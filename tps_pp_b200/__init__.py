"""tps_pp_b200 -- B200-native (sm_100a) TPS++ rectifier hot path behind the reference's module API.

Public surface (mirrors what a user of simplify23/TPS_PP touches for this path):

    from tps_pp_b200 import TPS_PP, TPSPreprocessor, BasePreprocessor, MORAN, ResNetABI_v2_large
    from tps_pp_b200 import build_backbone, build_preprocessor     # dict(type='TPS_PP', ...)
    from tps_pp_b200 import NRTREncoder, NRTRDecoder, AttnConvertor, NRTR, build_recognizer   # image -> text
    from tps_pp_b200 import TFLoss, build_loss          # NRTR.forward_train: teacher-forced loss on native kernels
    from tps_pp_b200 import init_recognizer, model_inference, TestPipeline    # uint8 images / files -> strings
    from tps_pp_b200.functional import tps_warp, grid_sample_border
"""
from .registry import (BACKBONES, CONVERTORS, DECODERS, ENCODERS, LOSSES, PIPELINES, PREPROCESSOR, RECOGNIZERS, build_backbone,
                       build_convertor, build_decoder, build_encoder, build_loss, build_preprocessor, build_recognizer,
                       register_into_mmocr)
from .rectifier import TPS_PP
from .classical import MORAN, BasePreprocessor, TPSPreprocessor
from .backbone import ResNetABI_v2_large
from .nrtr import NRTRDecoder, NRTREncoder
from .recognizer import NRTR, AttnConvertor, TFLoss
from .pipeline import TestPipeline
from .apis import init_recognizer, model_inference

__all__ = ["TPS_PP", "TPSPreprocessor", "BasePreprocessor", "MORAN", "ResNetABI_v2_large", "NRTRDecoder", "NRTREncoder",
           "AttnConvertor", "NRTR", "TFLoss", "TestPipeline", "init_recognizer", "model_inference", "BACKBONES", "PREPROCESSOR", "DECODERS",
           "ENCODERS", "CONVERTORS", "RECOGNIZERS", "LOSSES", "PIPELINES",
           "build_backbone", "build_preprocessor", "build_decoder", "build_encoder", "build_convertor", "build_loss", "build_recognizer",
           "register_into_mmocr"]
__version__ = "0.1.0"
