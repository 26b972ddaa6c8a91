"""Minimal stand-in for ``mmocr.models.builder`` (reference mmocr/models/builder.py:10-26,50-72):
registries that honour ``dict(type='TPS_PP', **kwargs)`` / ``dict(type='TPSPreprocessor', ...)``.
When the real mmocr registries are importable, :func:`register_into_mmocr` adds our modules to
them under the reference's names so existing configs pick them up unchanged (INTEGRATION.md)."""
from __future__ import annotations

from typing import Any, Callable, Dict, Optional


class Registry:
    def __init__(self, name: str):
        self.name = name
        self._modules: Dict[str, type] = {}

    @property
    def module_dict(self):
        return self._modules

    def get(self, key: str):
        return self._modules.get(key)

    def register_module(self, name: Optional[str] = None, force: bool = False, module: Optional[type] = None):
        def _register(cls):
            key = name or cls.__name__
            if key in self._modules and not force:
                raise KeyError(f"{key} is already registered in {self.name}")
            self._modules[key] = cls
            return cls
        if module is not None:
            return _register(module)
        return _register

    def build(self, cfg: Dict[str, Any]):
        if not isinstance(cfg, dict) or "type" not in cfg:
            raise TypeError(f"cfg must be a dict with a 'type' key, got {cfg!r}")
        args = dict(cfg)
        kind = args.pop("type")
        cls = kind if isinstance(kind, type) else self._modules.get(kind)
        if cls is None:
            raise KeyError(f"{kind} is not in the {self.name} registry")
        return cls(**args)


BACKBONES = Registry("backbone")
PREPROCESSOR = Registry("preprocessor")
DECODERS = Registry("decoder")
ENCODERS = Registry("encoder")
CONVERTORS = Registry("convertor")
RECOGNIZERS = Registry("recognizer")
# the recogniser's losses (TFLoss); not registered into mmocr, which has its own
LOSSES = Registry("loss")
# the batched GPU test pipeline (tps_pp_b200/pipeline.py); not registered into mmocr: its transforms run per image on the host
PIPELINES = Registry("pipeline")


def build_backbone(cfg):
    """reference mmocr/models/builder.py:70-72; used for ``tpsnet`` at
    recognizer/encode_decode_recognizer.py:50-51."""
    return BACKBONES.build(cfg)


def build_preprocessor(cfg):
    """reference mmocr/models/builder.py:50-52."""
    return PREPROCESSOR.build(cfg)


def build_decoder(cfg):
    """reference mmocr/models/builder.py (``DECODERS``); used for ``decoder`` at recognizer/encode_decode_recognizer.py:60-66."""
    return DECODERS.build(cfg)


def build_encoder(cfg):
    """reference mmocr/models/builder.py (``ENCODERS``); used for ``encoder`` at recognizer/encode_decode_recognizer.py."""
    return ENCODERS.build(cfg)


def build_convertor(cfg):
    """reference mmocr/models/builder.py (``CONVERTORS``); used for ``label_convertor`` at recognizer/encode_decode_recognizer.py."""
    return CONVERTORS.build(cfg)


def build_loss(cfg):
    """reference mmocr/models/builder.py (``LOSSES``); used for ``loss`` at recognizer/encode_decode_recognizer.py."""
    return LOSSES.build(cfg)


def build_recognizer(cfg):
    """``dict(type='NRTR', backbone=..., tpsnet=..., encoder=..., decoder=..., label_convertor=...)`` -> the recogniser."""
    return RECOGNIZERS.build(cfg)


def register_into_mmocr(force: bool = True) -> bool:
    """Register the B200 modules into a real MMOCR install, replacing the stock classes (``ENCODERS`` too where the install
    exposes that registry)."""
    try:
        from mmocr.models.builder import BACKBONES as MB, DECODERS as MD, PREPROCESSOR as MP  # type: ignore
    except Exception:
        return False
    pairs = [(MB, BACKBONES), (MP, PREPROCESSOR), (MD, DECODERS)]
    try:
        from mmocr.models.builder import ENCODERS as ME  # type: ignore
        pairs.append((ME, ENCODERS))
    except Exception:
        pass
    for reg, ours in pairs:
        for key, cls in ours.module_dict.items():
            reg.register_module(name=key, force=force, module=cls)
    return True
