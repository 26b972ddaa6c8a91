"""Image-to-text NRTR recogniser built from the drop-in modules, so that ``nrtr_tps++.py`` runs without mmocr installed.

``AttnConvertor`` (registry ``CONVERTORS``; reference mmocr/models/textrecog/convertors/base.py + attn.py): the label
dictionary and the decode of class probabilities into strings.  ``NRTR`` (registry ``RECOGNIZERS``; reference
recognizer/nrtr.py over ``EncodeDecodeRecognizer``, recognizer/encode_decode_recognizer.py): ``backbone`` (with ``tpsnet``
called mid-way), ``encoder``, ``decoder`` and ``label_convertor`` built from config dicts, under the reference's sub-module
names so that ``backbone.*`` / ``tpsnet.*`` / ``encoder.*`` / ``decoder.*`` checkpoint keys load with ``strict=True``.
Inference only: ``simple_test`` (encode_decode_recognizer.py:184-225); training runs in mmocr.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch
import torch.nn as nn

from .registry import CONVERTORS, RECOGNIZERS, build_backbone, build_convertor, build_decoder, build_encoder, build_preprocessor

DICT36 = tuple("0123456789abcdefghijklmnopqrstuvwxyz")
DICT90 = tuple("0123456789abcdefghijklmnopqrstuvwxyz"
               "ABCDEFGHIJKLMNOPQRSTUVWXYZ!\"#$%&'()"
               "*+,-./:;<=>?@[\\]_`~")


@CONVERTORS.register_module()
class AttnConvertor:
    """Index order: the dictionary's characters, then ``<UKN>`` (``with_unknown``), ``<BOS/EOS>`` (start = end when
    ``start_end_same``), ``<PAD>``.  DICT90 with ``<UKN>``: 93 classes, start = end = 91, padding 92."""

    def __init__(self, dict_type="DICT90", dict_file=None, dict_list=None, with_unknown=True, max_seq_len=40, lower=False,
                 start_end_same=True):
        if dict_file is not None:
            raise ValueError("tps_pp_b200.AttnConvertor: dict_file is not supported; pass dict_type='DICT36' / 'DICT90' or dict_list")
        if dict_list is not None:
            self.idx2char = list(dict_list)
        elif dict_type in ("DICT36", "DICT90"):
            self.idx2char = list(DICT36 if dict_type == "DICT36" else DICT90)
        else:
            raise ValueError(f"tps_pp_b200.AttnConvertor: dict_type must be 'DICT36' or 'DICT90', got {dict_type!r}")
        self.max_seq_len = max_seq_len
        self.lower = lower
        self.start_end_same = start_end_same
        self.unknown_idx = None
        if with_unknown:
            self.idx2char.append("<UKN>")
            self.unknown_idx = len(self.idx2char) - 1
        self.idx2char.append("<BOS/EOS>")
        self.start_idx = len(self.idx2char) - 1
        if not start_end_same:
            self.idx2char.append("<BOS/EOS>")
        self.end_idx = len(self.idx2char) - 1
        self.idx2char.append("<PAD>")
        self.padding_idx = len(self.idx2char) - 1
        self.char2idx = {c: i for i, c in enumerate(self.idx2char)}

    def num_classes(self) -> int:
        return len(self.idx2char)

    def tensor2idx(self, outputs: torch.Tensor, img_metas=None):
        """Class probabilities [N, T, C] -> (indexes, scores): per image the arg-max of each step, padding skipped, cut at the
        end index.  The arg-max runs on the tensor's device and one copy brings index and score of every step to the host."""
        val, idx = torch.max(outputs.detach(), -1)
        both = torch.stack([idx.double(), val.double()]).cpu()      # indices < 2**53 and fp32 scores are exact in fp64
        indexes, scores = [], []
        for ids, vals in zip(both[0].long().tolist(), both[1].tolist()):
            str_index, str_score = [], []
            for i, v in zip(ids, vals):
                if i == self.padding_idx:
                    continue
                if i == self.end_idx:
                    break
                str_index.append(i)
                str_score.append(v)
            indexes.append(str_index)
            scores.append(str_score)
        return indexes, scores

    def idx2str(self, indexes: Sequence[Sequence[int]]) -> List[str]:
        return ["".join(self.idx2char[i] for i in index) for index in indexes]


@RECOGNIZERS.register_module()
class NRTR(nn.Module):
    """``EncodeDecodeRecognizer`` inference over the drop-in modules.  As in the reference, the decoder config is completed
    from the convertor (``num_classes``, ``start_idx``, ``padding_idx``) and ``max_seq_len``."""

    def __init__(self, preprocessor=None, backbone=None, encoder=None, decoder=None, loss=None, label_convertor=None,
                 train_cfg=None, test_cfg=None, max_seq_len=40, pretrained=None, init_cfg=None, tpsnet=None):
        super().__init__()
        if backbone is None or decoder is None or label_convertor is None:
            raise ValueError("tps_pp_b200.NRTR needs backbone, decoder and label_convertor configs")
        self.preprocessor = build_preprocessor(preprocessor) if preprocessor is not None else None
        self.backbone = build_backbone(backbone)
        self.tpsnet = build_backbone(tpsnet) if tpsnet is not None else None
        self.encoder = build_encoder(encoder) if encoder is not None else None
        self.label_convertor = build_convertor(dict(label_convertor, max_seq_len=max_seq_len))
        self.decoder = build_decoder(dict(decoder, num_classes=self.label_convertor.num_classes(),
                                          start_idx=self.label_convertor.start_idx, padding_idx=self.label_convertor.padding_idx,
                                          max_seq_len=max_seq_len))
        self.loss_cfg, self.train_cfg, self.test_cfg, self.init_cfg = loss, train_cfg, test_cfg, init_cfg
        self.max_seq_len = max_seq_len

    def extract_feat(self, img):
        """encode_decode_recognizer.py: optional preprocessor, then the backbone with the rectifier called mid-way."""
        if self.preprocessor is not None:
            img = self.preprocessor(img)
        return self.backbone(img, self.tpsnet, True)["output"]

    def simple_test(self, img, img_metas: Optional[list] = None, **kwargs):
        """Images [N, 3, H, W] -> ``[dict(text=str, score=[per-character probabilities])]`` (encode_decode_recognizer.py:184-225).
        Without ``img_metas`` every image has ``valid_ratio`` 1.0."""
        if img_metas is None:
            img_metas = [dict(valid_ratio=1.0) for _ in range(img.shape[0])]
        feat = self.extract_feat(img)
        out_enc = self.encoder(feat, img_metas) if self.encoder is not None else None
        out_dec = self.decoder(feat, out_enc, None, img_metas, train_mode=False)
        indexes, scores = self.label_convertor.tensor2idx(out_dec, img_metas)
        strings = self.label_convertor.idx2str(indexes)
        return [dict(text=s, score=sc) for s, sc in zip(strings, scores)]

    def forward(self, img, img_metas=None, return_loss=False, **kwargs):
        if return_loss:
            raise RuntimeError("tps_pp_b200.NRTR is the inference recogniser: training (return_loss=True) runs in mmocr, with "
                               "the drop-in modules registered by tps_pp_b200.register_into_mmocr()")
        return self.simple_test(img, img_metas, **kwargs)
