"""Image-to-text NRTR recogniser built from the drop-in modules, so that ``nrtr_tps++.py`` runs without mmocr installed.

``AttnConvertor`` (registry ``CONVERTORS``; reference mmocr/models/textrecog/convertors/base.py + attn.py): the label
dictionary and the decode of class probabilities into strings.  ``NRTR`` (registry ``RECOGNIZERS``; reference
recognizer/nrtr.py over ``EncodeDecodeRecognizer``, recognizer/encode_decode_recognizer.py): ``backbone`` (with ``tpsnet``
called mid-way), ``encoder``, ``decoder`` and ``label_convertor`` built from config dicts, under the reference's sub-module
names so that ``backbone.*`` / ``tpsnet.*`` / ``encoder.*`` / ``decoder.*`` checkpoint keys load with ``strict=True``.
Inference: ``simple_test`` (encode_decode_recognizer.py:184-225).  Training: ``forward_train`` (encode_decode_recognizer.py:
``forward_train``) -- the labels through ``AttnConvertor.str2tensor``, the encoder and the teacher-forced decoder on native
attention and dense kernels (``nrtr_train``), ``TFLoss`` (registry ``LOSSES``; reference losses/ce_loss.py).
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch
import torch.nn as nn

from . import functional as TF
from . import nrtr_train
from .nrtr import NRTRDecoder, NRTREncoder, valid_lengths
from .registry import (CONVERTORS, LOSSES, RECOGNIZERS, build_backbone, build_convertor, build_decoder, build_encoder, build_loss,
                       build_preprocessor)

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

    def str2idx(self, strings: Sequence[str]) -> List[List[int]]:
        """convertors/base.py ``str2idx``: each string (lower-cased with ``lower``) to its character indexes; a character outside
        the dictionary is ``<UKN>``, or raises ``ValueError`` without ``with_unknown``."""
        if not isinstance(strings, (list, tuple)) or not all(isinstance(s, str) for s in strings):
            raise TypeError("tps_pp_b200.AttnConvertor.str2idx takes a list of strings")
        indexes = []
        for string in strings:
            if self.lower:
                string = string.lower()
            index = []
            for char in string:
                i = self.char2idx.get(char, self.unknown_idx)
                if i is None:
                    raise ValueError(f"tps_pp_b200.AttnConvertor: character {char!r} is not in the dictionary; use a dictionary that "
                                     "holds it or with_unknown=True")
                index.append(i)
            indexes.append(index)
        return indexes

    def str2tensor(self, strings: Sequence[str]):
        """convertors/attn.py ``str2tensor``: ``targets`` (per string its character indexes, LongTensor) and ``padded_targets``
        [N, max_seq_len] -- ``[start, chars..., end]`` filled up with ``padding_idx``, cut at ``max_seq_len`` when longer."""
        targets, padded = [], []
        for index in self.str2idx(strings):
            targets.append(torch.LongTensor(index))
            seq = [self.start_idx] + index + [self.end_idx]
            row = torch.full((self.max_seq_len,), self.padding_idx, dtype=torch.long)
            seq = seq[:self.max_seq_len]
            row[:len(seq)] = torch.LongTensor(seq)
            padded.append(row)
        return dict(targets=targets, padded_targets=torch.stack(padded, 0))


@LOSSES.register_module()
class TFLoss(nn.Module):
    """mmocr 0.4 ``TFLoss`` (losses/ce_loss.py): the cross-entropy of ``outputs[:, :-1]`` against ``padded_targets[:, 1:]``
    (each step predicts the next token), flattened, with ``reduction='none'`` -- one loss per (image, step), 0 where the target is
    ``ignore_index`` (the recogniser sets it to the padding index).  Returns ``dict(loss_ce=...)``."""

    def __init__(self, ignore_index=-1, reduction="none", flatten=True, **kwargs):
        super().__init__()
        if not isinstance(flatten, bool):
            raise TypeError("tps_pp_b200.TFLoss: flatten must be a bool")
        self.flatten = flatten
        self.loss_ce = nn.CrossEntropyLoss(ignore_index=ignore_index, reduction=reduction)

    def format(self, outputs, targets_dict):
        outputs = outputs[:, :-1, :].contiguous()
        targets = targets_dict["padded_targets"][:, 1:].contiguous()
        if self.flatten:
            return outputs.view(-1, outputs.size(-1)), targets.view(-1)
        return outputs.permute(0, 2, 1).contiguous(), targets

    def forward(self, outputs, targets_dict, img_metas=None):
        outputs, targets = self.format(outputs, targets_dict)
        return dict(loss_ce=self.loss_ce(outputs, targets.to(outputs.device)))


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
        # as EncodeDecodeRecognizer.__init__: the loss ignores the padding index
        self.loss = build_loss(dict(loss if loss is not None else dict(type="TFLoss"), ignore_index=self.label_convertor.padding_idx))
        self.last_train_native = None

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

    def forward_train(self, img, img_metas):
        """encode_decode_recognizer.py ``forward_train``: images [N, 3, H, W] and one meta per image with its ground-truth
        ``text`` -> ``dict(loss_ce=[N * (max_seq_len - 1)] per-step losses)``.  Each image's ``valid_ratio`` is
        ``resize_shape[1] / W`` where the meta has ``resize_shape``, else its ``valid_ratio`` (default 1.0).  The backbone runs in
        its training form (``TPS_PP`` on its native training path); the encoder and the teacher-forced decoder run on native
        attention and dense kernels, forward and backward (``nrtr_train``); ``last_train_native`` records whether every attention
        call of both halves ran the native kernels."""
        if img_metas is None or any(not isinstance(m, dict) or "text" not in m for m in img_metas):
            raise RuntimeError("tps_pp_b200.NRTR.forward_train: each image's ground-truth `text` must come in img_metas, as mmocr's "
                               "training pipeline provides it")
        if len(img_metas) != img.shape[0]:
            raise ValueError(f"tps_pp_b200.NRTR.forward_train: {img.shape[0]} images but {len(img_metas)} img_metas")
        if not isinstance(self.encoder, NRTREncoder) or not isinstance(self.decoder, NRTRDecoder):
            raise RuntimeError("tps_pp_b200.NRTR.forward_train needs the NRTREncoder and NRTRDecoder of this package")
        self.last_train_native = False
        calls = TF._Attention.calls
        metas = []
        for m in img_metas:
            ratio = m["resize_shape"][1] / img.shape[-1] if "resize_shape" in m else m.get("valid_ratio", 1.0)
            metas.append(dict(m, valid_ratio=ratio))
        feat = self.extract_feat(img)
        targets_dict = self.label_convertor.str2tensor([m["text"] for m in metas])
        lens = valid_lengths(feat.shape[2] * feat.shape[3], metas)
        out_enc = nrtr_train.encoder_train(self.encoder, feat, lens)
        out_dec = nrtr_train.decoder_train(self.decoder, targets_dict["padded_targets"], out_enc, lens)
        # every attention call of both halves ran the native kernels: one per encoder layer, two per decoder layer
        self.last_train_native = TF._Attention.calls - calls == len(self.encoder.layer_stack) + 2 * len(self.decoder.layer_stack)
        return self.loss(out_dec, targets_dict, metas)

    def forward(self, img, img_metas=None, return_loss=False, **kwargs):
        if return_loss:
            return self.forward_train(img, img_metas)
        return self.simple_test(img, img_metas, **kwargs)
