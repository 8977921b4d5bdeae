"""References for Style-Bert-VITS2's assist text (assist_text / assist_text_weight).

``assist_features`` is upstream's loop (style_bert_vits2/nlp/japanese/bert_feature.py, extract_bert_feature) in torch, in
float32 or float64.  ``restated_features`` is the library's numerical contract (include/sbv2_b200.h, sbv2_assist_text) in
numpy: the device kernels and the host restatement in host/tts.cpp must equal it bit for bit.
"""
from __future__ import annotations

import numpy as np
import torch


def assist_features(res, style_res, word2ph, weight: float, dtype=torch.float64) -> torch.Tensor:
    """res: DeBERTa rows of the text [T_tok, H]; style_res: those of the assist text [T_a, H], CLS and SEP included.
    -> phone-level features [H, sum(word2ph)] (upstream returns ``phone_level_feature.T``)."""
    res = torch.as_tensor(np.asarray(res)).to(dtype)
    style_res = torch.as_tensor(np.asarray(style_res)).to(dtype)
    style_res_mean = style_res.mean(0)
    phone_level_feature = []
    for i in range(len(word2ph)):
        repeat_feature = (res[i].repeat(int(word2ph[i]), 1) * (1 - weight)
                          + style_res_mean.repeat(int(word2ph[i]), 1) * weight)
        phone_level_feature.append(repeat_feature)
    phone_level_feature = torch.cat(phone_level_feature, dim=0)
    return phone_level_feature.T


def restated_mean(style_res: np.ndarray) -> np.ndarray:
    """(float)((sum_t (double)F[t][c]) / n): one fp64 accumulator per column, summed in token order."""
    f = np.asarray(style_res, dtype=np.float32)
    acc = np.zeros(f.shape[1], np.float64)
    for t in range(f.shape[0]):
        acc += f[t].astype(np.float64)
    return (acc / np.float64(f.shape[0])).astype(np.float32)


def restated_features(res: np.ndarray, style_res, word2ph, weight: float) -> np.ndarray:
    """The library's blend: rows fl(fl(row * (float)(1 - (double)w)) + fl(mean * w)); style_res None or w == 0: the plain
    repeat.  -> float32 [H, sum(word2ph)]."""
    rows = np.repeat(np.asarray(res, dtype=np.float32), np.asarray(word2ph), axis=0)
    w = np.float32(weight)
    if style_res is not None and w != 0:
        c_row, c_mean = np.float32(1.0 - np.float64(w)), w
        rows = rows * c_row + restated_mean(style_res) * c_mean  # two float32 products and a float32 sum (numpy forms no FMA)
    return np.ascontiguousarray(rows.T)
