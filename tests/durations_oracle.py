"""Reference for synthesis at given phoneme durations.

``infer_with_durations`` restates ``SynthesizerTrn.infer`` (oracle/vits.py) with ``w_ceil`` replaced by the caller's
integer durations: the duration predictors' outputs are not used, so their statements are left out.  The CPU test
tests/test_durations_oracle.py holds it equal to ``infer`` when the given durations are the predicted ones.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import vits as ov


@torch.no_grad()
def infer_with_durations(model, u, durations, dtype=torch.float32):
    """u: a tests/util.make_utterance dict (its noise_zp must have >= T_y frames); durations: int [t_x].
    -> (audio [1, 1, T_y * hop], dict(attn [1, 1, T_y, t_x], y_lengths [1], w_ceil [1, 1, t_x]))"""
    m = model if dtype == torch.float32 else model.double()
    cast = lambda t: t.to(dtype) if t.is_floating_point() else t
    g = m.emb_g(torch.tensor([u["sid"]])).unsqueeze(-1)
    x, m_p, logs_p, x_mask = m.enc_p(u["x"], torch.tensor([u["t_x"]]), u["tone"], u["lang"], cast(u["bert"]), cast(u["style"]), g=g)
    w_ceil = torch.as_tensor(np.asarray(durations, dtype=np.int64)).to(x_mask.dtype).reshape(1, 1, -1) * x_mask
    y_lengths = torch.clamp_min(torch.sum(w_ceil, [1, 2]), 1).long()
    y_mask = ov.sequence_mask(y_lengths, None).unsqueeze(1).to(x_mask.dtype)
    attn_mask = x_mask.unsqueeze(2) * y_mask.unsqueeze(-1)
    attn = ov.generate_path(w_ceil, attn_mask)
    m_p = torch.matmul(attn.squeeze(1), m_p.transpose(1, 2)).transpose(1, 2)
    logs_p = torch.matmul(attn.squeeze(1), logs_p.transpose(1, 2)).transpose(1, 2)
    eps = cast(u["noise_zp"])[:, :, :m_p.shape[2]]
    z_p = m_p + eps * torch.exp(logs_p) * u["noise_scale"]
    z = m.flow.forward_reverse(z_p, y_mask, g)
    o = m.dec(z * y_mask, g=g)
    if dtype != torch.float32:
        model.float()
    return o, dict(attn=attn, y_lengths=y_lengths, w_ceil=w_ceil)
