"""CPU check of the given-durations reference (tests/durations_oracle.py): with the predicted durations it reproduces
SynthesizerTrn.infer exactly, and edited durations give the alignment and length the contract states."""
import numpy as np
import torch

import util
from durations_oracle import infer_with_durations
from util import ov


def test_predicted_durations_reproduce_infer():
    hp = ov.tiny_hparams()
    model = ov.build_model(hp, seed=0)
    u = util.make_utterance(hp, 17, seed=3, sdp_ratio=0.4)
    ref, inter = util.oracle_run(model, u)
    d = inter["w_ceil"][0, 0].numpy().astype(np.int64)
    got, gi = infer_with_durations(model, u, d)
    assert torch.equal(gi["attn"], inter["attn"])
    assert torch.equal(got, ref)


def test_edited_durations_alignment_and_length():
    hp = ov.tiny_hparams()
    model = ov.build_model(hp, seed=0)
    u = util.make_utterance(hp, 9, seed=4, max_frames=64)
    d = np.array([0, 3, 1, 0, 0, 5, 2, 0, 1])
    audio, gi = infer_with_durations(model, u, d)
    assert int(gi["y_lengths"][0]) == d.sum() and audio.shape[-1] == d.sum() * hp.hop
    f2p = gi["attn"][0, 0].argmax(1).numpy()
    assert np.array_equal(f2p, np.repeat(np.arange(d.size), d))
    audio0, g0 = infer_with_durations(model, u, np.zeros(9, np.int64))
    assert int(g0["y_lengths"][0]) == 1 and audio0.shape[-1] == hp.hop and not g0["attn"].any()
