"""CPU checks of the assist-text references (tests/assist_oracle.py): upstream's loop as ``assist_features`` against a
literal transcription of it, the limits w = 0 and w = 1, the mean over every token (CLS and SEP included), and the
library's restated numerics against the float64 blend."""
import numpy as np
import pytest
import torch

from assist_oracle import assist_features, restated_features, restated_mean


def _inputs(seed=0, t_tok=9, t_a=6, hidden=16):
    rng = np.random.default_rng(seed)
    res = rng.standard_normal((t_tok, hidden)).astype(np.float32)
    style_res = rng.standard_normal((t_a, hidden)).astype(np.float32)
    word2ph = np.array([3, 1, 2, 0, 4, 1, 2, 2, 1], np.int32)[:t_tok]
    return res, style_res, word2ph


def _literal_loop(res, style_res, word2ph, w):
    """style_bert_vits2/nlp/japanese/bert_feature.py, extract_bert_feature, line by line in numpy (float64)."""
    res, style_res = res.astype(np.float64), style_res.astype(np.float64)
    style_res_mean = style_res.mean(0)
    phone_level_feature = []
    for i in range(len(word2ph)):
        repeat_feature = np.tile(res[i], (word2ph[i], 1)) * (1 - w) + np.tile(style_res_mean, (word2ph[i], 1)) * w
        phone_level_feature.append(repeat_feature)
    return np.concatenate(phone_level_feature, axis=0).T


@pytest.mark.parametrize("w", [0.3, 0.7, 1.0, -0.5, 2.0])
def test_assist_features_is_upstreams_loop(w):
    res, style_res, word2ph = _inputs()
    got = assist_features(res, style_res, word2ph, w, torch.float64).numpy()
    want = _literal_loop(res, style_res, word2ph, w)
    assert got.shape == (res.shape[1], int(word2ph.sum()))
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-14)
    got32 = assist_features(res, style_res, word2ph, w, torch.float32).numpy()
    assert got32.dtype == np.float32
    np.testing.assert_allclose(got32, want, rtol=0, atol=1e-5)


def test_weight_zero_is_the_plain_repeat():
    res, style_res, word2ph = _inputs(1)
    plain = np.repeat(res, word2ph, axis=0).T
    assert np.array_equal(assist_features(res, style_res, word2ph, 0.0, torch.float32).numpy(), plain)
    assert np.array_equal(restated_features(res, style_res, word2ph, 0.0), plain)
    assert np.array_equal(restated_features(res, None, word2ph, 0.7), plain)


def test_weight_one_gives_the_mean_in_every_phoneme_column():
    res, style_res, word2ph = _inputs(2)
    got = assist_features(res, style_res, word2ph, 1.0).numpy()
    mean = style_res.astype(np.float64).mean(0)
    np.testing.assert_allclose(got, np.repeat(mean[:, None], got.shape[1], axis=1), rtol=0, atol=1e-15)
    r = restated_features(res, style_res, word2ph, 1.0)
    assert (r == restated_mean(style_res)[:, None]).all()  # c_row = 0 and c_mean = 1 are exact


def test_mean_covers_cls_and_sep():
    res, style_res, word2ph = _inputs(3)
    style_res[0] += 100.0   # CLS
    style_res[-1] -= 40.0   # SEP
    got = assist_features(res, style_res, word2ph, 1.0).numpy()[:, 0]
    np.testing.assert_allclose(got, style_res.astype(np.float64).mean(0), rtol=0, atol=1e-12)
    assert np.abs(got - style_res[1:-1].astype(np.float64).mean(0)).min() > 1.0


def test_restated_numerics_against_the_float64_blend():
    rng = np.random.default_rng(4)
    res = rng.standard_normal((40, 1024)).astype(np.float32) * 3
    style_res = rng.standard_normal((30, 1024)).astype(np.float32) * 3
    word2ph = rng.integers(0, 5, size=40).astype(np.int32)
    for w in (0.3, 0.7, 1.0):
        got = restated_features(res, style_res, word2ph, w)
        want = assist_features(res, style_res, word2ph, float(np.float32(w))).numpy()
        # two float32 products and a float32 sum: a few ulps of the magnitudes involved
        assert np.abs(got - want).max() <= 4 * np.finfo(np.float32).eps * (np.abs(res).max() + np.abs(want).max())
    # the mean is the fp64 sum in token order, rounded once: within half an ulp of the exact mean
    m = restated_mean(style_res)
    exact = style_res.astype(np.float64).mean(0)
    assert np.abs(m - exact).max() <= np.abs(exact).max() * np.finfo(np.float32).eps
