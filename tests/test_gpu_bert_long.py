"""DeBERTa on sentences longer than 512 tokens (up to kMaxBertTokens = 32768), on a B200 (-m gpu).

* The multi-tile attention kernels (bert_attention_tc.cu) through sbv2_debug_deberta_attention against float64 on the
  exact fp16 operands they read, on a ragged batch up to 2048 tokens.  The position tables make rows 0, 1, 510 and 511
  differ strongly, so an index clamped at +-511 instead of the table's bound +-512 (rel <= -512 reading row 1, not 0) fails
  the bar; the test checks that it would.  Far tile pairs (|qt - kt| >= 5) take a reduced path that must be bit-identical
  to the generic one, and each utterance alone must be bit-identical to its rows in the batch.
* The whole forward (tiny configuration, both numerics modes) against HF at 513 ... 2048 tokens, and the tensor-core
  attention against the CUDA-core kernel (SBV2_B200_BERT_ATTN=simt) on a ragged batch mixing 1 ... 2048 tokens.
* The cap: 32768 tokens run, 32769 return SBV2_ERR_INVALID_ARGUMENT.
* DeBERTa-large at 2048 tokens against HF fp32, and the device-resident chain with a ~1200-token sentence.
"""
import importlib.util
import os

import numpy as np
import pytest
import torch
from transformers.models.deberta_v2.modeling_deberta_v2 import make_log_bucket_position

import util
from util import ov
from oracle import deberta as od

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TOL = {"exact": (2e-4, 2e-5), "fp16": (3e-2, 5e-3)}        # the feature bars of test_gpu_bert.py
FEAT_TOL = {"exact": (6e-4, 1.5e-4), "fp16": (3e-2, 5e-3)}  # the DeBERTa-large bars of test_gpu_fullsize.py
SPAN, HEADS, SC = 256, 2, 16.0


@pytest.fixture(scope="module")
def S(lib_built):
    spec = importlib.util.spec_from_file_location("sbv2_b200_build", os.path.join(ROOT, "sbv2-api_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()  # the debug library carries the attention hook; a no-op when up to date
    import sbv2_b200
    if sbv2_b200.device_count() < 1:
        pytest.fail("GPU tests selected but no B200 is visible")
    return sbv2_b200


def close(got, ref, tol):
    err = float(np.abs(got - ref).max())
    rel = float(np.linalg.norm(got - ref) / (np.linalg.norm(ref) + 1e-30))
    assert err <= tol[0] and rel <= tol[1], f"max-abs {err:.3e}, rel-fro {rel:.3e} (|ref| max {np.abs(ref).max():.2f})"
    return err, rel


def make_model(S, onnx, mode, simt=False):
    env = {"SBV2_B200_BERT": "fp16"} if mode == "fp16" else {}
    if simt:
        env["SBV2_B200_BERT_ATTN"] = "simt"
    os.environ.update(env)
    try:
        return S.Model(onnx, bert=True)
    finally:
        for k in env:
            del os.environ[k]


# ---- the attention kernels alone -------------------------------------------------------------------------------------
LENS = [2048, 513, 640, 641, 768, 769, 1, 130, 1100]


def hf_index(rel: np.ndarray) -> np.ndarray:
    b = make_log_bucket_position(torch.from_numpy(rel), SPAN, 2 * SPAN)
    return torch.clamp(b + SPAN, 0, 2 * SPAN - 1).long().numpy()


def ref_attention(q, k, v, pk, pq, clamp=None):
    """float64 DeBERTa attention of one head: q, k, v [L, 64], pk, pq [2*span, 64].  clamp: distances clipped to +-clamp
    first (the mistake the test must catch)."""
    L = len(q)
    rel = np.arange(L)[:, None] - np.arange(L)[None, :]
    if clamp is not None:
        rel = np.clip(rel, -clamp, clamp)
    ix = hf_index(rel)
    c2p = np.take_along_axis(q @ pk.T, ix, axis=1)             # q_i . pk[ix(i - j)]
    p2c = np.take_along_axis(k @ pq.T, ix.T, axis=1).T         # k_j . pq[ix(i - j)]
    s = (q @ k.T + c2p + p2c) / np.sqrt(3 * 64)
    s -= s.max(axis=1, keepdims=True)
    p = np.exp(s)
    return (p / p.sum(axis=1, keepdims=True)) @ v


@pytest.fixture(scope="module")
def attn_inputs():
    rng = np.random.default_rng(7)
    n, H = sum(LENS), HEADS * 64
    qkv = rng.standard_normal((n, 3 * H))
    pos = [0.5 * rng.standard_normal((2 * SPAN, H)) for _ in range(2)]
    for t in pos:  # rows 0 / 1 and 510 / 511 strongly different: a clamp at +-511 reads the wrong one of each pair
        u, w = 2.0 * rng.standard_normal(H), 2.0 * rng.standard_normal(H)
        t[0], t[1], t[510], t[511] = u, -u, w, -w
    split = lambda x: (lambda h0: np.stack([h0, (x * SC - h0.astype(np.float64)).astype(np.float16)]))(
        (x * SC).astype(np.float16))  # two fp16 terms of x * sc
    ops = {"fp16": (qkv.astype(np.float16)[None], pos[0].astype(np.float16)[None], pos[1].astype(np.float16)[None])}
    ops["exact"] = (split(qkv), split(pos[0]), split(pos[1]))
    # the values each mode's kernel reads, in float64
    val = {m: tuple(a.astype(np.float64).sum(axis=0) / (SC if m == "exact" else 1.0) for a in o) for m, o in ops.items()}
    return ops, val


def per_head(x, h):
    return x[:, h * 64:(h + 1) * 64]


@pytest.mark.parametrize("kernel", ["multi", "exact-multi", "simt"])
def test_attention_against_float64(S, attn_inputs, kernel):
    """Bars: fp16 operands (multi, simt) round the two bias terms and P to fp16 and the context once more; with |c2p| up
    to ~50 that is ~2e-3 in a logit, <= ~1e-2 in a context of magnitude ~3.  Exact: every product is fp32-grade (two-term
    splits), the bias fp32, P and the context two fp16 terms: ~1e-6 relative, bar 1e-4.  The ±511 clamp moves contexts by O(1)."""
    ops, val = attn_inputs
    mode = "exact" if kernel == "exact-multi" else "fp16"
    qkv, pk, pq = ops[mode]
    got = S.debug_deberta_attention(qkv, pk, pq, LENS, HEADS, kernel, far_pairs=True, sc=SC).astype(np.float64)
    ctx = got.sum(axis=0) / (SC if mode == "exact" else 1.0)
    vq, vk, vv = (lambda a: (a[:, :HEADS * 64], a[:, HEADS * 64:2 * HEADS * 64], a[:, 2 * HEADS * 64:]))(val[mode][0])
    bar = 1e-4 if mode == "exact" else 2e-2
    worst, wrong_min = 0.0, np.inf
    off = 0
    for L in LENS:
        for h in range(HEADS):
            sl = slice(off, off + L)
            args = (per_head(vq[sl], h), per_head(vk[sl], h), per_head(vv[sl], h), per_head(val[mode][1], h), per_head(val[mode][2], h))
            g = per_head(ctx[sl], h)
            err = float(np.abs(g - ref_attention(*args)).max())
            worst = max(worst, err)
            assert err <= bar, f"{kernel} L={L} head {h}: max-abs {err:.3e} > {bar}"
            if L >= 640:  # queries with keys at rel <= -512 exist: the wrong clamp must be visible
                wrong_min = min(wrong_min, float(np.abs(g - ref_attention(*args, clamp=511)).max()))
        off += L
    print(f"{kernel}: max-abs error vs float64 {worst:.3e} (bar {bar}); vs the +-511-clamp reference >= {wrong_min:.3e}")
    assert wrong_min > 5 * bar


@pytest.mark.parametrize("kernel", ["multi", "exact-multi"])
def test_far_pairs_bit_identical_and_batch_equals_singles(S, attn_inputs, kernel):
    """The reduced far-pair path against the generic path (far_pairs off), and each utterance alone against the batch."""
    ops, _ = attn_inputs
    qkv, pk, pq = ops["exact" if kernel == "exact-multi" else "fp16"]
    far = S.debug_deberta_attention(qkv, pk, pq, LENS, HEADS, kernel, far_pairs=True, sc=SC)
    gen = S.debug_deberta_attention(qkv, pk, pq, LENS, HEADS, kernel, far_pairs=False, sc=SC)
    diff = np.flatnonzero((far.view(np.uint16) != gen.view(np.uint16)).any(axis=(0, 2)))
    assert diff.size == 0, f"{diff.size} rows differ between the far-pair and the generic path"
    off = 0
    for L in LENS:
        one = S.debug_deberta_attention(qkv[:, off:off + L], pk, pq, [L], HEADS, kernel, far_pairs=True, sc=SC)
        assert np.array_equal(one.view(np.uint16), far[:, off:off + L].view(np.uint16)), f"L={L}"
        off += L


# ---- the whole forward -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tiny(S):
    from sbv2_b200 import assets
    cfg = od.tiny_config()
    hf = od.build_model(cfg, seed=1)
    onnx = assets.deberta_onnx(od.state_dict_numpy(hf))
    return cfg, hf, onnx, {m: make_model(S, onnx, m) for m in ("exact", "fp16")}


@pytest.mark.parametrize("s", [513, 641, 769, 1024, 1500, 2048])
def test_tiny_matches_hf_beyond_512(tiny, s):
    cfg, hf, _, models = tiny
    ids = torch.randint(3, cfg.vocab_size, (1, s), generator=torch.Generator().manual_seed(300 + s))
    ref = od.predict(hf, ids, torch.ones_like(ids))[0].numpy()
    for mode, model in models.items():
        got = model.predict(ids[0].numpy(), np.ones(s, np.int64))
        e = close(got, ref, TOL[mode])
        print(f"tiny S={s} [{mode}] vs HF: max-abs {e[0]:.3e}, rel-Frobenius {e[1]:.3e}")


@pytest.mark.parametrize("mode", ["fp16", "exact"])
def test_tensor_core_vs_cuda_core_ragged(S, tiny, mode):
    """Right-padded ragged batch across the single-tile, multi-tile and far-pair regimes.  Each row is compared with its own
    single call: bit for bit where the two calls' GEMMs take the same path, else within the mode's bar (a call's token
    count decides split-K and the weight packing, so in this configuration most rows do not)."""
    cfg, _, onnx, models = tiny
    tc, simt = models[mode], make_model(S, onnx, mode, simt=True)
    lens = [1, 128, 129, 512, 513, 1300, 2048]
    smax = max(lens)
    ids = torch.randint(3, cfg.vocab_size, (len(lens), smax), generator=torch.Generator().manual_seed(31)).numpy()
    mask = np.zeros_like(ids)
    for b, n in enumerate(lens):
        mask[b, :n] = 1
    a, b_ = tc.predict_batch(ids, mask), simt.predict_batch(ids, mask)
    assert a.shape == (len(lens), smax, cfg.hidden_size) and np.isfinite(a).all()
    same = 0
    for i, n in enumerate(lens):
        assert not a[i, n:].any() and not b_[i, n:].any()
        close(a[i, :n], b_[i, :n], TOL[mode])
        single = tc.predict(ids[i, :n], np.ones(n, np.int64))
        if np.array_equal(single, a[i, :n]):
            same += 1
        else:  # the bar test_gpu_fullsize.py sets between a split-K call and the same sentence in a batch
            close(single, a[i, :n], (TOL[mode][0], 2 * FEAT_TOL[mode][1]))
    print(f"[{mode}] rows bit-identical to their single call: {same} of {len(lens)}")


def test_cap(S, tiny):
    cfg, _, onnx, models = tiny
    model, simt = models["fp16"], make_model(S, onnx, "fp16", simt=True)
    n = 32768
    ids = np.random.default_rng(1).integers(3, cfg.vocab_size, n).astype(np.int64)
    a = model.predict(ids, np.ones(n, np.int64))
    assert a.shape == (n, cfg.hidden_size) and np.isfinite(a).all()
    e = close(a, simt.predict(ids, np.ones(n, np.int64)), TOL["fp16"])
    print(f"32768 tokens [fp16] tensor-core vs CUDA-core attention: max-abs {e[0]:.3e}, rel-Frobenius {e[1]:.3e}")
    with pytest.raises(S.Sbv2Error) as ex:
        model.predict(np.append(ids, 5), np.ones(n + 1, np.int64))
    assert ex.value.status == S.ERR_INVALID_ARGUMENT
    with pytest.raises(S.Sbv2Error) as ex:
        model.predict_batch(np.ones((2, n + 1), np.int64), np.ones((2, n + 1), np.int64))
    assert ex.value.status == S.ERR_INVALID_ARGUMENT


def test_deberta_large_2048(S):
    from sbv2_b200 import assets
    cfg = od.deberta_config()
    hf = od.build_model(cfg, seed=1)
    onnx = assets.deberta_onnx(od.state_dict_numpy(hf))
    ids = torch.randint(3, cfg.vocab_size, (1, 2048), generator=torch.Generator().manual_seed(24))
    ref = od.predict(hf, ids, torch.ones_like(ids))[0].numpy()
    del hf
    for mode in ("exact", "fp16"):
        got = make_model(S, onnx, mode).predict(ids[0].numpy(), np.ones(2048, np.int64))
        e = close(got, ref, FEAT_TOL[mode])
        print(f"DeBERTa-large S=2048 [{mode}] vs HF fp32: max-abs {e[0]:.3e}, rel-Frobenius {e[1]:.3e}")


# ---- the chain -------------------------------------------------------------------------------------------------------
def test_long_sentence_chain(S):
    """A ~1200-token sentence (one line with split_sentences = false) through the device-resident chain and the holder."""
    from sbv2_b200 import assets
    hp = ov.tiny_hparams(bert_dim=128)
    _, onnx = util.synth_assets(hp, seed=0)
    cfg = od.tiny_config()
    bert_onnx = assets.deberta_onnx(od.state_dict_numpy(od.build_model(cfg, seed=1)))
    synth, bert = S.Model(onnx, bert=False), S.Model(bert_onnx, bert=True)
    t_x = 4201  # odd, as the frontend's blank interleave gives
    w2p = util.word2ph_for(t_x, 77)
    assert 1100 <= w2p.size <= 1300
    ids = np.random.default_rng(77).integers(3, cfg.vocab_size, size=w2p.size).astype(np.int64)
    x, tone, lang, _, style = ov.synthetic_inputs(hp, t_x, seed=77)
    x, tone, lang, style = x[0].numpy(), tone[0].numpy(), lang[0].numpy(), style[0].numpy()
    mask = np.ones_like(ids)
    feats = bert.predict(ids, mask)
    synth.seed(9)
    a = synth.synthesize(util.expand_features(feats, w2p), x, [0], tone, lang, style, 0.2, 1.0, 0.677, 0.8).reshape(-1)
    synth.seed(9)
    b = synth.synthesize_from_tokens(bert, ids, mask, w2p, x, 0, tone, lang, style, 0.2, 1.0, 0.677, 0.8)
    assert a.size > 0 and np.array_equal(a, b)
    # the holder: token path against host features, each on a fresh holder (same generator state)
    sv = np.random.default_rng(3).standard_normal((2, 256)).astype(np.float32) * 0.1
    wavs = []
    for tokens in (False, True):
        h = S.TTSModelHolder(bert_onnx, b"")
        h.load("m", assets.style_json(sv), onnx)
        if tokens:
            wavs.append(h.easy_synthesize_tokens("m", [dict(token_ids=ids, word2ph=w2p, phones=x, tones=tone, lang_ids=lang)], 1, 0))
        else:
            f = h.bert_features(ids, mask, w2p)
            assert f.shape == (128, t_x)
            wavs.append(h.easy_synthesize("m", [dict(bert=f, phones=x, tones=tone, lang_ids=lang)], 1, 0))
        h.close()
    assert len(wavs[0]) > 1000 and wavs[0] == wavs[1]
