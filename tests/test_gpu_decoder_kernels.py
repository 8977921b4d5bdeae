"""Layer-level tests of the tensor-core HiFi-GAN decoder (umma_conv.cu, umma_decoder.cu) against float64 references,
through the hooks of libsbv2_b200_debug.so (csrc/debug_kernels.cu); the GPU tests run with -m gpu on a B200.

Every reference is float64 (numpy) evaluated on exactly the operands the kernel reads: fp16-rounded inputs and weights
(np.float16 rounds to nearest even, like __float2half_rn), fp32 biases, each utterance zero-padded at its own
boundaries.  Ragged batches include lengths 1, 2, 3 and lengths at the layer's tile edges: a work item covers 128 * mt
rows (input rows of an upsampling layer), mt from MT below, and the batches hold 128 * mt +- 1 and 256 * mt +- 1.

Bars (per element; "terms" are all addends of that output before the epilogue's division and activation: the products
w * x, the bias, the recovered residuals and the previous accumulate value):

* fp16 outputs:  |got - ref| <= ulp16(ref) + KAPPA * sum|term|,  ulp16(v) = 2^(floor(log2|v|) - 10), at least 2^-24.
  The kernel forms the value in fp32 and rounds it once to fp16: half an ulp of the stored value, which is at most one
  ulp16(ref) when the fp32 value crosses a binade.  The fp32 part is the accumulation error, below.
* KAPPA = 2^-14.  Products of fp16 operands are exact in fp32.  Every later step adds one rounding of at most one fp32
  ulp (2^-23, allowing the tensor core's truncating alignment) relative to the running partial sum, which is bounded
  by sum|term|.  The longest chain in the decoder is a 256-channel, 11-tap conv.  That is 176 MMA steps of K = 16,
  each with its in-MMA sum and the accumulator add, plus at most four epilogue adds and a division: fewer than 512
  roundings of 2^-23, so 512 * 2^-23 = 2^-14.  conv_post's chain is C * k sequential fmaf of 2^-24 each, at most
  64 * 11 = 704 < 1024 here: the same 2^-14.  One KAPPA for every layer.
* fp32 accumulate buffer (UACC_SET / UACC_ADD): |got - ref| <= KAPPA * sum|term|.  The reference adds the previous
  accumulate value the kernel read, so errors do not compound along the chain.
* fused ResBlock pair: the fp64 reference rounds the intermediate t1 to fp16 as the kernel does, but the kernel's fp32
  t1 may round to the neighbouring fp16 value.  The bar adds sum_j,c |w2| * (ulp16(t1) + KAPPA * sum|term of t1|).
* conv_post: |got - tanh(ref)| <= KAPPA * sum|w * x| + 2 ulp32(tanh(ref)).  tanh is 1-Lipschitz and tanhf is within
  2 ulp (CUDA C Programming Guide, mathematical functions).
* whole decoders: the waveform within WAVE_TOL = 1e-3 of the oracle's float64 decoder, as the parity tests require, and
  the CUDA-core fp32 decoder within 2e-5 of it.

Where a batch must equal its utterances run alone, or two kernels must agree, the comparison is bit for bit.  No layer
may write a planar row outside its utterances: every conv reads its halo from those rows and relies on them being zero.

test_bars_catch_mutants (CPU) checks that these bars are not vacuous: on the same inputs, each of a set of plausible
kernel mistakes moves at least one element beyond its bar.
"""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import util
from util import ov

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

pf = C.POINTER(C.c_float)
pi = C.POINTER(C.c_int)
pll = C.POINTER(C.c_longlong)
HOOKS = {
    "sbv2_debug_umma_layer": [pf, pf, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, pf, pi, C.c_int, pf, C.c_int,
                              pf, pf, C.c_float, C.c_int, pf, C.c_float, C.c_int, pf, pll, pi],
    "sbv2_debug_dec_post": [pf, pi, pll, C.c_int, pf, C.c_int, C.c_int, C.c_int, pf, C.c_longlong],
}
ACT_LRELU, ACT_LRELU01 = 2, 4  # kernels.h Act
SLOPE = {ACT_LRELU: 0.1, ACT_LRELU01: 0.01}
UACC_NONE, UACC_SET, UACC_ADD, UACC_FINAL = 0, 1, 2, 3
KAPPA = 2.0 ** -14
WAVE_TOL = 1e-3
MT_PREF = 16  # as umma_decoder_create asks for every layer
WAVE_SENTINEL = np.uint32(0x7FC0BEEF)  # an fp32 NaN payload no kernel writes

# 128-row tiles per work item that make_layer picks at MT_PREF (the test checks the hook reports the same)
MT_CONV = {(256, 256): 1, (256, 128): 2, (128, 256): 2, (64, 256): 4, (32, 256): 8, (16, 256): 16}  # (C, nb_max)
# upsampling layers (cin, cout, k, u): the five JP-Extra stages, one k = 2u and one k = u case
UP_CASES = [(512, 256, 16, 8, 1), (256, 128, 16, 8, 2), (128, 64, 8, 2, 2), (64, 32, 2, 2, 4), (32, 16, 2, 2, 8),
            (64, 32, 4, 2, 4), (32, 16, 4, 4, 8)]  # last: mt
RES_KD = [(3, 1), (7, 3), (11, 5)]
CONV_SHAPES = [(c, k, d, nb) for c in (256, 128, 64, 32, 16) for k, d in RES_KD for nb in ((256, 128) if c == 256 else (256,))]
CONV_MODES = ["res", "mrf", "chain2", "chain4"]
POST_CASES = [(16, 7, 0), (16, 7, 1), (32, 7, 1), (64, 11, 1)]  # (C, k, generic kernel)


def f16(a):
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


def lrelu(v, s=0.1):
    return np.where(v >= 0, v, v * s)


def xrec(y):
    """The residual the epilogue recovers from a stored post-lrelu(0.1) value: exact for fp16 y."""
    y = np.asarray(y, np.float64)
    return np.where(y >= 0, y, 10.0 * y)


def ulp16(v):
    a = np.abs(np.asarray(v, np.float64))
    e = np.floor(np.log2(np.where(a > 0, a, 1.0)))
    return np.maximum(np.where(a > 0, np.exp2(e - 10), 0.0), 2.0 ** -24)


def ulp32(v):
    a = np.abs(np.asarray(v, np.float64))
    e = np.floor(np.log2(np.where(a > 0, a, 1.0)))
    return np.maximum(np.where(a > 0, np.exp2(e - 23), 0.0), 2.0 ** -149)


def edge_lens(mt):
    t = 128 * mt
    return np.asarray([1, 2, 3, t - 1, t, t + 1, 2 * t - 1, 2 * t, 2 * t + 1], np.int32)


def starts(lens, mul=1):
    return np.concatenate([[0], np.cumsum(np.asarray(lens, np.int64) * mul)])


# ---------------------------------------------------------------------------------------------------------------------
# float64 references
# ---------------------------------------------------------------------------------------------------------------------

def taps_ref(x, w, offs, lens):
    """out[t] = sum_j w[:, :, j] @ x[t + offs[j]] per utterance, zero outside it.  x [rows, cin], w [cout, cin, k].
    -> (out, sum of |w * x|), float64 [rows, cout]"""
    x = np.asarray(x, np.float64)
    w = np.asarray(w, np.float64)
    H = max(abs(o) for o in offs)
    out = np.zeros((x.shape[0], w.shape[0]))
    mag = np.zeros_like(out)
    for o, T in zip(starts(lens)[:-1], lens):
        xp = np.zeros((T + 2 * H, x.shape[1]))
        xp[H:H + T] = x[o:o + T]
        for j, s in enumerate(offs):
            seg = xp[H + s:H + s + T]
            out[o:o + T] += seg @ w[:, :, j].T
            mag[o:o + T] += np.abs(seg) @ np.abs(w[:, :, j]).T
    return out, mag


def conv_offs(k, dil):
    return [(j - (k - 1) // 2) * dil for j in range(k)]


def convT_ref(x, w, u, lens, pad=None):
    """ConvTranspose1d(stride u, padding pad = (k - u) / 2) per utterance, w [cin, cout, k]: T * u output rows.
    -> (out, sum of |w * x|) float64"""
    x = np.asarray(x, np.float64)
    w = np.asarray(w, np.float64)
    k = w.shape[2]
    pad = (k - u) // 2 if pad is None else pad
    outs, mags = [], []
    for o, T in zip(starts(lens)[:-1], lens):
        full = np.zeros(((T - 1) * u + k + 2, w.shape[1]))
        fm = np.zeros_like(full)
        xu = x[o:o + T]
        for j in range(k):
            full[j:j + (T - 1) * u + 1:u] += xu @ w[:, :, j]
            fm[j:j + (T - 1) * u + 1:u] += np.abs(xu) @ np.abs(w[:, :, j])
        outs.append(full[pad:pad + T * u])
        mags.append(fm[pad:pad + T * u])
    return np.concatenate(outs), np.concatenate(mags)


def excess(got, ref, bar):
    """largest (|got - ref| - bar) and its element; NaN in got counts as unbounded"""
    d = np.abs(np.asarray(got, np.float64) - ref) - bar
    d = np.where(np.isnan(d), np.inf, d)
    i = np.unravel_index(np.argmax(d), d.shape)
    return float(d[i]), i


def assert_within(got, ref, bar, what):
    ex, i = excess(got, ref, bar)
    rel = np.abs(np.asarray(got, np.float64) - ref) / np.maximum(bar, 1e-300)
    print(f"{what}: max |err| / bar = {float(np.nanmax(rel)):.3f}")
    assert ex <= 0, f"{what}: element {i}: got {float(got[i])!r}, ref {float(ref[i])!r}, bar {float(bar[i]):.3e}"


# ---------------------------------------------------------------------------------------------------------------------
# inputs (shared by the GPU tests and the CPU mutant test)
# ---------------------------------------------------------------------------------------------------------------------

def up_inputs(case):
    cin, cout, k, u, mt = case
    g = np.random.default_rng([7, cin, k, u])
    lens = edge_lens(mt)
    x = f16(lrelu(g.standard_normal((int(lens.sum()), cin))))
    w = f16(g.standard_normal((cin, cout, k)) / np.sqrt(cin * k / u))
    b = (g.standard_normal(cout) * 0.1).astype(np.float32)
    return dict(x=x, w=w, b=b, lens=lens, u=u, mt=mt)


def up_reference(inp, pad=None, w=None):
    v, mag = convT_ref(inp["x"], inp["w"] if w is None else w, inp["u"], inp["lens"], pad)
    b = inp["b"].astype(np.float64)
    return lrelu(v + b), mag + np.abs(b)


def conv_inputs(c, k, dil, nb, step=0, cin=None):
    """one ResBlock conv2-like layer: input = residual (stored post-lrelu values), two more ResBlock outputs for the MRF,
    a garbage accumulate buffer"""
    cin = cin or c
    g = np.random.default_rng([11, c, cin, k, dil, nb, step])
    lens = edge_lens(MT_CONV[(c, nb)] if cin == c else 1)
    rows = int(lens.sum())
    return dict(x=f16(lrelu(g.standard_normal((rows, cin)))), w=f16(g.standard_normal((c, cin, k)) / np.sqrt(cin * k)),
                b=(g.standard_normal(c) * 0.1).astype(np.float32), r2=f16(lrelu(g.standard_normal((rows, c)))),
                r3=f16(lrelu(g.standard_normal((rows, c)))), garbage=(g.standard_normal((rows, c)) * 100).astype(np.float32),
                lens=lens, k=k, dil=dil)


def conv_value(inp, offs=None, rec=xrec):
    """conv + bias + recovered residual (the layer's input) -> (value, sum|term|) before any division / activation"""
    v, mag = taps_ref(inp["x"], inp["w"], offs or conv_offs(inp["k"], inp["dil"]), inp["lens"])
    b = inp["b"].astype(np.float64)
    xr = rec(inp["x"])
    return v + b + xr, mag + np.abs(b) + np.abs(xr)


def mrf_reference(inp, act, divide_first=False, offs=None, rec=xrec):
    v, mag = conv_value(inp, offs, rec)
    r = rec(inp["r2"]) + rec(inp["r3"])
    f = (r / 3.0 + v) if divide_first else (r + v) / 3.0
    return lrelu(f, SLOPE[act]), mag + np.abs(rec(inp["r2"])) + np.abs(rec(inp["r3"]))


def post_inputs(c, k):
    g = np.random.default_rng([13, c, k])
    lens = np.asarray([1, 2, 3, 255, 256, 257, 511, 512, 513], np.int32)  # 256-sample blocks
    x = f16(lrelu(g.standard_normal((int(lens.sum()), c)), 0.01))
    w = (g.standard_normal((c, k)) / np.sqrt(c * k)).astype(np.float32)
    wstart = np.zeros(len(lens), np.int64)
    pos = 5
    for b, T in enumerate(lens):  # 5 + b free samples before each utterance
        wstart[b] = pos
        pos += int(T) + 6 + b
    return dict(x=x, w=w, lens=lens, wstart=wstart, wave_len=pos + 300, k=k)


def post_reference(inp, pad=None):
    k = inp["k"]
    pad = (k - 1) // 2 if pad is None else pad
    v, mag = taps_ref(inp["x"], inp["w"][None], [j - pad for j in range(k)], inp["lens"])
    return v[:, 0], mag[:, 0]


# ---------------------------------------------------------------------------------------------------------------------
# hooks
# ---------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def D():
    """Builds first (a no-op when up to date): the session's lib_built fixture builds only when the product library is
    missing, so an older debug library without these hooks would go unnoticed."""
    spec = importlib.util.spec_from_file_location("sbv2_b200_build", os.path.join(ROOT, "sbv2-api_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()
    import sbv2_b200 as S
    if S.device_count() < 1:
        pytest.fail("GPU tests selected but no B200 is visible: " + S.lib.sbv2_last_error().decode())
    lib = S.debug_lib()
    missing = [h for h in HOOKS if not hasattr(lib, h)]
    if missing:
        pytest.fail(f"libsbv2_b200_debug.so does not export {missing}: rebuild it with `python sbv2-api_b200/build.py`")
    for name, args in HOOKS.items():
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = args
    return lib


def _p(a, t=pf):
    return None if a is None else a.ctypes.data_as(t)


def _f32(a):
    return None if a is None else np.ascontiguousarray(a, np.float32)


def run_layer(D, w, b, x, lens, *, dil=1, up=0, nb_max=256, bias_utt=None, residual=False, r2=None, r3=None, out_div=1.0,
              accum_mode=UACC_NONE, accum=None, accum_div=1.0, act=ACT_LRELU):
    """-> (out [out rows, cout] with NaN where nothing was stored, accum after the launch, pad_rows[2], cfg[3])"""
    w, b, x, bias_utt, r2, r3 = map(_f32, (w, b, x, bias_utt, r2, r3))
    lens = np.ascontiguousarray(lens, np.int32)
    cin = x.shape[1]
    cout = w.shape[1] if up else w.shape[0]
    out = np.full((int(lens.sum()) * (up or 1), cout), np.nan, np.float32)
    acc = None if accum is None else np.array(accum, np.float32, copy=True)
    pad = np.zeros(2, np.int64)
    cfg = np.zeros(3, np.int32)
    st = D.sbv2_debug_umma_layer(_p(w), _p(b), cin, cout, w.shape[2], dil, up, MT_PREF, nb_max, _p(x), _p(lens, pi), len(lens),
                                 _p(bias_utt), int(residual), _p(r2), _p(r3), out_div, accum_mode, _p(acc), accum_div, act, _p(out),
                                 _p(pad, pll), _p(cfg, pi))
    assert st == 0, D.sbv2_last_error().decode()
    return out, acc, pad, cfg


def run_post(D, inp, generic):
    x = _f32(inp["x"])
    w = _f32(inp["w"])
    lens = np.ascontiguousarray(inp["lens"], np.int32)
    ws = np.ascontiguousarray(inp["wstart"], np.int64)
    wave = np.full(inp["wave_len"], WAVE_SENTINEL, np.uint32).view(np.float32)
    st = D.sbv2_debug_dec_post(_p(x), _p(lens, pi), _p(ws, pll), len(lens), _p(w), w.shape[0], w.shape[1], int(generic), _p(wave),
                               len(wave))
    assert st == 0, D.sbv2_last_error().decode()
    return wave


# ---------------------------------------------------------------------------------------------------------------------
# upsampling (polyphase ConvTranspose1d)
# ---------------------------------------------------------------------------------------------------------------------

def test_convT_reference_matches_torch():
    """The numpy ConvTranspose1d reference is torch's conv_transpose1d (float64) per utterance."""
    for case in ((32, 16, 2, 2, 1), (64, 32, 8, 2, 1), (64, 32, 16, 8, 1), (32, 16, 4, 4, 1)):
        cin, cout, k, u, _ = case
        inp = up_inputs(case)
        lens = inp["lens"][:6]
        rows = int(lens.sum())
        got, _ = convT_ref(inp["x"][:rows], inp["w"], u, lens)
        o = starts(lens, u)
        for i, (s, T) in enumerate(zip(starts(lens)[:-1], lens)):
            xt = torch.from_numpy(inp["x"][s:s + T].T.astype(np.float64))[None]
            ref = F.conv_transpose1d(xt, torch.from_numpy(inp["w"].astype(np.float64)), stride=u, padding=(k - u) // 2)[0].T.numpy()
            assert ref.shape == (T * u, cout)
            assert np.abs(got[o[i]:o[i + 1]] - ref).max() <= 1e-12


@gpu
@pytest.mark.parametrize("case", UP_CASES, ids=lambda c: f"{c[0]}to{c[1]}-k{c[2]}-u{c[3]}")
def test_upsample_layer(D, case):
    """make_upsample_layer + launch_umma(out_mul = u), lrelu(0.1) as the decoder launches it: every element within its
    bar, the batch bit-identical to each utterance alone, no row outside the utterances written."""
    inp = up_inputs(case)
    u, lens = inp["u"], inp["lens"]
    out, _, pad, cfg = run_layer(D, inp["w"], inp["b"], inp["x"], lens, up=u, act=ACT_LRELU)
    ref, mag = up_reference(inp)
    assert_within(out, ref, ulp16(ref) + KAPPA * mag, f"upsample {case[:4]}")
    assert pad[0] == 0, f"{pad[0]} planar rows outside the utterances written"
    xs, os_ = starts(lens), starts(lens, u)
    for i, T in enumerate(lens):
        one, _, pad1, _ = run_layer(D, inp["w"], inp["b"], inp["x"][xs[i]:xs[i + 1]], [T], up=u, act=ACT_LRELU)
        assert np.array_equal(one, out[os_[i]:os_[i + 1]]), f"utterance of {T} rows differs alone and in the batch"
        assert pad1[0] == 0
    assert cfg[0] == inp["mt"], f"the layer runs {cfg[0]} tiles per item; MT of this test assumes {inp['mt']}"


# ---------------------------------------------------------------------------------------------------------------------
# ResBlock convs: epilogue variants
# ---------------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("act", [ACT_LRELU, ACT_LRELU01], ids=["lrelu", "lrelu01"])
@pytest.mark.parametrize("mode", CONV_MODES)
@pytest.mark.parametrize("shape", CONV_SHAPES, ids=lambda s: f"C{s[0]}-k{s[1]}d{s[2]}-nb{s[3]}")
def test_resblock_conv_epilogue(D, shape, mode, act):
    """One unfused ResBlock conv with the residual (its input), the MRF mean folded in (residual2/3, out_div 3), or as
    the UACC_SET -> ADD -> FINAL chain of a decoder with 2 or 4 ResBlocks per stage."""
    c, k, dil, nb = shape
    if mode in ("res", "mrf"):
        inp = conv_inputs(c, k, dil, nb)
        if mode == "res":
            out, _, pad, cfg = run_layer(D, inp["w"], inp["b"], inp["x"], inp["lens"], dil=dil, nb_max=nb, residual=True, act=act)
            v, mag = conv_value(inp)
            ref = lrelu(v, SLOPE[act])
        else:
            out, _, pad, cfg = run_layer(D, inp["w"], inp["b"], inp["x"], inp["lens"], dil=dil, nb_max=nb, residual=True, r2=inp["r2"],
                                         r3=inp["r3"], out_div=3.0, act=act)
            ref, mag = mrf_reference(inp, act)
        assert_within(out, ref, ulp16(ref) + KAPPA * mag, f"{mode} {shape}")
        assert pad[0] == 0, f"{pad[0]} planar rows outside the utterances written"
    else:
        n = int(mode[-1])
        prev = conv_inputs(c, k, dil, nb)["garbage"]  # UACC_SET must not read the buffer
        for j in range(n):
            inp = conv_inputs(c, k, dil, nb, step=j)
            am = UACC_SET if j == 0 else (UACC_FINAL if j == n - 1 else UACC_ADD)
            out, acc, pad, cfg = run_layer(D, inp["w"], inp["b"], inp["x"], inp["lens"], dil=dil, nb_max=nb, residual=True, accum_mode=am,
                                           accum=prev, accum_div=float(n), act=act)
            v, mag = conv_value(inp)
            s = 0.0 if am == UACC_SET else prev.astype(np.float64)
            assert pad.tolist() == [0, 0], f"step {j}: planar rows outside the utterances written (out, accum): {pad.tolist()}"
            if am == UACC_FINAL:
                assert np.array_equal(acc.view(np.uint32), prev.view(np.uint32)), "UACC_FINAL wrote the accumulate buffer"
                ref = lrelu((v + s) / n, SLOPE[act])
                assert_within(out, ref, ulp16(ref) + KAPPA * (mag + np.abs(s)), f"{mode} FINAL {shape}")
            else:
                assert np.isnan(out).all(), f"step {j} (UACC_{'SET' if am == UACC_SET else 'ADD'}) stored an fp16 output"
                assert_within(acc, v + s, KAPPA * (mag + np.abs(s)), f"{mode} step {j} accumulate {shape}")
                prev = acc
    assert cfg[0] == MT_CONV[(c, nb)], f"the layer runs {cfg[0]} tiles per item; MT_CONV assumes {MT_CONV[(c, nb)]}"


@gpu
def test_conv_pre_with_per_utterance_bias(D):
    """conv_pre (192 -> 512, k 7) with the speaker conditioning as bias_utt, one different row per utterance."""
    inp = conv_inputs(512, 7, 1, 256, cin=192)
    g = np.random.default_rng(17)
    bu = (g.standard_normal((len(inp["lens"]), 512)) * 0.5).astype(np.float32)
    out, _, pad, cfg = run_layer(D, inp["w"], inp["b"], inp["x"], inp["lens"], bias_utt=bu, act=ACT_LRELU)
    v, mag = taps_ref(inp["x"], inp["w"], conv_offs(7, 1), inp["lens"])
    rows_utt = np.repeat(np.arange(len(inp["lens"])), inp["lens"])
    bias = inp["b"].astype(np.float64)[None, :] + bu.astype(np.float64)[rows_utt]
    ref = lrelu(v + bias)
    assert_within(out, ref, ulp16(ref) + KAPPA * (mag + np.abs(inp["b"])[None, :] + np.abs(bu)[rows_utt]), "conv_pre")
    assert pad[0] == 0
    assert cfg[0] == 1


# ---------------------------------------------------------------------------------------------------------------------
# conv_post
# ---------------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("case", POST_CASES, ids=["16x7-const", "16x7-generic", "32x7", "64x11"])
def test_conv_post(D, case):
    c, k, generic = case
    inp = post_inputs(c, k)
    wave = run_post(D, inp, generic)
    v, mag = post_reference(inp)
    ref = np.tanh(v)
    inside = np.zeros(inp["wave_len"], bool)
    got = np.empty(len(v), np.float32)
    for o, s, T in zip(starts(inp["lens"])[:-1], inp["wstart"], inp["lens"]):
        inside[s:s + T] = True
        got[o:o + T] = wave[s:s + T]
    assert_within(got, ref, KAPPA * mag + 2 * ulp32(ref), f"conv_post {case}")
    stray = np.nonzero(wave.view(np.uint32)[~inside] != WAVE_SENTINEL)[0]
    assert len(stray) == 0, f"{len(stray)} samples outside the utterances written"
    if c == 16 and k == 7 and generic:
        const = run_post(D, inp, False)
        assert np.array_equal(wave.view(np.uint32), const.view(np.uint32)), "generic and 16 x 7 kernels differ"


# ---------------------------------------------------------------------------------------------------------------------
# whole decoders of other architectures
# ---------------------------------------------------------------------------------------------------------------------

ARCHS = {
    "one_resblock": dict(resblock_kernel_sizes=(3,), resblock_dilation_sizes=((1, 3, 5),)),
    "two_resblocks": dict(resblock_kernel_sizes=(3, 7), resblock_dilation_sizes=((1, 3, 5), (1, 3, 5))),
    "two_dilations": dict(resblock_kernel_sizes=(3, 7, 11), resblock_dilation_sizes=((1, 3), (1, 5), (3, 5))),
    "four_stages": dict(upsample_rates=(8, 8, 2, 2), upsample_kernel_sizes=(16, 16, 4, 4)),
}
DEC_LENS = (1, 33, 86, 120)


def _model(S, onnx, env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return S.Model(onnx, bert=False)  # umma_decoder_create reads the switches
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


def _decode_setup(arch_kw, seed):
    hp = ov.tiny_hparams(**arch_kw)
    oracle, onnx = util.synth_assets(hp, seed=seed)
    g = torch.Generator().manual_seed(31)
    zs = [torch.randn(hp.inter_channels, t, generator=g) for t in DEC_LENS]
    spk = oracle.emb_g(torch.tensor([0])).unsqueeze(-1)
    dec = oracle.dec.double()
    with torch.no_grad():
        refs = [dec(z.double()[None], g=spk.double())[0, 0].numpy() for z in zs]
    oracle.dec.float()
    return hp, onnx, [z.numpy() for z in zs], refs


def _wave_err(outs, refs):
    for o, r in zip(outs, refs):
        assert o.shape == r.shape
    return max(float(np.abs(o - r).max()) for o, r in zip(outs, refs))


@gpu
@pytest.mark.parametrize("arch", list(ARCHS))
def test_decoder_architectures(arch):
    import sbv2_b200 as S
    hp, onnx, zs, refs = _decode_setup(ARCHS[arch], seed=5)
    outs = _model(S, onnx, {}).decode_batch(zs)
    err = _wave_err(outs, refs)
    peak = max(float(np.abs(r).max()) for r in refs)
    print(f"{arch}: tensor-core decoder max |err| {err:.3e}, waveform peak {peak:.3f}")
    fp32 = _model(S, onnx, {"SBV2_B200_DECODER": "fp32"}).decode_batch(zs)
    err32 = _wave_err(fp32, refs)
    print(f"{arch}: fp32 decoder max |err| {err32:.3e}")
    assert err32 <= 2e-5, f"the CUDA-core fp32 decoder is {err32:.3e} from the oracle: assets or oracle, not the tensor cores"
    assert err <= WAVE_TOL, f"tensor-core decoder {err:.3e} from the oracle (peak {peak:.3f})"


@gpu
def test_decoder_switches_on_default_architecture():
    """SBV2_B200_PAIR_MAXC=0 (no fused ResBlock pairs) is bit-identical to the default, since a fused pair is bit-identical
    to its two convs; SBV2_B200_DEC_WIDE_NB=128 (N block 128 at C >= 256) stays within WAVE_TOL of the oracle."""
    import sbv2_b200 as S
    hp, onnx, zs, refs = _decode_setup({}, seed=0)
    base = _model(S, onnx, {}).decode_batch(zs)
    nofuse = _model(S, onnx, {"SBV2_B200_PAIR_MAXC": "0"}).decode_batch(zs)
    wide = _model(S, onnx, {"SBV2_B200_DEC_WIDE_NB": "128"}).decode_batch(zs)
    print(f"default: max |err| {_wave_err(base, refs):.3e}; wide_nb 128: {_wave_err(wide, refs):.3e}")
    for i, (a, b) in enumerate(zip(base, nofuse)):
        assert np.array_equal(a, b), f"utterance {i}: unfused ResBlock pairs change the waveform"
    assert _wave_err(base, refs) <= WAVE_TOL
    assert _wave_err(wide, refs) <= WAVE_TOL


# ---------------------------------------------------------------------------------------------------------------------
# the bars are not vacuous (CPU)
# ---------------------------------------------------------------------------------------------------------------------

def _caught(mut, ref, bar):
    return excess(mut, ref, bar)[0] > 0


def test_bars_catch_mutants():
    """Each mutant of a layer, on the inputs the GPU tests use, differs from the correct float64 reference by more than
    the bar at one element at least."""
    for case in UP_CASES[2:]:  # the two widest stages cost seconds of numpy each and add nothing here
        inp = up_inputs(case)
        u, k = inp["u"], case[2]
        ref, mag = up_reference(inp)
        bar = ulp16(ref) + KAPPA * mag
        swapped = ref.reshape(-1, u, ref.shape[1])[:, [1, 0] + list(range(2, u))].reshape(ref.shape)
        assert _caught(swapped, ref, bar), f"{case}: phases 0 and 1 swapped"
        assert _caught(up_reference(inp, w=inp["w"][:, :, ::-1])[0], ref, bar), f"{case}: taps reversed"
        assert _caught(up_reference(inp, pad=(k - u) // 2 + 1)[0], ref, bar), f"{case}: padding off by one"
    for c, kk, dil in ((16, 11, 5), (64, 7, 3), (128, 3, 1)):
        inp = conv_inputs(c, kk, dil, 256)
        offs = conv_offs(kk, dil)
        v, mag = conv_value(inp)
        ref = lrelu(v)
        bar = ulp16(ref) + KAPPA * mag
        shifted = [o + (dil if j == kk - 1 else 0) for j, o in enumerate(offs)]
        assert _caught(lrelu(conv_value(inp, offs=shifted)[0]), ref, bar), f"C{c} k{kk}: a tap shifted by dil"
        assert _caught(lrelu(conv_value(inp, rec=lambda y: np.asarray(y, np.float64))[0]), ref, bar), f"C{c}: residual without x10"
        mref, mmag = mrf_reference(inp, ACT_LRELU)
        assert _caught(mrf_reference(inp, ACT_LRELU, divide_first=True)[0], mref, ulp16(mref) + KAPPA * mmag), \
            f"C{c}: MRF mean divided before the add"
    for c, kk, _ in POST_CASES:
        inp = post_inputs(c, kk)
        v, mag = post_reference(inp)
        ref = np.tanh(v)
        bar = KAPPA * mag + 2 * ulp32(ref)
        assert _caught(np.tanh(post_reference(inp, pad=(kk - 1) // 2 + 1)[0]), ref, bar), f"conv_post {c}x{kk}: padding off by one"
