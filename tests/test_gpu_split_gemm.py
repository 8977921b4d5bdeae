"""Layer-level tests of the split-fp16 tensor-core GEMMs (make_split_conv1d_layer, launch_split_planar, the fp32 row-major
epilogue and its fused split producer, split-K and multicast clusters), the WaveNet gate epilogue and DeBERTa's
LayerNorms against float64 references, through the hooks of libsbv2_b200_debug.so (csrc/debug_kernels.cu); the GPU
tests run with -m gpu on a B200.

Every reference is float64 numpy on the fp32 values the layer receives.  The fp16 split of the operands is the
kernel's job, so the references do not pre-round it; numpy's float32 -> float16 conversion rounds to nearest even, like
__float2half_rn, and gives the bit-exact expected split planes.  u = 2^-24 is the fp32 unit roundoff.

Split layers.  X = s_x x and W = s_w w are the scaled operands: s_x = in_scale = 16, s_w = 2^(13 - e) with
max|w| = m 2^e, m in [0.5, 1) (frexp), so max|W| is in [2^12, 2^13).  Both scalings are exact.

* Representation, per product x w.  fp16 keeps 11 significant bits: h0 = fp16(X) leaves |X - h0| <= 2^-11 |X|, or an
  absolute 2^-25 below 2^-14 where fp16 is subnormal.  The remainder r = X - h0 is exact in fp32, and h1 = fp16(r)
  leaves |X - h0 - h1| <= 2^-22 |X| + 2^-25 (the 2^-25 only when r falls below 2^-14).  The same holds for W.  A two-term
  layer forms h0 w0 + h1 w0 + h0 w1; against X W it errs by the dropped h1 w1 (<= 2^-22 |X||W|) plus both operands'
  representation errors (2^-22 |X||W| each), plus second-order terms: at most REP_REL[2] |X||W| + REP_ABS (|X| + |W|)
  + REP_C, with REP_REL[2] = 2^-20 > 3 * 2^-22, REP_ABS = 2^-24 > 2^-25 (1 + 2^-10) and REP_C = 2^-48.  With three terms
  each operand is represented to 2^-33 |X| + 2^-25 (one more fp16 term of the remainder) and the dropped h1 w2 + h2 w1 +
  h2 w2 are below 2^-32 |X||W|: REP_REL[3] = 2^-30 > 2^-31.  Over one output, in the layer's units (divided by
  s_x s_w):  rep = REP_REL mag + REP_ABS (Sx / s_w + Sw / s_x) + REP_C N / (s_x s_w), where mag = sum |x||w|, Sx the sum
  of |x| the output reads, Sw the sum of its |w| and N = cin k.
* Accumulation.  Products of fp16 values are exact in fp32.  Each K = 16 MMA step adds two roundings of at most 2^-23
  of the running sum's magnitude, bounded by the sum of |terms|: the tensor core's truncating in-MMA sum and the add into
  the fp32 accumulator.  A layer runs steps = n Cin k / 16 of them (n = 3 plane blocks for two terms, 6 for three); under
  split-K each CTA's chain is steps / S long and the rank-ordered sum adds S fp32 adds.  The epilogue's * out_scale is
  exact (a power of two); the bias add is one rounding, the per-utterance bias one more.  With the split terms'
  magnitudes at most (1 + 2^-9) |X||W|:  acc = (2 chain + S + 2) 2^-23 (mag (1 + 2^-9) + |bias|).  The assumption
  that one MMA step's in-MMA sum loses at most 2^-23 of the sum of |terms| (the tensor core aligns its products to the
  largest and truncates) is the one constant here that rests on the hardware, not on IEEE arithmetic; the decoder's
  KAPPA (test_gpu_decoder_kernels.py) rests on the same one.  DeBERTa's f2 (K = 3 * 4096) is a 768-step chain, so every
  layer has its own bar.
* Activation.  ReLU is 1-Lipschitz and exact.  GELU(v) = v Phi(v) has |GELU'| <= GELU_LIP = 1.13; act_apply's erff is
  within 2 ulp (CUDA C Programming Guide, mathematical functions), and its argument v * fp32(1/sqrt 2), the 1 + erf,
  the halving and the product add at most four more roundings relative to v / 2 or v: |fl(GELU(v)) - GELU(v)| <=
  2^-21 |v|.  So the bar after GELU is GELU_LIP (rep + acc) + 2^-21 |v|.
* Aggregate.  The worst-case bar grows with K, a dropped split term only with sqrt(K), so at DeBERTa's depths the
  per-element bar alone cannot tell the split from single-term fp16 operands.  For every launch whose chain is at most
  AGG_MAX_CHAIN = 512 steps the rel-Frobenius error must stay within AGG_FRAC = 1/4 of that of single-term fp16
  operands on the same inputs (numpy).  The accumulation model above, with the truncation's bias all in one direction,
  gives about 512 * 2^-24 = 2^-15 rel-Frobenius at 512 steps; single-term operands give about 2^-12.  The 1/4 is that
  model's 1/8 with a factor of two of margin; it is not taken from a measurement, and every case prints its measured
  ratio.  On a B200 (1000 W) the largest measured ratio was 0.041, for the text encoder's FFN conv_2 (432 steps).

Bit-for-bit: launch_split_planar's planes and the fused split_out planes (ConvCall::split_out, store_split8) equal
numpy's split of the values they stand for; the small and batch packings, tmap on and off, and cluster = 2 against
the plain launch give identical outputs whenever neither launch split K (split-K sums in another order); a batch equals
each utterance run alone with split-K off; split-K gives the same bits twice.  No launch writes a planar row outside
its utterances.  The hook reports what launch_umma chose (ConvCall::report), and the tests pick row counts so that
S = 2, 4 and 8 and two-CTA multicast clusters are each taken.

WaveNet gate (make_gated_conv1d_layer, epilogue_gate).  out = tanh(a) sigmoid(s), a and s the tanh and sigmoid halves
of conv + bias + cond.  Plain fp16 operands (the layer rounds the weights; the tests pass fp16 values): a and s are each
within acc = (2 cin k / 16 + 2) 2^-23 (mag + |bias| + |cond|).  |d out / da| <= 1 and |d out / ds| <= 1/4.  tanhf is
within 2 ulp and __expf(x) within 2 + floor(1.173 |x|) ulp (CUDA C Programming Guide); the sigmoid's 1 + e, the IEEE
division and the product add three roundings: the computed value is within |out| (2^-22 + (2 + floor(1.173 |s|)) 2^-23 +
2^-22) of tanh(a) sigmoid(s) at the kernel's a, s.  The fp16 store adds ulp16(out).

LayerNorm (ln_split_kernel, ln_planar_wide_kernel): two-pass fp32 statistics, each sum a lane-sequential chain of up to
8 * 4 values and a 5-level butterfly, depth D = 37.  v = a + addin is one rounding.  The mean is within
e_mu = (D + 2) u sum|v| / C; each d_i = v_i - mean within eps_i = u |v_i| + e_mu + u |d_i|.  sqrt(sum d^2 / C + eps) moves
by at most ||eps||_2 / sqrt(C) when d does (it is 1/sqrt(C)-Lipschitz in d), and its own roundings (sum, division,
eps add, sqrtf, 1/x) add (D + 1) / 2 + 3 u relatively, so rstd is within rel_r = rstd ||eps||_2 / sqrt(C) +
((D + 1) / 2 + 3) u of rstd*.  Then out_i = d_i rstd g_i + b_i is within |g_i| rstd (eps_i + |d_i| (rel_r + 2 u)) +
u |out_i|, times 1.1 for second-order terms.  The bar is in sum|v| and rstd, never in max|ref|.

test_bars_catch_mutants (CPU) checks that these bars bite: on the same inputs, each of a set of plausible mistakes
moves an element past its bar or fails the aggregate check.
"""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest
from scipy.special import erf

from test_gpu_decoder_kernels import conv_offs, excess, starts, taps_ref, ulp16

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

pf = C.POINTER(C.c_float)
pi = C.POINTER(C.c_int)
pll = C.POINTER(C.c_longlong)
pu16 = C.POINTER(C.c_uint16)
ci, cf = C.c_int, C.c_float
HOOKS = {
    "sbv2_debug_split_layer": [pf, pf, ci, ci, ci, ci, ci, ci, ci, pf, pi, ci, pf, ci, ci, ci, cf, ci, ci, ci, pf, pu16, pu16, pll, pi, pf, pi],
    "sbv2_debug_gated_layer": [pf, pf, ci, ci, ci, ci, ci, pf, pi, ci, pf, pf, pll, pi],
    "sbv2_debug_bert_layernorm": [ci, pf, pf, pf, pf, cf, ci, pi, ci, cf, pf, pu16, pll],
}
ACT_NONE, ACT_RELU, ACT_GELU = 0, 1, 3  # kernels.h Act
VARIANT_SPLITK, VARIANT_CLUSTER, VARIANT_RM = 16, 2, 4  # umma_conv_kernel VARIANT bits

U = 2.0 ** -24
S_X = 16.0
REP_REL = {2: 2.0 ** -20, 3: 2.0 ** -30}
REP_ABS = 2.0 ** -24
REP_C = 2.0 ** -48
GELU_LIP = 1.13
AGG_MAX_CHAIN = 512
AGG_FRAC = 0.25
LN_DEPTH = 37
EPS = 1e-7  # DeBERTa-v3 layer_norm_eps

LENS = np.asarray([1, 2, 3, 127, 128, 129, 255, 256, 257, 300], np.int32)
# (name, cin, cout, k, act): the synthesizer's split layers at HParams defaults (text encoder, FFN, duration predictor)
SYN = [("bert_proj", 1024, 192, 1, ACT_NONE), ("qkv", 192, 576, 1, ACT_NONE), ("o", 192, 192, 1, ACT_NONE), ("proj", 192, 384, 1, ACT_NONE),
       ("ffn1", 192, 768, 3, ACT_RELU), ("ffn2", 768, 192, 3, ACT_NONE), ("dp1", 192, 256, 3, ACT_RELU), ("dp2", 256, 256, 3, ACT_RELU)]
SYN_PACKINGS = [(2, 256), (1, 16)]  # (mt_pref, nb_max) of text_tc and text_tc_small
# DeBERTa-v3-large (1024 hidden) and the tiny test config (128 hidden); f1 feeds the next GEMM as split_out only
DEB = [("qkv", 1024, 3072, 1, ACT_NONE), ("o", 1024, 1024, 1, ACT_NONE), ("f1", 1024, 4096, 1, ACT_GELU), ("f2", 4096, 1024, 1, ACT_NONE),
       ("conv", 1024, 1024, 3, ACT_GELU), ("tiny_qkv", 128, 384, 1, ACT_NONE), ("tiny_o", 128, 128, 1, ACT_NONE),
       ("tiny_f1", 128, 512, 1, ACT_GELU), ("tiny_f2", 512, 128, 1, ACT_NONE)]
DEB_PACKINGS = [256, 64]  # nb_max of the batch and the small-call packing (mt_pref 1)
DEB_SHAPE = {d[0]: d for d in DEB}
# split-K launches of one sentence or a small batch at the small packing: (layer, lens, S that launch_umma must pick).
# B200: 148 SMs; S is the largest of 8, 4, 2 with items * S <= 148 that divides the layer's K chunks.
SPLITK_CASES = [("o", [7], 8), ("conv", [7], 8), ("f2", [7], 8), ("tiny_f2", [7], 8), ("o", [129], 4), ("conv", [129], 4),
                ("o", [3, 5], 4), ("qkv", [7], 2), ("f1", [7], 2)]


def f16(a):
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


def np_split(v, terms):
    """fp32 values -> their fp16 terms (h0, h1[, h2]) as numpy float16, each the RN-even fp16 of the fp32 remainder"""
    v = np.asarray(v, np.float32)
    out = []
    with np.errstate(over="ignore", invalid="ignore"):
        for _ in range(terms):
            h = v.astype(np.float16)
            out.append(h)
            v = v - h.astype(np.float32)  # exact in fp32
    return out


def split_planes(v, terms, scale=S_X):
    """the plane blocks a split layer reads, [h0 | h1 | h0] or [h0 | h1 | h2 | h0 | h1 | h0], as uint16 [rows, n * C]"""
    h = np_split(np.asarray(v, np.float32) * np.float32(scale), terms)
    order = [0, 1, 0] if terms == 2 else [0, 1, 2, 0, 1, 0]
    return np.concatenate([h[i] for i in order], axis=-1).view(np.uint16)


def weight_scale(w):
    """make_split_conv1d_layer's s_w: the largest power of two with max|w| s_w < 2^13 (frexp)"""
    wmax = float(np.abs(np.asarray(w, np.float32)).max())
    if wmax == 0.0:
        return 1.0
    return 2.0 ** (13 - np.frexp(np.float32(wmax))[1])


def act_ref(v, act):
    if act == ACT_RELU:
        return np.maximum(v, 0.0)
    if act == ACT_GELU:
        return 0.5 * v * (1.0 + erf(v / np.sqrt(2.0)))
    return v


def rel_frob(got, ref):
    return float(np.linalg.norm(np.asarray(got, np.float64) - ref) / np.linalg.norm(ref))


# ---------------------------------------------------------------------------------------------------------------------
# split layers: inputs, float64 reference, bars
# ---------------------------------------------------------------------------------------------------------------------

def split_inputs(cin, cout, k, seed, lens=LENS, edge=None, bias_utt=False):
    g = np.random.default_rng([23, cin, cout, k, seed])
    lens = np.asarray(lens, np.int32)
    rows = int(lens.sum())
    x = g.standard_normal((rows, cin)).astype(np.float32)
    w = (g.standard_normal((cout, cin, k)) / np.sqrt(cin * k)).astype(np.float32)
    b = (g.standard_normal(cout) * 0.1).astype(np.float32)
    if edge == "big_x":  # |x| up to the fp16 bound of 16 x, both signs, and the largest fp32 below 4095 that stays finite
        x = (g.uniform(-1, 1, (rows, cin)) * 4094).astype(np.float32)
        x[0, :4] = [4094.0, -4094.0, 4094.97, -4094.97]
    elif edge == "tiny_x":  # 16 x below 2^-3: h1 is subnormal; 16 x below 2^-14: h0 is too
        x = (x * np.where(g.random((rows, cin)) < 0.5, 1e-3, 1e-6)).astype(np.float32)
    elif edge == "wide_w":  # weights from 2^-30 to 1 of max|w| in one layer
        w = (np.sign(w) * 2.0 ** -g.uniform(0, 30, w.shape)).astype(np.float32)
        w.flat[0] = 1.0
    elif edge == "wmax_pow2":  # max|w| exactly a power of two: s_w puts it at 2^12
        w.flat[np.argmax(np.abs(w))] = 0.0
        w = (w / np.abs(w).max() * 0.25).astype(np.float32)
        w.flat[5] = -0.5
    elif edge == "wmax_below":  # max|w| one fp32 ulp below a power of two: s_w puts it just below 2^13
        w = (w / np.abs(w).max() * 0.25).astype(np.float32)
        w.flat[5] = np.nextafter(np.float32(0.5), np.float32(0))
    elif edge == "zero_w":
        w = np.zeros_like(w)
    bu = (g.standard_normal((len(lens), cout)) * 0.5).astype(np.float32) if bias_utt else None
    return dict(x=x, w=w, b=b, bu=bu, lens=lens, k=k)


def split_value(inp, w=None, x=None):
    """float64 conv + bias (+ per-utterance bias) before the activation -> (value, mag = sum|x||w|, |bias| total)"""
    v, mag = taps_ref(inp["x"] if x is None else x, inp["w"] if w is None else w, conv_offs(inp["k"], 1), inp["lens"])
    bias = np.broadcast_to(inp["b"].astype(np.float64), v.shape)
    if inp["bu"] is not None:
        bias = bias + inp["bu"].astype(np.float64)[np.repeat(np.arange(len(inp["lens"])), inp["lens"])]
    return v + bias, mag, np.abs(bias)


def split_bar(inp, terms, S, act, v, mag, babs):
    cin, k = inp["x"].shape[1], inp["k"]
    sw = weight_scale(inp["w"])
    sx_sum, _ = taps_ref(np.abs(inp["x"]), np.ones((1, cin, k)), conv_offs(k, 1), inp["lens"])
    sw_sum = np.abs(inp["w"].astype(np.float64)).sum(axis=(1, 2))[None, :]
    rep = REP_REL[terms] * mag + REP_ABS * (sx_sum / sw + sw_sum / S_X) + REP_C * cin * k / (S_X * sw)
    chain = (3 if terms == 2 else 6) * cin * k // 16 // S
    acc = (2 * chain + S + 2) * 2.0 ** -23 * (mag * (1 + 2.0 ** -9) + babs)
    if act == ACT_GELU:
        return GELU_LIP * (rep + acc) + 2.0 ** -21 * np.abs(v), chain
    return rep + acc, chain


def single_term(inp, act):
    """the same layer on single-term fp16 operands (fp16 of the scaled values), float64"""
    sw = weight_scale(inp["w"])
    xs = f16(inp["x"] * np.float32(S_X)).astype(np.float64) / S_X
    ws = f16(inp["w"] * np.float32(sw)).astype(np.float64) / sw
    return act_ref(split_value(inp, w=ws, x=xs)[0], act)


# ---------------------------------------------------------------------------------------------------------------------
# hooks
# ---------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def D():
    """Builds first (a no-op when up to date), so that an older debug library without these hooks cannot be used."""
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


def run_split(D, inp, terms, act, *, mt_pref=1, nb_max=256, rm=True, split=False, tmap=False, splitk=False, cluster=0, lens=None,
              x=None):
    """-> dict(out [rows, cout] fp32 or None, split [rows, 3 cout] uint16 or None, insplit [rows, n cin] uint16, pad[2],
    cfg = (mt, nb, n_nblk, nkc), scales = (in_scale, out_scale), S, nc, variant, tmap)"""
    w, b, x, bu = map(_f32, (inp["w"], inp["b"], inp["x"] if x is None else x, inp["bu"]))
    lens = np.ascontiguousarray(inp["lens"] if lens is None else lens, np.int32)
    rows, cin = x.shape
    cout, k = w.shape[0], w.shape[2]
    out = np.full((rows, cout), np.nan, np.float32) if rm else None
    spl = np.zeros((rows, 3 * cout), np.uint16) if split else None
    ins = np.zeros((rows, (3 if terms == 2 else 6) * cin), np.uint16)
    pad = np.zeros(2, np.int64)
    cfg = np.zeros(4, np.int32)
    sc = np.zeros(2, np.float32)
    rep = np.zeros(4, np.int32)
    st = D.sbv2_debug_split_layer(_p(w), _p(b), cin, cout, k, 1, terms, mt_pref, nb_max, _p(x), _p(lens, pi), len(lens),
                                  _p(bu if lens.size == len(inp["lens"]) else None), act, int(rm), int(split), S_X, int(tmap),
                                  int(splitk), cluster, _p(out), _p(spl, pu16), _p(ins, pu16), _p(pad, pll), _p(cfg, pi), _p(sc),
                                  _p(rep, pi))
    assert st == 0, D.sbv2_last_error().decode()
    return dict(out=out, split=spl, insplit=ins, pad=pad, cfg=tuple(cfg), scales=tuple(sc), variant=int(rep[0]), nc=int(rep[1]),
                S=int(rep[2]), tmap=int(rep[3]))


def check_split(D, name, inp, terms, act, r, aggregate=True):
    """every element within its bar, the aggregate check where the chain allows it, the input planes and the layer's
    scales exactly as derived, no stray rows; prints the case's figures"""
    sw = weight_scale(inp["w"])
    assert r["scales"] == (np.float32(S_X), np.float32(1.0 / (S_X * sw))), f"{name}: in/out scale {r['scales']}, s_w {sw}"
    assert np.array_equal(r["insplit"], split_planes(inp["x"], terms)), f"{name}: launch_split_planar's planes differ from numpy's split"
    assert r["pad"].tolist() == [0, 0], f"{name}: planar rows outside the utterances written (input, split_out): {r['pad'].tolist()}"
    assert r["S"] >= 1 and r["nc"] >= 1 and (r["S"] > 1) == bool(r["variant"] & VARIANT_SPLITK)
    v, mag, babs = split_value(inp)
    ref = act_ref(v, act)
    bar, chain = split_bar(inp, terms, r["S"], act, v, mag, babs)
    got = r["out"]
    ex, i = excess(got, ref, bar)
    ratio = float(np.nanmax(np.abs(got.astype(np.float64) - ref) / np.maximum(bar, 1e-300)))
    agg = ""
    if aggregate and chain <= AGG_MAX_CHAIN:
        e_k, e_1 = rel_frob(got, ref), rel_frob(single_term(inp, act), ref)
        agg = f", rel-Frobenius {e_k:.2e} = {e_k / e_1:.4f} x single-term fp16 ({e_1:.2e})"
    print(f"{name}: S {r['S']}, nc {r['nc']}, tmap {r['tmap']}, chain {chain}: max |err| / bar = {ratio:.3f}{agg}")
    assert ex <= 0, f"{name}: element {i}: got {float(got[i])!r}, ref {float(ref[i])!r}, bar {float(bar[i]):.3e}"
    if agg:
        assert e_k <= AGG_FRAC * e_1, f"{name}: rel-Frobenius {e_k:.3e} is not within {AGG_FRAC} of single-term fp16's {e_1:.3e}"


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


# ---------------------------------------------------------------------------------------------------------------------
# the synthesizer's split layers
# ---------------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("terms", [2, 3])
@pytest.mark.parametrize("shape", SYN, ids=lambda s: s[0])
def test_synth_split_layer(D, shape, terms):
    """Both packings the model builds, each within its bars, bit-identical to each other; dp1 with a per-utterance bias."""
    name, cin, cout, k, act = shape
    inp = split_inputs(cin, cout, k, 0, bias_utt=name == "dp1")
    outs = []
    for mt_pref, nb_max in SYN_PACKINGS:
        r = run_split(D, inp, terms, act, mt_pref=mt_pref, nb_max=nb_max)
        assert r["S"] == 1 and r["nc"] == 1 and r["variant"] == VARIANT_RM
        check_split(D, f"{name} terms {terms} packing {mt_pref}/{nb_max} (mt {r['cfg'][0]}, nb {r['cfg'][1]})", inp, terms, act, r)
        outs.append(r["out"])
    assert same_bits(outs[0], outs[1]), f"{name}: the small and batch packings differ"


@gpu
@pytest.mark.parametrize("shape", [SYN[4], SYN[6]], ids=lambda s: s[0])
def test_synth_split_batch_equals_alone(D, shape):
    name, cin, cout, k, act = shape
    inp = split_inputs(cin, cout, k, 1, bias_utt=name == "dp1")
    full = run_split(D, inp, 2, act, mt_pref=2)["out"]
    for i, (o, T) in enumerate(zip(starts(inp["lens"])[:-1], inp["lens"])):
        one = dict(inp, x=inp["x"][o:o + T], lens=np.asarray([T], np.int32), bu=None if inp["bu"] is None else inp["bu"][i:i + 1])
        r = run_split(D, one, 2, act, mt_pref=2)
        assert same_bits(r["out"], full[o:o + T]), f"{name}: utterance of {T} rows differs alone and in the batch"


EDGES = ["big_x", "tiny_x", "wide_w", "wmax_pow2", "wmax_below", "zero_w"]


@gpu
@pytest.mark.parametrize("terms", [2, 3])
@pytest.mark.parametrize("edge", EDGES)
def test_split_range_edges(D, edge, terms):
    """The operand ranges the power-of-two scalings are built for, on the text encoder's o (192 -> 192) and FFN conv_2."""
    for name, cin, cout, k, act in (SYN[2], SYN[5]):
        inp = split_inputs(cin, cout, k, 2, edge=edge)
        r = run_split(D, inp, terms, act, mt_pref=2)
        assert np.isfinite(r["out"]).all(), f"{edge} {name}: non-finite output"
        check_split(D, f"{edge} {name} terms {terms}", inp, terms, act, r, aggregate=False)
        if edge == "zero_w":
            assert same_bits(r["out"], np.broadcast_to(inp["b"], r["out"].shape).copy()), f"{name}: an all-zero layer must return its bias"


# ---------------------------------------------------------------------------------------------------------------------
# DeBERTa's split GEMMs
# ---------------------------------------------------------------------------------------------------------------------

def deb_run(D, name, inp, nb_max, **kw):
    """as bert_model.cu launches its GEMMs: tmap, splitk and cluster = 2 unless overridden"""
    act = DEB_SHAPE[name][4]
    opts = dict(tmap=True, splitk=True, cluster=2)
    opts.update(kw)
    return run_split(D, inp, 2, act, nb_max=nb_max, **opts)


@gpu
@pytest.mark.parametrize("shape", DEB, ids=lambda s: s[0])
def test_deberta_split_gemm(D, shape):
    """Ragged batch at both packings, with the model's launch options.  qkv also writes split_out; f1 writes split_out
    only, which must equal the split of the same launch's row-major values.  The packings give the same bits when neither
    split K."""
    name, cin, cout, k, act = shape
    inp = split_inputs(cin, cout, k, 3)
    runs = []
    for nb in DEB_PACKINGS:
        if name in ("f1", "tiny_f1"):
            so = deb_run(D, name, inp, nb, rm=False, split=True)
            r = deb_run(D, name, inp, nb)
            assert (so["S"], so["nc"]) == (r["S"], r["nc"])
            assert np.array_equal(so["split"], split_planes(r["out"], 2)), f"{name}: split_out differs from the split of its values"
        else:
            r = deb_run(D, name, inp, nb, split=name.endswith("qkv"))
            if r["split"] is not None:
                assert np.array_equal(r["split"], split_planes(r["out"], 2)), f"{name}: split_out differs from the split of its values"
        assert r["tmap"] == 1, f"{name}: the launch did not use the tensor map"
        check_split(D, f"deberta {name} nb_max {nb} (nb {r['cfg'][1]}, nkc {r['cfg'][3]})", inp, 2, act, r)
        runs.append(r)
    if runs[0]["S"] == 1 and runs[1]["S"] == 1:
        assert same_bits(runs[0]["out"], runs[1]["out"]), f"{name}: the small and batch packings differ"


@gpu
def test_deberta_tmap_and_cluster_bit_identical(D):
    """o at nb_max 256 on the ragged batch: 17 row tiles, so a two-CTA cluster launch runs one dummy tile.  tmap off, no
    cluster and the model's launch give the same bits."""
    name = "o"
    inp = split_inputs(*DEB_SHAPE[name][1:4], 4)
    base = deb_run(D, name, inp, 256)
    assert base["nc"] == 2 and base["S"] == 1 and base["variant"] & VARIANT_CLUSTER, f"expected a 2-CTA multicast launch: {base}"
    assert sum(-(-int(t) // 128) for t in inp["lens"]) % 2 == 1
    check_split(D, "deberta o, 2-CTA clusters", inp, 2, ACT_NONE, base)
    plain = deb_run(D, name, inp, 256, cluster=0)
    assert plain["nc"] == 1
    assert same_bits(base["out"], plain["out"]), "cluster = 2 differs from the plain launch"
    notmap = deb_run(D, name, inp, 256, tmap=False)
    assert notmap["tmap"] == 0
    assert same_bits(base["out"], notmap["out"]), "tmap on and off differ"


@gpu
def test_deberta_batch_equals_alone(D):
    """ConvLayer (k = 3: the halo reads the neighbouring gap rows) at nb_max 256, split-K off."""
    name = "conv"
    inp = split_inputs(*DEB_SHAPE[name][1:4], 5, lens=[1, 2, 129, 300])
    full = deb_run(D, name, inp, 256, splitk=False)
    assert full["S"] == 1
    for o, T in zip(starts(inp["lens"])[:-1], inp["lens"]):
        one = dict(inp, x=inp["x"][o:o + T], lens=np.asarray([T], np.int32))
        r = deb_run(D, name, one, 256, splitk=False)
        assert same_bits(r["out"], full["out"][o:o + T]), f"utterance of {T} rows differs alone and in the batch"


@gpu
@pytest.mark.parametrize("case", SPLITK_CASES, ids=lambda c: f"{c[0]}-T{'+'.join(map(str, c[1]))}-S{c[2]}")
def test_deberta_split_k(D, case):
    """One sentence or a small batch at the small packing takes split-K with the expected S; within the bars (the
    per-CTA chain is short enough for the aggregate check on every layer), and the same bits twice."""
    name, lens, S = case
    _, cin, cout, k, act = DEB_SHAPE[name]
    inp = split_inputs(cin, cout, k, 6, lens=lens)
    r = deb_run(D, name, inp, 64)
    assert r["S"] == S and r["nc"] == S and r["variant"] & VARIANT_SPLITK, f"{name} {lens}: launch_umma chose {r}, expected S = {S}"
    check_split(D, f"split-K {name} T {lens}", inp, 2, act, r)
    again = deb_run(D, name, inp, 64)
    assert same_bits(r["out"], again["out"]), f"{name}: split-K is not deterministic"
    off = deb_run(D, name, inp, 64, splitk=False)
    assert off["S"] == 1
    check_split(D, f"no split-K {name} T {lens}", inp, 2, act, off)


# ---------------------------------------------------------------------------------------------------------------------
# WaveNet gate
# ---------------------------------------------------------------------------------------------------------------------

GATE_H, GATE_K = 192, 5


def gate_perm(H):
    """make_gated_conv1d_layer's channel permutation: packed channel i = original perm[i]"""
    hb = next(v for v in range(min(H, 128) // 16 * 16, 15, -16) if H % v == 0)
    perm = []
    for j in range(H // hb):
        perm += list(range(j * hb, (j + 1) * hb)) + list(range(H + j * hb, H + (j + 1) * hb))
    return np.asarray(perm)


def gate_inputs():
    H, k = GATE_H, GATE_K
    g = np.random.default_rng(29)
    lens = LENS
    x = f16(g.standard_normal((int(lens.sum()), H)))
    w = f16(g.standard_normal((2 * H, H, k)) / np.sqrt(H * k))
    b = (g.standard_normal(2 * H) * 0.1).astype(np.float32)
    cond = (g.standard_normal((len(lens), 2 * H)) * 2).astype(np.float32)
    cond[1::2, ::7] *= 12.0  # pre-activations at +-20 and beyond: tanh and the sigmoid saturate
    cond[2, 3], cond[2, H + 3], cond[3, 5], cond[3, H + 5] = 40.0, -40.0, -95.0, 95.0
    return dict(x=x, w=w, b=b, cond=cond, lens=lens)


def gate_reference(inp, cond=None, swap=False):
    H = GATE_H
    v, mag = taps_ref(inp["x"], inp["w"], conv_offs(GATE_K, 1), inp["lens"])
    c = (inp["cond"] if cond is None else cond).astype(np.float64)[np.repeat(np.arange(len(inp["lens"])), inp["lens"])]
    pre = v + inp["b"].astype(np.float64) + c
    a, s = pre[:, :H], pre[:, H:]
    if swap:
        a, s = s, a
    out = np.tanh(a) / (1.0 + np.exp(-s))
    absb = np.abs(inp["b"]).astype(np.float64) + np.abs(c)
    acc = (2 * H * GATE_K // 16 + 2) * 2.0 ** -23 * (mag + absb)
    fn = np.abs(out) * (2.0 ** -22 + (2 + np.floor(1.173 * np.abs(s) + 1e-6)) * 2.0 ** -23 + 2.0 ** -22)
    return out, ulp16(out) + acc[:, :H] + acc[:, H:] / 4 + fn


@gpu
def test_wavenet_gate(D):
    """Ragged batch, a different conditioning vector per utterance and channel, saturated pre-activations.  The hook
    applies the layer's perm to the conditioning as the model does; a perm on one side only fails the bar."""
    inp = gate_inputs()
    H = GATE_H
    lens = np.ascontiguousarray(inp["lens"], np.int32)
    out = np.full((int(lens.sum()), H), np.nan, np.float32)
    pad = np.zeros(1, np.int64)
    cfg = np.zeros(4, np.int32)
    st = D.sbv2_debug_gated_layer(_p(_f32(inp["w"])), _p(_f32(inp["b"])), H, H, GATE_K, 1, 2, _p(_f32(inp["x"])), _p(lens, pi), len(lens),
                                  _p(_f32(inp["cond"])), _p(out), _p(pad, pll), _p(cfg, pi))
    assert st == 0, D.sbv2_last_error().decode()
    ref, bar = gate_reference(inp)
    ex, i = excess(out, ref, bar)
    print(f"gate H {H} k {GATE_K} (gate_half {cfg[0]}, nb {cfg[1]}, mt {cfg[3]}): max |err| / bar = "
          f"{float(np.nanmax(np.abs(out - ref) / bar)):.3f}")
    assert cfg[0] * 2 == cfg[1] and np.array_equal(gate_perm(H)[:cfg[1]] % H, np.tile(np.arange(cfg[0]), 2))
    assert ex <= 0, f"gate: element {i}: got {float(out[i])!r}, ref {float(ref[i])!r}, bar {float(bar[i]):.3e}"
    assert pad[0] == 0, f"{pad[0]} planar rows outside the utterances written"


# ---------------------------------------------------------------------------------------------------------------------
# DeBERTa's LayerNorms
# ---------------------------------------------------------------------------------------------------------------------

LN_C = [128, 200, 256, 520, 768, 1024]
LN_LENS = np.asarray([1, 2, 3, 7, 8, 9, 31, 33], np.int32)


def ln_inputs(C, with_addin):
    g = np.random.default_rng([31, C, with_addin])
    rows = int(LN_LENS.sum())
    a = g.standard_normal((rows, C)).astype(np.float32)
    a[1] = 1000.0 + 0.1 * a[1]  # large common offset, mean >> spread
    a[2] = np.float32(3.3)  # constant row
    a[3] = 0.5 + 1e-4 * a[3]  # spread below sqrt(eps)
    a[4] *= 30.0
    addin = (g.standard_normal((rows, C)) * 0.5).astype(np.float32) if with_addin else None
    if with_addin:
        addin[1:4] = 0.0  # keep the special rows special
    gamma = (1.0 + 0.2 * g.standard_normal(C)).astype(np.float32)
    beta = (0.1 * g.standard_normal(C)).astype(np.float32)
    return dict(a=a, addin=addin, gamma=gamma, beta=beta, C=C)


def ln_reference(inp, ddof=0, eps_outside=False):
    v = inp["a"].astype(np.float64)
    if inp["addin"] is not None:
        v = v + inp["addin"]
    C = inp["C"]
    mu = v.mean(axis=1, keepdims=True)
    d = v - mu
    var = (d * d).sum(axis=1, keepdims=True) / (C - ddof)
    rstd = 1.0 / (np.sqrt(var) + EPS) if eps_outside else 1.0 / np.sqrt(var + EPS)
    g, b = inp["gamma"].astype(np.float64), inp["beta"].astype(np.float64)
    out = d * rstd * g + b
    e_mu = (LN_DEPTH + 2) * U * np.abs(v).sum(axis=1, keepdims=True) / C
    eps_i = U * np.abs(v) + e_mu + U * np.abs(d)
    rel_r = rstd * np.sqrt((eps_i * eps_i).sum(axis=1, keepdims=True)) / np.sqrt(C) + ((LN_DEPTH + 1) / 2 + 3) * U
    bar = 1.1 * (np.abs(g) * rstd * (eps_i + np.abs(d) * (rel_r + 2 * U)) + U * np.abs(out))
    return out, bar


@gpu
@pytest.mark.parametrize("with_addin", [False, True], ids=["a", "a+addin"])
@pytest.mark.parametrize("mode", [0, 1], ids=["ln_split", "ln_planar_wide"])
@pytest.mark.parametrize("C", LN_C)
def test_bert_layernorm(D, C, mode, with_addin):
    inp = ln_inputs(C, with_addin)
    rows = inp["a"].shape[0]
    nbuf = 3 if mode == 0 else 2
    out = np.zeros((rows, C), np.float32)
    planes = np.zeros((rows, nbuf * C), np.uint16)
    pad = np.zeros(1, np.int64)
    st = D.sbv2_debug_bert_layernorm(mode, _p(_f32(inp["a"])), _p(_f32(inp["addin"])), _p(inp["gamma"]), _p(inp["beta"]), EPS, C,
                                     _p(LN_LENS, pi), len(LN_LENS), S_X, _p(out), _p(planes, pu16), _p(pad, pll))
    assert st == 0, D.sbv2_last_error().decode()
    ref, bar = ln_reference(inp)
    ex, i = excess(out, ref, bar)
    print(f"LayerNorm {'ln_split' if mode == 0 else 'ln_planar_wide'} C {C} addin {with_addin}: max |err| / bar = "
          f"{float(np.nanmax(np.abs(out - ref) / bar)):.3f}")
    assert ex <= 0, f"element {i}: got {float(out[i])!r}, ref {float(ref[i])!r}, bar {float(bar[i]):.3e}"
    assert pad[0] == 0, f"{pad[0]} planar rows outside the utterances written"
    if mode == 0:
        assert np.array_equal(planes, split_planes(out, 2)), "ln_split's planes differ from the split of its own output"
    else:
        hp = out.astype(np.float16).view(np.uint16)
        assert np.array_equal(planes[:, :C], hp) and np.array_equal(planes[:, C:], hp), "hp / hp2 differ from fp16(h)"


# ---------------------------------------------------------------------------------------------------------------------
# the bars bite (CPU)
# ---------------------------------------------------------------------------------------------------------------------

def _caught(mut, ref, bar, single=None, chain=None):
    if excess(mut, ref, bar)[0] > 0:
        return True
    return single is not None and chain <= AGG_MAX_CHAIN and rel_frob(mut, ref) > AGG_FRAC * rel_frob(single, ref)


def _split_term_value(inp, drop):
    """float64 output of the two-term product sum with one cross term dropped ("h1w0" or "h0w1")"""
    sw = weight_scale(inp["w"])
    h = [t.astype(np.float64) / S_X for t in np_split(inp["x"] * np.float32(S_X), 2)]
    wt = [t.astype(np.float64) / sw for t in np_split(inp["w"] * np.float32(sw), 2)]
    v = split_value(inp, w=wt[0], x=h[0])[0]
    if drop != "h1w0":
        v += split_value(dict(inp, b=0 * inp["b"], bu=None), w=wt[0], x=h[1])[0]
    if drop != "h0w1":
        v += split_value(dict(inp, b=0 * inp["b"], bu=None), w=wt[1], x=h[0])[0]
    return v


def test_bars_catch_mutants():
    """Each mutant, on the inputs the GPU tests use, moves an element past its bar or fails the aggregate check."""
    # split layers: the tiny config's f1 (GELU, 24 steps) and the text encoder's FFN conv_2 (k = 3, 432 steps)
    for name, cin, cout, k, act in (DEB_SHAPE["tiny_f1"], SYN[5]):
        inp = split_inputs(cin, cout, k, 3)
        v, mag, babs = split_value(inp)
        ref = act_ref(v, act)
        bar, chain = split_bar(inp, 2, 1, act, v, mag, babs)
        single = single_term(inp, act)
        assert not _caught(ref, ref, bar, single, chain)
        for drop in ("h1w0", "h0w1"):
            assert _caught(act_ref(_split_term_value(inp, drop), act), ref, bar, single, chain), f"{name}: {drop} dropped"
        assert _caught(act_ref(2 * (v - inp["b"]) + inp["b"], act), ref, bar, single, chain), f"{name}: out_scale x2"
        sw = weight_scale(inp["w"])
        assert _caught(act_ref(v - inp["b"] + inp["b"] / (S_X * sw), act), ref, bar, single, chain), f"{name}: bias before the scale-back"
        if act == ACT_GELU:
            tanh_gelu = 0.5 * v * (1 + np.tanh(np.sqrt(2 / np.pi) * (v + 0.044715 * v ** 3)))
            assert _caught(tanh_gelu, ref, bar, single, chain), f"{name}: tanh-approximate GELU"
    # split-K: one rank's K chunks dropped or doubled.  Rank r of S sums the 64-channel chunks [r nkc / S, (r + 1) nkc / S)
    # of the stacked operand [h0 | h1 | h0] against [w0 | w0 | w1].
    for name, lens, S in SPLITK_CASES[:4]:
        _, cin, cout, k, act = DEB_SHAPE[name]
        inp = split_inputs(cin, cout, k, 6, lens=lens)
        v, mag, babs = split_value(inp)
        ref = act_ref(v, act)
        bar, chain = split_bar(inp, 2, S, act, v, mag, babs)
        single = single_term(inp, act)
        sw = weight_scale(inp["w"])
        h = np_split(inp["x"] * np.float32(S_X), 2)
        wt = np_split(inp["w"] * np.float32(sw), 2)
        xs = np.concatenate([h[0], h[1], h[0]], axis=1).astype(np.float64) / S_X
        ws = np.concatenate([wt[0], wt[0], wt[1]], axis=1).astype(np.float64) / sw
        nkc = 3 * cin // 64
        lo, hi = nkc * 3 // S * 64, nkc * 4 // S * 64  # rank 3
        part = taps_ref(xs[:, lo:hi], ws[:, lo:hi], conv_offs(k, 1), inp["lens"])[0]
        for sign, what in ((-1, "dropped"), (1, "doubled")):
            assert _caught(act_ref(v + sign * part, act), ref, bar, single, chain), f"{name}: a split-K rank's partial sum {what}"
    # WaveNet gate
    inp = gate_inputs()
    ref, bar = gate_reference(inp)
    assert excess(ref, ref, bar)[0] <= 0
    assert _caught(gate_reference(inp, swap=True)[0], ref, bar), "gate halves swapped"
    perm = gate_perm(GATE_H)
    unperm = np.empty_like(inp["cond"])
    unperm[:, perm] = inp["cond"]  # the kernel adds cond[i] at packed channel i: original channel perm[i] gets cond[i]
    assert _caught(gate_reference(inp, cond=unperm)[0], ref, bar), "perm not applied to the conditioning vector"
    # LayerNorm
    for C in LN_C:
        inp = ln_inputs(C, True)
        ref, bar = ln_reference(inp)
        assert _caught(ln_reference(inp, ddof=1)[0], ref, bar), f"C {C}: variance over C - 1"
        assert _caught(ln_reference(inp, eps_outside=True)[0], ref, bar), f"C {C}: eps outside the square root"
