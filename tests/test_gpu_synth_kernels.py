"""Kernel unit tests of the synthesizer between the text encoder and the decoder, through the hooks of
libsbv2_b200_debug.so (csrc/debug_kernels.cu); the GPU tests run with -m gpu on a B200.

Every reference is oracle/vits.py evaluated in float64 on exactly the inputs the kernel reads (rounded to fp16 where
the kernel reads fp16, relative tables fp16-representable so that both attention kernels and the reference see the
same values).  Each bar follows from the kernel's rounding points and is derived next to its assertion; -s prints the
measured error of every case.

* window attention of the transformer flow: tensor-core kernel (flow_attention_tc.cu) and planar CUDA-core kernel on a
  ragged batch of 21 lengths around the 32-row chunk and 128-key tile edges, each length also alone;
* the text encoder's fp32 attention, both CTA shapes (16 and 64 queries);
* the inverse rational-quadratic spline of the stochastic duration predictor at its edges (tails, bounds, knots,
  saturated softmaxes, both softplus branches);
* durations, their per-utterance scan and the frame -> phoneme expansion, including a total beyond int32;
* the default (transformer) flow of the full model stage by stage against the oracle.
"""
import ctypes as C
import functools
import importlib.util
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import util
from util import ov

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

pf = C.POINTER(C.c_float)
pi = C.POINTER(C.c_int)
pu16 = C.POINTER(C.c_uint16)
HOOKS = {
    "sbv2_debug_flow_attention": [pu16, pi, C.c_int, C.c_int, pf, pf, C.c_int, C.c_uint16, pu16, C.POINTER(C.c_longlong)],
    "sbv2_debug_rel_attention": [pf, pi, C.c_int, C.c_int, pf, pf, pf],
    "sbv2_debug_convflow_spline": [pf, pf, C.c_int, C.c_int, C.c_float, C.c_float],
    "sbv2_debug_durations": [pf, pf, pf, pf, pi, C.c_int, pf, pi, pi, pi, pi],
}
INT_MAX = 2 ** 31 - 1
HD = 96  # head_dim of every attention of the model


def _ptr(a, t):
    return None if a is None else a.ctypes.data_as(t)


@pytest.fixture(scope="module")
def built():
    """conftest.lib_built builds only when the product library is missing, so a debug library older than the hooks used
    here would go unnoticed: build first (a no-op when everything is up to date)."""
    spec = importlib.util.spec_from_file_location("sbv2_b200_build", os.path.join(ROOT, "sbv2-api_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()
    import sbv2_b200
    return mod, sbv2_b200


@pytest.fixture(scope="module")
def D(built):
    _, S = built
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


def _check(lib, status):
    assert status == 0, lib.sbv2_last_error().decode()


def _dynamic_symbols(path):
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    return {line.split()[-1] for line in out.splitlines() if line.strip()}


def test_debug_hooks_are_only_in_the_debug_library(built):
    """The product library exports the ABI of include/sbv2_b200.h: of the sbv2_debug_* names only those the header
    declares (sbv2_debug_fetch); the kernel hooks are in libsbv2_b200_debug.so."""
    mod, _ = built
    header = open(os.path.join(ROOT, "include", "sbv2_b200.h")).read()
    declared = set(re.findall(r"\b(sbv2_debug_\w+)\s*\(", header))
    product = {s for s in _dynamic_symbols(mod.LIB) if s.startswith("sbv2_debug_")}
    assert product == declared, f"product library exports debug symbols {sorted(product - declared)}"
    debug = _dynamic_symbols(mod.DEBUG_LIB)
    assert set(HOOKS) <= debug, f"debug library lacks {sorted(set(HOOKS) - debug)}"


# ---------------------------------------------------------------------------------------------------------------------
# window attention
# ---------------------------------------------------------------------------------------------------------------------

FLOW_LENS = [1, 2, 4, 5, 9, 10, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 700, 1300, 5200]
GAP_FILLS = {"0": 0x0000, "+65504": 0x7BFF, "-65504": 0xFBFF}  # finite: the kernels' precondition on padding rows


def f16(a):
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


def rel_tables(seed):
    g = np.random.default_rng(seed)
    return f16(g.standard_normal((9, HD)) * 0.5), f16(g.standard_normal((9, HD)) * 0.5)


def attention_inputs(lens, heads, regime, seed):
    """q, k, v [rows, heads, 96] for one regime of the softmax:
    normal    N(0,1) logits;
    peak_band each query row aims at one key of its +-4 band (the relative terms carry the result) with a scaled logit of
              about +30, and at one random key with about -30;
    peak_far  the same with the +30 key far from the band;
    equal     q = 0: every logit of a row is 0 (uniform softmax, every key and every masking error counts)."""
    g = np.random.default_rng(seed)
    rows = int(sum(lens))
    k = g.standard_normal((rows, heads, HD))
    v = g.standard_normal((rows, heads, HD))
    if regime == "normal":
        q = g.standard_normal((rows, heads, HD))
    elif regime == "equal":
        q = np.zeros((rows, heads, HD))
    else:
        kn = k / np.linalg.norm(k, axis=-1, keepdims=True)
        q = np.zeros((rows, heads, HD))
        o = 0
        for n in lens:
            i = np.arange(n)
            if regime == "peak_band":
                hit = np.clip(i + g.integers(-4, 5, n), 0, n - 1)
            else:
                hit = (i + n // 2) % n
            miss = g.integers(0, n, n)
            # logit(i, j) = q_i . k_j / sqrt(96): +30 * |k_hit| / sqrt(96) ~ +30 at the hit, ~ -30 at the miss
            q[o:o + n] = 30.0 * (kn[o + hit] - kn[o + miss] * (miss != hit)[:, None, None])
            o += n
    return f16(q), f16(k), f16(v)


def attention_reference(q, k, v, lens, heads, rel_k, rel_v):
    """oracle MultiHeadAttention.attention in float64, utterance by utterance -> [rows, heads*96]"""
    m = ov.MultiHeadAttention(heads * HD, heads * HD, heads, 4).double()
    with torch.no_grad():
        m.emb_rel_k.copy_(torch.from_numpy(rel_k.astype(np.float64))[None])
        m.emb_rel_v.copy_(torch.from_numpy(rel_v.astype(np.float64))[None])
        out = []
        o = 0
        for n in lens:
            cm = [torch.from_numpy(a[o:o + n].reshape(n, heads * HD).T.astype(np.float64))[None] for a in (q, k, v)]
            out.append(m.attention(*cm)[0].T.numpy())
            o += n
    return np.concatenate(out)


@functools.lru_cache(maxsize=None)
def flow_case(heads, regime):
    seed = {"normal": 1, "peak_band": 2, "peak_far": 3, "equal": 4}[regime] * 10 + heads
    q, k, v = attention_inputs(FLOW_LENS, heads, regime, seed)
    rel_k, rel_v = rel_tables(seed)
    rows = q.shape[0]
    qkv = np.concatenate([a.reshape(rows, heads * HD) for a in (q, k, v)], axis=1).astype(np.float16)
    return qkv, rel_k, rel_v, attention_reference(q, k, v, FLOW_LENS, heads, rel_k, rel_v), float(np.abs(v).max())


def run_flow_attention(lib, qkv, lens, heads, rel_k, rel_v, mode, gap):
    lens_a = np.asarray(lens, np.int32)
    qkv = np.ascontiguousarray(qkv)
    out = np.zeros((qkv.shape[0], heads * HD), np.float16)
    pad = C.c_longlong(-1)
    _check(lib, lib.sbv2_debug_flow_attention(_ptr(qkv.view(np.uint16), pu16), _ptr(lens_a, pi), len(lens), heads, _ptr(rel_k, pf),
                                              _ptr(rel_v, pf), mode, gap, _ptr(out.view(np.uint16), pu16), C.byref(pad)))
    return out, pad.value


@gpu
@pytest.mark.parametrize("regime", ["normal", "peak_band", "peak_far", "equal"])
@pytest.mark.parametrize("heads", [2, 1])
def test_flow_window_attention(D, heads, regime):
    qkv, rel_k, rel_v, ref, vmax = flow_case(heads, regime)
    offs = np.concatenate([[0], np.cumsum(FLOW_LENS)])
    for mode, name in ((0, "tensor-core"), (1, "planar CUDA-core")):
        batch = None
        for gname, gap in GAP_FILLS.items():
            out, pad = run_flow_attention(D, qkv, FLOW_LENS, heads, rel_k, rel_v, mode, gap)
            assert pad == 0, f"{name}: {pad} padding rows written"
            assert not np.isnan(out).any(), f"{name}: NaN in the output"
            err = np.abs(out.astype(np.float64) - ref)
            if mode == 0:
                # P goes through fp16 (<= 2^-11 relative per probability, so <= 2^-11 max|v| on the output) and so does the
                # output (another 2^-11 of a value <= max|v|): ~1e-3 max|v|.  A dropped band term or an unmasked key moves
                # the output by O(0.1).
                bar = 2e-3 * vmax
            else:
                bar = 1e-3 * float(np.abs(ref).max())  # fp32 arithmetic, only the output is rounded to fp16 (2^-11)
            worst = int(np.argmax(err.max(axis=1)))
            b = int(np.searchsorted(offs, worst, side="right") - 1)
            print(f"\nflow attention {name} heads={heads} {regime:9s} gap={gname:7s}: max|err| {err.max():.3e} "
                  f"(bar {bar:.3e}; worst at row {worst - offs[b]} of length {FLOW_LENS[b]})", end="")
            assert err.max() <= bar
            if gap == 0:
                batch = out
        for b, n in enumerate(FLOW_LENS):
            single, pad = run_flow_attention(D, qkv[offs[b]:offs[b + 1]], [n], heads, rel_k, rel_v, mode, 0)
            assert pad == 0
            assert np.array_equal(single.view(np.uint16), batch[offs[b]:offs[b + 1]].view(np.uint16)), \
                f"{name}: length {n} alone differs from the same utterance in the batch"


TEXT_CASES = {"one utterance, 16-query CTAs": [1000], "one utterance, 64-query CTAs": [1100],
              "ragged, 16-query CTAs": [1, 5, 33, 64, 129], "ragged, 64-query CTAs": [1, 5, 31, 64, 65, 129, 300, 17]}


@gpu
@pytest.mark.parametrize("case", list(TEXT_CASES))
def test_text_encoder_attention(D, case):
    """launch_rel_attention takes 16-query CTAs when max_len * n <= 1024 and 64-query CTAs otherwise; both against the
    fp64 oracle at the bar of the fp32 path's end-to-end test."""
    lens, heads = TEXT_CASES[case], 2
    g = np.random.default_rng(len(case))
    rows = sum(lens)
    q, k, v = (g.standard_normal((rows, heads, HD)).astype(np.float32) for _ in range(3))
    rel_k, rel_v = rel_tables(7)
    qkv = np.ascontiguousarray(np.concatenate([a.reshape(rows, heads * HD) for a in (q, k, v)], axis=1))
    out = np.zeros((rows, heads * HD), np.float32)
    lens_a = np.asarray(lens, np.int32)
    _check(D, D.sbv2_debug_rel_attention(_ptr(qkv, pf), _ptr(lens_a, pi), len(lens), heads, _ptr(rel_k, pf), _ptr(rel_v, pf), _ptr(out, pf)))
    ref = attention_reference(q, k, v, lens, heads, rel_k, rel_v)
    err = np.abs(out - ref).max()
    bar = 2e-5 * max(1.0, float(np.abs(ref).max()))
    print(f"\ntext attention {case}: max|err| {err:.3e} (bar {bar:.3e})", end="")
    assert err <= bar


# ---------------------------------------------------------------------------------------------------------------------
# inverse rational-quadratic spline (stochastic duration predictor)
# ---------------------------------------------------------------------------------------------------------------------

NB, LD, TB = 10, 29, 5.0
INV_SQRT = np.float32(1.0 / np.sqrt(192.0))


def spline_proj_rows():
    g = np.random.default_rng(5)
    rows, names = [], []

    def add(name, p):
        rows.append(np.asarray(p, np.float32))
        names.append(name)
    add("zeros", np.zeros(LD))
    for s in (1, 10, 100):
        for i in range(2):
            add(f"N(0,1)*{s}#{i}", g.standard_normal(LD) * s)
    for i in (0, 4, 9):  # one saturated width / height logit: every other bin at the minimum size
        p = np.zeros(LD)
        p[i] = 1e4
        add(f"width[{i}]=1e4", p)
        p = np.zeros(LD)
        p[NB + i] = 1e4
        add(f"height[{i}]=1e4", p)
    for dv in (-50.0, 20.0, 20.0001, 25.0):  # softplus: log1p(exp(x)) and the x > 20 branch
        p = g.standard_normal(LD)
        p[2 * NB:] = dv
        add(f"derivatives={dv}", p)
    p = g.standard_normal(LD)
    p[2 * NB:] = np.resize([-50.0, 20.0, 20.0001, 25.0], NB - 1)
    add("derivatives mixed", p)
    return names, np.stack(rows)


def kernel_knots(p):
    """cumheights as convflow_spline_kernel forms them in fp32 (same operations, same order)"""
    f = np.float32
    uh = p[NB:2 * NB].astype(f) * INV_SQRT
    e = np.exp(uh - uh.max()).astype(f)
    sh = f(0)
    for x in e:
        sh = f(sh + x)
    ah, knots = f(0), []
    for x in e:
        ah = f(ah + f(f(1e-3) + f(f(1) - f(1e-3) * f(NB)) * f(x / sh)))
        knots.append(f(f(f(2) * f(TB)) * ah) + f(-TB))
    return np.asarray(knots[:-1], f)  # the last one is replaced by tail_bound


def spline_inputs(p):
    f = np.float32
    up, dn = lambda x: np.nextafter(f(x), f(np.inf)), lambda x: np.nextafter(f(x), f(-np.inf))
    special = np.asarray([TB, -TB, dn(TB), up(TB), up(-TB), dn(-TB), 0.0, np.inf, -np.inf, np.nan], f)
    kn = kernel_knots(p)
    knots = np.concatenate([kn, up(kn), dn(kn)])
    sweep = np.linspace(-TB, TB, 10000, dtype=f)
    return np.concatenate([special, knots, sweep]), len(special) + len(knots)


def spline_reference(x, p):
    """oracle unconstrained_rqs_inverse in float64"""
    t = torch.from_numpy(p.astype(np.float64))
    with torch.no_grad():
        return ov.unconstrained_rqs_inverse(torch.from_numpy(np.asarray(x, np.float64)), t[:, :NB] * float(INV_SQRT),
                                            t[:, NB:2 * NB] * float(INV_SQRT), t[:, 2 * NB:].clone(), TB).numpy()


@gpu
def test_convflow_spline_inverse(D):
    names, prows = spline_proj_rows()
    xs, ps, n_pts = [], [], None
    for p in prows:
        x, n_edge = spline_inputs(p)
        xs.append(x)
        ps.append(np.tile(p, (len(x), 1)))
        n_pts = len(x)
    x = np.concatenate(xs)
    proj = np.ascontiguousarray(np.concatenate(ps))
    g = np.random.default_rng(6)
    z = np.stack([g.standard_normal(len(x)).astype(np.float32), x], axis=1)
    z = np.ascontiguousarray(z)
    z_in = z.copy()
    _check(D, D.sbv2_debug_convflow_spline(_ptr(z, pf), _ptr(proj, pf), LD, len(x), TB, INV_SQRT))
    assert np.array_equal(z[:, 0].view(np.uint32), z_in[:, 0].view(np.uint32)), "column 0 was written"
    y = z[:, 1].astype(np.float64)
    outside = ~((x >= -TB) & (x <= TB))  # also NaN: the oracle passes it through as the kernel does
    assert np.array_equal(z[outside, 1].view(np.uint32), x[outside].view(np.uint32)), "linear tails are not the identity"
    inside = ~outside
    xi = x[inside].astype(np.float64)
    pi_ = proj[inside]
    ref = spline_reference(xi, pi_)
    lo, hi = spline_reference(xi - 1e-5, pi_), spline_reference(xi + 1e-5, pi_)
    yi = y[inside]
    assert np.isfinite(yi).all()
    # Bracket: robust where min-height bins make the inverse steep (a 1e-5 move of x moves the result a lot).  Where the
    # inverse is flat the bracket is narrower than the output's own fp32 error: the width knots are 2 * tail_bound times
    # a sum of 10 fp32 softmax terms (~24 roundings of 2^-24 -> 1.5e-5 at worst, 1e-5 seen in a float32 model of the
    # kernel), so the bracket is widened by Y_TOL in the output.  Dropping the end derivative moves the output by O(1e-2).
    Y_TOL = 2e-5
    below = np.minimum(lo, hi) - Y_TOL - yi
    above = yi - np.maximum(lo, hi) - Y_TOL
    slope = np.abs(hi - lo) / 2e-5
    tame = slope <= 10
    fwd = np.abs(yi - ref)[tame]
    row_of = np.repeat(np.arange(len(names)), n_pts)[inside]
    for r, name in enumerate(names):
        sel = row_of == r
        sel_t = sel[tame]
        print(f"\nspline proj={name:20s}: max fwd err (slope<=10) {fwd[sel_t].max() if sel_t.any() else 0:.2e}, "
              f"outside the x-bracket by {max(below[sel].max(), above[sel].max()) + Y_TOL:.2e}, max slope {slope[sel].max():.1e}",
              end="")
    assert (below <= 0).all() and (above <= 0).all(), "output outside the fp64 inverse of [x - 1e-5, x + 1e-5] (+- 2e-5)"
    # where the inverse is not steep the knot errors (~1e-6 typical) dominate: 2e-5
    assert fwd.max() <= 2e-5
    sweep = y.reshape(len(names), n_pts)[:, n_edge:]
    assert (np.diff(sweep, axis=1) >= 0).all(), "the inverse is not monotone on the sweep"


# ---------------------------------------------------------------------------------------------------------------------
# durations, scan and expansion
# ---------------------------------------------------------------------------------------------------------------------

DUR_LENS = [1, 31, 32, 33, 64, 65, 1000, 1801]


def run_durations(lib, logw_dp, z_sdp, ratio, ls, lens, want_f2p=True):
    rows, n = len(logw_dp), len(lens)
    a = lambda v, t=np.float32: np.ascontiguousarray(v, t)
    logw_dp, ratio, ls, lens_a = a(logw_dp), a(ratio), a(ls), a(lens, np.int32)
    z_sdp = None if z_sdp is None else a(z_sdp)
    w = np.zeros(rows, np.float32)
    dur, cum, ylen = np.zeros(rows, np.int32), np.zeros(rows, np.int32), np.zeros(n, np.int32)
    tot = None
    f2p = None
    _check(lib, lib.sbv2_debug_durations(_ptr(logw_dp, pf), _ptr(z_sdp, pf), _ptr(ratio, pf), _ptr(ls, pf), _ptr(lens_a, pi), n,
                                         _ptr(w, pf), _ptr(dur, pi), _ptr(cum, pi), _ptr(ylen, pi), None))
    if want_f2p:
        tot = int(ylen.astype(np.int64).sum())
        f2p = np.full(tot, -7, np.int32)
        _check(lib, lib.sbv2_debug_durations(_ptr(logw_dp, pf), _ptr(z_sdp, pf), _ptr(ratio, pf), _ptr(ls, pf), _ptr(lens_a, pi), n,
                                             _ptr(w, pf), _ptr(dur, pi), _ptr(cum, pi), _ptr(ylen, pi), _ptr(f2p, pi)))
    return w, dur, cum, ylen, f2p


def check_scan(lens, dur, cum, ylen, f2p):
    offs = np.concatenate([[0], np.cumsum(lens)])
    yo = np.concatenate([[0], np.cumsum(ylen.astype(np.int64))])
    for b in range(len(lens)):
        d = dur[offs[b]:offs[b + 1]].astype(np.int64)
        assert np.array_equal(cum[offs[b]:offs[b + 1]], np.cumsum(d)), f"cum of utterance {b}"
        assert ylen[b] == max(1, int(d.sum()))
        want = np.repeat(np.arange(len(d), dtype=np.int32), d) if d.sum() > 0 else np.asarray([-1], np.int32)
        assert np.array_equal(f2p[yo[b]:yo[b + 1]], want), f"frame2ph of utterance {b}"


@gpu
@pytest.mark.parametrize("with_sdp", [True, False], ids=["sdp", "no_sdp"])
@pytest.mark.parametrize("rot", range(3))
def test_durations_and_expansion(D, with_sdp, rot):
    g = np.random.default_rng(10 * rot + with_sdp)
    rows, n = sum(DUR_LENS), len(DUR_LENS)
    ratios, scales = [0.0, 0.4, 1.0], [0.5, 1.0, 2.3]
    ratio = np.asarray([ratios[(b + rot) % 3] for b in range(n)], np.float32)
    ls = np.asarray([scales[(b // 3 + b + rot) % 3] for b in range(n)], np.float32)
    logw_dp = g.uniform(-1.5, 2.5, rows).astype(np.float32)
    z_sdp = None
    if with_sdp:
        # column 1 is the other SDP channel: huge, so that reading it instead of column 0 cannot go unnoticed
        z_sdp = np.stack([g.uniform(-1.5, 2.5, rows), np.full(rows, 80.0)], axis=1).astype(np.float32)
    w, dur, cum, ylen, f2p = run_durations(D, logw_dp, z_sdp, ratio, ls, DUR_LENS)
    # reference: float32 with the kernel's operation order, expf replaced by a correctly rounded exp
    r = np.repeat(ratio, DUR_LENS)
    s = np.repeat(ls, DUR_LENS)
    one = np.float32(1)
    logw = logw_dp * (one - r)
    if with_sdp:
        logw = (z_sdp[:, 0] * r) + logw
    e_ref = np.exp(logw.astype(np.float64)).astype(np.float32)
    w_ref = e_ref * s
    # expf is within 2 ulp of exp; the product with length_scale is rounded once more: 2 ulp(e) * ls + 1 ulp(w)
    # (2 ulp of w when length_scale is a power of two, up to ~3.3 for 2.3)
    tol = 2 * np.spacing(e_ref).astype(np.float64) * s + np.spacing(np.abs(w_ref))
    dev = np.abs(w.astype(np.float64) - w_ref)
    ulps = dev / np.spacing(np.abs(w_ref))
    assert (dev <= tol).all(), f"w differs from float32(exp(logw)) * length_scale by up to {ulps.max():.1f} ulp"
    assert np.array_equal(dur, np.clip(np.ceil(w), 0, 1e6).astype(np.int32)), "dur != ceil(w)"
    # where w_ref is this close to an integer, ceil may legitimately go either way (w = exp(0) * ls is exact, not a tie)
    near = (np.abs(w_ref - np.round(w_ref)) <= np.maximum(4 * np.spacing(np.abs(w_ref)), tol)) & (w != w_ref)
    print(f"\ndurations rot={rot} sdp={with_sdp}: max {ulps.max():.1f} ulp, {int(near.sum())} near-integer w, T_y {ylen.tolist()}", end="")
    assert near.sum() == 0
    assert np.array_equal(dur, np.ceil(w_ref).astype(np.int32))
    check_scan(DUR_LENS, dur, cum, ylen, f2p)


@gpu
def test_durations_crafted_values(D):
    """w = exp(log k) on both sides of k; a duration at the 1e6 clamp; an utterance whose durations are all zero maps
    its single frame to no phoneme (-1)."""
    k = np.arange(1, 65)
    lens = [64, 1, 5]
    logw_dp = np.concatenate([np.log(k).astype(np.float32), [100.0], np.zeros(5)]).astype(np.float32)
    w, dur, cum, ylen, f2p = run_durations(D, logw_dp, None, np.zeros(3), np.asarray([1.0, 1.0, 0.0]), lens)
    assert ((dur[:64] == k) | (dur[:64] == k + 1)).all()
    assert np.array_equal(dur[:64], np.ceil(w[:64]).astype(np.int32))
    assert dur[64] == 1_000_000 and np.isinf(w[64])
    assert (dur[65:] == 0).all() and ylen[2] == 1
    check_scan(lens, dur, cum, ylen, f2p)
    print(f"\ncrafted durations: {int((dur[:64] != k).sum())} of 64 exp(log k) rounded above k", end="")


@gpu
def test_durations_total_beyond_int32(D):
    """2200 phonemes at the 1e6-frame clamp: 2.2e9 frames.  ylen saturates at INT_MAX, which the host rejects as too
    long, instead of wrapping around to a plausible (or clamped-to-1) T_y."""
    lens = [2200, 7]
    logw_dp = np.concatenate([np.full(2200, 20.0), np.log(np.arange(2, 9))]).astype(np.float32)
    w, dur, cum, ylen, _ = run_durations(D, logw_dp, None, np.zeros(2), np.ones(2), lens, want_f2p=False)
    assert (dur[:2200] == 1_000_000).all()
    assert ylen[0] == INT_MAX, f"T_y of a 2.2e9-frame utterance reported as {ylen[0]}"
    assert ylen[1] == int(dur[2200:].sum()) and np.array_equal(cum[2200:], np.cumsum(dur[2200:]))


# ---------------------------------------------------------------------------------------------------------------------
# the default flow, stage by stage
# ---------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def flow_models(built, D):
    """the full model, and the same with one coupling layer: the flow ping-pongs between the buffer that holds z_p and a
    second one, so after a run debug_fetch("z_p") still holds z_p only when there is a single coupling layer"""
    _, S = built
    out = {}
    for n_flow in (4, 1):
        hp = ov.HParams(n_flow_layer=n_flow)
        oracle, onnx = util.synth_assets(hp, seed=0)
        model = S.Model(onnx, bert=False)
        assert model.describe()["use_transformer_flow"] is True
        out[n_flow] = (hp, oracle, model)
    return out


def _run_stages(hp, oracle, model, t_x, seed):
    u = util.make_utterance(hp, t_x, seed=seed, sdp_ratio=0.4)
    _, inter = util.oracle_run(oracle, u)
    _, dur, _ = model.synthesize_with_noise(u["bert"][0].numpy(), u["x"][0].numpy(), u["sid"], u["tone"][0].numpy(),
                                            u["lang"][0].numpy(), u["style"][0].numpy(), u["sdp_ratio"], u["length_scale"],
                                            u["noise_scale"], u["noise_scale_w"], u["noise_sdp"][0].numpy(), u["noise_zp"][0].numpy())
    assert np.array_equal(dur, inter["w_ceil"][0, 0].numpy().astype(np.int32)), "durations differ: the stages are not comparable"
    return inter


def _errors(got, ref):
    assert got.shape == ref.shape
    return float(np.abs(got - ref).max()), float(np.linalg.norm(got - ref) / np.linalg.norm(ref))


@gpu
@pytest.mark.parametrize("t_x,seed", [(23, 13), (241, 341)])
def test_transformer_flow_stages_against_oracle(flow_models, t_x, seed):
    """SDP output, prior sample z_p and flow output z (tensor-core window attention in every layer) against the oracle."""
    hp, oracle, model = flow_models[4]
    inter = _run_stages(hp, oracle, model, t_x, seed)
    zs_err = np.abs(model.debug_fetch("z_sdp")[:, 0] - inter["logw_sdp"][0, 0].numpy()).max()
    z_err = _errors(model.debug_fetch("z"), inter["z"][0].numpy().T)
    hp1, oracle1, model1 = flow_models[1]
    inter1 = _run_stages(hp1, oracle1, model1, t_x, seed)
    zp_err = _errors(model1.debug_fetch("z_p"), inter1["z_p"][0].numpy().T)
    print(f"\nflow stages T_x={t_x}: z_sdp max|err| {zs_err:.2e}; z_p max|err| {zp_err[0]:.2e} rel {zp_err[1]:.2e}; "
          f"z max|err| {z_err[0]:.2e} rel {z_err[1]:.2e}", end="")
    # the SDP runs on the text encoder's split-fp16 convs: ~1e-5 relative (test_text_split_convs_match_fp32_path)
    assert zs_err <= 1e-4
    assert zp_err[1] <= 1e-5
    # fp16 operands of the flow's tensor-core convs and attention: the bars of the WN flow's z (test_wn_flow_variant)
    assert z_err[0] <= 2e-2 and z_err[1] <= 2e-3
