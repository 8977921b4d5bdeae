"""DeBERTa attention of sentences of at most 128 tokens against float64, kernel by kernel, through the hooks of
libsbv2_b200_debug.so (csrc/debug_kernels.cu); the GPU tests run with -m gpu on a B200.

Kernels: the single-tile tcgen05 kernels of bert_attention_tc.cu, deberta_attention_tc_kernel (fp16 mode, "single") and
deberta_attention_tc_exact_kernel (exact mode, the default, "exact-single"), and the fp32 CUDA-core kernel
deberta_attention_kernel<true> (launch_deberta_attention_f32, exact mode beyond the tensor-core kernels and their
cross-check), with its fp32 output and with its split output.  The single-tile kernels assume the bucket map linear for
|i - j| <= 127 and bulk-copy one 256-row position window from win0 = span - 127; every 128-row tile reads past the end of
its utterance into the 32-row gap and the next utterance's rows.  The reference assumes neither: it takes each (i, j)'s
position row from HF `make_log_bucket_position` (max_position = 2 span, the model's table) and attends over exactly the
utterance's keys.

Reference.  HF's disentangled attention in float64 numpy on exactly the values the kernel reads: the fp16 operands, the
float64 sum of the two split terms divided by sc, or the fp32 operands.  z_ij = (q_i.k_j + q_i.pk[b(i-j)] +
k_j.pq[b(i-j)]) / sqrt(3 * 64), p = softmax_j(z), ctx = p v.  Inputs: q, k ~ s N(0, 1) with s = 1 and s = 3 (near
one-hot rows), v ~ N(0, 1), position tables 0.5 N(0, 1) with independent rows and one table per head.  Spans 256 (the
model's), 254 (the smallest deberta_attention_tc_supported accepts) and 512; 2 and 16 heads.  The batch puts short
utterances directly before long ones, so that each short tile over-reads real rows of its neighbour.

Bars, per element, from each kernel's rounding points.  u = 2^-24.  mag = sum_d |a_d b_d| of a product, over the
operands the kernel reads; MS, MC, MP the magnitudes of q.k, q.pk and k.pq, A_ic = sum_j p_ij |v_jc|.

* Accumulation.  Products of fp16 values are exact in fp32; each K = 16 MMA step adds two roundings of at most 2^-23 of
  the running sum's magnitude, bounded by mag (STEP = 2^-22 per step).  That the in-MMA sum loses at most 2^-23 is the
  hardware assumption of KAPPA (test_gpu_decoder_kernels.py) and of test_gpu_split_gemm.py.  q.k, q.posK and k.posQ are
  4 steps (K = 64) per operand pair, P V 8 steps (K = 128).
* Split representation (exact kernel).  The reference reads h0 + h1 of each operand, so the only representation error
  of a product is the dropped h1 g1: |h1| <= 2^-11 |X| (1 + 2^-10) + 2^-25 in the scaled units X = sc x, so
  |h1 g1| <= REP |x||g| + 2^-36 (|x| + |g|) / sc + 2^-50 / sc^2, REP = 2^-22 (1 + 2^-9).  (test_gpu_split_gemm.py's
  REP_REL[2] = 2^-20 also covers the representation of fp32 values; here the split values are the reference's.)
  Each product is three cross terms in 12 MMA steps; their magnitudes are at most (1 + 2^-9) mag.
* Logits, raw units (before / sqrt 192):
  - single:  12 STEP-steps (S, C2P, P2C: 4 each) of MS, MC, MP; C2P and P2C rounded to fp16 in the skewed tiles,
    2^-11 (|c2p| + its accumulation error) + 2^-25 each; the fp32 sum S + c2p + p2c, two roundings: 2u (MS + MC + MP).
  - exact-single:  12 STEP-steps per product with the (1 + 2^-9) term magnitudes, REP per product, the fp32 bias tile
    (c2p written, p2c added: one rounding) and S + bias (one more): 2u (MS + MC + MP).
  - f32:  64 sequential fmaf per product (64 u mag), q pre-multiplied by fl(1 / sqrtf(192)) (3 u) and K.posQ
    multiplied after (2 u), C2P + P2C then + S: 2u.  69 u (MS + MC + MP) in all.
  Then the exponent, natural units: the tile kernels form 2^(fmaf(s, c, -fl(m c))) with c = fl(log2 e / sqrtf(192))
  (3 u relative) and one fmaf rounding; a constant error per row cancels in the softmax (the row sum uses the same p),
  the rest is 4u |z - z_max|.  ex2.approx.ftz.f32 has a maximum relative error of 2^-22 (2 ulp) over its range (PTX ISA,
  "ex2" instruction, floating-point notes): EX2 = 2^-22 more.  The f32 kernel's expf is within 2 ulp (CUDA C++
  Programming Guide, single-precision mathematical functions): 2^-22 per exponential, and its online softmax rescales
  the earlier keys by expf(m_old - m_new) once per 64-key tile: (tiles (2^-22 + u) + u (z_max - z_min)) more.
* Softmax.  With logit errors |dz_ij| <= d_ij, p_j is increasing in z_j and decreasing in every other z_k, so
  p~_j <= p_j e^{d_j} / (p_j e^{d_j} + sum_{k != j} p_k e^{-d_k}) and the mirror bound below: each |p~_j - p_j| has a
  closed-form bound dp_j.  With one row-wide D_i = max_j d_ij this is at most p_j (1 - p_j) (e^{2 D_i} - 1), tighter
  than p_j (e^{2 D_i} - 1) for near one-hot rows.  Logit part of the bar: L_ic = sum_j dp_ij |v_jc|.
* After the logits, relative to A~ = A + L:
  - single:  P rounded to fp16 (2^-11 p + 2^-25), 8 STEP-steps of P V, the row sum l summed in fp32 over the unrounded
    p ((len - 1) u), 1 / l and O / l (2u); abs 2^-25 sum_j |v_jc| / l.  The fp16 store: half an ulp16 of the result.
  - exact-single:  P as two terms (2^-22 p + 2^-25 each), the dropped P1 V1 (2^-22 p |v| + 2^-35 |v|), 24 STEP-steps
    of P V (three cross terms), l and the division as above; the output as two terms of ctx sc: 2^-22 |ctx| + 2^-25 / sc.
  - f32:  the fmaf chain of P V and the rescales ((L + tiles) u), l ((L + 3 tiles) u), the division (2u); the split
    output adds 2^-22 |ctx| + 2^-25 / split_scale.
  Everything after the logits is multiplied by (1 + 2^-10) for second-order terms.
On inputs distributed as test_gpu_bert_long.py's (q, k ~ N(0, 1)) every bar is within the multi-tile kernels' bars there
(2e-2 fp16, 1e-4 exact), which test_bars_within_the_multi_tile_bars asserts; at 3 N(0, 1) the exact bar reaches ~6e-4
through the accumulation term of logits ~9x larger.  -s prints every case's max |err| / bar.

Bit-level checks: a batch equals each utterance run alone; two launches give the same bits; the output is the same
whether the padding rows (gaps, tail) hold zeros or seeded finite fp16 values, as rows an earlier batch leaves behind;
no planar row outside the utterances is written (the output planes hold a sentinel before).  The exact kernels (single-
and multi-tile) write block 3 equal to block 1 and |h1| <= ulp16(h0) / 2; the f32 kernel's split planes are numpy's split
of its own fp32 output times split_scale.

test_bars_catch_mutants (CPU) checks on the same inputs that each of a set of plausible mistakes moves some element past
its bar: the window shifted by one row either way, c2p or p2c read at b(j - i), posK and posQ swapped, sqrt(2 * 64)
instead of sqrt(3 * 64), the last valid key dropped or the key at j = len admitted (with a zero V row, as the kernels
zero V there), heads reading each other's tables; for the exact bars, the h1 term of q, of posK or of P dropped.
"""
import functools

import numpy as np
import pytest
import torch
from transformers.models.deberta_v2.modeling_deberta_v2 import make_log_bucket_position

from test_gpu_decoder_kernels import excess, ulp16
from test_gpu_split_gemm import np_split

gpu = pytest.mark.gpu

U = 2.0 ** -24
STEP = 2.0 ** -22           # two roundings of 2^-23 per K = 16 MMA step
REP = 2.0 ** -22 * (1 + 2.0 ** -9)
EX2 = 2.0 ** -22            # ex2.approx.f32, PTX ISA
EXPF = 2.0 ** -22           # expf, 2 ulp
SECOND = 1 + 2.0 ** -10
SQ = np.sqrt(3 * 64)
BAR_MAX = {"single": 2e-2, "exact-single": 1e-4}  # the multi-tile kernels' bars (test_gpu_bert_long.py)

# short utterances before long ones: every short tile over-reads real rows of its neighbour
LENS = [1, 128, 2, 127, 7, 97, 8, 96, 9, 128, 16, 97, 17, 96, 31, 65, 32, 64, 33, 63, 64, 65, 96, 127, 128]
LENS_LONG = LENS + [129, 300, 700]  # the f32 kernel at every length
SPANS = [256, 254, 512]
HEADS = [2, 16]
SCALES = [1.0, 3.0]
SCS = [16.0, 4.0]  # exact-single: the model's split scale and another power of two
KINDS = ["single", "exact-single", "f32", "f32-split"]


# ---------------------------------------------------------------------------------------------------------------------
# inputs and the float64 reference
# ---------------------------------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def bucket_index(n, span):
    """position row of each (i, j) of an n-token sentence: HF make_log_bucket_position(i - j, span, 2 span) + span,
    clamped to the table"""
    rel = np.arange(n)[:, None] - np.arange(n)[None, :]
    b = make_log_bucket_position(torch.from_numpy(rel), span, 2 * span)
    return torch.clamp(b + span, 0, 2 * span - 1).long().numpy()


@functools.lru_cache(maxsize=None)
def base_inputs(span, heads, scale, long):
    lens = LENS_LONG if long else LENS
    rng = np.random.default_rng(1000 * span + 10 * heads + int(scale) + (5 if long else 0))
    H = heads * 64
    qkv = rng.standard_normal((sum(lens), 3 * H))
    qkv[:, :2 * H] *= scale
    pk = 0.5 * rng.standard_normal((2 * span, H))
    pq = 0.5 * rng.standard_normal((2 * span, H))
    return lens, qkv, pk, pq


def split_terms(x, sc):
    """two fp16 terms of x * sc"""
    h0 = (x * sc).astype(np.float16)
    return np.stack([h0, (x * sc - h0.astype(np.float64)).astype(np.float16)])


def operands(kind, span, heads, scale, sc=16.0):
    """(what the hook takes, the float64 values the kernel reads, the split terms or None)"""
    lens, qkv, pk, pq = base_inputs(span, heads, scale, kind.startswith("f32"))
    if kind == "single":
        ops = tuple(a.astype(np.float16) for a in (qkv, pk, pq))
        return lens, ops, tuple(a.astype(np.float64) for a in ops), None
    if kind == "exact-single":
        terms = tuple(split_terms(a, sc) for a in (qkv, pk, pq))
        return lens, terms, tuple(t.astype(np.float64).sum(axis=0) / sc for t in terms), terms
    ops = tuple(a.astype(np.float32) for a in (qkv, pk, pq))
    return lens, ops, tuple(a.astype(np.float64) for a in ops), None


def heads_of(qkv, heads, h):
    H = heads * 64
    return qkv[:, h * 64:(h + 1) * 64], qkv[:, H + h * 64:H + (h + 1) * 64], qkv[:, 2 * H + h * 64:2 * H + (h + 1) * 64]


def logits(q, k, pk, pq, span, mut=None):
    """raw scores (q.k, c2p, p2c) of one head, with HF's bucket rows; mut: a mistake to restate"""
    n = len(q)
    ix = bucket_index(n, span)
    if mut in ("win+1", "win-1"):
        ix = np.clip(ix + (1 if mut == "win+1" else -1), 0, 2 * span - 1)
    if mut == "swap":
        pk, pq = pq, pk
    c2p = np.take_along_axis(q @ pk.T, ix.T if mut == "c2p_ji" else ix, axis=1)   # q_i . pk[b(i - j)]
    p2c = np.take_along_axis(k @ pq.T, ix if mut == "p2c_ji" else ix.T, axis=1).T  # k_j . pq[b(i - j)]
    return q @ k.T, c2p, p2c


def attend(q, k, v, pk, pq, span, mut=None, p_h0=False):
    """float64 context of one head; p_h0: P rounded to one fp16 term before P V (the row sum unrounded)"""
    if mut == "admit":  # the key at j = len with a zero k row (the gap) and a zero V row
        z1 = np.zeros((1, k.shape[1]))
        k, v = np.vstack([k, z1]), np.vstack([v, z1])
        q = np.vstack([q, z1])
    if mut == "drop" and len(q) > 1:
        k, v = k[:-1], v[:-1]
    n = len(q)
    if len(k) != n:  # square the score matrix for the gather; the extra query row is dropped below
        m = max(n, len(k))
        q = np.vstack([q, np.zeros((m - n, q.shape[1]))])
        k2 = np.vstack([k, np.zeros((m - len(k), k.shape[1]))])
        s, c2p, p2c = logits(q, k2, pk, pq, span, mut)
        s, c2p, p2c = (a[:n, :len(k)] for a in (s, c2p, p2c))
    else:
        s, c2p, p2c = logits(q, k, pk, pq, span, mut)
    z = (s + c2p + p2c) / (np.sqrt(2 * 64) if mut == "sqrt2" else SQ)
    p = np.exp(z - z.max(axis=1, keepdims=True))
    l = p.sum(axis=1, keepdims=True)
    if p_h0:
        p = p.astype(np.float32).astype(np.float16).astype(np.float64)
    out = (p / l) @ v
    return out[:-1] if mut == "admit" else out


def head_bar(kind, q, k, v, pk, pq, span, sc):
    """(float64 context, per-element bar) of one head; see the module docstring"""
    n = len(q)
    ix = bucket_index(n, span)
    s, c2p, p2c = logits(q, k, pk, pq, span)
    aq, ak, apk, apq = np.abs(q), np.abs(k), np.abs(pk), np.abs(pq)
    MS = aq @ ak.T
    MC = np.take_along_axis(aq @ apk.T, ix, axis=1)
    MP = np.take_along_axis(ak @ apq.T, ix.T, axis=1).T
    M = MS + MC + MP
    z = (s + c2p + p2c) / SQ
    zmax = z.max(axis=1, keepdims=True)
    zr = zmax - z
    tiles = -(-n // 64)
    if kind == "single":
        eC = 4 * STEP * MC
        eP = 4 * STEP * MP
        raw = 4 * STEP * MS + eC + eP + 2.0 ** -11 * (np.abs(c2p) + eC + np.abs(p2c) + eP) + 2 * 2.0 ** -25 + 2 * U * M * SECOND
    elif kind == "exact-single":
        sq, sk = aq.sum(axis=1), ak.sum(axis=1)
        spk, spq = apk.sum(axis=1)[ix], apq.sum(axis=1)[ix.T].T
        rep_abs = 2.0 ** -36 / sc * (2 * sq[:, None] + 2 * sk[None, :] + spk + spq) + 3 * 64 * 2.0 ** -50 / sc ** 2
        raw = (12 * STEP * (1 + 2.0 ** -9) + REP + 2 * U) * M + rep_abs
    else:
        raw = 69 * U * M
    d_raw = raw / SQ
    if kind.startswith("f32"):
        d = d_raw + EXPF + U * zr + tiles * (EXPF + U) + U * (zmax - z.min(axis=1, keepdims=True))
    else:
        d = d_raw + EX2 + 4 * U * (zr + 2 * d_raw.max(axis=1, keepdims=True))
    p = np.exp(-zr)
    p /= p.sum(axis=1, keepdims=True)
    ctx = p @ v
    # closed-form bound of |p~ - p| under |dz_j| <= d_j
    e_hi, e_lo = p * np.exp(d), p * np.exp(-d)
    s_hi, s_lo = e_hi.sum(axis=1, keepdims=True), e_lo.sum(axis=1, keepdims=True)
    dp = np.maximum(e_hi / (e_hi + s_lo - e_lo) - p, p - e_lo / (e_lo + s_hi - e_hi))
    av = np.abs(v)
    L = dp @ av
    A = p @ av + L
    sv = av.sum(axis=0)[None, :] * np.exp(d.max(axis=1, keepdims=True)) / np.exp(-zr).sum(axis=1, keepdims=True)  # sum|v| / l
    if kind == "single":
        rel = 2.0 ** -11 + 8 * STEP * (1 + 2.0 ** -11) + (n - 1) * U + 2 * U
        post = rel * A + 2.0 ** -25 * sv
    elif kind == "exact-single":
        rel = 2.0 ** -22 + 2.0 ** -22 + 24 * STEP * (1 + 2.0 ** -9) + (n - 1) * U + 2 * U
        post = rel * A + (2.0 ** -25 + 2.0 ** -35) * sv
    else:
        rel = (n + tiles) * U + (n + 3 * tiles) * U + 2 * U
        post = rel * A
    pre = L + SECOND * post
    if kind == "single":
        bar = pre + ulp16(np.abs(ctx) + pre) / 2
    elif kind == "exact-single":
        bar = pre + 2.0 ** -22 * (np.abs(ctx) + pre) + 2.0 ** -25 / sc
    elif kind == "f32-split":
        bar = pre + 2.0 ** -22 * (np.abs(ctx) + pre) + 2.0 ** -25 / SC_F32
    else:
        bar = pre
    return ctx, bar


SC_F32 = 16.0  # the split output's scale (the model's kSplitScale)


def reference(kind, span, heads, scale, sc=16.0):
    """(lens, hook operands, split terms, float64 context [rows, H], bar [rows, H])"""
    lens, ops, val, terms = operands(kind, span, heads, scale, sc)
    qkv, pk, pq = val
    rows, H = qkv.shape[0], heads * 64
    ref, bar = np.zeros((rows, H)), np.zeros((rows, H))
    off = 0
    for n in lens:
        sl = slice(off, off + n)
        for h in range(heads):
            q, k, v = heads_of(qkv[sl], heads, h)
            c = slice(h * 64, (h + 1) * 64)
            ref[sl, c], bar[sl, c] = head_bar(kind, q, k, v, pk[:, c], pq[:, c], span, sc)
        off += n
    return lens, ops, terms, ref, bar


def mutant(kind, span, heads, scale, mut, sc=16.0, drop_h1=None):
    """float64 context [rows, H] of a mistaken kernel on the same inputs"""
    lens, _, val, terms = operands(kind, span, heads, scale, sc)
    qkv, pk, pq = (a.copy() for a in val)
    H = heads * 64
    if drop_h1 == "q":
        qkv[:, :H] = terms[0][0][:, :H].astype(np.float64) / sc
    elif drop_h1 == "posK":
        pk = terms[1][0].astype(np.float64) / sc
    out = np.zeros((qkv.shape[0], H))
    off = 0
    for n in lens:
        sl = slice(off, off + n)
        for h in range(heads):
            q, k, v = heads_of(qkv[sl], heads, h)
            t = (h + 1) % heads if mut == "heads" else h
            c, ct = slice(h * 64, (h + 1) * 64), slice(t * 64, (t + 1) * 64)
            out[sl, c] = attend(q, k, v, pk[:, ct], pq[:, ct], span, mut, p_h0=drop_h1 == "P")
        off += n
    return out


def ratio(got, ref, bar):
    return float(np.nanmax(np.where(np.isnan(got), np.inf, np.abs(got - ref)) / bar))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference and the bars
# ---------------------------------------------------------------------------------------------------------------------

def test_reference_restates_hf_attention():
    """attend() against HF's DisentangledSelfAttention (oracle/deberta.py's tiny model, one layer, float64; HF forms
    sqrt(3 d) in float32, a relative 1e-8 on every logit)."""
    from oracle import deberta as od
    cfg = od.tiny_config()
    hf = od.build_model(cfg, seed=1).double()
    layer = hf.encoder.layer[0].attention.self
    n, heads = 100, cfg.num_attention_heads
    d = cfg.hidden_size // heads
    assert d == 64
    rng = np.random.default_rng(3)
    x = torch.from_numpy(rng.standard_normal((1, n, cfg.hidden_size)))
    rel_emb = torch.from_numpy(0.5 * rng.standard_normal((2 * cfg.position_buckets, cfg.hidden_size)))
    rel_pos = hf.encoder.get_rel_pos(x)
    with torch.no_grad():
        got = layer(x, torch.ones(1, 1, n, n, dtype=torch.bool), output_attentions=False, relative_pos=rel_pos, rel_embeddings=rel_emb)
        got = (got[0] if isinstance(got, tuple) else got)[0].numpy()
        q = layer.query_proj(x)[0].numpy()
        k = layer.key_proj(x)[0].numpy()
        v = layer.value_proj(x)[0].numpy()
        pk = layer.key_proj(rel_emb).numpy()
        pq = layer.query_proj(rel_emb).numpy()
    span = cfg.position_buckets
    for h in range(heads):
        c = slice(h * d, (h + 1) * d)
        np.testing.assert_allclose(attend(q[:, c], k[:, c], v[:, c], pk[:, c], pq[:, c], span), got[:, c], rtol=0, atol=1e-7)


def test_single_tile_window_is_linear():
    """What the single-tile kernels assume and the reference does not: b(i - j) = i - j + span for |i - j| <= 127 at every
    span they accept (>= 254), so their window starts at row span - 127."""
    for span in SPANS:
        ix = bucket_index(128, span)
        rel = np.arange(128)[:, None] - np.arange(128)[None, :]
        assert np.array_equal(ix, rel + span), span


@pytest.mark.parametrize("kind", ["single", "exact-single"])
def test_bars_within_the_multi_tile_bars(kind):
    """On inputs distributed as test_gpu_bert_long.py's (q, k ~ N(0, 1)) every bar is within the multi-tile kernels' bar.
    At 3 N(0, 1) the exact bar grows with the logits' magnitude (the MMA accumulation term): printed, not asserted."""
    worst = {}
    for span in SPANS:
        for heads in HEADS:
            for scale in SCALES:
                for sc in (SCS if kind == "exact-single" else [16.0]):
                    worst[scale] = max(worst.get(scale, 0.0), float(reference(kind, span, heads, scale, sc)[4].max()))
    print(f"\n{kind}: largest bar {worst[1.0]:.3e} at q, k ~ N(0, 1), {worst[3.0]:.3e} at 3 N(0, 1) (the multi-tile kernels' bar "
          f"{BAR_MAX[kind]})", end="")
    assert worst[1.0] <= BAR_MAX[kind]


GENERIC_MUTANTS = ["win+1", "win-1", "c2p_ji", "p2c_ji", "swap", "sqrt2", "drop", "admit", "heads"]


def test_bars_catch_mutants():
    """Each mutant, on the inputs the GPU tests use, moves some element past its bar."""
    for kind in ("single", "exact-single", "f32", "f32-split"):
        for span in SPANS:
            _, _, _, ref, bar = reference(kind, span, 2, 1.0)
            assert ratio(ref, ref, bar) == 0
            for mut in GENERIC_MUTANTS:
                r = ratio(mutant(kind, span, 2, 1.0, mut), ref, bar)
                assert r > 1, f"{kind} span {span}: mutant {mut} stays within the bars (max |err| / bar {r:.3f})"
    for sc in SCS:
        for scale in SCALES:
            _, _, _, ref, bar = reference("exact-single", 256, 2, scale, sc)
            for what in ("q", "posK", "P"):
                r = ratio(mutant("exact-single", 256, 2, scale, None, sc, drop_h1=what), ref, bar)
                print(f"\nexact-single sc {sc} scale {scale}: h1 of {what} dropped: max |err| / bar {r:.1f}", end="")
                assert r > 1, f"sc {sc} scale {scale}: h1 of {what} dropped stays within the bars ({r:.3f})"


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def S(lib_built):
    """Builds first (a no-op when up to date), so that an older debug library without these hooks cannot be used."""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("sbv2_b200_build", os.path.join(root, "sbv2-api_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()
    import sbv2_b200
    if sbv2_b200.device_count() < 1:
        pytest.fail("GPU tests selected but no B200 is visible")
    return sbv2_b200


def run(S, kind, lens, ops, heads, sc=16.0, pad_seed=0):
    """-> (float64 context [rows, H], raw output: fp16 blocks or the f32 kernel's (ctx, split), stray rows)"""
    if kind in ("single", "exact-single"):
        out, stray = S.debug_deberta_attention(*ops, lens, heads, kind, sc=sc, all_blocks=kind == "exact-single", pad_seed=pad_seed,
                                               with_stray=True)
        o = out.astype(np.float64)
        return (o[0] if kind == "single" else (o[0] + o[1]) / sc), out, stray
    ctx, split, stray = S.debug_deberta_attention_f32(*ops, lens, heads, out=kind == "f32", split_scale=SC_F32 if kind == "f32-split" else 0.0)
    got = ctx.astype(np.float64) if kind == "f32" else split[:2].astype(np.float64).sum(axis=0) / SC_F32
    return got, (ctx, split), stray


def check_split_blocks(blocks, what):
    """[h0 | h1 | h0]: block 3 equals block 1 bit for bit and |h1| <= ulp16(h0) / 2"""
    assert np.array_equal(blocks[2].view(np.uint16), blocks[0].view(np.uint16)), f"{what}: block 3 differs from block 1"
    h0, h1 = blocks[0].astype(np.float64), blocks[1].astype(np.float64)
    assert np.isfinite(h0).all() and np.isfinite(h1).all(), f"{what}: non-finite split terms"
    ex, i = excess(np.abs(h1), 0.0, ulp16(h0) / 2)
    assert ex <= 0, f"{what}: |h1| {abs(h1[i]):.3e} > ulp16(h0) / 2 at {i} (h0 {h0[i]:.6e})"


CASES = [(k, span, heads, scale, sc) for k in KINDS for span in SPANS for heads in HEADS for scale in SCALES
         for sc in (SCS if k == "exact-single" else [16.0])]


@gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-span{c[1]}-h{c[2]}-s{c[3]:g}" + (f"-sc{c[4]:g}" if c[0] == "exact-single" else ""))
def test_against_float64(S, case):
    kind, span, heads, scale, sc = case
    lens, ops, _, ref, bar = reference(kind, span, heads, scale, sc)
    got, raw, stray = run(S, kind, lens, ops, heads, sc)
    assert stray == 0, f"{stray} planar rows outside the utterances written"
    r = ratio(got, ref, bar)
    err = np.where(np.isnan(got), np.inf, np.abs(got - ref))
    print(f"\n{kind} span {span} heads {heads} q,k ~ {scale:g} N(0,1)" + (f" sc {sc:g}" if kind == "exact-single" else "")
          + f": max |err| {err.max():.3e}, max bar {bar.max():.3e}, max |err| / bar = {r:.4f}", end="")
    if r > 1:
        ex, i = excess(got, ref, bar)
        row = i[0]
        utt = int(np.searchsorted(np.cumsum(lens), row, side="right"))
        pytest.fail(f"element {i} (utterance {utt}, length {lens[utt]}, head {i[1] // 64}): got {got[i]!r}, ref {ref[i]!r}, bar {bar[i]:.3e}")
    if kind == "exact-single":
        check_split_blocks(raw, kind)
    if kind == "f32-split":
        check_split_blocks(raw[1], kind)


@gpu
@pytest.mark.parametrize("kind", KINDS)
def test_bits(S, kind):
    """Two launches give the same bits, seeded padding the same bits as zero padding (the tile kernels read it), and
    each utterance alone the bits of its rows in the batch."""
    span, heads = 256, 16
    lens, ops, _, _, _ = reference(kind, span, heads, 1.0)
    bits = lambda raw: (raw.view(np.uint16) if kind in ("single", "exact-single") else
                        (raw[0].view(np.uint32) if kind == "f32" else raw[1].view(np.uint16)))
    a = bits(run(S, kind, lens, ops, heads)[1])
    assert np.array_equal(a, bits(run(S, kind, lens, ops, heads)[1])), "two launches differ"
    if kind in ("single", "exact-single"):
        for seed in (1, 0xDEADBEEF):
            _, raw, stray = run(S, kind, lens, ops, heads, pad_seed=seed)
            assert stray == 0
            assert np.array_equal(bits(raw), a), f"padding seed {seed}: the output depends on the padding rows' contents"
    off = 0
    for n in lens:
        one_ops = ((ops[0][:, off:off + n] if kind == "exact-single" else ops[0][off:off + n]),) + ops[1:]
        one = bits(run(S, kind, [n], one_ops, heads)[1])
        batch = a[:, off:off + n] if a.ndim == 3 else a[off:off + n]
        assert np.array_equal(one, batch), f"length {n} at row {off}: alone differs from the batch"
        off += n


@gpu
def test_f32_split_output_is_numpy_split(S):
    """The split output of the f32 kernel is numpy's two-term split of its own fp32 output times split_scale."""
    for span, heads in ((256, 16), (512, 2)):
        lens, ops, _, _, _ = reference("f32", span, heads, 3.0)
        ctx, split, stray = S.debug_deberta_attention_f32(*ops, lens, heads, out=True, split_scale=SC_F32)
        assert stray == 0
        h0, h1 = np_split(ctx * np.float32(SC_F32), 2)
        assert np.array_equal(split[0].view(np.uint16), h0.view(np.uint16)), f"span {span}: h0 differs from numpy's split"
        assert np.array_equal(split[1].view(np.uint16), h1.view(np.uint16)), f"span {span}: h1 differs from numpy's split"
        check_split_blocks(split, f"f32 span {span}")


@gpu
def test_exact_multi_tile_blocks(S):
    """The exact multi-tile kernel's three output blocks, on a batch reaching 700 tokens: [h0 | h1 | h0], no stray rows."""
    _, _, _, terms = operands("exact-single", 256, 2, 1.0)
    lens_long = LENS_LONG
    rng = np.random.default_rng(11)
    H = 2 * 64
    qkv = split_terms(rng.standard_normal((sum(lens_long), 3 * H)), 16.0)
    out, stray = S.debug_deberta_attention(qkv, terms[1], terms[2], lens_long, 2, "exact-multi", sc=16.0, all_blocks=True,
                                           pad_seed=7, with_stray=True)
    assert stray == 0
    check_split_blocks(out, "exact-multi")
    two = S.debug_deberta_attention(qkv, terms[1], terms[2], lens_long, 2, "exact-multi", sc=16.0)
    assert np.array_equal(two.view(np.uint16), out[:2].view(np.uint16)), "the two-block call differs from the three-block call"
