"""GPU unit tests of individual tensor-core kernels through their debug hooks (run with -m gpu on a B200).

* fused ResBlock pair (umma_pair.cu) against the two unfused tensor-core convs (bit-identical: same fp16
  rounding points, same fp32 accumulation order), against a numpy fp32 evaluation of
  oracle/vits.py ResBlock1 (one conv1/conv2 pair), and per element against a float64 evaluation with the bars of
  test_gpu_decoder_kernels.py, on ragged batches that exercise tile boundaries;
* split-fp16 text-encoder convs against the CUDA-core fp32 path of the same model.
"""
import ctypes as C
import os

import numpy as np
import pytest

import util
from test_gpu_decoder_kernels import KAPPA, conv_offs, taps_ref, ulp16, xrec
from util import ov

pytestmark = pytest.mark.gpu

pf = C.POINTER(C.c_float)
pi = C.POINTER(C.c_int)


@pytest.fixture(scope="module")
def S(lib_built):
    import sbv2_b200
    if sbv2_b200.device_count() < 1:
        pytest.fail("GPU tests selected but no B200 is visible: " + sbv2_b200.lib.sbv2_last_error().decode())
    fn = sbv2_b200.debug_lib().sbv2_debug_pair_compare   # unit-test hooks live in libsbv2_b200_debug.so only
    fn.restype = C.c_int
    fn.argtypes = [pf, pi, C.c_int, C.c_int, C.c_int, C.c_int, pf, pf, pf, pf, C.c_int, C.c_int, pf, pf, pf, pi, C.POINTER(C.c_longlong)]
    return sbv2_b200


def lrelu(v, s=0.1):
    return np.where(v >= 0, v, v * s)


def conv_np(x, w, b, dil):  # x [T, C], w [Co, Ci, k], "same" zero padding
    T = x.shape[0]
    k = w.shape[2]
    pad = dil * (k - 1) // 2
    xp = np.zeros((T + 2 * pad, x.shape[1]), np.float32)
    xp[pad:pad + T] = x
    out = np.tile(b[None, :], (T, 1)).astype(np.float32)
    for j in range(k):
        out += xp[j * dil:j * dil + T] @ w[:, :, j].T
    return out


def f16(a):
    return a.astype(np.float16).astype(np.float32)


@pytest.mark.parametrize("c,k,dil,mrf", [(16, 3, 1, 0), (16, 11, 5, 0), (16, 7, 3, 1), (32, 3, 5, 0), (32, 11, 1, 0), (32, 7, 5, 1),
                                         (64, 3, 1, 0), (64, 7, 3, 0), (64, 11, 5, 0), (64, 11, 5, 1),
                                         (128, 3, 1, 0), (128, 7, 3, 0), (128, 3, 5, 1), (128, 7, 5, 1)])
def test_fused_resblock_pair(S, c, k, dil, mrf):
    rng = np.random.default_rng(c * 100 + k * 10 + dil)
    lens = np.asarray([50, 1, 700, 1300, 129, 2500, 1022, 1023], np.int32)  # tile-edge lengths included
    tot = int(lens.sum())
    x = rng.standard_normal((tot, c)).astype(np.float32)
    w1 = f16(rng.standard_normal((c, c, k)) / np.sqrt(c * k))
    w2 = f16(rng.standard_normal((c, c, k)) / np.sqrt(c * k))
    b1 = (rng.standard_normal(c) * 0.1).astype(np.float32)
    b2 = (rng.standard_normal(c) * 0.1).astype(np.float32)
    fused = np.zeros((tot, c), np.float32)
    unfused = np.zeros((tot, c), np.float32)
    ms = np.zeros(2, np.float32)
    cfg = np.zeros(8, np.int32)
    st = S.debug_lib().sbv2_debug_pair_compare(x.ctypes.data_as(pf), lens.ctypes.data_as(pi), len(lens), c, k, dil, w1.ctypes.data_as(pf),
                                       b1.ctypes.data_as(pf), w2.ctypes.data_as(pf), b2.ctypes.data_as(pf), mrf, 0,
                                       fused.ctypes.data_as(pf), unfused.ctypes.data_as(pf), ms.ctypes.data_as(pf),
                                       cfg.ctypes.data_as(pi), None)
    assert st == 0, S.debug_lib().sbv2_last_error().decode()
    assert np.array_equal(fused, unfused), "fused pair differs from the two unfused tensor-core convs"
    # numpy evaluation with the kernels' rounding points: stored activations and the intermediate are fp16
    y = f16(lrelu(x))
    xr = np.where(y >= 0, y, y * 10.0)
    ref = np.zeros_like(x)
    o = 0
    for n in lens:
        t1 = f16(lrelu(conv_np(y[o:o + n], w1, b1, dil)))
        ref[o:o + n] = conv_np(t1, w2, b2, 1) + xr[o:o + n]
        o += n
    if mrf:  # the hook feeds lrelu(x) and x (stored as-is) as the two other ResBlock outputs
        yb = f16(x)
        ref = (xr + np.where(yb >= 0, yb, yb * 10.0) + ref) / 3.0
    ref = lrelu(ref)
    assert np.abs(fused - ref).max() <= 4e-3 * max(1.0, np.abs(ref).max())  # fp16 output rounding of values up to ~6
    # float64 per element.  t1 is rounded to fp16 as the kernel stores it; the kernel's fp32 t1 (off by up to KAPPA * its
    # sum of |terms|) may round to the neighbouring fp16 value, which conv2 weighs with |w2|.
    p1, m1 = taps_ref(y, w1, conv_offs(k, dil), lens)
    p1 += b1
    m1 += np.abs(b1)
    t1 = f16(lrelu(p1))
    e1 = KAPPA * m1 + ulp16(np.abs(t1) + KAPPA * m1)
    v, mag = taps_ref(t1, w2, conv_offs(k, 1), lens)
    v += b2 + xr
    mag += np.abs(b2) + np.abs(xr)
    if mrf:
        rb = xrec(f16(x))
        v = ((xr + rb) + v) / 3.0
        mag += np.abs(xr) + np.abs(rb)
    ref64 = lrelu(v)
    bar = ulp16(ref64) + KAPPA * mag + taps_ref(e1, np.abs(w2), conv_offs(k, 1), lens)[0]
    err = np.abs(fused - ref64) - bar
    i = np.unravel_index(np.argmax(err), err.shape)
    print(f"pair C{c} k{k} d{dil} mrf{mrf}: max |err| / bar = {float((np.abs(fused - ref64) / bar).max()):.3f}")
    assert err[i] <= 0, f"element {i}: fused {fused[i]!r}, float64 {ref64[i]!r}, bar {bar[i]:.3e}"


def test_text_split_convs_match_fp32_path(S):
    """Text encoder + duration predictor on tensor cores (two-term fp16 split) against the CUDA-core fp32 kernels of the
    same model: same integer durations, hidden states within 1e-4."""
    hp = ov.HParams()
    oracle, onnx = util.synth_assets(hp, seed=0)
    u = util.make_utterance(hp, 97, seed=5, sdp_ratio=0.0)
    got = {}
    for mode in ("split2", "fp32", "split3"):
        os.environ["SBV2_B200_TEXT"] = mode
        try:
            model = S.Model(onnx, bert=False)
        finally:
            del os.environ["SBV2_B200_TEXT"]
        audio, dur, f2p = model.synthesize_with_noise(u["bert"][0].numpy(), u["x"][0].numpy(), u["sid"], u["tone"][0].numpy(),
                                                      u["lang"][0].numpy(), u["style"][0].numpy(), u["sdp_ratio"], u["length_scale"],
                                                      u["noise_scale"], u["noise_scale_w"], u["noise_sdp"][0].numpy(),
                                                      u["noise_zp"][0].numpy())
        got[mode] = (dur.copy(), model.debug_fetch("enc_x").copy(), model.debug_fetch("logw_dp").copy(), audio.copy())
        del model
    for mode in ("split2", "split3"):
        assert np.array_equal(got[mode][0], got["fp32"][0])
        assert np.abs(got[mode][1] - got["fp32"][1]).max() <= 1e-4 * max(1.0, np.abs(got["fp32"][1]).max())
        assert np.abs(got[mode][2] - got["fp32"][2]).max() <= 2e-5
        assert np.abs(got[mode][3] - got["fp32"][3]).max() <= 1e-3


@pytest.mark.parametrize("env", [{"SBV2_B200_CLUSTER": "2"}, {"SBV2_B200_CLUSTER": "4"},
                                 {"SBV2_B200_PAIR2": "1", "SBV2_B200_TEST_NBMAX": "128"}], ids=["cluster2", "cluster4", "pair2"])
def test_conv_kernel_cluster_and_pair_variants(S, env):
    """The optional launch modes of umma_conv_kernel — thread-block clusters with multicast weight stages and CTA pairs
    (tcgen05 cta_group::2, M = 256) — against the fp32 CUDA-core conv on 20 shapes (tools/umma_conv_check.py).  The
    switches are read once per process, hence the subprocess."""
    import subprocess
    import sys
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "umma_conv_check.py")], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, **env))
    lines = [l for l in r.stdout.splitlines() if l.startswith(("OK", "BAD")) or "ERROR" in l]
    assert r.returncode == 0 and len(lines) >= 20, r.stderr[-1500:]
    assert all(l.startswith("OK") for l in lines), "\n".join(l for l in lines if not l.startswith("OK"))
