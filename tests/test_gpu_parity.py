"""GPU parity tests (run with -m gpu on a B200): the CUDA path through the C ABI against the CPU
oracle on the same seeded inputs with the noise injected explicitly.

Bars (BASELINE.json north_star): durations and frame->phoneme alignment bit-exact; waveform
max-abs <= 1e-3 (fp16 tensor-core operands, fp32 accumulate; synthetic weights calibrated so the
waveform peaks at ~0.3, i.e. 1e-3 is a ~0.3 % bound).  A duration may legitimately differ only when
the fp64 oracle shows w within 1e-4 of an integer (documented tie, SURVEY.md §7.3.1).
"""
import os

import numpy as np
import pytest
import torch

import util
from util import ov

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
WAVE_TOL = 1e-3


@pytest.fixture(scope="module")
def S(lib_built):
    import sbv2_b200
    if sbv2_b200.device_count() < 1:
        pytest.fail("GPU tests selected but no B200 is visible: " + sbv2_b200.lib.sbv2_last_error().decode())
    return sbv2_b200


@pytest.fixture(scope="module")
def full(S):
    hp = ov.HParams()
    oracle, onnx = util.synth_assets(hp, seed=0)
    model = S.Model(onnx, bert=False)
    return hp, oracle, model


@pytest.fixture(scope="module")
def tiny(S):
    hp = ov.tiny_hparams()
    oracle, onnx = util.synth_assets(hp, seed=0)
    model = S.Model(onnx, bert=False)
    return hp, oracle, model


def run_gpu(model, u):
    return model.synthesize_with_noise(u["bert"][0].numpy(), u["x"][0].numpy(), u["sid"], u["tone"][0].numpy(),
                                       u["lang"][0].numpy(), u["style"][0].numpy(), u["sdp_ratio"], u["length_scale"],
                                       u["noise_scale"], u["noise_scale_w"], u["noise_sdp"][0].numpy(), u["noise_zp"][0].numpy())


def check_alignment(oracle, u, inter, dur, f2p):
    ref_d = inter["w_ceil"][0, 0].numpy().astype(np.int32)
    if not np.array_equal(dur, ref_d):
        # only near-ties of the real-valued duration may differ
        _, i64 = util.oracle_run(oracle, u, dtype=torch.float64)
        w64 = i64["w"][0, 0].numpy()
        bad = np.nonzero(dur != ref_d)[0]
        margin = np.abs(w64[bad] - np.round(w64[bad]))
        assert (margin < 1e-4).all(), f"durations differ at {bad} with fp64 margins {margin}"
        pytest.skip(f"documented duration tie at phonemes {bad.tolist()} (fp64 margin {margin.max():.2e})")
    attn = inter["attn"][0, 0].numpy()
    assert len(f2p) == attn.shape[0]
    assert np.array_equal(f2p, attn.argmax(1).astype(np.int32))


@pytest.mark.parametrize("sdp_ratio", [0.0, 0.4, 1.0])
def test_cfg1_short_utterance(full, sdp_ratio):
    """BASELINE config 1: one short utterance (T_x = 23, 'こんにちは'-shaped)."""
    hp, oracle, model = full
    u = util.make_utterance(hp, 23, seed=13, sdp_ratio=sdp_ratio)
    ref, inter = util.oracle_run(oracle, u)
    audio, dur, f2p = run_gpu(model, u)
    check_alignment(oracle, u, inter, dur, f2p)
    assert audio.shape[0] == ref.shape[-1] == 512 * len(f2p)
    err = np.abs(audio - ref[0, 0].numpy()).max()
    assert err <= WAVE_TOL, f"waveform max-abs {err:.3e} (peak {float(ref.abs().max()):.3f})"


@pytest.mark.parametrize("t_x,length_scale", [(1, 1.0), (3, 1.0), (101, 0.5), (241, 1.0), (77, 2.0)])
def test_lengths_and_length_scale(full, t_x, length_scale):
    hp, oracle, model = full
    u = util.make_utterance(hp, t_x, seed=100 + t_x, sdp_ratio=0.2, length_scale=length_scale)
    ref, inter = util.oracle_run(oracle, u)
    audio, dur, f2p = run_gpu(model, u)
    check_alignment(oracle, u, inter, dur, f2p)
    err = np.abs(audio - ref[0, 0].numpy()).max()
    assert err <= WAVE_TOL, f"waveform max-abs {err:.3e}"


def test_golden_fixture(tiny):
    hp, oracle, model = tiny
    g = np.load(os.path.join(GOLDEN, "synth_tiny_tx23.npz"))
    u = util.make_utterance(hp, int(g["t_x"]), seed=int(g["input_seed"]), sdp_ratio=float(g["sdp_ratio"]))
    audio, dur, f2p = run_gpu(model, u)
    assert np.array_equal(dur, g["durations"])
    assert np.array_equal(f2p, g["frame2ph"])
    assert np.abs(audio - g["audio"]).max() <= WAVE_TOL


def test_batch_is_bit_identical_to_singles(full):
    """The reference is batch 1 (model.rs:66-79); the var-len batched extension must not change
    any utterance: waveforms, durations and alignment are compared bit for bit."""
    hp, oracle, model = full
    us = [util.make_utterance(hp, t, seed=200 + i, sdp_ratio=r, length_scale=ls)
          for i, (t, r, ls) in enumerate([(23, 0.0, 1.0), (151, 0.4, 1.0), (57, 0.0, 1.3), (5, 1.0, 0.8), (241, 0.2, 1.0)])]
    singles = [run_gpu(model, u) for u in us]
    audios, durs, f2ps = model.synthesize_batch([util.to_api(u) for u in us], want_alignment=True)
    for i in range(len(us)):
        assert np.array_equal(durs[i], singles[i][1])
        assert np.array_equal(f2ps[i], singles[i][2])
        assert audios[i].shape == singles[i][0].shape
        assert np.array_equal(audios[i], singles[i][0]), f"utterance {i} differs between batch and single run"


def test_alignment_properties_full_batch(full):
    """Size-independent properties at the benchmark's batch size (32 x ~8 s)."""
    hp, oracle, model = full
    us = [util.make_utterance(hp, 201 + 2 * (i % 41), seed=300 + i) for i in range(32)]
    audios, durs, f2ps = model.synthesize_batch([util.to_api(u) for u in us], want_alignment=True)
    audios2 = model.synthesize_batch([util.to_api(u) for u in us])
    for i, u in enumerate(us):
        d, f = durs[i], f2ps[i]
        assert (d >= 1).all()                      # exp(.) > 0 -> ceil >= 1
        assert d.sum() == len(f)                   # T_y = sum of durations
        assert (np.diff(f) >= 0).all()             # monotonic path
        assert np.array_equal(np.bincount(f, minlength=u["t_x"]), d)  # each phoneme owns exactly d frames
        assert audios[i].shape[0] == 512 * len(f)
        assert np.isfinite(audios[i]).all() and np.abs(audios[i]).max() <= 1.0
        assert np.array_equal(audios[i], audios2[i])  # deterministic with injected noise
    # every utterance of this batch is compared with the oracle in tests/test_gpu_fullsize.py
    # (test_cfg4_batch32_every_utterance_against_the_oracle)


def test_decoder_alone_cfg3_shape(full):
    """BASELINE config 3 (HiFi-GAN alone) at reduced length: z [B,192,T] -> waveform."""
    hp, oracle, model = full
    g = torch.Generator().manual_seed(31)
    zs = [torch.randn(192, t, generator=g) for t in (86, 33, 120, 1)]
    outs = model.decode_batch([z.numpy() for z in zs])
    spk = oracle.emb_g(torch.tensor([0])).unsqueeze(-1)
    for z, o in zip(zs, outs):
        with torch.no_grad():
            ref = oracle.dec(z.unsqueeze(0), g=spk)[0, 0].numpy()
        assert o.shape == ref.shape
        assert np.abs(o - ref).max() <= WAVE_TOL


def test_fp32_cuda_path_matches_oracle_tightly(S):
    """The CUDA-core fp32 kernels (selected with SBV2_B200_DECODER/FLOW/TEXT=fp32) reproduce the oracle
    to fp32 round-off; this separates kernel-logic errors from fp16 operand rounding."""
    hp = ov.HParams()
    oracle, onnx = util.synth_assets(hp, seed=0)
    os.environ["SBV2_B200_DECODER"] = "fp32"
    os.environ["SBV2_B200_FLOW"] = "fp32"
    os.environ["SBV2_B200_TEXT"] = "fp32"
    try:
        model = S.Model(onnx, bert=False)
    finally:
        del os.environ["SBV2_B200_DECODER"]
        del os.environ["SBV2_B200_FLOW"]
        del os.environ["SBV2_B200_TEXT"]
    u = util.make_utterance(hp, 61, seed=77, sdp_ratio=0.5)
    ref, inter = util.oracle_run(oracle, u)
    audio, dur, f2p = run_gpu(model, u)
    check_alignment(oracle, u, inter, dur, f2p)
    assert np.abs(audio - ref[0, 0].numpy()).max() <= 2e-5
    got_logw = model.debug_fetch("logw_dp")[:, 0]
    assert np.abs(got_logw - inter["logw_dp"][0, 0].numpy()).max() <= 2e-5


def test_wn_flow_variant(S):
    """north_star names the WN residual-coupling flow; JP-Extra uses the transformer flow by default
    (SURVEY.md D1).  Both are supported; the variant is inferred from the initializer names."""
    hp = ov.HParams(use_transformer_flow=False)
    oracle, onnx = util.synth_assets(hp, seed=3)
    model = S.Model(onnx, bert=False)
    assert model.describe()["use_transformer_flow"] is False and model.describe()["wn_layers"] == 4
    for t_x, seed in ((45, 5), (241, 6)):
        u = util.make_utterance(hp, t_x, seed=seed, sdp_ratio=0.3)
        ref, inter = util.oracle_run(oracle, u)
        audio, dur, f2p = run_gpu(model, u)
        check_alignment(oracle, u, inter, dur, f2p)
        err = np.abs(audio - ref[0, 0].numpy()).max()
        assert err <= WAVE_TOL, f"WN flow, T_x={t_x}: waveform max-abs {err:.3e}"
        # the flow output itself: z after the four coupling layers, against the oracle's
        z = model.debug_fetch("z")
        zr = inter["z"][0].numpy().T
        assert z.shape == zr.shape and np.abs(z - zr).max() <= 2e-2 and np.linalg.norm(z - zr) / np.linalg.norm(zr) <= 2e-3
    # tensor-core WN (gate fused into the in_layer conv's epilogue) vs the CUDA-core fp32 kernels of the same model, ragged batch
    os.environ["SBV2_B200_FLOW"] = "fp32"
    try:
        simt = S.Model(onnx, bert=False)
    finally:
        del os.environ["SBV2_B200_FLOW"]
    us = [util.to_api(util.make_utterance(hp, t, seed=40 + i, sdp_ratio=0.0)) for i, t in enumerate((33, 1, 131, 77))]
    a, da, fa = model.synthesize_batch(us, want_alignment=True)
    b, db_, fb = simt.synthesize_batch(us, want_alignment=True)
    for i in range(len(us)):
        assert np.array_equal(da[i], db_[i]) and np.array_equal(fa[i], fb[i])
        assert np.abs(a[i] - b[i]).max() <= WAVE_TOL
    singles = [model.synthesize_batch([u])[0] for u in us]
    for i in range(len(us)):
        assert np.array_equal(a[i], singles[i])          # batched == batch-1, bit for bit


def test_structural_binding_of_anonymous_weights(S):
    """Real exports constant-fold weight-normed convs to onnx::Conv_N names (SURVEY.md §A.7)."""
    from sbv2_b200 import assets
    hp = ov.tiny_hparams()
    oracle = ov.build_model(hp, seed=0)
    sd = ov.state_dict_numpy(oracle)
    named = S.Model(assets.synth_onnx(sd, hp.upsample_rates, hp.resblock_dilation_sizes), bert=False)
    anon = S.Model(assets.synth_onnx(sd, hp.upsample_rates, hp.resblock_dilation_sizes, anonymize_weight_norm=True), bert=False)
    assert anon.describe()["structural_binding"] is True and named.describe()["structural_binding"] is False
    u = util.make_utterance(hp, 31, seed=9)
    a, da, fa = run_gpu(named, u)
    b, db, fb = run_gpu(anon, u)
    assert np.array_equal(a, b) and np.array_equal(da, db) and np.array_equal(fa, fb)


def test_multi_speaker_and_sid(tiny):
    hp, oracle, model = tiny
    u0 = util.make_utterance(hp, 21, seed=4, sid=0)
    u1 = util.make_utterance(hp, 21, seed=4, sid=1)
    a0 = run_gpu(model, u0)[0]
    a1 = run_gpu(model, u1)[0]
    r1, _ = util.oracle_run(oracle, u1)
    assert not np.array_equal(a0[: min(len(a0), len(a1))], a1[: min(len(a0), len(a1))])
    assert np.abs(a1 - r1[0, 0].numpy()).max() <= WAVE_TOL


def test_error_paths(tiny, S):
    hp, oracle, model = tiny
    u = util.make_utterance(hp, 11, seed=1)
    api = util.to_api(u)
    bad = dict(api, x_tst=api["x_tst"].copy())
    bad["x_tst"][3] = hp.n_vocab
    with pytest.raises(S.Sbv2Error) as e:
        model.synthesize_batch([bad])
    assert e.value.status == S.ERR_INVALID_ARGUMENT
    with pytest.raises(S.Sbv2Error):
        model.synthesize_batch([dict(api, sid=hp.n_speakers)])
    short = dict(api, noise_zp=api["noise_zp"][:, :2])
    with pytest.raises(S.Sbv2Error) as e:
        model.synthesize_batch([short])
    assert "noise_zp" in e.value.message
    with pytest.raises(S.Sbv2Error):
        model.predict([1, 2, 3], [1, 1, 1])  # bert entry point on a synthesizer
    with pytest.raises(S.Sbv2Error):
        S.Model(b"\x08\x01", bert=False)  # a ModelProto without a graph
    from sbv2_b200 import assets
    with pytest.raises(S.Sbv2Error) as e:
        S.Model(assets.model_proto({"foo": np.zeros(4, np.float32)}), bert=False)
    assert e.value.status == S.ERR_UNSUPPORTED
    # 2201 phonemes at the 1e6-frame duration clamp: 2.2e9 frames, more than an int32 total (and 2^31 samples) can hold
    long = dict(util.to_api(util.make_utterance(hp, 2201, seed=5, max_frames=1)), length_scale=1e30, noise_zp=None)
    with pytest.raises(S.Sbv2Error) as e:
        model.synthesize_batch([long])
    assert e.value.status == S.ERR_INVALID_ARGUMENT and "too long" in e.value.message
    # the model is still usable after errors
    assert run_gpu(model, u)[0].size > 0


def test_zero_durations(full):
    """length_scale = 0: every duration is 0, T_y is clamped to 1 and that frame belongs to no phoneme (frame2ph -1); the
    oracle synthesizes it from m_p = logs_p = 0."""
    hp, oracle, model = full
    u = util.make_utterance(hp, 7, seed=17, sdp_ratio=0.4, length_scale=0.0)
    ref, inter = util.oracle_run(oracle, u)
    audio, dur, f2p = run_gpu(model, u)
    assert (dur == 0).all() and (inter["w_ceil"] == 0).all()
    assert np.array_equal(f2p, [-1])
    assert audio.shape[0] == ref.shape[-1] == 512
    err = np.abs(audio - ref[0, 0].numpy()).max()
    assert err <= WAVE_TOL, f"waveform max-abs {err:.3e}"


def test_internal_noise_is_seeded(tiny):
    hp, oracle, model = tiny
    u = util.make_utterance(hp, 15, seed=2, sdp_ratio=0.5)
    args = (u["bert"][0].numpy(), u["x"][0].numpy(), [0], u["tone"][0].numpy(), u["lang"][0].numpy(), u["style"][0].numpy(),
            0.5, 1.0, 0.677, 0.8)
    model.seed(42)
    a = model.synthesize(*args)
    model.seed(42)
    b = model.synthesize(*args)
    model.seed(43)
    c = model.synthesize(*args)
    assert a.shape[:2] == (1, 1) and np.array_equal(a, b)
    assert a.shape != c.shape or not np.array_equal(a, c)
    assert a.shape[2] % 512 == 0 and np.isfinite(a).all()


def test_programmatic_dependent_launch_does_not_change_results(S):
    """The tensor-core kernels are launched with programmatic stream serialization by default; SBV2_B200_PDL=0 launches
    them normally.  Same inputs and noise -> bit-identical audio and alignment."""
    hp = ov.HParams()
    oracle, onnx = util.synth_assets(hp, seed=0)
    u = util.make_utterance(hp, 45, seed=21, sdp_ratio=0.3)
    outs = []
    for pdl in ("1", "0"):
        os.environ["SBV2_B200_PDL"] = pdl
        try:
            model = S.Model(onnx, bert=False)
        finally:
            del os.environ["SBV2_B200_PDL"]
        outs.append(run_gpu(model, u))
        del model
    assert np.array_equal(outs[0][0], outs[1][0])
    assert np.array_equal(outs[0][1], outs[1][1]) and np.array_equal(outs[0][2], outs[1][2])
