"""GPU tests of phoneme durations in and out (include/sbv2_b200.h, "phoneme durations"): the timing queries return the
durations synthesis uses, synthesis at those durations reproduces the plain call bit for bit under the same generator
state, edited durations match the reference (tests/durations_oracle.py), mixed batches keep the batch-1 guarantee, the
holder reports where every phoneme lands in its WAV, and out-of-range durations are rejected before anything runs."""
import numpy as np
import pytest
import torch

import util
from durations_oracle import infer_with_durations
from oracle import deberta as od
from util import ov

pytestmark = pytest.mark.gpu

WAVE_TOL = 1e-3
HOP = 512


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
    assert model.describe()["hop"] == HOP
    return hp, oracle, model


@pytest.fixture(scope="module")
def tiny(S):
    """tiny synthesizer (bert_dim 128) + tiny DeBERTa: -> (hp, synth onnx, cfg, bert onnx, synth, bert)"""
    from sbv2_b200 import assets
    hp = ov.tiny_hparams(bert_dim=128)
    _, onnx = util.synth_assets(hp, seed=0)
    cfg = od.tiny_config()
    bert_onnx = assets.deberta_onnx(od.state_dict_numpy(od.build_model(cfg, seed=1)))
    return hp, onnx, cfg, bert_onnx, S.Model(onnx, bert=False), S.Model(bert_onnx, bert=True)


def _six(hp, sdp_ratio):
    return [util.make_utterance(hp, t, seed=500 + i, sdp_ratio=sdp_ratio, length_scale=ls)
            for i, (t, ls) in enumerate([(23, 1.0), (151, 1.0), (57, 1.3), (5, 0.8), (101, 1.0), (41, 0.9)])]


def _sentence(hp, cfg, t_x, seed, **kw):
    w2p = util.word2ph_for(t_x, seed)
    ids = np.random.default_rng(seed).integers(3, cfg.vocab_size, size=w2p.size).astype(np.int64)
    x, tone, lang, _, style = ov.synthetic_inputs(hp, t_x, seed=seed)
    return dict(token_ids=ids, word2ph=w2p, x_tst=x[0].numpy(), tones=tone[0].numpy(), lang_ids=lang[0].numpy(),
                style_vec=style[0].numpy(), **kw)


@pytest.mark.parametrize("sdp_ratio", [0.0, 0.4])
def test_query_equals_synthesis_and_the_oracle(full, sdp_ratio):
    hp, oracle, model = full
    us = _six(hp, sdp_ratio)
    api = [util.to_api(u) for u in us]
    q = model.predict_durations_batch(api)
    _, durs, _ = model.synthesize_batch(api, want_alignment=True)
    ties = 0
    for i, u in enumerate(us):
        assert np.array_equal(q[i], durs[i]), f"utterance {i}: query differs from synthesis"
        ref = util.oracle_durations(oracle, u)["w_ceil"]
        bad = np.nonzero(q[i] != ref)[0]
        if bad.size:
            w64 = util.oracle_durations(oracle, u, dtype=torch.float64)["w"]
            margin = np.abs(w64[bad] - np.round(w64[bad]))
            assert (margin < 1e-4).all(), f"utterance {i}: durations differ at {bad} with fp64 margins {margin}"
            ties += bad.size
    print(f"sdp_ratio {sdp_ratio}: query == synthesis for 6 utterances, {ties} fp64-margin ties against the oracle")


@pytest.mark.parametrize("sdp_ratio", [0.0, 0.4])
def test_round_trip_is_bit_exact(full, sdp_ratio):
    hp, _, model = full
    api = [util.to_api(u) for u in _six(hp, sdp_ratio)]
    d = model.predict_durations_batch(api)
    a0, d0, f0 = model.synthesize_batch(api, want_alignment=True)
    a1, d1, f1 = model.synthesize_batch_with_durations(api, d)
    for i in range(len(api)):
        assert np.array_equal(d1[i], d0[i]) and np.array_equal(f1[i], f0[i])
        assert np.array_equal(a1[i], a0[i]), f"utterance {i}"


def test_edited_durations_against_the_oracle(full):
    """Doubled and zeroed phonemes, an all-zero utterance and a ~60 s one: frame2ph equals the reference's attn.argmax,
    T_y = max(1, sum d), and the waveform is within 1e-3 of infer with w_ceil replaced by d."""
    hp, oracle, model = full
    us = [util.make_utterance(hp, t, seed=600 + i, sdp_ratio=0.4, length_scale=ls, max_frames=mf)
          for i, (t, ls, mf) in enumerate([(41, 1.0, 2000), (23, 1.0, 64), (151, 1.0, 5300), (9, 2.0, 400)])]
    api = [util.to_api(u) for u in us]
    pred = model.predict_durations_batch(api)
    d0 = pred[0].copy()
    d0[::3] *= 2
    d0[1::5] = 0
    d3 = pred[3].copy()
    d3[[0, 4]] = 0
    d3[2] += 7
    given = [d0, np.zeros(23, np.int32), np.full(151, 34, np.int32), d3]   # 151 x 34 frames = 59.6 s
    audios, durs, f2ps = model.synthesize_batch_with_durations(api, given)
    for i, (u, d) in enumerate(zip(us, given)):
        ty = max(1, int(d.sum()))
        assert np.array_equal(durs[i], d)
        assert len(f2ps[i]) == ty and audios[i].size == ty * HOP
        ref, gi = infer_with_durations(oracle, u, d)
        assert int(gi["y_lengths"][0]) == ty
        if d.sum() == 0:
            assert np.array_equal(f2ps[i], [-1])       # one frame from a zero prior mean and log-scale
        else:
            assert np.array_equal(f2ps[i], gi["attn"][0, 0].numpy().argmax(1).astype(np.int32))
        err = float(np.abs(audios[i] - ref[0, 0].numpy()).max())
        print(f"utterance {i}: T_y {ty}, waveform max-abs {err:.3e}")
        assert err <= WAVE_TOL, f"utterance {i}: waveform max-abs {err:.3e}"


def test_mixed_batch_equals_batch1_calls(full):
    hp, _, model = full
    us = [util.make_utterance(hp, t, seed=700 + i, sdp_ratio=r, max_frames=1500) for i, (t, r) in
          enumerate([(31, 0.4), (77, 0.0), (19, 0.4), (121, 0.2), (45, 0.0)])]
    api = [util.to_api(u) for u in us]
    pred = model.predict_durations_batch(api)
    given = [pred[0] + 1, None, np.maximum(pred[2] - 1, 0), None, pred[4] * 2]
    audios, durs, f2ps = model.synthesize_batch_with_durations(api, given)
    for i, u in enumerate(api):
        if given[i] is None:
            a1, d1, f1 = model.synthesize_batch([u], want_alignment=True)
            assert np.array_equal(durs[i], pred[i])
        else:
            a1, d1, f1 = model.synthesize_batch_with_durations([u], [given[i]])
        assert np.array_equal(durs[i], d1[0]) and np.array_equal(f2ps[i], f1[0])
        assert np.array_equal(audios[i], a1[0]), f"utterance {i} ({'given' if given[i] is not None else 'predicted'})"


def test_token_path_round_trip_with_the_internal_generator(S, tiny):
    hp, _, cfg, _, synth, bert = tiny
    ids = np.random.default_rng(9).integers(3, cfg.vocab_size, size=14).astype(np.int64)
    ids[0], ids[-1] = 1, 2
    assists = [dict(token_ids=ids, weight=0.7)]
    sents = [_sentence(hp, cfg, t, 800 + i, sdp_ratio=r, assist=a) for i, (t, r, a) in
             enumerate([(19, 0.4, None), (33, 0.0, 0), (11, 0.4, None), (27, 0.0, None)])]
    pauses = [22050, 0, 300, 0]
    tx = [s["x_tst"].size for s in sents]

    def launches(fn):
        l0 = synth.launch_count
        r = fn()
        return r, synth.launch_count - l0

    synth.seed(21)
    (a_plain, n_plain), l_plain = launches(lambda: synth.synthesize_from_tokens_batch(bert, sents, pauses, assists=assists))
    synth.seed(21)
    D, l_query = launches(lambda: synth.predict_durations_from_tokens(bert, sents, assists=assists))
    assert [d.size for d in D] == tx
    synth.seed(21)
    (a_timed, n_timed, d_used), l_timed = launches(
        lambda: synth.synthesize_from_tokens_with_durations(bert, sents, D, pauses, assists=assists))
    assert np.array_equal(a_timed, a_plain) and np.array_equal(n_timed, n_plain)
    assert all(np.array_equal(a, b) for a, b in zip(d_used, D))
    assert list(n_plain) == [HOP * max(1, int(d.sum())) for d in D]
    # a mixed call launches what the plain call launches (the ingest kernel replaces the durations kernel) and gives the
    # same audio; the all-given call launches neither the DP nor the SDP
    synth.seed(21)
    (a_mixed, _, _), l_mixed = launches(
        lambda: synth.synthesize_from_tokens_with_durations(bert, sents, [D[0], None, D[2], None], pauses, assists=assists))
    assert np.array_equal(a_mixed, a_plain) and l_mixed == l_plain
    nosdp = [dict(s, sdp_ratio=0.0) for s in sents]
    _, l_plain_nosdp = launches(lambda: synth.synthesize_from_tokens_batch(bert, nosdp, pauses, assists=assists))
    _, l_timed_nosdp = launches(lambda: synth.synthesize_from_tokens_with_durations(bert, nosdp, D, pauses, assists=assists))
    n_sdp = l_plain - l_plain_nosdp
    n_dp = l_plain_nosdp - l_timed_nosdp
    assert n_sdp > 0 and n_dp >= 7     # DP: cond, add, conv_1, norm_1, conv_2, norm_2, proj
    assert l_timed == l_timed_nosdp == l_plain - n_sdp - n_dp
    print(f"token path launches: plain {l_plain}, query {l_query}, all given {l_timed} (DP {n_dp}, SDP {n_sdp} not launched)")


def test_query_is_cheap(full):
    hp, _, model = full
    x, tone, lang, bert, style = ov.synthetic_inputs(hp, 151, 77)   # bench.py's latency utterance
    u = dict(bert=bert[0].numpy(), x_tst=x[0].numpy(), tones=tone[0].numpy(), lang_ids=lang[0].numpy(), style_vec=style[0].numpy())
    model.synthesize_batch([u])
    l0 = model.launch_count
    model.synthesize_batch([u])
    l_plain = model.launch_count - l0
    l0 = model.launch_count
    model.predict_durations_batch([u])
    l_query = model.launch_count - l0
    print(f"one ~5 s utterance (T_x = 151): plain call {l_plain} launches, timing query {l_query}")
    assert l_query < 0.5 * l_plain


def _wav_samples(wav: bytes) -> np.ndarray:
    i = wav.index(b"data")
    n = int.from_bytes(wav[i + 4:i + 8], "little")
    return np.frombuffer(wav[i + 8:i + 8 + n], dtype=np.float32)


def test_holder_timing(S, tiny):
    from sbv2_b200 import assets
    hp, onnx, cfg, bert_onnx, _, _ = tiny
    sv = np.random.default_rng(3).standard_normal((2, 256)).astype(np.float32) * 0.1
    h = S.TTSModelHolder(bert_onnx, b"")

    def fresh():   # the voice's generator back to its creation state
        h.unload("m")
        h.load("m", assets.style_json(sv), onnx)

    lines = []
    for i, t in enumerate((21, None, 35, 13)):
        if t is None:
            lines.append(None)
            continue
        s = _sentence(hp, cfg, t, 900 + i)
        lines.append(dict(token_ids=s["token_ids"], word2ph=s["word2ph"], phones=s["x_tst"], tones=s["tones"], lang_ids=s["lang_ids"]))
    kw = dict(sdp_ratio=0.4, length_scale=1.1)
    fresh()
    w_plain = h.easy_synthesize_tokens("m", lines, 1, 0, **kw)
    fresh()
    w_timed, d_timed, starts = h.easy_synthesize_tokens_timed("m", lines, 1, 0, **kw)
    assert w_timed == w_plain
    fresh()
    d_query = h.predict_durations_tokens("m", lines, 1, 0, **kw)
    assert all(np.array_equal(a, b) for a, b in zip(d_query, d_timed))
    fresh()
    w_given, d_given, starts_given = h.easy_synthesize_tokens_timed("m", lines, 1, 0, durations=d_query, **kw)
    assert w_given == w_plain
    assert all(np.array_equal(a, b) for a, b in zip(d_given, d_query))
    assert all(np.array_equal(a, b) for a, b in zip(starts_given, starts))
    samples = _wav_samples(w_plain)
    pauses = [22050, 22050, 0]   # after every line but the last one of the text
    pos = 0
    for k, (d, st) in enumerate(zip(d_timed, starts)):
        assert st[0] == pos
        assert np.array_equal(np.diff(st), d[:-1].astype(np.int64) * HOP)
        n = HOP * max(1, int(d.sum()))
        assert np.abs(samples[pos:pos + n]).max() > 0
        assert not samples[pos + n:pos + n + pauses[k]].any()
        pos += n + pauses[k]
    assert pos == samples.size
    h.close()


def test_invalid_durations_are_rejected(S, full):
    hp, _, model = full
    u = util.to_api(util.make_utterance(hp, 9, seed=950))
    bad = [np.array([3, 2, -1, 4, 1, 1, 2, 2, 1]), np.array([3, 2, 1, 1_000_001, 1, 1, 2, 2, 1]),
           np.full(9, 1_000_000)]   # 9e6 frames * 512 samples > 2^31
    for d in bad:
        with pytest.raises(S.Sbv2Error) as e:
            model.synthesize_batch_with_durations([u], [d])
        assert e.value.status == S.ERR_INVALID_ARGUMENT and e.value.message, e.value.message
        print(e.value.message)
    audios, durs, f2ps = model.synthesize_batch_with_durations([u], [np.full(9, 5)])
    assert audios[0].size == 45 * HOP and np.isfinite(audios[0]).all() and np.array_equal(durs[0], np.full(9, 5))


def test_token_path_rejects_before_launching(S, tiny):
    hp, _, cfg, _, synth, bert = tiny
    sents = [_sentence(hp, cfg, t, 960 + i) for i, t in enumerate((13, 9))]
    lb, ls = bert.launch_count, synth.launch_count
    with pytest.raises(S.Sbv2Error) as e:
        synth.synthesize_from_tokens_with_durations(bert, sents, [None, np.array([1, 2, 3, 1_000_001, 1, 1, 1, 1, 1])])
    assert e.value.status == S.ERR_INVALID_ARGUMENT
    assert bert.launch_count == lb and synth.launch_count == ls   # DeBERTa did not run either
    audio, ns, d = synth.synthesize_from_tokens_with_durations(bert, sents, [None, np.full(9, 2)])
    assert ns[1] == 18 * HOP and np.array_equal(d[1], np.full(9, 2)) and np.isfinite(audio).all()
