"""GPU tests of Style-Bert-VITS2's assist text (sbv2_synthesize_from_tokens_assist, sbv2_holder_bert_features_assist,
sbv2_holder_easy_synthesize_tokens_assist): the device blend is bit-identical to the restated numerics
(tests/assist_oracle.py) over the documented DeBERTa batch layout [sentences..., used assists...], the host path equals
the device path, weight 0 is the old path, and the full-size chain agrees with upstream's loop fed by HF features."""
import time

import numpy as np
import pytest
import torch

import util
from assist_oracle import assist_features, restated_features
from oracle import deberta as od
from oracle import vits as ov

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def S(lib_built):
    import sbv2_b200
    if sbv2_b200.device_count() < 1:
        pytest.fail("GPU tests selected but no B200 is visible")
    return sbv2_b200


@pytest.fixture(scope="module")
def tiny(S):
    """tiny synthesizer (bert_dim 128) + tiny DeBERTa (hidden 128): -> (hp, oracle, synth onnx, cfg, bert onnx, synth, bert)"""
    from sbv2_b200 import assets
    hp = ov.tiny_hparams(bert_dim=128)
    oracle, onnx = util.synth_assets(hp, seed=0)
    cfg = od.tiny_config()
    bert_onnx = assets.deberta_onnx(od.state_dict_numpy(od.build_model(cfg, seed=1)))
    return hp, oracle, onnx, cfg, bert_onnx, S.Model(onnx, bert=False), S.Model(bert_onnx, bert=True)


def _sentence(hp, cfg, t_x, seed, **kw):
    w2p = util.word2ph_for(t_x, seed)
    ids = np.random.default_rng(seed).integers(3, cfg.vocab_size, size=w2p.size).astype(np.int64)
    x, tone, lang, _, style = ov.synthetic_inputs(hp, t_x, seed=seed)
    return dict(token_ids=ids, word2ph=w2p, x_tst=x[0].numpy(), tones=tone[0].numpy(), lang_ids=lang[0].numpy(),
                style_vec=style[0].numpy(), **kw)


def _assist(cfg, t_tok, seed, weight):
    ids = np.random.default_rng(seed).integers(3, cfg.vocab_size, size=t_tok).astype(np.int64)
    ids[0], ids[-1] = 1, 2  # CLS ... SEP
    return dict(token_ids=ids, weight=weight)


def _padded(rows):
    s = max(len(r) for r in rows)
    ids = np.zeros((len(rows), s), np.int64)
    mask = np.zeros((len(rows), s), np.int64)
    for b, r in enumerate(rows):
        ids[b, :len(r)] = r
        mask[b, :len(r)] = 1
    return ids, mask


def test_device_blend_is_bit_identical_to_the_restatement(S, tiny):
    hp, _, _, cfg, _, synth, bert = tiny
    A, B = _assist(cfg, 13, 1, 0.7), _assist(cfg, 27, 2, 1.0)
    sents = [_sentence(hp, cfg, t, 80 + i, assist=a) for i, (t, a) in enumerate(((19, 0), (25, None), (15, 1)))]
    synth.seed(1)
    audio, ns = synth.synthesize_from_tokens_batch(bert, sents, assists=[A, B])
    got = synth.debug_fetch("bert")                                   # [sum t_x, 128], the rows as gathered
    assert got.shape == (sum(s["x_tst"].size for s in sents), 128) and np.isfinite(audio).all()
    ids, mask = _padded([s["token_ids"] for s in sents] + [A["token_ids"], B["token_ids"]])   # [s0, s1, s2, A, B]
    feat = bert.predict_batch(ids, mask)
    a_rows = {0: feat[3, :A["token_ids"].size], 1: feat[4, :B["token_ids"].size]}
    off = 0
    for i, s in enumerate(sents):
        n = s["x_tst"].size
        t = s["token_ids"].size
        a = s["assist"]
        want = restated_features(feat[i, :t], a_rows[a] if a is not None else None, s["word2ph"],
                                 [A, B][a]["weight"] if a is not None else 0.0)
        assert np.array_equal(got[off:off + n].T, want), f"sentence {i}"
        if a is None:
            assert np.array_equal(got[off:off + n], np.repeat(feat[i, :t], s["word2ph"], axis=0))
        off += n


def test_holder_features_against_hf_and_the_restatement(S):
    from sbv2_b200 import assets
    cfg = od.deberta_config(hidden_size=1024, num_hidden_layers=3, num_attention_heads=16, intermediate_size=256, vocab_size=300)
    hf = od.build_model(cfg, seed=1)
    onnx = assets.deberta_onnx(od.state_dict_numpy(hf))
    h = S.TTSModelHolder(onnx, b"")
    bert = S.Model(onnx, bert=True)
    ids = np.array([1, 17, 33, 5, 250, 2], np.int64)
    word2ph = np.array([3, 4, 2, 0, 4, 2], np.int32)
    A = _assist(cfg, 11, 3, 0.7)
    got = h.bert_features(ids, np.ones_like(ids), word2ph, assist=A)
    res = od.predict(hf, torch.from_numpy(ids)[None], torch.ones(1, ids.size, dtype=torch.long))[0].numpy()
    style = od.predict(hf, torch.from_numpy(A["token_ids"])[None], torch.ones(1, A["token_ids"].size, dtype=torch.long))[0].numpy()
    want = assist_features(res, style, word2ph, float(np.float32(A["weight"])), torch.float64).numpy()
    assert got.shape == want.shape == (1024, int(word2ph.sum()))
    err = float(np.abs(got - want).max())
    print(f"holder bert_features with assist vs float64 blend of HF features: max-abs {err:.3e}")
    assert err <= 3e-2
    pid, pmask = _padded([ids, A["token_ids"]])
    feat = bert.predict_batch(pid, pmask)
    assert np.array_equal(got, restated_features(feat[0, :ids.size], feat[1, :A["token_ids"].size], word2ph, A["weight"]))
    # weight 0 is the plain path
    assert np.array_equal(h.bert_features(ids, np.ones_like(ids), word2ph, assist=dict(A, weight=0.0)),
                          h.bert_features(ids, np.ones_like(ids), word2ph))
    with pytest.raises(S.Sbv2Error) as e:
        h.bert_features(ids, np.ones_like(ids), word2ph, assist=dict(A, weight=float("nan")))
    assert e.value.status == S.ERR_INVALID_ARGUMENT
    h.close()


def test_host_path_equals_device_path(S, tiny):
    hp, _, onnx, cfg, bert_onnx, synth, bert = tiny
    from sbv2_b200 import assets
    h = S.TTSModelHolder(bert_onnx, b"")
    s = _sentence(hp, cfg, 31, 90)
    A = _assist(cfg, 17, 4, 0.7)
    feats = h.bert_features(s["token_ids"], np.ones_like(s["token_ids"]), s["word2ph"], assist=A)
    synth.seed(7)
    a = synth.synthesize(feats, s["x_tst"], [0], s["tones"], s["lang_ids"], s["style_vec"], 0.2, 1.0, 0.677, 0.8).reshape(-1)
    synth.seed(7)
    b, n = synth.synthesize_from_tokens_batch(bert, [dict(s, sdp_ratio=0.2, assist=0)], assists=[A])
    assert a.size == b.size == n[0] > 0
    assert np.array_equal(a, b)
    # the holder's easy_synthesize_tokens with the assist gives the durations of the host feature path (sdp_ratio 0)
    sv = np.random.default_rng(3).standard_normal((2, 256)).astype(np.float32) * 0.1
    h.load("m", assets.style_json(sv), onnx)
    line_tok = dict(token_ids=s["token_ids"], word2ph=s["word2ph"], phones=s["x_tst"], tones=s["tones"], lang_ids=s["lang_ids"])
    line_feat = dict(bert=feats, phones=s["x_tst"], tones=s["tones"], lang_ids=s["lang_ids"])
    wa = h.easy_synthesize("m", [line_feat], 1, 0)
    wb = h.easy_synthesize_tokens("m", [line_tok], 1, 0, assist=A)
    assert len(wa) == len(wb)
    h.close()


def test_weight_zero_is_the_old_path(S, tiny):
    hp, _, _, cfg, _, synth, bert = tiny
    sents = [_sentence(hp, cfg, t, 100 + i) for i, t in enumerate((21, 13))]
    A = _assist(cfg, 23, 5, 0.0)
    synth.seed(11)
    l0 = bert.launch_count
    ref, nr = synth.synthesize_from_tokens_batch(bert, sents, [100, 0])
    d_ref = bert.launch_count - l0
    synth.seed(11)
    l0 = bert.launch_count
    got, ng = synth.synthesize_from_tokens_batch(bert, [dict(s, assist=0) for s in sents], [100, 0], assists=[A])
    d_got = bert.launch_count - l0
    assert np.array_equal(ref, got) and np.array_equal(nr, ng)
    assert d_got == d_ref > 0, (d_got, d_ref)


def test_mixed_batch_equals_single_calls(S, tiny):
    hp, _, _, cfg, _, synth, bert = tiny
    A, B = _assist(cfg, 19, 6, 0.7), _assist(cfg, 9, 7, 1.0)
    sents = [_sentence(hp, cfg, t, 110 + i, assist=a) for i, (t, a) in enumerate(((19, 0), (7, None), (33, 1), (11, 0)))]
    singles = []
    for s in sents:
        synth.seed(5)
        singles.append(synth.synthesize_from_tokens_batch(bert, [s], assists=[A, B])[0])
    pauses = [22050, 0, 22050, 100]
    synth.seed(5)
    audio, ns = synth.synthesize_from_tokens_batch(bert, sents, pauses, assists=[A, B])
    assert [int(n) for n in ns] == [a.size for a in singles]
    assert audio.size == int(ns.sum()) + sum(pauses)
    off = 0
    for i, n in enumerate(ns):
        assert np.isfinite(audio[off:off + n]).all() and np.abs(audio[off:off + n]).max() > 1e-4
        off += int(n)
        assert not audio[off:off + pauses[i]].any()
        off += pauses[i]


def test_invalid_assists_are_rejected(S, tiny):
    hp, _, _, cfg, _, synth, bert = tiny
    s = _sentence(hp, cfg, 15, 120, assist=0)
    A = _assist(cfg, 10, 8, 0.5)
    bad = [[dict(A, weight=float("nan"))], [dict(A, weight=float("inf"))],
           [dict(A, attention_mask=np.array([1, 1, 0, 1, 1, 1, 1, 1, 1, 1], np.int64))],
           [dict(token_ids=np.arange(3, 3 + 32769) % 400 + 3, weight=0.5)], [dict(token_ids=np.zeros(0, np.int64), weight=0.5)]]
    for assists in bad:
        with pytest.raises(S.Sbv2Error) as e:
            synth.synthesize_from_tokens_batch(bert, [s], assists=assists)
        assert e.value.status == S.ERR_INVALID_ARGUMENT, e.value.message
    for k in (1, -2):
        with pytest.raises(S.Sbv2Error) as e:
            synth.synthesize_from_tokens_batch(bert, [dict(s, assist=k)], assists=[A])
        assert e.value.status == S.ERR_INVALID_ARGUMENT
    with pytest.raises(S.Sbv2Error):
        bert.synthesize_from_tokens_batch(synth, [s], assists=[A])
    synth.seed(3)
    audio, ns = synth.synthesize_from_tokens_batch(bert, [s], assists=[A])
    assert audio.size == ns[0] > 0 and np.isfinite(audio).all()


FEAT_TOL_EXACT = (6e-4, 1.5e-4)   # tests/test_gpu_fullsize.py FEAT_TOL["exact"]
WAVE_TOL = 1e-3


def test_fullsize_chain_with_assists_against_upstreams_loop(S):
    """32 cfg4-shaped utterances (DeBERTa-large shape, exact mode; T_x odd in 201..281), assists of 20-60 tokens with weights
    {0.3, 0.7, 1.0}.  GPU: one call of sbv2_synthesize_from_tokens_assist, its gathered features read back.  Oracle: HF fp32
    features -> upstream's loop in float64 -> fp32 -> oracle synthesizer.  Features within the exact mode's tolerance,
    durations equal except fp64-margin < 1e-4 ties (counted), waveforms of the first 4 matching utterances <= 1e-3."""
    from sbv2_b200 import assets
    t0 = time.time()
    hp = ov.HParams()
    oracle, onnx = util.synth_assets(hp, seed=0)
    synth = S.Model(onnx, bert=False)
    cfg = od.deberta_config()
    hf = od.build_model(cfg, seed=1)
    bert = S.Model(assets.deberta_onnx(od.state_dict_numpy(hf)), bert=True)
    assert bert.describe()["numerics"] == "exact"
    rng = np.random.default_rng(77)
    weights = (0.3, 0.7, 1.0)
    assists = []
    for k in range(6):
        ids = rng.integers(3, cfg.vocab_size, size=int(rng.integers(20, 61))).astype(np.int64)
        ids[0], ids[-1] = 1, 2
        assists.append(dict(token_ids=ids, weight=weights[k % 3]))
    specs, sents = [], []
    for i in range(32):
        t_x = int(rng.integers(100, 141)) * 2 + 1
        w2p = util.word2ph_for(t_x, seed=7700 + i)
        ids = rng.integers(3, cfg.vocab_size, size=w2p.size).astype(np.int64)
        a = None if i % 7 == 3 else i % len(assists)
        u = util.make_utterance(hp, t_x, seed=77000 + i, sdp_ratio=0.0 if i % 4 else 0.2)
        specs.append((u, w2p, ids, a))
        sents.append(dict(token_ids=ids, word2ph=w2p, x_tst=u["x"][0].numpy(), tones=u["tone"][0].numpy(), lang_ids=u["lang"][0].numpy(),
                          style_vec=u["style"][0].numpy(), sdp_ratio=u["sdp_ratio"], assist=a))
    audio, ns = synth.synthesize_from_tokens_batch(bert, sents, assists=assists)
    gathered = synth.debug_fetch("bert")
    assert np.isfinite(audio).all() and gathered.shape == (sum(u["t_x"] for u, *_ in specs), 1024)
    # ---- oracle features: HF fp32 per text, upstream's loop in float64
    def hf_rows(ids):
        return od.predict(hf, torch.from_numpy(ids)[None], torch.ones(1, ids.size, dtype=torch.long))[0].numpy()
    style_rows = [hf_rows(a["token_ids"]) for a in assists]
    feat_worst = [0.0, 0.0]
    utts_gpu, us_ref = [], []
    off = 0
    for u, w2p, ids, a in specs:
        res = hf_rows(ids)
        if a is None:
            ref = util.expand_features(res, w2p).astype(np.float64)
        else:
            ref = assist_features(res, style_rows[a], w2p, float(np.float32(assists[a]["weight"])), torch.float64).numpy()
        got = gathered[off:off + u["t_x"]].T
        off += u["t_x"]
        e = (float(np.abs(got - ref).max()), float(np.linalg.norm(got - ref) / np.linalg.norm(ref)))
        feat_worst = [max(feat_worst[0], e[0]), max(feat_worst[1], e[1])]
        us_ref.append(dict(u, bert=torch.from_numpy(ref.astype(np.float32)).unsqueeze(0)))
        utts_gpu.append(util.to_api(dict(u, bert=torch.from_numpy(np.ascontiguousarray(got)).unsqueeze(0))))
    # ---- durations and waveforms: the GPU synthesizer on the GPU's blended features vs the oracle chain (same noise)
    audios, durs, _ = synth.synthesize_batch(utts_gpu, want_alignment=True)
    flips = ties = total_ph = compared = 0
    worst_wave = 0.0
    for i, u_ref in enumerate(us_ref):
        o32 = util.oracle_durations(oracle, u_ref)
        bad = np.nonzero(durs[i] != o32["w_ceil"])[0]
        total_ph += len(durs[i])
        if bad.size:
            w64 = util.oracle_durations(oracle, u_ref, dtype=torch.float64)["w"]
            margin = np.abs(w64[bad] - np.round(w64[bad]))
            n_tie = int((margin < 1e-4).sum())
            ties += n_tie
            flips += int(bad.size) - n_tie
            if bad.size - n_tie:
                print(f"utterance {i}: duration flips at {bad.tolist()} fp64 margins {margin}")
        elif compared < 4:
            ref, _ = util.oracle_run(oracle, u_ref)
            err = float(np.abs(audios[i] - ref[0, 0].numpy()).max())
            worst_wave = max(worst_wave, err)
            compared += 1
            assert err <= WAVE_TOL, f"utterance {i}: waveform max-abs {err:.3e}"
        if specs[i][0]["sdp_ratio"] == 0.0:   # durations do not depend on the noise: the token call's lengths agree
            assert ns[i] == 512 * int(durs[i].sum())
    print(f"assist chain: 32 utterances, {total_ph} phonemes, blended features vs HF + float64 loop: max-abs {feat_worst[0]:.3e}, "
          f"rel-Frobenius {feat_worst[1]:.3e}; duration flips {flips}, fp64-margin ties {ties}; worst waveform max-abs "
          f"{worst_wave:.3e} over {compared} utterances ({time.time() - t0:.0f} s)")
    assert feat_worst[0] <= FEAT_TOL_EXACT[0] and feat_worst[1] <= FEAT_TOL_EXACT[1], feat_worst
    assert flips == 0
    assert compared == 4
