"""What a timing query and synthesis at given durations cost: wall-time p50 / p99 and kernel launches of the plain call,
the timing query and the timed call (all durations given) for
  - one ~5 s utterance (bench.py's latency utterance, T_x = 151): sbv2_synthesize_batch, sbv2_predict_durations_batch,
    sbv2_synthesize_batch_with_durations;
  - an 8-sentence request through DeBERTa-large (exact mode) and the full-size synthesizer:
    sbv2_synthesize_from_tokens_batch, sbv2_predict_durations_from_tokens, sbv2_synthesize_from_tokens_with_durations.
The card's name and power limit are printed first: the numbers belong to them.

  python tools/durations_cost.py [--calls 100] [--out profiles/durations_cost.log]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "sbv2-api_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import util  # noqa: E402
from oracle import deberta as od  # noqa: E402
from oracle import vits as ov  # noqa: E402
import sbv2_b200 as S  # noqa: E402
from sbv2_b200 import assets  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True)
        card = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"
    except OSError:
        card = "unknown (nvidia-smi not found)"
    emit(f"# card (name, power limit, max SM clock): {card}")
    if S.device_count() < 1:
        raise SystemExit("no GPU visible: nothing measured")
    hp = ov.HParams()
    _, synth_onnx = util.synth_assets(hp, seed=0)
    synth = S.Model(synth_onnx, bert=False)
    cfg = od.deberta_config()
    bert = S.Model(assets.deberta_onnx(od.state_dict_numpy(od.build_model(cfg, seed=1))), bert=True)
    assert bert.describe()["numerics"] == "exact"

    def measure(fn):
        for _ in range(5):
            fn()
        ts = []
        for _ in range(args.calls):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e3
        l0 = synth.launch_count
        fn()
        return np.median(ts), np.percentile(ts, 99), synth.launch_count - l0

    emit(f"# wall time over {args.calls} calls after 5 warm-up calls; launches of the synthesizer model per call")
    emit("request                         call      p50_ms   p99_ms   synth_launches")

    x, tone, lang, feat, style = ov.synthetic_inputs(hp, 151, 77)   # bench.py's latency utterance
    u = dict(bert=S.pinned_copy(feat[0].numpy()), x_tst=x[0].numpy(), tones=tone[0].numpy(), lang_ids=lang[0].numpy(),
             style_vec=style[0].numpy())
    d = synth.predict_durations_batch([u])
    for name, fn in (("plain", lambda: synth.synthesize_batch([u])), ("query", lambda: synth.predict_durations_batch([u])),
                     ("timed", lambda: synth.synthesize_batch_with_durations([u], d))):
        p50, p99, nl = measure(fn)
        emit(f"{'1 x T_x 151 (~5 s)':30s}  {name:8s}  {p50:7.3f}  {p99:7.3f}  {nl:14d}")

    rng = np.random.default_rng(5)
    sents = []
    for t_tok in rng.integers(30, 51, size=8):
        w2p = np.concatenate([[1], rng.integers(2, 6, size=int(t_tok) - 2), [1]]).astype(np.int32)
        w2p[1] += 1 - int(w2p.sum()) % 2
        ids = rng.integers(3, cfg.vocab_size, size=int(t_tok)).astype(np.int64)
        x, tone, lang, _, style = ov.synthetic_inputs(hp, int(w2p.sum()), seed=int(rng.integers(1 << 30)))
        sents.append(dict(token_ids=ids, word2ph=w2p, x_tst=x[0].numpy(), tones=tone[0].numpy(), lang_ids=lang[0].numpy(),
                          style_vec=style[0].numpy()))
    pauses = [22050] * 7 + [0]
    t_x = sum(s["x_tst"].size for s in sents)
    dt = synth.predict_durations_from_tokens(bert, sents)
    label = f"8 sentences, T_x {t_x}"
    for name, fn in (("plain", lambda: synth.synthesize_from_tokens_batch(bert, sents, pauses)),
                     ("query", lambda: synth.predict_durations_from_tokens(bert, sents)),
                     ("timed", lambda: synth.synthesize_from_tokens_with_durations(bert, sents, dt, pauses))):
        p50, p99, nl = measure(fn)
        emit(f"{label:30s}  {name:8s}  {p50:7.3f}  {p99:7.3f}  {nl:14d}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
