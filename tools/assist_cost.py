"""What Style-Bert-VITS2's assist text costs a request: wall-time p50 / p99 of TTSModelHolder.easy_synthesize_tokens
(DeBERTa-large shape in exact mode, the full-size JP-Extra synthesizer) for one sentence (T_tok ~ 40) and for 8 sentences,
each without an assist and with a 30-token assist at weight 0.7, plus the kernel launches of one call per model.
The assist adds its rows to the request's one DeBERTa batch and two small kernels (token mean, blended gather).
The card's name and power limit are printed first: the numbers belong to them.

  python tools/assist_cost.py [--calls 100] [--out profiles/assist_cost.log]
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
    cfg = od.deberta_config()
    bert_onnx = assets.deberta_onnx(od.state_dict_numpy(od.build_model(cfg, seed=1)))
    hp = ov.HParams()
    _, synth_onnx = util.synth_assets(hp, seed=0)
    sv = np.random.default_rng(3).standard_normal((2, 256)).astype(np.float32) * 0.1
    holder = S.TTSModelHolder(bert_onnx, b"")
    holder.load("m", assets.style_json(sv), synth_onnx)
    synth, bert = S.Model(synth_onnx, bert=False), S.Model(bert_onnx, bert=True)
    assert bert.describe()["numerics"] == "exact"
    rng = np.random.default_rng(5)

    def sentence(t_tok):
        w2p = np.concatenate([[1], rng.integers(2, 6, size=t_tok - 2), [1]]).astype(np.int32)  # ~3.5 phonemes per token
        w2p[1] += 1 - int(w2p.sum()) % 2  # odd T_x, as the frontend's blank interleave gives
        ids = rng.integers(3, cfg.vocab_size, size=t_tok).astype(np.int64)
        x, tone, lang, _, style = ov.synthetic_inputs(hp, int(w2p.sum()), seed=int(rng.integers(1 << 30)))
        return dict(token_ids=ids, word2ph=w2p, phones=x[0].numpy(), tones=tone[0].numpy(), lang_ids=lang[0].numpy(),
                    style_vec=style[0].numpy())

    a_ids = rng.integers(3, cfg.vocab_size, size=30).astype(np.int64)
    a_ids[0], a_ids[-1] = 1, 2
    assist = dict(token_ids=a_ids, weight=0.7)
    requests = {1: [sentence(40)], 8: [sentence(int(t)) for t in rng.integers(30, 51, size=8)]}
    emit(f"# easy_synthesize_tokens wall time over {args.calls} calls after 5 warm-up calls; assist: 30 tokens, weight 0.7")
    emit("sentences  T_tok  T_x    assist  p50_ms   p99_ms   bert_launches  synth_launches")
    for n, sents in requests.items():
        t_tok = sum(s["token_ids"].size for s in sents)
        t_x = sum(s["phones"].size for s in sents)
        for with_assist in (False, True):
            a = assist if with_assist else None
            for _ in range(5):
                holder.easy_synthesize_tokens("m", sents, 0, 0, assist=a)
            ts = []
            for _ in range(args.calls):
                t0 = time.perf_counter()
                holder.easy_synthesize_tokens("m", sents, 0, 0, assist=a)
                ts.append(time.perf_counter() - t0)
            ts = np.array(ts) * 1e3
            # launches of the same request through the model-level entry easy_synthesize_tokens calls
            api = [dict(s, x_tst=s["phones"], assist=0 if with_assist else None) for s in sents]
            synth.synthesize_from_tokens_batch(bert, api, assists=[assist] if with_assist else None)
            lb, ls = bert.launch_count, synth.launch_count
            synth.synthesize_from_tokens_batch(bert, api, assists=[assist] if with_assist else None)
            emit(f"{n:9d}  {t_tok:5d}  {t_x:5d}  {'yes' if with_assist else 'no':6s}  {np.median(ts):7.3f}  {np.percentile(ts, 99):7.3f}  "
                 f"{bert.launch_count - lb:13d}  {synth.launch_count - ls:14d}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
