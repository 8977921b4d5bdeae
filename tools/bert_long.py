"""Long-sentence DeBERTa timings (DeBERTa-v2-large shape, random weights).

  python tools/bert_long.py [--out FILE]

1. The whole forward, both numerics modes, S in {512, 1024, 2048, 4096} x batch {1, 4}: the "bert" region of the model's
   CUDA events (median of 5 calls after 2 warm-up calls).
2. The attention alone (one layer's launch, 16 heads) through sbv2_debug_deberta_attention, far-pair path on and off in
   the same process, alternating, each the mean of 20 launches timed with CUDA events, median of 5 alternations.
The card's name and power limit are printed first: the numbers belong to them."""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "sbv2-api_b200"))

import sbv2_b200 as S  # noqa: E402
from sbv2_b200 import assets  # noqa: E402
from oracle import deberta as od  # noqa: E402

SEQS, BATCHES, HEADS = (512, 1024, 2048, 4096), (1, 4), 16


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    emit(f"# card: {q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'}")
    if S.device_count() < 1:
        raise SystemExit("no GPU visible: nothing measured")
    cfg = od.deberta_config()
    onnx = assets.deberta_onnx(od.state_dict_numpy(od.build_model(cfg, seed=1)))
    emit("# whole forward, kernel ms ('bert' region events), median of 5 after 2 warm-up calls")
    emit("mode   batch x S      kernel_ms   tokens/s")
    for mode in ("exact", "fp16"):
        if mode == "fp16":
            os.environ["SBV2_B200_BERT"] = "fp16"
        try:
            model = S.Model(onnx, bert=True)
        finally:
            os.environ.pop("SBV2_B200_BERT", None)
        model.enable_timing(True)
        for s in SEQS:
            for b in BATCHES:
                ids = torch.randint(3, cfg.vocab_size, (b, s), generator=torch.Generator().manual_seed(s + b)).numpy()
                mask = np.ones_like(ids)
                ts = []
                for i in range(7):
                    model.predict_batch(ids, mask)
                    if i >= 2:
                        ts.append(model.region_ms("bert"))
                ms = float(np.median(ts))
                emit(f"{mode:6s} {b} x {s:5d}   {ms:10.2f}   {b * s / (ms * 1e-3):10.0f}")
        del model
    emit("# attention alone (one layer, 16 heads), ms per launch: far-pair path on / off, alternated, median of 5 x 20 launches")
    emit("kernel       batch x S   far_on_ms   far_off_ms   far_pairs/pairs")
    rng = np.random.default_rng(0)
    H = HEADS * 64
    pk, pq = (rng.standard_normal((512, H)) * 0.5 for _ in range(2))
    for kernel in ("exact-multi", "multi"):
        for s in SEQS:
            for b in BATCHES:
                lens = [s] * b
                x = rng.standard_normal((b * s, 3 * H))
                if kernel == "exact-multi":
                    split = lambda v: np.stack([(v * 16).astype(np.float16), (v * 16 - (v * 16).astype(np.float16)).astype(np.float16)])
                    ops = (split(x), split(pk), split(pq))
                else:
                    ops = (x.astype(np.float16), pk.astype(np.float16), pq.astype(np.float16))
                t = {True: [], False: []}
                for _ in range(5):
                    for far in (True, False):
                        t[far].append(S.debug_deberta_attention(*ops, lens, HEADS, kernel, far_pairs=far, reps=20)[1])
                nt = (s + 127) // 128
                nfar = sum(1 for a in range(nt) for c in range(nt) if abs(a - c) >= 5)
                emit(f"{kernel:11s} {b} x {s:5d}   {np.median(t[True]):9.3f}   {np.median(t[False]):10.3f}   {nfar}/{nt * nt}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
