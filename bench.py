#!/usr/bin/env python
"""Benchmark of the synthesis hot path (BASELINE.json metric: audio-sec/sec, JP-Extra 44.1 kHz,
batch 32 per GPU; p50 latency of a 5 s utterance).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the full JP-Extra synthesizer (enc_p, duration predictors, length
regulator, flow, HiFi-GAN decoder) over one batch of 32 synthetic ~8 s utterances (BASELINE config 4
per-GPU shard: T_x odd in U{201..281}, BERT features given, sdp_ratio 0, device-side noise).
Weak scaling: every rank owns a model replica and its own batch, no collective on the data path.

  value : audio-seconds per second with the step's inputs already resident in HBM, timed with CUDA
          events on the models' streams, max over ranks (--e2e-replicas model replicas per GPU on their own
          streams; `single_stream` repeats it with ONE replica / ONE stream).
  e2e   : the same metric through the C-ABI call a user makes (`sbv2_synthesize_batch`): host
          buffers in (page-locked, as the bench contract prescribes), waveforms in pinned host
          memory out, all copies inside the timed region.
  latency : p50 / p99 wall time of ONE ~5 s utterance, batch 1, through `sbv2_synthesize`
          (host in -> host out) — the reference's production call (model.rs:53-111, main.rs:86).
  roofline : HiFi-GAN decoder (tcgen05 implicit-GEMM convs), algorithmic FLOPs per step
          (651.6 MFLOP per latent frame, SURVEY.md §8d) / measured decoder time.
  configs : the other BASELINE.json configurations on rank 0 (cfg1 short utterance, cfg2 DeBERTa 32x128 in
          both numerics modes, cfg3 decoder alone 32x861, cfg5 one 60 s utterance).
  cpu_baseline : the reference's CPU path timed on the host cores on a bounded sample of the same
          batch: ONNX Runtime with the reference's session options if `onnxruntime` is importable and the
          graph can be exported here (probed at run time), else the PyTorch-CPU restatement (kind "port").
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "sbv2-api_b200"))

SR = 44100
BATCH = 32
DEC_FLOP_PER_FRAME = 651.6e6   # SURVEY.md §8d / §C.1 (flop-counter verified)
BERT_FLOP_PER_TOKEN = 0.605e9  # SURVEY.md §8d: 22 live layers of deberta-v2-large


def make_batch(hp, batch: int, seed: int):
    """cfg4 per-GPU shard: T_x odd ~ U{201..281}; synthetic ids / BERT features / style."""
    from oracle import vits as ov
    rng = np.random.default_rng(seed)
    utts, raw = [], []
    for i in range(batch):
        t_x = int(rng.integers(100, 141)) * 2 + 1
        x, tone, lang, bert, style = ov.synthetic_inputs(hp, t_x, seed * 1000 + i)
        raw.append((x, tone, lang, bert, style, t_x))
        utts.append(dict(bert=bert[0].numpy(), x_tst=x[0].numpy(), tones=tone[0].numpy(), lang_ids=lang[0].numpy(),
                         style_vec=style[0].numpy(), sid=0, sdp_ratio=0.0, length_scale=1.0, noise_scale=0.677,
                         noise_scale_w=0.8))
    return utts, raw


def one_utt(hp, t_x, seed):
    from oracle import vits as ov
    x, tone, lang, bert, style = ov.synthetic_inputs(hp, t_x, seed)
    return dict(bert=bert[0].numpy(), x_tst=x[0].numpy(), tones=tone[0].numpy(), lang_ids=lang[0].numpy(), style_vec=style[0].numpy(),
                sid=0, sdp_ratio=0.0, length_scale=1.0, noise_scale=0.677, noise_scale_w=0.8)


class ClockSampler:
    """nvidia-smi in loop mode (-lms 100) for the duration of the timed region, as the profiling recipe does."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw"

    def __init__(self, index: int):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
        time.sleep(0.15)

    def stop(self):
        rows = []
        if self.proc is not None:
            time.sleep(0.12)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            rows = [[c.strip() for c in line.split(",")] for line in out.splitlines() if line.strip()]
        num = lambda x: x.replace(".", "", 1).isdigit()
        sm = [float(r[0]) for r in rows if r and num(r[0])]
        mx = [float(r[1]) for r in rows if len(r) > 1 and num(r[1])]
        pw = [float(r[6]) for r in rows if len(r) > 6 and num(r[6])]
        reasons = []
        for name, col in (("hw_slowdown", 2), ("hw_thermal_slowdown", 3), ("sw_thermal_slowdown", 4), ("sw_power_cap", 5)):
            if any(len(r) > col and r[col].lower().startswith("active") for r in rows):
                reasons.append(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(rows)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs
# ---------------------------------------------------------------------------------------------------------------------
def try_ort_session(model, hp, threads: int):
    """ONNX Runtime CPU with the reference's session options (crates/sbv2_core/src/model.rs:43-49: graph optimisation level
    3, intra- and inter-op threads = physical cores).  Needs `onnxruntime` AND an exportable graph (`onnx` for
    torch.onnx.export); neither ships in the offline image, so this normally returns (None, reason)."""
    try:
        import onnxruntime as ort  # noqa: F401
    except Exception as e:  # noqa: BLE001
        return None, f"onnxruntime not importable ({type(e).__name__})"
    try:
        import io
        import torch

        class Wrap(torch.nn.Module):  # scripts/convert/convert_model.py:97-110 (argument order as exported)
            def __init__(self, m):
                super().__init__()
                self.m = m

            def forward(self, x, xl, sid, tone, lang, bert, style, length_scale, sdp_ratio, noise_scale, noise_scale_w):
                t = x.shape[1]
                return self.m.infer(x, xl, sid, tone, lang, bert, style, noise_sdp=torch.randn(1, 2, t),
                                    noise_zp=lambda b, c, n: torch.randn(b, c, n), noise_scale=noise_scale, length_scale=length_scale,
                                    noise_scale_w=noise_scale_w, sdp_ratio=sdp_ratio)
        from oracle import vits as ov
        x, tone, lang, bert, style = ov.synthetic_inputs(hp, 31, 1)
        buf = io.BytesIO()
        torch.onnx.export(Wrap(model), (x, torch.tensor([31]), torch.tensor([0]), tone, lang, bert, style, torch.tensor(1.0),
                                        torch.tensor(0.0), torch.tensor(0.677), torch.tensor(0.8)), buf,
                          input_names=["x_tst", "x_tst_lengths", "sid", "tones", "language", "bert", "style_vec", "length_scale",
                                       "sdp_ratio", "noise_scale", "noise_scale_w"], output_names=["output"],
                          dynamic_axes={"x_tst": {1: "t"}, "tones": {1: "t"}, "language": {1: "t"}, "bert": {2: "t"}})
        so = ort.SessionOptions()
        so.graph_optimization_level = ort.GraphOptimizationLevel.ORT_ENABLE_ALL
        so.intra_op_num_threads = threads
        so.inter_op_num_threads = threads
        return ort.InferenceSession(buf.getvalue(), so, providers=["CPUExecutionProvider"]), "onnxruntime " + ort.__version__
    except Exception as e:  # noqa: BLE001
        return None, f"onnxruntime importable but the graph could not be exported/loaded here ({type(e).__name__}: {str(e)[:80]})"


def cpu_rate(model, hp, raw, n_utts: int, threads: int):
    """audio-sec/sec of the reference's CPU path, batch 1 per utterance like the reference (model.rs:66-79).
    -> (rate, audio_s, seconds, kind, note)"""
    import torch
    torch.set_num_threads(threads)
    sess, note = try_ort_session(model, hp, threads)
    g = torch.Generator().manual_seed(7)
    audio_s, t0 = 0.0, None
    for i in range(n_utts + 1):  # the first call is an untimed warm-up
        x, tone, lang, bert, style, t_x = raw[i % len(raw)]
        if i == 1:
            t0 = time.perf_counter()
            audio_s = 0.0
        if sess is not None:
            o = sess.run(["output"], {"x_tst": x.numpy(), "x_tst_lengths": np.array([t_x], np.int64), "sid": np.array([0], np.int64),
                                      "tones": tone.numpy(), "language": lang.numpy(), "bert": bert.numpy(), "style_vec": style.numpy(),
                                      "length_scale": np.array(1.0, np.float32), "sdp_ratio": np.array(0.0, np.float32),
                                      "noise_scale": np.array(0.677, np.float32), "noise_scale_w": np.array(0.8, np.float32)})[0]
        else:
            nsdp = torch.randn(1, 2, t_x, generator=g)
            o = model.infer(x, torch.tensor([t_x]), torch.tensor([0]), tone, lang, bert, style, noise_sdp=nsdp,
                            noise_zp=lambda b, c, t: torch.randn(b, c, t, generator=g), noise_scale=0.677, length_scale=1.0,
                            noise_scale_w=0.8, sdp_ratio=0.0)
        audio_s += o.shape[-1] / SR
    dt = time.perf_counter() - t0
    kind = "reference" if sess is not None else "port"
    return audio_s / dt, audio_s, dt, kind, note


def sources_digest() -> str:
    """sha1 over the CUDA sources: ties the committed ncu traffic figure to the kernels it was measured on."""
    h = hashlib.sha1()
    d = os.path.join(ROOT, "sbv2-api_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.startswith("umma_") and f.endswith((".cu", ".cuh", ".h")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()


DUMP_LIMIT = 64 << 20  # bytes written by --dump-outputs


def dump_outputs(out_dir: str, waves, suffix: str = "") -> None:
    """Writes one batch's waveforms as sbv2_batch_download hands them to its caller: the samples of every utterance back to
    back (audio, float32) and the samples per utterance (audio_lengths, float64).  Past DUMP_LIMIT bytes, audio keeps a fixed,
    seeded sample of the samples, in order, and audio_index (float64) gives their positions."""
    os.makedirs(out_dir, exist_ok=True)
    audio = np.concatenate(waves).astype(np.float32, copy=False)
    arrays = {"audio_lengths": np.array([w.size for w in waves], np.float64)}
    if audio.nbytes + arrays["audio_lengths"].nbytes > DUMP_LIMIT:
        k = (DUMP_LIMIT - arrays["audio_lengths"].nbytes - 1024) // 12  # 4 B per sample + 8 B per index; 1 KB for the headers
        idx = np.sort(np.random.default_rng(0).choice(audio.size, size=k, replace=False))
        arrays["audio_index"] = idx.astype(np.float64)
        audio = audio[idx]
    arrays["audio"] = audio
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def wall(fn, n, warm=3):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n):
        t = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t)
    return np.array(ts)


def other_configs(S, assets, ov, hp, oracle, model, peak_tf, which):
    """BASELINE.json configs 1, 2, 3, 5 on this GPU (rank 0 only; the headline is config 4)."""
    import torch
    out = {}
    if "cfg1" in which:
        u = one_utt(hp, 23, 12)
        ts = wall(lambda: model.synthesize_batch([u]), 30)
        n = model.synthesize_batch([u])[0].size
        out["cfg1"] = {"what": "one short utterance T_x=23, batch 1, host in -> host out", "audio_s": n / SR,
                       "latency_ms_p50": float(np.median(ts) * 1e3), "latency_ms_p99": float(np.percentile(ts, 99) * 1e3)}
    if "cfg5" in which:
        u = one_utt(hp, 1801, 51)
        ts = wall(lambda: model.synthesize_batch([u]), 8, warm=2)
        n = model.synthesize_batch([u])[0].size
        out["cfg5"] = {"what": "one long-form utterance T_x=1801 (~60 s), batch 1, host in -> host out", "audio_s": n / SR,
                       "latency_ms_p50": float(np.median(ts) * 1e3), "audio_s_per_s": n / SR / float(np.median(ts))}
    if "cfg3" in which:
        g = torch.Generator().manual_seed(31)
        zs = [S.pinned_copy(torch.randn(192, 861, generator=g).numpy()) for _ in range(32)]
        model.enable_timing(True)
        ts = wall(lambda: model.decode_batch(zs), 5, warm=2)
        dec_ms = model.region_ms("decoder")
        model.enable_timing(False)
        audio_s = 32 * 861 * 512 / SR
        tf = DEC_FLOP_PER_FRAME * 32 * 861 / (dec_ms * 1e-3) / 1e12
        out["cfg3"] = {"what": "HiFi-GAN decoder alone, 32 x 861 frames (10 s)", "audio_s": audio_s, "decoder_ms": dec_ms, "tflops": tf,
                       "frac_of_peak": tf / peak_tf, "audio_s_per_s_kernel": audio_s / (dec_ms * 1e-3),
                       "audio_s_per_s_e2e": audio_s / float(np.median(ts))}
        del zs
    if "cfg2" in which:
        from oracle import deberta as od
        cfg = od.deberta_config()
        onnx = assets.deberta_onnx(od.state_dict_numpy(od.build_model(cfg, seed=1)))
        ids = torch.randint(3, cfg.vocab_size, (32, 128), generator=torch.Generator().manual_seed(21)).numpy()
        mask = np.ones_like(ids)
        res = {"what": "DeBERTa-v2-large shape (22 live layers), batch 32 x seq 128; exact = two-term fp16 splits (default, "
                       "duration-exact downstream), fp16 = single-term operands (SBV2_B200_BERT=fp16)"}
        for mode in ("exact", "fp16"):
            if mode == "fp16":
                os.environ["SBV2_B200_BERT"] = "fp16"
            try:
                bert = S.Model(onnx, bert=True)
            finally:
                os.environ.pop("SBV2_B200_BERT", None)
            bert.enable_timing(True)
            ts = wall(lambda: bert.predict_batch(ids, mask), 8, warm=3)
            k_ms = bert.region_ms("bert")
            t1 = wall(lambda: bert.predict(ids[0, :7], np.ones(7, np.int64)), 20)
            mul = 3.0 if mode == "exact" else 1.0  # tensor FLOPs issued per algorithmic FLOP
            res[mode] = {"kernel_ms": k_ms, "e2e_ms": float(np.median(ts) * 1e3), "tokens_per_s": 4096 / (k_ms * 1e-3),
                         "algorithmic_tflops": BERT_FLOP_PER_TOKEN * 4096 / (k_ms * 1e-3) / 1e12,
                         "issued_tflops": mul * BERT_FLOP_PER_TOKEN * 4096 / (k_ms * 1e-3) / 1e12,
                         "frac_of_peak_issued": mul * BERT_FLOP_PER_TOKEN * 4096 / (k_ms * 1e-3) / 1e12 / peak_tf,
                         "latency_ms_T_tok_7": float(np.median(t1) * 1e3)}
            del bert
        out["cfg2"] = res
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--configs", default="cfg1,cfg2,cfg3,cfg5", help="other BASELINE configs measured on rank 0 ('' = none)")
    ap.add_argument("--e2e-replicas", type=int, default=3,
                    help="model replicas per GPU driven by separate host threads: the synchronous call's H2D / T_y read-back / D2H "
                         "phases of one replica overlap the kernels of the others (measured 1/2/3 replicas: 8.2k/8.3k/8.9k audio-s/s, "
                         "profiles/r2_e2e_replicas.log)")
    ap.add_argument("--tiny", action="store_true", help="reduced model (tests only; not a benchmark configuration)")
    ap.add_argument("--flow", default="transformer", choices=["transformer", "wn"],
                    help="flow variant of the synthetic model: JP-Extra's transformer coupling layers (the headline) or the WN "
                         "residual-coupling layers north_star names (non-JP-Extra Style-Bert-VITS2 models)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the waveforms of the last timed batch of replica 0 to DIR as .npy "
                         "(see dump_outputs); the same arguments give the same inputs, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    threads = os.cpu_count() or 1

    import torch
    from oracle import vits as ov

    flow_kw = {} if args.flow == "transformer" else {"use_transformer_flow": False}
    hp = ov.tiny_hparams(**flow_kw) if args.tiny else ov.HParams(**flow_kw)
    workload = f"cfg4 shard: full JP-Extra pipeline, {args.batch} synthetic ~8 s utterances per GPU per step " \
               f"(T_x odd U{{201..281}}, BERT features given, sdp_ratio 0, " + \
               ("transformer flow L=6)" if args.flow == "transformer" else "WN residual-coupling flow, 4 x 4 layers)")

    # ------------------------------------------------------------------ reference arm (the reference's CPU path)
    if args.impl == "reference":
        if rank != 0:
            return
        model = ov.build_model(hp, seed=0)
        _, raw = make_batch(hp, args.batch, seed=100)
        rate, audio_s, dt, kind, note = cpu_rate(model, hp, raw, max(1, args.steps), threads)
        label = "ONNX Runtime CPU, the reference's session options" if kind == "reference" else \
            "PyTorch-CPU restatement of the reference's ONNX graph (ONNX Runtime probe: " + note + ")"
        line = {
            "impl": "reference", "metric": "audio-sec/sec", "value": rate, "unit": "audio-s/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * dt / max(1, args.steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "batch_per_gpu": args.batch,
                       "sample": f"{args.steps} utterances of the batch, batch 1 each (as the reference runs)"},
            "cpu_baseline": {"value": rate, "unit": "audio-s/s", "cores": threads, "kind": kind,
                             "sample": f"{args.steps} x 1 utterance (~8 s audio each) of the same synthetic batch; " + label},
            "e2e": {"value": rate, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm
    import sbv2_b200 as S
    from sbv2_b200 import assets
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    oracle = ov.build_model(hp, seed=0)
    onnx = assets.synth_onnx(ov.state_dict_numpy(oracle), hp.upsample_rates, hp.resblock_dilation_sizes)
    model = S.Model(onnx, bert=False, device=local_rank)
    model.seed(1234 + rank)
    utts, raw = make_batch(hp, args.batch, seed=100 + rank)
    # the e2e arm's inputs live in page-locked host memory (bench contract: "host->device copy ... from pinned host memory")
    utts_pinned = [dict(u, bert=S.pinned_copy(u["bert"])) for u in utts]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- kernel-only: inputs resident in HBM.  R replicas (one CUDA stream + one host thread each) run their
    # own resident batch concurrently, so the mid-pipeline T_y read-back of one overlaps kernels of the other.
    R = max(1, args.e2e_replicas)
    replicas = [model] + [S.Model(onnx, bert=False, device=local_rank) for _ in range(R - 1)]
    del onnx
    for i, m in enumerate(replicas[1:]):
        m.seed(4321 + rank + i)
    dbs = [S.DeviceBatch(m, utts) for m in replicas]
    streams = [torch.cuda.ExternalStream(m.stream, device=local_rank) for m in replicas]
    samples = 0
    for db in dbs:
        for _ in range(args.warmup):
            samples = db.run()

    def timed_kernel_run(n_rep: int, steps: int):
        """steps batches over the first n_rep replicas -> (ms, launches)"""
        counts = [steps // n_rep + (1 if i < steps % n_rep else 0) for i in range(n_rep)]
        ev0 = torch.cuda.Event(enable_timing=True)
        ev_end = [torch.cuda.Event(enable_timing=True) for _ in range(n_rep)]
        go = threading.Barrier(n_rep)
        l0 = sum(m.launch_count for m in replicas)

        def kworker(i):
            go.wait()
            for _ in range(counts[i]):
                dbs[i].run()
            ev_end[i].record(streams[i])

        for st in streams:
            st.synchronize()
        ev0.record(streams[0])
        for st in streams[1:n_rep]:
            st.wait_event(ev0)  # nothing of any replica starts before ev0
        ths = [threading.Thread(target=kworker, args=(i,)) for i in range(n_rep)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        for st in streams:
            st.synchronize()
        return max(ev0.elapsed_time(e) for e in ev_end), sum(m.launch_count for m in replicas) - l0

    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms, launches = timed_kernel_run(R, args.steps)
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs:
        # replica 0 runs at least one of the timed steps, and its device noise is seeded and advances per run by an amount
        # its inputs set, so its last batch depends on the arguments only
        dump_outputs(args.dump_outputs, dbs[0].download(), f"_rank{rank}" if world > 1 else "")
    # one replica on one stream (no overlap between replicas): what a single in-flight batch achieves
    ms_single, _ = timed_kernel_run(1, max(2, args.steps // 2))
    single_steps = max(2, args.steps // 2)
    barrier()
    db = dbs[0]
    # region split (CUDA events inside the library), measured on extra steps outside the timed region
    model.enable_timing(True)
    dec_ms = flow_ms = text_ms = 0.0
    n_reg = min(3, args.steps)
    for _ in range(n_reg):
        db.run()
        dec_ms += model.region_ms("decoder") / n_reg
        flow_ms += model.region_ms("flow") / n_reg
        text_ms += model.region_ms("text") / n_reg
    model.enable_timing(False)
    frames = samples // hp.hop
    audio_s_step = samples / SR

    # ---- end to end through the C ABI with host buffers
    # (a) one replica, one host thread: the latency-oriented number; (b) R replicas on this GPU, one host
    # thread each (ctypes releases the GIL): H2D / D2H of one replica overlap the kernels of the other.
    for _ in range(2):
        model.synthesize_batch(utts_pinned)
    barrier()
    t0 = time.perf_counter()
    single_audio = 0.0
    n_single = max(2, args.steps // 2)
    for _ in range(n_single):
        out = model.synthesize_batch(utts_pinned)
        single_audio += sum(a.size for a in out) / SR
    torch.cuda.synchronize()
    e2e_single = single_audio / (time.perf_counter() - t0)
    # the same from pageable caller memory (staged through the library's pinned block)
    t0 = time.perf_counter()
    pageable_audio = 0.0
    for _ in range(max(2, n_single // 2)):
        out = model.synthesize_batch(utts)
        pageable_audio += sum(a.size for a in out) / SR
    torch.cuda.synchronize()
    e2e_pageable = pageable_audio / (time.perf_counter() - t0)
    for m in replicas[1:]:
        for _ in range(2):
            m.synthesize_batch(utts_pinned)
    per_thread = [0.0] * R
    counts = [args.steps // R + (1 if i < args.steps % R else 0) for i in range(R)]

    def worker(i):
        for _ in range(counts[i]):
            o = replicas[i].synthesize_batch(utts_pinned)
            per_thread[i] += sum(a.size for a in o) / SR

    # untimed warm-up of the concurrent pattern itself: with R calls in flight the library's pool of pinned result blocks
    # grows to its steady-state size here (a cudaMallocHost of 45 MB costs ~10 ms) instead of inside the timed region
    def warm(i):
        for _ in range(max(args.warmup, 3)):
            replicas[i].synthesize_batch(utts_pinned)

    wthreads = [threading.Thread(target=warm, args=(i,)) for i in range(R)]
    for th in wthreads:
        th.start()
    for th in wthreads:
        th.join()
    barrier()
    t0 = time.perf_counter()
    ethreads = [threading.Thread(target=worker, args=(i,)) for i in range(R)]
    for th in ethreads:
        th.start()
    for th in ethreads:
        th.join()
    torch.cuda.synchronize()
    e2e_dt = time.perf_counter() - t0
    e2e_audio = sum(per_thread)
    barrier()
    h2d = sum(u["bert"].nbytes + 3 * 4 * u["x_tst"].size + u["style_vec"].nbytes + 8 * 4 for u in utts)
    d2h = int(samples * 4)

    # ---- the latency half of the metric: ONE ~5 s utterance, batch 1, host in -> host out (rank 0)
    latency = None
    if rank == 0:
        u5 = one_utt(hp, 151, 77)  # T_x = 151 -> ~4.9 s of audio with the synthetic duration calibration
        u5p = dict(u5, bert=S.pinned_copy(u5["bert"]))
        ts = wall(lambda: model.synthesize_batch([u5p]), 100, warm=5)
        n5 = model.synthesize_batch([u5p])[0].size
        l0 = model.launch_count
        model.synthesize_batch([u5p])
        latency = {"what": "one ~5 s utterance (T_x=151), batch 1, sbv2_synthesize_batch host in -> pinned host out, 100 calls",
                   "audio_s": n5 / SR, "p50_ms": float(np.median(ts) * 1e3), "p99_ms": float(np.percentile(ts, 99) * 1e3),
                   "min_ms": float(ts.min() * 1e3), "launches_per_call": int(model.launch_count - l0)}

    t = torch.tensor([ms, e2e_dt * 1000.0, ms_single], dtype=torch.float64, device="cuda")
    tot = torch.tensor([audio_s_step * args.steps, e2e_audio, float(launches)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_max, e2e_ms_max, ms_single_max = float(t[0]), float(t[1]), float(t[2])
    audio_total, e2e_audio_total, launches_total = float(tot[0]), float(tot[1]), int(tot[2])

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained")
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained; fp16 has the same tensor rate)"
        if not peak_tf:
            peak_tf, peak_src = 1400.0, "fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)"
        dec_flop = DEC_FLOP_PER_FRAME * frames
        achieved = dec_flop / (dec_ms * 1e-3) / 1e12 if dec_ms > 0 else None
        # DRAM traffic of the decoder's launches: an ncu figure, so it cannot be measured inside this run; the committed
        # figure is used only while the kernel sources it was measured on are unchanged (digest recorded beside it)
        traffic, traffic_note = None, "no ncu capture for the current kernel sources (tools/decoder_traffic.py)"
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "decoder_traffic.json")))
            if tj.get("sources_sha1") == sources_digest():
                traffic = tj.get("dram_bytes_per_step")
                traffic_note = "ncu dram__bytes_read.sum + dram__bytes_write.sum over the decoder's launches of one step of this workload " \
                               "(profiles/decoder_traffic.json, same kernel sources)"
        except Exception:
            pass
        line = {
            "metric": "audio-sec/sec", "value": audio_total / (ms_max * 1e-3), "unit": "audio-s/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16 operands / f32 accumulate on tcgen05 (decoder, flow; text encoder with two-term fp16 splits); f32 elsewhere",
            "data": "synthetic",
            "config": {"workload": workload, "batch_per_gpu": args.batch, "audio_s_per_step_per_gpu": audio_s_step,
                       "frames_per_step_per_gpu": int(frames), "weights": "random-init tsukuyomi-shaped JP-Extra, seed 0",
                       "l2": "activations per step (>2 GB) exceed the 126 MB L2; no explicit flush",
                       "region_ms_per_step_rank0": {"text": text_ms, "flow": flow_ms, "decoder": dec_ms}},
            "single_stream": {"value": audio_s_step * single_steps * world / (ms_single_max * 1e-3), "unit": "audio-s/s",
                              "ms_per_step": ms_single_max / single_steps,
                              "what": f"kernel-only, ONE replica on ONE stream per GPU (value above: {R} replicas / streams per GPU)"},
            "e2e": {"value": e2e_audio_total / (e2e_ms_max * 1e-3), "unit": "audio-s/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": d2h, "replicas_per_gpu": R, "single_replica_rank0": e2e_single,
                    "single_replica_pageable_inputs_rank0": e2e_pageable,
                    "api": "sbv2_synthesize_batch (page-locked host buffers in, pinned host waveforms out)"},
            "latency": latency,
            "gpu_launches": launches_total,
            "replicas_per_gpu": R,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "umma_conv_kernel + umma_pair_kernel (HiFi-GAN decoder, timed region = whole decoder)",
                         "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": (achieved / peak_tf) if achieved else None, "traffic": traffic, "traffic_note": traffic_note,
                         "peak_source": peak_src},
        }
        which = [c for c in args.configs.split(",") if c] if not args.tiny else []
        if which:
            try:
                line["configs"] = other_configs(S, assets, ov, hp, oracle, model, peak_tf, which)
            except Exception as e:  # noqa: BLE001  (the headline line must still print)
                line["configs"] = {"error": f"{type(e).__name__}: {e}"}
        if not args.no_cpu_baseline:
            n = 3
            rate, a_s, dt, kind, note = cpu_rate(oracle, hp, raw, n, threads)
            label = "ONNX Runtime CPU, the reference's session options" if kind == "reference" else \
                "PyTorch-CPU restatement (ONNX Runtime probe: " + note + ")"
            line["cpu_baseline"] = {"value": rate, "unit": "audio-s/s", "cores": threads, "kind": kind,
                                    "sample": f"{n} utterances (~{a_s:.0f} s audio) of the same batch, batch 1 each; " + label}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
