"""The bench contract end to end on a GPU box: default arm (with the CPU baseline leg) on a reduced batch, and the JSON keys
the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")


def test_bench_line_has_the_contract_keys(lib_built, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch", "4", "--steps", "2", "--warmup", "3", "--configs", "cfg1,cfg3",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline", "latency", "single_stream", "configs"):
        assert k in line, k
    assert line["metric"] == "audio-sec/sec" and line["value"] > 0 and line["gpu_launches"] > 0
    assert line["e2e"]["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert line["roofline"]["bound"] == "tensor" and 0 < line["roofline"]["frac"] < 1
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["value"] > 0
    assert "probe" in line["cpu_baseline"]["sample"] or line["cpu_baseline"]["kind"] == "reference"   # ORT probed at run time
    assert line["latency"]["p50_ms"] > 0 and line["latency"]["p99_ms"] >= line["latency"]["p50_ms"] and 4 < line["latency"]["audio_s"] < 6
    assert line["single_stream"]["value"] > 0
    assert line["configs"]["cfg1"]["latency_ms_p50"] > 0 and line["configs"]["cfg3"]["decoder_ms"] > 0
    assert line["e2e"]["single_replica_rank0"] > 0 and line["e2e"]["single_replica_pageable_inputs_rank0"] > 0
    # --dump-outputs: the last timed batch of 4 utterances, whole (well under the size limit), finite and not silent
    audio, lengths = np.load(tmp_path / "audio.npy"), np.load(tmp_path / "audio_lengths.npy")
    assert sorted(os.listdir(tmp_path)) == ["audio.npy", "audio_lengths.npy"]
    assert audio.dtype == np.float32 and lengths.dtype == np.float64 and lengths.size == 4 and lengths.sum() == audio.size
    assert np.isfinite(audio).all() and np.abs(audio).max() > 0
