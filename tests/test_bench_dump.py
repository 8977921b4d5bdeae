"""CPU test of bench.py --dump-outputs: the waveforms of one batch are written whole while they fit the size limit, and as the
same fixed, seeded sample (values and positions) past it."""
import os

import numpy as np

import bench


def _waves(seed):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal(int(n)).astype(np.float32) for n in rng.integers(1, 2000, 7)]


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_whole_batch(tmp_path):
    waves = _waves(0)
    bench.dump_outputs(str(tmp_path), waves)
    got = _load(tmp_path)
    assert sorted(got) == ["audio", "audio_lengths"]
    assert got["audio"].dtype == np.float32 and got["audio_lengths"].dtype == np.float64
    np.testing.assert_array_equal(got["audio"], np.concatenate(waves))
    assert got["audio_lengths"].tolist() == [w.size for w in waves]


def test_dump_sample_past_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT", 1024 + 7 * 8 + 12 * 500)
    waves = _waves(1)
    flat = np.concatenate(waves)
    runs = []
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), waves, "_rank1")
        runs.append(_load(tmp_path / name))
    a, b = runs
    assert sorted(a) == ["audio_index_rank1", "audio_lengths_rank1", "audio_rank1"]
    idx = a["audio_index_rank1"]
    assert idx.dtype == np.float64 and idx.size == 500 and np.all(np.diff(idx) > 0) and idx[-1] < flat.size
    np.testing.assert_array_equal(a["audio_rank1"], flat[idx.astype(np.int64)])
    assert a["audio_lengths_rank1"].sum() == flat.size
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_LIMIT
