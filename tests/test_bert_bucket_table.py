"""The DeBERTa relative-position bucket table (bert_bucket_table in bert_model.cu, through sbv2_debug_bert_bucket_table of
libsbv2_b200_debug.so; no GPU needed) against HF make_log_bucket_position followed by the clamp of the c2p / p2c indices.

The kernels clamp a distance to +-R and read entry d + R, so the table is only right if every |d| >= R maps to the row of
+-R.  For HF's span of 256 that bound is 512, not 511: idx(-512) = 0 but idx(-511) = 1."""
import importlib.util
import os

import numpy as np
import pytest
import torch
from transformers.models.deberta_v2.modeling_deberta_v2 import make_log_bucket_position

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def S(lib_built):
    spec = importlib.util.spec_from_file_location("sbv2_b200_build", os.path.join(ROOT, "sbv2-api_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()  # the debug library carries the hook; a no-op when up to date
    import sbv2_b200
    return sbv2_b200


def hf_index(d: np.ndarray, span: int) -> np.ndarray:
    b = make_log_bucket_position(torch.from_numpy(d), span, 2 * span)
    return torch.clamp(b + span, 0, 2 * span - 1).long().numpy()


@pytest.mark.parametrize("span", [256, 128, 64])
def test_bucket_table_matches_hf_for_every_distance(S, span):
    tab = S.debug_bert_bucket_table(span)
    R = (tab.size - 1) // 2
    d = np.arange(-40000, 40001, dtype=np.int64)
    got = tab[np.clip(d, -R, R) + R]
    want = hf_index(d, span)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"span {span}: {bad.size} distances differ, first d = {d[bad[0]]}: {got[bad[0]]} vs {want[bad[0]]}"
    # R is the smallest bound with that property
    assert hf_index(np.array([-(R - 1)]), span)[0] != 0 or hf_index(np.array([R - 1]), span)[0] != 2 * span - 1


def test_bucket_table_bound_for_span_256(S):
    tab = S.debug_bert_bucket_table(256)
    R = (tab.size - 1) // 2
    assert R == 512
    assert tab[-512 + R] == 0 and tab[-511 + R] == 1
    assert tab[511 + R] == tab[512 + R] == 511
