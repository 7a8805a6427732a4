"""The shared-memory model of the 16-bit pair kernel (scripts/p16_smem_model.py) and the substitution-table index it models
(p16_tab_entry in csrc/pair16.cuh): CPU only."""
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import p16_smem_model as m  # noqa: E402


def test_entry_map_is_a_bijection_with_acgt_on_distinct_bank_pairs():
    a, b = np.meshgrid(np.arange(5), np.arange(5), indexing="ij")
    e = m.tab_new(a, b)
    assert sorted(e.ravel().tolist()) == list(range(25))
    ia, ib = m.inv_new(e)
    assert (ia == a).all() and (ib == b).all()
    acgt = e[:4, :4].ravel()
    assert sorted(acgt.tolist()) == list(range(16))          # entry e sits on bank pair e % 16


def test_model_mirrors_the_header():
    """the Python map is the one pair16.cuh compiles"""
    src = open(os.path.join(ROOT, "mapping-iterative-assembler_b200", "csrc", "pair16.cuh")).read()
    assert "a < 4 && b < 4 ? a * 4 + b : a == 4 ? 16 + b : 21 + a" in src
    assert re.search(r"constexpr int P16_PAD_CODE = 0;", src)


def test_table_wavefronts_rule():
    assert m.table_wavefronts(np.zeros(16, int)) == 1                      # one address: broadcast
    assert m.table_wavefronts(np.arange(16)) == 1                          # sixteen bank pairs
    assert m.table_wavefronts(np.array([0, 16] + [1] * 14)) == 2           # 0 and 16 share a bank pair


def test_benchmark_workload_model():
    res = m.model(20000)
    assert {9, 10, 11} <= set(res)
    for K in (9, 10, 11):
        old, new = res[K]["old"], res[K]["new"]
        assert abs(new["table"] - 2.0) < 1e-9             # the reference has no N: one wavefront per half-warp
        assert 3.5 < old["table"] < 3.9                    # a*5+b with N padding
        assert old["rowoff"] == 4.0 and new["rowoff"] == 1.0
        assert new["total"] < 0.65 * old["total"]
    o = res[11]["old"]
    assert o["total"] <= m.CAPTURE_K11 <= o["total"] + o["shfl"] + 3     # the parent's capture lies in the model's range
