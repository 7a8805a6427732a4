"""-m gpu: the 16-bit SIMD pair kernel (csrc/pair16.cuh) against the 32-bit kernel and the oracle, and the
one-call iteration (miagpu_iterate_host) against the separate calls.  Bit-exact."""
import os

import numpy as np
import pytest

import gpu_checks

pytestmark = pytest.mark.gpu


def _realign(gpu, case, sm, pair16):
    ref, bases, off, rc, as_, ae = case
    os.environ["MIAGPU_PAIR16"] = "1" if pair16 else "0"
    try:
        gpu.set_pssm(sm)
        gpu.set_reference(ref, circular=1, with_rc=0)
        out = gpu.realign_host(bases, off, rc, as_, ae)
        pb, fb, lmax = gpu.last_pair_buckets()
    finally:
        os.environ.pop("MIAGPU_PAIR16", None)
    return out, sum(b["reads"] for b in pb), fb, lmax


@pytest.mark.parametrize("matrix,lens,div,indel", [("onepass", (35, 75), 0.005, 0.0), ("ancient", (30, 140), 0.03, 0.004),
                                                    ("onepass", (20, 60), 0.10, 0.005)])
def test_pair16_equals_32bit_kernel(gpu, matrix, lens, div, indel):
    case = gpu_checks.make_case(20000, 5000, seed=17 + lens[0], divergence=div, indel_rate=indel, min_len=lens[0], max_len=lens[1])
    sm = gpu_checks.load_pssm(matrix)
    a, taken, handed, lmax = _realign(gpu, case, sm, True)
    b, taken0, _, _ = _realign(gpu, case, sm, False)
    assert taken0 == 0 and taken > 10000 and lmax >= 130, (taken, taken0, lmax)
    assert handed < taken
    for k in ("score", "as_out", "ae_out", "abr", "n_runs", "status"):
        assert (a[k] == b[k]).all(), (k, np.flatnonzero(a[k] != b[k])[:5])
    nr = np.maximum(a["n_runs"], 0)
    mask = np.arange(a["runs"].shape[1])[None, :] < nr[:, None]
    assert (a["runs"][mask] == b["runs"][mask]).all()


def test_pair16_vs_oracle_exact_windows(gpu, oracle):
    # as/ae exact (bench-like): almost every read stays in the pair kernel
    ref, bases, off, rc, as_, ae = gpu_checks.make_case(3000, 4000, seed=5, divergence=0.004, indel_rate=0.0)
    bad, out = gpu_checks.check_realign(gpu, oracle, ref, bases, off, rc, as_, ae, gpu_checks.load_pssm("onepass"))
    assert not bad, bad[:3]
    pb, fb, _ = gpu.last_pair_buckets()
    assert sum(b["reads"] for b in pb) > 2500 and fb < 600


def test_iterate_host_equals_separate_calls(gpu):
    from mia_b200 import api
    ref, bases, off, rc, as_, ae = gpu_checks.make_case(30000, 6000, seed=23, divergence=0.02, indel_rate=0.004)
    gpu.set_pssm(gpu_checks.load_pssm("onepass"))
    gpu.set_reference(ref, circular=1, with_rc=0)
    n = len(off) - 1
    seq_len = np.diff(off).astype(np.int32)
    out = gpu.realign_host(bases, off, rc, as_, ae)
    packed = np.zeros(n * 4, np.uint16)
    tot, _, _ = gpu.get_runs_packed(None, packed)
    sticky = (np.arange(n) % 97 == 0).astype(np.uint8)              # flags left by earlier rounds
    below = api.cull_flags(seq_len, out["score"])
    drop = (sticky | below).astype(np.uint8)
    cons, gaps, _ = gpu.consensus_natural(drop, drop, 1)
    d2 = sticky.copy()
    packed2 = np.zeros(n * 4, np.uint16)
    cons2, out2, tot2, gaps2 = gpu.iterate_host(bases, off, rc, as_, ae, seq_len, d2, packed=packed2, want_gaps=True)
    assert cons2 == cons and tot2 == tot and (gaps2 == gaps).all()
    assert (d2 == drop).all()
    assert (packed2[:tot] == packed[:tot]).all()
    for k in ("score", "as_out", "ae_out", "abr", "n_runs", "status"):
        assert (out2[k] == out[k]).all(), k


@pytest.mark.parametrize("matrix,div,indel", [("pe", 0.01, 0.001), ("onepass", 0.12, 0.006), ("ancient", 0.30, 0.01)])
def test_pair16_rebased_frame_takes_long_reads(gpu, monkeypatch, matrix, div, indel):
    # reads of 100-156 bases are beyond the low 16-bit frame (~130 rows): the RB variant (pair16.cuh 5.) takes them -- exact against the
    # 32-bit kernel field for field, including reads that diverge so much that they sink to the poison bound and are handed over
    case = gpu_checks.make_case(16000, 6000, seed=301, divergence=div, indel_rate=indel, min_len=100, max_len=156)
    sm = gpu_checks.load_pssm(matrix)
    a, taken, handed, _ = _realign(gpu, case, sm, True)
    b, taken0, _, _ = _realign(gpu, case, sm, False)
    monkeypatch.setenv("MIAGPU_PAIR_RB", "0")
    _, taken_low, _, _ = _realign(gpu, case, sm, True)
    monkeypatch.delenv("MIAGPU_PAIR_RB")
    assert taken0 == 0 and taken > 15000 and taken_low < 9000, (taken, taken_low)
    for k in ("score", "as_out", "ae_out", "abr", "n_runs", "status"):
        assert (a[k] == b[k]).all(), (k, np.flatnonzero(a[k] != b[k])[:5], a[k][a[k] != b[k]][:5], b[k][a[k] != b[k]][:5])
    nr = np.maximum(a["n_runs"], 0)
    mask = np.arange(a["runs"].shape[1])[None, :] < nr[:, None]
    assert (a["runs"][mask] == b["runs"][mask]).all()
