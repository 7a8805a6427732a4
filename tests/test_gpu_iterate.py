"""GPU: whole rounds (miagpu_iterate_host / miagpu_iterate_resident, score cut on the device) against the
separate calls with the host-side score cut.  Bit-exact: slope, intercept (as IEEE doubles), flags, gaps, consensus."""
import struct

import numpy as np
import pytest

import gpu_checks

pytestmark = pytest.mark.gpu


def _bits(x):
    return struct.pack("<d", x)


def _separate(gpu, api, bases, off, rc, as_, ae, seq_len, sticky, unique_best=None, hard_cut=0, score_cut=None):
    out = gpu.realign_host(bases, off, rc, as_, ae)
    if score_cut is None:
        fit = api.score_cut(seq_len, out["score"], unique_best)
        below = api.cull_flags(seq_len, out["score"], unique_best, hard_cut, 1, fit[0], fit[1])
    else:
        fit = score_cut
        below = api.cull_flags(seq_len, out["score"], unique_best, hard_cut, 1, fit[0], fit[1])
    tested = np.ones(len(sticky), bool) if unique_best is None else unique_best.astype(bool)
    drop = (sticky | (below & tested)).astype(np.uint8)             # a read that is not unique_best is not tested (mia.c:466)
    flags = np.where(tested, drop, 2).astype(np.uint8)              # ... and not in the culled list at all
    cons, gaps, _ = gpu.consensus_natural(flags, flags, 1)
    return out, fit, drop, cons, gaps


@pytest.mark.parametrize("n_reads,ref_len,seed,heavy", [(300, 1500, 3, 0.0), (9000, 3000, 4, 0.0), (120000, 6000, 5, 0.0), (20000, 3000, 6, 0.2)],
                         ids=["300-1500-3", "9000-3000-4", "120000-6000-5", "20000-3000-6-heavy"])
def test_iterate_resident_equals_separate_calls(gpu, n_reads, ref_len, seed, heavy):
    from mia_b200 import api
    ref, bases, off, rc, as_, ae = gpu_checks.make_case(n_reads, ref_len, seed=seed, divergence=0.02, indel_rate=0.004)
    n = len(off) - 1
    if heavy:
        # a `heavy` share of the reads with a quarter of their bases substituted: low scores, no indels, few runs, no status bits.
        # Round 1 then drops more than an eighth of the reads, so round 2 flags the entries before it accumulates the columns.
        rng = np.random.default_rng(seed)
        read_of = np.repeat(np.arange(n), np.diff(off))
        sub = (rng.random(n) < heavy)[read_of] & (rng.random(len(bases)) < 0.25)
        code = np.searchsorted(np.frombuffer(b"ACGT", np.uint8), bases[sub]) % 4
        bases = bases.copy()
        bases[sub] = np.frombuffer(b"ACGT", np.uint8)[(code + rng.integers(1, 4, len(code))) % 4]
    gpu.set_pssm(gpu_checks.load_pssm("onepass"))
    gpu.set_reference(ref, circular=1, with_rc=0)
    seq_len = np.diff(off).astype(np.int32)
    sticky = (np.arange(n) % 89 == 0).astype(np.uint8)
    out, fit, drop, cons, gaps = _separate(gpu, api, bases, off, rc, as_, ae, seq_len, sticky)
    gpu.upload_reads(bases, off)
    gpu.set_alignment_inputs(rc, as_, ae)
    gpu.set_cut_inputs(seq_len, None, sticky)
    d2 = np.zeros(n, np.uint8)
    cons2, fit2, gaps2 = gpu.iterate_resident(dropped=d2, want_gaps=True)
    assert _bits(fit2[0]) == _bits(fit[0]) and _bits(fit2[1]) == _bits(fit[1]), (fit, fit2)
    assert (d2 == drop).all()
    assert cons2 == cons and (gaps2 == gaps).all()
    if heavy:
        assert int(((d2 == 1) & (sticky == 0)).sum()) * 8 > n
    # a second round on the same inputs: the flags are sticky on the device, nothing changes
    d3 = np.zeros(n, np.uint8)
    cons3, fit3, _ = gpu.iterate_resident(dropped=d3)
    assert cons3 == cons and (d3 == drop).all() and _bits(fit3[0]) == _bits(fit[0])
    gpu.reset_dropped()
    d4 = np.zeros(n, np.uint8)
    gpu.iterate_resident(dropped=d4)
    below = api.cull_flags(seq_len, out["score"], None, 0, 1, fit[0], fit[1])
    assert (d4 == below).all()


def test_iterate_host_policy_variants(gpu):
    from mia_b200 import api
    ref, bases, off, rc, as_, ae = gpu_checks.make_case(40000, 5000, seed=31, divergence=0.03, indel_rate=0.004)
    gpu.set_pssm(gpu_checks.load_pssm("onepass"))
    gpu.set_reference(ref, circular=1, with_rc=0)
    n = len(off) - 1
    seq_len = np.diff(off).astype(np.int32)
    sticky = (np.arange(n) % 101 == 0).astype(np.uint8)
    rng = np.random.default_rng(1)
    unique = (rng.random(n) < 0.8).astype(np.uint8)
    for kw in (dict(unique_best=unique), dict(hard_cut=9000), dict(score_cut=(150.0, -500.0)), dict(unique_best=unique, hard_cut=7000)):
        out, fit, drop, cons, gaps = _separate(gpu, api, bases, off, rc, as_, ae, seq_len, sticky, **kw)
        d2 = sticky.copy()
        cons2, out2, _, gaps2 = gpu.iterate_host(bases, off, rc, as_, ae, seq_len, d2, want_gaps=True, **kw)
        assert (d2 == drop).all(), kw
        assert cons2 == cons and (gaps2 == gaps).all(), kw
        assert (out2["score"] == out["score"]).all()


def test_iterate_reports_bad_seq_len(gpu):
    from mia_b200 import api
    ref, bases, off, rc, as_, ae = gpu_checks.make_case(5000, 2000, seed=2)
    gpu.set_pssm(gpu_checks.load_pssm("onepass"))
    gpu.set_reference(ref, circular=1, with_rc=0)
    seq_len = np.diff(off).astype(np.int32)
    seq_len[1234] = 300
    with pytest.raises(api.MiaGpuError, match="seq_len"):
        gpu.iterate_host(bases, off, rc, as_, ae, seq_len, np.zeros(len(seq_len), np.uint8))
