"""-m gpu: the damage profile on the device (miagpu_misincorporation) against the `.maln`-to-table oracle of
tests/test_misinc_oracle.py -- on the unmodified reference binary's `.maln` files through host/mia_gpu -d and through
driver.ResidentAssembler in every round, on the library's own file for 200 k damaged synthetic reads, over shards, and the
refusals.  Every comparison is exact."""
import gzip
import json
import os
import subprocess

import numpy as np
import pytest

import gpu_checks
from test_host_c import HOST, ensure_host, matrix_text
from test_misinc_oracle import misinc_table, read_damage_file

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
A, C, G, T = 0, 1, 2, 3
MATRIX = {"ancient.submat.txt": "ancient", "ancient.submat.solexa.pe.txt": "pe", "ancient.submat.solexa.onepass.txt": "onepass"}


def _sessions():
    s = json.load(gzip.open(os.path.join(HERE, "golden", "maln_session.json.gz"), "rt"))["sessions"]
    r2 = json.load(gzip.open(os.path.join(HERE, "golden", "maln_session_r2.json.gz"), "rt"))
    hp = json.load(gzip.open(os.path.join(HERE, "golden", "hp.json.gz"), "rt"))["sessions"]
    return {**s, **r2, **hp}


SESSIONS = ["circ_k10", "lin_pe", "tr1_tf_lin", "tr1_tf_lin_k8", "tr1_tf_c", "dups_c_k10_u", "dups_c_k10_U", "circ_k10_H", "circ_k10_SN",
            "circ_k10_p2", "flat_2000_c", "origin305_splitflip_c", "synth3k_div10_c_k12_D", "synth1k_N_lin_D", "hp2k_c_k10_h", "hp2k_lin_k12_hD"]
# what driver.ResidentAssembler runs as the reference's main loop: no cut given (-H / -S -N), no repeat filter (-u / -U)
RESIDENT = [n for n in SESSIONS if not ({"-H", "-S", "-u", "-U"} & set(_sessions()[n]["flags"]))]


def _run_host(exe, s, golden, tmp_path, extra=()):
    (tmp_path / "ref.fa").write_text(s.get("ref_text") or f">{s['ref_id']} {s['ref_desc']}\n{s['ref']}\n")
    (tmp_path / "reads.fq").write_text(s["fastq"])
    (tmp_path / "m.txt").write_text(matrix_text(golden[MATRIX.get(s["matrix"], s["matrix"])]))
    r = subprocess.run([exe, *extra, "-r", "ref.fa", "-f", "reads.fq", "-s", "m.txt", "-m", "out", "-d", "damage.tsv"] + s["flags"], cwd=tmp_path,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return r


@pytest.mark.parametrize("name", SESSIONS)
def test_host_damage_file_equals_oracle_on_the_reference_final_maln(golden, name, tmp_path):
    s = _sessions()[name]
    if s.get("complete") is False:
        pytest.skip("the golden session stops before convergence: its last file is not the host's final round")
    ensure_host()
    _run_host(HOST, s, golden, tmp_path)
    n = len(s["malns"])
    assert os.path.exists(tmp_path / f"out.{n}") and not os.path.exists(tmp_path / f"out.{n + 1}")
    got = read_damage_file(tmp_path / "damage.tsv")
    want = misinc_table(s["malns"][-1])
    assert (got == want).all(), (name, np.argwhere(got != want).tolist()[:10])


def _flag(flags, f, default=0):
    return int(flags[flags.index(f) + 1]) if f in flags else default


@pytest.mark.parametrize("name", RESIDENT)
def test_resident_rounds_table_equals_oracle_every_round(gpu, golden, name, tmp_path):
    import _pkg
    _pkg.load()
    from mia_b200 import api, driver
    s = _sessions()[name]
    fl = s["flags"]
    ref = s.get("ref") or "".join(s["ref_text"].split("\n")[1:]).replace(" ", "").replace("\r", "")
    (tmp_path / "reads.fq").write_text(s["fastq"])
    rdr = api.FastxReader(path=str(tmp_path / "reads.fq"))
    batch = rdr.next()
    rdr.close()
    try:
        R = driver.ResidentAssembler(gpu, ref, golden[MATRIX.get(s["matrix"], s["matrix"])], int("-c" in fl), _flag(fl, "-k"), 0, cons_code=_flag(fl, "-p", 1),
                                     distant_ref=int("-D" in fl), hp=int("-h" in fl))
        R.pass1(batch["bases"], batch["offsets"])
        for it, body in enumerate(s["malns"]):
            R.iterate()
            got, want = R.misincorporation(), misinc_table(body)
            assert got.dtype == np.int64 and got.shape == (31, 6, 6)
            assert (got == want).all(), (name, it + 1, np.argwhere(got != want).tolist()[:10])
            assert (R.misincorporation() == got).all()                   # the call reads the round's state, changes none of it
    finally:
        gpu.set_homopolymer(0)


def test_200k_damaged_reads_to_convergence(gpu, tmp_path):
    # synth defaults: 35-75 bp, both strands, 5' C->T and 3' G->A at 0.3 * 0.5**d.  Without the pointer state every read owns its
    # AlnSeqs: the model miagpu_write_maln writes, so the library's own final file is the reference for the table
    import _pkg
    _pkg.load()
    from mia_b200 import driver, synth
    ref = synth.random_reference(16569, seed=41)
    bases, off, _ = synth.make_reads(ref, 200_000, seed=42)
    R = driver.ResidentAssembler(gpu, ref, gpu_checks.load_pssm("ancient"), 1, 12, 0, pointer_state=False, strand_unknown="drop")
    R.pass1(bases, off)
    conv = False
    while not conv and R.iter < 10:
        _, conv = R.iterate(want_gaps=True)
    assert conv
    t = R.misincorporation()
    n = len(off) - 1
    ids = b"".join(b"r%d\0" % i for i in range(n))
    id_off = np.concatenate([[0], np.cumsum([len(b"r%d" % i) + 1 for i in range(n)])]).astype(np.int64)
    batch = dict(bases=bases, offsets=off, ids=ids, id_off=id_off)
    R.write_maln(str(tmp_path / "final"), batch, "ref")
    body = open(tmp_path / "final").read().split("\n", 1)[1]
    assert (t == misinc_table(body)).all()
    ct0 = t[0, C, T] / t[0, C].sum()
    ga30 = t[30, G, A] / t[30, G].sum()
    ct15 = t[15, C, T] / t[15, C].sum()
    assert abs(ct0 - 0.30) <= 0.02 and abs(ga30 - 0.30) <= 0.02 and ct15 < 0.01, (ct0, ga30, ct15)


@pytest.mark.parametrize("parts", [2, 3])
def test_sharded_tables_sum_to_the_single_gpu_table(gpu, parts):
    from mia_b200 import api, driver, shard
    ref, bases, off, rc, as_, ae = gpu_checks.make_case(60000, 4000, seed=17, divergence=0.02, indel_rate=0.004)
    n = len(off) - 1
    seq_len = np.diff(off).astype(np.int32)
    sticky = (np.arange(n) % 97 == 0).astype(np.uint8)
    gpu.set_pssm(gpu_checks.load_pssm("onepass"))
    gpu.set_reference(ref, circular=1, with_rc=0)
    gpu.upload_reads(bases, off)
    gpu.set_alignment_inputs(rc, as_, ae)
    gpu.set_cut_inputs(seq_len, None, sticky)
    cons, _, _ = gpu.iterate_resident(dropped=np.zeros(n, np.uint8))
    single = gpu.misincorporation()
    assert single.sum() > 0
    bnd = [n * r // parts for r in range(parts + 1)]
    ctxs = [api.MiaGpu(0) for _ in range(parts)]
    try:
        for r, g in enumerate(ctxs):
            lo, hi = bnd[r], bnd[r + 1]
            g.set_pssm(gpu_checks.load_pssm("onepass"))
            g.set_reference(ref, circular=1, with_rc=0)
            g.upload_reads(np.ascontiguousarray(bases[off[lo]:off[hi]]), np.ascontiguousarray(off[lo:hi + 1] - off[lo]))
            g.set_alignment_inputs(rc[lo:hi].copy(), as_[lo:hi].copy(), ae[lo:hi].copy())
            g.set_cut_inputs(seq_len[lo:hi].copy(), None, sticky[lo:hi].copy())
        res = shard.LocalShards(ctxs).resident(max(bnd[r + 1] - bnd[r] for r in range(parts)),
                                               dropped=[np.zeros(bnd[r + 1] - bnd[r], np.uint8) for r in range(parts)])
        assert all(c == cons for c, _, _ in res)
        tables = [g.misincorporation() for g in ctxs]
        assert (sum(tables) == single).all()

        # driver.ResidentAssembler's sum over the ranks: each rank hands in its own table, the others' come from their contexts
        class Exchange:
            def __init__(self, rank):
                self.rank = rank

            def all_gather_host(self, a):
                return np.concatenate([a if k == self.rank else g.misincorporation().ravel() for k, g in enumerate(ctxs)])
        for r, g in enumerate(ctxs):
            R = object.__new__(driver.ResidentAssembler)
            R.g, R.x = g, Exchange(r)
            assert (R.misincorporation() == single).all(), r
    finally:
        for g in ctxs:
            g.close()


def test_multi_gpu_host_writes_the_same_damage_file(golden, tmp_path):
    import _pkg
    _pkg.load()
    from mia_b200 import api
    mg = os.path.join(os.path.dirname(HOST), "mia_gpu_mg")
    if not os.path.exists(mg):
        pytest.skip("host/mia_gpu_mg not built (needs nccl.h / libnccl at build time)")
    ensure_host()
    s = _sessions()["circ_k10"]
    (tmp_path / "one").mkdir()
    _run_host(HOST, s, golden, tmp_path / "one")
    want = open(tmp_path / "one" / "damage.tsv").read()
    for gpus in (1, 2):
        if api.load_library().miagpu_device_count() < gpus:
            continue
        d = tmp_path / f"g{gpus}"
        d.mkdir()
        _run_host(mg, s, golden, d, ("-g", str(gpus)))
        assert open(d / "damage.tsv").read() == want, gpus


def test_refusals_say_why(gpu):
    import _pkg
    _pkg.load()
    from mia_b200 import api
    g = api.MiaGpu(0)
    try:
        with pytest.raises(api.MiaGpuError, match="no round has ended with base calling"):
            g.misincorporation()
        ref, bases, off, rc, as_, ae = gpu_checks.make_case(3000, 2000, seed=23)
        g.set_pssm(gpu_checks.load_pssm("ancient"))
        g.set_reference(ref, circular=1, with_rc=0)
        g.upload_reads(bases, off)
        with pytest.raises(api.MiaGpuError, match="no round has ended"):          # still none: the first reason stands
            g.misincorporation()
        g.set_alignment_inputs(rc, as_, ae)
        g.set_cut_inputs(np.diff(off).astype(np.int32))
        cons, _, _ = g.iterate_resident()
        t = g.misincorporation()
        assert t.sum() > 0
        g.adopt_alignment()                                             # the next round's inputs: the table stays
        assert (g.misincorporation() == t).all()
        g.set_reference(cons, circular=1, with_rc=0)
        with pytest.raises(api.MiaGpuError, match="miagpu_set_reference"):
            g.misincorporation()
        g.iterate_resident()
        assert g.misincorporation().sum() > 0
        g.realign_resident()
        with pytest.raises(api.MiaGpuError, match="realign"):
            g.misincorporation()
        g.consensus_natural()
        assert g.misincorporation().sum() > 0
    finally:
        g.close()
