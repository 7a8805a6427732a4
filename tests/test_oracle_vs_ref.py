"""CPU: the oracle restatement against the UNMODIFIED reference compiled into oracle/_ref
(only where that library exists: the build container, or a box the prebuilt .so travelled to)."""
import os
import random
import tempfile

import numpy as np
import pytest

from oracle_driver import OracleRun


def _fuzz(rng):
    n1 = rng.randint(5, 160)
    ref = "".join(rng.choice("ACGT" if rng.random() < 0.97 else "N") for _ in range(n1))
    n2 = rng.randint(1, 70)
    if rng.random() < 0.7 and n1 > n2:
        s = rng.randint(0, n1 - n2)
        rd = list(ref[s:s + n2])
        for i in range(len(rd)):
            x = rng.random()
            if x < 0.05:
                rd[i] = rng.choice("ACGT")
            elif x < 0.07:
                rd[i] = ""
            elif x < 0.09:
                rd[i] = rd[i] + rng.choice("ACGT")
        rd = "".join(rd)[:256] or "A"
    else:
        rd = "".join(rng.choice("ACGT") for _ in range(n2))
    mask = None
    if rng.random() < 0.5:
        mask = np.zeros(n1, np.uint8)
        for _ in range(rng.randint(1, 3)):
            a = rng.randint(0, n1 - 1)
            mask[a:min(n1, a + rng.randint(1, 90))] = 1
    return ref, rd, mask


def test_align_fuzz_full_matrices(oracle, ref, golden):
    rng = random.Random(99)
    mats = [golden["flat"], golden["ancient"], golden["ancient_rc"], golden["pe"]]
    for it in range(1500):
        s1, s2, mask = _fuzz(rng)
        sm, sg5 = rng.choice(mats), rng.randint(0, 1)
        a = ref.align(s1, s2, sm, sg5, mask, matrices=True)
        b = oracle.align(s1, s2, sm, sg5, mask, matrices=True)
        for k in ("score", "abr", "abc", "aer", "aec", "ref_gapped", "read_gapped"):
            assert a[k] == b[k], (it, k)
        assert (a["S"] == b["S"]).all() and (a["T"] == b["T"]).all(), it


def _fuzz_hp(rng):
    # homopolymer-rich sequences: runs of 1-9 equal bases, the read a copy with run lengths changed here and there
    runs = [(rng.choice("ACGT"), max(1, int(rng.expovariate(0.45)))) for _ in range(rng.randint(4, 45))]
    ref = "".join(b * min(n, 9) for b, n in runs)
    a = rng.randint(0, max(0, len(runs) - 3))
    sub = runs[a:a + rng.randint(2, 25)]
    rd = []
    for b, n in sub:
        x = rng.random()
        if x < 0.25:
            n = max(1, n + rng.choice((-2, -1, 1, 2)))
        elif x < 0.30:
            b = rng.choice("ACGT")
        rd.append(b * min(n, 9))
    rd = "".join(rd)[:250] or "A"
    mask = None
    if rng.random() < 0.3:
        mask = np.zeros(len(ref), np.uint8)
        for _ in range(rng.randint(1, 3)):
            s = rng.randint(0, len(ref) - 1)
            mask[s:min(len(ref), s + rng.randint(1, 90))] = 1
    return ref, rd, mask


def test_align_fuzz_homopolymer_discount(oracle, ref, golden):
    # mia -h: the two extra gap candidates (mia.c:882-905), their place in the cascade, hp_discount_penalty's truncation
    rng = random.Random(431)
    mats = [golden["flat"], golden["ancient"], golden["ancient_rc"], golden["onepass"]]
    used = 0
    for it in range(1200):
        s1, s2, mask = _fuzz_hp(rng) if it % 4 else _fuzz(rng)
        sm, sg5 = rng.choice(mats), rng.randint(0, 1)
        a = ref.align(s1, s2, sm, sg5, mask, matrices=True, hp=1)
        b = oracle.align(s1, s2, sm, sg5, mask, matrices=True, hp=1)
        for k in ("score", "abr", "abc", "aer", "aec", "ref_gapped", "read_gapped"):
            assert a[k] == b[k], (it, k)
        assert (a["S"] == b["S"]).all() and (a["T"] == b["T"]).all(), it
        used += int((a["S"] != oracle.align(s1, s2, sm, sg5, mask, matrices=True)["S"]).any())
    ref.set_hp(0)
    assert used > 300, used              # the discount changed the matrix in that many cases: the candidates are exercised


def test_session_homopolymer_discount(oracle, ref, golden):
    import _pkg
    _pkg.load()
    from mia_b200 import synth
    refseq = _hp_reference(2200, 7)
    g = synth.diverge(refseq, 0.02, seed=3, indel_rate=0.01)
    b, off, _ = synth.make_reads(g, 260, 35, 90, seed=4)
    reads = [synth.read_str(b, off, i) for i in range(260)]
    try:
        _session_compare(oracle, ref, refseq, reads, golden["onepass"], 1, 10, hp=1)
        _session_compare(oracle, ref, refseq, reads[:100], golden["ancient"], 0, 0, hp=1)
    finally:
        ref.set_hp(0)


def _hp_reference(n, seed):
    rng = random.Random(seed)
    out = []
    while sum(len(x) for x in out) < n:
        out.append(rng.choice("ACGT") * min(9, max(1, int(rng.expovariate(0.5)))))
    return "".join(out)[:n]


def test_kmer_table_and_filter(oracle, ref):
    import _pkg
    _pkg.load()
    from mia_b200 import synth
    # low-complexity reference so that the 128-position cap and saturation trigger
    rng = random.Random(5)
    seq = synth.random_reference(1500, seed=9) + "AC" * 400 + "c" * 300 + synth.random_reference(500, seed=10).lower()
    for k, soft in ((6, 0), (8, 1), (11, 0)):
        ft, fo = ref.kmer_new(seq, k, soft), oracle.kmer_build(seq, k, soft)
        for inx in [rng.randrange(4 ** k) for _ in range(300)] + [0, 4 ** k - 1, int("01" * k, 2) if k < 16 else 0]:
            assert (ref.kmer_lookup(ft, inx) == oracle.kmer_lookup(fo, inx)).all()
        for _ in range(150):
            p = rng.randint(0, len(seq) - 80)
            rd = seq[p:p + rng.randint(k - 2 if k > 2 else 1, 70)].upper()
            if rng.random() < 0.3:
                rd = "".join(rng.choice("ACGT") for _ in range(40))
            a = ref.kmer_filter(ft, ft, k, rd, len(seq))
            b = oracle.kmer_filter(fo, fo, k, rd, len(seq))
            assert a[0] == b[0]
            if a[0]:
                assert (a[1] == b[1]).all() and (a[2] == b[2]).all()
        ref.kmer_free(ft, k)
        oracle.kmer_free(fo)


def _session_compare(oracle, ref, refseq, reads, sm, circular, k, soft_mask=0, hp=0):
    with tempfile.NamedTemporaryFile("w", suffix=".fa", delete=False) as f:
        f.write(">ref\n" + refseq + "\n")
        path = f.name
    s = ref.sess_new(path, circular, sm, k=k, soft_mask=soft_mask, hp=hp)
    R = OracleRun(oracle, refseq, sm, circular, k, soft_mask, hp=hp)
    for i, rd in enumerate(reads):
        a, b = ref.sess_pass1(s, "r%d" % i, rd), R.pass1(rd)
        for key in a:
            if not a["hits"] and key not in ("hits", "added"):
                continue
            assert a[key] == b[key], (i, key)
    ref.sess_end_pass1(s)
    R.end_pass1()
    for it in range(30):
        ca, conva = ref.sess_iterate(s, sort=0)
        cb, convb = R.iterate()
        fa = ref.sess_reads(s)
        assert [[x[k2] for k2 in ("score", "as_", "ae", "rc", "seq")] for x in fa] == \
               [[x[k2] for k2 in ("score", "as_", "ae", "rc", "seq")] for x in R.fsdb], it
        sa, sb = ref.sess_slots(s), oracle.asm_entries(R.asm)
        keys = ("start", "end", "score", "revcom", "dropped", "segment", "seq", "smp", "ins")
        assert [[x[k2] for k2 in keys] for x in sa] == [[x[k2] for k2 in keys] for x in sb], it
        gb = oracle.asm_gaps(R.asm, R.wrap_len)
        assert (ref.sess_gaps(s)[:len(gb)] == gb).all()
        assert ca == cb and conva == convb, it
        if conva:
            break
    os.unlink(path)
    return it + 1


def test_session_synthetic(oracle, ref, golden):
    import _pkg
    _pkg.load()
    from mia_b200 import synth
    refseq = synth.random_reference(2500, seed=1)
    g = synth.diverge(refseq, 0.03, seed=3, indel_rate=0.004)
    b, off, _ = synth.make_reads(g, 300, 35, 75, seed=4, n_rate=0.003)
    reads = [synth.read_str(b, off, i) for i in range(300)]
    _session_compare(oracle, ref, refseq, reads, golden["onepass"], 1, 10)
    _session_compare(oracle, ref, refseq, reads[:120], golden["pe"], 0, 0)


def test_score_cut_matches_reference_regression(oracle):
    # a12 is checked through the sessions above (dropped flags); here the product's own host
    # implementation (libmiagpu: miagpu_score_cut) against the oracle's on random data
    import _pkg
    _pkg.load()
    from mia_b200 import api
    rng = np.random.default_rng(3)
    for _ in range(20):
        n = int(rng.integers(5, 4000))
        sl = rng.integers(30, 140, n).astype(np.int32)
        sc = (sl * rng.integers(120, 200, n) + rng.integers(-3000, 800, n)).astype(np.int32)
        assert api.score_cut(sl, sc) == oracle.score_cut(sl, sc)
        below = api.cull_flags(sl, sc)
        s, i = oracle.score_cut(sl, sc)
        s = 100.0 if s <= 0 else s
        assert (below == (sc < (i + s * sl))).all()


def test_repeat_filter_oracle_equals_reference(oracle, ref):
    # f1: sort_fsdb / sort_fsdb_qscore + set_uniq_in_fsdb (fsdb.c:240-252, 440-508) on FSDBs full of ties, both sort keys,
    # both just_outer_coords settings, with and without a tolerance
    rng = np.random.default_rng(1)
    for trial in range(25):
        n = int(rng.integers(1, 3000))
        rc = rng.integers(0, 2, n).astype(np.uint8)
        as_ = rng.integers(0, 60, n).astype(np.int32)
        ae = (as_ + rng.integers(30, 40, n)).astype(np.int32)
        k4 = rng.integers(2000, 2010, n).astype(np.int32)
        tr = rng.integers(0, 2, n).astype(np.uint8)
        for uq in (0, 1):
            for jo in (0, 1):
                for tol in (0, 2):
                    a = oracle.repeat_filter(rc, as_, ae, k4, tr, jo, tol)
                    b = ref.repeat_filter(rc, as_, ae, k4, tr, jo, tol, use_qscore=uq)
                    assert (a[0] == b[0]).all() and (a[1] == b[1]).all(), (trial, uq, jo, tol)


def test_trim_oracle_equals_reference(oracle, ref):
    # f4: trim_frag (mia.c:1318-1368) on reads with damaged adapter prefixes, adapters of 1 .. 44 bases, reads with N
    rng = random.Random(3)
    adapters = ["GTCAGACACGCAACAGGGGATAGGCAAGGCACACAGGGGATAGG", "CTGAGACACGCAACAGGGGATAGGCAAGGCACACAGGGGATAGG", "ACGTTGCA", "A"]
    for t in range(1500):
        ad = rng.choice(adapters)
        rd = "".join(rng.choice("ACGT") for _ in range(rng.randint(1, 120)))
        if rng.random() < 0.6:
            frag = list(ad[: rng.randint(1, len(ad))])
            for i in range(len(frag)):
                y = rng.random()
                if y < 0.05:
                    frag[i] = rng.choice("ACGT")
                elif y < 0.07:
                    frag[i] = ""
                elif y < 0.09:
                    frag[i] += rng.choice("ACGT")
            rd = (rd + "".join(frag))[:256]
        if rng.random() < 0.05:
            rd = rd[: len(rd) // 2] + "N" + rd[len(rd) // 2 + 1:]
        rd = rd or "A"
        assert oracle.trim(rd, ad) == ref.trim(rd, ad), (t, rd, ad)


@pytest.mark.parametrize("checker_name", ["ref", "oracle"])
def test_columns_right_of_the_end_cell_do_not_matter(request, checker_name):
    # What the 16-bit kernels rely on when they hand a gapped read to the 32-bit kernels with its window cut at the end cell
    # (pair16.cuh): every candidate of a dyn_prog cell comes from a lower column (mia.c:838-871) and max_sg_score takes the FIRST
    # maximum of the last row (mia.c:1278-1302), so the alignment against window[0 .. aec] equals the alignment against the whole
    # window -- checked here on the unmodified reference itself and on the oracle, reads with indels, every matrix, both sg5.
    import numpy as np
    import gpu_checks
    checker = request.getfixturevalue(checker_name)
    rng = np.random.default_rng(11)
    n_gapped = 0
    for t in range(300):
        sm = gpu_checks.load_pssm(["onepass", "ancient", "pe", "flat"][t % 4])
        L = int(rng.integers(20, 90))
        W = L + int(rng.integers(20, 130))
        window = "".join("ACGT"[i] for i in rng.integers(0, 4, W))
        s0 = int(rng.integers(0, W - L + 1))
        read = list(window[s0:s0 + L])
        for _ in range(int(rng.integers(0, 4))):                       # a few substitutions, an insert or a deletion
            read[int(rng.integers(0, len(read)))] = "ACGT"[int(rng.integers(0, 4))]
        if t % 3 == 0 and len(read) > 12:
            p = int(rng.integers(4, len(read) - 4))
            read[p:p] = list("ACGT"[int(rng.integers(0, 4))] * int(rng.integers(1, 4)))
        elif t % 3 == 1 and len(read) > 16:
            p = int(rng.integers(4, len(read) - 8))
            del read[p:p + int(rng.integers(1, 4))]
        read = "".join(read)
        for sg5 in (1, 0):
            full = checker.align(window, read, sm, sg5=sg5)
            cut = checker.align(window[: full["aec"] + 1], read, sm, sg5=sg5)
            for k in ("score", "abr", "abc", "aer", "aec", "ref_gapped", "read_gapped"):
                assert cut[k] == full[k], (t, sg5, k, cut[k], full[k])
        n_gapped += "-" in full["ref_gapped"] or "-" in full["read_gapped"]
    assert n_gapped > 60
