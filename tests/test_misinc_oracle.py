"""CPU: the damage profile's definition (include/miagpu.h, miagpu_misincorporation) as a `.maln`-to-table oracle, checked against a
hand-written file whose table is written out by hand; and the hosts' -d option refusing a missing file name before touching a GPU.
tests/test_gpu_misinc.py compares the device's tables with this oracle on the unmodified reference binary's `.maln` files."""
import os
import subprocess

import numpy as np
import pytest

from test_hostio import parse_maln
from test_host_c import ensure_host, HOST

CODES = "ACGTN-"
COMP = [3, 2, 1, 0, 4, 5]                  # A<->T, C<->G; N and - stay


def _code(ch):
    i = CODES.find(ch)
    return 4 if i < 0 else i


def misinc_table(body):
    """the misincorporation table of a `.maln` file (after its first line): int64[31, 6, 6], depth x reference x read over A C G T N -"""
    h, seqs = parse_maln(body)
    t = np.zeros((31, 6, 6), np.int64)
    L, ref = h["len"], h["seq"]
    for a in seqs:
        if a["dr"]:
            continue
        rev = a["rc"] == 1
        for c, ch in enumerate(a["seq"]):
            pos = a["start"] + c
            if pos >= L:
                continue
            d = ord(a["smp"][c]) - ord("A")
            r, q = _code(ref[pos]), _code(ch)
            ins = [_code(b) for b in a["ins"].get(c, "")]
            if rev:
                d, r, q, ins = 30 - d, COMP[r], COMP[q], [COMP[b] for b in ins]
            t[d, r, q] += 1
            for b in ins:
                t[d, 5, b] += 1
    return t


def read_damage_file(path):
    """the text the hosts write with -d -> int64[31, 6, 6]"""
    lines = open(path).read().split("\n")
    assert lines[0] == "depth\tref\tread\tcount" and lines[-1] == ""
    rows = [ln.split("\t") for ln in lines[1:-1]]
    assert len(rows) == 31 * 36
    for k, (d, r, q, _) in enumerate(rows):
        assert (int(d), r, q) == (k // 36, CODES[k // 6 % 6], CODES[k % 6]), k
    return np.array([int(x[3]) for x in rows], np.int64).reshape(31, 6, 6)


def _record(rid, start, rc, dr, seq, smp, ins=""):
    return "\n".join([f"ID {rid}", "DESC ", "SCORE 3000", "NUM_INPUTS 1", f"START {start}", f"END {start + len(seq) - 1}", f"RC {rc}", "TR 0",
                      f"DR {dr}", "SEG a", f"SEQ {seq}", f"SMP {smp}", "INS_POS" + (" " + ins if ins else "")])


def _maln(ref, records):
    pssm = "".join(f"{w}:\n" + "".join("0 0 0 0 0\n" * 5 + "\n" for _ in range(31)) for w in ("FPSM", "RPSM"))
    head = (f"MALN_NAS {len(records)}\nMALN_SIZ {len(records)}\nMALN_COC 1\n__REFERENCE__\nID r\nDESC \nLEN {len(ref)}\nSIZE {len(ref)}\n"
            f"SEQ {ref}\nGAPS" + " 0" * len(ref) + f"\n__PSSM__\nDEPTH 15\n{pssm}__ALNSEQS__\n")
    return head + "".join(r + "\n" for r in records)


def test_oracle_on_a_hand_written_maln():
    body = _maln("ACGTACGTACGT", [
        # forward: ref A C G T A against read A C T T A, depths 0..4
        _record("fw", 0, 0, 0, "ACTTA", "ABCDE"),
        # reverse strand: a deletion in column 1, two inserted bases (T G) in front of column 2; depths 30, 29, 28, 27 mirror to 0..3
        _record("rv", 2, 1, 0, "G-AC", "_^]\\", "2 TG"),
        # dropped: counts nowhere
        _record("dr", 0, 0, 1, "AAAA", "AAAA"),
        # columns 2 and 3 (and the insert in front of column 2) lie at or past LEN; an N in the read
        _record("end", 10, 0, 0, "GNNA", "PPQR", "2 C"),
    ])
    want = np.zeros((31, 6, 6), np.int64)
    A, C, G, T, N, GAP = range(6)
    for d, r, q in [(0, A, A), (1, C, C), (2, G, T), (3, T, T), (4, A, A),          # fw
                    (0, C, C), (1, A, GAP), (2, T, T), (2, GAP, A), (2, GAP, C), (3, G, G),   # rv, complemented and mirrored
                    (15, G, G), (15, T, N)]:                                        # end
        want[d, r, q] += 1
    got = misinc_table(body)
    assert (got == want).all(), np.argwhere(got != want).tolist()


@pytest.mark.parametrize("prog", ["mia_gpu", "mia_gpu_mg"])
def test_damage_option_without_a_file_is_a_usage_error(prog, tmp_path):
    ensure_host()
    exe = os.path.join(os.path.dirname(HOST), prog)
    if not os.path.exists(exe):
        pytest.skip(f"host/{prog} not built (mia_gpu_mg needs nccl.h / libnccl at build time)")
    r = subprocess.run([exe, "-r", "r.fa", "-f", "q.fq", "-s", "m.txt", "-d"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 2 and "-d needs a file name" in r.stderr, r.stderr
    r = subprocess.run([exe], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 2 and "[-d damage.tsv" in r.stderr and "extension of this host" in r.stderr
