"""CPU: the C side of the boundary -- include/miagpu.h is plain C99, miagpu_read_pssm equals the reference's read_pssm
(the golden matrices in tests/golden/pssm.npz came out of the reference's own reader), and the plain-C host
(host/mia_gpu.c) fails loudly without a GPU instead of falling back to anything."""
import json
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "host", "mia_gpu")


import _pkg  # noqa: E402

_pkg.load()
from mia_b200.synth import matrix_text  # noqa: E402,F401


def ensure_host():
    """host/mia_gpu is built by __graft_entry__.build(); build it here if a fresh checkout has not run that yet"""
    if not os.path.exists(HOST):
        pkg = os.path.join(ROOT, "mapping-iterative-assembler_b200")
        subprocess.run(["gcc", "-std=c99", "-O2", "-I" + os.path.join(ROOT, "include"), "-o", HOST, os.path.join(ROOT, "host", "mia_gpu.c"),
                        "-L" + pkg, "-lmiagpu", "-Wl,-rpath,$ORIGIN/../mapping-iterative-assembler_b200"], check=True)
    return HOST


def _api():
    import _pkg
    _pkg.load()
    from mia_b200 import api
    return api


def test_header_is_plain_c99(tmp_path):
    src = tmp_path / "t.c"
    src.write_text('#include "miagpu.h"\nint main(void) { miagpu_maln_header h; miagpu_maln_reads r; (void)h; (void)r; return MIAGPU_MAX_READ == 256 ? 0 : 1; }\n')
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-fsyntax-only", "-I" + os.path.join(ROOT, "include"), str(src)], check=True)


@pytest.mark.parametrize("name", ["ancient", "onepass", "pe", "ancient_rc"])
def test_read_pssm_equals_reference(golden, name, tmp_path):
    api = _api()
    p = tmp_path / "m.txt"
    p.write_text(matrix_text(golden[name]))
    got = api.read_pssm(str(p)).reshape(-1)
    want = np.asarray(golden[name]).reshape(31, 5, 5).copy()
    want[:, :4, 4] = -100                                  # io.c:443-448: N column / non-ACGT reference row are constants
    want[:, 4, :] = -10
    assert (got == want.reshape(-1)).all()


def test_read_pssm_shipped_files_and_errors(golden, tmp_path):
    api = _api()
    # the text of the reference's matrices/ancient.submat.solexa.onepass.txt, stored with the golden vectors
    shipped = tmp_path / "ancient.submat.solexa.onepass.txt"
    shipped.write_text(json.load(open(os.path.join(ROOT, "tests", "golden", "onepass_matrix_fixture.json")))["text"])
    assert (api.read_pssm(str(shipped)).reshape(-1) == golden["onepass"]).all()
    bad = tmp_path / "bad.txt"
    bad.write_text(matrix_text(golden["ancient"]).replace("MIDDLE", "16"))
    with pytest.raises(api.MiaGpuError, match="MIDDLE"):
        api.read_pssm(str(bad))
    with pytest.raises(api.MiaGpuError, match="cannot open"):
        api.read_pssm(str(tmp_path / "none.txt"))


def test_c_host_has_no_cpu_fallback(golden, tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    ensure_host()
    (tmp_path / "m.txt").write_text(matrix_text(golden["ancient"]))
    (tmp_path / "r.fa").write_text(">r\nACGTACGTACGTACGTACGT\n")
    (tmp_path / "q.fq").write_text("@a\nACGTACGTAC\n+\nIIIIIIIIII\n")
    r = subprocess.run([HOST, "-r", "r.fa", "-f", "q.fq", "-s", "m.txt", "-m", "out"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 1 and "no CUDA device" in r.stderr and "no CPU fallback" in r.stderr
    assert not os.path.exists(tmp_path / "out.1")


def test_c_host_argument_errors(golden, tmp_path):
    # what the host refuses, it refuses before touching the GPU: reference options it does not carry, missing files
    ensure_host()
    run = lambda *a: subprocess.run([HOST] + list(a), cwd=tmp_path, capture_output=True, text=True)
    r = run()
    assert r.returncode == 2 and "usage: mia_gpu" in r.stderr
    for opt in ("-T", "-C3", "-I"):
        r = run("-r", "r.fa", "-f", "q.fq", "-s", "m.txt", opt)
        assert r.returncode == 2 and "not handled by this host" in r.stderr, opt
    r = run("-r", "r.fa", "-f", "q.fq", "-s", "m.txt", "-u", "-H", "3000")
    assert r.returncode == 2 and "-u / -U" in r.stderr
    r = run("-r", "r.fa", "-f", "q.fq", "-s", "m.txt", "-u", "-D")
    assert r.returncode == 2 and "-u / -U" in r.stderr
    (tmp_path / "r.fa").write_text(">r\nACGTACGTACGTACGTACGT\n")
    (tmp_path / "q.fq").write_text("@a\nACGTACGTAC\n+\nIIIIIIIIII\n")
    r = run("-r", "r.fa", "-f", "q.fq", "-s", "none.txt")
    assert r.returncode == 1 and "miagpu_read_pssm" in r.stderr and "cannot open" in r.stderr
    (tmp_path / "m.txt").write_text(matrix_text(golden["ancient"]).replace("MIDDLE", "16"))
    r = run("-r", "r.fa", "-f", "q.fq", "-s", "m.txt")
    assert r.returncode == 1 and "MIDDLE" in r.stderr
    r = run("-r", "missing.fa", "-f", "q.fq", "-s", "m.txt")
    assert r.returncode == 1 and "cannot read reference" in r.stderr
