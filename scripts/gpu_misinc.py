"""GPU: what the damage profile (miagpu_misincorporation) costs after one resident round of the benchmark's default workload
(bench.make_workload: 1 M reads of 35-75 bp, 16.5 kb circular reference, onepass matrix):
    python scripts/gpu_misinc.py [reads] [calls]
Prints the round time (CUDA events on the library's stream, median of 10 warm rounds), the call's kernel time (the library's own
events around memset + kernel, miagpu_last_timing) and its whole time with the download (events around the call on the library's
stream) over `calls` warm calls, the bytes the walk has to read with the HBM floor they give, and the card with its power limit,
read in the same run.  The working set (146 MB at one run per read) is larger than the 126 MB L2, and each call reads it once."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import _pkg
_pkg.load()
from mia_b200 import api
import bench

HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name(0) + " (power limit: nvidia-smi unavailable)"


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
    calls = int(sys.argv[2]) if len(sys.argv) > 2 else 200
    ref, bases, off, rc, as_, ae = bench.make_workload(n, seed=1000)
    g = api.MiaGpu(0)
    g.set_pssm(bench.load_pssm("onepass"))
    g.set_reference(ref, circular=1, with_rc=0)
    g.upload_reads(bases, off)
    g.set_alignment_inputs(rc, as_, ae)
    g.set_cut_inputs(np.diff(off).astype(np.int32))
    st = torch.cuda.ExternalStream(g.lib.miagpu_stream(g.h), device=torch.device("cuda", 0))
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def timed(fn, k):
        out = []
        for _ in range(k):
            a, b = ev(), ev()
            a.record(st)
            fn()
            b.record(st)
            b.synchronize()
            out.append(a.elapsed_time(b))
        return out

    def round_():
        g.reset_dropped()                               # every round starts from the same state
        g.iterate_resident()
    for _ in range(3):
        round_()
    round_ms = timed(round_, 10)
    t = g.misincorporation()
    for _ in range(10):
        assert (g.misincorporation() == t).all()
    kern, whole = [], []
    for _ in range(calls):
        whole += timed(g.misincorporation, 1)
        kern.append(g.last_timing()["ms_kernels"])
    # what the walk reads: the entries (2 per read, 32 bytes), every read's run list (its n_runs words), bases, per-read words
    # (n_runs, abr, rc: 4 + 4 + 1 bytes; two 8-byte offsets)
    al = g.get_alignment()
    runs = int(np.maximum(al["n_runs"], 0).sum())
    nbytes = dict(entries=2 * n * 32, runs=2 * runs, bases=int(off[-1]), per_read=n * (4 + 4 + 1 + 16))
    total = sum(nbytes.values())
    ct0 = float(t[0, 1, 3] / max(1, t[0, 1].sum()))
    res = dict(card=card(), reads=n, round_ms_median=float(np.median(round_ms)), calls=calls,
               kernel_us_median=1e3 * float(np.median(kern)), kernel_us_min=1e3 * float(np.min(kern)),
               call_with_download_us_median=1e3 * float(np.median(whole)), bytes=nbytes, bytes_total=total,
               hbm_floor_us=1e6 * total / HBM_BYTES_PER_S, share_of_round=float(np.median(kern) / np.median(round_ms)),
               table_total=int(t.sum()), ct_depth0=ct0)
    print(f"card: {res['card']}")
    print(f"round (iterate_resident, {n} reads): {res['round_ms_median']:.3f} ms median of 10")
    print(f"miagpu_misincorporation over {calls} warm calls: kernel (memset + misinc_kernel) {res['kernel_us_median']:.1f} us median, "
          f"{res['kernel_us_min']:.1f} us min; with the 9 kB download {res['call_with_download_us_median']:.1f} us median")
    print(f"bytes the walk reads: {total / 1e6:.1f} MB {nbytes} -> HBM floor {res['hbm_floor_us']:.1f} us at 7.7 TB/s")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
