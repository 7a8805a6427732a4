#!/usr/bin/env python
"""bench.py -- MIA per-iteration hot path on B200 (BASELINE.json metric/config).

A "step" is ONE ITERATION of the hot path over one batch of synthetic aDNA reads:
windowed PSSM semi-global DP + on-device traceback of every read against the current
consensus (reiterate_assembly, mia_main.c:178-257), then per-column accumulation and base
calling (consensus_assembly_string, mia.c:515-603).  Workload at N=1 is BASELINE.json
configs[1]: 1 M synthetic 35-75 bp aDNA-damaged reads vs a 16,569 bp circular reference,
ancient.submat.solexa.onepass, single iteration.  The step also holds the iteration's score cut
(cull_maln_from_fsdb / find_fsdb_score_cut, mia.c:418-479, fsdb.c:269-383) between the two, at every N.
Reads shard across ranks (weak scaling: 1 M reads per GPU, consensus replicated; per round one
all-reduce MAX (insert maxima, best scores, the ranks' integer sums), one all-gather of the regression's
block records (~50 B per 512 reads) and one all-reduce SUM of the column planes over NCCL, enqueued on
the library's stream: mia_b200/shard.py).

  value : reads/s, whole job, inputs resident in HBM, device time (CUDA events on the
          library's stream), max over ranks.
  e2e   : the same through the C ABI with HOST buffers (miagpu_iterate_host): H2D of reads +
          rc/as/ae/seq_len/flags from pinned memory, realign, score cut, consensus, D2H of the
          per-read results, packed run lists, flags and consensus -- wall clock around the call.
  --impl reference : the unmodified reference (oracle/_ref, built from /root/reference/src)
          running its own per-read realign sequence on the host cores, one process per core
          on disjoint shards (the reference itself is single-threaded).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "aligned reads/sec per iteration (windowed PSSM DP + traceback + score cut + consensus)"
UNIT = "reads/s"
REF_LEN = 16569
INT_OPS_PER_CELL = 15          # SURVEY.md 8d: minimum straight-line INT32 work per DP cell


def load_pssm(name="onepass"):
    return np.load(os.path.join(ROOT, "tests", "golden", "pssm.npz"))[name]


def make_workload(n_reads, seed, ref=None, divergence=0.005, indel_rate=0.0, min_len=35, max_len=75):
    import _pkg
    _pkg.load()
    from mia_b200 import synth
    ref = ref or synth.random_reference(REF_LEN, seed=1)
    genome = synth.diverge(ref, divergence, seed=2, indel_rate=indel_rate)
    bases, off, truth = synth.make_reads(genome, n_reads, min_len, max_len, seed=seed)
    rc = truth["strand"].astype(np.uint8)
    # stored orientation: reverse-strand reads are kept reverse-complemented (fsdb.c:209-227)
    comp = np.zeros(256, np.uint8)
    for a, b in zip(b"ACGTN", b"TGCAN"):
        comp[a] = b
    rid = np.repeat(np.arange(n_reads), np.diff(off))
    pos = np.arange(len(bases)) - off[rid]
    src = np.where(rc[rid] == 1, off[rid] + (off[rid + 1] - off[rid]) - 1 - pos, np.arange(len(bases)))
    stored = np.where(rc[rid] == 1, comp[bases[src]], bases)
    as_ = np.minimum(truth["start"], len(ref) - 1).astype(np.int32)      # (a sample with indels is a little longer / shorter than the reference)
    ae = (as_ + truth["length"] - 1).astype(np.int32)
    return ref, np.ascontiguousarray(stored, np.uint8), off, rc, as_, ae


def windows(off, as_, ae, wrap_len):
    """mia_main.c:190-212"""
    L = np.diff(off).astype(np.int64)
    rs = np.maximum(as_.astype(np.int64) - 50, 0)
    re = np.where(ae.astype(np.int64) + 51 > wrap_len, wrap_len, ae.astype(np.int64) + 50)
    whole = rs + L > re
    rs = np.where(whole, 0, rs)
    re = np.where(whole, wrap_len, re)
    return rs.astype(np.int32), (re - rs).astype(np.int32)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.start = [], None, 0
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def mark(self):
        """samples before this point (start-up, warm-up) are dropped"""
        self.start = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        self.rows = self.rows[self.start:]
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs next to its GPU (sysfs local_cpulist of the GPU's PCI function), so that the pinned host buffers
    of the end-to-end arm are first touched on the GPU's own NUMA node: with one process per GPU on a two-socket host half of the
    uploads otherwise cross the socket interconnect.  Returns the CPU list, or None when the information is not there."""
    try:
        bdf = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=10).stdout.strip().lower()
        if bdf.startswith("00000000:"):
            bdf = bdf[4:]
        cpus = open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        ids &= os.sched_getaffinity(0)
        if ids:
            os.sched_setaffinity(0, ids)
            return cpus
    except Exception:
        pass
    return None


def run_ours(args):
    import torch
    import torch.distributed as dist
    import _pkg
    _pkg.load()
    from mia_b200 import api

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None       # before any pinned buffer is allocated (first touch decides the node)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.reads
    ref, bases, off, rc, as_, ae = make_workload(n, seed=1000 + rank)
    sm = load_pssm("onepass")
    g = api.MiaGpu(local)
    g.set_pssm(sm)
    g.set_reference(ref, circular=1, with_rc=0)
    lib_stream = torch.cuda.ExternalStream(g.lib.miagpu_stream(g.h), device=torch.device("cuda", local))
    seq_len = np.diff(off).astype(np.int32)

    from mia_b200 import shard
    S = shard.ShardedRounds(g, local, world, rank, n) if world > 1 else None     # weak scaling: n reads on every rank

    launches = {"n": 0}

    def step_resident():
        """the whole round on resident inputs: realign, score cut, consensus (N > 1: the sharded protocol,
        2 all-reduces + 1 small all-gather over NCCL on the library's stream; same work per read at every N)"""
        g.reset_dropped()                               # every timed step starts from the same state
        cons, cut, _ = g.iterate_resident() if world == 1 else S.resident()
        launches["n"] += g.last_timing()["launches"]
        return cons, cut

    # pinned host buffers for the end-to-end path
    def pin(a):
        t = torch.from_numpy(a).pin_memory()
        return t
    h_bases, h_off, h_rc, h_as, h_ae = pin(bases), pin(off), pin(rc), pin(as_), pin(ae)
    h_out = api.MiaGpu.alloc_realign_outputs(n, pinned=True)
    del h_out["runs"]                                   # run lists come back packed (sum(n_runs) words, not n*24)
    h_packed = torch.empty(4 * n, dtype=torch.int16).pin_memory()
    packed_total = {"n": 0}

    h_seq_len = pin(seq_len)
    dropped = torch.zeros(n, dtype=torch.uint8).pin_memory()

    def step_e2e():
        """one call sequence through the C ABI with host buffers: upload, realign, score cut, consensus, downloads"""
        dropped.zero_()                                 # every timed step starts from the same state
        if world == 1:
            cons, _, tot, _ = g.iterate_host(h_bases, h_off, h_rc, h_as, h_ae, h_seq_len, dropped, h_out, h_packed)
        else:
            cons, _, tot, _ = S.host(h_bases, h_off, h_rc, h_as, h_ae, h_seq_len, dropped, h_out, h_packed)
        packed_total["n"] = tot
        return cons

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident arm: device time per step via events on the library's stream
    g.upload_reads(bases, off)
    g.set_alignment_inputs(rc, as_, ae)
    g.set_cut_inputs(seq_len)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    sampler = ClockSampler(local) if rank == 0 else None      # nvidia-smi needs a few hundred ms to start: launched before the warm-up
    for _ in range(max(args.warmup, 3)):
        cons, _ = step_resident()
    tim = g.last_timing()
    barrier()
    if sampler:
        t_wait = time.perf_counter()
        while not sampler.rows and time.perf_counter() - t_wait < 3.0:      # first sample in: the sampling loop is running
            time.sleep(0.01)
        sampler.mark()
    barrier()
    launches["n"] = 0
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for k in range(args.steps):
        flush.zero_()                       # L2 flush between timed iterations (outside the timed events)
        barrier()
        ev[k][0].record(lib_stream)
        cons, cut = step_resident()
        ev[k][1].record(lib_stream)
        torch.cuda.synchronize()
    barrier()
    if args.dump_outputs and rank == 0:
        # what a caller of the round receives: the consensus and the cut here, the per-read alignment and the run lists
        # from the device (miagpu_get_alignment + miagpu_get_runs_packed), before the per-class timing below overwrites them
        total_runs = g.get_runs_packed()[0]
        packed = g.get_runs_packed(None, np.zeros(total_runs, np.uint16))[2]
        dumped = {"consensus": cons, "score_cut": cut, "aln": g.get_alignment(), "runs": packed}
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = float(sum(step_ms))
    # resident realigns on the measurement path (one width class after the other, events around each) just to read the
    # per-class kernel times; the first call only sizes that path's scratch buffers
    g.realign_resident()
    g.realign_resident()
    buckets = [dict(b, kernel=f"realign_kernel<{b['K']}>") for b in g.last_buckets()]
    pbuckets, n_fallback, lmax16 = g.last_pair_buckets()
    pbuckets = [dict(b, kernel=f"pair16_kernel<{b['K']}>") for b in pbuckets]
    tim_realign = g.last_timing()
    dom = max(buckets + pbuckets, key=lambda x: x["ms"])
    int_peak = g.int32_peak()

    # ---- end-to-end arm
    for _ in range(2):
        step_e2e()
    barrier()
    e2e_times = []
    for k in range(args.steps):
        flush.zero_()
        barrier()
        t0 = time.perf_counter()
        cons_e2e = step_e2e()
        torch.cuda.synchronize()
        e2e_times.append(time.perf_counter() - t0)
    barrier()
    clocks = sampler.stop() if sampler else None
    e2e_total = float(sum(e2e_times))
    if args.dump_outputs and rank == 0:
        e2e = {"consensus": cons_e2e, "aln": {k: v.numpy() for k, v in h_out.items()}, "dropped": dropped.numpy(),
               "runs": h_packed[: packed_total["n"]].numpy().view(np.uint16)}
        dump_outputs(args.dump_outputs, dumped, e2e, n)

    if world > 1:
        t = torch.tensor([total_ms, e2e_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_total = t.tolist()
    cut_stats = g.last_cut_stats()
    parity = None
    if not args.no_parity:
        parity = parity_block(g, args, world, rank, local, ref, bases, off, rc, as_, ae, sm, cons)
        g.set_reference(ref, circular=1, with_rc=0)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ms_per_step = total_ms / args.steps
    value = world * n / (ms_per_step * 1e-3)
    cells = tim_realign["dp_cells"]
    gcups = world * cells / (ms_per_step * 1e-3) / 1e9
    h2d = world * int(len(bases) + off.nbytes + rc.nbytes + as_.nbytes + ae.nbytes + seq_len.nbytes + n)
    d2h = world * int(sum(v.numel() * v.element_size() for v in h_out.values()) + 2 * packed_total["n"] + len(cons_e2e) + n)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    # algorithmic bytes of the dominant realign launch: read bases + offset(8) + rc/as/ae(9) in,
    # score/as/ae/abr/n_runs/status(21) + one run word(2) out, per read
    # DRAM traffic and SASS warp instructions of the dominant kernel: from the committed ncu capture of THIS round's build
    # (profiles/r02_kernels.json, written by profiles/summarize.py from the .ncu-rep), per read / per cell of the captured launch
    traffic, traffic_src, ipc, ipc_src = None, None, None, None
    try:
        kj = json.load(open(os.path.join(ROOT, "profiles", "r02_kernels.json")))
        ent = kj.get(dom["kernel"]) or next((v for k, v in kj.items() if k.split("<")[0] == dom["kernel"].split("<")[0]), None)
        if ent:
            traffic = ent["dram_bytes_per_launch"] / ent["reads_per_launch"] * dom["reads"]
            ipc = ent["warp_inst_per_launch"] / ent["cells_per_launch"]
            traffic_src = ipc_src = ent["source"]
    except Exception:
        pass
    frac_reads = dom["reads"] / n
    alg_bytes = frac_reads * (len(bases) + n * (8 + 9 + 21 + 2))
    dom_s = dom["ms"] * 1e-3
    clk = (clocks or {}).get("sm_mhz") or 1965.0
    issue_peak = 4 * 148 * clk / 1e3                    # G warp instructions / s: 4 schedulers x 148 SMs x SM clock under load
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
        "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: 1M synthetic 35-75 bp aDNA-damaged reads per GPU vs 16,569 bp circular "
                               "R-rand reference, ancient.submat.solexa.onepass, single iteration (realign + score cut + consensus)",
                   "reads_per_gpu": n, "ref_len": REF_LEN, "l2": "256 MiB buffer written between timed steps",
                   "host_cpus_of_rank0": numa,
                   "parallelism": f"reads sharded x{world}, consensus replicated; per round all-reduce MAX (insert maxima + the ranks' sums) + "
                                  f"all-gather (regression block records, ~50 B per 512 reads) + all-reduce SUM (column planes) over NCCL on the library stream"},
        "gcups": gcups, "dp_cells_per_step": world * cells,
        "e2e": {"value": world * n / (e2e_total / args.steps), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_total / args.steps * 1e3,
                "ms_min_median_max": [round(float(np.min(e2e_times)) * 1e3, 3), round(float(np.median(e2e_times)) * 1e3, 3),
                                      round(float(np.max(e2e_times)) * 1e3, 3)]},
        "gpu_launches": launches["n"],
        "clocks": clocks,
        # the bound of the dominant kernel is the issue slot (max-plus recurrence in 16x2 SIMD: no dense contraction, ~0.01 B per cell):
        # SASS warp instructions per cell (ncu smsp__inst_executed.sum / cells of the captured launch) x cells/s of the launch timed
        # here, against 4 schedulers x 148 SMs x the SM clock sampled under load
        "roofline": {"bound": "issue", "achieved": None if ipc is None else ipc * dom["cells"] / dom_s / 1e9, "peak": issue_peak,
                     "unit": "G warp-inst/s", "frac": None if ipc is None else ipc * dom["cells"] / dom_s / 1e9 / issue_peak,
                     "traffic": traffic, "traffic_algorithmic": alg_bytes, "warp_inst_per_cell": ipc, "source": ipc_src,
                     "kernel": dom["kernel"], "kernel_ms": dom["ms"], "kernel_reads": dom["reads"], "kernel_gcups": dom["cells"] / dom_s / 1e9,
                     "kernel_share_of_step": dom["ms"] / ms_per_step, "sm_mhz": clk,
                     "peak_source": "4 x 148 x SM clock (nvidia-smi median during the timed region)",
                     # the tighter view of the same bound: 84 of the row loop's 164 SASS instructions (K = 11) are ALU-pipe instructions
                     # (VIMNMX* / VIADDMNMX / LOP3 .U16x2), and that pipe takes one warp instruction per two cycles and scheduler
                     "alu_pipe": None if ipc is None else {"share_of_instructions": 84 / 164, "peak": issue_peak / 2, "unit": "G warp-inst/s",
                                                           "frac": ipc * (84 / 164) * dom["cells"] / dom_s / 1e9 / (issue_peak / 2),
                                                           "source": "cuobjdump -sass of pair16_kernel<11,16> (DESIGN 4.2); ncu sm__inst_executed_pipe_alu 63 % (profiles/r02j_ncu_pair16_full.md)"}},
        "roofline_hbm": {"bound": "hbm", "achieved": alg_bytes / dom_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": alg_bytes / dom_s / 1e9 / hbm_peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst)" if peaks else "fallback 6650 GB/s",
                         "note": "reported to show that HBM is NOT the limiter"},
        "roofline_int32": {"bound": "int32 ops", "achieved": INT_OPS_PER_CELL * dom["cells"] / dom_s / 1e12,
                           "peak": int_peak / 1e12, "unit": "Tops/s", "frac": INT_OPS_PER_CELL * dom["cells"] / dom_s / int_peak,
                           "ops_per_cell": INT_OPS_PER_CELL,
                           "peak_source": "miagpu_int32_peak micro-benchmark (32-bit IADD3 / IMNMX / SEL), same run",
                           "note": "the pair kernels do TWO 16-bit cells per 32-bit SIMD operation, so SURVEY 8d's 15-ops-per-cell figure can "
                                   "exceed the 32-bit peak (frac > 1): not a roofline, kept for comparison with the 32-bit kernels"},
        "buckets": pbuckets + buckets,
        "pair16": {"reads_handed_to_32bit_kernels": n_fallback, "max_read_len": lmax16},
        "consensus_matches_e2e": bool(cons == cons_e2e),
        "score_cut": cut_stats,
        "parity": parity,
    }
    # ---- the other read shapes of BASELINE.json (indel-bearing divergent reads, 30-140 bp merged pairs), with their own parity checks
    if world == 1 and not args.no_shapes:
        line["shapes"] = shaped_rounds(g, args, flush, lib_stream)
    # ---- the same round on R-mt (SURVEY 8d: the reference's mt311 consensus, real composition and low-complexity stretches)
    if world == 1 and not args.no_rmt:
        line["r_mt"] = rmt_numbers(g, args, flush, lib_stream)
    # ---- pass 1 (k-mer seeding + whole-reference both-strand DP), reported beside the headline
    if world == 1 and not args.no_pass1:
        line["pass1"] = pass1_numbers(g, ref, bases, off, rc, args)
    # ---- the widened rows (SURVEY 8f) and a whole assembly, measured beside the headline
    if world == 1 and not args.no_extras:
        line["extras"] = extras(g, ref, bases, off, rc, as_, ae, sm)
    # ---- CPU baseline: the reference's own realign sequence on a bounded sample, 1 thread
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline(ref, bases, off, rc, as_, ae, sm, args.cpu_sample)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_READS = 200_000            # per-read sample of --dump-outputs: 13 arrays, 2 x 24 run words and an index, at most 51 MB


def _runs_of(packed, n_runs, idx):
    """the packed run words of reads idx (sorted) out of a read-order packing with n_runs words per read"""
    first = np.concatenate(([0], np.cumsum(n_runs, dtype=np.int64)))[idx]
    lens = n_runs[idx].astype(np.int64)
    start = np.concatenate(([0], np.cumsum(lens)))
    return packed[np.repeat(first - start[:-1], lens) + np.arange(start[-1])]


def dump_outputs(d, resident, e2e, n):
    """--dump-outputs: what the last timed step of each arm handed back -- consensus (byte codes), score cut (slope, intercept),
    per-read alignment and packed run lists, and from the end-to-end arm also the sticky dropped flags -- as DIR/<name>.npy,
    float32 (float64 for the cut and the read indices).  The inputs are a function of the arguments, so two builds run with the
    same arguments can be compared file by file.  Per-read arrays cover a fixed seeded sample of DUMP_READS reads when there
    are more (read indices in reads.npy)."""
    os.makedirs(d, exist_ok=True)
    idx = np.arange(n) if n <= DUMP_READS else np.sort(np.random.default_rng(0).choice(n, DUMP_READS, replace=False))
    out = {"reads": idx.astype(np.float64)}
    for prefix, arm in (("", resident), ("e2e_", e2e)):
        out[prefix + "consensus"] = np.frombuffer(arm["consensus"].encode(), np.uint8).astype(np.float32)
        for k, v in arm["aln"].items():
            out[prefix + k] = v[idx].astype(np.float32)
        out[prefix + "runs"] = _runs_of(arm["runs"], arm["aln"]["n_runs"], idx).astype(np.float32)
    out["score_cut"] = np.asarray(resident["score_cut"], np.float64)
    out["e2e_dropped"] = e2e["dropped"][idx].astype(np.float32)
    for k, v in out.items():
        np.save(os.path.join(d, k + ".npy"), v)


def parity_block(g, args, world, rank, local, ref, bases, off, rc, as_, ae, sm, cons_full):
    """Untimed: ties what was just measured to the CPU checker (oracle/_ref = the unmodified reference where it was built).
    (1) the first `--parity-reads` reads of rank 0's workload through one resident round on ONE GPU: every read's score / as /
    ae / abr / gapped strings and the round's consensus against the checker; (2) N > 1: every rank holds the same consensus
    after the timed sharded round, and the sharded round over that common prefix (each rank its contiguous slice) gives the
    consensus of the one-GPU round of (1)."""
    import hashlib
    import torch
    import torch.distributed as dist
    import gpu_checks
    from mia_b200 import shard
    P = min(args.parity_reads, len(off) - 1)
    out = {}
    # rank 0's workload is a function of its seed: every rank regenerates its prefix
    if rank == 0:
        r0 = (ref, bases, off, rc, as_, ae)
    else:
        r0 = make_workload(args.reads, seed=1000)
    _, b0, o0, rc0, as0, ae0 = r0
    pb, po = np.ascontiguousarray(b0[: o0[P]]), np.ascontiguousarray(o0[: P + 1])
    if world > 1:
        h = int(hashlib.md5(cons_full.encode()).hexdigest()[:15], 16)
        t = torch.tensor([h], dtype=torch.int64, device="cuda")
        allh = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allh, t)
        out["ranks_hold_one_consensus"] = bool(all(int(x) == h for x in allh))
        # the sharded round over the common prefix
        lo, hi = P * rank // world, P * (rank + 1) // world
        g.set_reference(ref, circular=1, with_rc=0)
        g.upload_reads(np.ascontiguousarray(pb[po[lo]:po[hi]]), np.ascontiguousarray(po[lo:hi + 1] - po[lo]))
        g.set_alignment_inputs(rc0[lo:hi], as0[lo:hi], ae0[lo:hi])
        g.set_cut_inputs(np.diff(po[lo:hi + 1]).astype(np.int32))
        Sp = shard.ShardedRounds(g, local, world, rank, -(-P // world))
        cons_sh = Sp.resident()[0]
        hs = int(hashlib.md5(cons_sh.encode()).hexdigest()[:15], 16)
        t = torch.tensor([hs], dtype=torch.int64, device="cuda")
        dist.all_gather(allh, t)
        out["sharded_prefix_ranks_agree"] = bool(all(int(x) == hs for x in allh))
    if rank == 0:
        t0 = time.perf_counter()
        res = gpu_checks.round_parity(g, ref, pb, po, rc0[:P], as0[:P], ae0[:P], sm)
        cons_1 = res.pop("consensus")
        out.update(res)
        if world > 1:
            out["sharded_equals_single_gpu"] = bool(cons_sh == cons_1)
        out["wall_s"] = round(time.perf_counter() - t0, 1)
    return out


def shaped_rounds(g, args, flush, lib_stream):
    """The resident round on the other BASELINE read shapes, 1 GPU, beside the headline (same timing rules): configs[3] -- reads of
    a sample 10 % + 0.5 % indels away from the reference they are realigned to (the first rounds of a divergent-seed assembly:
    about every fourth read carries a gap) -- and configs[2] -- merged paired-end reads, 30-140 bp, ancient.submat.solexa.pe.
    Each with its own parity check of a prefix against the CPU checker."""
    import torch
    import gpu_checks
    res = {}
    for tag, kw, mat in (("c4_divergent_indels", dict(divergence=0.10, indel_rate=0.005), "ancient"),
                         ("c3_merged_pe_30_140", dict(divergence=0.005, indel_rate=0.0005, min_len=30, max_len=140), "pe")):
        n = args.reads
        sm = load_pssm(mat)
        ref, bases, off, rc, as_, ae = make_workload(n, seed=3000, **kw)
        g.set_pssm(sm)
        g.set_reference(ref, circular=1, with_rc=0)
        g.upload_reads(bases, off)
        g.set_alignment_inputs(rc, as_, ae)
        g.set_cut_inputs(np.diff(off).astype(np.int32))
        for _ in range(3):
            g.reset_dropped()
            g.iterate_resident()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for k in range(args.steps):
            flush.zero_()
            torch.cuda.synchronize()
            ev[k][0].record(lib_stream)
            g.reset_dropped()
            g.iterate_resident()
            ev[k][1].record(lib_stream)
            torch.cuda.synchronize()
        ms = float(sum(a.elapsed_time(b) for a, b in ev)) / args.steps
        g.realign_resident()
        g.realign_resident()
        cells = g.last_timing()["dp_cells"]
        pb, n_fallback, lmax16 = g.last_pair_buckets()
        b32 = g.last_buckets()
        al = g.get_alignment()
        P = min(args.parity_reads // 4, n)
        par = gpu_checks.round_parity(g, ref, np.ascontiguousarray(bases[: off[P]]), np.ascontiguousarray(off[: P + 1]), rc[:P], as_[:P], ae[:P], sm)
        par.pop("consensus")
        # pass 1 (k = 12) on the same reads: what the read shape does to the k-mer-filtered first pass
        p1 = None
        if not args.no_pass1:
            g.set_reference(ref, circular=1, with_rc=1)
            g.build_kmers(12)
            g.upload_reads(bases, off)                 # (the parity check above left its prefix on the device)
            p1_ms = []
            for _ in range(3):
                flush.zero_()
                torch.cuda.synchronize()
                g.pass1(fields=("score",))
                p1_ms.append(g.last_timing()["ms_kernels"])
            fastp, generalp, skippedp = g.last_pass1_stats()
            nominal, effective = g.last_pass1_cells()
            p1 = {"k": 12, "ms": float(min(p1_ms[1:])), "reads_per_s": n / (min(p1_ms[1:]) * 1e-3), "windowed_16bit": int(fastp), "general_kernel": int(generalp),
                  "no_kmer_hit": int(skippedp), "effective_gcups": effective / (min(p1_ms[1:]) * 1e-3) / 1e9}
            g.set_reference(ref, circular=1, with_rc=0)
        res[tag] = {"reads": n, "matrix": mat, "ms_per_step": ms, "value": n / (ms * 1e-3), "gcups": cells / (ms * 1e-3) / 1e9, "pass1": p1,
                    "gapped_fraction": float((al["n_runs"] > 1).mean()), "reads_in_16bit_kernels": int(sum(b["reads"] for b in pb)),
                    "fallback_fraction": n_fallback / n, "reads_handed_to_32bit_kernels": n_fallback, "max_read_len_16bit": lmax16,
                    "ms_16bit_kernels": float(sum(b["ms"] for b in pb)), "ms_32bit_kernels": float(sum(b["ms"] for b in b32)), "parity": par}
    g.set_pssm(load_pssm("onepass"))
    return res


def rmt_numbers(g, args, flush, lib_stream):
    """Resident rounds + k = 12 pass 1 with R-mt as the reference (derived from the reference's mt311 consensus by
    oracle/pyoracle.write_r_mt at build time, where /root/reference exists; a data file, nothing of oracle/ is executed)."""
    import torch
    path = os.path.join(ROOT, "oracle", "_ref", "r_mt.fa")
    if not os.path.exists(path):
        return {"unavailable": "oracle/_ref/r_mt.fa was not generated (no /root/reference at build time)"}
    rmt = "".join(l.strip() for l in open(path) if not l.startswith(">"))
    n = args.reads
    ref, bases, off, rc, as_, ae = make_workload(n, seed=2000, ref=rmt)
    g.set_reference(ref, circular=1, with_rc=0)
    g.upload_reads(bases, off)
    g.set_alignment_inputs(rc, as_, ae)
    g.set_cut_inputs(np.diff(off).astype(np.int32))
    for _ in range(3):
        g.reset_dropped()
        g.iterate_resident()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for k in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        ev[k][0].record(lib_stream)
        g.reset_dropped()
        g.iterate_resident()
        ev[k][1].record(lib_stream)
        torch.cuda.synchronize()
    ms = float(sum(a.elapsed_time(b) for a, b in ev)) / args.steps
    g.realign_resident()
    cells = g.last_timing()["dp_cells"]
    _, n_fallback, _ = g.last_pair_buckets()
    res = {"ref_len": len(ref), "reads": n, "value": n / (ms * 1e-3), "ms_per_step": ms, "gcups": cells / (ms * 1e-3) / 1e9,
           "reads_handed_to_32bit_kernels": n_fallback}
    if not args.no_pass1:
        res["pass1_k12"] = pass1_numbers(g, ref, bases, off, rc, args, only_k12=True)["k12"]
    return res


def extras(g, ref, stored, off, rc, as_, ae, sm):
    """8f1 repeat filter and 8f4 adapter trimming on the same 1 M reads, and a whole assembly (pass 1 with k = 12, then rounds
    until the consensus stops changing) with everything resident -- wall clock around the library calls."""
    from mia_b200 import driver
    n = len(off) - 1
    res = {}
    score = (200 * np.diff(off)).astype(np.int32)
    g.repeat_filter(rc, as_, ae, score)
    t0 = time.perf_counter()
    _, uniq = g.repeat_filter(rc, as_, ae, score)
    t = g.last_timing()
    res["repeat_filter"] = {"reads": n, "wall_ms": (time.perf_counter() - t0) * 1e3, "kernel_ms": t["ms_kernels"], "unique": int(uniq.sum())}
    adapter = "GTCAGACACGCAACAGGGGATAGGCAAGGCACACAGGGGATAGG"                 # mia_main.c:462
    g.trim(stored, off, adapter)
    t0 = time.perf_counter()
    tr = g.trim(stored, off, adapter)
    t = g.last_timing()
    res["trim"] = {"reads": n, "wall_ms": (time.perf_counter() - t0) * 1e3, "kernel_ms": t["ms_kernels"],
                   "gcups": t["dp_cells"] / (t["ms_kernels"] * 1e-3) / 1e9, "trimmed": int(tr["trimmed"].sum())}
    comp = np.zeros(256, np.uint8)
    for a, b in zip(b"ACGTN", b"TGCAN"):
        comp[a] = b
    rid = np.repeat(np.arange(n), np.diff(off))
    pos = np.arange(len(stored)) - off[rid]
    src = np.where(rc[rid] == 1, off[rid] + (off[rid + 1] - off[rid]) - 1 - pos, np.arange(len(stored)))
    orig = np.ascontiguousarray(np.where(rc[rid] == 1, comp[stored[src]], stored), np.uint8)
    for rep in range(2):
        A = driver.ResidentAssembler(g, ref, sm, circular=1, k=12)
        t0 = time.perf_counter()
        A.pass1(orig, off)
        t1 = time.perf_counter()
        conv = False
        while not conv and A.iter < 30:
            _, conv = A.iterate()
        t2 = time.perf_counter()
    res["assembly"] = {"reads": n, "rounds": A.iter, "converged": bool(conv), "pass1_wall_ms": (t1 - t0) * 1e3,
                       "rounds_wall_ms": (t2 - t1) * 1e3, "total_wall_ms": (t2 - t0) * 1e3, "consensus_len": len(A.cons),
                       "note": "driver.ResidentAssembler: pass 1 (k = 12) + rounds to convergence, everything resident; wall clock incl. "
                               "the host-side numpy bookkeeping between the library calls"}
    g.build_kmers(0)
    res["files"] = file_to_file(ref, orig, off)
    return res


def pass1_numbers(g, ref, stored, off, rc, args, only_k12=False):
    """Pass 1 on the original (un-revcomped) reads: (a) k = 12 filter on all reads, (b) no filter on a prefix."""
    comp = np.zeros(256, np.uint8)
    for a, b in zip(b"ACGTN", b"TGCAN"):
        comp[a] = b
    n = len(off) - 1
    rid = np.repeat(np.arange(n), np.diff(off))
    pos = np.arange(len(stored)) - off[rid]
    src = np.where(rc[rid] == 1, off[rid] + (off[rid + 1] - off[rid]) - 1 - pos, np.arange(len(stored)))
    orig = np.ascontiguousarray(np.where(rc[rid] == 1, comp[stored[src]], stored), np.uint8)
    g.set_reference(ref, circular=1, with_rc=1)
    res = {}
    for tag, k, m in (("k12", 12, n), ("unmasked", 0, min(n, args.pass1_unmasked_reads)))[: 1 if only_k12 else 2]:
        g.build_kmers(k)
        g.upload_reads(orig[: off[m]], off[: m + 1])
        g.pass1()                                   # warm-up
        out = g.pass1()
        t = g.last_timing()
        nominal, effective = g.last_pass1_cells()
        res[tag] = {"reads": m, "kernel_ms": t["ms_kernels"], "reads_per_s": m / (t["ms_kernels"] * 1e-3),
                    "nominal_cells": nominal, "effective_cells": effective,
                    # SURVEY 8d: GCUPS on nominal cells for unmasked runs, on EFFECTIVE cells (L x unmasked columns) for -k runs; both printed
                    "gcups": (effective if k > 0 else nominal) / (t["ms_kernels"] * 1e-3) / 1e9,
                    "nominal_gcups": nominal / (t["ms_kernels"] * 1e-3) / 1e9,
                    "effective_gcups": effective / (t["ms_kernels"] * 1e-3) / 1e9,
                    "accepted": int((out["score"] >= 2000).sum()), "rc_fraction": float(out["rc"].mean()),
                    "skipped_by_filter": int(((out["status"] & 2) != 0).sum()),
                    "reads_windowed_pair_kernels": g.last_pass1_stats()[0], "reads_general_kernel": g.last_pass1_stats()[1]}
    g.build_kmers(0)
    return res


def file_to_file(ref, orig, off, ref_sample=5000):
    """SURVEY 8 f2 / f3 and the plain-C host: FASTQ file -> reader -> pass 1 (k = 12) -> rounds -> `.maln` file, as a PROGRAM
    (host/mia_gpu, C, linked against libmiagpu.so only), wall clock with its own phase timing; the reader alone; and the
    unmodified reference binary (oracle/_ref/mia, 1 thread) on the first `ref_sample` reads of the same file with the same
    flags, whose final `.maln` must equal ours byte for byte after line 1 (checked here, reported as maln_identical)."""
    import ctypes as C
    import re
    import subprocess
    import tempfile
    from mia_b200 import api, synth
    root = os.path.dirname(os.path.abspath(__file__))
    host = os.path.join(root, "host", "mia_gpu")
    out = {}
    if not os.path.exists(host):
        return {"skipped": "host/mia_gpu not built"}
    n = len(off) - 1
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "ref.fa"), "w").write(">ref synthetic\n" + ref + "\n")
        open(os.path.join(d, "m.txt"), "w").write(synth.matrix_text(load_pssm()))
        open(os.path.join(d, "all.fq"), "wb").write(synth.fastq_text(orig, off))
        open(os.path.join(d, "part.fq"), "wb").write(synth.fastq_text(orig, off, 0, min(ref_sample, n)))
        fq_bytes = os.path.getsize(os.path.join(d, "all.fq"))
        # the reader alone (miagpu_fastx_open + _next over the whole file), second pass = page cache warm
        L = api.load_library()
        for _ in range(2):
            h, cnt = C.c_void_p(), C.c_int64()
            t0 = time.perf_counter()
            L.miagpu_fastx_open(C.byref(h), os.path.join(d, "all.fq").encode())
            L.miagpu_fastx_next(h, 1 << 40, C.byref(cnt))
            t = time.perf_counter() - t0
            L.miagpu_fastx_close(h)
        out["reader"] = {"reads": cnt.value, "file_mb": fq_bytes / 1e6, "wall_ms": t * 1e3, "mb_per_s": fq_bytes / 1e6 / t, "reads_per_s": cnt.value / t,
                         "cursors": min(os.cpu_count() or 1, 16),
                         "note": "miagpu_fastx_open + _next over the whole file, page cache warm; above 8 MB the file is parsed by several cursors "
                                 "at once, pieces kept only where the one-cursor parse would have stood in the same state"}

        def run(cmd):
            t0 = time.perf_counter()
            r = subprocess.run(cmd, cwd=d, capture_output=True, text=True)
            return time.perf_counter() - t0, r
        flags = ["-s", "m.txt", "-c", "-k", "12", "-F"]
        t, r = run([host, "-r", "ref.fa", "-f", "all.fq", "-m", "ours_all"] + flags)
        if r.returncode != 0:
            return {"error": r.stderr[-300:]}
        ph = re.search(r"timing ms: init ([\d.]+) parse ([\d.]+) pass1 ([\d.]+) rounds ([\d.]+) write ([\d.]+) total ([\d.]+)", r.stderr)
        rounds = int(re.search(r"after (\d+) rounds", r.stderr).group(1))
        final = os.path.join(d, f"ours_all.{rounds}")
        out["program"] = {"reads": n, "rounds": rounds, "wall_s": t, "reads_per_s": n / t, "maln_mb": os.path.getsize(final) / 1e6,
                          "phases_ms": dict(zip(("init", "parse", "pass1", "rounds", "write", "total"), map(float, ph.groups()))) if ph else None,
                          "note": "host/mia_gpu -c -k 12 -F: process start to exit incl. CUDA context creation, FASTQ parse, pass 1, all rounds, "
                                  "final .maln written to a tmpfs/overlay file; context creation and first-use allocations vary run to run (0.5-3.7 s and "
                                  "0.15-1.7 s observed), parse and write do not"}
        t_o, r_o = run([host, "-r", "ref.fa", "-f", "part.fq", "-m", "ours_part"] + flags)
        mia = os.path.join(root, "oracle", "_ref", "mia")
        if os.path.exists(mia) and r_o.returncode == 0:
            t_r, r_r = run([mia, "-r", "ref.fa", "-f", "part.fq", "-m", "ref_part"] + flags)
            ro = int(re.search(r"after (\d+) rounds", r_o.stderr).group(1))
            ours = open(os.path.join(d, f"ours_part.{ro}")).read().split("\n", 1)[1]
            refs = sorted(f for f in os.listdir(d) if f.startswith("ref_part."))
            theirs = open(os.path.join(d, refs[-1])).read().split("\n", 1)[1] if refs else ""
            out["vs_reference_binary"] = {"reads": min(ref_sample, n), "ours_wall_s": t_o, "reference_wall_s": t_r, "reference_cores": 1,
                                          "speedup_wall": t_r / t_o, "rounds": ro, "reference_final_file": refs[-1] if refs else None,
                                          "maln_identical": bool(refs) and ours == theirs,
                                          "note": "oracle/_ref/mia = the unmodified reference compiled with gcc -O2; same FASTA / FASTQ / matrix / flags; "
                                                  "ours includes ~0.3-0.5 s of CUDA context creation per process"}
    return out


def cpu_baseline(ref, bases, off, rc, as_, ae, sm, sample):
    from oracle.pyoracle import Oracle, Ref, have_ref
    o = Oracle()
    wrap = ref + ref[:256]
    s = min(sample, len(off) - 1)
    ws, wl = windows(off[: s + 1], as_[:s], ae[:s], len(wrap))
    smr = o.revcom_pssm(sm)
    if have_ref():
        r = Ref()
        t, cells, _ = r.time_realign(wrap, bases, off[: s + 1], ws, wl, rc[:s], sm, smr)
        kind = "reference"
    else:
        ctx = o.ctx_new(ref, 1, sm, with_rc=0, k=0)
        t0 = time.perf_counter()
        cells = 0
        for i in range(s):
            o.realign(ctx, bases[off[i]:off[i + 1]].tobytes(), int(rc[i]), int(as_[i]), int(ae[i]))
            cells += int(off[i + 1] - off[i]) * int(wl[i])
        t = time.perf_counter() - t0
        kind = "port"
    return {"value": s / t, "unit": UNIT, "cores": 1, "kind": kind, "gcups": cells / t / 1e9,
            "sample": f"first {s} reads of the same workload, realign sequence only (pop_s1c/pop_s2c/dyn_prog/max_sg_score/"
                      f"find_align_begin/populate_pwaln_to_begin), {t:.1f} s wall; the O(ref_len x N) consensus scan is NOT included"}


def _ref_worker(q, ref, bases, off, rc, as_, ae, sm, smr, lo, hi, steps, warmup):
    from oracle.pyoracle import Ref
    r = Ref()
    wrap = ref + ref[:256]
    o = np.ascontiguousarray(off[lo:hi + 1] - off[lo])
    b = np.ascontiguousarray(bases[off[lo]:off[hi]])
    ws, wl = windows(off[lo:hi + 1], as_[lo:hi], ae[lo:hi], len(wrap))
    rcs = np.ascontiguousarray(rc[lo:hi])
    m = max(1, (hi - lo) // 8)                           # a warm-up pass takes an eighth of the shard: every array cut to it
    for _ in range(warmup):
        r.time_realign(wrap, b, np.ascontiguousarray(o[: m + 1]), ws[:m].copy(), wl[:m].copy(), rcs[:m].copy(), sm, smr)
    ts, cells = [], 0
    for _ in range(steps):
        t, cells, _ = r.time_realign(wrap, b, o, ws, wl, rcs, sm, smr)
        ts.append(t)
    q.put((ts, cells))


def run_reference(args):
    """The reference's CPU implementation of the path, all host cores (one process per core)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle.pyoracle import Oracle, Ref, have_ref
    if not have_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libmia_ref.so missing (reference sources not on this box)"}))
        return
    Ref()                                                # the parent maps oracle/_ref/libmia_ref.so too (the workers are forked from it)
    cores = os.cpu_count() or 1
    per_core = args.ref_reads_per_core
    n = cores * per_core
    ref, bases, off, rc, as_, ae = make_workload(n, seed=1000)
    sm = load_pssm("onepass")
    smr = Oracle().revcom_pssm(sm)
    q = mp.Queue()
    procs = [mp.Process(target=_ref_worker, args=(q, ref, bases, off, rc, as_, ae, sm, smr, i * per_core, (i + 1) * per_core,
                                                  args.steps, args.warmup)) for i in range(cores)]
    t0 = time.perf_counter()
    for p in procs:
        p.start()
    res = [q.get() for _ in procs]
    for p in procs:
        p.join()
    wall = time.perf_counter() - t0
    step_t = [max(r[0][k] for r in res) for k in range(args.steps)]       # slowest shard per step
    cells = sum(r[1] for r in res)
    ms = float(np.mean(step_t)) * 1e3
    value = n / (ms * 1e-3)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1] (same generator), bounded sample per step", "reads_per_step": n,
                   "ref_len": REF_LEN},
        "gcups": cells / (ms * 1e-3) / 1e9,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference",
                         "sample": f"{per_core} reads per core x {cores} processes per step; unmodified reference realign sequence "
                                   f"(dyn_prog + traceback), consensus scan not included; total wall {wall:.1f} s"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=1_000_000, help="reads per GPU")
    ap.add_argument("--cpu-sample", type=int, default=60000)
    ap.add_argument("--ref-reads-per-core", type=int, default=4000)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-pass1", action="store_true")
    ap.add_argument("--no-rmt", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-shapes", action="store_true")
    ap.add_argument("--parity-reads", type=int, default=20000, help="prefix of rank 0's workload checked against the CPU reference")
    ap.add_argument("--pass1-unmasked-reads", type=int, default=1000000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
