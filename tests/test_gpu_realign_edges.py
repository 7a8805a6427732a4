"""-m gpu: a round's per-read realign against the oracle on every route classify_kernel can send a read down, read by read
(score, as, ae, abr and both gapped strings).  Nothing here is compared with another GPU configuration.

The routes: the eight 16-bit pair classes (128 ... 256 columns) in the low and the re-based (RB) frame, the nine
realign_kernel<K> buckets (<= 64 ... <= 512 columns), and the chunked strip kernels (team and warp) for windows over 512
columns and the whole-reference fallback (rs + L > re).  A read the pair kernels cannot finish is handed to a
32-bit bucket with its window cut at its end cell; the cases below make that window land in bucket 0 and come out narrower
than the read.

The case generator places every read so that the window rule of reiterate_assembly (mia_main.c:190-212) gives an exact width:
in the middle of the reference (ae - as = width - 100), at both clamps (as < 50, ae + 51 > wrap_len), across the end of a
circular reference into its 256-base wrap copy, and beyond the window (the whole-reference fallback).  The widths are every
edge E of the pair classes and the buckets at E and E + 1; the lengths 1, 2, 255, 256, the window's own width and the longest
read of every pair class's low 16-bit frame and one more (pair16.cuh p16_lmax, which moves with the matrix's maximum), and the
same at twice the columns per lane for the classes up to 176 columns (lengths just below those limits).  The
contents: exact copies, substitutions, indels, insertions at the window's start, unrelated reads, low-complexity stretches
(many tied end cells), N in the read and in the reference, and reads with 10 to 13 gaps around the 24-run limit.

Paths: realign_host (timed, one stream, the routing counters), iterate_host in three chunks (four streams, windows over 512
columns in every chunk) and the resident one-call round under set_fsdb (four streams)."""
import random

import numpy as np
import pytest

import gpu_checks

pytestmark = pytest.mark.gpu

GOP, GEP, PSSM_ABS_LIMIT, MAX_READ, MAX_RUNS, BUFFER = 1000, 200, 2000, 256, 24, 50
ST_RUNS_OVERFLOW = 1
P16_COLS = (128, 144, 160, 176, 192, 208, 224, 256)
NEAR_LIMIT_K = (16, 18, 20, 22, 12, 13, 14, 16)        # per pair class: the columns per lane of a second, lower length limit
BUCKET_EDGES = (64, 128, 160, 192, 224, 256, 320, 384, 512)
EDGES = sorted(set(P16_COLS) | set(BUCKET_EDGES))
WIDTHS = sorted({w for e in EDGES for w in (e, e + 1)} | {1000})
MATRICES = ("onepass", "ancient", "pe", "flat")
KINDS = ("exact", "sub", "indel", "ins_head", "random", "lowcx", "nread", "nref")
CONFIGS = {"default": {}, "pair16_off": {"MIAGPU_PAIR16": "0"}, "rb_off": {"MIAGPU_PAIR_RB": "0"},
           "no_narrow": {"MIAGPU_NO_NARROW": "1"}, "strip_warp": {"MIAGPU_STRIP_TEAM": "0"}, "strip_team": {"MIAGPU_STRIP_TEAM": "1"}}
ENV_KEYS = sorted({k for c in CONFIGS.values() for k in c} | {"MIAGPU_CHUNKS"})


def p16_lmax(K, max_entry):
    """pair16.cuh p16_off / p16_lmax: the longest read the low 16-bit frame of a K-column-per-lane class holds"""
    off = 32768 - 2 * GOP - GEP - PSSM_ABS_LIMIT - GEP * K - 32
    inc = max_entry + GEP
    return (32767 + off - GEP * (K - 2)) // inc if inc > 0 else MAX_READ


def low_frame_limits(sm):
    """per pair class: the low frame's longest read, and the same at NEAR_LIMIT_K columns per lane"""
    mx = int(np.max(sm))
    return [(min(p16_lmax(c // 16, mx), MAX_READ), min(p16_lmax(k, mx), MAX_READ)) for c, k in zip(P16_COLS, NEAR_LIMIT_K)]


def window(as_, ae, L, W):
    """classify_kernel's window rule -> (rs, width, whole-reference fallback)"""
    rs = max(0, as_ - BUFFER)
    re = W if ae + BUFFER + 1 > W else ae + BUFFER
    if rs + L > re:
        return 0, W, True
    return rs, re - rs, False


def n_runs_of(rg, fg):
    kinds = ["I" if a == "-" else "D" if b == "-" else "M" for a, b in zip(rg, fg)]
    return sum(1 for i, k in enumerate(kinds) if i == 0 or k != kinds[i - 1])


def make_reference(n, seed):
    """uniform ACGT with a 300-base homopolymer, a 300-base dinucleotide repeat, a 240-base triplet repeat and a stretch
    with 3 % N"""
    rng = np.random.default_rng(seed)
    s = bytearray(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].tobytes())
    lo = n // 4
    s[lo:lo + 300] = b"A" * 300
    s[lo + 700:lo + 1000] = b"AC" * 150
    s[lo + 1400:lo + 1640] = b"AAT" * 80
    nlo = n // 2 + 500
    for p in rng.choice(np.arange(nlo, nlo + 600), 18, replace=False):
        s[p] = ord("N")
    return s.decode(), (lo, lo + 1640), (nlo, nlo + 600)


class Case:
    """One batch of reads against one reference and matrix, with the oracle's realign of every read."""

    def __init__(self, oracle, matrix, circular, ref_len, seed, per_combo=2, n_whole=4):
        self.name = f"{matrix}/{'circular' if circular else 'linear'}/{ref_len}"
        self.sm = gpu_checks.load_pssm(matrix)
        self.circular = circular
        self.ref, self.lowcx, self.nreg = make_reference(ref_len, seed)
        W = len(self.ref) + (min(256, len(self.ref)) if circular else 0)
        self.wref = self.ref + (self.ref[:W - len(self.ref)])
        rng = random.Random(seed)
        limits = low_frame_limits(self.sm)
        reads, meta = [], []                                   # meta: (as, ae, rc, description)
        kind_i = 0

        def add(kind, place, w, L, as_, ae, src):
            nonlocal kind_i
            read = self._content(rng, kind, src, L)
            rs, wl, whole = window(as_, ae, L, W)
            assert (wl, whole) == ((W, True) if place == "whole" else (w, False)), (place, w, L, as_, ae, rs, wl, whole)
            reads.append(read)
            meta.append((as_, ae, rng.randint(0, 1), (kind, place, w, L)))

        for w in WIDTHS:
            cls = next((k for k, c in enumerate(P16_COLS) if w <= c), None)
            lens = {1, 2, 255, 256, w, w - 1, rng.randint(3, 254)}
            for lim, near in limits:
                lens |= {lim, lim + 1, near, near + 1}
            lens = sorted(L for L in lens if 1 <= L <= min(w, MAX_READ))
            places = ["left", "right"] + (["middle"] + (["wrap"] if circular else []) if w >= 100 else [])
            for place in places:
                for L in lens:
                    for _ in range(per_combo):
                        kind = KINDS[kind_i % len(KINDS)]
                        kind_i += 1
                        as_, ae, src = self._place(rng, place, kind, w, L, W)
                        add(kind, place, w, L, as_, ae, src)
            # the low frame's limit and one more with exact copies (the highest path a read can take) at every end-column phase
            if cls is not None:
                for L in sorted({x for pair in limits[cls:cls + 1] for y in pair for x in (y, y + 1) if x <= w}):
                    for _ in range(6):
                        place = rng.choice(["left", "right", "middle"] if w >= 100 else ["left", "right"])
                        as_, ae, src = self._place(rng, place, "exact", w, L, W)
                        add("exact", place, w, L, as_, ae, src)
        # the whole-reference fallback: the read does not fit its window
        for k in range(n_whole):
            L = (101, 180, 256, 130)[k % 4]
            if k % 2:
                as_ = ae = rng.randint(BUFFER, W - BUFFER - 2)
            else:
                as_, ae = rng.randint(0, 10), rng.randint(10, 30)
            src = min(max(0, as_ - 20), W - L)
            add(("sub", "indel", "exact", "lowcx")[k % 4], "whole", W, L, as_, ae, src)
        # 10 .. 13 single-base gaps, spread over the read: 21 .. 27 runs around the limit of 24
        for L in (150, 200, 256):
            for g in (10, 11, 12, 13):
                for _ in range(2):
                    w = L + 120
                    as_, ae, src = self._place(rng, "middle", "exact", w, L, W)
                    reads.append(self._gapped(self.wref[src:], L, g))
                    meta.append((as_, ae, rng.randint(0, 1), ("gaps%d" % g, "middle", w, L)))
        order = list(range(len(reads)))
        rng.shuffle(order)                                     # every class and bucket in every chunk of iterate_host
        self.reads = [reads[i] for i in order]
        self.desc = [meta[i][3] for i in order]
        n = len(self.reads)
        self.as_ = np.array([meta[i][0] for i in order], np.int32)
        self.ae = np.array([meta[i][1] for i in order], np.int32)
        self.rc = np.array([meta[i][2] for i in order], np.uint8)
        self.off = np.zeros(n + 1, np.int64)
        np.cumsum([len(r) for r in self.reads], out=self.off[1:])
        self.bases = np.frombuffer("".join(self.reads).encode(), np.uint8).copy()
        self.win = [window(int(self.as_[i]), int(self.ae[i]), len(self.reads[i]), W) for i in range(n)]
        ctx = oracle.ctx_new(self.ref, circular, self.sm, with_rc=0, k=0)
        assert oracle.ctx_seq(ctx) == self.wref
        self.exp = []
        for i in range(n):
            o = oracle.realign(ctx, self.reads[i], int(self.rc[i]), int(self.as_[i]), int(self.ae[i]))
            o["n_runs"] = n_runs_of(o["ref_gapped"], o["read_gapped"])
            self.exp.append(o)
        oracle.ctx_free(ctx)
        self.over = np.array([e["n_runs"] > MAX_RUNS for e in self.exp])

    def _place(self, rng, place, kind, w, L, W):
        """(as, ae, source position of the read) such that the window is exactly w columns"""
        if place == "middle":                                  # rs = as - 50, re = ae + 50
            if kind == "lowcx":
                p = rng.randint(self.lowcx[0], self.lowcx[1] - L)
            elif kind == "nref":
                p = rng.randint(self.nreg[0], self.nreg[1] - min(L, 300))
            else:
                p = rng.randint(0, W - L)
            rs = rng.randint(max(0, p + L - w), min(p, W - w - 1)) if max(0, p + L - w) <= min(p, W - w - 1) else rng.randint(0, W - w - 1)
            as_ = rs + BUFFER
            ae = as_ + w - 2 * BUFFER
        elif place == "left":                                  # as < 50: rs = 0, re = ae + 50
            rs, ae = 0, w - BUFFER
            as_ = rng.randint(0, min(BUFFER - 1, ae))
        elif place == "right":                                 # ae + 51 > W: re = W, rs = as - 50
            rs = W - w
            as_ = rs + BUFFER
            ae = rng.randint(max(as_, W - BUFFER), W - 1)
        else:                                                  # circular: the window crosses seq_len into the wrap copy
            seq_len = len(self.ref)
            rs = rng.randint(max(0, seq_len - w + 1), min(seq_len - 1, W - w - 1))
            as_ = rs + BUFFER
            ae = as_ + w - 2 * BUFFER
        if place != "middle" or not rs <= p <= rs + w - L:
            p = rs if kind == "ins_head" else rng.randint(rs, rs + w - L)
        if kind == "ins_head":
            p = rs
        return as_, ae, p

    def _content(self, rng, kind, p, L):
        src = self.wref[p:]
        if kind == "random":
            return "".join(rng.choice("ACGT") for _ in range(L))
        if kind == "exact":
            return src[:L]
        if kind in ("sub", "lowcx", "nref"):
            rate = 0.04 if kind == "sub" else 0.02
            return "".join(rng.choice("ACGT") if rng.random() < rate else ch for ch in src[:L])
        if kind == "nread":
            return "".join("N" if rng.random() < 0.03 else ch for ch in src[:L])
        out, i = [], 0
        n_ins = 3 if kind == "ins_head" else 0
        while len(out) < L and i < len(src):
            x = rng.random()
            if kind == "ins_head" and n_ins and len(out) >= 4 and x < 0.15:
                out.append(rng.choice("ACGT"))
                n_ins -= 1
            elif kind == "indel" and x < 0.02:
                out.append(rng.choice("ACGT"))
            elif kind == "indel" and x < 0.04:
                i += rng.randint(1, 3)
            else:
                out.append(src[i])
                i += 1
        return "".join(out)[:L].ljust(L, "A")

    @staticmethod
    def _gapped(src, L, g):
        """L bases of src with g single-base gaps, alternately an insertion and a deletion, evenly spaced"""
        step = L // (g + 1)
        out, i = [], 0
        for k in range(g):
            out.append(src[i:i + step])
            i += step
            if k % 2:
                out.append("ACGT"[(ord(src[i]) + 1) % 4])
            else:
                i += 1
        out.append(src[i:i + L])
        return "".join(out)[:L]

    def subset(self, keep):
        """the same reads without the ones the one-call rounds refuse (more than 24 runs)"""
        c = object.__new__(Case)
        c.__dict__.update(self.__dict__)
        idx = np.flatnonzero(keep)
        c.reads = [self.reads[i] for i in idx]
        c.desc = [self.desc[i] for i in idx]
        c.exp = [self.exp[i] for i in idx]
        c.win = [self.win[i] for i in idx]
        c.as_, c.ae, c.rc, c.over = self.as_[idx], self.ae[idx], self.rc[idx], self.over[idx]
        c.off = np.zeros(len(idx) + 1, np.int64)
        np.cumsum([len(r) for r in c.reads], out=c.off[1:])
        c.bases = np.frombuffer("".join(c.reads).encode(), np.uint8).copy()
        return c


def mismatches(case, score, as_out, ae_out, abr, n_runs, status, runs_of):
    """reads whose GPU result differs from the oracle's.  A read whose oracle alignment has more than 24 runs must carry the
    overflow bit (n_runs = -1) with exact score / as / ae / abr; every other read must not."""
    import _pkg
    _pkg.load()
    from mia_b200 import api
    bad = []
    for i, e in enumerate(case.exp):
        st, nr = int(status[i]), int(n_runs[i])
        head = (int(score[i]), int(as_out[i]), int(ae_out[i]), int(abr[i]))
        want_head = (e["score"], e["as_"], e["ae"], e["abr"])
        if e["n_runs"] > MAX_RUNS:
            got, want = head + (st, nr), want_head + (ST_RUNS_OVERFLOW, -1)
        else:
            strings = api.expand_runs(case.wref, case.reads[i], int(as_out[i]), int(abr[i]), runs_of(i), nr) if nr > 0 else None
            got, want = head + (strings, st), want_head + ((e["ref_gapped"], e["read_gapped"]), 0)
        if got != want:
            bad.append((i, case.desc[i], int(case.rc[i]), int(case.as_[i]), int(case.ae[i]), got, want))
    return bad


def set_config(monkeypatch, env):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def realign_host(gpu, case):
    gpu.set_pssm(case.sm)
    gpu.set_reference(case.ref, circular=case.circular, with_rc=0)
    out = gpu.realign_host(case.bases, case.off, case.rc, case.as_, case.ae)
    pb, fb, _ = gpu.last_pair_buckets()
    return out, gpu.last_buckets(), pb, fb


@pytest.fixture(scope="module")
def cases(oracle):
    return [Case(oracle, m, circ, 6000, seed=1000 + 10 * k + circ) for k, m in enumerate(MATRICES) for circ in (1, 0)]


@pytest.fixture(scope="module")
def big_case(oracle):
    # 200 kb: too big for the kernels' shared-memory copy of the reference, read through L2.  Each whole-reference read costs the
    # oracle L x 200 k cells: only three of them.
    return Case(oracle, "onepass", 1, 200_000, seed=77, per_combo=1, n_whole=3)


@pytest.mark.parametrize("config", list(CONFIGS))
def test_realign_host_every_route_equals_oracle(gpu, monkeypatch, cases, big_case, config):
    set_config(monkeypatch, CONFIGS[config])
    report = []
    for case in cases + [big_case]:
        out, buckets, pairs, fb = realign_host(gpu, case)
        bad = mismatches(case, out["score"], out["as_out"], out["ae_out"], out["abr"], out["n_runs"], out["status"], lambda i: out["runs"][i])
        assert not bad, f"{config} {case.name}: {len(bad)} of {len(case.reads)} reads differ from the oracle; first: {bad[:3]}"
        report.append((case.name, [(b["K"], b["reads"]) for b in buckets], [(p["K"], p["reads"]) for p in pairs], fb))
        # both sides of the 24-run limit were reached, and the overflow bit was checked read by read above
        assert case.over.sum() > 0 and sum(1 for e in case.exp if 21 <= e["n_runs"] <= MAX_RUNS) > 0
        if config == "pair16_off":                      # every realign_kernel<K> and the chunked kernel take reads
            assert len(buckets) == 10 and not pairs, (case.name, buckets, pairs)
    print(f"\nrouting {config}:")
    for name, b, p, fb in report:
        print(f"  {name}: buckets (K, reads) {b}  pair classes (K, reads) {p}  handed over {fb}")


def test_routing_reaches_every_class_and_frame(gpu, monkeypatch, cases):
    """The cases reach every route: all eight pair classes, the RB frame in a class of at most 176 columns, hand-overs, the
    whole-reference fallback; hand-overs whose cut window lands in bucket 0 or is narrower than the read."""
    for case in cases:
        set_config(monkeypatch, {})
        out, buckets, pairs, fb = realign_host(gpu, case)
        assert len(pairs) == 8 and fb > 0, (case.name, pairs, fb)
        assert any(b["K"] == 0 for b in buckets), (case.name, buckets)         # the chunked kernel
        assert sum(wh for _, _, wh in case.win) >= 4, case.name                  # among its reads: the whole-reference fallback
        set_config(monkeypatch, {"MIAGPU_PAIR_RB": "0"})
        _, _, pairs_low, _ = realign_host(gpu, case)
        low = {p["K"]: p["reads"] for p in pairs_low}
        assert any(p["reads"] > low.get(p["K"], 0) for p in pairs if p["K"] <= 11), (case.name, pairs, pairs_low)
        # the pair kernels' hand-overs: the end cell cuts the window to aec + 1 columns (pair16.cuh); those cut narrower than
        # the read and into bucket 0 (<= 64 columns) are among them
        cut = [(i, case.exp[i]["ae"] - rs + 1) for i, (rs, wl, wh) in enumerate(case.win)
               if not wh and wl <= 256 and len(case.reads[i]) > 1 and "-" in case.exp[i]["ref_gapped"] + case.exp[i]["read_gapped"]]
        assert any(c < len(case.reads[i]) for i, c in cut) and any(c <= 64 for _, c in cut), case.name


@pytest.mark.parametrize("team", [None, "0"])
def test_iterate_host_chunks_equal_oracle(gpu, monkeypatch, cases, team):
    """miagpu_iterate_host in three chunks: every chunk holds windows over 512 columns (the chunked kernel's pointers are offset
    by the chunk's first read) and every pair class; per-read outputs and the packed run lists against the oracle."""
    set_config(monkeypatch, {"MIAGPU_CHUNKS": "3"} | ({"MIAGPU_STRIP_TEAM": team} if team else {}))
    for full in cases:
        case = full.subset(~full.over)
        n = len(case.reads)
        bounds = [0, n // 5, n * 3 // 5, n]                    # n (2k - 1) / (2C - 1) for C = 3
        for k in range(3):
            assert any(case.win[i][1] > 512 for i in range(bounds[k], bounds[k + 1])), (case.name, k)
        gpu.set_pssm(case.sm)
        gpu.set_reference(case.ref, circular=case.circular, with_rc=0)
        packed = np.zeros(n * MAX_RUNS, np.uint16)
        dropped = np.zeros(n, np.uint8)
        _, out, tot, _ = gpu.iterate_host(case.bases, case.off, case.rc, case.as_, case.ae, np.diff(case.off).astype(np.int32), dropped,
                                          packed=packed)
        run_off = np.zeros(n + 1, np.int64)
        np.cumsum(np.maximum(out["n_runs"], 0), out=run_off[1:])
        assert tot == run_off[-1]
        bad = mismatches(case, out["score"], out["as_out"], out["ae_out"], out["abr"], out["n_runs"], out["status"],
                         lambda i: packed[run_off[i]:run_off[i + 1]])
        assert not bad, f"{case.name}: {len(bad)} of {n} reads differ from the oracle; first: {bad[:3]}"


def test_resident_round_equals_oracle(gpu, monkeypatch, cases, big_case):
    """the resident one-call round under set_fsdb (four streams) on the same reads: per read and the round's consensus.
    Left out: reads with more than 24 runs (the round refuses them) and, on a circular reference, reads the clamped window left
    wholly in the wrap copy (as >= seq_len): their front AlnSeq's `over` positions are stale bytes in the reference (DESIGN §5)."""
    set_config(monkeypatch, {})
    ck = gpu_checks.Checker()
    for full in cases + [big_case]:
        in_wrap = np.array([full.circular and e["as_"] >= len(full.ref) for e in full.exp])
        case = full.subset(~full.over & ~in_wrap)
        r = gpu_checks.round_parity(gpu, case.ref, case.bases, case.off, case.rc, case.as_, case.ae, case.sm, circular=case.circular, checker=ck)
        assert r["per_read_equal"] and r["consensus_equal"], (case.name, r["n_diff"], r["first_diff"], r["checker"])


# ------------------------------------------------------------------------------------------------ miagpu_align_windows
def _windows_case(seed):
    rng = random.Random(seed)
    ref, _, _ = make_reference(6000, seed)
    reads, ws, wl = [], [], []
    for w in sorted(set(WIDTHS) | {1999}):
        for L in (1, 2, 40, 127, 200, 256):
            for kind in ("exact", "sub", "indel", "random", "short"):
                width = max(1, L // 2) if kind == "short" else w            # windows shorter than the read
                s = rng.randint(0, len(ref) - width)
                p = rng.randint(s, max(s, s + width - L))
                src = ref[p:] if p + L + 10 <= len(ref) else ref[len(ref) - L - 10:]
                if kind == "random":
                    read = "".join(rng.choice("ACGT") for _ in range(L))
                elif kind == "indel":
                    read = "".join(src[:L // 3] + "G" + src[L // 3:2 * L // 3] + src[2 * L // 3 + 2:])[:L]
                elif kind == "sub":
                    read = "".join(rng.choice("ACGT") if rng.random() < 0.04 else ch for ch in src[:L])
                else:
                    read = src[:L]
                reads.append(read.ljust(L, "C"))
                ws.append(s)
                wl.append(width)
    return ref, reads, np.array(ws, np.int32), np.array(wl, np.int32)


@pytest.mark.parametrize("sg5", [1, 0])
@pytest.mark.parametrize("rc", [0, 1])
def test_align_windows_every_width_equals_oracle(gpu, monkeypatch, oracle, sg5, rc):
    """explicit windows at every bucket edge, 513 and 1999 columns (the chunked kernel) and shorter than their reads, with the
    forward or the strand-reversed matrix, sg5 as given -- against oracle.align on the window's piece"""
    import _pkg
    _pkg.load()
    from mia_b200 import api
    sm = gpu_checks.load_pssm("ancient")
    ref, reads, ws, wl = _windows_case(11 + 2 * sg5 + rc)
    smx = oracle.revcom_pssm(sm) if rc else sm
    exp = []
    for i, read in enumerate(reads):
        a = oracle.align(ref[ws[i]:ws[i] + wl[i]], read, smx, sg5)
        exp.append(dict(score=a["score"], as_=a["abc"] + int(ws[i]), ae=a["aec"] + int(ws[i]), abr=a["abr"], ref_gapped=a["ref_gapped"],
                        read_gapped=a["read_gapped"], n_runs=n_runs_of(a["ref_gapped"], a["read_gapped"])))
    case = object.__new__(Case)
    case.exp, case.reads, case.wref = exp, reads, ref
    case.desc = [("window", int(w), len(r)) for w, r in zip(wl, reads)]
    case.rc, case.as_, case.ae = np.full(len(reads), rc, np.uint8), ws, ws + wl
    off = np.zeros(len(reads) + 1, np.int64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    assert (wl > 512).sum() >= 60 and (wl < np.diff(off)).sum() >= 60
    for team in (None, "0", "1"):
        set_config(monkeypatch, {"MIAGPU_STRIP_TEAM": team} if team else {})
        gpu.set_pssm(sm)
        gpu.set_reference(ref, circular=0, with_rc=0)
        gpu.upload_reads(np.frombuffer("".join(reads).encode(), np.uint8), off)
        out = gpu.align_windows(case.rc, ws, wl, sg5)
        runs = out["runs"].view(np.uint16).reshape(-1, api.MAX_RUNS)
        bad = mismatches(case, out["score"], out["as_out"], out["ae_out"], out["abr"], out["n_runs"], out["status"], lambda i: runs[i])
        assert not bad, f"sg5 {sg5} rc {rc} team {team}: {len(bad)} of {len(reads)} windows differ from the oracle; first: {bad[:3]}"
