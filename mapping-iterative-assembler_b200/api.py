"""ctypes binding of libmiagpu.so (include/miagpu.h) -- the host-side mirror of the
reference's call sites.  Python is plumbing only: every compute call goes through
the C ABI into hand-written sm_100a kernels; there is no CPU fallback and this
module raises if the library is missing or a call fails.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MIAGPU_LIB") or os.path.join(HERE, "libmiagpu.so")      # MIAGPU_LIB: a differently built libmiagpu.so (kernel experiments)
MAX_RUNS = 24
RUN_M, RUN_I, RUN_D = 0, 1, 2
MISINC_SHAPE = (31, 6, 6)          # miagpu_misincorporation: depth, reference, read
MISINC_CODES = "ACGTN-"            # the codes of both base axes (N = any other character)

_i32p = C.POINTER(C.c_int32)
_u8p = C.POINTER(C.c_uint8)
_u16p = C.POINTER(C.c_uint16)
_i64p = C.POINTER(C.c_int64)


class MiaGpuError(RuntimeError):
    pass


ENTRY_DTYPE = np.dtype([("read", np.int32), ("col_begin", np.int32), ("col_count", np.int32), ("ref_pos", np.int32),
                        ("front_len", np.int32), ("total_len", np.int32), ("act_bias", np.int32), ("dropped", np.uint8),
                        ("back_formula", np.uint8), ("reserved", np.uint8, 2)])
assert ENTRY_DTYPE.itemsize == 32

_lib = None


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MiaGpuError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.miagpu_last_error.restype = C.c_char_p
    L.miagpu_version.restype = C.c_char_p
    L.miagpu_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.miagpu_destroy.argtypes = [C.c_void_p]
    L.miagpu_destroy.restype = None
    L.miagpu_set_pssm.argtypes = [C.c_void_p, _i32p]
    L.miagpu_get_pssm.argtypes = [C.c_void_p, _i32p, _i32p]
    L.miagpu_set_reference.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int]
    L.miagpu_ref_wrap_len.argtypes = [C.c_void_p]
    L.miagpu_build_kmers.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.miagpu_upload_reads.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.miagpu_pass1.argtypes = [C.c_void_p] + [C.c_void_p] * 13
    L.miagpu_last_pass1_stats.argtypes = [C.c_void_p, _i64p, _i64p, _i64p]
    L.miagpu_set_homopolymer.argtypes = [C.c_void_p, C.c_int]
    L.miagpu_set_cons_capacity.argtypes = [C.c_void_p, C.c_int64]
    L.miagpu_last_pass1_route.argtypes = [C.c_void_p, C.c_void_p]
    L.miagpu_last_pass1_cells.argtypes = [C.c_void_p, _i64p, _i64p]
    L.miagpu_compact_reads.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, _i64p]
    L.miagpu_realign.argtypes = [C.c_void_p] + [C.c_void_p] * 10
    L.miagpu_get_runs_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, _i64p]
    L.miagpu_realign_host.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 12
    L.miagpu_consensus.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, _i32p]
    L.miagpu_accumulate_gaps.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_void_p), _i64p]
    L.miagpu_accumulate_counts.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), _i64p]
    L.miagpu_call.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, _i32p]
    L.miagpu_consensus_natural.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, _i32p]
    L.miagpu_accumulate_gaps_natural.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), _i64p]
    L.miagpu_score_cut.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.miagpu_cull_flags.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
    L.miagpu_set_alignment_inputs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.miagpu_realign_resident.argtypes = [C.c_void_p]
    L.miagpu_adopt_alignment.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.miagpu_set_cut_inputs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.miagpu_reset_dropped.argtypes = [C.c_void_p]
    L.miagpu_iterate_resident.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.POINTER(C.c_double),
                                          C.POINTER(C.c_double), C.c_void_p, C.c_void_p, C.c_void_p, _i32p]
    L.miagpu_last_buckets.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.miagpu_iterate_host.argtypes = ([C.c_void_p, C.c_int64] + [C.c_void_p] * 12 + [C.c_int64, _i64p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                      C.c_double, C.c_double, C.c_void_p, C.c_int, C.c_void_p, C.c_char_p, _i32p])
    _vpp = C.POINTER(C.c_void_p)
    L.miagpu_shard_begin.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_double, _vpp, _i64p]
    L.miagpu_shard_begin_host.argtypes = ([C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int64] + [C.c_void_p] * 14 +
                                          [C.c_int, C.c_int, C.c_double, C.c_double, _vpp, _i64p])
    L.miagpu_shard_fit.argtypes = [C.c_void_p, _vpp, _vpp, _i64p]
    L.miagpu_shard_cut.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), _vpp, _i64p]
    L.miagpu_shard_finish.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, _i64p, C.c_void_p, C.c_char_p, _i32p]
    L.miagpu_last_cut_stats.argtypes = [C.c_void_p, _i64p, _i64p]
    L.miagpu_trim.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int] + [C.c_void_p] * 6
    L.miagpu_repeat_filter.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.miagpu_last_pair_buckets.argtypes = [C.c_void_p] + [C.c_void_p] * 5 + [_i32p, _i32p]
    L.miagpu_last_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float), _i64p, _i32p]
    L.miagpu_int32_peak.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    L.miagpu_get_alignment.argtypes = [C.c_void_p] + [C.c_void_p] * 6
    L.miagpu_align_windows.argtypes = [C.c_void_p] + [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 7
    L.miagpu_fastx_open.argtypes = [_vpp, C.c_char_p]
    L.miagpu_fastx_open_memory.argtypes = [_vpp, C.c_void_p, C.c_int64]
    L.miagpu_fastx_format.argtypes = [C.c_void_p]
    L.miagpu_fastx_next.argtypes = [C.c_void_p, C.c_int64, _i64p]
    L.miagpu_fastx_batch.argtypes = [C.c_void_p] + [_vpp] * 7
    L.miagpu_fastx_close.argtypes = [C.c_void_p]
    L.miagpu_fastx_close.restype = None
    L.miagpu_maln_ref_size.argtypes = [C.c_int, C.c_int]
    L.miagpu_read_pssm.argtypes = [C.c_char_p, _i32p]
    L.miagpu_write_maln.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, _i64p]
    L.miagpu_write_maln_fsdb.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p, _i64p]
    L.miagpu_set_fsdb.argtypes = [C.c_void_p] + [C.c_void_p] * 6 + [C.c_int64, C.c_void_p, C.c_int]
    L.miagpu_get_fsdb.argtypes = [C.c_void_p] + [C.c_void_p] * 6 + [_i64p]
    L.miagpu_last_fsdb_stats.argtypes = [C.c_void_p, _i64p, _i64p, _i64p, _i64p]
    L.miagpu_distant_retry.argtypes = [C.c_void_p, _i64p, _i64p]
    L.miagpu_distant_retry_begin.argtypes = [C.c_void_p, _i64p, _i32p]
    L.miagpu_distant_retry_end.argtypes = [C.c_void_p, C.c_int, _i64p]
    L.miagpu_misincorporation.argtypes = [C.c_void_p, _i64p]
    L.miagpu_stream.restype = C.c_void_p
    L.miagpu_stream.argtypes = [C.c_void_p]
    _lib = L
    return L


EXPORTS = ["miagpu_device_count", "miagpu_create", "miagpu_destroy", "miagpu_last_error", "miagpu_version", "miagpu_set_pssm",
           "miagpu_get_pssm", "miagpu_set_reference", "miagpu_ref_wrap_len", "miagpu_build_kmers", "miagpu_upload_reads",
           "miagpu_pass1", "miagpu_last_pass1_stats", "miagpu_last_pass1_route", "miagpu_compact_reads", "miagpu_realign", "miagpu_realign_host", "miagpu_iterate_host", "miagpu_get_runs_packed",
           "miagpu_consensus", "miagpu_accumulate_gaps", "miagpu_accumulate_counts", "miagpu_call", "miagpu_consensus_natural", "miagpu_accumulate_gaps_natural",
           "miagpu_score_cut", "miagpu_cull_flags",
           "miagpu_set_alignment_inputs", "miagpu_realign_resident", "miagpu_adopt_alignment", "miagpu_set_cut_inputs", "miagpu_reset_dropped", "miagpu_iterate_resident", "miagpu_last_buckets", "miagpu_last_pair_buckets", "miagpu_last_timing",
           "miagpu_int32_peak", "miagpu_stream", "miagpu_shard_begin", "miagpu_shard_begin_host", "miagpu_shard_fit", "miagpu_shard_cut", "miagpu_shard_finish",
           "miagpu_last_cut_stats", "miagpu_repeat_filter", "miagpu_trim", "miagpu_get_alignment",
           "miagpu_fastx_open", "miagpu_fastx_open_memory", "miagpu_fastx_format", "miagpu_fastx_next", "miagpu_fastx_batch", "miagpu_fastx_close",
           "miagpu_maln_ref_size", "miagpu_write_maln", "miagpu_read_pssm", "miagpu_align_windows",
           "miagpu_set_fsdb", "miagpu_get_fsdb", "miagpu_last_fsdb_stats", "miagpu_distant_retry", "miagpu_write_maln_fsdb", "miagpu_last_pass1_cells", "miagpu_set_homopolymer", "miagpu_shard_flags", "miagpu_set_cons_capacity",
           "miagpu_distant_retry_begin", "miagpu_distant_retry_end", "miagpu_misincorporation"]


def _ptr(a):
    """Raw address of a numpy array / torch tensor / None."""
    if a is None:
        return None
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    return C.c_void_p(a.ctypes.data)


class MiaGpu:
    """One context = one GPU = one stream (SURVEY.md 8b)."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = C.c_void_p()
        if not self.lib.miagpu_create(C.byref(h), device):
            raise MiaGpuError(self.lib.miagpu_last_error().decode())
        self.h = h
        self.n = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.miagpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, ok):
        if not ok:
            raise MiaGpuError(self.lib.miagpu_last_error().decode())

    # -- setup
    def set_pssm(self, sm):
        sm = np.ascontiguousarray(sm, np.int32)
        assert sm.size == 775
        self._ck(self.lib.miagpu_set_pssm(self.h, sm.ctypes.data_as(_i32p)))

    def get_pssm(self):
        f, r = np.zeros(775, np.int32), np.zeros(775, np.int32)
        self._ck(self.lib.miagpu_get_pssm(self.h, f.ctypes.data_as(_i32p), r.ctypes.data_as(_i32p)))
        return f, r

    def set_reference(self, seq, circular=1, with_rc=0):
        b = seq if isinstance(seq, bytes) else seq.encode()
        self._ck(self.lib.miagpu_set_reference(self.h, b, len(b), int(circular), int(with_rc)))
        self.seq_len = len(b)
        self.wrap_len = self.lib.miagpu_ref_wrap_len(self.h)

    def build_kmers(self, k, soft_mask=0):
        self._ck(self.lib.miagpu_build_kmers(self.h, int(k), int(soft_mask)))

    def upload_reads(self, bases, offsets):
        n = len(offsets) - 1
        self._ck(self.lib.miagpu_upload_reads(self.h, n, _ptr(bases), _ptr(offsets)))
        self.n = n

    # -- pass 1
    def pass1(self, fields=None):
        """new_kmer_filter + sg_align's compute over the resident reads (mia_main.c:781-796).
        fields: the outputs wanted (default: all); the others are not downloaded."""
        n = self.n
        spec = dict(hits=np.int32, score=np.int32, fw_score=np.int32, rc_score=np.int32, rc=np.uint8, as_=np.int32, ae=np.int32,
                    start=np.int32, end=np.int32, abr=np.int32, n_runs=np.int32, runs=np.uint16, status=np.uint8)
        o = {k: (np.zeros((n, MAX_RUNS) if k == "runs" else n, dt) if (fields is None or k in fields) else None) for k, dt in spec.items()}
        self._ck(self.lib.miagpu_pass1(self.h, *[_ptr(o[k]) for k in ("hits", "score", "fw_score", "rc_score", "rc", "as_", "ae",
                                                                     "start", "end", "abr", "n_runs", "runs", "status")]))
        return {k: v for k, v in o.items() if v is not None}

    def set_homopolymer(self, on=True):
        """mia -h: the homopolymer-discounted gap candidates in every alignment of this context"""
        self._ck(self.lib.miagpu_set_homopolymer(self.h, int(bool(on))))

    def last_pass1_stats(self):
        """(reads finished by the windowed pair kernels, reads the general kernel took, reads without a k-mer hit)"""
        f, g, k = C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(self.lib.miagpu_last_pass1_stats(self.h, C.byref(f), C.byref(g), C.byref(k)))
        return f.value, g.value, k.value

    def last_pass1_cells(self):
        """(nominal, effective) DP cells of the last pass 1 (SURVEY 8d)"""
        a, b = C.c_int64(), C.c_int64()
        self._ck(self.lib.miagpu_last_pass1_cells(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def last_pass1_route(self):
        r = np.zeros(self.n, np.uint8)
        self._ck(self.lib.miagpu_last_pass1_route(self.h, _ptr(r)))
        return r

    def compact_reads(self, keep, revcomp=None):
        keep = np.ascontiguousarray(keep, np.uint8)
        rv = None if revcomp is None else np.ascontiguousarray(revcomp, np.uint8)
        n = C.c_int64()
        self._ck(self.lib.miagpu_compact_reads(self.h, _ptr(keep), _ptr(rv), C.byref(n)))
        self.n = n.value
        return self.n

    # -- iteration regime
    @staticmethod
    def alloc_realign_outputs(n, pinned=False):
        def mk(shape, dt):
            if pinned:
                import torch
                return torch.empty(shape, dtype=getattr(torch, dt), pin_memory=True)
            return np.empty(shape, dtype=dt)
        return dict(score=mk(n, "int32"), as_out=mk(n, "int32"), ae_out=mk(n, "int32"), abr=mk(n, "int32"),
                    n_runs=mk(n, "int32"), runs=mk((n, MAX_RUNS), "int16" if pinned else "uint16"), status=mk(n, "uint8"))

    def realign(self, rc, as_, ae, out=None):
        """reiterate_assembly's per-read body over the resident reads (mia_main.c:178-257)."""
        n = self.n
        out = out or self.alloc_realign_outputs(n)
        self._ck(self.lib.miagpu_realign(self.h, _ptr(rc), _ptr(as_), _ptr(ae), _ptr(out["score"]), _ptr(out["as_out"]),
                                         _ptr(out["ae_out"]), _ptr(out["abr"]), _ptr(out["n_runs"]), _ptr(out.get("runs")),
                                         _ptr(out["status"])))
        return out

    def align_windows(self, rc, win_start, win_len, sg5=1, out=None):
        """the bare dyn_prog client sequence (ccheck.cc:571-603) of every resident read against its own reference stretch"""
        out = out or self.alloc_realign_outputs(self.n)
        rc, ws, wl = np.ascontiguousarray(rc, np.uint8), np.ascontiguousarray(win_start, np.int32), np.ascontiguousarray(win_len, np.int32)
        self._ck(self.lib.miagpu_align_windows(self.h, _ptr(rc), _ptr(ws), _ptr(wl), int(sg5), _ptr(out["score"]), _ptr(out["as_out"]),
                                               _ptr(out["ae_out"]), _ptr(out["abr"]), _ptr(out["n_runs"]), _ptr(out.get("runs")),
                                               _ptr(out["status"])))
        return out

    def get_runs_packed(self, run_off=None, packed=None):
        """(total, run_off, packed): packed run lists of the last realign / pass 1."""
        tot = C.c_int64()
        cap = 0 if packed is None else (packed.numel() if hasattr(packed, "numel") else packed.size)
        self._ck(self.lib.miagpu_get_runs_packed(self.h, _ptr(run_off), _ptr(packed), cap, C.byref(tot)))
        return tot.value, run_off, packed

    def realign_host(self, bases, offsets, rc, as_, ae, out=None):
        n = len(offsets) - 1
        out = out or self.alloc_realign_outputs(n)
        self._ck(self.lib.miagpu_realign_host(self.h, n, _ptr(bases), _ptr(offsets), _ptr(rc), _ptr(as_), _ptr(ae),
                                              _ptr(out["score"]), _ptr(out["as_out"]), _ptr(out["ae_out"]), _ptr(out["abr"]),
                                              _ptr(out["n_runs"]), _ptr(out.get("runs")), _ptr(out["status"])))
        self.n = n
        return out

    def iterate_host(self, bases, offsets, rc, as_, ae, seq_len, dropped, out=None, packed=None, cons_code=1, unique_best=None,
                     hard_cut=0, score_cut=None, want_gaps=False):
        """One whole iteration for a host-resident batch (miagpu_iterate_host).  `dropped` is updated in place (sticky).
        Returns (consensus, out, total_runs, gaps)."""
        n = len(offsets) - 1
        out = out or self.alloc_realign_outputs(n)
        if not hasattr(self, "_consbuf") or len(self._consbuf) < self.seq_len * 4 + 4096:
            self._consbuf = C.create_string_buffer(self.seq_len * 4 + 4096)
        cap = 0 if packed is None else (packed.numel() if hasattr(packed, "numel") else packed.size)
        tot, cl = C.c_int64(), C.c_int32()
        gaps = np.zeros(self.seq_len, np.int32) if want_gaps else None
        slope, icpt = score_cut if score_cut is not None else (0.0, 0.0)
        self._ck(self.lib.miagpu_iterate_host(self.h, n, _ptr(bases), _ptr(offsets), _ptr(rc), _ptr(as_), _ptr(ae), _ptr(out["score"]),
                                              _ptr(out["as_out"]), _ptr(out["ae_out"]), _ptr(out["abr"]), _ptr(out["n_runs"]),
                                              _ptr(out["status"]), _ptr(packed), cap, C.byref(tot), _ptr(seq_len), _ptr(unique_best),
                                              hard_cut, 0 if score_cut is None else 1, slope, icpt, _ptr(dropped), cons_code,
                                              _ptr(gaps), self._consbuf, C.byref(cl)))
        self.n = n
        return self._consbuf.value.decode(), out, tot.value, gaps

    def set_cut_inputs(self, seq_len, unique_best=None, dropped=None):
        """Per-read inputs of the score cut, resident from here on (miagpu_set_cut_inputs)."""
        self._ck(self.lib.miagpu_set_cut_inputs(self.h, _ptr(np.ascontiguousarray(seq_len, np.int32)), _ptr(unique_best), _ptr(dropped)))

    def set_fsdb(self, seq_len, score, unique_best=None, strand_known=None, front_slot=None, back_slot=None, n_slots=0, slot_dropped=None,
                 distant_ref=0):
        """The FSDB's pointer state after pass 1 (miagpu_set_fsdb): from here on iterate_resident follows the reference's
        FragSeq -> AlnSeq pointers (slot-indexed sticky flags, stale back pointers, strand-unknown reads)."""
        a = lambda x, dt: None if x is None else np.ascontiguousarray(x, dt)
        sl, sc, uq, sk = a(seq_len, np.int32), a(score, np.int32), a(unique_best, np.uint8), a(strand_known, np.uint8)
        fs, bs, sd = a(front_slot, np.int32), a(back_slot, np.int32), a(slot_dropped, np.uint8)
        self._ck(self.lib.miagpu_set_fsdb(self.h, _ptr(sl), _ptr(uq), _ptr(sc), _ptr(sk), _ptr(fs), _ptr(bs), int(n_slots), _ptr(sd), int(distant_ref)))

    def get_fsdb(self):
        n = self.n
        o = dict(strand_known=np.zeros(n, np.uint8), rc=np.zeros(n, np.uint8), front_slot=np.zeros(n, np.int32), back_slot=np.zeros(n, np.int32),
                 dropped_front=np.zeros(n, np.uint8), dropped_back=np.zeros(n, np.uint8))
        ns = C.c_int64()
        self._ck(self.lib.miagpu_get_fsdb(self.h, *[_ptr(o[k]) for k in ("strand_known", "rc", "front_slot", "back_slot", "dropped_front",
                                                                        "dropped_back")], C.byref(ns)))
        o["n_slots"] = ns.value
        return o

    def last_fsdb_stats(self):
        v = [C.c_int64() for _ in range(4)]
        self._ck(self.lib.miagpu_last_fsdb_stats(self.h, *[C.byref(x) for x in v]))
        return dict(n_slots=v[0].value, stale_pointers=v[1].value, extra_entries=v[2].value, frozen=v[3].value)

    def distant_retry(self):
        """-D: whole-reference attempts of the strand-unknown reads (miagpu_distant_retry) -> (tried, learned)"""
        a, b = C.c_int64(), C.c_int64()
        self._ck(self.lib.miagpu_distant_retry(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def distant_retry_begin(self):
        """-D over several shards, step 1 (miagpu_distant_retry_begin) -> (tried, [state after the last local read if the first
        is entered with the forward matrix, ... with the strand-reversed one])"""
        a, st = C.c_int64(), (C.c_int32 * 2)()
        self._ck(self.lib.miagpu_distant_retry_begin(self.h, C.byref(a), st))
        return a.value, [int(st[0]), int(st[1])]

    def distant_retry_end(self, state_in):
        """step 2: the local chain entered with state_in -> learned"""
        b = C.c_int64()
        self._ck(self.lib.miagpu_distant_retry_end(self.h, int(state_in), C.byref(b)))
        return b.value

    def misincorporation(self):
        """Damage profile of the last round (miagpu_misincorporation): int64[31, 6, 6] = counts[depth][reference][read] over
        MISINC_CODES, in the orientation of the molecule (depth 0 = its 5' end), cell for cell the forward matrix's."""
        t = np.zeros(MISINC_SHAPE, np.int64)
        self._ck(self.lib.miagpu_misincorporation(self.h, t.ctypes.data_as(_i64p)))
        return t

    def reset_dropped(self):
        self._ck(self.lib.miagpu_reset_dropped(self.h))

    def iterate_resident(self, cons_code=1, hard_cut=0, score_cut=None, dropped=None, want_gaps=False):
        """One whole iteration over resident inputs (miagpu_iterate_resident).
        Returns (consensus, (slope, intercept), gaps); `dropped` (uint8[n], optional) receives the sticky flags."""
        if not hasattr(self, "_consbuf") or len(self._consbuf) < self.seq_len * 4 + 4096:
            self._consbuf = C.create_string_buffer(self.seq_len * 4 + 4096)
        cl = C.c_int32()
        gaps = np.zeros(self.seq_len, np.int32) if want_gaps else None
        slope, icpt = score_cut if score_cut is not None else (0.0, 0.0)
        so, io = C.c_double(), C.c_double()
        self._ck(self.lib.miagpu_iterate_resident(self.h, hard_cut, 0 if score_cut is None else 1, slope, icpt, cons_code, C.byref(so),
                                                  C.byref(io), _ptr(dropped), _ptr(gaps), self._consbuf, C.byref(cl)))
        return self._consbuf.value.decode(), (so.value, io.value), gaps

    # -- sharded rounds (SURVEY 8e): three phases with one collective after each of the first two (see shard.py)
    def shard_begin(self, world, rank, n_max, hard_cut=0, score_cut=None):
        """-> (ptr, words) of the device buffer to MAX-reduce (insert maxima, best scores, the ranks' header rows)"""
        mb, mw = C.c_void_p(), C.c_int64()
        slope, icpt = score_cut if score_cut is not None else (0.0, 0.0)
        self._ck(self.lib.miagpu_shard_begin(self.h, world, rank, n_max, hard_cut, 0 if score_cut is None else 1, slope, icpt,
                                             C.byref(mb), C.byref(mw)))
        return mb.value, mw.value

    def shard_begin_host(self, world, rank, n_max, bases, offsets, rc, as_, ae, seq_len, dropped, out, unique_best=None, hard_cut=0,
                         score_cut=None):
        n = len(offsets) - 1
        mb, mw = C.c_void_p(), C.c_int64()
        slope, icpt = score_cut if score_cut is not None else (0.0, 0.0)
        self._ck(self.lib.miagpu_shard_begin_host(self.h, world, rank, n_max, n, _ptr(bases), _ptr(offsets), _ptr(rc), _ptr(as_), _ptr(ae),
                                                  _ptr(out["score"]), _ptr(out["as_out"]), _ptr(out["ae_out"]), _ptr(out["abr"]),
                                                  _ptr(out["n_runs"]), _ptr(out["status"]), _ptr(seq_len), _ptr(unique_best), _ptr(dropped),
                                                  hard_cut, 0 if score_cut is None else 1, slope, icpt, C.byref(mb), C.byref(mw)))
        self.n = n
        return mb.value, mw.value

    def shard_fit(self):
        """-> dict(send=(ptr, words), recv=(ptr, world * words)) of the block records to all-gather (words = 0: nothing to gather)"""
        gs, gr, gw = C.c_void_p(), C.c_void_p(), C.c_int64()
        self._ck(self.lib.miagpu_shard_fit(self.h, C.byref(gs), C.byref(gr), C.byref(gw)))
        return dict(send=(gs.value, gw.value), recv=(gr.value, gw.value))

    def shard_cut(self):
        """-> ((slope, intercept), (ptr, words) of the column planes to SUM-reduce)"""
        so, io, sb, sw = C.c_double(), C.c_double(), C.c_void_p(), C.c_int64()
        self._ck(self.lib.miagpu_shard_cut(self.h, C.byref(so), C.byref(io), C.byref(sb), C.byref(sw)))
        return (so.value, io.value), (sb.value, sw.value)

    def shard_finish(self, cons_code=1, dropped=None, packed=None, want_gaps=False, want_total_runs=False):
        """-> (consensus, gaps or None, total_runs or None)"""
        if not hasattr(self, "_consbuf") or len(self._consbuf) < self.seq_len * 4 + 4096:
            self._consbuf = C.create_string_buffer(self.seq_len * 4 + 4096)
        cl, tot = C.c_int32(), C.c_int64()
        gaps = np.zeros(self.seq_len, np.int32) if want_gaps else None
        cap = 0 if packed is None else (packed.numel() if hasattr(packed, "numel") else packed.size)
        want_tot = want_total_runs or packed is not None
        self._ck(self.lib.miagpu_shard_finish(self.h, cons_code, _ptr(dropped), _ptr(packed), cap, C.byref(tot) if want_tot else None,
                                              _ptr(gaps), self._consbuf, C.byref(cl)))
        return self._consbuf.value.decode(), gaps, (tot.value if want_tot else None)

    def shard_flags(self):
        """-> (ptr, bytes) of the slot flags to MAX-reduce over the ranks after shard_finish (bytes = 0: no pointer state)"""
        b, n = C.c_void_p(), C.c_int64()
        self.lib.miagpu_shard_flags.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), _i64p]
        self._ck(self.lib.miagpu_shard_flags(self.h, C.byref(b), C.byref(n)))
        return b.value, n.value

    def last_cut_stats(self):
        a, b = C.c_int64(), C.c_int64()
        self._ck(self.lib.miagpu_last_cut_stats(self.h, C.byref(a), C.byref(b)))
        return dict(serial_blocks=a.value, fetched_blocks=b.value)

    # -- adapter trimming (8f4)
    def trim(self, bases, offsets, adapter):
        """trim_frag for a batch: -> dict(score, abr, abc, aer, trimmed, trim_point) of numpy arrays"""
        n = len(offsets) - 1
        o = dict(score=np.zeros(n, np.int32), abr=np.zeros(n, np.int32), abc=np.zeros(n, np.int32), aer=np.zeros(n, np.int32),
                 trimmed=np.zeros(n, np.uint8), trim_point=np.zeros(n, np.int32))
        ad = adapter if isinstance(adapter, bytes) else adapter.encode()
        self._ck(self.lib.miagpu_trim(self.h, n, _ptr(bases), _ptr(offsets), ad, len(ad), _ptr(o["score"]), _ptr(o["abr"]), _ptr(o["abc"]),
                                      _ptr(o["aer"]), _ptr(o["trimmed"]), _ptr(o["trim_point"])))
        return o

    # -- repeat filter (8f1)
    def repeat_filter(self, rc, as_, ae, key4, trimmed=None, just_outer_coords=1, tolerance=0, want_order=True):
        """sort_fsdb[_qscore] + set_uniq_in_fsdb: -> (order int64[n] or None, unique_best uint8[n] by input index)"""
        n = len(rc)
        rc = np.ascontiguousarray(rc, np.uint8); as_ = np.ascontiguousarray(as_, np.int32); ae = np.ascontiguousarray(ae, np.int32)
        key4 = np.ascontiguousarray(key4, np.int32)
        tr = None if trimmed is None else np.ascontiguousarray(trimmed, np.uint8)
        order = np.zeros(n, np.int64) if want_order else None
        uniq = np.zeros(n, np.uint8)
        self._ck(self.lib.miagpu_repeat_filter(self.h, n, _ptr(rc), _ptr(as_), _ptr(ae), _ptr(key4), _ptr(tr), int(just_outer_coords),
                                               int(tolerance), _ptr(order), _ptr(uniq)))
        return order, uniq

    # -- consensus
    def consensus(self, entries, cons_code=1, want_counts=False):
        """consensus_assembly_string over the culled entry list (mia.c:515-603).
        Returns (consensus, gaps[seq_len], counts[seq_len,10] or None)."""
        entries = np.ascontiguousarray(entries, ENTRY_DTYPE)
        gaps = np.zeros(self.seq_len, np.int32)
        counts = np.zeros((self.seq_len, 10), np.int32) if want_counts else None
        buf = C.create_string_buffer(self.seq_len * 2 + 1024 + len(entries) * 4)
        n = C.c_int32()
        self._ck(self.lib.miagpu_consensus(self.h, len(entries), _ptr(entries), cons_code, _ptr(gaps), _ptr(counts), buf, C.byref(n)))
        return buf.value.decode(), gaps, counts

    def consensus_natural(self, dropped_front=None, dropped_back=None, cons_code=1, want_counts=False, want_gaps=True):
        gaps = np.zeros(self.seq_len, np.int32) if want_gaps else None
        counts = np.zeros((self.seq_len, 10), np.int32) if want_counts else None
        if not hasattr(self, "_consbuf") or len(self._consbuf) < self.seq_len * 4 + 4096:
            self._consbuf = C.create_string_buffer(self.seq_len * 4 + 4096)
        n = C.c_int32()
        self._ck(self.lib.miagpu_consensus_natural(self.h, _ptr(dropped_front), _ptr(dropped_back), cons_code, _ptr(gaps),
                                                   _ptr(counts), self._consbuf, C.byref(n)))
        return self._consbuf.value.decode(), gaps, counts

    def accumulate_gaps_natural(self, dropped_front=None, dropped_back=None):
        ptr, n = C.c_void_p(), C.c_int64()
        self._ck(self.lib.miagpu_accumulate_gaps_natural(self.h, _ptr(dropped_front), _ptr(dropped_back), C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def set_alignment_inputs(self, rc, as_, ae):
        self._ck(self.lib.miagpu_set_alignment_inputs(self.h, _ptr(rc), _ptr(as_), _ptr(ae)))

    def adopt_alignment(self, want=True):
        """this round's as / ae become the next round's inputs; -> (score, as, ae) of this round if want"""
        if not want:
            self._ck(self.lib.miagpu_adopt_alignment(self.h, None, None, None))
            return None
        sc, a, e = np.zeros(self.n, np.int32), np.zeros(self.n, np.int32), np.zeros(self.n, np.int32)
        self._ck(self.lib.miagpu_adopt_alignment(self.h, _ptr(sc), _ptr(a), _ptr(e)))
        return sc, a, e

    def get_alignment(self):
        """the alignment the last round left on the device (miagpu_get_alignment) -> dict like realign's, without runs"""
        out = {k: np.zeros(self.n, np.int32) for k in ("score", "as_out", "ae_out", "abr", "n_runs")}
        out["status"] = np.zeros(self.n, np.uint8)
        self._ck(self.lib.miagpu_get_alignment(self.h, *[_ptr(out[k]) for k in ("score", "as_out", "ae_out", "abr", "n_runs", "status")]))
        return out

    def realign_resident(self):
        self._ck(self.lib.miagpu_realign_resident(self.h))

    def last_buckets(self):
        k, r, cells, ms = np.zeros(10, np.int32), np.zeros(10, np.int32), np.zeros(10, np.int64), np.zeros(10, np.float32)
        self._ck(self.lib.miagpu_last_buckets(self.h, _ptr(k), _ptr(r), _ptr(cells), _ptr(ms)))
        return [dict(K=int(k[i]), reads=int(r[i]), cells=int(cells[i]), ms=float(ms[i])) for i in range(10) if r[i]]

    def last_pair_buckets(self):
        """16-bit pair kernels of the last realign: (list of per-class dicts, reads handed to the 32-bit kernels, max read length)."""
        k, r, pr = np.zeros(8, np.int32), np.zeros(8, np.int32), np.zeros(8, np.int32)       # MIAGPU_NPAIRCLASS
        cells, ms = np.zeros(8, np.int64), np.zeros(8, np.float32)
        fb, ml = C.c_int32(), C.c_int32()
        self._ck(self.lib.miagpu_last_pair_buckets(self.h, _ptr(k), _ptr(r), _ptr(pr), _ptr(cells), _ptr(ms), C.byref(fb), C.byref(ml)))
        return ([dict(K=int(k[i]), reads=int(r[i]), pairs=int(pr[i]), cells=int(cells[i]), ms=float(ms[i])) for i in range(8) if r[i]],
                fb.value, ml.value)

    def accumulate_gaps(self, entries):
        entries = np.ascontiguousarray(entries, ENTRY_DTYPE)
        ptr, n = C.c_void_p(), C.c_int64()
        self._ck(self.lib.miagpu_accumulate_gaps(self.h, len(entries), _ptr(entries), C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def accumulate_counts(self):
        ptr, n = C.c_void_p(), C.c_int64()
        self._ck(self.lib.miagpu_accumulate_counts(self.h, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def call(self, cons_code=1, want_counts=False, max_len=None):
        gaps = np.zeros(self.seq_len, np.int32)
        counts = np.zeros((self.seq_len, 10), np.int32) if want_counts else None
        buf = C.create_string_buffer(max_len or (self.seq_len * 4 + 4096))
        n = C.c_int32()
        self._ck(self.lib.miagpu_call(self.h, cons_code, _ptr(gaps), _ptr(counts), buf, C.byref(n)))
        return buf.value.decode(), gaps, counts

    def last_timing(self):
        k, h, d = C.c_float(), C.c_float(), C.c_float()
        cells, launches = C.c_int64(), C.c_int32()
        self._ck(self.lib.miagpu_last_timing(self.h, C.byref(k), C.byref(h), C.byref(d), C.byref(cells), C.byref(launches)))
        return dict(ms_kernels=k.value, ms_h2d=h.value, ms_d2h=d.value, dp_cells=cells.value, launches=launches.value)

    def int32_peak(self):
        v = C.c_double()
        self._ck(self.lib.miagpu_int32_peak(self.h, C.byref(v)))
        return v.value


def expand_runs(ref, read, start, abr, runs, n_runs):
    """Gapped strings (PWAlnFrag.ref_seq / frag_seq, mia.c:1440-1497) from a run list.
    ref must be indexable at reference coordinates (wrapped); start = first ref column."""
    rg, fg = [], []
    c, r = start, abr
    for x in runs[:n_runs]:
        x = int(x) & 0xFFFF
        t, ln = x >> 14, x & 0x3FFF
        if t == RUN_M:
            rg.append(ref[c:c + ln]); fg.append(read[r:r + ln]); c += ln; r += ln
        elif t == RUN_I:
            rg.append("-" * ln); fg.append(read[r:r + ln]); r += ln
        else:
            rg.append(ref[c:c + ln]); fg.append("-" * ln); c += ln
    return "".join(rg), "".join(fg)


def score_cut(seq_len, score, unique_best=None):
    """find_fsdb_score_cut (fsdb.c:269-383) -> (slope, intercept)."""
    L = load_library()
    sl, sc = np.ascontiguousarray(seq_len, np.int32), np.ascontiguousarray(score, np.int32)
    s, i = C.c_double(), C.c_double()
    if not L.miagpu_score_cut(len(sl), _ptr(sl), _ptr(sc), _ptr(unique_best), C.byref(s), C.byref(i)):
        raise MiaGpuError(L.miagpu_last_error().decode())
    return s.value, i.value


def cull_flags(seq_len, score, unique_best=None, hard_cut=0, score_cut_set=0, slope=200.0, intercept=0.0, out=None):
    """Per-read `score < min_score_for_len` of cull_maln_from_fsdb (mia.c:418-479)."""
    L = load_library()
    n = len(seq_len)
    out = np.zeros(n, np.uint8) if out is None else out
    if not L.miagpu_cull_flags(n, _ptr(seq_len), _ptr(score), _ptr(unique_best), hard_cut, score_cut_set, slope, intercept, _ptr(out)):
        raise MiaGpuError(L.miagpu_last_error().decode())
    return out


# ---------------------------------------------------------------- host formats either side of the path (SURVEY 8 f2 / f3)
class FastxReader:
    """find_input_type + read_fasta / read_fastq (io.c:11-281) as mia_main.c:746-759 drives them: batches of records
    ready for upload_reads (miagpu_fastx_*).  Host only."""

    def __init__(self, path=None, text=None):
        self.lib = load_library()
        self.h = C.c_void_p()
        if path is not None:
            ok = self.lib.miagpu_fastx_open(C.byref(self.h), os.fsencode(path))
        else:
            self._text = text if isinstance(text, bytes) else text.encode("latin-1")
            ok = self.lib.miagpu_fastx_open_memory(C.byref(self.h), self._text, len(self._text))
        if not ok:
            raise MiaGpuError(self.lib.miagpu_last_error().decode())
        self.format = self.lib.miagpu_fastx_format(self.h)

    def close(self):
        if self.h:
            self.lib.miagpu_fastx_close(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def next(self, max_reads=1 << 20):
        """-> dict(n, bases uint8, offsets int64[n+1], ids bytes, id_off, descs bytes, desc_off, qual_sum) (copies) or None at the end"""
        n = C.c_int64()
        if not self.lib.miagpu_fastx_next(self.h, max_reads, C.byref(n)):
            raise MiaGpuError(self.lib.miagpu_last_error().decode())
        n = n.value
        if n == 0:
            return None
        p = [C.c_void_p() for _ in range(7)]
        self.lib.miagpu_fastx_batch(self.h, *[C.byref(x) for x in p])

        def arr(ptr, count, dt):
            if count == 0:
                return np.zeros(0, dt)
            nbytes = count * np.dtype(dt).itemsize
            return np.frombuffer(C.string_at(ptr.value, nbytes), dt).copy()
        off = arr(p[1], n + 1, np.int64)
        id_off = arr(p[3], n + 1, np.int64)
        desc_off = arr(p[5], n + 1, np.int64)
        return dict(n=n, bases=arr(p[0], int(off[-1]), np.uint8), offsets=off, ids=C.string_at(p[2].value, int(id_off[-1])), id_off=id_off,
                    descs=C.string_at(p[4].value, int(desc_off[-1])), desc_off=desc_off, qual_sum=arr(p[6], n, np.int32))

    @staticmethod
    def strings(blob, off):
        return [blob[off[i]:off[i + 1] - 1].decode("latin-1") for i in range(len(off) - 1)]


class _MalnHeader(C.Structure):
    _fields_ = [("ref_id", C.c_char_p), ("ref_desc", C.c_char_p), ("ref_seq", C.c_char_p), ("ref_len", C.c_int32), ("circular", C.c_int32),
                ("ref_size", C.c_int32), ("maln_size", C.c_int32), ("cons_code", C.c_int32), ("gaps", C.c_void_p), ("fpsm", C.c_void_p),
                ("rpsm", C.c_void_p)]


class _MalnReads(C.Structure):
    _fields_ = [("n", C.c_int64)] + [(k, C.c_void_p) for k in
                                     ("bases", "offsets", "ids", "id_off", "descs", "desc_off", "rc", "trimmed", "num_inputs", "score", "as_",
                                      "ae", "abr", "run_off", "packed", "unique_best", "dropped_front", "dropped_back", "fsdb_order")]


def read_pssm(path):
    """read_pssm (io.c:408-503) -> int32[31, 5, 5]"""
    L = load_library()
    sm = np.zeros(775, np.int32)
    if not L.miagpu_read_pssm(os.fsencode(path), sm.ctypes.data_as(_i32p)):
        raise MiaGpuError(L.miagpu_last_error().decode())
    return sm.reshape(31, 5, 5)


def maln_ref_size(ref_len, circular):
    return load_library().miagpu_maln_ref_size(ref_len, circular)


def write_maln(path, ref_id, ref_desc, ref_seq, circular, maln_size, cons_code, gaps, fpsm, rpsm, reads):
    """write_ma (map_alignment.c:283-382) from per-read device results (miagpu_write_maln).  `reads`: dict with bases (STORED
    orientation), offsets, ids (bytes blob), id_off, descs, desc_off, rc, score, as_, ae, abr, run_off, packed and optionally
    trimmed, num_inputs, unique_best, dropped_front, dropped_back.  -> number of AlnSeqs written."""
    L = load_library()
    keep = []

    def a(x, dt):
        if x is None:
            return None
        x = np.ascontiguousarray(x, dt)
        keep.append(x)
        return x.ctypes.data

    def blob(x):
        if x is None:
            return None
        b = C.create_string_buffer(bytes(x), len(x))
        keep.append(b)
        return C.addressof(b)
    hd = _MalnHeader(ref_id.encode(), ref_desc.encode(), ref_seq.encode(), len(ref_seq), int(circular), 0, int(maln_size), int(cons_code),
                     a(gaps, np.int32), a(fpsm, np.int32), a(rpsm, np.int32))
    r = reads
    rd = _MalnReads(len(r["offsets"]) - 1, a(r["bases"], np.uint8), a(r["offsets"], np.int64), blob(r["ids"]), a(r["id_off"], np.int64),
                    blob(r.get("descs")), a(r.get("desc_off"), np.int64), a(r["rc"], np.uint8), a(r.get("trimmed"), np.uint8),
                    a(r.get("num_inputs"), np.int32), a(r["score"], np.int32), a(r["as_"], np.int32), a(r["ae"], np.int32),
                    a(r["abr"], np.int32), a(r["run_off"], np.int64), a(r["packed"], np.uint16), a(r.get("unique_best"), np.uint8),
                    a(r.get("dropped_front"), np.uint8), a(r.get("dropped_back"), np.uint8), a(r.get("fsdb_order"), np.int64))
    n_out = C.c_int64()
    if not L.miagpu_write_maln(os.fsencode(path), C.byref(hd), C.byref(rd), C.byref(n_out)):
        raise MiaGpuError(L.miagpu_last_error().decode())
    return n_out.value
