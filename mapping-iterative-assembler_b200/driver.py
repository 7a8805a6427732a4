"""Host-side mirror of mia_main.c's control flow (lines 759-976) on top of the C ABI.

The reference's host code stays what it is -- one pass over the reads, then
"reiterate_assembly -> pop_smp -> cull -> consensus" until the consensus stops changing.
This module is that loop with the hot calls replaced by libmiagpu entry points, plus the
reference's own bookkeeping that decides WHAT is fed to the consensus:

  * AlnSeq slots are numbered in merge order, 1 per read, 2 per wrap-split read
    (merge_pwaln_into_maln, map_align.c:866-954);
  * AlnSeq.dropped is sticky per slot (H10: cull only sets it, mia.c:471-478; merge copies
    every field except it, map_align.c:885-893);
  * FragSeq.back_asp is never cleared by reiterate_assembly (mia_main.c:273-276): a read that
    was split once keeps pointing at its old back slot; pop_smp, cull and the consensus follow
    that pointer.  A stale pointer to a slot that is live this round is described to the
    device as an extra entry on the owner's segment (with the smp parameters of whichever
    pointer pop_smp visits last); a stale pointer to a slot beyond this round's slot count
    (content from an older round) is not reproduced and is reported in `self.ghosts`.

Used by tests and bench; a C host would make the same calls (INTEGRATION.md).
"""
import numpy as np

from . import api
from .api import ENTRY_DTYPE, MAX_RUNS

FIRST_ROUND_SCORE_CUTOFF = 2000
MAX_ITER = 30


def _geom(runs_i, n, cut=None):
    """(cols, ins, dels) of the alignment columns [0,cut) and [cut, end) (cut=None: everything in the first)."""
    g = [[0, 0, 0], [0, 0, 0]]
    col = 0
    for x in runs_i[:n]:
        x = int(x)
        t, ln = x >> 14, x & 0x3FFF
        if t == 1:
            g[0 if (cut is None or col < cut) else 1][1] += ln
            continue
        for _ in range(ln):                      # rare path (split reads only): per-column is fine
            s = 0 if (cut is None or col < cut) else 1
            g[s][0] += 1
            if t == 2:
                g[s][2] += 1
            col += 1
    return g


class Assembler:
    def __init__(self, gpu, ref, sm, circular=1, k=0, soft_mask=0, cons_code=1):
        self.g, self.sm, self.circular, self.k, self.soft_mask, self.cons_code = gpu, sm, circular, k, soft_mask, cons_code
        self.ref0 = ref
        self.ghosts = 0
        gpu.set_pssm(sm)

    # ------------------------------------------------------------------ pass 1
    def pass1(self, bases, off):
        g = self.g
        g.set_reference(self.ref0, self.circular, with_rc=1)
        g.build_kmers(self.k, self.soft_mask)
        g.upload_reads(bases, off)
        p = g.pass1()
        self.p1 = p
        n = len(off) - 1
        seq_len = np.diff(off).astype(np.int32)
        aligned = p["hits"] > 0
        keep = aligned & (p["score"] >= FIRST_ROUND_SCORE_CUTOFF)                   # mia.c:1614
        strand_known = keep & (p["score"] > FIRST_ROUND_SCORE_CUTOFF)               # mia.c:1653
        idx = np.flatnonzero(keep)
        # pass-1 AlnSeq slots, in merge order (mia.c:1619-1643); back_asp = NULL unless split
        split = p["start"][idx] > p["end"][idx]
        nsl = 1 + split.astype(np.int64)
        first = np.concatenate([[0], np.cumsum(nsl)[:-1]]) if len(idx) else np.zeros(0, np.int64)
        self.dropped_slot = np.zeros(int(nsl.sum()) + 16, np.uint8)
        self.seq_len = seq_len[idx]
        self.score = p["score"][idx].copy()
        self.rc = p["rc"][idx].copy()
        self.as_ = p["as_"][idx].copy()
        self.ae = p["ae"][idx].copy()
        self.strand_known = strand_known[idx]
        self.front = first.astype(np.int64)
        self.back = np.where(split, first + 1, -1).astype(np.int64)
        # pass-1 cull (mia_main.c:848): only its dropped flags survive
        self._cull()
        # clean_FSDB (mia.c:400-406) and stored orientation (fsdb.c:209-227)
        ok = self.score > 0
        keep_dev = np.zeros(n, np.uint8)
        keep_dev[idx[ok]] = 1
        rev = np.zeros(n, np.uint8)
        rev[idx] = (self.rc == 1) & self.strand_known
        g.compact_reads(keep_dev, rev)
        for name in ("seq_len", "score", "rc", "as_", "ae", "strand_known", "front", "back"):
            setattr(self, name, getattr(self, name)[ok])
        if not self.strand_known.all():
            raise NotImplementedError("reads with score == 2000 keep strand_known = 0 and are never realigned (mia.c:1653)")
        self.iter = 0
        self.cons = None
        self.last = self.ref0.upper()
        return p

    def _cull(self):
        below = api.cull_flags(self.seq_len, self.score)
        need = int(max(self.front.max(initial=0), self.back.max(initial=0))) + 2
        if need > len(self.dropped_slot):
            self.dropped_slot = np.concatenate([self.dropped_slot, np.zeros(need, np.uint8)])
        f = self.front[below > 0]
        self.dropped_slot[f] = 1
        b = self.back[(below > 0) & (self.back >= 0)]
        self.dropped_slot[b] = 1

    # --------------------------------------------------------------- one round
    def iterate(self):
        """mia_main.c:878-900 / 918-963: realign everything against the current consensus, cull, call."""
        g = self.g
        if self.cons is not None:
            self.last = self.cons
        self.iter += 1
        ref = self.last
        g.set_reference(ref, self.circular, with_rc=0)
        out = g.realign(self.rc, self.as_, self.ae)
        self.out = out
        if (out["status"] != 0).any():
            raise api.MiaGpuError(f"realign status bits set on {(out['status'] != 0).sum()} reads")
        self.as_, self.ae, self.score = out["as_out"].copy(), out["ae_out"].copy(), out["score"].copy()
        n, L = len(self.as_), len(ref)
        runs = out["runs"].view(np.uint16).reshape(-1, MAX_RUNS)
        end = np.where(self.ae > L, self.ae - L, self.ae)
        split = self.as_ > end
        nsl = 1 + split.astype(np.int64)
        first = np.concatenate([[0], np.cumsum(nsl)[:-1]])
        n_slots = int(nsl.sum())
        self.front = first
        self.back = np.where(split, first + 1, self.back)              # NOT cleared when not split: mia_main.c:273-276
        self._cull()
        # ---- natural entries (vectorised), then the alias fix-ups
        from .entries import natural_entries
        ent, _, _ = natural_entries(self.as_, self.ae, out["n_runs"], runs, L)
        slot_entry = np.arange(n_slots)                                # natural entry index of slot k == k
        ent["dropped"] = self.dropped_slot[:n_slots]
        stale = np.flatnonzero(~split & (self.back >= 0))
        extra = []
        if len(stale):
            owner = np.repeat(np.arange(n), nsl)                       # slot -> owning read
            last_holder = {}
            for i in stale:
                kslot = int(self.back[i])
                if kslot >= n_slots:
                    self.ghosts += 1
                    continue
                j = int(owner[kslot])
                seg = kslot - int(first[j])
                e_own = ent[slot_entry[kslot]]
                gi = _geom(runs[i], int(out["n_runs"][i]))[0]
                fl_i = gi[0] + gi[1]
                bases_f_i = gi[0] - gi[2] + gi[1]
                bl = int(e_own["col_count"]) + self._slot_ins(runs[j], int(out["n_runs"][j]), int(e_own["col_begin"]), int(e_own["col_count"]))
                # the holder's own front AlnSeq sees back_seq_len = asp_len(stale slot) (fsdb.c:554-559)
                ent["total_len"][slot_entry[first[i]]] = fl_i + bl
                rb = 0
                if seg == 1:
                    gj = _geom(runs[j], int(out["n_runs"][j]), int(e_own["col_begin"]))[0]
                    rb = gj[0] - gj[2] + gj[1]
                x = e_own.copy()
                x["back_formula"], x["front_len"], x["total_len"], x["act_bias"] = 1, fl_i, fl_i + bl, bases_f_i - rb
                extra.append((kslot, i, x))
                if i > j and i > last_holder.get(kslot, (-1,))[0]:
                    last_holder[kslot] = (i, x)
            for kslot, (_, x) in last_holder.items():                  # pop_smp visits this pointer last: its smp sticks
                for fld in ("back_formula", "front_len", "total_len", "act_bias"):
                    ent[fld][slot_entry[kslot]] = x[fld]
            add = []
            for kslot, i, x in extra:                                  # every pointer is one list entry; same AlnSeq => same smp
                y = ent[slot_entry[kslot]].copy()
                add.append(y)
            if add:
                ent = np.concatenate([ent, np.array(add, ENTRY_DTYPE)])
        self.entries = ent
        cons, gaps, _ = g.consensus(ent, self.cons_code)
        self.gaps = gaps
        self.cons = cons
        return cons, cons == self.last

    @staticmethod
    def _slot_ins(runs_i, n, cb, cc):
        """inserted bases attached to alignment columns [cb, cb+cc) (asp_len's second term)"""
        col, tot = 0, 0
        for x in runs_i[:n]:
            x = int(x)
            t, ln = x >> 14, x & 0x3FFF
            if t == 1:
                if cb <= col < cb + cc:
                    tot += ln
            else:
                col += ln
        return tot

    def run(self, bases, off, max_iter=MAX_ITER):
        self.pass1(bases, off)
        conv = False
        while not conv and self.iter < max_iter:
            _, conv = self.iterate()
        return self.cons, self.iter, conv


class ResidentAssembler:
    """The same loop with everything resident in HBM and one library call per round (miagpu_iterate_resident, or the
    sharded protocol when `world` > 1): the path for large read sets (BASELINE configs[2]..[4]).

    On one GPU the FSDB's pointer state goes to the device after pass 1 (miagpu_set_fsdb) and the rounds follow the reference's
    FragSeq -> AlnSeq pointers there: slot-indexed sticky dropped flags (H10), never-cleared back pointers (mia_main.c:273-276),
    reads that score exactly 2000 (strand_known = 0, mia.c:1653) and -D (`distant_ref`: mia.c:1614, mia_main.c:120-174,
    find_alignable_len in the cull).  Sharded rounds do the same with `pointer_state=True` (global slot numbers, slot flags
    replicated, the -D chain passed from shard to shard: `retry_begin` / `retry_end`); without it every read gets its own
    fresh segments and one sticky flag, and what that misses is counted in `split_changes`.

    `exchange`: None for one GPU; otherwise an object with
        all_gather_host(np_array) -> concatenation over ranks in rank order
        rounds                    -> shard.ShardedRounds (or anything with .resident(...))
    """

    def __init__(self, gpu, ref, sm, circular=1, k=0, soft_mask=0, cons_code=1, exchange=None, strand_unknown="raise", distant_ref=0,
                 pointer_state=None, hp=0):
        """strand_unknown ("raise" / "drop") only matters without the pointer state (sharded rounds), which does not model reads that
        score exactly 2000.  pointer_state: None = on unless `exchange` is given.  hp: mia -h (miagpu_set_homopolymer; the caller's
        context keeps the mode until it is switched off)."""
        self.g, self.sm, self.circular, self.k, self.soft_mask, self.cons_code = gpu, sm, circular, k, soft_mask, cons_code
        self.ref0, self.x = ref, exchange
        self.split_changes = 0
        self.strand_unknown, self.strand_unknown_reads = strand_unknown, 0
        self.distant_ref = int(distant_ref)
        self.fs = (exchange is None) if pointer_state is None else bool(pointer_state)
        if self.distant_ref and not self.fs:
            raise NotImplementedError("-D needs the pointer state (pointer_state=True)")
        self.matrix_state = 0                                                        # H6 over shards: which matrix the last read of the last shard left
        self._manual_retry = False                                                   # True: the caller drives retry_begin / retry_end (shards without an exchange object)
        gpu.set_pssm(sm)
        gpu.set_homopolymer(hp)

    def _gather(self, a):
        return a if self.x is None else self.x.all_gather_host(a)

    def pass1(self, bases, off, defer_cull=False):
        g = self.g
        g.set_reference(self.ref0, self.circular, with_rc=1)
        g.build_kmers(self.k, self.soft_mask)
        g.upload_reads(bases, off)
        p = g.pass1(fields=("hits", "score", "rc", "as_", "ae", "start", "end"))
        self.p1 = p
        seq_len = np.diff(off).astype(np.int32)
        keep = (p["hits"] > 0) & ((p["score"] >= FIRST_ROUND_SCORE_CUTOFF) | bool(self.distant_ref))   # mia.c:1614
        unknown = keep & (p["score"] <= FIRST_ROUND_SCORE_CUTOFF)                                       # mia.c:1653
        if not self.fs and unknown.any():
            if self.strand_unknown != "drop":
                raise NotImplementedError("sharded rounds: reads with score == 2000 keep strand_known = 0 and are never realigned (mia.c:1653)")
            self.strand_unknown_reads = int(unknown.sum())
            keep &= ~unknown
            unknown[:] = False
        idx = np.flatnonzero(keep)
        self._idx, self._n_all = idx, len(seq_len)
        self.seq_len, self.score = seq_len[idx], p["score"][idx].copy()
        self.rc, self.as_, self.ae = p["rc"][idx].copy(), p["as_"][idx].copy(), p["ae"][idx].copy()
        self.strand_known = ~unknown[idx]
        self.split = p["start"][idx] > p["end"][idx]                                 # mia.c:1619
        self.maln_size = int(len(idx) + self.split.sum())                            # culled_maln->size (mia.c:54): AlnSeqs of pass 1
        if self.x is not None:
            counts = self._gather(np.array([len(self.seq_len)], np.int64))            # reads per rank, in rank order
            lo = int(counts[: self.x.rank].sum()) if self.fs else 0
            self.pass1_cull(self._gather(self.seq_len), self._gather(self.score), self._gather(self.split.astype(np.uint8)) if self.fs else None, lo,
                            self._gather(self.cull_len()) if self.fs and self.distant_ref else None)
        elif not defer_cull:
            self.pass1_cull(self.seq_len, self.score)
        return p

    def _alignable_len(self, ref_wrapped_upper, wrap_len):
        """find_alignable_len (mia.c:69-91) of every FSDB read against the (wrapped, upper-cased) reference"""
        isn = np.concatenate([[0], np.cumsum(np.frombuffer(ref_wrapped_upper.encode(), np.uint8) == ord("N"))])
        a = np.clip(self.as_.astype(np.int64), 0, wrap_len)
        e = np.clip(np.minimum(self.ae.astype(np.int64), wrap_len), a, wrap_len)
        return np.maximum(self.seq_len - (isn[e] - isn[a]), 15).astype(np.int32)     # MIN_ALIGNABLE_LEN

    def cull_len(self):
        """the length that picks a read's threshold in the pass-1 cull (mia.c:460-463): seq_len, or find_alignable_len under -D"""
        if not self.distant_ref:
            return self.seq_len
        ru = self.ref0.upper()
        rw = ru + (ru[:min(256, len(ru))] if self.circular else "")
        return self._alignable_len(rw, len(rw))

    def pass1_cull(self, all_seq_len, all_score, all_split=None, lo=0, all_cull_len=None):
        """pass-1 cull (mia_main.c:848) with the fit over the reads of ALL ranks in FSDB order: only its dropped flags survive.
        all_split / lo (pointer state over several shards): the wrap-split flags of all ranks' reads and where this shard's reads
        begin among them -- AlnSeq slots are numbered over all reads, every shard keeps the flags of all slots; all_cull_len: the
        ranks' cull_len() under -D."""
        g, idx = self.g, self._idx
        fit = api.score_cut(all_seq_len, all_score)
        thr_len = self.cull_len()
        dropped = api.cull_flags(thr_len, self.score, None, 0, 1, fit[0], fit[1])
        # AlnSeq slots of pass 1 in merge order (mia.c:1619-1643): one per accepted read, two when wrap-split
        if all_split is None:
            nsl = 1 + self.split.astype(np.int64)
            first = np.cumsum(nsl) - nsl
            n_slots = int(nsl.sum())
            slot_dropped = np.zeros(n_slots + 1, np.uint8)
            slot_dropped[first[dropped > 0]] = 1
            slot_dropped[first[(dropped > 0) & self.split] + 1] = 1
        else:
            asp = np.asarray(all_split).astype(bool)
            ansl = 1 + asp.astype(np.int64)
            afirst = np.cumsum(ansl) - ansl
            n_slots = int(ansl.sum())
            if self.distant_ref and all_cull_len is None:
                raise ValueError("-D over several shards: pass1_cull needs the cull_len() of all ranks")
            adrop = api.cull_flags(np.asarray(all_seq_len if all_cull_len is None else all_cull_len, np.int32), np.asarray(all_score, np.int32), None, 0, 1, fit[0], fit[1])
            slot_dropped = np.zeros(n_slots + 1, np.uint8)
            slot_dropped[afirst[adrop > 0]] = 1
            slot_dropped[afirst[(adrop > 0) & asp] + 1] = 1
            first = afirst[lo: lo + len(self.seq_len)]
        ok = self.score > 0                                                          # clean_FSDB (mia.c:400-406)
        keep_dev = np.zeros(self._n_all, np.uint8)
        keep_dev[idx[ok]] = 1
        rev = np.zeros(self._n_all, np.uint8)
        rev[idx] = (self.rc == 1) & self.strand_known                               # stored orientation (fsdb.c:209-227)
        g.compact_reads(keep_dev, rev)
        self.fsdb_idx = idx[ok]                                                      # input index of every FSDB read
        front, back = first[ok].astype(np.int32), np.where(self.split, first + 1, -1)[ok].astype(np.int32)
        for name in ("seq_len", "score", "rc", "as_", "ae", "split", "strand_known"):
            setattr(self, name, getattr(self, name)[ok])
        self.dropped = np.ascontiguousarray(dropped[ok], np.uint8)
        g.set_alignment_inputs(self.rc, self.as_, self.ae)
        if self.fs:
            g.set_fsdb(self.seq_len, self.score, None, self.strand_known.astype(np.uint8), front, back, n_slots, slot_dropped[:n_slots],
                       self.distant_ref)
        else:
            g.set_cut_inputs(self.seq_len, None, self.dropped)
        self.iter, self.cons, self.last = 0, None, self.ref0.upper()

    def begin_round(self):
        if self.cons is not None:
            self.last = self.cons
        self.iter += 1
        self.g.set_reference(self.last, self.circular, with_rc=0)
        if self.distant_ref and self.x is not None:                                  # mia_main.c:120-174 over shards: the matrix state crosses their boundaries (H6)
            after = self._gather(np.array(self.retry_begin(), np.int32)).reshape(-1, 2)
            self.retry_end(after, self.x.rank)
        elif self.distant_ref and not self._manual_retry:
            self.retried = self.g.distant_retry()                                    # mia_main.c:120-174 (iteration 2 on)

    def retry_begin(self):
        """-D over shards, step 1: the local attempts -> [state after this shard if entered with 0, ... with 1]"""
        self._tried, after = self.g.distant_retry_begin()
        return after

    def retry_end(self, all_after, rank):
        """step 2: all_after = the retry_begin() results of all shards in rank order; enters the local chain with what the shards
        before this one leave, and keeps what the last shard leaves for the next round"""
        s = self.matrix_state
        for r in range(rank):
            s = int(all_after[r][s])
        self.retried = (self._tried, self.g.distant_retry_end(s))
        for r in range(rank, len(all_after)):
            s = int(all_after[r][s])
        self.matrix_state = s

    def iterate(self, want_gaps=False):
        g = self.g
        self.begin_round()
        if self.x is None:
            res = g.iterate_resident(self.cons_code, dropped=self.dropped, want_gaps=want_gaps)
        else:
            res = self.x.rounds.resident(self.cons_code, dropped=self.dropped, want_gaps=want_gaps)
        return self.end_round(*res)

    def end_round(self, cons, fit, gaps):
        self.fit, self.gaps = fit, gaps
        self.score, self.as_, self.ae = self.g.adopt_alignment()
        if self.fs and not self.strand_known.all():
            st = self.g.get_fsdb()
            self.strand_known, self.rc = st["strand_known"].astype(bool), st["rc"]
        L = len(self.last)
        split = (self.as_ > np.where(self.ae > L, self.ae - L, self.ae)) & self.strand_known
        if not self.fs:
            self.split_changes += int((split != self.split).sum())
        self.split = split
        self.cons = cons
        return cons, cons == self.last

    def misincorporation(self):
        """Damage profile of the last round: int64[31, 6, 6] (api.MiaGpu.misincorporation); with an `exchange`, the sum over the
        ranks -- the table of the whole round, the same as one GPU's."""
        t = self.g.misincorporation()
        if self.x is None:
            return t
        return self._gather(t.ravel()).reshape((-1,) + api.MISINC_SHAPE).sum(0)

    def write_maln(self, path, batch, ref_id, ref_desc=""):
        """write_ma of this round's culled_maln (mia_main.c:905 / 958) from the device's results: `batch` is the FastxReader batch
        (or any dict with bases / offsets / ids / id_off / descs / desc_off) the reads came from, in input order; call after
        iterate(want_gaps=True).  Reference id / desc follow mia_main.c:47, 62-65."""
        from .synth import revcomp_bytes
        g = self.g
        al = g.get_alignment()
        if (al["status"] != 0).any():
            raise api.MiaGpuError(f"status bits set on {(al['status'] != 0).sum()} reads: not written as if they were fine")
        tot, _, _ = g.get_runs_packed()
        run_off, packed = np.zeros(len(self.rc) + 1, np.int64), np.zeros(max(tot, 1), np.uint16)
        g.get_runs_packed(run_off, packed)
        off, bases = np.asarray(batch["offsets"]), np.asarray(batch["bases"])
        stored, ids, descs = [], [], []
        idb, ido = batch["ids"], batch["id_off"]
        dsb, dso = batch.get("descs"), batch.get("desc_off")
        for j, i in enumerate(self.fsdb_idx):                                        # stored orientation: fsdb.c:209-227
            r = bases[off[i]:off[i + 1]]
            stored.append(revcomp_bytes(r) if self.rc[j] else r)
            ids.append(idb[ido[i]:ido[i + 1]])
            descs.append(dsb[dso[i]:dso[i + 1]] if dsb is not None else b"\0")
        so = np.zeros(len(stored) + 1, np.int64)
        np.cumsum([len(x) for x in stored], out=so[1:])
        cum = lambda xs: np.concatenate([[0], np.cumsum([len(x) for x in xs])]).astype(np.int64)
        fpsm, rpsm = g.get_pssm()
        if self.iter > 1:
            ref_id, ref_desc = f"ConsAssem.{self.iter}", "iteration assembly"
        rd = dict(bases=np.concatenate(stored) if stored else np.zeros(0, np.uint8), offsets=so, ids=b"".join(ids), id_off=cum(ids),
                  descs=b"".join(descs), desc_off=cum(descs), rc=self.rc, score=al["score"], as_=al["as_out"], ae=al["ae_out"], abr=al["abr"],
                  run_off=run_off, packed=packed, dropped_front=self.dropped, dropped_back=self.dropped)
        return api.write_maln(path, ref_id, ref_desc, self.last, self.circular, self.maln_size, self.cons_code, self.gaps, fpsm, rpsm, rd)

    def run(self, bases, off, max_iter=MAX_ITER):
        self.pass1(bases, off)
        conv = False
        while not conv and self.iter < max_iter:
            _, conv = self.iterate()
        return self.cons, self.iter, conv


class RepeatFilterAssembler:
    """mia -u / -U on the device: every round re-sorts the FSDB (sort_fsdb, fsdb.c:240-252), marks the first of every group
    of reads with the same strand, start and end as unique_best (set_uniq_in_fsdb, fsdb.c:440-508) and leaves the others
    out of the regression and of the consensus (mia.c:466).  Reads, alignments and the DP stay resident; the filter is
    miagpu_repeat_filter; the host keeps what the reference keeps per FSDB POSITION rather than per read:

      * the FSDB order itself (the next sort's ties are resolved by it);
      * AlnSeq slots are numbered in FSDB order at every merge, and AlnSeq.dropped is sticky per slot (H10): a flag set
        for the read at position k stays with position k when the next sort puts another read there.

    Stale back pointers (a read that was wrap-split in an earlier round, mia_main.c:273-276) are counted in
    `split_changes`, not reproduced (driver.Assembler does that, without the filter)."""

    def __init__(self, gpu, ref, sm, circular=1, k=0, soft_mask=0, cons_code=1, just_outer_coords=1, key="score"):
        self.g, self.sm, self.circular, self.k, self.soft_mask, self.cons_code = gpu, sm, circular, k, soft_mask, cons_code
        self.just_outer_coords, self.ref0 = just_outer_coords, ref
        self.split_changes = 0
        if key not in ("score", "qual"):
            raise ValueError("key is 'score' (-u: sort_fsdb) or 'qual' (-U: sort_fsdb_qscore on FragSeq.qual_sum)")
        self.key = key
        gpu.set_pssm(sm)

    def _filter_and_cull(self, split):
        """sort + unique flags + cull over the current FSDB; returns per-read flags for miagpu_consensus_natural"""
        g, fo = self.g, self.order
        key4 = self.score if self.key == "score" else self.qual                     # -u: FragSeq.score, -U: FragSeq.qual_sum
        order, uniq = g.repeat_filter(self.rc[fo], self.as_[fo], self.ae[fo], key4[fo], None, self.just_outer_coords, 0)
        # slots were numbered in the FSDB order the merges ran in (BEFORE this sort)
        nsl = 1 + split.astype(np.int64)
        first = np.zeros(len(nsl), np.int64)
        first[fo] = np.cumsum(nsl[fo]) - nsl[fo]
        need = int(nsl.sum()) + 2
        if need > len(self.dropped_slot):
            self.dropped_slot = np.concatenate([self.dropped_slot, np.zeros(need - len(self.dropped_slot) + 64, np.uint8)])
        self.unique = np.zeros(len(fo), np.uint8)
        self.unique[fo] = uniq
        self.order = fo[order]                                                       # the sort's effect on fsdb->fss
        fo = self.order
        fit = api.score_cut(self.seq_len[fo], self.score[fo], self.unique[fo])       # sums run in FSDB order (H8)
        below = api.cull_flags(self.seq_len, self.score, None, 0, 1, fit[0], fit[1]).astype(bool) & (self.unique > 0)
        self.dropped_slot[first[below]] = 1
        self.dropped_slot[first[below & split] + 1] = 1
        df = np.where(self.unique > 0, self.dropped_slot[first], 2).astype(np.uint8)
        db = np.where(self.unique > 0, self.dropped_slot[np.minimum(first + 1, len(self.dropped_slot) - 1)], 2).astype(np.uint8)
        self.fit = fit
        return df, db

    def pass1(self, bases, off, qual_sum=None):
        """qual_sum (per input read; FastxReader's `qual_sum`, read_fastq's sum(q - 33)) is the fourth sort key with key='qual'"""
        g = self.g
        g.set_reference(self.ref0, self.circular, with_rc=1)
        g.build_kmers(self.k, self.soft_mask)
        g.upload_reads(bases, off)
        p = g.pass1()
        seq_len = np.diff(off).astype(np.int32)
        keep = (p["hits"] > 0) & (p["score"] >= FIRST_ROUND_SCORE_CUTOFF)            # mia.c:1614
        if (keep & (p["score"] == FIRST_ROUND_SCORE_CUTOFF)).any():
            raise NotImplementedError("reads with score == 2000 keep strand_known = 0 and are never realigned (mia.c:1653)")
        idx = np.flatnonzero(keep)
        self.ids = idx.copy()                                                        # input index of every FSDB read
        if self.key == "qual":
            if qual_sum is None:
                raise ValueError("key='qual' (-U) needs qual_sum per input read")
            self.qual = np.ascontiguousarray(np.asarray(qual_sum)[idx], np.int32)
        else:
            self.qual = np.zeros(len(idx), np.int32)
        self.seq_len, self.score = seq_len[idx], p["score"][idx].copy()
        self.rc, self.as_, self.ae = p["rc"][idx].copy(), p["as_"][idx].copy(), p["ae"][idx].copy()
        split = p["start"][idx] > p["end"][idx]                                      # mia.c:1619
        self.maln_size = int(len(idx) + split.sum())                                 # culled_maln->size (mia.c:54)
        self.order = np.arange(len(idx))
        self.dropped_slot = np.zeros(2 * len(idx) + 64, np.uint8)
        self._filter_and_cull(split)                                                 # mia_main.c:827-848: only the flags survive
        ok = self.score > 0                                                          # clean_FSDB (mia.c:400-406)
        keep_dev = np.zeros(len(seq_len), np.uint8)
        keep_dev[idx[ok]] = 1
        rev = np.zeros(len(seq_len), np.uint8)
        rev[idx] = self.rc == 1
        g.compact_reads(keep_dev, rev)
        newpos = np.cumsum(ok) - 1
        self.order = newpos[self.order[ok[self.order]]]
        for name in ("seq_len", "score", "rc", "as_", "ae", "ids", "qual"):
            setattr(self, name, getattr(self, name)[ok])
        self.split = split[ok]
        g.set_alignment_inputs(self.rc, self.as_, self.ae)
        self.iter, self.cons, self.last = 0, None, self.ref0.upper()
        return p

    def iterate(self):
        g = self.g
        if self.cons is not None:
            self.last = self.cons
        self.iter += 1
        g.set_reference(self.last, self.circular, with_rc=0)
        g.realign_resident()
        self.score, self.as_, self.ae = g.adopt_alignment()
        L = len(self.last)
        split = self.as_ > np.where(self.ae > L, self.ae - L, self.ae)
        self.split_changes += int((split != self.split).sum())
        self.split = split
        df, db = self._filter_and_cull(split)
        self.df, self.db = df, db
        cons, self.gaps, _ = g.consensus_natural(df, db, self.cons_code)
        self.cons = cons
        return cons, cons == self.last

    def write_maln(self, path, batch, ref_id, ref_desc=""):
        """write_ma of this round's culled_maln (mia_main.c:905 / 958) under -u / -U: the reads in the FSDB order this round's
        sort left, the non-unique ones left out (mia.c:466), AlnSeq.dropped from the slot-indexed sticky flags."""
        from .synth import revcomp_bytes
        g, fo = self.g, self.order
        al = g.get_alignment()
        if (al["status"] != 0).any():
            raise api.MiaGpuError(f"status bits set on {(al['status'] != 0).sum()} reads: not written as if they were fine")
        tot, _, _ = g.get_runs_packed()
        run_off, packed = np.zeros(len(self.rc) + 1, np.int64), np.zeros(max(tot, 1), np.uint16)
        g.get_runs_packed(run_off, packed)
        nr = np.diff(run_off)[fo]
        new_off = np.concatenate([[0], np.cumsum(nr)]).astype(np.int64)
        src = np.repeat(run_off[:-1][fo] - new_off[:-1], nr) + np.arange(int(new_off[-1]))
        off, bases = np.asarray(batch["offsets"]), np.asarray(batch["bases"])
        idb, ido, dsb, dso = batch["ids"], batch["id_off"], batch.get("descs"), batch.get("desc_off")
        stored, ids, descs = [], [], []
        for j in fo:                                                                 # stored orientation: fsdb.c:209-227
            i = self.ids[j]
            r = bases[off[i]:off[i + 1]]
            stored.append(revcomp_bytes(r) if self.rc[j] else r)
            ids.append(idb[ido[i]:ido[i + 1]])
            descs.append(dsb[dso[i]:dso[i + 1]] if dsb is not None else b"\0")
        cum = lambda xs: np.concatenate([[0], np.cumsum([len(x) for x in xs])]).astype(np.int64)
        fpsm, rpsm = g.get_pssm()
        if self.iter > 1:
            ref_id, ref_desc = f"ConsAssem.{self.iter}", "iteration assembly"
        rd = dict(bases=np.concatenate(stored) if stored else np.zeros(0, np.uint8), offsets=cum(stored), ids=b"".join(ids), id_off=cum(ids),
                  descs=b"".join(descs), desc_off=cum(descs), rc=self.rc[fo], score=al["score"][fo], as_=al["as_out"][fo], ae=al["ae_out"][fo],
                  abr=al["abr"][fo], run_off=new_off, packed=packed[src] if len(src) else packed[:0], unique_best=self.unique[fo],
                  dropped_front=(self.df[fo] == 1), dropped_back=(self.db[fo] == 1))
        return api.write_maln(path, ref_id, ref_desc, self.last, self.circular, self.maln_size, self.cons_code, self.gaps, fpsm, rpsm, rd)
