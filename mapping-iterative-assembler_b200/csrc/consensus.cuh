// consensus.cuh -- per-column accumulation and base calling (sm_100a).
//
// Replaces consensus_assembly_string (mia.c:515-603) and what feeds it:
// merge_pwaln_into_maln's seq/ins/gaps (map_align.c:866-954), pop_smp_from_FSDB
// (fsdb.c:542-619), cull_maln_from_fsdb's gaps rescan (mia.c:486-504), add_base
// (map_align.c:229-263), find_ins_cons (444-510) and find_consensus (294-391).
//
// The reference scans ALL AlnSeqs for EVERY reference position: O(ref_len x N).
// Here one warp walks one AlnSeq entry (O(sum read_len) total): lanes take
// consecutive reference columns, locate them in the run list, derive the base,
// the PSSM depth code (smp) and the four column scores, and add into plane-major
// int32 accumulators with coalesced RED.ADDs (lane i -> address base+i).
// Integer sums commute, so the result is bit-identical for any schedule and any
// number of GPUs (the planes are all-reduced between accumulate and call).
#pragma once
#include "common.cuh"

namespace miagpu {

constexpr int NPLANE = MIAGPU_COUNTS_PER_COL;   // As,Cs,Gs,Ts,gaps,cov,sA,sC,sG,sT
constexpr int PL_GAPS = 4, PL_COV = 5, PL_SCORE = 6;

struct ConsParams {
  const miagpu_entry* entries;
  int64_t n_entries;
  const uint8_t* bases;
  const int64_t* off;
  const uint8_t* rc;
  const int32_t* abr;
  const int32_t* n_runs;
  const uint16_t* runs;
  const int32_t* sm;          // [2][775] forward then strand-reversed, reference layout sm[d][ref][read]
  int32_t seq_len;
  int32_t* gaps;              // [seq_len]
  const int32_t* ins_off;     // [seq_len+1] exclusive scan of gaps (gaps[0] forced to 0)
  int32_t* acc;               // [NPLANE][n_cols], n_cols = seq_len + ins_off[seq_len]
  int64_t n_cols;
  // entry.read >= n_reads names a FROZEN alignment (slots.cuh): the content an earlier round left in a slot that is no longer
  // live but still pointed at -- own bases (FZ_BASES bytes each), M / D runs only, first row 0
  int64_t n_reads;
  const uint8_t* fz_bases;
  const uint16_t* fz_runs;
  const int32_t* fz_nruns;
  const uint8_t* fz_rc;
};
constexpr int FZ_BASES_STRIDE = MAX_READ;
__device__ __forceinline__ int cons_nruns(const ConsParams& p, int rd) { return rd >= p.n_reads ? p.fz_nruns[rd - p.n_reads] : p.n_runs[rd]; }

// an entry as two 16-byte loads (the struct's own alignment is 4: the compiler would load it word by word); entry arrays are
// cudaMalloc'ed and 32 bytes per element
__device__ __forceinline__ miagpu_entry load_entry(const miagpu_entry* p) {
  static_assert(sizeof(miagpu_entry) == 32, "miagpu_entry is eight 32-bit words");
  const uint4 a = *reinterpret_cast<const uint4*>(p), b = *(reinterpret_cast<const uint4*>(p) + 1);
  miagpu_entry e;
  e.read = (int32_t)a.x; e.col_begin = (int32_t)a.y; e.col_count = (int32_t)a.z; e.ref_pos = (int32_t)a.w;
  e.front_len = (int32_t)b.x; e.total_len = (int32_t)b.y; e.act_bias = (int32_t)b.z;
  e.dropped = (uint8_t)(b.w & 0xffu); e.back_formula = (uint8_t)((b.w >> 8) & 0xffu); e.reserved[0] = e.reserved[1] = 0;
  return e;
}

__device__ __forceinline__ int smp_depth(const miagpu_entry& e, int act) {   // fsdb.c:569-580 / 598-609
  const int dfront = e.back_formula ? e.front_len + act : act;
  const int dback = e.total_len - act - 1;
  return dfront <= PSSM_DEPTH ? dfront : (dback < PSSM_DEPTH ? 2 * PSSM_DEPTH - dback : PSSM_DEPTH);
}

// add_base (map_align.c:229-263) into column `col` of the plane-major accumulators.
// GlobalAdder: RED.ADD straight into the global planes (coalesced: lane i -> address base+i).
struct GlobalAdder {
  int32_t* acc;
  int64_t n_cols;
  __device__ __forceinline__ void add(int plane, int64_t col, int v) const { atomicAdd(acc + plane * n_cols + col, v); }
};
// NegGlobalAdder: takes a contribution back out of the global planes (one-call rounds accumulate every read while the host
// still stitches the score cut's chains, then remove the base columns of the reads this round's cut dropped)
struct NegGlobalAdder {
  int32_t* acc;
  int64_t n_cols;
  __device__ __forceinline__ void add(int plane, int64_t col, int v) const { atomicAdd(acc + plane * n_cols + col, -v); }
};
// TileAdder: a block owns the padded columns [c0, c0 + TILE_COLS) in shared memory; whatever an entry
// adds outside that window (its tail past the tile, at most a read length) goes to the global planes.
constexpr int TILE_POS = 1792;                  // reference positions per tile
constexpr int TILE_COLS = 2304;                 // padded columns a tile holds in shared memory (positions + overhang + inserts)
struct TileAdder {
  int32_t* s_acc;                               // [NPLANE][TILE_COLS]
  int64_t c0;
  int32_t* acc;
  int64_t n_cols;
  __device__ __forceinline__ void add(int plane, int64_t col, int v) const {
    const int64_t d = col - c0;
    if ((uint64_t)d < (uint64_t)TILE_COLS) atomicAdd(s_acc + plane * TILE_COLS + (int)d, v);
    else atomicAdd(acc + plane * n_cols + col, v);
  }
};
// LocalAdder: every column of the entry lies inside the tile's shared window: plain 32-bit indices, no range test
struct LocalAdder {
  int32_t* s_acc;
  __device__ __forceinline__ void add(int plane, int col, int v) const { atomicAdd(s_acc + plane * TILE_COLS + col, v); }
};
template <typename Adder, typename Col>
__device__ __forceinline__ void add_base_dev(const Adder& A, Col col, int ch_code /*0..4, 5 = '-'*/, const int32_t* sm_strand, int depth) {
  A.add(PL_COV, col, 1);
  if (ch_code == 5) { A.add(PL_GAPS, col, 1); return; }
  if (ch_code < 4) A.add(ch_code, col, 1);
  const int32_t* m = sm_strand + depth * 25 + ch_code;          // sm[depth][X][b]
#pragma unroll
  for (int x = 0; x < 4; x++) A.add(PL_SCORE + x, col, m[x * 5]);
}

// Misincorporation table (miagpu_misincorporation): counts[depth][ref][read] over A C G T N -, in the orientation of the molecule
// (a reverse-strand entry is complemented and mirrored, depth -> 30 - depth, so every cell is the cell of the FORWARD matrix that
// scored the base).  The bins are skewed: with 35-75 bp reads about half of all columns are matches at depth 15, where the 32
// lanes of a warp would hit four shared addresses.  Those four cells are lane-private register counters, summed over the warp
// once per block; everything else (the depths of the read ends, where consecutive lanes have consecutive depths, mismatches,
// deletions, inserted bases) is a shared-memory atomic into the block's table.
constexpr int MISINC_CODES = 6;                 // A C G T N -
struct MisincAdder {
  uint32_t* s_tab;                              // [31][6][6] of this block
  const uint8_t* ref;                           // reference codes 0..4
  mutable uint32_t hot0 = 0, hot1 = 0, hot2 = 0, hot3 = 0;   // depth-15 matches of this lane, by forward base
  __device__ __forceinline__ static int comp(int b) { return b < 4 ? 3 - b : b; }
  // an aligned column: reference position pos, read code qc (5 = the read has a deletion)
  __device__ __forceinline__ void base(int depth, int pos, int qc, bool rev) const {
    int r = ref[pos];
    if (rev) { r = comp(r); qc = comp(qc); depth = 2 * PSSM_DEPTH - depth; }
    if (depth == PSSM_DEPTH && r == qc && r < 4) {
      hot0 += r == 0; hot1 += r == 1; hot2 += r == 2; hot3 += r == 3;
    } else {
      atomicAdd(s_tab + (depth * MISINC_CODES + r) * MISINC_CODES + qc, 1u);
    }
  }
  // an inserted base in front of a column of depth `depth`: reference '-'
  __device__ __forceinline__ void ins(int depth, int qc, bool rev) const {
    if (rev) { qc = comp(qc); depth = 2 * PSSM_DEPTH - depth; }
    atomicAdd(s_tab + (depth * MISINC_CODES + 5) * MISINC_CODES + qc, 1u);
  }
};

// One entry, walked by a whole warp (lanes take consecutive reference columns).
// MODE 0: ref->gaps = max insert length per position over the culled list (mia.c:486-504;
//         positions with start < pos <= end only, so an insert in front of an entry's first
//         column never counts)
// MODE 1: base columns + insert columns
// MODE 2: base columns only (what AlnSeq.dropped decides, mia.c:571-579; insert columns count dropped reads too)
// MODE 3: the misincorporation table (MisincAdder): every column below seq_len and every inserted base in front of one, of the
//         entries that are not dropped -- what the AlnSeq's SEQ / INS_POS / SMP in the `.maln` file list
// Where the columns of a reference position lie.  GlobalLay: the padded layout of the whole alignment, straight from ins_off / gaps.
// TileLay: the same for an entry that lies wholly inside a tile's shared window -- columns relative to the window, insert offsets
// and lengths from the tile's copy of ins_off (gaps[pos] = ins_off[pos + 1] - ins_off[pos] for pos > 0, the only positions asked).
struct GlobalLay {
  const int32_t* ins_off;
  const int32_t* gaps;
  __device__ __forceinline__ int64_t col(int pos) const { return (int64_t)pos + ins_off[pos + 1]; }    // the base column sits after its insert columns
  __device__ __forceinline__ int64_t icol(int pos) const { return (int64_t)pos + ins_off[pos]; }
  __device__ __forceinline__ int gap(int pos) const { return gaps[pos]; }
};
struct TileLay {
  const int32_t* s_ins;     // ins_off[t0 + i]
  int t0, ins0;
  __device__ __forceinline__ int col(int pos) const { return pos - t0 + s_ins[pos - t0 + 1] - ins0; }
  __device__ __forceinline__ int icol(int pos) const { return pos - t0 + s_ins[pos - t0] - ins0; }
  __device__ __forceinline__ int gap(int pos) const { return s_ins[pos - t0 + 1] - s_ins[pos - t0]; }
};

template <int MODE, typename Adder, typename Lay>
__device__ __forceinline__ void walk_entry(const ConsParams& p, const miagpu_entry& e, int lane, const Adder& A, const Lay& Y, const int32_t* sm) {
  if (e.col_count <= 0 || (MODE == 3 && e.dropped)) return;
  const int rd = e.read;
  const bool fz = rd >= p.n_reads;
  const int64_t q = rd - p.n_reads;
  const int nr = fz ? p.fz_nruns[q] : p.n_runs[rd];
  if (nr <= 0) return;
  const uint16_t* runs = fz ? p.fz_runs + q * MAX_RUNS : p.runs + (int64_t)rd * MAX_RUNS;
  const uint8_t* read = fz ? p.fz_bases + q * FZ_BASES_STRIDE : p.bases + p.off[rd];
  const bool rev = fz ? p.fz_rc[q] : p.rc[rd];
  const int32_t* sm_strand = sm + (rev ? MIAGPU_PSSM_INTS : 0);
  const int cb = e.col_begin, ce = e.col_begin + e.col_count;

  int colpos = 0;                 // reference columns before this run
  int rpos = fz ? 0 : p.abr[rd];  // read rows consumed before this run (absolute row)
  const int row0 = rpos;
  int pend = 0;                   // inserted bases waiting for the next column
  for (int k = 0; k < nr; k++) {
    const int x = runs[k];
    const int type = x >> 14, len = x & 0x3fff;
    if (type == MIAGPU_RUN_I) { pend = len; rpos += len; continue; }
    const int lo = max(colpos, cb), hi = min(colpos + len, ce);
    for (int i = lo + lane; i < hi; i += 32) {
      const int pos = e.ref_pos + (i - cb);
      if (pos >= p.seq_len) continue;                       // consensus loop stops at seq_len (mia.c:555)
      const bool isM = type == MIAGPU_RUN_M;
      const int row = rpos + (i - colpos);                  // read row of an M column
      const int q = (i == colpos) ? pend : 0;               // insert length in front of this column
      if (MODE == 0) {
        if (q > 0 && i > cb && pos > 0) atomicMax(p.gaps + pos, q);
      } else if constexpr (MODE == 3) {
        const int depth = smp_depth(e, e.act_bias + (isM ? row - row0 : rpos - row0));
        A.base(depth, pos, isM ? base_code(read[row]) : 5, rev);
        for (int j = 0; j < q; j++) A.ins(depth, base_code(read[row - q + j]), rev);   // INS_POS: every insert, first column too
      } else {
        // act = read bases consumed before the column, inserted ones included (fsdb.c:564-583)
        const int act = e.act_bias + (isM ? row - row0 : rpos - row0);
        const int depth = smp_depth(e, act);
        if (!e.dropped) {
          const int ch = isM ? base_code(read[row]) : 5;
          add_base_dev(A, Y.col(pos), ch, sm_strand, depth);
        }
        if (MODE == 2) continue;
        const int g = (i > cb && pos > 0) ? Y.gap(pos) : 0;  // find_ins_cons: start < pos <= end, dropped NOT checked
        for (int j = 0; j < g; j++) {
          const int ch = j < q ? base_code(read[row - q + j]) : 5;
          add_base_dev(A, Y.icol(pos) + j, ch, sm_strand, depth);
        }
      }
    }
    colpos += len;
    if (type == MIAGPU_RUN_M) rpos += len;
    pend = 0;
  }
}

template <int MODE, typename Adder>
__device__ __forceinline__ void walk_entry(const ConsParams& p, const miagpu_entry& e, int lane, const Adder& A) {
  walk_entry<MODE>(p, e, lane, A, GlobalLay{p.ins_off, p.gaps}, p.sm);
}

// MODE 0 / 1 over the whole entry list, accumulators in global memory: one warp per entry.
template <int MODE>
__global__ void __launch_bounds__(256) entry_kernel(ConsParams p) {
  const int lane = threadIdx.x & 31;
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= p.n_entries) return;
  const miagpu_entry e = load_entry(p.entries + w);
  walk_entry<MODE>(p, e, lane, GlobalAdder{p.acc, p.n_cols});
}

// MODE 0 with a cheap filter in front: a lane looks at one entry, only entries whose alignment has more
// than one run (an insert needs at least M I M) are walked by the warp.
__global__ void __launch_bounds__(256) gaps_kernel(ConsParams p) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32;
  const int64_t idx = w0 + lane;
  bool want = false;
  if (idx < p.n_entries) {
    const int32_t rd = p.entries[idx].read;
    want = p.entries[idx].col_count > 0 && rd < p.n_reads && p.n_runs[rd] > 2;      // a frozen alignment has no inserts
  }
  unsigned m = __ballot_sync(0xffffffffu, want);
  while (m) {
    const int b = __ffs(m) - 1;
    m &= m - 1;
    const miagpu_entry e = load_entry(p.entries + w0 + b);
    walk_entry<0>(p, e, lane, GlobalAdder{p.acc, p.n_cols});
  }
}

// MODE 1 with the accumulators of one reference tile private to the block (shared-memory atomics), flushed
// once at the end.  grid = (slices, tiles): block (s, t) scans slice s of ent_pos[] (start position of every
// entry, -1 = empty) and walks the entries that start inside tile t.  Used when the reference is short enough
// for every tile to be scanned by many blocks (high coverage per column = the case where global atomics
// contend); integer sums, so the result does not depend on the path taken.
// Shared memory: [NPLANE][TILE_COLS] accumulators, ins_off[t0 .. t0+TILE_COLS], both PSSMs.
// A lane first loads the metadata of "its" entry (32 independent loads in flight), then the warp walks the
// flagged entries one by one; the common alignment -- a single M run -- takes a loop that touches global
// memory only for the read bases.
constexpr int TILE_THREADS = 512;
constexpr int TILE_SMEM_INTS = NPLANE * TILE_COLS + (TILE_COLS + 1) + 2 * MIAGPU_PSSM_INTS + 64 + 32;   // + base-code table (256 bytes) + a sink word per lane
// What tile_kernel needs of a binned entry, 32 bytes, written in bin order by ent_bin_scatter_kernel so that a warp reads 32 of them
// in one contiguous kilobyte: no per-read look-ups (n_runs, runs, abr, rc, off) while the tile is walked.
//   a = { byte offset of read row `abr` in p.bases (lo, hi), ref_pos, col_begin | hi_col << 16 }
//   b = { front_len | total_len << 16 (signed halves), act_bias (signed low half) | flags << 16, entry index, 0 }
// flags: 1 dropped, 2 back_formula, 4 reverse strand, 8 FAST = the alignment is one M run (everything above is valid); without
// FAST only the entry index counts and the warp takes the general walk.  hi_col = min(run length, col_begin + col_count).
struct TileRec { uint4 a, b; };
constexpr uint32_t TR_DROPPED = 1, TR_BACKF = 2, TR_STRAND = 4, TR_FAST = 8;

__global__ void __launch_bounds__(TILE_THREADS) tile_kernel(ConsParams p, const TileRec* __restrict__ recs, const int32_t* __restrict__ bin_start) {
  extern __shared__ int32_t s_acc[];                       // [NPLANE][TILE_COLS]
  int32_t* s_ins = s_acc + NPLANE * TILE_COLS;             // ins_off[t0 + i], i <= TILE_COLS
  int32_t* s_sm = s_ins + TILE_COLS + 1;
  uint8_t* s_code = reinterpret_cast<uint8_t*>(s_sm + 2 * MIAGPU_PSSM_INTS);   // base_code() of every byte value: one LDS instead of four compares
  int32_t* s_sink = s_sm + 2 * MIAGPU_PSSM_INTS + 64;                          // where the count of an N goes (no base plane of its own)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int t0 = blockIdx.y * TILE_POS;
  const int64_t c0 = (int64_t)t0 + p.ins_off[t0];
  for (int i = threadIdx.x; i < NPLANE * TILE_COLS; i += blockDim.x) s_acc[i] = 0;
  for (int i = threadIdx.x; i <= TILE_COLS; i += blockDim.x) s_ins[i] = p.ins_off[min(t0 + i, p.seq_len)];
  for (int i = threadIdx.x; i < 2 * MIAGPU_PSSM_INTS; i += blockDim.x) s_sm[i] = p.sm[i];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_code[i] = (uint8_t)base_code((uint8_t)i);
  __syncthreads();
  const TileAdder A{s_acc, c0, p.acc, p.n_cols};
  // the entries that start inside this tile were binned (ent_bin_*_kernel): slice blockIdx.x of the tile's records
  const int64_t b0 = bin_start[blockIdx.y], b1 = bin_start[blockIdx.y + 1];
  const int64_t per = (b1 - b0 + gridDim.x - 1) / gridDim.x;
  const int64_t lo = b0 + per * blockIdx.x, hi = min(lo + per, b1);
  const int ins0 = s_ins[0];
  for (int64_t base = lo + warp * 32; base < hi; base += nwarps * 32) {
    const int64_t at = base + lane;
    const bool mine = at < hi;
    TileRec r{};
    if (mine) { r.a = __ldg(&recs[at].a); r.b = __ldg(&recs[at].b); }
    if (mine && ((r.b.y >> 16) & TR_FAST)) {               // the 32 entries' bases on their way into L2 while the warp walks them one by one
      const uint8_t* q = p.bases + (((int64_t)r.a.y << 32) | r.a.x);
      asm volatile("prefetch.global.L2 [%0];" ::"l"(q + (r.a.w & 0xffffu)));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(q + (r.a.w >> 16) - 1));
    }
    unsigned m = __ballot_sync(0xffffffffu, mine);
    while (m) {
      const int b = __ffs(m) - 1;
      m &= m - 1;
      const uint32_t bf = __shfl_sync(0xffffffffu, r.b.y, b);
      const uint32_t flags = bf >> 16;
      const int rp = (int)__shfl_sync(0xffffffffu, r.a.z, b);
      const uint32_t ch = __shfl_sync(0xffffffffu, r.a.w, b);
      if (flags & TR_DROPPED) {
        // a dropped entry only counts in insert columns (mia.c:571-579): none between its first and last position => nothing to add
        const int df = rp - t0, dl = min(rp + (int)(ch >> 16) - (int)(ch & 0xffffu) - 1, p.seq_len - 1) - t0;
        if (dl < TILE_COLS && dl >= df && s_ins[dl + 1] == s_ins[df]) continue;
      }
      if (!(flags & TR_FAST)) {                            // gaps in the alignment, or a frozen one: the general walk
        const miagpu_entry eb = load_entry(p.entries + __shfl_sync(0xffffffffu, r.b.z, b));
        // wholly inside the shared window (its last position and that position's columns): layout, scores and sums from shared memory
        const int dl = min(eb.ref_pos + eb.col_count - 1, p.seq_len - 1) - t0;
        if (dl >= 0 && dl < TILE_COLS && dl + (s_ins[min(dl + 1, TILE_COLS)] - ins0) < TILE_COLS)
          walk_entry<1>(p, eb, lane, LocalAdder{s_acc}, TileLay{s_ins, t0, ins0}, s_sm);
        else
          walk_entry<1>(p, eb, lane, A);
        continue;
      }
      const uint32_t alo = __shfl_sync(0xffffffffu, r.a.x, b), ahi = __shfl_sync(0xffffffffu, r.a.y, b);
      const uint32_t ft = __shfl_sync(0xffffffffu, r.b.x, b);
      const int cb = (int)(ch & 0xffffu), hi_col = (int)(ch >> 16);
      const int fl = (int)(int16_t)(ft & 0xffffu), tl = (int)(int16_t)(ft >> 16), bias = (int)(int16_t)(bf & 0xffffu);
      const bool dropped = flags & TR_DROPPED, backf = flags & TR_BACKF;
      const int32_t* sms = s_sm + ((flags & TR_STRAND) ? MIAGPU_PSSM_INTS : 0);
      const uint8_t* read = p.bases + (((int64_t)ahi << 32) | alo);
      // the entry's last column inside the shared window => all of them are (positions and insert offsets grow together)
      const int d_last = min(rp + (hi_col - 1 - cb), p.seq_len - 1) - t0;
      const bool inside = hi_col > cb && d_last >= 0 && d_last < TILE_COLS && d_last + (s_ins[min(d_last + 1, TILE_COLS)] - ins0) < TILE_COLS;
      if (inside) {
        const LocalAdder LA{s_acc};
        for (int i = cb + lane; i < hi_col; i += 32) {
          const int pos = rp + (i - cb);
          if (pos >= p.seq_len) continue;
          const int act = bias + i;
          const int dfront = backf ? fl + act : act, dback = tl - act - 1;
          const int depth = dfront <= PSSM_DEPTH ? dfront : (dback < PSSM_DEPTH ? 2 * PSSM_DEPTH - dback : PSSM_DEPTH);
          const int d = pos - t0;
          const int io0 = s_ins[d] - ins0, io1 = s_ins[d + 1] - ins0;
          if (!dropped) {                                    // add_base_dev for a base (never '-'), without its branches
            const int ch = s_code[read[i]], col = d + io1;
            int32_t* cell = s_acc + col;
            atomicAdd(cell + PL_COV * TILE_COLS, 1);
            atomicAdd(ch < 4 ? cell + ch * TILE_COLS : s_sink + lane, 1);
            const int32_t* m = sms + depth * 25 + ch;        // sm[depth][X][b]
#pragma unroll
            for (int x = 0; x < 4; x++) atomicAdd(cell + (PL_SCORE + x) * TILE_COLS, m[x * 5]);
          }
          if (i > cb && pos > 0)                             // find_ins_cons: start < pos <= end, dropped NOT checked
            for (int j = io0; j < io1; j++) add_base_dev(LA, d + j, 5, sms, depth);
        }
        continue;
      }
      for (int i = cb + lane; i < hi_col; i += 32) {
        const int pos = rp + (i - cb);
        if (pos >= p.seq_len) continue;
        const int act = bias + i;
        const int dfront = backf ? fl + act : act, dback = tl - act - 1;
        const int depth = dfront <= PSSM_DEPTH ? dfront : (dback < PSSM_DEPTH ? 2 * PSSM_DEPTH - dback : PSSM_DEPTH);
        const int d = pos - t0;
        int io0, io1;
        if (d < TILE_COLS) { io0 = s_ins[d]; io1 = s_ins[d + 1]; }
        else { io0 = p.ins_off[pos]; io1 = p.ins_off[pos + 1]; }
        if (!dropped) add_base_dev(A, (int64_t)pos + io1, base_code(read[i]), sms, depth);
        if (i > cb && pos > 0)                               // find_ins_cons: start < pos <= end, dropped NOT checked
          for (int j = io0; j < io1; j++) add_base_dev(A, (int64_t)pos + j, 5, sms, depth);
      }
    }
  }
  __syncthreads();
  const int64_t room = min((int64_t)TILE_COLS, p.n_cols - c0);
  for (int i = threadIdx.x; i < NPLANE * TILE_COLS; i += blockDim.x) {
    const int pl = i / TILE_COLS, d = i - pl * TILE_COLS;
    const int v = s_acc[i];
    if (v != 0 && d < room) atomicAdd(p.acc + pl * p.n_cols + c0 + d, v);
  }
}

// The reads this round's cut dropped (newly[i] = below the cut now, not dropped before): their base columns come back out
// of the planes and their entries take the flag.  A lane looks at one read, the warp walks the flagged ones.
__global__ void __launch_bounds__(256) undo_kernel(ConsParams p, int64_t n_reads, const uint8_t* __restrict__ newly, miagpu_entry* entries) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32;
  const int64_t i = w0 + lane;
  unsigned m = __ballot_sync(0xffffffffu, i < n_reads && newly[i]);
  while (m) {
    const int b = __ffs(m) - 1;
    m &= m - 1;
    for (int h = 0; h < 2; h++) {
      const int64_t idx = 2 * (w0 + b) + h;
      const miagpu_entry e = load_entry(entries + idx);
      if (e.dropped) continue;
      walk_entry<2>(p, e, lane, NegGlobalAdder{p.acc, p.n_cols});
      __syncwarp();
      if (lane == 0) entries[idx].dropped = 1;
    }
  }
}

// The misincorporation table of the entry list (MODE 3 of walk_entry), read only: a block takes MISINC_PER_BLOCK consecutive
// entries (at most 2 M columns: the block-private 32-bit cells cannot overflow) and adds its table into the global 64-bit one once.
// A warp takes 32 entries at a time; each lane first touches the per-read words and the bases of its entry, so that 32 of those
// dependent loads are in flight at once before the warp walks the 32 entries one by one (DESIGN 4.12: the walk is latency-bound).
constexpr int MISINC_THREADS = 256;
constexpr int MISINC_PER_BLOCK = 4096;
__global__ void __launch_bounds__(MISINC_THREADS) misinc_kernel(ConsParams p, const uint8_t* __restrict__ ref, unsigned long long* out) {
  __shared__ uint32_t s_tab[MIAGPU_MISINC_INTS];
  for (int i = threadIdx.x; i < MIAGPU_MISINC_INTS; i += blockDim.x) s_tab[i] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const MisincAdder A{s_tab, ref};
  const int64_t b0 = (int64_t)blockIdx.x * MISINC_PER_BLOCK, b1 = min(b0 + MISINC_PER_BLOCK, p.n_entries);
  for (int64_t base = b0 + warp * 32; base < b1; base += nwarps * 32) {
    if (base + lane < b1) {
      const int rd = p.entries[base + lane].read;
      if (rd < p.n_reads) {
        asm volatile("prefetch.global.L1 [%0];" ::"l"(p.n_runs + rd));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(p.abr + rd));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(p.rc + rd));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(p.runs + (int64_t)rd * MAX_RUNS));
        const int64_t o0 = p.off[rd], o1 = p.off[rd + 1];
        if (o1 > o0) {
          asm volatile("prefetch.global.L1 [%0];" ::"l"(p.bases + o0));
          asm volatile("prefetch.global.L1 [%0];" ::"l"(p.bases + o1 - 1));
        }
      }
    }
    const int m = (int)min((int64_t)32, b1 - base);
    for (int k = 0; k < m; k++) walk_entry<3>(p, load_entry(p.entries + base + k), lane, A);
  }
  uint32_t h[4] = {A.hot0, A.hot1, A.hot2, A.hot3};
#pragma unroll
  for (int r = 0; r < 4; r++) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) h[r] += __shfl_xor_sync(0xffffffffu, h[r], s);
    if (lane == 0 && h[r]) atomicAdd(s_tab + (PSSM_DEPTH * MISINC_CODES + r) * MISINC_CODES + r, h[r]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < MIAGPU_MISINC_INTS; i += blockDim.x)
    if (s_tab[i]) atomicAdd(out + i, (unsigned long long)s_tab[i]);
}

// Entries binned by the tile their first column lies in (a counting sort in two kernels; the order inside a bin does not
// matter: integer sums).  ent_bin_count_kernel: tile of every entry (-1 = nothing to add) + entries per tile;
// ent_bin_scan_kernel: bin starts + cursors; ent_bin_scatter_kernel: entry indices into their bins.
constexpr int MAX_TILES = 64;
__global__ void __launch_bounds__(256) ent_bin_count_kernel(ConsParams p, int32_t* ent_tile, int32_t* counts) {
  __shared__ int s_cnt[MAX_TILES];
  if (threadIdx.x < MAX_TILES) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int t = -1;
  if (i < p.n_entries) {
    const uint4 a = *reinterpret_cast<const uint4*>(p.entries + i);        // read, col_begin, col_count, ref_pos
    const int e_read = (int)a.x, e_cols = (int)a.z, e_pos = (int)a.w;
    if (e_cols > 0 && cons_nruns(p, e_read) > 0 && e_pos >= 0 && e_pos < p.seq_len) t = e_pos / TILE_POS;
    ent_tile[i] = t;
  }
  const unsigned peers = __match_any_sync(0xffffffffu, t);
  if (t >= 0 && (peers & ((1u << (threadIdx.x & 31)) - 1)) == 0) atomicAdd(&s_cnt[t], __popc(peers));
  __syncthreads();
  if (threadIdx.x < MAX_TILES && s_cnt[threadIdx.x]) atomicAdd(&counts[threadIdx.x], s_cnt[threadIdx.x]);
}
__global__ void ent_bin_scan_kernel(int n_tiles, const int32_t* counts, int32_t* bin_start, int32_t* cursor) {
  if (threadIdx.x != 0) return;
  int run = 0;
  for (int t = 0; t < n_tiles; t++) { bin_start[t] = run; cursor[t] = run; run += counts[t]; }
  bin_start[n_tiles] = run;
}
__global__ void __launch_bounds__(256) ent_bin_scatter_kernel(ConsParams p, const int32_t* __restrict__ ent_tile, int32_t* cursor, TileRec* recs) {
  __shared__ int s_cnt[MAX_TILES], s_base[MAX_TILES];
  if (threadIdx.x < MAX_TILES) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int t = i < p.n_entries ? ent_tile[i] : -1;
  const int lane = threadIdx.x & 31;
  const unsigned peers = __match_any_sync(0xffffffffu, t);
  int slot = 0;
  TileRec r{};
  if (t >= 0) {
    const int leader = __ffs(peers) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(&s_cnt[t], __popc(peers));
    base = __shfl_sync(peers, base, leader);
    slot = base + __popc(peers & ((1u << lane) - 1));
    // the record (entries come in read order here: the per-read look-ups are next to each other)
    const miagpu_entry e = load_entry(p.entries + i);
    r.b.z = (uint32_t)i;
    r.a.z = (uint32_t)e.ref_pos;                           // every record: where the entry lies and whether it is dropped (tile_kernel skips
    r.a.w = (uint32_t)min(e.col_begin, 0xffff) | ((uint32_t)min(e.col_begin + e.col_count, 0xffff) << 16);   // dropped entries without insert columns)
    r.b.y = (e.dropped ? TR_DROPPED : 0u) << 16;
    if (e.read < p.n_reads && p.n_runs[e.read] == 1) {
      const int run0 = p.runs[(int64_t)e.read * MAX_RUNS];
      const int len = run0 & 0x3fff;
      const bool fits = e.front_len >= -32768 && e.front_len <= 32767 && e.total_len >= -32768 && e.total_len <= 32767 &&
                        e.act_bias >= -32768 && e.act_bias <= 32767 && e.col_begin <= 0xffff;
      if ((run0 >> 14) == MIAGPU_RUN_M && fits) {
        const int64_t addr = p.off[e.read] + p.abr[e.read];
        const int hi_col = min(len, e.col_begin + e.col_count);
        const uint32_t flags = TR_FAST | (e.dropped ? TR_DROPPED : 0u) | (e.back_formula ? TR_BACKF : 0u) | (p.rc[e.read] ? TR_STRAND : 0u);
        r.a = make_uint4((uint32_t)addr, (uint32_t)(addr >> 32), (uint32_t)e.ref_pos, (uint32_t)e.col_begin | ((uint32_t)hi_col << 16));
        r.b.x = ((uint32_t)e.front_len & 0xffffu) | ((uint32_t)e.total_len << 16);
        r.b.y = ((uint32_t)e.act_bias & 0xffffu) | (flags << 16);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < MAX_TILES) s_base[threadIdx.x] = s_cnt[threadIdx.x] ? atomicAdd(&cursor[threadIdx.x], s_cnt[threadIdx.x]) : 0;
  __syncthreads();
  if (t >= 0) { recs[s_base[t] + slot].a = r.a; recs[s_base[t] + slot].b = r.b; }
}

// find_consensus (map_align.c:294-391) for every column of the padded layout.
// out[col] = called character ('-' for a gap consensus, dropped on the host side).
__global__ void call_kernel(const int32_t* acc, int64_t n_cols, int cons_code, char* out) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cols) return;
  const int cov = acc[PL_COV * n_cols + c], gaps = acc[PL_GAPS * n_cols + c];
  char r;
  if (cov == 0) r = 'N';
  else if ((double)gaps / (double)cov >= 0.5) r = '-';
  else {
    const int sA = acc[(PL_SCORE + 0) * n_cols + c], sC = acc[(PL_SCORE + 1) * n_cols + c];
    const int sG = acc[(PL_SCORE + 2) * n_cols + c], sT = acc[(PL_SCORE + 3) * n_cols + c];
    int top = sA, second = INT_MIN;
    char base = 'A';
    if (sC >= top) { second = top; top = sC; base = 'C'; } else second = sC;        // '>=': later base wins ties
    if (sG >= top) { second = top; top = sG; base = 'G'; } else if (sG >= second) second = sG;
    if (sT >= top) { second = top; top = sT; base = 'T'; } else if (sT >= second) second = sT;
    if (cons_code == 2) r = (top >= 0 || (top - 2400) > second) ? base : 'N';       // MIN_SC_DIFF_CONS
    else r = top >= -399 ? base : 'N';                                              // MIN_SCORE_CONS
  }
  out[c] = r;
}

// Device-side construction of the "natural" entry list: read i owns entries 2i (whole
// alignment or front part) and 2i+1 (wrapped back part, col_count = 0 when not split).
// Mirrors mia_main.c:259-276 (end fix, split test), split_pwaln (mia.c:1376-1438) and
// asp_len (fsdb.c:518-530); used when the host has no stale AlnSeq pointers to describe.
// A read that is not unique_best (-u / -U) is not in the culled list at all (mia.c:466): flag value 2 in dropped_front /
// dropped_back, or unique[i] == 0, leaves its entries empty.
__global__ void natural_entries_kernel(int64_t n, const int32_t* as_out, const int32_t* ae_out, const int32_t* n_runs,
                                       const uint16_t* runs, const uint8_t* status, int seq_len, const uint8_t* dropped_front,
                                       const uint8_t* dropped_back, miagpu_entry* out, const uint8_t* unique = nullptr,
                                       const uint8_t* known = nullptr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  miagpu_entry f{}, b{};
  f.read = b.read = (int32_t)i;
  const int nr = n_runs[i];
  // (known: a strand-unknown read merges no AlnSeq of its own, mia_main.c:178)
  const bool absent = (unique && !unique[i]) || (dropped_front && dropped_front[i] == 2) || (known && !known[i]);
  if (nr > 0 && !(status[i] & MIAGPU_ST_UNSUPPORTED) && !absent) {
    const int start = as_out[i];
    int end = ae_out[i];
    if (end > seq_len) end -= seq_len;
    const bool split = start > end;
    const int cf = split ? seq_len - start : 0x7fffffff;     // alignment columns that stay in front
    int cols = 0, ins = 0, fins = 0;
    const uint16_t* r = runs + i * MAX_RUNS;
    for (int k = 0; k < nr; k++) {
      const int x = r[k], t = x >> 14, len = x & 0x3fff;
      if (t == MIAGPU_RUN_I) { ins += len; if (cols < cf) fins += len; }
      else cols += len;
    }
    // a read that starts beyond seq_len (the window rule can leave it in the wrap): split_pwaln moves ALL of it to the back AlnSeq
    // at START 0 (mia.c:1400-1422) and the front AlnSeq has the negative length asp_len computes from end - start + 1
    const int fcols = split ? min(max(cf, 0), cols) : cols;
    const int fl = (split && cf < 0) ? cf : fcols + fins, bl = split ? (cols + ins) - fl : 0;
    f.col_begin = 0; f.col_count = fcols; f.ref_pos = start; f.front_len = fl; f.total_len = fl + bl;
    f.dropped = dropped_front ? (dropped_front[i] != 0) : 0;
    if (split) {
      b = f;
      b.col_begin = fcols; b.col_count = cols - fcols; b.ref_pos = 0; b.back_formula = 1;
      b.dropped = dropped_back ? (dropped_back[i] != 0) : f.dropped;
    }
  }
  // two 16-byte stores per entry (the struct's own alignment is 4: the compiler would store it word by word)
  static_assert(sizeof(miagpu_entry) == 32, "miagpu_entry is eight 32-bit words");
  uint4* q = reinterpret_cast<uint4*>(out + 2 * i);
  q[0] = make_uint4((uint32_t)f.read, (uint32_t)f.col_begin, (uint32_t)f.col_count, (uint32_t)f.ref_pos);
  q[1] = make_uint4((uint32_t)f.front_len, (uint32_t)f.total_len, (uint32_t)f.act_bias, (uint32_t)f.dropped | ((uint32_t)f.back_formula << 8));
  q[2] = make_uint4((uint32_t)b.read, (uint32_t)b.col_begin, (uint32_t)b.col_count, (uint32_t)b.ref_pos);
  q[3] = make_uint4((uint32_t)b.front_len, (uint32_t)b.total_len, (uint32_t)b.act_bias, (uint32_t)b.dropped | ((uint32_t)b.back_formula << 8));
}

// gaps[0] is ignored by the consensus (mia.c:557 "ref_pos > 0"); force it to 0 so the scan
// allocates no columns for it
__global__ void zero_first_kernel(int32_t* gaps) { gaps[0] = 0; }

}  // namespace miagpu
