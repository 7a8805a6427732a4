// sweep16.cuh -- pass 1 WITHOUT the k-mer filter: both whole strands of a read in packed 16-bit SIMD (sm_100a).
//
// sg_align (mia.c:1500-1610) runs dyn_prog over the read against the whole wrapped reference, forward strand and
// reverse-complement strand, both with the forward matrix (H5), and keeps the better strand.  The two matrices have the
// same rows (same read, same substitution profile) and the same width, so they ride in the two halves of one
// register: low half = forward strand, high half = reverse-complement strand -- the lane frame, the 25-entry
// per-row table, the FMA-pipe adds and the folded pure-diagonal verdict are those of pair16.cuh (read 1. - 4.
// there), with K = 16 columns per lane and 16 lanes per read: a warp carries two reads of equal length.
//
// The strands are 16,825 columns (1 Mb + 256 for the nuclear case), not a window: the sweep goes CHUNK by chunk of
// 256 columns, all L rows per chunk, and hands the next chunk, per row, exactly what a lane's left neighbour hands
// over inside a chunk -- the last two cells of the row, the verdict carry of the last cell, and the running
// column-gap maximum (best_gap_col as a value: mia.c:838-850) -- through a per-read ring in shared memory.  In the
// lane frame a hand-over is the constant shift -GEP*K whether the neighbour is a lane or the previous chunk.
//
// Per strand the kernel keeps the first maximum of the last row over all chunks (max_sg_score, mia.c:1278-1302)
// and the verdict at that cell; it writes them as the two "jobs" of the read, and p1_merge_kernel (pass1.cuh)
// picks the strand, applies sg_align's coordinates, or hands the read to the general kernel (strip.cuh) when the
// winner's path is not one plain diagonal.  Reads longer than the 16-bit frame holds never come here.
#pragma once
#include "common.cuh"
#include "pair16.cuh"

namespace miagpu {

constexpr int SW_K = 16;                            // columns per lane
constexpr int SW_G = 16;                            // lanes per read
constexpr int SW_CW = SW_K * SW_G;                  // chunk width
constexpr int SW_CLASS = 7;                         // the pair class whose frame limits apply (K = 16)

struct Sweep16Params {
  const uint8_t* bases;
  const int64_t* off;
  const int32_t* pairs;          // [n_items][2 half-warps][2] JOBS whose reads have one length; -1 = empty slot
  const int32_t* n_items;
  const int32_t* first_item;     // nullable: the launch's items begin at *first_item (the re-based launch follows the plain one's)
  int32_t* counter;
  const int32_t* job_read;       // job -> read, bit 31 = reverse-complement strand
  const uint8_t* ref2;           // codes of the wrapped forward strand, then (strand_stride bytes on) of the reverse-complement strand
  int32_t strand_stride;
  int32_t len1;
  int32_t rows_cap;              // rows the per-job arrays in shared memory hold (>= the longest read of the launch): sized per launch,
                                 // because the hand-over rings decide how many blocks an SM takes
  const int16_t* prof16;
  uint32_t gep2;
  int32_t rb_off, rb_d, rb_thresh;   // RB: the re-based frame of pair16.cuh 5. (K = 16)
  // per job, the layout p1_merge_kernel reads
  int32_t* jscore; int32_t* jabc; int32_t* jaec; int32_t* jabr;
  uint8_t* jstatus;
};

// dynamic shared memory: [prof16][rowoff WARPS*rows_cap*2 u32][tab WARPS*2*2*P16_TAB_WORDS u32][ring WARPS*2*2*rows_cap*4 u32]
// rowoff as in pair16.cuh: per warp, row r of half-warp hw in word r*2 + hw = {shared address of job A's profile row, job B's << 16}
// (SAME: the one read's, whole word)
__host__ __device__ constexpr int sw_smem(int rows_cap) {
  return (PROF16_N + 8) * 2 + WARPS_PER_BLOCK * rows_cap * 2 * 4 + WARPS_PER_BLOCK * 2 * 2 * P16_TAB_WORDS * 4 +
         WARPS_PER_BLOCK * 2 * 2 * rows_cap * 16;
}

// A half-warp (16 lanes x 16 columns) carries TWO jobs in the halves of its registers: job A in the low half, job B in the high
// half -- (read, strand) pairs whose reads have one length.  Without the k-mer filter they are the two strands of one read; with
// it they are the strands the filter saturated (kmer.c:283-285: the whole strand is unmasked) of any two reads of one length.
// RB: the re-based frame (pair16.cuh 5.) for reads beyond the plain one; every chunk goes through the same re-basings, so what a
// chunk hands to the next stays in step: the last two cells of row r-1 are re-based by the consumer when row r begins with one.
// SAME: the two jobs of a half-warp are the two strands of ONE read (pass 1 without the filter): `pairs` holds reads, two per
// item, job = 2 * read + strand; one row array, one table row -- the kernel of round 1, kept because the general pairing costs it
// eight more registers' worth of spills.
template <bool RB, bool SAME = false>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, 4) sweep16_kernel(Sweep16Params p) {
  constexpr int K = SW_K, G = SW_G;
  constexpr int NE = (25 + G - 1) / G;
  extern __shared__ __align__(16) uint8_t smem[];
  int16_t* s_prof = reinterpret_cast<int16_t*>(smem);
  constexpr int PROF_BYTES = (PROF16_N + 8) * 2;
  const int RC = p.rows_cap;                           // a multiple of 8: the sections stay 16-byte aligned
  const int ROWOFF_BYTES = WARPS_PER_BLOCK * RC * 2 * 4;
  constexpr int TAB_BYTES = WARPS_PER_BLOCK * 2 * 2 * P16_TAB_WORDS * 4;
  uint32_t* s_rowoff = reinterpret_cast<uint32_t*>(smem + PROF_BYTES);
  uint32_t* s_tab = reinterpret_cast<uint32_t*>(smem + PROF_BYTES + ROWOFF_BYTES);
  uint4* s_ring = reinterpret_cast<uint4*>(smem + PROF_BYTES + ROWOFF_BYTES + TAB_BYTES);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int sub = lane & (G - 1), hw = lane / G;
  const unsigned gmask = 0xffffu << (hw * 16);
  for (int i = tid; i < PROF16_N + 8; i += blockDim.x) s_prof[i] = p.prof16[i];
  __syncthreads();

  uint32_t* rowAB = s_rowoff + warp * RC * 2 + hw;                     // row r: rowAB[2 * r]
  uint32_t* tab = s_tab + (warp * 2 + hw) * 2 * P16_TAB_WORDS;
  uint4* ring = s_ring + (size_t)(warp * 2 + hw) * 2 * RC;            // two buffers of RC rows: {l2, l1, acc, scan total}
  const uint32_t prof_base = smem_u32(s_prof);
  const uint32_t tab_addr = smem_u32(tab);

  constexpr int OFFN = p16_off(K);
  const int OFF = RB ? p.rb_off : OFFN;
  constexpr int CONV = GEP * K;
  constexpr int SENT = -32768 + GOP;
  constexpr uint32_t RB_NMIN = B2(-(GOP + 3 * GEP) - OFFN), RB_CELLMIN = B2(-(GOP + 3 * GEP) - OFFN + 2 * GEP - PSSM_ABS_LIMIT);
  const uint32_t rb_d2 = RB ? K2(p.rb_d) : 0u;
  const int n_items = *p.n_items;

  const uint32_t gep2 = p.gep2;
  const int len1 = p.len1;

  uint32_t eoa[NE], eob[NE];
#pragma unroll
  for (int t = 0; t < NE; t++) {
    const int e = min(sub + G * t, 24);
    eoa[t] = p16_tab_a(e) * 2;
    eob[t] = p16_tab_b(e) * 2;
  }
  // entry p16_tab_entry(a, b) = { sub_A(r, a), sub_B(r, b) << 16 }
  auto build_table = [&](int r, uint32_t* dst) {
    const uint32_t ab = rowAB[2 * r];
    const uint32_t pa = SAME ? ab : ab & 0xffffu, pb = SAME ? pa : ab >> 16;
#pragma unroll
    for (int t = 0; t < NE; t++) {
      const uint2 v = make_uint2((uint32_t)lds_s16(pa + eoa[t]), lds_u16(pb + eob[t]) << 16);
      if (sub + G * t < 25) reinterpret_cast<uint2*>(dst)[sub + G * t] = v;
    }
  };

  for (;;) {
    int item = 0;
    if (lane == 0) item = atomicAdd(p.counter, 1);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= n_items) break;
    if (p.first_item) item += *p.first_item;
    // (the jobs are read again at the end instead of being kept in registers through the sweep)
    int soA = 0, soB = 0, L;                         // strand offsets into ref2; rows
    if (SAME) {
      int rd = p.pairs[2 * (int64_t)item + hw];
      if (rd < 0) rd = p.pairs[2 * (int64_t)item];   // an empty slot recomputes the item's first read and writes nothing
      const int64_t o = p.off[rd];
      L = (int)(p.off[rd + 1] - o);
      __syncwarp();
      for (int r = sub; r < L; r += G) rowAB[2 * r] = prof_base + prof_row_index(0, sm_depth(r, L), base_code(p.bases[o + r])) * 2;
      __syncwarp();
    } else {
      int jobA = p.pairs[4 * (int64_t)item + 2 * hw], jobB = p.pairs[4 * (int64_t)item + 2 * hw + 1];
      if (jobA < 0) jobA = p.pairs[4 * (int64_t)item];     // an empty half-warp recomputes the item's first job and writes nothing
      if (jobB < 0) jobB = jobA;                           // an empty B slot rides along as a copy of A
      const int jrA = p.job_read[jobA], jrB = p.job_read[jobB];
      const int rdA = jrA & 0x7fffffff, rdB = jrB & 0x7fffffff;
      soA = jrA < 0 ? p.strand_stride : 0;
      soB = jrB < 0 ? p.strand_stride : 0;
      const int64_t oA = p.off[rdA], oB = p.off[rdB];
      L = (int)(p.off[rdA + 1] - oA);                // the same for every read of the item
      __syncwarp();
      for (int r = sub; r < L; r += G) {
        const int d = sm_depth(r, L);
        rowAB[2 * r] = (prof_base + prof_row_index(0, d, base_code(p.bases[oA + r])) * 2) |
                       (prof_base + prof_row_index(0, d, base_code(p.bases[oB + r])) * 2) << 16;
      }
      __syncwarp();
    }

    int bestv[2] = {INT_MIN, INT_MIN}, bestc[2] = {0, 0}, rb_shift = 0;
    bool bestbad[2] = {false, false}, bestsunk[2] = {false, false};
    int cur = 0;                                     // ring buffer the current chunk WRITES; it reads the other one
    for (int c0 = 0; c0 < len1; c0 += SW_CW, cur ^= 1) {
      const bool first = c0 == 0;
      uint4* rin = ring + (cur ^ 1) * RC;
      uint4* rout = ring + cur * RC;
      // lane masks of the group's first lane: in the first chunk it has no left neighbour (one LOP3 instead of a select)
      const bool edge = sub == 0 && first;
      const uint32_t keep = edge ? 0u : 0xffffffffu;
      const uint32_t sentm = edge ? B2(SENT) : 0u;
      uint32_t cur_n = RB ? ((uint32_t)(-(GOP + 3 * GEP) - OFF + 32768) & 0xffffu) * 0x10001u : B2(-(GOP + 3 * GEP) - OFFN);
      uint32_t ncmp0m = edge ? cur_n : 0u;
      rb_shift = 0;
      uint32_t comb[K];
#pragma unroll
      for (int j = 0; j < K; j++) {
        const int c = c0 + sub * K + j;
        int a = P16_PAD_CODE, b = P16_PAD_CODE;      // padding columns: see P16_PAD_CODE (pair16.cuh)
        if (c < len1) {
          if (SAME) { a = __ldg(p.ref2 + c); b = __ldg(p.ref2 + p.strand_stride + c); }
          else { a = __ldg(p.ref2 + soA + c); b = __ldg(p.ref2 + soB + c); }
        }
        comb[j] = tab_addr + (uint32_t)p16_tab_entry(a, b) * 8;
      }
      __syncwarp();
      build_table(0, tab);
      __syncwarp();
      // ---- row 0 (mia.c:769-785)
      uint32_t W[K], Rg[K], acc[K];
      if (L > 1) build_table(1, tab + P16_TAB_WORDS);
#pragma unroll
      for (int j = 0; j < K; j++) {
        const uint2 e = lds_entry<0>(comb[j]);
        if (RB) W[j] = ((uint32_t)(GEP * j - OFF + 32768) & 0xffffu) * 0x10001u + e.x + e.y;
        else W[j] = B2(GEP * j - OFFN) + e.x + e.y;
        Rg[j] = B2(-32768);
        acc[j] = 0;
      }
      if (sub == G - 1) rout[0] = make_uint4(W[K - 2], W[K - 1], 0u, 0u);
      __syncwarp();

      auto dp_row = [&](int r, auto par, const uint32_t (&W)[K], const uint32_t (&acc)[K], uint32_t (&Wn)[K], uint32_t (&accn)[K]) {
        constexpr int PAR = decltype(par)::value;
        if (r + 1 < L) build_table(r + 1, tab + (PAR ^ 1) * P16_TAB_WORDS);
        uint32_t l2 = __shfl_up_sync(0xffffffffu, W[K - 2], 1, G);
        uint32_t l1 = __shfl_up_sync(0xffffffffu, W[K - 1], 1, G);
        uint32_t ain = __shfl_up_sync(0xffffffffu, acc[K - 1], 1, G);
        uint32_t qin = 0;                                            // biased -infinity
        if (sub == 0 && !first) {                                    // the previous chunk's last lane is this lane's left neighbour
          const uint4 a = rin[r - 1], b = rin[r];
          l2 = a.x; l1 = a.y; ain = a.z; qin = b.w;
          if (RB && (r & (P16_RB_ROWS - 1)) == 1 && r > 1) {         // row r begins with a re-basing: row r-1's cells follow it
            l2 = __vmaxu2(__vsubus2(l2, rb_d2), RB_CELLMIN);
            l1 = __vmaxu2(__vsubus2(l1, rb_d2), RB_CELLMIN);
          }
        }
        l2 = and_or(__vadd2(l2, K2(-CONV)), keep, sentm);
        const uint32_t l1c = __vadd2(l1, K2(-CONV));
        l1 = and_or(l1c, keep, sentm);
        ain &= keep;
        // lane total of the column-gap candidates E = {l2, l1, W[0..K-3]}
        uint32_t X = __vimax3_u16x2(l2, l1, W[0]);
#pragma unroll
        for (int j = 1; j + 1 < K - 2; j += 2) X = __vimax3_u16x2(X, W[j], W[j + 1]);
        if ((K - 3) & 1) X = __vmaxu2(X, W[K - 3]);
        X = __vadd2(X, K2(-GOP));
        // what the previous chunk's scan carried up to its last lane, one lane hop away (0 = -infinity stays 0)
        const uint32_t qc = sub == 0 ? __vadd2(__vmaxu2(qin, B2(-32768 + CONV)), K2(-CONV)) : 0u;
        X = __vmaxu2(X, qc);
#pragma unroll
        for (int d = 1; d < G; d <<= 1) {
          const uint32_t y = __shfl_up_sync(0xffffffffu, X, d, G);
          X = __viaddmax_u16x2(__vmaxu2(y, B2(-32768 + CONV * d)), K2(-CONV * d), X);
        }
        uint32_t q = __shfl_up_sync(0xffffffffu, X, 1, G);
        q = __vadd2(__vmaxu2(q, B2(-32768 + CONV)), K2(-CONV));
        if (sub == 0) q = qc;
        uint32_t Q[K];
        Q[0] = __viaddmax_u16x2(l2, K2(-GOP), q);
        Q[1] = __viaddmax_u16x2(l1, K2(-GOP), Q[0]);
#pragma unroll
        for (int j = 2; j < K; j++) Q[j] = __viaddmax_u16x2(W[j - 2], K2(-GOP), Q[j - 1]);
#pragma unroll
        for (int j = 0; j < K; j++) {
          const uint32_t ncmpj = (RB ? cur_n : B2(-(GOP + 3 * GEP) - OFFN)) + K2(GEP * j);
          uint32_t D, ad;
          if (j > 0) { D = W[j - 1]; ad = acc[j - 1]; }
          else { D = and_or(l1c, keep, ncmp0m); ad = ain; }          // matrix column 0: S = sub + N, never start-new (mia.c:805-822)
          const uint32_t best = __vimax3_u16x2(D, Q[j], Rg[j]);
          Rg[j] = __viaddmax_u16x2(D, K2(-GOP), Rg[j]);
          const uint2 e = lds_entry<PAR * P16_TAB_WORDS * 4>(comb[j]);
          uint32_t bp;
          Wn[j] = cell_pair(best, ncmpj, e.x, e.y, gep2, bp);
          accn[j] = ad | (bp ^ D);
        }
        if (sub == G - 1) {                                          // hand-over to the next chunk: this row's cells, this row's scan total
          rout[r] = make_uint4(Wn[K - 2], Wn[K - 1], accn[K - 1], X);
        }
        __syncwarp();
      };
      auto rebase = [&](uint32_t (&W)[K]) {                          // pair16.cuh 5.
#pragma unroll
        for (int j = 0; j < K; j++) {
          W[j] = __vmaxu2(__vsubus2(W[j], rb_d2), RB_CELLMIN);
          Rg[j] = __vsubus2(Rg[j], rb_d2);
        }
        cur_n = __vmaxu2(__vsubus2(cur_n, rb_d2), RB_NMIN);
        rb_shift += p.rb_d;
        ncmp0m = edge ? cur_n : 0u;
      };
      {
        uint32_t W1[K], acc1[K];
        int r = 1;
        for (; r + 1 < L; r += 2) {
          if (RB && (r & (P16_RB_ROWS - 1)) == 1 && r > 1) rebase(W);
          dp_row(r, std::integral_constant<int, 1>{}, W, acc, W1, acc1);
          dp_row(r + 1, std::integral_constant<int, 0>{}, W1, acc1, W, acc);
        }
        if (r < L) {
          if (RB && (r & (P16_RB_ROWS - 1)) == 1 && r > 1) rebase(W);
          dp_row(r, std::integral_constant<int, 1>{}, W, acc, W1, acc1);
#pragma unroll
          for (int j = 0; j < K; j++) { W[j] = W1[j]; acc[j] = acc1[j]; }
        }
      }
      // ---- this chunk's part of max_sg_score: first maximum of the last row, strict '>' across chunks
#pragma unroll
      for (int h = 0; h < 2; h++) {
        int best = INT_MIN;
#pragma unroll
        for (int j = 0; j < K; j++) {
          const int cl = sub * K + j;
          const int v = (int)(h ? (W[j] >> 16) : (W[j] & 0xffffu)) - 32768 - GEP * j;
          const int key = (c0 + cl < len1) ? v * 512 + (KEY_IDX_MASK - cl) : INT_MIN;
          best = max(best, key);
        }
        best = __reduce_max_sync(gmask, best);
        const int cl = KEY_IDX_MASK - (best & KEY_IDX_MASK);
        const int v = best >> 9;
        bool bad = false;
#pragma unroll
        for (int j = 0; j < K; j++)
          if (sub * K + j == cl) bad = (h ? (acc[j] >> 16) : (acc[j] & 0xffffu)) != 0;
        bad = __any_sync(gmask, bad);
        if (best != INT_MIN && v > bestv[h]) {
          bestv[h] = v; bestc[h] = c0 + cl; bestbad[h] = bad;
          bestsunk[h] = RB && v + GEP * (cl % K) <= p.rb_thresh;      // an end value in the poisoned range: only an upper bound
        }
      }
      __syncwarp();
    }
    int jobA, jobB;
    if (SAME) { const int rd = p.pairs[2 * (int64_t)item + hw]; jobA = rd < 0 ? -1 : 2 * rd; jobB = 2 * rd + 1; }
    else { jobA = p.pairs[4 * (int64_t)item + 2 * hw]; jobB = p.pairs[4 * (int64_t)item + 2 * hw + 1]; }
    if (sub == 0 && jobA >= 0) {
#pragma unroll
      for (int h = 0; h < 2; h++) {
        if (h && jobB < 0) continue;
        const int64_t j = h ? jobB : jobA;
        const int aec = bestc[h];
        const int nsteps = min(L - 1, aec);
        p.jscore[j] = bestv[h] + OFF - GEP * (L - 1) + rb_shift;
        p.jaec[j] = aec;
        p.jabc[j] = aec - nsteps;
        p.jabr[j] = L - 1 - nsteps;
        p.jstatus[j] = bestsunk[h] ? P16_ST_SUNK : bestbad[h] ? P16_ST_GENERAL : MIAGPU_ST_OK;
      }
    }
  }
}

// ---- work items of the sweep: jobs grouped by read length, four to an item (two per half-warp, two half-warps that must run
// the same number of rows).  A counting sort over the lengths; every length's run is padded with -1 to a multiple of four.
//   cnt[0 .. 256] jobs per length | start[0 .. 257] first slot of a length (start[257] = all slots) | cursor[0 .. 256]
constexpr int SW_LAYOUT_WORDS = 3 * (MAX_READ + 2) + 4;      // + n_items[2], work counters[2]
// (job_read == nullptr: the list holds reads, not jobs)
__global__ void __launch_bounds__(256) sw_hist_kernel(int64_t m, const int32_t* __restrict__ jobs, const int32_t* __restrict__ job_read,
                                                      const int64_t* __restrict__ off, int32_t* cnt) {
  __shared__ int s_cnt[MAX_READ + 1];
  for (int l = threadIdx.x; l <= MAX_READ; l += blockDim.x) s_cnt[l] = 0;
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const int e = jobs ? jobs[i] : (int32_t)i;
    const int rd = job_read ? job_read[e] & 0x7fffffff : e;
    atomicAdd(&s_cnt[min((int)(off[rd + 1] - off[rd]), MAX_READ)], 1);
  }
  __syncthreads();
  for (int l = threadIdx.x; l <= MAX_READ; l += blockDim.x) if (s_cnt[l]) atomicAdd(cnt + l, s_cnt[l]);
}
// n_items[0] = items whose reads are at most lmax_low long (the plain frame), n_items[1] = the others (the re-based frame)
// per_item: list entries per work item (4 jobs, or 2 reads)
__global__ void sw_layout_kernel(const int32_t* cnt, int32_t* start, int32_t* cursor, int lmax_low, int32_t* n_items, int per_item) {
  if (threadIdx.x != 0) return;
  int run = 0, low = 0;
  for (int l = 0; l <= MAX_READ; l++) {
    start[l] = run; cursor[l] = run;
    run += (cnt[l] + per_item - 1) / per_item * per_item;
    if (l == lmax_low) low = run;
  }
  start[MAX_READ + 1] = run;
  n_items[0] = low / per_item;
  n_items[1] = (run - low) / per_item;
}
__global__ void __launch_bounds__(256) sw_scatter_kernel(int64_t m, const int32_t* __restrict__ jobs, const int32_t* __restrict__ job_read,
                                                         const int64_t* __restrict__ off, int32_t* cursor, int32_t* out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const int job = jobs ? jobs[i] : (int32_t)i;
  const int rd = job_read ? job_read[job] & 0x7fffffff : job;
  out[atomicAdd(cursor + min((int)(off[rd + 1] - off[rd]), MAX_READ), 1)] = job;
}

// every read becomes two "jobs" (forward strand, reverse-complement strand) of the sweep; reads the 16-bit frame does
// not hold go to the general kernel.  new_kmer_filter returns 1 without a filter (kmer.c:251-255).
struct SweepPrepParams {
  int64_t n;
  const int64_t* off;
  int lmax;
  uint8_t* route; int32_t* jfirst; uint16_t* jcount; uint8_t* jkind; int32_t* job_read; int32_t* sw_jobs; int32_t* hits;
  int32_t* general_list; int32_t* meta;
};
__global__ void sweep_prep_kernel(SweepPrepParams p, int p1_ngeneral) {
  const int64_t rd = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (rd >= p.n) return;
  const int L = (int)(p.off[rd + 1] - p.off[rd]);
  p.hits[rd] = 1;
  p.job_read[2 * rd] = (int32_t)rd;
  p.job_read[2 * rd + 1] = (int32_t)((uint32_t)rd | 0x80000000u);
  if (L >= 1 && L <= p.lmax) {
    p.route[rd] = 1;
    p.jfirst[rd] = (int32_t)(2 * rd);
    p.jcount[rd] = 0x0101;
    p.jkind[2 * rd] = p.jkind[2 * rd + 1] = (uint8_t)(16 + SW_CLASS);
    p.sw_jobs[atomicAdd(&p.meta[META_PREADS + SW_CLASS], 1)] = (int32_t)rd;      // the sweep's list holds READS here (SAME kernels)
  } else {
    p.route[rd] = 2;
    p.jcount[rd] = 0;
    p.general_list[atomicAdd(p.meta + p1_ngeneral, 1)] = (int32_t)rd;
  }
}

}  // namespace miagpu
