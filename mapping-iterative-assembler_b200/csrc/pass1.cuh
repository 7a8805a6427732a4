// pass1.cuh -- pass 1 with the k-mer filter on: seeding and the windowed fast path (sm_100a).
//
// new_kmer_filter (kmer.c:239-331) unmasks, for every k-mer hit (read offset p, reference position q), the columns
// [q-p-10, q+(L-p)+10] (one less on the reverse strand) of that strand's matrix; sg_align (mia.c:1500-1610) then
// runs dyn_prog over both whole strands, where masked cells are HIM.  For a read whose hits on a strand all lie on
// neighbouring diagonals the unmasked columns form ONE stretch of about L+20 columns, and the masked DP over the
// whole strand equals a DP over that stretch alone (pair16.cuh, JOB kernels, explains the one cell rule that
// differs).  Several stretches on one strand (chance k-mer hits elsewhere, the rule on a long reference) are
// independent DPs as well when enough masked columns lie between them: the only state dyn_prog carries across masked
// columns is best_gap_col (H3), a candidate worth at most S - P(g) = r*max(sm) - GOP - GEP*g in row r after g masked
// columns, and a column-gap candidate below the start-new value N(r) = -P(r+1) can never be chosen nor change which
// other candidate is (mia.c:910-965: every branch compares against N first).  So with
//     GEP*g > (L-1)*(max(sm) + GEP) + GEP          [`need` in p1_seed_kernel]
// every stretch is its own job, and max_sg_score's first maximum of the last row is the first maximum over the
// jobs in column order.  So:
//   p1_seed_kernel   warp per read: k-mer lookups on both strands -> hits and their diagonals, chained into stretches;
//                    a strand becomes up to P1_JPS jobs (allocated from one counter, a read's jobs are contiguous) when every stretch is
//                    at most 256 columns wide, the stretches are far enough apart and the read fits the 16-bit
//                    frame; a read whose strands with hits are all jobs goes to the pair kernels, a read without hits
//                    is skipped (mia_main.c:781), everything else (close stretches, saturated strand, long read)
//                    goes to the general kernel (strip.cuh)
//   pair16_kernel<K, true>      the jobs, two per register
//   p1_merge_kernel  first best job per strand, strand pick (forward only if strictly better, mia.c:1549-1554),
//                    sg_align's coordinates (c2rcc, as / ae / start / end fix-ups, mia.c:1568-1610), or hand-over to
//                    the general kernel when the winning job's alignment was not one plain diagonal
#pragma once
#include "common.cuh"
#include "pair16.cuh"
#include "strip.cuh"

namespace miagpu {

// p1 meta block (int32 words) -- laid out like the realign meta block where pair_layout / pair_scatter read it
constexpr int P1_NGENERAL = META_P1;      // reads handed to the general kernel (list fill counter)
constexpr int P1_NFAST = META_P1 + 1;     // reads finished by the pair kernels
constexpr int P1_NSKIPPED = META_P1 + 2;  // reads without a k-mer hit
constexpr int P1_WORK = META_P1 + 3;      // work-fetch counter of the general kernel

constexpr int P1_WORK2 = META_P1 + 5;       // work-fetch counter of the general kernel's second launch (reads the merge handed over)
constexpr int P1_NJOBS = META_P1 + 4;       // jobs allocated (may exceed the capacity: reads that did not fit go to the general kernel)
constexpr int P1_EFF = META_P1 + 6;         // [2] int64: effective DP cells = sum over strands of L x unmasked columns (SURVEY 8d)
constexpr int P1_NTRACE = META_COUNT;       // winning jobs whose path is not one plain diagonal: traced by realign_kernel<K, false, true> (list fill counter)
constexpr int P1_TWORK = META_WORK;         // [3] work-fetch counters of those launches (the pass-1 meta block has no 32-bit work lists of its own)
constexpr int P1_NSWEEP = META_COUNT + 1;   // strands the filter saturated: whole-strand jobs of sweep16_kernel (list fill counter)
constexpr int P1_NSUNK = META_COUNT + 2;    // jobs that left the 16-bit frame (pair16.cuh 5.): computed by the 32-bit JOB kernel before the merge (list fill counter)
constexpr int P1_SWORK = META_WORK + 3;     // [3] work-fetch counters of those launches
constexpr uint8_t P1_KIND_SWEEP = 1;        // jkind of such a job (a pair-class job has 16 + class, 0 = no job)
constexpr int P1_JPS = 12;           // stretches per strand that become jobs
constexpr int P1_MAXD = 128;         // diagonals kept per strand: KMER_SATURATE hits unmask the whole strand anyway

struct Stretches { int hits, n; int lo[P1_JPS], hi[P1_JPS]; };   // n > P1_JPS: too many

// The read as 2-bit codes, 16 bases per 32-bit word, first base in the top bits (so that a k-mer's index -- first base
// most significant, kmer2inx kmer.c:18-48 -- is a funnel shift away), plus one validity bit per base (A/C/G/T after
// upper-casing, kmer.c:27), 32 bases per word.  Lane l packs bases [8l, 8l+8).  s_code: 17 words, s_valid: 9 words.
__device__ __forceinline__ void pack_read(const uint8_t* __restrict__ read, const int L, uint32_t* s_code, uint32_t* s_valid) {
  const int lane = threadIdx.x & 31;
  uint32_t code = 0, valid = 0;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const int i = lane * 8 + j;
    const int c = i < L ? kmer_code(read[i]) : -1;
    code = (code << 2) | (uint32_t)(c & 3);
    valid = (valid << 1) | (c >= 0 ? 1u : 0u);
  }
  reinterpret_cast<uint16_t*>(s_code)[lane ^ 1] = (uint16_t)code;      // word = (even lane << 16) | odd lane
  reinterpret_cast<uint8_t*>(s_valid)[lane ^ 3] = (uint8_t)valid;      // word = lanes 4j .. 4j+3, first in the top byte
  if (lane == 0) { s_code[16] = 0; s_valid[8] = 0; }
  __syncwarp();
}

// new_kmer_filter's hit loop (kmer.c:275-327) without the mask, both strands in one pass over the read's k-mers:
// the hit diagonals (reference position - read offset) of strand t go to s_diag[t] (the first P1_MAXD), s_n[t] counts.
__device__ __forceinline__ void seed_hits(const KmerTable (&kt)[2], const int k, const int L, const uint32_t* s_code, const uint32_t* s_valid,
                                          int (*s_diag)[P1_MAXD], int* s_n) {
  const int lane = threadIdx.x & 31;
  if (lane < 2) s_n[lane] = 0;
  __syncwarp();
  const uint32_t full = (1u << k) - 1;
  for (int p = lane; p + k <= L; p += 32) {
    const uint32_t v = __funnelshift_l(s_valid[(p >> 5) + 1], s_valid[p >> 5], p & 31) >> (32 - k);
    if (v != full) continue;                                             // a base other than A/C/G/T: kmer2inx fails
    const uint32_t inx = __funnelshift_l(s_code[(p >> 4) + 1], s_code[p >> 4], 2 * (p & 15)) >> (32 - 2 * k);
#pragma unroll
    for (int t = 0; t < 2; t++) {
      const int b = (int)(inx >> kt[t].bucket_shift);
      const int e0 = __ldg(kt[t].bucket_start + b), e1 = __ldg(kt[t].bucket_start + b + 1);
      for (int e = e0; e < e1; e++) {
        if (__ldg(kt[t].kmer + e) != inx) continue;
        const int slot = atomicAdd(&s_n[t], 1);
        if (slot < P1_MAXD) s_diag[t][slot] = __ldg(kt[t].pos + e) - p;
      }
    }
  }
  __syncwarp();
}

// The hit diagonals of one strand chained into stretches: two hits belong to one stretch when their unmasked
// intervals [d - 10, d + span - 10] overlap or adjoin, i.e. their diagonals differ by at most span + 1.
__device__ __forceinline__ Stretches chain_stretches(const int hits, const int* s_diag, const int span) {
  const int lane = threadIdx.x & 31;
  Stretches r;
  r.hits = hits;
  r.n = 0;
  if (r.hits == 0 || r.hits >= KMER_SATURATE) return r;
  int v[P1_MAXD / 32];
#pragma unroll
  for (int i = 0; i < P1_MAXD / 32; i++) v[i] = lane + 32 * i < r.hits ? s_diag[lane + 32 * i] : INT_MAX;
  int lo = INT_MAX;
#pragma unroll
  for (int i = 0; i < P1_MAXD / 32; i++) lo = min(lo, v[i]);
  lo = __reduce_min_sync(0xffffffffu, lo);
  while (lo != INT_MAX) {
    int hi = lo;
    for (;;) {                                        // extend the stretch while some diagonal is within reach
      int m = hi;
#pragma unroll
      for (int i = 0; i < P1_MAXD / 32; i++)
        if (v[i] != INT_MAX && v[i] > hi && v[i] <= hi + span + 1) m = max(m, v[i]);
      m = __reduce_max_sync(0xffffffffu, m);
      if (m == hi) break;
      hi = m;
    }
    if (r.n < P1_JPS) { r.lo[r.n] = lo; r.hi[r.n] = hi; }
    r.n++;
    if (r.n > P1_JPS) break;
    int nx = INT_MAX;
#pragma unroll
    for (int i = 0; i < P1_MAXD / 32; i++)
      if (v[i] != INT_MAX && v[i] > hi) nx = min(nx, v[i]);
    lo = __reduce_min_sync(0xffffffffu, nx);
  }
  return r;
}

struct P1SeedParams {
  const uint8_t* bases;
  const int64_t* off;
  int64_t n;
  int32_t k, len1, strand_stride, pssm_max;
  KmerTable kt[2];
  PairLmax lm;
  int32_t sw_lmax;               // longest read sweep16_kernel takes (0: saturated strands go to the general kernel)
  int32_t* sw_jobs;              // jobs of the saturated strands
  // per job (zeroed jkind: a slot nobody filled is no job)
  int64_t job_cap;
  uint8_t* jkind;                // 16 + pair class, 0 = no job
  int32_t* jws;                  // first column of the stretch, as an index into the concatenated codes
  int32_t* jwl;                  // columns
  int32_t* jread;                // read, bit 31 = reverse strand
  // per read
  int32_t* jfirst;               // first job of the read; its forward stretches in column order, then the reverse ones
  uint16_t* jcount;              // forward | reverse << 8
  int32_t* hits;
  uint8_t* route;                // 0 skipped, 1 pair kernels, 2 general kernel
  int32_t* general_list;
  int32_t* score; int32_t* n_runs; uint8_t* status;
  int32_t* meta;
};

__global__ void __launch_bounds__(256) p1_seed_kernel(P1SeedParams p) {
  __shared__ int s_hist[P16_KEYS];
  __shared__ int s_preads[P16_NKB], s_pmaxl[P16_NKB];
  __shared__ unsigned long long s_pcells[P16_NKB];
  __shared__ int s_counts[3];
  __shared__ int s_diag[8][2][P1_MAXD];
  __shared__ int s_nd[8][2];
  __shared__ uint32_t s_code[8][17], s_valid[8][9];
  __shared__ int s_need[8];
  __shared__ long long s_first[8];
  __shared__ unsigned long long s_eff;
  if (threadIdx.x == 0) s_eff = 0;
  for (int i = threadIdx.x; i < P16_KEYS; i += blockDim.x) s_hist[i] = 0;
  if (threadIdx.x < P16_NKB) { s_preads[threadIdx.x] = 0; s_pcells[threadIdx.x] = 0; s_pmaxl[threadIdx.x] = 0; }
  if (threadIdx.x < 3) s_counts[threadIdx.x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  // block-uniform rounds of 8 reads: the jobs of a round are allocated with ONE atomic on the global counter
  for (int64_t rd0 = (int64_t)blockIdx.x * (blockDim.x >> 5); rd0 < p.n; rd0 += warps) {
    const int64_t rd = rd0 + w;
    const bool live = rd < p.n;
    const int64_t o = live ? p.off[rd] : 0;
    const int L = live ? (int)(p.off[rd + 1] - o) : 0;
    const bool odd = live && (L <= 0 || L > MAX_READ);                    // the general kernel reports it
    Stretches st[2];
    st[0].hits = st[1].hits = 0; st[0].n = st[1].n = 0;
    if (live && !odd && L >= p.k) {
      pack_read(p.bases + o, L, s_code[w], s_valid[w]);
      seed_hits(p.kt, p.k, L, s_code[w], s_valid[w], s_diag[w], s_nd[w]);
      // every hit unmasks [d - 10, d + L + 10 - s] (kmer.c:294, 319)
      st[0] = chain_stretches(s_nd[w][0], s_diag[w][0], L + 2 * ALIGN_MASK_BUFFER);
      st[1] = chain_stretches(s_nd[w][1], s_diag[w][1], L + 2 * ALIGN_MASK_BUFFER - 1);
      __syncwarp();                                                        // everybody is done with the shared lists
    }
    const int total = st[0].hits + st[1].hits;
    if (live && lane == 0) p.hits[rd] = odd ? 0 : total;
    if (live && lane == 0 && !odd && total > 0) {                         // effective cells: L x the columns new_kmer_filter unmasks
      unsigned long long eff = 0;
      for (int s = 0; s < 2; s++) {
        if (!st[s].hits) continue;
        if (st[s].hits >= KMER_SATURATE || st[s].n > P1_JPS) { eff += (unsigned long long)L * p.len1; continue; }   // (> 12 stretches: counted whole)
        for (int t = 0; t < st[s].n; t++) {
          const int a = max(st[s].lo[t] - ALIGN_MASK_BUFFER, 0), z = min(st[s].hi[t] + L + ALIGN_MASK_BUFFER - s, p.len1 - 1);
          if (z >= a) eff += (unsigned long long)L * (z - a + 1);
        }
      }
      atomicAdd(&s_eff, eff);
    }
    bool fast = live && !odd && total > 0;
    // masked columns needed between two stretches so that no column-gap candidate crosses (see the header)
    const int need = (L - 1) * (max(p.pssm_max, 0) + GEP) + GEP;
    bool sat[2] = {false, false};
    for (int s = 0; s < 2 && fast; s++) {
      if (!st[s].hits) continue;
      if (st[s].hits >= KMER_SATURATE) {                                   // kmer.c:283-285: the whole strand is unmasked -> one whole-strand job
        if (L > p.sw_lmax) { fast = false; break; }
        sat[s] = true; st[s].n = 1;
        continue;
      }
      if (st[s].n > P1_JPS) { fast = false; break; }
      const int span = L + 2 * ALIGN_MASK_BUFFER - s;                    // last column of a hit's interval minus its first
      int prev_z = -1;
      for (int t = 0; t < st[s].n; t++) {
        int a = st[s].lo[t] - ALIGN_MASK_BUFFER, z = st[s].hi[t] + span - ALIGN_MASK_BUFFER;
        if (a < 0) a = 0;
        if (z >= p.len1) z = p.len1 - 1;
        const int kb = z < a ? -1 : p16_job_class(z - a + 1);
        if (kb < 0 || L > p.lm.v[kb]) { fast = false; break; }
        if (t > 0 && !(GEP * (a - prev_z - 1) > need)) { fast = false; break; }
        prev_z = z;
        st[s].lo[t] = a; st[s].hi[t] = z;                                // from here on: first / last unmasked column
      }
    }
    if (lane == 0) s_need[w] = fast ? st[0].n + st[1].n : 0;
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int i = 0; i < 8; i++) tot += s_need[i];
      long long base = tot ? (long long)atomicAdd(reinterpret_cast<unsigned int*>(p.meta + P1_NJOBS), (unsigned)tot) : 0;
      for (int i = 0; i < 8; i++) { s_first[i] = base; base += s_need[i]; }
    }
    __syncthreads();
    if (lane != 0 || !live) continue;
    const int64_t first = s_first[w];
    if (fast && first + st[0].n + st[1].n > p.job_cap) fast = false;     // no room: the slots stay "no job"
    if (odd) {
      p.route[rd] = 2; p.jcount[rd] = 0; p.general_list[atomicAdd(p.meta + P1_NGENERAL, 1)] = (int32_t)rd;
    } else if (!total) {
      p.route[rd] = 0;
      p.status[rd] = MIAGPU_ST_SKIPPED; p.n_runs[rd] = 0; p.score[rd] = INT_MIN;      // mia_main.c:781: not aligned at all
      p.jcount[rd] = 0;
      atomicAdd(&s_counts[0], 1);
    } else if (!fast) {
      p.route[rd] = 2;
      p.jcount[rd] = 0;
      p.general_list[atomicAdd(p.meta + P1_NGENERAL, 1)] = (int32_t)rd;
    } else {
      p.route[rd] = 1;
      p.jfirst[rd] = (int32_t)first;
      p.jcount[rd] = (uint16_t)(st[0].n | (st[1].n << 8));
      int64_t job = first;
      for (int s = 0; s < 2; s++)
        for (int t = 0; t < st[s].n; t++, job++) {
          if (sat[s]) {
            p.jkind[job] = P1_KIND_SWEEP;
            p.jws[job] = s * p.strand_stride;
            p.jwl[job] = p.len1;
            p.jread[job] = (int32_t)((uint32_t)rd | ((uint32_t)s << 31));
            p.sw_jobs[atomicAdd(p.meta + P1_NSWEEP, 1)] = (int32_t)job;
            continue;
          }
          const int a = st[s].lo[t], wl = st[s].hi[t] - a + 1;
          const int kb = p16_job_class(wl);
          p.jkind[job] = (uint8_t)(16 + kb);
          p.jws[job] = s * p.strand_stride + a;
          p.jwl[job] = wl;
          p.jread[job] = (int32_t)((uint32_t)rd | ((uint32_t)s << 31));
          atomicAdd(&s_hist[kb * (P16_MAXL + 1) + L], 1);
          atomicAdd(&s_preads[kb], 1);
          atomicMax(&s_pmaxl[kb], L);
          atomicAdd(&s_pcells[kb], (unsigned long long)L * wl);
        }
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < P16_KEYS; k += blockDim.x)
    if (s_hist[k]) atomicAdd(&p.meta[META_HIST + k], s_hist[k]);
  if (threadIdx.x < P16_NKB && s_preads[threadIdx.x]) {
    atomicAdd(&p.meta[META_PREADS + threadIdx.x], s_preads[threadIdx.x]);
    atomicAdd(reinterpret_cast<unsigned long long*>(p.meta + META_PCELLS) + threadIdx.x, s_pcells[threadIdx.x]);
    atomicMax(&p.meta[META_PMAXL + threadIdx.x], s_pmaxl[threadIdx.x]);
  }
  if (threadIdx.x == 0 && s_counts[0]) atomicAdd(&p.meta[P1_NSKIPPED], s_counts[0]);
  if (threadIdx.x == 0 && s_eff) atomicAdd(reinterpret_cast<unsigned long long*>(p.meta + P1_EFF), s_eff);
}

struct P1MergeParams {
  int64_t n;
  const int64_t* off;
  int32_t seq_len;
  uint8_t* route;                // 3 = handed to the general kernel by the merge
  const int32_t* jfirst; const uint16_t* jcount;
  const uint8_t* jkind; const uint8_t* jstatus;
  const int32_t* jscore; const int32_t* jabc; const int32_t* jaec; const int32_t* jabr;
  int32_t* general_list;
  int32_t* trace_list;           // nullable (whole-strand jobs of sweep16.cuh: no window to trace in); else the winning jobs the 32-bit JOB kernels trace
  int32_t* meta;
  int32_t *score, *fw_score, *rc_score, *as_out, *ae_out, *start, *end, *abr, *n_runs;
  uint8_t* rc_out;
  uint16_t* runs;
  uint8_t* status;
};

__global__ void p1_merge_kernel(P1MergeParams p) {
  const int64_t rd = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (rd >= p.n || p.route[rd] != 1) return;
  int best[2] = {HIM, HIM};                         // a strand without a hit is masked everywhere: max_sg_score finds HIM in column 0
  int64_t bj[2] = {-1, -1};
  int64_t j0 = p.jfirst[rd];
  const int cnt[2] = {p.jcount[rd] & 0xff, p.jcount[rd] >> 8};
  bool sunk = false;                                // a job whose score is only an upper bound (pair16.cuh 5.): both strands' scores are outputs
  for (int s = 0; s < 2; s++)
    for (int t = 0; t < cnt[s]; t++, j0++) {        // stretches in column order: the first maximum wins (mia.c:1278-1302)
      sunk |= (p.jstatus[j0] & P16_ST_SUNK) != 0;
      if (p.jscore[j0] > best[s]) { best[s] = p.jscore[j0]; bj[s] = j0; }
    }
  const int s = !(best[0] > best[1]) ? 1 : 0;       // forward only if strictly better (mia.c:1549-1554)
  const int64_t j = bj[s];
  if (j >= 0 && !sunk && p.jstatus[j] == P16_ST_GENERAL && p.trace_list && p.jkind[j] != P1_KIND_SWEEP) {
    // every job's score is exact, so the winner is known; only its path is not: the 32-bit kernel runs the winner's stretch with a trace
    p.trace_list[atomicAdd(p.meta + P1_NTRACE, 1)] = (int32_t)j;
    atomicAdd(p.meta + P1_NFAST, 1);
    p.route[rd] = 4;
    p.rc_out[rd] = (uint8_t)s;
    p.fw_score[rd] = best[0]; p.rc_score[rd] = best[1];
    p.score[rd] = best[s];
    return;
  }
  if (j < 0 || sunk || p.jstatus[j] != MIAGPU_ST_OK) {      // a sunk job, or no window to trace in: the general kernel computes the read
    p.general_list[atomicAdd(p.meta + P1_NGENERAL, 1)] = (int32_t)rd;
    p.route[rd] = 3;
    return;
  }
  atomicAdd(p.meta + P1_NFAST, 1);
  const int L = (int)(p.off[rd + 1] - p.off[rd]);
  const int abc = p.jabc[j], aec = p.jaec[j], abr = p.jabr[j];
  int start = abc, end = aec;
  if (s == 1) {                                     // c2rcc, mia.c:26-30
    start = p.seq_len - (aec % p.seq_len) - 1;
    end = p.seq_len - (abc % p.seq_len) - 1;
  }
  int as = start, ae = end;
  if (as > ae) ae = p.seq_len + as;                 // mia.c:1600-1604
  if (end > p.seq_len) end -= p.seq_len;            // mia.c:1606-1610
  p.as_out[rd] = as; p.ae_out[rd] = ae; p.start[rd] = start; p.end[rd] = end;
  p.rc_out[rd] = (uint8_t)s;
  p.fw_score[rd] = best[0]; p.rc_score[rd] = best[1];
  p.abr[rd] = s == 1 ? 0 : abr;                     // row of the run's first base in the STORED orientation
  p.score[rd] = best[s];
  p.n_runs[rd] = 1;
  p.runs[rd * MAX_RUNS] = (uint16_t)((MIAGPU_RUN_M << 14) | (L - abr));
  p.status[rd] = MIAGPU_ST_OK;
}

}  // namespace miagpu
