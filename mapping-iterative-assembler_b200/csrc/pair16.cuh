// pair16.cuh -- windowed PSSM semi-global DP in packed 16-bit SIMD (u16x2), TWO READS PER REGISTER,
// with the pure-diagonal traceback folded into the forward pass (sm_100a).
//
// Same contract as realign.cuh (reiterate_assembly's per-read body, mia_main.c:178-257:
// dyn_prog mia.c:740-981, max_sg_score 1278-1302, find_align_begin 612-637,
// populate_pwaln_to_begin 1440-1497), for the common case: short reads whose path is a plain
// diagonal.  Everything else is handed, read by read, to the 32-bit kernel of realign.cuh through
// its work list -- never approximated.
//
// 1. Two reads of equal length share a group of 16 lanes: every 32-bit register holds the same DP
//    cell of read A (low half) and read B (high half), so one VIADDMNMX.U16x2 / VIMNMX3.U16x2 does
//    two cells.  Lane l of the group owns columns [l*K, l*K+K) as in realign.cuh.  A warp carries
//    two such pairs (four reads of equal length).
//
// 2. Lane frame (checked lane for lane against the oracle by tests/model/pair16_model.c).  A cell of
//    column c = l*K + j is held as  V(r,c) = S(r,c) + GEP*r + GEP*j - OFF  (stored biased, V + 32768,
//    so that the halves order as unsigned numbers); a value taken from another lane is converted by
//    -GEP*K per lane of distance.  In this frame none of dyn_prog's candidates decays:
//      diagonal    V(r-1,c-1)                    + 2*GEP
//      column gap  max_{k<=c-2} V(r-1,k) - GOP   + 2*GEP      (mia.c:838-850: a plain running maximum,
//                                                              per-lane chain seeded by a cross-lane scan)
//      row gap     max_{i<=r-2} V(i,c-1) - GOP   + 2*GEP      (mia.c:856-868: a plain running maximum)
//    and the start-new candidate N_r (mia.c:877-880) is the per-column constant NCMP_j + 2*GEP.
//    A candidate below NCMP_j can never be chosen nor change the start-new test, so the scan clamps
//    from below before converting: no 16-bit operation wraps.  OFF and the longest read the frame
//    holds follow from the matrices' extreme entries (pair16_limits in miagpu.cu).
//
// 3. One table read per cell pair, adds on the FMA pipe.  The substitution scores of a DP row depend
//    on the column only through the two reference codes (a of read A's window, b of read B's), so each
//    group keeps a 25-entry table of 64-bit entries  tab[p16_tab_entry(a,b)] = { (int32) subA(r,a), subB(r,b) << 16 }
//    for the current row in shared memory (double-buffered, built for row r+1 while row r is
//    computed): one LDS.64 per cell pair.  The kernel is bound by the shared-memory data pipe (DESIGN 4.2), so
//    the table is laid out for it: a 64-bit load is served per half-warp (= one group), and the sixteen
//    A/C/G/T pairs sit in entries 0..15, i.e. on sixteen distinct bank pairs -- one wavefront whatever the
//    columns hold, where a*5+b put 0/16, 1/17 and 2/18 on one bank pair (1.82 wavefronts on random
//    columns).  The row offsets of both reads of a group share one 32-bit word.  Because the halves are biased-unsigned and never leave
//    [0, 65535], plain 32-bit adds (IMAD, FMA pipe -- the 16x2 min/max unit is the busy one) add each
//    half exactly: the sign extension of the low entry cancels its borrow.  The start-new rule
//    "S = N, substitution score NOT added" (mia.c:910-915) is the predicate on those two adds; the
//    predicates come out of the VIMNMX.U16x2 that applies the floor NCMP_j.
//
// 4. Traceback without a trace.  find_align_begin walks a plain diagonal exactly when every cell on it
//    (rows and columns >= 1) stored trace 0, i.e. max(D, Gc, Gr, NCMP_j) == D there.  The kernel ORs
//    bad(r,c) = max(...) ^ D down the diagonals (acc(r,c) = acc(r-1,c-1) | bad(r,c), one LOP3 per cell
//    pair, the carry moving with the diagonal operand): acc == 0 in the first-maximum cell of the last
//    row means the alignment is one M run from (abr, abc) = (L-1-n, aec-n), n = min(L-1, aec).
//    Otherwise (gap, start-new cell on the path, jump stored as trace 0) the read is appended to the
//    32-bit kernel's list.  No trace matrix, no band, no scratch memory.
//
// 5. Reads beyond the 16-bit frame (RB = true).  In the frame of 2. a cell on a good path gains up to max(sm) + GEP per row, so
//    a read of more than ~130 rows runs out of the 16-bit range.  The RB variant starts the frame near the TOP of the range and
//    subtracts D = 8 * (max(sm) + GEP) from all state every 8 rows (saturating), so that exact values never rise above their
//    start (+ a bounded fluctuation: within 8 rows, and the GEP*K a path regains each time it crosses into the next lane) while a
//    real read sinks by (max(sm) - its entries) per row.  The start-new level and every cell are clamped from below at the
//    levels the frame of 2. guarantees, so no operation wraps; a clamped value is too HIGH (poisoned), and so is everything
//    derived from it -- but never above clamp level + fluctuation.  If the end cell lies above that bound, every cell of its path
//    does too (values do not rise along a path beyond the fluctuation), none of them was poisoned, and every poisoned candidate
//    they met was strictly lower: score, end cell and verdict are exact.  Otherwise the read goes to the 32-bit kernel.
#pragma once
#include "common.cuh"
#include "realign.cuh"
#include <type_traits>

namespace miagpu {

constexpr int P16_MAXL = MAX_READ;                  // rows the shared row-offset arrays hold
constexpr int PROF16_N = 2 * NMAT * 5 * PROF_ROW_INTS;   // int16 entries
constexpr int P16_NKB = 12;                         // width classes: 128 / 144 / 160 / 176 / 192 / 208 / 224 / 256 columns (K = columns / 16),
                                                    // then the narrow classes of pass-1 jobs: 64 / 80 / 96 / 112 (K = 4 .. 7)
constexpr int P16_NKB_WIDE = 8;                     // classes reiterate_assembly's windows use (a window is at least 100 columns + the read)
constexpr int P16_TAB_WORDS = 64;                   // 25 64-bit entries, padded to 32
constexpr int P16_G = 16;                           // lanes per pair (1. in the header)
constexpr int P16_NP = 32 / P16_G;                  // pairs per warp = per work item

// Entry of the reference codes (a, b) in a group's substitution table (3. in the header): the A/C/G/T pairs at a*4+b, then
// the nine pairs with an N (code 4): (N, b) at 16+b, (a, N) at 21+a.  p16_tab_a / p16_tab_b invert it for the table build.
__host__ __device__ constexpr int p16_tab_entry(int a, int b) { return a < 4 && b < 4 ? a * 4 + b : a == 4 ? 16 + b : 21 + a; }
__host__ __device__ constexpr int p16_tab_a(int e) { return e < 16 ? e >> 2 : e < 21 ? 4 : e - 21; }
__host__ __device__ constexpr int p16_tab_b(int e) { return e < 16 ? e & 3 : e < 21 ? e - 16 : 4; }
constexpr bool p16_tab_bijective() {
  for (int e = 0; e < 25; e++)
    if (p16_tab_a(e) > 4 || p16_tab_b(e) > 4 || p16_tab_entry(p16_tab_a(e), p16_tab_b(e)) != e) return false;
  return true;
}
static_assert(p16_tab_bijective(), "p16_tab_entry maps the 25 code pairs onto 0..24");
// Code of a padding column (c >= the window's length; the last lanes of a group).  Exact whatever it is: dyn_prog's candidates
// of a cell all come from lower columns (mia.c:838-871), so a padding column feeds only padding columns; the end-cell key and
// the verdict (max_sg_score) skip c >= len1; and the frame's bounds (2. and 5. above) use only the matrix's extreme entries,
// never a column's code, so no value wraps.  Code 0 keeps a padding column's entry among the sixteen of distinct bank pairs,
// where code 4 would share a bank pair with one of them.
constexpr int P16_PAD_CODE = 0;

// OFF of the lane frame: the lowest intermediate, (lowest cell = -OFF-GOP-GEP+min entry) converted to the next lane
// (-GEP*K) minus GOP, must stay above -32768 for every matrix set_pssm accepts (|entry| <= PSSM_ABS_LIMIT).
__host__ __device__ constexpr int p16_off(int K) { return 32768 - 2 * GOP - GEP - PSSM_ABS_LIMIT - GEP * K - 32; }
// longest read the frame holds: L*max_entry + GEP*(L-1) + GEP*(K-1) - OFF <= 32767
__host__ __device__ inline int p16_lmax(int K, int max_entry) {
  const int inc = max_entry + GEP;
  return inc > 0 ? (32767 + p16_off(K) - GEP * (K - 2)) / inc : MAX_READ;
}
__host__ __device__ inline int p16_class(int len1) {
  return len1 <= 128 ? 0 : len1 <= 144 ? 1 : len1 <= 160 ? 2 : len1 <= 176 ? 3 : len1 <= 192 ? 4 : len1 <= 208 ? 5 : len1 <= 224 ? 6 : len1 <= 256 ? 7 : -1;
}
// pass-1 jobs (a stretch is about L + 20 columns): the narrow classes first
__host__ __device__ inline int p16_job_class(int len1) {
  return len1 <= 64 ? 8 : len1 <= 80 ? 9 : len1 <= 96 ? 10 : len1 <= 112 ? 11 : p16_class(len1);
}
__host__ __device__ inline int bucket32_of(int len1) {
  return len1 <= 64 ? 0 : len1 <= 128 ? 1 : len1 <= 160 ? 2 : len1 <= 192 ? 3 : len1 <= 224 ? 4 : len1 <= 256 ? 5 : len1 <= 320 ? 6 : len1 <= 384 ? 7 : len1 <= 512 ? 8 : 9;
}

struct PairLmax { int v[P16_NKB]; };                 // longest read each pair class takes (0 = pair kernels off)

// Meta block of a realign / pass-1 job (int32 words): classification counters, pair layout, work-fetch counters
constexpr int META_COUNT = 0;        // [16] fill counters of the 32-bit work lists
constexpr int META_WORK = 16;        // [16] dynamic work-fetch counters of the 32-bit kernels
constexpr int META_MAXL = 32;        // [16] longest read per width class (all reads of the class)
constexpr int META_CELLS = 48;       // [16] int64 DP cells per width class (all reads of the class)
constexpr int META_POP = 80;         // [16] reads per width class (direct + pair-eligible)
constexpr int META_NPAIRS = 96;      // [12] work items per pair class
constexpr int META_PWORK = 108;      // [12] work-fetch counters of the pair kernels
constexpr int META_PREADS = 120;     // [12] eligible reads per pair class
constexpr int META_PCELLS = 132;     // [12] int64 cells of the eligible reads
constexpr int META_MAXLEN = 156;     // scratch of max_len_kernel
constexpr int META_NFALL = 157;      // reads handed from the pair kernels to the 32-bit kernels
constexpr int META_P1 = 158;         // [8]  pass-1 counters (pass1.cuh)
constexpr int META_CELLS32 = 168;    // [10] int64 DP cells the 32-bit kernels actually computed, per width bucket
constexpr int META_PMAXL = 192;      // [12] longest eligible read per pair class (decides between the low and the RB frame)
constexpr int META_HOST = 208;       // words copied to the host after classification
constexpr int P16_KEYS = P16_NKB * (P16_MAXL + 1);
constexpr int META_KEYS = 3200;      // room per key table
constexpr int META_HIST = 256;       // [P16_KEYS] eligible reads per (pair class, read length)
constexpr int META_PSTART = META_HIST + META_KEYS;    // [P16_KEYS] first pair of the key
constexpr int META_CURSOR = META_PSTART + META_KEYS;  // [P16_KEYS] scatter cursors
constexpr int META_WORDS = META_CURSOR + META_KEYS;
static_assert(P16_KEYS <= META_KEYS && P16_NKB == 12 && META_PCELLS % 2 == 0, "meta layout");

struct Pair16Params {
  const uint8_t* bases;
  const int64_t* off;
  const uint8_t* rc;
  const int32_t* win_start;
  const int32_t* win_len;
  int32_t* win_len_narrow;       // realign windows only (null = off): a read handed to the 32-bit kernels keeps the columns up to its end cell
  const int32_t* pairs;          // [n_items][P16_NP][2] read ids; -1 = empty slot (a work item's first slot is never empty)
  const int32_t* n_items;        // device counter (layout kernel wrote it)
  int32_t* counter;
  const uint8_t* ref_codes;
  int32_t ref_bytes;
  int32_t ref_in_smem;
  const int16_t* prof16;
  int32_t* score;
  int32_t* as_out;
  int32_t* ae_out;
  int32_t* abr;
  int32_t* n_runs;
  uint16_t* runs;
  uint8_t* status;
  int32_t* lists;                // 32-bit kernel work lists [NBUCKET][n]
  int32_t* list_counts;          // their fill counters
  int64_t n_reads;
  int32_t* n_fallback;           // statistics
  int32_t* sunk_list;            // JOB + RB kernels: jobs whose end value lies in the poisoned range (list + fill counter): the 32-bit
  int32_t* sunk_count;           // JOB kernel computes them exactly before the merge
  uint32_t gep2;                 // K2(2*GEP), passed as data so that ptxas keeps this add an IMAD (FMA pipe) instead of folding it into a VIADD
  int32_t strand_stride;         // JOB kernels: bytes between the forward and the reverse-complement codes in ref_codes
  const int32_t* job_read;       // JOB kernels: read of a job, bit 31 = reverse strand
  // RB kernels (see 5. in the header): OFF of the high frame, the amount subtracted every P16_RB_ROWS rows, the lowest end value that is exact
  int32_t rb_off, rb_d, rb_thresh;
};

constexpr int P16_RB_ROWS = 8;
// parameters of the RB frame for K columns per lane and the largest matrix entry; feasible = a real read has room to sink
struct RbFrame { int off, d, thresh, room; };
__host__ __device__ inline RbFrame p16_rb_frame(int K, int max_entry) {
  const int mx = max_entry > 0 ? max_entry : 0;
  const int G = P16_RB_ROWS * (mx + 2 * GEP) + GEP * K;                          // fluctuation of an exact value above its long-run level
  RbFrame f;
  f.d = P16_RB_ROWS * (mx + GEP);
  f.off = mx + GEP * (K - 1) + G + 64 - 32767;                                   // row 0 starts at most G + 64 below the top
  const int clamp_cell = -(GOP + 3 * GEP) - (32768 - 2 * GOP - GEP - PSSM_ABS_LIMIT - GEP * K - 32) + 2 * GEP + PSSM_ABS_LIMIT;   // p16_off(K), see below
  f.thresh = clamp_cell + 2 * G + 2 * GOP;                                       // unbiased; above it nothing is poisoned
  f.room = (-f.off) - f.thresh;                                                  // how far a read may sink below the top of row 0
  return f;
}

constexpr uint8_t P16_ST_GENERAL = 0x40;   // JOB kernels: the alignment is not one plain diagonal, the general kernel takes the read
constexpr uint8_t P16_ST_SUNK = 0x20;      // JOB + RB kernels: the job's end value lies in the poisoned range, its score is only an upper bound

// packed constants: B2(v) = the cell value v in both halves (biased), K2(k) = the addend k in both halves
__host__ __device__ constexpr uint32_t B2(int v) { return ((uint32_t)(v + 32768) & 0xffffu) * 0x10001u; }
__host__ __device__ constexpr uint32_t K2(int k) { return ((uint32_t)k & 0xffffu) * 0x10001u; }

__device__ __forceinline__ int lds_s16(uint32_t addr) {
  int v;
  asm volatile("ld.shared.s16 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t and_or(uint32_t a, uint32_t b, uint32_t c) {   // (a & b) | c in one LOP3
  uint32_t d;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
// table entry {eA, eB} at a shared address plus a compile-time offset (the table buffer)
template <int OFS>
__device__ __forceinline__ uint2 lds_entry(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2+%3];" : "=r"(v.x), "=r"(v.y) : "r"(addr), "n"(OFS));
  return v;
}
// One DP cell pair.  bp = max(best, ncmp) per half; w = bp + 2*GEP + (start-new ? 0 : sub) per half, as 32-bit adds
// (exact, see 3. above).  The setp.eq pattern is the one ptxas folds into VIMNMX.U16x2 with two predicate
// outputs; mad.lo keeps the adds on the FMA pipe.
__device__ __forceinline__ uint32_t cell_pair(uint32_t best, uint32_t ncmp, uint32_t ea, uint32_t eb, uint32_t gep2, uint32_t& bp) {
  uint32_t w;
  asm("{.reg .pred pu, pv;\n\t"
      ".reg .u16 h0, h1, h2, h3;\n\t"
      "max.u16x2 %1, %2, %3;\n\t"
      "mov.b32 {h0, h1}, %1;\n\t"
      "mov.b32 {h2, h3}, %2;\n\t"
      "setp.eq.u16 pv, h0, h2;\n\t"
      "setp.eq.u16 pu, h1, h3;\n\t"
      "mad.lo.u32 %0, %1, 1, %6;\n\t"
      "@pv mad.lo.u32 %0, %4, 1, %0;\n\t"
      "@pu mad.lo.u32 %0, %5, 1, %0;}\n\t"
      : "=&r"(w), "=&r"(bp)
      : "r"(best), "r"(ncmp), "r"(ea), "r"(eb), "r"(gep2));
  return w;
}

// dynamic shared memory: [prof16 (PROF16_N + 8) int16][rowoff WARPS*P16_MAXL*P16_NP u32][tab WARPS*P16_NP*2*P16_TAB_WORDS u32][ref codes]
// rowoff: per warp, row r of pair hw in word r*P16_NP + hw = {shared address of read A's profile row, read B's << 16}: one LDS.32
// per row, and the pairs of a warp, which run the same row, read adjacent banks.  The profile is the first section of the block's
// shared memory (after at most a few bytes of static shared memory), so its addresses fit 16 bits.
constexpr int P16_SMEM_FIXED = (PROF16_N + 8) * 2 + WARPS_PER_BLOCK * P16_MAXL * P16_NP * 4 + WARPS_PER_BLOCK * P16_NP * 2 * P16_TAB_WORDS * 4;

// JOB = false: a work item names reads (reiterate_assembly's windows, matrix by strand).
// JOB = true : pass 1 with the k-mer filter (sg_align, mia.c:1500-1610).  A work item names jobs (pass1.cuh;
//   job_read[job] = read, bit 31 = strand): the read against ONE stretch of columns its k-mer hits unmasked on that strand (new_kmer_filter, kmer.c:239-331),
//   always with the forward matrix (H5).  The masked matrix differs from a window in one place: when the stretch does
//   not begin at column 0 its first column has a masked left neighbour, so there dyn_prog starts a new alignment
//   (S = N, substitution score not added, mia.c:910-915) instead of applying the column-0 rule (mia.c:805-822).
//   Everything to the left / right of the stretch is HIM and can neither be chosen nor become the best end cell.
//   Outputs are per job, in strand coordinates: as_out = abc, ae_out = aec.
template <int K, bool JOB, bool RB = false>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, (K <= 5 ? 8 : K <= 7 ? 6 : K <= 12 ? 5 : 4)) pair16_kernel(Pair16Params p) {
  static_assert(K >= 4 && K <= 16, "columns per lane");
  constexpr int NE = (25 + P16_G - 1) / P16_G;       // table entries a lane builds per row
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ __align__(8) uint64_t ref_bar;
  int16_t* s_prof = reinterpret_cast<int16_t*>(smem);
  constexpr int PROF_BYTES = (PROF16_N + 8) * 2;
  constexpr int ROWOFF_BYTES = WARPS_PER_BLOCK * P16_MAXL * P16_NP * 4;
  uint32_t* s_rowoff = reinterpret_cast<uint32_t*>(smem + PROF_BYTES);
  uint32_t* s_tab = reinterpret_cast<uint32_t*>(smem + PROF_BYTES + ROWOFF_BYTES);
  uint8_t* s_ref = smem + P16_SMEM_FIXED;

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int sub = lane & (P16_G - 1);                // lane within the pair's group
  const int hw = lane / P16_G;                       // which pair of the warp
  const unsigned gmask = 0xffffu << (hw * P16_G);

  if (p.ref_in_smem) {
    if (tid == 0) {
      mbar_init(&ref_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
      mbar_expect_tx(&ref_bar, (uint32_t)p.ref_bytes);
      for (int o = 0; o < p.ref_bytes; o += 32768) bulk_g2s(s_ref + o, p.ref_codes + o, (uint32_t)min(32768, p.ref_bytes - o), &ref_bar);
    }
  }
  for (int i = tid; i < PROF16_N + 8; i += blockDim.x) s_prof[i] = p.prof16[i];
  if (p.ref_in_smem) mbar_wait(&ref_bar, 0);
  __syncthreads();

  uint32_t* rowAB = s_rowoff + warp * P16_MAXL * P16_NP + hw;          // row r: rowAB[r * P16_NP]
  uint32_t* tab = s_tab + (warp * P16_NP + hw) * 2 * P16_TAB_WORDS;     // two buffers of P16_TAB_WORDS
  const uint32_t prof_base = smem_u32(s_prof);
  const uint32_t tab_addr = smem_u32(tab);

  constexpr int OFFN = p16_off(K);
  const int OFF = RB ? p.rb_off : OFFN;              // (a compile-time constant without RB)
  constexpr int CONV = GEP * K;                      // frame shift per lane of distance
  constexpr int SENT = -32768 + GOP;                 // "-infinity" that survives one -GOP
  const int n_items = *p.n_items;
  const uint32_t gep2 = p.gep2;
  const uint32_t keep = sub ? 0xffffffffu : 0u;      // lane masks for the group's first lane (one LOP3 instead of a select)
  const uint32_t sentm = sub ? 0u : B2(SENT);
  uint32_t ncmp0m = sub ? 0u : B2(-(GOP + 3 * GEP) - OFFN);
  // RB: the start-new level N(r) in the frame, sinking with the frame but never below the level of the low frame; the cells' clamp
  constexpr uint32_t RB_NMIN = B2(-(GOP + 3 * GEP) - OFFN), RB_CELLMIN = B2(-(GOP + 3 * GEP) - OFFN + 2 * GEP - PSSM_ABS_LIMIT);
  const uint32_t rb_d2 = RB ? K2(p.rb_d) : 0u;
  uint32_t cur_n = 0;

  // table entries this lane builds every row: e = sub + P16_G*t -> (a, b) = (p16_tab_a(e), p16_tab_b(e))
  uint32_t eoa[NE], eob[NE];
#pragma unroll
  for (int t = 0; t < NE; t++) {
    const int e = min(sub + P16_G * t, 24);
    eoa[t] = p16_tab_a(e) * 2;
    eob[t] = p16_tab_b(e) * 2;
  }
  auto build_table = [&](int r, uint32_t* dst) {
    const uint32_t ab = rowAB[r * P16_NP];
    const uint32_t pa = ab & 0xffffu, pb = ab >> 16;
#pragma unroll
    for (int t = 0; t < NE; t++) {
      const uint2 v = make_uint2((uint32_t)lds_s16(pa + eoa[t]), lds_u16(pb + eob[t]) << 16);
      if (sub + P16_G * t < 25) reinterpret_cast<uint2*>(dst)[sub + P16_G * t] = v;
    }
  };

  for (;;) {
    int item = 0;
    if (lane == 0) item = atomicAdd(p.counter, 1);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= n_items) break;
    int rdA = p.pairs[2 * (item * P16_NP + hw)];
    int rdB = p.pairs[2 * (item * P16_NP + hw) + 1];
    const bool hasA = rdA >= 0;                       // an empty pair slot recomputes the warp's first pair and writes nothing
    if (!hasA) rdA = p.pairs[2 * (item * P16_NP)];
    const bool hasB = hasA && rdB >= 0;
    if (rdB < 0 || !hasA) rdB = rdA;
    const int jrA = JOB ? p.job_read[rdA] : 0, jrB = JOB ? p.job_read[rdB] : 0;
    const int rrA = JOB ? jrA & 0x7fffffff : rdA, rrB = JOB ? jrB & 0x7fffffff : rdB;      // the reads behind the jobs
    const int64_t oA = p.off[rrA], oB = p.off[rrB];
    const int L = (int)(p.off[rrA + 1] - oA);         // the same for every read of the work item
    const int wsA = p.win_start[rdA], wsB = p.win_start[rdB];
    const int lenA = p.win_len[rdA], lenB = p.win_len[rdB];
    const int sA = JOB ? 0 : (p.rc[rdA] ? 1 : 0), sB = JOB ? 0 : (p.rc[rdB] ? 1 : 0);
    bool mlA = false, mlB = false;
    if (JOB) {                                        // first column: column 0 of the matrix, or a column with a masked left neighbour
      mlA = wsA - (jrA < 0 ? p.strand_stride : 0) > 0; mlB = wsB - (jrB < 0 ? p.strand_stride : 0) > 0;
      const uint32_t real = B2(-(GOP + 3 * GEP) - OFFN), cut = B2(SENT);
      if (!RB) ncmp0m = sub ? 0u : (((mlA ? cut : real) & 0xffffu) | ((mlB ? cut : real) & 0xffff0000u));
    }
    int rb_shift = 0;                                 // RB: what has been subtracted from the frame so far
    auto rb_ncmp0 = [&]() {                           // RB: column 0's operand follows the start-new level
      if (!JOB) { ncmp0m = sub ? 0u : cur_n; return; }
      const uint32_t cut = B2(SENT);
      ncmp0m = sub ? 0u : (((mlA ? cut : cur_n) & 0xffffu) | ((mlB ? cut : cur_n) & 0xffff0000u));
    };
    if (RB) { cur_n = ((uint32_t)(-(GOP + 3 * GEP) - OFF + 32768) & 0xffffu) * 0x10001u; rb_ncmp0(); }

    __syncwarp();
    for (int r = sub; r < L; r += P16_G) {
      const int d = sm_depth(r, L);
      rowAB[r * P16_NP] = (prof_base + prof_row_index(sA, d, base_code(p.bases[oA + r])) * 2) |
                          (prof_base + prof_row_index(sB, d, base_code(p.bases[oB + r])) * 2) << 16;
    }
    uint32_t comb[K];                                 // shared address of the column's (a, b) entry in table buffer 0
#pragma unroll
    for (int j = 0; j < K; j++) {
      const int c = sub * K + j;
      int a = P16_PAD_CODE, b = P16_PAD_CODE;
      if (c < lenA) a = p.ref_in_smem ? s_ref[wsA + c] : p.ref_codes[wsA + c];
      if (c < lenB) b = p.ref_in_smem ? s_ref[wsB + c] : p.ref_codes[wsB + c];
      comb[j] = tab_addr + (uint32_t)p16_tab_entry(a, b) * 8;
    }
    __syncwarp();
    build_table(0, tab);
    __syncwarp();

    // ---- row 0 (mia.c:769-785): V = sub + GEP*j - OFF
    uint32_t W[K], Rg[K], acc[K];
    {
      if (L > 1) build_table(1, tab + P16_TAB_WORDS);
#pragma unroll
      for (int j = 0; j < K; j++) {
        const uint2 e = lds_entry<0>(comb[j]);
        if (RB) W[j] = ((uint32_t)(GEP * j - OFF + 32768) & 0xffffu) * 0x10001u + e.x + e.y;
        else W[j] = B2(GEP * j - OFFN) + e.x + e.y;   // biased seed + entries: 32-bit adds, as in cell_pair
        Rg[j] = B2(-32768);
        acc[j] = 0;
      }
      __syncwarp();
    }

    // Exclusive prefix over the group's lanes of the lane totals X (each in its own lane's frame): q of lane i = max over the lanes
    // l < i of X_l - CONV * (i - l), clamped so that nothing wraps (a clamped value ends at the bottom of the range, below every
    // start-new level): four doubling steps + the shift by one lane.
    auto lane_prefix = [&](uint32_t X) -> uint32_t {
      // inclusive cross-lane scan, converting by CONV per lane, clamped so nothing wraps
#pragma unroll
      for (int d = 1; d < P16_G; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, X, d, P16_G);
        X = __viaddmax_u16x2(__vmaxu2(y, B2(-32768 + CONV * d)), K2(-CONV * d), X);    // lanes < d get their own X back: max(X, max(X,cl)-dec) = X
      }
      const uint32_t q = __shfl_up_sync(0xffffffffu, X, 1, P16_G);
      return __vadd2(__vmaxu2(q, B2(-32768 + CONV)), K2(-CONV)) & keep;         // B2(-32768) = 0
    };
    // One DP row: row r-1 in W / acc -> row r in Wn / accn (Rg in place).  PAR = r & 1 selects the table buffer at
    // compile time (an immediate offset of the LDS), so the row loop below is unrolled by two and ping-pongs
    // between two register sets (no moves at the back edge).
    auto dp_row = [&](int r, auto par, const uint32_t (&W)[K], const uint32_t (&acc)[K], uint32_t (&Wn)[K], uint32_t (&accn)[K]) {
      constexpr int PAR = decltype(par)::value;
      if (r + 1 < L) build_table(r + 1, tab + (PAR ^ 1) * P16_TAB_WORDS);
      uint32_t l2 = __shfl_up_sync(0xffffffffu, W[K - 2], 1, P16_G);
      uint32_t l1 = __shfl_up_sync(0xffffffffu, W[K - 1], 1, P16_G);
      uint32_t ain = __shfl_up_sync(0xffffffffu, acc[K - 1], 1, P16_G);
      l2 = and_or(__vadd2(l2, K2(-CONV)), keep, sentm);          // first lane of the group: no left neighbour
      const uint32_t l1c = __vadd2(l1, K2(-CONV));
      l1 = and_or(l1c, keep, sentm);
      ain &= keep;
      // lane total of the column-gap candidates E = {l2, l1, W[0..K-3]}
      uint32_t X = __vimax3_u16x2(l2, l1, W[0]);
#pragma unroll
      for (int j = 1; j + 1 < K - 2; j += 2) X = __vimax3_u16x2(X, W[j], W[j + 1]);
      if ((K - 3) & 1) X = __vmaxu2(X, W[K - 3]);
      X = __vadd2(X, K2(-GOP));
      const uint32_t q = lane_prefix(X);
      // column-gap chain (mia.c:838-850): Q[j] = max over columns <= c-2 of V - GOP
      uint32_t Q[K];
      Q[0] = __viaddmax_u16x2(l2, K2(-GOP), q);
      Q[1] = __viaddmax_u16x2(l1, K2(-GOP), Q[0]);
#pragma unroll
      for (int j = 2; j < K; j++) Q[j] = __viaddmax_u16x2(W[j - 2], K2(-GOP), Q[j - 1]);
#pragma unroll
      for (int j = 0; j < K; j++) {
        const uint32_t ncmpj = (RB ? cur_n : B2(-(GOP + 3 * GEP) - OFFN)) + K2(GEP * j);     // NCMP_j: compile-time after unrolling (without RB)
        uint32_t D, ad;
        if (j > 0) { D = W[j - 1]; ad = acc[j - 1]; }
        else { D = and_or(l1c, keep, ncmp0m); ad = ain; }   // column 0: S = sub + N, never start-new (mia.c:805-822)
        const uint32_t best = __vimax3_u16x2(D, Q[j], Rg[j]);
        Rg[j] = __viaddmax_u16x2(D, K2(-GOP), Rg[j]);          // row r-1 joins the row-gap candidates of column c-1
        const uint2 e = lds_entry<PAR * P16_TAB_WORDS * 4>(comb[j]);
        uint32_t bp;
        Wn[j] = cell_pair(best, ncmpj, e.x, e.y, gep2, bp);
        if (JOB && j == 0) accn[j] = and_or(bp ^ D, keep, ad);   // a start-new cell in the stretch's first column ends the walk like column 0 does
        else accn[j] = ad | (bp ^ D);
      }
      __syncwarp();
    };
    // RB: every P16_RB_ROWS rows the frame sinks by rb_d (see 5. in the header); cells and the start-new level keep the low frame's floors
    auto rebase = [&](uint32_t (&W)[K]) {
#pragma unroll
      for (int j = 0; j < K; j++) {
        W[j] = __vmaxu2(__vsubus2(W[j], rb_d2), RB_CELLMIN);
        Rg[j] = __vsubus2(Rg[j], rb_d2);
      }
      cur_n = __vmaxu2(__vsubus2(cur_n, rb_d2), RB_NMIN);
      rb_shift += p.rb_d;
      rb_ncmp0();
    };
    uint32_t W1[K], acc1[K];
    int r = 1;
    for (; r + 1 < L; r += 2) {
      if (RB && (r & (P16_RB_ROWS - 1)) == 1 && r > 1) rebase(W);
      dp_row(r, std::integral_constant<int, 1>{}, W, acc, W1, acc1);
      dp_row(r + 1, std::integral_constant<int, 0>{}, W1, acc1, W, acc);
    }
    if (r < L) {
      dp_row(r, std::integral_constant<int, 1>{}, W, acc, W1, acc1);
#pragma unroll
      for (int j = 0; j < K; j++) { W[j] = W1[j]; acc[j] = acc1[j]; }
    }

    // ---- max_sg_score (first maximum of the last row) + the diagonal verdict, one read (half) at a time
#pragma unroll 1
    for (int h = 0; h < 2; h++) {
      const bool live = h ? hasB : hasA;              // uniform within the group
      const int rd = h ? rdB : rdA;
      const int ws = h ? wsB : wsA;
      const int len1 = h ? lenB : lenA;
      int best = INT_MIN;
#pragma unroll
      for (int j = 0; j < K; j++) {
        const int c = sub * K + j;
        const int v = (int)(h ? (W[j] >> 16) : (W[j] & 0xffffu)) - 32768 - GEP * j;
        const int key = (c < len1) ? v * 512 + (KEY_IDX_MASK - c) : INT_MIN;
        best = max(best, key);
      }
      best = __reduce_max_sync(gmask, best);
      const int aec = KEY_IDX_MASK - (best & KEY_IDX_MASK);
      const int score = (best >> 9) + OFF - GEP * (L - 1) + rb_shift;
      bool bad = false;
#pragma unroll
      for (int j = 0; j < K; j++)
        if (sub * K + j == aec) bad = (h ? (acc[j] >> 16) : (acc[j] & 0xffffu)) != 0;
      // RB: an end value at or below the poison bound may have met clamped cells: the 32-bit kernel takes the read
      const bool sunk = RB && (best >> 9) + GEP * (aec % K) <= p.rb_thresh;
      const bool ok = !__any_sync(gmask, bad) && !sunk;
      const int nsteps = min(L - 1, aec);
      if (JOB) {
        if (sub == 0 && live) {
          const int lo = ws - ((h ? jrB : jrA) < 0 ? p.strand_stride : 0);
          p.score[rd] = score;                          // exact whatever the path looks like (unless sunk): a losing job needs no more
          if (sunk) {
            p.status[rd] = P16_ST_SUNK;                 // sg_align reports both strands' scores: the 32-bit JOB kernel computes this job
            if (p.sunk_list) p.sunk_list[atomicAdd(p.sunk_count, 1)] = rd;
          } else if (ok) {
            p.as_out[rd] = aec - nsteps + lo;           // abc
            p.ae_out[rd] = aec + lo;                    // aec
            p.abr[rd] = L - 1 - nsteps;
            p.status[rd] = MIAGPU_ST_OK;
          } else {
            p.status[rd] = P16_ST_GENERAL;
          }
        }
      } else if (sub == 0 && live) {
        if (ok) {
          p.score[rd] = score;
          p.as_out[rd] = aec - nsteps + ws;
          p.ae_out[rd] = aec + ws;
          p.abr[rd] = L - 1 - nsteps;
          p.n_runs[rd] = 1;
          p.runs[(int64_t)rd * MAX_RUNS] = (uint16_t)((MIAGPU_RUN_M << 14) | (nsteps + 1));
          p.status[rd] = MIAGPU_ST_OK;
        } else {
          // dyn_prog's candidates of a cell all come from lower columns (mia.c:838-871), so the columns to the right of the end cell
          // -- exact here unless sunk -- can reach neither its value nor its path, and being the FIRST maximum of the last row
          // (mia.c:1278-1302) it stays the only one of the narrower window: the 32-bit kernel sweeps [ws, ws + aec] alone
          int wl = len1;
          if (p.win_len_narrow && !sunk) { wl = aec + 1; p.win_len_narrow[rd] = wl; }
          const int b = bucket32_of(wl);
          const int slot = atomicAdd(p.list_counts + b, 1);
          p.lists[(int64_t)b * p.n_reads + slot] = rd;
          atomicAdd(p.n_fallback, 1);
        }
      }
    }
  }
}

}  // namespace miagpu
