// strip.cuh -- general (chunked, maskable) PSSM DP for pass 1 and for windows wider than the
// register-tiled kernels of realign.cuh (sm_100a).
//
// Replaces new_kmer_filter (kmer.c:239-331) + sg_align's compute (mia.c:1500-1610): both
// strands x whole wrapped reference with the forward matrix, masked by the k-mer filter,
// strand pick, traceback, coordinate fix-ups; and the whole-reference fallback of
// reiterate_assembly (mia_main.c:209-212).
//
// Same row-parallel scheme as realign.cuh (a row has no internal dependency), but the columns
// are processed in CHUNKS of CW = 32*K columns: for each chunk the warp runs all L rows, and
// per row hands the next chunk {S[r][last], S[r][last-1], best_gap_col state} through a
// checkpoint array in global memory.  Fully masked chunks are skipped (best_gap_col persists
// across them, exactly like the reference's running variable, H3).  The forward sweep keeps
// no trace; the traceback re-runs only the chunk(s) the path crosses from their checkpoints
// with a full int32 trace (the reference's own encoding, so the trace==0 collision H2 is
// reproduced by construction).  Arg-maxes are (value, index) pairs in plain int32 with the real
// HIM = INT_MIN/2 sentinel: no packing limits, any reference length.
#pragma once
#include "common.cuh"
#include "realign.cuh"

namespace miagpu {

constexpr int SK = 8;                 // columns per lane
constexpr int CW = 32 * SK;           // chunk width
constexpr int KMER_SATURATE = 128;    // params.h:85
constexpr int MAX_KMER_POS = 128;     // params.h:83
constexpr int ALIGN_MASK_BUFFER = 10; // params.h:86

struct KmerTable {                    // one strand; sorted (kmer, pos), <= 128 positions per k-mer
  const int32_t* bucket_start;        // [nbuckets+1]
  const uint32_t* kmer;               // full k-mer index of entry
  const int32_t* pos;
  int32_t bucket_shift;               // bucket = kmer >> bucket_shift
};

struct StripParams {
  const uint8_t* bases;
  const int64_t* off;
  int64_t n;
  int32_t* counter;
  // mode 0: pass 1 (both strands, forward matrix, k-mer masks).  mode 1: single strand, unmasked,
  // explicit work list + per-read strand matrix (wide realign).  mode 2: like 1, but the matrix columns are the read's own
  // window [win_start, win_start + win_len) of the forward strand (the rounds of mia -h, which only this kernel computes)
  int32_t mode;
  const int32_t* win_start;
  const int32_t* win_len;
  // mia -h (strip_kernel<true>): start of the homopolymer every strand column belongs to (pop_hpl_and_hps over the whole wrapped
  // strand, mia_main.c:735-739; a window clips it, mia_main.c:221-224), and one more checkpoint value per row and processed chunk
  const int32_t* hps[2];
  int32_t* ckh;                       // [warp][2][(max_chunks+1)][Lmax]
  const int32_t* list;
  int32_t n_list;
  const int32_t* n_list_ptr;          // nullable: the list's length on the device (mode 0 with a list)
  const uint8_t* rc_in;
  const uint8_t* ref_codes[2];        // forward / reverse-complement strand, wrapped
  int32_t len1;                       // columns (wrap_len if circular else seq_len)
  int32_t seq_len;
  const int32_t* prof;
  int32_t sg5;                        // start-new level of a row (mia.c:877-880): 1 everywhere but miagpu_align_windows(..., sg5 = 0)
  int32_t k;                          // k-mer length, <= 0: no filter
  KmerTable kt[2];
  // per-warp scratch
  uint32_t* mask;                     // [warp][2][mask_words]
  int32_t mask_words;
  int4* ckpt;                         // [warp][2][(max_chunks+1)][Lmax]
  int32_t* chunk_ids;                 // [warp][2][max_chunks]
  int32_t max_chunks;
  int32_t Lmax;
  int32_t* trace;                     // [warp][(Lmax)][CW]
  // outputs
  int32_t *hits, *score, *fw_score, *rc_score, *as_out, *ae_out, *start, *end, *abr, *n_runs;
  uint8_t* rc_out;
  uint16_t* runs;
  uint8_t* status;
};

// mia -h.  The two extra candidates of a cell (mia.c:882-905) need, beyond what a row-parallel sweep holds anyway:
//   column candidate (rows where a read homopolymer starts): S[r-1][hs-1], hs = start of the column's reference homopolymer --
//       any earlier column: the chunk's previous row is kept in shared memory (srow); for the homopolymer that crosses the chunk's
//       left edge the value comes from the previous processed chunk, which recorded that one column for every row (ckh);
//   row candidate (rows inside a read homopolymer that started at row rs): S[rs-1][c-1] -- a snapshot of row rs-1 taken when the
//       homopolymer starts (registers HS), shifted by one column.
// hp_discount_penalty(gap_len, ., hprl) = GEP * gap_len + trunc(GOP * f(hprl)) (mia.c:1096-1134; the row candidate passes the
// COLUMN distance, which is 0 there).
struct HpRow {
  const uint8_t* rch;                 // per row: the read's raw byte as 0..4 (exactly 'A','C','G','T','N') times 4, 28 for anything else
  const uint16_t* hprs;               // per row: first row of its homopolymer (raw bytes compared, mia.c:1193-1234)
  const int32_t* hpg;                 // per row: trunc(GOP * f(length of its homopolymer))
  int32_t* srow;                      // CW ints of the warp: the chunk's previous row
};
struct HpChunk {
  HpRow row;
  const int32_t* hps;                 // indexed by matrix column (already offset by the window start), absolute strand columns
  int32_t clip;                       // absolute strand column of matrix column 0
  const int32_t* ckh_in;              // per row: S[row][hs(c0) - 1], valid when in_valid
  int32_t* ckh_out;                   // per row: S[row][hs(c0 + CW) - 1] for the next processed chunk (nullable)
  bool in_valid;
};
__device__ __forceinline__ int hp_gop_part(int len) {      // trunc(GOP * f): 1000 x {1, .5, .33, .25, .2, .17, .14, .13, .11, .10}, exact in double
  return len <= 1 ? GOP : len == 2 ? 500 : len == 3 ? 330 : len == 4 ? 250 : len == 5 ? 200 : len == 6 ? 170 : len == 7 ? 140 : len == 8 ? 130
       : len == 9 ? 110 : 100;
}
static_assert(GOP == 1000, "hp_gop_part spells out trunc(GOP * f) for GOP = 1000");

struct PV { int v, i; };
__device__ __forceinline__ PV pv_better(PV a, PV b) { return (b.v > a.v) ? b : a; }   // strict '>' keeps the earlier

// One chunk, all rows.  TRACE: also write trace ints for rows 1..L-1 into trace[(r)*CW + cc].
// ck_in: checkpoint of this chunk (per row {S1,S2,PV,PI}); adjacent: S1/S2 valid (previous chunk is c0-CW).
// ck_out: written for the next processed chunk.  Returns via best/best_col the running first-max of the last row.
// PIPE (strip_team_kernel): the previous processed chunk is swept by ANOTHER warp of the block at the same time, one row
// ahead: row r waits until *flag_prev > r (that warp has written its row r candidate state and its row r-1 scores) and
// announces its own progress through *flag_mine.  The hand-over goes through shared memory (ring_in = that warp's
// per-row {S1, S2, PV, PI}, ring_out = mine); the global checkpoints are still written, for the traceback.
template <bool TRACE, bool PIPE = false, bool HP = false>
__device__ void strip_chunk(const int L, const int len1, const int c0, const uint8_t* __restrict__ ref, const uint32_t* __restrict__ mask,
                            const uint16_t* rowoff, const uint32_t prof_base, const int sg5, const int4* ck_in, const bool adjacent, const bool have_in,
                            int4* ck_out, int32_t* trace, int& best, int& best_col, volatile int* flag_prev = nullptr,
                            volatile int* flag_mine = nullptr, volatile int* ring_in = nullptr, volatile int* ring_out = nullptr,
                            const HpChunk* hp = nullptr) {
  static_assert(!(PIPE && HP), "the team schedule does not carry the homopolymer checkpoints");
  const int lane = threadIdx.x & 31;
  const int cbase = c0 + lane * SK;
  int hsj[SK], HS[SK], HS0 = HIM;                   // HP: homopolymer start per column (matrix columns); snapshot of row rs-1
  int tb = -1;                                      // HP: the column the next processed chunk needs from this one, -1 none
  if (HP) {
#pragma unroll
    for (int j = 0; j < SK; j++) {
      const int c = cbase + j;
      hsj[j] = c < len1 ? max(hp->hps[c], hp->clip) - hp->clip : c;
      HS[j] = HIM;
    }
    if (c0 + CW < len1) tb = max(hp->hps[c0 + CW], hp->clip) - hp->clip - 1;
  }
  auto put_ckh = [&](const int r, const int (&Srow)[SK]) {
    if (!HP || !hp->ckh_out || tb < 0) return;
    if (tb >= c0) {
      const int tl = (tb - c0) / SK, tj = (tb - c0) - tl * SK;
      if (lane == tl) {
        int v = Srow[0];
#pragma unroll
        for (int j = 1; j < SK; j++) if (j == tj) v = Srow[j];
        hp->ckh_out[r] = v;
      }
    } else if (lane == 0) hp->ckh_out[r] = hp->in_valid ? hp->ckh_in[r] : HIM;     // one homopolymer covers the whole chunk
  };
  int code4[SK];
  bool mb[SK];
  {
    const uint32_t mword = mask ? __ldcg(mask + (cbase >> 5)) : 0xffffffffu;       // SK = 8 divides 32: one word per lane
#pragma unroll
    for (int j = 0; j < SK; j++) {
      const int c = cbase + j;
      code4[j] = (c < len1 ? ref[c] : 4) * 4;
      mb[j] = c < len1 && ((mword >> ((cbase & 31) + j)) & 1u);
    }
  }
  int Sp[SK], RV[SK], RI[SK];
  {
    const uint32_t pa = prof_base + rowoff[0];
#pragma unroll
    for (int j = 0; j < SK; j++) {
      Sp[j] = mb[j] ? lds_s32(pa + code4[j]) : HIM;                     // mia.c:769-785
      RV[j] = INT_MIN; RI[j] = 0;
    }
  }
  if (ck_out && lane == 31) {
    ck_out[0] = make_int4(Sp[SK - 1], Sp[SK - 2], 0, 0);
    if (PIPE) { ring_out[0] = Sp[SK - 1]; ring_out[1] = Sp[SK - 2]; }
  }
  if (HP) {
    __syncwarp();
#pragma unroll
    for (int j = 0; j < SK; j++) hp->row.srow[lane * SK + j] = Sp[j];
    put_ckh(0, Sp);
    __syncwarp();
  }
  for (int r = 1; r < L; r++) {
    const uint32_t pa = prof_base + rowoff[r];
    const int N = sg5 ? -(GOP + GEP * (r + 1)) : 0;                      // mia.c:877-880
    // left neighbours of this lane's first column in row r-1
    int l1 = __shfl_up_sync(0xffffffffu, Sp[SK - 1], 1);
    int l2 = __shfl_up_sync(0xffffffffu, Sp[SK - 2], 1);
    PV seed;
    if (lane == 0) {
      if (PIPE && have_in) {
        while (*flag_prev <= r) {}
        __threadfence_block();
      }
      int4 ci = make_int4(HIM, HIM, 0, 0);
      if (have_in) {
        if (PIPE) { ci.x = ring_in[4 * (r - 1)]; ci.y = ring_in[4 * (r - 1) + 1]; }
        else ci = ck_in[r - 1];
      }
      l1 = adjacent ? ci.x : HIM;
      l2 = adjacent ? ci.y : HIM;
      // best_gap_col entering this chunk at row r: the previous processed chunk's state, or the row-start
      // state bgc = 0 (mia.c:825) = (S[r-1][0], 0)
      if (c0 == 0) seed = PV{Sp[0], 0};
      else if (have_in) {
        if (PIPE) seed = PV{ring_in[4 * r + 2], ring_in[4 * r + 3]};
        else { int4 cr = ck_in[r]; seed = PV{cr.z, cr.w}; }
      }
      else seed = PV{HIM, 0};
    }
    // candidates: column k = c-2 joins when column c is unmasked and c >= 2 (mia.c:827-843)
    PV cand[SK];
#pragma unroll
    for (int j = 0; j < SK; j++) {
      const int c = cbase + j, k = c - 2;
      const int s = j == 0 ? l2 : j == 1 ? l1 : Sp[j - 2];
      cand[j] = (mb[j] && k >= 0) ? PV{s + GEP * k, k} : PV{INT_MIN, 0};
    }
    PV t = cand[0];
#pragma unroll
    for (int j = 1; j < SK; j++) t = pv_better(t, cand[j]);
    if (lane == 0) t = pv_better(seed, t);                              // seed is earlier than every candidate
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      PV o{__shfl_up_sync(0xffffffffu, t.v, d), __shfl_up_sync(0xffffffffu, t.i, d)};
      if (lane >= d) t = pv_better(o, t);
    }
    PV P{__shfl_up_sync(0xffffffffu, t.v, 1), __shfl_up_sync(0xffffffffu, t.i, 1)};
    if (lane == 0) P = seed;
    if (ck_out && lane == 31) {
      ck_out[r] = make_int4(0, 0, t.v, t.i);                            // S1/S2 patched below
      if (PIPE) {
        ring_out[4 * r + 2] = t.v; ring_out[4 * r + 3] = t.i;
        __threadfence_block();
        *flag_mine = r + 1;                                             // row r-1's scores went out before (program order)
      }
    }

    int D = l1;
    int tr[SK];
    int rs = 0, pg = 0, rcl = 28;
    bool rstart = false;
    if (HP) {
      rs = hp->row.hprs[r]; pg = hp->row.hpg[r]; rcl = hp->row.rch[r];
      rstart = rs == r;
      if (rstart) {                                                      // a read homopolymer starts: keep row r-1 (HS0: the column left of this lane)
#pragma unroll
        for (int j = 0; j < SK; j++) HS[j] = Sp[j];
        HS0 = l1;
      }
    }
#pragma unroll
    for (int j = 0; j < SK; j++) {
      const int c = cbase + j;
      P = pv_better(P, cand[j]);
      int S = HIM, trace_v = 0;
      if (mb[j]) {
        const int sub = lds_s32(pa + code4[j]);
        if (c == 0) {
          S = sub + N;                                                   // mia.c:805-822
        } else {
          const int Gc = c >= 2 ? P.v - (GOP - GEP) - GEP * c : HIM;     // mia.c:838-850
          const int Gr = r >= 2 ? RV[j] - (GOP - GEP) - GEP * r : HIM;   // mia.c:856-868
          int hc = HIM, hr = HIM;                                        // mia.c:882-905
          if (HP && code4[j] == rcl) {                                   // seq1[col] == seq2[row]
            const int hs = hsj[j];
            if (rstart) {
              if (hs != c && hs > 0) {
                const int src = hs - 1;
                const int v = src >= c0 ? hp->row.srow[src - c0] : (hp->in_valid ? hp->ckh_in[r - 1] : HIM);
                hc = v - (GEP * (c - hs) + pg);
              }
            } else if (rs > 0 && hs == c) {
              hr = (j ? HS[j - 1] : HS0) - pg;                           // gap_len = col - hpcs[col] = 0, as written
            }
          }
          if (N > D && N > Gc && N > Gr && N > hc && N > hr) { S = N; trace_v = c; }         // mia.c:910-918
          else if (D >= Gc && D >= Gr && D >= hc && D >= hr) { S = sub + D; trace_v = 0; }
          else if (Gc >= Gr && Gc >= hc && Gc >= hr) { S = sub + Gc; trace_v = P.i; }
          else if (Gr >= hc && Gr >= hr) { S = sub + Gr; trace_v = -RI[j]; }
          else if (hc >= hr) { S = sub + hc; trace_v = hsj[j] - 1; }                         // mia.c:950-955
          else { S = sub + hr; trace_v = -(rs - 1); }                                        // mia.c:956-961
          // row r-1 joins best_gap_row[c-1] (used from row r+1 on)
          const int cv = D + GEP * (r - 1);
          if (cv > RV[j]) { RV[j] = cv; RI[j] = r - 1; }
        }
      }
      tr[j] = trace_v;
      D = Sp[j];
      Sp[j] = S;
    }
    if (ck_out && lane == 31) {
      ck_out[r].x = Sp[SK - 1]; ck_out[r].y = Sp[SK - 2];
      if (PIPE) { ring_out[4 * r] = Sp[SK - 1]; ring_out[4 * r + 1] = Sp[SK - 2]; }
    }
    if (TRACE) {
      int4* trow = reinterpret_cast<int4*>(trace + (int64_t)r * CW + lane * SK);
      trow[0] = make_int4(tr[0], tr[1], tr[2], tr[3]);
      trow[1] = make_int4(tr[4], tr[5], tr[6], tr[7]);
    }
    if (HP) {
      __syncwarp();                                                      // every lane has read row r-1
#pragma unroll
      for (int j = 0; j < SK; j++) hp->row.srow[lane * SK + j] = Sp[j];
      put_ckh(r, Sp);
      __syncwarp();
    }
  }
  // max_sg_score over this chunk's columns (mia.c:1293-1299): strict '>' in column order
  int lb = INT_MIN, lc = 0;
#pragma unroll
  for (int j = 0; j < SK; j++) {
    const int c = cbase + j;
    if (c < len1 && Sp[j] > lb) { lb = Sp[j]; lc = c; }
  }
  const int wb = __reduce_max_sync(0xffffffffu, lb);
  const int wc = __reduce_min_sync(0xffffffffu, lb == wb ? lc : 0x7fffffff);
  if (wb > best) { best = wb; best_col = wc; }
}

__device__ __forceinline__ int kmer_code(uint8_t b) {                   // kmer2inx upper-cases (kmer.c:27)
  if (b >= 'a' && b <= 'z') b -= 32;
  return b == 'A' ? 0 : b == 'C' ? 1 : b == 'G' ? 2 : b == 'T' ? 3 : -1;
}

// new_kmer_filter for one strand: sets mask bits, returns the hit count (kmer.c:275-327)
__device__ int seed_strand(const KmerTable& kt, const int k, const uint8_t* read, const int L, const int len1, const int strand,
                           uint32_t* mask, const int mask_words) {
  const int lane = threadIdx.x & 31;
  int hits = 0;
  for (int p = lane; p + k <= L; p += 32) {
    uint32_t inx = 0;
    bool ok = true;
    for (int i = 0; i < k; i++) {
      const int c = kmer_code(read[p + i]);
      if (c < 0) { ok = false; break; }
      inx = (inx << 2) | (uint32_t)c;
    }
    if (!ok) continue;
    const int b = (int)(inx >> kt.bucket_shift);
    for (int e = kt.bucket_start[b]; e < kt.bucket_start[b + 1]; e++) {
      if (kt.kmer[e] != inx) continue;
      hits++;
      const int q = kt.pos[e];
      int lo = q - p - ALIGN_MASK_BUFFER;
      int hi = q + (L - p) + ALIGN_MASK_BUFFER - strand;                // rc bound is one shorter: kmer.c:294 vs 319
      if (lo < 0) lo = 0;
      if (hi >= len1) hi = len1 - 1;
      for (int w = lo >> 5; w <= (hi >> 5); w++) {
        const int a = max(lo, w << 5) & 31, z = min(hi, (w << 5) + 31) & 31;
        atomicOr(mask + w, (0xffffffffu >> (31 - z)) & (0xffffffffu << a));
      }
    }
  }
  hits = __reduce_add_sync(0xffffffffu, hits);
  if (hits >= KMER_SATURATE) {                                           // kmer.c:283-285
    __syncwarp();
    for (int w = lane; w < mask_words; w += 32) mask[w] = 0xffffffffu;
  }
  return hits;
}

// mia -h: what processed chunk q of a strand takes from / leaves to its neighbours (uniform over the warp)
__device__ __forceinline__ HpChunk hp_chunk(const StripParams& p, const HpRow& row, const int s, const int ws, const int len1, const int32_t* ids,
                                            const int q, int32_t* ckh, const bool want_out) {
  HpChunk h;
  h.row = row; h.hps = p.hps[s] + ws; h.clip = ws;
  const int c0 = ids[q] * CW;
  const int hs0 = max(h.hps[c0], ws) - ws;
  h.in_valid = false;
  if (q > 0 && hs0 < c0) {                            // the first column's homopolymer began before the chunk: did the previous processed chunk record it?
    const int pb = (ids[q - 1] + 1) * CW;             // that chunk recorded column hs(pb) - 1
    h.in_valid = pb < len1 && max(h.hps[pb], ws) - ws == hs0;
  }
  h.ckh_in = ckh + (int64_t)q * p.Lmax;
  h.ckh_out = want_out ? ckh + (int64_t)(q + 1) * p.Lmax : nullptr;
  return h;
}

// One warp: strand pick, traceback (re-running the chunks the path crosses from their checkpoints) and the outputs of read rd.
// len1 / ws: the matrix columns of this read (the whole strand, or its window in mode 2).
template <bool HP = false>
__device__ void strip_finish(const StripParams& p, const int rd, const int L, const int nstrand, const bool masked, const int (&best)[2],
                             const int (&bcol)[2], const int (&nch)[2], const uint32_t* mask0, const int32_t* ids0, const int4* ck0,
                             int32_t* trace, const uint16_t* rowoff, const uint32_t prof_base, const int len1, const int ws = 0,
                             const HpRow* hprow = nullptr, int32_t* ckh0 = nullptr) {
  const int lane = threadIdx.x & 31;
  // ---- strand pick: fw only if strictly better (mia.c:1549-1554)
  const int s = (nstrand == 2 && !(best[0] > best[1])) ? 1 : 0;
  const int score = best[s];
  const int aec = bcol[s];
  // ---- traceback: re-run the chunks the path crosses, with trace
  const uint32_t* mask = masked ? mask0 + s * p.mask_words : nullptr;
  const int32_t* ids = ids0 + s * p.max_chunks;
  const int4* ck = ck0 + (int64_t)s * (p.max_chunks + 1) * p.Lmax;
  int row = L - 1, col = aec, nrun = 0, curM = 0, ncols = 0, loaded = -1;
  uint16_t* my_runs = p.runs + (int64_t)rd * MAX_RUNS;
  auto push = [&](int type, int len) {
    while (len > 0) {                                                  // a run longer than 14 bits is split
      const int l = min(len, 0x3fff);
      if (nrun < MAX_RUNS && lane == 0) my_runs[nrun] = (uint16_t)((type << 14) | l);
      nrun++; len -= l;
    }
  };
  bool lost = false;
  while (row > 0 && col > 0) {
    const int ch = col / CW;
    if (ch != loaded) {
      int q = -1;                                                      // position of chunk ch in the processed list
      for (int base = 0; base < nch[s]; base += 32) {
        const bool hit = base + lane < nch[s] && ids[base + lane] == ch;
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (bal) { q = base + __ffs(bal) - 1; break; }
      }
      if (q < 0) { lost = true; break; }                               // cannot happen: the path only visits unmasked cells
      int dummy_b = INT_MIN, dummy_c = 0;
      __syncwarp();
      if (HP) {
        const HpChunk h = hp_chunk(p, *hprow, s, ws, len1, ids, q, ckh0 + (int64_t)s * (p.max_chunks + 1) * p.Lmax, false);
        strip_chunk<true, false, true>(L, len1, ch * CW, p.ref_codes[s] + ws, mask, rowoff, prof_base, p.sg5, ck + (int64_t)q * p.Lmax,
                                       q > 0 && ids[q - 1] == ch - 1, q > 0, nullptr, trace, dummy_b, dummy_c, nullptr, nullptr, nullptr, nullptr, &h);
      } else {
        strip_chunk<true>(L, len1, ch * CW, p.ref_codes[s] + ws, mask, rowoff, prof_base, p.sg5, ck + (int64_t)q * p.Lmax,
                          q > 0 && ids[q - 1] == ch - 1, q > 0, nullptr, trace, dummy_b, dummy_c);
      }
      __syncwarp();
      loaded = ch;
    }
    const int t = __ldcg(trace + (int64_t)row * CW + (col - ch * CW));
    if (t == col || t == -row) break;                                  // mia.c:617-618
    curM++;
    if (t == 0) { row--; col--; }
    else if (t < 0) { push(MIAGPU_RUN_M, curM); ncols += curM; curM = 0; push(MIAGPU_RUN_I, row - 1 + t); ncols += row - 1 + t; row = -t; col--; }
    else { push(MIAGPU_RUN_M, curM); ncols += curM; curM = 0; push(MIAGPU_RUN_D, col - 1 - t); ncols += col - 1 - t; col = t; row--; }
  }
  push(MIAGPU_RUN_M, curM + 1); ncols += curM + 1;
  if (lane == 0) {
    uint8_t st = lost ? MIAGPU_ST_UNSUPPORTED : MIAGPU_ST_OK;
    if (nrun > MAX_RUNS) { st |= MIAGPU_ST_RUNS_OVERFLOW; nrun = -1; }
    if (ncols > 2 * MAX_READ) st |= MIAGPU_ST_STR_OVERFLOW;
    const int abc = col, abr = row;
    if (p.mode == 0) {
      // sg_align's coordinates (mia.c:1568-1610); runs go out in forward-reference orientation
      int start = abc, end = aec;
      if (s == 1) {                                                     // c2rcc, mia.c:26-30; revcom_PWAF reverses the columns
        start = p.seq_len - (aec % p.seq_len) - 1;
        end = p.seq_len - (abc % p.seq_len) - 1;
      } else {
        for (int a = 0, b = nrun - 1; a < b; a++, b--) { uint16_t x = my_runs[a]; my_runs[a] = my_runs[b]; my_runs[b] = x; }
      }
      int as = start, ae = end;
      if (as > ae) ae = p.seq_len + as;                                 // mia.c:1600-1604
      if (end > p.seq_len) end -= p.seq_len;                            // mia.c:1606-1610
      p.as_out[rd] = as; p.ae_out[rd] = ae; p.start[rd] = start; p.end[rd] = end;
      p.rc_out[rd] = (uint8_t)s;
      p.fw_score[rd] = best[0]; p.rc_score[rd] = best[1];
      p.abr[rd] = s == 1 ? 0 : abr;                                     // row of the returned runs' first base in the STORED orientation
    } else {
      for (int a = 0, b = nrun - 1; a < b; a++, b--) { uint16_t x = my_runs[a]; my_runs[a] = my_runs[b]; my_runs[b] = x; }
      p.as_out[rd] = abc + ws; p.ae_out[rd] = aec + ws;                 // mia_main.c:250-255 (ws = 0 for the whole reference, 209-212)
      p.abr[rd] = abr;
    }
    p.score[rd] = score;
    p.n_runs[rd] = nrun;
    p.status[rd] = st;
  }
}

// dynamic smem: [prof PROF_INTS ints][rowoff WARPS*256 u16]; HP: + per warp [srow CW ints][hpg 256 ints][hprs 256 u16][rch 256 u8]
constexpr int STRIP_HP_SMEM_PER_WARP = CW * 4 + MAX_READ * 4 + MAX_READ * 2 + MAX_READ;
template <bool HP = false>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) strip_kernel(StripParams p) {
  extern __shared__ __align__(16) uint8_t smem[];
  int32_t* s_prof = reinterpret_cast<int32_t*>(smem);
  uint16_t* s_rowoff = reinterpret_cast<uint16_t*>(smem + PROF_INTS * 4);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < PROF_INTS; i += blockDim.x) s_prof[i] = p.prof[i];
  __syncthreads();
  uint16_t* rowoff = s_rowoff + warp * MAX_READ;
  HpRow hprow{};
  if (HP) {
    uint8_t* base = smem + PROF_INTS * 4 + WARPS_PER_BLOCK * MAX_READ * 2 + (size_t)warp * STRIP_HP_SMEM_PER_WARP;
    hprow.srow = reinterpret_cast<int32_t*>(base);
    hprow.hpg = reinterpret_cast<int32_t*>(base + CW * 4);
    hprow.hprs = reinterpret_cast<uint16_t*>(base + CW * 4 + MAX_READ * 4);
    hprow.rch = base + CW * 4 + MAX_READ * 4 + MAX_READ * 2;
  }
  const uint32_t prof_base = smem_u32(s_prof);
  const int64_t gw = (int64_t)blockIdx.x * WARPS_PER_BLOCK + warp;
  uint32_t* mask0 = p.mask + gw * 2 * p.mask_words;
  int4* ck0 = p.ckpt + gw * 2 * (int64_t)(p.max_chunks + 1) * p.Lmax;
  int32_t* ids0 = p.chunk_ids + gw * 2 * p.max_chunks;
  int32_t* trace = p.trace + gw * (int64_t)p.Lmax * CW;
  int32_t* ckh0 = HP ? p.ckh + gw * 2 * (int64_t)(p.max_chunks + 1) * p.Lmax : nullptr;
  const int total = p.n_list_ptr ? *p.n_list_ptr : (p.mode == 0 && !p.list) ? (int)p.n : p.n_list;

  for (;;) {
    int item = 0;
    if (lane == 0) item = atomicAdd(p.counter, 1);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= total) break;
    const int rd = p.list ? p.list[item] : item;
    const int64_t o0 = p.off[rd];
    const int L = (int)(p.off[rd + 1] - o0);
    const uint8_t* read = p.bases + o0;
    const int ws = p.mode == 2 ? p.win_start[rd] : 0;                    // the matrix columns: the whole strand, or the read's window
    const int len1 = p.mode == 2 ? p.win_len[rd] : p.len1;
    if (L <= 0 || L > MAX_READ) {
      if (lane == 0) { p.status[rd] = MIAGPU_ST_UNSUPPORTED; p.n_runs[rd] = -1; p.score[rd] = INT_MIN; if (p.hits) p.hits[rd] = 0; }
      continue;
    }
    const int nstrand = p.mode == 0 ? 2 : 1;
    const int mat = p.mode == 0 ? 0 : (p.rc_in[rd] ? 1 : 0);             // pass 1 scores BOTH strands with the forward matrix (H5)
    __syncwarp();
    for (int r = lane; r < L; r += 32) rowoff[r] = (uint16_t)(prof_row_index(mat, sm_depth(r, L), base_code(read[r])) * 4);
    if (HP) {                                                            // pop_hpl_and_hps over the read (mia.c:1527-1531 / mia_main.c:222)
      uint8_t* rch = const_cast<uint8_t*>(hprow.rch);
      uint16_t* hprs = const_cast<uint16_t*>(hprow.hprs);
      int32_t* hpg = const_cast<int32_t*>(hprow.hpg);
      for (int r = lane; r < L; r += 32) {
        const uint8_t b = read[r];
        rch[r] = (uint8_t)(b == 'A' ? 0 : b == 'C' ? 4 : b == 'G' ? 8 : b == 'T' ? 12 : b == 'N' ? 16 : 28);
      }
      if (lane == 0) {
        int start = 0;
        for (int r = 1; r <= L; r++)
          if (r == L || read[r] != read[r - 1]) {
            const int g = hp_gop_part(r - start);
            for (int q = start; q < r; q++) { hprs[q] = (uint16_t)start; hpg[q] = g; }
            start = r;
          }
      }
      __syncwarp();
    }
    // ---- k-mer filter
    int hits[2] = {1, 0};
    const bool masked = p.mode == 0 && p.k > 0;
    if (masked) {
      for (int w = lane; w < 2 * p.mask_words; w += 32) mask0[w] = 0;
      __syncwarp();
      hits[0] = hits[1] = 0;
      if (L >= p.k) {
        hits[0] = seed_strand(p.kt[0], p.k, read, L, len1, 0, mask0, p.mask_words);
        hits[1] = seed_strand(p.kt[1], p.k, read, L, len1, 1, mask0 + p.mask_words, p.mask_words);
      }
      __syncwarp();
    }
    if (p.hits && lane == 0) p.hits[rd] = hits[0] + hits[1];
    if (masked && hits[0] + hits[1] == 0) {                              // mia_main.c:781: the read is not aligned at all
      if (lane == 0) { p.status[rd] = MIAGPU_ST_SKIPPED; p.n_runs[rd] = 0; p.score[rd] = INT_MIN; }
      continue;
    }
    // ---- forward sweeps
    int best[2] = {INT_MIN, INT_MIN}, bcol[2] = {0, 0}, nch[2] = {0, 0};
    const int n_chunks_all = (len1 + CW - 1) / CW;
    for (int s = 0; s < nstrand; s++) {
      const uint32_t* mask = masked ? mask0 + s * p.mask_words : nullptr;
      int32_t* ids = ids0 + s * p.max_chunks;
      int4* ck = ck0 + (int64_t)s * (p.max_chunks + 1) * p.Lmax;
      // chunk list: chunks with at least one unmasked column
      int n = 0;
      for (int base = 0; base < n_chunks_all; base += 32) {
        const int ch = base + lane;
        bool any = false;
        if (ch < n_chunks_all) {
          if (!mask) any = true;
          else for (int w = 0; w < CW / 32; w++) { const int wi = ch * (CW / 32) + w; if (wi < p.mask_words && __ldcg(mask + wi)) any = true; }
        }
        const unsigned bal = __ballot_sync(0xffffffffu, any);
        if (any) ids[n + __popc(bal & ((1u << lane) - 1))] = ch;
        n += __popc(bal);
      }
      __syncwarp();
      nch[s] = n;
      // the reference's scan starts at column 0: S[L-1][0] (HIM if masked) is the first incumbent
      best[s] = HIM; bcol[s] = 0;
      int prev = -2;
      for (int q = 0; q < n; q++) {
        const int ch = ids[q];
        if (HP) {
          const HpChunk h = hp_chunk(p, hprow, s, ws, len1, ids, q, ckh0 + (int64_t)s * (p.max_chunks + 1) * p.Lmax, true);
          strip_chunk<false, false, true>(L, len1, ch * CW, p.ref_codes[s] + ws, mask, rowoff, prof_base, p.sg5, ck + (int64_t)q * p.Lmax, prev == ch - 1,
                                          q > 0, ck + (int64_t)(q + 1) * p.Lmax, nullptr, best[s], bcol[s], nullptr, nullptr, nullptr, nullptr, &h);
        } else {
          strip_chunk<false>(L, len1, ch * CW, p.ref_codes[s] + ws, mask, rowoff, prof_base, p.sg5, ck + (int64_t)q * p.Lmax, prev == ch - 1, q > 0,
                             ck + (int64_t)(q + 1) * p.Lmax, nullptr, best[s], bcol[s]);
        }
        prev = ch;
        __syncwarp();
      }
    }
    strip_finish<HP>(p, rd, L, nstrand, masked, best, bcol, nch, mask0, ids0, ck0, trace, rowoff, prof_base, len1, ws, &hprow, ckh0);
  }
}

// The same for FEW reads with MANY chunks to sweep (a strand the k-mer filter saturated, an unmasked strand, a wide
// realign window): a block of TEAM_WARPS warps takes one read; warp w sweeps processed chunks w, w + TEAM_WARPS, ...,
// each one row behind the warp that holds the chunk to its left (strip_chunk's PIPE mode: row r of a chunk needs only
// row r-1 / the row-r candidate state of the chunks before it).  L + chunks/TEAM_WARPS row steps instead of L * chunks.
// A warp alternates between two rings from one of its chunks to the next: when it re-uses a ring (two chunks later, 2 *
// TEAM_WARPS chunks further right) its own previous chunk is finished, hence -- every chunk trails its left neighbour --
// so is the reader of the ring's old content, which the next warp swept before ITS previous chunk.
// dynamic smem: [prof PROF_INTS ints][rowoff 256 u16][flags max_chunks ints][rings 2 x TEAM_WARPS x Lmax x 4 ints]
constexpr int TEAM_WARPS = 16;
__global__ void __launch_bounds__(TEAM_WARPS * 32) strip_team_kernel(StripParams p) {
  extern __shared__ __align__(16) uint8_t smem[];
  int32_t* s_prof = reinterpret_cast<int32_t*>(smem);
  uint16_t* rowoff = reinterpret_cast<uint16_t*>(smem + PROF_INTS * 4);
  volatile int* s_flag = reinterpret_cast<volatile int*>(smem + PROF_INTS * 4 + MAX_READ * 2);
  volatile int* s_ring = s_flag + ((p.max_chunks + 3) & ~3);
  __shared__ int s_item, s_hits[2], s_n, s_wb[TEAM_WARPS], s_wc[TEAM_WARPS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < PROF_INTS; i += blockDim.x) s_prof[i] = p.prof[i];
  __syncthreads();
  const uint32_t prof_base = smem_u32(s_prof);
  const int64_t gw = blockIdx.x;
  uint32_t* mask0 = p.mask + gw * 2 * p.mask_words;
  int4* ck0 = p.ckpt + gw * 2 * (int64_t)(p.max_chunks + 1) * p.Lmax;
  int32_t* ids0 = p.chunk_ids + gw * 2 * p.max_chunks;
  int32_t* trace = p.trace + gw * (int64_t)p.Lmax * CW;
  const int total = p.n_list_ptr ? *p.n_list_ptr : (p.mode == 0 && !p.list) ? (int)p.n : p.n_list;

  for (;;) {
    __syncthreads();
    if (tid == 0) s_item = atomicAdd(p.counter, 1);
    __syncthreads();
    const int item = s_item;
    if (item >= total) break;
    const int rd = p.list ? p.list[item] : item;
    const int64_t o0 = p.off[rd];
    const int L = (int)(p.off[rd + 1] - o0);
    const uint8_t* read = p.bases + o0;
    const int ws = p.mode == 2 ? p.win_start[rd] : 0;                    // the matrix columns: the whole strand, or the read's window
    const int len1 = p.mode == 2 ? p.win_len[rd] : p.len1;
    const int n_chunks_all = (len1 + CW - 1) / CW;
    if (L <= 0 || L > MAX_READ) {
      if (tid == 0) { p.status[rd] = MIAGPU_ST_UNSUPPORTED; p.n_runs[rd] = -1; p.score[rd] = INT_MIN; if (p.hits) p.hits[rd] = 0; }
      continue;
    }
    const int nstrand = p.mode == 0 ? 2 : 1;
    const int mat = p.mode == 0 ? 0 : (p.rc_in[rd] ? 1 : 0);             // pass 1 scores BOTH strands with the forward matrix (H5)
    for (int r = tid; r < L; r += blockDim.x) rowoff[r] = (uint16_t)(prof_row_index(mat, sm_depth(r, L), base_code(read[r])) * 4);
    const bool masked = p.mode == 0 && p.k > 0;
    if (masked) {
      for (int w = tid; w < 2 * p.mask_words; w += blockDim.x) mask0[w] = 0;
      __syncthreads();
      if (warp == 0) {
        int h0 = 0, h1 = 0;
        if (L >= p.k) {
          h0 = seed_strand(p.kt[0], p.k, read, L, len1, 0, mask0, p.mask_words);
          h1 = seed_strand(p.kt[1], p.k, read, L, len1, 1, mask0 + p.mask_words, p.mask_words);
        }
        if (lane == 0) { s_hits[0] = h0; s_hits[1] = h1; }
      }
    } else if (tid == 0) { s_hits[0] = 1; s_hits[1] = 0; }
    __syncthreads();
    const int hits[2] = {s_hits[0], s_hits[1]};
    if (p.hits && tid == 0) p.hits[rd] = hits[0] + hits[1];
    if (masked && hits[0] + hits[1] == 0) {                              // mia_main.c:781: the read is not aligned at all
      if (tid == 0) { p.status[rd] = MIAGPU_ST_SKIPPED; p.n_runs[rd] = 0; p.score[rd] = INT_MIN; }
      continue;
    }
    int best[2] = {INT_MIN, INT_MIN}, bcol[2] = {0, 0}, nch[2] = {0, 0};
    for (int s = 0; s < nstrand; s++) {
      const uint32_t* mask = masked ? mask0 + s * p.mask_words : nullptr;
      int32_t* ids = ids0 + s * p.max_chunks;
      int4* ck = ck0 + (int64_t)s * (p.max_chunks + 1) * p.Lmax;
      if (warp == 0) {                                                   // chunk list: chunks with at least one unmasked column
        int n = 0;
        for (int base = 0; base < n_chunks_all; base += 32) {
          const int ch = base + lane;
          bool any = false;
          if (ch < n_chunks_all) {
            if (!mask) any = true;
            else for (int w = 0; w < CW / 32; w++) { const int wi = ch * (CW / 32) + w; if (wi < p.mask_words && __ldcg(mask + wi)) any = true; }
          }
          const unsigned bal = __ballot_sync(0xffffffffu, any);
          if (any) ids[n + __popc(bal & ((1u << lane) - 1))] = ch;
          n += __popc(bal);
        }
        if (lane == 0) s_n = n;
      }
      for (int q = tid; q < n_chunks_all; q += blockDim.x) s_flag[q] = 0;
      __syncthreads();
      const int n = s_n;
      nch[s] = n;
      int wb = INT_MIN, wc = 0x7fffffff;
      for (int q = warp; q < n; q += TEAM_WARPS) {
        const int ch = ids[q];
        strip_chunk<false, true>(L, len1, ch * CW, p.ref_codes[s] + ws, mask, rowoff, prof_base, p.sg5, ck + (int64_t)q * p.Lmax,
                                 q > 0 && ids[q - 1] == ch - 1, q > 0, ck + (int64_t)(q + 1) * p.Lmax, nullptr, wb, wc,
                                 q > 0 ? s_flag + (q - 1) : nullptr, s_flag + q,
                                 s_ring + (size_t)((((q - 1) / TEAM_WARPS) & 1) * TEAM_WARPS + (q + TEAM_WARPS - 1) % TEAM_WARPS) * p.Lmax * 4,
                                 s_ring + (size_t)(((q / TEAM_WARPS) & 1) * TEAM_WARPS + warp) * p.Lmax * 4);
        __syncwarp();
      }
      if (lane == 0) { s_wb[warp] = wb; s_wc[warp] = wc; }
      __syncthreads();
      // the reference's scan starts at column 0: S[L-1][0] (HIM if masked) is the first incumbent; first maximum in column order
      int b = HIM, bc = 0;
      for (int w = 0; w < TEAM_WARPS; w++)
        if (s_wb[w] > b || (s_wb[w] == b && s_wc[w] < bc)) { b = s_wb[w]; bc = s_wc[w]; }
      best[s] = b; bcol[s] = bc;
      __syncthreads();
    }
    if (warp == 0) strip_finish(p, rd, L, nstrand, masked, best, bcol, nch, mask0, ids0, ck0, trace, rowoff, prof_base, len1, ws);
  }
}

}  // namespace miagpu
