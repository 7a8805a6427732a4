// miagpu.cu -- C ABI (include/miagpu.h) + host orchestration for libmiagpu.so.
// sm_100a only; no CPU fallback: every compute entry point needs a CUDA device.
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>

#include <algorithm>
#include <functional>
#include <chrono>
#include <thread>
#include <vector>

#include "common.cuh"
#include "realign.cuh"
#include "pair16.cuh"
#include "consensus.cuh"
#include "strip.cuh"
#include "pass1.cuh"
#include "sweep16.cuh"
#include "scorecut.hpp"
#include "scorecut.cuh"
#include "repeat.cuh"
#include "slots.cuh"
#include <unordered_map>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_radix_sort.cuh>

namespace miagpu {

static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ------------------------------------------------------------------ buffers
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;
  int reserve(size_t n) {
    if (n <= cap) return 1;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = n + n / 8 + 64;
    MIAGPU_CUDA(cudaMalloc(&p, want * sizeof(T)));
    cap = want;
    return 1;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

constexpr int NBUCKET = 10;                                  // 9 register-tiled widths + "big"
static const int BUCKET_K[NBUCKET] = {2, 4, 5, 6, 7, 8, 10, 12, 16, 0};
constexpr int P16_COLS[P16_NKB] = {128, 144, 160, 176, 192, 208, 224, 256, 64, 80, 96, 112};   // columns of the pair kernels' width classes

constexpr int MAX_CHUNKS = 16;
constexpr int MAX_DEVICES = 64;

}  // namespace miagpu

using namespace miagpu;

// The score-cut policy of a whole round (miagpu_iterate_* or miagpu_shard_begin* .. _finish) and where its reads came from
struct RoundPolicy {
  int hard_cut = 0, score_cut_set = 0;          // -H, or a cut the caller gave (-S -N)
  double slope = 0, intercept = 0;
  bool unique_best = false;                     // the repeat filter's unique_best takes part in the cut
  int host_chunks = 0;                          // > 0: the reads came from the host in that many chunks (host_round_front)
  bool fit() const { return !score_cut_set && hard_cut <= 0; }
  bool host_fed() const { return host_chunks > 0; }
};

struct miagpu_ctx {
  int device = 0;
  int num_sms = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[8] = {};
  cudaEvent_t p1ev[3] = {};                    // pass-1 fast path: after seeding, after the pair kernels, after the merge
  bool p1ev_valid = false;
  cudaEvent_t bev[2 * NBUCKET] = {};           // per width-bucket start/stop
  float bucket_ms[NBUCKET] = {};
  int64_t bucket_cells[NBUCKET] = {};
  int32_t bucket_reads[NBUCKET] = {};
  // scoring
  bool have_pssm = false;
  int32_t sm_f[MIAGPU_PSSM_INTS], sm_r[MIAGPU_PSSM_INTS];
  DevBuf<int32_t> d_prof;
  // reference
  bool have_ref = false;
  std::string raw_wrapped, raw_rc_wrapped;     // case preserved (k-mer soft mask)
  int seq_len = 0, wrap_len = 0, circular = 0, with_rc = 0;
  int64_t cut_prev_newly = -1;                       // reads the previous one-call round's cut dropped (-1: unknown)
  int64_t cons_capacity = 0;                         // bytes behind the caller's cons_out (0 = the header's default)
  bool explicit_windows = false;   // miagpu_align_windows: d_as / d_ae hold [start, end) of every read's window, no window rule
  int explicit_sg5 = 1;
  DevBuf<uint8_t> d_ref, d_rcref, d_ref2;      // codes 0..4, padded to 16 B; d_ref2 = both strands back to back
  int ref_bytes = 0;
  // reads
  int64_t n = 0, total_bases = 0;
  DevBuf<uint8_t> d_bases;
  DevBuf<int64_t> d_off;
  // per-read
  DevBuf<uint8_t> d_rc, d_status;
  DevBuf<int32_t> d_as, d_ae, d_score, d_as_out, d_ae_out, d_abr, d_nruns, d_win_start, d_win_len, d_lists;
  DevBuf<uint16_t> d_runs;
  DevBuf<int32_t> d_meta;                      // META_* layout below
  DevBuf<uint32_t> d_scratch[4];               // trace scratch of the 32-bit kernels, one per launch stream
  DevBuf<int32_t> d_p1trace;                   // pass 1: winning jobs the 32-bit JOB kernels trace
  DevBuf<int32_t> d_sw_jobs, d_sw_layout, d_sw_pairs;   // pass 1: whole-strand jobs of sweep16_kernel, their work items
  DevBuf<int32_t> d_p1sunk;                    // pass 1: jobs that left the 16-bit frame
  int p1_traced = 0, p1_swept = 0;
  // mia -h (miagpu_set_homopolymer): every DP runs in the chunked kernel with the two homopolymer-discounted gap candidates
  bool hp = false, hps_valid = false;
  DevBuf<int32_t> d_hps[2];                    // start of the homopolymer of every (wrapped) strand column
  DevBuf<int32_t> d_ckh;                       // one more checkpoint value per row and processed chunk (strip.cuh)
  cudaStream_t s_aux[4] = {};                  // [0] = stream; [1..3] side streams of the concurrent DP launches
  cudaEvent_t aev[8] = {};                     // fork / join events of those
  cudaStream_t launch_stream = nullptr;        // where launch_realign / launch_pair16 / launch_strip put their kernel
  int launch_slot = 0;
  // 16-bit SIMD pair kernel (pair16.cuh)
  DevBuf<int16_t> d_prof16;
  DevBuf<uint8_t> d_kind;
  DevBuf<int32_t> d_pairs;
  int pssm_min = 0, pssm_max = 0, lmax16 = 0;
  cudaEvent_t pev[2 * P16_NKB] = {};
  float pair_ms[P16_NKB] = {};
  int32_t pair_reads[P16_NKB] = {}, pair_pairs[P16_NKB] = {};
  int64_t pair_cells[P16_NKB] = {};
  int32_t n_fallback = 0;
  // chunked pipeline of miagpu_iterate_host: upload / download streams, per-chunk events, pinned meta copies
  cudaStream_t s_up = nullptr, s_down = nullptr;
  cudaEvent_t cev[4 * 16] = {};                 // [MAX_CHUNKS][4]: classified, realigned, scores on host, spare
  cudaEvent_t xev[4] = {};
  int32_t* h_meta = nullptr;                    // pinned, MAX_CHUNKS * META_HOST
  // device score cut (scorecut.cuh): seq_len / unique_best copies, integer sums, tables, thresholds, chain blocks
  DevBuf<int32_t> d_seqlen;
  DevBuf<uint8_t> d_unique;
  DevBuf<CutStatsDev> d_cstats;
  DevBuf<CutTables> d_ctab;
  DevBuf<double> d_thr;
  DevBuf<CutBlockDev> d_cblk;
  struct CutHost* h_cut = nullptr;              // pinned
  CutBlockDev* h_cblk = nullptr;                // pinned
  int64_t h_cblk_cap = 0;
  char* h_call = nullptr;                       // pinned staging of miagpu_call
  size_t h_call_cap = 0;
  int32_t* h_score = nullptr;                   // pinned copy of the scores (resident rounds)
  int64_t h_score_cap = 0;
  std::vector<int32_t> h_seqlen;                // host copies for the chains' unproven blocks (resident rounds)
  std::vector<uint8_t> h_unique;
  int64_t cut_inputs_n = -1;
  int64_t cut_serial_blocks = 0;                // chain blocks the last round summed read by read on the host
  // adapter trimming
  DevBuf<int32_t> tr_prof, tr_ws, tr_wl, tr_out, tr_cnt;
  DevBuf<uint8_t> tr_codes, tr_ad, tr_st;
  // repeat filter (repeat.cuh)
  DevBuf<uint8_t> rf_rc, rf_tr, rf_uq, rf_tmp;
  DevBuf<int32_t> rf_as, rf_ae, rf_k4, rf_idx, rf_idx2;
  DevBuf<uint64_t> rf_key, rf_key2;
  DevBuf<int64_t> rf_ord;
  DevBuf<int> rf_bad;
  RoundPolicy round;                            // the round in flight (one-GPU and sharded)
  // sharded rounds (SURVEY 8e): this rank's part of the all-gather, what came back
  int sh_world = 0, sh_rank = 0, sh_phase = 0;
  int64_t sh_stride = 0;
  DevBuf<uint32_t> d_sh_send, d_sh_recv;
  DevBuf<ShardPrep> d_sh_prep;
  int64_t sh_nb = 0;
  uint32_t* h_sh_recv = nullptr;                // pinned: what the all-gather of the block records brought
  size_t h_sh_cap = 0;
  // pass 1 / wide windows
  int kmer_k = 0;
  DevBuf<int32_t> d_kb[2], d_kp[2];
  DevBuf<uint32_t> d_kk[2];
  int kmer_shift[2] = {0, 0};
  int max_read_len = 0;
  DevBuf<uint32_t> d_smask;
  DevBuf<int4> d_ckpt;
  DevBuf<int32_t> d_chunk_ids, d_strace, d_hits, d_fw, d_rcs, d_start, d_end;
  DevBuf<uint8_t> d_rc_out, d_bases2;
  // pass-1 fast path (pass1.cuh): per job (8 slots per read: strand x stretch) inputs / outputs, per read route, general-kernel list
  DevBuf<uint8_t> d_jkind, d_jstatus, d_route;
  DevBuf<int32_t> d_jws, d_jwl, d_jscore, d_jabc, d_jaec, d_jabr, d_p1list, d_p1meta, d_jpairs, d_jread, d_jfirst;
  DevBuf<uint16_t> d_jcount;
  int64_t p1_fast = 0, p1_general = 0, p1_skipped = 0, p1_eff = 0, dp_cells_p1 = 0;
  DevBuf<uint16_t> d_packed;
  DevBuf<int64_t> d_off2;
  DevBuf<int32_t> d_src;
  // consensus
  DevBuf<miagpu_entry> d_entries;
  DevBuf<int32_t> d_ent_pos;                   // start position per entry (tile_kernel's scan list)
  int64_t n_entries = 0;
  DevBuf<int32_t> d_sm, d_gaps, d_ins_off, d_acc;
  DevBuf<uint8_t> d_cub, d_dropf, d_dropb, d_newly;
  DevBuf<char> d_called;
  int64_t n_cols = 0;
  int cons_stage = 0;                          // 0 none, 1 gaps done, 2 counts done
  // FSDB pointer state (slots.cuh): FragSeq.front_asp / back_asp as slot indices, AlnSeq.dropped per slot
  bool fs_on = false;                          // miagpu_set_fsdb: the one-call rounds follow the reference's pointer semantics
  int fs_distant = 0;                          // maln->distant_ref (-D)
  int fs_submat_rc = 0;                        // which matrix a->submat was left pointing at (H6)
  std::vector<int32_t> dr_U, dr_sc, dr_a0, dr_a1, dr_score;   // miagpu_distant_retry_begin -> _end: the strand-unknown reads, their three attempts, fs->score
  bool dr_ready = false;
  int fs_round = 0;                            // rounds since miagpu_set_fsdb
  int64_t fs_slot_cap = 0, fs_nslots = 0, fs_nslots_prev = 0;
  bool fs_sharded = false;                     // the round in flight numbers its slots over all ranks (miagpu_shard_*)
  int fs_prev_seq_len = 0;
  bool fs_prev_valid = false, fs_prev_pass1 = false, fs_seed_read_flags = false;
  DevBuf<uint8_t> d_known, d_slot_flag, d_slot_new, d_flip_prev;
  DevBuf<int32_t> d_front_slot, d_back_slot, d_first, d_nsl, d_slot_owner, d_slot_owner_prev, d_ent_slot, d_stale, d_fs_cnt, d_fs_tmp, d_nprefix;
  DevBuf<uint16_t> d_runs_prev;                // previous round's alignment: ping-pong partners of d_runs / d_nruns / d_abr / d_as_out / d_ae_out
  DevBuf<int32_t> d_nruns_prev, d_abr_prev, d_as_prev, d_ae_prev, d_score_prev;
  DevBuf<uint8_t> d_fz_bases, d_fz_rc;         // frozen alignments
  DevBuf<uint16_t> d_fz_runs;
  DevBuf<int32_t> d_fz_nruns;
  struct FzHost { int32_t start, cols, dels, rc, score, seg, read, num_inputs; };
  std::vector<FzHost> fz;                      // geometry of the frozen alignments
  std::unordered_map<int64_t, int> fz_of_slot; // slot that is no longer live -> its frozen content
  std::vector<uint8_t> h_known, h_rc;          // host mirrors (the -D chain is resolved on the host)
  int64_t fs_n_extra = 0, fs_n_stale = 0, fs_n_ghost = 0;
  struct FsExtra { int32_t holder, kind, slot, live_entry, frozen, front_len, total_len, act_bias, back_formula, listed; };
  std::vector<FsExtra> fs_extra;               // this round's stale pointers, in FSDB order (front before back)
  std::vector<int32_t> fs_patch_host;          // smp parameters the writer needs for slots whose last visitor is a stale pointer
  miagpu_ctx* aux = nullptr;                   // scratch context of the -D attempts
  // miagpu_misincorporation: whether the entry list, alignments, reads and reference on the device are still those of the last
  // round that ended with base calling, and if not, the call that changed them
  const char* misinc_stale = "no round has ended with base calling on this context";
  DevBuf<unsigned long long> d_misinc;
  cudaEvent_t misinc_ev[3] = {};               // its own timing events: the rounds' events may still be read between their calls
  // timing of the last call
  float ms_kernels = 0, ms_h2d = 0, ms_d2h = 0;
  int64_t dp_cells = 0;
  int launches = 0;
};


// the table of miagpu_misincorporation belongs to the state the last round left: the first call after it that changes that state
// is what a refusal names (before any round: that there was none)
static void misinc_invalidate(miagpu_ctx* c, const char* why) {
  if (!c->misinc_stale) c->misinc_stale = why;
}

// -------------------------------------------------------------------- misc
extern "C" const char* miagpu_last_error(void) { return g_err; }
extern "C" const char* miagpu_version(void) { return "miagpu 0.1 (sm_100a)"; }

extern "C" int miagpu_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

extern "C" int miagpu_create(miagpu_ctx** out, int device) {
  if (!out) { set_error("miagpu_create: out is NULL"); return 0; }
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    set_error("miagpu_create: no CUDA device (%s); this library has no CPU fallback", e == cudaSuccess ? "count = 0" : cudaGetErrorString(e));
    return 0;
  }
  if (device < 0 || device >= n) { set_error("miagpu_create: device %d out of range (0..%d)", device, n - 1); return 0; }
  MIAGPU_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  MIAGPU_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) { set_error("miagpu_create: device %d is sm_%d%d; this build is sm_100a only", device, prop.major, prop.minor); return 0; }
  miagpu_ctx* c = new miagpu_ctx();
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  MIAGPU_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  for (auto& ev : c->ev) MIAGPU_CUDA(cudaEventCreate(&ev));
  for (auto& ev : c->p1ev) MIAGPU_CUDA(cudaEventCreate(&ev));
  for (auto& ev : c->bev) MIAGPU_CUDA(cudaEventCreate(&ev));
  for (auto& ev : c->pev) MIAGPU_CUDA(cudaEventCreate(&ev));
  c->s_aux[0] = c->stream; c->launch_stream = c->stream;
  for (int i = 1; i < 4; i++) MIAGPU_CUDA(cudaStreamCreateWithFlags(&c->s_aux[i], cudaStreamNonBlocking));
  for (auto& ev : c->aev) MIAGPU_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  // the upload stream also classifies the next chunk while this chunk's persistent DP blocks hold every SM slot:
  // highest priority, so that its few blocks are placed first whenever a DP class drains
  int prio_lo = 0, prio_hi = 0;
  MIAGPU_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  MIAGPU_CUDA(cudaStreamCreateWithPriority(&c->s_up, cudaStreamNonBlocking, prio_hi));
  MIAGPU_CUDA(cudaStreamCreateWithFlags(&c->s_down, cudaStreamNonBlocking));
  for (auto& ev : c->cev) MIAGPU_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  for (auto& ev : c->xev) MIAGPU_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  MIAGPU_CUDA(cudaMallocHost(&c->h_meta, sizeof(int32_t) * MAX_CHUNKS * META_HOST));
  *out = c;
  return 1;
}

extern "C" void miagpu_destroy(miagpu_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  c->d_jkind.release(); c->d_jstatus.release(); c->d_route.release(); c->d_jws.release(); c->d_jwl.release(); c->d_jscore.release();
  c->d_jabc.release(); c->d_jaec.release(); c->d_jabr.release(); c->d_p1list.release(); c->d_p1trace.release(); c->d_sw_jobs.release(); c->d_sw_layout.release(); c->d_sw_pairs.release(); c->d_p1sunk.release(); c->d_p1meta.release(); c->d_jpairs.release();
  c->d_jread.release(); c->d_jfirst.release(); c->d_jcount.release();
  c->d_prof.release(); c->d_ref.release(); c->d_rcref.release(); c->d_ref2.release(); c->d_bases.release(); c->d_off.release();
  c->d_rc.release(); c->d_status.release(); c->d_as.release(); c->d_ae.release(); c->d_score.release();
  c->d_as_out.release(); c->d_ae_out.release(); c->d_abr.release(); c->d_nruns.release(); c->d_win_start.release();
  c->d_win_len.release(); c->d_lists.release(); c->d_runs.release(); c->d_meta.release();
  for (auto& b : c->d_scratch) b.release();
  for (int i = 1; i < 4; i++) cudaStreamDestroy(c->s_aux[i]);
  for (auto& ev : c->aev) cudaEventDestroy(ev);
  for (int t = 0; t < 2; t++) { c->d_kb[t].release(); c->d_kp[t].release(); c->d_kk[t].release(); }
  c->d_smask.release(); c->d_ckpt.release(); c->d_chunk_ids.release(); c->d_strace.release(); c->d_hits.release(); c->d_fw.release();
  c->d_rcs.release(); c->d_start.release(); c->d_end.release(); c->d_rc_out.release(); c->d_bases2.release(); c->d_packed.release(); c->d_off2.release(); c->d_src.release();
  c->d_entries.release(); c->d_ent_pos.release(); c->d_sm.release(); c->d_gaps.release(); c->d_ins_off.release(); c->d_acc.release(); c->d_cub.release(); c->d_called.release(); c->d_dropf.release(); c->d_dropb.release(); c->d_newly.release();
  for (auto& ev : c->ev) cudaEventDestroy(ev);
  for (auto& ev : c->p1ev) cudaEventDestroy(ev);
  for (auto& ev : c->bev) cudaEventDestroy(ev);
  for (auto& ev : c->pev) cudaEventDestroy(ev);
  c->d_prof16.release(); c->d_kind.release(); c->d_pairs.release();
  for (auto& ev : c->cev) cudaEventDestroy(ev);
  for (auto& ev : c->xev) cudaEventDestroy(ev);
  cudaStreamDestroy(c->s_up);
  cudaStreamDestroy(c->s_down);
  cudaFreeHost(c->h_meta);
  if (c->h_cut) cudaFreeHost(c->h_cut);
  if (c->h_cblk) cudaFreeHost(c->h_cblk);
  if (c->h_score) cudaFreeHost(c->h_score);
  if (c->h_call) cudaFreeHost(c->h_call);
  if (c->h_sh_recv) cudaFreeHost(c->h_sh_recv);
  c->d_sh_prep.release();
  c->d_sh_send.release(); c->d_sh_recv.release();
  c->tr_prof.release(); c->tr_ws.release(); c->tr_wl.release(); c->tr_out.release(); c->tr_cnt.release(); c->tr_codes.release();
  c->tr_ad.release(); c->tr_st.release();
  c->rf_rc.release(); c->rf_tr.release(); c->rf_uq.release(); c->rf_tmp.release(); c->rf_as.release(); c->rf_ae.release(); c->rf_k4.release();
  c->rf_idx.release(); c->rf_idx2.release(); c->rf_key.release(); c->rf_key2.release(); c->rf_ord.release(); c->rf_bad.release();
  c->d_seqlen.release(); c->d_unique.release(); c->d_cstats.release(); c->d_ctab.release(); c->d_thr.release(); c->d_cblk.release();
  c->d_known.release(); c->d_slot_flag.release(); c->d_slot_new.release(); c->d_flip_prev.release(); c->d_front_slot.release();
  c->d_back_slot.release(); c->d_first.release(); c->d_nsl.release(); c->d_slot_owner.release(); c->d_slot_owner_prev.release();
  c->d_ent_slot.release(); c->d_stale.release(); c->d_fs_cnt.release(); c->d_fs_tmp.release(); c->d_nprefix.release();
  c->d_runs_prev.release(); c->d_nruns_prev.release(); c->d_abr_prev.release(); c->d_as_prev.release(); c->d_ae_prev.release(); c->d_score_prev.release();
  c->d_fz_bases.release(); c->d_fz_rc.release(); c->d_fz_runs.release(); c->d_fz_nruns.release(); c->d_misinc.release();
  for (auto& ev : c->misinc_ev) if (ev) cudaEventDestroy(ev);
  if (c->aux) miagpu_destroy(c->aux);
  cudaStreamDestroy(c->stream);
  delete c;
}

extern "C" void* miagpu_stream(miagpu_ctx* c) { return c ? (void*)c->stream : nullptr; }

// -------------------------------------------------------------------- PSSM
static void revcom_pssm(const int32_t* in, int32_t* out) {      // pssm.c:53-93
  for (int d = 0; d < NMAT; d++)
    for (int i = 0; i < 5; i++)
      for (int j = 0; j < 5; j++) {
        int ci = i < 4 ? 3 - i : 4, cj = j < 4 ? 3 - j : 4;
        out[((NMAT - 1 - d) * 5 + i) * 5 + j] = in[(d * 5 + ci) * 5 + cj];
      }
}

extern "C" int miagpu_set_pssm(miagpu_ctx* c, const int32_t* fwd) {
  if (!c || !fwd) { set_error("miagpu_set_pssm: NULL argument"); return 0; }
  for (int i = 0; i < MIAGPU_PSSM_INTS; i++)
    if (fwd[i] > PSSM_ABS_LIMIT || fwd[i] < -PSSM_ABS_LIMIT) {
      set_error("miagpu_set_pssm: entry %d = %d exceeds the supported magnitude %d", i, fwd[i], PSSM_ABS_LIMIT);
      return 0;
    }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  memcpy(c->sm_f, fwd, sizeof(c->sm_f));
  revcom_pssm(c->sm_f, c->sm_r);
  std::vector<int32_t> prof(PROF_INTS, 0);
  for (int s = 0; s < 2; s++)
    for (int d = 0; d < NMAT; d++)
      for (int rb = 0; rb < 5; rb++)
        for (int fb = 0; fb < 5; fb++)   // sm[depth][ref_base][read_base]
          prof[prof_row_index(s, d, rb) + fb] = (s ? c->sm_r : c->sm_f)[(d * 5 + fb) * 5 + rb];
  if (!c->d_prof.reserve(PROF_INTS) || !c->d_sm.reserve(2 * MIAGPU_PSSM_INTS)) return 0;
  MIAGPU_CUDA(cudaMemcpyAsync(c->d_prof.p, prof.data(), PROF_INTS * 4, cudaMemcpyHostToDevice, c->stream));
  MIAGPU_CUDA(cudaMemcpyAsync(c->d_sm.p, c->sm_f, sizeof(c->sm_f), cudaMemcpyHostToDevice, c->stream));
  MIAGPU_CUDA(cudaMemcpyAsync(c->d_sm.p + MIAGPU_PSSM_INTS, c->sm_r, sizeof(c->sm_r), cudaMemcpyHostToDevice, c->stream));
  // 16-bit profile of the pair kernel
  std::vector<int16_t> prof16(PROF16_N + 8, 0);
  for (int i = 0; i < PROF16_N; i++) prof16[i] = (int16_t)prof[i];
  if (!c->d_prof16.reserve(PROF16_N + 8)) return 0;
  MIAGPU_CUDA(cudaMemcpyAsync(c->d_prof16.p, prof16.data(), (PROF16_N + 8) * 2, cudaMemcpyHostToDevice, c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  c->pssm_min = *std::min_element(fwd, fwd + MIAGPU_PSSM_INTS);
  c->pssm_max = *std::max_element(fwd, fwd + MIAGPU_PSSM_INTS);
  c->lmax16 = std::min(p16_lmax(4, c->pssm_max), P16_MAXL);   // longest read any pair class holds (fewest columns per lane)
  if (c->pssm_max + GEP <= 0) c->lmax16 = 0;                   // degenerate matrices: 32-bit kernels only
  c->have_pssm = true;
  return 1;
}

extern "C" int miagpu_get_pssm(miagpu_ctx* c, int32_t* fwd, int32_t* rev) {
  if (!c || !c->have_pssm) { set_error("miagpu_get_pssm: no matrices set"); return 0; }
  if (fwd) memcpy(fwd, c->sm_f, sizeof(c->sm_f));
  if (rev) memcpy(rev, c->sm_r, sizeof(c->sm_r));
  return 1;
}

// --------------------------------------------------------------- reference
static int fs_upload_nprefix(miagpu_ctx* c);
static char revcom_char(char b) {                                // map_align.c:418-431
  static const char* from = "ABCDGHKMNRSTUVWXY";
  static const char* to = "TVGHCDMKNYSAABWXR";
  if (b == '-') return '-';
  bool lower = b >= 'a' && b <= 'z';
  char u = lower ? (char)(b - 32) : b;
  const char* q = (u >= 'A' && u <= 'Z') ? strchr(from, u) : nullptr;
  if (!q || !*q) return 'N';
  return lower ? (char)(to[q - from] + 32) : to[q - from];
}

static int upload_codes(miagpu_ctx* c, const std::string& s, DevBuf<uint8_t>& dst) {
  int padded = ((int)s.size() + 15) / 16 * 16 + 16;
  std::vector<uint8_t> codes(padded, 4);
  for (size_t i = 0; i < s.size(); i++) {
    char u = s[i];
    if (u >= 'a' && u <= 'z') u = (char)(u - 32);               // make_ref_upper, mia.c:642-648
    codes[i] = (uint8_t)base_code((uint8_t)u);
  }
  if (!dst.reserve(padded)) return 0;
  MIAGPU_CUDA(cudaMemcpyAsync(dst.p, codes.data(), padded, cudaMemcpyHostToDevice, c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  c->ref_bytes = padded;
  return 1;
}

extern "C" int miagpu_set_reference(miagpu_ctx* c, const char* seq, int seq_len, int circular, int with_rc) {
  if (!c || !seq || seq_len <= 0) { set_error("miagpu_set_reference: bad argument"); return 0; }
  misinc_invalidate(c, "miagpu_set_reference has replaced the reference of that round");
  MIAGPU_CUDA(cudaSetDevice(c->device));
  int wrap = circular ? std::min(seq_len, MAX_READ) : 0;         // add_ref_wrap, mia.c:657-689
  c->seq_len = seq_len;
  c->wrap_len = seq_len + wrap;
  c->circular = circular;
  c->with_rc = with_rc;
  c->raw_wrapped.assign(seq, seq_len);
  c->raw_wrapped.append(seq, wrap);
  if (!upload_codes(c, c->raw_wrapped, c->d_ref)) return 0;
  c->raw_rc_wrapped.clear();
  if (with_rc) {                                                 // io.c:388-398, then the same wrap
    std::string rcs(seq_len, 'N');
    for (int i = 0; i < seq_len; i++) rcs[i] = revcom_char(seq[seq_len - 1 - i]);
    c->raw_rc_wrapped = rcs;
    c->raw_rc_wrapped.append(rcs, 0, wrap);
    if (!upload_codes(c, c->raw_rc_wrapped, c->d_rcref)) return 0;
    // both strands back to back for the pass-1 pair kernels (a job's window start carries the strand)
    if (!c->d_ref2.reserve(2 * (size_t)c->ref_bytes)) return 0;
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_ref2.p, c->d_ref.p, c->ref_bytes, cudaMemcpyDeviceToDevice, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_ref2.p + c->ref_bytes, c->d_rcref.p, c->ref_bytes, cudaMemcpyDeviceToDevice, c->stream));
    MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  }
  c->have_ref = true;
  c->hps_valid = false;
  if (c->fs_on && c->fs_distant && !fs_upload_nprefix(c)) return 0;
  return 1;
}

// mia -h: hp_special (mia_main.c:424, 497).  From now on dyn_prog's two homopolymer-discounted gap candidates (mia.c:882-905) take part
// in every alignment of this context: pass 1 (homopolymers of the whole strands, mia_main.c:735-739), the rounds (of the read's window,
// mia_main.c:221-224), the -D attempts (mia_main.c:132-134, 158-160).  All of them run in the chunked 32-bit kernel (strip.cuh); the
// 16-bit kernels do not carry the candidates.  miagpu_trim and explicit windows with sg5 = 0 refuse a context in this mode.
extern "C" int miagpu_set_homopolymer(miagpu_ctx* c, int on) {
  if (!c) { set_error("miagpu_set_homopolymer: no context"); return 0; }
  c->hp = on != 0;
  return 1;
}

// pop_hpl_and_hps (mia.c:1193-1234) over the upper-cased wrapped strands: only the starts are needed (hp_discount_penalty ignores
// the column homopolymer's length).  The kernel compares the read's raw byte with the reference base it knows as a code 0..4, so a
// reference with other letters than A C G T N cannot be served exactly and is refused.
static int ensure_hps(miagpu_ctx* c) {
  if (c->hps_valid) return 1;
  const int len1 = c->wrap_len;
  std::vector<int32_t> h(len1);
  for (int s = 0; s < (c->with_rc ? 2 : 1); s++) {
    const std::string& t = s ? c->raw_rc_wrapped : c->raw_wrapped;
    int start = 0;
    for (int i = 0; i < len1; i++) {
      const char b = (char)toupper((unsigned char)t[i]);
      if (b != 'A' && b != 'C' && b != 'G' && b != 'T' && b != 'N') {
        set_error("homopolymer mode: reference base '%c' at %d: only A C G T N can be compared with the reads on the device", t[i], i);
        return 0;
      }
      if (i > 0 && b != (char)toupper((unsigned char)t[i - 1])) start = i;
      h[i] = start;
    }
    if (!c->d_hps[s].reserve(len1 + 1)) return 0;
    MIAGPU_CUDA(cudaMemcpy(c->d_hps[s].p, h.data(), (size_t)len1 * 4, cudaMemcpyHostToDevice));
  }
  c->hps_valid = true;
  return 1;
}

extern "C" int miagpu_ref_wrap_len(miagpu_ctx* c) { return c ? c->wrap_len : 0; }

// ------------------------------------------------------------------- reads
static int reserve_per_read(miagpu_ctx* c, int64_t n) {
  return c->d_rc.reserve(n) && c->d_status.reserve(n) && c->d_as.reserve(n) && c->d_ae.reserve(n) && c->d_score.reserve(n) &&
         c->d_as_out.reserve(n) && c->d_ae_out.reserve(n) && c->d_abr.reserve(n) && c->d_nruns.reserve(n) &&
         c->d_win_start.reserve(n) && c->d_win_len.reserve(n) && c->d_lists.reserve(n * NBUCKET) &&
         c->d_runs.reserve(n * MAX_RUNS) && c->d_meta.reserve(META_WORDS * MAX_CHUNKS) && c->d_kind.reserve(n + 1) &&
         c->d_pairs.reserve(n + MAX_CHUNKS * (8 * P16_KEYS + 64));
}

extern "C" int miagpu_upload_reads(miagpu_ctx* c, int64_t n, const uint8_t* bases, const int64_t* offsets) {
  if (!c || n < 0 || (n > 0 && (!bases || !offsets))) { set_error("miagpu_upload_reads: bad argument"); return 0; }
  misinc_invalidate(c, "miagpu_upload_reads has replaced the reads of that round");
  MIAGPU_CUDA(cudaSetDevice(c->device));
  if (n > 0x7fffffffLL / NBUCKET) { set_error("miagpu_upload_reads: at most %lld reads per batch", 0x7fffffffLL / NBUCKET); return 0; }
  int64_t total = n ? offsets[n] : 0;
  if (n && offsets[0] != 0) { set_error("miagpu_upload_reads: offsets[0] must be 0"); return 0; }
  if (!c->d_bases.reserve(total + 16) || !c->d_off.reserve(n + 1) || !reserve_per_read(c, n)) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->ev[0], c->stream));
  if (n) {
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_bases.p, bases, total, cudaMemcpyHostToDevice, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_off.p, offsets, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
  }
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]));
  c->n = n;
  c->total_bases = total;
  c->cut_inputs_n = -1;
  c->fs_on = false; c->fs_prev_valid = false;
  c->max_read_len = -1;                      // computed on demand (device reduction) by the chunked kernel's launcher
  return 1;
}

// ----------------------------------------------------------------- realign
// Window rule of reiterate_assembly (mia_main.c:190-212) + width class.  A read goes either to the
// work list of its 32-bit width bucket or, when the 16-bit pair kernel can take it (short enough for
// the 16-bit frame of its width class, at most 256 columns), into the (pair class, read length)
// histogram that pairs reads of equal length.
// Block-level statistics go through shared-memory counters; lanes of a warp that hit the same counter are
// merged first (match.any + redux), so a counter sees one atomic per warp instead of up to 32.
__global__ void classify_kernel(int64_t n, const int64_t* off, const int32_t* as, const int32_t* ae, int wrap_len, PairLmax lm,
                                int32_t* win_start, int32_t* win_len, int32_t* lists, uint8_t* kind, int32_t* meta, int explicit_win = 0,
                                const uint8_t* __restrict__ known = nullptr) {
  int lmax16 = 0;
  for (int k = 0; k < P16_NKB; k++) lmax16 = max(lmax16, lm.v[k]);
  __shared__ int s_cnt[NBUCKET], s_base[NBUCKET], s_maxL[NBUCKET], s_pop[NBUCKET];
  __shared__ unsigned long long s_cells[NBUCKET];
  __shared__ int s_hist[P16_KEYS];
  __shared__ int s_preads[P16_NKB], s_pmaxl[P16_NKB];
  __shared__ unsigned long long s_pcells[P16_NKB];
  if (threadIdx.x < NBUCKET) { s_cnt[threadIdx.x] = 0; s_maxL[threadIdx.x] = 0; s_pop[threadIdx.x] = 0; s_cells[threadIdx.x] = 0; }
  if (threadIdx.x < P16_NKB) { s_preads[threadIdx.x] = 0; s_pcells[threadIdx.x] = 0; s_pmaxl[threadIdx.x] = 0; }
  if (lmax16 > 0) for (int i = threadIdx.x; i < P16_KEYS; i += blockDim.x) s_hist[i] = 0;
  __syncthreads();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1;
  int b = -1, slot = 0, L = 0, key = -1, kb = -1;
  unsigned cells = 0;
  bool direct = false;
  if (i < n && known && !known[i]) {
    kind[i] = 15;                                       // strand unknown: not realigned (mia_main.c:178)
  } else if (i < n) {
    L = (int)(off[i + 1] - off[i]);
    int rs = as[i] - REALIGN_BUFFER < 0 ? 0 : as[i] - REALIGN_BUFFER;
    int re = (ae[i] + REALIGN_BUFFER + 1 > wrap_len) ? wrap_len : ae[i] + REALIGN_BUFFER;
    bool whole = rs + L > re;
    if (whole) { rs = 0; re = wrap_len; }
    if (explicit_win) { rs = as[i]; re = ae[i]; whole = true; }          // caller's window as it is; 32-bit kernels only (whole => not pair-eligible)
    int len1 = re - rs;
    win_start[i] = rs;
    win_len[i] = len1;
    b = bucket32_of(len1);
    if (L <= 0 || L > MAX_READ) b = NBUCKET - 1;
    kb = p16_class(len1);
    const bool elig = b != NBUCKET - 1 && kb >= 0 && !whole && L <= lm.v[kb < 0 ? 0 : kb];
    cells = (unsigned)max(L, 0) * (unsigned)len1;                       // <= 256 * wrap_len: a warp's sum fits 32 bits up to 500 kb windows
    if (elig) { kind[i] = (uint8_t)(16 + kb); key = kb * (P16_MAXL + 1) + L; }
    else { kind[i] = (uint8_t)b; direct = true; kb = -1; }
  }
  // per width bucket: population, longest read, cells
  {
    const unsigned peers = __match_any_sync(0xffffffffu, b);
    const int mx = __reduce_max_sync(peers, L);
    const unsigned long long cs = (unsigned long long)__reduce_add_sync(peers, cells & 0xffffu) +
                                  ((unsigned long long)__reduce_add_sync(peers, cells >> 16) << 16);
    if (b >= 0 && (peers & lt) == 0) {
      atomicAdd(&s_pop[b], __popc(peers));
      atomicMax(&s_maxL[b], mx);
      atomicAdd(&s_cells[b], cs);
    }
  }
  // pair-eligible reads: histogram per (class, length), reads and cells per class
  if (lmax16 > 0) {
    const unsigned pk = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && (pk & lt) == 0) atomicAdd(&s_hist[key], __popc(pk));
    const unsigned pc = __match_any_sync(0xffffffffu, kb);
    const unsigned long long cs = (unsigned long long)__reduce_add_sync(pc, cells & 0xffffu) + ((unsigned long long)__reduce_add_sync(pc, cells >> 16) << 16);
    const int mxl = __reduce_max_sync(pc, L);
    if (kb >= 0 && (pc & lt) == 0) { atomicAdd(&s_preads[kb], __popc(pc)); atomicAdd(&s_pcells[kb], cs); atomicMax(&s_pmaxl[kb], mxl); }
  }
  // reads that go straight to a 32-bit list take consecutive slots
  {
    const int db = direct ? b : -1;
    const unsigned pd = __match_any_sync(0xffffffffu, db);
    int base = 0;
    if (direct && (pd & lt) == 0) base = atomicAdd(&s_cnt[b], __popc(pd));
    base = __shfl_sync(0xffffffffu, base, __ffs(pd) - 1);
    slot = base + __popc(pd & lt);
  }
  __syncthreads();
  if (threadIdx.x < NBUCKET) {
    const int t = threadIdx.x;
    s_base[t] = s_cnt[t] ? atomicAdd(&meta[META_COUNT + t], s_cnt[t]) : 0;
    if (s_maxL[t]) atomicMax(&meta[META_MAXL + t], s_maxL[t]);
    if (s_pop[t]) atomicAdd(&meta[META_POP + t], s_pop[t]);
    if (s_cells[t]) atomicAdd(reinterpret_cast<unsigned long long*>(meta + META_CELLS) + t, s_cells[t]);
  }
  if (threadIdx.x < P16_NKB && s_preads[threadIdx.x]) {
    atomicAdd(&meta[META_PREADS + threadIdx.x], s_preads[threadIdx.x]);
    atomicAdd(reinterpret_cast<unsigned long long*>(meta + META_PCELLS) + threadIdx.x, s_pcells[threadIdx.x]);
    atomicMax(&meta[META_PMAXL + threadIdx.x], s_pmaxl[threadIdx.x]);
  }
  if (lmax16 > 0)
    for (int k = threadIdx.x; k < P16_KEYS; k += blockDim.x)
      if (s_hist[k]) atomicAdd(&meta[META_HIST + k], s_hist[k]);
  __syncthreads();
  if (direct) lists[(int64_t)b * n + s_base[b] + slot] = (int32_t)i;
}

// Pairs per (class, length) key: ceil(count / 2), rounded up to whole work items of P16_NP pairs (a warp's reads all
// have one length), laid out class after class.  META_PSTART is in pairs, META_NPAIRS in work items.
// One block: a thread takes LAYOUT_PER consecutive keys, the block scans the per-thread totals.
constexpr int LAYOUT_THREADS = 256;
constexpr int LAYOUT_PER = (P16_KEYS + LAYOUT_THREADS - 1) / LAYOUT_THREADS;
__global__ void __launch_bounds__(LAYOUT_THREADS) pair_layout_kernel(int32_t* meta) {
  __shared__ int s_tot[LAYOUT_THREADS];
  __shared__ int s_start[P16_KEYS + 1];
  const int t = threadIdx.x;
  int items[LAYOUT_PER], sum = 0;
#pragma unroll
  for (int q = 0; q < LAYOUT_PER; q++) {
    const int k = t * LAYOUT_PER + q;
    const int pairs = k < P16_KEYS ? (meta[META_HIST + k] + 1) >> 1 : 0;
    items[q] = (pairs + P16_NP - 1) / P16_NP * P16_NP;
    sum += items[q];
  }
  s_tot[t] = sum;
  __syncthreads();
  for (int d = 1; d < LAYOUT_THREADS; d <<= 1) {           // Hillis-Steele inclusive scan
    const int v = t >= d ? s_tot[t - d] : 0;
    __syncthreads();
    s_tot[t] += v;
    __syncthreads();
  }
  int run = s_tot[t] - sum;
#pragma unroll
  for (int q = 0; q < LAYOUT_PER; q++) {
    const int k = t * LAYOUT_PER + q;
    if (k < P16_KEYS) { meta[META_PSTART + k] = run; s_start[k] = run; }
    run += items[q];
  }
  if (t == LAYOUT_THREADS - 1) s_start[P16_KEYS] = s_tot[t];
  __syncthreads();
  if (t < P16_NKB) meta[META_NPAIRS + t] = (s_start[(t + 1) * (P16_MAXL + 1)] - s_start[t * (P16_MAXL + 1)]) / P16_NP;
}

// Eligible reads take the next free slot of their key: slot s is member s&1 of pair pstart + s/2.
// item_read (nullable): the items are pass-1 jobs, item_read[i] & 0x7fffffff is the job's read and off[] is per read.
__global__ void pair_scatter_kernel(int64_t n, const int64_t* off, const uint8_t* kind, int32_t* meta, int32_t* pairs,
                                    const int32_t* item_read = nullptr) {
  __shared__ int s_cnt[P16_KEYS], s_base[P16_KEYS];
  for (int i = threadIdx.x; i < P16_KEYS; i += blockDim.x) s_cnt[i] = 0;
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int key = -1, slot = 0;
  if (i < n && kind[i] >= 16) {
    const int64_t rd = item_read ? (int64_t)(item_read[i] & 0x7fffffff) : i;
    key = (kind[i] - 16) * (P16_MAXL + 1) + (int)(off[rd + 1] - off[rd]);
    slot = atomicAdd(&s_cnt[key], 1);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < P16_KEYS; k += blockDim.x)
    if (s_cnt[k]) s_base[k] = atomicAdd(&meta[META_CURSOR + k], s_cnt[k]);
  __syncthreads();
  if (key >= 0) {
    const int g = s_base[key] + slot;
    pairs[2 * (int64_t)(meta[META_PSTART + key] + (g >> 1)) + (g & 1)] = (int32_t)i;
  }
}

// OR of the per-read status bytes of a round (reads the consensus would silently leave out: more than MAX_RUNS runs, a window
// no kernel takes): the one-call rounds fail instead
__global__ void status_or_kernel(int64_t n, const uint8_t* __restrict__ status, const int32_t* __restrict__ n_runs, int32_t* out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int st = 0;
  if (i < n) st = status[i] | (n_runs[i] <= 0 ? MIAGPU_ST_RUNS_OVERFLOW : 0);
  st = __reduce_or_sync(0xffffffffu, st);
  if ((threadIdx.x & 31) == 0 && st) atomicOr(out, st);
}

__global__ void flag_big_kernel(const int32_t* list, int n_list, int32_t* score, int32_t* n_runs, uint8_t* status) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_list) { int rd = list[i]; score[rd] = INT_MIN; n_runs[rd] = -1; status[rd] = 0x80; }
}

// ------------------------------------------------ chunked kernel (pass 1, wide windows)
__global__ void max_len_kernel(int64_t n, const int64_t* off, int32_t* out) {
  int m = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = max(m, (int)(off[i + 1] - off[i]));
  m = __reduce_max_sync(0xffffffffu, m);
  if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

static int ensure_max_read_len(miagpu_ctx* c) {
  if (c->max_read_len >= 0) return 1;
  int32_t m = 0;
  if (c->n) {
    MIAGPU_CUDA(cudaMemsetAsync(c->d_meta.p + META_MAXLEN, 0, 4, c->stream));
    max_len_kernel<<<256, 256, 0, c->stream>>>(c->n, c->d_off.p, c->d_meta.p + META_MAXLEN);
    MIAGPU_CUDA(cudaMemcpyAsync(&m, c->d_meta.p + META_MAXLEN, 4, cudaMemcpyDeviceToHost, c->stream));
    MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  }
  c->max_read_len = m;
  return 1;
}

// mode 0 with a list: pass 1 over the listed reads only; n_list is then an upper bound and n_list_ptr the list's
// length on the device (the seeding / merge kernels of pass1.cuh fill it).
static int launch_strip(miagpu_ctx* c, int mode, const int32_t* list, int n_list, int32_t* counter, int64_t lo = 0, const int32_t* n_list_ptr = nullptr) {
  if (!ensure_max_read_len(c)) return 0;
  const int len1 = c->circular ? c->wrap_len : c->seq_len;                 // mia_main.c:721-728
  const int n_chunks = (len1 + CW - 1) / CW;
  const int Lmax = std::min(std::max(c->max_read_len, 1), MAX_READ);
  const int mask_words = n_chunks * (CW / 32);
  const int64_t total = (mode == 0 && !list) ? c->n : n_list;
  if (total == 0) return 1;
  // few reads: a team of warps per read (strip_team_kernel), else a warp per read
  bool team = total <= (int64_t)2 * c->num_sms * 4;
  if (const char* e = getenv("MIAGPU_STRIP_TEAM")) team = atoi(e) != 0;
  const bool hp = c->hp;
  if (hp) { team = false; if (!ensure_hps(c)) return 0; }          // the team schedule does not carry the homopolymer checkpoints
  const size_t smem = team ? PROF_INTS * 4 + MAX_READ * 2 + (size_t)((n_chunks + 3) & ~3) * 4 + (size_t)2 * TEAM_WARPS * Lmax * 16
                           : PROF_INTS * 4 + WARPS_PER_BLOCK * MAX_READ * 2 + (hp ? WARPS_PER_BLOCK * STRIP_HP_SMEM_PER_WARP : 0);
  if (team && smem > 200 * 1024) team = false;
  int per_sm = 0;
  if (team) {
    if (smem > 40 * 1024) MIAGPU_CUDA(cudaFuncSetAttribute(strip_team_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   // + static
    MIAGPU_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, strip_team_kernel, TEAM_WARPS * 32, smem));
  } else if (hp) {
    MIAGPU_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, strip_kernel<true>, WARPS_PER_BLOCK * 32, smem));
  } else {
    MIAGPU_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, strip_kernel<false>, WARPS_PER_BLOCK * 32, smem));
  }
  if (per_sm < 1) { set_error("strip_kernel does not fit on an SM (team %d, %zu bytes of shared memory, Lmax %d, %d chunks)", (int)team, smem, Lmax, n_chunks); return 0; }
  // per-warp (per-team) scratch: keep the total under ~6 GB
  const size_t per_warp = (size_t)2 * mask_words * 4 + (size_t)2 * (n_chunks + 1) * Lmax * (hp ? 20 : 16) + (size_t)2 * n_chunks * 4 + (size_t)Lmax * CW * 4;
  const int units_per_block = team ? 1 : WARPS_PER_BLOCK;
  per_sm = std::min(per_sm, 4);
  while (per_sm > 1 && per_warp * c->num_sms * per_sm * units_per_block > ((size_t)6 << 30)) per_sm--;
  int blocks = (int)std::min<int64_t>((int64_t)c->num_sms * per_sm, (total + units_per_block - 1) / units_per_block);
  const size_t warps = (size_t)blocks * units_per_block;
  if (!c->d_smask.reserve(warps * 2 * mask_words) || !c->d_ckpt.reserve(warps * 2 * (n_chunks + 1) * Lmax) ||
      !c->d_chunk_ids.reserve(warps * 2 * n_chunks) || !c->d_strace.reserve(warps * Lmax * CW)) return 0;
  if (hp && !c->d_ckh.reserve(warps * 2 * (n_chunks + 1) * Lmax)) return 0;
  StripParams p{};
  p.bases = c->d_bases.p; p.off = c->d_off.p; p.n = c->n; p.counter = counter; p.mode = mode;
  p.list = list; p.n_list = n_list; p.n_list_ptr = n_list_ptr; p.rc_in = c->d_rc.p;
  p.ref_codes[0] = c->d_ref.p; p.ref_codes[1] = c->with_rc ? c->d_rcref.p : c->d_ref.p;
  p.len1 = len1; p.seq_len = c->seq_len; p.prof = c->d_prof.p;
  p.sg5 = c->explicit_windows ? c->explicit_sg5 : 1;            // miagpu_align_windows' windows over 512 columns come here
  p.k =mode == 0 ? c->kmer_k : 0;
  for (int t = 0; t < 2; t++) p.kt[t] = KmerTable{c->d_kb[t].p, c->d_kk[t].p, c->d_kp[t].p, c->kmer_shift[t]};
  p.mask = c->d_smask.p; p.mask_words = mask_words; p.ckpt = c->d_ckpt.p; p.chunk_ids = c->d_chunk_ids.p;
  p.max_chunks = n_chunks; p.Lmax = Lmax; p.trace = c->d_strace.p;
  p.hits = mode == 0 ? c->d_hits.p : nullptr; p.score = c->d_score.p; p.fw_score = c->d_fw.p; p.rc_score = c->d_rcs.p;
  p.as_out = c->d_as_out.p; p.ae_out = c->d_ae_out.p; p.start = c->d_start.p; p.end = c->d_end.p; p.abr = c->d_abr.p;
  p.n_runs = c->d_nruns.p; p.rc_out = c->d_rc_out.p; p.runs = c->d_runs.p; p.status = c->d_status.p;
  p.win_start = c->d_win_start.p; p.win_len = c->d_win_len.p;
  p.hps[0] = c->d_hps[0].p; p.hps[1] = c->with_rc ? c->d_hps[1].p : c->d_hps[0].p; p.ckh = c->d_ckh.p;
  if (mode >= 1 && lo) {                       // a chunk of the batch: list entries count from read `lo`
    p.off += lo; p.rc_in += lo; p.score += lo; p.as_out += lo; p.ae_out += lo; p.abr += lo; p.n_runs += lo;
    p.runs += lo * MAX_RUNS; p.status += lo; p.win_start += lo; p.win_len += lo;
  }
  if (team) strip_team_kernel<<<blocks, TEAM_WARPS * 32, smem, c->launch_stream>>>(p);
  else if (hp) strip_kernel<true><<<blocks, WARPS_PER_BLOCK * 32, smem, c->launch_stream>>>(p);
  else strip_kernel<false><<<blocks, WARPS_PER_BLOCK * 32, smem, c->launch_stream>>>(p);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches++;
  return 1;
}

// Blocks of KERNEL one SM holds with `smem` bytes of dynamic shared memory; 0 with the error set when the kernel does not fit or a
// CUDA call fails.  Cached per instantiation AND per device (function attributes belong to a device; several contexts of one process
// may drive several GPUs): the attribute / occupancy calls cost more than the launch.
template <auto KERNEL>
static int blocks_per_sm(miagpu_ctx* c, size_t smem, const char* name, int K) {
  static size_t cached_smem_d[MAX_DEVICES];
  static int cached_per_sm_d[MAX_DEVICES];
  size_t& cached_smem = cached_smem_d[c->device % MAX_DEVICES];
  int& cached_per_sm = cached_per_sm_d[c->device % MAX_DEVICES];
  if (cached_smem != smem + 1) {
    MIAGPU_CUDA(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MIAGPU_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cached_per_sm, KERNEL, WARPS_PER_BLOCK * 32, smem));
    cached_smem = smem + 1;
  }
  if (cached_per_sm < 1) set_error("%s<%d> does not fit on an SM (smem %zu)", name, K, smem);
  return std::max(cached_per_sm, 0);
}

// realign_kernel over a work list: a width bucket of reiterate_assembly's windows (JOB = false), or pass 1's winning jobs whose
// path is not one plain diagonal, stretch by stretch with a trace (JOB = true)
template <int K, bool JOB = false>
static int launch_realign(miagpu_ctx* c, RealignParams p, int maxL) {
  using TL = TraceLayout<K>;
  const bool ref_in_smem = p.ref_bytes <= 160 * 1024;
  const size_t smem = PROF_INTS * 4 + WARPS_PER_BLOCK * MAX_READ * 2 + (ref_in_smem ? p.ref_bytes : 0);
  const int per_sm = blocks_per_sm<realign_kernel<K, false, JOB>>(c, smem, JOB ? "realign_kernel (pass-1 jobs)" : "realign_kernel", K);
  if (per_sm < 1) return 0;
  // at most 8 blocks = 32 warps per SM (measured best on B200); bounds the trace scratch
  const int blocks = std::min(c->num_sms * std::min(per_sm, 8), (p.n_list + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK);
  if (blocks < 1) return 1;
  const int64_t words = (int64_t)std::max(maxL - 1, 1) * TL::ROW_WORDS;
  DevBuf<uint32_t>& scratch = c->d_scratch[c->launch_slot];
  if (!scratch.reserve((size_t)words * blocks * WARPS_PER_BLOCK)) return 0;
  p.scratch = scratch.p;
  p.scratch_words_per_warp = words;
  p.ref_in_smem = ref_in_smem;
  realign_kernel<K, false, JOB><<<blocks, WARPS_PER_BLOCK * 32, smem, c->launch_stream>>>(p);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches++;
  return 1;
}

template <int K, bool JOB, bool RB>
static int launch_pair16(miagpu_ctx* c, Pair16Params p, int n_items) {
  const bool ref_in_smem = p.ref_bytes <= 160 * 1024;
  const size_t smem = P16_SMEM_FIXED + (ref_in_smem ? p.ref_bytes : 0);
  const int per_sm = blocks_per_sm<pair16_kernel<K, JOB, RB>>(c, smem, "pair16_kernel", K);
  if (per_sm < 1) return 0;
  if (RB) { const RbFrame f = p16_rb_frame(K, c->pssm_max); p.rb_off = f.off; p.rb_d = f.d; p.rb_thresh = f.thresh; }
  const int blocks = std::min(c->num_sms * std::min(per_sm, 8), (n_items + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK);
  if (blocks < 1) return 1;
  p.ref_in_smem = ref_in_smem;
  p.gep2 = K2(2 * GEP);
  pair16_kernel<K, JOB, RB><<<blocks, WARPS_PER_BLOCK * 32, smem, c->launch_stream>>>(p);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches++;
  return 1;
}

// is pair class kb built in the RB frame (pair16.cuh 5.)?  The wide classes only (K = 8 .. 16); for pass-1 jobs K = 10 .. 16 (a
// stretch is about L + 20 columns)
constexpr bool pair_rb_built(int kb, bool job) { return kb < P16_NKB_WIDE && !(job && kb < 2); }

// The pair kernel of class kb in the low or the RB frame.  Realign windows use the wide classes only; pass-1 jobs also the narrow
// ones, in the low frame.  A (class, frame) without a kernel is an error.
template <bool JOB, int KB = 0>
static int launch_pair_class(miagpu_ctx* c, const Pair16Params& p, int kb, bool rb, int n_items) {
  if constexpr (KB < P16_NKB) {
    if (kb != KB) return launch_pair_class<JOB, KB + 1>(c, p, kb, rb, n_items);
    constexpr int K = P16_COLS[KB] / P16_G;
    if constexpr (JOB || KB < P16_NKB_WIDE) {
      if (!rb) return launch_pair16<K, JOB, false>(c, p, n_items);
    }
    if constexpr (pair_rb_built(KB, JOB)) {
      if (rb) return launch_pair16<K, JOB, true>(c, p, n_items);
    }
  }
  set_error("pair class %d has no %s kernel in the %s frame", kb, JOB ? "pass-1 job" : "realign window", rb ? "RB" : "low");
  return 0;
}

// One realign job = reads [lo, lo + n) of the resident batch with their own meta block, work lists and pair
// table, so that several jobs (the chunks of miagpu_iterate_host's pipeline) can be in flight.
struct RealignJob {
  int64_t lo = 0, n = 0;
  int32_t* d_meta = nullptr;     // META_WORDS
  int32_t* d_lists = nullptr;    // NBUCKET * n
  int32_t* d_pairs = nullptr;    // n + 4 * P16_KEYS + 64
  int32_t* h_meta = nullptr;     // META_HOST words on the host (pinned for an asynchronous copy)
  bool timed = false;            // per-class events, one kernel after the other (the measurement path)
};

// Untimed jobs spread their DP kernels over four streams: the kernels are persistent (every block fetches work
// until its class runs dry), so the next class's blocks move in as the previous class's tail drains.
static int fork_streams(miagpu_ctx* c, int ev) {
  MIAGPU_CUDA(cudaEventRecord(c->aev[ev], c->stream));
  for (int i = 1; i < 4; i++) MIAGPU_CUDA(cudaStreamWaitEvent(c->s_aux[i], c->aev[ev], 0));
  return 1;
}
static int join_streams(miagpu_ctx* c, int ev) {
  for (int i = 1; i < 4; i++) {
    MIAGPU_CUDA(cudaEventRecord(c->aev[ev + i], c->s_aux[i]));
    MIAGPU_CUDA(cudaStreamWaitEvent(c->stream, c->aev[ev + i], 0));
  }
  c->launch_stream = c->stream; c->launch_slot = 0;
  return 1;
}
static void pick_stream(miagpu_ctx* c, bool concurrent, int& rr) {
  c->launch_slot = concurrent ? (rr++ & 3) : 0;
  c->launch_stream = c->s_aux[c->launch_slot];
}

// longest read every pair class takes in the low frame (pair16.cuh 2.)
static PairLmax pair_lmax_low(miagpu_ctx* c) {
  int lmax16 = c->lmax16;
  if (const char* e = getenv("MIAGPU_PAIR16")) if (atoi(e) == 0) lmax16 = 0;
  PairLmax lm{};
  for (int kb = 0; kb < P16_NKB; kb++) lm.v[kb] = lmax16 > 0 ? std::min(p16_lmax(P16_COLS[kb] / P16_G, c->pssm_max), P16_MAXL) : 0;
  return lm;
}
// does the class have an RB instantiation with room for real reads under the current matrices?
static bool pair_rb_class(miagpu_ctx* c, int kb, bool job) {
  if (const char* e = getenv("MIAGPU_PAIR_RB")) if (atoi(e) == 0) return false;
  if (!pair_rb_built(kb, job)) return false;
  return p16_rb_frame(P16_COLS[kb] / P16_G, c->pssm_max).room >= 16384;
}
// longest read every pair class takes at all: the RB frame holds any read of the class's width
static PairLmax pair_lmax(miagpu_ctx* c, bool job = false) {
  PairLmax lm = pair_lmax_low(c);
  for (int kb = 0; kb < P16_NKB; kb++)
    if (lm.v[kb] > 0 && pair_rb_class(c, kb, job)) lm.v[kb] = P16_MAXL;
  return lm;
}

static void realign_reset_stats(miagpu_ctx* c) {
  c->launches = 0;
  c->dp_cells = 0;
  c->n_fallback = 0;
  for (int kb = 0; kb < P16_NKB; kb++) { c->pair_ms[kb] = 0; c->pair_reads[kb] = 0; c->pair_pairs[kb] = 0; c->pair_cells[kb] = 0; }
  for (int b = 0; b < NBUCKET; b++) { c->bucket_ms[b] = 0; c->bucket_reads[b] = 0; c->bucket_cells[b] = 0; }
}

// window rule + width classes + pair layout of one job on stream st; the meta block is copied to j.h_meta
static int realign_classify(miagpu_ctx* c, const RealignJob& j, cudaStream_t st) {
  if (j.n == 0) return 1;
  PairLmax lm = pair_lmax(c);
  if (c->hp) for (int kb = 0; kb < P16_NKB; kb++) lm.v[kb] = 0;      // mia -h: no read is pair-eligible
  MIAGPU_CUDA(cudaMemsetAsync(j.d_meta, 0, META_WORDS * sizeof(int32_t), st));
  classify_kernel<<<(unsigned)((j.n + 255) / 256), 256, 0, st>>>(j.n, c->d_off.p + j.lo, c->d_as.p + j.lo, c->d_ae.p + j.lo, c->wrap_len, lm,
                                                                c->d_win_start.p + j.lo, c->d_win_len.p + j.lo, j.d_lists, c->d_kind.p + j.lo, j.d_meta,
                                                                c->explicit_windows ? 1 : 0, (c->fs_on && !c->explicit_windows) ? c->d_known.p + j.lo : nullptr);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches++;
  if (lm.v[0] > 0) {
    pair_layout_kernel<<<1, LAYOUT_THREADS, 0, st>>>(j.d_meta);
    MIAGPU_CUDA(cudaGetLastError());
    c->launches++;
  }
  MIAGPU_CUDA(cudaMemcpyAsync(j.h_meta, j.d_meta, sizeof(int32_t) * META_HOST, cudaMemcpyDeviceToHost, st));
  return 1;
}

// the DP kernels of one job on c->stream; j.h_meta must have arrived
static int realign_launch(miagpu_ctx* c, const RealignJob& j) {
  const int64_t n = j.n, lo = j.lo;
  if (n == 0) return 1;
  const int32_t* meta = j.h_meta;
  const PairLmax lm_low = pair_lmax_low(c);
  const bool concurrent = !j.timed && !getenv("MIAGPU_SERIAL_LAUNCH") && !c->hp;     // the chunked kernel's launches share their scratch
  int rr = 0;
  int64_t cells[NBUCKET], pcells[P16_NKB];
  memcpy(cells, meta + META_CELLS, sizeof(cells));
  memcpy(pcells, meta + META_PCELLS, sizeof(pcells));
  for (int b = 0; b < NBUCKET; b++) { c->bucket_cells[b] += cells[b]; c->dp_cells += cells[b]; }
  int pair_items[P16_NKB];
  int total_pairs = 0;                               // pair slots of all classes (a work item holds P16_NP pairs)
  for (int kb = 0; kb < P16_NKB; kb++) {
    pair_items[kb] = meta[META_NPAIRS + kb];
    c->pair_pairs[kb] += pair_items[kb]; c->pair_reads[kb] += meta[META_PREADS + kb]; c->pair_cells[kb] += pcells[kb];
    total_pairs += pair_items[kb] * P16_NP;
  }

  // ---- 16-bit pair kernels first: the reads they cannot finish join the 32-bit lists
  if (total_pairs) {
    MIAGPU_CUDA(cudaMemsetAsync(j.d_pairs, 0xff, (size_t)2 * total_pairs * sizeof(int32_t), c->stream));
    pair_scatter_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(n, c->d_off.p + lo, c->d_kind.p + lo, j.d_meta, j.d_pairs);
    MIAGPU_CUDA(cudaGetLastError());
    c->launches++;
    int base_of[P16_NKB], base = 0, order[P16_NKB];
    for (int kb = 0; kb < P16_NKB; kb++) { base_of[kb] = base; base += pair_items[kb] * P16_NP; order[kb] = kb; }   // in pair slots
    if (concurrent) {                                 // biggest class first: the small ones fill its tail
      std::sort(order, order + P16_NKB, [&](int a, int b) { return pcells[a] > pcells[b]; });
      if (!fork_streams(c, 0)) return 0;
    }
    for (int oi = 0; oi < P16_NKB; oi++) {
      const int kb = order[oi];
      const int ni = pair_items[kb];
      if (!ni) continue;
      const int base = base_of[kb];
      pick_stream(c, concurrent, rr);
      if (j.timed) MIAGPU_CUDA(cudaEventRecord(c->pev[2 * kb], c->stream));
      Pair16Params p{};
      p.bases = c->d_bases.p; p.off = c->d_off.p + lo; p.rc = c->d_rc.p + lo; p.win_start = c->d_win_start.p + lo; p.win_len = c->d_win_len.p + lo;
      p.win_len_narrow = getenv("MIAGPU_NO_NARROW") ? nullptr : c->d_win_len.p + lo;
      p.pairs = j.d_pairs + 2 * (int64_t)base; p.n_items = j.d_meta + META_NPAIRS + kb; p.counter = j.d_meta + META_PWORK + kb;
      p.ref_codes = c->d_ref.p; p.ref_bytes = c->ref_bytes; p.prof16 = c->d_prof16.p;
      p.score = c->d_score.p + lo; p.as_out = c->d_as_out.p + lo; p.ae_out = c->d_ae_out.p + lo; p.abr = c->d_abr.p + lo;
      p.n_runs = c->d_nruns.p + lo; p.runs = c->d_runs.p + lo * MAX_RUNS; p.status = c->d_status.p + lo;
      p.lists = j.d_lists; p.list_counts = j.d_meta + META_COUNT; p.n_reads = n; p.n_fallback = j.d_meta + META_NFALL;
      const bool rb = meta[META_PMAXL + kb] > lm_low.v[kb];         // a read of the class is beyond the low frame: the whole class takes the RB frame
      if (!launch_pair_class<false>(c, p, kb, rb, ni)) return 0;
      if (j.timed) MIAGPU_CUDA(cudaEventRecord(c->pev[2 * kb + 1], c->stream));
    }
    if (concurrent && !join_streams(c, 0)) return 0;
  }

  // ---- 32-bit kernels over the direct lists plus whatever the pair kernels appended
  if (concurrent && !fork_streams(c, 4)) return 0;
  // A read the pair kernels hand over arrives with the window cut at its end cell (pair16.cuh), i.e. in its own bucket or a narrower
  // one: the bound of a list's final length and of its longest read take in the pair-eligible reads of every wider bucket.
  int pop_ub[NBUCKET], maxL_ub[NBUCKET];
  {
    int wider = 0, widerL = 0;                        // pair-eligible reads of the buckets >= b, their longest read
    for (int b = NBUCKET - 1; b >= 0; b--) {
      const int elig = total_pairs && b != NBUCKET - 1 ? meta[META_POP + b] - meta[META_COUNT + b] : 0;
      if (elig > 0) { wider += elig; widerL = std::max(widerL, meta[META_MAXL + b]); }
      pop_ub[b] = meta[META_COUNT + b] + (b != NBUCKET - 1 ? wider : 0);
      maxL_ub[b] = std::max(meta[META_MAXL + b], b != NBUCKET - 1 ? widerL : 0);
    }
  }
  for (int b = 0; b < NBUCKET; b++) {
    const int pop = pop_ub[b];                        // upper bound of the final list length
    if (!pop) continue;
    if (!total_pairs && !meta[META_COUNT + b]) continue;
    pick_stream(c, concurrent, rr);
    if (j.timed) MIAGPU_CUDA(cudaEventRecord(c->bev[2 * b], c->stream));
    RealignParams p{};
    p.bases = c->d_bases.p; p.off = c->d_off.p + lo; p.rc = c->d_rc.p + lo;
    p.win_start = c->d_win_start.p + lo; p.win_len = c->d_win_len.p + lo;
    p.list = j.d_lists + (int64_t)b * n; p.n_list = total_pairs ? pop : meta[META_COUNT + b];
    p.n_list_ptr = j.d_meta + META_COUNT + b; p.counter = j.d_meta + META_WORK + b;
    p.ref_codes = c->d_ref.p; p.ref_bytes = c->ref_bytes; p.prof = c->d_prof.p; p.sg5 = c->explicit_windows ? c->explicit_sg5 : 1;
    p.score = c->d_score.p + lo; p.as_out = c->d_as_out.p + lo; p.ae_out = c->d_ae_out.p + lo; p.abr = c->d_abr.p + lo;
    p.n_runs = c->d_nruns.p + lo; p.runs = c->d_runs.p + lo * MAX_RUNS; p.status = c->d_status.p + lo;
    p.cells_done = j.timed ? reinterpret_cast<unsigned long long*>(j.d_meta + META_CELLS32) + b : nullptr;
    int ok = 1, maxL = maxL_ub[b];
    if (c->hp) {                                      // mia -h: the chunked kernel, the read's window as the matrix (the widest class: the whole reference)
      if (c->explicit_windows && !c->explicit_sg5) { set_error("homopolymer mode: explicit windows need sg5 = 1"); return 0; }
      ok = launch_strip(c, 2, p.list, meta[META_COUNT + b], j.d_meta + META_WORK + b, lo);
      if (!ok) return 0;
      if (j.timed) MIAGPU_CUDA(cudaEventRecord(c->bev[2 * b + 1], c->stream));
      if (j.timed) c->bucket_reads[b] = -1;
      continue;
    }
    switch (BUCKET_K[b]) {
      case 2: ok = launch_realign<2>(c, p, maxL); break;
      case 4: ok = launch_realign<4>(c, p, maxL); break;
      case 5: ok = launch_realign<5>(c, p, maxL); break;
      case 6: ok = launch_realign<6>(c, p, maxL); break;
      case 7: ok = launch_realign<7>(c, p, maxL); break;
      case 8: ok = launch_realign<8>(c, p, maxL); break;
      case 10: ok = launch_realign<10>(c, p, maxL); break;
      case 12: ok = launch_realign<12>(c, p, maxL); break;
      case 16: ok = launch_realign<16>(c, p, maxL); break;
      default:
        ok = launch_strip(c, 2, p.list, meta[META_COUNT + b], j.d_meta + META_WORK + b, lo);   // too wide for either kernel (its window, or the whole reference, as the matrix): never pair-eligible
    }
    if (!ok) return 0;
    if (j.timed) MIAGPU_CUDA(cudaEventRecord(c->bev[2 * b + 1], c->stream));
    if (j.timed) c->bucket_reads[b] = -1;            // launched; the final list length is read back with the timings
  }
  if (concurrent && !join_streams(c, 4)) return 0;
  return 1;
}

static RealignJob whole_batch_job(miagpu_ctx* c) {
  RealignJob j;
  j.lo = 0; j.n = c->n; j.d_meta = c->d_meta.p; j.d_lists = c->d_lists.p; j.d_pairs = c->d_pairs.p; j.h_meta = c->h_meta; j.timed = true;
  return j;
}

static int realign_device(miagpu_ctx* c, bool timed = true) {
  realign_reset_stats(c);
  if (c->n == 0) return 1;
  RealignJob j = whole_batch_job(c);
  j.timed = timed;
  if (!realign_classify(c, j, c->stream)) return 0;
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  return realign_launch(c, j);
}

static int realign_bucket_times(miagpu_ctx* c) {
  if (c->n == 0) return 1;
  int32_t meta[META_HOST];
  MIAGPU_CUDA(cudaMemcpyAsync(meta, c->d_meta.p, sizeof(meta), cudaMemcpyDeviceToHost, c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  c->n_fallback = meta[META_NFALL];
  int64_t cells32[NBUCKET];
  memcpy(cells32, meta + META_CELLS32, sizeof(cells32));
  for (int b = 0; b < NBUCKET; b++)
    if (c->bucket_reads[b]) {
      c->bucket_reads[b] = meta[META_COUNT + b];
      if (b != NBUCKET - 1) c->bucket_cells[b] = cells32[b];               // what the 32-bit kernel of this bucket computed, not the class's total
      MIAGPU_CUDA(cudaEventElapsedTime(&c->bucket_ms[b], c->bev[2 * b], c->bev[2 * b + 1]));
    }
  for (int kb = 0; kb < P16_NKB; kb++)
    if (c->pair_pairs[kb]) MIAGPU_CUDA(cudaEventElapsedTime(&c->pair_ms[kb], c->pev[2 * kb], c->pev[2 * kb + 1]));
  return 1;
}

static int realign_common(miagpu_ctx* c, const uint8_t* rc, const int32_t* as, const int32_t* ae, int32_t* score,
                          int32_t* as_out, int32_t* ae_out, int32_t* abr, int32_t* n_runs, uint16_t* runs, uint8_t* status,
                          bool time_h2d_from_upload) {
  if (!c || !c->have_pssm || !c->have_ref) { set_error("miagpu_realign: set_pssm and set_reference first"); return 0; }
  misinc_invalidate(c, "a realign has replaced the alignments of that round");
  if (c->n && (!rc || !as || !ae)) { set_error("miagpu_realign: rc/as/ae are required"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n;
  MIAGPU_CUDA(cudaEventRecord(c->ev[0], c->stream));
  if (n) {
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_rc.p, rc, n, cudaMemcpyHostToDevice, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_as.p, as, n * 4, cudaMemcpyHostToDevice, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_ae.p, ae, n * 4, cudaMemcpyHostToDevice, c->stream));
  }
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], c->stream));
  if (!realign_device(c)) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], c->stream));
  if (n) {
    if (score) MIAGPU_CUDA(cudaMemcpyAsync(score, c->d_score.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (as_out) MIAGPU_CUDA(cudaMemcpyAsync(as_out, c->d_as_out.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (ae_out) MIAGPU_CUDA(cudaMemcpyAsync(ae_out, c->d_ae_out.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (abr) MIAGPU_CUDA(cudaMemcpyAsync(abr, c->d_abr.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (n_runs) MIAGPU_CUDA(cudaMemcpyAsync(n_runs, c->d_nruns.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (runs) MIAGPU_CUDA(cudaMemcpyAsync(runs, c->d_runs.p, n * MAX_RUNS * 2, cudaMemcpyDeviceToHost, c->stream));
    if (status) MIAGPU_CUDA(cudaMemcpyAsync(status, c->d_status.p, n, cudaMemcpyDeviceToHost, c->stream));
  }
  MIAGPU_CUDA(cudaEventRecord(c->ev[3], c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  float h2d = 0;
  MIAGPU_CUDA(cudaEventElapsedTime(&h2d, c->ev[0], c->ev[1]));
  c->ms_h2d = time_h2d_from_upload ? c->ms_h2d + h2d : h2d;
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_kernels, c->ev[1], c->ev[2]));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_d2h, c->ev[2], c->ev[3]));
  return realign_bucket_times(c);
}

extern "C" int miagpu_realign(miagpu_ctx* c, const uint8_t* rc, const int32_t* as, const int32_t* ae, int32_t* score,
                              int32_t* as_out, int32_t* ae_out, int32_t* abr, int32_t* n_runs, uint16_t* runs, uint8_t* status) {
  return realign_common(c, rc, as, ae, score, as_out, ae_out, abr, n_runs, runs, status, false);
}

extern "C" int miagpu_realign_host(miagpu_ctx* c, int64_t n, const uint8_t* bases, const int64_t* offsets, const uint8_t* rc,
                                   const int32_t* as, const int32_t* ae, int32_t* score, int32_t* as_out, int32_t* ae_out,
                                   int32_t* abr, int32_t* n_runs, uint16_t* runs, uint8_t* status) {
  if (!miagpu_upload_reads(c, n, bases, offsets)) return 0;
  return realign_common(c, rc, as, ae, score, as_out, ae_out, abr, n_runs, runs, status, true);
}

// 8f4: the bare dyn_prog client sequence (ccheck.cc:571-603): pop_s1c_in_a / pop_s2c_in_a / dyn_prog / max_sg_score /
// find_align_begin / populate_pwaln_to_begin of every resident read against ITS OWN stretch of the resident reference,
// unmasked, no window rule.  Runs the 32-bit kernels (realign.cuh) for every read.
extern "C" int miagpu_align_windows(miagpu_ctx* c, const uint8_t* rc, const int32_t* win_start, const int32_t* win_len, int sg5,
                                    int32_t* score, int32_t* as_out, int32_t* ae_out, int32_t* abr, int32_t* n_runs, uint16_t* runs,
                                    uint8_t* status) {
  if (!c || !c->have_pssm || !c->have_ref) { set_error("miagpu_align_windows: set_pssm and set_reference first"); return 0; }
  misinc_invalidate(c, "miagpu_align_windows has replaced the alignments of that round");
  const int64_t n = c->n;
  if (n && (!rc || !win_start || !win_len)) { set_error("miagpu_align_windows: rc / win_start / win_len are required"); return 0; }
  std::vector<int32_t> win_end((size_t)n);
  for (int64_t i = 0; i < n; i++) {
    if (win_start[i] < 0 || win_len[i] < 1 || (int64_t)win_start[i] + win_len[i] > c->wrap_len) {
      set_error("miagpu_align_windows: window %lld = [%d, %d + %d) leaves the reference (%d columns)", (long long)i, win_start[i],
                win_start[i], win_len[i], c->wrap_len);
      return 0;
    }
    win_end[i] = win_start[i] + win_len[i];
  }
  c->explicit_windows = true;
  c->explicit_sg5 = sg5 ? 1 : 0;
  const int ok = realign_common(c, rc, win_start, win_end.data(), score, as_out, ae_out, abr, n_runs, runs, status, false);
  c->explicit_windows = false;
  return ok;
}

extern "C" int miagpu_last_timing(miagpu_ctx* c, float* ms_kernels, float* ms_h2d, float* ms_d2h, int64_t* dp_cells, int32_t* launches) {
  if (!c) { set_error("miagpu_last_timing: NULL ctx"); return 0; }
  if (ms_kernels) *ms_kernels = c->ms_kernels;
  if (ms_h2d) *ms_h2d = c->ms_h2d;
  if (ms_d2h) *ms_d2h = c->ms_d2h;
  if (dp_cells) *dp_cells = c->dp_cells;
  if (launches) *launches = c->launches;
  return 1;
}

extern "C" int miagpu_last_buckets(miagpu_ctx* c, int32_t* k, int32_t* reads, int64_t* cells, float* ms) {
  if (!c) { set_error("miagpu_last_buckets: NULL ctx"); return 0; }
  for (int b = 0; b < NBUCKET; b++) {
    if (k) k[b] = BUCKET_K[b];
    if (reads) reads[b] = c->bucket_reads[b];
    if (cells) cells[b] = c->bucket_cells[b];
    if (ms) ms[b] = c->bucket_ms[b];
  }
  return 1;
}

extern "C" int miagpu_last_pair_buckets(miagpu_ctx* c, int32_t* k, int32_t* reads, int32_t* pairs, int64_t* cells, float* ms, int32_t* fallback_reads, int32_t* max_len16) {
  if (!c) { set_error("miagpu_last_pair_buckets: NULL ctx"); return 0; }
  for (int kb = 0; kb < P16_NKB_WIDE; kb++) {            // MIAGPU_NPAIRCLASS slots: the classes realign windows use
    if (k) k[kb] = P16_COLS[kb] / P16_G;
    if (reads) reads[kb] = c->pair_reads[kb];
    if (pairs) pairs[kb] = c->pair_pairs[kb];
    if (cells) cells[kb] = c->pair_cells[kb];
    if (ms) ms[kb] = c->pair_ms[kb];
  }
  if (fallback_reads) *fallback_reads = c->n_fallback;
  if (max_len16) *max_len16 = c->lmax16;
  return 1;
}

// Device-resident round: rc/as/ae already on the device (from miagpu_realign / _set_alignment_inputs);
// nothing crosses PCIe except the consensus string.
extern "C" int miagpu_set_alignment_inputs(miagpu_ctx* c, const uint8_t* rc, const int32_t* as, const int32_t* ae) {
  if (!c || (c->n && (!rc || !as || !ae))) { set_error("miagpu_set_alignment_inputs: bad argument"); return 0; }
  misinc_invalidate(c, "miagpu_set_alignment_inputs has replaced the strands of that round's reads");
  MIAGPU_CUDA(cudaSetDevice(c->device));
  if (c->n) {
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_rc.p, rc, c->n, cudaMemcpyHostToDevice, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_as.p, as, c->n * 4, cudaMemcpyHostToDevice, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_ae.p, ae, c->n * 4, cudaMemcpyHostToDevice, c->stream));
  }
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  c->h_rc.assign(rc, rc + c->n);
  return 1;
}

// fs->as / fs->ae / fs->score of the next round are this round's results (mia_main.c:252-256)
extern "C" int miagpu_adopt_alignment(miagpu_ctx* c, int32_t* score, int32_t* as, int32_t* ae) {
  if (!c) { set_error("miagpu_adopt_alignment: no context"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n;
  if (n) {
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_as.p, c->d_as_out.p, n * 4, cudaMemcpyDeviceToDevice, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_ae.p, c->d_ae_out.p, n * 4, cudaMemcpyDeviceToDevice, c->stream));
    if (score) MIAGPU_CUDA(cudaMemcpyAsync(score, c->d_score.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (as) MIAGPU_CUDA(cudaMemcpyAsync(as, c->d_as_out.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (ae) MIAGPU_CUDA(cudaMemcpyAsync(ae, c->d_ae_out.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
  }
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  return 1;
}

// The resident alignment of the last round as miagpu_realign would have returned it (all outputs nullable): what
// miagpu_write_maln needs beside the packed run lists after a one-call round.
extern "C" int miagpu_get_alignment(miagpu_ctx* c, int32_t* score, int32_t* as_out, int32_t* ae_out, int32_t* abr, int32_t* n_runs,
                                    uint8_t* status) {
  if (!c) { set_error("miagpu_get_alignment: no context"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n;
  if (n) {
    if (score) MIAGPU_CUDA(cudaMemcpyAsync(score, c->d_score.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (as_out) MIAGPU_CUDA(cudaMemcpyAsync(as_out, c->d_as_out.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (ae_out) MIAGPU_CUDA(cudaMemcpyAsync(ae_out, c->d_ae_out.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (abr) MIAGPU_CUDA(cudaMemcpyAsync(abr, c->d_abr.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (n_runs) MIAGPU_CUDA(cudaMemcpyAsync(n_runs, c->d_nruns.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (status) MIAGPU_CUDA(cudaMemcpyAsync(status, c->d_status.p, n, cudaMemcpyDeviceToHost, c->stream));
  }
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  return 1;
}

extern "C" int miagpu_realign_resident(miagpu_ctx* c) {
  if (!c || !c->have_pssm || !c->have_ref) { set_error("miagpu_realign_resident: set_pssm and set_reference first"); return 0; }
  misinc_invalidate(c, "miagpu_realign_resident has replaced the alignments of that round");
  MIAGPU_CUDA(cudaSetDevice(c->device));
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], c->stream));
  if (!realign_device(c)) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_kernels, c->ev[1], c->ev[2]));
  c->ms_h2d = c->ms_d2h = 0;
  return realign_bucket_times(c);
}

// Packed run lists: the n_runs[i] valid runs of every read, concatenated in read order.
__global__ void pack_runs_kernel(int64_t n, const int32_t* n_runs, const int64_t* run_off, const uint16_t* runs, uint16_t* packed) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int k = n_runs[i] > 0 ? n_runs[i] : 0;
  const int64_t o = run_off[i];
  for (int j = 0; j < k; j++) packed[o + j] = runs[i * MAX_RUNS + j];
}
__global__ void clamp_runs_kernel(int64_t n, const int32_t* n_runs, int64_t* cnt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) cnt[i] = n_runs[i] > 0 ? n_runs[i] : 0;
  if (i == n) cnt[i] = 0;
}

extern "C" int miagpu_get_runs_packed(miagpu_ctx* c, int64_t* run_off, uint16_t* packed, int64_t capacity, int64_t* total) {
  if (!c || !total) { set_error("miagpu_get_runs_packed: bad argument"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n;
  if (!c->d_off2.reserve(2 * (n + 2))) return 0;
  int64_t* cnt = c->d_off2.p;
  int64_t* offs = c->d_off2.p + (n + 2);
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], c->stream));
  clamp_runs_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, c->stream>>>(n, c->d_nruns.p, cnt);
  size_t tmp = 0;
  MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, cnt, offs, n + 1, c->stream));
  if (!c->d_cub.reserve(tmp + 16)) return 0;
  MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, cnt, offs, n + 1, c->stream));
  int64_t tot = 0;
  MIAGPU_CUDA(cudaMemcpyAsync(&tot, offs + n, 8, cudaMemcpyDeviceToHost, c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  *total = tot;
  if (packed && tot > capacity) { set_error("miagpu_get_runs_packed: %lld runs, capacity %lld", (long long)tot, (long long)capacity); return 0; }
  if (!c->d_packed.reserve(tot + 1)) return 0;
  if (n) pack_runs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(n, c->d_nruns.p, offs, c->d_runs.p, c->d_packed.p);
  MIAGPU_CUDA(cudaGetLastError());
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], c->stream));
  if (run_off) MIAGPU_CUDA(cudaMemcpyAsync(run_off, offs, (n + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
  if (packed && tot) MIAGPU_CUDA(cudaMemcpyAsync(packed, c->d_packed.p, tot * 2, cudaMemcpyDeviceToHost, c->stream));
  MIAGPU_CUDA(cudaEventRecord(c->ev[3], c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_kernels, c->ev[1], c->ev[2]));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_d2h, c->ev[2], c->ev[3]));
  c->launches = 4;
  return 1;
}

// ------------------------------------------------ integer peak micro-benchmark
// 8 independent chains per thread of IADD3 / IMNMX / SEL-style ops, no memory.
__global__ void int_peak_kernel(int* out, int iters, int seed) {
  int a[8];
#pragma unroll
  for (int i = 0; i < 8; i++) a[i] = seed + threadIdx.x * (i + 1);
  int b = seed ^ 0x5bd1e995, c = seed + 77;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      a[i] = a[i] + b + it;               // IADD3
      a[i] = max(a[i], c - i);            // IMNMX
      a[i] = (a[i] > b) ? a[i] - c : a[i] + 3;   // ISETP + SEL(+IADD)
      a[i] = min(a[i], 0x3fffffff);
    }
  }
  int s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s ^= a[i];
  if (s == 0x7fffffff) out[0] = s;
}

extern "C" int miagpu_int32_peak(miagpu_ctx* c, double* ops_per_s) {
  if (!c || !ops_per_s) { set_error("miagpu_int32_peak: NULL argument"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  if (!c->d_meta.reserve(META_WORDS)) return 0;
  const int iters = 4096, threads = 256, blocks = c->num_sms * 8;
  // ops per inner statement group: IADD3(1) + IMNMX(1) + ISETP/SEL/IADD(3) + IMNMX(1) = 6 per chain element
  for (int rep = 0; rep < 2; rep++) {
    MIAGPU_CUDA(cudaEventRecord(c->ev[4], c->stream));
    int_peak_kernel<<<blocks, threads, 0, c->stream>>>(c->d_meta.p + META_WORDS - 4, iters, 12345);
    MIAGPU_CUDA(cudaEventRecord(c->ev[5], c->stream));
    MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  }
  float ms = 0;
  MIAGPU_CUDA(cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]));
  *ops_per_s = (double)blocks * threads * iters * 8.0 * 6.0 / (ms * 1e-3);
  return 1;
}

// --------------------------------------------------------------- consensus
static ConsParams cons_params(miagpu_ctx* c) {
  ConsParams p{};
  p.entries = c->d_entries.p; p.n_entries = c->n_entries;
  p.bases = c->d_bases.p; p.off = c->d_off.p; p.rc = c->d_rc.p; p.abr = c->d_abr.p;
  p.n_runs = c->d_nruns.p; p.runs = c->d_runs.p; p.sm = c->d_sm.p; p.seq_len = c->seq_len;
  p.gaps = c->d_gaps.p; p.ins_off = c->d_ins_off.p; p.acc = c->d_acc.p; p.n_cols = c->n_cols;
  p.n_reads = c->n; p.fz_bases = c->d_fz_bases.p; p.fz_runs = c->d_fz_runs.p; p.fz_nruns = c->d_fz_nruns.p; p.fz_rc = c->d_fz_rc.p;
  return p;
}

// MODE 0 (per-position insert maxima) over the current entry list
static int launch_gaps(miagpu_ctx* c, cudaStream_t st) {
  if (!c->n_entries) return 1;
  ConsParams p = cons_params(c);
  gaps_kernel<<<(unsigned)((c->n_entries + 255) / 256), 256, 0, st>>>(p);          // a warp filters 32 entries
  MIAGPU_CUDA(cudaGetLastError());
  c->launches++;
  return 1;
}

// MODE 1 (base + insert columns) over the current entry list: tile-private shared-memory accumulators when the
// reference is short (many reads per column), global REDs otherwise.
// Small results the host waits for (integer sums, insert-column total, chain blocks, the called consensus) go to PINNED host memory
// by a kernel that stores through the mapped address instead of by cudaMemcpyAsync: a copy queues on the device-to-host copy
// engine behind the bulk downloads of the per-read results (24 MB per 1 M reads in miagpu_iterate_host), and the round then waits
// for a few hundred bytes (measured: 0.09 ms per e2e round).  cudaMallocHost memory is mapped under unified addressing; the stores
// are visible to the host once an event recorded behind the kernel has completed.  bytes is rounded up to whole 32-bit words
// (callers pad).
__global__ void to_host_kernel(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, int64_t words) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (int64_t)gridDim.x * blockDim.x) dst[i] = src[i];
}
static cudaError_t small_to_host(void* host_pinned, const void* dev, size_t bytes, cudaStream_t st) {
  if (((uintptr_t)host_pinned & 3) || ((uintptr_t)dev & 3)) return cudaMemcpyAsync(host_pinned, dev, bytes, cudaMemcpyDeviceToHost, st);
  const int64_t words = (int64_t)(bytes + 3) / 4;
  if (!words) return cudaSuccess;
  to_host_kernel<<<(unsigned)std::min<int64_t>(32, (words + 255) / 256), 256, 0, st>>>(static_cast<uint32_t*>(host_pinned), static_cast<const uint32_t*>(dev), words);
  return cudaGetLastError();
}

static int launch_accumulate(miagpu_ctx* c, cudaStream_t st) {
  if (!c->n_entries) return 1;
  ConsParams p = cons_params(c);
  const int n_tiles = (c->seq_len + TILE_POS - 1) / TILE_POS;
  bool tiles = n_tiles <= MAX_TILES && c->n_entries >= 4096;
  if (const char* e = getenv("MIAGPU_CONS_TILES")) tiles = atoi(e) != 0;
  if (tiles) {
    // d_ent_pos: the records in bin order (TileRec, 8 words each) | [n_entries] tile of every entry | counts[64] | starts[65] | cursors[64]
    const int64_t ne = c->n_entries;
    if (!c->d_ent_pos.reserve(9 * ne + 3 * MAX_TILES + 16)) return 0;
    TileRec* recs = reinterpret_cast<TileRec*>(c->d_ent_pos.p);
    int32_t *ent_tile = c->d_ent_pos.p + 8 * ne, *counts = ent_tile + ne, *starts = counts + MAX_TILES, *cursor = starts + MAX_TILES + 1;
    MIAGPU_CUDA(cudaMemsetAsync(counts, 0, MAX_TILES * sizeof(int32_t), st));
    ent_bin_count_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(p, ent_tile, counts);
    ent_bin_scan_kernel<<<1, 32, 0, st>>>(n_tiles, counts, starts, cursor);
    ent_bin_scatter_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(p, ent_tile, cursor, recs);
    MIAGPU_CUDA(cudaGetLastError());
    const size_t smem = (size_t)TILE_SMEM_INTS * sizeof(int32_t);
    MIAGPU_CUDA(cudaFuncSetAttribute(tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int slices = std::max(1, (2 * c->num_sms + n_tiles - 1) / n_tiles);
    tile_kernel<<<dim3(slices, n_tiles), TILE_THREADS, smem, st>>>(p, recs, starts);
    MIAGPU_CUDA(cudaGetLastError());
    c->launches += 4;
  } else {
    entry_kernel<1><<<(unsigned)((c->n_entries * 32 + 255) / 256), 256, 0, st>>>(p);
    MIAGPU_CUDA(cudaGetLastError());
    c->launches++;
  }
  return 1;
}

extern "C" int miagpu_accumulate_gaps(miagpu_ctx* c, int64_t n_entries, const miagpu_entry* entries, void** dev_gaps, int64_t* n_gaps) {
  if (!c || !c->have_ref || !c->have_pssm) { set_error("miagpu_accumulate_gaps: set_pssm / set_reference / realign first"); return 0; }
  misinc_invalidate(c, "miagpu_accumulate_gaps has replaced the entry list of that round");
  if (n_entries < 0 || (n_entries && !entries)) { set_error("miagpu_accumulate_gaps: bad entries"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  for (int64_t i = 0; i < n_entries; i++) {
    const miagpu_entry& e = entries[i];
    if (e.read < 0 || e.read >= c->n) { set_error("miagpu_accumulate_gaps: entry %lld names read %d of %lld", (long long)i, e.read, (long long)c->n); return 0; }
    if (e.ref_pos < 0 || e.col_begin < 0 || e.col_count < 0 || e.col_count > 2 * MAX_READ || e.col_begin > 2 * MAX_READ) {
      set_error("miagpu_accumulate_gaps: entry %lld has ref_pos %d, columns [%d, +%d)", (long long)i, e.ref_pos, e.col_begin, e.col_count);
      return 0;
    }
  }
  c->launches = 0;
  if (!c->d_entries.reserve(n_entries) || !c->d_gaps.reserve(c->seq_len + 2) || !c->d_ins_off.reserve(c->seq_len + 2)) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->ev[0], c->stream));
  if (n_entries) MIAGPU_CUDA(cudaMemcpyAsync(c->d_entries.p, entries, n_entries * sizeof(miagpu_entry), cudaMemcpyHostToDevice, c->stream));
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], c->stream));
  c->n_entries = n_entries;
  MIAGPU_CUDA(cudaMemsetAsync(c->d_gaps.p, 0, (c->seq_len + 2) * sizeof(int32_t), c->stream));
  if (!launch_gaps(c, c->stream)) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_kernels, c->ev[1], c->ev[2]));
  c->ms_d2h = 0;
  c->cons_stage = 1;
  if (dev_gaps) *dev_gaps = c->d_gaps.p;
  if (n_gaps) *n_gaps = c->seq_len;
  return 1;
}

extern "C" int miagpu_accumulate_counts(miagpu_ctx* c, void** dev_counts, int64_t* n_counts) {
  if (!c || c->cons_stage < 1) { set_error("miagpu_accumulate_counts: call miagpu_accumulate_gaps first"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], c->stream));
  // insert-column layout: exclusive scan of gaps[0..seq_len] (gaps[seq_len] = 0 pad)
  size_t tmp = 0;
  MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, c->d_gaps.p, c->d_ins_off.p, c->seq_len + 1, c->stream));
  if (!c->d_cub.reserve(tmp + 16)) return 0;
  MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, c->d_gaps.p, c->d_ins_off.p, c->seq_len + 1, c->stream));
  int32_t total_ins = 0;
  MIAGPU_CUDA(cudaMemcpyAsync(&total_ins, c->d_ins_off.p + c->seq_len, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  c->n_cols = (int64_t)c->seq_len + total_ins;
  if (!c->d_acc.reserve(c->n_cols * NPLANE) || !c->d_called.reserve(c->n_cols + 16)) return 0;
  MIAGPU_CUDA(cudaMemsetAsync(c->d_acc.p, 0, c->n_cols * NPLANE * sizeof(int32_t), c->stream));
  if (!launch_accumulate(c, c->stream)) return 0;
  c->launches++;                                     // the scan
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  float ms = 0;
  MIAGPU_CUDA(cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]));
  c->ms_kernels += ms;
  c->cons_stage = 2;
  if (dev_counts) *dev_counts = c->d_acc.p;
  if (n_counts) *n_counts = c->n_cols * NPLANE;
  return 1;
}

extern "C" int miagpu_call(miagpu_ctx* c, int cons_code, int32_t* gaps_out, int32_t* counts_out, char* cons_out, int32_t* cons_len) {
  if (!c || c->cons_stage < 2) { set_error("miagpu_call: call miagpu_accumulate_counts first"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  const int64_t nc = c->n_cols;
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], c->stream));
  call_kernel<<<(unsigned)((nc + 255) / 256), 256, 0, c->stream>>>(c->d_acc.p, nc, cons_code, c->d_called.p);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches++;
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], c->stream));
  // pinned staging: the called columns (and the gaps when asked for) come back at full PCIe speed
  const size_t need = (size_t)nc + 16 + (size_t)c->seq_len * sizeof(int32_t);
  if (c->h_call_cap < need) {
    if (c->h_call) cudaFreeHost(c->h_call);
    c->h_call = nullptr; c->h_call_cap = 0;
    MIAGPU_CUDA(cudaMallocHost(&c->h_call, need + need / 8));
    c->h_call_cap = need + need / 8;
  }
  char* called = c->h_call;
  int32_t* gaps = reinterpret_cast<int32_t*>(c->h_call + ((nc + 15) / 16) * 16);
  std::vector<int32_t> ins_off, acc;
  MIAGPU_CUDA(small_to_host(called, c->d_called.p, nc, c->stream));             // (both buffers are padded to whole words)
  if (gaps_out) MIAGPU_CUDA(small_to_host(gaps, c->d_gaps.p, c->seq_len * sizeof(int32_t), c->stream));
  if (counts_out) {
    acc.resize(nc * NPLANE);
    ins_off.resize(c->seq_len + 1);
    MIAGPU_CUDA(cudaMemcpyAsync(ins_off.data(), c->d_ins_off.p, (c->seq_len + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(acc.data(), c->d_acc.p, nc * NPLANE * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  }
  MIAGPU_CUDA(cudaEventRecord(c->ev[3], c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  float ms = 0;
  MIAGPU_CUDA(cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]));
  c->ms_kernels += ms;
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_d2h, c->ev[2], c->ev[3]));
  if (gaps_out) memcpy(gaps_out, gaps, c->seq_len * sizeof(int32_t));
  if (counts_out)
    for (int pos = 0; pos < c->seq_len; pos++)
      for (int pl = 0; pl < NPLANE; pl++) counts_out[(int64_t)pos * NPLANE + pl] = acc[(int64_t)pl * nc + pos + ins_off[pos + 1]];
  // consensus string: columns in layout order, gap calls dropped (mia.c:562-570, 600-601)
  int64_t n = 0;
  for (int64_t i = 0; i < nc; i++) n += called[i] != '-' && called[i] != ' ';
  // the caller's buffer: seq_len * 4 + 4096 bytes by contract (miagpu.h), or what miagpu_set_cons_capacity announced
  const int64_t cap = c->cons_capacity > 0 ? c->cons_capacity : (int64_t)c->seq_len * 4 + 4096;
  if (cons_out && n + 1 > cap) {
    set_error("miagpu_call: the consensus has %lld characters, cons_out holds %lld (miagpu_set_cons_capacity announces a larger buffer)", (long long)n, (long long)cap);
    return 0;
  }
  n = 0;
  for (int64_t i = 0; i < nc; i++)
    if (called[i] != '-' && called[i] != ' ') { if (cons_out) cons_out[n] = called[i]; n++; }
  if (cons_out) cons_out[n] = 0;
  if (cons_len) *cons_len = (int32_t)n;
  return 1;
}

extern "C" int miagpu_set_cons_capacity(miagpu_ctx* c, int64_t bytes) {
  if (!c || bytes < 0) { set_error("miagpu_set_cons_capacity: bad argument"); return 0; }
  c->cons_capacity = bytes;                          // 0 = back to the contract's seq_len * 4 + 4096
  return 1;
}

// Entries built on the device from the resident alignments (every read points at its own
// fresh segments).  dropped_front/back: host arrays of n (nullable = nothing dropped).
extern "C" int miagpu_accumulate_gaps_natural(miagpu_ctx* c, const uint8_t* dropped_front, const uint8_t* dropped_back,
                                              void** dev_gaps, int64_t* n_gaps) {
  if (!c || !c->have_ref || !c->have_pssm) { set_error("miagpu_accumulate_gaps_natural: set_pssm / set_reference / realign first"); return 0; }
  misinc_invalidate(c, "miagpu_accumulate_gaps_natural has replaced the entry list of that round");
  MIAGPU_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n;
  c->launches = 0;
  if (!c->d_entries.reserve(2 * n + 2) || !c->d_gaps.reserve(c->seq_len + 2) || !c->d_ins_off.reserve(c->seq_len + 2) ||
      !c->d_dropf.reserve(n + 1) || !c->d_dropb.reserve(n + 1)) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->ev[0], c->stream));
  if (n && dropped_front) MIAGPU_CUDA(cudaMemcpyAsync(c->d_dropf.p, dropped_front, n, cudaMemcpyHostToDevice, c->stream));
  if (n && dropped_back) MIAGPU_CUDA(cudaMemcpyAsync(c->d_dropb.p, dropped_back, n, cudaMemcpyHostToDevice, c->stream));
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], c->stream));
  c->n_entries = 2 * n;
  MIAGPU_CUDA(cudaMemsetAsync(c->d_gaps.p, 0, (c->seq_len + 2) * sizeof(int32_t), c->stream));
  if (n) {
    natural_entries_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(
        n, c->d_as_out.p, c->d_ae_out.p, c->d_nruns.p, c->d_runs.p, c->d_status.p, c->seq_len, dropped_front ? c->d_dropf.p : nullptr,
        dropped_back ? c->d_dropb.p : nullptr, c->d_entries.p);
    MIAGPU_CUDA(cudaGetLastError());
    c->launches++;
    if (!launch_gaps(c, c->stream)) return 0;
  }
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_kernels, c->ev[1], c->ev[2]));
  c->ms_d2h = 0;
  c->cons_stage = 1;
  if (dev_gaps) *dev_gaps = c->d_gaps.p;
  if (n_gaps) *n_gaps = c->seq_len;
  return 1;
}

extern "C" int miagpu_consensus_natural(miagpu_ctx* c, const uint8_t* dropped_front, const uint8_t* dropped_back, int cons_code,
                                        int32_t* gaps_out, int32_t* counts_out, char* cons_out, int32_t* cons_len) {
  if (!miagpu_accumulate_gaps_natural(c, dropped_front, dropped_back, nullptr, nullptr)) return 0;
  float h2d = c->ms_h2d;
  if (!miagpu_accumulate_counts(c, nullptr, nullptr)) return 0;
  if (!miagpu_call(c, cons_code, gaps_out, counts_out, cons_out, cons_len)) return 0;
  c->ms_h2d = h2d;
  c->misinc_stale = nullptr;
  return 1;
}

// ------------------------------------------------------- host policy (a12)
// find_fsdb_score_cut (fsdb.c:269-383): double-precision sums in FSDB order (scorecut.hpp explains how the two
// rounded chains are evaluated block-wise without changing a bit of the result).
static int host_threads(int64_t n) {
  int t = (int)std::thread::hardware_concurrency();
  t = std::max(1, std::min(t, 8));
  if (const char* e = getenv("MIAGPU_HOST_THREADS")) t = std::max(1, atoi(e));
  return (int)std::min<int64_t>(t, std::max<int64_t>(1, n / 65536));
}

// order-independent part of the regression, mergeable across slices (and across the chunks of a pipeline)
struct CutSums {
  int64_t sx = 0, sy = 0, cnt = 0, bad = -1;
  int32_t best[MAX_READ + 1];
  CutSums() { for (int l = 0; l <= MAX_READ; l++) best[l] = INT_MIN; }
  void scan(const int32_t* seq_len, const int32_t* score, const uint8_t* unique_best, int64_t lo, int64_t hi) {
    // xbar / ybar are sums of integers: exact in double in any order (< 2^53), so they are taken in int64.
    // max slope_delta: for a fixed length the quotient is monotone in the score, so the maximum over reads
    // is the maximum over lengths of the quotient at that length's best score (same doubles, same result).
    for (int64_t i = lo; i < hi; i++)
      if ((!unique_best || unique_best[i]) && score[i] >= FIRST_ROUND_SCORE_CUTOFF) {
        const int l = seq_len[i];
        if (l < 0 || l > MAX_READ) { bad = i; return; }
        sx += l; sy += score[i]; cnt++;
        if (score[i] > best[l]) best[l] = score[i];
      }
  }
  void merge(const CutSums& q) {
    if (q.bad >= 0 && bad < 0) bad = q.bad;
    sx += q.sx; sy += q.sy; cnt += q.cnt;
    for (int l = 0; l <= MAX_READ; l++) best[l] = std::max(best[l], q.best[l]);
  }
};

// xbar / ybar and the per-length tables: the same doubles the reference forms per read (fsdb.c:296-316)
struct CutFit { double xbar, ybar; double dx_of[MAX_READ + 1], dx2_of[MAX_READ + 1]; };
static void cut_fit_tables(const CutSums& S, CutFit& F) {
  F.xbar = (double)S.sx; F.ybar = (double)S.sy;
  F.xbar /= S.cnt; F.ybar /= S.cnt;
  for (int l = 0; l <= MAX_READ; l++) { F.dx_of[l] = l - F.xbar; F.dx2_of[l] = F.dx_of[l] * F.dx_of[l]; }
}
// slope / intercept from the two chains (fsdb.c:318-383)
static void cut_fit_slope(const CutSums& S, const CutFit& F, double ssxy, double ssxx, double* slope, double* intercept) {
  double max_delta = 0;
  const double bf = ssxy / ssxx, ib = F.ybar - bf * F.xbar;
  for (int l = 0; l <= MAX_READ; l++)
    if (S.best[l] != INT_MIN) {
      double d = (S.best[l] - ((bf * l) + ib)) / l;
      if (d > max_delta) max_delta = d;
    }
  *intercept = ib;
  if ((bf - max_delta) > 0) *slope = bf - (max_delta * 2.0);
  else *slope = (double)(bf * (80 / 100.0));                     // SCORE_CUTOFF_BUFFER, params.h:24
}
// min_score_for_len of cull_maln_from_fsdb (mia.c:452-470): the threshold depends on the length only
static void cut_thresholds(int hard_cut, double slope, double intercept, double* min_score) {
  if (slope <= 0) slope = 100.0;
  for (int l = 0; l <= MAX_READ; l++) min_score[l] = hard_cut > 0 ? (double)hard_cut : (double)(intercept + (slope * l));
}

// slope / intercept from the merged sums plus the two rounded chains over all reads in order
static int score_cut_finish(int64_t n, const int32_t* seq_len, const int32_t* score, const uint8_t* unique_best, const CutSums& S,
                            HostTeam& team, double* slope, double* intercept) {
  if (S.bad >= 0) { set_error("miagpu_score_cut: seq_len[%lld] = %d out of range", (long long)S.bad, seq_len[S.bad]); return 0; }
  CutFit F;
  cut_fit_tables(S, F);
  auto used = [&](int64_t i) { return (!unique_best || unique_best[i]) && score[i] >= FIRST_ROUND_SCORE_CUTOFF; };
  const double ssxy = chained_sum(n, [&](int64_t i) { return used(i) ? F.dx_of[seq_len[i]] * (score[i] - F.ybar) : 0.0; }, team);
  const double ssxx = chained_sum(n, [&](int64_t i) { return used(i) ? F.dx2_of[seq_len[i]] : 0.0; }, team);
  cut_fit_slope(S, F, ssxy, ssxx, slope, intercept);
  return 1;
}

static int score_cut_team(int64_t n, const int32_t* seq_len, const int32_t* score, const uint8_t* unique_best, HostTeam& team,
                          double* slope, double* intercept) {
  std::vector<CutSums> parts(team.size());
  team.chunks(n, [&](int t, int64_t lo, int64_t hi) { parts[t].scan(seq_len, score, unique_best, lo, hi); });
  CutSums S;
  for (const CutSums& q : parts) S.merge(q);
  return score_cut_finish(n, seq_len, score, unique_best, S, team, slope, intercept);
}

extern "C" int miagpu_score_cut(int64_t n, const int32_t* seq_len, const int32_t* score, const uint8_t* unique_best,
                                double* slope, double* intercept) {
  if (n < 0 || !seq_len || !score || !slope || !intercept) { set_error("miagpu_score_cut: bad argument"); return 0; }
  HostTeam team(host_threads(n));
  return score_cut_team(n, seq_len, score, unique_best, team, slope, intercept);
}

// The per-read test of cull_maln_from_fsdb (mia.c:418-479): below[i] = score < min_score_for_len.
// sticky (nullable): the caller's dropped flags, updated in place (dropped |= below, H10); newly (nullable):
// below & !dropped-before.
static int cull_flags_team(int64_t n, const int32_t* seq_len, const int32_t* score, int hard_cut, double slope, double intercept,
                           HostTeam& team, uint8_t* below, uint8_t* sticky, uint8_t* newly) {
  double min_score[MAX_READ + 1];
  cut_thresholds(hard_cut, slope, intercept, min_score);
  std::vector<int64_t> bad(team.size(), -1);
  team.chunks(n, [&](int t, int64_t lo, int64_t hi) {
    for (int64_t i = lo; i < hi; i++) {
      const int l = seq_len[i];
      if (l < 0 || l > MAX_READ) { bad[t] = i; return; }
      const uint8_t b = score[i] < min_score[l];
      if (below) below[i] = b;
      if (newly) newly[i] = b & !sticky[i];
      if (sticky) sticky[i] |= b;
    }
  });
  for (int64_t x : bad)
    if (x >= 0) { set_error("miagpu_cull_flags: seq_len[%lld] = %d out of range", (long long)x, seq_len[x]); return 0; }
  return 1;
}

extern "C" int miagpu_cull_flags(int64_t n, const int32_t* seq_len, const int32_t* score, const uint8_t* unique_best, int hard_cut,
                                 int score_cut_set, double slope_in, double intercept_in, uint8_t* below) {
  if (n < 0 || !seq_len || !score || !below) { set_error("miagpu_cull_flags: bad argument"); return 0; }
  double slope = slope_in, intercept = intercept_in;
  HostTeam team(host_threads(n));
  if (!score_cut_set && !score_cut_team(n, seq_len, score, unique_best, team, &slope, &intercept)) return 0;
  return cull_flags_team(n, seq_len, score, hard_cut, slope, intercept, team, below, nullptr, nullptr);
}

extern "C" int miagpu_consensus(miagpu_ctx* c, int64_t n_entries, const miagpu_entry* entries, int cons_code, int32_t* gaps_out,
                                int32_t* counts_out, char* cons_out, int32_t* cons_len) {
  if (!miagpu_accumulate_gaps(c, n_entries, entries, nullptr, nullptr)) return 0;
  float h2d = c->ms_h2d;
  if (!miagpu_accumulate_counts(c, nullptr, nullptr)) return 0;
  if (!miagpu_call(c, cons_code, gaps_out, counts_out, cons_out, cons_len)) return 0;
  c->ms_h2d = h2d;
  c->misinc_stale = nullptr;
  return 1;
}

// ---- damage profile: the misincorporation table of the entry list the last round's consensus walked (misinc_kernel, MODE 3 of
// walk_entry).  Reads the entries, alignments, reads and reference as the round left them and writes only its own buffer.
extern "C" int miagpu_misincorporation(miagpu_ctx* c, int64_t* counts) {
  if (!c || !counts) { set_error("miagpu_misincorporation: NULL argument"); return 0; }
  if (c->misinc_stale) { set_error("miagpu_misincorporation: no table of the last round: %s", c->misinc_stale); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  for (auto& ev : c->misinc_ev) if (!ev) MIAGPU_CUDA(cudaEventCreate(&ev));
  if (!c->d_misinc.reserve(MIAGPU_MISINC_INTS)) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->misinc_ev[0], c->stream));
  MIAGPU_CUDA(cudaMemsetAsync(c->d_misinc.p, 0, MIAGPU_MISINC_INTS * sizeof(unsigned long long), c->stream));
  if (c->n_entries) {
    misinc_kernel<<<(unsigned)((c->n_entries + MISINC_PER_BLOCK - 1) / MISINC_PER_BLOCK), MISINC_THREADS, 0, c->stream>>>(cons_params(c), c->d_ref.p,
                                                                                                                       c->d_misinc.p);
    MIAGPU_CUDA(cudaGetLastError());
  }
  MIAGPU_CUDA(cudaEventRecord(c->misinc_ev[1], c->stream));
  MIAGPU_CUDA(cudaMemcpyAsync(counts, c->d_misinc.p, MIAGPU_MISINC_INTS * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
  MIAGPU_CUDA(cudaEventRecord(c->misinc_ev[2], c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_kernels, c->misinc_ev[0], c->misinc_ev[1]));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_d2h, c->misinc_ev[1], c->misinc_ev[2]));
  c->ms_h2d = 0;
  c->launches = c->n_entries ? 1 : 0;
  return 1;
}


// ------------------------------------------------------------------ FSDB pointer state (slots.cuh)
// grow a device buffer and keep what it holds (the rare paths that append to a round's entry list)
template <typename T>
static int grow_keep(DevBuf<T>& b, size_t need, size_t used, cudaStream_t st) {
  if (need <= b.cap) return 1;
  DevBuf<T> nb;
  if (!nb.reserve(need + need / 4)) return 0;
  if (used && b.p) MIAGPU_CUDA(cudaMemcpyAsync(nb.p, b.p, used * sizeof(T), cudaMemcpyDeviceToDevice, st));
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  b.release();
  b = nb;
  return 1;
}

// -D: number of 'N' in ref[0, x) over the wrapped, upper-cased reference (find_alignable_len, mia.c:69-91)
static int fs_upload_nprefix(miagpu_ctx* c) {
  std::vector<int32_t> pre((size_t)c->wrap_len + 1, 0);
  for (int i = 0; i < c->wrap_len; i++) {
    const char ch = c->raw_wrapped[i];
    pre[i + 1] = pre[i] + (ch == 'N' || ch == 'n');
  }
  if (!c->d_nprefix.reserve(pre.size())) return 0;
  MIAGPU_CUDA(cudaMemcpyAsync(c->d_nprefix.p, pre.data(), pre.size() * 4, cudaMemcpyHostToDevice, c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  return 1;
}

static FsDev fs_dev(miagpu_ctx* c) {
  FsDev f{};
  f.known = c->d_known.p; f.front_slot = c->d_front_slot.p; f.back_slot = c->d_back_slot.p; f.slot_flag = c->d_slot_flag.p;
  f.slot_new = c->d_slot_new.p; f.first = c->d_first.p; f.slot_owner = c->d_slot_owner.p; f.ent_slot = c->d_ent_slot.p;
  f.stale = c->d_stale.p; f.counters = c->d_fs_cnt.p; f.stale_cap = (int32_t)std::min<size_t>(c->d_stale.cap / 3, 0x7fffffff);
  f.slot_base = c->fs_sharded ? c->d_fs_cnt.p + FS_CNT_BASE : nullptr;
  return f;
}

static int fs_reserve_round(miagpu_ctx* c) {
  const int64_t n = c->n;
  const size_t slots = (size_t)c->fs_slot_cap;
  return c->d_first.reserve(n + 2) && c->d_nsl.reserve(n + 2) && c->d_slot_owner.reserve(slots) && c->d_slot_owner_prev.reserve(slots) &&
         c->d_ent_slot.reserve(2 * n + 2) && c->d_stale.reserve(3 * (2 * n + 16)) && c->d_fs_cnt.reserve(FS_CNT_WORDS) &&
         c->d_runs_prev.reserve((size_t)n * MAX_RUNS) && c->d_nruns_prev.reserve(n) && c->d_abr_prev.reserve(n) && c->d_as_prev.reserve(n) &&
         c->d_ae_prev.reserve(n) && c->d_score_prev.reserve(n + 1) && c->d_dropf.reserve(n + 1) && c->d_dropb.reserve(n + 1);
}

// the previous round's alignment stays where it is: this round's results go to the partner buffers
static void fs_begin_round(miagpu_ctx* c) {
  if (c->fs_round > 0) {
    std::swap(c->d_runs, c->d_runs_prev); std::swap(c->d_nruns, c->d_nruns_prev); std::swap(c->d_abr, c->d_abr_prev);
    std::swap(c->d_as_out, c->d_as_prev); std::swap(c->d_ae_out, c->d_ae_prev); std::swap(c->d_slot_owner, c->d_slot_owner_prev);
    c->fs_nslots_prev = c->fs_nslots;
    c->fs_prev_pass1 = false; c->fs_prev_valid = true;
  }
  if (c->n) cudaMemcpyAsync(c->d_score_prev.p, c->d_score.p, c->n * sizeof(int32_t), cudaMemcpyDeviceToDevice, c->stream);   // AlnSeq.score of the slots as they are
  c->fs_round++;
}

// which matrix a->submat points at after the last read of a round (mia_main.c:126-184, H6): a read whose strand is known leaves
// the matrix of its strand; a strand-unknown read is not touched at all in iteration 1 and leaves the strand-reversed matrix
// from iteration 2 on (mia_main.c:151)
static void fs_carry_submat(miagpu_ctx* c) {
  if (!c->fs_distant) return;
  for (int64_t i = c->n - 1; i >= 0; i--) {
    if (c->h_known[i]) { c->fs_submat_rc = c->h_rc[i] ? 1 : 0; return; }
    if (c->fs_round > 1) { c->fs_submat_rc = 1; return; }
  }
}

static int fs_number(miagpu_ctx* c);
static int fs_entries(miagpu_ctx* c, bool has_unique);
static int fs_number_and_entries(miagpu_ctx* c, bool has_unique) { return fs_number(c) && fs_entries(c, has_unique); }

// slot numbers of this round: exclusive scan of the AlnSeqs every read merges, FSDB order (sharded rounds: of this rank's reads)
static int fs_number(miagpu_ctx* c) {
  cudaStream_t main = c->stream;
  const int64_t n = c->n;
  const unsigned grid = (unsigned)((n + 255) / 256);
  MIAGPU_CUDA(cudaMemsetAsync(c->d_fs_cnt.p, 0, FS_CNT_WORDS * sizeof(int32_t), main));
  MIAGPU_CUDA(cudaMemsetAsync(c->d_nsl.p + n, 0, sizeof(int32_t), main));
  fs_nsl_kernel<<<grid, 256, 0, main>>>(n, c->d_known.p, c->d_as.p, c->d_ae.p, c->d_as_out.p, c->d_ae_out.p, c->d_nruns.p, c->d_status.p, c->seq_len,
                                        c->d_nsl.p, c->d_fs_cnt.p);
  size_t tmp = 0;
  MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, c->d_nsl.p, c->d_first.p, n + 1, main));
  if (!c->d_cub.reserve(tmp + 16)) return 0;
  MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, c->d_nsl.p, c->d_first.p, n + 1, main));
  MIAGPU_CUDA(cudaMemcpyAsync(c->d_fs_cnt.p + FS_CNT_NSLOTS, c->d_first.p + n, sizeof(int32_t), cudaMemcpyDeviceToDevice, main));
  MIAGPU_CUDA(cudaGetLastError());
  c->launches += 3;
  return 1;
}

// natural entries with the flags of their slots, slot owners, this round's pointers, the list of stale pointers
static int fs_entries(miagpu_ctx* c, bool has_unique) {
  cudaStream_t main = c->stream;
  const int64_t n = c->n;
  const unsigned grid = (unsigned)((n + 255) / 256);
  if (c->fs_seed_read_flags) {                       // per-read flags of miagpu_set_fsdb( slot numbers = NULL ): they belong to the slots of this numbering
    fs_seed_flags_kernel<<<grid, 256, 0, main>>>(n, c->d_first.p, c->d_nsl.p, c->d_dropf.p, c->d_slot_flag.p);
    c->fs_seed_read_flags = false;
  }
  fs_entries_kernel<<<grid, 256, 0, main>>>(n, fs_dev(c), c->d_as_out.p, c->d_ae_out.p, c->d_nruns.p, c->d_runs.p, c->seq_len,
                                            has_unique ? c->d_unique.p : nullptr, c->d_entries.p);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches += 1;
  return 1;
}

// asp_len (fsdb.c:518-530) of a segment from fs_geom_kernel's record (front_len carries the negative-length quirk)
static inline int fs_asp_len(const int32_t* g, int seg) { return seg ? g[7] - g[6] : g[6]; }

// Resolve this round's stale pointers (see slots.cuh): which content each one sees, the smp parameters every touched slot ends
// up with (the LAST pointer pop_smp_from_FSDB visits writes them), one extra list entry per stale pointer.
static int fs_resolve(miagpu_ctx* c, int n_stale, bool has_unique) {
  cudaStream_t st = c->stream;
  const int64_t n = c->n;
  if (n_stale > (int64_t)c->d_stale.cap / 3) { set_error("miagpu: %d stale AlnSeq pointers overflow the list", n_stale); return 0; }
  if (!c->d_fs_tmp.reserve((size_t)n_stale * 8 * 4 + 64)) return 0;
  int32_t* d_rec = c->d_fs_tmp.p;
  fs_gather_kernel<<<(n_stale + 255) / 256, 256, 0, st>>>(n_stale, c->d_stale.p, c->d_slot_owner.p, c->fs_nslots,
                                                          c->fs_prev_valid ? c->d_slot_owner_prev.p : nullptr, c->fs_nslots_prev, c->d_known.p, c->d_front_slot.p, d_rec);
  MIAGPU_CUDA(cudaGetLastError());
  std::vector<int32_t> rec((size_t)n_stale * 8);
  MIAGPU_CUDA(cudaMemcpyAsync(rec.data(), d_rec, rec.size() * 4, cudaMemcpyDeviceToHost, st));
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  std::vector<int> order(n_stale);
  for (int q = 0; q < n_stale; q++) order[q] = q;
  std::sort(order.begin(), order.end(), [&](int a, int b) {
    return rec[8 * a] != rec[8 * b] ? rec[8 * a] < rec[8 * b] : rec[8 * a + 1] < rec[8 * b + 1];
  });
  // ---- content that is no longer live: frozen already, or frozen now from the previous round's results
  std::vector<int32_t> fz_which, fz_dst;
  std::vector<int64_t> fz_slot;
  for (int q = 0; q < n_stale; q++) {
    const int32_t* r = &rec[8 * q];
    const int64_t k = r[2];
    if (r[3] < 0 && r[7] && c->fs_sharded) {
      set_error("miagpu: sharded rounds: local read %d holds a stale pointer to AlnSeq slot %lld, which a read of another rank owns this round "
                "(a pointer that crosses a shard boundary is not served)", r[0], (long long)k);
      return 0;
    }
    if (r[3] >= 0 || c->fz_of_slot.count(k)) continue;
    if (r[4] < 0) {
      set_error("miagpu: read %d points at AlnSeq slot %lld, which neither this nor the previous round filled%s", r[0], (long long)k,
                c->fs_sharded ? " on this rank (sharded rounds: its last content lives on another rank)" : "");
      return 0;
    }
    c->fz_of_slot[k] = (int)(c->fz.size() + fz_which.size());
    fz_which.push_back(r[4]); fz_dst.push_back((int32_t)(c->fz.size() + fz_which.size() - 1)); fz_slot.push_back(k);
  }
  if (!fz_which.empty()) {
    const size_t m = fz_which.size(), tot = c->fz.size() + m;
    if (!grow_keep(c->d_fz_bases, tot * FZ_BASES, c->fz.size() * FZ_BASES, st) || !grow_keep(c->d_fz_runs, tot * MAX_RUNS, c->fz.size() * MAX_RUNS, st) ||
        !grow_keep(c->d_fz_nruns, tot, c->fz.size(), st) || !grow_keep(c->d_fz_rc, tot, c->fz.size(), st)) return 0;
    DevBuf<int32_t> d_list;
    if (!d_list.reserve(m * 10 + 16)) return 0;
    MIAGPU_CUDA(cudaMemcpyAsync(d_list.p, fz_which.data(), m * 4, cudaMemcpyHostToDevice, st));
    MIAGPU_CUDA(cudaMemcpyAsync(d_list.p + m, fz_dst.data(), m * 4, cudaMemcpyHostToDevice, st));
    const AlnView pv{c->d_as_prev.p, c->d_ae_prev.p, c->d_nruns_prev.p, c->d_runs_prev.p, c->d_abr_prev.p, c->fs_prev_seq_len};
    fs_freeze_kernel<<<(unsigned)((m + 127) / 128), 128, 0, st>>>((int)m, d_list.p, d_list.p + m, pv, c->d_bases.p, c->d_off.p, c->d_rc.p,
                                                                  c->fs_prev_pass1 ? c->d_flip_prev.p : nullptr, c->d_score_prev.p, c->d_fz_bases.p,
                                                                  c->d_fz_runs.p, c->d_fz_nruns.p, c->d_fz_rc.p, d_list.p + 2 * m);
    MIAGPU_CUDA(cudaGetLastError());
    std::vector<int32_t> geo(m * 8);
    MIAGPU_CUDA(cudaMemcpyAsync(geo.data(), d_list.p + 2 * m, m * 32, cudaMemcpyDeviceToHost, st));
    MIAGPU_CUDA(cudaStreamSynchronize(st));
    d_list.release();
    for (size_t q = 0; q < m; q++) {
      const int32_t* g = &geo[8 * q];
      // AlnSeq.num_inputs of a pass-1 AlnSeq is what sg_align leaves in the PWAlnFrag: nothing (mia.c:1558-1573 never sets it) = 0
      c->fz.push_back(miagpu_ctx::FzHost{g[0], g[1], g[2], g[3], g[4], g[5], g[6], c->fs_prev_pass1 ? 0 : 1});
    }
  }
  // ---- geometry of the live segments involved: the targets and the holders' own fresh front segments
  std::vector<int32_t> want;
  std::unordered_map<int32_t, int> at;               // 2 * read + seg -> index into geo
  auto need = [&](int32_t e) { if (e >= 0 && !at.count(e)) { at[e] = (int)want.size(); want.push_back(e); } };
  for (int q = 0; q < n_stale; q++) {
    need(rec[8 * q + 3]);
    if (rec[8 * q + 5]) need(2 * rec[8 * q]);
  }
  std::vector<int32_t> geo(want.size() * 8);
  if (!want.empty()) {
    DevBuf<int32_t> d_w;
    if (!d_w.reserve(want.size() * 9 + 16)) return 0;
    MIAGPU_CUDA(cudaMemcpyAsync(d_w.p, want.data(), want.size() * 4, cudaMemcpyHostToDevice, st));
    const AlnView cv{c->d_as_out.p, c->d_ae_out.p, c->d_nruns.p, c->d_runs.p, c->d_abr.p, c->seq_len};
    fs_geom_kernel<<<(unsigned)((want.size() + 127) / 128), 128, 0, st>>>((int)want.size(), d_w.p, cv, d_w.p + want.size());
    MIAGPU_CUDA(cudaGetLastError());
    MIAGPU_CUDA(cudaMemcpyAsync(geo.data(), d_w.p + want.size(), geo.size() * 4, cudaMemcpyDeviceToHost, st));
    MIAGPU_CUDA(cudaStreamSynchronize(st));
    d_w.release();
  }
  struct Content { int aln, cb, cc, ref_pos, asp, bases, rb; };
  auto live_content = [&](int32_t e) {
    const int32_t* g = &geo[8 * at[e]];
    return Content{e >> 1, g[0], g[1], g[2], fs_asp_len(g, e & 1), g[1] - g[4] + g[3], g[5]};
  };
  auto slot_content = [&](const int32_t* r) {
    if (r[3] >= 0) return live_content(r[3]);
    const int fid = c->fz_of_slot[r[2]];
    const miagpu_ctx::FzHost& z = c->fz[fid];
    return Content{(int)(n + fid), 0, z.cols, z.start, z.cols, z.cols - z.dels, 0};      // inserts freed: mia_main.c:80-92
  };
  // ---- visits of pop_smp_from_FSDB (fsdb.c:542-619) by the holders of stale pointers, in FSDB order.  For a read with front
  // content F and back content B: front_len = asp_len(F), total = asp_len(F) + asp_len(B); the running position starts at 0 in
  // F and goes on in B; a content that begins in mid-alignment (a back segment) has consumed rb read bases before its first column.
  struct Visit { int64_t key; int fl, total, bias, bf; };
  std::unordered_map<int64_t, Visit> last;           // slot -> the last visit
  auto visit = [&](int64_t slot, int64_t key, int fl, int total, int bias, int bf) {
    auto it = last.find(slot);
    if (it == last.end() || it->second.key < key) last[slot] = Visit{key, fl, total, bias, bf};
  };
  struct Ptr { int holder, kind; int64_t slot; Content ct; int32_t live_e; bool listed; };
  std::vector<Ptr> ptrs;
  std::unordered_map<int64_t, int32_t> live_entry;   // slot -> its natural entry
  std::unordered_map<int, char> known_holder;
  for (int a = 0; a < n_stale;) {
    int b = a;
    while (b < n_stale && rec[8 * order[b]] == rec[8 * order[a]]) b++;
    const int i = rec[8 * order[a]];
    const bool known = rec[8 * order[a] + 5] != 0;
    const bool listed = !has_unique || c->h_unique.empty() || c->h_unique[i];
    const int32_t *rf = nullptr, *rb = nullptr;
    for (int q = a; q < b; q++) (rec[8 * order[q] + 1] ? rb : rf) = &rec[8 * order[q]];
    Content F{}, B{};
    int64_t slotF = rec[8 * order[a] + 6];           // front_asp: this round's own slot (known), or the stale pass-1 pointer
    if (known) { F = live_content(2 * i); live_entry[slotF] = 2 * i; known_holder[i] = 1; }   // (a known holder is not split this round)
    else if (rf) { F = slot_content(rf); slotF = rf[2]; }
    else { set_error("miagpu: strand-unknown read %d has no front AlnSeq pointer", i); return 0; }
    if (rb) B = slot_content(rb);
    const int fl = F.asp, bl = rb ? B.asp : 0;
    visit(slotF, 2 * (int64_t)i, fl, fl + bl, -F.rb, 0);
    if (!known) ptrs.push_back(Ptr{i, 0, slotF, F, rf[3], listed});
    if (rb) {
      visit(rb[2], 2 * (int64_t)i + 1, fl, fl + bl, F.bases - B.rb, 1);
      ptrs.push_back(Ptr{i, 1, rb[2], B, rb[3], listed});
    }
    a = b;
  }
  // the owners' own visits of the live slots that stale pointers touch (an owner that holds a stale pointer itself is done above)
  for (int q = 0; q < n_stale; q++) {
    const int32_t* r = &rec[8 * q];
    if (r[3] < 0) continue;
    live_entry[r[2]] = r[3];
    const int j = r[3] >> 1, seg = r[3] & 1;
    if (known_holder.count(j)) continue;
    const int32_t* g = &geo[8 * at[r[3]]];
    visit(r[2], 2 * (int64_t)j + seg, g[6], g[7], 0, seg);
  }
  // ---- every touched live slot's natural entry takes the parameters of the slot's last visit; one extra entry per stale pointer
  // of a listed read (cull_maln_from_fsdb copies front_asp and back_asp of every unique_best read into the list, mia.c:469-476)
  std::vector<int32_t> pat;
  std::vector<miagpu_entry> extra;
  c->fs_extra.clear(); c->fs_patch_host.clear();
  for (auto& kv : last) {
    auto le = live_entry.find(kv.first);
    if (le == live_entry.end()) continue;
    const Visit& v = kv.second;
    const int32_t row[6] = {le->second, v.fl, v.total, v.bias, v.bf, -2};
    pat.insert(pat.end(), row, row + 6);
    c->fs_patch_host.insert(c->fs_patch_host.end(), row, row + 5);
  }
  int64_t n_extra = 0;
  for (const Ptr& p : ptrs) {
    const Visit& v = last[p.slot];
    c->fs_extra.push_back(miagpu_ctx::FsExtra{p.holder, p.kind, (int32_t)p.slot, p.live_e, p.ct.aln >= n ? (int32_t)(p.ct.aln - n) : -1,
                                              v.fl, v.total, v.bias, v.bf, (int32_t)p.listed});
    if (!p.listed) continue;
    miagpu_entry x{};
    x.read = p.ct.aln; x.col_begin = p.ct.cb; x.col_count = p.ct.cc; x.ref_pos = p.ct.ref_pos;
    x.front_len = v.fl; x.total_len = v.total; x.act_bias = v.bias; x.back_formula = (uint8_t)v.bf;
    const int32_t row[6] = {(int32_t)(2 * n + n_extra), v.fl, v.total, v.bias, v.bf, (int32_t)p.slot};
    pat.insert(pat.end(), row, row + 6);
    extra.push_back(x);
    n_extra++;
  }
  if (n_extra) {
    if (!grow_keep(c->d_entries, (size_t)(2 * n + n_extra + 2), (size_t)(2 * n), st) ||
        !grow_keep(c->d_ent_slot, (size_t)(2 * n + n_extra + 2), (size_t)(2 * n), st)) return 0;
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_entries.p + 2 * n, extra.data(), extra.size() * sizeof(miagpu_entry), cudaMemcpyHostToDevice, st));
  }
  if (!pat.empty()) {
    DevBuf<int32_t> d_p;
    if (!d_p.reserve(pat.size() + 16)) return 0;
    MIAGPU_CUDA(cudaMemcpyAsync(d_p.p, pat.data(), pat.size() * 4, cudaMemcpyHostToDevice, st));
    const int m = (int)(pat.size() / 6);
    fs_patch_kernel<<<(m + 255) / 256, 256, 0, st>>>(m, d_p.p, c->d_entries.p, c->d_ent_slot.p, c->d_slot_flag.p);
    MIAGPU_CUDA(cudaGetLastError());
    MIAGPU_CUDA(cudaStreamSynchronize(st));
    d_p.release();
  }
  c->n_entries = 2 * n + n_extra;
  c->fs_n_extra = n_extra;
  return 1;
}

// after the host has this round's counters: status of the reads, slot count, stale pointers
static int fs_after_numbering(miagpu_ctx* c, bool has_unique, const int32_t* cnt, int32_t* total_ins) {
  const int status = cnt[FS_CNT_STATUS];
  c->fs_nslots = c->fs_sharded ? cnt[FS_CNT_TOTAL] : cnt[FS_CNT_NSLOTS];
  c->fs_n_stale = cnt[FS_CNT_STALE];
  c->fs_n_extra = 0;
  c->fs_extra.clear(); c->fs_patch_host.clear();
  if (status) {
    set_error("miagpu: reads came back with status bits 0x%x (more than %d alignment runs, or a window no kernel takes): the round is not usable", status, MAX_RUNS);
    return 0;
  }
  if (c->fs_nslots > c->fs_slot_cap) { set_error("miagpu: %lld AlnSeq slots, room for %lld", (long long)c->fs_nslots, (long long)c->fs_slot_cap); return 0; }
  if (!c->fs_n_stale) return 1;
  if (!fs_resolve(c, (int)c->fs_n_stale, has_unique)) return 0;
  if (c->fs_n_extra && has_unique) {                 // a slot whose owner is not listed may bring inserts into the list through a stale pointer
    ConsParams p = cons_params(c);
    p.entries = c->d_entries.p + 2 * c->n; p.n_entries = c->fs_n_extra;
    gaps_kernel<<<(unsigned)((c->fs_n_extra + 255) / 256), 256, 0, c->stream>>>(p);
    size_t tmp = 0;
    MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, c->d_gaps.p, c->d_ins_off.p, c->seq_len + 1, c->stream));
    if (!c->d_cub.reserve(tmp + 16)) return 0;
    MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, c->d_gaps.p, c->d_ins_off.p, c->seq_len + 1, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(total_ins, c->d_ins_off.p + c->seq_len, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  }
  return 1;
}

// this round's cull through the pointers, the newly flagged slots' base columns back out of the planes, flags made sticky
static int fs_flags_and_undo(miagpu_ctx* c, bool has_unique) {
  cudaStream_t main = c->stream;
  const int64_t n = c->n;
  const unsigned grid = (unsigned)((n + 255) / 256);
  fs_flags_kernel<<<grid, 256, 0, main>>>(n, c->d_seqlen.p, c->d_score.p, c->d_thr.p, has_unique ? c->d_unique.p : nullptr, fs_dev(c), c->d_as_out.p,
                                          c->d_ae_out.p, c->fs_distant ? c->d_nprefix.p : nullptr, c->wrap_len, c->d_cstats.p);
  ConsParams p = cons_params(c);
  fs_undo_kernel<<<(unsigned)((c->n_entries + 255) / 256), 256, 0, main>>>(p, c->d_ent_slot.p, c->d_slot_new.p, c->d_entries.p);
  fs_commit_kernel<<<(unsigned)((c->fs_slot_cap + 255) / 256), 256, 0, main>>>(c->fs_slot_cap, c->d_slot_flag.p, c->d_slot_new.p);
  fs_read_flags_kernel<<<grid, 256, 0, main>>>(n, c->d_front_slot.p, c->d_back_slot.p, c->d_slot_flag.p, c->d_dropf.p, c->d_dropb.p);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches += 4;
  return 1;
}


// ------------------------------------------------------------------ FSDB state: entry points
extern "C" int miagpu_set_fsdb(miagpu_ctx* c, const int32_t* seq_len, const uint8_t* unique_best, const int32_t* score,
                               const uint8_t* strand_known, const int32_t* front_slot, const int32_t* back_slot, int64_t n_slots,
                               const uint8_t* slot_dropped, int distant_ref) {
  if (!c || (c->n && (!seq_len || !score))) { set_error("miagpu_set_fsdb: seq_len and score are required"); return 0; }
  misinc_invalidate(c, "miagpu_set_fsdb has replaced the pointer state of that round");
  if ((front_slot == nullptr) != (back_slot == nullptr) || n_slots < 0) { set_error("miagpu_set_fsdb: front_slot and back_slot come together"); return 0; }
  if (!miagpu_set_cut_inputs(c, seq_len, unique_best, nullptr)) return 0;
  const int64_t n = c->n;
  if (c->h_rc.size() != (size_t)n) { set_error("miagpu_set_fsdb: call miagpu_set_alignment_inputs first"); return 0; }
  cudaStream_t st = c->stream;
  c->fs_slot_cap = std::max<int64_t>(2 * n_slots, 2 * n) + 64;     // (sharded rounds: n_slots counts the slots of ALL ranks; a round takes at most two per read)
  if (!c->d_known.reserve(n + 1) || !c->d_front_slot.reserve(n + 1) || !c->d_back_slot.reserve(n + 1) ||
      !c->d_slot_flag.reserve(c->fs_slot_cap) || !c->d_slot_new.reserve(c->fs_slot_cap) || !fs_reserve_round(c)) return 0;
  c->h_known.assign((size_t)n, 1);
  if (strand_known) for (int64_t i = 0; i < n; i++) c->h_known[i] = strand_known[i] != 0;
  std::vector<int32_t> nat;
  const int32_t *fs = front_slot, *bs = back_slot;
  if (!front_slot) {                                 // no pass-1 numbering: the reads stand for themselves until the first round numbers them
    nat.assign((size_t)2 * n, -1);
    for (int64_t i = 0; i < n; i++) nat[i] = (int32_t)i;
    fs = nat.data(); bs = nat.data() + n;
    if (!n_slots) n_slots = n;
  }
  for (int64_t i = 0; i < n; i++)
    if (fs[i] < 0 || fs[i] >= c->fs_slot_cap || bs[i] < -1 || bs[i] >= c->fs_slot_cap) {
      set_error("miagpu_set_fsdb: read %lld points at slots %d / %d of %lld", (long long)i, fs[i], bs[i], (long long)n_slots);
      return 0;
    }
  MIAGPU_CUDA(cudaMemsetAsync(c->d_slot_flag.p, 0, c->fs_slot_cap, st));
  MIAGPU_CUDA(cudaMemsetAsync(c->d_slot_new.p, 0, c->fs_slot_cap, st));
  MIAGPU_CUDA(cudaMemsetAsync(c->d_slot_owner_prev.p, 0xff, c->fs_slot_cap * sizeof(int32_t), st));
  if (n) {
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_known.p, c->h_known.data(), n, cudaMemcpyHostToDevice, st));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_front_slot.p, fs, n * 4, cudaMemcpyHostToDevice, st));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_back_slot.p, bs, n * 4, cudaMemcpyHostToDevice, st));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_score.p, score, n * 4, cudaMemcpyHostToDevice, st));
    fs_owner_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, c->d_front_slot.p, c->d_back_slot.p, n_slots, c->d_slot_owner_prev.p);
    MIAGPU_CUDA(cudaGetLastError());
  }
  c->fs_seed_read_flags = false;
  if (slot_dropped && front_slot && n_slots) MIAGPU_CUDA(cudaMemcpyAsync(c->d_slot_flag.p, slot_dropped, n_slots, cudaMemcpyHostToDevice, st));
  else if (slot_dropped && n) {                      // per READ: the flags go to the slots the reads take at the first numbering
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_dropf.p, slot_dropped, n, cudaMemcpyHostToDevice, st));
    c->fs_seed_read_flags = true;
  }
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  c->fs_on = true; c->fs_distant = distant_ref ? 1 : 0; c->fs_submat_rc = 0; c->fs_round = 0; c->fs_sharded = false;
  c->fs_nslots = c->fs_nslots_prev = n_slots;
  if (!front_slot) c->fs_prev_valid = false;         // nothing was merged before the first round
  c->fz.clear(); c->fz_of_slot.clear(); c->fs_extra.clear(); c->fs_patch_host.clear();
  c->fs_n_extra = c->fs_n_stale = 0;
  if (c->fs_distant && c->have_ref && !fs_upload_nprefix(c)) return 0;
  return 1;
}

extern "C" int miagpu_get_fsdb(miagpu_ctx* c, uint8_t* strand_known, uint8_t* rc, int32_t* front_slot, int32_t* back_slot,
                               uint8_t* dropped_front, uint8_t* dropped_back, int64_t* n_slots) {
  if (!c || !c->fs_on) { set_error("miagpu_get_fsdb: call miagpu_set_fsdb first"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  const int64_t n = c->n;
  if (n) {
    if (dropped_front || dropped_back) {
      fs_read_flags_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, c->d_front_slot.p, c->d_back_slot.p, c->d_slot_flag.p, c->d_dropf.p, c->d_dropb.p);
      MIAGPU_CUDA(cudaGetLastError());
    }
    if (strand_known) MIAGPU_CUDA(cudaMemcpyAsync(strand_known, c->d_known.p, n, cudaMemcpyDeviceToHost, st));
    if (rc) MIAGPU_CUDA(cudaMemcpyAsync(rc, c->d_rc.p, n, cudaMemcpyDeviceToHost, st));
    if (front_slot) MIAGPU_CUDA(cudaMemcpyAsync(front_slot, c->d_front_slot.p, n * 4, cudaMemcpyDeviceToHost, st));
    if (back_slot) MIAGPU_CUDA(cudaMemcpyAsync(back_slot, c->d_back_slot.p, n * 4, cudaMemcpyDeviceToHost, st));
    if (dropped_front) MIAGPU_CUDA(cudaMemcpyAsync(dropped_front, c->d_dropf.p, n, cudaMemcpyDeviceToHost, st));
    if (dropped_back) MIAGPU_CUDA(cudaMemcpyAsync(dropped_back, c->d_dropb.p, n, cudaMemcpyDeviceToHost, st));
  }
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  if (n_slots) *n_slots = c->fs_nslots;
  return 1;
}

extern "C" int miagpu_last_fsdb_stats(miagpu_ctx* c, int64_t* n_slots, int64_t* stale_pointers, int64_t* extra_entries, int64_t* frozen) {
  if (!c) { set_error("miagpu_last_fsdb_stats: no context"); return 0; }
  if (n_slots) *n_slots = c->fs_nslots;
  if (stale_pointers) *stale_pointers = c->fs_n_stale;
  if (extra_entries) *extra_entries = c->fs_n_extra;
  if (frozen) *frozen = (int64_t)c->fz.size();
  return 1;
}

// -D: the strand-unknown reads' attempts against the whole current reference (mia_main.c:120-174), before the round's realign.
// -D in two steps, so that shards can pass the matrix state (H6) from one to the next between them:
//   _begin  the whole-reference attempts of the local strand-unknown reads on the device (three per read: as stored with either
//           matrix, reverse-complemented with the strand-reversed one); state_after[s] = which matrix the LAST local read leaves
//           in the Alignment when the first one is entered with s (0 = forward, 1 = strand-reversed) -- the identity for a shard
//           without reads, a constant as soon as one read's strand was known before;
//   _end    the chain over the local reads in FSDB order entered with state_in, results applied.
// In the first round (iter_num == 1, mia_main.c:122) nothing is tried: a strand-unknown read is not touched and leaves the matrix alone.
static int distant_after(const miagpu_ctx* c, int s) {
  for (int64_t i = c->n - 1; i >= 0; i--) {
    if (c->h_known[i]) return c->h_rc[i] ? 1 : 0;
    if (c->fs_round >= 1) return 1;                    // tried and still unknown: the reverse attempt's matrix stays (mia_main.c:151)
  }
  return s;
}
// one pass of the chain; apply = false: only the state after the last local read is wanted (h_known / h_rc are put back)
static int distant_chain(miagpu_ctx* c, int state_in, bool apply, std::vector<int32_t>* upd, int64_t* learned) {
  const std::vector<int32_t>& U = c->dr_U;
  const int64_t m = (int64_t)U.size();
  std::vector<uint8_t> sk, sr;
  if (!apply) { sk = c->h_known; sr = c->h_rc; }
  for (int64_t q = 0; q < m; q++) {
    const int32_t i = U[q];
    int state = state_in;                              // read 0: what the read before it (the previous round's last, or the previous shard's) left
    if (i > 0) state = c->h_known[i - 1] ? (c->h_rc[i - 1] ? 1 : 0) : 1;      // (a read that stays unknown leaves the strand-reversed matrix)
    const int64_t fwd = 3 * q + (state ? 1 : 0), rev = 3 * q + 2;
    int known = 0, rc = 0, as = 0, ae = 0, score = c->dr_score[q];
    if (c->dr_sc[fwd] > FIRST_ROUND_SCORE_CUTOFF) { known = 1; rc = 0; as = c->dr_a0[fwd]; ae = c->dr_a1[fwd]; score = c->dr_sc[fwd]; }
    if (c->dr_sc[rev] > FIRST_ROUND_SCORE_CUTOFF && c->dr_sc[rev] > score) { known = 1; rc = 1; as = c->dr_a0[rev]; ae = c->dr_a1[rev]; score = c->dr_sc[rev]; }
    if (known) {
      c->h_known[i] = 1; c->h_rc[i] = (uint8_t)rc;
      if (upd) {
        const int32_t row[6] = {i, rc, as, ae, score, rc};                     // strcpy( fs->seq, tmp_rc ) when the reverse attempt wins
        upd->insert(upd->end(), row, row + 6);
      }
      if (learned) ++*learned;
    }
  }
  const int after = distant_after(c, state_in);
  if (!apply) { c->h_known = sk; c->h_rc = sr; }
  return after;
}

extern "C" int miagpu_distant_retry_begin(miagpu_ctx* c, int64_t* n_tried, int32_t* state_after) {
  if (n_tried) *n_tried = 0;
  if (!c || !c->fs_on || !c->have_ref || !c->have_pssm) { set_error("miagpu_distant_retry: set_pssm, set_reference and miagpu_set_fsdb first"); return 0; }
  misinc_invalidate(c, "miagpu_distant_retry has realigned reads of that round");
  c->dr_U.clear(); c->dr_sc.clear(); c->dr_a0.clear(); c->dr_a1.clear(); c->dr_score.clear();
  c->dr_ready = true;
  if (!c->fs_distant) { if (state_after) { state_after[0] = 0; state_after[1] = 1; } return 1; }
  if (c->fs_round < 1) {                               // iter_num > 1 only (mia_main.c:122)
    if (state_after) { state_after[0] = distant_after(c, 0); state_after[1] = distant_after(c, 1); }
    return 1;
  }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n;
  std::vector<int32_t>& U = c->dr_U;
  for (int64_t i = 0; i < n; i++) if (!c->h_known[i]) U.push_back((int32_t)i);
  const int64_t m = (int64_t)U.size();
  if (n_tried) *n_tried = m;
  if (m) {
    cudaStream_t st = c->stream;
    if (!c->aux && !miagpu_create(&c->aux, c->device)) return 0;
    miagpu_ctx* x = c->aux;
    if (!miagpu_set_pssm(x, c->sm_f)) return 0;
    if (!miagpu_set_reference(x, c->raw_wrapped.c_str(), c->seq_len, c->circular, 0)) return 0;
    x->hp = c->hp;                                     // mia_main.c:132-134, 158-160
    // the scratch batch: three items per read (fs_retry_reads_kernel)
    std::vector<int64_t> off_new((size_t)3 * m + 1, 0);
    for (int64_t q = 0; q < 3 * m; q++) off_new[q + 1] = off_new[q] + c->h_seqlen[U[q / 3]];
    const int64_t total = off_new.back();
    if (!x->d_bases.reserve(total + 16) || !x->d_off.reserve(3 * m + 1) || !reserve_per_read(x, 3 * m) || !c->d_fs_tmp.reserve((size_t)m * 6 + 64)) return 0;
    MIAGPU_CUDA(cudaMemcpyAsync(x->d_off.p, off_new.data(), (3 * m + 1) * 8, cudaMemcpyHostToDevice, st));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_fs_tmp.p, U.data(), m * 4, cudaMemcpyHostToDevice, st));
    fs_retry_reads_kernel<<<(unsigned)((3 * m * 32 + 255) / 256), 256, 0, st>>>((int)m, c->d_fs_tmp.p, c->d_bases.p, c->d_off.p, x->d_off.p, x->d_bases.p);
    MIAGPU_CUDA(cudaGetLastError());
    MIAGPU_CUDA(cudaStreamSynchronize(st));
    x->n = 3 * m; x->total_bases = total; x->cut_inputs_n = -1; x->max_read_len = -1;
    std::vector<uint8_t> vrc((size_t)3 * m), vst((size_t)3 * m);
    std::vector<int32_t> ws((size_t)3 * m, 0), wl((size_t)3 * m, c->wrap_len);
    c->dr_sc.resize((size_t)3 * m); c->dr_a0.resize((size_t)3 * m); c->dr_a1.resize((size_t)3 * m);
    for (int64_t q = 0; q < 3 * m; q++) vrc[q] = q % 3 != 0;
    if (!miagpu_align_windows(x, vrc.data(), ws.data(), wl.data(), 1, c->dr_sc.data(), c->dr_a0.data(), c->dr_a1.data(), nullptr, nullptr, nullptr, vst.data())) return 0;
    for (int64_t q = 0; q < 3 * m; q++)
      if (vst[q] & ~(MIAGPU_ST_RUNS_OVERFLOW | MIAGPU_ST_STR_OVERFLOW)) { set_error("miagpu_distant_retry: whole-reference attempt %lld came back with status 0x%x", (long long)q, vst[q]); return 0; }
    // fs->score of the strand-unknown reads (the reverse attempt must beat it)
    std::vector<int32_t> all((size_t)n);
    MIAGPU_CUDA(cudaMemcpyAsync(all.data(), c->d_score.p, n * 4, cudaMemcpyDeviceToHost, st));
    MIAGPU_CUDA(cudaStreamSynchronize(st));
    c->dr_score.resize((size_t)m);
    for (int64_t q = 0; q < m; q++) c->dr_score[q] = all[U[q]];
  }
  if (state_after)
    for (int s = 0; s < 2; s++) state_after[s] = distant_chain(c, s, false, nullptr, nullptr);
  return 1;
}

extern "C" int miagpu_distant_retry_end(miagpu_ctx* c, int state_in, int64_t* n_learned) {
  if (n_learned) *n_learned = 0;
  if (!c || !c->fs_on || !c->dr_ready) { set_error("miagpu_distant_retry_end: call miagpu_distant_retry_begin first"); return 0; }
  misinc_invalidate(c, "miagpu_distant_retry_end has realigned reads of that round");
  c->dr_ready = false;
  if (state_in != 0 && state_in != 1) { set_error("miagpu_distant_retry_end: state_in is 0 (forward matrix) or 1 (strand-reversed)"); return 0; }
  if (c->dr_U.empty()) return 1;
  MIAGPU_CUDA(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  std::vector<int32_t> upd;
  int64_t learned = 0;
  distant_chain(c, state_in, true, &upd, &learned);    // the chain over the reads in FSDB order: the forward attempt runs with whatever matrix the read before left (H6)
  if (learned) {
    DevBuf<int32_t> d_u;
    if (!d_u.reserve(upd.size() + 16)) return 0;
    MIAGPU_CUDA(cudaMemcpyAsync(d_u.p, upd.data(), upd.size() * 4, cudaMemcpyHostToDevice, st));
    fs_apply_kernel<<<(unsigned)((learned * 32 + 255) / 256), 256, 0, st>>>((int)learned, d_u.p, c->d_known.p, c->d_rc.p, c->d_as.p, c->d_ae.p, c->d_score.p,
                                                                           c->d_bases.p, c->d_off.p);
    MIAGPU_CUDA(cudaGetLastError());
    MIAGPU_CUDA(cudaStreamSynchronize(st));
    d_u.release();
  }
  c->dr_U.clear();
  if (n_learned) *n_learned = learned;
  return 1;
}

// one GPU: the chain is entered with what the last read of the previous round left (fs_carry_submat)
extern "C" int miagpu_distant_retry(miagpu_ctx* c, int64_t* n_tried, int64_t* n_learned) {
  if (n_tried) *n_tried = 0;
  if (n_learned) *n_learned = 0;
  if (!c || !c->fs_on || !c->have_ref || !c->have_pssm) { set_error("miagpu_distant_retry: set_pssm, set_reference and miagpu_set_fsdb first"); return 0; }
  misinc_invalidate(c, "miagpu_distant_retry has realigned reads of that round");
  if (!c->fs_distant || c->fs_round < 1) return 1;   // iter_num > 1 only (mia_main.c:122)
  return miagpu_distant_retry_begin(c, n_tried, nullptr) && miagpu_distant_retry_end(c, c->fs_submat_rc, n_learned);
}

// ---------------------------------------------------- one whole round (a9..a13), score cut on the device
struct Trace {                                       // MIAGPU_TRACE=1: host-side timeline of one iteration call on stderr
  bool on = getenv("MIAGPU_TRACE") != nullptr;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  void mark(const char* what) const {
    if (on) fprintf(stderr, "[miagpu trace] %8.3f ms  %s\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(), what);
  }
};

static int pick_chunks(int64_t n) {
  int ch = (int)std::min<int64_t>(8, std::max<int64_t>(1, (n + 125000) / 250000));
  if (const char* e = getenv("MIAGPU_CHUNKS")) ch = std::max(1, std::min(MAX_CHUNKS, atoi(e)));
  return (int)std::min<int64_t>(ch, std::max<int64_t>(1, n));
}

// pinned staging of the device score cut
struct CutHost {
  CutStatsDev stats;
  CutTables tab;
  double thr[MAX_READ + 1];
  int64_t tot_runs;
  int32_t total_ins;
  long long bad_after;
  int32_t newly_dropped;
  int32_t fs_cnt[FS_CNT_WORDS];
  ShardPrep prep;
};

static int cut_reserve(miagpu_ctx* c, int64_t n) {
  const int64_t nb = (n + CUT_BLOCK - 1) / CUT_BLOCK;
  if (!c->d_cstats.reserve(1) || !c->d_ctab.reserve(1) || !c->d_thr.reserve(MAX_READ + 1) || !c->d_cblk.reserve(nb + 1) || !c->d_fs_cnt.reserve(FS_CNT_WORDS)) return 0;
  if (!c->h_cut) MIAGPU_CUDA(cudaMallocHost(&c->h_cut, sizeof(CutHost)));
  if (c->h_cblk_cap < nb) {
    if (c->h_cblk) cudaFreeHost(c->h_cblk);
    c->h_cblk = nullptr; c->h_cblk_cap = 0;
    MIAGPU_CUDA(cudaMallocHost(&c->h_cblk, sizeof(CutBlockDev) * (nb + nb / 8 + 16)));
    c->h_cblk_cap = nb + nb / 8 + 16;
  }
  return 1;
}

// integer sums + per-length maxima of the reads [lo, hi) on the compute stream (after their DP)
static int cut_launch_stats(miagpu_ctx* c, int64_t lo, int64_t hi, bool has_unique) {
  if (hi <= lo) return 1;
  const unsigned grid = (unsigned)std::min<int64_t>(4 * c->num_sms, (hi - lo + CUT_THREADS * 4 - 1) / (CUT_THREADS * 4));
  cut_stats_kernel<<<grid, CUT_THREADS, 0, c->stream>>>(lo, hi, c->d_seqlen.p, c->d_score.p, has_unique ? c->d_unique.p : nullptr, c->d_cstats.p);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches++;
  return 1;
}

// ---- the phases of a round, one copy each for the one-GPU round (iterate_tail) and the sharded round (miagpu_shard_*).  The policy
// is c->round.  Compute stream unless a phase takes one.

// drains every stream a round puts work on: a round that fails leaves nothing of itself in flight
static int round_abort(miagpu_ctx* c) {
  if (c)
    for (cudaStream_t st : {c->stream, c->s_up, c->s_down, c->s_aux[2]}) cudaStreamSynchronize(st);
  return 0;
}

// a round over resident reads: pointer state (this round's results go to the partner buffers), integer sums zeroed, the DP (ev[1]..ev[2])
static int round_start_resident(miagpu_ctx* c, bool sharded) {
  if (c->fs_on) {
    if (!fs_reserve_round(c)) return 0;
    c->fs_sharded = sharded;
    fs_begin_round(c);
  }
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], c->stream));
  cut_init_kernel<<<1, 256, 0, c->stream>>>(c->d_cstats.p);
  MIAGPU_CUDA(cudaGetLastError());
  if (!realign_device(c, false)) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], c->stream));
  return 1;
}

// entries (with the sticky flags of EARLIER rounds) + per-position insert maxima; none of it depends on this round's cut.  A host-fed
// round's earlier flags arrive on the upload stream (xev[1]).
static int round_entries(miagpu_ctx* c) {
  cudaStream_t main = c->stream;
  const int64_t n = c->n;
  c->n_entries = 2 * n;
  MIAGPU_CUDA(cudaMemsetAsync(c->d_gaps.p, 0, (c->seq_len + 2) * sizeof(int32_t), main));
  if (c->round.host_fed()) MIAGPU_CUDA(cudaStreamWaitEvent(main, c->xev[1], 0));
  if (c->fs_on) {
    if (!fs_number_and_entries(c, c->round.unique_best)) return 0;
  } else {
    MIAGPU_CUDA(cudaMemsetAsync(c->d_fs_cnt.p, 0, FS_CNT_WORDS * sizeof(int32_t), main));
    if (n) {
      status_or_kernel<<<(unsigned)((n + 255) / 256), 256, 0, main>>>(n, c->d_status.p, c->d_nruns.p, c->d_fs_cnt.p + FS_CNT_STATUS);
      natural_entries_kernel<<<(unsigned)((n + 255) / 256), 256, 0, main>>>(n, c->d_as_out.p, c->d_ae_out.p, c->d_nruns.p, c->d_runs.p,
                                                                            c->d_status.p, c->seq_len, c->d_dropf.p, c->d_dropf.p, c->d_entries.p,
                                                                            c->round.unique_best ? c->d_unique.p : nullptr);
      MIAGPU_CUDA(cudaGetLastError());
      c->launches += 2;
    }
  }
  return launch_gaps(c, main);
}

// insert-column layout from the insert maxima; its total and the round's counters go to the host (aev[6])
static int round_layout(miagpu_ctx* c) {
  cudaStream_t main = c->stream;
  CutHost* H = c->h_cut;
  size_t tmp = 0;
  MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, c->d_gaps.p, c->d_ins_off.p, c->seq_len + 1, main));
  if (!c->d_cub.reserve(tmp + 16)) return 0;
  MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, c->d_gaps.p, c->d_ins_off.p, c->seq_len + 1, main));
  MIAGPU_CUDA(small_to_host(&H->total_ins, c->d_ins_off.p + c->seq_len, sizeof(int32_t), main));
  MIAGPU_CUDA(small_to_host(H->fs_cnt, c->d_fs_cnt.p, sizeof(H->fs_cnt), main));
  MIAGPU_CUDA(cudaEventRecord(c->aev[6], main));
  c->launches += 2;
  return 1;
}

// the column planes, sized on the host from the layout (one short wait) and zeroed on st; never a consensus that silently lacks reads
static int round_planes(miagpu_ctx* c, cudaStream_t st) {
  CutHost* H = c->h_cut;
  MIAGPU_CUDA(cudaEventSynchronize(c->aev[6]));
  if (c->fs_on) {
    if (!fs_after_numbering(c, c->round.unique_best, H->fs_cnt, &H->total_ins)) return 0;
  } else if (H->fs_cnt[FS_CNT_STATUS]) {
    set_error("miagpu: reads came back with status bits 0x%x (more than %d alignment runs, or a window no kernel takes): the round is not usable", H->fs_cnt[FS_CNT_STATUS], MAX_RUNS);
    return 0;
  }
  c->n_cols = (int64_t)c->seq_len + H->total_ins;
  if (!c->d_acc.reserve(c->n_cols * NPLANE) || !c->d_called.reserve(c->n_cols + 16)) return 0;
  MIAGPU_CUDA(cudaStreamWaitEvent(st, c->aev[6], 0));
  MIAGPU_CUDA(cudaMemsetAsync(c->d_acc.p, 0, c->n_cols * NPLANE * sizeof(int32_t), st));
  return 1;
}

// this round's flags (cull_maln_from_fsdb, mia.c:452-470), sticky (H10), and the newly dropped reads out of the base columns (xev[2]:
// the flags are final).  Pointer state: through the pointers.  cut_first: the entries take this round's flags, then the one
// accumulation.  Otherwise the columns were accumulated with the earlier flags and the newly dropped reads are taken back out.
static int round_flags(miagpu_ctx* c, double slope, double intercept, bool cut_first) {
  cudaStream_t main = c->stream;
  const int64_t n = c->n;
  CutHost* H = c->h_cut;
  cut_thresholds(c->round.hard_cut, slope, intercept, H->thr);
  MIAGPU_CUDA(cudaMemcpyAsync(c->d_thr.p, H->thr, sizeof(H->thr), cudaMemcpyHostToDevice, main));
  if (n && c->fs_on) {
    if (!fs_flags_and_undo(c, c->round.unique_best)) return 0;
  } else if (n) {
    cut_flags_kernel<<<(unsigned)((n + 255) / 256), 256, 0, main>>>(n, c->d_seqlen.p, c->d_score.p, c->d_thr.p, c->d_dropf.p, cut_first ? c->d_entries.p : nullptr,
                                                                    c->d_cstats.p, c->round.unique_best ? c->d_unique.p : nullptr, c->d_newly.p);
    MIAGPU_CUDA(cudaGetLastError());
    c->launches++;
    if (cut_first) {
      if (!launch_accumulate(c, main)) return 0;
    } else {
      undo_kernel<<<(unsigned)((n + 255) / 256), 256, 0, main>>>(cons_params(c), n, c->d_newly.p, c->d_entries.p);
      MIAGPU_CUDA(cudaGetLastError());
      c->launches++;
    }
  }
  MIAGPU_CUDA(cudaEventRecord(c->xev[2], main));
  return 1;
}

// base calling (consensus_assembly_string); the flags go to the host on the download stream meanwhile
static int round_call(miagpu_ctx* c, int cons_code, uint8_t* dropped, int32_t* gaps_out, char* cons_out, int32_t* cons_len) {
  if (dropped && c->n) {
    MIAGPU_CUDA(cudaStreamWaitEvent(c->s_down, c->xev[2], 0));
    MIAGPU_CUDA(cudaMemcpyAsync(dropped, c->d_dropf.p, c->n, cudaMemcpyDeviceToHost, c->s_down));   // fs mode: AlnSeq.dropped behind front_asp (fs_flags_and_undo)
  }
  c->cons_stage = 2;
  const int launches = c->launches;
  if (!miagpu_call(c, cons_code, gaps_out, nullptr, cons_out, cons_len)) return 0;
  c->launches = launches + 1;
  return 1;
}

// after base calling: the round's timing and fallback count; the device state is now that of a round that called its bases
static int round_end(miagpu_ctx* c) {
  if (c->round.host_fed()) {
    c->ms_h2d = 0; c->ms_kernels = 0; c->ms_d2h = 0;   // the phases overlap: only the caller's wall clock means something
    MIAGPU_CUDA(cudaStreamSynchronize(c->s_up));
    for (int k = 0; k < c->round.host_chunks; k++) {
      int32_t nf = 0;
      MIAGPU_CUDA(cudaMemcpy(&nf, c->d_meta.p + (size_t)META_WORDS * k + META_NFALL, 4, cudaMemcpyDeviceToHost));
      c->n_fallback += nf;
    }
  } else {
    MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_kernels, c->ev[1], c->ev[2]));
    c->ms_h2d = c->ms_d2h = 0;
    MIAGPU_CUDA(cudaMemcpy(&c->n_fallback, c->d_meta.p + META_NFALL, 4, cudaMemcpyDeviceToHost));
    if (c->fs_on) c->fs_prev_seq_len = c->seq_len;   // the geometry of this round's alignments, should the next round have to freeze one
  }
  c->misinc_stale = nullptr;
  return 1;
}

struct IterTail {
  // what the host knows about the reads (fallback blocks of the chains are summed on the host, read by read)
  const int32_t* h_seq_len; const uint8_t* h_unique; const int32_t* h_score; cudaEvent_t scores_on_host;
  int cons_code;
  // outputs (host, nullable)
  uint16_t* packed_runs; int64_t capacity; int64_t* total_runs; uint8_t* dropped; int32_t* gaps_out; char* cons_out; int32_t* cons_len;
  double* slope_out; double* intercept_out;
};

// Everything after the DP of a one-GPU round: score cut (stats kernels already enqueued per chunk), entries, insert maxima,
// column accumulation, base calling.  Compute stream throughout; two short host waits (the integer sums, the blocks).
static int iterate_tail(miagpu_ctx* c, const IterTail& a, const Trace& tr) {
  cudaStream_t main = c->stream, down = c->s_down, side = c->s_aux[2];
  const int64_t n = c->n;
  const bool fit = c->round.fit();
  const bool has_unique = c->round.unique_best;
  CutHost* H = c->h_cut;
  const int64_t nb = (n + CUT_BLOCK - 1) / CUT_BLOCK;
  if (!c->d_newly.reserve(n + 1)) return 0;
  if (fit) {
    MIAGPU_CUDA(small_to_host(&H->stats, c->d_cstats.p, sizeof(CutStatsDev), main));
    MIAGPU_CUDA(cudaEventRecord(c->xev[0], main));
  }
  // ---- packed run lists + entries + per-position insert maxima.  The reads this round drops are taken back out of the planes
  // afterwards (round_flags), so that the column accumulation runs while the host stitches the regression's chains.
  int64_t* cnt = c->d_off2.p;
  int64_t* offs = c->d_off2.p + (n + 2);
  H->tot_runs = 0;
  if (a.packed_runs || a.total_runs) {
    size_t tmp = 0;
    MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, cnt, offs, n + 1, main));
    if (!c->d_cub.reserve(tmp + 16)) return 0;
    clamp_runs_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, main>>>(n, c->d_nruns.p, cnt);
    MIAGPU_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, cnt, offs, n + 1, main));
    MIAGPU_CUDA(small_to_host(&H->tot_runs, offs + n, 8, main));
    c->launches += 3;
  }
  if (!round_entries(c) || !round_layout(c)) return 0;
  tr.mark("entries + insert maxima enqueued");
  // ---- regression: integer sums -> tables -> block kernels (side stream) -> stitch (find_fsdb_score_cut, fsdb.c:269-383)
  CutSums S;
  CutFit F;
  if (fit) {
    MIAGPU_CUDA(cudaEventSynchronize(c->xev[0]));
    tr.mark("integer sums on host");
    S.sx = H->stats.sx; S.sy = H->stats.sy; S.cnt = H->stats.cnt; S.bad = H->stats.bad == LLONG_MAX ? -1 : H->stats.bad;
    memcpy(S.best, H->stats.best, sizeof(S.best));
    if (S.bad >= 0) { set_error("miagpu_score_cut: seq_len[%lld] = %d out of range", (long long)S.bad, a.h_seq_len[S.bad]); return 0; }
    cut_fit_tables(S, F);
    H->tab.ybar = F.ybar;
    memcpy(H->tab.dx, F.dx_of, sizeof(F.dx_of));
    memcpy(H->tab.dx2, F.dx2_of, sizeof(F.dx2_of));
    MIAGPU_CUDA(cudaStreamWaitEvent(side, c->xev[0], 0));                              // the scores are final
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_ctab.p, &H->tab, sizeof(CutTables), cudaMemcpyHostToDevice, side));
    const uint8_t* du = has_unique ? c->d_unique.p : nullptr;
    CutSrc src{};
    src.seq_len = c->d_seqlen.p; src.score = c->d_score.p; src.unique_best = du;
    cut_approx_kernel<false><<<(unsigned)nb, CUT_THREADS, 0, side>>>(n, src, c->d_ctab.p, c->d_cblk.p);
    cut_prefix_kernel<<<1, CUT_PREFIX_THREADS, 0, side>>>(nb, c->d_cblk.p);
    cut_exact_kernel<false><<<(unsigned)nb, CUT_THREADS, 0, side>>>(n, src, c->d_ctab.p, c->d_cblk.p, nullptr, nullptr);
    MIAGPU_CUDA(cudaGetLastError());
    MIAGPU_CUDA(small_to_host(c->h_cblk, c->d_cblk.p, sizeof(CutBlockDev) * nb, side));
    MIAGPU_CUDA(cudaEventRecord(c->aev[7], side));
    c->launches += 2;
  }
  // ---- column accumulation of every read that is not yet dropped (needs the insert-column layout: one short wait)
  if (!round_planes(c, main)) return 0;
  const int64_t tot = H->tot_runs;
  if (a.total_runs) *a.total_runs = tot;
  if (a.packed_runs && tot > a.capacity) { set_error("miagpu_iterate: %lld runs, capacity %lld", (long long)tot, (long long)a.capacity); return 0; }
  if (!c->d_packed.reserve(tot + 1)) return 0;
  // Normally the columns of every read not yet dropped are accumulated while the host stitches the chains, and the few reads this
  // round's cut drops are taken back out afterwards.  When the previous round dropped more than an eighth of the reads (the first
  // rounds on a divergent seed: mia.c:452-470 cuts most of them), the same is likely now: wait for the cut, flag the entries,
  // and accumulate once.  Integer sums: the planes are the same either way.
  // (a cut the caller gave -- -H / -S -N -- is known at once: flags first, always)
  const bool cut_first = !c->fs_on && (!fit || (c->cut_prev_newly >= 0 && c->cut_prev_newly * 8 > n));
  if (!cut_first && !launch_accumulate(c, main)) return 0;
  if (a.packed_runs) {
    pack_runs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, main>>>(n, c->d_nruns.p, offs, c->d_runs.p, c->d_packed.p);
    MIAGPU_CUDA(cudaEventRecord(c->xev[3], main));
    MIAGPU_CUDA(cudaStreamWaitEvent(down, c->xev[3], 0));
    if (tot) MIAGPU_CUDA(cudaMemcpyAsync(a.packed_runs, c->d_packed.p, tot * 2, cudaMemcpyDeviceToHost, down));
    c->launches++;
  }
  tr.mark("accumulation enqueued");
  double slope = c->round.slope, intercept = c->round.intercept;
  if (fit) {
    MIAGPU_CUDA(cudaEventSynchronize(c->aev[7]));
    MIAGPU_CUDA(cudaEventSynchronize(a.scores_on_host));
    tr.mark("chain blocks on host");
    std::vector<ChainBlock> bxy(nb), bxx(nb);
    for (int64_t b = 0; b < nb; b++) {
      const CutBlockDev& B = c->h_cblk[b];
      bxy[b] = ChainBlock{B.approx[0], B.T[0], B.A[0], B.e[0], B.ok[0] != 0};
      bxx[b] = ChainBlock{B.approx[1], B.T[1], B.A[1], B.e[1], B.ok[1] != 0};
    }
    const int32_t* seq_len = a.h_seq_len; const int32_t* score = a.h_score; const uint8_t* ub = a.h_unique;
    auto used = [&](int64_t i) { return (!ub || ub[i]) && score[i] >= FIRST_ROUND_SCORE_CUTOFF; };
    int64_t ser0 = 0, ser1 = 0;
    const double ssxy = chain_stitch(n, [&](int64_t i) { return used(i) ? F.dx_of[seq_len[i]] * (score[i] - F.ybar) : 0.0; }, bxy.data(), nb, &ser0);
    const double ssxx = chain_stitch(n, [&](int64_t i) { return used(i) ? F.dx2_of[seq_len[i]] : 0.0; }, bxx.data(), nb, &ser1);
    c->cut_serial_blocks = ser0 + ser1;
    cut_fit_slope(S, F, ssxy, ssxx, &slope, &intercept);
    tr.mark("chains stitched, slope / intercept known");
  }
  if (a.slope_out) *a.slope_out = slope;
  if (a.intercept_out) *a.intercept_out = intercept;
  if (!round_flags(c, slope, intercept, cut_first)) return 0;
  MIAGPU_CUDA(small_to_host(&H->newly_dropped, &c->d_cstats.p->pad, sizeof(int32_t), main));
  MIAGPU_CUDA(small_to_host(&H->bad_after, &c->d_cstats.p->bad, sizeof(long long), main));
  tr.mark("flags + undo enqueued");
  if (!round_call(c, a.cons_code, a.dropped, a.gaps_out, a.cons_out, a.cons_len)) return 0;
  tr.mark("consensus called and downloaded");
  if (H->bad_after != LLONG_MAX) { set_error("miagpu_cull_flags: seq_len[%lld] = %d out of range", H->bad_after, a.h_seq_len[H->bad_after]); return 0; }
  c->cut_prev_newly = c->fs_on ? -1 : H->newly_dropped;
  MIAGPU_CUDA(cudaStreamSynchronize(down));
  tr.mark("download stream drained");
  return 1;
}

// One iteration of mia_main.c:931-963 for a batch that arrives in host memory: upload, realign every read
// (reiterate_assembly), score cut (cull_maln_from_fsdb), column accumulation and base calling
// (consensus_assembly_string).  Same results as miagpu_realign_host + miagpu_get_runs_packed +
// miagpu_cull_flags + miagpu_consensus_natural called one after the other, as a pipeline over three streams:
//   upload stream   chunk k's reads + rc/as/ae/seq_len, then its classification (window rule, width classes, pairs)
//   compute stream  chunk k's DP kernels as soon as chunk k is classified, then its share of the regression's
//                   integer sums; afterwards entries, insert maxima, column accumulation of every read not yet
//                   dropped, this round's flags, the newly dropped reads taken back out, base calling
//   side stream     the regression's block kernels + their records to the host (the host stitches the chains while the
//                   compute stream accumulates)
//   download stream chunk k's scores (first) and the other per-read outputs while chunk k+1 computes
// upload, per-chunk classification + DP + downloads of a host-resident batch (the front half of a round); returns the
// number of chunks C, 0 on error (the last chunk's "scores on host" event is c->cev[4 * (C - 1) + 2])
static int host_round_front(miagpu_ctx* c, const char* who, int64_t n, const uint8_t* bases, const int64_t* offsets, const uint8_t* rc,
                            const int32_t* as, const int32_t* ae, int32_t* score, int32_t* as_out, int32_t* ae_out, int32_t* abr,
                            int32_t* n_runs, uint8_t* status, const int32_t* seq_len, const uint8_t* unique_best, bool stats,
                            const uint8_t* dropped, const Trace& tr) {
  if (!c || !c->have_pssm || !c->have_ref) { set_error("%s: set_pssm and set_reference first", who); return 0; }
  misinc_invalidate(c, "a new round has started and not ended");
  if (n <= 0 || !bases || !offsets || !rc || !as || !ae || !score || !seq_len || !dropped) { set_error("%s: bad argument", who); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  if (n > 0x7fffffffLL / NBUCKET) { set_error("%s: at most %lld reads per batch", who, 0x7fffffffLL / NBUCKET); return 0; }
  if (offsets[0] != 0) { set_error("%s: offsets[0] must be 0", who); return 0; }
  const int64_t total = offsets[n];
  if (!c->d_bases.reserve(total + 16) || !c->d_off.reserve(n + 1) || !reserve_per_read(c, n)) return 0;
  if (!c->d_entries.reserve(2 * n + 2) || !c->d_gaps.reserve(c->seq_len + 2 + MAX_READ + 8) || !c->d_ins_off.reserve(c->seq_len + 2) ||
      !c->d_dropf.reserve(n + 1) || !c->d_off2.reserve(2 * (n + 2)) || !c->d_seqlen.reserve(n + 1) || !c->d_unique.reserve(n + 1) ||
      !cut_reserve(c, n)) return 0;
  cudaStream_t main = c->stream, up = c->s_up, down = c->s_down;
  const int C = pick_chunks(n);
  tr.mark("buffers reserved");
  realign_reset_stats(c);
  c->n = n; c->total_bases = total; c->cut_inputs_n = -1;
  c->fs_on = false; c->fs_prev_valid = false;
  c->max_read_len = C > 1 ? MAX_READ : -1;            // chunked: the longest read is not known before the last upload
  // the side streams start after whatever the compute stream still has queued
  cut_init_kernel<<<1, 256, 0, main>>>(c->d_cstats.p);
  MIAGPU_CUDA(cudaGetLastError());
  MIAGPU_CUDA(cudaEventRecord(c->ev[0], main));
  MIAGPU_CUDA(cudaStreamWaitEvent(up, c->ev[0], 0));
  MIAGPU_CUDA(cudaStreamWaitEvent(down, c->ev[0], 0));
  // ---- upload stream: every chunk's inputs and classification, then the flags of earlier rounds
  RealignJob jobs[MAX_CHUNKS];
  // the first chunk is half the size of the others: the DP starts after its upload, and from then on the uploads (about
  // twice as fast as the DP) stay ahead
  auto bound = [&](int k) { return k <= 0 ? (int64_t)0 : k >= C ? n : n * (2 * k - 1) / (2 * C - 1); };
  for (int k = 0; k < C; k++) {
    const int64_t lo = bound(k), hi = bound(k + 1);
    RealignJob& j = jobs[k];
    j.lo = lo; j.n = hi - lo; j.d_meta = c->d_meta.p + (size_t)META_WORDS * k; j.d_lists = c->d_lists.p + (size_t)NBUCKET * lo;
    j.d_pairs = c->d_pairs.p + lo + (size_t)k * (8 * P16_KEYS + 64); j.h_meta = c->h_meta + (size_t)META_HOST * k; j.timed = false;
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_bases.p + offsets[lo], bases + offsets[lo], offsets[hi] - offsets[lo], cudaMemcpyHostToDevice, up));
    if (k == 0) MIAGPU_CUDA(cudaMemcpyAsync(c->d_off.p, offsets, sizeof(int64_t), cudaMemcpyHostToDevice, up));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_off.p + lo + 1, offsets + lo + 1, (hi - lo) * sizeof(int64_t), cudaMemcpyHostToDevice, up));   // every element once
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_rc.p + lo, rc + lo, hi - lo, cudaMemcpyHostToDevice, up));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_as.p + lo, as + lo, (hi - lo) * 4, cudaMemcpyHostToDevice, up));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_ae.p + lo, ae + lo, (hi - lo) * 4, cudaMemcpyHostToDevice, up));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_seqlen.p + lo, seq_len + lo, (hi - lo) * 4, cudaMemcpyHostToDevice, up));
    if (unique_best) MIAGPU_CUDA(cudaMemcpyAsync(c->d_unique.p + lo, unique_best + lo, hi - lo, cudaMemcpyHostToDevice, up));
    if (!realign_classify(c, j, up)) return 0;
    MIAGPU_CUDA(cudaEventRecord(c->cev[4 * k], up));
  }
  MIAGPU_CUDA(cudaMemcpyAsync(c->d_dropf.p, dropped, n, cudaMemcpyHostToDevice, up));       // sticky flags of earlier rounds (H10)
  MIAGPU_CUDA(cudaEventRecord(c->xev[1], up));
  tr.mark("uploads + classification enqueued");
  // ---- compute + download streams, chunk by chunk
  for (int k = 0; k < C; k++) {
    const RealignJob& j = jobs[k];
    MIAGPU_CUDA(cudaEventSynchronize(c->cev[4 * k]));           // the chunk's meta block is on the host
    tr.mark("chunk classified");
    MIAGPU_CUDA(cudaStreamWaitEvent(main, c->cev[4 * k], 0));
    if (tr.on && k == 0) MIAGPU_CUDA(cudaEventRecord(c->ev[6], main));
    if (!realign_launch(c, j)) return 0;
    if (tr.on && k == C - 1) MIAGPU_CUDA(cudaEventRecord(c->ev[7], main));
    MIAGPU_CUDA(cudaEventRecord(c->cev[4 * k + 1], main));
    if (stats && !cut_launch_stats(c, j.lo, j.lo + j.n, unique_best != nullptr)) return 0;
    MIAGPU_CUDA(cudaStreamWaitEvent(down, c->cev[4 * k + 1], 0));
    MIAGPU_CUDA(cudaMemcpyAsync(score + j.lo, c->d_score.p + j.lo, j.n * 4, cudaMemcpyDeviceToHost, down));
    MIAGPU_CUDA(cudaEventRecord(c->cev[4 * k + 2], down));            // this chunk's scores
    if (as_out) MIAGPU_CUDA(cudaMemcpyAsync(as_out + j.lo, c->d_as_out.p + j.lo, j.n * 4, cudaMemcpyDeviceToHost, down));
    if (ae_out) MIAGPU_CUDA(cudaMemcpyAsync(ae_out + j.lo, c->d_ae_out.p + j.lo, j.n * 4, cudaMemcpyDeviceToHost, down));
    if (abr) MIAGPU_CUDA(cudaMemcpyAsync(abr + j.lo, c->d_abr.p + j.lo, j.n * 4, cudaMemcpyDeviceToHost, down));
    if (n_runs) MIAGPU_CUDA(cudaMemcpyAsync(n_runs + j.lo, c->d_nruns.p + j.lo, j.n * 4, cudaMemcpyDeviceToHost, down));
    if (status) MIAGPU_CUDA(cudaMemcpyAsync(status + j.lo, c->d_status.p + j.lo, j.n, cudaMemcpyDeviceToHost, down));
  }
  tr.mark("DP + downloads enqueued");
  return C;
}

extern "C" int miagpu_iterate_host(miagpu_ctx* c, int64_t n, const uint8_t* bases, const int64_t* offsets, const uint8_t* rc,
                                   const int32_t* as, const int32_t* ae, int32_t* score, int32_t* as_out, int32_t* ae_out,
                                   int32_t* abr, int32_t* n_runs, uint8_t* status, uint16_t* packed_runs, int64_t capacity,
                                   int64_t* total_runs, const int32_t* seq_len, const uint8_t* unique_best, int hard_cut,
                                   int score_cut_set, double slope, double intercept, uint8_t* dropped, int cons_code,
                                   int32_t* gaps_out, char* cons_out, int32_t* cons_len) {
  const Trace tr;
  RoundPolicy pol{hard_cut, score_cut_set, slope, intercept, unique_best != nullptr};
  const int C = host_round_front(c, "miagpu_iterate_host", n, bases, offsets, rc, as, ae, score, as_out, ae_out, abr, n_runs, status, seq_len,
                                 unique_best, pol.fit(), dropped, tr);
  if (!C) return round_abort(c);
  pol.host_chunks = C;
  c->round = pol;
  IterTail t{};
  t.h_seq_len = seq_len; t.h_unique = unique_best; t.h_score = score; t.scores_on_host = c->cev[4 * (C - 1) + 2]; t.cons_code = cons_code;
  t.packed_runs = packed_runs; t.capacity = capacity; t.total_runs = total_runs; t.dropped = dropped;
  t.gaps_out = gaps_out; t.cons_out = cons_out; t.cons_len = cons_len;
  if (!iterate_tail(c, t, tr)) return round_abort(c);
  if (tr.on) {                                       // device time from the first chunk's DP launch to the last chunk's last DP kernel
    float ms = 0;
    if (cudaEventElapsedTime(&ms, c->ev[6], c->ev[7]) == cudaSuccess) fprintf(stderr, "[miagpu trace] DP of %d chunk(s) on the device: %.3f ms\n", C, ms);
  }
  if (!round_end(c)) return round_abort(c);
  return 1;
}

// The same round over reads, rc/as/ae, seq_len / unique_best and sticky flags that are already resident:
extern "C" int miagpu_set_cut_inputs(miagpu_ctx* c, const int32_t* seq_len, const uint8_t* unique_best, const uint8_t* dropped) {
  if (!c || (c->n && !seq_len)) { set_error("miagpu_set_cut_inputs: bad argument"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n;
  if (!c->d_seqlen.reserve(n + 1) || !c->d_unique.reserve(n + 1) || !c->d_dropf.reserve(n + 1)) return 0;
  c->h_seqlen.assign(seq_len, seq_len + n);
  c->h_unique.clear();
  if (unique_best) c->h_unique.assign(unique_best, unique_best + n);
  if (n) {
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_seqlen.p, seq_len, n * 4, cudaMemcpyHostToDevice, c->stream));
    if (unique_best) MIAGPU_CUDA(cudaMemcpyAsync(c->d_unique.p, unique_best, n, cudaMemcpyHostToDevice, c->stream));
    if (dropped) MIAGPU_CUDA(cudaMemcpyAsync(c->d_dropf.p, dropped, n, cudaMemcpyHostToDevice, c->stream));
    else MIAGPU_CUDA(cudaMemsetAsync(c->d_dropf.p, 0, n, c->stream));
  }
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  c->cut_inputs_n = n;
  return 1;
}

extern "C" int miagpu_reset_dropped(miagpu_ctx* c) {
  if (!c || c->cut_inputs_n != c->n) { set_error("miagpu_reset_dropped: call miagpu_set_cut_inputs first"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  if (c->n) MIAGPU_CUDA(cudaMemsetAsync(c->d_dropf.p, 0, c->n, c->stream));
  return 1;
}

extern "C" int miagpu_iterate_resident(miagpu_ctx* c, int hard_cut, int score_cut_set, double slope, double intercept, int cons_code,
                                       double* slope_out, double* intercept_out, uint8_t* dropped, int32_t* gaps_out, char* cons_out,
                                       int32_t* cons_len) {
  if (!c || !c->have_pssm || !c->have_ref) { set_error("miagpu_iterate_resident: set_pssm and set_reference first"); return 0; }
  misinc_invalidate(c, "a new round has started and not ended");
  if (c->n <= 0 || c->cut_inputs_n != c->n) { set_error("miagpu_iterate_resident: upload reads, alignment inputs and cut inputs first"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n;
  if (!c->d_entries.reserve(2 * n + 2) || !c->d_gaps.reserve(c->seq_len + 2) || !c->d_ins_off.reserve(c->seq_len + 2) ||
      !c->d_off2.reserve(2 * (n + 2)) || !cut_reserve(c, n)) return 0;
  if (c->h_score_cap < n) {
    if (c->h_score) cudaFreeHost(c->h_score);
    c->h_score = nullptr; c->h_score_cap = 0;
    MIAGPU_CUDA(cudaMallocHost(&c->h_score, sizeof(int32_t) * (n + 64)));
    c->h_score_cap = n;
  }
  c->round = RoundPolicy{hard_cut, score_cut_set, slope, intercept, !c->h_unique.empty()};
  const Trace tr;
  if (!round_start_resident(c, false)) return round_abort(c);
  if (c->round.fit()) {
    cudaStream_t down = c->s_down;
    MIAGPU_CUDA(cudaStreamWaitEvent(down, c->ev[2], 0));
    MIAGPU_CUDA(cudaMemcpyAsync(c->h_score, c->d_score.p, n * 4, cudaMemcpyDeviceToHost, down));    // only the chains' unproven blocks read them
    MIAGPU_CUDA(cudaEventRecord(c->cev[2], down));
    if (!cut_launch_stats(c, 0, n, c->round.unique_best)) return round_abort(c);
  }
  tr.mark("DP enqueued");
  IterTail t{};
  t.h_seq_len = c->h_seqlen.data(); t.h_unique = c->round.unique_best ? c->h_unique.data() : nullptr; t.h_score = c->h_score;
  t.scores_on_host = c->cev[2]; t.cons_code = cons_code;
  t.dropped = dropped; t.gaps_out = gaps_out; t.cons_out = cons_out; t.cons_len = cons_len;
  t.slope_out = slope_out; t.intercept_out = intercept_out;
  if (!iterate_tail(c, t, tr) || !round_end(c)) return round_abort(c);
  if (c->fs_on) fs_carry_submat(c);
  return 1;
}

// ------------------------------------------------------------------ sharded rounds (SURVEY 8e)
// One round of mia_main.c:931-963 with the reads sharded over `world` GPUs, one context (one process) per GPU,
// the consensus replicated.  The library does not link a communication library: between the three phases the
// caller runs one collective each on the buffers the library hands out, on miagpu_stream (NCCL in bench.py and
// driver.py; INTEGRATION.md shows the C calls):
//   miagpu_shard_begin[_host]   DP of the local reads; integer sums + per-length maxima of the regression; the local
//                               reads' keys; entries; per-position insert maxima
//       -> all-gather  gather_send -> gather_recv   (stride words per rank)
//       -> all-reduce  MAX over max_buf             (insert maxima + per-length best scores)
//   miagpu_shard_cut            the regression over the gathered keys of every rank in rank order = FSDB order (the
//                               same block-wise exact chains as a single-GPU round, evaluated redundantly on every
//                               rank: identical slope / intercept everywhere), flags of the local reads, insert-column
//                               layout from the reduced maxima, column accumulation of the local reads
//       -> all-reduce  SUM over sum_buf             (the column planes)
//   miagpu_shard_finish         base calling (every rank calls the same bases), downloads
// Integer sums and maxima commute and the chains are evaluated exactly: the results are bit-identical to a
// single-GPU round over the concatenated reads for any number of ranks.
static int shard_reserve(miagpu_ctx* c, int world, int64_t n_max) {
  const int64_t nb = (n_max + CUT_BLOCK - 1) / CUT_BLOCK;                    // chain blocks per rank (the same on every rank)
  // what a rank sends in the all-gather: nb block records | count + SHARD_PF_SLOTS block ids | SHARD_PF_SLOTS blocks of keys
  const int64_t words = (nb * (int64_t)sizeof(ShardBlockRec) + 3) / 4 + (SHARD_PF_SLOTS + 8) + (int64_t)SHARD_PF_SLOTS * CUT_BLOCK;
  c->sh_stride = (words + 3) / 4 * 4;
  c->sh_nb = nb;
  if (!c->d_sh_send.reserve(c->sh_stride) || !c->d_sh_recv.reserve((size_t)world * c->sh_stride) || !c->d_sh_prep.reserve(1) || !cut_reserve(c, nb * CUT_BLOCK)) return 0;
  const size_t need = (size_t)world * c->sh_stride * sizeof(uint32_t);
  if (c->h_sh_cap < need) {
    if (c->h_sh_recv) cudaFreeHost(c->h_sh_recv);
    c->h_sh_recv = nullptr; c->h_sh_cap = 0;
    MIAGPU_CUDA(cudaMallocHost(&c->h_sh_recv, need + need / 8));
    c->h_sh_cap = need + need / 8;
  }
  return 1;
}

// after the DP: this rank's entries and insert maxima, and its header row + insert maxima + best scores for the all-reduce(MAX)
static int shard_after_dp(miagpu_ctx* c, void** max_buf, int64_t* max_words) {
  cudaStream_t main = c->stream;
  const int64_t n = c->n;
  int32_t* best = c->d_gaps.p + c->seq_len + 2;
  int32_t* hdr = best + MAX_READ + 1;
  if (c->fs_on) {
    // pointer state: this rank's slot count goes out with the header; the slots can only be numbered (and the entries take their
    // flags) once every rank's count is back -- miagpu_shard_fit.  The insert maxima need the entries' geometry only.
    c->n_entries = 2 * n;
    MIAGPU_CUDA(cudaMemsetAsync(c->d_gaps.p, 0, (c->seq_len + 2) * sizeof(int32_t), main));
    if (!fs_number(c)) return 0;
    if (n) {
      natural_entries_kernel<<<(unsigned)((n + 255) / 256), 256, 0, main>>>(n, c->d_as_out.p, c->d_ae_out.p, c->d_nruns.p, c->d_runs.p,
                                                                            c->d_status.p, c->seq_len, nullptr, nullptr, c->d_entries.p, nullptr, c->d_known.p);
      MIAGPU_CUDA(cudaGetLastError());
      c->launches++;
    }
    if (!launch_gaps(c, main)) return 0;
  } else if (!round_entries(c)) {
    return 0;
  }
  shard_hdr2_kernel<<<1, 256, 0, main>>>(c->d_cstats.p, best, hdr, c->sh_world, c->sh_rank, (int)n, c->fs_on ? c->d_fs_cnt.p + FS_CNT_NSLOTS : nullptr);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches++;
  if (max_buf) *max_buf = c->d_gaps.p;
  if (max_words) *max_words = c->seq_len + 2 + MAX_READ + 1 + (int64_t)c->sh_world * SHARD_HDR2;
  c->sh_phase = 1;
  return 1;
}

static int shard_args(miagpu_ctx* c, const char* who, int world, int rank, int64_t n_max, int64_t n) {
  if (!c || !c->have_pssm || !c->have_ref) { set_error("%s: set_pssm and set_reference first", who); return 0; }
  misinc_invalidate(c, "a new round has started and not ended");
  if (world < 1 || rank < 0 || rank >= world || n_max < n || n_max < 1) { set_error("%s: bad world / rank / n_max (n_max must be the largest read count of any rank)", who); return 0; }
  if ((int64_t)world * (n_max + CUT_BLOCK) > 0x7fffffffLL * 64) { set_error("%s: too many reads", who); return 0; }
  return 1;
}

static int shard_reserve_common(miagpu_ctx* c, int world, int64_t n_max) {
  const int64_t n = c->n;
  return c->d_entries.reserve(2 * n + 2) && c->d_gaps.reserve(c->seq_len + 2 + MAX_READ + 8 + (size_t)world * SHARD_HDR2) &&
         c->d_ins_off.reserve(c->seq_len + 2) && c->d_off2.reserve(2 * (n + 2)) && c->d_seqlen.reserve(n + 1) && c->d_score.reserve(n + 1) &&
         c->d_newly.reserve(n + 1) && shard_reserve(c, world, n_max);
}

extern "C" int miagpu_shard_begin(miagpu_ctx* c, int world, int rank, int64_t n_max, int hard_cut, int score_cut_set, double slope,
                                  double intercept, void** max_buf, int64_t* max_words) {
  if (!shard_args(c, "miagpu_shard_begin", world, rank, n_max, c ? c->n : 0)) return 0;
  if (c->cut_inputs_n != c->n) { set_error("miagpu_shard_begin: upload reads, alignment inputs and cut inputs first"); return 0; }
  if (c->fs_on && !c->h_unique.empty()) { set_error("miagpu_shard_begin: the pointer state in sharded rounds goes without the repeat filter"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  if (!shard_reserve_common(c, world, n_max)) return 0;
  c->sh_world = world; c->sh_rank = rank; c->sh_phase = 0;
  c->round = RoundPolicy{hard_cut, score_cut_set, slope, intercept, !c->h_unique.empty()};
  if (!round_start_resident(c, true) || !cut_launch_stats(c, 0, c->n, c->round.unique_best) || !shard_after_dp(c, max_buf, max_words)) return round_abort(c);
  return 1;
}

extern "C" int miagpu_shard_begin_host(miagpu_ctx* c, int world, int rank, int64_t n_max, int64_t n, const uint8_t* bases,
                                       const int64_t* offsets, const uint8_t* rc, const int32_t* as, const int32_t* ae, int32_t* score,
                                       int32_t* as_out, int32_t* ae_out, int32_t* abr, int32_t* n_runs, uint8_t* status,
                                       const int32_t* seq_len, const uint8_t* unique_best, const uint8_t* dropped, int hard_cut,
                                       int score_cut_set, double slope, double intercept, void** max_buf, int64_t* max_words) {
  if (!shard_args(c, "miagpu_shard_begin_host", world, rank, n_max, n)) return 0;
  if (c->fs_on) { set_error("miagpu_shard_begin_host: the pointer state goes with resident reads (miagpu_shard_begin)"); return 0; }
  const Trace tr;
  c->sh_phase = 0;
  const int C = host_round_front(c, "miagpu_shard_begin_host", n, bases, offsets, rc, as, ae, score, as_out, ae_out, abr, n_runs, status, seq_len,
                                 unique_best, true, dropped, tr);
  if (!C || !shard_reserve_common(c, world, n_max)) return round_abort(c);
  c->sh_world = world; c->sh_rank = rank;
  c->round = RoundPolicy{hard_cut, score_cut_set, slope, intercept, unique_best != nullptr, C};
  if (!shard_after_dp(c, max_buf, max_words)) return round_abort(c);
  return 1;
}

// After the all-reduce(MAX): this rank's part of the regression -- the sums of all ranks, the tables, the block records of the local
// reads (scorecut.cuh) -- into gather_send for the all-gather; beside it (side stream) the column accumulation of the local reads
// with the flags of earlier rounds, laid out by the reduced insert maxima.  *gather_words = 0: nothing to gather (the cut is given).
extern "C" int miagpu_shard_fit(miagpu_ctx* c, void** gather_send, void** gather_recv, int64_t* gather_words) {
  if (!c || c->sh_phase != 1) { set_error("miagpu_shard_fit: call miagpu_shard_begin first"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  cudaStream_t main = c->stream, side = c->s_aux[2];
  const int64_t n = c->n, nb = c->sh_nb;
  int32_t* best = c->d_gaps.p + c->seq_len + 2;
  int32_t* hdr = best + MAX_READ + 1;
  if (c->fs_on) {
    // every rank's slot count is back: global slot numbers (the ranks' reads one after the other), entries with the flags of their
    // slots, owners of the local slots (-1: another rank's), this round's pointers and the list of stale ones
    fs_base_kernel<<<1, 32, 0, main>>>(c->sh_world, c->sh_rank, hdr, SHARD_HDR2, c->d_fs_cnt.p);
    MIAGPU_CUDA(cudaMemsetAsync(c->d_slot_owner.p, 0xff, (size_t)c->fs_slot_cap * sizeof(int32_t), main));
    if (!fs_entries(c, false)) return round_abort(c);
    c->launches += 2;
  }
  if (!round_layout(c)) return round_abort(c);          // from the reduced maxima
  if (c->round.fit()) {
    uint32_t* send = c->d_sh_send.p;
    ShardBlockRec* recs = reinterpret_cast<ShardBlockRec*>(send);
    int32_t* pf_ids = reinterpret_cast<int32_t*>(send + (nb * sizeof(ShardBlockRec) + 3) / 4);
    uint32_t* pf_keys = reinterpret_cast<uint32_t*>(pf_ids + SHARD_PF_SLOTS + 8);
    shard_prep_kernel<<<1, 256, 0, main>>>(c->sh_world, c->sh_rank, hdr, best, c->d_cstats.p, c->d_ctab.p, c->d_sh_prep.p, pf_ids);
    CutSrc src{};
    src.seq_len = c->d_seqlen.p; src.score = c->d_score.p; src.unique_best = c->round.unique_best ? c->d_unique.p : nullptr;
    cut_approx_kernel<false><<<(unsigned)nb, CUT_THREADS, 0, main>>>(n, src, c->d_ctab.p, c->d_cblk.p);
    cut_prefix_kernel<<<1, CUT_PREFIX_THREADS, 0, main>>>(nb, c->d_cblk.p, c->d_sh_prep.p->start);
    cut_exact_kernel<false><<<(unsigned)nb, CUT_THREADS, 0, main>>>(n, src, c->d_ctab.p, c->d_cblk.p, pf_keys, pf_ids);
    shard_records_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, main>>>(nb, c->d_cblk.p, recs);
    MIAGPU_CUDA(cudaGetLastError());
    c->launches += 5;
  }
  // the column planes (pointer state: stale pointers -> extra entries / patched smp parameters / frozen content, all of it local to
  // this rank), accumulated on the side stream beside the regression.  The planes are followed by nothing yet: the caller
  // all-reduces exactly n_cols * NPLANE words.
  if (!round_planes(c, side) || !launch_accumulate(c, side)) return round_abort(c);
  MIAGPU_CUDA(cudaEventRecord(c->aev[7], side));
  if (gather_send) *gather_send = c->d_sh_send.p;
  if (gather_recv) *gather_recv = c->d_sh_recv.p;
  if (gather_words) *gather_words = c->round.fit() ? c->sh_stride : 0;
  c->sh_phase = 2;
  return 1;
}

extern "C" int miagpu_shard_cut(miagpu_ctx* c, double* slope_out, double* intercept_out, void** sum_buf, int64_t* sum_words) {
  if (!c || c->sh_phase != 2) { set_error("miagpu_shard_cut: call miagpu_shard_fit first"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  cudaStream_t main = c->stream;
  const int64_t stride = c->sh_stride, nb = c->sh_nb;
  const int world = c->sh_world;
  CutHost* H = c->h_cut;
  double slope = c->round.slope, intercept = c->round.intercept;
  if (c->round.fit()) {
    // every rank's records, ids and the first SHARD_PF_FIRST key blocks in one strided copy; the other key blocks only if a rank used them
    const size_t pitch = (size_t)stride * sizeof(uint32_t);
    const size_t ids_at = ((size_t)nb * sizeof(ShardBlockRec) + 3) / 4 * 4;
    const size_t first = ids_at + (size_t)(SHARD_PF_SLOTS + 8) * 4 + (size_t)SHARD_PF_FIRST * CUT_BLOCK * 4;
    MIAGPU_CUDA(cudaMemcpy2DAsync(c->h_sh_recv, pitch, c->d_sh_recv.p, pitch, first, world, cudaMemcpyDeviceToHost, main));
    MIAGPU_CUDA(cudaMemcpyAsync(&H->prep, c->d_sh_prep.p, sizeof(ShardPrep), cudaMemcpyDeviceToHost, main));
    MIAGPU_CUDA(cudaMemcpyAsync(&H->stats, c->d_cstats.p, sizeof(CutStatsDev), cudaMemcpyDeviceToHost, main));
    MIAGPU_CUDA(cudaStreamSynchronize(main));
    int most = 0;
    for (int r = 0; r < world; r++) most = std::max(most, *reinterpret_cast<const int32_t*>(reinterpret_cast<const char*>(c->h_sh_recv) + r * pitch + ids_at));
    if (most > SHARD_PF_FIRST) {
      MIAGPU_CUDA(cudaMemcpy2DAsync(reinterpret_cast<char*>(c->h_sh_recv) + first, pitch, reinterpret_cast<const char*>(c->d_sh_recv.p) + first, pitch,
                                    pitch - first, world, cudaMemcpyDeviceToHost, main));
      MIAGPU_CUDA(cudaStreamSynchronize(main));
    }
    CutSums S;
    CutFit F;
    S.sx = H->prep.sx; S.sy = H->prep.sy; S.cnt = H->prep.cnt; S.bad = H->stats.bad == LLONG_MAX ? -1 : H->stats.bad;
    memcpy(S.best, H->stats.best, sizeof(S.best));
    if (S.bad >= 0) { set_error("miagpu_shard_cut: seq_len of local read %lld out of range", (long long)S.bad); return round_abort(c); }
    if (S.cnt <= 0) { set_error("miagpu_shard_cut: no read of any rank scores >= %d: nothing to fit", FIRST_ROUND_SCORE_CUTOFF); return round_abort(c); }
    cut_fit_tables(S, F);
    const int64_t nbt = (int64_t)world * nb;
    std::vector<ChainBlock> bxy(nbt), bxx(nbt);
    auto rank_words = [&](int r) { return c->h_sh_recv + (size_t)r * stride; };
    for (int r = 0; r < world; r++) {
      const ShardBlockRec* recs = reinterpret_cast<const ShardBlockRec*>(rank_words(r));
      for (int64_t b = 0; b < nb; b++) {
        const ShardBlockRec& B = recs[b];
        bxy[r * nb + b] = ChainBlock{0.0, B.T[0], B.A[0], B.e[0], B.ok[0] != 0};
        bxx[r * nb + b] = ChainBlock{0.0, B.T[1], B.A[1], B.e[1], B.ok[1] != 0};
      }
    }
    // keys of a block the stitch cannot prove: they came with the records of the rank that owns the block
    int missing = 0;
    char first_missing[200] = "";
    auto block_keys = [&](int64_t gb, double Sum, const ChainBlock& B, int chain) -> const uint32_t* {
      const int r = (int)(gb / nb);
      const int64_t b = gb % nb;
      const int32_t* pf_ids = reinterpret_cast<const int32_t*>(rank_words(r) + (nb * sizeof(ShardBlockRec) + 3) / 4);
      const uint32_t* pf_keys = reinterpret_cast<const uint32_t*>(pf_ids + SHARD_PF_SLOTS + 8);
      const int npf = std::min<int>(pf_ids[0], SHARD_PF_SLOTS);
      for (int k = 0; k < npf; k++)
        if (pf_ids[1 + k] == b) return pf_keys + (size_t)k * CUT_BLOCK;
      if (!missing++)
        snprintf(first_missing, sizeof first_missing, "first: rank %d block %lld chain %d, running sum %.17g, record e=%d ok=%d T=%g A=%g, %d blocks of that rank sent keys",
                 r, (long long)b, chain, Sum, B.e, (int)B.ok, B.T, B.A, pf_ids[0]);
      return nullptr;
    };
    int64_t ser0 = 0, ser1 = 0;
    const double ssxy = chain_stitch_blocks(bxy.data(), nbt, [&](int64_t b, double Sum) {
      const uint32_t* k = block_keys(b, Sum, bxy[b], 0);
      if (!k) return Sum;
      for (int i = 0; i < CUT_BLOCK; i++) Sum += k[i] == CUT_KEY_UNUSED ? 0.0 : F.dx_of[k[i] & 511] * ((double)(int)(k[i] >> 9) - F.ybar);
      return Sum;
    }, &ser0);
    const double ssxx = chain_stitch_blocks(bxx.data(), nbt, [&](int64_t b, double Sum) {
      const uint32_t* k = block_keys(b, Sum, bxx[b], 1);
      if (!k) return Sum;
      for (int i = 0; i < CUT_BLOCK; i++) Sum += k[i] == CUT_KEY_UNUSED ? 0.0 : F.dx2_of[k[i] & 511];
      return Sum;
    }, &ser1);
    if (missing) {
      set_error("miagpu_shard_cut: %d blocks of the regression's chains could not be proven and their keys did not travel (at most %d blocks per rank send keys; %s)", missing, SHARD_PF_SLOTS, first_missing);
      return round_abort(c);
    }
    c->cut_serial_blocks = ser0 + ser1;
    cut_fit_slope(S, F, ssxy, ssxx, &slope, &intercept);
  }
  if (slope_out) *slope_out = slope;
  if (intercept_out) *intercept_out = intercept;
  // flags of the local reads; with pointer state, every slot a local pointer reaches is local (miagpu_shard_fit)
  MIAGPU_CUDA(cudaStreamWaitEvent(main, c->aev[7], 0));                                // the accumulation of shard_fit
  if (!round_flags(c, slope, intercept, false)) return round_abort(c);
  if (sum_buf) *sum_buf = c->d_acc.p;
  if (sum_words) *sum_words = c->n_cols * NPLANE;
  c->sh_phase = 3;
  return 1;
}

extern "C" int miagpu_shard_finish(miagpu_ctx* c, int cons_code, uint8_t* dropped, uint16_t* packed_runs, int64_t capacity,
                                   int64_t* total_runs, int32_t* gaps_out, char* cons_out, int32_t* cons_len) {
  if (!c || c->sh_phase != 3) { set_error("miagpu_shard_finish: call miagpu_shard_cut first"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  c->sh_phase = 0;
  if (!round_call(c, cons_code, dropped, gaps_out, cons_out, cons_len) || !round_end(c)) return round_abort(c);
  if (packed_runs || total_runs) {                   // the round's launch count and times stand
    const int launches = c->launches;
    const float ms_kernels = c->ms_kernels, ms_d2h = c->ms_d2h;
    int64_t tot = 0;
    if (!miagpu_get_runs_packed(c, nullptr, packed_runs, capacity, &tot)) return round_abort(c);
    c->launches = launches + 4; c->ms_kernels = ms_kernels; c->ms_d2h = ms_d2h;
    if (total_runs) *total_runs = tot;
  }
  MIAGPU_CUDA(cudaStreamSynchronize(c->s_down));
  return 1;
}

// Pointer state in sharded rounds: AlnSeq.dropped lives in the slots, slot numbers run over the reads of all ranks, and the slots a
// rank's reads take drift from round to round -- so every rank keeps the flags of ALL slots.  After miagpu_shard_cut the flags this
// round set are in this buffer (one byte per slot); the caller MAX-reduces it over the ranks before the next miagpu_shard_begin.
// *bytes = 0: the context has no pointer state, nothing to do.
extern "C" int miagpu_shard_flags(miagpu_ctx* c, void** flag_buf, int64_t* bytes) {
  if (!c) { set_error("miagpu_shard_flags: no context"); return 0; }
  if (flag_buf) *flag_buf = c->fs_on ? c->d_slot_flag.p : nullptr;
  if (bytes) *bytes = c->fs_on ? c->fs_slot_cap : 0;
  return 1;
}

extern "C" int miagpu_last_cut_stats(miagpu_ctx* c, int64_t* serial_blocks, int64_t* fetched_blocks) {
  if (!c) { set_error("miagpu_last_cut_stats: no context"); return 0; }
  if (serial_blocks) *serial_blocks = c->cut_serial_blocks;
  if (fetched_blocks) *fetched_blocks = 0;
  return 1;
}

// ------------------------------------------------------------------ adapter trimming (8f4)
__global__ void trim_codes_kernel(int64_t total, uint8_t* bases_to_codes) {          // pop_s1c_in_a: ASCII -> 0..4, in place
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) bases_to_codes[i] = (uint8_t)base_code(bases_to_codes[i]);
}
__global__ void trim_windows_kernel(int64_t n, const int64_t* off, int32_t* ws, int32_t* wl, int* bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t l = off[i + 1] - off[i];
  if (l < 1 || l > MAX_READ) atomicMin(bad, (int)i);
  ws[i] = (int32_t)off[i]; wl[i] = (int32_t)min(max(l, (int64_t)1), (int64_t)MAX_READ);
}

template <int K>
static int launch_trim(miagpu_ctx* c, RealignParams p, int maxL, int n) {
  using TL = TraceLayout<K>;
  const size_t smem = PROF_INTS * 4 + WARPS_PER_BLOCK * MAX_READ * 2;
  int per_sm = 0;
  MIAGPU_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (realign_kernel<K, true>), WARPS_PER_BLOCK * 32, smem));
  if (per_sm < 1) { set_error("realign_kernel<%d, trim> does not fit on an SM", K); return 0; }
  per_sm = std::min(per_sm, 8);
  const int blocks = std::min(c->num_sms * per_sm, (n + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK);
  const int64_t words = (int64_t)std::max(maxL - 1, 1) * TL::ROW_WORDS;
  DevBuf<uint32_t>& scratch = c->d_scratch[0];
  if (!scratch.reserve((size_t)words * blocks * WARPS_PER_BLOCK)) return 0;
  p.scratch = scratch.p; p.scratch_words_per_warp = words; p.ref_in_smem = 0;
  realign_kernel<K, true><<<blocks, WARPS_PER_BLOCK * 32, smem, c->stream>>>(p);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches++;
  return 1;
}

extern "C" int miagpu_trim(miagpu_ctx* c, int64_t n, const uint8_t* bases, const int64_t* offsets, const char* adapter, int adapter_len,
                           int32_t* max_score, int32_t* abr, int32_t* abc, int32_t* aer, uint8_t* trimmed, int32_t* trim_point) {
  if (!c || n < 0 || (n && (!bases || !offsets)) || !adapter || adapter_len < 1 || adapter_len > 127) {   // mia_main.c:559: "That adapter is too big!"
    set_error("miagpu_trim: bad argument (the adapter holds 1..127 bases)");
    return 0;
  }
  if (n == 0) return 1;
  if (c->hp) { set_error("miagpu_trim: adapter trimming with the homopolymer discount (mia -T -h) is not built"); return 0; }
  if (n > 0x7fffffffLL || offsets[n] > 0x7fffffffLL) { set_error("miagpu_trim: batch too large"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  // flat matrix (init_flatsubmat, pssm.c:96-126) as a scoring profile: prof[depth][row base][column code]
  int32_t flat[MIAGPU_PSSM_INTS];
  for (int d = 0; d < NMAT; d++)
    for (int a = 0; a < 5; a++)
      for (int b = 0; b < 5; b++) flat[(d * 5 + a) * 5 + b] = a == 4 ? NR_SCORE_FLAT : b == 4 ? N_SCORE_FLAT : a == b ? FLAT_MATCH : FLAT_MISMATCH;
  std::vector<int32_t> prof(PROF_INTS, 0);
  for (int d = 0; d < NMAT; d++)
    for (int rb = 0; rb < 5; rb++)
      for (int fb = 0; fb < 5; fb++) prof[prof_row_index(0, d, rb) + fb] = flat[(d * 5 + fb) * 5 + rb];
  const int64_t total = offsets[n];
  std::vector<uint8_t> ad(adapter_len);
  for (int i = 0; i < adapter_len; i++) ad[i] = (uint8_t)adapter[i];
  DevBuf<int32_t>&d_prof = c->tr_prof, &d_ws = c->tr_ws, &d_wl = c->tr_wl, &d_out = c->tr_out, &d_cnt = c->tr_cnt;
  DevBuf<uint8_t>&d_codes = c->tr_codes, &d_ad = c->tr_ad, &d_st = c->tr_st;
  if (!d_prof.reserve(PROF_INTS) || !d_ws.reserve(n) || !d_wl.reserve(n) || !d_out.reserve(5 * n) || !d_cnt.reserve(4) ||
      !d_codes.reserve(total + 16) || !d_ad.reserve(adapter_len + 16) || !d_st.reserve(n) || !c->d_off2.reserve(n + 2)) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->ev[0], st));
  MIAGPU_CUDA(cudaMemcpyAsync(d_prof.p, prof.data(), PROF_INTS * 4, cudaMemcpyHostToDevice, st));
  MIAGPU_CUDA(cudaMemcpyAsync(c->d_off2.p, offsets, (n + 1) * 8, cudaMemcpyHostToDevice, st));
  MIAGPU_CUDA(cudaMemcpyAsync(d_codes.p, bases, total, cudaMemcpyHostToDevice, st));
  MIAGPU_CUDA(cudaMemcpyAsync(d_ad.p, ad.data(), adapter_len, cudaMemcpyHostToDevice, st));
  MIAGPU_CUDA(cudaMemsetAsync(d_cnt.p, 0, 16, st));
  int bad_read = 0x7fffffff, maxL = 0;
  MIAGPU_CUDA(cudaMemcpyAsync(d_cnt.p + 1, &bad_read, 4, cudaMemcpyHostToDevice, st));
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], st));
  trim_codes_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(total, d_codes.p);
  trim_windows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, c->d_off2.p, d_ws.p, d_wl.p, d_cnt.p + 1);
  max_len_kernel<<<256, 256, 0, st>>>(n, c->d_off2.p, d_cnt.p + 2);
  MIAGPU_CUDA(cudaGetLastError());
  int chk[2] = {0, 0};
  MIAGPU_CUDA(cudaMemcpyAsync(chk, d_cnt.p + 1, 8, cudaMemcpyDeviceToHost, st));
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  if (chk[0] != 0x7fffffff) { set_error("miagpu_trim: read %d has %lld bases (1..%d)", chk[0], (long long)(offsets[chk[0] + 1] - offsets[chk[0]]), MAX_READ); return 0; }
  maxL = std::min(chk[1], MAX_READ);
  RealignParams p{};
  p.bases = d_ad.p; p.off = nullptr; p.rc = nullptr; p.win_start = d_ws.p; p.win_len = d_wl.p; p.list = nullptr; p.n_list = (int)n;
  p.n_list_ptr = nullptr; p.counter = d_cnt.p; p.ref_codes = d_codes.p; p.ref_bytes = 0; p.prof = d_prof.p; p.sg5 = 1;   // mia_main.c:711-712
  p.score = d_out.p; p.as_out = d_out.p + n; p.ae_out = d_out.p + 2 * n; p.abr = d_out.p + 3 * n; p.aer_out = d_out.p + 4 * n;
  p.n_runs = nullptr; p.runs = nullptr; p.status = d_st.p; p.shared_rows = adapter_len;
  c->launches = 0;
  const int K = (maxL + 31) / 32;
  int ok;
  if (K <= 2) ok = launch_trim<2>(c, p, adapter_len, (int)n);
  else if (K <= 4) ok = launch_trim<4>(c, p, adapter_len, (int)n);
  else ok = launch_trim<8>(c, p, adapter_len, (int)n);
  if (!ok) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], st));
  std::vector<int32_t> out(5 * n);
  MIAGPU_CUDA(cudaMemcpyAsync(out.data(), d_out.p, 5 * n * 4, cudaMemcpyDeviceToHost, st));
  MIAGPU_CUDA(cudaEventRecord(c->ev[3], st));
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_kernels, c->ev[1], c->ev[2]));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_d2h, c->ev[2], c->ev[3]));
  c->dp_cells = total * adapter_len;
  for (int64_t i = 0; i < n; i++) {
    const int sc = out[i], col = out[n + i], row = out[3 * n + i], er = out[4 * n + i];
    const int t = (sc >= TRIM_SCORE_CUT) || (sc >= (er - row + 1) * FLAT_MATCH);       // mia.c:1358-1366
    if (max_score) max_score[i] = sc;
    if (abr) abr[i] = row;
    if (abc) abc[i] = col;
    if (aer) aer[i] = er;
    if (trimmed) trimmed[i] = (uint8_t)t;
    if (trim_point) trim_point[i] = t ? col - 1 : 0;
  }
  return 1;
}

// ------------------------------------------------------------------ repeat filter (8f1)
extern "C" int miagpu_repeat_filter(miagpu_ctx* c, int64_t n, const uint8_t* rc, const int32_t* as, const int32_t* ae, const int32_t* key4,
                                    const uint8_t* trimmed, int just_outer_coords, int tolerance, int64_t* order, uint8_t* unique_best) {
  if (!c || n < 0 || (n && (!rc || !as || !ae || !key4 || !unique_best)) || tolerance < 0) { set_error("miagpu_repeat_filter: bad argument"); return 0; }
  if (n > 0x7fffffffLL) { set_error("miagpu_repeat_filter: at most %d reads", 0x7fffffff); return 0; }
  if (n == 0) return 1;
  MIAGPU_CUDA(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  // scratch of the filter stays with the context (the call comes once per iteration)
  DevBuf<uint8_t>&d_rc = c->rf_rc, &d_tr = c->rf_tr, &d_uq = c->rf_uq, &d_tmp = c->rf_tmp;
  DevBuf<int32_t>&d_as = c->rf_as, &d_ae = c->rf_ae, &d_k4 = c->rf_k4, &d_idx = c->rf_idx, &d_idx2 = c->rf_idx2;
  DevBuf<uint64_t>&d_key = c->rf_key, &d_key2 = c->rf_key2;
  DevBuf<int64_t>& d_ord = c->rf_ord;
  DevBuf<int>& d_bad = c->rf_bad;
  if (!d_rc.reserve(n) || !d_as.reserve(n) || !d_ae.reserve(n) || !d_k4.reserve(n) || !d_idx.reserve(n) || !d_idx2.reserve(n) ||
      !d_key.reserve(n) || !d_key2.reserve(n) || !d_uq.reserve(n) || !d_bad.reserve(1) || (trimmed && !d_tr.reserve(n)) ||
      (order && !d_ord.reserve(n))) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->ev[0], st));
  MIAGPU_CUDA(cudaMemcpyAsync(d_rc.p, rc, n, cudaMemcpyHostToDevice, st));
  MIAGPU_CUDA(cudaMemcpyAsync(d_as.p, as, n * 4, cudaMemcpyHostToDevice, st));
  MIAGPU_CUDA(cudaMemcpyAsync(d_ae.p, ae, n * 4, cudaMemcpyHostToDevice, st));
  MIAGPU_CUDA(cudaMemcpyAsync(d_k4.p, key4, n * 4, cudaMemcpyHostToDevice, st));
  if (trimmed) MIAGPU_CUDA(cudaMemcpyAsync(d_tr.p, trimmed, n, cudaMemcpyHostToDevice, st));
  MIAGPU_CUDA(cudaMemsetAsync(d_bad.p, 0, sizeof(int), st));
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], st));
  const unsigned grid = (unsigned)((n + 255) / 256);
  rf_key_kernel<<<grid, 256, 0, st>>>(n, d_rc.p, d_as.p, d_ae.p, d_k4.p, d_key.p, d_idx.p, d_bad.p);
  MIAGPU_CUDA(cudaGetLastError());
  size_t tmp = 0;
  MIAGPU_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, d_key.p, d_key2.p, d_idx.p, d_idx2.p, (int)n, 0, 64, st));
  if (!d_tmp.reserve(tmp + 16)) return 0;
  MIAGPU_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp.p, tmp, d_key.p, d_key2.p, d_idx.p, d_idx2.p, (int)n, 0, 64, st));
  int bad = 0;
  MIAGPU_CUDA(cudaMemcpyAsync(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  c->launches = 2;
  if (tolerance == 0) {
    rf_unique_kernel<<<grid, 256, 0, st>>>(n, d_idx2.p, d_rc.p, d_as.p, d_ae.p, trimmed ? d_tr.p : nullptr, just_outer_coords, d_uq.p);
    MIAGPU_CUDA(cudaGetLastError());
    c->launches++;
  }
  if (order) {
    rf_widen_kernel<<<grid, 256, 0, st>>>(n, d_idx2.p, d_ord.p);
    MIAGPU_CUDA(cudaGetLastError());
    c->launches++;
  }
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], st));
  std::vector<int32_t> h_idx;
  if (tolerance == 0) MIAGPU_CUDA(cudaMemcpyAsync(unique_best, d_uq.p, n, cudaMemcpyDeviceToHost, st));
  else { h_idx.resize(n); MIAGPU_CUDA(cudaMemcpyAsync(h_idx.data(), d_idx2.p, n * 4, cudaMemcpyDeviceToHost, st)); }
  if (order) MIAGPU_CUDA(cudaMemcpyAsync(order, d_ord.p, n * 8, cudaMemcpyDeviceToHost, st));
  MIAGPU_CUDA(cudaEventRecord(c->ev[3], st));
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_kernels, c->ev[1], c->ev[2]));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_d2h, c->ev[2], c->ev[3]));
  if (bad) { set_error("miagpu_repeat_filter: coordinates must lie in [0, %d] and the fourth key in [%d, %d)", RF_COORD_MAX, -RF_KEY4_HALF, RF_KEY4_HALF); return 0; }
  if (tolerance > 0) {                                 // set_uniq_in_fsdb's greedy grouping (fsdb.c:452-506) over the sorted order
    int64_t f = h_idx[0];
    int curr_rc = rc[f] != 0, curr_as = as[f], curr_ae = ae[f];
    unique_best[f] = 1;
    for (int64_t k = 1; k < n; k++) {
      f = h_idx[k];
      const int frc = rc[f] != 0;
      if (frc == curr_rc && abs(as[f] - curr_as) <= tolerance && abs(ae[f] - curr_ae) <= tolerance) { unique_best[f] = 0; continue; }
      if (just_outer_coords) unique_best[f] = 1;
      else if (!frc) unique_best[f] = as[f] == curr_as ? (trimmed && trimmed[f] ? 1 : 0) : 1;
      else unique_best[f] = ae[f] == curr_ae ? (trimmed && trimmed[f] ? 1 : 0) : 1;
      curr_rc = frc; curr_as = as[f]; curr_ae = ae[f];
    }
  }
  return 1;
}

// ------------------------------------------------------------------ pass 1
// populate_kpa / add_kmer (kmer.c:63-85, 153-168) as a bucketed, sorted (k-mer, position) table
static int build_kmer_strand(miagpu_ctx* c, int t, const std::string& seq, int k, int soft_mask) {
  std::vector<uint64_t> all;
  all.reserve(seq.size());
  for (size_t i = 0; i + k <= seq.size(); i++) {
    bool ok = true;
    uint64_t inx = 0;
    for (int j = 0; j < k && ok; j++) {
      char ch = seq[i + j];
      if (soft_mask && ch >= 'a' && ch <= 'z') ok = false;                  // all_upper, kmer.c:140-148
      if (ch >= 'a' && ch <= 'z') ch = (char)(ch - 32);                     // kmer2inx upper-cases, kmer.c:27
      int code = ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : ch == 'T' ? 3 : -1;
      if (code < 0) ok = false;
      inx = (inx << 2) | (uint64_t)(code & 3);
    }
    if (ok) all.push_back((inx << 32) | (uint64_t)i);
  }
  std::sort(all.begin(), all.end());
  const int bucket_bits = std::min(2 * k, 16);
  const int shift = 2 * k - bucket_bits;
  const int nb = 1 << bucket_bits;
  std::vector<int32_t> bstart(nb + 1, 0), pos;
  std::vector<uint32_t> km;
  int run = 0;
  for (size_t i = 0; i < all.size(); i++) {
    run = (i > 0 && (all[i] >> 32) == (all[i - 1] >> 32)) ? run + 1 : 0;
    if (run >= MAX_KMER_POS) continue;                                      // add_kmer keeps the first 128 positions
    km.push_back((uint32_t)(all[i] >> 32));
    pos.push_back((int32_t)(all[i] & 0xffffffffu));
    bstart[(km.back() >> shift) + 1]++;
  }
  for (int b = 0; b < nb; b++) bstart[b + 1] += bstart[b];
  if (!c->d_kb[t].reserve(nb + 1) || !c->d_kk[t].reserve(km.size() + 1) || !c->d_kp[t].reserve(pos.size() + 1)) return 0;
  MIAGPU_CUDA(cudaMemcpyAsync(c->d_kb[t].p, bstart.data(), (nb + 1) * 4, cudaMemcpyHostToDevice, c->stream));
  if (!km.empty()) {
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_kk[t].p, km.data(), km.size() * 4, cudaMemcpyHostToDevice, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_kp[t].p, pos.data(), pos.size() * 4, cudaMemcpyHostToDevice, c->stream));
  }
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  c->kmer_shift[t] = shift;
  return 1;
}

extern "C" int miagpu_build_kmers(miagpu_ctx* c, int k, int soft_mask) {
  if (!c || !c->have_ref) { set_error("miagpu_build_kmers: set_reference first"); return 0; }
  if (k > 14) { set_error("Cannot use kmer length greater than 14"); return 0; }   // init_kpa, kmer.c:93-97
  MIAGPU_CUDA(cudaSetDevice(c->device));
  if (k <= 0) { c->kmer_k = 0; return 1; }
  if (!c->with_rc) { set_error("miagpu_build_kmers: the reference was set without its reverse complement"); return 0; }
  if ((int)c->raw_wrapped.size() < k) { set_error("miagpu_build_kmers: reference shorter than k"); return 0; }
  if (!build_kmer_strand(c, 0, c->raw_wrapped, k, soft_mask) || !build_kmer_strand(c, 1, c->raw_rc_wrapped, k, soft_mask)) return 0;
  c->kmer_k = k;
  return 1;
}

// Pass 1 with the k-mer filter on (pass1.cuh): seed every read, run the strands' separate stretches through the pair
// kernels, merge, and leave the rest to the general kernel.
// longest read sweep16_kernel takes: the whole frame with the re-based variant when the matrices leave it room
static int sweep_lmax(miagpu_ctx* c, const PairLmax& lm_low) {
  bool rb = p16_rb_frame(SW_K, c->pssm_max).room >= 16384;
  if (const char* e = getenv("MIAGPU_PAIR_RB")) if (atoi(e) == 0) rb = false;
  return lm_low.v[SW_CLASS] > 0 ? (rb ? P16_MAXL : lm_low.v[SW_CLASS]) : 0;
}

// Whole-strand 16-bit sweeps of m jobs (jobs: device list, nullptr = jobs 0 .. m-1; d_jread names their reads and strands): work
// items by read length, the plain frame for the reads it holds, the re-based frame for the longer ones.  On c->launch_stream.
// same_read: the list holds reads; a half-warp takes both strands of one (pass 1 without the filter).
static int launch_sweep(miagpu_ctx* c, const int32_t* jobs, int64_t m, int lmax_low, bool same_read = false) {
  if (m <= 0) return 1;
  cudaStream_t st = c->launch_stream;
  const int len1 = c->circular ? c->wrap_len : c->seq_len;
  if (!c->d_sw_layout.reserve(SW_LAYOUT_WORDS) || !c->d_sw_pairs.reserve((size_t)m + 4 * (MAX_READ + 2) + 8)) return 0;
  int32_t *cnt = c->d_sw_layout.p, *start = cnt + (MAX_READ + 2), *cursor = start + (MAX_READ + 2), *n_items = cursor + (MAX_READ + 2), *work = n_items + 2;
  MIAGPU_CUDA(cudaMemsetAsync(cnt, 0, SW_LAYOUT_WORDS * sizeof(int32_t), st));
  MIAGPU_CUDA(cudaMemsetAsync(c->d_sw_pairs.p, 0xff, ((size_t)m + 4 * (MAX_READ + 2) + 8) * sizeof(int32_t), st));
  const int32_t* jr = same_read ? nullptr : c->d_jread.p;
  const int per_item = same_read ? 2 : 4;
  sw_hist_kernel<<<(unsigned)std::min<int64_t>(2 * c->num_sms, (m + 255) / 256), 256, 0, st>>>(m, jobs, jr, c->d_off.p, cnt);
  sw_layout_kernel<<<1, 32, 0, st>>>(cnt, start, cursor, lmax_low, n_items, per_item);
  sw_scatter_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(m, jobs, jr, c->d_off.p, cursor, c->d_sw_pairs.p);
  MIAGPU_CUDA(cudaGetLastError());
  Sweep16Params sp{};
  sp.bases = c->d_bases.p; sp.off = c->d_off.p; sp.pairs = c->d_sw_pairs.p; sp.job_read = c->d_jread.p;
  sp.ref2 = c->d_ref2.p; sp.strand_stride = c->ref_bytes; sp.len1 = len1; sp.prof16 = c->d_prof16.p; sp.gep2 = K2(2 * GEP);
  sp.jscore = c->d_jscore.p; sp.jabc = c->d_jabc.p; sp.jaec = c->d_jaec.p; sp.jabr = c->d_jabr.p; sp.jstatus = c->d_jstatus.p;
  const RbFrame f = p16_rb_frame(SW_K, c->pssm_max);
  sp.rb_off = f.off; sp.rb_d = f.d; sp.rb_thresh = f.thresh;
  // shared memory follows the longest read (the hand-over rings are the bulk of it): short reads leave room for four blocks per SM
  if (!ensure_max_read_len(c)) return 0;
  const int rows_cap = std::min((std::max(c->max_read_len, 8) + 7) & ~7, P16_MAXL);
  sp.rows_cap = rows_cap;
  const size_t smem = sw_smem(rows_cap);
  static int per_sm_d[MAX_DEVICES][2], cached_rows_d[MAX_DEVICES];
  int* per_sm = per_sm_d[c->device % MAX_DEVICES];
  int& cached_rows = cached_rows_d[c->device % MAX_DEVICES];
  if (cached_rows != rows_cap) {
    MIAGPU_CUDA(cudaFuncSetAttribute((sweep16_kernel<false, false>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MIAGPU_CUDA(cudaFuncSetAttribute((sweep16_kernel<true, false>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MIAGPU_CUDA(cudaFuncSetAttribute((sweep16_kernel<false, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MIAGPU_CUDA(cudaFuncSetAttribute((sweep16_kernel<true, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MIAGPU_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[0], (sweep16_kernel<false, false>), WARPS_PER_BLOCK * 32, smem));
    MIAGPU_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[1], (sweep16_kernel<true, false>), WARPS_PER_BLOCK * 32, smem));
    cached_rows = rows_cap;
  }
  if (per_sm[0] < 1 || per_sm[1] < 1) { set_error("sweep16_kernel does not fit on an SM (smem %zu)", smem); return 0; }
  const int64_t items_max = m / per_item + (MAX_READ + 2);                  // every length's run is padded to whole items
  const int blocks0 = (int)std::min<int64_t>((int64_t)c->num_sms * per_sm[0], (items_max + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK);
  const int blocks1 = (int)std::min<int64_t>((int64_t)c->num_sms * per_sm[1], (items_max + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK);
  sp.n_items = n_items; sp.first_item = nullptr; sp.counter = work;
  if (same_read) sweep16_kernel<false, true><<<blocks0, WARPS_PER_BLOCK * 32, smem, st>>>(sp);
  else sweep16_kernel<false, false><<<blocks0, WARPS_PER_BLOCK * 32, smem, st>>>(sp);
  sp.n_items = n_items + 1; sp.first_item = n_items; sp.counter = work + 1;
  if (same_read) sweep16_kernel<true, true><<<blocks1, WARPS_PER_BLOCK * 32, smem, st>>>(sp);
  else sweep16_kernel<true, false><<<blocks1, WARPS_PER_BLOCK * 32, smem, st>>>(sp);
  MIAGPU_CUDA(cudaGetLastError());
  c->launches += 5;
  return 1;
}

static int pass1_fast(miagpu_ctx* c, const PairLmax& lm) {
  const PairLmax lm_low = pair_lmax_low(c);
  const int64_t n = c->n, nj = 10 * n + 4096;          // job capacity; reads whose jobs do not fit go to the general kernel
  if (n > 0x7fffffffLL / 8) { set_error("miagpu_pass1: at most %d reads per batch", 0x7fffffff / 8); return 0; }
  if (!c->d_jread.reserve(nj + 1) || !c->d_jfirst.reserve(n + 1) || !c->d_jcount.reserve(n + 1)) return 0;
  if (!c->d_jkind.reserve(nj + 1) || !c->d_jstatus.reserve(nj + 1) || !c->d_route.reserve(n + 1) || !c->d_jws.reserve(nj + 1) ||
      !c->d_jwl.reserve(nj + 1) || !c->d_jscore.reserve(nj + 1) || !c->d_jabc.reserve(nj + 1) || !c->d_jaec.reserve(nj + 1) ||
      !c->d_jabr.reserve(nj + 1) || !c->d_p1list.reserve(n + 1) || !c->d_p1trace.reserve(n + 1) || !c->d_sw_jobs.reserve(2 * n + 1) || !c->d_p1sunk.reserve(nj + 1) || !c->d_p1meta.reserve(META_WORDS) ||
      !c->d_jpairs.reserve(nj + 4 * P16_KEYS + 64)) return 0;
  cudaStream_t st = c->stream;
  int32_t* meta = c->d_p1meta.p;
  const int len1 = c->circular ? c->wrap_len : c->seq_len;
  MIAGPU_CUDA(cudaMemsetAsync(meta, 0, META_WORDS * sizeof(int32_t), st));
  MIAGPU_CUDA(cudaMemsetAsync(c->d_jkind.p, 0, nj, st));
  P1SeedParams sp{};
  sp.bases = c->d_bases.p; sp.off = c->d_off.p; sp.n = n; sp.k = c->kmer_k; sp.len1 = len1; sp.strand_stride = c->ref_bytes; sp.pssm_max = c->pssm_max;
  for (int t = 0; t < 2; t++) sp.kt[t] = KmerTable{c->d_kb[t].p, c->d_kk[t].p, c->d_kp[t].p, c->kmer_shift[t]};
  sp.lm = lm;
  sp.sw_lmax = getenv("MIAGPU_P1_NO_SWEEP") ? 0 : sweep_lmax(c, lm_low); sp.sw_jobs = c->d_sw_jobs.p;
  sp.job_cap = nj; sp.jread = c->d_jread.p; sp.jfirst = c->d_jfirst.p; sp.jcount = c->d_jcount.p;
  sp.jkind = c->d_jkind.p; sp.jws = c->d_jws.p; sp.jwl = c->d_jwl.p; sp.hits = c->d_hits.p; sp.route = c->d_route.p;
  sp.general_list = c->d_p1list.p; sp.score = c->d_score.p; sp.n_runs = c->d_nruns.p; sp.status = c->d_status.p; sp.meta = meta;
  const unsigned seed_blocks = (unsigned)std::min<int64_t>((int64_t)c->num_sms * 8, (n + 7) / 8);
  p1_seed_kernel<<<seed_blocks, 256, 0, st>>>(sp);
  MIAGPU_CUDA(cudaGetLastError());
  pair_layout_kernel<<<1, LAYOUT_THREADS, 0, st>>>(meta);
  MIAGPU_CUDA(cudaGetLastError());
  MIAGPU_CUDA(cudaEventRecord(c->p1ev[0], st));
  MIAGPU_CUDA(cudaMemcpyAsync(c->h_meta, meta, sizeof(int32_t) * META_HOST, cudaMemcpyDeviceToHost, st));
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  c->launches += 2;
  int pair_items[P16_NKB], total_pairs = 0;
  for (int kb = 0; kb < P16_NKB; kb++) { pair_items[kb] = c->h_meta[META_NPAIRS + kb]; total_pairs += pair_items[kb]; }
  // The reads the seeding already sent to the general kernel (saturated strands above all: a whole strand on one
  // warp, milliseconds per read) start first, on a side stream, and run beside the pair kernels.
  const int n_general0 = c->h_meta[P1_NGENERAL];
  const int n_sweep = c->h_meta[P1_NSWEEP];
  c->p1_swept = n_sweep;
  if (n_general0 || n_sweep) {
    MIAGPU_CUDA(cudaEventRecord(c->aev[0], st));
    MIAGPU_CUDA(cudaStreamWaitEvent(c->s_aux[1], c->aev[0], 0));
    c->launch_stream = c->s_aux[1];
    // the strands the filter saturated (error-free reads of 128 + k - 1 bases and more): whole-strand sweeps in 16 bits, two jobs per
    // half-warp; the merge below needs their scores
    int ok = launch_sweep(c, c->d_sw_jobs.p, n_sweep, lm_low.v[SW_CLASS]);
    if (ok && n_sweep) MIAGPU_CUDA(cudaEventRecord(c->aev[5], c->s_aux[1]));
    if (ok && n_general0) ok = launch_strip(c, 0, c->d_p1list.p, n_general0, meta + P1_WORK, 0, nullptr);
    c->launch_stream = st;
    if (!ok) return 0;
    MIAGPU_CUDA(cudaEventRecord(c->aev[1], c->s_aux[1]));
  }
  if (total_pairs) {
    MIAGPU_CUDA(cudaMemsetAsync(c->d_jpairs.p, 0xff, (size_t)2 * P16_NP * total_pairs * sizeof(int32_t), st));
    const int64_t njobs = std::min<int64_t>(nj, (uint32_t)c->h_meta[P1_NJOBS]);
    pair_scatter_kernel<<<(unsigned)((njobs + 255) / 256), 256, 0, st>>>(njobs, c->d_off.p, c->d_jkind.p, meta, c->d_jpairs.p, c->d_jread.p);
    MIAGPU_CUDA(cudaGetLastError());
    c->launches++;
    int base = 0;
    // the classes' kernels are persistent (blocks fetch work until the class runs dry): spread over three streams, the next
    // class's blocks move in as the previous class's tail drains (s_aux[1] belongs to the general kernel)
    cudaStream_t lanes3[3] = {st, c->s_aux[2], c->s_aux[3]};
    MIAGPU_CUDA(cudaEventRecord(c->aev[2], st));
    MIAGPU_CUDA(cudaStreamWaitEvent(c->s_aux[2], c->aev[2], 0));
    MIAGPU_CUDA(cudaStreamWaitEvent(c->s_aux[3], c->aev[2], 0));
    int rr = 0;
    c->launch_slot = 0;
    for (int kb = 0; kb < P16_NKB; kb++) {
      const int ni = pair_items[kb];
      if (!ni) continue;
      c->launch_stream = lanes3[rr++ % 3];
      Pair16Params p{};
      p.bases = c->d_bases.p; p.off = c->d_off.p; p.rc = nullptr; p.win_start = c->d_jws.p; p.win_len = c->d_jwl.p;
      p.pairs = c->d_jpairs.p + 2 * (int64_t)P16_NP * base; p.n_items = meta + META_NPAIRS + kb; p.counter = meta + META_PWORK + kb;
      p.ref_codes = c->d_ref2.p; p.ref_bytes = 2 * c->ref_bytes; p.strand_stride = c->ref_bytes; p.prof16 = c->d_prof16.p; p.job_read = c->d_jread.p;
      p.score = c->d_jscore.p; p.as_out = c->d_jabc.p; p.ae_out = c->d_jaec.p; p.abr = c->d_jabr.p; p.status = c->d_jstatus.p;
      p.n_reads = nj;
      p.sunk_list = c->d_p1sunk.p; p.sunk_count = meta + P1_NSUNK;
      const bool rb = c->h_meta[META_PMAXL + kb] > lm_low.v[kb];
      if (!launch_pair_class<true>(c, p, kb, rb, ni)) { c->launch_stream = st; return 0; }
      base += ni;
    }
    c->launch_stream = st;
    for (int i = 2; i < 4; i++) {
      MIAGPU_CUDA(cudaEventRecord(c->aev[1 + i], c->s_aux[i]));
      MIAGPU_CUDA(cudaStreamWaitEvent(st, c->aev[1 + i], 0));
    }
  }
  if (total_pairs && !getenv("MIAGPU_P1_NO_SUNK32")) {
    // jobs whose alignment left the 16-bit frame (a chance stretch of a long read sinks fast): exact scores from the 32-bit JOB
    // kernel, so that the merge sees no job it cannot use; the list's length stays on the device (usually a per cent of the reads)
    if (!ensure_max_read_len(c)) return 0;
    const int maxL = std::min(std::max(c->max_read_len, 2), MAX_READ);
    RealignParams p{};
    p.bases = c->d_bases.p; p.off = c->d_off.p; p.rc = nullptr; p.win_start = c->d_jws.p; p.win_len = c->d_jwl.p;
    p.list = c->d_p1sunk.p; p.n_list = 2 * WARPS_PER_BLOCK * c->num_sms; p.n_list_ptr = meta + P1_NSUNK;
    p.ref_codes = c->d_ref2.p; p.ref_bytes = 2 * c->ref_bytes; p.prof = c->d_prof.p; p.sg5 = 1;
    p.score = c->d_score.p; p.status = c->d_status.p;
    p.job_read = c->d_jread.p; p.strand_stride = c->ref_bytes; p.seq_len = c->seq_len;
    p.job_score = c->d_jscore.p; p.job_abc = c->d_jabc.p; p.job_aec = c->d_jaec.p; p.job_abr = c->d_jabr.p; p.job_status = c->d_jstatus.p;
    for (int t = 0; t < 3; t++) {
      c->launch_slot = 1 + t;
      p.counter = meta + P1_SWORK + t;
      p.job_wl_lo = t == 0 ? 0 : t == 1 ? 64 : 128;
      p.job_wl_hi = t == 0 ? 64 : t == 1 ? 128 : 256;
      const int ok = t == 0 ? launch_realign<2, true>(c, p, maxL) : t == 1 ? launch_realign<4, true>(c, p, maxL) : launch_realign<8, true>(c, p, maxL);
      if (!ok) { c->launch_slot = 0; return 0; }
    }
    c->launch_slot = 0;
  }
  if (n_sweep) MIAGPU_CUDA(cudaStreamWaitEvent(st, c->aev[5], 0));
  MIAGPU_CUDA(cudaEventRecord(c->p1ev[1], st));
  P1MergeParams mp{};
  mp.n = n; mp.off = c->d_off.p; mp.seq_len = c->seq_len; mp.route = c->d_route.p; mp.jfirst = c->d_jfirst.p; mp.jcount = c->d_jcount.p; mp.jkind = c->d_jkind.p; mp.jstatus = c->d_jstatus.p;
  mp.jscore = c->d_jscore.p; mp.jabc = c->d_jabc.p; mp.jaec = c->d_jaec.p; mp.jabr = c->d_jabr.p; mp.general_list = c->d_p1list.p; mp.meta = meta;
  mp.score = c->d_score.p; mp.fw_score = c->d_fw.p; mp.rc_score = c->d_rcs.p; mp.as_out = c->d_as_out.p; mp.ae_out = c->d_ae_out.p;
  mp.start = c->d_start.p; mp.end = c->d_end.p; mp.abr = c->d_abr.p; mp.n_runs = c->d_nruns.p; mp.rc_out = c->d_rc_out.p;
  mp.runs = c->d_runs.p; mp.status = c->d_status.p;
  mp.trace_list = getenv("MIAGPU_P1_NO_TRACE") ? nullptr : c->d_p1trace.p;
  p1_merge_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(mp);
  MIAGPU_CUDA(cudaGetLastError());
  MIAGPU_CUDA(cudaEventRecord(c->p1ev[2], st));
  c->launches++;
  // the general kernel over whatever is left (list length read on the device; the grid is sized for the seeding's share)
  MIAGPU_CUDA(cudaMemcpyAsync(c->h_meta, meta, sizeof(int32_t) * META_HOST, cudaMemcpyDeviceToHost, st));
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  const int n_general = c->h_meta[P1_NGENERAL];
  c->p1_general = n_general; c->p1_fast = c->h_meta[P1_NFAST]; c->p1_skipped = c->h_meta[P1_NSKIPPED];
  c->p1_traced = c->h_meta[P1_NTRACE];
  if (c->p1_traced) {
    if (!ensure_max_read_len(c)) return 0;
    const int maxL = std::min(std::max(c->max_read_len, 2), MAX_READ);
    // gapped winners (reads with an indel against the reference, or a mismatch close to an end that a gap buys out): their stretch
    // alone, 32-bit with a trace, three widths; every launch walks the whole list and takes its own widths
    RealignParams p{};
    p.bases = c->d_bases.p; p.off = c->d_off.p; p.rc = nullptr; p.win_start = c->d_jws.p; p.win_len = c->d_jwl.p;
    p.list = c->d_p1trace.p; p.n_list = c->p1_traced; p.n_list_ptr = nullptr;
    p.ref_codes = c->d_ref2.p; p.ref_bytes = 2 * c->ref_bytes; p.prof = c->d_prof.p; p.sg5 = 1;
    p.score = c->d_score.p; p.as_out = c->d_as_out.p; p.ae_out = c->d_ae_out.p; p.abr = c->d_abr.p; p.n_runs = c->d_nruns.p;
    p.runs = c->d_runs.p; p.status = c->d_status.p; p.start = c->d_start.p; p.end = c->d_end.p;
    p.job_read = c->d_jread.p; p.strand_stride = c->ref_bytes; p.seq_len = c->seq_len;
    cudaStream_t lanes3[3] = {c->s_aux[2], c->s_aux[3], st};
    MIAGPU_CUDA(cudaEventRecord(c->aev[2], st));
    int ok = 1;
    for (int t = 0; t < 3 && ok; t++) {
      c->launch_stream = lanes3[t];
      c->launch_slot = 1 + t;                          // scratch 0 may still serve the general kernel's first launch
      if (lanes3[t] != st) MIAGPU_CUDA(cudaStreamWaitEvent(lanes3[t], c->aev[2], 0));
      p.counter = meta + P1_TWORK + t;
      p.job_wl_lo = t == 0 ? 0 : t == 1 ? 64 : 128;
      p.job_wl_hi = t == 0 ? 64 : t == 1 ? 128 : 256;
      ok = t == 0 ? launch_realign<2, true>(c, p, maxL) : t == 1 ? launch_realign<4, true>(c, p, maxL) : launch_realign<8, true>(c, p, maxL);
    }
    c->launch_stream = st; c->launch_slot = 0;
    if (!ok) return 0;
    for (int i = 2; i < 4; i++) {
      MIAGPU_CUDA(cudaEventRecord(c->aev[1 + i], c->s_aux[i]));
      MIAGPU_CUDA(cudaStreamWaitEvent(st, c->aev[1 + i], 0));
    }
  }
  if (n_general0) MIAGPU_CUDA(cudaStreamWaitEvent(st, c->aev[1], 0));      // the two general launches share their scratch
  if (n_general > n_general0 &&
      !launch_strip(c, 0, c->d_p1list.p + n_general0, n_general - n_general0, meta + P1_WORK2, 0, nullptr)) return 0;
  return 1;
}

// Pass 1 without the k-mer filter (sweep16.cuh): both whole strands of every read in one 16-bit sweep, two reads per warp;
// the merge kernel of the fast path finishes the reads whose winning path is a plain diagonal, the general kernel the rest.
static int pass1_sweep(miagpu_ctx* c, const PairLmax& lm) {
  const int64_t n = c->n, nj = 2 * n;
  if (n > 0x3fffffffLL) { set_error("miagpu_pass1: at most %d reads per batch", 0x3fffffff); return 0; }
  if (!c->d_jfirst.reserve(n + 1) || !c->d_jcount.reserve(n + 1) || !c->d_jkind.reserve(nj + 1) || !c->d_jstatus.reserve(nj + 1) ||
      !c->d_route.reserve(n + 1) || !c->d_jscore.reserve(nj + 1) || !c->d_jabc.reserve(nj + 1) || !c->d_jaec.reserve(nj + 1) ||
      !c->d_jabr.reserve(nj + 1) || !c->d_p1list.reserve(n + 1) || !c->d_p1meta.reserve(META_WORDS) || !c->d_jread.reserve(nj + 1) ||
      !c->d_sw_jobs.reserve(nj + 1)) return 0;
  cudaStream_t st = c->stream;
  int32_t* meta = c->d_p1meta.p;
  MIAGPU_CUDA(cudaMemsetAsync(meta, 0, META_WORDS * sizeof(int32_t), st));
  const int lmax_low = lm.v[SW_CLASS];
  SweepPrepParams pp{};
  pp.n = n; pp.off = c->d_off.p; pp.lmax = sweep_lmax(c, lm); pp.route = c->d_route.p; pp.jfirst = c->d_jfirst.p;
  pp.jcount = c->d_jcount.p; pp.jkind = c->d_jkind.p; pp.job_read = c->d_jread.p; pp.sw_jobs = c->d_sw_jobs.p; pp.hits = c->d_hits.p;
  pp.general_list = c->d_p1list.p; pp.meta = meta;
  sweep_prep_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(pp, P1_NGENERAL);
  MIAGPU_CUDA(cudaGetLastError());
  MIAGPU_CUDA(cudaEventRecord(c->p1ev[0], st));
  MIAGPU_CUDA(cudaMemcpyAsync(c->h_meta, meta, sizeof(int32_t) * META_HOST, cudaMemcpyDeviceToHost, st));
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  c->launches += 1;
  const int64_t n_sweep_reads = c->h_meta[META_PREADS + SW_CLASS];
  const int n_general0 = c->h_meta[P1_NGENERAL];
  if (n_general0) {                                   // reads no 16-bit frame holds: the general kernel, beside the sweep
    MIAGPU_CUDA(cudaEventRecord(c->aev[0], st));
    MIAGPU_CUDA(cudaStreamWaitEvent(c->s_aux[1], c->aev[0], 0));
    c->launch_stream = c->s_aux[1];
    const int ok = launch_strip(c, 0, c->d_p1list.p, n_general0, meta + P1_WORK, 0, nullptr);
    c->launch_stream = st;
    if (!ok) return 0;
    MIAGPU_CUDA(cudaEventRecord(c->aev[1], c->s_aux[1]));
  }
  c->launch_stream = st;
  if (!launch_sweep(c, c->d_sw_jobs.p, n_sweep_reads, lmax_low, true)) return 0;
  MIAGPU_CUDA(cudaEventRecord(c->p1ev[1], st));
  P1MergeParams mp{};
  mp.n = n; mp.off = c->d_off.p; mp.seq_len = c->seq_len; mp.route = c->d_route.p; mp.jfirst = c->d_jfirst.p; mp.jcount = c->d_jcount.p;
  mp.jkind = c->d_jkind.p; mp.jstatus = c->d_jstatus.p;
  mp.jscore = c->d_jscore.p; mp.jabc = c->d_jabc.p; mp.jaec = c->d_jaec.p; mp.jabr = c->d_jabr.p; mp.general_list = c->d_p1list.p; mp.meta = meta;
  mp.score = c->d_score.p; mp.fw_score = c->d_fw.p; mp.rc_score = c->d_rcs.p; mp.as_out = c->d_as_out.p; mp.ae_out = c->d_ae_out.p;
  mp.start = c->d_start.p; mp.end = c->d_end.p; mp.abr = c->d_abr.p; mp.n_runs = c->d_nruns.p; mp.rc_out = c->d_rc_out.p;
  mp.runs = c->d_runs.p; mp.status = c->d_status.p;
  p1_merge_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(mp);
  MIAGPU_CUDA(cudaGetLastError());
  MIAGPU_CUDA(cudaEventRecord(c->p1ev[2], st));
  c->launches++;
  MIAGPU_CUDA(cudaMemcpyAsync(c->h_meta, meta, sizeof(int32_t) * META_HOST, cudaMemcpyDeviceToHost, st));
  MIAGPU_CUDA(cudaStreamSynchronize(st));
  const int n_general = c->h_meta[P1_NGENERAL];
  c->p1_general = n_general; c->p1_fast = c->h_meta[P1_NFAST]; c->p1_skipped = 0;
  if (n_general0) MIAGPU_CUDA(cudaStreamWaitEvent(st, c->aev[1], 0));
  if (n_general > n_general0 &&
      !launch_strip(c, 0, c->d_p1list.p + n_general0, n_general - n_general0, meta + P1_WORK2, 0, nullptr)) return 0;
  return 1;
}

extern "C" int miagpu_pass1(miagpu_ctx* c, int32_t* hits, int32_t* score, int32_t* fw_score, int32_t* rc_score, uint8_t* rc, int32_t* as,
                            int32_t* ae, int32_t* start, int32_t* end, int32_t* abr, int32_t* n_runs, uint16_t* runs, uint8_t* status) {
  if (!c || !c->have_pssm || !c->have_ref || !c->with_rc) { set_error("miagpu_pass1: set_pssm and set_reference(with_rc=1) first"); return 0; }
  misinc_invalidate(c, "miagpu_pass1 has replaced the alignments of that round");
  MIAGPU_CUDA(cudaSetDevice(c->device));
  const int64_t n = c->n;
  c->launches = 0;
  if (!c->d_hits.reserve(n + 1) || !c->d_fw.reserve(n + 1) || !c->d_rcs.reserve(n + 1) || !c->d_start.reserve(n + 1) ||
      !c->d_end.reserve(n + 1) || !c->d_rc_out.reserve(n + 1)) return 0;
  MIAGPU_CUDA(cudaMemsetAsync(c->d_meta.p, 0, 128 * sizeof(int32_t), c->stream));
  MIAGPU_CUDA(cudaEventRecord(c->ev[1], c->stream));
  const PairLmax lm = c->kmer_k > 0 ? pair_lmax(c, true) : pair_lmax_low(c);      // (the whole-strand sweep has no RB frame)
  bool fast = c->kmer_k > 0 && lm.v[0] > 0 && n > 0 && !c->hp;             // mia -h: the chunked kernel only
  if (const char* e = getenv("MIAGPU_PASS1_FAST")) fast = fast && atoi(e) != 0;
  bool sweep = c->kmer_k <= 0 && lm.v[SW_CLASS] > 0 && n > 0 && !c->hp;
  if (const char* e = getenv("MIAGPU_PASS1_FAST")) sweep = sweep && atoi(e) != 0;
  c->p1_fast = c->p1_general = c->p1_skipped = 0;
  c->p1ev_valid = fast || sweep;
  if (sweep) {
    if (!pass1_sweep(c, lm)) return 0;
  } else if (!fast) {
    if (!launch_strip(c, 0, nullptr, 0, c->d_meta.p + 16)) return 0;
    c->p1_general = n;
  } else if (!pass1_fast(c, lm)) {
    return 0;
  }
  MIAGPU_CUDA(cudaEventRecord(c->ev[2], c->stream));
  if (n) {
    auto dl = [&](void* h, const void* d, size_t bytes) { return h ? cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, c->stream) : cudaSuccess; };
    MIAGPU_CUDA(dl(hits, c->d_hits.p, n * 4)); MIAGPU_CUDA(dl(score, c->d_score.p, n * 4)); MIAGPU_CUDA(dl(fw_score, c->d_fw.p, n * 4));
    MIAGPU_CUDA(dl(rc_score, c->d_rcs.p, n * 4)); MIAGPU_CUDA(dl(rc, c->d_rc_out.p, n)); MIAGPU_CUDA(dl(as, c->d_as_out.p, n * 4));
    MIAGPU_CUDA(dl(ae, c->d_ae_out.p, n * 4)); MIAGPU_CUDA(dl(start, c->d_start.p, n * 4)); MIAGPU_CUDA(dl(end, c->d_end.p, n * 4));
    MIAGPU_CUDA(dl(abr, c->d_abr.p, n * 4)); MIAGPU_CUDA(dl(n_runs, c->d_nruns.p, n * 4)); MIAGPU_CUDA(dl(runs, c->d_runs.p, n * MAX_RUNS * 2));
    MIAGPU_CUDA(dl(status, c->d_status.p, n));
  }
  MIAGPU_CUDA(cudaEventRecord(c->ev[3], c->stream));
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_kernels, c->ev[1], c->ev[2]));
  MIAGPU_CUDA(cudaEventElapsedTime(&c->ms_d2h, c->ev[2], c->ev[3]));
  c->ms_h2d = 0;
  if (c->p1ev_valid && getenv("MIAGPU_TRACE")) {
    float a = 0, b = 0, d = 0, e = 0;
    cudaEventElapsedTime(&a, c->ev[1], c->p1ev[0]); cudaEventElapsedTime(&b, c->p1ev[0], c->p1ev[1]);
    cudaEventElapsedTime(&d, c->p1ev[1], c->p1ev[2]); cudaEventElapsedTime(&e, c->p1ev[2], c->ev[2]);
    fprintf(stderr, "[miagpu trace] pass 1: seeding %.3f ms, pair kernels (+ host sync) %.3f ms, merge %.3f ms, general tail %.3f ms\n", a, b, d, e);
  }
  const int len1 = c->circular ? c->wrap_len : c->seq_len;
  c->dp_cells = 2 * (int64_t)len1 * c->total_bases;                        // nominal cells (SURVEY 8d)
  c->dp_cells_p1 = c->dp_cells;
  c->p1_eff = c->dp_cells;                                                 // without the filter every cell is computed
  if (fast) memcpy(&c->p1_eff, c->h_meta + P1_EFF, sizeof(int64_t));
  return 1;
}

extern "C" int miagpu_last_pass1_route(miagpu_ctx* c, uint8_t* route) {
  if (!c || !route) { set_error("miagpu_last_pass1_route: bad argument"); return 0; }
  if (c->p1_fast + c->p1_skipped == 0 && c->p1_general == c->n) { memset(route, 2, c->n); return 1; }   // the fast path was off
  MIAGPU_CUDA(cudaSetDevice(c->device));
  MIAGPU_CUDA(cudaMemcpy(route, c->d_route.p, c->n, cudaMemcpyDeviceToHost));
  return 1;
}

extern "C" int miagpu_last_pass1_cells(miagpu_ctx* c, int64_t* nominal, int64_t* effective) {
  if (!c) { set_error("miagpu_last_pass1_cells: bad argument"); return 0; }
  if (nominal) *nominal = c->dp_cells_p1;
  if (effective) *effective = c->p1_eff;
  return 1;
}

extern "C" int miagpu_last_pass1_stats(miagpu_ctx* c, int64_t* fast_reads, int64_t* general_reads, int64_t* skipped_reads) {
  if (!c) { set_error("miagpu_last_pass1_stats: bad argument"); return 0; }
  if (fast_reads) *fast_reads = c->p1_fast;
  if (general_reads) *general_reads = c->p1_general;
  if (skipped_reads) *skipped_reads = c->p1_skipped;
  return 1;
}

// keep / reverse-complement the resident reads in place (sg_align's accept + add_virgin_fs2fsdb + clean_FSDB)
__global__ void compact_kernel(int64_t n_new, const int32_t* src, const uint8_t* revcomp, const int64_t* off_old, const uint8_t* bases_old,
                               const int64_t* off_new, uint8_t* bases_new) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n_new) return;
  const int i = src[w];
  const int64_t o = off_old[i], L = off_old[i + 1] - o, d = off_new[w];
  const bool rcv = revcomp[w];
  for (int64_t j = lane; j < L; j += 32) {
    uint8_t b = rcv ? bases_old[o + L - 1 - j] : bases_old[o + j];
    if (rcv) {                                                             // revcom_char, map_align.c:418-431
      const char* from = "ABCDGHKMNRSTUVWXY";
      const char* to = "TVGHCDMKNYSAABWXR";
      uint8_t r = 'N';
      for (int q = 0; q < 17; q++) if (from[q] == b) r = to[q];
      b = b == '-' ? '-' : r;
    }
    bases_new[d + j] = b;
  }
}

extern "C" int miagpu_compact_reads(miagpu_ctx* c, const uint8_t* keep, const uint8_t* revcomp, int64_t* n_out) {
  if (!c || (c->n && !keep)) { set_error("miagpu_compact_reads: bad argument"); return 0; }
  misinc_invalidate(c, "miagpu_compact_reads has replaced the reads of that round");
  MIAGPU_CUDA(cudaSetDevice(c->device));
  std::vector<int64_t> off_old(c->n + 1), off_new(1, 0);
  if (c->n) MIAGPU_CUDA(cudaMemcpy(off_old.data(), c->d_off.p, (c->n + 1) * 8, cudaMemcpyDeviceToHost));
  std::vector<int32_t> src;
  std::vector<uint8_t> rcv;
  int maxL = 0;
  for (int64_t i = 0; i < c->n; i++)
    if (keep[i]) {
      src.push_back((int32_t)i);
      rcv.push_back(revcomp ? revcomp[i] : 0);
      off_new.push_back(off_new.back() + off_old[i + 1] - off_old[i]);
      maxL = std::max<int64_t>(maxL, off_old[i + 1] - off_old[i]);
    }
  const int64_t m = (int64_t)src.size();
  if (!c->d_bases2.reserve(off_new.back() + 16) || !c->d_off2.reserve(m + 1) || !c->d_src.reserve(m + 1) || !c->d_dropf.reserve(m + 1)) return 0;
  if (m) {
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_src.p, src.data(), m * 4, cudaMemcpyHostToDevice, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_dropf.p, rcv.data(), m, cudaMemcpyHostToDevice, c->stream));
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_off2.p, off_new.data(), (m + 1) * 8, cudaMemcpyHostToDevice, c->stream));
    compact_kernel<<<(unsigned)((m * 32 + 255) / 256), 256, 0, c->stream>>>(m, c->d_src.p, c->d_dropf.p, c->d_off.p, c->d_bases.p, c->d_off2.p, c->d_bases2.p);
    MIAGPU_CUDA(cudaGetLastError());
  } else {
    MIAGPU_CUDA(cudaMemcpyAsync(c->d_off2.p, off_new.data(), 8, cudaMemcpyHostToDevice, c->stream));
  }
  // the pass-1 alignment of the reads that stay, in FSDB order, becomes "the previous round" of the first round: slots that
  // pass 1 filled and no later round re-uses keep that content (slots.cuh)
  c->fs_prev_valid = false;
  if (m && c->d_start.cap && c->d_rc_out.cap &&
      c->d_runs_prev.reserve((size_t)m * MAX_RUNS) && c->d_nruns_prev.reserve(m) && c->d_abr_prev.reserve(m) && c->d_as_prev.reserve(m) &&
      c->d_ae_prev.reserve(m) && c->d_flip_prev.reserve(m)) {
    fs_prev_from_pass1_kernel<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(m, c->d_src.p, c->d_dropf.p, c->d_start.p, c->d_end.p, c->d_abr.p,
                                                                                 c->d_nruns.p, c->d_runs.p, c->d_rc_out.p, c->d_as_prev.p, c->d_ae_prev.p,
                                                                                 c->d_abr_prev.p, c->d_nruns_prev.p, c->d_runs_prev.p, c->d_flip_prev.p);
    MIAGPU_CUDA(cudaGetLastError());
    c->fs_prev_valid = true; c->fs_prev_pass1 = true; c->fs_prev_seq_len = c->seq_len;
  }
  MIAGPU_CUDA(cudaStreamSynchronize(c->stream));
  std::swap(c->d_bases, c->d_bases2);
  std::swap(c->d_off, c->d_off2);
  c->fs_on = false;
  c->n = m; c->cut_inputs_n = -1;
  c->total_bases = off_new.back();
  c->max_read_len = maxL;
  if (n_out) *n_out = m;
  return 1;
}


// host-side formats either side of the path (SURVEY 8 f2 / f3): FASTA / FASTQ reader, .maln writer
#include "hostio.hpp"

// write_ma of the round miagpu_iterate_resident just ran under miagpu_set_fsdb: the culled list follows the pointers
// (cull_maln_from_fsdb mia.c:463-476: front_asp, then back_asp of every unique_best read in FSDB order), so an AlnSeq that stale
// pointers reach appears once per pointer, with the smp codes of the last visit (fsdb.c:542-619) and the slot's sticky dropped flag.
// rd as for miagpu_write_maln (dropped_front / dropped_back / fsdb_order are not read: the slot flags come from the device).
extern "C" int miagpu_write_maln_fsdb(miagpu_ctx* c, const char* path, const miagpu_maln_header* hd, const miagpu_maln_reads* rd,
                                      int64_t* n_alnseqs_out) {
  using namespace hostio;
  if (!c || !c->fs_on || !path || !hd || !rd) { set_error("miagpu_write_maln_fsdb: call miagpu_set_fsdb and a round first"); return 0; }
  const int64_t n = c->n;
  if (rd->n != n || (n && (!rd->bases || !rd->offsets || !rd->rc || !rd->score || !rd->as || !rd->ae || !rd->abr || !rd->run_off || !rd->packed ||
                           !rd->ids || !rd->id_off))) { set_error("miagpu_write_maln_fsdb: incomplete read arrays"); return 0; }
  MIAGPU_CUDA(cudaSetDevice(c->device));
  std::vector<int32_t> front((size_t)n), back((size_t)n);
  std::vector<uint8_t> known((size_t)n), flag((size_t)c->fs_slot_cap);
  MIAGPU_CUDA(cudaMemcpy(flag.data(), c->d_slot_flag.p, flag.size(), cudaMemcpyDeviceToHost));
  if (n) {
    MIAGPU_CUDA(cudaMemcpy(front.data(), c->d_front_slot.p, n * 4, cudaMemcpyDeviceToHost));
    MIAGPU_CUDA(cudaMemcpy(back.data(), c->d_back_slot.p, n * 4, cudaMemcpyDeviceToHost));
    MIAGPU_CUDA(cudaMemcpy(known.data(), c->d_known.p, n, cudaMemcpyDeviceToHost));
  }
  const size_t nfz = c->fz.size();
  std::vector<uint8_t> fzb(nfz * FZ_BASES + 1);
  std::vector<uint16_t> fzr(nfz * MAX_RUNS + 1);
  std::vector<int32_t> fzn(nfz + 1);
  if (nfz) {
    MIAGPU_CUDA(cudaMemcpy(fzb.data(), c->d_fz_bases.p, nfz * FZ_BASES, cudaMemcpyDeviceToHost));
    MIAGPU_CUDA(cudaMemcpy(fzr.data(), c->d_fz_runs.p, nfz * MAX_RUNS * 2, cudaMemcpyDeviceToHost));
    MIAGPU_CUDA(cudaMemcpy(fzn.data(), c->d_fz_nruns.p, nfz * 4, cudaMemcpyDeviceToHost));
  }
  const FrozenView fzv{fzb.data(), fzr.data(), fzn.data(), FZ_BASES, MAX_RUNS};
  std::unordered_map<int32_t, const int32_t*> ov;                              // natural entry -> parameters of its slot's last visit
  for (size_t q = 0; q + 5 <= c->fs_patch_host.size(); q += 5) ov[c->fs_patch_host[q]] = &c->fs_patch_host[q];
  std::unordered_map<int64_t, const miagpu_ctx::FsExtra*> stale;                // 2 * holder + kind -> what the pointer sees
  for (const auto& x : c->fs_extra) stale[2 * (int64_t)x.holder + x.kind] = &x;
  const int L = hd->ref_len;
  auto with_params = [](Seg& sg, int fl, int total, int bias, int bf) { sg.ov = 1; sg.fl = fl; sg.total = total; sg.bias = bias; sg.bf = bf; };
  std::vector<Seg> segs;
  segs.reserve((size_t)n + 16);
  for (int64_t i = 0; i < n; i++) {
    if (rd->unique_best && !rd->unique_best[i]) continue;
    Seg f, b;
    bool split = false;
    if (known[i]) {
      split = natural_segs(rd, L, i, f, b) != 0;
      f.dropped = flag[front[i]];
      auto it = ov.find((int32_t)(2 * i));
      if (it != ov.end()) with_params(f, it->second[1], it->second[2], it->second[3], it->second[4]);
      segs.push_back(f);
      if (split) {
        b.dropped = flag[back[i]];
        it = ov.find((int32_t)(2 * i + 1));
        if (it != ov.end()) with_params(b, it->second[1], it->second[2], it->second[3], it->second[4]);
        segs.push_back(b);
      }
    }
    for (int kind = known[i] ? 1 : 0; kind < 2; kind++) {
      if (kind == 1 && (split || back[i] < 0)) continue;
      auto it = stale.find(2 * i + kind);
      if (it == stale.end()) { set_error("miagpu_write_maln_fsdb: the pointer of read %lld was not resolved by the last round", (long long)i); return 0; }
      const miagpu_ctx::FsExtra& x = *it->second;
      Seg sg;
      if (x.frozen >= 0) {
        const miagpu_ctx::FzHost& z = c->fz[x.frozen];
        sg.read = z.read; sg.start = z.start; sg.end = z.start + z.cols - 1; sg.col0 = 0; sg.ncol = z.cols; sg.smp_n = z.cols; sg.seg = (char)z.seg;
        sg.fz = x.frozen; sg.fz_score = z.score; sg.fz_rc = z.rc; sg.fz_num_inputs = z.num_inputs;
      } else {
        Seg of, ob;
        const int64_t j = x.live_entry >> 1;
        natural_segs(rd, L, j, of, ob);
        sg = (x.live_entry & 1) ? ob : of;
      }
      sg.dropped = flag[x.slot];
      with_params(sg, x.front_len, x.total_len, x.act_bias, x.back_formula);
      segs.push_back(sg);
    }
  }
  return maln_emit(path, hd, rd, segs, &fzv, n_alnseqs_out);
}
