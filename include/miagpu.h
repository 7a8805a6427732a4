/* miagpu.h -- C ABI of the B200-native hot path for the Mapping Iterative
 * Assembler (MIA).  Plain C, no CUDA / torch types in any signature.
 *
 * Every entry point sits at a call site of the reference's own C host code
 * (citations are /root/reference/src/<file>:<line>); INTEGRATION.md shows the
 * stubs a maintainer of the reference would add.  Conventions follow the
 * reference (SURVEY.md section 8b): functions return 1 on success and 0 on
 * failure, never throw; the message of the last failure is available from
 * miagpu_last_error().  There is NO CPU fallback: without a CUDA device every
 * compute call fails loudly.
 *
 * Compile-time limits are the reference's (params.h): reads <= 256 bases
 * (INIT_ALN_SEQ_LEN), alignment strings <= 512 columns, k <= 14
 * (MAX_KMER_LEN), <= 128 positions per k-mer (MAX_KMER_POS), saturation at 128
 * hits (KMER_SATURATE), mask buffer 10 (ALIGN_MASK_BUFFER), realign buffer 50
 * (REALIGN_BUFFER), GOP 1000, GEP 200, PSSM depth 15, first-round cutoff 2000.
 */
#ifndef MIAGPU_H
#define MIAGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MIAGPU_MAX_READ      256      /* INIT_ALN_SEQ_LEN, params.h:71 */
#define MIAGPU_PSSM_INTS     775      /* int sm[31][5][5], types.h:155-158 */
#define MIAGPU_MAX_RUNS      24       /* alignment runs returned per read */
#define MIAGPU_NBUCKET       10       /* window-width buckets of the realign kernels */
#define MIAGPU_COUNTS_PER_COL 10      /* As,Cs,Gs,Ts,gaps,cov,scoreA,scoreC,scoreG,scoreT (types.h:198-211) */

/* Alignment run: (type << 14) | length, in 5'->3' order of the stored read.
 *   type 0  M  read base aligned to reference base (both strings advance)
 *   type 1  I  read bases against '-' in the reference string (mia.c:1466-1476)
 *   type 2  D  reference bases against '-' in the read string   (mia.c:1477-1487)
 * The pair of gapped strings populate_pwaln_to_begin builds (mia.c:1440-1497)
 * is exactly the expansion of these runs starting at reference column `as`
 * and read row `abr`. */
#define MIAGPU_RUN_M 0
#define MIAGPU_RUN_I 1
#define MIAGPU_RUN_D 2
#define MIAGPU_RUN_TYPE(x) ((x) >> 14)
#define MIAGPU_RUN_LEN(x)  ((x) & 0x3fff)

/* per-read status bits (status[] outputs) */
#define MIAGPU_ST_OK          0
#define MIAGPU_ST_RUNS_OVERFLOW 1     /* more than MIAGPU_MAX_RUNS runs: n_runs = -1 */
#define MIAGPU_ST_SKIPPED     2       /* pass 1: no k-mer hit, read not aligned (mia_main.c:781) */
#define MIAGPU_ST_STR_OVERFLOW 4      /* alignment longer than the reference's 512-column buffers */
#define MIAGPU_ST_UNSUPPORTED  0x80    /* window wider than the register-tiled kernels handle (reported, never silent) */

typedef struct miagpu_ctx miagpu_ctx;

/* ---- lifetime.  Replaces init_alignment x2 + init_kpa (mia_main.c:659-690). */
int         miagpu_device_count( void );
int         miagpu_create( miagpu_ctx** out, int device );
void        miagpu_destroy( miagpu_ctx* ctx );
const char* miagpu_last_error( void );
const char* miagpu_version( void );

/* ---- a1. Scoring matrices.  fwd is PSSM.sm as read_pssm / init_flatsubmat
 * fill it (io.c:408-503, pssm.c:96-126); the strand-reversed copy
 * (revcom_submat, pssm.c:53-93) is derived inside.  Entries must satisfy
 * |x| <= 2000 (the packed-key DP needs 256*|x| + 200*511 < 2^20). */
int miagpu_set_pssm( miagpu_ctx* ctx, const int32_t* fwd );
int miagpu_get_pssm( miagpu_ctx* ctx, int32_t* fwd, int32_t* rev );
/* read_pssm (io.c:408-503; call site mia_main.c:299-335): the matrix file -> int fwd[31][5][5] for miagpu_set_pssm, with the
 * reference's N column (-100) and non-ACGT reference row (-10).  Host only.  A malformed file returns 0 (the reference exits). */
int miagpu_read_pssm( const char* path, int32_t* fwd );

/* ---- reference / current consensus.  seq is what read_fasta_ref left in
 * RefSeq.seq (case preserved, so that -M soft masking still works); the
 * library appends the circular wrap (add_ref_wrap, mia.c:657-689), builds the
 * reverse complement when with_rc (make_reverse_complement, io.c:388-398) and
 * upper-cases both (make_ref_upper, mia.c:642-648).  Called once before pass 1
 * (mia_main.c:637-733) and once per iteration with the new consensus
 * (reiterate_assembly, mia_main.c:43-78; with_rc = 0 there). */
int miagpu_set_reference( miagpu_ctx* ctx, const char* seq, int seq_len,
                          int circular, int with_rc );
int miagpu_ref_wrap_len( miagpu_ctx* ctx );

/* ---- a2. k-mer tables of both strands over the wrapped, NOT yet upper-cased
 * reference (populate_kpa, kmer.c:153-168; call site mia_main.c:659-672).
 * k <= 0 disables the filter (all masks ones, new_kmer_filter kmer.c:251-255). */
int miagpu_build_kmers( miagpu_ctx* ctx, int k, int soft_mask );

/* ---- reads.  bases = all reads concatenated, upper-case ASCII as read_fasta /
 * read_fastq store them (io.c:102, 251); offsets[n+1].  The batch stays
 * resident in HBM until the next upload.  store_rc (nullable): 1 = replace the
 * read by its reverse complement on upload (what add_virgin_fs2fsdb does once
 * the strand is known, fsdb.c:209-227). */
int miagpu_upload_reads( miagpu_ctx* ctx, int64_t n, const uint8_t* bases,
                         const int64_t* offsets );

/* ---- a3+a5..a8. Pass 1 over the resident reads: k-mer filter, both-strand
 * whole-reference DP with the forward matrix, strand pick, traceback and the
 * coordinate fix-ups of sg_align (mia_main.c:781-796; mia.c:1500-1610).
 * Outputs (host arrays of n, any may be NULL):
 *   hits      return value of new_kmer_filter (0 => skipped)
 *   score     best_score of the chosen strand; fw_score / rc_score both strands
 *   rc        1 if the reverse strand won (ties go to rc, mia.c:1549-1554)
 *   as, ae    FragSeq.as / ae after mia.c:1587-1604
 *   start,end PWAlnFrag start / end after the "end > seq_len" fix (mia.c:1606-1610)
 *   abr       first aligned read row (soft clip), in the orientation aligned
 *   n_runs, runs[n*MIAGPU_MAX_RUNS]  alignment of the chosen strand, already
 *             reverse-complemented for rc (revcom_PWAF), i.e. in forward
 *             reference orientation starting at `start`
 * The accept / strand_known / split decisions (mia.c:1614-1658) are pure
 * functions of these and stay in the host code. */
int miagpu_pass1( miagpu_ctx* ctx, int32_t* hits, int32_t* score,
                  int32_t* fw_score, int32_t* rc_score, uint8_t* rc,
                  int32_t* as, int32_t* ae, int32_t* start, int32_t* end,
                  int32_t* abr, int32_t* n_runs, uint16_t* runs,
                  uint8_t* status );

/* How the last miagpu_pass1 was computed: reads finished by the windowed 16-bit
 * pair kernels (k-mer filter on, all hits of a strand on neighbouring diagonals:
 * csrc/pass1.cuh), reads the general chunked kernel took, reads without a hit. */
int miagpu_last_pass1_stats( miagpu_ctx* ctx, int64_t* fast_reads,
                             int64_t* general_reads, int64_t* skipped_reads );
/* DP cells of the last miagpu_pass1 (SURVEY 8d): nominal = 2 * L * len1 per read (what the reference visits), effective = L * the
 * columns new_kmer_filter unmasks, summed over both strands (a strand with >= 128 hits, or with more than 12 separate stretches,
 * counts whole); equal without the filter */
int miagpu_last_pass1_cells( miagpu_ctx* ctx, int64_t* nominal, int64_t* effective );
/* ---- f4. mia -h (hp_special, mia_main.c:424, 497; init_alignment( ..., hp_special ) mia.c:988-1028): from now on
 * dyn_prog's two homopolymer-discounted gap candidates (mia.c:882-905, hp_discount_penalty mia.c:1096-1134,
 * pop_hpl_and_hps mia.c:1193-1234) take part in every alignment of this context: pass 1 (homopolymers of the whole
 * strands, mia_main.c:735-739), the rounds (of the read's window, mia_main.c:221-224), the -D attempts
 * (mia_main.c:132-134, 158-160).  They all run in the chunked 32-bit kernel; the 16-bit kernels do not carry the
 * candidates.  The reads' raw bytes are compared with the reference's bases (mia.c:886): the reference may hold
 * A C G T N only (anything else is refused at the first alignment).  miagpu_trim and miagpu_align_windows with
 * sg5 = 0 refuse a context in this mode. */
int miagpu_set_homopolymer( miagpu_ctx* ctx, int on );

/* per read of the last miagpu_pass1: 0 no k-mer hit, 1 finished by the pair kernels, 2 general kernel
 * (decided while seeding), 3 general kernel (a job of the read left the 16-bit frame), 4 pair kernels for the scores +
 * the windowed 32-bit kernel for the winning stretch's trace (the winner's path was not a plain diagonal; counted with 1
 * in miagpu_last_pass1_stats) */
int miagpu_last_pass1_route( miagpu_ctx* ctx, uint8_t* route );

/* After pass 1 the host tells the device which resident reads to keep and in
 * which orientation (sg_align's accept test + add_virgin_fs2fsdb + clean_FSDB):
 * keep[i] in {0,1}; revcomp[i] = 1 stores the reverse complement.  Reads are
 * compacted in order; returns the new count through n_out. */
int miagpu_compact_reads( miagpu_ctx* ctx, const uint8_t* keep,
                          const uint8_t* revcomp, int64_t* n_out );

/* ---- a9 (+a5..a7). One round of reiterate_assembly's per-read body
 * (mia_main.c:178-257) over the resident reads against the current reference:
 * window [max(0,as-50), ae+50) with the clamp at mia_main.c:197-212, matrix by
 * strand (179-184), sg5 = 1, unmasked DP, first-max end cell, traceback.
 * Inputs (host, n each): rc, as, ae.  Outputs (host, n each, nullable):
 *   score, as_out, ae_out (absolute), abr, n_runs, runs[n*MIAGPU_MAX_RUNS],
 *   status.  Results are in input order. */
int miagpu_realign( miagpu_ctx* ctx, const uint8_t* rc, const int32_t* as,
                    const int32_t* ae, int32_t* score, int32_t* as_out,
                    int32_t* ae_out, int32_t* abr, int32_t* n_runs,
                    uint16_t* runs, uint8_t* status );

/* The run lists of the last realign / pass 1 in packed form: the n_runs[i] valid runs
 * of every read concatenated in read order (run_off[n+1], nullable; packed nullable
 * = only report *total).  Moves sum(n_runs)*2 bytes instead of n*MIAGPU_MAX_RUNS*2. */
int miagpu_get_runs_packed( miagpu_ctx* ctx, int64_t* run_off, uint16_t* packed,
                            int64_t capacity, int64_t* total );

/* Convenience form used by the end-to-end benchmark: upload + realign +
 * download in one call with host buffers only. */
int miagpu_realign_host( miagpu_ctx* ctx, int64_t n, const uint8_t* bases,
                         const int64_t* offsets, const uint8_t* rc,
                         const int32_t* as, const int32_t* ae, int32_t* score,
                         int32_t* as_out, int32_t* ae_out, int32_t* abr,
                         int32_t* n_runs, uint16_t* runs, uint8_t* status );

/* ---- a10..a13. Column accumulation and base calling over the alignments the
 * last miagpu_pass1 / miagpu_realign left on the device.
 *
 * The host keeps the reference's own bookkeeping -- which AlnSeq slot belongs
 * to which read (FragSeq.front_asp / back_asp), the sticky AlnSeq.dropped flag
 * (H10), the back pointer that reiterate_assembly never clears
 * (mia_main.c:273-276) -- and describes culled_maln->AlnSeqArray to the device
 * as a list of entries, one per AlnSeq in the list (duplicates allowed).
 * The device derives AlnSeq.seq / ins / smp on the fly from the run lists
 * (merge_pwaln_into_maln map_align.c:866-954, split_pwaln mia.c:1376-1438,
 * pop_smp_from_FSDB fsdb.c:542-619), takes the per-position maximum insert
 * length (ref->gaps as left by cull_maln_from_fsdb, mia.c:486-504), adds every
 * covered column into the BaseCounts accumulators (add_base
 * map_align.c:229-263, find_ins_cons 444-510) and calls bases (find_consensus
 * map_align.c:294-391; consensus_assembly_string mia.c:515-603).
 *
 * An alignment is a sequence of reference columns (M and D runs) numbered from
 * 0 at its first column; an entry covers columns [col_begin, col_begin +
 * col_count) and places the first of them at reference position ref_pos
 * (AlnSeq.start).  Inserted bases belong to the column that follows them
 * (AlnSeq.ins[], map_align.c:906-927).  For a whole alignment: col_begin = 0,
 * ref_pos = start; for a wrap-split one the 'f' entry ends at seq_len-1 and the
 * 'b' entry has ref_pos = 0 (mia.c:1419-1422).
 * smp (fsdb.c:563-614): with act = act_bias + (read bases consumed before the
 * column, inserted ones included),
 *     dist_front = back_formula ? front_len + act : act
 *     dist_back  = total_len - act - 1
 *     depth = dist_front <= 15 ? dist_front : dist_back < 15 ? 30 - dist_back : 15
 */
typedef struct {
  int32_t read;         /* index into the resident reads */
  int32_t col_begin;
  int32_t col_count;
  int32_t ref_pos;      /* AlnSeq.start */
  int32_t front_len;    /* asp_len(front_asp) of the read that holds the pointer (fsdb.c:553) */
  int32_t total_len;    /* front_seq_len + back_seq_len (fsdb.c:554-559) */
  int32_t act_bias;     /* 0 for a read's own segments */
  uint8_t dropped;      /* AlnSeq.dropped: excluded from base columns, NOT from insert columns */
  uint8_t back_formula; /* 0 = front loop (fsdb.c:563-584), 1 = back loop (588-614) */
  uint8_t reserved[2];
} miagpu_entry;

/* Accumulate + call in one step (single GPU).  Outputs are host arrays, any may
 * be NULL: gaps_out[seq_len] = ref->gaps for positions < seq_len;
 * counts_out[seq_len*10] = BaseCounts of every base column (MIAGPU_COUNTS_PER_COL
 * order); cons_out receives at most seq_len + sum(gaps) + 1 chars and must hold
 * seq_len * 4 + 4096 bytes unless miagpu_set_cons_capacity said otherwise: a consensus
 * that does not fit fails the call (nothing is written); *cons_len its strlen. */
int miagpu_consensus( miagpu_ctx* ctx, int64_t n_entries,
                      const miagpu_entry* entries, int cons_code,
                      int32_t* gaps_out, int32_t* counts_out, char* cons_out,
                      int32_t* cons_len );

/* Multi-GPU (SURVEY 8e): the same in three steps so that the caller can
 * all-reduce between them (reads are sharded, the reference is replicated):
 *   _accumulate_gaps   -> device int32 gaps[seq_len]          reduce with MAX
 *   _accumulate_counts -> device int32 counts[10][n_cols]      reduce with SUM
 *                         (n_cols = seq_len + sum(gaps); plane-major)
 *   _call              -> consensus from the reduced buffers
 * The insert-column layout is a function of the reduced gaps only, so every
 * rank derives the same layout.  Integer sums: bit-identical for any number
 * of GPUs and any order. */
int miagpu_accumulate_gaps( miagpu_ctx* ctx, int64_t n_entries,
                            const miagpu_entry* entries, void** dev_gaps,
                            int64_t* n_gaps );
int miagpu_accumulate_counts( miagpu_ctx* ctx, void** dev_counts,
                              int64_t* n_counts );
int miagpu_call( miagpu_ctx* ctx, int cons_code, int32_t* gaps_out,
                 int32_t* counts_out, char* cons_out, int32_t* cons_len );
/* Size in bytes of the buffer the caller passes as cons_out to the calls of this context
 * (0 = the default, seq_len * 4 + 4096).  The reference sizes its consensus string from
 * the gaps it has just counted (consensus_assembly_string, mia.c:527-533); a caller of
 * this library allocates before the gaps are known, so it announces its buffer and a
 * longer consensus fails the call rather than overrunning it. */
int miagpu_set_cons_capacity( miagpu_ctx* ctx, int64_t bytes );

/* The same with the entry list built ON THE DEVICE from the resident alignments:
 * every read contributes its own fresh segment(s) (no stale AlnSeq pointers to
 * describe).  dropped_front / dropped_back: host arrays of n flags for the
 * read's whole-or-front and back AlnSeq (nullable = nothing dropped): 0 = in the
 * culled list, 1 = AlnSeq.dropped, 2 (in dropped_front) = the read is not
 * unique_best and therefore not in the culled list at all (mia.c:466). */
int miagpu_consensus_natural( miagpu_ctx* ctx, const uint8_t* dropped_front,
                              const uint8_t* dropped_back, int cons_code,
                              int32_t* gaps_out, int32_t* counts_out,
                              char* cons_out, int32_t* cons_len );

int miagpu_accumulate_gaps_natural( miagpu_ctx* ctx, const uint8_t* dropped_front,
                                    const uint8_t* dropped_back, void** dev_gaps,
                                    int64_t* n_gaps );

/* ---- a12 on the host (H8; scores in host memory, e.g. gathered from several
 * GPUs): the score/length regression of
 * find_fsdb_score_cut (fsdb.c:269-383, double sums in FSDB order) and the
 * per-read test of cull_maln_from_fsdb (mia.c:418-479): below[i] = 1 iff
 * score[i] < (hard_cut > 0 ? hard_cut : intercept + slope*seq_len[i]).  The
 * caller ORs below[] into its sticky per-slot dropped flags (H10). */
int miagpu_score_cut( int64_t n, const int32_t* seq_len, const int32_t* score,
                      const uint8_t* unique_best, double* slope,
                      double* intercept );
int miagpu_cull_flags( int64_t n, const int32_t* seq_len, const int32_t* score,
                       const uint8_t* unique_best, int hard_cut,
                       int score_cut_set, double slope, double intercept,
                       uint8_t* below );

/* ---- a9..a13 in one call for a batch that lives in host memory: one iteration of
 * mia_main.c:931-963.  Equivalent to miagpu_realign_host + miagpu_get_runs_packed +
 * miagpu_cull_flags (dropped[i] |= below[i], sticky as in H10) + miagpu_consensus_natural
 * (every read owns its fresh AlnSeq segments; dropped[] serves the front and the back
 * segment), pipelined over upload / compute / download streams.  The score cut runs
 * on the device over the scores where they are (csrc/scorecut.cuh): integer sums,
 * then the two double-precision chains of find_fsdb_score_cut block by block with
 * a proof per block that the block-wise result equals the reference's read-by-read
 * rounding; blocks without a proof are summed read by read on the host.  Slope,
 * intercept and flags are bit-identical to miagpu_score_cut / miagpu_cull_flags.
 * seq_len / unique_best / hard_cut / score_cut_set / slope / intercept as in
 * miagpu_cull_flags; a read that is not unique_best is left out of the fit, is not
 * tested against the cut and is absent from the consensus (mia.c:466).
 * packed_runs (nullable) as in miagpu_get_runs_packed. */
int miagpu_iterate_host( miagpu_ctx* ctx, int64_t n, const uint8_t* bases,
                         const int64_t* offsets, const uint8_t* rc, const int32_t* as,
                         const int32_t* ae, int32_t* score, int32_t* as_out,
                         int32_t* ae_out, int32_t* abr, int32_t* n_runs, uint8_t* status,
                         uint16_t* packed_runs, int64_t capacity, int64_t* total_runs,
                         const int32_t* seq_len, const uint8_t* unique_best, int hard_cut,
                         int score_cut_set, double slope, double intercept,
                         uint8_t* dropped, int cons_code, int32_t* gaps_out,
                         char* cons_out, int32_t* cons_len );

/* The same round with everything resident in HBM (reads from miagpu_upload_reads,
 * rc/as/ae from miagpu_set_alignment_inputs, and the score cut's per-read inputs
 * from miagpu_set_cut_inputs: FragSeq.seq_len, unique_best (nullable = all 1),
 * the sticky AlnSeq.dropped flags of earlier rounds (nullable = none)).  The
 * sticky flags stay on the device and keep accumulating from round to round
 * (H10); miagpu_reset_dropped clears them.  Outputs are nullable host arrays:
 * slope_out / intercept_out (the fit, or the values passed in when
 * score_cut_set), dropped[n] (sticky flags after this round), gaps_out[seq_len],
 * cons_out / cons_len as in miagpu_consensus. */
int miagpu_set_cut_inputs( miagpu_ctx* ctx, const int32_t* seq_len,
                           const uint8_t* unique_best, const uint8_t* dropped );
int miagpu_reset_dropped( miagpu_ctx* ctx );
int miagpu_iterate_resident( miagpu_ctx* ctx, int hard_cut, int score_cut_set,
                             double slope, double intercept, int cons_code,
                             double* slope_out, double* intercept_out,
                             uint8_t* dropped, int32_t* gaps_out, char* cons_out,
                             int32_t* cons_len );

/* ---- a8 / a9: the reference's FragSeq -> AlnSeq POINTER semantics in the one-call rounds.
 * In the reference an AlnSeq is an object in maln->AlnSeqArray[k] ("slot" k) that every round re-uses for the k-th segment it
 * merges in FSDB order (merge_pwaln_into_maln map_align.c:866-954: one slot per read, two per wrap-split read), and a FragSeq
 * holds pointers to its slots.  Three consequences that a "every read owns its fresh AlnSeqs" model misses:
 *   - AlnSeq.dropped is sticky per SLOT (H10: mia.c:471-478 only sets it, map_align.c:885-893 copies everything else): when
 *     the split pattern changes, later reads slide onto slots whose flags other reads set;
 *   - reiterate_assembly never clears back_asp (mia_main.c:273-276): a read that was wrap-split once keeps a stale pointer;
 *   - a read whose pass-1 score is <= 2000 has strand_known = 0 (mia.c:1653; accepted at exactly 2000, or at any score under
 *     -D, mia.c:1614) and is never realigned (mia_main.c:178): both its pass-1 pointers stay for ever.
 * pop_smp_from_FSDB, cull_maln_from_fsdb and consensus_assembly_string follow the pointers, whatever they point at.
 * miagpu_set_fsdb hands the state after pass 1 to the device (call it after miagpu_compact_reads, which keeps the pass-1
 * alignments of the reads that stay, and miagpu_set_alignment_inputs); from then on miagpu_iterate_resident reproduces all of
 * the above: slot numbers by a scan over the reads, flags per slot, stale pointers resolved into extra list entries, slot
 * content that is no longer live kept as it was (its inserts freed, mia_main.c:80-92).
 *   seq_len, unique_best (nullable), score     FragSeq.seq_len / unique_best / score in FSDB order
 *   strand_known (nullable = all 1)            FragSeq.strand_known
 *   front_slot, back_slot (-1 = NULL)          FragSeq.front_asp / back_asp as indices into the pass-1 AlnSeqArray, n_slots its
 *                                              length (maln->num_aln_seqs after pass 1); both NULL = nothing merged yet
 *   slot_dropped                               AlnSeq.dropped after the pass-1 cull (mia_main.c:848), n_slots flags; with
 *                                              front_slot == NULL: one flag per READ, applied to the slots of the first round
 *   distant_ref                                -D: miagpu_distant_retry before every round but the first; find_alignable_len
 *                                              (mia.c:69-91) decides a read's threshold in the cull (mia.c:460-463) */
int miagpu_set_fsdb( miagpu_ctx* ctx, const int32_t* seq_len, const uint8_t* unique_best, const int32_t* score,
                     const uint8_t* strand_known, const int32_t* front_slot, const int32_t* back_slot, int64_t n_slots,
                     const uint8_t* slot_dropped, int distant_ref );
/* the state after the last round (host arrays of n, all nullable): strand_known, rc, the pointers, AlnSeq.dropped behind them */
int miagpu_get_fsdb( miagpu_ctx* ctx, uint8_t* strand_known, uint8_t* rc, int32_t* front_slot, int32_t* back_slot,
                     uint8_t* dropped_front, uint8_t* dropped_back, int64_t* n_slots );
/* last round: AlnSeq slots merged, stale pointers followed, list entries they added, slot contents kept frozen so far */
int miagpu_last_fsdb_stats( miagpu_ctx* ctx, int64_t* n_slots, int64_t* stale_pointers, int64_t* extra_entries, int64_t* frozen );
/* -D, from iteration 2 on (mia_main.c:120-174): every strand-unknown read against the WHOLE current reference -- as it is stored,
 * with whatever matrix the read before it left in the Alignment (H6: both variants are computed on the device, the chain over the
 * reads is resolved on the host), then reverse-complemented with the strand-reversed matrix; a read that scores above 2000 learns
 * its strand, as / ae / score (and is stored reverse-complemented when the reverse attempt wins).  Call after
 * miagpu_set_reference and before miagpu_iterate_resident; does nothing in the first round or without distant_ref. */
int miagpu_distant_retry( miagpu_ctx* ctx, int64_t* n_tried, int64_t* n_learned );
/* The same in two steps, for reads sharded over several contexts (miagpu_shard_*): the matrix the forward attempt of a shard's
 * FIRST read runs with is the one the LAST read of the shard before it left (H6 does not stop at a shard boundary).
 *   _begin  the attempts of the local strand-unknown reads on the device; state_after[s] (two ints) = the matrix the last local
 *           read leaves -- 0 forward, 1 strand-reversed -- if the first one is entered with s: the identity for a shard without
 *           reads, a constant as soon as one local read's strand is known.  In the first round nothing is tried (iter_num > 1,
 *           mia_main.c:122) and state_after describes the untouched reads.
 *   the caller all-gathers the ranks' state_after pairs (two ints per rank) and folds them in rank order, starting from what
 *   the last round left (0 before the first round)
 *   _end    the local chain entered with state_in, the reads that learned their strand updated on the device.
 * miagpu_distant_retry = _begin + _end with the state this context carried over from its own previous round. */
int miagpu_distant_retry_begin( miagpu_ctx* ctx, int64_t* n_tried, int32_t* state_after );
int miagpu_distant_retry_end( miagpu_ctx* ctx, int state_in, int64_t* n_learned );

/* ---- 8e. The same round with the reads sharded over `world` GPUs of one box: one context per GPU (one process per GPU, or one
 * host thread per GPU: host/mia_gpu.c), reads partitioned contiguously in FSDB order (rank 0 holds the first reads), reference,
 * matrices and k-mer tables replicated.  The library links no communication library; between the phases the caller runs ONE
 * collective each, on miagpu_stream(), over device buffers the library hands out (ncclAllReduce / ncclAllGather in C,
 * torch.distributed in bench.py; INTEGRATION.md shows both):
 *
 *   miagpu_shard_begin       realign the resident local reads (inputs as for miagpu_iterate_resident); or
 *   miagpu_shard_begin_host  the same for a local batch in host memory (arguments as for miagpu_iterate_host)
 *        -> all-reduce  MAX, int32, max_words words at max_buf: per-position insert maxima, best score per read length, and one
 *                       header row per rank with that rank's integer sums (zero elsewhere: the MAX gathers them)
 *   miagpu_shard_fit         this rank's part of find_fsdb_score_cut (fsdb.c:269-383): xbar / ybar from the sums of all ranks, then
 *                            the two chains over the LOCAL reads as block records (integer increments per 512 reads in the binade
 *                            the running sum is predicted to be in, with a proof per block), plus the keys of the few blocks that
 *                            may have to be added read by read; beside it the column accumulation of the local reads
 *        -> all-gather  gather_send (gather_words uint32) into gather_recv (world * gather_words, rank order): about 50 bytes per
 *                       512 reads.  gather_words = 0 (the cut was given: -H / -S -N): nothing to gather
 *   miagpu_shard_cut         every rank stitches the same chains from the records of ALL ranks in rank order = FSDB order and gets the
 *                            same slope / intercept, bit for bit what one GPU computes over the concatenated reads; cull flags of
 *                            the local reads (mia.c:452-470, sticky as in H10), the newly dropped reads leave the base columns
 *        -> all-reduce  SUM, int32, sum_words words at sum_buf (the column planes)
 *   miagpu_shard_finish      base calling (identical on every rank) and downloads: dropped[n] = the local reads' sticky flags,
 *                            packed_runs / total_runs as in miagpu_get_runs_packed, gaps_out / cons_out / cons_len as in
 *                            miagpu_consensus.  All nullable.
 *
 * n_max = the largest local read count of any rank (the same value on every rank).  hard_cut / score_cut_set / slope / intercept
 * as in miagpu_cull_flags.  world = 1 needs no collectives (gather_recv must still receive a copy of gather_send) and equals
 * miagpu_iterate_resident / miagpu_iterate_host.  With miagpu_set_cut_inputs a sharded round gives every read its own AlnSeqs
 * and one sticky flag; with miagpu_set_fsdb it follows the reference's pointers (see miagpu_shard_flags below). */
int miagpu_shard_begin( miagpu_ctx* ctx, int world, int rank, int64_t n_max, int hard_cut,
                        int score_cut_set, double slope, double intercept,
                        void** max_buf, int64_t* max_words );
int miagpu_shard_begin_host( miagpu_ctx* ctx, int world, int rank, int64_t n_max, int64_t n,
                             const uint8_t* bases, const int64_t* offsets, const uint8_t* rc,
                             const int32_t* as, const int32_t* ae, int32_t* score,
                             int32_t* as_out, int32_t* ae_out, int32_t* abr, int32_t* n_runs,
                             uint8_t* status, const int32_t* seq_len, const uint8_t* unique_best,
                             const uint8_t* dropped, int hard_cut, int score_cut_set,
                             double slope, double intercept, void** max_buf, int64_t* max_words );
int miagpu_shard_fit( miagpu_ctx* ctx, void** gather_send, void** gather_recv, int64_t* gather_words );
int miagpu_shard_cut( miagpu_ctx* ctx, double* slope_out, double* intercept_out,
                      void** sum_buf, int64_t* sum_words );
int miagpu_shard_finish( miagpu_ctx* ctx, int cons_code, uint8_t* dropped,
                         uint16_t* packed_runs, int64_t capacity, int64_t* total_runs,
                         int32_t* gaps_out, char* cons_out, int32_t* cons_len );

/* Pointer state (miagpu_set_fsdb) in sharded rounds.  Slot numbers run over the reads of ALL ranks in FSDB order: a rank passes
 * miagpu_set_fsdb the GLOBAL slot numbers of its reads' pass-1 pointers, the global slot count and the flags of all slots.  A
 * round numbers its slots from the ranks' slot counts (they travel in the header rows of the MAX all-reduce), follows the local
 * reads' pointers as a one-GPU round does, and refuses a stale pointer whose slot a read of another rank owns this round (or
 * whose last content lives on another rank): without -D such a pointer sits within a few reads of a shard boundary; under -D the
 * stale pass-1 pointers of strand-unknown reads reach as far as there are such reads before them, so large -D runs belong on one
 * GPU (BASELINE configs[3], 2 M reads: 1.8 s, profiles/r02_c4_distant.md).  AlnSeq.dropped lives in
 * the slots, and the slots a rank's reads take drift from round to round, so every rank keeps the flags of all slots: after
 * miagpu_shard_finish the caller MAX-reduces this buffer (one byte per slot) over the ranks, before the next miagpu_shard_begin.
 * *bytes = 0: no pointer state, nothing to do.  -D: miagpu_distant_retry_begin / _end before miagpu_shard_begin.  The repeat
 * filter is not available in sharded rounds. */
int miagpu_shard_flags( miagpu_ctx* ctx, void** flag_buf, int64_t* bytes );
/* chain blocks of the last round's regression that were summed read by read on the host, and how many of
 * those needed an extra device fetch (sharded rounds prefetch the likely ones with the block records) */
int miagpu_last_cut_stats( miagpu_ctx* ctx, int64_t* serial_blocks, int64_t* fetched_blocks );

/* Device-resident round (reads, rc, as, ae stay in HBM between calls): */
int miagpu_set_alignment_inputs( miagpu_ctx* ctx, const uint8_t* rc,
                                 const int32_t* as, const int32_t* ae );
int miagpu_realign_resident( miagpu_ctx* ctx );
/* The last round's as_out / ae_out become the resident as / ae of the next round (fs->as, fs->ae:
 * mia_main.c:252-256); score / as / ae (nullable host arrays of n) receive this round's values. */
int miagpu_adopt_alignment( miagpu_ctx* ctx, int32_t* score, int32_t* as, int32_t* ae );

/* ---- 8f4 (second client). The bare alignment sequence that ccheck runs per read (ccheck.cc:571-603: pop_s1c_in_a,
 * pop_s2c_in_a, dyn_prog, max_sg_score, find_align_begin, populate_pwaln_to_begin) and that reiterate_assembly runs after
 * its window rule: every resident read against its own stretch [win_start, win_start + win_len) of the resident reference
 * (for ccheck: the lifted-over consensus pieces back to back, set with miagpu_set_reference( circular = 0 ); matrix =
 * init_flatsubmat through miagpu_set_pssm), unmasked, sg5 as given at every window width (windows over 512 columns go to the
 * chunked kernel, which takes sg5 too; homopolymer mode refuses sg5 = 0), rc[i] picks the strand-reversed matrix.  No window rule,
 * no fall-back to the whole reference; a window may be shorter than its read.  Outputs as miagpu_realign (as_out / ae_out are
 * reference coordinates: abc + win_start, aec + win_start).  Overwrites the resident as / ae of
 * miagpu_set_alignment_inputs. */
int miagpu_align_windows( miagpu_ctx* ctx, const uint8_t* rc, const int32_t* win_start,
                          const int32_t* win_len, int sg5, int32_t* score, int32_t* as_out,
                          int32_t* ae_out, int32_t* abr, int32_t* n_runs, uint16_t* runs,
                          uint8_t* status );

/* The alignment the last round left on the device, as miagpu_realign returns it (host arrays of n, all nullable):
 * after miagpu_iterate_resident / miagpu_shard_finish this plus miagpu_get_runs_packed is what miagpu_write_maln takes. */
int miagpu_get_alignment( miagpu_ctx* ctx, int32_t* score, int32_t* as_out, int32_t* ae_out,
                          int32_t* abr, int32_t* n_runs, uint8_t* status );

/* ---- 8f4. Adapter trimming (-T): trim_frag (mia.c:1318-1368) for every read of a batch in
 * host memory (call site mia_main.c:773-777; set-up 692-713): dyn_prog of the adapter (rows)
 * against the read (columns) with the flat matrix (init_flatsubmat, pssm.c:96-126), sg5 = 1, the
 * first maximum of the last column, find_align_begin.  Outputs (host arrays of n, nullable):
 * max_score, abr, abc, aer as trim_frag leaves them in the Alignment; trimmed / trim_point =
 * FragSeq.trimmed / trim_point (trim_point 0 when not trimmed).  No homopolymer discount (-h). */
int miagpu_trim( miagpu_ctx* ctx, int64_t n, const uint8_t* bases, const int64_t* offsets,
                 const char* adapter, int adapter_len, int32_t* max_score, int32_t* abr,
                 int32_t* abc, int32_t* aer, uint8_t* trimmed, int32_t* trim_point );

/* ---- 8f1. The repeat filter (-u / -U): sort_fsdb / sort_fsdb_qscore (fsdb.c:13-88, 90-180,
 * 240-252) + set_uniq_in_fsdb (fsdb.c:440-508) at the call sites mia_main.c:827-844, 883-890,
 * 938-945.  Inputs are host arrays of n in FSDB order: FragSeq.rc / as / ae, key4 = FragSeq.score
 * (-u) or FragSeq.qual_sum (-U), trimmed (nullable).  Outputs: order[k] (nullable) = input index of
 * the FragSeq that stands at position k of fsdb->fss after the sort (a stable sort, as glibc's
 * qsort is while its merge buffer fits: equal reads keep their order); unique_best[i] by INPUT
 * index.  Coordinates must lie in [0, 2^21), key4 in [-2^20, 2^20).  Sort and flags run on the
 * device (64-bit keys, LSD radix sort); with tolerance > 0 (-C) the greedy grouping of
 * set_uniq_in_fsdb runs on the host over the device-sorted order. */
int miagpu_repeat_filter( miagpu_ctx* ctx, int64_t n, const uint8_t* rc, const int32_t* as,
                          const int32_t* ae, const int32_t* key4, const uint8_t* trimmed,
                          int just_outer_coords, int tolerance, int64_t* order,
                          uint8_t* unique_best );

/* ---- 8f2. Streaming FASTA / FASTQ record reader: find_input_type (io.c:11-25), read_fastq
 * (io.c:46-167) and read_fasta (io.c:190-281) as mia_main.c:746-759 drives them, over a
 * memory-mapped file, filling batch arrays that go straight into miagpu_upload_reads /
 * miagpu_trim / miagpu_write_maln.  Host only (no device work).  Record rules are the reference's:
 * ids end at the first blank or after 100 characters (the character that ends an over-long id is
 * consumed and starts the description), descriptions are cut at 128, FASTA descriptions repeat
 * their first character (the ungetc at io.c:224), bases are upper-cased and cut at 256 per read,
 * qual_sum = sum(q - 33); the input ends at the first record that does not start with '@' / '>',
 * at a FASTQ record whose quality line differs in length from its sequence, or at end of file.
 *   miagpu_fastx_next  parses up to max_reads records into the handle's batch (replacing the
 *                      previous batch); *n_out = records parsed, 0 at the end of the input.
 *   miagpu_fastx_batch borrows the batch arrays (valid until the next _next / _close):
 *                      bases (ASCII), offsets[n+1], ids / descs as NUL-terminated strings
 *                      back to back with id_off[n+1] / desc_off[n+1], qual_sum[n]. */
typedef struct miagpu_fastx miagpu_fastx;
int  miagpu_fastx_open( miagpu_fastx** out, const char* path );
int  miagpu_fastx_open_memory( miagpu_fastx** out, const void* text, int64_t len );  /* text is borrowed */
int  miagpu_fastx_format( miagpu_fastx* h );            /* 0 FASTA, 1 FASTQ (seq_code, io.c:11-25) */
int  miagpu_fastx_next( miagpu_fastx* h, int64_t max_reads, int64_t* n_out );
int  miagpu_fastx_batch( miagpu_fastx* h, const uint8_t** bases, const int64_t** offsets,
                         const char** ids, const int64_t** id_off, const char** descs,
                         const int64_t** desc_off, const int32_t** qual_sum );
void miagpu_fastx_close( miagpu_fastx* h );

/* ---- 8f3. write_ma (map_alignment.c:283-382) fed from the device's per-read results, at the call
 * sites mia_main.c:905, 958, 974.  The AlnSeq list is rebuilt on the host from the packed run
 * lists: AlnSeq.seq / ins as merge_pwaln_into_maln (map_align.c:866-954) and split_pwaln
 * (mia.c:1376-1438, "_f" / "_b" ids) make them, AlnSeq.smp as pop_smp_from_FSDB (fsdb.c:542-619),
 * list order = FSDB order of the unique_best reads, front before back (cull_maln_from_fsdb
 * mia.c:463-476), then sort_aln_frags by (start, end) (map_alignment.c:630; stable, as glibc's
 * merge-sort qsort).  The file is byte-identical to the reference's after line 1 (its time stamp).
 * Every read owns its fresh AlnSeqs here (the model of miagpu_iterate_resident); the reference's
 * never-cleared back pointers (mia_main.c:273-276) are not reproduced. */
typedef struct {
  const char*    ref_id;      /* maln->ref->id: the input's id in round 1, "ConsAssem.<iter>" later (mia_main.c:47, 62-65) */
  const char*    ref_desc;    /* "iteration assembly" from round 2 on */
  const char*    ref_seq;     /* the reference of THIS round (ref_len characters) */
  int32_t        ref_len;
  int32_t        circular;
  int32_t        ref_size;    /* RefSeq.size; 0 = derive with miagpu_maln_ref_size */
  int32_t        maln_size;   /* culled_maln->size = number of AlnSeqs after pass 1 (mia.c:54) */
  int32_t        cons_code;
  const int32_t* gaps;        /* ref->gaps after the cull (gaps output of miagpu_call / _iterate_*), ref_len entries */
  const int32_t* fpsm;        /* int sm[31][5][5] x 2, as miagpu_get_pssm returns them */
  const int32_t* rpsm;
} miagpu_maln_header;

typedef struct {
  int64_t        n;           /* FragSeqs in FSDB order */
  const uint8_t* bases;       /* STORED orientation (fsdb.c:209-227: rc reads are kept reverse-complemented), ASCII */
  const int64_t* offsets;     /* n+1 */
  const char*    ids;         /* NUL-terminated strings back to back (the layout miagpu_fastx_batch returns) */
  const int64_t* id_off;      /* n+1 */
  const char*    descs;       /* nullable */
  const int64_t* desc_off;
  const uint8_t* rc;
  const uint8_t* trimmed;     /* nullable = 0 */
  const int32_t* num_inputs;  /* nullable = 1 */
  const int32_t* score;       /* outputs of miagpu_realign / miagpu_iterate_*: */
  const int32_t* as;          /*   as_out (absolute)                           */
  const int32_t* ae;          /*   ae_out (absolute, may exceed ref_len)       */
  const int32_t* abr;         /*   first aligned read row (soft clip)          */
  const int64_t* run_off;     /* n+1, miagpu_get_runs_packed                   */
  const uint16_t* packed;
  const uint8_t* unique_best;   /* nullable = all 1 */
  const uint8_t* dropped_front; /* AlnSeq.dropped of the front / only segment; nullable = 0 */
  const uint8_t* dropped_back;  /* nullable = dropped_front */
  const int64_t* fsdb_order;    /* nullable = identity: fsdb_order[k] = index (into the arrays above) of the read at position k of
                                   fsdb->fss, i.e. what sort_fsdb left (-u / -U); the AlnSeq list is built in this order */
} miagpu_maln_reads;

int miagpu_maln_ref_size( int ref_len, int circular );   /* mia_main.c:67 + add_ref_wrap mia.c:669-675 */
int miagpu_write_maln( const char* path, const miagpu_maln_header* hd,
                       const miagpu_maln_reads* rd, int64_t* n_alnseqs_out );

/* The same for the round miagpu_iterate_resident just ran under miagpu_set_fsdb: the list follows the pointers (front_asp, then
 * back_asp of every unique_best read in FSDB order, mia.c:463-476), so an AlnSeq that stale pointers reach is written once per
 * pointer, with the smp codes the last visit of pop_smp_from_FSDB left and the slot's sticky dropped flag; content of slots that
 * are no longer live is written as the earlier round left it.  rd->dropped_front / dropped_back / fsdb_order are not read. */
int miagpu_write_maln_fsdb( miagpu_ctx* ctx, const char* path, const miagpu_maln_header* hd,
                            const miagpu_maln_reads* rd, int64_t* n_alnseqs_out );

/* ---- Damage profile of the last round: the misincorporation table of its culled alignments, computed on the device from the
 * entry list the consensus walked (no `.maln` file needed).  counts[d][r][q], int64 [31][6][6], r (reference) and q (read) over
 * A C G T N - (N = any other character), summed over every AlnSeq of the round's `.maln` with DR 0:
 *   aligned columns  every column c of SEQ with START + c < LEN: d = SMP[c] - 'A', r = the reference's SEQ at START + c,
 *                    q = SEQ[c] ('-': the read has a deletion there)
 *   inserted bases   every base of INS_POS in front of such a column c: r = '-', q = the inserted base, d = SMP[c]
 *   orientation      an AlnSeq with RC 1 has both bases complemented (A<->T, C<->G; N and - stay) and d -> 30 - d, so depth 0
 *                    is always the molecule's 5' end and every cell is the cell of the FORWARD matrix (miagpu_set_pssm) that
 *                    scored the base (revcom_pssm: rev[30-d][i][j] = fwd[d][comp i][comp j]).
 * Records that stale pointers reach and frozen slot content count as the file lists them; dropped AlnSeqs and reads that are not
 * unique_best (-u / -U) count nowhere.  Integer sums: the same for any schedule; the table of a sharded round is the sum of the
 * ranks' tables.  Valid after a call that ends a round with base calling on this context (miagpu_iterate_resident,
 * miagpu_iterate_host, miagpu_consensus, miagpu_consensus_natural, miagpu_shard_finish); a later call that changes the reference,
 * the reads, their strands, their alignments or the entry list (miagpu_set_reference, miagpu_upload_reads, miagpu_compact_reads,
 * miagpu_set_alignment_inputs, the realign / pass-1 / window calls, miagpu_accumulate_gaps*, miagpu_set_fsdb,
 * miagpu_distant_retry*, miagpu_shard_begin*) makes the call fail with a miagpu_last_error that says which.  Changes no state the next round reads. */
#define MIAGPU_MISINC_INTS 1116       /* 31 depths x 6 reference codes x 6 read codes */
int miagpu_misincorporation( miagpu_ctx* ctx, int64_t* counts );

/* ---- measurement helpers (bench.py) */
/* per width bucket of the last realign: columns-per-lane K (0 = too wide),
 * reads, DP cells, kernel ms (CUDA events on the library's stream); MIAGPU_NBUCKET entries */
int miagpu_last_buckets( miagpu_ctx* ctx, int32_t* k, int32_t* reads,
                         int64_t* cells, float* ms );
/* the 16-bit SIMD pair kernels of the last realign (csrc/pair16.cuh): per width class (MIAGPU_NPAIRCLASS entries)
 * columns-per-lane K, reads taken, pairs formed, DP cells of those reads, kernel ms; plus the number
 * of reads the pair kernels handed on to the 32-bit kernels (counted in miagpu_last_buckets as well)
 * and the longest read the 16-bit frame holds with the current matrices (0 = pair kernels off) */
#define MIAGPU_NPAIRCLASS 8
int miagpu_last_pair_buckets( miagpu_ctx* ctx, int32_t* k, int32_t* reads, int32_t* pairs,
                              int64_t* cells, float* ms, int32_t* fallback_reads,
                              int32_t* max_len16 );
/* device time in ms of the kernels launched by the last call, per phase */
int miagpu_last_timing( miagpu_ctx* ctx, float* ms_kernels, float* ms_h2d,
                        float* ms_d2h, int64_t* dp_cells, int32_t* launches );
/* dependent-free INT32 ALU micro-benchmark; returns achieved ops/s (IADD3 /
 * IMNMX / SEL mix) so the roofline can quote a measured integer peak */
int miagpu_int32_peak( miagpu_ctx* ctx, double* ops_per_s );
void* miagpu_stream( miagpu_ctx* ctx );   /* cudaStream_t the library launches on */

#ifdef __cplusplus
}
#endif
#endif
