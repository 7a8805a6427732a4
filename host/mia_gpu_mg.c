/* mia_gpu_mg.c -- the plain-C host of libmiagpu.so for the GPUs of ONE box (SURVEY 8e): one process, one context and one host
 * thread per GPU, reads sharded contiguously in FSDB order, the consensus replicated, three NCCL collectives per round on the
 * library's own streams (the sequence INTEGRATION.md gives, compiled and run):
 *
 *     mia_gpu_mg -g N -r ref.fa -f reads.fq -s matrix.txt -m out [-c] [-k K] [-p 1|2] [-H cut | -S slope -N icpt] [-F] [-d damage.tsv]
 *
 *       miagpu_shard_begin   -> ncclAllReduce( max_buf, MAX )        insert maxima, best scores, the ranks' integer sums
 *       miagpu_shard_fit     -> ncclAllGather( gather_send/recv )    block records of the regression's two chains
 *       miagpu_shard_cut     -> ncclAllReduce( sum_buf, SUM )        column planes
 *       miagpu_shard_finish     every rank calls the same bases
 *
 * It writes the `.maln` files the one-GPU host (host/mia_gpu.c) and the reference write (tests/test_gpu_host_c.py runs both).
 * Sharded rounds give every read its own AlnSeqs and one sticky flag: input that needs the reference's pointer state (a read that
 * scores exactly 2000, -D) is refused here -- host/mia_gpu.c takes it.  -u / -U / -T / -h / -C / -I are not handled.
 * -d FILE is an extension of this host, not a flag of the reference: the damage profile of the final round (miagpu_misincorporation
 * of every GPU's context, summed here) in the text format of host/mia_gpu.c -d.  Without -d every output is what it is without it.
 * No CPU fallback: without CUDA devices miagpu_create fails and so does this program. */
#define _POSIX_C_SOURCE 200809L
#include <ctype.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <cuda_runtime_api.h>
#include <nccl.h>

#include "miagpu.h"

#define FIRST_ROUND_SCORE_CUTOFF 2000   /* params.h */
#define MAX_ITER 30
#define MAX_GPUS 16

static void* xmalloc( size_t n ) {
  void* p = calloc( n ? n : 1, 1 );
  if ( !p ) { fprintf( stderr, "mia_gpu_mg: out of memory\n" ); exit( 1 ); }
  return p;
}
static double now_ms( void ) {
  struct timespec t;
  clock_gettime( CLOCK_MONOTONIC, &t );
  return t.tv_sec * 1e3 + t.tv_nsec * 1e-6;
}

/* first record of a FASTA file (read_fasta_ref io.c:288-386), case kept */
static char* read_reference( const char* fn, char* id, char* desc, int* len_out ) {
  FILE* f = fopen( fn, "r" );
  size_t cap = 1 << 16, n = 0;
  char* seq = (char*)xmalloc( cap );
  int c, k = 0;
  if ( !f || fgetc( f ) != '>' ) { fprintf( stderr, "mia_gpu_mg: cannot read reference %s\n", fn ); exit( 1 ); }
  while ( ( c = fgetc( f ) ) != EOF && !isspace( c ) && k < 100 ) id[k++] = (char)c;
  id[k] = 0;
  k = 0;
  if ( c != '\n' && c != EOF )
    while ( ( c = fgetc( f ) ) != EOF && c != '\n' && k < 128 ) desc[k++] = (char)c;
  desc[k] = 0;
  while ( c != '\n' && c != EOF ) c = fgetc( f );
  while ( ( c = fgetc( f ) ) != EOF && c != '>' ) {
    if ( isspace( c ) ) continue;
    if ( n + 2 > cap ) { cap *= 2; seq = (char*)realloc( seq, cap ); if ( !seq ) exit( 1 ); }
    seq[n++] = (char)c;
  }
  seq[n] = 0;
  fclose( f );
  *len_out = (int)n;
  return seq;
}

/* ---- what all threads share */
typedef struct {
  int world, circular, k, cons_code, hard_cut, score_cut_set, final_only, hp_special;
  double user_slope, user_icpt;
  const char *root, *ref_id, *ref_desc;
  char* ref; int ref_len;
  int32_t fwd[MIAGPU_PSSM_INTS], fpsm[MIAGPU_PSSM_INTS], rpsm[MIAGPU_PSSM_INTS];
  /* the input, in input order */
  int64_t n;
  const uint8_t* bases; const int64_t *off, *id_off, *desc_off; const char *ids, *descs;
  int64_t in_lo[MAX_GPUS + 1];                 /* input reads of rank r: [in_lo[r], in_lo[r + 1]) */
  int32_t *hits, *score, *as, *ae, *start, *end; uint8_t *rc, *keep;
  /* the FSDB (accepted reads, input order) */
  int64_t m, fs_lo[MAX_GPUS + 1], n_max;
  int64_t* src;
  int32_t *f_len, *f_score, *f_as, *f_ae, *f_abr; uint8_t *f_rc, *f_dropped, *f_status;
  int64_t *s_off, *f_id_off, *f_desc_off;
  uint8_t* stored; char *f_ids, *f_descs;
  int32_t maln_size;
  /* per round */
  char *last, *cons; int32_t* gaps; size_t cons_cap;
  int64_t run_total[MAX_GPUS]; int64_t *run_off, *run_off_r[MAX_GPUS]; uint16_t* packed[MAX_GPUS]; int64_t packed_cap[MAX_GPUS];
  int iter, converged, failed;
  const char* damage_fn;
  int64_t damage[MAX_GPUS][MIAGPU_MISINC_INTS];  /* -d: the final round's table of every rank */
  ncclComm_t comm[MAX_GPUS];
  pthread_barrier_t bar;
  double t_rounds, t_write;
} Shared;

typedef struct { Shared* S; int rank; } Arg;

static unsigned char comp[256];
static void init_comp( void ) {
  const char* a = "ACGTRYKMBDHVNSWacgtrykmbdhvnsw-";
  const char* b = "TGCAYRMKVHDBNSWtgcayrmkvhdbnsw-";
  int i;
  for ( i = 0; i < 256; i++ ) comp[i] = 'N';
  for ( i = 0; a[i]; i++ ) comp[(unsigned char)a[i]] = (unsigned char)b[i];
}

/* -d: the table of miagpu_misincorporation as text (the format of host/mia_gpu.c) */
static int write_damage( const char* fn, const int64_t* t ) {
  static const char code[] = "ACGTN-";
  FILE* f = fopen( fn, "w" );
  int c;
  if ( !f ) return 0;
  fprintf( f, "depth\tref\tread\tcount\n" );
  for ( c = 0; c < MIAGPU_MISINC_INTS; c++ ) fprintf( f, "%d\t%c\t%c\t%lld\n", c / 36, code[c / 6 % 6], code[c % 6], (long long)t[c] );
  return fclose( f ) == 0;
}

#define FAIL( S, ... ) do { fprintf( stderr, "mia_gpu_mg: " __VA_ARGS__ ); (S)->failed = 1; } while ( 0 )
#define CK( S, call ) do { if ( !(S)->failed && !( call ) ) { fprintf( stderr, "mia_gpu_mg: rank %d: %s: %s\n", rank, #call, miagpu_last_error() ); (S)->failed = 1; } } while ( 0 )
#define NC( S, call ) do { if ( !(S)->failed ) { ncclResult_t r_ = ( call ); if ( r_ != ncclSuccess ) { fprintf( stderr, "mia_gpu_mg: rank %d: %s: %s\n", rank, #call, ncclGetErrorString( r_ ) ); (S)->failed = 1; } } } while ( 0 )
/* every thread leaves together: a failure anywhere is seen by all after the next barrier */
#define SYNC( S ) do { pthread_barrier_wait( &(S)->bar ); if ( (S)->failed ) return NULL; } while ( 0 )

static void* worker( void* arg_ ) {
  Arg* A = (Arg*)arg_;
  Shared* S = A->S;
  const int rank = A->rank, world = S->world;
  miagpu_ctx* g = NULL;
  int64_t j;
  CK( S, miagpu_create( &g, rank ) );
  CK( S, miagpu_set_homopolymer( g, S->hp_special ) );
  CK( S, miagpu_set_cons_capacity( g, (int64_t)S->cons_cap ) );      /* what the cons buffers of this program hold */
  CK( S, miagpu_set_pssm( g, S->fwd ) );
  CK( S, miagpu_set_reference( g, S->ref, S->ref_len, S->circular, 1 ) );
  CK( S, miagpu_build_kmers( g, S->k, 0 ) );
  SYNC( S );
  cudaStream_t st = (cudaStream_t)miagpu_stream( g );
  /* ---- pass 1 over this rank's share of the input (mia_main.c:746-805) */
  const int64_t lo = S->in_lo[rank], hi = S->in_lo[rank + 1], nl = hi - lo;
  {
    int64_t* loff = xmalloc( ( nl + 1 ) * 8 );
    for ( j = 0; j <= nl; j++ ) loff[j] = S->off[lo + j] - S->off[lo];
    CK( S, miagpu_upload_reads( g, nl, S->bases + S->off[lo], loff ) );
    CK( S, miagpu_pass1( g, S->hits + lo, S->score + lo, NULL, NULL, S->rc + lo, S->as + lo, S->ae + lo, S->start + lo, S->end + lo, NULL, NULL,
                         NULL, NULL ) );
    free( loff );
  }
  SYNC( S );
  /* ---- rank 0: sg_align's accept test (mia.c:1614), the FSDB, the pass-1 cull with the fit over ALL reads (mia_main.c:848) */
  if ( rank == 0 ) {
    int64_t m = 0, r;
    double slope = 0, icpt = 0;
    for ( j = 0; j < S->n; j++ ) {
      S->keep[j] = ( S->hits[j] > 0 && S->score[j] >= FIRST_ROUND_SCORE_CUTOFF );
      if ( S->keep[j] && S->score[j] == FIRST_ROUND_SCORE_CUTOFF ) {
        FAIL( S, "a read scores exactly 2000 (strand_known = 0, mia.c:1653): the pointer state it needs is a one-GPU feature (host/mia_gpu)\n" );
        break;
      }
      if ( S->keep[j] ) { S->maln_size += 1 + ( S->start[j] > S->end[j] ); m++; }
    }
    S->m = m;
    S->src = xmalloc( m * 8 );
    S->f_len = xmalloc( m * 4 ); S->f_score = xmalloc( m * 4 ); S->f_as = xmalloc( m * 4 ); S->f_ae = xmalloc( m * 4 ); S->f_abr = xmalloc( m * 4 );
    S->f_rc = xmalloc( m ); S->f_dropped = xmalloc( m ); S->f_status = xmalloc( m );
    S->s_off = xmalloc( ( m + 1 ) * 8 ); S->f_id_off = xmalloc( ( m + 1 ) * 8 ); S->f_desc_off = xmalloc( ( m + 1 ) * 8 ); S->run_off = xmalloc( ( m + 1 ) * 8 );
    for ( j = 0, m = 0, r = 0; j < S->n; j++ ) {
      while ( r < world && j >= S->in_lo[r] ) S->fs_lo[r++] = m;
      if ( !S->keep[j] ) continue;
      S->src[m] = j;
      S->f_len[m] = (int32_t)( S->off[j + 1] - S->off[j] ); S->f_score[m] = S->score[j]; S->f_as[m] = S->as[j]; S->f_ae[m] = S->ae[j]; S->f_rc[m] = S->rc[j];
      S->s_off[m + 1] = S->s_off[m] + S->f_len[m];
      S->f_id_off[m + 1] = S->f_id_off[m] + ( S->id_off[j + 1] - S->id_off[j] );
      S->f_desc_off[m + 1] = S->f_desc_off[m] + ( S->desc_off[j + 1] - S->desc_off[j] );
      m++;
    }
    while ( r <= world ) S->fs_lo[r++] = m;
    S->stored = xmalloc( (size_t)S->s_off[m] + 1 );
    S->f_ids = xmalloc( (size_t)S->f_id_off[m] + 1 ); S->f_descs = xmalloc( (size_t)S->f_desc_off[m] + 1 );
    for ( j = 0; j < m; j++ ) {                                     /* stored orientation (fsdb.c:209-227), ids, descriptions */
      int64_t q = S->src[j], L = S->f_len[j], t;
      if ( !S->f_rc[j] ) memcpy( S->stored + S->s_off[j], S->bases + S->off[q], (size_t)L );
      else for ( t = 0; t < L; t++ ) S->stored[S->s_off[j] + t] = comp[S->bases[S->off[q] + L - 1 - t]];
      memcpy( S->f_ids + S->f_id_off[j], S->ids + S->id_off[q], (size_t)( S->id_off[q + 1] - S->id_off[q] ) );
      memcpy( S->f_descs + S->f_desc_off[j], S->descs + S->desc_off[q], (size_t)( S->desc_off[q + 1] - S->desc_off[q] ) );
    }
    if ( !S->failed && m == 0 ) FAIL( S, "no read aligned in pass 1\n" );
    if ( !S->failed ) {
      if ( S->hard_cut > 0 || S->score_cut_set ) {
        if ( !miagpu_cull_flags( m, S->f_len, S->f_score, NULL, S->hard_cut, S->score_cut_set, S->user_slope, S->user_icpt, S->f_dropped ) ) FAIL( S, "%s\n", miagpu_last_error() );
      }
      else if ( !miagpu_score_cut( m, S->f_len, S->f_score, NULL, &slope, &icpt ) ||
                !miagpu_cull_flags( m, S->f_len, S->f_score, NULL, 0, 1, slope, icpt, S->f_dropped ) ) FAIL( S, "%s\n", miagpu_last_error() );
    }
    S->n_max = 1;
    for ( r = 0; r < world; r++ ) if ( S->fs_lo[r + 1] - S->fs_lo[r] > S->n_max ) S->n_max = S->fs_lo[r + 1] - S->fs_lo[r];
    fprintf( stderr, "mia_gpu_mg: %lld reads read, %lld aligned in pass 1, %d GPUs\n", (long long)S->n, (long long)m, world );
  }
  SYNC( S );
  /* ---- this rank's part of the FSDB stays resident */
  const int64_t flo = S->fs_lo[rank], fhi = S->fs_lo[rank + 1], ml = fhi - flo;
  {
    int64_t kept = 0;
    CK( S, miagpu_compact_reads( g, S->keep + lo, S->rc + lo, &kept ) );
    if ( !S->failed && kept != ml ) FAIL( S, "rank %d: compact_reads kept %lld of %lld\n", rank, (long long)kept, (long long)ml );
    CK( S, miagpu_set_alignment_inputs( g, S->f_rc + flo, S->f_as + flo, S->f_ae + flo ) );
    CK( S, miagpu_set_cut_inputs( g, S->f_len + flo, NULL, S->f_dropped + flo ) );
  }
  SYNC( S );
  /* ---- rounds (mia_main.c:878-976) */
  char* cons = xmalloc( S->cons_cap );
  int32_t* gaps = xmalloc( S->cons_cap * 4 );
  for ( ;; ) {
    int32_t cons_len = 0, L = (int32_t)strlen( S->last );
    double t1 = now_ms(), slope = 0, icpt = 0;
    void *mb = NULL, *gs = NULL, *gr = NULL, *sb = NULL;
    int64_t mw = 0, gw = 0, sw = 0;
    CK( S, miagpu_set_reference( g, S->last, L, S->circular, 0 ) );
    CK( S, miagpu_shard_begin( g, world, rank, S->n_max, S->hard_cut, S->score_cut_set, S->user_slope, S->user_icpt, &mb, &mw ) );
    SYNC( S );                                                      /* a rank that failed must not leave the others inside a collective */
    NC( S, ncclAllReduce( mb, mb, (size_t)mw, ncclInt32, ncclMax, S->comm[rank], st ) );
    CK( S, miagpu_shard_fit( g, &gs, &gr, &gw ) );
    SYNC( S );
    if ( gw ) NC( S, ncclAllGather( gs, gr, (size_t)gw, ncclUint32, S->comm[rank], st ) );
    CK( S, miagpu_shard_cut( g, &slope, &icpt, &sb, &sw ) );
    SYNC( S );
    NC( S, ncclAllReduce( sb, sb, (size_t)sw, ncclInt32, ncclSum, S->comm[rank], st ) );
    CK( S, miagpu_shard_finish( g, S->cons_code, S->f_dropped + flo, NULL, 0, NULL, gaps, cons, &cons_len ) );
    CK( S, miagpu_adopt_alignment( g, S->f_score + flo, S->f_as + flo, S->f_ae + flo ) );
    cons[cons_len] = 0;
    if ( rank == 0 ) {
      S->iter++;
      memcpy( S->cons, cons, (size_t)cons_len + 1 );
      memcpy( S->gaps, gaps, (size_t)L * 4 );
      S->converged = !strcmp( cons, S->last );
      S->t_rounds += now_ms() - t1;
    }
    SYNC( S );
    if ( !S->final_only || S->converged || S->iter == MAX_ITER ) {   /* every rank hands its alignments to rank 0, which writes */
      int64_t total = 0;
      CK( S, miagpu_get_alignment( g, NULL, NULL, NULL, S->f_abr + flo, NULL, S->f_status + flo ) );
      CK( S, miagpu_get_runs_packed( g, NULL, NULL, 0, &total ) );
      if ( total > S->packed_cap[rank] ) { free( S->packed[rank] ); S->packed_cap[rank] = total + total / 4 + 16; S->packed[rank] = xmalloc( (size_t)S->packed_cap[rank] * 2 ); }
      if ( !S->run_off_r[rank] ) S->run_off_r[rank] = xmalloc( ( ml + 1 ) * 8 );
      CK( S, miagpu_get_runs_packed( g, S->run_off_r[rank], S->packed[rank], S->packed_cap[rank], &total ) );
      S->run_total[rank] = total;
      SYNC( S );
      if ( rank == 0 ) {
        double t2 = now_ms();
        int64_t all = 0, base = 0, n_aln = 0, r;
        uint16_t* packed;
        char fn[4096], iter_id[64];
        miagpu_maln_header hd;
        miagpu_maln_reads rd;
        for ( j = 0; j < S->m; j++ )
          if ( S->f_status[j] != MIAGPU_ST_OK ) { FAIL( S, "read %lld came back with status 0x%x in iteration %d\n", (long long)S->src[j], S->f_status[j], S->iter ); break; }
        for ( r = 0; r < world; r++ ) all += S->run_total[r];
        packed = xmalloc( (size_t)all * 2 + 2 );
        for ( r = 0; r < world; r++ ) {                             /* the ranks' packed run lists back to back, offsets rebased */
          memcpy( packed + base, S->packed[r], (size_t)S->run_total[r] * 2 );
          for ( j = S->fs_lo[r]; j < S->fs_lo[r + 1]; j++ ) S->run_off[j] = S->run_off_r[r][j - S->fs_lo[r]] + base;
          base += S->run_total[r];
        }
        S->run_off[S->m] = base;
        memset( &hd, 0, sizeof hd );
        memset( &rd, 0, sizeof rd );
        snprintf( iter_id, sizeof iter_id, "ConsAssem.%d", S->iter );
        hd.ref_id = S->iter > 1 ? iter_id : S->ref_id;               /* mia_main.c:47, 62-65 */
        hd.ref_desc = S->iter > 1 ? "iteration assembly" : S->ref_desc;
        hd.ref_seq = S->last; hd.ref_len = L; hd.circular = S->circular; hd.maln_size = S->maln_size; hd.cons_code = S->cons_code;
        hd.gaps = S->gaps; hd.fpsm = S->fpsm; hd.rpsm = S->rpsm;
        rd.n = S->m; rd.bases = S->stored; rd.offsets = S->s_off; rd.ids = S->f_ids; rd.id_off = S->f_id_off; rd.descs = S->f_descs;
        rd.desc_off = S->f_desc_off; rd.rc = S->f_rc; rd.score = S->f_score; rd.as = S->f_as; rd.ae = S->f_ae; rd.abr = S->f_abr;
        rd.run_off = S->run_off; rd.packed = packed; rd.dropped_front = S->f_dropped; rd.dropped_back = S->f_dropped;
        snprintf( fn, sizeof fn, "%s.%d", S->root, S->iter );
        if ( !S->failed && !miagpu_write_maln( fn, &hd, &rd, &n_aln ) ) FAIL( S, "%s\n", miagpu_last_error() );
        if ( !S->failed ) fprintf( stderr, "mia_gpu_mg: iteration %d: %lld AlnSeqs -> %s\n", S->iter, (long long)n_aln, fn );
        free( packed );
        S->t_write += now_ms() - t2;
      }
    }
    if ( rank == 0 ) { char* t = S->last; S->last = S->cons; S->cons = t; }
    SYNC( S );
    if ( S->converged || S->iter >= MAX_ITER ) break;
  }
  if ( S->damage_fn ) {                                             /* the contexts still hold the final round: the ranks' tables, summed */
    CK( S, miagpu_misincorporation( g, S->damage[rank] ) );
    SYNC( S );
    if ( rank == 0 ) {
      int r, c;
      for ( r = 1; r < world; r++ )
        for ( c = 0; c < MIAGPU_MISINC_INTS; c++ ) S->damage[0][c] += S->damage[r][c];
      if ( !write_damage( S->damage_fn, S->damage[0] ) ) FAIL( S, "cannot write %s\n", S->damage_fn );
    }
  }
  miagpu_destroy( g );
  return NULL;
}

int main( int argc, char** argv ) {
  static Shared S;
  const char *ref_fn = NULL, *frag_fn = NULL, *mat_fn = NULL;
  static char ref_id[128], ref_desc[160];
  int i, ngpu = 0, devs[MAX_GPUS];
  double t0 = now_ms();
  S.root = "assembly.maln.iter"; S.k = -1; S.cons_code = 1; S.user_slope = 200.0; S.user_icpt = 0.0;
  for ( i = 1; i < argc; i++ ) {
    if ( !strcmp( argv[i], "-c" ) ) S.circular = 1;
    else if ( !strcmp( argv[i], "-F" ) ) S.final_only = 1;
    else if ( !strcmp( argv[i], "-h" ) ) S.hp_special = 1;
    else if ( !strcmp( argv[i], "-i" ) ) ;
    else if ( !strcmp( argv[i], "-d" ) ) {
      if ( i + 1 >= argc ) { fprintf( stderr, "mia_gpu_mg: -d needs a file name (the damage profile of the final round)\n" ); return 2; }
      S.damage_fn = argv[++i];
    }
    else if ( i + 1 < argc && !strcmp( argv[i], "-g" ) ) ngpu = atoi( argv[++i] );
    else if ( i + 1 < argc && !strcmp( argv[i], "-r" ) ) ref_fn = argv[++i];
    else if ( i + 1 < argc && !strcmp( argv[i], "-f" ) ) frag_fn = argv[++i];
    else if ( i + 1 < argc && !strcmp( argv[i], "-s" ) ) mat_fn = argv[++i];
    else if ( i + 1 < argc && !strcmp( argv[i], "-m" ) ) S.root = argv[++i];
    else if ( i + 1 < argc && !strcmp( argv[i], "-k" ) ) S.k = atoi( argv[++i] );
    else if ( i + 1 < argc && !strcmp( argv[i], "-p" ) ) S.cons_code = atoi( argv[++i] );
    else if ( i + 1 < argc && !strcmp( argv[i], "-H" ) ) S.hard_cut = atoi( argv[++i] );
    else if ( i + 1 < argc && !strcmp( argv[i], "-S" ) ) { S.user_slope = atof( argv[++i] ); S.score_cut_set = 1; }
    else if ( i + 1 < argc && !strcmp( argv[i], "-N" ) ) { S.user_icpt = atof( argv[++i] ); S.score_cut_set = 1; }
    else { fprintf( stderr, "mia_gpu_mg: option %s is not handled by this host (see the header of host/mia_gpu_mg.c)\n", argv[i] ); return 2; }
  }
  if ( !ref_fn || !frag_fn || !mat_fn ) {
    fprintf( stderr, "usage: mia_gpu_mg -g N -r ref.fa -f reads.fa|fq -s matrix.txt [-m root] [-c] [-k K] [-p code] [-H cut | -S slope -N icpt] [-F]\n"
                     "                  [-d damage.tsv  (extension of this host: the final round's misincorporation table)]\n" );
    return 2;
  }
  init_comp();
  S.ref = read_reference( ref_fn, ref_id, ref_desc, &S.ref_len );
  S.ref_id = ref_id; S.ref_desc = ref_desc;
  if ( !miagpu_read_pssm( mat_fn, S.fwd ) ) { fprintf( stderr, "mia_gpu_mg: miagpu_read_pssm: %s\n", miagpu_last_error() ); return 1; }
  if ( ngpu <= 0 ) ngpu = miagpu_device_count();
  if ( ngpu < 1 || ngpu > MAX_GPUS || ngpu > miagpu_device_count() ) {
    fprintf( stderr, "mia_gpu_mg: %d GPUs asked for, %d CUDA devices here; this program has no CPU fallback\n", ngpu, miagpu_device_count() );
    return 1;
  }
  S.world = ngpu;
  { /* the strand-reversed copy of the matrices for the .maln header */
    miagpu_ctx* g0;
    if ( !miagpu_create( &g0, 0 ) || !miagpu_set_pssm( g0, S.fwd ) || !miagpu_get_pssm( g0, S.fpsm, S.rpsm ) ) { fprintf( stderr, "mia_gpu_mg: %s\n", miagpu_last_error() ); return 1; }
    miagpu_destroy( g0 );
  }
  /* ---- the whole input, one batch (mia_main.c:746-759), shared by the ranks */
  miagpu_fastx* fx;
  const int32_t* qual_sum;
  if ( !miagpu_fastx_open( &fx, frag_fn ) || !miagpu_fastx_next( fx, (int64_t)1 << 40, &S.n ) ||
       !miagpu_fastx_batch( fx, &S.bases, &S.off, &S.ids, &S.id_off, &S.descs, &S.desc_off, &qual_sum ) ) { fprintf( stderr, "mia_gpu_mg: %s\n", miagpu_last_error() ); return 1; }
  if ( S.n < 1 ) { fprintf( stderr, "mia_gpu_mg: no reads in %s\n", frag_fn ); return 1; }
  for ( i = 0; i <= ngpu; i++ ) S.in_lo[i] = S.n * i / ngpu;
  S.hits = xmalloc( S.n * 4 ); S.score = xmalloc( S.n * 4 ); S.as = xmalloc( S.n * 4 ); S.ae = xmalloc( S.n * 4 ); S.start = xmalloc( S.n * 4 );
  S.end = xmalloc( S.n * 4 ); S.rc = xmalloc( S.n ); S.keep = xmalloc( S.n );
  S.cons_cap = (size_t)S.ref_len * 4 + 65536;
  S.last = xmalloc( S.cons_cap ); S.cons = xmalloc( S.cons_cap ); S.gaps = xmalloc( S.cons_cap * 4 );
  for ( i = 0; i < S.ref_len; i++ ) S.last[i] = (char)toupper( (unsigned char)S.ref[i] );      /* make_ref_upper mia.c:642-648 */
  for ( i = 0; i < ngpu; i++ ) devs[i] = i;
  { ncclResult_t r = ncclCommInitAll( S.comm, ngpu, devs );
    if ( r != ncclSuccess ) { fprintf( stderr, "mia_gpu_mg: ncclCommInitAll: %s\n", ncclGetErrorString( r ) ); return 1; } }
  pthread_barrier_init( &S.bar, NULL, (unsigned)ngpu );
  pthread_t th[MAX_GPUS];
  Arg args[MAX_GPUS];
  for ( i = 0; i < ngpu; i++ ) { args[i].S = &S; args[i].rank = i; pthread_create( &th[i], NULL, worker, &args[i] ); }
  for ( i = 0; i < ngpu; i++ ) pthread_join( th[i], NULL );
  if ( S.failed ) return 3;
  for ( i = 0; i < ngpu; i++ ) ncclCommDestroy( S.comm[i] );
  miagpu_fastx_close( fx );
  fprintf( stderr, S.converged ? "Assembly convergence after %d rounds\n" : "Assembly did not converge after %d rounds, quitting\n", S.iter );
  fprintf( stderr, "mia_gpu_mg: timing ms: rounds %.1f write %.1f total %.1f\n", S.t_rounds, S.t_write, now_ms() - t0 );
  return 0;
}
