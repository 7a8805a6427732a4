/* mia_gpu.c -- a plain-C host for libmiagpu.so: the call sequence INTEGRATION.md gives a maintainer of the reference,
 * compiled and run.  It is NOT the reference's CLI (SURVEY 8: out of scope): it covers the default assembly mode only
 *
 *     mia_gpu -r ref.fa -f reads.fq -s matrix.txt -m out [-c] [-k K] [-p 1|2] [-H cut | -S slope -N icpt] [-F] [-u | -U] [-A] [-D] [-h]
 *             [-d damage.tsv]
 *
 * and exists to show (and test, tests/test_gpu_host_c.py) that the C ABI alone -- no Python, no torch -- reproduces
 * the reference's `.maln` files: reader (miagpu_fastx_*), matrices (miagpu_read_pssm), pass 1, score cut, one library
 * call per round with everything resident, writer (miagpu_write_maln).  The host keeps what mia_main.c keeps: which
 * reads enter the FSDB (mia.c:1614), their strand, the convergence test (mia_main.c:909-976), the file names.
 * -u / -U (the repeat filter, mia_main.c:827-844, 883-890, 938-945) run the per-phase calls instead of the one-call round, with
 * the FSDB order and the slot-indexed sticky AlnSeq.dropped flags kept here as mia_main.c keeps them.
 * The one-call rounds follow the reference's FragSeq -> AlnSeq pointers on the device (miagpu_set_fsdb): reads that score exactly
 * 2000 (strand_known = 0, mia.c:1653), never-cleared back pointers, slot-indexed sticky flags, and -D (mia.c:1614,
 * mia_main.c:120-174: miagpu_distant_retry).  -h (mia_main.c:497: the homopolymer discount in every alignment) is
 * miagpu_set_homopolymer.  -T, -C, -I are not handled here.
 * -d FILE is an extension of this host, not a flag of the reference: the damage profile of the final round (miagpu_misincorporation,
 * the misincorporation table of its `.maln` file by depth) as text, a header line depth / ref / read / count, then one line per cell
 * of the [31][6][6] table in index order, bases as A C G T N -.  Without -d every output is what it is without the extension.
 * There is no CPU fallback: without a CUDA device miagpu_create fails and so does this program. */
#define _POSIX_C_SOURCE 199309L
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <ctype.h>
#include <time.h>
#include "miagpu.h"

#define FIRST_ROUND_SCORE_CUTOFF 2000   /* params.h */
#define MAX_ITER 30

static void die( const char* what ) {
  fprintf( stderr, "mia_gpu: %s: %s\n", what, miagpu_last_error() );
  exit( 1 );
}
#define CK( call ) do { if ( !( call ) ) die( #call ); } while ( 0 )

static double now_ms( void ) {
  struct timespec t;
  clock_gettime( CLOCK_MONOTONIC, &t );
  return t.tv_sec * 1e3 + t.tv_nsec * 1e-6;
}

static void* xmalloc( size_t n ) {
  void* p = calloc( n ? n : 1, 1 );
  if ( !p ) { fprintf( stderr, "mia_gpu: out of memory\n" ); exit( 1 ); }
  return p;
}

/* first record of a FASTA file: id = up to the first blank, desc = rest of the line after ONE blank, sequence with
 * white space removed, case kept (read_fasta_ref io.c:288-386; the -M soft mask needs the case) */
static char* read_reference( const char* fn, char* id, char* desc, int* len_out ) {
  FILE* f = fopen( fn, "r" );
  size_t cap = 1 << 16, n = 0;
  char* seq = (char*)xmalloc( cap );
  int c, k = 0;
  if ( !f || fgetc( f ) != '>' ) { fprintf( stderr, "mia_gpu: cannot read reference %s\n", fn ); exit( 1 ); }
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

/* -d: the table of miagpu_misincorporation as text */
static void write_damage( const char* fn, const int64_t* t ) {
  static const char code[] = "ACGTN-";
  FILE* f = fopen( fn, "w" );
  int c;
  if ( !f ) { fprintf( stderr, "mia_gpu: cannot write %s\n", fn ); exit( 1 ); }
  fprintf( f, "depth\tref\tread\tcount\n" );
  for ( c = 0; c < MIAGPU_MISINC_INTS; c++ ) fprintf( f, "%d\t%c\t%c\t%lld\n", c / 36, code[c / 6 % 6], code[c % 6], (long long)t[c] );
  if ( fclose( f ) != 0 ) { fprintf( stderr, "mia_gpu: cannot write %s\n", fn ); exit( 1 ); }
}

static unsigned char comp[256];
static void init_comp( void ) {
  const char* a = "ACGTRYKMBDHVNSWacgtrykmbdhvnsw-";
  const char* b = "TGCAYRMKVHDBNSWtgcayrmkvhdbnsw-";
  int i;
  for ( i = 0; i < 256; i++ ) comp[i] = 'N';
  for ( i = 0; a[i]; i++ ) comp[(unsigned char)a[i]] = (unsigned char)b[i];
}

/* ---- -u / -U: sort_fsdb[_qscore] + set_uniq_in_fsdb + cull_maln_from_fsdb over the current FSDB (mia_main.c:827-848, 883-891).
 * Arrays are indexed by read (device order); order[k] = read at position k of fsdb->fss. */
typedef struct {
  int64_t m;
  int joc, by_qual;
  int32_t *len, *score, *as, *ae, *qual;
  uint8_t *rc, *split, *unique, *df, *db, *slot;      /* slot: AlnSeq.dropped per maln slot, sticky (H10) */
  int64_t *order, slot_cap;
} Fsdb;

static void filter_and_cull( miagpu_ctx* g, Fsdb* F ) {
  int64_t m = F->m, k, s = 0;
  uint8_t *rc = xmalloc( m ), *uq = xmalloc( m ), *below = xmalloc( m ), *uo = xmalloc( m );
  int32_t *as = xmalloc( m * 4 ), *ae = xmalloc( m * 4 ), *k4 = xmalloc( m * 4 ), *lo = xmalloc( m * 4 ), *so = xmalloc( m * 4 );
  int64_t *ord = xmalloc( m * 8 ), *first = xmalloc( m * 8 ), *neworder = xmalloc( m * 8 );
  double slope = 0, icpt = 0;
  for ( k = 0; k < m; k++ ) {
    int64_t j = F->order[k];
    rc[k] = F->rc[j]; as[k] = F->as[j]; ae[k] = F->ae[j]; k4[k] = F->by_qual ? F->qual[j] : F->score[j];
    first[j] = s; s += 1 + F->split[j];               /* slots were numbered in the order the merges ran in: BEFORE this sort */
  }
  CK( miagpu_repeat_filter( g, m, rc, as, ae, k4, NULL, F->joc, 0, ord, uq ) );
  for ( k = 0; k < m; k++ ) F->unique[F->order[k]] = uq[k];
  for ( k = 0; k < m; k++ ) neworder[k] = F->order[ord[k]];
  memcpy( F->order, neworder, (size_t)m * 8 );
  for ( k = 0; k < m; k++ ) { int64_t j = F->order[k]; lo[k] = F->len[j]; so[k] = F->score[j]; uo[k] = F->unique[j]; }
  CK( miagpu_score_cut( m, lo, so, uo, &slope, &icpt ) );                /* sums run in FSDB order */
  CK( miagpu_cull_flags( m, F->len, F->score, NULL, 0, 1, slope, icpt, below ) );
  if ( s + 2 > F->slot_cap ) {
    F->slot = realloc( F->slot, (size_t)s + 66 );
    memset( F->slot + F->slot_cap, 0, (size_t)( s + 66 - F->slot_cap ) );
    F->slot_cap = s + 66;
  }
  for ( k = 0; k < m; k++ )
    if ( below[k] && F->unique[k] ) { F->slot[first[k]] = 1; if ( F->split[k] ) F->slot[first[k] + 1] = 1; }
  for ( k = 0; k < m; k++ ) {
    int64_t b = first[k] + 1 < F->slot_cap ? first[k] + 1 : F->slot_cap - 1;
    F->df[k] = F->unique[k] ? F->slot[first[k]] : 2;
    F->db[k] = F->unique[k] ? F->slot[b] : 2;
  }
  free( rc ); free( uq ); free( below ); free( uo ); free( as ); free( ae ); free( k4 ); free( lo ); free( so ); free( ord ); free( first );
  free( neworder );
}

int main( int argc, char** argv ) {
  const char *ref_fn = NULL, *frag_fn = NULL, *mat_fn = NULL, *root = "assembly.maln.iter", *damage_fn = NULL;
  int circular = 0, k = -1, cons_code = 1, hard_cut = 0, final_only = 0, repeat_filt = 0, just_outer_coords = 1, i;
  int score_cut_set = 0, distant_ref = 0, n_unknown = 0, hp_special = 0;
  double user_slope = 200.0, user_icpt = 0.0;           /* DEF_S, DEF_N (params.h:36-37); -S / -N: mia_main.c:579-586 */
  for ( i = 1; i < argc; i++ ) {
    if ( !strcmp( argv[i], "-c" ) ) circular = 1;
    else if ( !strcmp( argv[i], "-F" ) ) final_only = 1;
    else if ( !strcmp( argv[i], "-u" ) ) repeat_filt = 1;
    else if ( !strcmp( argv[i], "-U" ) ) repeat_filt = 2;
    else if ( !strcmp( argv[i], "-A" ) ) just_outer_coords = 0;
    else if ( !strcmp( argv[i], "-D" ) ) distant_ref = 1;
    else if ( !strcmp( argv[i], "-h" ) ) hp_special = 1;
    else if ( !strcmp( argv[i], "-i" ) ) ;
    else if ( i + 1 < argc && !strcmp( argv[i], "-r" ) ) ref_fn = argv[++i];
    else if ( i + 1 < argc && !strcmp( argv[i], "-f" ) ) frag_fn = argv[++i];
    else if ( i + 1 < argc && !strcmp( argv[i], "-s" ) ) mat_fn = argv[++i];
    else if ( i + 1 < argc && !strcmp( argv[i], "-m" ) ) root = argv[++i];
    else if ( !strcmp( argv[i], "-d" ) ) {
      if ( i + 1 >= argc ) { fprintf( stderr, "mia_gpu: -d needs a file name (the damage profile of the final round)\n" ); return 2; }
      damage_fn = argv[++i];
    }
    else if ( i + 1 < argc && !strcmp( argv[i], "-k" ) ) k = atoi( argv[++i] );
    else if ( i + 1 < argc && !strcmp( argv[i], "-p" ) ) cons_code = atoi( argv[++i] );
    else if ( i + 1 < argc && !strcmp( argv[i], "-H" ) ) hard_cut = atoi( argv[++i] );
    else if ( i + 1 < argc && !strcmp( argv[i], "-S" ) ) { user_slope = atof( argv[++i] ); score_cut_set = 1; }
    else if ( i + 1 < argc && !strcmp( argv[i], "-N" ) ) { user_icpt = atof( argv[++i] ); score_cut_set = 1; }
    else { fprintf( stderr, "mia_gpu: option %s is not handled by this host (see the header of host/mia_gpu.c)\n", argv[i] ); return 2; }
  }
  if ( repeat_filt && ( hard_cut > 0 || score_cut_set || distant_ref ) ) { fprintf( stderr, "mia_gpu: -H / -S / -N / -D together with -u / -U are not handled by this host\n" ); return 2; }
  if ( !ref_fn || !frag_fn || !mat_fn ) {
    fprintf( stderr, "usage: mia_gpu -r ref.fa -f reads.fa|fq -s matrix.txt [-m root] [-c] [-k K] [-p code] [-H cut] [-F] [-u|-U] [-A]\n"
                     "               [-d damage.tsv  (extension of this host: the final round's misincorporation table)]\n" );
    return 2;
  }
  init_comp();

  /* ---- set-up: mia_main.c:299-335 (matrices), 618-733 (reference, k-mer tables) */
  static int32_t fwd[MIAGPU_PSSM_INTS], fpsm[MIAGPU_PSSM_INTS], rpsm[MIAGPU_PSSM_INTS];
  char ref_id[128], ref_desc[160];
  int ref_len;
  char* ref = read_reference( ref_fn, ref_id, ref_desc, &ref_len );
  miagpu_ctx* g;
  double t0 = now_ms(), t_init, t_parse, t_pass1, t_rounds = 0, t_write = 0, t1;
  CK( miagpu_read_pssm( mat_fn, fwd ) );
  CK( miagpu_create( &g, 0 ) );
  CK( miagpu_set_homopolymer( g, hp_special ) );
  CK( miagpu_set_pssm( g, fwd ) );
  CK( miagpu_get_pssm( g, fpsm, rpsm ) );
  CK( miagpu_set_reference( g, ref, ref_len, circular, 1 ) );
  CK( miagpu_build_kmers( g, k, 0 ) );
  t_init = now_ms() - t0;

  /* ---- pass 1 over the whole file (mia_main.c:746-805), one batch */
  miagpu_fastx* fx;
  int64_t n = 0, j, m = 0;
  const uint8_t* bases; const int64_t *off, *id_off, *desc_off; const char *ids, *descs; const int32_t* qual_sum;
  CK( miagpu_fastx_open( &fx, frag_fn ) );
  CK( miagpu_fastx_next( fx, (int64_t)1 << 40, &n ) );
  CK( miagpu_fastx_batch( fx, &bases, &off, &ids, &id_off, &descs, &desc_off, &qual_sum ) );
  t_parse = now_ms() - t0 - t_init;
  CK( miagpu_upload_reads( g, n, bases, off ) );
  int32_t *hits = xmalloc( n * 4 ), *score = xmalloc( n * 4 ), *as = xmalloc( n * 4 ), *ae = xmalloc( n * 4 ), *start = xmalloc( n * 4 ),
          *end = xmalloc( n * 4 );
  uint8_t *rc = xmalloc( n ), *keep = xmalloc( n );
  CK( miagpu_pass1( g, hits, score, NULL, NULL, rc, as, ae, start, end, NULL, NULL, NULL, NULL ) );

  /* sg_align's accept test (mia.c:1614), the AlnSeq slots pass 1 merges in input order (mia.c:1619-1643), the pass-1 cull over
     every accepted read (mia_main.c:848), then clean_FSDB (mia.c:400-406): reads that scored <= 0 (-D only) leave the FSDB */
  int64_t* src = xmalloc( n * 8 );
  int32_t maln_size = 0;
  int64_t n_acc = 0;
  int32_t *a_len = xmalloc( n * 4 ), *a_thr = xmalloc( n * 4 ), *a_score = xmalloc( n * 4 ), *a_first = xmalloc( n * 4 );
  uint8_t* a_below = xmalloc( n );
  int64_t* a_src = xmalloc( n * 8 );
  {
    /* find_alignable_len (mia.c:69-91) against the wrapped, upper-cased input reference: -D only */
    int wrap = circular ? ( ref_len < MIAGPU_MAX_READ ? ref_len : MIAGPU_MAX_READ ) : 0, wl = ref_len + wrap;
    int32_t* npre = xmalloc( ( (size_t)wl + 1 ) * 4 );
    for ( j = 0; j < wl; j++ ) npre[j + 1] = npre[j] + ( toupper( (unsigned char)ref[j % ref_len] ) == 'N' );
    for ( j = 0; j < n; j++ ) {
      int L = (int32_t)( off[j + 1] - off[j] ), al = L;
      keep[j] = ( hits[j] > 0 && ( score[j] >= FIRST_ROUND_SCORE_CUTOFF || distant_ref ) );
      if ( !keep[j] ) continue;
      if ( distant_ref ) {
        int64_t a = as[j], e = ae[j] > wl ? wl : ae[j];
        if ( a >= 0 && e > a ) al -= npre[e] - npre[a];
        if ( al < 15 ) al = 15;                                                          /* MIN_ALIGNABLE_LEN */
      }
      a_len[n_acc] = L; a_thr[n_acc] = al; a_score[n_acc] = score[j]; a_first[n_acc] = maln_size; a_src[n_acc] = j;
      maln_size += 1 + ( start[j] > end[j] );
      n_acc++;
    }
    free( npre );
  }
  /* pass-1 cull (mia_main.c:848): the fit over the accepted reads that score >= 2000, the threshold by (alignable) length; only
     the sticky flags of the AlnSeq slots survive */
  double slope = 0, icpt = 0;
  uint8_t* slot_dropped = xmalloc( (size_t)maln_size + 2 );
  if ( !repeat_filt ) {
    if ( hard_cut > 0 || score_cut_set ) CK( miagpu_cull_flags( n_acc, a_thr, a_score, NULL, hard_cut, score_cut_set, user_slope, user_icpt, a_below ) );
    else {
      CK( miagpu_score_cut( n_acc, a_len, a_score, NULL, &slope, &icpt ) );
      CK( miagpu_cull_flags( n_acc, a_thr, a_score, NULL, 0, 1, slope, icpt, a_below ) );
    }
    for ( j = 0; j < n_acc; j++ )
      if ( a_below[j] ) {
        slot_dropped[a_first[j]] = 1;
        if ( start[a_src[j]] > end[a_src[j]] ) slot_dropped[a_first[j] + 1] = 1;
      }
  }
  for ( j = 0; j < n_acc; j++ ) {
    int64_t q = a_src[j];
    if ( score[q] > 0 ) src[m++] = q; else keep[q] = 0;
  }
  int32_t *f_len = xmalloc( m * 4 ), *f_score = xmalloc( m * 4 ), *f_as = xmalloc( m * 4 ), *f_ae = xmalloc( m * 4 ), *abr = xmalloc( m * 4 );
  uint8_t *f_rc = xmalloc( m ), *dropped = xmalloc( m ), *f_known = xmalloc( m ), *known_now = xmalloc( m ), *rc_now = xmalloc( m ), *revc = xmalloc( n );
  int32_t *f_front = xmalloc( m * 4 ), *f_back = xmalloc( m * 4 );
  int64_t *s_off = xmalloc( ( m + 1 ) * 8 ), *f_id_off = xmalloc( ( m + 1 ) * 8 ), *f_desc_off = xmalloc( ( m + 1 ) * 8 );
  for ( j = 0; j < m; j++ ) {
    int64_t q = src[j];
    f_len[j] = (int32_t)( off[q + 1] - off[q] ); f_score[j] = score[q]; f_as[j] = as[q]; f_ae[j] = ae[q]; f_rc[j] = rc[q];
    f_known[j] = score[q] > FIRST_ROUND_SCORE_CUTOFF;                                    /* mia.c:1653 */
    n_unknown += !f_known[j];
    s_off[j + 1] = s_off[j] + f_len[j];
    f_id_off[j + 1] = f_id_off[j] + ( id_off[q + 1] - id_off[q] );
    f_desc_off[j + 1] = f_desc_off[j] + ( desc_off[q + 1] - desc_off[q] );
  }
  { int64_t k = 0;                                                                        /* front_asp / back_asp as slot indices */
    for ( j = 0; j < m; j++ ) {
      while ( a_src[k] != src[j] ) k++;
      f_front[j] = a_first[k];
      f_back[j] = start[src[j]] > end[src[j]] ? a_first[k] + 1 : -1;
    } }
  /* host copy of the FSDB: stored orientation (fsdb.c:209-227), ids, descriptions -- what the writer needs */
  uint8_t* stored = xmalloc( (size_t)s_off[m] + 1 );
  char *f_ids = xmalloc( (size_t)f_id_off[m] + 1 ), *f_descs = xmalloc( (size_t)f_desc_off[m] + 1 );
  for ( j = 0; j < m; j++ ) {
    int64_t q = src[j], L = f_len[j], t;
    if ( !( f_rc[j] && f_known[j] ) ) memcpy( stored + s_off[j], bases + off[q], (size_t)L );   /* revcomped only when the strand is known */
    else for ( t = 0; t < L; t++ ) stored[s_off[j] + t] = comp[bases[off[q] + L - 1 - t]];
    memcpy( f_ids + f_id_off[j], ids + id_off[q], (size_t)( id_off[q + 1] - id_off[q] ) );
    memcpy( f_descs + f_desc_off[j], descs + desc_off[q], (size_t)( desc_off[q + 1] - desc_off[q] ) );
  }
  Fsdb F;
  memset( &F, 0, sizeof F );
  if ( repeat_filt ) {
    F.m = m; F.joc = just_outer_coords; F.by_qual = repeat_filt == 2;
    F.len = f_len; F.score = f_score; F.as = f_as; F.ae = f_ae; F.rc = f_rc;
    F.qual = xmalloc( m * 4 ); F.split = xmalloc( m ); F.unique = xmalloc( m ); F.df = xmalloc( m ); F.db = xmalloc( m );
    F.order = xmalloc( m * 8 ); F.slot_cap = 2 * m + 64; F.slot = xmalloc( (size_t)F.slot_cap );
    for ( j = 0; j < m; j++ ) { F.qual[j] = qual_sum[src[j]]; F.split[j] = start[src[j]] > end[src[j]]; F.order[j] = j; }
    filter_and_cull( g, &F );
  }
  int64_t n_kept = 0;
  for ( j = 0; j < n; j++ ) revc[j] = rc[j] && score[j] > FIRST_ROUND_SCORE_CUTOFF;       /* add_virgin_fs2fsdb, fsdb.c:209-227 */
  CK( miagpu_compact_reads( g, keep, revc, &n_kept ) );
  if ( n_kept != m ) { fprintf( stderr, "mia_gpu: compact_reads kept %lld of %lld\n", (long long)n_kept, (long long)m ); return 3; }
  CK( miagpu_set_alignment_inputs( g, f_rc, f_as, f_ae ) );
  if ( repeat_filt ) {
    if ( n_unknown ) { fprintf( stderr, "mia_gpu: reads that score exactly 2000 together with -u / -U are not handled by this host\n" ); return 3; }
    CK( miagpu_set_cut_inputs( g, f_len, NULL, dropped ) );
  }
  else CK( miagpu_set_fsdb( g, f_len, NULL, f_score, f_known, f_front, f_back, maln_size, slot_dropped, distant_ref ) );
  memcpy( known_now, f_known, (size_t)m );
  miagpu_fastx_close( fx );
  fprintf( stderr, "mia_gpu: %lld reads read, %lld aligned in pass 1 (%d with unknown strand)\n", (long long)n, (long long)m, n_unknown );
  t_pass1 = now_ms() - t0 - t_init - t_parse;

  /* ---- rounds (mia_main.c:878-976): one library call each */
  size_t cons_cap = (size_t)ref_len * 4 + 4096;
  char *last = xmalloc( cons_cap ), *cons = xmalloc( cons_cap ), fn[4096], iter_id[64];
  int32_t* gaps = xmalloc( cons_cap * 4 );
  int64_t *run_off = xmalloc( ( m + 1 ) * 8 ), total = 0, cap = 0, n_aln = 0;
  uint16_t* packed = NULL;
  uint8_t* st = xmalloc( m );
  int iter = 0, converged = 0;
  for ( j = 0; j < ref_len; j++ ) last[j] = (char)toupper( (unsigned char)ref[j] );      /* make_ref_upper mia.c:642-648 */
  last[ref_len] = 0;
  while ( !converged && iter < MAX_ITER ) {
    int32_t cons_len = 0, L = (int32_t)strlen( last );
    if ( (size_t)L * 4 + 4096 > cons_cap ) {            /* the consensus grew: seq_len + sum(gaps) + 1 characters come back */
      cons_cap = (size_t)L * 4 + 4096;
      last = realloc( last, cons_cap ); cons = realloc( cons, cons_cap ); gaps = realloc( gaps, cons_cap * 4 );
      if ( !last || !cons || !gaps ) { fprintf( stderr, "mia_gpu: out of memory\n" ); return 1; }
    }
    iter++;
    t1 = now_ms();
    CK( miagpu_set_cons_capacity( g, (int64_t)cons_cap ) );
    CK( miagpu_set_reference( g, last, L, circular, 0 ) );
    if ( repeat_filt ) {
      CK( miagpu_realign_resident( g ) );
      CK( miagpu_adopt_alignment( g, f_score, f_as, f_ae ) );
      for ( j = 0; j < m; j++ ) F.split[j] = f_as[j] > ( f_ae[j] > L ? f_ae[j] - L : f_ae[j] );
      filter_and_cull( g, &F );
      CK( miagpu_consensus_natural( g, F.df, F.db, cons_code, gaps, NULL, cons, &cons_len ) );
    }
    else {
      if ( distant_ref ) {                                                              /* mia_main.c:120-174, from iteration 2 on */
        int64_t tried = 0, learned = 0;
        CK( miagpu_distant_retry( g, &tried, &learned ) );
        if ( tried ) fprintf( stderr, "mia_gpu: iteration %d: %lld strand-unknown reads re-tried, %lld learned their strand\n", iter, (long long)tried, (long long)learned );
        if ( learned ) {                                                                /* strcpy( fs->seq, tmp_rc ): the host copy follows */
          CK( miagpu_get_fsdb( g, known_now, rc_now, NULL, NULL, NULL, NULL, NULL ) );
          for ( j = 0; j < m; j++ )
            if ( known_now[j] && !f_known[j] ) {
              int64_t a = s_off[j], b = s_off[j + 1] - 1;
              f_known[j] = 1; f_rc[j] = rc_now[j];
              if ( rc_now[j] )
                for ( ; a <= b; a++, b-- ) { unsigned char x = stored[a], y = stored[b]; stored[a] = comp[y]; stored[b] = comp[x]; }
            }
        }
      }
      CK( miagpu_iterate_resident( g, hard_cut, score_cut_set, user_slope, user_icpt, cons_code, &slope, &icpt, dropped, gaps, cons, &cons_len ) );
      CK( miagpu_adopt_alignment( g, f_score, f_as, f_ae ) );
    }
    cons[cons_len] = 0;
    converged = !strcmp( cons, last );
    t_rounds += now_ms() - t1;
    t1 = now_ms();
    if ( !final_only || converged || iter == MAX_ITER ) {
      miagpu_maln_header hd;
      miagpu_maln_reads rd;
      CK( miagpu_get_alignment( g, NULL, NULL, NULL, abr, NULL, st ) );
      for ( j = 0; j < m; j++ )
        if ( st[j] != MIAGPU_ST_OK && f_known[j] ) {   /* e.g. more runs than MIAGPU_MAX_RUNS: never written as if it were fine */
          fprintf( stderr, "mia_gpu: read %lld came back with status 0x%x in iteration %d\n", (long long)src[j], st[j], iter );
          return 4;
        }
      CK( miagpu_get_runs_packed( g, NULL, NULL, 0, &total ) );
      if ( total > cap ) { free( packed ); cap = total + total / 4 + 16; packed = xmalloc( (size_t)cap * 2 ); }
      CK( miagpu_get_runs_packed( g, run_off, packed, cap, &total ) );
      memset( &hd, 0, sizeof hd );
      memset( &rd, 0, sizeof rd );
      snprintf( iter_id, sizeof iter_id, "ConsAssem.%d", iter );
      hd.ref_id = iter > 1 ? iter_id : ref_id;                                           /* mia_main.c:47, 62-65 */
      hd.ref_desc = iter > 1 ? "iteration assembly" : ref_desc;
      hd.ref_seq = last; hd.ref_len = L; hd.circular = circular; hd.maln_size = maln_size; hd.cons_code = cons_code;
      hd.gaps = gaps; hd.fpsm = fpsm; hd.rpsm = rpsm;
      rd.n = m; rd.bases = stored; rd.offsets = s_off; rd.ids = f_ids; rd.id_off = f_id_off; rd.descs = f_descs; rd.desc_off = f_desc_off;
      rd.rc = f_rc; rd.score = f_score; rd.as = f_as; rd.ae = f_ae; rd.abr = abr; rd.run_off = run_off; rd.packed = packed;
      rd.dropped_front = dropped; rd.dropped_back = dropped;
      if ( repeat_filt ) {
        for ( j = 0; j < m; j++ ) { F.df[j] = F.df[j] == 1; F.db[j] = F.db[j] == 1; }      /* 2 = not unique: see unique_best */
        rd.unique_best = F.unique; rd.dropped_front = F.df; rd.dropped_back = F.db; rd.fsdb_order = F.order;
      }
      snprintf( fn, sizeof fn, "%s.%d", root, iter );
      if ( repeat_filt ) CK( miagpu_write_maln( fn, &hd, &rd, &n_aln ) );
      else CK( miagpu_write_maln_fsdb( g, fn, &hd, &rd, &n_aln ) );
      fprintf( stderr, "mia_gpu: iteration %d: %lld AlnSeqs -> %s\n", iter, (long long)n_aln, fn );
    }
    t_write += now_ms() - t1;
    { char* t = last; last = cons; cons = t; }
  }
  fprintf( stderr, converged ? "Assembly convergence after %d rounds\n" : "Assembly did not converge after %d rounds, quitting\n", iter );
  if ( damage_fn ) {                                    /* the device still holds the final round */
    static int64_t table[MIAGPU_MISINC_INTS];
    CK( miagpu_misincorporation( g, table ) );
    write_damage( damage_fn, table );
  }
  fprintf( stderr, "mia_gpu: timing ms: init %.1f parse %.1f pass1 %.1f rounds %.1f write %.1f total %.1f\n", t_init, t_parse, t_pass1,
           t_rounds, t_write, now_ms() - t0 );
  miagpu_destroy( g );
  return 0;
}
