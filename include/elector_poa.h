/* elector_poa.h -- C-ABI of the B200-native ELECTOR POA hot path.
 *
 * The reference has no in-process API for this path: its boundary is the `poa`
 * executable (src/poa-graph/main.c) driven by elector/alignment.py:59-63, and the
 * tally is elector/computeStats.py reading msa.fa.  These entry points are what a
 * cgo / ctypes / JNI binding of that path would bind; each cites the reference
 * interface it replaces (paths relative to the reference tree).  Plain pointers and
 * sizes only; the caller owns every host buffer; all functions return 0 on success
 * and a negative ELECTOR_E* code on error (elector_last_error() gives the text).
 * There is no CPU fallback: without a CUDA device elector_poa_init fails.
 */
#ifndef ELECTOR_POA_H
#define ELECTOR_POA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ELECTOR_OK 0
#define ELECTOR_EINVAL (-1)   /* bad argument (NULL pointer, empty window, ...) */
#define ELECTOR_EMATRIX (-2)  /* matrix file unreadable / malformed (main.c:149-155 -> exit 1) */
#define ELECTOR_EUNSUPPORTED (-3) /* matrix outside the supported class (see DESIGN.md) */
#define ELECTOR_ECUDA (-4)    /* CUDA runtime error, no device, out of memory */
#define ELECTOR_EIO (-5)      /* FASTA / output file unreadable (main.c:245-262 -> exit 1) */
#define ELECTOR_ETOOLARGE (-6) /* window larger than the large tier supports */
#define ELECTOR_ECAPACITY (-7) /* caller's output buffer too small */

typedef struct elector_ctx elector_ctx;

/* Number of per-read tally counters written by elector_tally_run (see ELECTOR_T_*). */
#define ELECTOR_TALLY_K 24
enum {
  ELECTOR_T_TP = 0, ELECTOR_T_FP, ELECTOR_T_FN,
  ELECTOR_T_COR, ELECTOR_T_UNCOR,           /* corBases / uncorBases   (computeStats.py:371-393) */
  ELECTOR_T_UNCORCOR, ELECTOR_T_UNCORUNCOR, /* uncorCorBases / uncorUncorBases */
  ELECTOR_T_INSC, ELECTOR_T_DELC, ELECTOR_T_SUBSC, /* indels() corrected (:309-317) */
  ELECTOR_T_INSU, ELECTOR_T_DELU, ELECTOR_T_SUBSU, /* indels() uncorrected (:318-328) */
  ELECTOR_T_GCREF, ELECTOR_T_GCCOR,         /* GC counts over all columns (:421-424) */
  ELECTOR_T_LENREF, ELECTOR_T_LENCOR, ELECTOR_T_LENUNC, /* non-gap lengths (getLen :268) */
  ELECTOR_T_GAPSLEFT, ELECTOR_T_GAPSRIGHT,  /* gapsAndExtensions (:472-488) */
  ELECTOR_T_MISSING,                        /* missingSize after clamping (:489-495) */
  ELECTOR_T_EXTENDED,                       /* extended bases, -1 when the read is not extended */
  ELECTOR_T_NCOLS,                          /* msa line length */
  ELECTOR_T_ASSESSED                        /* 1 when len(reference row) > 10 (:577) */
};

/* Replaces: process start of `poa` -- black_flag_init + read_score_matrix
 * (main.c:38,149-155; seq_util.c:82-217).  device = CUDA ordinal.  matrix_path may be
 * NULL for the shipped blosum80.mat values (identity 0/-10, gaps 10 5 5, T=10, D=5). */
int elector_poa_init(int device, const char *matrix_path, elector_ctx **ctx);

/* Replaces: process exit of `poa` (main.c:293-312). */
void elector_poa_free(elector_ctx *ctx);

/* Text of the last error on this context (or of the last failed init when ctx==NULL). */
const char *elector_last_error(const elector_ctx *ctx);

/* Replaces: the per-window loop of `poa` (main.c:265-284): for each window
 * initialize_seqs_as_lpo x3, buildup_progressive_lpo (align_lpo_po + fuse_lpo, twice)
 * and xlate_lpo_to_al.  Inputs are raw FASTA letters (any case; normalised on the
 * device like create_seq.c:39-43 + seq_util.c:253-263,37-52), concatenated, with
 * n+1 offsets per sequence kind; every window must have >=1 letter in each sequence.
 * Outputs (host): nring[w] = MSA columns; the three rows of window w start at
 * rows_out + row_off[w] + s*row_stride[w], s = 0 ref, 1 corrected, 2 uncorrected
 * (lpo_format.c:407-421 order), row_stride[w] = nring[w] rounded up to 4;
 * score1/score2 = best_score of the two align_lpo_po calls (align_lpo_po2.c:486);
 * cells[w] = DP inner-loop iterations (align_lpo_po2.c:309-320).  score1, score2 and
 * cells may be NULL.  rows_cap >= elector_poa_rows_bound(...) always suffices. */
int elector_poa_run(elector_ctx *ctx, int64_t n_windows,
                    const char *ref, const int64_t *ref_off,
                    const char *cor, const int64_t *cor_off,
                    const char *unc, const int64_t *unc_off,
                    char *rows_out, int64_t rows_cap, int64_t *row_off, int32_t *row_stride,
                    int32_t *nring, int32_t *score1, int32_t *score2, int64_t *cells);

/* Upper bound of the bytes elector_poa_run / elector_pipeline_run can write to rows_out: O(1), 3 bytes per letter of the
 * call plus 9 per window, in 16-byte granules.  Row positions inside the buffer are arbitrary (row_off[] says where
 * each window's rows are); with a buffer of at least this size the pipelined entry point returns the rows in several
 * regions while later windows still compute.  A smaller buffer is accepted as long as the exact need fits. */
int64_t elector_poa_rows_bound(int64_t n_windows, const int64_t *ref_off,
                               const int64_t *cor_off, const int64_t *unc_off);

/* Same computation with every buffer already resident in device memory (pointers
 * from cudaMalloc / torch); nothing is copied to the host.  Used for the
 * device-resident throughput figure and by callers that chain the tally on device.
 * d_rows_used receives (on the device) the bytes used in d_rows_out.  lens_host_*
 * are host copies of the offsets (needed to bin windows by size). */
int elector_poa_run_device(elector_ctx *ctx, int64_t n_windows,
                           const char *d_ref, const int64_t *d_ref_off,
                           const char *d_cor, const int64_t *d_cor_off,
                           const char *d_unc, const int64_t *d_unc_off,
                           const int64_t *h_ref_off, const int64_t *h_cor_off,
                           const int64_t *h_unc_off,
                           char *d_rows_out, int64_t rows_cap, int64_t *d_row_off,
                           int32_t *d_row_stride, int32_t *d_nring, int32_t *d_score1,
                           int32_t *d_score2, int64_t *d_cells, int64_t *d_rows_used);

/* Replaces: the whole `poa` process body for one shard (main.c:241-287) -- reads the
 * three FASTA files (fasta_format.c:10-66 semantics), aligns every record triplet and
 * writes the PIR file (lpo_format.c:398-426 format).  print_perm != 0 also prints the
 * reference's "0 1 2 \n" line per window on stdout (buildup_lpo.c:545).  Returns 0, or
 * ELECTOR_EIO when a file cannot be opened / holds no record (reference exit code 1). */
int elector_poa_files(elector_ctx *ctx, const char *ref_fasta, const char *cor_fasta,
                      const char *unc_fasta, const char *pir_out, int print_perm);

/* Replaces: Donatello's per-read merge (src/split/Donatello.cpp:13-31,50-84: windows
 * concatenated per read, columns whose corrected row is 'n' dropped) followed by the
 * integer part of computeStats.py's per-read tally (gapsAndExtensions :472-498,
 * findGapStretches :104-189, getCorrectedPositions :712-752, getTPFNFP :399-440).
 * Input: n_reads merged reads; row pointers are given as offsets into three
 * concatenated row buffers (ref, corrected, uncorrected; n_reads+1 offsets shared by
 * the three, all rows of one read have equal length).  counters_out[r*ELECTOR_TALLY_K+k].
 * Ratios (recall, precision, rates) stay with the caller, as in computeStats.py:444-468. */
int elector_tally_run(elector_ctx *ctx, int64_t n_reads, const char *row_ref,
                      const char *row_cor, const char *row_unc, const int64_t *row_off,
                      int64_t *counters_out);

/* Replaces: `Donatello smsa<i> msa.fa` (Donatello.cpp:50-84) on in-memory window MSAs: the
 * windows read_first[r] .. read_first[r+1]-1 (consecutive records with the same header) are
 * concatenated and every column whose corrected row is 'n' is dropped (clean_msa :13-31).
 * Window rows are addressed as in elector_poa_run's output.  Merged read r occupies
 * m_len[r] bytes at offset m_off[r] in each of m_ref / m_cor / m_unc (m_cap bytes each;
 * the sum of nring plus 16 bytes per read always suffices). */
int elector_merge_run(elector_ctx *ctx, int64_t n_reads, const int64_t *read_first, int64_t n_windows,
                      const char *rows, int64_t rows_bytes, const int64_t *row_off, const int32_t *row_stride,
                      const int32_t *nring, char *m_ref, char *m_cor, char *m_unc, int64_t m_cap,
                      int64_t *m_off, int32_t *m_len);

/* The same merge followed by the tally, chained on the device-resident output of
 * elector_poa_run_device (nothing returns to the host except through d_counters_out, which
 * is device memory: n_reads*ELECTOR_TALLY_K int64).  h_read_first is a host array. */
int elector_merge_tally_device(elector_ctx *ctx, int64_t n_reads, const int64_t *h_read_first,
                               int64_t n_windows, const char *d_rows, int64_t rows_bytes,
                               const int64_t *d_row_off, const int32_t *d_row_stride,
                               const int32_t *d_nring, int64_t *d_counters_out);

/* Replaces: one round of elector/alignment.py:98-129 plus the integer part of
 * computeStats.py for the windows of n_reads reads -- Pool(fpoa) (main.c:265-284 per window),
 * Donatello (Donatello.cpp:50-84) and the per-read tally (computeStats.py:371-498) -- as ONE
 * call on host buffers.  Windows read_first[r] .. read_first[r+1]-1 belong to read r.  The work
 * is cut into chunks of whole reads, each processed by one of a few worker contexts the library
 * creates (own host thread and streams): a chunk's inputs arrive and its results leave while
 * other chunks compute (pin the host buffers for that).  Not reentrant per context.  Outputs as in
 * elector_poa_run plus counters_out[r*ELECTOR_TALLY_K + k] and sums_out[k] = sum over reads
 * (k = ELECTOR_T_EXTENDED sums the extended bases of extended reads only).  With n_reads == 0
 * (read_first, counters_out, sums_out NULL) only the alignment runs. */
int elector_pipeline_run(elector_ctx *ctx, int64_t n_windows,
                         const char *ref, const int64_t *ref_off,
                         const char *cor, const int64_t *cor_off,
                         const char *unc, const int64_t *unc_off,
                         int64_t n_reads, const int64_t *read_first,
                         char *rows_out, int64_t rows_cap, int64_t *row_off, int32_t *row_stride,
                         int32_t *nring, int32_t *score1, int32_t *score2, int64_t *cells,
                         int64_t *counters_out, int64_t *sums_out);

/* ---- compact wire format of the pipelined call ------------------------------------------------------------------------
 * elector_pipeline_run moves 1 byte per letter and three 8-byte offsets per window to the device and 3 bytes per MSA column
 * back: at 10 000 triplets of 10 kb that is 0.35 GB each way, and the call is bound by the host link, not by the kernels.
 * elector_pipeline_run2 is the same call (alignment.py:98-129 + Donatello + the integer part of computeStats.py) with
 *   - letters as 2 bits each plus a list of the few that are not A, C, G or T (elector_pack_letters; the reads of ELECTOR are
 *     DNA: `N` placeholder windows and IUPAC codes are the exceptions), window offsets sent as 32-bit values;
 *   - outputs chosen by the caller: the per-window rows (what `poa -pir` writes; temporary files in ELECTOR,
 *     alignment.py:128-129), the merged rows per read (what Donatello appends to msa.fa) as bytes or as 4 bits per column,
 *     the per-read counters and their sums.  Any output pointer may be NULL; with all row pointers NULL only counters return. */
typedef struct elector_packed {
  const uint8_t *bits;      /* letter i in bits 2*(i&3)..2*(i&3)+1 of byte i>>2: A/a = 0, C/c = 1, G/g = 2, T/t = 3 */
  int64_t n_letters;
  const int64_t *exc_pos;   /* ascending positions of the letters that are none of these (their two bits are ignored) ... */
  const uint8_t *exc_byte;  /* ... and their bytes, as in the FASTA file */
  int64_t n_exc;
} elector_packed;

/* Packs n letters (host side, outside the timed call: the caller packs once what it reads from its FASTA files).  bits must
 * hold (n + 3) / 4 bytes.  Returns the number of exceptions; when it exceeds exc_cap only the first exc_cap were stored and
 * the call has to be repeated with larger arrays. */
int64_t elector_pack_letters(const char *letters, int64_t n, uint8_t *bits, int64_t *exc_pos, uint8_t *exc_byte, int64_t exc_cap);

/* 4-bit column codes of the merged rows (m_nibbles != 0): column i of a row in bits 4*(i&1).. of byte i>>1 */
#define ELECTOR_NIBBLE_CHARS ".acgtnA"   /* codes 0..6; code 15 = any other character: listed in m_esc_* */
/* one byte per column for the three rows together (m_nibbles == 2): ref + 6 * cor + 36 * unc, each row's character coded
 * 0..5 over ELECTOR_COLUMN_CHARS; 255 = some character of the column is outside the code: its three characters are listed
 * in m_esc_*.  A third of the bytes of the 4-bit form: what Donatello appends to msa.fa (Donatello.cpp:50-84) in 1 B / column. */
#define ELECTOR_COLUMN_CHARS ".acgtn"
/* host side: the three rows of n columns back from their codes (escaped columns come out as '?': patch them from m_esc_*) */
void elector_unpack_columns(const uint8_t *codes, int64_t n, char *ref, char *cor, char *unc);

typedef struct elector_pipeline_io {
  int64_t n_windows, n_reads;
  /* letters: bytes (ref / cor / unc) or packed (pref / pcor / punc); offsets as in elector_pipeline_run */
  const char *ref, *cor, *unc;
  const elector_packed *pref, *pcor, *punc;
  const int64_t *ref_off, *cor_off, *unc_off, *read_first;
  /* optional with packed letters: the window lengths as 32-bit values (n_windows each), prepared by the caller like the packed
   * letters.  They are what crosses the link (the device adds them up); without them the call derives 32-bit offsets from the
   * 64-bit ones itself, a pass over 24 bytes per window on the calling thread. */
  const int32_t *ref_len, *cor_len, *unc_len;
  /* per window, each may be NULL (rows_out NULL: row_off / row_stride unused) */
  char *rows_out; int64_t rows_cap; int64_t *row_off; int32_t *row_stride;
  int32_t *nring, *score1, *score2; int64_t *cells;
  /* merged rows per read (Donatello.cpp:50-84), each may be NULL: read r's three rows are m_len[r] columns from column
   * m_off[r] of m_ref / m_cor / m_unc (m_off[r] is a multiple of 16; m_cap columns per buffer, elector_merged_bound()
   * always suffices).  m_nibbles == 1: two columns per byte (ELECTOR_NIBBLE_CHARS), the buffers hold m_cap / 2 bytes, and the
   * columns with code 15 are listed in m_esc_pos (3 * column + row, unordered) / m_esc_byte (at most m_esc_cap; *m_n_esc
   * receives their number).  m_nibbles == 2: the three rows in one byte per column (ELECTOR_COLUMN_CHARS) in m_ref alone
   * (m_cap bytes; m_cor / m_unc unused), code 255 = the column's three characters are in the escape list. */
  char *m_ref, *m_cor, *m_unc; int64_t m_cap; int m_nibbles;
  int64_t *m_off; int32_t *m_len;
  int64_t *m_esc_pos; uint8_t *m_esc_byte; int64_t m_esc_cap; int64_t *m_n_esc;
  /* per read / per call */
  int64_t *counters_out, *sums_out;
  /* optional, instead of ref_len / cor_len / unc_len: the window lengths as 16-bit values (every window shorter than 65 536
   * letters, which the alignment requires anyway: 16-bit node indices).  Half the bytes of the 32-bit lengths on the link. */
  const uint16_t *ref_len16, *cor_len16, *unc_len16;
} elector_pipeline_io;

int64_t elector_merged_bound(int64_t n_windows, int64_t n_reads, const int64_t *ref_off, const int64_t *cor_off, const int64_t *unc_off);
int elector_pipeline_run2(elector_ctx *ctx, const elector_pipeline_io *io);

/* ---- window cutting (SURVEY.md 8f-1) -----------------------------------------------------------------------------------
 * Replaces: the body of one `masterSplitter` round (src/split/Master_Splitter.cpp:352-472 minus the file I/O) -- best_split
 * (:310-332: split() at k = 15, 13, 11, 9) for each of n triplets, given as three letter arrays with n + 1 offsets each
 * (reference, uncorrected, corrected: the splitter's argv[1..3]) and the length of each triplet's header line (it takes part
 * in largest_fragment(), :158-169).  threshold = argv[10] (SIZE_CORRECTED_READ_THRESHOLD).  Triplets whose reference read has
 * at most 2 letters are the caller's to drop (:414).
 * Outputs: status[t] (0 cut, 1 corrected read too short = small_reads, 2 not cut = wrongly_cor_reads; 1 and 2 give the
 * placeholder record AAA / AAA / AAA, :417-431), k_used[t], and the windows of all triplets in triplet order as three letter
 * arrays with offsets -- the records the reference writes to out1<i> / out2<i> / out3<i>, ready for elector_pipeline_run*
 * (read_first[t] = first window of triplet t).  elector_split_bounds gives capacities that always suffice. */
int elector_split_bounds(int64_t n_triplets, const int64_t *ref_off, const int64_t *unc_off, const int64_t *cor_off,
                         int64_t *win_cap, int64_t *ref_cap, int64_t *unc_cap, int64_t *cor_cap);
int elector_split_run(elector_ctx *ctx, int64_t n_triplets, const char *ref, const int64_t *ref_off, const char *unc,
                      const int64_t *unc_off, const char *cor, const int64_t *cor_off, const int32_t *header_len, double threshold,
                      int32_t *status, int32_t *k_used, int64_t *read_first, int64_t win_cap, int64_t *w_ref_off,
                      int64_t *w_unc_off, int64_t *w_cor_off, char *w_ref, int64_t w_ref_cap, char *w_unc, int64_t w_unc_cap,
                      char *w_cor, int64_t w_cor_cap, int64_t *n_windows);

/* Replaces: one round of elector/alignment.py:98-129 from the READS on -- masterSplitter (Master_Splitter.cpp:352-472), Pool(fpoa)
 * (main.c:265-284 per window), Donatello (Donatello.cpp:50-84) and the integer part of computeStats.py -- as one call in which the
 * windows never leave the device: cut by elector_split_run's kernels, aligned where they are, merged per triplet (the records of a
 * triplet share its header, :283-285, so a triplet is one Donatello read) and tallied.  Inputs as elector_split_run.  Outputs:
 * status / k_used / read_first (n_triplets + 1) / n_windows as elector_split_run (each may be NULL), counters_out[t*ELECTOR_TALLY_K+k],
 * sums_out[k] (may be NULL), and optionally the merged rows of every triplet (what Donatello appends to msa.fa): m_len[t] columns at
 * m_off[t] of m_ref / m_cor / m_unc (m_cap bytes each; letters of the call + 32 per triplet suffices). */
int elector_reads_run(elector_ctx *ctx, int64_t n_triplets, const char *ref, const int64_t *ref_off, const char *unc,
                      const int64_t *unc_off, const char *cor, const int64_t *cor_off, const int32_t *header_len, double threshold,
                      int32_t *status, int32_t *k_used, int64_t *read_first, int64_t *n_windows, int64_t *counters_out,
                      int64_t *sums_out, char *m_ref, char *m_cor, char *m_unc, int64_t m_cap, int64_t *m_off, int32_t *m_len);
/* Device time of the last elector_reads_run or elector_reads_pipeline_run (summed over its chunks): window cutting, alignment,
 * merge + tally (CUDA events, ms). */
int elector_last_reads_ms(const elector_ctx *ctx, float *ms_split, float *ms_poa, float *ms_merge_tally);

/* ---- pipelined reads-in call ------------------------------------------------------------------------------------------
 * Replaces: one or more rounds of elector/alignment.py:98-129 -- masterSplitter (Master_Splitter.cpp:352-472), Pool(fpoa)
 * (main.c:265-284 per window), Donatello (Donatello.cpp:50-84) and the integer part of computeStats.py -- for any number of
 * triplets in one call.  The call is cut into chunks of whole triplets (balanced by letters); each chunk runs the body of
 * elector_reads_run start to finish on one worker context (own host thread and stream), so that one chunk's copies overlap
 * another chunk's kernels, and the workers may sit on several devices.  Inputs as elector_reads_run, plus the devices:
 * devices[0 .. n_devices - 1] (NULL / 0: the context's own device; a device may be listed more than once); every listed device
 * gets ELECTOR_PIPELINE_WORKERS worker contexts (default 2), created on first use and kept until elector_poa_free.
 * ELECTOR_PIPELINE_CHUNKS forces the number of chunks.  Every output may be NULL and is byte-identical to one elector_reads_run
 * over the same triplets, however the call is chunked, except where m_off places the merged rows:
 *   status[n], k_used[n], read_first[n + 1] (global window indices), *n_windows,
 *   counters_out[n][ELECTOR_TALLY_K], sums_out[ELECTOR_TALLY_K],
 *   stretches_out[n][ELECTOR_STRETCH_K]: what elector_last_stretches gives after elector_reads_run,
 *   the merged rows of triplet t: m_len[t] bytes at m_off[t] of m_ref / m_cor / m_unc (all five or none).
 * Placement rule: the rows of triplet t start at or after the bound of the triplets before it, B(t) = (letters of triplets
 * 0 .. t-1 in the three kinds + 32 * t) rounded down to 16, so that every chunk writes into the caller's buffers at once.
 * m_cap must be at least the bound of the call, letters of all triplets + 32 * n rounded up to 16; a smaller m_cap
 * returns ELECTOR_ECAPACITY before any work.  A failure on any worker stops the others at their next chunk; the call returns
 * that error and its text. */
typedef struct elector_reads_io {
  int64_t n_triplets;
  const char *ref, *unc, *cor;                    /* letters as bytes, as in the FASTA files */
  const int64_t *ref_off, *unc_off, *cor_off;     /* n_triplets + 1 offsets each */
  const int32_t *header_len;                      /* length of each triplet's header line */
  double threshold;                               /* SIZE_CORRECTED_READ_THRESHOLD */
  const int *devices; int n_devices;
  int32_t *status, *k_used;
  int64_t *read_first, *n_windows;
  int64_t *counters_out, *sums_out;
  int32_t *stretches_out;
  char *m_ref, *m_cor, *m_unc; int64_t *m_off; int32_t *m_len; int64_t m_cap;
} elector_reads_io;

int elector_reads_pipeline_run(elector_ctx *ctx, const elector_reads_io *io);

/* ---- report (SURVEY.md 8f-2) -------------------------------------------------------------------------------------------
 * The border gap stretches of every read of the last tally on this context (elector_tally_run, elector_merge_tally_device,
 * elector_reads_run; not the chunked elector_pipeline_run*; elector_reads_pipeline_run returns them in stretches_out): what findGapStretches keeps (computeStats.py:179-189), as
 * stretches_out[r*ELECTOR_STRETCH_K] = their number and (first, last) column pairs behind it.  With gapsLeft / gapsRight they
 * rebuild the column mask of getCorrectedPositions (:712-752). */
#define ELECTOR_STRETCH_K 17
int elector_last_stretches(elector_ctx *ctx, int64_t n_reads, int32_t *stretches_out);

/* What computeStats.outputRecallPrecision returns and prints (computeStats.py:196-264), as numbers. */
typedef struct elector_report_summary {
  int64_t assessed_reads, throughput_uncorrected, throughput_corrected;
  double recall, precision;                 /* means over reads, round(.., 7) */
  double correct_rate_uncorrected;          /* not rounded by the reference */
  double correct_rate_corrected, error_rate; /* round(.., 7); error_rate = 1 - corrected bases / all bases (:669) */
  int64_t trimmed_or_split, split_reads, trimmed_reads;
  double mean_missing;
  int64_t extended_reads;
  double mean_extension, gc_ref, gc_cor;    /* gc_*: per cent */
  int64_t small_reads, wrongly_cor_reads;
  int64_t ins_u, del_u, subs_u, ins_c, del_c, subs_c;
  double homopolymer_ratio;
  int32_t size_distribution_complete;       /* 0: trimmed / split reads present but corrected_fasta missing: no "sequences" lines */
} elector_report_summary;

/* Replaces: computeStats.outputRecallPrecision (computeStats.py:196-264) with computeMetrics (:519-675), outputMetrics (:444-468)
 * and outputReadSizeDistribution (:273-288) on the per-record counters of the device tally instead of a Python pass over msa.fa.
 * Records are those of msa.fa in file order: headers (without '>', header_off[n + 1] offsets into `headers`), counters
 * [n][ELECTOR_TALLY_K], stretches [n][ELECTOR_STRETCH_K], and the merged rows (m_ref / m_cor, record i at m_off[i]): rows are
 * read for split reads (consecutive records with one header: the missing size of :595-599) and for the last read (the homopolymer
 * ratio: the reference keeps the last read's only, :560); m_cor == NULL leaves the ratio at 1.  small_reads / wrongly_cor_reads: the
 * splitter's two counters; size_threshold: SIZE_CORRECTED_READ_THRESHOLD; homopolymer_threshold: reportedHomopolThreshold;
 * compensated_sum: 0 adds the per-read ratios left to right like sum() of Python < 3.12 (the README example of the reference),
 * 1 with Neumaier's compensation like Python >= 3.12 (the means can differ in their 16th digit);
 * corrected_fasta: the sorted corrected reads (read for the "sequences" lines when there are trimmed / split reads; may be NULL).
 * Writes <out_dir>/[<soft>_]per_read_metrics.txt and <out_dir>/<size_file_name> (out_dir NULL: nothing is written), the text the
 * reference appends to its log file (log_text) and the text it prints (stdout_text); host only, no device needed.
 * Errors: elector_last_error(NULL). */
int elector_report_write(int64_t n_records, const char *headers, const int64_t *header_off, const int64_t *counters,
                         const int32_t *stretches, const char *m_ref, const char *m_cor, const int64_t *m_off,
                         int small_reads, int wrongly_cor_reads, double size_threshold, int homopolymer_threshold, int compensated_sum,
                         const char *corrected_fasta, const char *out_dir, const char *soft, const char *size_file_name,
                         elector_report_summary *summary, char *log_text, int64_t log_cap, char *stdout_text, int64_t stdout_cap);

/* The same from the merged rows alone (the records of msa.fa in memory): the tally runs on the device, the report on its counters. */
int elector_report_run(elector_ctx *ctx, int64_t n_records, const char *headers, const int64_t *header_off, const char *m_ref,
                       const char *m_cor, const char *m_unc, const int64_t *m_off, int small_reads, int wrongly_cor_reads,
                       double size_threshold, int homopolymer_threshold, int compensated_sum, const char *corrected_fasta, const char *out_dir,
                       const char *soft, const char *size_file_name, elector_report_summary *summary, char *log_text,
                       int64_t log_cap, char *stdout_text, int64_t stdout_cap);

/* ---- file preparation in front of the splitter (SURVEY.md 8f-4; host only) ---------------------------------------------
 * Replaces: readAndSortFasta (elector/readAndSortFiles.py:150-166): the records of a FASTA file (Bio.SeqIO semantics: multi-line
 * sequences joined, blanks dropped) sorted by their whole header line, ties in file order, written two lines per record. */
int elector_sort_fasta(const char *in_path, const char *out_path, int64_t *n_records);
/* Replaces: duplicateRefReads (:171-191) fed by the occurrence table readAndSortFasta returns for the corrected reads (:520-522):
 * every reference / uncorrected record with k corrected records of the same header is written k times as header_0 .. header_(k-1),
 * the others are dropped: as many triplets as there are corrected reads. */
int elector_duplicate_reads(const char *sorted_ref, const char *sorted_unc, const char *sorted_cor, const char *new_ref,
                            const char *new_unc, int64_t *n_triplets);

/* Global counters on the device: d_sums[k] += sum over reads of d_counters[r*ELECTOR_TALLY_K+k]
 * (ELECTOR_T_EXTENDED: extended reads only).  d_sums is ELECTOR_TALLY_K int64 the caller zeroes;
 * with one rank per GPU this vector is what the final all-reduce carries. */
int elector_tally_sum_device(elector_ctx *ctx, int64_t n_reads, const int64_t *d_counters, int64_t *d_sums);

/* Device-side timing for callers (bench.py): which = 0 records the start event, 1 the stop
 * event, both on the context's launching stream; elapsed returns the milliseconds between
 * them after synchronising on the stop event. */
int elector_event_record(elector_ctx *ctx, int which);
int elector_event_elapsed_ms(elector_ctx *ctx, float *ms);

/* Measured INT32 issue peak of this device (the roofline denominator of the DP kernel):
 * a register-only chain of IMAD / IADD3 / VIMNMX on every SM; returns tera integer
 * lane-operations per second (an fma-pipe IMAD counts once, like an alu-pipe op). */
int elector_int32_peak(elector_ctx *ctx, double *tiops_mixed, double *tiops_alu_only);

/* Timing of the kernels launched by the last run on this context, measured with CUDA
 * events on the launching stream: total ms and number of kernel launches. */
int elector_last_kernel_ms(const elector_ctx *ctx, float *ms, int *launches);

/* Split of that time for the last alignment run: ms_phase1 = sort 1 + the DP1-phase kernels
 * (poa_dp1_kernel), ms_total - ms_phase1 = sort 2 + the DP2-phase kernels (poa_dp2_kernel). */
int elector_last_phase_ms(const elector_ctx *ctx, float *ms_phase1, float *ms_total);

#ifdef __cplusplus
}
#endif
#endif
