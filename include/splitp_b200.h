/* splitp_b200 -- C ABI of the B200 (sm_100a) engine for the SplitP hot path.
 *
 * The reference (js51/SplitP v0.3.2) is pure Python and has no FFI layer: its boundary is the set of
 * callables re-exported at splitp/__init__.py:15-18.  The entry points below are what a ctypes
 * binding inside those callables would call (see INTEGRATION.md); each one names the reference
 * function it replaces.  All pointers are DEVICE pointers unless the name says `h_`; the caller owns
 * every buffer; the library keeps no state besides a thread-local error string.  Every call is
 * asynchronous on `stream` (a cudaStream_t passed as void*) unless documented as synchronising.
 * Return value: 0 = ok, otherwise an spb_status; spb_last_error() describes the failure.
 *
 * Encodings (fixed by splitp/constants.py:7-8): A=0 C=1 G=2 T=3.
 *   key      : base-4 number of a site pattern, taxon 0 most significant (same significance as
 *              `__index_of`, splitp/constructions.py:166-171).  n <= 31 taxa -> uint64.
 *   sm       : "site-major" packed alignment, a little-endian bit stream of 2n-bit keys, site s at
 *              bits [2n*s, 2n*s+2n).  N*n/4 bytes.  Allocate spb_sm_words(n, N) uint32.
 *   planes   : "taxon-major" bit planes, uint32 [n][2][Wp]; plane 0 = low code bit, plane 1 = high
 *              code bit, site s = bit (s%32) of word s/32.  N*n/4 bytes.  Wp = spb_plane_words(N).
 *   valid    : uint32 [Wp] bit mask, 1 = every taxon has A/C/G/T at that site
 *              (splitp/parsers/fasta.py:55-57).
 *   split    : spb_split -- ordered taxon positions of both sides; order = digit significance.
 */
#ifndef SPLITP_B200_H
#define SPLITP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  SPB_OK = 0,
  SPB_ERR_ARG = 1,      /* maps to ValueError */
  SPB_ERR_CUDA = 2,     /* maps to RuntimeError */
  SPB_ERR_CAPACITY = 3, /* a caller-provided buffer is too small; maps to MemoryError */
  SPB_ERR_UNSUPPORTED = 4 /* maps to NotImplementedError */
} spb_status;

#define SPB_MAX_TAXA 64
#define SPB_MAX_BATCH 64 /* splits per batched flatten launch (their descriptors travel as ONE 9 KB kernel parameter) */
#define SPB_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull

typedef struct {
  int32_t n;            /* taxa in the pattern */
  int32_t a, b;         /* side sizes */
  uint8_t idx_a[SPB_MAX_TAXA]; /* positions (0..n-1) of side A, most significant digit first */
  uint8_t idx_b[SPB_MAX_TAXA];
} spb_split;

int spb_version(void);
const char* spb_last_error(void);
/* number of CUDA kernels this library has launched in this process so far (bench.py's gpu_launches) */
uint64_t spb_launch_count(void);
/* number of SMs / compute capability of the current device; -1 when there is no device */
int spb_device_info(int* sm_count, int* cc_major, int* cc_minor);

int64_t spb_sm_words(int n_taxa, int64_t n_sites);
int64_t spb_plane_words(int64_t n_sites);

/* ---- f1: FASTA text -> packed alignment (parsers/fasta.py:20-35 reads, :48-57 validity rule) ---- */
/* d_chars: uint8 [n][row_stride]; is_ascii=1: bytes are characters (ACGTacgt valid), 0: bytes are
 * codes 0..3 (anything else invalid).  Any of d_sm / d_planes may be NULL.  d_sm needs n <= 32. */
int spb_pack(const uint8_t* d_chars, int n_taxa, int64_t n_sites, int64_t row_stride, int is_ascii,
             uint32_t* d_sm, uint32_t* d_planes, uint32_t* d_valid, void* stream);

/* ---- a1: get_pattern_counts (parsers/fasta.py:48-63) ---- */
/* Direct-indexed table, n <= 14: d_table uint32 [4^n] must be zeroed by the caller (or hold partial
 * counts to accumulate into, e.g. another site range).  d_first (optional, uint32 [4^n], filled with
 * 0xFFFFFFFF) receives the first site index of each pattern (dict insertion order).
 * d_usable (uint64, optional) accumulates the number of valid sites in [site_begin, site_end). */
int spb_count_direct(const uint32_t* d_sm, const uint32_t* d_valid, int n_taxa, int64_t site_begin,
                     int64_t site_end, uint32_t* d_table, uint32_t* d_first, uint64_t* d_usable,
                     void* stream);
/* Non-zero cells of a direct table -> (keys ascending = lexicographic A<C<G<T order of
 * simulation.py:50-54, counts, first).  d_tmp: uint32 [spb_compact_tmp_words(cells)].
 * Writes P to d_num (uint64).  capacity = length of the output arrays. */
int64_t spb_compact_tmp_words(int64_t cells);
int spb_compact_direct(const uint32_t* d_table, const uint32_t* d_first, int64_t cells, uint64_t* d_keys,
                       uint32_t* d_counts, uint32_t* d_first_out, int64_t capacity, uint64_t* d_num,
                       uint32_t* d_tmp, void* stream);
/* Open-addressing hash table for 15 <= n <= 31 (works for any n <= 31): d_hkeys uint64 [cap] filled
 * with 0xFF bytes, d_hcounts uint32 [cap] zeroed, d_hfirst optional (0xFF filled).  cap = power of 2.
 * d_overflow (uint32) is set non-zero if the table filled up (SPB_ERR_CAPACITY must then be raised
 * by the caller after reading it). */
int spb_count_hash(const uint32_t* d_sm, const uint32_t* d_valid, int n_taxa, int64_t site_begin,
                   int64_t site_end, uint64_t* d_hkeys, uint32_t* d_hcounts, uint32_t* d_hfirst,
                   int64_t cap, uint64_t* d_usable, uint32_t* d_overflow, void* stream);
int spb_compact_hash(const uint64_t* d_hkeys, const uint32_t* d_hcounts, const uint32_t* d_hfirst,
                     int64_t cap, uint64_t* d_keys, uint32_t* d_counts, uint32_t* d_first_out,
                     int64_t capacity, uint64_t* d_num, uint32_t* d_tmp, void* stream);
/* Multi-GPU merge of direct tables without reducing all 4^n cells: every rank compacts its table, the (key, count) lists
 * are all-gathered (a few hundred KB instead of a 64 MB allreduce at 12 taxa) and added into a zeroed table with this call
 * (d_table uint32 [cells], keys < cells), which spb_compact_direct then turns into the sorted global list. */
int spb_direct_merge(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, int64_t cells, uint32_t* d_table, void* stream);
/* Merge a (keys, counts) list into a hash table (multi-GPU merge of hashed tables). */
int spb_hash_merge(const uint64_t* d_keys, const uint32_t* d_counts, const uint32_t* d_first, int64_t num,
                   uint64_t* d_hkeys, uint32_t* d_hcounts, uint32_t* d_hfirst, int64_t cap,
                   uint32_t* d_overflow, void* stream);

/* ---- wide keys, up to 64 taxa (BASELINE config 4): 128-bit base-4 pattern keys stored as two uint64 {lo, hi} ---- */
/* d_wide: uint64 [n_sites][2], 16-byte aligned; d_valid: uint32 [spb_plane_words(n_sites)] (zero-filled by the caller). */
int spb_pack_wide(const uint8_t* d_chars, int n_taxa, int64_t n_sites, int64_t row_stride, int is_ascii, uint64_t* d_wide,
                  uint32_t* d_valid, void* stream);
/* get_pattern_counts (parsers/fasta.py:48-63) with 128-bit keys: open addressing, d_hkeys uint64 [cap][2] filled with
 * 0xFF bytes (16-byte aligned), d_hcounts uint32 [cap] zeroed, cap = power of 2.  The all-ones key (all-T pattern at
 * 64 taxa) is the EMPTY marker, its count goes to *d_special (uint64, zeroed by the caller).
 * d_hfirst (optional, uint32 [cap + 1], 0xFF filled) receives the first site of every pattern (dict insertion order);
 * its last cell belongs to the all-ones key. */
int spb_count_hash_wide(const uint64_t* d_wide, const uint32_t* d_valid, int64_t site_begin, int64_t site_end,
                        uint64_t* d_hkeys, uint32_t* d_hcounts, uint32_t* d_hfirst, int64_t cap, uint64_t* d_special,
                        uint64_t* d_usable, uint32_t* d_overflow, void* stream);
int spb_hash_merge_wide(const uint64_t* d_keys, const uint32_t* d_counts, const uint32_t* d_first, int64_t num,
                        uint64_t* d_hkeys, uint32_t* d_hcounts, uint32_t* d_hfirst, int64_t cap, uint64_t* d_special,
                        uint32_t* d_overflow, void* stream);
/* Non-empty slots -> (keys uint64 [capacity][2], counts, optional first) in arbitrary order; *d_num = their number. */
int spb_compact_hash_wide(const uint64_t* d_hkeys, const uint32_t* d_hcounts, const uint32_t* d_hfirst, int64_t cap,
                          uint64_t* d_keys, uint32_t* d_counts, uint32_t* d_first, int64_t capacity, uint64_t* d_num,
                          void* stream);
/* Exact Gram F F^T (double [4^a][4^a], a = 1, 2 or 3) of the reduced flattening (constructions.py:31-55) of the split
 * {h_idx_a} | {all other taxa}, computed from the hashed table by one lookup per (pattern, row). */
int spb_thin_gram_wide(const uint64_t* d_hkeys, const uint32_t* d_hcounts, int64_t cap, const uint64_t* d_special, int n_taxa,
                       const uint8_t* h_idx_a, int a, double* d_G, void* stream);
/* The same Gram with a column filter (two bitmaps of filter_words uint32 each in d_filter, zeroed here;
 * spb_thin_filter_words(cap) = 8 x cap bits per bitmap): patterns whose column holds no second pattern skip their
 * 4^a - 1 table lookups.  Bit-identical result; d_filter == NULL is spb_thin_gram_wide. */
int64_t spb_thin_filter_words(int64_t cap);
int spb_thin_gram_wide_filtered(const uint64_t* d_hkeys, const uint32_t* d_hcounts, int64_t cap, const uint64_t* d_special,
                                int n_taxa, const uint8_t* h_idx_a, int a, uint32_t* d_filter, int64_t filter_words,
                                double* d_G, void* stream);
/* Pattern LISTS with 128-bit keys (d_keys uint64 [num][2] = {lo, hi}, 16-byte aligned), e.g. a {pattern: value} mapping of
 * 32..64 taxa.  Projection: the digits of the m <= n_taxa positions h_pos (HOST array, most significant first) of every key,
 * as a base-4 number: d_out uint64 [num] for m <= 31 (flattening row / column indices), uint64 [num][2] {lo, hi} (16-byte
 * aligned) for m >= 32 (keys of a sub-alignment). */
int spb_project_wide(const uint64_t* d_keys, int64_t num, int n_taxa, const uint8_t* h_pos, int m, uint64_t* d_out, void* stream);
/* Joint tables N double [n][n][4][4] (N[i][j][x][y] = sum of the values d_vals[p] of the patterns with taxon i in state x
 * and taxon j in state y; written in full) of a weighted pattern list, for spb_pair_transform.  Computed as E^T diag(v) E
 * (E = one-hot digits) on the fp64 tensor cores with a fixed summation order: bitwise reproducible, exact for
 * integer values below 2^53.  Values must be finite.  d_ws: double [spb_pair_tables_wide_ws(num, n_taxa)]. */
int64_t spb_pair_tables_wide_ws(int64_t num, int n_taxa);
int spb_pair_tables_wide(const uint64_t* d_keys, const double* d_vals, int64_t num, int n_taxa, double* d_N, double* d_ws,
                         void* stream);

/* ---- a7-a10: flattening (constructions.py:7-102) ---- */
/* value kinds for the pattern table handed to the flattening kernels */
#define SPB_VAL_U32 0 /* counts; written value = count / divisor (one IEEE division, fasta.py:66-70), divisor<=0 -> count */
#define SPB_VAL_F64 1 /* values copied verbatim (dict inputs) */
/* rows/cols of every pattern (int64) -- the COO triplets behind FlatFormat.sparse (:86-102) */
int spb_flatten_coo(const uint64_t* d_keys, int64_t num, const spb_split* split, int64_t* d_rows,
                    int64_t* d_cols, void* stream);
/* FlatFormat.dense := sparse.todense(): d_out double [4^a][4^b], zero-filled by this call. */
int spb_flatten_dense(const uint64_t* d_keys, const void* d_vals, int val_kind, double divisor, int64_t num,
                      const spb_split* split, double* d_out, void* stream);
/* FlatFormat.reduced (:31-55) in two steps.  plan: marks used rows/cols and ranks them
 * (sorted-unique), returns the reduced shape in h_shape[2] (SYNCHRONISES).  d_rank_r uint32 [4^a + 1],
 * d_rank_c uint32 [4^b + 1], d_tmp uint32 [spb_compact_tmp_words(max(4^a,4^b))].  Sides are limited to
 * 13 taxa each.  fill: d_out double [R][C] zero-filled by the call. */
int spb_flatten_reduced_plan(const uint64_t* d_keys, int64_t num, const spb_split* split, uint32_t* d_rank_r,
                             uint32_t* d_rank_c, uint32_t* d_tmp, int64_t* h_shape, void* stream);
int spb_flatten_reduced_fill(const uint64_t* d_keys, const void* d_vals, int val_kind, double divisor,
                             int64_t num, const spb_split* split, const uint32_t* d_rank_r,
                             const uint32_t* d_rank_c, int64_t R, int64_t C, double* d_out, void* stream);
/* Variants with a winner workspace d_win (uint32 per output cell): required only when the split does not
 * cover all taxa, where the reference's assignment semantics (last pattern wins, constructions.py:43,101)
 * need a tie-break.  The plain entry points above pass d_win = NULL and fail with SPB_ERR_ARG in that case. */
int spb_flatten_dense_w(const uint64_t* d_keys, const void* d_vals, int val_kind, double divisor, int64_t num,
                        const spb_split* split, double* d_out, uint32_t* d_win, void* stream);
int spb_flatten_reduced_fill_w(const uint64_t* d_keys, const void* d_vals, int val_kind, double divisor,
                               int64_t num, const spb_split* split, const uint32_t* d_rank_r,
                               const uint32_t* d_rank_c, int64_t R, int64_t C, double* d_out, uint32_t* d_win,
                               void* stream);
/* Scoring layout of a count flattening: low byte of every count into d_s0 (uint8, rows_pad x pitch cells;
 * rows_pad >= R, pitch >= C) and the remainder (count - (count & 255)) of counts >= 256 as COO triplets
 * (d_hi_rc int32 [cap][2], d_hi_val uint32 [cap]), *d_hi_num (uint32, zeroed by the call) = number of
 * triplets (may exceed cap -> caller must check).  layout: SPB_S0_ROWMAJOR = [rows_pad][pitch], pitch % 16 == 0
 * (plain layout, accepted by spb_gram_u8_simt and the correction kernels only); SPB_S0_K4MAJOR = 32-bit words of 4
 * consecutive k stored at word (k/4) * rows_pad + r (the dp4a operand layout, rows_pad % 4 == 0, pitch % 16 == 0);
 * SPB_S0_TILED = 128 x 128-byte tiles in the tensor-core operand layout (see csrc/gram.cu), rows_pad % 128 ==
 * 0 and pitch % 128 == 0.  flags & SPB_U8_NO_MEMSET: d_s0 is known to be all zero (see spb_flatten_u8_clear),
 * skip the memset.  If d_rank_r/d_rank_c are non-NULL the reduced row/col ranks are used instead of the raw
 * base-4 indices.  Requires the split to cover all n taxa (otherwise cells would collide). */
#define SPB_S0_ROWMAJOR 0
#define SPB_S0_TILED 1
#define SPB_S0_K4MAJOR 2
#define SPB_U8_NO_MEMSET 1
int spb_flatten_u8(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, const spb_split* split,
                   const uint32_t* d_rank_r, const uint32_t* d_rank_c, uint8_t* d_s0, int64_t rows_pad,
                   int64_t pitch, int layout, int flags, int32_t* d_hi_rc, uint32_t* d_hi_val, uint32_t* d_hi_num,
                   int64_t hi_cap, void* stream);
/* Writes zeros back to exactly the cells spb_flatten_u8 touched for this split (P byte stores instead of a
 * rows_pad * pitch memset), restoring the all-zero state for the next split. */
int spb_flatten_u8_clear(const uint64_t* d_keys, int64_t num, const spb_split* split, const uint32_t* d_rank_r,
                         const uint32_t* d_rank_c, uint8_t* d_s0, int64_t rows_pad, int64_t pitch, int layout,
                         void* stream);
/* Batched forms (one launch for nb <= SPB_MAX_BATCH splits of equal shape, raw base-4 indices only): entry b uses
 * h_splits[b] (HOST array), the S0 buffer d_s0 + b * s0_stride (bytes) and the high-part buffers
 * d_hi_rc + b * 2 * hi_cap, d_hi_val + b * hi_cap, d_hi_num + b. */
int spb_flatten_u8_batch(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, const spb_split* h_splits, int nb,
                         uint8_t* d_s0, int64_t s0_stride, int64_t rows_pad, int64_t pitch, int layout, int flags,
                         int32_t* d_hi_rc, uint32_t* d_hi_val, uint32_t* d_hi_num, int64_t hi_cap, void* stream);
int spb_flatten_u8_clear_batch(const uint64_t* d_keys, int64_t num, const spb_split* h_splits, int nb, uint8_t* d_s0,
                               int64_t s0_stride, int64_t rows_pad, int64_t pitch, int layout, void* stream);

/* ---- a11: subflattening (constructions.py:108-198) ---- */
/* Raw pair statistics of sites [32*word_begin, 32*word_end) accumulated (atomicAdd) into d_raw
 * (uint64 [spb_pair_raw_words(n)], zeroed by the caller; sum-reducible across GPUs). */
int64_t spb_pair_raw_words(int n_taxa);
int spb_pair_tables(const uint32_t* d_planes, const uint32_t* d_valid, int n_taxa, int64_t plane_words,
                    int64_t word_begin, int64_t word_end, uint64_t* d_raw, void* stream);
/* raw -> N double [n][n][4][4] (joint tables, N[i][i] diagonal = marginal) and the Hadamard-type
 * basis change T[i][j] = H N[i][j] H^T (H = sign table of constructions.py:143-161).  divisor > 0
 * turns counts into probabilities first (count / divisor); divisor < 0 divides by the number of usable sites held in
 * d_raw (fasta.py:66-70) without a host round trip; divisor == 0 keeps counts.  d_total (double) = sum of all values. */
int spb_pair_finalize(const uint64_t* d_raw, int n_taxa, double divisor, double* d_N, double* d_T,
                      double* d_total, void* stream);
/* Same tables from a weighted pattern list (dict inputs): d_N must be zeroed by the caller. */
int spb_pair_tables_weighted(const uint64_t* d_keys, const double* d_vals, int64_t num, int n_taxa,
                             double* d_N, void* stream);
int spb_pair_transform(const double* d_N, int n_taxa, double* d_T, double* d_total, void* stream);
/* One subflattening matrix, row-major double [(3a+1)][(3b+1)]. */
int spb_subflatten(const double* d_T, const double* d_total, int n_taxa, const spb_split* split, double* d_out,
                   void* stream);
/* Batched: scores of `num` splits given as bit masks over taxon positions (bit t set = taxon t on
 * side A; side B = d_masks_b[s] if non-NULL else the complement).  d_scores double [num].
 * Up to 21 taxa: one warp per split (Gram, Householder tridiagonalisation, the 4 largest eigenvalues by bisection,
 * score = sqrt((trace - top4) / trace)); above: one CTA per split with a shared-memory Jacobi solver.
 * SPB_SUBFLATTEN_WARP=0 in the environment forces the second kernel. */
int spb_subflatten_score(const double* d_T, const double* d_total, int n_taxa, const uint64_t* d_masks_a,
                         const uint64_t* d_masks_b, int64_t num, double* d_scores, void* stream);

/* The same scores through TRIPLE tables (the round-2 kernel, up to 43 taxa: sides of at most 21 taxa, k = 3 min(a, b) + 1
 * <= 64): one pass tabulates P[x][x'][y] = T3[x][y] T3[x'][y]^T (3 x 3 blocks) and the margin terms into d_tables (double
 * [spb_subflatten_tables_doubles(n)]), after which the Gram matrix of a subflattening is a sum of a b gathered blocks --
 * no staged matrix, one warp per split with two rows per lane, division-free Sturm counts.  tables_ready != 0 skips the
 * tabulation (d_tables already holds the tables of this d_T). */
int64_t spb_subflatten_tables_doubles(int n_taxa);
int spb_subflatten_score_tables(const double* d_T, const double* d_total, int n_taxa, const uint64_t* d_masks_a,
                                const uint64_t* d_masks_b, int64_t num, double* d_scores, double* d_tables, int tables_ready,
                                void* stream);

/* ---- a12-a14: split_score (phylogenetics.py:280-328), K = 4 hard-coded ---- */
/* G = A A^T for row-major double A [batch][R][C] (lda = C): d_G double [batch][R][R].
 * d_ws: double workspace of spb_gram_f64_ws(R, C, batch) elements (may be NULL when that is 0). */
int64_t spb_gram_f64_ws(int64_t R, int64_t C, int64_t batch);
int spb_gram_f64(const double* d_A, int64_t R, int64_t C, int64_t batch, double* d_G, double* d_ws, void* stream);
/* Exact integer Gram of a u8 matrix (see spb_flatten_u8): d_G double [rows_pad][rows_pad] is OVERWRITTEN with
 * S0 S0^T.  SPB_S0_K4MAJOR: rows_pad <= 64, dp4a kernel.  SPB_S0_TILED: rows_pad == 128 or rows_pad % 256 == 0,
 * tcgen05 (tensor core, kind::i8) kernel.  K = pitch.  d_ws: uint64 [spb_gram_u8_ws(...)] (NULL when that is 0);
 * it holds exact 64-bit partial sums when K is split across CTAs. */
int64_t spb_s0_bytes(int64_t rows_pad, int64_t pitch);
int64_t spb_gram_u8_ws(int64_t rows_pad, int64_t pitch, int layout, int nb);
int spb_gram_u8(const uint8_t* d_s0, int64_t rows_pad, int64_t pitch, int layout, double* d_G, uint64_t* d_ws,
                void* stream);
/* nb matrices in one launch: S0 of entry b at d_s0 + b * s0_stride (bytes), its Gram at d_G + b * g_stride (doubles).
 * The tensor-core kernel schedules the tiles of all matrices over the SMs and splits K only when nb * tiles < #SMs.
 * d_ws: uint64 [spb_gram_u8_ws(rows_pad, pitch, layout, nb)]. */
int spb_gram_u8_batch(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch, int layout,
                      double* d_G, int64_t g_stride, uint64_t* d_ws, void* stream);
/* Same result from a plain SIMT loop, any layout and size: the on-device cross-check used by the tests. */
int spb_gram_u8_simt(const uint8_t* d_s0, int64_t rows_pad, int64_t pitch, int layout, double* d_G, void* stream);
/* Adds the terms of the sparse high part H (F = S0 + H): G += S0 H^T + H S0^T + H H^T, so that G = F F^T. */
int spb_gram_hi_correction(const uint8_t* d_s0, int64_t rows_pad, int64_t pitch, int layout, const int32_t* d_hi_rc,
                           const uint32_t* d_hi_val, const uint32_t* d_hi_num, int64_t hi_cap, double* d_G,
                           void* stream);
int spb_gram_hi_correction_batch(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch,
                                 int layout, const int32_t* d_hi_rc, const uint32_t* d_hi_val, const uint32_t* d_hi_num,
                                 int64_t hi_cap, double* d_G, int64_t g_stride, void* stream);
/* Scores from symmetric PSD Gram matrices d_G double [batch][ld][ld] using the leading k x k block
 * (k <= 128): cyclic Jacobi in shared memory, score = sqrt(sum_{i>=4} lambda_i / sum_i lambda_i).
 * d_eig (optional) double [batch][k] receives the eigenvalues in descending order. */
int spb_score_gram_small(const double* d_G, int64_t k, int64_t ld, int64_t batch, double* d_scores,
                         double* d_eig, void* stream);
/* Scores from large Gram matrices (k > 128): restarted block-Krylov Rayleigh-Ritz for the 4 largest
 * eigenvalues (the role of LAPACK gesdd at phylogenetics.py:281-285), score = sqrt(1 - top4 / trace).
 * d_ws: double [spb_score_gram_large_ws(k, batch)].
 * d_info (optional) double [batch][SPB_SCORE_INFO] = {top4 sum, trace, residual of the top-4 Ritz pairs relative to
 * theta_1, krylov dim, cycles, |change of top4| / trace in the last cycle, theta_4, theta_5, converged (1 / 0), 0}.
 * A matrix that exhausts the cycle budget keeps its last score and reports converged = 0; the call still returns
 * SPB_OK and spb_score_last_unconverged() (thread-local, last call) returns how many matrices did so. */
#define SPB_SCORE_INFO 10
int64_t spb_score_gram_large_ws(int64_t k, int64_t batch);
int spb_score_last_unconverged(void);
int spb_score_gram_large(const double* d_G, int64_t k, int64_t ld, int64_t batch, double* d_scores,
                         double* d_info, double* d_ws, void* stream);
/* The same with a cycle budget max_cycles in 1..40 (40 = spb_score_gram_large).  Every matrix of a batch stays in the
 * cycle until the last one is accepted and the cycles grow (2, 2, 4, 4, 12, ... Krylov blocks), so a caller with a large
 * batch runs the first cycles with a small budget and calls again with the few matrices whose d_info reports
 * converged = 0. */
int spb_score_gram_large_n(const double* d_G, int64_t k, int64_t ld, int64_t batch, double* d_scores, double* d_info,
                           double* d_ws, int max_cycles, void* stream);

/* ---- 32-bit integer form of the exact Gram (halves the HBM traffic of the eigen stage for large matrices) ----
 * spb_gram_u8_batch_i32: G0 = S0 S0^T as int32 [nb][rows_pad][rows_pad] straight from the tensor-core accumulators
 * (tiled layout, rows_pad % 256 == 0, pitch <= 32768 so that one accumulation stays below 2^31).
 * spb_gram_hi_strip_batch: the correction C = S0 H^T + H S0^T + H H^T is non-zero only in the rows / columns of the m
 * distinct rows that hold a high entry; it is returned as the strip d_Cs [nb][cs_rows][rows_pad] (fp64, exact
 * integers, zero-filled here) of those rows, with d_pos [nb][rows_pad] = strip index of a row or -1, d_hr
 * [nb][cs_rows] = the rows, d_hm [nb] = m.  cs_rows must be >= the number of high entries of the table.
 * spb_score_gram_large_i32: spb_score_gram_large on G = G0 + C (same workspace size, same d_info).  d_Gi must hold
 * the FULL symmetric matrix (both triangles, as spb_gram_u8_batch_i32 writes it) with entries in [0, 2^31): the
 * product kernel reads it column-wise. */
int spb_gram_u8_batch_i32(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch, int32_t* d_Gi,
                          int64_t g_stride, void* stream);
int spb_gram_hi_strip_batch(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch, int layout,
                            const int32_t* d_hi_rc, const uint32_t* d_hi_val, const uint32_t* d_hi_num, int64_t hi_cap,
                            double* d_Cs, int64_t cs_rows, int32_t* d_pos, int32_t* d_hr, int32_t* d_hm, void* stream);
/* spb_gram_hi_strip_batch with the cross terms S0 H^T + H S0^T taken from the PATTERN TABLE (a join of the pattern list with
 * the high list on the column index) instead of from column scans of S0: same d_Cs / d_pos / d_hr / d_hm, bit for bit.
 * h_splits: the nb <= SPB_MAX_BATCH splits the S0 buffers were scattered with (every split covers all taxa);
 * d_ws: spb_gram_hi_strip_table_ws(nb, pitch, hi_cap) int32 of scratch.  Only the first d_hm[b] rows of a strip are written
 * (and read by spb_score_gram_large_i32). */
int64_t spb_gram_hi_strip_table_ws(int nb, int64_t pitch, int64_t hi_cap);
int spb_gram_hi_strip_batch_table(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, const spb_split* h_splits, int nb,
                                  int64_t rows_pad, int64_t pitch, const int32_t* d_hi_rc, const uint32_t* d_hi_val,
                                  const uint32_t* d_hi_num, int64_t hi_cap, double* d_Cs, int64_t cs_rows, int32_t* d_pos, int32_t* d_hr,
                                  int32_t* d_hm, int32_t* d_ws, void* stream);
int spb_score_gram_large_i32(const int32_t* d_Gi, int64_t k, int64_t ld, int64_t batch, const double* d_Cs, int64_t cs_rows,
                             const int32_t* d_pos, const int32_t* d_hr, const int32_t* d_hm, double* d_scores, double* d_info,
                             double* d_ws, void* stream);
int spb_score_gram_large_i32_n(const int32_t* d_Gi, int64_t k, int64_t ld, int64_t batch, const double* d_Cs, int64_t cs_rows,
                               const int32_t* d_pos, const int32_t* d_hr, const int32_t* d_hm, double* d_scores, double* d_info,
                               double* d_ws, int max_cycles, void* stream);
/* Diagnostic: d_AQ = G0 d_Q for `batch` int32 Gram matrices through ONE of the product kernels of the eigen-solver
 * (variant 0: column-owning FMA kernel; 1..6: fp64 tensor-core (DMMA) kernels), launched exactly as the solver launches
 * them.  d_Q, d_AQ: [batch][8][k] doubles; d_Qt: spb_symv_i32_ws(k, batch) doubles of scratch.  For tests and
 * scripts/symv_bench.py; the product path reaches these kernels through spb_score_gram_large_i32. */
int64_t spb_symv_i32_ws(int64_t k, int64_t batch);
int spb_symv_i32(const int32_t* d_Gi, int64_t k, int64_t ld, int64_t batch, const double* d_Q, double* d_AQ, double* d_Qt, int variant,
                 void* stream);

/* ---- marginals, rank-1 approximation and rank-1 divergence of a flattening ----
 * reference: phylogenetics.py:331-341 (r = column sums, c = row sums, approximation = r^T c),
 * phylogenetics.py:364-373 (divergence = sum over non-zero cells of F[x,y] log(F[x,y] / (r[y] c[x]))),
 * constructions.py:94-101 (entries whose row / column pattern holds the banned state more than once are zeroed; used by
 * phylogenetics.py:344-361).  States are 0..3 = A,C,G,T; -1 = nothing banned. */
int64_t spb_mi_partials(void); /* doubles of d_partials below */
/* matrix route: F is double [rows][ld] on the device */
int spb_marginals_dense(const double* d_F, int64_t rows, int64_t cols, int64_t ld, double* d_rowsum, double* d_colsum,
                        void* stream);
int spb_mi_dense(const double* d_F, int64_t rows, int64_t cols, int64_t ld, const double* d_rowsum, const double* d_colsum,
                 double* d_partials, double* d_out, void* stream);
/* d_out[i][j] (+)= x[i] * y[j] */
int spb_outer_f64(const double* d_x, int64_t nx, const double* d_y, int64_t ny, double* d_out, int accumulate, void* stream);
/* rows / cols of every pattern as spb_flatten_coo, plus d_banned[i] = 1 where the banned-state rule zeroes the entry */
int spb_flatten_coo_banned(const uint64_t* d_keys, int64_t num, const spb_split* split, int ban_row, int ban_col,
                           int64_t* d_rows, int64_t* d_cols, uint8_t* d_banned, void* stream);
/* pattern-table route, for a split that places every taxon on exactly one side (SPB_ERR_UNSUPPORTED otherwise).
 * Side sums of the RAW values (counts or doubles) are ADDED into d_rowsum / d_colsum (caller zero-fills).  A side is
 * either direct-indexed (d_?keys NULL, ?cap >= 4^side entries, side <= 15 taxa) or an open-addressing table
 * (d_?keys uint64 [?cap] filled with 0xFF bytes, ?cap a power of two >= 2 x distinct side patterns; the sums then sit
 * at the slots of their keys).  d_overflow (uint32, zeroed) is set when a table fills up. */
int spb_table_marginals(const uint64_t* d_keys, const void* d_vals, int val_kind, int64_t num, const spb_split* split,
                        int ban_row, int ban_col, double* d_rowsum, uint64_t* d_rkeys, int64_t rcap, double* d_colsum,
                        uint64_t* d_ckeys, int64_t ccap, uint32_t* d_overflow, void* stream);
/* divergence from the table and the side sums above; values and sums are divided by `divisor` when it is > 0 */
int spb_mi_table(const uint64_t* d_keys, const void* d_vals, int val_kind, double divisor, int64_t num,
                 const spb_split* split, const double* d_rowsum, const uint64_t* d_rkeys, int64_t rcap,
                 const double* d_colsum, const uint64_t* d_ckeys, int64_t ccap, double* d_partials, double* d_out,
                 void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPLITP_B200_H */
