/*
 * b200repair.h -- C ABI of libb200repair.so (hand-written sm_100a CUDA behind the
 * `delphi.repair` API).
 *
 * This is the drop-in boundary for the hot path: each entry point replaces one Py4J static call
 * the reference's Python driver makes into its Scala side (SURVEY.md section 8b).  Reference
 * paths below are relative to maropu/spark-data-repair-plugin @ 7701550d.
 *
 * Conventions
 *   - C linkage, plain pointers and sizes, no C++/torch types.
 *   - every function returns 0 on success, non-zero on failure; dr_last_error(ctx) explains.
 *     Nothing throws across the boundary, nothing aborts.
 *   - "device" pointers are caller-owned device memory (the Python host passes
 *     torch.Tensor.data_ptr()); the library never allocates long-lived device memory except a
 *     small per-context scratch buffer.  "host" pointers are caller-owned host memory.
 *   - `stream` is a cudaStream_t passed as void* (0 = default stream).  Calls that return a
 *     host value (counts, quartiles) synchronise that stream; all others are asynchronous.
 *   - table layout: one device array of int32 codes per column, NULL = -1 (column-major,
 *     label-encoded; numeric columns additionally as float64 with NaN = NULL).
 *   - a cell set is a bitmap per column: uint32 words, bit (r & 31) of word (r >> 5) = row r.
 *   - one dr_ctx per GPU; a ctx is not thread-safe; independent ctxs may run concurrently.
 */
#ifndef B200REPAIR_H
#define B200REPAIR_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DR_MAX_COLS 64 /* computeFreqStats' own limit, RepairApi.scala:241-244 */
#define DR_MAX_PREDS 8     /* predicates of one denial constraint evaluated by dr_dc_exists */
#define DR_MAX_SEGMENTS 32 /* segments of one packed exchange buffer (dr_combine_counts) */
#define DR_OK 0
#define DR_ERR_INVALID 1
#define DR_ERR_CUDA 2
#define DR_ERR_UNSUPPORTED 3

typedef struct dr_ctx dr_ctx;

/* ---- context ------------------------------------------------------------------------------- */
int dr_ctx_create(int device, dr_ctx** out);
int dr_ctx_destroy(dr_ctx* ctx);
const char* dr_last_error(const dr_ctx* ctx);
int dr_abi_version(void);
/* Number of kernels this context has launched so far (bench.py's `gpu_launches`). */
int64_t dr_launch_count(const dr_ctx* ctx);

/* ---- ingest ----------------------------------------------------------------------------------------
 * Replaces handing Spark view names across Py4J (model.py:477-480): label-encoded columns whose
 * dictionary has <= 254 entries travel host -> device as ONE byte per cell (255 = NULL) and are
 * widened to the int32 table layout here (4x less PCIe traffic than int32 codes). */
int dr_widen_u8(dr_ctx* ctx, const uint8_t* src, int64_t n, int32_t* dst, void* stream);

/* Arrow ingest (replaces `spark_df.toPandas()` / the view hand-off of model.py:477-480 with the raw Arrow
 * buffers of the collected table; nothing is re-encoded on the host).
 *
 * dr_h2d_copy / dr_d2h_copy: PAGEABLE host memory <-> device through a ring of pinned 4 MB chunks fed by
 * `n_threads` worker threads (<= 0: a default), each on its own copy stream.  Both calls block until
 * every byte has arrived; `stream` is synchronised first (its earlier work may still use the buffers).
 *
 * dr_index_presence: `used` (device uint32[ceil(dict_size/32)], caller zeroes) gets bit v set iff some
 * valid row holds dictionary index v.  idx: device array of `width`-byte signed integers (1, 2 or 4:
 * Arrow int8 / int16 / int32 dictionary indices); validity: device copy of the Arrow validity bitmap
 * (bit (bit_offset + i) = row i is not NULL) or NULL when the column has no NULLs.
 * dr_index_remap: dst[i] = lut[idx[i]] (device int32[dict_size], -1 for entries to drop), -1 for NULL
 * rows and indices outside [0, dict_size).
 *
 * dr_ids_unique_i64: RepairApi.checkInputTable's uniqueness gate (RepairApi.scala:53-62) on the device:
 * one pass when the ids are strictly increasing, else a radix sort + adjacent compare (allocates
 * 2 * 8 * n bytes for its duration).  *out_unique = 1 / 0.  Synchronises `stream`.
 * dr_gather_i64: out[i] = col[rows[i]] (row ids of the output cells).
 * dr_valid_bits: Arrow validity bitmap of a code array, bit i = codes[i] >= 0 (uint32 words). */
int dr_h2d_copy(dr_ctx* ctx, const void* const* src_host, void* const* dst_dev, const int64_t* bytes, int n_bufs,
                int n_threads, void* stream);
int dr_d2h_copy(dr_ctx* ctx, const void* const* src_dev, void* const* dst_host, const int64_t* bytes, int n_bufs,
                int n_threads, void* stream);
int dr_index_presence(dr_ctx* ctx, const void* idx, int width, const uint8_t* validity, int64_t bit_offset,
                      int64_t n_rows, int32_t dict_size, uint32_t* used, void* stream);
int dr_index_remap(dr_ctx* ctx, const void* idx, int width, const uint8_t* validity, int64_t bit_offset,
                   int64_t n_rows, const int32_t* lut, int32_t dict_size, int32_t* dst, void* stream);
int dr_ids_unique_i64(dr_ctx* ctx, const int64_t* ids, int64_t n, int* out_unique, void* stream);
int dr_gather_i64(dr_ctx* ctx, const int64_t* col, const int32_t* rows, int64_t n, int64_t* out, void* stream);
int dr_valid_bits(dr_ctx* ctx, const int32_t* codes, int64_t n, uint32_t* bits, void* stream);

/* ---- a2 + a7/a8: NULL scan fused with per-column histograms ------------------------------------
 * Replaces ErrorDetectorApi.detectNullCells (ErrorDetectorApi.scala:30-34,128-157: K_t UNION-ALL
 * scans) and the single-attribute GROUPING SETS of RepairApi.computeFreqStats
 * (RepairApi.scala:231-273) plus the NULL/ndv part of computeAndGetTableStats (:108-118).
 *   cols[i]      device int32[n_rows]
 *   dom[i]       domain size of column i (codes are in [-1, dom[i]))
 *   bitmaps[i]   device uint32[ceil(n_rows/32)] or NULL; NULL cells are OR-ed in
 *   hist         device int64[sum(dom[i] + 1)], ACCUMULATED (caller zeroes); column i occupies
 *                slots [off_i, off_i + dom[i] + 1), slot 0 = NULL, slot c + 1 = code c
 * One pass over the n_cols columns: 4 * n_cols algorithmic bytes per row. */
int dr_scan_hist(dr_ctx* ctx, const int32_t* const* cols, const int32_t* dom, int n_cols, int64_t n_rows,
                 uint32_t* const* bitmaps, int64_t* hist, void* stream);

/* ---- a5: RegExErrorDetector / DomainValues ----------------------------------------------------
 * Replaces ErrorDetectorApi.detectErrorCellsFromRegEx (ErrorDetectorApi.scala:36-46,159-187).
 * The regex is evaluated once per dictionary entry on the host; lut[c] = 1 iff entry c does NOT
 * match.  Flags  code < 0 (NULL)  or  lut[code] != 0. */
int dr_lut_scan(dr_ctx* ctx, const int32_t* col, int64_t n_rows, const uint8_t* lut, int32_t dict_size,
                uint32_t* bitmap, void* stream);

/* ---- a4: GaussianOutlierErrorDetector ---------------------------------------------------------
 * Replaces ErrorDetectorApi.detectErrorCellsFromOutliers (ErrorDetectorApi.scala:60-70,249-300).
 * dr_quartiles: exact Spark `percentile(col, [0.25, 0.75])` over non-NaN values (linear
 * interpolation at p*(n-1)); out_q host double[2]; out_n host int64 = number of non-NaN values.
 * dr_range_flag: flags  v < lower || v > upper  (NaN never flagged). */
int dr_quartiles(dr_ctx* ctx, const double* col, int64_t n_rows, double* out_q, int64_t* out_n, void* stream);
int dr_range_flag(dr_ctx* ctx, const double* col, int64_t n_rows, double lower, double upper, uint32_t* bitmap,
                  void* stream);

/* ---- a3: ConstraintErrorDetector --------------------------------------------------------------
 * Replaces ErrorDetectorApi.detectErrorCellsFromConstraints (ErrorDetectorApi.scala:48-58,
 * 189-244); the constraint text is parsed on the host (DenialConstraints.scala:82-225).
 *
 * dr_dc_const: single-tuple DC  t1&OP(t1.A, const)&...  -> row_bitmap bit set iff ALL predicates
 * hold.  Predicate p compares cols[p] (dictionary sorted, so order = code order) with a constant:
 *   DR_OP_EQ   code == arg[p]                       (arg = code of the constant, -2 if absent)
 *   DR_OP_IQ   code != arg[p]                       (NOT(<=>): NULL differs from a constant)
 *   DR_OP_LT   code >= 0 && code <  arg[p]          (arg = lower_bound rank of the constant)
 *   DR_OP_GT   code >= 0 && code >= arg[p]          (arg = upper_bound rank of the constant)
 *
 * dr_dc_fd_build / dr_dc_fd_flag: two-tuple DC  EQ(a_1)..EQ(a_m) & IQ(b).  A row violates iff its
 * NULL-safe key group holds >= 2 distinct b (NULL counted as a value).  Keys are mixed-radix
 * numbers  key = sum (code_i + 1) * stride_i  over [0, key_space); lo/hi are device
 * int32[key_space] tables (caller initialises lo = INT32_MAX, hi = INT32_MIN) holding min/max of
 * (b + 1) per key -- both are idempotent reductions, so per-GPU tables combine with one
 * MIN / MAX all-reduce.  flag sets row_bitmap where lo[key] != hi[key]. */
#define DR_OP_EQ 0
#define DR_OP_IQ 1
#define DR_OP_LT 2
#define DR_OP_GT 3
int dr_dc_const(dr_ctx* ctx, const int32_t* const* cols, const int32_t* ops, const int32_t* args, int n_preds,
                int64_t n_rows, uint32_t* row_bitmap, void* stream);
int dr_dc_fd_build(dr_ctx* ctx, const int32_t* const* key_cols, const int64_t* strides, int n_keys,
                   const int32_t* b_col, int64_t n_rows, int64_t key_space, int32_t* lo, int32_t* hi,
                   void* stream);
int dr_dc_fd_flag(dr_ctx* ctx, const int32_t* const* key_cols, const int64_t* strides, int n_keys,
                  int64_t n_rows, int64_t key_space, const int32_t* lo, const int32_t* hi, uint32_t* row_bitmap,
                  void* stream);
/* The same two reductions for key spaces too large for direct tables: an open-addressing hash table of
 * `capacity` (power of two, >= 2 * n_rows) slots keyed by the 64-bit mixed-radix key.  The caller
 * initialises table_keys = all ones (empty), lo = INT32_MAX, hi = INT32_MIN.  dr_dc_hash_flag: mode 0
 * flags lo != hi (EQ.. & IQ(b)), mode 1 flags x >= 0 && x + 1 < hi (EQ.. & LT(x), table built with b = x).
 * Single GPU only: slot positions differ between tables, so they cannot be combined by an all-reduce. */
int dr_dc_hash_build(dr_ctx* ctx, const int32_t* const* key_cols, const int64_t* strides, int n_keys,
                     const int32_t* b_col, int64_t n_rows, int64_t capacity, uint64_t* table_keys, int32_t* lo,
                     int32_t* hi, void* stream);
int dr_dc_hash_flag(dr_ctx* ctx, const int32_t* const* key_cols, const int64_t* strides, int n_keys,
                    const int32_t* x_col, int mode, int64_t n_rows, int64_t capacity, const uint64_t* table_keys,
                    const int32_t* lo, const int32_t* hi, uint32_t* row_bitmap, void* stream);
/* Two-tuple DC  EQ(a_1)..EQ(a_m) & LT(t1.x, t2.x): a row is matched iff another row of its NULL-safe key
 * group has a larger x (`<` is never true for NULL).  hi = the max table dr_dc_fd_build makes for b = x;
 * flags rows with x >= 0 and x + 1 < hi[key].  GT(t1.x, t2.x) is the same test on the reversed codes
 * x' = dom - 1 - x (NULL kept), which the caller materialises. */
int dr_dc_lt_flag(dr_ctx* ctx, const int32_t* const* key_cols, const int64_t* strides, int n_keys,
                  const int32_t* x_col, int64_t n_rows, int64_t key_space, const int32_t* hi, uint32_t* row_bitmap,
                  void* stream);

/* ---- bitmap plumbing (a6: union + distinct of detector outputs, errors.py:405-421) ------------
 * dr_bitmap_or:      dst |= src                                  (n_rows bits)
 * dr_bitmap_andnot:  dst &= ~src
 * dr_bitmap_count:   popcount -> host int64
 * dr_bitmap_to_rows: ascending row indices of set bits -> device int32[capacity]; host count.
 *                    Fails with DR_ERR_INVALID if count > capacity.
 * dr_bitmap_gather:  out bit i = src bit rows[i]                 (n bits out)
 * dr_bitmap_clear_rows: clears bit rows[i] for every i with flags[i] != 0 */
int dr_bitmap_or(dr_ctx* ctx, uint32_t* dst, const uint32_t* src, int64_t n_rows, void* stream);
int dr_bitmap_andnot(dr_ctx* ctx, uint32_t* dst, const uint32_t* src, int64_t n_rows, void* stream);
int dr_bitmap_count(dr_ctx* ctx, const uint32_t* bitmap, int64_t n_rows, int64_t* out_count, void* stream);
int dr_bitmap_to_rows(dr_ctx* ctx, const uint32_t* bitmap, int64_t n_rows, int32_t* out_rows, int64_t capacity,
                      int64_t* out_count, void* stream);
/* Second half of the ordered compaction when the count was already taken: must directly follow
 * dr_bitmap_count on the SAME bitmap (it reuses the per-block offsets left in the context scratch). */
int dr_bitmap_rows_after_count(dr_ctx* ctx, const uint32_t* bitmap, int64_t n_rows, int32_t* out_rows,
                               int64_t capacity, void* stream);
/* Fewer host round trips: the popcounts of up to DR_MAX_COUNT_MANY bitmaps with ONE synchronisation, and
 * the ordered compaction of a bitmap whose count the caller already knows (no synchronisation; writes
 * at most `count` indices).  Both use the context scratch like dr_bitmap_count. */
#define DR_MAX_COUNT_MANY 128
int dr_bitmap_count_many(dr_ctx* ctx, const uint32_t* const* bitmaps, int n_bitmaps, int64_t n_rows,
                         int64_t* out_counts, void* stream);
int dr_bitmap_to_rows_async(dr_ctx* ctx, const uint32_t* bitmap, int64_t n_rows, int32_t* out_rows, int64_t count,
                            void* stream);
/* The same ordered compaction for up to DR_MAX_COUNT_MANY bitmaps (all over n_rows rows) in three launches;
 * counts[i] = popcount of bitmap i (0: skipped), out_rows[i]: device int32[counts[i]].  Asynchronous. */
int dr_bitmaps_to_rows_many(dr_ctx* ctx, const uint32_t* const* bitmaps, int n_bitmaps, int64_t n_rows,
                            int32_t* const* out_rows, const int64_t* counts, void* stream);
int dr_bitmap_gather(dr_ctx* ctx, const uint32_t* src, const int32_t* rows, int64_t n, uint32_t* out,
                     void* stream);
int dr_bitmap_clear_rows(dr_ctx* ctx, uint32_t* bitmap, const int32_t* rows, const uint8_t* flags, int64_t n,
                         void* stream);

/* ---- a3 (general): any two-tuple denial constraint -----------------------------------------------
 * Replaces the generic `EXISTS (SELECT .. WHERE p1 AND p2 ..)` self semi-join of
 * ErrorDetectorApi.scala:211-229 for predicate lists that are not of the FD / single-inequality
 * shapes above.  A row's answer only depends on its projection onto the attributes the constraint
 * references:
 *   dr_key_presence  bit (sum_i (code_i + 1) * strides[i]) of `bits` is set for every row (OR-accumulated;
 *                    key_space bits).  The set bits are the DISTINCT projections of the table.
 *   dr_dc_exists     for distinct projection i (n of them, sorted so that the members of an equality
 *                    group are contiguous): out[i] = 1 iff some j in [group_begin[i], group_end[i])
 *                    satisfies every predicate q: sign[q](left[q][i], right[q][j]); operands are RANKS in
 *                    a per-predicate common order (-1 = NULL): EQ is `<=>`, IQ is NOT(<=>), LT / GT are
 *                    false on NULL (DenialConstraints.scala:66-79).
 *   dr_key_flag      row bit |= viol_bits[key(row)].
 * ---- 8(e): the exchange step of the row-sharded path --------------------------------------------
 * dr_combine_counts: `gathered` = world copies (rank-major) of an n-element int64 buffer, the result
 * of ONE all-gather; segment s = [seg_off[s], seg_off[s+1]) is reduced with seg_op[s] into out[0..n).
 * Replaces the driver-side aggregation Spark does after every scan (SURVEY.md 8e). */
#define DR_RED_SUM 0
#define DR_RED_MIN 1
#define DR_RED_MAX 2
#define DR_RED_OR 3
int dr_key_presence(dr_ctx* ctx, const int32_t* const* cols, const int64_t* strides, int n_keys, int64_t n_rows,
                    int64_t key_space, uint32_t* bits, void* stream);
int dr_key_flag(dr_ctx* ctx, const int32_t* const* cols, const int64_t* strides, int n_keys, int64_t n_rows,
                int64_t key_space, const uint32_t* viol_bits, uint32_t* row_bitmap, void* stream);
int dr_dc_exists(dr_ctx* ctx, const int32_t* const* left, const int32_t* const* right, const int32_t* sign,
                 int n_preds, int64_t n, const int32_t* group_begin, const int32_t* group_end, uint8_t* out,
                 void* stream);
int dr_combine_counts(dr_ctx* ctx, const int64_t* gathered, int world, int64_t n, const int64_t* seg_off,
                      const int32_t* seg_op, int n_seg, int64_t* out, void* stream);

/* ---- a7: discretisation of continuous attributes ----------------------------------------------
 * Replaces the projection of RepairApi.convertToDiscretizedTable (RepairApi.scala:126-169):
 *   out = (int)((v - vmin) / denom * thres)   (truncation toward zero), NaN -> -1; denom == 0 -> -1 */
int dr_discretize(dr_ctx* ctx, const double* vals, int64_t n_rows, double vmin, double denom, int32_t thres,
                  int32_t* out, void* stream);

/* ---- a8: attribute-pair statistics -------------------------------------------------------------
 * Replaces the K_t*(K-1) approx_count_distinct(struct(x, y)) scans (RepairApi.scala:430-448) and
 * the pair GROUPING SETS of computeFreqStats (:231-273).
 *
 * dr_pair_presence: for every pair p = (px[p], py[p]) sets bit  (cx+1)*(dom[y]+1) + (cy+1)  of
 * the pair's bit table for the rows of `n_blocks` row blocks of `block_rows` rows spread evenly
 * over the table (block_rows * n_blocks >= n_rows -> every row).  bits: device uint32, pair p at
 * word offset bit_off[p] (host int64[n_pairs+1], in words), OR-accumulated.  A sample gives lower
 * bounds of the distinct-pair counts, the full table gives them exactly.
 *
 * dr_cooc: exact co-occurrence counts.  out: device int64, pair p occupies
 * [tab_off[p], tab_off[p+1]) with entry (cx+1)*(dom[y]+1) + (cy+1); ACCUMULATED (caller zeroes). */
int dr_pair_presence(dr_ctx* ctx, const int32_t* const* cols, const int32_t* dom, int n_cols, const int32_t* px,
                     const int32_t* py, int n_pairs, const int64_t* bit_off, int64_t n_rows, int64_t block_rows,
                     int64_t n_blocks, uint32_t* bits, void* stream);
int dr_cooc(dr_ctx* ctx, const int32_t* const* cols, const int32_t* dom, int n_cols, const int32_t* px,
            const int32_t* py, int n_pairs, const int64_t* tab_off, int64_t n_rows, int64_t* out, void* stream);
/* dr_cooc_skip: dr_cooc that leaves ONE entry per x value uncounted: rows with cy + 1 == skip[skip_off[p] + cx + 1]
 * are not counted (skip: device int32, -1 = count everything; skip_off: host int64[n_pairs + 1], pair p has
 * dom[px[p]] + 1 entries).  The caller restores table[x][skip[x]] = hist_x[x] - sum_y table[x][y] from the
 * column histogram of the same rows.  With the skipped entry = the most frequent partner of every x the
 * shared-memory atomics -- what bounds dr_cooc -- all but vanish on correlated pairs (the pairs the
 * statistics select), at identical results. */
int dr_cooc_skip(dr_ctx* ctx, const int32_t* const* cols, const int32_t* dom, int n_cols, const int32_t* px,
                 const int32_t* py, int n_pairs, const int64_t* tab_off, int64_t n_rows, const int32_t* skip,
                 const int64_t* skip_off, int64_t* out, void* stream);

/* ---- a9: cell-domain analysis (weak labelling) -------------------------------------------------
 * Replaces RepairApi.computeDomainInErrorCells (RepairApi.scala:479-675) + the weak-label test
 * of errors.py:517-524 for ONE target attribute.
 *   rows          device int32[n_cells]      noisy cells of the target (row indices)
 *   target        device int32[n_rows]       discretised target column (dom_t values)
 *   corr[j]       device int32[n_rows]       discretised correlated attribute j, j < n_corr <= 8
 *   cooc[j]       device int64[(dom_c[j]+1)*(dom_t+1)]  counts, entry (c+1)*(dom_t+1)+(t+1), i.e. the
 *                                            candidate (target) index varies fastest
 *   hist_t        device int64[dom_t+1]      single-attribute counts of the target
 *   tau[j]        co-occurrence threshold (cnt > tau[j]), RepairApi.scala:572-576
 *   out_top1      device int32[n_cells]      candidate with the highest probability among those
 *                                            with prob > beta, -1 if none (ties: lowest code)
 *   out_prob      device double[n_cells]     its probability (0 if none)
 *   out_weak      device uint8[n_cells]      1 iff the cell's current code == out_top1 (the cell is
 *                                            weak-labelled clean), else 0 */
int dr_domain_score(dr_ctx* ctx, const int32_t* rows, int64_t n_cells, const int32_t* target, int32_t dom_t,
                    const int32_t* const* corr, const int32_t* dom_c, const int64_t* const* cooc, int n_corr,
                    const int64_t* hist_t, const int64_t* tau, int64_t n_total_rows, double beta,
                    int32_t* out_top1, double* out_prob, uint8_t* out_weak, void* stream);

/* The same analysis for ALL targets of a pass in three launches, applied to the error bitmaps in place:
 * a cell's verdict only depends on its correlated values, so the top-1 candidate is computed once per
 * combination of correlated values (the per-cell loop of dr_domain_score, identical doubles) and the pass
 * over the cells is a table look-up driven by the bitmap -- bits of cells whose current value is their
 * top-1 candidate are cleared (errors.py:507-530); removed[i] (device int64, accumulated) counts them.
 * DR_ERR_UNSUPPORTED when a target has more than 2^20 combinations (use dr_domain_score).  Synchronises
 * `stream`. */
typedef struct dr_domain_target {
    const int32_t* target;    /* device int32[n_rows]: discretised target column */
    uint32_t* bitmap;         /* device: error cells of the target, updated in place */
    const int64_t* hist_t;    /* device int64[dom_t + 1], HAVING applied */
    int32_t dom_t;
    int32_t n_corr;           /* 1 .. 8 */
    const int32_t* corr[8];   /* device columns of the correlated attributes */
    const int64_t* cooc[8];   /* device int64[(dom_c + 1) * (dom_t + 1)], HAVING applied */
    int64_t tau[8];
    int32_t dom_c[8];
} dr_domain_target;
int dr_domain_prune(dr_ctx* ctx, const dr_domain_target* targets, int n_targets, int64_t n_rows,
                    int64_t n_total_rows, double beta, int64_t* removed, void* stream);

/* ---- a10: repair base = error cells masked to NULL, restricted to the rows that matter ---------
 * Replaces RepairApi.convertErrorCellsToNull (RepairApi.scala:171-211) and the dirty/clean split
 * (model.py:550-555) without materialising the N x K masked table: gathers the given rows into a
 * ROW-MAJOR int32[n][n_cols] tile, writing -1 where bitmaps[c] has the row's bit set
 * (bitmaps[c] may be NULL = column is not a target).  Also used to pull training samples. */
int dr_gather_rows_masked(dr_ctx* ctx, const int32_t* const* cols, uint32_t* const* bitmaps, int n_cols,
                          const int32_t* rows, int64_t n, int32_t* out, void* stream);
/* Same for float64 side arrays of continuous attributes (NaN where masked). */
/* Same, and on the way: null_out[c * null_words_per_col + w] bit i = (out[32 * w + i][c] < 0), the NULL
 * bitmap of every tile column (what dr_tile_null_bitmaps computes with a second pass over the tile). */
int dr_gather_rows_masked_nulls(dr_ctx* ctx, const int32_t* const* cols, uint32_t* const* bitmaps, int n_cols,
                                const int32_t* rows, int64_t n, int32_t* out, uint32_t* null_out,
                                int64_t null_words_per_col, void* stream);
int dr_gather_rows_masked_f64(dr_ctx* ctx, const double* const* cols, uint32_t* const* bitmaps, int n_cols,
                              const int32_t* rows, int64_t n, double* out, void* stream);
/* out bit i = (tile[i][col] < 0): the cells model `col` has to fill (model.py:1128-1133). */
int dr_tile_null_bitmap(dr_ctx* ctx, const int32_t* tile, int64_t n, int n_cols, int col, uint32_t* out,
                        void* stream);
int dr_tile_null_bitmap_f64(dr_ctx* ctx, const double* tile, int64_t n, int n_cols, int col, uint32_t* out,
                            void* stream);
/* All columns at once: out[c * words_per_col + w] (one coalesced pass over the tile; a model only
 * ever fills its own column, so the bitmaps taken before the chain stay valid for every target). */
int dr_tile_null_bitmaps(dr_ctx* ctx, const int32_t* tile, int64_t n, int n_cols, int64_t words_per_col,
                         uint32_t* out, void* stream);
/* out[i] = col[rows[i]]  (current values of error cells, RepairApi.withCurrentValues :69-104). */
int dr_gather_i32(dr_ctx* ctx, const int32_t* col, const int32_t* rows, int64_t n, int32_t* out, void* stream);
int dr_gather_f64(dr_ctx* ctx, const double* col, const int32_t* rows, int64_t n, double* out, void* stream);
/* out[i] = tile[drows[i]][col]  (repaired values read back from the dirty-row tile). */
int dr_tile_gather_i32(dr_ctx* ctx, const int32_t* tile, int n_cols, int col, const int32_t* drows, int64_t n,
                       int32_t* out, void* stream);
int dr_tile_gather_f64(dr_ctx* ctx, const double* tile, int n_cols, int col, const int32_t* drows, int64_t n,
                       double* out, void* stream);
/* a14 filter on codes: out bit i = repaired[i] < 0 (NULL) || repaired[i] != current[i], i.e. the
 * reference's `repaired IS NULL OR NOT(current_value <=> repaired)` (model.py:1401). */
int dr_changed_bitmap(dr_ctx* ctx, const int32_t* current, const int32_t* repaired, int64_t n, uint32_t* out,
                      void* stream);
/* out[i] = position of keys[i] in the ascending array sorted[n_sorted] (binary search), -1 if
 * absent: maps an error cell's row to its dirty-tile row. */
int dr_lookup_sorted(dr_ctx* ctx, const int32_t* sorted, int64_t n_sorted, const int32_t* keys, int64_t n,
                     int32_t* out, void* stream);

/* ---- a13: repair-model inference ---------------------------------------------------------------
 * Replaces the `repair` pandas UDF (model.py:1095-1135): transformer.transform + model.predict
 * + fill-NULL-only, for ONE target attribute over the dirty-row tile, in place.
 *
 * Forest (device arrays, caller-owned; layout in DESIGN.md "flat forest"):
 *   n_seq sequences (1 = regression or binary, C = multiclass), trees grouped by sequence:
 *   seq_tree_off int32[n_seq+1]; tree_node_off int32[n_trees+1];
 *   node_thr double[n_nodes] (threshold, or leaf value on leaves); node_meta uint32[n_nodes]:
 *     bits 0..11  feature index, 0xFFF = leaf
 *     bit  12     NaN goes left
 *     bits 13..21 left child, bits 22..30 right child (node index relative to the tree root)
 *   baseline double[n_seq].
 * Features: encoded feature f of a row = enc_lut[f][ tile[row][feat_col[f]] + 1 ] when
 *   feat_col[f] >= 0 refers to a discrete tile column (enc_lut_off int32[n_feat+1] into the
 *   double LUT; entry 0 = NULL), or ctile[row][-feat_col[f]-1] for continuous columns
 *   (passthrough, NaN = NULL).
 * Margin of sequence s = baseline[s] + sum of its trees' leaves in tree order (sequential float64
 * adds: bit-identical to the oracle).  Output per cell i (tile row cells[i]):
 *   kind 0 (classifier)  code = class_code[argmax_s margin] (binary: margin > 0 ? class 1 : 0),
 *                        ties -> lowest s; written to tile[row][target_col]
 *   kind 1 (regressor)   value (rounded half-to-even like numpy.round when `integral`) written
 *                        to ctile[row][target_ccol]
 * out_margin (optional, device double[n_cells * n_seq]) receives the margins (pmf modes). */
typedef struct dr_forest {
    int32_t n_seq, n_trees, n_nodes, n_feat;
    const int32_t* seq_tree_off;
    const int32_t* tree_node_off;
    const double* node_thr;
    const uint32_t* node_meta;
    const double* baseline;
    const int32_t* feat_col;
    const int32_t* enc_lut_off;
    const double* enc_lut;
    const int32_t* class_code; /* int32[n_classes], kind 0 only */
    int32_t kind, integral, n_classes;
} dr_forest;
int dr_forest_predict(dr_ctx* ctx, const dr_forest* forest, int32_t* tile, int n_cols, double* ctile, int n_ccols,
                      const int32_t* cells, int64_t n_cells, int target_col, double* out_margin, void* stream);
/* Rank-coded variant for all-discrete models (the common case: every feature is a label-encoded
 * attribute).  An encoded feature then takes only a handful of distinct values, so the host replaces
 * every value by its RANK among the feature's sorted distinct values and every threshold by the
 * number of values <= threshold: `x <= thr` becomes `rank < thr_rank` -- same decisions, but a node is
 * ONE 32-bit word and a cell's feature vector is one byte per rank slot, which is what lets 16 warps
 * per SM stay resident.  Leaf values stay float64 and are summed in tree order, so margins remain
 * bit-identical to dr_forest_predict / the oracle.
 *   rank slot: one (encoded feature, NaN direction) combination that some node tests.  Slot s of a
 *              row = rank_lut[rank_lut_off[s] + tile[row][slot_col[s]] + 1] when the code lies inside
 *              the slot's LUT, else slot_nan[s]; LUT entries are rank + 1 (1..254) with NaN already
 *              folded to 0 (the slot's nodes send NaN left) or 255 (right).  At most 255 slots.
 *   node word: bits 24-31 = rank slot, bits 8-23 = index of the LEFT child in the chunk's node array
 *              (the right child is the next word: siblings are adjacent), bits 0-7 = 256 -
 *              (thr_rank + 1).  Adding the row's rank byte to the word carries into the child field
 *              exactly when rank >= thr_rank + 1, i.e. when the row goes right: a level is load rank,
 *              add, load word[bits 8-23].  A LEAF is (own index << 8): slot 0, never carries, the
 *              walk stays put -- every tree is walked max_depth levels without a branch.
 *   leaf values: the LAST level only computes the index c of the node the walk ends on (no load of
 *              that node's word); its value is slot chunk_leaf_off[chunk] + bias + c of the leaf table, where
 *              bias (signed) is the second header word of the tree.  The table is stored as 32-bit words,
 *              chunk by chunk: chunk c with L = chunk_leaf_off[c+1] - chunk_leaf_off[c] slots occupies
 *              leaf_value[2 * chunk_leaf_off[c] ..): the L low words of its float64 values, then the L high
 *              words (two conflict-free 32-bit shared-memory loads instead of one 64-bit load).  The host orders the nodes of a
 *              tree so that all leaves sit in its tail and stores values for that tail only.
 *   max_depth: deepest leaf of any tree.
 *   Forest chunks are streamed into shared memory by the TMA engine (cp.async.bulk, double buffered).
 *   The host supplies the chunk table: chunk c = trees [chunk_tree_off[c], chunk_tree_off[c+1]) of
 *   sequence chunk_seq[c] (never straddling a sequence; every sequence has at least one tree), at
 *   most DR_RANKED_CHUNK_TREES trees, DR_RANKED_CHUNK_NODES node words and DR_RANKED_CHUNK_LEAVES leaf
 *   values; its words are node_word[chunk_node_off[c] .. chunk_node_off[c+1]), its leaf values
 *   the leaf planes described above, its tree headers tree_hdr[2 * chunk_hdr_off[c] ..): two words
 *   per tree = (root node word, value bias).  chunk_node_off and chunk_leaf_off are multiples of 4,
 *   chunk_hdr_off a multiple of 2 (16-byte TMA granules). */
#define DR_RANKED_CHUNK_NODES 4096
#define DR_RANKED_CHUNK_LEAVES 2560
#define DR_RANKED_CHUNK_TREES 256
typedef struct dr_forest_ranked {
    int32_t n_seq, n_trees, n_nodes, n_leaves, n_slots, max_depth, n_chunks;
    int32_t layout;          /* shared-memory rank tile: 0 = choose, 1 = bytes, 2 / 3 = one word per rank
                                with 8 / 16 trees in flight per thread (DR_ERR_UNSUPPORTED if it does not fit) */
    const int32_t* chunk_tree_off;
    const int32_t* chunk_seq;
    const int32_t* chunk_node_off;
    const int32_t* chunk_leaf_off;
    const int32_t* chunk_hdr_off;
    const uint32_t* tree_hdr;
    const uint32_t* node_word;
    const uint32_t* leaf_value;   /* float64 leaf values, per chunk: low words of its leaves, then high words */
    const double* baseline;
    const int32_t* slot_col;      /* int32[n_slots]: tile column the slot reads */
    const int32_t* rank_lut_off;  /* int32[n_slots + 1] */
    const uint8_t* rank_lut;
    const uint8_t* slot_nan;      /* uint8[n_slots]: rank byte of a code outside the slot's LUT */
    const int32_t* class_code;
    int32_t n_classes;
} dr_forest_ranked;
int dr_forest_predict_ranked(dr_ctx* ctx, const dr_forest_ranked* forest, int32_t* tile, int n_cols,
                             const int32_t* cells, int64_t n_cells, int target_col, double* out_margin,
                             void* stream);
/* ---- a12 ("next" #1): repair-model training ------------------------------------------------------
 * Replaces train.build_model (train.py:89-234: LightGBM under a hyperopt search) with a histogram
 * GBDT trained on the GPU with the reference's fixed parameters (train.py:102-115; LightGBM defaults
 * for the rest).  The algorithm is specified in oracle/gbdt.py and reproduced bit for bit: integer
 * (quantised-gradient) histograms, explicit round-to-nearest arithmetic, level-wise growth under a
 * num_leaves budget, all class sequences of a boosting round grown together, no host
 * synchronisation inside the boosting loop.
 *   bins      device uint8[n_rows][n_features]: value bins 0..n_bins[f]-2, missing = n_bins[f]-1
 *   n_bins    host int32[n_features]  (sum of bins * 12 bytes must fit in shared memory)
 *   qscale    gradient quantisation scale; the caller chooses it so that n_rows * max|g| * qscale < 2^31
 *             (oracle/gbdt.py: 2^min(24, 30 - ceil(log2 n)) / max weight)
 *   y_class   device int32[n_rows] (n_classes >= 2) / y_value device double[n_rows] (n_classes == 1)
 *   weight    device double[n_rows] (class weights; classification only)
 *   init      host double[S] initial scores, S = 1 for regression / binary, n_classes otherwise
 *   workspace device scratch of dr_gbdt_workspace_bytes(n_rows, S) bytes
 *   out_nodes device dr_gbdt_node[n_iter][S][64], out_counts device int32[n_iter][S] (nodes used) */
typedef struct dr_gbdt_params {
    int32_t n_rows, n_features, n_classes, n_iter, max_depth, num_leaves, min_data_in_leaf;
    double learning_rate, min_sum_hessian, qscale;
    /* the remaining parameters of the reference's search space (train.py:148-156); defaults 0 / 1 / 1 / 0:
     * reg_lambda is added to every hessian sum (gain and leaf value); feature f takes part in tree
     * (iteration, sequence) iff hash(seed, iteration, sequence, f) < colsample_bytree (the feature with
     * the smallest hash always does); every subsample_freq iterations row i is (re)drawn into the bag iff
     * hash(seed, bag, i) < subsample -- oracle/gbdt.py states the hashes */
    double reg_lambda, colsample_bytree, subsample;
    int32_t subsample_freq, seed;
} dr_gbdt_params;
typedef struct dr_gbdt_node {
    int16_t feature; /* -1 = leaf */
    uint8_t thr_bin, missing_left, left, right, pad[2];
    double value; /* leaf value (already scaled by the learning rate) */
} dr_gbdt_node;
int64_t dr_gbdt_workspace_bytes(int32_t n_rows, int32_t n_seq);
int dr_gbdt_train(dr_ctx* ctx, const dr_gbdt_params* params, const uint8_t* bins, const int32_t* n_bins,
                  const int32_t* y_class, const double* y_value, const double* weight, const double* init,
                  void* workspace, int64_t workspace_bytes, dr_gbdt_node* out_nodes, int32_t* out_counts,
                  void* stream);

/* ---- 8f #4: rule-based repairs -----------------------------------------------------------------
 * dr_scatter_*: col[rows[i]] = vals[i] -- repairs decided by a rule join the repair base
 *   (RepairModel._repair_attrs, model.py:1250-1257 -> RepairMiscApi.repairAttrsFrom :184-247).
 * dr_fd_map_build: the map behind FunctionalDepModel (model.py:64-100), replacing
 *   DepGraph.computeFunctionalDepMap (DepGraph.scala:300-316: GROUP BY x HAVING size(collect_set(y)) = 1).
 *   For every row whose x and y are non-NULL and not masked (x_mask / y_mask: error-cell bitmaps, may be
 *   NULL): lo[x] = min(lo[x], y), hi[x] = max(hi[x], y); lo/hi are device int32[dom_x], caller
 *   initialises lo = INT32_MAX, hi = INT32_MIN.  x determines y iff lo[x] == hi[x]; both reductions are
 *   idempotent, so per-GPU tables combine with one MIN / MAX all-reduce.
 * dr_tile_lut_fill: FunctionalDepModel.predict on the dirty-row tile:
 *   tile[cells[i]][y_col] = lut[tile[cells[i]][x_col] + 1]  (lut[0] = what a NULL x maps to, -1 = NULL). */
int dr_scatter_i32(dr_ctx* ctx, int32_t* col, const int32_t* rows, const int32_t* vals, int64_t n, void* stream);
int dr_scatter_f64(dr_ctx* ctx, double* col, const int32_t* rows, const double* vals, int64_t n, void* stream);
int dr_fd_map_build(dr_ctx* ctx, const int32_t* x_col, const uint32_t* x_mask, const int32_t* y_col,
                    const uint32_t* y_mask, int64_t n_rows, int32_t dom_x, int32_t* lo, int32_t* hi, void* stream);
int dr_tile_lut_fill(dr_ctx* ctx, int32_t* tile, int n_cols, int x_col, int y_col, const int32_t* cells,
                     int64_t n_cells, const int32_t* lut, int32_t lut_size, void* stream);

/* ---- LOFOutlierErrorDetector: exact one-dimensional local outlier factor ---------------------------
 * Replaces LOFOutlierErrorDetector (errors.py:302-312: sklearn LocalOutlierFactor per column).
 *   col        device double[n], the whole column (NaN = NULL); when the table is sharded, the gathered
 *              global column
 *   k          neighbours, 1 <= k <= min(64, n - 1) (the detector uses min(20, n - 1))
 *   bitmap     device uint32 words; only rows in [row_begin, row_begin + row_count) set bits, at bit
 *              (row - row_begin); flagged iff lof > 1.5
 *   out_lof    device double[n] (nullable): scores in row order; NaN when nothing was scored
 *              (n < 2 or an all-NULL column)
 *   out_flagged host int64 (nullable): number of rows flagged inside the range; non-NULL synchronises
 *   workspace  device scratch of dr_lof_workspace_bytes(n) bytes (no allocation inside the call)
 * Definition: NULL -> median of the non-NULL values (np.median), -0.0 -> +0.0; stable sort by
 * (value, row); for sorted position i, the leftmost window [l, l + k] around i minimising
 * max(s[i] - s[l], s[l + k] - s[i]) gives kdist and the neighbours; then scikit-learn's lrd / lof with
 * the sums in ascending sorted position and round-to-nearest double arithmetic. */
int64_t dr_lof_workspace_bytes(int64_t n);
int dr_lof_flag(dr_ctx* ctx, const double* col, int64_t n, int k, int64_t row_begin, int64_t row_count,
                uint32_t* bitmap, double* out_lof, int64_t* out_flagged, void* workspace, int64_t workspace_bytes,
                void* stream);

/* PoorModel (model.py:44-61): constant fill of the listed tile rows. */
int dr_tile_fill_i32(dr_ctx* ctx, int32_t* tile, int n_cols, int col, const int32_t* cells, int64_t n_cells,
                     int32_t value, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200REPAIR_H */
