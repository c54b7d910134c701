/*
 * nvtb200.h — C-ABI of libnvtb200.so, the B200 (sm_100a) engine behind the
 * nvtabular.ops operator API for the Categorify / Normalize / FillMissing /
 * HashBucket / JoinGroupby / TargetEncoding hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference has no FFI on
 * this path: its operators call cuDF / pandas through merlin.core.dispatch
 * (reference nvtabular/dispatch.py:21).  Each entry point below replaces the
 * dataframe-library call(s) the reference makes at the cited file:line; the
 * Python operator classes in nvtabular_b200/ops bind these with ctypes
 * (see INTEGRATION.md for the binding a reference maintainer would add).
 *
 * Conventions
 *   - every function returns 0 on success or a negative nvtb_status_t;
 *     nvtb_last_error() gives a thread-local message.  No C++ exception ever
 *     crosses this boundary.
 *   - all data pointers are DEVICE pointers owned by the caller unless the
 *     parameter name ends in `_host`.
 *   - `stream` is a cudaStream_t passed as void*.  All kernels are stream
 *     ordered; only the functions documented as "synchronises" block the host.
 *   - a column is (data, validity, dtype).  `validity` is an Arrow-style
 *     bitmask: bit (i & 7) of byte (i >> 3) is 1 when row i is non-null;
 *     NULL means "no nulls".  Data pointers should be 32-byte aligned for
 *     the vectorised (256-bit) path; a scalar path is taken otherwise.
 *   - handles (nvtb_hashagg_t, nvtb_vocab_t, nvtb_groupstats_t) are created
 *     and destroyed explicitly; build-phase calls on one handle must not be
 *     issued concurrently; finalised vocab / groupstats handles are immutable
 *     and may be probed from any number of streams.
 *   - ONE device per process (the one-process-per-GPU model of SURVEY §8e): the
 *     hashagg build phase keeps grow-only scratch (two accumulator arenas, the
 *     partition buffer, the sort / bucket scratch) in process-global pools on the device
 *     that was current at the first call.  The pools are mutex-guarded and a use
 *     on another stream waits on an event of the previous one, so build calls
 *     of DIFFERENT handles may come from different streams of that device; a
 *     second device in the same process is not supported and not detected.
 */
#ifndef NVTB200_H
#define NVTB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  NVTB_OK = 0,
  NVTB_EINVAL = -1,  /* bad argument (dtype, null pointer, size)          */
  NVTB_ENOMEM = -2,  /* device allocation failed                          */
  NVTB_ECUDA = -3,   /* a CUDA runtime call or kernel launch failed       */
  NVTB_ESTATE = -4,  /* handle used in the wrong phase                    */
  NVTB_ENCCL = -5    /* an NCCL call failed / NCCL is not loadable         */
} nvtb_status_t;

typedef enum {
  NVTB_I32 = 0,
  NVTB_I64 = 1,
  NVTB_F32 = 2,
  NVTB_F64 = 3,
  NVTB_U8 = 4,  /* bool / fold ids */
  NVTB_H64 = 5  /* hash columns only: a precomputed 64-bit value hash (e.g. the
                   pandas string hash of a dictionary entry), used as-is   */
} nvtb_dtype_t;

typedef struct {
  const void* data;        /* device, n elements of `dtype`               */
  const uint8_t* validity; /* device bitmask or NULL                      */
  int32_t dtype;           /* nvtb_dtype_t                                */
  int32_t _pad;
} nvtb_col_t;

/* library identity ------------------------------------------------------- */
int nvtb_version(void);              /* 1000*major + minor                 */
const char* nvtb_last_error(void);   /* thread-local, never NULL           */
int nvtb_device_sm_count(int* out_host); /* SMs of the current device      */

/* ---- Normalize / NormalizeMinMax statistics ---------------------------
 * Replaces _chunkwise_moments (reference nvtabular/ops/moments.py:64-77:
 * count(), sum(), astype(f64).pow(2).sum() — three cuDF reductions per
 * column) and ddf.min()/ddf.max() (reference nvtabular/ops/normalize.py:
 * 166-170) with ONE fused scan over all columns.  FillMissing upstream
 * (reference nvtabular/ops/fill.py:49-57) is fused: when fill_vals_host[c]
 * is not NaN, null rows count as that value instead of being skipped.
 *
 * acc: device double[ncols * 5] = {count, sum, sumsq, min, max} per column.
 * The call ADDS this batch into acc (min/max: combines), so batches and the
 * tree reduction of moments.py:80-86 become repeated calls.  Initialise with
 * nvtb_moments_init.  Deterministic: fixed grid + ordered final reduction.
 */
int nvtb_moments_init(double* acc, int ncols, void* stream);
int nvtb_moments_accumulate(const nvtb_col_t* cols_host, int ncols, int64_t n,
                            const double* fill_vals_host, double* acc,
                            void* stream);
/* _finalize_moments (reference nvtabular/ops/moments.py:89-116), host math:
 * mean = sum/n; var = (sumsq - sum^2/n) / max(n-1,1), NaN when n-1 == 0;
 * std = sqrt(var).  acc_host is a HOST copy of acc.  out_host: double
 * [ncols*3] = {mean, var, std}. */
int nvtb_moments_finalize(const double* acc_host, int ncols, double* out_host);

/* ---- FillMissing / Normalize transforms --------------------------------
 * nvtb_fill_apply: FillMissing.transform (reference nvtabular/ops/fill.py:
 * 49-57, C++ twin cpp/nvtabular/inference/fill.cc:91-102): out = valid ? x :
 * (T)fill, dtype preserved; filled_out[c] (may be NULL) receives the
 * `<col>_filled` indicator as uint8 0/1.
 *
 * nvtb_normalize_apply: Normalize.transform (reference nvtabular/ops/
 * normalize.py:71-90) fused with an upstream FillMissing:
 * y = std>0 ? (x-mean)/std : (x-mean); float32 inputs are computed in float32
 * exactly like numpy does, everything else in float64; out_dtype F32|F64.
 * With fill NaN, null rows produce NaN (nulls propagate).
 *
 * nvtb_minmax_apply: NormalizeMinMax.transform (normalize.py:150-161):
 * (x-min)/(max-min) when max>min, x/(2x) when max==min.
 */
int nvtb_fill_apply(const nvtb_col_t* cols_host, int ncols, int64_t n,
                    const double* fill_vals_host, void* const* out_host,
                    uint8_t* const* filled_out_host, void* stream);
int nvtb_normalize_apply(const nvtb_col_t* cols_host, int ncols, int64_t n,
                         const double* fill_vals_host,
                         const double* means_host, const double* stds_host,
                         void* const* out_host, int out_dtype, void* stream);
int nvtb_minmax_apply(const nvtb_col_t* cols_host, int ncols, int64_t n,
                      const double* fill_vals_host, const double* mins_host,
                      const double* maxs_host, void* const* out_host,
                      int out_dtype, void* stream);

/* Clip (reference nvtabular/ops/clip.py:46-53) and Clip + LogOp (ops/logop.py:47-56) in one
 * pass, with an upstream FillMissing fused in (fill_vals[c] NaN = none): x = fill if null;
 * x = max(x, min_vals[c]); x = min(x, max_vals[c]) (NaN bound / NULL array = none);
 * take_log == 0: out[c] has the column's own dtype; take_log != 0: out[c] (out_dtype float32 |
 * float64) = log(x cast to out_dtype + 1).  Rows that stay null are written as 0 / NaN. */
int nvtb_cliplog_apply(const nvtb_col_t* cols, int ncols, int64_t n,
                       const double* fill_vals, const double* min_vals,
                       const double* max_vals, int take_log, void* const* out,
                       int out_dtype, void* stream);

/* ---- HashBucket ---------------------------------------------------------
 * dispatch.hash_series(col) % nb  (reference nvtabular/ops/hash_bucket.py:
 * 86-100, nvtabular/ops/categorify.py:1837-1852).  The hash is the value-only
 * pandas hash (pandas/core/util/hashing.py::_hash_ndarray): bits of the value
 * zero-extended to u64 by itemsize, then the splitmix64 finaliser.  ncols > 1
 * XORs the per-column hashes first (encode_type="combo", categorify.py:
 * 1847-1851; HashedCross).  out[i] = (int32)(h % nb) + add.  Null rows hash
 * the float64 NaN pattern (what the pandas path sees for a null).
 */
int nvtb_hash_bucket_apply(const nvtb_col_t* cols_host, int ncols, int64_t n,
                           uint64_t num_buckets, int64_t add, void* out,
                           int out_dtype, void* stream);
/* raw 64-bit hashes (testing / host-side composition) */
int nvtb_hash_values(const nvtb_col_t* col_host, int64_t n, uint64_t* out,
                     void* stream);

/* ---- hash aggregation: groupby(key, dropna=False).agg(size[,sum,...]) ----
 * Replaces _top_level_groupby / _mid_level_groupby / _bottom_level_groupby
 * (reference nvtabular/ops/categorify.py:955-1137): cuDF hash-groupby per
 * partition + tree of concat+groupby.  One handle per column group holds an
 * open-addressing device table {key:int64, size:int64 [, per cont col: sum,
 * sumsq, min, max : double]} that every batch is inserted into (block-level
 * shared-memory pre-aggregation, then global atomics).  The null key
 * (dropna=False) is kept out of the table in a dedicated group.
 *
 *   size  = rows in the group                       (agg "size", Categorify)
 *   count : the reference attaches agg "count" to the FIRST KEY column
 *           (categorify.py:989-999), so count == size when that key component
 *           is non-null and 0 otherwise — derived by the caller from the key,
 *           not stored.
 *   per cont column: sum / sumsq over non-null values, min, max
 *           (NaN when the group has no non-null value).
 *
 * n_agg = number of continuous columns (0 for Categorify).  capacity_hint =
 * expected number of distinct keys (0 = unknown: the first 2^20 rows are
 * inserted on their own and their exact distinct count sizes the table).
 * The hint only affects speed; results never depend on it.
 * key dtype I32 or I64 (multi-column keys are packed to I64 with
 * nvtb_pack_keys2 first).
 */
typedef struct nvtb_hashagg nvtb_hashagg_t;
int nvtb_hashagg_create(nvtb_hashagg_t** out, int n_agg,
                        int64_t capacity_hint);
int nvtb_hashagg_destroy(nvtb_hashagg_t* h);
/* empty the table but keep its capacity and cardinality estimate (a second fit
 * over similar data then needs neither growth nor the sampling pass) */
int nvtb_hashagg_reset(nvtb_hashagg_t* h, void* stream);
/* insert one batch of raw rows; agg_cols_host may be NULL when n_agg == 0.
 * int32 keys without payload are folded in SHARED memory (one kernel), after a
 * one-pass hash partition of the column (three more kernels) when the expected
 * number of distinct keys exceeds what one SM's shared memory holds
 * (csrc/fold_i32.cuh); other keys take one kernel that updates the table directly.  Waits for the handle's PREVIOUS launch (its counters are
 * read back), never for the one it enqueues. */
int nvtb_hashagg_insert(nvtb_hashagg_t* h, const nvtb_col_t* key_host,
                        const nvtb_col_t* agg_cols_host, int64_t n,
                        void* stream);
/* merge pre-aggregated partials (the cross-GPU unique-merge and the
 * _mid_level_groupby concat+groupby, categorify.py:1054-1070).  vals layout:
 * double[n * 4 * n_agg] row-major {sum,sumsq,min,max} per cont col, or NULL. */
int nvtb_hashagg_merge(nvtb_hashagg_t* h, const int64_t* keys,
                       const int64_t* sizes, const double* vals, int64_t n,
                       void* stream);
int nvtb_hashagg_add_null_group(nvtb_hashagg_t* h, int64_t size,
                                const double* vals_host);
/* synchronises; number of distinct non-null keys, and the null group's size */
int nvtb_hashagg_size(nvtb_hashagg_t* h, int64_t* n_unique_host,
                      int64_t* null_size_host, void* stream);
/* compact the table into caller arrays of length n_unique (unordered).
 * vals_out may be NULL when n_agg == 0.  null_vals_host: host double
 * [4*n_agg] for the null group, may be NULL. */
int nvtb_hashagg_export(nvtb_hashagg_t* h, int64_t* keys_out,
                        int64_t* sizes_out, double* vals_out,
                        double* null_vals_host, void* stream);

/* 0 = resident hash table, 1 = sorted accumulator.  int32 key columns whose expected number
 * of distinct keys exceeds NVTB_RUNS_MIN_KEYS (default 2^23: the table would leave the L2)
 * are accumulated as a key-ordered array of packed (key, count) pairs: every batch is
 * radix-sorted, run-length encoded and merged in (csrc/sortagg.cuh) — the streaming
 * replacement of the per-partition groupby + concat/groupby tree of reference
 * nvtabular/ops/categorify.py:955-1137 for the C20/C1/C22/C10 class of Criteo columns. */
int nvtb_hashagg_mode(nvtb_hashagg_t* h, int* mode_host);
/* A sorted accumulator only COPIES a batch (keys + validity bytes) into its staging buffer; the
 * sort + run-length encode + merge of everything staged runs when NVTB_STAGE_ROWS rows (default
 * 2^28) are waiting, when the handle is read (size / export / vocabulary build), or here. */
int nvtb_hashagg_flush(nvtb_hashagg_t* h, void* stream);

/* ---- sorted-pair primitives of the cross-GPU vocabulary merge (SURVEY.md 8e) --------------
 * A high-cardinality column is exchanged between GPUs as key-ordered packed pairs
 * word = (uint32)(key ^ 2^31) << 32 | (uint32)count (unsigned order of the word == key order),
 * split by KEY RANGE (the local accumulator is already grouped by owner: no partition pass),
 * merged by the owner, ordered by count on the owner, and the owners' count-ordered shards
 * are interleaved into the global (count desc, key asc) order group by group.  Replaces the
 * dask tree + shared-filesystem hop of reference nvtabular/ops/categorify.py:1036-1049,
 * 1399-1540.  The collectives themselves are issued by the host (torch.distributed / NCCL). */
/* make the handle a sorted accumulator (no-op if it is one); NVTB_ESTATE when the handle holds
 * int64 keys, payload columns or >= 2^32 rows */
int nvtb_hashagg_to_sorted(nvtb_hashagg_t* h, void* stream);
/* copy the packed pairs of a sorted accumulator (key order) to `out` (may be NULL: size query) */
int nvtb_hashagg_export_packed(nvtb_hashagg_t* h, uint64_t* out, int64_t* n_host, void* stream);
/* out_dev[j] = number of pairs whose unsigned key is < bounds_dev[j]  (the split points of the
 * key-range exchange) */
int nvtb_pairs_lower_bounds(const uint64_t* pairs, int64_t n, const uint32_t* bounds_dev, int m,
                            int64_t* out_dev, void* stream);
/* merge two key-sorted, key-unique pair arrays adding the counts of equal keys (the owner-side
 * _mid_level_groupby, categorify.py:1054-1070); out holds na + nb pairs; synchronises */
int nvtb_pairs_merge(const uint64_t* a, int64_t na, const uint64_t* b, int64_t nb, uint64_t* out,
                     int64_t* n_out_host, void* stream);
/* copy nseg contiguous segments [seg_src[s], seg_src[s+1]) of src to dst + seg_dst[s] */
int nvtb_segment_copy_u64(const uint64_t* src, uint64_t* dst, const int64_t* seg_src_dev,
                          const int64_t* seg_dst_dev, int nseg, int64_t n, void* stream);

/* Stable LSD radix sort of device arrays by bits [lo_bit, hi_bit) of every element
 * (csrc/radix.cuh; ascending, or descending on that bit field).  data/tmp: n elements
 * each, 16-byte aligned; the result ends in data (*result_in_tmp_host = 0) or tmp (= 1).
 * This is the ordering primitive behind sort_values in reference
 * nvtabular/ops/categorify.py:1300,1316. */
int nvtb_radix_sort_u32(uint32_t* data, uint32_t* tmp, int64_t n, int lo_bit, int hi_bit,
                        int descending, int* result_in_tmp_host, void* stream);
int nvtb_radix_sort_u64(uint64_t* data, uint64_t* tmp, int64_t n, int lo_bit, int hi_bit,
                        int descending, int* result_in_tmp_host, void* stream);

/* owner = mix(key) % n_parts for the key-hash sharding across GPUs
 * (SURVEY.md §8e; the reference's split_out shuffle_group,
 * categorify.py:1036-1049).  perm_out receives a permutation that groups
 * rows by owner; part_counts_host the rows per owner.  Synchronises. */
int nvtb_partition_by_owner(const int64_t* keys, int64_t n, int n_parts,
                            int64_t* perm_out, int64_t* part_counts_host,
                            void* stream);
/* same grouping without a host round trip: the per-owner row counts stay on the
 * device (part_counts_dev, int64[n_parts]); nothing synchronises, so the 26
 * columns of a Categorify fit are partitioned back to back and their counts read
 * with ONE copy (nvtabular_b200/dist.py global_merge_many). */
int nvtb_partition_by_owner_async(const int64_t* keys, int64_t n, int n_parts,
                                  int64_t* perm_out, int64_t* part_counts_dev, void* stream);
int nvtb_gather_i64(const int64_t* src, const int64_t* perm, int64_t n,
                    int64_t* dst, void* stream);
int nvtb_gather_f64_rows(const double* src, const int64_t* perm, int64_t n,
                         int row_width, double* dst, void* stream);

/* pack two key columns into one order-preserving int64 key:
 * (a << 32) | (b ^ 0x80000000), both I32.  Rows where BOTH are null become
 * null (validity_out bit cleared); a single null becomes INT32_MIN so the
 * tuple sorts first (categorify.py:1689-1692 all-null rule; KAT
 * tests/unit/ops/test_categorify.py:288-297). */
int nvtb_pack_keys2(const nvtb_col_t* a_host, const nvtb_col_t* b_host,
                    int64_t n, int64_t* keys_out, uint8_t* validity_out,
                    void* stream);

/* ---- vocabulary: ordering, cut, lookup table, encode ----------------------
 * nvtb_vocab_build replaces _write_uniques + _save_encodings (reference
 * nvtabular/ops/categorify.py:1149-1337, 719-822): order the (key,size) rows
 * by (size desc, key asc), apply freq_threshold (keep size >= t) or max_size
 * (keep the first max_size - (num_buckets or 1) - 2), and build the
 * key -> position lookup used by the encode.  keys/sizes are device arrays of
 * length n (unordered, distinct keys, null group NOT included).
 *
 * nvtb_vocab_from_arrays: keys already in label order (user `vocabs=`,
 * categorify.py:421-454, or a unique.<col>.parquet read back); sizes may be
 * NULL.
 */
typedef struct nvtb_vocab nvtb_vocab_t;
typedef struct {
  int64_t n_kept;      /* rows written to unique.<col>.parquet            */
  int64_t n_total;     /* distinct non-null keys seen                     */
  int64_t null_size;   /* meta num_observed[null]                         */
  int64_t oov_size;    /* meta num_observed[oov]: rows of dropped keys    */
  int64_t unique_size; /* meta num_observed[unique]                       */
} nvtb_vocab_info_t;
/* key_bits: 32 when every key is known to be an int32 value (halves the radix passes),
 * else 0; size_bound: an upper bound on any size (e.g. rows seen), 0 = unknown.
 * Both are speed hints only.  The build is ENQUEUED: n_kept and the meta numbers are read
 * back by the first nvtb_vocab_info / export / encode call on the handle. */
int nvtb_vocab_build(nvtb_vocab_t** out, const int64_t* keys,
                     const int64_t* sizes, int64_t n, int64_t null_size,
                     int64_t freq_threshold, int64_t max_size,
                     int64_t num_buckets, int key_bits, int64_t size_bound,
                     void* stream);
/* the same straight from a group-by handle (single GPU: _write_uniques reads the result of
 * _bottom_level_groupby without leaving the device, categorify.py:1149-1337).  A handle
 * holding a sorted accumulator is already in key order, so the ordering is one stable
 * radix sort on the size bits in use; null_size comes from the handle. */
int nvtb_vocab_build_from_hashagg(nvtb_vocab_t** out, nvtb_hashagg_t* h,
                                  int64_t freq_threshold, int64_t max_size,
                                  int64_t num_buckets, int key_bits, int64_t size_bound,
                                  void* stream);
/* the same from packed pairs that are ALREADY in (count desc, key asc) order (assembled by the
 * cross-GPU merge); the array is copied */
int nvtb_vocab_build_from_pairs(nvtb_vocab_t** out, const uint64_t* ordered_pairs, int64_t n,
                                int64_t null_size, int64_t freq_threshold, int64_t max_size,
                                int64_t num_buckets, void* stream);
int nvtb_vocab_from_arrays(nvtb_vocab_t** out, const int64_t* keys,
                           const int64_t* sizes, int64_t n, void* stream);
int nvtb_vocab_destroy(nvtb_vocab_t* v);
int nvtb_vocab_info(const nvtb_vocab_t* v, nvtb_vocab_info_t* info_host);
/* copy the kept keys / sizes in label order into caller device arrays */
int nvtb_vocab_export(const nvtb_vocab_t* v, int64_t* keys_out,
                      int64_t* sizes_out, void* stream);

/* _encode (reference nvtabular/ops/categorify.py:1558-1807), without the
 * join + sort: label = null_label for null rows; first_label + position for
 * keys in the vocab; otherwise oov_label (+ hash(key) % num_buckets when
 * num_buckets > 1, categorify.py:1709-1715).  For the default layout
 * null_label=1, oov_label=2, first_label=2+(num_buckets or 1); single_table
 * shifts all three (categorify.py:1683-1685).  hash_cols_host: the original
 * column(s) to hash for OOV (NULL = hash `key` itself); out_dtype I32|I64. */
int nvtb_encode_apply(const nvtb_vocab_t* v, const nvtb_col_t* key_host,
                      int64_t n, int64_t null_label, int64_t oov_label,
                      int64_t first_label, uint64_t num_buckets,
                      const nvtb_col_t* hash_cols_host, int n_hash_cols,
                      void* out, int out_dtype, void* stream);

/* ---- group statistics gather: JoinGroupby / TargetEncoding transforms -----
 * Replaces the left-merge + sort_values("__tmp__") of reference
 * nvtabular/ops/join_groupby.py:200-215 and target_encoding.py:357-384.
 * The handle maps key -> row of a caller-provided stats matrix (device,
 * row-major double[n_groups][width]); nvtb_groupstats_gather writes, for
 * column j of the matrix, out[j][i] = stats[row(key_i)][j] cast to
 * out_dtypes[j] (I32|I64|F32|F64), or miss_vals[j] (NaN == null; the global
 * mean for TargetEncoding, target_encoding.py:378-380) when the key is
 * absent. */
typedef struct nvtb_groupstats nvtb_groupstats_t;
/* null_row: row of `stats` that null keys join to (pandas/cuDF merge matches
 * null with null, and dropna=False makes the null key a group), or -1. */
int nvtb_groupstats_create(nvtb_groupstats_t** out, const int64_t* keys,
                           int64_t n_groups, const double* stats, int width,
                           int64_t null_row, void* stream);
int nvtb_groupstats_destroy(nvtb_groupstats_t* g);
int nvtb_groupstats_gather(const nvtb_groupstats_t* g,
                           const nvtb_col_t* key_host, int64_t n,
                           const int* cols_host, int ncols_out,
                           const double* miss_vals_host,
                           void* const* out_host, const int* out_dtypes_host,
                           void* stream);

/* ---- cross-GPU collectives of the fit path (SURVEY.md 8e) ---------------------------------
 * nvtb_comm_t wraps an ncclComm_t: created here (rank 0 makes a unique id, the host runtime
 * hands it to every rank — torch.distributed broadcast, MPI, a file) or provided by the caller.
 * These are all the exchanges the path has: moments all-reduce, variable-block all-to-all of
 * group-by partials, all-gather of vocabulary shards.  They replace the dask tree reduction and
 * the shared-filesystem broadcast of reference nvtabular/ops/categorify.py:1399-1540, 1627-1643
 * and ops/moments.py:34-57.  Stream-ordered; NVTB_ENCCL on failure. */
typedef struct nvtb_comm nvtb_comm_t;
int nvtb_comm_available(void);
int nvtb_comm_unique_id(uint8_t* id_out128);
int nvtb_comm_create(nvtb_comm_t** out, const uint8_t* id128, int rank, int world);
int nvtb_comm_wrap(nvtb_comm_t** out, void* nccl_comm, int rank, int world);
int nvtb_comm_destroy(nvtb_comm_t* c);
int nvtb_comm_rank(const nvtb_comm_t* c, int* rank, int* world);
/* in place; op: 0 sum, 1 min, 2 max */
int nvtb_comm_allreduce_f64(nvtb_comm_t* c, double* buf_dev, int64_t n, int op, void* stream);
int nvtb_comm_allreduce_i64(nvtb_comm_t* c, int64_t* buf_dev, int64_t n, int op, void* stream);
/* acc_dev: [ncols][5] = {count, sum, sumsq, min, max} (nvtb_moments_accumulate's accumulator) */
int nvtb_moments_allreduce(nvtb_comm_t* c, double* acc_dev, int ncols, void* stream);
/* recv holds world blocks of `bytes` bytes in rank order */
int nvtb_comm_allgather(nvtb_comm_t* c, const void* send_dev, void* recv_dev, int64_t bytes, void* stream);
/* send_counts_host[r] elements (elem_bytes each, consecutive in send) go to rank r;
 * recv_counts_host[r] arrive from rank r (consecutive in recv) */
int nvtb_comm_alltoallv(nvtb_comm_t* c, const void* send_dev, const int64_t* send_counts_host,
                        void* recv_dev, const int64_t* recv_counts_host, int elem_bytes, void* stream);

/* ---- session ops: Groupby, ListSlice, Dataset.shuffle_by_keys (csrc/groupby.cu) ----------
 * Replace cuDF sort_values + groupby(sort=True, dropna=True).agg + list.get of reference
 * nvtabular/ops/groupby.py:114-150, 213-240, 290-319, and the numba kernels _calculate_row_sizes
 * / _slice_rows of nvtabular/ops/list_slice.py:180-228.  A partition is ordered once
 * (nvtb_sort_rows), cut into groups once (nvtb_segments: the ONE host synchronisation per
 * Groupby per partition that sizes the outputs, besides the key-range read of the sort), and
 * every output column is one more pass over that order. */

/* Stable lexicographic row order over nkeys (<= 8) key columns, keys[0] most significant
 * (reference groupby.py:116 sort_values + :236 groupby(sort=True)).  descending[k] != 0 orders
 * key k descending (NULL: all ascending).  Rows with a null in any of the first n_drop_null keys
 * are dropped (dropna=True): they go after the *n_kept_dev kept rows of perm_out.  The other keys
 * order their nulls last in either direction (na_position="last").  Floating -0.0 equals +0.0.
 * perm_out: int32[n] row numbers, n < 2^31.  Synchronises once (the keys' value ranges, which
 * trim the radix passes to the bits in use). */
int nvtb_sort_rows(const nvtb_col_t* keys_host, const int* descending_host, int nkeys, int n_drop_null,
                   int64_t n, int32_t* perm_out, int64_t* n_kept_dev, void* stream);
/* group boundaries of the first *n_kept_dev rows of perm (keys equal <=> same group):
 * offsets_out[0..n_groups] (int64, room for n_max + 1), offsets_out[n_groups] = n_kept.
 * Synchronises: the group count and the kept-row count come back to the host. */
int nvtb_segments(const nvtb_col_t* keys_host, int nkeys, const int32_t* perm, int64_t n_max,
                  const int64_t* n_kept_dev, int64_t* offsets_out, int64_t* n_groups_host,
                  int64_t* n_kept_host, void* stream);
/* out[i] = src[perm[idx[i] + idx_shift]] (idx NULL: perm[i]; perm NULL: no permutation) for
 * i < n, any 1/4/8-byte dtype; validity_out (4-byte aligned, padded to a multiple of 4 bytes)
 * is required when src has a validity mask.  The group keys (idx = offsets) and "list"
 * (the whole permutation) of Groupby. */
int nvtb_gather_rows(const nvtb_col_t* src_host, const int32_t* perm, const int64_t* idx,
                     int idx_shift, int64_t n, void* out, uint8_t* validity_out, void* stream);
/* Scalar aggregations of every group of a value column (reference groupby.py:213-240, pandas
 * semantics; accumulated in double).  out_host / validity_out_host: 9 slots in the order
 * count, sum, mean, min, max, std, var, first, last; NULL = not requested.  Output dtypes:
 * count int32; sum, mean, std, var float32; min, max, first, last the value dtype.  count and
 * sum (0 when no value) have no validity; mean, min, max (null without a non-null value), std,
 * var (ddof 1, null below 2 values) need one; first / last (the group's first / last row, a
 * null stays null) need one when the column has nulls.  Groups of up to 32 rows are reduced by
 * one thread, longer ones in chunks of 2048 rows, one CTA each, merged with atomics. */
int nvtb_segment_agg(const nvtb_col_t* val_host, const int32_t* perm, const int64_t* offsets,
                     int64_t n_groups, void* const* out_host, uint8_t* const* validity_out_host,
                     void* stream);
/* median (float32, mean of the two middle values, null without values) and nunique (int32,
 * distinct non-null values) of groups whose rows are in value order with nulls last: perm from
 * nvtb_sort_rows over (group keys..., value), offsets from nvtb_segments of the group keys.
 * n_rows = kept rows.  Either output may be NULL. */
int nvtb_segment_sorted_agg(const nvtb_col_t* val_host, const int32_t* perm, const int64_t* offsets,
                            int64_t n_groups, int64_t n_rows, float* median_out,
                            uint8_t* median_validity_out, int32_t* nunique_out, void* stream);
/* ListSlice (reference list_slice.py:58-75, 104-142): output row r is the Python slice
 * row[start:end] of source row s(r) = perm[idx[r] + idx_shift] (NULL perm / idx as in
 * nvtb_gather_rows), padded at the end to max_elements when pad != 0.  Also the list-row gather
 * of first / last on list columns (start 0, end INT64_MAX).  Step 1 writes offsets_out[n_rows+1]
 * and the leaf count; it synchronises unless pad != 0 (offsets r * max_elements).  Step 2 copies
 * the leaves (pad_value cast to the leaf dtype); validity_out is required when the leaves have
 * nulls and pads are valid. */
int nvtb_list_slice_offsets(const int64_t* offsets, int64_t n_rows, const int32_t* perm,
                            const int64_t* idx, int idx_shift, int64_t start, int64_t end, int pad,
                            int64_t max_elements, int64_t* offsets_out, int64_t* total_host,
                            void* stream);
int nvtb_list_slice(const int64_t* offsets, const nvtb_col_t* leaves_host, int64_t n_rows,
                    const int32_t* perm, const int64_t* idx, int idx_shift, int64_t start,
                    int64_t end, int pad, int64_t max_elements, double pad_value,
                    const int64_t* offsets_out, int64_t total, void* leaves_out,
                    uint8_t* validity_out, void* stream);

/* ---- inference-time transforms on HOST arrays --------------------------------------------
 * The twin of the reference's pybind11 module nvtabular_cpp.inference
 * (cpp/nvtabular/inference/categorify.cc:31-347, fill.cc:32-124; bound at
 * nvtabular/ops/categorify.py:602-609, ops/fill.py:59-65): dict-of-numpy requests of a serving
 * process are encoded by probing a host table of the kept keys (built once from the device
 * vocabulary) with a few host threads — a serving batch is too small to pay for a PCIe round
 * trip.  Labels are identical to nvtb_encode_apply's. */
typedef struct nvtb_infer_vocab nvtb_infer_vocab_t;
/* label = first_label + position of the key in keys_host */
int nvtb_infer_vocab_create(nvtb_infer_vocab_t** out, const int64_t* keys_host, int64_t n);
int nvtb_infer_vocab_from_device(nvtb_infer_vocab_t** out, const nvtb_vocab_t* v, void* stream);
int nvtb_infer_vocab_destroy(nvtb_infer_vocab_t* v);
/* keys_host: int32 | int64 [n]; validity_host: Arrow bitmask or NULL; labels_out_host: int32 |
 * int64 [n]; n_threads <= 0: hardware concurrency (one thread per 16 Ki rows at most) */
int nvtb_infer_categorify_host(const nvtb_infer_vocab_t* v, const void* keys_host, int key_dtype,
                               const uint8_t* validity_host, int64_t n, int64_t null_label,
                               int64_t oov_label, int64_t first_label, uint64_t num_buckets,
                               void* labels_out_host, int out_dtype, int n_threads);
/* FillMissing in place on a host float32 / float64 array (NaN -> fill); integer arrays pass */
int nvtb_infer_fill_host(void* data_host, int dtype, int64_t n, double fill);

#ifdef __cplusplus
}
#endif
#endif /* NVTB200_H */
