/*
 * b200agg.h — C ABI of libb200agg.so: the B200-native replacement for the binned-statistics /
 * groupby hot path of vaexio/vaex (superagg Grid/Binner/Agg kernels + ordered_set ordinal encoder).
 *
 * Plain C: pointers, sizes, enums; no torch / pybind / C++ types cross this boundary.  Every entry
 * point returns 0 on success or a negative b200_status; the message for the calling thread is at
 * b200_last_error().  Nothing throws across the ABI.  There is NO CPU fallback: every compute entry
 * point fails with B200_ERR_CUDA when no sm_100 device is usable.
 *
 * What each entry point replaces in the reference (paths under /root/reference/packages/vaex-core/):
 *
 *   b200_ctx_*            the per-thread state the reference keeps inside each Binner/Aggregator
 *                         (data_ptr[thread], data_mask_ptr[thread]; src/agg_base.hpp:18-30, src/binners.cpp:84-91)
 *                         plus ThreadPoolIndex's thread index (vaex/multithreading.py:64-80): a `slot`
 *                         here is that thread index, bound to one CUDA stream + one H2D staging arena.
 *   b200_agg_create       Agg{Count,Sum,SumMoment,Min,Max,First}_<dtype>(grid, grids, threads[, arg])
 *                         (src/agg.cpp:52-69, src/agg_base.hpp:11-31) and initial_fill()
 *                         (src/agg_count.cpp:13, src/agg_sum.cpp:137, src/agg_minmax.cpp:13-18,83-87,
 *                         src/agg_first.cpp:19-26).  One device grid replaces the `grids` per-thread copies.
 *   b200_bin              Grid::bin / Grid::bin_ (src/agg.hpp:76-137) fused with every
 *                         Binner::to_bins (src/binners.cpp:13-57, src/binner_ordinal.cpp:20-176) and
 *                         Aggregator::aggregate (src/agg_count.cpp:43-67, src/agg_sum.cpp:98-127,
 *                         src/agg_minmax.cpp:45-74,120-145, src/agg_first.cpp:115-165) it would call.
 *   b200_agg_read         Aggregator::get_result (src/agg_count.cpp:24-41, src/agg_sum.cpp:77-96,
 *                         src/agg_first.cpp:61-114) — the multi-grid fold is gone, this is a D2H copy.
 *   b200_agg_merge        Aggregator::merge (src/agg_count.cpp:15-23, src/agg_sum.cpp:69-76, ...).
 *   b200_agg_device_ptr   (no reference counterpart) exposes the device grid so the host side can run
 *                         the NCCL all-reduce across row-sharded GPUs on it in place.
 *   b200_set_*            ordered_set<T> (src/hash_primitives.hpp:437-725, bound in
 *                         src/hash_primitives.cpp:45-56): update / merge / key_array / map_ordinal /
 *                         isin / create-from-keys, and hash<T> (src/hash.hpp:40-152).
 *   b200_minmax           the limits pre-pass: vaexfast statisticNd OP_MIN_MAX (src/vaexfast.cpp:1089-1101).
 *   b200_hash64           superutils.hash (src/superutils.cpp:265) — test hook, host only.
 */
#ifndef B200AGG_H
#define B200AGG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_ABI_VERSION 1
#define B200_MAX_BINNERS 8 /* binners per b200_bin call (reference MAX_DIM is 16, src/agg.hpp:29) */
#define B200_MAX_AGGS 8    /* aggregators fused into one launch; more are split into several launches */

typedef enum {
    B200_OK = 0,
    B200_ERR_INVALID = -1,     /* bad argument ("Expected a 1d array", unknown dtype, ...) */
    B200_ERR_CUDA = -2,        /* CUDA runtime error or no usable device */
    B200_ERR_NODATA = -3,      /* "data not set" (src/agg_sum.cpp:101-103) */
    B200_ERR_UNSUPPORTED = -4, /* valid in the reference but not implemented here */
    B200_ERR_STATE = -5,       /* e.g. merge of sets with unequal nmaps, sealed set */
    B200_ERR_NOMEM = -6
} b200_status;

/* order of src/create_alltypes.hpp */
typedef enum {
    B200_F64 = 0, B200_F32, B200_I64, B200_I32, B200_I16, B200_I8,
    B200_U64, B200_U32, B200_U16, B200_U8, B200_BOOL, B200_NDTYPE
} b200_dtype;

typedef enum {
    B200_BINNER_SCALAR = 0,  /* BinnerScalar_<T>  */
    B200_BINNER_ORDINAL = 1, /* BinnerOrdinal_<T> */
    B200_BINNER_HASH = 2     /* ordinal binner fed by a fused ordered_set probe: the reference's
                                `_ordinal_values(key, set)` expression (vaex/functions.py:2454-2463) +
                                BinnerOrdinal (vaex/groupby.py:303-317) without materialising the codes */
} b200_binner_kind;

typedef enum {
    B200_AGG_COUNT = 0, B200_AGG_SUM, B200_AGG_SUM_MOMENT, B200_AGG_MIN, B200_AGG_MAX,
    B200_AGG_FIRST, B200_AGG_LAST,
    B200_AGG_NUNIQUE /* AggNUnique_<T>(grid, grids, threads, dropmissing, dropnan) (src/agg_nunique.cpp): `moment` bit 0 = dropmissing,
                        bit 1 = dropnan.  b200_agg_input: `mask` = validity (1 = value present, 0 = null row: the reference's
                        data mask), `order` = selection mask (uint8, 1 = the row takes part: set_selection_mask); both nullable */,
    B200_AGG_LIST /* AggList_<T>(grid, grids, threads, dropnan, dropnull) (src/agg_list.cpp:5-127): `moment` bit 0 = dropnan, bit 1 =
                     dropnull; read with b200_agg_list_finish / b200_agg_list_read, not b200_agg_read */,
    B200_AGG_LIST_STRING /* AggList_string_int64(grid, grids, threads, dropnan, dropnull) (src/agg_list.cpp:122-222): per cell the
                            strings in arrival order, a null string as a null element where it arrived (unless dropnull).  `moment` bit 1
                            = dropnull; bit 0 (dropnan) is accepted and has no effect, like in the reference; `dtype` is B200_U8.
                            b200_agg_input: `data` = int64 string offsets[nrows + 1] (arrow large_string; offsets[0] may be > 0),
                            `order` = the bytes they index (NULL only when no row has a byte), `mask` = null mask of the strings
                            (1 = null; nullable).  There is no data mask: the reference never reads it.  Read with
                            b200_agg_list_string_finish / b200_agg_list_string_read.  Fewer than 2^32 rows per aggregator. */
} b200_agg_op;

/* where the column pointers of a call live.  MIXED: every pointer is classified on its own (cudaPointerGetAttributes);
   host columns are staged, device columns are used in place — e.g. device-computed group codes next to host value columns */
typedef enum { B200_MEM_HOST = 0, B200_MEM_DEVICE = 1, B200_MEM_MIXED = 2 } b200_memspace;

/* flags for b200_bin / b200_set_update */
/* Host chunks (B200_MEM_HOST) are by default memcpy'd into the slot's page-locked bounce ring inside the call: the caller's buffers
 * are only read during the call (vaex/cpu.py:708-710) and the call returns without waiting for the device.  With
 * B200_FLAG_ASYNC_HOST the copies are issued straight from the caller's buffers, which must then stay valid (and should be
 * page-locked, b200_host_register) until b200_ctx_sync(slot). */
#define B200_FLAG_ASYNC_HOST 1u

typedef struct b200_ctx b200_ctx;
typedef struct b200_agg b200_agg;
typedef struct b200_set b200_set;

/* One binner + its column for this call.  `mask`: numpy convention, 1 = masked (src/binners.cpp:29). */
typedef struct {
    int32_t kind;        /* b200_binner_kind */
    int32_t dtype;       /* b200_dtype of `data` */
    int32_t byteswap;    /* 1 = the `_non_native` class variant (FlipEndian) */
    int32_t allow_other; /* ordinal */
    int32_t invert;      /* ordinal */
    int32_t reserved;
    double vmin, vmax;   /* scalar */
    uint64_t bins;       /* scalar */
    int64_t ordinal_count, min_value; /* ordinal (for HASH: ordinal_count = number of codes, min_value 0) */
    const b200_set *set; /* HASH only */
    const void *data;
    const uint8_t *mask; /* nullable */
} b200_binner;

/* One aggregator + its columns for this call.  `mask`: aggregator convention, 1 = use the row
 * (src/agg_sum.cpp:107); nullable.  `data` may be NULL only for COUNT (count(*)). */
typedef struct {
    b200_agg *agg;
    const void *data;
    const void *order;   /* FIRST/LAST: order column of dtype2, NULL = chunk-local row index (src/agg_first.cpp:134) */
    const uint8_t *mask;
} b200_agg_input;

/* ---- context ------------------------------------------------------------------------------- */
const char *b200_last_error(void);
int b200_abi_version(void);
int b200_device_count(void);
int b200_ctx_create(int device, int nslots, b200_ctx **out);
int b200_ctx_destroy(b200_ctx *ctx);
int b200_ctx_sync(b200_ctx *ctx, int slot /* -1 = all */);
int b200_ctx_device(const b200_ctx *ctx);
/* raw cudaStream_t of a slot, so host code can order its own work (NCCL, timing events) after ours */
int b200_ctx_stream(b200_ctx *ctx, int slot, void **stream_out);
/* Counters of the last partitioned count(*) batch on this slot (csrc/ringcount.cu), read back from the device after a stream
 * sync — bench.py derives the scratch traffic of the timed build from them instead of quoting a profiler constant:
 * out[0] rows of the batch, out[1] 16-bit entries written to (and read back from) the scratch pool, pads included,
 * out[2] chunks reserved, out[3] entries per chunk, out[4] bytes memset before the batch, out[5] (warp, part) lists.
 * All zero when the slot has not run that path.  No reference counterpart (instrumentation). */
int b200_ctx_path_stats(b200_ctx *ctx, int slot, uint64_t out[6]);
/* Wall-clock accounting of the host-chunk path (b200_bin with B200_MEM_HOST), summed over the slots: out[0..3] nanoseconds spent
 * waiting for a free piece of the page-locked bounce ring, in memcpy into the ring, enqueueing the pieces' copies, and in b200_bin
 * as a whole; out[4] pieces copied, out[5] calls.  reset != 0 zeroes the counters.  No reference counterpart (instrumentation). */
int b200_ctx_host_stats(b200_ctx *ctx, uint64_t out[6], int reset);
/* Measurement aid: enqueue on `slot`'s stream a kernel of `ctas` CTAs x `threads` threads with `smem_bytes` of shared memory that
 * does nothing for `nanoseconds` — it stands in for another stream's kernel holding SMs (an NCCL all-reduce) so that one GPU can
 * show what that costs a persistent kernel on a different slot (tools/ab_headline.py --occupy).  No reference counterpart. */
int b200_ctx_occupy(b200_ctx *ctx, int slot, int ctas, int threads, int smem_bytes, uint64_t nanoseconds);

/* ---- aggregators --------------------------------------------------------------------------- */
int b200_agg_create(b200_ctx *ctx, int op, int dtype, int dtype2, int byteswap, uint32_t moment, uint64_t cells, b200_agg **out);
int b200_agg_destroy(b200_agg *agg);
int b200_agg_reset(b200_agg *agg); /* initial_fill() again (synchronises every slot first) */
/* stream-ordered variants for pipelined drivers: reset / D2H of the device grid enqueued on the slot's stream, no host sync.
 * b200_agg_read_on copies the DEVICE cell type (b200_agg_device_dtype) into `values_out`, which must stay valid until
 * b200_ctx_sync(slot); not available for FIRST/LAST. */
int b200_agg_reset_on(b200_agg *agg, int slot);
int b200_agg_read_on(b200_agg *agg, int slot, void *values_out);
uint64_t b200_agg_cells(const b200_agg *agg);
int b200_agg_result_dtype(const b200_agg *agg); /* count: I64; sum: upcast; min/max/first: dtype */
size_t b200_agg_bytes(const b200_agg *agg);     /* sizeof(result dtype) * cells — the reference's bytes_used() for grids == 1 */
/* which: 0 = primary device grid (cell type b200_agg_device_dtype; NUNIQUE: its three u64 planes), 1 = first/last packed
   {order key, global row} state (2 x u64 per cell), 2 = first/last order values (dtype2), 3 = first/last cell_masked (u8) */
int b200_agg_device_ptr(b200_agg *agg, int which, void **ptr, size_t *bytes);
int b200_agg_device_dtype(const b200_agg *agg);
/* D2H of the finished grid in result dtype; `cell_masked` (nullable) is filled for FIRST/LAST (1 = empty cell) */
int b200_agg_read(b200_agg *agg, void *values_out, uint8_t *cell_masked_out);
int b200_agg_merge(b200_agg *agg, b200_agg *const *others, int nothers);
/* AggList results (src/agg_list.cpp:47-83 get_result): per cell the values in arrival order, then one NaN per NaN value seen (unless
 * dropnan), then one slot per null row (unless dropnull).  finish: sorts the appended records, returns the flat length; read: int64
 * offsets[cells + 1] and `total` values of the aggregator's dtype.  merge() is a no-op like the reference's (:46). */
int b200_agg_list_finish(b200_agg *agg, int64_t *total_out);
int b200_agg_list_read(b200_agg *agg, int64_t *offsets_out, void *values_out);
/* AggListString::get_result (src/agg_list.cpp:141-182).  finish: sorts the appended records (stable, by cell) and builds the result on
 * the device; nelem = elements over all cells, nbytes = their bytes.  read: one D2H per buffer, any may be NULL: list_offsets =
 * int64[cells + 1], str_offsets = int64[nelem + 1] (arrow large_string offsets, starting at 0), bytes[nbytes], nulls[nelem] (1 = null
 * element, which has no bytes).  merge() is a no-op like the reference's (:140). */
int b200_agg_list_string_finish(b200_agg *agg, int64_t *nelem_out, int64_t *nbytes_out);
int b200_agg_list_string_read(b200_agg *agg, int64_t *list_offsets, int64_t *str_offsets, uint8_t *bytes, uint8_t *nulls);
/* load a full grid (result dtype, `cells` long) — TaskPartAggregation initial_values (vaex/cpu.py:654-658) */
int b200_agg_write(b200_agg *agg, const void *values);

/* ---- the hot path --------------------------------------------------------------------------- */
int b200_bin(b200_ctx *ctx, int slot, const b200_binner *binners, int nbinners, const b200_agg_input *aggs, int naggs,
             int64_t nrows, int64_t row_offset, int memspace, uint32_t flags);

/* ---- ordinal encoder ------------------------------------------------------------------------ */
int b200_set_create(b200_ctx *ctx, int dtype, int nmaps, int64_t limit, b200_set **out);
int b200_set_from_keys(b200_ctx *ctx, int dtype, const void *keys, int64_t nkeys, int64_t null_index, int64_t nan_count, int64_t null_count, b200_set **out);
int b200_set_destroy(b200_set *set);
/* masks: 1 = null.  return_values: out_values[nrows] (int64 shard-local ordinals) + out_map_index[nrows] (int16), host memory */
int b200_set_update(b200_set *set, int slot, const void *keys, const uint8_t *masks, int64_t nrows, int64_t start_index,
                    int return_values, int64_t *out_values, int16_t *out_map_index, int memspace, uint32_t flags);
int b200_set_merge(b200_set *set, b200_set *const *others, int nothers);
int64_t b200_set_count(b200_set *set);
int64_t b200_set_nan_count(b200_set *set);
int64_t b200_set_null_count(b200_set *set);
int64_t b200_set_nan_index(b200_set *set);
int64_t b200_set_null_index(b200_set *set);
int b200_set_nmaps(const b200_set *set);
int b200_set_dtype(const b200_set *set);

/* ---- string key sets: vaex.superutils.ordered_set_string (src/hash_string.hpp:56-180, bound at src/hash_string.cpp:86-99) ---------
 * Strings arrive in the arrow large_string layout StringList64 uses: int64 offsets[nrows + 1] into `bytes`, plus an optional byte
 * mask (1 = null; the reference reads the arrow validity bitmap).  shard = std::hash<string_view>(key) % nmaps (libstdc++ 64-bit
 * Murmur-2), ordinal = insertion rank in the shard, nulls join shard 0 at the end of the call that first sees one.  The getters
 * b200_set_count / null_count / null_index / offsets / nmaps / destroy apply.  A 64-bit hash collision between two different
 * strings is detected and reported (B200_ERR_UNSUPPORTED), never merged silently. */
int b200_strset_create(b200_ctx *ctx, int nmaps, int64_t limit /* must be -1 */, b200_set **out);
int b200_strset_update(b200_set *set, int slot, const int64_t *offsets, const uint8_t *bytes, const uint8_t *masks, int64_t nrows, int return_values,
                       int64_t *out_values /* local ordinals */, int16_t *out_map_index, int memspace);
/* global ordinals (-1: not a member); out is host memory, or a device buffer when out_is_device (consume it on the same slot) */
int b200_strset_map_ordinal(b200_set *set, int slot, const int64_t *offsets, const uint8_t *bytes, const uint8_t *masks, int64_t nrows, int64_t *out,
                            int memspace, int out_is_device);
int b200_strset_key_bytes(b200_set *set, int64_t *nbytes_out);
int b200_strset_key_array(b200_set *set, int64_t *offsets_out /* count + 1 */, uint8_t *bytes_out /* key_bytes */);
int b200_set_offsets(b200_set *set, int64_t *out /* nmaps */);
int b200_set_key_array(b200_set *set, void *keys_out /* count * itemsize, host */);
/* out dtype follows the reference: count < 2^7 -> I8, < 2^15 -> I16, < 2^31 -> I32, else I64 */
int b200_set_ordinal_dtype(b200_set *set);
int b200_set_map_ordinal(b200_set *set, int slot, const void *keys, int64_t nrows, void *out, int memspace, uint32_t flags);
int b200_set_isin(b200_set *set, int slot, const void *keys, int64_t nrows, uint8_t *out, int memspace, uint32_t flags);
size_t b200_set_bytes(b200_set *set);
/* Sparse multi-key groupby (vaex/groupby.py:526-584 `_combine`: `sum_k _ordinal_values(key_k) * cumulative_counts[k+1]`,
   vaex/functions.py:2454-2463): per row, the ordinal of every key column in its own set (null rows -> the set's null ordinal,
   NaN -> its NaN ordinal) fused into ONE int64 code = sum_k ordinal_k * multipliers[k]; -1 when a key is in none of the
   sets.  `masks[k]` may be NULL; `out` holds nrows int64 in the call's memspace. */
#define B200_MAX_COMBINE 8
int b200_set_combine(b200_ctx *ctx, int slot, int nkeys, b200_set *const *sets, const void *const *keys, const uint8_t *const *masks,
                     const int64_t *multipliers, int64_t nrows, int64_t *out, int memspace, uint32_t flags);
/* counter_<T> (src/hash_primitives.hpp:344-433, value_counts / unique): an ordered set that also counts the occurrences of each
 * key; `b200_set_counts` returns them in the order of b200_set_key_array (NaN / null slots hold their own counts). */
int b200_counter_create(b200_ctx *ctx, int dtype, int nmaps, b200_set **out);
int b200_set_counts(b200_set *set, int64_t *counts_out);

/* ---- limits pre-pass ------------------------------------------------------------------------ */
/* out[0] = min, out[1] = max over non-NaN, unmasked values, as double; out = {+inf,-inf} when empty.
 */
int b200_minmax(b200_ctx *ctx, int slot, int dtype, int byteswap, const void *data, const uint8_t *mask, int64_t nrows, int memspace, double *out);

/* ---- device-side expressions and filter compaction (SURVEY.md section 8f row 2) ------------------------------------------------
 * Replaces the per-chunk Python `eval` of virtual columns / filters / selections (vaex/scopes.py:108-128 _BlockScope.evaluate) and
 * the pre-filter compression of every dependent column (vaex/execution.py:516-522).  A program is the expression in postfix order;
 * vaex_b200/expression.py builds it from the expression's AST and decides every node's numpy result type (so the results are
 * bit-identical to numpy's).  `cls` is the class the operation computes in (for CAST / ORDINAL: the class of its operand). */
typedef enum {
    B200_EX_INPUT = 0, /* push inputs[arg][row] */
    B200_EX_CONST_F64, /* push f (as float32 when cls == B200_EXC_F32) */
    B200_EX_CONST_I64, /* push i */
    B200_EX_ADD, B200_EX_SUB, B200_EX_MUL, B200_EX_DIV, /* one correctly rounded IEEE operation; integers wrap */
    B200_EX_NEG, B200_EX_ABS, B200_EX_SQRT,
    B200_EX_LT, B200_EX_LE, B200_EX_GT, B200_EX_GE, B200_EX_EQ, B200_EX_NE, /* -> bool */
    B200_EX_AND, B200_EX_OR, B200_EX_NOT,                                   /* on bools */
    B200_EX_CAST,   /* astype(b200_dtype arg) */
    B200_EX_ORDINAL /* _ordinal_values(value, sets[arg]) -> int64 ordinal, -1 when absent (vaex/functions.py:2454-2463) */
} b200_expr_opcode;
typedef enum { B200_EXC_F64 = 0, B200_EXC_F32, B200_EXC_I64 /* any signed integer, sign-extended */, B200_EXC_U64, B200_EXC_BOOL } b200_expr_class;
typedef struct {
    int32_t op, cls, arg, reserved;
    double f;
    int64_t i;
} b200_expr_op;
typedef struct {
    const void *data;
    int32_t dtype; /* b200_dtype, native byte order */
    int32_t reserved;
} b200_expr_input;
/* out_device: device buffer of nrows elements of out_dtype; the kernel is enqueued on the slot's stream (consume the result on the
 * same slot).  <= 64 ops, 8 inputs, 4 sets, stack depth 12. */
int b200_eval(b200_ctx *ctx, int slot, const b200_expr_op *prog, int nops, const b200_expr_input *inputs, int ninputs, b200_set *const *sets, int nsets,
              int64_t nrows, int memspace, int out_dtype, void *out_device);
/* stable compaction of up to 16 columns by a keep-mask (1 byte per row, non-zero = keep): outs_device[c] receives the kept rows of
 * cols[c] in order; *count_out = rows kept (the call waits for it). */
int b200_compact(b200_ctx *ctx, int slot, const uint8_t *keep, int ncols, const void *const *cols, const int32_t *dtypes, int64_t nrows, int memspace,
                 void *const *outs_device, int64_t *count_out);


/* ---- host-chunk ingestion (SURVEY.md 8f row 2) ---------------------------------------------- */
/* Page-lock a host column once (cudaHostRegister) so that the per-chunk H2D copies of b200_bin(HOST) run at PCIe rate and
 * truly asynchronously; the reference has no counterpart (its columns are mmapped/numpy memory read by the CPU in place). */
int b200_host_register(const void *ptr, size_t bytes);
int b200_host_unregister(const void *ptr);

/* ---- test hook ------------------------------------------------------------------------------ */
uint64_t b200_hash64(uint64_t x);

#ifdef __cplusplus
}
#endif
#endif /* B200AGG_H */
