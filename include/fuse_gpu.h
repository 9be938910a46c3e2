/*
 * fuse_gpu.h — C ABI of libfuse_gpu.so: the B200 (sm_100a) replacement for fuse-query's vectorised
 * Source -> Filter -> Projection -> AggregatePartial / Limit hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  A Rust FFI crate
 * (`extern "C"` block, see INTEGRATION.md) binds exactly these symbols; the C++ host mirror under
 * fuse_query_b200/csrc/host and the Python ctypes layer call nothing else.  Citations are
 * file:line under /root/reference/src and name the reference interface each entry point replaces.
 *
 * Conventions
 *   - every function returns an fq_status (0 = ok); fq_last_error(ctx) returns the message, which
 *     reproduces the reference's FuseQueryError Display text where one exists (error.rs:10-20);
 *   - nothing throws or aborts across the ABI;
 *   - handles are opaque, created/destroyed by the library; host buffers belong to the caller;
 *   - every launch takes a CUDA stream (cudaStream_t / CUstream passed as void*, NULL = the
 *     legacy default stream) and is asynchronous; results are read with the matching *_fetch call;
 *   - a context binds one CUDA device; calls set the device themselves, so any host thread may
 *     drive any context (the reference runs one tokio task per partition pipe,
 *     processors/processor_merge.rs:46-62).  Contexts and columns may be shared between threads; a pipe
 *     owns running state (aggregate state, result slots) and is driven by one thread at a time — the
 *     reference clones its Function per pipe for the same reason (pipeline_builder.rs:50-65).
 */
#ifndef FUSE_GPU_H
#define FUSE_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FQ_ABI_VERSION 2

/* status codes; FQ_ERR_INTERNAL/FQ_ERR_PLAN map onto FuseQueryError::{Internal,Plan} (error.rs:10-20) */
typedef int32_t fq_status;
enum {
  FQ_OK = 0,
  FQ_ERR_INTERNAL = 1,       /* "Internal Error: ..." */
  FQ_ERR_PLAN = 2,           /* "Error during plan: ..." */
  FQ_ERR_DIVIDE_BY_ZERO = 3, /* arrow DivideByZero -> "Internal Error: Divide by zero error" */
  FQ_ERR_UNSUPPORTED = 4,    /* well-formed request the device path does not implement (never a silent fallback) */
  FQ_ERR_CUDA = 5,           /* CUDA runtime / driver / NVRTC failure */
  FQ_ERR_INVALID = 6,        /* bad handle / argument */
  FQ_ERR_CAPACITY = 7        /* a GROUP BY pipe met more groups than its table was reserved for: reserve more and relaunch */
};

/* DataType / DataValue tags in the declaration order of datavalues/data_value.rs:19-35 */
typedef int32_t fq_dtype;
enum {
  FQ_NULL = 0, FQ_BOOL = 1, FQ_I8 = 2, FQ_I16 = 3, FQ_I32 = 4, FQ_I64 = 5, FQ_U8 = 6, FQ_U16 = 7,
  FQ_U32 = 8, FQ_U64 = 9, FQ_F32 = 10, FQ_F64 = 11, FQ_UTF8 = 12, FQ_STRUCT = 13
};

/* operator enums of datavalues/data_value_operator.rs:5-81 */
enum { FQ_AGG_MIN = 0, FQ_AGG_MAX = 1, FQ_AGG_SUM = 2, FQ_AGG_COUNT = 3 };
enum { FQ_CMP_EQ = 0, FQ_CMP_LT = 1, FQ_CMP_LTEQ = 2, FQ_CMP_GT = 3, FQ_CMP_GTEQ = 4 };
enum { FQ_AR_ADD = 0, FQ_AR_SUB = 1, FQ_AR_MUL = 2, FQ_AR_DIV = 3 };
enum { FQ_LG_AND = 0, FQ_LG_OR = 1 };

/* ---------------------------------------------------------------------------------------------
 * Expression trees: a flat array of nodes restating `enum Function` (functions/function.rs:16-25).
 * Children are indexes into the same array; every expression handed to the library is a root index.
 * ------------------------------------------------------------------------------------------- */
enum {
  FQ_EXPR_ALIAS = 0,      /* function_alias.rs: transparent, child in `left` */
  FQ_EXPR_CONSTANT = 1,   /* function_constant.rs: dtype + value */
  FQ_EXPR_FIELD = 2,      /* function_field.rs: input column index in `column` */
  FQ_EXPR_ARITHMETIC = 3, /* function_arithmetic.rs: op in FQ_AR_* */
  FQ_EXPR_COMPARISON = 4, /* function_comparison.rs: op in FQ_CMP_* */
  FQ_EXPR_LOGIC = 5,      /* function_logic.rs: op in FQ_LG_* */
  FQ_EXPR_AGGREGATOR = 6, /* function_aggregator.rs: op in FQ_AGG_*, argument in `left` */
  FQ_EXPR_LOOKUP = 7      /* Boolean: bit `left` of the bit table bound to slot `op` (fq_pipe_set_lookup); `left` is an unsigned
                             integer expression (normally a dictionary codes column) and not a constant, op in
                             [0, FQ_MAX_LOOKUPS); a value at or beyond the table's bit count gives false; NULL where `left` is */
};

typedef union fq_scalar_bits {
  int64_t i;  /* FQ_BOOL, FQ_I8..FQ_I64 */
  uint64_t u; /* FQ_U8..FQ_U64 */
  double f;   /* FQ_F32 (rounded to float by the library), FQ_F64 */
} fq_scalar_bits;

typedef struct fq_expr_node {
  int32_t kind;   /* FQ_EXPR_* */
  int32_t op;     /* operator for ARITHMETIC / COMPARISON / LOGIC / AGGREGATOR, slot for LOOKUP */
  int32_t left;   /* child index or -1 */
  int32_t right;  /* child index or -1 */
  int32_t column; /* FIELD: index into the pipe's input columns */
  fq_dtype dtype; /* CONSTANT: value type */
  fq_scalar_bits value;
} fq_expr_node;

/* DataValue restricted to what crosses the boundary (aggregate states, scalar results) */
typedef struct fq_value {
  fq_dtype dtype; /* FQ_NULL = DataValue::Null */
  int32_t some;   /* 0 = Type(None) */
  fq_scalar_bits v;
} fq_value;

/* ---------------------------------------------------------------------------------------------
 * Context
 * ------------------------------------------------------------------------------------------- */
typedef struct fq_ctx fq_ctx;

uint32_t fq_abi_version(void);
fq_status fq_ctx_create(int32_t device, fq_ctx **out);
void fq_ctx_destroy(fq_ctx *ctx);
/* message of the last failing call on this context from the calling thread ("" if none);
 * ctx == NULL returns the message of a failed fq_ctx_create */
const char *fq_last_error(const fq_ctx *ctx);
/* number of kernels this context has launched (bench.py's gpu_launches) */
uint64_t fq_ctx_launch_count(const fq_ctx *ctx);
/* multiprocessor count of the bound device (grid sizing is the library's job; exposed for reports) */
int32_t fq_ctx_sm_count(const fq_ctx *ctx);

/* ---------------------------------------------------------------------------------------------
 * Columns — device-resident Arrow-layout buffers replacing ArrayRef inside DataBlock
 * (datablocks/data_block.rs:10-14): contiguous little-endian values, 256-byte aligned.
 * numbers_mt's column is NOT NULL (datasources/system/numbers_table.rs:21-25) and carries nothing else.
 * A nullable column additionally points at a validity column: FQ_BOOL, one byte per row (1 = valid) — Arrow's
 * bit-packed validity is unpacked when it is uploaded, so that slicing and compaction stay byte-addressed.
 * ------------------------------------------------------------------------------------------- */
typedef struct fq_column fq_column;

fq_status fq_column_alloc(fq_ctx *ctx, fq_dtype dtype, uint64_t len, fq_column **out);
/* borrow device memory owned by the caller (e.g. a torch tensor); must be 16-byte aligned */
fq_status fq_column_wrap(fq_ctx *ctx, fq_dtype dtype, uint64_t len, void *device_values, fq_column **out);
/* zero-copy view of rows [offset, offset+len) of `parent` (arrow slice); parent must outlive it */
fq_status fq_column_slice(fq_ctx *ctx, const fq_column *parent, uint64_t offset, uint64_t len, fq_column **out);
/* attach (validity != NULL) or detach a validity column; it is borrowed and must outlive `col`; slices of `col`
 * made afterwards slice it too */
fq_status fq_column_set_validity(fq_ctx *ctx, fq_column *col, const fq_column *validity);
/* The same with Arrow's own validity buffer, left bit-packed: `bitmap` is an FQ_U8 column holding the LSB-first bitmap
 * (bit = 1: valid), row 0 of `col` = bit `bit_offset` (arrow's array offset).  Pipes compiled with col_nullable = 2 read
 * the bits in place: 1 bit of validity traffic per row instead of 1 byte (12.5 % -> 1.6 % on a UInt64 column, 100 % ->
 * 12.5 % on a UInt8 one).  Borrowed like a byte validity column; slices of `col` keep it with a moved offset. */
fq_status fq_column_set_validity_bitmap(fq_ctx *ctx, fq_column *col, const fq_column *bitmap, uint64_t bit_offset);
const fq_column *fq_column_validity(const fq_column *col);
void fq_column_free(fq_ctx *ctx, fq_column *col);
fq_dtype fq_column_dtype(const fq_column *col);
uint64_t fq_column_len(const fq_column *col);
void *fq_column_device_ptr(const fq_column *col);
/* async copies of `n_rows` values starting at row `row_offset`; host memory should be pinned */
fq_status fq_column_upload(fq_ctx *ctx, fq_column *col, uint64_t row_offset, const void *host, uint64_t n_rows, void *stream);
fq_status fq_column_download(fq_ctx *ctx, const fq_column *col, uint64_t row_offset, void *host, uint64_t n_rows, void *stream);
/* Arrow bitmaps <-> the device's one byte per row.  The reference's BooleanArray values and every array's validity
 * are LSB-first bitmaps (arrow 2.0.0 bitmap.rs / buffer.rs; `DataBlock` columns are arrow ArrayRef,
 * datablocks/data_block.rs:10-14).  `col` must be a Boolean column (values, or the validity column of another).
 * upload: rows [row_offset, row_offset + n_rows) = bits [bit_offset, bit_offset + n_rows) of `host_bits`, expanded by
 * a kernel (one source byte -> one 8-byte store); download: the inverse, `host_bits` receives ceil(n_rows / 8)
 * bytes starting at bit 0, padding bits zero.  Async on `stream` like the plain copies. */
fq_status fq_column_upload_bits(fq_ctx *ctx, fq_column *col, uint64_t row_offset, const void *host_bits, uint64_t bit_offset,
                                uint64_t n_rows, void *stream);
fq_status fq_column_download_bits(fq_ctx *ctx, const fq_column *col, uint64_t row_offset, void *host_bits, uint64_t n_rows,
                                  void *stream);
/* device-to-device: dst[dst_offset .. +n_rows) = src[src_offset .. +n_rows) (same type; values only) */
fq_status fq_column_copy(fq_ctx *ctx, fq_column *dst, uint64_t dst_offset, const fq_column *src, uint64_t src_offset, uint64_t n_rows,
                         void *stream);
fq_status fq_stream_synchronize(fq_ctx *ctx, void *stream);
/* `stream` arguments are cudaStream_t handles of the caller (NULL = the default stream).  A host without CUDA bindings of
 * its own gets one here: a non-blocking stream on the context's device. */
fq_status fq_stream_create(fq_ctx *ctx, void **stream);
void fq_stream_destroy(fq_ctx *ctx, void *stream);
/* pinned host staging memory */
fq_status fq_host_alloc(fq_ctx *ctx, uint64_t bytes, void **out);
void fq_host_free(fq_ctx *ctx, void *p);

/* ---------------------------------------------------------------------------------------------
 * Utf8 arrays — Arrow string layout on the device: int32 offsets[len + 1] + the value bytes (+ an optional validity column,
 * one byte per row).  What the reference does with strings on this path: the *_utf8 comparison kernels for array (op) array
 * and array (op) scalar (datavalues/macros.rs:29-36, 102-113 <- data_array_comparison.rs:29-85), min_string / max_string
 * (macros.rs:162 <- data_array_aggregate.rs:139-154) and count.  Strings compare bytewise (Rust `str` ordering, which
 * arrow's comparison kernels use).  Results are ordinary Boolean columns, so they feed filters like any predicate.
 * ------------------------------------------------------------------------------------------- */
typedef struct fq_utf8 fq_utf8;
/* copies offsets (len + 1 entries, host) and the value bytes (offsets[len] bytes, host) to the device; `validity` (FQ_BOOL,
 * borrowed, may be NULL) marks NULL slots */
fq_status fq_utf8_create(fq_ctx *ctx, const int32_t *offsets, const void *data, uint64_t len, const fq_column *validity, void *stream,
                         fq_utf8 **out);
void fq_utf8_free(fq_ctx *ctx, fq_utf8 *a);
uint64_t fq_utf8_len(const fq_utf8 *a);
/* out[row] = l[row] op r[row] (op in FQ_CMP_*), out_valid[row] = both valid; out_valid may be NULL when neither side
 * carries validity.  Arrays must have the same length. */
fq_status fq_utf8_compare(fq_ctx *ctx, int32_t op, const fq_utf8 *l, const fq_utf8 *r, fq_column *out, fq_column *out_valid, void *stream);
fq_status fq_utf8_compare_scalar(fq_ctx *ctx, int32_t op, const fq_utf8 *l, const void *scalar, uint64_t scalar_len, fq_column *out,
                                 fq_column *out_valid, void *stream);
/* row index of the smallest (FQ_AGG_MIN) / largest (FQ_AGG_MAX) valid string, first occurrence; -1 when there is none
 * (arrow min_string / max_string return None).  Waits for the result. */
fq_status fq_utf8_minmax(fq_ctx *ctx, int32_t op, const fq_utf8 *a, int64_t *row, void *stream);
/* value bytes of the array (offsets[len]) */
uint64_t fq_utf8_bytes(const fq_utf8 *a);
/* async copy to host memory: offsets_host receives len + 1 entries, data_host fq_utf8_bytes(a) bytes */
fq_status fq_utf8_download(fq_ctx *ctx, const fq_utf8 *a, int32_t *offsets_host, void *data_host, void *stream);
/* Gather by index: *out[i] = src[rows[i]] for i < n (`rows` a UInt32 column, every index < len(src)).  rows_validity (FQ_BOOL,
 * may be NULL, borrowed: it becomes the validity of *out and must outlive it) marks output slots that are NULL; their rows are
 * not read.  Fails, instead of truncating, when the result would exceed 2 GiB of value bytes.  Waits for the result. */
fq_status fq_utf8_take(fq_ctx *ctx, const fq_utf8 *src, const fq_column *rows, uint64_t n, const fq_column *rows_validity, fq_utf8 **out,
                       void *stream);
/* Dictionary encoding (fewer than 2^32 - 1 rows).  codes (FQ_U32, at least len(src) slots) receives, for every valid row, the
 * position of its string in *dict: the distinct valid strings of `src` in bytewise order, with no validity.  NULL rows get code
 * 0; the caller gives `codes` the source's validity.  Because the dictionary is sorted, code order is string order, and a
 * Utf8 column `s` with codes `c` lowers to integer work (lb / ub = fq_utf8_bounds of the literal, D = dictionary length):
 *   s = 'x'                 c = lb when lb < ub (the literal is in the dictionary), else c = D (no row has that code)
 *   s < 'x', s <= 'x'       c < lb, c < ub
 *   s > 'x', s >= 'x'       c >= ub, c >= lb
 *   'x' op s                flip the operator first (data_array_comparison.rs:75-85)
 *   s op s2                 c op c2, when both columns hold codes of the SAME dictionary
 *   GROUP BY s / ORDER BY s group / sort by c (NULL rows stay NULL through the codes' validity), then decode with fq_utf8_take
 *   min(s), max(s)          min / max of c, then the dictionary entry;  count(s) is unchanged
 * Waits for the result. */
fq_status fq_utf8_dict_encode(fq_ctx *ctx, const fq_utf8 *src, fq_column *codes, fq_utf8 **dict, void *stream);
/* lower = the first index of the sorted array `dict` whose string is >= the literal, upper = the first one > it.  Waits. */
fq_status fq_utf8_bounds(fq_ctx *ctx, const fq_utf8 *dict, const void *scalar, uint64_t scalar_len, uint64_t *lower, uint64_t *upper,
                         void *stream);
/* SQL LIKE against one pattern: bit i of `bits` (an FQ_U8 column of at least ceil(len(a) / 8) bytes, LSB-first like Arrow's
 * bitmaps) = a[i] LIKE pattern, negated when `negate` is set (NOT LIKE); NULL rows get bit 0 in both cases, the caller keeps
 * a's validity.  `%` matches any run of characters (newlines included), `_` one character (one UTF-8 code point), `\` makes
 * the next pattern character literal (`\%`, `\_`, `\\`); there is no ESCAPE clause.  Matching is bytewise and case-sensitive,
 * the equality fq_utf8_compare uses.  A pattern that ends in an unpaired `\` is FQ_ERR_INVALID.  Waits for the result.
 * Over a dictionary the pattern is matched once per distinct string, and a Utf8 column `s` with codes `c` lowers to
 *   s LIKE 'p'              (lookup k c)  with slot k bound to fq_utf8_like(dict, 'p', 0)   (FQ_EXPR_LOOKUP)
 *   s NOT LIKE 'p'          (lookup k c)  with slot k bound to fq_utf8_like(dict, 'p', 1)
 * so the pipe's generated source depends on the slot, not on the pattern: one compiled pipe serves every pattern. */
fq_status fq_utf8_like(fq_ctx *ctx, const fq_utf8 *a, const void *pattern, uint64_t pattern_len, int32_t negate, fq_column *bits,
                       void *stream);

/* ---------------------------------------------------------------------------------------------
 * Source — system.numbers_mt shards.  Replaces NumbersStream::poll_next materialising 10 000-row
 * UInt64Arrays (datasources/system/numbers_stream.rs:68-83): one fill kernel writes the whole
 * shard [begin, end] (inclusive, like the partition names of numbers_table.rs:29-55) into HBM.
 * The "generated" mode has no column at all: see fq_source.numbers_begin.
 * ------------------------------------------------------------------------------------------- */
fq_status fq_numbers_fill(fq_ctx *ctx, fq_column *col, uint64_t row_offset, uint64_t begin, uint64_t n_rows, void *stream);

typedef struct fq_source {
  uint64_t n_rows;
  int32_t n_cols;             /* materialised input columns (0 in generated mode) */
  int32_t generated;          /* 1: column 0 is UInt64 `numbers_begin + row`, produced in-kernel */
  const fq_column *const *cols;
  uint64_t numbers_begin;
} fq_source;

/* ---------------------------------------------------------------------------------------------
 * Pipes — one fused kernel per Source -> [Filter] -> (Projection | AggregatePartial) [-> Limit]
 * chain of processors/pipeline_builder.rs:26-106.  Compiling a pipe specialises the kernel for the
 * expression trees (precompiled table for the README shapes, NVRTC for everything else).
 * ------------------------------------------------------------------------------------------- */
#define FQ_MAX_COLS 8
#define FQ_MAX_EXPRS 8
#define FQ_MAX_KEYS 4
/* bit tables one pipe reads through FQ_EXPR_LOOKUP nodes */
#define FQ_MAX_LOOKUPS 4

enum { FQ_PIPE_PROJECT = 0, FQ_PIPE_AGGREGATE = 1, FQ_PIPE_GROUPBY = 2 };

typedef struct fq_pipe_desc {
  int32_t n_cols;                   /* input schema */
  fq_dtype col_dtypes[FQ_MAX_COLS];
  int32_t col_nullable[FQ_MAX_COLS]; /* 1: the column carries validity, one byte per row (fq_column_set_validity);
                                        2: validity is an Arrow bitmap (fq_column_set_validity_bitmap) */
  int32_t generated;                /* specialise for fq_source.generated (column 0 = UInt64 numbers) */
  const fq_expr_node *nodes;
  int32_t n_nodes;
  int32_t predicate;                /* root of the WHERE predicate (transform_filter.rs:38-55) or -1 */
  int32_t kind;                     /* FQ_PIPE_PROJECT (transform_projection.rs:45-56) or FQ_PIPE_AGGREGATE
                                       (transform_aggregate_partial.rs:50-78) */
  int32_t n_exprs;
  int32_t exprs[FQ_MAX_EXPRS];      /* roots of the select expressions */
  int32_t n_keys;                   /* FQ_PIPE_GROUPBY: GROUP BY expressions (plan_parser.rs:279-308), else 0 */
  int32_t keys[FQ_MAX_KEYS];        /* their roots; `exprs` are the aggregate expressions (AggregatePlan.aggr_expr) */
} fq_pipe_desc;

typedef struct fq_pipe fq_pipe;

fq_status fq_pipe_compile(fq_ctx *ctx, const fq_pipe_desc *desc, fq_pipe **out);
void fq_pipe_destroy(fq_ctx *ctx, fq_pipe *pipe);
/* Kernel variant the pipe's launches prefer: aggregate pipes "tma" (bulk-copy staged, default) | "u4" (LDG.128 x 4), filter +
 * projection pipes "tma" | "sparse" | "dense" | "ldg", projection pipes "tma" | "ldg"; GROUP BY pipes have none.  The default
 * comes from FQ_AGG_VARIANT / FQ_SEL_VARIANT / FQ_MAP_VARIANT, read once when the pipe is compiled (never on the launch path);
 * another word is FQ_ERR_INVALID, there and here.  A variant the pipe's module does not hold falls back to one it does. */
fq_status fq_pipe_set_variant(fq_ctx *ctx, fq_pipe *pipe, const char *variant);
/* Binds bit table `slot` of the pipe's FQ_EXPR_LOOKUP nodes: `bits` is an FQ_U8 column holding at least ceil(n_bits / 8) bytes,
 * LSB-first (fq_utf8_like writes one).  Borrowed: it must outlive the launches that follow, which read it; binding the slot
 * again replaces it for later launches.  A launch of a pipe with an unbound slot is FQ_ERR_INVALID. */
fq_status fq_pipe_set_lookup(fq_ctx *ctx, fq_pipe *pipe, int32_t slot, const fq_column *bits, uint64_t n_bits);
/* 1 if the kernel came from the library's precompiled table, 0 if NVRTC built it */
int32_t fq_pipe_is_precompiled(const fq_pipe *pipe);
/* where the pipe's kernels came from: 0 = the library's precompiled table, 1 = built by NVRTC in this process,
 * 2 = a cubin from the on-disk JIT cache ($FQ_JIT_CACHE_DIR, default .jit_cache next to the library; FQ_JIT_CACHE=0
 * disables it) */
int32_t fq_pipe_build_kind(const fq_pipe *pipe);
/* generated CUDA source of the specialised part (diagnostics / DESIGN.md) */
const char *fq_pipe_source(const fq_pipe *pipe);
/* Function::return_type of select expression i over the pipe's schema (functions/function.rs:28-38) */
fq_status fq_pipe_expr_dtype(fq_ctx *ctx, const fq_pipe *pipe, int32_t i, fq_dtype *out);
/* projection pipes: 1 when select expression i can yield NULL (a nullable input, or a coercion cast that arrow turns
 * into NULL when the value does not fit): the launch then needs a validity output column for it */
fq_status fq_pipe_expr_nullable(fq_ctx *ctx, const fq_pipe *pipe, int32_t i, int32_t *out);

/* ---- aggregate pipes: Function::accumulate over a whole shard (function_aggregator.rs:57-100) ----
 * The device keeps one running state per Aggregator leaf.  FQ_RUN_ACCUMULATE folds this launch into
 * the running state (successive blocks of one partition); without it the state restarts from Null.
 * FQ_RUN_BLOCK_STATS additionally records, for pipes with a WHERE predicate and a Sum leaf, how many of
 * the reference's 10 000-row blocks (numbers_stream.rs:29, counted from row 0 of each launch) kept no row:
 * the reference folds Sum per block and an empty block poisons its state (SURVEY F8).  The counts are
 * reported by fq_pipe_fetch_block_stats; what to do with them is the caller's decision. */
enum { FQ_RUN_ACCUMULATE = 1, FQ_RUN_LIMIT_EARLY_EXIT = 2, FQ_RUN_BLOCK_STATS = 4 };

fq_status fq_pipe_launch_aggregate(fq_ctx *ctx, fq_pipe *pipe, const fq_source *src, uint32_t flags, void *stream);
/* Waits for the last launch and returns, for each Aggregator leaf in node-index order, the state
 * Function::accumulate_result would hold (function_aggregator.rs:102-104): Null if no launch folded
 * any block, Type(None) for Sum/Min/Max over zero rows, else Type(Some(v)).  rows_selected is the
 * post-filter row count.  A zero divisor anywhere in the scanned rows yields FQ_ERR_DIVIDE_BY_ZERO. */
fq_status fq_pipe_fetch_aggregate(fq_ctx *ctx, fq_pipe *pipe, fq_value *states, int32_t cap, int32_t *n_states,
                                  uint64_t *rows_selected);
/* after fq_pipe_fetch_aggregate: reference blocks scanned / left empty by the predicate over the launches folded so far
 * (both 0 when the pipe has no predicate + Sum leaf or FQ_RUN_BLOCK_STATS was not set) */
fq_status fq_pipe_fetch_block_stats(fq_ctx *ctx, fq_pipe *pipe, uint64_t *blocks, uint64_t *empty_blocks);
/* node indexes of the Aggregator leaves, in the order fetch reports them */
fq_status fq_pipe_aggregator_nodes(fq_ctx *ctx, const fq_pipe *pipe, int32_t *nodes, int32_t cap, int32_t *n);
/* device address of the raw running state: FQ_STATE_HEADER_SLOTS 8-byte header slots (rows selected, error bits,
 * launches folded, rows scanned, reference blocks, empty reference blocks) then one slot per leaf — for collectives
 * that merge states on the device (ncclAllGather of n_bytes) */
#define FQ_STATE_HEADER_SLOTS 6
fq_status fq_pipe_state_device(fq_ctx *ctx, const fq_pipe *pipe, void **dev_ptr, uint64_t *n_bytes);

/* ---- GROUP BY pipes: hash aggregation (SURVEY 8 f4) ----
 * The reference plans GROUP BY (plan_parser.rs:279-308: AggregatePlan{group_expr, aggr_expr}, schema = the group fields
 * followed by the aggregate fields) but its pipeline builder only ever uses aggr_expr (pipeline_builder.rs:50-65): the
 * operator is not executed there.  This is the operator the plan describes, with the reference's own aggregate protocol
 * applied per group: one output row per distinct tuple of key values (a NULL key is a group of its own); Sum / Min / Max
 * skip NULL slots and are Type(None) for a group without a valid row, Count is the group's row count
 * (function_aggregator.rs:57-100, data_array_aggregate.rs:29); integer sums wrap.  Row order of the result is unspecified.
 *
 * A FQ_PIPE_GROUPBY pipe keeps an open-addressing hash table in HBM: packed keys (the key expressions' value bits, plus
 * one bit per nullable key: one 64-bit word for up to 64 bits in all, two words for 65..128 bits, claimed by one 16-byte
 * compare-and-swap; wider key sets are refused) and one 8-byte state per Aggregator leaf per group, updated with atomics;
 * every CTA pre-aggregates in a shared-memory table first, so low-cardinality keys never leave the SM.
 * fq_pipe_groupby_reserve sizes (and clears) the table; a launch that meets more groups than reserved makes
 * fq_pipe_fetch_groupby return FQ_ERR_CAPACITY (reserve more, relaunch).  Every reservation after a pipe's first also hashes
 * the keys with a new seed, so keys whose hashes clustered in one table (a probe chain too long: FQ_ERR_CAPACITY with room
 * to spare) are spread in the next.  No scan needs room for more groups than the rows it reads: an overflow at that size
 * is worth one more reservation of the same size, not a larger one.  FQ_RUN_ACCUMULATE keeps the table between launches.
 * fq_pipe_export_groups writes the groups, in table order, to dense columns: key_cols[j] (+ key_valid[j] for nullable
 * keys, one byte per row) and one column per Aggregator leaf in fq_pipe_aggregator_nodes order (+ leaf_valid[k] for
 * leaves fq_pipe_leaf_nullable reports) — the caller evaluates arithmetic over aggregates (sum(x) / count(x)) as an
 * ordinary projection over those columns, exactly like merge_result re-applies it (function_arithmetic.rs:82-88). */
fq_status fq_pipe_key_dtype(fq_ctx *ctx, const fq_pipe *pipe, int32_t j, fq_dtype *out, int32_t *nullable);
fq_status fq_pipe_leaf_dtype(fq_ctx *ctx, const fq_pipe *pipe, int32_t k, fq_dtype *out, int32_t *nullable);
fq_status fq_pipe_groupby_reserve(fq_ctx *ctx, fq_pipe *pipe, uint64_t groups);
fq_status fq_pipe_launch_groupby(fq_ctx *ctx, fq_pipe *pipe, const fq_source *src, uint32_t flags, void *stream);
fq_status fq_pipe_fetch_groupby(fq_ctx *ctx, fq_pipe *pipe, uint64_t *n_groups);
fq_status fq_pipe_export_groups(fq_ctx *ctx, fq_pipe *pipe, fq_column *const *key_cols, fq_column *const *key_valid,
                                fq_column *const *leaf_cols, fq_column *const *leaf_valid, uint64_t capacity, void *stream);
/* Multi-GPU exchange of partial groups (one process per GPU).  fq_pipe_export_partials writes this rank's groups as raw
 * table entries — `entries` is a UInt64 column of n_groups x fq_pipe_group_entry_slots rows: the packed key, 1 or 2
 * words, then the state slots — ordered by owner rank = hash(key) mod world, and reports how many go to each rank (counts[world], host
 * memory, valid after fq_stream_synchronize).  The host moves the runs to their owners (NCCL all-to-all over NVLink);
 * fq_pipe_merge_partials folds received entries into this pipe's table with the merge_state rules.  Afterwards every rank
 * owns a disjoint set of complete groups and exports them with fq_pipe_export_groups. */
fq_status fq_pipe_group_entry_slots(fq_ctx *ctx, const fq_pipe *pipe, int32_t *slots);
fq_status fq_pipe_export_partials(fq_ctx *ctx, fq_pipe *pipe, int32_t world, fq_column *entries, uint64_t *counts, void *stream);
fq_status fq_pipe_merge_partials(fq_ctx *ctx, fq_pipe *pipe, const fq_column *entries, uint64_t n_entries, uint32_t flags, void *stream);

/* ---- multi-GPU merge point (processors/processor_merge.rs:37-66 feeding transform_aggregate_final.rs:50-78 /
 * the LimitTransform after the merge, pipeline_builder.rs:31-41) without a collective call ----
 * One process per GPU.  A group is a set of 1..8 ranks, each owning an exchange window in its GPU's memory
 * (2 parities x world rows of `row_bytes`).  Every rank creates its group, exports the window with fq_group_handle
 * (64-byte CUDA IPC handle, exchanged by the host however it likes: torch.distributed, MPI, a socket) and hands the
 * `world * 64` bytes of all handles, in rank order, to fq_group_connect (ranks in ONE process pass raw window addresses
 * to fq_group_connect_ptrs instead: IPC handles cannot be opened by the process that made them).
 *
 * Aggregate pipes: after fq_pipe_set_group every fq_pipe_launch_aggregate ends with the merge point INSIDE the kernel —
 * its last CTA stores the running state into its row of every rank's window over NVLink peer memory (release at system
 * scope), waits until the rows of all ranks for this operation have arrived in its own window, folds them in rank order
 * (wrapping add / min / max — the merge_state rules, function_aggregator.rs:106-139) and leaves the merged state of the
 * whole group on every rank: fq_pipe_fetch_merged.  No host round trip, no collective library call.
 * Projection pipes: fq_group_gather_project concatenates the rows every rank's launch wrote, in rank (= partition) order,
 * cut at `limit`, into `final_cols` on every rank.
 *
 * Like a communicator, a group numbers its operations: every rank must issue the same sequence of group operations
 * (launches of pipes bound to the group, gathers).  A rank that never shows up makes the others fail with FQ_ERR_CUDA
 * after FQ_GROUP_TIMEOUT_MS (default 20 000) instead of hanging the GPU. */
typedef struct fq_group fq_group;
fq_status fq_group_create(fq_ctx *ctx, int32_t rank, int32_t world, uint64_t row_bytes, fq_group **out);
fq_status fq_group_handle(fq_ctx *ctx, const fq_group *group, void *handle64);
fq_status fq_group_window(fq_ctx *ctx, const fq_group *group, void **dev_ptr, uint64_t *n_bytes);
fq_status fq_group_connect(fq_ctx *ctx, fq_group *group, const void *handles /* world x 64 bytes, rank order */);
fq_status fq_group_connect_ptrs(fq_ctx *ctx, fq_group *group, void *const *windows /* world device addresses */);
void fq_group_destroy(fq_ctx *ctx, fq_group *group);
/* group == NULL detaches the pipe; the group must outlive the pipes bound to it */
fq_status fq_pipe_set_group(fq_ctx *ctx, fq_pipe *pipe, fq_group *group);
/* like fq_pipe_fetch_aggregate, for the state merged over all ranks by the last launch (Count = rows of all ranks) */
fq_status fq_pipe_fetch_merged(fq_ctx *ctx, fq_pipe *pipe, fq_value *states, int32_t cap, int32_t *n_states,
                               uint64_t *rows_selected);
/* after fq_pipe_launch_project(pipe, ..., local_cols, local_valid, ...) on the same stream; final_* must hold
 * min(limit, world * capacity) rows; limit < 0 = none */
fq_status fq_group_gather_project(fq_ctx *ctx, fq_group *group, fq_pipe *pipe, fq_column *const *local_cols,
                                  fq_column *const *local_valid, fq_column *const *final_cols, fq_column *const *final_valid,
                                  int64_t limit, void *stream);
/* the same for columns the caller already holds (any producer): `rows_local` rows of `local_cols` (and `local_valid`, entries
 * may be NULL), `capacity` = the most rows any rank brings (the same value on every rank: it fixes the window layout) */
fq_status fq_group_gather_columns(fq_ctx *ctx, fq_group *group, const fq_column *const *local_cols, const fq_column *const *local_valid,
                                  int32_t n_cols, uint64_t rows_local, uint64_t rows_selected_local, uint64_t capacity,
                                  fq_column *const *final_cols, fq_column *const *final_valid, int64_t limit, void *stream);
fq_status fq_group_fetch_gather(fq_ctx *ctx, fq_group *group, uint64_t *rows_selected, uint64_t *rows_final);

/* ---- projection pipes: filter_record_batch + projection (+ LimitStream) in one pass ----
 * out_cols[i] receives select expression i for the rows that pass the predicate, in row order
 * (arrow filter keeps order, transform_filter.rs:51-54).  At most min(limit, capacity) rows are
 * written (limit < 0 = none; stream_limit.rs:28-48); rows_selected reports every matching row
 * unless FQ_RUN_LIMIT_EARLY_EXIT let the scan stop once `limit` rows were found (without a predicate:
 * after the 10 000-row reference block that completes the limit, like LimitStream stops pulling blocks). */
/* out_valid[i] (FQ_BOOL, one byte per output row) is required for expressions fq_pipe_expr_nullable reports; the
 * array itself may be NULL when no expression is nullable. */
fq_status fq_pipe_launch_project(fq_ctx *ctx, fq_pipe *pipe, const fq_source *src, fq_column *const *out_cols,
                                 fq_column *const *out_valid, uint64_t capacity, int64_t limit, uint32_t flags, void *stream);
fq_status fq_pipe_fetch_project(fq_ctx *ctx, fq_pipe *pipe, uint64_t *rows_selected, uint64_t *rows_written);
/* When the last launch filled min(limit, capacity) output rows: the source row (index into the launch's source) that
 * produced the LAST of them — the row that completes the LIMIT.  The reference evaluates predicate and projection over
 * every row of the 10 000-row block holding that row before LimitStream cuts it (transform_projection.rs:45-56 runs
 * before stream_limit.rs:28-48), and of the block after it (LimitStream polls its input before it checks its counter,
 * :58-62); a caller that wants exactly the reference's errors evaluates up to the end of that block and no further. */
fq_status fq_pipe_fetch_limit_row(fq_ctx *ctx, fq_pipe *pipe, uint64_t *row);

/* ---- ORDER BY ----
 * The reference lists sorting as not implemented (README.md:28; plan_parser.rs never reads `query.order_by`); the order is
 * arrow's with the crate's default SortOptions: ascending unless descending[j], NULLs first, ties in input order (stable),
 * floats by IEEE total order.  Several keys: lexicographic, keys[0] most significant.
 * fq_sort_indices writes the permutation (row indexes in sorted order, UInt32, so fewer than 2^32 rows) and fq_column_take
 * applies it to a column: out[i] = src[rows[i]], validity (bytes or bitmap) gathered into out_valid when the source has one.
 * Stable LSD radix sort, one pass per 8-bit digit that differs between some two rows; scratch is 24 bytes per row, kept by
 * the context between sorts (fq_ctx_trim returns it); sorts of one context run one at a time. */
fq_status fq_ctx_trim(fq_ctx *ctx);   /* frees cached scratch memory (synchronises the device) */
fq_status fq_sort_indices(fq_ctx *ctx, const fq_column *const *keys, const uint8_t *descending, int32_t n_keys, uint64_t n_rows,
                          fq_column *indices, void *stream);
/* ORDER BY ... LIMIT: the first min(limit, n_rows) indexes of the same order (`indices` needs only that many slots).  When one
 * NOT NULL key decides the order and the result is a small part of the table the rows are found by radix select (a
 * histogram and a partition per digit, from the most significant one down) and only what is left is sorted. */
fq_status fq_sort_indices_limit(fq_ctx *ctx, const fq_column *const *keys, const uint8_t *descending, int32_t n_keys, uint64_t n_rows,
                                uint64_t limit, fq_column *indices, uint64_t *n_out, void *stream);
fq_status fq_column_take(fq_ctx *ctx, const fq_column *src, const fq_column *rows, uint64_t n, fq_column *out, fq_column *out_valid,
                         void *stream);

/* ---- replaying a query: the launches of one or more pipes recorded once as a CUDA graph ----
 * The reference rebuilds its pipeline for every query (interpreter_select.rs:27-40); a prepared statement that is executed
 * again and again pays here only one graph launch instead of one launch per memset / probe / kernel / copy-back.
 *   fq_graph_begin(ctx, stream);  fq_pipe_launch_*(..., stream) ...;  fq_graph_end(ctx, stream, &g);
 *   for every execution: fq_graph_launch(ctx, g, stream);  fq_pipe_fetch_*(...) as after a direct launch.
 * Sources, output columns, limits and flags are frozen as recorded.  Between begin and end nothing runs; only launches
 * on `stream` belong to the recording, one recording at a time per context.  A pipe with a group attached is refused
 * (its merge carries an epoch that advances with every execution).  Lookup tables (fq_pipe_set_lookup) are frozen too: a
 * replay reads the tables that were bound when the launch was recorded, whatever is bound to the pipe since. */
typedef struct fq_graph fq_graph;
fq_status fq_graph_begin(fq_ctx *ctx, void *stream);
fq_status fq_graph_end(fq_ctx *ctx, void *stream, fq_graph **out);
fq_status fq_graph_launch(fq_ctx *ctx, fq_graph *graph, void *stream);
void fq_graph_destroy(fq_ctx *ctx, fq_graph *graph);

#ifdef __cplusplus
}
#endif
#endif /* FUSE_GPU_H */
