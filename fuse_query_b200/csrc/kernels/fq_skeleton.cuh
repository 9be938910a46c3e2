// fq_skeleton.cuh — hand-written sm_100a kernel skeletons of the fused fuse-query pipes.
//
// A pipe's expression trees are lowered by codegen.cc into a struct `Q` (typed row loaders, the WHERE
// predicate, per-row accumulate / projection code); the templates below supply everything around it:
// the coalesced 128-bit streaming loads, the register -> warp-shuffle -> shared-memory -> grid
// reductions, the ballot/popc stream compaction with a decoupled look-back across tiles.
//
// The same text is compiled twice: by nvcc into libfuse_gpu.so for the precompiled pipes
// (aot_kernels.cu) and by NVRTC at fq_pipe_compile time for any other expression tree.  It therefore
// includes nothing and relies on compiler builtins only.
//
// What each kernel replaces in the reference (/root/reference/src):
//   fq_agg_kernel     AggregatePartialTransform's loop (transforms/transform_aggregate_partial.rs:53-59) =
//                     per block, per aggregate: Function::eval of the argument (one Arrow pass and one
//                     intermediate array per node, datavalues/data_array_arithmetic.rs:14-55), one Arrow
//                     sum/min/max pass (data_array_aggregate.rs:103-114) and a scalar fold
//                     (functions/function_aggregator.rs:57-100) — here ONE pass, 8 B read per row.
//   fq_select_kernel  FilterTransform + ProjectionTransform (+ LimitStream): predicate -> BooleanArray ->
//                     filter_record_batch -> per-expression arrays (transform_filter.rs:38-55,
//                     transform_projection.rs:45-56, datastreams/stream_limit.rs:28-48).
//   fq_map_kernel     ProjectionTransform without a filter.
//   fq_fill_numbers   NumbersStream::poll_next (datasources/system/numbers_stream.rs:68-83).
#pragma once

typedef unsigned long long fq_u64;
typedef long long fq_i64;
typedef unsigned int fq_u32;
typedef int fq_i32;
typedef unsigned short fq_u16;
typedef short fq_i16;
typedef unsigned char fq_u8;
typedef signed char fq_i8;

#define FQ_E_DIVZERO 1u  // arrow DivideByZero

// launch shapes (the host reads the same macros through fq_skeleton_config.h)
#ifndef FQ_AGG_THREADS
#define FQ_AGG_THREADS 256
#define FQ_AGG_MIN_BLOCKS 4
#define FQ_TMA_THREADS 256   // consumer threads (+32 for the producer warp)
#define FQ_TMA_UNROLL 8      // tile = 256 * 8 vector groups = 32 KB of a UInt64 column per bulk copy
#define FQ_TMA_STAGES 8      // upper bound of the ring; the host picks stages so that ~128 KB are in flight per SM
#define FQ_TMA_MIN_BLOCKS 1
#define FQ_SEL_THREADS 352
#define FQ_SEL_MIN_BLOCKS 2
#define FQ_SEL_UNROLL 4
#define FQ_SEL_SEG 8
#define FQ_SEL_LOOK 5        // look-back window = 160 descriptors per poll (>= the CTAs of a 1-CTA/SM grid)
#define FQ_MAP_THREADS 256
#define FQ_MAP_MIN_BLOCKS 4
#define FQ_MAP_UNROLL 4
#endif
#ifndef FQ_GB_THREADS
#define FQ_GB_THREADS 256    // GROUP BY kernel
#define FQ_GB_MIN_BLOCKS 2
#endif
#ifndef FQ_GB_UNROLL
#define FQ_GB_UNROLL 4
#endif
#ifndef FQ_GB_ADMIT_SHIFT
#define FQ_GB_ADMIT_SHIFT 2  // the CTA's shared-memory table admits new keys until it is 1 - 2^-SHIFT full
#endif
#ifndef FQ_SELT_THREADS
#define FQ_SELT_THREADS 512  // staged select kernel, sparse-tuned build: consumer threads (+32 scan warp, +32 producer warp)
#define FQ_SELT_UNROLL 4     // tile = 512 * 4 vector groups = 32 KB of a UInt64 column per bulk copy
#define FQ_SELT_SEG 8        // tiles per segment (one look-back each): 256 KB of a UInt64 column
#define FQ_SELT_STAGES 8     // upper bound of the ring; the host picks the depth (~192 KB in flight per SM)
#define FQ_SELT_LAG 3        // pass 2 of SPARSE segments runs this many segments behind pass 1 (dense ones: 1)
#endif
// The dense-tuned build of the staged select kernel (fqk_*_select_dense): both passes through the ring, smaller tiles and
// segments so that what lies between a tile's two reads (one segment + the read-ahead, times 148 SMs) stays near 35 MB and
// the second read hits L2 (measured with ncu on 1e9 rows, every row kept: 14.2 GB from HBM for the 8 GB column with 28-KB
// tiles x 8, 8.2 GB with 14-KB tiles x 8).  The sparse-tuned build (fqk_*_select_tma) has no staged pass 2 compiled in.
#ifndef FQ_SELD_THREADS
#define FQ_SELD_THREADS 448  // + scan warp + producer warp = 16 warps: 128 registers per thread
#define FQ_SELD_UNROLL 2     // tile = 448 * 2 vector groups = 14 KB of a UInt64 column
#define FQ_SELD_SEG 8        // 112-KB segments
#define FQ_SELD_PROBE_ROWS 512   // rows per CTA of the density probe
#endif

#define FQ_STATE_HDR 6        // state / partial slots: [0] rows selected, [1] error bits, [2] launches folded, [3] rows scanned,
                              // [4] reference (10 000-row) blocks seen, [5] of which had no selected row (SURVEY F8)
#define FQ_REF_BLOCK_ROWS 10000ull   // NumbersStream block size, datasources/system/numbers_stream.rs:29
#define FQ_MAX_WARPS 32

// Kernel parameter block (one struct for every kernel so the host launch path is uniform).
struct fq_launch_params {
  fq_u64 n_rows;
  const void *cols[8];
  const void *cols_valid[8];  // per input column: validity — one byte per row (1 = valid), or an Arrow LSB-first bitmap (the pipe is
                              // compiled for one or the other), or null when the column is NOT NULL
  fq_u64 cols_valid_bit0[8];  // bitmap validity: bit of row 0 of the source
  fq_u64 numbers_begin;  // generated mode: column 0 = numbers_begin + row
  // bit tables of the pipe's FQ_EXPR_LOOKUP nodes (FQ_MAX_LOOKUPS slots): LSB-first bitmaps, read a byte at a time so that a
  // table needs no alignment and no padding past its last byte; the row functions (pred, consume, gb_row, emit) receive them here
  const fq_u8 *lookup[4];
  fq_u64 lookup_bits[4];
  // aggregate
  fq_u64 *partials;      // [gridDim.x][FQ_STATE_HDR + Q::NSLOTS]
  fq_u64 *state;         // [FQ_STATE_HDR + Q::NSLOTS] running state of the pipe
  fq_u32 *ticket;
  fq_u32 accumulate;
  fq_u32 *block_hit;     // one bit per reference block of this launch (zeroed before it), or null: block tracking off
  fq_u32 stages;         // bulk-copy staged kernel: ring depth actually used (<= its STAGES template bound)
  fq_u32 stages2;        // staged select kernel: != 0 when pass 2 of dense segments is staged too (slots hold every referenced column)
  const fq_u32 *sel_mode; // null, or which build of the staged select kernel runs: 0 sparse-tuned, 1 dense-tuned (written by the probe)
  fq_u32 *probe;          // density probe: [0] rows sampled, [1] rows kept, [2] = the mode it decided
  fq_u32 bits_unstaged;  // a validity bitmap starts off the 128-row grid: the host launches the LDG variant (no bulk copies)
  fq_u32 unaligned;      // some input column (a slice) does not start on a 16-byte boundary: no vector / bulk loads, every row by fq_ld1
  // multi-GPU merge point fused into the aggregate kernel (fq_group, include/fuse_gpu.h): after the fold the last CTA
  // stores the running state into its row of EVERY rank's exchange window (peer GPUs' memory over NVLink), waits until
  // every rank's row of this epoch has arrived in its own window, folds them in rank order and writes `merged`.
  // Window layout: [parity = epoch & 1][writer rank][group_row_slots] 8-byte slots, slot 0 of a row = the epoch it holds.
  // group_world = 0: off
  fq_u64 *group_windows[8];
  fq_u64 group_epoch;
  fq_u64 group_timeout_ns;
  fq_u64 *merged;          // [FQ_STATE_HDR + Q::NSLOTS] merged state of all ranks (local)
  fq_u64 *host_state;      // pinned host mirrors of `state` / `merged`, written by the kernel itself (no copy operation queued
  fq_u64 *host_merged;     // behind the launch: a 10^7-row query is launch-latency bound and the copy cost as much as the kernel)
  fq_u32 group_rank, group_world, group_row_slots;
  // group by: open-addressing table in HBM, gb_cap (a power of two) slots + 1 for the key that equals the EMPTY mark
  fq_u64 *gb_keys;        // [gb_cap + 1] packed keys (Q::Key: one or two words), every word FQ_GB_EMPTY = free
  fq_u64 *gb_slots;       // [gb_cap + 1][Q::G] group states
  fq_u64 gb_cap;
  fq_u32 *gb_flags;       // [0] != 0: the table overflowed (results void), [1] != 0: the EMPTY-valued key occurred
  fq_u32 gb_smem_cap;     // slots of the CTA's shared-memory table (a power of two, 0 = none)
  const fq_u64 *gb_entries;  // merge kernel: n_rows partial entries of KW + Q::G slots each (packed key's KW words, state)
  fq_u64 *gb_rep_keys;    // [gb_reps - 1][gb_cap + 1] replicas of the table: CTA b aggregates into replica b % gb_reps (0 = the
  fq_u64 *gb_rep_slots;   // table itself), the merge kernel folds them into the table and leaves them empty again
  fq_u32 gb_reps;         // >= 1
  fq_u64 gb_seed;         // xored into every key before it is hashed for this table's slots (0 at a pipe's first reservation)
  // select / map
  void *outs[8];
  void *outs_valid[8];   // per select expression that can yield NULL: one byte per output row
  fq_u64 capacity;       // rows written are those with rank < capacity (min(limit, capacity) on the host)
  fq_u64 *tile_status;   // decoupled look-back descriptors, zeroed before the launch
  fq_u32 *tile_counter;  // dynamic tile ids (forward progress for the look-back), zeroed before the launch
  fq_u64 *result;        // [0] rows selected, [1] error bits, [5] source row of output row capacity - 1 (the row that completes a LIMIT)
  fq_u64 n_tiles;
  fq_u64 stop_after;     // early exit: stop scanning once this many rows were selected (0 = never)
  fq_u32 *done;          // early-exit flag, zeroed before the launch
};

// ---------------------------------------------------------------------------------------------
// memory access helpers
// ---------------------------------------------------------------------------------------------
struct fq_b16 { fq_u32 x, y, z, w; };

// streaming 128-bit load: read-only path, do not allocate in L1 (every byte is touched once)
__device__ __forceinline__ fq_b16 fq_ld16(const void *p) {
  fq_b16 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ fq_u64 fq_ld_volatile(const fq_u64 *p) {
  fq_u64 v;
  asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void fq_st_volatile(fq_u64 *p, fq_u64 v) {
  asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ fq_u32 fq_ld_volatile32(const fq_u32 *p) {
  fq_u32 v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ fq_u64 fq_ld_cg(const fq_u64 *p) {
  fq_u64 v;
  asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(p));
  return v;
}

// Arrow validity bitmaps, read in place (datablocks/data_block.rs:10-14 columns are arrow arrays: LSB-first, bit = 1 valid).
// A thread owns V consecutive rows, i.e. V consecutive bits: one byte (two for V = 16) that the neighbouring lanes share,
// so a warp load touches 32 * V / 8 bytes of the bitmap — 1/64 of the traffic of a UInt64 column, 1/8 of a UInt8 one,
// instead of one validity BYTE per row.  `bit` is a multiple of V on the vector path (the host routes anything else
// through the row-by-row path).
__device__ __forceinline__ bool fq_ld_bit(const void *bitmap, fq_u64 bit) {
  return (__ldg((const fq_u8 *)bitmap + (bit >> 3)) >> (bit & 7)) & 1u;
}
template <int V> __device__ __forceinline__ void fq_load_bits(bool (&dst)[V], const void *bitmap, fq_u64 bit) {
  if constexpr (V <= 8) {
    const fq_u32 w = (fq_u32)__ldg((const fq_u8 *)bitmap + (bit >> 3)) >> (bit & 7);
#pragma unroll
    for (int v = 0; v < V; v++) dst[v] = (w >> v) & 1u;
  } else {
#pragma unroll
    for (int b = 0; b < V / 8; b++) {
      const fq_u32 w = __ldg((const fq_u8 *)bitmap + (bit >> 3) + b);
#pragma unroll
      for (int v = 0; v < 8; v++) dst[8 * b + v] = (w >> v) & 1u;
    }
  }
}

// FQ_EXPR_LOOKUP: bit c of a bit table of n bits, false at or beyond n (the table of an empty dictionary has no bits)
__device__ __forceinline__ bool fq_lookup(const fq_u8 *table, fq_u64 n, fq_u64 c) {
  return c < n && ((__ldg(table + (c >> 3)) >> (c & 7)) & 1u);
}

// one value (scalar tails, ragged last tile)
template <class T> __device__ __forceinline__ T fq_ld1(const void *base, fq_u64 row) { return __ldg((const T *)base + row); }
template <> __device__ __forceinline__ bool fq_ld1<bool>(const void *base, fq_u64 row) { return __ldg((const fq_u8 *)base + row) != 0; }

// Load V consecutive values of type T (V * sizeof(T) bytes, a multiple of 16 or a power of two below)
template <class T, int V>
__device__ __forceinline__ void fq_load_vec(T (&dst)[V], const void *base, fq_u64 group) {
  constexpr int BYTES = V * (int)sizeof(T);
  const char *p = (const char *)base + group * (fq_u64)BYTES;
  if constexpr (BYTES >= 16) {
    union { fq_b16 q[BYTES / 16]; T t[V]; } u;
#pragma unroll
    for (int k = 0; k < BYTES / 16; k++) u.q[k] = fq_ld16(p + 16 * k);
#pragma unroll
    for (int k = 0; k < V; k++) dst[k] = u.t[k];
  } else if constexpr (BYTES == 8) {
    union { fq_u64 q; T t[V]; } u;
    u.q = __ldg((const fq_u64 *)p);
#pragma unroll
    for (int k = 0; k < V; k++) dst[k] = u.t[k];
  } else if constexpr (BYTES == 4) {
    union { fq_u32 q; T t[V]; } u;
    u.q = __ldg((const fq_u32 *)p);
#pragma unroll
    for (int k = 0; k < V; k++) dst[k] = u.t[k];
  } else {
#pragma unroll
    for (int k = 0; k < V; k++) dst[k] = fq_ld1<T>(p, k);
  }
}

// Outputs are written once and never read by the kernel: streaming stores (.cs: evict-first) keep them from pushing the
// input lines that pass 2 of the select kernel will read again out of L2.
#ifndef FQ_STORE_CS
#define FQ_STORE_CS 1
#endif
template <class T> __device__ __forceinline__ void fq_st1(void *base, fq_u64 idx, T v) {
#if FQ_STORE_CS
  __stcs((T *)base + idx, v);
#else
  ((T *)base)[idx] = v;
#endif
}
// Store V consecutive values (the mirror of fq_load_vec): one 16/8/4/2-byte store when the run is that wide.
// `base + first` is aligned to V * sizeof(T) because vector groups start at multiples of V rows.
template <class T, int V>
__device__ __forceinline__ void fq_store_vec(void *base, fq_u64 first, const T (&src)[V]) {
  constexpr int BYTES = V * (int)sizeof(T);
  char *p = (char *)base + first * sizeof(T);
  if constexpr (BYTES >= 16) {
    union { fq_b16 q[BYTES / 16]; T t[V]; } u;
#pragma unroll
    for (int k = 0; k < V; k++) u.t[k] = src[k];
#pragma unroll
    for (int k = 0; k < BYTES / 16; k++) {
#if FQ_STORE_CS
      asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p + 16 * k), "r"(u.q[k].x), "r"(u.q[k].y), "r"(u.q[k].z), "r"(u.q[k].w) : "memory");
#else
      asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p + 16 * k), "r"(u.q[k].x), "r"(u.q[k].y), "r"(u.q[k].z), "r"(u.q[k].w) : "memory");
#endif
    }
  } else if constexpr (BYTES == 8) {
    union { fq_u64 q; T t[V]; } u;
#pragma unroll
    for (int k = 0; k < V; k++) u.t[k] = src[k];
    *(fq_u64 *)p = u.q;
  } else if constexpr (BYTES == 4) {
    union { fq_u32 q; T t[V]; } u;
#pragma unroll
    for (int k = 0; k < V; k++) u.t[k] = src[k];
    *(fq_u32 *)p = u.q;
  } else if constexpr (BYTES == 2) {
    union { fq_u16 q; T t[V]; } u;
#pragma unroll
    for (int k = 0; k < V; k++) u.t[k] = src[k];
    *(fq_u16 *)p = u.q;
  } else {
#pragma unroll
    for (int k = 0; k < V; k++) ((T *)p)[k] = src[k];
  }
}

// ---------------------------------------------------------------------------------------------
// arithmetic helpers used by generated code (semantics of arrow 2.0 as the reference calls it)
// ---------------------------------------------------------------------------------------------
template <class T> struct fq_traits;
#define FQ_TRAITS(T, UT, ISF, ISS, LO, HI)                                          \
  template <> struct fq_traits<T> {                                                 \
    typedef UT unsigned_t;                                                          \
    enum { is_float = ISF, is_signed = ISS };                                       \
    __device__ static __forceinline__ T lo() { return LO; }                         \
    __device__ static __forceinline__ T hi() { return HI; }                         \
  };
FQ_TRAITS(fq_i8, fq_u8, 0, 1, (fq_i8)-128, (fq_i8)127)
FQ_TRAITS(fq_i16, fq_u16, 0, 1, (fq_i16)-32768, (fq_i16)32767)
FQ_TRAITS(fq_i32, fq_u32, 0, 1, (fq_i32)(-2147483647 - 1), (fq_i32)2147483647)
FQ_TRAITS(fq_i64, fq_u64, 0, 1, (fq_i64)(-9223372036854775807ll - 1), (fq_i64)9223372036854775807ll)
FQ_TRAITS(fq_u8, fq_u8, 0, 0, (fq_u8)0, (fq_u8)255)
FQ_TRAITS(fq_u16, fq_u16, 0, 0, (fq_u16)0, (fq_u16)65535)
FQ_TRAITS(fq_u32, fq_u32, 0, 0, 0u, 4294967295u)
FQ_TRAITS(fq_u64, fq_u64, 0, 0, 0ull, 18446744073709551615ull)
FQ_TRAITS(float, float, 1, 1, -__int_as_float(0x7f800000), __int_as_float(0x7f800000))
FQ_TRAITS(double, double, 1, 1, -__longlong_as_double(0x7ff0000000000000ll), __longlong_as_double(0x7ff0000000000000ll))
#undef FQ_TRAITS

// wrapping integer add / sub / mul (arrow `add` etc. on integer lanes).  Float lanes use the round-to-nearest
// intrinsics, which the compiler never contracts into FMAs: `a * b + c` must round twice like the reference's
// separate Arrow passes do (a contracted FMA differs in the last bit).
__device__ __forceinline__ float fq_fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double fq_fadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float fq_fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double fq_fsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float fq_fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double fq_fmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float fq_fdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double fq_fdiv(double a, double b) { return __ddiv_rn(a, b); }
template <class T> __device__ __forceinline__ T fq_add(T a, T b) {
  if constexpr (fq_traits<T>::is_float) return fq_fadd(a, b);
  else { typedef typename fq_traits<T>::unsigned_t U; return (T)(U)((U)a + (U)b); }
}
template <class T> __device__ __forceinline__ T fq_sub(T a, T b) {
  if constexpr (fq_traits<T>::is_float) return fq_fsub(a, b);
  else { typedef typename fq_traits<T>::unsigned_t U; return (T)(U)((U)a - (U)b); }
}
template <class T> __device__ __forceinline__ T fq_mul(T a, T b) {
  if constexpr (fq_traits<T>::is_float) return fq_fmul(a, b);
  else { typedef typename fq_traits<T>::unsigned_t U; return (T)(U)((U)a * (U)b); }
}
// arrow `divide`: a zero divisor in a VALID slot is an error (integer and float lanes alike; null slots are skipped,
// math_divide checks the combined validity bitmap first); integers truncate
template <class T> __device__ __forceinline__ T fq_div(T a, T b, bool valid, fq_u32 &err) {
  if (b == (T)0) {
    if (valid) err |= FQ_E_DIVZERO;
    return (T)0;
  }
  if constexpr (fq_traits<T>::is_float) return fq_fdiv(a, b);
  else if constexpr (fq_traits<T>::is_signed) {
    typedef typename fq_traits<T>::unsigned_t U;
    if (b == (T)-1) return (T)(U)((U)0 - (U)a);  // MIN / -1 wraps instead of trapping
    return (T)(a / b);
  } else return (T)(a / b);
}
template <class T> __device__ __forceinline__ T fq_min(T a, T b) { return b < a ? b : a; }
template <class T> __device__ __forceinline__ T fq_max(T a, T b) { return b > a ? b : a; }

// arrow numeric `cast` (num::cast): a value that does not fit the target becomes NULL.  fq_cast_ok says whether the
// value is representable, fq_cast_v converts it (0 when it is not); codegen ANDs fq_cast_ok into the row's validity.
template <class T, class S> __device__ __forceinline__ bool fq_cast_ok(S x) {
  if constexpr (fq_traits<T>::is_float) return true;
  else if constexpr (fq_traits<S>::is_float) {
    const double d = (double)x;
    if (d != d) return false;
    const double t = d < 0 ? -floor(-d) : floor(d);
    if constexpr (sizeof(T) == 8 && fq_traits<T>::is_signed) return t >= -9223372036854775808.0 && t < 9223372036854775808.0;
    else if constexpr (sizeof(T) == 8) return t > -1.0 && t < 18446744073709551616.0;
    else return t >= (double)fq_traits<T>::lo() && t <= (double)fq_traits<T>::hi();
  } else if constexpr (fq_traits<S>::is_signed && !fq_traits<T>::is_signed) {
    return x >= 0 && (fq_u64)x <= (fq_u64)fq_traits<T>::hi();
  } else if constexpr (!fq_traits<S>::is_signed && fq_traits<T>::is_signed) {
    return (fq_u64)x <= (fq_u64)fq_traits<T>::hi();
  } else {
    if constexpr (sizeof(S) > sizeof(T)) return x >= (S)fq_traits<T>::lo() && x <= (S)fq_traits<T>::hi();
    else return true;
  }
}
template <class T, class S> __device__ __forceinline__ T fq_cast_v(S x) {
  if constexpr (fq_traits<S>::is_float && !fq_traits<T>::is_float) {
    if (!fq_cast_ok<T, S>(x)) return (T)0;
    const double d = (double)x;
    return (T)(d < 0 ? -floor(-d) : floor(d));
  } else {
    return (T)x;
  }
}

// 64-bit slot packing of accumulator values (what crosses to the host / between launches)
template <class T> __device__ __forceinline__ fq_u64 fq_pack(T x) {
  if constexpr (fq_traits<T>::is_float) return (fq_u64)__double_as_longlong((double)x);
  else if constexpr (fq_traits<T>::is_signed) return (fq_u64)(fq_i64)x;
  else return (fq_u64)x;
}
template <class T> __device__ __forceinline__ T fq_unpack(fq_u64 s) {
  if constexpr (fq_traits<T>::is_float) return (T)__longlong_as_double((fq_i64)s);
  else return (T)s;
}
template <class T> __device__ __forceinline__ T fq_shfl_xor(T x, int m) {
  if constexpr (sizeof(T) == 8) return fq_unpack<T>(__shfl_xor_sync(0xffffffffu, fq_pack<T>(x), m));
  else if constexpr (fq_traits<T>::is_float) return __shfl_xor_sync(0xffffffffu, x, m);
  else return (T)__shfl_xor_sync(0xffffffffu, (fq_i32)x, m);
}

// ---------------------------------------------------------------------------------------------
// block-level reduction of a generated accumulator:  registers -> warp shuffles -> shared -> warp 0
// result valid in thread 0
// ---------------------------------------------------------------------------------------------
template <class Q>
__device__ __forceinline__ void fq_block_reduce(typename Q::Acc &acc, fq_u64 &nsel, fq_u32 &err,
                                                fq_u64 (*sm)[FQ_STATE_HDR + Q::NSLOTS]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) {
    typename Q::Acc o = acc;
    Q::shfl(o, m);
    Q::merge(acc, o);
    nsel += __shfl_xor_sync(0xffffffffu, nsel, m);
    err |= __shfl_xor_sync(0xffffffffu, err, m);
  }
  __syncthreads();  // sm may still be read by a previous use
  if (lane == 0) {
    sm[warp][0] = nsel;
    sm[warp][1] = err;
    Q::store(acc, &sm[warp][FQ_STATE_HDR]);
  }
  __syncthreads();
  if (warp == 0) {
    Q::init(acc);
    nsel = 0;
    err = 0;
    if (lane < nwarps) {
      nsel = sm[lane][0];
      err = (fq_u32)sm[lane][1];
      Q::unpack(acc, &sm[lane][FQ_STATE_HDR]);
    }
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) {
      typename Q::Acc o = acc;
      Q::shfl(o, m);
      Q::merge(acc, o);
      nsel += __shfl_xor_sync(0xffffffffu, nsel, m);
      err |= __shfl_xor_sync(0xffffffffu, err, m);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Reference-block tracking (SURVEY F8).  The reference folds Sum per 10 000-row block: a block in which the WHERE
// clause keeps no row yields arrow sum(empty) = None, and `state + None` fails ("DataValue to array cannot be NONE",
// datavalues/data_value.rs:104-109 via data_value_arithmetic.rs:19-24).  To be able to report the same outcome the
// fused scan records which reference blocks saw at least one selected row: one bit per block, warp-aggregated.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void fq_mark_one(fq_u32 *hit, fq_u64 blk) {
  fq_u32 *w = hit + (blk >> 5);
  const fq_u32 bit = 1u << (blk & 31);
  if (!(*(volatile fq_u32 *)w & bit)) atomicOr(w, bit);
}
// per-lane form (divergent callers): `kept` has bit v set when row row0 + v was selected
template <int V> __device__ __forceinline__ void fq_mark_blocks_lane(const fq_launch_params &p, fq_u64 row0, fq_u32 kept) {
  if (!kept) return;
  const fq_u64 first = row0 / FQ_REF_BLOCK_ROWS, last = (row0 + V - 1) / FQ_REF_BLOCK_ROWS;
  if (first == last) { fq_mark_one(p.block_hit, first); return; }
#pragma unroll
  for (int v = 0; v < V; v++)
    if ((kept >> v) & 1u) fq_mark_one(p.block_hit, (row0 + v) / FQ_REF_BLOCK_ROWS);
}
// whole-warp form: the lanes hold 32 consecutive vector groups (32 * V consecutive rows)
template <int V> __device__ __forceinline__ void fq_mark_blocks_warp(const fq_launch_params &p, fq_u64 row0, fq_u32 kept) {
  if (!__any_sync(0xffffffffu, kept != 0)) return;
  const fq_u64 first = __shfl_sync(0xffffffffu, row0, 0) / FQ_REF_BLOCK_ROWS;
  const fq_u64 last = (__shfl_sync(0xffffffffu, row0, 31) + V - 1) / FQ_REF_BLOCK_ROWS;
  if (first == last) {
    if ((threadIdx.x & 31) == 0) fq_mark_one(p.block_hit, first);
  } else {
    fq_mark_blocks_lane<V>(p, row0, kept);
  }
}

#define FQ_E_MERGE_TIMEOUT 2u  // a rank's state did not arrive in the exchange window in time

// Out of line (see fq_group_merge): the running state into its pinned host mirror, posted writes over PCIe
static __device__ __noinline__ void fq_mirror_state(fq_u64 *host, const fq_u64 *dev, int n) {
  for (int k = 0; k < n; k++) host[k] = dev[k];
  __threadfence_system();
}


__device__ __forceinline__ void fq_st_release_sys(fq_u64 *p, fq_u64 v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ fq_u64 fq_ld_acquire_sys(const fq_u64 *p) {
  fq_u64 v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ fq_u64 fq_globaltimer() {
  fq_u64 t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// Row of `writer` in a window, for the epoch's parity.  A rank can be at most one epoch ahead of another (it cannot finish
// epoch e + 1 before every rank has published e + 1, which they do after finishing e), so two row sets suffice.
__device__ __forceinline__ fq_u64 *fq_group_row(const fq_launch_params &p, int window_of, int writer) {
  return p.group_windows[window_of] + ((p.group_epoch & 1ull) * p.group_world + (fq_u64)writer) * p.group_row_slots;
}
// lanes 0 .. world-1 of one warp: lane r stores `n` payload slots into this rank's row of rank r's window, then the epoch
// (release at system scope: the payload is visible to whoever acquires the epoch).  Returns after the stores were issued.
__device__ __forceinline__ void fq_group_publish(const fq_launch_params &p, const fq_u64 *payload, int n) {
  const int lane = threadIdx.x & 31;
  if (lane < (int)p.group_world) {
    fq_u64 *row = fq_group_row(p, lane, (int)p.group_rank);
    for (int k = 0; k < n; k++) row[1 + k] = payload[k];
    __threadfence_system();
    fq_st_release_sys(row, p.group_epoch);
  }
}
// lanes 0 .. world-1: lane r waits for rank r's row of this epoch in the LOCAL window; false on timeout (a dead peer must
// not hang the GPU: the caller reports FQ_E_MERGE_TIMEOUT)
__device__ __forceinline__ bool fq_group_wait(const fq_launch_params &p) {
  const int lane = threadIdx.x & 31;
  bool ok = true;
  if (lane < (int)p.group_world) {
    const fq_u64 *row = fq_group_row(p, (int)p.group_rank, lane);
    const fq_u64 t0 = fq_globaltimer();
    while (fq_ld_acquire_sys(row) != p.group_epoch) {
      if (fq_globaltimer() - t0 > p.group_timeout_ns) { ok = false; break; }
    }
  }
  return __all_sync(0xffffffffu, ok);
}

// The exchange + final fold of the merge point (processors/processor_merge.rs:37-66 feeding
// transforms/transform_aggregate_final.rs:50-78), run by warp 0 of the aggregate kernel's last CTA.  Out of line on
// purpose: inlined, this cold code changed the register allocation and unrolling of the hot loops of the ALU-bound
// generated-source kernels (sum(number) over 1e10 generated rows: 1.15 -> 1.70 ms).
template <class Q>
static __device__ __noinline__ void fq_group_merge(const fq_launch_params &p) {
  constexpr int S = FQ_STATE_HDR + Q::NSLOTS;
  fq_group_publish(p, p.state, S);
  const bool ok = fq_group_wait(p);
  if ((threadIdx.x & 31) == 0) {
    typename Q::Acc acc;
    Q::init(acc);
    fq_u64 hdr[FQ_STATE_HDR];
#pragma unroll
    for (int k = 0; k < FQ_STATE_HDR; k++) hdr[k] = 0;
    for (int r = 0; r < (int)p.group_world; r++) {   // rank order = partition order: float sums fold deterministically
      const fq_u64 *row = fq_group_row(p, (int)p.group_rank, r) + 1;
      fq_u64 tmp[Q::NSLOTS > 0 ? Q::NSLOTS : 1];
#pragma unroll
      for (int k = 0; k < Q::NSLOTS; k++) tmp[k] = fq_ld_cg(row + FQ_STATE_HDR + k);
      typename Q::Acc o;
      Q::unpack(o, tmp);
      Q::merge(acc, o);
#pragma unroll
      for (int k = 0; k < FQ_STATE_HDR; k++) {
        const fq_u64 x = fq_ld_cg(row + k);
        hdr[k] = k == 1 ? (hdr[k] | x) : (hdr[k] + x);
      }
    }
    if (!ok) hdr[1] |= FQ_E_MERGE_TIMEOUT;
#pragma unroll
    for (int k = 0; k < FQ_STATE_HDR; k++) p.merged[k] = hdr[k];
    Q::store(acc, p.merged + FQ_STATE_HDR);
    if (p.host_merged) fq_mirror_state(p.host_merged, p.merged, S);
  }
}

// CTA partial -> global partial row -> last CTA (ticket) folds every partial into (or restarts) the running state
template <class Q>
__device__ __forceinline__ void fq_agg_finish(const fq_launch_params &p, typename Q::Acc &acc, fq_u64 &nsel, fq_u32 &err,
                                              fq_u64 (*sm)[FQ_STATE_HDR + Q::NSLOTS], fq_u32 *s_last_p, fq_u32 *s_hits_p) {
  constexpr int S = FQ_STATE_HDR + Q::NSLOTS;
  fq_u32 &s_last = *s_last_p;
  fq_u32 &s_hits = *s_hits_p;
  fq_block_reduce<Q>(acc, nsel, err, sm);
  if (threadIdx.x == 0) {
    fq_u64 *out = p.partials + (fq_u64)blockIdx.x * S;
    out[0] = nsel;
    out[1] = err;
    Q::store(acc, out + FQ_STATE_HDR);
    __threadfence();
    s_last = (atomicAdd(p.ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
    s_hits = 0;
  }
  __syncthreads();
  if (!s_last) return;

  // reference blocks of this launch that saw a selected row
  fq_u64 ref_blocks = 0;
  if constexpr (Q::TRACK_BLOCKS) {
    if (p.block_hit) {
      ref_blocks = (p.n_rows + FQ_REF_BLOCK_ROWS - 1) / FQ_REF_BLOCK_ROWS;
      const fq_u64 words = (ref_blocks + 31) / 32;
      fq_u32 h = 0;
      for (fq_u64 w = threadIdx.x; w < words; w += blockDim.x) {
        fq_u32 x;
        asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(x) : "l"(p.block_hit + w));
        h += __popc(x);
      }
      if (h) atomicAdd(&s_hits, h);
    }
  }

  // last CTA: fold every CTA's partial, then fold into (or restart) the running state
  __threadfence();
  Q::init(acc);
  nsel = 0;
  err = 0;
  for (fq_u32 i = threadIdx.x; i < gridDim.x; i += blockDim.x) {
    const fq_u64 *in = p.partials + (fq_u64)i * S;
    fq_u64 tmp[Q::NSLOTS > 0 ? Q::NSLOTS : 1];
#pragma unroll
    for (int k = 0; k < Q::NSLOTS; k++) tmp[k] = fq_ld_cg(in + FQ_STATE_HDR + k);
    typename Q::Acc o;
    Q::unpack(o, tmp);
    Q::merge(acc, o);
    nsel += fq_ld_cg(in);
    err |= (fq_u32)fq_ld_cg(in + 1);
  }
  fq_block_reduce<Q>(acc, nsel, err, sm);
  if (threadIdx.x == 0) {
    if (!Q::HAS_PRED) nsel = p.n_rows;
    fq_u64 folded = 1, scanned = p.n_rows;
    fq_u64 blocks = ref_blocks, empty_blocks = ref_blocks - s_hits;   // s_hits is complete: fq_block_reduce synchronised the CTA
    if (p.accumulate) {
      typename Q::Acc o;
      Q::unpack(o, p.state + FQ_STATE_HDR);
      Q::merge(acc, o);
      nsel += p.state[0];
      err |= (fq_u32)p.state[1];
      folded += p.state[2];
      scanned += p.state[3];
      blocks += p.state[4];
      empty_blocks += p.state[5];
    }
    p.state[0] = nsel;
    p.state[1] = err;
    p.state[2] = folded;
    p.state[3] = scanned;
    p.state[4] = blocks;
    p.state[5] = empty_blocks;
    Q::store(acc, p.state + FQ_STATE_HDR);
    *p.ticket = 0;
    if (p.host_state) fq_mirror_state(p.host_state, p.state, S);
  }
  // the merge point across GPUs, fused: exchange over peer memory + final fold (see fq_group_merge)
  if (p.group_world) {
    __syncthreads();   // p.state is complete
    if (threadIdx.x < 32) fq_group_merge<Q>(p);
  }
}

// ---------------------------------------------------------------------------------------------
// fq_agg_kernel — single-pass multi-aggregate scan.
//
// Grid: persistent, (SM count x resident CTAs) blocks.  Each CTA walks contiguous chunks of
// blockDim.x * UNROLL vector groups (16 B per thread per load, UNROLL independent loads in flight
// per thread, consecutive lanes on consecutive 16-B words -> every warp load is one 512-B run).
// Algorithmic traffic: sizeof(row) bytes read per row, (FQ_STATE_HDR + NSLOTS) * 8 B written per CTA.
// ---------------------------------------------------------------------------------------------
template <class Q, int UNROLL>
__device__ __forceinline__ void fq_agg_kernel(const fq_launch_params &p) {
  constexpr int V = Q::V;
  constexpr int S = FQ_STATE_HDR + Q::NSLOTS;
  __shared__ fq_u64 sm[FQ_MAX_WARPS][S];
  __shared__ fq_u32 s_last;
  __shared__ fq_u32 s_hits;

  typename Q::Acc acc;
  Q::init(acc);
  fq_u32 err = 0;
  fq_u64 nsel = 0;

  const fq_u64 nvec = p.unaligned ? 0 : p.n_rows / V;   // unaligned slices: everything through the row-by-row tail
  const fq_u64 chunk = (fq_u64)blockDim.x * UNROLL;
  const fq_u64 nfull = nvec / chunk;
  for (fq_u64 c = blockIdx.x; c < nfull; c += gridDim.x) {
    const fq_u64 g0 = c * chunk + threadIdx.x;
    typename Q::Rows rows[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; u++) Q::load(rows[u], p, g0 + (fq_u64)u * blockDim.x);
#pragma unroll
    for (int u = 0; u < UNROLL; u++) {
      fq_u32 kept = 0;
#pragma unroll
      for (int v = 0; v < V; v++) kept |= (Q::consume(p, acc, rows[u], v, nsel, err) ? 1u : 0u) << v;
      if constexpr (Q::TRACK_BLOCKS) {
        if (p.block_hit) fq_mark_blocks_warp<V>(p, (g0 + (fq_u64)u * blockDim.x) * V, kept);
      }
    }
  }
  // remainder groups (< one chunk) and the scalar tail (< V rows), spread over the whole grid
  const fq_u64 tid = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x;
  const fq_u64 nthreads = (fq_u64)gridDim.x * blockDim.x;
  for (fq_u64 g = nfull * chunk + tid; g < nvec; g += nthreads) {
    typename Q::Rows r;
    Q::load(r, p, g);
    fq_u32 kept = 0;
#pragma unroll
    for (int v = 0; v < V; v++) kept |= (Q::consume(p, acc, r, v, nsel, err) ? 1u : 0u) << v;
    if constexpr (Q::TRACK_BLOCKS) {
      if (p.block_hit) fq_mark_blocks_lane<V>(p, g * V, kept);
    }
  }
  for (fq_u64 row = nvec * V + tid; row < p.n_rows; row += nthreads) {
    typename Q::Rows r;
    Q::load1(r, p, row);
    const bool kept = Q::consume(p, acc, r, 0, nsel, err);
    if constexpr (Q::TRACK_BLOCKS) {
      if (p.block_hit && kept) fq_mark_one(p.block_hit, row / FQ_REF_BLOCK_ROWS);
    }
  }

  fq_agg_finish<Q>(p, acc, nsel, err, sm, &s_last, &s_hits);
}

// ---------------------------------------------------------------------------------------------
// fq_agg_tma_kernel — the same single-pass multi-aggregate scan, staged through shared memory by the bulk-copy
// engine (cp.async.bulk, SASS UBLKCP) instead of per-thread LDG.
//
// CTA = C consumer warps + 1 producer warp.  Tile = 32 * C * U vector groups of every referenced column; a ring
// of STAGES tiles lives in dynamic shared memory.  Producer (one elected lane): wait empty[s] -> arrive.expect_tx
// full[s] -> one cp.async.bulk per column (contiguous tile_rows * sizeof(T) bytes, completes on full[s]).
// Consumers: wait full[s] -> LDS.128 (consecutive lanes on consecutive 16-B words: conflict-free) -> accumulate in
// registers -> one arrive per warp on empty[s].  Bytes in flight are set by stages * tile bytes, not by registers:
// one CTA per SM with 4 x 32 KB measured best on B200 (10.70 ms for 80 GB vs 11.04 ms for the LDG kernel; more
// than 128 KB in flight per SM is slower again).  Rows past the last full tile take the LDG path.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ fq_u32 fq_smem_addr(const void *p) { return (fq_u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void fq_mbar_init(fq_u32 bar, fq_u32 count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fq_mbar_expect_tx(fq_u32 bar, fq_u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fq_mbar_arrive(fq_u32 bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void fq_mbar_wait(fq_u32 bar, fq_u32 parity) {
  fq_u32 ok;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  } while (!ok);
}
// global -> shared bulk copy (16-byte aligned, size a multiple of 16), completion counted in bytes on `bar`.
// HINT: L2 eviction priority of the lines the copy touches — 0 default, 1 evict_last (they will be read again: pass 1 of
// the select kernel), 2 evict_first (last use: its pass 2).
#ifndef FQ_L2_HINTS
#define FQ_L2_HINTS 1
#endif
template <int HINT = 0>
__device__ __forceinline__ void fq_bulk_g2s(fq_u32 dst, const void *src, fq_u32 bytes, fq_u32 bar) {
  if constexpr (HINT == 0 || !FQ_L2_HINTS) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
  } else {
    fq_u64 pol;
    if constexpr (HINT == 1) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    else asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
  }
}
// V consecutive values of one staged column from shared memory
template <class T, int V>
__device__ __forceinline__ void fq_lds_vec(T (&dst)[V], const unsigned char *col, fq_u32 group) {
  constexpr int BYTES = V * (int)sizeof(T);
  if constexpr (BYTES >= 16) {
    union { uint4 q[BYTES / 16]; T t[V]; } u;
#pragma unroll
    for (int k = 0; k < BYTES / 16; k++) u.q[k] = *(const uint4 *)(col + (size_t)group * BYTES + 16 * k);
#pragma unroll
    for (int k = 0; k < V; k++) dst[k] = u.t[k];
  } else {
#pragma unroll
    for (int k = 0; k < V; k++) dst[k] = ((const T *)col)[(size_t)group * V + k];
  }
}

// V consecutive validity bits of a staged bitmap (tile-relative bit = group * V)
template <int V> __device__ __forceinline__ void fq_lds_bits(bool (&dst)[V], const unsigned char *bits, fq_u32 group) {
  const fq_u32 bit = group * V;
  if constexpr (V <= 8) {
    const fq_u32 w = (fq_u32)bits[bit >> 3] >> (bit & 7);
#pragma unroll
    for (int v = 0; v < V; v++) dst[v] = (w >> v) & 1u;
  } else {
#pragma unroll
    for (int b = 0; b < V / 8; b++) {
      const fq_u32 w = bits[(bit >> 3) + b];
#pragma unroll
      for (int v = 0; v < 8; v++) dst[8 * b + v] = (w >> v) & 1u;
    }
  }
}

template <class Q, int U, int STAGES>
__device__ __forceinline__ void fq_agg_tma_kernel(const fq_launch_params &p) {
  constexpr int V = Q::V;
  constexpr int S = FQ_STATE_HDR + Q::NSLOTS;
  extern __shared__ __align__(128) unsigned char fq_dyn_smem[];
  __shared__ fq_u64 sm[FQ_MAX_WARPS][S];
  __shared__ fq_u32 s_last;
  __shared__ fq_u32 s_hits;
  __shared__ __align__(8) fq_u64 s_bars[2 * STAGES];   // full[0..STAGES), empty[0..STAGES)

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cthreads = (int)blockDim.x - 32, cwarps = cthreads >> 5;
  const bool is_producer = (int)threadIdx.x >= cthreads;
  const fq_u32 tile_groups = (fq_u32)cthreads * U;
  const fq_u64 tile_rows = (fq_u64)tile_groups * V;
  const fq_u32 stage_bytes = Q::stage_bytes((fq_u32)tile_rows);
  const fq_u64 n_tiles = p.unaligned ? 0 : p.n_rows / tile_rows;   // full tiles only (none when a column is an unaligned slice)
  const int stages = (int)p.stages;

  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; s++) {
      fq_mbar_init(fq_smem_addr(&s_bars[s]), 1);                 // full: the producer's expect_tx arrive
      fq_mbar_init(fq_smem_addr(&s_bars[STAGES + s]), cwarps);   // empty: one arrive per consumer warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  typename Q::Acc acc;
  Q::init(acc);
  fq_u32 err = 0;
  fq_u64 nsel = 0;

  if (is_producer) {
    if (lane == 0) {
      fq_u64 i = 0;
      for (fq_u64 t = blockIdx.x; t < n_tiles; t += gridDim.x, i++) {
        const int s = (int)(i % stages);
        if (i >= (fq_u64)stages) fq_mbar_wait(fq_smem_addr(&s_bars[STAGES + s]), (fq_u32)(((i / stages) - 1) & 1));
        const fq_u32 full = fq_smem_addr(&s_bars[s]);
        fq_mbar_expect_tx(full, stage_bytes);
        Q::tma_issue(p, fq_smem_addr(fq_dyn_smem + (size_t)s * stage_bytes), full, t, (fq_u32)tile_rows);
      }
    }
  } else {
    fq_u64 i = 0;
    for (fq_u64 t = blockIdx.x; t < n_tiles; t += gridDim.x, i++) {
      const int s = (int)(i % stages);
      fq_mbar_wait(fq_smem_addr(&s_bars[s]), (fq_u32)((i / stages) & 1));
      const unsigned char *stage = fq_dyn_smem + (size_t)s * stage_bytes;
      typename Q::Rows rows[U];
#pragma unroll
      for (int u = 0; u < U; u++)
        Q::load_smem(rows[u], p, stage, (fq_u32)tile_rows, (fq_u32)(u * cthreads + (int)threadIdx.x), t * tile_groups + (fq_u64)u * cthreads + threadIdx.x);
#pragma unroll
      for (int u = 0; u < U; u++) {
        fq_u32 kept = 0;
#pragma unroll
        for (int v = 0; v < V; v++) kept |= (Q::consume(p, acc, rows[u], v, nsel, err) ? 1u : 0u) << v;
        if constexpr (Q::TRACK_BLOCKS) {
          if (p.block_hit) fq_mark_blocks_warp<V>(p, (t * tile_groups + (fq_u64)u * cthreads + threadIdx.x) * V, kept);
        }
      }
      __syncwarp();
      if (lane == 0) fq_mbar_arrive(fq_smem_addr(&s_bars[STAGES + s]));
    }
    // rows past the last full tile: plain loads, spread over the consumers of the whole grid
    const fq_u64 ctid = (fq_u64)blockIdx.x * cthreads + threadIdx.x;
    const fq_u64 cn = (fq_u64)gridDim.x * cthreads;
    const fq_u64 nvec = p.unaligned ? 0 : p.n_rows / V;
    for (fq_u64 g = n_tiles * tile_groups + ctid; g < nvec; g += cn) {
      typename Q::Rows r;
      Q::load(r, p, g);
      fq_u32 kept = 0;
#pragma unroll
      for (int v = 0; v < V; v++) kept |= (Q::consume(p, acc, r, v, nsel, err) ? 1u : 0u) << v;
      if constexpr (Q::TRACK_BLOCKS) {
        if (p.block_hit) fq_mark_blocks_lane<V>(p, g * V, kept);
      }
    }
    for (fq_u64 row = nvec * V + ctid; row < p.n_rows; row += cn) {
      typename Q::Rows r;
      Q::load1(r, p, row);
      const bool kept = Q::consume(p, acc, r, 0, nsel, err);
      if constexpr (Q::TRACK_BLOCKS) {
        if (p.block_hit && kept) fq_mark_one(p.block_hit, row / FQ_REF_BLOCK_ROWS);
      }
    }
  }
  fq_agg_finish<Q>(p, acc, nsel, err, sm, &s_last, &s_hits);
}

// ---------------------------------------------------------------------------------------------
// fq_select_kernel — fused predicate + order-preserving stream compaction + projection (+ limit).
//
// CTA = W worker warps + 1 scan warp (warp-specialised).  Work unit = SEGMENT of SEG consecutive tiles
// (tile = 32 * W * U vector groups; worker warp w owns the contiguous run of 32 * U groups at
// tile_base + w * 32 * U, so row order inside a tile is (warp, u, lane, v)).  Segments are claimed dynamically
// (atomicAdd) by the CTAs of a persistent grid.
//   workers, pass 1   stream the segment once from HBM, evaluate the predicate in registers, keep ONE BIT per
//                     row (U * V * SEG <= 64 bits per thread) and per-(tile, warp) selected counts in shared memory;
//                     the last warp to finish publishes the segment's aggregate descriptor (fq_sel_publish_agg);
//   scan warp         turns the counts into exclusive offsets and resolves the segment's global base by a look-back
//                     over 64-bit descriptors {flag:2, count:62} that stops at the CTA's own previous segment
//                     (fq_sel_lookback), then publishes the inclusive prefix;
//   workers, pass 2   (two segments behind) warps that selected something in a tile re-read those rows (still in
//                     the 126 MB L2: <= resident CTAs * 3 * 128 KB are in flight), rank them with __ballot_sync /
//                     __popc of the lower-lane mask and write each selected row once, projected at scatter time.
// The look-back of segment k overlaps the workers' pass 1 of segments k + 1 and k + 2: named barriers FULL[k % 3]
// (workers arrive, scan waits) and DONE[k % 3] (scan arrives, workers wait) form a three-slot ring.  With block-wide
// barriers instead, ncu showed 16-25 warp-cycles of barrier stall per issued instruction and 2.1 TB/s; a look-back
// per 16-KB tile cannot keep up with HBM at all (0.7 TB/s measured).  fq_select_tma_kernel below is the same
// algorithm with pass 1 staged by bulk copies; this kernel serves generated sources (nothing to copy).
// Rows beyond min(limit, capacity) are counted, not written.  Early exit: the segment that reaches `stop_after`
// raises a flag; a CTA that sees it when claiming publishes a saturated prefix for the claimed segment and leaves.
// Algorithmic traffic: sizeof(row) read per row from HBM + sum(sizeof(out_i)) written per selected row.
// ---------------------------------------------------------------------------------------------
#define FQ_TILE_AGG (1ull << 62)
#define FQ_TILE_PREFIX (2ull << 62)
#define FQ_TILE_VALUE(x) ((x) & ((1ull << 62) - 1))
#define FQ_TILE_FLAG(x) ((x) >> 62)

__device__ __forceinline__ void fq_bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void fq_bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// Tile access is split in two so that a tile's loads can be in flight while the previous tile is ranked:
// fq_tile_load only issues the loads (full tiles vectorised, the ragged last one row by row), fq_tile_pred
// evaluates the predicate on rows that exist: bit (u * V + v) of the returned mask is set for kept rows.
// `wthreads` = worker threads of the CTA (the tile geometry ignores the scan warp).
// PRED: only the predicate's columns (pass 1); otherwise every referenced column (pass 2 projects from them).
template <class Q, int U, bool PRED = false>
__device__ __forceinline__ void fq_tile_load(const fq_launch_params &p, fq_u64 tile, int wthreads, typename Q::Rows (&rows)[U]) {
  constexpr int V = Q::V;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const fq_u64 tile_groups = (fq_u64)wthreads * U;
  const fq_u64 g0 = tile * tile_groups + (fq_u64)warp * 32 * U + lane;
  if ((tile + 1) * tile_groups * V <= p.n_rows && !p.unaligned) {
#pragma unroll
    for (int u = 0; u < U; u++) {
      if constexpr (PRED) Q::load_pred(rows[u], p, g0 + 32ull * u);
      else Q::load(rows[u], p, g0 + 32ull * u);
    }
  } else if (tile * tile_groups * V < p.n_rows) {
#pragma unroll
    for (int u = 0; u < U; u++) {
      const fq_u64 row0 = (g0 + 32ull * u) * V;
#pragma unroll
      for (int v = 0; v < V; v++) {
        if (row0 + v < p.n_rows) {
          typename Q::Rows one;
          if constexpr (PRED) Q::load1_pred(one, p, row0 + v);
          else Q::load1(one, p, row0 + v);
          Q::copy_row(rows[u], v, one);
        }
      }
    }
  }
}
template <class Q, int U>
__device__ __forceinline__ fq_u32 fq_tile_pred(const fq_launch_params &p, fq_u64 tile, int wthreads, const typename Q::Rows (&rows)[U], fq_u32 &err) {
  constexpr int V = Q::V;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const fq_u64 tile_groups = (fq_u64)wthreads * U;
  fq_u32 keep = 0;
  if ((tile + 1) * tile_groups * V <= p.n_rows && !p.unaligned) {
#pragma unroll
    for (int u = 0; u < U; u++)
#pragma unroll
      for (int v = 0; v < V; v++) keep |= (Q::pred(p, rows[u], v, err) ? 1u : 0u) << (u * V + v);
  } else if (tile * tile_groups * V < p.n_rows) {
    const fq_u64 g0 = tile * tile_groups + (fq_u64)warp * 32 * U + lane;
#pragma unroll
    for (int u = 0; u < U; u++) {
      const fq_u64 row0 = (g0 + 32ull * u) * V;
#pragma unroll
      for (int v = 0; v < V; v++)
        if (row0 + v < p.n_rows) keep |= (Q::pred(p, rows[u], v, err) ? 1u : 0u) << (u * V + v);
    }
  }
  return keep;
}

// tile / segment shape for a given vector width: at most 32 predicate bits per thread per tile and 64 per segment
template <int V> struct fq_sel_shape {
  static constexpr int U = (FQ_SEL_UNROLL * V <= 32) ? FQ_SEL_UNROLL : (32 / V);
  static constexpr int SEG = (FQ_SEL_SEG * U * V <= 64) ? FQ_SEL_SEG : (64 / (U * V));
};

enum { FQ_BAR_FULL = 2, FQ_BAR_DONE = 5, FQ_SEL_RING = 3 };  // named barrier ids (FULL/DONE take +0..+2; 0 is __syncthreads)

// scan warp, step 1: per-(tile, worker warp) selected counts -> exclusive offsets inside the segment (in place,
// (tile, warp) order); returns the segment total.  Called by all 32 lanes of the scan warp.
template <int SEG>
__device__ __forceinline__ fq_u32 fq_sel_scan_counts(fq_u32 (*cnt)[FQ_MAX_WARPS], int nwarps) {
  const int lane = threadIdx.x & 31;
  const int entries = SEG * nwarps;
  const int per = (entries + 31) / 32;
  fq_u32 local = 0;
  for (int j = 0; j < per; j++) {
    const int i = lane * per + j;
    if (i < entries) local += cnt[i / nwarps][i % nwarps];
  }
  fq_u32 incl_lane = local;
#pragma unroll
  for (int m = 1; m < 32; m <<= 1) {
    const fq_u32 o = __shfl_up_sync(0xffffffffu, incl_lane, m);
    if (lane >= m) incl_lane += o;
  }
  const fq_u32 tot = __shfl_sync(0xffffffffu, incl_lane, 31);
  fq_u32 run = incl_lane - local;
  for (int j = 0; j < per; j++) {
    const int i = lane * per + j;
    if (i < entries) {
      const fq_u32 c = cnt[i / nwarps][i % nwarps];
      cnt[i / nwarps][i % nwarps] = run;
      run += c;
    }
  }
  return tot;
}

// Workers, end of pass 1: lane 0 of every worker warp adds the warp's selected count of the segment to a packed
// shared-memory word {arrivals:32, count:32}; the last warp to arrive publishes the segment's descriptor (aggregate;
// prefix for segment 0).  The aggregate therefore becomes visible the moment the segment has been streamed and never
// queues behind the scan warp, which may still be looking back for the previous segment — with the scan warp
// publishing it, every look-back waited for the look-backs before it (a convoy: 7-10 us per segment per CTA).
// Returns true in the warp that arrived last, with the segment total in *tot_out.
__device__ __forceinline__ bool fq_sel_publish_agg(const fq_launch_params &p, fq_u64 seg, unsigned long long *acc, fq_u32 wsum, int nwarps,
                                                   fq_u32 *tot_out = nullptr) {
  const unsigned long long old = atomicAdd(acc, (1ull << 32) | (unsigned long long)wsum);
  if ((int)(old >> 32) == nwarps - 1) {
    const fq_u64 tot = (fq_u64)((fq_u32)old + wsum);
    *acc = 0ull;   // the slot is reused three segments later, after two named barriers
    fq_st_volatile(p.tile_status + seg, (seg == 0 ? FQ_TILE_PREFIX : FQ_TILE_AGG) | tot);
    if (tot_out) *tot_out = (fq_u32)tot;
    return true;
  }
  return false;
}

// scan warp, step 2: resolve the segment's exclusive global base by a look-back over the 64-bit descriptors
// {flag:2, count:62} of its predecessors, publish the inclusive prefix.
//
// A CTA claims segments in increasing order, and its scan warp resolves them one after the other.  So when it
// looks back from segment `seg` it already knows the inclusive prefix `prev_incl` of the segment `prev_seg` it
// resolved before: the walk only has to add the AGGREGATES of the segments in between (about one per resident CTA)
// and never has to wait for anybody's PREFIX.  That matters: a classic decoupled look-back ends at the nearest
// published prefix, prefixes are published only when a look-back ends, and with hundreds of segments in flight the
// chain costs 7-10 us per segment per CTA (measured: the kernel ran at 1 segment per look-back latency).  Bounded by
// the CTA's own history the walk is 1-2 polls of FQ_SEL_LOOK * 32 descriptors, independent of the others' progress.
// A nearer published prefix still ends the walk early; the first segment of a CTA (prev_seg < 0) walks to one.
__device__ __forceinline__ fq_u64 fq_sel_lookback(const fq_launch_params &p, fq_u64 seg, fq_u32 tot, fq_i64 prev_seg, fq_u64 prev_incl) {
  const int lane = threadIdx.x & 31;
  fq_u64 excl = 0;
  if (seg == 0) return 0;   // its descriptor (a prefix) was published by the workers, like every aggregate
  fq_i64 look = (fq_i64)seg - 1;
  for (;;) {
    // FQ_SEL_LOOK * 32 predecessors per poll: lane l inspects look - 32 * j - l for j = 0 .. FQ_SEL_LOOK - 1
    fq_u64 st[FQ_SEL_LOOK];
    bool ready;
    do {
      ready = true;
#pragma unroll
      for (int j = 0; j < FQ_SEL_LOOK; j++) {
        const fq_i64 idx = look - 32 * j - lane;
        if (idx < 0) st[j] = FQ_TILE_PREFIX;                                            // before segment 0: prefix 0
        else if (idx <= prev_seg) st[j] = FQ_TILE_PREFIX | (idx == prev_seg ? prev_incl : 0ull);   // own history
        else st[j] = fq_ld_volatile(p.tile_status + idx);
        ready = ready && FQ_TILE_FLAG(st[j]) != 0;
      }
    } while (!ready);   // lanes whose descriptors are published leave the poll; the ballot below reconverges the warp
    fq_u64 contrib = 0;
    bool found = false;
#pragma unroll
    for (int j = 0; j < FQ_SEL_LOOK; j++) {
      if (!found) {
        const fq_u32 pm = __ballot_sync(0xffffffffu, FQ_TILE_FLAG(st[j]) == 2);
        if (pm) {
          if (lane <= __ffs(pm) - 1) contrib += FQ_TILE_VALUE(st[j]);
          found = true;
        } else {
          contrib += FQ_TILE_VALUE(st[j]);
        }
      }
    }
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, m);
    excl += contrib;
    if (found) break;
    look -= 32 * FQ_SEL_LOOK;
  }
  if (lane == 0) fq_st_volatile(p.tile_status + seg, FQ_TILE_PREFIX | (excl + tot));
  return excl;
}

// Pass 2 of one segment (kept out of line: it runs once per 128 KB and would otherwise double the register
// pressure of the streaming loop).  `cnt` = this segment's ring slot of exclusive offsets, `base` its global base.
// One vector group (V rows) of a tile for the calling thread: group u of worker warp `warp`, i.e. the rows
// fq_tile_load puts in rows[u].  Ragged tiles row by row.
template <class Q, int U>
__device__ __forceinline__ void fq_group_load(const fq_launch_params &p, fq_u64 tile, int wthreads, int u, typename Q::Rows &r) {
  constexpr int V = Q::V;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const fq_u64 tile_groups = (fq_u64)wthreads * U;
  const fq_u64 g = tile * tile_groups + (fq_u64)warp * 32 * U + lane + 32ull * u;
  if ((tile + 1) * tile_groups * V <= p.n_rows && !p.unaligned) {
    Q::load(r, p, g);
  } else {
#pragma unroll
    for (int v = 0; v < V; v++) {
      if (g * V + v < p.n_rows) {
        typename Q::Rows one;
        Q::load1(one, p, g * V + v);
        Q::copy_row(r, v, one);
      }
    }
  }
}

// The (tile, worker warp) run that holds output row capacity - 1 records which source row produced it (result[5],
// fq_pipe_fetch_limit_row): one run per launch at most, so the ranking is simply redone here, off the hot path.
template <class Q, int U>
__device__ __noinline__ void fq_note_limit_row(const fq_launch_params &p, fq_u64 tile, int wthreads, fq_u32 keep, fq_u64 pos0) {
  constexpr int V = Q::V;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const fq_u32 lt_mask = (1u << lane) - 1u;
  for (int u = 0; u < U; u++) {
    fq_u32 before = 0, tot = 0;
    for (int v = 0; v < V; v++) {
      const fq_u32 bmask = __ballot_sync(0xffffffffu, (keep >> (u * V + v)) & 1u);
      before += __popc(bmask & lt_mask);
      tot += __popc(bmask);
    }
    fq_u64 pos = pos0 + before;
    const fq_u64 row0 = ((tile * (fq_u64)wthreads + (fq_u64)warp * 32) * U + lane + 32ull * u) * V;   // first row of this group
    for (int v = 0; v < V; v++) {
      if ((keep >> (u * V + v)) & 1u) {
        if (pos + 1 == p.capacity) p.result[5] = row0 + v;
        pos++;
      }
    }
    pos0 += tot;
  }
}

// Scatter of one (tile, worker warp) run whose rows are in registers (loaded from L2 or from a staged tile): rank every
// kept row with ballots over the warp, project at scatter time.  `pos0` = output position of the run's first kept row.
template <class Q, int U>
__device__ __forceinline__ void fq_scatter_rows(const fq_launch_params &p, fq_u64 tile, int wthreads, fq_u32 keep, fq_u64 pos0,
                                                const typename Q::Rows (&rows)[U], fq_u32 &err) {
  constexpr int V = Q::V;
  const int lane = threadIdx.x & 31;
  const fq_u32 lt_mask = (1u << lane) - 1u;
#pragma unroll
  for (int u = 0; u < U; u++) {
    fq_u32 before = 0, tot = 0;
#pragma unroll
    for (int v = 0; v < V; v++) {
      const fq_u32 bmask = __ballot_sync(0xffffffffu, (keep >> (u * V + v)) & 1u);
      before += __popc(bmask & lt_mask);
      tot += __popc(bmask);
    }
    fq_u64 pos = pos0 + before;
    if (tot == 32u * V && (pos0 % V) == 0 && pos + V <= p.capacity) {
      // the warp kept the whole group (range predicates over sorted data: groups are all-or-nothing) and the
      // output position keeps the vector alignment: one vector store per output column instead of V scalar ones
      Q::emit_vec(rows[u], p, pos, err);
    } else {
#pragma unroll
      for (int v = 0; v < V; v++) {
        if ((keep >> (u * V + v)) & 1u) {
          if (pos < p.capacity) Q::emit(rows[u], v, p, pos, err);
          pos++;
        }
      }
    }
    pos0 += tot;
  }
}

// Pass 2 of one (tile, worker warp) run from global memory (L2).  Dense runs (the warp kept at least 1/8 of its rows)
// re-read the warp's whole run with all loads in flight; sparse runs load only the vector groups of the threads that kept
// something (a 1/1024 selection re-reads 3 % of the tile instead of 25 %).  Per-thread predicated loads for both cases
// were measured slower on dense selections (7.9 vs 5.9 ms for all of 1e9 rows).
template <class Q, int U>
__device__ __forceinline__ void fq_scatter_tile_global(const fq_launch_params &p, fq_u64 tile, int wthreads, fq_u32 keep, fq_u32 wkept,
                                                       fq_u64 pos0, fq_u32 &err) {
  constexpr int V = Q::V;
  constexpr int BITS = U * V;
  const int lane = threadIdx.x & 31;
  const fq_u32 lt_mask = (1u << lane) - 1u;
  if (pos0 < p.capacity && p.capacity <= pos0 + wkept) fq_note_limit_row<Q, U>(p, tile, wthreads, keep, pos0);
  if (wkept * 8 >= 32 * BITS) {
    typename Q::Rows rows[U];
    fq_tile_load<Q, U>(p, tile, wthreads, rows);   // L2 hit
    fq_scatter_rows<Q, U>(p, tile, wthreads, keep, pos0, rows, err);
  } else {
#pragma unroll 1
    for (int u = 0; u < U; u++) {
      const fq_u32 ku = (keep >> (u * V)) & ((1u << V) - 1u);
      if (__ballot_sync(0xffffffffu, ku != 0) == 0) continue;
      typename Q::Rows r;
      if (ku) fq_group_load<Q, U>(p, tile, wthreads, u, r);
      fq_u32 before = 0, tot = 0;
#pragma unroll
      for (int v = 0; v < V; v++) {
        const fq_u32 bmask = __ballot_sync(0xffffffffu, (ku >> v) & 1u);
        before += __popc(bmask & lt_mask);
        tot += __popc(bmask);
      }
      fq_u64 pos = pos0 + before;
#pragma unroll
      for (int v = 0; v < V; v++) {
        if ((ku >> v) & 1u) {
          if (pos < p.capacity) Q::emit(r, v, p, pos, err);
          pos++;
        }
      }
      pos0 += tot;
    }
  }
}

// Pass 2 of one segment from global memory (kept out of line: it runs once per segment and would otherwise double the
// register pressure of the streaming loop).  `cnt` = this segment's ring slot of exclusive offsets, `base` its global
// base.  The re-reads hit L2: at most resident CTAs * LAG segments are between the passes.
template <class Q, int U, int SEG>
__device__ __noinline__ void fq_select_scatter(const fq_launch_params &p, fq_u64 sseg, fq_u64 skeep, const fq_u32 (*cnt)[FQ_MAX_WARPS],
                                               fq_u64 base, int wthreads, fq_u32 *err_out) {
  constexpr int V = Q::V;
  constexpr int BITS = U * V;
  const int warp = threadIdx.x >> 5;
  fq_u32 err = 0;
  if (base >= p.capacity) return;
#pragma unroll
  for (int t = 0; t < SEG; t++) {
    const fq_u32 keep = (fq_u32)(skeep >> (t * BITS)) & (BITS >= 32 ? 0xffffffffu : ((1u << (BITS & 31)) - 1u));
    const fq_u32 wkept = __reduce_add_sync(0xffffffffu, (fq_u32)__popc(keep));
    if (wkept == 0) continue;
    fq_scatter_tile_global<Q, U>(p, sseg * SEG + t, wthreads, keep, wkept, base + cnt[t][warp], err);
  }
  if (err) *err_out |= err;
}

// Pass 2 of one DENSE segment of the staged select kernel: the producer staged the segment's full tiles again (every
// referenced column).  Every consumer warp takes every slot (work or not), copies its rows to registers, hands the slot
// back and then ranks + writes.  sr = {ring slot, round} of the next staged tile, updated.  Out of line like
// fq_select_scatter, for the same reason.
template <class Q, int U, int SEG, int STAGES>
__device__ __noinline__ void fq_select_scatter_staged(const fq_launch_params &p, fq_u64 sseg, fq_u64 skeep, const fq_u32 (*cnt)[FQ_MAX_WARPS],
                                                      fq_u64 base, int cthreads, fq_u64 *bars, fq_u32 stage_bytes, fq_u64 n_full_tiles,
                                                      fq_u32 (&sr)[2], fq_u32 *err_out) {
  constexpr int V = Q::V;
  constexpr int BITS = U * V;
  extern __shared__ __align__(128) unsigned char fq_dyn_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const fq_u32 tile_rows = (fq_u32)cthreads * U * V;
  const int stages = (int)p.stages;
  int slot = (int)sr[0];
  fq_u32 round = sr[1];
  fq_u32 err = 0;
  const bool live = base < p.capacity;
#pragma unroll 1
  for (int t = 0; t < SEG; t++) {
    const fq_u64 tile = sseg * SEG + t;
    const fq_u32 keep = (fq_u32)(skeep >> (t * BITS)) & (BITS >= 32 ? 0xffffffffu : ((1u << (BITS & 31)) - 1u));
    const fq_u32 wkept = __reduce_add_sync(0xffffffffu, (fq_u32)__popc(keep));
    const fq_u64 pos0 = base + cnt[t][warp];
    if (tile < n_full_tiles) {
      fq_mbar_wait(fq_smem_addr(&bars[slot]), round & 1);
      typename Q::Rows rows[U];
      if (live && wkept) {
        const unsigned char *stage = fq_dyn_smem + (size_t)slot * stage_bytes;
#pragma unroll
        for (int u = 0; u < U; u++)
          Q::load_smem(rows[u], p, stage, tile_rows, (fq_u32)(warp * 32 * U + 32 * u + lane), tile * ((fq_u64)cthreads * U) + (fq_u64)(warp * 32 * U + 32 * u + lane));
      }
      __syncwarp();
      if (lane == 0) fq_mbar_arrive(fq_smem_addr(&bars[STAGES + slot]));   // the rows are in registers: hand the slot back
      if (++slot == stages) { slot = 0; round++; }
      if (live && wkept) {
        if (pos0 < p.capacity && p.capacity <= pos0 + wkept) fq_note_limit_row<Q, U>(p, tile, cthreads, keep, pos0);
        fq_scatter_rows<Q, U>(p, tile, cthreads, keep, pos0, rows, err);
      }
    } else if (live && wkept) {
      fq_scatter_tile_global<Q, U>(p, tile, cthreads, keep, wkept, pos0, err);
    }
  }
  sr[0] = (fq_u32)slot;
  sr[1] = round;
  if (err) *err_out |= err;
}

template <class Q, int U, int SEG>
__device__ __forceinline__ void fq_select_kernel(const fq_launch_params &p) {
  constexpr int V = Q::V;
  constexpr int BITS = U * V;                 // predicate bits per thread per tile
  static_assert(BITS <= 32 && BITS * SEG <= 64, "one keep bit per row must fit two registers");
  __shared__ fq_u32 s_cnt[FQ_SEL_RING][SEG][FQ_MAX_WARPS];  // per (tile, worker warp): selected count, then exclusive offset in the segment
  __shared__ fq_u64 s_excl[FQ_SEL_RING];                    // global base of the segment in each ring slot
  __shared__ unsigned long long s_acc[FQ_SEL_RING];         // {arrived worker warps, selected rows} of the segment being streamed
  __shared__ volatile fq_u64 s_seg[4];           // claimed segment ids: ring of 4 (the scan warp lags the workers by up to 2)
  __shared__ volatile fq_u32 s_stop[4];
  __shared__ volatile int s_ready[4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wthreads = (int)blockDim.x - 32, nwarps = wthreads >> 5, allthreads = (int)blockDim.x;
  const bool is_scan = (int)threadIdx.x >= wthreads;
  const fq_u32 lt_mask = (1u << lane) - 1u;
  const fq_u64 n_seg = p.n_tiles;
  fq_u32 err = 0;

  // Segments are claimed dynamically (atomicAdd): only running CTAs own segments, so every predecessor of a running
  // segment has started and the look-back makes progress whatever else shares the GPU.  Claiming and observing the
  // early-exit flag happen together: a claimed segment is ALWAYS published (a successor may already be polling it); a CTA
  // that sees the flag publishes a saturated prefix for the segment it just claimed and leaves.
  // Thread 0 claims the segment of iteration k + 1 at the start of iteration k and hands it to the other warps through a
  // shared-memory ring (s_ready[slot] == k + 2): no block-wide barrier per segment, warps run ahead on their own.
  auto publish_claim = [&](int k, fq_u64 c, fq_u32 st) {   // claim of iteration k
    s_seg[k & 3] = c;
    s_stop[k & 3] = st;
    __threadfence_block();
    s_ready[k & 3] = k + 1;
  };
  if (threadIdx.x >= 1 && threadIdx.x < 4) s_ready[threadIdx.x] = 0;
  if (threadIdx.x < FQ_SEL_RING) s_acc[threadIdx.x] = 0ull;
  if (threadIdx.x == 0) {
    const fq_u64 c = atomicAdd(p.tile_counter, 1u);
    const fq_u32 st = (p.stop_after != 0 && fq_ld_volatile32(p.done) != 0) ? 1u : 0u;
    if (st && c < n_seg) fq_st_volatile(p.tile_status + c, FQ_TILE_PREFIX | p.stop_after);
    publish_claim(0, c, st);
  }
  __syncthreads();

  if (is_scan) {
    // ================= scan warp =================
    fq_i64 prev_seg = -1;      // the segment this CTA resolved last and its inclusive prefix (see fq_sel_lookback)
    fq_u64 prev_incl = 0;
    for (int k = 0;; k++) {
      const int b = k % FQ_SEL_RING;
      fq_bar_sync(FQ_BAR_FULL + b, allthreads);
      const fq_u64 seg = s_seg[k & 3];
      if (!(seg < n_seg) || s_stop[k & 3]) break;
      const fq_u32 tot = fq_sel_scan_counts<SEG>(s_cnt[b], nwarps);
      const fq_u64 excl = fq_sel_lookback(p, seg, tot, prev_seg, prev_incl);
      prev_seg = (fq_i64)seg;
      prev_incl = excl + tot;
      if (lane == 0) {
        s_excl[b] = excl;
        const fq_u64 incl = excl + tot;
        if (p.stop_after != 0 && incl >= p.stop_after) {
          *(volatile fq_u32 *)p.done = 1u;
          atomicMax(p.result, incl);   // the last segment may never run: report what is known
        }
        if (seg == n_seg - 1) atomicMax(p.result, incl);
      }
      __syncwarp();
      fq_bar_arrive(FQ_BAR_DONE + b, allthreads);
    }
    return;
  }

  // ================= worker warps =================
  // scatter of segment j: its look-back had two segment-streaming times to complete
  auto scatter = [&](fq_u64 sseg, fq_u64 skeep, int sb) {
    fq_bar_sync(FQ_BAR_DONE + sb, allthreads);
    fq_select_scatter<Q, U, SEG>(p, sseg, skeep, s_cnt[sb], s_excl[sb], wthreads, &err);
  };
  fq_u64 keep1 = 0, seg1 = 0, keep2 = 0, seg2 = 0;   // segments k-1 and k-2, still to be scattered
  int pending = 0;
  for (int k = 0;; k++) {
    const int b = k % FQ_SEL_RING;
    if (lane == 0) {
      while (s_ready[k & 3] != k + 1) {}   // claim of this iteration (made one segment ago by thread 0)
    }
    __syncwarp();
    const fq_u64 seg = s_seg[k & 3];
    const bool stop = s_stop[k & 3] != 0;
    const bool active = seg < n_seg && !stop;

    // thread 0: claim the next segment now, publish it after pass 1 (the atomic's round trip hides behind the streaming)
    fq_u64 next_c = 0;
    fq_u32 next_st = 0;
    if (threadIdx.x == 0 && active) {
      next_c = atomicAdd(p.tile_counter, 1u);
      next_st = (p.stop_after != 0 && fq_ld_volatile32(p.done) != 0) ? 1u : 0u;
    }

    // ---- pass 1: one streaming read of the segment, one bit per row ----
    fq_u64 keepbits = 0;
    if (active) {
      typename Q::Rows rows0[U], rows_n[U];
      fq_u32 wsum = 0;
      fq_tile_load<Q, U, true>(p, seg * SEG, wthreads, rows0);
#pragma unroll
      for (int t = 0; t < SEG; t++) {
        if (t + 1 < SEG) fq_tile_load<Q, U, true>(p, seg * SEG + t + 1, wthreads, rows_n);   // next tile's loads in flight
        const fq_u32 keep = fq_tile_pred<Q, U>(p, seg * SEG + t, wthreads, rows0, err);
        keepbits |= (fq_u64)keep << (t * BITS);
        const fq_u32 wcount = __reduce_add_sync(0xffffffffu, (fq_u32)__popc(keep));
        if (lane == 0) s_cnt[b][t][warp] = wcount;
        wsum += wcount;
        if (t + 1 < SEG) {
#pragma unroll
          for (int u = 0; u < U; u++) rows0[u] = rows_n[u];
        }
      }
      if (lane == 0) fq_sel_publish_agg(p, seg, &s_acc[b], wsum, nwarps);
    }
    if (threadIdx.x == 0 && active) {
      if (next_st && next_c < n_seg) fq_st_volatile(p.tile_status + next_c, FQ_TILE_PREFIX | p.stop_after);
      publish_claim(k + 1, next_c, next_st);
    }
    __syncwarp();
    fq_bar_arrive(FQ_BAR_FULL + b, allthreads);   // hand the counts (or the end marker) to the scan warp

    // ---- pass 2 of segment k-2 (while the scan warp resolves k-1 and k) ----
    if (pending == 2) {
      scatter(seg2, keep2, (k + 1) % FQ_SEL_RING);   // (k - 2) mod 3
      pending = 1;
    }
    if (!active) {
      if (pending == 1) scatter(seg1, keep1, (k + 2) % FQ_SEL_RING);   // (k - 1) mod 3
      break;
    }
    keep2 = keep1;
    seg2 = seg1;
    keep1 = keepbits;
    seg1 = seg;
    pending += 1;   // no block-wide sync here: warps run ahead into the next segment on their own
  }
  if (err) atomicOr((fq_u32 *)(p.result + 1), err);
}

// ---------------------------------------------------------------------------------------------
// fq_select_tma_kernel — the select kernel with BOTH passes staged by the bulk-copy engine.
//
// One CTA per SM = C consumer warps + 1 scan warp + 1 producer warp.  The producer lane claims segments
// (atomicAdd), hands the ids to the other warps through a shared-memory ring and keeps a ring of `stages` tiles
// in flight with cp.async.bulk (one copy per column per tile, completion on full[s]); bytes in flight per
// SM are therefore independent of the consumers' registers and of the time they spend in pass 2.
//   pass 1   consumers read each staged tile (the predicate's columns) with LDS.128 (lane l of warp w, group u: vector
//            group w * 32U + 32u + l — the row order of fq_tile_load, so the ranking code is shared with
//            fq_select_kernel), evaluate the predicate, keep one bit per row and per-(tile, warp) counts, and release
//            the slot (one arrive per warp on empty[s]).  The warp that finishes a segment last publishes its
//            aggregate and decides whether the segment is DENSE (>= 1/8 of its rows kept and the output not yet full).
//   pass 2   LAG segments later, when the scan warp has resolved the segment's base.  Sparse segments: the warps that
//            kept something re-read just those vector groups from L2 (fq_scatter_tile_global).  Dense segments: the
//            producer stages the segment's tiles AGAIN (every referenced column this time; an L2 hit when LAG * SEG
//            tiles per SM fit) behind the pass-1 tiles of the current segment, so the re-read is as asynchronous as the
//            first read: consumers find the rows in shared memory, copy them to registers, release the slot, rank with
//            ballots and write.  With per-thread L2 re-reads instead (round 1) the L2 latency was exposed once per
//            tile and a selection keeping every row ran at 0.70 of the copy peak.
// Producer and consumers walk the same sequence of staged tiles: per iteration k the full tiles of the claimed segment,
// then, if the segment of iteration k - LAG is dense, its full tiles again; at the end the pending segments oldest
// first.  Tiles that are not entirely inside the source (the ragged end) are never staged: consumers load them with
// fq_tile_load.  Scan warp, look-back and the named-barrier ring FULL/DONE are those of fq_select_kernel.
// p.stages2 != 0 switches the staged pass 2 on (the host does when a stage of all referenced columns fits the ring).
// ---------------------------------------------------------------------------------------------
template <int V> struct fq_selt_shape {
  static constexpr int U = (FQ_SELT_UNROLL * V <= 32) ? FQ_SELT_UNROLL : (32 / V);
  static constexpr int SEG = (FQ_SELT_SEG * U * V <= 64) ? FQ_SELT_SEG : (64 / (U * V));
};
template <int V> struct fq_seld_shape {
  static constexpr int U = (FQ_SELD_UNROLL * V <= 32) ? FQ_SELD_UNROLL : (32 / V);
  static constexpr int SEG = (FQ_SELD_SEG * U * V <= 64) ? FQ_SELD_SEG : (64 / (U * V));
};
// Density probe: every CTA evaluates the predicate over FQ_SELD_PROBE_ROWS rows at an evenly spaced position of the source;
// the last CTA decides the build (dense when at least 1/16 of the sampled rows are kept) — on the device, so that no host
// round trip sits between the probe and the two launches that follow it (the build that is not chosen returns at once).
template <class Q>
__device__ __forceinline__ void fq_select_probe_kernel(const fq_launch_params &p) {
  constexpr int V = Q::V;
  __shared__ fq_u32 s_kept;
  if (threadIdx.x == 0) s_kept = 0;
  __syncthreads();
  const fq_u64 groups_total = p.n_rows / V;
  const fq_u64 per_cta = FQ_SELD_PROBE_ROWS / V;
  fq_u32 err = 0, kept = 0, sampled = 0;
  if (groups_total >= per_cta * gridDim.x && !p.unaligned) {
    const fq_u64 g0 = (groups_total / gridDim.x) * blockIdx.x;
    for (fq_u64 g = threadIdx.x; g < per_cta; g += blockDim.x) {
      typename Q::Rows r;
      Q::load_pred(r, p, g0 + g);
#pragma unroll
      for (int v = 0; v < V; v++) kept += Q::pred(p, r, v, err) ? 1u : 0u;
      sampled += V;
    }
  }
  kept = __reduce_add_sync(0xffffffffu, kept);
  sampled = __reduce_add_sync(0xffffffffu, sampled);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(p.probe, sampled);
    atomicAdd(p.probe + 1, kept);
    __threadfence();
  }
  __syncthreads();
  if (threadIdx.x == 0 && atomicAdd(p.probe + 3, 1u) == gridDim.x - 1) {
    __threadfence();
    const fq_u32 n = *(volatile fq_u32 *)p.probe, k = *(volatile fq_u32 *)(p.probe + 1);
    p.probe[2] = (n > 0 && (fq_u64)k * 16 >= n) ? 1u : 0u;
  }
}
#define FQ_SELT_CLAIMS 16   // claim ring: the producer runs at most stages/SEG + 1 segments ahead of pass 1, the scan warp 2 behind

template <class Q, int U, int SEG, int STAGES, bool STAGE2>
__device__ __forceinline__ void fq_select_tma_kernel(const fq_launch_params &p) {
  constexpr int V = Q::V;
  // two builds share the launch parameters; the density probe (or the host) says which one runs this launch
  if (p.sel_mode && *(volatile const fq_u32 *)p.sel_mode != (STAGE2 ? 1u : 0u)) return;
  constexpr int BITS = U * V;
  static_assert(BITS <= 32 && BITS * SEG <= 64, "one keep bit per row must fit two registers");
  constexpr int LAG = FQ_SELT_LAG;            // pass 2 runs this many segments behind pass 1 (absorbs the skew between CTAs)
  constexpr int R = LAG + 1;                  // ring of count / base slots and of FULL / DONE named barriers
  constexpr int BAR_FULL = 2, BAR_DONE = 2 + R;
  static_assert(2 + 2 * R <= 16, "named barriers");
  static_assert(LAG + 1 <= FQ_SELT_CLAIMS, "claim ring");
  extern __shared__ __align__(128) unsigned char fq_dyn_smem[];
  __shared__ fq_u32 s_cnt[R][SEG][FQ_MAX_WARPS];
  __shared__ fq_u64 s_excl[R];
  __shared__ unsigned long long s_acc[R];
  __shared__ volatile fq_u64 s_seg[FQ_SELT_CLAIMS];
  __shared__ volatile fq_u32 s_stop[FQ_SELT_CLAIMS];
  __shared__ volatile int s_ready[FQ_SELT_CLAIMS];
  __shared__ volatile int s_p1[R];            // iteration k finished pass 1: (k + 1) << 1 | dense
  __shared__ volatile fq_u64 s_lastbase;      // base of the segment this CTA resolved last (monotone)
  __shared__ __align__(8) fq_u64 s_bars[2 * STAGES];   // full[0..STAGES), empty[0..STAGES)

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cthreads = (int)blockDim.x - 64, cwarps = cthreads >> 5, barthreads = cthreads + 32;
  const bool is_scan = (int)threadIdx.x >= cthreads && (int)threadIdx.x < cthreads + 32;
  const bool is_producer = (int)threadIdx.x >= cthreads + 32;
  const fq_u32 tile_groups = (fq_u32)cthreads * U;
  const fq_u64 tile_rows = (fq_u64)tile_groups * V;
  const bool stage2 = STAGE2 && p.stages2 != 0;
  // one slot holds a pass-1 tile (the predicate's columns) or, with the staged pass 2, a tile of every referenced column
  const fq_u32 pred_bytes = Q::pred_stage_bytes((fq_u32)tile_rows), all_bytes = Q::stage_bytes((fq_u32)tile_rows);
  const fq_u32 stage_bytes = stage2 ? all_bytes : pred_bytes;
  const fq_u64 n_full_tiles = p.unaligned ? 0 : p.n_rows / tile_rows;   // staged tiles; the others go through fq_tile_load
  const fq_u64 n_seg = p.n_tiles;
  const int stages = (int)p.stages;
  fq_u32 err = 0;

  if (threadIdx.x < FQ_SELT_CLAIMS) s_ready[threadIdx.x] = 0;
  if (threadIdx.x < R) { s_acc[threadIdx.x] = 0ull; s_p1[threadIdx.x] = 0; }
  if (threadIdx.x == 0) {
    s_lastbase = 0;
    for (int s = 0; s < stages; s++) {
      fq_mbar_init(fq_smem_addr(&s_bars[s]), 1);
      fq_mbar_init(fq_smem_addr(&s_bars[STAGES + s]), cwarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (is_producer) {
    // ================= producer warp (one lane) =================
    if (lane == 0) {
      int slot = 0;          // ring slot and round of the next staged tile (no 64-bit divisions in the loop)
      fq_u32 round = 0;
      fq_u64 hist[1] = {0};  // segment of the previous iteration
      auto stage_tile = [&](fq_u64 tile, bool all_cols) {
        if (round >= 1) fq_mbar_wait(fq_smem_addr(&s_bars[STAGES + slot]), (round - 1) & 1);
        const fq_u32 full = fq_smem_addr(&s_bars[slot]);
        const fq_u32 dst = fq_smem_addr(fq_dyn_smem + (size_t)slot * stage_bytes);
        if (all_cols) {
          fq_mbar_expect_tx(full, all_bytes);
          Q::template tma_issue<2>(p, dst, full, tile, (fq_u32)tile_rows);          // last use of these lines
        } else {
          fq_mbar_expect_tx(full, pred_bytes);
          if (stage2) Q::template tma_issue_pred<1>(p, dst, full, tile, (fq_u32)tile_rows);   // dense segments read them again
          else Q::template tma_issue_pred<0>(p, dst, full, tile, (fq_u32)tile_rows);
        }
        if (++slot == stages) { slot = 0; round++; }
      };
      // pass 2 of iteration j (segment sj): staged again when the consumers found it dense
      auto stage_pass2 = [&](int j, fq_u64 sj) {
        int v;
        while (((v = s_p1[j % R]) >> 1) != j + 1) {}
        if (!(v & 1)) return;
#pragma unroll 1
        for (int t = 0; t < SEG; t++)
          if (sj * SEG + t < n_full_tiles) stage_tile(sj * SEG + t, true);
      };
      fq_u64 c = atomicAdd(p.tile_counter, 1u);
      for (int k = 0;; k++) {
        const fq_u32 st = (p.stop_after != 0 && fq_ld_volatile32(p.done) != 0) ? 1u : 0u;
        // a claimed segment is always published: a successor's look-back may already be polling it
        if (st && c < n_seg) fq_st_volatile(p.tile_status + c, FQ_TILE_PREFIX | p.stop_after);
        s_seg[k % FQ_SELT_CLAIMS] = c;
        s_stop[k % FQ_SELT_CLAIMS] = st;
        __threadfence_block();
        s_ready[k % FQ_SELT_CLAIMS] = k + 1;
        if (!(c < n_seg) || st) {
          if (stage2 && k >= 1) stage_pass2(k - 1, hist[0]);   // drain: only the last segment can still be waiting for its pass 2
          break;
        }
        // the next claim's round trip to L2 overlaps the copies of this segment (its value is first used next iteration)
        const fq_u64 c_next = atomicAdd(p.tile_counter, 1u);
#pragma unroll 1
        for (int t = 0; t < SEG; t++) {
          const fq_u64 tile = c * SEG + t;
          if (tile < n_full_tiles) stage_tile(tile, false);
        }
        if (stage2 && k >= 1) stage_pass2(k - 1, hist[0]);   // a dense segment is staged again right behind its successor
        hist[0] = c;          // segment of iteration k - 1 at the next iteration
        c = c_next;
      }
    }
    return;
  }

  if (is_scan) {
    // ================= scan warp =================
    fq_i64 prev_seg = -1;      // the segment this CTA resolved last and its inclusive prefix (see fq_sel_lookback)
    fq_u64 prev_incl = 0;
    for (int k = 0;; k++) {
      const int b = k % R;
      fq_bar_sync(BAR_FULL + b, barthreads);
      const fq_u64 seg = s_seg[k % FQ_SELT_CLAIMS];
      if (!(seg < n_seg) || s_stop[k % FQ_SELT_CLAIMS]) break;
      const fq_u32 tot = fq_sel_scan_counts<SEG>(s_cnt[b], cwarps);
      const fq_u64 excl = fq_sel_lookback(p, seg, tot, prev_seg, prev_incl);
      prev_seg = (fq_i64)seg;
      prev_incl = excl + tot;
      if (lane == 0) {
        s_excl[b] = excl;
        s_lastbase = excl;
        const fq_u64 incl = excl + tot;
        if (p.stop_after != 0 && incl >= p.stop_after) {
          *(volatile fq_u32 *)p.done = 1u;
          atomicMax(p.result, incl);
        }
        if (seg == n_seg - 1) atomicMax(p.result, incl);
      }
      __syncwarp();
      fq_bar_arrive(BAR_DONE + b, barthreads);
    }
    return;
  }

  // ================= consumer warps =================
  int slot = 0;          // ring slot and round of the next staged tile (same count as the producer's)
  fq_u32 round = 0;
  auto scatter = [&](fq_u64 sseg, fq_u64 skeep, int sb) {
    fq_bar_sync(BAR_DONE + sb, barthreads);
    if (!(stage2 && (s_p1[sb] & 1))) {
      fq_select_scatter<Q, U, SEG>(p, sseg, skeep, s_cnt[sb], s_excl[sb], cthreads, &err);
      return;
    }
    // dense segment: its full tiles were staged again (every referenced column) — consume every slot, work or not
    fq_u32 sr[2] = {(fq_u32)slot, round};
    fq_select_scatter_staged<Q, U, SEG, STAGES>(p, sseg, skeep, s_cnt[sb], s_excl[sb], cthreads, s_bars, stage_bytes, n_full_tiles, sr, &err);
    slot = (int)sr[0];
    round = sr[1];
  };
  // Segments streamed but not yet scattered, newest first (registers: constant indexes): entry j = iteration k - 1 - j,
  // valid when bit j of `pend` is set.  A DENSE segment is scattered one iteration after its pass 1 (its tiles come
  // through the ring again right behind the next segment's: the shorter the distance, the more of the re-read hits L2 —
  // at LAG = 3 the 148 SMs hold 100 MB between the passes and every re-read went to HBM); a SPARSE one LAG iterations
  // after, when its look-back has long finished (waiting for it any earlier stalls the streaming: 1.2 -> 1.5 ms on the
  // README predicate), re-reading the few kept groups with plain loads.
  fq_u64 keepq[LAG], segq[LAG];
#pragma unroll
  for (int j = 0; j < LAG; j++) keepq[j] = segq[j] = 0;
  fq_u32 pend = 0;
  for (int k = 0;; k++) {
    const int b = k % R;
    if (lane == 0) {
      while (s_ready[k % FQ_SELT_CLAIMS] != k + 1) {}
    }
    __syncwarp();
    const fq_u64 seg = s_seg[k % FQ_SELT_CLAIMS];
    const bool active = seg < n_seg && s_stop[k % FQ_SELT_CLAIMS] == 0;

    fq_u64 keepbits = 0;
    if (active) {
      fq_u32 wsum = 0;
#pragma unroll
      for (int t = 0; t < SEG; t++) {
        const fq_u64 tile = seg * SEG + t;
        fq_u32 keep = 0;
        if (tile < n_full_tiles) {
          fq_mbar_wait(fq_smem_addr(&s_bars[slot]), round & 1);
          const unsigned char *stage = fq_dyn_smem + (size_t)slot * stage_bytes;
          typename Q::Rows rows[U];
#pragma unroll
          for (int u = 0; u < U; u++)
            Q::load_smem_pred(rows[u], p, stage, (fq_u32)tile_rows, (fq_u32)(warp * 32 * U + 32 * u + lane), tile * tile_groups + (fq_u64)(warp * 32 * U + 32 * u + lane));
#pragma unroll
          for (int u = 0; u < U; u++)
#pragma unroll
            for (int v = 0; v < V; v++) keep |= (Q::pred(p, rows[u], v, err) ? 1u : 0u) << (u * V + v);
          __syncwarp();
          if (lane == 0) fq_mbar_arrive(fq_smem_addr(&s_bars[STAGES + slot]));
          if (++slot == stages) { slot = 0; round++; }
        } else {   // ragged or empty tile at the end of the source
          typename Q::Rows rows[U];
          fq_tile_load<Q, U, true>(p, tile, cthreads, rows);
          keep = fq_tile_pred<Q, U>(p, tile, cthreads, rows, err);
        }
        keepbits |= (fq_u64)keep << (t * BITS);
        const fq_u32 wcount = __reduce_add_sync(0xffffffffu, (fq_u32)__popc(keep));
        if (lane == 0) s_cnt[b][t][warp] = wcount;
        wsum += wcount;
      }
      if (lane == 0) {
        fq_u32 tot = 0;
        if (fq_sel_publish_agg(p, seg, &s_acc[b], wsum, cwarps, &tot)) {
          // last warp of the segment: dense segments get their pass 2 staged (producer and consumers read this one flag)
          const bool dense = stage2 && (fq_u64)tot * 8 >= tile_rows * SEG && s_lastbase < p.capacity;
          __threadfence_block();
          s_p1[b] = ((k + 1) << 1) | (dense ? 1 : 0);
        }
      }
    }
    __syncwarp();
    fq_bar_arrive(BAR_FULL + b, barthreads);

    // the previous segment, if dense: its tiles are next in the ring
    if ((pend & 1u) && stage2) {
      if (lane == 0) {
        while ((s_p1[(k - 1) % R] >> 1) != k) {}   // every warp finished its pass 1 (the flag is written by the last one)
      }
      __syncwarp();
      if (s_p1[(k - 1) % R] & 1) {
        scatter(segq[0], keepq[0], (k - 1) % R);
        pend &= ~1u;
      }
    }
    // the segment of iteration k - LAG, if it is still waiting (sparse)
    if (pend & (1u << (LAG - 1))) {
      scatter(segq[LAG - 1], keepq[LAG - 1], (k + 1) % R);
      pend &= ~(1u << (LAG - 1));
    }
    if (!active) {          // drain, oldest first: entry j is the segment of iteration k - 1 - j
#pragma unroll
      for (int j = LAG - 2; j >= 0; j--)
        if (pend & (1u << j)) scatter(segq[j], keepq[j], (k - 1 - j) % R);
      break;
    }
#pragma unroll
    for (int j = LAG - 1; j > 0; j--) { keepq[j] = keepq[j - 1]; segq[j] = segq[j - 1]; }
    keepq[0] = keepbits;
    segq[0] = seg;
    pend = (pend << 1) | 1u;
  }
  if (err) atomicOr((fq_u32 *)(p.result + 1), err);
}

// ---------------------------------------------------------------------------------------------
// fq_groupby_kernel — hash aggregation (GROUP BY), one pass over the source.
//
// The reference plans GROUP BY but never executes it (pipeline_builder.rs:50-65 uses only aggr_expr); this is the
// operator AggregatePlan{group_expr, aggr_expr} describes, with the aggregate protocol of function_aggregator.rs:57-100
// applied per group.  Generated code (codegen.cc) supplies, per row, the packed key (Q::Key: fq_u64 for keys of up to 64
// bits, fq_gb_key2 for 65..128) and the encoded value of every Aggregator leaf (Q::gb_row), and the atomics that fold a row /
// a partial state into a group's Q::G slots.
// Two levels of open-addressing tables: every CTA aggregates into a table in shared memory first (gb_smem_cap slots, new
// keys admitted until it is 3/4 full) — with few distinct keys nothing but the final flush leaves the SM; a row whose key
// is not admitted there goes straight to the table in HBM (atomicCAS on the key, then atomics on the state).  At the end
// the CTA flushes its shared-memory groups into the HBM table.  Both searches keep the warp together (one probe step per
// trip, the trip count is the warp's longest chain): the atomics that follow are issued once per warp, not once per chain
// length.  A table that runs full raises gb_flags[0]: the host reserves
// a bigger one and relaunches.  Every reservation after a pipe's first hashes with a new seed (gb_seed): fq_gb_hash is a
// bijection, so keys can share the low bits of their hashes, and a cluster that overflowed one table would overflow every
// larger one under the same hash.  Algorithmic traffic: sizeof(row) read per row + the table.
// ---------------------------------------------------------------------------------------------
#define FQ_GB_EMPTY 0xffffffffffffffffull

// order-preserving 64-bit code of a double (min / max of float columns through integer atomics)
__device__ __forceinline__ fq_u64 fq_f64_ordered(double x) {
  const fq_u64 b = (fq_u64)__double_as_longlong(x);
  return (b >> 63) ? ~b : (b | (1ull << 63));
}
__device__ __forceinline__ double fq_f64_unordered(fq_u64 c) {
  return __longlong_as_double((fq_i64)((c >> 63) ? (c & ~(1ull << 63)) : ~c));
}
__device__ __forceinline__ fq_u64 fq_gb_hash(fq_u64 k) {
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdull;
  k ^= k >> 33;
  k *= 0xc4ceb9fe1a85ec53ull;
  k ^= k >> 33;
  return k;
}
// hash of a 128-bit key under `seed`.  fq_gb_hash is a bijection, so two distinct keys with the same lo never collide, and
// two with different lo collide only for particular seeds: the reseeded table after an overflow spreads a cluster again.
// (A form such as hash(lo ^ hash(hi)) ^ seed would keep every collision under every seed.)
__device__ __forceinline__ fq_u64 fq_gb_hash2(fq_u64 lo, fq_u64 hi, fq_u64 seed) {
  return fq_gb_hash(hi ^ fq_gb_hash(lo ^ seed));
}

// The table key: one 8-byte word, or two for keys of 65..128 bits.  Either is claimed by ONE compare-and-swap (sm_100a has
// a native 16-byte CAS in shared and global memory), so a slot goes from EMPTY to its key in one step and never changes
// again.  The overloads below are the only code that knows the width; the fq_u64 ones are the expressions of the 64-bit
// table, so its kernels compile as before.
struct __align__(16) fq_gb_key2 {
  fq_u64 lo, hi;
};
template <class K> __device__ __forceinline__ K fq_gb_empty();
template <> __device__ __forceinline__ fq_u64 fq_gb_empty<fq_u64>() { return FQ_GB_EMPTY; }
template <> __device__ __forceinline__ fq_gb_key2 fq_gb_empty<fq_gb_key2>() { return {FQ_GB_EMPTY, FQ_GB_EMPTY}; }
__device__ __forceinline__ bool fq_gb_eq(fq_u64 a, fq_u64 b) { return a == b; }
__device__ __forceinline__ bool fq_gb_eq(const fq_gb_key2 &a, const fq_gb_key2 &b) { return a.lo == b.lo && a.hi == b.hi; }
__device__ __forceinline__ bool fq_gb_is_empty(fq_u64 k) { return k == FQ_GB_EMPTY; }
__device__ __forceinline__ bool fq_gb_is_empty(const fq_gb_key2 &k) { return k.lo == FQ_GB_EMPTY && k.hi == FQ_GB_EMPTY; }
__device__ __forceinline__ fq_u64 fq_gb_seeded(fq_u64 k, fq_u64 seed) { return fq_gb_hash(k ^ seed); }
__device__ __forceinline__ fq_u64 fq_gb_seeded(const fq_gb_key2 &k, fq_u64 seed) { return fq_gb_hash2(k.lo, k.hi, seed); }
// a key stored as words (a partial entry: the key's words, then the group state)
__device__ __forceinline__ void fq_gb_from_words(fq_u64 &k, const fq_u64 *w) { k = w[0]; }
__device__ __forceinline__ void fq_gb_from_words(fq_gb_key2 &k, const fq_u64 *w) {
  k.lo = w[0];
  k.hi = w[1];
}
// The look before the CAS.  A 16-byte look is two 8-byte loads and is NOT taken to be single-copy atomic: it can mix one
// half of EMPTY (~0) with one half of a key being written, the looking lane's own key included, and skipping that as
// "another key" would insert the key twice.  Slots only go from EMPTY to a key, so a look whose halves are both not ~0 is
// the whole key and is trusted.  Any other look, a fully EMPTY one included, is "unsure": the lane CASes (EMPTY -> its
// key) and decides on the value the CAS returns.  That costs one extra CAS only for real keys with an all-ones half.
__device__ __forceinline__ fq_u64 fq_gb_look(const fq_u64 *k) { return fq_ld_volatile(k); }
__device__ __forceinline__ fq_gb_key2 fq_gb_look(const fq_gb_key2 *k) { return {fq_ld_volatile(&k->lo), fq_ld_volatile(&k->hi)}; }
__device__ __forceinline__ fq_u64 fq_gb_look_s(const fq_u64 *k) { return *(volatile fq_u64 *)k; }
__device__ __forceinline__ fq_gb_key2 fq_gb_look_s(const fq_gb_key2 *k) {
  const volatile fq_u64 *w = (const volatile fq_u64 *)k;
  return {w[0], w[1]};
}
__device__ __forceinline__ bool fq_gb_unsure(fq_u64 k) { return k == FQ_GB_EMPTY; }
__device__ __forceinline__ bool fq_gb_unsure(const fq_gb_key2 &k) { return k.lo == FQ_GB_EMPTY || k.hi == FQ_GB_EMPTY; }
// EMPTY -> key in one atomic; returns what the slot held (EMPTY: the caller claimed it)
__device__ __forceinline__ fq_u64 fq_gb_cas(fq_u64 *k, fq_u64 key) {
  return atomicCAS((unsigned long long *)k, FQ_GB_EMPTY, (unsigned long long)key);
}
__device__ __forceinline__ fq_gb_key2 fq_gb_cas(fq_gb_key2 *k, const fq_gb_key2 &key) { return atomicCAS(k, fq_gb_empty<fq_gb_key2>(), key); }

// slot of `key` in the HBM table (claimed on the spot when new); gb_cap for the key that equals the EMPTY mark; -1 = full
// or not wanted.  Called by every lane that is active at the call site, `want` says which of them search.  The loop's exit
// is a warp vote, so the lanes leave it together whatever their chain lengths: with an early `return slot` the compiler
// threads each exit straight into the caller's atomics and they run once per distinct chain length (ncu: 25 instead of
// 5 atomic instructions per 32 rows at 1000 keys).
template <class Key>
__device__ __forceinline__ fq_i64 fq_gb_find(const fq_launch_params &p, Key *tkeys, Key key, fq_u64 h, bool want) {
  const fq_u32 warp = __activemask();
  fq_i64 slot = -1;
  if (fq_gb_is_empty(key) && want) {
    if (*(volatile fq_u32 *)(p.gb_flags + 1) == 0) p.gb_flags[1] = 1u;
    slot = (fq_i64)p.gb_cap;
    want = false;
  }
  const fq_u64 mask = p.gb_cap - 1;
  const fq_u32 limit = p.gb_cap < 4096 ? (fq_u32)p.gb_cap : 4096u;   // a table that needs longer chains is as good as full
  fq_u64 i = h & mask;
  fq_u32 probe = 0;
  while (__any_sync(warp, want)) {
    if (want) {
      Key cur = fq_gb_look(tkeys + i);
      if (fq_gb_unsure(cur)) cur = fq_gb_cas(tkeys + i, key);
      if (fq_gb_is_empty(cur) || fq_gb_eq(cur, key)) {
        slot = (fq_i64)i;
        want = false;
      } else if (++probe >= limit) {
        if (*(volatile fq_u32 *)p.gb_flags == 0) p.gb_flags[0] = 1u;
        want = false;
      } else {
        i = (i + 1) & mask;
      }
    }
  }
  return slot;
}

// wrapping 64-bit add on a shared-memory slot with two native 32-bit atomics (low word, then the carry into the high word)
__device__ __forceinline__ void fq_atom_add64_s(fq_u64 *slot, fq_u64 x) {
  fq_u32 *w = (fq_u32 *)slot;
  const fq_u32 lo = (fq_u32)x, hi = (fq_u32)(x >> 32);
  fq_u32 carry = 0;
  if (lo) {
    const fq_u32 old = atomicAdd(w, lo);
    carry = (old + lo < old) ? 1u : 0u;
  }
  if (hi + carry) atomicAdd(w + 1, hi + carry);
}

// one group state (Q::G slots: rows, leaves, valid counts) into the CTA's shared-memory table or the table in HBM; called by
// every active lane, `live` says which of them hold a row.  Finding the slot and updating it are kept apart and the search
// keeps the warp together (see fq_gb_find): the warp issues the atomics once, ATOMS for the lanes whose key lives in shared
// memory and ATOMG for the others.
//
// The shared-memory table is searched like any linear-probing table: until the key or a free slot turns up.  A key that
// fits there must NEVER be sent to HBM: all its rows would hit one L2 line (measured: one such key among 1000 costs 40 ms
// per 1e9 rows).  New keys are admitted until the table is 3/4 full (s_used), which keeps the chains short; after that
// unknown keys go to HBM.  smem_try is the lane's patience, +1 per hit and -1 per miss from 64: once fewer than half of
// its rows find their key here, a lane stops looking (an unsuccessful search of a 3/4-full table costs more than the HBM
// atomics it tries to avoid — 1e9 rows, 5000 keys: 53 ms with the search, 33 ms without).
template <class Q>
__device__ __forceinline__ void fq_gb_put(const fq_launch_params &p, typename Q::Key *tkeys, fq_u64 *tslots, typename Q::Key *skeys, fq_u64 *sslots,
                                          fq_u32 *s_used, const typename Q::Key &key, const fq_u64 *st, bool live, int &smem_try) {
  const fq_u32 warp = __activemask();
  const fq_u64 h = fq_gb_seeded(key, p.gb_seed);
  const fq_u32 smask = p.gb_smem_cap - 1;
  const fq_u32 admit = p.gb_smem_cap - (p.gb_smem_cap >> FQ_GB_ADMIT_SHIFT);
  bool in_smem = false;
  bool look = live && p.gb_smem_cap && !fq_gb_is_empty(key) && smem_try > 0;
  const bool looked = look;
  // double hashing (an odd step walks the whole power-of-two table): no primary clustering, so the longest chain among the
  // warp's 32 lanes — the loop's trip count — stays short even at 3/4 load
  const fq_u32 step = ((fq_u32)(h >> 12) | 1u) & smask;
  fq_u32 i = (fq_u32)(h >> 32) & smask, probe = 0;
  while (__any_sync(warp, look)) {
    if (look) {
      typename Q::Key cur = fq_gb_look_s(skeys + i);
      if (fq_gb_unsure(cur)) {
        // an EMPTY look when admissions are closed sends the row to HBM: right whatever the slot really holds
        if (fq_gb_is_empty(cur) && *(volatile fq_u32 *)s_used >= admit) {
          look = false;          // not admitted: this key lives in HBM
        } else {
          cur = fq_gb_cas(skeys + i, key);
          if (fq_gb_is_empty(cur)) atomicAdd(s_used, 1u);
        }
      }
      if (look) {
        if (fq_gb_is_empty(cur) || fq_gb_eq(cur, key)) {
          in_smem = true;
          look = false;
        } else if (++probe >= p.gb_smem_cap) {
          look = false;          // admissions race past 3/4 on a tiny table: full
        } else {
          i = (i + step) & smask;
        }
      }
    }
  }
  if (looked) smem_try = in_smem ? (smem_try < 64 ? smem_try + 1 : 64) : smem_try - 1;
  const fq_i64 slot = fq_gb_find(p, tkeys, key, h, live && !in_smem);
  if (in_smem) Q::gb_merge_s(sslots + (size_t)i * Q::G, st);
  else if (slot >= 0) Q::gb_merge(tslots + (fq_u64)slot * Q::G, st);
}

// One row per lane.  (Folding the lanes of a warp that share a key first — MATCH.ANY + REDUX over the match groups — was
// measured on 1e9 rows, number % 7: 42 ms against 8.2 ms with plain native shared-memory atomics, and removed.)
template <class Q>
__device__ __forceinline__ void fq_gb_row(const fq_launch_params &p, typename Q::Key *tkeys, fq_u64 *tslots, typename Q::Key *skeys, fq_u64 *sslots,
                                          fq_u32 *s_used, const typename Q::Rows &r, int v, fq_u32 &err, int &smem_try) {
  typename Q::Key key = {};
  fq_u64 val[Q::NSLOTS > 0 ? Q::NSLOTS : 1] = {};
  fq_u32 vmask = 0;
  const bool live = Q::gb_row(p, r, v, err, key, val, vmask);
  fq_u64 st[Q::G];
  Q::gb_one(st, val, vmask);
  fq_gb_put<Q>(p, tkeys, tslots, skeys, sslots, s_used, key, st, live, smem_try);
}

template <class Q, int UNROLL>
__device__ __forceinline__ void fq_groupby_kernel(const fq_launch_params &p) {
  constexpr int V = Q::V;
  using Key = typename Q::Key;
  extern __shared__ __align__(128) unsigned char fq_dyn_smem[];
  Key *skeys = (Key *)fq_dyn_smem;   // the keys (16-byte aligned when two words), then the states
  fq_u64 *sslots = (fq_u64 *)(skeys + p.gb_smem_cap);
  __shared__ fq_u32 s_used;   // keys admitted to the shared-memory table
  if (threadIdx.x == 0) s_used = 0;
  for (fq_u32 i = threadIdx.x; i < p.gb_smem_cap; i += blockDim.x) {
    skeys[i] = fq_gb_empty<Key>();
    Q::gb_init(sslots + (size_t)i * Q::G);
  }
  __syncthreads();
  // this CTA's table in HBM: replica blockIdx % gb_reps.  A key that overflows the shared-memory table is hit by every CTA
  // on the same few L2 lines; with replicas only the CTAs that share one collide (1e9 rows, 5000 keys: 117 ms with one table)
  Key *tkeys = (Key *)p.gb_keys;
  fq_u64 *tslots = p.gb_slots;
  if (p.gb_reps > 1) {
    const fq_u32 rep = blockIdx.x % p.gb_reps;
    if (rep) {
      tkeys = (Key *)p.gb_rep_keys + (fq_u64)(rep - 1) * (p.gb_cap + 1);
      tslots = p.gb_rep_slots + (fq_u64)(rep - 1) * (p.gb_cap + 1) * Q::G;
    }
  }
  fq_u32 err = 0;
  int smem_try = 64;
  const fq_u64 nvec = p.unaligned ? 0 : p.n_rows / V;
  const fq_u64 chunk = (fq_u64)blockDim.x * UNROLL;
  const fq_u64 nfull = nvec / chunk;
  for (fq_u64 c = blockIdx.x; c < nfull; c += gridDim.x) {
    const fq_u64 g0 = c * chunk + threadIdx.x;
    typename Q::Rows rows[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; u++) Q::load(rows[u], p, g0 + (fq_u64)u * blockDim.x);
#pragma unroll
    for (int u = 0; u < UNROLL; u++)
#pragma unroll
      for (int v = 0; v < V; v++) fq_gb_row<Q>(p, tkeys, tslots, skeys, sslots, &s_used, rows[u], v, err, smem_try);
  }
  const fq_u64 tid = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x;
  const fq_u64 nthreads = (fq_u64)gridDim.x * blockDim.x;
  for (fq_u64 g = nfull * chunk + tid; g < nvec; g += nthreads) {
    typename Q::Rows r;
    Q::load(r, p, g);
#pragma unroll
    for (int v = 0; v < V; v++) fq_gb_row<Q>(p, tkeys, tslots, skeys, sslots, &s_used, r, v, err, smem_try);
  }
  for (fq_u64 row = nvec * V + tid; row < p.n_rows; row += nthreads) {
    typename Q::Rows r;
    Q::load1(r, p, row);
    fq_gb_row<Q>(p, tkeys, tslots, skeys, sslots, &s_used, r, 0, err, smem_try);
  }
  __syncthreads();
  // flush the CTA's groups into the table in HBM
  for (fq_u32 i = threadIdx.x; i < p.gb_smem_cap; i += blockDim.x) {
    const Key key = skeys[i];
    const fq_i64 slot = fq_gb_find(p, tkeys, key, fq_gb_seeded(key, p.gb_seed), !fq_gb_is_empty(key));
    if (slot >= 0) Q::gb_merge(tslots + (fq_u64)slot * Q::G, sslots + (size_t)i * Q::G);
  }
  if (err) atomicOr((fq_u32 *)(p.result + 1), err);
}

// partial groups folded into the table.  With gb_entries: n_rows entries of KW + Q::G slots (the packed key's KW words,
// the state — what fq_pipe_export_partials writes).  Without: the (gb_reps - 1) replicas the aggregation kernel filled,
// n_rows = (gb_reps - 1) * (gb_cap + 1) of their slots; every group met is folded into the table and its replica slot is
// reset (every word of its key), so the replicas are empty again when the kernel ends.
template <class Q>
__device__ __forceinline__ void fq_groupby_merge_kernel(const fq_launch_params &p) {
  using Key = typename Q::Key;
  constexpr int KW = sizeof(Key) / 8;
  const fq_u64 tid = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x;
  const fq_u64 nthreads = (fq_u64)gridDim.x * blockDim.x;
  if (p.gb_entries) {
    for (fq_u64 e = tid; e < p.n_rows; e += nthreads) {
      const fq_u64 *ent = p.gb_entries + e * (KW + Q::G);
      Key key;
      fq_gb_from_words(key, ent);
      const fq_i64 slot = fq_gb_find(p, (Key *)p.gb_keys, key, fq_gb_seeded(key, p.gb_seed), true);
      if (slot >= 0) Q::gb_merge(p.gb_slots + (fq_u64)slot * Q::G, ent + KW);
    }
    return;
  }
  for (fq_u64 e = tid; e < p.n_rows; e += nthreads) {
    const bool special = e % (p.gb_cap + 1) == p.gb_cap;   // the slot of the key that equals the EMPTY mark
    const Key key = special ? fq_gb_empty<Key>() : ((Key *)p.gb_rep_keys)[e];
    fq_u64 *from = p.gb_rep_slots + e * Q::G;
    const bool occupied = special ? from[0] != 0 : !fq_gb_is_empty(key);   // from[0] = the group's row count
    const fq_i64 slot = fq_gb_find(p, (Key *)p.gb_keys, key, fq_gb_seeded(key, p.gb_seed), occupied);
    if (slot >= 0) Q::gb_merge(p.gb_slots + (fq_u64)slot * Q::G, from);
    if (occupied) {
      if (!special) ((Key *)p.gb_rep_keys)[e] = fq_gb_empty<Key>();
      Q::gb_init(from);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// fq_map_kernel — projection of every row (no predicate): out_i[row] = expr_i(row)
// ---------------------------------------------------------------------------------------------
template <class Q, int UNROLL>
__device__ __forceinline__ void fq_map_kernel(const fq_launch_params &p) {
  constexpr int V = Q::V;
  fq_u32 err = 0;
  const fq_u64 nvec = p.unaligned ? 0 : p.n_rows / V;
  const fq_u64 chunk = (fq_u64)blockDim.x * UNROLL;
  const fq_u64 nfull = nvec / chunk;
  for (fq_u64 c = blockIdx.x; c < nfull; c += gridDim.x) {
    const fq_u64 g0 = c * chunk + threadIdx.x;
    typename Q::Rows rows[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; u++) Q::load(rows[u], p, g0 + (fq_u64)u * blockDim.x);
#pragma unroll
    for (int u = 0; u < UNROLL; u++) {
      const fq_u64 row0 = (g0 + (fq_u64)u * blockDim.x) * V;
      if (row0 + V <= p.capacity) {
        Q::emit_vec(rows[u], p, row0, err);   // one vector store per output column
      } else {
#pragma unroll
        for (int v = 0; v < V; v++)
          if (row0 + v < p.capacity) Q::emit(rows[u], v, p, row0 + v, err);
      }
    }
  }
  const fq_u64 tid = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x;
  const fq_u64 nthreads = (fq_u64)gridDim.x * blockDim.x;
  for (fq_u64 g = nfull * chunk + tid; g < nvec; g += nthreads) {
    typename Q::Rows r;
    Q::load(r, p, g);
    if (g * V + V <= p.capacity) {
      Q::emit_vec(r, p, g * V, err);
    } else {
#pragma unroll
      for (int v = 0; v < V; v++)
        if (g * V + v < p.capacity) Q::emit(r, v, p, g * V + v, err);
    }
  }
  for (fq_u64 row = nvec * V + tid; row < p.n_rows; row += nthreads) {
    typename Q::Rows r;
    Q::load1(r, p, row);
    if (row < p.capacity) Q::emit(r, 0, p, row, err);
  }
  if (err) atomicOr((fq_u32 *)(p.result + 1), err);
  if (tid == 0) p.result[0] = p.n_rows;
}

// ---------------------------------------------------------------------------------------------
// fq_map_tma_kernel — fq_map_kernel with its reads staged by the bulk-copy engine (same ring as fq_agg_tma_kernel):
// the loads in flight no longer compete with the output vectors for registers.  Consumers read a staged tile with
// LDS.128, evaluate every select expression and write one vector store per output column per group.
// ---------------------------------------------------------------------------------------------
template <class Q, int U, int STAGES>
__device__ __forceinline__ void fq_map_tma_kernel(const fq_launch_params &p) {
  constexpr int V = Q::V;
  extern __shared__ __align__(128) unsigned char fq_dyn_smem[];
  __shared__ __align__(8) fq_u64 s_bars[2 * STAGES];
  const int lane = threadIdx.x & 31;
  const int cthreads = (int)blockDim.x - 32, cwarps = cthreads >> 5;
  const bool is_producer = (int)threadIdx.x >= cthreads;
  const fq_u32 tile_groups = (fq_u32)cthreads * U;
  const fq_u64 tile_rows = (fq_u64)tile_groups * V;
  const fq_u32 stage_bytes = Q::stage_bytes((fq_u32)tile_rows);
  const fq_u64 n_tiles = p.unaligned ? 0 : p.n_rows / tile_rows;
  const int stages = (int)p.stages;
  fq_u32 err = 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; s++) {
      fq_mbar_init(fq_smem_addr(&s_bars[s]), 1);
      fq_mbar_init(fq_smem_addr(&s_bars[STAGES + s]), cwarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (is_producer) {
    if (lane == 0) {
      int slot = 0;
      fq_u32 round = 0;
      for (fq_u64 t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        if (round >= 1) fq_mbar_wait(fq_smem_addr(&s_bars[STAGES + slot]), (round - 1) & 1);
        const fq_u32 full = fq_smem_addr(&s_bars[slot]);
        fq_mbar_expect_tx(full, stage_bytes);
        Q::tma_issue(p, fq_smem_addr(fq_dyn_smem + (size_t)slot * stage_bytes), full, t, (fq_u32)tile_rows);
        if (++slot == stages) { slot = 0; round++; }
      }
    }
    return;
  }
  int slot = 0;
  fq_u32 round = 0;
  for (fq_u64 t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    fq_mbar_wait(fq_smem_addr(&s_bars[slot]), round & 1);
    const unsigned char *stage = fq_dyn_smem + (size_t)slot * stage_bytes;
    typename Q::Rows rows[U];
#pragma unroll
    for (int u = 0; u < U; u++)
      Q::load_smem(rows[u], p, stage, (fq_u32)tile_rows, (fq_u32)(u * cthreads + (int)threadIdx.x), t * tile_groups + (fq_u64)u * cthreads + threadIdx.x);
    __syncwarp();
    if (lane == 0) fq_mbar_arrive(fq_smem_addr(&s_bars[STAGES + slot]));   // the tile is in registers: hand the slot back
    if (++slot == stages) { slot = 0; round++; }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const fq_u64 row0 = (t * tile_groups + (fq_u64)u * cthreads + threadIdx.x) * V;
      if (row0 + V <= p.capacity) {
        Q::emit_vec(rows[u], p, row0, err);
      } else {
#pragma unroll
        for (int v = 0; v < V; v++)
          if (row0 + v < p.capacity) Q::emit(rows[u], v, p, row0 + v, err);
      }
    }
  }
  // rows past the last full tile: plain loads, spread over the consumers of the whole grid
  const fq_u64 ctid = (fq_u64)blockIdx.x * cthreads + threadIdx.x;
  const fq_u64 cn = (fq_u64)gridDim.x * cthreads;
  const fq_u64 nvec = p.unaligned ? 0 : p.n_rows / V;
  for (fq_u64 g = n_tiles * tile_groups + ctid; g < nvec; g += cn) {
    typename Q::Rows r;
    Q::load(r, p, g);
    if (g * V + V <= p.capacity) {
      Q::emit_vec(r, p, g * V, err);
    } else {
#pragma unroll
      for (int v = 0; v < V; v++)
        if (g * V + v < p.capacity) Q::emit(r, v, p, g * V + v, err);
    }
  }
  for (fq_u64 row = nvec * V + ctid; row < p.n_rows; row += cn) {
    typename Q::Rows r;
    Q::load1(r, p, row);
    if (row < p.capacity) Q::emit(r, 0, p, row, err);
  }
  if (err) atomicOr((fq_u32 *)(p.result + 1), err);
  if (ctid == 0) p.result[0] = p.n_rows;
}
