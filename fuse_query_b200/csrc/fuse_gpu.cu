// fuse_gpu.cu — implementation of the C ABI in include/fuse_gpu.h.
//
// Host side of libfuse_gpu.so: contexts, device columns, the pipe compiler front end (codegen ->
// precompiled table lookup -> NVRTC), launch shapes and result decoding.  No torch, no Python.
// libcuda and libnvrtc are dlopen'ed on first use so the library loads (and exports its symbols) on a
// machine without a GPU; every data-path entry point then fails loudly with FQ_ERR_CUDA.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <cinttypes>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/fuse_gpu.h"
#include "codegen.h"
#include "kernels/fq_skeleton.cuh"
#include "kernels/fq_sort.cuh"
#include "kernels/fq_utf8.cuh"
#include "generated/skeleton_embed.h"  // static const char fq_skeleton_src[]

// ---------------------------------------------------------------------------------------------
// precompiled kernels (generated/aot_kernels.cu)
// ---------------------------------------------------------------------------------------------
struct fq_aot_entry { const char *name; const void *fn; };
extern "C" const fq_aot_entry fq_aot_table[];
extern "C" const int fq_aot_count;

namespace {

thread_local std::string g_err;

fq_status set_err(fq_status st, const char *f, ...) __attribute__((format(printf, 2, 3)));
fq_status set_err(fq_status st, const char *f, ...) {
  char buf[2048];
  va_list ap;
  va_start(ap, f);
  vsnprintf(buf, sizeof buf, f, ap);
  va_end(ap);
  g_err = buf;
  return st;
}
#define CUDA_TRY(expr)                                                                                \
  do {                                                                                                \
    cudaError_t e_ = (expr);                                                                          \
    if (e_ != cudaSuccess) return set_err(FQ_ERR_CUDA, "CUDA error: %s (%s)", cudaGetErrorString(e_), #expr); \
  } while (0)

// ---- driver API + NVRTC through dlopen ----
typedef int CUresult_;
typedef struct CUmod_st *CUmodule_;
typedef struct CUfunc_st *CUfunction_;
struct Driver {
  void *h = nullptr;
  CUresult_ (*cuModuleLoadData)(CUmodule_ *, const void *) = nullptr;
  CUresult_ (*cuModuleGetFunction)(CUfunction_ *, CUmodule_, const char *) = nullptr;
  CUresult_ (*cuModuleUnload)(CUmodule_) = nullptr;
  CUresult_ (*cuLaunchKernel)(CUfunction_, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, void *, void **,
                              void **) = nullptr;
  CUresult_ (*cuOccupancyMaxActiveBlocksPerMultiprocessor)(int *, CUfunction_, int, size_t) = nullptr;
  CUresult_ (*cuFuncSetAttribute)(CUfunction_, int, int) = nullptr;
  CUresult_ (*cuGetErrorString)(CUresult_, const char **) = nullptr;
  std::string why;
  bool load() {
    if (h) return true;
    h = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { why = dlerror(); return false; }
#define SYM(n) *(void **)(&n) = dlsym(h, #n)
    SYM(cuModuleLoadData); SYM(cuModuleGetFunction); SYM(cuModuleUnload); SYM(cuLaunchKernel);
    SYM(cuOccupancyMaxActiveBlocksPerMultiprocessor); SYM(cuGetErrorString); SYM(cuFuncSetAttribute);
#undef SYM
    if (!cuModuleLoadData || !cuModuleGetFunction || !cuLaunchKernel || !cuOccupancyMaxActiveBlocksPerMultiprocessor) {
      why = "libcuda.so.1 lacks required symbols";
      return false;
    }
    return true;
  }
  std::string err(CUresult_ r) {
    const char *s = nullptr;
    if (cuGetErrorString) cuGetErrorString(r, &s);
    return s ? s : "unknown driver error";
  }
};
typedef struct _nvrtcProgram *nvrtcProgram_;
struct Nvrtc {
  void *h = nullptr;
  int (*nvrtcCreateProgram)(nvrtcProgram_ *, const char *, const char *, int, const char *const *, const char *const *) = nullptr;
  int (*nvrtcCompileProgram)(nvrtcProgram_, int, const char *const *) = nullptr;
  int (*nvrtcGetCUBINSize)(nvrtcProgram_, size_t *) = nullptr;
  int (*nvrtcGetCUBIN)(nvrtcProgram_, char *) = nullptr;
  int (*nvrtcGetProgramLogSize)(nvrtcProgram_, size_t *) = nullptr;
  int (*nvrtcGetProgramLog)(nvrtcProgram_, char *) = nullptr;
  int (*nvrtcDestroyProgram)(nvrtcProgram_ *) = nullptr;
  const char *(*nvrtcGetErrorString)(int) = nullptr;
  int (*nvrtcVersion)(int *, int *) = nullptr;
  std::string why;
  bool load() {
    if (h) return true;
    const char *cands[] = {"libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12", "libnvrtc.so",
                           "/usr/local/cuda/lib64/libnvrtc.so"};
    for (const char *c : cands) {
      h = dlopen(c, RTLD_NOW);
      if (h) break;
    }
    if (!h) { why = dlerror(); return false; }
#define SYM(n) *(void **)(&n) = dlsym(h, #n)
    SYM(nvrtcCreateProgram); SYM(nvrtcCompileProgram); SYM(nvrtcGetCUBINSize); SYM(nvrtcGetCUBIN);
    SYM(nvrtcGetProgramLogSize); SYM(nvrtcGetProgramLog); SYM(nvrtcDestroyProgram); SYM(nvrtcGetErrorString); SYM(nvrtcVersion);
#undef SYM
    if (!nvrtcCreateProgram || !nvrtcCompileProgram || !nvrtcGetCUBIN) { why = "libnvrtc lacks required symbols"; return false; }
    return true;
  }
};
Driver g_drv;
Nvrtc g_nvrtc;
std::mutex g_mu;

// Launch shapes.  Defaults are the macros the precompiled kernels were built with; FQ_TUNE_* environment
// overrides (kernel tuning experiments only) force the NVRTC path so kernel and host agree.
struct Shapes {
  int agg_threads = FQ_AGG_THREADS, agg_min_blocks = FQ_AGG_MIN_BLOCKS;
  int tma_threads = FQ_TMA_THREADS, tma_unroll = FQ_TMA_UNROLL, tma_stages = FQ_TMA_STAGES, tma_min_blocks = FQ_TMA_MIN_BLOCKS;
  int tma_stages_env = 0;   // FQ_TUNE_TMA_STAGES: ring depth override (<= FQ_TMA_STAGES)
  int sel_threads = FQ_SEL_THREADS, sel_min_blocks = FQ_SEL_MIN_BLOCKS, sel_unroll = FQ_SEL_UNROLL, sel_seg = FQ_SEL_SEG, sel_look = FQ_SEL_LOOK;
  int map_threads = FQ_MAP_THREADS, map_min_blocks = FQ_MAP_MIN_BLOCKS, map_unroll = FQ_MAP_UNROLL;
  int selt_threads = FQ_SELT_THREADS, selt_unroll = FQ_SELT_UNROLL, selt_seg = FQ_SELT_SEG, selt_lag = FQ_SELT_LAG;
  int seld_threads = FQ_SELD_THREADS, seld_unroll = FQ_SELD_UNROLL, seld_seg = FQ_SELD_SEG, seld_stages = 12;   // 12 x 14 KB in flight: 4.04 ms for a selection that keeps all of 1e9 rows (8 stages: 4.33)
  int selt_stages_env = 0;  // FQ_TUNE_SELT_STAGES: ring depth override (<= FQ_SELT_STAGES)
  bool tuned = false;
  Shapes() {
    auto env = [&](const char *name, int *v) {
      const char *e = getenv(name);
      if (e && atoi(e) > 0) { *v = atoi(e); tuned = true; }
    };
    env("FQ_TUNE_AGG_THREADS", &agg_threads); env("FQ_TUNE_AGG_MIN_BLOCKS", &agg_min_blocks);
    env("FQ_TUNE_TMA_THREADS", &tma_threads); env("FQ_TUNE_TMA_UNROLL", &tma_unroll);
    if (getenv("FQ_TUNE_TMA_STAGES") && atoi(getenv("FQ_TUNE_TMA_STAGES")) > 0) tma_stages_env = atoi(getenv("FQ_TUNE_TMA_STAGES"));
    env("FQ_TUNE_TMA_MIN_BLOCKS", &tma_min_blocks);
    env("FQ_TUNE_SEL_THREADS", &sel_threads); env("FQ_TUNE_SEL_MIN_BLOCKS", &sel_min_blocks); env("FQ_TUNE_SEL_UNROLL", &sel_unroll); env("FQ_TUNE_SEL_SEG", &sel_seg); env("FQ_TUNE_SEL_LOOK", &sel_look);
    env("FQ_TUNE_SELT_THREADS", &selt_threads); env("FQ_TUNE_SELT_UNROLL", &selt_unroll); env("FQ_TUNE_SELT_SEG", &selt_seg); env("FQ_TUNE_SELT_LAG", &selt_lag);
    if (getenv("FQ_TUNE_SELT_STAGES") && atoi(getenv("FQ_TUNE_SELT_STAGES")) > 0) selt_stages_env = atoi(getenv("FQ_TUNE_SELT_STAGES"));
    env("FQ_TUNE_SELD_THREADS", &seld_threads); env("FQ_TUNE_SELD_UNROLL", &seld_unroll); env("FQ_TUNE_SELD_SEG", &seld_seg); env("FQ_TUNE_SELD_STAGES", &seld_stages);
    env("FQ_TUNE_MAP_THREADS", &map_threads); env("FQ_TUNE_MAP_MIN_BLOCKS", &map_min_blocks); env("FQ_TUNE_MAP_UNROLL", &map_unroll);
    if (getenv("FQ_TUNE_EXTRA")) tuned = true;
  }
  std::string defines() const {
    char b[2048];
    snprintf(b, sizeof b,
             "#define FQ_SELD_THREADS %d\n#define FQ_SELD_UNROLL %d\n#define FQ_SELD_SEG %d\n#define FQ_SELD_PROBE_ROWS 512\n"
             "#define FQ_SELT_THREADS %d\n#define FQ_SELT_UNROLL %d\n#define FQ_SELT_SEG %d\n#define FQ_SELT_STAGES 8\n#define FQ_SELT_LAG %d\n"
             "#define FQ_AGG_THREADS %d\n#define FQ_AGG_MIN_BLOCKS %d\n#define FQ_TMA_THREADS %d\n"
             "#define FQ_TMA_UNROLL %d\n#define FQ_TMA_STAGES %d\n#define FQ_TMA_MIN_BLOCKS %d\n#define FQ_SEL_THREADS %d\n"
             "#define FQ_SEL_MIN_BLOCKS %d\n#define FQ_SEL_UNROLL %d\n#define FQ_SEL_SEG %d\n#define FQ_SEL_LOOK %d\n#define FQ_MAP_THREADS %d\n#define FQ_MAP_MIN_BLOCKS %d\n#define FQ_MAP_UNROLL %d\n",
             seld_threads, seld_unroll, seld_seg, selt_threads, selt_unroll, selt_seg, selt_lag, agg_threads, agg_min_blocks, tma_threads, tma_unroll, tma_stages, tma_min_blocks, sel_threads, sel_min_blocks, sel_unroll, sel_seg, sel_look, map_threads, map_min_blocks, map_unroll);
    std::string out = b;
    // FQ_TUNE_EXTRA: raw preprocessor text for A/B experiments, ';' separates lines ("#define FQ_STORE_CS 0;#define FQ_L2_HINTS 0")
    if (const char *x = getenv("FQ_TUNE_EXTRA")) {
      std::string t = x;
      for (char &c : t) if (c == ';') c = '\n';
      out += t + "\n";
    }
    return out;
  }
};
const Shapes &shapes() {
  static Shapes s;
  return s;
}

// The kernels a pipe can launch, one slot per wrapper fq::generate emits
enum Slot { K_AGG_U4, K_AGG_TMA, K_SELECT, K_SELECT_TMA, K_SELECT_DENSE, K_SELECT_PROBE, K_MAP, K_MAP_TMA, K_GROUPBY, K_GBMERGE, K_SLOTS };

struct Kernel {
  // planned by plan_kernels
  const char *suffix = nullptr;   // of the wrapper fqk_<tag><suffix>; null when the pipe cannot launch this slot
  bool staged = false;            // on the bulk-copy staged path (the density probe goes with the dense build)
  bool one_per_sm = false;        // at most one CTA per SM whatever the occupancy
  int threads = 256;
  unsigned smem = 0;              // dynamic shared memory per CTA
  unsigned stages = 0;            // ring depth (fq_launch_params::stages)
  uint64_t rows = 0;              // source rows one CTA claims at a time (chunk or segment): the unit of a persistent grid
  // filled in by resolve_kernel
  const void *aot = nullptr;   // host stub of a precompiled kernel (cudaLaunchKernel)
  CUfunction_ jit = nullptr;   // NVRTC-built (cuLaunchKernel)
  int blocks_per_sm = 1;
  bool valid() const { return aot || jit; }
};

// Every kernel the pipe can launch with its launch shape: the wrappers fq::generate emits for the pipe's kind, less a staged
// one whose ring does not fit 200 KB.  Also the CTA's shared-memory table size of a GROUP BY pipe.
void plan_kernels(const fq::Generated &gen, Kernel *k, unsigned *gb_smem_cap) {
  const Shapes &s = shapes();
  const int V = gen.vec;
  auto unroll = [&](int u) { return u * V <= 32 ? u : 32 / V; };   // fq_sel{,t,d}_shape<V>::U
  auto seg_rows = [&](int threads, int cfg_u, int cfg_seg) {        // threads x U x V x fq_sel{,t,d}_shape<V>::SEG
    const int u = unroll(cfg_u);
    return (uint64_t)threads * u * V * (cfg_seg * u * V <= 64 ? cfg_seg : 64 / (u * V));
  };
  auto plan = [&](Slot slot, const char *suffix, int threads, uint64_t rows) {
    k[slot].suffix = suffix;
    k[slot].threads = threads;
    k[slot].rows = rows;
    return &k[slot];
  };
  // a staged kernel: a ring of tiles of `trows` rows, `row_bytes` per row plus `bitmaps` validity bitmaps; as many tiles as
  // fit `budget` (or the FQ_TUNE_* depth `env`), within [lo, hi]
  auto staged = [&](Slot slot, const char *suffix, int threads, uint64_t rows, unsigned trows, int row_bytes, int bitmaps, int env,
                    unsigned budget, unsigned lo, unsigned hi) {
    const unsigned tile = trows * row_bytes + bitmaps * (trows / 8);
    const unsigned stages = std::min(std::max(env > 0 ? (unsigned)env : budget / tile, lo), hi);
    if (stages * tile > 200u * 1024u) return false;
    Kernel *e = plan(slot, suffix, threads, rows);
    e->staged = true;
    e->stages = stages;
    e->smem = stages * tile;
    return true;
  };
  const unsigned tma_rows = (unsigned)s.tma_threads * s.tma_unroll * V;
  if (gen.kind == FQ_PIPE_GROUPBY) {
    // shared-memory table of the CTA: the largest power of two of (key words + state) slots within 96 KB (two CTAs per SM)
    const unsigned entry = 8u * ((unsigned)gen.key_words + 1u + (unsigned)gen.n_slots);
    unsigned cap = 1;
    while (cap * 2 * entry <= 96u * 1024u) cap *= 2;
    static const int smem_env = getenv("FQ_GB_SMEM_SLOTS") ? atoi(getenv("FQ_GB_SMEM_SLOTS")) : -1;
    if (smem_env >= 0) { cap = 1; while ((int)cap * 2 <= smem_env) cap *= 2; if (smem_env == 0) cap = 0; }
    *gb_smem_cap = cap;
    plan(K_GROUPBY, "_groupby", FQ_GB_THREADS, (uint64_t)FQ_GB_THREADS * FQ_GB_UNROLL * V)->smem = cap * entry;
    plan(K_GBMERGE, "_gbmerge", 256, 0);
  } else if (gen.kind == FQ_PIPE_AGGREGATE) {
    plan(K_AGG_U4, "_agg_u4", s.agg_threads, (uint64_t)s.agg_threads * 4 * V);
    // producer warp + consumers; ring of ~128 KB per CTA (measured optimum on B200)
    if (gen.tma_ok)
      staged(K_AGG_TMA, "_agg_tma", s.tma_threads + 32, tma_rows, tma_rows, gen.row_bytes, gen.row_bitmaps, s.tma_stages_env, 128u * 1024u, 2,
             FQ_TMA_STAGES);
  } else if (gen.has_pred) {
    plan(K_SELECT, "_select", s.sel_threads + 32, seg_rows(s.sel_threads, s.sel_unroll, s.sel_seg));   // worker warps + one scan warp
    // sparse-tuned build: consumer warps + scan warp + producer warp; pass 1 stages the predicate's columns.  ~192 KB in
    // flight per SM measured best here (1.19 -> 1.14 ms at 1e9 rows; the aggregate kernel peaks at 128 KB)
    // dense-tuned build: both passes staged, so a slot holds a tile of EVERY referenced column; small tiles, a ring of
    // ~112 KB, and one CTA per SM (the look-back window covers a grid of one CTA per SM)
    if (gen.sel_tma_ok &&
        staged(K_SELECT_TMA, "_select_tma", s.selt_threads + 64, seg_rows(s.selt_threads, s.selt_unroll, s.selt_seg),
               (unsigned)s.selt_threads * unroll(s.selt_unroll) * V, gen.pred_row_bytes, gen.pred_row_bitmaps, s.selt_stages_env, 192u * 1024u, 2,
               FQ_SELT_STAGES) &&
        staged(K_SELECT_DENSE, "_select_dense", s.seld_threads + 64, seg_rows(s.seld_threads, s.seld_unroll, s.seld_seg),
               (unsigned)s.seld_threads * unroll(s.seld_unroll) * V, gen.row_bytes, gen.row_bitmaps, s.seld_stages, 0, 3, 16)) {
      k[K_SELECT_DENSE].one_per_sm = true;
      plan(K_SELECT_PROBE, "_select_probe", 128, 0)->staged = true;
    }
  } else {
    plan(K_MAP, "_map", s.map_threads, (uint64_t)s.map_threads * s.map_unroll * V);
    if (gen.tma_ok)
      staged(K_MAP_TMA, "_map_tma", s.tma_threads + 32, tma_rows, tma_rows, gen.row_bytes, gen.row_bitmaps, s.tma_stages_env, 128u * 1024u, 2,
             FQ_TMA_STAGES);
  }
}

// Kernel variant a pipe's launches prefer.  tma: the staged kernel (a selection: the sparse-tuned build, and the dense-tuned
// one when the density probe says so); sparse / dense: that staged select build alone; ldg: the LDG kernel.
enum Variant { V_TMA, V_SPARSE, V_DENSE, V_LDG };
// the words each kind of pipe accepts, by the variable that sets its default; a GROUP BY pipe has no variant
const struct { const char *env, *word; Variant v; } kVariants[] = {
    {"FQ_AGG_VARIANT", "tma", V_TMA},    {"FQ_AGG_VARIANT", "u4", V_LDG},       {"FQ_SEL_VARIANT", "tma", V_TMA},
    {"FQ_SEL_VARIANT", "sparse", V_SPARSE}, {"FQ_SEL_VARIANT", "dense", V_DENSE}, {"FQ_SEL_VARIANT", "ldg", V_LDG},
    {"FQ_MAP_VARIANT", "tma", V_TMA},    {"FQ_MAP_VARIANT", "ldg", V_LDG}};
const char *variant_env(const fq::Generated &gen) {
  return gen.kind == FQ_PIPE_GROUPBY ? nullptr : gen.kind == FQ_PIPE_AGGREGATE ? "FQ_AGG_VARIANT" : gen.has_pred ? "FQ_SEL_VARIANT" : "FQ_MAP_VARIANT";
}
fq_status parse_variant(const fq::Generated &gen, const char *word, Variant *out) {
  const char *env = variant_env(gen);
  for (const auto &w : kVariants)
    if (env && strcmp(w.env, env) == 0 && strcmp(w.word, word) == 0) { *out = w.v; return FQ_OK; }
  return set_err(FQ_ERR_INVALID, "Internal Error: unknown kernel variant %s", word);
}

struct Module {  // one compiled specialisation, shared by every pipe with the same tag
  std::map<std::string, Kernel> kernels;
  std::vector<std::string> built;   // JIT: suffixes of the kernels in the module
  bool from_disk_cache = false;     // JIT: the cubin came from the on-disk cache instead of NVRTC
  bool precompiled = false;
  CUmodule_ mod = nullptr;
};

}  // namespace

// launches recorded between fq_graph_begin and fq_graph_end
struct fq_graph {
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  std::vector<cudaEvent_t> done;   // the "results are ready" events of the pipes launched inside, recorded after every replay
  uint64_t launches = 0;           // kernels per replay (fq_ctx_launch_count)
};

struct fq_ctx {
  int device = 0;
  int sm_count = 0;
  std::atomic<uint64_t> launches{0};
  std::mutex mu;
  std::map<std::string, Module> modules;  // tag -> module
  // ORDER BY scratch: kept between sorts (growing a 24-bytes-per-row buffer costs ~0.3 s per GB of fresh device memory, far
  // more than the sort itself); fq_ctx_trim gives it back
  std::mutex sort_mu;
  void *sort_scratch = nullptr;
  size_t sort_scratch_bytes = 0;
  cudaEvent_t sort_done = nullptr;        // the last sort's final copy out of the scratch
  fq_graph *recording = nullptr;          // set between fq_graph_begin and fq_graph_end
  cudaStream_t recording_stream = nullptr;
  uint64_t recording_launches0 = 0;
};

struct fq_column {
  fq_dtype dtype = FQ_NULL;
  uint64_t len = 0;
  void *ptr = nullptr;
  bool owned = false;
  const fq_column *validity = nullptr;   // FQ_BOOL, one byte per row; borrowed unless owns_validity (slices)
  bool owns_validity = false;
  const fq_column *validity_bits = nullptr;   // or: FQ_U8 column holding an Arrow LSB-first bitmap (borrowed), row 0 = bit validity_bit0
  uint64_t validity_bit0 = 0;
};

// Exchange windows of a group of ranks (one process per GPU): the merge point across GPUs (processor_merge.rs:37-66).
struct fq_group {
  int rank = 0, world = 1;
  uint32_t row_slots = 0;          // 8-byte slots per (parity, writer) row, slot 0 = epoch
  uint64_t *window = nullptr;      // local: 2 * world * row_slots slots
  uint64_t *windows[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  bool ipc_opened[8] = {false, false, false, false, false, false, false, false};
  bool connected = false;
  uint64_t epoch = 0;              // one per group operation; every rank issues the same sequence of operations
  uint64_t timeout_ns = 20ull * 1000 * 1000 * 1000;
  uint64_t *d_result = nullptr, *h_result = nullptr;   // gather: [0] rows selected by all ranks, [1] final rows, [2] error bits
  cudaEvent_t ev = nullptr;
  bool gathered = false;
};

struct fq_pipe {
  fq::Generated gen;
  Kernel k[K_SLOTS];   // plan_kernels, resolved by fq_pipe_compile
  // GROUP BY: the hash table in HBM
  uint64_t *gb_keys = nullptr, *gb_slots = nullptr;
  uint64_t *gb_rep_keys = nullptr, *gb_rep_slots = nullptr;   // gb_reps - 1 more tables of gb_cap + 1 slots (see fq_groupby_kernel)
  unsigned gb_reps = 1;
  bool gb_reps_dirty = false;        // freshly allocated replicas: fill them once; afterwards the fold leaves them empty
  uint64_t gb_cap = 0;
  uint64_t gb_seed = 0;              // hash seed of the current table (fq_launch_params::gb_seed)
  uint64_t gb_reservations = 0;
  uint32_t *gb_flags = nullptr;      // [0] overflow, [1] EMPTY-valued key seen, [2..3] group count (u64), [4..5] error bits
  uint64_t *h_gb = nullptr;          // pinned mirror of gb_flags (4 x u64)
  uint64_t *gb_identity = nullptr;   // device copy of a fresh group's state
  unsigned gb_smem_cap = 0;
  bool launched_groupby = false;

  int build_kind = 0;   // 0 precompiled, 1 NVRTC in this process, 2 on-disk JIT cache
  Variant variant = V_TMA;   // FQ_{AGG,SEL,MAP}_VARIANT when the pipe was compiled, or fq_pipe_set_variant
  fq_group *group = nullptr;   // aggregate launches end with the in-kernel cross-GPU merge when set
  uint64_t *d_merged = nullptr, *h_merged = nullptr;
  bool launched_merged = false;
  bool precompiled = false;
  int n_slots = 0;          // FQ_STATE_HDR + leaves
  uint64_t *d_state = nullptr, *d_partials = nullptr, *d_ctl = nullptr, *d_tiles = nullptr;
  uint32_t *d_blocks = nullptr;   // reference-block hit bitmap (FQ_RUN_BLOCK_STATS)
  uint64_t blocks_cap = 0;
  uint64_t *h_state = nullptr, *h_result = nullptr;  // pinned
  int partials_cap = 0;
  uint64_t tiles_cap = 0;
  cudaEvent_t ev = nullptr;
  bool launched = false, launched_project = false;
  uint64_t capacity_eff = 0;
  bool skipped = false;     // project launch over zero rows
  bool project_has_pred_launch = false;
  // bit tables of the pipe's FQ_EXPR_LOOKUP nodes (fq_pipe_set_lookup), borrowed
  const fq_u8 *lookup[FQ_MAX_LOOKUPS] = {nullptr, nullptr, nullptr, nullptr};
  uint64_t lookup_bits[FQ_MAX_LOOKUPS] = {0, 0, 0, 0};
  unsigned lookup_bound = 0;   // bit k: slot k is bound
};
static_assert(sizeof(((fq_launch_params *)nullptr)->lookup) / sizeof(void *) == FQ_MAX_LOOKUPS, "fq_launch_params holds FQ_MAX_LOOKUPS tables");

namespace {

fq_status use(fq_ctx *ctx) {
  if (!ctx) return set_err(FQ_ERR_INVALID, "Internal Error: null context");
  CUDA_TRY(cudaSetDevice(ctx->device));
  return FQ_OK;
}

__global__ void __launch_bounds__(256) fq_fill_numbers(fq_u64 *dst, fq_u64 begin, fq_u64 n) {
  // two values (16 B) per thread per step; dst is 16-byte aligned when (dst offset) is even
  const fq_u64 tid = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x;
  const fq_u64 nthreads = (fq_u64)gridDim.x * blockDim.x;
  const bool aligned = (((fq_u64)dst) & 15) == 0;
  if (aligned) {
    const fq_u64 nvec = n / 2;
    // each CTA writes contiguous 16-KB chunks: 4 independent 16-byte stores in flight per thread, every warp store one 512-B run
    const fq_u64 chunk = 4ull * blockDim.x, nfull = nvec / chunk;
    for (fq_u64 c = blockIdx.x; c < nfull; c += gridDim.x) {
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const fq_u64 g = c * chunk + (fq_u64)k * blockDim.x + threadIdx.x;
        ulonglong2 v;
        v.x = begin + 2 * g;
        v.y = begin + 2 * g + 1;
        reinterpret_cast<ulonglong2 *>(dst)[g] = v;
      }
    }
    for (fq_u64 g = nfull * chunk + tid; g < nvec; g += nthreads) {
      ulonglong2 v;
      v.x = begin + 2 * g;
      v.y = begin + 2 * g + 1;
      reinterpret_cast<ulonglong2 *>(dst)[g] = v;
    }
    if (tid == 0 && (n & 1)) dst[n - 1] = begin + n - 1;
  } else {
    for (fq_u64 i = tid; i < n; i += nthreads) dst[i] = begin + i;
  }
}

// ---- on-disk cache of JIT-built cubins ----
// NVRTC + ptxas cost about a second per kernel; the cubin of a specialisation is a pure function of the program text, so
// it is kept under $FQ_JIT_CACHE_DIR (default: .jit_cache next to libfuse_gpu.so) as <hash of the text>.cubin,
// written to a temporary name and renamed (ranks and threads may race for the same entry).  FQ_JIT_CACHE=0 disables it.
static uint64_t fnv1a64(const std::string &s) {
  uint64_t h = 1469598103934665603ull;
  for (unsigned char c : s) { h ^= c; h *= 1099511628211ull; }
  return h;
}
static std::string jit_cache_dir() {
  const char *off = getenv("FQ_JIT_CACHE");
  if (off && atoi(off) == 0) return "";
  std::string dir;
  if (const char *d = getenv("FQ_JIT_CACHE_DIR")) {
    dir = d;
  } else {   // next to the library itself: <dir of libfuse_gpu.so>/.jit_cache
    Dl_info info;
    if (dladdr((const void *)&jit_cache_dir, &info) && info.dli_fname) {
      dir = info.dli_fname;
      const size_t slash = dir.rfind('/');
      dir = (slash == std::string::npos ? std::string(".") : dir.substr(0, slash)) + "/.jit_cache";
    }
  }
  if (dir.empty()) return "";
  std::string cur;
  for (size_t i = 0; i <= dir.size(); i++) {   // mkdir -p
    if (i == dir.size() || dir[i] == '/') {
      if (!cur.empty() && mkdir(cur.c_str(), 0755) != 0 && errno != EEXIST) return "";
    }
    if (i < dir.size()) cur += dir[i];
  }
  return dir;
}
static bool jit_cache_read(const std::string &path, std::vector<char> *out) {
  FILE *f = fopen(path.c_str(), "rb");
  if (!f) return false;
  fseek(f, 0, SEEK_END);
  long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  bool ok = n > 0;
  if (ok) {
    out->resize((size_t)n);
    ok = fread(out->data(), 1, (size_t)n, f) == (size_t)n;
  }
  fclose(f);
  return ok;
}
static void jit_cache_write(const std::string &path, const std::vector<char> &data) {
  const std::string tmp = path + ".tmp" + std::to_string((long)getpid()) + "_" + std::to_string((unsigned long)(uintptr_t)&data);
  FILE *f = fopen(tmp.c_str(), "wb");
  if (!f) return;
  const bool ok = fwrite(data.data(), 1, data.size(), f) == data.size();
  fclose(f);
  if (!ok || rename(tmp.c_str(), path.c_str()) != 0) remove(tmp.c_str());
}

static const char *const kNvrtcOpts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo"};

// builds the kernels whose suffixes m->built lists
fq_status compile_jit(fq_ctx *ctx, const fq::Generated &gen, Module *m) {
  if (!g_nvrtc.load()) return set_err(FQ_ERR_CUDA, "NVRTC unavailable: %s", g_nvrtc.why.c_str());
  if (!g_drv.load()) return set_err(FQ_ERR_CUDA, "CUDA driver unavailable: %s", g_drv.why.c_str());
  std::string src = shapes().defines() + std::string(fq_skeleton_src) + "\n" + gen.struct_source;
  for (auto &k : gen.kernels)
    if (std::find(m->built.begin(), m->built.end(), k.first) != m->built.end()) src += k.second;
  const std::string cache_dir = jit_cache_dir();
  // key = program text + everything else the cubin depends on: NVRTC's version and the compile options
  int nv_major = 0, nv_minor = 0;
  if (g_nvrtc.nvrtcVersion) g_nvrtc.nvrtcVersion(&nv_major, &nv_minor);
  std::string key_text = src + "\n//nvrtc " + std::to_string(nv_major) + "." + std::to_string(nv_minor);
  for (const char *o : kNvrtcOpts) key_text += std::string(" ") + o;
  char key[40];
  snprintf(key, sizeof key, "%016" PRIx64 "%08x", fnv1a64(key_text), (unsigned)key_text.size());
  const std::string cache_path = cache_dir.empty() ? "" : cache_dir + "/" + key + ".sm_100a.cubin";
  std::vector<char> cached;
  if (!cache_path.empty() && jit_cache_read(cache_path, &cached)) {
    cudaFree(nullptr);
    if (g_drv.cuModuleLoadData(&m->mod, cached.data()) == 0) { m->from_disk_cache = true; return FQ_OK; }
    remove(cache_path.c_str());   // unreadable entry (another driver / truncated): rebuild it
  }
  nvrtcProgram_ prog = nullptr;
  int r = g_nvrtc.nvrtcCreateProgram(&prog, src.c_str(), ("fq_" + gen.tag + ".cu").c_str(), 0, nullptr, nullptr);
  if (r) return set_err(FQ_ERR_CUDA, "nvrtcCreateProgram: %s", g_nvrtc.nvrtcGetErrorString(r));
  r = g_nvrtc.nvrtcCompileProgram(prog, (int)(sizeof kNvrtcOpts / sizeof kNvrtcOpts[0]), kNvrtcOpts);
  if (r) {
    size_t n = 0;
    g_nvrtc.nvrtcGetProgramLogSize(prog, &n);
    std::string log(n, 0);
    if (n) g_nvrtc.nvrtcGetProgramLog(prog, &log[0]);
    g_nvrtc.nvrtcDestroyProgram(&prog);
    return set_err(FQ_ERR_CUDA, "NVRTC compile failed: %s\n%.1500s", g_nvrtc.nvrtcGetErrorString(r), log.c_str());
  }
  size_t n = 0;
  g_nvrtc.nvrtcGetCUBINSize(prog, &n);
  std::vector<char> cubin(n);
  g_nvrtc.nvrtcGetCUBIN(prog, cubin.data());
  g_nvrtc.nvrtcDestroyProgram(&prog);
  if (!cache_path.empty()) jit_cache_write(cache_path, cubin);
  cudaFree(nullptr);  // make sure the primary context exists and is current
  CUresult_ cr = g_drv.cuModuleLoadData(&m->mod, cubin.data());
  if (cr) return set_err(FQ_ERR_CUDA, "cuModuleLoadData: %s", g_drv.err(cr).c_str());
  (void)ctx;
  return FQ_OK;
}

// Finds a planned kernel in the pipe's module.  A JIT module holds only the kernels it was built with: a missing one stays
// invalid (the launch falls back).
fq_status resolve_kernel(Module *m, const std::string &tag, Kernel *k) {
  const std::string name = "fqk_" + tag + k->suffix;
  auto it = m->kernels.find(name);
  if (it != m->kernels.end()) { *k = it->second; return FQ_OK; }
  if (!m->precompiled && std::find(m->built.begin(), m->built.end(), k->suffix) == m->built.end()) return FQ_OK;
  const unsigned smem = k->smem;
  if (m->precompiled) {
    for (int i = 0; i < fq_aot_count; i++)
      if (name == fq_aot_table[i].name) k->aot = fq_aot_table[i].fn;
    if (!k->aot) return set_err(FQ_ERR_INTERNAL, "Internal Error: precompiled kernel %s missing", name.c_str());
    if (smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(k->aot, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&k->blocks_per_sm, k->aot, k->threads, smem));
  } else {
    CUresult_ cr = g_drv.cuModuleGetFunction(&k->jit, m->mod, name.c_str());
    if (cr) return set_err(FQ_ERR_CUDA, "cuModuleGetFunction(%s): %s", name.c_str(), g_drv.err(cr).c_str());
    if (smem > 48 * 1024) {
      if (!g_drv.cuFuncSetAttribute) return set_err(FQ_ERR_CUDA, "cuFuncSetAttribute unavailable");
      cr = g_drv.cuFuncSetAttribute(k->jit, 8 /* CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES */, (int)smem);
      if (cr) return set_err(FQ_ERR_CUDA, "cuFuncSetAttribute(%s): %s", name.c_str(), g_drv.err(cr).c_str());
    }
    cr = g_drv.cuOccupancyMaxActiveBlocksPerMultiprocessor(&k->blocks_per_sm, k->jit, k->threads, smem);
    if (cr) return set_err(FQ_ERR_CUDA, "cuOccupancy: %s", g_drv.err(cr).c_str());
  }
  if (k->blocks_per_sm < 1 || k->one_per_sm) k->blocks_per_sm = 1;
  m->kernels[name] = *k;
  return FQ_OK;
}

fq_status launch(fq_ctx *ctx, const Kernel &k, unsigned grid, const fq_launch_params &p, void *stream) {
  void *args[] = {(void *)&p};
  if (k.aot) {
    CUDA_TRY(cudaLaunchKernel(k.aot, dim3(grid), dim3(k.threads), args, k.smem, (cudaStream_t)stream));
  } else {
    CUresult_ cr = g_drv.cuLaunchKernel(k.jit, grid, 1, 1, (unsigned)k.threads, 1, 1, k.smem, stream, args, nullptr);
    if (cr) return set_err(FQ_ERR_CUDA, "cuLaunchKernel: %s", g_drv.err(cr).c_str());
  }
  ctx->launches++;
  return FQ_OK;
}

// Aggregate, select and map launches: the staged kernel when the variant allows it and the source's validity bitmaps can be
// bulk-copied, else the LDG kernel; a module that holds only one of the two (a JIT build) launches that one.
fq_status pick_kernel(const fq_pipe *pipe, Slot staged, Slot ldg, const fq_launch_params &p, const char *what, const Kernel **out) {
  const Kernel &ks = pipe->k[staged], &kl = pipe->k[ldg];
  if (p.bits_unstaged && !kl.valid())
    return set_err(FQ_ERR_INTERNAL, "Internal Error: validity bitmap off the 128-row grid needs the LDG kernel, which this pipe was not built with");
  *out = !p.bits_unstaged && ((pipe->variant != V_LDG && ks.valid()) || !kl.valid()) ? &ks : &kl;
  if (!(*out)->valid()) return set_err(FQ_ERR_INTERNAL, "Internal Error: no %s kernel was built for this pipe", what);
  return FQ_OK;
}

// persistent grid: every resident CTA slot of every SM, fewer when the source has fewer units of k.rows rows
unsigned persistent_grid(const fq_ctx *ctx, const Kernel &k, uint64_t n_rows) {
  return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)ctx->sm_count * k.blocks_per_sm, (n_rows + k.rows - 1) / k.rows));
}

// "the results of this launch are ready" for the fetch calls: an event on the stream, or — while a graph is being recorded
// — a note to record it after every replay (an event recorded into a capturing stream cannot be waited for)
fq_status mark_done(fq_ctx *ctx, cudaEvent_t ev, cudaStream_t s) {
  if (ctx->recording && s == ctx->recording_stream) {
    std::vector<cudaEvent_t> &d = ctx->recording->done;
    if (std::find(d.begin(), d.end(), ev) == d.end()) d.push_back(ev);
    return FQ_OK;
  }
  CUDA_TRY(cudaEventRecord(ev, s));
  return FQ_OK;
}

fq_status bind_source(const fq_pipe *pipe, const fq_source *src, fq_launch_params *p) {
  if (!src) return set_err(FQ_ERR_INVALID, "Internal Error: null source");
  if ((src->generated != 0) != pipe->gen.generated_source)
    return set_err(FQ_ERR_INVALID, "Internal Error: pipe was compiled for a %s source", pipe->gen.generated_source ? "generated" : "materialised");
  p->n_rows = src->n_rows;
  p->numbers_begin = src->numbers_begin;
  for (int k = 0; k < FQ_MAX_LOOKUPS; k++) {
    if (!(pipe->gen.lookup_slots & (1u << k))) continue;
    if (!(pipe->lookup_bound & (1u << k))) return set_err(FQ_ERR_INVALID, "Internal Error: lookup slot %d of the pipe is not bound (fq_pipe_set_lookup)", k);
    p->lookup[k] = pipe->lookup[k];
    p->lookup_bits[k] = pipe->lookup_bits[k];
  }
  for (int c : pipe->gen.used_cols) {
    if (pipe->gen.generated_source && c == 0) continue;
    if (c >= src->n_cols || !src->cols || !src->cols[c]) return set_err(FQ_ERR_INVALID, "Internal Error: source lacks column %d", c);
    const fq_column *col = src->cols[c];
    if (col->len < src->n_rows) return set_err(FQ_ERR_INVALID, "Internal Error: column %d has %" PRIu64 " rows, source says %" PRIu64, c, col->len, src->n_rows);
    if (((uintptr_t)col->ptr & 15) != 0) p->unaligned = 1;   // a slice off the 16-byte grid: the kernels read it row by row
    p->cols[c] = col->ptr;
    const auto nit = std::find(pipe->gen.null_cols.begin(), pipe->gen.null_cols.end(), c);
    const bool want_valid = nit != pipe->gen.null_cols.end();
    const int want_kind = want_valid ? pipe->gen.null_kind[(size_t)(nit - pipe->gen.null_cols.begin())] : 0;
    if (want_kind == 2) {
      if (!col->validity_bits) return set_err(FQ_ERR_INVALID, "Internal Error: pipe was compiled for a bitmap-validity column %d but the column carries no validity bitmap", c);
      if (col->validity_bits->len * 8 < col->validity_bit0 + src->n_rows) return set_err(FQ_ERR_INVALID, "Internal Error: validity bitmap of column %d is shorter than the source", c);
      if (col->validity_bit0 % (uint64_t)pipe->gen.vec != 0) p->unaligned = 1;   // a thread's V bits would straddle its byte: row-by-row path
      if (col->validity_bit0 % 128 != 0) p->bits_unstaged = 1;   // a tile's bitmap bytes would not start on a 16-byte boundary: no bulk copies
      p->cols_valid[c] = col->validity_bits->ptr;
      p->cols_valid_bit0[c] = col->validity_bit0;
    } else if (want_valid) {
      if (!col->validity) return set_err(FQ_ERR_INVALID, "Internal Error: pipe was compiled for a nullable column %d but the column carries no validity", c);
      if (col->validity->len < src->n_rows) return set_err(FQ_ERR_INVALID, "Internal Error: validity of column %d is shorter than the source", c);
      if (((uintptr_t)col->validity->ptr & 15) != 0) p->unaligned = 1;
      p->cols_valid[c] = col->validity->ptr;
    } else if (col->validity || col->validity_bits) {
      return set_err(FQ_ERR_INVALID, "Internal Error: column %d carries validity but the pipe was compiled for a NOT NULL column", c);
    }
  }
  return FQ_OK;
}

// every group operation takes the next epoch; all ranks issue the same sequence of operations (like a communicator)
void bind_group(fq_group *g, fq_launch_params *p) {
  for (int r = 0; r < g->world; r++) p->group_windows[r] = (fq_u64 *)g->windows[r];
  p->group_epoch = ++g->epoch;
  p->group_timeout_ns = g->timeout_ns;
  p->group_rank = (fq_u32)g->rank;
  p->group_world = (fq_u32)g->world;
  p->group_row_slots = g->row_slots;
}

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

uint32_t fq_abi_version(void) { return FQ_ABI_VERSION; }

const char *fq_last_error(const fq_ctx *) { return g_err.c_str(); }

fq_status fq_ctx_create(int32_t device, fq_ctx **out) {
  if (!out) return set_err(FQ_ERR_INVALID, "Internal Error: null out pointer");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return set_err(FQ_ERR_CUDA, "CUDA error: no usable CUDA device (%s); libfuse_gpu has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= n) return set_err(FQ_ERR_INVALID, "Internal Error: device %d out of range (%d devices)", device, n);
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaFree(nullptr));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return set_err(FQ_ERR_CUDA, "CUDA error: device %d is sm_%d%d; libfuse_gpu is built for sm_100a (B200) only", device, prop.major, prop.minor);
  fq_ctx *c = new fq_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  *out = c;
  return FQ_OK;
}

void fq_ctx_destroy(fq_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  for (auto &kv : ctx->modules)
    if (kv.second.mod && g_drv.cuModuleUnload) g_drv.cuModuleUnload(kv.second.mod);
  cudaFree(ctx->sort_scratch);
  if (ctx->sort_done) cudaEventDestroy(ctx->sort_done);
  delete ctx;
}

fq_status fq_ctx_trim(fq_ctx *ctx) {
  if (fq_status st = use(ctx)) return st;
  std::lock_guard<std::mutex> lock(ctx->sort_mu);
  CUDA_TRY(cudaDeviceSynchronize());
  cudaFree(ctx->sort_scratch);
  ctx->sort_scratch = nullptr;
  ctx->sort_scratch_bytes = 0;
  cudaMemPool_t pool = nullptr;
  if (cudaDeviceGetDefaultMemPool(&pool, ctx->device) == cudaSuccess && pool) cudaMemPoolTrimTo(pool, 0);
  cudaGetLastError();
  return FQ_OK;
}

uint64_t fq_ctx_launch_count(const fq_ctx *ctx) { return ctx ? ctx->launches.load() : 0; }
int32_t fq_ctx_sm_count(const fq_ctx *ctx) { return ctx ? ctx->sm_count : 0; }

// ---- columns ----
fq_status fq_column_alloc(fq_ctx *ctx, fq_dtype dtype, uint64_t len, fq_column **out) {
  if (fq_status st = use(ctx)) return st;
  size_t w = fq::dtype_size(dtype);
  if (!w) return set_err(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: column of type %s", fq::dtype_name(dtype));
  fq_column *c = new fq_column();
  c->dtype = dtype;
  c->len = len;
  c->owned = true;
  size_t bytes = (size_t)len * w;
  bytes = (bytes + 255) & ~(size_t)255;  // whole vector groups stay in bounds
  cudaError_t e = cudaMalloc(&c->ptr, bytes ? bytes : 256);
  if (e != cudaSuccess) {
    delete c;
    return set_err(FQ_ERR_CUDA, "CUDA error: %s (cudaMalloc of %zu bytes)", cudaGetErrorString(e), bytes);
  }
  *out = c;
  return FQ_OK;
}
fq_status fq_column_wrap(fq_ctx *ctx, fq_dtype dtype, uint64_t len, void *device_values, fq_column **out) {
  if (!ctx || !out) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (!fq::dtype_size(dtype)) return set_err(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: column of type %s", fq::dtype_name(dtype));
  if (((uintptr_t)device_values & 15) != 0) return set_err(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: wrapped buffer is not 16-byte aligned");
  fq_column *c = new fq_column();
  c->dtype = dtype;
  c->len = len;
  c->ptr = device_values;
  *out = c;
  return FQ_OK;
}
fq_status fq_column_slice(fq_ctx *ctx, const fq_column *parent, uint64_t offset, uint64_t len, fq_column **out) {
  if (!ctx || !parent || !out) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (offset + len > parent->len) return set_err(FQ_ERR_INVALID, "Internal Error: slice [%" PRIu64 ", +%" PRIu64 ") exceeds %" PRIu64 " rows", offset, len, parent->len);
  fq_column *c = new fq_column();
  c->dtype = parent->dtype;
  c->len = len;
  c->ptr = (char *)parent->ptr + offset * fq::dtype_size(parent->dtype);
  if (parent->validity) {
    fq_column *v = nullptr;
    if (fq_status st = fq_column_slice(ctx, parent->validity, offset, len, &v)) { delete c; return st; }
    c->validity = v;
    c->owns_validity = true;
  }
  c->validity_bits = parent->validity_bits;
  c->validity_bit0 = parent->validity_bit0 + offset;
  *out = c;
  return FQ_OK;
}
fq_status fq_column_set_validity(fq_ctx *ctx, fq_column *col, const fq_column *validity) {
  if (!ctx || !col) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (validity && (validity->dtype != FQ_BOOL || validity->len < col->len))
    return set_err(FQ_ERR_INVALID, "Internal Error: validity must be a Boolean column at least as long as the values");
  if (col->owns_validity && col->validity) fq_column_free(ctx, const_cast<fq_column *>(col->validity));
  col->validity = validity;
  col->owns_validity = false;
  col->validity_bits = nullptr;
  col->validity_bit0 = 0;
  return FQ_OK;
}
fq_status fq_column_set_validity_bitmap(fq_ctx *ctx, fq_column *col, const fq_column *bitmap, uint64_t bit_offset) {
  if (!ctx || !col) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (bitmap && (bitmap->dtype != FQ_U8 || bitmap->len * 8 < bit_offset + col->len))
    return set_err(FQ_ERR_INVALID, "Internal Error: the validity bitmap must be a UInt8 column of at least ceil((offset + rows) / 8) bytes");
  if (col->owns_validity && col->validity) fq_column_free(ctx, const_cast<fq_column *>(col->validity));
  col->validity = nullptr;
  col->owns_validity = false;
  col->validity_bits = bitmap;
  col->validity_bit0 = bitmap ? bit_offset : 0;
  return FQ_OK;
}
const fq_column *fq_column_validity(const fq_column *col) { return col ? col->validity : nullptr; }

void fq_column_free(fq_ctx *ctx, fq_column *col) {
  if (!col) return;
  if (col->owns_validity && col->validity) fq_column_free(ctx, const_cast<fq_column *>(col->validity));
  if (col->owned && col->ptr) {
    if (ctx) cudaSetDevice(ctx->device);
    cudaFree(col->ptr);
  }
  delete col;
}
fq_dtype fq_column_dtype(const fq_column *col) { return col ? col->dtype : FQ_NULL; }
uint64_t fq_column_len(const fq_column *col) { return col ? col->len : 0; }
void *fq_column_device_ptr(const fq_column *col) { return col ? col->ptr : nullptr; }

fq_status fq_column_upload(fq_ctx *ctx, fq_column *col, uint64_t row_offset, const void *host, uint64_t n_rows, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!col || row_offset + n_rows > col->len) return set_err(FQ_ERR_INVALID, "Internal Error: upload out of range");
  size_t w = fq::dtype_size(col->dtype);
  CUDA_TRY(cudaMemcpyAsync((char *)col->ptr + row_offset * w, host, n_rows * w, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return FQ_OK;
}
fq_status fq_column_download(fq_ctx *ctx, const fq_column *col, uint64_t row_offset, void *host, uint64_t n_rows, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!col || row_offset + n_rows > col->len) return set_err(FQ_ERR_INVALID, "Internal Error: download out of range");
  size_t w = fq::dtype_size(col->dtype);
  CUDA_TRY(cudaMemcpyAsync(host, (const char *)col->ptr + row_offset * w, n_rows * w, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return FQ_OK;
}
// ---- Arrow LSB-first bitmaps <-> one byte per row ----
__global__ void __launch_bounds__(256) fq_bits_expand(fq_u8 *dst, const fq_u8 *bits, unsigned shift, fq_u64 n_rows) {
  // thread i -> rows [8i, 8i + 8): source bits [shift + 8i, shift + 8i + 8) straddle bytes i and i + 1 (the staging buffer has one spare byte)
  const fq_u64 groups = (n_rows + 7) / 8;
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i < groups; i += (fq_u64)gridDim.x * blockDim.x) {
    const unsigned w = ((unsigned)bits[i] | ((unsigned)bits[i + 1] << 8)) >> shift;
    fq_u64 out = 0;
#pragma unroll
    for (int b = 0; b < 8; b++) out |= (fq_u64)((w >> b) & 1u) << (8 * b);
    if (8 * i + 8 <= n_rows && (((uintptr_t)dst) & 7) == 0) {
      *(fq_u64 *)(dst + 8 * i) = out;
    } else {
      for (int b = 0; b < 8 && 8 * i + b < n_rows; b++) dst[8 * i + b] = (fq_u8)(out >> (8 * b));
    }
  }
}
__global__ void __launch_bounds__(256) fq_bits_pack(fq_u8 *bits, const fq_u8 *src, fq_u64 n_rows) {
  const fq_u64 groups = (n_rows + 7) / 8;
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i < groups; i += (fq_u64)gridDim.x * blockDim.x) {
    unsigned w = 0;
    for (int b = 0; b < 8 && 8 * i + b < n_rows; b++) w |= (src[8 * i + b] ? 1u : 0u) << b;
    bits[i] = (fq_u8)w;
  }
}
fq_status fq_column_upload_bits(fq_ctx *ctx, fq_column *col, uint64_t row_offset, const void *host_bits, uint64_t bit_offset,
                                uint64_t n_rows, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!col || col->dtype != FQ_BOOL) return set_err(FQ_ERR_INVALID, "Internal Error: bitmap upload needs a Boolean column");
  if (row_offset + n_rows > col->len) return set_err(FQ_ERR_INVALID, "Internal Error: upload out of range");
  if (n_rows == 0) return FQ_OK;
  if (!host_bits) return set_err(FQ_ERR_INVALID, "Internal Error: null bitmap");
  cudaStream_t s = (cudaStream_t)stream;
  const uint64_t first = bit_offset / 8, nbytes = (bit_offset % 8 + n_rows + 7) / 8;
  fq_u8 *stage = nullptr;
  CUDA_TRY(cudaMallocAsync((void **)&stage, nbytes + 1, s));
  CUDA_TRY(cudaMemsetAsync(stage + nbytes, 0, 1, s));
  CUDA_TRY(cudaMemcpyAsync(stage, (const char *)host_bits + first, nbytes, cudaMemcpyHostToDevice, s));
  const uint64_t groups = (n_rows + 7) / 8;
  const unsigned grid = (unsigned)std::min<uint64_t>((groups + 255) / 256, (uint64_t)ctx->sm_count * 8);
  fq_bits_expand<<<grid, 256, 0, s>>>((fq_u8 *)col->ptr + row_offset, stage, (unsigned)(bit_offset % 8), n_rows);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  CUDA_TRY(cudaFreeAsync(stage, s));
  return FQ_OK;
}
fq_status fq_column_download_bits(fq_ctx *ctx, const fq_column *col, uint64_t row_offset, void *host_bits, uint64_t n_rows,
                                  void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!col || col->dtype != FQ_BOOL) return set_err(FQ_ERR_INVALID, "Internal Error: bitmap download needs a Boolean column");
  if (row_offset + n_rows > col->len) return set_err(FQ_ERR_INVALID, "Internal Error: download out of range");
  if (n_rows == 0) return FQ_OK;
  if (!host_bits) return set_err(FQ_ERR_INVALID, "Internal Error: null bitmap");
  cudaStream_t s = (cudaStream_t)stream;
  const uint64_t nbytes = (n_rows + 7) / 8;
  fq_u8 *stage = nullptr;
  CUDA_TRY(cudaMallocAsync((void **)&stage, nbytes, s));
  const unsigned grid = (unsigned)std::min<uint64_t>((nbytes + 255) / 256, (uint64_t)ctx->sm_count * 8);
  fq_bits_pack<<<grid, 256, 0, s>>>(stage, (const fq_u8 *)col->ptr + row_offset, n_rows);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  CUDA_TRY(cudaMemcpyAsync(host_bits, stage, nbytes, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaFreeAsync(stage, s));
  return FQ_OK;
}
fq_status fq_column_copy(fq_ctx *ctx, fq_column *dst, uint64_t dst_offset, const fq_column *src, uint64_t src_offset, uint64_t n_rows,
                         void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!dst || !src) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (dst->dtype != src->dtype) return set_err(FQ_ERR_INVALID, "Internal Error: copy between columns of different types");
  if (dst_offset + n_rows > dst->len || src_offset + n_rows > src->len) return set_err(FQ_ERR_INVALID, "Internal Error: copy exceeds a column");
  const size_t w = fq::dtype_size(src->dtype);
  if (n_rows) CUDA_TRY(cudaMemcpyAsync((char *)dst->ptr + dst_offset * w, (const char *)src->ptr + src_offset * w, n_rows * w, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return FQ_OK;
}
fq_status fq_stream_synchronize(fq_ctx *ctx, void *stream) {
  if (fq_status st = use(ctx)) return st;
  CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return FQ_OK;
}
fq_status fq_stream_create(fq_ctx *ctx, void **stream) {
  if (fq_status st = use(ctx)) return st;
  if (!stream) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  cudaStream_t s = nullptr;
  CUDA_TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  *stream = (void *)s;
  return FQ_OK;
}
void fq_stream_destroy(fq_ctx *ctx, void *stream) {
  if (!stream) return;
  if (ctx) cudaSetDevice(ctx->device);
  cudaStreamDestroy((cudaStream_t)stream);
}
fq_status fq_host_alloc(fq_ctx *ctx, uint64_t bytes, void **out) {
  if (fq_status st = use(ctx)) return st;
  CUDA_TRY(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
  return FQ_OK;
}
void fq_host_free(fq_ctx *ctx, void *p) {
  if (ctx) cudaSetDevice(ctx->device);
  if (p) cudaFreeHost(p);
}

fq_status fq_numbers_fill(fq_ctx *ctx, fq_column *col, uint64_t row_offset, uint64_t begin, uint64_t n_rows, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!col || col->dtype != FQ_U64) return set_err(FQ_ERR_INVALID, "Internal Error: numbers column must be UInt64");
  if (row_offset + n_rows > col->len) return set_err(FQ_ERR_INVALID, "Internal Error: fill out of range");
  if (n_rows == 0) return FQ_OK;
  uint64_t want = (n_rows / 2 + 255) / 256;
  unsigned grid = (unsigned)std::min<uint64_t>(std::max<uint64_t>(want, 1), (uint64_t)ctx->sm_count * 8);
  fq_fill_numbers<<<grid, 256, 0, (cudaStream_t)stream>>>((fq_u64 *)col->ptr + row_offset, begin, n_rows);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  return FQ_OK;
}

// ---- pipes ----
fq_status fq_pipe_compile(fq_ctx *ctx, const fq_pipe_desc *desc, fq_pipe **out) {
  if (fq_status st = use(ctx)) return st;
  if (!desc || !out) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  *out = nullptr;
  fq_pipe *pipe = new fq_pipe();
  std::string err;
  int st = fq::generate(*desc, &pipe->gen, &err);
  if (st) {
    delete pipe;
    return set_err(st, "%s", err.c_str());
  }
  const fq::Generated &gen = pipe->gen;
  plan_kernels(gen, pipe->k, &pipe->gb_smem_cap);
  // the environment is read here, once per pipe — never on the launch path
  const char *env = variant_env(gen);
  if (const char *word = env ? getenv(env) : nullptr) {
    if (fq_status s2 = parse_variant(gen, word, &pipe->variant)) { delete pipe; return s2; }
  }
  {
    std::lock_guard<std::mutex> lk(ctx->mu);
    auto it = ctx->modules.find(gen.tag);
    if (it == ctx->modules.end()) {
      Module mod;
      const std::string probe = "fqk_" + gen.tag + "_";
      for (int i = 0; i < fq_aot_count; i++)
        if (strncmp(fq_aot_table[i].name, probe.c_str(), probe.size()) == 0) mod.precompiled = true;
      if (getenv("FQ_FORCE_JIT") || shapes().tuned) mod.precompiled = false;
      if (!mod.precompiled) {
        // NVRTC + ptxas cost about a second per kernel: build only the path this pipe will launch (the staged one when the
        // variant allows it and its ring fits, else the LDG one; both handle ragged and unaligned sources).  A validity bitmap
        // that starts off the 128-row grid (a slice) cannot be bulk-copied: such pipes also get the LDG kernel.
        // FQ_JIT_ALL_VARIANTS=1 builds every planned kernel.
        const bool all = getenv("FQ_JIT_ALL_VARIANTS") && atoi(getenv("FQ_JIT_ALL_VARIANTS")) != 0;
        bool staged = false;
        for (const Kernel &k : pipe->k) staged |= k.staged && pipe->variant != V_LDG;
        for (const Kernel &k : pipe->k)
          if (k.suffix && (all || k.staged == staged || (!k.staged && gen.row_bitmaps > 0))) mod.built.push_back(k.suffix);
        std::lock_guard<std::mutex> lk2(g_mu);
        if (fq_status s2 = compile_jit(ctx, gen, &mod)) { delete pipe; return s2; }
      }
      it = ctx->modules.emplace(gen.tag, mod).first;
    }
    Module *m = &it->second;
    pipe->precompiled = m->precompiled;
    pipe->build_kind = m->precompiled ? 0 : m->from_disk_cache ? 2 : 1;
    for (Kernel &k : pipe->k) {
      if (!k.suffix) continue;
      if (fq_status s2 = resolve_kernel(m, gen.tag, &k)) { delete pipe; return s2; }
    }
  }
  pipe->n_slots = FQ_STATE_HDR + gen.n_slots;
  cudaError_t e = cudaMalloc(&pipe->d_state, sizeof(uint64_t) * pipe->n_slots);
  if (e == cudaSuccess && gen.kind == FQ_PIPE_AGGREGATE) {
    // one partial row per CTA of the largest persistent grid any variant can launch: no allocation on the launch path
    int bps = 1;
    for (const Kernel *k : {&pipe->k[K_AGG_U4], &pipe->k[K_AGG_TMA]})
      if (k->valid()) bps = std::max(bps, k->blocks_per_sm);
    pipe->partials_cap = ctx->sm_count * bps;
    e = cudaMalloc(&pipe->d_partials, sizeof(uint64_t) * pipe->n_slots * pipe->partials_cap);
  }
  if (e == cudaSuccess) e = cudaMemset(pipe->d_state, 0, sizeof(uint64_t) * pipe->n_slots);
  if (e == cudaSuccess) e = cudaMalloc(&pipe->d_ctl, 64);
  if (e == cudaSuccess) e = cudaMemset(pipe->d_ctl, 0, 64);
  if (e == cudaSuccess) e = cudaHostAlloc(&pipe->h_state, sizeof(uint64_t) * pipe->n_slots, cudaHostAllocDefault);
  if (e == cudaSuccess) e = cudaHostAlloc(&pipe->h_result, 64, cudaHostAllocDefault);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&pipe->ev, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    fq_pipe_destroy(ctx, pipe);
    return set_err(FQ_ERR_CUDA, "CUDA error: %s (pipe buffers)", cudaGetErrorString(e));
  }
  memset(pipe->h_state, 0, sizeof(uint64_t) * pipe->n_slots);
  memset(pipe->h_result, 0, 64);
  *out = pipe;
  return FQ_OK;
}

void fq_pipe_destroy(fq_ctx *ctx, fq_pipe *pipe) {
  if (!pipe) return;
  if (ctx) cudaSetDevice(ctx->device);
  cudaFree(pipe->d_state);
  cudaFree(pipe->d_partials);
  cudaFree(pipe->d_ctl);
  cudaFree(pipe->d_tiles);
  cudaFree(pipe->d_blocks);
  cudaFree(pipe->d_merged);
  cudaFree(pipe->gb_keys);
  cudaFree(pipe->gb_slots);
  cudaFree(pipe->gb_rep_keys);
  cudaFree(pipe->gb_rep_slots);
  cudaFree(pipe->gb_flags);
  cudaFree(pipe->gb_identity);
  if (pipe->h_gb) cudaFreeHost(pipe->h_gb);
  if (pipe->h_merged) cudaFreeHost(pipe->h_merged);
  if (pipe->h_state) cudaFreeHost(pipe->h_state);
  if (pipe->h_result) cudaFreeHost(pipe->h_result);
  if (pipe->ev) cudaEventDestroy(pipe->ev);
  delete pipe;
}

fq_status fq_pipe_set_variant(fq_ctx *, fq_pipe *pipe, const char *variant) {
  if (!pipe || !variant) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  return parse_variant(pipe->gen, variant, &pipe->variant);
}
fq_status fq_pipe_set_lookup(fq_ctx *, fq_pipe *pipe, int32_t slot, const fq_column *bits, uint64_t n_bits) {
  if (!pipe || !bits) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (slot < 0 || slot >= FQ_MAX_LOOKUPS) return set_err(FQ_ERR_INVALID, "Internal Error: lookup slot %d out of range [0, %d)", slot, FQ_MAX_LOOKUPS);
  if (bits->dtype != FQ_U8 || bits->len < (n_bits + 7) / 8)
    return set_err(FQ_ERR_INVALID, "Internal Error: a lookup table of %" PRIu64 " bits is a UInt8 column of at least %" PRIu64 " bytes", n_bits, (n_bits + 7) / 8);
  pipe->lookup[slot] = (const fq_u8 *)bits->ptr;
  pipe->lookup_bits[slot] = n_bits;
  pipe->lookup_bound |= 1u << slot;
  return FQ_OK;
}
int32_t fq_pipe_is_precompiled(const fq_pipe *pipe) { return pipe && pipe->precompiled; }
int32_t fq_pipe_build_kind(const fq_pipe *pipe) { return pipe ? pipe->build_kind : 0; }
const char *fq_pipe_source(const fq_pipe *pipe) { return pipe ? pipe->gen.source.c_str() : ""; }

fq_status fq_pipe_expr_dtype(fq_ctx *, const fq_pipe *pipe, int32_t i, fq_dtype *out) {
  if (!pipe || !out || i < 0 || i >= (int)pipe->gen.expr_dtypes.size()) return set_err(FQ_ERR_INVALID, "Internal Error: bad expression index");
  *out = pipe->gen.expr_dtypes[i];
  return FQ_OK;
}

fq_status fq_pipe_expr_nullable(fq_ctx *, const fq_pipe *pipe, int32_t i, int32_t *out) {
  if (!pipe || !out || i < 0 || i >= (int)pipe->gen.expr_dtypes.size()) return set_err(FQ_ERR_INVALID, "Internal Error: bad expression index");
  *out = i < (int)pipe->gen.expr_nullable.size() ? pipe->gen.expr_nullable[i] : 0;
  return FQ_OK;
}

fq_status fq_pipe_aggregator_nodes(fq_ctx *, const fq_pipe *pipe, int32_t *nodes, int32_t cap, int32_t *n) {
  if (!pipe || !n) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  *n = (int32_t)pipe->gen.agg_nodes.size();
  for (int i = 0; i < *n && i < cap && nodes; i++) nodes[i] = pipe->gen.agg_nodes[i];
  return FQ_OK;
}

fq_status fq_pipe_state_device(fq_ctx *, const fq_pipe *pipe, void **dev_ptr, uint64_t *n_bytes) {
  if (!pipe || !dev_ptr || !n_bytes) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  *dev_ptr = pipe->d_state;
  *n_bytes = sizeof(uint64_t) * pipe->n_slots;
  return FQ_OK;
}

fq_status fq_pipe_launch_aggregate(fq_ctx *ctx, fq_pipe *pipe, const fq_source *src, uint32_t flags, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!pipe || pipe->gen.kind != FQ_PIPE_AGGREGATE) return set_err(FQ_ERR_INVALID, "Internal Error: not an aggregate pipe");
  fq_launch_params p;
  memset(&p, 0, sizeof p);
  if (fq_status st = bind_source(pipe, src, &p)) return st;
  const Kernel *k;
  if (fq_status st = pick_kernel(pipe, K_AGG_TMA, K_AGG_U4, p, "aggregate", &k)) return st;
  const unsigned grid = persistent_grid(ctx, *k, src->n_rows);
  if ((int)grid > pipe->partials_cap) return set_err(FQ_ERR_INTERNAL, "Internal Error: grid of %u CTAs exceeds the pipe's %d partial rows", grid, pipe->partials_cap);
  p.partials = (fq_u64 *)pipe->d_partials;
  p.state = (fq_u64 *)pipe->d_state;
  p.ticket = (fq_u32 *)(pipe->d_ctl + 4);
  p.accumulate = (flags & FQ_RUN_ACCUMULATE) ? 1u : 0u;
  p.stages = pipe->k[K_AGG_TMA].stages;   // the staged kernel's ring (the LDG kernel does not read it)
  if (fq_group *g = pipe->group) {
    if (ctx->recording) return set_err(FQ_ERR_INVALID, "Internal Error: a pipe with a group attached cannot be recorded into a graph (the merge epoch advances per launch)");
    if (!g->connected) return set_err(FQ_ERR_INVALID, "Internal Error: the pipe's group is not connected to its peers");
    if ((uint32_t)pipe->n_slots + 1 > g->row_slots) return set_err(FQ_ERR_INVALID, "Internal Error: group rows are too small for this pipe's state");
    bind_group(g, &p);
    p.merged = (fq_u64 *)pipe->d_merged;
  }
  if ((flags & FQ_RUN_BLOCK_STATS) && pipe->gen.track_blocks && src->n_rows > 0) {
    const uint64_t words = ((src->n_rows + FQ_REF_BLOCK_ROWS - 1) / FQ_REF_BLOCK_ROWS + 31) / 32;
    if (words > pipe->blocks_cap) {
      cudaFree(pipe->d_blocks);
      pipe->d_blocks = nullptr;
      CUDA_TRY(cudaMalloc(&pipe->d_blocks, sizeof(uint32_t) * words));
      pipe->blocks_cap = words;
    }
    CUDA_TRY(cudaMemsetAsync(pipe->d_blocks, 0, sizeof(uint32_t) * words, (cudaStream_t)stream));
    p.block_hit = pipe->d_blocks;
  }
  // the kernel's last CTA writes state (and merged state) straight into the pinned host mirrors: nothing is queued behind it
  p.host_state = (fq_u64 *)pipe->h_state;
  p.host_merged = pipe->group ? (fq_u64 *)pipe->h_merged : nullptr;
  if (fq_status st = launch(ctx, *k, grid, p, stream)) return st;
  pipe->launched_merged = pipe->group != nullptr;
  if (fq_status st = mark_done(ctx, pipe->ev, (cudaStream_t)stream)) return st;
  pipe->launched = true;
  return FQ_OK;
}

static fq_status decode_err(uint64_t bits) {
  if (bits & FQ_E_MERGE_TIMEOUT) return set_err(FQ_ERR_CUDA, "CUDA error: a rank of the group did not publish its state in time (cross-GPU merge timed out)");
  if (bits & FQ_E_DIVZERO) return set_err(FQ_ERR_DIVIDE_BY_ZERO, "Internal Error: Divide by zero error");
  return FQ_OK;
}

// raw state slots -> the DataValues Function::accumulate_result / merge_result would hold
static fq_status decode_states(const fq_pipe *pipe, const uint64_t *slots, bool launched, fq_value *states, int32_t cap, int32_t *n_states,
                               uint64_t *rows_selected) {
  const int n = (int)pipe->gen.agg_nodes.size();
  if (n_states) *n_states = n;
  const uint64_t nsel = slots[0], folded = slots[2];
  if (rows_selected) *rows_selected = nsel;
  if (fq_status st = decode_err(slots[1])) return st;
  for (int k = 0; k < n && k < cap && states; k++) {
    fq_value &v = states[k];
    memset(&v, 0, sizeof v);
    if (!launched || folded == 0) { v.dtype = FQ_NULL; continue; }  // state still DataValue::Null
    const int op = pipe->gen.agg_ops[k];
    const fq_dtype t = pipe->gen.agg_dtypes[k];
    const uint64_t bits = slots[FQ_STATE_HDR + k];
    v.dtype = t;
    if (op == FQ_AGG_COUNT) {  // state (+) UInt64(rows) per block, function_aggregator.rs:61-66
      v.some = 1;
      v.v.u = nsel;
      continue;
    }
    // arrow sum/min/max skip nulls and are None when no valid row was seen (empty input included)
    v.some = pipe->gen.agg_count_slot[k] >= 0 ? slots[FQ_STATE_HDR + pipe->gen.agg_count_slot[k]] > 0 : nsel > 0;
    if (!v.some) continue;
    if (t == FQ_F32 || t == FQ_F64) memcpy(&v.v.f, &bits, 8);
    else v.v.u = bits;
  }
  return FQ_OK;
}

fq_status fq_pipe_fetch_aggregate(fq_ctx *ctx, fq_pipe *pipe, fq_value *states, int32_t cap, int32_t *n_states,
                                  uint64_t *rows_selected) {
  if (fq_status st = use(ctx)) return st;
  if (!pipe || pipe->gen.kind != FQ_PIPE_AGGREGATE) return set_err(FQ_ERR_INVALID, "Internal Error: not an aggregate pipe");
  if (pipe->launched) CUDA_TRY(cudaEventSynchronize(pipe->ev));
  return decode_states(pipe, pipe->h_state, pipe->launched, states, cap, n_states, rows_selected);
}

fq_status fq_pipe_fetch_merged(fq_ctx *ctx, fq_pipe *pipe, fq_value *states, int32_t cap, int32_t *n_states,
                               uint64_t *rows_selected) {
  if (fq_status st = use(ctx)) return st;
  if (!pipe || pipe->gen.kind != FQ_PIPE_AGGREGATE) return set_err(FQ_ERR_INVALID, "Internal Error: not an aggregate pipe");
  if (!pipe->launched_merged) return set_err(FQ_ERR_INVALID, "Internal Error: the last launch of this pipe did not merge across a group");
  CUDA_TRY(cudaEventSynchronize(pipe->ev));
  return decode_states(pipe, pipe->h_merged, true, states, cap, n_states, rows_selected);
}

fq_status fq_pipe_fetch_block_stats(fq_ctx *ctx, fq_pipe *pipe, uint64_t *blocks, uint64_t *empty_blocks) {
  if (fq_status st = use(ctx)) return st;
  if (!pipe || pipe->gen.kind != FQ_PIPE_AGGREGATE) return set_err(FQ_ERR_INVALID, "Internal Error: not an aggregate pipe");
  if (pipe->launched) CUDA_TRY(cudaEventSynchronize(pipe->ev));
  if (blocks) *blocks = pipe->launched ? pipe->h_state[4] : 0;
  if (empty_blocks) *empty_blocks = pipe->launched ? pipe->h_state[5] : 0;
  return FQ_OK;
}

// ---- merge point over peer memory ----
static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the ABI passes IPC handles as 64 opaque bytes");
fq_status fq_group_create(fq_ctx *ctx, int32_t rank, int32_t world, uint64_t row_bytes, fq_group **out) {
  if (fq_status st = use(ctx)) return st;
  if (!out) return set_err(FQ_ERR_INVALID, "Internal Error: null out pointer");
  *out = nullptr;
  if (world < 1 || world > 8 || rank < 0 || rank >= world) return set_err(FQ_ERR_INVALID, "Internal Error: a group has 1..8 ranks");
  if (row_bytes < 256 || row_bytes > (64u << 20)) return set_err(FQ_ERR_INVALID, "Internal Error: group rows hold 256 B .. 64 MB");
  fq_group *g = new fq_group();
  g->rank = rank;
  g->world = world;
  g->row_slots = (uint32_t)((row_bytes + 7) / 8);
  if (const char *t = getenv("FQ_GROUP_TIMEOUT_MS")) {
    if (atoll(t) > 0) g->timeout_ns = (uint64_t)atoll(t) * 1000000ull;
  }
  const size_t bytes = sizeof(uint64_t) * 2 * (size_t)world * g->row_slots;
  cudaError_t e = cudaMalloc(&g->window, bytes);
  if (e == cudaSuccess) e = cudaMemset(g->window, 0, bytes);
  if (e == cudaSuccess) e = cudaMalloc(&g->d_result, 64);
  if (e == cudaSuccess) e = cudaMemset(g->d_result, 0, 64);
  if (e == cudaSuccess) e = cudaHostAlloc(&g->h_result, 64, cudaHostAllocDefault);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->ev, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    fq_group_destroy(ctx, g);
    return set_err(FQ_ERR_CUDA, "CUDA error: %s (group buffers)", cudaGetErrorString(e));
  }
  g->windows[rank] = g->window;
  g->connected = world == 1;
  *out = g;
  return FQ_OK;
}
fq_status fq_group_handle(fq_ctx *ctx, const fq_group *g, void *handle64) {
  if (fq_status st = use(ctx)) return st;
  if (!g || !handle64) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  cudaIpcMemHandle_t h;
  CUDA_TRY(cudaIpcGetMemHandle(&h, g->window));
  memcpy(handle64, &h, sizeof h);
  return FQ_OK;
}
fq_status fq_group_window(fq_ctx *, const fq_group *g, void **dev_ptr, uint64_t *n_bytes) {
  if (!g || !dev_ptr) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  *dev_ptr = g->window;
  if (n_bytes) *n_bytes = sizeof(uint64_t) * 2 * (uint64_t)g->world * g->row_slots;
  return FQ_OK;
}
fq_status fq_group_connect(fq_ctx *ctx, fq_group *g, const void *handles) {
  if (fq_status st = use(ctx)) return st;
  if (!g || !handles) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (g->world == 1) return FQ_OK;   // nothing to connect
  if (g->connected) return set_err(FQ_ERR_INVALID, "Internal Error: the group is already connected");
  for (int r = 0; r < g->world; r++) {
    if (r == g->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char *)handles + 64 * (size_t)r, sizeof h);
    void *ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      for (int q = 0; q < r; q++)
        if (g->ipc_opened[q]) { cudaIpcCloseMemHandle(g->windows[q]); g->ipc_opened[q] = false; g->windows[q] = nullptr; }
      return set_err(FQ_ERR_CUDA, "CUDA error: %s (cudaIpcOpenMemHandle of rank %d's window)", cudaGetErrorString(e), r);
    }
    g->windows[r] = (uint64_t *)ptr;
    g->ipc_opened[r] = true;
  }
  g->connected = true;
  return FQ_OK;
}
fq_status fq_group_connect_ptrs(fq_ctx *ctx, fq_group *g, void *const *windows) {
  if (!ctx || !g || !windows) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (g->world == 1) return FQ_OK;   // nothing to connect
  if (g->connected) return set_err(FQ_ERR_INVALID, "Internal Error: the group is already connected");
  for (int r = 0; r < g->world; r++) {
    if (r == g->rank) continue;
    if (!windows[r]) return set_err(FQ_ERR_INVALID, "Internal Error: missing window of rank %d", r);
    g->windows[r] = (uint64_t *)windows[r];
  }
  g->connected = true;
  return FQ_OK;
}
void fq_group_destroy(fq_ctx *ctx, fq_group *g) {
  if (!g) return;
  if (ctx) cudaSetDevice(ctx->device);
  for (int r = 0; r < 8; r++)
    if (g->ipc_opened[r]) cudaIpcCloseMemHandle(g->windows[r]);
  cudaFree(g->window);
  cudaFree(g->d_result);
  if (g->h_result) cudaFreeHost(g->h_result);
  if (g->ev) cudaEventDestroy(g->ev);
  delete g;
}
fq_status fq_pipe_set_group(fq_ctx *ctx, fq_pipe *pipe, fq_group *g) {
  if (fq_status st = use(ctx)) return st;
  if (!pipe) return set_err(FQ_ERR_INVALID, "Internal Error: null pipe");
  if (g && pipe->gen.kind == FQ_PIPE_AGGREGATE) {
    if ((uint32_t)pipe->n_slots + 1 > g->row_slots) return set_err(FQ_ERR_INVALID, "Internal Error: group rows are too small for this pipe's state");
    if (!pipe->d_merged) {
      CUDA_TRY(cudaMalloc(&pipe->d_merged, sizeof(uint64_t) * pipe->n_slots));
      CUDA_TRY(cudaMemset(pipe->d_merged, 0, sizeof(uint64_t) * pipe->n_slots));
      CUDA_TRY(cudaHostAlloc(&pipe->h_merged, sizeof(uint64_t) * pipe->n_slots, cudaHostAllocDefault));
      memset(pipe->h_merged, 0, sizeof(uint64_t) * pipe->n_slots);
    }
  }
  pipe->group = g;
  return FQ_OK;
}

// Ordered concatenation of every rank's filtered + projected rows, cut at `limit` — MergeProcessor + the LimitTransform
// after it (processor_merge.rs:37-66, pipeline_builder.rs:31-41), ranks in partition order (a legal merge order, SURVEY F9).
// One CTA: publish this rank's {selected, written, error bits, rows} into every rank's window, wait for all rows of
// the epoch, copy the first `limit` rows in rank order into the final columns.
struct fq_gather_params {
  fq_launch_params g;          // group_* fields only
  const void *src[2 * FQ_MAX_EXPRS];
  void *dst[2 * FQ_MAX_EXPRS];
  fq_u32 elem[2 * FQ_MAX_EXPRS];
  fq_u32 col_slot[2 * FQ_MAX_EXPRS];   // first slot of column c inside a row's payload
  fq_u32 n_cols;
  fq_u64 local_selected, local_rows;   // used instead of local_result when use_imm != 0 (columns of any producer)
  fq_u32 use_imm;
  const fq_u64 *local_result;  // the projection launch's result block: [0] rows selected, [1] error bits
  fq_u64 cap_local;            // rows the local launch may have written
  fq_u64 limit;                // final rows = min(limit, sum of written)
  fq_u64 *out_result;          // [0] rows selected by all ranks, [1] final rows, [2] error bits
};
__global__ void __launch_bounds__(256) fq_group_gather_rows(const __grid_constant__ fq_gather_params a) {
  const fq_launch_params &p = a.g;
  __shared__ fq_u64 s_off[9], s_take[8], s_sel, s_err;
  __shared__ int s_ok;
  const fq_u64 selected = a.use_imm ? a.local_selected : a.local_result[0];
  const fq_u64 written = a.use_imm ? a.local_rows : (selected < a.cap_local ? selected : a.cap_local);
  // payload into every rank's window: 8-byte words (columns are 256-byte padded, rows 8-byte slotted)
  for (fq_u32 r = 0; r < p.group_world; r++) {
    fq_u64 *row = fq_group_row(p, (int)r, (int)p.group_rank);
    for (fq_u32 c = 0; c < a.n_cols; c++) {
      const fq_u64 words = (written * a.elem[c] + 7) / 8;
      const fq_u64 *src = (const fq_u64 *)a.src[c];
      fq_u64 *dst = row + a.col_slot[c];
      for (fq_u64 i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
    }
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < p.group_world) {
    fq_u64 *row = fq_group_row(p, (int)threadIdx.x, (int)p.group_rank);
    row[1] = selected;
    row[2] = written;
    row[3] = a.use_imm ? 0ull : a.local_result[1];
    __threadfence_system();
    fq_st_release_sys(row, p.group_epoch);
  }
  if (threadIdx.x < 32) {
    const bool ok = fq_group_wait(p);
    if (threadIdx.x == 0) {
      s_ok = ok ? 1 : 0;
      fq_u64 off = 0, sel = 0, err = ok ? 0 : FQ_E_MERGE_TIMEOUT;
      for (fq_u32 r = 0; r < p.group_world; r++) {
        const fq_u64 *row = fq_group_row(p, (int)p.group_rank, (int)r);
        const fq_u64 w = ok ? fq_ld_cg(row + 2) : 0;
        const fq_u64 take = off + w <= a.limit ? w : a.limit - off;
        s_off[r] = off;
        s_take[r] = take;
        off += take;
        sel += ok ? fq_ld_cg(row + 1) : 0;
        err |= ok ? fq_ld_cg(row + 3) : 0;
      }
      s_off[p.group_world] = off;
      s_sel = sel;
      s_err = err;
    }
  }
  __syncthreads();
  for (fq_u32 r = 0; r < p.group_world; r++) {
    const fq_u64 *row = fq_group_row(p, (int)p.group_rank, (int)r);
    for (fq_u32 c = 0; c < a.n_cols; c++) {
      const unsigned char *src = (const unsigned char *)(row + a.col_slot[c]);
      unsigned char *dst = (unsigned char *)a.dst[c] + s_off[r] * a.elem[c];
      const fq_u64 bytes = s_take[r] * a.elem[c];
      if (a.elem[c] == 8) {
        for (fq_u64 i = threadIdx.x; i < s_take[r]; i += blockDim.x) ((fq_u64 *)dst)[i] = fq_ld_cg((const fq_u64 *)src + i);
      } else {
        for (fq_u64 i = threadIdx.x; i < bytes; i += blockDim.x) dst[i] = *(const volatile unsigned char *)(src + i);
      }
    }
  }
  if (threadIdx.x == 0) {
    a.out_result[0] = s_sel;
    a.out_result[1] = s_off[p.group_world];
    a.out_result[2] = s_err;
  }
}

fq_status fq_group_gather_project(fq_ctx *ctx, fq_group *g, fq_pipe *pipe, fq_column *const *local_cols, fq_column *const *local_valid,
                                  fq_column *const *final_cols, fq_column *const *final_valid, int64_t limit, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!g || !pipe || pipe->gen.kind != FQ_PIPE_PROJECT || !pipe->launched_project)
    return set_err(FQ_ERR_INVALID, "Internal Error: gather needs a group and a projection pipe that was launched");
  if (!g->connected) return set_err(FQ_ERR_INVALID, "Internal Error: the group is not connected to its peers");
  if (ctx->recording) return set_err(FQ_ERR_INVALID, "Internal Error: a group operation cannot be recorded into a graph (its epoch advances per call)");
  fq_gather_params a;
  memset(&a, 0, sizeof a);
  const int ne = (int)pipe->gen.expr_dtypes.size();
  const uint64_t cap = pipe->capacity_eff;
  const uint64_t lim = limit < 0 ? cap * (uint64_t)g->world : (uint64_t)limit;
  uint64_t slot = 4;   // [0] epoch, [1] selected, [2] written, [3] error bits
  for (int e = 0; e < ne; e++) {
    for (int v = 0; v < 2; v++) {
      const bool nullable = e < (int)pipe->gen.expr_nullable.size() && pipe->gen.expr_nullable[e];
      if (v == 1 && !nullable) continue;
      const fq_column *lc = v ? (local_valid ? local_valid[e] : nullptr) : (local_cols ? local_cols[e] : nullptr);
      const fq_column *fc = v ? (final_valid ? final_valid[e] : nullptr) : (final_cols ? final_cols[e] : nullptr);
      const fq_dtype want = v ? (fq_dtype)FQ_BOOL : pipe->gen.expr_dtypes[e];
      if (!lc || !fc || lc->dtype != want || fc->dtype != want)
        return set_err(FQ_ERR_INVALID, "Internal Error: gather column %d%s missing or of the wrong type", e, v ? " (validity)" : "");
      if (lc->len < cap || fc->len < std::min<uint64_t>(lim, cap * (uint64_t)g->world))
        return set_err(FQ_ERR_INVALID, "Internal Error: gather column %d is shorter than the rows it may receive", e);
      const uint32_t w = (uint32_t)fq::dtype_size(want);
      const int c = (int)a.n_cols++;
      a.src[c] = lc->ptr;
      a.dst[c] = fc->ptr;
      a.elem[c] = w;
      a.col_slot[c] = (fq_u32)slot;
      slot += (cap * w + 7) / 8;
    }
  }
  if (slot > g->row_slots)
    return set_err(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: %" PRIu64 " rows per rank do not fit the group's %u-byte rows", cap,
                   g->row_slots * 8u);
  bind_group(g, &a.g);
  a.local_result = (const fq_u64 *)pipe->d_ctl;
  a.cap_local = cap;
  a.limit = lim;
  a.out_result = (fq_u64 *)g->d_result;
  fq_group_gather_rows<<<1, 256, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  CUDA_TRY(cudaMemcpyAsync(g->h_result, g->d_result, 24, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CUDA_TRY(cudaEventRecord(g->ev, (cudaStream_t)stream));
  g->gathered = true;
  return FQ_OK;
}
fq_status fq_group_gather_columns(fq_ctx *ctx, fq_group *g, const fq_column *const *local_cols, const fq_column *const *local_valid,
                                  int32_t n_cols, uint64_t rows_local, uint64_t rows_selected_local, uint64_t capacity,
                                  fq_column *const *final_cols, fq_column *const *final_valid, int64_t limit, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!g || !local_cols || !final_cols || n_cols < 1 || n_cols > FQ_MAX_EXPRS) return set_err(FQ_ERR_INVALID, "Internal Error: gather needs a group and 1..8 columns");
  if (!g->connected) return set_err(FQ_ERR_INVALID, "Internal Error: the group is not connected to its peers");
  if (rows_local > capacity) return set_err(FQ_ERR_INVALID, "Internal Error: more local rows than the capacity every rank agreed on");
  if (ctx->recording) return set_err(FQ_ERR_INVALID, "Internal Error: a group operation cannot be recorded into a graph (its epoch advances per call)");
  fq_gather_params a;
  memset(&a, 0, sizeof a);
  const uint64_t lim = limit < 0 ? capacity * (uint64_t)g->world : (uint64_t)limit;
  uint64_t slot = 4;
  for (int e = 0; e < n_cols; e++) {
    for (int v = 0; v < 2; v++) {
      const fq_column *lc = v ? (local_valid ? local_valid[e] : nullptr) : local_cols[e];
      const fq_column *fc = v ? (final_valid ? final_valid[e] : nullptr) : final_cols[e];
      if (v == 1 && !fc) continue;    // this column has no validity (every rank must agree)
      if (!fc || (rows_local && !lc) || (lc && lc->dtype != fc->dtype) || (v == 1 && fc->dtype != FQ_BOOL))
        return set_err(FQ_ERR_INVALID, "Internal Error: gather column %d%s missing or of the wrong type", e, v ? " (validity)" : "");
      if ((lc && lc->len < rows_local) || fc->len < std::min<uint64_t>(lim, capacity * (uint64_t)g->world))
        return set_err(FQ_ERR_INVALID, "Internal Error: gather column %d is shorter than the rows it may receive", e);
      const uint32_t w = (uint32_t)fq::dtype_size(fc->dtype);
      const int c = (int)a.n_cols++;
      a.src[c] = lc ? lc->ptr : fc->ptr;   // (no local rows: never read)
      a.dst[c] = fc->ptr;
      a.elem[c] = w;
      a.col_slot[c] = (fq_u32)slot;
      slot += (capacity * w + 7) / 8;
    }
  }
  if (slot > g->row_slots)
    return set_err(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: %" PRIu64 " rows per rank do not fit the group's %u-byte rows", capacity,
                   g->row_slots * 8u);
  bind_group(g, &a.g);
  a.use_imm = 1;
  a.local_selected = rows_selected_local;
  a.local_rows = rows_local;
  a.cap_local = capacity;
  a.limit = lim;
  a.out_result = (fq_u64 *)g->d_result;
  fq_group_gather_rows<<<1, 256, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  CUDA_TRY(cudaMemcpyAsync(g->h_result, g->d_result, 24, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CUDA_TRY(cudaEventRecord(g->ev, (cudaStream_t)stream));
  g->gathered = true;
  return FQ_OK;
}
fq_status fq_group_fetch_gather(fq_ctx *ctx, fq_group *g, uint64_t *rows_selected, uint64_t *rows_final) {
  if (fq_status st = use(ctx)) return st;
  if (!g || !g->gathered) return set_err(FQ_ERR_INVALID, "Internal Error: no gather to fetch");
  CUDA_TRY(cudaEventSynchronize(g->ev));
  if (rows_selected) *rows_selected = g->h_result[0];
  if (rows_final) *rows_final = g->h_result[1];
  return decode_err(g->h_result[2]);
}

fq_status fq_pipe_launch_project(fq_ctx *ctx, fq_pipe *pipe, const fq_source *src, fq_column *const *out_cols,
                                 fq_column *const *out_valid, uint64_t capacity, int64_t limit, uint32_t flags, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!pipe || pipe->gen.kind != FQ_PIPE_PROJECT) return set_err(FQ_ERR_INVALID, "Internal Error: not a projection pipe");
  fq_launch_params p;
  memset(&p, 0, sizeof p);
  if (fq_status st = bind_source(pipe, src, &p)) return st;
  uint64_t cap = capacity;
  if (limit >= 0 && (uint64_t)limit < cap) cap = (uint64_t)limit;
  const int ne = (int)pipe->gen.expr_dtypes.size();
  for (int e = 0; e < ne; e++) {
    const fq_column *c = out_cols ? out_cols[e] : nullptr;
    if (!c) return set_err(FQ_ERR_INVALID, "Internal Error: missing output column %d", e);
    if (c->dtype != pipe->gen.expr_dtypes[e])
      return set_err(FQ_ERR_INVALID, "Internal Error: output column %d is %s, expression yields %s", e, fq::dtype_name(c->dtype),
                     fq::dtype_name(pipe->gen.expr_dtypes[e]));
    if (c->len < cap && c->len < capacity) return set_err(FQ_ERR_INVALID, "Internal Error: output column %d shorter than capacity", e);
    p.outs[e] = c->ptr;
    if (e < (int)pipe->gen.expr_nullable.size() && pipe->gen.expr_nullable[e]) {
      const fq_column *vcol = out_valid ? out_valid[e] : nullptr;
      if (!vcol || vcol->dtype != FQ_BOOL || (vcol->len < cap && vcol->len < capacity))
        return set_err(FQ_ERR_INVALID, "Internal Error: select expression %d can yield NULL: a Boolean validity output column is required", e);
      p.outs_valid[e] = vcol->ptr;
    }
  }
  p.capacity = cap;
  pipe->capacity_eff = cap;
  p.result = (fq_u64 *)pipe->d_ctl;
  p.tile_counter = (fq_u32 *)(pipe->d_ctl + 2);
  p.done = (fq_u32 *)(pipe->d_ctl + 3);
  p.stop_after = ((flags & FQ_RUN_LIMIT_EARLY_EXIT) && limit > 0) ? (uint64_t)limit : 0;
  CUDA_TRY(cudaMemsetAsync(pipe->d_ctl, 0, 64, (cudaStream_t)stream));
  pipe->skipped = false;
  pipe->project_has_pred_launch = false;
  if (src->n_rows == 0) {
    pipe->skipped = true;
  } else if (pipe->gen.has_pred) {
    const Kernel *k;
    if (fq_status st = pick_kernel(pipe, K_SELECT_TMA, K_SELECT, p, "select", &k)) return st;
    const Kernel &kd = pipe->k[K_SELECT_DENSE];
    // the dense-tuned build pays off when a good part of the rows is written: outputs of at least 1/16 of a large source
    const bool dense_ok = k->staged && kd.valid() && pipe->k[K_SELECT_PROBE].valid() && !p.unaligned;
    const bool force_dense = dense_ok && pipe->variant == V_DENSE;
    const bool probe = dense_ok && pipe->variant == V_TMA && src->n_rows >= (4u << 20) && cap >= src->n_rows / 16 && p.stop_after == 0;
    const uint64_t segs_sparse = (src->n_rows + k->rows - 1) / k->rows;
    const uint64_t segs_dense = (probe || force_dense) ? (src->n_rows + kd.rows - 1) / kd.rows : 0;
    const uint64_t segs_max = std::max(segs_sparse, segs_dense);
    if (segs_max > pipe->tiles_cap) {
      cudaFree(pipe->d_tiles);
      pipe->d_tiles = nullptr;
      CUDA_TRY(cudaMalloc(&pipe->d_tiles, sizeof(uint64_t) * segs_max));
      pipe->tiles_cap = segs_max;
    }
    p.tile_status = (fq_u64 *)pipe->d_tiles;
    CUDA_TRY(cudaMemsetAsync(pipe->d_tiles, 0, sizeof(uint64_t) * segs_max, (cudaStream_t)stream));
    fq_u32 *probe_words = (fq_u32 *)(pipe->d_ctl + 6);   // [0] sampled, [1] kept, [2] mode, [3] CTA ticket
    if (probe) {
      fq_launch_params pp = p;
      pp.probe = probe_words;
      if (fq_status st = launch(ctx, pipe->k[K_SELECT_PROBE], (unsigned)ctx->sm_count, pp, stream)) return st;
      p.sel_mode = probe_words + 2;
    }
    if (!force_dense) {   // the sparse-tuned build (or the LDG kernel)
      fq_launch_params ps = p;
      ps.stages = pipe->k[K_SELECT_TMA].stages;
      ps.stages2 = 0;
      ps.n_tiles = segs_sparse;
      if (fq_status st = launch(ctx, *k, persistent_grid(ctx, *k, src->n_rows), ps, stream)) return st;
    }
    if (probe || force_dense) {   // the dense-tuned build: returns at once when the probe chose the other one
      fq_launch_params pd = p;
      pd.stages = kd.stages;
      pd.stages2 = 1;
      pd.n_tiles = segs_dense;
      if (fq_status st = launch(ctx, kd, persistent_grid(ctx, kd, src->n_rows), pd, stream)) return st;
    }
    pipe->project_has_pred_launch = true;
  } else {
    // LIMIT without a filter: rows past the 10 000-row block that completes the limit are neither read nor evaluated.
    // (The reference's LimitStream polls its input once more before it ends, stream_limit.rs:58-62, so it still evaluates
    // the FOLLOWING block: a caller that wants the reference's errors checks the rows up to the end of that block itself —
    // fq_pipe_fetch_limit_row tells where; the host mirror's GpuPipeTransform does.)
    if ((flags & FQ_RUN_LIMIT_EARLY_EXIT) && limit >= 0) {
      const uint64_t blocks = ((uint64_t)limit + FQ_REF_BLOCK_ROWS - 1) / FQ_REF_BLOCK_ROWS;
      p.n_rows = std::min<uint64_t>(p.n_rows, std::max<uint64_t>(blocks, 1) * FQ_REF_BLOCK_ROWS);
    }
    const Kernel *k;
    if (fq_status st = pick_kernel(pipe, K_MAP_TMA, K_MAP, p, "projection", &k)) return st;
    p.stages = pipe->k[K_MAP_TMA].stages;
    if (fq_status st = launch(ctx, *k, persistent_grid(ctx, *k, p.n_rows), p, stream)) return st;
  }
  CUDA_TRY(cudaMemcpyAsync(pipe->h_result, pipe->d_ctl, 48, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  if (fq_status st = mark_done(ctx, pipe->ev, (cudaStream_t)stream)) return st;
  pipe->launched_project = true;
  return FQ_OK;
}

fq_status fq_pipe_fetch_project(fq_ctx *ctx, fq_pipe *pipe, uint64_t *rows_selected, uint64_t *rows_written) {
  if (fq_status st = use(ctx)) return st;
  if (!pipe || !pipe->launched_project) return set_err(FQ_ERR_INVALID, "Internal Error: no projection launch to fetch");
  CUDA_TRY(cudaEventSynchronize(pipe->ev));
  const uint64_t sel = pipe->skipped ? 0 : pipe->h_result[0];
  if (rows_selected) *rows_selected = sel;
  if (rows_written) *rows_written = std::min(sel, pipe->capacity_eff);
  return decode_err(pipe->h_result[1]);
}


fq_status fq_pipe_fetch_limit_row(fq_ctx *ctx, fq_pipe *pipe, uint64_t *row) {
  if (fq_status st = use(ctx)) return st;
  if (!pipe || !pipe->launched_project || !row) return set_err(FQ_ERR_INVALID, "Internal Error: no projection launch to fetch");
  CUDA_TRY(cudaEventSynchronize(pipe->ev));
  const uint64_t sel = pipe->skipped ? 0 : pipe->h_result[0];
  if (pipe->capacity_eff == 0 || sel < pipe->capacity_eff) return set_err(FQ_ERR_INVALID, "Internal Error: the launch did not fill its capacity");
  *row = pipe->project_has_pred_launch ? pipe->h_result[5] : pipe->capacity_eff - 1;
  return FQ_OK;
}

}  // extern "C"

// =============================================================================================
// GROUP BY pipes (hash aggregation)
// =============================================================================================
namespace {
// The host-compiled kernels below serve every GROUP BY pipe: `kw` is its key width in 64-bit words (Generated::key_words),
// and key i of a table is words [i * kw, i * kw + kw) of its key array.
__global__ void __launch_bounds__(256) fq_gb_fill(fq_u64 *keys, int kw, fq_u64 *slots, fq_u64 n_entries, int G, const fq_u64 *identity) {
  const fq_u64 tid = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (fq_u64)gridDim.x * blockDim.x;
  for (fq_u64 i = tid; i < n_entries * (fq_u64)kw; i += nthreads) keys[i] = FQ_GB_EMPTY;
  for (fq_u64 i = tid; i < n_entries * (fq_u64)G; i += nthreads) slots[i] = identity[i % (fq_u64)G];
}
// the words of key i: hi = 0 for one-word keys
__device__ __forceinline__ fq_gb_key2 fq_gb_key_at(const fq_u64 *keys, int kw, fq_u64 i) {
  return {keys[i * kw], kw == 2 ? keys[i * kw + 1] : 0ull};
}
__device__ __forceinline__ bool fq_gb_occupied(const fq_u64 *keys, int kw, fq_u64 cap, const fq_u32 *flags, fq_u64 i) {
  return i < cap ? keys[i * kw] != FQ_GB_EMPTY || (kw == 2 && keys[i * kw + 1] != FQ_GB_EMPTY) : (i == cap && flags[1] != 0);
}
__global__ void __launch_bounds__(256) fq_gb_count(const fq_u64 *keys, int kw, fq_u64 cap, fq_u32 *flags) {
  const fq_u64 tid = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (fq_u64)gridDim.x * blockDim.x;
  fq_u64 n = 0;
  for (fq_u64 i = tid; i <= cap; i += nthreads) n += fq_gb_occupied(keys, kw, cap, flags, i) ? 1 : 0;
  for (int m = 16; m > 0; m >>= 1) n += __shfl_xor_sync(0xffffffffu, n, m);
  if ((threadIdx.x & 31) == 0 && n) atomicAdd((unsigned long long *)(flags + 2), (unsigned long long)n);
}
struct fq_gb_export_params {
  const fq_u64 *keys, *slots;
  fq_u64 cap;
  const fq_u32 *flags;
  int kw, G, n_keys, n_leaves;
  int key_shift[FQ_MAX_KEYS], key_bits[FQ_MAX_KEYS], key_nullable[FQ_MAX_KEYS];
  void *key_out[FQ_MAX_KEYS], *key_valid[FQ_MAX_KEYS];
  int leaf_op[16], leaf_dtype[16], leaf_count_slot[16];
  void *leaf_out[16], *leaf_valid[16];
  fq_u64 capacity;
  fq_u64 *counter;
};
__device__ __forceinline__ void fq_store_low(void *base, fq_u64 idx, int bytes, fq_u64 v) {
  switch (bytes) {
    case 1: ((fq_u8 *)base)[idx] = (fq_u8)v; break;
    case 2: ((fq_u16 *)base)[idx] = (fq_u16)v; break;
    case 4: ((fq_u32 *)base)[idx] = (fq_u32)v; break;
    default: ((fq_u64 *)base)[idx] = v;
  }
}
__global__ void __launch_bounds__(256) fq_gb_export(const __grid_constant__ fq_gb_export_params a) {
  const fq_u64 tid = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (fq_u64)gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  const fq_u64 rounds = (a.cap + 1 + nthreads - 1) / nthreads;
  for (fq_u64 k = 0; k < rounds; k++) {
    const fq_u64 i = k * nthreads + tid;
    const bool occ = i <= a.cap && fq_gb_occupied(a.keys, a.kw, a.cap, a.flags, i);
    const fq_u32 m = __ballot_sync(0xffffffffu, occ);
    if (!m) continue;
    fq_u64 base = 0;
    if (lane == 0) base = atomicAdd((unsigned long long *)a.counter, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (!occ) continue;
    const fq_u64 pos = base + __popc(m & ((1u << lane) - 1u));
    if (pos >= a.capacity) continue;
    const fq_gb_key2 key = i < a.cap ? fq_gb_key_at(a.keys, a.kw, i) : fq_gb_key2{FQ_GB_EMPTY, FQ_GB_EMPTY};
    for (int j = 0; j < a.n_keys; j++) {
      // the field's value bits at [s, s + w), possibly across lo / hi, and its null flag at bit s + w
      const int s = a.key_shift[j], w = a.key_bits[j], f = s + w;
      fq_u64 bits = s >= 64 ? key.hi >> (s - 64) : s == 0 ? key.lo : (key.lo >> s) | (key.hi << (64 - s));
      if (w < 64) bits &= (1ull << w) - 1ull;
      fq_store_low(a.key_out[j], pos, w / 8, bits);
      if (a.key_nullable[j]) ((fq_u8 *)a.key_valid[j])[pos] = (fq_u8)((((f >= 64 ? key.hi >> (f - 64) : key.lo >> f)) & 1ull) ? 0 : 1);
    }
    const fq_u64 *st = a.slots + i * (fq_u64)a.G;
    for (int l = 0; l < a.n_leaves; l++) {
      const int op = a.leaf_op[l], t = a.leaf_dtype[l];
      fq_u64 x = op == FQ_AGG_COUNT ? st[0] : st[1 + l];
      if (t == FQ_F32 || t == FQ_F64) {
        const double d = op == FQ_AGG_SUM ? __longlong_as_double((fq_i64)x) : fq_f64_unordered(x);
        if (t == FQ_F32) ((float *)a.leaf_out[l])[pos] = (float)d;
        else ((double *)a.leaf_out[l])[pos] = d;
      } else {
        fq_store_low(a.leaf_out[l], pos, t == FQ_BOOL || t == FQ_I8 || t == FQ_U8 ? 1 : t == FQ_I16 || t == FQ_U16 ? 2 : t == FQ_I32 || t == FQ_U32 ? 4 : 8, x);
      }
      if (a.leaf_count_slot[l] >= 0 && a.leaf_valid[l]) ((fq_u8 *)a.leaf_valid[l])[pos] = st[1 + a.leaf_count_slot[l]] > 0 ? 1 : 0;
    }
  }
}
// partial groups ordered by owner rank: pass 0 counts (cursor[d] += ...), pass 1 writes entries at cursor positions
__global__ void __launch_bounds__(256) fq_gb_partials(const fq_u64 *keys, int kw, const fq_u64 *slots, fq_u64 cap, const fq_u32 *flags, int G, int world,
                                                      unsigned long long *cursor, fq_u64 *entries, int pass) {
  __shared__ fq_u32 cnt[8], base_lo[8];
  __shared__ unsigned long long base[8];
  const fq_u64 nthreads = (fq_u64)gridDim.x * blockDim.x;
  const fq_u64 rounds = (cap + 1 + nthreads - 1) / nthreads;
  (void)base_lo;
  for (fq_u64 k = 0; k < rounds; k++) {
    const fq_u64 i = (k * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
    if (threadIdx.x < 8) cnt[threadIdx.x] = 0;
    __syncthreads();
    const bool occ = i <= cap && fq_gb_occupied(keys, kw, cap, flags, i);
    const fq_gb_key2 key = occ && i < cap ? fq_gb_key_at(keys, kw, i) : fq_gb_key2{FQ_GB_EMPTY, kw == 2 ? FQ_GB_EMPTY : 0ull};
    // the owner rank: the unseeded hash the pipe's first table uses, so every rank agrees whatever its own table's seed
    const fq_u64 h = kw == 2 ? fq_gb_seeded(key, 0) : fq_gb_hash(key.lo);
    const int dest = (int)((h >> 40) % (fq_u64)world);
    fq_u32 r = 0;
    if (occ) r = atomicAdd(&cnt[dest], 1u);
    __syncthreads();
    if ((int)threadIdx.x < world && cnt[threadIdx.x]) base[threadIdx.x] = atomicAdd(cursor + threadIdx.x, (unsigned long long)cnt[threadIdx.x]);
    __syncthreads();
    if (occ && pass == 1) {
      fq_u64 *e = entries + (base[dest] + r) * (fq_u64)(kw + G);
      e[0] = key.lo;
      if (kw == 2) e[1] = key.hi;
      for (int s = 0; s < G; s++) e[kw + s] = slots[i * (fq_u64)G + s];
    }
    __syncthreads();
  }
}
__global__ void fq_gb_prefix(unsigned long long *cursor, unsigned long long *counts_out, int world) {
  unsigned long long run = 0;
  for (int d = 0; d < world; d++) {
    const unsigned long long c = cursor[d];
    counts_out[d] = c;
    cursor[d] = run;
    run += c;
  }
}

std::vector<uint64_t> gb_identity(const fq::Generated &gen) {
  std::vector<uint64_t> idn(1 + gen.n_slots, 0);
  for (size_t k = 0; k < gen.agg_ops.size(); k++) {
    const int op = gen.agg_ops[k];
    const fq_dtype t = gen.agg_dtypes[k];
    const bool sgn = t >= FQ_I8 && t <= FQ_I64;
    if (op == FQ_AGG_MIN) idn[1 + k] = sgn ? (uint64_t)INT64_MAX : ~0ull;
    else if (op == FQ_AGG_MAX) idn[1 + k] = sgn ? (uint64_t)INT64_MIN : 0ull;
  }
  return idn;
}
uint64_t splitmix64(uint64_t x) {
  x += 0x9e3779b97f4a7c15ull;
  x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
  x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
  return x ^ (x >> 31);
}
fq_status gb_check(const fq_pipe *pipe) {
  if (!pipe || pipe->gen.kind != FQ_PIPE_GROUPBY) return set_err(FQ_ERR_INVALID, "Internal Error: not a GROUP BY pipe");
  return FQ_OK;
}
// empty table on `stream`: keys = EMPTY, states = the aggregates' identities, flags = 0
fq_status gb_clear(fq_ctx *ctx, fq_pipe *pipe, cudaStream_t s) {
  const int G = 1 + pipe->gen.n_slots;
  CUDA_TRY(cudaMemsetAsync(pipe->gb_flags, 0, 64, s));
  const unsigned grid = (unsigned)std::min<uint64_t>((pipe->gb_cap + 256) / 256, (uint64_t)ctx->sm_count * 8);
  const int kw = pipe->gen.key_words;
  fq_gb_fill<<<grid, 256, 0, s>>>((fq_u64 *)pipe->gb_keys, kw, (fq_u64 *)pipe->gb_slots, pipe->gb_cap + 1, G, (const fq_u64 *)pipe->gb_identity);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  if (pipe->gb_reps > 1 && pipe->gb_reps_dirty) {
    const uint64_t n = (pipe->gb_cap + 1) * (pipe->gb_reps - 1);
    const unsigned g2 = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * 8);
    fq_gb_fill<<<g2, 256, 0, s>>>((fq_u64 *)pipe->gb_rep_keys, kw, (fq_u64 *)pipe->gb_rep_slots, n, G, (const fq_u64 *)pipe->gb_identity);
    CUDA_TRY(cudaGetLastError());
    ctx->launches++;
    pipe->gb_reps_dirty = false;
  }
  pipe->launched_groupby = false;
  return FQ_OK;
}
}  // namespace

extern "C" {

fq_status fq_pipe_key_dtype(fq_ctx *, const fq_pipe *pipe, int32_t j, fq_dtype *out, int32_t *nullable) {
  if (fq_status st = gb_check(pipe)) return st;
  if (j < 0 || j >= (int)pipe->gen.key_dtypes.size() || !out) return set_err(FQ_ERR_INVALID, "Internal Error: bad key index");
  *out = pipe->gen.key_dtypes[j];
  if (nullable) *nullable = pipe->gen.key_nullable[j];
  return FQ_OK;
}
fq_status fq_pipe_leaf_dtype(fq_ctx *, const fq_pipe *pipe, int32_t k, fq_dtype *out, int32_t *nullable) {
  if (!pipe || pipe->gen.kind == FQ_PIPE_PROJECT) return set_err(FQ_ERR_INVALID, "Internal Error: not an aggregate or GROUP BY pipe");
  if (k < 0 || k >= (int)pipe->gen.agg_dtypes.size() || !out) return set_err(FQ_ERR_INVALID, "Internal Error: bad leaf index");
  *out = pipe->gen.agg_dtypes[k];
  if (nullable) *nullable = pipe->gen.agg_count_slot[k] >= 0 ? 1 : 0;
  return FQ_OK;
}
fq_status fq_pipe_group_entry_slots(fq_ctx *, const fq_pipe *pipe, int32_t *slots) {
  if (fq_status st = gb_check(pipe)) return st;
  if (!slots) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  *slots = pipe->gen.key_words + 1 + pipe->gen.n_slots;
  return FQ_OK;
}

fq_status fq_pipe_groupby_reserve(fq_ctx *ctx, fq_pipe *pipe, uint64_t groups) {
  if (fq_status st = use(ctx)) return st;
  if (fq_status st = gb_check(pipe)) return st;
  uint64_t cap = 1024;
  while (cap < groups * 2 && cap < (1ull << 40)) cap *= 2;   // load factor <= 1/2
  const int G = 1 + pipe->gen.n_slots, kw = pipe->gen.key_words;
  // Replicas of a small table (CTA b aggregates into replica b % reps, folded into the table after the scan): as many as
  // fit FQ_GB_REPLICA_BYTES (default 32 MB, a quarter of L2), at most 32.  A table beyond that budget has enough slots that
  // the CTAs rarely meet on one line and stays single.
  uint64_t budget = 32ull << 20;
  unsigned max_reps = 32;
  if (const char *e = getenv("FQ_GB_REPLICA_BYTES")) budget = strtoull(e, nullptr, 10);
  if (const char *e = getenv("FQ_GB_REPLICAS")) max_reps = (unsigned)std::max(1, atoi(e));
  unsigned reps = 1;
  while (reps * 2 <= max_reps && (uint64_t)(reps * 2) * (cap + 1) * 8 * (kw + G) <= budget) reps *= 2;
  if (cap != pipe->gb_cap || reps != pipe->gb_reps) {
    cudaFree(pipe->gb_keys);
    cudaFree(pipe->gb_slots);
    cudaFree(pipe->gb_rep_keys);
    cudaFree(pipe->gb_rep_slots);
    pipe->gb_keys = pipe->gb_slots = pipe->gb_rep_keys = pipe->gb_rep_slots = nullptr;
    pipe->gb_cap = 0;
    pipe->gb_reps = 1;
    cudaError_t e = cudaMalloc(&pipe->gb_keys, sizeof(uint64_t) * kw * (cap + 1));
    if (e == cudaSuccess) e = cudaMalloc(&pipe->gb_slots, sizeof(uint64_t) * (cap + 1) * G);
    if (e == cudaSuccess && reps > 1) e = cudaMalloc(&pipe->gb_rep_keys, sizeof(uint64_t) * kw * (cap + 1) * (reps - 1));
    if (e == cudaSuccess && reps > 1) e = cudaMalloc(&pipe->gb_rep_slots, sizeof(uint64_t) * (cap + 1) * G * (reps - 1));
    if (e != cudaSuccess) {
      cudaFree(pipe->gb_keys);
      cudaFree(pipe->gb_slots);
      cudaFree(pipe->gb_rep_keys);
      cudaFree(pipe->gb_rep_slots);
      pipe->gb_keys = pipe->gb_slots = pipe->gb_rep_keys = pipe->gb_rep_slots = nullptr;
      return set_err(FQ_ERR_CUDA, "CUDA error: %s (GROUP BY table of %" PRIu64 " slots)", cudaGetErrorString(e), cap);
    }
    pipe->gb_cap = cap;
    pipe->gb_reps = reps;
    pipe->gb_reps_dirty = true;
  }
  if (!pipe->gb_flags) {
    CUDA_TRY(cudaMalloc(&pipe->gb_flags, 64));
    CUDA_TRY(cudaHostAlloc(&pipe->h_gb, 64, cudaHostAllocDefault));
  }
  if (!pipe->gb_identity) {
    const std::vector<uint64_t> idn = gb_identity(pipe->gen);
    CUDA_TRY(cudaMalloc(&pipe->gb_identity, sizeof(uint64_t) * idn.size()));
    CUDA_TRY(cudaMemcpy(pipe->gb_identity, idn.data(), sizeof(uint64_t) * idn.size(), cudaMemcpyHostToDevice));
  }
  // a new seed for every table after the first: keys whose hashes clustered in the last one (fq_gb_hash is a bijection)
  // are spread again, while a pipe's first table hashes the keys themselves
  pipe->gb_seed = pipe->gb_reservations++ ? splitmix64(pipe->gb_reservations) : 0;
  if (fq_status st = gb_clear(ctx, pipe, nullptr)) return st;
  CUDA_TRY(cudaDeviceSynchronize());
  return FQ_OK;
}

static fq_status gb_after_launch(fq_ctx *ctx, fq_pipe *pipe, cudaStream_t s) {
  // count the groups, mirror {overflow, count, error bits} to the host
  CUDA_TRY(cudaMemsetAsync(pipe->gb_flags + 2, 0, 8, s));
  const unsigned grid = (unsigned)std::min<uint64_t>((pipe->gb_cap + 256) / 256, (uint64_t)ctx->sm_count * 8);
  fq_gb_count<<<grid, 256, 0, s>>>((const fq_u64 *)pipe->gb_keys, pipe->gen.key_words, pipe->gb_cap, (fq_u32 *)pipe->gb_flags);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  CUDA_TRY(cudaMemcpyAsync(pipe->h_gb, pipe->gb_flags, 32, cudaMemcpyDeviceToHost, s));
  if (fq_status st = mark_done(ctx, pipe->ev, s)) return st;
  pipe->launched_groupby = true;
  return FQ_OK;
}

fq_status fq_pipe_launch_groupby(fq_ctx *ctx, fq_pipe *pipe, const fq_source *src, uint32_t flags, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (fq_status st = gb_check(pipe)) return st;
  if (!pipe->gb_cap) return set_err(FQ_ERR_INVALID, "Internal Error: fq_pipe_groupby_reserve was not called");
  if (!(flags & FQ_RUN_ACCUMULATE) && pipe->launched_groupby) {
    if (fq_status st = gb_clear(ctx, pipe, (cudaStream_t)stream)) return st;   // restart from an empty table
  }
  fq_launch_params p;
  memset(&p, 0, sizeof p);
  if (fq_status st = bind_source(pipe, src, &p)) return st;
  p.gb_keys = (fq_u64 *)pipe->gb_keys;
  p.gb_slots = (fq_u64 *)pipe->gb_slots;
  p.gb_cap = pipe->gb_cap;
  p.gb_flags = (fq_u32 *)pipe->gb_flags;
  p.gb_smem_cap = pipe->gb_smem_cap;
  p.gb_rep_keys = (fq_u64 *)pipe->gb_rep_keys;
  p.gb_rep_slots = (fq_u64 *)pipe->gb_rep_slots;
  p.gb_reps = pipe->gb_reps;
  p.gb_seed = pipe->gb_seed;
  p.result = (fq_u64 *)(pipe->gb_flags + 2);   // [0] = count (u64 at flags[2..3]), [1] = error bits (flags[4..5])
  const Kernel &k = pipe->k[K_GROUPBY];
  if (!k.valid()) return set_err(FQ_ERR_INTERNAL, "Internal Error: no GROUP BY kernel was built for this pipe");
  if (src->n_rows > 0) {
    const unsigned grid = persistent_grid(ctx, k, src->n_rows);
    if (grid < p.gb_reps) p.gb_reps = 1;   // a small scan: every CTA on the table itself, nothing to fold
    if (fq_status st = launch(ctx, k, grid, p, stream)) return st;
    if (p.gb_reps > 1) {
      // fold the replicas into the table (and leave them empty): the merge kernel without an entry list
      const Kernel &km = pipe->k[K_GBMERGE];
      if (!km.valid()) return set_err(FQ_ERR_INTERNAL, "Internal Error: no GROUP BY merge kernel was built for this pipe");
      fq_launch_params q = p;
      q.n_rows = (pipe->gb_cap + 1) * (uint64_t)(pipe->gb_reps - 1);
      q.gb_entries = nullptr;
      const unsigned g2 = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((q.n_rows + 255) / 256, (uint64_t)ctx->sm_count * 8));
      if (fq_status st = launch(ctx, km, g2, q, stream)) return st;
    }
  }
  return gb_after_launch(ctx, pipe, (cudaStream_t)stream);
}

fq_status fq_pipe_fetch_groupby(fq_ctx *ctx, fq_pipe *pipe, uint64_t *n_groups) {
  if (fq_status st = use(ctx)) return st;
  if (fq_status st = gb_check(pipe)) return st;
  if (!pipe->launched_groupby) return set_err(FQ_ERR_INVALID, "Internal Error: no GROUP BY launch to fetch");
  CUDA_TRY(cudaEventSynchronize(pipe->ev));
  const uint32_t *f = (const uint32_t *)pipe->h_gb;
  if (n_groups) *n_groups = pipe->h_gb[1];
  if (f[0]) return set_err(FQ_ERR_CAPACITY, "Internal Error: GROUP BY met more groups than the %" PRIu64 " reserved: reserve more and relaunch", pipe->gb_cap / 2);
  return decode_err(pipe->h_gb[2]);
}

fq_status fq_pipe_export_groups(fq_ctx *ctx, fq_pipe *pipe, fq_column *const *key_cols, fq_column *const *key_valid,
                                fq_column *const *leaf_cols, fq_column *const *leaf_valid, uint64_t capacity, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (fq_status st = gb_check(pipe)) return st;
  if (!pipe->gb_cap) return set_err(FQ_ERR_INVALID, "Internal Error: fq_pipe_groupby_reserve was not called");
  const fq::Generated &gen = pipe->gen;
  fq_gb_export_params a;
  memset(&a, 0, sizeof a);
  a.keys = (const fq_u64 *)pipe->gb_keys;
  a.slots = (const fq_u64 *)pipe->gb_slots;
  a.cap = pipe->gb_cap;
  a.flags = (const fq_u32 *)pipe->gb_flags;
  a.kw = gen.key_words;
  a.G = 1 + gen.n_slots;
  a.n_keys = (int)gen.key_dtypes.size();
  a.n_leaves = (int)gen.agg_nodes.size();
  if (a.n_leaves > 16) return set_err(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: more than 16 aggregates in a GROUP BY");
  for (int j = 0; j < a.n_keys; j++) {
    const fq_column *c = key_cols ? key_cols[j] : nullptr;
    if (!c || c->dtype != gen.key_dtypes[j] || c->len < capacity) return set_err(FQ_ERR_INVALID, "Internal Error: key output column %d missing, mistyped or short", j);
    a.key_out[j] = c->ptr;
    a.key_shift[j] = gen.key_shift[j];
    a.key_bits[j] = gen.key_bits[j];
    a.key_nullable[j] = gen.key_nullable[j];
    if (gen.key_nullable[j]) {
      const fq_column *v = key_valid ? key_valid[j] : nullptr;
      if (!v || v->dtype != FQ_BOOL || v->len < capacity) return set_err(FQ_ERR_INVALID, "Internal Error: key %d can be NULL: a Boolean validity output column is required", j);
      a.key_valid[j] = v->ptr;
    }
  }
  for (int l = 0; l < a.n_leaves; l++) {
    const fq_column *c = leaf_cols ? leaf_cols[l] : nullptr;
    if (!c || c->dtype != gen.agg_dtypes[l] || c->len < capacity) return set_err(FQ_ERR_INVALID, "Internal Error: leaf output column %d missing, mistyped or short", l);
    a.leaf_out[l] = c->ptr;
    a.leaf_op[l] = gen.agg_ops[l];
    a.leaf_dtype[l] = gen.agg_dtypes[l];
    a.leaf_count_slot[l] = gen.agg_count_slot[l];
    if (gen.agg_count_slot[l] >= 0) {
      const fq_column *v = leaf_valid ? leaf_valid[l] : nullptr;
      if (!v || v->dtype != FQ_BOOL || v->len < capacity) return set_err(FQ_ERR_INVALID, "Internal Error: aggregate %d can be NULL: a Boolean validity output column is required", l);
      a.leaf_valid[l] = v->ptr;
    }
  }
  a.capacity = capacity;
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(cudaMemsetAsync(pipe->gb_flags + 6, 0, 8, s));
  a.counter = (fq_u64 *)(pipe->gb_flags + 6);
  const unsigned grid = (unsigned)std::min<uint64_t>((pipe->gb_cap + 256) / 256, (uint64_t)ctx->sm_count * 8);
  fq_gb_export<<<grid, 256, 0, s>>>(a);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  return FQ_OK;
}

fq_status fq_pipe_export_partials(fq_ctx *ctx, fq_pipe *pipe, int32_t world, fq_column *entries, uint64_t *counts, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (fq_status st = gb_check(pipe)) return st;
  if (world < 1 || world > 8 || !counts) return set_err(FQ_ERR_INVALID, "Internal Error: 1..8 ranks and a counts array");
  if (!pipe->launched_groupby) return set_err(FQ_ERR_INVALID, "Internal Error: no GROUP BY launch to export");
  CUDA_TRY(cudaEventSynchronize(pipe->ev));
  const uint64_t n_groups = pipe->h_gb[1];
  const int G = 1 + pipe->gen.n_slots, kw = pipe->gen.key_words;
  if (!entries || entries->dtype != FQ_U64 || entries->len < n_groups * (uint64_t)(kw + G))
    return set_err(FQ_ERR_INVALID, "Internal Error: the entries column must be UInt64 with groups x %d rows", kw + G);
  cudaStream_t s = (cudaStream_t)stream;
  unsigned long long *cursor = nullptr;
  CUDA_TRY(cudaMalloc(&cursor, 16 * sizeof(unsigned long long)));
  CUDA_TRY(cudaMemsetAsync(cursor, 0, 16 * sizeof(unsigned long long), s));
  const unsigned grid = (unsigned)std::min<uint64_t>((pipe->gb_cap + 256) / 256, (uint64_t)ctx->sm_count * 8);
  fq_gb_partials<<<grid, 256, 0, s>>>((const fq_u64 *)pipe->gb_keys, kw, (const fq_u64 *)pipe->gb_slots, pipe->gb_cap, (const fq_u32 *)pipe->gb_flags, G,
                                      world, cursor, nullptr, 0);
  fq_gb_prefix<<<1, 1, 0, s>>>(cursor, cursor + 8, world);
  fq_gb_partials<<<grid, 256, 0, s>>>((const fq_u64 *)pipe->gb_keys, kw, (const fq_u64 *)pipe->gb_slots, pipe->gb_cap, (const fq_u32 *)pipe->gb_flags, G,
                                      world, cursor, (fq_u64 *)entries->ptr, 1);
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 3;
  unsigned long long h[8];
  CUDA_TRY(cudaMemcpyAsync(h, cursor + 8, sizeof h, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  cudaFree(cursor);
  for (int d = 0; d < world; d++) counts[d] = h[d];
  return FQ_OK;
}

fq_status fq_pipe_merge_partials(fq_ctx *ctx, fq_pipe *pipe, const fq_column *entries, uint64_t n_entries, uint32_t flags, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (fq_status st = gb_check(pipe)) return st;
  if (!pipe->gb_cap) return set_err(FQ_ERR_INVALID, "Internal Error: fq_pipe_groupby_reserve was not called");
  const int G = 1 + pipe->gen.n_slots, kw = pipe->gen.key_words;
  if (n_entries && (!entries || entries->dtype != FQ_U64 || entries->len < n_entries * (uint64_t)(kw + G)))
    return set_err(FQ_ERR_INVALID, "Internal Error: the entries column must be UInt64 with entries x %d rows", kw + G);
  if (!(flags & FQ_RUN_ACCUMULATE) && pipe->launched_groupby) {
    if (fq_status st = gb_clear(ctx, pipe, (cudaStream_t)stream)) return st;
  }
  if (n_entries) {
    fq_launch_params p;
    memset(&p, 0, sizeof p);
    p.n_rows = n_entries;
    p.gb_keys = (fq_u64 *)pipe->gb_keys;
    p.gb_slots = (fq_u64 *)pipe->gb_slots;
    p.gb_cap = pipe->gb_cap;
    p.gb_flags = (fq_u32 *)pipe->gb_flags;
    p.gb_seed = pipe->gb_seed;
    p.gb_entries = (const fq_u64 *)entries->ptr;
    const Kernel &k = pipe->k[K_GBMERGE];
    if (!k.valid()) return set_err(FQ_ERR_INTERNAL, "Internal Error: no GROUP BY merge kernel was built for this pipe");
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n_entries + 255) / 256, (uint64_t)ctx->sm_count * 8));
    if (fq_status st = launch(ctx, k, grid, p, stream)) return st;
  }
  return gb_after_launch(ctx, pipe, (cudaStream_t)stream);
}

// ---- ORDER BY: stable radix sort of row indexes, and the gather that applies them (kernels/fq_sort.cuh) ----
namespace {
// exclusive scan of m u32 counters in place; `sums` holds ceil(m / FQ_SCAN_TILE) scratch words
fq_status sort_scan(fq_ctx *ctx, fq_u32 *a, uint64_t m, fq_u32 *sums, cudaStream_t s) {
  const unsigned nb = (unsigned)((m + FQ_SCAN_TILE - 1) / FQ_SCAN_TILE);
  fq_scan_tile_sums<<<nb, FQ_SCAN_THREADS, 0, s>>>(a, m, sums);
  fq_scan_sums<<<1, FQ_SCAN_THREADS, 0, s>>>(sums, nb);
  fq_scan_tiles<<<nb, FQ_SCAN_THREADS, 0, s>>>(a, m, sums);
  CUDA_TRY(cudaGetLastError());
  ctx->launches += 3;
  return FQ_OK;
}
}  // namespace

namespace {
// One ORDER BY over the context's scratch (held under ctx->sort_mu by the caller): (code, row) pairs in code[cur] / idx[cur].
struct SortJob {
  fq_ctx *ctx;
  cudaStream_t s;
  fq_u64 *code[2] = {nullptr, nullptr}, *and_or = nullptr;
  fq_u32 *idx[2] = {nullptr, nullptr}, *hist = nullptr, *sums = nullptr, *small = nullptr;   // small: 256 + 2 counters (radix select)
  int cur = 0;

  // scratch for n rows: two (code, row) buffers, the (digit, tile) counters, the scan's tile sums, a few words
  fq_status acquire(uint64_t n) {
    const uint64_t n_tiles = (n + FQ_SORT_TILE - 1) / FQ_SORT_TILE, hist_len = 256 * n_tiles;
    const uint64_t scan_blocks = (hist_len + FQ_SCAN_TILE - 1) / FQ_SCAN_TILE;
    auto up = [](uint64_t b) { return (b + 255) & ~255ull; };
    const uint64_t need = 2 * up(8 * n) + 2 * up(4 * n) + up(4 * hist_len) + up(4 * scan_blocks) + 256 + 2048;
    if (!ctx->sort_done) CUDA_TRY(cudaEventCreateWithFlags(&ctx->sort_done, cudaEventDisableTiming));
    if (need > ctx->sort_scratch_bytes) {
      cudaFree(ctx->sort_scratch);   // (synchronises the device: nothing still reads the old buffer)
      ctx->sort_scratch = nullptr;
      ctx->sort_scratch_bytes = 0;
      cudaError_t e = cudaMalloc(&ctx->sort_scratch, need);
      if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(FQ_ERR_CUDA, "CUDA error: %s (sort scratch of %" PRIu64 " bytes for %" PRIu64 " rows)", cudaGetErrorString(e), need, n);
      }
      ctx->sort_scratch_bytes = need;
    } else {
      CUDA_TRY(cudaStreamWaitEvent(s, ctx->sort_done, 0));   // an earlier sort on another stream may still be copying its result out
    }
    char *at = (char *)ctx->sort_scratch;
    auto carve = [&](uint64_t b) { char *p = at; at += up(b); return p; };
    code[0] = (fq_u64 *)carve(8 * n);
    code[1] = (fq_u64 *)carve(8 * n);
    idx[0] = (fq_u32 *)carve(4 * n);
    idx[1] = (fq_u32 *)carve(4 * n);
    hist = (fq_u32 *)carve(4 * hist_len);
    sums = (fq_u32 *)carve(4 * scan_blocks);
    and_or = (fq_u64 *)carve(16);
    small = (fq_u32 *)carve(2048);
    CUDA_TRY(cudaFuncSetAttribute(fq_sort_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, FQ_SORT_SMEM));   // per device: not cached
    return FQ_OK;
  }

  // one stable pass over digit d of the first m pairs
  fq_status radix_pass(uint64_t m, int d) {
    const unsigned n_tiles = (unsigned)((m + FQ_SORT_TILE - 1) / FQ_SORT_TILE);
    fq_sort_hist<<<n_tiles, FQ_SORT_THREADS, 0, s>>>(code[cur], m, n_tiles, 8 * d, hist);
    ctx->launches++;
    if (fq_status st = sort_scan(ctx, hist, 256ull * n_tiles, sums, s)) return st;
    fq_sort_scatter<<<n_tiles, FQ_SORT_THREADS, FQ_SORT_SMEM, s>>>(code[cur], idx[cur], code[cur ^ 1], idx[cur ^ 1], hist, m, n_tiles, 8 * d);
    CUDA_TRY(cudaGetLastError());
    ctx->launches++;
    cur ^= 1;
    return FQ_OK;
  }

  // codes of one key (phase 0: values, phase 1: the NULLs-first flag) for the first m pairs, through idx[cur] when have_perm;
  // *varying = the bits that differ between some two codes
  fq_status encode(const fq_column *k, bool desc, int phase, bool have_perm, uint64_t m, uint64_t *varying) {
    static const uint64_t init[2] = {~0ull, 0ull};
    CUDA_TRY(cudaMemcpyAsync(and_or, init, 16, cudaMemcpyHostToDevice, s));
    fq_sort_encode_params a;
    memset(&a, 0, sizeof a);
    a.col = k->ptr;
    a.valid_bytes = k->validity ? (const fq_u8 *)k->validity->ptr : nullptr;
    a.valid_bits = (!k->validity && k->validity_bits) ? k->validity_bits->ptr : nullptr;
    a.valid_bit0 = k->validity_bit0;
    a.perm = have_perm ? idx[cur] : nullptr;
    a.code_out = code[cur];
    a.idx_out = idx[cur];
    a.and_or = and_or;
    a.n = m;
    a.dtype = (int)k->dtype;
    a.bits = 8 * (int)fq::dtype_size(k->dtype);
    a.descending = desc ? 1 : 0;
    a.flags_only = phase;
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((m + 255) / 256, (uint64_t)ctx->sm_count * 8));
    fq_sort_encode<<<grid, 256, 0, s>>>(a);
    CUDA_TRY(cudaGetLastError());
    ctx->launches++;
    uint64_t h[2];
    CUDA_TRY(cudaMemcpyAsync(h, and_or, 16, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    *varying = h[0] ^ h[1];
    return FQ_OK;
  }

  // one stable sort per key, last key first; inside a key: its value digits, then (nullable keys) the NULLs-first bit
  fq_status sort_by_keys(const fq_column *const *keys, const uint8_t *descending, int n_keys, uint64_t m, bool have_perm) {
    for (int j = n_keys - 1; j >= 0; j--) {
      const fq_column *k = keys[j];
      const bool nullable = k->validity || k->validity_bits;
      for (int phase = 0; phase < (nullable ? 2 : 1); phase++) {
        uint64_t varying = 0;
        if (fq_status st = encode(k, descending && descending[j], phase, have_perm, m, &varying)) return st;
        have_perm = true;
        const int digits = phase ? 1 : (int)fq::dtype_size(k->dtype);
        for (int d = 0; d < digits; d++) {
          if (((varying >> (8 * d)) & 255) == 0) continue;   // every row has the same digit: the pass would be the identity
          if (fq_status st = radix_pass(m, d)) return st;
        }
      }
    }
    return FQ_OK;
  }

  fq_status finish(fq_column *indices, uint64_t count) {
    if (count) CUDA_TRY(cudaMemcpyAsync(indices->ptr, idx[cur], 4 * count, cudaMemcpyDeviceToDevice, s));
    CUDA_TRY(cudaEventRecord(ctx->sort_done, s));
    return FQ_OK;
  }

  // ORDER BY one NOT NULL key LIMIT `limit` (limit < n): radix select, then a sort of what is left
  fq_status top_k(const fq_column *key, bool desc, uint64_t n, uint64_t limit, fq_column *indices) {
    uint64_t varying = 0;
    if (fq_status st = encode(key, desc, 0, false, n, &varying)) return st;   // code[cur] = codes, idx[cur] = 0 .. n-1
    if (varying == 0) return finish(indices, limit);   // every key is the same: the first rows, in input order
    uint64_t m = n, need = limit, winners = 0;
    fq_u32 *win = (fq_u32 *)indices->ptr;   // winners collect in the result column (fewer than `limit` of them), unordered
    for (int d = (int)fq::dtype_size(key->dtype) - 1; d >= 0; d--) {
      if (((varying >> (8 * d)) & 255) == 0) continue;
      if (m <= std::max<uint64_t>(4 * need, 1ull << 16)) break;   // small enough to sort
      CUDA_TRY(cudaMemsetAsync(small, 0, 4 * 258, s));
      const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((m + 255) / 256, (uint64_t)ctx->sm_count * 8));
      fq_topk_hist<<<grid, 256, 0, s>>>(code[cur], m, 8 * d, small);
      CUDA_TRY(cudaGetLastError());
      ctx->launches++;
      uint32_t h[256];
      CUDA_TRY(cudaMemcpyAsync(h, small, sizeof h, cudaMemcpyDeviceToHost, s));
      CUDA_TRY(cudaStreamSynchronize(s));
      uint64_t below = 0;
      unsigned bucket = 0;
      for (; bucket < 255 && below + h[bucket] < need; bucket++) below += h[bucket];   // the bucket that holds the need-th smallest
      fq_topk_partition<<<grid, 256, 0, s>>>(code[cur], idx[cur], m, 8 * d, bucket, win + winners, code[cur ^ 1], idx[cur ^ 1], small + 256);
      CUDA_TRY(cudaGetLastError());
      ctx->launches++;
      winners += below;
      need -= below;
      m = h[bucket];
      cur ^= 1;
    }
    // what is left: the winners and the last candidates, first in input order, then (stable) by key
    if (winners) CUDA_TRY(cudaMemcpyAsync(idx[cur] + m, win, 4 * winners, cudaMemcpyDeviceToDevice, s));
    const uint64_t t = m + winners;
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((t + 255) / 256, (uint64_t)ctx->sm_count * 8));
    fq_sort_rows_as_codes<<<grid, 256, 0, s>>>(idx[cur], code[cur], t);
    CUDA_TRY(cudaGetLastError());
    ctx->launches++;
    for (int d = 0; d < 4; d++)
      if (((n - 1) >> (8 * d)) != 0)
        if (fq_status st = radix_pass(t, d)) return st;
    const uint8_t dflag = desc ? 1 : 0;
    if (fq_status st = sort_by_keys(&key, &dflag, 1, t, true)) return st;
    return finish(indices, std::min(limit, t));
  }
};

fq_status sort_check(fq_ctx *ctx, const fq_column *const *keys, int32_t n_keys, uint64_t n_rows, uint64_t slots, const fq_column *indices) {
  if (!keys || n_keys < 1 || !indices) return set_err(FQ_ERR_INVALID, "Internal Error: sort needs at least one key column and an index column");
  if (indices->dtype != FQ_U32 || indices->len < slots) return set_err(FQ_ERR_INVALID, "Internal Error: the index column must be UInt32 with a slot per result row");
  if (n_rows >= (1ull << 32)) return set_err(FQ_ERR_INVALID, "Internal Error: sort handles fewer than 2^32 rows per call");
  if (ctx->recording) return set_err(FQ_ERR_INVALID, "Internal Error: a sort cannot be recorded into a graph (its passes depend on the data)");
  for (int j = 0; j < n_keys; j++) {
    if (!keys[j] || keys[j]->len < n_rows) return set_err(FQ_ERR_INVALID, "Internal Error: sort key %d is shorter than n_rows", j);
    if (keys[j]->dtype == FQ_NULL || keys[j]->dtype == FQ_UTF8) return set_err(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: sort key of type %s", fq::dtype_name(keys[j]->dtype));
  }
  return FQ_OK;
}
}  // namespace

fq_status fq_sort_indices(fq_ctx *ctx, const fq_column *const *keys, const uint8_t *descending, int32_t n_keys, uint64_t n_rows,
                          fq_column *indices, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (fq_status st = sort_check(ctx, keys, n_keys, n_rows, n_rows, indices)) return st;
  if (n_rows == 0) return FQ_OK;
  std::lock_guard<std::mutex> sort_lock(ctx->sort_mu);
  SortJob job{ctx, (cudaStream_t)stream};
  if (fq_status st = job.acquire(n_rows)) return st;
  if (fq_status st = job.sort_by_keys(keys, descending, n_keys, n_rows, false)) return st;
  return job.finish(indices, n_rows);
}

fq_status fq_sort_indices_limit(fq_ctx *ctx, const fq_column *const *keys, const uint8_t *descending, int32_t n_keys, uint64_t n_rows,
                                uint64_t limit, fq_column *indices, uint64_t *n_out, void *stream) {
  if (fq_status st = use(ctx)) return st;
  const uint64_t count = std::min(limit, n_rows);
  if (fq_status st = sort_check(ctx, keys, n_keys, n_rows, count, indices)) return st;
  if (n_out) *n_out = count;
  if (count == 0) return FQ_OK;
  std::lock_guard<std::mutex> sort_lock(ctx->sort_mu);
  SortJob job{ctx, (cudaStream_t)stream};
  if (fq_status st = job.acquire(n_rows)) return st;
  // radix select pays when the result is a small part of the table and the order is decided by one NOT NULL key
  const bool select = n_keys == 1 && !keys[0]->validity && !keys[0]->validity_bits && limit < n_rows / 64 && n_rows >= (1ull << 20);
  if (select) return job.top_k(keys[0], descending && descending[0], n_rows, limit, indices);
  if (fq_status st = job.sort_by_keys(keys, descending, n_keys, n_rows, false)) return st;
  return job.finish(indices, count);
}

fq_status fq_column_take(fq_ctx *ctx, const fq_column *src, const fq_column *rows, uint64_t n, fq_column *out, fq_column *out_valid,
                         void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!src || !rows || !out) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (rows->dtype != FQ_U32 || rows->len < n) return set_err(FQ_ERR_INVALID, "Internal Error: row indexes must be a UInt32 column with at least n slots");
  if (out->dtype != src->dtype || out->len < n) return set_err(FQ_ERR_INVALID, "Internal Error: the output column must have the source's type and at least n slots");
  const bool nullable = src->validity || src->validity_bits;
  if (nullable && (!out_valid || out_valid->dtype != FQ_BOOL || out_valid->len < n))
    return set_err(FQ_ERR_INVALID, "Internal Error: the source has validity: a Boolean output validity column is required");
  if (n == 0) return FQ_OK;
  fq_take_params a;
  memset(&a, 0, sizeof a);
  a.src = src->ptr;
  a.out = out->ptr;
  a.rows = (const fq_u32 *)rows->ptr;
  a.n = n;
  a.width = (int)fq::dtype_size(src->dtype);
  a.valid_bytes = src->validity ? (const fq_u8 *)src->validity->ptr : nullptr;
  a.valid_bits = (!src->validity && src->validity_bits) ? src->validity_bits->ptr : nullptr;
  a.valid_bit0 = src->validity_bit0;
  a.out_valid = out_valid ? (fq_u8 *)out_valid->ptr : nullptr;
  const unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * 16);
  fq_take_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  return FQ_OK;
}

// ---- recorded launches (CUDA graph) ----
fq_status fq_graph_begin(fq_ctx *ctx, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (ctx->recording) return set_err(FQ_ERR_INVALID, "Internal Error: a graph is already being recorded on this context");
  if (!stream) return set_err(FQ_ERR_INVALID, "Internal Error: a graph is recorded on an explicit stream, not the default stream");
  // relaxed mode: a pipe may grow a scratch buffer (cudaMalloc) on its first launch inside the recording
  CUDA_TRY(cudaStreamBeginCapture((cudaStream_t)stream, cudaStreamCaptureModeRelaxed));
  ctx->recording = new fq_graph();
  ctx->recording_stream = (cudaStream_t)stream;
  ctx->recording_launches0 = ctx->launches.load();
  return FQ_OK;
}

fq_status fq_graph_end(fq_ctx *ctx, void *stream, fq_graph **out) {
  if (fq_status st = use(ctx)) return st;
  if (!ctx->recording || (cudaStream_t)stream != ctx->recording_stream || !out)
    return set_err(FQ_ERR_INVALID, "Internal Error: fq_graph_end without a matching fq_graph_begin on this stream");
  fq_graph *g = ctx->recording;
  ctx->recording = nullptr;
  ctx->recording_stream = nullptr;
  g->launches = ctx->launches.load() - ctx->recording_launches0;
  ctx->launches -= g->launches;   // nothing ran yet
  cudaError_t e = cudaStreamEndCapture((cudaStream_t)stream, &g->graph);
  if (e == cudaSuccess) e = cudaGraphInstantiate(&g->exec, g->graph, 0);
  if (e != cudaSuccess) {
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
    cudaGetLastError();
    return set_err(FQ_ERR_CUDA, "CUDA error: %s (recording a graph)", cudaGetErrorString(e));
  }
  *out = g;
  return FQ_OK;
}

fq_status fq_graph_launch(fq_ctx *ctx, fq_graph *graph, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!graph || !graph->exec) return set_err(FQ_ERR_INVALID, "Internal Error: null graph");
  if (ctx->recording) return set_err(FQ_ERR_INVALID, "Internal Error: a graph cannot be launched while another is being recorded");
  CUDA_TRY(cudaGraphLaunch(graph->exec, (cudaStream_t)stream));
  for (cudaEvent_t ev : graph->done) CUDA_TRY(cudaEventRecord(ev, (cudaStream_t)stream));
  ctx->launches += graph->launches;
  return FQ_OK;
}

void fq_graph_destroy(fq_ctx *ctx, fq_graph *graph) {
  if (!graph) return;
  if (ctx) cudaSetDevice(ctx->device);
  if (graph->exec) cudaGraphExecDestroy(graph->exec);
  if (graph->graph) cudaGraphDestroy(graph->graph);
  delete graph;
}

}  // extern "C"

// =============================================================================================
// Utf8 arrays
// =============================================================================================
struct fq_utf8 {
  uint64_t len = 0;
  int32_t *offsets = nullptr;   // device, len + 1
  unsigned char *data = nullptr;
  uint64_t bytes = 0;           // offsets[len]
  const fq_column *validity = nullptr;
};

namespace {
__device__ __forceinline__ bool fq_cmp_holds(int op, int c) {
  switch (op) {
    case FQ_CMP_EQ: return c == 0;
    case FQ_CMP_LT: return c < 0;
    case FQ_CMP_LTEQ: return c <= 0;
    case FQ_CMP_GT: return c > 0;
    default: return c >= 0;
  }
}
__global__ void __launch_bounds__(256) fq_utf8_compare_kernel(int op, const int32_t *lo, const unsigned char *ld, const fq_u8 *lv, const int32_t *ro,
                                                             const unsigned char *rd, const fq_u8 *rv, fq_u32 scalar_len, fq_u64 n, fq_u8 *out,
                                                             fq_u8 *out_valid) {
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (fq_u64)gridDim.x * blockDim.x) {
    const unsigned char *a = ld + lo[i];
    const fq_u32 la = (fq_u32)(lo[i + 1] - lo[i]);
    const unsigned char *b = ro ? rd + ro[i] : rd;       // ro == null: the right side is one scalar
    const fq_u32 lb = ro ? (fq_u32)(ro[i + 1] - ro[i]) : scalar_len;
    const bool ok = (!lv || lv[i]) && (!rv || rv[i]);
    out[i] = (ok && fq_cmp_holds(op, fq_utf8_cmp(a, la, b, lb))) ? 1 : 0;
    if (out_valid) out_valid[i] = ok ? 1 : 0;
  }
}
// better(i, j): does row i beat row j for op?  ties keep the smaller row index (first occurrence)
__device__ __forceinline__ long long fq_utf8_pick(int op, const int32_t *o, const unsigned char *d, long long i, long long j) {
  if (i < 0) return j;
  if (j < 0) return i;
  const int c = fq_utf8_cmp(d + o[i], (fq_u32)(o[i + 1] - o[i]), d + o[j], (fq_u32)(o[j + 1] - o[j]));
  const bool i_wins = op == FQ_AGG_MIN ? (c < 0 || (c == 0 && i < j)) : (c > 0 || (c == 0 && i < j));
  return i_wins ? i : j;
}
__global__ void __launch_bounds__(256) fq_utf8_minmax_kernel(int op, const int32_t *o, const unsigned char *d, const fq_u8 *valid, fq_u64 n,
                                                            long long *partials, fq_u32 *ticket, long long *result) {
  __shared__ long long s_best[256];
  __shared__ fq_u32 s_last;
  long long best = -1;
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (fq_u64)gridDim.x * blockDim.x)
    if (!valid || valid[i]) best = fq_utf8_pick(op, o, d, best, (long long)i);
  s_best[threadIdx.x] = best;
  __syncthreads();
  for (int m = 128; m > 0; m >>= 1) {
    if ((int)threadIdx.x < m) s_best[threadIdx.x] = fq_utf8_pick(op, o, d, s_best[threadIdx.x], s_best[threadIdx.x + m]);
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = s_best[0];
    __threadfence();
    s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1u : 0u;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  best = -1;
  for (fq_u32 b = threadIdx.x; b < gridDim.x; b += blockDim.x) best = fq_utf8_pick(op, o, d, best, *(volatile long long *)(partials + b));
  s_best[threadIdx.x] = best;
  __syncthreads();
  for (int m = 128; m > 0; m >>= 1) {
    if ((int)threadIdx.x < m) s_best[threadIdx.x] = fq_utf8_pick(op, o, d, s_best[threadIdx.x], s_best[threadIdx.x + m]);
    __syncthreads();
  }
  if (threadIdx.x == 0) { *result = s_best[0]; *ticket = 0; }
}
}  // namespace

extern "C" {

fq_status fq_utf8_create(fq_ctx *ctx, const int32_t *offsets, const void *data, uint64_t len, const fq_column *validity, void *stream,
                         fq_utf8 **out) {
  if (fq_status st = use(ctx)) return st;
  if (!out || (len && !offsets)) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  *out = nullptr;
  const uint64_t bytes = len ? (uint64_t)offsets[len] - (uint64_t)offsets[0] : 0;
  if (len && (offsets[0] != 0 || offsets[len] < 0)) return set_err(FQ_ERR_INVALID, "Internal Error: Utf8 offsets must start at 0 and stay within int32");
  if (validity && (validity->dtype != FQ_BOOL || validity->len < len)) return set_err(FQ_ERR_INVALID, "Internal Error: validity must be a Boolean column as long as the array");
  if (bytes && !data) return set_err(FQ_ERR_INVALID, "Internal Error: null value buffer");
  fq_utf8 *a = new fq_utf8();
  a->len = len;
  a->bytes = bytes;
  a->validity = validity;
  cudaError_t e = cudaMalloc(&a->offsets, sizeof(int32_t) * (len + 1));
  if (e == cudaSuccess) e = cudaMalloc(&a->data, bytes ? bytes : 1);
  static const int32_t zero = 0;
  if (e == cudaSuccess) e = cudaMemcpyAsync(a->offsets, len ? offsets : &zero, sizeof(int32_t) * (len + 1), cudaMemcpyHostToDevice, (cudaStream_t)stream);
  if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(a->data, data, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);   // the host buffers may go away after the call
  if (e != cudaSuccess) {
    fq_utf8_free(ctx, a);
    return set_err(FQ_ERR_CUDA, "CUDA error: %s (Utf8 array of %" PRIu64 " rows)", cudaGetErrorString(e), len);
  }
  *out = a;
  return FQ_OK;
}
void fq_utf8_free(fq_ctx *ctx, fq_utf8 *a) {
  if (!a) return;
  if (ctx) cudaSetDevice(ctx->device);
  cudaFree(a->offsets);
  cudaFree(a->data);
  delete a;
}
uint64_t fq_utf8_len(const fq_utf8 *a) { return a ? a->len : 0; }

static fq_status utf8_compare(fq_ctx *ctx, int32_t op, const fq_utf8 *l, const fq_utf8 *r, const unsigned char *scalar_dev, uint32_t scalar_len,
                              fq_column *out, fq_column *out_valid, void *stream) {
  if (op < FQ_CMP_EQ || op > FQ_CMP_GTEQ) return set_err(FQ_ERR_INVALID, "Internal Error: operator code %d out of range", op);
  if (!l || !out || out->dtype != FQ_BOOL || out->len < l->len) return set_err(FQ_ERR_INVALID, "Internal Error: a Boolean output column as long as the arrays is required");
  if (r && r->len != l->len) return set_err(FQ_ERR_INTERNAL, "Internal Error: Compute error: Cannot perform comparison operation on arrays of different length");
  const bool nullable = l->validity || (r && r->validity);
  if (nullable && (!out_valid || out_valid->dtype != FQ_BOOL || out_valid->len < l->len))
    return set_err(FQ_ERR_INVALID, "Internal Error: the operands carry validity: a Boolean validity output column is required");
  if (l->len == 0) return FQ_OK;
  const unsigned grid = (unsigned)std::min<uint64_t>((l->len + 255) / 256, (uint64_t)ctx->sm_count * 8);
  fq_utf8_compare_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(op, l->offsets, l->data, l->validity ? (const fq_u8 *)l->validity->ptr : nullptr,
                                                               r ? r->offsets : nullptr, r ? r->data : scalar_dev,
                                                               r && r->validity ? (const fq_u8 *)r->validity->ptr : nullptr, scalar_len, l->len,
                                                               (fq_u8 *)out->ptr, out_valid ? (fq_u8 *)out_valid->ptr : nullptr);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  return FQ_OK;
}
fq_status fq_utf8_compare(fq_ctx *ctx, int32_t op, const fq_utf8 *l, const fq_utf8 *r, fq_column *out, fq_column *out_valid, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!r) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  return utf8_compare(ctx, op, l, r, nullptr, 0, out, out_valid, stream);
}
fq_status fq_utf8_compare_scalar(fq_ctx *ctx, int32_t op, const fq_utf8 *l, const void *scalar, uint64_t scalar_len, fq_column *out,
                                 fq_column *out_valid, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (scalar_len && !scalar) return set_err(FQ_ERR_INVALID, "Internal Error: null scalar");
  unsigned char *dev = nullptr;
  CUDA_TRY(cudaMallocAsync((void **)&dev, scalar_len ? scalar_len : 1, (cudaStream_t)stream));
  if (scalar_len) CUDA_TRY(cudaMemcpyAsync(dev, scalar, scalar_len, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  const fq_status st = utf8_compare(ctx, op, l, nullptr, dev, (uint32_t)scalar_len, out, out_valid, stream);
  cudaFreeAsync(dev, (cudaStream_t)stream);
  if (st == FQ_OK) CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));   // `scalar` may go away after the call
  return st;
}
fq_status fq_utf8_minmax(fq_ctx *ctx, int32_t op, const fq_utf8 *a, int64_t *row, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!a || !row || (op != FQ_AGG_MIN && op != FQ_AGG_MAX)) return set_err(FQ_ERR_INVALID, "Internal Error: Min or Max over a Utf8 array");
  *row = -1;
  if (a->len == 0) return FQ_OK;
  const unsigned grid = (unsigned)std::min<uint64_t>((a->len + 255) / 256, (uint64_t)ctx->sm_count * 4);
  long long *scratch = nullptr;
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(cudaMallocAsync((void **)&scratch, sizeof(long long) * (grid + 2), s));
  CUDA_TRY(cudaMemsetAsync(scratch + grid, 0, sizeof(long long) * 2, s));
  fq_utf8_minmax_kernel<<<grid, 256, 0, s>>>(op, a->offsets, a->data, a->validity ? (const fq_u8 *)a->validity->ptr : nullptr, a->len, scratch,
                                            (fq_u32 *)(scratch + grid), scratch + grid + 1);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  long long h = -1;
  CUDA_TRY(cudaMemcpyAsync(&h, scratch + grid + 1, sizeof h, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  cudaFreeAsync(scratch, s);
  *row = h;
  return FQ_OK;
}

}  // extern "C"

// ---- dictionary encoding (kernels/fq_utf8.cuh) ----
namespace {
// device buffers of one call, given back in stream order whatever way the call ends
struct StreamScratch {
  cudaStream_t s;
  std::vector<void *> bufs;
  explicit StreamScratch(cudaStream_t st) : s(st) {}
  ~StreamScratch() {
    for (void *p : bufs) cudaFreeAsync(p, s);
  }
  template <class T>
  cudaError_t get(T **out, uint64_t bytes) {
    void *p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, bytes ? bytes : 1, s);
    if (e == cudaSuccess) bufs.push_back(p);
    *out = (T *)p;
    return e;
  }
};

unsigned grid_for(const fq_ctx *ctx, uint64_t n, uint64_t per_sm = 8) {
  return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * per_sm));
}

// strings rows[0 .. n) of `src` (NULL where rows_valid says so) as a new array; waits for the result
fq_status utf8_take(fq_ctx *ctx, const fq_utf8 *src, const fq_u32 *rows, uint64_t n, const fq_column *rows_valid, cudaStream_t s, fq_utf8 **out) {
  if (n >= 0xFFFFFFFFull) return set_err(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: a Utf8 array of 2^32 - 1 rows or more");
  StreamScratch scratch(s);
  fq_utf8 *a = new fq_utf8();
  a->len = n;
  a->validity = rows_valid;
  auto fail = [&](fq_status st) { fq_utf8_free(ctx, a); return st; };
  unsigned long long *total = nullptr;
  fq_u32 *sums = nullptr;
  cudaError_t e = cudaMalloc(&a->offsets, sizeof(int32_t) * (n + 1));
  if (e == cudaSuccess) e = scratch.get(&total, 16);
  if (e == cudaSuccess) e = scratch.get(&sums, 4 * ((n + 1 + FQ_SCAN_TILE - 1) / FQ_SCAN_TILE));
  if (e == cudaSuccess) e = cudaMemsetAsync(total, 0, 16, s);
  if (e != cudaSuccess) return fail(set_err(FQ_ERR_CUDA, "CUDA error: %s (Utf8 take of %" PRIu64 " rows)", cudaGetErrorString(e), n));
  const fq_u8 *rv = rows_valid ? (const fq_u8 *)rows_valid->ptr : nullptr;
  fq_utf8_lens<<<grid_for(ctx, n + 1), 256, 0, s>>>(src->offsets, src->len, rows, rv, n, (fq_u32 *)a->offsets, total);
  ctx->launches++;
  unsigned long long h[2] = {0, 0};
  e = cudaMemcpyAsync(h, total, 16, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return fail(set_err(FQ_ERR_CUDA, "CUDA error: %s (Utf8 take of %" PRIu64 " rows)", cudaGetErrorString(e), n));
  if (h[1]) return fail(set_err(FQ_ERR_INVALID, "Internal Error: a row index of the Utf8 take is out of range"));
  if (h[0] > (unsigned long long)INT32_MAX)
    return fail(set_err(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: a Utf8 array of more than 2 GiB of string bytes (%llu)", h[0]));
  if (fq_status st = sort_scan(ctx, (fq_u32 *)a->offsets, n + 1, sums, s)) return fail(st);
  a->bytes = h[0];
  e = cudaMalloc(&a->data, a->bytes ? a->bytes : 1);
  if (e != cudaSuccess) return fail(set_err(FQ_ERR_CUDA, "CUDA error: %s (Utf8 take of %llu bytes)", cudaGetErrorString(e), h[0]));
  if (n && a->bytes) {
    fq_utf8_gather_bytes<<<grid_for(ctx, 32 * n, 16), 256, 0, s>>>(src->offsets, src->data, rows, rv, n, a->offsets, a->data);
    ctx->launches++;
  }
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return fail(set_err(FQ_ERR_CUDA, "CUDA error: %s (Utf8 take of %" PRIu64 " rows)", cudaGetErrorString(e), n));
  *out = a;
  return FQ_OK;
}
}  // namespace

extern "C" {

uint64_t fq_utf8_bytes(const fq_utf8 *a) { return a ? a->bytes : 0; }

fq_status fq_utf8_download(fq_ctx *ctx, const fq_utf8 *a, int32_t *offsets_host, void *data_host, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!a || !offsets_host || (a->bytes && !data_host)) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  CUDA_TRY(cudaMemcpyAsync(offsets_host, a->offsets, sizeof(int32_t) * (a->len + 1), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  if (a->bytes) CUDA_TRY(cudaMemcpyAsync(data_host, a->data, a->bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return FQ_OK;
}

fq_status fq_utf8_take(fq_ctx *ctx, const fq_utf8 *src, const fq_column *rows, uint64_t n, const fq_column *rows_validity, fq_utf8 **out,
                       void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!src || !rows || !out) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  *out = nullptr;
  if (rows->dtype != FQ_U32 || rows->len < n) return set_err(FQ_ERR_INVALID, "Internal Error: row indexes must be a UInt32 column with at least n slots");
  if (rows_validity && (rows_validity->dtype != FQ_BOOL || rows_validity->len < n))
    return set_err(FQ_ERR_INVALID, "Internal Error: the validity of the row indexes must be a Boolean column with at least n slots");
  return utf8_take(ctx, src, (const fq_u32 *)rows->ptr, n, rows_validity, (cudaStream_t)stream, out);
}

fq_status fq_utf8_dict_encode(fq_ctx *ctx, const fq_utf8 *src, fq_column *codes, fq_utf8 **dict, void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!src || !codes || !dict) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  *dict = nullptr;
  const uint64_t n = src->len;
  if (codes->dtype != FQ_U32 || codes->len < n) return set_err(FQ_ERR_INVALID, "Internal Error: the codes column must be UInt32 with a slot per row");
  if (n >= 0xFFFFFFFFull) return set_err(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: dictionary encoding of 2^32 - 1 rows or more");
  if (ctx->recording) return set_err(FQ_ERR_INVALID, "Internal Error: dictionary encoding cannot be recorded into a graph (it depends on the data)");
  cudaStream_t s = (cudaStream_t)stream;
  const fq_u8 *valid = src->validity ? (const fq_u8 *)src->validity->ptr : nullptr;
  // table: a power of two of at least 2 slots per row (at most 2^32, which still exceeds the row count: no retry)
  uint64_t cap = 1024;
  while (cap < 2 * n && cap < (1ull << 32)) cap <<= 1;
  StreamScratch scratch(s);
  unsigned long long *table = nullptr;
  fq_u32 *slot_of = nullptr, *ids = nullptr, *sums = nullptr, *small = nullptr;
  CUDA_TRY(scratch.get(&table, 8 * cap));
  CUDA_TRY(scratch.get(&slot_of, 4 * n));
  CUDA_TRY(scratch.get(&ids, 4 * cap));
  CUDA_TRY(scratch.get(&sums, 4 * ((cap + FQ_SCAN_TILE - 1) / FQ_SCAN_TILE)));
  CUDA_TRY(scratch.get(&small, 16));
  CUDA_TRY(cudaMemsetAsync(small, 0, 16, s));
  fq_dict_clear<<<grid_for(ctx, cap), 256, 0, s>>>(table, cap);
  if (n) fq_dict_insert<<<grid_for(ctx, n, 16), 256, 0, s>>>(src->offsets, src->data, valid, n, table, cap - 1, slot_of);
  fq_dict_flag<<<grid_for(ctx, cap), 256, 0, s>>>(table, cap, ids);
  CUDA_TRY(cudaGetLastError());
  ctx->launches += n ? 3 : 2;
  uint32_t last[2] = {0, 0};
  CUDA_TRY(cudaMemcpyAsync(&last[0], ids + cap - 1, 4, cudaMemcpyDeviceToHost, s));
  if (fq_status st = sort_scan(ctx, ids, cap, sums, s)) return st;
  CUDA_TRY(cudaMemcpyAsync(&last[1], ids + cap - 1, 4, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  const uint64_t d = (uint64_t)last[0] + last[1];   // distinct valid strings
  fq_u32 *rep = nullptr, *lens = nullptr, *rank = nullptr, *rows = nullptr;
  fq_u64 *chunk = nullptr;
  CUDA_TRY(scratch.get(&rep, 4 * d));
  CUDA_TRY(scratch.get(&lens, 4 * d));
  CUDA_TRY(scratch.get(&rank, 4 * d));
  CUDA_TRY(scratch.get(&rows, 4 * d));
  CUDA_TRY(scratch.get(&chunk, 8 * d));
  if (d) {
    fq_dict_compact<<<grid_for(ctx, cap), 256, 0, s>>>(table, cap, ids, src->offsets, rep, lens, small);
    CUDA_TRY(cudaGetLastError());
    ctx->launches++;
    uint32_t max_len = 0;
    CUDA_TRY(cudaMemcpyAsync(&max_len, small, 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    // bytewise order of the distinct strings: stable LSD sort by length, then by chunk K-1 down to chunk 0
    std::lock_guard<std::mutex> sort_lock(ctx->sort_mu);
    SortJob job{ctx, s};
    if (fq_status st = job.acquire(d)) return st;
    fq_column key;
    key.dtype = FQ_U32;
    key.len = d;
    key.ptr = lens;
    const fq_column *kp = &key;
    if (fq_status st = job.sort_by_keys(&kp, nullptr, 1, d, false)) return st;
    key.dtype = FQ_U64;
    key.ptr = chunk;
    for (int64_t j = ((int64_t)max_len + 7) / 8 - 1; j >= 0; j--) {
      fq_dict_chunk<<<grid_for(ctx, d), 256, 0, s>>>(src->offsets, src->data, rep, d, (fq_u32)j, chunk);
      CUDA_TRY(cudaGetLastError());
      ctx->launches++;
      if (fq_status st = job.sort_by_keys(&kp, nullptr, 1, d, true)) return st;
    }
    fq_dict_rank<<<grid_for(ctx, d), 256, 0, s>>>(job.idx[job.cur], d, rep, rank, rows);
    CUDA_TRY(cudaGetLastError());
    ctx->launches++;
    CUDA_TRY(cudaEventRecord(ctx->sort_done, s));   // the sort scratch is free again after this point of the stream
  }
  if (n) {
    fq_dict_codes<<<grid_for(ctx, n, 16), 256, 0, s>>>(valid, n, slot_of, ids, rank, (fq_u32 *)codes->ptr);
    CUDA_TRY(cudaGetLastError());
    ctx->launches++;
  }
  // the dictionary: the representative rows in sorted order (waits for the stream)
  return utf8_take(ctx, src, rows, d, nullptr, s, dict);
}

fq_status fq_utf8_like(fq_ctx *ctx, const fq_utf8 *a, const void *pattern, uint64_t pattern_len, int32_t negate, fq_column *bits,
                       void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!a || !bits || (pattern_len && !pattern)) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (bits->dtype != FQ_U8 || bits->len < (a->len + 7) / 8)
    return set_err(FQ_ERR_INVALID, "Internal Error: LIKE bits of %" PRIu64 " rows need a UInt8 column of at least %" PRIu64 " bytes", a->len, (a->len + 7) / 8);
  if (pattern_len > (uint64_t)INT32_MAX) return set_err(FQ_ERR_INVALID, "Internal Error: LIKE pattern over 2 GiB");
  // a `\` escapes the byte after it: the pattern ends in an unpaired one when the run of `\` at its end is odd
  const unsigned char *pat = (const unsigned char *)pattern;
  uint64_t run = 0;
  while (run < pattern_len && pat[pattern_len - 1 - run] == '\\') run++;
  if (run & 1) return set_err(FQ_ERR_INVALID, "Internal Error: LIKE pattern ends with the escape character \\");
  if (a->len == 0) return FQ_OK;
  cudaStream_t s = (cudaStream_t)stream;
  StreamScratch scratch(s);
  unsigned char *dev = nullptr;
  CUDA_TRY(scratch.get(&dev, pattern_len));
  if (pattern_len) CUDA_TRY(cudaMemcpyAsync(dev, pattern, pattern_len, cudaMemcpyHostToDevice, s));
  fq_utf8_like_kernel<<<grid_for(ctx, a->len, 16), 256, 0, s>>>(a->offsets, a->data, a->validity ? (const fq_u8 *)a->validity->ptr : nullptr, a->len,
                                                                dev, (fq_u32)pattern_len, negate ? 1 : 0, (fq_u8 *)bits->ptr);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  CUDA_TRY(cudaStreamSynchronize(s));   // `pattern` may go away after the call
  return FQ_OK;
}

fq_status fq_utf8_bounds(fq_ctx *ctx, const fq_utf8 *dict, const void *scalar, uint64_t scalar_len, uint64_t *lower, uint64_t *upper,
                         void *stream) {
  if (fq_status st = use(ctx)) return st;
  if (!dict || !lower || !upper || (scalar_len && !scalar)) return set_err(FQ_ERR_INVALID, "Internal Error: null argument");
  if (scalar_len > (uint64_t)INT32_MAX) return set_err(FQ_ERR_INVALID, "Internal Error: literal over 2 GiB");
  cudaStream_t s = (cudaStream_t)stream;
  StreamScratch scratch(s);
  unsigned char *x = nullptr;
  unsigned long long *out = nullptr;
  CUDA_TRY(scratch.get(&x, scalar_len));
  CUDA_TRY(scratch.get(&out, 16));
  if (scalar_len) CUDA_TRY(cudaMemcpyAsync(x, scalar, scalar_len, cudaMemcpyHostToDevice, s));
  fq_utf8_bounds_kernel<<<1, 1, 0, s>>>(dict->offsets, dict->data, dict->len, x, (fq_u32)scalar_len, out);
  CUDA_TRY(cudaGetLastError());
  ctx->launches++;
  unsigned long long h[2];
  CUDA_TRY(cudaMemcpyAsync(h, out, 16, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  *lower = h[0];
  *upper = h[1];
  return FQ_OK;
}

}  // extern "C"
