// host_internal.h — helpers shared by the host mirror's translation units (not part of the mirrored surface)
#pragma once
#include <map>

#include "fq_host.h"

namespace fuse {

struct Lowering {
  std::vector<fq_expr_node> nodes;
  std::vector<int> block_cols;        // pipe column -> block column
  std::vector<DataType> col_dtypes;
  std::vector<int> col_nullable;
  std::map<const Function *, int> node_of;
  std::map<const Function *, Utf8DictRef> leaf_dict;   // min / max leaves over a dictionary column: their state is a code
  std::vector<std::pair<DataArrayRef, uint64_t>> lookups;   // slot k of the pipe's LOOKUP nodes: bit table, bits (one per LIKE)
  bool generated = false;
  int column_of(const DataBlock &block, const std::string &name);
  int lower(const Function &f, const DataBlock &block);
  fq_pipe_desc desc(int kind, int predicate, const std::vector<int> &roots) const;
  // the state of Aggregator leaf `leaf` as the reference holds it: a code of a dictionary column becomes its string
  DataValue decode_leaf(const Function &leaf, DataValue v) const;
};

// the dictionary of `f` when it is a dictionary-encoded Utf8 column of `block` (possibly under aliases), else null
Utf8DictRef dict_of(const Function &f, const DataBlock &block);

struct BoundSource {
  fq_source src;
  std::vector<const fq_column *> cols;
};
void bind_source(const Lowering &lw, const DataBlock &block, BoundSource *b);
// compiles the pipe `d` lowered by `lw` and binds its lookup tables
PipeRef compile_pipe(GpuContextRef ctx, const Lowering &lw, const fq_pipe_desc &d);

struct ProjectResult {
  std::vector<DataArrayRef> columns;
  uint64_t rows_selected = 0, rows_written = 0;
  bool limit_reached = false;   // the launch filled `limit` rows; limit_row = the source row that produced the last of them
  uint64_t limit_row = 0;
};
// One fused launch: rows of `block` passing `predicate` (may be null), projected through `funcs`, at most
// `limit` rows (-1 = all), in row order.  With `deferred_error` an evaluation error (zero divisor) is stored there
// instead of thrown, so that the caller can decide whether the reference would have evaluated the offending row at all.
ProjectResult run_project(GpuContextRef ctx, const DataBlock &block, const Function *predicate,
                          const std::vector<const Function *> &funcs, int64_t limit, bool early_exit,
                          std::string *deferred_error = nullptr);

}  // namespace fuse
