// codegen.h — lowers a pipe description (expression trees over typed input columns) to the CUDA
// source of the struct `Q` that specialises the kernel skeletons in kernels/fq_skeleton.cuh.
#pragma once

#include <cstdint>
#include <string>
#include <utility>
#include <vector>

#include "../../include/fuse_gpu.h"

namespace fq {

struct Generated {
  std::string source;      // struct Q_<hash> + every extern "C" kernel wrapper (skeleton not included)
  std::string struct_source;                                   // struct Q_<hash> alone
  std::vector<std::pair<std::string, std::string>> kernels;   // (suffix such as "_agg_tma", wrapper source): a JIT build picks a subset
  std::string tag;         // 16 hex digits: FNV-1a of the specialised text, names the kernels
  int kind = 0;            // FQ_PIPE_*
  bool has_pred = false;
  bool generated_source = false;
  int vec = 2;             // rows per thread per vector load group (Q::V)
  int row_bytes = 0;       // bytes read per row (materialised columns actually referenced)
  int pred_row_bytes = 0;  // filter + projection pipes: bytes per row of the predicate's columns (what pass 1 streams)
  int row_bitmaps = 0, pred_row_bitmaps = 0;   // validity bitmaps staged behind them: tile_rows / 8 bytes each
  std::vector<int> used_cols;
  std::vector<int> null_cols;           // referenced columns that carry validity
  std::vector<int> null_kind;           // per entry of null_cols: 1 = one byte per row, 2 = Arrow LSB-first bitmap
  // aggregate pipes: Aggregator leaves in node-index order
  std::vector<int> agg_nodes, agg_ops;
  std::vector<fq_dtype> agg_dtypes;     // state type of each leaf (Count -> UInt64)
  std::vector<int> agg_count_slot;      // slot holding the leaf's count of valid rows, -1 when its argument is never NULL
  int n_slots = 0;                      // leaves + valid-row counts
  // select expressions
  std::vector<fq_dtype> expr_dtypes;    // Function::return_type
  std::vector<int> expr_nullable;       // projection pipes: can select expression i yield NULL?
  std::vector<fq_dtype> node_dtypes;    // per node, FQ_NULL when not reachable
  // GROUP BY pipes: how the key expressions pack into the table key of key_words 64-bit words (lo, then hi), lowest bits
  // first; a field may straddle the two words
  std::vector<fq_dtype> key_dtypes;
  std::vector<int> key_nullable, key_shift, key_bits;   // per key: can it be NULL, first bit, value bits (the null flag sits above them)
  int key_words = 1;                    // 1: keys of up to 64 bits (Q::Key = fq_u64), 2: 65..128 bits (Q::Key = fq_gb_key2)
  bool tma_ok = false;                  // every referenced column is materialised: the bulk-copy staged kernel exists
  bool sel_tma_ok = false;              // ... and the predicate reads at least one column: the staged select kernel exists
  bool track_blocks = false;            // aggregate pipe with a predicate and a Sum leaf: reference-block tracking compiled in
  bool const_divide_by_zero = false;    // a literal zero divisor is evaluated for every scanned row
  unsigned lookup_slots = 0;            // bit k: an FQ_EXPR_LOOKUP node reads table k, which every launch needs bound
};

// Returns FQ_OK or an fq_status; `err` receives the FuseQueryError-style message.
int generate(const fq_pipe_desc &desc, Generated *out, std::string *err);

// numerical_coercion / equal_coercion of datavalues/data_type.rs:27-98
int numerical_coercion(const char *op, fq_dtype l, fq_dtype r, fq_dtype *out, std::string *err);
const char *dtype_name(fq_dtype t);   // arrow DataType Debug
size_t dtype_size(fq_dtype t);

// Tiny s-expression reader used by the build-time AOT generator and the C++ tests:
//   (col number) (u64 1) (+ a b) (sum a) (alias c1 a) (lookup 0 a) ...   `cols` maps names to column indexes.
int parse_sexpr(const std::string &text, const std::vector<std::string> &cols, std::vector<fq_expr_node> *nodes,
                int *root, std::string *err);

}  // namespace fq
