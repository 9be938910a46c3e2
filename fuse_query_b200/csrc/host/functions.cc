// functions.cc — enum Function (functions/*.rs) on device-resident blocks.
//
// eval() lowers the whole expression tree under the node it is called on into ONE fused kernel (the
// reference materialises one Arrow array per node, data_array_arithmetic.rs:14-55); accumulate() lowers
// `Aggregator(arg)` into one single-pass reduction kernel.  State plumbing (accumulate_result /
// merge_state / merge_result, depth indexing) is host logic restated 1:1.
#include <algorithm>
#include <climits>
#include <cstring>

#include "host_internal.h"

namespace fuse {

static const char *arith_sym(int op) { static const char *s[] = {"+", "-", "*", "/"}; return s[op & 3]; }
static const char *cmp_sym(int op) { static const char *s[] = {"=", "<", "<=", ">", ">="}; return s[op % 5]; }
static const char *logic_sym(int op) { return op == FQ_LG_AND ? "and" : "or"; }
static const char *like_sym(int op) { return op ? "NOT LIKE" : "LIKE"; }

// ---------------------------------------------------------------------------------------------
// lowering: Function tree + block -> fq_pipe_desc
// ---------------------------------------------------------------------------------------------
int Lowering::column_of(const DataBlock &block, const std::string &name) {
  int bi = block.schema()->index_of(name);
  for (size_t k = 0; k < block_cols.size(); k++)
    if (block_cols[k] == bi) return (int)k;
  if (block_cols.size() == FQ_MAX_COLS) throw FuseQueryError::internal("Unsupported on the device path: more than 8 input columns in one expression");
  DataType t = block.generated ? (DataType)FQ_U64 : block.column((size_t)bi)->data_type();
  if (block.generated) {
    // generated numbers block: its only column must be pipe column 0
    if (!block_cols.empty() || bi != 0) throw FuseQueryError::internal("generated block column must be referenced first");
    generated = true;
  } else if (t == FQ_UTF8) {
    if (!block.column((size_t)bi)->dict()) throw FuseQueryError::internal("Unsupported on the device path: Utf8 column in an expression");
    t = FQ_U32;   // a dictionary column enters the pipe as its codes
  }
  block_cols.push_back(bi);
  col_dtypes.push_back(t);
  col_nullable.push_back(!block.generated && block.column((size_t)bi)->validity() ? 1 : 0);
  return (int)block_cols.size() - 1;
}
Utf8DictRef dict_of(const Function &f, const DataBlock &block) {
  const Function *g = &f;
  while (g->kind == Function::Alias) g = g->left.get();
  if (g->kind != Function::Variable || block.generated) return nullptr;
  const auto &fields = block.schema()->fields;
  for (size_t i = 0; i < fields.size() && i < block.num_columns(); i++)
    if (fields[i].name == g->name) return block.column(i)->dict();
  return nullptr;   // not a column of the block: lowering reports it

}
DataValue Lowering::decode_leaf(const Function &leaf, DataValue v) const {
  auto it = leaf_dict.find(&leaf);
  if (it == leaf_dict.end()) return v;
  return v.some ? DataValue::String(it->second->at((uint32_t)v.u)) : DataValue::None(FQ_UTF8);
}
// `col op literal` over the codes of a sorted dictionary (the lowering table of fq_utf8_dict_encode in fuse_gpu.h)
static void dict_comparison(const Utf8Dict &d, int op, const DataValue &lit, int *code_op, uint64_t *code) {
  if (!lit.some) throw FuseQueryError::internal("DataValue to array cannot be NONE " + lit.to_string());
  const auto [lb, ub] = d.bounds(lit.s);
  switch (op) {
    case FQ_CMP_EQ: *code_op = FQ_CMP_EQ; *code = lb < ub ? lb : d.size; break;
    case FQ_CMP_LT: *code_op = FQ_CMP_LT; *code = lb; break;
    case FQ_CMP_LTEQ: *code_op = FQ_CMP_LT; *code = ub; break;
    case FQ_CMP_GT: *code_op = FQ_CMP_GTEQ; *code = ub; break;
    default: *code_op = FQ_CMP_GTEQ; *code = lb; break;
  }
}
// `s [NOT] LIKE 'pattern'` over a dictionary column: the pattern is matched once per dictionary entry (Utf8Dict::like), and
// the pipe reads the bit of each row's code through a lookup slot, so its generated source does not depend on the pattern
static const Function &like_pattern(const Function &f) {
  const Function *pat = f.right.get();
  while (pat->kind == Function::Alias) pat = pat->left.get();
  return *pat;
}
// what LIKE accepts: a Utf8 operand and a string literal pattern (checked when the plan is typed and when it is lowered)
static void check_like(const Function &f, const DataSchema &s) {
  const DataType lt = f.left->return_type(s), rt = f.right->return_type(s);
  if (lt != FQ_UTF8)
    throw FuseQueryError::internal(std::string("Unsupported (") + data_type_name(lt) + ") " + like_sym(f.op) + " (" + data_type_name(rt) + ")");
  const Function &pat = like_pattern(f);
  if (pat.kind != Function::Constant || pat.value.tag != FQ_UTF8 || !pat.value.some)
    throw FuseQueryError::internal("Unsupported on the device path: LIKE with a pattern that is not a string literal");
}
static int lower_like(Lowering &lw, const Function &f, const DataBlock &block) {
  check_like(f, *block.schema());
  const Utf8DictRef d = dict_of(*f.left, block);
  if (!d) throw FuseQueryError::internal("Unsupported on the device path: LIKE over a Utf8 value that is not a dictionary-encoded column");
  if (lw.lookups.size() == (size_t)FQ_MAX_LOOKUPS)
    throw FuseQueryError::internal("Unsupported on the device path: more than " + std::to_string(FQ_MAX_LOOKUPS) + " LIKE predicates in one pipe");
  const int slot = (int)lw.lookups.size();
  lw.lookups.push_back({d->like(like_pattern(f).value.s, f.op != 0), d->size});
  fq_expr_node n;
  memset(&n, 0, sizeof n);
  n.right = -1;
  n.kind = FQ_EXPR_LOOKUP;
  n.op = slot;
  n.left = lw.lower(*f.left, block);
  lw.nodes.push_back(n);
  lw.node_of[&f] = (int)lw.nodes.size() - 1;
  return (int)lw.nodes.size() - 1;
}
int Lowering::lower(const Function &f, const DataBlock &block) {
  if (f.kind == Function::Like) return lower_like(*this, f, block);
  fq_expr_node n;
  memset(&n, 0, sizeof n);
  n.left = n.right = -1;
  if (f.kind == Function::Arithmetic || f.kind == Function::Comparison || f.kind == Function::Logic) {
    const Utf8DictRef ld = dict_of(*f.left, block), rd = dict_of(*f.right, block);
    if (ld || rd) {
      const DataSchema &sc = *block.schema();
      const DataType lt = f.left->return_type(sc), rt = f.right->return_type(sc);
      if (f.kind == Function::Arithmetic) numerical_coercion(arith_sym(f.op), lt, rt);   // throws "Unsupported (Utf8) + (..)"
      if (f.kind != Function::Comparison)
        throw FuseQueryError::internal(std::string("Unsupported on the device path: Utf8 operand of ") +
                                       (f.kind == Function::Arithmetic ? arith_sym(f.op) : logic_sym(f.op)));
      if (lt != FQ_UTF8 || rt != FQ_UTF8) numerical_coercion(cmp_sym(f.op), lt, rt);   // throws "Unsupported (Utf8) = (Int8)"
      if (ld && rd && ld != rd)
        throw FuseQueryError::internal("Unsupported on the device path: comparison of two Utf8 columns with different dictionaries");
      if (!(ld && rd)) {
        // column (op) literal, or literal (op) column flipped first (data_array_comparison.rs:75-85)
        static const int flipped[] = {FQ_CMP_EQ, FQ_CMP_GT, FQ_CMP_GTEQ, FQ_CMP_LT, FQ_CMP_LTEQ};
        const Function &col = ld ? *f.left : *f.right, &other = ld ? *f.right : *f.left;
        const Function *lit = &other;
        while (lit->kind == Function::Alias) lit = lit->left.get();
        if (lit->kind != Function::Constant)
          throw FuseQueryError::internal("Unsupported on the device path: Utf8 comparison with a computed string");
        int code_op = 0;
        uint64_t code = 0;
        dict_comparison(ld ? *ld : *rd, ld ? f.op % 5 : flipped[f.op % 5], lit->value, &code_op, &code);
        n.kind = FQ_EXPR_COMPARISON;
        n.op = code_op;
        n.left = lower(col, block);
        fq_expr_node c;
        memset(&c, 0, sizeof c);
        c.left = c.right = -1;
        c.kind = FQ_EXPR_CONSTANT;
        c.dtype = FQ_U32;
        c.value.u = code;
        nodes.push_back(c);
        n.right = (int)nodes.size() - 1;
        nodes.push_back(n);
        node_of[&f] = (int)nodes.size() - 1;
        return (int)nodes.size() - 1;
      }
    }
  }
  if (f.kind == Function::Aggregator) {
    if (Utf8DictRef d = dict_of(*f.left, block)) {
      if (f.op == FQ_AGG_SUM) throw FuseQueryError::internal("Unsupported data_array_sum for data type: Utf8");
      if (f.op != FQ_AGG_COUNT) leaf_dict[&f] = d;
    }
  }
  switch (f.kind) {
    case Function::Variable:
      n.kind = FQ_EXPR_FIELD;
      n.column = column_of(block, f.name);
      break;
    case Function::Constant:
      n.kind = FQ_EXPR_CONSTANT;
      n.dtype = f.value.tag;
      if (f.value.tag == FQ_NULL || !f.value.some)  // DataValue::to_array refuses Type(None), data_value.rs:104-109
        throw FuseQueryError::internal("DataValue to array cannot be NONE " + f.value.to_string());
      if (f.value.tag == FQ_F32 || f.value.tag == FQ_F64) n.value.f = f.value.f;
      else if (f.value.tag >= FQ_U8 && f.value.tag <= FQ_U64) n.value.u = f.value.u;
      else n.value.i = f.value.i;
      break;
    case Function::Alias:
      n.kind = FQ_EXPR_ALIAS;
      n.left = lower(*f.left, block);
      break;
    case Function::Aggregator:
      n.kind = FQ_EXPR_AGGREGATOR;
      n.op = f.op;
      n.left = lower(*f.left, block);
      break;
    default:
      n.kind = f.kind == Function::Arithmetic ? FQ_EXPR_ARITHMETIC : f.kind == Function::Comparison ? FQ_EXPR_COMPARISON : FQ_EXPR_LOGIC;
      n.op = f.op;
      n.left = lower(*f.left, block);
      n.right = lower(*f.right, block);
  }
  nodes.push_back(n);
  node_of[&f] = (int)nodes.size() - 1;
  return (int)nodes.size() - 1;
}
fq_pipe_desc Lowering::desc(int kind, int predicate, const std::vector<int> &roots) const {
  fq_pipe_desc d;
  memset(&d, 0, sizeof d);
  d.n_cols = (int)col_dtypes.size();
  for (size_t k = 0; k < col_dtypes.size(); k++) d.col_dtypes[k] = col_dtypes[k];
  for (size_t k = 0; k < col_nullable.size(); k++) d.col_nullable[k] = col_nullable[k];
  d.generated = generated;
  d.nodes = nodes.data();
  d.n_nodes = (int)nodes.size();
  d.predicate = predicate;
  d.kind = kind;
  // fq_pipe_desc::exprs holds FQ_MAX_EXPRS roots; callers with more split them into several pipes (run_project) or refuse
  if (roots.size() > (size_t)FQ_MAX_EXPRS)
    throw FuseQueryError::internal("Unsupported on the device path: more than 8 select expressions in one pipe");
  d.n_exprs = (int)roots.size();
  for (size_t k = 0; k < roots.size(); k++) d.exprs[k] = roots[k];
  return d;
}

void bind_source(const Lowering &lw, const DataBlock &block, BoundSource *b) {
  memset(&b->src, 0, sizeof b->src);
  b->cols.clear();
  for (int bi : lw.block_cols) b->cols.push_back(block.generated ? nullptr : block.column((size_t)bi)->column());
  b->src.n_rows = block.rows();
  b->src.n_cols = (int)b->cols.size();
  b->src.generated = lw.generated;
  b->src.cols = b->cols.data();
  b->src.numbers_begin = block.numbers_begin;
}

PipeRef compile_pipe(GpuContextRef ctx, const Lowering &lw, const fq_pipe_desc &d) {
  auto h = std::make_shared<PipeHandle>();
  h->ctx = ctx;
  ctx->check(fq_pipe_compile(ctx->raw(), &d, &h->pipe));
  for (size_t k = 0; k < lw.lookups.size(); k++) {
    ctx->check(fq_pipe_set_lookup(ctx->raw(), h->pipe, (int32_t)k, lw.lookups[k].first->column(), lw.lookups[k].second));
    h->lookups.push_back(lw.lookups[k].first);
  }
  return h;
}

// One fused launch evaluating `funcs` over `block` (optionally only the rows passing `predicate`, at most
// `limit` of them).  Used by Function::eval, the Filter/Projection transforms and GpuPipeTransform.
ProjectResult run_project(GpuContextRef ctx, const DataBlock &block, const Function *predicate, const std::vector<const Function *> &funcs,
                          int64_t limit, bool early_exit, std::string *deferred_error) {
  if (funcs.size() > (size_t)FQ_MAX_EXPRS) {
    // a pipe holds at most FQ_MAX_EXPRS select expressions: wider projections (and filters over wide tables, which gather
    // every column) run as several launches with the same predicate — the compaction is deterministic, so every launch
    // keeps the same rows in the same order
    ProjectResult all;
    for (size_t b = 0; b < funcs.size(); b += FQ_MAX_EXPRS) {
      std::vector<const Function *> part(funcs.begin() + b, funcs.begin() + std::min(funcs.size(), b + (size_t)FQ_MAX_EXPRS));
      ProjectResult r = run_project(ctx, block, predicate, part, limit, early_exit, deferred_error);
      if (b == 0) { all.rows_selected = r.rows_selected; all.rows_written = r.rows_written; all.limit_reached = r.limit_reached; all.limit_row = r.limit_row; }
      for (auto &c : r.columns) all.columns.push_back(c);
    }
    return all;
  }
  Lowering lw;
  // a generated block's column must be pipe column 0: touch it first
  if (block.generated) lw.column_of(block, block.schema()->fields[0].name);
  int pred = predicate ? lw.lower(*predicate, block) : -1;
  std::vector<int> roots;
  for (const Function *f : funcs) roots.push_back(lw.lower(*f, block));
  fq_pipe_desc d = lw.desc(FQ_PIPE_PROJECT, pred, roots);
  PipeRef pipe = compile_pipe(ctx, lw, d);
  const uint64_t rows = block.rows();
  uint64_t cap = rows;
  if (limit >= 0 && (uint64_t)limit < cap) cap = (uint64_t)limit;
  ProjectResult res;
  std::vector<fq_column *> outs, outs_valid;
  std::vector<DataArrayRef> valids;
  for (size_t e = 0; e < funcs.size(); e++) {
    fq_dtype t;
    int32_t nullable = 0;
    ctx->check(fq_pipe_expr_dtype(ctx->raw(), pipe->pipe, (int)e, &t));
    ctx->check(fq_pipe_expr_nullable(ctx->raw(), pipe->pipe, (int)e, &nullable));
    res.columns.push_back(DataArray::alloc(ctx, t, cap));
    outs.push_back(res.columns.back()->column());
    valids.push_back(nullable ? DataArray::alloc(ctx, FQ_BOOL, cap) : nullptr);
    outs_valid.push_back(nullable ? valids.back()->column() : nullptr);
  }
  BoundSource bs;
  bind_source(lw, block, &bs);
  ctx->check(fq_pipe_launch_project(ctx->raw(), pipe->pipe, &bs.src, outs.data(), outs_valid.data(), cap, limit,
                                    early_exit ? FQ_RUN_LIMIT_EARLY_EXIT : 0, ctx->stream));
  const fq_status fst = fq_pipe_fetch_project(ctx->raw(), pipe->pipe, &res.rows_selected, &res.rows_written);
  if (fst != FQ_OK && deferred_error && fst == FQ_ERR_DIVIDE_BY_ZERO) {
    if (deferred_error->empty()) *deferred_error = fq_last_error(ctx->raw());
  } else {
    ctx->check(fst);
  }
  if (limit > 0 && res.rows_written == (uint64_t)limit && res.rows_selected >= (uint64_t)limit) {
    res.limit_reached = true;
    ctx->check(fq_pipe_fetch_limit_row(ctx->raw(), pipe->pipe, &res.limit_row));
  }
  for (size_t e = 0; e < funcs.size(); e++) {
    if (valids[e]) res.columns[e]->set_validity(valids[e]);
    if (Utf8DictRef d = dict_of(*funcs[e], block)) res.columns[e] = DataArray::with_dict(res.columns[e], d);   // codes out: strings again
  }
  if (res.rows_written < cap)
    for (auto &c : res.columns) c = c->slice(0, res.rows_written);
  return res;
}

// ---------------------------------------------------------------------------------------------
// constructors
// ---------------------------------------------------------------------------------------------
FunctionRef Function::FieldFunction(const std::string &name) {
  auto f = FunctionRef(new Function(Variable));
  f->name = name;
  return f;
}
FunctionRef Function::ConstantFunction(const DataValue &v) {
  auto f = FunctionRef(new Function(Constant));
  f->value = v;
  return f;
}
FunctionRef Function::AliasFunction(const std::string &alias, FunctionRef inner) {
  auto f = FunctionRef(new Function(Alias));
  f->name = alias;
  f->left = std::move(inner);
  return f;
}
static FunctionRef binary(FunctionRef f, const std::vector<FunctionRef> &args) {
  if (args.size() < 2) throw FuseQueryError::internal("index out of bounds: the len is " + std::to_string(args.size()) + " but the index is 1");
  f->left = args[0]->clone();
  f->right = args[1]->clone();
  return f;
}
FunctionRef Function::ArithmeticFunction(int op, const std::vector<FunctionRef> &args) {
  auto f = FunctionRef(new Function(Arithmetic));
  f->op = op;
  return binary(f, args);
}
FunctionRef Function::ComparisonFunction(int op, const std::vector<FunctionRef> &args) {
  auto f = FunctionRef(new Function(Comparison));
  f->op = op;
  return binary(f, args);
}
FunctionRef Function::LogicFunction(int op, const std::vector<FunctionRef> &args) {
  auto f = FunctionRef(new Function(Logic));
  f->op = op;
  return binary(f, args);
}
FunctionRef Function::LikeFunction(bool negate, const std::vector<FunctionRef> &args) {
  auto f = FunctionRef(new Function(Like));
  f->op = negate ? 1 : 0;
  return binary(f, args);
}
FunctionRef Function::AggregatorFunction(int op, const std::vector<FunctionRef> &args) {
  if (args.empty()) throw FuseQueryError::internal("index out of bounds: the len is 0 but the index is 0");
  auto f = FunctionRef(new Function(Aggregator));
  f->op = op;
  f->left = args[0]->clone();
  f->value = DataValue::Null();
  return f;
}
// function_factory.rs:17-39
FunctionRef Function::factory_get(const std::string &name, const std::vector<FunctionRef> &args) {
  std::string n = name;
  std::transform(n.begin(), n.end(), n.begin(), ::tolower);
  if (n == "+") return ArithmeticFunction(FQ_AR_ADD, args);
  if (n == "-") return ArithmeticFunction(FQ_AR_SUB, args);
  if (n == "*") return ArithmeticFunction(FQ_AR_MUL, args);
  if (n == "/") return ArithmeticFunction(FQ_AR_DIV, args);
  if (n == "=") return ComparisonFunction(FQ_CMP_EQ, args);
  if (n == "<") return ComparisonFunction(FQ_CMP_LT, args);
  if (n == ">") return ComparisonFunction(FQ_CMP_GT, args);
  if (n == "<=") return ComparisonFunction(FQ_CMP_LTEQ, args);
  if (n == ">=") return ComparisonFunction(FQ_CMP_GTEQ, args);
  if (n == "and") return LogicFunction(FQ_LG_AND, args);
  if (n == "or") return LogicFunction(FQ_LG_OR, args);
  if (n == "like") return LikeFunction(false, args);
  if (n == "not like") return LikeFunction(true, args);
  if (n == "count") return AggregatorFunction(FQ_AGG_COUNT, args);
  if (n == "min") return AggregatorFunction(FQ_AGG_MIN, args);
  if (n == "max") return AggregatorFunction(FQ_AGG_MAX, args);
  if (n == "sum") return AggregatorFunction(FQ_AGG_SUM, args);
  throw FuseQueryError::internal("Unsupported Function: " + name);
}

FunctionRef Function::clone() const {
  auto f = FunctionRef(new Function(kind));
  f->op = op;
  f->depth = depth;
  f->name = name;
  f->value = value;
  if (left) f->left = left->clone();
  if (right) f->right = right->clone();
  return f;
}

// ---------------------------------------------------------------------------------------------
// typing and display
// ---------------------------------------------------------------------------------------------
DataType Function::return_type(const DataSchema &s) const {
  switch (kind) {
    case Alias: return left->return_type(s);
    case Constant: return value.data_type();
    case Variable: return s.field_with_name(name).data_type;
    case Arithmetic: return numerical_coercion(arith_sym(op), left->return_type(s), right->return_type(s));  // function_arithmetic.rs:36-42
    case Comparison: case Logic: return FQ_BOOL;
    case Like: check_like(*this, s); return FQ_BOOL;
    default: return op == FQ_AGG_COUNT ? (DataType)FQ_U64 : left->return_type(s);  // function_aggregator.rs:38-43
  }
}
bool Function::nullable(const DataSchema &s) const {
  switch (kind) {
    case Alias: return left->nullable(s);
    case Constant: return value.is_null();
    case Variable: return s.field_with_name(name).nullable;
    case Like: return left->nullable(s);
    default: return false;
  }
}
std::string Function::to_string() const {
  static const char *agg[] = {"Min", "Max", "Sum", "Count"};
  switch (kind) {
    case Alias: case Variable: return name;
    case Constant: return value.to_string();
    case Arithmetic: return left->to_string() + " " + arith_sym(op) + " " + right->to_string();
    case Comparison: return left->to_string() + " " + cmp_sym(op) + " " + right->to_string();
    case Logic: return left->to_string() + " " + logic_sym(op) + " " + right->to_string();
    case Like: return left->to_string() + " " + like_sym(op) + " " + right->to_string();
    default: return std::string(agg[op & 3]) + "(" + left->to_string() + ")";
  }
}
void Function::set_depth(size_t d) {
  switch (kind) {
    case Constant: break;
    case Arithmetic:  // function_arithmetic.rs:48-52
      left->set_depth(d);
      right->set_depth(d + 1);
      depth = d;
      break;
    default: depth = d;  // alias does not propagate, function_alias.rs:36-38
  }
}

// ---------------------------------------------------------------------------------------------
// eval / accumulate
// ---------------------------------------------------------------------------------------------
DataColumnarValue Function::eval(GpuContextRef ctx, const DataBlock &block) {
  switch (kind) {
    case Alias: case Aggregator: return left->eval(ctx, block);      // function_aggregator.rs:53-55
    case Constant: return DataColumnarValue::Scalar(value);           // function_constant.rs:30-32
    case Variable:
      if (!block.generated) return DataColumnarValue::Array(block.column_by_name(name));  // function_field.rs:43-47
      [[fallthrough]];
    default: {
      if (kind == Comparison && !block.generated) {
        // string comparisons go to the *_utf8 kernels (datavalues/macros.rs:29-36, 102-113): operands are a Utf8 column or literal
        auto is_utf8 = [&](const Function &f) {
          const Function *g = &f;
          while (g->kind == Alias) g = g->left.get();
          if (g->kind == Constant) return g->value.tag == FQ_UTF8;
          if (g->kind == Variable) {
            const int i = block.schema()->index_of(g->name);
            return block.column((size_t)i)->is_utf8();
          }
          return false;
        };
        if (is_utf8(*left) || is_utf8(*right))
          return DataColumnarValue::Array(data_array_comparison_op(ctx, op, left->eval(ctx, block), right->eval(ctx, block)));
      }
      ProjectResult r = run_project(ctx, block, nullptr, {this}, -1, false);
      return DataColumnarValue::Array(r.columns[0]);
    }
  }
}

static const char *unsupported_agg_name(const Function &f) {
  if (f.kind == Function::Variable) return "field";
  if (f.kind == Function::Like) return like_sym(f.op);
  return f.kind == Function::Comparison ? cmp_sym(f.op) : logic_sym(f.op);
}

void Function::accumulate(GpuContextRef ctx, const DataBlock &block) {
  switch (kind) {
    case Alias: left->accumulate(ctx, block); return;
    case Constant: case Variable: return;
    case Arithmetic: case Comparison: case Logic: case Like:
      left->accumulate(ctx, block);
      right->accumulate(ctx, block);
      return;
    default: break;
  }
  // function_aggregator.rs:57-100
  const uint64_t rows = block.rows();
  DataValue part;
  if (rows == 0) {
    // arrow sum/min/max over an empty array is None; count adds UInt64(0).  The argument is still typed.
    DataType t = left->return_type(*block.schema());
    part = op == FQ_AGG_COUNT ? DataValue::UInt64(0) : DataValue::None(t);
  } else {
    Lowering lw;
    if (block.generated) lw.column_of(block, block.schema()->fields[0].name);
    int root = lw.lower(*this, block);
    fq_pipe_desc d = lw.desc(FQ_PIPE_AGGREGATE, -1, {root});
    PipeRef pipe = compile_pipe(ctx, lw, d);
    BoundSource bs;
    bind_source(lw, block, &bs);
    ctx->check(fq_pipe_launch_aggregate(ctx->raw(), pipe->pipe, &bs.src, 0, ctx->stream));
    fq_value st[4];
    int32_t n = 0;
    uint64_t sel = 0;
    ctx->check(fq_pipe_fetch_aggregate(ctx->raw(), pipe->pipe, st, 4, &n, &sel));
    part = lw.decode_leaf(*this, DataValue::from_abi(st[0]));
  }
  if (op == FQ_AGG_COUNT || op == FQ_AGG_SUM) value = data_value_arithmetic_op(FQ_AR_ADD, value, part);
  else value = data_value_aggregate_op(op, value, part);
}

std::vector<DataValue> Function::accumulate_result() {
  switch (kind) {
    case Alias: return left->accumulate_result();
    case Constant: case Aggregator: return {value};
    case Arithmetic: {  // function_arithmetic.rs:69-75
      auto l = left->accumulate_result(), r = right->accumulate_result();
      l.insert(l.end(), r.begin(), r.end());
      return l;
    }
    default: throw FuseQueryError::internal(std::string("Unsupported aggregate operation for function ") + unsupported_agg_name(*this));
  }
}
void Function::merge_state(const std::vector<DataValue> &states) {
  switch (kind) {
    case Alias: left->merge_state(states); return;
    case Constant: return;
    case Arithmetic:
      left->merge_state(states);
      right->merge_state(states);
      return;
    case Aggregator: {  // function_aggregator.rs:106-139
      if (depth >= states.size())
        throw FuseQueryError::internal("index out of bounds: the len is " + std::to_string(states.size()) + " but the index is " + std::to_string(depth));
      const DataValue &val = states[depth];
      if (op == FQ_AGG_COUNT || op == FQ_AGG_SUM) value = data_value_arithmetic_op(FQ_AR_ADD, value, val);
      else value = data_value_aggregate_op(op, value, val);
      return;
    }
    default: throw FuseQueryError::internal(std::string("Unsupported aggregate operation for function ") + unsupported_agg_name(*this));
  }
}
DataValue Function::merge_result() {
  switch (kind) {
    case Alias: return left->merge_result();
    case Constant: case Aggregator: return value;
    case Arithmetic: return data_value_arithmetic_op(op, left->merge_result(), right->merge_result());  // function_arithmetic.rs:82-88
    default: throw FuseQueryError::internal(std::string("Unsupported aggregate operation for function ") + unsupported_agg_name(*this));
  }
}
void Function::sync_state() {}

// ---------------------------------------------------------------------------------------------
// datavalues array ops: thin wrappers that build a one-node expression over the operands
// ---------------------------------------------------------------------------------------------
static DataArrayRef binary_array_op(GpuContextRef ctx, Function::Kind kind, int op, const DataColumnarValue &l, const DataColumnarValue &r) {
  auto schema = std::make_shared<DataSchema>();
  std::vector<DataArrayRef> cols;
  auto operand = [&](const DataColumnarValue &v, const char *name) -> FunctionRef {
    if (v.is_scalar) return Function::ConstantFunction(v.scalar);
    schema->fields.push_back({name, v.array->data_type(), false});
    cols.push_back(v.array);
    return Function::FieldFunction(name);
  };
  FunctionRef a = operand(l, "l"), b = operand(r, "r");
  FunctionRef f = kind == Function::Arithmetic ? Function::ArithmeticFunction(op, {a, b})
                  : kind == Function::Comparison ? Function::ComparisonFunction(op, {a, b}) : Function::LogicFunction(op, {a, b});
  if (cols.size() == 2 && cols[0]->len() != cols[1]->len())
    throw FuseQueryError::internal(kind == Function::Arithmetic ? "Compute error: Cannot perform math operation on arrays of different length"
                                   : kind == Function::Comparison ? "Compute error: Cannot perform comparison operation on arrays of different length"
                                                                  : "Compute error: Cannot perform bitwise operation on arrays of different length");
  DataBlock block(schema, cols);
  return f->eval(ctx, block).array;
}
DataArrayRef data_array_arithmetic_op(GpuContextRef ctx, int op, const DataColumnarValue &l, const DataColumnarValue &r) {
  return binary_array_op(std::move(ctx), Function::Arithmetic, op, l, r);
}
// A host Utf8 DataArray keeps its strings on the host; for a kernel it is packed into Arrow's offsets + bytes and uploaded.
// A dictionary array is decoded on the device, with its validity.
namespace {
struct DeviceUtf8 {
  GpuContextRef ctx;
  fq_utf8 *raw = nullptr;
  DeviceUtf8(GpuContextRef c, const DataArray &a) : ctx(std::move(c)) {
    if (a.dict()) {
      ctx->check(fq_utf8_take(ctx->raw(), a.dict()->raw, a.column(), a.len(), a.validity() ? a.validity()->column() : nullptr, &raw, ctx->stream));
      return;
    }
    const auto &strs = a.strings();
    std::vector<int32_t> offsets(strs.size() + 1, 0);
    std::string data;
    for (size_t i = 0; i < strs.size(); i++) {
      data += strs[i];
      if (data.size() > (size_t)INT32_MAX) throw FuseQueryError::internal("Utf8 array exceeds 2 GiB of values");
      offsets[i + 1] = (int32_t)data.size();
    }
    ctx->check(fq_utf8_create(ctx->raw(), offsets.data(), data.data(), strs.size(), nullptr, ctx->stream, &raw));
  }
  ~DeviceUtf8() { fq_utf8_free(ctx->raw(), raw); }
  DeviceUtf8(const DeviceUtf8 &) = delete;
  DeviceUtf8 &operator=(const DeviceUtf8 &) = delete;
};
}  // namespace

DataArrayRef data_array_comparison_op(GpuContextRef ctx, int op, const DataColumnarValue &l, const DataColumnarValue &r) {
  const bool l8 = l.data_type() == FQ_UTF8, r8 = r.data_type() == FQ_UTF8;
  if (!l8 && !r8) return binary_array_op(std::move(ctx), Function::Comparison, op, l, r);
  // data_array_comparison.rs:14-94 with a Utf8 side: equal_coercion only accepts Utf8 (op) Utf8
  static const char *sym[] = {"=", "<", "<=", ">", ">="};
  if (!(l8 && r8)) numerical_coercion(sym[op % 5], l.data_type(), r.data_type());   // throws "Unsupported (..) = (..)"
  if (l.is_scalar && r.is_scalar)   // :87-92
    throw FuseQueryError::internal(std::string("Cannot do data_array ") + sym[op % 5] + ", left:Utf8, right:Utf8");
  static const int flipped[] = {FQ_CMP_EQ, FQ_CMP_GT, FQ_CMP_GTEQ, FQ_CMP_LT, FQ_CMP_LTEQ};   // scalar (op) array = array (flipped op) scalar, :75-85
  const DataArrayRef &arr = l.is_scalar ? r.array : l.array;
  DataArrayRef out = DataArray::alloc(ctx, FQ_BOOL, arr->len());
  // NULL slots of dictionary arrays compare to NULL
  const bool nullable = (!l.is_scalar && l.array->validity()) || (!r.is_scalar && r.array->validity());
  DataArrayRef out_valid = nullable ? DataArray::alloc(ctx, FQ_BOOL, arr->len()) : nullptr;
  fq_column *ov = out_valid ? out_valid->column() : nullptr;
  DeviceUtf8 a(ctx, *arr);
  if (l.is_scalar || r.is_scalar) {
    const DataValue &sc = l.is_scalar ? l.scalar : r.scalar;
    if (!sc.some) throw FuseQueryError::internal("DataValue to array cannot be NONE " + sc.to_string());
    ctx->check(fq_utf8_compare_scalar(ctx->raw(), l.is_scalar ? flipped[op % 5] : op, a.raw, sc.s.data(), sc.s.size(), out->column(), ov, ctx->stream));
  } else {
    if (l.array->len() != r.array->len())
      throw FuseQueryError::internal("Compute error: Cannot perform comparison operation on arrays of different length");
    DeviceUtf8 b(ctx, *r.array);
    ctx->check(fq_utf8_compare(ctx->raw(), op, a.raw, b.raw, out->column(), ov, ctx->stream));
    ctx->check(fq_stream_synchronize(ctx->raw(), ctx->stream));
  }
  if (out_valid) out->set_validity(out_valid);
  return out;
}
DataArrayRef data_array_logic_op(GpuContextRef ctx, int op, const DataColumnarValue &l, const DataColumnarValue &r) {
  return binary_array_op(std::move(ctx), Function::Logic, op, l, r);
}
DataValue data_array_aggregate_op(GpuContextRef ctx, int op, const DataArrayRef &a) {
  auto schema = std::make_shared<DataSchema>();
  schema->fields.push_back({"a", a->data_type(), false});
  DataBlock block(schema, {a});
  if (op == FQ_AGG_COUNT) return DataValue::UInt64(a->len());  // data_array_aggregate.rs:113
  if (a->is_utf8()) {   // min_string / max_string, data_array_aggregate.rs:139-154 (macros.rs:162)
    if (op == FQ_AGG_SUM) throw FuseQueryError::internal("Unsupported data_array_sum for data type: Utf8");
    DeviceUtf8 d(ctx, *a);
    int64_t row = -1;
    ctx->check(fq_utf8_minmax(ctx->raw(), op, d.raw, &row, ctx->stream));
    return row < 0 ? DataValue::None(FQ_UTF8) : DataValue::String(a->strings()[(size_t)row]);
  }
  auto f = Function::AggregatorFunction(op, {Function::FieldFunction("a")});
  if (a->len() == 0) return DataValue::None(a->data_type());
  f->accumulate(ctx, block);
  return f->value;
}

}  // namespace fuse
