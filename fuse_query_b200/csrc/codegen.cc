// codegen.cc — expression trees -> CUDA source of the specialising struct Q (see codegen.h).
//
// Typing follows the reference exactly: Function::return_type (functions/function.rs:28-38),
// numerical_coercion / equal_coercion (datavalues/data_type.rs:27-98), Count -> UInt64
// (functions/function_aggregator.rs:38-43); the emitted arithmetic restates what the reference asks
// of arrow 2.0 (cast both sides to the coerced type, wrapping integer lanes, truncating divide that
// errors on a zero divisor: datavalues/data_array_arithmetic.rs:33-54).
#include "codegen.h"

#include <cctype>
#include <cinttypes>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <set>

namespace fq {

const char *dtype_name(fq_dtype t) {
  static const char *n[] = {"Null", "Boolean", "Int8", "Int16", "Int32", "Int64", "UInt8",
                            "UInt16", "UInt32", "UInt64", "Float32", "Float64", "Utf8", "Struct"};
  return (t >= 0 && t <= FQ_STRUCT) ? n[t] : "?";
}
size_t dtype_size(fq_dtype t) {
  switch (t) {
    case FQ_BOOL: case FQ_I8: case FQ_U8: return 1;
    case FQ_I16: case FQ_U16: return 2;
    case FQ_I32: case FQ_U32: case FQ_F32: return 4;
    case FQ_I64: case FQ_U64: case FQ_F64: return 8;
    default: return 0;
  }
}
static bool is_numeric(fq_dtype t) { return t >= FQ_I8 && t <= FQ_F64; }
static bool is_float(fq_dtype t) { return t == FQ_F32 || t == FQ_F64; }
static bool is_signed_int(fq_dtype t) { return t >= FQ_I8 && t <= FQ_I64; }

static const char *ctype(fq_dtype t) {
  static const char *n[] = {"void", "bool", "fq_i8", "fq_i16", "fq_i32", "fq_i64", "fq_u8",
                            "fq_u16", "fq_u32", "fq_u64", "float", "double", "void", "void"};
  return n[t];
}
static const char *arith_sym(int op) { static const char *s[] = {"+", "-", "*", "/"}; return s[op & 3]; }
static const char *cmp_sym(int op) { static const char *s[] = {"=", "<", "<=", ">", ">="}; return s[op % 5]; }
static const char *cmp_c(int op) { static const char *s[] = {"==", "<", "<=", ">", ">="}; return s[op % 5]; }
static const char *agg_name(int op) { static const char *s[] = {"min", "max", "sum", "count"}; return s[op & 3]; }

static std::string fmt(const char *f, ...) __attribute__((format(printf, 1, 2)));
static std::string fmt(const char *f, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, f);
  vsnprintf(buf, sizeof buf, f, ap);
  va_end(ap);
  return buf;
}

int numerical_coercion(const char *op, fq_dtype l, fq_dtype r, fq_dtype *out, std::string *err) {
  if (!is_numeric(l) || !is_numeric(r)) {
    *err = fmt("Internal Error: Unsupported (%s) %s (%s)", dtype_name(l), op, dtype_name(r));
    return FQ_ERR_INTERNAL;
  }
  if (l == r) { *out = l; return FQ_OK; }
  static const fq_dtype order[] = {FQ_F64, FQ_F32, FQ_I64, FQ_I32, FQ_I16, FQ_I8, FQ_U64, FQ_U32, FQ_U16, FQ_U8};
  for (fq_dtype t : order)
    if (l == t || r == t) { *out = t; return FQ_OK; }
  *err = fmt("Internal Error: Unsupported (%s) %s (%s)", dtype_name(l), op, dtype_name(r));
  return FQ_ERR_INTERNAL;
}
static int equal_coercion(const char *op, fq_dtype l, fq_dtype r, fq_dtype *out, std::string *err) {
  if (l == r) { *out = l; return FQ_OK; }
  return numerical_coercion(op, l, r, out, err);
}

namespace {

struct Gen {
  const fq_pipe_desc &d;
  std::vector<fq_dtype> ty;     // inferred, FQ_NULL = not visited
  std::vector<char> visited, scalar;
  std::set<int> used_cols;
  std::string err;
  int status = FQ_OK;
  bool const_div0 = false;
  int quiet_depth = 0;
  unsigned lookup_slots = 0;   // bit k: some FQ_EXPR_LOOKUP node reads table k

  // columns referenced below node i (any depth)
  void cols_below(int i, std::set<int> *out, int depth = 0) const {
    if (i < 0 || i >= d.n_nodes || depth > 130) return;
    const fq_expr_node &n = d.nodes[i];
    if (n.kind == FQ_EXPR_FIELD) { out->insert(n.column); return; }
    if (n.kind == FQ_EXPR_CONSTANT) return;
    cols_below(n.left, out, depth + 1);
    if (n.kind != FQ_EXPR_ALIAS && n.kind != FQ_EXPR_AGGREGATOR) cols_below(n.right, out, depth + 1);
  }

  bool trivial(int i, int depth = 0) const {
    if (i < 0 || i >= d.n_nodes || depth > 130) return false;   // (an alias cycle is not trivial; infer() reports it)
    const fq_expr_node &n = d.nodes[i];
    if (n.kind == FQ_EXPR_FIELD || n.kind == FQ_EXPR_CONSTANT) return true;
    return n.kind == FQ_EXPR_ALIAS && trivial(n.left, depth + 1);
  }

  explicit Gen(const fq_pipe_desc &desc) : d(desc), ty(desc.n_nodes, FQ_NULL), visited(desc.n_nodes, 0), scalar(desc.n_nodes, 0) {}

  bool fail(int st, const std::string &m) {
    if (status == FQ_OK) { status = st; err = m; }
    return false;
  }
  const fq_expr_node *node(int i) {
    if (i < 0 || i >= d.n_nodes) { fail(FQ_ERR_INVALID, fmt("Internal Error: expression node index %d out of range", i)); return nullptr; }
    return &d.nodes[i];
  }
  fq_dtype col_dtype(int c) const { return (d.generated && c == 0) ? (fq_dtype)FQ_U64 : d.col_dtypes[c]; }

  // Function::return_type + the checks eval would make
  bool infer(int i, int depth = 0) {
    const fq_expr_node *n = node(i);
    if (!n) return false;
    if (depth > 128) return fail(FQ_ERR_PLAN, "Error during plan: expression depth more than 128");
    if (visited[i] == 2) return status == FQ_OK;   // typed before (a node shared by two parents)
    if (visited[i] == 1)                            // still being typed: the "tree" has a cycle — every later walk would not end
      return fail(FQ_ERR_INVALID, fmt("Internal Error: expression node %d is its own ancestor", i));
    visited[i] = 1;
    const bool typed = infer_node(i, n, depth);
    visited[i] = 2;
    return typed;
  }
  bool infer_node(int i, const fq_expr_node *n, int depth) {
    // operator codes index symbol tables below and in the emitter: refuse anything outside the enums up front
    const int n_ops = n->kind == FQ_EXPR_ARITHMETIC ? 4 : n->kind == FQ_EXPR_COMPARISON ? 5 : n->kind == FQ_EXPR_LOGIC ? 2
                      : n->kind == FQ_EXPR_AGGREGATOR ? 4 : 0;
    if (n_ops && (n->op < 0 || n->op >= n_ops))
      return fail(FQ_ERR_INVALID, fmt("Internal Error: operator code %d out of range for expression node kind %d", n->op, n->kind));
    switch (n->kind) {
      case FQ_EXPR_FIELD: {
        if (n->column < 0 || n->column >= d.n_cols)
          return fail(FQ_ERR_INTERNAL, fmt("Internal Error: Invalid argument error: Unable to get field at index %d", n->column));
        fq_dtype t = col_dtype(n->column);
        if (!is_numeric(t) && t != FQ_BOOL)
          return fail(FQ_ERR_UNSUPPORTED, fmt("Unsupported on the device path: column of type %s", dtype_name(t)));
        ty[i] = t;
        if (quiet_depth == 0) used_cols.insert(n->column);
        return true;
      }
      case FQ_EXPR_CONSTANT:
        if (!(is_numeric(n->dtype) || n->dtype == FQ_BOOL))
          return fail(FQ_ERR_UNSUPPORTED, fmt("Unsupported on the device path: constant of type %s", dtype_name(n->dtype)));
        ty[i] = n->dtype;
        scalar[i] = 1;
        return true;
      case FQ_EXPR_ALIAS:
      case FQ_EXPR_AGGREGATOR: {
        // Count(arg) evaluates and discards its argument (function_aggregator.rs:58-66).  A bare column or literal cannot
        // fail, so nothing has to be read for it: the column is typed but not marked as used.
        const bool quiet = n->kind == FQ_EXPR_AGGREGATOR && n->op == FQ_AGG_COUNT && trivial(n->left) && d.kind != FQ_PIPE_PROJECT;
        if (quiet) quiet_depth++;
        const bool ok = infer(n->left, depth + 1);
        if (quiet) quiet_depth--;
        if (!ok) return false;
        ty[i] = ty[n->left];
        scalar[i] = scalar[n->left];
        return true;
      }
      case FQ_EXPR_ARITHMETIC: {
        if (!infer(n->left, depth + 1) || !infer(n->right, depth + 1)) return false;
        fq_dtype t;
        int st = numerical_coercion(arith_sym(n->op), ty[n->left], ty[n->right], &t, &err);
        if (st) { status = st; return false; }
        if (scalar[n->left] && scalar[n->right])
          return fail(FQ_ERR_UNSUPPORTED, "Unsupported on the device path: arithmetic between two constants (the reference yields a 1-row array)");
        ty[i] = t;
        return true;
      }
      case FQ_EXPR_COMPARISON: {
        if (!infer(n->left, depth + 1) || !infer(n->right, depth + 1)) return false;
        if (scalar[n->left] && scalar[n->right])  // data_array_comparison.rs:87-92
          return fail(FQ_ERR_INTERNAL, fmt("Internal Error: Cannot do data_array %s, left:%s, right:%s", cmp_sym(n->op),
                                          dtype_name(ty[n->left]), dtype_name(ty[n->right])));
        fq_dtype t;
        int st = equal_coercion(cmp_sym(n->op), ty[n->left], ty[n->right], &t, &err);
        if (st) { status = st; return false; }
        if (t == FQ_BOOL)  // macros.rs:55-76: no Boolean arm
          return fail(FQ_ERR_INTERNAL, fmt("Internal Error: Unsupported arithmetic_compute::%s for data type: Boolean",
                                          (const char *[]){"eq", "lt", "lt_eq", "gt", "gt_eq"}[n->op % 5]));
        ty[i] = FQ_BOOL;
        return true;
      }
      case FQ_EXPR_LOGIC: {
        if (!infer(n->left, depth + 1) || !infer(n->right, depth + 1)) return false;
        const char *sym = n->op == FQ_LG_AND ? "and" : "or";
        if (scalar[n->left] || scalar[n->right])  // data_array_logic.rs:25-30
          return fail(FQ_ERR_INTERNAL, fmt("Internal Error: Cannot do data_array %s, left:%s, right:%s", sym,
                                          dtype_name(ty[n->left]), dtype_name(ty[n->right])));
        for (int c : {n->left, n->right})
          if (ty[c] != FQ_BOOL)
            return fail(FQ_ERR_INTERNAL, fmt("Internal Error: Cannot downcast_array from datatype:%s item to:BooleanArray", dtype_name(ty[c])));
        ty[i] = FQ_BOOL;
        return true;
      }
      case FQ_EXPR_LOOKUP: {
        if (n->op < 0 || n->op >= FQ_MAX_LOOKUPS)
          return fail(FQ_ERR_INVALID, fmt("Internal Error: lookup slot %d out of range [0, %d)", n->op, FQ_MAX_LOOKUPS));
        if (!infer(n->left, depth + 1)) return false;
        const fq_dtype t = ty[n->left];
        if (t < FQ_U8 || t > FQ_U64)
          return fail(FQ_ERR_INVALID, fmt("Internal Error: a lookup takes an unsigned integer index, not %s", dtype_name(t)));
        if (scalar[n->left]) return fail(FQ_ERR_INVALID, "Internal Error: a lookup of a constant index");
        lookup_slots |= 1u << n->op;
        ty[i] = FQ_BOOL;
        return true;
      }
      default:
        return fail(FQ_ERR_INVALID, fmt("Internal Error: unknown expression node kind %d", n->kind));
    }
  }

  static std::string literal(fq_dtype t, fq_scalar_bits v) {
    switch (t) {
      case FQ_BOOL: return v.i ? "true" : "false";
      case FQ_I8: case FQ_I16: case FQ_I32:
        return fmt("((%s)(%" PRId64 "))", ctype(t), v.i);
      case FQ_I64:
        if (v.i == INT64_MIN) return "((fq_i64)(-9223372036854775807ll - 1))";
        return fmt("((fq_i64)(%" PRId64 "ll))", v.i);
      case FQ_U8: case FQ_U16: case FQ_U32:
        return fmt("((%s)(%" PRIu64 "u))", ctype(t), v.u);
      case FQ_U64: return fmt("((fq_u64)(%" PRIu64 "ull))", v.u);
      // %a prints ±inf and NaN as `inf` / `nan`, which are not CUDA identifiers: non-finite constants are written as
      // their bit patterns, which also keeps the sign and the NaN payload
      case FQ_F32: {
        const float x = (float)v.f;
        if (std::isfinite(x)) return fmt("((float)(%a))", (double)x);
        uint32_t b;
        memcpy(&b, &x, sizeof b);
        return fmt("__int_as_float((int)0x%08" PRIx32 "u)", b);
      }
      case FQ_F64:
        if (std::isfinite(v.f)) return fmt("((double)(%a))", v.f);
        return fmt("__longlong_as_double((long long)0x%016" PRIx64 "ull)", v.u);
      default: return "0";
    }
  }
  bool nullable_col(int c) const { return !(d.generated && c == 0) && d.col_nullable[c] != 0; }
  bool bitmap_col(int c) const { return nullable_col(c) && d.col_nullable[c] == 2; }   // validity = Arrow LSB-first bitmap
  // arrow cast S -> T yields NULL for values T cannot represent (num::cast): can that happen at all?
  static bool cast_fallible(fq_dtype from, fq_dtype to) {
    if (from == to || is_float(to) || from == FQ_BOOL || to == FQ_BOOL) return false;
    if (is_float(from)) return true;
    const int bf = (int)dtype_size(from) * 8, bt = (int)dtype_size(to) * 8;
    if (is_signed_int(to)) return is_signed_int(from) ? bf > bt : bf >= bt;
    return is_signed_int(from) ? true : bf > bt;
  }

  // Row-level code of one generated function, in SSA form: every node is evaluated once into `n<i>` (value) and, when
  // it can be NULL at all, `k<i>` (validity).  Validity follows arrow: a slot is null when either operand is null
  // (combine_option_bitmap) or a coercion cast cannot represent the value; "true" means statically never null.
  struct Emitter {
    Gen &g;
    std::string body;   // statements, indented by `ind`
    std::string ind;
    std::vector<std::string> val, ok;
    std::vector<char> done;
    Emitter(Gen &gen, const std::string &indent) : g(gen), ind(indent), val(gen.d.n_nodes), ok(gen.d.n_nodes), done(gen.d.n_nodes, 0) {}

    static std::string conj(const std::vector<std::string> &terms) {
      std::string o;
      for (const auto &t : terms)
        if (!t.empty() && t != "true") o += (o.empty() ? "" : " & ") + t;
      return o.empty() ? "true" : o;
    }
    // operand `c` converted to type `t`: value expression and (possibly empty) representability check
    std::pair<std::string, std::string> coerce(int c, fq_dtype t) {
      const fq_dtype from = g.ty[c];
      if (from == t) return {val[c], ""};
      std::string v = fmt("fq_cast_v<%s, %s>(", ctype(t), ctype(from)) + val[c] + ")";
      std::string k = cast_fallible(from, t) ? fmt("fq_cast_ok<%s, %s>(", ctype(t), ctype(from)) + val[c] + ")" : "";
      return {v, k};
    }
    void node(int i) {
      if (done[i]) return;
      done[i] = 1;
      const fq_expr_node &n = g.d.nodes[i];
      switch (n.kind) {
        case FQ_EXPR_FIELD:
          val[i] = fmt("r.c%d[v]", n.column);
          ok[i] = g.nullable_col(n.column) ? fmt("r.k%d[v]", n.column) : "true";
          return;
        case FQ_EXPR_CONSTANT:
          val[i] = literal(n.dtype, n.value);
          ok[i] = "true";
          return;
        case FQ_EXPR_ALIAS: case FQ_EXPR_AGGREGATOR:   // Aggregator::eval is transparent, function_aggregator.rs:53-55
          node(n.left);
          val[i] = val[n.left];
          ok[i] = ok[n.left];
          return;
        case FQ_EXPR_LOOKUP:   // the row functions receive the launch parameters, which hold the bound tables
          node(n.left);
          body += ind + fmt("const bool n%d = fq_lookup(p.lookup[%d], p.lookup_bits[%d], (fq_u64)(", i, n.op, n.op) + val[n.left] + "));\n";
          val[i] = fmt("n%d", i);
          ok[i] = ok[n.left];
          return;
        default: break;
      }
      node(n.left);
      node(n.right);
      fq_dtype t = g.ty[i];
      if (n.kind == FQ_EXPR_COMPARISON) {
        std::string e;
        equal_coercion(cmp_sym(n.op), g.ty[n.left], g.ty[n.right], &t, &e);
      } else if (n.kind == FQ_EXPR_LOGIC) {
        t = FQ_BOOL;
      }
      auto a = coerce(n.left, t), b = coerce(n.right, t);
      const std::string valid = conj({ok[n.left], ok[n.right], a.second, b.second});
      const std::string name = fmt("n%d", i);
      std::string rhs;
      const char *T = n.kind == FQ_EXPR_ARITHMETIC ? ctype(t) : "bool";
      if (n.kind == FQ_EXPR_ARITHMETIC) {
        if (n.op == FQ_AR_DIV) {
          const fq_expr_node &rn = g.d.nodes[n.right];
          if (g.scalar[n.right] && rn.kind == FQ_EXPR_CONSTANT && (is_float(rn.dtype) ? rn.value.f == 0.0 : rn.value.u == 0))
            g.const_div0 = true;
          rhs = fmt("fq_div<%s>(", ctype(t)) + a.first + ", " + b.first + ", " + valid + ", err)";
        } else {
          const char *f = n.op == FQ_AR_ADD ? "fq_add" : n.op == FQ_AR_SUB ? "fq_sub" : "fq_mul";
          rhs = fmt("%s<%s>(", f, ctype(t)) + a.first + ", " + b.first + ")";
        }
      } else if (n.kind == FQ_EXPR_COMPARISON) {
        rhs = "(" + a.first + " " + cmp_c(n.op) + " " + b.first + ")";
      } else {  // non-short-circuit: both sides are evaluated (and may raise) in the reference
        rhs = "(" + a.first + (n.op == FQ_LG_AND ? " & " : " | ") + b.first + ")";
      }
      body += ind + "const " + T + " " + name + " = " + rhs + ";\n";
      val[i] = name;
      if (valid == "true") {
        ok[i] = "true";
      } else {
        body += ind + fmt("const bool k%d = ", i) + valid + ";\n";
        ok[i] = fmt("k%d", i);
      }
    }
  };
  // can node i ever be NULL?  (same rules as the emitter, without emitting)
  bool maybe_null(int i) {
    Emitter e(*this, "");
    e.node(i);
    return e.ok[i] != "true";
  }

  // Aggregator leaves reachable without crossing another Aggregator
  void collect_aggs(int i, std::set<int> &out) {
    const fq_expr_node &n = d.nodes[i];
    switch (n.kind) {
      case FQ_EXPR_AGGREGATOR: out.insert(i); break;
      case FQ_EXPR_ALIAS: case FQ_EXPR_LOOKUP: collect_aggs(n.left, out); break;
      case FQ_EXPR_ARITHMETIC: case FQ_EXPR_COMPARISON: case FQ_EXPR_LOGIC:
        collect_aggs(n.left, out);
        collect_aggs(n.right, out);
        break;
      default: break;
    }
  }
};

uint64_t fnv1a(const std::string &s) {
  uint64_t h = 1469598103934665603ull;
  for (unsigned char c : s) { h ^= c; h *= 1099511628211ull; }
  return h;
}

std::string identity_of(int op, fq_dtype t) {
  if (op == FQ_AGG_SUM || op == FQ_AGG_COUNT) return fmt("(%s)0", ctype(t));
  if (op == FQ_AGG_MIN) return fmt("fq_traits<%s>::hi()", ctype(t));
  return fmt("fq_traits<%s>::lo()", ctype(t));
}

}  // namespace

int generate(const fq_pipe_desc &d, Generated *out, std::string *err) {
  *out = Generated();
  const bool groupby = d.kind == FQ_PIPE_GROUPBY;
  const bool agg_like = d.kind == FQ_PIPE_AGGREGATE || groupby;   // select expressions are trees over Aggregator leaves
  if (d.n_cols < 0 || d.n_cols > FQ_MAX_COLS || d.n_exprs < (groupby ? 0 : 1) || d.n_exprs > FQ_MAX_EXPRS || !d.nodes || d.n_nodes < 1) {
    *err = "Error during plan: pipe needs 1..8 select expressions over at most 8 input columns";
    return FQ_ERR_PLAN;
  }
  if (d.kind != FQ_PIPE_PROJECT && d.kind != FQ_PIPE_AGGREGATE && !groupby) {
    *err = "Error during plan: unknown pipe kind";
    return FQ_ERR_PLAN;
  }
  if (groupby ? (d.n_keys < 1 || d.n_keys > FQ_MAX_KEYS) : d.n_keys != 0) {
    *err = groupby ? "Error during plan: a GROUP BY pipe needs 1..4 key expressions" : "Error during plan: only GROUP BY pipes take key expressions";
    return FQ_ERR_PLAN;
  }
  if (d.generated && d.n_cols < 1) {
    *err = "Error during plan: generated numbers source needs column 0";
    return FQ_ERR_PLAN;
  }
  Gen g(d);
  if (d.predicate >= 0) {
    if (!g.infer(d.predicate)) { *err = g.err; return g.status; }
    if (g.ty[d.predicate] != FQ_BOOL || g.scalar[d.predicate]) {  // transform_filter.rs:45-50
      *err = "Internal Error: cannot downcast to boolean array";
      return FQ_ERR_INTERNAL;
    }
  }
  for (int e = 0; e < d.n_exprs; e++) {
    if (!g.infer(d.exprs[e])) { *err = g.err; return g.status; }
    out->expr_dtypes.push_back(g.ty[d.exprs[e]]);
  }
  out->kind = d.kind;
  out->has_pred = d.predicate >= 0;
  out->generated_source = d.generated != 0;

  // GROUP BY keys: typed like any expression; no aggregates, no bare constants
  struct KeyInfo { int node; fq_dtype t; bool nullable; int shift, bits; };
  std::vector<KeyInfo> keys;
  if (groupby) {
    int shift = 0;
    for (int k = 0; k < d.n_keys; k++) {
      if (!g.infer(d.keys[k])) { *err = g.err; return g.status; }
      std::set<int> inner;
      g.collect_aggs(d.keys[k], inner);
      if (!inner.empty()) { *err = "Internal Error: Aggregate function is found in GROUP BY in query"; return FQ_ERR_INTERNAL; }
      if (g.scalar[d.keys[k]]) { *err = "Unsupported on the device path: a constant GROUP BY expression"; return FQ_ERR_UNSUPPORTED; }
      KeyInfo ki;
      ki.node = d.keys[k];
      ki.t = g.ty[d.keys[k]];
      ki.nullable = g.maybe_null(d.keys[k]);
      ki.bits = (int)dtype_size(ki.t) * 8;
      ki.shift = shift;
      shift += ki.bits + (ki.nullable ? 1 : 0);
      keys.push_back(ki);
      out->key_dtypes.push_back(ki.t);
      out->key_nullable.push_back(ki.nullable ? 1 : 0);
      out->key_shift.push_back(ki.shift);
      out->key_bits.push_back(ki.bits);
    }
    if (shift > 128) {
      *err = fmt("Unsupported on the device path: GROUP BY keys of %d bits (values plus one bit per nullable key) do not pack into 64 or 128", shift);
      return FQ_ERR_UNSUPPORTED;
    }
    out->key_words = shift > 64 ? 2 : 1;
  }

  std::set<int> aggs;
  if (agg_like) {
    for (int e = 0; e < d.n_exprs; e++) g.collect_aggs(d.exprs[e], aggs);
    for (int a : aggs) {
      const fq_expr_node &n = d.nodes[a];
      fq_dtype t = n.op == FQ_AGG_COUNT ? (fq_dtype)FQ_U64 : g.ty[n.left];
      if (n.op != FQ_AGG_COUNT && !is_numeric(t)) {  // data_array_aggregate.rs:153-161
        *err = fmt("Internal Error: Unsupported data_array_%s for data type: %s", agg_name(n.op), dtype_name(t));
        return FQ_ERR_INTERNAL;
      }
      out->agg_nodes.push_back(a);
      out->agg_ops.push_back(n.op);
      out->agg_dtypes.push_back(t);
    }
    // select expression types: Count -> UInt64 at the leaf (function_aggregator.rs:38-43)
    std::function<int(int, fq_dtype *)> rtype = [&](int i, fq_dtype *t) -> int {
      const fq_expr_node &n = d.nodes[i];
      if (n.kind == FQ_EXPR_AGGREGATOR && n.op == FQ_AGG_COUNT) { *t = FQ_U64; return FQ_OK; }
      if (n.kind == FQ_EXPR_ALIAS) return rtype(n.left, t);
      if (n.kind == FQ_EXPR_ARITHMETIC) {
        fq_dtype a, b;
        if (int st = rtype(n.left, &a)) return st;
        if (int st = rtype(n.right, &b)) return st;
        return numerical_coercion(arith_sym(n.op), a, b, t, err);
      }
      *t = g.ty[i];
      return FQ_OK;
    };
    for (int e = 0; e < d.n_exprs; e++)
      if (int st = rtype(d.exprs[e], &out->expr_dtypes[e])) return st;
  }

  // ---- vector width and Rows layout ----
  size_t min_w = 8;
  for (int c : g.used_cols) { size_t w = dtype_size(g.col_dtype(c)); if (w < min_w) min_w = w; }
  int V = (int)(16 / min_w);
  if (V < 2) V = 2;
  out->vec = V;
  out->used_cols.assign(g.used_cols.begin(), g.used_cols.end());
  for (int c : g.used_cols)
    if (!(d.generated && c == 0)) out->row_bytes += (int)dtype_size(g.col_dtype(c));

  // nullable inputs that are actually referenced; validity travels as one byte per row next to the values
  std::vector<int> null_cols;
  for (int c : g.used_cols)
    if (g.nullable_col(c)) null_cols.push_back(c);
  // per aggregate leaf: does its argument ever yield NULL?  then the leaf counts its valid rows (sum/min/max of no valid
  // row is None, arrow sum / min / max skip nulls)
  std::vector<int> leaf_counted;
  for (size_t k = 0; k < out->agg_nodes.size(); k++) {
    const fq_expr_node &an = d.nodes[out->agg_nodes[k]];
    const bool counted = an.op != FQ_AGG_COUNT && g.maybe_null(an.left);
    leaf_counted.push_back(counted ? 1 : 0);
  }
  const int n_leaves = (int)out->agg_nodes.size();
  int n_slots = n_leaves;
  out->agg_count_slot.assign(n_leaves, -1);
  for (int k = 0; k < n_leaves; k++)
    if (leaf_counted[k]) out->agg_count_slot[k] = n_slots++;
  out->n_slots = n_slots;
  out->null_cols = null_cols;
  for (int c : null_cols) out->null_kind.push_back(g.bitmap_col(c) ? 2 : 1);
  out->expr_nullable.assign(d.n_exprs, 0);
  if (d.kind == FQ_PIPE_PROJECT)
    for (int e = 0; e < d.n_exprs; e++) out->expr_nullable[e] = g.maybe_null(d.exprs[e]) ? 1 : 0;

  std::string s;
  s += "struct Q_@ {\n";
  bool has_sum = false;
  for (int op : out->agg_ops) has_sum = has_sum || op == FQ_AGG_SUM;
  out->track_blocks = out->has_pred && has_sum && !groupby;   // only Sum is poisoned by an empty block (SURVEY F8)
  s += fmt("  static constexpr int V = %d;\n  static constexpr int NSLOTS = %d;\n  static constexpr bool HAS_PRED = %s;\n"
           "  static constexpr bool TRACK_BLOCKS = %s;\n", V, n_slots, out->has_pred ? "true" : "false", out->track_blocks ? "true" : "false");
  s += "  struct Rows {";
  for (int c : g.used_cols) s += fmt(" %s c%d[V];", ctype(g.col_dtype(c)), c);
  for (int c : null_cols) s += fmt(" bool k%d[V];", c);
  out->lookup_slots = g.lookup_slots;
  s += " };\n";
  s += "  __device__ static __forceinline__ void load(Rows &r, const fq_launch_params &p, fq_u64 g) {\n";
  for (int c : g.used_cols) {
    if (d.generated && c == 0) s += "#pragma unroll\n    for (int v = 0; v < V; v++) r.c0[v] = p.numbers_begin + g * V + v;\n";
    else s += fmt("    fq_load_vec<%s, V>(r.c%d, p.cols[%d], g);\n", ctype(g.col_dtype(c)), c, c);
  }
  auto valid_vec = [&](int c) {
    return g.bitmap_col(c) ? fmt("    fq_load_bits<V>(r.k%d, p.cols_valid[%d], p.cols_valid_bit0[%d] + g * V);\n", c, c, c)
                           : fmt("    fq_load_vec<bool, V>(r.k%d, p.cols_valid[%d], g);\n", c, c);
  };
  auto valid_one = [&](int c) {
    return g.bitmap_col(c) ? fmt("    r.k%d[0] = fq_ld_bit(p.cols_valid[%d], p.cols_valid_bit0[%d] + row);\n", c, c, c)
                           : fmt("    r.k%d[0] = fq_ld1<bool>(p.cols_valid[%d], row);\n", c, c);
  };
  for (int c : null_cols) s += valid_vec(c);
  s += "  }\n";
  s += "  __device__ static __forceinline__ void load1(Rows &r, const fq_launch_params &p, fq_u64 row) {\n";
  for (int c : g.used_cols) {
    if (d.generated && c == 0) s += "    r.c0[0] = p.numbers_begin + row;\n";
    else s += fmt("    r.c%d[0] = fq_ld1<%s>(p.cols[%d], row);\n", c, ctype(g.col_dtype(c)), c);
  }
  for (int c : null_cols) s += valid_one(c);
  s += "  }\n";
  s += "  __device__ static __forceinline__ void copy_row(Rows &dst, int v, const Rows &one) {\n";
  for (int c : g.used_cols) s += fmt("    dst.c%d[v] = one.c%d[0];\n", c, c);
  for (int c : null_cols) s += fmt("    dst.k%d[v] = one.k%d[0];\n", c, c);
  s += "  }\n";
  // Filter + projection pipes read only the predicate's columns in pass 1 (one streaming read of every row); the
  // projection-only columns are read in pass 2, for the rows that were kept.
  std::set<int> pred_cols;
  if (d.kind == FQ_PIPE_PROJECT && out->has_pred) {
    g.cols_below(d.predicate, &pred_cols);
    std::vector<int> pred_null;
    for (int c : pred_cols)
      if (g.nullable_col(c)) pred_null.push_back(c);
    out->pred_row_bytes = 0;
    for (int c : pred_cols)
      if (!(d.generated && c == 0)) out->pred_row_bytes += (int)dtype_size(g.col_dtype(c));
    for (int c : pred_null)
      if (!g.bitmap_col(c)) out->pred_row_bytes += 1;   // byte validity is staged like a column; bitmaps are read in place
    s += fmt("  static constexpr int PRED_ROW_BYTES = %d;\n", out->pred_row_bytes);
    {
      int nb = 0;
      for (int c : pred_null) nb += g.bitmap_col(c) ? 1 : 0;
      s += fmt("  __device__ static constexpr fq_u32 pred_stage_bytes(fq_u32 tile_rows) { return tile_rows * %du + %du * (tile_rows >> 3); }\n", out->pred_row_bytes, nb);
    }
    s += "  __device__ static __forceinline__ void load_pred(Rows &r, const fq_launch_params &p, fq_u64 g) {\n";
    for (int c : pred_cols) {
      if (d.generated && c == 0) s += "#pragma unroll\n    for (int v = 0; v < V; v++) r.c0[v] = p.numbers_begin + g * V + v;\n";
      else s += fmt("    fq_load_vec<%s, V>(r.c%d, p.cols[%d], g);\n", ctype(g.col_dtype(c)), c, c);
    }
    for (int c : pred_null) s += valid_vec(c);
    s += "  }\n";
    s += "  __device__ static __forceinline__ void load1_pred(Rows &r, const fq_launch_params &p, fq_u64 row) {\n";
    for (int c : pred_cols) {
      if (d.generated && c == 0) s += "    r.c0[0] = p.numbers_begin + row;\n";
      else s += fmt("    r.c%d[0] = fq_ld1<%s>(p.cols[%d], row);\n", c, ctype(g.col_dtype(c)), c);
    }
    for (int c : pred_null) s += valid_one(c);
    s += "  }\n";
    out->sel_tma_ok = !pred_cols.empty() && !(d.generated && g.used_cols.count(0)) && !g.used_cols.empty();
    if (out->sel_tma_ok) {
      s += "  template <int HINT = 0> __device__ static __forceinline__ void tma_issue_pred(const fq_launch_params &p, fq_u32 stage, fq_u32 bar, fq_u64 tile, fq_u32 tile_rows) {\n";
      int prefix = 0;
      for (int c : pred_cols) {
        int w = (int)dtype_size(g.col_dtype(c));
        s += fmt("    fq_bulk_g2s<HINT>(stage + tile_rows * %du, (const char *)p.cols[%d] + tile * tile_rows * %dull, tile_rows * %du, bar);\n", prefix, c, w, w);
        prefix += w;
      }
      for (int c : pred_null) {
        if (g.bitmap_col(c)) continue;
        s += fmt("    fq_bulk_g2s<HINT>(stage + tile_rows * %du, (const char *)p.cols_valid[%d] + tile * tile_rows, tile_rows, bar);\n", prefix, c);
        prefix += 1;
      }
      {   // validity bitmaps: tile_rows / 8 bytes each, behind the byte columns (the host stages only 128-row aligned bitmaps)
        int j = 0;
        for (int c : pred_null)
          if (g.bitmap_col(c)) {
            s += fmt("    fq_bulk_g2s<HINT>(stage + tile_rows * %du + %du * (tile_rows >> 3), (const char *)p.cols_valid[%d] + ((p.cols_valid_bit0[%d] + tile * tile_rows) >> 3), tile_rows >> 3, bar);\n",
                     out->pred_row_bytes, j, c, c);
            j++;
          }
        out->pred_row_bitmaps = j;
      }
      s += "  }\n";
      s += "  __device__ static __forceinline__ void load_smem_pred(Rows &r, const fq_launch_params &p, const unsigned char *stage, fq_u32 tile_rows, fq_u32 group, fq_u64 g) {\n";
      prefix = 0;
      for (int c : pred_cols) {
        int w = (int)dtype_size(g.col_dtype(c));
        s += fmt("    fq_lds_vec<%s, V>(r.c%d, stage + (size_t)tile_rows * %d, group);\n", ctype(g.col_dtype(c)), c, prefix);
        prefix += w;
      }
      {
        int j = 0;
        for (int c : pred_null) {
          if (g.bitmap_col(c)) {
            s += fmt("    fq_lds_bits<V>(r.k%d, stage + (size_t)tile_rows * %d + %d * (tile_rows >> 3), group);\n", c, out->pred_row_bytes, j++);
            continue;
          }
          s += fmt("    fq_lds_vec<bool, V>(r.k%d, stage + (size_t)tile_rows * %d, group);\n", c, prefix);
          prefix += 1;
        }
      }
      s += "  }\n";
    }
  }
  // staged (bulk-copy) access: every referenced column must be materialised; validity bytes are staged like a column
  out->tma_ok = !g.used_cols.empty() && !(d.generated && g.used_cols.count(0));
  for (int c : null_cols)
    if (!g.bitmap_col(c)) out->row_bytes += 1;
  s += fmt("  static constexpr int ROW_BYTES = %d;\n", out->row_bytes);
  for (int c : null_cols) out->row_bitmaps += g.bitmap_col(c) ? 1 : 0;
  s += fmt("  __device__ static constexpr fq_u32 stage_bytes(fq_u32 tile_rows) { return tile_rows * %du + %du * (tile_rows >> 3); }\n", out->row_bytes, out->row_bitmaps);
  if (out->tma_ok) {
    s += "  template <int HINT = 0> __device__ static __forceinline__ void tma_issue(const fq_launch_params &p, fq_u32 stage, fq_u32 bar, fq_u64 tile, fq_u32 tile_rows) {\n";
    int prefix = 0;
    for (int c : g.used_cols) {
      int w = (int)dtype_size(g.col_dtype(c));
      s += fmt("    fq_bulk_g2s<HINT>(stage + tile_rows * %du, (const char *)p.cols[%d] + tile * tile_rows * %dull, tile_rows * %du, bar);\n", prefix, c, w, w);
      prefix += w;
    }
    for (int c : null_cols) {
      if (g.bitmap_col(c)) continue;
      s += fmt("    fq_bulk_g2s<HINT>(stage + tile_rows * %du, (const char *)p.cols_valid[%d] + tile * tile_rows, tile_rows, bar);\n", prefix, c);
      prefix += 1;
    }
    {
      int j = 0;
      for (int c : null_cols)
        if (g.bitmap_col(c))
          s += fmt("    fq_bulk_g2s<HINT>(stage + tile_rows * %du + %du * (tile_rows >> 3), (const char *)p.cols_valid[%d] + ((p.cols_valid_bit0[%d] + tile * tile_rows) >> 3), tile_rows >> 3, bar);\n",
                   out->row_bytes, j++, c, c);
    }
    s += "  }\n";
    s += "  __device__ static __forceinline__ void load_smem(Rows &r, const fq_launch_params &p, const unsigned char *stage, fq_u32 tile_rows, fq_u32 group, fq_u64 g) {\n";
    prefix = 0;
    for (int c : g.used_cols) {
      int w = (int)dtype_size(g.col_dtype(c));
      s += fmt("    fq_lds_vec<%s, V>(r.c%d, stage + (size_t)tile_rows * %d, group);\n", ctype(g.col_dtype(c)), c, prefix);
      prefix += w;
    }
    {
      int j = 0;
      for (int c : null_cols) {
        if (g.bitmap_col(c)) {
          s += fmt("    fq_lds_bits<V>(r.k%d, stage + (size_t)tile_rows * %d + %d * (tile_rows >> 3), group);\n", c, out->row_bytes, j++);
          continue;
        }
        s += fmt("    fq_lds_vec<bool, V>(r.k%d, stage + (size_t)tile_rows * %d, group);\n", c, prefix);
        prefix += 1;
      }
    }
    s += "  }\n";
  }
  // WHERE: a NULL predicate keeps nothing
  s += "  __device__ static __forceinline__ bool pred(const fq_launch_params &p, const Rows &r, int v, fq_u32 &err) {\n";
  if (out->has_pred) {
    Gen::Emitter e(g, "    ");
    e.node(d.predicate);
    s += e.body + "    return " + Gen::Emitter::conj({e.val[d.predicate], e.ok[d.predicate]}) + ";\n  }\n";
  } else {
    s += "    return true;\n  }\n";
  }

  if (groupby) {
    // ---- hash aggregation: per row the packed key and the encoded value of every leaf; per group G 8-byte slots ----
    const int n = n_leaves;
    auto is_f = [&](int k) { return is_float(out->agg_dtypes[k]); };
    auto is_s = [&](int k) { return is_signed_int(out->agg_dtypes[k]); };
    const bool wide = out->key_words == 2;
    s += fmt("  static constexpr int G = %d;\n", 1 + n_slots);
    s += wide ? "  using Key = fq_gb_key2;\n" : "  using Key = fq_u64;\n";
    s += "  __device__ static __forceinline__ bool gb_row(const fq_launch_params &p, const Rows &r, int v, fq_u32 &err, Key &key, fq_u64 (&val)[NSLOTS > 0 ? NSLOTS : 1], fq_u32 &vmask) {\n";
    if (out->has_pred) s += "    if (!pred(p, r, v, err)) return false;\n";
    {
      Gen::Emitter e(g, "    ");
      std::string st = wide ? "    key.lo = 0ull;\n    key.hi = 0ull;\n    vmask = 0u;\n" : "    key = 0ull;\n    vmask = 0u;\n";
      for (const KeyInfo &ki : keys) {
        e.node(ki.node);
        std::string bits;
        const std::string &x = e.val[ki.node];
        switch (ki.t) {
          case FQ_F32: bits = "(fq_u64)__float_as_uint(" + x + ")"; break;
          case FQ_F64: bits = "(fq_u64)__double_as_longlong(" + x + ")"; break;
          case FQ_BOOL: bits = "(fq_u64)((" + x + ") ? 1u : 0u)"; break;
          default: bits = fmt("(fq_u64)(fq_traits<%s>::unsigned_t)(", ctype(ki.t)) + x + ")";
        }
        if (!wide) {
          if (ki.nullable) st += fmt("    key |= (%s) ? (%s << %d) : (1ull << %d);\n", e.ok[ki.node].c_str(), bits.c_str(), ki.shift, ki.shift + ki.bits);
          else st += fmt("    key |= %s << %d;\n", bits.c_str(), ki.shift);
          continue;
        }
        // two words: the field's value bits at [shift, shift + bits), which may straddle lo / hi, then its null flag
        const std::string b = ki.nullable ? fmt("((%s) ? %s : 0ull)", e.ok[ki.node].c_str(), bits.c_str()) : bits;
        st += "    {\n      const fq_u64 b = " + b + ";\n";
        if (ki.shift < 64) st += fmt("      key.lo |= b << %d;\n", ki.shift);
        if (ki.shift + ki.bits > 64) st += ki.shift < 64 ? fmt("      key.hi |= b >> %d;\n", 64 - ki.shift) : fmt("      key.hi |= b << %d;\n", ki.shift - 64);
        if (ki.nullable) {
          const int f = ki.shift + ki.bits;
          st += fmt("      key.%s |= (%s) ? 0ull : (1ull << %d);\n", f < 64 ? "lo" : "hi", e.ok[ki.node].c_str(), f < 64 ? f : f - 64);
        }
        st += "    }\n";
      }
      for (int k = 0; k < n; k++) {
        const fq_expr_node &an = d.nodes[out->agg_nodes[k]];
        if (an.op == FQ_AGG_COUNT) {
          // Count evaluates (and discards) its argument, function_aggregator.rs:58-66: only its error checks remain
          if (!g.trivial(an.left)) { e.node(an.left); st += "    (void)" + e.val[an.left] + ";\n"; }
          st += fmt("    val[%d] = 0ull;\n", k);
          continue;
        }
        e.node(an.left);
        const std::string &x = e.val[an.left];
        std::string enc;
        if (is_f(k)) enc = an.op == FQ_AGG_SUM ? "(fq_u64)__double_as_longlong((double)(" + x + "))" : "fq_f64_ordered((double)(" + x + "))";
        else if (is_s(k)) enc = "(fq_u64)(fq_i64)(" + x + ")";
        else enc = "(fq_u64)(" + x + ")";
        st += fmt("    val[%d] = %s;\n", k, enc.c_str());
        if (leaf_counted[k]) st += fmt("    vmask |= (%s) ? %uu : 0u;\n", e.ok[an.left].c_str(), 1u << k);
      }
      s += e.body + st;
    }
    s += "    return true;\n  }\n";
    // identities of a fresh group
    s += "  __device__ static __forceinline__ void gb_init(fq_u64 *slots) {\n    slots[0] = 0ull;\n";
    for (int k = 0; k < n; k++) {
      const int op = out->agg_ops[k];
      const char *idn = (op == FQ_AGG_SUM || op == FQ_AGG_COUNT) ? "0ull"
                        : op == FQ_AGG_MIN ? (is_s(k) ? "(fq_u64)9223372036854775807ll" : "~0ull")
                                           : (is_s(k) ? "(fq_u64)(-9223372036854775807ll - 1)" : "0ull");
      s += fmt("    slots[%d] = %s;\n", 1 + k, idn);
      if (leaf_counted[k]) s += fmt("    slots[%d] = 0ull;\n", 1 + out->agg_count_slot[k]);
    }
    s += "  }\n";
    // a row as a group state st[G]: rows, leaves, valid counts
    s += "  __device__ static __forceinline__ void gb_one(fq_u64 (&st)[G], const fq_u64 (&val)[NSLOTS > 0 ? NSLOTS : 1], fq_u32 vmask) {\n    st[0] = 1ull;\n";
    for (int k = 0; k < n; k++) {
      s += fmt("    st[%d] = val[%d];\n", 1 + k, k);
      if (leaf_counted[k]) s += fmt("    st[%d] = (vmask >> %d) & 1u;\n", 1 + out->agg_count_slot[k], k);
    }
    s += "  }\n";
    // a group state into a group of a table.  gb_merge: the table in HBM (native 64-bit ATOMG).  gb_merge_s: the CTA's table
    // in shared memory — sm_100a has no 64-bit shared-memory atomics (the compiler emits ATOMS.CAST.SPIN loops, which under
    // contention cost hundreds of instructions per row), so counts and wrapping integer sums go through native 32-bit
    // atomics: low word first, and whoever sees it wrap carries one into the high word (exact mod 2^64 in any order).
    for (int pass = 0; pass < 2; pass++) {
      const bool shared = pass == 1;
      s += shared ? "  __device__ static __forceinline__ void gb_merge_s(fq_u64 *slots, const fq_u64 *src) {\n"
                  : "  __device__ static __forceinline__ void gb_merge(fq_u64 *slots, const fq_u64 *src) {\n";
      auto add64 = [&](int slot, const std::string &x) {
        return shared ? fmt("fq_atom_add64_s(slots + %d, %s);", slot, x.c_str())
                      : fmt("atomicAdd((unsigned long long *)(slots + %d), (unsigned long long)%s);", slot, x.c_str());
      };
      s += "    " + add64(0, "src[0]") + "\n";
      for (int k = 0; k < n; k++) {
        const int op = out->agg_ops[k];
        if (op == FQ_AGG_COUNT) continue;
        const std::string x = fmt("src[%d]", 1 + k);
        std::string stmt;
        if (op == FQ_AGG_SUM) {
          stmt = is_f(k) ? fmt("atomicAdd((double *)(slots + %d), __longlong_as_double((fq_i64)%s));", 1 + k, x.c_str()) : add64(1 + k, x);
        } else {
          // after the first rows of a group a new minimum / maximum is rare: look before paying for the atomic
          const char *f = op == FQ_AGG_MIN ? "atomicMin" : "atomicMax";
          const char *cmp = op == FQ_AGG_MIN ? "<" : ">";
          stmt = is_s(k) ? fmt("if ((long long)%s %s *(volatile long long *)(slots + %d)) %s((long long *)(slots + %d), (long long)%s);", x.c_str(), cmp,
                               1 + k, f, 1 + k, x.c_str())
                         : fmt("if ((unsigned long long)%s %s *(volatile unsigned long long *)(slots + %d)) %s((unsigned long long *)(slots + %d), (unsigned long long)%s);",
                               x.c_str(), cmp, 1 + k, f, 1 + k, x.c_str());
        }
        if (leaf_counted[k]) {
          const int cs = 1 + out->agg_count_slot[k];
          s += fmt("    if (src[%d]) { %s %s }\n", cs, stmt.c_str(), add64(cs, fmt("src[%d]", cs)).c_str());
        } else {
          s += "    " + stmt + "\n";
        }
      }
      s += "  }\n";
    }
  } else if (d.kind == FQ_PIPE_AGGREGATE) {
    const int n = n_leaves;
    s += "  struct Acc {";
    for (int k = 0; k < n; k++) s += fmt(" %s a%d;", ctype(out->agg_dtypes[k]), k);
    for (int k = 0; k < n; k++)
      if (leaf_counted[k]) s += fmt(" fq_u64 c%d;", k);
    s += " };\n";
    s += "  __device__ static __forceinline__ void init(Acc &a) {\n";
    for (int k = 0; k < n; k++) s += fmt("    a.a%d = %s;\n", k, identity_of(out->agg_ops[k], out->agg_dtypes[k]).c_str());
    for (int k = 0; k < n; k++)
      if (leaf_counted[k]) s += fmt("    a.c%d = 0;\n", k);
    s += "  }\n";
    s += "  __device__ static __forceinline__ bool consume(const fq_launch_params &p, Acc &a, const Rows &r, int v, fq_u64 &nsel, fq_u32 &err) {\n";
    if (out->has_pred) s += "    if (!pred(p, r, v, err)) return false;\n    nsel += 1;\n";
    {
      Gen::Emitter e(g, "    ");
      std::string upd;
      for (int k = 0; k < n; k++) {
        const fq_expr_node &an = d.nodes[out->agg_nodes[k]];
        const char *T = ctype(out->agg_dtypes[k]);
        if (an.op == FQ_AGG_COUNT) {
          // Count evaluates (and discards) its argument, function_aggregator.rs:58-66: only its error checks remain
          if (!g.trivial(an.left)) { e.node(an.left); upd += "    (void)" + e.val[an.left] + ";\n"; }
          continue;
        }
        e.node(an.left);
        const char *f = an.op == FQ_AGG_SUM ? "fq_add" : an.op == FQ_AGG_MIN ? "fq_min" : "fq_max";
        std::string step = fmt("a.a%d = %s<%s>(a.a%d, ", k, f, T, k) + e.val[an.left] + ");";
        if (leaf_counted[k]) upd += "    if (" + e.ok[an.left] + ") { " + step + fmt(" a.c%d += 1; }\n", k);
        else upd += "    " + step + "\n";
      }
      s += e.body + upd;
    }
    s += "    return true;\n  }\n";
    s += "  __device__ static __forceinline__ void merge(Acc &a, const Acc &b) {\n";
    for (int k = 0; k < n; k++) {
      const char *T = ctype(out->agg_dtypes[k]);
      const char *f = out->agg_ops[k] == FQ_AGG_MIN ? "fq_min" : out->agg_ops[k] == FQ_AGG_MAX ? "fq_max" : "fq_add";
      s += fmt("    a.a%d = %s<%s>(a.a%d, b.a%d);\n", k, f, T, k, k);
      if (leaf_counted[k]) s += fmt("    a.c%d += b.c%d;\n", k, k);
    }
    s += "  }\n";
    s += "  __device__ static __forceinline__ void shfl(Acc &a, int m) {\n";
    for (int k = 0; k < n; k++) {
      s += fmt("    a.a%d = fq_shfl_xor<%s>(a.a%d, m);\n", k, ctype(out->agg_dtypes[k]), k);
      if (leaf_counted[k]) s += fmt("    a.c%d = fq_shfl_xor<fq_u64>(a.c%d, m);\n", k, k);
    }
    s += "  }\n";
    s += "  __device__ static __forceinline__ void store(const Acc &a, fq_u64 *o) {\n";
    for (int k = 0; k < n; k++) {
      s += fmt("    o[%d] = fq_pack<%s>(a.a%d);\n", k, ctype(out->agg_dtypes[k]), k);
      if (leaf_counted[k]) s += fmt("    o[%d] = a.c%d;\n", out->agg_count_slot[k], k);
    }
    s += "  }\n";
    s += "  __device__ static __forceinline__ void unpack(Acc &a, const fq_u64 *o) {\n";
    for (int k = 0; k < n; k++) {
      s += fmt("    a.a%d = fq_unpack<%s>(o[%d]);\n", k, ctype(out->agg_dtypes[k]), k);
      if (leaf_counted[k]) s += fmt("    a.c%d = o[%d];\n", k, out->agg_count_slot[k]);
    }
    s += "  }\n";
  } else {
    s += "  __device__ static __forceinline__ void emit(const Rows &r, int v, const fq_launch_params &p, fq_u64 pos, fq_u32 &err) {\n";
    {
      Gen::Emitter e(g, "    ");
      std::string st;
      for (int x = 0; x < d.n_exprs; x++) {
        fq_dtype t = out->expr_dtypes[x];
        e.node(d.exprs[x]);
        st += fmt("    fq_st1<%s>(p.outs[%d], pos, ", t == FQ_BOOL ? "fq_u8" : ctype(t), x) + e.val[d.exprs[x]] + ");\n";
        if (out->expr_nullable[x]) st += fmt("    fq_st1<fq_u8>(p.outs_valid[%d], pos, ", x) + e.ok[d.exprs[x]] + ");\n";
      }
      s += e.body + st;
    }
    s += "  }\n";
    // whole vector group at once (projection without a filter): V values per output column, one vector store each
    s += "  __device__ static __forceinline__ void emit_vec(const Rows &r, const fq_launch_params &p, fq_u64 row0, fq_u32 &err) {\n";
    for (int x = 0; x < d.n_exprs; x++) {
      fq_dtype t = out->expr_dtypes[x];
      s += fmt("    %s o%d[V];\n", t == FQ_BOOL ? "fq_u8" : ctype(t), x);
      if (out->expr_nullable[x]) s += fmt("    fq_u8 q%d[V];\n", x);
    }
    s += "#pragma unroll\n    for (int v = 0; v < V; v++) {\n";
    {
      Gen::Emitter e(g, "      ");
      std::string st;
      for (int x = 0; x < d.n_exprs; x++) {
        e.node(d.exprs[x]);
        st += fmt("      o%d[v] = ", x) + e.val[d.exprs[x]] + ";\n";
        if (out->expr_nullable[x]) st += fmt("      q%d[v] = ", x) + e.ok[d.exprs[x]] + ";\n";
      }
      s += e.body + st;
    }
    s += "    }\n";
    for (int x = 0; x < d.n_exprs; x++) {
      fq_dtype t = out->expr_dtypes[x];
      s += fmt("    fq_store_vec<%s, V>(p.outs[%d], row0, o%d);\n", t == FQ_BOOL ? "fq_u8" : ctype(t), x, x);
      if (out->expr_nullable[x]) s += fmt("    fq_store_vec<fq_u8, V>(p.outs_valid[%d], row0, q%d);\n", x, x);
    }
    s += "  }\n";
  }
  s += "};\n";
  // kernel wrappers: the ahead-of-time build compiles all of them, a JIT build only the variant it will launch
  std::vector<std::pair<std::string, std::string>> wrappers;
  if (groupby) {
    wrappers.push_back({"_groupby", "extern \"C\" __global__ void __launch_bounds__(FQ_GB_THREADS, FQ_GB_MIN_BLOCKS) fqk_@_groupby(const __grid_constant__ fq_launch_params p) { fq_groupby_kernel<Q_@, FQ_GB_UNROLL>(p); }\n"});
    wrappers.push_back({"_gbmerge", "extern \"C\" __global__ void __launch_bounds__(256) fqk_@_gbmerge(const __grid_constant__ fq_launch_params p) { fq_groupby_merge_kernel<Q_@>(p); }\n"});
  } else if (d.kind == FQ_PIPE_AGGREGATE) {
    wrappers.push_back({"_agg_u4", "extern \"C\" __global__ void __launch_bounds__(FQ_AGG_THREADS, FQ_AGG_MIN_BLOCKS) fqk_@_agg_u4(const __grid_constant__ fq_launch_params p) { fq_agg_kernel<Q_@, 4>(p); }\n"});
    if (out->tma_ok)
      wrappers.push_back({"_agg_tma", "extern \"C\" __global__ void __launch_bounds__(FQ_TMA_THREADS + 32, FQ_TMA_MIN_BLOCKS) fqk_@_agg_tma(const __grid_constant__ fq_launch_params p) { fq_agg_tma_kernel<Q_@, FQ_TMA_UNROLL, FQ_TMA_STAGES>(p); }\n"});
  } else if (out->has_pred) {
    wrappers.push_back({"_select", "extern \"C\" __global__ void __launch_bounds__(FQ_SEL_THREADS + 32, FQ_SEL_MIN_BLOCKS) fqk_@_select(const __grid_constant__ fq_launch_params p) { fq_select_kernel<Q_@, fq_sel_shape<Q_@::V>::U, fq_sel_shape<Q_@::V>::SEG>(p); }\n"});
    if (out->sel_tma_ok) {
      wrappers.push_back({"_select_tma", "extern \"C\" __global__ void __launch_bounds__(FQ_SELT_THREADS + 64, 1) fqk_@_select_tma(const __grid_constant__ fq_launch_params p) { fq_select_tma_kernel<Q_@, fq_selt_shape<Q_@::V>::U, fq_selt_shape<Q_@::V>::SEG, FQ_SELT_STAGES, false>(p); }\n"});
      wrappers.push_back({"_select_dense", "extern \"C\" __global__ void __launch_bounds__(FQ_SELD_THREADS + 64, 1) fqk_@_select_dense(const __grid_constant__ fq_launch_params p) { fq_select_tma_kernel<Q_@, fq_seld_shape<Q_@::V>::U, fq_seld_shape<Q_@::V>::SEG, 16, true>(p); }\n"});
      wrappers.push_back({"_select_probe", "extern \"C\" __global__ void __launch_bounds__(128) fqk_@_select_probe(const __grid_constant__ fq_launch_params p) { fq_select_probe_kernel<Q_@>(p); }\n"});
    }
  } else {
    wrappers.push_back({"_map", "extern \"C\" __global__ void __launch_bounds__(FQ_MAP_THREADS, FQ_MAP_MIN_BLOCKS) fqk_@_map(const __grid_constant__ fq_launch_params p) { fq_map_kernel<Q_@, FQ_MAP_UNROLL>(p); }\n"});
    if (out->tma_ok)
      wrappers.push_back({"_map_tma", "extern \"C\" __global__ void __launch_bounds__(FQ_TMA_THREADS + 32, FQ_TMA_MIN_BLOCKS) fqk_@_map_tma(const __grid_constant__ fq_launch_params p) { fq_map_tma_kernel<Q_@, FQ_TMA_UNROLL, FQ_TMA_STAGES>(p); }\n"});
  }
  const std::string struct_text = s;
  for (auto &w : wrappers) s += w.second;

  if (g.status != FQ_OK) { *err = g.err; return g.status; }
  out->const_divide_by_zero = g.const_div0;
  char tag[32];
  snprintf(tag, sizeof tag, "%016" PRIx64, fnv1a(s));
  out->tag = tag;
  auto with_tag = [&](const std::string &text) {
    std::string src;
    for (char c : text) {
      if (c == '@') src += out->tag; else src += c;
    }
    return src;
  };
  out->source = with_tag(s);
  out->struct_source = with_tag(struct_text);
  out->kernels.clear();
  for (auto &w : wrappers) out->kernels.push_back({w.first, with_tag(w.second)});
  out->node_dtypes = g.ty;
  return FQ_OK;
}

// ---------------------------------------------------------------------------------------------
// s-expression reader (build-time AOT list, C++ tests)
// ---------------------------------------------------------------------------------------------
namespace {
struct SexprParser {
  const std::string &t;
  size_t i = 0;
  const std::vector<std::string> &cols;
  std::vector<fq_expr_node> *nodes;
  std::string err;

  std::string tok() {
    while (i < t.size() && isspace((unsigned char)t[i])) i++;
    size_t b = i;
    if (i < t.size() && (t[i] == '(' || t[i] == ')')) { i++; return t.substr(b, 1); }
    while (i < t.size() && !isspace((unsigned char)t[i]) && t[i] != '(' && t[i] != ')') i++;
    // a NaN with a payload is written as strtod reads it, `nan(0x...)`: the parenthesis belongs to the token
    const std::string w = t.substr(b, i - b);
    if (i < t.size() && t[i] == '(' && (w == "nan" || w == "-nan" || w == "+nan")) {
      const size_t close = t.find(')', i);
      if (close != std::string::npos) i = close + 1;
    }
    return t.substr(b, i - b);
  }
  int push(fq_expr_node n) { nodes->push_back(n); return (int)nodes->size() - 1; }
  int parse() {
    if (tok() != "(") { err = "expected ("; return -1; }
    std::string h = tok();
    fq_expr_node n;
    memset(&n, 0, sizeof n);
    n.left = n.right = -1;
    static const struct { const char *name; int kind, op; } ops[] = {
        {"+", FQ_EXPR_ARITHMETIC, FQ_AR_ADD}, {"-", FQ_EXPR_ARITHMETIC, FQ_AR_SUB}, {"*", FQ_EXPR_ARITHMETIC, FQ_AR_MUL},
        {"/", FQ_EXPR_ARITHMETIC, FQ_AR_DIV}, {"=", FQ_EXPR_COMPARISON, FQ_CMP_EQ}, {"<", FQ_EXPR_COMPARISON, FQ_CMP_LT},
        {"<=", FQ_EXPR_COMPARISON, FQ_CMP_LTEQ}, {">", FQ_EXPR_COMPARISON, FQ_CMP_GT}, {">=", FQ_EXPR_COMPARISON, FQ_CMP_GTEQ},
        {"and", FQ_EXPR_LOGIC, FQ_LG_AND}, {"or", FQ_EXPR_LOGIC, FQ_LG_OR}, {"min", FQ_EXPR_AGGREGATOR, FQ_AGG_MIN},
        {"max", FQ_EXPR_AGGREGATOR, FQ_AGG_MAX}, {"sum", FQ_EXPR_AGGREGATOR, FQ_AGG_SUM}, {"count", FQ_EXPR_AGGREGATOR, FQ_AGG_COUNT}};
    static const struct { const char *name; fq_dtype t; } tys[] = {
        {"bool", FQ_BOOL}, {"i8", FQ_I8}, {"i16", FQ_I16}, {"i32", FQ_I32}, {"i64", FQ_I64}, {"u8", FQ_U8},
        {"u16", FQ_U16}, {"u32", FQ_U32}, {"u64", FQ_U64}, {"f32", FQ_F32}, {"f64", FQ_F64}};
    bool done = false;
    if (h == "col") {
      std::string name = tok();
      n.kind = FQ_EXPR_FIELD;
      n.column = -1;
      for (size_t c = 0; c < cols.size(); c++) if (cols[c] == name) n.column = (int)c;
      if (n.column < 0) { err = "unknown column " + name; return -1; }
      done = true;
    } else if (h == "alias") {
      tok();
      n.kind = FQ_EXPR_ALIAS;
      n.left = parse();
      if (n.left < 0) return -1;
      done = true;
    } else if (h == "lookup") {   // (lookup <slot> <index expression>)
      n.kind = FQ_EXPR_LOOKUP;
      n.op = (int)strtol(tok().c_str(), nullptr, 10);
      n.left = parse();
      if (n.left < 0) return -1;
      done = true;
    }
    for (auto &ty : tys)
      if (!done && h == ty.name) {
        std::string lit = tok();
        n.kind = FQ_EXPR_CONSTANT;
        n.dtype = ty.t;
        if (ty.t == FQ_BOOL) n.value.i = lit == "true";
        else if (is_float(ty.t)) n.value.f = ty.t == FQ_F32 ? (double)strtof(lit.c_str(), nullptr) : strtod(lit.c_str(), nullptr);
        else if (is_signed_int(ty.t)) n.value.i = strtoll(lit.c_str(), nullptr, 10);
        else n.value.u = strtoull(lit.c_str(), nullptr, 10);
        done = true;
      }
    for (auto &o : ops)
      if (!done && h == o.name) {
        n.kind = o.kind;
        n.op = o.op;
        n.left = parse();
        if (n.left < 0) return -1;
        if (o.kind != FQ_EXPR_AGGREGATOR) {
          n.right = parse();
          if (n.right < 0) return -1;
        }
        done = true;
      }
    if (!done) { err = "unknown head " + h; return -1; }
    if (tok() != ")") { err = "expected )"; return -1; }
    return push(n);
  }
};
}  // namespace

int parse_sexpr(const std::string &text, const std::vector<std::string> &cols, std::vector<fq_expr_node> *nodes, int *root,
                std::string *err) {
  SexprParser p{text, 0, cols, nodes, {}};
  int r = p.parse();
  if (r < 0) { *err = "Error during plan: " + p.err + " in `" + text + "`"; return FQ_ERR_PLAN; }
  *root = r;
  return FQ_OK;
}

}  // namespace fq
