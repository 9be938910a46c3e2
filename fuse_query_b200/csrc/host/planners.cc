// planners.cc — host mirror of src/planners + src/optimizers: SQL text -> PlanNode tree -> alias rewrite.
// Pure host logic (microseconds per query); it only exists so that the reference's plan_select /
// executor_select entry points accept the README queries unchanged and drive the GPU pipeline.
#include <algorithm>
#include <cctype>
#include <cstring>

#include "fq_host.h"

namespace fuse {

// ---------------------------------------------------------------------------------------------
// ExpressionPlan — plan_expression.rs
// ---------------------------------------------------------------------------------------------
FunctionRef ExpressionPlan::to_function(size_t depth) const {   // plan_to_function, :40-71
  switch (kind) {
    case Field: return Function::FieldFunction(name);
    case Constant: return Function::ConstantFunction(value);
    case BinaryExpression: {
      FunctionRef l = args[0].to_function(depth), r = args[1].to_function(depth + 1);
      FunctionRef f = Function::factory_get(name, {l, r});
      f->set_depth(depth);
      return f;
    }
    case Function: {
      std::vector<FunctionRef> funcs;
      for (const auto &a : args) {
        FunctionRef f = a.to_function(depth + 1);
        f->set_depth(depth);
        funcs.push_back(f);
      }
      FunctionRef f = Function::factory_get(name, funcs);
      f->set_depth(depth);
      return f;
    }
    case Alias: {
      FunctionRef f = args[0].to_function(depth);
      f->set_depth(depth);
      return Function::AliasFunction(name, f);
    }
    default: throw FuseQueryError::internal("Cannot transform wildcard to function");
  }
}
DataField ExpressionPlan::to_field(const DataSchema &input_schema) const {   // :31-38
  FunctionRef f = to_function();
  return DataField{f->to_string(), f->return_type(input_schema), f->nullable(input_schema)};
}
bool ExpressionPlan::is_aggregate() const {   // :77-89
  switch (kind) {
    case Alias: return args[0].is_aggregate();
    case BinaryExpression: return args[0].is_aggregate() || args[1].is_aggregate();
    case Function: {
      std::string n = name;
      std::transform(n.begin(), n.end(), n.begin(), ::tolower);
      return n == "max" || n == "min" || n == "avg" || n == "count" || n == "sum";
    }
    default: return false;
  }
}
std::string ExpressionPlan::to_string() const {   // Debug, :92-105
  switch (kind) {
    case Alias: return args[0].to_string() + " as " + name;
    case Field: return name;
    case Constant: return value.to_string();
    case BinaryExpression: return "(" + args[0].to_string() + " " + name + " " + args[1].to_string() + ")";
    case Function: {
      std::string o = name + "([";
      for (size_t i = 0; i < args.size(); i++) o += (i ? ", " : "") + args[i].to_string();
      return o + "])";
    }
    default: return "*";
  }
}

// ---------------------------------------------------------------------------------------------
// PlanNode — plan_node.rs, plan_display.rs
// ---------------------------------------------------------------------------------------------
DataSchemaRef PlanNode::schema() const {
  switch (kind) {
    case Filter: case Limit: case Select: case Sort: return input->schema();   // plan_filter.rs / plan_limit.rs forward the input schema
    case Explain: throw FuseQueryError::internal("not implemented");   // unimplemented!() in the reference
    default: return schema_ ? schema_ : std::make_shared<DataSchema>();
  }
}
const char *PlanNode::name() const {
  static const char *n[] = {"EmptyPlan", "ProjectionPlan", "AggregatePlan", "FilterPlan", "LimitPlan", "ScanPlan", "ReadSourcePlan", "ExplainPlan", "SelectPlan", "SortPlan"};
  return n[kind];
}
static std::vector<PlanNode> to_array(const PlanNode &root, bool with_parent) {   // plan_node.rs:55-125
  std::vector<PlanNode> result;
  const PlanNode *plan = &root;
  for (int depth = 0;; depth++) {
    if (depth > 128) throw FuseQueryError::plan("PlanNode depth more than 128");
    bool stop = false;
    switch (plan->kind) {
      case PlanNode::Aggregate: case PlanNode::Projection: case PlanNode::Filter: case PlanNode::Limit: case PlanNode::Sort:
        result.push_back(*plan);
        plan = plan->input.get();
        break;
      case PlanNode::Select: case PlanNode::Explain:
        if (with_parent) result.push_back(*plan);
        plan = plan->input.get();
        break;
      case PlanNode::Empty: stop = true; break;
      default: result.push_back(*plan); stop = true;
    }
    if (stop || !plan) break;
  }
  std::reverse(result.begin(), result.end());
  return result;
}
std::vector<PlanNode> PlanNode::children_to_plans() const { return to_array(*this, false); }
std::vector<PlanNode> PlanNode::node_to_plans() const { return to_array(*this, true); }
PlanNode PlanNode::plans_to_node(const std::vector<PlanNode> &plans) {   // :135-162
  PlanBuilder b = PlanBuilder::empty(false);
  for (const auto &p : plans) {
    switch (p.kind) {
      case Projection: b = b.project(p.expr); break;
      case Aggregate: b = b.aggregate(p.group_expr, p.expr); break;
      case Filter: b = b.filter(p.predicate); break;
      case Limit: b = b.limit(p.n); break;
      case Sort: b = b.sort(p.expr, p.descending); break;
      case ReadSource: b = PlanBuilder::from(p); break;
      case Explain: b = b.explain(); break;
      case Select: b = b.select(); break;
      default: break;
    }
  }
  return b.build();
}
std::string PlanNode::to_string() const {   // plan_display.rs:66-88
  std::vector<PlanNode> plans = children_to_plans();
  std::reverse(plans.begin(), plans.end());
  std::string out;
  size_t indent = 0;
  for (const auto &node : plans) {
    if (indent > 0) {
      out += "\n";
      for (size_t i = 0; i < indent; i++) out += "  ";
    }
    const std::string prefix = "└─";   // └─
    switch (node.kind) {
      case Projection:
        out += prefix + " Projection: ";
        for (size_t i = 0; i < node.expr.size(); i++) out += (i ? ", " : "") + node.expr[i].to_string();
        break;
      case Aggregate:
        out += prefix + " Aggregate: ";
        for (size_t i = 0; i < node.expr.size(); i++) out += (i ? ", " : "") + node.expr[i].to_string();
        for (size_t i = 0; i < node.group_expr.size(); i++) out += (i ? ", " : "") + node.group_expr[i].to_string();
        break;
      case Filter: out += prefix + " Filter: " + node.predicate.to_string(); break;
      case Limit: out += prefix + " Limit: " + std::to_string(node.n); break;
      case Sort:
        out += prefix + " Sort: ";
        for (size_t i = 0; i < node.expr.size(); i++) out += (i ? ", " : "") + node.expr[i].to_string() + (node.descending[i] ? " desc" : "");
        break;
      case ReadSource:
        out += prefix + " ReadDataSource: scan parts [" + std::to_string(node.partitions.size()) + "]" + node.description;
        break;
      default: break;
    }
    indent++;
  }
  return out;
}

// ---------------------------------------------------------------------------------------------
// PlanBuilder — plan_builder.rs
// ---------------------------------------------------------------------------------------------
PlanBuilder PlanBuilder::create(DataSchemaRef schema) {
  PlanNode p;
  p.kind = PlanNode::Empty;
  p.schema_ = std::move(schema);
  return PlanBuilder(p);
}
PlanBuilder PlanBuilder::empty(bool) { return create(std::make_shared<DataSchema>()); }
PlanBuilder PlanBuilder::scan(const std::string &schema_name, const std::string &, const DataSchema &table_schema,
                              std::optional<ExpressionPlan> table_args) {
  PlanNode p;
  p.kind = PlanNode::Scan;
  p.schema_name = schema_name;
  p.schema_ = std::make_shared<DataSchema>(table_schema);
  p.table_args = std::move(table_args);
  return PlanBuilder(p);
}
PlanBuilder PlanBuilder::project(const std::vector<ExpressionPlan> &exprs) const {   // :38-61
  DataSchemaRef in = plan_.schema();
  PlanNode p;
  p.kind = PlanNode::Projection;
  for (const auto &e : exprs) {
    if (e.kind == ExpressionPlan::Wildcard)
      for (const auto &f : in->fields) p.expr.push_back(ExpressionPlan::field(f.name));
    else p.expr.push_back(e);
  }
  auto schema = std::make_shared<DataSchema>();
  for (const auto &e : p.expr) schema->fields.push_back(e.to_field(*in));
  p.schema_ = schema;
  p.input = std::make_shared<PlanNode>(plan_);
  return PlanBuilder(p);
}
PlanBuilder PlanBuilder::aggregate(const std::vector<ExpressionPlan> &group_expr, const std::vector<ExpressionPlan> &aggr_expr) const {   // :64-83
  DataSchemaRef in = plan_.schema();
  PlanNode p;
  p.kind = PlanNode::Aggregate;
  p.group_expr = group_expr;
  p.expr = aggr_expr;
  auto schema = std::make_shared<DataSchema>();
  for (const auto &e : group_expr) schema->fields.push_back(e.to_field(*in));
  for (const auto &e : aggr_expr) schema->fields.push_back(e.to_field(*in));
  p.schema_ = schema;
  p.input = std::make_shared<PlanNode>(plan_);
  return PlanBuilder(p);
}
PlanBuilder PlanBuilder::filter(const ExpressionPlan &expr) const {
  PlanNode p;
  p.kind = PlanNode::Filter;
  p.predicate = expr;
  p.input = std::make_shared<PlanNode>(plan_);
  return PlanBuilder(p);
}
PlanBuilder PlanBuilder::limit(size_t n) const {
  PlanNode p;
  p.kind = PlanNode::Limit;
  p.n = n;
  p.input = std::make_shared<PlanNode>(plan_);
  return PlanBuilder(p);
}
PlanBuilder PlanBuilder::sort(const std::vector<ExpressionPlan> &keys, const std::vector<bool> &descending) const {
  DataSchemaRef in = plan_.schema();
  PlanNode p;
  p.kind = PlanNode::Sort;
  for (const auto &e : keys) {
    if (e.is_aggregate())
      throw FuseQueryError::plan("ORDER BY sorts the query's output columns: name the aggregate's column (or its alias) instead of " + e.to_string());
    (void)e.to_field(*in);   // every column a key names must be an output column of the input plan
  }
  p.expr = keys;
  p.descending = descending;
  p.descending.resize(keys.size(), false);
  p.input = std::make_shared<PlanNode>(plan_);
  return PlanBuilder(p);
}
PlanBuilder PlanBuilder::select() const {
  PlanNode p;
  p.kind = PlanNode::Select;
  p.input = std::make_shared<PlanNode>(plan_);
  return PlanBuilder(p);
}
PlanBuilder PlanBuilder::explain() const {
  PlanNode p;
  p.kind = PlanNode::Explain;
  p.input = std::make_shared<PlanNode>(plan_);
  return PlanBuilder(p);
}

// ---------------------------------------------------------------------------------------------
// SQL front end.  The reference uses sqlparser 0.6 (+ DataFusion's DFParser for EXPLAIN,
// planners/parser.rs:92-185); this recursive-descent parser accepts the SELECT subset the planner
// supports (plan_parser.rs:90-133) and produces what sql_to_rex would (plan_parser.rs:216-262).
// ---------------------------------------------------------------------------------------------
namespace {
struct Tok { enum K { Word, Number, String, Sym, End } k; std::string text; };

std::vector<Tok> lex(const std::string &sql) {
  std::vector<Tok> out;
  size_t i = 0;
  while (i < sql.size()) {
    char c = sql[i];
    if (isspace((unsigned char)c)) { i++; continue; }
    if (isalpha((unsigned char)c) || c == '_') {
      size_t b = i;
      while (i < sql.size() && (isalnum((unsigned char)sql[i]) || sql[i] == '_')) i++;
      out.push_back({Tok::Word, sql.substr(b, i - b)});
    } else if (isdigit((unsigned char)c) || (c == '.' && i + 1 < sql.size() && isdigit((unsigned char)sql[i + 1]))) {
      size_t b = i;
      while (i < sql.size() && (isdigit((unsigned char)sql[i]) || sql[i] == '.')) i++;
      out.push_back({Tok::Number, sql.substr(b, i - b)});
    } else if (c == '\'') {
      size_t b = ++i;
      while (i < sql.size() && sql[i] != '\'') i++;
      if (i >= sql.size()) throw FuseQueryError::sql("sql parser error: Unterminated string literal");
      out.push_back({Tok::String, sql.substr(b, i - b)});
      i++;
    } else {
      static const char *two[] = {"<=", ">=", "<>", "!="};
      std::string s(1, c);
      for (const char *t : two)
        if (sql.compare(i, 2, t) == 0) s = t;
      out.push_back({Tok::Sym, s});
      i += s.size();
    }
  }
  out.push_back({Tok::End, "EOF"});
  return out;
}

// sqlparser's Display of an expression it parsed but sql_to_rex refuses (plan_parser.rs:262-265 formats the AST, not the
// ExpressionPlan): binary operators without added parentheses, functions as name(args).  Parentheses of the original
// text are not kept by this parser, so `NOT (a > 1)` prints as `NOT a > 1`.
static std::string sql_display(const ExpressionPlan &e) {
  switch (e.kind) {
    case ExpressionPlan::Field: return e.name;
    case ExpressionPlan::Constant: return e.value.data_type() == FQ_UTF8 ? "'" + e.value.to_string() + "'" : e.value.to_string();
    case ExpressionPlan::BinaryExpression: return sql_display(e.args[0]) + " " + e.name + " " + sql_display(e.args[1]);
    case ExpressionPlan::Function: {
      std::string out = e.name + "(";
      for (size_t i = 0; i < e.args.size(); i++) out += (i ? ", " : "") + sql_display(e.args[i]);
      return out + ")";
    }
    case ExpressionPlan::Alias: return sql_display(e.args[0]) + " AS " + e.name;
    default: return "*";
  }
}

struct SqlParser {
  std::vector<Tok> t;
  size_t p = 0;
  // nesting of parentheses / function calls / derived tables currently open: the parser is recursive-descent, so a query
  // of 20 000 opening parentheses would otherwise overflow the host stack long before any plan check runs
  int nesting = 0;
  struct Nest {
    SqlParser &sp;
    explicit Nest(SqlParser &s, const char *what) : sp(s) {
      if (++sp.nesting > ExpressionPlan::kMaxDepth) { --sp.nesting; throw FuseQueryError::plan(std::string(what) + " depth more than 128"); }
    }
    ~Nest() { --sp.nesting; }
  };
  const Tok &peek() const { return t[p]; }
  bool is_kw(const char *kw) const {
    if (peek().k != Tok::Word) return false;
    std::string w = peek().text;
    std::transform(w.begin(), w.end(), w.begin(), ::toupper);
    return w == kw;
  }
  bool eat_kw(const char *kw) { if (is_kw(kw)) { p++; return true; } return false; }
  bool eat_sym(const char *s) { if (peek().k == Tok::Sym && peek().text == s) { p++; return true; } return false; }
  [[noreturn]] void expected(const std::string &what) { throw FuseQueryError::sql("sql parser error: Expected " + what + ", found: " + peek().text); }
  void expect_sym(const char *s) { if (!eat_sym(s)) expected(s); }

  static bool reserved(const std::string &w0) {
    std::string w = w0;
    std::transform(w.begin(), w.end(), w.begin(), ::toupper);
    static const char *kws[] = {"FROM", "WHERE", "GROUP", "HAVING", "LIMIT", "ORDER", "AS", "AND", "OR", "BY", "SELECT", "UNION", "ASC", "DESC"};
    for (const char *k : kws) if (w == k) return true;
    return false;
  }

  bool next_is_kw(const char *kw) const {
    if (t[p].k == Tok::End || t[p + 1].k != Tok::Word) return false;
    std::string w = t[p + 1].text;
    std::transform(w.begin(), w.end(), w.begin(), ::toupper);
    return w == kw;
  }

  // precedence climbing as sqlparser: OR(5) < AND(10) < comparisons, LIKE, NOT LIKE(20) < + -(30) < * / %(40)
  ExpressionPlan expr(int min_prec = 0) {
    ExpressionPlan lhs = prefix();
    for (;;) {
      int prec = 0, width = 1;
      std::string op;
      if (is_kw("OR")) { prec = 5; op = "OR"; }
      else if (is_kw("AND")) { prec = 10; op = "AND"; }
      else if (is_kw("LIKE")) { prec = 20; op = "LIKE"; }
      else if (is_kw("NOT") && next_is_kw("LIKE")) { prec = 20; op = "NOT LIKE"; width = 2; }
      else if (peek().k == Tok::Sym) {
        const std::string &s = peek().text;
        if (s == "=" || s == "<" || s == ">" || s == "<=" || s == ">=" || s == "<>" || s == "!=") { prec = 20; op = s == "!=" ? "<>" : s; }
        else if (s == "+" || s == "-") { prec = 30; op = s; }
        else if (s == "*" || s == "/" || s == "%") { prec = 40; op = s; }
      }
      if (prec == 0 || prec <= min_prec) return lhs;
      p += width;
      ExpressionPlan rhs = expr(prec);
      lhs = ExpressionPlan::binary(std::move(lhs), op, std::move(rhs));   // op: format!("{}", op), plan_parser.rs:241-247
    }
  }
  ExpressionPlan prefix() {
    const Tok tok = peek();
    if (tok.k == Tok::Number) {   // plan_parser.rs:223-235
      p++;
      bool integral = tok.text.find('.') == std::string::npos;
      if (integral) {
        errno = 0;
        char *end = nullptr;
        long long v = strtoll(tok.text.c_str(), &end, 10);
        if (errno == 0 && *end == 0) return ExpressionPlan::constant(v >= 0 ? DataValue::UInt64((uint64_t)v) : DataValue::Int64(v));
      }
      return ExpressionPlan::constant(DataValue::Float64(strtod(tok.text.c_str(), nullptr)));
    }
    if (tok.k == Tok::String) { p++; return ExpressionPlan::constant(DataValue::String(tok.text)); }
    if (tok.k == Tok::Sym && tok.text == "(") {   // Expr::Nested
      p++;
      Nest nest(*this, "expression");
      ExpressionPlan e = expr();
      expect_sym(")");
      return e;
    }
    if (tok.k == Tok::Sym && (tok.text == "-" || tok.text == "+")) {   // UnaryOp: not handled by sql_to_rex
      p++;
      Nest nest(*this, "expression");
      ExpressionPlan inner = expr(50);
      throw FuseQueryError::plan("Unsupported ExpressionPlan: " + tok.text + " " + sql_display(inner));
    }
    if (is_kw("NOT")) {   // UnaryOp { op: Not }: parsed by sqlparser, refused by sql_to_rex
      p++;
      Nest nest(*this, "expression");
      ExpressionPlan inner = expr(15);   // NOT binds looser than the comparisons, tighter than AND / OR
      throw FuseQueryError::plan("Unsupported ExpressionPlan: NOT " + sql_display(inner));
    }
    if (tok.k == Tok::Word && !reserved(tok.text)) {
      p++;
      if (eat_sym("(")) {   // Expr::Function
        Nest nest(*this, "expression");
        std::vector<ExpressionPlan> args;
        if (!eat_sym(")")) {
          do {
            if (eat_sym("*")) throw FuseQueryError::plan("Unsupported ExpressionPlan: *");
            args.push_back(expr());
          } while (eat_sym(","));
          expect_sym(")");
        }
        return ExpressionPlan::function(tok.text, std::move(args));
      }
      if (peek().k == Tok::Sym && peek().text == ".") throw FuseQueryError::plan("Unsupported ExpressionPlan: " + tok.text + "." + t[p + 1].text);
      return ExpressionPlan::field(tok.text);
    }
    expected("an expression");
  }
};

PlanNode select_to_plan(FuseQueryContextRef ctx, SqlParser &sp) {   // plan_parser.rs:90-133
  if (!sp.eat_kw("SELECT")) sp.expected("SELECT");
  // projection list (planned after FROM/WHERE like the reference)
  struct Item { ExpressionPlan e; };
  std::vector<ExpressionPlan> projection;
  do {
    if (sp.eat_sym("*")) { projection.push_back(ExpressionPlan::wildcard()); continue; }
    ExpressionPlan e = sp.expr();
    if (sp.eat_kw("AS")) {
      if (sp.peek().k != Tok::Word) sp.expected("an identifier after AS");
      e = ExpressionPlan::alias(sp.t[sp.p++].text, std::move(e));
    } else if (sp.peek().k == Tok::Word && !SqlParser::reserved(sp.peek().text)) {
      e = ExpressionPlan::alias(sp.t[sp.p++].text, std::move(e));
    }
    projection.push_back(std::move(e));
  } while (sp.eat_sym(","));

  // FROM: plan_tables_with_joins / create_relation, :155-213
  PlanNode plan = PlanBuilder::empty(true).build();
  if (sp.eat_kw("FROM")) {
    if (sp.eat_sym("(")) {
      // TableFactor::Derived: the subquery's plan (a SelectPlan node) is the input, plan_parser.rs:206-208;
      // children_to_plans flattens nested selects into one chain of transforms
      {
        SqlParser::Nest nest(sp, "PlanNode");
        plan = select_to_plan(ctx, sp);
      }
      sp.expect_sym(")");
      if (sp.eat_kw("AS")) {
        if (sp.peek().k != Tok::Word) sp.expected("an identifier after AS");
        sp.p++;
      } else if (sp.peek().k == Tok::Word && !SqlParser::reserved(sp.peek().text)) {
        sp.p++;   // table alias: parsed, not used (columns are resolved by name only)
      }
    } else {
      if (sp.peek().k != Tok::Word) sp.expected("a table name");
      std::string db = ctx->get_current_database(), table = sp.t[sp.p++].text;
      if (sp.eat_sym(".")) {
        db = table;
        if (sp.peek().k != Tok::Word) sp.expected("a table name");
        table = sp.t[sp.p++].text;
      }
      ITableRef tbl = ctx->get_table(db, table);
      DataSchemaRef schema = tbl->schema();
      std::optional<ExpressionPlan> table_args;
      if (sp.eat_sym("(")) {
        if (!sp.eat_sym(")")) {
          table_args = sp.expr();
          while (sp.eat_sym(",")) sp.expr();   // only args[0] is used, :195-197
          sp.expect_sym(")");
        }
      }
      PlanNode scan = PlanBuilder::scan(db, table, *schema, table_args).build();
      plan = tbl->read_plan(scan);
    }
    if (sp.eat_sym(",") || sp.is_kw("JOIN")) throw FuseQueryError::internal("Cannot support JOIN clause");
  }
  // WHERE -> FilterPlan (below the projection), :265-276
  if (sp.eat_kw("WHERE")) plan = PlanBuilder::from(plan).filter(sp.expr()).build();
  std::vector<ExpressionPlan> group_by;
  if (sp.eat_kw("GROUP")) {
    if (!sp.eat_kw("BY")) sp.expected("BY");
    do { group_by.push_back(sp.expr()); } while (sp.eat_sym(","));
  }
  if (sp.eat_kw("HAVING")) throw FuseQueryError::internal("HAVING is not implemented yet");
  // projection or aggregate, :104-125
  std::vector<ExpressionPlan> aggr;
  for (const auto &e : projection)
    if (e.is_aggregate()) aggr.push_back(e);
  if (!group_by.empty() || !aggr.empty()) {
    if (group_by.size() + aggr.size() != projection.size()) throw FuseQueryError::plan("Projection references non-aggregate values");
    plan = PlanBuilder::from(plan).aggregate(group_by, aggr).build();
  } else {
    plan = PlanBuilder::from(plan).project(projection).build();
  }
  if (sp.eat_kw("ORDER")) {   // no counterpart in plan_parser.rs (query.order_by is never read): SortPlan over the output columns
    if (!sp.eat_kw("BY")) sp.expected("BY");
    std::vector<ExpressionPlan> keys;
    std::vector<bool> desc;
    do {
      keys.push_back(sp.expr());
      bool d = false;
      if (sp.eat_kw("DESC")) d = true;
      else sp.eat_kw("ASC");
      desc.push_back(d);
    } while (sp.eat_sym(","));
    plan = PlanBuilder::from(plan).sort(keys, desc).build();
  }
  if (sp.eat_kw("LIMIT")) {   // :311-328
    ExpressionPlan l = sp.expr();
    if (!(l.kind == ExpressionPlan::Constant && l.value.tag == FQ_U64 && l.value.some)) throw FuseQueryError::plan("Unexpected expression for LIMIT clause");
    plan = PlanBuilder::from(plan).limit((size_t)l.value.u).build();
  }
  return PlanBuilder::from(plan).select().build();
}
}  // namespace

PlanNode Planner::build_from_sql(FuseQueryContextRef ctx, const std::string &query) const {
  SqlParser sp{lex(query)};
  while (sp.eat_sym(";")) {}
  bool explain = false;
  if (sp.is_kw("EXPLAIN")) {
    sp.p++;
    explain = true;
    sp.eat_kw("VERBOSE");
  }
  if (!sp.is_kw("SELECT")) {
    if (sp.peek().k == Tok::End) throw FuseQueryError::internal("Only support single query");
    throw FuseQueryError::internal("Unsupported statement " + sp.peek().text + " for planner.statement_to_plan");
  }
  PlanNode plan = select_to_plan(ctx, sp);
  while (sp.eat_sym(";")) {}
  if (sp.peek().k != Tok::End) {
    if (sp.is_kw("SELECT") || sp.is_kw("EXPLAIN")) throw FuseQueryError::internal("Only support single query");
    sp.expected("end of statement");
  }
  if (explain) return PlanBuilder::from(plan).explain().build();   // explain_statement_to_plan, :57-67
  return plan;
}

// ---------------------------------------------------------------------------------------------
// optimizers — optimizer_filter_push_down.rs:19-82: substitute SELECT aliases into the WHERE predicate
// ---------------------------------------------------------------------------------------------
static ExpressionPlan rewrite_alias_expr(const ExpressionPlan &e, const std::map<std::string, ExpressionPlan> &projection) {
  if (e.kind == ExpressionPlan::Field) {
    auto it = projection.find(e.name);
    if (it != projection.end()) return it->second;
    return e;
  }
  ExpressionPlan out = e;
  for (auto &a : out.args) a = rewrite_alias_expr(a, projection);
  return out;
}
PlanNode FilterPushDownOptimizer::optimize(const PlanNode &plan) const {
  std::vector<PlanNode> plans = plan.node_to_plans();
  // Optimizer::projection_to_map (optimizer.rs:34-57): alias name -> aliased expression
  std::map<std::string, ExpressionPlan> map;
  for (const auto &p : plans)
    if (p.kind == PlanNode::Projection)
      for (const auto &e : p.expr)
        if (e.kind == ExpressionPlan::Alias) map[e.name] = e.args[0];
  for (auto &p : plans)
    if (p.kind == PlanNode::Filter) p.predicate = rewrite_alias_expr(p.predicate, map);
  return PlanNode::plans_to_node(plans);
}
PlanNode Optimizer::optimize(const PlanNode &plan) const { return FilterPushDownOptimizer().optimize(plan); }

}  // namespace fuse
