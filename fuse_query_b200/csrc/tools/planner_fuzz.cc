// planner_fuzz.cc — robustness harness for the hand-written SQL front end and plan / pipeline builders of the host mirror
// (csrc/host/planners.cc, pipeline.cc): random token sequences must end in a plan or a FuseQueryError.  Built with
// -fsanitize=address,undefined by tests/test_abi_exports.py; needs no device (plans are built, never executed).
//
// usage: planner_fuzz [iterations] [seed]
#include <cstdio>
#include <cstdlib>
#include <functional>
#include <random>
#include <string>
#include <vector>

#include "../host/fq_host.h"

using namespace fuse;

int main(int argc, char **argv) {
  const int iters = argc > 1 ? atoi(argv[1]) : 20000;
  std::mt19937_64 rng(argc > 2 ? strtoull(argv[2], nullptr, 10) : 12345);
  const std::vector<std::string> toks = {
      "select", "from", "where", "limit", "group", "by", "as", "and", "or", "not", "explain", "system", ".", "numbers_mt", "number",
      "(", ")", ",", "*", "+", "-", "/", "%", "=", "<", ">", "<=", ">=", "<>", "!=", "1", "0", "10000", "1.5", "'a'", "sum", "count",
      "max", "min", "avg", "x", "t", ";", "having", "order", "asc", "desc", "join", "union", "-1", "1e10", "99999999999999999999", "\"q\"", "`b`",
      "'", "''", "\\", "/*", "--", "\t", "\n", "0x10", "1.", ".5", "e", "1e", "select(", "))", "((", "system.numbers_mt(10)", "like", "'%a_'", "'\\'"};
  auto pick = [&](size_t n) { return (size_t)(rng() % n); };
  // a grammar-shaped generator beside the token soup, so that the optimizer, EXPLAIN and the pipeline builder see plans too
  std::function<std::string(int)> expr = [&](int depth) -> std::string {
    static const char *leaf[] = {"number", "1", "0", "2.5", "'s'", "x", "c1", "10000"};
    static const char *ops[] = {"+", "-", "*", "/", "=", "<", ">", "<=", ">=", "and", "or", "%", "<>", "like", "not like"};
    static const char *fns[] = {"sum", "count", "max", "min", "avg", "nosuch"};
    if (depth <= 0 || pick(3) == 0) return leaf[pick(8)];
    switch (pick(4)) {
      case 0: return "(" + expr(depth - 1) + ")";
      case 1: return std::string(fns[pick(6)]) + "(" + expr(depth - 1) + ")";
      default: return expr(depth - 1) + " " + ops[pick(15)] + " " + expr(depth - 1);
    }
  };
  std::function<std::string(int)> query = [&](int nest) -> std::string {
    std::string q = "select ";
    for (size_t i = 0, m = 1 + pick(3); i < m; i++) q += (i ? ", " : "") + expr(3) + (pick(3) == 0 ? " as c" + std::to_string(i + 1) : "");
    if (nest > 0 && pick(3) == 0) q += " from (" + query(nest - 1) + ")" + (pick(2) ? " t" : "");
    else q += " from system.numbers_mt(" + std::string(pick(5) ? "100000" : "number") + ")";
    if (pick(2)) q += " where " + expr(3);
    if (pick(6) == 0) q += " group by " + expr(1);
    if (pick(4) == 0) {   // ORDER BY: output columns, arbitrary expressions, both directions
      q += " order by ";
      for (size_t i = 0, m = 1 + pick(2); i < m; i++) q += (i ? ", " : "") + (pick(2) ? "c" + std::to_string(1 + pick(3)) : expr(2)) + (pick(3) == 0 ? " desc" : pick(2) ? " asc" : "");
    }
    if (pick(3) == 0) q += " limit " + std::string(pick(4) ? "3" : "x");
    return (pick(5) == 0 ? "explain " : "") + q;
  };
  FuseQueryContextRef ctx = FuseQueryContext::create_ctx(8, nullptr, nullptr);
  long planned = 0, refused = 0;
  for (int it = 0; it < iters; it++) {
    std::string q;
    const size_t k = 1 + pick(16);
    if (pick(2)) {
      q = query(2);
    } else if (pick(2)) {
      q = "select ";
      for (size_t i = 0; i < k; i++) q += toks[pick(toks.size())] + " ";
      q += "from system.numbers_mt(" + toks[pick(toks.size())] + ") ";
      for (size_t i = 0, m = pick(7); i < m; i++) q += toks[pick(toks.size())] + " ";
    } else {
      for (size_t i = 0; i < k; i++) q += toks[pick(toks.size())] + (pick(4) ? " " : "");
    }
    try {
      PlanNode plan = Planner().build_from_sql(ctx, q);
      plan = Optimizer::create().optimize(plan);
      (void)plan.to_string();
      try {
        Pipeline p = PipelineBuilder::create(ctx, plan).build();
        (void)p.to_string();
      } catch (const FuseQueryError &) {
      }
      planned++;
    } catch (const FuseQueryError &) {
      refused++;
    }
  }
  printf("planner_fuzz: %ld planned, %ld refused\n", planned, refused);
  return 0;
}
