// codegen_fuzz.cc — robustness harness for the expression-tree code generator (codegen.cc): random pipe descriptions,
// most of them malformed (dangling / cyclic child indexes, wrong kinds, non-numeric types, too many columns), must
// come back as an fq_status with a message — never crash, never read out of bounds.  Built and run by
// tests/test_host_planner.py with -fsanitize=address,undefined.
//
// usage: codegen_fuzz [iterations] [seed]
#include <cstdio>
#include <cstdlib>
#include <random>
#include <string>
#include <vector>

#include "../codegen.h"

int main(int argc, char **argv) {
  const int iters = argc > 1 ? atoi(argv[1]) : 20000;
  std::mt19937_64 rng(argc > 2 ? strtoull(argv[2], nullptr, 10) : 12345);
  auto pick = [&](int lo, int hi) { return (int)(rng() % (uint64_t)(hi - lo + 1)) + lo; };
  long ok = 0, rejected = 0;
  for (int it = 0; it < iters; it++) {
    fq_pipe_desc d = {};
    const bool wild = pick(0, 3) == 0;                      // a quarter of the cases ignores every range
    d.n_cols = wild ? pick(-2, 12) : pick(1, FQ_MAX_COLS);
    for (int c = 0; c < FQ_MAX_COLS; c++) {
      d.col_dtypes[c] = wild ? pick(-1, 15) : pick(FQ_BOOL, FQ_F64);
      d.col_nullable[c] = pick(0, 1);
    }
    d.generated = pick(0, 1);
    if (d.generated) d.col_dtypes[0] = FQ_U64;
    const int n = pick(1, 24);
    std::vector<fq_expr_node> nodes((size_t)n);
    for (int i = 0; i < n; i++) {
      fq_expr_node &x = nodes[(size_t)i];
      x.kind = wild ? pick(-1, 9) : pick(FQ_EXPR_ALIAS, FQ_EXPR_LOOKUP);
      x.op = wild ? pick(-1, 9) : pick(0, 4);
      if (x.kind == FQ_EXPR_LOOKUP && !wild) x.op = pick(0, 4) ? pick(0, FQ_MAX_LOOKUPS - 1) : pick(-2, FQ_MAX_LOOKUPS + 2);   // slots, a few out of range
      // children mostly point backwards (a DAG), sometimes anywhere (cycles, self references, out of range)
      x.left = pick(0, 9) ? (i ? pick(0, i - 1) : -1) : pick(-3, n + 2);
      x.right = pick(0, 9) ? (i ? pick(0, i - 1) : -1) : pick(-3, n + 2);
      x.column = wild ? pick(-2, 12) : pick(0, d.n_cols > 0 ? d.n_cols - 1 : 0);
      x.dtype = wild ? pick(-1, 15) : pick(FQ_BOOL, FQ_F64);
      x.value.u = rng() >> pick(0, 63);
    }
    d.nodes = nodes.data();
    d.n_nodes = n;
    d.predicate = pick(0, 2) ? -1 : pick(-2, n + 1);
    d.kind = wild ? pick(-1, 3) : pick(FQ_PIPE_PROJECT, FQ_PIPE_AGGREGATE);
    d.n_exprs = wild ? pick(-1, 10) : pick(1, FQ_MAX_EXPRS);
    for (int e = 0; e < FQ_MAX_EXPRS; e++) d.exprs[e] = pick(0, 7) ? pick(0, n - 1) : pick(-3, n + 2);
    fq::Generated g;
    std::string err;
    const int st = fq::generate(d, &g, &err);
    if (st == FQ_OK) {
      ok++;
      if (g.source.empty() || g.tag.size() != 16) { fprintf(stderr, "iteration %d: FQ_OK without a program\n", it); return 1; }
    } else {
      rejected++;
      if (err.empty()) { fprintf(stderr, "iteration %d: status %d without a message\n", it, st); return 1; }
    }
  }
  printf("codegen_fuzz: %ld generated, %ld rejected\n", ok, rejected);
  return 0;
}
