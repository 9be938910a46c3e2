"""LIKE without a device: the oracle against pyarrow's match_like, the kernel's matcher (cut from kernels/fq_utf8.cuh and
compiled for the host) against the oracle, the SQL front end's LIKE / NOT LIKE, and pipes with lookup nodes compiled for
sm_100a."""
import ctypes as C
import os
import random
import re
import subprocess

import pyarrow as pa
import pyarrow.compute as pc
import pytest

from oracle import like as oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = os.path.join(ROOT, "fuse_query_b200", "csrc", "kernels")
ALPHABET = ["a", "b", "%", "_", "\\", "é", "中", "😀", "\0", "\n"]
TRAILING_ESCAPE = ["\\", "a\\", "%\\", "\\\\\\", "中\\", "a\\%\\"]


def _strings(rng, n, max_len=12):
    return ["".join(rng.choice(ALPHABET) for _ in range(rng.randint(0, max_len))) for _ in range(n)]


def _cases():
    """seeded strings and patterns over the alphabet: lengths 0-12 plus a few 300-character strings"""
    rng = random.Random(20201)
    strings = _strings(rng, 300) + ["".join(rng.choice(ALPHABET) for _ in range(300)) for _ in range(4)] + ["a" * 300, "a" * 299 + "b"]
    patterns = [p for p in _strings(rng, 80, 6) if _well_formed(p)]
    patterns += ["", "%", "%%", "_", "\\%", "\\_", "\\\\", "a%", "%a", "%a%", "_%_", "a%b%a", "%\0%", "%\n", "😀_", "%é_中%"]
    return strings, patterns


def _well_formed(p):
    run = len(p) - len(p.rstrip("\\"))
    return run % 2 == 0


STRINGS, PATTERNS = _cases()


def test_oracle_equals_pyarrow_match_like():
    arr = pa.array(STRINGS + [None])
    n = 0
    for p in PATTERNS:
        want = pc.match_like(arr, p).to_pylist()
        got = [oracle.match_like(s, p) for s in STRINGS + [None]]
        assert got == want, p
        n += len(STRINGS)
    assert n > 5000


@pytest.mark.parametrize("pattern", TRAILING_ESCAPE)
def test_oracle_refuses_a_trailing_escape(pattern):
    with pytest.raises(ValueError, match=re.escape(oracle.TRAILING_ESCAPE)):
        oracle.match_like("a", pattern)


def _cut_function(path, name):
    src = open(path).read()
    m = re.search(r"^__device__ [^\n]*\b" + name + r"\(", src, re.M)
    assert m, f"{name} not found in {path}"
    depth = 0
    for j in range(src.index("{", m.end()), len(src)):
        depth += {"{": 1, "}": -1}.get(src[j], 0)
        if depth == 0:
            return src[m.start():j + 1]
    raise AssertionError(f"unbalanced braces after {name}")


@pytest.fixture(scope="module")
def kernel_like(tmp_path_factory):
    """fq_like_match as the kernel defines it, compiled for the host"""
    d = tmp_path_factory.mktemp("kernel_like")
    src = "\n".join([
        "#include <cstdint>",
        "typedef uint32_t fq_u32;",
        "#define __device__",
        "#define __forceinline__ inline",
        _cut_function(os.path.join(KERNELS, "fq_utf8.cuh"), "fq_like_match"),
        'extern "C" int like(const unsigned char *s, fq_u32 n, const unsigned char *p, fq_u32 m) { return fq_like_match(s, n, p, m); }',
    ])
    (d / "l.cc").write_text(src)
    lib_path = str(d / "libl.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Werror", "-shared", "-fPIC", "-o", lib_path, str(d / "l.cc")], check=True, capture_output=True)
    lib = C.CDLL(lib_path)
    lib.like.restype, lib.like.argtypes = C.c_int, [C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32]
    return lambda s, p: bool(lib.like(s, len(s), p, len(p)))


def test_kernel_matcher_equals_the_oracle(kernel_like):
    bad = []
    for p in PATTERNS:
        pb = p.encode()
        for s in STRINGS:
            if kernel_like(s.encode(), pb) != oracle.match_like(s, p):
                bad.append((s, p))
    assert not bad, bad[:10]


def test_kernel_matcher_on_long_patterns(kernel_like):
    """no staging limit: patterns of 10 000+ bytes, and the worst case of the one-backtrack-point matcher"""
    s = ("ab" * 6000).encode()
    for p in ["ab" * 6000, "%" + "ab" * 5000 + "%", "%" + "b" * 10001, "a" + "_" * 11998 + "b", "_" * 12000, "_" * 12001]:
        assert kernel_like(s, p.encode()) == oracle.match_like(s.decode(), p), p[:20]
    assert kernel_like(b"a" * 3000, ("%a" * 1000 + "%b").encode()) is False


# ---- SQL front end ----
@pytest.fixture(scope="module")
def h():
    from fuse_query_b200 import _fuse_host
    return _fuse_host


@pytest.fixture(scope="module")
def ctx(h):
    return h.FuseQueryContext.create_ctx(8)


def _explain(h, ctx, sql):
    return h.execute_sql(ctx, "explain " + sql)[0].column(0).to_list()[0]


@pytest.mark.parametrize("where,want", [
    ("number like 'a%' and number = 1 or number like '_'", "((number LIKE a%) AND (number = 1)) OR (number LIKE _)"),
    ("number = 1 and number not like 'a\\%' ", "(number = 1) AND (number NOT LIKE a\\%)"),
    ("number + 1 like 'a' ", "((number + 1) LIKE a)"),
    ("number like 'a' = number", "((number LIKE a) = number)"),
    ("number not like 'x' or number < 2", "((number NOT LIKE x) OR (number < 2))"),
])
def test_like_binds_like_a_comparison(h, ctx, where, want):
    """precedence 20 as in sqlparser 0.6: tighter than AND / OR, looser than + -, left-associative with the comparisons"""
    text = _explain(h, ctx, f"select number from system.numbers_mt(10) where {where}")
    assert f"Filter: {want.strip()}" in text or f"Filter: ({want.strip()})" in text, text


def test_like_column_names_and_types(h, ctx):
    plan = h.Planner().build_from_sql(ctx, "select 'abc' like 'a%', 'abc' not like '_b_' as f from system.numbers_mt(10)")
    fields = plan.schema().fields
    assert [f.name for f in fields] == ["abc LIKE a%", "f"]
    assert all(f.data_type == h.DataType.Boolean for f in fields)


@pytest.mark.parametrize("sql,err", [
    ("select 'abc' like number from system.numbers_mt(10)", "Internal Error: Unsupported on the device path: LIKE with a pattern that is not a string literal"),
    ("select number like 'a%' from system.numbers_mt(10)", "Internal Error: Unsupported (UInt64) LIKE (Utf8)"),
    ("select number not like 'a%' from system.numbers_mt(10)", "Internal Error: Unsupported (UInt64) NOT LIKE (Utf8)"),
    ("select number from system.numbers_mt(10) where not number like 'a%'", "Error during plan: Unsupported ExpressionPlan: NOT number LIKE 'a%'"),
    ("select number from system.numbers_mt(10) where not (number > 1)", "Error during plan: Unsupported ExpressionPlan: NOT number > 1"),
])
def test_like_refusals_at_plan_time(h, ctx, sql, err):
    with pytest.raises(h.FuseQueryError) as e:
        h.Planner().build_from_sql(ctx, sql)
    assert str(e.value) == err


# ---- pipes with lookup nodes, compiled for sm_100a ----
def _codegen(tmp_path, pred, exprs, kind, cols, dtypes):
    """the generated source of a pipe, through the library's own code generator (aotgen's reader)"""
    from fuse_query_b200 import cabi
    src = ["#include <cstdio>", '#include "codegen.h"', "int main() {", "  std::vector<fq_expr_node> nodes; std::string err; int r;",
           "  fq_pipe_desc d = {};", f"  d.n_cols = {len(cols)};"]
    names = ", ".join(f'"{c}"' for c in cols)
    src.append(f"  std::vector<std::string> cols = {{{names}}};")
    for i, t in enumerate(dtypes):
        src.append(f"  d.col_dtypes[{i}] = {t};")
    src.append("  d.predicate = -1;")
    if pred:
        src.append(f'  if (fq::parse_sexpr("{pred}", cols, &nodes, &r, &err)) {{ puts(err.c_str()); return 1; }}')
        src.append("  d.predicate = r;")
    for k, e in enumerate(exprs):
        src.append(f'  if (fq::parse_sexpr("{e}", cols, &nodes, &r, &err)) {{ puts(err.c_str()); return 1; }}')
        src.append(f"  d.exprs[{k}] = r;")
    src += [f"  d.n_exprs = {len(exprs)};", f"  d.kind = {kind};", "  d.nodes = nodes.data(); d.n_nodes = (int)nodes.size();",
            "  fq::Generated g;", "  if (int st = fq::generate(d, &g, &err)) { printf(\"%d %s\\n\", st, err.c_str()); return 1; }",
            "  fputs(g.source.c_str(), stdout);", "  return 0;", "}"]
    (tmp_path / "gen.cc").write_text("\n".join(src))
    csrc = os.path.join(ROOT, "fuse_query_b200", "csrc")
    exe = str(tmp_path / "gen")
    subprocess.run(["g++", "-std=c++17", "-O1", "-I", csrc, "-I", os.path.join(ROOT, "include"), str(tmp_path / "gen.cc"), os.path.join(csrc, "codegen.cc"),
                    "-o", exe], check=True, capture_output=True)
    return subprocess.run([exe], check=True, capture_output=True, text=True).stdout


def _ptxas(tmp_path, source, name):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    skel = open(os.path.join(KERNELS, "fq_skeleton.cuh")).read()
    cu = tmp_path / f"{name}.cu"
    cu.write_text(skel + "\n" + source)
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-Xptxas", "-v", "-c", str(cu), "-o", str(tmp_path / f"{name}.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    usage, spills = {}, {}
    for chunk in r.stderr.split("Compiling entry function '")[1:]:
        name = chunk.split("'")[0]
        usage[name] = int(re.search(r"Used (\d+) registers", chunk).group(1))
        spills[name] = int(re.search(r"(\d+) bytes spill stores", chunk).group(1))
    return usage, spills, r.stderr


def test_lookup_pipes_compile_for_sm100a_without_new_spills(tmp_path):
    """a LIKE pipe (lookup of a codes column) against the same pipe with `=`: every kernel variant builds, and no build of
    the LIKE pipe spills more than the `=` one (the dense select build has a budget of 128 registers per thread)"""
    from fuse_query_b200 import cabi
    cols, dtypes = ["s", "x"], [cabi.U32, cabi.U32]
    usage = {}
    for name, pred in (("like", "(lookup 0 (col s))"), ("eq", "(= (col s) (u32 42))")):
        src = _codegen(tmp_path, pred, ["(col x)"], cabi.PIPE_PROJECT, cols, dtypes)
        u, sp, _ = _ptxas(tmp_path, src, name)
        usage[name] = {k.rsplit("_select", 1)[-1] or "ldg": (u[k], sp[k]) for k in u}
    print("select builds (registers, spill bytes): LIKE", usage["like"], "| =", usage["eq"])
    assert set(usage["like"]) == {"ldg", "_tma", "_dense", "_probe"}
    for variant, (regs, spill) in usage["like"].items():
        assert spill <= usage["eq"][variant][1], (variant, usage)
    assert usage["like"]["_dense"][0] <= 128
    assert "fq_lookup(p.lookup[0], p.lookup_bits[0]" in _codegen(tmp_path, "(lookup 0 (col s))", ["(col x)"], cabi.PIPE_PROJECT, cols, dtypes)
    for kind, pred, exprs, suffixes in ((cabi.PIPE_AGGREGATE, "(lookup 1 (col s))", ["(count (col s))", "(sum (col x))"], ("_agg_tma", "_agg_u4")),
                                        (cabi.PIPE_PROJECT, None, ["(lookup 3 (col s))", "(col x)"], ("_map_tma", "_map"))):
        u, sp, _ = _ptxas(tmp_path, _codegen(tmp_path, pred, exprs, kind, cols, dtypes), f"k{kind}")
        assert all(any(k.endswith(x) for k in u) for x in suffixes), sorted(u)


@pytest.mark.parametrize("bad,msg", [
    ("(lookup 4 (col s))", "lookup slot 4 out of range"),
    ("(lookup -1 (col s))", "lookup slot -1 out of range"),
    ("(lookup 0 (u32 3))", "a lookup of a constant index"),
    ("(lookup 0 (col x))", "a lookup takes an unsigned integer index, not Int64"),
])
def test_malformed_lookup_nodes_are_refused(tmp_path, bad, msg):
    from fuse_query_b200 import cabi
    with pytest.raises(subprocess.CalledProcessError) as e:
        _codegen(tmp_path, bad, ["(col s)"], cabi.PIPE_PROJECT, ["s", "x"], [cabi.U32, cabi.I64])
    assert msg in e.value.stdout and e.value.stdout.startswith(str(cabi.ERR_INVALID))
