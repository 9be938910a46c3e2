"""Both select kernels (FQ_SEL_VARIANT = ldg | tma) against closed forms and the oracle: order-preserving compaction
over ragged sizes around every tile / segment / ring boundary, dense and sparse selections, limits, early exit,
several input columns of different widths, validity.  (transform_filter.rs:38-55, transform_projection.rs:45-56,
stream_limit.rs:28-48.)  Integer results bit-exact."""
import os

import numpy as np
import pytest

from fuse_query_b200 import cabi
from oracle import binding as o

pytestmark = pytest.mark.gpu
NUM = "(col number)"
README_PRED = f"(< (+ (+ (+ {NUM} (u64 1)) (/ {NUM} (u64 2))) (u64 1)) (u64 100))"
PROJ = [f"(alias c1 (+ {NUM} (u64 1)))", f"(alias c2 (/ {NUM} (u64 2)))"]


@pytest.fixture(scope="module", autouse=True)
def all_jit_variants():
    """A JIT build normally holds only the kernel variant it will launch; this file switches variants per test."""
    os.environ["FQ_JIT_ALL_VARIANTS"] = "1"
    yield
    os.environ.pop("FQ_JIT_ALL_VARIANTS", None)


@pytest.fixture(params=["ldg", "tma", "dense"])
def variant(request):
    old = os.environ.get("FQ_SEL_VARIANT")
    os.environ["FQ_SEL_VARIANT"] = request.param     # read by the library when a pipe is compiled
    yield request.param
    if old is None:
        os.environ.pop("FQ_SEL_VARIANT", None)
    else:
        os.environ["FQ_SEL_VARIANT"] = old


@pytest.fixture(scope="module")
def ctx():
    c = cabi.Context(0)
    yield c
    c.close()


# tile = 4096 rows (tma) / 3072 rows (ldg); segment = 32768 / 24576 rows; 148 CTAs x 4-slot ring
SIZES = [1, 2, 15, 4095, 4096, 4097, 16385, 24576, 24577, 32767, 32768, 32769, 65536 + 1, 148 * 32768 - 1, 148 * 32768,
         148 * 32768 * 3 + 4097, 20_000_019]


@pytest.mark.parametrize("n", SIZES)
def test_every_kth_row_is_kept_in_order(ctx, variant, n):
    k = 7
    col = ctx.numbers(0, n)
    pipe = ctx.pipe(PROJ, predicate=f"(= (* (/ {NUM} (u64 {k})) (u64 {k})) {NUM})")
    want = np.arange(0, n, k, dtype=np.uint64)
    outs = [ctx.column(cabi.U64, len(want) + 5), ctx.column(cabi.U64, len(want) + 5)]
    pipe.launch_project(cabi.make_source([col], n), outs, len(want) + 5)
    sel, written = pipe.fetch_project()
    assert sel == written == len(want)
    assert np.array_equal(outs[0].to_numpy(written), want + 1)
    assert np.array_equal(outs[1].to_numpy(written), want // 2)
    for c in outs + [col]:
        c.free()
    pipe.destroy()


@pytest.mark.parametrize("n", [4097, 148 * 16384 + 33, 5_000_001])
def test_all_rows_kept_and_none_kept(ctx, variant, n):
    col = ctx.numbers(0, n)
    src = cabi.make_source([col], n)
    pipe = ctx.pipe(PROJ, predicate=f"(>= {NUM} (u64 0))")
    outs = [ctx.column(cabi.U64, n), ctx.column(cabi.U64, n)]
    pipe.launch_project(src, outs, n)
    assert pipe.fetch_project() == (n, n)
    assert np.array_equal(outs[0].to_numpy(n), np.arange(1, n + 1, dtype=np.uint64))
    assert np.array_equal(outs[1].to_numpy(n), np.arange(n, dtype=np.uint64) // 2)
    none = ctx.pipe(PROJ, predicate=f"(< {NUM} (u64 0))")
    none.launch_project(src, outs, n)
    assert none.fetch_project() == (0, 0)


@pytest.mark.parametrize("lo,hi", [(0, 2_500_001), (12_345, 4_000_000), (12_346, 5_000_000), (4_999_999, 5_000_001), (77, 78)])
def test_range_predicates_keep_whole_groups(ctx, variant, lo, hi):
    """Range predicates over sorted data keep vector groups all-or-nothing: pass 2 writes them with vector stores when
    the output position keeps the alignment (even `lo`) and row by row when it does not (odd `lo`)."""
    n = 5_000_001
    col = ctx.numbers(0, n)
    pipe = ctx.pipe(PROJ + [NUM], predicate=f"(and (>= {NUM} (u64 {lo})) (< {NUM} (u64 {hi})))")
    hi = min(hi, n)
    k = hi - lo
    for cap in (k, k - 1 if k > 1 else k, k + 7):
        outs = [ctx.column(cabi.U64, cap) for _ in range(3)]
        pipe.launch_project(cabi.make_source([col], n), outs, cap)
        sel, written = pipe.fetch_project()
        assert sel == k and written == min(k, cap)
        want = np.arange(lo, lo + written, dtype=np.uint64)
        assert np.array_equal(outs[0].to_numpy(written), want + 1)
        assert np.array_equal(outs[1].to_numpy(written), want // 2)
        assert np.array_equal(outs[2].to_numpy(written), want)
        for c in outs:
            c.free()


@pytest.mark.parametrize("limit,early", [(3, False), (3, True), (1000, True), (0, False)])
def test_readme_query_with_limit(ctx, variant, limit, early):
    n = 30_000_011
    col = ctx.numbers(0, n)
    pipe = ctx.pipe(PROJ, predicate=README_PRED)
    outs = [ctx.column(cabi.U64, 128), ctx.column(cabi.U64, 128)]
    pipe.launch_project(cabi.make_source([col], n), outs, 128, limit=limit, early_exit=early)
    sel, written = pipe.fetch_project()
    w = min(limit, 66)
    assert written == w
    assert sel >= w if early else sel == 66          # with early exit only a lower bound is known
    assert np.array_equal(outs[0].to_numpy(w), np.arange(1, w + 1, dtype=np.uint64))
    assert np.array_equal(outs[1].to_numpy(w), np.arange(w, dtype=np.uint64) // 2)


def test_early_exit_in_the_middle_of_a_long_scan(ctx, variant):
    n = 40_000_000
    col = ctx.numbers(0, n)
    pipe = ctx.pipe([NUM], predicate=f"(>= {NUM} (u64 20000000))")
    outs = [ctx.column(cabi.U64, 10)]
    pipe.launch_project(cabi.make_source([col], n), outs, 10, limit=10, early_exit=True)
    sel, written = pipe.fetch_project()
    assert written == 10 and sel >= 10
    assert np.array_equal(outs[0].to_numpy(10), np.arange(20_000_000, 20_000_010, dtype=np.uint64))


def test_mixed_width_nullable_columns_match_oracle(ctx, variant):
    n = 300_017
    rng = np.random.default_rng(3)
    a = rng.integers(0, 1 << 40, n, dtype=np.uint64)
    b = rng.integers(-1000, 1000, n).astype(np.int16)
    c = rng.normal(0, 100, n)
    av = (rng.random(n) > 0.25).astype(np.uint8)
    cols = [ctx.from_numpy(a, av), ctx.from_numpy(b), ctx.from_numpy(c)]
    table = {"a": o.array(o.U64, a, av), "b": o.array(o.I16, b), "c": o.array(o.F64, c)}
    exprs = ["(+ (col a) (col b))", "(* (col c) (col b))", "(col b)"]
    pred = "(and (> (col b) (i16 -500)) (< (col a) (u64 800000000000)))"
    want = o.run_query(exprs, table=table, predicate=pred, worker_threads=1, tail_quirk=False)
    pipe = ctx.pipe(exprs, columns=["a", "b", "c"], dtypes=[cabi.U64, cabi.I16, cabi.F64], predicate=pred, nullable=[True, False, False])
    outs = [ctx.column(pipe.expr_dtype(i), n) for i in range(3)]
    ov = [ctx.column(cabi.BOOL, n) if pipe.expr_nullable(i) else None for i in range(3)]
    pipe.launch_project(cabi.make_source(cols, n), outs, n, out_valid=ov)
    sel, written = pipe.fetch_project()
    assert sel == written == want.n_rows > 0
    for i, wc in enumerate(want.columns):
        wv = np.ones(written, np.uint8) if wc.valid is None else wc.valid
        gv = np.ones(written, np.uint8) if ov[i] is None else ov[i].to_numpy(written)
        assert np.array_equal(gv, wv)
        m = wv.astype(bool)
        assert np.array_equal(outs[i].to_numpy(written)[m].astype(wc.values.dtype), wc.values[m], equal_nan=wc.dtype == o.F64)


@pytest.mark.parametrize("off", [1, 3, 8, 13, 16, 10_001])
def test_unaligned_slices_fall_back_to_row_loads(ctx, variant, off):
    """A slice that does not start on a 16-byte boundary (MemoryTable partitions of odd sizes, arrow::Array::slice in the
    reference) is read row by row: select, projection-only and aggregate pipes, both aggregate kernels."""
    n_all, n = 700_000, 650_003
    rng = np.random.default_rng(off)
    a = rng.integers(0, 1 << 40, n_all, dtype=np.uint64)
    b = rng.integers(-100, 100, n_all).astype(np.int8)
    bv = (rng.random(n_all) > 0.3).astype(np.uint8)
    A, B = ctx.from_numpy(a), ctx.from_numpy(b, bv)
    sa, sb = A.slice(off, n), B.slice(off, n)
    src = cabi.make_source([sa, sb], n)
    x, y, yv = a[off:off + n], b[off:off + n].astype(np.int64), bv[off:off + n].astype(bool)
    kw = dict(columns=["a", "b"], dtypes=[cabi.U64, cabi.I8], nullable=[False, True])
    # filter + projection
    pipe = ctx.pipe(["(col a)", "(* (col b) (i8 2))"], predicate="(> (col b) (i8 10))", **kw)
    outs = [ctx.column(cabi.U64, n), ctx.column(cabi.I8, n)]
    ov = [None, ctx.column(cabi.BOOL, n)]
    pipe.launch_project(src, outs, n, out_valid=ov)
    sel, written = pipe.fetch_project()
    keep = yv & (y > 10)
    assert sel == written == int(keep.sum())
    assert np.array_equal(outs[0].to_numpy(written), x[keep])
    assert np.array_equal(outs[1].to_numpy(written), (y[keep] * 2).astype(np.int8))   # Int8 * Int8 wraps
    assert ov[1].to_numpy(written).all()
    # projection only
    pipe = ctx.pipe(["(* (col a) (u64 3))"], **kw)
    out = ctx.column(cabi.U64, n)
    pipe.launch_project(src, [out], n)
    assert pipe.fetch_project() == (n, n)
    assert np.array_equal(out.to_numpy(n), x * np.uint64(3))
    # aggregates (bulk-copy staged and LDG kernels)
    for agg_variant in ("tma", "u4"):
        os.environ["FQ_AGG_VARIANT"] = agg_variant
        try:
            pipe = ctx.pipe(["(sum (col a))", "(max (col b))", "(count (col a))", "(min (col a))"], aggregate=True, **kw)
            pipe.launch_aggregate(src)
            states, rows = pipe.fetch_aggregate()
        finally:
            os.environ.pop("FQ_AGG_VARIANT", None)
        assert rows == n
        assert [v for _, v in states] == [int(x.sum(dtype=np.uint64)), int(y[yv].max()), n, int(x.min())]


@pytest.mark.parametrize("map_variant", ["ldg", "tma"])
@pytest.mark.parametrize("n", [1, 4095, 4096, 4097, 148 * 4096 + 5, 3_000_001])
def test_projection_without_filter_both_variants(ctx, map_variant, n):
    """ProjectionTransform alone (transform_projection.rs:45-56): every row, every expression, both load styles."""
    os.environ["FQ_MAP_VARIANT"] = map_variant
    try:
        rng = np.random.default_rng(n)
        a = rng.integers(0, 1 << 50, n, dtype=np.uint64)
        b = rng.integers(-30000, 30000, n).astype(np.int16)
        cols = [ctx.from_numpy(a), ctx.from_numpy(b)]
        pipe = ctx.pipe(["(+ (col a) (u64 1))", "(/ (col a) (u64 2))", "(* (col b) (i16 3))", "(< (col b) (i16 0))"], columns=["a", "b"],
                        dtypes=[cabi.U64, cabi.I16])
        outs = [ctx.column(pipe.expr_dtype(i), n) for i in range(4)]
        for cap in (n, max(1, n - 3)):
            pipe.launch_project(cabi.make_source(cols, n), outs, cap)
            assert pipe.fetch_project() == (n, cap)
            assert np.array_equal(outs[0].to_numpy(cap), a[:cap] + 1)
            assert np.array_equal(outs[1].to_numpy(cap), a[:cap] // 2)
            assert np.array_equal(outs[2].to_numpy(cap), (b[:cap] * np.int16(3)).astype(np.int16))
            assert np.array_equal(outs[3].to_numpy(cap).astype(bool), b[:cap] < 0)
    finally:
        os.environ.pop("FQ_MAP_VARIANT", None)


def test_limit_without_filter_stops_after_the_block_that_completes_it(ctx):
    """stream_limit.rs:28-31: LimitStream ends the pipe, so blocks after the one that completes the limit are never
    evaluated — a zero divisor in row 10 000 does not surface with LIMIT 5."""
    n = 50_000
    x = np.ones(n, dtype=np.uint64)
    x[10_000:] = 0
    col = ctx.from_numpy(x)
    pipe = ctx.pipe(["(/ (u64 10) (col x))"], columns=["x"], dtypes=[cabi.U64])
    out = ctx.column(cabi.U64, 5)
    pipe.launch_project(cabi.make_source([col], n), [out], 5, limit=5, early_exit=True)
    sel, written = pipe.fetch_project()
    assert written == 5 and sel == 10_000 and out.to_numpy(5).tolist() == [10] * 5
    # without the early exit every row is counted; projection expressions are still evaluated only for rows that are
    # written (DESIGN.md, known deviations), so the zero divisors beyond the limit stay silent
    pipe.launch_project(cabi.make_source([col], n), [out], 5, limit=5, early_exit=False)
    assert pipe.fetch_project() == (n, 5)
    # ... and are an error as soon as such a row is written
    out2 = ctx.column(cabi.U64, n)
    pipe.launch_project(cabi.make_source([col], n), [out2], n)
    with pytest.raises(cabi.FuseGpuError) as e:
        pipe.fetch_project()
    assert str(e.value) == "Internal Error: Divide by zero error"


def test_variants_launch_different_kernels(ctx):
    """The environment switch must really select another kernel (both are precompiled for the README pipe)."""
    pipe = ctx.pipe(PROJ, predicate=README_PRED)
    assert pipe.precompiled
    src = pipe.source
    assert "_select_tma(" in src and "_select(" in src
