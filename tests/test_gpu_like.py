"""LIKE / NOT LIKE on the device: fq_utf8_like over Utf8 arrays against the oracle (oracle/like.py), the FQ_EXPR_LOOKUP node
in every kernel variant against numpy's bits[codes], and SQL over a registered table with a nullable string column
against pyarrow's match_like."""
import os
import random

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pytest

from oracle import like as oracle

pytestmark = pytest.mark.gpu

ALPHABET = ["a", "b", "%", "_", "\\", "é", "中", "😀", "\0", "\n"]
PATTERNS = ["", "%", "%%", "_", "\\%", "a%", "%b", "%a_%", "_%😀", "\\\\%", "%\0%"]


@pytest.fixture(scope="module")
def cctx():
    from fuse_query_b200 import cabi
    os.environ["FQ_JIT_ALL_VARIANTS"] = "1"   # JIT builds hold every kernel variant, so that set_variant picks each of them
    ctx = cabi.Context(0)
    yield ctx
    ctx.close()
    os.environ.pop("FQ_JIT_ALL_VARIANTS", None)


def unpack(col, n):
    nbytes = max(1, (n + 7) // 8)
    raw = col.to_numpy(nbytes).astype(np.uint8)
    bits = np.unpackbits(raw, bitorder="little")
    assert not bits[n:].any(), "padding bits must be zero"
    return bits[:n].astype(bool)


def random_strings(n, seed, null_every=7):
    rng = random.Random(seed)
    out = ["".join(rng.choice(ALPHABET) for _ in range(rng.randint(0, 12))) for _ in range(n)]
    return [None if null_every and i % null_every == 3 else v for i, v in enumerate(out)]


# ---- fq_utf8_like over arrays ----
@pytest.mark.parametrize("n", [0, 1, 31, 32, 33, 255, 256, 257, 100_003])
def test_like_over_arrays(cctx, n):
    values = random_strings(n, n)
    arr = cctx.utf8(values)
    for p in PATTERNS:
        for negate in (False, True):
            got = unpack(arr.like(p, negate), n)
            assert got.tolist() == oracle.like_bits(values, p, negate), (p, negate)
    arr.free()


def test_like_pattern_over_ten_thousand_bytes(cctx):
    long = "ab" * 5001 + "%"
    values = ["ab" * 5001 + "tail", "ab" * 5000, "x" + "ab" * 5001, None, "ab" * 5001]
    arr = cctx.utf8(values)
    for p in (long, "%" + "ab" * 5001, "_" * 10002 + "%"):
        assert unpack(arr.like(p), len(values)).tolist() == oracle.like_bits(values, p), p[:10]


def test_like_refuses_a_trailing_escape(cctx):
    from fuse_query_b200 import cabi
    arr = cctx.utf8(["a\\", "b"])
    for p in ("\\", "a\\", "\\\\\\"):
        with pytest.raises(cabi.FuseGpuError) as e:
            arr.like(p)
        assert e.value.status == cabi.ERR_INVALID
        assert str(e.value) == "Internal Error: LIKE pattern ends with the escape character \\"
    assert unpack(arr.like("a\\\\"), 2).tolist() == [True, False]


# ---- the lookup node in every kernel ----
def lookup_case(cctx, n_bits, n_rows, validity, seed, offset=0):
    """codes in [0, n_bits + 3) (some at or beyond the table), a random table, x = row index"""
    rng = np.random.default_rng(seed)
    table = rng.integers(0, 256, max(1, (n_bits + 7) // 8)).astype(np.uint8)
    bits = np.unpackbits(table, bitorder="little")[:n_bits].astype(bool)
    codes = rng.integers(0, n_bits + 3, n_rows + offset).astype(np.uint32)
    hit = np.concatenate([bits, np.zeros(3, bool)])[codes[offset:]]
    valid = rng.random(n_rows + offset) > 0.2
    if validity == "bytes":
        col = cctx.from_numpy(codes, valid)
    elif validity == "bitmap":   # row 0 at bit 3 of the bitmap: off the 128-row grid, the row-by-row validity path
        bitmap = np.packbits(np.concatenate([np.zeros(3, bool), valid]), bitorder="little")
        col = cctx.from_numpy(codes, valid_bitmap=bitmap, bit_offset=3)
    else:
        col = cctx.from_numpy(codes)
        valid[:] = True
    if offset:
        col = col.slice(offset, n_rows)
    x = cctx.from_numpy(np.arange(n_rows, dtype=np.uint32))
    return cctx.from_numpy(table), col, x, hit, valid[offset:]


NULLABLE = {"none": 0, "bytes": 1, "bitmap": 2}
CASES = [(0, "none", 0), (1, "bytes", 0), (33, "bitmap", 0), (4097, "none", 1), (4097, "bytes", 0), (1_000_000, "bitmap", 0), (33, "none", 3)]


@pytest.mark.parametrize("n_bits,validity,offset", CASES)
@pytest.mark.parametrize("variant", ["tma", "sparse", "dense", "ldg"])
def test_lookup_in_select(cctx, n_bits, validity, offset, variant):
    from fuse_query_b200 import cabi
    n = 300_001
    table, col, x, hit, valid = lookup_case(cctx, n_bits, n, validity, n_bits + offset, offset)
    pipe = cctx.pipe(["(col x)"], columns=["c", "x"], dtypes=[cabi.U32, cabi.U32], nullable=[NULLABLE[validity], 0],
                     predicate="(lookup 2 (col c))")
    pipe.set_variant(variant)
    pipe.set_lookup(2, table, n_bits)
    want = np.nonzero(hit & valid)[0]
    out = cctx.column(cabi.U32, n)
    pipe.launch_project(cabi.make_source([col, x], n), [out], n)
    sel, written = pipe.fetch_project()
    assert sel == written == len(want)
    assert np.array_equal(out.to_numpy(written), want)
    # LIMIT with the early exit: the first rows in order
    pipe.launch_project(cabi.make_source([col, x], n), [out], 10, limit=10, early_exit=True)
    _, written = pipe.fetch_project()
    assert out.to_numpy(written).tolist() == want[:10].tolist()


@pytest.mark.parametrize("n_bits,validity,offset", CASES)
@pytest.mark.parametrize("variant", ["tma", "u4"])
def test_lookup_in_aggregate(cctx, n_bits, validity, offset, variant):
    from fuse_query_b200 import cabi
    n = 300_001
    table, col, x, hit, valid = lookup_case(cctx, n_bits, n, validity, 7 + n_bits + offset, offset)
    pipe = cctx.pipe(["(count (col x))", "(sum (col x))"], columns=["c", "x"], dtypes=[cabi.U32, cabi.U32], nullable=[NULLABLE[validity], 0],
                     predicate="(or (lookup 0 (col c)) (= (col x) (u32 5)))", aggregate=True)
    pipe.set_variant(variant)
    pipe.set_lookup(0, table, n_bits)
    pipe.launch_aggregate(cabi.make_source([col, x], n))
    states, rows = pipe.fetch_aggregate()
    keep = valid & (hit | (np.arange(n) == 5))   # a NULL operand makes the OR NULL: the row is dropped
    assert rows == int(keep.sum())
    assert states[1][1] == (int(np.arange(n)[keep].sum()) & 0xFFFFFFFF if keep.any() else None)


@pytest.mark.parametrize("n_bits,validity,offset", CASES)
@pytest.mark.parametrize("variant", ["tma", "ldg"])
def test_lookup_in_map(cctx, n_bits, validity, offset, variant):
    from fuse_query_b200 import cabi
    n = 100_003
    table, col, x, hit, valid = lookup_case(cctx, n_bits, n, validity, 11 + n_bits + offset, offset)
    pipe = cctx.pipe(["(lookup 1 (col c))"], columns=["c"], dtypes=[cabi.U32], nullable=[NULLABLE[validity]])
    pipe.set_variant(variant)
    pipe.set_lookup(1, table, n_bits)
    out = cctx.column(cabi.BOOL, n)
    ov = cctx.column(cabi.BOOL, n) if validity != "none" else None
    pipe.launch_project(cabi.make_source([col], n), [out], n, out_valid=[ov] if ov is not None else None)
    assert pipe.fetch_project() == (n, n)
    got = out.to_numpy(n).astype(bool)
    if ov is not None:
        ok = ov.to_numpy(n).astype(bool)
        assert np.array_equal(ok, valid)
        assert np.array_equal(got[ok], hit[ok])
    else:
        assert np.array_equal(got, hit)


@pytest.mark.parametrize("n_bits,validity,offset", CASES)
def test_lookup_in_group_by(cctx, n_bits, validity, offset):
    from fuse_query_b200 import cabi
    n = 200_003
    table, col, x, hit, valid = lookup_case(cctx, n_bits, n, validity, 13 + n_bits + offset, offset)
    # key = the lookup, WHERE = a second lookup into the same table in another slot
    pipe = cctx.pipe(["(count (col x))"], columns=["c", "x"], dtypes=[cabi.U32, cabi.U32], nullable=[NULLABLE[validity], 0],
                     keys=["(lookup 0 (col c))"], predicate="(or (lookup 3 (col c)) (< (col x) (u32 1000)))")
    pipe.set_lookup(0, table, n_bits)
    pipe.set_lookup(3, table, n_bits)
    groups = pipe.run_groupby(cabi.make_source([col, x], n))
    keys, key_valid, leaves, _ = pipe.export_groups(groups)
    k = keys[0].to_numpy(groups).astype(bool).tolist()
    if key_valid[0] is not None:
        kv = key_valid[0].to_numpy(groups).astype(bool).tolist()
        k = [a if b else None for a, b in zip(k, kv)]
    got = dict(zip(k, leaves[0].to_numpy(groups).tolist()))
    keep = valid & (hit | (np.arange(n) < 1000))
    want = {}
    for h_, v_ in zip(hit[keep], valid[keep]):
        key = bool(h_) if v_ else None
        want[key] = want.get(key, 0) + 1
    assert got == want


def test_unbound_slot_and_bad_bindings(cctx):
    from fuse_query_b200 import cabi
    table, col, x, hit, valid = lookup_case(cctx, 100, 1000, "none", 1)
    pipe = cctx.pipe(["(count (col x))"], columns=["c", "x"], dtypes=[cabi.U32, cabi.U32], predicate="(lookup 1 (col c))", aggregate=True)
    with pytest.raises(cabi.FuseGpuError) as e:
        pipe.launch_aggregate(cabi.make_source([col, x], 1000))
    assert e.value.status == cabi.ERR_INVALID and "lookup slot 1" in str(e.value)
    for slot, bits in ((4, 100), (-1, 100), (1, 8 * 13 + 1)):
        with pytest.raises(cabi.FuseGpuError) as e:
            pipe.set_lookup(slot, table, bits)
        assert e.value.status == cabi.ERR_INVALID
    pipe.set_lookup(1, table, 100)
    pipe.launch_aggregate(cabi.make_source([col, x], 1000))
    assert pipe.fetch_aggregate()[1] == int(hit.sum())


def test_graph_replays_the_recorded_binding(cctx):
    from fuse_query_b200 import cabi
    table, col, x, hit, valid = lookup_case(cctx, 4097, 50_000, "none", 5)
    other = cctx.from_numpy(np.zeros(513, dtype=np.uint8))
    pipe = cctx.pipe(["(count (col x))"], columns=["c", "x"], dtypes=[cabi.U32, cabi.U32], predicate="(lookup 0 (col c))", aggregate=True)
    pipe.set_lookup(0, table, 4097)
    s = cctx.stream_create()
    src = cabi.make_source([col, x], 50_000)
    cctx.graph_begin(s)
    pipe.launch_aggregate(src, stream=s)
    g = cctx.graph_end(s)
    pipe.set_lookup(0, other, 4097)
    g.launch(s)
    assert pipe.fetch_aggregate()[1] == int(hit.sum())
    pipe.launch_aggregate(src, stream=s)
    assert pipe.fetch_aggregate()[1] == 0
    g.destroy()
    cctx.stream_destroy(s)


# ---- SQL ----
POOL = ["apple", "apricot", "banana", "a_b", "a%b", "Axe", "xylophone", "box", "", "a", "éa", "中文x", "😀x😀", "line\nx", "nul\0x", "a\\b"]


def make_table(n, pool, seed):
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, len(pool), n)
    nulls = rng.random(n) < 0.1
    s = [None if nulls[i] else pool[idx[i]] for i in range(n)]
    x = rng.integers(-1000, 1000, n).astype(np.int64)
    return pa.table({"s": pa.array(s, type=pa.string()), "x": x, "s2": pa.array([pool[(i * 7) % len(pool)] for i in range(n)])})


@pytest.fixture(scope="module")
def sql():
    from fuse_query_b200 import _fuse_host as h
    from fuse_query_b200.tables import register_table
    gpu = h.GpuContext.create(0)
    fctx = h.FuseQueryContext.create_ctx(4, gpu)
    small = make_table(60_000, POOL, 3)
    register_table(fctx, gpu, "default", "t", small)
    rng = np.random.default_rng(9)
    big_pool = [f"{v:09d}" for v in rng.permutation(1_000_000)]
    big = make_table(4_000_000, big_pool, 4)   # ~980 000 distinct strings
    register_table(fctx, gpu, "default", "big", big)

    def rows(q):
        out = []
        for b in h.execute_sql(fctx, q):
            out += list(zip(*[b.column(c).to_list() for c in range(b.num_columns())]))
        return out
    return {"h": h, "ctx": fctx, "tables": {"t": small, "big": big}, "rows": rows}


def arrow_mask(tbl, pattern, negate=False):
    m = pc.match_like(tbl["s"], pattern)
    return pc.invert(m) if negate else m


def smin(vals):
    vals = [v for v in vals if v is not None]
    return min(vals, key=str.encode) if vals else None


def smax(vals):
    vals = [v for v in vals if v is not None]
    return max(vals, key=str.encode) if vals else None


@pytest.mark.parametrize("table", ["t", "big"])
@pytest.mark.parametrize("pattern", ["a%", "%x%", "_", "a\\_b", "a\\%b", "%😀", "%\\\\%", "", "%", "%42%", "nul%"])
@pytest.mark.parametrize("negate", [False, True])
def test_aggregates_under_like(sql, table, pattern, negate):
    tbl = sql["tables"][table]
    kept = tbl.filter(arrow_mask(tbl, pattern, negate))
    op = "not like" if negate else "like"
    # (no sum under a WHERE that can empty a 10 000-row block: the reference's per-block Sum fold raises there, SURVEY F8; and
    # min / max only where some row is kept)
    if kept.num_rows == 0:
        assert sql["rows"](f"select count(x), count(s) from {table} where s {op} '{pattern}'") == [(0, 0)]
        return
    got = sql["rows"](f"select count(x), min(x), max(x), min(s), max(s), count(s) from {table} where s {op} '{pattern}'")
    s = kept["s"].to_pylist()
    want = (kept.num_rows, pc.min(kept["x"]).as_py(), pc.max(kept["x"]).as_py(), smin(s), smax(s), kept.num_rows)
    assert got == [want]


def test_like_with_numeric_predicates(sql):
    tbl = sql["tables"]["t"]
    m = arrow_mask(tbl, "a%")
    x = tbl["x"]
    for where, mask in [   # NULL in either operand of AND / OR drops the row, as every logic node of the device path("s like 'a%' and x > 0", pc.and_(m, pc.greater(x, 0))),
                        ("x < 500 or s not like '%b%'", pc.or_(pc.less(x, 500), arrow_mask(tbl, "%b%", True))),
                        ("s like 'a%' and s not like '%p%' or x = 7", pc.or_(pc.and_(m, arrow_mask(tbl, "%p%", True)), pc.equal(x, 7)))]:
        kept = tbl.filter(mask)
        assert sql["rows"](f"select count(x), max(x) from t where {where}") == [(kept.num_rows, pc.max(kept["x"]).as_py())], where


def test_like_as_a_projection(sql):
    tbl = sql["tables"]["t"]
    got = sql["rows"]("select s like 'a%' as f, s not like 'a%', x from t")
    want = list(zip(pc.match_like(tbl["s"], "a%").to_pylist(), pc.invert(pc.match_like(tbl["s"], "a%")).to_pylist(), tbl["x"].to_pylist()))
    assert got == want
    assert any(r[0] is None for r in got)


def test_group_by_like(sql):
    tbl = sql["tables"]["t"]
    got = sorted(sql["rows"]("select s like '%x%', count(x), sum(x) from t group by s like '%x%'"), key=repr)
    m = pc.match_like(tbl["s"], "%x%").to_pylist()
    want = {}
    for k, v in zip(m, tbl["x"].to_pylist()):
        c, t_ = want.get(k, (0, 0))
        want[k] = (c + 1, t_ + v)
    assert got == sorted([(k, c, t_) for k, (c, t_) in want.items()], key=repr)


def test_order_by_limit_under_like(sql):
    tbl = sql["tables"]["big"]
    got = sql["rows"]("select s, x from big where s like '%42%' order by s limit 10")
    kept = tbl.filter(arrow_mask(tbl, "%42%"))
    want = sorted(zip(kept["s"].to_pylist(), kept["x"].to_pylist()), key=lambda r: r[0].encode())
    assert [r[0] for r in got] == [r[0] for r in want[:10]]


def test_a_second_pattern_reuses_the_compiled_pipe(sql, tmp_path, monkeypatch):
    """the generated source depends on the lookup slot only: a query with another pattern finds the module of the first in
    the context's cache and builds nothing (no new cubin in the on-disk JIT cache)"""
    monkeypatch.setenv("FQ_JIT_CACHE_DIR", str(tmp_path))
    q = "select count(x), max(x) from t where s like '{}' and x > 11"
    sql["rows"](q.format("ap%"))
    built = sorted(os.listdir(tmp_path))
    assert built, "the first query builds its pipe"
    tbl = sql["tables"]["t"]
    kept = tbl.filter(pc.and_(arrow_mask(tbl, "%an%"), pc.greater(tbl["x"], 11)))
    assert sql["rows"](q.format("%an%")) == [(kept.num_rows, pc.max(kept["x"]).as_py())]
    assert sorted(os.listdir(tmp_path)) == built


def test_lookup_pipe_source_names_the_slot_not_the_pattern(cctx):
    from fuse_query_b200 import cabi
    arr = cctx.utf8(["x", "y"])
    codes, dictionary = arr.dict_encode()
    p1 = cctx.pipe(["(count (col c))"], columns=["c"], dtypes=[cabi.U32], predicate="(lookup 0 (col c))", aggregate=True)
    p2 = cctx.pipe(["(count (col c))"], columns=["c"], dtypes=[cabi.U32], predicate="(lookup 0 (col c))", aggregate=True)
    for pipe, pattern, want in ((p1, "x", 1), (p2, "%", 2)):
        pipe.set_lookup(0, dictionary.like(pattern), len(dictionary))
        pipe.launch_aggregate(cabi.make_source([codes], 2))
        assert pipe.fetch_aggregate()[1] == want
    assert p1.source == p2.source


@pytest.mark.parametrize("q,err", [
    ("select count(x) from t where s like s2", "Internal Error: Unsupported on the device path: LIKE with a pattern that is not a string literal"),
    ("select count(x) from t where x like 'a%'", "Internal Error: Unsupported (Int64) LIKE (Utf8)"),
    ("select count(x) from t where s like 'a\\'", "Internal Error: LIKE pattern ends with the escape character \\"),
    ("select count(x) from t where s like 'a' or s like 'b' or s like 'c' or s like 'd' or s like 'e'",
     "Internal Error: Unsupported on the device path: more than 4 LIKE predicates in one pipe"),
    ("select count(x) from t where not (s like 'a')", "Error during plan: Unsupported ExpressionPlan: NOT s LIKE 'a'"),
])
def test_refusals(sql, q, err):
    with pytest.raises(sql["h"].FuseQueryError) as e:
        sql["rows"](q)
    assert str(e.value) == err
