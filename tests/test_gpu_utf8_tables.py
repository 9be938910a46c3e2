"""Utf8 columns on the device: dictionary encoding through the C ABI, and SQL over a registered table with a string column
(WHERE, GROUP BY, ORDER BY, count / min / max), checked against plain Python bytewise order."""
import bisect
import operator

import numpy as np
import pyarrow as pa
import pyarrow.parquet as pq
import pytest

pytestmark = pytest.mark.gpu

OPS = {"=": operator.eq, "<": operator.lt, "<=": operator.le, ">": operator.gt, ">=": operator.ge}
FLIP = {"=": "=", "<": ">", "<=": ">=", ">": "<", ">=": "<="}


@pytest.fixture(scope="module")
def cctx():
    from fuse_query_b200 import cabi
    ctx = cabi.Context(0)
    yield ctx
    ctx.close()


def encode(ctx, values):
    arr = ctx.utf8(values)
    codes, dictionary = arr.dict_encode()
    return arr, codes, dictionary


def check_encoding(ctx, values):
    arr, codes, dictionary = encode(ctx, values)
    want = sorted({v.encode() for v in values if v is not None})
    got_dict = dictionary.to_list()
    assert got_dict == want
    rank = {b: i for i, b in enumerate(want)}
    got = codes.to_numpy(len(values)).tolist() if values else []
    for v, c in zip(values, got):
        if v is not None:
            assert c == rank[v.encode()], (v, c)
    # decoding the codes through the dictionary gives the column back, NULLs included
    if values:
        back = dictionary.take(codes, len(values), arr._valid).to_list()
        assert back == [None if v is None else v.encode() for v in values]
    return want, dictionary


LENGTHS = ["", "a" * 7, "a" * 8, "a" * 9, "a" * 15, "a" * 16, "a" * 17, "a" * 300, "a" * 299 + "b", "b" * 8, "a" * 8 + "\0"]
PREFIXES = ["abc", "ab", "abcd", "ab\0", "ab\0\0", "a", "", "ab\x01", "abc\0", "abb"]
LONG_PREFIX = ["p" * 100 + s for s in ("", "a", "b", "ab", "\0", "zz", "a" * 40)]
NON_ASCII = ["é", "e", "日本", "日", "z", "ÿ", "Ä", "ä", "€", "\x7f"]


@pytest.mark.parametrize("values", [
    LENGTHS * 3,
    PREFIXES + PREFIXES[::-1],
    LONG_PREFIX * 2,
    NON_ASCII + [None] + NON_ASCII,
    [None] * 5,
    [],
    ["same"] * 1000,
    ["x", None, "x", None],
], ids=["lengths", "prefixes", "long_prefix", "non_ascii", "all_null", "zero_rows", "one_value", "one_value_nulls"])
def test_encoder_codes_are_ranks(cctx, values):
    check_encoding(cctx, values)


@pytest.mark.parametrize("distinct", [4095, 4096, 4097, 8193])
def test_encoder_around_the_sort_tile(cctx, distinct):
    rng = np.random.default_rng(distinct)
    pool = [f"k{i:06d}" * int(rng.integers(1, 4)) for i in range(distinct)]
    values = [pool[i] for i in rng.permutation(np.concatenate([np.arange(distinct), rng.integers(0, distinct, 3000)]))]
    check_encoding(cctx, values)


def test_encoder_a_million_unique_strings(cctx):
    rng = np.random.default_rng(1)
    values = [f"{v:x}" for v in rng.permutation(1_000_000)]
    check_encoding(cctx, values)


def test_bounds_of_literals(cctx):
    values = PREFIXES + NON_ASCII + LENGTHS
    want, dictionary = check_encoding(cctx, values)
    for lit in ["", "a", "ab", "ab\0", "aa", "abz", "é", "zzz", "\0", "a" * 8, "a" * 301]:
        b = lit.encode()
        assert dictionary.bounds(lit) == (bisect.bisect_left(want, b), bisect.bisect_right(want, b)), lit


# ---- SQL over a registered table ----
POOL = ["Paris", "paris", "Paris\0", "", "a", "ab", "abc", "b", "zz", "Zurich", "日本", "é", "x" * 20, "x" * 21, "Lyon", "Berlin"]
N = 50_000


def make_table():
    rng = np.random.default_rng(7)
    idx = rng.integers(0, len(POOL), N)
    nulls = rng.random(N) < 0.1
    s = [None if nulls[i] else POOL[idx[i]] for i in range(N)]
    s2 = [POOL[(i * 7) % len(POOL)] for i in range(N)]
    x = rng.integers(-1000, 1000, N).astype(np.int64)
    ranks = {b: i for i, b in enumerate(sorted({v.encode() for v in s if v is not None}))}
    k = np.array([0 if v is None else ranks[v.encode()] for v in s], dtype=np.uint32)
    tbl = pa.table({"s": pa.array(s, type=pa.string()), "x": x, "k": pa.array(k, mask=nulls), "s2": pa.array(s2).dictionary_encode()})
    return tbl, s, s2, x.tolist()


@pytest.fixture(scope="module")
def sql():
    from fuse_query_b200 import _fuse_host as h
    from fuse_query_b200.tables import register_table
    gpu = h.GpuContext.create(0)
    fctx = h.FuseQueryContext.create_ctx(4, gpu)
    tbl, s, s2, x = make_table()
    register_table(fctx, gpu, "default", "t", tbl)

    def rows(q):
        out = []
        for b in h.execute_sql(fctx, q):
            out += list(zip(*[b.column(c).to_list() for c in range(b.num_columns())]))
        return out
    return {"h": h, "gpu": gpu, "ctx": fctx, "tbl": tbl, "s": s, "s2": s2, "x": x, "rows": rows}


def key(v):
    return (v is not None, b"" if v is None else v.encode())


LITERALS = ["Paris", "", "zz", "ab", "Pari", "m", "zzz", "Berlin", "日本", "aa"]


@pytest.mark.parametrize("op", list(OPS))
@pytest.mark.parametrize("lit", LITERALS)
def test_comparisons_against_literals(sql, op, lit):
    want = sum(1 for v in sql["s"] if v is not None and OPS[op](v.encode(), lit.encode()))
    assert sql["rows"](f"select count(x) from t where s {op} '{lit}'") == [(want,)]
    assert sql["rows"](f"select count(x) from t where '{lit}' {FLIP[op]} s") == [(want,)]


def test_filtered_projection(sql):
    want = [(v, x) for v, x in zip(sql["s"], sql["x"]) if v is not None and v.encode() < b"b" and x > 0]
    assert sorted(sql["rows"]("select s, x from t where s < 'b' and x > 0"), key=repr) == sorted(want, key=repr)


def test_count_min_max_of_a_string(sql):
    valid = [v for v in sql["s"] if v is not None]
    (cnt_k,) = sql["rows"]("select count(k) from t")[0]
    got = sql["rows"]("select count(s), min(s), max(s) from t")
    assert got == [(cnt_k, min(valid, key=str.encode), max(valid, key=str.encode))]
    sel = [v for v, x in zip(sql["s"], sql["x"]) if v is not None and x > 500]
    (cnt_k2,) = sql["rows"]("select count(k) from t where x > 500")[0]
    got = sql["rows"]("select count(s), min(s), max(s) from t where x > 500")
    assert got == [(cnt_k2, min(sel, key=str.encode), max(sel, key=str.encode))]


def groups(sql):
    g = {}
    for v, x in zip(sql["s"], sql["x"]):
        g.setdefault(v, []).append(x)
    return g


def test_group_by_a_string(sql):
    got = sql["rows"]("select s, sum(x), count(x), min(x), max(x), min(s), max(s) from t group by s")
    want = [(v, sum(xs), len(xs), min(xs), max(xs), v, v) for v, xs in groups(sql).items()]
    assert sorted(got, key=lambda r: key(r[0])) == sorted(want, key=lambda r: key(r[0]))


def test_group_by_order_by_desc_limit(sql):
    got = sql["rows"]("select s, count(x) from t group by s order by s desc limit 5")
    g = groups(sql)
    keys = [None] + sorted([v for v in g if v is not None], key=str.encode, reverse=True)   # NULLs first, both directions
    assert got == [(v, len(g[v])) for v in keys[:5]]


def test_order_by_string_then_number(sql):
    got = sql["rows"]("select s, x from t order by s, x")
    want = sorted(zip(sql["s"], sql["x"]), key=lambda r: (key(r[0]), r[1]))
    assert got == want


def test_parquet_round_trip(sql, tmp_path):
    from fuse_query_b200.tables import register_parquet
    path = tmp_path / "t.parquet"
    pq.write_table(sql["tbl"], str(path))
    register_parquet(sql["ctx"], sql["gpu"], "default", "tp", path, columns=["s", "x"])
    q = "select s, count(x), sum(x) from {} where s >= 'Paris' group by s"
    assert sorted(sql["rows"](q.format("tp")), key=repr) == sorted(sql["rows"](q.format("t")), key=repr)


@pytest.mark.parametrize("q, text", [
    ("select s + 1 from t", "Unsupported (Utf8) + ("),
    ("select count(x) from t where s = 1", "Unsupported (Utf8) = ("),
    ("select sum(s) from t", "Unsupported data_array_sum for data type: Utf8"),
    ("select count(x) from t where s = s2", "Unsupported on the device path: comparison of two Utf8 columns with different dictionaries"),
])
def test_error_texts(sql, q, text):
    with pytest.raises(sql["h"].FuseQueryError) as e:
        sql["rows"](q)
    assert text in str(e.value)


@pytest.mark.parametrize("q", [
    "select s, x from t where s < 'b' and x > 0",
    "select s, s2, x from t",
    "select count(s), min(s), max(s), sum(x) from t where s >= 'Paris'",
    "select min(s2), max(s2), count(x) from t where s2 < 'x'",
])
def test_fused_and_reference_shaped_pipelines_agree(sql, q):
    fused = sorted(sql["rows"](q), key=repr)
    sql["ctx"].options.fuse = False
    try:
        plain = sorted(sql["rows"](q), key=repr)
    finally:
        sql["ctx"].options.fuse = True
    assert fused == plain


@pytest.mark.parametrize("op", ["Eq", "Lt", "LtEq", "Gt", "GtEq"])
def test_array_comparison_op_agrees_with_sql(sql, op):
    h = sql["h"]
    from fuse_query_b200.tables import utf8_parts
    arr = h.DataArray.from_utf8(sql["gpu"], *utf8_parts(sql["tbl"].column("s")))
    lit = h.DataValue(h.DataType.Utf8, "Paris")
    got = h.data_array_comparison_op(sql["gpu"], getattr(h.ops, op), h.DataColumnarValue.Array(arr), h.DataColumnarValue.Scalar(lit)).to_list()
    sym = {"Eq": "=", "Lt": "<", "LtEq": "<=", "Gt": ">", "GtEq": ">="}[op]
    assert got == [None if v is None else OPS[sym](v.encode(), b"Paris") for v in sql["s"]]
    flipped = h.data_array_comparison_op(sql["gpu"], getattr(h.ops, op), h.DataColumnarValue.Scalar(lit), h.DataColumnarValue.Array(arr)).to_list()
    assert flipped == [None if v is None else OPS[sym](b"Paris", v.encode()) for v in sql["s"]]
    # the SQL path (codes against the literal's bounds) gives the same value per string
    assert sorted(sql["rows"](f"select s, s {sym} 'Paris' from t"), key=repr) == sorted(zip(sql["s"], got), key=repr)
    assert arr.dictionary() == sorted({v for v in sql["s"] if v is not None}, key=str.encode)
