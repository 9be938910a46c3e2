"""GROUP BY keys of 65..128 bits on the device (two-word table keys claimed by one 16-byte compare-and-swap): a nullable
64-bit key, pairs of 64-bit keys, mixed key sets and two nullable Utf8 keys, through the C ABI and SQL.  Checked against
the GROUP BY oracle (oracle/groupby.py) on a few 10^5 rows, against numpy closed forms at high cardinality and against
pyarrow's group_by for SQL.  Row order of a GROUP BY is unspecified: results are compared as sorted row lists, exactly;
float keys group, and are compared, by bit pattern."""
import numpy as np
import pyarrow as pa
import pytest

from fuse_query_b200 import cabi
from oracle import binding as o
from oracle.groupby import run_group_by
from test_groupby_wide_keys_host import wide_keys

pytestmark = pytest.mark.gpu
NUM = "(col number)"
M64 = (1 << 64) - 1
LEAVES = [f"(sum {NUM})", f"(count {NUM})", f"(min {NUM})", f"(max (+ {NUM} (u64 1)))"]


@pytest.fixture(scope="module")
def ctx():
    c = cabi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sql():
    from fuse_query_b200 import _fuse_host as h
    from fuse_query_b200.tables import register_table
    gpu = h.GpuContext.create(0)
    fctx = h.FuseQueryContext.create_ctx(4, gpu)

    def rows(q):
        out = []
        for b in h.execute_sql(fctx, q):
            out += list(zip(*[b.column(c).to_list() for c in range(b.num_columns())]))
        return out

    def register(name, table):
        register_table(fctx, gpu, "default", name, table)
    return {"h": h, "rows": rows, "register": register}


def mod(k):
    return f"(- {NUM} (* (/ {NUM} (u64 {k})) (u64 {k})))"


def wide(k):
    """number % k, number % k * 3: 128 bits, k groups"""
    return [mod(k), f"(* {mod(k)} (u64 3))"]


def fetch_rows(pipe, n_groups, float_keys=()):
    """exported groups as sorted python rows: keys then leaves, None for NULL; keys listed in float_keys as their bits"""
    keys, kval, leaves, lval = pipe.export_groups(n_groups)
    cols = []
    for j, (c, v) in enumerate(list(zip(keys, kval)) + list(zip(leaves, lval))):
        a = c.to_numpy(n_groups)
        vals = a.view(np.uint64 if a.itemsize == 8 else np.uint32).tolist() if j in float_keys else a.tolist()
        if v is not None:
            ok = v.to_numpy(n_groups).astype(bool).tolist()
            vals = [x if f else None for x, f in zip(vals, ok)]
        cols.append(vals)
    rows = list(zip(*cols)) if n_groups else []
    nk = len(keys)
    rows.sort(key=lambda r: tuple((x is not None, x) for x in r[:nk]))
    for c in keys + leaves + [x for x in kval + lval if x is not None]:
        c.free()
    return rows


def bitmap(valid, offset):
    """Arrow LSB-first bitmap of `valid` starting at bit `offset`"""
    bits = np.concatenate([np.zeros(offset, dtype=bool), valid])
    return np.packbits(bits, bitorder="little")


# ---- 1. a nullable UInt64 key: 65 bits ----
@pytest.mark.parametrize("validity", ["bytes", "bitmap"])
def test_nullable_u64_key(ctx, validity):
    rng = np.random.default_rng(11)
    n = 200_003
    pool = np.array([0, 1, 2, M64, M64 - 1, 1 << 63, 12345678901234567890] + rng.integers(0, 1 << 63, 90, dtype=np.uint64).tolist(), dtype=np.uint64)
    a = pool[rng.integers(0, len(pool), n)]
    a_ok = rng.random(n) > 0.07
    v = rng.integers(-10**9, 10**9, n).astype(np.int64)
    v_ok = rng.random(n) > 0.15
    if validity == "bytes":
        ca = ctx.from_numpy(a, a_ok)
    else:
        ca = ctx.from_numpy(a, valid_bitmap=bitmap(a_ok, 3), bit_offset=3)
    cols = [ca, ctx.from_numpy(v, v_ok)]
    aggs = ["(sum (col v))", "(count (col v))", "(min (col v))", "(max (col v))"]
    pipe = ctx.pipe(aggs, keys=["(col a)"], columns=["a", "v"], dtypes=[cabi.U64, cabi.I64],
                    nullable=[2 if validity == "bitmap" else True, True])
    groups = pipe.run_groupby(cabi.make_source(cols, n), groups_hint=4)
    table = {"a": o.Array(o.U64, a, a_ok.astype(np.uint8)), "v": o.Array(o.I64, v, v_ok.astype(np.uint8))}
    _, want = run_group_by(["(col a)"], aggs, table=table)
    assert groups == len(want) == len(np.unique(a[a_ok])) + 1
    assert fetch_rows(pipe, groups) == want
    pipe.destroy()


# ---- 2. two 64-bit keys (128 bits) with the all-ones pair; a nullable Float64 key with an Int32 key (97 bits) ----
def test_u64_i64_pair_with_the_empty_mark_key(ctx):
    rng = np.random.default_rng(12)
    n = 150_001
    a = rng.choice(np.array([0, 5, M64, M64 - 1, 1 << 63], dtype=np.uint64), n)
    b = rng.choice(np.array([-1, 0, 7, -(1 << 63), (1 << 63) - 1], dtype=np.int64), n)
    a[::101], b[::101] = np.uint64(M64), -1            # (2^64 - 1, -1): both words all ones, the table's EMPTY mark
    v = rng.integers(-1000, 1000, n).astype(np.int32)
    cols = [ctx.from_numpy(a), ctx.from_numpy(b), ctx.from_numpy(v)]
    aggs = ["(sum (col v))", "(count (col v))", "(min (col v))", "(max (col v))"]
    pipe = ctx.pipe(aggs, keys=["(col a)", "(col b)"], columns=["a", "b", "v"], dtypes=[cabi.U64, cabi.I64, cabi.I32])
    groups = pipe.run_groupby(cabi.make_source(cols, n))
    _, want = run_group_by(["(col a)", "(col b)"], aggs, table={"a": o.from_numpy(a), "b": o.from_numpy(b), "v": o.from_numpy(v)})
    assert groups == len(want) == 25
    got = fetch_rows(pipe, groups)
    assert got == want
    assert (M64, -1) in [r[:2] for r in got]
    pipe.destroy()


def test_nullable_f64_key_with_an_i32_key(ctx):
    rng = np.random.default_rng(13)
    n = 120_007
    nan_bits = np.array([0x7FF8000000000000, 0x7FF8000000012345, 0xFFF8000000000005, 0x7FF0000000000001], dtype=np.uint64)
    pool = np.concatenate([np.array([0.0, -0.0, 1.5, -2.25, np.inf, -np.inf, 5e-324]), nan_bits.view(np.float64)])
    f = pool[rng.integers(0, len(pool), n)]
    f_ok = rng.random(n) > 0.1
    k = rng.integers(-3, 3, n).astype(np.int32)
    v = rng.integers(-10**6, 10**6, n).astype(np.int64)
    cols = [ctx.from_numpy(f, f_ok), ctx.from_numpy(k), ctx.from_numpy(v)]
    aggs = ["(sum (col v))", "(count (col v))", "(min (col v))", "(max (col v))"]
    pipe = ctx.pipe(aggs, keys=["(col f)", "(col k)"], columns=["f", "k", "v"], dtypes=[cabi.F64, cabi.I32, cabi.I64], nullable=[True, False, False])
    groups = pipe.run_groupby(cabi.make_source(cols, n))
    # numpy reference, grouped by (validity, bit pattern, k)
    fb = np.where(f_ok, f.view(np.uint64), 0)
    ref = {}
    for fv, ok, kv, vv in zip(fb.tolist(), f_ok.tolist(), k.tolist(), v.tolist()):
        g = ref.setdefault((fv if ok else None, kv), [0, 0, None, None])
        g[0] += vv
        g[1] += 1
        g[2] = vv if g[2] is None else min(g[2], vv)
        g[3] = vv if g[3] is None else max(g[3], vv)
    want = sorted([key + tuple(s) for key, s in ref.items()], key=lambda r: tuple((x is not None, x) for x in r[:2]))
    assert groups == len(want) == (len(pool) + 1) * 6
    assert fetch_rows(pipe, groups, float_keys=(0,)) == want
    pipe.destroy()


# ---- 3. every table level and growth, materialised and generated ----
def closed_form(n, k):
    x = np.arange(n, dtype=np.uint64)
    key = (x % np.uint64(k)).astype(np.int64)
    g = min(k, n)
    cnt = np.bincount(key, minlength=g)
    sm = np.zeros(g, dtype=np.uint64)
    np.add.at(sm, key, x)
    mn = np.arange(g, dtype=np.uint64)                  # the first row of group r is r
    mx = mn + np.uint64(k) * ((np.uint64(n) - 1 - mn) // np.uint64(k))
    return list(zip(range(g), (3 * np.arange(g)).tolist(), sm.tolist(), cnt.tolist(), mn.tolist(), (mx + np.uint64(1)).tolist()))


@pytest.mark.parametrize("generated", [False, True])
@pytest.mark.parametrize("k", [7, 1000, 5000, 1_000_000])     # shared memory, shared memory and replicas, replicas, HBM only
def test_wide_keys_at_every_table_level(ctx, k, generated):
    n = 3_000_000
    col = None if generated else ctx.numbers(0, n)
    pipe = ctx.pipe(LEAVES, keys=wide(k), generated=generated)
    src = cabi.make_source([] if generated else [col], n, generated=generated)
    groups = pipe.run_groupby(src, groups_hint=4)
    assert groups == k
    assert fetch_rows(pipe, groups) == closed_form(n, k)
    pipe.destroy()
    if col is not None:
        col.free()


def test_wide_keys_match_the_oracle(ctx):
    n = 200_003
    pipe = ctx.pipe(LEAVES, keys=wide(1000))
    groups = pipe.run_groupby(cabi.make_source([ctx.numbers(0, n)], n), groups_hint=4)
    _, want = run_group_by(wide(1000), LEAVES, total=n)
    assert fetch_rows(pipe, groups) == want
    pipe.destroy()


# ---- 4. accumulate across launches; partial exchange among three ranks ----
def test_accumulate_and_partial_exchange(ctx):
    n, k = 1_000_000, 5003
    col = ctx.numbers(0, n)
    keys = wide(k)
    pipe = ctx.pipe(LEAVES, keys=keys)
    assert pipe.group_entry_slots() == 2 + 1 + len(LEAVES)      # two key words + G state slots (rows, 4 leaves)
    pipe.groupby_reserve(k)
    half = 500_000
    pipe.launch_groupby(cabi.make_source([col.slice(0, half)], half))
    pipe.launch_groupby(cabi.make_source([col.slice(half, n - half)], n - half), accumulate=True)
    assert pipe.fetch_groupby() == k
    want = closed_form(n, k)
    assert fetch_rows(pipe, k) == want
    world, bounds, parts = 3, [0, 333_334, 666_668, n], []
    for r in range(world):
        p = ctx.pipe(LEAVES, keys=keys)
        m = bounds[r + 1] - bounds[r]
        g = p.run_groupby(cabi.make_source([col.slice(bounds[r], m)], m))
        ent = ctx.column(cabi.U64, g * p.group_entry_slots())
        counts = p.export_partials(world, ent)
        assert sum(counts) == g == k
        parts.append((p, ent, counts))
    slots = parts[0][0].group_entry_slots()
    owned = []
    for owner in range(world):
        q = ctx.pipe(LEAVES, keys=keys)
        q.groupby_reserve(k)
        for i, (p, ent, counts) in enumerate(parts):
            off = sum(counts[:owner])
            q.merge_partials(ent.slice(off * slots, counts[owner] * slots), counts[owner], accumulate=i > 0)
        owned.append(fetch_rows(q, q.fetch_groupby()))
        q.destroy()
    owner_keys = [{r[:2] for r in rows} for rows in owned]
    assert all(not (owner_keys[i] & owner_keys[j]) for i in range(world) for j in range(i + 1, world))
    assert sorted(r for rows in owned for r in rows) == want
    for p, ent, _ in parts:
        p.destroy()
        ent.free()
    pipe.destroy()


# ---- 5. constructed collisions: every key in one probe chain of the first table ----
def collision_table(count, rows=200_000, seed=0):
    rng = np.random.default_rng(seed)
    pairs = np.array(wide_keys(count), dtype=np.uint64)
    idx = rng.permutation(np.concatenate([np.arange(count), rng.integers(0, count, rows - count)]))
    v = rng.integers(-10**6, 10**6, rows).astype(np.int64)
    return pairs[idx, 0].copy(), pairs[idx, 1].copy(), v


def collision_groups(lo, hi, v):
    ref = {}
    for a, b, x in zip(lo.tolist(), hi.tolist(), v.tolist()):
        g = ref.setdefault((a, b), [0, 0, x, x])
        g[0] += x
        g[1] += 1
        g[2] = min(g[2], x)
        g[3] = max(g[3], x)
    return sorted(key + tuple(s) for key, s in ref.items())


COLLISION_AGGS = ["(sum (col v))", "(count (col v))", "(min (col v))", "(max (col v))"]


@pytest.mark.parametrize("count", [3000, 6000])
def test_constructed_collisions(ctx, count):
    lo, hi, v = collision_table(count)
    cols = [ctx.from_numpy(lo), ctx.from_numpy(hi), ctx.from_numpy(v)]
    kw = dict(columns=["lo", "hi", "v"], dtypes=[cabi.U64, cabi.U64, cabi.I64])
    src = cabi.make_source(cols, len(v))
    pipe = ctx.pipe(COLLISION_AGGS, keys=["(col lo)", "(col hi)"], **kw)
    pipe.groupby_reserve(1 << 16)
    pipe.launch_groupby(src)
    if count > 4096:                                    # a chain longer than the probe limit: the seed-0 table overflows
        with pytest.raises(cabi.FuseGpuError) as e:
            pipe.fetch_groupby()
        assert e.value.status == cabi.ERR_CAPACITY
        pipe.groupby_reserve(1 << 16)                   # same size, a new seed
        pipe.launch_groupby(src)
    groups = pipe.fetch_groupby()
    assert groups == count
    assert fetch_rows(pipe, groups) == collision_groups(lo, hi, v)
    pipe.destroy()


def test_sql_constructed_collisions(sql):
    lo, hi, v = collision_table(6000, seed=1)
    sql["register"]("wide_collisions", {"lo": lo, "hi": hi, "v": v})
    got = sql["rows"]("select lo, hi, sum(v), count(v), min(v), max(v) from wide_collisions group by lo, hi")
    assert sorted(got) == collision_groups(lo, hi, v)


# ---- 6. SQL over a registered table against pyarrow ----
def sql_table(n=100_000, seed=21):
    rng = np.random.default_rng(seed)
    a = rng.integers(-(1 << 62), 1 << 62, 50)[rng.integers(0, 50, n)]
    a_null = rng.random(n) < 0.08
    b = rng.integers(-5, 5, n)
    b_null = rng.random(n) < 0.1
    c = rng.integers(0, 1000, n)
    c_null = rng.random(n) < 0.05
    words = ["alpha", "beta", "gamma", "", "delta", "日本", "zz"]
    s1 = [None if rng.random() < 0.1 else words[i] for i in rng.integers(0, len(words), n)]
    s2 = [None if rng.random() < 0.2 else words[i] for i in rng.integers(0, 4, n)]
    f = np.array([0.5, -1.0, 2.0, 1e300, -0.25])[rng.integers(0, 5, n)]
    f_null = rng.random(n) < 0.1
    i = rng.integers(-(1 << 40), 1 << 40, 20)[rng.integers(0, 20, n)]
    j = rng.integers(-3, 3, n).astype(np.int32)
    m = rng.integers(-(1 << 31), (1 << 31) - 1, 8)[rng.integers(0, 8, n)].astype(np.int32)
    m_null = rng.random(n) < 0.1
    x = rng.integers(-1000, 1000, n)
    return pa.table({"a": pa.array(a, mask=a_null), "b": pa.array(b, mask=b_null), "c": pa.array(c, mask=c_null), "s1": pa.array(s1, type=pa.string()),
                     "s2": pa.array(s2, type=pa.string()), "f": pa.array(f, mask=f_null), "i": pa.array(i), "j": pa.array(j),
                     "m": pa.array(m, mask=m_null), "x": pa.array(x)})


@pytest.fixture(scope="module")
def sql_t(sql):
    tbl = sql_table()
    sql["register"]("wt", tbl)
    return tbl


def arrow_groups(tbl, keys, where=None):
    """pyarrow's group_by: key columns, then sum / count / min / max of x, as python rows sorted with NULL first"""
    if where is not None:
        tbl = tbl.filter(where)
    g = tbl.group_by(keys).aggregate([("x", "sum"), ("x", "count"), ("x", "min"), ("x", "max")])
    g = g.select(keys + ["x_sum", "x_count", "x_min", "x_max"])
    rows = list(zip(*[g.column(i).to_pylist() for i in range(g.num_columns)]))
    return sorted(rows, key=lambda r: tuple((v is not None, v.encode() if isinstance(v, str) else v) for v in r[:len(keys)]))


def sorted_sql(rows, nk):
    return sorted(rows, key=lambda r: tuple((v is not None, v.encode() if isinstance(v, str) else v) for v in r[:nk]))


# 65, 2 x 33, 32 + 65 and 64 + 33 bits
@pytest.mark.parametrize("keys", [["a"], ["s1", "s2"], ["j", "f"], ["i", "m"]], ids=["nullable_i64", "two_nullable_utf8", "i32_nullable_f64", "i64_nullable_i32"])
def test_sql_group_by_against_pyarrow(sql, sql_t, keys):
    import pyarrow.compute as pc
    k = ", ".join(keys)
    got = sql["rows"](f"select {k}, sum(x), count(x), min(x), max(x) from wt group by {k}")
    assert sorted_sql(got, len(keys)) == arrow_groups(sql_t, keys)
    got = sql["rows"](f"select {k}, sum(x), count(x), min(x), max(x) from wt where x > 100 group by {k}")
    assert sorted_sql(got, len(keys)) == arrow_groups(sql_t, keys, pc.field("x") > 100)


def test_sql_order_by_and_limit_after_a_wide_group_by(sql, sql_t):
    want = arrow_groups(sql_t, ["s1", "s2"])[:7]        # NULL first, then bytewise, last key fastest
    got = sql["rows"]("select s1, s2, sum(x), count(x), min(x), max(x) from wt group by s1, s2 order by s1, s2 limit 7")
    assert got == want
    want = arrow_groups(sql_t, ["a"])
    got = sql["rows"]("select a, sum(x), count(x), min(x), max(x) from wt group by a order by a limit 5")
    assert got == want[:5]


@pytest.mark.parametrize("keys, bits", [("a, b, c", 195), ("i, f", 129)])
def test_sql_keys_over_128_bits_are_refused(sql, sql_t, keys, bits):
    with pytest.raises(sql["h"].FuseQueryError) as e:
        sql["rows"](f"select {keys}, count(x) from wt group by {keys}")
    assert f"GROUP BY keys of {bits} bits" in str(e.value) and "do not pack into 64 or 128" in str(e.value)
