"""Inputs that random data does not produce: strings whose 64-bit hashes are equal (the dictionary encoder's byte compare
behind a matching tag), GROUP BY keys whose hashes share their low 43 bits (one probe chain in every table size), and
sizes at which the shared exclusive scan (fq_scan_sums) needs more than one round of its single CTA (ORDER BY, dictionary
encoding and the Utf8 take).  The CPU tests restate the two device hashes in Python, pin them to the kernel source compiled
with g++, and prove that every constructed input collides under the kernel's own code; the GPU tests then run those inputs
against Python, numpy and closed forms."""
import collections
import ctypes as C
import functools
import os
import random
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = os.path.join(ROOT, "fuse_query_b200", "csrc", "kernels")

M64 = (1 << 64) - 1
K0 = 0x9E3779B97F4A7C15
C1, C2 = 0xFF51AFD7ED558CCD, 0xC4CEB9FE1A85EC53
INV1, INV2 = pow(C1, -1, 1 << 64), pow(C2, -1, 1 << 64)
GB_EMPTY = M64                      # FQ_GB_EMPTY: the key that equals the GROUP BY table's free mark
CLUSTER_BITS = 43                   # low hash bits the clustered GROUP BY keys share: one home slot up to 2^43 slots
SAFE = bytes(b for b in range(0x20, 0x7F) if b not in b"'\\")   # printable, and usable inside a SQL string literal


# ---- the two device hashes, their inverses and the constructors (pure Python) ----
def _xs(x, s):
    return x ^ (x >> s)


def _unxs(y, s):
    x = y
    for _ in range(64 // s + 1):
        x = y ^ (x >> s)
    return x


def _utf8_round(h, w):
    return _xs(((h ^ w) * C1) & M64, 32)


def _utf8_unround(after, before):
    """the 8-byte word w with _utf8_round(before, w) == after"""
    return ((_unxs(after, 32) * INV1) & M64) ^ before


def _utf8_fin(x):
    return _xs((_xs((x * C2) & M64, 29) * C1) & M64, 32)


def _utf8_unfin(h):
    return (_unxs((_unxs(h, 32) * INV1) & M64, 29) * INV2) & M64


def utf8_hash(b: bytes) -> int:
    """fq_utf8_hash (kernels/fq_utf8.cuh): 8-byte little-endian words, then the zero-padded tail and a finaliser"""
    h, i = K0 ^ len(b), 0
    while i + 8 <= len(b):
        h = _utf8_round(h, int.from_bytes(b[i:i + 8], "little"))
        i += 8
    return _utf8_fin(h ^ int.from_bytes(b[i:], "little"))


def gb_hash(k: int) -> int:
    """fq_gb_hash (kernels/fq_skeleton.cuh): murmur3's fmix64, a bijection of u64"""
    k = (_xs(k, 33) * C1) & M64
    k = (_xs(k, 33) * C2) & M64
    return _xs(k, 33)


def gb_unhash(h: int) -> int:
    h = (_unxs(h, 33) * INV2) & M64
    h = (_unxs(h, 33) * INV1) & M64
    return _unxs(h, 33)


def string_with_hash(target: int, n: int, rng: random.Random) -> bytes:
    """n (>= 8) printable bytes whose fq_utf8_hash is `target`: every byte but the last full 8-byte word is drawn at random,
    that word is solved for (each step of the hash inverts), and the draw is repeated until the solved word is printable
    too (about 1 draw in 2800 for this alphabet)."""
    free = 8 * (n // 8 - 1)
    while True:
        head = bytes(rng.choice(SAFE) for _ in range(free))
        tail = bytes(rng.choice(SAFE) for _ in range(n % 8))
        h = K0 ^ n
        for i in range(0, free, 8):
            h = _utf8_round(h, int.from_bytes(head[i:i + 8], "little"))
        w = _utf8_unround(_utf8_unfin(target) ^ int.from_bytes(tail, "little"), h).to_bytes(8, "little")
        if all(c in SAFE for c in w):
            return head + w + tail


@functools.lru_cache(maxsize=None)
def colliders():
    """(64 distinct 16-byte strings with one 64-bit hash, a 12-byte string with the same hash, a 16-byte string whose hash
    tag (upper 32 bits) is 0xFFFFFFFF: next to FQ_DICT_EMPTY once the row is packed beside it)"""
    rng = random.Random(20261020)
    target = rng.getrandbits(64)
    same = []
    while len(same) < 64:
        s = string_with_hash(target, 16, rng)
        if s not in same:
            same.append(s)
    short = string_with_hash(target, 12, rng)
    ones = string_with_hash((0xFFFFFFFF << 32) | rng.getrandbits(32), 16, rng)
    return [s.decode() for s in same], short.decode(), ones.decode()


@functools.lru_cache(maxsize=None)
def clustered_keys(count: int, low: int = 0x5A5A5A5A5A5):
    """`count` distinct u64 keys whose fq_gb_hash agree in their low CLUSTER_BITS bits"""
    return tuple(gb_unhash((i << CLUSTER_BITS) | low) for i in range(count))


# ---- pinned to the kernel source ----
def _cut_function(path, name):
    """the definition of device function `name` in `path`, from its return type to its closing brace"""
    with open(path) as f:
        src = f.read()
    m = re.search(r"^__device__ [^\n]*\b" + name + r"\(", src, re.M)
    assert m, f"{name} not found in {path}"
    depth = 0
    for j in range(src.index("{", m.end()), len(src)):
        depth += {"{": 1, "}": -1}.get(src[j], 0)
        if depth == 0:
            return src[m.start():j + 1]
    raise AssertionError(f"unbalanced braces after {name}")


@pytest.fixture(scope="module")
def kernel_hash(tmp_path_factory):
    """fq_utf8_hash and fq_gb_hash as the kernels define them, compiled for the host"""
    d = tmp_path_factory.mktemp("kernel_hash")
    src = "\n".join([
        "#include <cstdint>",
        "typedef uint32_t fq_u32;",
        "typedef uint64_t fq_u64;",
        "#define __device__",
        "#define __forceinline__ inline",
        _cut_function(os.path.join(KERNELS, "fq_utf8.cuh"), "fq_utf8_hash"),
        _cut_function(os.path.join(KERNELS, "fq_skeleton.cuh"), "fq_gb_hash"),
        'extern "C" fq_u64 utf8_hash(const unsigned char *p, fq_u32 n) { return fq_utf8_hash(p, n); }',
        'extern "C" fq_u64 gb_hash(fq_u64 k) { return fq_gb_hash(k); }',
    ])
    (d / "h.cc").write_text(src)
    lib_path = str(d / "libh.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", "-o", lib_path, str(d / "h.cc")], check=True, capture_output=True)
    lib = C.CDLL(lib_path)
    lib.utf8_hash.restype, lib.utf8_hash.argtypes = C.c_uint64, [C.c_char_p, C.c_uint32]
    lib.gb_hash.restype, lib.gb_hash.argtypes = C.c_uint64, [C.c_uint64]
    return {"utf8": lambda b: lib.utf8_hash(b, len(b)), "gb": lib.gb_hash}


def test_python_hashes_equal_the_kernel_source(kernel_hash):
    rng = np.random.default_rng(3)
    for n in list(range(41)) * 50 + rng.integers(41, 300, 200).tolist():
        b = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert utf8_hash(b) == kernel_hash["utf8"](b), b
    for k in rng.integers(0, 1 << 63, 3000, dtype=np.uint64).tolist() + [0, 1, GB_EMPTY, 1 << 63]:
        k = int(k) | (int(rng.integers(0, 2)) << 63)
        assert gb_hash(k) == kernel_hash["gb"](k), k
        assert gb_unhash(gb_hash(k)) == k


def test_constructed_strings_collide_under_the_kernel_hash(kernel_hash):
    same, short, ones = colliders()
    enc = [s.encode() for s in same]
    assert len(set(enc)) == 64 and all(len(b) == 16 and set(b) <= set(SAFE) for b in enc)
    h = {kernel_hash["utf8"](b) for b in enc + [short.encode()]}
    assert len(h) == 1 and len(short) == 12 and set(short.encode()) <= set(SAFE)
    assert kernel_hash["utf8"](ones.encode()) >> 32 == 0xFFFFFFFF and len(ones) == 16


@pytest.mark.parametrize("count", [3000, 6000])
def test_constructed_keys_cluster_under_the_kernel_hash(kernel_hash, count):
    keys = clustered_keys(count)
    assert len(set(keys)) == count and GB_EMPTY not in keys
    hs = [kernel_hash["gb"](k) for k in keys]
    low = (1 << CLUSTER_BITS) - 1
    assert len({x & low for x in hs}) == 1
    # one start and one step in the CTA's shared-memory table (fq_gb_put) for every table of up to 2^11 slots
    smask = (1 << 11) - 1
    assert len({((x >> 32) & smask, ((x >> 12) | 1) & smask) for x in hs}) == 1


# ---- GPU: fixtures and helpers ----
@pytest.fixture(scope="module")
def ctx():
    from fuse_query_b200 import cabi
    c = cabi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sql():
    from fuse_query_b200 import _fuse_host as h
    gpu = h.GpuContext.create(0)
    fctx = h.FuseQueryContext.create_ctx(4, gpu)

    def rows(q):
        out = []
        for b in h.execute_sql(fctx, q):
            out += list(zip(*[b.column(c).to_list() for c in range(b.num_columns())]))
        return out

    def register(name, columns):
        from fuse_query_b200.tables import register_table
        register_table(fctx, gpu, "default", name, columns)
    return {"h": h, "rows": rows, "register": register}


def scan_constants():
    """FQ_SORT_TILE, FQ_SCAN_TILE and FQ_SCAN_THREADS as kernels/fq_sort.cuh defines them"""
    with open(os.path.join(KERNELS, "fq_sort.cuh")) as f:
        defs = dict(re.findall(r"^#define (FQ_\w+) ([^/\n]+)", f.read(), re.M))

    def ev(name):
        return int(eval(re.sub(r"FQ_\w+", lambda m: str(ev(m.group(0))), defs[name]), {"__builtins__": {}}))
    return ev("FQ_SORT_TILE"), ev("FQ_SCAN_TILE"), ev("FQ_SCAN_THREADS")


def assert_scan_needs_rounds(counters):
    """an exclusive scan of `counters` words has more tile sums than fq_scan_sums' one CTA covers in one round"""
    _, tile, threads = scan_constants()
    assert -(-counters // tile) > threads, (counters, tile, threads)


def utf8_from_numpy(ctx, offsets, data, valid=None):
    from fuse_query_b200 import cabi
    n = len(offsets) - 1
    vcol = None
    if valid is not None:
        vcol = ctx.column(cabi.BOOL, n)
        v = np.ascontiguousarray(valid, dtype=np.uint8)
        ctx.check(cabi.lib().fq_column_upload(ctx._h, vcol._h, 0, C.c_void_p(v.ctypes.data), n, None))
    offsets = np.ascontiguousarray(offsets, dtype=np.int32)
    data = np.ascontiguousarray(data if len(data) else np.zeros(1, np.uint8), dtype=np.uint8)
    h = C.c_void_p()
    ctx.check(cabi.lib().fq_utf8_create(ctx._h, C.c_void_p(offsets.ctypes.data), C.c_void_p(data.ctypes.data), n,
                                        vcol._h if vcol is not None else None, None, C.byref(h)))
    ctx.synchronize()
    return cabi.Utf8Array(ctx, h, vcol)


def utf8_to_numpy(ctx, arr):
    """(offsets int32[n + 1], bytes uint8) of a device Utf8 array"""
    from fuse_query_b200 import cabi
    off = np.zeros(len(arr) + 1, dtype=np.int32)
    data = np.zeros(max(1, arr.nbytes()), dtype=np.uint8)
    ctx.check(cabi.lib().fq_utf8_download(ctx._h, arr._h, C.c_void_p(off.ctypes.data), C.c_void_p(data.ctypes.data), None))
    ctx.synchronize()
    return off, data[:off[-1]]


HEX = np.frombuffer(b"0123456789abcdef", dtype=np.uint8)


def hex_bytes(v, width):
    """zero-padded lower-case hex of every value, `width` digits each, as one flat uint8 array"""
    shifts = 4 * np.arange(width - 1, -1, -1, dtype=np.uint64)
    return HEX[((v.astype(np.uint64)[:, None] >> shifts) & np.uint64(15)).astype(np.intp)].ravel()


# ---- B. dictionary encoder under full hash collisions ----
def collider_values(rng, ordinary):
    same, short, ones = colliders()
    vals = (same + [short, ones]) * 3 + [None] * 40 + ordinary
    rng.shuffle(vals)
    return vals


def check_encoding(ctx, values):
    """codes = bytewise ranks, dictionary = the sorted distinct strings, decoding gives the column back"""
    arr = ctx.utf8(values)
    codes, dictionary = arr.dict_encode()
    want = sorted({v.encode() for v in values if v is not None})
    assert dictionary.to_list() == want
    rank = {b: i for i, b in enumerate(want)}
    valid = np.array([v is not None for v in values])
    exp = np.array([rank[v.encode()] if v is not None else 0 for v in values], dtype=np.uint32)
    assert np.array_equal(codes.to_numpy(len(values))[valid], exp[valid])
    assert dictionary.take(codes, len(values), arr._valid).to_list() == [None if v is None else v.encode() for v in values]


@pytest.mark.gpu
def test_encoder_separates_strings_with_one_hash(ctx):
    rng = random.Random(1)
    check_encoding(ctx, collider_values(rng, [f"o{i}" for i in range(200)] + ["", "a" * 16]))


@pytest.mark.gpu
def test_encoder_separates_strings_with_one_hash_among_a_million(ctx):
    rng = random.Random(2)
    ordinary = [f"{v:x}" for v in np.random.default_rng(2).integers(0, 1 << 62, 1_000_000).tolist()]
    check_encoding(ctx, collider_values(rng, ordinary))


@pytest.mark.gpu
def test_sql_over_strings_with_one_hash(sql):
    same, short, ones = colliders()
    vals = collider_values(random.Random(3), [f"o{i % 50}" for i in range(5000)])
    n = len(vals)
    sql["register"]("collide", {"s": np.array(vals, dtype=object), "x": np.arange(n, dtype=np.int64)})
    got = sql["rows"]("select s, count(x) from collide group by s")
    assert sorted(got, key=repr) == sorted(collections.Counter(vals).items(), key=repr)
    want = collections.Counter(vals)
    for lit in [same[0], same[63], short, ones]:
        assert sql["rows"](f"select count(x) from collide where s = '{lit}'") == [(want[lit],)], lit


# ---- C. GROUP BY on clustered keys ----
GB_LEAVES = ["(sum (col v))", "(count (col v))", "(min (col v))", "(max (col v))"]


def clustered_table(count, rows=200_000, seed=0):
    rng = np.random.default_rng(seed)
    keys = np.array(clustered_keys(count) + (GB_EMPTY,), dtype=np.uint64)
    k = rng.permutation(np.concatenate([keys, keys[rng.integers(0, len(keys), rows - len(keys))]]))
    v = rng.integers(-10**6, 10**6, rows).astype(np.int64)
    return k, v


def expected_groups(k, v):
    """sorted rows (key, sum, count, min, max), exact"""
    uniq, inv = np.unique(k, return_inverse=True)
    sums = np.zeros(len(uniq), np.int64)
    np.add.at(sums, inv, v)
    mins = np.full(len(uniq), np.iinfo(np.int64).max)
    np.minimum.at(mins, inv, v)
    maxs = np.full(len(uniq), np.iinfo(np.int64).min)
    np.maximum.at(maxs, inv, v)
    return list(zip(uniq.tolist(), sums.tolist(), np.bincount(inv).tolist(), mins.tolist(), maxs.tolist()))


def exported_groups(pipe, n_groups):
    keys, _, leaves, _ = pipe.export_groups(n_groups)
    cols = [c.to_numpy(n_groups).tolist() for c in keys + leaves]
    for c in keys + leaves:
        c.free()
    return sorted(zip(*cols))


@pytest.mark.gpu
@pytest.mark.parametrize("count", [3000, 6000])
def test_group_by_clustered_keys(ctx, count):
    """At most three growths of the table (the way run_groupby grows it): a cluster that overflows every table size fails
    here in seconds instead of reserving ever larger tables."""
    from fuse_query_b200 import cabi
    k, v = clustered_table(count)
    cols = [ctx.from_numpy(k), ctx.from_numpy(v)]
    pipe = ctx.pipe(GB_LEAVES, keys=["(col k)"], columns=["k", "v"], dtypes=[cabi.U64, cabi.I64])
    src = cabi.make_source(cols, len(k))
    hint, groups = 1 << 16, None
    for _ in range(4):
        pipe.groupby_reserve(hint)
        pipe.launch_groupby(src)
        try:
            groups = pipe.fetch_groupby()
            break
        except cabi.FuseGpuError as e:
            if e.status != cabi.ERR_CAPACITY:
                raise
            hint *= 8
    assert groups is not None, f"{count + 1} groups overflowed tables for up to {hint // 8} groups"
    assert exported_groups(pipe, groups) == expected_groups(k, v)
    pipe.destroy()
    # a new pipe's run_groupby with room for every row from the start: its first table (seed 0) keeps the cluster, and
    # its second, of the same size, is hashed with another seed
    pipe = ctx.pipe(GB_LEAVES, keys=["(col k)"], columns=["k", "v"], dtypes=[cabi.U64, cabi.I64])
    assert pipe.run_groupby(src, groups_hint=len(k)) == count + 1
    assert exported_groups(pipe, count + 1) == expected_groups(k, v)
    pipe.destroy()


@pytest.mark.gpu
def test_sql_group_by_clustered_keys(sql):
    k, v = clustered_table(6000, seed=1)
    sql["register"]("clustered", {"k": k, "v": v})
    got = sql["rows"]("select k, sum(v), count(v), min(v), max(v) from clustered group by k")
    assert sorted(got) == expected_groups(k, v)


# ---- D. the shared scan past one round ----
@pytest.mark.gpu
@pytest.mark.parametrize("descending", [False, True])
def test_order_by_past_one_scan_round(ctx, descending):
    sort_tile, _, _ = scan_constants()
    n = (1 << 27) + (1 << 20) + 3
    assert_scan_needs_rounds(256 * -(-n // sort_tile))
    key = ctx.from_numpy(np.resize(np.arange(1000, dtype=np.uint32), n))
    got = ctx.sort_indices([key], n, descending=[descending]).to_numpy(n)
    key.free()
    pos = 0
    for r in (range(999, -1, -1) if descending else range(1000)):
        want = np.arange(r, n, 1000, dtype=np.uint32)       # stable: rows of one key stay in row order
        assert np.array_equal(got[pos:pos + len(want)], want), (r, pos)
        pos += len(want)
    assert pos == n


def hex_column(n, distinct, width, null_share, seed):
    """every value of [0, distinct) at least once in a valid row, then random duplicates of which some are NULL"""
    rng = np.random.default_rng(seed)
    v = np.concatenate([np.arange(distinct), rng.integers(0, distinct, n - distinct)]).astype(np.int64)
    valid = np.concatenate([np.ones(distinct, bool), rng.random(n - distinct) >= null_share])
    p = rng.permutation(n)
    v, valid = v[p], valid[p]
    return v, valid, np.arange(0, width * n + 1, width, dtype=np.int32), hex_bytes(v, width)


@pytest.mark.gpu
def test_dictionary_encoding_past_one_scan_round(ctx):
    n, distinct, width = (1 << 22) + 300_001, 3_000_000, 6
    cap = 1024
    while cap < 2 * n:
        cap *= 2                                              # the encoder's table: the next power of two >= 2n slots
    assert_scan_needs_rounds(cap)
    v, valid, off, data = hex_column(n, distinct, width, 0.1, seed=5)
    arr = utf8_from_numpy(ctx, off, data, valid)
    codes, dictionary = arr.dict_encode()
    got = codes.to_numpy(n)
    assert np.array_equal(got[valid], v[valid])               # fixed-width hex order is numeric order
    d_off, d_data = utf8_to_numpy(ctx, dictionary)
    assert np.array_equal(d_off, np.arange(0, width * distinct + 1, width)) and np.array_equal(d_data, hex_bytes(np.arange(distinct), width))
    back_off, back_data = utf8_to_numpy(ctx, dictionary.take(codes, n, arr._valid))
    assert np.array_equal(back_off[1:], np.cumsum(width * valid)) and np.array_equal(back_data, hex_bytes(v[valid], width))


@pytest.mark.gpu
def test_utf8_take_past_one_scan_round(ctx):
    from fuse_query_b200 import cabi
    n = (1 << 23) + 4097
    assert_scan_needs_rounds(n + 1)                           # one length per output row + the total
    rng = np.random.default_rng(6)
    lens = rng.integers(0, 17, 100_000).astype(np.int64)
    src_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    src_data = rng.integers(0x20, 0x7F, int(src_off[-1])).astype(np.uint8)
    src = utf8_from_numpy(ctx, src_off, src_data)
    rows = rng.integers(0, len(lens), n).astype(np.uint32)
    ok = rng.random(n) >= 0.1
    rows_col = ctx.from_numpy(rows)
    ok_col = ctx.column(cabi.BOOL, n)
    ok8 = ok.astype(np.uint8)
    ctx.check(cabi.lib().fq_column_upload(ctx._h, ok_col._h, 0, C.c_void_p(ok8.ctypes.data), n, None))
    off, data = utf8_to_numpy(ctx, src.take(rows_col, n, ok_col))
    out_len = lens[rows] * ok
    want_off = np.concatenate([[0], np.cumsum(out_len)])
    assert np.array_equal(off, want_off)
    want = src_data[np.repeat(src_off[rows].astype(np.int64) - want_off[:-1], out_len) + np.arange(want_off[-1])]
    assert np.array_equal(data, want)


@pytest.mark.gpu
def test_sql_order_by_limit_over_a_large_string_column(sql):
    import pyarrow as pa
    n, distinct, width = (1 << 22) + 300_001, 2_000_000, 6
    v, _, off, data = hex_column(n, distinct, width, 0.0, seed=7)
    s = pa.StringArray.from_buffers(n, pa.py_buffer(off), pa.py_buffer(data))
    sql["register"]("big", {"s": s, "x": np.arange(n, dtype=np.int64)})
    srt = np.sort(v)
    assert sql["rows"]("select s from big order by s limit 10") == [(f"{x:06x}",) for x in srt[:10]]
    assert sql["rows"]("select s from big order by s desc limit 10") == [(f"{x:06x}",) for x in srt[::-1][:10]]
    counts = np.bincount(v)
    assert sql["rows"]("select s, count(x) from big group by s order by s limit 5") == [(f"{x:06x}", int(counts[x])) for x in range(5)]


# ---- E. the encoder's degenerate sizes ----
@pytest.mark.gpu
def test_all_null_string_column(sql):
    import pyarrow as pa
    n = 1000
    sql["register"]("allnull", {"s": pa.array([None] * n, type=pa.string()), "x": np.arange(n, dtype=np.int64)})
    q = sql["rows"]
    assert q("select count(x) from allnull where s = 'a'") == [(0,)]
    assert q("select count(x) from allnull where s < 'a'") == [(0,)]
    assert q("select count(x) from allnull where s >= ''") == [(0,)]
    assert q("select count(s), min(s), max(s) from allnull") == [(n, None, None)]
    assert q("select s, count(x) from allnull group by s") == [(None, n)]
    assert q("select s, x from allnull order by s") == [(None, i) for i in range(n)]


@pytest.mark.gpu
def test_all_empty_string_column(sql):
    n = 1000
    sql["register"]("allempty", {"s": np.array([""] * n, dtype=object), "x": np.arange(n, dtype=np.int64)})
    q = sql["rows"]
    assert q("select count(x) from allempty where s = ''") == [(n,)]
    assert q("select count(x) from allempty where s < 'a'") == [(n,)]
    assert q("select count(x) from allempty where s > ''") == [(0,)]
    assert q("select count(s), min(s), max(s) from allempty") == [(n, "", "")]
    assert q("select s, count(x) from allempty group by s") == [("", n)]
    assert q("select s, x from allempty order by s desc limit 3") == [("", 0), ("", 1), ("", 2)]
