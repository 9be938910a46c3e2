"""Utf8 columns on the device: dictionary-encoding throughput, string queries against the same queries over a plain UInt32
column holding the codes, LIKE queries against `s = '...'` on the same column, fq_utf8_like over dictionaries, and pyarrow
on the host CPU as a baseline.  Writes <out>/r03_utf8_<rows>.json (or r04_like_<rows>.json for --sections like) with the
GPU's name and power limit.

    python tools/bench_utf8.py [--rows 100000000] [--out profiles] [--sections encode,queries,like]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from fuse_query_b200 import cabi  # noqa: E402
from fuse_query_b200 import _fuse_host as h  # noqa: E402

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def strings(values, width, prefix=b""):
    """fixed-width strings: `prefix` + the decimal digits of `values`, zero-padded to `width` bytes in all"""
    digits = width - len(prefix)
    mat = np.empty((len(values), width), dtype=np.uint8)
    mat[:, :len(prefix)] = np.frombuffer(prefix, dtype=np.uint8)
    v = values.astype(np.int64)
    for j in range(digits):
        mat[:, width - 1 - j] = 48 + v % 10
        v //= 10
    offsets = np.arange(len(values) + 1, dtype=np.int64) * width
    assert offsets[-1] < 2**31
    return offsets.astype(np.int32), mat.reshape(-1)


def device_utf8(ctx, offsets, data):
    hdl = C.c_void_p()
    ctx.check(cabi.lib().fq_utf8_create(ctx._h, C.c_void_p(offsets.ctypes.data), C.c_void_p(data.ctypes.data), len(offsets) - 1, None, None,
                                        C.byref(hdl)))
    return cabi.Utf8Array(ctx, hdl, None)


def median_time(fn, reps):
    fn()   # warm-up: module loads, scratch growth, JIT of new pipes
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()   # every measured call ends with a device synchronise (results come back to the host)
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), [round(t, 6) for t in ts]


def encode_case(ctx, rows, distinct, width, prefix, rng, reps):
    values = rng.permutation(rows) if distinct >= rows else rng.integers(0, distinct, rows)
    offsets, data = strings(values, width, prefix)
    arr = device_utf8(ctx, offsets, data)
    cap = 1024
    while cap < 2 * rows:
        cap *= 2

    def run():
        codes, d = arr.dict_encode()
        run.d = len(d)
        d.free()
        codes.free()
    sec, all_t = median_time(run, reps)
    stream_bytes = rows * (4 + width + 4)   # offsets + string bytes read, codes written
    table_bytes = cap * 8 * 3 + cap * 4 * 3 + rows * 8   # clear, flag and compact passes over the table, the scan, one probe per row
    arr.free()
    return {"rows": rows, "distinct": run.d, "width": width, "shared_prefix": len(prefix), "seconds": sec, "all_seconds": all_t,
            "rows_per_s": rows / sec, "stream_bytes": stream_bytes, "stream_GBps": stream_bytes / sec / 1e9,
            "stream_share_of_hbm_bound": stream_bytes / HBM_BYTES_PER_S / sec, "hash_table_bytes": table_bytes}


def query_cases(rows, distinct, rng, reps):
    """the same four queries over the Utf8 column s and over k, a plain nullable-free UInt32 column holding s's codes"""
    import pyarrow as pa
    import pyarrow.compute as pc
    values = rng.integers(0, distinct, rows)
    offsets, data = strings(values, 16)
    x = rng.integers(0, 1000, rows).astype(np.uint64)
    gpu = h.GpuContext.create(0)
    fctx = h.FuseQueryContext.create_ctx(8, gpu)
    s = h.DataArray.from_utf8(gpu, offsets, data.tobytes(), None)
    dictionary = s.dictionary()
    ranks = np.searchsorted(np.array([d.encode() for d in dictionary], dtype="S16"), np.array([f"{v:016d}".encode() for v in range(distinct)], dtype="S16"))
    k = h.DataArray.from_numpy(gpu, ranks[values].astype(np.uint32))
    xs = h.DataArray.from_numpy(gpu, x)
    schema = h.DataSchema([h.DataField("s", h.DataType.Utf8, False), h.DataField("k", h.DataType.UInt32, False), h.DataField("x", h.DataType.UInt64, False)])
    ds = fctx.datasource()
    ds.add_database("b")
    ds.add_table("b", h.MemoryTable("b", "t", schema, [s, k, xs]))
    lit = dictionary[len(dictionary) // 2]
    lit_code = len(dictionary) // 2
    queries = {
        "eq": (f"select count(x) from b.t where s = '{lit}'", f"select count(x) from b.t where k = {lit_code}"),
        "lt": (f"select count(x) from b.t where s < '{lit}'", f"select count(x) from b.t where k < {lit_code}"),
        "group_by": ("select s, count(x) from b.t group by s", "select k, count(x) from b.t group by k"),
        "order_by_limit": ("select s from b.t order by s limit 10", "select k from b.t order by k limit 10"),
    }
    out = {}
    for name, (qs, qk) in queries.items():
        ts, tk = [], []
        for _ in range(2):   # warm-up both
            h.execute_sql(fctx, qs), h.execute_sql(fctx, qk)
        for _ in range(reps):   # alternate the two so that drift on a shared host hits both alike
            t0 = time.perf_counter(); h.execute_sql(fctx, qs); ts.append(time.perf_counter() - t0)
            t0 = time.perf_counter(); h.execute_sql(fctx, qk); tk.append(time.perf_counter() - t0)
        out[name] = {"utf8_sql": qs, "uint32_sql": qk, "utf8_seconds": float(np.median(ts)), "uint32_seconds": float(np.median(tk)),
                     "utf8_all": [round(t, 6) for t in ts], "uint32_all": [round(t, 6) for t in tk]}
    # pyarrow on the host CPU, same data
    arr = pa.Array.from_buffers(pa.string(), rows, [None, pa.py_buffer(offsets), pa.py_buffer(data)])
    tbl = pa.table({"s": arr, "x": x})
    base = {}
    for name, fn in {"dictionary_encode": lambda: arr.dictionary_encode(),
                     "filter_eq_count": lambda: pc.sum(pc.equal(arr, lit)).as_py(),
                     "filter_lt_count": lambda: pc.sum(pc.less(arr, lit)).as_py(),
                     "group_by_count": lambda: tbl.group_by("s").aggregate([("x", "count")]),
                     "sort_indices": lambda: pc.sort_indices(arr)}.items():
        t0 = time.perf_counter(); fn(); base[name] = time.perf_counter() - t0
    return {"rows": rows, "distinct": distinct, "queries": out, "pyarrow_host_seconds": base}


def alternate(fctx, qa, qb, reps):
    """median seconds of two queries, run in turn so that drift on a shared host hits both alike"""
    ta, tb = [], []
    for _ in range(2):   # warm-up both (module loads, the pattern's bit table)
        h.execute_sql(fctx, qa), h.execute_sql(fctx, qb)
    for _ in range(reps):
        t0 = time.perf_counter(); h.execute_sql(fctx, qa); ta.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); h.execute_sql(fctx, qb); tb.append(time.perf_counter() - t0)
    return float(np.median(ta)), float(np.median(tb)), [round(t, 6) for t in ta], [round(t, 6) for t in tb]


def like_cases(rows, distinct, rng, reps):
    """LIKE and NOT LIKE over the Utf8 column s of the query table, each beside `s = '...'` over the same column; the matching
    kernel alone over sorted dictionaries of 10^4, 10^6 and 10^8 distinct 16-byte strings; pyarrow match_like on the host"""
    import pyarrow as pa
    import pyarrow.compute as pc
    values = rng.integers(0, distinct, rows)
    offsets, data = strings(values, 16)
    x = rng.integers(0, 1000, rows).astype(np.uint64)
    gpu = h.GpuContext.create(0)
    fctx = h.FuseQueryContext.create_ctx(8, gpu)
    s = h.DataArray.from_utf8(gpu, offsets, data.tobytes(), None)
    schema = h.DataSchema([h.DataField("s", h.DataType.Utf8, False), h.DataField("x", h.DataType.UInt64, False)])
    ds = fctx.datasource()
    ds.add_database("b")
    ds.add_table("b", h.MemoryTable("b", "t", schema, [s, h.DataArray.from_numpy(gpu, x)]))
    lit = f"{distinct // 2:016d}"
    eq = f"select count(x) from b.t where s = '{lit}'"
    queries = {"prefix": "select count(x) from b.t where s like '00000000000042%'",
               "infix": "select count(x) from b.t where s like '%42%'",
               "not_like": "select count(x) from b.t where s not like '%42%'"}
    out = {}
    for name, q in queries.items():
        tl, te, al, ae = alternate(fctx, q, eq, reps)
        out[name] = {"like_sql": q, "eq_sql": eq, "like_seconds": tl, "eq_seconds": te, "like_over_eq": tl / te, "like_all": al, "eq_all": ae,
                     "rows": rows, "result": h.execute_sql(fctx, q)[0].column(0).to_list()[0]}
    arr = pa.Array.from_buffers(pa.string(), rows, [None, pa.py_buffer(offsets), pa.py_buffer(data)])
    base = {}
    for name, pat in (("prefix", "00000000000042%"), ("infix", "%42%")):
        t0 = time.perf_counter(); pc.sum(pc.match_like(arr, pat)).as_py(); base[name] = time.perf_counter() - t0
    kernel = []
    ctx = cabi.Context(0)
    for d in (10**4, 10**6, 10**8):
        offs, dat = strings(np.arange(d), 16)   # zero-padded decimals: already in bytewise order, a dictionary as fq_utf8_dict_encode leaves it
        dictionary = device_utf8(ctx, offs, dat)
        for pat in ("%42%", "00000000000042%"):
            sec, all_t = median_time(lambda: dictionary.like(pat).free(), reps)
            kernel.append({"distinct": d, "pattern": pat, "seconds": sec, "all_seconds": all_t, "strings_per_s": d / sec,
                           "bytes_read": d * (16 + 4), "GBps": d * 20 / sec / 1e9})
            print(json.dumps(kernel[-1]), flush=True)
        dictionary.free()
    ctx.close()
    return {"rows": rows, "distinct": distinct, "queries": out, "fq_utf8_like": kernel, "pyarrow_match_like_host_seconds": base}


def device_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--prefix-rows", type=int, default=20_000_000, help="rows of the 100-byte case (int32 offsets: at most 2 GiB of bytes)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="profiles")
    ap.add_argument("--sections", default="encode,queries", help="comma-separated: encode, queries, like")
    a = ap.parse_args()
    sections = a.sections.split(",")
    rng = np.random.default_rng(2026)
    res = {"device": device_info(), "encode": [], "note": "seconds are host wall time around calls that end with a device synchronise"}
    if "like" in sections:
        res["like"] = like_cases(a.rows, 10**4, rng, max(a.reps, 5))
        print(json.dumps(res["like"]["queries"]), flush=True)
    if sections == ["like"]:
        os.makedirs(a.out, exist_ok=True)
        path = os.path.join(a.out, f"r04_like_{a.rows}.json")
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print("wrote", path)
        return
    ctx = cabi.Context(0)
    for distinct in (10, 10**4, 10**6, a.rows):
        res["encode"].append(encode_case(ctx, a.rows, distinct, 16, b"", rng, a.reps))
        print(json.dumps(res["encode"][-1]), flush=True)
    res["encode"].append(encode_case(ctx, a.prefix_rows, 10**6, 100, b"p" * 84, rng, a.reps))
    print(json.dumps(res["encode"][-1]), flush=True)
    ctx.close()
    res["queries"] = query_cases(a.rows, 10**4, rng, max(a.reps, 5))
    print(json.dumps(res["queries"]), flush=True)
    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, f"r03_utf8_{a.rows}.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
