"""GROUP BY with a 128-bit or 65-bit table key against the same grouping with a 64-bit key, on one GPU.

Three shapes over the same materialised numbers column, with sum / count / min / max, for each k:
  narrow    group by number % k                        64-bit key
  wide      group by number % k, number % k * 3        128-bit key, the same k groups
  nullable  group by x, x = number % k as a column with an all-valid Arrow validity bitmap: 65-bit key
Every shape is warmed up, then the shapes are timed alternating, each run a launch plus the fetch that synchronises
(host clock).  The median of --reps runs is reported, and every result is checked against closed forms.  Writes
<out>/<name>_<rows>.json with the GPU's name and power limit.  FQ_GB_SMEM_SLOTS fixes the shared-memory table's size
for every shape (the run that separates the key width from the table size).

    python tools/bench_groupby_wide.py [--rows 1000000000] [--ks 7,1000,1500,5000,1000000] [--reps 7] [--out profiles]
                                       [--name r05_groupby_wide]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from fuse_query_b200 import cabi  # noqa: E402

NUM = "(col number)"


def mod(k, col=NUM):
    return f"(- {col} (* (/ {col} (u64 {k})) (u64 {k})))"


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


def closed_form(n, k, of_number):
    """per group r = 0..k-1, sorted: (count, sum, min, max) of number (of_number) or of x = number % k"""
    r = np.arange(min(k, n), dtype=np.uint64)
    c = np.uint64(n // k) + (r < np.uint64(n % k)).astype(np.uint64)
    if of_number:
        s = c * r + np.uint64(k) * (c * (c - np.uint64(1)) // np.uint64(2))
        return c, s, r, r + np.uint64(k) * (c - np.uint64(1))
    return c, c * r, r, r


def check(pipe, n, k, n_keys, of_number):
    groups = pipe.fetch_groupby()
    assert groups == min(k, n), (groups, k)
    keys, _, leaves, _ = pipe.export_groups(groups)
    kv = [c.to_numpy(groups) for c in keys]
    order = np.argsort(kv[0], kind="stable")
    assert np.array_equal(kv[0][order], np.arange(groups, dtype=np.uint64))
    if n_keys == 2:
        assert np.array_equal(kv[1][order], kv[0][order] * np.uint64(3))
    got = [c.to_numpy(groups)[order] for c in leaves]     # sum, count, min, max
    c, s, lo, hi = closed_form(n, k, of_number)
    for g, w, name in zip(got, (s, c, lo, hi), ("sum", "count", "min", "max")):
        assert np.array_equal(g.astype(np.uint64), w), (k, n_keys, name)
    for col in keys + leaves:
        col.free()


def smem_slots():
    """slots of the CTA's shared-memory table per shape, as plan_kernels sizes it: the largest power of two of entries of
    8 * (key words + G) bytes within 96 KB, or FQ_GB_SMEM_SLOTS; G = rows + 4 leaves (+ 3 valid-row counts when the
    aggregated column is nullable)"""
    env = os.environ.get("FQ_GB_SMEM_SLOTS")
    out = {}
    for name, words, g in (("narrow", 1, 5), ("wide", 2, 5), ("nullable", 1, 8)):
        cap = 1
        while cap * 2 * 8 * (words + g) <= 96 * 1024:
            cap *= 2
        if env is not None:
            cap = 1
            while cap * 2 <= int(env):
                cap *= 2
        out[name] = cap
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000_000)
    ap.add_argument("--ks", default="7,1000,1500,5000,1000000")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default="profiles")
    ap.add_argument("--name", default="r05_groupby_wide", help="output file: <out>/<name>_<rows>.json")
    a = ap.parse_args()
    n = a.rows
    ctx = cabi.Context(0)
    number = ctx.numbers(0, n)
    src = cabi.make_source([number], n)
    bits = ctx.from_numpy(np.full((n + 7) // 8, 0xFF, dtype=np.uint8))
    results = []
    for k in [int(x) for x in a.ks.split(",")]:
        aggs = lambda c: [f"(sum {c})", f"(count {c})", f"(min {c})", f"(max {c})"]
        # x = number % k on the device, then an all-valid validity bitmap attached: a nullable UInt64 column
        x = ctx.column(cabi.U64, n)
        proj = ctx.pipe([mod(k)])
        proj.launch_project(src, [x], n)
        proj.fetch_project()
        proj.destroy()
        ctx.check(cabi.lib().fq_column_set_validity_bitmap(ctx._h, x._h, bits._h, 0))
        shapes = {
            "narrow": (ctx.pipe(aggs(NUM), keys=[mod(k)]), src, 1, True),
            "wide": (ctx.pipe(aggs(NUM), keys=[mod(k), f"(* {mod(k)} (u64 3))"]), src, 2, True),
            "nullable": (ctx.pipe(aggs("(col x)"), keys=["(col x)"], columns=["x"], dtypes=[cabi.U64], nullable=[2]),
                         cabi.make_source([x], n), 1, False),
        }
        times = {name: [] for name in shapes}
        for name, (pipe, s, _, _) in shapes.items():
            pipe.run_groupby(s, groups_hint=min(k, n))          # reserve once, warm up (module load, first launch)
        for _ in range(a.reps):
            for name, (pipe, s, _, _) in shapes.items():
                t0 = time.perf_counter()
                pipe.launch_groupby(s)
                pipe.fetch_groupby()                             # synchronises
                times[name].append(time.perf_counter() - t0)
        for name, (pipe, s, nk, of_number) in shapes.items():
            check(pipe, n, k, nk, of_number)
        entry = {"k": k, "rows": n, "smem_slots": smem_slots(),
                 "median_s": {name: float(np.median(t)) for name, t in times.items()},
                 "runs_s": {name: [round(v, 6) for v in t] for name, t in times.items()}}
        entry["ratio_wide_over_narrow"] = entry["median_s"]["wide"] / entry["median_s"]["narrow"]
        entry["ratio_nullable_over_narrow"] = entry["median_s"]["nullable"] / entry["median_s"]["narrow"]
        print(json.dumps(entry), flush=True)
        results.append(entry)
        for pipe, _, _, _ in shapes.values():
            pipe.destroy()
        x.free()
    res = {"device": device_info(), "results": results,
           "note": "seconds are host wall time around a GROUP BY launch and the fetch that synchronises; sum / count / min / max; "
                   "every result checked against closed forms"}
    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, f"{a.name}_{n}.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)
    ctx.close()


if __name__ == "__main__":
    main()
