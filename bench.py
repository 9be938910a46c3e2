#!/usr/bin/env python3
"""bench.py — throughput of the fuse-query hot path on B200 (and of the CPU reference arm).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--rows R] [--mode materialised|generated]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[3], the README headline query):
    SELECT sum(number)/count(number), max(number), min(number) FROM system.numbers_mt(10_000_000_000)
One "step" = one COMPLETE query over the 10^10-row UInt64 column (materialised in HBM, 80 GB at N=1): every rank runs the
fused Source -> AggregatePartial kernel over its shard and the kernel itself finishes with the merge point
(processors/processor_merge.rs:37-66 -> transforms/transform_aggregate_final.rs:50-78): its last CTA stores the 80-byte
running state into every rank's exchange window over NVLink peer memory, waits for the states of all ranks of this step
and folds them, so that when the step's kernel has ended EVERY rank holds the merged answer (copied to pinned host
memory behind the kernel).  `--merge nccl` (or an IPC failure) does the same exchange with an NCCL all-gather + fold
after each launch.  Strong scaling: the 10^10 rows are partitioned across ranks exactly like the reference chunks its 8
partitions over workers (processors/pipeline_builder.rs:73-95).

Prints ONE JSON line (see the contract in the task statement): `value` = whole-job rows/s with inputs resident in HBM,
merge included; `throughput_no_merge` = back-to-back kernels without the cross-rank wait (round 1's figure); `e2e` = the
same query through the C ABI with HOST (pinned) column buffers, H2D copies and the D2H state read inside the timed
region, with `e2e.roofline` = the plain cudaMemcpyAsync rate of the same copies on all ranks at once; `roofline` for the
aggregate kernel; `per_query` = every README query x {materialised, generated} as whole-job numbers at this N with the
merged result verified against the closed form; `cpu_baseline` = the CPU oracle's reference-shaped pipeline timed on this
box's host cores (rank 0, N=1 only).

--impl reference times the reference's CPU algorithm (oracle port; the reference itself is Rust and cannot be built in
this image) with the 8-way parallelism the reference uses.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from as it found it (it may be read-only)

TOTAL_ROWS = 10_000_000_000
NUM = "(col number)"
HEADLINE = [f"(/ (sum {NUM}) (count {NUM}))", f"(max {NUM})", f"(min {NUM})"]
HEADLINE_SQL = "SELECT sum(number)/count(number), max(number), min(number) FROM system.numbers_mt(10000000000)"
README_PUBLISHED_SECONDS = 6.40  # README.md:62 (8 vCPU KVM), BASELINE.md §1
M64 = (1 << 64) - 1


def _sum(n, b=0):     # wrapping sum of b .. b+n-1
    return ((2 * b + n - 1) * n // 2) & M64


# name -> (select expressions, expected Aggregator-leaf states in node order as functions of the row count, README seconds, note)
README_QUERIES = {
    "sum(number)": ([f"(sum {NUM})"], lambda n: [_sum(n)], 1.77, None),
    "max(number)": ([f"(max {NUM})"], lambda n: [n - 1], 2.83, None),
    "max(number+1)": ([f"(max (+ {NUM} (u64 1)))"], lambda n: [n], 6.13, None),
    "count(number)": ([f"(count {NUM})"], lambda n: [n], 1.55,
                      "metadata-only: Count of a bare column reads no data (the row count is known); no bytes, no GB/s"),
    "count(number) [honest 8N scan]": ([f"(count (+ {NUM} (u64 0)))"], lambda n: [n], 1.55,
                                       "Count(number + 0): the argument is evaluated for every row like the reference does "
                                       "(function_aggregator.rs:58-59), so the column is streamed once"),
    "sum(number)/count(number)": ([f"(/ (sum {NUM}) (count {NUM}))"], lambda n: [_sum(n), n], 2.04, None),
    "sum(number)/count(number),max(number),min(number)": (HEADLINE, lambda n: [_sum(n), n, n - 1, 0], 6.40, None),
}
CFG1 = [f"(max (+ {NUM} (u64 1)))", f"(min {NUM})", f"(count {NUM})"]
CFG2_PRED = f"(< (+ (+ (+ {NUM} (u64 1)) (/ {NUM} (u64 2))) (u64 1)) (u64 100))"
CFG2_PROJ = [f"(alias c1 (+ {NUM} (u64 1)))", f"(alias c2 (/ {NUM} (u64 2)))"]


def agg_kernel_name(generated: bool) -> str:
    v = os.environ.get("FQ_AGG_VARIANT", "tma")
    if generated or v != "tma":
        return "fq_agg_kernel (fqk_*_agg_%s): LDG.128 streaming" % ("u8" if v == "u8" else "u4")
    return "fq_agg_tma_kernel (fqk_*_agg_tma): cp.async.bulk staged, 4 x 32 KB ring per SM"


def ncu_traffic(rows_per_launch: int, generated: bool):
    """dram__bytes_read.sum + dram__bytes_write.sum of the aggregate kernel from the committed ncu --set full capture of THIS
    workload (profiles/*traffic_headline_1e10.json, newest round first); None when the launch differs from the captured one."""
    if generated:
        return None
    for name in ("r02_traffic_headline_1e10.json", "r01_traffic_headline_1e10.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            with open(path) as f:
                t = json.load(f)
            if t["rows"] == rows_per_launch:
                return t["traffic"]
    return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.lines:
            if not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def shard_of(rank: int, world: int, total: int):
    """Consecutive reference partitions per rank (numbers_table.rs:29-55 + pipeline_builder.rs:73-95)."""
    from fuse_query_b200.shards import shard_for_rank
    return shard_for_rank(rank, world, total)


def expected(total: int):
    return {"sum": _sum(total), "count": total, "avg": _sum(total) // total, "max": total - 1, "min": 0}


def dump_outputs(out_dir: str, arrays: dict):
    """--dump-outputs: each array as <out_dir>/<name>.npy in float64, so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def u64_hi_lo(values):
    """u64 values as exact (high 32 bits, low 32 bits) pairs: a wrapped u64 sum does not fit float64's 53-bit mantissa."""
    return [[v >> 32, v & 0xFFFFFFFF] for v in values]


def common_config(total: int):
    """The part of `config` both arms print identically (the driver compares them)."""
    sql = HEADLINE_SQL if total == TOTAL_ROWS else HEADLINE_SQL.replace("10000000000", str(total))
    return {"workload": sql, "rows_total": total}


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle's reference-shaped pipeline on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_reference_run(rows: int):
    from oracle import binding as o
    r = o.run_query(HEADLINE, total=rows, is_aggregate=True, worker_threads=8, use_threads=True)
    return r.seconds, r.rows()[0]


def cpu_sample_rows(target_s: float = 8.0) -> int:
    secs, _ = cpu_reference_run(400_000_000)
    rate = 400_000_000 / secs
    rows = int(min(TOTAL_ROWS, max(400_000_000, rate * target_s)))
    return (rows // 80_000) * 80_000  # 8 partitions of whole 10 000-row blocks (SURVEY F7 stays out of the way)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = min(8, os.cpu_count() or 1)
    # bounded sample: the whole --steps/--warmup run stays within ~2.5 minutes whatever K the driver passes
    rows = args.rows or cpu_sample_rows(max(0.5, min(8.0, 150.0 / max(1, args.steps + args.warmup))))
    times = []
    for i in range(args.warmup + args.steps):
        secs, res = cpu_reference_run(rows)
        if i >= args.warmup:
            times.append(secs)
    t = sum(times)
    value = rows * len(times) / t
    exp = expected(rows)
    assert list(res) == [exp["avg"], exp["max"], exp["min"]], (res, exp)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"result": list(res)})
    total = args.rows or TOTAL_ROWS
    sample = (f"{rows} rows of numbers_mt per step (the {total}-row workload is {total / rows:.1f}x this; rows/s is size-independent), "
              f"8 partitions on {cores} threads, 10 000-row blocks, one Arrow-style pass per aggregate")
    out = {
        "impl": "reference", "metric": "rows_per_s", "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / len(times), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": value / (TOTAL_ROWS / README_PUBLISHED_SECONDS), "dtype": "u64", "data": "synthetic",
        "config": common_config(total),
        "note": "CPU oracle port of the reference pipeline (the reference is Rust; no rustc in this image), bounded sample per step",
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "cpu_model": cpu_model(),
    }
    print(json.dumps(out), flush=True)


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def _cpulist(text: str):
    ids = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        ids.update(range(int(a), int(b or a) + 1))
    return ids


def bind_to_gpu_cpus(local: int):
    """Pin this process (and so the placement of the pinned host buffers it allocates afterwards) to the CPUs next to its GPU:
    with 8 ranks the e2e leg otherwise pulls part of its host column across the socket interconnect.  Sources, in order: the
    PCI device's numa_node, its local_cpulist (present even where numa_node says -1).  Returns a description for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{getattr(pr, 'pci_domain_id', 0):04x}:{pr.pci_bus_id:02x}:{getattr(pr, 'pci_device_id', 0):02x}.0"
        base = f"/sys/bus/pci/devices/{bdf}"
        allowed_now = os.sched_getaffinity(0)
        node = int(open(f"{base}/numa_node").read().strip())
        cpus, src = set(), ""
        if node >= 0:
            cpus, src = _cpulist(open(f"/sys/devices/system/node/node{node}/cpulist").read()), f"numa node {node}"
        else:
            cpus, src = _cpulist(open(f"{base}/local_cpulist").read()), "pci local_cpulist (numa_node = -1)"
        pick = cpus & allowed_now
        n_nodes = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()])
        if pick and len(pick) < len(allowed_now):
            os.sched_setaffinity(0, pick)
            return f"{bdf}: bound to {len(pick)} cpus of {src}; host has {n_nodes} numa node(s)"
        return f"{bdf}: {src} covers every allowed cpu ({len(allowed_now)}): nothing to bind; host has {n_nodes} numa node(s)"
    except Exception as e:  # sysfs layout differs / container hides it: keep the default placement
        return f"not bound ({type(e).__name__}: {e})"


def mem_available_bytes():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


class DevPtr:
    """__cuda_array_interface__ view of a raw device buffer (the pipe's running state) for torch."""

    def __init__(self, ptr: int, n_u64: int):
        self.__cuda_array_interface__ = {"shape": (n_u64,), "typestr": "<i8", "data": (ptr, False), "version": 2}


class Rig:
    """Everything a measurement needs: context, stream, ranks, the group, max-over-ranks reductions."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from fuse_query_b200 import cabi
        self.torch, self.dist, self.cabi, self.args = torch, dist, cabi, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one process per GPU)")
        torch.cuda.set_device(self.local)
        self.dev = f"cuda:{self.local}"
        self.affinity = bind_to_gpu_cpus(self.local)
        if self.world > 1:
            # stdout carries the one JSON line.  NCCL_DEBUG=VERSION (set in the GPU image) makes NCCL printf "NCCL version ..."
            # to stdout, past NCCL_DEBUG_FILE; the level logs nothing else, so it is dropped.  Other levels go to stderr.
            if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
                del os.environ["NCCL_DEBUG"]
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.ctx = cabi.Context(self.local)
        self.stream = torch.cuda.current_stream().cuda_stream
        self.group, self.merge = None, "single GPU: the kernel's own fold is the final state"
        if self.world > 1:
            self.merge = "nccl all_gather of the running state + fold on the device after each launch"
            if args.merge == "peer":
                ok = torch.ones(1, device=self.dev)
                try:
                    g = self.ctx.group(self.rank, self.world)
                    handles = [None] * self.world
                    dist.all_gather_object(handles, g.handle())
                    g.connect(handles)
                    self.group = g
                except Exception as e:  # IPC not permitted in this container / no peer access: keep NCCL
                    sys.stderr.write(f"[bench] rank {self.rank}: peer-memory merge unavailable ({e}); using NCCL\n")
                    ok = torch.zeros(1, device=self.dev)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)   # all ranks or none
                if ok.item() != 1:
                    self.group = None
                else:
                    self.merge = ("in-kernel: the aggregate kernel's last CTA stores its state into every rank's exchange window over NVLink "
                                  "peer memory, waits for all ranks' states of the step and folds them (fq_group)")

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, values, op="max"):
        if self.world == 1:
            return list(values)
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return t.tolist()

    def event(self):
        return self.torch.cuda.Event(enable_timing=True)


class MergedPipe:
    """An aggregate pipe whose launch completes the query across ranks: in-kernel group merge, or NCCL all-gather + device fold."""

    def __init__(self, rig: Rig, exprs, generated: bool, leaf_ops):
        self.rig, self.leaf_ops = rig, leaf_ops
        self.pipe = rig.ctx.pipe(exprs, aggregate=True, generated=generated)
        self.use_nccl = rig.world > 1 and rig.group is None
        if rig.group is not None:
            self.pipe.set_group(rig.group)
        if self.use_nccl:
            t = rig.torch
            ptr, nbytes = self.pipe.state_device()
            self.n_slots = nbytes // 8
            self.state_t = t.as_tensor(DevPtr(ptr, self.n_slots), device=rig.dev)
            self.gathered = t.zeros((rig.world, self.n_slots), dtype=t.int64, device=rig.dev)
            self.folded = t.zeros(self.n_slots, dtype=t.int64, device=rig.dev)
            self.host = t.zeros(self.n_slots, dtype=t.int64).pin_memory()

    def launch(self, src):
        self.pipe.launch_aggregate(src, stream=self.rig.stream)
        self.exchange()

    def exchange(self):
        """NCCL arm only: the collective part of the step (the in-kernel merge needs nothing after the launch)."""
        if not self.use_nccl:
            return
        H = self.rig.cabi.STATE_HEADER_SLOTS
        self.rig.dist.all_gather_into_tensor(self.gathered.view(-1), self.state_t)
        self.folded[:H] = self.gathered[:, :H].sum(0)
        for k, op in enumerate(self.leaf_ops):     # this workload's values stay below 2^63 for min/max; sums wrap like u64
            col = self.gathered[:, H + k]
            self.folded[H + k] = col.sum() if op in ("sum", "count") else (col.max() if op == "max" else col.min())
        self.host.copy_(self.folded, non_blocking=True)

    def result(self):
        """-> (leaf values, rows) of the whole job, on this rank"""
        if self.rig.world == 1:
            states, rows = self.pipe.fetch_aggregate()
        elif not self.use_nccl:
            states, rows = self.pipe.fetch_merged()
        else:
            self.rig.torch.cuda.synchronize()
            H = self.rig.cabi.STATE_HEADER_SLOTS
            raw = [int(x) & M64 for x in self.host.tolist()]
            return [raw[0] if op == "count" else raw[H + k] for k, op in enumerate(self.leaf_ops)], raw[0]
        return [s[1] for s in states], rows

    def destroy(self):
        self.pipe.destroy()


def leaf_ops_of(exprs):
    """Aggregator leaves in node order (post-order of each expression in turn)."""
    import re
    ops = []
    for e in exprs:
        ops += re.findall(r"\((sum|count|max|min) ", e)
    return ops


def timed(rig: Rig, launch, reps: int, warm: int = 2):
    """ms per call of `launch` on this rig's stream, max over ranks; ranks enter together."""
    for _ in range(warm):
        launch()
    rig.barrier()
    a, b = rig.event(), rig.event()
    a.record()
    for _ in range(reps):
        launch()
    b.record()
    rig.torch.cuda.synchronize()
    return rig.reduce([a.elapsed_time(b) / reps])[0]


def run_ours(args):
    rig = Rig(args)
    torch, cabi, ctx, rank, world = rig.torch, rig.cabi, rig.ctx, rig.rank, rig.world
    total = args.rows or TOTAL_ROWS
    generated = args.mode == "generated"
    begin, n = shard_of(rank, world, total)

    # ---- resident shard (untimed): one fill kernel writes this rank's range into HBM ----
    col = None if generated else ctx.numbers(begin, n, rig.stream)
    src = cabi.make_source([] if generated else [col], n, generated=generated, begin=begin)
    head = MergedPipe(rig, HEADLINE, generated, leaf_ops_of(HEADLINE))

    # ---- the timed region: K complete queries ----
    for _ in range(max(args.warmup, 3)):
        head.launch(src)
    rig.barrier()
    sampler = ClockSampler(rig.local)
    sampler.start()
    time.sleep(0.25)
    launches0 = ctx.launch_count
    k_ev = [(rig.event(), rig.event()) for _ in range(args.steps)]
    e0, e1 = rig.event(), rig.event()
    rig.barrier()
    wall0 = time.time()
    e0.record()
    for i in range(args.steps):
        k_ev[i][0].record()
        head.pipe.launch_aggregate(src, stream=rig.stream)
        k_ev[i][1].record()
        head.exchange()
    e1.record()
    rig.barrier()
    wall1 = time.time()
    clocks = sampler.stop(wall0, wall1)
    launches = ctx.launch_count - launches0
    ms = e0.elapsed_time(e1)
    kernel_ms = statistics.mean(a.elapsed_time(b) for a, b in k_ev)
    ms, kernel_ms = rig.reduce([ms, kernel_ms])
    launches = int(rig.reduce([float(launches)], "sum")[0])
    # ---- validity: the merged result every rank holds after the last step must be the reference's answer, bit-exact ----
    vals, rows = head.result()
    exp = expected(total)
    got = {"sum": vals[0], "count": vals[1], "avg": vals[0] // vals[1], "max": vals[2], "min": vals[3]}
    assert got == exp and rows == total, f"rank {rank}: result mismatch: {got} != {exp}"
    if args.dump_outputs and rank == 0:
        # the query's row, the merged Aggregator-leaf states (sum, count, max, min) and the rows the last step scanned
        dump_outputs(args.dump_outputs, {"result": [got["avg"], got["max"], got["min"]], "leaf_states_hi_lo": u64_hi_lo(vals), "rows": [rows]})

    # ---- the same kernels back to back without the cross-rank merge (what round 1 reported as the step) ----
    no_merge = None
    if world > 1 and rig.group is not None:
        head.pipe.set_group(None)
        t_ms = timed(rig, lambda: head.pipe.launch_aggregate(src, stream=rig.stream), args.steps, warm=2)
        head.pipe.set_group(rig.group)
        no_merge = {"ms_per_step": t_ms, "rows_per_s": total / (t_ms * 1e-3),
                    "note": "kernels back to back, no exchange and no wait for the other ranks: NOT a complete query"}

    # ---- every README query x {materialised, generated}: whole-job numbers at this N, merged result verified ----
    per_query = {}
    group_by = None
    order_by = None
    if not args.no_query_table:
        per_query = query_table(rig, col, begin, n, total, generated)
        if col is not None:
            group_by = group_by_table(rig, col)
            order_by = order_by_table(rig, col) if world == 1 else None

    # ---- e2e: host-resident (pinned) column -> H2D chunks overlapped with the kernel -> D2H state ----
    e2e = run_e2e(rig, col, begin, n, total, generated)

    rig.barrier()
    sql_e2e = None
    if rank == 0 and world == 1 and not args.no_query_table:
        if col is not None:
            col.free()
            col = None
        sql_e2e = run_sql_e2e(rig.local, total)

    if rank == 0:
        peak, which = peaks()
        secs = ms * 1e-3
        value = total * args.steps / secs
        kernel_s = kernel_ms * 1e-3
        row_bytes = 0 if generated else 8
        achieved = row_bytes * n / kernel_s / 1e9
        cfg = common_config(total)
        out = {
            "metric": "rows_per_s", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": value / (TOTAL_ROWS / README_PUBLISHED_SECONDS), "dtype": "u64", "data": "synthetic",
            "config": cfg,
            "setup": {"rows_per_gpu": n, "source": args.mode,
                      "partitioning": f"{8 // world if world <= 8 else 1} of the reference's 8 partitions per GPU",
                      "host_affinity": rig.affinity,
                      "l2": "inputs (>= 10 GB per GPU) are far larger than the 126 MB L2; no flush needed",
                      "merge": rig.merge,
                      "step": "one complete query: every rank's kernel + the cross-rank merge; each rank holds the merged state when its kernel ends",
                      "vs_baseline_ref": "README.md:62 FuseQuery 6.40 s for this query on an 8 vCPU KVM instance"},
            "hbm_gb_per_s": row_bytes * total * args.steps / secs / 1e9,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(n, generated),
                         "kernel": agg_kernel_name(generated), "kernel_ms": kernel_ms, "peak_source": which,
                         "algorithmic_bytes_per_launch": row_bytes * n,
                         "note": "kernel_ms includes the in-kernel wait for the slowest rank when N > 1"},
            "throughput_no_merge": no_merge,
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "result": got, "per_query": per_query, "group_by": group_by, "order_by": order_by,
            "sql_e2e": sql_e2e,
        }
        if world == 1 and not args.no_cpu_baseline:
            rows_cpu = cpu_sample_rows()
            secs_cpu, _ = cpu_reference_run(rows_cpu)
            out["cpu_baseline"] = {"value": rows_cpu / secs_cpu, "unit": "rows/s", "cores": min(8, os.cpu_count() or 1), "kind": "port",
                                   "sample": f"{rows_cpu} rows of the same query through the oracle's reference-shaped pipeline "
                                             f"(8 partitions, 10 000-row blocks, one pass per aggregate), {secs_cpu:.2f} s; cpu: {cpu_model()}"}
            # SURVEY 8d-i: the best a CPU could do with this query, NOT the reference's structure: one fused pass per
            # thread over numbers generated in registers, all host threads.  Reported beside the baseline, not as it.
            from oracle import binding as _o
            nthreads = os.cpu_count() or 1
            _o.fused_headline(1_000_000_000, nthreads)
            secs_best, res_best = _o.fused_headline(TOTAL_ROWS, nthreads)
            assert res_best == [_sum(TOTAL_ROWS), TOTAL_ROWS, TOTAL_ROWS - 1, 0], res_best
            out["cpu_baseline"]["best_case_fused"] = {"value": TOTAL_ROWS / secs_best, "unit": "rows/s", "cores": nthreads,
                                                      "note": "hand-fused single pass, generated in registers, vectorised by gcc -O3 -march=native; "
                                                              "compare with per_query[...]['generated'], not with the materialised scan"}
        print(json.dumps(out), flush=True)
    rig.barrier()
    head.destroy()
    if rig.group is not None:
        rig.group.destroy()
    if world > 1:
        rig.dist.destroy_process_group()


def query_table(rig: Rig, col, begin, n, total, generated_only):
    """Whole-job time of every README query (and BASELINE configs 0-2) at this N: all ranks launch together, the launch ends
    with the merged state on every rank, max over ranks, result asserted against the closed form on EVERY rank."""
    cabi, ctx, world, rank, torch = rig.cabi, rig.ctx, rig.world, rig.rank, rig.torch
    per_query = {}
    reps = 3

    def record(name, mode, ms, rows, nbytes, extra=None):
        d = {"ms": round(ms, 4), "rows_per_s": rows / (ms * 1e-3), "gb_per_s": (nbytes / (ms * 1e-3) / 1e9) if nbytes else None,
             "verified": True, "n_gpus": world}
        if extra:
            d.update(extra)
        per_query.setdefault(name, {})[mode] = d

    for name, (exprs, want, readme_s, note) in README_QUERIES.items():
        for mode in ("materialised", "generated"):
            g = mode == "generated"
            if not g and generated_only:
                continue
            mp = MergedPipe(rig, exprs, g, leaf_ops_of(exprs))
            s = cabi.make_source([] if g else [col], n, generated=g, begin=begin)
            ms = timed(rig, lambda: mp.launch(s), reps)
            vals, rows = mp.result()
            assert rows == total and vals == want(total), f"rank {rank}: {name} [{mode}]: {vals} != {want(total)}"
            reads = (not g) and not name.startswith("count(number)") or (not g and "honest" in name)
            extra = {"readme_seconds_8vcpu": readme_s}
            if note:
                extra["note"] = note
            record(name, mode, ms, total, 8 * total if reads else 0, extra)
            mp.destroy()

    # BASELINE configs[0] (the reference's own CPU-runnable case: 80 MB per job, L2-resident — a latency figure, not bandwidth)
    t0 = 10_000_000
    b0, n0 = shard_of(rank, world, t0)
    for mode in ("materialised", "generated"):
        g = mode == "generated"
        if not g and generated_only:
            continue
        if not g:
            ctx.fill_numbers(col, b0, n0, rig.stream)
        mp = MergedPipe(rig, [f"(sum {NUM})"], g, ["sum"])
        s0 = cabi.make_source([] if g else [col], n0, generated=g, begin=b0)
        ms = timed(rig, lambda: mp.launch(s0), 20, warm=5)
        vals, rows = mp.result()
        assert rows == t0 and vals == [_sum(t0)], (vals, rows)
        record("cfg0: sum(number) @1e7", mode, ms, t0, 0, {"note": "80 MB per job: L2-resident and launch-latency bound; no bandwidth claim"})
        mp.destroy()

    # BASELINE configs[1] and [2] over numbers_mt(10^9), sharded like the headline
    t2 = min(total, 1_000_000_000)
    b2, n2 = shard_of(rank, world, t2)
    if col is not None:
        ctx.fill_numbers(col, b2, n2, rig.stream)      # this rank's shard of numbers_mt(10^9) (overwrites the head of the column)
        ms = timed(rig, lambda: ctx.fill_numbers(col, b2, n2, rig.stream), reps)
        record("source: fill numbers_mt(1e9)", "materialised", ms, t2, 8 * t2, {"note": "fq_fill_numbers, write-only"})
    for mode in ("materialised", "generated"):
        g = mode == "generated"
        if not g and generated_only:
            continue
        s2 = cabi.make_source([] if g else [col], n2, generated=g, begin=b2)
        mp = MergedPipe(rig, CFG1, g, leaf_ops_of(CFG1))
        ms = timed(rig, lambda: mp.launch(s2), reps)
        vals, rows = mp.result()
        assert rows == t2 and vals == [t2, 0, t2], (vals, rows)
        record("cfg1: max(number+1),min(number),count(number) @1e9", mode, ms, t2, 0 if g else 8 * t2)
        mp.destroy()

        # cfg2: every rank filters + projects its shard with LIMIT 3; the rows of all ranks meet in rank order and are cut
        # at LIMIT 3 again (pipeline_builder.rs:31-41) — on the device, over the group's windows, when there is one
        p = ctx.pipe(CFG2_PROJ, predicate=CFG2_PRED, generated=g)
        outs = [ctx.column(cabi.U64, 3), ctx.column(cabi.U64, 3)]
        fin = [ctx.column(cabi.U64, 3 * world), ctx.column(cabi.U64, 3 * world)]
        for early in (False, True):
            def one():
                p.launch_project(s2, outs, 3, limit=3, early_exit=early, stream=rig.stream)
                if rig.group is not None:
                    rig.group.gather_project(p, outs, fin, limit=3, stream=rig.stream)
            ms = timed(rig, one, reps)
            if rig.group is not None:
                sel, nfin = rig.group.fetch_gather()
                rows_out = list(zip(fin[0].to_numpy(nfin).tolist(), fin[1].to_numpy(nfin).tolist()))
            else:
                sel, written = p.fetch_project()
                mine = list(zip(outs[0].to_numpy(written).tolist(), outs[1].to_numpy(written).tolist()))
                if world > 1:
                    allrows = [None] * world
                    rig.dist.all_gather_object(allrows, (sel, mine))
                    sel, rows_out = sum(a for a, _ in allrows), [r for _, rr in allrows for r in rr][:3]
                else:
                    rows_out = mine
            assert rows_out == [(1, 0), (2, 0), (3, 1)] and (early or sel == 66), (rows_out, sel)
            key = "cfg2: filter+projection+limit 3 @1e9" + (" (limit early exit)" if early else " (full scan)")
            record(key, mode, ms, t2, 0 if (g or early) else 8 * t2,
                   {"note": "early exit: the scan stops once LIMIT rows were found; rows/s counts rows of the table, not rows read"} if early else None)
        if rig.group is None and world == 1:
            # the same query as a prepared statement: its launches (memset, kernel, copy-back of the counters) recorded once
            # as a CUDA graph and replayed (fq_graph_*), next to direct launches of the same pipe on the same stream
            torch.cuda.synchronize()
            gs = torch.cuda.Stream()
            with torch.cuda.stream(gs):
                ctx.graph_begin(gs.cuda_stream)
                p.launch_project(s2, outs, 3, limit=3, early_exit=True, stream=gs.cuda_stream)
                graph = ctx.graph_end(gs.cuda_stream)
                ms_direct = timed(rig, lambda: p.launch_project(s2, outs, 3, limit=3, early_exit=True, stream=gs.cuda_stream), 50, warm=5)
                ms = timed(rig, lambda: graph.launch(gs.cuda_stream), 50, warm=5)
                sel, written = p.fetch_project()
                got = list(zip(outs[0].to_numpy(written, stream=gs.cuda_stream).tolist(), outs[1].to_numpy(written, stream=gs.cuda_stream).tolist()))
            assert got == [(1, 0), (2, 0), (3, 1)], got
            record("cfg2: filter+projection+limit 3 @1e9 (limit early exit, graph replay)", mode, ms, t2, 0,
                   {"direct_launch_ms": round(ms_direct, 5),
                    "note": "launch-latency figure: one cudaGraphLaunch per query instead of one launch per memset / kernel / copy"})
            graph.destroy()
        p.destroy()
        for c in outs + fin:
            c.free()
    return per_query


def group_by_table(rig: Rig, col):
    """GROUP BY hash aggregation (SURVEY 8 f4) over numbers_mt(10^9): SELECT number % k, sum, count, min, max ... GROUP BY
    number % k (written number - number / k * k: the reference has no % operator).  Whole-job time at this N: every rank
    aggregates its shard into its own hash table; at N > 1 the partial groups then travel to their owner rank
    (hash(key) mod N) with one NCCL all-to-all over NVLink and are folded there (fq_pipe_export_partials /
    fq_pipe_merge_partials).  Verified: number of groups, and the column sums of count / sum / min / max against closed forms."""
    cabi, ctx, world, rank, torch, dist = rig.cabi, rig.ctx, rig.world, rig.rank, rig.torch, rig.dist
    total = 1_000_000_000
    b, n = shard_of(rank, world, total)
    ctx.fill_numbers(col, b, n, rig.stream)
    src = cabi.make_source([col], n)
    out = {}
    aggs = [f"(sum {NUM})", f"(count {NUM})", f"(min {NUM})", f"(max {NUM})"]
    if world > 1:
        # NCCL opens its peer-to-peer channels on first use per pair: a full all-to-all now, so that the first timed key count
        # (7 groups: most pairs exchange nothing) does not pay for connections the later ones need
        w = torch.ones(world * 16, dtype=torch.int64, device=rig.dev)
        dist.all_to_all_single(torch.empty_like(w), w)
        torch.cuda.synchronize()
    for k in (7, 1000, 5000, 1_000_000, 100_000_000):
        key = f"(- {NUM} (* (/ {NUM} (u64 {k})) (u64 {k})))"
        pipe = ctx.pipe(aggs, keys=[key])
        owner = ctx.pipe(aggs, keys=[key]) if world > 1 else None
        slots = pipe.group_entry_slots()
        local_groups = min(k, n)
        pipe.groupby_reserve(local_groups)
        if owner is not None:
            owner.groupby_reserve(k // world + k // (4 * world) + 1024)
        ent = ctx.column(cabi.U64, local_groups * slots) if world > 1 else None
        recv = None

        def one():
            nonlocal recv
            pipe.launch_groupby(src, stream=rig.stream)
            if world == 1:
                return
            g = pipe.fetch_groupby()
            counts = pipe.export_partials(world, ent, stream=rig.stream)
            send_counts = torch.tensor(counts, dtype=torch.int64, device=rig.dev)
            recv_counts = torch.empty_like(send_counts)
            dist.all_to_all_single(recv_counts, send_counts)
            rc = recv_counts.tolist()
            send_t = torch.as_tensor(DevPtr(ent.device_ptr, g * slots), device=rig.dev)
            if recv is None or recv[1] < sum(rc) * slots:
                recv = (ctx.column(cabi.U64, max(1, sum(rc) * slots)), sum(rc) * slots)
            recv_t = torch.as_tensor(DevPtr(recv[0].device_ptr, max(1, sum(rc) * slots)), device=rig.dev)[:sum(rc) * slots]
            dist.all_to_all_single(recv_t, send_t[:g * slots], [c * slots for c in rc], [c * slots for c in counts])
            torch.cuda.current_stream().synchronize()
            owner.merge_partials(recv[0], sum(rc), stream=rig.stream)

        reps = 2 if k >= 1_000_000 else 3
        ms = timed(rig, one, reps, warm=1)
        final = owner if owner is not None else pipe
        groups = final.fetch_groupby()
        keys, kval, leaves, lval = final.export_groups(groups)
        lv = [torch.as_tensor(DevPtr(c.device_ptr, max(1, groups)), device=rig.dev)[:groups] for c in leaves]
        # checks that need no sort: totals over all groups (and all ranks)
        sums = [int(lv[0].sum().item()) & M64, int(lv[1].sum().item()), int(lv[2].sum().item()) & M64, int(lv[3].sum().item()) & M64, groups]
        if world > 1:
            gathered = [None] * world
            dist.all_gather_object(gathered, sums)
            sums = [sum(x[i] for x in gathered) & M64 for i in range(5)]
        kk = min(k, total)
        # group r's max is the largest number below `total` congruent to r
        max_sum = (kk * (total - kk) + _sum(kk)) if total % kk == 0 else sum(((total - 1 - r) // kk) * kk + r for r in range(kk))
        want = [_sum(total), total, _sum(kk), max_sum & M64, kk]
        assert sums == want, f"group by k={k}: {sums} != {want}"
        table_bytes = (2 * local_groups) * 8 * slots
        out[f"number % {k}"] = {"ms": round(ms, 4), "rows_per_s": total / (ms * 1e-3), "groups": kk, "verified": True, "n_gpus": world,
                                "read_gb_per_s": 8 * total / (ms * 1e-3) / 1e9,
                                "bytes": {"column_read": 8 * total, "table_per_gpu_at_least": table_bytes},
                                "note": "whole job: scan + hash aggregation" + (" + all-to-all of partial groups + merge" if world > 1 else "")}
        for c in keys + leaves:
            c.free()
        pipe.destroy()
        if owner is not None:
            owner.destroy()
        if ent is not None:
            ent.free()
        if recv is not None:
            recv[0].free()
    return out


def order_by_table(rig: Rig, col):
    """ORDER BY (SURVEY 8 f4) over numbers_mt(10^9) on one GPU: fq_sort_indices (stable LSD radix sort of row indexes) +
    fq_column_take of the payload.  Two key shapes: `number DESC` (input already ordered the other way; 4 of 8 digits vary)
    and a 64-bit scrambled key `number * 0x9E3779B97F4A7C15` (every digit varies: 8 passes).  Verified on the device: the
    gathered keys are ordered and the row indexes are a permutation (sum and xor of 0 .. n-1)."""
    cabi, ctx, torch = rig.cabi, rig.ctx, rig.torch
    n = 1_000_000_000
    ctx.fill_numbers(col, 0, n, rig.stream)
    keycol = col.slice(0, n)
    out = {}
    scr = ctx.pipe([f"(* {NUM} (u64 {0x9E3779B97F4A7C15}))"])
    scrambled = ctx.column(cabi.U64, n)
    scr.launch_project(cabi.make_source([keycol], n), [scrambled], n, stream=rig.stream)
    assert scr.fetch_project()[1] == n
    scr.destroy()
    for name, key, desc in (("number desc", keycol, True), ("number * 0x9E3779B97F4A7C15 (64-bit scrambled)", scrambled, False)):
        idx = ctx.column(cabi.U32, n)
        ms_sort = timed(rig, lambda: ctx.sort_indices([key], n, [desc], stream=rig.stream, out=idx), 2, warm=1)
        a, b = rig.event(), rig.event()
        a.record()
        taken = ctx.take(key, idx, n, stream=rig.stream)
        b.record()
        torch.cuda.synchronize()
        ms_take = a.elapsed_time(b)
        t = torch.as_tensor(DevPtr(taken.device_ptr, n), device=rig.dev)
        rows = torch.as_tensor(DevPtr(idx.device_ptr, n // 2), device=rig.dev).view(torch.int32)     # u32 indexes, 2 per i64
        if desc:
            ordered = bool((t[1:] < t[:-1]).all().item())
        else:   # unsigned order of i64 views: flip the sign bit
            u = t ^ (-(1 << 63))
            ordered = bool((u[1:] >= u[:-1]).all().item())
            del u
        perm_ok = int(rows.sum(dtype=torch.int64).item()) == n * (n - 1) // 2
        assert ordered and perm_ok, (name, ordered, perm_ok)
        passes = 4 if desc else 8
        out[name] = {"sort_ms": round(ms_sort, 3), "take_ms": round(ms_take, 3), "rows_per_s": n / (ms_sort * 1e-3), "passes": passes, "verified": True,
                     "bytes": {"algorithmic_per_pass": 36 * n, "note": "12 B read for the histogram + 12 B read + 12 B written by the scatter, per row and pass"},
                     "gb_per_s": passes * 36 * n / (ms_sort * 1e-3) / 1e9}
        del t, rows
        idx.free()
        taken.free()
        # ORDER BY key LIMIT 10: radix select instead of the full sort; checked against the head of the full order
        def top():
            i2, _ = ctx.sort_indices_limit([key], n, 10, [desc], stream=rig.stream)
            i2.free()
        ms_top = timed(rig, top, 3, warm=1)
        i2, cnt = ctx.sort_indices_limit([key], n, 10, [desc], stream=rig.stream)
        head10 = ctx.take(key, i2, cnt, stream=rig.stream).to_numpy(cnt)
        if desc:
            assert head10.tolist() == [n - 1 - j for j in range(10)], head10
        else:
            assert bool((head10[1:] >= head10[:-1]).all()) and int(head10[0]) == int(torch.as_tensor(DevPtr(key.device_ptr, n), device=rig.dev).view(torch.int64).bitwise_xor(-(1 << 63)).min().item() ^ -(1 << 63)) & M64
        out[name]["limit_10_ms"] = round(ms_top, 3)
        i2.free()
    scrambled.free()
    ctx.trim()           # 24 GB of sort scratch back to the device before the e2e leg
    return out


def run_sql_e2e(device, total):
    """The call a user of the reference makes: SQL text in, result rows out (Planner -> Optimizer -> PipelineBuilder ->
    SelectExecutor, mysql_handler.rs:52-75), wall clock including planning, kernel launches and the D2H of the result.
    numbers_mt is a generator table: `generated` computes it in-kernel, `materialised` scans the shard resident in HBM
    (filled on first use, like a table load; that first query is reported separately)."""
    from fuse_query_b200 import _fuse_host as h
    gpu = h.GpuContext.create(device)
    sql = HEADLINE_SQL.replace("10000000000", str(total))
    exp = expected(total)
    out = {}
    for mode in ("generated", "materialised"):
        c = h.FuseQueryContext.create_ctx(1, gpu)
        c.options.generated = mode == "generated"
        t0 = time.time()
        rows = [tuple(b.column(i).to_list()[0] for i in range(b.num_columns())) for b in h.execute_sql(c, sql)]
        first = time.time() - t0
        assert rows == [(exp["avg"], exp["max"], exp["min"])], rows
        reps = 5
        t0 = time.time()
        for _ in range(reps):
            h.execute_sql(c, sql)[0].column(0).to_list()
        dt = (time.time() - t0) / reps
        out[mode] = {"ms_per_query": 1e3 * dt, "rows_per_s": total / dt, "first_query_ms": 1e3 * first}
    h.numbers_cache_clear()
    return out


def run_e2e(rig: Rig, col, begin_full, n_full, total_full, generated):
    """Same query, inputs in HOST memory: each step copies this rank's share of the column from pinned memory in chunks
    (double-buffered against the kernel, which folds chunk after chunk into the running state; the last chunk's launch
    ends with the cross-rank merge) and reads the merged state back.  Also measured: the plain cudaMemcpyAsync rate of the
    very same copies without any kernel, on all ranks at once — the roofline of this leg."""
    import ctypes as C

    import numpy as np
    args, torch, cabi, ctx, world, rank = rig.args, rig.torch, rig.cabi, rig.ctx, rig.world, rig.rank
    L = cabi.lib()
    # the headline's 10^10 rows when the host can pin them (80 GB at N=1), else --e2e-rows
    total = args.e2e_rows or total_full
    why = None
    avail = -rig.reduce([-float(mem_available_bytes())])[0]      # min over ranks (they share the host)
    if not args.e2e_rows and (8 * total * 1.25 + (24 << 30) > avail or generated):
        total, why = min(total_full, 1_000_000_000), f"host MemAvailable {avail / 2**30:.0f} GiB cannot pin {8 * total_full / 2**30:.0f} GiB safely"
    hp = C.c_void_p()
    while True:
        begin, n = shard_of(rank, world, total)
        t_pin = time.time()
        ok = 1.0
        try:
            ctx.check(L.fq_host_alloc(ctx._h, max(n, 1) * 8, C.byref(hp)))
        except cabi.FuseGpuError as e:
            ok, why = 0.0, f"pinning {8 * n / 2**30:.0f} GiB failed ({e})"
        t_pin = time.time() - t_pin
        if -rig.reduce([-ok])[0] == 1.0:
            break
        if ok:
            L.fq_host_free(ctx._h, hp)
        if total <= 1_000_000_000:
            raise SystemExit("cannot pin host memory for the e2e leg")
        total = 1_000_000_000
    # the host-side DataBlocks of the reference (numbers_stream.rs:68-83): written by D2H copies of the resident column where
    # it holds exactly these numbers (fast), else by numpy
    if col is not None and (begin, n) == (begin_full, n_full):
        ctx.fill_numbers(col, begin, n, rig.stream)   # query_table may have overwritten the head of the column
        step_rows = 1 << 27
        for i in range(0, n, step_rows):
            m = min(step_rows, n - i)
            ctx.check(L.fq_column_download(ctx._h, col._h, i, C.c_void_p(hp.value + i * 8), m, C.c_void_p(rig.stream)))
        ctx.synchronize(rig.stream)
    else:
        host = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_uint64)), shape=(max(n, 1),))
        step_rows = 1 << 24
        for i in range(0, n, step_rows):
            host[i:i + step_rows] = np.arange(begin + i, begin + min(n, i + step_rows), dtype=np.uint64)
    chunk = max(1, min(n, args.e2e_chunk_rows))
    bufs = [ctx.column(cabi.U64, chunk), ctx.column(cabi.U64, chunk)]
    mp = MergedPipe(rig, HEADLINE, False, leaf_ops_of(HEADLINE))
    pipe = mp.pipe
    if rig.group is not None:
        pipe.set_group(None)      # only the last chunk's launch of a step merges across ranks
    state_bytes = pipe.state_device()[1]
    copy_s, comp_s = torch.cuda.Stream(), torch.cuda.Stream()
    free_ev = [torch.cuda.Event(), torch.cuda.Event()]
    full_ev = [torch.cuda.Event(), torch.cuda.Event()]
    n_chunks = (n + chunk - 1) // chunk
    counts = {"h2d": 0, "d2h": 0}

    def one(with_kernel=True):
        counts["h2d"] = counts["d2h"] = 0
        k = 0
        for off in range(0, n, chunk):
            m = min(chunk, n - off)
            b = k & 1
            copy_s.wait_event(free_ev[b])
            ctx.check(L.fq_column_upload(ctx._h, bufs[b]._h, 0, C.c_void_p(hp.value + off * 8), m, C.c_void_p(copy_s.cuda_stream)))
            full_ev[b].record(copy_s)
            counts["h2d"] += m * 8
            if with_kernel:
                comp_s.wait_event(full_ev[b])
                last = k == n_chunks - 1
                if last and rig.group is not None:
                    pipe.set_group(rig.group)
                pipe.launch_aggregate(cabi.make_source([bufs[b]], m), accumulate=k > 0, stream=comp_s.cuda_stream)
                if last and rig.group is not None:
                    pipe.set_group(None)
                free_ev[b].record(comp_s)
                counts["d2h"] += state_bytes * (2 if last and rig.group is not None else 1)   # every launch queues the D2H of its state
            else:
                free_ev[b].record(copy_s)
            k += 1
        if not with_kernel:
            copy_s.synchronize()
            return None
        if rig.group is not None:
            return pipe.fetch_merged()
        return pipe.fetch_aggregate()   # waits for the last launch, D2H of the state

    def measure(with_kernel, steps):
        for _ in range(2 if with_kernel else 1):
            one(with_kernel)
        rig.barrier()
        t0 = time.time()
        for _ in range(steps):
            res = one(with_kernel)
        torch.cuda.synchronize()
        mine = time.time() - t0
        rig.barrier()
        return res, mine

    res, dt_mine = measure(True, args.e2e_steps)
    h2d, d2h = counts["h2d"], counts["d2h"]
    dt = rig.reduce([dt_mine])[0]
    h2d_all, d2h_all = rig.reduce([float(h2d), float(d2h)], "sum")
    states, rows = res
    vals = [s[1] for s in states]
    if rig.group is not None or world == 1:
        assert rows == total and vals == [_sum(total), total, total - 1, 0], (vals, rows)
    else:
        assert rows == n and vals == [_sum(n, begin), n, begin + n - 1, begin], (vals, rows)
    # roofline of the leg: the same pinned -> device copies, one plain cudaMemcpyAsync per chunk, no kernel, all ranks at once
    _, roof_mine = measure(False, args.e2e_steps)
    roof_dt = rig.reduce([roof_mine])[0]
    per_rank = [0.0] * world
    per_rank[rank] = 8 * n * args.e2e_steps / roof_mine / 1e9
    per_rank = rig.reduce(per_rank, "sum")
    for b in bufs:
        b.free()
    mp.destroy()
    L.fq_host_free(ctx._h, hp)
    value = total * args.e2e_steps / dt
    roof_gbs = 8 * total * args.e2e_steps / roof_dt / 1e9
    return {"value": value, "unit": "rows/s", "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all),
            "rows_per_step": total, "ms_per_step": 1e3 * dt / args.e2e_steps, "h2d_gb_per_s": 8 * value / 1e9,
            "chunk_rows": chunk, "pinned_alloc_s": round(t_pin, 2),
            "roofline": {"bound": "pcie", "achieved": 8 * value / 1e9, "peak": roof_gbs, "unit": "GB/s", "frac": 8 * value / 1e9 / roof_gbs,
                         "per_gpu_gb_per_s": [round(x, 2) for x in per_rank],
                         "how": "the same chunks copied pinned -> device with one cudaMemcpyAsync each (fq_column_upload), no kernel, "
                                "all ranks concurrently; aggregate = bytes of all ranks / slowest rank's time"},
            "rows_note": why or "the headline's own table (same_config)",
            "note": "host-resident UInt64 column in pinned memory, chunked H2D overlapped with the kernel; PCIe-bound"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=0, help="override the 10^10-row workload (debug)")
    ap.add_argument("--mode", default="materialised", choices=["materialised", "generated"])
    ap.add_argument("--merge", choices=["peer", "nccl"], default="peer", help="N > 1: how the per-rank states meet")
    ap.add_argument("--e2e-rows", type=int, default=0, help="rows of the host-buffer leg (default: the workload's, if the host can pin them)")
    ap.add_argument("--e2e-chunk-rows", type=int, default=1 << 25)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-query-table", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if "FQ_JIT_CACHE_DIR" not in os.environ:
        # kernels compiled at run time are cached in a directory of this run's own, not next to the library in the tree
        jit_dir = tempfile.mkdtemp(prefix="fq_jit_")
        atexit.register(shutil.rmtree, jit_dir, True)
        os.environ["FQ_JIT_CACHE_DIR"] = jit_dir
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
