"""Multi-GPU execution of a SELECT: one process per GPU (torch.distributed), partitions split across ranks.

The reference runs one pipe per chunk of partitions and merges them at MergeProcessor
(processors/pipeline_builder.rs:73-95, processor_merge.rs:37-66).  Here each rank runs the fused GpuPipeTransform
over ITS consecutive partitions; what crosses ranks is exactly what crosses the reference's merge channel:
the partial-state block (one Utf8/JSON row per aggregate expression, transform_aggregate_partial.rs:61-72) or the
filtered + projected rows.  The final stage (AggregateFinalTransform / LimitTransform) is the unchanged host logic; an
ORDER BY (GpuSortTransform, no counterpart in the reference) runs on every rank over the merged rows.
torch.distributed is plumbing: NCCL (or gloo) carries a few hundred bytes per rank.
"""
from __future__ import annotations

from typing import List, Tuple

import numpy as np

from . import _fuse_host as h


def _my_partitions(parts: list, rank: int, world: int) -> list:
    per = max(1, len(parts) // world)
    return parts[rank * per:(rank + 1) * per] if rank < world - 1 else parts[rank * per:]


def execute_sql_distributed(ctx, sql: str, rank: int, world: int, all_gather_object, gpu=None) -> Tuple[List[str], List[tuple]]:
    """Returns (column names, rows) on every rank.  `all_gather_object(obj) -> list` is the collective
    (torch.distributed.all_gather_object bound to a group).  With `gpu` (the rank's GpuContext) the rows of a LIMIT query
    meet on the device (fq_group) instead of travelling through the host."""
    plan = h.Optimizer.create().optimize(h.Planner().build_from_sql(ctx, sql))
    plans = plan.children_to_plans()
    src = plans[0]
    if src.name() != "ReadSourcePlan":
        raise h.FuseQueryError("Internal Error: distributed execution needs a table source")
    i = 1
    pred = None
    if i < len(plans) and plans[i].name() == "FilterPlan":
        pred = plans[i].predicate
        i += 1
    sel = plans[i]
    is_agg = sel.name() == "AggregatePlan"
    i += 1
    sort = None
    if i < len(plans) and plans[i].name() == "SortPlan":
        sort = plans[i]
        i += 1
    limit = None
    if i < len(plans) and plans[i].name() == "LimitPlan":
        limit = plans[i].n
        i += 1
    if i != len(plans) or sel.name() not in ("AggregatePlan", "ProjectionPlan"):
        # e.g. a derived table: its outer Filter / Projection would have to run after the cross-rank merge
        raise h.FuseQueryError("Internal Error: distributed execution supports ReadSource [Filter] (Projection | Aggregate) [Sort] [Limit], got "
                               + " -> ".join(p.name() for p in plans))
    if sort is not None and (sel.name() != "ProjectionPlan" or gpu is None):
        raise h.FuseQueryError("Internal Error: distributed ORDER BY needs a projection query and the rank's device context")
    if h.DataType.Utf8 in src.schema().types():
        # dictionary codes are local to the rank's table: rows of different ranks cannot be merged as codes
        raise h.FuseQueryError("Internal Error: Unsupported on the device path: distributed execution over a table with a Utf8 column")
    parts = _my_partitions(list(src.partitions), rank, world)
    names = sel.schema().names()
    local_blocks = []
    if parts:
        pipe = h.GpuPipeTransform.try_create(ctx, src.db, src.table, parts, pred, is_agg, sel.schema(), sel.expr,
                                             None if (is_agg or sort is not None) else limit)
        local_blocks = pipe.execute().collect()
    if sort is not None:
        # A sort is a pipeline breaker: every rank's rows meet (rank order = partition order, so ties keep the order one
        # process would give them) and every rank sorts the whole on its device.  Merge-then-sort: right, not scalable — a
        # range-partitioned sort (sample, all-to-all, local sorts) is what a large result would need.
        mine = [[b.column(c).to_numpy() for c in range(b.num_columns())] for b in local_blocks if b.num_rows() > 0]
        valid = [[(b.column(c).validity().to_numpy() if b.column(c).validity() is not None else None) for c in range(b.num_columns())]
                 for b in local_blocks if b.num_rows() > 0]
        gathered = all_gather_object((mine, valid))
        blocks = []
        for per_rank, per_rank_valid in gathered:
            for cols, vals in zip(per_rank, per_rank_valid):
                arrays = [h.DataArray.from_numpy(gpu, np.ascontiguousarray(a)) if v is None else h.DataArray.from_numpy_masked(gpu, np.ascontiguousarray(a), np.asarray(v) != 0)
                          for a, v in zip(cols, vals)]
                blocks.append(h.DataBlock.create(sel.schema(), arrays))
        if not blocks:
            return names, []
        srt = h.GpuSortTransform.try_create(ctx, sort.expr, list(sort.descending))
        srt.connect_to(h.DataBlockSource(blocks))
        out = srt.execute().collect()
        rows = [r for b in out for r in zip(*[b.column(c).to_list() for c in range(b.num_columns())])]
        return names, rows[:limit] if limit is not None else rows
    if is_agg:
        mine = [b.column(0).to_list() for b in local_blocks]            # JSON rows of this rank's partial block(s)
        gathered = all_gather_object(mine)
        blocks = [h.DataBlock.create(sel.schema(), [h.DataArray.utf8(rows)]) for per_rank in gathered for rows in per_rank]
        final = h.AggregateFinalTransform.try_create(ctx, sel.schema(), sel.expr)
        final.connect_to(h.DataBlockSource(blocks))
        out = final.execute().collect()
        rows = [tuple(b.column(c).to_list()[0] for c in range(b.num_columns())) for b in out]
        if limit is not None:
            rows = rows[:limit]
        return names, rows
    n_cols = len(names)
    if limit is not None and gpu is not None and world > 1:
        # MergeProcessor + the LimitTransform after it (processor_merge.rs:37-66, pipeline_builder.rs:31-41) on the device: every
        # rank's rows meet in every rank's exchange window over peer memory and the first `limit` rows, in rank (= partition)
        # order, are copied out — nothing but the 64-byte window handles ever crosses the host.
        group = _group_for(gpu, rank, world, all_gather_object)
        cols = [None] * n_cols
        rows_local = 0
        if local_blocks:                       # a fused pipe with a LIMIT yields at most `limit` rows, usually in one block
            merged = [b for b in local_blocks if b.num_rows() > 0]
            if len(merged) > 1:                # several runs of partitions: concatenate on the host side of this rank only
                mine = [np.concatenate([b.column(c).to_numpy() for b in merged])[:limit] for c in range(n_cols)]
                cols = [h.DataArray.from_numpy(gpu, a) for a in mine]
                rows_local = len(mine[0])
            elif merged:
                rows_local = min(merged[0].num_rows(), limit)
                cols = [merged[0].column(c).slice(0, rows_local) for c in range(n_cols)]
        types = [f.data_type for f in sel.schema().fields]
        finals, _selected = group.gather(cols, types, rows_local, rows_local, max(limit, 1), limit)
        rows = list(zip(*[a.to_list() for a in finals])) if finals and len(finals[0]) else []
        return names, rows
    mine = [[b.column(c).to_numpy() for c in range(b.num_columns())] for b in local_blocks]
    gathered = all_gather_object(mine)
    rows: List[tuple] = []
    for per_rank in gathered:                                           # rank order = partition order (a legal merge order)
        for cols in per_rank:
            rows.extend(zip(*[np.asarray(c).tolist() for c in cols]))
    if limit is not None:                                               # LimitTransform x 1 after the merge
        rows = rows[:limit]
    return names, rows


_GROUPS = {}


def _group_for(gpu, rank: int, world: int, all_gather_object):
    """One exchange window per (device context, world): created on first use, handles exchanged once."""
    key = (id(gpu), rank, world)
    if key not in _GROUPS:
        g = h.GpuGroup(gpu, rank, world, 1 << 20)
        g.connect(all_gather_object(g.handle()))
        _GROUPS[key] = g
    return _GROUPS[key]
