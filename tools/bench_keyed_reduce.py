#!/usr/bin/env python
"""bench_keyed_reduce.py -- group-by on a stored tag across GPUs (bydb_scan_reduce_keyed), next to bench.py:

    bench.py's 1e9-datapoint part (10,000 series x 100,000 points, tag default/region with 8 values) sharded by series range over
    N ranks, two queries through the keyed collective:
      region:          sum(latency), count(latency) GROUP BY region        -- bench.py's stored_tag_group_by leg (no series groups)
      service_region:  the same GROUP BY (service, region), service = (sid - 1) % 1000, Top 100 by sum(latency)

    python tools/bench_keyed_reduce.py --steps 20 --check                                        # one GPU (N = 1)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/bench_keyed_reduce.py --check

ms/step: host clock around one collective call (it returns after a synchronisation) after a barrier, median over the timed
steps, as seen by the root (rank 0); per-rank scan_kernel_ms is the sum of the rank's per-value scan passes.  Every rank runs
one scan pass per key value, so the fixed cost of a pass (block selection, reduce, read-back, host round trip) is paid once per
value on every rank and does not shrink with N.  --check runs the same collective over a 1/64 sample of the series (every 64th
series, drawn across all shards) and compares the root's answer with the oracle.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench as B  # noqa: E402

SERVICES = 1000
ARGS = None


def sample_part(n_series: int, sid0: int):
    """Every 64th series of bench.py's part from sid0 on: its generators are seeded per series, so the rows are the same."""
    from importlib import import_module
    S = import_module("bydb_b200.synth")
    fields = [("latency", S.F_LATENCY), ("walk", S.F_WALK3), ("ints", S.F_INT1000), ("uniform", S.F_UNIFORM)]
    return S.synth_part(n_series, ARGS.points, fields, sid0=sid0, sid_step=64, t0=B.T0, t_step=B.STEP, region_values=8, region_run=16, seed=B.SEED)


def gpu_identity(index: int):
    """-> (GPU name, enforced power limit in W) read now through nvidia-smi (a read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return out[0].strip(), float(out[1])
    except Exception:  # noqa: BLE001
        return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--series", type=int, default=10_000)
    ap.add_argument("--points", type=int, default=100_000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--check", action="store_true")
    args = ap.parse_args()
    global ARGS
    ARGS = args
    args.steps = max(args.steps, 20)
    rank, world, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = B.load_pkg()
    ctx = pkg.Context(device=local_rank)
    lo, hi = rank * args.series // world, (rank + 1) * args.series // world
    n_mine, sid0 = hi - lo, 1 + lo
    t0 = time.perf_counter()
    img = B.make_part(pkg, n_mine, args.points, sid0)
    t_gen = time.perf_counter() - t0
    h = ctx.register_part(1 + rank, img.files())
    del img
    sids = np.arange(sid0, sid0 + n_mine, dtype=np.uint64)
    aggs = [("latency", pkg.AGG_SUM), ("latency", pkg.AGG_COUNT)]

    def queries(handles, s):
        groups = ((s - 1) % SERVICES).astype(np.int32)
        return {"region": pkg.Query(parts=handles, series_ids=s, aggs=aggs),
                "service_region": pkg.Query(parts=handles, series_ids=s, aggs=aggs, series_group=groups, n_groups=SERVICES, top_n=100, top_agg=0,
                                            top_desc=True)}
    qs = queries([h], sids)
    slot = max(ctx.keyed_reduce_layout(q, "default", "region") for q in qs.values())
    mine_h = ctx.comm_export(slot, world)
    if world > 1:
        t = torch.frombuffer(bytearray(mine_h), dtype=torch.uint8).cuda()
        all_h = torch.empty(world * 128, dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(all_h, t)
        raw = all_h.cpu().numpy().tobytes()
        handles = [raw[i * 128:(i + 1) * 128] for i in range(world)]
    else:
        handles = [mine_h]
    ctx.comm_connect(rank, world, handles)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    name, plimit = gpu_identity(local_rank)
    results = {}
    for qname, q in qs.items():
        for _ in range(args.warmup):
            ctx.scan_reduce_keyed(q, "default", "region", root=0)
        times, scan_ms = [], []
        last = None
        for _ in range(args.steps):
            barrier()
            t = time.perf_counter()
            last = ctx.scan_reduce_keyed(q, "default", "region", root=0)
            times.append(time.perf_counter() - t)
            scan_ms.append(last.stats.scan_kernel_ms)
        per_rank = [float(np.median(scan_ms))]
        rows = float(last.stats.rows_scanned)
        if world > 1:
            g = [None] * world
            dist.all_gather_object(g, (float(np.median(scan_ms)), rows))
            per_rank = [x[0] for x in g]
            rows = sum(x[1] for x in g)
        results[qname] = {"ms_per_step": float(np.median(times)) * 1e3, "ms_per_step_min": float(np.min(times)) * 1e3,
                          "scan_kernel_ms_per_rank": per_rank, "datapoints_per_step": float(args.series * args.points),
                          "rows_scanned_all_passes": rows,   # every rank scans its shard once per key value
                          "rows_out": int(last.rows.size) if rank == 0 else None, "n_keys": int(last.n_keys) if rank == 0 else None}
        if rank == 0:
            results[qname]["datapoints_per_s"] = args.series * args.points / (results[qname]["ms_per_step"] * 1e-3)
            results[qname]["keys"] = [k.decode() for k in last.key[:8]]
    single = None
    if world == 1:   # the same query through bydb_scan_agg_keyed, for the record next to the collective at N = 1
        q = qs["region"]
        for _ in range(args.warmup):
            ctx.scan_agg_keyed(q, "default", "region")
        ts = []
        for _ in range(args.steps):
            t = time.perf_counter()
            ctx.scan_agg_keyed(q, "default", "region")
            ts.append(time.perf_counter() - t)
        single = {"api": "bydb_scan_agg_keyed", "query": "region", "ms_per_step": float(np.median(ts)) * 1e3}

    check = None
    if args.check:
        # every 64th series of the whole measure, each rank the ones in its shard; the collective runs on the same mailboxes
        first = lo + ((-lo) % 64)
        s_mine = np.arange(1 + first, 1 + hi, 64, dtype=np.uint64)
        simg = sample_part(len(s_mine), int(s_mine[0])) if len(s_mine) else None
        hs = ctx.register_part(900 + rank, simg.files()) if simg is not None else h   # an empty sample: the rank's shard selects no block
        sq = queries([hs], s_mine)
        got = {k: ctx.scan_reduce_keyed(q, "default", "region", root=0) for k, q in sq.items()}
        if rank == 0:
            import dataclasses
            from oracle import oracle as O
            s_all = np.arange(1, 1 + args.series, 64, dtype=np.uint64)
            whole = sample_part(len(s_all), 1)   # kept alive: files() are views into its memory
            op = O.Part.open({k: bytes(v) for k, v in whole.files().items()})
            ok = True
            detail = {}
            for k, q in queries([], s_all).items():
                oq = O.Query([op], s_all, aggs, groups=None if q.series_group is None else np.asarray(q.series_group), n_groups=q.n_groups,
                             top_n=q.top_n, top_agg=q.top_agg, top_desc=q.top_desc, threads=os.cpu_count() or 1)
                want = O.run_query(dataclasses.replace(oq, group_key=("default", "region")))
                g = got[k]
                same = (g.key == want.key and g.group_id.tolist() == want.group_id.tolist() and g.rows.tolist() == want.rows.tolist()
                        and g.val_i64.tolist() == want.val_i64.tolist())
                err = float(np.max(np.abs(g.val_f64 - want.val_f64) / np.maximum(np.abs(want.val_f64), 1e-300))) if want.val_f64.size else 0.0
                detail[k] = {"rows_out": int(g.rows.size), "exact_rows_keys_ints": bool(same), "float_max_rel_err": err}
                ok = ok and same and err <= 1e-9
            check = {"sample_series": int(s_all.size), "agrees_with_oracle": bool(ok), **detail}
    if rank == 0:
        print(json.dumps({"benchmark": "keyed_reduce", "n_gpus": world, "gpu": name, "power_limit_w": plimit, "steps": args.steps,
                          "workload": f"{args.series * args.points:.0e} datapoints ({args.series} x {args.points}), sharded by series range",
                          "queries": {"region": "sum(latency), count(latency) GROUP BY region (stored tag, 8 values)",
                                      "service_region": f"the same GROUP BY (service, region), {SERVICES} services x 8 values, Top 100 by sum"},
                          "results": results, "single_context_scan_agg_keyed": single, "generate_s_rank0": t_gen, "oracle_check": check}))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
