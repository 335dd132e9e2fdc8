#!/usr/bin/env python
"""bench.py -- the measure-query hot path on B200: scanned datapoints/s and achieved HBM GB/s.

Workload = BASELINE.json's north-star configuration (configs[2] / configs[3], SURVEY.md 8d C3 / C4):
    1e9 datapoints (10 000 series x 100 000 points), 4 float64 fields (latency, walk, ints, uniform) + a dictionary tag,
    query  GROUP BY service_id (1000 services x 10 series)  sum(latency), count(latency)  ->  Top 100 by the sum.
A "step" is one pass of the hot path (block selection -> page decode -> filter -> aggregate -> Top-N) over all of it.

``--gpus 1``  one part of 1e9 datapoints resident in one B200's HBM.
``--gpus N``  (torchrun) the SAME 1e9 datapoints sharded by series range over N ranks -- STRONG scaling (C4): every rank
              scans its shard into a partial table on its GPU, the tables meet on rank 0, which finalises (MEAN / Top-N).

``value``        datapoints scanned+aggregated per second with the parts already resident in HBM (whole job).
``e2e``          the same metric through the host-buffer entry point of the C ABI (bydb_scan_agg_host): part file images in
                 HOST memory in, result out, every step; legs for a caller whose images are pinned and for one whose are not.
``roofline``     algorithmic bytes (SURVEY.md 8d: 8 B per scanned datapoint for this query -- one float64 column; the group
                 id is per series, never read per row) / the scan kernel's CUDA-event time, against MEASURED_PEAKS.json.
``c2_query``     second leg on the same part: BASELINE configs[1]'s query (time range AND region == "r3", avg(latency) +
                 max(walk)), 25 algorithmic B per datapoint.
``cpu_baseline`` the oracle (C restatement of the reference's Go path; Go cannot be built in this image) on the host cores
                 over a stated sample of the same series, reference-shaped and all-core, with the GPU's answer on exactly
                 that sample compared against it (``agrees_with_gpu``).
``--impl reference`` times that CPU port alone on parts written by the oracle's own writer; the product library is not loaded.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T0 = 1_700_000_000_000_000_000
STEP = 60_000_000_000
SEED = 0xB200
B_ALG_C3 = 8    # sum(latency): one float64 column per scanned row (SURVEY.md 8d, C3)
B_ALG_C2 = 25   # 8 (timestamp) + 1 (dictionary tag) + 2 x 8 (fields)            (SURVEY.md 8d, C2)
METRIC = "measure datapoints scanned+aggregated/sec"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--series", type=int, default=10_000)
    ap.add_argument("--points", type=int, default=100_000)
    ap.add_argument("--services", type=int, default=1000)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target duration of each CPU baseline run")
    ap.add_argument("--sustained-steps", type=int, default=200, help="extra resident steps timed as one long region")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the sustained / graph / C2-query legs (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result of the last timed step as DIR/<name>.npy (float64), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        # the reference arm's sample is sized by the host's core count, so its inputs are not the same from machine to machine
        ap.error("--dump-outputs needs --impl b200")
    return args


def dump_outputs(out_dir, res):
    """The arrays a caller of the timed path receives (capi.Result), as float64 .npy files.  The int64 columns of this
    query are row numbers, counts and group ids, far below 2**53, so the conversion is exact."""
    os.makedirs(out_dir, exist_ok=True)
    for name in ("group_id", "rows", "is_float", "val_i64", "val_f64"):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(getattr(res, name), dtype=np.float64))


def load_pkg():
    import __graft_entry__ as ge
    if not os.path.exists(os.path.join(ge.PKG_DIR, "libbydbgpu.so")):
        ge.build()
    return ge.load_package()


def workload_text(n_series, n_points, services, world):
    s = (f"{n_series * n_points:.0e} datapoints ({n_series} series x {n_points} points), 4 float64 fields, GROUP BY service_id "
         f"({services} services), sum(latency)+count(latency), Top 100 desc by the sum")
    if world > 1:
        s += f"; the same data sharded by series range over {world} ranks (strong scaling)"
    return s


def traffic_from_profile():
    """dram__bytes_read.sum + dram__bytes_write.sum of one scan launch of this query, from the committed
    ncu --set full capture (profiles/traffic.json names it); None when there is none."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return int(t["dram_bytes_read"]) + int(t["dram_bytes_write"])
    except Exception:
        return None


FIELD_KINDS = ("latency", "walk", "ints", "uniform")


def make_part(pkg, n_series, n_points, sid0):
    """The synthetic part of SURVEY.md 8(d): per-series generators seeded by (SEED, series id), so a shard of the series
    holds exactly the rows the whole part holds for them."""
    from importlib import import_module
    S = import_module("bydb_b200.synth")
    fields = [("latency", S.F_LATENCY), ("walk", S.F_WALK3), ("ints", S.F_INT1000), ("uniform", S.F_UNIFORM)]
    return S.synth_part(n_series, n_points, fields, sid0=sid0, sid_step=1, t0=T0, t_step=STEP, region_values=8, region_run=16, seed=SEED)


def c3_query(pkg, handles, sids, services, flags=0):
    groups = ((np.asarray(sids, dtype=np.uint64) - 1) % services).astype(np.int32)   # service_id of a series comes from the index
    return pkg.Query(parts=handles, series_ids=sids, aggs=[("latency", pkg.AGG_SUM), ("latency", pkg.AGG_COUNT)], series_group=groups,
                     n_groups=services, top_n=100, top_agg=0, top_desc=True, flags=flags)


def c2_query(pkg, handles, sids, n_points):
    return pkg.Query(parts=handles, series_ids=sids, aggs=[("latency", pkg.AGG_MEAN), ("walk", pkg.AGG_MAX)], tmin=T0 + (n_points // 4) * STEP,
                     tmax=T0 + (3 * n_points // 4) * STEP, preds=[pkg.Pred("default", "region", pkg.OP_EQ, b"r3")])


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed regions (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index),
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU side (oracle)
def oracle_c3(O, parts, sids, services, threads, per_thread_partials=False):
    groups = ((np.asarray(sids, dtype=np.uint64) - 1) % services).astype(np.int32)
    return O.Query(parts, sids, [("latency", O.AGG_SUM), ("latency", O.AGG_COUNT)], groups=groups, n_groups=services, top_n=100, top_agg=0,
                   top_desc=True, threads=threads, per_thread_partials=per_thread_partials)


def timed_oracle(O, q):
    t = time.perf_counter()
    r = O.run_query(q)
    return time.perf_counter() - t, r


def oracle_written_parts(O, n_series, n_points, n_parts, threads):
    """Parts of the bench shape written by the ORACLE's own writer (oracle/part.c), n_parts series ranges built on a thread
    pool (the C calls release the GIL).  Values follow the same distributions as the product generator (numpy streams, not
    the same bits): they only feed the CPU arm."""
    from concurrent.futures import ThreadPoolExecutor
    per = max(1, n_series // n_parts)
    ranges = [(i * per, min(n_series, (i + 1) * per)) for i in range(n_parts) if i * per < n_series]
    ranges[-1] = (ranges[-1][0], n_series)

    def build(rg):
        a, b = rg
        ns = b - a
        rng = np.random.default_rng(SEED + a)
        n = ns * n_points
        sids = np.repeat(np.arange(1 + a, 1 + b, dtype=np.uint64), n_points)
        ts = np.tile(T0 + np.arange(n_points, dtype=np.int64) * STEP, ns)
        lat = np.round(25 + rng.normal(0, 5, n), 2)
        walk = np.round(50 + np.cumsum(rng.uniform(-0.1, 0.1, (ns, n_points)), axis=1), 3).reshape(-1)
        ints = rng.integers(0, 1000, n).astype(np.float64)
        uni = rng.uniform(0, 100, n)
        reg_vals = [b"r%d" % v for v in range(8)]
        runs = rng.integers(0, 8, n // 16 + 1)
        region = [reg_vals[v] for v in np.repeat(runs, 16)[:n]]
        pb = O.PartBuilder()
        pb.append(sids, ts, np.ones(n, np.int64),
                  [("latency", O.VT_FLOAT64, lat, None), ("walk", O.VT_FLOAT64, walk, None), ("ints", O.VT_FLOAT64, ints, None),
                   ("uniform", O.VT_FLOAT64, uni, None)], [("default", [("region", O.VT_STR, region, None)])])
        return pb.finish()

    with ThreadPoolExecutor(max_workers=max(1, min(threads, len(ranges)))) as ex:
        return list(ex.map(build, ranges))


def c1_cpu_number(O, cores):
    """BASELINE configs[0]: single part, 1k series x 1k points, 1 float64 field, sum() no filter -- the reference's own
    CPU-runnable case (template: banyand/measure/block_batch_benchmark_test.go:212-247), on the oracle."""
    rng = np.random.default_rng(SEED)
    ns, npts = 1000, 1000
    sids = np.repeat(np.arange(1, ns + 1, dtype=np.uint64), npts)
    ts = np.tile(T0 + np.arange(npts, dtype=np.int64) * STEP, ns)
    lat = np.round(25 + rng.normal(0, 5, sids.size), 2)
    pb = O.PartBuilder()
    pb.append(sids, ts, np.ones(sids.size, np.int64), [("latency", O.VT_FLOAT64, lat, None)])
    part = pb.finish()
    usid = np.arange(1, ns + 1, dtype=np.uint64)
    out = {}
    for label, thr, ptp in (("reference_shaped", cores, False), ("all_core_partials", cores, True), ("one_core", 1, False)):
        q = O.Query([part], usid, [("latency", O.AGG_SUM)], threads=thr, per_thread_partials=ptp)
        O.run_query(q)
        best = min(timed_oracle(O, q)[0] for _ in range(5))
        out[label] = {"value": ns * npts / best, "unit": "datapoints/s", "ms": best * 1e3, "threads": thr}
    out["workload"] = "1 part, 1000 series x 1000 points, 1 float64 field, sum(latency), no filter (BASELINE configs[0]); best of 5"
    return out


def reference_arm(args, cores):
    from oracle import oracle as O   # the product library is never loaded in this arm
    n_points, services = args.points, args.services
    steps, warmup = max(args.steps, 1), args.warmup
    # bounded sample: the oracle's writer spends ~13 us per full-precision `uniform` cell, so the sample is sized for the
    # writer (a few tens of seconds on the pool), not for the query
    n_sample = max(8, min(args.series, 2 * cores))
    n_parts = max(1, min(128, n_sample // 2))
    t0 = time.perf_counter()
    parts = oracle_written_parts(O, n_sample, n_points, n_parts, cores)
    t_build = time.perf_counter() - t0
    sids = np.arange(1, n_sample + 1, dtype=np.uint64)
    q = oracle_c3(O, parts, sids, services, cores)
    for _ in range(warmup):
        O.run_query(q)
    t = time.perf_counter()
    rows = 0
    for _ in range(steps):
        rows += O.run_query(q).rows_scanned
    dt = time.perf_counter() - t
    val = rows / dt
    q2 = oracle_c3(O, parts, sids, services, cores, per_thread_partials=True)
    O.run_query(q2)
    dt2, r2 = timed_oracle(O, q2)
    sample = (f"{n_sample} of {args.series} series x {n_points} points per step ({rows // steps} datapoints/step) in {len(parts)} parts written by "
              f"the oracle's writer in {t_build:.1f} s; C port of the reference Go path: decode on a thread pool, single-threaded merge+fold")
    cfg = {"workload": workload_text(args.series, n_points, services, 1), "n_series": args.series, "n_points": n_points, "services": services,
           "query": "sum(latency), count(latency) GROUP BY service_id, Top 100"}
    print(json.dumps({"metric": METRIC, "value": val, "unit": "datapoints/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
                      "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "n/a", "vs_baseline": None,
                      "dtype": "f64", "data": "synthetic", "impl": "reference", "config": cfg,
                      "cpu_baseline": {"value": val, "unit": "datapoints/s", "cores": cores, "kind": "port", "sample": sample,
                                       "all_core_partials_variant": {"value": r2.rows_scanned / dt2, "unit": "datapoints/s", "cores": cores,
                                                                     "sample": "same parts, one run; per-thread partial aggregates"},
                                       "c1": c1_cpu_number(O, cores)},
                      "e2e": {"value": val, "unit": "datapoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


def cpu_sample(pkg, args, cores, target_seconds, ctx, h, sid0, n_mine):
    """The oracle over the first n series of this rank's shard (a part of exactly those series from the same generator, so
    the rows are the resident part's), reference-shaped and all-core, and the GPU's answer on exactly that sample."""
    from oracle import oracle as O
    n_points, services = args.points, args.services
    probe_n = max(1, min(n_mine, 16))
    img = make_part(pkg, probe_n, n_points, sid0)
    part = O.Part.open({k: bytes(v) for k, v in img.files().items()})
    sids = np.arange(sid0, sid0 + probe_n, dtype=np.uint64)
    dt, r = timed_oracle(O, oracle_c3(O, [part], sids, services, cores))
    rate = r.rows_scanned / max(dt, 1e-9)
    n_sample = int(max(probe_n, min(n_mine, target_seconds * rate / n_points)))
    if n_sample != probe_n:
        img = make_part(pkg, n_sample, n_points, sid0)
        part = O.Part.open({k: bytes(v) for k, v in img.files().items()})
        sids = np.arange(sid0, sid0 + n_sample, dtype=np.uint64)
    del img
    dt, r = timed_oracle(O, oracle_c3(O, [part], sids, services, cores))
    out = {"value": r.rows_scanned / dt, "unit": "datapoints/s", "cores": cores, "kind": "port",
           "sample": f"the first {n_sample} of {args.series} series x {n_points} points ({r.rows_scanned} datapoints, {dt:.1f} s), same query; "
                     "C port of the reference Go path: decode on a thread pool, single-threaded merge+fold"}
    dt2, r2 = timed_oracle(O, oracle_c3(O, [part], sids, services, cores, per_thread_partials=True))
    out["all_core_partials_variant"] = {"value": r2.rows_scanned / dt2, "unit": "datapoints/s", "cores": cores,
                                        "sample": f"same sample, {dt2:.1f} s; per-thread partial aggregates (optimistic: not how the reference folds)"}
    g = ctx.scan_agg(c3_query(pkg, [h], sids, services))
    same_rows = g.group_id.tolist() == r.group_id.tolist() and g.rows.tolist() == r.rows.tolist()
    same_cnt = g.val_i64[:, 1].tolist() == r.val_i64[:, 1].tolist()
    rel = float(np.max(np.abs(g.val_f64[:, 0] - r.val_f64[:, 0]) / np.maximum(np.abs(r.val_f64[:, 0]), 1e-300))) if same_rows and len(r.rows) else None
    out["agrees_with_gpu"] = bool(same_rows and same_cnt and rel is not None and rel <= 1e-9)
    out["agreement"] = {"top100_groups_and_order_equal": bool(same_rows), "counts_bit_equal": bool(same_cnt), "max_rel_err_of_sums": rel, "tolerance": 1e-9}
    try:
        out["c1"] = c1_cpu_number(O, cores)
    except Exception as ex:  # noqa: BLE001
        out["c1"] = {"error": str(ex)[:120]}
    return out


# ------------------------------------------------------------------------------------------------ main
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_series, n_points, services = args.series, args.points, args.services
    cores = os.cpu_count() or 1
    cfg = {"workload": workload_text(n_series, n_points, services, world), "n_series": n_series, "n_points": n_points, "services": services,
           "query": "sum(latency), count(latency) GROUP BY service_id, Top 100",
           "timing": "inputs larger than L2 (no flush needed): the encoded latency pages of one step are ~1.9 GB per 1e9 datapoints vs 126 MB L2"}

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, cores)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the measure scan path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = load_pkg()
    ctx = pkg.Context(device=local_rank)
    # strong scaling: rank r owns the contiguous series range [lo, hi) of the ONE workload
    lo, hi = rank * n_series // world, (rank + 1) * n_series // world
    n_mine, sid0 = hi - lo, 1 + lo
    t0 = time.perf_counter()
    img = make_part(pkg, n_mine, n_points, sid0)
    t_gen = time.perf_counter() - t0
    files = img.files()
    t0 = time.perf_counter()
    h = ctx.register_part(1 + rank, files)
    admission = {"generate_s": t_gen, "register_ms": (time.perf_counter() - t0) * 1e3, **ctx.part_info(h), "file_bytes": int(sum(v.size for v in files.values())),
                 "note": "one-time per part: upload to HBM, block-index parse, device unpack of the fallback pages (the `uniform` field is "
                         "full-precision float64 = zstd-compressed EncodeTypePlain pages)"}
    sids = np.arange(sid0, sid0 + n_mine, dtype=np.uint64)   # a rank resolves the series of its own shard (a data node's index lookup)
    q = c3_query(pkg, [h], sids, services)
    pq = ctx.prepare(q)   # marshalled to the C struct once, like a cgo caller would hold it

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    stats_acc = []
    phase = {"scan_enqueue": 0.0, "all_gather_enqueue": 0.0, "combine_finalize_sync": 0.0}
    if world == 1:
        def step(want_stats=True):
            r = ctx.scan_agg(pq)
            stats_acc.append(r.stats)
            return r
    else:
        # the reduce lives behind the C ABI: peer mailboxes over NVLink (bydb_comm_*).  torch.distributed only carries the
        # 128-byte mailbox handles once, at set-up -- it is not on the data path
        lay = ctx.partials_layout(q)
        mine_h = torch.frombuffer(bytearray(ctx.comm_export(int(lay["total_bytes"]), world)), dtype=torch.uint8).cuda()
        all_h = torch.empty(world * 128, dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(all_h, mine_h)
        raw = bytes(all_h.cpu().numpy().tobytes())
        ctx.comm_connect(rank, world, [raw[i * 128:(i + 1) * 128] for i in range(world)])

        def step(want_stats=True):
            # ONE collective call per rank: scan -> the partial table lands in rank 0's mailbox (P2P stores) -> rank 0 waits for
            # the arrival flags on the device, combines in rank order, finalises MEAN / Top-N and reads the rows back
            r = ctx.scan_reduce(pq, root=0)
            stats_acc.append(r.stats)
            return r if rank == 0 else None

    if world > 1:
        words = lay["total_bytes"] // 8
        table = torch.zeros(words, dtype=torch.float64, device="cuda")
        gathered = torch.zeros(world * words, dtype=torch.float64, device="cuda")
        stream = torch.cuda.current_stream().cuda_stream

        def nccl_step(want_stats=False):
            # the library-collective variant, measured beside the mailbox reduce: every rank scans its shard into a partial table
            # on its GPU (asynchronous), ONE NCCL all-gather ships the tables, rank 0 combines in rank order and finalises
            ta = time.perf_counter()
            ctx.scan_partials(pq, table.data_ptr(), lay["total_bytes"], stream, want_stats=False)
            tb = time.perf_counter()
            dist.all_gather_into_tensor(gathered, table)
            tc = time.perf_counter()
            res = None
            if rank == 0:
                ctx.partials_combine(pq, gathered.data_ptr(), world, lay["total_bytes"], stream)
                res = ctx.reduce_finalize(pq, gathered.data_ptr(), lay["total_bytes"], stream)
            else:
                torch.cuda.current_stream().synchronize()
            td = time.perf_counter()
            phase["scan_enqueue"] += tb - ta
            phase["all_gather_enqueue"] += tc - tb
            phase["combine_finalize_sync"] += td - tc
            return res

    if world > 1:
        from importlib import import_module
        multi = import_module("bydb_b200.multi")

        def allreduce_step():
            # north_star's literal form: the partial table all-reduced in place over NVLink (SUM / MAX over its four typed ranges,
            # skywalking-banyandb_b200/multi.py), finalised on rank 0.  Float sums then depend on NCCL's reduction order.
            ctx.scan_partials(pq, table.data_ptr(), lay["total_bytes"], stream, want_stats=False)
            multi.allreduce_partial_table(table, lay, dist)
            if rank == 0:
                return ctx.reduce_finalize(pq, table.data_ptr(), lay["total_bytes"], stream)
            torch.cuda.current_stream().synchronize()
            return None

    def timed(fn, steps):
        barrier()
        t = time.perf_counter()
        last = None
        for _ in range(steps):
            last = fn()
        barrier()
        d = time.perf_counter() - t
        if world > 1:
            m = torch.tensor([d], dtype=torch.float64, device="cuda")
            dist.all_reduce(m, op=dist.ReduceOp.MAX)
            d = float(m[0])
        return d, last

    warm = max(args.warmup, 3)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- (1) the plain calls (bydb_scan_agg / bydb_scan_reduce): they carry the per-kernel CUDA-event times the roofline uses
    for _ in range(warm):
        step()
    stats_acc.clear()
    d_plain, last_plain = timed(step, args.steps)
    # ---- (2) the timed region of `value`: the same query as a PREPARED query (bydb_query_prepare + bydb_scan_agg_prepared /
    #      bydb_scan_reduce_prepared -- what a cgo caller holds for a dashboard or alert-rule query): the whole step, on every rank,
    #      is one captured CUDA graph -- one launch + one synchronisation per call, every execution scans all the data again
    graph_note = None
    try:
        gq = ctx.prepare_graph(q)

        def gstep():
            r = gq.run() if world == 1 else gq.run_reduce(root=0)
            return r if rank == 0 else None
        for _ in range(warm + 2):
            gstep()
        dt, last = timed(gstep, args.steps)
        same = None
        if rank == 0 and last is not None and last_plain is not None:
            same = bool(last.group_id.tolist() == last_plain.group_id.tolist() and last.val_i64.tolist() == last_plain.val_i64.tolist()
                        and last.val_f64.tolist() == last_plain.val_f64.tolist())
        graph_note = {"api": "bydb_scan_agg_prepared" if world == 1 else "bydb_scan_reduce_prepared", "same_result_as_plain_call": same}
        timed_step = gstep
    except Exception as ex:  # noqa: BLE001 -- keep the bench line alive: the plain call is then the timed one
        graph_note = {"error": str(ex)[:200]}
        dt, last, timed_step = d_plain, last_plain, step
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    kernel_timing = "cuda events inside the plain calls of the same step (a graph replay has no per-kernel events); value is timed on the prepared-query path"
    rows_step = stats_acc[-1].rows_scanned
    scan_ms = float(np.mean([s.scan_kernel_ms for s in stats_acc]))
    dev_ms = float(np.mean([s.device_ms for s in stats_acc]))
    launches = int(sum(s.kernel_launches for s in stats_acc[:args.steps]))
    page_bytes = stats_acc[-1].page_bytes
    slow_blocks, slow_why = int(stats_acc[-1].blocks_slow_lane), int(stats_acc[-1].slow_lane_reasons)
    total_rows_step = float(rows_step)
    scan_ms_max = scan_ms
    if world > 1:
        sm = torch.tensor([float(rows_step)], dtype=torch.float64, device="cuda")
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        total_rows_step = float(sm[0])
        mx = torch.tensor([scan_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        scan_ms_max = float(mx[0])
    value = total_rows_step * args.steps / dt

    extra = {}
    if not args.no_extra:
        # a long resident region (the timed K steps above last only tens of ms: too short for the 100 ms clock sampler alone)
        ns = max(args.sustained_steps, args.steps)
        d2, _ = timed(timed_step, ns)
        extra["sustained"] = {"steps": ns, "ms_per_step": d2 / ns * 1e3, "value": total_rows_step * ns / d2, "unit": "datapoints/s"}
        stats_acc[:] = stats_acc[:args.steps]
        if world > 1:
            for _ in range(warm):
                nccl_step()
            for k in phase:
                phase[k] = 0.0
            dn, _ = timed(nccl_step, args.steps)
            extra["nccl_allgather_variant"] = {"steps": args.steps, "ms_per_step": dn / args.steps * 1e3, "value": total_rows_step * args.steps / dn, "unit": "datapoints/s",
                                               "host_phase_ms_per_step_rank0": {k: v / args.steps * 1e3 for k, v in phase.items()},
                                               "note": "bydb_scan_partials (asynchronous) -> one NCCL all-gather of the partial tables -> bydb_partials_combine + "
                                                       "bydb_reduce_finalize on rank 0"}
        if world > 1:
            for _ in range(warm):
                allreduce_step()
            da, ra = timed(allreduce_step, args.steps)
            extra["nccl_allreduce_variant"] = {"steps": args.steps, "ms_per_step": da / args.steps * 1e3, "value": total_rows_step * args.steps / da, "unit": "datapoints/s",
                                               "same_top100_groups": bool(ra.group_id.tolist() == last.group_id.tolist()) if rank == 0 and ra is not None and last is not None else None,
                                               "note": "bydb_scan_partials -> NCCL all-reduce of the table in place (4 typed ranges) -> bydb_reduce_finalize on rank 0"}
        if world == 1:
            # second leg: BASELINE configs[1]'s query over the same part
            q2 = ctx.prepare(c2_query(pkg, [h], sids, n_points))
            for _ in range(3):
                r2 = ctx.scan_agg(q2)
            n2 = max(5, args.steps)
            acc2 = []

            def step2():
                r = ctx.scan_agg(q2)
                acc2.append(r.stats)
                return r
            d2q, r2 = timed(step2, n2)
            s2 = float(np.mean([s.scan_kernel_ms for s in acc2]))
            extra["c2_query"] = {"query": "time range (middle 50%) AND region==\"r3\", avg(latency)+max(walk), scalar", "ms_per_step": d2q / n2 * 1e3,
                                 "datapoints_per_step": int(r2.stats.rows_scanned), "value": r2.stats.rows_scanned * n2 / d2q, "unit": "datapoints/s",
                                 "scan_kernel_ms": s2, "algorithmic_bytes_per_datapoint": B_ALG_C2,
                                 "achieved_GBps": r2.stats.rows_scanned * B_ALG_C2 / (s2 * 1e-3) / 1e9, "encoded_page_bytes": int(r2.stats.page_bytes),
                                 "rows_matched": int(r2.rows[0]), "mean_latency": float(r2.val_f64[0, 0]), "max_walk": float(r2.val_f64[0, 1]),
                                 "blocks_slow_lane": int(r2.stats.blocks_slow_lane)}
            # third leg: group-by on a STORED tag (a12): sum + count of latency per value of default/region (8 values) -- one
            # scan pass per value behind bydb_scan_agg_keyed
            qk = pkg.Query(parts=[h], series_ids=sids, aggs=[("latency", pkg.AGG_SUM), ("latency", pkg.AGG_COUNT)])
            try:
                rk = ctx.scan_agg_keyed(qk, "default", "region")
                nk = 3
                dk, rk = timed(lambda: ctx.scan_agg_keyed(qk, "default", "region"), nk)
            except Exception as ex:  # noqa: BLE001 -- a side leg must never cost the headline line
                rk = None
                extra["stored_tag_group_by"] = {"error": str(ex)[:200]}
            if rk is not None:
                extra["stored_tag_group_by"] = {"query": "sum(latency), count(latency) GROUP BY region (a stored tag, 8 values)", "api": "bydb_scan_agg_keyed",
                                            "ms_per_step": dk / nk * 1e3, "datapoints_per_step": int(rows_step), "value": rows_step * nk / dk,
                                            "unit": "datapoints/s", "groups": [k.decode() for k in rk.key],
                                            "rows_per_group": [int(x) for x in rk.rows], "all_rows_accounted": bool(int(rk.rows.sum()) == int(rows_step)),
                                            "kernel_launches": int(rk.stats.kernel_launches)}

    # ------------------------------------------------------------------ end to end: host buffers in, result out
    e2e = None
    if not args.no_e2e:
        from bydb_b200.capi import Q_HOST_ZERO_COPY
        t0 = time.perf_counter()
        pinned, keep_pinned = {}, []
        for k, v in files.items():
            tns = torch.empty(v.size + 256, dtype=torch.uint8, pin_memory=True)   # 256 B of readable slack after each image
            tns[:v.size].copy_(torch.from_numpy(np.ascontiguousarray(v)))
            keep_pinned.append(tns)
            pinned[k] = tns[:v.size].numpy()
        t_pin = time.perf_counter() - t0

        def e2e_leg(flags, steps, bufs):
            qh = c3_query(pkg, [], sids, services, flags=flags)
            st = [None]

            def one():
                r = ctx.scan_agg_host([bufs], qh) if world == 1 else ctx.scan_reduce_host([bufs], qh, root=0)
                st[0] = r.stats
                return r if rank == 0 else None
            one()
            d, r = timed(one, steps)
            s = st[0]
            hb = torch.tensor([float(s.h2d_bytes), float(s.d2h_bytes)], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(hb, op=dist.ReduceOp.SUM)
            return {"value": total_rows_step * steps / d, "unit": "datapoints/s", "h2d_bytes_per_step": int(hb[0]), "d2h_bytes_per_step": int(hb[1]),
                    "ms_per_step": d / steps * 1e3, "steps": steps, "scan_kernel_ms": s.scan_kernel_ms, "device_ms": s.device_ms}, r

        e2e_steps = max(3, min(args.steps, 5))
        e2e, r_e2e = e2e_leg(Q_HOST_ZERO_COPY, e2e_steps, pinned)
        e2e["pinned_by_caller"] = True
        e2e["note"] = ("bydb_scan_agg_host(BYDB_Q_HOST_ZERO_COPY): the part's file images stay in the caller's pinned host memory; every step parses "
                       "the block index, uploads the block directory and the kernels pull exactly the pages the query touches over PCIe "
                       "(h2d = directory + page bytes), result copied back"
                       + ("; bydb_scan_reduce_host on every rank: host images in on all ranks, the partial tables meet in rank 0's mailbox, one "
                          "result out on rank 0 -- the collective is inside the timed call" if world > 1 else ""))
        e2e["pin_copy_s_outside_timed_region"] = t_pin
        if world == 1:
            # one more, untimed, step with the library's host-side timeline (BYDB_TRACE) captured from stderr: shows whether a slow
            # step waited for the block-index parsers (host cores) or for the copies (PCIe)
            import tempfile
            try:
                with tempfile.TemporaryFile() as tf:
                    sys.stderr.flush()
                    saved = os.dup(2)
                    os.dup2(tf.fileno(), 2)
                    os.environ["BYDB_TRACE"] = "1"
                    try:
                        t1 = time.perf_counter()
                        ctx.scan_agg_host([pinned], c3_query(pkg, [], sids, services, flags=Q_HOST_ZERO_COPY))
                        traced_ms = (time.perf_counter() - t1) * 1e3
                    finally:
                        os.environ.pop("BYDB_TRACE", None)
                        os.dup2(saved, 2)
                        os.close(saved)
                    tf.seek(0)
                    lines = [ln.strip() for ln in tf.read().decode(errors="replace").splitlines() if "[bydb cold]" in ln]
                e2e["traced_step"] = {"ms": traced_ms, "timeline": lines[:40]}
            except Exception as ex:  # noqa: BLE001
                e2e["traced_step"] = {"error": str(ex)[:200]}
        if last is not None and r_e2e is not None:
            # the cold path scans in slices and combines their tables: float sums may differ from the resident run in the last bits
            e2e["same_result_as_resident"] = bool(r_e2e.group_id.tolist() == last.group_id.tolist() and r_e2e.val_i64.tolist() == last.val_i64.tolist()
                                                  and np.allclose(r_e2e.val_f64, last.val_f64, rtol=1e-12, atol=0))
        try:
            if world > 1:
                raise RuntimeError("single-GPU leg")
            staged, _ = e2e_leg(0, 3, files)
            staged["pinned_by_caller"] = False
            staged["note"] = ("bydb_scan_agg_host on PAGEABLE images (not pinned by the caller, like BanyanDB's mmap'd part files): the block index "
                              "is parsed, the host selects the blocks and gathers only the pages the query reads into a pinned staging ring "
                              "(64 MB chunks, worker pool), asynchronous copies, scan, result copied back")
            e2e["unpinned_gather"] = staged
        except Exception as ex:  # noqa: BLE001
            e2e["unpinned_gather"] = {"error": str(ex)[:200]}
        del pinned, keep_pinned

    clocks = None
    if rank == 0:
        clocks = sampler.stop()
        clocks["window"] = "resident timed steps + sustained / graph / C2 legs + e2e legs (100 ms sampling)"
    cpu = None
    if world == 1 and not args.no_cpu:
        cpu = cpu_sample(pkg, args, cores, args.cpu_seconds, ctx, h, sid0, n_mine)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = rows_step * B_ALG_C3 / (scan_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "scan_sum_express_kernel (timed with the two empty lanes launched behind it, ~6 us)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                "algorithmic_bytes_per_datapoint": B_ALG_C3, "algorithmic_bytes_per_launch": int(rows_step * B_ALG_C3), "kernel_ms": scan_ms,
                "kernel_ms_max_over_ranks": scan_ms_max, "encoded_page_bytes_per_launch": int(page_bytes),
                "encoded_GBps": page_bytes / (scan_ms * 1e-3) / 1e9, "frac_encoded": page_bytes / (scan_ms * 1e-3) / 1e9 / peak,
                "traffic": traffic_from_profile() if world == 1 else None, "kernel_timing": kernel_timing,
                "reading": "frac counts SURVEY 8(d)'s 8 decoded bytes per datapoint; the pages hold ~1.9 encoded bytes per datapoint, so frac can "
                           "pass 1 while DRAM runs at frac_encoded of the copy peak: the kernel is bound by the ALU pipe (ncu: 74 % busy), not by HBM",
                "note": "per launch on rank 0's shard" if world > 1 else "per launch"}
    out = {"metric": METRIC, "value": value, "unit": "datapoints/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
           "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong" if world > 1 else "n/a", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic", "config": cfg, "datapoints_per_step": total_rows_step, "device_ms_per_step": dev_ms,
           "scan_kernel_ms": scan_ms, "blocks_slow_lane": slow_blocks, "slow_lane_reasons": slow_why, "roofline": roofline, "clocks": clocks,
           "gpu_launches": launches, "e2e": e2e, "part_admission": admission}
    out["prepared_query"] = graph_note
    out["plain_call"] = {"api": "bydb_scan_agg" if world == 1 else "bydb_scan_reduce", "ms_per_step": d_plain / args.steps * 1e3,
                         "value": total_rows_step * args.steps / d_plain, "unit": "datapoints/s",
                         "note": "the same step through the unprepared call: ~25 runtime calls and the launch gaps between the small kernels every step"}
    out.update(extra)
    if world > 1:
        out["reduce"] = "bydb_scan_reduce: peer mailboxes over NVLink behind the C ABI (no library collective on the data path)"
    if last is not None:
        out["result"] = {"rows": int(last.group_id.size), "top3": [[int(g), float(s), int(c)] for g, s, c in zip(last.group_id[:3], last.val_f64[:3, 0], last.val_i64[:3, 1])],
                         "top_sorted_desc": bool((np.diff(last.val_f64[:, 0]) <= 0).all()), "total_count_top100": int(last.val_i64[:, 1].sum())}
    if cpu is not None:
        out["cpu_baseline"] = cpu
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
