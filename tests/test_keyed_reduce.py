"""bydb_scan_reduce_keyed: group-by on a stored tag as a collective over the peer mailboxes.  The root must return exactly what
bydb_scan_agg_keyed returns when one context scans every rank's parts and series (rows, order, key bytes, series groups, int64
values; float sums within 1e-12 relative), for several shardings of one measure, and every failure must leave the mailboxes
usable."""
import ctypes
import os
import shutil
import subprocess
import threading

import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import STEP, T0, assert_parity, build_part, grid, to_gpu_query

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 3
_pid = [70_000]


def _next_pid():
    _pid[0] += 100
    return _pid[0]


# ------------------------------------------------------------------ host only
def test_keyed_ranks_program_compiles_and_links(tmp_path, bydb):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    lib_dir = os.path.dirname(bydb.library_path())
    subprocess.check_call(["gcc", "-std=c99", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(tmp_path / "keyed_ranks"),
                           os.path.join(ROOT, "tests", "native", "keyed_ranks.c"), "-L", lib_dir, "-lbydbgpu", "-lm", "-Wl,-rpath," + lib_dir])


def test_keyed_collective_symbols_are_exported(bydb):
    lib = ctypes.CDLL(bydb.library_path())
    for name in ("bydb_keyed_reduce_layout", "bydb_scan_reduce_keyed"):
        assert hasattr(lib, name) and name in bydb.capi.EXPORTS


def _table_bytes(bydb, n_groups, aggs):
    q = bydb.Query(parts=[], series_ids=[], aggs=aggs, series_group=[], n_groups=n_groups)
    keep = []
    cq = bydb.capi._mk_query(q, keep)
    lay = bydb.capi._Layout()
    assert bydb.load_library().bydb_partials_layout(ctypes.byref(cq), ctypes.byref(lay)) == 0
    return lay.total_bytes


def test_keyed_reduce_layout_covers_table_dictionary_and_first_appearances(bydb):
    aggs = [("latency", O.AGG_SUM), ("calls", O.AGG_MAX), ("latency", O.AGG_COUNT)]   # two distinct fields
    for G in (1, 7, 1000):
        for max_values, cap in ((0, 64), (1, 1), (8, 8), (256, 256)):
            q = bydb.Query(parts=[], series_ids=[], aggs=aggs, series_group=[], n_groups=G)
            slot = bydb.capi.keyed_reduce_layout(q, "default", "region", max_values)
            need = _table_bytes(bydb, cap * G, aggs) + cap * (4 + 64) + cap * G * (8 + 8 + 4)
            assert slot >= need, (G, cap, slot, need)
    one = bydb.capi.keyed_reduce_layout(bydb.Query(parts=[], series_ids=[], aggs=aggs), "default", "region", 8)
    assert one >= _table_bytes(bydb, 8, aggs) + 8 * (4 + 64 + 20)
    with pytest.raises(bydb.BydbError) as e:
        bydb.capi.keyed_reduce_layout(bydb.Query(parts=[], series_ids=[], aggs=aggs), "default", "region", 257)
    assert e.value.code == bydb.capi.EINVAL


# ------------------------------------------------------------------ on the device
def _collective(fns):
    """Runs fns[r]() on one thread per rank; -> (results, error codes).  Non-BydbError exceptions fail the test."""
    got, codes, other = [None] * len(fns), [0] * len(fns), []

    def run(r):
        try:
            got[r] = fns[r]()
        except Exception as e:  # noqa: BLE001
            if hasattr(e, "code"):
                codes[r] = e.code
            else:
                other.append(repr(e))
    th = [threading.Thread(target=run, args=(r,)) for r in range(len(fns))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not other, other
    return got, codes


def _contexts(bydb, n_dev, table_bytes):
    ctxs = [bydb.Context(device=r % n_dev) for r in range(R)]
    handles = [c.comm_export(table_bytes, R) for c in ctxs]
    for r, c in enumerate(ctxs):
        c.comm_connect(r, R, handles)
    return ctxs


def _guarded(body):
    # The threaded collectives share the device on a one-GPU box: a finaliser of an unrelated object that runs on a rank's thread in
    # the middle of a collective frees page-locked memory -- an implicit device synchronisation that can wait on a peer.  No garbage
    # collection while they run; a stalled collective dumps every thread's stack.
    import faulthandler
    import gc
    gc.collect()
    gc.disable()
    faulthandler.dump_traceback_later(60, exit=False)
    try:
        body()
    finally:
        faulthandler.cancel_dump_traceback_later()
        gc.enable()


def _measure(rng, n_series=24, n_pts=4000):
    sids, ts, ver = grid(n_series, n_pts, sid0=5, sid_step=3)
    n = sids.size
    lat = np.round(30 + rng.normal(0, 6, n), 2)
    calls = rng.integers(-3000, 3000, n)
    code = rng.integers(0, 4, n) * 100
    region = []
    while len(region) < n:
        region.extend([b"region-%d" % int(rng.integers(0, 6))] * int(rng.integers(1, 50)))
    region = region[:n]
    for i in range(3, n, 911):
        region[i] = None          # nil and "" are one key
    for i in range(7, n, 1303):
        region[i] = b""
    for s in range(n_series):     # a value that only shows late in time, in every series
        region[s * n_pts + n_pts - 300: s * n_pts + n_pts - 290] = [b"late"] * 10
    for s in (20, 23):            # a value only these series have: in every sharding below, one rank holds it
        region[s * n_pts + 100: s * n_pts + 140] = [b"solo"] * 40
    return sids, ts, ver, lat, calls, code, region


def _part(sids, ts, ver, lat, calls, code, region, m):
    return build_part(sids[m], ts[m], ver[m], [("latency", O.VT_FLOAT64, lat[m], None), ("calls", O.VT_INT64, calls[m], None)],
                      [("default", [("region", O.VT_STR, [x for x, k in zip(region, m) if k], None), ("code", O.VT_INT64, code[m], None)])])


ALL5 = [("latency", O.AGG_SUM), ("latency", O.AGG_MAX), ("calls", O.AGG_MIN), ("calls", O.AGG_COUNT), ("latency", O.AGG_MEAN), ("calls", O.AGG_SUM)]


def _queries():
    return [
        dict(aggs=ALL5, grouped=True, preds=[O.Pred("default", "code", O.OP_NE, 300)], tmin=T0 + 150 * STEP, tmax=T0 + 3900 * STEP),
        dict(aggs=[("calls", O.AGG_SUM), ("calls", O.AGG_COUNT)], grouped=False),
        dict(aggs=[("calls", O.AGG_COUNT), ("latency", O.AGG_MAX)], grouped=True, top_n=6, top_agg=0, top_desc=True,
             tmin=T0 + 1000 * STEP, tmax=T0 + 1012 * STEP),   # few rows per composite group: COUNT ties
        dict(aggs=[("calls", O.AGG_COUNT), ("latency", O.AGG_MAX)], grouped=True, top_n=6, top_agg=0, top_desc=False,
             tmin=T0 + 1000 * STEP, tmax=T0 + 1012 * STEP),
    ]


def _assert_same(got, want, aggs, ctx):
    assert got.key == want.key, f"{ctx}: keys {got.key} vs {want.key}"
    assert got.group_id.tolist() == want.group_id.tolist() and got.rows.tolist() == want.rows.tolist(), ctx
    assert got.is_float.tolist() == want.is_float.tolist(), ctx
    assert got.val_i64.tolist() == want.val_i64.tolist(), ctx
    for a, (_, func) in enumerate(aggs):
        if want.is_float[a] and func in (O.AGG_MIN, O.AGG_MAX):
            assert got.val_f64[:, a].view(np.uint64).tolist() == want.val_f64[:, a].view(np.uint64).tolist(), ctx
    assert np.allclose(got.val_f64, want.val_f64, rtol=1e-12, atol=0), ctx


def _run_keyed(ctxs, qs, tag, root, max_values=0):
    return _collective([lambda r=r: ctxs[r].scan_reduce_keyed(qs[r], "default", tag, root=root, max_values=max_values) for r in range(R)])


@pytest.mark.gpu
def test_keyed_reduce_equals_one_context_over_every_shard(bydb, gpu_ctx):
    import torch
    n_dev = max(1, torch.cuda.device_count())
    _guarded(lambda: _parity_body(bydb, gpu_ctx, n_dev))


def _parity_body(bydb, gpu_ctx, n_dev):
    import dataclasses
    rng = np.random.default_rng(0x5EED)
    sids, ts, ver, lat, calls, code, region = _measure(rng)
    usid = np.unique(sids)
    groups = (np.arange(usid.size) % 3).astype(np.int32)
    full = _part(sids, ts, ver, lat, calls, code, region, np.ones(sids.size, bool))
    half = ts < T0 + 2000 * STEP
    early, late = (_part(sids, ts, ver, lat, calls, code, region, m) for m in (half, ~half))
    idx = np.arange(usid.size)
    # sharding -> (per rank: (part mask or None, the rank's query series mask)); every rank's query names only its own series
    shardings = {
        "contiguous": [(np.isin(sids, usid[(idx * R) // usid.size == r]), (idx * R) // usid.size == r) for r in range(R)],
        "interleaved": [(np.isin(sids, usid[idx % R == r]), idx % R == r) for r in range(R)],
        # every series: first half on rank 0, second half on rank 1; rank 2 holds a part but its shard selects no block
        "time split": [("early", np.ones(usid.size, bool)), ("late", np.ones(usid.size, bool)), ("early", np.zeros(usid.size, bool))],
    }
    whole = {"full": [gpu_ctx.register_part(_next_pid(), full.files())]}
    whole["split"] = [gpu_ctx.register_part(_next_pid(), p.files()) for p in (early, late)]
    probe = bydb.Query(parts=[], series_ids=[], aggs=ALL5, series_group=[], n_groups=3)
    ctxs = _contexts(bydb, n_dev, bydb.capi.keyed_reduce_layout(probe, "default", "region"))
    try:
        for name, shard in shardings.items():
            hs = []
            for r, (pm, _) in enumerate(shard):
                p = {"early": early, "late": late}[pm] if isinstance(pm, str) else _part(sids, ts, ver, lat, calls, code, region, pm)
                hs.append(ctxs[r].register_part(_next_pid(), p.files()))
            opart = [early, late] if name == "time split" else [full]
            wparts = whole["split"] if name == "time split" else whole["full"]
            for kw in _queries():
                kw = dict(kw)
                aggs, grouped = kw.pop("aggs"), kw.pop("grouped")
                preds = kw.pop("preds", [])
                g_all = groups if grouped else None
                oq = O.Query(opart, usid, aggs, groups=g_all, n_groups=3 if grouped else 1, preds=preds, **kw)
                for tag in ("region", "nosuchtag"):
                    want = gpu_ctx.scan_agg_keyed(to_gpu_query(bydb, wparts, oq), "default", tag)
                    oracle = O.run_query(dataclasses.replace(oq, group_key=("default", tag)))
                    assert want.key == oracle.key
                    assert_parity(want, oracle, aggs, f"{name}: single context vs oracle")
                    if tag == "nosuchtag":
                        assert set(want.key) <= {b""} and want.n_keys == 1
                    qs = [bydb.Query(parts=[hs[r]], series_ids=usid[m], aggs=aggs, series_group=groups[m] if grouped else None,
                                     n_groups=3 if grouped else 1, preds=[bydb.Pred(p.family, p.tag, p.op, p.value) for p in preds], **kw)
                          for r, (_, m) in enumerate(shard)]
                    for root in (0, 2):
                        got, codes = _run_keyed(ctxs, qs, tag, root)
                        ctx = f"{name}, {tag}, root {root}, {aggs}, {kw}"
                        assert codes == [0] * R, (ctx, codes)
                        _assert_same(got[root], want, aggs, ctx)
                        assert got[root].n_keys == want.n_keys, ctx
                        for r in range(R):
                            if r != root:
                                assert got[r].group_id.size == 0 and got[r].n_keys == 0, ctx
                                if shard[r][1].any() and "tmin" not in kw:
                                    assert got[r].stats.blocks_scanned > 0, ctx
            for r, h in enumerate(hs):
                ctxs[r].release_part(h)
        # the keyed collective and the plain one alternate on the same mailboxes
        hs = [ctxs[r].register_part(_next_pid(), _part(sids, ts, ver, lat, calls, code, region, shardings["contiguous"][r][0]).files()) for r in range(R)]
        masks = [m for _, m in shardings["contiguous"]]
        for it in range(4):
            plain, codes = _collective([lambda r=r: ctxs[r].scan_reduce(bydb.Query([hs[r]], usid[masks[r]], [("calls", O.AGG_SUM)]), root=it % R)
                                        for r in range(R)])
            assert codes == [0] * R and int(plain[it % R].val_i64[0, 0]) == int(calls.sum())
            qs = [bydb.Query([hs[r]], usid[masks[r]], [("calls", O.AGG_SUM)], series_group=groups[masks[r]], n_groups=3) for r in range(R)]
            got, codes = _run_keyed(ctxs, qs, "region", it % R)
            assert codes == [0] * R and b"solo" in got[it % R].key
            assert int(got[it % R].val_i64[:, 0].sum()) == int(calls.sum())
        for r, h in enumerate(hs):
            ctxs[r].release_part(h)
    finally:
        for c in ctxs:
            c.close()
        for hl in whole.values():
            for h in hl:
                gpu_ctx.release_part(h)


@pytest.mark.gpu
def test_keyed_reduce_failures_leave_the_mailboxes_usable(bydb, gpu_ctx):
    import torch
    n_dev = max(1, torch.cuda.device_count())
    _guarded(lambda: _failure_body(bydb, gpu_ctx, n_dev))


def _failure_body(bydb, gpu_ctx, n_dev):
    rng = np.random.default_rng(0xFA11)
    n_pts = 1500
    # rank r: 4 series whose tag "k" holds {a, b, c, x<r>}: 4 values per rank, 6 over the ranks
    data = []
    for r in range(R):
        sids, ts, ver = grid(4, n_pts, sid0=1 + 10 * r, t0=T0 + r * n_pts * STEP)   # one context over all the parts: none overlap in time
        vals = [b"a", b"b", b"c", b"x%d" % r]
        k = [vals[int(i)] for i in rng.integers(0, 4, sids.size)]
        calls = rng.integers(0, 1000, sids.size)
        data.append((sids, ts, ver, k, calls))

    def part(r, k_override=None, k_int=False):
        sids, ts, ver, k, calls = data[r]
        tag = ("k", O.VT_INT64, rng.integers(0, 5, sids.size), None) if k_int else ("k", O.VT_STR, k_override or k, None)
        return build_part(sids, ts, ver, [("calls", O.VT_INT64, calls, None)], [("default", [tag])])
    total = int(sum(int(d[4].sum()) for d in data))
    good = [part(r) for r in range(R)]
    probe = bydb.Query(parts=[], series_ids=[], aggs=[("calls", O.AGG_SUM)])
    ctxs = _contexts(bydb, n_dev, bydb.capi.keyed_reduce_layout(probe, "default", "k", 256))
    whole = [gpu_ctx.register_part(_next_pid(), p.files()) for p in good]

    def queries(handles):
        return [bydb.Query([handles[r]], np.unique(data[r][0]), [("calls", O.AGG_SUM), ("calls", O.AGG_COUNT)]) for r in range(R)]

    def still_usable(hs, root):
        plain, codes = _collective([lambda r=r: ctxs[r].scan_reduce(bydb.Query([hs[r]], np.unique(data[r][0]), [("calls", O.AGG_SUM)]), root=root)
                                    for r in range(R)])
        assert codes == [0] * R and int(plain[root].val_i64[0, 0]) == total
        got, codes = _run_keyed(ctxs, queries(hs), "k", root)
        want = gpu_ctx.scan_agg_keyed(bydb.Query(whole, np.unique(np.concatenate([d[0] for d in data])), [("calls", O.AGG_SUM), ("calls", O.AGG_COUNT)]),
                                      "default", "k")
        assert codes == [0] * R
        _assert_same(got[root], want, [("calls", O.AGG_SUM), ("calls", O.AGG_COUNT)], f"after a failure, root {root}")
    try:
        hs = [ctxs[r].register_part(_next_pid(), p.files()) for r, p in enumerate(good)]
        still_usable(hs, 0)
        # the union over the ranks exceeds max_values while every rank is within it
        _, codes = _run_keyed(ctxs, queries(hs), "k", 1, max_values=4)
        assert codes == [0, bydb.capi.ENOMEM, 0], codes
        still_usable(hs, 1)
        # one rank stores the key tag as int64: EINVAL there and at the root
        bad = list(hs)
        bad[1] = ctxs[1].register_part(_next_pid(), part(1, k_int=True).files())
        _, codes = _run_keyed(ctxs, queries(bad), "k", 0)
        assert codes == [bydb.capi.EINVAL, bydb.capi.EINVAL, 0], codes
        ctxs[1].release_part(bad[1])
        still_usable(hs, 2)
        # one rank's key block falls back to the plain bytes block (> 256 distinct values): ENOTSUP there and at the root
        bad = list(hs)
        many = [b"v%d" % (i % 400) for i in range(data[2][0].size)]
        bad[2] = ctxs[2].register_part(_next_pid(), part(2, k_override=many).files())
        _, codes = _run_keyed(ctxs, queries(bad), "k", 0, max_values=256)
        assert codes == [bydb.capi.ENOTSUP, 0, bydb.capi.ENOTSUP], codes
        ctxs[2].release_part(bad[2])
        still_usable(hs, 0)
        for r, h in enumerate(hs):
            ctxs[r].release_part(h)
    finally:
        for c in ctxs:
            c.close()
    # a mailbox exported too small for the keyed table: EINVAL on every rank, then a fitting keyed query and a plain one succeed
    small = bydb.capi.keyed_reduce_layout(probe, "default", "k", 8)
    ctxs = _contexts(bydb, n_dev, small)
    try:
        hs = [ctxs[r].register_part(_next_pid(), p.files()) for r, p in enumerate(good)]
        _, codes = _run_keyed(ctxs, queries(hs), "k", 2, max_values=64)
        assert codes == [bydb.capi.EINVAL] * R, codes
        plain, codes = _collective([lambda r=r: ctxs[r].scan_reduce(bydb.Query([hs[r]], np.unique(data[r][0]), [("calls", O.AGG_SUM)]), root=2)
                                    for r in range(R)])
        assert codes == [0] * R and int(plain[2].val_i64[0, 0]) == total
        got, codes = _run_keyed(ctxs, queries(hs), "k", 2, max_values=8)
        assert codes == [0] * R and sorted(got[2].key) == [b"a", b"b", b"c", b"x0", b"x1", b"x2"]
        for r, h in enumerate(hs):
            ctxs[r].release_part(h)
    finally:
        for c in ctxs:
            c.close()
        for h in whole:
            gpu_ctx.release_part(h)


@pytest.mark.gpu
def test_keyed_reduce_one_process_per_rank(tmp_path, bydb):
    """tests/native/keyed_ranks.c: one process per rank, handles over a pipe, bydb_scan_reduce_keyed with rotating roots (the
    cudaIpcOpenMemHandle path that threads of one process never take), checked against one context scanning all shards."""
    import torch
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    lib_dir = os.path.dirname(bydb.library_path())
    exe = tmp_path / "keyed_ranks"
    subprocess.check_call(["gcc", "-std=c99", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe),
                           os.path.join(ROOT, "tests", "native", "keyed_ranks.c"), "-L", lib_dir, "-lbydbgpu", "-lm", "-Wl,-rpath," + lib_dir])
    ndev = max(1, torch.cuda.device_count())
    for nranks in sorted({2, min(4, max(2, ndev))}):
        out = subprocess.run([str(exe), str(nranks), str(ndev)], capture_output=True, text=True, timeout=300)
        assert out.returncode == 0 and out.stdout.startswith("OK"), out.stdout + out.stderr
