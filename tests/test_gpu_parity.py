"""-m gpu: parity of the CUDA path (through the C ABI) against the oracle on the same seeded inputs.
Bar: bit-exact for int64 count/min/max/sum and float64 min/max; <= 1e-9 relative for float64 sum/mean."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import (E2E_CASES, QUERY_TEST_AGGS, QUERY_TEST_CASES, STEP, T0, assert_parity, build_part, check_e2e_rows,
                           check_query_test_case, grid, load_e2e_case, query_test_fixture, run_both)

pytestmark = pytest.mark.gpu

ALL5 = [O.AGG_SUM, O.AGG_COUNT, O.AGG_MIN, O.AGG_MAX, O.AGG_MEAN]
_pid = [10]


def _seed_of(kind: str) -> int:
    """A fixed seed per test-case name (crc32: the same in every process, unlike hash(str))."""
    import zlib
    return zlib.crc32(kind.encode()) & 0xFFFF


def _next_pid(n=1):
    _pid[0] += 100
    return _pid[0]


def test_c1_scalar_sum_no_filter(bydb, gpu_ctx):
    # BASELINE config 1: single part, 1k series x 1k points, 1 float64 field, sum() no filter
    rng = np.random.default_rng(0xB200)
    sids, ts, ver = grid(1000, 1000)
    lat = np.round(25 + rng.normal(0, 5, sids.size), 2)
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None)])
    oq = O.Query([part], np.unique(sids), [("latency", O.AGG_SUM)])
    got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
    assert_parity(got, want, oq.aggs, "C1")
    assert got.stats.rows_scanned == 1_000_000 and got.stats.rows_matched == 1_000_000
    # the exact decimal sum is an independent known answer
    exact = int(np.round(lat * 100).astype(np.int64).sum()) / 100.0
    assert abs(got.val_f64[0, 0] - exact) <= 1e-9 * abs(exact)


def test_groups_time_range_dict_pred_all_functions(bydb, gpu_ctx):
    rng = np.random.default_rng(11)
    sids, ts, ver = grid(37, 2500, sid0=5, sid_step=3)
    lat = np.round(25 + rng.normal(0, 5, sids.size), 2)
    calls = rng.integers(-5000, 5000, sids.size)
    region = [b"r%d" % v for v in rng.integers(0, 8, sids.size)]
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None), ("calls", O.VT_INT64, calls, None)],
                      [("default", [("region", O.VT_STR, region, None)])])
    usid = np.unique(sids)
    groups = (np.arange(usid.size) % 6).astype(np.int32)
    aggs = [("latency", f) for f in ALL5] + [("calls", f) for f in ALL5]
    oq = O.Query([part], usid, aggs, groups=groups, n_groups=6, tmin=T0 + 300 * STEP + 1, tmax=T0 + 2100 * STEP,
                 preds=[O.Pred("default", "region", O.OP_EQ, b"r3")])
    got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
    assert_parity(got, want, aggs, "grouped")
    assert got.stats.rows_matched == want.rows_matched


@pytest.mark.parametrize("kind", ["const", "delta_const", "delta_small", "delta_wide", "dod_monotone", "dod_counter_resets",
                                  "full_range", "negative", "two_byte", "one_byte"])
def test_int64_encodings(bydb, gpu_ctx, kind):
    rng = np.random.default_rng(_seed_of(kind))
    n_series, n_pts = 9, 8193 + 700   # 8193-row first block (measure.go:41-46 quirk) + a short tail block
    sids, ts, ver = grid(n_series, n_pts)
    n = sids.size
    if kind == "const":
        v = np.full(n, 42, dtype=np.int64)
    elif kind == "delta_const":
        v = np.tile(np.arange(n_pts, dtype=np.int64) * -7 + 100, n_series)
    elif kind == "delta_small":
        v = rng.integers(-50, 50, n)
    elif kind == "delta_wide":
        v = rng.integers(-(1 << 40), 1 << 40, n)
    elif kind == "dod_monotone":
        v = np.concatenate([np.cumsum(rng.integers(0, 1000, n_pts)) for _ in range(n_series)])
    elif kind == "dod_counter_resets":
        base = np.cumsum(rng.integers(1, 50, n_pts))
        base[n_pts // 3:] -= base[n_pts // 3]        # one reset -> isIncremental -> delta-of-delta
        base[n_pts // 3] = 0
        v = np.tile(base, n_series)
    elif kind == "full_range":
        v = rng.integers(-(1 << 62), 1 << 62, n) * 2 + rng.integers(0, 2, n)
        v[::1000] = np.iinfo(np.int64).max
        v[1::1000] = np.iinfo(np.int64).min
    elif kind == "negative":
        v = -np.abs(rng.integers(1, 1 << 20, n))
    elif kind == "two_byte":
        v = rng.integers(-700, 700, n).cumsum() % 100000
    else:
        v = np.cumsum(rng.integers(-3, 4, n))
    v = np.asarray(v, dtype=np.int64)
    part = build_part(sids, ts, ver, [("calls", O.VT_INT64, v, None)])
    usid = np.unique(sids)
    aggs = [("calls", f) for f in ALL5]
    for tmin, tmax in [(-(1 << 63), (1 << 63) - 1), (T0 + 17 * STEP, T0 + 8500 * STEP)]:
        oq = O.Query([part], usid, aggs, groups=(np.arange(usid.size) % 2).astype(np.int32), n_groups=2, tmin=tmin, tmax=tmax)
        got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
        assert_parity(got, want, aggs, f"int64/{kind}")


@pytest.mark.parametrize("kind", ["two_decimals", "ints_as_float", "mixed_exponents", "tiny", "huge_scale", "negative_mix", "random_walk_3dp"])
def test_float64_decimal_pages(bydb, gpu_ctx, kind):
    rng = np.random.default_rng(_seed_of(kind))
    n_series, n_pts = 6, 5000
    sids, ts, ver = grid(n_series, n_pts)
    n = sids.size
    if kind == "two_decimals":
        v = np.round(25 + rng.normal(0, 5, n), 2)
    elif kind == "ints_as_float":
        v = rng.integers(0, 1000, n).astype(np.float64) * 100.0   # trailing zeros -> positive exponent
    elif kind == "mixed_exponents":
        v = np.where(rng.random(n) < 0.5, np.round(rng.random(n) * 10, 4), rng.integers(0, 50, n) * 10.0)
    elif kind == "tiny":
        v = rng.integers(1, 9999, n) / 1e12     # exact division keeps the short decimal
    elif kind == "huge_scale":
        v = np.array([float("%de25" % k) for k in rng.integers(1, 999, n)])   # correctly rounded k*10^25
    elif kind == "negative_mix":
        v = np.round(rng.normal(0, 100, n), 1)
    else:
        v = np.round(np.cumsum(rng.normal(0, 0.1, n)), 3)
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, v, None)])
    usid = np.unique(sids)
    aggs = [("latency", f) for f in ALL5]
    oq = O.Query([part], usid, aggs, groups=(np.arange(usid.size) % 3).astype(np.int32), n_groups=3,
                 tmin=T0 + 3 * STEP, tmax=T0 + 4711 * STEP)
    got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
    assert_parity(got, want, aggs, f"float64/{kind}")


@pytest.mark.parametrize("kind", ["irregular", "accelerating", "single_row_blocks"])
def test_timestamp_encodings_and_ranges(bydb, gpu_ctx, kind):
    rng = np.random.default_rng(_seed_of(kind))
    n_series = 5
    rows = []
    for s in range(n_series):
        if kind == "irregular":      # Delta page
            t = T0 + np.cumsum(rng.integers(1, 10, 3000) * 1_000_000_000)
        elif kind == "accelerating":  # monotone deltas -> delta-of-delta page
            t = T0 + np.cumsum(np.arange(1, 3001, dtype=np.int64) * 1_000_000)
        else:
            t = T0 + np.arange(1, dtype=np.int64)
        rows.append((np.full(t.size, s + 1, np.uint64), t.astype(np.int64)))
    sids = np.concatenate([r[0] for r in rows])
    ts = np.concatenate([r[1] for r in rows])
    v = rng.integers(0, 1000, sids.size)
    part = build_part(sids, ts, np.ones(sids.size, np.int64), [("calls", O.VT_INT64, v, None)])
    usid = np.unique(sids)
    aggs = [("calls", O.AGG_SUM), ("calls", O.AGG_COUNT), ("calls", O.AGG_MIN)]
    lo, hi = int(ts.min()), int(ts.max())
    ranges = [(-(1 << 63), (1 << 63) - 1), (lo + (hi - lo) // 3, lo + 2 * (hi - lo) // 3), (lo, lo), (hi, hi + 5),
              (int(ts[min(7, ts.size - 1)]), int(ts[min(7, ts.size - 1)])),
              (int(ts[min(7, ts.size - 1)]) + 1, int(ts[9]) - 1 if ts.size > 9 else hi)]
    for tmin, tmax in ranges:
        oq = O.Query([part], usid, aggs, tmin=tmin, tmax=tmax)
        got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
        assert_parity(got, want, aggs, f"ts/{kind}/{tmin}-{tmax}")


def test_int64_tag_predicates_all_ops_and_conjunction(bydb, gpu_ctx):
    rng = np.random.default_rng(21)
    sids, ts, ver = grid(8, 4000)
    n = sids.size
    calls = rng.integers(0, 100, n)
    code = rng.integers(0, 6, n) * 100            # Delta page
    seq = np.tile(np.arange(4000, dtype=np.int64), 8)   # DeltaConst page
    flag = np.full(n, 3, dtype=np.int64)          # Const page
    region = [b"r%d" % v for v in np.repeat(rng.integers(0, 4, n // 50), 50)]   # runs of 50
    part = build_part(sids, ts, ver, [("calls", O.VT_INT64, calls, None)],
                      [("default", [("code", O.VT_INT64, code, None), ("seq", O.VT_INT64, seq, None),
                                    ("flag", O.VT_INT64, flag, None), ("region", O.VT_STR, region, None)])])
    usid = np.unique(sids)
    aggs = [("calls", O.AGG_SUM), ("calls", O.AGG_COUNT)]
    cases = []
    for op in (O.OP_EQ, O.OP_NE, O.OP_LT, O.OP_LE, O.OP_GT, O.OP_GE):
        cases.append([O.Pred("default", "code", op, 300)])
        cases.append([O.Pred("default", "seq", op, 1234)])
        cases.append([O.Pred("default", "flag", op, 3)])
        cases.append([O.Pred("default", "region", op, b"r2")])
    cases.append([O.Pred("default", "code", O.OP_GE, 200), O.Pred("default", "region", O.OP_NE, b"r0"), O.Pred("default", "seq", O.OP_LT, 3000)])
    cases.append([O.Pred("default", "nosuchtag", O.OP_EQ, b"x")])
    cases.append([O.Pred("default", "nosuchtag", O.OP_NE, b"x")])
    cases.append([O.Pred("nofamily", "region", O.OP_NE, 5)])
    cases.append([O.Pred("default", "region", O.OP_EQ, b"zzz")])
    for preds in cases:
        oq = O.Query([part], usid, aggs, tmin=T0 + 100 * STEP, tmax=T0 + 3900 * STEP, preds=preds)
        got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
        assert_parity(got, want, aggs, f"preds/{[(p.tag, p.op) for p in preds]}")


def test_dictionary_tag_shapes(bydb, gpu_ctx):
    rng = np.random.default_rng(5)
    sids, ts, ver = grid(6, 8193)
    n = sids.size
    calls = rng.integers(0, 100, n)
    per_row = [b"r%d" % v for v in rng.integers(0, 8, n)]                       # run length ~1
    per_series = [b"zone-%d" % (s % 3) for s in sids.tolist()]                   # one run per block
    many = [b"v%03d" % v for v in rng.integers(0, 25, n)]                        # 25 short values (<128 B of lens)
    with_nil = [None if v == 0 else (b"" if v == 1 else b"k%d" % v) for v in rng.integers(0, 5, n)]
    part = build_part(sids, ts, ver, [("calls", O.VT_INT64, calls, None)],
                      [("default", [("per_row", O.VT_STR, per_row, None), ("per_series", O.VT_STR, per_series, None),
                                    ("many", O.VT_STR, many, None), ("with_nil", O.VT_STR, with_nil, None)])])
    usid = np.unique(sids)
    aggs = [("calls", O.AGG_SUM), ("calls", O.AGG_MAX)]
    for preds in ([O.Pred("default", "per_row", O.OP_EQ, b"r5")], [O.Pred("default", "per_series", O.OP_EQ, b"zone-1")],
                  [O.Pred("default", "per_series", O.OP_GT, b"zone-0")], [O.Pred("default", "many", O.OP_LE, b"v010")],
                  [O.Pred("default", "with_nil", O.OP_EQ, b"")], [O.Pred("default", "with_nil", O.OP_NE, b"k3")],
                  [O.Pred("default", "per_row", O.OP_NE, b"r1"), O.Pred("default", "many", O.OP_EQ, b"v007")]):
        oq = O.Query([part], usid, aggs, groups=(np.arange(usid.size) % 2).astype(np.int32), n_groups=2, preds=preds)
        got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
        assert_parity(got, want, aggs, f"dict/{[(p.tag, p.op, p.value) for p in preds]}")


def test_multiple_parts_series_subset_and_topn(bydb, gpu_ctx):
    rng = np.random.default_rng(77)
    parts = []
    all_sids = np.arange(1, 201, dtype=np.uint64) * 7
    for k in range(3):   # time-disjoint parts, like consecutive flushes
        sids = np.repeat(all_sids, 400)
        ts = np.tile(T0 + (k * 400 + np.arange(400, dtype=np.int64)) * STEP, all_sids.size)
        lat = np.round(rng.gamma(2.0, 20.0, sids.size), 2)
        parts.append(build_part(sids, ts, np.ones(sids.size, np.int64), [("latency", O.VT_FLOAT64, lat, None)]))
    sel = all_sids[::2]                      # every other series
    groups = (np.arange(sel.size) // 4).astype(np.int32)     # 25 services x 4 series
    aggs = [("latency", O.AGG_SUM), ("latency", O.AGG_COUNT)]
    oq = O.Query(parts, sel, aggs, groups=groups, n_groups=25, tmin=T0 + 150 * STEP, tmax=T0 + 1000 * STEP, top_n=10, top_desc=True)
    got, want = run_both(bydb, gpu_ctx, parts, oq, _next_pid())
    assert got.group_id.tolist() == want.group_id.tolist()
    assert_parity(got, want, aggs, "multi-part top10")
    oq.top_desc, oq.top_n, oq.top_agg = False, 3, 1
    got, want = run_both(bydb, gpu_ctx, parts, oq, _next_pid())
    assert_parity(got, want, aggs, "multi-part bottom3")


def test_topn_adjacent_values_ties_and_float_order(bydb, gpu_ctx):
    # top.go:62-117: full-precision ordering (values differing by 1 / 1 ulp), ties -> earlier group, both directions
    rng = np.random.default_rng(31)
    n_groups = 300
    sids = np.arange(1, n_groups + 1, dtype=np.uint64)
    ivals = rng.integers(-5, 6, n_groups) + 1000            # many ties and neighbours
    fvals = np.round(rng.integers(-3, 4, n_groups) * 0.01 + 7.5, 2)
    part = build_part(sids, np.full(n_groups, T0, np.int64), np.ones(n_groups, np.int64),
                      [("calls", O.VT_INT64, ivals, None), ("latency", O.VT_FLOAT64, fvals, None)])
    groups = np.arange(n_groups, dtype=np.int32)
    aggs = [("calls", O.AGG_SUM), ("latency", O.AGG_MAX), ("calls", O.AGG_COUNT)]
    for top_agg in (0, 1, 2):
        for desc in (True, False):
            for n in (1, 7, 64, 299, 300, 1000):
                oq = O.Query([part], sids, aggs, groups=groups, n_groups=n_groups, top_n=n, top_agg=top_agg, top_desc=desc)
                got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
                assert_parity(got, want, aggs, f"top/{top_agg}/{desc}/{n}")


def test_empty_and_missing(bydb, gpu_ctx):
    sids, ts, ver = grid(4, 100)
    part = build_part(sids, ts, ver, [("calls", O.VT_INT64, np.arange(sids.size), None)])
    aggs = [("calls", O.AGG_SUM), ("nosuchfield", O.AGG_MAX), ("calls", O.AGG_COUNT)]
    for q in (O.Query([part], [99, 100], aggs),                                  # no series matches
              O.Query([part], np.unique(sids), aggs, tmin=T0 - 10, tmax=T0 - 1),  # nothing in range
              O.Query([part], np.unique(sids), aggs),                             # unknown field next to a real one
              O.Query([part], [], aggs)):
        got, want = run_both(bydb, gpu_ctx, [part], q, _next_pid())
        assert_parity(got, want, aggs, "empty/missing")


def _fallback_part(rng, n_series=5, n_pts=8193 + 700):
    """Every fallback shape of banyand/measure/column.go in one part: null cells (147-153, 192-195), floats that are
    not short decimals (203-208), few distinct values (dictionary inside the Plain page) and many (plain bytes block
    whose >= 128 B blocks are zstd frames, pkg/encoding/bytes.go:291-304)."""
    sids, ts, ver = grid(n_series, n_pts)
    n = sids.size
    calls = rng.integers(-10**12, 10**12, n)
    calls_null = (rng.random(n) < 0.1).astype(np.uint8)
    lat = rng.random(n) * 1e3 + rng.random(n) * 1e-7            # 16-17 significant digits, mixed exponents
    lat_null = (rng.random(n) < 0.05).astype(np.uint8)
    raw = rng.standard_normal(n) * 1e6                           # no nulls, just not decimal
    few = rng.choice(np.array([0.1 + 0.2, np.pi, -1e-300, 5e300, 2.0 / 3.0]), n)
    few_null = (rng.random(n) < 0.3).astype(np.uint8)
    few[sids == sids[0]] = np.e                                  # one value + nulls in the first series' blocks
    code = rng.integers(0, 50, n)
    code_null = (rng.random(n) < 0.05).astype(np.uint8)
    svc = [b"service-name-%03d" % v for v in rng.integers(0, 60, n)]          # 60 x 16 B values: zstd data block
    wide = [b"w%04d" % v for v in rng.integers(0, 200, n)]                     # 200 values: zstd lens + data blocks
    trace = [None if i % 97 == 0 else b"trace-%08d" % (i * 7919 % 100003) for i in range(n)]   # > 256 values: plain page
    part = build_part(sids, ts, ver,
                      [("calls", O.VT_INT64, calls, calls_null), ("latency", O.VT_FLOAT64, lat, lat_null),
                       ("raw", O.VT_FLOAT64, raw, None), ("few", O.VT_FLOAT64, few, few_null)],
                      [("default", [("code", O.VT_INT64, code, code_null), ("svc", O.VT_STR, svc, None), ("wide", O.VT_STR, wide, None),
                                    ("trace", O.VT_STR, trace, None)])])
    return part, sids, ts


FALLBACK_AGGS = [("calls", O.AGG_SUM), ("calls", O.AGG_COUNT), ("calls", O.AGG_MIN), ("calls", O.AGG_MAX), ("calls", O.AGG_MEAN),
                 ("latency", O.AGG_SUM), ("latency", O.AGG_COUNT), ("latency", O.AGG_MIN), ("latency", O.AGG_MAX), ("latency", O.AGG_MEAN),
                 ("raw", O.AGG_SUM), ("raw", O.AGG_MIN), ("raw", O.AGG_MAX), ("few", O.AGG_COUNT), ("few", O.AGG_MAX), ("few", O.AGG_MIN)]


def _assert_parity_abs(got, want, aggs, ctx):
    """assert_parity, except that float sums of mixed-sign data are compared against the magnitude of the terms."""
    sum_like = [a for a, (f, fn) in enumerate(aggs) if want.is_float[a] and fn in (O.AGG_SUM, O.AGG_MEAN)]
    keep = [a for a in range(len(aggs)) if a not in sum_like]
    sub = lambda r, idx: type("R", (), dict(group_id=r.group_id, rows=r.rows, is_float=r.is_float[idx], val_i64=r.val_i64[:, idx],
                                            val_f64=r.val_f64[:, idx]))
    assert_parity(sub(got, keep), sub(want, keep), [aggs[a] for a in keep], ctx)
    for a in sum_like:
        g, w = got.val_f64[:, a], want.val_f64[:, a]
        assert (np.abs(g - w) <= 1e-9 * np.maximum(np.abs(w), 1e6)).all(), f"{ctx}: float agg {a} {aggs[a]}: {g} vs {w}"


def test_fallback_numeric_pages_nulls_and_non_decimal_floats(bydb, gpu_ctx):
    rng = np.random.default_rng(41)
    part, sids, ts = _fallback_part(rng)
    usid = np.unique(sids)
    h = gpu_ctx.register_part(_next_pid(), part.files())
    info = gpu_ctx.part_info(h)
    assert info["fallback_unpacked"] >= 4 * 2 * usid.size and info["fallback_left"] == 0, info
    gpu_ctx.release_part(h)
    groups = (np.arange(usid.size) % 2).astype(np.int32)
    for kw in (dict(), dict(tmin=T0 + 100 * STEP, tmax=T0 + 8500 * STEP), dict(groups=groups, n_groups=2),
               dict(preds=[O.Pred("default", "code", O.OP_LT, 25)]),
               dict(preds=[O.Pred("default", "code", O.OP_NE, 7)], tmin=T0 + 8000 * STEP, tmax=T0 + 8400 * STEP, groups=groups, n_groups=2)):
        oq = O.Query([part], usid, FALLBACK_AGGS, **kw)
        got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
        _assert_parity_abs(got, want, FALLBACK_AGGS, f"fallback/{sorted(kw)}")
    # Top-N over a float sum of raw cells, and a group whose only column is all-null in range
    oq = O.Query([part], usid, [("raw", O.AGG_MAX), ("few", O.AGG_COUNT)], groups=np.arange(usid.size, dtype=np.int32), n_groups=usid.size,
                 top_n=3, top_agg=0, top_desc=True)
    got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
    assert_parity(got, want, oq.aggs, "fallback/top")


def test_fallback_string_pages_zstd_dictionary_and_plain(bydb, gpu_ctx):
    rng = np.random.default_rng(43)
    part, sids, ts = _fallback_part(rng, n_series=4)
    usid = np.unique(sids)
    aggs = [("calls", O.AGG_COUNT), ("raw", O.AGG_MAX), ("latency", O.AGG_MIN)]
    for preds in ([O.Pred("default", "svc", O.OP_EQ, b"service-name-017")], [O.Pred("default", "svc", O.OP_GE, b"service-name-040")],
                  [O.Pred("default", "wide", O.OP_NE, b"w0100")], [O.Pred("default", "wide", O.OP_LT, b"w0050"), O.Pred("default", "svc", O.OP_GT, b"service-name-010")],
                  [O.Pred("default", "trace", O.OP_EQ, b"trace-%08d" % (5 * 7919 % 100003))], [O.Pred("default", "trace", O.OP_GT, b"trace-00050000")],
                  [O.Pred("default", "trace", O.OP_NE, b"trace-00000000")], [O.Pred("default", "trace", O.OP_LE, b"trace-0001")],
                  [O.Pred("default", "trace", O.OP_LT, b"trace-00070000"), O.Pred("default", "code", O.OP_GE, 10)]):
        oq = O.Query([part], usid, aggs, groups=(np.arange(usid.size) % 2).astype(np.int32), n_groups=2, preds=preds)
        got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
        assert_parity(got, want, aggs, f"fallback-str/{[(p.tag, p.op, p.value) for p in preds]}")


def test_fallback_pages_on_the_cold_host_path(bydb, gpu_ctx):
    # bydb_scan_agg_host scans the pages as they are and only unpacks (then rescans) when it meets a fallback page
    import torch
    rng = np.random.default_rng(47)
    part, sids, ts = _fallback_part(rng, n_series=3, n_pts=9000)
    usid = np.unique(sids)
    aggs = [("latency", O.AGG_MEAN), ("calls", O.AGG_MAX), ("few", O.AGG_COUNT)]
    oq = O.Query([part], usid, aggs, preds=[O.Pred("default", "svc", O.OP_LE, b"service-name-030")])
    want = O.run_query(oq)
    files = {k: np.frombuffer(v, dtype=np.uint8) for k, v in part.files().items()}
    q = bydb.Query([], usid, aggs, preds=[bydb.Pred("default", "svc", O.OP_LE, b"service-name-030")])
    got = gpu_ctx.scan_agg_host([files], q)
    _assert_parity_abs(got, want, aggs, "fallback/host staged")
    keep, pinned = [], {}
    for k, v in files.items():
        t = torch.empty(v.size + 256, dtype=torch.uint8, pin_memory=True)
        t[:v.size].copy_(torch.from_numpy(v.copy()))
        keep.append(t)
        pinned[k] = t[:v.size].numpy()
    q.flags = 1
    got = gpu_ctx.scan_agg_host([pinned], q)
    _assert_parity_abs(got, want, aggs, "fallback/host zero-copy")


def test_version_dedup_across_overlapping_parts(bydb, gpu_ctx):
    # query.go:995-1004 / query_batch.go:151-161: a (series, timestamp) present in several parts keeps the highest version
    rng = np.random.default_rng(17)
    n_series, n_pts = 12, 9000
    sids, ts, _ = grid(n_series, n_pts)
    base = rng.integers(0, 1000, sids.size)
    lat = np.round(rng.normal(20, 3, sids.size), 2)
    p1 = build_part(sids, ts, np.full(sids.size, 5, np.int64), [("calls", O.VT_INT64, base, None), ("latency", O.VT_FLOAT64, lat, None)])
    # part 2 rewrites a random 30% of the points of the even series: half of them newer (version 9), half stale (version 2)
    m = (rng.random(sids.size) < 0.3) & (sids % 2 == 0)
    ver2 = np.where(rng.random(m.sum()) < 0.5, 9, 2).astype(np.int64)
    p2 = build_part(sids[m], ts[m], ver2, [("calls", O.VT_INT64, base[m] + 100000, None), ("latency", O.VT_FLOAT64, lat[m] + 1000, None)])
    # part 3: late data for series 3 only, newest version, plus points beyond the others' range
    m3 = sids == 3
    ts3 = np.concatenate([ts[m3][::7], ts[m3][-1] + (1 + np.arange(50)) * STEP])
    p3 = build_part(np.full(ts3.size, 3, np.uint64), ts3, np.full(ts3.size, 11, np.int64),
                    [("calls", O.VT_INT64, np.arange(ts3.size) - 7, None), ("latency", O.VT_FLOAT64, np.full(ts3.size, 0.5), None)])
    usid = np.unique(sids)
    aggs = [("calls", f) for f in ALL5] + [("latency", O.AGG_SUM), ("latency", O.AGG_MAX)]
    for kw in (dict(), dict(tmin=T0 + 1000 * STEP, tmax=T0 + 8500 * STEP),
               dict(groups=(np.arange(usid.size) % 3).astype(np.int32), n_groups=3)):
        oq = O.Query([p1, p2, p3], usid, aggs, **kw)
        got, want = run_both(bydb, gpu_ctx, [p1, p2, p3], oq, _next_pid())
        assert_parity(got, want, aggs, f"dedup/{list(kw)}")
    # order of the parts must not matter
    oq = O.Query([p3, p1, p2], usid, aggs)
    got, want = run_both(bydb, gpu_ctx, [p3, p1, p2], oq, _next_pid())
    assert_parity(got, want, aggs, "dedup/reordered")


def test_version_dedup_irregular_timestamps_and_predicate(bydb, gpu_ctx):
    rng = np.random.default_rng(23)
    rows1, rows2 = [], []
    for s in range(1, 6):
        t = T0 + np.cumsum(rng.integers(1, 10, 4000)) * 1_000_000_000
        rows1.append((np.full(t.size, s, np.uint64), t))
        pick = rng.random(t.size) < 0.4
        rows2.append((np.full(pick.sum(), s, np.uint64), t[pick]))
    sid1, ts1 = np.concatenate([r[0] for r in rows1]), np.concatenate([r[1] for r in rows1])
    sid2, ts2 = np.concatenate([r[0] for r in rows2]), np.concatenate([r[1] for r in rows2])
    v1, v2 = rng.integers(0, 100, sid1.size), rng.integers(1000, 2000, sid2.size)
    reg1 = [b"r%d" % x for x in rng.integers(0, 3, sid1.size)]
    reg2 = [b"r%d" % x for x in rng.integers(0, 3, sid2.size)]
    p1 = build_part(sid1, ts1, np.full(sid1.size, 1, np.int64), [("calls", O.VT_INT64, v1, None)], [("default", [("region", O.VT_STR, reg1, None)])])
    p2 = build_part(sid2, ts2, np.full(sid2.size, 2, np.int64), [("calls", O.VT_INT64, v2, None)], [("default", [("region", O.VT_STR, reg2, None)])])
    aggs = [("calls", O.AGG_SUM), ("calls", O.AGG_COUNT), ("calls", O.AGG_MAX)]
    for preds in ([], [O.Pred("default", "region", O.OP_EQ, b"r1")]):
        oq = O.Query([p1, p2], np.arange(1, 6, dtype=np.uint64), aggs, preds=preds, tmin=int(ts1.min()) + 5, tmax=int(ts1.max()) - 5)
        got, want = run_both(bydb, gpu_ctx, [p1, p2], oq, _next_pid())
        assert_parity(got, want, aggs, f"dedup-irregular/{len(preds)}")


def test_scan_agg_host_and_idempotent_register(bydb, gpu_ctx):
    rng = np.random.default_rng(3)
    sids, ts, ver = grid(20, 1000)
    lat = np.round(rng.normal(50, 10, sids.size), 2)
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None)])
    aggs = [("latency", O.AGG_MEAN), ("latency", O.AGG_MAX)]
    oq = O.Query([part], np.unique(sids), aggs)
    want = O.run_query(oq)
    files = {k: np.frombuffer(v, dtype=np.uint8) for k, v in part.files().items()}
    got = gpu_ctx.scan_agg_host([files], bydb.Query([], np.unique(sids), aggs))
    assert_parity(got, want, aggs, "host path")
    assert got.stats.h2d_bytes >= sum(v.size for k, v in files.items() if k in ("timestamps.bin", "fv.bin"))
    # zero-copy: pinned, padded host buffers are read in place by the kernels
    import torch
    keep, pinned = [], {}
    for k, v in files.items():
        t = torch.empty(v.size + 256, dtype=torch.uint8, pin_memory=True)
        t[:v.size].copy_(torch.from_numpy(v.copy()))
        keep.append(t)
        pinned[k] = t[:v.size].numpy()
    got = gpu_ctx.scan_agg_host([pinned], bydb.Query([], np.unique(sids), aggs, flags=1))
    assert_parity(got, want, aggs, "host zero-copy path")
    assert got.stats.h2d_bytes >= got.stats.page_bytes      # directory + the pages the kernels pulled over PCIe
    with pytest.raises(bydb.BydbError):     # pageable memory must be refused, not silently copied
        gpu_ctx.scan_agg_host([files], bydb.Query([], np.unique(sids), aggs, flags=1))
    pid = _next_pid()
    h1 = gpu_ctx.register_part(pid, part.files())
    h2 = gpu_ctx.register_part(pid, part.files())
    assert h1 == h2
    info = gpu_ctx.part_info(h1)
    assert info["n_rows"] == sids.size and info["n_blocks"] == 20
    gpu_ctx.release_part(h1)
    with pytest.raises(bydb.BydbError):
        gpu_ctx.part_info(h1)


def test_operator_gpuscanagg_matches_batch_aggregation_contract(bydb, gpu_ctx):
    # reads like pkg/query/vectorized/measure/aggregation_test.go: schema (tag key + field), AggSpecs, NextBatch until EOF
    rng = np.random.default_rng(8)
    sids, ts, ver = grid(30, 500)
    calls = rng.integers(0, 50, sids.size)
    part = build_part(sids, ts, ver, [("calls", O.VT_INT64, calls, None)])
    h = gpu_ctx.register_part(_next_pid(), part.files())
    V = bydb
    schema = V.BatchSchema([V.ColumnDef("service_id", V.ColumnRole.RoleTag, V.ColumnType.ColumnTypeString, "default"),
                            V.ColumnDef("calls", V.ColumnRole.RoleField, V.ColumnType.ColumnTypeInt64)])
    usid = np.unique(sids)[::-1].copy()      # index order is not ascending
    svc = ["svc_%02d" % (int(s) % 7) for s in usid]
    op = V.GPUScanAgg(gpu_ctx, schema, [0], [V.AggSpec("sum_v", V.AggSum, 1), V.AggSpec("n", V.AggCount, 1), V.AggSpec("mean_v", V.AggMean, 1)],
                      V.ScanSpec(parts=[h], series_ids=usid, series_tags={("default", "service_id"): svc}), batch_size=4)
    op.Init()
    assert [c.Name for c in op.OutputSchema().Columns] == ["service_id", "sum_v", "n", "mean_v"]
    out = {}
    order = []
    while True:
        b = op.NextBatch()
        if b is None:
            break
        assert 0 < b.Len <= 4 and b.Selection is None
        for i in range(b.Len):
            out[b.Columns[0][i]] = (int(b.Columns[1][i]), int(b.Columns[2][i]), int(b.Columns[3][i]))
            order.append(b.Columns[0][i])
    assert op.NextBatch() is None
    op.Close()
    op.Close()   # idempotent
    first_seen = []
    for s in svc:
        if s not in first_seen:
            first_seen.append(s)
    assert order == first_seen           # group-insertion order (aggregation.go:211-213)
    sid_svc = dict(zip(usid.tolist(), svc))
    for name in first_seen:
        m = np.array([sid_svc[int(s)] == name for s in sids])
        tot, n = int(calls[m].sum()), int(m.sum())
        assert out[name] == (tot, n, max(tot // n, 1))
    # BatchLimit windows over the same output stream (limit_test.go:52-129): first N, rows N..N+M, offset beyond the data
    def names_of(limit):
        o = V.GPUScanAgg(gpu_ctx, schema, [0], [V.AggSpec("sum_v", V.AggSum, 1)],
                         V.ScanSpec(parts=[h], series_ids=usid, series_tags={("default", "service_id"): svc}), batch_size=2, limit=limit)
        o.Init()
        got_names = []
        while (bt := o.NextBatch()) is not None:
            assert 0 < bt.Len <= 2
            got_names += list(bt.Columns[0])
        o.Close()
        return got_names
    assert names_of(V.LimitSpec(0, 3)) == first_seen[:3]
    assert names_of(V.LimitSpec(2, 4)) == first_seen[2:6]
    assert names_of(V.LimitSpec(5, 100)) == first_seen[5:]
    assert names_of(V.LimitSpec(50, 10)) == []
    assert names_of(V.LimitSpec(1, 0)) == []
    gpu_ctx.release_part(h)


def test_large_property_checks(bydb, gpu_ctx):
    # size-independent properties at a size the oracle would take long on: count == rows, sum over groups ==
    # scalar sum (int64, exact), min <= mean <= max, idempotence (same query twice -> identical bits)
    rng = np.random.default_rng(99)
    n_series, n_pts = 200, 20000
    sids, ts, ver = grid(n_series, n_pts)
    lat = np.round(25 + rng.normal(0, 5, sids.size), 2)
    calls = rng.integers(0, 1000, sids.size)
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None), ("calls", O.VT_INT64, calls, None)])
    h = gpu_ctx.register_part(_next_pid(), part.files())
    usid = np.unique(sids)
    aggs = [("calls", O.AGG_SUM), ("calls", O.AGG_COUNT), ("latency", O.AGG_MIN), ("latency", O.AGG_MEAN), ("latency", O.AGG_MAX), ("latency", O.AGG_SUM)]
    q1 = bydb.Query([h], usid, aggs)
    qg = bydb.Query([h], usid, aggs, series_group=(np.arange(usid.size) % 16).astype(np.int32), n_groups=16)
    a, b, g = gpu_ctx.scan_agg(q1), gpu_ctx.scan_agg(q1), gpu_ctx.scan_agg(qg)
    assert a.val_i64.tolist() == b.val_i64.tolist() and a.val_f64.view(np.uint64).tolist() == b.val_f64.view(np.uint64).tolist()
    assert a.val_i64[0, 1] == sids.size == a.rows[0]
    assert a.val_i64[0, 0] == int(calls.sum()) == int(g.val_i64[:, 0].sum())
    assert g.val_i64[:, 1].sum() == sids.size
    assert a.val_f64[0, 2] == lat.min() and a.val_f64[0, 4] == lat.max()
    assert a.val_f64[0, 2] <= a.val_f64[0, 3] <= a.val_f64[0, 4]
    exact = int(np.round(lat * 100).astype(np.int64).sum()) / 100.0
    assert abs(a.val_f64[0, 5] - exact) <= 1e-9 * exact
    assert abs(g.val_f64[:, 5].sum() - exact) <= 1e-9 * exact
    gpu_ctx.release_part(h)


def test_c3_shape_grouped_sum_top(bydb, gpu_ctx):
    # BASELINE config 3 scaled down: GROUP BY service_id (100 services x 10 series) sum(latency) -> Top 10 desc
    rng = np.random.default_rng(0xC3)
    n_series, n_pts = 1000, 3000
    sids, ts, ver = grid(n_series, n_pts, sid0=17, sid_step=3)
    lat = np.round(rng.gamma(2.0, 12.0, sids.size), 2)
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None)])
    usid = np.unique(sids)
    groups = (np.arange(usid.size) // 10).astype(np.int32)
    aggs = [("latency", O.AGG_SUM), ("latency", O.AGG_COUNT)]
    oq = O.Query([part], usid, aggs, groups=groups, n_groups=100, top_n=10, top_desc=True, threads=4)
    got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
    assert_parity(got, want, aggs, "C3 shape")
    assert got.stats.blocks_slow_lane == 0


@pytest.mark.timeout(120)
def test_corrupt_pages_fail_or_answer_but_never_hang(bydb, gpu_ctx):
    # flipped / truncated page bytes must surface as an error code (or a wrong-but-terminating answer), never a hang or a crash
    rng = np.random.default_rng(404)
    sids, ts, ver = grid(6, 3000)
    lat = np.round(rng.normal(20, 4, sids.size), 2)
    wide = rng.integers(-(1 << 40), 1 << 40, sids.size)
    region = [b"r%d" % v for v in rng.integers(0, 5, sids.size)]
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None), ("wide", O.VT_INT64, wide, None)],
                      [("default", [("region", O.VT_STR, region, None)])])
    files = part.files()
    q_aggs = [("latency", O.AGG_SUM), ("wide", O.AGG_MAX)]
    outcomes = {"ok": 0, "error": 0}
    for trial in range(24):
        bad = dict(files)
        target = ["fv.bin", "default.tf", "timestamps.bin"][trial % 3]
        buf = bytearray(bad[target])
        if trial % 4 == 3:
            buf = buf[: max(16, len(buf) // 2)]                     # truncation -> registration must refuse
        else:
            for pos in rng.integers(0, len(buf), 6):
                buf[int(pos)] ^= int(rng.integers(1, 256))          # bit rot inside the pages
        bad[target] = bytes(buf)
        try:
            h = gpu_ctx.register_part(_next_pid(), bad)
        except bydb.BydbError:
            outcomes["error"] += 1
            continue
        try:
            gpu_ctx.scan_agg(bydb.Query([h], np.unique(sids), q_aggs, preds=[bydb.Pred("default", "region", bydb.OP_EQ, b"r2")]))
            outcomes["ok"] += 1
        except bydb.BydbError as e:
            assert e.code in (-22, -95, -5)
            outcomes["error"] += 1
        finally:
            gpu_ctx.release_part(h)
    assert outcomes["error"] > 0
    # the context is still healthy afterwards
    h = gpu_ctx.register_part(_next_pid(), files)
    got = gpu_ctx.scan_agg(bydb.Query([h], np.unique(sids), q_aggs))
    want = O.run_query(O.Query([part], np.unique(sids), q_aggs))
    assert_parity(got, want, q_aggs, "after corruption trials")
    gpu_ctx.release_part(h)


def test_partial_tables_async_scan_combine_finalize(bydb, gpu_ctx):
    # the multi-GPU reduce on one device: two "ranks" = two series-disjoint parts, each scanned into its own partial table
    # (one synchronously with statistics, one asynchronously), rank-ordered combine, finalisation.  Same answer as one query.
    import torch
    rng = np.random.default_rng(61)
    parts, all_sids = [], []
    for r in range(2):
        sids, ts, ver = grid(40, 700, sid0=1 + 1000 * r)
        lat = np.round(rng.gamma(2.0, 15.0, sids.size), 2)
        calls = rng.integers(-500, 500, sids.size)
        region = [b"r%d" % v for v in rng.integers(0, 4, sids.size)]
        parts.append(build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None), ("calls", O.VT_INT64, calls, None)],
                                [("default", [("region", O.VT_STR, region, None)])]))
        all_sids.append(np.unique(sids))
    usid = np.concatenate(all_sids)
    groups = (np.arange(usid.size) % 7).astype(np.int32)
    aggs = [("latency", O.AGG_MEAN), ("latency", O.AGG_MIN), ("calls", O.AGG_SUM), ("calls", O.AGG_MAX), ("calls", O.AGG_COUNT)]
    preds = [O.Pred("default", "region", O.OP_NE, b"r1")]
    want = O.run_query(O.Query(parts, usid, aggs, groups=groups, n_groups=7, preds=preds, tmin=T0 + 10 * STEP, tmax=T0 + 650 * STEP))
    handles = [gpu_ctx.register_part(_next_pid(), p.files()) for p in parts]
    stream = torch.cuda.current_stream().cuda_stream
    try:
        def q_of(hs, preds_):
            return bydb.Query(hs, usid, aggs, series_group=groups, n_groups=7, tmin=T0 + 10 * STEP, tmax=T0 + 650 * STEP,
                              preds=[bydb.Pred(p.family, p.tag, p.op, p.value) for p in preds_])
        lay = gpu_ctx.partials_layout(q_of([handles[0]], preds))
        words = lay["total_bytes"] // 8
        tables = torch.zeros(2 * words, dtype=torch.float64, device="cuda")
        st = gpu_ctx.scan_partials(q_of([handles[0]], preds), tables.data_ptr(), lay["total_bytes"], stream)
        assert st.rows_scanned > 0
        pq1 = gpu_ctx.prepare(q_of([handles[1]], preds))
        assert gpu_ctx.scan_partials(pq1, tables.data_ptr() + lay["total_bytes"], lay["total_bytes"], stream, want_stats=False) is None
        qf = q_of([], preds)
        gpu_ctx.partials_combine(qf, tables.data_ptr(), 2, lay["total_bytes"], stream)
        got = gpu_ctx.reduce_finalize(qf, tables.data_ptr(), lay["total_bytes"], stream)
        assert_parity(got, want, aggs, "partials/async")
        # a device-side failure of an asynchronous scan travels in the table and fails the finalisation
        bad = [O.Pred("default", "region", O.OP_EQ, 5)]            # int64 literal against a string tag
        assert gpu_ctx.scan_partials(q_of([handles[1]], bad), tables.data_ptr(), lay["total_bytes"], stream, want_stats=False) is None
        with pytest.raises(bydb.BydbError) as ei:
            gpu_ctx.reduce_finalize(q_of([], bad), tables.data_ptr(), lay["total_bytes"], stream)
        assert ei.value.code == -22
        with pytest.raises(bydb.BydbError):                          # the synchronous form reports it itself
            gpu_ctx.scan_partials(q_of([handles[1]], bad), tables.data_ptr(), lay["total_bytes"], stream)
    finally:
        for h in handles:
            gpu_ctx.release_part(h)


@pytest.mark.parametrize("name", E2E_CASES)
def test_reference_e2e_cases_on_the_device(bydb, gpu_ctx, name):
    # the reference's own end-to-end cases (test/cases/measure/data, tests/golden/e2e_cases.json): expected rows of the want/*.yaml
    part, oq, names, want, ordered = load_e2e_case(name)
    got, oracle_res = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
    check_e2e_rows(got, names, want, ordered, name)
    assert_parity(got, oracle_res, oq.aggs, f"e2e/{name}")


@pytest.mark.parametrize("name", [c for c in E2E_CASES if c.startswith("gen_feat_") or c.startswith("float_top") or c == "top"])
def test_reference_e2e_cases_through_the_operator(bydb, gpu_ctx, name):
    # the same cases through the PullOperator mirror: row order (group first-appearance under the request's order-by, or Top order),
    # the non-key projected tag's first-seen value, values -- exactly the rows of the reference's want/*.yaml
    import json, os
    case = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "e2e_cases.json")))[name]
    part, oq, names, want, ordered = load_e2e_case(name)
    V = bydb
    h = gpu_ctx.register_part(_next_pid(), part.files())
    try:
        tags, q = case["tags"], case["query"]
        proj = q["projected_tags"]
        is_float = next(f["type"] for f in case["fields"] if f["name"] == q["field"]) == "float"
        schema = V.BatchSchema([V.ColumnDef(t, V.ColumnRole.RoleTag, V.ColumnType.ColumnTypeString, case["family"]) for t in proj] +
                               [V.ColumnDef(q["field"], V.ColumnRole.RoleField, V.ColumnType.ColumnTypeFloat64 if is_float else V.ColumnType.ColumnTypeInt64)])
        # per-series tag values in series order (= first appearance in the data, which is time order)
        ent_rows = {}
        for r in case["rows"]:
            ent_rows.setdefault(tuple(r["tags"][tags.index(t)] for t in case["entity"]), r)
        series_rows = list(ent_rows.values())
        series_tags = {(case["family"], t): [r["tags"][tags.index(t)] for r in series_rows] for t in proj}
        func = {"SUM": V.AggSum, "COUNT": V.AggCount, "MIN": V.AggMin, "MAX": V.AggMax, "MEAN": V.AggMean}[q["agg"]]
        preds = [V.Pred(p.family, p.tag, p.op, p.value) for p in oq.preds]
        op = V.GPUScanAgg(gpu_ctx, schema, [proj.index(q["group_by"])], [V.AggSpec(q["field"], func, len(proj))],
                          V.ScanSpec(parts=[h], series_ids=np.asarray(oq.sids, dtype=np.uint64), series_tags=series_tags, preds=preds,
                                     order_desc=q["order"] == "SORT_DESC"),
                          batch_size=2, top=V.TopSpec(q["top"]["n"], 0, q["top"]["desc"]) if q["top"] else None)
        op.Init()
        rows = []
        while (b := op.NextBatch()) is not None:
            for i in range(b.Len):
                rows.append(({t: b.Columns[k][i] for k, t in enumerate(proj)}, b.Columns[len(proj)][i]))
        op.Close()
        assert len(rows) == len(want), (rows, want)
        for (gt, gv), w in zip(rows, want):
            assert gt == {t: w["tags"][t] for t in proj}, f"{name}: tags {gt} vs {w['tags']}"
            assert abs(float(gv) - float(w["value"])) <= 1e-9 * max(abs(float(w["value"])), 1e-300), f"{name}: {gv} vs {w['value']}"
    finally:
        gpu_ctx.release_part(h)


@pytest.mark.parametrize("case", sorted(QUERY_TEST_CASES))
def test_reference_query_test_fixtures_on_the_device(bydb, gpu_ctx, case):
    # banyand/measure/query_test.go TestQueryResult on dpsTS1 / dpsTS11 / dpsTS2: cross-part version dedup in either part order,
    # series without a field (all-null fallback pages), per-series aggregates of the surviving rows
    names, expect, _ = QUERY_TEST_CASES[case]
    parts = [query_test_fixture(n) for n in names]
    oq = O.Query(parts, [1, 2, 3], QUERY_TEST_AGGS, groups=np.arange(3, dtype=np.int32), n_groups=3, tmin=1, tmax=2)
    got, want = run_both(bydb, gpu_ctx, parts, oq, _next_pid())
    check_query_test_case(got, expect, case)
    assert_parity(got, want, QUERY_TEST_AGGS, f"query_test/{case}")
    # the int64 tag with null cells as a row predicate on top of the dedup (series 1 only carries it)
    oq.preds = [O.Pred("singleTag", "intTag", O.OP_GE, 10)]
    got, want = run_both(bydb, gpu_ctx, parts, oq, _next_pid())
    assert_parity(got, want, QUERY_TEST_AGGS, f"query_test/{case}/pred")


def test_equal_version_duplicates_keep_the_earlier_part(bydb, gpu_ctx):
    # same (series, timestamp, version) in two parts with different values: unspecified in the reference (heap order), defined
    # here as "the earlier part of the query wins" -- oracle and device must agree for both part orders
    ts_a = T0 + np.array([5, 6, 7], dtype=np.int64) * STEP
    ts_b = T0 + np.array([1, 5, 6, 9], dtype=np.int64) * STEP
    pa = build_part(np.full(3, 4, np.uint64), ts_a, np.array([2, 2, 1], np.int64), [("calls", O.VT_INT64, np.array([10, 20, 30]), None)])
    pb = build_part(np.full(4, 4, np.uint64), ts_b, np.array([2, 2, 3, 2], np.int64), [("calls", O.VT_INT64, np.array([100, 200, 300, 400]), None)])
    aggs = [("calls", O.AGG_SUM), ("calls", O.AGG_COUNT), ("calls", O.AGG_MIN)]
    for parts, want in (([pa, pb], 840), ([pb, pa], 1030)):
        got, ora = run_both(bydb, gpu_ctx, parts, O.Query(parts, [4], aggs), _next_pid())
        assert_parity(got, ora, aggs, "equal-version duplicates")
        assert int(got.val_i64[0, 0]) == want and int(got.val_i64[0, 1]) == 5


@pytest.mark.parametrize("seed", range(24))
def test_random_sweep_device_vs_oracle(bydb, gpu_ctx, seed):
    # the generator of tests/test_oracle_model_sweep.py (1-3 overlapping parts, versions incl. equal ones, nil cells, int/str
    # predicates, groups, all five functions): device vs oracle; float sums against the magnitude of the terms
    from tests.test_oracle_model_sweep import AGGS, case_query, random_case
    parts, _, kw = random_case(seed)
    oq = case_query(parts, kw)
    got, want = run_both(bydb, gpu_ctx, parts, oq, _next_pid())
    # Bound on |device - oracle| for a float64 sum or mean, first order in u = 2^-53, over the stored cells v of field f in the
    # case's parts (sum|v|).  The oracle adds the cells one at a time: at most rows - 1 roundings per term.  The device sums a
    # decimal page exactly, rounds that sum to float64 (up to twice) and scales it by 10^exp (once); with the rounding of each
    # decoded cell that is 4 u * sum|v| per block, plus blocks - 1 additions across blocks.  The mean's one division adds
    # u * |mean| <= u * sum|v|.  Together: (rows + blocks + 4) * u * sum|v|.  A raw-cell page (nulls, or floats with no exact
    # decimal form) is summed in float64 instead, lane-strided then by a 5-level warp tree: ceil(count / 32) + 4 roundings per
    # term at most, with count <= 8193 rows per block, which the last term adds.
    rows = sum(p.meta()["total_count"] for p in parts)
    blocks = sum(p.meta()["blocks_count"] for p in parts)
    abs_sum = 0.0
    for p in parts:
        sids = sorted({int(s) for s in O.scan_rows(O.Query([p], list(range(1, kw["nser"] + 1)), [("f", O.AGG_SUM)]))["sid"]})
        _, _, vals, nulls = O.scan_rows(O.Query([p], sids, [("f", O.AGG_SUM)]))["fields"][0]
        abs_sum += float(np.abs(vals[~nulls]).sum())
    ftol = (rows + blocks + 4 + (min(rows, 8193) + 31) // 32 + 4) * 2.0 ** -53 * abs_sum
    assert got.group_id.tolist() == want.group_id.tolist() and got.rows.tolist() == want.rows.tolist()
    assert got.is_float.tolist() == want.is_float.tolist()
    for a, (_, fn) in enumerate(AGGS):
        if not want.is_float[a]:
            assert got.val_i64[:, a].tolist() == want.val_i64[:, a].tolist(), (seed, a)
        elif fn in (O.AGG_MIN, O.AGG_MAX):
            assert got.val_f64[:, a].view(np.uint64).tolist() == want.val_f64[:, a].view(np.uint64).tolist(), (seed, a)
        else:
            assert (np.abs(got.val_f64[:, a] - want.val_f64[:, a]) <= ftol).all(), (seed, a, got.val_f64[:, a], want.val_f64[:, a], ftol)


def test_block_selection_part_iter_test_go(bydb, gpu_ctx):
    # banyand/measure/part_iter_test.go Test_partIter_nextBlock on `dps`: the blocks plan_blocks selects for each series list
    from tests.helpers import PART_ITER_CASES, part_iter_fixture
    part = part_iter_fixture()
    for sids, want_sids in PART_ITER_CASES:
        oq = O.Query([part], sids, [("intField", O.AGG_COUNT)], groups=np.arange(len(sids), dtype=np.int32), n_groups=max(len(sids), 1), tmin=1, tmax=220)
        got, want = run_both(bydb, gpu_ctx, [part], oq, _next_pid())
        assert_parity(got, want, oq.aggs, f"part_iter/{sids}")
        assert got.stats.blocks_scanned == len(want_sids) and got.stats.rows_scanned == 2 * len(want_sids)


def test_concurrent_callers_share_one_context(bydb, gpu_ctx):
    # the cgo contract (SURVEY 8b): many goroutines call into one bydb_ctx concurrently -> one stream / staging slot per call.
    # 8 threads x 25 queries of three shapes (resident scan, Top-N, cold host path) must all return the sequential answers.
    import threading
    rng = np.random.default_rng(71)
    sids, ts, ver = grid(40, 3000)
    lat = np.round(rng.normal(30, 6, sids.size), 2)
    calls = rng.integers(0, 500, sids.size)
    region = [b"r%d" % v for v in rng.integers(0, 4, sids.size)]
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None), ("calls", O.VT_INT64, calls, None)], [("default", [("region", O.VT_STR, region, None)])])
    usid = np.unique(sids)
    h = gpu_ctx.register_part(_next_pid(), part.files())
    files = {k: np.frombuffer(v, dtype=np.uint8) for k, v in part.files().items()}
    groups = (np.arange(usid.size) % 5).astype(np.int32)
    shapes = [
        lambda: gpu_ctx.scan_agg(bydb.Query([h], usid, [("latency", O.AGG_MEAN), ("calls", O.AGG_MAX)], preds=[bydb.Pred("default", "region", O.OP_EQ, b"r2")])),
        lambda: gpu_ctx.scan_agg(bydb.Query([h], usid, [("calls", O.AGG_SUM)], series_group=groups, n_groups=5, top_n=3, top_desc=True)),
        lambda: gpu_ctx.scan_agg_host([files], bydb.Query([], usid, [("latency", O.AGG_SUM), ("calls", O.AGG_COUNT)], tmin=T0 + 100 * STEP, tmax=T0 + 2500 * STEP)),
    ]
    want = [f() for f in shapes]
    errors = []

    def worker(seed):
        r = np.random.default_rng(seed)
        try:
            for _ in range(25):
                k = int(r.integers(0, len(shapes)))
                got = shapes[k]()
                w = want[k]
                if not (got.group_id.tolist() == w.group_id.tolist() and got.rows.tolist() == w.rows.tolist()
                        and got.val_i64.tolist() == w.val_i64.tolist() and got.val_f64.view(np.uint64).tolist() == w.val_f64.view(np.uint64).tolist()):
                    errors.append(f"shape {k}: result differs under concurrency")
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))

    threads = [threading.Thread(target=worker, args=(s,)) for s in range(8)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    gpu_ctx.release_part(h)
    assert not errors, errors[:3]


def test_prepared_query_graph_replay_equals_scan_agg(bydb, gpu_ctx):
    # bydb_query_prepare / bydb_scan_agg_prepared: run 1 = ordinary path, run 2 = capture, runs 3.. = graph replays; every run must
    # return exactly what bydb_scan_agg returns, for a masked scalar query, a grouped Top-N and a fallback-page query
    rng = np.random.default_rng(88)
    part, sids, ts = _fallback_part(rng, n_series=4)
    usid = np.unique(sids)
    h = gpu_ctx.register_part(_next_pid(), part.files())
    groups = (np.arange(usid.size) % 2).astype(np.int32)
    queries = [
        bydb.Query([h], usid, [("raw", O.AGG_MAX), ("calls", O.AGG_COUNT)], preds=[bydb.Pred("default", "svc", O.OP_LE, b"service-name-030")],
                   tmin=T0 + 100 * STEP, tmax=T0 + 8500 * STEP),
        bydb.Query([h], usid, [("calls", O.AGG_SUM), ("latency", O.AGG_MIN)], series_group=groups, n_groups=2, top_n=1, top_desc=True),
        bydb.Query([h], usid, [("few", O.AGG_COUNT), ("raw", O.AGG_MEAN)]),
    ]
    try:
        for q in queries:
            want = gpu_ctx.scan_agg(q)
            g = gpu_ctx.prepare_graph(q)
            try:
                for run in range(6):
                    got = g.run()
                    assert got.group_id.tolist() == want.group_id.tolist() and got.rows.tolist() == want.rows.tolist(), run
                    assert got.val_i64.tolist() == want.val_i64.tolist(), run
                    assert got.val_f64.view(np.uint64).tolist() == want.val_f64.view(np.uint64).tolist(), run
                    assert got.stats.rows_scanned == want.stats.rows_scanned and got.stats.blocks_scanned == want.stats.blocks_scanned, run
            finally:
                g.close()
        # a device-side failure inside a replay is reported like on the ordinary path
        bad = bydb.Query([h], usid, [("calls", O.AGG_SUM)], preds=[bydb.Pred("default", "svc", O.OP_EQ, 5)])
        g = gpu_ctx.prepare_graph(bad)
        try:
            for run in range(4):
                with pytest.raises(bydb.BydbError) as ei:
                    g.run()
                assert ei.value.code == -22, run
        finally:
            g.close()
    finally:
        gpu_ctx.release_part(h)


def _c5_part(bydb, n_series, n_points, sid0=1):
    """BASELINE configs[4] shape (SURVEY.md 8d C5): 4 int64 fields (monotone delta / small fluctuations / random < 100 / counter with
    resets) + 4 float64 fields, two dictionary string tags and one int64 tag, from the product's synthetic generator."""
    from importlib import import_module
    S = import_module("bydb_b200.synth")
    fields = [("i_delta", S.I_DELTA), ("i_fluct", S.I_FLUCT), ("i_rand", S.I_RANDOM100), ("i_counter", S.I_COUNTER),
              ("latency", S.F_LATENCY), ("walk", S.F_WALK3), ("ints", S.F_INT1000), ("f_lat2", S.F_LATENCY)]
    return S.synth_part(n_series, n_points, fields, sid0=sid0, t0=T0, t_step=STEP, region_values=8, region_run=16, code_tag=True, zone_tag=True, seed=0xC5)


def test_c5_shape_three_conjunctive_predicates_eight_fields(bydb, gpu_ctx):
    # 1e6 datapoints, 8-field mixed int64 + float64 measure, region == "r3" AND zone != "z1" AND code >= 200 AND time range;
    # every aggregation function the reference has (pkg/query/aggregation/aggregation.go:63-82: there is no percentile) over the 8 fields
    n_series, n_points = 100, 10_000
    img = _c5_part(bydb, n_series, n_points)
    files = {k: v.tobytes() for k, v in img.files().items()}
    part = O.Part.open(files)
    usid = np.arange(1, n_series + 1, dtype=np.uint64)
    groups = ((usid - 1) % 10).astype(np.int32)
    names = ["i_delta", "i_fluct", "i_rand", "i_counter", "latency", "walk", "ints", "f_lat2"]
    preds = [O.Pred("default", "region", O.OP_EQ, b"r3"), O.Pred("default", "zone", O.OP_NE, b"z1"), O.Pred("default", "code", O.OP_GE, 200)]
    tmin, tmax = T0 + (n_points // 4) * STEP, T0 + (3 * n_points // 4) * STEP
    for funcs in ([O.AGG_SUM, O.AGG_COUNT], [O.AGG_MIN, O.AGG_MAX], [O.AGG_MEAN]):
        aggs = [(n, f) for n in names for f in funcs]
        oq = O.Query([part], usid, aggs, groups=groups, n_groups=10, tmin=tmin, tmax=tmax, preds=preds)
        h = gpu_ctx.register_part(_next_pid(), files)
        try:
            got = gpu_ctx.scan_agg(bydb.Query([h], usid, aggs, series_group=groups, n_groups=10, tmin=tmin, tmax=tmax,
                                              preds=[bydb.Pred(p.family, p.tag, p.op, p.value) for p in preds]))
        finally:
            gpu_ctx.release_part(h)
        want = O.run_query(oq)
        assert_parity(got, want, aggs, f"C5/{funcs}")
        assert got.stats.rows_matched == want.rows_matched and 0 < want.rows_matched < want.rows_scanned
    # the same shape without predicates and over the full range: the all-rows sum path over delta and delta-of-delta pages
    aggs = [(n, O.AGG_SUM) for n in names] + [("latency", O.AGG_COUNT)]
    oq = O.Query([part], usid, aggs, groups=groups, n_groups=10)
    h = gpu_ctx.register_part(_next_pid(), files)
    try:
        got = gpu_ctx.scan_agg(bydb.Query([h], usid, aggs, series_group=groups, n_groups=10))
    finally:
        gpu_ctx.release_part(h)
    assert_parity(got, O.run_query(oq), aggs, "C5/all-rows sums")


def test_hbm_budget_is_the_acquire_resource_mirror(bydb):
    # banyand/measure/query.go:608-633: the reference refuses a query whose blocks exceed the protector's quota; the library's mirror is
    # bydb_cfg.hbm_budget_bytes -> BYDB_ENOMEM at part admission (resident parts) and inside bydb_scan_agg_host (transient parts)
    rng = np.random.default_rng(5)
    sids, ts, ver = grid(8, 4000)
    lat = np.round(rng.normal(30, 6, sids.size), 2)
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None)])
    files = part.files()
    size = sum(len(v) for v in files.values())
    q = lambda h: bydb.Query(h, np.unique(sids), [("latency", O.AGG_SUM)])  # noqa: E731
    with bydb.Context(device=0, hbm_budget_bytes=size // 2) as small:
        with pytest.raises(bydb.BydbError) as ei:
            small.register_part(1, files)
        assert ei.value.code == bydb.capi.ENOMEM and "budget" in ei.value.msg
        with pytest.raises(bydb.BydbError) as ei:
            small.scan_agg_host([files], q([]))
        assert ei.value.code == bydb.capi.ENOMEM
    with bydb.Context(device=0) as probe:
        per = probe.part_info(probe.register_part(1, files))["hbm_bytes"]     # what one resident copy of this part accounts for
    with bydb.Context(device=0, hbm_budget_bytes=int(3.5 * per)) as roomy:
        h1 = roomy.register_part(1, files)
        info = roomy.part_info(h1)
        assert info["hbm_bytes"] == per
        want = roomy.scan_agg(q([h1]))
        # the budget is an account, not a high-water mark: releasing gives the bytes back, and a failed admission leaves nothing behind
        for i in range(6):
            h2 = roomy.register_part(100 + i, files)
            roomy.release_part(h2)
        got = roomy.scan_agg_host([files], q([]))
        assert got.val_f64.tolist() == want.val_f64.tolist()
        h3 = roomy.register_part(2, files)
        with pytest.raises(bydb.BydbError) as ei:
            for i in range(8):
                roomy.register_part(200 + i, files)
        assert ei.value.code == bydb.capi.ENOMEM
        assert roomy.scan_agg(q([h1, ])).val_f64.tolist() == want.val_f64.tolist()
        roomy.release_part(h3)


def _comm_pair(bydb, n_ranks, devices):
    """n contexts (one per rank) with their mailboxes connected; same process, so the handles carry plain pointers."""
    ctxs = [bydb.Context(device=d) for d in devices]
    handles = [c.comm_export(1 << 20, n_ranks) for c in ctxs]
    for r, c in enumerate(ctxs):
        c.comm_connect(r, n_ranks, handles)
    return ctxs


def test_scan_reduce_peer_mailboxes_equal_the_single_context_answer(bydb, gpu_ctx):
    # bydb_comm_export / _connect / bydb_scan_reduce: the series of one measure sharded over R ranks (R contexts; on a one-GPU box
    # they share the device, on a multi-GPU box each takes its own), every rank scans its shard and writes its partial table into
    # the root's mailbox, the root combines in rank order and finalises -- the liaison reduce of measure_plan_aggregation.go:96-124.
    # Must equal one context scanning everything, for grouped Top-N, MEAN / MIN / MAX finalisation and a rank without matching rows.
    import faulthandler
    import gc
    import threading
    import torch
    n_dev = torch.cuda.device_count()
    # On a one-GPU box the ranks share the device.  A finaliser of some earlier test's object (a prepared query, a context) that runs
    # on a rank's thread in the middle of a collective frees page-locked memory -- an implicit device synchronisation that waits for
    # the peers' spinning wait kernels, i.e. for the very rank that is stuck in it.  Nothing unrelated may be torn down here.
    gc.collect()
    gc.disable()
    faulthandler.dump_traceback_later(25, exit=False)   # a stalled collective shows where every thread sits
    try:
        _scan_reduce_body(bydb, gpu_ctx, threading, n_dev)
    finally:
        faulthandler.cancel_dump_traceback_later()
        gc.enable()


def _scan_reduce_body(bydb, gpu_ctx, threading, n_dev):
    rng = np.random.default_rng(314)
    R = 3
    sids, ts, ver = grid(30, 2600)
    lat = np.round(rng.normal(30, 6, sids.size), 2)
    calls = rng.integers(-50, 500, sids.size)
    region = [b"r%d" % v for v in rng.integers(0, 4, sids.size)]
    usid = np.unique(sids)
    shard_of = (np.arange(usid.size) * R) // usid.size
    parts = []
    for r in range(R):
        m = np.isin(sids, usid[shard_of == r])
        parts.append(build_part(sids[m], ts[m], ver[m], [("latency", O.VT_FLOAT64, lat[m], None), ("calls", O.VT_INT64, calls[m], None)],
                                [("default", [("region", O.VT_STR, [x for x, k in zip(region, m) if k], None)])]))
    groups = (np.arange(usid.size) % 7).astype(np.int32)
    queries = [
        dict(aggs=[("latency", O.AGG_SUM), ("latency", O.AGG_COUNT)], top_n=3, top_agg=0, top_desc=True),
        dict(aggs=[("latency", O.AGG_MEAN), ("calls", O.AGG_MIN), ("calls", O.AGG_MAX), ("latency", O.AGG_MAX), ("calls", O.AGG_MEAN)],
             preds=[bydb.Pred("default", "region", O.OP_EQ, b"r2")], tmin=T0 + 200 * STEP, tmax=T0 + 2300 * STEP),
        dict(aggs=[("calls", O.AGG_SUM)], tmin=T0 + 10 * STEP, tmax=T0 + 20 * STEP),
    ]
    whole = [gpu_ctx.register_part(_next_pid(), p.files()) for p in parts]
    ctxs = _comm_pair(bydb, R, [r % n_dev for r in range(R)])
    try:
        hs = [c.register_part(1, p.files()) for c, p in zip(ctxs, parts)]
        for root in (0, 2):
            for kw in queries:
                want = gpu_ctx.scan_agg(bydb.Query(whole, usid, series_group=groups, n_groups=7, **kw))
                got, errs = [None] * R, []

                def run(r):
                    try:
                        mine = shard_of == r
                        got[r] = ctxs[r].scan_reduce(bydb.Query([hs[r]], usid[mine], series_group=groups[mine], n_groups=7, **kw), root=root)
                    except Exception as e:  # noqa: BLE001
                        errs.append(repr(e))
                th = [threading.Thread(target=run, args=(r,)) for r in range(R)]
                for t in th:
                    t.start()
                for t in th:
                    t.join()
                assert not errs, errs
                g = got[root]
                assert g.group_id.tolist() == want.group_id.tolist() and g.rows.tolist() == want.rows.tolist()
                assert g.val_i64.tolist() == want.val_i64.tolist()
                assert np.allclose(g.val_f64, want.val_f64, rtol=1e-12, atol=0)
                for r in range(R):
                    if r != root:
                        assert got[r].group_id.size == 0 and got[r].stats.blocks_scanned > 0
        # the collective as a prepared query (bydb_scan_reduce_prepared): run 1 plain, then one captured graph per (root, slot parity);
        # ranks 0 and 1 use the prepared form, rank 2 keeps calling bydb_scan_reduce -- the two mix within one collective
        for kw in (queries[0], queries[1]):
            want = gpu_ctx.scan_agg(bydb.Query(whole, usid, series_group=groups, n_groups=7, **kw))
            qs = [bydb.Query([hs[r]], usid[shard_of == r], series_group=groups[shard_of == r], n_groups=7, **kw) for r in range(R)]
            gqs = [ctxs[r].prepare_graph(qs[r]) for r in range(2)]
            try:
                for it in range(7):
                    root = it % 2
                    got, errs = [None] * R, []

                    def run_p(r):
                        try:
                            got[r] = gqs[r].run_reduce(root=root) if r < 2 else ctxs[r].scan_reduce(qs[r], root=root)
                        except Exception as e:  # noqa: BLE001
                            errs.append(repr(e))
                    th = [threading.Thread(target=run_p, args=(r,)) for r in range(R)]
                    for t in th:
                        t.start()
                    for t in th:
                        t.join()
                    assert not errs, (it, errs)
                    g = got[root]
                    assert g.group_id.tolist() == want.group_id.tolist() and g.rows.tolist() == want.rows.tolist(), it
                    assert g.val_i64.tolist() == want.val_i64.tolist() and np.allclose(g.val_f64, want.val_f64, rtol=1e-12, atol=0), it
                    assert got[1 - root].group_id.size == 0 and got[1 - root].stats.blocks_scanned > 0
            finally:
                for gq in gqs:
                    gq.close()
        # the same collective with HOST file images on every rank (bydb_scan_reduce_host: the cold distributed query, end to end)
        kw = queries[1]
        want = gpu_ctx.scan_agg(bydb.Query(whole, usid, series_group=groups, n_groups=7, **kw))
        got, errs = [None] * R, []

        def run_host(r):
            try:
                mine = shard_of == r
                got[r] = ctxs[r].scan_reduce_host([parts[r].files()], bydb.Query([], usid[mine], series_group=groups[mine], n_groups=7, **kw), root=1)
            except Exception as e:  # noqa: BLE001
                errs.append(repr(e))
        th = [threading.Thread(target=run_host, args=(r,)) for r in range(R)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        assert not errs, errs
        assert got[1].group_id.tolist() == want.group_id.tolist() and got[1].val_i64.tolist() == want.val_i64.tolist()
        assert np.allclose(got[1].val_f64, want.val_f64, rtol=1e-12, atol=0) and got[1].stats.h2d_bytes > 0
        # a device-side failure on ONE rank (predicate literal of the wrong type) fails the root's call with that error
        res = [None] * R

        def run_bad(r):
            preds = [bydb.Pred("default", "region", O.OP_EQ, 5)] if r == 1 else []
            mine = shard_of == r
            try:
                ctxs[r].scan_reduce(bydb.Query([hs[r]], usid[mine], [("calls", O.AGG_SUM)], preds=preds), root=0)
                res[r] = 0
            except bydb.BydbError as e:
                res[r] = e.code
        th = [threading.Thread(target=run_bad, args=(r,)) for r in range(R)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        assert res[0] == -22 and res[1] == -22 and res[2] == 0, res
        # and the mailboxes stay usable afterwards
        got = [None] * R

        def run_ok(r):
            mine = shard_of == r
            got[r] = ctxs[r].scan_reduce(bydb.Query([hs[r]], usid[mine], [("calls", O.AGG_SUM)]), root=0)
        th = [threading.Thread(target=run_ok, args=(r,)) for r in range(R)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        assert int(got[0].val_i64[0, 0]) == int(calls.sum())
    finally:
        for c in ctxs:
            c.close()
        for h in whole:
            gpu_ctx.release_part(h)


def test_partial_rows_in_the_reference_wire_shape(bydb, gpu_ctx):
    # a18 / f3: bydb_partials_rows turns a data node's partial table into the rows mapAccumulator.Result(emitPartial) ships
    # (Partial.Value, + Partial.Count as "__agg_count" for MEAN; everything N-typed by the field, function.go:42-44,91-93,129-131,
    # 169-171,211-213).  Two "data nodes" (two shards of the series); the liaison's reduceAccumulator.Combine + Val()
    # (function.go:57-71,104-110,142-148,182-190,224-232), restated here in a few lines, must reproduce the oracle's whole-query answer.
    import torch
    rng = np.random.default_rng(2718)
    sids, ts, ver = grid(24, 1500)
    lat = np.round(rng.normal(0.4, 0.3, sids.size), 2)        # means below 1: the MEAN clamp of function.go:31-40 matters
    calls = rng.integers(-20, 90, sids.size)
    usid = np.unique(sids)
    groups = (np.arange(usid.size) % 5).astype(np.int32)
    aggs = [("latency", O.AGG_MEAN), ("latency", O.AGG_COUNT), ("latency", O.AGG_MAX), ("calls", O.AGG_MEAN), ("calls", O.AGG_MIN), ("calls", O.AGG_SUM),
            ("calls", O.AGG_COUNT), ("latency", O.AGG_SUM), ("latency", O.AGG_MIN), ("calls", O.AGG_MAX)]
    shards = [usid[:9], usid[9:]]     # group 4 has no series in ... both shards hold every group; a time range empties some
    tmin, tmax = T0 + 100 * STEP, T0 + 1200 * STEP
    whole = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None), ("calls", O.VT_INT64, calls, None)])
    want = O.run_query(O.Query([whole], usid, aggs, groups=groups, n_groups=5, tmin=tmin, tmax=tmax))
    node_rows = []
    for sh in shards:
        m = np.isin(sids, sh)
        part = build_part(sids[m], ts[m], ver[m], [("latency", O.VT_FLOAT64, lat[m], None), ("calls", O.VT_INT64, calls[m], None)])
        h = gpu_ctx.register_part(_next_pid(), part.files())
        try:
            q = bydb.Query([h], sh, aggs, series_group=groups[np.isin(usid, sh)], n_groups=5, tmin=tmin, tmax=tmax)
            lay = gpu_ctx.partials_layout(q)
            table = torch.zeros(lay["total_bytes"] // 8, dtype=torch.float64, device="cuda")
            gpu_ctx.scan_partials(q, table.data_ptr(), lay["total_bytes"], torch.cuda.current_stream().cuda_stream)
            rows = gpu_ctx.partials_rows(q, table.data_ptr(), lay["total_bytes"], torch.cuda.current_stream().cuda_stream)
            # the map rows of one node against the oracle run on that node's part alone: Value / Count per function
            own_parts = [O.run_query(O.Query([part], sh, [(f, fn) for fn in (O.AGG_SUM, O.AGG_COUNT, O.AGG_MAX, O.AGG_MIN)], groups=groups[np.isin(usid, sh)],
                                             n_groups=5, tmin=tmin, tmax=tmax)) for f, _ in aggs]

            class own:   # the per-aggregate oracle runs side by side: columns 4a .. 4a+3 belong to aggregate a
                group_id = own_parts[0].group_id
                val_i64 = np.concatenate([o.val_i64 for o in own_parts], axis=1)
                val_f64 = np.concatenate([o.val_f64 for o in own_parts], axis=1)
            assert rows["group_id"].tolist() == own.group_id.tolist()
            assert rows["is_float"].tolist() == [f == "latency" for f, _ in aggs]     # N-typed: COUNT over a float field is a float
            for a, (f, fn) in enumerate(aggs):
                isf = f == "latency"
                got_v = rows["val_f64"][:, a] if isf else rows["val_i64"][:, a]
                got_c = rows["cnt_f64"][:, a] if isf else rows["cnt_i64"][:, a]
                o_sum = own.val_f64[:, 4 * a] if isf else own.val_i64[:, 4 * a]
                o_cnt, o_max, o_min = own.val_i64[:, 4 * a + 1], (own.val_f64 if isf else own.val_i64)[:, 4 * a + 2], (own.val_f64 if isf else own.val_i64)[:, 4 * a + 3]
                exp_v = {O.AGG_SUM: o_sum, O.AGG_MEAN: o_sum, O.AGG_COUNT: o_cnt.astype(got_v.dtype), O.AGG_MAX: o_max, O.AGG_MIN: o_min}[fn]
                if isf and fn in (O.AGG_SUM, O.AGG_MEAN):
                    assert np.allclose(got_v, exp_v, rtol=1e-9, atol=0), (a, got_v, exp_v)
                else:
                    assert got_v.tolist() == exp_v.tolist(), (a, got_v, exp_v)
                assert got_c.tolist() == (o_cnt.astype(got_c.dtype).tolist() if fn == O.AGG_MEAN else [0] * len(got_c)), a
            node_rows.append(rows)
        finally:
            gpu_ctx.release_part(h)
    # liaison: reduceAccumulator.Combine over the nodes' rows, then Val()
    for gi, g in enumerate(want.group_id.tolist()):
        for a, (f, fn) in enumerate(aggs):
            isf = f == "latency"
            parts = []
            for rows in node_rows:
                k = np.nonzero(rows["group_id"] == g)[0]
                if k.size:
                    parts.append(((rows["val_f64"] if isf else rows["val_i64"])[k[0], a].item(), (rows["cnt_f64"] if isf else rows["cnt_i64"])[k[0], a].item()))
            assert parts
            if fn == O.AGG_MEAN:
                s_, c_ = sum(p[0] for p in parts), sum(p[1] for p in parts)
                val = 0 if c_ == 0 else (s_ / c_ if isf else int(s_ / c_))
                val = 1 if (c_ != 0 and val < 1) else val
            elif fn in (O.AGG_SUM, O.AGG_COUNT):
                val = sum(p[0] for p in parts)
            elif fn == O.AGG_MAX:
                val = max(p[0] for p in parts)
            else:
                val = min(p[0] for p in parts)
            ref = want.val_f64[gi, a] if want.is_float[a] else want.val_i64[gi, a]
            if isf and fn in (O.AGG_SUM, O.AGG_MEAN):
                assert abs(val - ref) <= 1e-9 * max(abs(ref), 1e-300), (g, a, val, ref)
            else:
                assert val == ref, (g, a, fn, val, ref)     # COUNT over a float field: 1380.0 == 1380 (vec types it int64, the row path float)


def test_gather_path_for_pageable_host_images(bydb, gpu_ctx):
    # bydb_scan_agg_host on PAGEABLE images (BanyanDB's mmap'd part files are not pinned): the host selects the blocks like plan_blocks
    # and stages only the pages the query reads, in 64 MB chunks through a pinned ring.  3e7 datapoints x 2 touched fields = more
    # than one chunk; a series subset + time range + predicate exercises the block selection and the rewritten page offsets.
    from importlib import import_module
    S = import_module("bydb_b200.synth")
    n_series, n_points = 300, 100_000
    img = S.synth_part(n_series, n_points, [("latency", S.F_LATENCY), ("walk", S.F_WALK3), ("ints", S.F_INT1000)], sid0=1, t0=T0, t_step=STEP,
                       region_values=8, region_run=16, seed=0x6A7)
    files = img.files()
    usid = np.arange(1, n_series + 1, dtype=np.uint64)
    groups = ((usid - 1) % 11).astype(np.int32)
    h = gpu_ctx.register_part(_next_pid(), files)
    try:
        cases = [
            dict(series=usid, kw=dict(aggs=[("latency", O.AGG_SUM), ("walk", O.AGG_MAX), ("latency", O.AGG_COUNT)], series_group=groups, n_groups=11)),
            dict(series=usid[5::3], kw=dict(aggs=[("walk", O.AGG_MEAN), ("ints", O.AGG_MIN)], series_group=groups[5::3], n_groups=11,
                                            tmin=T0 + 20_000 * STEP + 7, tmax=T0 + 71_234 * STEP, preds=[bydb.Pred("default", "region", O.OP_NE, b"r5")])),
            dict(series=np.array([400, 500], dtype=np.uint64), kw=dict(aggs=[("latency", O.AGG_SUM)])),   # selects nothing at all
        ]
        for c in cases:
            want = gpu_ctx.scan_agg(bydb.Query([h], c["series"], **c["kw"]))
            got = gpu_ctx.scan_agg_host([files], bydb.Query([], c["series"], **c["kw"]))
            assert got.group_id.tolist() == want.group_id.tolist() and got.rows.tolist() == want.rows.tolist()
            assert got.is_float.tolist() == want.is_float.tolist() and got.val_i64.tolist() == want.val_i64.tolist()
            assert np.allclose(got.val_f64, want.val_f64, rtol=1e-12, atol=0)
            assert got.stats.rows_scanned == want.stats.rows_scanned and got.stats.page_bytes == want.stats.page_bytes
            total = sum(v.size for v in files.values())
            assert got.stats.h2d_bytes < 0.8 * total, "only the touched pages may travel"
    finally:
        gpu_ctx.release_part(h)


def test_row_path_result_typing_flag(bydb, gpu_ctx):
    # a14 / a15: the reference's ROW path types every aggregate like its field -- countFunc[N] is N-typed (function.go:78-93,
    # measure_plan_aggregation.go:152-175): COUNT over a float64 field is a float64; the vectorized path types COUNT int64
    # (aggregation.go:425-430, the default here).  BYDB_Q_ROW_PATH_TYPES selects the former; values are the same numbers.
    from bydb_b200.capi import Q_ROW_PATH_TYPES
    rng = np.random.default_rng(99)
    sids, ts, ver = grid(6, 700)
    lat = np.round(rng.normal(30, 6, sids.size), 2)
    calls = rng.integers(0, 50, sids.size)
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None), ("calls", O.VT_INT64, calls, None)])
    h = gpu_ctx.register_part(_next_pid(), part.files())
    try:
        aggs = [("latency", O.AGG_COUNT), ("calls", O.AGG_COUNT), ("latency", O.AGG_MEAN), ("calls", O.AGG_SUM)]
        vec = gpu_ctx.scan_agg(bydb.Query([h], np.unique(sids), aggs))
        row = gpu_ctx.scan_agg(bydb.Query([h], np.unique(sids), aggs, flags=Q_ROW_PATH_TYPES))
        assert vec.is_float.tolist() == [False, False, True, False] and row.is_float.tolist() == [True, False, True, False]
        assert float(row.val_f64[0, 0]) == float(vec.val_i64[0, 0]) == sids.size
        assert row.val_i64[0, 1] == vec.val_i64[0, 1] and row.val_f64[0, 2] == vec.val_f64[0, 2] and row.val_i64[0, 3] == vec.val_i64[0, 3]
    finally:
        gpu_ctx.release_part(h)


def test_block_index_decoded_on_the_device_equals_the_host_parser(bydb):
    # f1: bydb_part_register inflates meta.bin / primary.bin with the device zstd decoder and walks the blockMetadata records in
    # kernels (index_kernels.cu; part_iter.go:184-208, block_metadata.go:133-168, column_metadata.go:108-122, primary_metadata.go:47-83).
    # The directory it builds must be the host parser's (csrc/part_dir.cc, BYDB_CFG_HOST_INDEX) byte for byte, up to the numbering
    # of the interned column names (an arbitrary per-context id): many primary blocks, several tag columns, fallback pages, nulls.
    from importlib import import_module
    S = import_module("bydb_b200.synth")
    rng = np.random.default_rng(1234)
    parts = {}
    keep = [S.synth_part(6000, 40, [("latency", S.F_LATENCY), ("calls", S.I_FLUCT)], sid0=7, sid_step=2, t0=T0, t_step=STEP, region_values=8,
                         region_run=4, code_tag=True, zone_tag=True, seed=5), _c5_part(bydb, 40, 20_000)]   # files() are views into the images
    parts["many primary blocks"] = keep[0].files()
    parts["eight fields, long blocks"] = keep[1].files()
    fb, _, _ = _fallback_part(rng, n_series=3)
    parts["fallback pages"] = fb.files()
    sids, ts, ver = grid(5, 300)
    parts["no tags"] = build_part(sids, ts, ver, [("v", O.VT_INT64, rng.integers(0, 9, sids.size), None)]).files()
    col_dt = np.dtype([("off", "<u8"), ("size", "<u4"), ("name_id", "<u2"), ("value_type", "u1"), ("file_id", "u1")])
    with bydb.Context(device=0, host_index=True) as host, bydb.Context(device=0) as dev:
        for name, files in parts.items():
            hh, hd = host.register_part(1, files), dev.register_part(1, files)
            try:
                hb, hc = host.part_directory(hh)
                db, dc = dev.part_directory(hd)
                assert hb.shape == db.shape and hb.shape[0] > 0, name
                assert (hb == db).all(), f"{name}: DevBlock records differ"
                hcv, dcv = hc.view(col_dt).reshape(-1), dc.view(col_dt).reshape(-1)
                for f in ("size", "value_type", "file_id"):
                    assert (hcv[f] == dcv[f]).all(), f"{name}: DevCol.{f} differs"
                # pages unpacked at admission live in a side arena whose slots are handed out by an atomic counter: their offsets are
                # not reproducible from one registration to the next, everything else is
                in_arena = (hcv["file_id"] == hcv["file_id"].max()) if host.part_info(hh)["fallback_unpacked"] else np.zeros(hcv.size, bool)
                assert ((hcv["off"] == dcv["off"]) | in_arena).all(), f"{name}: DevCol.off differs"
                pairs = set(zip(hcv["name_id"].tolist(), dcv["name_id"].tolist()))
                assert len(pairs) == len({a for a, _ in pairs}) == len({b for _, b in pairs}), f"{name}: name ids are not a relabelling"
                assert host.part_info(hh) == dev.part_info(hd), name
                # and the scans agree
                usid = np.unique(hb[:, :8].copy().view("<u8").reshape(-1))
                fld = "latency" if name != "no tags" and name != "fallback pages" else ("v" if name == "no tags" else "calls")
                q = lambda h: bydb.Query([h], usid, [(fld, O.AGG_SUM), (fld, O.AGG_MAX), (fld, O.AGG_COUNT)])  # noqa: E731
                a, b = host.scan_agg(q(hh)), dev.scan_agg(q(hd))
                assert a.val_i64.tolist() == b.val_i64.tolist() and a.val_f64.view(np.uint64).tolist() == b.val_f64.view(np.uint64).tolist(), name
            finally:
                host.release_part(hh)
                dev.release_part(hd)
        # a corrupt index fails on the device like on the host: truncated primary.bin, garbage meta.bin
        files = dict(parts["no tags"])
        bad = dict(files)
        bad["primary.bin"] = bytes(files["primary.bin"])[:-7]
        for ctx in (host, dev):
            with pytest.raises(bydb.BydbError) as ei:
                ctx.register_part(9, bad)
            assert ei.value.code == -22
        bad = dict(files)
        bad["meta.bin"] = b"\x28\xb5\x2f\xfd" + bytes(20)
        for ctx in (host, dev):
            with pytest.raises(bydb.BydbError):
                ctx.register_part(9, bad)
            h = ctx.register_part(10, files)   # and the context is still usable
            ctx.release_part(h)


def _keyed_both(bydb, gpu_ctx, parts, oq, family, tag, max_values=0):
    from tests.helpers import to_gpu_query
    pid0 = _next_pid()
    handles = [gpu_ctx.register_part(pid0 + i, p.files()) for i, p in enumerate(parts)]
    try:
        got = gpu_ctx.scan_agg_keyed(to_gpu_query(bydb, handles, oq), family, tag, max_values)
    finally:
        for h in handles:
            gpu_ctx.release_part(h)
    import dataclasses
    want = O.run_query(dataclasses.replace(oq, group_key=(family, tag)))
    return got, want


def test_group_by_stored_tag_insertion_order_and_topn(bydb, gpu_ctx):
    # a12: the group key is a stored dictionary tag, so it changes from row to row (aggregation.go:193-254); nil and "" are one key
    rng = np.random.default_rng(0xA12)
    sids, ts, ver = grid(23, 9000, sid0=3, sid_step=2)   # 8193-row block + a tail block per series
    n = sids.size
    lat = np.round(25 + rng.normal(0, 5, n), 2)
    calls = rng.integers(-5000, 5000, n)
    code = rng.integers(0, 4, n) * 100
    # runs of equal values of random length (what RLE dictionary pages hold), a few nil and "" cells, one value only late in time
    region = []
    while len(region) < n:
        v = rng.integers(0, 7)
        region.extend([b"region-%d" % v] * int(rng.integers(1, 40)))
    region = region[:n]
    for i in range(0, n, 977):
        region[i] = None
    for i in range(5, n, 1409):
        region[i] = b""
    for s in range(23):
        region[s * 9000 + 8800: s * 9000 + 8810] = [b"late"] * 10
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None), ("calls", O.VT_INT64, calls, None)],
                      [("default", [("region", O.VT_STR, region, None), ("code", O.VT_INT64, code, None)])])
    usid = np.unique(sids)
    groups = (np.arange(usid.size) % 3).astype(np.int32)
    aggs = [("latency", O.AGG_SUM), ("latency", O.AGG_MAX), ("calls", O.AGG_SUM), ("calls", O.AGG_MIN), ("calls", O.AGG_COUNT),
            ("latency", O.AGG_MEAN)]
    oq = O.Query([part], usid, aggs, groups=groups, n_groups=3, tmin=T0 + 100 * STEP, tmax=T0 + 8900 * STEP,
                 preds=[O.Pred("default", "code", O.OP_NE, 300)])
    got, want = _keyed_both(bydb, gpu_ctx, [part], oq, "default", "region")
    assert got.key == want.key, "key values in insertion order"
    assert_parity(got, want, aggs, "keyed")
    assert b"" in got.key and b"late" in got.key and len(got.key) == 3 * 9
    # no series groups: pure group-by-tag
    oq1 = O.Query([part], usid[::2], [("calls", O.AGG_SUM), ("calls", O.AGG_COUNT)], tmin=T0 + 50 * STEP, tmax=T0 + 8700 * STEP)
    got, want = _keyed_both(bydb, gpu_ctx, [part], oq1, "default", "region")
    assert got.key == want.key and b"late" not in got.key
    assert_parity(got, want, oq1.aggs, "keyed, one series group")
    # Top-N over the composite groups, both directions; COUNT ties go to the group inserted first
    for desc in (True, False):
        oqt = O.Query([part], usid, [("calls", O.AGG_COUNT), ("latency", O.AGG_MAX)], groups=groups, n_groups=3, top_n=7, top_agg=0,
                      top_desc=desc)
        got, want = _keyed_both(bydb, gpu_ctx, [part], oqt, "default", "region")
        assert got.key == want.key
        assert_parity(got, want, oqt.aggs, f"keyed top desc={desc}")
    # two parts that follow each other in time: a value that first shows in the second part is inserted later
    half = ts < T0 + 4000 * STEP
    pa = build_part(sids[half], ts[half], ver[half], [("calls", O.VT_INT64, calls[half], None)],
                    [("default", [("region", O.VT_STR, [r for r, h in zip(region, half) if h], None)])])
    pb = build_part(sids[~half], ts[~half], ver[~half], [("calls", O.VT_INT64, calls[~half], None)],
                    [("default", [("region", O.VT_STR, [r for r, h in zip(region, half) if not h], None)])])
    oq2 = O.Query([pa, pb], usid, [("calls", O.AGG_SUM), ("calls", O.AGG_MAX)], groups=groups, n_groups=3)
    got, want = _keyed_both(bydb, gpu_ctx, [pa, pb], oq2, "default", "region")
    assert got.key == want.key
    assert_parity(got, want, oq2.aggs, "keyed, two parts")
    # a tag no block stores: every cell is nil -> the single key ""
    got, want = _keyed_both(bydb, gpu_ctx, [part], oq1, "default", "nosuchtag")
    assert got.key == want.key == [b""]
    assert_parity(got, want, oq1.aggs, "keyed, absent tag")
    # nothing selected
    oq0 = O.Query([part], np.array([999999], dtype=np.uint64), [("calls", O.AGG_SUM)])
    got, want = _keyed_both(bydb, gpu_ctx, [part], oq0, "default", "region")
    assert got.key == want.key == [] and got.rows.size == 0


def test_group_by_stored_tag_limits(bydb, gpu_ctx):
    rng = np.random.default_rng(7)
    sids, ts, ver = grid(4, 3000)
    n = sids.size
    calls = rng.integers(0, 100, n)
    region = [b"r%d" % v for v in rng.integers(0, 12, n)]
    longv = [b"x" * 70 if i % 500 == 0 else b"ok" for i in range(n)]
    code = rng.integers(0, 4, n)
    part = build_part(sids, ts, ver, [("calls", O.VT_INT64, calls, None)],
                      [("default", [("region", O.VT_STR, region, None), ("long", O.VT_STR, longv, None), ("code", O.VT_INT64, code, None)])])
    h = gpu_ctx.register_part(_next_pid(), part.files())
    try:
        q = bydb.Query(parts=[h], series_ids=np.unique(sids), aggs=[("calls", O.AGG_SUM)])
        with pytest.raises(bydb.BydbError) as e:
            gpu_ctx.scan_agg_keyed(q, "default", "region", max_values=8)   # 12 distinct values
        assert e.value.code == bydb.capi.ENOMEM
        assert len(gpu_ctx.scan_agg_keyed(q, "default", "region", max_values=12).key) == 12
        with pytest.raises(bydb.BydbError) as e:
            gpu_ctx.scan_agg_keyed(q, "default", "long")
        assert e.value.code == bydb.capi.ENOTSUP
        with pytest.raises(bydb.BydbError) as e:
            gpu_ctx.scan_agg_keyed(q, "default", "code")                   # an int64 tag is not a dictionary page
        assert e.value.code == bydb.capi.EINVAL
        with pytest.raises(bydb.BydbError) as e:
            gpu_ctx.scan_agg_keyed(q, "default", "region", max_values=1000)
        assert e.value.code == bydb.capi.EINVAL
        # the context is still healthy
        assert gpu_ctx.scan_agg(q).val_i64[0, 0] == int(calls.sum())
    finally:
        gpu_ctx.release_part(h)


def _oracle_numeric_page(values: np.ndarray) -> bytes:
    if values.dtype == np.float64:
        raw = values.astype(">f8").tobytes()
        vt = O.VT_FLOAT64
    else:
        raw = (values.astype(np.int64).view(np.uint64) ^ np.uint64(1 << 63)).astype(">u8").tobytes()
        vt = O.VT_INT64
    return O.column_encode(vt, [raw[8 * i:8 * i + 8] for i in range(values.size)])


def _int_blocks(rng):
    i64 = np.iinfo(np.int64)
    n = 1500
    t = np.arange(n, dtype=np.int64)
    resets = np.cumsum(rng.integers(1, 10, n)).astype(np.int64)
    resets[700:] -= resets[700] - 3       # a counter that restarts once: still "incremental" (int_list.go:150-179)
    many = np.cumsum(rng.integers(1, 10, n)).astype(np.int64) % 50   # restarts all the time: plain delta
    return [np.full(n, 42, np.int64), np.array([-7], np.int64), np.array([5, 9], np.int64), t * 60_000_000_000 + 1_700_000_000_000_000_000,
            t * -7 + 100, np.cumsum(rng.integers(0, 10, n)).astype(np.int64), -np.cumsum(rng.integers(0, 10, n)).astype(np.int64) - 5,
            resets, many, rng.integers(-1000, 1000, n).astype(np.int64), rng.integers(i64.min, i64.max, n, dtype=np.int64, endpoint=True),
            np.array([i64.min, i64.max, 0, -1, i64.max, i64.min], np.int64), np.array([3, 3, 3, 4], np.int64),
            np.array([10, 8, 6, 4, 2, 0, -2], np.int64), rng.integers(0, 100, 8193).astype(np.int64), 25 + np.cumsum(rng.integers(-5, 6, 8193)).astype(np.int64),
            np.array([0, 1 << 62, -(1 << 62), 1 << 62], np.int64)]


def _float_blocks(rng):
    n = 1200
    return [np.round(25 + rng.normal(0, 5, n), 2), np.round(np.cumsum(rng.uniform(-0.1, 0.1, n)) + 50, 3), rng.integers(0, 1000, n).astype(np.float64),
            np.full(n, 0.5), np.array([0.0, -0.0, 1.5, -2.25, 1e6, 120.0, 3e-7]), np.round(rng.uniform(-1e6, 1e6, n), 6),
            rng.integers(-50, 50, n) * 1000.0, np.array([1e15, 123456789012345.0, 0.001]), np.round(rng.uniform(0, 1, n), 15),
            np.array([1e300, 1.0]),                         # common exponent overflows -> CPU (the fallback page)
            rng.uniform(0, 100, n),                         # full precision: the general shortest-digits search -> CPU
            np.array([1.0, np.nan]), np.array([np.inf, 2.0]), np.array([0.1 + 0.2, 1.0]), np.array([9007199254740993.0, 2.0 ** 63, -2.0 ** 63, 2.0 ** 70])]


def test_device_page_encoder_matches_the_reference_writer(bydb, gpu_ctx):
    # f4: fv.bin pages of numeric field blocks encoded on the device, byte for byte the writer's (column.go:113-234)
    rng = np.random.default_rng(0xF4)
    for blocks, kind in ((_int_blocks(rng), "int64"), (_float_blocks(rng), "float64")):
        values = np.concatenate(blocks)
        pages, ms = gpu_ctx.encode_pages(values, [b.size for b in blocks])
        assert len(pages) == len(blocks) and ms >= 0
        n_cpu = 0
        for i, (blk, page) in enumerate(zip(blocks, pages)):
            want = _oracle_numeric_page(blk)
            if page is None:
                n_cpu += 1
                assert kind == "float64", f"{kind} block {i} was left to the CPU"
                continue
            assert page == want, f"{kind} block {i}: {page[:24].hex()} vs {want[:24].hex()} (len {len(page)} vs {len(want)})"
            assert page[0] in (1, 2, 3, 4)
        if kind == "float64":
            # what the device declined: overflow on the common exponent, full-precision values, NaN, Inf, 0.1+0.2 and the 17-digit integers
            assert 3 <= n_cpu <= 7, n_cpu
    # a whole synthetic column: every block of the bench generators is encoded on the device and decodes back
    sids, ts, ver = grid(12, 9000)
    lat = np.round(25 + rng.normal(0, 5, sids.size), 2)
    rows = [8193, 807] * 12
    pages, _ = gpu_ctx.encode_pages(lat, rows)
    off = 0
    for r, page in zip(rows, pages):
        assert page is not None and page == _oracle_numeric_page(lat[off:off + r])
        off += r
    pages, _ = gpu_ctx.encode_pages(np.zeros(0, np.int64), [])
    assert pages == []
    with pytest.raises(bydb.BydbError):
        gpu_ctx.encode_pages(np.zeros(3, np.int64), [0, 3])   # a block without rows


@pytest.mark.parametrize("seed", range(10))
def test_random_sweep_stored_tag_group_by(bydb, gpu_ctx, seed):
    # randomised a12 queries: key cardinality, run lengths, nil cells, series groups, predicates, ranges, aggregates, Top-N
    rng = np.random.default_rng(0xA1200 + seed)
    n_series, n_pts = int(rng.integers(3, 18)), int(rng.integers(200, 9500))
    sids, ts, ver = grid(n_series, n_pts, sid0=int(rng.integers(1, 50)), sid_step=int(rng.integers(1, 4)))
    n = sids.size
    lat = np.round(rng.normal(40, 15, n), int(rng.integers(0, 4)))
    calls = rng.integers(-(10 ** int(rng.integers(1, 7))), 10 ** int(rng.integers(1, 7)), n)
    code = rng.integers(0, 5, n) * 100
    n_vals, max_run = int(rng.integers(1, 10)), int(rng.integers(1, 60))
    key = []
    while len(key) < n:
        v = int(rng.integers(0, n_vals))
        key.extend([b"k%d" % v if v else b""] * int(rng.integers(1, max_run + 1)))   # value 0 is the empty string
    key = key[:n]
    if rng.random() < 0.5:
        for i in rng.integers(0, n, max(1, n // 300)):
            key[int(i)] = None
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None), ("calls", O.VT_INT64, calls, None)],
                      [("default", [("key", O.VT_STR, key, None), ("code", O.VT_INT64, code, None)])])
    usid = np.unique(sids)
    pick = usid[rng.random(usid.size) < 0.8] if usid.size > 3 else usid
    if pick.size == 0:
        pick = usid[:1]
    n_groups = int(rng.integers(1, 5))
    groups = rng.integers(0, n_groups, pick.size).astype(np.int32)
    # group ids in first-appearance order of the series, like the caller densifies them
    remap, dense = {}, []
    for g in groups.tolist():
        dense.append(remap.setdefault(g, len(remap)))
    groups = np.array(dense, dtype=np.int32)
    funcs = [O.AGG_SUM, O.AGG_COUNT, O.AGG_MIN, O.AGG_MAX, O.AGG_MEAN]
    aggs = [(str(rng.choice(["latency", "calls"])), int(rng.choice(funcs))) for _ in range(int(rng.integers(1, 5)))]
    kw = {}
    if rng.random() < 0.6:
        kw["preds"] = [O.Pred("default", "code", int(rng.choice([O.OP_EQ, O.OP_NE, O.OP_GE, O.OP_LT])), int(rng.integers(0, 5)) * 100)]
    if rng.random() < 0.6:
        a, b = sorted(rng.integers(0, n_pts, 2).tolist())
        kw["tmin"], kw["tmax"] = T0 + a * STEP, T0 + b * STEP
    if rng.random() < 0.4:
        kw["top_n"], kw["top_agg"], kw["top_desc"] = int(rng.integers(1, 8)), int(rng.integers(0, len(aggs))), bool(rng.integers(0, 2))
    oq = O.Query([part], pick, aggs, groups=groups, n_groups=len(remap), **kw)
    got, want = _keyed_both(bydb, gpu_ctx, [part], oq, "default", "key")
    assert got.key == want.key, (seed, got.key, want.key)
    assert_parity(got, want, aggs, f"keyed sweep {seed}")
