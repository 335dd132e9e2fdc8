"""-m gpu: the SWAR sum decoders on pages that need their three-class fall-back.

The scan decodes a delta page with two byte classes (the first and the second byte of a varint) and decodes a 2 KB chunk again
with three classes only when it holds the third byte of a varint.  Metric columns at a fixed precision almost never produce
such varints, so the parity suite rarely reaches that path on the device.  Here `latency` carries rare spikes whose deltas take
3 bytes (|delta| >= 8192 in units of the last decimal), at densities from a few per page to one row in three, so that they fall
on lane and chunk edges, and some series carry one 4-byte delta (the page then goes to the general decoder).  Each query runs
through the C ABI and is compared with the oracle under the parity contract:
  * sum + count grouped by service with a Top N, no filter (the express lane, swar_chunk);
  * mean under a time range and under a tag predicate (the masked SWAR pass);
  * sum + count grouped by a stored tag (bydb_scan_agg_keyed).
"""
import dataclasses

import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import STEP, T0, assert_parity, build_part, grid, run_both, to_gpu_query

pytestmark = pytest.mark.gpu

N_SERIES, N_PTS = 48, 6000


def _spiky_part():
    rng = np.random.default_rng(20261017)
    sids, ts, ver = grid(N_SERIES, N_PTS)
    lat = np.round(25 + rng.normal(0, 5, sids.size), 2).reshape(N_SERIES, N_PTS)
    for s in range(N_SERIES):
        density = [0.0, 0.001, 0.01, 0.05, 0.3][s % 5]
        hit = rng.random(N_PTS) < density
        lat[s, hit] += np.round(rng.choice([-1.0, 1.0], hit.sum()) * rng.uniform(100, 5000, hit.sum()), 2)
        if s % 8 == 3:
            lat[s, rng.integers(1, N_PTS)] += 20000.0  # a 4-byte delta into and out of the spike
    lat = lat.reshape(-1)
    region = [b"r%d" % v for v in np.repeat(rng.integers(0, 8, sids.size // 16 + 1), 16)[:sids.size]]
    part = build_part(sids, ts, ver, [("latency", O.VT_FLOAT64, lat, None)], [("default", [("region", O.VT_STR, region, None)])])
    return part, sids, lat


@pytest.fixture(scope="module")
def spiky():
    part, sids, lat = _spiky_part()
    # the deltas the encoder sees (per series, in units of 0.01): make sure the data holds what the test is about
    d = np.diff(np.round(lat * 100).astype(np.int64).reshape(N_SERIES, N_PTS), axis=1)
    zz = np.where(d >= 0, 2 * d, -2 * d - 1)
    assert (zz >= 1 << 14).sum() > 1000, "3-byte varints"
    assert (zz >= 1 << 21).any(), "4-byte varints"
    return part, np.unique(sids)


def test_express_lane_group_sum_count_topn(bydb, gpu_ctx, spiky):
    part, usid = spiky
    groups = (np.arange(usid.size) % 10).astype(np.int32)
    aggs = [("latency", O.AGG_SUM), ("latency", O.AGG_COUNT)]
    oq = O.Query([part], usid, aggs, groups=groups, n_groups=10, top_n=6, top_agg=0, top_desc=True)
    got, want = run_both(bydb, gpu_ctx, [part], oq, 91000)
    assert_parity(got, want, aggs, "spiky C3 shape")
    assert got.stats.rows_matched == N_SERIES * N_PTS


@pytest.mark.parametrize("shape", ["time_range", "tag_pred"])
def test_masked_swar_mean(bydb, gpu_ctx, spiky, shape):
    part, usid = spiky
    aggs = [("latency", O.AGG_MEAN), ("latency", O.AGG_SUM), ("latency", O.AGG_COUNT)]
    groups = (np.arange(usid.size) % 4).astype(np.int32)
    if shape == "time_range":
        oq = O.Query([part], usid, aggs, groups=groups, n_groups=4, tmin=T0 + 777 * STEP, tmax=T0 + 5123 * STEP)
    else:
        oq = O.Query([part], usid, aggs, groups=groups, n_groups=4, preds=[O.Pred("default", "region", O.OP_EQ, b"r3")])
    got, want = run_both(bydb, gpu_ctx, [part], oq, 92000 if shape == "time_range" else 93000)
    assert_parity(got, want, aggs, f"spiky masked mean ({shape})")


def test_stored_tag_group_by(bydb, gpu_ctx, spiky):
    part, usid = spiky
    aggs = [("latency", O.AGG_SUM), ("latency", O.AGG_COUNT)]
    oq = O.Query([part], usid, aggs)
    h = gpu_ctx.register_part(94000, part.files())
    try:
        got = gpu_ctx.scan_agg_keyed(to_gpu_query(bydb, [h], oq), "default", "region")
    finally:
        gpu_ctx.release_part(h)
    want = O.run_query(dataclasses.replace(oq, group_key=("default", "region")))
    assert got.key == want.key
    assert_parity(got, want, aggs, "spiky keyed group-by")
