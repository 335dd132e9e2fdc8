"""Page geometry of the scan decoders, checked against exact references computed here from the generated values.

The per-lane arithmetic of the varint decoders is tested on the host (tests/native/lane_decode_test.cc).  What this file
pins down is the warp-level glue around it in csrc/scan_kernels.cu: the neighbour-word shuffle and the carries across
32 B / 64 B lanes and 1 KB / 2 KB chunks, the first and last chunk masks (pstart = (page + header) & 15), the two-stage
2 KB TMA ring and its wrap on pages longer than 4 KB, the bail-out on a varint of 4+ bytes in the middle of a page and the
stage bookkeeping the warp's next page depends on, the terminator / last-byte checks, and the express lane's continuous
ring over a batch of up to 8 pages.

The generator below chooses the deltas of each page so that a varint of a chosen width starts at a chosen byte of the TMA
window (window offset = pstart + body offset).  A CPU test re-encodes every generated column with the oracle writer and
checks those claims; the device tests compare every answer with exact Python arithmetic on the generated values:
int64 bit-exact (sums modulo 2^64), float64 min/max bit-exact and float64 sums within a bound derived from how the
device sums (see float_sum_tol).
"""
from fractions import Fraction

import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import STEP, T0, build_part

I64_MIN, I64_MAX = -(1 << 63), (1 << 63) - 1
U = 2.0 ** -53  # unit roundoff of float64

# boundaries of the device decoders, as offsets in a page's 16 B aligned TMA window
B_LANE32, B_LANE64, B_CHUNK1K, B_CHUNK2K, B_RING, B_STAGE3 = 3 * 32, 3 * 64, 1024, 2048, 4096, 6144
BOUNDARIES = (B_LANE32, B_LANE64, B_CHUNK1K, B_CHUNK2K, B_RING, B_STAGE3)
# |delta| range of a zig-zag varint width, either sign: 1 byte below 64, 2 below 8192, 3 below 2^20, 4 below 2^27
# (-64, -8192, -2^20 zig-zag to 2^k - 1: still the narrower width, so the lower ends start one above)
MAG = {1: (1, 63), 2: (65, 8191), 3: (8193, (1 << 20) - 1), 4: ((1 << 20) + 1, (1 << 27) - 1)}
BACKGROUND = (1, 1, 2, 3, 3)  # widths of the filler varints: 3-byte deltas (the 8192 * T2 class of the SWAR sum) are common
MAX_BLOCK = 8193              # rows of a full block: the writer cuts after 8192 + 1 (measure.go:41-46, oracle/part.c)


def wrap64(x):
    x &= (1 << 64) - 1
    return x - (1 << 64) if x >> 63 else x


def varint_spans(body):
    """(start, width) of every varint of a page body: a varint ends on a byte below 0x80."""
    out, start = [], 0
    for i, c in enumerate(body):
        if c < 0x80:
            out.append((start, i + 1 - start))
            start = i + 1
    assert start == len(body), "the body must end on a terminator"
    return out


# ------------------------------------------------------------------ generator
def fill_widths(rng, nbytes, nvar=None):
    """Widths of filler varints covering exactly nbytes: nvar of them when given (each 1..3 bytes), else drawn from BACKGROUND."""
    if nvar is None:
        out = []
        while nbytes > 0:
            w = min(int(rng.choice(BACKGROUND)), nbytes)
            out.append(w)
            nbytes -= w
        return out
    assert nvar <= nbytes <= 3 * nvar, (nvar, nbytes)
    grow = rng.choice(2 * nvar, nbytes - nvar, replace=False) % nvar  # each varint can grow by two bytes
    return (1 + np.bincount(grow, minlength=nvar)).tolist()


def layout(rng, pieces):
    """pieces: ("fill", nbytes[, nvar]) or ("put", width) -> (varint widths, [(body offset, width) of every put])."""
    widths, puts = [], []
    for pc in pieces:
        if pc[0] == "fill":
            widths += fill_widths(rng, pc[1], pc[2] if len(pc) > 2 else None)
        else:
            puts.append((sum(widths), pc[1]))
            widths.append(pc[1])
    return widths, puts


def signed_all(rng, widths):
    """A delta of each given varint width, random magnitude and sign."""
    w = np.asarray(widths, np.int64)
    lo = np.array([0] + [MAG[k][0] for k in (1, 2, 3, 4)], np.int64)[w]
    hi = np.array([0] + [MAG[k][1] for k in (1, 2, 3, 4)], np.int64)[w]
    return (rng.integers(lo, hi + 1) * np.where(rng.random(w.size) < 0.5, 1, -1)).tolist()


def delta_walk(rng, widths, first, lo, hi):
    """EncodeTypeDelta values: first >= 0, deltas of the given widths whose signs differ (not is_delta) and every value above
    an eighth of its predecessor (not is_incremental), inside [lo, hi]."""
    assert 0 <= first and lo > hi >> 3
    ds = signed_all(rng, widths)
    if len(ds) >= 2 and len({d > 0 for d in ds[1:]} | {ds[0] > 0}) == 1:
        ds[-1] = -ds[-1]
    vals, v = [first], first
    for i, d in enumerate(ds):
        if not lo <= v + d <= hi:
            d = -d
        v += d
        vals.append(v)
    return vals


def dod_walk(rng, widths, first):
    """Delta-of-delta values: first < 0 makes the writer take delta-of-delta (is_incremental); widths[0] is the first delta's."""
    assert first < 0
    dd = signed_all(rng, widths)
    d = dd[0]
    vals = [first, first + d]
    for x in dd[1:]:
        d += x
        vals.append(vals[-1] + d)
    return vals


class Column:
    """One column's pages, written in block order into one file; tracks the file offset so the next page's pstart is known."""

    def __init__(self, name, is_float=False, exp=0, fname="fv.bin"):
        self.name, self.is_float, self.exp, self.fname = name, is_float, exp, fname
        self.hdr = 11 if is_float else 9
        self.off = 0
        self.pages = []

    def next_pstart(self):
        return (self.off + self.hdr) % 16

    def skip(self, nbytes):
        self.off += nbytes

    def add(self, ints, enc=None, puts=(), wp=None, skip=0):
        """ints: decimal integers of one block; puts: claimed (window offset, width) of varints in the decoder's stream window,
        which starts at the 16 B aligned address at or below body + skip (skip: the first delta of a delta-of-delta page,
        read before the stream is opened) and has pstart wp.  `wide`: a varint of 4+ bytes in the stream, which sends the
        block to the general decoder (a delta-of-delta page's first delta is read on its own, at any width)."""
        body, got_enc, first = O.int64_list_encode(ints)
        page = dict(off=self.off, pstart=self.next_pstart(), enc=got_enc, want_enc=enc, ints=list(ints), body=body, first=first,
                    puts=list(puts), wp=self.next_pstart() if wp is None else wp, skip=skip,
                    wide=any(w >= 4 for _, w in varint_spans(body)[got_enc == 4:]) if got_enc in (3, 4) else False)
        self.pages.append(page)
        self.off += self.hdr + len(body)
        return page

    def value(self, m):
        """The float64 a decimal page of exponent exp decodes m to (one correctly rounded operation, as scale_decimal)."""
        if not self.is_float:
            return m
        return float(m * 10 ** self.exp) if self.exp >= 0 else m / 10 ** -self.exp


def geometry_cases():
    """(name, window offset -> pieces): a straddling 2- / 3-byte varint at split 1 or 2, a 4-byte varint just before, on and
    just after each boundary; pages that end one byte before, on and after each boundary; bodies of 2..17 bytes."""
    cases = []
    for B in BOUNDARIES:
        for w, s in ((2, 1), (3, 1), (3, 2)):
            cases.append((f"straddle{w}s{s}@{B}", lambda p, rng, B=B, w=w, s=s: [("fill", B - s - p), ("put", w), ("fill", int(rng.integers(1, 600)))]))
        for d in (-1, 0, 1):
            cases.append((f"wide{d:+d}@{B}", lambda p, rng, B=B, d=d: [("fill", B + d - p), ("put", 4), ("fill", int(rng.integers(1, 600)))]))
        for d in (-1, 0, 1):
            cases.append((f"end{d:+d}@{B}", lambda p, rng, B=B, d=d: [("fill", B + d - p)]))
    for n in range(2, 18):
        cases.append((f"short{n}", lambda p, rng, n=n: [("fill", n, n)]))
    return cases


def w_values(s, n):
    """The second field of series s: a delta-const page (or a const one every third series)."""
    return [5 + 3 * i for i in range(n)] if s % 3 else [11] * n


def build_geometry_rows(rng, col, family):
    """-> per-series decimal-int lists of the geometry field `v` of a family, its claims recorded in col.pages.  The pages of
    the field `w` follow each `v` page in fv.bin and are accounted for, so every page's pstart is known in advance."""
    series = []
    dod = family_enc(family) == 4

    def add_series(pieces_of, tail=0):
        s, p = len(series), col.next_pstart()
        # a delta-of-delta decoder reads the first delta (1 byte here) before it opens the stream on the rest of the body
        wp = (p + 1) % 16 if dod else p
        widths, puts = layout(rng, ([("put", 1)] if dod else []) + pieces_of(wp, rng))
        claims = [(wp + o - dod, w) for o, w in puts[dod:]]
        ints = family_walk(rng, family, widths + fill_widths(rng, tail, tail))
        for b0 in range(0, len(ints), MAX_BLOCK):
            first = b0 == 0
            col.add(ints[b0:b0 + MAX_BLOCK], enc=family_enc(family) if first else None, puts=claims if first else (),
                    wp=wp if first else None, skip=int(dod) if first else 0)
            col.skip(9 + len(O.int64_list_encode(w_values(s, len(ints))[b0:b0 + MAX_BLOCK])[0]))
        series.append(ints)

    for _, pieces_of in geometry_cases():
        add_series(pieces_of)
    # the 8193-row first block of a longer series, and its 5-row tail as a second block
    add_series(lambda p, rng: [("fill", 2 * (MAX_BLOCK - 1), MAX_BLOCK - 1 - dod)], tail=5)
    # short pages until the field pages have taken every pstart: each one's length is chosen so that the next page starts at
    # a value not seen yet
    for _ in range(64):
        seen = {pg["pstart"] for pg in col.pages}
        if len(seen) == 16:
            break
        p, s = col.next_pstart(), len(series)
        for n in range(4, 20):
            nxt = (col.off + col.hdr + n + dod + 9 + len(O.int64_list_encode(w_values(s, n + dod + 1))[0]) + col.hdr) % 16
            if nxt not in seen | {p}:
                break
        add_series(lambda p, rng, n=n: [("fill", n, n)])
    return series


FAMILY = {  # name -> (value type, exponent, encoding, first value)
    "delta": (O.VT_INT64, 0, 3, 1 << 40),
    "dod": (O.VT_INT64, 0, 4, -(1 << 40)),
    "near_max": (O.VT_INT64, 0, 3, I64_MAX - (1 << 37)),
    "near_min": (O.VT_INT64, 0, 4, I64_MIN + (1 << 58)),
    # EncodeTypeDelta with every value but `first` near INT64_MIN: a page that starts below zero is always delta-of-delta
    # (is_incremental, oracle/codec.c:150-155), so the narrow delta page starts at INT64_MAX and its first delta wraps
    "wrap_to_min": (O.VT_INT64, 0, 3, I64_MAX),
    "float_neg_exp": (O.VT_FLOAT64, -2, 3, 10 ** 12 + 7),
    "float_pos_exp": (O.VT_FLOAT64, 3, 4, -(10 ** 12 + 7)),
}


def family_enc(family):
    return FAMILY[family][2]


def family_walk(rng, family, widths):
    _, _, enc, first = FAMILY[family]
    if enc == 4:
        return dod_walk(rng, widths, first)
    if family == "wrap_to_min":
        # walked above INT64_MAX without wrapping (so the first delta is positive), then stored modulo 2^64
        # the walk starts at its lower bound, so the signs can come out all positive (a delta-of-delta page): draw again
        for _ in range(200):
            vals = delta_walk(rng, widths, first, I64_MAX + 1, I64_MAX + (1 << 38))
            vals = [first] + [wrap64(v) for v in vals[1:]]
            if O.int64_list_encode(vals)[1] == 3:
                return vals
        raise AssertionError("no EncodeTypeDelta walk for these widths")
    hi = min(first + (1 << 37), I64_MAX)
    return delta_walk(rng, widths, first, first - (1 << 37), hi)


def tag_walk(rng, col, n, B):
    """Values of the narrow int64 tag page of an n-row block: a 2- or 3-byte varint straddles window offset B when the block
    is long enough.  -> (ints, row whose delta straddles B, or None)."""
    if n < 3:
        ints = [7] * n if n < 2 else [7, 9]
        col.add(ints)
        return ints, None
    p = col.next_pstart()
    k = (B - 1 - p) // 2
    if n - 2 - k >= 1 and k >= 1:
        widths, puts = layout(rng, [("fill", B - 1 - p, k), ("put", int(rng.choice((2, 3)))), ("fill", n - 2 - k, n - 2 - k)])
        ints = delta_walk(rng, widths, 1 << 30, (1 << 30) - (1 << 26), (1 << 30) + (1 << 26))
        col.add(ints, enc=3, puts=[(p + o, w) for o, w in puts])
        return ints, k + 1
    ints = delta_walk(rng, fill_widths(rng, n - 1, n - 1), 1 << 30, (1 << 30) - (1 << 26), (1 << 30) + (1 << 26))
    col.add(ints, enc=3)
    return ints, None


def mask_pattern(rng, kind, n):
    if kind == 0:
        return np.zeros(n, bool)
    if kind == 1:
        m = np.zeros(n, bool)
        m[int(rng.integers(0, n))] = True
        return m
    if kind == 2:
        return np.arange(n) % 2 == 1
    if kind == 3:
        m, pos, on = np.zeros(n, bool), 0, bool(rng.integers(0, 2))
        while pos < n:
            run = int(rng.integers(1, 200))
            m[pos:pos + run] = on
            pos, on = pos + run, not on
        return m
    return np.ones(n, bool)


class Case:
    """One part of a geometry family: series s (sid s + 1) holds the geometry field `v`, the delta-const field `w`, the dictionary
    tag m/k and the narrow int64 tag n/t."""

    def __init__(self, family, seed):
        rng = np.random.default_rng(seed)
        vt, exp, _, _ = FAMILY[family]
        self.v = Column("v", vt == O.VT_FLOAT64, exp)
        self.t = Column("t", fname="n.tf")
        v_series = build_geometry_rows(rng, self.v, family)
        self.series = []
        tag_bounds = (B_CHUNK1K, B_CHUNK2K, B_LANE64)
        for s, ints in enumerate(v_series):
            n = len(ints)
            ws = w_values(s, n)
            tint, trow = [], None
            for b0 in range(0, n, MAX_BLOCK):                              # one tag page per block, like the field pages
                part_ints, r = tag_walk(rng, self.t, min(MAX_BLOCK, n - b0), tag_bounds[s % 3])
                if r is not None and b0 == 0:
                    trow = r
                tint += part_ints
            self.series.append(dict(v=ints, w=ws, t=tint, trow=trow, k=mask_pattern(rng, s % 5, n)))
        self.family = family

    def fields_and_tags(self):
        sids = np.concatenate([np.full(len(s["v"]), i + 1, np.uint64) for i, s in enumerate(self.series)])
        ts = np.concatenate([T0 + np.arange(len(s["v"]), dtype=np.int64) * STEP for s in self.series])
        vv = [m for s in self.series for m in s["v"]]
        vals = np.array([self.v.value(m) for m in vv], np.float64) if self.v.is_float else np.array(vv, np.int64)
        fields = [("v", O.VT_FLOAT64 if self.v.is_float else O.VT_INT64, vals, None),
                  ("w", O.VT_INT64, np.array([x for s in self.series for x in s["w"]], np.int64), None)]
        k = [b"a" if on else b"b" for s in self.series for on in s["k"]]
        t = np.array([x for s in self.series for x in s["t"]], np.int64)
        fams = [("m", [("k", O.VT_STR, k, None)]), ("n", [("t", O.VT_INT64, t, None)])]
        return sids, ts, fields, fams

    def part(self):
        sids, ts, fields, fams = self.fields_and_tags()
        return build_part(sids, ts, np.ones(sids.size, np.int64), fields, fams)


_CASES = {}


def case_of(family):
    if family not in _CASES:
        import zlib
        _CASES[family] = Case(family, zlib.crc32(family.encode()))
    return _CASES[family]


# ------------------------------------------------------------------ CPU: the generator's claims against the writer
@pytest.mark.parametrize("family", sorted(FAMILY))
def test_generator_places_varints_where_it_claims(family):
    c = case_of(family)
    files = c.part().files()
    fv, tf = files["fv.bin"], files["n.tf"]
    # the writer lays the pages out block after block, field after field: v then w in fv.bin, t alone in n.tf.  Walk fv.bin with
    # the page sizes of the generated pages to find every v page, and check that the writer put exactly those bytes there.
    off = 0
    vpages = iter(c.v.pages)
    for s in c.series:
        n = len(s["v"])
        for b0 in range(0, n, MAX_BLOCK):
            pg = next(vpages)
            hdr = bytes([pg["enc"]]) + ((c.v.exp & 0xFFFF).to_bytes(2, "big") if c.v.is_float else b"") + O.conv_int64_to_bytes(pg["first"])
            assert fv[off:off + len(hdr) + len(pg["body"])] == hdr + pg["body"], f"{family}: v page of block at row {b0}"
            assert (off + c.v.hdr) % 16 == pg["pstart"]
            off += len(hdr) + len(pg["body"])
            wb, _, _ = O.int64_list_encode(s["w"][b0:b0 + MAX_BLOCK])
            off += 9 + len(wb)
    assert off == len(fv)
    for pg in c.v.pages + c.t.pages:
        if pg["want_enc"] is not None:
            assert pg["enc"] == pg["want_enc"], (family, pg["puts"], pg["enc"])
        if pg["enc"] in (3, 4):
            spans = set(varint_spans(pg["body"]))
            for wo, w in pg["puts"]:
                assert (wo - pg["wp"] + pg["skip"], w) in spans, f"{family}: no {w}-byte varint at window offset {wo} (pstart {pg['wp']})"
    toff = 0
    for pg in c.t.pages:
        assert tf[toff + 9:toff + 9 + len(pg["body"])] == pg["body"] and (toff + 9) % 16 == pg["pstart"]
        toff += 9 + len(pg["body"])
    if c.v.is_float:
        for s in c.series:
            ints, e = O.float64_to_decimal_list([c.v.value(m) for m in s["v"][:MAX_BLOCK]])
            assert e == c.v.exp and ints.tolist() == s["v"][:MAX_BLOCK], f"{family}: the decimal page must hold the generated integers"
    # every boundary class is hit by a straddling varint at split 1 and 2 and by a 4-byte varint before / on / after it
    claimed = {(wo, w) for pg in c.v.pages for wo, w in pg["puts"]}
    for B in BOUNDARIES:
        assert {(B - 1, 2), (B - 1, 3), (B - 2, 3), (B - 1, 4), (B, 4), (B + 1, 4)} <= claimed, B
    assert {pg["pstart"] for pg in c.v.pages} == set(range(16)), f"{family}: pstart values {sorted({pg['pstart'] for pg in c.v.pages})}"


def test_range_rows_end_on_boundaries():
    rc = range_case()
    for pg, (ba, bb) in zip(rc.col.pages, rc.bounds):
        ends = np.cumsum([w for _, w in varint_spans(pg["body"])])
        assert pg["pstart"] + ends[RANGE_R0 - 1] == ba and pg["pstart"] + ends[RANGE_R1 - 1] == bb, (pg["pstart"], ba, bb)


# ------------------------------------------------------------------ the time-range part: rows r0 / r1 end on boundaries
RANGE_R0, RANGE_R1 = 400, 1500
RANGE_BOUNDS = [(416, 2048), (448, 2048), (1024, 3072), (1024, 4096), (448, 3072), (1088, 4096), (480, 2048)]


class RangeCase:
    def __init__(self, seed=0x5A):
        rng = np.random.default_rng(seed)
        self.col, self.bounds, self.series = Column("v"), [], []
        for i in range(48):
            ba, bb = RANGE_BOUNDS[i % len(RANGE_BOUNDS)]
            p = self.col.next_pstart()
            widths, _ = layout(rng, [("fill", ba - p, RANGE_R0), ("fill", bb - ba, RANGE_R1 - RANGE_R0), ("fill", int(rng.integers(2, 900)))])
            ints = delta_walk(rng, widths, 1 << 40, (1 << 40) - (1 << 37), (1 << 40) + (1 << 37))
            self.col.add(ints, enc=3)
            self.bounds.append((ba, bb))
            self.series.append(ints)

    def part(self):
        sids = np.concatenate([np.full(len(s), i + 1, np.uint64) for i, s in enumerate(self.series)])
        ts = np.concatenate([T0 + np.arange(len(s), dtype=np.int64) * STEP for s in self.series])
        return build_part(sids, ts, np.ones(sids.size, np.int64), [("v", O.VT_INT64, np.concatenate(self.series).astype(np.int64), None)])


_RANGE = []


def range_case():
    if not _RANGE:
        _RANGE.append(RangeCase())
    return _RANGE[0]


# ------------------------------------------------------------------ exact references
def float_sum_tol(n_blocks, abs_sum):
    """Bound on |device float64 sum - exact sum of the decoded cells| for one group.

    Per block the device adds the page's decimal integers exactly (128 bits), converts that sum to float64 (one rounding, or
    two when it does not fit 64 bits: hi * 2^64 + lo) and scales it by 10^exp once (scale_decimal: one more rounding while
    |exp| <= 22, so 10^|exp| is exact).  Each decoded cell is itself a rounded m * 10^exp, within U * |v| of the decimal value,
    so the block sum is within 4 * U * sum|v| of the exact sum of the decoded cells.  The n_blocks - 1 additions across
    blocks (series, then group) add at most U * sum|v| each.  First order: (n_blocks + 4) * U * sum|v|."""
    return (n_blocks + 4) * U * abs_sum


def ref_group(col, vals, n_blocks, func):
    """Exact answer of one aggregate over the active cells `vals` (decimal integers) of one group. -> (value, tolerance)."""
    if func == O.AGG_COUNT:
        return len(vals), 0
    if col.is_float:
        fl = [col.value(m) for m in vals]
        if func == O.AGG_MIN:
            return min(fl), 0
        if func == O.AGG_MAX:
            return max(fl), 0
        exact = sum((Fraction(x) for x in fl), Fraction(0))
        tol = float_sum_tol(n_blocks, sum(abs(x) for x in fl))
        if func == O.AGG_SUM:
            return float(exact), tol
        mean = exact / len(fl)   # function.go Val(): sum / count, and a mean below 1 reads as 1 (oracle/query.c:431-434)
        return (1.0 if mean < 1 else float(mean)), tol / len(fl) + U * abs(float(mean))
    if func == O.AGG_MIN:
        return min(vals), 0
    if func == O.AGG_MAX:
        return max(vals), 0
    total = wrap64(sum(vals))  # Go's int64 sum wraps modulo 2^64
    if func == O.AGG_SUM:
        return total, 0
    mean = abs(total) // len(vals) * (1 if total >= 0 else -1)  # oracle/query.c:419-423: truncating division, then max(v, 1)
    return max(mean, 1), 0


def check_result(res, want, aggs, ctx):
    """want: {group: (rows, [(value, tol) per agg])}."""
    assert sorted(want) == res.group_id.tolist(), f"{ctx}: groups {res.group_id.tolist()[:20]} vs {sorted(want)[:20]}"
    for i, g in enumerate(res.group_id.tolist()):
        rows, vals = want[g]
        assert int(res.rows[i]) == rows, f"{ctx}: group {g} rows {int(res.rows[i])} vs {rows}"
        for a, (v, tol) in enumerate(vals):
            got = res.value(i, a)
            if isinstance(v, float) and tol == 0:
                assert got == v, f"{ctx}: group {g} agg {aggs[a]}: {got!r} vs {v!r} (bit-exact)"
            elif isinstance(v, float):
                assert abs(got - v) <= tol, f"{ctx}: group {g} agg {aggs[a]}: {got!r} vs {v!r} (|diff| {abs(got - v):.3g} > {tol:.3g})"
            else:
                assert got == v, f"{ctx}: group {g} agg {aggs[a]}: {got} vs {v}"


NEEDS = {  # which decoder the aggregates pick: SWAR sum / express count / delta_page_fast<MinMax> / both / mean
    "sum": [O.AGG_SUM],
    "count": [O.AGG_COUNT],
    "minmax": [O.AGG_MIN, O.AGG_MAX],
    "sum_min": [O.AGG_SUM, O.AGG_MIN],
    "mean": [O.AGG_MEAN],
}
CMP = {O.OP_LT: lambda a, b: a < b, O.OP_GE: lambda a, b: a >= b, O.OP_EQ: lambda a, b: a == b}


def expected(col, series_vals, actives, funcs, extra=None):
    """Per-series groups: series i -> group i.  series_vals[i]: decimal ints; actives[i]: bool mask of the active rows."""
    want = {}
    for g, (vals, act) in enumerate(zip(series_vals, actives)):
        sel = [m for m, a in zip(vals, act) if a]
        if not sel:
            continue
        nb = len(range(0, len(vals), MAX_BLOCK))
        want[g] = (len(sel), [ref_group(col, sel, nb, f) for f in funcs] + (extra(g, sel) if extra else []))
    return want


def device_query(bydb, ctx, h, n_series, aggs, **kw):
    return ctx.scan_agg(bydb.Query([h], np.arange(1, n_series + 1, dtype=np.uint64), aggs,
                                   series_group=np.arange(n_series, dtype=np.int32), n_groups=n_series, **kw))


def pstarts_on_device(ctx, h, n_fields, hdr_of):
    """pstart of every field page the device holds: column offset + header size, modulo 16 (the file images are 256 B aligned).
    hdr_of: field position -> header size."""
    blocks, cols = ctx.part_directory(h)
    out = []
    for b in blocks:
        # DevBlock: col_begin u32 at byte 52, n_cols u16 at 56.  DevCol: off u64 at 0, file_id u8 at 15; file 1 is fv.bin, where
        # a block's fields lie in order
        col_begin, n_cols = int(b[52:56].view(np.uint32)[0]), int(b[56:58].view(np.uint16)[0])
        offs = sorted(int(c[0:8].view(np.uint64)[0]) for c in cols[col_begin:col_begin + n_cols] if c[15] == 1)
        assert len(offs) == n_fields
        out += [(j, (o + hdr_of[j]) % 16) for j, o in enumerate(offs)]
    return out


# ------------------------------------------------------------------ device: every family through every decoder and row mode
@pytest.mark.gpu
@pytest.mark.parametrize("family", sorted(FAMILY))
def test_geometry_device_matrix(bydb, gpu_ctx, family):
    c = case_of(family)
    ns = len(c.series)
    h = gpu_ctx.register_part(7100 + sorted(FAMILY).index(family), c.part().files())
    try:
        # the field pages take every pstart, read back from the device's own directory
        ps = pstarts_on_device(gpu_ctx, h, 2, {0: c.v.hdr, 1: 9})
        assert sorted({p for j, p in ps if j == 0}) == list(range(16))
        assert [p for j, p in ps if j == 0] == [pg["pstart"] for pg in c.v.pages]
        vals = [s["v"] for s in c.series]
        all_rows = [np.ones(len(v), bool) for v in vals]
        wide_blocks = sum(pg["wide"] for pg in c.v.pages)
        lo_row, hi_row = 37, 1999
        in_range = [(np.arange(len(v)) >= lo_row) & (np.arange(len(v)) <= hi_row) for v in vals]
        lits = [(s["t"][s["trow"]], s["trow"]) for s in c.series if s["trow"] is not None][:3]
        assert len(lits) == 3
        for need, funcs in NEEDS.items():
            aggs = [("v", f) for f in funcs]
            ctx = f"{family}/{need}"
            # all rows
            res = device_query(bydb, gpu_ctx, h, ns, aggs)
            check_result(res, expected(c.v, vals, all_rows, funcs), aggs, ctx + "/all")
            if need != "count":
                assert res.stats.blocks_slow_lane == wide_blocks, (ctx, res.stats.blocks_slow_lane, wide_blocks)
                assert bool(res.stats.slow_lane_reasons & 4) == (wide_blocks > 0), (ctx, res.stats.slow_lane_reasons)
            else:
                assert res.stats.blocks_slow_lane == 0, ctx  # COUNT never reads the page body
            # time range
            res = device_query(bydb, gpu_ctx, h, ns, aggs, tmin=T0 + lo_row * STEP, tmax=T0 + hi_row * STEP)
            check_result(res, expected(c.v, vals, in_range, funcs), aggs, ctx + "/range")
            # dictionary tag mask: none / one row / alternating / runs / all, by series
            res = device_query(bydb, gpu_ctx, h, ns, aggs, preds=[bydb.Pred("m", "k", bydb.OP_EQ, b"a")])
            check_result(res, expected(c.v, vals, [s["k"] for s in c.series], funcs), aggs, ctx + "/dict")
            # int64 tag mask from the narrow delta tag page; literal = a value its walk reaches on a straddling varint
            for (lit, _), op in zip(lits, CMP):
                res = device_query(bydb, gpu_ctx, h, ns, aggs, preds=[bydb.Pred("n", "t", op, int(lit))])
                act = [np.array([CMP[op](x, lit) for x in s["t"]]) for s in c.series]
                check_result(res, expected(c.v, vals, act, funcs), aggs, f"{ctx}/int-tag op {op}")
                assert res.stats.slow_lane_reasons & 2 == 0, "the narrow tag page must be compared by delta_pred_fast"
        # the same narrow field alone (express lane) and next to a delta-const / const field (the express lane refuses the
        # block, the regular fast lane takes it whole and the first field goes through delta_page_sum_all)
        wv = [s["w"] for s in c.series]
        for aggs in ([("v", O.AGG_SUM)], [("v", O.AGG_SUM), ("w", O.AGG_SUM)], [("w", O.AGG_SUM), ("v", O.AGG_SUM)]):
            res = device_query(bydb, gpu_ctx, h, ns, aggs)
            want = {}
            for g in range(ns):
                parts = {"v": ref_group(c.v, vals[g], len(range(0, len(vals[g]), MAX_BLOCK)), O.AGG_SUM),
                         "w": (wrap64(sum(wv[g])), 0)}
                want[g] = (len(vals[g]), [parts[f] for f, _ in aggs])
            check_result(res, want, aggs, f"{family}/lanes {aggs}")
            assert res.stats.blocks_slow_lane == wide_blocks
            if wide_blocks:
                assert res.stats.slow_lane_reasons & (4 << [f for f, _ in aggs].index("v")), res.stats.slow_lane_reasons
    finally:
        gpu_ctx.release_part(h)


@pytest.mark.gpu
def test_time_range_rows_on_boundaries(bydb, gpu_ctx):
    rc = range_case()
    ns = len(rc.series)
    h = gpu_ctx.register_part(7200, rc.part().files())
    try:
        for r0, r1 in ((RANGE_R0, RANGE_R1), (RANGE_R0 + 1, RANGE_R1 + 1), (RANGE_R0 + 1, RANGE_R1)):
            act = [(np.arange(len(v)) >= r0) & (np.arange(len(v)) <= r1) for v in rc.series]
            for need, funcs in NEEDS.items():
                aggs = [("v", f) for f in funcs]
                res = device_query(bydb, gpu_ctx, h, ns, aggs, tmin=T0 + r0 * STEP, tmax=T0 + r1 * STEP)
                check_result(res, expected(rc.col, rc.series, act, funcs), aggs, f"range [{r0},{r1}] {need}")
                assert res.stats.blocks_slow_lane == 0
    finally:
        gpu_ctx.release_part(h)


# ------------------------------------------------------------------ bail-out in the middle of a block, then more fields
def bailout_part(seed=0xBA11):
    """Blocks of five SUM fields over ~6.5 KB pages (four TMA stages): in block (j, where) field j holds one 4-byte varint in
    chunk 0, in the third stage or in the last chunk; every other field is narrow.  Plus narrow blocks in between."""
    rng = np.random.default_rng(seed)
    nf, n = 5, 3000
    cols = [Column(f"f{j}") for j in range(nf)]
    series = []
    for j in range(nf):
        for where in ("chunk0", "stage3", "last", None):
            row = []
            for i, col in enumerate(cols):
                p = col.next_pstart()
                body = 6400 + 16 * i + j - p
                wpos = {"chunk0": 200, "stage3": 4096 + 500, "last": body + p - 40}.get(where)
                if i == j and wpos is not None:
                    b1, b2 = wpos - p, body - (wpos - p) - 4
                    k = max(-(-b1 // 3), n - 2 - b2)          # varints before the wide one: both fills need 1..3 bytes per varint
                    pieces = [("fill", b1, k), ("put", 4), ("fill", b2, n - 2 - k)]
                else:
                    pieces = [("fill", body, n - 1)]
                widths, puts = layout(rng, pieces)
                ints = delta_walk(rng, widths, 1 << 40, (1 << 40) - (1 << 37), (1 << 40) + (1 << 37))
                col.add(ints, enc=3, puts=[(p + o, w) for o, w in puts])
                row.append(ints)
            series.append(row)
    return cols, series


@pytest.mark.gpu
def test_slow_lane_decodes_the_fields_after_a_bailout(bydb, gpu_ctx):
    """A block with a wide page goes whole to the slow lane, where one warp decodes its fields in order: field j's fast
    decoder bails out mid-page (drain, sm->seq fix-up), the general decoder opens the same page again, then fields j+1..
    open theirs.  Every one of those streams starts from the ring bookkeeping the previous one left."""
    cols, series = bailout_part()
    nf, ns = len(cols), len(series)
    sids = np.concatenate([np.full(len(r[0]), s + 1, np.uint64) for s, r in enumerate(series)])
    ts = np.concatenate([T0 + np.arange(len(r[0]), dtype=np.int64) * STEP for r in series])
    fields = [(f"f{j}", O.VT_INT64, np.concatenate([r[j] for r in series]).astype(np.int64), None) for j in range(nf)]
    h = gpu_ctx.register_part(7300, build_part(sids, ts, np.ones(sids.size, np.int64), fields).files())
    wide = sum(any(c.pages[s]["wide"] for c in cols) for s in range(ns))
    assert wide == nf * 3
    try:
        for funcs in ([O.AGG_SUM], [O.AGG_SUM, O.AGG_MAX], [O.AGG_MEAN]):
            aggs = [(f"f{j}", f) for j in range(nf) for f in funcs]
            res = device_query(bydb, gpu_ctx, h, ns, aggs)
            want = {g: (len(series[g][0]), [ref_group(cols[0], series[g][int(f[1:])], 1, fn) for f, fn in aggs]) for g in range(ns)}
            check_result(res, want, aggs, f"bail-out {funcs}")
            assert res.stats.blocks_slow_lane == wide
            assert res.stats.slow_lane_reasons & 0b1111100 == 0b1111100, res.stats.slow_lane_reasons
            for tmin, tmax in ((T0 + 5 * STEP, T0 + 2990 * STEP),):
                res = device_query(bydb, gpu_ctx, h, ns, aggs, tmin=tmin, tmax=tmax)
                want = {g: (2986, [ref_group(cols[0], series[g][int(f[1:])][5:2991], 1, fn) for f, fn in aggs]) for g in range(ns)}
                check_result(res, want, aggs, f"bail-out ranged {funcs}")
    finally:
        gpu_ctx.release_part(h)


def test_bailout_part_claims():
    cols, series = bailout_part()
    for s in range(len(series)):
        wides = [j for j, c in enumerate(cols) if c.pages[s]["wide"]]
        assert wides == ([s // 4] if s % 4 != 3 else []), (s, wides)
        for c in cols:
            pg = c.pages[s]
            assert pg["enc"] == 3 and len(pg["ints"]) == 3000
            spans = set(varint_spans(pg["body"]))
            for wo, w in pg["puts"]:
                assert (wo - pg["pstart"], w) in spans
            assert (pg["pstart"] + len(pg["body"])) > 3 * 2048, "every page spans four TMA stages"


# ------------------------------------------------------------------ many blocks per warp: express batches, fast-lane grabs
EXPRESS_KINDS = ("plain", "single", "long", "wide", "bail_chunk0", "bail_stage3", "bail_last")
BAIL_ROWS, BAIL_BODY = 3000, 6400   # bail pages: four TMA stages
X_OFF = 1 << 40


def bail_page(rng, where):
    """A 6.4 KB narrow page with one 4-byte varint starting at body offset 200 (chunk 0), 4596 (third stage) or 40 bytes
    before the end (last chunk), or none (where=None)."""
    n, body = BAIL_ROWS, BAIL_BODY
    if where is None:
        widths = fill_widths(rng, body, n - 1)
    else:
        b1 = {"chunk0": 200, "stage3": 4096 + 500, "last": body - 40}[where]
        b2 = body - b1 - 4
        k = max(-(-b1 // 3), n - 2 - b2)          # varints before the wide one: both fills need 1..3 bytes per varint
        widths, _ = layout(rng, [("fill", b1, k), ("put", 4), ("fill", b2, n - 2 - k)])
    return delta_walk(rng, widths, X_OFF, X_OFF - (1 << 37), X_OFF + (1 << 37))


def express_blocks(rng, n_blocks):
    """Per block: dict(kind, x, y, z, wide_x, wide_y).  single: one row (a const page, which the express lane hands on);
    long: a page of more than 4 KB (the ring wraps inside the page); wide: one 4-byte varint in x; bail_*: 6.4 KB pages in
    x and y, one of them with a 4-byte varint in chunk 0, the third stage or the last chunk.  z is a delta-const page."""
    kinds = rng.choice(len(EXPRESS_KINDS), size=n_blocks, p=[0.854, 0.07, 0.01, 0.06, 0.002, 0.002, 0.002])
    out = []
    for k in kinds.tolist():
        kind = EXPRESS_KINDS[k]
        wide_x = wide_y = False
        if kind.startswith("bail"):
            where = kind[5:]
            wide_x = bool(rng.integers(0, 2))
            wide_y = not wide_x
            x, y = bail_page(rng, where if wide_x else None), bail_page(rng, where if wide_y else None)
        else:
            n = 1 if kind == "single" else int(rng.integers(2600, 4000)) if kind == "long" else int(rng.integers(3, 40))
            lo = 4200 if kind == "long" else n - 1
            widths = fill_widths(rng, int(rng.integers(lo, 2 * (n - 1) + 1)), n - 1) if n > 1 else []
            if kind == "wide":
                widths[int(rng.integers(0, len(widths)))] = 4
                wide_x = True
            x = delta_walk(rng, widths, X_OFF, X_OFF - (1 << 37), X_OFF + (1 << 37)) if n > 1 else [int(rng.integers(0, X_OFF))]
            y = delta_walk(rng, fill_widths(rng, n - 1, n - 1), 1 << 20, 1 << 19, 1 << 21) if n > 2 else [3] * n
        z = [7 + 5 * i for i in range(len(x))]
        out.append(dict(kind=kind, x=x, y=y, z=z, wide_x=wide_x, wide_y=wide_y))
    return out


@pytest.mark.gpu
def test_many_blocks_per_warp_express_batches_and_fast_lane_grabs(bydb):
    """One CTA of 8 warps per SM and ~20 blocks per warp, so the scheduler hands out several blocks per grab: the express lane
    streams full 8-page batches through one ring, and the regular fast lane takes 4 blocks at a time.  Pages that bail out
    mid-batch (wide, bail_*) are followed on the same warp by the rest of the batch or the next grabbed block, which depend
    on the ring bookkeeping the bail-out left."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    warps = sms * 8                                  # warps_per_sm=8: one CTA of 8 warps per SM
    n_blocks = 20 * warps                            # grab_work hands out 8 blocks while more than 16 per warp are left
    rng = np.random.default_rng(0xE8)
    blocks = express_blocks(rng, n_blocks)
    n_missing = n_blocks // 5                        # part B: no field y
    # part B lies after part A in time: parts that overlap in time take the version-dedup path, which the express lane skips
    b_t0 = T0 + 10_000 * STEP
    G = 64
    parts = []
    for lo, hi, with_y, t0 in ((0, n_missing, False, b_t0), (n_missing, n_blocks, True, T0)):
        bl = blocks[lo:hi]
        sids = np.concatenate([np.full(len(b["x"]), lo + i + 1, np.uint64) for i, b in enumerate(bl)])
        ts = np.concatenate([t0 + np.arange(len(b["x"]), dtype=np.int64) * STEP for b in bl])
        fields = [("x", O.VT_INT64, np.concatenate([b["x"] for b in bl]).astype(np.int64), None),
                  ("z", O.VT_INT64, np.concatenate([b["z"] for b in bl]).astype(np.int64), None)]
        if with_y:
            fields.append(("y", O.VT_INT64, np.concatenate([b["y"] for b in bl]).astype(np.int64), None))
        parts.append(build_part(sids, ts, np.ones(sids.size, np.int64), fields))
    groups = (np.arange(n_blocks) * 7919 % G).astype(np.int32)

    def want_of(aggs, first_row):
        """Exact per-group answers; rows of part A below first_row are cut by the time range."""
        acc = {}
        for b, blk in enumerate(blocks):
            r0 = first_row if b >= n_missing else 0
            if r0 >= len(blk["x"]):
                continue
            a = acc.setdefault(int(groups[b]), dict(rows=0, x=[], y=[], z=[]))
            a["rows"] += len(blk["x"]) - r0
            for f in ("x", "z") + (("y",) if b >= n_missing else ()):
                a[f] += blk[f][r0:]
        out = {}
        for g, a in acc.items():
            vals = []
            for f, fn in aggs:
                v = a[f]
                vals.append((len(v), 0) if fn == O.AGG_COUNT else (max(v), 0) if fn == O.AGG_MAX else (wrap64(sum(v)), 0))
            out[g] = (a["rows"], vals)
        return out

    def wide_blocks(fields, first_row=0):
        return sum(1 for b, blk in enumerate(blocks) if len(blk["x"]) > (first_row if b >= n_missing else 0)
                   and (("x" in fields and blk["wide_x"]) or ("y" in fields and blk["wide_y"] and b >= n_missing)))

    sums = [("x", O.AGG_SUM), ("x", O.AGG_COUNT), ("y", O.AGG_SUM), ("y", O.AGG_COUNT)]
    ctx = bydb.Context(device=0, warps_per_sm=8)
    try:
        hs = [ctx.register_part(7400 + i, p.files()) for i, p in enumerate(parts)]

        def run(aggs, name, first_row=0, fields=("x", "y")):
            tmin = T0 + first_row * STEP if first_row else -(1 << 63)
            res = ctx.scan_agg(bydb.Query(hs, np.arange(1, n_blocks + 1, dtype=np.uint64), aggs, series_group=groups, n_groups=G, tmin=tmin))
            check_result(res, want_of(aggs, first_row), aggs, name)
            assert res.stats.blocks_slow_lane == wide_blocks(fields, first_row), (name, res.stats.blocks_slow_lane)
            assert res.stats.slow_lane_reasons & 4, name
            return res

        # SUM / COUNT only: the express lane
        express = run(sums, "express batches")
        assert express.stats.blocks_scanned == n_blocks and express.stats.rows_scanned == sum(len(b["x"]) for b in blocks)
        # + MAX: no express lane; the fast lane takes the whole list, 4 blocks per grab (delta_page_fast, delta_page_sum_all)
        fast = run(sums + [("x", O.AGG_MAX)], "fast lane grabs")
        # the express kernel is launched for the sums-only query and not for the other (capi.cu counts it as one launch)
        assert express.stats.kernel_launches == fast.stats.kernel_launches + 1
        # next to a delta-const field the express lane refuses every block: the fast lane takes them all through delta_page_sum_all
        run([("x", O.AGG_SUM), ("z", O.AGG_SUM)], "express refuses", fields=("x",))
        # a time range that cuts every block of part A: delta_page_sum_masked on those, the express lane on part B
        run([("x", O.AGG_SUM), ("y", O.AGG_SUM)], "ranged", first_row=2)
    finally:
        ctx.close()


def test_express_blocks_are_what_they_claim():
    rng = np.random.default_rng(0xE8)
    kinds = set()
    for b in express_blocks(rng, 6000):
        kinds.add(b["kind"])
        body, enc, _ = O.int64_list_encode(b["x"])
        assert O.int64_list_encode(b["z"])[1] == (2 if len(b["z"]) > 1 else 1)
        if b["kind"] == "single":
            assert enc == 1 and body == b""
            continue
        assert enc == 3, b["kind"]
        widest = max(w for _, w in varint_spans(body))
        assert (widest >= 4) == b["wide_x"], b["kind"]
        if b["kind"].startswith("bail"):
            ybody, yenc, _ = O.int64_list_encode(b["y"])
            assert yenc == 3 and (max(w for _, w in varint_spans(ybody)) >= 4) == b["wide_y"]
            assert len(body) == len(ybody) == BAIL_BODY and b["wide_x"] != b["wide_y"]
            wide_at = [o for o, w in varint_spans(body if b["wide_x"] else ybody) if w >= 4]
            assert wide_at == [{"chunk0": 200, "stage3": 4596, "last": BAIL_BODY - 40}[b["kind"][5:]]]
        if b["kind"] == "long":
            assert len(body) > 4096
    assert kinds == set(EXPRESS_KINDS)
