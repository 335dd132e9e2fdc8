"""ctypes binding of include/bydb_gpu.h (the same calls a cgo shim would make; see INTEGRATION.md)."""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Union

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

VT_STR, VT_INT64, VT_FLOAT64, VT_BINARY = 1, 2, 3, 4
AGG_MEAN, AGG_MAX, AGG_MIN, AGG_COUNT, AGG_SUM = 1, 2, 3, 4, 5
OP_EQ, OP_NE, OP_LT, OP_LE, OP_GT, OP_GE = 1, 2, 3, 4, 5, 6
ENOENT, EIO, ENOMEM, EINVAL, ENOTSUP = -2, -5, -12, -22, -95


class BydbError(RuntimeError):
    """A negative return code of the C ABI plus bydb_last_error()."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"bydb error {code}: {msg}")
        self.code = code
        self.msg = msg


class _Cfg(C.Structure):
    _fields_ = [("device", C.c_int32), ("warps_per_sm", C.c_int32), ("hbm_budget_bytes", C.c_uint64),
                ("flags", C.c_uint32), ("reserved", C.c_uint32)]


class _File(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("len", C.c_uint64)]


class _PartFiles(C.Structure):
    _fields_ = [("n_files", C.c_uint32), ("files", C.POINTER(_File))]


class _Pred(C.Structure):
    _fields_ = [("family", C.c_char_p), ("tag", C.c_char_p), ("op", C.c_int32), ("value_type", C.c_int32),
                ("lit", C.c_void_p), ("lit_len", C.c_uint64), ("lit_i64", C.c_int64)]


class _Agg(C.Structure):
    _fields_ = [("field", C.c_char_p), ("func", C.c_int32), ("reserved", C.c_int32)]


class _Query(C.Structure):
    _fields_ = [("n_parts", C.c_uint32), ("parts", C.POINTER(C.c_uint64)), ("n_series", C.c_uint64),
                ("series_ids", C.c_void_p), ("series_group", C.c_void_p), ("n_groups", C.c_int32),
                ("reserved0", C.c_int32), ("tmin", C.c_int64), ("tmax", C.c_int64), ("n_preds", C.c_uint32),
                ("preds", C.POINTER(_Pred)), ("n_aggs", C.c_uint32), ("aggs", C.POINTER(_Agg)),
                ("top_n", C.c_int32), ("top_agg", C.c_int32), ("top_desc", C.c_int32), ("flags", C.c_uint32)]


class _Stats(C.Structure):
    _fields_ = [("rows_scanned", C.c_uint64), ("rows_matched", C.c_uint64), ("blocks_scanned", C.c_uint64),
                ("page_bytes", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("scan_kernel_ms", C.c_double), ("device_ms", C.c_double), ("kernel_launches", C.c_uint32),
                ("blocks_slow_lane", C.c_uint32), ("slow_lane_reasons", C.c_uint32), ("reserved", C.c_uint32)]


class _Result(C.Structure):
    _fields_ = [("n_rows", C.c_int32), ("n_aggs", C.c_int32), ("group_id", C.POINTER(C.c_int32)),
                ("rows", C.POINTER(C.c_int64)), ("is_float", C.POINTER(C.c_uint8)),
                ("val_i64", C.POINTER(C.c_int64)), ("val_f64", C.POINTER(C.c_double)), ("stats", _Stats),
                ("owner", C.c_void_p)]


class _GroupKey(C.Structure):
    _fields_ = [("family", C.c_char_p), ("tag", C.c_char_p), ("max_values", C.c_uint32), ("reserved", C.c_uint32)]


class _KeyedResult(C.Structure):
    _fields_ = [("base", _Result), ("key_id", C.POINTER(C.c_int32)), ("n_keys", C.c_int32), ("reserved", C.c_int32),
                ("key_off", C.POINTER(C.c_uint32)), ("key_bytes", C.POINTER(C.c_uint8)), ("owner", C.c_void_p)]


class _EncodeInput(C.Structure):
    _fields_ = [("value_type", C.c_int32), ("n_blocks", C.c_uint32), ("block_rows", C.c_void_p), ("values", C.c_void_p)]


class _EncodedPages(C.Structure):
    _fields_ = [("n_blocks", C.c_uint32), ("reserved", C.c_uint32), ("page_off", C.POINTER(C.c_uint64)), ("bytes", C.POINTER(C.c_uint8)),
                ("needs_cpu", C.POINTER(C.c_uint8)), ("n_cpu_blocks", C.c_uint64), ("device_ms", C.c_double), ("owner", C.c_void_p)]


class _PartialRows(C.Structure):
    _fields_ = [("n_rows", C.c_int32), ("n_aggs", C.c_int32), ("group_id", C.POINTER(C.c_int32)), ("is_float", C.POINTER(C.c_uint8)),
                ("val_i64", C.POINTER(C.c_int64)), ("val_f64", C.POINTER(C.c_double)), ("cnt_i64", C.POINTER(C.c_int64)),
                ("cnt_f64", C.POINTER(C.c_double)), ("owner", C.c_void_p)]


class _Layout(C.Structure):
    _fields_ = [("total_bytes", C.c_uint64), ("off_sum_f64", C.c_uint64), ("off_max_f64", C.c_uint64),
                ("off_sum_i64", C.c_uint64), ("off_max_i64", C.c_uint64), ("n_sum_f64", C.c_uint64),
                ("n_max_f64", C.c_uint64), ("n_sum_i64", C.c_uint64), ("n_max_i64", C.c_uint64)]


# every symbol include/bydb_gpu.h declares (tests/test_capi_symbols.py checks the list against the header)
EXPORTS = ["bydb_init", "bydb_shutdown", "bydb_part_register", "bydb_part_release", "bydb_part_info", "bydb_part_fallback_pages", "bydb_part_directory",
           "bydb_scan_agg", "bydb_scan_agg_host", "bydb_result_free", "bydb_query_prepare", "bydb_scan_agg_prepared",
           "bydb_query_release", "bydb_partials_layout",
           "bydb_scan_partials", "bydb_partials_combine", "bydb_reduce_finalize", "bydb_partials_rows", "bydb_partial_rows_free", "bydb_comm_export", "bydb_comm_connect",
           "bydb_scan_reduce", "bydb_scan_reduce_prepared", "bydb_scan_reduce_host", "bydb_scan_agg_keyed", "bydb_keyed_result_free",
           "bydb_keyed_reduce_layout", "bydb_scan_reduce_keyed",
           "bydb_encode_pages", "bydb_encoded_pages_free", "bydb_last_error", "bydb_version"]

_lib = None


def library_path() -> str:
    # BYDB_GPU_LIB: a differently built libbydbgpu.so (kernel-variant experiments); still the CUDA library, never a fallback
    return os.environ.get("BYDB_GPU_LIB") or os.path.join(_HERE, "libbydbgpu.so")


def load_library():
    """Loads libbydbgpu.so.  Fails loudly when the CUDA extension is missing: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: build it with `make -C {_HERE}` (or __graft_entry__.build()); "
                          "the measure scan path has no CPU fallback")
    L = C.CDLL(path)
    L.bydb_last_error.restype = C.c_char_p
    L.bydb_version.restype = C.c_char_p
    L.bydb_init.argtypes = [C.POINTER(_Cfg), C.POINTER(C.c_void_p)]
    L.bydb_shutdown.argtypes = [C.c_void_p]
    L.bydb_part_register.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(_PartFiles), C.POINTER(C.c_uint64)]
    L.bydb_part_release.argtypes = [C.c_void_p, C.c_uint64]
    L.bydb_part_info.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.bydb_part_fallback_pages.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.bydb_part_directory.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.bydb_scan_agg.argtypes = [C.c_void_p, C.POINTER(_Query), C.POINTER(_Result)]
    L.bydb_scan_agg_host.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(_PartFiles), C.POINTER(_Query), C.POINTER(_Result)]
    L.bydb_result_free.argtypes = [C.c_void_p, C.POINTER(_Result)]
    L.bydb_scan_agg_keyed.argtypes = [C.c_void_p, C.POINTER(_Query), C.POINTER(_GroupKey), C.POINTER(_KeyedResult)]
    L.bydb_keyed_result_free.argtypes = [C.c_void_p, C.POINTER(_KeyedResult)]
    L.bydb_keyed_result_free.restype = None
    L.bydb_keyed_reduce_layout.argtypes = [C.POINTER(_Query), C.POINTER(_GroupKey), C.POINTER(C.c_uint64)]
    L.bydb_scan_reduce_keyed.argtypes = [C.c_void_p, C.POINTER(_Query), C.POINTER(_GroupKey), C.c_int32, C.POINTER(_KeyedResult)]
    L.bydb_encode_pages.argtypes = [C.c_void_p, C.POINTER(_EncodeInput), C.POINTER(_EncodedPages)]
    L.bydb_encoded_pages_free.argtypes = [C.c_void_p, C.POINTER(_EncodedPages)]
    L.bydb_encoded_pages_free.restype = None
    L.bydb_query_prepare.argtypes = [C.c_void_p, C.POINTER(_Query), C.POINTER(C.c_void_p)]
    L.bydb_scan_agg_prepared.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(_Result)]
    L.bydb_query_release.argtypes = [C.c_void_p, C.c_void_p]
    L.bydb_query_release.restype = None
    L.bydb_partials_layout.argtypes = [C.POINTER(_Query), C.POINTER(_Layout)]
    L.bydb_scan_partials.argtypes = [C.c_void_p, C.POINTER(_Query), C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(_Stats)]
    L.bydb_partials_combine.argtypes = [C.c_void_p, C.POINTER(_Query), C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p]
    L.bydb_reduce_finalize.argtypes = [C.c_void_p, C.POINTER(_Query), C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(_Result)]
    L.bydb_partials_rows.argtypes = [C.c_void_p, C.POINTER(_Query), C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(_PartialRows)]
    L.bydb_partial_rows_free.argtypes = [C.c_void_p, C.POINTER(_PartialRows)]
    L.bydb_partial_rows_free.restype = None
    L.bydb_comm_export.argtypes = [C.c_void_p, C.c_uint64, C.c_int32, C.c_void_p]
    L.bydb_comm_connect.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
    L.bydb_scan_reduce.argtypes = [C.c_void_p, C.POINTER(_Query), C.c_int32, C.POINTER(_Result)]
    L.bydb_scan_reduce_prepared.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(_Result)]
    L.bydb_scan_reduce_host.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(_PartFiles), C.POINTER(_Query), C.c_int32, C.POINTER(_Result)]
    _lib = L
    return L


def _check(rc: int):
    if rc != 0:
        raise BydbError(rc, (load_library().bydb_last_error() or b"").decode())


@dataclass
class Pred:
    family: str
    tag: str
    op: int
    value: Union[int, bytes, str]


@dataclass
class Query:
    """model.MeasureQueryOptions after series resolution (see bydb_query in bydb_gpu.h)."""
    parts: Sequence[int]                      # part handles
    series_ids: Sequence[int]                 # ascending
    aggs: Sequence[tuple]                     # (field, AGG_*)
    series_group: Optional[Sequence[int]] = None
    n_groups: int = 1
    tmin: int = -(1 << 63)
    tmax: int = (1 << 63) - 1
    preds: Sequence[Pred] = field(default_factory=list)
    top_n: int = 0
    top_agg: int = 0
    top_desc: bool = True
    flags: int = 0


Q_HOST_ZERO_COPY = 1
Q_ROW_PATH_TYPES = 2


@dataclass
class Stats:
    rows_scanned: int = 0
    rows_matched: int = 0
    blocks_scanned: int = 0
    page_bytes: int = 0
    h2d_bytes: int = 0
    d2h_bytes: int = 0
    scan_kernel_ms: float = 0.0
    device_ms: float = 0.0
    kernel_launches: int = 0
    blocks_slow_lane: int = 0
    slow_lane_reasons: int = 0

    @staticmethod
    def of(s: _Stats) -> "Stats":
        return Stats(s.rows_scanned, s.rows_matched, s.blocks_scanned, s.page_bytes, s.h2d_bytes, s.d2h_bytes,
                     s.scan_kernel_ms, s.device_ms, s.kernel_launches, s.blocks_slow_lane, s.slow_lane_reasons)


@dataclass
class Result:
    group_id: np.ndarray
    rows: np.ndarray
    is_float: np.ndarray
    val_i64: np.ndarray   # [n_rows, n_aggs]
    val_f64: np.ndarray
    stats: Stats
    key: Optional[List[bytes]] = None   # scan_agg_keyed only: key value of each row
    n_keys: int = 0                      # scan_agg_keyed only: distinct key values found in the selected blocks

    def value(self, row: int, agg: int):
        return float(self.val_f64[row, agg]) if self.is_float[agg] else int(self.val_i64[row, agg])


def _part_files(files: Dict[str, Union[bytes, np.ndarray]], keep: list) -> _PartFiles:
    arr = (_File * len(files))()
    for i, (name, data) in enumerate(files.items()):
        nb = name.encode()
        keep.append(nb)
        arr[i].name = nb
        if isinstance(data, np.ndarray):
            a = np.ascontiguousarray(data, dtype=np.uint8)
            keep.append(a)
            arr[i].data = a.ctypes.data
            arr[i].len = a.size
        elif hasattr(data, "data_ptr"):      # a (pinned) torch uint8 tensor
            keep.append(data)
            arr[i].data = data.data_ptr()
            arr[i].len = data.numel()
        else:
            b = bytes(data)
            buf = C.create_string_buffer(b, max(len(b), 1))
            keep.append(buf)
            arr[i].data = C.cast(buf, C.c_void_p).value
            arr[i].len = len(b)
    keep.append(arr)
    pf = _PartFiles()
    pf.n_files = len(files)
    pf.files = arr
    return pf


def _mk_query(q: Query, keep: list) -> _Query:
    cq = _Query()
    parts = (C.c_uint64 * max(len(q.parts), 1))(*[int(p) for p in q.parts])
    keep.append(parts)
    cq.n_parts, cq.parts = len(q.parts), parts
    sids = np.ascontiguousarray(q.series_ids, dtype=np.uint64)
    keep.append(sids)
    cq.n_series, cq.series_ids = sids.size, sids.ctypes.data
    if q.series_group is not None:
        g = np.ascontiguousarray(q.series_group, dtype=np.int32)
        keep.append(g)
        cq.series_group, cq.n_groups = g.ctypes.data, q.n_groups
    else:
        cq.series_group, cq.n_groups = None, 1
    cq.tmin, cq.tmax = q.tmin, q.tmax
    preds = (_Pred * max(len(q.preds), 1))()
    for i, p in enumerate(q.preds):
        fb, tb = p.family.encode(), p.tag.encode()
        keep.extend([fb, tb])
        preds[i].family, preds[i].tag, preds[i].op = fb, tb, p.op
        if isinstance(p.value, (int, np.integer)):
            preds[i].value_type, preds[i].lit_i64 = VT_INT64, int(p.value)
        else:
            vb = p.value.encode() if isinstance(p.value, str) else bytes(p.value)
            buf = C.create_string_buffer(vb, max(len(vb), 1))
            keep.append(buf)
            preds[i].value_type = VT_STR
            preds[i].lit = C.cast(buf, C.c_void_p).value
            preds[i].lit_len = len(vb)
    keep.append(preds)
    cq.n_preds, cq.preds = len(q.preds), preds
    aggs = (_Agg * max(len(q.aggs), 1))()
    for i, (fname, func) in enumerate(q.aggs):
        nb = fname.encode()
        keep.append(nb)
        aggs[i].field, aggs[i].func = nb, int(func)
    keep.append(aggs)
    cq.n_aggs, cq.aggs = len(q.aggs), aggs
    cq.top_n, cq.top_agg, cq.top_desc = q.top_n, q.top_agg, int(q.top_desc)
    cq.flags = q.flags
    return cq


def keyed_reduce_layout(q: Query, family: str, tag: str, max_values: int = 0) -> int:
    """Mailbox slot bytes the keyed collective needs for q (bydb_keyed_reduce_layout; host only, no device)."""
    keep: list = []
    cq = _mk_query(q, keep)
    gk = _GroupKey(family.encode(), tag.encode(), max_values, 0)
    out = C.c_uint64(0)
    _check(load_library().bydb_keyed_reduce_layout(C.byref(cq), C.byref(gk), C.byref(out)))
    return out.value


class PreparedQuery:
    """A Query marshalled once into the C struct (with everything it points at kept alive): repeated calls skip
    the per-call ctypes work.  Context methods take a Query or a PreparedQuery."""

    def __init__(self, q: Query):
        self.query = q
        self._keep: list = []
        self.c = _mk_query(q, self._keep)


def _cq(q):
    """-> (ctypes struct, keepalive) for a Query or a PreparedQuery."""
    if isinstance(q, PreparedQuery):
        return q.c, q
    keep: list = []
    return _mk_query(q, keep), keep


def _read_result(r: _Result) -> Result:
    n, a = r.n_rows, r.n_aggs

    def arr(ptr, count, dtype):
        if count == 0:
            return np.zeros(0, dtype=dtype)
        if count <= 256:   # typical aggregate results are a handful of rows: slicing the pointer beats wrapping it (~2 us per array)
            return np.array(ptr[:count], dtype=dtype)
        return np.ctypeslib.as_array(ptr, (count,)).copy()

    return Result(group_id=arr(r.group_id, n, np.int32), rows=arr(r.rows, n, np.int64),
                  is_float=arr(r.is_float, a, np.uint8).astype(bool),
                  val_i64=arr(r.val_i64, n * a, np.int64).reshape(n, a),
                  val_f64=arr(r.val_f64, n * a, np.float64).reshape(n, a), stats=Stats.of(r.stats))


class GraphQuery:
    """A query held by the library (deep copy) whose step is replayed as one CUDA graph from its third run on."""

    def __init__(self, ctx: "Context", handle):
        self._ctx, self._h = ctx, handle

    def run(self) -> Result:
        r = _Result()
        _check(self._ctx._L.bydb_scan_agg_prepared(self._ctx._h, self._h, C.byref(r)))
        try:
            return _read_result(r)
        finally:
            self._ctx._L.bydb_result_free(self._ctx._h, C.byref(r))

    def run_reduce(self, root: int = 0) -> Result:
        """The collective form (bydb_scan_reduce_prepared): graph replay from the second execution on."""
        r = _Result()
        _check(self._ctx._L.bydb_scan_reduce_prepared(self._ctx._h, self._h, root, C.byref(r)))
        try:
            return _read_result(r)
        finally:
            self._ctx._L.bydb_result_free(self._ctx._h, C.byref(r))

    def close(self):
        if self._h:
            self._ctx._L.bydb_query_release(self._ctx._h, self._h)
            self._h = None


class Context:
    """bydb_ctx: one device, its streams and the HBM part cache."""

    def __init__(self, device: int = 0, warps_per_sm: int = 0, hbm_budget_bytes: int = 0, host_index: bool = False):
        self._L = load_library()
        cfg = _Cfg(device, warps_per_sm, hbm_budget_bytes, 1 if host_index else 0, 0)
        h = C.c_void_p()
        _check(self._L.bydb_init(C.byref(cfg), C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._L.bydb_shutdown(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        self.close()

    # ---- parts
    def register_part(self, part_id: int, files: Dict[str, Union[bytes, np.ndarray]]) -> int:
        keep: list = []
        pf = _part_files(files, keep)
        out = C.c_uint64(0)
        _check(self._L.bydb_part_register(self._h, part_id, C.byref(pf), C.byref(out)))
        return out.value

    def release_part(self, handle: int):
        _check(self._L.bydb_part_release(self._h, handle))

    def part_info(self, handle: int) -> Dict[str, int]:
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        _check(self._L.bydb_part_info(self._h, handle, C.byref(a), C.byref(b), C.byref(c)))
        u, l = C.c_uint64(), C.c_uint64()
        _check(self._L.bydb_part_fallback_pages(self._h, handle, C.byref(u), C.byref(l)))
        return dict(hbm_bytes=a.value, n_blocks=b.value, n_rows=c.value, fallback_unpacked=u.value, fallback_left=l.value)

    def part_directory(self, handle: int):
        """-> (blocks [n, 64] uint8, cols [n, 16] uint8): the part's device block directory, byte for byte (diagnostics)."""
        nb, nc = C.c_uint64(), C.c_uint64()
        _check(self._L.bydb_part_directory(self._h, handle, None, 0, None, 0, C.byref(nb), C.byref(nc)))
        blocks = np.zeros((nb.value, 64), dtype=np.uint8)
        cols = np.zeros((nc.value, 16), dtype=np.uint8)
        _check(self._L.bydb_part_directory(self._h, handle, blocks.ctypes.data, blocks.nbytes, cols.ctypes.data, cols.nbytes, C.byref(nb), C.byref(nc)))
        return blocks, cols

    # ---- queries
    def prepare(self, q: Query) -> PreparedQuery:
        return PreparedQuery(q)

    def scan_agg(self, q) -> Result:
        cq, keep = _cq(q)
        r = _Result()
        _check(self._L.bydb_scan_agg(self._h, C.byref(cq), C.byref(r)))
        try:
            return _read_result(r)
        finally:
            self._L.bydb_result_free(self._h, C.byref(r))

    def scan_agg_keyed(self, q: Query, family: str, tag: str, max_values: int = 0) -> Result:
        """Group-by on a stored tag (bydb_scan_agg_keyed): rows carry (series group, key value)."""
        keep: list = []
        cq = _mk_query(q, keep)
        fb, tb = family.encode(), tag.encode()
        gk = _GroupKey(fb, tb, max_values, 0)
        r = _KeyedResult()
        _check(self._L.bydb_scan_agg_keyed(self._h, C.byref(cq), C.byref(gk), C.byref(r)))
        return self._read_keyed(r, len(q.aggs))

    def _read_keyed(self, r: _KeyedResult, n_aggs: int) -> Result:
        try:
            if r.base.n_rows == 0 and not r.base.owner:
                a = n_aggs
                res = Result(np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(a, bool), np.zeros((0, a), np.int64),
                             np.zeros((0, a), np.float64), Stats.of(r.base.stats))
            else:
                res = _read_result(r.base)
            keys = [bytes(r.key_bytes[r.key_off[k]:r.key_off[k + 1]]) for k in range(r.n_keys)]
            res.key = [keys[r.key_id[i]] for i in range(r.base.n_rows)]
            res.n_keys = r.n_keys
            return res
        finally:
            self._L.bydb_keyed_result_free(self._h, C.byref(r))

    def encode_pages(self, values: np.ndarray, block_rows: Sequence[int]):
        """Write side (bydb_encode_pages): int64 / float64 value blocks -> ([page bytes or None per block], device ms).
        None = the block needs the CPU writer."""
        vt = VT_FLOAT64 if values.dtype == np.float64 else VT_INT64
        vals = np.ascontiguousarray(values, dtype=np.float64 if vt == VT_FLOAT64 else np.int64)
        rows = np.ascontiguousarray(block_rows, dtype=np.uint32)
        assert int(rows.sum()) == vals.size
        inp = _EncodeInput(vt, rows.size, rows.ctypes.data, vals.ctypes.data)
        r = _EncodedPages()
        _check(self._L.bydb_encode_pages(self._h, C.byref(inp), C.byref(r)))
        try:
            n = r.n_blocks
            off = np.ctypeslib.as_array(r.page_off, (n + 1,)).copy() if n else np.zeros(1, np.uint64)
            total = int(off[-1])
            data = np.ctypeslib.as_array(r.bytes, (max(total, 1),))[:total].tobytes()
            pages = [None if r.needs_cpu[b] else data[int(off[b]):int(off[b + 1])] for b in range(n)]
            return pages, float(r.device_ms)
        finally:
            self._L.bydb_encoded_pages_free(self._h, C.byref(r))

    # ---- prepared queries replayed as one captured CUDA graph (bydb_query_prepare / bydb_scan_agg_prepared)
    def prepare_graph(self, q: Query) -> "GraphQuery":
        keep: list = []
        cq = _mk_query(q, keep)
        h = C.c_void_p()
        _check(self._L.bydb_query_prepare(self._h, C.byref(cq), C.byref(h)))
        return GraphQuery(self, h)

    def scan_agg_host(self, parts: Sequence[Dict[str, Union[bytes, np.ndarray]]], q: Query) -> Result:
        keep: list = []
        arr = (_PartFiles * len(parts))()
        for i, files in enumerate(parts):
            arr[i] = _part_files(files, keep)
        cq = _mk_query(q, keep)
        r = _Result()
        _check(self._L.bydb_scan_agg_host(self._h, len(parts), arr, C.byref(cq), C.byref(r)))
        try:
            return _read_result(r)
        finally:
            self._L.bydb_result_free(self._h, C.byref(r))

    # ---- multi-GPU map / reduce
    def partials_layout(self, q: Query) -> Dict[str, int]:
        keep: list = []
        cq = _mk_query(q, keep)
        lay = _Layout()
        _check(self._L.bydb_partials_layout(C.byref(cq), C.byref(lay)))
        return {k: getattr(lay, k) for k, _ in _Layout._fields_}

    def scan_partials(self, q, d_ptr: int, nbytes: int, stream: int = 0, want_stats: bool = True) -> Optional[Stats]:
        """want_stats=False is the asynchronous form: returns as soon as the scan is enqueued on `stream`; failures
        surface in reduce_finalize (they travel in the table)."""
        cq, keep = _cq(q)
        if not want_stats:
            _check(self._L.bydb_scan_partials(self._h, C.byref(cq), d_ptr, nbytes, stream or None, None))
            return None
        st = _Stats()
        _check(self._L.bydb_scan_partials(self._h, C.byref(cq), d_ptr, nbytes, stream or None, C.byref(st)))
        return Stats.of(st)

    def partials_rows(self, q, d_ptr: int, nbytes: int, stream: int = 0) -> Dict[str, np.ndarray]:
        """Map-phase rows of a partial table in the reference's wire shape (emitPartial): per group and aggregate
        Partial.Value (+ Partial.Count for MEAN), typed like the field."""
        cq, keep = _cq(q)
        r = _PartialRows()
        _check(self._L.bydb_partials_rows(self._h, C.byref(cq), d_ptr, nbytes, stream or None, C.byref(r)))
        try:
            n, a = r.n_rows, r.n_aggs
            f = lambda ptr, cnt, dt: np.array(ptr[:cnt], dtype=dt)  # noqa: E731
            return dict(group_id=f(r.group_id, n, np.int32), is_float=f(r.is_float, a, np.uint8).astype(bool),
                        val_i64=f(r.val_i64, n * a, np.int64).reshape(n, a), val_f64=f(r.val_f64, n * a, np.float64).reshape(n, a),
                        cnt_i64=f(r.cnt_i64, n * a, np.int64).reshape(n, a), cnt_f64=f(r.cnt_f64, n * a, np.float64).reshape(n, a))
        finally:
            self._L.bydb_partial_rows_free(self._h, C.byref(r))

    # ---- multi-GPU reduce behind the C ABI (peer mailboxes over NVLink; no torch / NCCL on the data path)
    def comm_export(self, max_table_bytes: int, max_ranks: int) -> bytes:
        """-> this rank's 128-byte mailbox handle; exchange the handles of all ranks, then comm_connect."""
        buf = C.create_string_buffer(128)
        _check(self._L.bydb_comm_export(self._h, max_table_bytes, max_ranks, buf))
        return buf.raw

    def comm_connect(self, rank: int, nranks: int, handles: Sequence[bytes]) -> None:
        assert len(handles) == nranks and all(len(h) == 128 for h in handles)
        buf = C.create_string_buffer(b"".join(handles), 128 * nranks)
        _check(self._L.bydb_comm_connect(self._h, rank, nranks, buf))

    def scan_reduce(self, q, root: int = 0) -> Result:
        """Collective: every rank scans its parts, the partial tables meet in the root's mailbox, the root finalises.
        Non-root ranks get an empty result (n_rows = 0) with their own scan statistics."""
        cq, keep = _cq(q)
        r = _Result()
        _check(self._L.bydb_scan_reduce(self._h, C.byref(cq), root, C.byref(r)))
        try:
            return _read_result(r)
        finally:
            self._L.bydb_result_free(self._h, C.byref(r))

    def keyed_reduce_layout(self, q: Query, family: str, tag: str, max_values: int = 0) -> int:
        """Mailbox slot bytes scan_reduce_keyed needs for q: pass the largest over the queries to come to comm_export."""
        return keyed_reduce_layout(q, family, tag, max_values)

    def scan_reduce_keyed(self, q: Query, family: str, tag: str, root: int = 0, max_values: int = 0) -> Result:
        """Group-by on a stored tag as a collective (bydb_scan_reduce_keyed): the root gets what scan_agg_keyed over every rank's
        parts and series returns, .key and .n_keys included; the other ranks get an empty result with their own scan statistics."""
        keep: list = []
        cq = _mk_query(q, keep)
        gk = _GroupKey(family.encode(), tag.encode(), max_values, 0)
        r = _KeyedResult()
        _check(self._L.bydb_scan_reduce_keyed(self._h, C.byref(cq), C.byref(gk), root, C.byref(r)))
        return self._read_keyed(r, len(q.aggs))

    def scan_reduce_host(self, parts: Sequence[Dict[str, Union[bytes, np.ndarray]]], q: Query, root: int = 0) -> Result:
        keep: list = []
        arr = (_PartFiles * len(parts))()
        for i, files in enumerate(parts):
            arr[i] = _part_files(files, keep)
        cq = _mk_query(q, keep)
        r = _Result()
        _check(self._L.bydb_scan_reduce_host(self._h, len(parts), arr, C.byref(cq), root, C.byref(r)))
        try:
            return _read_result(r)
        finally:
            self._L.bydb_result_free(self._h, C.byref(r))

    def partials_combine(self, q, d_ptr: int, n_tables: int, bytes_each: int, stream: int = 0) -> None:
        cq, keep = _cq(q)
        _check(self._L.bydb_partials_combine(self._h, C.byref(cq), d_ptr, n_tables, bytes_each, stream or None))

    def reduce_finalize(self, q, d_ptr: int, nbytes: int, stream: int = 0) -> Result:
        cq, keep = _cq(q)
        r = _Result()
        _check(self._L.bydb_reduce_finalize(self._h, C.byref(cq), d_ptr, nbytes, stream or None, C.byref(r)))
        try:
            return _read_result(r)
        finally:
            self._L.bydb_result_free(self._h, C.byref(r))
