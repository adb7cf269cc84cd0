"""ctypes binding of libpinot_b200.so (include/pinot_b200.h + include/pinot_b200_host.h).

This is what tests and bench.py call; it is the Python twin of the JNI shim (jni/pinot_b200_jni.c).  There is no
fallback: if the shared library is missing or no CUDA device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Sequence

import numpy as np

from .query import AggOp, QueryContext
from .segment_writer import DataType, Segment

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PB_LIB_PATH") or os.path.join(_HERE, "libpinot_b200.so")      # (PB_LIB_PATH: a scratch build, see build.py)

PB_Q_COMBINE = 1
PB_Q_DEFER_FINALIZE = 2
PB_Q_GENERIC_KERNEL = 4
PB_Q_NO_TMA = 8
PB_Q_GATHER_IN_PLACE = 16
PB_Q_ALL_RANKS = 32
PB_COMM_ID_BYTES = 128


class PbColumnDesc(C.Structure):
    _fields_ = [("name", C.c_char_p), ("stored_type", C.c_int32), ("has_dictionary", C.c_int32),
                ("is_sorted", C.c_int32), ("cardinality", C.c_int32), ("bits_per_element", C.c_int32),
                ("dict_entry_bytes", C.c_int32),
                ("forward_index", C.c_void_p), ("forward_index_len", C.c_uint64),
                ("dictionary", C.c_void_p), ("dictionary_len", C.c_uint64),
                ("inverted_index", C.c_void_p), ("inverted_index_len", C.c_uint64),
                ("null_value_vector", C.c_void_p), ("null_value_vector_len", C.c_uint64)]


class PbSegmentDesc(C.Structure):
    _fields_ = [("segment_name", C.c_char_p), ("num_docs", C.c_int32), ("num_columns", C.c_int32),
                ("columns", C.POINTER(PbColumnDesc))]


class PbAggregationDesc(C.Structure):
    _fields_ = [("op", C.c_int32), ("column", C.c_char_p)]


class PbExecStats(C.Structure):
    _fields_ = [("num_docs_scanned", C.c_int64), ("num_entries_scanned_in_filter", C.c_int64),
                ("num_entries_scanned_post_filter", C.c_int64), ("num_total_docs", C.c_int64),
                ("num_groups_limit_reached", C.c_int32), ("num_segments", C.c_int32)]


class PbhPredicate(C.Structure):
    _fields_ = [("type", C.c_int32), ("column", C.c_char_p), ("num_values", C.c_int32),
                ("values", C.POINTER(C.c_char_p)), ("lower", C.c_char_p), ("upper", C.c_char_p),
                ("lower_inclusive", C.c_int32), ("upper_inclusive", C.c_int32)]


class PbhFilterNode(C.Structure):
    _fields_ = [("kind", C.c_int32), ("num_children", C.c_int32), ("predicate", C.c_int32)]


class PbhFilterProgram(C.Structure):
    _fields_ = [("num_filter_nodes", C.c_int32), ("filter_nodes", C.POINTER(PbhFilterNode)),
                ("predicates", C.POINTER(PbhPredicate))]


class PbOrderBy(C.Structure):
    _fields_ = [("kind", C.c_int32), ("index", C.c_int32), ("descending", C.c_int32)]


class PbhQueryContext(C.Structure):
    _fields_ = [("num_filter_nodes", C.c_int32), ("filter_nodes", C.POINTER(PbhFilterNode)),
                ("predicates", C.POINTER(PbhPredicate)),
                ("num_group_by", C.c_int32), ("group_by_columns", C.POINTER(C.c_char_p)),
                ("num_aggregations", C.c_int32), ("aggregations", C.POINTER(PbAggregationDesc)),
                ("num_groups_limit", C.c_int32), ("max_initial_result_holder_capacity", C.c_int32),
                ("num_skip_inverted", C.c_int32), ("skip_inverted_columns", C.POINTER(C.c_char_p)),
                ("num_agg_filters", C.c_int32), ("agg_filters", C.POINTER(PbhFilterProgram)),
                ("agg_filter_of", C.POINTER(C.c_int32)),
                ("num_order_by", C.c_int32), ("order_by", C.POINTER(PbOrderBy)), ("trim_size", C.c_int32), ("trim_threshold", C.c_int32),
                ("null_handling", C.c_int32)]


_lib = None


def lib():
    """Load the native library; raises if it has not been built (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the executor has no CPU fallback)")
    l = C.CDLL(LIB_PATH)
    l.pb_last_error.restype = C.c_char_p
    l.pb_init.argtypes = [C.POINTER(C.c_int), C.c_int, C.c_size_t]
    l.pb_device_count.restype = C.c_int
    l.pb_comm_unique_id.argtypes = [C.c_void_p, C.c_size_t]
    l.pb_comm_init.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_size_t]
    l.pb_comm_info.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_int)]
    l.pb_result_comm_ms.argtypes = [C.c_void_p]
    l.pb_result_comm_ms.restype = C.c_double
    l.pb_segment_stage.argtypes = [C.POINTER(PbSegmentDesc), C.c_int, C.POINTER(C.c_void_p)]
    l.pb_segment_release.argtypes = [C.c_void_p]
    l.pb_cache_stats.argtypes = [C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    l.pb_segment_device_bytes.argtypes = [C.c_void_p]
    l.pb_segment_device_bytes.restype = C.c_int64
    l.pb_segment_group_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]
    l.pb_segment_group_release.argtypes = [C.c_void_p]
    l.pb_segment_group_export_dictionary.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p),
                                                     C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
    l.pb_segment_group_set_global_dictionary.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.c_int32]
    l.pb_segment_group_remap.argtypes = [C.c_void_p, C.c_char_p, C.c_int32, C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.c_int32)]
    l.pbh_execute.argtypes = [C.c_void_p, C.POINTER(PbhQueryContext), C.c_uint32, C.POINTER(C.c_void_p)]
    l.pbh_is_eligible.argtypes = [C.c_void_p, C.POINTER(PbhQueryContext)]
    l.pbh_explain_filter.argtypes = [C.c_void_p, C.c_int32, C.POINTER(PbhQueryContext), C.c_char_p, C.c_int32]
    l.pbh_explain_agg_filter.argtypes = [C.c_void_p, C.c_int32, C.POINTER(PbhQueryContext), C.c_int32, C.c_char_p, C.c_int32]
    l.pbh_dump_lowered.argtypes = [C.c_void_p, C.c_int32, C.POINTER(PbhQueryContext), C.c_int32, C.c_char_p, C.c_int32]
    l.pbh_null_clause_plan.argtypes = [C.c_void_p, C.POINTER(PbhQueryContext), C.POINTER(C.c_int32), C.c_int32]
    l.pbh_null_clause_plan.restype = C.c_int32
    l.pb_result_free.argtypes = [C.c_void_p]
    l.pb_result_finalize.argtypes = [C.c_void_p]
    l.pb_result_num_tables.argtypes = [C.c_void_p]
    l.pb_result_num_tables.restype = C.c_int32
    l.pb_result_num_groups.argtypes = [C.c_void_p, C.c_int32]
    l.pb_result_num_groups.restype = C.c_int64
    l.pb_result_group_dict_ids.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    l.pb_result_group_dict_ids.restype = C.POINTER(C.c_int32)
    l.pb_result_group_key_values.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    l.pb_result_group_key_values.restype = C.c_void_p
    l.pb_result_double.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    l.pb_result_double.restype = C.POINTER(C.c_double)
    l.pb_result_long.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    l.pb_result_long.restype = C.POINTER(C.c_int64)
    l.pb_result_distinct_offsets.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    l.pb_result_distinct_offsets.restype = C.POINTER(C.c_int64)
    l.pb_result_distinct_dict_ids.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    l.pb_result_distinct_dict_ids.restype = C.POINTER(C.c_int32)
    l.pb_result_distinct_values.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    l.pb_result_distinct_values.restype = C.POINTER(C.c_int64)
    l.pb_result_stats.argtypes = [C.c_void_p, C.c_int32]
    l.pb_result_stats.restype = C.POINTER(PbExecStats)
    l.pb_result_device_ms.argtypes = [C.c_void_p]
    l.pb_result_device_ms.restype = C.c_double
    l.pb_result_scan_kernel_ms.argtypes = [C.c_void_p]
    l.pb_result_scan_kernel_ms.restype = C.c_double
    l.pb_result_kernel_launches.argtypes = [C.c_void_p]
    l.pb_result_kernel_launches.restype = C.c_int32
    l.pb_result_in_place_columns.argtypes = [C.c_void_p]
    l.pb_result_in_place_columns.restype = C.c_int32
    l.pb_result_residual_leaves.argtypes = [C.c_void_p]
    l.pb_result_residual_leaves.restype = C.c_int32
    l.pb_result_stream.argtypes = [C.c_void_p]
    l.pb_result_stream.restype = C.c_void_p
    l.pb_result_wait.argtypes = [C.c_void_p]
    l.pb_result_merge_gathered.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
    l.pb_result_phase_ms.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    l.pb_result_host_timing.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    l.pb_host_register.argtypes = [C.c_void_p, C.c_size_t]
    l.pb_host_unregister.argtypes = [C.c_void_p]
    l.pb_result_device_buffer.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
    _lib = l
    return l


class PinotB200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"pinot_b200 error {code}: {msg}")
        self.code = code


def _check(rc: int):
    if rc != 0:
        raise PinotB200Error(rc, lib().pb_last_error().decode("utf-8", "replace"))


def init(device=None, hbm_cache_bytes: int = 0):
    """pb_init.  device: None = the current CUDA device, an int, or a list of CUDA device ordinals driven by this process
    (segments are then staged on a device_index into that list)."""
    if device is None:
        _check(lib().pb_init(None, 0, hbm_cache_bytes))
    else:
        ids = [device] if isinstance(device, int) else list(device)
        arr = (C.c_int * len(ids))(*ids)
        _check(lib().pb_init(arr, len(ids), hbm_cache_bytes))


def cache_stats(device_index: int = 0):
    """(bytes staged in HBM right now, segments evicted so far) of one device's segment cache"""
    b, e = C.c_int64(), C.c_int64()
    _check(lib().pb_cache_stats(device_index, C.byref(b), C.byref(e)))
    return b.value, e.value


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(PB_COMM_ID_BYTES)
    _check(lib().pb_comm_unique_id(buf, PB_COMM_ID_BYTES))
    return buf.raw


def comm_init(n_ranks: int, rank: int, unique_id: bytes):
    """ncclCommInitRank inside libpinot_b200.so (collective: every rank calls it with rank 0's id)."""
    assert len(unique_id) == PB_COMM_ID_BYTES
    buf = C.create_string_buffer(unique_id, PB_COMM_ID_BYTES)
    _check(lib().pb_comm_init(n_ranks, rank, buf, PB_COMM_ID_BYTES))


def comm_info():
    n, r = C.c_int(), C.c_int()
    has = lib().pb_comm_info(C.byref(n), C.byref(r))
    return bool(has), n.value, r.value


def comm_destroy():
    _check(lib().pb_comm_destroy())


class StagedSegment:
    """IndexSegment handle on the device (pb_segment_stage).  Keeps the host buffers alive."""

    def __init__(self, seg: Segment, columns: Optional[Sequence[str]] = None, device_index: int = 0):
        self.segment = seg
        self.device_index = device_index
        names = list(columns) if columns is not None else seg.column_names()
        self._keep = []
        cols = (PbColumnDesc * len(names))()
        for i, n in enumerate(names):
            c = seg.columns[n]
            d = cols[i]
            d.name = n.encode()
            d.stored_type = int(c.data_type)
            d.has_dictionary = int(c.has_dictionary)
            d.is_sorted = int(c.is_sorted)
            d.cardinality = c.cardinality
            d.bits_per_element = c.bits_per_element
            d.dict_entry_bytes = c.dict_entry_bytes
            d.forward_index = c.forward_index.ctypes.data
            d.forward_index_len = c.forward_index.size
            if c.dictionary is not None:
                d.dictionary = c.dictionary.ctypes.data
                d.dictionary_len = c.dictionary.size
            if c.inverted_index is not None:
                d.inverted_index = c.inverted_index.ctypes.data
                d.inverted_index_len = c.inverted_index.size
            if getattr(c, "null_value_vector", None) is not None:
                d.null_value_vector = c.null_value_vector.ctypes.data
                d.null_value_vector_len = c.null_value_vector.size
        desc = PbSegmentDesc(seg.name.encode(), seg.num_docs, len(names), cols)
        self._keep.append((cols, desc))
        h = C.c_void_p()
        _check(lib().pb_segment_stage(C.byref(desc), device_index, C.byref(h)))
        self.handle = h

    def device_bytes(self) -> int:
        return lib().pb_segment_device_bytes(self.handle)

    def release(self):
        if self.handle:
            lib().pb_segment_release(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class SegmentGroup:
    def __init__(self, staged: Sequence[StagedSegment]):
        self.staged = list(staged)
        arr = (C.c_void_p * len(self.staged))(*[s.handle for s in self.staged])
        h = C.c_void_p()
        _check(lib().pb_segment_group_create(arr, len(self.staged), C.byref(h)))
        self.handle = h

    def export_dictionary(self, column: str) -> np.ndarray:
        p, n, eb = C.c_void_p(), C.c_int64(), C.c_int32()
        _check(lib().pb_segment_group_export_dictionary(self.handle, column.encode(), C.byref(p), C.byref(n), C.byref(eb)))
        raw = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n.value * eb.value,)).copy()
        return raw.reshape(n.value, eb.value)

    def set_global_dictionary(self, column: str, entries: np.ndarray):
        e = np.ascontiguousarray(entries, dtype=np.uint8)
        _check(lib().pb_segment_group_set_global_dictionary(self.handle, column.encode(), e.ctypes.data, e.shape[0], e.shape[1]))

    def remap(self, column: str, segment_index: int) -> np.ndarray:
        p, n = C.POINTER(C.c_int32)(), C.c_int32()
        _check(lib().pb_segment_group_remap(self.handle, column.encode(), segment_index, C.byref(p), C.byref(n)))
        return np.ctypeslib.as_array(p, shape=(n.value,)).copy()

    def release(self):
        if self.handle:
            lib().pb_segment_group_release(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


_KEY_DT = {0: np.int32, 1: np.int64, 2: np.float32, 3: np.float64}


class ResultTable:
    """One GroupByResultsBlock / AggregationResultsBlock.  Arrays are zero-copy views of the result handle's pinned
    host memory, created on first access (valid until Result.free())."""

    def __init__(self, rh, t: int, q: QueryContext, parent=None):
        l = lib()
        self._rh, self._t, self.query = rh, t, q
        self._parent = parent          # the views below point into the Result's pinned memory: keep it alive
        self.num_groups = int(l.pb_result_num_groups(rh, t))
        st = l.pb_result_stats(rh, t).contents
        self.stats = {k: getattr(st, k) for k, _ in PbExecStats._fields_}
        self._cache = {}

    def _view(self, name, fn):
        if name not in self._cache:
            self._cache[name] = fn()
        return self._cache[name]

    @property
    def key_dict_ids(self):
        def load():
            n = max(self.num_groups, 1)
            return [np.ctypeslib.as_array(lib().pb_result_group_dict_ids(self._rh, self._t, j), shape=(n,))[:self.num_groups]
                    for j in range(len(self.query.group_by))]
        return self._view("ids", load)

    @property
    def key_values(self):
        def load():
            out, n = [], max(self.num_groups, 1)
            for j in range(len(self.query.group_by)):
                ty, eb = C.c_int32(), C.c_int32()
                p = lib().pb_result_group_key_values(self._rh, self._t, j, C.byref(ty), C.byref(eb))
                raw = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n * eb.value,))[:self.num_groups * eb.value]
                if ty.value == 4:
                    out.append(np.array([bytes(r).rstrip(b"\0") for r in raw.reshape(self.num_groups, eb.value)], dtype=object))
                else:
                    out.append(raw.view(_KEY_DT[ty.value]))
            return out
        return self._view("vals", load)

    @property
    def doubles(self):
        n = max(self.num_groups, 1)
        return self._view("dbl", lambda: [np.ctypeslib.as_array(lib().pb_result_double(self._rh, self._t, a), shape=(n,))[:self.num_groups]
                                          for a in range(len(self.query.aggregations))])

    @property
    def longs(self):
        n = max(self.num_groups, 1)
        return self._view("lng", lambda: [np.ctypeslib.as_array(lib().pb_result_long(self._rh, self._t, a), shape=(n,))[:self.num_groups]
                                          for a in range(len(self.query.aggregations))])

    @property
    def distinct(self):
        def load():
            out = []
            for a, agg in enumerate(self.query.aggregations):
                if agg.op == AggOp.DISTINCTCOUNT:
                    off = np.ctypeslib.as_array(lib().pb_result_distinct_offsets(self._rh, self._t, a), shape=(self.num_groups + 1,))
                    tot = int(off[-1])
                    p = lib().pb_result_distinct_dict_ids(self._rh, self._t, a)
                    if not p:       # raw column: the value sets as bits (int64)
                        p = lib().pb_result_distinct_values(self._rh, self._t, a)
                    ids = np.ctypeslib.as_array(p, shape=(max(tot, 1),))[:tot]
                    out.append((off, ids))
                else:
                    out.append(None)
            return out
        return self._view("dc", load)

    def keys(self) -> List[tuple]:
        vals = self.key_values
        return [tuple(v[g].item() if hasattr(v[g], "item") else v[g] for v in vals) for g in range(self.num_groups)]

    def rows(self) -> Dict[tuple, list]:
        """key -> [per-aggregation value]: COUNT int, SUM/MIN/MAX float, AVG (sum, count), DISTINCTCOUNT count."""
        ks = self.keys() if self.query.group_by else [()]
        dbl, lng = self.doubles, self.longs
        out = {}
        nh = getattr(self.query, "null_handling", False)      # the long array then holds the inputs every function saw: 0 = SQL NULL
        for g, k in enumerate(ks):
            row = []
            for a, agg in enumerate(self.query.aggregations):
                if agg.op in (AggOp.COUNT, AggOp.DISTINCTCOUNT):
                    row.append(int(lng[a][g]))
                elif nh and int(lng[a][g]) == 0:
                    row.append(None)
                elif agg.op == AggOp.AVG:
                    row.append((float(dbl[a][g]), int(lng[a][g])))
                else:
                    row.append(float(dbl[a][g]))
            out[k] = row
        return out


class Result:
    def __init__(self, rh, q: QueryContext, deferred: bool = False):
        self._rh = rh
        self.query = q
        self._finalized = not deferred
        self.in_place_columns = lib().pb_result_in_place_columns(rh)     # known as soon as the call is planned
        self.residual_leaves = lib().pb_result_residual_leaves(rh)       # filter leaves tested by the aggregation kernel
        if not deferred:
            self._load()

    @property
    def tables(self) -> List[ResultTable]:
        """Built on access and not cached: a table keeps its Result alive (its arrays are views of the Result's pinned
        memory) but the Result does not reference its tables, so no reference cycle is left for the GC."""
        if not self._finalized:
            return []
        return [ResultTable(self._rh, t, self.query, self) for t in range(lib().pb_result_num_tables(self._rh))]

    def _load(self):
        l = lib()
        self._finalized = True
        self.device_ms = l.pb_result_device_ms(self._rh)
        self.scan_kernel_ms = l.pb_result_scan_kernel_ms(self._rh)
        self.kernel_launches = l.pb_result_kernel_launches(self._rh)
        self.in_place_columns = l.pb_result_in_place_columns(self._rh)

    def device_buffer(self, which: int, agg: int = 0):
        p, n = C.c_void_p(), C.c_int64()
        _check(lib().pb_result_device_buffer(self._rh, which, agg, C.byref(p), C.byref(n)))
        return p.value, n.value

    def merge_gathered(self, gathered_ptr: int, n_ranks: int):
        _check(lib().pb_result_merge_gathered(self._rh, gathered_ptr, n_ranks))

    def stream(self) -> int:
        return lib().pb_result_stream(self._rh) or 0

    def phase_ms(self):
        f, a = C.c_double(), C.c_double()
        _check(lib().pb_result_phase_ms(self._rh, C.byref(f), C.byref(a)))
        return f.value, a.value

    def host_timing_us(self):
        arr = (C.c_double * 8)()
        _check(lib().pb_result_host_timing(self._rh, arr))
        return list(arr)

    def wait(self):
        _check(lib().pb_result_wait(self._rh))

    def comm_ms(self) -> float:
        """device time of the cross-rank merge of this call (collective + merge kernel), 0 without PB_Q_ALL_RANKS"""
        return lib().pb_result_comm_ms(self._rh)

    def scan_ms(self) -> float:
        return lib().pb_result_scan_kernel_ms(self._rh)

    def finalize(self):
        _check(lib().pb_result_finalize(self._rh))
        self._load()

    def free(self):
        if self._rh:
            lib().pb_result_free(self._rh)
            self._rh = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class _MarshalledQuery:
    def _filter(self, flt):
        """one filter expression -> (n_nodes, PbhFilterNode[], PbhPredicate[])"""
        from .query import postfix_of
        nodes, preds = postfix_of(flt)
        cn = (PbhFilterNode * max(1, len(nodes)))()
        for i, (k, n, p) in enumerate(nodes):
            cn[i].kind, cn[i].num_children, cn[i].predicate = k, n, p
        cp = (PbhPredicate * max(1, len(preds)))()
        for i, p in enumerate(preds):
            o = cp[i]
            o.type = int(p.type)
            o.column = p.column.encode()
            if int(p.type) == 4:
                o.lower = p.lower.encode() if p.lower is not None else None
                o.upper = p.upper.encode() if p.upper is not None else None
                o.lower_inclusive = int(p.lower_inclusive)
                o.upper_inclusive = int(p.upper_inclusive)
            else:
                arr = (C.c_char_p * max(1, len(p.values)))(*[v.encode() for v in p.values])
                self.keep.append(arr)
                o.values = arr
                o.num_values = len(p.values)
        self.keep.append((cn, cp))
        return len(nodes), cn, cp

    def __init__(self, q: QueryContext):
        self.keep = []
        n_nodes, self.nodes, self.preds = self._filter(q.filter)
        nodes = [None] * n_nodes
        self.gb = (C.c_char_p * max(1, len(q.group_by)))(*[c.encode() for c in q.group_by])
        self.aggs = (PbAggregationDesc * max(1, len(q.aggregations)))()
        for i, a in enumerate(q.aggregations):
            self.aggs[i].op = int(a.op)
            keep_col = a.column is not None and (int(a.op) != 0 or getattr(q, "null_handling", False))   # COUNT(col) = COUNT(*) unless nulls are handled
            self.aggs[i].column = a.column.encode() if keep_col else None
        skip = [c for c, kinds in q.skip_indexes.items() if "inverted" in kinds]
        self.skip = (C.c_char_p * max(1, len(skip)))(*[c.encode() for c in skip])
        filters, filter_of = q.agg_filters()
        self.progs = (PbhFilterProgram * max(1, len(filters)))()
        for i, f in enumerate(filters):
            n, cn, cp = self._filter(f)
            self.progs[i].num_filter_nodes, self.progs[i].filter_nodes, self.progs[i].predicates = n, cn, cp
        self.filter_of = (C.c_int32 * max(1, len(filter_of)))(*filter_of)
        self.ctx = PbhQueryContext(len(nodes), self.nodes, self.preds, len(q.group_by), self.gb,
                                   len(q.aggregations), self.aggs, q.num_groups_limit,
                                   q.max_initial_result_holder_capacity, len(skip), self.skip,
                                   len(filters), self.progs, self.filter_of)
        self.order = (PbOrderBy * max(1, len(q.order_by)))()
        for i, (kind, index, desc) in enumerate(q.order_by):
            self.order[i].kind, self.order[i].index, self.order[i].descending = kind, index, int(desc)
        self.ctx.num_order_by, self.ctx.order_by = len(q.order_by), self.order
        self.ctx.null_handling = int(getattr(q, "null_handling", False))
        self.trims = {True: q.trim(True), False: q.trim(False)}


def prepare(q: QueryContext) -> "_MarshalledQuery":
    """Marshal a QueryContext once; pass it to execute(prepared=...) when the same query runs many times."""
    return _MarshalledQuery(q)


def execute(group: SegmentGroup, q: QueryContext, flags: int = 0, prepared: Optional["_MarshalledQuery"] = None) -> Result:
    """Plan (host layer) + run (device) a query over every segment of the group."""
    m = prepared if prepared is not None else _MarshalledQuery(q)
    # ORDER BY ... LIMIT trim: the server-level trim of the combine layer for a merged table, the segment-level one otherwise
    m.ctx.trim_size, m.ctx.trim_threshold = m.trims[bool(flags & PB_Q_COMBINE)]
    rh = C.c_void_p()
    _check(lib().pbh_execute(group.handle, C.byref(m.ctx), flags, C.byref(rh)))
    return Result(rh, q, deferred=bool(flags & PB_Q_DEFER_FINALIZE))


def host_register(arr: np.ndarray):
    _check(lib().pb_host_register(arr.ctypes.data, arr.nbytes))


def host_unregister(arr: np.ndarray):
    _check(lib().pb_host_unregister(arr.ctypes.data))


def is_eligible(group: SegmentGroup, q: QueryContext) -> bool:
    m = _MarshalledQuery(q)
    return lib().pbh_is_eligible(group.handle, C.byref(m.ctx)) == 0


def dump_lowered(group: SegmentGroup, q: QueryContext, clause: int = -1, segment_index: int = 0) -> List[str]:
    """The lowered pb_filter_node program of one segment (clause -1 = WHERE filter), one postfix node per line."""
    m = _MarshalledQuery(q)
    cap = 1 << 16
    while True:
        buf = C.create_string_buffer(cap)
        n = lib().pbh_dump_lowered(group.handle, segment_index, C.byref(m.ctx), clause, buf, cap)
        if n < 0:
            _check(n)
        if n < cap:
            return buf.value.decode().splitlines()
        cap = n + 1


def clause_plan(group: SegmentGroup, q: QueryContext):
    """(number of FILTER clauses the device runs for q, clause index per aggregation): the query's own clauses, or with
    enableNullHandling the (own clause, nullable input column) pairs (pbh_null_clause_plan)."""
    m = _MarshalledQuery(q)
    n = len(q.aggregations)
    of = (C.c_int32 * max(1, n))()
    k = lib().pbh_null_clause_plan(group.handle, C.byref(m.ctx), of, n)
    if k < 0:
        _check(k)
    return k, list(of)[:n]


def explain_agg_filter(group: SegmentGroup, q: QueryContext, clause: int, segment_index: int = 0) -> str:
    """EXPLAIN of FILTER clause `clause` (index into QueryContext.agg_filters()[0]) as planned for one segment."""
    m = _MarshalledQuery(q)
    buf = C.create_string_buffer(8192)
    n = lib().pbh_explain_agg_filter(group.handle, segment_index, C.byref(m.ctx), clause, buf, 8192)
    if n < 0:
        _check(n)
    return buf.value.decode()


def explain_filter(group: SegmentGroup, q: QueryContext, segment_index: int = 0) -> str:
    m = _MarshalledQuery(q)
    buf = C.create_string_buffer(8192)
    n = lib().pbh_explain_filter(group.handle, segment_index, C.byref(m.ctx), buf, 8192)
    if n < 0:
        _check(n)
    return buf.value.decode()
