"""ctypes binding of libb200vs.so (include/b200vs.h) — harness glue for tests/ and bench.py.

The product is the C-ABI shared library; this module only loads it and marshals numpy / torch buffers.
It fails loudly when the CUDA library is missing: there is no CPU fallback anywhere in the product path.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
PKG_ROOT = os.path.abspath(os.path.join(_HERE, "..", ".."))       # dingo-store_b200/
REPO_ROOT = os.path.abspath(os.path.join(PKG_ROOT, ".."))
LIB_PATH = os.path.join(PKG_ROOT, "libb200vs.so")

FLAT, IVF_FLAT, IVF_PQ, HNSW, BINARY_FLAT, BINARY_IVF_FLAT = 0, 1, 2, 3, 4, 5
L2, IP, COSINE, HAMMING = 1, 2, 3, 4
BINARY_TYPES = (BINARY_FLAT, BINARY_IVF_FLAT)
OK, EILLEGAL_PARAMETERS, EVECTOR_INVALID, EVECTOR_NOT_TRAIN, EVECTOR_NOT_SUPPORT, EINTERNAL, EVECTOR_ID_DUPLICATED = range(7)

# every symbol include/b200vs.h declares (checked by tests/test_abi.py without a GPU)
ABI_SYMBOLS = [
    "b200vs_create", "b200vs_destroy", "b200vs_train", "b200vs_set_trained_state", "b200vs_get_trained_state",
    "b200vs_add_with_ids", "b200vs_remove_ids", "b200vs_search", "b200vs_search_device", "b200vs_coarse_device", "b200vs_search_probes_device", "b200vs_range_search",
    "b200vs_count", "b200vs_deleted_count", "b200vs_memory_size", "b200vs_is_trained", "b200vs_dimension",
    "b200vs_save", "b200vs_load", "b200vs_export_lists", "b200vs_merge_topk_device", "b200vs_last_search_stats", "b200vs_last_phase_times", "b200vs_calc_distance",
    "b200vs_scan_begin", "b200vs_scan_push", "b200vs_scan_finish", "b200vs_scan_abort", "b200vs_set_profiling",
    "b200vs_last_error", "b200vs_version",
    "b200vs_add_with_ids_device", "b200vs_assign_device", "b200vs_reserve_lists", "b200vs_export_list", "b200vs_set_coalescing", "b200vs_reconstruct", "b200vs_sub_type",
    "b200vs_shard_unique_id", "b200vs_shard_create", "b200vs_shard_destroy", "b200vs_shard_list_range", "b200vs_shard_train",
    "b200vs_shard_broadcast_state", "b200vs_shard_add", "b200vs_shard_add_device", "b200vs_shard_remove_ids", "b200vs_shard_plan_add_device",
    "b200vs_shard_plan_commit", "b200vs_shard_search", "b200vs_shard_search_device",
    "b200vs_train_binary", "b200vs_add_binary_with_ids", "b200vs_search_binary", "b200vs_search_binary_device",
    "b200vs_range_search_binary", "b200vs_calc_distance_binary",
]


class Params(ctypes.Structure):
    _fields_ = [("nlist", ctypes.c_int32), ("pq_m", ctypes.c_int32), ("pq_nbits", ctypes.c_int32),
                ("hnsw_m", ctypes.c_int32), ("hnsw_efc", ctypes.c_int32), ("max_elements", ctypes.c_int64),
                ("device", ctypes.c_int32), ("hnsw_build_threads", ctypes.c_int32)]


class SearchParams(ctypes.Structure):
    _fields_ = [("nprobe", ctypes.c_int32), ("efsearch", ctypes.c_int32), ("has_range", ctypes.c_int32),
                ("negate", ctypes.c_int32), ("range_min", ctypes.c_int64), ("range_max", ctypes.c_int64),
                ("sorted_ids", ctypes.c_void_p), ("n_ids", ctypes.c_int64), ("exact_only", ctypes.c_int32),
                ("reserved", ctypes.c_int32)]


class B200VSError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"b200vs status {code}: {msg}")
        self.code = code
        self.msg = msg


_lib = None


def lib():
    """Load libb200vs.so; raise (never fall back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not built — run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float
    L.b200vs_create.argtypes = [ctypes.c_int, ctypes.c_int, i32, ctypes.POINTER(Params), ctypes.POINTER(vp)]
    L.b200vs_destroy.argtypes = [vp]
    L.b200vs_destroy.restype = None
    L.b200vs_train.argtypes = [vp, i64, vp]
    L.b200vs_set_trained_state.argtypes = [vp, vp, ctypes.c_size_t]
    L.b200vs_get_trained_state.argtypes = [vp, vp, ctypes.c_size_t]
    L.b200vs_get_trained_state.restype = i64
    L.b200vs_add_with_ids.argtypes = [vp, i64, vp, vp, ctypes.c_int]
    L.b200vs_remove_ids.argtypes = [vp, i64, vp, ctypes.POINTER(i64)]
    L.b200vs_search.argtypes = [vp, i64, vp, i32, ctypes.POINTER(SearchParams), vp, vp]
    L.b200vs_search_device.argtypes = [vp, i64, vp, i32, ctypes.POINTER(SearchParams), vp, vp, vp]
    L.b200vs_coarse_device.argtypes = [vp, i64, vp, i32, i32, i32, vp, vp, vp]
    L.b200vs_search_probes_device.argtypes = [vp, i64, vp, i32, vp, i32, ctypes.POINTER(SearchParams), vp, vp, vp]
    L.b200vs_range_search.argtypes = [vp, i64, vp, f32, i32, ctypes.POINTER(SearchParams), vp, vp, vp]
    L.b200vs_count.argtypes = [vp, ctypes.POINTER(i64)]
    L.b200vs_deleted_count.argtypes = [vp, ctypes.POINTER(i64)]
    L.b200vs_memory_size.argtypes = [vp, ctypes.POINTER(i64)]
    L.b200vs_is_trained.argtypes = [vp]
    L.b200vs_dimension.argtypes = [vp]
    L.b200vs_save.argtypes = [vp, ctypes.c_char_p]
    L.b200vs_load.argtypes = [vp, ctypes.c_char_p]
    L.b200vs_export_lists.argtypes = [vp, vp, vp, vp, vp]
    L.b200vs_merge_topk_device.argtypes = [i32, i32, i64, i32, vp, vp, vp, vp, vp]
    L.b200vs_last_search_stats.argtypes = [vp, ctypes.POINTER(i64 * 8)]
    L.b200vs_last_phase_times.argtypes = [vp, ctypes.POINTER(ctypes.c_float * 16)]
    L.b200vs_calc_distance.argtypes = [i32, i32, ctypes.c_int, i32, i64, vp, i64, vp, vp, vp, vp]
    L.b200vs_scan_begin.argtypes = [i32, ctypes.c_int, i32, i64, vp, i32, ctypes.POINTER(SearchParams), ctypes.POINTER(vp)]
    L.b200vs_scan_push.argtypes = [vp, i64, vp, vp]
    L.b200vs_scan_finish.argtypes = [vp, vp, vp]
    L.b200vs_scan_abort.argtypes = [vp]
    L.b200vs_scan_abort.restype = None
    L.b200vs_set_profiling.argtypes = [vp, ctypes.c_int]
    L.b200vs_last_error.restype = ctypes.c_char_p
    L.b200vs_version.restype = ctypes.c_char_p
    L.b200vs_add_with_ids_device.argtypes = [vp, i64, vp, vp, vp, ctypes.c_int]
    L.b200vs_assign_device.argtypes = [vp, i64, vp, vp]
    L.b200vs_reserve_lists.argtypes = [vp, vp, i32]
    L.b200vs_export_list.argtypes = [vp, i32, i64, vp, vp, ctypes.POINTER(i64)]
    L.b200vs_set_coalescing.argtypes = [vp, ctypes.c_int, ctypes.POINTER(i64 * 2)]
    L.b200vs_reconstruct.argtypes = [vp, i64, vp, vp, vp]
    L.b200vs_sub_type.argtypes = [vp]
    L.b200vs_shard_unique_id.argtypes = [vp]
    L.b200vs_shard_create.argtypes = [vp, i32, i32, vp, i32, ctypes.POINTER(vp)]
    L.b200vs_shard_destroy.argtypes = [vp]
    L.b200vs_shard_destroy.restype = None
    L.b200vs_shard_list_range.argtypes = [vp, i32, ctypes.POINTER(i32), ctypes.POINTER(i32)]
    L.b200vs_shard_train.argtypes = [vp, i64, vp]
    L.b200vs_shard_broadcast_state.argtypes = [vp, i32]
    L.b200vs_shard_add.argtypes = [vp, i64, vp, vp]
    L.b200vs_shard_add_device.argtypes = [vp, i64, vp, vp]
    L.b200vs_shard_remove_ids.argtypes = [vp, i64, vp, ctypes.POINTER(i64)]
    L.b200vs_shard_plan_add_device.argtypes = [vp, i64, vp]
    L.b200vs_shard_plan_commit.argtypes = [vp]
    L.b200vs_shard_search.argtypes = [vp, i64, i64, vp, i32, ctypes.POINTER(SearchParams), vp, vp]
    L.b200vs_shard_search_device.argtypes = [vp, i64, i64, vp, i32, ctypes.POINTER(SearchParams), vp, vp, vp]
    L.b200vs_train_binary.argtypes = [vp, i64, vp]
    L.b200vs_add_binary_with_ids.argtypes = [vp, i64, vp, vp, ctypes.c_int]
    L.b200vs_search_binary.argtypes = [vp, i64, vp, i32, ctypes.POINTER(SearchParams), vp, vp]
    L.b200vs_search_binary_device.argtypes = [vp, i64, vp, i32, ctypes.POINTER(SearchParams), vp, vp, vp]
    L.b200vs_range_search_binary.argtypes = [vp, i64, vp, f32, i32, ctypes.POINTER(SearchParams), vp, vp, vp]
    L.b200vs_calc_distance_binary.argtypes = [i32, i32, i64, vp, i64, vp, vp]
    _lib = L
    return L


def _check(rc):
    if rc != OK:
        raise B200VSError(rc, lib().b200vs_last_error().decode("utf-8", "replace"))


def _f32(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def make_search_params(nprobe=0, efsearch=0, id_range=None, sorted_ids=None, negate=False, exact_only=False):
    sp = SearchParams()
    sp.nprobe, sp.efsearch, sp.exact_only = int(nprobe), int(efsearch), int(bool(exact_only))
    keep = None
    if id_range is not None:
        sp.has_range, sp.range_min, sp.range_max = 1, int(id_range[0]), int(id_range[1])
    if sorted_ids is not None:
        keep = _i64(sorted_ids)
        sp.sorted_ids = keep.ctypes.data
        sp.n_ids = keep.size
        sp.negate = int(bool(negate))
    return sp, keep


class Index:
    """Thin owner of a b200vs_index handle.  Method names follow the reference plugin virtuals
    (src/vector/vector_index.h:148-202): train / add / upsert / delete / search / range_search / get_count ..."""

    def __init__(self, index_type, metric, dim, nlist=0, pq_m=0, pq_nbits=0, hnsw_m=0, hnsw_efc=0, max_elements=0,
                 device=0, hnsw_build_threads=0):
        self.L = lib()
        self.dim, self.type, self.metric = int(dim), int(index_type), int(metric)
        p = Params(nlist, pq_m, pq_nbits, hnsw_m, hnsw_efc, max_elements, device, hnsw_build_threads)
        self.params = p
        h = ctypes.c_void_p()
        _check(self.L.b200vs_create(index_type, metric, dim, ctypes.byref(p), ctypes.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.b200vs_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def binary(self):
        """BINARY_FLAT / BINARY_IVF_FLAT: dim is in bits, rows are uint8 [n, dim // 8]."""
        return self.type in BINARY_TYPES

    def _rows(self, x):
        """(contiguous rows, row count) in the index's value type."""
        if self.binary:
            x = _u8(x)
            return x, (x.shape[0] if x.ndim == 2 else x.size // (self.dim // 8))
        x = _f32(x)
        return x, (x.shape[0] if x.ndim == 2 else x.size // self.dim)

    # ---- write path ----
    def train(self, x):
        if self.binary:
            x, n = self._rows(x)
            _check(self.L.b200vs_train_binary(self.h, n, x.ctypes.data if x.size else None))
            return
        x = _f32(x)
        n = x.shape[0] if x.ndim == 2 else x.size // self.dim
        _check(self.L.b200vs_train(self.h, n, x.ctypes.data))

    def set_trained_state(self, blob):
        blob = np.ascontiguousarray(np.frombuffer(bytes(blob), dtype=np.uint8)) if not isinstance(blob, np.ndarray) else np.ascontiguousarray(blob.view(np.uint8))
        _check(self.L.b200vs_set_trained_state(self.h, blob.ctypes.data, blob.nbytes))

    def get_trained_state(self):
        need = self.L.b200vs_get_trained_state(self.h, None, 0)
        if need < 0:
            _check(-need)
        buf = np.zeros(max(int(need), 1), dtype=np.uint8)
        got = self.L.b200vs_get_trained_state(self.h, buf.ctypes.data, buf.nbytes)
        if got < 0:
            _check(-got)
        return buf[:got]

    def add(self, x, ids, upsert=False):
        if self.binary:
            x, ids = _u8(x), _i64(ids)
            _check(self.L.b200vs_add_binary_with_ids(self.h, ids.size, x.ctypes.data if x.size else None, ids.ctypes.data if ids.size else None, int(upsert)))
            return
        x, ids = _f32(x), _i64(ids)
        _check(self.L.b200vs_add_with_ids(self.h, ids.size, x.ctypes.data if x.size else None, ids.ctypes.data if ids.size else None, int(upsert)))

    def upsert(self, x, ids):
        self.add(x, ids, upsert=True)

    def add_device(self, n, x_dev_ptr, ids_dev_ptr, lists_dev_ptr=None, upsert=False):
        _check(self.L.b200vs_add_with_ids_device(self.h, n, x_dev_ptr, ids_dev_ptr, lists_dev_ptr, int(upsert)))

    def assign_device(self, n, x_dev_ptr, out_lists_dev_ptr):
        _check(self.L.b200vs_assign_device(self.h, n, x_dev_ptr, out_lists_dev_ptr))

    def reserve_lists(self, rows_per_list):
        r = _i64(rows_per_list)
        _check(self.L.b200vs_reserve_lists(self.h, r.ctypes.data, r.size))

    def delete(self, ids):
        ids = _i64(ids)
        n = ctypes.c_int64(0)
        _check(self.L.b200vs_remove_ids(self.h, ids.size, ids.ctypes.data if ids.size else None, ctypes.byref(n)))
        return n.value

    # ---- read path ----
    def search(self, xq, k, **kw):
        xq, nq = self._rows(xq)
        sp, keep = make_search_params(**kw)
        D = np.zeros((nq, max(k, 0)), dtype=np.float32)
        I = np.full((nq, max(k, 0)), -1, dtype=np.int64)
        fn = self.L.b200vs_search_binary if self.binary else self.L.b200vs_search
        _check(fn(self.h, nq, xq.ctypes.data if xq.size else None, k, ctypes.byref(sp), D.ctypes.data, I.ctypes.data))
        return D, I

    def search_raw(self, nq, xq_ptr, k, out_dist_ptr, out_ids_ptr, sp=None):
        """Host-pointer call with caller-owned (e.g. pinned) buffers — the e2e benchmark leg."""
        _check(self.L.b200vs_search(self.h, nq, xq_ptr, k, ctypes.byref(sp) if sp is not None else None, out_dist_ptr, out_ids_ptr))

    def search_device(self, nq, xq_dev_ptr, k, out_dist_dev_ptr, out_ids_dev_ptr, stream=None, sp=None):
        fn = self.L.b200vs_search_binary_device if self.binary else self.L.b200vs_search_device
        _check(fn(self.h, nq, xq_dev_ptr, k, ctypes.byref(sp) if sp is not None else None,
                                           out_dist_dev_ptr, out_ids_dev_ptr, stream))

    def coarse_device(self, nq, xq_dev_ptr, nprobe, list_begin, list_end, out_score_dev_ptr, out_lists_dev_ptr, stream=None):
        _check(self.L.b200vs_coarse_device(self.h, nq, xq_dev_ptr, nprobe, list_begin, list_end, out_score_dev_ptr, out_lists_dev_ptr, stream))

    def search_probes_device(self, nq, xq_dev_ptr, k, probes_dev_ptr, nprobe, out_dist_dev_ptr, out_ids_dev_ptr, stream=None, sp=None):
        _check(self.L.b200vs_search_probes_device(self.h, nq, xq_dev_ptr, k, probes_dev_ptr, nprobe, ctypes.byref(sp) if sp is not None else None,
                                                  out_dist_dev_ptr, out_ids_dev_ptr, stream))

    def range_search(self, xq, radius, max_results=1024, **kw):
        xq, nq = self._rows(xq)
        sp, keep = make_search_params(**kw)
        D = np.zeros((nq, max_results), dtype=np.float32)
        I = np.full((nq, max_results), -1, dtype=np.int64)
        C = np.zeros(nq, dtype=np.int32)
        fn = self.L.b200vs_range_search_binary if self.binary else self.L.b200vs_range_search
        _check(fn(self.h, nq, xq.ctypes.data if xq.size else None, float(radius), max_results,
                                          ctypes.byref(sp), D.ctypes.data, I.ctypes.data, C.ctypes.data))
        return D, I, C

    # ---- introspection ----
    def get_count(self):
        n = ctypes.c_int64(0)
        _check(self.L.b200vs_count(self.h, ctypes.byref(n)))
        return n.value

    def get_deleted_count(self):
        n = ctypes.c_int64(0)
        _check(self.L.b200vs_deleted_count(self.h, ctypes.byref(n)))
        return n.value

    def get_memory_size(self):
        n = ctypes.c_int64(0)
        _check(self.L.b200vs_memory_size(self.h, ctypes.byref(n)))
        return n.value

    def is_trained(self):
        return bool(self.L.b200vs_is_trained(self.h))

    def stats(self):
        a = (ctypes.c_int64 * 8)()
        _check(self.L.b200vs_last_search_stats(self.h, ctypes.byref(a)))
        return list(a)

    PHASES = ("coarse_prep", "coarse_scan", "coarse_final", "plan", "sample", "tau", "capture", "final", "fallback", "other", "comm", "merge")

    def phase_times(self):
        """{phase: device ms} of the last search (profiling mode only)."""
        a = (ctypes.c_float * 16)()
        _check(self.L.b200vs_last_phase_times(self.h, ctypes.byref(a)))
        return {n: float(a[i]) for i, n in enumerate(self.PHASES)}

    def set_profiling(self, on):
        _check(self.L.b200vs_set_profiling(self.h, int(bool(on))))

    def export_lists(self, nlist, with_vectors=True, code_size=0):
        """(list_off, vectors, codes, ids).  Binary indexes return their rows as codes [n, dim // 8] (vectors None)."""
        if self.binary:
            with_vectors, code_size = False, self.dim // 8
        n = self.get_count()
        off = np.zeros(nlist + 1, dtype=np.int64)
        vec = np.zeros((n, self.dim), dtype=np.float32) if with_vectors else None
        codes = np.zeros((n, code_size), dtype=np.uint8) if code_size else None
        ids = np.zeros(n, dtype=np.int64)
        _check(self.L.b200vs_export_lists(self.h, off.ctypes.data, vec.ctypes.data if vec is not None and vec.size else None,
                                          codes.ctypes.data if codes is not None and codes.size else None,
                                          ids.ctypes.data if ids.size else None))
        return off, vec, codes, ids

    def reconstruct(self, ids):
        ids = _i64(ids)
        out = np.zeros((ids.size, self.dim), dtype=np.float32)
        found = np.zeros(ids.size, dtype=np.uint8)
        _check(self.L.b200vs_reconstruct(self.h, ids.size, ids.ctypes.data, out.ctypes.data, found.ctypes.data))
        return out, found.astype(bool)

    def sub_type(self):
        return int(self.L.b200vs_sub_type(self.h))

    def coalescing(self, on=-1):
        """Switch (1 / 0) or just read (-1) request coalescing; returns (batches run, requests served)."""
        a = (ctypes.c_int64 * 2)()
        _check(self.L.b200vs_set_coalescing(self.h, on, ctypes.byref(a)))
        return int(a[0]), int(a[1])

    def export_list(self, list_id):
        """(vectors [n, dim], ids [n]) of one inverted list (live rows, stored order)."""
        n = ctypes.c_int64(0)
        _check(self.L.b200vs_export_list(self.h, list_id, 0, None, None, ctypes.byref(n)))
        vec = np.zeros((n.value, self.dim), dtype=np.float32)
        ids = np.zeros(n.value, dtype=np.int64)
        if n.value:
            _check(self.L.b200vs_export_list(self.h, list_id, n.value, vec.ctypes.data, ids.ctypes.data, ctypes.byref(n)))
        return vec, ids

    def save(self, path):
        _check(self.L.b200vs_save(self.h, path.encode()))

    def load(self, path):
        _check(self.L.b200vs_load(self.h, path.encode()))


class Shard:
    """One rank of a list-sharded IVF_FLAT index (b200vs_shard_*).  `id_bytes`: the 128-byte rendezvous blob made by
    Shard.unique_id() on rank 0 and distributed by the host (tests: torch.distributed broadcast)."""

    @staticmethod
    def unique_id():
        buf = np.zeros(128, dtype=np.uint8)
        _check(lib().b200vs_shard_unique_id(buf.ctypes.data))
        return buf

    def __init__(self, index, rank, world, id_bytes=None, lanes=2):
        self.ix, self.rank, self.world = index, int(rank), int(world)
        self.h = ctypes.c_void_p()
        idb = np.ascontiguousarray(id_bytes, dtype=np.uint8) if id_bytes is not None else None
        _check(lib().b200vs_shard_create(index.h, rank, world, idb.ctypes.data if idb is not None else None, lanes, ctypes.byref(self.h)))

    def close(self):
        if getattr(self, "h", None):
            lib().b200vs_shard_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def list_range(self, rank=None):
        b, e = ctypes.c_int32(0), ctypes.c_int32(0)
        _check(lib().b200vs_shard_list_range(self.h, self.rank if rank is None else rank, ctypes.byref(b), ctypes.byref(e)))
        return b.value, e.value

    def train(self, x):
        x = _f32(x)
        _check(lib().b200vs_shard_train(self.h, x.shape[0], x.ctypes.data))

    def broadcast_state(self, root=0):
        _check(lib().b200vs_shard_broadcast_state(self.h, root))

    def add(self, x, ids):
        x, ids = _f32(x), _i64(ids)
        _check(lib().b200vs_shard_add(self.h, ids.size, x.ctypes.data if x.size else None, ids.ctypes.data if ids.size else None))

    def add_device(self, n, x_dev_ptr, ids_dev_ptr):
        _check(lib().b200vs_shard_add_device(self.h, n, x_dev_ptr, ids_dev_ptr))

    def delete(self, ids):
        """Collective delete: every rank passes the same ids; returns the rows removed over all ranks."""
        ids = _i64(ids)
        n = ctypes.c_int64(0)
        _check(lib().b200vs_shard_remove_ids(self.h, ids.size, ids.ctypes.data if ids.size else None, ctypes.byref(n)))
        return n.value

    def plan_add_device(self, n, x_dev_ptr):
        _check(lib().b200vs_shard_plan_add_device(self.h, n, x_dev_ptr))

    def plan_commit(self):
        _check(lib().b200vs_shard_plan_commit(self.h))

    def search(self, xq, k, seq=-1, **kw):
        xq = _f32(xq)
        nq = xq.shape[0]
        sp, keep = make_search_params(**kw)
        D = np.zeros((nq, k), dtype=np.float32)
        I = np.full((nq, k), -1, dtype=np.int64)
        _check(lib().b200vs_shard_search(self.h, seq, nq, xq.ctypes.data, k, ctypes.byref(sp), D.ctypes.data, I.ctypes.data))
        return D, I

    def search_raw(self, nq, xq_ptr, k, out_dist_ptr, out_ids_ptr, sp=None, seq=-1):
        _check(lib().b200vs_shard_search(self.h, seq, nq, xq_ptr, k, ctypes.byref(sp) if sp is not None else None, out_dist_ptr, out_ids_ptr))

    def search_device(self, nq, xq_dev_ptr, k, out_dist_dev_ptr, out_ids_dev_ptr, stream=None, sp=None, seq=-1):
        _check(lib().b200vs_shard_search_device(self.h, seq, nq, xq_dev_ptr, k, ctypes.byref(sp) if sp is not None else None,
                                                out_dist_dev_ptr, out_ids_dev_ptr, stream))


def ivf_state_blob(centroids, metric):
    """Trained-state blob of an IVF-Flat index (DESIGN.md §Trained-state blobs)."""
    c = _f32(centroids)
    hdr = np.array([0x43465649, c.shape[0], c.shape[1], metric], dtype=np.int64)
    return np.concatenate([hdr.view(np.uint8), c.reshape(-1).view(np.uint8)])


def binary_ivf_state_blob(centroids):
    """Trained-state blob of a BINARY_IVF_FLAT index: packed centroids uint8 [nlist, dim // 8] (DESIGN.md §5)."""
    c = _u8(centroids)
    hdr = np.array([0x46564942, c.shape[0], c.shape[1] * 8, HAMMING], dtype=np.int64)
    return np.concatenate([hdr.view(np.uint8), c.reshape(-1)])


def merge_topk_device(device, nparts, nq, k, parts_dist_ptr, parts_ids_ptr, out_dist_ptr, out_ids_ptr, stream=None):
    _check(lib().b200vs_merge_topk_device(device, nparts, nq, k, parts_dist_ptr, parts_ids_ptr, out_dist_ptr, out_ids_ptr, stream))


ALGORITHM_FAISS, ALGORITHM_HNSWLIB = 1, 2


def calc_distance(algorithm, metric, left, right, return_normalized=False, device=0):
    """Pairwise distance matrix [nl, nr] (VectorCalcDistance); optionally the (normalised) operands as well."""
    left, right = _f32(left), _f32(right)
    nl, nr = left.shape[0], right.shape[0]
    d = left.shape[1] if left.ndim == 2 else 0
    out = np.zeros((nl, nr), dtype=np.float32)
    lo = np.zeros_like(left) if return_normalized else None
    ro = np.zeros_like(right) if return_normalized else None
    _check(lib().b200vs_calc_distance(device, algorithm, metric, d, nl, left.ctypes.data if left.size else None, nr,
                                      right.ctypes.data if right.size else None, out.ctypes.data if out.size else None,
                                      lo.ctypes.data if lo is not None and lo.size else None, ro.ctypes.data if ro is not None and ro.size else None))
    return (out, lo, ro) if return_normalized else out


def calc_distance_binary(left, right, device=0):
    """Pairwise Hamming matrix [nl, nr] of packed rows uint8 [n, dim // 8] (VectorCalcDistance, METRIC_TYPE_HAMMING)."""
    left, right = _u8(left), _u8(right)
    nl, nr = left.shape[0], right.shape[0]
    out = np.zeros((nl, nr), dtype=np.float32)
    _check(lib().b200vs_calc_distance_binary(device, left.shape[1] * 8, nl, left.ctypes.data if left.size else None, nr,
                                             right.ctypes.data if right.size else None, out.ctypes.data if out.size else None))
    return out


class BruteForceScan:
    """Streaming brute-force top-k over tiles of vectors that are not in an index (VectorReader::BruteForceSearch)."""

    def __init__(self, metric, dim, xq, k, device=0, **kw):
        xq = _f32(xq)
        self.nq, self.k = xq.shape[0], k
        sp, self._keep = make_search_params(**kw)
        self.h = ctypes.c_void_p()
        _check(lib().b200vs_scan_begin(device, metric, dim, self.nq, xq.ctypes.data if xq.size else None, k, ctypes.byref(sp), ctypes.byref(self.h)))

    def push(self, x, ids):
        x, ids = _f32(x), _i64(ids)
        _check(lib().b200vs_scan_push(self.h, ids.size, x.ctypes.data if x.size else None, ids.ctypes.data if ids.size else None))

    def finish(self):
        D = np.zeros((self.nq, self.k), dtype=np.float32)
        I = np.full((self.nq, self.k), -1, dtype=np.int64)
        h, self.h = self.h, None
        _check(lib().b200vs_scan_finish(h, D.ctypes.data, I.ctypes.data))
        return D, I

    def __del__(self):
        if getattr(self, "h", None):
            lib().b200vs_scan_abort(self.h)
            self.h = None


def ivfpq_state_blob(centroids, codebooks, metric):
    """Trained-state blob of an IVF-PQ index: centroids [nlist, d] + codebooks [M, 256, d/M]."""
    c, cb = _f32(centroids), _f32(codebooks)
    hdr = np.array([0x51505649, c.shape[0], c.shape[1], metric, cb.shape[0], 8], dtype=np.int64)
    return np.concatenate([hdr.view(np.uint8), c.reshape(-1).view(np.uint8), cb.reshape(-1).view(np.uint8)])
