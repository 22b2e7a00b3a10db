"""ctypes access to the CPU oracle of the binary (Hamming) indexes (tests/native/_build/liboracle_binary.so).
TEST INFRASTRUCTURE: imported only from tests/, __graft_entry__.smoke() and bench_binary.py."""
import ctypes
import os

import numpy as np

import oracle_lib

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "native", "_build", "liboracle_binary.so")


def _u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


class BinaryOracle:
    def __init__(self, path=SO):
        L = ctypes.CDLL(path)
        vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float
        fp, c_int = ctypes.POINTER(oracle_lib.Filter), ctypes.c_int
        L.oracle_hamming.argtypes = [vp, vp, i32]
        L.oracle_hamming.restype = i32
        L.oracle_binary_flat_search.argtypes = [i32, i64, vp, vp, i64, vp, i32, fp, c_int, vp, vp]
        L.oracle_binary_flat_range_search.argtypes = [i32, i64, vp, vp, i64, vp, f32, i32, fp, c_int, vp, vp, vp]
        L.oracle_binary_to_real.argtypes = [i64, i32, vp, vp]
        L.oracle_binary_to_real.restype = None
        L.oracle_real_to_binary.argtypes = [i64, i32, vp, vp]
        L.oracle_real_to_binary.restype = None
        L.oracle_binary_kmeans.argtypes = [i32, i64, vp, i32, i32, i32, i64, c_int, vp]
        L.oracle_binary_assign.argtypes = [i32, i64, vp, i32, vp, c_int, vp]
        L.oracle_binary_ivf_search.argtypes = [i32, i32, vp, vp, vp, vp, i64, vp, i32, i32, fp, c_int, vp, vp]
        L.oracle_binary_ivf_range_search.argtypes = [i32, i32, vp, vp, vp, vp, i64, vp, f32, i32, i32, fp, c_int, vp, vp, vp]
        L.oracle_calc_distance_hamming.argtypes = [i32, i64, vp, i64, vp, vp]
        self.L = L

    @staticmethod
    def _ptr(a):
        return a.ctypes.data if a.size else None

    def hamming(self, a, b):
        a, b = _u8(a), _u8(b)
        return int(self.L.oracle_hamming(a.ctypes.data, b.ctypes.data, a.size * 8))

    def flat_search(self, xb, ids, xq, k, nthreads=8, **filt):
        xb, ids, xq = _u8(xb), _i64(ids), _u8(xq)
        nq, dim = xq.shape[0], xq.shape[1] * 8
        D = np.zeros((nq, k), np.float32)
        I = np.full((nq, k), -1, np.int64)
        f, keep = oracle_lib.Oracle._filter(**filt)
        rc = self.L.oracle_binary_flat_search(dim, ids.size, self._ptr(xb), self._ptr(ids), nq, xq.ctypes.data, k,
                                              ctypes.byref(f) if f else None, nthreads, D.ctypes.data, I.ctypes.data)
        assert rc == 0
        return D, I

    def flat_range_search(self, xb, ids, xq, radius, max_results, nthreads=8, **filt):
        xb, ids, xq = _u8(xb), _i64(ids), _u8(xq)
        nq, dim = xq.shape[0], xq.shape[1] * 8
        D = np.zeros((nq, max_results), np.float32)
        I = np.full((nq, max_results), -1, np.int64)
        C = np.zeros(nq, np.int32)
        f, keep = oracle_lib.Oracle._filter(**filt)
        rc = self.L.oracle_binary_flat_range_search(dim, ids.size, self._ptr(xb), self._ptr(ids), nq, xq.ctypes.data, float(radius),
                                                    max_results, ctypes.byref(f) if f else None, nthreads, D.ctypes.data,
                                                    I.ctypes.data, C.ctypes.data)
        assert rc == 0
        return D, I, C

    def binary_to_real(self, x):
        x = _u8(x)
        out = np.zeros((x.shape[0], x.shape[1] * 8), np.float32)
        self.L.oracle_binary_to_real(x.shape[0], x.shape[1] * 8, x.ctypes.data, out.ctypes.data)
        return out

    def real_to_binary(self, x):
        x = np.ascontiguousarray(x, dtype=np.float32)
        out = np.zeros((x.shape[0], x.shape[1] // 8), np.uint8)
        self.L.oracle_real_to_binary(x.shape[0], x.shape[1], x.ctypes.data, out.ctypes.data)
        return out

    def kmeans(self, x, k, niter=10, max_pts=256, seed=1234, nthreads=8):
        x = _u8(x)
        c = np.zeros((k, x.shape[1]), np.uint8)
        rc = self.L.oracle_binary_kmeans(x.shape[1] * 8, x.shape[0], x.ctypes.data, k, niter, max_pts, seed, nthreads, c.ctypes.data)
        assert rc == 0, rc
        return c

    def assign(self, x, centroids, nthreads=8):
        x, c = _u8(x), _u8(centroids)
        out = np.zeros(x.shape[0], np.int32)
        rc = self.L.oracle_binary_assign(x.shape[1] * 8, x.shape[0], x.ctypes.data, c.shape[0], c.ctypes.data, nthreads, out.ctypes.data)
        assert rc == 0
        return out

    def ivf_search(self, centroids, list_off, xb, ids, xq, k, nprobe, nthreads=8, **filt):
        c, off, xb, ids, xq = _u8(centroids), _i64(list_off), _u8(xb), _i64(ids), _u8(xq)
        nq, dim = xq.shape[0], xq.shape[1] * 8
        D = np.zeros((nq, k), np.float32)
        I = np.full((nq, k), -1, np.int64)
        f, keep = oracle_lib.Oracle._filter(**filt)
        rc = self.L.oracle_binary_ivf_search(dim, c.shape[0], c.ctypes.data, off.ctypes.data, self._ptr(xb), self._ptr(ids), nq,
                                             xq.ctypes.data, k, nprobe, ctypes.byref(f) if f else None, nthreads, D.ctypes.data,
                                             I.ctypes.data)
        assert rc == 0
        return D, I

    def ivf_range_search(self, centroids, list_off, xb, ids, xq, radius, max_results, nprobe, nthreads=8, **filt):
        c, off, xb, ids, xq = _u8(centroids), _i64(list_off), _u8(xb), _i64(ids), _u8(xq)
        nq, dim = xq.shape[0], xq.shape[1] * 8
        D = np.zeros((nq, max_results), np.float32)
        I = np.full((nq, max_results), -1, np.int64)
        C = np.zeros(nq, np.int32)
        f, keep = oracle_lib.Oracle._filter(**filt)
        rc = self.L.oracle_binary_ivf_range_search(dim, c.shape[0], c.ctypes.data, off.ctypes.data, self._ptr(xb), self._ptr(ids), nq,
                                                   xq.ctypes.data, float(radius), max_results, nprobe, ctypes.byref(f) if f else None,
                                                   nthreads, D.ctypes.data, I.ctypes.data, C.ctypes.data)
        assert rc == 0
        return D, I, C

    def calc_distance(self, left, right):
        left, right = _u8(left), _u8(right)
        out = np.zeros((left.shape[0], right.shape[0]), np.float32)
        rc = self.L.oracle_calc_distance_hamming(left.shape[1] * 8, left.shape[0], left.ctypes.data, right.shape[0], right.ctypes.data,
                                                 out.ctypes.data)
        assert rc == 0
        return out


def load():
    if not os.path.exists(SO):
        raise ImportError(f"{SO} not built — run __graft_entry__.build()")
    return BinaryOracle(SO)
