"""BINARY_FLAT on the GPU against the CPU binary oracle: ids and distances bit-equal under the (distance, id) rule, filters,
delete / upsert, range search at the truncated radius, Save / Load and the status codes of the binary contract."""
import os

import numpy as np
import pytest

import b200vs
import oracle_binary_lib
from gpu_util import assert_same_results, require_gpu

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bo():
    return oracle_binary_lib.load()


def rows_with_duplicates(rng, n, nbytes, distinct):
    """n rows drawn from `distinct` random rows plus fresh ones: many exact distance ties."""
    base = rng.integers(0, 256, (distinct, nbytes), dtype=np.uint8)
    x = rng.integers(0, 256, (n, nbytes), dtype=np.uint8)
    pick = rng.random(n) < 0.5
    x[pick] = base[rng.integers(0, distinct, pick.sum())]
    return x


@pytest.mark.parametrize("dim", [8, 24, 64, 256, 1024, 4096])
@pytest.mark.parametrize("k", [1, 10, 100, 1024])
def test_flat_parity(bo, dim, k):
    require_gpu()
    rng = np.random.default_rng(dim * 7 + k)
    n = 3000
    xb = rows_with_duplicates(rng, n, dim // 8, 40)
    ids = rng.permutation(n).astype(np.int64) * 5 + 3  # not in insertion order
    ix = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, dim)
    ix.add(xb, ids)
    assert ix.get_count() == n
    for nq in (1, 300):
        xq = rng.integers(0, 256, (nq, dim // 8), dtype=np.uint8)
        xq[: nq // 3] = xb[rng.integers(0, n, nq // 3)]  # exact hits
        D, I = ix.search(xq, k)
        Do, Io = bo.flat_search(xb, ids, xq, k)
        assert_same_results(D, I, Do, Io)


def test_flat_large_single_query_spreads_and_matches(bo):
    require_gpu()
    rng = np.random.default_rng(11)
    n, dim = 200000, 1024
    xb = rows_with_duplicates(rng, n, dim // 8, 500)
    ids = np.arange(n, dtype=np.int64)
    ix = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, dim)
    ix.add(xb, ids)
    xq = rng.integers(0, 256, (3, dim // 8), dtype=np.uint8)
    for q in range(3):
        D, I = ix.search(xq[q:q + 1], 10)
        Do, Io = bo.flat_search(xb, ids, xq[q:q + 1], 10)
        assert_same_results(D, I, Do, Io)


def test_flat_filters(bo):
    require_gpu()
    rng = np.random.default_rng(2)
    n, dim = 5000, 128
    xb = rows_with_duplicates(rng, n, dim // 8, 30)
    ids = np.arange(100, 100 + n, dtype=np.int64)
    ix = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, dim)
    ix.add(xb, ids)
    xq = rng.integers(0, 256, (64, dim // 8), dtype=np.uint8)
    allow = np.sort(rng.choice(ids, 700, replace=False))
    for kw in (dict(id_range=(1000, 3000)), dict(sorted_ids=allow), dict(sorted_ids=allow, negate=True)):
        D, I = ix.search(xq, 20, **kw)
        Do, Io = bo.flat_search(xb, ids, xq, 20, **kw)
        assert_same_results(D, I, Do, Io)


def test_flat_delete_upsert_then_search(bo):
    require_gpu()
    rng = np.random.default_rng(3)
    n, dim = 4000, 64
    xb = rows_with_duplicates(rng, n, dim // 8, 20)
    ids = np.arange(n, dtype=np.int64)
    ix = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, dim)
    ix.add(xb, ids)
    gone = rng.choice(n, 2500, replace=False)  # enough to trigger compaction
    assert ix.delete(np.concatenate([gone, [10 ** 9]])) == 2500  # unknown ids are ignored
    assert ix.get_count() == n - 2500
    new = rng.integers(0, 256, (300, dim // 8), dtype=np.uint8)
    up_ids = np.concatenate([gone[:150], np.setdiff1d(ids, gone)[:150]])
    ix.upsert(new, up_ids)
    ix.add(new[:50], up_ids[:50])  # Flat add replaces pre-existing ids too (flat.cc:121-162)
    live = dict(zip(np.setdiff1d(ids, gone).tolist(), xb[np.setdiff1d(ids, gone)]))
    for i, r in zip(up_ids, new):
        live[int(i)] = r
    for i, r in zip(up_ids[:50], new[:50]):
        live[int(i)] = r
    ref_ids = np.array(sorted(live), np.int64)
    ref_x = np.stack([live[i] for i in ref_ids])
    assert ix.get_count() == len(ref_ids)
    xq = rng.integers(0, 256, (50, dim // 8), dtype=np.uint8)
    D, I = ix.search(xq, 30)
    Do, Io = bo.flat_search(ref_x, ref_ids, xq, 30)
    assert_same_results(D, I, Do, Io)
    off, vec, codes, eids = ix.export_lists(1)
    assert vec is None and codes.shape == (len(ref_ids), dim // 8)
    got = dict(zip(eids.tolist(), codes))
    assert sorted(got) == ref_ids.tolist() and all(np.array_equal(got[i], live[i]) for i in got)


def test_flat_range_search_truncated_radius(bo):
    require_gpu()
    rng = np.random.default_rng(4)
    n, dim = 6000, 64
    xb = rows_with_duplicates(rng, n, dim // 8, 50)
    ids = np.arange(n, dtype=np.int64) * 2
    ix = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, dim)
    ix.add(xb, ids)
    xq = xb[rng.integers(0, n, 40)] ^ rng.integers(0, 2, (40, dim // 8), dtype=np.uint8)
    for radius in (0.0, 1.0, 10.1, 20.0, 26.9):
        D, I, C = ix.range_search(xq, radius, max_results=512)
        Do, Io, Co = bo.flat_range_search(xb, ids, xq, radius, 512)
        assert np.array_equal(C, Co), radius
        assert_same_results(D, I, Do, Io)
    D, I, C = ix.range_search(xq, 10.1, max_results=512, id_range=(0, 5000))
    Do, Io, Co = bo.flat_range_search(xb, ids, xq, 10.1, 512, id_range=(0, 5000))
    assert np.array_equal(C, Co)
    assert_same_results(D, I, Do, Io)


def test_flat_save_load_round_trip(bo, tmp_path):
    require_gpu()
    rng = np.random.default_rng(5)
    n, dim = 3000, 200
    xb = rows_with_duplicates(rng, n, dim // 8, 10)
    ids = rng.permutation(n).astype(np.int64)
    ix = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, dim)
    ix.add(xb, ids)
    ix.delete(ids[:100])
    p1, p2 = str(tmp_path / "a.idx"), str(tmp_path / "b.idx")
    ix.save(p1)
    iy = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, dim)
    iy.load(p1)
    assert iy.get_count() == n - 100
    iy.save(p2)
    assert open(p1, "rb").read() == open(p2, "rb").read()
    xq = rng.integers(0, 256, (20, dim // 8), dtype=np.uint8)
    D1, I1 = ix.search(xq, 50)
    D2, I2 = iy.search(xq, 50)
    assert_same_results(D2, I2, D1, I1)
    # a float index file is rejected by a binary index, and the other way round
    fl = b200vs.Index(b200vs.FLAT, b200vs.L2, dim)
    fl.add(rng.random((10, dim), dtype=np.float32), np.arange(10))
    pf = str(tmp_path / "f.idx")
    fl.save(pf)
    iz = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, dim)
    with pytest.raises(b200vs.B200VSError):
        iz.load(pf)
    fz = b200vs.Index(b200vs.FLAT, b200vs.L2, dim)
    with pytest.raises(b200vs.B200VSError):
        fz.load(p1)


def code_of(fn):
    with pytest.raises(b200vs.B200VSError) as e:
        fn()
    return e.value.code


def test_status_codes():
    require_gpu()
    L = b200vs.lib()
    # create: wrong metric for the type, bad binary dimension, HAMMING on a float type
    for t in b200vs.BINARY_TYPES:
        assert code_of(lambda: b200vs.Index(t, b200vs.L2, 64)) == b200vs.EILLEGAL_PARAMETERS
        assert code_of(lambda: b200vs.Index(t, b200vs.HAMMING, 12)) == b200vs.EILLEGAL_PARAMETERS
        assert code_of(lambda: b200vs.Index(t, b200vs.HAMMING, 32776)) == b200vs.EILLEGAL_PARAMETERS
    b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, 32768).close()
    assert code_of(lambda: b200vs.Index(b200vs.FLAT, b200vs.HAMMING, 64)) == b200vs.EILLEGAL_PARAMETERS
    ix = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, 64)
    x = np.arange(80, dtype=np.uint8).reshape(10, 8)
    ix.add(x, np.arange(10))
    # duplicate ids inside one batch
    assert code_of(lambda: ix.add(x[:2], np.array([5, 5]))) == b200vs.EVECTOR_ID_DUPLICATED
    # empty batch / topk 0
    assert code_of(lambda: ix.add(x[:0], np.arange(0))) == b200vs.EILLEGAL_PARAMETERS
    D, I = ix.search(x[:2], 0)
    assert D.shape == (2, 0)
    assert code_of(lambda: ix.search(x[:0], 5)) == b200vs.EILLEGAL_PARAMETERS
    assert ix.delete(np.arange(0)) == 0
    # float entry points on a binary index and binary ones on a float index: EVECTOR_INVALID
    f = np.zeros((2, 64), np.float32)
    ids2 = np.arange(2, dtype=np.int64)
    sp = b200vs.SearchParams()
    D2, I2 = np.zeros((2, 3), np.float32), np.zeros((2, 3), np.int64)
    C2 = np.zeros(2, np.int32)
    assert L.b200vs_add_with_ids(ix.h, 2, f.ctypes.data, ids2.ctypes.data, 0) == b200vs.EVECTOR_INVALID
    assert L.b200vs_search(ix.h, 2, f.ctypes.data, 3, None, D2.ctypes.data, I2.ctypes.data) == b200vs.EVECTOR_INVALID
    assert L.b200vs_range_search(ix.h, 2, f.ctypes.data, 1.0, 3, None, D2.ctypes.data, I2.ctypes.data, C2.ctypes.data) == b200vs.EVECTOR_INVALID
    assert L.b200vs_train(ix.h, 2, f.ctypes.data) == b200vs.EVECTOR_INVALID
    fl = b200vs.Index(b200vs.FLAT, b200vs.L2, 64)
    xb8 = np.zeros((2, 8), np.uint8)
    assert L.b200vs_add_binary_with_ids(fl.h, 2, xb8.ctypes.data, ids2.ctypes.data, 0) == b200vs.EVECTOR_INVALID
    assert L.b200vs_search_binary(fl.h, 2, xb8.ctypes.data, 3, None, D2.ctypes.data, I2.ctypes.data) == b200vs.EVECTOR_INVALID
    assert L.b200vs_range_search_binary(fl.h, 2, xb8.ctypes.data, 1.0, 3, None, D2.ctypes.data, I2.ctypes.data, C2.ctypes.data) == b200vs.EVECTOR_INVALID
    assert L.b200vs_train_binary(fl.h, 2, xb8.ctypes.data) == b200vs.EVECTOR_INVALID
    # not supported on binary indexes
    assert code_of(lambda: ix.reconstruct(np.arange(2))) == b200vs.EVECTOR_NOT_SUPPORT
    import torch  # real device buffers: rejected before use, harmless if that order ever changes
    xd = torch.zeros((2, 64), dtype=torch.float32, device="cuda")
    idd = torch.arange(2, dtype=torch.int64, device="cuda")
    assert L.b200vs_add_with_ids_device(ix.h, 2, xd.data_ptr(), idd.data_ptr(), None, 0) == b200vs.EVECTOR_NOT_SUPPORT
    torch.cuda.synchronize()
    assert L.b200vs_reserve_lists(ix.h, ids2.ctypes.data, 1) == b200vs.EVECTOR_NOT_SUPPORT
    assert code_of(lambda: b200vs.Shard(ix, 0, 1, None)) == b200vs.EVECTOR_NOT_SUPPORT
    # Flat: no trained state
    assert ix.is_trained() and ix.sub_type() == b200vs.BINARY_FLAT and len(ix.get_trained_state()) <= 1
    assert ix.get_memory_size() > 0 and ix.get_deleted_count() == 0
    # the float distance matrix still rejects HAMMING and metric 0
    for m in (0, b200vs.HAMMING):
        assert code_of(lambda: b200vs.calc_distance(b200vs.ALGORITHM_FAISS, m, f, f)) == b200vs.EILLEGAL_PARAMETERS


def test_search_binary_device_matches_host(bo):
    require_gpu()
    import torch
    rng = np.random.default_rng(6)
    n, dim, nq, k = 5000, 512, 128, 16
    xb = rows_with_duplicates(rng, n, dim // 8, 25)
    ids = np.arange(n, dtype=np.int64)
    ix = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, dim)
    ix.add(xb, ids)
    xq = rng.integers(0, 256, (nq, dim // 8), dtype=np.uint8)
    q = torch.from_numpy(xq).cuda()
    od = torch.zeros((nq, k), dtype=torch.float32, device="cuda")
    oi = torch.zeros((nq, k), dtype=torch.int64, device="cuda")
    ix.search_device(nq, q.data_ptr(), k, od.data_ptr(), oi.data_ptr())
    Do, Io = bo.flat_search(xb, ids, xq, k)
    assert_same_results(od.cpu().numpy(), oi.cpu().numpy(), Do, Io)
