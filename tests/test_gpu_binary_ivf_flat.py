"""BINARY_IVF_FLAT on the GPU against the CPU binary oracle on a shared trained state: probes chosen by the
(distance, list id) rule (forced centroid ties included), list assignment, range search, delete / upsert, GPU training
vs oracle training, Save / Load and the untrained contract."""
import numpy as np
import pytest

import b200vs
import oracle_binary_lib
from gpu_util import assert_same_results, recall, require_gpu

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bo():
    return oracle_binary_lib.load()


def build(bo, dim, nlist, xb, ids, cent):
    ix = b200vs.Index(b200vs.BINARY_IVF_FLAT, b200vs.HAMMING, dim, nlist=nlist)
    ix.set_trained_state(b200vs.binary_ivf_state_blob(cent))
    assert ix.is_trained()
    ix.add(xb, ids)
    off, _, codes, lids = ix.export_lists(nlist)
    return ix, off, codes, lids


def clustered(rng, n, nbytes, nclusters, flip=0.08):
    centers = rng.integers(0, 256, (nclusters, nbytes), dtype=np.uint8)
    x = centers[rng.integers(0, nclusters, n)]
    noise = np.packbits(rng.random((n, nbytes * 8)) < flip, axis=1, bitorder="little")
    return x ^ noise


@pytest.mark.parametrize("dim", [8, 24, 64, 256, 1024, 4096])
@pytest.mark.parametrize("k", [1, 10, 100, 1024])
def test_ivf_parity_shared_state(bo, dim, k):
    require_gpu()
    rng = np.random.default_rng(dim + k)
    n, nlist = 8000, 32
    xb = clustered(rng, n, dim // 8, 64)
    xb[::5] = xb[1::5]  # duplicated rows
    ids = rng.permutation(n).astype(np.int64) + 7
    cent = bo.kmeans(xb, nlist)
    ix, off, codes, lids = build(bo, dim, nlist, xb, ids, cent)
    assign = bo.assign(xb, cent)
    assert np.array_equal(np.diff(off), np.bincount(assign, minlength=nlist))  # adds go to the (distance, list id) nearest list
    for nq in (1, 300):
        xq = clustered(rng, nq, dim // 8, 64)
        for nprobe in (1, 4, nlist):
            D, I = ix.search(xq, k, nprobe=nprobe)
            Do, Io = bo.ivf_search(cent, off, codes, lids, xq, k, nprobe)
            assert_same_results(D, I, Do, Io)


def test_forced_centroid_ties_probe_the_same_lists(bo):
    require_gpu()
    rng = np.random.default_rng(21)
    dim, nlist, n = 32, 16, 6000
    cent = rng.integers(0, 256, (nlist, dim // 8), dtype=np.uint8)
    cent[3] = cent[2] ^ np.array([1, 0, 0, 0], np.uint8)
    cent[8:] = cent[:8]  # every centroid has a twin: equal distances everywhere, only the list id decides
    xb = rng.integers(0, 256, (n, dim // 8), dtype=np.uint8)
    ids = np.arange(n, dtype=np.int64)[::-1].copy()
    ix, off, codes, lids = build(bo, dim, nlist, xb, ids, cent)
    assert (np.diff(off)[8:] == 0).all()  # the higher twin never receives a row
    xq = np.concatenate([cent[:4], rng.integers(0, 256, (60, dim // 8), dtype=np.uint8)])
    for nprobe in (1, 2, 3, 5, 9):
        D, I = ix.search(xq, 50, nprobe=nprobe)
        Do, Io = bo.ivf_search(cent, off, codes, lids, xq, 50, nprobe)
        assert_same_results(D, I, Do, Io)


def test_ivf_filters_delete_upsert_range(bo):
    require_gpu()
    rng = np.random.default_rng(22)
    dim, nlist, n = 128, 24, 10000
    xb = clustered(rng, n, dim // 8, 40)
    ids = np.arange(n, dtype=np.int64)
    cent = bo.kmeans(xb, nlist)
    ix, _, _, _ = build(bo, dim, nlist, xb, ids, cent)
    assert ix.delete(ids[:6000]) == 6000
    assert pytest.raises(b200vs.B200VSError, ix.delete, np.array([10 ** 9])).value.code == b200vs.EVECTOR_INVALID
    ix.upsert(xb[6000:6500] ^ np.uint8(1), ids[6000:6500])
    ix.add(xb[:300], ids[:300])
    off, _, codes, lids = ix.export_lists(nlist)
    assert ix.get_count() == 4300
    xq = clustered(rng, 80, dim // 8, 40)
    allow = np.sort(rng.choice(ids, 2000, replace=False))
    for kw in ({}, dict(id_range=(100, 8000)), dict(sorted_ids=allow), dict(sorted_ids=allow, negate=True)):
        D, I = ix.search(xq, 25, nprobe=6, **kw)
        Do, Io = bo.ivf_search(cent, off, codes, lids, xq, 25, 6, **kw)
        assert_same_results(D, I, Do, Io)
    for radius in (5.5, 10.1, 30.0):
        D, I, C = ix.range_search(xq, radius, max_results=256, nprobe=5)
        Do, Io, Co = bo.ivf_range_search(cent, off, codes, lids, xq, radius, 256, 5)
        assert np.array_equal(C, Co)
        assert_same_results(D, I, Do, Io)


def test_gpu_training_matches_oracle_training(bo):
    require_gpu()
    rng = np.random.default_rng(23)
    dim, nlist = 256, 64
    xb = clustered(rng, 40000, dim // 8, 100)  # > nlist * 256: the training subsample is exercised
    ix = b200vs.Index(b200vs.BINARY_IVF_FLAT, b200vs.HAMMING, dim, nlist=nlist)
    ix.train(xb)
    assert ix.is_trained()
    blob = ix.get_trained_state()
    hdr = blob[:32].view(np.int64)
    assert hdr[0] == 0x46564942 and hdr[1] == nlist and hdr[2] == dim and hdr[3] == b200vs.HAMMING
    cg = blob[32:].reshape(nlist, dim // 8)
    co = bo.kmeans(xb, nlist)
    # +-1 sums are exact integers and the assignment scan is the reference-order exact L2, so the two agree bit for bit
    same = (cg == co).all(axis=1).mean()
    assert same == 1.0, f"{same:.3f} of the centroids agree"
    ix.add(xb, np.arange(len(xb)))
    xq = xb[:200]
    D, I = ix.search(xq, 10, nprobe=8)
    Df, If = bo.flat_search(xb, np.arange(len(xb)), xq, 10)
    assert recall(I, If) > 0.8


def test_untrained_and_degenerate_nlist(bo, tmp_path):
    require_gpu()
    rng = np.random.default_rng(24)
    dim = 64
    ix = b200vs.Index(b200vs.BINARY_IVF_FLAT, b200vs.HAMMING, dim)  # nlist defaults to 2048
    assert not ix.is_trained()
    x = rng.integers(0, 256, (500, dim // 8), dtype=np.uint8)
    D, I = ix.search(x[:3], 5)  # untrained search -> OK + empty results
    assert (I == -1).all() and (D == 0).all()
    assert pytest.raises(b200vs.B200VSError, ix.add, x, np.arange(500)).value.code == b200vs.EVECTOR_NOT_TRAIN
    assert ix.delete(np.arange(3)) == 0  # untrained delete -> OK
    ix.train(x)  # 500 rows < nlist 2048 -> nlist degenerates to 1
    assert ix.get_trained_state()[8:16].view(np.int64)[0] == 1
    ix.train(x[:10])  # already trained: no-op
    ix.add(x, np.arange(500))
    D, I = ix.search(x[:20], 7)  # default nprobe 80, clamped to nlist
    Do, Io = bo.flat_search(x, np.arange(500), x[:20], 7)
    assert_same_results(D, I, Do, Io)
    # Save / Load round trip: byte-identical files, identical results
    p1, p2 = str(tmp_path / "a.idx"), str(tmp_path / "b.idx")
    ix.save(p1)
    iy = b200vs.Index(b200vs.BINARY_IVF_FLAT, b200vs.HAMMING, dim)
    iy.load(p1)
    iy.save(p2)
    assert open(p1, "rb").read() == open(p2, "rb").read()
    D2, I2 = iy.search(x[:20], 7)
    assert_same_results(D2, I2, D, I)
    fl = b200vs.Index(b200vs.IVF_FLAT, b200vs.L2, dim, nlist=4)
    pf = str(tmp_path / "f.idx")
    fl.save(pf)
    iz = b200vs.Index(b200vs.BINARY_IVF_FLAT, b200vs.HAMMING, dim)
    assert pytest.raises(b200vs.B200VSError, iz.load, pf).value.code == b200vs.EINTERNAL
    # IVF-only building blocks are not offered on a binary index
    # (real device buffers: the calls are rejected before they touch them, and must stay harmless if that order changes)
    import torch
    L = b200vs.lib()
    q = torch.zeros((1, dim), dtype=torch.float32, device="cuda")
    score = torch.zeros((1, 1), dtype=torch.float32, device="cuda")
    lists = torch.zeros((1, 1), dtype=torch.int64, device="cuda")
    assert L.b200vs_coarse_device(iy.h, 1, q.data_ptr(), 1, 0, 1, score.data_ptr(), lists.data_ptr(), None) == b200vs.EVECTOR_NOT_SUPPORT
    assert L.b200vs_search_probes_device(iy.h, 1, q.data_ptr(), 1, lists.data_ptr(), 1, None, score.data_ptr(), lists.data_ptr(),
                                         None) == b200vs.EVECTOR_NOT_SUPPORT
    assert L.b200vs_assign_device(iy.h, 1, q.data_ptr(), lists.data_ptr()) == b200vs.EVECTOR_NOT_SUPPORT
    torch.cuda.synchronize()
    bad = b200vs.binary_ivf_state_blob(np.zeros((2, dim // 8), np.uint8))
    bad[24:32] = np.array([b200vs.L2], np.int64).view(np.uint8)  # 'BIVF' magic with a non-HAMMING metric
    assert pytest.raises(b200vs.B200VSError, iz.set_trained_state, bad).value.code == b200vs.EILLEGAL_PARAMETERS
    assert pytest.raises(b200vs.B200VSError, b200vs.Shard, iy, 0, 1, None).value.code == b200vs.EVECTOR_NOT_SUPPORT
