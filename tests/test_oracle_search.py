"""Behavioural checks of the oracle's search restatements (the reference's unit tests assert contracts, not
numbers: SURVEY.md §4) plus cross-checks against float64 numpy brute force."""
import json
import os

import numpy as np
import pytest

import oracle_lib
from oracle_lib import COSINE, IP, L2


def brute(metric, xb, xq, k):
    xb64, xq64 = xb.astype(np.float64), xq.astype(np.float64)
    if metric == L2:
        d = ((xq64[:, None, :] - xb64[None, :, :]) ** 2).sum(-1)
    else:
        d = -(xq64 @ xb64.T)
    return np.argsort(d, axis=1, kind="stable")[:, :k]


@pytest.mark.parametrize("metric", [L2, IP, COSINE])
def test_flat_matches_float64_bruteforce(oracle, metric):
    rng = np.random.default_rng(3)
    xb = rng.random((500, 24)).astype(np.float32)
    xq = rng.random((7, 24)).astype(np.float32)
    ids = np.arange(1000, 1500, dtype=np.int64)
    stored = oracle.normalize_faiss(xb) if metric == COSINE else xb
    D, I = oracle.flat_search(metric, stored, ids, xq, 10)
    qn = oracle.normalize_faiss(xq) if metric == COSINE else xq
    want = ids[brute(L2 if metric == L2 else IP, stored, qn, 10)]
    assert (I == want).mean() > 0.98  # float32 vs float64 may swap near-ties
    assert np.all(np.diff(D, axis=1) >= 0)  # ascending in API semantics
    if metric != L2:  # 1 - ip
        ip = (qn.astype(np.float64) @ stored.astype(np.float64).T)
        assert np.allclose(D[:, 0], 1 - ip.max(1), atol=1e-5)


def test_flat_reference_fixture_contract(oracle):
    # reference Flat fixture: 10 x 8 (test_vector_index_flat.cc:44-47,:491-500); self query -> itself at rank 0
    xb = oracle.fixture(10, 8)
    ids = np.arange(1, 11, dtype=np.int64)
    D, I = oracle.flat_search(L2, xb, ids, xb[:3], 3)
    assert list(I[:, 0]) == [1, 2, 3] and np.all(D[:, 0] == 0)
    # fewer vectors than k -> padded with -1 (labels pre-filled -1, flat.cc:218-219)
    D, I = oracle.flat_search(L2, xb, ids, xb[:1], 20)
    assert (I[0, 10:] == -1).all() and (I[0, :10] >= 1).all()


def test_flat_filters_and_removed_slots(oracle):
    rng = np.random.default_rng(4)
    xb = rng.random((200, 16)).astype(np.float32)
    ids = np.arange(1, 201, dtype=np.int64)
    ids[10:20] = -1  # removed
    xq = rng.random((4, 16)).astype(np.float32)
    D, I = oracle.flat_search(L2, xb, ids, xq, 50, id_range=(50, 100))
    assert ((I >= 50) & (I < 100)).all()
    allow = np.array([3, 5, 77, 150], np.int64)
    D, I = oracle.flat_search(L2, xb, ids, xq, 10, sorted_ids=allow)
    assert set(I[0][I[0] >= 0]) == set(allow)
    D, I = oracle.flat_search(L2, xb, ids, xq, 200, sorted_ids=allow, negate=True)
    got = set(I[0][I[0] >= 0])
    assert not (got & set(allow)) and not (got & set(range(11, 21))) and len(got) == 200 - 10 - 4


def test_ties_break_by_id(oracle):
    xb = np.ones((6, 4), np.float32)
    ids = np.array([9, 3, 7, 1, 5, 2], np.int64)
    D, I = oracle.flat_search(L2, xb, ids, np.zeros((1, 4), np.float32), 4)
    assert list(I[0]) == [1, 2, 3, 5]


def make_ivf(oracle, metric, n=3000, d=16, nlist=20, seed=5):
    rng = np.random.default_rng(seed)
    xb = rng.random((n, d)).astype(np.float32)
    stored = oracle.normalize_faiss(xb) if metric == COSINE else xb
    cent = oracle.kmeans(metric, stored, nlist)
    asg = oracle.assign(metric, stored, cent)
    order = np.argsort(asg, kind="stable")
    off = np.zeros(nlist + 1, np.int64)
    off[1:] = np.cumsum(np.bincount(asg, minlength=nlist))
    ids = np.arange(1, n + 1, dtype=np.int64)
    return xb, stored, cent, off, stored[order], ids[order], ids


@pytest.mark.parametrize("metric", [L2, IP, COSINE])
def test_ivfflat_full_probe_equals_flat(oracle, metric):
    xb, stored, cent, off, lx, lids, ids = make_ivf(oracle, metric)
    xq = np.random.default_rng(6).random((9, 16)).astype(np.float32)
    Df, If = oracle.flat_search(metric, stored, ids, xq, 10)
    Di, Ii = oracle.ivfflat_search(metric, cent, off, lx, lids, xq, 10, nprobe=20)
    assert np.array_equal(If, Ii) and np.array_equal(Df, Di)
    # nprobe is clamped to nlist (ivf_flat.cc:234); <= 0 means the default 80 (constant.h:178)
    Dc, Ic = oracle.ivfflat_search(metric, cent, off, lx, lids, xq, 10, nprobe=500)
    Dd, Id = oracle.ivfflat_search(metric, cent, off, lx, lids, xq, 10, nprobe=0)
    assert np.array_equal(Ic, If) and np.array_equal(Id, If)


def test_ivfflat_partial_probe_recall_and_subset(oracle):
    xb, stored, cent, off, lx, lids, ids = make_ivf(oracle, L2)
    xq = np.random.default_rng(7).random((20, 16)).astype(np.float32)
    Df, If = oracle.flat_search(L2, stored, ids, xq, 10)
    Di, Ii = oracle.ivfflat_search(L2, cent, off, lx, lids, xq, 10, nprobe=5)
    recall = np.mean([len(set(a) & set(b)) / 10 for a, b in zip(If, Ii)])
    assert recall > 0.6
    assert np.all(np.diff(Di, axis=1) >= 0)


def test_kmeans_is_deterministic_and_reasonable(oracle):
    rng = np.random.default_rng(8)
    centers = rng.random((8, 6)).astype(np.float32) * 10
    x = (centers[rng.integers(0, 8, 4000)] + rng.standard_normal((4000, 6)) * 0.1).astype(np.float32)
    c1 = oracle.kmeans(L2, x, 8, nthreads=1)
    c2 = oracle.kmeans(L2, x, 8, nthreads=4)
    assert np.array_equal(c1, c2)
    asg = oracle.assign(L2, x, c1)
    err = ((x - c1[asg]) ** 2).sum(1).mean()
    assert err < 0.3 * x.var(0).sum()  # Lloyd from random points: a local optimum, far below the data variance


def test_ivfpq_search_sanity(oracle):
    rng = np.random.default_rng(9)
    n, d, nlist, M = 6000, 32, 16, 8
    xb = rng.standard_normal((n, d)).astype(np.float32)
    for metric in (L2, IP):
        cent = oracle.kmeans(metric, xb, nlist)
        asg = oracle.assign(metric, xb, cent)
        cb = oracle.pq_train(xb - cent[asg], M)
        codes = oracle.ivfpq_encode(cb, cent, xb, asg)
        order = np.argsort(asg, kind="stable")
        off = np.zeros(nlist + 1, np.int64)
        off[1:] = np.cumsum(np.bincount(asg, minlength=nlist))
        ids = np.arange(n, dtype=np.int64)
        xq = xb[:50] + 0.01 * rng.standard_normal((50, d)).astype(np.float32)
        D, I = oracle.ivfpq_search(metric, cent, cb, off, codes[order], ids[order], xq, 10, nprobe=nlist)
        Df, If = oracle.flat_search(metric, xb, ids, xq, 10)
        recall = np.mean([len(set(a) & set(b)) / 10 for a, b in zip(If, I)])
        assert recall > 0.35, (metric, recall)
        assert np.all(np.diff(D, axis=1) >= 0)
        # distances approximate the true ones (PQ reconstruction error only)
        recon = cent[asg] + np.stack([cb[m, codes[:, m]] for m in range(M)], 1).reshape(n, d)
        j = I[0, 0]
        true = ((xq[0] - recon[j]) ** 2).sum() if metric == L2 else 1 - xq[0] @ recon[j]
        assert abs(D[0, 0] - true) < 1e-3 * max(1, abs(true))


@pytest.mark.parametrize("metric", [L2, IP, COSINE])
def test_hnsw_recall_and_contract(oracle, metric):
    rng = np.random.default_rng(10)
    n, d = 2000, 16
    xb = rng.random((n, d)).astype(np.float32)
    labels = np.arange(100, 100 + n, dtype=np.int64)
    h = oracle_lib.OracleHnsw(oracle, metric, d, n, 16, 200)
    h.add(xb, labels)
    xq = rng.random((30, d)).astype(np.float32)
    D, I, nd, nh = h.search(xq, 10, ef=128)
    assert (I >= 100).all() and np.all(np.diff(D, axis=1) >= 0)  # exactly k hits, ascending (hnsw.cc:400-419)
    stored = oracle.normalize_hnsw(xb) if metric == COSINE else xb
    qn = oracle.normalize_hnsw(xq) if metric == COSINE else xq
    want = labels[brute(L2 if metric == L2 else IP, stored, qn, 10)]
    recall = np.mean([len(set(a) & set(b)) / 10 for a, b in zip(want, I)])
    assert recall > 0.9, recall
    assert (nd > 0).all() and (nh > 0).all()
    # filter: traversed but never returned
    D2, I2, _, _ = h.search(xq, 10, ef=128, id_range=(100, 600))
    assert ((I2 >= 100) & (I2 < 600) | (I2 == -1)).all()
    blob = h.export()
    hdr = blob[:64].view(np.int64)
    assert hdr[0] == 0x57534E48 and hdr[1] == n and hdr[2] == d


@pytest.mark.parametrize("algorithm", [1, 2])
def test_calc_distance_pinned_to_reference_kernels(oracle, algorithm):
    """oracle_calc_distance (vector_index_utils.cc:48-124): every entry is the hooked kernel's value — checked against
    what the reference's own src/simd objects returned on these inputs (tests/golden/simd_ref_samples.json) — and the
    two normalisers differ."""
    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "simd_ref_samples.json")))["calc_distance"]
    rng = np.random.default_rng(gold["seed"])
    left = rng.random(tuple(gold["left"]), dtype=np.float32)
    right = rng.random(tuple(gold["right"]), dtype=np.float32) * 2 - 0.5
    ref_l2 = np.array([[int(h, 16) for h in row] for row in gold["l2"]], np.uint32).view(np.float32)
    ref_ip = np.array([[int(h, 16) for h in row] for row in gold["ip"]], np.uint32).view(np.float32)
    d2, lo, ro = oracle.calc_distance(algorithm, oracle_lib.L2, left, right)
    ip, _, _ = oracle.calc_distance(algorithm, oracle_lib.IP, left, right)
    assert np.array_equal(lo, left) and np.array_equal(ro, right)
    assert d2.shape == ref_l2.shape == ip.shape == ref_ip.shape
    for i in range(5):
        for j in range(6):
            assert d2[i, j] == ref_l2[i, j]
            assert ip[i, j] == np.float32(1.0) - ref_ip[i, j]
            assert abs(d2[i, j] - float(((left[i].astype(np.float64) - right[j]) ** 2).sum())) < 1e-3
    cs, ln, rn = oracle.calc_distance(algorithm, oracle_lib.COSINE, left, right)
    want_l = oracle.normalize_faiss(left) if algorithm == 1 else oracle.normalize_hnsw(left)
    assert np.array_equal(ln, want_l)
    cos64 = 1 - (left.astype(np.float64) @ right.T.astype(np.float64)) / np.outer(np.linalg.norm(left.astype(np.float64), axis=1), np.linalg.norm(right.astype(np.float64), axis=1))
    assert np.abs(cs - cos64).max() < 1e-5
    # hand-checkable: (1,2,3) vs (4,6,8)
    a, b = np.array([[1, 2, 3]], np.float32), np.array([[4, 6, 8]], np.float32)
    assert oracle.calc_distance(algorithm, oracle_lib.L2, a, b)[0][0, 0] == 50.0
    assert oracle.calc_distance(algorithm, oracle_lib.IP, a, b)[0][0, 0] == -39.0


def test_hnsw_reference_hand_written_rows(oracle):
    """The reference's hand-written HNSW fixture (test/unit_test/vector/test_vector_index_hnsw.cc:181-223): ten parallel
    16-d rows j * m, m in {1, 3, 4, ..., 11}, ids 0..9, M = 2 links — small enough to reason about by hand."""
    base = np.arange(16, dtype=np.float32)
    xb = np.stack([base * m for m in (1, 3, 4, 5, 6, 7, 8, 9, 10, 11)]).astype(np.float32)
    labels = np.arange(10, dtype=np.int64)
    q = xb[[2, 7]]
    # L2: a row is its own nearest neighbour at distance 0, then its neighbours in the progression
    h = oracle_lib.OracleHnsw(oracle, L2, 16, 100, 2, 200)
    h.add(xb, labels)
    D, I, _, _ = h.search(q, 3, ef=10)
    assert I[:, 0].tolist() == [2, 7] and D[:, 0].tolist() == [0.0, 0.0]
    assert set(I[0, 1:]) == {1, 3} and set(I[1, 1:]) == {6, 8}
    h.close()
    # inner product (distance 1 - ip): the longest row wins for every positive query
    h = oracle_lib.OracleHnsw(oracle, IP, 16, 100, 2, 200)
    h.add(xb, labels)
    D, I, _, _ = h.search(q, 2, ef=10)
    assert I[:, 0].tolist() == [9, 9] and I[:, 1].tolist() == [8, 8]
    assert D[0, 0] == np.float32(1.0) - np.float32(np.dot(xb[2].astype(np.float64), xb[9].astype(np.float64)))
    h.close()
    # cosine: every row is parallel to every other one -> every returned distance is ~0 (with M = 2 links the graph
    # over identical normalised points need not reach all ten, so only the hits that do come back are checked)
    h = oracle_lib.OracleHnsw(oracle, COSINE, 16, 100, 2, 200)
    h.add(xb, labels)
    D, I, _, _ = h.search(q, 10, ef=16)
    hit = I >= 0
    assert hit[:, 0].all() and len(set(I[0][hit[0]].tolist())) == int(hit[0].sum()) and np.abs(D[hit]).max() < 1e-5
    h.close()


def test_hnsw_import_adopts_an_exported_graph(oracle):
    """oracle_hnsw_import: a graph exported by one oracle (or by the engine, same layout) and adopted by a fresh one is searched
    identically — the mechanism behind parity runs on graphs built by concurrent writers (not reproducible by re-insertion)."""
    import oracle_lib
    rng = np.random.default_rng(21)
    n, d, M, efc = 1500, 24, 8, 60
    xb = rng.random((n, d)).astype(np.float32)
    labels = np.arange(10, 10 + n, dtype=np.int64)
    for metric in (oracle_lib.L2, oracle_lib.COSINE):
        a = oracle_lib.OracleHnsw(oracle, metric, d, n, M, efc)
        a.add(xb, labels)
        blob = a.export()
        b = oracle_lib.OracleHnsw(oracle, metric, d, n, M, efc)
        b.load(blob)
        assert np.array_equal(b.export(), blob)
        xq = rng.random((30, d)).astype(np.float32)
        Da, Ia, nda, nha = a.search(xq, 7, ef=40, nthreads=2)
        Db, Ib, ndb, nhb = b.search(xq, 7, ef=40, nthreads=2)
        assert np.array_equal(Ia, Ib) and np.array_equal(Da.view(np.uint32), Db.view(np.uint32))
        assert np.array_equal(nda, ndb) and np.array_equal(nha, nhb)
        # a blob of another shape is refused
        c = oracle_lib.OracleHnsw(oracle, metric, d + 8, n, M, efc)
        with pytest.raises(AssertionError):
            c.load(blob)
