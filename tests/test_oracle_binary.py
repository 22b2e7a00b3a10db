"""CPU oracle of the binary (Hamming) indexes against numpy restatements: distances, the +-1 / threshold round trip,
Flat / IVF search with mass ties, and the truncated range-search radius.  No GPU needed."""
import numpy as np
import pytest

import oracle_binary_lib


@pytest.fixture(scope="module")
def bo():
    return oracle_binary_lib.load()


def np_hamming(a, b):
    """[na, nb] Hamming matrix via np.unpackbits."""
    ua = np.unpackbits(a, axis=1).astype(np.int32)
    ub = np.unpackbits(b, axis=1).astype(np.int32)
    return (ua[:, None, :] != ub[None, :, :]).sum(-1)


def np_topk(dist, ids, k, keep=None):
    """(distance, id) ascending top-k per row, -1 / 0 padded."""
    nq = dist.shape[0]
    D = np.zeros((nq, k), np.float32)
    I = np.full((nq, k), -1, np.int64)
    for q in range(nq):
        cand = [(int(dist[q, j]), int(ids[j])) for j in range(len(ids)) if ids[j] >= 0 and (keep is None or keep(q, j))]
        cand.sort()
        for r, (d, i) in enumerate(cand[:k]):
            D[q, r], I[q, r] = d, i
    return D, I


def test_hamming_hand_values(bo):
    assert bo.hamming(np.array([0x00], np.uint8), np.array([0xFF], np.uint8)) == 8
    assert bo.hamming(np.array([0b1010, 0], np.uint8), np.array([0b0110, 0x80], np.uint8)) == 3
    a = np.zeros(4096, np.uint8)
    assert bo.hamming(a, a) == 0
    assert bo.hamming(a, np.full(4096, 0xFF, np.uint8)) == 32768


@pytest.mark.parametrize("nbytes", [1, 3, 8, 32, 128, 512])
def test_hamming_matrix_matches_unpackbits(bo, nbytes):
    rng = np.random.default_rng(nbytes)
    a = rng.integers(0, 256, (7, nbytes), dtype=np.uint8)
    b = rng.integers(0, 256, (5, nbytes), dtype=np.uint8)
    assert np.array_equal(bo.calc_distance(a, b), np_hamming(a, b).astype(np.float32))


def test_binary_to_real_is_lsb_first_and_round_trips(bo):
    x = np.array([[0b00000001, 0b10000000]], np.uint8)
    r = bo.binary_to_real(x)
    expect = -np.ones(16, np.float32)
    expect[0] = 1.0   # bit 0 of byte 0
    expect[15] = 1.0  # bit 7 of byte 1
    assert np.array_equal(r[0], expect)
    rng = np.random.default_rng(1)
    y = rng.integers(0, 256, (50, 16), dtype=np.uint8)
    assert np.array_equal(bo.real_to_binary(bo.binary_to_real(y)), y)
    # threshold is strictly > 0: zero components give 0 bits
    assert np.array_equal(bo.real_to_binary(np.array([[0.0, 1e-9, -1e-9, 0, 0, 0, 0, 2.0]], np.float32)), np.array([[0b10000010]], np.uint8))


@pytest.mark.parametrize("dim,k", [(8, 5), (64, 10), (256, 33)])
def test_flat_search_matches_numpy_with_mass_ties(bo, dim, k):
    rng = np.random.default_rng(dim)
    n, nq = 300, 9
    # few distinct rows: every distance is shared by many rows, so the id tie-break decides the order
    base = rng.integers(0, 256, (6, dim // 8), dtype=np.uint8)
    xb = base[rng.integers(0, 6, n)]
    ids = rng.permutation(np.arange(1000, 1000 + n)).astype(np.int64)  # not in insertion order
    ids[::17] = -1  # removed slots
    xq = rng.integers(0, 256, (nq, dim // 8), dtype=np.uint8)
    D, I = bo.flat_search(xb, ids, xq, k)
    De, Ie = np_topk(np_hamming(xq, xb), ids, k)
    assert np.array_equal(I, Ie) and np.array_equal(D, De)


def test_flat_search_filters(bo):
    rng = np.random.default_rng(3)
    xb = rng.integers(0, 256, (200, 4), dtype=np.uint8)
    ids = np.arange(200, dtype=np.int64)
    xq = rng.integers(0, 256, (4, 4), dtype=np.uint8)
    dist = np_hamming(xq, xb)
    D, I = bo.flat_search(xb, ids, xq, 10, id_range=(50, 120))
    assert np.array_equal(I, np_topk(dist, ids, 10, lambda q, j: 50 <= ids[j] < 120)[1])
    allow = np.arange(0, 200, 7)
    D, I = bo.flat_search(xb, ids, xq, 10, sorted_ids=allow)
    assert np.array_equal(I, np_topk(dist, ids, 10, lambda q, j: ids[j] % 7 == 0)[1])
    D, I = bo.flat_search(xb, ids, xq, 10, sorted_ids=allow, negate=True)
    assert np.array_equal(I, np_topk(dist, ids, 10, lambda q, j: ids[j] % 7 != 0)[1])


def test_range_search_truncates_radius(bo):
    xb = np.array([[0x00], [0x01], [0x03], [0x07], [0x0F], [0x1F]], np.uint8)  # distances 0..5 from 0x00
    ids = np.arange(10, 16, dtype=np.int64)
    xq = np.zeros((1, 1), np.uint8)
    for radius, hits in [(3.0, 3), (3.9, 3), (4.0, 4), (0.5, 0), (0.0, 0), (-2.0, 0), (10.1, 6)]:
        D, I, C = bo.flat_range_search(xb, ids, xq, radius, 8)
        assert C[0] == hits, (radius, C[0])
        assert list(I[0, :hits]) == list(range(10, 10 + hits)) and (I[0, hits:] == -1).all()
    D, I, C = bo.flat_range_search(xb, ids, xq, 10.1, 2)  # at most max_results, closest first
    assert C[0] == 2 and list(I[0]) == [10, 11]


def test_assign_and_ivf_search_with_centroid_ties(bo):
    rng = np.random.default_rng(5)
    dim, nlist, n, nq = 32, 8, 400, 16
    cent = rng.integers(0, 256, (nlist, dim // 8), dtype=np.uint8)
    cent[5] = cent[1]  # identical centroids: the (distance, list id) rule must pick list 1 first
    xb = rng.integers(0, 256, (n, dim // 8), dtype=np.uint8)
    a = bo.assign(xb, cent)
    dc = np_hamming(xb, cent)
    assert np.array_equal(a, np.argmin(dc, axis=1))  # argmin returns the first (smallest index) minimum
    assert not (a == 5).any()
    order = np.argsort(a, kind="stable")
    xs, ids = xb[order], np.arange(n, dtype=np.int64)[order] * 3 + 1
    off = np.concatenate([[0], np.cumsum(np.bincount(a, minlength=nlist))]).astype(np.int64)
    xq = rng.integers(0, 256, (nq, dim // 8), dtype=np.uint8)
    for nprobe in (1, 3, nlist):
        D, I = bo.ivf_search(cent, off, xs, ids, xq, 10, nprobe)
        dq = np_hamming(xq, cent)
        for q in range(nq):
            probes = sorted(range(nlist), key=lambda c: (dq[q, c], c))[:nprobe]
            rows = np.concatenate([np.arange(off[c], off[c + 1]) for c in probes]).astype(np.int64)
            De, Ie = np_topk(np_hamming(xq[q:q + 1], xs[rows]), ids[rows], 10)
            assert np.array_equal(I[q], Ie[0]) and np.array_equal(D[q], De[0])
    D, I, C = bo.ivf_range_search(cent, off, xs, ids, xq, 12.7, 64, nlist)
    Df, If, Cf = bo.flat_range_search(xs, ids, xq, 12, 64)
    assert np.array_equal(C, Cf) and np.array_equal(I, If)


def test_kmeans_is_threshold_of_float_kmeans(bo):
    import oracle_lib
    o = oracle_lib.load()
    rng = np.random.default_rng(7)
    x = rng.integers(0, 256, (600, 8), dtype=np.uint8)
    c = bo.kmeans(x, 4)
    cf = o.kmeans(oracle_lib.L2, bo.binary_to_real(x), 4)
    assert np.array_equal(c, bo.real_to_binary(cf))
