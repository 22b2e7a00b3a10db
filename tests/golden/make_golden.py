"""Regenerates tests/golden/simd_kat.json and tests/golden/simd_ref_samples.json from the REFERENCE's own kernels
(oracle/_ref, built from the reference's src/simd by oracle/Makefile).  Needs oracle/_ref, so it runs only where the
reference tree is available:
    python tests/golden/make_golden.py
Inputs are reproducible: (a) the reference's unit-test fixture generator (default-seeded std::mt19937,
test/unit_test/vector/test_vector_index_flat.cc:491-500) restated by oracle_fixture_mt19937, and
(b) numpy default_rng(seed) draws.  Outputs are the bit patterns returned by
fvec_{L2sqr,inner_product}_avx512 (src/simd/distances_avx512.cc:48-143)."""
import json
import os
import struct
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle_lib  # noqa: E402


def hx(f):
    return "0x%08x" % struct.unpack("<I", struct.pack("<f", f))[0]


def main():
    o = oracle_lib.load()
    r = oracle_lib.load_ref()
    assert r is not None, "build oracle/_ref first (make -C oracle)"
    assert r.ref_simd_type() == b"AVX512"
    cases = []
    for d in [1, 2, 3, 4, 5, 7, 8, 9, 12, 15, 16, 17, 23, 24, 31, 32, 33, 64, 100, 128, 256, 512, 768, 1000, 1536, 4096]:
        x = o.fixture(10, d)
        a, b = x[0], x[1]
        cases.append({"gen": "fixture", "d": d,
                      "l2": hx(r.ref_fvec_L2sqr_avx512(a.ctypes.data, b.ctypes.data, d)),
                      "ip": hx(r.ref_fvec_inner_product_avx512(a.ctypes.data, b.ctypes.data, d)),
                      "l2_hooked": hx(r.ref_fvec_L2sqr(a.ctypes.data, b.ctypes.data, d)),
                      "ip_hooked": hx(r.ref_fvec_inner_product(a.ctypes.data, b.ctypes.data, d))})
    for seed, d in [(1, 6), (2, 13), (3, 40), (4, 128), (5, 768), (6, 769), (7, 1537)]:
        g = np.random.default_rng(seed)
        a = g.standard_normal(d).astype(np.float32)
        b = g.standard_normal(d).astype(np.float32)
        cases.append({"gen": "normal", "seed": seed, "d": d,
                      "l2": hx(r.ref_fvec_L2sqr_avx512(a.ctypes.data, b.ctypes.data, d)),
                      "ip": hx(r.ref_fvec_inner_product_avx512(a.ctypes.data, b.ctypes.data, d))})
    row0 = o.fixture(10, 8)[0]
    out = {"source": "reference src/simd compiled by oracle/Makefile (dingo-store dc8c439c), AVX512 variant",
           "fixture_d8_row0": [hx(float(v)) for v in row0], "cases": cases}
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "simd_kat.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", len(cases), "cases")
    write_samples(r)


def write_samples(r):
    """simd_ref_samples.json: the reference's answers on the seeded inputs that
    tests/test_oracle_simd.py::test_bitwise_against_reference_objects and
    tests/test_oracle_search.py::test_calc_distance_pinned_to_reference_kernels draw."""
    def both(x, y, d):
        return (hx(r.ref_fvec_L2sqr_avx512(x.ctypes.data, y.ctypes.data, d)),
                hx(r.ref_fvec_inner_product_avx512(x.ctypes.data, y.ctypes.data, d)))

    dims, per_dim = list(range(1, 70)) + [127, 128, 129, 767, 768, 769, 1536, 4096], 10
    rng = np.random.default_rng(0)
    l2, ip = [], []
    for d in dims:
        for _ in range(per_dim):
            x = rng.standard_normal(d).astype(np.float32)
            y = (rng.standard_normal(d) * 3).astype(np.float32)
            a, b = both(x, y, d)
            l2.append(a)
            ip.append(b)
    pairs = {"seed": 0, "dims": dims, "pairs_per_dim": per_dim, "l2": l2, "ip": ip}

    rng = np.random.default_rng(3)
    left = rng.random((5, 77), dtype=np.float32)
    right = rng.random((6, 77), dtype=np.float32) * 2 - 0.5
    grid = [[both(left[i], right[j], 77) for j in range(6)] for i in range(5)]
    calc = {"seed": 3, "left": [5, 77], "right": [6, 77],
            "l2": [[c[0] for c in row] for row in grid], "ip": [[c[1] for c in row] for row in grid]}

    out = {"source": "reference src/simd compiled by oracle/Makefile (dingo-store dc8c439c), AVX512 variant",
           "pairs": pairs, "calc_distance": calc}
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "simd_ref_samples.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")
    print("wrote", len(l2), "pairs and a 5 x 6 calc_distance grid")


if __name__ == "__main__":
    main()
