"""Pins the oracle's distance arithmetic: (1) against the reference's known-answer values (SURVEY.md §0 and
tests/golden/simd_kat.json), (2) bit-for-bit against the reference's answers on 770 seeded random pairs
(tests/golden/simd_ref_samples.json).  Both files hold what the reference's own src/simd objects returned
(tests/golden/make_golden.py)."""
import json
import os
import struct

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "simd_kat.json")
SAMPLES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "simd_ref_samples.json")


def hx(f):
    return "0x%08x" % struct.unpack("<I", struct.pack("<f", f))[0]


def test_fixture_generator_matches_survey_kat(oracle):
    # SURVEY.md §0: d=8 row0 of the reference's unit-test fixture
    want = ["0x3e0aba7c", "0x3f55c31f", "0x3f7807b8", "0x3e6256c0", "0x3e9dc812", "0x3f0c16a6", "0x3e40e734", "0x3f7e2d78"]
    row0 = oracle.fixture(10, 8)[0]
    assert [hx(float(v)) for v in row0] == want


def test_survey_known_answers(oracle):
    # SURVEY.md §0, AVX-512 column (the canonical arithmetic)
    kat = {8: ("0x401f384a", "0x40194098"), 128: ("0x41ba12ea", "0x4200ccb1"), 768: ("0x43072e00", "0x4341d979")}
    for d, (l2, ip) in kat.items():
        x = oracle.fixture(10, d)
        assert hx(oracle.l2sqr(x[0], x[1])) == l2
        assert hx(oracle.ip(x[0], x[1])) == ip


def test_golden_vectors(oracle):
    gold = json.load(open(GOLD))
    assert [hx(float(v)) for v in oracle.fixture(10, 8)[0]] == gold["fixture_d8_row0"]
    for c in gold["cases"]:
        d = c["d"]
        if c["gen"] == "fixture":
            x = oracle.fixture(10, d)
            a, b = x[0], x[1]
        else:
            g = np.random.default_rng(c["seed"])
            a = g.standard_normal(d).astype(np.float32)
            b = g.standard_normal(d).astype(np.float32)
        assert hx(oracle.l2sqr(a, b)) == c["l2"], c
        assert hx(oracle.ip(a, b)) == c["ip"], c


def test_bitwise_against_reference_objects(oracle):
    gold = json.load(open(SAMPLES))["pairs"]
    rng = np.random.default_rng(gold["seed"])
    i = 0
    for d in gold["dims"]:
        for _ in range(gold["pairs_per_dim"]):
            x = rng.standard_normal(d).astype(np.float32)
            y = (rng.standard_normal(d) * 3).astype(np.float32)
            assert hx(oracle.l2sqr(x, y)) == gold["l2"][i], (d, i)
            assert hx(oracle.ip(x, y)) == gold["ip"][i], (d, i)
            i += 1
    assert i == len(gold["l2"]) == len(gold["ip"])


def test_normalizers(oracle):
    rng = np.random.default_rng(1)
    x = rng.random((5, 33)).astype(np.float32)
    nf = oracle.normalize_faiss(x)
    nh = oracle.normalize_hnsw(x)
    for a in (nf, nh):
        assert np.allclose(np.linalg.norm(a.astype(np.float64), axis=1), 1.0, atol=1e-6)
    # already-normalised rows are left untouched by the faiss flavour (|1-n2| <= 1e-5), utils.cc:485
    again = oracle.normalize_faiss(nf)
    assert np.array_equal(again, nf)
    z = np.zeros((1, 8), np.float32)
    assert np.array_equal(oracle.normalize_faiss(z), z)
