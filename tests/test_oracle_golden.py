"""CPU: pins the oracle against the reference's own golden vectors (tests/golden/, transcribed by
oracle/make_golden.py from the reference test-suite) and against an independent float64 NumPy
computation.  No GPU, no product code."""
import json
import os

import numpy as np
import pytest

import oracle

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_vectors.json")))


@pytest.mark.parametrize("case", GOLD["cases"], ids=lambda c: c["name"])
def test_reference_known_answers(case):
    ds = np.array(case["dataset"], np.float32)
    qs = np.array(case["queries"], np.float32)
    keep = case.get("filter_keep")
    if keep is not None:
        sub = ds[keep]
        dist, idx = oracle.knn(sub, qs, case["k"], case["metric"])
        idx = np.array(keep)[idx]
    else:
        dist, idx = oracle.knn(ds, qs, case["k"], case["metric"])
    assert idx.tolist() == case["neighbors"]
    np.testing.assert_allclose(dist, np.array(case["distances"], np.float32), atol=case["eps"])


def test_reference_label_case():
    lc = GOLD["label_case"]
    pts = np.array(lc["points"], np.float32)
    labels = np.array(lc["labels"])
    _, idx = oracle.knn(pts, pts, lc["k"], lc["metric"])
    assert (labels[idx] == labels[:, None]).all()


def test_fp8_known_answers():
    for v, code in GOLD["fp8"]["unsigned"]:
        assert int(oracle.fp8_encode([v])[0]) == code, v
    for code, v in GOLD["fp8"]["decode_unsigned"]:
        assert float(oracle.fp8_decode([code])[0]) == v
    # signed variant: sign lives in the LSB (ivf_pq_fp_8bit.cuh:56-60, 76-80)
    x = np.array([-1.0, 1.0, -3.5, 0.0], np.float32)
    enc = oracle.fp8_encode(x, signed=True)
    assert (enc & 1).tolist() == [1, 0, 1, 0]
    dec = oracle.fp8_decode(enc, signed=True)
    assert np.sign(dec[:3]).tolist() == [-1.0, 1.0, -1.0]
    # monotone and within 2^-3 relative error (3 value bits, truncation + half-ulp bias)
    v = np.exp(np.linspace(np.log(1e-4), np.log(6e4), 2000)).astype(np.float32)
    r = oracle.fp8_decode(oracle.fp8_encode(v))
    assert (np.diff(r) >= 0).all()
    assert np.max(np.abs(r - v) / v) <= 0.125 / 2 + 1e-6


@pytest.mark.parametrize("metric", ["sqeuclidean", "l2_unexpanded", "inner_product", "cosine", "euclidean"])
def test_knn_against_float64(metric):
    rng = np.random.default_rng(1234)
    ds = rng.uniform(-1, 1, (500, 33)).astype(np.float32)
    qs = rng.uniform(-1, 1, (40, 33)).astype(np.float32)
    k = 7
    dist, idx = oracle.knn(ds, qs, k, metric)
    a, b = qs.astype(np.float64), ds.astype(np.float64)
    if metric in ("sqeuclidean", "l2_unexpanded", "euclidean"):
        full = ((a[:, None, :] - b[None, :, :]) ** 2).sum(-1)
        if metric == "euclidean":
            full = np.sqrt(full)
        order = np.argsort(full, axis=1, kind="stable")[:, :k]
    elif metric == "inner_product":
        full = a @ b.T
        order = np.argsort(-full, axis=1, kind="stable")[:, :k]
    else:
        full = 1 - (a @ b.T) / (np.linalg.norm(a, axis=1)[:, None] * np.linalg.norm(b, axis=1)[None, :])
        order = np.argsort(full, axis=1, kind="stable")[:, :k]
    ref = np.take_along_axis(full, order, axis=1)
    assert oracle.knn_match(idx, dist, order, ref, eps=1e-4) == 0


def test_knn_fewer_rows_than_k():
    ds = np.eye(3, dtype=np.float32)
    dist, idx = oracle.knn(ds, ds[:1], 5)
    assert idx[0, :3].tolist() == [0, 1, 2] and idx[0, 3:].tolist() == [-1, -1]


def test_select_k_ties_and_padding():
    v = np.array([[3, 1, 1, 2, 1], [5, 4, 3, 2, 1]], np.float32)
    ov, oi = oracle.select_k(v, 3, True)
    assert oi.tolist() == [[1, 2, 4], [4, 3, 2]]
    ov, oi = oracle.select_k(v, 2, False)
    assert oi.tolist() == [[0, 3], [0, 1]]
    ov, oi = oracle.select_k(v[:, :2], 4, True)
    assert oi[0].tolist() == [1, 0, -1, -1]


def test_pq_packing_roundtrip():
    rng = np.random.default_rng(0)
    for bits in (4, 5, 6, 7, 8):
        codes = rng.integers(0, 1 << bits, (70, 24), dtype=np.uint8)
        packed = oracle.pack_pq_interleaved(codes, bits)
        assert packed.shape == (3, -(-24 // (128 // bits)), 32, 16)
        back = oracle.unpack_pq_interleaved(packed, 70, 24, bits)
        assert (back == codes).all()
    # 8-bit: code j of vector v is simply byte j%16 of chunk j/16 (SURVEY Appendix B)
    codes = rng.integers(0, 256, (33, 32), dtype=np.uint8)
    packed = oracle.pack_pq_interleaved(codes, 8)
    assert packed[1, 1, 0, 5] == codes[32, 21]


def test_ivf_flat_interleave_layout():
    rows = np.arange(40 * 8, dtype=np.float32).reshape(40, 8)
    flat = oracle.interleave_ivf_flat(rows)
    veclen = 4
    for r, k in [(0, 0), (5, 3), (5, 4), (33, 7)]:
        off = (r // 32) * 32 * 8 + (k // veclen) * 32 * veclen + (r % 32) * veclen + k % veclen
        assert flat[off] == rows[r, k]


def test_blocked_gemm_formulation_agrees_with_the_pinned_scan():
    """oracle.knn_blocked (SGEMM + top-k, the throughput formulation used as bench.py's CPU baseline) returns the same
    neighbours as oracle.knn (sequential fmaf chains, the parity checker) up to last-ulp rounding of the expanded form."""
    rng = np.random.default_rng(11)
    ds = rng.standard_normal((30000, 48)).astype(np.float32)
    qs = rng.standard_normal((300, 48)).astype(np.float32)
    for metric in ("sqeuclidean", "inner_product"):
        d0, i0 = oracle.knn(ds, qs, 7, metric)
        d1, i1 = oracle.knn_blocked(ds, qs, 7, metric, rows_per_block=7000, queries_per_block=128)
        assert oracle.recall_with_ties(i1, d1, i0, d0, eps=1e-3) >= 0.9999
        assert (i0 == i1).mean() >= 0.999
        np.testing.assert_allclose(d1, d0, rtol=1e-4, atol=2e-4)


# ---- fixtures produced by the REFERENCE's own CPU search, executed in the build container (oracle/make_golden_cuvs_bench.py)
def _ref_exec_cases():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cuvs_bench_cpu_groundtruth.json")
    return json.load(open(path))["cases"]


def _ref_exec_inputs(case):
    rng = np.random.default_rng(case["seed"])  # the same Generator calls as oracle/make_golden_cuvs_bench.py: inputs()
    ds = rng.standard_normal((case["n"], case["d"]), dtype=np.float32)
    qs = rng.standard_normal((case["nq"], case["d"]), dtype=np.float32)
    return ds, qs


@pytest.mark.parametrize("case", _ref_exec_cases(), ids=lambda c: c["name"])
def test_oracle_knn_reproduces_the_reference_cpu_search(case):
    """python/cuvs_bench/cuvs_bench/generate_groundtruth/__main__.py:104-214 (cpu_search / calc_truth, numpy) is the one CPU
    implementation of exact kNN the reference ships.  Its outputs on seeded inputs are committed; the oracle must return the
    same neighbours (the reference sums in numpy's pairwise order, the oracle in fmaf chains: distances to 1e-5 relative,
    ids identical except where two distances tie within that tolerance)."""
    ds, qs = _ref_exec_inputs(case)
    metric = "sqeuclidean" if case["metric"] == "squeclidean" else "inner_product"
    d, i = oracle.knn(ds, qs, case["k"], metric)
    ri, rd = np.array(case["ids"]), np.array(case["distances"], np.float32)
    np.testing.assert_allclose(d, rd, rtol=2e-5, atol=1e-5)
    same = (i == ri)
    assert same.mean() >= 0.999, f"{(~same).sum()} of {same.size} neighbour ids differ from the reference's CPU search"
    for q, j in zip(*np.nonzero(~same)):  # a differing slot must be a tie within the arithmetic tolerance
        assert abs(float(d[q, j]) - float(rd[q, j])) <= 2e-5 * max(1.0, abs(float(rd[q, j])))
        assert set(i[q].tolist()) == set(ri[q].tolist()) or abs(float(rd[q, -1]) - float(d[q, -1])) <= 2e-5 * max(1.0, abs(float(rd[q, -1])))


def test_fp8_restatement_equals_the_reference_code_compiled_here():
    """The REFERENCE's fp_8bit<5, Signed> (cpp/src/neighbors/ivf_pq/ivf_pq_fp_8bit.cuh:31-100), compiled from the reference
    source by oracle/ref_fp8/Makefile, recorded every decode and a dense sweep of encodes in tests/golden/reference_fp8.npz
    (oracle/make_golden_fp8.py).  The oracle's restatement must agree with it on every byte and on every float of the sweep,
    for both the unsigned and the signed variant."""
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_fp8.npz"))
    floats = gold["floats"]
    for signed in (0, 1):
        codes = np.arange(256, dtype=np.uint8)
        dec_ref, dec_half = gold[f"decode_{signed}"], gold[f"decode_half_{signed}"]
        np.testing.assert_array_equal(oracle.fp8_decode(codes, signed=bool(signed)), dec_ref)
        # the reference's HALF decode (fp_8bit2half, :88-99) is the same bit trick on a 5-bit fp16 exponent: it agrees with the
        # float decode wherever the value is a normal fp16 number, and differs only in the lowest exponent (codes 0..7: fp16
        # subnormals) and the highest one (codes 248..255: beyond fp16's range) — a property of the reference, recorded here
        np.testing.assert_array_equal(dec_half[8:248], dec_ref[8:248])
        assert set(np.nonzero(~(dec_half == dec_ref))[0].tolist()) <= set(range(8)) | set(range(248, 256))
        xs = floats if signed else floats[floats >= 0]
        xs = np.concatenate([xs, -xs]) if signed else xs
        np.testing.assert_array_equal(oracle.fp8_encode(xs, signed=bool(signed)), gold[f"encode_{signed}"])
    # unsigned encode of negative inputs: "all small and negative numbers are truncated to zero" (ivf_pq_fp_8bit.cuh:62-63)
    neg = -np.abs(floats[1:200])
    np.testing.assert_array_equal(oracle.fp8_encode(neg), gold["encode_negative_0"])
