#!/usr/bin/env python
"""Golden vectors of the reference's fp_8bit<5, Signed> (the LUT element type of its IVF-PQ scan), from the reference's own
code (test infrastructure).

oracle/ref_fp8/Makefile compiles cpp/src/neighbors/ivf_pq/ivf_pq_fp_8bit.cuh of a reference checkout into
oracle/_ref/libref_fp8.so (git-ignored).  This script loads it, runs every encode / decode the tests check and writes inputs
and outputs to tests/golden/reference_fp8.npz, so the comparison needs neither the checkout nor the library.

    make -C oracle/ref_fp8 REF=<reference checkout>
    python oracle/make_golden_fp8.py                  # rewrites the fixture
"""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "oracle", "_ref", "libref_fp8.so")
OUT = os.path.join(ROOT, "tests", "golden", "reference_fp8.npz")


def sweep():
    """Special values, a log-uniform and a normal sample, powers of two and their lower neighbours."""
    rng = np.random.default_rng(0)
    return np.concatenate([
        np.array([0.0, -0.0, 1e-30, 1e-8, 2.0 ** -16, 2.0 ** -15, 2.0 ** -14, 0.5, 1.0, 1.5, 2.0, 3.999, 1000.0, 65504.0, 1e9,
                  1e30, np.inf], np.float32),
        (10.0 ** rng.uniform(-7, 7, 4000)).astype(np.float32),
        rng.standard_normal(2000).astype(np.float32) * 100.0,
        np.float32(2.0) ** np.arange(-20, 20, dtype=np.float32),
        np.nextafter(np.float32(2.0) ** np.arange(-18, 18, dtype=np.float32), np.float32(0)),
    ]).astype(np.float32)


def main():
    ref = C.CDLL(SO)
    ref.ref_fp8_encode.restype, ref.ref_fp8_encode.argtypes = C.c_uint8, [C.c_float, C.c_int]
    ref.ref_fp8_decode.restype, ref.ref_fp8_decode.argtypes = C.c_float, [C.c_uint8, C.c_int]
    ref.ref_fp8_decode_half.restype, ref.ref_fp8_decode_half.argtypes = C.c_float, [C.c_uint8, C.c_int]
    floats = sweep()
    out = {"floats": floats}
    for signed in (0, 1):
        out[f"decode_{signed}"] = np.array([ref.ref_fp8_decode(b, signed) for b in range(256)], np.float32)
        out[f"decode_half_{signed}"] = np.array([ref.ref_fp8_decode_half(b, signed) for b in range(256)], np.float32)
        xs = np.concatenate([floats, -floats]) if signed else floats[floats >= 0]
        out[f"encode_{signed}"] = np.array([ref.ref_fp8_encode(float(v), signed) for v in xs], np.uint8)
    # unsigned encode of negative inputs
    out["encode_negative_0"] = np.array([ref.ref_fp8_encode(float(v), 0) for v in -np.abs(floats[1:200])], np.uint8)
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
