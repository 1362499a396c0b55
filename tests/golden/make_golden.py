"""Generates tests/golden/*.npz from the REFERENCE ITSELF: oracle/_ref/libref.so is compiled from the
reference's own sources (oracle/Makefile `ref`, which needs the reference tree), so every array below is an
output of reference code.  The tests only read these fixtures; none of them needs the reference.

    python tests/golden/make_golden.py [vectors] [oracle] [harness]     # default: all three files

reference_vectors.npz (vectors)
  fp32 cases:  inputs from cuda/random_matrix.cpp after srand48(seed) (called as the harness calls it,
               cuda/test_MMult.cpp:77-78), outputs of cuda/REF_MMult.cpp (OpenBLAS cblas_sgemm) and of
               aarch64/REF_MMult.cpp (naive, fused by the reference's own flags).
  ones case:   aarch64/random_matrix.cpp (all 1.0f) -> every C element == K (SURVEY §8c fixture 3).
  int8 cases:  aarch64-int8/random_matrix.c ramp + aarch64-int8/REF_MMult.c.
oracle_vs_reference.npz (oracle): what tests/test_oracle_vs_ref.py compares the oracle against.
reference_harness.npz (harness): what the reference's harnesses compare MY_MMult against, for
  tests/test_ref_harness_gpu.py: the cuda/ sweep's OpenBLAS results (N = 256..4096 step 256, a seeded sample
  of entries per size, plus digests of the inputs), the aarch64/ 256^3 result and the aarch64-int8/ results.
Bit-exact results are stored as SHA-256 digests of the whole array (tests/_libs.py sha256); results that are
compared within a tolerance are stored as values.
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import _libs  # noqa: E402

P = _libs.P
libc = C.CDLL(None)
libc.srand48.argtypes = [C.c_long]

# the parameters of tests/test_oracle_vs_ref.py and tests/test_ref_harness_gpu.py
SHAPES = [(1, 1, 1), (3, 5, 7), (64, 48, 80), (67, 45, 129), (128, 128, 128), (200, 9, 300)]
BLAS_SHAPES = [(64, 48, 80), (130, 70, 257), (256, 256, 256)]
I8_SHAPES = [(1, 1, 1), (4, 8, 16), (77, 77, 77), (33, 130, 65)]
HARNESS_SIZES = range(256, 4097, 256)          # cuda/parameters.h sweep as the harness was built (oracle/Makefile)
HARNESS_SAMPLE = 1024                          # stored OpenBLAS entries per size
I8_HARNESS_SHAPES = [(77, 77, 77), (64, 64, 64), (33, 130, 65), (512, 768, 1024)]   # (77,77,77): no CLI arguments


def key(*dims):
    return "x".join(str(d) for d in dims)


def reference_vectors(r):
    out = {}
    for idx, (m, n, k, seed) in enumerate([(64, 48, 80, 1), (96, 128, 160, 2), (130, 70, 257, 3), (128, 256, 64, 4)]):
        libc.srand48(seed)
        a = np.zeros(m * k, np.float32)
        b = np.zeros(k * n, np.float32)
        r.cuda_random_matrix(m, k, P(a), m)      # cuda/test_MMult.cpp:77
        r.cuda_random_matrix(k, n, P(b), k)      # cuda/test_MMult.cpp:78
        a, b = a.reshape(m, k), b.reshape(k, n)
        c_blas = np.zeros((m, n), np.float32)
        r.cuda_REF_MMult(m, n, k, P(a), k, P(b), n, P(c_blas), n)
        c_naive = np.zeros((m, n), np.float32)
        r.a64_REF_MMult(m, n, k, P(a), P(b), P(c_naive))
        out[f"f32_{idx}_shape"] = np.array([m, n, k, seed])
        out[f"f32_{idx}_a"], out[f"f32_{idx}_b"] = a, b
        out[f"f32_{idx}_c_openblas"], out[f"f32_{idx}_c_naive"] = c_blas, c_naive
    m = n = k = 96
    a = np.zeros((m, k), np.float32)
    b = np.zeros((k, n), np.float32)
    r.a64_random_matrix(m, k, P(a))
    r.a64_random_matrix(k, n, P(b))
    c = np.zeros((m, n), np.float32)
    r.a64_REF_MMult(m, n, k, P(a), P(b), P(c))
    out["ones_a"], out["ones_b"], out["ones_c"] = a, b, c
    for idx, (m, n, k) in enumerate([(77, 77, 77), (64, 96, 128), (5, 130, 33)]):
        a = np.zeros((m, k), np.int8)
        b = np.zeros((k, n), np.int8)
        r.i8_random_matrix(m, k, P(a), k)
        r.i8_random_matrix(k, n, P(b), n)
        c = np.zeros((m, n), np.int32)
        r.i8_REF_MMult(m, n, k, P(a), k, P(b), n, P(c), n)
        out[f"s8_{idx}_a"], out[f"s8_{idx}_b"], out[f"s8_{idx}_c"] = a, b, c
    return out


def oracle_pins(r, o):
    """The reference side of every comparison in tests/test_oracle_vs_ref.py, on the same inputs."""
    out = {}
    for m, n, k in SHAPES:
        libc.srand48(42)
        a = np.zeros(m * k, np.float32)
        r.cuda_random_matrix(m, k, P(a), m)
        out[f"rand_{key(m, n, k)}_sha256"] = _libs.sha256(a)
        # inputs from the oracle's generator (pinned by the digest above), C += A*B from a random C
        a, b = _libs.gen_f32(o, m, k, 5), _libs.gen_f32(o, k, n, 6)
        c0 = _libs.gen_f32(o, m, n, 7)
        c = c0.copy()
        r.a64_REF_MMult(m, n, k, P(a), P(b), P(c))
        out[f"naive_{key(m, n, k)}_sha256"] = _libs.sha256(c)
        c = c0.copy()
        r.a64_MY_MMult(m, n, k, P(a), k, P(b), n, P(c), n)
        out[f"mmult0_{key(m, n, k)}_sha256"] = _libs.sha256(c)
    m, n = 37, 53
    a = np.zeros((m, n), np.float32)
    r.a64_random_matrix(m, n, P(a))
    i = np.zeros((m, n), np.int8)
    r.i8_random_matrix(m, n, P(i), n)
    out[f"ones_{key(m, n)}"], out[f"ramp_{key(m, n)}"] = a, i
    rng = np.random.default_rng(2024)
    for m, n, k in BLAS_SHAPES:
        a, b = _libs.gen_f32(o, m, k, 8), _libs.gen_f32(o, k, n, 9)
        c = np.full((m, n), 123.0, np.float32)          # beta = 0 must overwrite
        r.cuda_REF_MMult(m, n, k, P(a), k, P(b), n, P(c), n)
        idx = np.sort(rng.choice(m * n, min(m * n, 2048), replace=False)).astype(np.int32)
        out[f"blas_{key(m, n, k)}_idx"], out[f"blas_{key(m, n, k)}_val"] = idx, c.ravel()[idx]
    for m, n, k in I8_SHAPES:
        a, b = _libs.gen_s8(o, m, k, 3), _libs.gen_s8(o, k, n, 4)
        c = (np.arange(m * n, dtype=np.int32).reshape(m, n) % 11) - 5
        r.i8_REF_MMult(m, n, k, P(a), k, P(b), n, P(c), n)
        out[f"i8_{key(m, n, k)}_sha256"] = _libs.sha256(c)
    # compare_matrices of each family on the pairs the test builds
    m, n = 40, 50
    a = _libs.gen_f32(o, m, n, 1)
    b = a.copy()
    b[17, 23] += 0.25
    out["cmp_cuda"] = np.float32(r.cuda_compare_matrices(m, n, P(a), n, P(b), n))
    out["cmp_a64"] = np.float32(r.a64_compare_matrices(m, n, P(a), P(b)))
    ia = np.arange(m * n, dtype=np.int32).reshape(m, n)
    ib = ia.copy()
    ib[3, 4] -= 9
    out["cmp_i8"] = np.int32(r.i8_compare_matrices(m, n, P(ia), n, P(ib), n))
    return out


def harness_vectors(r):
    """cuda/test_MMult.cpp draws A, B and a C it then zeroes from one never-seeded drand48 stream, size after
    size, and compares MY_MMult against REF_MMult (OpenBLAS).  Kept per size: digests of A and B, and REF_MMult
    at HARNESS_SAMPLE seeded positions (flat row-major index)."""
    out = {"cuda_sizes": np.array(list(HARNESS_SIZES), np.int32)}
    _libs.seed_unseeded_drand48()
    for p in HARNESS_SIZES:
        a, b, cold = (np.zeros(p * p, np.float32) for _ in range(3))
        r.cuda_random_matrix(p, p, P(a), p)      # cuda/test_MMult.cpp:77-79
        r.cuda_random_matrix(p, p, P(b), p)
        r.cuda_random_matrix(p, p, P(cold), p)
        cref = np.zeros(p * p, np.float32)
        r.cuda_REF_MMult(p, p, p, P(a), p, P(b), p, P(cref), p)
        idx = np.sort(np.random.default_rng(p).choice(p * p, HARNESS_SAMPLE, replace=False)).astype(np.int32)
        out[f"cuda_{p}_a_sha256"], out[f"cuda_{p}_b_sha256"] = _libs.sha256(a), _libs.sha256(b)
        out[f"cuda_{p}_idx"], out[f"cuda_{p}_cref"] = idx, cref[idx]
    # aarch64/test_MMult.cpp at 256^3: random_matrix fills 1.0f, cref = 0 then REF_MMult (C += A*B)
    p = 256
    a, b = np.zeros((p, p), np.float32), np.zeros((p, p), np.float32)
    r.a64_random_matrix(p, p, P(a))
    r.a64_random_matrix(p, p, P(b))
    c = np.zeros((p, p), np.float32)
    r.a64_REF_MMult(p, p, p, P(a), P(b), P(c))
    out["a64_256_cref"] = c
    # aarch64-int8/test_MMult.c: ramp inputs (lda = k, ldb = n), cref = 0 then REF_MMult
    for m, n, k in I8_HARNESS_SHAPES:
        a, b = np.zeros((m, k), np.int8), np.zeros((k, n), np.int8)
        r.i8_random_matrix(m, k, P(a), k)
        r.i8_random_matrix(k, n, P(b), n)
        c = np.zeros((m, n), np.int32)
        r.i8_REF_MMult(m, n, k, P(a), k, P(b), n, P(c), n)
        out[f"i8_{key(m, n, k)}_cref_sha256"] = _libs.sha256(c)
    return out


def main(which):
    r = _libs.load_ref()
    r.openblas_set_num_threads(1)
    o = _libs.load_oracle()
    files = {"vectors": ("reference_vectors.npz", lambda: reference_vectors(r)),
             "oracle": ("oracle_vs_reference.npz", lambda: oracle_pins(r, o)),
             "harness": ("reference_harness.npz", lambda: harness_vectors(r))}
    for name in which or files:
        fn, make = files[name]
        out = make()
        np.savez_compressed(os.path.join(HERE, fn), **out)
        print("wrote", os.path.join(HERE, fn), len(out), "arrays")


if __name__ == "__main__":
    main(sys.argv[1:])
