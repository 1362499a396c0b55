"""Pins the oracle (oracle/oracle.c) against the reference itself: tests/golden/oracle_vs_reference.npz holds
what the reference's own sources (compiled into oracle/_ref/libref.so) produced on the inputs below, written
by tests/golden/make_golden.py.  Bit-exact results are stored as SHA-256 digests of the whole array.  CPU only."""
import os

import numpy as np
import pytest

import _libs
from _libs import P

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "oracle_vs_reference.npz"))

SHAPES = [(1, 1, 1), (3, 5, 7), (64, 48, 80), (67, 45, 129), (128, 128, 128), (200, 9, 300)]


def key(*dims):
    return "x".join(str(d) for d in dims)


def same_bits(x, name):
    return np.array_equal(_libs.sha256(x), G[name])


@pytest.mark.parametrize("m,n,k", SHAPES)
def test_random_matrix_cuda_bit_exact(oracle, m, n, k):
    """cuda/random_matrix.cpp after srand48(42)."""
    oracle.oracle_seed(42)
    a2 = np.zeros(m * k, np.float32)
    oracle.oracle_random_matrix_cuda(m, k, P(a2), m)
    assert same_bits(a2, f"rand_{key(m, n, k)}_sha256")
    assert a2.min() >= -1.0 and a2.max() < 1.0


def test_random_matrix_ones_and_int8_ramp(oracle):
    m, n = 37, 53
    a1, a2 = G[f"ones_{key(m, n)}"], np.zeros((m, n), np.float32)
    oracle.oracle_random_matrix_ones(m, n, P(a2))
    assert np.array_equal(a1, a2) and (a1 == 1.0).all()
    i1, i2 = G[f"ramp_{key(m, n)}"], np.zeros((m, n), np.int8)
    oracle.oracle_random_int8_ramp(m, n, P(i2), n)
    assert np.array_equal(i1, i2) and set(np.unique(i1)) == {0, 1, 2}


@pytest.mark.parametrize("m,n,k", SHAPES)
def test_naive_ref_mmult_matches_reference_build(oracle, m, n, k):
    """aarch64/REF_MMult.cpp built with the reference's flags fuses multiply-add: the oracle's
    _fma variant (and its threaded _fast form) must be bit-identical, with C += semantics."""
    a, b = _libs.gen_f32(oracle, m, k, 5), _libs.gen_f32(oracle, k, n, 6)
    c0 = _libs.gen_f32(oracle, m, n, 7)
    c1 = c0.copy()
    oracle.oracle_ref_mmult_f32_fma(m, n, k, P(a), k, P(b), n, P(c1), n)
    c2 = c0.copy()
    oracle.oracle_ref_mmult_f32_fma_fast(m, n, k, P(a), k, P(b), n, P(c2), n)
    assert same_bits(c1, f"naive_{key(m, n, k)}_sha256") and np.array_equal(c1, c2)
    c_ref = c1                      # bit-identical to the reference's result
    # the reference's CPU MY_MMult (aarch64/MMult0.cpp) is the same loop nest
    assert same_bits(c_ref, f"mmult0_{key(m, n, k)}_sha256")
    # un-fused variant: same sequence, separately rounded; agrees to fp32 rounding noise
    c4 = c0.copy()
    oracle.oracle_ref_mmult_f32(m, n, k, P(a), k, P(b), n, P(c4), n)
    c5 = c0.copy()
    oracle.oracle_ref_mmult_f32_fast(m, n, k, P(a), k, P(b), n, P(c5), n)
    assert np.array_equal(c4, c5)
    assert np.abs(c4 - c_ref).max() <= 2e-6 * max(1.0, k ** 0.5) * 4


@pytest.mark.parametrize("m,n,k", [(64, 48, 80), (130, 70, 257), (256, 256, 256)])
def test_openblas_ref_mmult_close_to_oracle(oracle, m, n, k):
    """cuda/REF_MMult.cpp is cblas_sgemm (beta = 0, into a C holding 123.0): different summation order, so the
    pin is the fp64 truth: both within fp32 accumulation noise of it.  The stored OpenBLAS entries are a seeded
    sample of C (all of it for the smallest shape)."""
    a, b = _libs.gen_f32(oracle, m, k, 8), _libs.gen_f32(oracle, k, n, 9)
    idx, c_blas = G[f"blas_{key(m, n, k)}_idx"], G[f"blas_{key(m, n, k)}_val"]
    assert len(idx) == min(m * n, 2048)
    t = _libs.ref_f64(oracle, a, b)
    c_or = _libs.ref_f32_fma(oracle, a, b)
    tol = 4e-7 * k ** 0.5 * np.abs(t).max() + 1e-6
    assert np.abs(c_blas - t.ravel()[idx]).max() <= tol
    assert np.abs(c_or - t).max() <= tol
    assert np.allclose(t, a.astype(np.float64) @ b.astype(np.float64), rtol=0, atol=1e-9)


@pytest.mark.parametrize("m,n,k", [(1, 1, 1), (4, 8, 16), (77, 77, 77), (33, 130, 65)])
def test_int8_ref_bit_exact(oracle, m, n, k):
    a, b = _libs.gen_s8(oracle, m, k, 3), _libs.gen_s8(oracle, k, n, 4)
    assert a.min() >= -127 and b.min() >= -127
    c0 = (np.arange(m * n, dtype=np.int32).reshape(m, n) % 11) - 5
    c1 = c0.copy()
    oracle.oracle_ref_mmult_s8s32(m, n, k, P(a), k, P(b), n, P(c1), n)
    c2 = c0.copy()
    oracle.oracle_ref_mmult_s8s32_fast(m, n, k, P(a), k, P(b), n, P(c2), n)
    assert same_bits(c1, f"i8_{key(m, n, k)}_sha256") and np.array_equal(c1, c2)
    assert np.array_equal(c1 - c0, a.astype(np.int64) @ b.astype(np.int64))


def test_compare_matrices(oracle):
    m, n = 40, 50
    a = _libs.gen_f32(oracle, m, n, 1)
    b = a.copy()
    b[17, 23] += 0.25
    assert oracle.oracle_compare_matrices_f32(m, n, P(a), n, P(b), n) == pytest.approx(float(G["cmp_cuda"]))
    assert float(G["cmp_a64"]) == pytest.approx(0.25)
    ia = np.arange(m * n, dtype=np.int32).reshape(m, n)
    ib = ia.copy()
    ib[3, 4] -= 9
    assert oracle.oracle_compare_matrices_s32(m, n, P(ia), n, P(ib), n) == 9 == int(G["cmp_i8"])
    # the reference's macro abs() hides NaN (SURVEY Appendix B-7); the oracle must not
    b[0, 0] = np.nan
    assert np.isnan(oracle.oracle_compare_matrices_f32(m, n, P(a), n, P(b), n))
