"""Test-side loaders: the CPU oracle (oracle/liboracle.so), the compiled reference
(oracle/_ref/libref.so, optional) and the product package.  Only tests/, smoke() and bench.py's
cpu_baseline / --impl reference legs may import this."""
import ctypes as C
import hashlib
import importlib
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libref.so")
PKG = "how-to-optimize-gemm_b200"


def P(a):
    return a.ctypes.data_as(C.c_void_p)


def sha256(a):
    """SHA-256 of an array's bytes as a uint8[32]: pins a bit-exact result of any size in 32 bytes."""
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def seed_unseeded_drand48():
    """Puts drand48 back in glibc's start state (X = 0), the stream a program that never seeds it draws
    (cuda/test_MMult.cpp calls random_matrix without srand48); srand48 cannot reach that state."""
    C.CDLL(None).seed48((C.c_ushort * 3)(0, 0, 0))


def load_oracle():
    if not os.path.exists(ORACLE_SO):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"])
    o = C.CDLL(ORACLE_SO)
    o.oracle_seed.argtypes = [C.c_long]
    o.oracle_compare_matrices_f32.restype = C.c_float
    o.oracle_max_abs_f32.restype = C.c_float
    o.oracle_max_err_vs_f64.restype = C.c_double
    o.oracle_f32_to_bf16.restype = C.c_uint16
    o.oracle_f32_to_bf16.argtypes = [C.c_float]
    o.oracle_bf16_to_f32.restype = C.c_float
    o.oracle_bf16_to_f32.argtypes = [C.c_uint16]
    o.oracle_random_int8_uniform.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_uint64]
    o.oracle_round_to_bf16_inplace.argtypes = [C.c_size_t, C.c_void_p]
    return o


def have_ref():
    return os.path.exists(REF_SO)


def load_ref():
    r = C.CDLL(REF_SO)
    # C++-mangled entry points of the reference's own sources (see oracle/Makefile)
    r.cuda_REF_MMult = r._Z9REF_MMultiiiPfiS_iS_i            # cuda/REF_MMult.cpp:9 (cblas_sgemm)
    r.cuda_random_matrix = r._Z13random_matrixiiPfi          # cuda/random_matrix.cpp:6
    r.cuda_compare_matrices = r._Z16compare_matricesiiPfiS_i  # cuda/compare_matrices.cpp:7
    r.cuda_compare_matrices.restype = C.c_float
    r.a64_REF_MMult = r._Z9REF_MMultiiiPfS_S_                # aarch64/REF_MMult.cpp:18
    r.a64_random_matrix = r._Z13random_matrixiiPf            # aarch64/random_matrix.cpp:3
    r.a64_compare_matrices = r._Z16compare_matricesiiPfS_    # aarch64/compare_matrices.cpp:5
    r.a64_compare_matrices.restype = C.c_float
    r.a64_MY_MMult = r._Z8MY_MMultiiiPfiS_iS_i               # aarch64/MMult0.cpp:3
    r.i8_REF_MMult = r.REF_MMult                              # aarch64-int8/REF_MMult.c:10
    r.i8_random_matrix = r.random_int8_matrix                 # aarch64-int8/random_matrix.c:9
    r.i8_compare_matrices = r.compare_matrices                # aarch64-int8/compare_matrices.c:8
    r.i8_compare_matrices.restype = C.c_int32
    r.openblas_set_num_threads.argtypes = [C.c_int]
    return r


def load_pkg():
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    return importlib.import_module(PKG)


# ---- oracle-backed numpy conveniences -----------------------------------------------------------
def gen_f32(o, m, n, seed):
    """uniform(-1,1) exactly as cuda/random_matrix.cpp fills an m x n buffer called with lda=m
    (cuda/test_MMult.cpp:77), returned as the ROW-MAJOR m x n view the harness then uses."""
    a = np.zeros(m * n, np.float32)
    o.oracle_seed(seed)
    o.oracle_random_matrix_cuda(m, n, P(a), m)
    return a.reshape(m, n)


def ref_f32_fma(o, a, b, c0=None):
    m, k = a.shape
    n = b.shape[1]
    c = np.zeros((m, n), np.float32) if c0 is None else c0.copy()
    o.oracle_ref_mmult_f32_fma_fast(m, n, k, P(a), a.strides[0] // 4, P(b), b.strides[0] // 4, P(c), n)
    return c


def ref_f64(o, a, b):
    m, k = a.shape
    n = b.shape[1]
    c = np.zeros((m, n), np.float64)
    o.oracle_ref_mmult_f64acc(m, n, k, P(a), a.strides[0] // 4, P(b), b.strides[0] // 4, P(c), n)
    return c


def ref_s8(o, a, b):
    m, k = a.shape
    n = b.shape[1]
    c = np.zeros((m, n), np.int32)
    o.oracle_ref_mmult_s8s32_fast(m, n, k, P(a), a.strides[0], P(b), b.strides[0], P(c), n)
    return c


def requant_s8(o, c32, scales, bias=None):
    """oracle_requant_s32_to_s8 over an int32 matrix (aarch64-int8/int8kernel_m4.S:386-426)."""
    c32 = np.ascontiguousarray(c32, np.int32)
    m, n = c32.shape
    scales = np.ascontiguousarray(scales, np.float32)
    out = np.zeros((m, n), np.int8)
    bp = None
    if bias is not None:
        bias = np.ascontiguousarray(bias, np.float32)
        bp = P(bias)
    o.oracle_requant_s32_to_s8(m, n, P(c32), n, P(scales), bp, P(out), n)
    return out


def gen_s8(o, m, n, seed):
    a = np.zeros((m, n), np.int8)
    o.oracle_random_int8_uniform(m, n, P(a), n, seed)
    return a


def round_bf16(o, a):
    a = np.ascontiguousarray(a, np.float32).copy()
    o.oracle_round_to_bf16_inplace(a.size, P(a))
    return a
