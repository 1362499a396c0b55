"""The reference's harnesses, replayed through the entry points the MY_MMult shims call (shim/*.cpp), against
what the reference computed: tests/golden/reference_harness.npz (tests/golden/make_golden.py) holds REF_MMult's
results for the harnesses' own inputs, which the oracle regenerates bit for bit.  This is the drop-in claim of
SURVEY §8b checked end to end on the GPU.

The fp32 harnesses run in a fresh process each, as the harness binaries did, so that B200GEMM_F32_MODE picks
the library's default mode exactly as it does for a program linked against the shim:
    python tests/test_ref_harness_gpu.py cuda|a64
prints one JSON line of rows [N, GFLOP/s, max|diff|, inputs_match, finite]."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import _libs
from _libs import P

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_harness.npz"))
NREPEATS = 20                   # cuda/parameters.h as the harness was built


def cuda_harness():
    """cuda/test_MMult.cpp:55-129: per size, A, B and a C it then zeroes from one never-seeded drand48 stream,
    NREPEATS launches of MY_MMult(handle, ...) (= b200_gemm_f32, AUTO, legacy default stream), then max|C - cref|
    over the stored sample of REF_MMult (OpenBLAS) entries."""
    import torch
    o, g = _libs.load_oracle(), _libs.load_pkg()
    assert torch.cuda.get_device_capability(0)[0] == 10, torch.cuda.get_device_name(0)
    _libs.seed_unseeded_drand48()
    rows = []
    for p in (int(x) for x in G["cuda_sizes"]):
        a, b, cold = (np.zeros(p * p, np.float32) for _ in range(3))
        o.oracle_random_matrix_cuda(p, p, P(a), p)
        o.oracle_random_matrix_cuda(p, p, P(b), p)
        o.oracle_random_matrix_cuda(p, p, P(cold), p)
        same = (np.array_equal(_libs.sha256(a), G[f"cuda_{p}_a_sha256"])
                and np.array_equal(_libs.sha256(b), G[f"cuda_{p}_b_sha256"]))
        dA, dB = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        dC = torch.empty(p * p, device="cuda")
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(NREPEATS):
            g.MY_MMult_cuda(None, p, p, p, dA.data_ptr(), p, dB.data_ptr(), p, dC.data_ptr(), p)
        e.record()
        e.synchronize()
        c = dC.cpu().numpy()
        gflops = 2.0 * p ** 3 / (s.elapsed_time(e) / NREPEATS) / 1e6
        diff = float(np.abs(c[G[f"cuda_{p}_idx"]].astype(np.float64) - G[f"cuda_{p}_cref"]).max())
        rows.append([p, gflops, diff, bool(same), bool(np.isfinite(c).all())])
    return rows


def a64_harness():
    """aarch64/test_MMult.cpp at 256^3: inputs all 1.0f, NREPEATS = 10 of (C = 0; MY_MMult(m, n, k, a, ...)),
    the 9-argument host form (= b200_gemm_f32_host, AUTO, C += A*B), then max|C - cref|."""
    o, g = _libs.load_oracle(), _libs.load_pkg()
    p = 256
    a, b = np.zeros((p, p), np.float32), np.zeros((p, p), np.float32)
    o.oracle_random_matrix_ones(p, p, P(a))
    o.oracle_random_matrix_ones(p, p, P(b))
    c = np.zeros((p, p), np.float32)
    for _ in range(10):
        c[:] = 0
        g.MY_MMult(p, p, p, a, p, b, p, c, p)
    return [[p, 0.0, float(np.abs(c - G["a64_256_cref"]).max()), True, bool(np.isfinite(c).all())]]


def replay(kind, env):
    r = subprocess.run([sys.executable, os.path.abspath(__file__), kind], capture_output=True, text=True,
                       timeout=600, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    return json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("[")][-1])


@pytest.mark.parametrize("mode", ["default", "0", "1", "2", "5"])   # shim default (AUTO -> F16X2), STRICT, TF32, BF16X3, F16X2
def test_cuda_harness_unmodified(mode):
    """cuda/test_MMult.cpp + REF_MMult.cpp (OpenBLAS) + compare_matrices.cpp, N = 256..4096 step 256.  "default" is
    what bench.py measures: the shim passes B200_F32_AUTO and no environment override is set."""
    env = {k: v for k, v in os.environ.items() if k != "B200GEMM_F32_MODE"}
    if mode != "default":
        env["B200GEMM_F32_MODE"] = mode
    rs = replay("cuda", env)
    assert [x[0] for x in rs] == list(range(256, 4097, 256))
    for n, gflops, diff, same_inputs, finite in rs:
        assert same_inputs and finite, n
        assert gflops > 0
        # gate: cuda/test_MMult.cpp:124 (0.5); the fp32-class modes sit at OpenBLAS's own summation-order noise
        assert diff < (0.5 if mode == "1" else 2e-3), (n, diff)


def test_aarch64_harness_config1():
    """aarch64/test_MMult.cpp at 256^3 through the 9-arg host shim (C += A*B), diff must be 0."""
    rs = replay("a64", dict(os.environ, B200GEMM_F32_MODE="0"))
    assert len(rs) == 1 and rs[0][0] == 256 and rs[0][2] == 0.0 and rs[0][4]


@pytest.mark.parametrize("mnk", [None, ("64", "64", "64"), ("33", "130", "65"), ("512", "768", "1024")])
def test_int8_harness(gemm, oracle, mnk):
    """aarch64-int8/test_MMult.c (no arguments: 77^3): ramp inputs, C = 0, MY_MMult (= b200_gemm_s8s32_host); it
    exits silently (no row printed) on ANY mismatch with REF_MMult (test_MMult.c:108-111)."""
    m, n, k = (int(x) for x in (mnk or (77, 77, 77)))
    a, b = np.zeros((m, k), np.int8), np.zeros((k, n), np.int8)
    oracle.oracle_random_int8_ramp(m, k, P(a), k)
    oracle.oracle_random_int8_ramp(k, n, P(b), n)
    c = np.zeros((m, n), np.int32)
    gemm.MY_MMult_int8(m, n, k, a, k, b, n, c, n)
    assert np.array_equal(_libs.sha256(c), G[f"i8_{m}x{n}x{k}_cref_sha256"])


if __name__ == "__main__":
    print(json.dumps({"cuda": cuda_harness, "a64": a64_harness}[sys.argv[1]]()), flush=True)
