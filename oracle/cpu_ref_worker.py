#!/usr/bin/env python
"""CPU timing worker for bench.py's reference arm and cpu_baseline leg (test infrastructure, like the
rest of oracle/: only bench.py's `--impl reference` / cpu_baseline legs and tests/ may run it).

Times the reference's own CPU implementation of the path on this box's host cores in a FRESH process:
cuda/REF_MMult.cpp -> cblas_sgemm of the vendored OpenBLAS-0.2.20 (oracle/_ref/libref.so, kind
"reference"), else the oracle port of the naive loop nest (kind "port").

Why a separate process: OpenBLAS-0.2.20 sizes its thread pool when the library is loaded, from
OPENBLAS_NUM_THREADS / OMP_NUM_THREADS.  torchrun exports OMP_NUM_THREADS=1 into every rank, and growing
the pool afterwards with openblas_set_num_threads(128) dead-locks (reproduced here: round-1 SCALE run,
rc 124 at N=2/4, SIGSEGV at N=8).  So the parent strips OMP_NUM_THREADS, sets OPENBLAS_NUM_THREADS and
never resizes the pool; a watchdog (the parent's subprocess timeout) bounds the run.

usage: cpu_ref_worker.py KIND M N K THREADS STEPS WARMUP [BUDGET_S]
  KIND = sgemm  : cblas_sgemm via cuda/REF_MMult.cpp (falls back to the port when libref.so is absent)
         naive  : the naive REF_MMult loop nest (aarch64/REF_MMult.cpp:18-28) on M rows, 1 thread
prints one JSON object on stdout.
"""
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))


def main():
    kind, M, N, K, threads, steps, warmup = sys.argv[1], *[int(x) for x in sys.argv[2:8]]
    budget = float(sys.argv[8]) if len(sys.argv) > 8 else 1e9
    import numpy as np
    import _libs
    rng = np.random.default_rng(0)
    a = rng.uniform(-1, 1, (M, K)).astype(np.float32)
    b = rng.uniform(-1, 1, (K, N)).astype(np.float32)
    c = np.zeros((M, N), np.float32)
    if kind == "sgemm" and _libs.have_ref():
        r = _libs.load_ref()          # pool size comes from OPENBLAS_NUM_THREADS (set by the parent)
        fn = lambda: r.cuda_REF_MMult(M, N, K, _libs.P(a), K, _libs.P(b), N, _libs.P(c), N)
        out_kind, what = "reference", "cuda/REF_MMult.cpp -> cblas_sgemm (vendored OpenBLAS-0.2.20, HASWELL kernels)"
    elif kind == "sgemm":
        o = _libs.load_oracle()
        o.oracle_set_threads(threads)
        def fn():
            c[:] = 0
            o.oracle_ref_mmult_f32_fma_fast(M, N, K, _libs.P(a), K, _libs.P(b), N, _libs.P(c), N)
        out_kind, what = "port", "oracle_ref_mmult_f32_fma_fast (naive REF_MMult arithmetic, row-parallel)"
    else:
        o = _libs.load_oracle()
        threads = 1
        def fn():
            c[:] = 0
            o.oracle_ref_mmult_f32_fma(M, N, K, _libs.P(a), K, _libs.P(b), N, _libs.P(c), N)
        out_kind, what = "port", "naive REF_MMult loop nest (aarch64/REF_MMult.cpp:18-28)"
    for _ in range(warmup):
        fn()
    done, t0 = 0, time.perf_counter()
    while done < steps:
        fn()
        done += 1
        if time.perf_counter() - t0 > budget:
            break
    dt = (time.perf_counter() - t0) / done
    print(json.dumps({"ms_per_step": dt * 1e3, "gflops": 2.0 * M * N * K / dt / 1e9, "threads": threads, "steps_done": done,
                      "kind": out_kind, "what": what, "M": M, "N": N, "K": K}))


if __name__ == "__main__":
    main()
