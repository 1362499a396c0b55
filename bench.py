#!/usr/bin/env python
"""bench.py — the driver-facing benchmark of the GEMM hot path (contract: see DESIGN.md §Measurement).

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  the reference's CPU path on the host cores

Workload (BASELINE.json configs[1], headline point): fp32 SGEMM, row-major, M = 4096*N_gpus,
N = K = 4096.  At 1 GPU this is the 4096^3 point the reference quotes (cuda/output_MMult_cuda_12.m:29);
at N GPUs C is sharded by row panels (one 4096-row panel per rank, per-GPU work fixed => "weak"), B lives
on rank 0 and is broadcast over NVLink inside the timed region (SURVEY §8e) by the C-ABI row-panel plan
(b200_gemm_f32_rowpanel).  A "step" is one such GEMM.  value = 2*M*N*K / max-over-ranks time.

After the timed loop every rank checks rows of its C panel against the oracle (verified / max_rel_err);
a failed check fails the run.  The JSON line also carries: c5 (BASELINE configs[4]: 16384^3 strong-scaled
over the same ranks), modes, sweep (GFLOP/s vs N), configs34 (bf16 and int8 records), sustained,
roofline, cpu_baseline, e2e, clocks, gpu_launches.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from
# stdout must carry exactly one JSON line.  NCCL prints its version banner with a C-level printf to
# fd 1 on the first communicator (seen on the 2-GPU box even with NCCL_DEBUG_FILE set), so the real
# stdout is set aside at start-up, fd 1 is pointed at stderr for everything else this process or its
# libraries print, and the JSON line alone is written to the saved descriptor.
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
_JSON_FD = None


def _claim_stdout():
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(obj):
    sys.stdout.flush()
    data = (json.dumps(obj) + "\n").encode()
    fd = _JSON_FD if _JSON_FD is not None else 1
    while data:
        data = data[os.write(fd, data):]


sys.path.insert(0, os.path.join(ROOT, "tests"))

N0 = 4096                     # headline size
N5 = 16384                    # BASELINE configs[4]
METRIC = "SGEMM GFLOP/s (square N=4096 point of the 256..4096 sweep)"
MODE_NAMES = {0: "strict_ffma", 1: "tf32", 2: "bf16x3", 3: "bf16x2", 5: "f16x2_scaled"}
MODE_DTYPE = {0: "f32", 1: "tf32", 2: "bf16x3(split-f32)", 3: "bf16x2(split-f32)", 5: "f16x2(scaled split-f32)"}
MODE_PRODUCTS = {2: 6, 3: 3, 5: 3}                      # tensor-core products per k-step (no roofline credit)
MODE_TOL = {0: 1e-5, 1: 1e-3, 2: 1e-5, 3: 4e-5, 5: 1e-5}  # max |C - C_f64| / max |C_f64| (north_star bar: 1e-3)
DUMP_ROWS = 1024              # --dump-outputs: rows of C written (16 MiB at N = 4096), shared among the ranks


def workload_str(M, N):
    """One string for both arms (the driver compares config.workload of the two lines)."""
    return f"fp32 SGEMM row-major M={M} N=K={N} (BASELINE configs[1], N=4096 point)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, tag=""):
        self.index, self.proc, self.path = index, None, f"/tmp/b200_clocks_{os.getpid()}{tag}.csv"

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "10"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.03)
        self.proc.terminate()
        self.proc.wait()
        self.f.close()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in open(self.path):
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 8:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], c[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = [s for s, p in zip(sm, pw) if p >= 0.5 * max(pw)] or sm
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def cpu_worker(kind, M, N, K, threads, steps, warmup, budget_s, timeout_s):
    """oracle/cpu_ref_worker.py in a fresh process with a clean threading environment (see its header:
    torchrun's OMP_NUM_THREADS=1 + a later openblas_set_num_threads dead-locks OpenBLAS-0.2.20)."""
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "GOTO_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        env.pop(k, None)
    env["OPENBLAS_NUM_THREADS"] = str(threads)
    cmd = [sys.executable, "-B", os.path.join(ROOT, "oracle", "cpu_ref_worker.py"), kind, str(M), str(N), str(K), str(threads),
           str(steps), str(warmup), str(budget_s)]
    try:
        r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout_s)
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        if r.returncode == 0 and line:
            return json.loads(line[-1])
        return {"error": f"rc={r.returncode} {r.stderr[-300:]}"}
    except subprocess.TimeoutExpired:
        return {"error": f"watchdog: no result within {timeout_s} s"}


def run_reference(args):
    """The reference's own CPU implementation of the path: cuda/REF_MMult.cpp (cblas_sgemm of the
    vendored OpenBLAS-0.2.20) from oracle/_ref/libref.so on all host threads (oracle port when libref.so is
    absent).  Rank 0 alone runs it; a step is one full SGEMM of the arm's workload, bounded by a time budget."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cores = os.cpu_count() or 1
    threads = min(cores, 128)                       # OpenBLAS-0.2.20 was built NUM_THREADS=128
    if os.environ.get("B200_REF_THREADS"):          # test hook: oversubscribe a small box like the 128-thread pool of the GPU host
        threads = int(os.environ["B200_REF_THREADS"])
    M = N0 * args.gpus
    warm = max(1, min(args.warmup, 3))
    res = cpu_worker("sgemm", M, N0, N0, threads, args.steps, warm, budget_s=150.0, timeout_s=420)
    if "error" in res and threads > 16:             # belt and braces: retry small before giving up
        res = cpu_worker("sgemm", M, N0, N0, 16, args.steps, 1, budget_s=100.0, timeout_s=300)
    if "error" in res:
        _emit({"impl": "reference", "unavailable": res["error"]})
        return
    gf, dt = res["gflops"], res["ms_per_step"]
    sample = (f"{res['steps_done']} of {args.steps} full SGEMMs M={M} N=K={N0} ({res['what']}), {res['threads']} threads"
              + ("" if res["steps_done"] == args.steps else " (150 s budget reached)"))
    _emit({
        "impl": "reference", "metric": METRIC, "value": gf,
        "unit": "GFLOP/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_str(M, N0)},
        "cpu_baseline": {"value": gf, "unit": "GFLOP/s", "cores": res["threads"], "kind": res["kind"], "sample": sample},
        "e2e": {"value": gf, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def cpu_baseline():
    """Timed beside the GPU number on this box's host cores (rank 0, N=1), each in its own process: the
    reference's OpenBLAS REF_MMult on all cores and on 1 core (BASELINE.md §3), and the naive REF_MMult
    loop nest on a row subset."""
    cores = os.cpu_count() or 1
    threads = min(cores, 128)
    allc = cpu_worker("sgemm", N0, N0, N0, threads, 12, 1, budget_s=8.0, timeout_s=120)
    one = cpu_worker("sgemm", 1024, N0, N0, 1, 3, 1, budget_s=8.0, timeout_s=120)
    naive = cpu_worker("naive", 64, N0, N0, 1, 1, 0, budget_s=30.0, timeout_s=120)
    out = {}
    if "error" not in allc:
        out = {"value": allc["gflops"], "unit": "GFLOP/s", "cores": allc["threads"], "kind": allc["kind"],
               "sample": f"{allc['steps_done']} full 4096^3 calls: {allc['what']}"}
    if "error" not in one:
        out["openblas_1_thread"] = {"value": one["gflops"], "unit": "GFLOP/s", "cores": 1, "kind": one["kind"],
                                    "sample": f"{one['steps_done']} calls on 1024 of 4096 rows (M=1024, N=K=4096): {one['what']}"}
    if "error" not in naive:
        nv = {"value": naive["gflops"], "unit": "GFLOP/s", "cores": 1, "kind": "port",
              "sample": f"{naive['what']} on 64 of 4096 rows, extrapolated"}
        out["naive_ref_mmult"] = nv
        if "value" not in out:
            out.update(nv)
    for name, r in (("all_cores", allc), ("one_thread", one), ("naive", naive)):
        if "error" in r:
            out.setdefault("errors", {})[name] = r["error"]
    return out


def dump_last_step(out_dir, Cm, rank, world):
    """C of the last timed step, as the caller receives it, for output-by-output comparison of two builds.  The
    rows are a fixed seeded sample of the whole M = rows_per_rank * world, so they do not change between runs."""
    import numpy as np
    import torch
    m = Cm.shape[0]
    rows = np.sort(np.random.default_rng(0).choice(m * world, min(DUMP_ROWS, m * world), replace=False))
    mine = rows[(rows >= rank * m) & (rows < (rank + 1) * m)] - rank * m
    torch.cuda.synchronize()
    c = Cm[torch.from_numpy(mine).to(Cm.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "c.npy" if world == 1 else f"c_rank{rank}.npy"), c)


_T0 = time.time()


def _phase(name):
    if os.environ.get("B200_BENCH_TRACE"):
        print(f"[bench +{time.time() - _T0:6.1f}s] {name}", file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--mode", type=int, default=-1, help="fp32 precision mode of the headline (default: library default)")
    ap.add_argument("--no-extras", action="store_true", help="skip sweep / modes / configs34 / cpu_baseline (quick runs)")
    ap.add_argument("--no-c5", action="store_true", help="skip the BASELINE configs[4] record (16384^3)")
    ap.add_argument("--slices", default="", help="K-slices of the B exchange, e.g. '512,1536,2048' (default: the plan's)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help=f"write C of the last timed step as DIR/c.npy (DIR/c_rank<r>.npy with several GPUs): float32, "
                         f"a fixed seeded sample of {DUMP_ROWS} rows of the whole C, in increasing row order")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    _claim_stdout()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    import _libs

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _phase("torch/nccl up")
    g = _libs.load_pkg()            # raises if libb200gemm.so is missing: no fallback
    o = _libs.load_oracle()         # the checker (verification after the timed loops only)
    rowpanel = __import__("importlib").import_module(_libs.PKG + ".rowpanel")
    mode = args.mode if args.mode >= 0 else g.lib.b200_gemm_default_f32_mode()
    comm = rowpanel.nccl_comm_ptr(dist, dev) if world > 1 else 0
    pk = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def verify_rows(A, B, Cm, nrows, tol):
        """This rank's rows of C against the fp64-accumulated oracle product of the SAME device operands
        (B is read back from this rank's buffer, so the exchange is covered), plus bit-agreement of B across
        ranks.  Returns (ok, max_rel_err)."""
        m = A.shape[0]
        rows = torch.unique(torch.linspace(0, m - 1, nrows, device=dev).long())
        a_np, b_np = A[rows].cpu().numpy(), B.cpu().numpy()
        truth = _libs.ref_f64(o, a_np, b_np)
        got = Cm[rows].cpu().numpy()
        err = float(np.abs(got - truth).max() / max(np.abs(truth).max(), 1e-30))
        ok = bool(np.isfinite(got).all()) and err <= tol
        if mode == 0:               # strict: bit-exact against the reference's naive (fused) REF_MMult
            ok = ok and bool(np.array_equal(got, _libs.ref_f32_fma(o, a_np, b_np)))
        if world > 1:
            h = B.view(torch.int32).sum(dtype=torch.int64).reshape(1)
            hs = [torch.zeros_like(h) for _ in range(world)]
            dist.all_gather(hs, h)
            ok = ok and all(int(x.item()) == int(hs[0].item()) for x in hs)
        err_all = allmax(err)
        ok_all = allmax(0.0 if ok else 1.0) == 0.0
        return ok_all, err_all

    # ================= headline: M = 4096 * world, N = K = 4096 (weak) ==============================
    K = N = N0
    Mloc = N0
    R = 3                           # rotating operand sets: consecutive steps never see a warm L2
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    sets = []
    for _ in range(R):
        A = torch.rand((Mloc, K), device=dev, generator=gen) * 2 - 1
        B = torch.rand((K, N), device=dev, generator=gen) * 2 - 1 if rank == 0 else torch.full((K, N), float("nan"), device=dev)
        Cm = torch.empty((Mloc, N), device=dev)
        sets.append((A, B, Cm))
    plan = None
    if world > 1:
        sl = None
        if args.slices:
            v = [int(x) for x in args.slices.split(",")]
            e = [0]
            for x in v:
                e.append(e[-1] + x)
            sl = list(zip(e[:-1], e[1:]))
        plan = rowpanel.RowPanelPlan(g, comm, Mloc, N, K, mode, sl)

    def step(i):
        A, B, Cm = sets[i % R]
        if plan is None:
            g.gemm_f32(A, B, out=Cm, mode=mode)
        else:
            plan.run(A, B, Cm)      # b200_gemm_f32_rowpanel: ncclBroadcast of B's K-slices pipelined with the K-sliced GEMM

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()              # nvidia-smi needs ~0.1 s to start: launch it ahead of the warm-up
    for i in range(max(args.warmup, 3)):
        step(i)
    if rank == 0:
        time.sleep(0.15)             # let the sampler come up; BEFORE the barrier so all ranks start together
    barrier()
    l0 = g.launch_count()
    g.lib.b200_gemm_debug_kernel_timing(1)      # event pair around every dominant-kernel launch, same stream
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    barrier()
    ms = allmax(e0.elapsed_time(e1)) / args.steps
    launches = g.launch_count() - l0
    kern_ms_sum, kern_launches = g.kernel_time_ms()
    g.lib.b200_gemm_debug_kernel_timing(0)
    clocks = sampler.stop() if rank == 0 else None
    flops_step = 2.0 * (Mloc * world) * N * K
    value = flops_step / (ms * 1e-3) / 1e9
    kernel_name = g.last_kernel()
    _phase("timed region done")
    if args.dump_outputs:            # before anything below overwrites the C buffers
        dump_last_step(args.dump_outputs, sets[(args.steps - 1) % R][2], rank, world)

    # ---- verification of the timed path (every rank, after the timed loop) --------------------------
    step(0)
    torch.cuda.synchronize()
    verified, max_rel_err = verify_rows(*sets[0], 64, MODE_TOL.get(mode, 1e-5))
    _phase("verified")

    # ---- sustained: the same step back to back for >= 2 s (the part sits at its power cap) ---------
    sustained = None
    if not args.no_extras:
        s_sampler = ClockSampler(local, "s")
        if rank == 0:
            s_sampler.start()
        n_sus = max(200, int(2200.0 / ms))
        barrier()
        e0.record()
        for i in range(n_sus):
            step(i)
        e1.record()
        barrier()
        s_ms = allmax(e0.elapsed_time(e1)) / n_sus
        s_clk = s_sampler.stop() if rank == 0 else None
        sustained = {"gflops": flops_step / (s_ms * 1e-3) / 1e9, "ms_per_step": s_ms, "steps": n_sus,
                     "seconds": s_ms * n_sus / 1e3, "clocks": s_clk}
        _phase("sustained done")

    # ================= c5: BASELINE configs[4], M = N = K = 16384 sharded over the same ranks (strong) =====
    c5 = None
    if not args.no_c5:
        del sets[1:]                                        # headline sets 1.. are not needed any more
        torch.cuda.empty_cache()
        M5 = N5 // world
        A5 = torch.empty((M5, N5), device=dev).uniform_(-1, 1, generator=gen)
        B5 = torch.empty((N5, N5), device=dev)
        if rank == 0:
            B5.uniform_(-1, 1, generator=gen)
        else:
            B5.fill_(float("nan"))
        C5 = torch.empty((M5, N5), device=dev)
        plan5 = rowpanel.RowPanelPlan(g, comm, M5, N5, N5, mode) if world > 1 else None

        def step5():
            if plan5 is None:
                g.gemm_f32(A5, B5, out=C5, mode=mode)
            else:
                plan5.run(A5, B5, C5)

        c_sampler = ClockSampler(local, "c5")
        if rank == 0:
            c_sampler.start()
        step5()
        step5()
        barrier()
        c5_steps = 4
        e0.record()
        for _ in range(c5_steps):
            step5()
        e1.record()
        barrier()
        c5_ms = allmax(e0.elapsed_time(e1)) / c5_steps
        c5_clk = c_sampler.stop() if rank == 0 else None
        ok5, err5 = verify_rows(A5, B5, C5, 8, MODE_TOL.get(mode, 1e-5))
        gf5 = 2.0 * N5 ** 3 / (c5_ms * 1e-3) / 1e9
        c5 = {"workload": f"fp32 SGEMM row-major M=N=K={N5} (BASELINE configs[4]), C row-panel sharded over {world} rank(s), "
                          "B broadcast from rank 0 inside every step (strong scaling)",
              "gflops": gf5, "ms_per_step": c5_ms, "steps": c5_steps, "warmup": 2, "scaling": "strong",
              "frac_of_n_x_bf16_burst": gf5 / 1e3 / (world * pk["bf16_tflops"]),
              "frac_of_n_x_bf16_sustained": gf5 / 1e3 / (world * pk["bf16_tflops_sustained"]) if pk["bf16_tflops_sustained"] else None,
              "k_slices": [k1 - k0 for k0, k1 in plan5.chunks] if plan5 else [N5],
              "kernel": g.last_kernel(), "verified": ok5, "max_rel_err": err5, "rows_checked_per_rank": 8, "clocks": c5_clk}
        if plan5 is not None:
            plan5.close()
        del A5, B5, C5
        torch.cuda.empty_cache()
        _phase("c5 done")

    # ================= e2e: the host-pointer plug-in call (9-arg MY_MMult contract, C += A*B) ==========
    # world == 1: b200_gemm_f32_host.  world > 1: b200_gemm_f32_rowpanel_host — the SAME sharded product with
    # host operands: B host->device on rank 0, broadcast, every rank stages its own A/C panel.
    e2e_steps = max(3, min(args.steps, 8))
    hA = torch.empty((Mloc, K), dtype=torch.float32).pin_memory().uniform_(-1, 1)
    hB = torch.empty((K, N), dtype=torch.float32).pin_memory().uniform_(-1, 1) if rank == 0 else None
    hC = torch.zeros((Mloc, N), dtype=torch.float32).pin_memory()

    def e2e_step():
        if plan is None:
            rc = g.lib.b200_gemm_f32_host(Mloc, N, K, hA.data_ptr(), K, hB.data_ptr(), N, hC.data_ptr(), N, mode)
            assert rc == 0, rc
        else:
            plan.run_host(hA, hB, hC)
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()                      # synchronous: returns when C is back in host memory
    barrier()
    e2e_ms = allmax((time.perf_counter() - t0) * 1e3 / e2e_steps)
    e2e = {"value": flops_step / (e2e_ms * 1e-3) / 1e9, "unit": "GFLOP/s",
           "h2d_bytes_per_step": (Mloc * K + Mloc * N) * 4 * world + K * N * 4, "d2h_bytes_per_step": Mloc * N * 4 * world,
           "ms_per_step": e2e_ms,
           "api": ("b200_gemm_f32_host (9-arg MY_MMult contract, pinned host buffers)" if plan is None else
                   "b200_gemm_f32_rowpanel_host (9-arg contract, row-panel sharded: B uploaded on rank 0 and broadcast, "
                   "A/C panels staged per rank; bytes are the whole job's)")}
    # e2e result check on rank 0's panel: C was zero, then (1 + e2e_steps) x (C += A*B)
    rows = torch.arange(0, Mloc, 257)[:16]
    hBd = sets[0][1] if plan is None else None
    if rank == 0:
        t = _libs.ref_f64(o, hA[rows].numpy(), hB.numpy()) * (1 + e2e_steps)
        e2e["max_rel_err"] = float(np.abs(hC[rows].numpy() - t).max() / np.abs(t).max())
        e2e["verified"] = bool(e2e["max_rel_err"] <= 4 * MODE_TOL.get(mode, 1e-5))
    del hBd
    _phase("e2e done")

    if plan is not None:
        plan.close()
    if world > 1:
        dist.destroy_process_group()        # every rank, right after the last collective
    if not (verified and (c5 is None or c5["verified"])):
        if rank == 0:
            print(f"VERIFICATION FAILED: headline {verified} ({max_rel_err}), c5 {c5 and (c5['verified'], c5['max_rel_err'])}",
                  file=sys.stderr)
        sys.exit(3)
    if rank != 0:
        return

    out = {
        "metric": METRIC, "value": value, "unit": "GFLOP/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": MODE_DTYPE.get(mode, str(mode)), "data": "synthetic",
        "verified": verified, "max_rel_err": max_rel_err,
        "config": {"workload": workload_str(Mloc * world, N),
                   "sharding": (f"C row-panel sharded over {world} ranks; B broadcast from rank 0 inside every step as K-slices "
                                f"{[k1 - k0 for k0, k1 in plan.chunks]} (ncclBroadcast, in place) pipelined with the K-sliced GEMM "
                                "through the C ABI (b200_gemm_f32_rowpanel)") if world > 1 else "single GPU (b200_gemm_f32)",
                   "precision_mode": MODE_NAMES.get(mode, str(mode)), "kernel": kernel_name,
                   "l2": f"{R} rotating input/output sets of {3 * N0 * N0 * 4 / 1e6:.0f} MB each (> 126 MB L2 between reuses)",
                   "inputs": "uniform(-1,1), row-major, lda=k ldb=n ldc=n (cuda/test_MMult.cpp:62)",
                   "verification": "64 rows of every rank's C panel vs the fp64-accumulated oracle after the timed loop "
                                   f"(tolerance {MODE_TOL.get(mode, 1e-5)} * max|C|), B bit-compared across ranks"},
        "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e,
        "published_reference": {"MMult_cuda_12 @4096 on RTX 3090": 21410.87, "note": "other hardware; BASELINE.json.published is {}"},
    }
    if sustained:
        out["sustained"] = sustained
    if c5:
        out["c5"] = c5
    # roofline of the dominant kernel: its own launch durations (CUDA events on the launching stream,
    # recorded inside the timed region); algorithmic flops = 2*M*N*K, no credit for the split products
    if world == 1:
        kern_ms = kern_ms_sum / max(kern_launches, 1)
        achieved = 2.0 * N0 ** 3 / (kern_ms * 1e-3) / 1e12
        prods = MODE_PRODUCTS.get(mode, 1)
        out["roofline"] = {"bound": "tensor", "achieved": achieved, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                           "frac": achieved / pk["bf16_tflops"], "traffic": None,
                           "kernel_ms": kern_ms, "kernel_launches_timed": kern_launches,
                           "kernel_share_of_step": kern_ms / ms,
                           "tensor_pipe_flops_per_launch": 2.0 * N0 ** 3 * prods,
                           "tensor_pipe_frac": achieved * prods / ({1: 0.5}.get(mode, 1.0) * pk["bf16_tflops"]),
                           "peak_source": pk["source"] + ", burst bf16; sustained " + str(pk["bf16_tflops_sustained"]),
                           "frac_of_sustained": achieved / pk["bf16_tflops_sustained"] if pk["bf16_tflops_sustained"] else None,
                           "algorithmic_flops_per_launch": 2.0 * N0 ** 3,
                           "algorithmic_bytes_per_launch": 3 * N0 * N0 * 4,
                           "achieved_hbm_gbs": 3 * N0 * N0 * 4 / (ms * 1e-3) / 1e9,
                           "kernel": kernel_name}
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                # bytes per launch (dram read+write) of this kernel at this size from the committed
                # `ncu --set full` capture (profiles/, tools/summarize_ncu.py); null if not captured
                tj = json.load(open(tp))
                out["roofline"]["traffic"] = tj.get(f"{kernel_name}@{N0}")
                out["roofline"]["traffic_source"] = tj.get("_source", "profiles/ ncu capture (not measured in this run)")
            except Exception:
                pass

    if not args.no_extras and world == 1:
        A, B, Cm = sets[0]
        # ---- every precision mode at the headline size, with its error against the oracle --------
        rows = torch.arange(0, N0, 67, device=dev)[:48]
        a_np, b_np = A[rows].cpu().numpy(), B.cpu().numpy()
        truth = _libs.ref_f64(o, a_np, b_np)
        ref_naive = _libs.ref_f32_fma(o, a_np, b_np)
        A2, B2 = torch.rand_like(A) * 2 - 1, torch.rand_like(B) * 2 - 1
        C2 = torch.empty_like(Cm)
        rot = [(A, B, Cm), (A2, B2, C2)]
        modes = {}
        for md, name in MODE_NAMES.items():
            try:
                g.gemm_f32(A, B, out=Cm, mode=md)
            except g.B200GemmError:
                continue
            kn = g.last_kernel()
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(10):
                a_, b_, c_ = rot[i % 2]
                g.gemm_f32(a_, b_, out=c_, mode=md)
            e.record()
            torch.cuda.synchronize()
            t_ms = s.elapsed_time(e) / 10
            g.gemm_f32(A, B, out=Cm, mode=md)
            got = Cm[rows].cpu().numpy()
            modes[name] = {"gflops": 2.0 * N0 ** 3 / t_ms / 1e6, "ms": t_ms, "kernel": kn,
                           "max_abs_err_vs_f64": float(np.abs(got - truth).max()),
                           "max_rel_err_vs_maxabs": float(np.abs(got - truth).max() / np.abs(truth).max()),
                           "max_abs_diff_vs_REF_MMult_naive": float(np.abs(got - ref_naive).max()),
                           "bit_exact_vs_REF_MMult_naive": bool(np.array_equal(got, ref_naive)),
                           "frac_of_bf16_peak": 2.0 * N0 ** 3 / t_ms / 1e9 / pk["bf16_tflops"]}
        out["modes"] = modes
        fp32_peak = 2 * 128 * torch.cuda.get_device_properties(dev).multi_processor_count * (clocks["sm_max_mhz"] or 1965.0) * 1e6 / 1e12
        out["fp32_cuda_core_peak_tflops"] = fp32_peak
        if "strict_ffma" in modes:
            modes["strict_ffma"]["frac_of_fp32_cuda_core_peak"] = modes["strict_ffma"]["gflops"] / 1e3 / fp32_peak
        del A2, B2, C2, rot
        _phase("modes done")

        # ---- BASELINE configs[2] (bf16) and configs[3] (int8): driver-run records -------------------
        def timed_kernel(fn, iters):
            for i in range(3):
                fn(i)
            torch.cuda.synchronize()
            g.lib.b200_gemm_debug_kernel_timing(1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(iters):
                fn(i)
            e.record()
            torch.cuda.synchronize()
            ksum, kn = g.kernel_time_ms()
            g.lib.b200_gemm_debug_kernel_timing(0)
            return s.elapsed_time(e) / iters, ksum / max(kn, 1)

        rec34 = []
        for n in (4096, 8192):
            Rn = 3 if n == 4096 else 2
            ops = [(((torch.rand((n, n), device=dev) * 2 - 1)).bfloat16(), ((torch.rand((n, n), device=dev) * 2 - 1)).bfloat16())
                   for _ in range(Rn)]
            rws = torch.arange(0, n, 131, device=dev)[:24]
            tr = _libs.ref_f64(o, ops[0][0][rws].float().cpu().numpy(), ops[0][1].float().cpu().numpy())
            for od, oname, s_out in ((torch.bfloat16, "bf16->bf16", 2), (torch.float32, "bf16->fp32", 4)):
                outs = [torch.empty((n, n), device=dev, dtype=od) for _ in range(Rn)]
                t_ms, k_ms = timed_kernel(lambda i: g.gemm_bf16(ops[i % Rn][0], ops[i % Rn][1], out=outs[i % Rn]), 20)
                g.gemm_bf16(ops[0][0], ops[0][1], out=outs[0])
                got = outs[0][rws].float().cpu().numpy()
                tf = 2.0 * n ** 3 / k_ms / 1e9
                rec34.append({"config": f"{oname} N={n} (BASELINE configs[2])", "kernel": g.last_kernel(), "ms_per_call": t_ms,
                              "kernel_ms": k_ms, "tflops": tf, "frac_of_bf16_burst": tf / pk["bf16_tflops"],
                              "frac_of_bf16_sustained": tf / pk["bf16_tflops_sustained"] if pk["bf16_tflops_sustained"] else None,
                              "algorithmic_bytes": 2 * n * n * 2 + n * n * s_out,
                              "achieved_hbm_gbs": (2 * n * n * 2 + n * n * s_out) / k_ms / 1e6,
                              "traffic": None,
                              "max_rel_err_vs_f64": float(np.abs(got - tr).max() / np.abs(tr).max())})
                del outs
            del ops
        for n in (4096, 8192):
            Rn = 3 if n == 4096 else 2
            ops = [(torch.randint(-127, 128, (n, n), device=dev, dtype=torch.int8), torch.randint(-127, 128, (n, n), device=dev, dtype=torch.int8))
                   for _ in range(Rn)]
            outs = [torch.empty((n, n), device=dev, dtype=torch.int32) for _ in range(Rn)]
            t_ms, k_ms = timed_kernel(lambda i: g.gemm_s8s32(ops[i % Rn][0], ops[i % Rn][1], out=outs[i % Rn]), 20)
            g.gemm_s8s32(ops[0][0], ops[0][1], out=outs[0])
            rws = torch.arange(0, n, 131, device=dev)[:24]
            exact = bool(np.array_equal(outs[0][rws].cpu().numpy(), _libs.ref_s8(o, ops[0][0][rws].cpu().numpy(), ops[0][1].cpu().numpy())))
            tops = 2.0 * n ** 3 / k_ms / 1e9
            rec34.append({"config": f"int8->int32 N={n} (BASELINE configs[3], chgemm semantics)", "kernel": g.last_kernel(),
                          "ms_per_call": t_ms, "kernel_ms": k_ms, "tops": tops,
                          "frac_of_2x_bf16_burst": tops / (2 * pk["bf16_tflops"]),
                          "algorithmic_bytes": 2 * n * n + 4 * n * n, "achieved_hbm_gbs": (2 * n * n + 4 * n * n) / k_ms / 1e6,
                          "traffic": None, "bit_exact_vs_REF_MMult": exact})
            del ops, outs
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            for r in rec34:
                nn = 4096 if "N=4096" in r["config"] else 8192
                r["traffic"] = tj.get(f"{r['kernel']}@{nn}")
        except Exception:
            pass
        out["configs34"] = rec34
        torch.cuda.empty_cache()
        _phase("configs 3/4 done")

        # ---- GFLOP/s-vs-N curve in the reference's output_*.m format ------------------------------
        sweep, sweep_kernels = [], []
        sweep_mode = args.mode if args.mode >= 0 else g.F32_AUTO    # the library default, size heuristic included
        for n in range(256, 4097, 256):
            a = torch.rand((n, n), device=dev) * 2 - 1
            b = torch.rand((n, n), device=dev) * 2 - 1
            c = torch.empty((n, n), device=dev)
            for _ in range(3):
                g.gemm_f32(a, b, out=c, mode=sweep_mode)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(20):            # NREPEATS = 20 back-to-back launches (cuda/parameters.h:24)
                g.gemm_f32(a, b, out=c, mode=sweep_mode)
            e.record()
            torch.cuda.synchronize()
            sweep.append([n, round(2.0 * n ** 3 / (s.elapsed_time(e) / 20) / 1e6, 2)])
            sweep_kernels.append(g.last_kernel())
        out["sweep"] = sweep
        out["sweep_kernels"] = sweep_kernels       # AUTO takes the single-launch strict kernel up to ~512^3
        out["cpu_baseline"] = cpu_baseline()
    _phase("extras done")
    _emit(out)


if __name__ == "__main__":
    main()
