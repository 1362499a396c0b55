"""The C-ABI row-panel plan on hardware (-m gpu).

  * one rank, comm = NULL: the whole K-sliced schedule (A split once, every slice of B split and multiplied
    as it "lands", products accumulated) without the exchange — runs on the driver's 1-GPU box;
  * two NCCL ranks (skipped with < 2 GPUs): the full path, the complete C of both ranks against the oracle,
    B bit-identical on both ranks afterwards, device and host variants, every precision mode.
"""
import os
import socket
import sys

import numpy as np
import pytest

import _libs

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TOL = {0: 0.0, 1: 1e-3, 2: 1e-5, 3: 4e-5, 5: 1e-5}


def _rowpanel():
    import importlib
    sys.path.insert(0, _libs.ROOT)
    return importlib.import_module(_libs.PKG + ".rowpanel")


def rel(c, t):
    return float(np.abs(c.astype(np.float64) - t).max() / max(np.abs(t).max(), 1e-30))


@pytest.mark.parametrize("mode", [5, 2, 0, 1])
@pytest.mark.parametrize("m,n,k,slices", [(300, 520, 1280, None), (1000, 1104, 2048, [(0, 256), (256, 1024), (1024, 2048)]),
                                          (77, 96, 80, [(0, 16), (16, 80)]), (2304, 2304, 1024, [(0, 128), (128, 1024)])])
def test_rowpanel_single_rank_k_sliced(gemm, oracle, m, n, k, slices, mode):
    rp = _rowpanel()
    a, b = _libs.gen_f32(oracle, m, k, 71), _libs.gen_f32(oracle, k, n, 72)
    A, B = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    plan = rp.RowPanelPlan(gemm, 0, m, n, k, mode, slices)
    assert plan.chunks == (slices or [(0, k)])
    C = torch.full((m, n), float("nan"), device="cuda")
    plan.run(A, B, C)
    c = C.cpu().numpy()
    if mode == 0:       # K-sliced strict: one fused chain per element continuing through C — still the naive loop's bits
        assert np.array_equal(c, _libs.ref_f32_fma(oracle, a, b)), gemm.last_kernel()
    else:
        assert rel(c, _libs.ref_f64(oracle, a, b)) <= TOL[mode], (gemm.last_kernel(), mode)
    # a smaller panel through the same plan (m_local <= m_local_max), then the host variant: C += A*B
    C2 = torch.empty((m // 2, n), device="cuda")
    plan.run(A[: m // 2], B, C2)
    if mode == 0:
        assert torch.equal(C2, C[: m // 2])
    else:                                                    # other tile shapes may be picked for the smaller panel
        assert rel(C2.cpu().numpy(), _libs.ref_f64(oracle, a[: m // 2], b)) <= TOL[mode]
    hA, hB = torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory()
    hC = torch.ones((m, n)).pin_memory()
    plan.run_host(hA, hB, hC)
    if mode == 0:
        assert np.array_equal(hC.numpy(), _libs.ref_f32_fma(oracle, a, b, np.ones((m, n), np.float32)))
    else:
        assert rel(hC.numpy() - 1.0, _libs.ref_f64(oracle, a, b)) <= 2 * max(TOL[mode], 1e-6)
    plan.close()


def test_rowpanel_default_slices_match_the_python_model(gemm):
    rp = _rowpanel()
    for k in (512, 1100, 4096, 16384):
        plan = rp.RowPanelPlan(gemm, 0, 128, 256, k, 5)
        assert plan.chunks == rp.default_slices(k, 1)
        plan.close()
    with pytest.raises(gemm.B200GemmError):
        rp.RowPanelPlan(gemm, 0, 128, 256, 1024, 5, [(0, 100), (100, 1024)])     # slice boundary not a multiple of 8


# ---- two NCCL ranks ---------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, M, N, K, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import torch.distributed as dist
    import _libs as L
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    g = L.load_pkg()
    o = L.load_oracle()
    import importlib
    rp = importlib.import_module(L.PKG + ".rowpanel")
    comm = rp.nccl_comm_ptr(dist, dev)
    a, b = L.gen_f32(o, M, K, 100), L.gen_f32(o, K, N, 200)
    r0, r1 = rp.row_panel(rank, world, M)
    A = torch.from_numpy(a[r0:r1]).to(dev)
    res = {}
    for mode in (5, 2, 0):
        for slices in (None, [(0, K // 2), (K // 2, K)]):
            B = torch.from_numpy(b).to(dev) if rank == 0 else torch.full((K, N), float("nan"), device=dev)
            C = torch.full((r1 - r0, N), float("nan"), device=dev)
            plan = rp.RowPanelPlan(g, comm, r1 - r0, N, K, mode, slices)
            assert plan.chunks == (slices or rp.default_slices(K, world, N)), plan.chunks      # the C++ default == its Python model
            for _ in range(3):                       # back-to-back steps reuse the plan's buffers and events
                plan.run(A, B, C)
            torch.cuda.synchronize()
            res[f"c_{mode}_{0 if slices is None else 1}"] = C.cpu().numpy()
            res[f"b_ok_{mode}_{0 if slices is None else 1}"] = np.array([bool(torch.equal(B.cpu(), torch.from_numpy(b)))])
            if slices is None:
                hA = torch.from_numpy(a[r0:r1]).pin_memory()
                hB = torch.from_numpy(b).pin_memory() if rank == 0 else None
                hC = torch.zeros((r1 - r0, N)).pin_memory()
                plan.run_host(hA, hB, hC)
                res[f"h_{mode}"] = hC.numpy().copy()
            plan.close()
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_rowpanel_two_nccl_ranks_full_c(tmp_path, oracle):
    import torch.multiprocessing as mp
    world, M, N, K = 2, 1000, 1104, 2048
    mp.spawn(_worker, args=(world, _free_port(), M, N, K, str(tmp_path)), nprocs=world, join=True)
    a, b = _libs.gen_f32(oracle, M, K, 100), _libs.gen_f32(oracle, K, N, 200)
    t, naive = _libs.ref_f64(oracle, a, b), _libs.ref_f32_fma(oracle, a, b)
    parts = [np.load(tmp_path / f"r{r}.npz") for r in range(world)]
    for mode in (5, 2, 0):
        for s in (0, 1):
            C = np.concatenate([p[f"c_{mode}_{s}"] for p in parts], axis=0)
            assert all(bool(p[f"b_ok_{mode}_{s}"][0]) for p in parts), "B differs from the root's after the exchange"
            if mode == 0:
                assert np.array_equal(C, naive)
            else:
                assert rel(C, t) <= TOL[mode], (mode, s, rel(C, t))
        H = np.concatenate([p[f"h_{mode}"] for p in parts], axis=0)
        if mode == 0:
            assert np.array_equal(H, naive)
        else:
            assert rel(H, t) <= TOL[mode]


def _demo(*args):
    import subprocess
    exe = os.path.join(_libs.ROOT, _libs.PKG, "harness", "rowpanel_demo.x")
    if not os.path.exists(exe):
        pytest.skip(f"{exe} not built (make -C {_libs.PKG} host)")
    r = subprocess.run([exe, *[str(a) for a in args]], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    row = r.stdout.split("MY_MMult = [")[1].split("];")[0].split()
    return int(row[0]), float(row[1]), float(row[2])


def test_cxx_host_single_gpu():
    """harness/rowpanel_demo.cpp: a C++ program (no Python, no torch) driving the plan through include/b200gemm.h."""
    gpus, gflops, err = _demo(1, 1024, 1280, 1536, 5)
    assert gpus == 1 and gflops > 0 and err <= 1e-5


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_cxx_host_two_gpus_one_thread_each():
    """One process, one host thread per GPU (per-device library state), NCCL communicator made through the C ABI
    (b200_comm_unique_id / b200_comm_init_rank), libnccl resolved by dlopen."""
    gpus, gflops, err = _demo(2, 1024, 1280, 1536, 5)
    assert gpus == 2 and gflops > 0 and err <= 1e-5
