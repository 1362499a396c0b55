"""how-to-optimize-gemm_b200 — Python host binding of libb200gemm.so (ctypes over the C ABI).

The product is the CUDA library; this module only loads it and forwards pointers.  PyTorch is
plumbing (device memory, streams, torch.distributed) and is imported lazily, only by the helpers
that take tensors.  There is NO CPU fallback: if the shared library is missing, import fails
loudly; if no sm_100 GPU is present, every compute call raises B200GemmError(-2).

Interface mirrored from the reference (file:line in /root/reference):
  MY_MMult(m, n, k, a, lda, b, ldb, c, ldc)                 aarch64/MMult0.cpp:3   (host, C += A*B)
  MY_MMult_cuda(handle, m, n, k, dA, lda, dB, ldb, dC, ldc)  cuda/test_MMult.cpp:13 (device, C = A*B)
  MY_MMult_int8(m, n, k, a, lda, b, ldb, c, ldc)             aarch64-int8/test_MMult.c:9
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200gemm.so")

F32_STRICT, F32_TF32, F32_BF16X3, F32_BF16X2, F32_AUTO, F32_F16X2 = 0, 1, 2, 3, 4, 5
OUT_F32, OUT_BF16 = 0, 1

EXPORTS = [
    "b200_gemm_version", "b200_gemm_device_ok", "b200_gemm_strerror", "b200_gemm_last_kernel",
    "b200_gemm_launch_count", "b200_gemm_default_f32_mode", "b200_gemm_set_default_f32_mode",
    "b200_gemm_f32", "b200_gemm_f32_acc", "b200_gemm_f32_ex", "b200_gemm_workspace_bytes", "b200_gemm_reserve_workspace", "b200_mxf4_q_bytes", "b200_mxf4_sf_bytes",
    "b200_mxf4_quantize_a", "b200_mxf4_quantize_b", "b200_gemm_mxf4", "b200_gemm_f32_host", "b200_gemm_bf16", "b200_gemm_s8s32",
    "b200_gemm_s8s32_host", "b200_gemm_s8s8_requant", "b200_gemm_f32_pack_b", "b200_gemm_f32_packed",
    "b200_gemm_f32_pack_free", "b200_nccl_load", "b200_nccl_last_error", "b200_comm_unique_id", "b200_comm_init_rank",
    "b200_comm_destroy", "b200_rowpanel_create", "b200_rowpanel_destroy", "b200_rowpanel_slices", "b200_rowpanel_set_reserve_sms", "b200_rowpanel_trace", "b200_rowpanel_trace_dump", "b200_gemm_f32_rowpanel",
    "b200_gemm_f32_rowpanel_host", "b200_gemm_f32_pack_a", "b200_gemm_f32_packed_ab", "b200_gemm_f32_pack_free_a",
    "b200_convert_f32_to_bf16", "b200_gemm_debug_set_b_desc", "b200_gemm_debug_set_bn",
    "b200_gemm_debug_set_split_chunk", "b200_gemm_debug_kernel_timing", "b200_gemm_debug_kernel_time_ms",
    "b200_gemm_debug_set_cta_group", "b200_gemm_debug_set_split_tail", "b200_gemm_debug_set_group_rows",
    "b200_gemm_debug_set_ffma_variant", "b200_gemm_debug_set_epilogue", "b200_gemm_debug_set_pdl", "b200_gemm_debug_set_dynamic_sched",
    "b200_gemm_debug_last_schedule",
]


class B200GemmError(RuntimeError):
    def __init__(self, code, what=""):
        self.code = code
        super().__init__(f"b200gemm error {code}: {what}")


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc, sm_100a). There is no CPU or PyTorch fallback for this path.")

lib = C.CDLL(LIB_PATH)
_vp, _i = C.c_void_p, C.c_int
lib.b200_gemm_version.restype = C.c_char_p
lib.b200_gemm_strerror.restype = C.c_char_p
lib.b200_gemm_strerror.argtypes = [_i]
lib.b200_gemm_last_kernel.restype = C.c_char_p
lib.b200_gemm_launch_count.restype = C.c_ulonglong
lib.b200_gemm_f32.argtypes = [_i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _i, _vp]
lib.b200_gemm_f32_acc.argtypes = [_i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _i, _vp]
lib.b200_gemm_f32_ex.argtypes = [_i, _i, _i, C.c_float, _vp, _i, _vp, _i, C.c_float, _vp, _i, _i, _vp]
lib.b200_gemm_workspace_bytes.argtypes = [_i, _i, _i, _i]
lib.b200_gemm_workspace_bytes.restype = C.c_size_t
lib.b200_gemm_reserve_workspace.argtypes = [C.c_size_t]
lib.b200_mxf4_q_bytes.argtypes = [_i, _i]
lib.b200_mxf4_q_bytes.restype = C.c_size_t
lib.b200_mxf4_sf_bytes.argtypes = [_i, _i]
lib.b200_mxf4_sf_bytes.restype = C.c_size_t
lib.b200_mxf4_quantize_a.argtypes = [_i, _i, _vp, _i, _vp, _vp, _vp]
lib.b200_mxf4_quantize_b.argtypes = [_i, _i, _vp, _i, _vp, _vp, _vp]
lib.b200_gemm_mxf4.argtypes = [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp]
lib.b200_gemm_f32_host.argtypes = [_i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _i]
lib.b200_gemm_bf16.argtypes = [_i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _i, _vp]
lib.b200_gemm_s8s32.argtypes = [_i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp]
lib.b200_gemm_s8s32_host.argtypes = [_i, _i, _i, _vp, _i, _vp, _i, _vp, _i]
lib.b200_gemm_f32_pack_b.argtypes = [_i, _i, _vp, _i, _i, C.POINTER(_vp), _vp]
lib.b200_gemm_f32_packed.argtypes = [_i, _i, _i, _vp, _i, _vp, _vp, _i, _i, _vp]
lib.b200_gemm_f32_pack_free.argtypes = [_vp]
lib.b200_gemm_f32_pack_free.restype = None
lib.b200_gemm_f32_pack_a.argtypes = [_i, _i, _vp, _i, _i, C.POINTER(_vp), _vp]
lib.b200_gemm_f32_packed_ab.argtypes = [_i, _i, _i, _vp, _i, _vp, _vp, _i, _i, _vp]
lib.b200_gemm_f32_pack_free_a.argtypes = [_vp]
lib.b200_gemm_f32_pack_free_a.restype = None
lib.b200_nccl_load.argtypes = [C.c_char_p]
lib.b200_nccl_last_error.restype = C.c_char_p
lib.b200_comm_unique_id.argtypes = [_vp]
lib.b200_comm_init_rank.argtypes = [C.POINTER(_vp), _vp, _i, _i]
lib.b200_comm_destroy.argtypes = [_vp]
lib.b200_rowpanel_create.argtypes = [C.POINTER(_vp), _vp, _i, _i, _i, _i, C.POINTER(_i), _i]
lib.b200_rowpanel_destroy.argtypes = [_vp]
lib.b200_rowpanel_destroy.restype = None
lib.b200_rowpanel_slices.argtypes = [_vp, C.POINTER(_i), _i]
lib.b200_rowpanel_set_reserve_sms.argtypes = [_vp, _i]
lib.b200_rowpanel_trace.argtypes = [_vp, _i]
lib.b200_rowpanel_trace.restype = None
lib.b200_rowpanel_trace_dump.argtypes = [_vp, C.POINTER(C.c_float), _i]
lib.b200_gemm_f32_rowpanel.argtypes = [_vp, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _i, _vp]
lib.b200_gemm_f32_rowpanel_host.argtypes = [_vp, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _i]
lib.b200_gemm_s8s8_requant.argtypes = [_i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _vp, _vp]
lib.b200_convert_f32_to_bf16.argtypes = [_vp, _vp, C.c_size_t, _vp]
lib.b200_gemm_debug_set_b_desc.argtypes = [_i, _i]
lib.b200_gemm_set_default_f32_mode.argtypes = [_i]
lib.b200_gemm_debug_set_bn.argtypes = [_i]
lib.b200_gemm_debug_set_split_chunk.argtypes = [_i, _i]
lib.b200_gemm_debug_kernel_timing.argtypes = [_i]
lib.b200_gemm_debug_set_cta_group.argtypes = [_i]
lib.b200_gemm_debug_set_split_tail.argtypes = [_i]
lib.b200_gemm_debug_set_pdl.argtypes = [_i]
lib.b200_gemm_debug_set_dynamic_sched.argtypes = [_i]
lib.b200_gemm_debug_kernel_time_ms.argtypes = [C.POINTER(C.c_double)]
lib.b200_gemm_debug_last_schedule.argtypes = [C.POINTER(_i), _i]

SCHEDULE_FIELDS = ("tile_m", "bn", "cta_group", "epilogue_warps", "tiles", "grid_units", "full_tiles", "split",
                   "halfn", "dynamic")


def kernel_time_ms():
    """(sum_ms, launches) of the dominant GEMM kernel since kernel timing was enabled."""
    s = C.c_double(0.0)
    n = lib.b200_gemm_debug_kernel_time_ms(C.byref(s))
    return s.value, n


def _check(rc):
    if rc != 0:
        what = lib.b200_gemm_strerror(rc).decode()
        if rc == -5:
            what += ": " + lib.b200_nccl_last_error().decode()
        raise B200GemmError(rc, what)


def version():
    return lib.b200_gemm_version().decode()


def last_kernel():
    return lib.b200_gemm_last_kernel().decode()


def launch_count():
    return int(lib.b200_gemm_launch_count())


def last_schedule():
    """Work schedule of this thread's last tensor-core or strict-FFMA launch as a dict (SCHEDULE_FIELDS), or
    None when the last launch was another kernel (b200_gemm_debug_last_schedule)."""
    buf = (_i * len(SCHEDULE_FIELDS))()
    n = lib.b200_gemm_debug_last_schedule(buf, len(buf))
    return dict(zip(SCHEDULE_FIELDS, buf[:n])) if n else None


def _stream_ptr(stream):
    if stream is None:
        import torch
        return torch.cuda.current_stream().cuda_stream
    return getattr(stream, "cuda_stream", stream)


# ---- raw-pointer forms (exact mirrors of the reference signatures) ------------------------------
def MY_MMult_cuda(handle, m, n, k, dA, lda, dB, ldb, dC, ldc, mode=F32_AUTO, stream=0):
    """cuda/test_MMult.cpp:13-14 — device pointers (ints), C = A*B.  `handle` is ignored, as the
    reference's hand kernels ignore it (cuda/MMult_cuda_12.cu:228)."""
    _check(lib.b200_gemm_f32(m, n, k, dA, lda, dB, ldb, dC, ldc, mode, stream))


def MY_MMult(m, n, k, a, lda, b, ldb, c, ldc, mode=F32_AUTO):
    """aarch64/MMult0.cpp:3-4 — numpy float32 host arrays, C += A*B in place."""
    _check(lib.b200_gemm_f32_host(m, n, k, a.ctypes.data, lda, b.ctypes.data, ldb, c.ctypes.data, ldc, mode))


def MY_MMult_int8(m, n, k, a, lda, b, ldb, c, ldc):
    """aarch64-int8/test_MMult.c:9,98 — numpy int8 host arrays, int32 C = A*B."""
    _check(lib.b200_gemm_s8s32_host(m, n, k, a.ctypes.data, lda, b.ctypes.data, ldb, c.ctypes.data, ldc))


# ---- tensor forms (torch CUDA tensors; row-major, last dim contiguous) --------------------------
def _ld(t):
    assert t.dim() == 2 and (t.stride(1) == 1 or t.shape[1] <= 1), "row-major 2-D tensor with unit inner stride expected"
    if t.shape[1] <= 1:              # a single column: any stride is reported for the size-1 dimension
        return max(1, t.stride(0)) if t.shape[0] > 1 else 1
    return t.stride(0) if t.shape[0] > 1 else max(t.shape[1], t.stride(0))


def gemm_f32(A, B, out=None, mode=F32_AUTO, stream=None, accumulate=False):
    """C = A*B, or C += A*B into `out` when accumulate is set (b200_gemm_f32_acc)."""
    import torch
    assert A.dtype == torch.float32 and B.dtype == torch.float32 and A.is_cuda and B.is_cuda
    m, k = A.shape
    k2, n = B.shape
    assert k == k2
    if out is None:
        out = torch.empty((m, n), dtype=torch.float32, device=A.device)
    fn = lib.b200_gemm_f32_acc if accumulate else lib.b200_gemm_f32
    assert not accumulate or out is not None
    _check(fn(m, n, k, A.data_ptr(), _ld(A), B.data_ptr(), _ld(B), out.data_ptr(), _ld(out), mode, _stream_ptr(stream)))
    return out


def gemm_f32_ex(alpha, A, B, beta, out, mode=F32_AUTO, stream=None):
    """out = alpha * A*B + beta * out (b200_gemm_f32_ex; cuBLAS sgemm semantics, cuda/MMult_cuBLAS_1.cpp:11-19)."""
    m, k = A.shape
    n = B.shape[1]
    _check(lib.b200_gemm_f32_ex(m, n, k, alpha, A.data_ptr(), _ld(A), B.data_ptr(), _ld(B), beta, out.data_ptr(), _ld(out),
                                mode, _stream_ptr(stream)))
    return out


def mxf4_quantize(X, transpose=False, stream=None):
    """fp32 CUDA matrix -> (q, sf, rows, k): packed E2M1 rows + UE8M0 scale atoms (b200_mxf4_quantize_a / _b).
    transpose=False: X is A (m x k), rows = m.  transpose=True: X is B (k x n) and the result is B^T (rows = n)."""
    import torch
    assert X.dtype == torch.float32 and X.is_cuda and X.dim() == 2
    r, c = X.shape
    rows, k = (c, r) if transpose else (r, c)
    q = torch.empty(lib.b200_mxf4_q_bytes(rows, k), dtype=torch.uint8, device=X.device)
    sf = torch.empty(lib.b200_mxf4_sf_bytes(rows, k), dtype=torch.uint8, device=X.device)
    fn = lib.b200_mxf4_quantize_b if transpose else lib.b200_mxf4_quantize_a
    _check(fn(r, c, X.data_ptr(), _ld(X), q.data_ptr(), sf.data_ptr(), _stream_ptr(stream)))
    return q, sf, rows, k


def gemm_mxf4(qa, sfa, qb, sfb, m, n, k, out=None, stream=None):
    """C (m x n fp32) = dequant(A_q) * dequant(B_q)^T from mxf4_quantize outputs (b200_gemm_mxf4)."""
    import torch
    if out is None:
        out = torch.empty((m, n), dtype=torch.float32, device=qa.device)
    _check(lib.b200_gemm_mxf4(m, n, k, qa.data_ptr(), sfa.data_ptr(), qb.data_ptr(), sfb.data_ptr(), out.data_ptr(), _ld(out),
                              _stream_ptr(stream)))
    return out


def gemm_bf16(A, B, out=None, out_dtype=None, stream=None):
    import torch
    assert A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16 and A.is_cuda and B.is_cuda
    m, k = A.shape
    k2, n = B.shape
    assert k == k2
    if out is None:
        out = torch.empty((m, n), dtype=out_dtype or torch.float32, device=A.device)
    ot = OUT_F32 if out.dtype == torch.float32 else OUT_BF16
    assert out.dtype in (torch.float32, torch.bfloat16)
    _check(lib.b200_gemm_bf16(m, n, k, A.data_ptr(), _ld(A), B.data_ptr(), _ld(B), out.data_ptr(), _ld(out),
                              ot, _stream_ptr(stream)))
    return out


class PackedB:
    """Pre-split B (b200_gemm_f32_pack_b): holds the handle, frees it with the object."""

    def __init__(self, B, mode=F32_AUTO, stream=None):
        import torch
        assert B.dtype == torch.float32 and B.is_cuda and B.dim() == 2
        self.k, self.n = B.shape
        self.handle = _vp()
        _check(lib.b200_gemm_f32_pack_b(self.k, self.n, B.data_ptr(), _ld(B), mode, C.byref(self.handle),
                                        _stream_ptr(stream)))

    def close(self):
        if getattr(self, "handle", None):
            lib.b200_gemm_f32_pack_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:      # interpreter shutdown: module globals may already be gone
            pass


class PackedA:
    """Pre-split A (b200_gemm_f32_pack_a, F16X2): holds the handle, frees it with the object."""

    def __init__(self, A, mode=F32_AUTO, stream=None):
        import torch
        assert A.dtype == torch.float32 and A.is_cuda and A.dim() == 2
        self.m, self.k = A.shape
        self.handle = _vp()
        _check(lib.b200_gemm_f32_pack_a(self.m, self.k, A.data_ptr(), _ld(A), mode, C.byref(self.handle),
                                        _stream_ptr(stream)))

    def close(self):
        if getattr(self, "handle", None):
            lib.b200_gemm_f32_pack_free_a(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def gemm_f32_packed_ab(packedA, packedB, out, a_k0=0, stream=None, accumulate=False):
    """C (+)= A[:, a_k0:a_k0+k] * B from two pre-split operands (b200_gemm_f32_packed_ab)."""
    _check(lib.b200_gemm_f32_packed_ab(packedA.m, packedB.n, packedB.k, packedA.handle, a_k0, packedB.handle,
                                       out.data_ptr(), _ld(out), 1 if accumulate else 0, _stream_ptr(stream)))
    return out


def gemm_f32_packed(A, packedB, out=None, stream=None, accumulate=False):
    import torch
    assert A.dtype == torch.float32 and A.is_cuda
    m, k = A.shape
    if out is None:
        assert not accumulate
        out = torch.empty((m, packedB.n), dtype=torch.float32, device=A.device)
    _check(lib.b200_gemm_f32_packed(m, packedB.n, k, A.data_ptr(), _ld(A), packedB.handle, out.data_ptr(), _ld(out),
                                    1 if accumulate else 0, _stream_ptr(stream)))
    return out


def gemm_s8s8_requant(A, B, scales, bias=None, out=None, stream=None):
    """int8 x int8 -> int8 with per-row scales / bias (aarch64-int8/int8kernel_m4.S:40,386-426)."""
    import torch
    assert A.dtype == torch.int8 and B.dtype == torch.int8 and A.is_cuda and B.is_cuda
    m, k = A.shape
    k2, n = B.shape
    assert k == k2
    assert scales.dtype == torch.float32 and scales.is_cuda and scales.is_contiguous() and scales.numel() == m
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.is_cuda and bias.is_contiguous() and bias.numel() == m
    if out is None:
        out = torch.empty((m, n), dtype=torch.int8, device=A.device)
    assert out.dtype == torch.int8
    _check(lib.b200_gemm_s8s8_requant(m, n, k, A.data_ptr(), _ld(A), B.data_ptr(), _ld(B), out.data_ptr(), _ld(out),
                                      scales.data_ptr(), bias.data_ptr() if bias is not None else None,
                                      _stream_ptr(stream)))
    return out


def gemm_s8s32(A, B, out=None, stream=None):
    import torch
    assert A.dtype == torch.int8 and B.dtype == torch.int8 and A.is_cuda and B.is_cuda
    m, k = A.shape
    k2, n = B.shape
    assert k == k2
    if out is None:
        out = torch.empty((m, n), dtype=torch.int32, device=A.device)
    _check(lib.b200_gemm_s8s32(m, n, k, A.data_ptr(), _ld(A), B.data_ptr(), _ld(B), out.data_ptr(), _ld(out),
                               _stream_ptr(stream)))
    return out


def convert_f32_to_bf16(src, stream=None):
    import torch
    out = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    _check(lib.b200_convert_f32_to_bf16(src.data_ptr(), out.data_ptr(), src.numel(), _stream_ptr(stream)))
    return out
