/*
 * b200gemm.h — C ABI of the B200-native row-major GEMM (libb200gemm.so).
 *
 * This header is the drop-in boundary for the hot path of
 * tpoisonooo/how-to-optimize-gemm: the free function MY_MMult that the
 * reference's harness links against exactly one object for.  Every entry point
 * below cites the reference interface it stands behind:
 *
 *   b200_gemm_f32     <- cuda/test_MMult.cpp:13-14  (10-arg MY_MMult, device
 *                        pointers, C = A*B; wrapper cuda/MMult_cuda_12.cu:228-235)
 *   b200_gemm_f32_host<- aarch64/MMult0.cpp:3-23 / aarch64/test_MMult.cpp:17
 *                        (9-arg MY_MMult, host pointers, C += A*B)
 *   b200_gemm_bf16    <- same contraction, bf16 operands (BASELINE config 3; no
 *                        reference precedent, semantics of cuda/test_MMult.cpp)
 *   b200_gemm_s8s32   <- aarch64-int8/MMult_4x8_21.c:81-86 (12-arg MY_MMult,
 *                        int8 x int8 -> int32, C = A*B, any m,n,k)
 *   b200_gemm_s8s32_host <- aarch64-int8/test_MMult.c:9,98 (host pointers)
 *   b200_gemm_s8s8_requant <- aarch64-int8/int8kernel_m4.S:40 (int8kernel_m4_requant:
 *                        int8 x int8 -> int8 through per-row scales / bias, :386-426)
 *
 * All matrices are ROW-MAJOR: A is m x k (leading dimension lda >= k),
 * B is k x n (ldb >= n), C is m x n (ldc >= n); leading dimensions are in
 * ELEMENTS.  The reference only ever passes lda=k, ldb=n, ldc=n
 * (cuda/test_MMult.cpp:62) and silently ignores them
 * (cuda/MMult_cuda_12.cu:231-234); this library honours them.
 *
 * Device entry points are fully asynchronous on `stream` (a cudaStream_t passed
 * as void*; NULL = the legacy default stream the reference harness uses,
 * cuda/test_MMult.cpp:98-110), never synchronise or allocate in steady state (see
 * b200_gemm_reserve_workspace for the first call) and may be called on any stream of any
 * sm_100 device (per-device state; make the device current on the calling thread).  They return 0 on success or a cudaError_t /
 * negative B200_ERR_* code.  There is NO CPU fallback: without a CUDA device of
 * compute capability 10.x every compute entry point returns
 * B200_ERR_NO_DEVICE.
 */
#ifndef B200GEMM_H_
#define B200GEMM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes (negative; positive values are cudaError_t) ------------ */
#define B200_OK                 0
#define B200_ERR_BAD_ARG       -1   /* null pointer, negative size, ld too small */
#define B200_ERR_NO_DEVICE     -2   /* no sm_100 device / driver entry point missing */
#define B200_ERR_UNSUPPORTED   -3   /* mode not available for this dtype */
#define B200_ERR_TENSORMAP     -4   /* cuTensorMapEncodeTiled rejected the operand */
#define B200_ERR_NCCL          -5   /* libnccl missing or an NCCL call failed: b200_nccl_last_error() */

/* ---- fp32 precision modes (the SURVEY §7 H1 decision, made explicit) ------ */
enum b200_f32_mode {
  B200_F32_STRICT = 0,   /* CUDA-core FFMA, fp32 multiply-add, k ascending: the
                            arithmetic of cuda/MMult_cuda_12.cu:200-206          */
  B200_F32_TF32   = 1,   /* one tcgen05 kind::tf32 pass (10-bit mantissa inputs,
                            fp32 accumulate in TMEM)                              */
  B200_F32_BF16X3 = 2,   /* split-bf16: a=a1+a2+a3, 6 tcgen05 kind::f16 products per
                            k-step, two-level accumulation (K chunks of 512, each a
                            fresh TMEM accumulator added with a rounded fp32 add to a
                            running sum held in registers): fp32-class error on the
                            tensor cores, elementwise.  The round-1 default.      */
  B200_F32_BF16X2 = 3,   /* split-bf16: a=a1+a2, 3 products, ~2^-17 relative       */
  B200_F32_AUTO   = 4,   /* library default: F16X2 unless the environment variable
                            B200GEMM_F32_MODE or b200_gemm_set_default_f32_mode
                            says otherwise; problems up to ~512^3 with TMA-able
                            operands take the single-launch STRICT kernel, problems
                            up to ~1100^3 the two-launch BF16X3 path               */
  B200_F32_F16X2  = 5    /* scaled split-fp16: rows of A / columns of B are scaled by
                            exact powers of two into [-1,1], a'=h1+h2 in fp16 (22
                            bits), 3 tcgen05 kind::f16 products, two-level
                            accumulation, epilogue unscales.  fp32-class NORMWISE
                            error (elements far below their row/column maximum keep
                            absolute, not relative, precision): half the tensor-core
                            work of BF16X3 at the same measured error.
                            THE LIBRARY DEFAULT.                                   */
};

/* ---- bf16 output selector -------------------------------------------------- */
enum b200_out_type {
  B200_OUT_F32  = 0,     /* C written as float   (4 B/elem) */
  B200_OUT_BF16 = 1      /* C written as bf16    (2 B/elem) */
};

/* Library / device ---------------------------------------------------------- */
const char* b200_gemm_version(void);
/* 0 if a usable sm_100 device is current, else B200_ERR_NO_DEVICE. */
int  b200_gemm_device_ok(void);
/* Human-readable text for a code returned by this library. */
const char* b200_gemm_strerror(int code);
/* Name of the kernel the last call on this thread dispatched to
 * ("tc_bf16_128x256", "ffma_128x128", ...), for tests and bench evidence. */
const char* b200_gemm_last_kernel(void);
/* Number of kernel launches this library has issued since load. */
unsigned long long b200_gemm_launch_count(void);
int  b200_gemm_default_f32_mode(void);
void b200_gemm_set_default_f32_mode(int mode);

/* The split-precision fp32 modes keep the planes of A and B in a per-device, grow-only workspace.  Its first
 * use and every growth allocate (and synchronise the device); steady-state calls never do.  Reserve it up front
 * — b200_gemm_reserve_workspace(b200_gemm_workspace_bytes(m, n, k, mode)) on the device that will run the
 * calls — to keep even the first call allocation-free (e.g. ahead of CUDA-graph capture).  State is per device:
 * one process may drive several GPUs (make the device current on the calling thread); calls on different
 * streams of one device are serialised on the workspace by an event, not by the host. */
size_t b200_gemm_workspace_bytes(int m, int n, int k, int precision_mode);
int    b200_gemm_reserve_workspace(size_t bytes);

/* fp32: C = A*B.  Replaces MY_MMult(cublasHandle_t,m,n,k,dA,lda,dB,ldb,dC,ldc)
 * (cuda/test_MMult.cpp:13-14,100-103).  DEVICE pointers. */
int b200_gemm_f32(int m, int n, int k,
                  const float* dA, int lda, const float* dB, int ldb,
                  float* dC, int ldc, int precision_mode, void* stream);

/* fp32: C += A*B on DEVICE pointers — the CPU harnesses' contract (aarch64/MMult0.cpp:16) without
 * the staging copies; also what lets a K-sliced operand stream (B arriving in row chunks over
 * NVLink) be consumed chunk by chunk.  STRICT keeps one fused chain per element starting from C(i,j);
 * the tensor-core modes fold their fp32 partial sums into C with rounded adds. */
int b200_gemm_f32_acc(int m, int n, int k,
                      const float* dA, int lda, const float* dB, int ldb,
                      float* dC, int ldc, int precision_mode, void* stream);

/* fp32: C = alpha * A*B + beta * C on DEVICE pointers — the contract of the reference's cuBLAS comparator
 * (cublasSgemm, cuda/MMult_cuBLAS_1.cpp:11-19; the harness only ever passes alpha = 1, beta = 0).  beta == 0
 * never reads C.  (1, 0) and (1, 1) are b200_gemm_f32 / b200_gemm_f32_acc exactly; any other pair is fused
 * into the epilogue of the tensor-core modes, and costs two element-wise passes over C around the kernel in
 * STRICT mode and on the generic (unaligned-operand) path. */
int b200_gemm_f32_ex(int m, int n, int k, float alpha,
                     const float* dA, int lda, const float* dB, int ldb, float beta,
                     float* dC, int ldc, int precision_mode, void* stream);

/* fp32 with HOST pointers and the CPU harness contract C += A*B
 * (aarch64/MMult0.cpp:11-19; harness zeroes C first, aarch64/test_MMult.cpp:107).
 * Stages H2D, runs b200_gemm_f32 on the device, adds into C on the device,
 * copies back, synchronises.  Plumbing/parity only, never a reported number. */
int b200_gemm_f32_host(int m, int n, int k,
                       const float* A, int lda, const float* B, int ldb,
                       float* C, int ldc, int precision_mode);

/* bf16 operands (raw uint16 bit patterns), fp32 accumulate; C is float or bf16
 * according to out_type.  DEVICE pointers. */
int b200_gemm_bf16(int m, int n, int k,
                   const uint16_t* dA, int lda, const uint16_t* dB, int ldb,
                   void* dC, int ldc, int out_type, void* stream);

/* int8 x int8 -> int32, exact: C = A*B (aarch64-int8/README.md:8; oracle
 * aarch64-int8/REF_MMult.c:10-23).  DEVICE pointers. */
int b200_gemm_s8s32(int m, int n, int k,
                    const int8_t* dA, int lda, const int8_t* dB, int ldb,
                    int32_t* dC, int ldc, void* stream);

/* int8 with HOST pointers: what aarch64-int8/test_MMult.c:98 passes. */
int b200_gemm_s8s32_host(int m, int n, int k,
                         const int8_t* A, int lda, const int8_t* B, int ldb,
                         int32_t* C, int ldc);

/* Pre-split operands for the split-precision modes (AUTO = the library default): the reference
 * leaves its "packAB interface open" for callers that reuse one operand (README.md:85; PackMatrixA/B,
 * aarch64/MMult_4x4_13.cpp:259,361).  TMA needs no repacking of row-major operands, but the fp32 ->
 * plane split is per-call work (the pre-pass) that a constant operand can pay once.
 *   b200_gemm_f32_pack_b   splits the k x n matrix B (F16X2, BF16X3, BF16X2) into a handle that owns its
 *                          device memory;
 *   b200_gemm_f32_pack_a   does the same for the m x k matrix A (F16X2 only);
 *   b200_gemm_f32_packed   computes C = A*B (accumulate = 0) or C += A*B (1) from fp32 A and packed B and
 *                          is bit-identical to b200_gemm_f32 / b200_gemm_f32_acc in the handle's mode;
 *   b200_gemm_f32_packed_ab  uses both handles and multiplies columns [a_k0, a_k0 + k) of packed A
 *                          (a_k0 a multiple of 8) by a packed B of exactly k rows: a K-sliced consumer
 *                          (B arriving in row blocks over NVLink) splits A once and each block of B as
 *                          it lands.
 * DEVICE pointers; a handle may be used by any number of later calls (stream-ordered after the pack
 * call) on the device it was made on and is released with b200_gemm_f32_pack_free / _free_a.  Modes
 * without a split (STRICT, TF32) return B200_ERR_UNSUPPORTED. */
typedef struct b200_packed_b b200_packed_b;
typedef struct b200_packed_a b200_packed_a;
int b200_gemm_f32_pack_b(int k, int n, const float* dB, int ldb, int precision_mode,
                         b200_packed_b** out, void* stream);
int b200_gemm_f32_pack_a(int m, int k, const float* dA, int lda, int precision_mode,
                         b200_packed_a** out, void* stream);
int b200_gemm_f32_packed(int m, int n, int k, const float* dA, int lda,
                         const b200_packed_b* packedB, float* dC, int ldc,
                         int accumulate, void* stream);
int b200_gemm_f32_packed_ab(int m, int n, int k, const b200_packed_a* packedA, int a_k0,
                            const b200_packed_b* packedB, float* dC, int ldc,
                            int accumulate, void* stream);
void b200_gemm_f32_pack_free(b200_packed_b* packedB);
void b200_gemm_f32_pack_free_a(b200_packed_a* packedA);

/* int8 x int8 -> int8 with the requantising tail of chgemm's kernels fused into the
 * GEMM epilogue (aarch64-int8/int8kernel_m4.S:386-426; signature :40):
 *   C(i,j) = sat_int8( round_ties_away( float(sum_p A(i,p)*B(p,j)) * dScales[i] (+ dBias[i]) ) )
 * int32 -> fp32 conversion rounds to nearest even, the multiply and the add round
 * separately (fmul, fadd), NaN converts to 0.  dScales has m entries, dBias has m
 * entries or is NULL (the kernel's `cmp bias, #0`).  C is written once as int8
 * (1 byte per element instead of 4).  DEVICE pointers; ldc in elements (bytes). */
int b200_gemm_s8s8_requant(int m, int n, int k,
                           const int8_t* dA, int lda, const int8_t* dB, int ldb,
                           int8_t* dC, int ldc, const float* dScales,
                           const float* dBias, void* stream);

/* ---- multi-GPU: C sharded by row panels, one exchange step (BASELINE config 5; SURVEY §8e) ------------
 * The reference has no multi-GPU code; north_star asks for "row-panels across the box's GPUs with one
 * NCCL broadcast of B over NVLink" behind this C ABI.  One process (or host thread) per GPU; rank i owns
 * A_i (m_local x k) and C_i (m_local x n); B (k x n) is valid on `root` before the call and on every rank
 * after it.  B crosses NVLink as K-slices (contiguous row blocks of the row-major operand, broadcast in
 * place with ncclBroadcast on the plan's own stream); A_i is split into its planes while the first slice
 * travels and slice j is multiplied while slices j+1.. are in flight.  Timing convention of the
 * reference's harness: operands resident, the exchange inside the call (cuda/test_MMult.cpp:84-112).
 *
 * NCCL is resolved with dlopen at first use (the libnccl.so.2 already loaded in the process, e.g. torch's,
 * else the system one; b200_nccl_load(path) forces one): libb200gemm.so itself does not link NCCL.
 *   nccl_comm   an ncclComm_t (as void*): the caller's own (torch: ProcessGroupNCCL._comm_ptr()) or one
 *               made with b200_comm_unique_id + b200_comm_init_rank (rank 0 creates the 128-byte id and
 *               hands it to the other ranks by whatever means the host has).  NULL = single rank.
 *   slice_rows  rows of B per K-slice (sum k, every boundary a multiple of 8), or NULL / n_slices 0 for the
 *               default (one slice on one rank; two slices weighted 1:3 up to 256 MB of B; equal ~256 MB slices, at most 8, beyond).
 * The plan owns all scratch (planes, events, streams): the compute calls never allocate. */
typedef struct b200_rowpanel b200_rowpanel;
int  b200_nccl_load(const char* libnccl_path_or_null);
const char* b200_nccl_last_error(void);
int  b200_comm_unique_id(void* id128);
int  b200_comm_init_rank(void** nccl_comm_out, const void* id128, int rank, int world);
int  b200_comm_destroy(void* nccl_comm);
int  b200_rowpanel_create(b200_rowpanel** out, void* nccl_comm, int m_local_max, int n, int k,
                          int precision_mode, const int* slice_rows, int n_slices);
void b200_rowpanel_destroy(b200_rowpanel* plan);
/* Tuning.  While a later K-slice is still being broadcast, the GEMM of the current slice shares the GPU with NCCL's
 * copy kernels; those GEMMs therefore draw their tiles from an atomic counter (dynamic schedule: a CTA that gets its
 * SM late draws fewer tiles) and may leave `sms` SMs unused (default 0).  sms = -1 switches the dynamic schedule off. */
int  b200_rowpanel_set_reserve_sms(b200_rowpanel* plan, int sms);
/* Diagnostics: with tracing on, timing events bracket every stage of a call; the dump synchronises the device and
 * writes, in ms after the call began: A split done, then per K-slice {broadcast begin, broadcast end, slice visible
 * on the compute stream, split done, GEMM done}.  Returns the number of values. */
void b200_rowpanel_trace(b200_rowpanel* plan, int enable);
int  b200_rowpanel_trace_dump(b200_rowpanel* plan, float* out_ms, int cap);
/* K-slice boundaries of the plan: writes min(n_slices + 1, cap) row offsets, returns n_slices. */
int  b200_rowpanel_slices(const b200_rowpanel* plan, int* bounds, int cap);
/* C_local = A_local * B on DEVICE pointers (dB: the operand on root, the receive buffer elsewhere; ldb == n
 * unless single-rank).  Asynchronous on `stream`. */
int  b200_gemm_f32_rowpanel(b200_rowpanel* plan, int m_local, int n, int k,
                            const float* dA_local, int lda, float* dB, int ldb,
                            float* dC_local, int ldc, int root, void* stream);
/* C_local += A_local * B with HOST pointers (the 9-arg MY_MMult contract, aarch64/MMult0.cpp:3-23, sharded):
 * B is read on root only; H2D, exchange, math and D2H are pipelined inside; synchronous. */
int  b200_gemm_f32_rowpanel_host(b200_rowpanel* plan, int m_local, int n, int k,
                                 const float* A_local, int lda, const float* B, int ldb,
                                 float* C_local, int ldc, int root);

/* ---- the 4-bit path (SURVEY §8 f-4) ------------------------------------------------------------------
 * The reference lists a cuda-int4 back-end and ships only the word "WIP" (cuda-int4/README.md:1;
 * README.md:13-15,118-120), so there is no interface to mirror: this is the chgemm idea (quantised operands,
 * wide accumulate) on Blackwell's only 4-bit tensor type, OCP MXFP4 — E2M1 elements with one power-of-two
 * UE8M0 scale per 32 consecutive K elements (tcgen05.mma.kind::mxf4.block_scale), fp32 accumulate and output.
 *   quantize_a   A (m x k fp32, row-major)  -> dQ (m rows of kpad/2 bytes, two elements per byte, low nibble
 *                first; kpad = k rounded up to 128) + dSF (scale atoms, b200_mxf4_sf_bytes(m, k) bytes)
 *   quantize_b   B (k x n fp32, row-major)  -> B^T quantised along K: dQ has n rows (4-bit operands must be
 *                K-major for the tensor core: the one transposing pass of this library) + dSF(n, k)
 *   gemm_mxf4    C (m x n fp32) = dequant(A) * dequant(B)
 * Scale atom layout: [rows/128][kpad/128][512 bytes], byte (r%32)*16 + ((r/32)%4)*4 + (kblock%4).
 * DEVICE pointers, 16-byte aligned; asynchronous on `stream`. */
size_t b200_mxf4_q_bytes(int rows, int k);
size_t b200_mxf4_sf_bytes(int rows, int k);
int b200_mxf4_quantize_a(int m, int k, const float* dA, int lda, uint8_t* dQ, uint8_t* dSF, void* stream);
int b200_mxf4_quantize_b(int k, int n, const float* dB, int ldb, uint8_t* dQ, uint8_t* dSF, void* stream);
int b200_gemm_mxf4(int m, int n, int k, const uint8_t* dAq, const uint8_t* dSFA,
                   const uint8_t* dBq, const uint8_t* dSFB, float* dC, int ldc, void* stream);

/* Element-wise helper the bf16 config needs on the device: round-to-nearest-
 * even fp32 -> bf16 (the rounding SURVEY §8d prescribes for config 3 inputs). */
int b200_convert_f32_to_bf16(const float* dSrc, uint16_t* dDst, size_t count,
                             void* stream);

/* Test/diagnostic hook: overrides for the UMMA shared-memory descriptor of the
 * MN-major B operand (bytes; 0 = library default).  Used only by the probe in
 * tests/ to pin the descriptor semantics on real hardware. */
void b200_gemm_debug_set_b_desc(int lbo_bytes, int sbo_bytes);
/* Tuning hook: 0 = launch without programmatic dependent launch (default 1: the library's tensor-core and
 * pre-pass kernels are launched with the programmatic-serialisation attribute and order themselves with
 * griddepcontrol.wait, so a kernel's prologue overlaps the tail of its predecessor in the stream). */
void b200_gemm_debug_set_pdl(int mask);   /* bit 0: PDL on; bit 1: keep the F16X2 pre-pass of B on the caller's stream (default: auxiliary stream beside A's) */
/* Tuning hook: 1 = a scheduler warp hands tiles out from an atomic counter, so CTAs that start late because a
 * co-running kernel holds their SM draw fewer tiles; 0 (default) = static round-robin tile schedule, except where
 * the row-panel plan asks for the dynamic one. */
void b200_gemm_debug_set_dynamic_sched(int on);
/* Tuning hook: force the tensor-core tile width (128, 192 or 256; 0 = built-in heuristic). */
void b200_gemm_debug_set_bn(int bn);
/* Tuning hook: 1 = single-CTA tiles only, 2 = CTA pairs (tcgen05 cta_group::2) always, 0 = auto. */
void b200_gemm_debug_set_cta_group(int cg);
/* Tuning hook: 1 (default) = the last partial round of tiles is split along K across the idle
 * CTAs and folded into C in order; 0 = whole tiles only. */
void b200_gemm_debug_set_split_tail(int on);
/* Tuning hook: K extent the tensor core accumulates before the epilogue folds the partial sum
 * into C with a rounded fp32 add (two-level accumulation of the split modes); 0 = whole K.
 * bf16x2_k sets the F16X2 mode's extent as well.  A negative argument restores the built-in
 * defaults of all three modes (BF16X3 512, BF16X2 512, F16X2 1024). */
void b200_gemm_debug_set_split_chunk(int bf16x3_k, int bf16x2_k);
/* Test hook: the work schedule of the calling thread's last tensor-core or strict-FFMA kernel launch, as
 * {tile_m, bn, cta_group, epilogue_warps, tiles, grid_units, full_tiles, split, halfn, dynamic}:
 * rows and columns of one tile (tile_m = 256 for a CTA pair), CTAs per tile, epilogue warps per CTA
 * (0 for the FFMA kernels), tiles of C, CTAs or CTA pairs launched, work items that are whole tiles,
 * K parts of each tail tile, 1 if tail tiles are issued as two half-width tiles (the FFMA kernels'
 * half tiles), 1 if the dynamic tile scheduler ran.  Writes min(10, cap) values to out and returns the
 * count; returns 0 when the last launch of the thread was another kernel (generic, fill, pre-pass). */
int  b200_gemm_debug_last_schedule(int* out, int cap);
/* Tuning hook: rows of A per raster group of the persistent tile schedule (0 = 2048). */
void b200_gemm_debug_set_group_rows(int rows);
/* Tuning hook for the strict fp32 kernels: bit 0 = half tiles in the last partial round (default on),
 * bit 1 = force the 128x256 fat-thread kernel; a negative value restores selection by size. */
void b200_gemm_debug_set_ffma_variant(int v);
/* Tuning hook, bit mask: bit 0 = non-folding epilogue passes store straight from registers instead of through
 * the shared-memory transpose (measured no faster on B200; default off); bit 1 = drain the CTA-pair kernels of
 * the plain kinds (bf16, tf32, int8) with 4 epilogue warps instead of the default 8 (two warps per TMEM lane
 * quadrant, half the column passes each; results are bit-identical). */
void b200_gemm_debug_set_epilogue(int mask);
/* Measurement hook: while enabled, a CUDA-event pair is recorded on the launching stream around
 * every dominant GEMM kernel launch (not the split pre-pass).  b200_gemm_debug_kernel_time_ms
 * synchronises those events, stores the summed kernel time and returns the number of launches
 * covered (then resets).  bench.py's roofline.achieved comes from here. */
void b200_gemm_debug_kernel_timing(int enable);
int  b200_gemm_debug_kernel_time_ms(double* sum_ms);

#ifdef __cplusplus
}
#endif
#endif /* B200GEMM_H_ */
