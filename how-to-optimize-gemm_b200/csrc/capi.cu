// capi.cu — the C ABI of libb200gemm.so (include/b200gemm.h): argument checks, tensor-map
// construction and caching, kernel selection and launch.  Host-side counterpart of the reference's
// MY_MMult wrappers (cuda/MMult_cuda_12.cu:228-235; aarch64-int8/MMult_4x8_21.c:81-143).
//
// No cuBLAS, no CUTLASS, no CPU fallback: if no sm_100 device is usable every compute entry point
// fails with B200_ERR_NO_DEVICE.
#include "../../include/b200gemm.h"

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "gemm_ffma.cuh"
#include "gemm_generic.cuh"
#include "gemm_mxf4.cuh"
#include "gemm_tc.cuh"

using namespace b200;

namespace {

std::atomic<unsigned long long> g_launches{0};
int g_split_tail = 1;        // test/tuning hook (b200_gemm_debug_set_split_tail): 0 = whole tiles only

// Optional per-launch timing of the dominant GEMM kernel (bench.py's roofline.achieved): a pair of
// CUDA events is recorded on the launching stream around the kernel.  Off by default.
struct KernelTimer {
  static constexpr int CAP = 1024;
  bool on = false;
  int n = 0;
  cudaEvent_t ev[CAP][2] = {};
  void begin(cudaStream_t st) {
    if (!on || n >= CAP) return;
    if (!ev[n][0]) { cudaEventCreate(&ev[n][0]); cudaEventCreate(&ev[n][1]); }
    cudaEventRecord(ev[n][0], st);
  }
  void end(cudaStream_t st) {
    if (!on || n >= CAP) return;
    cudaEventRecord(ev[n][1], st);
    n++;
  }
} g_ktimer;
std::atomic<int> g_default_f32_mode{-1};
thread_local const char* t_last_kernel = "none";
// Work schedule of the calling thread's last tensor-core or FFMA launch (b200_gemm_debug_last_schedule), so that a
// test can confirm which kernel variant and which tail path it exercised.  n = 0: the last launch was neither.
struct SchedRecord {
  static constexpr int N = 10;
  int n = 0;
  int v[N] = {};   // tile_m, bn, cta_group, epilogue_warps, tiles, grid_units, full_tiles, split, halfn, dynamic
  void set(int tile_m, int bn, int cg, int epiw, int tiles, int units, int full, int split, int halfn, int dyn) {
    const int r[N] = {tile_m, bn, cg, epiw, tiles, units, full, split, halfn, dyn};
    for (int i = 0; i < N; i++) v[i] = r[i];
    n = N;
  }
  void clear() { n = 0; }
};
thread_local SchedRecord t_last_sched;
// General epilogue request of the current call (b200_gemm_f32_ex): read by launch_tc, reset by the entry point.
struct EpiOpts { int axpby = 0; float alpha = 1.f, beta = 0.f; };
thread_local EpiOpts t_epi;
// SMs the tensor-core launches of the current call leave free (the row-panel plan sets it while a later K-slice
// of B is still being broadcast: a persistent GEMM holding every SM would starve NCCL's copy kernels and
// serialise the exchange behind the math — measured on 2 x B200, DESIGN §7).
thread_local int t_sm_reserve = 0;
// The row-panel plan sets this for GEMMs that run while NCCL's copy kernels hold some SMs: CTAs that start late then
// draw fewer tiles instead of delaying a statically scheduled grid (measured on 2 x B200: a K = 1024 slice took 137 us
// instead of ~80 under the static schedule).
thread_local int t_dynamic_sched = 0;
int g_dbg_b_lbo = 0, g_dbg_b_sbo = 0;

// ---- per-device state ------------------------------------------------------------------------------
// Everything the library caches on a GPU lives in the context of THAT device (flags, split workspace,
// host-path staging buffers and streams, which kernels already had their dynamic shared memory limit
// raised), so one process may drive several GPUs (one host thread or one stream per GPU).  The split
// workspace is shared by all streams of a device: users are serialised by ws_mu on the host and by an
// event recorded after the consuming GEMM on the device (a call on another stream waits for it).
struct Scratch { void* p = nullptr; size_t bytes = 0; };
struct HostPipe {
  bool ready = false;
  cudaStream_t h2d = nullptr, comp = nullptr, d2h = nullptr;
  cudaEvent_t in[8] = {}, done[8] = {};
  cudaError_t init() {
    if (ready) return cudaSuccess;
    cudaError_t e;
    if ((e = cudaStreamCreateWithFlags(&h2d, cudaStreamNonBlocking)) != cudaSuccess) return e;
    if ((e = cudaStreamCreateWithFlags(&comp, cudaStreamNonBlocking)) != cudaSuccess) return e;
    if ((e = cudaStreamCreateWithFlags(&d2h, cudaStreamNonBlocking)) != cudaSuccess) return e;
    for (int i = 0; i < 8; i++) {
      if ((e = cudaEventCreateWithFlags(&in[i], cudaEventDisableTiming)) != cudaSuccess) return e;
      if ((e = cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming)) != cudaSuccess) return e;
    }
    ready = true;
    return cudaSuccess;
  }
};
struct DevCtx {
  int ok = 0;          // 1 usable, -1 not usable, 0 unknown
  int sms = 0;
  int dev = -1;
  int* flags = nullptr;      // tail-split ordering flags (zero between launches), 16 rotating slots of 1024 ints
  unsigned flag_slot = 0;
  int* sched_counters = nullptr;   // dynamic tile scheduler: 64 rotating work counters, zero between launches
  unsigned sched_slot = 0;
  // split-precision workspace (planes of A and B, row / column maxima): cached, grow-only
  std::mutex ws_mu;
  Scratch ws;
  cudaEvent_t ws_event = nullptr;    // recorded after the last GEMM that read the workspace
  cudaStream_t ws_stream = nullptr;  // stream of that GEMM
  bool ws_busy = false;
  unsigned cmax_slot = 0;            // F16X2: double-buffered column maxima (the idle one is re-zeroed by the pre-pass)
  float* cmax_buf = nullptr;
  size_t cmax_cap = 0;
  int cmax_dirty[2] = {0, 0};       // entries of each half that may be non-zero
  cudaStream_t aux = nullptr;        // B's pre-pass chain runs here, beside A's on the caller's stream
  cudaEvent_t aux_fork = nullptr, aux_join = nullptr;
  // host-pointer entry points
  std::mutex host_mu;
  Scratch scr[4];
  HostPipe pipe;
  std::vector<const void*> attr_done;   // kernels whose MaxDynamicSharedMemorySize was raised on this device
};
constexpr int kMaxDevices = 64;
DevCtx g_ctx[kMaxDevices];
std::mutex g_mu;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;

thread_local DevCtx* t_ctx = nullptr;   // context of the device current on this thread (set by ensure_device)

// Binds t_ctx to the CUDA device current on the calling thread, initialising its context on first use.
int ensure_device() {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) { cudaGetLastError(); t_ctx = nullptr; return B200_ERR_NO_DEVICE; }
  DevCtx* c = &g_ctx[dev];
  t_ctx = c;
  if (c->ok == 1) return 0;
  std::lock_guard<std::mutex> lk(g_mu);
  if (c->ok == 1) return 0;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) { cudaGetLastError(); c->ok = -1; return B200_ERR_NO_DEVICE; }
  if (prop.major != 10) { c->ok = -1; return B200_ERR_NO_DEVICE; }
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess || !fn) {
      cudaGetLastError();
      c->ok = -1;
      return B200_ERR_NO_DEVICE;
    }
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  if (!c->flags) {
    if (cudaMalloc(&c->flags, 16 * 1024 * sizeof(int)) != cudaSuccess || cudaMemset(c->flags, 0, 16 * 1024 * sizeof(int)) != cudaSuccess) {
      cudaGetLastError(); c->flags = nullptr; c->ok = -1; return B200_ERR_NO_DEVICE;
    }
  }
  if (!c->sched_counters) {
    if (cudaMalloc(&c->sched_counters, 64 * sizeof(int)) != cudaSuccess || cudaMemset(c->sched_counters, 0, 64 * sizeof(int)) != cudaSuccess) {
      cudaGetLastError(); c->sched_counters = nullptr; c->ok = -1; return B200_ERR_NO_DEVICE;
    }
  }
  if (!c->ws_event && cudaEventCreateWithFlags(&c->ws_event, cudaEventDisableTiming) != cudaSuccess) {
    cudaGetLastError(); c->ok = -1; return B200_ERR_NO_DEVICE;
  }
  c->dev = dev;
  c->sms = prop.multiProcessorCount;
  c->ok = 1;
  return 0;
}

// Raises a kernel's dynamic shared memory limit once per (kernel, device).
template <typename Kern>
int ensure_smem_attr(Kern kern, int bytes) {
  const void* key = reinterpret_cast<const void*>(kern);
  {
    std::lock_guard<std::mutex> lk(g_mu);
    for (const void* k : t_ctx->attr_done) if (k == key) return 0;
  }
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
  std::lock_guard<std::mutex> lk(g_mu);
  t_ctx->attr_done.push_back(key);
  return 0;
}

// ---- tensor-map cache: cuTensorMapEncodeTiled costs microseconds, the harness calls MY_MMult 20x
// back to back on the same operands (cuda/test_MMult.cpp:100-103).
struct MapKey {
  const void* ptr; int dtype; unsigned long long d0, d1, ld_bytes; unsigned b0, b1; int swz; int dev;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && dtype == o.dtype && d0 == o.d0 && d1 == o.d1 && ld_bytes == o.ld_bytes &&
           b0 == o.b0 && b1 == o.b1 && swz == o.swz && dev == o.dev;
  }
};
struct MapEntry { MapKey key; CUtensorMap map; };
std::vector<MapEntry> g_maps;
size_t g_map_next = 0;
constexpr size_t kMapCache = 64;

// 2-D row-major tensor: dim0 (inner, contiguous) x dim1 rows with pitch ld_bytes.
int get_map(CUtensorMap* out, const void* ptr, CUtensorMapDataType dt, int elem_bytes,
            unsigned long long inner, unsigned long long rows, unsigned long long ld_bytes,
            unsigned box_inner, unsigned box_rows, int swizzle /*0 none, 1 = 128B, 2 = 128B atom 32B, 3 = 64B*/) {
  MapKey key{ptr, (int)dt, inner, rows, ld_bytes, box_inner, box_rows, swizzle, t_ctx->dev};
  std::lock_guard<std::mutex> lk(g_mu);
  for (auto& e : g_maps)
    if (e.key == key) { *out = e.map; return 0; }
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {ld_bytes};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMap m;
  CUresult r = g_encode(&m, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE,
                        swizzle == 1 ? CU_TENSOR_MAP_SWIZZLE_128B
                        : swizzle == 2 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B
                        : swizzle == 3 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  (void)elem_bytes;
  if (r != CUDA_SUCCESS) return B200_ERR_TENSORMAP;
  if (g_maps.size() < kMapCache) g_maps.push_back({key, m});
  else { g_maps[g_map_next] = {key, m}; g_map_next = (g_map_next + 1) % kMapCache; }
  *out = m;
  return 0;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int check_args(int m, int n, int k, const void* A, int lda, const void* B, int ldb, const void* C, int ldc) {
  if (m < 0 || n < 0 || k < 0) return B200_ERR_BAD_ARG;
  if (m == 0 || n == 0) return 1;            // nothing to do
  if (!C || ldc < n) return B200_ERR_BAD_ARG;
  if (k > 0 && (!A || !B || lda < k || ldb < n)) return B200_ERR_BAD_ARG;
  return 0;
}

int last_launch_status() {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
  return 0;
}

// Launch with the programmatic-serialisation (PDL) attribute: the kernel may start while the previous kernel of
// the stream drains; every kernel launched through here calls griddep_wait before it touches global memory.
int g_pdl = 1;                // tuning hook (b200_gemm_debug_set_pdl)
int g_prepass_fork = 1;       // F16X2: B's pre-pass chain on an auxiliary stream beside A's (b200_gemm_debug_set_pdl bit 1 = off)
int g_dynamic_sched = 0;      // 1: every tensor-core launch draws its tiles from an atomic counter (b200_gemm_debug_set_dynamic_sched).  Default: static
                              // round robin (measured 0-8 % faster when the GPU is ours alone) except where t_dynamic_sched asks for it
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[2];
  int n = 0;
  if (cluster > 1) {
    at[n].id = cudaLaunchAttributeClusterDimension;
    at[n].val.clusterDim.x = cluster; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
    n++;
  }
  if (g_pdl) {
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    n++;
  }
  cfg.attrs = at; cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

template <typename T>
int launch_zero(int m, int n, T* C, int ldc, cudaStream_t st) {
  dim3 grid((n + 255) / 256, m < 4096 ? m : 4096);
  fill_zero_kernel<T><<<grid, 256, 0, st>>>(m, n, C, ldc);
  g_launches++;
  t_last_kernel = "fill_zero";
  t_last_sched.clear();
  return last_launch_status();
}

template <typename InT, typename OutT>
int launch_generic(int m, int n, int k, const InT* A, int lda, const InT* B, int ldb, OutT* C, int ldc,
                   int accumulate, cudaStream_t st, const char* name) {
  dim3 grid((n + 63) / 64, (m + 63) / 64);
  gemm_generic_kernel<InT, OutT><<<grid, 256, 0, st>>>(m, n, k, A, lda, B, ldb, C, ldc, accumulate);
  g_launches++;
  t_last_kernel = name;
  t_last_sched.clear();
  return last_launch_status();
}

int launch_generic_requant(int m, int n, int k, const int8_t* A, int lda, const int8_t* B, int ldb, int8_t* C,
                           int ldc, const float* scales, const float* bias, cudaStream_t st) {
  dim3 grid((n + 63) / 64, (m + 63) / 64);
  gemm_generic_kernel<int8_t, int8_t><<<grid, 256, 0, st>>>(m, n, k, A, lda, B, ldb, C, ldc, 0, scales, bias);
  g_launches++;
  t_last_kernel = "generic_s8_requant_64x64";
  t_last_sched.clear();
  return last_launch_status();
}

// ---- tensor-core launch -------------------------------------------------------------------
int g_force_bn = 0;          // test/tuning hook (b200_gemm_debug_set_bn): 0 = heuristic
int g_group_rows = 0;         // tuning hook: rows per raster group of the tensor-core kernels (0 = 2048)
int g_force_cg = 0;           // test/tuning hook (b200_gemm_debug_set_cta_group): 0 = auto, 1, 2
int g_epi8 = 1;               // pair kernels of the plain kinds drain with 8 epilogue warps (tuning hook b200_gemm_debug_set_epilogue bit 1 = back to 4):
                              // measured int8 4096^3 2.07 -> 2.32 POP/s, bf16->fp32 2304^3 692 -> 823 TFLOP/s, bit-identical results
constexpr int kStreamCDefault = 0;
int g_stream_c = -1;          // split modes: streaming stores for C (-1 = unresolved: B200GEMM_STREAM_C or the default above)
int g_epi_direct = 0;         // tuning hook (b200_gemm_debug_set_epilogue): 1 = direct register stores for non-folding passes
int g_ffma_fat = -1;          // strict kernel: 1 = 128x256 fat-thread variant, 0 = 128x128, -1 = by size
int g_ffma_halves = 1;        // strict kernel: split the tail round into half tiles (tuning hook)

template <int KIND, int BN, int STAGES, typename OutT, class Prod = ProdSingle, int A_ROW_BYTES = 128, int CG = 1, int EPIW = 4>
int launch_tc(int m, int n, int k, const void* A, long long lda, int a_rows_total, int a_plane_rows,
              const void* B, long long ldb, int b_rows_total, int b_plane_rows, void* C, int ldc,
              cudaStream_t st, const char* name, int chunk_k = 0, const float* row_max = nullptr,
              const float* col_max = nullptr, int accumulate = 0) {
  using Cfg = TcConfig<KIND, BN, STAGES, Prod, A_ROW_BYTES, CG, EPIW>;
  using T = KindTraits<KIND>;
  constexpr CUtensorMapDataType dt = KIND == KIND_F16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                   : KIND == KIND_FP16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                   : KIND == KIND_TF32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                                       : CU_TENSOR_MAP_DATA_TYPE_UINT8;
  CUtensorMap tmA, tmB;
  int rc = get_map(&tmA, A, dt, T::ELEM, k, a_rows_total, (unsigned long long)lda * T::ELEM, Cfg::BK, Cfg::BM,
                   A_ROW_BYTES == 128 ? 1 : 3);
  if (rc) return rc;
  rc = get_map(&tmB, B, dt, T::ELEM, n, b_rows_total, (unsigned long long)ldb * T::ELEM, Cfg::B_BOX_COLS, Cfg::BK,
               T::B_LAYOUT == 1 ? 2 : 1);
  if (rc) return rc;
  TcParams p;
  p.C = C; p.ldc = ldc; p.M = m; p.N = n; p.K = k;
  p.tiles_m = (m + Cfg::TILE_M - 1) / Cfg::TILE_M;
  p.tiles_n = (n + BN - 1) / BN;
  p.group_m = (g_group_rows > 0 ? g_group_rows : 2048) / Cfg::TILE_M;     // rows of A per raster group
  if (p.group_m < 1) p.group_m = 1;
  constexpr int OB = OutBytes<OutT>::V;
  p.vec_ok = aligned16(C) && ((long long)ldc * OB) % 16 == 0;
  p.a_plane_rows = a_plane_rows; p.b_plane_rows = b_plane_rows;
  p.chunk_kb = chunk_k > 0 ? (chunk_k + Cfg::BK - 1) / Cfg::BK : (k + Cfg::BK - 1) / Cfg::BK;
  if (p.chunk_kb < 1) p.chunk_kb = 1;
  p.dbg_b_lbo = g_dbg_b_lbo; p.dbg_b_sbo = g_dbg_b_sbo;
  p.row_max = row_max; p.col_max = col_max;
  p.accumulate = accumulate;
  p.axpby = t_epi.axpby; p.alpha = t_epi.alpha; p.beta = t_epi.beta;
  p.epi_direct = g_epi_direct;
  p.stream_c = g_stream_c < 0 ? (g_stream_c = (getenv("B200GEMM_STREAM_C") ? atoi(getenv("B200GEMM_STREAM_C")) : kStreamCDefault)) : g_stream_c;
  auto kern = gemm_tc_kernel<KIND, BN, STAGES, OutT, Prod, A_ROW_BYTES, CG, EPIW>;
  if (int arc = ensure_smem_attr(kern, Cfg::SMEM_BYTES)) return arc;
  int tiles = p.tiles_m * p.tiles_n;
  const int units_max = (t_ctx->sms - t_sm_reserve > 2 * CG ? t_ctx->sms - t_sm_reserve : t_ctx->sms) / CG;   // CTAs, or CTA pairs (one per TPC)
  // Wave quantisation: the last, partial round of tiles (or the only round of a small problem) is
  // cut along K so that every CTA/pair has work: rem tiles x split parts <= units.
  const int num_kb = (k + Cfg::BK - 1) / Cfg::BK;
  const int rem = tiles % units_max;
  int split = 1;
  if (g_split_tail && OB == 4 && rem > 0) {
    split = units_max / rem;
    if (split > 4) split = 4;
    if (split > num_kb / 8) split = num_kb / 8;       // keep >= 8 k-blocks per part
    if (split < 1) split = 1;
    if (rem * CG * Cfg::EPI_WARPS > 1024) split = 1;  // flag slot capacity
  }
  // When at least one full round exists, the partial last round is better served by half-width tiles
  // (no K split, no fold): 2*rem items of half the duration.  Needs BN/2 to be a whole number of
  // B column blocks per CTA.
  p.halfn = 0;
  if (g_split_tail == 1 && tiles >= units_max && rem > 0 && 2 * rem <= units_max &&
      ((BN / 2 / CG) % Cfg::B_BOX_COLS) == 0 && (BN / 2) % 16 == 0 && (BN / 2) % OutPack<OutT>::COLS == 0) {
    p.halfn = 1;
    split = 1;
  }
  p.split = split;
  p.full_tiles = (split > 1 || p.halfn) ? tiles - rem : tiles;
  p.flags = t_ctx->flags + (t_ctx->flag_slot++ % 16) * 1024;
  p.sched_counter = (g_dynamic_sched || t_dynamic_sched) ? t_ctx->sched_counters + (t_ctx->sched_slot++ % 64) : nullptr;
  if (split > 1) {          // the ordering flags start from zero whatever an aborted earlier launch left behind
    cudaError_t e = cudaMemsetAsync(p.flags, 0, 1024 * sizeof(int), st);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
  }
  const int items = p.full_tiles + (tiles - p.full_tiles) * (p.halfn ? 2 : split);
  const int units = items < units_max ? items : units_max;
  g_ktimer.begin(st);
  {
    cudaError_t e = launch_pdl(kern, dim3(units * CG), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, st, CG, tmA, tmB, p);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
  }
  g_ktimer.end(st);
  g_launches++;
  t_last_kernel = name;
  t_last_sched.set(Cfg::TILE_M, BN, CG, Cfg::EPI_WARPS, tiles, units, p.full_tiles, split, p.halfn, p.sched_counter != nullptr);
  return last_launch_status();
}

// Tile width: fewest "wave x tile-time" units over the persistent grid (tile time ~ BN plus a
// fixed per-tile cost); 128 x 256 has the best operand reuse, narrower tiles quantise better.
int pick_bn(int m, int n, bool allow256, bool allow192 = true) {
  if (g_force_bn == 128 || (g_force_bn == 192 && allow192) || (g_force_bn == 256 && allow256)) return g_force_bn;
  const int cands[3] = {256, 192, 128};
  // relative efficiency of the 1-CTA kernels, measured on B200 at N=4096 (bf16: 1347 / 1317 / 1058
  // TFLOP/s; the CTA-pair kernel: 1538): narrower tiles amortise shared-memory operand reads worse
  const double eff[3] = {1.00, 0.97, 0.80};
  int best = 128;
  double best_cost = 1e300;
  const int tm = (m + 127) / 128;
  for (int i = 0; i < 3; i++) {
    if (cands[i] == 256 && !allow256) continue;
    if (cands[i] == 192 && !allow192) continue;
    const long long tiles = (long long)tm * ((n + cands[i] - 1) / cands[i]);
    const long long waves = (tiles + t_ctx->sms - 1) / t_ctx->sms;
    const double cost = (double)waves * (cands[i] / eff[i] + 8.0);
    if (cost < best_cost) { best_cost = cost; best = cands[i]; }
  }
  return best;
}

// CTA pairs (tcgen05 cta_group::2, 256 x BN per pair): each CTA stages only its half of B, halving the
// shared-memory operand traffic per MMA that bounds the 1-CTA kernel (1538 vs 1347 TFLOP/s, bf16 4096^3).
// Used once the 256 x 256 pair tiles fill most of the 74 pairs; below that the 1-CTA tiles fill the
// machine better (N = 1536, BF16X3: 128x128 tiles 143 TFLOP/s, pair tiles 95).
bool use_pair(int m, int n) {
  if (g_force_cg == 1) return false;
  if (g_force_cg == 2) return m > 128 && n > 128;
  if (m <= 128 || n <= 128) return false;
  const long long tiles = (long long)((m + 255) / 256) * ((n + 255) / 256);
  return tiles * 5 >= (long long)(t_ctx->sms / 2) * 4;
}

#define TC_PLAIN(KIND, OUT, NAME)                                                                     \
  if (use_pair(m, n) && g_epi8)                                                                       \
    return launch_tc<KIND, 256, 6, OUT, ProdSingle, 128, 2, 8>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, NAME "_2cta_256x256_e8"); \
  if (use_pair(m, n))                                                                                 \
    return launch_tc<KIND, 256, 6, OUT, ProdSingle, 128, 2>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, NAME "_2cta_256x256"); \
  switch (pick_bn(m, n, true)) {                                                                      \
    case 256: return launch_tc<KIND, 256, 4, OUT>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, NAME "_128x256"); \
    case 192: return launch_tc<KIND, 192, 5, OUT>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, NAME "_128x192"); \
    default:  return launch_tc<KIND, 128, 6, OUT>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, NAME "_128x128"); \
  }

int tc_tf32(int m, int n, int k, const float* A, int lda, const float* B, int ldb, float* C, int ldc, cudaStream_t st, int acc = 0) {
  if (use_pair(m, n) && g_epi8)
    return launch_tc<KIND_TF32, 256, 6, float, ProdSingle, 128, 2, 8>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_tf32_2cta_256x256_e8", 0, nullptr, nullptr, acc);
  if (use_pair(m, n))
    return launch_tc<KIND_TF32, 256, 6, float, ProdSingle, 128, 2>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_tf32_2cta_256x256", 0, nullptr, nullptr, acc);
  switch (pick_bn(m, n, true)) {
    case 256: return launch_tc<KIND_TF32, 256, 4, float>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_tf32_128x256", 0, nullptr, nullptr, acc);
    case 192: return launch_tc<KIND_TF32, 192, 5, float>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_tf32_128x192", 0, nullptr, nullptr, acc);
    default:  return launch_tc<KIND_TF32, 128, 6, float>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_tf32_128x128", 0, nullptr, nullptr, acc);
  }
}
int tc_bf16_f32(int m, int n, int k, const void* A, int lda, const void* B, int ldb, void* C, int ldc, cudaStream_t st) {
  TC_PLAIN(KIND_F16, float, "tc_bf16")
}
int tc_bf16_bf16(int m, int n, int k, const void* A, int lda, const void* B, int ldb, void* C, int ldc, cudaStream_t st) {
  TC_PLAIN(KIND_F16, bf16_out, "tc_bf16_obf16")
}
int tc_s8(int m, int n, int k, const void* A, int lda, const void* B, int ldb, void* C, int ldc, cudaStream_t st) {
  // int8 column blocks are 128 elements wide (128 B): BN = 192 is not a whole number of them
  if (use_pair(m, n) && g_epi8)
    return launch_tc<KIND_I8, 256, 6, int32_t, ProdSingle, 128, 2, 8>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_s8_2cta_256x256_e8");
  if (use_pair(m, n))
    return launch_tc<KIND_I8, 256, 6, int32_t, ProdSingle, 128, 2>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_s8_2cta_256x256");
  if (pick_bn(m, n, true, false) == 256)
    return launch_tc<KIND_I8, 256, 4, int32_t>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_s8_128x256");
  return launch_tc<KIND_I8, 128, 6, int32_t>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_s8_128x128");
}

// int8 in, int8 out through the requantising epilogue (scales / bias ride in the row_max / col_max slots)
int tc_s8_requant(int m, int n, int k, const void* A, int lda, const void* B, int ldb, void* C, int ldc,
                  const float* scales, const float* bias, cudaStream_t st) {
  if (use_pair(m, n) && g_epi8)
    return launch_tc<KIND_I8, 256, 6, s8_out, ProdSingle, 128, 2, 8>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_s8_requant_2cta_256x256_e8", 0, scales, bias);
  if (use_pair(m, n))
    return launch_tc<KIND_I8, 256, 6, s8_out, ProdSingle, 128, 2>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_s8_requant_2cta_256x256", 0, scales, bias);
  if (pick_bn(m, n, true, false) == 256)
    return launch_tc<KIND_I8, 256, 4, s8_out>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_s8_requant_128x256", 0, scales, bias);
  return launch_tc<KIND_I8, 128, 6, s8_out>(m, n, k, A, lda, m, 0, B, ldb, k, 0, C, ldc, st, "tc_s8_requant_128x128", 0, scales, bias);
}

// ---- split-precision fp32 on the tensor cores ---------------------------------------------------
// Workspace for the bf16 planes: cached, grow-only (no per-call cudaMalloc in steady state).  Calls
// in split modes are serialised on this buffer by stream order; use one stream per library instance.
// K extent accumulated inside the tensor core before folding into C (0 = whole K): [0] BF16X3, [1] BF16X2
constexpr int kSplitChunkDefault[3] = {512, 512, 1024};   // BF16X3, BF16X2, F16X2
int g_split_chunk_k[3] = {kSplitChunkDefault[0], kSplitChunkDefault[1], kSplitChunkDefault[2]};
// Grows the device's split workspace to `need` bytes.  Starts at 256 MiB (every size of the reference's
// 256..4096 sweep fits: its harness averages the first, cold call into each row, and a cudaFree +
// cudaMalloc there costs tens of ms) and at least doubles.  Growth synchronises the device (other
// streams may still read the old buffer); steady-state calls never allocate.  Caller holds ws_mu.
int split_ws_reserve(size_t need) {
  DevCtx* c = t_ctx;
  if (c->ws.bytes >= need) return B200_OK;
  size_t want = c->ws.bytes ? 2 * c->ws.bytes : ((size_t)256 << 20);
  if (want < need) want = need;
  if (c->ws.p) { cudaDeviceSynchronize(); cudaFree(c->ws.p); }
  c->ws.p = nullptr; c->ws.bytes = 0; c->ws_busy = false;
  cudaError_t e = cudaMalloc(&c->ws.p, want);
  if (e != cudaSuccess && want > need) { cudaGetLastError(); want = need; e = cudaMalloc(&c->ws.p, want); }
  if (e != cudaSuccess) { cudaGetLastError(); c->ws.p = nullptr; return (int)e; }
  c->ws.bytes = want;
  return B200_OK;
}
// Stream ordering of workspace users: a call on a stream other than the last user's waits (on the device)
// for that user's GEMM; ws_release records the event the next foreign-stream user will wait on.
void ws_acquire(cudaStream_t st) {
  DevCtx* c = t_ctx;
  if (c->ws_busy && c->ws_stream != st) cudaStreamWaitEvent(st, c->ws_event, 0);
}
void ws_release(cudaStream_t st) {
  DevCtx* c = t_ctx;
  cudaEventRecord(c->ws_event, st);
  c->ws_stream = st;
  c->ws_busy = true;
}

// Plane geometry shared by the per-call pre-pass and the pre-split B handle (b200_gemm_f32_pack_b).
inline long long plane_pitch(int cols) { return ((long long)cols + 7) & ~7LL; }   // elements, 16-byte multiple
inline int b_plane_rows(int k) { return (k + 31) & ~31; }                           // zero rows pad K to the k-block

// Splits one operand (jobs == 1) or both (jobs == 2) in a single launch.
template <int NP>
int launch_split(const SplitJob& ja, const SplitJob& jb, int jobs, cudaStream_t st) {
  const long long wide = jobs == 2 && jb.dld > ja.dld ? jb.dld : ja.dld;
  const int tall = jobs == 2 && jb.plane_rows > ja.plane_rows ? jb.plane_rows : ja.plane_rows;
  const int gx = (int)((wide + 2047) / 2048);
  int gy = (t_ctx->sms * 8 + jobs * gx - 1) / (jobs * gx);        // ~8 blocks per SM over the launch
  if (gy > (tall + 1) / 2) gy = (tall + 1) / 2;
  if (gy < 1) gy = 1;
  launch_pdl(split_planes_kernel<NP>, dim3(gx, gy, jobs), dim3(256), 0, st, 1, ja, jb);
  g_launches += 1;
  return last_launch_status();
}

// prepB: bf16 planes of B split earlier by b200_gemm_f32_pack_b (then only A is split here), or null.
template <int NP>
int gemm_f32_split(int m, int n, int k, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                   cudaStream_t st, int acc = 0, const uint16_t* prepB = nullptr) {
  const long long pka = plane_pitch(k), pnb = plane_pitch(n);
  const int kp = b_plane_rows(k);
  const size_t a_bytes = (size_t)NP * m * pka * 2, b_bytes = (size_t)NP * kp * pnb * 2;
  const size_t a_off = (a_bytes + 1023) & ~(size_t)1023;
  std::lock_guard<std::mutex> wlk(t_ctx->ws_mu);
  if (int rc = split_ws_reserve(prepB ? a_off : a_off + b_bytes)) return rc;
  ws_acquire(st);
  struct Release { cudaStream_t s; ~Release() { ws_release(s); } } rel{st};
  uint16_t* pA = reinterpret_cast<uint16_t*>(t_ctx->ws.p);
  const uint16_t* pB = prepB ? prepB
                             : reinterpret_cast<uint16_t*>(reinterpret_cast<uint8_t*>(t_ctx->ws.p) + a_off);
  const SplitJob ja{A, lda, m, k, pA, pka, m}, jb{B, ldb, k, n, const_cast<uint16_t*>(pB), pnb, kp};
  int rc = launch_split<NP>(ja, jb, prepB ? 1 : 2, st);
  if (rc) return rc;
  if (use_pair(m, n)) {
    if constexpr (NP == 3)
      return launch_tc<KIND_F16, 256, 4, float, ProdX3, 64, 2>(m, n, k, pA, pka, NP * m, m, pB, pnb, NP * kp, kp, C, ldc, st, "tc_bf16x3_2cta_256x256", g_split_chunk_k[0], nullptr, nullptr, acc);
    else
      return launch_tc<KIND_F16, 256, 6, float, ProdX2, 64, 2>(m, n, k, pA, pka, NP * m, m, pB, pnb, NP * kp, kp, C, ldc, st, "tc_bf16x2_2cta_256x256", g_split_chunk_k[1], nullptr, nullptr, acc);
  }
  const int bn = pick_bn(m, n, NP == 2);
  if constexpr (NP == 3) {
    if (bn == 192)
      return launch_tc<KIND_F16, 192, 3, float, ProdX3, 64>(m, n, k, pA, pka, NP * m, m, pB, pnb, NP * kp, kp, C, ldc, st, "tc_bf16x3_128x192", g_split_chunk_k[0], nullptr, nullptr, acc);
    return launch_tc<KIND_F16, 128, 4, float, ProdX3, 64>(m, n, k, pA, pka, NP * m, m, pB, pnb, NP * kp, kp, C, ldc, st, "tc_bf16x3_128x128", g_split_chunk_k[0], nullptr, nullptr, acc);
  } else {
    if (bn == 256)
      return launch_tc<KIND_F16, 256, 4, float, ProdX2, 64>(m, n, k, pA, pka, NP * m, m, pB, pnb, NP * kp, kp, C, ldc, st, "tc_bf16x2_128x256", g_split_chunk_k[1], nullptr, nullptr, acc);
    if (bn == 192)
      return launch_tc<KIND_F16, 192, 4, float, ProdX2, 64>(m, n, k, pA, pka, NP * m, m, pB, pnb, NP * kp, kp, C, ldc, st, "tc_bf16x2_128x192", g_split_chunk_k[1], nullptr, nullptr, acc);
    return launch_tc<KIND_F16, 128, 6, float, ProdX2, 64>(m, n, k, pA, pka, NP * m, m, pB, pnb, NP * kp, kp, C, ldc, st, "tc_bf16x2_128x128", g_split_chunk_k[1], nullptr, nullptr, acc);
  }
}

// B200_F32_F16X2: scaled fp16 split, 3 products.  Row maxima of A and column maxima of B give exact
// power-of-two scalings that bring every operand into [-1, 1] (fp16 has 5 exponent bits); the
// epilogue multiplies them back.  Launches: rows of A (max + scale + split fused), column maxima of B,
// columns of B, GEMM.
struct F16Operand {           // one operand as two stacked fp16 planes + the maxima its scaling came from
  const uint16_t* planes;     // plane p at row p * plane_rows
  long long pitch;            // elements (multiple of 8)
  int plane_rows;
  const float* maxv;          // [rows of A] / [columns of B]
};
inline long long f16_pitch(int cols) { return ((long long)cols + 7) & ~7LL; }
inline int f16_b_rows(int k) { return (k + 31) & ~31; }

// A (rows x cols, scaled by row) -> planes + rmax.  One launch, each row read from HBM once.
int launch_f16_split_rows(const float* A, long long lda, int rows, int cols, float* rmax, uint16_t* planes,
                          long long pitch, int plane_rows, cudaStream_t st) {
  int blocks = (plane_rows + 7) / 8;                       // one warp per row, 8 rows per block
  const int cap = t_ctx->sms * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (cols <= 1024) launch_pdl(split_f16_rows_kernel<4>, dim3(blocks), dim3(256), 0, st, 1, A, (long long)lda, rows, cols, rmax, planes, pitch, plane_rows);
  else if (cols <= 2048) launch_pdl(split_f16_rows_kernel<8>, dim3(blocks), dim3(256), 0, st, 1, A, (long long)lda, rows, cols, rmax, planes, pitch, plane_rows);
  else if (cols <= 4096) launch_pdl(split_f16_rows_kernel<16>, dim3(blocks), dim3(256), 0, st, 1, A, (long long)lda, rows, cols, rmax, planes, pitch, plane_rows);
  else launch_pdl(split_f16_rows_kernel<0>, dim3(blocks), dim3(256), 0, st, 1, A, (long long)lda, rows, cols, rmax, planes, pitch, plane_rows);
  g_launches++;
  return last_launch_status();
}

// B (rows x cols, scaled by column) -> planes + cmax (must be zero on entry).  Two launches.  zero_buf:
// another buffer to clear on the way (the idle half of the double-buffered maxima), or null.
int launch_f16_split_cols(const float* B, long long ldb, int rows, int cols, float* cmax, uint16_t* planes,
                          long long pitch, int plane_rows, float* zero_buf, int zero_n, cudaStream_t st) {
  launch_pdl(col_absmax_kernel, dim3((cols + 1023) / 1024, (rows + 15) / 16), dim3(256), 0, st, 1, B, (long long)ldb, rows, cols,
             reinterpret_cast<unsigned int*>(cmax));
  const int gx = (int)((pitch + 2047) / 2048);
  int gy = (t_ctx->sms * 8 + gx - 1) / gx;
  if (gy > (plane_rows + 1) / 2) gy = (plane_rows + 1) / 2;
  if (gy < 1) gy = 1;
  if (zero_buf && zero_n > gx * 2048) {                    // wider than this launch covers: clear it separately
    cudaMemsetAsync(zero_buf, 0, (size_t)zero_n * 4, st);
    zero_buf = nullptr;
  }
  launch_pdl(split_f16_cols_kernel, dim3(gx, gy), dim3(256), 0, st, 1, B, (long long)ldb, rows, cols, (const float*)cmax, planes, pitch, plane_rows, zero_buf, zero_n);
  g_launches += 2;
  return last_launch_status();
}

int gemm_f16x2_core(int m, int n, int k, const F16Operand& a, const F16Operand& b, float* C, int ldc, int acc,
                    cudaStream_t st) {
  constexpr int NP = 2;
  if (use_pair(m, n))
    return launch_tc<KIND_FP16, 256, 6, float, ProdX2, 64, 2>(m, n, k, a.planes, a.pitch, NP * a.plane_rows, a.plane_rows,
                                                              b.planes, b.pitch, NP * b.plane_rows, b.plane_rows, C, ldc, st,
                                                              "tc_f16x2_2cta_256x256", g_split_chunk_k[2], a.maxv, b.maxv, acc);
  const int bn = pick_bn(m, n, true);
  if (bn == 256)
    return launch_tc<KIND_FP16, 256, 4, float, ProdX2, 64>(m, n, k, a.planes, a.pitch, NP * a.plane_rows, a.plane_rows,
                                                           b.planes, b.pitch, NP * b.plane_rows, b.plane_rows, C, ldc, st,
                                                           "tc_f16x2_128x256", g_split_chunk_k[2], a.maxv, b.maxv, acc);
  if (bn == 192)
    return launch_tc<KIND_FP16, 192, 4, float, ProdX2, 64>(m, n, k, a.planes, a.pitch, NP * a.plane_rows, a.plane_rows,
                                                           b.planes, b.pitch, NP * b.plane_rows, b.plane_rows, C, ldc, st,
                                                           "tc_f16x2_128x192", g_split_chunk_k[2], a.maxv, b.maxv, acc);
  return launch_tc<KIND_FP16, 128, 6, float, ProdX2, 64>(m, n, k, a.planes, a.pitch, NP * a.plane_rows, a.plane_rows,
                                                         b.planes, b.pitch, NP * b.plane_rows, b.plane_rows, C, ldc, st,
                                                         "tc_f16x2_128x128", g_split_chunk_k[2], a.maxv, b.maxv, acc);
}

// Column maxima are double-buffered outside the grow-only workspace: call i accumulates into half i % 2
// (atomicMax needs zeros) and its split launch re-zeroes the other half for call i + 1.
int cmax_reserve(int n, float** cur, float** other, int* other_dirty) {
  DevCtx* c = t_ctx;
  if (c->cmax_cap < (size_t)n) {
    size_t cap = c->cmax_cap ? 2 * c->cmax_cap : 16384;
    if (cap < (size_t)n) cap = (size_t)n;
    if (c->cmax_buf) { cudaDeviceSynchronize(); cudaFree(c->cmax_buf); }
    c->cmax_buf = nullptr; c->cmax_cap = 0;
    cudaError_t e = cudaMalloc(&c->cmax_buf, 2 * cap * sizeof(float));
    if (e == cudaSuccess) e = cudaMemset(c->cmax_buf, 0, 2 * cap * sizeof(float));
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    c->cmax_cap = cap;
    c->cmax_dirty[0] = c->cmax_dirty[1] = 0;
  }
  const unsigned slot = c->cmax_slot++ & 1u;
  *cur = c->cmax_buf + slot * c->cmax_cap;
  *other = c->cmax_buf + (slot ^ 1u) * c->cmax_cap;
  *other_dirty = c->cmax_dirty[slot ^ 1u];
  c->cmax_dirty[slot ^ 1u] = 0;
  c->cmax_dirty[slot] = n;
  return 0;
}

// prepA / prepB: operands split earlier (b200_gemm_f32_pack_a / _pack_b), or null = split here.
int gemm_f32_split_f16(int m, int n, int k, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                       cudaStream_t st, int acc = 0, const F16Operand* prepA = nullptr, const F16Operand* prepB = nullptr) {
  constexpr int NP = 2;
  const long long pka = f16_pitch(k), pnb = f16_pitch(n);
  const int kp = f16_b_rows(k);
  const size_t a_bytes = prepA ? 0 : (size_t)NP * m * pka * 2, b_bytes = prepB ? 0 : (size_t)NP * kp * pnb * 2;
  const size_t a_off = (a_bytes + 1023) & ~(size_t)1023;
  const size_t r_off = (a_off + b_bytes + 1023) & ~(size_t)1023;       // row maxima
  const size_t total = r_off + (prepA ? 0 : (size_t)m * 4);
  F16Operand oa, ob;
  if (prepA && prepB) return gemm_f16x2_core(m, n, k, *prepA, *prepB, C, ldc, acc, st);
  std::lock_guard<std::mutex> wlk(t_ctx->ws_mu);
  if (int rc = split_ws_reserve(total)) return rc;
  ws_acquire(st);
  struct Release { cudaStream_t s; ~Release() { ws_release(s); } } rel{st};
  uint8_t* base = reinterpret_cast<uint8_t*>(t_ctx->ws.p);
  // Neither pre-pass kernel saturates HBM on its own (ncu: 37-52 % of peak DRAM throughput each), and A's and B's
  // chains are independent: when both operands are split here, B's chain (column maxima, split) runs on the
  // context's auxiliary stream beside A's row split and joins before the GEMM.
  DevCtx* c = t_ctx;
  const bool fork = !prepA && !prepB && g_prepass_fork && (double)m * k + (double)k * n >= 4.0e6;
  cudaStream_t sb = st;
  if (fork) {
    if (!c->aux) {
      if (cudaStreamCreateWithFlags(&c->aux, cudaStreamNonBlocking) != cudaSuccess ||
          cudaEventCreateWithFlags(&c->aux_fork, cudaEventDisableTiming) != cudaSuccess ||
          cudaEventCreateWithFlags(&c->aux_join, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return B200_ERR_NO_DEVICE; }
    }
    cudaEventRecord(c->aux_fork, st);
    cudaStreamWaitEvent(c->aux, c->aux_fork, 0);
    sb = c->aux;
  }
  if (prepB) ob = *prepB;
  else {
    uint16_t* pB = reinterpret_cast<uint16_t*>(base + a_off);
    float *cmax, *other;
    int other_dirty;
    if (int rc = cmax_reserve(n, &cmax, &other, &other_dirty)) return rc;
    if (int rc = launch_f16_split_cols(B, ldb, k, n, cmax, pB, pnb, kp, other, other_dirty, sb)) return rc;
    ob = F16Operand{pB, pnb, kp, cmax};
  }
  if (prepA) oa = *prepA;
  else {
    uint16_t* pA = reinterpret_cast<uint16_t*>(base);
    float* rmax = reinterpret_cast<float*>(base + r_off);
    if (int rc = launch_f16_split_rows(A, lda, m, k, rmax, pA, pka, m, st)) return rc;
    oa = F16Operand{pA, pka, m, rmax};
  }
  if (fork) {
    cudaEventRecord(c->aux_join, c->aux);
    cudaStreamWaitEvent(st, c->aux_join, 0);
  }
  return gemm_f16x2_core(m, n, k, oa, ob, C, ldc, acc, st);
}

int launch_ffma(int m, int n, int k, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                int accumulate, cudaStream_t st) {
  using Cfg = FfmaCfg;
  CUtensorMap tmA, tmB;
  int rc = get_map(&tmA, A, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, k, m, (unsigned long long)lda * 4, Cfg::BK, Cfg::BM, 1);
  if (rc) return rc;
  rc = get_map(&tmB, B, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, n, k, (unsigned long long)ldb * 4, Cfg::BN, Cfg::BK, 0);
  if (rc) return rc;
  FfmaParams p;
  p.C = C; p.ldc = ldc; p.M = m; p.N = n; p.K = k;
  p.vec_ok = aligned16(C) && (ldc % 4) == 0;
  p.accumulate = accumulate;
  p.tiles_m = (m + Cfg::BM - 1) / Cfg::BM;
  p.tiles_n = (n + Cfg::BN - 1) / Cfg::BN;
  p.group_m = 8;
  // 2 CTAs per SM: tiles of the last, at most half-full round are issued as two half tiles each
  const int tiles = p.tiles_m * p.tiles_n, slots = 2 * t_ctx->sms;
  const int rem = tiles % slots;
  const bool halves = g_ffma_halves && rem > 0 && 2 * rem <= slots;
  p.full_tiles = halves ? tiles - rem : tiles;
  const int ctas = p.full_tiles + 2 * (tiles - p.full_tiles);
  if (int arc = ensure_smem_attr(gemm_ffma_kernel, Cfg::SMEM_BYTES)) return arc;
  g_ktimer.begin(st);
  gemm_ffma_kernel<<<ctas, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(tmA, tmB, p);
  g_ktimer.end(st);
  g_launches++;
  t_last_kernel = "ffma_128x128x32_tma";
  t_last_sched.set(Cfg::BM, Cfg::BN, 1, 0, tiles, ctas, p.full_tiles, 1, halves, 0);
  return last_launch_status();
}

int launch_ffma_fat(int m, int n, int k, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                int accumulate, cudaStream_t st) {
  using Cfg = FfmaFatCfg;
  CUtensorMap tmA, tmB;
  int rc = get_map(&tmA, A, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, k, m, (unsigned long long)lda * 4, Cfg::BK, Cfg::BM, 1);
  if (rc) return rc;
  rc = get_map(&tmB, B, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, n, k, (unsigned long long)ldb * 4, Cfg::BN, Cfg::BK, 0);
  if (rc) return rc;
  FfmaParams p;
  p.C = C; p.ldc = ldc; p.M = m; p.N = n; p.K = k;
  p.vec_ok = aligned16(C) && (ldc % 4) == 0;
  p.accumulate = accumulate;
  p.tiles_m = (m + Cfg::BM - 1) / Cfg::BM;
  p.tiles_n = (n + Cfg::BN - 1) / Cfg::BN;
  p.group_m = 8;
  // 1 CTA per SM: tiles of the last, at most half-full round are issued as two half tiles each
  const int tiles = p.tiles_m * p.tiles_n, slots = t_ctx->sms;
  const int rem = tiles % slots;
  const bool halves = g_ffma_halves && rem > 0 && 2 * rem <= slots;
  p.full_tiles = halves ? tiles - rem : tiles;
  const int ctas = p.full_tiles + 2 * (tiles - p.full_tiles);
  if (int arc = ensure_smem_attr(gemm_ffma_fat_kernel, Cfg::SMEM_BYTES)) return arc;
  g_ktimer.begin(st);
  gemm_ffma_fat_kernel<<<ctas, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(tmA, tmB, p);
  g_ktimer.end(st);
  g_launches++;
  t_last_kernel = "ffma_fat_128x256x32_tma";
  t_last_sched.set(Cfg::BM, Cfg::BN, 1, 0, tiles, ctas, p.full_tiles, 1, halves, 0);
  return last_launch_status();
}

bool tma_ok(const void* A, int lda, const void* B, int ldb, int elem) {
  return aligned16(A) && aligned16(B) && ((long long)lda * elem) % 16 == 0 && ((long long)ldb * elem) % 16 == 0;
}

int resolve_f32_mode(int mode) {
  if (mode == B200_F32_AUTO) {
    int d = g_default_f32_mode.load();
    if (d < 0) {
      const char* e = getenv("B200GEMM_F32_MODE");
      d = e ? atoi(e) : B200_F32_F16X2;
      if (d < 0 || d == B200_F32_AUTO || d > B200_F32_F16X2) d = B200_F32_F16X2;
      g_default_f32_mode.store(d);
    }
    return d;
  }
  return mode;
}

int gemm_f32_impl(int m, int n, int k, const float* dA, int lda, const float* dB, int ldb, float* dC,
                  int ldc, int mode, int accumulate, cudaStream_t st) {
  int rc = check_args(m, n, k, dA, lda, dB, ldb, dC, ldc);
  if (rc == 1) return 0;
  if (rc) return rc;
  rc = ensure_device();
  if (rc) return rc;
  if (k == 0) return accumulate ? 0 : launch_zero<float>(m, n, dC, ldc, st);
  const bool was_auto = mode == B200_F32_AUTO;
  mode = resolve_f32_mode(mode);
  const bool tma = tma_ok(dA, lda, dB, ldb, 4);
  // AUTO on a small problem: the split path costs two launches (pre-pass + GEMM); up to 512^3 the
  // single-launch strict FFMA2 kernel is within 15 % of it (measured, tools/probe_small.py: 9.3 vs 10.6
  // TFLOP/s at 512^3, 2.0 vs 2.0 at 256^3) and bit-exact against the reference oracle.  From 640^3 the
  // tensor-core path pulls away (19.2 vs 15.0; 63.0 vs 41.0 at 1024^3).
  if (was_auto && (mode == B200_F32_BF16X3 || mode == B200_F32_F16X2) && tma && (double)m * n * k <= 2.0e8) mode = B200_F32_STRICT;
  // AUTO between ~640^3 and ~1100^3: the two-launch BF16X3 path (one fused split + GEMM) beats the four-launch
  // F16X2 path while launches, not tensor work, dominate (tools/probe_crossover.py, TFLOP/s BF16X3 : F16X2 —
  // 768^3 23.6 : 20.1, 1024^3 61.5 : 53.4, 1152^3 98.5 : 98.7, 1536^3 170 : 193, 2048^3 201 : 252).  Both are fp32-class.
  else if (was_auto && mode == B200_F32_F16X2 && (double)m * n * k < 1.3e9) mode = B200_F32_BF16X3;
  switch (mode) {
    case B200_F32_STRICT:
      // 128x256 fat-thread tiles once they fill most of the machine (measured at N = 4096 / 3072 / 2048:
      // 58.9 / 57.7 / 50.8 TFLOP/s against 58.5 / 57.2 / 49.3 for 128x128; at 1024 the small tile wins 40.6 : 24.1)
      if (tma && (g_ffma_fat == 1 || (g_ffma_fat < 0 && (long long)((m + 127) / 128) * ((n + 255) / 256) >= 96)))
        return launch_ffma_fat(m, n, k, dA, lda, dB, ldb, dC, ldc, accumulate, st);
      if (tma) return launch_ffma(m, n, k, dA, lda, dB, ldb, dC, ldc, accumulate, st);
      return launch_generic<float, float>(m, n, k, dA, lda, dB, ldb, dC, ldc, accumulate, st, "generic_f32_64x64");
    case B200_F32_TF32:
      if (!tma) return launch_generic<float, float>(m, n, k, dA, lda, dB, ldb, dC, ldc, accumulate, st, "generic_f32_64x64");
      return tc_tf32(m, n, k, dA, lda, dB, ldb, dC, ldc, st, accumulate);
    case B200_F32_BF16X3:
      return gemm_f32_split<3>(m, n, k, dA, lda, dB, ldb, dC, ldc, st, accumulate);
    case B200_F32_BF16X2:
      return gemm_f32_split<2>(m, n, k, dA, lda, dB, ldb, dC, ldc, st, accumulate);
    case B200_F32_F16X2:
      return gemm_f32_split_f16(m, n, k, dA, lda, dB, ldb, dC, ldc, st, accumulate);
    default:
      return B200_ERR_UNSUPPORTED;
  }
}

}  // namespace

extern "C" {

const char* b200_gemm_version(void) { return "b200gemm 0.2 (sm_100a; tcgen05+TMA; round 2)"; }

int b200_gemm_device_ok(void) { return ensure_device(); }

const char* b200_gemm_strerror(int code) {
  switch (code) {
    case B200_OK: return "ok";
    case B200_ERR_BAD_ARG: return "bad argument";
    case B200_ERR_NO_DEVICE: return "no usable sm_100 CUDA device (there is no CPU fallback)";
    case B200_ERR_UNSUPPORTED: return "mode not supported for these operands";
    case B200_ERR_TENSORMAP: return "cuTensorMapEncodeTiled failed";
    case B200_ERR_NCCL: return "NCCL failure (b200_nccl_last_error has the text)";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown";
  }
}

const char* b200_gemm_last_kernel(void) { return t_last_kernel; }
unsigned long long b200_gemm_launch_count(void) { return g_launches.load(); }
int b200_gemm_default_f32_mode(void) { return resolve_f32_mode(B200_F32_AUTO); }
void b200_gemm_set_default_f32_mode(int mode) {
  if (mode >= 0 && mode != B200_F32_AUTO && mode <= B200_F32_F16X2) g_default_f32_mode.store(mode);
}
void b200_gemm_debug_set_b_desc(int lbo_bytes, int sbo_bytes) { g_dbg_b_lbo = lbo_bytes; g_dbg_b_sbo = sbo_bytes; }
void b200_gemm_debug_set_bn(int bn) { g_force_bn = bn; }
void b200_gemm_debug_set_pdl(int v) { g_pdl = (v & 1) != 0; g_prepass_fork = (v & 2) == 0; }
void b200_gemm_debug_set_dynamic_sched(int on) { g_dynamic_sched = on != 0; }
void b200_gemm_debug_set_cta_group(int cg) { g_force_cg = cg; }
void b200_gemm_debug_set_split_tail(int on) { g_split_tail = on; }
void b200_gemm_debug_set_epilogue(int v) { g_epi_direct = v & 1; g_epi8 = ((v >> 1) & 1) ^ 1; }
void b200_gemm_debug_set_group_rows(int rows) { g_group_rows = rows; }
void b200_gemm_debug_set_ffma_variant(int v) { g_ffma_halves = v & 1; g_ffma_fat = v < 0 ? -1 : (v >> 1) & 1; }
void b200_gemm_debug_set_split_chunk(int x3_k, int x2_k) {
  if (x3_k < 0 || x2_k < 0) {            // back to the built-in defaults, each mode its own
    g_split_chunk_k[0] = kSplitChunkDefault[0]; g_split_chunk_k[1] = kSplitChunkDefault[1]; g_split_chunk_k[2] = kSplitChunkDefault[2];
    return;
  }
  g_split_chunk_k[0] = x3_k; g_split_chunk_k[1] = x2_k; g_split_chunk_k[2] = x2_k;
}
int b200_gemm_debug_last_schedule(int* out, int cap) {
  if (!out || cap <= 0) return 0;
  const int n = t_last_sched.n < cap ? t_last_sched.n : cap;
  for (int i = 0; i < n; i++) out[i] = t_last_sched.v[i];
  return n;
}
void b200_gemm_debug_kernel_timing(int enable) { g_ktimer.on = enable != 0; g_ktimer.n = 0; }
int b200_gemm_debug_kernel_time_ms(double* sum_ms) {
  double sum = 0;
  int cnt = 0;
  for (int i = 0; i < g_ktimer.n; i++) {
    float ms = 0.f;
    if (cudaEventSynchronize(g_ktimer.ev[i][1]) == cudaSuccess &&
        cudaEventElapsedTime(&ms, g_ktimer.ev[i][0], g_ktimer.ev[i][1]) == cudaSuccess) { sum += ms; cnt++; }
  }
  cudaGetLastError();
  g_ktimer.n = 0;
  if (sum_ms) *sum_ms = sum;
  return cnt;
}

// Grows the split-precision workspace of the current device up front, so that no later compute call
// synchronises or allocates (first use and growth otherwise do: cudaMalloc of the plane buffers).
int b200_gemm_reserve_workspace(size_t bytes) {
  int rc = ensure_device();
  if (rc) return rc;
  std::lock_guard<std::mutex> wlk(t_ctx->ws_mu);
  return split_ws_reserve(bytes);
}
// Bytes b200_gemm_f32 needs for an m x n x k product in `precision_mode` (0 for modes without a split).
size_t b200_gemm_workspace_bytes(int m, int n, int k, int precision_mode) {
  const int mode = resolve_f32_mode(precision_mode);
  const int np = mode == B200_F32_BF16X3 ? 3 : (mode == B200_F32_BF16X2 || mode == B200_F32_F16X2) ? 2 : 0;
  if (!np || m <= 0 || n <= 0 || k <= 0) return 0;
  const size_t a = ((size_t)np * m * plane_pitch(k) * 2 + 1023) & ~(size_t)1023;
  const size_t b = ((size_t)np * b_plane_rows(k) * plane_pitch(n) * 2 + 1023) & ~(size_t)1023;
  return a + b + (size_t)m * 4 + 1024;
}

int b200_gemm_f32(int m, int n, int k, const float* dA, int lda, const float* dB, int ldb, float* dC,
                  int ldc, int precision_mode, void* stream) {
  return gemm_f32_impl(m, n, k, dA, lda, dB, ldb, dC, ldc, precision_mode, 0, (cudaStream_t)stream);
}

// C = alpha * A*B + beta * C (the contract of the reference's cuBLAS comparator, cuda/MMult_cuBLAS_1.cpp:11-19).
int b200_gemm_f32_ex(int m, int n, int k, float alpha, const float* dA, int lda, const float* dB, int ldb, float beta,
                     float* dC, int ldc, int precision_mode, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (alpha == 1.f && beta == 0.f) return gemm_f32_impl(m, n, k, dA, lda, dB, ldb, dC, ldc, precision_mode, 0, st);
  if (alpha == 1.f && beta == 1.f) return gemm_f32_impl(m, n, k, dA, lda, dB, ldb, dC, ldc, precision_mode, 1, st);
  int rc = check_args(m, n, k, dA, lda, dB, ldb, dC, ldc);
  if (rc == 1) return 0;
  if (rc) return rc;
  rc = ensure_device();
  if (rc) return rc;
  const int mode = resolve_f32_mode(precision_mode);
  const bool cuda_core = mode == B200_F32_STRICT || !tma_ok(dA, lda, dB, ldb, 4) || k == 0 ||
                         (precision_mode == B200_F32_AUTO && (double)m * n * k <= 2.0e8);
  const dim3 sg((n + 255) / 256, m < 4096 ? m : 4096);
  if (alpha == 0.f || cuda_core) {
    // CUDA-core paths (strict FFMA chain, generic kernels): C <- (beta/alpha) C, C += A*B, C <- alpha C.
    // beta == 0 must not read C (NaN-safe, as cuBLAS): start from C = A*B instead.
    if (alpha == 0.f || k == 0) {
      if (beta == 0.f) return launch_zero<float>(m, n, dC, ldc, st);
      scale_inplace_kernel<<<sg, 256, 0, st>>>(m, n, dC, ldc, beta);
      g_launches++;
      return last_launch_status();
    }
    if (beta != 0.f && beta != alpha) { scale_inplace_kernel<<<sg, 256, 0, st>>>(m, n, dC, ldc, beta / alpha); g_launches++; }
    rc = gemm_f32_impl(m, n, k, dA, lda, dB, ldb, dC, ldc, cuda_core && mode != B200_F32_STRICT && tma_ok(dA, lda, dB, ldb, 4) ? B200_F32_STRICT : mode,
                       beta != 0.f ? 1 : 0, st);
    if (rc) return rc;
    scale_inplace_kernel<<<sg, 256, 0, st>>>(m, n, dC, ldc, alpha);
    g_launches++;
    return last_launch_status();
  }
  t_epi.axpby = 1; t_epi.alpha = alpha; t_epi.beta = beta;      // tensor-core modes: fused into the epilogue
  rc = gemm_f32_impl(m, n, k, dA, lda, dB, ldb, dC, ldc, mode, 0, st);
  t_epi = EpiOpts();
  return rc;
}

int b200_gemm_f32_acc(int m, int n, int k, const float* dA, int lda, const float* dB, int ldb, float* dC,
                      int ldc, int precision_mode, void* stream) {
  return gemm_f32_impl(m, n, k, dA, lda, dB, ldb, dC, ldc, precision_mode, 1, (cudaStream_t)stream);
}

int b200_gemm_bf16(int m, int n, int k, const uint16_t* dA, int lda, const uint16_t* dB, int ldb,
                   void* dC, int ldc, int out_type, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (out_type != B200_OUT_F32 && out_type != B200_OUT_BF16) return B200_ERR_BAD_ARG;
  int rc = check_args(m, n, k, dA, lda, dB, ldb, dC, ldc);
  if (rc == 1) return 0;
  if (rc) return rc;
  rc = ensure_device();
  if (rc) return rc;
  if (k == 0)
    return out_type == B200_OUT_F32 ? launch_zero<float>(m, n, (float*)dC, ldc, st)
                                    : launch_zero<uint16_t>(m, n, (uint16_t*)dC, ldc, st);
  if (!tma_ok(dA, lda, dB, ldb, 2)) {
    if (out_type == B200_OUT_F32)
      return launch_generic<uint16_t, float>(m, n, k, dA, lda, dB, ldb, (float*)dC, ldc, 0, st, "generic_bf16_64x64");
    return launch_generic<uint16_t, uint16_t>(m, n, k, dA, lda, dB, ldb, (uint16_t*)dC, ldc, 0, st, "generic_bf16_64x64");
  }
  if (out_type == B200_OUT_F32) return tc_bf16_f32(m, n, k, dA, lda, dB, ldb, dC, ldc, st);
  return tc_bf16_bf16(m, n, k, dA, lda, dB, ldb, dC, ldc, st);
}

int b200_gemm_s8s32(int m, int n, int k, const int8_t* dA, int lda, const int8_t* dB, int ldb,
                    int32_t* dC, int ldc, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  int rc = check_args(m, n, k, dA, lda, dB, ldb, dC, ldc);
  if (rc == 1) return 0;
  if (rc) return rc;
  rc = ensure_device();
  if (rc) return rc;
  if (k == 0) return launch_zero<int32_t>(m, n, dC, ldc, st);
  if (!tma_ok(dA, lda, dB, ldb, 1))
    return launch_generic<int8_t, int32_t>(m, n, k, dA, lda, dB, ldb, dC, ldc, 0, st, "generic_s8_64x64");
  return tc_s8(m, n, k, dA, lda, dB, ldb, dC, ldc, st);
}

// ---- pre-split operands (the reference's "packAB interface is open" idea, README.md:85, for the split modes) ----
// One handle type for both sides: bf16 planes (BF16X3 / BF16X2, B only) or scaled fp16 planes with the
// maxima their scaling came from (F16X2, A or B).
struct b200_packed {
  int side;            // 0 = A (rows x cols = m x k), 1 = B (k x n)
  int rows, cols, mode, np, plane_rows;
  long long pitch;
  uint16_t* planes;
  float* maxv;         // F16X2 only
  int dev;
};
struct b200_packed_a : b200_packed {};
struct b200_packed_b : b200_packed {};

static int pack_operand(int side, int rows, int cols, const float* d, int ld, int precision_mode, b200_packed* h,
                        cudaStream_t st) {
  if (rows <= 0 || cols <= 0 || !d || ld < cols) return B200_ERR_BAD_ARG;
  const int mode = resolve_f32_mode(precision_mode);
  if (mode != B200_F32_F16X2 && (side != 1 || (mode != B200_F32_BF16X3 && mode != B200_F32_BF16X2))) return B200_ERR_UNSUPPORTED;
  int rc = ensure_device();
  if (rc) return rc;
  h->side = side; h->rows = rows; h->cols = cols; h->mode = mode; h->planes = nullptr; h->maxv = nullptr;
  h->dev = t_ctx->dev;
  if (mode == B200_F32_F16X2) {
    h->np = 2;
    h->pitch = f16_pitch(cols);
    h->plane_rows = side == 0 ? rows : f16_b_rows(rows);
    const size_t nmax = side == 0 ? (size_t)rows : (size_t)cols;
    cudaError_t e = cudaMalloc(&h->planes, (size_t)2 * h->plane_rows * h->pitch * 2);
    if (e == cudaSuccess) e = cudaMalloc(&h->maxv, nmax * 4);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    if (side == 0) return launch_f16_split_rows(d, ld, rows, cols, h->maxv, h->planes, h->pitch, h->plane_rows, st);
    e = cudaMemsetAsync(h->maxv, 0, nmax * 4, st);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    return launch_f16_split_cols(d, ld, rows, cols, h->maxv, h->planes, h->pitch, h->plane_rows, nullptr, 0, st);
  }
  h->np = mode == B200_F32_BF16X3 ? 3 : 2;
  h->pitch = plane_pitch(cols);
  h->plane_rows = b_plane_rows(rows);
  cudaError_t e = cudaMalloc(&h->planes, (size_t)h->np * h->plane_rows * h->pitch * 2);
  if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
  const SplitJob jb{d, ld, rows, cols, h->planes, h->pitch, h->plane_rows};
  return h->np == 3 ? launch_split<3>(jb, jb, 1, st) : launch_split<2>(jb, jb, 1, st);
}
static void pack_release(b200_packed* h) {
  if (!h) return;
  if (h->planes) cudaFree(h->planes);
  if (h->maxv) cudaFree(h->maxv);
}

int b200_gemm_f32_pack_b(int k, int n, const float* dB, int ldb, int precision_mode, b200_packed_b** out,
                         void* stream) {
  if (!out) return B200_ERR_BAD_ARG;
  *out = nullptr;
  b200_packed_b* h = new b200_packed_b();
  int rc = pack_operand(1, k, n, dB, ldb, precision_mode, h, (cudaStream_t)stream);
  t_last_kernel = "split_planes";
  t_last_sched.clear();
  if (rc) { pack_release(h); delete h; return rc; }
  *out = h;
  return B200_OK;
}

int b200_gemm_f32_pack_a(int m, int k, const float* dA, int lda, int precision_mode, b200_packed_a** out,
                         void* stream) {
  if (!out) return B200_ERR_BAD_ARG;
  *out = nullptr;
  b200_packed_a* h = new b200_packed_a();
  int rc = pack_operand(0, m, k, dA, lda, precision_mode, h, (cudaStream_t)stream);
  t_last_kernel = "split_planes";
  t_last_sched.clear();
  if (rc) { pack_release(h); delete h; return rc; }
  *out = h;
  return B200_OK;
}

// k0: first column of packed A / first row of B this product starts at (K-sliced consumers); the B handle
// always covers exactly the k rows multiplied.
static int gemm_packed_impl(int m, int n, int k, const float* dA, int lda, const b200_packed* pa, int a_k0,
                            const b200_packed* pb, float* dC, int ldc, int accumulate, cudaStream_t st) {
  if (!pb || pb->rows != k || pb->cols != n) return B200_ERR_BAD_ARG;
  if (pa && (pa->rows != m || a_k0 < 0 || a_k0 + k > pa->cols || (a_k0 & 7) || pa->mode != pb->mode)) return B200_ERR_BAD_ARG;
  int rc = check_args(m, n, k, pa ? (const void*)pa->planes : (const void*)dA, pa ? k : lda, pb->planes, n, dC, ldc);
  if (rc == 1) return 0;
  if (rc) return rc;
  rc = ensure_device();
  if (rc) return rc;
  if (pb->dev != t_ctx->dev || (pa && pa->dev != t_ctx->dev)) return B200_ERR_BAD_ARG;
  if (pb->mode == B200_F32_F16X2) {
    const F16Operand ob{pb->planes, pb->pitch, pb->plane_rows, pb->maxv};
    if (pa) {
      const F16Operand oa{pa->planes + a_k0, pa->pitch, pa->plane_rows, pa->maxv};
      return gemm_f32_split_f16(m, n, k, nullptr, 0, nullptr, 0, dC, ldc, st, accumulate ? 1 : 0, &oa, &ob);
    }
    return gemm_f32_split_f16(m, n, k, dA, lda, nullptr, 0, dC, ldc, st, accumulate ? 1 : 0, nullptr, &ob);
  }
  if (pa) return B200_ERR_UNSUPPORTED;
  return pb->np == 3 ? gemm_f32_split<3>(m, n, k, dA, lda, nullptr, 0, dC, ldc, st, accumulate ? 1 : 0, pb->planes)
                     : gemm_f32_split<2>(m, n, k, dA, lda, nullptr, 0, dC, ldc, st, accumulate ? 1 : 0, pb->planes);
}

int b200_gemm_f32_packed(int m, int n, int k, const float* dA, int lda, const b200_packed_b* pb, float* dC,
                         int ldc, int accumulate, void* stream) {
  return gemm_packed_impl(m, n, k, dA, lda, nullptr, 0, pb, dC, ldc, accumulate, (cudaStream_t)stream);
}

int b200_gemm_f32_packed_ab(int m, int n, int k, const b200_packed_a* pa, int a_k0, const b200_packed_b* pb,
                            float* dC, int ldc, int accumulate, void* stream) {
  if (!pa) return B200_ERR_BAD_ARG;
  return gemm_packed_impl(m, n, k, nullptr, 0, pa, a_k0, pb, dC, ldc, accumulate, (cudaStream_t)stream);
}

void b200_gemm_f32_pack_free(b200_packed_b* pb) {
  if (!pb) return;
  pack_release(pb);
  delete pb;
}
void b200_gemm_f32_pack_free_a(b200_packed_a* pa) {
  if (!pa) return;
  pack_release(pa);
  delete pa;
}

int b200_gemm_s8s8_requant(int m, int n, int k, const int8_t* dA, int lda, const int8_t* dB, int ldb,
                           int8_t* dC, int ldc, const float* dScales, const float* dBias, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  int rc = check_args(m, n, k, dA, lda, dB, ldb, dC, ldc);
  if (rc == 1) return 0;
  if (rc) return rc;
  if (!dScales) return B200_ERR_BAD_ARG;
  rc = ensure_device();
  if (rc) return rc;
  if (k == 0 || !tma_ok(dA, lda, dB, ldb, 1))         // K = 0: every element is requant(0) = sat(round(bias))
    return launch_generic_requant(m, n, k, dA, lda, dB, ldb, dC, ldc, dScales, dBias, st);
  return tc_s8_requant(m, n, k, dA, lda, dB, ldb, dC, ldc, dScales, dBias, st);
}

// ---- the 4-bit path: block-scaled MXFP4 (SURVEY §8 f-4; the reference's cuda-int4 is "WIP") ----------------
size_t b200_mxf4_q_bytes(int rows, int k) { return rows <= 0 || k <= 0 ? 0 : (size_t)rows * (size_t)(((k + 127) & ~127) / 2); }
size_t b200_mxf4_sf_bytes(int rows, int k) {
  return rows <= 0 || k <= 0 ? 0 : (size_t)((rows + 127) / 128) * (size_t)((k + 127) / 128) * 512;
}

int b200_mxf4_quantize_a(int m, int k, const float* dA, int lda, uint8_t* dQ, uint8_t* dSF, void* stream) {
  if (m <= 0 || k <= 0 || !dA || !dQ || !dSF || lda < k) return B200_ERR_BAD_ARG;
  int rc = ensure_device();
  if (rc) return rc;
  const int kpad = (k + 127) & ~127, rows_pad = (m + 127) & ~127;
  const long long total = (long long)rows_pad * (kpad / 32);
  long long blocks = (total + 255) / 256;
  if (blocks > t_ctx->sms * 16) blocks = t_ctx->sms * 16;
  mxf4_quantize_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(dA, lda, m, k, dQ, kpad, dSF, rows_pad);
  g_launches++;
  t_last_kernel = "mxf4_quantize_rows";
  t_last_sched.clear();
  return last_launch_status();
}

// B is k x n row-major; the output is B^T quantised along K: n rows of kpad/2 bytes (the K-major operand the
// 4-bit tensor path requires) + scale atoms indexed by (n, K-block).
int b200_mxf4_quantize_b(int k, int n, const float* dB, int ldb, uint8_t* dQ, uint8_t* dSF, void* stream) {
  if (n <= 0 || k <= 0 || !dB || !dQ || !dSF || ldb < n) return B200_ERR_BAD_ARG;
  int rc = ensure_device();
  if (rc) return rc;
  const int kpad = (k + 127) & ~127, n_pad = (n + 127) & ~127;
  mxf4_quantize_cols_t_kernel<<<dim3((n_pad + 255) / 256, kpad / 32), 256, 0, (cudaStream_t)stream>>>(dB, ldb, k, n, dQ, kpad, dSF, n_pad);
  g_launches++;
  t_last_kernel = "mxf4_quantize_cols_t";
  t_last_sched.clear();
  return last_launch_status();
}

int b200_gemm_mxf4(int m, int n, int k, const uint8_t* dAq, const uint8_t* dSFA, const uint8_t* dBq, const uint8_t* dSFB,
                   float* dC, int ldc, void* stream) {
  if (m < 0 || n < 0 || k < 0) return B200_ERR_BAD_ARG;
  if (m == 0 || n == 0) return 0;
  if (!dC || ldc < n) return B200_ERR_BAD_ARG;
  int rc = ensure_device();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (k == 0) return launch_zero<float>(m, n, dC, ldc, st);
  if (!dAq || !dSFA || !dBq || !dSFB || !aligned16(dAq) || !aligned16(dBq) || !aligned16(dSFA) || !aligned16(dSFB)) return B200_ERR_BAD_ARG;
  using Cfg = Mxf4Cfg<128>;
  const int kpad = (k + 127) & ~127;
  CUtensorMap tmA, tmB;
  rc = get_map(&tmA, dAq, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, kpad / 2, m, kpad / 2, 128, Cfg::BM, 1);
  if (rc) return rc;
  rc = get_map(&tmB, dBq, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, kpad / 2, n, kpad / 2, 128, 128, 1);
  if (rc) return rc;
  Mxf4Params p;
  p.C = dC; p.ldc = ldc; p.M = m; p.N = n; p.K = kpad;
  p.sfa = dSFA; p.sfb = dSFB;
  p.tiles_m = (m + 127) / 128; p.tiles_n = (n + 127) / 128;
  p.vec_ok = aligned16(dC) && (ldc % 4) == 0;
  auto kern = gemm_mxf4_kernel<128>;
  if (int arc = ensure_smem_attr(kern, Cfg::SMEM_BYTES)) return arc;
  const int tiles = p.tiles_m * p.tiles_n;
  g_ktimer.begin(st);
  kern<<<tiles < t_ctx->sms ? tiles : t_ctx->sms, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(tmA, tmB, p);
  g_ktimer.end(st);
  g_launches++;
  t_last_kernel = "tc_mxf4_128x128";
  t_last_sched.clear();
  return last_launch_status();
}

int b200_convert_f32_to_bf16(const float* dSrc, uint16_t* dDst, size_t count, void* stream) {
  if (count == 0) return 0;
  if (!dSrc || !dDst) return B200_ERR_BAD_ARG;
  int rc = ensure_device();
  if (rc) return rc;
  size_t blocks = (count + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  convert_f32_to_bf16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(dSrc, dDst, count);
  g_launches++;
  t_last_kernel = "convert_f32_to_bf16";
  t_last_sched.clear();
  return last_launch_status();
}

// ---- host-pointer entry points (plumbing / parity / e2e) ---------------------------------------
// Device staging buffers are cached and only ever grow, so repeated calls (the harness calls
// MY_MMult NREPEATS times, aarch64/test_MMult.cpp:105-117) pay no cudaMalloc after the first.
// Copies are asynchronous on the legacy stream; pinned host buffers run at full PCIe rate.
namespace {
cudaError_t scratch(int i, size_t bytes, void** out) {
  Scratch* scr = t_ctx->scr;
  if (scr[i].bytes < bytes) {
    if (scr[i].p) cudaFree(scr[i].p);
    scr[i].p = nullptr; scr[i].bytes = 0;
    cudaError_t e = cudaMalloc(&scr[i].p, bytes);
    if (e != cudaSuccess) return e;
    scr[i].bytes = bytes;
  }
  *out = scr[i].p;
  return cudaSuccess;
}
}  // namespace

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { cudaGetLastError(); return (int)e_; } } while (0)

int b200_gemm_f32_host(int m, int n, int k, const float* A, int lda, const float* B, int ldb, float* C,
                       int ldc, int precision_mode) {
  int rc = check_args(m, n, k, A, lda, B, ldb, C, ldc);
  if (rc == 1) return 0;
  if (rc) return rc;
  rc = ensure_device();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(t_ctx->host_mu);
  float *dA = nullptr, *dB = nullptr, *dC = nullptr;
  const int mode = precision_mode;   // unresolved: AUTO keeps its small-problem switch to the bit-exact STRICT kernel
  // device images: pitches rounded up to 4 floats so the TMA paths apply to any k, n
  const int pk = (k + 3) & ~3, pn = (n + 3) & ~3;
  const size_t pa = (size_t)pk * 4, pb = (size_t)pn * 4, pc = (size_t)pn * 4;
  if (k > 0) {
    CK(scratch(0, pa * m, (void**)&dA));
    CK(scratch(1, pb * k, (void**)&dB));
  }
  CK(scratch(2, pc * m, (void**)&dC));
  // Large problems: row-block pipeline over three streams, so the D2H of C block i overlaps the H2D
  // of block i+1 (PCIe is full duplex) and the GEMMs hide under the copies.  The path is copy-bound:
  // 268 MB cross the bus per 4096^3 call against 0.6 ms of math.
  const int blocks = (k > 0 && m >= 2048 && (double)m * n * k >= 8.0e9) ? 4 : 1;
  if (blocks == 1) {
    cudaStream_t st = 0;
    if (k > 0) {
      CK(cudaMemcpy2DAsync(dA, pa, A, (size_t)lda * 4, (size_t)k * 4, m, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpy2DAsync(dB, pb, B, (size_t)ldb * 4, (size_t)n * 4, k, cudaMemcpyHostToDevice, st));
    }
    CK(cudaMemcpy2DAsync(dC, pc, C, (size_t)ldc * 4, (size_t)n * 4, m, cudaMemcpyHostToDevice, st));
    rc = gemm_f32_impl(m, n, k, dA, pk, dB, pn, dC, pn, mode, /*accumulate=*/1, st);   // C += A*B on the device
    if (rc) return rc;
    CK(cudaMemcpy2DAsync(C, (size_t)ldc * 4, dC, pc, (size_t)n * 4, m, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
  }
  CK(t_ctx->pipe.init());
  CK(cudaMemcpy2DAsync(dB, pb, B, (size_t)ldb * 4, (size_t)n * 4, k, cudaMemcpyHostToDevice, t_ctx->pipe.h2d));
  const int rows_per = ((m + blocks - 1) / blocks + 255) & ~255;       // whole 256-row pair tiles per block
  int nb = 0;
  for (int r0 = 0; r0 < m; r0 += rows_per, nb++) {
    const int rows = m - r0 < rows_per ? m - r0 : rows_per;
    float* dAi = dA + (size_t)r0 * pk;
    float* dCi = dC + (size_t)r0 * pn;
    CK(cudaMemcpy2DAsync(dAi, pa, A + (size_t)r0 * lda, (size_t)lda * 4, (size_t)k * 4, rows, cudaMemcpyHostToDevice, t_ctx->pipe.h2d));
    CK(cudaMemcpy2DAsync(dCi, pc, C + (size_t)r0 * ldc, (size_t)ldc * 4, (size_t)n * 4, rows, cudaMemcpyHostToDevice, t_ctx->pipe.h2d));
    CK(cudaEventRecord(t_ctx->pipe.in[nb], t_ctx->pipe.h2d));
    CK(cudaStreamWaitEvent(t_ctx->pipe.comp, t_ctx->pipe.in[nb], 0));
    rc = gemm_f32_impl(rows, n, k, dAi, pk, dB, pn, dCi, pn, mode, /*accumulate=*/1, t_ctx->pipe.comp);
    if (rc) return rc;
    CK(cudaEventRecord(t_ctx->pipe.done[nb], t_ctx->pipe.comp));
    CK(cudaStreamWaitEvent(t_ctx->pipe.d2h, t_ctx->pipe.done[nb], 0));
    CK(cudaMemcpy2DAsync(C + (size_t)r0 * ldc, (size_t)ldc * 4, dCi, pc, (size_t)n * 4, rows, cudaMemcpyDeviceToHost, t_ctx->pipe.d2h));
  }
  CK(cudaStreamSynchronize(t_ctx->pipe.d2h));
  CK(cudaStreamSynchronize(t_ctx->pipe.comp));
  return 0;
}

int b200_gemm_s8s32_host(int m, int n, int k, const int8_t* A, int lda, const int8_t* B, int ldb,
                         int32_t* C, int ldc) {
  int rc = check_args(m, n, k, A, lda, B, ldb, C, ldc);
  if (rc == 1) return 0;
  if (rc) return rc;
  rc = ensure_device();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(t_ctx->host_mu);
  int8_t *dA = nullptr, *dB = nullptr;
  int32_t* dC = nullptr;
  // device images padded to 16-byte pitches so the tcgen05 path is taken for any m,n,k
  const size_t pa = ((size_t)k + 15) & ~(size_t)15, pb = ((size_t)n + 15) & ~(size_t)15;
  const size_t pc = (size_t)n * 4;
  cudaStream_t st = 0;
  if (k > 0) {
    CK(scratch(0, pa * m, (void**)&dA));
    CK(scratch(1, pb * k, (void**)&dB));
    CK(cudaMemcpy2DAsync(dA, pa, A, (size_t)lda, (size_t)k, m, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpy2DAsync(dB, pb, B, (size_t)ldb, (size_t)n, k, cudaMemcpyHostToDevice, st));
  }
  CK(scratch(2, pc * m, (void**)&dC));
  rc = b200_gemm_s8s32(m, n, k, dA, (int)pa, dB, (int)pb, dC, n, st);
  if (rc) return rc;
  CK(cudaMemcpy2DAsync(C, (size_t)ldc * 4, dC, pc, pc, m, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

}  // extern "C"

#include "rowpanel.cuh"
