// CUDA instantiation of the persistent tensor-core convolution that runs every dense conv layer the engine routes to the
// tensor cores: the body lives in conv2_body.inl, the primitives in tc_policy_dev.cuh, plan / pack / argument fill in
// conv2_host.h.  The same body runs on a CPU model of the primitives in tests/test_conv2_sim.py (every epilogue, every
// split precision, ragged batches); on the B200: tests/test_gpu_conv_kernels.py and the whole -m gpu suite.
#include "kernels.cuh"
#include "launch.cuh"

#include <cuda_bf16.h>

#include <cstdlib>
#include <stdexcept>

#define MRF_FN __device__ __forceinline__
#define MRF_NOINLINE __device__ __noinline__
#include "tc_policy_dev.cuh"
#include "conv2_host.h"
#include "conv2_body.inl"

namespace pb200 {
void count_launch();

namespace {

template <int PREC, int MT>
__global__ void __launch_bounds__(conv2::C2_THREADS, 1) conv2_kernel(const __grid_constant__ MmaConvArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) conv2::Barriers<uint64_t> bar;
  __shared__ uint32_t tmem_base_s;
  DevPrim::Ctx cx;
  conv2::conv2_body<DevPrim, PREC, MT>(a, cx, smem, bar, &tmem_base_s);
}

// Tensor-map variant (PIPER_B200_V2_TM=1): the activation window of a channel chunk is one cp.async.bulk.tensor copy.
// The dynamic shared memory is re-aligned to 128 bytes by hand (tensor copies require it; the launcher adds the slack).
// ASLOTS = 0: the A-stationary instantiation (operand ring with one slot per channel chunk, MmaConvArgs::a_slots)
template <int PREC, int MT, int ASLOTS = 2>
__global__ void __launch_bounds__(conv2::C2_THREADS, 1) conv2_tm_kernel(const __grid_constant__ MmaConvArgs a,
                                                                        const __grid_constant__ CUtensorMap tmx) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ __align__(8) conv2::Barriers<uint64_t> bar;
  __shared__ uint32_t tmem_base_s;
  uint8_t* smem = smem_raw + ((128u - ((uint32_t)__cvta_generic_to_shared(smem_raw) & 127u)) & 127u);
  DevPrim::Ctx cx;
  conv2::conv2_body<DevPrim, PREC, MT, true, ASLOTS>(a, cx, smem, bar, &tmem_base_s, &tmx);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda)
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}


}  // namespace

bool encode_tmap(const TmapDesc& d, void* out_cutensormap) {
  CUtensorMap* out = static_cast<CUtensorMap*>(out_cutensormap);
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)d.dims[0], (cuuint64_t)d.dims[1], (cuuint64_t)d.dims[2]};
  const cuuint64_t strides[2] = {(cuuint64_t)d.stride1, (cuuint64_t)d.stride2};
  const cuuint32_t box[3] = {(cuuint32_t)d.box[0], (cuuint32_t)d.box[1], (cuuint32_t)d.box[2]};
  const cuuint32_t estr[3] = {1, 1, 1};
  return fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(d.base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool conv2_plan(int ci, int rows, int k, int dil, int prec, int chains, Conv2Layer& l) {
  static int g_opts = -1;                               // PIPER_B200_V2_OPTS: plan options (conv2_host.h)
  if (g_opts < 0) {
    const char* e = std::getenv("PIPER_B200_V2_OPTS");
    g_opts = e ? std::atoi(e) : 0;
  }
  conv2::Plan p;
  if (!conv2::plan(ci, rows, k, dil, prec, chains, p, g_opts)) return false;
  l.tf32 = p.tf32; l.prec = p.prec; l.n_tile = p.n_tile; l.n_tiles = p.n_tiles; l.mt = p.mt; l.kc = p.kc; l.stage_rows = p.stage_rows;
  l.raw_stride = p.raw_stride; l.t_slots = p.t_slots; l.tmem_cols = p.tmem_cols; l.chains = p.chains; l.mh_stride = p.mh_stride;
  l.smem = p.smem; l.w_bytes = p.w_bytes;
  return true;
}

static conv2::Plan to_plan(const Conv2Layer& l) {
  conv2::Plan p;
  p.ok = true; p.tf32 = l.tf32; p.prec = l.prec; p.n_tile = l.n_tile; p.n_tiles = l.n_tiles; p.mt = l.mt; p.kc = l.kc; p.stage_rows = l.stage_rows;
  p.raw_stride = l.raw_stride; p.t_slots = l.t_slots; p.tmem_cols = l.tmem_cols; p.chains = l.chains; p.mh_stride = l.mh_stride;
  p.smem = l.smem; p.w_bytes = l.w_bytes;
  return p;
}

void conv2_pack(const float* wsrc, int ci, int k, int rows_p, const Conv2Layer& l, uint8_t* out) {
  conv2::pack(wsrc, ci, k, rows_p, to_plan(l), out);
}

// a: x / y / y2 / r / w (conv2_pack layout) / bias / len / shape / epilogue fields set by the caller
void launch_conv2(MmaConvArgs a, const Conv2Layer& l, int B, int max_len, cudaStream_t st) {
  if (B <= 0 || max_len <= 0) return;
  const conv2::Plan p = to_plan(l);
  static int g_tm = -1;                                 // PIPER_B200_V2_TM: tensor-map TMA for the activation window
  if (g_tm < 0) {
    const char* e = std::getenv("PIPER_B200_V2_TM");
    g_tm = (e ? std::atoi(e) > 0 : true) ? 1 : 0;       // default on (0 = one bulk copy per channel row)
  }
  static int g_mma3 = -1;                               // PIPER_B200_V2_MMA3: non-overlapping three-instruction k-step
  if (g_mma3 < 0) {
    const char* e = std::getenv("PIPER_B200_V2_MMA3");
    g_mma3 = (e && std::atoi(e) > 0) ? 1 : 0;
  }
  a.mma3 = g_mma3;
  TmapDesc td;
  CUtensorMap tmx;
  bool tm = g_tm != 0;
  // PIPER_B200_V2_ASTAT (default 1): A-stationary tile order with the whole converted window of a position resident
  // (conv2_body.inl, conv2_host.h).  The first version kept the two-slot ring and so applied to almost no layer (447.9 vs
  // 448.4 M samples/s); with one slot per channel chunk: 512.0 vs 493.4 M samples/s on the same box (first FFN conv 59 ->
  // 45 us, second upsampler 238 -> 168 us).
  static int g_astat = -1;
  if (g_astat < 0) {
    const char* e = std::getenv("PIPER_B200_V2_ASTAT");
    g_astat = e ? (std::atoi(e) != 0) : 1;
  }
  size_t smem = p.smem;                                 // (the A-stationary plan re-sizes the rings)
  int grid = conv2::fill_args(a, p, B, max_len, tm, &td, g_astat != 0, &smem);
  if (tm && !encode_tmap(td, &tmx)) {                    // (a view the encoder refuses: fall back to per-row copies)
    tm = false;
    grid = conv2::fill_args(a, p, B, max_len, false, nullptr, false, &smem);
  } else if (!tm && a.astat) {
    grid = conv2::fill_args(a, p, B, max_len, false, nullptr, false, &smem);   // (the A-stationary instantiations exist for the tensor-map kernel only)
  }
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev & 63]) {
    cudaFuncSetAttribute(conv2_kernel<0, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_kernel<0, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_kernel<1, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_kernel<2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_kernel<2, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_tm_kernel<0, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_tm_kernel<0, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_tm_kernel<1, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_tm_kernel<2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_tm_kernel<2, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_tm_kernel<0, 128, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_tm_kernel<0, 256, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_tm_kernel<1, 128, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_tm_kernel<2, 128, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    cudaFuncSetAttribute(conv2_tm_kernel<2, 256, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
    attr_set[dev & 63] = true;
  }
  if (tm && a.astat) {
    const size_t sm = smem + 128;
    if (p.prec == 1) launch_k(conv2_tm_kernel<1, 128, 0>, dim3(grid), dim3(conv2::C2_THREADS), sm, st, a, tmx);
    else if (p.prec == 2 && p.mt == 256) launch_k(conv2_tm_kernel<2, 256, 0>, dim3(grid), dim3(conv2::C2_THREADS), sm, st, a, tmx);
    else if (p.prec == 2) launch_k(conv2_tm_kernel<2, 128, 0>, dim3(grid), dim3(conv2::C2_THREADS), sm, st, a, tmx);
    else if (p.mt == 256) launch_k(conv2_tm_kernel<0, 256, 0>, dim3(grid), dim3(conv2::C2_THREADS), sm, st, a, tmx);
    else launch_k(conv2_tm_kernel<0, 128, 0>, dim3(grid), dim3(conv2::C2_THREADS), sm, st, a, tmx);
    count_launch();
    return;
  }
  if (tm) {
    const size_t sm = smem + 128;
    if (p.prec == 1) launch_k(conv2_tm_kernel<1, 128>, dim3(grid), dim3(conv2::C2_THREADS), sm, st, a, tmx);
    else if (p.prec == 2 && p.mt == 256) launch_k(conv2_tm_kernel<2, 256>, dim3(grid), dim3(conv2::C2_THREADS), sm, st, a, tmx);
    else if (p.prec == 2) launch_k(conv2_tm_kernel<2, 128>, dim3(grid), dim3(conv2::C2_THREADS), sm, st, a, tmx);
    else if (p.mt == 256) launch_k(conv2_tm_kernel<0, 256>, dim3(grid), dim3(conv2::C2_THREADS), sm, st, a, tmx);
    else launch_k(conv2_tm_kernel<0, 128>, dim3(grid), dim3(conv2::C2_THREADS), sm, st, a, tmx);
    count_launch();
    return;
  }
  if (p.prec == 1) launch_k(conv2_kernel<1, 128>, dim3(grid), dim3(conv2::C2_THREADS), smem, st, a);
  else if (p.prec == 2 && p.mt == 256) launch_k(conv2_kernel<2, 256>, dim3(grid), dim3(conv2::C2_THREADS), smem, st, a);
  else if (p.prec == 2) launch_k(conv2_kernel<2, 128>, dim3(grid), dim3(conv2::C2_THREADS), smem, st, a);
  else if (p.mt == 256) launch_k(conv2_kernel<0, 256>, dim3(grid), dim3(conv2::C2_THREADS), smem, st, a);
  else launch_k(conv2_kernel<0, 128>, dim3(grid), dim3(conv2::C2_THREADS), smem, st, a);
  count_launch();
}

}  // namespace pb200
