// Generator tail and audio epilogue.
//   conv_post: leaky_relu(slope 0.01) -> Conv1d(C -> 1, k=7, no bias) -> tanh      (models.py:364-366)
//   int16 epilogue: per-utterance peak, scale 32767 / max(0.01, peak), clamp, truncate  (piper.cpp:411-431)
#include "kernels.cuh"
#include "launch.cuh"

#include <stdexcept>

namespace pb200 {
void count_launch();

namespace {

constexpr int POST_TT = 256;
constexpr int POST_MAXK = 15;

// conv_post where the fused MRF stage does not apply.  The staging loads of eight channels are in flight at once: staging
// the C = 32 rows one exposed load latency after the other measured ~0.58 ms per step for 0.5 GB, 7x the HBM time.
__global__ void __launch_bounds__(256) conv_post_kernel2(View x, const float* __restrict__ w, int C, int k, float slope,
                                                         float* __restrict__ out, const long long* __restrict__ out_off,
                                                         const int* __restrict__ len, int len_scale) {
  pdl_launch_dependents();   // programmatic dependent launch (launch.cuh): the next grid may be scheduled now;
  pdl_wait();                // nothing below runs before the previous grid has completed
  extern __shared__ float sm[];   // weights [C][k] | activated input tile [C][POST_TT + k - 1]
  const int b = blockIdx.z;
  const int L = len[b] * len_scale;
  const int t0 = blockIdx.x * POST_TT;
  if (t0 >= L) return;
  const int half = (k - 1) / 2;
  const int span = POST_TT + k - 1;
  float* ws = sm;
  float* xs = sm + C * k;
  for (int i = threadIdx.x; i < C * k; i += 256) ws[i] = w[i];
  const float* xb = x.p + (long long)b * x.bs;
  for (int u = threadIdx.x; u < span; u += 256) {
    const int tt = t0 - half + u;
    const bool in = tt >= 0 && tt < L;
    for (int c0 = 0; c0 < C; c0 += 8) {
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = (in && c0 + e < C) ? __ldg(xb + (long long)(c0 + e) * x.cs + tt) : 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e)
        if (c0 + e < C) xs[(c0 + e) * span + u] = v[e] > 0.f ? v[e] : v[e] * slope;
    }
  }
  __syncthreads();
  const int t = t0 + threadIdx.x;
  if (t >= L) return;
  float acc = 0.f;
  for (int c = 0; c < C; ++c) {
    const float* xr = xs + c * span + threadIdx.x;
    const float* wr = ws + c * k;
    for (int j = 0; j < k; ++j) acc = fmaf(wr[j], xr[j], acc);
  }
  out[out_off[b] + t] = tanhf(acc);
}

__global__ void __launch_bounds__(256) peak_kernel(const float* __restrict__ audio, const long long* __restrict__ off,
                                                   const int* __restrict__ len, int len_scale,
                                                   unsigned int* __restrict__ peak) {
  pdl_launch_dependents();   // programmatic dependent launch (launch.cuh): the next grid may be scheduled now;
  pdl_wait();                // nothing below runs before the previous grid has completed
  const int b = blockIdx.z;
  const int L = len[b] * len_scale;
  const float* a = audio + off[b];
  float m = 0.f;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < L; t += (long long)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(a[t]));
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(peak + b, __float_as_uint(m));
}

__global__ void __launch_bounds__(256) to_int16_kernel(const float* __restrict__ audio,
                                                       const long long* __restrict__ off, const int* __restrict__ len,
                                                       int len_scale, const unsigned int* __restrict__ peak,
                                                       int16_t* __restrict__ out) {
  pdl_launch_dependents();   // programmatic dependent launch (launch.cuh): the next grid may be scheduled now;
  pdl_wait();                // nothing below runs before the previous grid has completed
  const int b = blockIdx.z;
  const int L = len[b] * len_scale;
  const float mx = fmaxf(0.01f, __uint_as_float(peak[b]));   // maxAudioValue starts at 0.01f
  const float scale = 32767.0f / fmaxf(0.01f, mx);
  const float* a = audio + off[b];
  int16_t* o = out + off[b];
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < L; t += (long long)gridDim.x * blockDim.x) {
    const float v = fminf(fmaxf(a[t] * scale, -32768.0f), 32767.0f);
    o[t] = (int16_t)v;   // static_cast<int16_t>(float): truncation toward zero
  }
}

}  // namespace

void launch_conv_post(View x, const float* w, int C, int k, float slope, float* out, const long long* out_off,
                      const int* len, int len_scale, int B, int max_len, cudaStream_t st) {
  if (B <= 0 || max_len <= 0) return;
  if (k > POST_MAXK) throw std::runtime_error("conv_post: kernel too wide");
  dim3 grid((max_len + POST_TT - 1) / POST_TT, 1, B);
  const size_t smem = (size_t(C) * k + size_t(C) * (POST_TT + k - 1)) * sizeof(float);
  if (smem > 96 * 1024) throw std::runtime_error("conv_post: too many channels");
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev & 63]) {
    cudaFuncSetAttribute(conv_post_kernel2, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    attr_set[dev & 63] = true;
  }
  launch_k(conv_post_kernel2, dim3(grid), dim3(256), smem, st, x, w, C, k, slope, out, out_off, len, len_scale);
  count_launch();
}

void launch_peak(const float* audio, const long long* off, const int* len, int len_scale, unsigned int* peak, int B,
                 int max_len, cudaStream_t st) {
  if (B <= 0 || max_len <= 0) return;
  int gx = (max_len + 256 * 8 - 1) / (256 * 8);
  if (gx < 1) gx = 1;
  dim3 grid(gx, 1, B);
  launch_k(peak_kernel, dim3(grid), dim3(256), 0, st, audio, off, len, len_scale, peak);
  count_launch();
}

void launch_to_int16(const float* audio, const long long* off, const int* len, int len_scale, const unsigned int* peak,
                     int16_t* out, int B, int max_len, cudaStream_t st) {
  if (B <= 0 || max_len <= 0) return;
  int gx = (max_len + 256 * 8 - 1) / (256 * 8);
  if (gx < 1) gx = 1;
  dim3 grid(gx, 1, B);
  launch_k(to_int16_kernel, dim3(grid), dim3(256), 0, st, audio, off, len, len_scale, peak, out);
  count_launch();
}

}  // namespace pb200
