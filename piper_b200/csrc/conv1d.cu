// Generic fp32 Conv1d / ConvTranspose1d as a register-tiled implicit GEMM (CUDA cores).
//
//   acc[row][t] = sum_ci sum_j W[ci][j][row] * act(x[ci][t - pad + j*dil])
//
// One CTA (256 threads, 8 warps) owns a ROWS x TT output tile: WR warps along rows (CPT rows per
// thread, weights read as warp-broadcast LDS.128) x WT warps along time (lanes own consecutive t, TPT
// positions per lane 32 apart -> conflict-free scalar LDS and coalesced global stores).  The input
// tile (with its dilated halo) and the weight slab of `cic` input channels are staged in shared
// memory per chunk; the pre-activation (leaky-relu) is applied once while staging, the epilogues
// (bias / relu / residual / WaveNet gate / WN residual+skip / coupling subtract / pixel-shuffle store /
// MRF average) are applied from registers, so every elementwise op of the reference graph between two
// convolutions costs zero extra HBM traffic.
//
// fp32 FFMA keeps the 1e-3 waveform parity bar (single-pass TF32/BF16 tensor-core math does not:
// SURVEY.md finding 7); the split-precision tcgen05 path for the large layers lives in conv_mma2.cu.
//
// Reference ops covered: every Conv / ConvTranspose node of the exported graph except the depthwise
// ones (SURVEY.md App. B.1; modules.py:184-209,301-314,355-364; models.py:348-368; attentions.py:386-407).
#include "kernels.cuh"
#include "launch.cuh"

#include <atomic>
#include <stdexcept>
#include <string>

namespace pb200 {

static std::atomic<unsigned long long> g_launches{0};
unsigned long long launch_count() { return g_launches.load(); }
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
void count_launches(unsigned long long n) { g_launches.fetch_add(n, std::memory_order_relaxed); }   // a replayed CUDA graph

namespace {

__device__ __forceinline__ float sigmoidf_acc(float v) { return 1.f / (1.f + expf(-v)); }

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc, int src_bytes) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// Two-stage cp.async pipeline: while chunk k is in the FMA loop, chunk k+1 (input tile with its dilated
// halo + weight slab) streams global -> shared with 16-byte LDGSTS; out-of-range bytes are zero-filled by
// the copy itself (src-size < 16), which is what gives every utterance its own zero padding.
template <int CPT, int WR, int TPT>
__global__ void __launch_bounds__(256) conv1d_kernel(const ConvArgs a) {
  pdl_launch_dependents();   // programmatic dependent launch (launch.cuh): the next grid may be scheduled now;
  pdl_wait();                // nothing below runs before the previous grid has completed
  constexpr int WT = 8 / WR;
  constexpr int ROWS = CPT * WR;
  constexpr int TT = WT * 32 * TPT;
  extern __shared__ __align__(16) float smem[];

  const int b = blockIdx.z;
  const int L = a.len[b] * a.len_scale;
  const int Lq = L + a.q_extra;
  const int t0 = blockIdx.x * TT;
  if (t0 >= Lq) return;
  const int row0 = blockIdx.y * ROWS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wr = warp % WR, wt = warp / WR;

  // the tile starts at the 16-byte boundary below t0 - pad so every row copy is a run of aligned float4
  const int tbase = t0 - a.pad;
  const int t_al = tbase & ~3;                 // floor to a multiple of 4 (two's complement: also for negatives)
  const int off = tbase - t_al;                // 0..3
  const int span4 = (TT + (a.k - 1) * a.dil + off + 3) >> 2;   // float4 per row
  const int span = span4 << 2;
  const int cic = a.cic;
  const int xs_floats = cic * span;
  const int ws_floats = cic * a.k * ROWS;
  const int stage_floats = xs_floats + ws_floats;               // both multiples of 4

  float acc[CPT][TPT];
#pragma unroll
  for (int r = 0; r < CPT; ++r)
#pragma unroll
    for (int i = 0; i < TPT; ++i) acc[r][i] = 0.f;

  const float* xb = a.x.p + (long long)b * a.x.bs;
  const int n_chunks = (a.ci + cic - 1) / cic;
  const int x4_total = cic * span4;
  const int w4_total = cic * a.k * (ROWS / 4);

  auto prefetch = [&](int chunk, float* stage) {
    const int ci0 = chunk * cic;
    float* xs = stage;
    float* ws = stage + xs_floats;
    for (int idx = tid; idx < x4_total; idx += 256) {
      const int c = idx / span4, u4 = idx - c * span4;
      const int ci = ci0 + c;
      const int t = t_al + (u4 << 2);
      int valid = 0;                                   // bytes of this float4 inside [0, L)
      if (ci < a.ci && t >= 0 && t < L) valid = min(4, L - t) * 4;
      const float* src = valid ? xb + (long long)ci * a.x.cs + t : xb;
      cp_async16(xs + c * span + (u4 << 2), src, valid);
    }
    for (int idx = tid; idx < w4_total; idx += 256) {
      const int r4 = idx % (ROWS / 4);
      const int cj = idx / (ROWS / 4);
      const int c = cj / a.k, j = cj - c * a.k;
      const int ci = ci0 + c;
      const int row = row0 + r4 * 4;
      const bool ok = ci < a.ci && row < a.rows_p;
      const float* src = ok ? a.w + ((long long)ci * a.k + j) * a.rows_p + row : a.w;
      cp_async16(ws + (idx << 2), src, ok ? 16 : 0);
    }
    cp_async_commit();
  };

  prefetch(0, smem);
  for (int chunk = 0; chunk < n_chunks; ++chunk) {
    float* stage = smem + (chunk & 1) * stage_floats;
    if (chunk + 1 < n_chunks) {
      prefetch(chunk + 1, smem + ((chunk + 1) & 1) * stage_floats);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    float* xs = stage;
    const float* ws = stage + xs_floats;
    if (a.pre == PRE_LRELU) {
      // each thread activates exactly the float4s it copied itself (visible to it after wait_group)
      for (int idx = tid; idx < x4_total; idx += 256) {
        const int c = idx / span4, u4 = idx - c * span4;
        float4* p = reinterpret_cast<float4*>(xs + c * span + (u4 << 2));
        float4 v = *p;
        v.x = v.x > 0.f ? v.x : v.x * a.slope;
        v.y = v.y > 0.f ? v.y : v.y * a.slope;
        v.z = v.z > 0.f ? v.z : v.z * a.slope;
        v.w = v.w > 0.f ? v.w : v.w * a.slope;
        *p = v;
      }
    }
    __syncthreads();

    // ---- FMA
    for (int c = 0; c < cic; ++c) {
      const float* xrow = xs + c * span + off + wt * (32 * TPT) + lane;
      const float* wrow = ws + c * a.k * ROWS + wr * CPT;
      for (int j = 0; j < a.k; ++j) {
        float wv[CPT];
#pragma unroll
        for (int r = 0; r < CPT; r += 4) {
          const float4 w4 = *reinterpret_cast<const float4*>(wrow + j * ROWS + r);
          wv[r] = w4.x; wv[r + 1] = w4.y; wv[r + 2] = w4.z; wv[r + 3] = w4.w;
        }
        float xv[TPT];
#pragma unroll
        for (int i = 0; i < TPT; ++i) xv[i] = xrow[j * a.dil + 32 * i];
#pragma unroll
        for (int r = 0; r < CPT; ++r)
#pragma unroll
          for (int i = 0; i < TPT; ++i) acc[r][i] = fmaf(wv[r], xv[i], acc[r][i]);
      }
    }
    __syncthreads();   // everyone is done with this stage before the next prefetch overwrites it
  }

  // ---- epilogue
  const int rbase = row0 + wr * CPT;
  float bv[CPT];
#pragma unroll
  for (int r = 0; r < CPT; ++r) {
    bv[r] = (a.bias != nullptr && rbase + r < a.rows) ? __ldg(a.bias + rbase + r) : 0.f;
    if (a.bias_item != nullptr && rbase + r < a.rows) bv[r] += __ldg(a.bias_item + (long long)b * a.bias_item_stride + rbase + r);
  }

  float* yb = a.y.p ? a.y.p + (long long)b * a.y.bs : nullptr;
  float* y2b = a.y2.p ? a.y2.p + (long long)b * a.y2.bs : nullptr;
  const float* rb = a.r.p ? a.r.p + (long long)b * a.r.bs : nullptr;

#pragma unroll
  for (int i = 0; i < TPT; ++i) {
    const int t = t0 + wt * (32 * TPT) + lane + 32 * i;
    if (t >= Lq) continue;
    if (a.epi == EPI_GATE) {
#pragma unroll
      for (int r = 0; r < CPT; r += 2) {
        const int row = rbase + r;
        if (row + 1 < a.rows) {
          const float ta = acc[r][i] + bv[r], sb = acc[r + 1][i] + bv[r + 1];
          yb[(long long)(row >> 1) * a.y.cs + t] = tanhf(ta) * sigmoidf_acc(sb);
        }
      }
      continue;
    }
#pragma unroll
    for (int r = 0; r < CPT; ++r) {
      const int row = rbase + r;
      if (row >= a.rows) continue;
      const float v = acc[r][i] + bv[r];
      switch (a.epi) {
        case EPI_BIAS: yb[(long long)row * a.y.cs + t] = v; break;
        case EPI_RELU: yb[(long long)row * a.y.cs + t] = fmaxf(v, 0.f); break;
        case EPI_RES: yb[(long long)row * a.y.cs + t] = v + rb[(long long)row * a.r.cs + t]; break;
        case EPI_WN:
          if (row < a.split) {
            yb[(long long)row * a.y.cs + t] = rb[(long long)row * a.r.cs + t] + v;
          } else {
            float* o = y2b + (long long)(row - a.split) * a.y2.cs + t;
            *o = a.first ? v : *o + v;
          }
          break;
        case EPI_SUBFROM: yb[(long long)row * a.y.cs + t] = rb[(long long)row * a.r.cs + t] - v; break;
        case EPI_UPSAMPLE: {
          const int co = row / a.up, phi = row - co * a.up;
          const int to = t * a.up + phi - a.up_pad;
          if (to >= 0 && to < L * a.up) yb[(long long)co * a.y.cs + to] = v;
          break;
        }
        case EPI_MRF: {
          const float v2 = v + rb[(long long)row * a.r.cs + t];
          float* o = y2b + (long long)row * a.y2.cs + t;
          if (a.mrf == 0) *o = v2;
          else if (a.mrf == 1) *o = *o + v2;
          else *o = (*o + v2) / (float)a.mrf_n;
          break;
        }
        default: break;
      }
    }
  }
}

template <int CPT, int WR, int TPT>
void launch_cfg(ConvArgs& a, int B, int max_len, cudaStream_t st) {
  constexpr int WT = 8 / WR, ROWS = CPT * WR, TT = WT * 32 * TPT;
  const int span = ((TT + (a.k - 1) * a.dil + 3 + 3) >> 2) << 2;   // worst-case alignment offset of 3
  // input-channel chunk: as deep as two pipeline stages allow (fewer barriers per FLOP), at most 64
  auto bytes = [&](int c) { return size_t(2) * size_t(c * span + c * a.k * ROWS) * sizeof(float); };
  int cic = a.ci < 64 ? a.ci : 64;
  while (cic > 2 && bytes(cic) > 100 * 1024) --cic;
  const int n_chunks = (a.ci + cic - 1) / cic;
  cic = (a.ci + n_chunks - 1) / n_chunks;              // even split: no mostly-empty last chunk
  a.cic = cic;
  const size_t smem = bytes(cic);
  if (smem > 200 * 1024) throw std::runtime_error("conv1d: tile does not fit shared memory (k*dil too large)");
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev & 63]) {
    cudaFuncSetAttribute(conv1d_kernel<CPT, WR, TPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_set[dev & 63] = true;
  }
  dim3 grid((max_len + TT - 1) / TT, (a.rows + ROWS - 1) / ROWS, B);
  launch_k(conv1d_kernel<CPT, WR, TPT>, dim3(grid), dim3(256), smem, st, a);
  count_launch();
}

}  // namespace

void launch_conv1d(ConvArgs a, int B, int max_len, cudaStream_t st) {
  if (B <= 0 || max_len <= 0) return;
  if (a.rows_p % 4 != 0) throw std::runtime_error("conv1d: rows_p must be a multiple of 4");
  if (a.epi == EPI_GATE && (a.rows % 2) != 0) throw std::runtime_error("conv1d: gated conv needs even rows");
  // Tile choice: fill >= ~2 waves of 148 SMs x 2 CTAs when the problem allows, else shrink the time tile.
  const long long target = 148LL * 2;
  auto blocks = [&](int rows_tile, int tt) {
    return (long long)((max_len + tt - 1) / tt) * ((a.rows + rows_tile - 1) / rows_tile) * B;
  };
  if (a.rows <= 32) {
    if (blocks(32, 256) >= target) launch_cfg<8, 4, 4>(a, B, max_len, st);
    else launch_cfg<8, 4, 1>(a, B, max_len, st);
  } else {
    if (blocks(64, 256) >= target) launch_cfg<8, 8, 8>(a, B, max_len, st);
    else if (blocks(64, 64) >= target) launch_cfg<8, 8, 2>(a, B, max_len, st);
    else launch_cfg<8, 8, 1>(a, B, max_len, st);
  }
}

}  // namespace pb200
