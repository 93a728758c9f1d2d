// Text-encoder kernels: embedding gather, relative-position multi-head attention, channel LayerNorm.
//
// Reference: TextEncoder.forward (models.py:198-209), Encoder.forward (attentions.py:60-74),
// MultiHeadAttention.attention (attentions.py:225-272) with the banded closed form of the
// relative-position terms (SURVEY.md App. A.1-3, validated there to 1.8e-7):
//     S[i,j]  = (q_i/sqrt(dk)) . k_j  +  [|j-i| <= w] (q_i/sqrt(dk)) . emb_rel_k[j-i+w]
//     O_i     = sum_j P[i,j] v_j      +  sum_{|j-i|<=w} P[i,j] emb_rel_v[j-i+w]
// and modules.LayerNorm (modules.py:23-26): LayerNorm over the CHANNEL axis, eps 1e-5.
#include "kernels.cuh"
#include <algorithm>
#include "launch.cuh"

#include <cstdlib>

#include <stdexcept>

namespace pb200 {
void count_launch();

namespace {

__global__ void embed_kernel(const int* __restrict__ ids, int ids_pitch, const float* __restrict__ emb, int H,
                             float scale, View x, const int* __restrict__ len, int Tmax) {
  pdl_launch_dependents();   // programmatic dependent launch (launch.cuh): the next grid may be scheduled now;
  pdl_wait();                // nothing below runs before the previous grid has completed
  const int b = blockIdx.z;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= len[b]) return;
  const int id = ids[(long long)b * ids_pitch + t];
  const float* e = emb + (long long)id * H;
  float* xb = x.p + (long long)b * x.bs;
  for (int c = blockIdx.y; c < H; c += gridDim.y) xb[(long long)c * x.cs + t] = __ldg(e + c) * scale;
}

// ATT_QPW query rows per warp, 8 warps per CTA.  Keys/values stream through shared memory in chunks of 32 with an
// online softmax; within a chunk every K element read feeds ATT_QPW score FMAs and every V element read feeds ATT_QPW
// accumulator FMAs (the probability of key jj for query qq comes by warp shuffle).  The banded relative-value term
// touches at most 2*window+1 keys per query and is added separately.  dk <= 128 (lane owns d = lane + 32*r, r < 4).
constexpr int ATT_QPW = 4;
constexpr int ATT_Q = 8 * ATT_QPW;
constexpr int ATT_MAXR = 4;

// CUDA-core attention: the fallback for shapes the tensor-core kernel (att_mma.cu) declines, and all of it under
// PIPER_B200_ATT3=0.  The staged queries are kept per warp as [d][4 queries], so the score loop issues one K load and ONE
// 16-byte broadcast load per 4 FMAs instead of one K load and four scalar broadcast loads - the loop is bound by the
// shared-memory pipe (DESIGN.md section 8).
static_assert(ATT_QPW == 4, "rel_attention_kernel2 packs the four queries of a warp into one float4");
__global__ void __launch_bounds__(256) rel_attention_kernel2(View qkv, View out, const float* __restrict__ rel_k,
                                                            const float* __restrict__ rel_v, int H, int dk, int window,
                                                            const int* __restrict__ len, int tail_thr) {
  pdl_launch_dependents();   // programmatic dependent launch (launch.cuh): the next grid may be scheduled now;
  pdl_wait();                // nothing below runs before the previous grid has completed
  extern __shared__ float sm[];
  const int b = blockIdx.z, h = blockIdx.y;
  const int T = len[b];
  int i0 = blockIdx.x * ATT_Q;
  if (tail_thr > 0) {
    // tail mode: only the rows of a short last 128-query tile, which the tensor-core kernel (att_body.inl) skipped
    const int q0 = ((T - 1) / 128) * 128;
    if (T <= 0 || q0 == 0 || T - q0 > tail_thr) return;
    i0 += q0;
  }
  if (i0 >= T) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nrel = 2 * window + 1;
  float* Ks = sm;                       // [dk][33]
  float* Vs = Ks + dk * 33;             // [dk][33]
  float* Qs = Vs + dk * 33;             // [ATT_Q][dk]
  float* Rl = Qs + ATT_Q * dk;          // [ATT_Q][nrel]   relative-key logits per query
  float* Ev = Rl + ATT_Q * nrel;        // [nrel][dk]      emb_rel_v

  const float* base = qkv.p + (long long)b * qkv.bs;
  const float* qg = base + (long long)(h * dk) * qkv.cs;
  const float* kg = base + (long long)(H + h * dk) * qkv.cs;
  const float* vg = base + (long long)(2 * H + h * dk) * qkv.cs;

  for (int idx = threadIdx.x; idx < ATT_Q * dk; idx += 256) {
    const int d = idx / ATT_Q, qi = idx - d * ATT_Q;          // consecutive threads -> consecutive query positions
    const int i = i0 + qi;
    // per-warp transposed layout [warp][d][ATT_QPW]: one 16-byte broadcast load brings q[d] of the warp's four queries
    Qs[((qi / ATT_QPW) * dk + d) * ATT_QPW + (qi % ATT_QPW)] = i < T ? qg[(long long)d * qkv.cs + i] / sqrtf((float)dk) : 0.f;
  }
  for (int idx = threadIdx.x; idx < nrel * dk; idx += 256) Ev[idx] = rel_v[idx];
  __syncthreads();
  // relative-key logits: Rl[qi][r] = q_i . emb_rel_k[r]
#pragma unroll
  for (int qq = 0; qq < ATT_QPW; ++qq) {
    const int qi = warp * ATT_QPW + qq;
    for (int r = 0; r < nrel; ++r) {
      float p = 0.f;
      for (int d = lane; d < dk; d += 32) p += Qs[(warp * dk + d) * ATT_QPW + qq] * __ldg(rel_k + r * dk + d);
      for (int o = 16; o; o >>= 1) p += __shfl_xor_sync(0xffffffffu, p, o);
      if (lane == 0) Rl[qi * nrel + r] = p;
    }
  }
  __syncwarp();

  float m_run[ATT_QPW], l_run[ATT_QPW], acc[ATT_QPW][ATT_MAXR];
#pragma unroll
  for (int qq = 0; qq < ATT_QPW; ++qq) {
    m_run[qq] = -INFINITY;
    l_run[qq] = 0.f;
#pragma unroll
    for (int r = 0; r < ATT_MAXR; ++r) acc[qq][r] = 0.f;
  }
  const int iq0 = i0 + warp * ATT_QPW;            // first query row of this warp

  for (int j0 = 0; j0 < T; j0 += 32) {
    __syncthreads();  // previous chunk fully consumed
    for (int idx = threadIdx.x; idx < dk * 32; idx += 256) {
      const int d = idx >> 5, jj = idx & 31;
      const int j = j0 + jj;
      float kv = 0.f, vv = 0.f;
      if (j < T) {
        kv = kg[(long long)d * qkv.cs + j];
        vv = vg[(long long)d * qkv.cs + j];
      }
      Ks[d * 33 + jj] = kv;
      Vs[d * 33 + jj] = vv;
    }
    __syncthreads();
    if (iq0 >= T) continue;                        // warp-uniform; the barriers above are still reached
    const int j = j0 + lane;
    const int jn = min(32, T - j0);
    float s[ATT_QPW];
#pragma unroll
    for (int qq = 0; qq < ATT_QPW; ++qq) s[qq] = 0.f;
    const float4* qw = reinterpret_cast<const float4*>(Qs) + warp * dk;
    for (int d = 0; d < dk; ++d) {
      const float kd = Ks[d * 33 + lane];
      const float4 q4 = qw[d];                          // 2 shared-memory instructions per 4 FMAs instead of 5
      s[0] = fmaf(q4.x, kd, s[0]);
      s[1] = fmaf(q4.y, kd, s[1]);
      s[2] = fmaf(q4.z, kd, s[2]);
      s[3] = fmaf(q4.w, kd, s[3]);
    }
    float p[ATT_QPW];
#pragma unroll
    for (int qq = 0; qq < ATT_QPW; ++qq) {
      const int i = iq0 + qq;
      float sc = s[qq];
      const int rel = j - i + window;
      if (rel >= 0 && rel < nrel) sc += Rl[(warp * ATT_QPW + qq) * nrel + rel];
      if (j >= T || i >= T) sc = -INFINITY;   // keys past the utterance: masked_fill(-1e4) -> exp underflows to exactly 0
      float cmax = sc;
      for (int o = 16; o; o >>= 1) cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
      const float m_new = fmaxf(m_run[qq], cmax);
      const float corr = (m_new == -INFINITY) ? 1.f : expf(m_run[qq] - m_new);
      p[qq] = (m_new == -INFINITY) ? 0.f : expf(sc - m_new);
      float psum = p[qq];
      for (int o = 16; o; o >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
      l_run[qq] = l_run[qq] * corr + psum;
#pragma unroll
      for (int r = 0; r < ATT_MAXR; ++r) acc[qq][r] *= corr;
      m_run[qq] = m_new;
      // banded relative values: keys j with |j - i| <= window inside this chunk
      const int jlo = max(j0, i - window), jhi = min(j0 + jn - 1, i + window);
      for (int jb = jlo; jb <= jhi; ++jb) {
        const float pj = __shfl_sync(0xffffffffu, p[qq], jb - j0);
        const int relj = jb - i + window;
#pragma unroll
        for (int r = 0; r < ATT_MAXR; ++r) {
          const int d = lane + 32 * r;
          if (d < dk) acc[qq][r] = fmaf(pj, Ev[relj * dk + d], acc[qq][r]);
        }
      }
    }
    // P.V: one V read per (key, channel) shared by the warp's queries
    for (int jj = 0; jj < jn; ++jj) {
      float pj[ATT_QPW];
#pragma unroll
      for (int qq = 0; qq < ATT_QPW; ++qq) pj[qq] = __shfl_sync(0xffffffffu, p[qq], jj);
#pragma unroll
      for (int r = 0; r < ATT_MAXR; ++r) {
        const int d = lane + 32 * r;
        if (d < dk) {
          const float v = Vs[d * 33 + jj];
#pragma unroll
          for (int qq = 0; qq < ATT_QPW; ++qq) acc[qq][r] = fmaf(pj[qq], v, acc[qq][r]);
        }
      }
    }
  }
  float* ob = out.p + (long long)b * out.bs + (long long)(h * dk) * out.cs;
#pragma unroll
  for (int qq = 0; qq < ATT_QPW; ++qq) {
    const int i = iq0 + qq;
    if (i >= T) continue;
#pragma unroll
    for (int r = 0; r < ATT_MAXR; ++r) {
      const int d = lane + 32 * r;
      if (d < dk) ob[(long long)d * out.cs + i] = acc[qq][r] / l_run[qq];
    }
  }
}

// The rows of a SHORT last 128-query tile (launch_rel_attention: tail mode), key-parallel: one CTA per (utterance, head,
// ATT_QPW rows); every warp walks its own share of the 32-key chunks (chunk c for warp c % n_w) with a private K / V
// stage and its own online-softmax state, the states are merged at the end (m = max, l and the accumulators rescaled).
// Same arithmetic per key as rel_attention_kernel2; only the order in which the chunks meet differs.  With the generic
// kernel in tail mode one warp per CTA walked all nine chunks of a 259-id utterance behind block-wide barriers (~60 us
// per launch, as long as the tensor-core CTAs it was meant to relieve).
__global__ void __launch_bounds__(256) rel_attention_tail_kernel(View qkv, View out, const float* __restrict__ rel_k,
                                                                 const float* __restrict__ rel_v, int H, int dk, int window,
                                                                 const int* __restrict__ len, int tail_thr, int n_w) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];
  const int b = blockIdx.z, h = blockIdx.y;
  const int T = len[b];
  const int q0 = T > 0 ? ((T - 1) / 128) * 128 : 0;
  if (T <= 0 || q0 == 0 || T - q0 > tail_thr) return;
  const int i0 = q0 + blockIdx.x * ATT_QPW;
  if (i0 >= T) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nrel = 2 * window + 1;
  float* Qs = sm;                               // [dk][ATT_QPW]
  float* Rl = Qs + dk * ATT_QPW;                // [ATT_QPW][nrel]
  float* Ev = Rl + ATT_QPW * nrel + (4 - (ATT_QPW * nrel) % 4) % 4;   // [nrel][dk]
  float* stage = Ev + nrel * dk;                // per warp: K [dk][33] | V [dk][33]; afterwards the partial states
  const float* base = qkv.p + (long long)b * qkv.bs;
  const float* qg = base + (long long)(h * dk) * qkv.cs;
  const float* kg = base + (long long)(H + h * dk) * qkv.cs;
  const float* vg = base + (long long)(2 * H + h * dk) * qkv.cs;
  for (int idx = threadIdx.x; idx < ATT_QPW * dk; idx += 256) {
    const int d = idx / ATT_QPW, qq = idx - d * ATT_QPW;
    const int i = i0 + qq;
    Qs[d * ATT_QPW + qq] = i < T ? qg[(long long)d * qkv.cs + i] / sqrtf((float)dk) : 0.f;
  }
  for (int idx = threadIdx.x; idx < nrel * dk; idx += 256) Ev[idx] = rel_v[idx];
  __syncthreads();
  for (int pr = warp; pr < ATT_QPW * nrel; pr += 8) {      // relative-key logits Rl[qq][r] = q . emb_rel_k[r]
    const int qq = pr / nrel, r = pr - qq * nrel;
    float p = 0.f;
    for (int d = lane; d < dk; d += 32) p += Qs[d * ATT_QPW + qq] * __ldg(rel_k + r * dk + d);
    for (int o = 16; o; o >>= 1) p += __shfl_xor_sync(0xffffffffu, p, o);
    if (lane == 0) Rl[pr] = p;
  }
  __syncthreads();

  float m_run[ATT_QPW], l_run[ATT_QPW], acc[ATT_QPW][ATT_MAXR];
#pragma unroll
  for (int qq = 0; qq < ATT_QPW; ++qq) {
    m_run[qq] = -INFINITY;
    l_run[qq] = 0.f;
#pragma unroll
    for (int r = 0; r < ATT_MAXR; ++r) acc[qq][r] = 0.f;
  }
  if (warp < n_w) {
    float* Ks = stage + (size_t)warp * 2 * dk * 33;
    float* Vs = Ks + dk * 33;
    for (int j0 = warp * 32; j0 < T; j0 += n_w * 32) {
      __syncwarp();
      const int j = j0 + lane;
      for (int d = 0; d < dk; ++d) {
        Ks[d * 33 + lane] = j < T ? kg[(long long)d * qkv.cs + j] : 0.f;
        Vs[d * 33 + lane] = j < T ? vg[(long long)d * qkv.cs + j] : 0.f;
      }
      __syncwarp();
      const int jn = min(32, T - j0);
      float s[ATT_QPW];
#pragma unroll
      for (int qq = 0; qq < ATT_QPW; ++qq) s[qq] = 0.f;
      const float4* qw = reinterpret_cast<const float4*>(Qs);
      for (int d = 0; d < dk; ++d) {
        const float kd = Ks[d * 33 + lane];
        const float4 q4 = qw[d];
        s[0] = fmaf(q4.x, kd, s[0]);
        s[1] = fmaf(q4.y, kd, s[1]);
        s[2] = fmaf(q4.z, kd, s[2]);
        s[3] = fmaf(q4.w, kd, s[3]);
      }
      float p[ATT_QPW];
#pragma unroll
      for (int qq = 0; qq < ATT_QPW; ++qq) {
        const int i = i0 + qq;
        float sc = s[qq];
        const int rel = j - i + window;
        if (rel >= 0 && rel < nrel) sc += Rl[qq * nrel + rel];
        if (j >= T || i >= T) sc = -INFINITY;
        float cmax = sc;
        for (int o = 16; o; o >>= 1) cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
        const float m_new = fmaxf(m_run[qq], cmax);
        const float corr = (m_new == -INFINITY) ? 1.f : expf(m_run[qq] - m_new);
        p[qq] = (m_new == -INFINITY) ? 0.f : expf(sc - m_new);
        float psum = p[qq];
        for (int o = 16; o; o >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
        l_run[qq] = l_run[qq] * corr + psum;
#pragma unroll
        for (int r = 0; r < ATT_MAXR; ++r) acc[qq][r] *= corr;
        m_run[qq] = m_new;
        const int jlo = max(j0, i - window), jhi = min(j0 + jn - 1, i + window);   // banded relative values
        for (int jb = jlo; jb <= jhi; ++jb) {
          const float pj = __shfl_sync(0xffffffffu, p[qq], jb - j0);
          const int relj = jb - i + window;
#pragma unroll
          for (int r = 0; r < ATT_MAXR; ++r) {
            const int d = lane + 32 * r;
            if (d < dk) acc[qq][r] = fmaf(pj, Ev[relj * dk + d], acc[qq][r]);
          }
        }
      }
      for (int jj = 0; jj < jn; ++jj) {
        float pj[ATT_QPW];
#pragma unroll
        for (int qq = 0; qq < ATT_QPW; ++qq) pj[qq] = __shfl_sync(0xffffffffu, p[qq], jj);
#pragma unroll
        for (int r = 0; r < ATT_MAXR; ++r) {
          const int d = lane + 32 * r;
          if (d < dk) {
            const float v = Vs[d * 33 + jj];
#pragma unroll
            for (int qq = 0; qq < ATT_QPW; ++qq) acc[qq][r] = fmaf(pj[qq], v, acc[qq][r]);
          }
        }
      }
    }
  }
  __syncthreads();                                   // every warp is done with its stage: reuse it for the partial states
  float* Pm = stage;                                 // [n_w][ATT_QPW]
  float* Pl = Pm + 8 * ATT_QPW;                      // [n_w][ATT_QPW]
  float* Pa = Pl + 8 * ATT_QPW;                      // [n_w][ATT_QPW][128]
  if (warp < n_w) {
#pragma unroll
    for (int qq = 0; qq < ATT_QPW; ++qq) {
      if (lane == 0) { Pm[warp * ATT_QPW + qq] = m_run[qq]; Pl[warp * ATT_QPW + qq] = l_run[qq]; }
#pragma unroll
      for (int r = 0; r < ATT_MAXR; ++r) Pa[(warp * ATT_QPW + qq) * 128 + lane + 32 * r] = acc[qq][r];
    }
  }
  __syncthreads();
  if (warp < ATT_QPW) {
    const int qq = warp, i = i0 + qq;
    if (i < T) {
      float M = -INFINITY;
      for (int w = 0; w < n_w; ++w) M = fmaxf(M, Pm[w * ATT_QPW + qq]);
      float Lsum = 0.f, o[ATT_MAXR] = {0.f, 0.f, 0.f, 0.f};
      for (int w = 0; w < n_w; ++w) {
        const float mw = Pm[w * ATT_QPW + qq];
        const float f = mw == -INFINITY ? 0.f : expf(mw - M);
        Lsum = fmaf(Pl[w * ATT_QPW + qq], f, Lsum);
#pragma unroll
        for (int r = 0; r < ATT_MAXR; ++r) o[r] = fmaf(Pa[(w * ATT_QPW + qq) * 128 + lane + 32 * r], f, o[r]);
      }
      float* ob = out.p + (long long)b * out.bs + (long long)(h * dk) * out.cs;
#pragma unroll
      for (int r = 0; r < ATT_MAXR; ++r) {
        const int d = lane + 32 * r;
        if (d < dk) ob[(long long)d * out.cs + i] = o[r] / Lsum;
      }
    }
  }
}

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f)); }

// LayerNorm over channels for a tile of 32 time steps; the warps split the channel axis.  Values are staged in shared
// memory [C][33] so the (optional) depthwise conv is evaluated once.  Every warp issues its global loads eight channel rows
// at a time before using any of them: walking 24 rows (C = 192) one dependent load -> store at a time in both passes
// measured ~28 us per launch (36 launches per step), ~2 x 24 exposed L2 / DRAM latencies with only 16 warps per SM to
// hide them.
constexpr int LN_U = 8;
// NW warps per CTA: 24 for C >= 96 (each warp then owns <= 8 channel rows: ONE batch of loads per pass instead of three)
template <int NW>
__global__ void __launch_bounds__(NW * 32) layernorm_kernel2(const LnArgs a) {
  pdl_launch_dependents();   // programmatic dependent launch (launch.cuh): the next grid may be scheduled now;
  pdl_wait();                // nothing below runs before the previous grid has completed
  extern __shared__ float sm[];  // [C][33] | gamma [C] | beta [C] | dw_b [C] | dw_w [C][dw_k]
  __shared__ float red[NW][32];
  const int b = blockIdx.z;
  const int T = a.len[b];
  const int t0 = blockIdx.x * 32;
  if (t0 >= T) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int t = t0 + lane;
  const bool live = t < T;
  const int C = a.C;
  const float* ab = a.a.p + (long long)b * a.a.bs;
  // Per-channel parameters go to shared memory once: read through __ldg inside the loops they were 24 dependent L2 round
  // trips per warp in the output pass alone (39 % of this kernel's stall samples, profiles/r02_ncu_ln.txt).
  float* gs = sm + C * 33;
  float* bs = gs + C;
  float* dwb = bs + C;
  float* dww = dwb + C;
  for (int c = threadIdx.x; c < C; c += NW * 32) {
    gs[c] = a.gamma[c];
    bs[c] = a.beta[c];
  }
  if (a.mode == LN_DW_GELU) {
    for (int c = threadIdx.x; c < C; c += NW * 32) dwb[c] = a.dw_b[c];
    for (int i = threadIdx.x; i < C * a.dw_k; i += NW * 32) dww[i] = a.dw_w[i];
    __syncthreads();                                     // (uniform branch) the depthwise taps are used in the load phase
  }
  for (int c0 = warp; c0 < C; c0 += NW * LN_U) {
    float v[LN_U];
    if (a.mode == LN_DW_GELU) {
      const int half = (a.dw_k - 1) / 2;
#pragma unroll
      for (int u = 0; u < LN_U; ++u) {
        const int c = c0 + NW * u;
        v[u] = 0.f;
        if (live && c < C) {
          const float* ar = ab + (long long)c * a.a.cs;
          float acc = dwb[c];
          for (int j = 0; j < a.dw_k; ++j) {
            const int tt = t + (j - half) * a.dw_dil;
            if (tt >= 0 && tt < T) acc = fmaf(dww[c * a.dw_k + j], ar[tt], acc);
          }
          v[u] = acc;
        }
      }
    } else {
      float w2[LN_U];
#pragma unroll
      for (int u = 0; u < LN_U; ++u) {
        const int c = c0 + NW * u;
        v[u] = 0.f;
        w2[u] = 0.f;
        if (live && c < C) {
          v[u] = ab[(long long)c * a.a.cs + t];
          if (a.mode == LN_ADD) w2[u] = a.b.p[(long long)b * a.b.bs + (long long)c * a.b.cs + t];
        }
      }
      if (a.mode == LN_ADD) {
#pragma unroll
        for (int u = 0; u < LN_U; ++u) v[u] += w2[u];
      }
    }
#pragma unroll
    for (int u = 0; u < LN_U; ++u) {
      const int c = c0 + NW * u;
      if (c < C) sm[c * 33 + lane] = v[u];
    }
  }
  __syncthreads();
  float s = 0.f;
  for (int c = warp; c < C; c += NW) s += sm[c * 33 + lane];
  red[warp][lane] = s;
  __syncthreads();
  float mean = 0.f;
#pragma unroll
  for (int w = 0; w < NW; ++w) mean += red[w][lane];
  mean /= (float)C;
  __syncthreads();
  float q = 0.f;
  for (int c = warp; c < C; c += NW) {
    const float d = sm[c * 33 + lane] - mean;
    q = fmaf(d, d, q);
  }
  red[warp][lane] = q;
  __syncthreads();
  float var = 0.f;
#pragma unroll
  for (int w = 0; w < NW; ++w) var += red[w][lane];
  var /= (float)C;
  const float rstd = 1.f / sqrtf(var + 1e-5f);
  if (!live) return;
  float* yb = a.y.p + (long long)b * a.y.bs;
  for (int c0 = warp; c0 < C; c0 += NW * LN_U) {
    float rv[LN_U];
#pragma unroll
    for (int u = 0; u < LN_U; ++u) {                      // the residual loads of the whole batch first
      const int c = c0 + NW * u;
      rv[u] = (a.mode == LN_GELU_RES && c < C) ? a.r.p[(long long)b * a.r.bs + (long long)c * a.r.cs + t] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < LN_U; ++u) {
      const int c = c0 + NW * u;
      if (c >= C) continue;
      float v = (sm[c * 33 + lane] - mean) * rstd * gs[c] + bs[c];
      if (a.mode == LN_GELU_RES || a.mode == LN_DW_GELU) v = gelu_erf(v);
      if (a.mode == LN_GELU_RES) v += rv[u];
      yb[(long long)c * a.y.cs + t] = v;
    }
  }
}

}  // namespace

void launch_embed(const int* ids, int ids_pitch, const float* emb, int H, float scale, View x, const int* len, int B,
                  int Tmax, cudaStream_t st) {
  if (B <= 0 || Tmax <= 0) return;
  dim3 grid((Tmax + 127) / 128, 8, B);
  launch_k(embed_kernel, dim3(grid), dim3(128), 0, st, ids, ids_pitch, emb, H, scale, x, len, Tmax);
  count_launch();
}

void launch_rel_attention(View qkv, View out, const float* rel_k, const float* rel_v, int H, int n_heads, int window,
                          const int* len, int B, int Tmax, cudaStream_t st) {
  if (B <= 0 || Tmax <= 0) return;
  const int dk = H / n_heads;
  if (dk > 32 * ATT_MAXR) throw std::runtime_error("attention: head width > 128 is not supported");
  const int nrel = 2 * window + 1;
  const size_t smem = size_t(2 * dk * 33 + ATT_Q * dk + ATT_Q * nrel + nrel * dk) * sizeof(float);
  int dev = 0;
  cudaGetDevice(&dev);
  auto kernel2_attr = [dev] {        // set where the CUDA-core kernel runs: the default path never loads it
    static bool attr_set[64] = {};
    if (!attr_set[dev & 63]) {
      cudaFuncSetAttribute(rel_attention_kernel2, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
      attr_set[dev & 63] = true;
    }
  };
  dim3 grid((Tmax + ATT_Q - 1) / ATT_Q, n_heads, B);
  static int g_att3 = -1;                                 // PIPER_B200_ATT3: tensor-core attention (att_mma.cu)
  if (g_att3 < 0) {
    const char* e = std::getenv("PIPER_B200_ATT3");
    g_att3 = e ? std::atoi(e) : 1;                       // default on (0 = CUDA-core kernel for every shape)
  }
  int tail_thr = 0;
  if (g_att3 && launch_rel_attention_tc(qkv, out, rel_k, rel_v, H, n_heads, window, len, B, Tmax, st, &tail_thr)) {
    if (tail_thr > 0) {                                  // short last tiles: the CUDA-core kernel, one CTA per ATT_Q rows
      static bool attr2[64] = {};
      if (!attr2[dev & 63]) {
        cudaFuncSetAttribute(rel_attention_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);
        attr2[dev & 63] = true;
      }
      // warps that walk key chunks: as many private K | V stages as fit (8 for dk = 96, 5 for dk = 128); the same region
      // later holds the 8 x ATT_QPW x (128 + 2) partial states
      const size_t fixed = size_t(dk * ATT_QPW + ATT_QPW * nrel + 4 + nrel * dk) * sizeof(float);
      const size_t per_warp = size_t(2) * dk * 33 * sizeof(float), part = size_t(8) * ATT_QPW * 130 * sizeof(float);
      int n_w = int(std::min<size_t>(8, (size_t(212) * 1024 - fixed) / per_warp));
      if (n_w >= 1) {
        const size_t smem_t = fixed + std::max(per_warp * n_w, part);
        launch_k(rel_attention_tail_kernel, dim3((tail_thr + ATT_QPW - 1) / ATT_QPW, n_heads, B), dim3(256), smem_t, st, qkv, out,
                 rel_k, rel_v, H, dk, window, len, tail_thr, n_w);
      } else {
        kernel2_attr();
        launch_k(rel_attention_kernel2, dim3((tail_thr + ATT_Q - 1) / ATT_Q, n_heads, B), dim3(256), smem, st, qkv, out, rel_k, rel_v, H,
                 dk, window, len, tail_thr);
      }
      count_launch();
    }
    return;
  }
  kernel2_attr();
  launch_k(rel_attention_kernel2, dim3(grid), dim3(256), smem, st, qkv, out, rel_k, rel_v, H, dk, window, len, 0);
  count_launch();
}

void launch_layernorm(const LnArgs& a, int B, int Tmax, cudaStream_t st) {
  if (B <= 0 || Tmax <= 0) return;
  const size_t smem = (size_t(a.C) * 33 + size_t(a.C) * (3 + (a.mode == LN_DW_GELU ? a.dw_k : 0))) * sizeof(float);
  if (smem > 96 * 1024) throw std::runtime_error("layernorm: channel count too large");
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev & 63]) {
    cudaFuncSetAttribute(layernorm_kernel2<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    cudaFuncSetAttribute(layernorm_kernel2<24>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    attr_set[dev & 63] = true;
  }
  dim3 grid((Tmax + 31) / 32, 1, B);
  static int g_ln_warps = -1;                             // PIPER_B200_LN_WARPS: 8 / 24 warps per CTA (default: by problem size)
  if (g_ln_warps < 0) {
    const char* e = std::getenv("PIPER_B200_LN_WARPS");
    g_ln_warps = e ? std::atoi(e) : 0;
  }
  // 24 warps (one batch of loads per pass) shorten a latency-bound launch; with several CTAs per SM already resident the
  // 8-warp form has the same loads in flight and less barrier traffic (measured: batch 1 prefers 24, batch 32 prefers 8)
  const bool wide = g_ln_warps ? g_ln_warps == 24 : (long long)grid.x * B <= 148;
  if (a.C >= 96 && wide) launch_k(layernorm_kernel2<24>, dim3(grid), dim3(24 * 32), smem, st, a);
  else launch_k(layernorm_kernel2<8>, dim3(grid), dim3(256), smem, st, a);
  count_launch();
}

}  // namespace pb200
