// Kernel launch interface of the sm_100a VITS engine (device code in *.cu next to this file).
//
// Layout convention everywhere: activations are fp32 [B][C][Lp], time contiguous (the reference's
// [B,C,T] channel-major layout, models.py / modules.py), Lp = padded row pitch (multiple of 4 floats
// so rows are 16-byte aligned).  Batches are RAGGED: item b is valid on [0, len[b]*len_scale); every
// kernel zero-fills reads outside that range and never stores outside it, which gives each utterance
// its own zero padding (SURVEY.md App. A.9: parity is per utterance against the B = 1 reference).
#pragma once
#include <cuda_runtime.h>

#include "voice.h"
#include <cstdint>
#include <cstring>
#include <vector>

namespace pb200 {

struct View {        // a [B][C][L] activation view
  float* p = nullptr;
  long long bs = 0;  // batch stride (floats)
  int cs = 0;        // channel stride (floats)
  __host__ __device__ View offset_channels(int c) const { return View{p + (long long)c * cs, bs, cs}; }
};

enum PreAct { PRE_NONE = 0, PRE_LRELU = 1 };

enum Epilogue {
  EPI_BIAS = 0,      // y = v
  EPI_RELU = 1,      // y = max(v, 0)
  EPI_RES = 2,       // y = v + r
  EPI_GATE = 3,      // rows interleaved (a_i, b_i): y[row/2] = tanh(a) * sigmoid(b)      (commons.py:99-106)
  EPI_WN = 4,        // row < split: y = r + v (residual stream, in place); row >= split: y2 (+)= v (skip sum)
  EPI_SUBFROM = 5,   // y = r - v                                                          (modules.py:464)
  EPI_UPSAMPLE = 6,  // ConvTranspose pixel-shuffle store: y[row/up][q*up + row%up - up_pad] = v
  EPI_MRF = 7,       // v' = v + r; mrf 0: y2 = v'; 1: y2 += v'; 2: y2 = (y2 + v') / mrf_n   (models.py:356-363)
};

struct ConvArgs {
  View x, y, y2, r;
  const float* w = nullptr;     // [ci][k][rows_p]
  const float* bias = nullptr;  // [rows] or null
  const float* bias_item = nullptr;  // optional per-item bias (speaker conditioning): + bias_item[b * bias_item_stride + row]
  int bias_item_stride = 0;
  const int* len = nullptr;     // per item
  int len_scale = 1;            // valid input length = len[b] * len_scale
  int ci = 0, rows = 0, rows_p = 0, k = 1, dil = 1, pad = 0;
  int q_extra = 0;              // output positions computed past the input length (ConvTranspose tail)
  int pre = PRE_NONE;
  float slope = 0.f;
  int epi = EPI_BIAS;
  int split = 0, first = 0;     // EPI_WN
  int up = 1, up_pad = 0;       // EPI_UPSAMPLE
  int mrf = 0, mrf_n = 1;       // EPI_MRF
  int cic = 16;                 // input-channel chunk staged in shared memory (set by the launcher)
  const ConvW* host_w = nullptr;  // host-side only: the layer this launch came from (tensor-core plan lookup)
};

// max_len = max over the batch of (len[b]*len_scale + q_extra): sizes the grid.
void launch_conv1d(ConvArgs a, int B, int max_len, cudaStream_t st);

// What a TMA tensor map over an activation view [B][C][pitch] is built from (conv_mma2.cu encodes the CUtensorMap from
// it; the CPU model in tests/sim executes it directly): element (x = time, y = channel, z = item), fp32, out-of-bounds
// elements of a box read as zero.
struct TmapDesc {
  const float* base = nullptr;
  int dims[3] = {0, 0, 0};                  // pitch, channels, items
  long long stride1 = 0, stride2 = 0;       // bytes between channels / items
  int box[3] = {0, 0, 1};                   // floats per row, rows, 1
};

// CUtensorMap (128 bytes, 64-byte aligned) from a TmapDesc through cuTensorMapEncodeTiled; false = the driver refused it.
bool encode_tmap(const TmapDesc& d, void* out_cutensormap);

// ---- persistent tensor-core (tcgen05) Conv1d / ConvTranspose1d with split precision (conv_mma2.cu) -------------
struct MmaConvArgs {
  View x, y, y2, r;
  const uint8_t* w = nullptr;    // packed by conv2_pack
  const float* bias = nullptr;
  const float* bias_item = nullptr;   // optional per-item bias (speaker conditioning)
  int bias_item_stride = 0;
  const int* len = nullptr;
  int len_scale = 1;
  int ci = 0, rows = 0, k = 1, dil = 1, pad = 0, q_extra = 0;
  int pre = PRE_NONE;
  float slope = 0.f;
  int epi = EPI_BIAS;
  int split = 0, first = 0, up = 1, up_pad = 0, mrf = 0, mrf_n = 1;
  int kc = 0, stage_rows = 0, n_tile = 0, tmem_cols = 0, a_slots = 1;   // from the Conv2Layer plan
  int chains = 1, mh_stride = 0;
  int raw_stride = 0, tiles_per_item = 0, total_tiles = 0, batch = 0, t_slots = 1;
  int tm_boxes = 0;              // conv2 tensor-map mode: boxes per channel chunk (0 = per-row bulk copies)
  int mma3 = 0;                  // conv2: three instructions per k-step on exactly matching accumulator regions (see conv2_body.inl)
  // conv2 flat mode: the views are laid out [channel][item][slot of flat_tg floats] (View.bs = flat_tg, View.cs = items *
  // flat_tg), the launch sees ONE item of length flat_n * flat_tg and tiles are cut on that concatenated time axis; a row
  // g belongs to item g / flat_tg at time g % flat_tg and is live while that is < len[item] * len_scale.
  int flat_tg = 0, flat_n = 0;
  // conv2 A-stationary order: output-row tiles of one position are consecutive tiles of ONE CTA, and the converted
  // activation window (all its channel chunks fit the operand ring) is loaded and converted once per position instead of
  // once per output-row tile.  n_tiles = output-row tiles per position.
  int astat = 0, n_tiles = 1;
  unsigned long long* prof = nullptr;   // optional: per-role stall cycle counters (tools/conv_diag.py)
};

struct Conv2Layer {          // tiling of one layer + where its stacked weights live (filled lazily by the engine)
  bool tf32 = false;
  int prec = 0;              // 0 bf16x3, 1 tf32x3, 2 fp16x3 (conv2_body.inl)
  int n_tile = 0, n_tiles = 0, mt = 128, kc = 0, stage_rows = 0, raw_stride = 0, t_slots = 1, tmem_cols = 0, chains = 1, mh_stride = 0;
  size_t smem = 0, w_bytes = 0;
  void* w_dev = nullptr;
};
bool conv2_plan(int ci, int rows, int k, int dil, int prec, int chains, Conv2Layer& l);
void conv2_pack(const float* wsrc, int ci, int k, int rows_p, const Conv2Layer& l, uint8_t* out);
void launch_conv2(MmaConvArgs a, const Conv2Layer& l, int B, int max_len, cudaStream_t st);

// ---- one whole MRF stage (three resblocks) of the generator per launch (mrf_fused.cu; default for 32-channel stages) ----
constexpr int MRF_MAX_CHAINS = 3, MRF_MAX_STEPS = 6;
struct MrfFusedPlan {
  bool ok = false;
  int n_chains = 0, n_steps = 0, pair = 1;      // pair: convs per residual unit (ResBlock2: 1, ResBlock1: 2)
  int k[MRF_MAX_CHAINS] = {0, 0, 0};
  int dil[MRF_MAX_CHAINS][MRF_MAX_STEPS] = {};
  int hv = 0, to = 0;                           // rows dropped on each side of a 256-row tile / positions stored per tile
  int post_k = 0;                               // > 0: conv_post (k taps, no bias) + tanh fused behind the stage; its half-width is in hv
  size_t w_bytes = 0;                           // packed tap tiles
  int n_bias = 0;                               // floats
};
struct MrfFusedArgs {
  View x, y;                                    // [B][32][L] fp32 in / out
  const int* len = nullptr;
  int len_scale = 1;
  const uint8_t* w = nullptr;                   // pack_mrf_fused
  const float* bias = nullptr;
  float slope = 0.1f;
  int n_chains = 0, n_steps = 0, pair = 1, hv = 0, to = 0;
  int k[MRF_MAX_CHAINS] = {0, 0, 0};
  int dil[MRF_MAX_CHAINS][MRF_MAX_STEPS] = {};
  int tiles_per_item = 0, total_tiles = 0;
  // optional fused generator tail: audio[out_off[b] + t] = tanh(conv_post(lrelu_post_slope(y)))  (models.py:364-366)
  const float* post_w = nullptr;                // [32][post_k]
  int post_k = 0;
  float post_slope = 0.01f;
  float* audio = nullptr;
  const long long* out_off = nullptr;
};
// plan -> launch arguments (shared by the CUDA launcher and the CPU model of the kernel in tests/sim)
inline void mrf_fill_args(MrfFusedArgs& a, const MrfFusedPlan& p, int B, int max_len) {
  a.n_chains = p.n_chains; a.n_steps = p.n_steps; a.pair = p.pair; a.hv = p.hv; a.to = p.to; a.post_k = p.post_k;
  for (int c = 0; c < MRF_MAX_CHAINS; ++c) {
    a.k[c] = p.k[c];
    for (int s = 0; s < MRF_MAX_STEPS; ++s) a.dil[c][s] = p.dil[c][s];
  }
  a.tiles_per_item = (max_len + p.to - 1) / p.to;
  a.total_tiles = a.tiles_per_item * B;
}
// post_k > 0 plans the stage with conv_post + tanh fused behind it (last stage of the generator only)
bool plan_mrf_fused(const std::vector<ResBlockW>& stage, int resblock_kind, int channels, int post_k, MrfFusedPlan& p);
void pack_mrf_fused(const float* blob, const std::vector<ResBlockW>& stage, const MrfFusedPlan& p, uint8_t* w, float* bias);
void launch_mrf_fused(MrfFusedArgs a, const MrfFusedPlan& p, int B, int max_len, cudaStream_t st);

// ---- text encoder -----------------------------------------------------------------------------
void launch_embed(const int* ids, int ids_pitch, const float* emb, int H, float scale, View x, const int* len, int B,
                  int Tmax, cudaStream_t st);
// qkv: [B][3H][Lp] (q | k | v rows), out: [B][H][Lp]
void launch_rel_attention(View qkv, View out, const float* rel_k, const float* rel_v, int H, int n_heads, int window,
                          const int* len, int B, int Tmax, cudaStream_t st);

// the same attention on the tensor cores (att_mma.cu; default, PIPER_B200_ATT3=0 = CUDA cores); false = shape not handled
bool launch_rel_attention_tc(View qkv, View out, const float* rel_k, const float* rel_v, int H, int n_heads, int window,
                             const int* len, int B, int Tmax, cudaStream_t st, int* tail_thr = nullptr);

enum LnMode {
  LN_ADD = 0,          // y = LN(a + b)
  LN_GELU_RES = 1,     // y = r + gelu(LN(a))
  LN_DW_GELU = 2,      // y = gelu(LN(dwconv_k(a)))      (modules.py:117-129, first half of a DDSConv layer)
  LN_PLAIN = 3,        // y = LN(a)
};
struct LnArgs {
  View a, b, r, y;
  const float* gamma = nullptr;
  const float* beta = nullptr;
  const float* dw_w = nullptr;  // [C][k]
  const float* dw_b = nullptr;  // [C]
  int dw_k = 3, dw_dil = 1;
  int C = 0, mode = LN_ADD;
  const int* len = nullptr;
};
void launch_layernorm(const LnArgs& a, int B, int Tmax, cudaStream_t st);

// cond[b][r] = bias[r] + sum_k w[r][k] * emb_g[sid[b]][k]        (g = emb_g(sid), then every 1x1 conditioning conv at once)
void launch_speaker_cond(const float* w, const float* bias, const float* emb_g, const int* sid, float* cond, int rows,
                         int gin, int B, cudaStream_t st);

// Per-call scalars (the graph's `scales` input, piper.cpp:357-365, and the noise seed).  They live in device memory so
// that a captured CUDA graph of the pipeline does not bake them in: a replay reads the values of the current call.
struct CallParams {
  unsigned long long seed;
  float noise_scale, length_scale, noise_w, pad_;
};

// ---- stochastic duration predictor ------------------------------------------------------------
// z[b][ch][t] = eps * noise_w  (eps explicit [sum_b 2*len_b] item-major, or Philox(seed) when eps == null)
void launch_dp_noise(View z, const float* eps, const long long* eps_off, const CallParams* cp,
                     const int* len, int B, int Tmax, cudaStream_t st);
// h[c][t] = w[c] * z[x0_ch][t] + b[c] + g[c][t]
void launch_cf_pre(View z, int x0_ch, const float* w, const float* b, View g, View h, int C, const int* len, int B,
                   int Tmax, cudaStream_t st);
// inverse rational-quadratic spline on z[x1_ch] with parameters h [B][3*bins-1][Lp]   (transforms.py:50-191)
void launch_spline_inverse(View z, int x1_ch, View h, int bins, float inv_sqrt_c, float bound, const int* len, int B,
                           int Tmax, cudaStream_t st);
// logw = (z0 - m)*s ; w = exp(logw)*length_scale ; w_ceil = ceil(w) ; cum = inclusive scan ; y_len = max(sum, 1)
void launch_durations(View z, float ea_m, float ea_scale, const CallParams* cp, const int* w_override,
                      int w_override_pitch, int* cum, int cum_pitch, int* y_len, float* logw_out, const int* len,
                      int B, int Tmax, cudaStream_t st);
// z_p[c][j] = m_p[c][i(j)] + eps * exp(logs_p[c][i(j)]) * noise_scale   for j < y_len  (models.py:705-718)
void launch_expand(View stats, int inter, const int* cum, int cum_pitch, const int* len, const int* y_len, View zp,
                   const float* eps, long long eps_bs, int eps_cs, const CallParams* cp, int B,
                   int Fmax, cudaStream_t st);

// ---- generator tail / audio epilogue ------------------------------------------------------------
// out[off[b] + t] = tanh( sum_c sum_j w[c][j] * lrelu_0.01(x[c][t + j - k/2]) )      (models.py:364-366)
void launch_conv_post(View x, const float* w, int C, int k, float slope, float* out, const long long* out_off,
                      const int* len, int len_scale, int B, int max_len, cudaStream_t st);
// peak[b] = max |x| over the item (as float bits, non-negative floats order like ints)
void launch_peak(const float* audio, const long long* off, const int* len, int len_scale, unsigned int* peak, int B,
                 int max_len, cudaStream_t st);
// int16 = clamp(x * 32767 / max(0.01, peak), -32768, 32767) truncated      (piper.cpp:411-431)
void launch_to_int16(const float* audio, const long long* off, const int* len, int len_scale, const unsigned int* peak,
                     int16_t* out, int B, int max_len, cudaStream_t st);

unsigned long long launch_count();  // kernels launched by this library since load (bench.py's gpu_launches)

}  // namespace pb200
