// C ABI of the engine (declared in include/piper_b200.h).
#include "../../include/piper_b200.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <exception>
#include <stdexcept>
#include <string>

#include "engine.h"

struct pb200_voice {
  pb200::Engine engine;
  pb200_voice(const char* path, int device, bool upload = true) : engine(path, device, upload) {}
};

namespace {
thread_local std::string g_error;

template <class F>
int guarded(F&& f) {
  try {
    f();
    return PB200_OK;
  } catch (const std::exception& e) {
    g_error = e.what();
  } catch (...) {
    g_error = "unknown error";
  }
  return PB200_ERROR;
}

pb200::NoiseSpec to_spec(const pb200_noise* n) {
  pb200::NoiseSpec s;
  if (n) {
    s.eps_dp = n->eps_dp;
    s.eps_z = n->eps_z;
    s.z_stride = n->z_stride;
    s.seed = n->seed;
  }
  return s;
}
}  // namespace

extern "C" {

int pb200_voice_load(const char* onnx_path, int device, pb200_voice** out) {
  return guarded([&] {
    if (!onnx_path || !out) throw std::runtime_error("pb200_voice_load: null argument");
    *out = new pb200_voice(onnx_path, device);
  });
}

int pb200_voice_load_ex(const char* onnx_path, int device, int32_t flags, pb200_voice** out) {
  return guarded([&] {
    if (!onnx_path || !out) throw std::runtime_error("pb200_voice_load_ex: null argument");
    *out = new pb200_voice(onnx_path, device, (flags & PB200_LOAD_NO_UPLOAD) == 0);
  });
}

int pb200_voice_weight_buffers(pb200_voice* v, void** fp32, int64_t* fp32_bytes) {
  return guarded([&] {
    if (!v || !fp32 || !fp32_bytes) throw std::runtime_error("pb200_voice_weight_buffers: null argument");
    v->engine.weight_buffers(fp32, fp32_bytes);
  });
}

void pb200_voice_free(pb200_voice* v) { delete v; }

int pb200_voice_get_info(const pb200_voice* v, pb200_voice_info* info) {
  return guarded([&] {
    if (!v || !info) throw std::runtime_error("pb200_voice_get_info: null argument");
    const pb200::VoiceSpec& s = v->engine.spec();
    info->n_vocab = s.n_vocab; info->hidden = s.hidden; info->inter = s.inter; info->filter = s.filter;
    info->n_heads = s.n_heads; info->n_layers = s.n_layers; info->window = s.window; info->resblock = s.resblock;
    info->n_upsamples = int32_t(s.up_rates.size()); info->hop = s.hop; info->up_initial = s.up_initial;
    info->device = v->engine.device();
    info->n_speakers = s.n_speakers; info->gin = s.gin;
    info->n_params = v->engine.voice().n_params;
    info->weight_bytes = v->engine.weight_bytes();
  });
}

int pb200_voice_describe(const char* onnx_path, char* buf, int64_t cap) {
  return guarded([&] {
    if (!onnx_path || !buf || cap <= 0) throw std::runtime_error("pb200_voice_describe: bad argument");
    pb200::PackedVoice pv;
    pb200::load_voice_file(onnx_path, pv);
    const std::string s = pb200::describe_voice(pv);
    const size_t n = std::min<size_t>(s.size(), size_t(cap - 1));
    std::memcpy(buf, s.data(), n);
    buf[n] = 0;
  });
}

int pb200_voice_pack(const char* onnx_path, float* blob, int64_t* n_floats) {
  return guarded([&] {
    if (!onnx_path || !n_floats) throw std::runtime_error("pb200_voice_pack: null argument");
    pb200::PackedVoice pv;
    pb200::load_voice_file(onnx_path, pv);
    const int64_t need = int64_t(pv.blob.size());
    if (blob) {
      if (*n_floats < need) throw std::runtime_error("pb200_voice_pack: buffer too small");
      std::memcpy(blob, pv.blob.data(), size_t(need) * 4);
    }
    *n_floats = need;
  });
}

int pb200_debug_mrf_pack(const char* onnx_path, int32_t stage, int32_t fuse_post, int32_t plan[32], uint8_t* w,
                         int64_t* w_bytes, float* bias, int64_t* n_bias) {
  return guarded([&] {
    if (!onnx_path || !plan || !w_bytes || !n_bias) throw std::runtime_error("pb200_debug_mrf_pack: null argument");
    pb200::PackedVoice pv;
    pb200::load_voice_file(onnx_path, pv);
    if (stage < 0 || stage >= int32_t(pv.ups.size())) throw std::runtime_error("pb200_debug_mrf_pack: stage out of range");
    pb200::MrfFusedPlan p;
    const int ch = pv.ups[stage].rows / pv.ups[stage].up;
    pb200::plan_mrf_fused(pv.resblocks[stage], pv.spec.resblock, ch, fuse_post ? pv.post_k : 0, p);
    std::memset(plan, 0, 32 * sizeof(int32_t));
    plan[0] = p.ok; plan[1] = p.n_chains; plan[2] = p.n_steps; plan[3] = p.pair; plan[4] = p.hv; plan[5] = p.to;
    for (int c = 0; c < pb200::MRF_MAX_CHAINS; ++c) {
      plan[6 + c] = p.k[c];
      for (int st = 0; st < pb200::MRF_MAX_STEPS; ++st) plan[9 + c * pb200::MRF_MAX_STEPS + st] = p.dil[c][st];
    }
    plan[27] = p.post_k;
    if (p.ok && w && bias) {
      if (*w_bytes < int64_t(p.w_bytes) || *n_bias < p.n_bias) throw std::runtime_error("pb200_debug_mrf_pack: buffer too small");
      pb200::pack_mrf_fused(pv.blob.data(), pv.resblocks[stage], p, w, bias);
    }
    *w_bytes = int64_t(p.w_bytes);
    *n_bias = p.n_bias;
  });
}

int pb200_synthesize(pb200_voice* v, const int64_t* ids, int64_t n_ids, const float scales[3], const int64_t* sid,
                     const pb200_noise* noise, const float** audio, int64_t* n_samples, double* infer_seconds) {
  return guarded([&] {
    if (!v || !ids || !scales || !audio || !n_samples) throw std::runtime_error("pb200_synthesize: null argument");
    // NULL = speaker 0 (include/piper_b200.h): never inherit the speaker of an earlier call
    v->engine.set_speakers(sid, sid ? 1 : 0);
    int64_t lens[1] = {n_ids};
    *audio = v->engine.synthesize(ids, lens, 1, scales, to_spec(noise), nullptr, n_samples, infer_seconds);
  });
}

int pb200_synthesize_batch(pb200_voice* v, const int64_t* ids_concat, const int64_t* lens, int32_t B,
                           const float scales[3], const pb200_noise* noise, const int32_t* w_ceil_override,
                           const float** audio, int64_t* n_samples, double* infer_seconds) {
  return guarded([&] {
    if (!v || !ids_concat || !lens || !scales || !audio || !n_samples)
      throw std::runtime_error("pb200_synthesize_batch: null argument");
    *audio = v->engine.synthesize(ids_concat, lens, B, scales, to_spec(noise), w_ceil_override, n_samples, infer_seconds);
  });
}

int pb200_synthesize_int16(pb200_voice* v, const int64_t* ids_concat, const int64_t* lens, int32_t B,
                           const float scales[3], const pb200_noise* noise, const int16_t** audio,
                           int64_t* n_samples, double* infer_seconds) {
  return guarded([&] {
    if (!v || !ids_concat || !lens || !scales || !audio || !n_samples)
      throw std::runtime_error("pb200_synthesize_int16: null argument");
    *audio = v->engine.synthesize_int16(ids_concat, lens, B, scales, to_spec(noise), n_samples, infer_seconds);
  });
}

int pb200_vocode(pb200_voice* v, const float* z, int32_t B, int64_t frames, const float** audio,
                 double* infer_seconds) {
  return guarded([&] {
    if (!v || !z || !audio) throw std::runtime_error("pb200_vocode: null argument");
    *audio = v->engine.vocode(z, B, frames, false, infer_seconds);
  });
}

int pb200_decode(pb200_voice* v, const float* z_p, int32_t B, int64_t frames, const float** audio,
                 double* infer_seconds) {
  return guarded([&] {
    if (!v || !z_p || !audio) throw std::runtime_error("pb200_decode: null argument");
    *audio = v->engine.vocode(z_p, B, frames, true, infer_seconds);
  });
}

int pb200_encode(pb200_voice* v, const int64_t* ids, int64_t n_ids, const float scales[3], const pb200_noise* noise,
                 const float** z_p, int64_t* frames, double* infer_seconds) {
  return guarded([&] {
    if (!v || !ids || !scales || !z_p || !frames) throw std::runtime_error("pb200_encode: null argument");
    *z_p = v->engine.encode(ids, n_ids, scales, to_spec(noise), frames, infer_seconds);
  });
}

int pb200_stage(pb200_voice* v, const int64_t* ids_concat, const int64_t* lens, int32_t B, const float scales[3],
                const pb200_noise* noise, const int32_t* w_ceil_override) {
  return guarded([&] {
    if (!v || !ids_concat || !lens || !scales) throw std::runtime_error("pb200_stage: null argument");
    v->engine.stage(ids_concat, lens, B, scales, to_spec(noise), w_ceil_override);
  });
}

int pb200_run_staged(pb200_voice* v, int64_t* total_samples, float* device_ms) {
  return guarded([&] {
    if (!v) throw std::runtime_error("pb200_run_staged: null argument");
    const int64_t n = v->engine.run_staged(device_ms);
    if (total_samples) *total_samples = n;
  });
}

int pb200_stage_times(const pb200_voice* v, float ms[5]) {
  return guarded([&] {
    if (!v || !ms) throw std::runtime_error("pb200_stage_times: null argument");
    v->engine.stage_times(ms);
  });
}

int pb200_set_profile(pb200_voice* v, int32_t on) {
  return guarded([&] {
    if (!v) throw std::runtime_error("pb200_set_profile: null argument");
    v->engine.set_profile(on != 0);
  });
}

int pb200_profile_read(pb200_voice* v, char* buf, int64_t cap) {
  return guarded([&] {
    if (!v || !buf || cap <= 0) throw std::runtime_error("pb200_profile_read: bad argument");
    const std::string s = v->engine.profile_json();
    const size_t n = std::min<size_t>(s.size(), size_t(cap - 1));
    std::memcpy(buf, s.data(), n);
    buf[n] = 0;
  });
}

int pb200_profile_read_launches(pb200_voice* v, char* buf, int64_t cap) {
  return guarded([&] {
    if (!v || !buf || cap <= 0) throw std::runtime_error("pb200_profile_read_launches: bad argument");
    const std::string s = v->engine.profile_launches_json();
    if (int64_t(s.size()) >= cap) throw std::runtime_error("pb200_profile_read_launches: buffer too small");
    std::memcpy(buf, s.data(), s.size());
    buf[s.size()] = 0;
  });
}

int pb200_set_mma(pb200_voice* v, int32_t on) {
  return guarded([&] {
    if (!v) throw std::runtime_error("pb200_set_mma: null argument");
    v->engine.set_mma(on);
  });
}

#define CK(expr)                                                                                         \
  do {                                                                                                   \
    cudaError_t _e = (expr);                                                                             \
    if (_e != cudaSuccess) throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(_e)); \
  } while (0)

}  // extern "C"

namespace {

// device allocations of one test-hook call, freed on every exit path
struct DevArena {
  std::vector<void*> ptrs;
  ~DevArena() {
    for (void* p : ptrs) cudaFree(p);
  }
  template <class T>
  T* upload(const T* host, size_t n) {
    if (!host || n == 0) return nullptr;
    void* d = nullptr;
    CK(cudaMalloc(&d, n * sizeof(T)));
    ptrs.push_back(d);
    CK(cudaMemcpy(d, host, n * sizeof(T), cudaMemcpyHostToDevice));
    return static_cast<T*>(d);
  }
};

[[noreturn]] void conv_reject(const std::string& why) { throw std::runtime_error("pb200_debug_conv: " + why); }

// One conv launch on host arrays, packed and launched the way Engine::conv does it (include/piper_b200.h)
void debug_conv(int backend, const int32_t* d, float slope, const float* x, const float* w, const float* bias,
                const float* bias_item, int bias_item_stride, const int32_t* len, int B, float* y, float* y2, const float* r) {
  using namespace pb200;
  if (backend < 0 || backend > 6) conv_reject("backend " + std::to_string(backend) + " is not 0..6");
  if (!d || !x || !w || !len || B <= 0) conv_reject("null argument");
  const int ci = d[0], rows = d[1], k = d[2], dil = d[3], pad = d[4], q_extra = d[5], pre = d[6], epi = d[7];
  const int split = d[8], first = d[9], up = d[10], up_pad = d[11], mrf = d[12], mrf_n = d[13], len_scale = d[14];
  const int flags = d[22];
  const bool alias = flags & PB200_CONV_Y_IS_R, flat = flags & PB200_CONV_FLAT, latency = flags & PB200_CONV_LATENCY;
  const int cs_x = d[15], cs_y = d[16], cs_y2 = d[17], C_y = d[19], C_y2 = d[20];
  const int cs_r = alias ? cs_y : d[18], C_r = alias ? C_y : d[21];          // y == r: r is y
  if (ci <= 0 || rows <= 0 || k <= 0 || dil <= 0 || pad < 0 || q_extra < 0 || len_scale <= 0 || up <= 0)
    conv_reject("bad shape");
  if (epi < EPI_BIAS || epi > EPI_MRF) conv_reject("unknown epilogue " + std::to_string(epi));
  if (pre != PRE_NONE && pre != PRE_LRELU) conv_reject("unknown pre-activation " + std::to_string(pre));
  // what the engine never launches
  if (epi == EPI_GATE && rows % 2) conv_reject("GATE needs an even number of rows");
  if (epi == EPI_UPSAMPLE ? rows % up != 0 : up != 1) conv_reject("rows % up != 0, or up != 1 without UPSAMPLE");
  if (q_extra && epi != EPI_UPSAMPLE) conv_reject("q_extra without UPSAMPLE");
  if (epi == EPI_WN && (split < 0 || split > rows || split % 16)) conv_reject("WN split must be a multiple of 16 in [0, rows]");
  if (epi == EPI_MRF && (mrf < 0 || mrf > 2 || mrf_n <= 0)) conv_reject("bad MRF mode");
  if (alias && epi != EPI_WN && epi != EPI_SUBFROM) conv_reject("y == r only for WN and SUBFROM");
  if (bias_item && bias_item_stride < rows) conv_reject("bias_item stride shorter than rows");
  // which buffers the epilogue reads and writes, and how many channels of each
  const bool uses_r = epi == EPI_RES || epi == EPI_WN || epi == EPI_SUBFROM || epi == EPI_MRF;
  const bool uses_y2 = epi == EPI_MRF || (epi == EPI_WN && split < rows);
  const bool uses_y = epi != EPI_MRF && !(epi == EPI_WN && split == 0);
  const int need_y = epi == EPI_GATE ? rows / 2 : epi == EPI_UPSAMPLE ? rows / up : epi == EPI_WN ? split : rows;
  const int need_r = epi == EPI_WN ? split : rows, need_y2 = epi == EPI_WN ? rows - split : rows;
  if (uses_y && (!y || C_y < need_y)) conv_reject("y needs " + std::to_string(need_y) + " channels");
  if (uses_y2 && (!y2 || C_y2 < need_y2)) conv_reject("y2 needs " + std::to_string(need_y2) + " channels");
  if (uses_r && ((!alias && !r) || (alias && !y) || C_r < need_r)) conv_reject("r needs " + std::to_string(need_r) + " channels");
  int max_in = 0;
  for (int b = 0; b < B; ++b) {
    if (len[b] < 0) conv_reject("negative length");
    max_in = std::max(max_in, len[b] * len_scale);
  }
  const int max_len = max_in + q_extra;
  // pitches: 16-byte rows (the CUDA-core kernel stages x with 16-byte copies); every valid column inside its row
  for (int cs : {cs_x, cs_y, cs_y2, cs_r})
    if (cs < 0 || cs % 4) conv_reject("pitches must be non-negative multiples of 4 floats");
  if (cs_x < max_in) conv_reject("x pitch shorter than the longest item");
  if (uses_y && cs_y < (epi == EPI_UPSAMPLE ? max_in * up : max_len)) conv_reject("y pitch too short");
  if (uses_y2 && cs_y2 < max_len) conv_reject("y2 pitch too short");
  if (uses_r && cs_r < max_len) conv_reject("r pitch too short");
  // the tensor-core plan, as Engine::conv2_layer makes it: 1, 3 = bf16x3; 2, 4 = tf32x3 (2 chains); 5 = fp16x3 (1 chain);
  // 6 = fp16x3 (2 chains); the latency plan (conv2_layer variant 1) takes two chains whatever the back end
  Conv2Layer l;
  if (backend) {
    const int prec = (backend == 1 || backend == 3) ? 0 : (backend == 2 || backend == 4) ? 1 : 2;
    const int chains = latency || backend == 2 || backend == 4 || backend == 6 ? 2 : 1;
    if (!conv2_plan(ci, rows, k, dil, prec, chains, l)) conv_reject("shape not supported by the tensor-core conv");
  }

  // weights in the engine's [ci][k][rows_p] layout (voice.cc), then the tensor-core packing of the plan
  const int rows_p = (rows + 3) & ~3;
  std::vector<float> pk(size_t(ci) * k * rows_p, 0.f);
  for (int i = 0; i < ci; ++i)
    for (int j = 0; j < k; ++j)
      for (int o = 0; o < rows; ++o) pk[(size_t(i) * k + j) * rows_p + o] = w[(size_t(o) * ci + i) * k + j];
  std::vector<uint8_t> packed;
  if (backend) {
    packed.resize(l.w_bytes);
    conv2_pack(pk.data(), ci, k, rows_p, l, packed.data());
  }

  // buffers: item-major [B][C][cs] or flat [C][B][cs] (the engine's flat layout: item b at b * cs of every channel row)
  DevArena m;
  const size_t nx = size_t(B) * ci * cs_x, ny = size_t(B) * C_y * cs_y, ny2 = size_t(B) * C_y2 * cs_y2, nr = size_t(B) * C_r * cs_r;
  float* dx = m.upload(x, nx);
  float* dy = uses_y || alias ? m.upload(y, ny) : nullptr;
  float* dy2 = uses_y2 ? m.upload(y2, ny2) : nullptr;
  float* dr = alias ? dy : uses_r ? m.upload(r, nr) : nullptr;
  const float* dbias = m.upload(bias, size_t(rows));
  const float* dbi = bias_item ? m.upload(bias_item, size_t(B - 1) * bias_item_stride + rows) : nullptr;
  const int* dlen = m.upload(len, size_t(B));
  auto view = [&](float* p, int C, int cs) {
    return flat ? View{p, (long long)cs, B * cs} : View{p, (long long)C * cs, cs};
  };
  const View vx = view(dx, ci, cs_x), vy = view(dy, C_y, cs_y), vy2 = view(dy2, C_y2, cs_y2),
             vr = alias ? vy : view(dr, C_r, cs_r);

  if (backend == 0) {
    ConvArgs a;
    a.x = vx; a.y = vy; a.y2 = vy2; a.r = vr;
    a.w = m.upload(pk.data(), pk.size());
    a.bias = dbias; a.bias_item = dbi; a.bias_item_stride = bias_item_stride;
    a.len = dlen; a.len_scale = len_scale;
    a.ci = ci; a.rows = rows; a.rows_p = rows_p; a.k = k; a.dil = dil; a.pad = pad; a.q_extra = q_extra;
    a.pre = pre; a.slope = slope; a.epi = epi; a.split = split; a.first = first;
    a.up = up; a.up_pad = up_pad; a.mrf = mrf; a.mrf_n = mrf_n;
    launch_conv1d(a, B, max_len, nullptr);
  } else {
    MmaConvArgs a;
    a.x = vx; a.y = vy; a.y2 = vy2; a.r = vr;
    a.w = m.upload(packed.data(), packed.size());
    a.bias = dbias; a.bias_item = dbi; a.bias_item_stride = bias_item_stride;
    a.len = dlen; a.len_scale = len_scale;
    a.ci = ci; a.rows = rows; a.k = k; a.dil = dil; a.pad = pad; a.q_extra = q_extra;
    a.pre = pre; a.slope = slope; a.epi = epi; a.split = split; a.first = first;
    a.up = up; a.up_pad = up_pad; a.mrf = mrf; a.mrf_n = mrf_n;
    // one launch item on the concatenated time axis under the conditions of Engine::conv (engine.cu), per-item tiles otherwise
    auto same_layout = [&](const View& v) { return v.p == nullptr || (v.bs == vx.bs && v.cs == vx.cs); };
    const bool flat_launch = flat && len_scale == 1 && q_extra == 0 && vx.bs < (long long)vx.cs && vx.bs >= 2 &&
                             ((long long)vx.cs + 1024) * vx.bs < (1LL << 32) && same_layout(a.y) && same_layout(a.y2) &&
                             same_layout(a.r);
    if (flat_launch) {
      a.flat_tg = int(vx.bs);
      a.flat_n = B;
      launch_conv2(a, l, 1, B * int(vx.bs), nullptr);
    } else {
      launch_conv2(a, l, B, max_len, nullptr);
    }
  }
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  if (uses_y || alias) CK(cudaMemcpy(y, dy, ny * 4, cudaMemcpyDeviceToHost));
  if (uses_y2) CK(cudaMemcpy(y2, dy2, ny2 * 4, cudaMemcpyDeviceToHost));
}

}  // namespace

extern "C" {

int pb200_debug_conv(int32_t backend, const int32_t desc[PB200_CONV_DESC_LEN], float slope, const float* x, const float* w,
                     const float* bias, const float* bias_item, int32_t bias_item_stride, const int32_t* len, int32_t B,
                     float* y, float* y2, const float* r) {
  return guarded([&] { debug_conv(backend, desc, slope, x, w, bias, bias_item, bias_item_stride, len, B, y, y2, r); });
}

int pb200_debug_conv1d(int32_t backend, const float* x, int32_t B, int32_t ci, int32_t L, const float* w,
                       const float* bias, int32_t co, int32_t k, int32_t dil, float pre_slope, const float* resid,
                       float* y) {
  return guarded([&] {
    using namespace pb200;
    if (!x || !w || !y || B <= 0 || L <= 0) throw std::runtime_error("pb200_debug_conv1d: bad argument");
    // every item L long, rows padded to a 16-byte pitch, y zeroed; only the valid columns come back
    const int Lp = (L + 3) & ~3;
    std::vector<float> xp(size_t(B) * ci * Lp, 0.f), yp(size_t(B) * co * Lp, 0.f), rp;
    for (size_t row = 0; row < size_t(B) * ci; ++row) std::memcpy(&xp[row * Lp], x + row * L, size_t(L) * 4);
    if (resid) {
      rp.assign(size_t(B) * co * Lp, 0.f);
      for (size_t row = 0; row < size_t(B) * co; ++row) std::memcpy(&rp[row * Lp], resid + row * L, size_t(L) * 4);
    }
    const std::vector<int32_t> lens(B, L);
    int32_t d[PB200_CONV_DESC_LEN] = {};
    d[0] = ci; d[1] = co; d[2] = k; d[3] = dil; d[4] = dil * (k - 1) / 2;
    d[6] = pre_slope != 0.f ? PRE_LRELU : PRE_NONE;
    d[7] = resid ? EPI_RES : EPI_BIAS;
    d[10] = 1; d[13] = 1; d[14] = 1;
    d[15] = Lp; d[16] = Lp; d[18] = resid ? Lp : 0; d[19] = co; d[21] = resid ? co : 0;
    debug_conv(backend, d, pre_slope, xp.data(), w, bias, nullptr, 0, lens.data(), B, yp.data(), nullptr,
               resid ? rp.data() : nullptr);
    for (size_t row = 0; row < size_t(B) * co; ++row) std::memcpy(y + row * L, &yp[row * Lp], size_t(L) * 4);
  });
}

void pb200_release(pb200_voice*, const void*) {
  // Output buffers are engine-owned pinned staging areas reused by the next call; nothing to free.
}

int pb200_set_speakers(pb200_voice* v, const int64_t* sids, int32_t n) {
  return guarded([&] {
    if (!v || (n > 0 && !sids)) throw std::runtime_error("pb200_set_speakers: null argument");
    v->engine.set_speakers(sids, n);
  });
}

int pb200_set_debug(pb200_voice* v, int32_t on) {
  return guarded([&] {
    if (!v) throw std::runtime_error("pb200_set_debug: null argument");
    v->engine.set_debug(on != 0);
  });
}

int pb200_tap_shape(const pb200_voice* v, const char* name, int32_t b, int32_t* channels, int32_t* len) {
  return guarded([&] {
    if (!v || !name) throw std::runtime_error("pb200_tap_shape: null argument");
    const pb200::HostTap* t = v->engine.tap(name);
    if (!t) throw std::runtime_error(std::string("no tap named '") + name + "' (debug off, or stage not run)");
    if (b < 0 || b >= t->B) throw std::runtime_error("tap: item index out of range");
    if (channels) *channels = t->C;
    if (len) *len = t->len[b];
  });
}

int pb200_tap_read(const pb200_voice* v, const char* name, int32_t b, float* buf, int64_t cap_floats) {
  return guarded([&] {
    if (!v || !name || !buf) throw std::runtime_error("pb200_tap_read: null argument");
    const pb200::HostTap* t = v->engine.tap(name);
    if (!t) throw std::runtime_error(std::string("no tap named '") + name + "'");
    if (b < 0 || b >= t->B) throw std::runtime_error("tap: item index out of range");
    const int L = t->len[b];
    if (int64_t(t->C) * L > cap_floats) throw std::runtime_error("tap: buffer too small");
    for (int c = 0; c < t->C; ++c)
      std::memcpy(buf + size_t(c) * L, t->data.data() + (size_t(b) * t->C + c) * t->pitch, size_t(L) * 4);
  });
}

uint64_t pb200_launch_count(void) { return pb200::launch_count(); }
const char* pb200_last_error(void) { return g_error.c_str(); }
const char* pb200_version(void) { return "piper_b200 0.1.0 (sm_100a)"; }

}  // extern "C"
