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

int pb200_debug_conv1d(int32_t backend, const float* x, int32_t B, int32_t ci, int32_t L, const float* w,
                       const float* bias, int32_t co, int32_t k, int32_t dil, float pre_slope, const float* resid,
                       float* y) {
  return guarded([&] {
    using namespace pb200;
    if (!x || !w || !y || B <= 0 || L <= 0) throw std::runtime_error("pb200_debug_conv1d: bad argument");
    if (backend < 0 || backend > 6)
      throw std::runtime_error("pb200_debug_conv1d: backend " + std::to_string(backend) + " is not 0..6");
    const int Lp = (L + 3) & ~3, pad = dil * (k - 1) / 2, rows_p = (co + 3) & ~3;
    float *dx = nullptr, *dy = nullptr, *dr = nullptr, *dw = nullptr, *db = nullptr;
    int* dlen = nullptr;
    uint8_t* dw16 = nullptr;
    CK(cudaMalloc(&dx, size_t(B) * ci * Lp * 4));
    CK(cudaMalloc(&dy, size_t(B) * co * Lp * 4));
    CK(cudaMemset(dy, 0, size_t(B) * co * Lp * 4));
    CK(cudaMemcpy2D(dx, size_t(Lp) * 4, x, size_t(L) * 4, size_t(L) * 4, size_t(B) * ci, cudaMemcpyHostToDevice));
    if (resid) {
      CK(cudaMalloc(&dr, size_t(B) * co * Lp * 4));
      CK(cudaMemcpy2D(dr, size_t(Lp) * 4, resid, size_t(L) * 4, size_t(L) * 4, size_t(B) * co, cudaMemcpyHostToDevice));
    }
    if (bias) {
      CK(cudaMalloc(&db, size_t(co) * 4));
      CK(cudaMemcpy(db, bias, size_t(co) * 4, cudaMemcpyHostToDevice));
    }
    std::vector<int> lens(B, L);
    CK(cudaMalloc(&dlen, size_t(B) * 4));
    CK(cudaMemcpy(dlen, lens.data(), size_t(B) * 4, cudaMemcpyHostToDevice));
    View vx{dx, (long long)ci * Lp, Lp}, vy{dy, (long long)co * Lp, Lp}, vr{dr, (long long)co * Lp, Lp};
    if (backend == 0) {
      std::vector<float> pk(size_t(ci) * k * rows_p, 0.f);
      for (int i = 0; i < ci; ++i)
        for (int j = 0; j < k; ++j)
          for (int o = 0; o < co; ++o) pk[(size_t(i) * k + j) * rows_p + o] = w[(size_t(o) * ci + i) * k + j];
      CK(cudaMalloc(&dw, pk.size() * 4));
      CK(cudaMemcpy(dw, pk.data(), pk.size() * 4, cudaMemcpyHostToDevice));
      ConvArgs a;
      a.x = vx; a.y = vy; a.r = vr; a.w = dw; a.bias = db; a.len = dlen; a.len_scale = 1;
      a.ci = ci; a.rows = co; a.rows_p = rows_p; a.k = k; a.dil = dil; a.pad = pad;
      a.pre = pre_slope != 0.f ? PRE_LRELU : PRE_NONE; a.slope = pre_slope;
      a.epi = resid ? EPI_RES : EPI_BIAS;
      launch_conv1d(a, B, L, nullptr);
    } else {
      // tensor-core kernel (conv_mma2.cu): 1, 3 = bf16x3; 2, 4 = tf32x3 (2 chains); 5 = fp16x3 (1 chain); 6 = fp16x3 (2 chains)
      const int prec = (backend == 1 || backend == 3) ? 0 : (backend == 2 || backend == 4) ? 1 : 2;
      const int chains = (backend == 2 || backend == 4 || backend == 6) ? 2 : 1;
      Conv2Layer l;
      if (!conv2_plan(ci, co, k, dil, prec, chains, l))
        throw std::runtime_error("shape not supported by the tensor-core conv");
      std::vector<float> pk(size_t(ci) * k * rows_p, 0.f);
      for (int i = 0; i < ci; ++i)
        for (int j = 0; j < k; ++j)
          for (int o = 0; o < co; ++o) pk[(size_t(i) * k + j) * rows_p + o] = w[(size_t(o) * ci + i) * k + j];
      std::vector<uint8_t> packed(l.w_bytes);
      conv2_pack(pk.data(), ci, k, rows_p, l, packed.data());
      CK(cudaMalloc(&dw16, packed.size()));
      CK(cudaMemcpy(dw16, packed.data(), packed.size(), cudaMemcpyHostToDevice));
      MmaConvArgs a;
      a.x = vx; a.y = vy; a.r = vr; a.w = dw16; a.bias = db; a.len = dlen; a.len_scale = 1;
      a.ci = ci; a.rows = co; a.k = k; a.dil = dil; a.pad = pad;
      a.pre = pre_slope != 0.f ? PRE_LRELU : PRE_NONE; a.slope = pre_slope;
      a.epi = resid ? EPI_RES : EPI_BIAS;
      launch_conv2(a, l, B, L, nullptr);
    }
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy2D(y, size_t(L) * 4, dy, size_t(Lp) * 4, size_t(L) * 4, size_t(B) * co, cudaMemcpyDeviceToHost));
    cudaFree(dx); cudaFree(dy); cudaFree(dr); cudaFree(dw); cudaFree(db); cudaFree(dlen); cudaFree(dw16);
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
