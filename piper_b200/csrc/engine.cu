#include "engine.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>

namespace pb200 {

#define CUDA_CHECK(expr)                                                                              \
  do {                                                                                                \
    cudaError_t _e = (expr);                                                                          \
    if (_e != cudaSuccess)                                                                            \
      throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(_e) + " at " #expr); \
  } while (0)

// Bumped whenever any workspace buffer is re-allocated: captured CUDA graphs hold raw pointers and are re-captured
// when the generation they were built against is stale.
static std::atomic<unsigned long long> g_ws_generation{1};
void count_launches(unsigned long long n);

void DeviceBuf::ensure(size_t bytes) {
  if (bytes <= cap) return;
  g_ws_generation.fetch_add(1);
  release();
  size_t want = bytes + bytes / 4 + 256;   // headroom: data-dependent lengths vary call to call
  CUDA_CHECK(cudaMalloc(&p, want));
  cap = want;
}
void DeviceBuf::release() {
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
}
void PinnedBuf::ensure(size_t bytes) {
  if (bytes <= cap) return;
  release();
  size_t want = bytes + bytes / 4 + 256;
  CUDA_CHECK(cudaMallocHost(&p, want));
  cap = want;
}
void PinnedBuf::release() {
  if (p) cudaFreeHost(p);
  p = nullptr;
  cap = 0;
}

static int round4(int v) { return (v + 3) & ~3; }

// Flat layout (PIPER_B200_FLAT, default on): phoneme- and frame-rate activations are stored [channel][item][slot] instead of
// [item][channel][pitch] - the same View struct with bs = slot and cs = items * slot - so that the conv kernel can cut its
// tiles on the concatenated time axis (T = 259 costs 3 x 128-row tiles per utterance, but 32 utterances x 264 = 66 tiles
// instead of 96).  The slot is the pitch plus a gap >= the largest one-sided conv halo, so a window never reaches live
// data of a neighbouring utterance.
bool Engine::flat_on() {
  if (flat_ < 0) {
    const char* e = std::getenv("PIPER_B200_FLAT");
    flat_ = e ? (std::atoi(e) != 0) : 1;
  }
  return flat_ != 0;
}
int Engine::slot(int max_len) { return round4(max_len) + (flat_on() ? 4 : 0); }
View Engine::fview(float* p, int C, int pitch) const {
  if (flat_ > 0) return View{p, (long long)pitch, B_ * pitch};
  return View{p, (long long)C * pitch, pitch};
}

Engine::Engine(const std::string& onnx_path, int device, bool upload) : device_(device) {
  load_voice_file(onnx_path, voice_);
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev <= 0)
    throw std::runtime_error(std::string("piper_b200 needs a CUDA device (no CPU fallback): ") +
                             (e != cudaSuccess ? cudaGetErrorString(e) : "no devices"));
  if (device < 0 || device >= n_dev) throw std::runtime_error("device index out of range");
  CUDA_CHECK(cudaSetDevice(device));
  cudaDeviceProp prop{};
  CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    throw std::runtime_error(std::string("piper_b200 kernels are built for sm_100a only; device is sm_") +
                             std::to_string(prop.major) + std::to_string(prop.minor));
  CUDA_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  for (auto& ev : ev_) CUDA_CHECK(cudaEventCreate(&ev));
  weights_.ensure(voice_.blob.size() * sizeof(float));
  if (upload)
    CUDA_CHECK(cudaMemcpyAsync(weights_.p, voice_.blob.data(), voice_.blob.size() * sizeof(float), cudaMemcpyHostToDevice, stream_));
  CUDA_CHECK(cudaStreamSynchronize(stream_));    // uploads from pageable memory: complete before the first kernel reads them
  if (const char* e = std::getenv("PIPER_B200_MMA")) mma_mask_ = std::atoi(e);
}

Engine::~Engine() {
  cudaSetDevice(device_);
  if (stream_) cudaStreamSynchronize(stream_);
  drop_graphs();
  DeviceBuf* dbs[] = {&weights_, &ids_d_, &len_d_, &ylen_d_, &cum_d_, &logw_d_, &override_d_, &epsdp_d_, &epsoff_d_,
                      &off_d_, &sid_d_, &cond_d_, &x_, &t1_, &qkv_, &att_, &ffn_, &stats_, &g_, &h_, &u_, &v_, &pr_, &z2_, &z_, &fh_,
                      &facts_, &fout_, &epsz_d_, &ga_, &gp_, &gq_, &gs_, &audio_d_, &audio16_d_, &peak_d_, &mrf_w_, &params_d_, &prof_d_};
  for (auto* d : dbs) d->release();
  for (auto& kv : conv2_layers_)
    if (kv.second.w_dev) cudaFree(kv.second.w_dev);
  PinnedBuf* pbs[] = {&ids_pin_, &misc_pin_, &audio_pin_, &audio16_pin_, &eps_pin_, &params_pin_, &override_pin_};
  for (auto* p : pbs) p->release();
  for (auto& ev : ev_)
    if (ev) cudaEventDestroy(ev);
  for (auto& ev : ev_pool_)
    if (ev) cudaEventDestroy(ev);
  if (stream_) cudaStreamDestroy(stream_);
}

ConvArgs Engine::conv_args(const ConvW& c, View x, const int* len, int len_scale) const {
  ConvArgs a;
  a.x = x;
  a.w = W(c.w);
  a.bias = W(c.b);
  a.len = len;
  a.len_scale = len_scale;
  a.ci = c.ci; a.rows = c.rows; a.rows_p = c.rows_p; a.k = c.k; a.dil = c.dil; a.pad = c.pad;
  a.up = c.up; a.up_pad = c.up_pad;
  a.host_w = &c;
  return a;
}

void Engine::conv(const char* tag, ConvArgs& a, int max_len, double len_sum) {
  // the tensor cores when the layer's family is enabled in the mask and the conv2 plan takes its shape, CUDA cores otherwise
  const ConvW* w = a.host_w;
  const int family = tag[0] == 'd' && tag[1] == 'e' ? 1 : tag[0] == 'f' ? 2 : tag[0] == 'e' ? 4 : tag[0] == 'd' && tag[1] == 'p' ? 8 : 0;
  const bool fp32_grade = family != 1;                 // flow, encoder, duration predictor: their outputs feed exp() / ceil()
  const Conv2Layer* l = w && (mma_mask_ & family) ? conv2_layer(*w, a, fp32_grade) : nullptr;
  if (l && fp32_grade) {
    // a launch of the throughput plan that would leave most SMs idle takes the latency plan instead (batch 1)
    const long long rows = a.x.bs < (long long)a.x.cs ? (long long)B_ * a.x.bs : (long long)B_ * max_len;
    const long long ctas = (rows + l->mt - 1) / l->mt * l->n_tiles;
    if (ctas < 74)
      if (const Conv2Layer* l1 = conv2_layer(*w, a, fp32_grade, 1)) l = l1;
  }
  auto go = [&] {
    if (!l) {
      launch_conv1d(a, B_, max_len, stream_);
      return;
    }
    MmaConvArgs m;
    m.x = a.x; m.y = a.y; m.y2 = a.y2; m.r = a.r;
    m.w = static_cast<const uint8_t*>(l->w_dev);
    m.bias = a.bias; m.bias_item = a.bias_item; m.bias_item_stride = a.bias_item_stride;
    m.len = a.len; m.len_scale = a.len_scale;
    m.ci = a.ci; m.rows = a.rows; m.k = a.k; m.dil = a.dil; m.pad = a.pad; m.q_extra = a.q_extra;
    m.pre = a.pre; m.slope = a.slope; m.epi = a.epi; m.split = a.split; m.first = a.first;
    m.up = a.up; m.up_pad = a.up_pad; m.mrf = a.mrf; m.mrf_n = a.mrf_n;
    if (profile_ && prof_d_.p && recs_.size() < kProfRecs)       // per-role wait counters of this launch (conv2_body.inl)
      m.prof = prof_d_.as<unsigned long long>() + 16 * recs_.size();
    // flat layout views (bs = slot < cs): one launch item of length items x slot, tiles on the concatenated time axis
    auto same_layout = [&](const View& v) { return v.p == nullptr || (v.bs == a.x.bs && v.cs == a.x.cs); };
    const bool flat = flat_ > 0 && a.len_scale == 1 && a.q_extra == 0 && a.x.bs < (long long)a.x.cs && a.x.bs * B_ == a.x.cs &&
                      a.x.bs >= 2 && ((long long)a.x.cs + 1024) * a.x.bs < (1LL << 32) &&   // (range of the kernel's reciprocal division)
                      same_layout(a.y) && same_layout(a.y2) && same_layout(a.r);   // (conv_pre writes an item-major generator buffer)
    if (flat) {
      m.flat_tg = int(a.x.bs);
      m.flat_n = B_;
      launch_conv2(m, *l, 1, B_ * int(a.x.bs), stream_);
    } else {
      launch_conv2(m, *l, B_, max_len, stream_);
    }
  };
  if (!profile_) {
    go();
    return;
  }
  if (ev_used_ + 2 > ev_pool_.size()) {
    const size_t old = ev_pool_.size();
    ev_pool_.resize(old + 256);
    for (size_t i = old; i < ev_pool_.size(); ++i) CUDA_CHECK(cudaEventCreate(&ev_pool_[i]));
  }
  ProfRec r;
  r.tag = tag;
  r.mma = l != nullptr;
  r.e0 = ev_pool_[ev_used_++];
  r.e1 = ev_pool_[ev_used_++];
  // algorithmic work of this launch (SURVEY.md §8d): fp32 in + out + weights once; elementwise ops free
  const double co = double(a.rows) / a.up, lin = len_sum, lout = len_sum * a.up;
  r.bytes = 4.0 * (lin * a.ci + lout * (a.epi == EPI_GATE ? co / 2 : co) + double(a.ci) * a.rows * a.k + a.rows);
  r.flops = 2.0 * lout * a.ci * co * a.k;
  r.ci = a.ci; r.rows = a.rows; r.k = a.k; r.dil = a.dil; r.up = a.up; r.max_len = max_len; r.len_sum = len_sum;
  CUDA_CHECK(cudaEventRecord(r.e0, stream_));
  go();
  CUDA_CHECK(cudaEventRecord(r.e1, stream_));
  recs_.push_back(r);
}

// variant 0: the throughput plan (one K-chain for short reductions -> 128-row output tiles); variant 1: the latency plan for
// launches that cannot fill the machine (two chains everywhere -> 64-row output tiles, i.e. more, lighter CTAs).
const Conv2Layer* Engine::conv2_layer(const ConvW& w, const ConvArgs& a, bool fp32_grade, int variant) {
  auto it = conv2_layers_.find({&w, variant});
  if (it == conv2_layers_.end()) {
    Conv2Layer l;
    // precision: fp16x3 for every family (tf32x3-class accuracy at bf16x3 instruction cost, conv2_body.inl) or, with
    // PIPER_B200_V2_PREC=std, bf16x3 for the generator and tf32x3 for the fp32-grade families; 2 K-chains for the latter
    static int g_f16 = -1;
    if (g_f16 < 0) {
      const char* e = std::getenv("PIPER_B200_V2_PREC");
      g_f16 = (e ? std::string(e) == "f16" : true) ? 1 : 0;      // default fp16x3 (PIPER_B200_V2_PREC=std: bf16x3 generator, tf32x3 elsewhere)
    }
    const int prec = g_f16 ? 2 : (fp32_grade ? 1 : 0);
    static int g_chains = -1;                            // PIPER_B200_V2_CHAINS: K-chains of the fp32-grade families (default 2)
    if (g_chains < 0) {
      const char* e = std::getenv("PIPER_B200_V2_CHAINS");
      g_chains = e ? std::max(1, std::min(2, std::atoi(e))) : 2;
    }
    // The tensor core adds into its fp32 accumulator with truncation, an error that grows with the number of accumulation
    // steps (DESIGN.md section 3): the fp32-grade families cut LONG reductions into two K-chains.  A short one (1x1 convs:
    // C_in / 16 = 12 steps) gains nothing from that, and a single chain frees TMEM for 128-row output tiles.
    static int g_chain_k = -1;                           // PIPER_B200_V2_CHAIN_K: reductions shorter than this use one chain
    if (g_chain_k < 0) {
      const char* e = std::getenv("PIPER_B200_V2_CHAIN_K");
      g_chain_k = e ? std::atoi(e) : 400;               // measured: +1.6 % on config 3; real-voice error 2.8e-4 -> <= 3.6e-4
    }
    const int chains = (fp32_grade && (variant == 1 || a.ci * a.k >= g_chain_k)) ? g_chains : 1;
    if (conv2_plan(a.ci, a.rows, a.k, a.dil, prec, chains, l)) {
      std::vector<uint8_t> host(l.w_bytes);
      conv2_pack(voice_.blob.data() + w.w, a.ci, a.k, a.rows_p, l, host.data());
      CUDA_CHECK(cudaMalloc(&l.w_dev, l.w_bytes));
      // On the engine's own stream and waited for: a synchronous cudaMemcpy from pageable memory may return before the DMA
      // has landed and orders only against the legacy stream, which this (non-blocking) stream does not synchronise with -
      // the first launch then raced the upload of its own weights (found on hardware: wrong first call, right ever after).
      CUDA_CHECK(cudaMemcpyAsync(l.w_dev, host.data(), l.w_bytes, cudaMemcpyHostToDevice, stream_));
      CUDA_CHECK(cudaStreamSynchronize(stream_));
    }
    it = conv2_layers_.emplace(std::make_pair(&w, variant), l).first;
  }
  return it->second.w_dev ? &it->second : nullptr;
}

void Engine::profile_begin() {
  recs_.clear();
  ev_used_ = 0;
  static const bool roles = std::getenv("PIPER_B200_PROF_ROLES") != nullptr;   // developer diagnostic (tools/layer_report.py --roles)
  if (roles) {
    prof_d_.ensure(kProfRecs * 16 * sizeof(unsigned long long));
    CUDA_CHECK(cudaMemsetAsync(prof_d_.p, 0, kProfRecs * 16 * sizeof(unsigned long long), stream_));
  }
}

std::string Engine::profile_json() {
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  struct Agg { long n = 0; double ms = 0, bytes = 0, flops = 0; };
  std::map<std::string, Agg> agg;
  for (const ProfRec& r : recs_) {
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, r.e0, r.e1));
    Agg& a = agg[std::string(r.tag) + (r.mma ? ".mma" : "")];
    a.n++; a.ms += ms; a.bytes += r.bytes; a.flops += r.flops;
  }
  std::string out = "{";
  bool first = true;
  for (const auto& kv : agg) {
    char buf[256];
    snprintf(buf, sizeof buf, "%s\"%s\":{\"launches\":%ld,\"ms\":%.6f,\"bytes\":%.0f,\"flops\":%.0f}", first ? "" : ",",
             kv.first.c_str(), kv.second.n, kv.second.ms, kv.second.bytes, kv.second.flops);
    out += buf;
    first = false;
  }
  return out + "}";
}

std::string Engine::profile_launches_json() {
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  std::vector<unsigned long long> roles;
  if (prof_d_.p) {
    roles.resize(kProfRecs * 16);
    CUDA_CHECK(cudaMemcpy(roles.data(), prof_d_.p, roles.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  }
  std::string out = "[";
  for (size_t i = 0; i < recs_.size(); ++i) {
    const ProfRec& r = recs_[i];
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, r.e0, r.e1));
    char buf[640];
    snprintf(buf, sizeof buf,
             "%s{\"tag\":\"%s\",\"mma\":%d,\"us\":%.3f,\"ci\":%d,\"rows\":%d,\"k\":%d,\"dil\":%d,\"up\":%d,"
             "\"max_len\":%d,\"len_sum\":%.0f,\"bytes\":%.0f,\"flops\":%.0f}",
             i ? "," : "", r.tag, r.mma ? 1 : 0, ms * 1e3, r.ci, r.rows, r.k, r.dil, r.up, r.max_len, r.len_sum, r.bytes, r.flops);
    out += buf;
    if (!roles.empty() && i < kProfRecs && roles[16 * i + 3]) {   // summed over CTAs, SM cycles: see conv2_body.inl for the slots
      out.pop_back();
      out += ",\"roles\":[";
      for (int j = 0; j < 9; ++j) out += (j ? "," : "") + std::to_string(roles[16 * i + j]);
      out += "]}";
    }
  }
  return out + "]";
}

void Engine::ensure_front(int B, int Tmax) {
  const VoiceSpec& s = voice_.spec;
  const int Tp = slot(Tmax);
  const size_t n = size_t(B) * Tp;
  ids_d_.ensure(n * 4); len_d_.ensure(size_t(B) * 4); ylen_d_.ensure(size_t(B) * 4);
  cum_d_.ensure(n * 4); logw_d_.ensure(n * 4); off_d_.ensure(size_t(B) * 8); epsoff_d_.ensure(size_t(B) * 8);
  x_.ensure(n * s.hidden * 4); t1_.ensure(n * s.hidden * 4); qkv_.ensure(n * 3 * s.hidden * 4);
  att_.ensure(n * s.hidden * 4); ffn_.ensure(n * s.filter * 4); stats_.ensure(n * 2 * s.inter * 4);
  g_.ensure(n * s.hidden * 4); h_.ensure(n * s.hidden * 4); u_.ensure(n * s.hidden * 4); v_.ensure(n * s.hidden * 4);
  pr_.ensure(n * 32 * 4 * ((3 * s.spline_bins - 1 + 31) / 32)); z2_.ensure(n * 2 * 4);
  peak_d_.ensure(size_t(B) * 4);
}

void Engine::ensure_back(int B, int Fmax) {
  const VoiceSpec& s = voice_.spec;
  const int Fp = slot(Fmax);
  const size_t n = size_t(B) * Fp;
  z_.ensure(n * s.inter * 4); fh_.ensure(n * s.hidden * 4); facts_.ensure(n * s.hidden * 4); fout_.ensure(n * s.hidden * 4);
  size_t per_frame = size_t(s.up_initial);
  int ch = s.up_initial, rate = 1;
  for (int u : s.up_rates) {
    ch /= 2;
    rate *= u;
    per_frame = std::max(per_frame, size_t(ch) * rate);
  }
  const size_t g = n * per_frame * 4;
  ga_.ensure(g); gp_.ensure(g); gq_.ensure(g); gs_.ensure(g);
  audio_d_.ensure(n * s.hop * 4);
}

void Engine::upload_inputs(const int64_t* ids_concat, const int64_t* lens, int B, const float scales[3],
                           const NoiseSpec& noise, const int32_t* w_ceil_override) {
  const VoiceSpec& s = voice_.spec;
  if (B <= 0) throw std::runtime_error("batch size must be positive");
  if (!ids_concat || !lens) throw std::runtime_error("null input pointer");
  CUDA_CHECK(cudaSetDevice(device_));
  int Tmax = 0;
  int64_t total = 0;
  for (int b = 0; b < B; ++b) {
    if (lens[b] <= 0) throw std::runtime_error("empty phoneme-id sequence (input_lengths must be >= 1)");
    if (lens[b] > (1 << 20)) throw std::runtime_error("phoneme-id sequence too long");
    Tmax = std::max<int>(Tmax, int(lens[b]));
    total += lens[b];
  }
  Tmax = bucket_ids(Tmax);                 // shape bucket (identity unless CUDA graphs are on): every kernel masks by len[b]
  B_ = B; Tmax_ = Tmax; Tp_ = slot(Tmax);
  sum_T_ = double(total);
  for (int i = 0; i < 3; ++i) scales_[i] = scales[i];
  seed_ = noise.seed;
  ensure_front(B, Tmax);
  // per-call scalars go to device memory (kernels.cuh CallParams): a replayed graph must see this call's values
  params_d_.ensure(sizeof(CallParams));
  params_pin_.ensure(sizeof(CallParams));
  CallParams* cp = params_pin_.as<CallParams>();
  cp->seed = seed_; cp->noise_scale = scales_[0]; cp->length_scale = scales_[1]; cp->noise_w = scales_[2]; cp->pad_ = 0.f;
  CUDA_CHECK(cudaMemcpyAsync(params_d_.p, cp, sizeof(CallParams), cudaMemcpyHostToDevice, stream_));
  len_h_.assign(B, 0);
  // ids: int64 host -> int32 [B][Tp] (validated: an out-of-range id would index past the embedding table)
  ids_pin_.ensure(size_t(B) * Tp_ * 4);
  int* ip = ids_pin_.as<int>();
  std::memset(ip, 0, size_t(B) * Tp_ * 4);
  int64_t pos = 0;
  for (int b = 0; b < B; ++b) {
    len_h_[b] = int(lens[b]);
    for (int t = 0; t < len_h_[b]; ++t) {
      const int64_t id = ids_concat[pos + t];
      if (id < 0 || id >= s.n_vocab)
        throw std::runtime_error("phoneme id " + std::to_string(id) + " outside the voice's symbol table [0," +
                                 std::to_string(s.n_vocab) + ")");
      ip[size_t(b) * Tp_ + t] = int(id);
    }
    pos += lens[b];
  }
  misc_pin_.ensure(size_t(B) * 32);
  int* lp = misc_pin_.as<int>();
  for (int b = 0; b < B; ++b) lp[b] = len_h_[b];
  CUDA_CHECK(cudaMemcpyAsync(ids_d_.p, ip, size_t(B) * Tp_ * 4, cudaMemcpyHostToDevice, stream_));
  CUDA_CHECK(cudaMemcpyAsync(len_d_.p, lp, size_t(B) * 4, cudaMemcpyHostToDevice, stream_));

  have_eps_dp_ = noise.eps_dp != nullptr;
  have_eps_z_ = noise.eps_z != nullptr;
  z_stride_ = noise.z_stride;
  if (have_eps_dp_) {
    epsdp_d_.ensure(size_t(total) * 2 * 4);
    CUDA_CHECK(cudaMemcpyAsync(epsdp_d_.p, noise.eps_dp, size_t(total) * 2 * 4, cudaMemcpyHostToDevice, stream_));
    long long* op = reinterpret_cast<long long*>(lp + B + (B & 1));
    long long o = 0;
    for (int b = 0; b < B; ++b) { op[b] = o; o += 2LL * len_h_[b]; }
    CUDA_CHECK(cudaMemcpyAsync(epsoff_d_.p, op, size_t(B) * 8, cudaMemcpyHostToDevice, stream_));
  }
  if (have_eps_z_) {
    if (z_stride_ <= 0) throw std::runtime_error("eps_z given without z_stride");
    const size_t n = size_t(B) * s.inter * size_t(z_stride_);
    epsz_d_.ensure(n * 4);
    CUDA_CHECK(cudaMemcpyAsync(epsz_d_.p, noise.eps_z, n * 4, cudaMemcpyHostToDevice, stream_));
  }
  have_override_ = w_ceil_override != nullptr;
  if (have_override_) {
    override_d_.ensure(size_t(total) * 4 + size_t(B) * Tp_ * 4);
    // ragged host array -> padded [B][Tp] (pinned: the copy leaves it before the next call, which starts after this
    // call's final stream synchronisation)
    override_pin_.ensure(size_t(B) * Tp_ * 4);
    int* tmp = override_pin_.as<int>();
    std::memset(tmp, 0, size_t(B) * Tp_ * 4);
    int64_t p2 = 0;
    for (int b = 0; b < B; ++b) {
      for (int t = 0; t < len_h_[b]; ++t) {
        const int v = w_ceil_override[p2 + t];
        if (v < 0) throw std::runtime_error("negative duration override");
        tmp[size_t(b) * Tp_ + t] = v;
      }
      p2 += len_h_[b];
    }
    CUDA_CHECK(cudaMemcpyAsync(override_d_.p, tmp, size_t(B) * Tp_ * 4, cudaMemcpyHostToDevice, stream_));
  }
  // No synchronisation here: the pinned staging buffers are next written by the NEXT call, and every public call ends
  // with a stream synchronisation; within this call the stream orders the copies before the kernels that read them.
}

void Engine::set_speakers(const int64_t* sids, int n) {
  sids_.clear();
  for (int i = 0; i < n; ++i) {
    if (sids[i] < 0 || sids[i] >= voice_.spec.n_speakers)
      throw std::runtime_error("speaker id " + std::to_string(sids[i]) + " outside [0," + std::to_string(voice_.spec.n_speakers) + ")");
    sids_.push_back(int(sids[i]));
  }
}

void Engine::upload_speakers(int B) {
  const VoiceSpec& s = voice_.spec;
  if (s.gin <= 0) return;
  std::vector<int> sid(B, 0);
  for (int b = 0; b < B; ++b)
    if (!sids_.empty()) sid[b] = sids_[std::min<size_t>(b, sids_.size() - 1)];
  sid_d_.ensure(size_t(B) * 4);
  cond_d_.ensure(size_t(B) * voice_.cond_rows * 4);
  // `sid` is pageable memory: cudaMemcpyAsync returns once it has been copied to the driver's staging buffer
  CUDA_CHECK(cudaMemcpyAsync(sid_d_.p, sid.data(), size_t(B) * 4, cudaMemcpyHostToDevice, stream_));
  launch_speaker_cond(W(voice_.cond_w), W(voice_.cond_b), W(voice_.emb_g), sid_d_.as<int>(), cond_d_.as<float>(),
                      voice_.cond_rows, s.gin, B, stream_);
}

void Engine::dds(const DDSW& d, View h, View u, View v, int C) {
  const int* len = len_d_.as<int>();
  for (const DDSLayerW& l : d.layers) {
    LnArgs a;
    a.a = h; a.y = u; a.gamma = W(l.n1.gamma); a.beta = W(l.n1.beta);
    a.dw_w = W(l.sep_w); a.dw_b = W(l.sep_b); a.dw_k = l.k; a.dw_dil = l.dil;
    a.C = C; a.mode = LN_DW_GELU; a.len = len;
    launch_layernorm(a, B_, Tmax_, stream_);
    ConvArgs c = conv_args(l.pw, u, len, 1);
    c.y = v; c.epi = EPI_BIAS;
    conv("dp", c, Tmax_, sum_T_);
    LnArgs b;
    b.a = v; b.r = h; b.y = h; b.gamma = W(l.n2.gamma); b.beta = W(l.n2.beta);
    b.C = C; b.mode = LN_GELU_RES; b.len = len;
    launch_layernorm(b, B_, Tmax_, stream_);
  }
}

void Engine::save_tap(const std::string& name, View v, int C, const int* len_host, int scale) {
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  // host copy is always [item][channel][pitch]; the device view may be that or the flat layout [channel][item][slot]
  const int pitch = v.bs < (long long)v.cs ? int(v.bs) : v.cs;
  HostTap t;
  t.B = B_; t.C = C; t.pitch = pitch;
  t.len.resize(B_);
  for (int b = 0; b < B_; ++b) t.len[b] = len_host[b] * scale;
  t.data.resize(size_t(B_) * C * pitch);
  for (int b = 0; b < B_; ++b)
    CUDA_CHECK(cudaMemcpy2D(t.data.data() + size_t(b) * C * pitch, size_t(pitch) * 4, v.p + (long long)b * v.bs, size_t(v.cs) * 4,
                            size_t(pitch) * 4, size_t(C), cudaMemcpyDeviceToHost));
  taps_[name] = std::move(t);
}

const HostTap* Engine::tap(const std::string& name) const {
  auto it = taps_.find(name);
  return it == taps_.end() ? nullptr : &it->second;
}

// ---- CUDA graphs ------------------------------------------------------------------------------------------------
bool Engine::graphs_on() {
  if (graph_mode_ < 0) {
    const char* e = std::getenv("PIPER_B200_GRAPH");
    graph_mode_ = e ? std::atoi(e) : 1;               // default on (PIPER_B200_GRAPH=0: direct launches)
  }
  return graph_mode_ > 0;
}
// Shape buckets: with graphs on, the grid-sizing lengths are rounded up so that one captured graph serves every call
// of the bucket (kernels read the true per-item lengths from device memory and skip tiles past them).
int Engine::bucket_ids(int t) const { return const_cast<Engine*>(this)->graphs_on() ? (t + 31) / 32 * 32 : t; }
int Engine::bucket_frames(int f) const { return const_cast<Engine*>(this)->graphs_on() ? (f + 63) / 64 * 64 : f; }

void Engine::record(int i) {
  // inside a capture a plain cudaEventRecord only expresses a dependency; the external flag makes it a record node
  if (capturing_) CUDA_CHECK(cudaEventRecordWithFlags(ev_[i], stream_, cudaEventRecordExternal));
  else CUDA_CHECK(cudaEventRecord(ev_[i], stream_));
}

void Engine::drop_graphs() {
  for (auto& kv : graphs_)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  graphs_.clear();
}

void Engine::run_graphed(unsigned long long key, const std::function<void()>& enqueue) {
  // explicit noise / duration overrides are test inputs with their own strides: only the production path is graphed
  if (!graphs_on() || debug_ || profile_ || have_eps_dp_ || have_eps_z_ || have_override_) {
    enqueue();
    return;
  }
  GraphSlot& g = graphs_[key];
  if (g.exec && g.gen == g_ws_generation.load()) {
    CUDA_CHECK(cudaGraphLaunch(g.exec, stream_));
    count_launches(g.launches);
    return;
  }
  if (g.exec) {
    cudaGraphExecDestroy(g.exec);
    g.exec = nullptr;
  }
  if (g.seen++ == 0) {                 // first call of a key runs directly: lazy weight packing, function attributes
    enqueue();
    return;
  }
  const unsigned long long n0 = launch_count();
  CUDA_CHECK(cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal));
  capturing_ = true;
  cudaGraph_t graph = nullptr;
  try {
    enqueue();
  } catch (...) {
    capturing_ = false;
    cudaStreamEndCapture(stream_, &graph);
    if (graph) cudaGraphDestroy(graph);
    throw;
  }
  capturing_ = false;
  CUDA_CHECK(cudaStreamEndCapture(stream_, &graph));
  cudaGraphExec_t exec = nullptr;
  cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) throw std::runtime_error(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
  g.exec = exec;
  g.gen = g_ws_generation.load();
  g.launches = launch_count() - n0;    // counted once while capturing; the launch below is that one execution
  CUDA_CHECK(cudaGraphLaunch(exec, stream_));
}

void Engine::run_front() {
  const int B = B_;
  if (debug_) taps_.clear();
  if (profile_) profile_begin();
  upload_speakers(B);
  CUDA_CHECK(cudaEventRecord(ev_[0], stream_));
  const unsigned long long key = (1ull << 60) | ((unsigned long long)B << 36) | ((unsigned long long)Tmax_ << 8) |
                                 (unsigned long long)(mma_mask_ & 0xff);
  run_graphed(key, [this] { enqueue_front(); });
  CUDA_CHECK(cudaGetLastError());
  CUDA_CHECK(cudaEventRecord(ev_[2], stream_));
  // ---- the one data-dependent host round trip: output lengths size everything downstream
  misc_pin_.ensure(size_t(B) * 32);
  int* yl = misc_pin_.as<int>();
  CUDA_CHECK(cudaMemcpyAsync(yl, ylen_d_.p, size_t(B) * 4, cudaMemcpyDeviceToHost, stream_));
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  ylen_h_.assign(yl, yl + B);
  if (debug_) {
    const int Tp = Tp_;
    HostTap t;
    t.B = B; t.C = 1; t.pitch = Tp; t.len = len_h_;
    t.data.resize(size_t(B) * Tp);
    CUDA_CHECK(cudaMemcpy(t.data.data(), logw_d_.p, size_t(B) * Tp * 4, cudaMemcpyDeviceToHost));
    taps_["logw"] = t;
    std::vector<int> cum(size_t(B) * Tp);
    CUDA_CHECK(cudaMemcpy(cum.data(), cum_d_.p, cum.size() * 4, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < cum.size(); ++i) t.data[i] = float(cum[i]);
    taps_["cum"] = t;
  }
}

void Engine::enqueue_front() {
  const VoiceSpec& s = voice_.spec;
  const int H = s.hidden, I = s.inter, Tp = Tp_, B = B_, T = Tmax_;
  const int* len = len_d_.as<int>();
  const CallParams* cp = params_d_.as<CallParams>();
  View x = fview(x_.as<float>(), H, Tp), t1 = fview(t1_.as<float>(), H, Tp), qkv = fview(qkv_.as<float>(), 3 * H, Tp),
       att = fview(att_.as<float>(), H, Tp), ffn = fview(ffn_.as<float>(), s.filter, Tp),
       stats = fview(stats_.as<float>(), 2 * I, Tp);
  // ---- text encoder (models.py:198-209)
  launch_embed(ids_d_.as<int>(), Tp, W(voice_.emb), H, std::sqrt(float(H)), x, len, B, T, stream_);
  for (const EncLayerW& e : voice_.enc) {
    ConvArgs c = conv_args(e.qkv, x, len, 1);
    c.y = qkv;
    conv("enc", c, T, sum_T_);
    launch_rel_attention(qkv, att, W(e.rel_k), W(e.rel_v), H, s.n_heads, s.window, len, B, T, stream_);
    c = conv_args(e.o, att, len, 1);
    c.y = t1; c.r = x; c.epi = EPI_RES;
    conv("enc", c, T, sum_T_);
    LnArgs l;
    l.a = t1; l.y = x; l.gamma = W(e.ln1.gamma); l.beta = W(e.ln1.beta); l.C = H; l.mode = LN_PLAIN; l.len = len;
    launch_layernorm(l, B, T, stream_);
    c = conv_args(e.ffn1, x, len, 1);
    c.y = ffn; c.epi = EPI_RELU;
    conv("enc", c, T, sum_T_);
    c = conv_args(e.ffn2, ffn, len, 1);
    c.y = t1; c.r = x; c.epi = EPI_RES;
    conv("enc", c, T, sum_T_);
    l.gamma = W(e.ln2.gamma); l.beta = W(e.ln2.beta);
    launch_layernorm(l, B, T, stream_);
  }
  {
    ConvArgs c = conv_args(voice_.enc_proj, x, len, 1);
    c.y = stats;
    conv("enc", c, T, sum_T_);
  }
  record(1);
  if (debug_) {
    save_tap("x", x, H, len_h_.data(), 1);
    save_tap("stats", stats, 2 * I, len_h_.data(), 1);
  }
  // ---- stochastic duration predictor, reverse (models.py:63-70,108-117)
  View g = fview(g_.as<float>(), H, Tp), h = fview(h_.as<float>(), H, Tp), u = fview(u_.as<float>(), H, Tp),
       v = fview(v_.as<float>(), H, Tp), z2 = fview(z2_.as<float>(), 2, Tp);
  const int pr_rows = 3 * s.spline_bins - 1;
  View pr = fview(pr_.as<float>(), pr_rows, Tp);
  {
    ConvArgs c = conv_args(voice_.dp_pre, x, len, 1);
    c.y = h;
    c.bias_item = cond_row(voice_.dp_cond_row);      // x = pre(x) + cond(g)  (models.py:66-68)
    c.bias_item_stride = voice_.cond_rows;
    conv("dp", c, T, sum_T_);
    dds(voice_.dp_dds, h, u, v, H);
    c = conv_args(voice_.dp_proj, h, len, 1);
    c.y = g;
    conv("dp", c, T, sum_T_);
  }
  launch_dp_noise(z2, have_eps_dp_ ? epsdp_d_.as<float>() : nullptr, epsoff_d_.as<long long>(), cp, len, B, T, stream_);
  bool flipped = false;
  for (const ConvFlowW& cf : voice_.dp_flows) {
    flipped = !flipped;                       // Flip precedes every ConvFlow in the reversed list
    const int x0 = flipped ? 1 : 0, x1 = 1 - x0;
    launch_cf_pre(z2, x0, W(cf.pre_w), W(cf.pre_b), g, h, H, len, B, T, stream_);
    dds(cf.dds, h, u, v, H);
    ConvArgs c = conv_args(cf.proj, h, len, 1);
    c.y = pr;
    conv("dp", c, T, sum_T_);
    launch_spline_inverse(z2, x1, pr, s.spline_bins, 1.f / std::sqrt(float(H)), 5.0f, len, B, T, stream_);
  }
  flipped = !flipped;                         // the Flip before ElementwiseAffine
  const int lw_ch = flipped ? 1 : 0;
  launch_durations(z2.offset_channels(lw_ch), voice_.ea_m[0], voice_.ea_scale[0], cp,
                   have_override_ ? override_d_.as<int>() : nullptr, Tp, cum_d_.as<int>(), Tp, ylen_d_.as<int>(),
                   logw_d_.as<float>(), len, B, T, stream_);
}

void Engine::plan_back() {
  const VoiceSpec& s = voice_.spec;
  int Fmax = 0;
  off_h_.assign(B_, 0);
  long long off = 0;
  for (int b = 0; b < B_; ++b) {
    if (ylen_h_[b] < 1) throw std::runtime_error("internal: non-positive output length");
    if (ylen_h_[b] > max_frames_)
      throw std::runtime_error("predicted utterance length " + std::to_string(ylen_h_[b]) + " frames exceeds the limit " +
                               std::to_string(max_frames_));
    if (have_eps_z_ && ylen_h_[b] > z_stride_)
      throw std::runtime_error("eps_z has " + std::to_string(z_stride_) + " columns but the utterance needs " +
                               std::to_string(ylen_h_[b]));
    Fmax = std::max(Fmax, ylen_h_[b]);
    off_h_[b] = off;
    off += (long long)ylen_h_[b] * s.hop;
  }
  total_samples_ = off;
  sum_F_ = double(off) / s.hop;
  Fmax = bucket_frames(Fmax);              // shape bucket (identity unless CUDA graphs are on)
  Fmax_ = Fmax;
  Fp_ = slot(Fmax);
  ensure_back(B_, Fmax);
  // tight audio layout: item b starts at off[b]
  audio_d_.ensure(size_t(std::max<long long>(off, 1)) * 4);
  long long* op = reinterpret_cast<long long*>(misc_pin_.as<int>() + B_ + (B_ & 1));
  for (int b = 0; b < B_; ++b) op[b] = off_h_[b];
  CUDA_CHECK(cudaMemcpyAsync(off_d_.p, op, size_t(B_) * 8, cudaMemcpyHostToDevice, stream_));
}

void Engine::run_generator() {
  const VoiceSpec& s = voice_.spec;
  const int B = B_, Fp = Fp_, F = Fmax_;
  const int* ylen = ylen_d_.as<int>();
  View z = fview(z_.as<float>(), s.inter, Fp);
  int ch = s.up_initial;
  View S = view(gs_.as<float>(), ch, Fp);
  {
    ConvArgs c = conv_args(voice_.dec_pre, z, ylen, 1);
    c.y = S;
    c.bias_item = cond_row(voice_.dec_cond_row);     // x = conv_pre(x) + cond(g)  (models.py:350-351)
    c.bias_item_stride = voice_.cond_rows;
    conv("dec.pre", c, F, sum_F_);
  }
  int rate = 1;
  const int nk = int(voice_.resblocks.at(0).size());
  // EPI_MRF mode 2 expects an accumulator initialised by an earlier resblock; every piper preset has 3 kernels
  if (nk < 2) throw std::runtime_error("generators with a single resblock kernel are not supported");
  for (size_t st = 0; st < voice_.ups.size(); ++st) {
    const ConvW& up = voice_.ups[st];
    const int co = up.rows / up.up;
    const int Lp_out = Fp * rate * up.up;
    View A = view(ga_.as<float>(), co, Lp_out);
    {
      ConvArgs c = conv_args(up, S, ylen, rate);
      c.pre = PRE_LRELU; c.slope = 0.1f;           // F.leaky_relu(x, LRELU_SLOPE) before every upsample (models.py:354)
      c.y = A; c.epi = EPI_UPSAMPLE; c.q_extra = up.k - 1;
      conv("dec.up", c, F * rate + c.q_extra, sum_F_ * rate);
    }
    rate *= up.up;
    ch = co;
    const int L = F * rate;
    View P = view(gp_.as<float>(), ch, Lp_out), Q = view(gq_.as<float>(), ch, Lp_out);
    S = view(gs_.as<float>(), ch, Lp_out);
    if (debug_) save_tap("up" + std::to_string(st), A, ch, ylen_h_.data(), rate);
    if ((mma_mask_ & 16) && !mrf_ready_) prepare_mrf_fused();
    if ((mma_mask_ & 16) && mrf_plans_[st].ok) {
      // the whole stage (all resblocks and the MRF average) in one launch
      MrfFusedArgs f;
      f.x = A; f.y = S; f.len = ylen; f.len_scale = rate; f.slope = 0.1f;
      f.w = mrf_w_.as<uint8_t>() + mrf_w_off_[st];
      f.bias = reinterpret_cast<const float*>(mrf_w_.as<uint8_t>() + mrf_b_off_[st]);
      // profile record: the layer-wise algorithmic work (SURVEY 8d) of everything this one launch replaces, so the
      // roofline fraction stays comparable with the layer-wise path (and may exceed 1: the fused kernel moves less)
      const bool tail = st + 1 == voice_.ups.size() && mrf_plan_post_.ok && !debug_;
      ProfRec pr{};
      if (profile_) {
        if (ev_used_ + 2 > ev_pool_.size()) {
          const size_t old_n = ev_pool_.size();
          ev_pool_.resize(old_n + 256);
          for (size_t i = old_n; i < ev_pool_.size(); ++i) CUDA_CHECK(cudaEventCreate(&ev_pool_[i]));
        }
        const MrfFusedPlan& pl = tail ? mrf_plan_post_ : mrf_plans_[st];
        const double Ls = sum_F_ * rate;
        double taps = 0;
        for (int c = 0; c < pl.n_chains; ++c) taps += double(pl.k[c]) * pl.n_steps;
        const double n_convs = double(pl.n_chains) * pl.n_steps;
        pr.tag = "dec.mrf"; pr.mma = true;
        pr.bytes = 4.0 * (n_convs * 2.0 * Ls * ch + taps * ch * ch + n_convs * ch);
        pr.flops = 2.0 * Ls * ch * ch * taps;
        if (tail) { pr.bytes += 4.0 * (Ls * ch + Ls + double(ch) * voice_.post_k); pr.flops += 2.0 * Ls * ch * voice_.post_k; }
        pr.ci = ch; pr.rows = ch; pr.k = int(taps); pr.dil = 0; pr.up = 1; pr.max_len = L; pr.len_sum = Ls;
        pr.e0 = ev_pool_[ev_used_++]; pr.e1 = ev_pool_[ev_used_++];
        CUDA_CHECK(cudaEventRecord(pr.e0, stream_));
      }
      auto done = [&] {
        if (!profile_) return;
        CUDA_CHECK(cudaEventRecord(pr.e1, stream_));
        recs_.push_back(pr);
      };
      if (tail) {
        // last stage: conv_post + tanh fused behind it, the stage output never goes to HBM (taps need it: debug off only)
        f.post_w = W(voice_.post_w); f.post_slope = 0.01f;
        f.audio = audio_d_.as<float>(); f.out_off = off_d_.as<long long>();
        launch_mrf_fused(f, mrf_plan_post_, B, L, stream_);
        done();
        return;
      }
      launch_mrf_fused(f, mrf_plans_[st], B, L, stream_);
      done();
      if (debug_) save_tap("stage" + std::to_string(st), S, ch, ylen_h_.data(), rate);
      continue;
    }
    for (int j = 0; j < nk; ++j) {
      const ResBlockW& rb = voice_.resblocks[st][j];
      const int mrf = nk == 1 ? 2 : (j == 0 ? 0 : (j == nk - 1 ? 2 : 1));
      const int n = int(rb.c1.size());
      View y = A;
      for (int c = 0; c < n; ++c) {
        const bool last = c == n - 1;
        if (s.resblock == 1) {
          ConvArgs a1 = conv_args(rb.c1[c], y, ylen, rate);
          a1.pre = PRE_LRELU; a1.slope = 0.1f; a1.y = P; a1.epi = EPI_BIAS;
          conv("dec.rb", a1, L, sum_F_ * rate);
          ConvArgs a2 = conv_args(rb.c2[c], P, ylen, rate);
          a2.pre = PRE_LRELU; a2.slope = 0.1f; a2.r = y;
          if (last) { a2.epi = EPI_MRF; a2.y2 = S; a2.mrf = mrf; a2.mrf_n = nk; }
          else { a2.epi = EPI_RES; a2.y = Q; }
          conv("dec.rb", a2, L, sum_F_ * rate);
          y = Q;
        } else {
          ConvArgs a1 = conv_args(rb.c1[c], y, ylen, rate);
          a1.pre = PRE_LRELU; a1.slope = 0.1f; a1.r = y;
          View dst = (c & 1) ? Q : P;
          if (last) { a1.epi = EPI_MRF; a1.y2 = S; a1.mrf = mrf; a1.mrf_n = nk; }
          else { a1.epi = EPI_RES; a1.y = dst; }
          conv("dec.rb", a1, L, sum_F_ * rate);
          y = dst;
        }
      }
    }
    if (debug_) save_tap("stage" + std::to_string(st), S, ch, ylen_h_.data(), rate);
  }
  launch_conv_post(S, W(voice_.post_w), voice_.post_c, voice_.post_k, 0.01f, audio_d_.as<float>(),
                   off_d_.as<long long>(), ylen, rate, B, F * rate, stream_);
}

void Engine::prepare_mrf_fused() {
  const size_t n = voice_.ups.size();
  mrf_plans_.assign(n, MrfFusedPlan{});
  mrf_w_off_.assign(n, 0);
  mrf_b_off_.assign(n, 0);
  std::vector<uint8_t> host;
  int ch = voice_.spec.up_initial;
  for (size_t st = 0; st < n; ++st) {
    ch = voice_.ups[st].rows / voice_.ups[st].up;
    MrfFusedPlan& p = mrf_plans_[st];
    if (!plan_mrf_fused(voice_.resblocks[st], voice_.spec.resblock, ch, 0, p)) continue;
    if (st + 1 == n && ch == voice_.post_c)
      plan_mrf_fused(voice_.resblocks[st], voice_.spec.resblock, ch, voice_.post_k, mrf_plan_post_);
    const size_t w_off = (host.size() + 127) & ~size_t(127);
    const size_t b_off = w_off + p.w_bytes;
    host.resize(b_off + size_t(p.n_bias) * 4);
    pack_mrf_fused(voice_.blob.data(), voice_.resblocks[st], p, host.data() + w_off,
                   reinterpret_cast<float*>(host.data() + b_off));
    mrf_w_off_[st] = w_off;
    mrf_b_off_[st] = b_off;
  }
  if (!host.empty()) {
    mrf_w_.ensure(host.size());
    CUDA_CHECK(cudaMemcpyAsync(mrf_w_.p, host.data(), host.size(), cudaMemcpyHostToDevice, stream_));   // (see conv2_layer)
    CUDA_CHECK(cudaStreamSynchronize(stream_));
  }
  mrf_ready_ = true;
}

void Engine::run_flow() {
  const VoiceSpec& s = voice_.spec;
  const int B = B_, H = s.hidden, I = s.inter, Fp = Fp_, F = Fmax_;
  const int* ylen = ylen_d_.as<int>();
  View z = fview(z_.as<float>(), I, Fp);
  // ---- flow, reverse (models.py:251-253; modules.py:447-466,184-209)
  View fh = fview(fh_.as<float>(), H, Fp), acts = fview(facts_.as<float>(), H, Fp), out = fview(fout_.as<float>(), H, Fp);
  const int half = I / 2;
  for (const CouplingW& cw : voice_.flow) {
    View x0 = cw.flipped ? z.offset_channels(half) : z;
    View x1 = cw.flipped ? z : z.offset_channels(half);
    ConvArgs c = conv_args(cw.pre, x0, ylen, 1);
    c.y = fh;
    conv("flow", c, F, sum_F_);
    const int nl = int(cw.in_layers.size());
    for (int i = 0; i < nl; ++i) {
      ConvArgs a = conv_args(cw.in_layers[i], fh, ylen, 1);
      a.y = acts; a.epi = EPI_GATE;
      if (cw.cond_row >= 0) {                          // in_act = x_in + g_l  (modules.py:188-199)
        a.bias_item = cond_row(cw.cond_row + i * 2 * H);
        a.bias_item_stride = voice_.cond_rows;
      }
      conv("flow", a, F, sum_F_);
      ConvArgs r = conv_args(cw.res_skip[i], acts, ylen, 1);
      r.epi = EPI_WN; r.y = fh; r.r = fh; r.y2 = out; r.first = i == 0;
      r.split = i < nl - 1 ? H : 0;
      conv("flow", r, F, sum_F_);
    }
    ConvArgs p = conv_args(cw.post, out, ylen, 1);
    p.epi = EPI_SUBFROM; p.y = x1; p.r = x1;
    conv("flow", p, F, sum_F_);
  }
}

void Engine::enqueue_back() {
  const VoiceSpec& s = voice_.spec;
  const int B = B_, I = s.inter, Fp = Fp_, F = Fmax_;
  const int* ylen = ylen_d_.as<int>();
  const int* len = len_d_.as<int>();
  View stats = fview(stats_.as<float>(), 2 * I, Tp_);
  View z = fview(z_.as<float>(), I, Fp);
  launch_expand(stats, I, cum_d_.as<int>(), Tp_, len, ylen, z, have_eps_z_ ? epsz_d_.as<float>() : nullptr,
                (long long)I * z_stride_, int(z_stride_), params_d_.as<CallParams>(), B, F, stream_);
  if (debug_) save_tap("z_p", z, I, ylen_h_.data(), 1);
  run_flow();
  if (debug_) save_tap("z", z, I, ylen_h_.data(), 1);
  record(4);
  run_generator();
}

void Engine::run_back() {
  CUDA_CHECK(cudaEventRecord(ev_[3], stream_));
  const unsigned long long key = (2ull << 60) | ((unsigned long long)B_ << 36) | ((unsigned long long)Fmax_ << 8) |
                                 (unsigned long long)(mma_mask_ & 0xff);
  run_graphed(key, [this] { enqueue_back(); });
  CUDA_CHECK(cudaGetLastError());
  CUDA_CHECK(cudaEventRecord(ev_[5], stream_));
}

void Engine::stage(const int64_t* ids_concat, const int64_t* lens, int B, const float scales[3], const NoiseSpec& noise,
                   const int32_t* w_ceil_override) {
  upload_inputs(ids_concat, lens, B, scales, noise, w_ceil_override);
}

int64_t Engine::run_staged(float* device_ms) {
  if (B_ <= 0) throw std::runtime_error("run_staged: nothing staged");
  CUDA_CHECK(cudaSetDevice(device_));
  run_front();
  plan_back();
  run_back();
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  collect_stage_times();
  if (device_ms) {
    float tot = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&tot, ev_[0], ev_[5]));
    *device_ms = tot;
  }
  return total_samples_;
}

void Engine::collect_stage_times() {
  for (int i = 0; i < 5; ++i) CUDA_CHECK(cudaEventElapsedTime(&stage_ms_[i], ev_[i], ev_[i + 1]));
}

void Engine::stage_times(float out_ms[5]) const {
  for (int i = 0; i < 5; ++i) out_ms[i] = stage_ms_[i];
}

const float* Engine::synthesize(const int64_t* ids_concat, const int64_t* lens, int B, const float scales[3],
                                const NoiseSpec& noise, const int32_t* w_ceil_override, int64_t* n_samples,
                                double* infer_seconds) {
  const auto t0 = std::chrono::steady_clock::now();
  upload_inputs(ids_concat, lens, B, scales, noise, w_ceil_override);
  run_front();
  plan_back();
  run_back();
  audio_pin_.ensure(size_t(std::max<int64_t>(total_samples_, 1)) * 4);
  CUDA_CHECK(cudaMemcpyAsync(audio_pin_.p, audio_d_.p, size_t(total_samples_) * 4, cudaMemcpyDeviceToHost, stream_));
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  collect_stage_times();
  if (debug_) {
    HostTap t;
    t.B = 1; t.C = 1; t.pitch = int(total_samples_); t.len = {int(total_samples_)};
    t.data.assign(audio_pin_.as<float>(), audio_pin_.as<float>() + total_samples_);
    taps_["audio"] = std::move(t);
  }
  for (int b = 0; b < B; ++b)
    if (n_samples) n_samples[b] = int64_t(ylen_h_[b]) * voice_.spec.hop;
  if (infer_seconds)
    *infer_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return audio_pin_.as<float>();
}

const int16_t* Engine::synthesize_int16(const int64_t* ids_concat, const int64_t* lens, int B, const float scales[3],
                                        const NoiseSpec& noise, int64_t* n_samples, double* infer_seconds) {
  const auto t0 = std::chrono::steady_clock::now();
  upload_inputs(ids_concat, lens, B, scales, noise, nullptr);
  run_front();
  plan_back();
  run_back();
  const int hop = voice_.spec.hop;
  audio16_d_.ensure(size_t(std::max<int64_t>(total_samples_, 1)) * 2);
  CUDA_CHECK(cudaMemsetAsync(peak_d_.p, 0, size_t(B) * 4, stream_));
  launch_peak(audio_d_.as<float>(), off_d_.as<long long>(), ylen_d_.as<int>(), hop, peak_d_.as<unsigned int>(), B,
              Fmax_ * hop, stream_);
  launch_to_int16(audio_d_.as<float>(), off_d_.as<long long>(), ylen_d_.as<int>(), hop, peak_d_.as<unsigned int>(),
                  audio16_d_.as<int16_t>(), B, Fmax_ * hop, stream_);
  audio16_pin_.ensure(size_t(std::max<int64_t>(total_samples_, 1)) * 2);
  CUDA_CHECK(cudaMemcpyAsync(audio16_pin_.p, audio16_d_.p, size_t(total_samples_) * 2, cudaMemcpyDeviceToHost, stream_));
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  collect_stage_times();
  for (int b = 0; b < B; ++b)
    if (n_samples) n_samples[b] = int64_t(ylen_h_[b]) * hop;
  if (infer_seconds)
    *infer_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return audio16_pin_.as<int16_t>();
}

const float* Engine::encode(const int64_t* ids, int64_t n_ids, const float scales[3], const NoiseSpec& noise,
                            int64_t* frames, double* infer_seconds) {
  // Encoder half of the reference's streaming split (export_onnx_streaming.py:19-58): text encoder, duration
  // predictor, length regulator and the prior sample z_p [inter][T'] - everything before the flow.
  const auto t0 = std::chrono::steady_clock::now();
  int64_t lens[1] = {n_ids};
  upload_inputs(ids, lens, 1, scales, noise, nullptr);
  run_front();
  plan_back();
  const VoiceSpec& s = voice_.spec;
  View stats = fview(stats_.as<float>(), 2 * s.inter, Tp_);
  View z = fview(z_.as<float>(), s.inter, Fp_);
  launch_expand(stats, s.inter, cum_d_.as<int>(), Tp_, len_d_.as<int>(), ylen_d_.as<int>(), z,
                have_eps_z_ ? epsz_d_.as<float>() : nullptr, (long long)s.inter * z_stride_, int(z_stride_),
                params_d_.as<CallParams>(), 1, Fmax_, stream_);
  const int F = ylen_h_[0];
  audio_pin_.ensure(size_t(s.inter) * F * 4);
  CUDA_CHECK(cudaMemcpy2DAsync(audio_pin_.p, size_t(F) * 4, z.p, size_t(z.cs) * 4, size_t(F) * 4, size_t(s.inter),
                               cudaMemcpyDeviceToHost, stream_));
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  if (frames) *frames = F;
  if (infer_seconds) *infer_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return audio_pin_.as<float>();
}

const float* Engine::vocode(const float* z, int B, int64_t frames, bool with_flow, double* infer_seconds) {
  const VoiceSpec& s = voice_.spec;
  if (B <= 0 || frames <= 0 || !z) throw std::runtime_error("vocode: bad arguments");
  if (frames > max_frames_) throw std::runtime_error("vocode: too many frames");
  const auto t0 = std::chrono::steady_clock::now();
  CUDA_CHECK(cudaSetDevice(device_));
  // Generator only: nothing here cuts tiles on a concatenated axis, and the host tensor is item-major - keep the per-item
  // layout so the upload stays ONE 2-D copy.  (With the flow - the streaming decoder - the flat layout is used; for B = 1
  // the two coincide.)
  flat_on();
  struct FlatGuard { int& f; int saved; ~FlatGuard() { f = saved; } } flat_guard{flat_, flat_};
  if (!with_flow) flat_ = 0;
  B_ = B; Tmax_ = 1; Tp_ = 4;
  ensure_front(B, 1);
  ylen_h_.assign(B, int(frames));
  len_h_.assign(B, 1);
  misc_pin_.ensure(size_t(B) * 32);
  int* yl = misc_pin_.as<int>();
  for (int b = 0; b < B; ++b) yl[b] = int(frames);
  CUDA_CHECK(cudaMemcpyAsync(ylen_d_.p, yl, size_t(B) * 4, cudaMemcpyHostToDevice, stream_));
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  have_eps_z_ = have_eps_dp_ = have_override_ = false;
  plan_back();
  upload_speakers(B);
  if (debug_) taps_.clear();
  // z host [B][inter][frames] -> the device view (per item: [inter] rows of `frames` floats at the view's channel stride)
  {
    const View zv = fview(z_.as<float>(), s.inter, Fp_);
    if (zv.bs == (long long)s.inter * zv.cs) {           // item-major device layout: one copy of B * inter rows
      CUDA_CHECK(cudaMemcpy2DAsync(zv.p, size_t(zv.cs) * 4, z, size_t(frames) * 4, size_t(frames) * 4, size_t(B) * s.inter,
                                   cudaMemcpyHostToDevice, stream_));
    } else {
      for (int b = 0; b < B; ++b)
        CUDA_CHECK(cudaMemcpy2DAsync(zv.p + (long long)b * zv.bs, size_t(zv.cs) * 4, z + size_t(b) * s.inter * frames,
                                     size_t(frames) * 4, size_t(frames) * 4, size_t(s.inter), cudaMemcpyHostToDevice, stream_));
    }
  }
  {
    const unsigned long long key = (3ull << 60) | ((unsigned long long)B << 36) | ((unsigned long long)Fmax_ << 8) |
                                   (unsigned long long)(mma_mask_ & 0x7f) | (with_flow ? 0x80ull : 0ull);   // (layout follows with_flow)
    run_graphed(key, [this, with_flow] {
      if (with_flow) run_flow();             // decoder half of the reference's streaming split (flow + generator)
      record(4);
      run_generator();
    });
  }
  CUDA_CHECK(cudaEventRecord(ev_[5], stream_));
  audio_pin_.ensure(size_t(total_samples_) * 4);
  CUDA_CHECK(cudaMemcpyAsync(audio_pin_.p, audio_d_.p, size_t(total_samples_) * 4, cudaMemcpyDeviceToHost, stream_));
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  CUDA_CHECK(cudaEventElapsedTime(&stage_ms_[4], ev_[4], ev_[5]));
  if (infer_seconds)
    *infer_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return audio_pin_.as<float>();
}

}  // namespace pb200
