// Host-side engine: owns one voice's packed weights in HBM, a grow-only activation workspace, one
// CUDA stream, and runs the VITS inference graph (SynthesizerTrn.infer, models.py:681-722) as a
// sequence of hand-written sm_100a kernels.  This is what stands behind `Ort::Session::Run` at
// /root/reference/src/cpp/piper.cpp:386-388.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <functional>
#include <map>
#include <utility>
#include <memory>
#include <string>
#include <vector>

#include "kernels.cuh"
#include "voice.h"

namespace pb200 {

struct DeviceBuf {
  void* p = nullptr;
  size_t cap = 0;
  DeviceBuf() = default;
  DeviceBuf(const DeviceBuf&) = delete;
  DeviceBuf& operator=(const DeviceBuf&) = delete;
  ~DeviceBuf() { release(); }        // an Engine constructor that throws half-way must not leak HBM
  void ensure(size_t bytes);
  void release();
  template <class T> T* as() const { return static_cast<T*>(p); }
};
struct PinnedBuf {
  void* p = nullptr;
  size_t cap = 0;
  PinnedBuf() = default;
  PinnedBuf(const PinnedBuf&) = delete;
  PinnedBuf& operator=(const PinnedBuf&) = delete;
  ~PinnedBuf() { release(); }
  void ensure(size_t bytes);
  void release();
  template <class T> T* as() const { return static_cast<T*>(p); }
};

struct NoiseSpec {
  const float* eps_dp = nullptr;  // host, item-major [sum_b 2*len_b]; null => Philox(seed)
  const float* eps_z = nullptr;   // host, [B][inter][z_stride]; null => Philox(seed)
  int64_t z_stride = 0;
  uint64_t seed = 0;
};

struct HostTap {
  int B = 0, C = 0;
  std::vector<int> len;           // valid length per item
  int pitch = 0;
  std::vector<float> data;        // [B][C][pitch]
};

class Engine {
 public:
  // upload = false: allocate the HBM weight buffer but leave it unfilled (a peer broadcasts into it)
  Engine(const std::string& onnx_path, int device, bool upload = true);
  ~Engine();
  Engine(const Engine&) = delete;
  Engine& operator=(const Engine&) = delete;

  const VoiceSpec& spec() const { return voice_.spec; }
  const PackedVoice& voice() const { return voice_; }
  int device() const { return device_; }
  int64_t weight_bytes() const { return int64_t(voice_.blob.size()) * 4; }
  // device pointer of the fp32 weight blob for load-time broadcast
  void weight_buffers(void** fp32, int64_t* fp32_bytes) const {
    *fp32 = weights_.p; *fp32_bytes = int64_t(voice_.blob.size()) * 4;
  }

  // ---- whole pipeline, host buffers in / host buffer out (the reference-facing call)
  // ids_concat: int64 [sum lens]; returns pointer to pinned fp32 audio (valid until the next call),
  // n_samples[b] = y_len[b] * hop, items concatenated in order.
  const float* synthesize(const int64_t* ids_concat, const int64_t* lens, int B, const float scales[3],
                          const NoiseSpec& noise, const int32_t* w_ceil_override, int64_t* n_samples,
                          double* infer_seconds);
  // Same, with the int16 peak-normalisation epilogue of piper.cpp:411-431 fused on the GPU.
  const int16_t* synthesize_int16(const int64_t* ids_concat, const int64_t* lens, int B, const float scales[3],
                                  const NoiseSpec& noise, int64_t* n_samples, double* infer_seconds);
  // Generator only: z host [B][inter][frames] -> audio [B][frames*hop]
  const float* vocode(const float* z, int B, int64_t frames, bool with_flow, double* infer_seconds);
  // encoder half of the streaming split: ids -> z_p [inter][frames] (host, pinned)
  const float* encode(const int64_t* ids, int64_t n_ids, const float scales[3], const NoiseSpec& noise, int64_t* frames,
                      double* infer_seconds);

  // ---- staged execution for device-resident timing (bench.py `value`)
  void stage(const int64_t* ids_concat, const int64_t* lens, int B, const float scales[3], const NoiseSpec& noise,
             const int32_t* w_ceil_override);
  // runs the kernels on the already-staged inputs; audio stays in HBM. Returns total valid samples and the
  // device time (CUDA events on the engine's stream) in ms.
  int64_t run_staged(float* device_ms);
  // per-stage device times of the last run_staged/synthesize: enc, dp, sync, flow(expand+flow), dec
  void stage_times(float out_ms[5]) const;

  // per-launch CUDA-event timing of the conv kernel family, aggregated by pipeline stage (bench.py roofline)
  void set_profile(bool on) { profile_ = on; }
  std::string profile_json();
  std::string profile_launches_json();   // every conv launch of the last call, in order
  void set_mma(int mask) { mma_mask_ = mask; }
  int mma() const { return mma_mask_; }
  // speaker ids for the next calls (multi-speaker voices); item b uses sids[min(b, n-1)], default speaker 0
  void set_speakers(const int64_t* sids, int n);
  void set_debug(bool on) { debug_ = on; }
  const HostTap* tap(const std::string& name) const;
  void set_max_frames(int64_t f) { max_frames_ = f; }

 private:
  void upload_inputs(const int64_t* ids_concat, const int64_t* lens, int B, const float scales[3],
                     const NoiseSpec& noise, const int32_t* w_ceil_override);
  void run_front();              // encoder + duration predictor, ends with the y_len D2H + sync
  void plan_back();              // host: sizes, offsets, workspace growth
  void run_back();               // expand + flow + generator -> audio_d_
  void run_flow();               // in place on z_
  void run_generator();
  void ensure_front(int B, int Tmax);
  void ensure_back(int B, int Fmax);
  void collect_stage_times();
  // every dense conv goes through here: the tensor-core kernel (conv_mma2.cu) when the layer's family (1 = generator,
  // 2 = flow, 4 = text encoder, 8 = duration predictor) is enabled and conv2_plan takes its shape, CUDA-core kernel otherwise
  void conv(const char* tag, ConvArgs& a, int max_len, double len_sum);
  void profile_begin();
  void save_tap(const std::string& name, View v, int C, const int* len_host, int scale);

  View view(float* p, int C, int pitch) const { return View{p, (long long)C * pitch, pitch}; }
  // phoneme- / frame-rate activations: [item][channel][pitch], or the flat layout [channel][item][slot] (engine.cu: flat_on)
  View fview(float* p, int C, int pitch) const;
  bool flat_on();
  int slot(int max_len);
  int flat_ = -1;
  const float* W(int64_t off) const { return off >= 0 ? weights_.as<float>() + off : nullptr; }
  ConvArgs conv_args(const ConvW& c, View x, const int* len, int len_scale) const;
  void dds(const DDSW& d, View h, View u, View v, int C);

  PackedVoice voice_;
  int device_ = 0;
  cudaStream_t stream_ = nullptr;
  cudaEvent_t ev_[8] = {};
  DeviceBuf weights_;
  // tensor-core conv (conv_mma2.cu): per-layer plan + stacked weights, packed lazily from the fp32 blob; null = not taken
  std::map<std::pair<const ConvW*, int>, Conv2Layer> conv2_layers_;   // (layer, variant): see conv2_layer
  const Conv2Layer* conv2_layer(const ConvW& w, const ConvArgs& a, bool fp32_grade, int variant = 0);
  // fused MRF stage (mask bit 16, mrf_fused.cu): packed lazily on first use
  void prepare_mrf_fused();
  bool mrf_ready_ = false;
  std::vector<MrfFusedPlan> mrf_plans_;
  MrfFusedPlan mrf_plan_post_;        // last stage with conv_post + tanh fused behind it (used when taps are off)
  std::vector<size_t> mrf_w_off_, mrf_b_off_;
  DeviceBuf mrf_w_;
  int mma_mask_ = 31;  // every conv family and the fused MRF stage on the tensor cores, fp16x3 (DESIGN.md §3)

  // request state
  int B_ = 0, Tmax_ = 0, Tp_ = 0, Fmax_ = 0, Fp_ = 0;
  float scales_[3] = {0.667f, 1.f, 0.8f};
  uint64_t seed_ = 0;
  bool have_eps_dp_ = false, have_eps_z_ = false, have_override_ = false;
  int64_t z_stride_ = 0;
  std::vector<int> len_h_, ylen_h_;
  std::vector<long long> off_h_;
  int64_t total_samples_ = 0;
  int64_t max_frames_ = 1 << 17;

  // phoneme-rate workspace
  std::vector<int> sids_;
  DeviceBuf sid_d_, cond_d_;
  void upload_speakers(int B);   // sid per item -> device, cond = W_cond * emb_g[sid] + b (no-op for single-speaker voices)
  const float* cond_row(int row) const { return row >= 0 && cond_d_.p ? cond_d_.as<float>() + row : nullptr; }
  DeviceBuf ids_d_, len_d_, ylen_d_, cum_d_, logw_d_, override_d_, epsdp_d_, epsoff_d_, off_d_;
  DeviceBuf x_, t1_, qkv_, att_, ffn_, stats_, g_, h_, u_, v_, pr_, z2_;
  // frame-rate workspace
  DeviceBuf z_, fh_, facts_, fout_, epsz_d_;
  // sample-rate workspace
  DeviceBuf ga_, gp_, gq_, gs_, audio_d_, audio16_d_, peak_d_;
  PinnedBuf ids_pin_, misc_pin_, audio_pin_, audio16_pin_, eps_pin_;

  // ---- CUDA graphs (PIPER_B200_GRAPH, engine.cu): the launch sequences of the front half (text encoder + duration
  // predictor) and of the back half (expand + flow + generator) are captured once per shape bucket and replayed; the
  // data-dependent output lengths are read from device memory by every kernel, so one graph serves a whole bucket.
  struct GraphSlot {
    cudaGraphExec_t exec = nullptr;
    unsigned long long gen = 0;      // workspace generation the graph's pointers belong to
    int seen = 0;                    // calls with this key so far (the first one runs un-captured: lazy initialisation)
    unsigned long long launches = 0; // kernel nodes (for launch_count)
  };
  std::map<unsigned long long, GraphSlot> graphs_;
  int graph_mode_ = -1;              // -1: read PIPER_B200_GRAPH on first use
  bool capturing_ = false;
  bool graphs_on();
  void run_graphed(unsigned long long key, const std::function<void()>& enqueue);
  void record(int ev);               // stage event, usable inside a captured region
  void drop_graphs();
  int bucket_ids(int t) const;       // shape buckets (identity when graphs are off)
  int bucket_frames(int f) const;
  void enqueue_front();
  void enqueue_back();
  DeviceBuf params_d_;               // CallParams of the current call
  PinnedBuf params_pin_, override_pin_;

  struct ProfRec { const char* tag; bool mma; cudaEvent_t e0, e1; double bytes, flops; int ci, rows, k, dil, up, max_len; double len_sum; };
  bool profile_ = false;
  static constexpr size_t kProfRecs = 1024;
  DeviceBuf prof_d_;                       // PIPER_B200_PROF_ROLES: 16 counters per profiled launch
  std::vector<cudaEvent_t> ev_pool_;
  size_t ev_used_ = 0;
  std::vector<ProfRec> recs_;
  double sum_T_ = 0, sum_F_ = 0;
  bool debug_ = false;
  std::map<std::string, HostTap> taps_;
  float stage_ms_[5] = {0, 0, 0, 0, 0};
};

}  // namespace pb200
