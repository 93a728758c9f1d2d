/* piper_b200 — C ABI of the B200-native VITS inference engine.
 *
 * Drop-in boundary: these entry points replace what piper's C++ host obtains from onnxruntime
 * for the phoneme-ids -> waveform path.  Each one names the reference interface it stands in for
 * (paths relative to the rhasspy/piper tree, commit 73c04d8):
 *
 *   pb200_voice_load        <- loadModel(): Ort::Env + Ort::SessionOptions + Ort::Session(modelPath)
 *                              src/cpp/piper.cpp:262-306 (called from loadVoice, :309-334)
 *   pb200_voice_free        <- ~ModelSession (Ort::Session release), src/cpp/piper.hpp:78-85
 *   pb200_synthesize        <- inside synthesize(): CreateTensor x3(4) + session.onnx.Run(...)
 *                              + GetTensorData/GetShape, src/cpp/piper.cpp:342-400
 *   pb200_release           <- Ort::detail::OrtRelease(outputTensors[i].release()), piper.cpp:434-440
 *   pb200_synthesize_int16  <- the same Run plus the host loops that peak-normalise to int16,
 *                              src/cpp/piper.cpp:411-431 (python twin: src/python_run/piper/util.py:5-12)
 *   pb200_synthesize_batch  <- the graph's dynamic batch axis (export_onnx.py:96-100); no reference
 *                              caller uses B > 1 (piper.cpp:352), semantics are B independent utterances
 *   pb200_vocode            <- the decoder half of the reference's streaming export
 *                              (src/python/piper_train/export_onnx_streaming.py:61-69)
 *   pb200_last_error        <- the std::runtime_error / Ort::Exception messages thrown up to main
 *                              (e.g. piper.cpp:391-393); the C ABI returns codes, the C++ shim rethrows.
 *
 * Plain C types only: no torch / CUDA types cross this boundary.  All calls are blocking and may be
 * issued repeatedly from one thread per voice handle (the reference's threading contract, SURVEY §8b).
 * There is NO CPU fallback: without a usable sm_100 device pb200_voice_load fails.
 */
#ifndef PIPER_B200_H_
#define PIPER_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB200_OK 0
#define PB200_ERROR 1

typedef struct pb200_voice pb200_voice;

/* Inferred from the .onnx initializer shapes (hyper-parameters are not in the voice JSON). */
typedef struct pb200_voice_info {
  int32_t n_vocab, hidden, inter, filter, n_heads, n_layers, window;
  int32_t resblock;        /* 1 (high) or 2 (x-low / low / medium) */
  int32_t n_upsamples;
  int32_t hop;             /* samples per frame = prod(upsample_rates) */
  int32_t up_initial;
  int32_t device;
  int32_t n_speakers;      /* rows of emb_g (1 for single-speaker voices) */
  int32_t gin;             /* speaker-embedding width, 0 for single-speaker voices */
  int64_t n_params;        /* fp32 parameters read from the file */
  int64_t weight_bytes;    /* packed blob resident in HBM */
} pb200_voice_info;

/* Noise for the graph's two RandomNormalLike nodes (unseeded in the reference export).
 * eps_dp : item-major, for item b a [2][len_b] block          (models.py:111)   or NULL
 * eps_z  : [B][inter][z_stride], only the first y_len_b columns are read (models.py:718) or NULL
 * NULL pointers draw N(0,1) on the device from a Philox stream keyed by `seed`. */
typedef struct pb200_noise {
  const float* eps_dp;
  const float* eps_z;
  int64_t z_stride;
  uint64_t seed;
} pb200_noise;

/* Parse `onnx_path`, pack the weights and upload them to CUDA device `device`. */
int pb200_voice_load(const char* onnx_path, int device, pb200_voice** out);
/* Multi-GPU load (SURVEY §8e): every rank parses the file (host only), rank 0 uploads, the other ranks pass
 * PB200_LOAD_NO_UPLOAD and receive the packed fp32 weight blob by an NCCL broadcast over NVLink into the device
 * buffer returned by pb200_voice_weight_buffers.  Every rank packs its own tensor-core weights from its host parse on
 * first use.  The hot path itself has no collective: utterances are independent. */
#define PB200_LOAD_NO_UPLOAD 1
int pb200_voice_load_ex(const char* onnx_path, int device, int32_t flags, pb200_voice** out);
int pb200_voice_weight_buffers(pb200_voice* v, void** fp32, int64_t* fp32_bytes);
void pb200_voice_free(pb200_voice* v);
int pb200_voice_get_info(const pb200_voice* v, pb200_voice_info* info);

/* Host-only (no GPU needed): parse + pack and describe the result as JSON into buf (NUL-terminated,
 * truncated to cap).  Returns PB200_OK or PB200_ERROR. */
int pb200_voice_describe(const char* onnx_path, char* buf, int64_t cap);
/* Host-only: copy the packed weight blob (for loader tests).  *n_floats in: capacity, out: size. */
int pb200_voice_pack(const char* onnx_path, float* blob, int64_t* n_floats);

/* One utterance.  ids: int64 [n_ids]; scales = {noise_scale, length_scale, noise_w};
 * sid: speaker id for multi-speaker voices (the graph's `sid` input, piper.cpp:367-377) or NULL (speaker 0).  On success *audio points at fp32 samples owned by the
 * engine (pinned host memory), valid until the next call on this voice or pb200_release(). */
int pb200_synthesize(pb200_voice* v, const int64_t* ids, int64_t n_ids, const float scales[3], const int64_t* sid,
                     const pb200_noise* noise, const float** audio, int64_t* n_samples, double* infer_seconds);

/* B utterances (ragged): ids_concat int64 [sum lens], lens int64 [B].  Audio is the concatenation of the
 * items' valid samples; n_samples[b] = y_len_b * hop.  w_ceil_override (int32, ids_concat layout) replaces
 * the predicted per-id frame counts when non-NULL (benchmark / test control of T'). */
int pb200_synthesize_batch(pb200_voice* v, const int64_t* ids_concat, const int64_t* lens, int32_t B,
                           const float scales[3], const pb200_noise* noise, const int32_t* w_ceil_override,
                           const float** audio, int64_t* n_samples, double* infer_seconds);

/* As above with the int16 peak-normalisation of piper.cpp:411-431 fused on the GPU (per utterance). */
int pb200_synthesize_int16(pb200_voice* v, const int64_t* ids_concat, const int64_t* lens, int32_t B,
                           const float scales[3], const pb200_noise* noise, const int16_t** audio,
                           int64_t* n_samples, double* infer_seconds);

/* Generator only: z fp32 [B][inter][frames] (host) -> audio [B][frames*hop]. */
int pb200_vocode(pb200_voice* v, const float* z, int32_t B, int64_t frames, const float** audio,
                 double* infer_seconds);

/* The reference's streaming split (src/python/piper_train/export_onnx_streaming.py:19-69):
 *   pb200_encode = VitsEncoder.forward  (text encoder, duration predictor, length regulator, prior sample)
 *                  ids -> z_p fp32 [inter][frames] (engine-owned host memory, valid until the next call)
 *   pb200_decode = VitsDecoder.forward  (flow reverse + generator) on z_p [B][inter][frames] -> audio [B][frames*hop]
 * The chunk / halo scheduling of infer_onnx_streaming.py:76-108 lives on the host (piper_b200/streaming.py). */
int pb200_encode(pb200_voice* v, const int64_t* ids, int64_t n_ids, const float scales[3], const pb200_noise* noise,
                 const float** z_p, int64_t* frames, double* infer_seconds);
int pb200_decode(pb200_voice* v, const float* z_p, int32_t B, int64_t frames, const float** audio,
                 double* infer_seconds);

/* Device-resident timing: stage inputs in HBM once, then run the kernels (no host<->device traffic except
 * the B-int output-length read-back the graph's data-dependent shape requires). */
int pb200_stage(pb200_voice* v, const int64_t* ids_concat, const int64_t* lens, int32_t B, const float scales[3],
                const pb200_noise* noise, const int32_t* w_ceil_override);
int pb200_run_staged(pb200_voice* v, int64_t* total_samples, float* device_ms);
/* enc, duration predictor, host length round-trip, expand+flow, generator — CUDA-event ms of the last run */
int pb200_stage_times(const pb200_voice* v, float ms[5]);

/* Per-launch CUDA-event timing of the convolution kernels of the last run, aggregated by pipeline stage,
 * as JSON {"stage": {"launches", "ms", "bytes", "flops"}} with the algorithmic bytes/flops of SURVEY §8d. */
int pb200_set_profile(pb200_voice* v, int32_t on);
int pb200_profile_read(pb200_voice* v, char* buf, int64_t cap);
/* Same records un-aggregated: a JSON array with one entry per conv launch of the last call, in launch order
 * (tag, tensor-core flag, microseconds, layer shape, algorithmic bytes / FLOP).  Fails if cap is too small. */
int pb200_profile_read_launches(pb200_voice* v, char* buf, int64_t cap);

/* Select which layer families run on the tcgen05 tensor cores (split precision, fp16x3 by default): bit 0 = generator,
 * bit 1 = flow, bit 2 = text encoder, bit 3 = duration predictor, bit 4 = the generator's MRF stages fused into one
 * launch each; cleared bits use the fp32 CUDA-core kernel.  Default 31.  The tensor core truncates (RZ) when adding into
 * its fp32 accumulator; the long reductions of the flow, encoder and duration predictor therefore run in 2 K-chains,
 * each with its own correction accumulator, combined in fp32 RN in the epilogue, which keeps fp32-grade accuracy on the
 * ill-conditioned real test voice (DESIGN.md §3).  Env PIPER_B200_MMA=<mask> sets the default at load. */
int pb200_set_mma(pb200_voice* v, int32_t mask);
/* Kernel-level test hook: one Conv1d (same-padded, pad = dil*(k-1)/2) on host arrays through the chosen back end:
 * 0 = CUDA-core kernel; tensor cores 1 (or 3) = bf16x3, 2 (or 4) = tf32x3 with 2 K-chains, 5 = fp16x3 with 1 chain,
 * 6 = fp16x3 with 2 chains.  Any other value is an error.  x [B][ci][L], w [co][ci][k], bias [co] or NULL, pre_slope != 0 applies
 * leaky-relu to the input, resid [B][co][L] or NULL is added, y [B][co][L]. */
int pb200_debug_conv1d(int32_t backend, const float* x, int32_t B, int32_t ci, int32_t L, const float* w,
                       const float* bias, int32_t co, int32_t k, int32_t dil, float pre_slope, const float* resid,
                       float* y);

/* Kernel-level test hook: ONE conv launch with any fused epilogue, on a ragged batch, through back end `backend` (numbered
 * as above), packed and launched the way the engine launches a layer.  The descriptor (the field order of the CPU model's
 * conv2_sim_run in tests/sim/conv2_sim.cpp, without its plan fields):
 *   desc = {ci, rows, k, dil, pad, q_extra, pre (0 none / 1 leaky-relu with `slope`), epi (kernels.cuh Epilogue), split,
 *           first, up, up_pad, mrf, mrf_n, len_scale, cs_x, cs_y, cs_y2, cs_r, C_y, C_y2, C_r, flags}
 * x has ci channels, y / y2 / r have C_y / C_y2 / C_r channels; cs_* are the row pitches in floats (multiples of 4).
 * Item-major layout [B][C][cs], or with PB200_CONV_FLAT the engine's flat layout [C][B][cs] (item b at column b * cs of
 * every channel row; the tensor-core kernel then tiles the concatenated time axis where the engine would).  Item b is
 * valid on [0, len[b] * len_scale).  w [rows][ci][k] (a ConvTranspose already lowered to rows = C_out * up stride-phase
 * rows), bias [rows] or NULL, bias_item [B][bias_item_stride] (per-item rows added to the bias) or NULL.  y, y2 and r are
 * uploaded whole and y, y2 copied back whole, so a caller can prefill them and see every store; pass NULL for a buffer the
 * epilogue does not use.  PB200_CONV_Y_IS_R: the launch reads r from y and writes it in place (WN, SUBFROM; r unused).
 * PB200_CONV_LATENCY: the latency plan of the tensor-core kernel (two K-chains).  A launch the engine never makes
 * (odd rows for GATE, rows not a multiple of up, a shape the tensor-core plan declines, ...) is an error. */
#define PB200_CONV_DESC_LEN 23
enum { PB200_CONV_Y_IS_R = 1, PB200_CONV_FLAT = 2, PB200_CONV_LATENCY = 4 };
int pb200_debug_conv(int32_t backend, const int32_t desc[PB200_CONV_DESC_LEN], float slope, const float* x, const float* w,
                     const float* bias, const float* bias_item, int32_t bias_item_stride, const int32_t* len, int32_t B,
                     float* y, float* y2, const float* r);

/* Host-only (no GPU): tiling and packed weights of the fused MRF stage (csrc/mrf_fused.cu, engine mask bit 16) for
 * upsample stage `stage` of a voice; fuse_post != 0 plans it with conv_post + tanh fused behind it.
 * plan = {ok, n_chains, n_steps, pair, hv, to, k[3], dil[3][6], post_k}; w = bf16 tap tiles in consumption order,
 * bias = [step][chain][32].  w / bias may be NULL to query sizes. */
int pb200_debug_mrf_pack(const char* onnx_path, int32_t stage, int32_t fuse_post, int32_t plan[32], uint8_t* w,
                         int64_t* w_bytes, float* bias, int64_t* n_bias);

void pb200_release(pb200_voice* v, const void* audio);

/* Speaker ids for the following batch / staged / decode calls on this voice: item b uses sids[min(b, n-1)]
 * (n = 0 resets to speaker 0).  Single-speaker voices ignore it. */
int pb200_set_speakers(pb200_voice* v, const int64_t* sids, int32_t n);

/* Test taps: when debug is on, intermediate tensors of the last call are kept on the host.
 * names: x, stats, logw, cum, z_p, z, up<i>, stage<i>, audio.  Copies item b as [C][len] into buf. */
int pb200_set_debug(pb200_voice* v, int32_t on);
int pb200_tap_shape(const pb200_voice* v, const char* name, int32_t b, int32_t* channels, int32_t* len);
int pb200_tap_read(const pb200_voice* v, const char* name, int32_t b, float* buf, int64_t cap_floats);

uint64_t pb200_launch_count(void);
const char* pb200_last_error(void);
const char* pb200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PIPER_B200_H_ */
