// Voice = one piper `.onnx` file turned into (a) inferred hyper-parameters and (b) one packed
// fp32 weight blob laid out for the sm_100a kernels, plus a table of where each layer lives.
//
// Replaces what `loadModel` delegates to Ort::Session
// (/root/reference/src/cpp/piper.cpp:262-306).  Hyper-parameters are not in the voice JSON; they
// are inferred from initializer shapes and Conv attributes (SURVEY.md App. B.3).  Naming traps of
// the reference exporter handled here (export_onnx.py:51-101): the embedding table is called `sid`,
// weight-normed flow convs are anonymous `onnx::Conv_*` (recovered through the bias name), and
// `dp.flows.0.logs` survives only as exp(-logs) in an anonymous [2,1] Mul operand.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

namespace pb200 {

// A Conv1d / ConvTranspose1d lowered to "rows x (Ci*K)" with weights stored [Ci][K][RowsP]
// (row index fastest) so a CTA's row tile is one contiguous, 16B-aligned run per (ci, tap).
struct ConvW {
  int64_t w = -1, b = -1;  // float offsets into the blob; b < 0 => no bias
  int ci = 0, rows = 0, rows_p = 0, k = 1, dil = 1, pad = 0;
  // ConvTranspose lowering: rows = Co * up, output t = q*up + (row % up) - up_pad
  int up = 1, up_pad = 0;
};

struct LayerNormW {
  int64_t gamma = -1, beta = -1;
  int c = 0;
};

struct DDSLayerW {
  int64_t sep_w = -1, sep_b = -1;  // depthwise [C][k], [C]
  int k = 3, dil = 1;
  ConvW pw;                        // 1x1
  LayerNormW n1, n2;
};
struct DDSW { std::vector<DDSLayerW> layers; };

struct EncLayerW {
  ConvW qkv, o, ffn1, ffn2;   // qkv rows = 3H in q,k,v order
  LayerNormW ln1, ln2;
  int64_t rel_k = -1, rel_v = -1;  // [2w+1][dk]
};

struct ConvFlowW {
  int64_t pre_w = -1, pre_b = -1;  // 1 -> H pointwise
  DDSW dds;
  ConvW proj;                      // H -> 3*bins-1
};

struct CouplingW {
  bool flipped = false;  // executes while the channel order is reversed (flip folded into weights)
  ConvW pre, post;
  std::vector<ConvW> in_layers;   // rows interleaved (tanh_i, sigmoid_i) for the gate epilogue
  std::vector<ConvW> res_skip;
  int cond_row = -1;              // first row of this coupling's WN cond_layer in the speaker-conditioning matrix
};

struct ResBlockW {
  int k = 3;
  std::vector<ConvW> c1, c2;  // ResBlock2: only c1 used
};

struct VoiceSpec {
  int n_vocab = 0, hidden = 0, inter = 0, filter = 0, n_heads = 0, n_layers = 0, window = 0, ffn_kernel = 0;
  int dds_layers = 0, spline_bins = 10, wn_layers = 0, wn_kernel = 0, wn_dilation_rate = 1;
  int resblock = 2, up_initial = 0, hop = 1;
  int n_speakers = 1, gin = 0;   // multi-speaker voices: emb_g [n_speakers][gin]
  std::vector<int> dp_flows, flow_layers, up_rates, up_kernels, up_pads, rb_kernels;
  std::vector<std::vector<int>> rb_dilations;
};

struct PackedVoice {
  VoiceSpec spec;
  std::vector<float> blob;
  int64_t emb = -1;
  std::vector<EncLayerW> enc;
  ConvW enc_proj;
  ConvW dp_pre, dp_proj;
  DDSW dp_dds;
  std::vector<ConvFlowW> dp_flows;  // execution order
  float ea_m[2] = {0, 0}, ea_scale[2] = {1, 1};  // (z - m) * exp(-logs)
  std::vector<CouplingW> flow;      // execution order
  ConvW dec_pre;
  std::vector<ConvW> ups;
  std::vector<std::vector<ResBlockW>> resblocks;  // [stage][kernel]
  int64_t post_w = -1;              // conv_post [C][k] (no bias, models.py:342)
  int post_c = 0, post_k = 7;
  // speaker conditioning (models.py:692-696; modules.py:188-197): one [cond_rows][gin] matrix holding dp.cond, every
  // WN cond_layer (rows in the gate-interleaved order of the in_layers) and dec.cond; cond = W * emb_g[sid] + b
  int64_t emb_g = -1, cond_w = -1, cond_b = -1;
  int cond_rows = 0, dp_cond_row = -1, dec_cond_row = -1;
  int64_t n_params = 0;             // fp32 parameters read from the file (before packing/padding)
};

// Parse + canonicalise + pack.  Throws std::runtime_error with a precise message on any
// structural surprise (the loader is topology-driven and refuses what it does not understand).
void load_voice_file(const std::string& onnx_path, PackedVoice& out);

// Human/test-readable description (JSON) of the inferred spec and packed layout.
std::string describe_voice(const PackedVoice& v);

}  // namespace pb200
