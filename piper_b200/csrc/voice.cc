#include "voice.h"

#include <cmath>
#include <cstring>
#include <map>
#include <regex>
#include <set>
#include <sstream>
#include <stdexcept>

#include "onnx_reader.h"

namespace pb200 {
namespace {

struct Attr {
  int k = 1, dil = 1, stride = 1, pad = 0, groups = 1;
};

struct Canon {
  std::map<std::string, const OnnxTensor*> w;
  std::map<std::string, Attr> attr;
  float ea_exp_neg_logs[2] = {1.f, 1.f};
  bool have_ea_scale = false;
};

[[noreturn]] void fail(const std::string& msg) { throw std::runtime_error("voice loader: " + msg); }

bool starts_with(const std::string& s, const char* p) { return s.rfind(p, 0) == 0; }
bool ends_with(const std::string& s, const std::string& p) {
  return s.size() >= p.size() && s.compare(s.size() - p.size(), p.size(), p) == 0;
}

void canonicalize(const OnnxModel& m, Canon& c) {
  std::set<std::string> anonymous;
  for (const auto& n : m.nodes) {
    if ((n.op_type != "Conv" && n.op_type != "ConvTranspose") || n.inputs.size() < 2) continue;
    const OnnxTensor* wt = m.find(n.inputs[1]);
    if (!wt) continue;
    std::string name = n.inputs[1];
    if (starts_with(name, "onnx::") && n.inputs.size() >= 3 && ends_with(n.inputs[2], ".bias")) {
      anonymous.insert(name);
      name = n.inputs[2].substr(0, n.inputs[2].size() - 5) + ".weight";
    }
    Attr a;
    a.k = int(n.attr("kernel_shape", wt->dims.empty() ? 1 : wt->dims.back()));
    a.dil = int(n.attr("dilations", 1));
    a.stride = int(n.attr("strides", 1));
    a.pad = int(n.attr("pads", 0));
    a.groups = int(n.attr("group", 1));
    c.attr[name] = a;
    c.w[name] = wt;
  }
  for (const auto& t : m.initializers) {
    if (t.dtype != 1 || starts_with(t.name, "onnx::") || anonymous.count(t.name)) continue;
    c.w.emplace(t.name, &t);
  }
  if (!c.w.count("enc_p.emb.weight")) {
    const OnnxTensor* sid = m.find("sid");
    if (sid && sid->dims.size() == 2 && sid->dtype == 1) {
      c.w["enc_p.emb.weight"] = sid;
      c.w.erase("sid");
    } else {
      fail("embedding table not found (neither enc_p.emb.weight nor a 2-D `sid` initializer)");
    }
  }
  if (const auto it = c.w.find("dp.flows.0.logs"); it != c.w.end()) {
    for (int i = 0; i < 2; ++i) c.ea_exp_neg_logs[i] = std::exp(-it->second->f32()[i]);
    c.have_ea_scale = true;
  } else {
    std::set<std::string> sub_out;
    for (const auto& n : m.nodes)
      if (n.op_type == "Sub")
        for (const auto& in : n.inputs)
          if (in == "dp.flows.0.m") sub_out.insert(n.outputs.at(0));
    for (const auto& n : m.nodes) {
      if (n.op_type != "Mul") continue;
      bool consumes = false;
      for (const auto& in : n.inputs) consumes |= sub_out.count(in) > 0;
      if (!consumes) continue;
      for (const auto& in : n.inputs) {
        const OnnxTensor* t = m.find(in);
        if (t && t->dtype == 1 && t->numel() == 2) {
          c.ea_exp_neg_logs[0] = t->f32()[0];
          c.ea_exp_neg_logs[1] = t->f32()[1];
          c.have_ea_scale = true;
        }
      }
    }
    if (!c.have_ea_scale) fail("dp.flows.0: exp(-logs) constant not found after Sub(., dp.flows.0.m)");
  }
}

struct Packer {
  const Canon& c;
  PackedVoice& v;
  Packer(const Canon& c_, PackedVoice& v_) : c(c_), v(v_) {}

  const OnnxTensor& get(const std::string& name, size_t rank) const {
    auto it = c.w.find(name);
    if (it == c.w.end()) fail("missing tensor '" + name + "'");
    if (it->second->dims.size() != rank)
      fail("tensor '" + name + "' has rank " + std::to_string(it->second->dims.size()) + ", expected " +
           std::to_string(rank));
    return *it->second;
  }
  bool has(const std::string& name) const { return c.w.count(name) > 0; }
  Attr attr(const std::string& wname) const {
    auto it = c.attr.find(wname);
    if (it == c.attr.end()) fail("no Conv node references '" + wname + "'");
    return it->second;
  }

  int64_t alloc(int64_t n) {  // 256-byte aligned sections
    int64_t off = (int64_t(v.blob.size()) + 63) / 64 * 64;
    v.blob.resize(size_t(off + n), 0.f);
    return off;
  }
  int64_t put(const OnnxTensor& t) {
    int64_t off = alloc(t.numel());
    std::memcpy(&v.blob[size_t(off)], t.f32(), size_t(t.numel()) * 4);
    v.n_params += t.numel();
    return off;
  }
  int64_t put_named(const std::string& name, size_t rank) { return put(get(name, rank)); }

  enum Perm { kPlain, kGate, kRevCi, kRevCo };

  // Conv1d weight [Co][Ci][K] (+ bias [Co]) -> [Ci][K][RowsP]
  ConvW conv(const std::string& prefix, Perm perm = kPlain, int want_ci = -1, int want_co = -1) {
    const OnnxTensor& w = get(prefix + ".weight", 3);
    Attr a = attr(prefix + ".weight");
    if (a.groups != 1) fail("'" + prefix + "': grouped conv in a dense slot");
    if (a.stride != 1) fail("'" + prefix + "': strided Conv1d is not part of the VITS graph");
    const int co = int(w.dims[0]), ci = int(w.dims[1]), k = int(w.dims[2]);
    if (want_ci >= 0 && ci != want_ci) fail("'" + prefix + "': C_in " + std::to_string(ci) + " != " + std::to_string(want_ci));
    if (want_co >= 0 && co != want_co) fail("'" + prefix + "': C_out " + std::to_string(co) + " != " + std::to_string(want_co));
    if (perm == kGate && (co % 2)) fail("'" + prefix + "': gated conv needs even C_out");
    ConvW r;
    r.ci = ci; r.rows = co; r.rows_p = (co + 3) / 4 * 4; r.k = k; r.dil = a.dil; r.pad = a.pad;
    r.w = alloc(int64_t(ci) * k * r.rows_p);
    const float* src = w.f32();
    auto row_src = [&](int row) {  // packed row -> source output channel
      switch (perm) {
        case kGate: return (row & 1) ? co / 2 + row / 2 : row / 2;
        case kRevCo: return co - 1 - row;
        default: return row;
      }
    };
    for (int i = 0; i < ci; ++i) {
      const int si = perm == kRevCi ? ci - 1 - i : i;
      for (int j = 0; j < k; ++j) {
        float* dst = &v.blob[size_t(r.w + (int64_t(i) * k + j) * r.rows_p)];
        for (int row = 0; row < co; ++row) dst[row] = src[(int64_t(row_src(row)) * ci + si) * k + j];
      }
    }
    v.n_params += w.numel();
    if (has(prefix + ".bias")) {
      const OnnxTensor& b = get(prefix + ".bias", 1);
      if (b.dims[0] != co) fail("'" + prefix + ".bias' size mismatch");
      r.b = alloc(co);
      for (int row = 0; row < co; ++row) v.blob[size_t(r.b + row)] = b.f32()[row_src(row)];
      v.n_params += co;
    }
    return r;
  }

  // ConvTranspose1d weight [Ci][Co][k], stride s, pad p with k = m*s, k - 2p = s  =>  L_out = s*L_in and
  // out[co, q*s + phi - p] = b[co] + sum_ci sum_{j<m} x[ci, q-(m-1)+j] * W[ci, co, phi + (m-1-j)*s]
  ConvW conv_transpose(const std::string& prefix) {
    const OnnxTensor& w = get(prefix + ".weight", 3);
    Attr a = attr(prefix + ".weight");
    const int ci = int(w.dims[0]), co = int(w.dims[1]), k = int(w.dims[2]), s = a.stride, p = a.pad;
    if (s < 1 || k % s != 0 || k - 2 * p != s || a.dil != 1 || a.groups != 1)
      fail("'" + prefix + "': ConvTranspose1d (k=" + std::to_string(k) + ", s=" + std::to_string(s) + ", p=" +
           std::to_string(p) + ") is outside the supported family k = m*s, k - 2p = s");
    const int m = k / s;
    ConvW r;
    r.ci = ci; r.rows = co * s; r.rows_p = (r.rows + 3) / 4 * 4; r.k = m; r.dil = 1; r.pad = m - 1;
    r.up = s; r.up_pad = p;
    r.w = alloc(int64_t(ci) * m * r.rows_p);
    const float* src = w.f32();
    for (int i = 0; i < ci; ++i)
      for (int j = 0; j < m; ++j) {
        float* dst = &v.blob[size_t(r.w + (int64_t(i) * m + j) * r.rows_p)];
        for (int c2 = 0; c2 < co; ++c2)
          for (int phi = 0; phi < s; ++phi) dst[c2 * s + phi] = src[(int64_t(i) * co + c2) * k + phi + (m - 1 - j) * s];
      }
    v.n_params += w.numel();
    if (has(prefix + ".bias")) {
      const OnnxTensor& b = get(prefix + ".bias", 1);
      r.b = alloc(r.rows);
      for (int row = 0; row < r.rows; ++row) v.blob[size_t(r.b + row)] = b.f32()[row / s];
      v.n_params += co;
    }
    return r;
  }

  LayerNormW ln(const std::string& prefix, int c_expected) {
    LayerNormW r;
    const OnnxTensor& g = get(prefix + ".gamma", 1);
    if (g.dims[0] != c_expected) fail("'" + prefix + "': LayerNorm width mismatch");
    r.c = c_expected;
    r.gamma = put(g);
    r.beta = put_named(prefix + ".beta", 1);
    return r;
  }

  DDSW dds(const std::string& prefix, int C, int n_layers) {
    DDSW d;
    for (int i = 0; i < n_layers; ++i) {
      DDSLayerW l;
      const std::string sep = prefix + ".convs_sep." + std::to_string(i);
      const OnnxTensor& w = get(sep + ".weight", 3);
      Attr a = attr(sep + ".weight");
      if (w.dims[0] != C || w.dims[1] != 1 || a.groups != C) fail("'" + sep + "': expected depthwise conv over " + std::to_string(C) + " channels");
      l.k = int(w.dims[2]);
      l.dil = a.dil;
      if (a.pad * 2 != a.dil * (l.k - 1)) fail("'" + sep + "': depthwise conv is not same-padded");
      l.sep_w = put(w);
      l.sep_b = put_named(sep + ".bias", 1);
      l.pw = conv(prefix + ".convs_1x1." + std::to_string(i), kPlain, C, C);
      l.n1 = ln(prefix + ".norms_1." + std::to_string(i), C);
      l.n2 = ln(prefix + ".norms_2." + std::to_string(i), C);
      d.layers.push_back(l);
    }
    return d;
  }
};

std::vector<int> indices(const Canon& c, const std::string& pattern) {
  std::regex rx(pattern);
  std::set<int> s;
  std::smatch m;
  for (const auto& kv : c.w)
    if (std::regex_match(kv.first, m, rx)) s.insert(std::stoi(m[1].str()));
  return std::vector<int>(s.begin(), s.end());
}

}  // namespace

void load_voice_file(const std::string& onnx_path, PackedVoice& v) {
  OnnxModel m;
  load_onnx(onnx_path, m);
  Canon c;
  canonicalize(m, c);
  Packer P(c, v);
  VoiceSpec& s = v.spec;

  // ---- hyper-parameters from shapes (SURVEY.md App. B.3)
  const OnnxTensor& emb = P.get("enc_p.emb.weight", 2);
  s.n_vocab = int(emb.dims[0]);
  s.hidden = int(emb.dims[1]);
  const OnnxTensor& relk = P.get("enc_p.encoder.attn_layers.0.emb_rel_k", 3);
  if (relk.dims[0] != 1) fail("per-head relative embeddings (heads_share=False) are not supported");
  const int dk = int(relk.dims[2]);
  if (dk <= 0 || s.hidden % dk) fail("emb_rel_k width does not divide hidden size");
  s.n_heads = s.hidden / dk;
  s.window = (int(relk.dims[1]) - 1) / 2;
  s.n_layers = int(indices(c, R"(enc_p\.encoder\.attn_layers\.(\d+)\.conv_q\.weight)").size());
  const OnnxTensor& f1 = P.get("enc_p.encoder.ffn_layers.0.conv_1.weight", 3);
  s.filter = int(f1.dims[0]);
  s.ffn_kernel = int(f1.dims[2]);
  s.inter = int(P.get("enc_p.proj.weight", 3).dims[0]) / 2;
  s.dds_layers = int(indices(c, R"(dp\.convs\.convs_sep\.(\d+)\.weight)").size());
  {
    auto cf = indices(c, R"(dp\.flows\.(\d+)\.pre\.weight)");
    if (cf.empty()) fail("no ConvFlow in the duration predictor (deterministic DurationPredictor voices are not supported)");
    // SynthesizerTrn's reverse pass drops self.flows[1], the first ConvFlow after the ElementwiseAffine ("remove a useless
    // vflow", models.py:110: flows[:-2] + [flows[-1]] of the reversed list).  The stock exporter prunes its weights from
    // the file; an exporter that keeps initializers must not make us run it.
    if (cf.size() > 1 && cf.front() == 1) cf.erase(cf.begin());
    s.dp_flows.assign(cf.rbegin(), cf.rend());
    s.spline_bins = (int(P.get("dp.flows." + std::to_string(cf[0]) + ".proj.weight", 3).dims[0]) + 1) / 3;
    auto fl = indices(c, R"(flow\.flows\.(\d+)\.pre\.weight)");
    if (fl.empty()) fail("no coupling layers found");
    s.flow_layers.assign(fl.rbegin(), fl.rend());
    const std::string f0 = "flow.flows." + std::to_string(fl[0]) + ".enc.in_layers.";
    s.wn_layers = int(indices(c, "flow\\.flows\\." + std::to_string(fl[0]) + R"(\.enc\.in_layers\.(\d+)\.weight)").size());
    s.wn_kernel = int(P.get(f0 + "0.weight", 3).dims[2]);
    s.wn_dilation_rate = s.wn_layers > 1 ? P.attr(f0 + "1.weight").dil : 1;
  }
  const int H = s.hidden, I = s.inter;
  if (I % 2) fail("inter_channels must be even");
  if (P.has("emb_g.weight")) {
    const OnnxTensor& eg = P.get("emb_g.weight", 2);
    s.n_speakers = int(eg.dims[0]);
    s.gin = int(eg.dims[1]);
  }

  // ---- text encoder
  v.emb = P.put(emb);
  for (int l = 0; l < s.n_layers; ++l) {
    EncLayerW e;
    const std::string a = "enc_p.encoder.attn_layers." + std::to_string(l);
    e.rel_k = P.put_named(a + ".emb_rel_k", 3);
    e.rel_v = P.put_named(a + ".emb_rel_v", 3);
    // fused q|k|v projection: three [H][H][1] convs stacked on the row axis
    ConvW q = P.conv(a + ".conv_q", Packer::kPlain, H, H), k = P.conv(a + ".conv_k", Packer::kPlain, H, H),
          vv = P.conv(a + ".conv_v", Packer::kPlain, H, H);
    if (q.k != 1 || q.rows_p != H) fail("attention projections must be 1x1 with H % 4 == 0");
    e.qkv = q;
    e.qkv.rows = e.qkv.rows_p = 3 * H;
    e.qkv.w = P.alloc(int64_t(H) * 3 * H);
    e.qkv.b = P.alloc(3 * H);
    const ConvW* parts[3] = {&q, &k, &vv};
    for (int i = 0; i < H; ++i)
      for (int pidx = 0; pidx < 3; ++pidx)
        std::memcpy(&v.blob[size_t(e.qkv.w + int64_t(i) * 3 * H + pidx * H)],
                    &v.blob[size_t(parts[pidx]->w + int64_t(i) * H)], size_t(H) * 4);
    for (int pidx = 0; pidx < 3; ++pidx) {
      if (parts[pidx]->b < 0) fail("attention projection without bias");
      std::memcpy(&v.blob[size_t(e.qkv.b + pidx * H)], &v.blob[size_t(parts[pidx]->b)], size_t(H) * 4);
    }
    e.o = P.conv(a + ".conv_o", Packer::kPlain, H, H);
    const std::string f = "enc_p.encoder.ffn_layers." + std::to_string(l);
    e.ffn1 = P.conv(f + ".conv_1", Packer::kPlain, H, s.filter);
    e.ffn2 = P.conv(f + ".conv_2", Packer::kPlain, s.filter, H);
    // FFN pads (k-1)/2 left, k/2 right with explicit Pad nodes (attentions.py:419-427); Conv pads are 0
    e.ffn1.pad = (e.ffn1.k - 1) / 2;
    e.ffn2.pad = (e.ffn2.k - 1) / 2;
    e.ln1 = P.ln("enc_p.encoder.norm_layers_1." + std::to_string(l), H);
    e.ln2 = P.ln("enc_p.encoder.norm_layers_2." + std::to_string(l), H);
    v.enc.push_back(e);
  }
  v.enc_proj = P.conv("enc_p.proj", Packer::kPlain, H, 2 * I);

  // ---- stochastic duration predictor (reverse)
  v.dp_pre = P.conv("dp.pre", Packer::kPlain, H, H);
  v.dp_proj = P.conv("dp.proj", Packer::kPlain, H, H);
  v.dp_dds = P.dds("dp.convs", H, s.dds_layers);
  for (int f : s.dp_flows) {
    ConvFlowW cf;
    const std::string p = "dp.flows." + std::to_string(f);
    const OnnxTensor& pw = P.get(p + ".pre.weight", 3);
    if (pw.dims[0] != H || pw.dims[1] != 1 || pw.dims[2] != 1) fail("'" + p + ".pre': expected 1 -> H pointwise conv");
    cf.pre_w = P.put(pw);
    cf.pre_b = P.put_named(p + ".pre.bias", 1);
    cf.dds = P.dds(p + ".convs", H, s.dds_layers);
    cf.proj = P.conv(p + ".proj", Packer::kPlain, H, 3 * s.spline_bins - 1);
    v.dp_flows.push_back(cf);
  }
  {
    const OnnxTensor& m0 = P.get("dp.flows.0.m", 2);
    v.ea_m[0] = m0.f32()[0];
    v.ea_m[1] = m0.f32()[1];
    v.ea_scale[0] = c.ea_exp_neg_logs[0];
    v.ea_scale[1] = c.ea_exp_neg_logs[1];
    v.n_params += 4;
  }

  // ---- flow (reverse): Flip, RCL_a, Flip, RCL_b, ... ; the flip is folded into pre/post weights
  bool flipped = false;
  for (int f : s.flow_layers) {
    flipped = !flipped;
    CouplingW cw;
    cw.flipped = flipped;
    const std::string p = "flow.flows." + std::to_string(f);
    cw.pre = P.conv(p + ".pre", flipped ? Packer::kRevCi : Packer::kPlain, I / 2, H);
    for (int i = 0; i < s.wn_layers; ++i) {
      ConvW in = P.conv(p + ".enc.in_layers." + std::to_string(i), Packer::kGate, H, 2 * H);
      if (in.pad * 2 != in.dil * (in.k - 1)) fail("WN in_layer is not same-padded");
      cw.in_layers.push_back(in);
      cw.res_skip.push_back(P.conv(p + ".enc.res_skip_layers." + std::to_string(i), Packer::kPlain, H,
                                   i < s.wn_layers - 1 ? 2 * H : H));
    }
    if (int(P.get(p + ".post.weight", 3).dims[0]) != I / 2) fail("'" + p + ".post': only mean-only couplings are supported");
    cw.post = P.conv(p + ".post", flipped ? Packer::kRevCo : Packer::kPlain, H, I / 2);
    v.flow.push_back(cw);
  }
  if (flipped) fail("odd number of coupling layers leaves the latent channel-reversed (unsupported)");

  // ---- generator
  v.dec_pre = P.conv("dec.conv_pre", Packer::kPlain, I, -1);
  s.up_initial = v.dec_pre.rows;
  auto ups = indices(c, R"(dec\.ups\.(\d+)\.weight)");
  if (ups.empty()) fail("generator has no upsampling stages");
  s.resblock = 2;
  for (const auto& kv : c.w)
    if (starts_with(kv.first, "dec.resblocks.0.convs1.")) s.resblock = 1;
  const int n_rb = int(indices(c, R"(dec\.resblocks\.(\d+)\..*)").size());
  if (n_rb % int(ups.size())) fail("resblock count is not a multiple of the upsample count");
  const int nk = n_rb / int(ups.size());
  int ch = s.up_initial;
  s.hop = 1;
  for (size_t i = 0; i < ups.size(); ++i) {
    ConvW u = P.conv_transpose("dec.ups." + std::to_string(ups[i]));
    if (u.ci != ch) fail("dec.ups." + std::to_string(i) + ": channel chain broken");
    ch = u.rows / u.up;
    s.up_rates.push_back(u.up);
    s.up_kernels.push_back(u.k * u.up);
    s.up_pads.push_back(u.up_pad);
    s.hop *= u.up;
    v.ups.push_back(u);
    std::vector<ResBlockW> stage;
    for (int j = 0; j < nk; ++j) {
      ResBlockW rb;
      const std::string r = "dec.resblocks." + std::to_string(int(i) * nk + j);
      const std::string first = s.resblock == 1 ? ".convs1." : ".convs.";
      auto ids = indices(c, "dec\\.resblocks\\." + std::to_string(int(i) * nk + j) +
                                (s.resblock == 1 ? R"(\.convs1\.(\d+)\.weight)" : R"(\.convs\.(\d+)\.weight)"));
      std::vector<int> dils;
      for (int id : ids) {
        ConvW c1 = P.conv(r + first + std::to_string(id), Packer::kPlain, ch, ch);
        if (c1.pad * 2 != c1.dil * (c1.k - 1)) fail("'" + r + "': resblock conv is not same-padded");
        rb.k = c1.k;
        dils.push_back(c1.dil);
        rb.c1.push_back(c1);
        if (s.resblock == 1) {
          ConvW c2 = P.conv(r + ".convs2." + std::to_string(id), Packer::kPlain, ch, ch);
          if (c2.pad * 2 != c2.dil * (c2.k - 1)) fail("'" + r + "': resblock conv is not same-padded");
          rb.c2.push_back(c2);
        }
      }
      if (i == 0) {
        s.rb_kernels.push_back(rb.k);
        s.rb_dilations.push_back(dils);
      }
      stage.push_back(rb);
    }
    v.resblocks.push_back(stage);
  }
  {
    const OnnxTensor& pw = P.get("dec.conv_post.weight", 3);
    if (pw.dims[0] != 1 || pw.dims[1] != ch) fail("dec.conv_post: expected [1][C][k]");
    if (P.has("dec.conv_post.bias")) fail("dec.conv_post with a bias is not part of the piper generator");
    Attr a = P.attr("dec.conv_post.weight");
    v.post_c = ch;
    v.post_k = int(pw.dims[2]);
    if (a.pad * 2 != v.post_k - 1 || a.dil != 1) fail("dec.conv_post is not same-padded");
    v.post_w = P.put(pw);
  }
  // ---- speaker conditioning matrix (multi-speaker voices)
  if (s.gin > 0) {
    v.emb_g = P.put_named("emb_g.weight", 2);
    std::vector<const OnnxTensor*> ws, bs;
    std::vector<int> perm_layers;   // > 0: rows are n WN layers of 2H rows each, to be gate-interleaved
    auto add = [&](const std::string& prefix, int expect_rows, int wn_layers_of) {
      const OnnxTensor& w = P.get(prefix + ".weight", 3);
      if (w.dims[0] != expect_rows || w.dims[1] != s.gin || w.dims[2] != 1)
        fail("'" + prefix + "': expected a " + std::to_string(expect_rows) + " x gin pointwise conditioning conv");
      ws.push_back(&w);
      bs.push_back(&P.get(prefix + ".bias", 1));
      perm_layers.push_back(wn_layers_of);
      const int row = v.cond_rows;
      v.cond_rows += expect_rows;
      return row;
    };
    v.dp_cond_row = add("dp.cond", H, 0);
    for (size_t ci = 0; ci < v.flow.size(); ++ci)
      v.flow[ci].cond_row = add("flow.flows." + std::to_string(s.flow_layers[ci]) + ".enc.cond_layer", 2 * H * s.wn_layers, s.wn_layers);
    v.dec_cond_row = add("dec.cond", s.up_initial, 0);
    v.cond_w = P.alloc(int64_t(v.cond_rows) * s.gin);
    v.cond_b = P.alloc(v.cond_rows);
    int row = 0;
    for (size_t t = 0; t < ws.size(); ++t) {
      const int rows = int(ws[t]->dims[0]);
      for (int r = 0; r < rows; ++r) {
        int src = r;
        if (perm_layers[t] > 0) {           // (tanh_j, sigmoid_j) interleave inside each layer's 2H rows
          const int layer = r / (2 * H), in = r % (2 * H);
          src = layer * 2 * H + ((in & 1) ? H + in / 2 : in / 2);
        }
        std::memcpy(&v.blob[size_t(v.cond_w + int64_t(row + r) * s.gin)], ws[t]->f32() + size_t(src) * s.gin, size_t(s.gin) * 4);
        v.blob[size_t(v.cond_b + row + r)] = bs[t]->f32()[src];
      }
      row += rows;
      v.n_params += ws[t]->numel() + rows;
    }
  }

  // pad the tail so 16-byte vector loads of the last rows never leave the allocation
  v.blob.resize((v.blob.size() + 63) / 64 * 64 + 64, 0.f);
}

namespace {
void jlist(std::ostringstream& o, const std::vector<int>& v) {
  o << "[";
  for (size_t i = 0; i < v.size(); ++i) o << (i ? "," : "") << v[i];
  o << "]";
}
void jconv(std::ostringstream& o, const char* name, const ConvW& c) {
  o << "\"" << name << "\":{\"w\":" << c.w << ",\"b\":" << c.b << ",\"ci\":" << c.ci << ",\"rows\":" << c.rows
    << ",\"rows_p\":" << c.rows_p << ",\"k\":" << c.k << ",\"dil\":" << c.dil << ",\"pad\":" << c.pad
    << ",\"up\":" << c.up << ",\"up_pad\":" << c.up_pad << "}";
}
}  // namespace

std::string describe_voice(const PackedVoice& v) {
  const VoiceSpec& s = v.spec;
  std::ostringstream o;
  o << "{\"n_vocab\":" << s.n_vocab << ",\"hidden\":" << s.hidden << ",\"inter\":" << s.inter << ",\"filter\":" << s.filter
    << ",\"n_heads\":" << s.n_heads << ",\"n_layers\":" << s.n_layers << ",\"window\":" << s.window
    << ",\"ffn_kernel\":" << s.ffn_kernel << ",\"dds_layers\":" << s.dds_layers << ",\"spline_bins\":" << s.spline_bins
    << ",\"wn_layers\":" << s.wn_layers << ",\"wn_kernel\":" << s.wn_kernel << ",\"wn_dilation_rate\":" << s.wn_dilation_rate
    << ",\"n_speakers\":" << s.n_speakers << ",\"gin\":" << s.gin << ",\"cond_rows\":" << v.cond_rows << ",\"resblock\":" << s.resblock << ",\"up_initial\":" << s.up_initial << ",\"hop\":" << s.hop << ",\"dp_flows\":";
  jlist(o, s.dp_flows);
  o << ",\"flow_layers\":";
  jlist(o, s.flow_layers);
  o << ",\"up_rates\":";
  jlist(o, s.up_rates);
  o << ",\"up_kernels\":";
  jlist(o, s.up_kernels);
  o << ",\"up_pads\":";
  jlist(o, s.up_pads);
  o << ",\"rb_kernels\":";
  jlist(o, s.rb_kernels);
  o << ",\"rb_dilations\":[";
  for (size_t i = 0; i < s.rb_dilations.size(); ++i) {
    o << (i ? "," : "");
    jlist(o, s.rb_dilations[i]);
  }
  o << "],\"n_params\":" << v.n_params << ",\"blob_floats\":" << v.blob.size() << ",\"ea_m\":[" << v.ea_m[0] << ","
    << v.ea_m[1] << "],\"ea_scale\":[" << v.ea_scale[0] << "," << v.ea_scale[1] << "],\"layers\":{";
  o << "\"emb\":" << v.emb << ",";
  jconv(o, "enc0_qkv", v.enc.at(0).qkv); o << ",";
  jconv(o, "enc0_ffn1", v.enc.at(0).ffn1); o << ",";
  jconv(o, "enc_proj", v.enc_proj); o << ",";
  jconv(o, "flow0_pre", v.flow.at(0).pre); o << ",";
  jconv(o, "flow0_in0", v.flow.at(0).in_layers.at(0)); o << ",";
  jconv(o, "flow0_post", v.flow.at(0).post); o << ",";
  jconv(o, "flow1_pre", v.flow.at(1).pre); o << ",";
  jconv(o, "dec_pre", v.dec_pre); o << ",";
  jconv(o, "up0", v.ups.at(0)); o << ",";
  jconv(o, "rb0_c0", v.resblocks.at(0).at(0).c1.at(0));
  o << ",\"post_w\":" << v.post_w << "}}";
  return o.str();
}

}  // namespace pb200
