// LW-DETR forward engine (host side).  Packs a reference-format checkpoint into kernel-native
// layouts once, then runs a fixed schedule of hand-written sm_100a kernels per batch:
//   patch gather -> [LN, qkv GEMM, fused attention, proj GEMM(+layer-scale+residual), LN, fc1 GEMM(GELU),
//   fc2 GEMM(+layer-scale+residual)] x depth -> projector (1x1 / implicit 3x3 / pixel-shuffle GEMMs,
//   channel LN writing the decoder memory directly) -> two-stage selection (GEMMs, row max, top-k,
//   gathers) -> 3 decoder layers (GEMMs, fused attention, fused deformable gather, LNs) -> heads.
// Reference call stack being replaced: SURVEY.md section 3.2 (lwdetr.py:111-174 and callees).
#include "engine.h"
#include "launch.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstring>

#include "attn.h"
#include "gemm_tc.h"
#include "msda.h"
#include "resize.h"
#include "rowops.h"

namespace lwb {

namespace {
struct Mat {
  void* p;
  int ld;
};
inline char* cptr(void* p) { return static_cast<char*>(p); }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
}  // namespace

// ------------------------------------------------------------------------------- host math helpers
// Bicubic resize, align_corners=False, cubic-convolution kernel with A = -0.75 and border clamping:
// the semantics of F.interpolate(mode="bicubic") used by get_abs_pos (vit.py:44-52).
static void cubic_coeffs(float t, float w[4]) {
  const float A = -0.75f;
  auto c1 = [&](float x) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; };            // |x| <= 1
  auto c2 = [&](float x) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; };      // 1 < |x| < 2
  w[0] = c2(t + 1.f);
  w[1] = c1(t);
  w[2] = c1(1.f - t);
  w[3] = c2(2.f - t);
}
void bicubic_resize_chlast(const float* src, int n_in, int C, int n_out, float* dst) {
  const float scale = static_cast<float>(n_in) / static_cast<float>(n_out);
  std::vector<int> idx(static_cast<size_t>(n_out) * 4);
  std::vector<float> wts(static_cast<size_t>(n_out) * 4);
  for (int o = 0; o < n_out; ++o) {
    const float s = (o + 0.5f) * scale - 0.5f;
    const float f = std::floor(s);
    cubic_coeffs(s - f, &wts[o * 4]);
    for (int k = 0; k < 4; ++k) idx[o * 4 + k] = std::min(std::max(static_cast<int>(f) - 1 + k, 0), n_in - 1);
  }
  for (int oy = 0; oy < n_out; ++oy)
    for (int ox = 0; ox < n_out; ++ox) {
      float* d = dst + (static_cast<size_t>(oy) * n_out + ox) * C;
      for (int c = 0; c < C; ++c) d[c] = 0.f;
      for (int ky = 0; ky < 4; ++ky)
        for (int kx = 0; kx < 4; ++kx) {
          const float w = wts[oy * 4 + ky] * wts[ox * 4 + kx];
          const float* s = src + (static_cast<size_t>(idx[oy * 4 + ky]) * n_in + idx[ox * 4 + kx]) * C;
          for (int c = 0; c < C; ++c) d[c] += w * s[c];
        }
    }
}

// ------------------------------------------------------------------------------- Engine basics
Engine::Engine(const lwdetr_config& cfg, int dtype) : cfg_(cfg), dtype_(dtype) { cudaGetDevice(&device_); }

namespace {
// Switches to the engine's device for the duration of a call (the caller's current device is restored afterwards).
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev); else prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
}  // namespace

void Engine::drop_graphs() {
  for (auto& kv : graphs_) cudaGraphExecDestroy(kv.second);
  graphs_.clear();
}

Engine::~Engine() {
  DeviceGuard guard(device_);
  drop_graphs();
  if (gstream_) cudaStreamDestroy(gstream_);
  if (ev_in_) cudaEventDestroy(ev_in_);
  if (ev_out_) cudaEventDestroy(ev_out_);
  if (warena_.p) cudaFree(warena_.p);
  if (sarena_.p) cudaFree(sarena_.p);
}

void* Engine::walloc(size_t bytes) {
  woff_ = align_up(woff_, 256);
  if (woff_ + bytes > warena_.bytes) return nullptr;
  void* p = cptr(warena_.p) + woff_;
  woff_ += bytes;
  return p;
}
void* Engine::salloc(size_t bytes) {
  soff_ = align_up(soff_, 1024);
  void* p = sarena_.p ? cptr(sarena_.p) + soff_ : nullptr;
  soff_ += bytes;
  return p;
}

std::vector<uint16_t> Engine::to16(const std::vector<float>& v) const {
  std::vector<uint16_t> h(v.size());
  if (dtype_ == DT_BF16) {
    for (size_t i = 0; i < v.size(); ++i) {
      __nv_bfloat16 b = __float2bfloat16_rn(v[i]);
      std::memcpy(&h[i], &b, 2);
    }
  } else {
    for (size_t i = 0; i < v.size(); ++i) {
      __half b = __float2half_rn(v[i]);
      std::memcpy(&h[i], &b, 2);
    }
  }
  return h;
}
void* Engine::upload16(const std::vector<float>& v) {
  void* d = walloc(v.size() * 2);
  if (!d) return nullptr;
  const std::vector<uint16_t> h = to16(v);
  cudaMemcpy(d, h.data(), h.size() * 2, cudaMemcpyHostToDevice);
  return d;
}

int Engine::upload_pos_table(int G, void* dst) {
  const int C = cfg_.vit_dim, T = G * G;
  std::vector<float> raw(static_cast<size_t>(196) * C), grid(static_cast<size_t>(T) * C), wm(static_cast<size_t>(T) * C);
  if (cudaMemcpy(raw.data(), F_.at("pos_raw"), raw.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  bicubic_resize_chlast(raw.data(), 14, C, G, grid.data());
  const int wh = G / 4, wsz = wh * wh;
  for (int r = 0; r < T; ++r) {   // window-major row r -> spatial (y, x)   (vit.py:353-358)
    const int win = r / wsz, t = r % wsz;
    const int y = (win >> 2) * wh + t / wh, x = (win & 3) * wh + t % wh;
    std::memcpy(&wm[static_cast<size_t>(r) * C], &grid[(static_cast<size_t>(y) * G + x) * C], C * sizeof(float));
  }
  const std::vector<uint16_t> h = to16(wm);
  return cudaMemcpy(dst, h.data(), h.size() * 2, cudaMemcpyHostToDevice) == cudaSuccess ? 0 : -1;
}
float* Engine::upload32(const std::vector<float>& v) {
  void* d = walloc(v.size() * 4);
  if (!d) return nullptr;
  cudaMemcpy(d, v.data(), v.size() * 4, cudaMemcpyHostToDevice);
  return static_cast<float*>(d);
}

int Engine::set_option(const char* name, int value) {
  if (std::strcmp(name, "fuse_layernorm") == 0) {
    fuse_ln_ = value;
    drop_graphs();
    planned_B_ = 0;
    return 0;
  }
  if (std::strcmp(name, "cuda_graph") == 0) {
    use_graph_ = value;
    drop_graphs();
    return 0;
  }
  if (std::strcmp(name, "pdl") == 0) {                 // programmatic dependent launch of every kernel (launch.h); process-wide
    pdl_enabled() = value ? 1 : 0;
    drop_graphs();
    return 0;
  }
  return -1;
}

// ------------------------------------------------------------------------------- weight packing
int Engine::load_weights(const std::map<std::string, HostTensor>& w, std::string* err) {
  DeviceGuard guard(device_);
  // Whatever happens below, the old packing is gone: a failed load must not leave a schedule pointing into a freed arena.
  weights_loaded_ = false;
  planned_B_ = 0;
  ops_.clear();
  const int C = cfg_.vit_dim, d = cfg_.hidden_dim, nq = cfg_.num_queries, ncls = cfg_.num_classes;
  const int G = cfg_.img_size / 16, T = G * G, ntap = cfg_.n_taps, c2 = d / 2;
  const int M = cfg_.ca_heads, L = cfg_.n_levels, P = cfg_.dec_points, ff = cfg_.dim_feedforward;
  bool missing = false;
  auto get = [&](const std::string& name, long long numel) -> const float* {
    auto it = w.find(name);
    if (it == w.end()) { if (!missing) *err = "missing tensor " + name; missing = true; return nullptr; }
    if (it->second.numel != numel) {
      if (!missing) *err = "tensor " + name + " has " + std::to_string(it->second.numel) + " elements, expected " + std::to_string(numel);
      missing = true; return nullptr;
    }
    return it->second.data;
  };
  auto vec = [&](const std::string& name, long long numel) {
    const float* p = get(name, numel);
    return p ? std::vector<float>(p, p + numel) : std::vector<float>(static_cast<size_t>(numel), 0.f);
  };
  // total parameter bytes bound: every tensor at most once in 16-bit + fp32 vectors + slack
  long long total = 0;
  for (auto& kv : w) total += kv.second.numel;
  drop_graphs();
  if (warena_.p) { cudaFree(warena_.p); warena_.p = nullptr; }
  warena_.bytes = static_cast<size_t>(total) * 4 + (96u << 20);
  if (cudaMalloc(&warena_.p, warena_.bytes) != cudaSuccess) { *err = "cudaMalloc(weight arena) failed"; return -1; }
  woff_ = 0;
  W_.clear(); F_.clear();
  bool oom = false;
  auto put16 = [&](const std::string& key, const std::vector<float>& v) { void* p = upload16(v); if (!p) oom = true; W_[key] = p; };
  auto put32 = [&](const std::string& key, const std::vector<float>& v) { float* p = upload32(v); if (!p) oom = true; F_[key] = p; };

  const int dtl = dtype_;
  auto round16 = [dtl](float f) -> float {
    return dtl == DT_BF16 ? __bfloat162float(__float2bfloat16_rn(f)) : __half2float(__float2half_rn(f));
  };
  // fold BatchNorm (eval, eps 1e-5) into a bias-free conv: returns (W', b') with W' laid out [Co][k-order]
  auto fold_convx = [&](const std::string& p, int co, int ci, int k, std::vector<float>* Wp, std::vector<float>* bp) {
    auto cw = vec(p + ".conv.weight", 1LL * co * ci * k * k);
    auto g = vec(p + ".bn.weight", co), b = vec(p + ".bn.bias", co), mu = vec(p + ".bn.running_mean", co), var = vec(p + ".bn.running_var", co);
    Wp->assign(static_cast<size_t>(co) * ci * k * k, 0.f);
    bp->assign(co, 0.f);
    for (int o = 0; o < co; ++o) {
      const float s = g[o] / std::sqrt(var[o] + 1e-5f);
      (*bp)[o] = b[o] - mu[o] * s;
      for (int i = 0; i < ci; ++i)
        for (int t = 0; t < k * k; ++t)      // [Co, Ci, kh, kw] -> [Co, (kh*k+kw)*Ci + ci]
          (*Wp)[(static_cast<size_t>(o) * k * k + t) * ci + i] = cw[(static_cast<size_t>(o) * ci + i) * k * k + t] * s;
    }
  };
  auto put_convx = [&](const std::string& key, const std::string& p, int co, int ci, int k) {
    std::vector<float> Wp, bp;
    fold_convx(p, co, ci, k, &Wp, &bp);
    put16(key + ".w", Wp);
    put32(key + ".b", bp);
  };
  auto put_linear = [&](const std::string& key, const std::string& p, int n_out, int n_in) {
    put16(key + ".w", vec(p + ".weight", 1LL * n_out * n_in));
    put32(key + ".b", vec(p + ".bias", n_out));
  };
  auto put_norm = [&](const std::string& key, const std::string& p, int n) {
    put32(key + ".w", vec(p + ".weight", n));
    put32(key + ".b", vec(p + ".bias", n));
  };
  // ConvTranspose2d(k=2,s=2) weight [Ci, Co, 2, 2] -> GEMM weight [(dy*2+dx)*Co + co, Ci], bias x4
  auto put_convT = [&](const std::string& key, const std::string& p, int ci, int co) {
    auto cw = vec(p + ".weight", 1LL * ci * co * 4);
    auto cb = vec(p + ".bias", co);
    std::vector<float> Wp(static_cast<size_t>(4) * co * ci), bp(static_cast<size_t>(4) * co);
    for (int i = 0; i < ci; ++i)
      for (int o = 0; o < co; ++o)
        for (int q = 0; q < 4; ++q) Wp[(static_cast<size_t>(q) * co + o) * ci + i] = cw[(static_cast<size_t>(i) * co + o) * 4 + q];
    for (int q = 0; q < 4; ++q)
      for (int o = 0; o < co; ++o) bp[q * co + o] = cb[o];
    put16(key + ".w", Wp);
    put32(key + ".b", bp);
  };

  // ---- ViT
  const std::string E = "backbone.0.encoder.";
  put16("patch.w", vec(E + "patch_embed.proj.weight", 1LL * C * 768));
  put32("patch.b", vec(E + "patch_embed.proj.bias", C));
  {
    // the raw table (cls slot dropped, vit.py:39-40) stays in the arena: plan() resizes it for other input resolutions
    auto pe = vec(E + "pos_embed", 197LL * C);
    put32("pos_raw", std::vector<float>(pe.begin() + C, pe.end()));
    void* p = walloc(static_cast<size_t>(T) * C * 2);   // the table at cfg.img_size, built once here
    W_["pos"] = p;
    if (!p) oom = true;
    else if (!oom && upload_pos_table(G, p)) { *err = "CUDA error while building the position table"; return -1; }
  }
  for (int i = 0; i < cfg_.vit_depth; ++i) {
    const std::string b = E + "blocks." + std::to_string(i) + ".", k = "blk" + std::to_string(i) + ".";
    put_norm(k + "ln1", b + "norm1", C);
    put16(k + "qkv.w", vec(b + "attn.qkv.weight", 3LL * C * C));
    {
      auto qb = vec(b + "attn.q_bias", C), vb = vec(b + "attn.v_bias", C);
      std::vector<float> bias(static_cast<size_t>(3) * C, 0.f);     // [q_bias, 0, v_bias]  (vit.py:123-125)
      std::copy(qb.begin(), qb.end(), bias.begin());
      std::copy(vb.begin(), vb.end(), bias.begin() + 2 * C);
      put32(k + "qkv.b", bias);
    }
    // LayerNorm-fused variants (consumer GEMMs run on the raw residual stream, see gemm_tc.h):
    //   W'[n,k] = W[n,k]*ln_w[k] ; colsum[n] = sum_k round16(W'[n,k]) ; bias'[n] = bias[n] + sum_k ln_b[k]*W[n,k]
    auto fold_ln = [&](const std::string& key, const std::vector<float>& Wm, const std::vector<float>& bias, const std::string& ln, int n_out) {
      auto lw = vec(ln + ".weight", C), lb = vec(ln + ".bias", C);
      std::vector<float> Wf(Wm.size()), cs(n_out), bf(n_out);
      for (int n = 0; n < n_out; ++n) {
        double acc_b = bias[n], acc_c = 0.0;
        for (int kk = 0; kk < C; ++kk) {
          const float wv = Wm[static_cast<size_t>(n) * C + kk];
          const float wf = wv * lw[kk];
          Wf[static_cast<size_t>(n) * C + kk] = wf;
          acc_c += round16(wf);
          acc_b += static_cast<double>(lb[kk]) * wv;
        }
        cs[n] = static_cast<float>(acc_c);
        bf[n] = static_cast<float>(acc_b);
      }
      put16(key + ".w", Wf);
      put32(key + ".b", bf);
      put32(key + ".cs", cs);
    };
    {
      auto qb = vec(b + "attn.q_bias", C), vb = vec(b + "attn.v_bias", C);
      std::vector<float> bias(static_cast<size_t>(3) * C, 0.f);
      std::copy(qb.begin(), qb.end(), bias.begin());
      std::copy(vb.begin(), vb.end(), bias.begin() + 2 * C);
      fold_ln(k + "qkv_ln", vec(b + "attn.qkv.weight", 3LL * C * C), bias, b + "norm1", 3 * C);
      fold_ln(k + "fc1_ln", vec(b + "mlp.fc1.weight", 4LL * C * C), vec(b + "mlp.fc1.bias", 4LL * C), b + "norm2", 4 * C);
    }
    put_linear(k + "proj", b + "attn.proj", C, C);
    put32(k + "g1", vec(b + "gamma_1", C));
    put_norm(k + "ln2", b + "norm2", C);
    put_linear(k + "fc1", b + "mlp.fc1", 4 * C, C);
    put_linear(k + "fc2", b + "mlp.fc2", C, 4 * C);
    put32(k + "g2", vec(b + "gamma_2", C));
  }
  // ---- projector
  const std::string PR = "backbone.0.projector.";
  for (int l = 0; l < L; ++l) {
    const int sc = cfg_.level_scale_log2[l];
    const std::string k = "lvl" + std::to_string(l) + ".";
    int cs = C;   // channels each tap contributes
    for (int t = 0; t < ntap; ++t) {
      const std::string s = PR + "stages_sampling." + std::to_string(l) + "." + std::to_string(t) + ".";
      const std::string ks = k + "samp" + std::to_string(t);
      if (sc == 1) {
        if (C > 512) {
          put_convx(ks + ".pre", s + "0", C / 2, C, 1);
          put_convT(ks + ".up", s + "1", C / 2, C / 4);
          cs = C / 4;
        } else {
          put_convT(ks + ".up", s + "0", C, C / 2);
          cs = C / 2;
        }
      } else if (sc == -1) {
        put_convx(ks + ".down", s + "0", C, C, 3);
      }
    }
    const std::string st = PR + "stages." + std::to_string(l) + ".";
    put_convx(k + "cv1", st + "0.cv1", 2 * c2, cs * ntap, 1);
    put_convx(k + "cv2", st + "0.cv2", d, 5 * c2, 1);
    for (int j = 0; j < 3; ++j) {
      put_convx(k + "m" + std::to_string(j) + "a", st + "0.m." + std::to_string(j) + ".cv1", c2, c2, 3);
      put_convx(k + "m" + std::to_string(j) + "b", st + "0.m." + std::to_string(j) + ".cv2", c2, c2, 3);
    }
    put_norm(k + "ln", st + "1", d);
  }
  // ---- two-stage + decoder (group 0 only in eval: lwdetr.py:141-144, transformer.py:229)
  const std::string TR = "transformer.";
  put_linear("enc_out", TR + "enc_output.0", d, d);
  put_norm("enc_ln", TR + "enc_output_norm.0", d);
  put_linear("enc_cls", TR + "enc_out_class_embed.0", ncls, d);
  for (int i = 0; i < 3; ++i) put_linear("enc_box" + std::to_string(i), TR + "enc_out_bbox_embed.0.layers." + std::to_string(i), i == 2 ? 4 : d, d);
  {
    auto re = vec("refpoint_embed.weight", 1LL * nq * cfg_.group_detr * 4);
    put32("refpoint_embed", std::vector<float>(re.begin(), re.begin() + static_cast<size_t>(nq) * 4));
    auto qf = vec("query_feat.weight", 1LL * nq * cfg_.group_detr * d);
    put16("query_feat", std::vector<float>(qf.begin(), qf.begin() + static_cast<size_t>(nq) * d));
  }
  put_linear("rph0", TR + "decoder.ref_point_head.layers.0", d, 2 * d);
  put_linear("rph1", TR + "decoder.ref_point_head.layers.1", d, d);
  std::vector<float> wval, bval;
  const int MLP = M * L * P;
  for (int i = 0; i < cfg_.dec_layers; ++i) {
    const std::string p = TR + "decoder.layers." + std::to_string(i) + ".", k = "dec" + std::to_string(i) + ".";
    auto ipw = vec(p + "self_attn.in_proj_weight", 3LL * d * d), ipb = vec(p + "self_attn.in_proj_bias", 3LL * d);
    put16(k + "qk.w", std::vector<float>(ipw.begin(), ipw.begin() + static_cast<size_t>(2) * d * d));
    put32(k + "qk.b", std::vector<float>(ipb.begin(), ipb.begin() + 2 * d));
    put16(k + "v.w", std::vector<float>(ipw.begin() + static_cast<size_t>(2) * d * d, ipw.end()));
    put32(k + "v.b", std::vector<float>(ipb.begin() + 2 * d, ipb.end()));
    put_linear(k + "so", p + "self_attn.out_proj", d, d);
    put_norm(k + "n1", p + "norm1", d);
    {
      auto ow = vec(p + "cross_attn.sampling_offsets.weight", 2LL * MLP * d), ob = vec(p + "cross_attn.sampling_offsets.bias", 2LL * MLP);
      auto aw = vec(p + "cross_attn.attention_weights.weight", 1LL * MLP * d), ab = vec(p + "cross_attn.attention_weights.bias", MLP);
      ow.insert(ow.end(), aw.begin(), aw.end());
      ob.insert(ob.end(), ab.begin(), ab.end());
      put16(k + "oa.w", ow);
      put32(k + "oa.b", ob);
    }
    {
      auto vw = vec(p + "cross_attn.value_proj.weight", 1LL * d * d), vb = vec(p + "cross_attn.value_proj.bias", d);
      wval.insert(wval.end(), vw.begin(), vw.end());
      bval.insert(bval.end(), vb.begin(), vb.end());
    }
    put_linear(k + "co", p + "cross_attn.output_proj", d, d);
    put_norm(k + "n2", p + "norm2", d);
    put_linear(k + "l1", p + "linear1", ff, d);
    put_linear(k + "l2", p + "linear2", d, ff);
    put_norm(k + "n3", p + "norm3", d);
  }
  put16("value.w", wval);
  put32("value.b", bval);
  put_norm("dec_norm", TR + "decoder.norm", d);
  put_linear("cls", "class_embed", ncls, d);
  for (int i = 0; i < 3; ++i) put_linear("box" + std::to_string(i), "bbox_embed.layers." + std::to_string(i), i == 2 ? 4 : d, d);
  if (missing) return -1;
  if (oom) { *err = "weight arena exhausted"; return -1; }
  if (cudaDeviceSynchronize() != cudaSuccess) { *err = "CUDA error while uploading weights"; return -1; }
  weights_loaded_ = true;
  planned_B_ = 0;   // pointers changed: re-plan
  return 0;
}

// ------------------------------------------------------------------------------- schedule
int Engine::plan(int B, int R, std::string* err) {
  const int C = cfg_.vit_dim, d = cfg_.hidden_dim, nq = cfg_.num_queries, ncls = cfg_.num_classes;
  const int G = R / 16, T = G * G, ntap = cfg_.n_taps, c2 = d / 2, heads = cfg_.vit_heads;
  const int M = cfg_.ca_heads, L = cfg_.n_levels, P = cfg_.dec_points, ff = cfg_.dim_feedforward, NL = cfg_.dec_layers;
  const long long BT = 1LL * B * T;
  int lvl_hw[2] = {0, 0}, lvl_start[2] = {0, 0}, S = 0;
  for (int l = 0; l < L; ++l) {
    const int sc = cfg_.level_scale_log2[l];
    lvl_hw[l] = sc == 1 ? 2 * G : (sc == -1 ? G / 2 : G);
    lvl_start[l] = S;
    S += lvl_hw[l] * lvl_hw[l];
  }
  const long long BS = 1LL * B * S, BQ = 1LL * B * nq;
  planned_B_ = 0;   // until this plan is complete, forward() must not run the old (or a half-built) schedule
  const int ldc = static_cast<int>(align_up(static_cast<size_t>(ncls), 32));   // row pitch of the fp32 class-logit buffers
  ldc_ = ldc;
  if (d / M != 16) { *err = "deformable attention head dim must be 16"; return -1; }
  if (C / heads != 16 && C / heads != 32 && C / heads != 64) { *err = "unsupported ViT head dim"; return -1; }

  for (int pass = 0; pass < 2; ++pass) {   // pass 0 sizes the workspace, pass 1 builds the ops
    soff_ = 0;
    ops_.clear();
    bool fail = false;
    auto buf16 = [&](long long rows, int cols) { return Mat{salloc(static_cast<size_t>(rows) * cols * 2), cols}; };
    auto buf32 = [&](long long n) { return static_cast<float*>(salloc(static_cast<size_t>(n) * 4)); };
    auto col = [&](Mat m, int c) { return Mat{cptr(m.p) + static_cast<size_t>(c) * 2, m.ld}; };
    auto w16 = [&](const std::string& k) -> void* { auto it = W_.find(k); if (it == W_.end()) { fail = true; *err = "internal: weight " + k; return nullptr; } return it->second; };
    auto w32 = [&](const std::string& k) -> float* { auto it = F_.find(k); if (it == F_.end()) { fail = true; *err = "internal: vector " + k; return nullptr; } return it->second; };

    struct GemmOpt {
      const float* gamma = nullptr; Mat resid{nullptr, 0}; int resid_mod = 0; int act = ACT_NONE; int out_fp32 = 0;
      int rows_in = ROWS_PLAIN, remap = 0, shuffle = 0, IH = 0, IW = 0;
      int conv = 0, cB = 0, cOH = 0, cOW = 0;   // conv: 1 = 3x3 s1, 2 = 3x3 s2
      int hm_S = 0, hm_heads = 0, hm_slices = 0; const uint8_t* row_zero = nullptr;
      float2* stats_out = nullptr; const float2* stats_in = nullptr; int ln_C = 0; float ln_eps = 0.f;
    };
    int stats_parts = 0;   // partial (sum, sumsq) pairs per row written by the N = C producer GEMMs
    auto add_gemm = [&](const std::string& label, Mat A, long long Mrows, int K, const std::string& wkey, int N, void* out, int ld_out,
                        const GemmOpt& o, long long out_rows = -1) {
      if (pass == 0) return;
      GemmDesc g;
      g.dtype = dtype_; g.A = A.p; g.lda = A.ld; g.M = static_cast<int>(Mrows); g.N = N; g.K = K;
      g.W = w16(wkey + ".w"); g.bias = F_.count(wkey + ".b") ? F_[wkey + ".b"] : nullptr;
      g.gamma = o.gamma; g.resid = o.resid.p; g.ld_resid = o.resid.ld; g.resid_mod = o.resid_mod; g.act = o.act;
      g.out = out; g.ld_out = ld_out; g.out_fp32 = o.out_fp32; g.rows_in = o.rows_in; g.remap_rows = o.remap;
      g.shuffle_cout = o.shuffle; g.IH = o.IH; g.IW = o.IW;
      g.hm_S = o.hm_S; g.hm_heads = o.hm_heads; g.hm_slices = o.hm_slices; g.row_zero = o.row_zero;
      if (o.conv) { g.a_mode = o.conv == 1 ? AMODE_CONV3_S1 : AMODE_CONV3_S2; g.B = o.cB; g.OH = o.cOH; g.OW = o.cOW; }
      g.stats_out = o.stats_out; g.stats_in = o.stats_in; g.stats_parts_in = stats_parts; g.ln_C = o.ln_C; g.ln_eps = o.ln_eps;
      if (o.stats_in) g.colsum = w32(wkey + ".cs");
      GemmOp op;
      std::string e;
      if (fail || gemm_build(g, &op, &e)) { if (!fail) *err = label + ": " + e; fail = true; return; }
      if (o.stats_out) {
        if (stats_parts == 0) stats_parts = op.args.stats_parts_out;
        if (stats_parts != op.args.stats_parts_out || stats_parts > 48) { *err = label + ": inconsistent LayerNorm partial count"; fail = true; return; }
      }
      Op P_;
      P_.label = label;
      P_.run = [op](cudaStream_t st) { return gemm_launch(op, st); };
      P_.out = out; P_.rows = out_rows >= 0 ? out_rows : (o.shuffle ? Mrows * 4 : Mrows); P_.cols = o.shuffle ? o.shuffle : (o.hm_S ? 16 : N);
      P_.ld = ld_out; P_.fp32 = o.out_fp32;
      P_.flops = op.flops;
      P_.bytes = 2.0 * (static_cast<double>(Mrows) * K + static_cast<double>(N) * K) + (o.out_fp32 ? 4.0 : 2.0) * Mrows * N + (o.resid.p ? 2.0 * Mrows * N : 0.0);
      ops_.push_back(P_);
    };
    auto add_ln = [&](const std::string& label, Mat x, Mat y, const std::string& nkey, float eps, long long rows, int Cn,
                      const uint8_t* flag = nullptr, int flag_mod = 0, const float* ovr = nullptr, Mat add = Mat{nullptr, 0},
                      Mat y2 = Mat{nullptr, 0}, long long ygroup = 0, long long ystride = 0, long long yoff = 0, long long out_rows = -1,
                      const std::string& nkey3 = std::string(), Mat y3 = Mat{nullptr, 0}, float eps3 = 0.f) {
      if (pass == 0) return;
      LayerNormArgs a;
      std::memset(&a, 0, sizeof a);
      if (y3.p) { a.w3 = w32(nkey3 + ".w"); a.b3 = w32(nkey3 + ".b"); a.eps3 = eps3; a.y3 = y3.p; a.ldy3 = y3.ld; }
      a.x = x.p; a.ldx = x.ld; a.y = y.p; a.ldy = y.ld; a.w = w32(nkey + ".w"); a.b = w32(nkey + ".b"); a.eps = eps;
      a.rows = rows; a.C = Cn; a.row_flag = flag; a.flag_mod = flag_mod > 0 ? flag_mod : 1; a.override_vec = ovr;
      a.add_src = add.p; a.ld_add = add.ld; a.y2 = y2.p; a.ldy2 = y2.ld; a.y_group = ygroup; a.y_group_stride = ystride; a.y_row_off = yoff;
      const int dt = dtype_;
      Op P_;
      P_.label = label;
      P_.run = [a, dt](cudaStream_t st) { return layernorm_launch(dt, a, st); };
      P_.out = y.p; P_.rows = out_rows >= 0 ? out_rows : rows; P_.cols = Cn; P_.ld = y.ld;
      P_.bytes = 4.0 * rows * Cn + (y2.p ? 4.0 * rows * Cn : 0.0) + (y3.p ? 2.0 * rows * Cn : 0.0);
      ops_.push_back(P_);
    };
    auto add_attn = [&](const std::string& label, Mat q, Mat k, Mat v, Mat o, int nseq, int seqlen, int nheads, int dh) {
      if (pass == 0) return;
      AttnArgs a;
      a.q = q.p; a.k = k.p; a.v = v.p; a.ldq = q.ld; a.ldk = k.ld; a.ldv = v.ld; a.o = o.p; a.ldo = o.ld;
      a.seqlen = seqlen; a.nseq = nseq; a.heads = nheads;
      a.scale_log2 = 1.4426950408889634f / std::sqrt(static_cast<float>(dh));
      const int dt = dtype_;
      Op P_;
      P_.label = label;
      P_.run = [a, dt, dh](cudaStream_t st) { return attention_launch(dt, a, dh, st); };
      P_.out = o.p; P_.rows = 1LL * nseq * seqlen; P_.cols = nheads * dh; P_.ld = o.ld;
      P_.flops = 4.0 * nseq * static_cast<double>(seqlen) * seqlen * nheads * dh;
      P_.bytes = 2.0 * 4.0 * nseq * seqlen * nheads * dh;
      ops_.push_back(P_);
    };
    auto add_op = [&](const std::string& label, std::function<int(cudaStream_t)> fn, const void* out, long long rows, int cols, int ld, int fp32, double bytes) {
      if (pass == 0) return;
      Op P_;
      P_.label = label; P_.run = std::move(fn); P_.out = out; P_.rows = rows; P_.cols = cols; P_.ld = ld; P_.fp32 = fp32; P_.bytes = bytes;
      ops_.push_back(P_);
    };
    const int dt = dtype_;

    // ================================================================ padding-mask tables (constants when the batch is unpadded)
    float* prop_b = buf32(BS * 4);
    float* vr_b = buf32(static_cast<long long>(B) * L * 2 + 4);
    uint8_t* invalid_b = static_cast<uint8_t*>(salloc(static_cast<size_t>(BS)));
    uint8_t* pad_b = static_cast<uint8_t*>(salloc(static_cast<size_t>(BS)));
    {
      const int img = R;
      const int lh0 = lvl_hw[0], lh1 = lvl_hw[1], ls0 = lvl_start[0], ls1 = lvl_start[1];
      add_op("mask_setup", [this, B, img, L, S, lh0, lh1, ls0, ls1, prop_b, invalid_b, pad_b, vr_b](cudaStream_t st) {
        const int lh[2] = {lh0, lh1}, ls[2] = {ls0, ls1};
        return mask_setup_launch(in_.mask, B, img, img, L, S, lh, lh, ls, prop_b, invalid_b, pad_b, vr_b, st);
      }, prop_b, BS, 4, 4, 1, 24.0 * BS);
      if (pass) ops_.back().reads_input = true;
    }
    // ================================================================ ViT encoder
    Mat a0 = buf16(BT, 768);
    Mat xa = buf16(BT, C), xb = buf16(BT, C), xm = buf16(BT, C), lnb = buf16(BT, C);
    Mat tapbuf = buf16(BT, ntap * C);
    Mat qkv = buf16(BT, 3 * C), att = buf16(BT, C), hid = buf16(BT, 4 * C);
    {
      void* a0p = a0.p;
      const int img = R;
      add_op("patch_gather", [this, a0p, B, img, dt](cudaStream_t st) {
               if (in_.kind == IN_U8_FRAMES) return resize_patch_gather_u8_launch(dt, frames_.data(), B, img, in_.mean, in_.stdv, a0p, st);
               if (in_.kind == IN_U8_NHWC) return patch_gather_u8_launch(dt, in_.images, in_.mean, in_.stdv, a0p, B, img, st);
               return patch_gather_launch(dt, in_.images, in_.kind == IN_F32_NCHW ? 1 : 0, a0p, B, img, st);
             },
             a0.p, BT, 768, 768, 0, 1.0 * B * 3 * img * img * 4 + 2.0 * BT * 768);
      if (pass) {
        ops_.back().reads_input = true;
        patch_op_ = static_cast<int>(ops_.size()) - 1;
        patch_bytes_ = ops_.back().bytes;
      }
    }
    float2* stats_x = static_cast<float2*>(salloc(static_cast<size_t>(BT) * 48 * sizeof(float2)));   // row stats of x (block input)
    float2* stats_m = static_cast<float2*>(salloc(static_cast<size_t>(BT) * 48 * sizeof(float2)));   // row stats of x + attn
    const bool fuse = fuse_ln_ != 0;
    Mat xcur = xa;
    {
      // position table: the load-time one at cfg.img_size, else one built for this grid in the workspace
      Mat pos = R == cfg_.img_size ? Mat{pass ? w16("pos") : nullptr, C} : buf16(T, C);
      if (pass && R != cfg_.img_size) {
        // earlier forwards may still read the workspace on the device: let them finish before the host writes into it
        if (cudaDeviceSynchronize() != cudaSuccess || upload_pos_table(G, pos.p)) { *err = "CUDA error while building the position table"; return -1; }
      }
      GemmOpt o; o.resid = pos; o.resid_mod = T;
      if (fuse) o.stats_out = stats_x;
      add_gemm("patch_embed", a0, BT, 768, "patch", C, xcur.p, xcur.ld, o);
    }
    int tap_slot = 0;
    for (int i = 0; i < cfg_.vit_depth; ++i) {
      const std::string k = "blk" + std::to_string(i) + ".", lb = "block" + std::to_string(i);
      const bool window = (cfg_.window_block_mask >> i) & 1;
      if (fuse) {
        GemmOpt o; o.stats_in = stats_x; o.ln_C = C; o.ln_eps = 1e-6f;
        add_gemm(lb + ".qkv", xcur, BT, C, k + "qkv_ln", 3 * C, qkv.p, qkv.ld, o);
      } else {
        add_ln(lb + ".ln1", xcur, lnb, k + "ln1", 1e-6f, BT, C);
        add_gemm(lb + ".qkv", lnb, BT, C, k + "qkv", 3 * C, qkv.p, qkv.ld, GemmOpt{});
      }
      add_attn(lb + (window ? ".win_attn" : ".glb_attn"), col(qkv, 0), col(qkv, C), col(qkv, 2 * C), att,
               window ? 16 * B : B, window ? T / 16 : T, heads, C / heads);
      { GemmOpt o; o.gamma = pass ? w32(k + "g1") : nullptr; o.resid = xcur; if (fuse) o.stats_out = stats_m;
        add_gemm(lb + ".proj", att, BT, C, k + "proj", C, xm.p, xm.ld, o); }
      if (fuse) {
        GemmOpt o; o.act = ACT_GELU; o.stats_in = stats_m; o.ln_C = C; o.ln_eps = 1e-6f;
        add_gemm(lb + ".fc1", xm, BT, C, k + "fc1_ln", 4 * C, hid.p, hid.ld, o);
      } else {
        add_ln(lb + ".ln2", xm, lnb, k + "ln2", 1e-6f, BT, C);
        GemmOpt o; o.act = ACT_GELU; add_gemm(lb + ".fc1", lnb, BT, C, k + "fc1", 4 * C, hid.p, hid.ld, o);
      }
      Mat xnext;
      bool is_tap = false;
      for (int t = 0; t < ntap; ++t) is_tap = is_tap || cfg_.taps[t] == i;
      if (is_tap) xnext = col(tapbuf, (tap_slot++) * C);
      else xnext = (xcur.p == xa.p) ? xb : xa;
      { GemmOpt o; o.gamma = pass ? w32(k + "g2") : nullptr; o.resid = xm; if (fuse && i + 1 < cfg_.vit_depth) o.stats_out = stats_x;
        add_gemm(lb, hid, BT, 4 * C, k + "fc2", C, xnext.p, xnext.ld, o); }
      xcur = xnext;
    }

    // ================================================================ projector -> decoder memory [B, S, d]
    Mat memory = buf16(BS, d);
    for (int l = 0; l < L; ++l) {
      const int sc = cfg_.level_scale_log2[l], H = lvl_hw[l];
      const long long rows = 1LL * B * H * H;
      const std::string k = "lvl" + std::to_string(l) + ".", lb = "level" + std::to_string(l);
      Mat c2f = buf16(rows, 5 * c2), tmp = buf16(rows, c2), pout = buf16(rows, d);
      if (sc == 0) {
        GemmOpt o; o.act = ACT_SILU; o.rows_in = ROWS_WINDOW_MAJOR; o.remap = 1; o.IH = G; o.IW = G;
        add_gemm(lb + ".cv1", tapbuf, BT, ntap * C, k + "cv1", 2 * c2, c2f.p, c2f.ld, o);
      } else if (sc == 1) {
        const int cs = C > 512 ? C / 4 : C / 2;
        Mat samp = buf16(rows, ntap * cs);
        Mat pre = C > 512 ? buf16(BT, C / 2) : Mat{nullptr, 0};
        for (int t = 0; t < ntap; ++t) {
          const std::string ks = k + "samp" + std::to_string(t);
          Mat src = col(tapbuf, t * C);
          int kin = C;
          if (C > 512) {
            GemmOpt o; o.act = ACT_RELU;
            add_gemm(lb + ".pre" + std::to_string(t), src, BT, C, ks + ".pre", C / 2, pre.p, pre.ld, o);
            src = pre; kin = C / 2;
          }
          GemmOpt o; o.rows_in = ROWS_WINDOW_MAJOR; o.shuffle = cs; o.IH = G; o.IW = G;
          Mat dst = col(samp, t * cs);
          add_gemm(lb + ".up" + std::to_string(t), src, BT, kin, ks + ".up", 4 * cs, dst.p, dst.ld, o);
        }
        GemmOpt o; o.act = ACT_SILU;
        add_gemm(lb + ".cv1", samp, rows, ntap * cs, k + "cv1", 2 * c2, c2f.p, c2f.ld, o);
      } else {
        Mat spat = buf16(BT, ntap * C), samp = buf16(rows, ntap * C);
        {
          void* sp = tapbuf.p; void* dp = spat.p; const int ldx = ntap * C;
          add_op(lb + ".unwindow", [sp, dp, ldx, BT, G, dt](cudaStream_t st) { return unwindow_launch(dt, sp, ldx, dp, ldx, BT, ldx, G, st); },
                 spat.p, BT, ldx, ldx, 0, 4.0 * BT * ldx);
        }
        for (int t = 0; t < ntap; ++t) {
          GemmOpt o; o.act = ACT_RELU; o.conv = 2; o.cB = B; o.cOH = H; o.cOW = H;
          Mat src = col(spat, t * C), dst = col(samp, t * C);
          add_gemm(lb + ".down" + std::to_string(t), src, rows, 9 * C, k + "samp" + std::to_string(t) + ".down", C, dst.p, dst.ld, o);
        }
        GemmOpt o; o.act = ACT_SILU;
        add_gemm(lb + ".cv1", samp, rows, ntap * C, k + "cv1", 2 * c2, c2f.p, c2f.ld, o);
      }
      for (int j = 0; j < 3; ++j) {
        GemmOpt o; o.act = ACT_SILU; o.conv = 1; o.cB = B; o.cOH = H; o.cOW = H;
        Mat src = col(c2f, (1 + j) * c2), dst = col(c2f, (2 + j) * c2);
        add_gemm(lb + ".m" + std::to_string(j) + "a", src, rows, 9 * c2, k + "m" + std::to_string(j) + "a", c2, tmp.p, tmp.ld, o);
        add_gemm(lb + ".m" + std::to_string(j) + "b", tmp, rows, 9 * c2, k + "m" + std::to_string(j) + "b", c2, dst.p, dst.ld, o);
      }
      { GemmOpt o; o.act = ACT_SILU; add_gemm(lb + ".cv2", c2f, rows, 5 * c2, k + "cv2", d, pout.p, pout.ld, o); }
      add_ln(lb, pout, memory, k + "ln", 1e-6f, rows, d, nullptr, 0, nullptr, Mat{nullptr, 0}, Mat{nullptr, 0}, 1LL * H * H, S, lvl_start[l], BS);
    }

    // ================================================================ two-stage query selection
    // value_proj of all decoder layers, HEAD-MAJOR [B][layer][head][S][16] (msda.cu stages whole (image, head) slabs)
    Mat value = buf16(BS, NL * d), om = buf16(BS, d), omn = buf16(BS, d);
    float* cls_all = buf32(BS * ldc);
    float* score = buf32(BS);
    int* topk_idx = static_cast<int*>(salloc(static_cast<size_t>(BQ) * 4));
    Mat sel = buf16(BQ, d), h1 = buf16(BQ, d), h2 = buf16(BQ, d);
    float* delta_ts = buf32(BQ * 4);
    float* enc_logits = buf32(BQ * ncls);
    float* enc_boxes = buf32(BQ * 4);
    float* refpoint = buf32(BQ * 4);
    Mat sine = buf16(BQ, 2 * d), qpos = buf16(BQ, d);
    { GemmOpt o; o.hm_S = S; o.hm_heads = M; o.hm_slices = NL; o.row_zero = pad_b; add_gemm("value_proj", memory, BS, d, "value", NL * d, value.p, 16, o, BS * NL * M); }
    add_gemm("enc_output", memory, BS, d, "enc_out", d, om.p, om.ld, GemmOpt{});
    add_ln("enc_output_norm", om, omn, "enc_ln", 1e-5f, BS, d, invalid_b, static_cast<int>(BS), pass ? w32("enc_out.b") : nullptr);
    { GemmOpt o; o.out_fp32 = 1; add_gemm("enc_class", omn, BS, d, "enc_cls", ncls, cls_all, ldc, o); }
    add_op("enc_score", [cls_all, ncls, ldc, score, BS](cudaStream_t st) { return rowmax_launch(cls_all, ldc, ncls, score, BS, st); }, score, BS, 1, 1, 1, 4.0 * BS * ncls);
    add_op("topk", [this, score, B, S, nq, topk_idx](cudaStream_t st) {
      if (in_topk_override_ != nullptr)
        return static_cast<int>(cudaMemcpyAsync(topk_idx, in_topk_override_, static_cast<size_t>(B) * nq * 4, cudaMemcpyDeviceToDevice, st));
      return topk_launch(score, B, S, nq, topk_idx, st);
    }, nullptr, 0, 0, 0, 0, 4.0 * BS);
    {
      void* omp = omn.p; void* selp = sel.p;
      add_op("gather_topk", [omp, d, cls_all, ncls, ldc, topk_idx, B, S, nq, selp, enc_logits, dt](cudaStream_t st) {
        return gather_topk_launch(dt, omp, d, cls_all, ldc, ncls, topk_idx, B, S, nq, d, selp, enc_logits, st);
      }, sel.p, BQ, d, d, 0, 4.0 * BQ * d);
    }
    { GemmOpt o; o.act = ACT_RELU; add_gemm("enc_box0", sel, BQ, d, "enc_box0", d, h1.p, h1.ld, o); }
    { GemmOpt o; o.act = ACT_RELU; add_gemm("enc_box1", h1, BQ, d, "enc_box1", d, h2.p, h2.ld, o); }
    { GemmOpt o; o.out_fp32 = 1; add_gemm("enc_box2", h2, BQ, d, "enc_box2", 4, delta_ts, 4, o); }
    {
      const float* rpe = pass ? w32("refpoint_embed") : nullptr;
      void* sp = sine.p;
      add_op("query_init", [delta_ts, prop_b, topk_idx, rpe, B, nq, d, enc_boxes, refpoint, sp, dt, S, L, vr_b](cudaStream_t st) {
        return query_init_launch(dt, delta_ts, prop_b, topk_idx, rpe, B, nq, d, enc_boxes, refpoint, sp, S, L, vr_b, st);
      }, refpoint, BQ, 4, 4, 1, 4.0 * BQ * d);
    }
    { GemmOpt o; o.act = ACT_RELU; add_gemm("ref_point_head0", sine, BQ, 2 * d, "rph0", d, h1.p, h1.ld, o); }
    add_gemm("query_pos", h1, BQ, d, "rph1", d, qpos.p, qpos.ld, GemmOpt{});

    // ================================================================ decoder
    Mat tgt = buf16(BQ, d), tq = buf16(BQ, d), t1 = buf16(BQ, d), ta = buf16(BQ, d), tb = buf16(BQ, d);
    Mat qk = buf16(BQ, 2 * d), vb = buf16(BQ, d), sa = buf16(BQ, d), oa = buf16(BQ, 3 * M * L * P), ms = buf16(BQ, d), ffh = buf16(BQ, ff);
    Mat hs = buf16(NL * BQ, d);
    {
      void* qf = pass ? w16("query_feat") : nullptr; void* tp = tgt.p; void* tqp = tq.p; void* qp = qpos.p;
      add_op("tgt_init", [qf, d, nq, tp, BQ, dt](cudaStream_t st) { return add_rows_launch(dt, qf, d, nq, nullptr, 0, tp, d, BQ, d, st); }, tgt.p, BQ, d, d, 0, 4.0 * BQ * d);
      add_op("tgt_plus_pos", [qf, d, nq, qp, tqp, BQ, dt](cudaStream_t st) { return add_rows_launch(dt, qf, d, nq, qp, d, tqp, d, BQ, d, st); }, tq.p, BQ, d, d, 0, 6.0 * BQ * d);
    }
    MsdaArgs mbase;
    std::memset(&mbase, 0, sizeof mbase);
    mbase.v_b_stride = 1LL * NL * M * S * MSDA_D; mbase.valid_ratio = vr_b; mbase.offs_logits = oa.p; mbase.ld_ol = oa.ld; mbase.ref = refpoint; mbase.out = ms.p; mbase.ld_out = ms.ld;
    mbase.batch = B; mbase.nq = nq; mbase.heads = M; mbase.levels = L; mbase.points = P; mbase.S = S;
    for (int l = 0; l < L; ++l) { mbase.lvl_h[l] = lvl_hw[l]; mbase.lvl_w[l] = lvl_hw[l]; mbase.lvl_start[l] = lvl_start[l]; }
    if (msda_plan(&mbase)) { *err = "deformable attention: a feature level is too wide to stage"; return -1; }
    Mat cur = tgt;
    for (int i = 0; i < NL; ++i) {
      const std::string k = "dec" + std::to_string(i) + ".", lb = "dec" + std::to_string(i);
      add_gemm(lb + ".qk", tq, BQ, d, k + "qk", 2 * d, qk.p, qk.ld, GemmOpt{});
      add_gemm(lb + ".v", cur, BQ, d, k + "v", d, vb.p, vb.ld, GemmOpt{});
      add_attn(lb + ".self_attn", col(qk, 0), col(qk, d), vb, sa, B, nq, cfg_.sa_heads, d / cfg_.sa_heads);
      { GemmOpt o; o.resid = cur; add_gemm(lb + ".sa_out", sa, BQ, d, k + "so", d, t1.p, t1.ld, o); }
      add_ln(lb + ".norm1", t1, ta, k + "n1", 1e-5f, BQ, d, nullptr, 0, nullptr, qpos, tq);
      add_gemm(lb + ".offs_attn", tq, BQ, d, k + "oa", 3 * M * L * P, oa.p, oa.ld, GemmOpt{});
      {
        MsdaArgs ma = mbase;
        ma.value = cptr(value.p) + static_cast<size_t>(i) * M * S * MSDA_D * 2;
        add_op(lb + ".msda", [ma, dt](cudaStream_t st) { return msda_launch(dt, ma, st); }, ms.p, BQ, d, d, 0,
               2.0 * std::min<double>(1.0 * BS * d, 1.0 * BQ * M * L * P * 4 * 16) + 2.0 * BQ * M * L * P * 3 + 2.0 * BQ * d);
      }
      { GemmOpt o; o.resid = ta; add_gemm(lb + ".ca_out", ms, BQ, d, k + "co", d, t1.p, t1.ld, o); }
      add_ln(lb + ".norm2", t1, tb, k + "n2", 1e-5f, BQ, d);
      { GemmOpt o; o.act = ACT_RELU; add_gemm(lb + ".linear1", tb, BQ, d, k + "l1", ff, ffh.p, ffh.ld, o); }
      { GemmOpt o; o.resid = tb; add_gemm(lb + ".linear2", ffh, BQ, ff, k + "l2", d, t1.p, t1.ld, o); }
      // norm3 and the decoder's output norm of this layer's hidden state (transformer.py:279-285) in one launch
      Mat hsl{cptr(hs.p) + static_cast<size_t>(i) * BQ * d * 2, d};
      add_ln(lb, t1, tgt, k + "n3", 1e-5f, BQ, d, nullptr, 0, nullptr, qpos, tq, 0, 0, 0, -1, "dec_norm", hsl, 1e-5f);
      cur = tgt;
    }
    // ================================================================ heads
    float* logits = buf32(NL * BQ * ldc);
    float* delta = buf32(NL * BQ * 4);
    float* boxes = buf32(NL * BQ * 4);
    Mat bh1 = buf16(NL * BQ, d), bh2 = buf16(NL * BQ, d);
    { GemmOpt o; o.out_fp32 = 1; add_gemm("class_embed", hs, NL * BQ, d, "cls", ncls, logits, ldc, o); }
    { GemmOpt o; o.act = ACT_RELU; add_gemm("bbox0", hs, NL * BQ, d, "box0", d, bh1.p, bh1.ld, o); }
    { GemmOpt o; o.act = ACT_RELU; add_gemm("bbox1", bh1, NL * BQ, d, "box1", d, bh2.p, bh2.ld, o); }
    { GemmOpt o; o.out_fp32 = 1; add_gemm("bbox2", bh2, NL * BQ, d, "box2", 4, delta, 4, o); }
    add_op("final_boxes", [delta, refpoint, BQ, NL, boxes](cudaStream_t st) { return final_boxes_launch(delta, refpoint, BQ, NL, boxes, st); },
           boxes, NL * BQ, 4, 4, 1, 32.0 * NL * BQ);
    out_logits_ = logits; out_boxes_ = boxes; out_enc_logits_ = enc_logits; out_enc_boxes_ = enc_boxes; topk_idx_ = topk_idx;

    if (pass == 0) {
      const size_t need = soff_ + 4096;
      if (need > sarena_.bytes) {
        if (sarena_.p) cudaFree(sarena_.p);
        sarena_.p = nullptr;
        if (cudaMalloc(&sarena_.p, need) != cudaSuccess) { *err = "cudaMalloc(workspace, " + std::to_string(need >> 20) + " MiB) failed"; sarena_.bytes = 0; return -1; }
        sarena_.bytes = need;
      }
    } else if (fail) {
      return -1;
    }
  }
  drop_graphs();
  eager_runs_ = 0;
  planned_B_ = B;
  planned_R_ = R;
  return 0;
}

int Engine::do_capture(const Op& op, cudaStream_t st) {
  for (auto& c : captures_) {
    if (c.label != op.label || op.out == nullptr) continue;
    if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
    const long long n = op.rows * op.cols;
    if (n > c.capacity) { c.written = -2; continue; }
    const size_t esz = op.fp32 ? 4 : 2;
    std::vector<uint8_t> raw(static_cast<size_t>(n) * esz);
    if (cudaMemcpy2D(raw.data(), op.cols * esz, op.out, static_cast<size_t>(op.ld) * esz, op.cols * esz, static_cast<size_t>(op.rows), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    if (op.fp32) std::memcpy(c.dst, raw.data(), raw.size());
    else if (dtype_ == DT_BF16) for (long long i = 0; i < n; ++i) { __nv_bfloat16 v; std::memcpy(&v, &raw[i * 2], 2); c.dst[i] = __bfloat162float(v); }
    else for (long long i = 0; i < n; ++i) { __half v; std::memcpy(&v, &raw[i * 2], 2); c.dst[i] = __half2float(v); }
    c.written = n;
  }
  return 0;
}

int Engine::forward(const ForwardIn& in, int B, int R, float* pred_logits, float* pred_boxes, const lwdetr_aux_out* aux,
                    const int32_t* topk_override, cudaStream_t st, std::string* err) {
  DeviceGuard guard(device_);
  if (!weights_loaded_) { *err = "lwdetr_forward: weights not loaded"; return -1; }
  if (B <= 0) { *err = "lwdetr_forward: batch must be positive"; return -1; }
  if ((B != planned_B_ || R != planned_R_) && plan(B, R, err)) return -1;
  if (in.kind == IN_U8_FRAMES ? !in.frames : !in.images) { *err = "lwdetr_forward: null images"; return -1; }
  in_ = in; in_topk_override_ = topk_override;
  // the input op's byte count follows the input: a frames batch reads the frames, whatever their sizes
  Op& gather = ops_[patch_op_];
  gather.bytes = patch_bytes_;
  if (in.kind == IN_U8_FRAMES) {
    frames_.assign(in.frames, in.frames + B);
    in_.frames = frames_.data();
    gather.bytes = 2.0 * gather.rows * gather.cols;
    for (const lwdetr_frame& f : frames_) gather.bytes += 3.0 * f.height * f.width;
  }
  // The first forward of a plan always runs eagerly (it also performs the one-time cudaFuncSetAttribute calls).
  const bool graph_ok = use_graph_ && captures_.empty() && eager_runs_ > 0;
  if (graph_ok) {
    if (!gstream_) {
      if (cudaStreamCreateWithFlags(&gstream_, cudaStreamNonBlocking) != cudaSuccess ||
          cudaEventCreateWithFlags(&ev_in_, cudaEventDisableTiming) != cudaSuccess ||
          cudaEventCreateWithFlags(&ev_out_, cudaEventDisableTiming) != cudaSuccess) { *err = "graph stream setup failed"; return -1; }
    }
    const GraphKey key{topk_override};
    auto it = graphs_.find(key);
    if (it == graphs_.end()) {
      if (graphs_.size() >= 8) drop_graphs();
      cudaGraph_t g = nullptr;
      if (cudaStreamBeginCapture(gstream_, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { *err = std::string("graph capture begin failed: ") + cudaGetErrorString(cudaGetLastError()); return -1; }
      int rc = 0;
      for (auto& op : ops_) { if (op.reads_input) continue; rc = op.run(gstream_); if (rc) break; }
      cudaError_t ce = cudaStreamEndCapture(gstream_, &g);
      if (rc || ce != cudaSuccess) { if (g) cudaGraphDestroy(g); *err = "graph capture failed"; return -1; }
      cudaGraphExec_t ex = nullptr;
      if (cudaGraphInstantiate(&ex, g, 0) != cudaSuccess) { cudaGraphDestroy(g); *err = "graph instantiate failed"; return -1; }
      cudaGraphDestroy(g);
      it = graphs_.emplace(key, ex).first;
    }
    // the input-reading ops on the caller's stream, then the graph ordered after them, then the caller's stream after the graph
    for (auto& op : ops_) {
      if (!op.reads_input) continue;
      const int rc = op.run(st);
      if (rc) { *err = "op " + op.label + " failed to launch"; return -1; }
    }
    if (cudaEventRecord(ev_in_, st) != cudaSuccess || cudaStreamWaitEvent(gstream_, ev_in_, 0) != cudaSuccess ||
        cudaGraphLaunch(it->second, gstream_) != cudaSuccess || cudaEventRecord(ev_out_, gstream_) != cudaSuccess ||
        cudaStreamWaitEvent(st, ev_out_, 0) != cudaSuccess) { *err = std::string("graph launch failed: ") + cudaGetErrorString(cudaGetLastError()); return -1; }
  } else {
    for (auto& op : ops_) {
      const int rc = op.run(st);
      if (rc) { *err = "op " + op.label + " failed to launch: " + (rc > 0 ? cudaGetErrorString(static_cast<cudaError_t>(rc)) : "bad arguments"); return -1; }
      if (!captures_.empty() && do_capture(op, st)) { *err = "capture after " + op.label + " failed: " + cudaGetErrorString(cudaGetLastError()); return -1; }
    }
    ++eager_runs_;
  }
  // results -> caller buffers (dense)
  const int nq = cfg_.num_queries, ncls = cfg_.num_classes, NL = cfg_.dec_layers;
  const long long BQ = 1LL * B * nq;
  auto copy_logits = [&](float* dst, int layer) {
    return cudaMemcpy2DAsync(dst, ncls * 4, out_logits_ + static_cast<size_t>(layer) * BQ * ldc_, static_cast<size_t>(ldc_) * 4, ncls * 4, static_cast<size_t>(BQ), cudaMemcpyDeviceToDevice, st);
  };
  cudaError_t e = cudaSuccess;
  if (pred_logits) e = copy_logits(pred_logits, NL - 1);
  if (e == cudaSuccess && pred_boxes) e = cudaMemcpyAsync(pred_boxes, out_boxes_ + static_cast<size_t>(NL - 1) * BQ * 4, BQ * 16, cudaMemcpyDeviceToDevice, st);
  if (aux) {
    for (int l = 0; l + 1 < NL && e == cudaSuccess; ++l) {
      if (aux->aux_logits) e = copy_logits(aux->aux_logits + static_cast<size_t>(l) * BQ * ncls, l);
      if (e == cudaSuccess && aux->aux_boxes) e = cudaMemcpyAsync(aux->aux_boxes + static_cast<size_t>(l) * BQ * 4, out_boxes_ + static_cast<size_t>(l) * BQ * 4, BQ * 16, cudaMemcpyDeviceToDevice, st);
    }
    if (e == cudaSuccess && aux->enc_logits) e = cudaMemcpyAsync(aux->enc_logits, out_enc_logits_, BQ * ncls * 4, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess && aux->enc_boxes) e = cudaMemcpyAsync(aux->enc_boxes, out_enc_boxes_, BQ * 16, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess && aux->topk_index) e = cudaMemcpyAsync(aux->topk_index, topk_idx_, BQ * 4, cudaMemcpyDeviceToDevice, st);
  }
  if (e != cudaSuccess) { *err = std::string("result copy failed: ") + cudaGetErrorString(e); return -1; }
  return 0;
}

int Engine::profile_ops(int iters, std::vector<float>* ms, cudaStream_t st, std::string* err) {
  DeviceGuard guard(device_);
  if (planned_B_ <= 0) { *err = "profile_ops: run a forward first"; return -1; }
  ms->assign(ops_.size(), 0.f);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (size_t i = 0; i < ops_.size(); ++i) {
    ops_[i].run(st);   // warm
    cudaEventRecord(e0, st);
    for (int k = 0; k < iters; ++k) ops_[i].run(st);
    cudaEventRecord(e1, st);
    if (cudaEventSynchronize(e1) != cudaSuccess) { *err = "profile_ops: op " + ops_[i].label + " failed"; return -1; }
    float t = 0.f;
    cudaEventElapsedTime(&t, e0, e1);
    (*ms)[i] = t / iters;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return 0;
}

}  // namespace lwb
