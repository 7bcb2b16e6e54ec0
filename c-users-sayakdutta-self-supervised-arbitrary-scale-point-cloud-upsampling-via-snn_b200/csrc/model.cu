// Model handles: weight registry, eval-mode folding, upload.
//
// Folding rules (all on the host, fp32 like torch's eval BatchNorm):
//   invstd = 1/sqrt(running_var + 1e-5) ; scale = weight*invstd ; shift = bias_bn - running_mean*scale
//   neuron parameters are clamped to the ranges the reference clamps to at every step
//   (fn/snn_coder.py:116-118, fd/snn_coder.py:231-235); fd temporal weights are soft-maxed (fd/snn_coder.py:327).
#include <cmath>
#include <algorithm>
#include <math.h>
#include <string.h>
#include "../../include/sapcu_b200.h"
#include "model.h"
#include "lif_table.cuh"

using namespace sapcu;

namespace {

// IEEE binary16 conversions on the host (round to nearest even, subnormals kept)
static uint16_t f32_to_f16_rn(float f) {
  uint32_t x; memcpy(&x, &f, 4);
  const uint32_t sign = (x >> 16) & 0x8000u;
  const uint32_t ax = x & 0x7FFFFFFFu;
  if (ax >= 0x7F800000u) return (uint16_t)(sign | 0x7C00u | (ax > 0x7F800000u ? 0x200u : 0));   // inf / nan
  if (ax >= 0x477FF000u) return (uint16_t)(sign | 0x7C00u);                                      // rounds to inf
  if (ax < 0x33000001u) return (uint16_t)sign;                                                   // below half the smallest subnormal
  int exp = (int)(ax >> 23) - 127;
  uint32_t man = (ax & 0x7FFFFFu) | 0x800000u;                        // 24-bit significand
  int shift = exp >= -14 ? 13 : 13 + (-14 - exp);                      // bits dropped
  uint32_t half_man = man >> shift;
  const uint32_t rem = man & ((1u << shift) - 1), halfway = 1u << (shift - 1);
  if (rem > halfway || (rem == halfway && (half_man & 1u))) ++half_man;
  uint32_t out;
  if (exp >= -14) out = ((uint32_t)(exp + 15) << 10) + (half_man - 0x400u);   // carry into the exponent is handled by +
  else out = half_man;                                                         // subnormal (may round up to the smallest normal)
  return (uint16_t)(sign | out);
}
static float f16_to_f32(uint16_t h) {
  const uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
  const int exp = (h >> 10) & 31; const uint32_t man = h & 0x3FFu;
  float v;
  if (exp == 0) v = std::ldexp((float)man, -24);
  else if (exp == 31) { uint32_t b = sign | 0x7F800000u | (man << 13); memcpy(&v, &b, 4); return v; }
  else v = std::ldexp((float)(man | 0x400u), exp - 25);
  uint32_t b; memcpy(&b, &v, 4); b |= sign; memcpy(&v, &b, 4);
  return v;
}

struct Builder {
  sapcu_model* m;
  std::vector<float> blob;
  std::string err;
  struct Fix { const float** dst; size_t off; };
  std::vector<Fix> fixes;

  const std::vector<float>* get(const std::string& name, size_t numel) {
    auto it = m->host.find(name);
    if (it == m->host.end()) { if (err.empty()) err = "missing tensor '" + name + "'"; return nullptr; }
    if (it->second.size() != numel) {
      if (err.empty()) err = "tensor '" + name + "' has " + std::to_string(it->second.size()) + " elements, expected " + std::to_string(numel);
      return nullptr;
    }
    return &it->second;
  }
  size_t put(const float* p, size_t n, const float** dst) {
    size_t off = (blob.size() + 63) / 64 * 64;   // 256-byte alignment
    blob.resize(off + n);
    if (p) memcpy(blob.data() + off, p, n * sizeof(float));
    fixes.push_back({dst, off});
    return off;
  }
  // weight matrix + its tensor-core splits (split_weights)
  void put_w(Layer& L, const float* w, size_t n) {
    put(w, n, &L.W);
    WeightSplit s;
    split_weights(w, n, &s);
    put(s.hi.data(), n, &L.Whi); put(s.lo.data(), n, &L.Wlo);
    put(reinterpret_cast<const float*>(s.h.data()), s.h.size() / 2, &L.Wh);
    put(reinterpret_cast<const float*>(s.l.data()), s.l.size() / 2, &L.Wl);
    L.winv = s.winv;
  }
  // conv/linear `wname`.weight [N,K(,1,1)], optional .bias; optional BatchNorm `bnname`
  void layer(Layer& L, const std::string& wname, const std::string& bnname, int N, int K, bool bias) {
    L.N = N; L.K = K;
    if (auto* w = get(wname + ".weight", (size_t)N * K)) put_w(L, w->data(), w->size());
    if (bias) { if (auto* b = get(wname + ".bias", N)) put(b->data(), N, &L.bias); }
    if (!bnname.empty()) {
      auto* g = get(bnname + ".weight", N); auto* b = get(bnname + ".bias", N);
      auto* mu = get(bnname + ".running_mean", N); auto* var = get(bnname + ".running_var", N);
      if (g && b && mu && var) {
        std::vector<float> sc(N), sh(N);
        for (int i = 0; i < N; ++i) {
          const float invstd = 1.0f / sqrtf((*var)[i] + 1e-5f);
          sc[i] = (*g)[i] * invstd;
          sh[i] = (*b)[i] - (*mu)[i] * sc[i];
        }
        put(sc.data(), N, &L.scale); put(sh.data(), N, &L.shift);
      }
    }
  }
  // several conv(+bias)+BN pairs `<name>.0` / `<name>.1` with a shared input, stacked along N
  void layer_cat(Layer& L, const std::vector<std::string>& names, int N_each, int K) {
    const int n = (int)names.size();
    L.N = N_each * n; L.K = K;
    std::vector<float> W((size_t)L.N * K), bi(L.N), sc(L.N), sh(L.N);
    for (int q = 0; q < n; ++q) {
      auto* w = get(names[q] + ".0.weight", (size_t)N_each * K); auto* b0 = get(names[q] + ".0.bias", N_each);
      auto* g = get(names[q] + ".1.weight", N_each); auto* b = get(names[q] + ".1.bias", N_each);
      auto* mu = get(names[q] + ".1.running_mean", N_each); auto* var = get(names[q] + ".1.running_var", N_each);
      if (!(w && b0 && g && b && mu && var)) return;
      memcpy(W.data() + (size_t)q * N_each * K, w->data(), w->size() * sizeof(float));
      for (int i = 0; i < N_each; ++i) {
        const float invstd = 1.0f / sqrtf((*var)[i] + 1e-5f);
        bi[q * N_each + i] = (*b0)[i];
        sc[q * N_each + i] = (*g)[i] * invstd;
        sh[q * N_each + i] = (*b)[i] - (*mu)[i] * sc[q * N_each + i];
      }
    }
    put_w(L, W.data(), W.size()); put(bi.data(), bi.size(), &L.bias);
    put(sc.data(), sc.size(), &L.scale); put(sh.data(), sh.size(), &L.shift);
  }
  static float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }
  // neuron parameter block(s) concatenated along the channel axis: np = [4][C_total]
  // tab_T > 0: also tabulate the T-step chain from the zero state (LIF only) for the fast mode
  void neuron(Neuron& nr, const std::vector<std::string>& names, int C_each, bool eif, int tab_T = 0) {
    const int n = (int)names.size(), C = C_each * n;
    nr.C = C;
    std::vector<float> np(4 * (size_t)C), ep(2 * (size_t)C);
    bool ok = true;
    for (int q = 0; q < n; ++q) {
      auto* d = get(names[q] + ".membrane_decay", C_each); auto* a = get(names[q] + ".threshold_adapt", C_each);
      auto* r = get(names[q] + ".refractory_decay", C_each); auto* t = get(names[q] + ".threshold_base", C_each);
      if (!(d && a && r && t)) { ok = false; break; }
      for (int i = 0; i < C_each; ++i) {
        np[0 * C + q * C_each + i] = clampf((*d)[i], 0.1f, 0.99f);
        np[1 * C + q * C_each + i] = clampf((*a)[i], 0.001f, 0.1f);
        np[2 * C + q * C_each + i] = clampf((*r)[i], 0.1f, 0.95f);
        np[3 * C + q * C_each + i] = (*t)[i];
      }
      if (eif) {
        auto* dt = get(names[q] + ".delta_T", C_each); auto* th = get(names[q] + ".theta_rh", C_each);
        if (!(dt && th)) { ok = false; break; }
        for (int i = 0; i < C_each; ++i) {
          ep[0 * C + q * C_each + i] = clampf((*dt)[i], 0.1f, 5.0f);
          ep[1 * C + q * C_each + i] = clampf((*th)[i], 0.1f, 2.0f);
        }
      }
    }
    if (!ok) return;
    put(np.data(), np.size(), &nr.np);
    if (eif) put(ep.data(), ep.size(), &nr.ep);
    if (tab_T > 0 && !eif) {
      LifTablePacked t;
      lif_table_pack(np.data(), C, tab_T, &t);
      put(t.img.data(), t.img.size(), &nr.tab);
      nr.tab_stride = t.stride; nr.tab_T = tab_T; nr.tab_ok = t.usable; nr.tab_err = t.max_err;
    }
  }
  void raw(const std::string& name, size_t n, const float** dst) {
    if (auto* v = get(name, n)) put(v->data(), n, dst);
  }
};

void build_fn(Builder& B) {
  FnNet& f = B.m->fn;
  const auto& c = B.m->cfg;
  f.kvals[0] = c[0]; f.kvals[1] = c[1]; f.kvals[2] = c[2]; f.emb = c[3]; f.T_enc = c[4]; f.heads = c[5];
  B.layer(f.conv1, "encoder.conv1.0", "encoder.conv1.1", 64, 3, true);
  B.neuron(f.snn_init, {"encoder.snn_init"}, 64, false, f.T_enc);
  const int Ds[3] = {128, 256, 512};
  for (int b = 0; b < 3; ++b) {
    FnBlock& k = f.blk[b];
    k.D = Ds[b]; k.k = f.kvals[b];
    const int D = k.D;
    const std::string p = "encoder.trans" + std::to_string(b + 1) + ".";
    B.layer(k.fc1, p + "fc1.0", p + "fc1.1", D, 64, true);
    B.neuron(k.snn1, {p + "snn1"}, D, false, 4);
    // q, k, v share their input: one [3D, D] contraction with concatenated weights / BN / neuron rows
    B.layer_cat(k.qkv, {p + "w_qs", p + "w_ks", p + "w_vs"}, D, D);
    B.neuron(k.snn_qkv, {p + "snn_q", p + "snn_k", p + "snn_v"}, D, false, 4);
    B.layer(k.fc_delta, p + "fc_delta.0", p + "fc_delta.1", D, 3, true);
    B.neuron(k.snn_delta, {p + "snn_delta"}, D, false, 4);
    B.layer(k.fc_delta2, p + "fc_delta2.0", p + "fc_delta2.1", D, D, true);
    B.neuron(k.snn_delta2, {p + "snn_delta2"}, D, false, 4);
    B.layer(k.fc_gamma, p + "fc_gamma.0", p + "fc_gamma.1", D, D, true);
    B.neuron(k.snn_gamma, {p + "snn_gamma"}, D, false, 4);
    B.layer(k.fc_gamma2, p + "fc_gamma2.0", p + "fc_gamma2.1", D, D, true);
    B.layer(k.out_proj, p + "out_proj.0", p + "out_proj.1", D, D, true);
    B.layer(k.fc2, p + "fc2.0", p + "fc2.1", 64, D, true);
  }
  B.layer(f.conv_final, "encoder.conv_final.0", "encoder.conv_final.1", f.emb, 192, true);
  B.neuron(f.snn_final, {"encoder.snn_final"}, f.emb, false, f.T_enc);
  B.layer(f.fc_out, "encoder.fc_out", "", 2048, f.emb, true);
  B.layer(f.mlp[0], "decoder.mlp.0", "decoder.mlp.1", 1024, 2048, true);
  B.layer(f.mlp[1], "decoder.mlp.4", "decoder.mlp.5", 512, 1024, true);
  B.layer(f.mlp[2], "decoder.mlp.8", "decoder.mlp.9", 256, 512, true);
  B.layer(f.head, "decoder.fc_out", "", 3, 256, true);
  B.raw("decoder.norm_out.weight", 3, &f.ln_w);
  B.raw("decoder.norm_out.bias", 3, &f.ln_b);
}

void build_fd(Builder& B) {
  FdNet& f = B.m->fd;
  const auto& c = B.m->cfg;
  f.k = c[0]; f.emb = c[1]; f.T = c[2]; f.heads = c[3]; f.nscales = c[4];
  for (int s = 0; s < f.nscales; ++s) f.kscales[s] = c[5 + s];
  for (int s = 0; s < f.nscales; ++s) {
    const std::string p = "encoder.multi_scale_first_conv." + std::to_string(s);
    B.layer(f.first[s], p + ".0", p + ".1", 64, 6, false);
  }
  B.layer(f.fusion, "encoder.scale_fusion.0", "encoder.scale_fusion.1", 64, 64 * f.nscales, false);
  B.neuron(f.blk[0], {"encoder.snn_blocks.0"}, 64, true);
  B.neuron(f.blk[1], {"encoder.snn_blocks.1"}, 128, true);
  B.neuron(f.blk[2], {"encoder.snn_blocks.2"}, 256, false);
  B.neuron(f.blk[3], {"encoder.snn_blocks.3"}, 512, false);
  const int cin[3] = {64, 128, 256}, cout[3] = {128, 256, 512};
  for (int b = 0; b < 3; ++b) {
    const std::string p = "encoder.conv_blocks." + std::to_string(b);
    B.layer(f.conv[b], p + ".0", p + ".1", cout[b], 2 * cin[b], false);
    if (auto* w = B.get(p + ".0.weight", (size_t)cout[b] * 2 * cin[b])) {
      // W = [Wa | Wb] acts on cat(x_j - x_i, x_j):  rows [0,Cout) = Wa + Wb (applied to x_j), rows [Cout,2Cout) = Wa (to x_i)
      std::vector<float> wf((size_t)2 * cout[b] * cin[b]);
      for (int o = 0; o < cout[b]; ++o)
        for (int i = 0; i < cin[b]; ++i) {
          const float wa = (*w)[(size_t)o * 2 * cin[b] + i], wb = (*w)[(size_t)o * 2 * cin[b] + cin[b] + i];
          wf[(size_t)o * cin[b] + i] = wa + wb;
          wf[((size_t)cout[b] + o) * cin[b] + i] = wa;
        }
      f.convf[b].N = 2 * cout[b]; f.convf[b].K = cin[b];
      B.put_w(f.convf[b], wf.data(), wf.size());
    }
  }
  B.layer(f.msc, "encoder.multi_scale_conv.0", "encoder.multi_scale_conv.1", f.emb, 960, false);
  B.neuron(f.snn_fc, {"encoder.snn_fc"}, f.emb, false);
  if (auto* w = B.get("encoder.temporal_integration.weights", f.T)) {
    std::vector<float> sm(f.T);
    float mx = -INFINITY;
    for (float v : *w) mx = fmaxf(mx, v);
    float sum = 0.0f;
    for (int t = 0; t < f.T; ++t) { sm[t] = expf((*w)[t] - mx); sum += sm[t]; }
    for (int t = 0; t < f.T; ++t) sm[t] /= sum;
    B.put(sm.data(), f.T, &f.tw);
  }
  const std::string d = "distance_decoder.";
  B.layer(f.fc_in, d + "fc_in.0", d + "fc_in.1", 256, f.emb, true);
  const int hin[2] = {256, 128}, hout[2] = {128, 64};
  for (int r = 0; r < 2; ++r) {
    const std::string p = d + "residual_blocks." + std::to_string(r) + ".";
    B.layer(f.rb_fc0[r], p + "fc.0", p + "fc.1", hout[r], hin[r], true);
    B.layer(f.rb_fc1[r], p + "fc.4", p + "fc.5", hout[r], hout[r], true);
    B.layer(f.rb_res[r], p + "res_proj", "", hout[r], hin[r], true);
  }
  B.layer(f.to_qkv, d + "attention.to_qkv", "", 192, 64, true);
  B.layer(f.to_out, d + "attention.to_out.0", "", 64, 64, true);
  B.raw(d + "attention.norm.weight", 64, &f.ln_w);
  B.raw(d + "attention.norm.bias", 64, &f.ln_b);
  B.layer(f.fc_hidden, d + "fc_hidden.0", d + "fc_hidden.1", 32, 64, true);
  B.layer(f.fc_dist, d + "fc_distance", "", 1, 32, true);
}

}  // namespace

namespace sapcu {

void split_weights(const float* w, size_t n, WeightSplit* s) {
  s->hi.resize(n); s->lo.resize(n);
  for (size_t i = 0; i < n; ++i) {
    uint32_t b; memcpy(&b, &w[i], 4);
    if ((b & 0x7F800000u) != 0x7F800000u) b = (b + 0x1000u) & 0xFFFFE000u;
    float h; memcpy(&h, &b, 4);
    s->hi[i] = h; s->lo[i] = w[i] - h;                                    // lo exact in fp32
  }
  // fp16 (hi, lo) of w * 2^e with max |w| * 2^e in [2^13, 2^14): both halves stay in fp16's normal range for every
  // weight within 2^-9 of the largest one, smaller ones keep 6e-8 absolute (scaled) precision
  float mx = 0.0f;
  for (size_t i = 0; i < n; ++i) if (std::isfinite(w[i])) mx = std::max(mx, std::fabs(w[i]));
  int e = 0;
  if (mx > 0.0f) { int ex; std::frexp(mx, &ex); e = 14 - ex; }          // mx = f * 2^ex, f in [0.5, 1)
  const float sc = std::ldexp(1.0f, e);
  s->h.assign((n + 1) & ~(size_t)1, 0); s->l.assign((n + 1) & ~(size_t)1, 0);
  for (size_t i = 0; i < n; ++i) {
    const float ws = w[i] * sc;                                           // exact (power of two)
    const uint16_t h = f32_to_f16_rn(ws);
    s->h[i] = h; s->l[i] = f32_to_f16_rn(ws - f16_to_f32(h));
  }
  s->winv = std::ldexp(1.0f, -e);
}

void lif_table_pack(const float* np4, int C, int T, LifTablePacked* out) {
  LifTableHost t;
  lif_table_build(np4, C, T, &t);
  const uint32_t stride = (t.max_block_bytes + 255u) / 256u * 256u;
  out->img.assign((size_t)stride / 4 * t.blocks.size(), 0.0f);
  for (size_t b = 0; b < t.blocks.size(); ++b)
    memcpy(reinterpret_cast<uint8_t*>(out->img.data()) + b * stride, t.image.data() + t.blocks[b].off_bytes, t.blocks[b].bytes);
  out->stride = stride; out->usable = t.usable; out->max_err = (float)t.max_err;
}

}  // namespace sapcu

extern "C" {

sapcu_model* sapcu_model_create(int kind, const int32_t* cfg, int ncfg) {
  if (kind != SAPCU_MODEL_FN && kind != SAPCU_MODEL_FD) { set_error("model_create: unknown kind %d", kind); return nullptr; }
  if (!cfg) { set_error("model_create: null cfg"); return nullptr; }
  if (kind == SAPCU_MODEL_FN) {
    if (ncfg != 6) { set_error("model_create(fn): expected 6 cfg ints {k0,k1,k2,emb,T_enc,heads}, got %d", ncfg); return nullptr; }
    for (int i = 0; i < 3; ++i) if (cfg[i] < 1 || cfg[i] > 32) { set_error("model_create(fn): k_values[%d]=%d outside [1,32]", i, cfg[i]); return nullptr; }
    if (cfg[3] < 16 || cfg[3] % 16) { set_error("model_create(fn): emb_dims=%d must be a positive multiple of 16", cfg[3]); return nullptr; }
    if (cfg[4] < 1 || cfg[5] < 1 || 128 % cfg[5]) { set_error("model_create(fn): bad time_steps_enc=%d / num_heads=%d", cfg[4], cfg[5]); return nullptr; }
  } else {
    if (ncfg < 6 || ncfg != 5 + cfg[4] || cfg[4] < 1 || cfg[4] > 8) { set_error("model_create(fd): expected {k,emb,T,heads,ns,k_scales[ns<=8]}"); return nullptr; }
    if (cfg[0] < 1 || cfg[1] < 16 || cfg[1] % 16 || cfg[2] < 1 || cfg[3] < 1 || cfg[3] > 16 || 64 % cfg[3]) { set_error("model_create(fd): bad hyper-parameters"); return nullptr; }
    for (int s = 0; s < cfg[4]; ++s) if (cfg[5 + s] < 1 || cfg[5 + s] > 64 || (s && cfg[5 + s] < cfg[4 + s])) { set_error("model_create(fd): k_scales must be ascending within [1,64]"); return nullptr; }
  }
  sapcu_model* m = new (std::nothrow) sapcu_model();
  if (!m) { set_error("model_create: out of host memory"); return nullptr; }
  m->kind = kind;
  m->cfg.assign(cfg, cfg + ncfg);
  return m;
}

int sapcu_model_set_tensor(sapcu_model* m, const char* name, const float* h_data, int64_t numel) {
  SAPCU_REQUIRE(m && name && (h_data || numel == 0) && numel >= 0, "model_set_tensor: bad argument");
  if (m->finalized) { set_error("model_set_tensor: model already finalized"); return SAPCU_ESTATE; }
  m->host[name].assign(h_data, h_data + numel);
  return 0;
}

int sapcu_model_finalize(sapcu_model* m) {
  SAPCU_REQUIRE(m, "model_finalize: null model");
  if (m->finalized) return 0;
  Builder B; B.m = m;
  if (m->kind == SAPCU_MODEL_FN) build_fn(B); else build_fd(B);
  if (!B.err.empty()) { set_error("model_finalize: %s", B.err.c_str()); return SAPCU_ESTATE; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_error("model_finalize: no CUDA device (this library has no CPU fallback)");
    return SAPCU_ECUDA;
  }
  SAPCU_CUDA_CHECK(cudaGetDevice(&m->device));
  const size_t n = (B.blob.size() + 63) / 64 * 64;
  B.blob.resize(n);
  SAPCU_CUDA_CHECK(cudaMalloc(&m->dev, n * sizeof(float)));
  SAPCU_CUDA_CHECK(cudaMemcpy(m->dev, B.blob.data(), n * sizeof(float), cudaMemcpyHostToDevice));
  m->dev_floats = n;
  for (auto& fx : B.fixes) *fx.dst = m->dev + fx.off;
  m->host.clear();
  m->finalized = true;
  return 0;
}

void sapcu_model_destroy(sapcu_model* m) {
  if (!m) return;
  if (m->dev) {
    // free on the device the weights live on, whichever device the caller has current, and leave the caller's device as it was
    int cur = -1;
    const bool other = cudaGetDevice(&cur) == cudaSuccess && cur != m->device && cudaSetDevice(m->device) == cudaSuccess;
    cudaFree(m->dev);
    if (other) cudaSetDevice(cur);
  }
  delete m;
}

}  // extern "C"
