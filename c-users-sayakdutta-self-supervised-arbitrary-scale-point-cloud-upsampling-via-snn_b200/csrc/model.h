// Model handle: host-side weight registry, folded device parameters and the per-chunk workspace plans
// of the fn / fd forwards.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <map>
#include <string>
#include <vector>
#include "common.cuh"

namespace sapcu {

struct Layer {     // 1x1 conv / Linear (+ folded eval BatchNorm):  y = (x W^T + bias) * scale + shift
  const float* W = nullptr; const float* Whi = nullptr; const float* Wlo = nullptr; const float* bias = nullptr; const float* scale = nullptr; const float* shift = nullptr;
  int N = 0, K = 0;
  // fp16 (hi, lo) split of W * 2^wexp for the fp16x3 tensor-core path (inputs known to lie in the LIF output range);
  // the pointers address raw half data inside the float blob, winv = 2^-wexp
  const float* Wh = nullptr; const float* Wl = nullptr; float winv = 1.0f;
};
struct Neuron {    // clamped per-channel parameters: np = [4][C] (d, a, r, th0); ep = [2][C] (dT, th_rh) for EIF
  const float* np = nullptr; const float* ep = nullptr; int C = 0;
  // SAPCU_MODE_FAST: tabulated LIF^T chain (lif_table.cuh), one image of `tab_stride` bytes per 128-channel block
  const float* tab = nullptr; uint32_t tab_stride = 0; int tab_T = 0; bool tab_ok = false; float tab_err = 0.0f;
};

// The tensor-core copies of one weight matrix w [n] (host fp32), as sapcu_model_finalize uploads them: tf32 (hi, lo) with
// hi = w rounded to 10 mantissa bits (round-to-nearest, ties away) and lo = w - hi, and fp16 (hi, lo) of w * 2^e with
// max |w| * 2^e in [2^13, 2^14), winv = 2^-e.  h / l are padded to an even count (the float blob's granularity).
struct WeightSplit { std::vector<float> hi, lo; std::vector<uint16_t> h, l; float winv = 1.0f; };
void split_weights(const float* w, size_t n, WeightSplit* out);
// The LIF^T table of np4 ([4][C] rows {d, a, r, th0}, clamped) for T steps, re-packed with one fixed stride per 128-channel
// block so that a kernel finds its block from (base, stride, block index) alone
struct LifTablePacked { std::vector<float> img; uint32_t stride = 0; bool usable = false; float max_err = 0.0f; };
void lif_table_pack(const float* np4, int C, int T, LifTablePacked* out);

struct FnBlock {
  int D = 0, k = 0;
  Layer fc1, qkv, fc_delta, fc_delta2, fc_gamma, fc_gamma2, out_proj, fc2;
  Neuron snn1, snn_qkv, snn_delta, snn_delta2, snn_gamma;
};
struct FnNet {
  int kvals[3] = {0, 0, 0}; int emb = 0, T_enc = 0, heads = 0;
  Layer conv1, conv_final, fc_out, mlp[3], head; Neuron snn_init, snn_final;
  const float* ln_w = nullptr; const float* ln_b = nullptr;
  FnBlock blk[3];
};
struct FdNet {
  int k = 0, emb = 0, T = 0, heads = 0, nscales = 0; int kscales[8] = {0};
  Layer first[8], fusion, conv[3], msc;
  Layer convf[3];              // factorised EdgeConv weights [(Wa+Wb) ; Wa] : [2*Cout, Cin] (tensor-core mode)
  Neuron blk[4], snn_fc;
  const float* tw = nullptr;   // softmax(temporal weights) [T]
  Layer fc_in, rb_fc0[2], rb_fc1[2], rb_res[2], to_qkv, to_out, fc_hidden, fc_dist;
  const float* ln_w = nullptr; const float* ln_b = nullptr;
};

}  // namespace sapcu

struct sapcu_model {
  int kind = 0;
  std::vector<int> cfg;
  std::map<std::string, std::vector<float>> host;   // raw state_dict tensors (host fp32)
  bool finalized = false;
  int device = -1;                                   // CUDA device current at finalize: the one `dev` lives on
  float* dev = nullptr;                              // one device allocation holding every derived array
  size_t dev_floats = 0;
  sapcu::FnNet fn;
  sapcu::FdNet fd;
  // storage format of the tapped spike tensors in the most recent forward on this handle (sapcu_model_tap_format)
  mutable std::atomic<int> tap_gamma{0}, tap_delta2{0}, tap_spk{0}, tap_snn1{0};
};
