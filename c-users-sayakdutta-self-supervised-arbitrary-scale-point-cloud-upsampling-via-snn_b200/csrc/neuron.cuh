// Membrane recurrences of the LIF / EIF neurons, evaluated entirely in registers.
//
// Semantics follow the reference neuron step in eval mode
// (fn/snn_coder.py:109-153, fd/snn_coder.py:117-155 LIF, fd/snn_coder.py:223-275 EIF):
//   x  = x * float(rho <= 0)
//   m  = m*d*(1-rho) + x (+ e)         e = dT*exp(clamp((m_prev - th_rh)/(dT+1e-6), -5, 5))   [EIF]
//   s  = 0.5*exp(-(vc^2)/2)/sqrt(2pi) + 0.5*sigmoid(10*vc),  vc = clamp(m - th, -10, 10)
//   m  = m*(1-s) ; rho = rho*r + s ; th = th + a*s ; th = th0 + (th - th0)*0.95
// The soft spike s is strictly positive, so rho > 0 after the first step and the gate
// `float(rho <= 0)` is closed for every later step (SURVEY.md fact 4); the gate is still
// evaluated literally here so the kernels stay faithful for any state.
#pragma once
#include <cuda_runtime.h>

namespace sapcu {

struct NeuronParams {   // per channel, already clamped to the reference's ranges
  float d;     // membrane_decay   in [0.1, 0.99]
  float a;     // threshold_adapt  in [0.001, 0.1]
  float r;     // refractory_decay in [0.1, 0.95]
  float th0;   // threshold_base
};
struct EifParams {      // per channel, clamped
  float dT;    // delta_T  in [0.1, 5]
  float thrh;  // theta_rh in [0.1, 2]
};

__device__ __forceinline__ float exp2f_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ordered flavours: `volatile` keeps their relative program order, which pins the phase-major MUFU schedule of
// lif_chain_vec_fast (ptxas otherwise re-serialises half of the elements)
__device__ __forceinline__ float exp2f_approx_ord(float x) {
  float y;
  asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx_ord(float x) {
  float y;
  asm volatile("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// also the reciprocal of the fast LIF step, where x = 2 + 2*exp2(.) may overflow to +inf (v << 0): the answer is then 0
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// PRECISE=true : libdevice expf (<= 1 ulp) -- the fp32 parity mode
// PRECISE=false: ex2.approx based __expf     -- the tensor-core mode
template <bool PRECISE>
__device__ __forceinline__ float sapcu_exp(float x) {
  if (PRECISE) return expf(x);
  return __expf(x);
}

// In PRECISE mode every product/sum is a separately rounded fp32 operation (the reference runs one
// ATen kernel per operation, so nothing is ever contracted into an FMA); the fast mode lets the
// compiler contract.
template <bool PRECISE> __device__ __forceinline__ float mulp(float a, float b) {
  return PRECISE ? __fmul_rn(a, b) : a * b;
}
template <bool PRECISE> __device__ __forceinline__ float addp(float a, float b) {
  return PRECISE ? __fadd_rn(a, b) : a + b;
}
template <bool PRECISE> __device__ __forceinline__ float subp(float a, float b) {
  return PRECISE ? __fsub_rn(a, b) : a - b;
}

template <bool PRECISE>
__device__ __forceinline__ float spike_fn(float v) {
  const float vc = fminf(fmaxf(v, -10.0f), 10.0f);
  const float inv_sqrt_2pi = 1.0f / 2.5066282746310002f;
  // CPU torch divides by the python scalar sqrt(2*pi) (rounded to fp32); the fast mode multiplies by 1/x
  const float e = sapcu_exp<PRECISE>(-mulp<PRECISE>(mulp<PRECISE>(vc, vc), 0.5f));
  const float g = PRECISE ? __fdiv_rn(e, 2.5066282746310002f) : e * inv_sqrt_2pi;
  float sg;
  if (PRECISE) sg = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-__fmul_rn(10.0f, vc))));
  else         sg = __fdividef(1.0f, 1.0f + __expf(-(10.0f * vc)));
  return addp<PRECISE>(mulp<PRECISE>(0.5f, g), mulp<PRECISE>(0.5f, sg));
}

struct NeuronState { float m, th, rho; };

__device__ __forceinline__ NeuronState neuron_init(const NeuronParams& p) {
  NeuronState s; s.m = 0.0f; s.th = p.th0; s.rho = 0.0f; return s;
}

// One step; returns the soft spike.
template <bool EIF, bool PRECISE>
__device__ __forceinline__ float neuron_step(float x, NeuronState& st, const NeuronParams& p,
                                             const EifParams& e) {
  float ex = 0.0f;
  if (EIF) {
    float arg = PRECISE ? __fdiv_rn(__fsub_rn(st.m, e.thrh), __fadd_rn(e.dT, 1e-6f))
                        : __fdividef(st.m - e.thrh, e.dT + 1e-6f);
    arg = fminf(fmaxf(arg, -5.0f), 5.0f);
    ex = mulp<PRECISE>(e.dT, sapcu_exp<PRECISE>(arg));
  }
  const float gate = (st.rho <= 0.0f) ? 1.0f : 0.0f;
  x = mulp<PRECISE>(x, gate);
  float m = addp<PRECISE>(mulp<PRECISE>(mulp<PRECISE>(st.m, p.d), subp<PRECISE>(1.0f, st.rho)), x);
  if (EIF) m = addp<PRECISE>(m, ex);
  const float s = spike_fn<PRECISE>(subp<PRECISE>(m, st.th));
  st.m = mulp<PRECISE>(m, subp<PRECISE>(1.0f, s));
  st.rho = addp<PRECISE>(mulp<PRECISE>(st.rho, p.r), s);
  const float th = addp<PRECISE>(st.th, mulp<PRECISE>(p.a, s));
  st.th = addp<PRECISE>(p.th0, mulp<PRECISE>(subp<PRECISE>(th, p.th0), 0.95f));
  return s;
}

// LIF^T(u): T steps from the zero state, the emitted spike fed back as the next input
// (fn/snn_coder.py:319-320 and every other `for t in range(T)` loop of the fn model).
template <bool PRECISE>
__device__ __forceinline__ float lif_chain(float u, const NeuronParams& p, int T) {
  NeuronState st = neuron_init(p);
  EifParams e{1.0f, 1.0f};
  float s = u;
#pragma unroll 1
  for (int t = 0; t < T; ++t) s = neuron_step<false, PRECISE>(s, st, p, e);
  return s;
}

// LIF^T on NV independent accumulators of one channel (interleaved for ILP); fast-math flavour.
// Algebraically identical to neuron_step, re-associated for the FMA pipe (12 FP + 3 MUFU per element-step):
//   * the soft spike is > 0, so the refractory gate is open at step 0 only: later steps take no input
//     (the +-10 clamp of the reference only matters below 1e-22 and is dropped here);
//   * m*d*(1-rho) = md - md*rho ; m*(1-s) = mm - mm*s ; 0.5*sigmoid(10v) = 1/(2 + 2*exp(-10v));
//   * th' = th0 + (th + a*s - th0)*0.95 = 0.95*th + (0.95*a*s + 0.05*th0).
template <int NV>
__device__ __forceinline__ void lif_chain_vec_fast(float (&u)[NV], const NeuronParams& p, int T) {
  float m[NV], th[NV], rho[NV];
  const float c_g = 0.5f / 2.5066282746310002f;        // 0.5 / sqrt(2 pi)
  const float k_g = -0.5f * 1.4426950408889634f;       // exp(-v^2/2) = 2^(k_g v^2)
  const float k_s = -10.0f * 1.4426950408889634f;      // exp(-10 v)  = 2^(k_s v)
  const float a95 = 0.95f * p.a, c05 = 0.05f * p.th0;
#pragma unroll
  for (int i = 0; i < NV; ++i) {                        // step 0: m = u, th = th0, rho = 0
    const float mm = u[i];
    const float v = mm - p.th0;
    const float g = exp2f_approx((k_g * v) * v);
    const float e = exp2f_approx(k_s * v);
    const float s = fmaf(c_g, g, rcp_approx(fmaf(2.0f, e, 2.0f)));
    m[i] = fmaf(-mm, s, mm);
    rho[i] = s;
    th[i] = fmaf(0.95f, p.th0, fmaf(a95, s, c05));
    u[i] = s;
  }
#pragma unroll 1
  for (int t = 1; t < T; ++t) {
    // phase-major over the NV elements: all EX2s are issued back to back, then all RCPs, so the MUFU pipe always
    // has independent work queued instead of one element's EX2 -> FFMA -> RCP -> FFMA dependency chain
    float mm[NV], g[NV], e[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float md = m[i] * p.d;
      mm[i] = fmaf(-md, rho[i], md);
      const float v = mm[i] - th[i];
      g[i] = (k_g * v) * v;
      e[i] = k_s * v;
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) e[i] = exp2f_approx_ord(e[i]);
#pragma unroll
    for (int i = 0; i < NV; ++i) g[i] = exp2f_approx_ord(g[i]);
#pragma unroll
    for (int i = 0; i < NV; ++i) e[i] = rcp_approx(fmaf(2.0f, e[i], 2.0f));
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float s = fmaf(c_g, g[i], e[i]);
      m[i] = fmaf(-mm[i], s, mm[i]);
      rho[i] = fmaf(rho[i], p.r, s);
      th[i] = fmaf(0.95f, th[i], fmaf(a95, s, c05));
      u[i] = s;
    }
  }
}

// SAPCU_MODE_FAST flavour of lif_chain_vec_fast: 0.5*sigmoid(10v) = 0.25 + 0.25*tanh(5v) with MUFU.TANH (tanh.approx.f32,
// relative error 2^-11) -- 2 MUFU operations per element-step instead of 3, 11 FP instead of 12.  Deviation from the exact
// chain <= 1.5e-4 absolute per step (reported with the fast mode's other deviations).
__device__ __forceinline__ float tanh_approx_ord(float x) {
  float y;
  asm volatile("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
template <int NV>
__device__ __forceinline__ void lif_chain_vec_fast2(float (&u)[NV], const NeuronParams& p, int T) {
  float m[NV], th[NV], rho[NV];
  const float c_g = 0.5f / 2.5066282746310002f, k_g = -0.5f * 1.4426950408889634f;
  const float a95 = 0.95f * p.a, c05 = 0.05f * p.th0;
#pragma unroll 1
  for (int t = 0; t < T; ++t) {
    float mm[NV], g[NV], e[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      if (t == 0) { mm[i] = u[i]; th[i] = p.th0; rho[i] = 0.0f; }
      else { const float md = m[i] * p.d; mm[i] = fmaf(-md, rho[i], md); }
      const float v = mm[i] - th[i];
      g[i] = (k_g * v) * v;
      e[i] = 5.0f * v;
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) e[i] = tanh_approx_ord(e[i]);
#pragma unroll
    for (int i = 0; i < NV; ++i) g[i] = exp2f_approx_ord(g[i]);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float s = fmaf(c_g, g[i], fmaf(0.25f, e[i], 0.25f));
      m[i] = fmaf(-mm[i], s, mm[i]);
      rho[i] = fmaf(rho[i], p.r, s);
      th[i] = fmaf(0.95f, th[i], fmaf(a95, s, c05));
      u[i] = s;
    }
  }
}

// One re-associated step (fast-math flavour of neuron_step) for kernels that need every step's spike.
// FIRST: the step from the zero state (m = 0, th = th0, rho = 0) with input u; later steps take no input
// (closed refractory gate).  Derived constants are passed in `k`.
struct FastNeuronK { float d, r, a95, c05, th0, dT, thrh, inv_dT; };
__device__ __forceinline__ FastNeuronK fast_neuron_k(const NeuronParams& p, const EifParams& e) {
  FastNeuronK k;
  k.d = p.d; k.r = p.r; k.a95 = 0.95f * p.a; k.c05 = 0.05f * p.th0; k.th0 = p.th0;
  k.dT = e.dT; k.thrh = e.thrh; k.inv_dT = 1.0f / (e.dT + 1e-6f);
  return k;
}
template <bool EIF, bool FIRST>
__device__ __forceinline__ float neuron_step_fast(float u, float& m, float& th, float& rho, const FastNeuronK& k) {
  const float c_g = 0.5f / 2.5066282746310002f, k_g = -0.5f * 1.4426950408889634f, k_s = -10.0f * 1.4426950408889634f;
  float mm;
  if (FIRST) {
    mm = u;
    if (EIF) mm += k.dT * exp2f_approx(fminf(fmaxf(-k.thrh * k.inv_dT, -5.0f), 5.0f) * 1.4426950408889634f);
  } else {
    const float md = m * k.d;
    mm = fmaf(-md, rho, md);
    if (EIF) mm += k.dT * exp2f_approx(fminf(fmaxf((m - k.thrh) * k.inv_dT, -5.0f), 5.0f) * 1.4426950408889634f);
  }
  const float v = mm - (FIRST ? k.th0 : th);
  const float g = exp2f_approx((k_g * v) * v);
  const float e = exp2f_approx(k_s * v);
  const float s = fmaf(c_g, g, rcp_approx(fmaf(2.0f, e, 2.0f)));
  m = fmaf(-mm, s, mm);
  rho = FIRST ? s : fmaf(rho, k.r, s);
  th = fmaf(0.95f, FIRST ? k.th0 : th, fmaf(k.a95, s, k.c05));
  return s;
}

// PRECISE: the reference-faithful step per element; otherwise the fast-math interleaved form above
template <int NV, bool PRECISE>
__device__ __forceinline__ void lif_chain_vec(float (&u)[NV], const NeuronParams& p, int T) {
  if (PRECISE) {
    NeuronState st[NV];
    EifParams e{1.0f, 1.0f};
#pragma unroll
    for (int i = 0; i < NV; ++i) st[i] = neuron_init(p);
#pragma unroll 1
    for (int t = 0; t < T; ++t) {
#pragma unroll
      for (int i = 0; i < NV; ++i) u[i] = neuron_step<false, true>(u[i], st[i], p, e);
    }
  } else {
    lif_chain_vec_fast<NV>(u, p, T);
  }
}

__device__ __forceinline__ float act_leaky(float x) { return x >= 0.0f ? x : 0.2f * x; }
__device__ __forceinline__ float act_gelu(float x) {   // exact (erf) GELU, torch default
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f));
}

}  // namespace sapcu
