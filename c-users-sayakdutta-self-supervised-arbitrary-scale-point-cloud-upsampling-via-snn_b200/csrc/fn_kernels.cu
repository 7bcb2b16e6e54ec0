// Non-GEMM kernels of the fn (normal estimation) forward, fn/snn_coder.py:294-396,430-476,542-549.
//   pointwise3_lif : 3 -> C pointwise conv + BN + LIF^T, on points (conv1, :453-456) or on edge offsets
//                    xyz_i - xyz_j (fc_delta, :308-310,355-358); K=3 is too thin for a GEMM tile
//   attn_out       : softmax over the k neighbours of a/sqrt(head_dim) and sum_j a_ij (v_j + pos_ij) (:379-391)
//   group_max      : max over the M points of a patch (adaptive_max_pool1d, :472; fd/snn_coder.py:479)
//   fn_head        : Linear 256->3, LayerNorm(3), L2 normalise (:545-548)
#include <cuda_fp16.h>
#include "common.cuh"
#include "kernels.h"
#include "neuron.cuh"
#include "lif_table.cuh"

namespace sapcu {

template <bool EDGE, bool PRECISE>
__global__ void pointwise3_lif_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ idx, int kk, int ldi,
                                      int Mpts, int64_t rows, int C, const float* __restrict__ W,
                                      const float* __restrict__ bias, const float* __restrict__ scale,
                                      const float* __restrict__ shift, const float* __restrict__ np, int T,
                                      float* __restrict__ out) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= rows * C) return;
  const int64_t row = e / C;
  const int c = (int)(e - row * C);
  float x0, x1, x2;
  if (EDGE) {
    const int64_t pt = row / kk;
    const int j = (int)(row - pt * kk);
    const int64_t nb = (pt / Mpts) * Mpts + idx[pt * ldi + j];
    x0 = __fsub_rn(xyz[3 * pt], xyz[3 * nb]);
    x1 = __fsub_rn(xyz[3 * pt + 1], xyz[3 * nb + 1]);
    x2 = __fsub_rn(xyz[3 * pt + 2], xyz[3 * nb + 2]);
  } else {
    x0 = xyz[3 * row]; x1 = xyz[3 * row + 1]; x2 = xyz[3 * row + 2];
  }
  float y = fmaf(W[3 * c + 2], x2, fmaf(W[3 * c + 1], x1, __fmul_rn(W[3 * c], x0)));
  y = __fadd_rn(y, bias[c]);
  y = __fadd_rn(__fmul_rn(y, scale[c]), shift[c]);
  NeuronParams p{np[c], np[C + c], np[2 * C + c], np[3 * C + c]};
  out[e] = lif_chain<PRECISE>(y, p, T);
}

// fc_delta on edge offsets + BN + LIF^T.  One CTA = one patch x 128 channels: the patch's coordinates and graph are
// staged in shared memory once, the per-channel parameters live in registers, and the CTA walks the patch's Mpts*kk
// edges in groups of EPL_G: the offsets xyz_i - xyz_j of the NEXT group are written to the other half of a double
// buffer before the T-step recurrence of the current one (8 interleaved edges per thread), so the single barrier per
// group never waits on memory and the MUFU pipe stays fed.
constexpr int EPL_G = 72;     // = 6 x 12 = 4 x 18 = 3 x 24 edges; a multiple of the 8-edge vector
template <bool PRECISE>
__global__ void __launch_bounds__(128)
edge_pos_lif_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ idx, int kk, int ldi, int Mpts, int C,
                    const float* __restrict__ W, const float* __restrict__ bias, const float* __restrict__ scale,
                    const float* __restrict__ shift, const float* __restrict__ np, int T, float* __restrict__ out,
                    int out_h2, int64_t plane) {
  extern __shared__ float esm[];
  float* xs = esm;                                              // [Mpts][3]
  float* pd = xs + 3 * Mpts;                                    // [2][EPL_G][3]
  uint8_t* nbs = reinterpret_cast<uint8_t*>(pd + 2 * EPL_G * 3);  // [Mpts][kk] local neighbour indices (Mpts <= 256)
  const int tid = threadIdx.x;
  const int64_t patch0 = (int64_t)blockIdx.x * Mpts;
  for (int i = tid; i < 3 * Mpts; i += 128) xs[i] = xyz[3 * patch0 + i];
  for (int pt = tid >> 5; pt < Mpts; pt += 4)
    for (int j = tid & 31; j < kk; j += 32) nbs[pt * kk + j] = (uint8_t)idx[(patch0 + pt) * ldi + j];
  __syncthreads();
  const int EP = Mpts * kk;
  const int G = (EP + EPL_G - 1) / EPL_G;
  auto stage = [&](int g, int buf) {
    const int e = g * EPL_G + tid;
    if (tid < EPL_G) {
      float d0 = 0.f, d1 = 0.f, d2 = 0.f;
      if (e < EP) {
        const int pt = e / kk;
        const int nb = nbs[e];
        d0 = __fsub_rn(xs[3 * pt], xs[3 * nb]);
        d1 = __fsub_rn(xs[3 * pt + 1], xs[3 * nb + 1]);
        d2 = __fsub_rn(xs[3 * pt + 2], xs[3 * nb + 2]);
      }
      float* q = pd + (buf * EPL_G + tid) * 3;
      q[0] = d0; q[1] = d1; q[2] = d2;
    }
  };
  const int g0 = blockIdx.z, gstep = gridDim.z;                  // grid.z CTAs share a patch slab (shorter-lived CTAs)
  if (g0 < G) stage(g0, 0);
  __syncthreads();
  const int c = blockIdx.y * 128 + tid;
  const bool cv = c < C;
  const int cc = cv ? c : 0;
  const float w0 = W[3 * cc], w1 = W[3 * cc + 1], w2 = W[3 * cc + 2];
  const float bi = bias[cc], sc = scale[cc], sh = shift[cc];
  const NeuronParams p{np[cc], np[C + cc], np[2 * C + cc], np[3 * C + cc]};
  float* o = out + patch0 * kk * (int64_t)C + c;
  int buf = 0;
#pragma unroll 1
  for (int g = g0; g < G; g += gstep, buf ^= 1) {
    if (g + gstep < G) stage(g + gstep, buf ^ 1);
    const float* q = pd + buf * EPL_G * 3;
    const int n = (EP - g * EPL_G) < EPL_G ? (EP - g * EPL_G) : EPL_G;
    if (cv) {
#pragma unroll 1
      for (int h = 0; h < EPL_G; h += 8) {
        if (h >= n) break;
        float u[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float y = fmaf(w2, q[(h + j) * 3 + 2], fmaf(w1, q[(h + j) * 3 + 1], __fmul_rn(w0, q[(h + j) * 3])));
          y = __fadd_rn(y, bi);
          u[j] = __fadd_rn(__fmul_rn(y, sc), sh);
        }
        lif_chain_vec<8, PRECISE>(u, p, T);
        if (out_h2) {                                             // fp16 (hi, lo) planes of y * 2^13 (tc_ptx.cuh)
          __half* hp = reinterpret_cast<__half*>(out) + (patch0 * kk + g * EPL_G + h) * (int64_t)C + c;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (h + j < n) {
              const float ys = u[j] * 8192.0f;
              const __half hv = __float2half_rn(ys);
              hp[(int64_t)j * C] = hv;
              hp[plane + (int64_t)j * C] = __float2half_rn(ys - __half2float(hv));
            }
          }
          continue;
        }
        float* og = o + (int64_t)(g * EPL_G + h) * C;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (h + j < n) og[(int64_t)j * C] = u[j];
      }
    }
    __syncthreads();
  }
}


// SAPCU_MODE_FAST flavour of edge_pos_lif: fc_delta (K = 3) + BN + LIF^T on the edge offsets, one fp16 plane of y * 2^13 out.
// Persistent CTAs (grid.y = 128-channel block, grid.x strides over the patches): the block's tabulated LIF^T chain
// (lif_table.cuh) is copied to shared memory once; per patch the coordinates and the graph are staged, the Mpts*kk edge
// offsets are expanded into shared memory, and 4 threads per channel walk the edges (lane = channel, so a warp's 32 stores
// of a row are 64 contiguous bytes).  LTAB = 0: no usable table -- the reduced-MUFU recurrence instead.
constexpr int EPF_THREADS = 512;
// LIF^T chain of NV rows of one channel from x = BN(.) - theta0 (LTAB: the table at lt_desc, exact chain out of its range) or
// from u = BN(.) (reduced-MUFU recurrence)
template <int LTAB, int NV>
__device__ __forceinline__ void lif_rows(float (&u)[NV], const NeuronParams& p, int T, uint32_t lt_desc) {
  if (LTAB) {
    float x0[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) x0[j] = u[j];
    if (lif_table_eval_vec<NV>(u, lt_desc)) {
#pragma unroll
      for (int j = 0; j < NV; ++j) if (lif_table_oob(x0[j])) u[j] = lif_chain<false>(x0[j] + p.th0, p, T);
    }
  } else {
    lif_chain_vec_fast2<NV>(u, p, T);
  }
}
// fc_delta (K = 3) with BN folded into (w0, w1, w2, b0), then the LIF^T chain: the same fmaf chain for edge and pair rows
template <int LTAB>
__device__ __forceinline__ void pos_lif4(const float4 (&d)[4], float w0, float w1, float w2, float b0, const NeuronParams& p, int T,
                                         uint32_t lt_desc, float (&u)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) u[j] = fmaf(w2, d[j].z, fmaf(w1, d[j].y, fmaf(w0, d[j].x, b0)));
  lif_rows<LTAB, 4>(u, p, T, lt_desc);
}
// rows j < n of y * 2^13 as an fp16 plane (+ the lo plane `plane` halfs behind it when PL2), row stride C
template <int PL2, int NV>
__device__ __forceinline__ void store_h(__half* o, int64_t C, int64_t plane, const float (&u)[NV], int n) {
#pragma unroll
  for (int j = 0; j < NV; ++j)
    if (j < n) {
      const float ys = u[j] * 8192.0f;
      const __half hv = __float2half_rn(ys);
      o[j * C] = hv;
      if (PL2) o[plane + j * C] = __float2half_rn(ys - __half2float(hv));
    }
}
// PL2: also write the lo plane (y * 2^13 - hi) `plane` halfs behind the hi plane -- the (hi, lo) hand-over format of the
// parity-grade tensor-core mode, whose LIF^T chains may use the same tables.
template <int LTAB, int CT, int PL2 = 0>     // CT: compile-time channel count (row stride of the output: store offsets become immediates), 0 = run-time
__global__ void __launch_bounds__(EPF_THREADS)
edge_pos_lif_fast_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ idx, int kk, int ldi, int Mpts, int C_rt,
                         int64_t S, const float* __restrict__ W, const float* __restrict__ bias,
                         const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ np,
                         int T, __half* __restrict__ out, const uint8_t* __restrict__ tab, uint32_t tab_stride, int64_t plane) {
  extern __shared__ __align__(16) uint8_t epf_sm[];
  const int C = CT ? CT : C_rt;
  const int EP = Mpts * kk;
  float4* pd = reinterpret_cast<float4*>(epf_sm);                               // [EP] edge offsets (w unused)
  float* xs = reinterpret_cast<float*>(epf_sm + (size_t)EP * 16);              // [Mpts][3]
  uint8_t* tsm = epf_sm + (((size_t)EP * 16 + (size_t)Mpts * 12 + 15) & ~(size_t)15);
  const int tid = threadIdx.x;
  const int cl = tid & 127, part = tid >> 7;                                   // channel inside the block, edge phase 0..3
  const int c = blockIdx.y * 128 + cl;
  const bool cv = c < C;
  const int cc = cv ? c : 0;
  if (LTAB) lif_table_load(tab + (size_t)blockIdx.y * tab_stride, tsm, tab_stride, tid, EPF_THREADS);
  const uint32_t lt_desc = (uint32_t)__cvta_generic_to_shared(tsm) + (uint32_t)cl * 8u;
  // y = ((w.d + b) * sc + sh) folded into one affine map of the offset
  const float sc = scale[cc];
  const float w0 = W[3 * cc] * sc, w1 = W[3 * cc + 1] * sc, w2 = W[3 * cc + 2] * sc;
  const NeuronParams p{np[cc], np[C + cc], np[2 * C + cc], np[3 * C + cc]};
  const float b0 = fmaf(bias[cc], sc, shift[cc]) - (LTAB ? p.th0 : 0.0f);     // table flavour: straight to x = u - theta0
  for (int64_t s = blockIdx.x; s < S; s += gridDim.x) {
    const int64_t patch0 = s * Mpts;
    __syncthreads();                                                           // previous patch fully consumed (and the table landed)
    for (int i = tid; i < 3 * Mpts; i += EPF_THREADS) xs[i] = xyz[3 * patch0 + i];
    __syncthreads();
    for (int e = tid; e < EP; e += EPF_THREADS) {
      const int pt = e / kk, j = e - pt * kk;
      const int nb = idx[(patch0 + pt) * ldi + j];
      pd[e] = make_float4(__fsub_rn(xs[3 * pt], xs[3 * nb]), __fsub_rn(xs[3 * pt + 1], xs[3 * nb + 1]),
                          __fsub_rn(xs[3 * pt + 2], xs[3 * nb + 2]), 0.0f);
    }
    __syncthreads();
    if (!cv) continue;
    __half* o = out + patch0 * kk * (int64_t)C + c + (int64_t)(part * 4) * C;   // this thread's first row; rounds advance it by 16 rows
    auto group = [&](int e0, bool full) {                                      // 4 consecutive edges of this thread's channel
      float4 d[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) d[j] = pd[(full || (e0 + j) < EP) ? (e0 + j) : (EP - 1)];
      float u[4];
      pos_lif4<LTAB>(d, w0, w1, w2, b0, p, T, lt_desc, u);
      store_h<PL2, 4>(o, C, plane, u, full ? 4 : EP - e0);
      o += 16 * C;
    };
    const int EPfull = EP & ~15;                                               // whole rounds of 4 phases x 4 edges: no bounds checks
#pragma unroll 1
    for (int e0 = part * 4; e0 < EPfull; e0 += 16) group(e0, true);
    if (EPfull + part * 4 < EP) group(EPfull + part * 4, false);
  }
}

// edge_pos_lif_fast (table flavour, (hi, lo) planes) on pair rows: row u's offset is delta[u]; persistent CTAs (grid.y = 128-channel block), 4 threads per channel
// each take 4 consecutive rows, the first *U_dev rows only.  `plane`: halfs between the hi and the lo plane (capacity * C).
template <int CT>
__global__ void __launch_bounds__(EPF_THREADS)
pair_pos_lif_kernel(const float4* __restrict__ delta, const int* __restrict__ U_dev, int C_rt, const float* __restrict__ W,
                    const float* __restrict__ bias, const float* __restrict__ scale, const float* __restrict__ shift,
                    const float* __restrict__ np, int T, __half* __restrict__ out, const uint8_t* __restrict__ tab, uint32_t tab_stride,
                    int64_t plane) {
  extern __shared__ __align__(16) uint8_t epf_sm[];
  const int C = CT ? CT : C_rt;
  const int tid = threadIdx.x;
  const int cl = tid & 127, part = tid >> 7;
  const int c = blockIdx.y * 128 + cl;
  const bool cv = c < C;
  const int cc = cv ? c : 0;
  lif_table_load(tab + (size_t)blockIdx.y * tab_stride, epf_sm, tab_stride, tid, EPF_THREADS);
  const uint32_t lt_desc = (uint32_t)__cvta_generic_to_shared(epf_sm) + (uint32_t)cl * 8u;
  const float sc = scale[cc];
  const float w0 = W[3 * cc] * sc, w1 = W[3 * cc + 1] * sc, w2 = W[3 * cc + 2] * sc;
  const NeuronParams p{np[cc], np[C + cc], np[2 * C + cc], np[3 * C + cc]};
  const float b0 = fmaf(bias[cc], sc, shift[cc]) - p.th0;
  __syncthreads();                                                             // the table landed
  if (!cv) return;
  const int64_t U = *U_dev;
  for (int64_t r0 = ((int64_t)blockIdx.x * 4 + part) * 4; r0 < U; r0 += (int64_t)gridDim.x * 16) {
    float4 d[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) d[j] = delta[r0 + j < U ? r0 + j : U - 1];
    float u[4];
    pos_lif4<1>(d, w0, w1, w2, b0, p, T, lt_desc, u);
    store_h<1, 4>(out + r0 * C + c, C, plane, u, (int)(U - r0 < 4 ? U - r0 : 4));
  }
}

// fc_gamma's table-flavour epilogue per edge, with the contraction W_gamma pos done per pair (WP, fp32, accumulator scale
// already undone): x = fmaf(WP[pid[e]], sc, fmaf(Wq[pt] - Wk[nb], sc, fmaf(bias, sc, shift) - theta0)) -- the expression of
// gemm_tc2_kernel's LT epilogue with the edge bias -- then the tabulated chain; (hi, lo) planes out as that epilogue writes them.
// Warp w of a CTA: channels (w & 3) * 32 + lane of the CTA's 128-channel block, rows in chunks of 32: lane l resolves row
// chunk*32 + l once (pair row, point, neighbour -> three element offsets), and the warp takes them by shuffle, 8 rows at a time,
// so no index arithmetic is repeated per channel.
constexpr int EGL_THREADS = 512;
template <int CT>
__global__ void __launch_bounds__(EGL_THREADS)
edge_gamma_lif_kernel(const float* __restrict__ WP, const int32_t* __restrict__ pid, const float* __restrict__ QK,
                      const int32_t* __restrict__ idx, int kk, int ldi, int Mpts, int64_t E, int C_rt, const float* __restrict__ bias,
                      const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ np, int T,
                      __half* __restrict__ out, const uint8_t* __restrict__ tab, uint32_t tab_stride, int64_t plane) {
  extern __shared__ __align__(16) uint8_t epf_sm[];
  const int C = CT ? CT : C_rt;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cl = (warp & 3) * 32 + lane, part = warp >> 2;
  const int c = blockIdx.y * 128 + cl;
  const bool cv = c < C;
  const int cc = cv ? c : 0;
  lif_table_load(tab + (size_t)blockIdx.y * tab_stride, epf_sm, tab_stride, tid, EGL_THREADS);
  const uint32_t lt_desc = (uint32_t)__cvta_generic_to_shared(epf_sm) + (uint32_t)cl * 8u;
  const float sc = scale[cc];
  const NeuronParams p{np[cc], np[C + cc], np[2 * C + cc], np[3 * C + cc]};
  const float bx = fmaf(bias[cc], sc, shift[cc]) - p.th0;
  __syncthreads();
  if (!cv) return;                                                // whole warps: C is a multiple of 32
  const float* wq = QK + c;
  const float* wk = QK + C + c;
  const float* wp = WP + c;
  const int64_t nch = (E + 31) / 32;
  for (int64_t ch = (int64_t)blockIdx.x * 4 + part; ch < nch; ch += (int64_t)gridDim.x * 4) {
    const int64_t r0 = ch * 32;
    uint32_t po, qo, ko;                                         // this lane's row: element offsets of WP, Wq and Wk
    {
      const uint32_t e = (uint32_t)(r0 + lane < E ? r0 + lane : E - 1);
      const uint32_t pt = e / (uint32_t)kk, jj = e - pt * (uint32_t)kk;
      const uint32_t nb = (pt / (uint32_t)Mpts) * (uint32_t)Mpts + (uint32_t)idx[(size_t)pt * ldi + jj];
      po = (uint32_t)pid[e] * (uint32_t)C; qo = pt * (uint32_t)(2 * C); ko = nb * (uint32_t)(2 * C);
    }
    const int nrow = (int)(E - r0 < 32 ? E - r0 : 32);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      if (g * 8 >= nrow) break;                                   // warp-uniform
      float u[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t a = __shfl_sync(0xffffffffu, po, g * 8 + j), b = __shfl_sync(0xffffffffu, qo, g * 8 + j),
                       d = __shfl_sync(0xffffffffu, ko, g * 8 + j);
        u[j] = fmaf(wp[a], sc, fmaf(wq[b] - wk[d], sc, bx));
      }
      lif_rows<1, 8>(u, p, T, lt_desc);
      store_h<1, 8>(out + (r0 + g * 8) * C + c, C, plane, u, nrow - g * 8);
    }
  }
}

// byte-packed copy of a patch-local graph (indices < 256): word w of point pt holds neighbours 4w .. 4w+3
__global__ void pack_idx_u8_kernel(const int32_t* __restrict__ idx, int ldi, int64_t P, int words, uint32_t* __restrict__ out) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= P * words) return;
  const int64_t pt = e / words;
  const int w = (int)(e - pt * words);
  uint32_t v = 0;
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    const int j = 4 * w + b;
    if (j < ldi) v |= ((uint32_t)idx[pt * ldi + j] & 255u) << (8 * b);
  }
  out[e] = v;
}
int launch_pack_idx_u8(const int32_t* idx, int ldi, int64_t P, uint32_t* out, cudaStream_t st) {
  if (P == 0) return 0;
  const int words = (ldi + 3) / 4;
  pack_idx_u8_kernel<<<(unsigned)ceil_div(P * words, 256), 256, 0, st>>>(idx, ldi, P, words, out);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

constexpr int ATT_KMAX = 32;

// softmax over the k neighbours + weighted sum.  CTA = 128 channels x APB points; KK is the compile-time
// neighbour count (12/18/24 for the yaml model, 32 = generic upper bound with run-time kk).
#ifndef SAPCU_APB
#define SAPCU_APB 8
#endif
constexpr int APB = SAPCU_APB;
template <bool PRECISE, int KK>
__global__ void __launch_bounds__(128)
attn_out_kernel(const float* __restrict__ logits, const float* __restrict__ pos, const float* __restrict__ V,
                int64_t ldv, const int32_t* __restrict__ idx, int ldi, int kk_rt, int Mpts, int P, int D,
                float sqrt_hd, float* __restrict__ out) {
  const int c = blockIdx.y * 128 + threadIdx.x;
  if (c >= D) return;
  const int kk = (KK == 32) ? kk_rt : KK;
  const float inv_s = 1.0f / sqrt_hd;
  for (int pi = 0; pi < APB; ++pi) {
    const int pt = blockIdx.x * APB + pi;
    if (pt >= P) return;
    const int patch0 = (pt / Mpts) * Mpts;
    const float* lg = logits + (int64_t)pt * kk * D + c;
    const float* ps = pos + (int64_t)pt * kk * D + c;
    float a[KK];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < KK; ++j) {
      if (j < kk) {
        const float l = lg[(int64_t)j * D];
        a[j] = PRECISE ? __fdiv_rn(l, sqrt_hd) : l * inv_s;
        mx = fmaxf(mx, a[j]);
      }
    }
    float sum = 0.0f;
#pragma unroll
    for (int j = 0; j < KK; ++j) {
      if (j < kk) {
        a[j] = PRECISE ? expf(__fsub_rn(a[j], mx)) : exp2f_approx((a[j] - mx) * 1.4426950408889634f);
        sum = __fadd_rn(sum, a[j]);
      }
    }
    const float inv_sum = 1.0f / sum;
    float res = 0.0f;
#pragma unroll
    for (int j = 0; j < KK; ++j) {
      if (j < kk) {
        const int nb = patch0 + idx[(int64_t)pt * ldi + j];
        const float vp = __fadd_rn(V[(int64_t)nb * ldv + c], ps[(int64_t)j * D]);
        if (PRECISE) res = __fadd_rn(res, __fmul_rn(__fdiv_rn(a[j], sum), vp));
        else res = fmaf(a[j] * inv_sum, vp, res);
      }
    }
    out[(int64_t)pt * D + c] = res;
  }
}

// fn attention input materialised for the tensor-core engine: out[e,c] = (q[pt,c] - k[nb,c]) + pos[e,c].
// One CTA = AIN_EDGES consecutive edges x D/4 float4 columns; a thread walks its column over the CTA's edges with
// incremental (pt, j) bookkeeping (one 32-bit division per thread instead of three 64-bit ones per element).
constexpr int AIN_EDGES = 16;
__global__ void __launch_bounds__(128)
attn_in_kernel(const float* __restrict__ Q, const float* __restrict__ Kf, int ldq, const float* __restrict__ pos,
               const int32_t* __restrict__ idx, int ldi, int kk, int Mpts, int E, int D, float* __restrict__ out) {
  const int D4 = D >> 2;
  const int c4 = threadIdx.x % D4;
  const int lane_e = threadIdx.x / D4;               // blockDim.x / D4 edges are processed side by side
  const int estep = blockDim.x / D4;
  const int e_begin = blockIdx.x * AIN_EDGES;
  const int e_end = min(e_begin + AIN_EDGES, E);
  int e = e_begin + lane_e;
  if (e >= e_end) return;
  int pt = e / kk, j = e - pt * kk;
  for (; e < e_end; e += estep) {
    const int nb = (pt / Mpts) * Mpts + idx[(int64_t)pt * ldi + j];
    const float4 q = reinterpret_cast<const float4*>(Q + (int64_t)pt * ldq)[c4];
    const float4 k = reinterpret_cast<const float4*>(Kf + (int64_t)nb * ldq)[c4];
    const float4 x = reinterpret_cast<const float4*>(pos + (int64_t)e * D)[c4];
    float4 o;
    o.x = __fadd_rn(__fsub_rn(q.x, k.x), x.x); o.y = __fadd_rn(__fsub_rn(q.y, k.y), x.y);
    o.z = __fadd_rn(__fsub_rn(q.z, k.z), x.z); o.w = __fadd_rn(__fsub_rn(q.w, k.w), x.w);
    reinterpret_cast<float4*>(out + (int64_t)e * D)[c4] = o;
    j += estep;
    while (j >= kk) { j -= kk; ++pt; }
  }
}

int launch_attn_in(const float* Q, const float* Kf, int64_t ldq, const float* pos, const int32_t* idx, int ldi, int kk,
                   int Mpts, int64_t E, int D, float* out, cudaStream_t st) {
  SAPCU_REQUIRE((D & 3) == 0 && (ldq & 3) == 0 && D <= 512 && (128 % (D >> 2)) == 0, "attn_in: unsupported D=%d", D);
  SAPCU_REQUIRE(E < ((int64_t)1 << 31) && ldq < (1 << 30), "attn_in: sizes must fit 32 bits");
  if (E == 0) return 0;
  attn_in_kernel<<<(unsigned)ceil_div(E, AIN_EDGES), 128, 0, st>>>(Q, Kf, (int)ldq, pos, idx, ldi, kk, Mpts, (int)E, D, out);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

// out[(s*Tt + t)*C + c] = max_m X[((s*M + m)*Tt + t)*C + c]
__global__ void group_max_kernel(const float* __restrict__ X, int64_t S, int M, int Tt, int C, float* __restrict__ out) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= S * Tt * C) return;
  const int c = (int)(e % C);
  const int64_t st = e / C;
  const int t = (int)(st % Tt);
  const int64_t s = st / Tt;
  const float* p = X + ((s * M) * Tt + t) * (int64_t)C + c;
  const int64_t stride = (int64_t)Tt * C;
  float m = -INFINITY;
  for (int i = 0; i < M; ++i) m = fmaxf(m, p[i * stride]);
  out[e] = m;
}

// one warp per patch: y = W[3,K] h + b ; LayerNorm(3) ; x / max(||x||, 1e-12)
__global__ void fn_head_kernel(const float* __restrict__ H, int K, int64_t S, const float* __restrict__ W,
                               const float* __restrict__ b, const float* __restrict__ lnw,
                               const float* __restrict__ lnb, float* __restrict__ out) {
  const int64_t s = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= S) return;
  float y[3] = {0.f, 0.f, 0.f};
  for (int c = lane; c < K; c += 32) {
    const float h = H[s * K + c];
#pragma unroll
    for (int o = 0; o < 3; ++o) y[o] = fmaf(W[o * K + c], h, y[o]);
  }
#pragma unroll
  for (int o = 0; o < 3; ++o)
    for (int off = 16; off; off >>= 1) y[o] += __shfl_xor_sync(0xffffffffu, y[o], off);
  if (lane == 0) {
#pragma unroll
    for (int o = 0; o < 3; ++o) y[o] += b[o];
    const float mean = (y[0] + y[1] + y[2]) / 3.0f;
    const float d0 = y[0] - mean, d1 = y[1] - mean, d2 = y[2] - mean;
    const float var = (d0 * d0 + d1 * d1 + d2 * d2) / 3.0f;
    const float rstd = 1.0f / sqrtf(var + 1e-5f);
    float z[3] = {d0 * rstd * lnw[0] + lnb[0], d1 * rstd * lnw[1] + lnb[1], d2 * rstd * lnw[2] + lnb[2]};
    const float nn = sqrtf(z[0] * z[0] + z[1] * z[1] + z[2] * z[2]);
    const float den = fmaxf(nn, 1e-12f);
    out[3 * s] = z[0] / den; out[3 * s + 1] = z[1] / den; out[3 * s + 2] = z[2] / den;
  }
}

int launch_pointwise3_lif(bool edge, bool precise, const float* xyz, const int32_t* idx, int kk, int ldi, int Mpts,
                          int64_t rows, int C, const float* W, const float* bias, const float* scale,
                          const float* shift, const float* np, int T, float* out, cudaStream_t st, int nsplit, bool out_h2) {
  if (rows == 0) return 0;
  if (edge) {
    SAPCU_REQUIRE(Mpts >= 1 && Mpts <= 256 && kk >= 1 && rows % ((int64_t)Mpts * kk) == 0, "pointwise3_lif: edge rows must be whole patches of <= 256 points");
    const int64_t S = rows / ((int64_t)Mpts * kk);
    const size_t smem = sizeof(float) * (3 * (size_t)Mpts + 2 * EPL_G * 3) + (size_t)Mpts * kk;
    dim3 grid((unsigned)S, (unsigned)ceil_div(C, 128), (unsigned)(nsplit < 1 ? 1 : nsplit));
    if (precise) edge_pos_lif_kernel<true><<<grid, 128, smem, st>>>(xyz, idx, kk, ldi, Mpts, C, W, bias, scale, shift, np, T, out, out_h2 ? 1 : 0, rows * C);
    else         edge_pos_lif_kernel<false><<<grid, 128, smem, st>>>(xyz, idx, kk, ldi, Mpts, C, W, bias, scale, shift, np, T, out, out_h2 ? 1 : 0, rows * C);
  } else {
    const unsigned grid = (unsigned)ceil_div(rows * C, 256);
    if (precise) pointwise3_lif_kernel<false, true><<<grid, 256, 0, st>>>(xyz, idx, kk, ldi, Mpts, rows, C, W, bias, scale, shift, np, T, out);
    else         pointwise3_lif_kernel<false, false><<<grid, 256, 0, st>>>(xyz, idx, kk, ldi, Mpts, rows, C, W, bias, scale, shift, np, T, out);
  }
  SAPCU_LAUNCH_CHECK();
  return 0;
}

// fast mode: single fp16 plane out, tabulated chain when `tab` is usable
int launch_edge_pos_lif_fast(const float* xyz, const int32_t* idx, int kk, int ldi, int Mpts, int64_t rows, int C,
                             const float* W, const float* bias, const float* scale, const float* shift, const float* np, int T,
                             float* out_h, const float* tab, uint32_t tab_stride, cudaStream_t st, bool two_planes) {
  if (rows == 0) return 0;
  SAPCU_REQUIRE(Mpts >= 1 && Mpts <= 256 && kk >= 1 && rows % ((int64_t)Mpts * kk) == 0, "edge_pos_lif_fast: edge rows must be whole patches of <= 256 points");
  const int64_t S = rows / ((int64_t)Mpts * kk);
  const bool lt = tab != nullptr && tab_stride > 0 && tab_stride <= LT_SMEM_BUDGET;
  const size_t smem = (((size_t)Mpts * kk * 16 + (size_t)Mpts * 12 + 15) & ~(size_t)15) + (lt ? tab_stride : 0);
  SAPCU_REQUIRE(smem <= 220 * 1024, "edge_pos_lif_fast: patch of %d x %d edges does not fit shared memory", Mpts, kk);
  static PerDeviceOnce once;
  {
    const int rc = once.run([]() -> int {
#define SAPCU_EPF_ATTR(L, CQ) SAPCU_CUDA_CHECK(cudaFuncSetAttribute(edge_pos_lif_fast_kernel<L, CQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024)); \
  SAPCU_CUDA_CHECK(cudaFuncSetAttribute(edge_pos_lif_fast_kernel<L, CQ, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024))
      SAPCU_EPF_ATTR(0, 0); SAPCU_EPF_ATTR(1, 0); SAPCU_EPF_ATTR(0, 128); SAPCU_EPF_ATTR(1, 128); SAPCU_EPF_ATTR(0, 256); SAPCU_EPF_ATTR(1, 256);
      SAPCU_EPF_ATTR(0, 512); SAPCU_EPF_ATTR(1, 512);
#undef SAPCU_EPF_ATTR
      return 0;
    });
    if (rc) return rc;
  }
  const int nblk = (int)ceil_div(C, 128);
  const uint8_t* tabp = lt ? reinterpret_cast<const uint8_t*>(tab) : nullptr;
  const uint32_t tstride = lt ? tab_stride : 0;
  __half* outp = reinterpret_cast<__half*>(out_h);
  const int64_t plane = rows * (int64_t)C;
#define SAPCU_EPF_GO(L, CQ)                                                                                             \
  do {                                                                                                                  \
    int occ = 1;                                                                                                        \
    SAPCU_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, edge_pos_lif_fast_kernel<L, CQ>, EPF_THREADS, smem)); \
    if (occ < 1) occ = 1;                                                                                               \
    int64_t gx = ((int64_t)kNumSMs * occ + nblk - 1) / nblk;                                                            \
    if (gx > S) gx = S;                                                                                                 \
    dim3 grid((unsigned)gx, (unsigned)nblk);                                                                            \
    if (two_planes) edge_pos_lif_fast_kernel<L, CQ, 1><<<grid, EPF_THREADS, smem, st>>>(xyz, idx, kk, ldi, Mpts, C, S, W, bias, scale, shift, np, T, \
                                                                                       outp, tabp, tstride, plane);     \
    else edge_pos_lif_fast_kernel<L, CQ><<<grid, EPF_THREADS, smem, st>>>(xyz, idx, kk, ldi, Mpts, C, S, W, bias, scale, shift, np, T, \
                                                                          outp, tabp, tstride, plane);                  \
  } while (0)
  if (lt) { if (C == 128) SAPCU_EPF_GO(1, 128); else if (C == 256) SAPCU_EPF_GO(1, 256); else if (C == 512) SAPCU_EPF_GO(1, 512); else SAPCU_EPF_GO(1, 0); }
  else { if (C == 128) SAPCU_EPF_GO(0, 128); else if (C == 256) SAPCU_EPF_GO(0, 256); else if (C == 512) SAPCU_EPF_GO(0, 512); else SAPCU_EPF_GO(0, 0); }
#undef SAPCU_EPF_GO
  SAPCU_LAUNCH_CHECK();
  return 0;
}

int launch_attn_out(bool precise, const float* logits, const float* pos, const float* V, int64_t ldv,
                    const int32_t* idx, int ldi, int kk, int Mpts, int64_t P, int D, float sqrt_hd, float* out,
                    cudaStream_t st) {
  SAPCU_REQUIRE(kk <= ATT_KMAX, "attn_out: k=%d > %d", kk, ATT_KMAX);
  SAPCU_REQUIRE(P < ((int64_t)1 << 31), "attn_out: too many points for 32-bit indexing");
  if (P == 0) return 0;
  dim3 grid((unsigned)ceil_div(P, APB), (unsigned)ceil_div(D, 128));
#define SAPCU_AO(PR, KK) attn_out_kernel<PR, KK><<<grid, 128, 0, st>>>(logits, pos, V, ldv, idx, ldi, kk, Mpts, (int)P, D, sqrt_hd, out)
  if (precise) {
    if (kk == 12) SAPCU_AO(true, 12); else if (kk == 18) SAPCU_AO(true, 18); else if (kk == 24) SAPCU_AO(true, 24); else SAPCU_AO(true, 32);
  } else {
    if (kk == 12) SAPCU_AO(false, 12); else if (kk == 18) SAPCU_AO(false, 18); else if (kk == 24) SAPCU_AO(false, 24); else SAPCU_AO(false, 32);
  }
#undef SAPCU_AO
  SAPCU_LAUNCH_CHECK();
  return 0;
}

int launch_group_max(const float* X, int64_t S, int M, int Tt, int C, float* out, cudaStream_t st) {
  if (S == 0) return 0;
  group_max_kernel<<<(unsigned)ceil_div(S * Tt * C, 256), 256, 0, st>>>(X, S, M, Tt, C, out);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

int launch_fn_head(const float* H, int K, int64_t S, const float* W, const float* b, const float* lnw,
                   const float* lnb, float* out, cudaStream_t st) {
  if (S == 0) return 0;
  fn_head_kernel<<<(unsigned)ceil_div(S * 32, 256), 256, 0, st>>>(H, K, S, W, b, lnw, lnb, out);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

}  // namespace sapcu

namespace sapcu {

#define SAPCU_TRY_RC(e) do { const int _r = (e); if (_r) return _r; } while (0)

namespace {
// persistent grid: as many CTAs per channel block as fit the SMs, never more than `steps` (rows / rows a CTA takes per step)
template <class K> int epf_grid(K kern, size_t smem, int nblk, int64_t steps, dim3& grid) {
  SAPCU_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  int occ = 1;
  SAPCU_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, EPF_THREADS, smem));
  if (occ < 1) occ = 1;
  int64_t gx = ((int64_t)kNumSMs * occ + nblk - 1) / nblk;
  if (gx > steps) gx = steps;
  if (gx < 1) gx = 1;
  grid = dim3((unsigned)gx, (unsigned)nblk);
  return 0;
}
}  // namespace

int launch_pair_pos_lif(const float4* delta, const int* U_dev, int64_t rows, int C, const float* W, const float* bias,
                        const float* scale, const float* shift, const float* np, int T, float* out_h, const float* tab,
                        uint32_t tab_stride, cudaStream_t st) {
  if (rows == 0) return 0;
  SAPCU_REQUIRE(tab != nullptr && tab_stride > 0 && tab_stride <= LT_SMEM_BUDGET, "pair_pos_lif: needs the layer's LIF table");
  const size_t smem = tab_stride;
  const int nblk = (int)ceil_div(C, 128);
  const uint8_t* tabp = reinterpret_cast<const uint8_t*>(tab);
  __half* o = reinterpret_cast<__half*>(out_h);
  const int64_t plane = rows * (int64_t)C;
  dim3 grid;
#define SAPCU_PPL_GO(CQ)                                                                                                \
  do {                                                                                                                  \
    SAPCU_TRY_RC(epf_grid(pair_pos_lif_kernel<CQ>, smem, nblk, ceil_div(rows, 16), grid));                              \
    pair_pos_lif_kernel<CQ><<<grid, EPF_THREADS, smem, st>>>(delta, U_dev, C, W, bias, scale, shift, np, T, o, tabp, tab_stride, plane); \
  } while (0)
  if (C == 128) SAPCU_PPL_GO(128); else if (C == 256) SAPCU_PPL_GO(256); else if (C == 512) SAPCU_PPL_GO(512); else SAPCU_PPL_GO(0);
#undef SAPCU_PPL_GO
  SAPCU_LAUNCH_CHECK();
  return 0;
}

int launch_edge_gamma_lif(const float* WP, const int32_t* pid, const float* QK, const int32_t* idx, int kk, int ldi, int Mpts,
                          int64_t rows, int C, const float* bias, const float* scale, const float* shift, const float* np, int T,
                          float* out_h, const float* tab, uint32_t tab_stride, cudaStream_t st) {
  if (rows == 0) return 0;
  SAPCU_REQUIRE(tab != nullptr && tab_stride > 0 && tab_stride <= LT_SMEM_BUDGET, "edge_gamma_lif: needs the layer's LIF table");
  SAPCU_REQUIRE(C % 32 == 0 && kk >= 1 && Mpts >= 1 && rows % ((int64_t)Mpts * kk) == 0, "edge_gamma_lif: edge rows must be whole patches, C %% 32 == 0");
  SAPCU_REQUIRE(rows < (1ll << 31) && (rows / kk) * 2 * C < (1ll << 32) && rows * C < (1ll << 32), "edge_gamma_lif: element offsets must fit 32 bits");
  const size_t smem = tab_stride;
  const int nblk = (int)ceil_div(C, 128);
  const uint8_t* tabp = reinterpret_cast<const uint8_t*>(tab);
  __half* o = reinterpret_cast<__half*>(out_h);
  const int64_t plane = rows * (int64_t)C;
  dim3 grid;
#define SAPCU_EGL_GO(CQ)                                                                                                \
  do {                                                                                                                  \
    SAPCU_TRY_RC(epf_grid(edge_gamma_lif_kernel<CQ>, smem, nblk, ceil_div(rows, 128), grid));                                \
    edge_gamma_lif_kernel<CQ><<<grid, EGL_THREADS, smem, st>>>(WP, pid, QK, idx, kk, ldi, Mpts, rows, C, bias, scale, shift, np, T, \
                                                               o, tabp, tab_stride, plane);                             \
  } while (0)
  if (C == 128) SAPCU_EGL_GO(128); else if (C == 256) SAPCU_EGL_GO(256); else if (C == 512) SAPCU_EGL_GO(512); else SAPCU_EGL_GO(0);
#undef SAPCU_EGL_GO
  SAPCU_LAUNCH_CHECK();
  return 0;
}

}  // namespace sapcu
