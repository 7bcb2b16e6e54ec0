// fp32 SIMT GEMM engine of the "fp32 parity mode":  Y[R,N] = epi( A[R,K] * W[N,K]^T ).
//
// Every 1x1 Conv1d/Conv2d and Linear of the two models (SURVEY.md appendix B) is this contraction
// with rows = points, edges or patches.  The A operand is produced by a loader policy so the
// per-edge inputs never exist in HBM:
//   A_PLAIN    A[r,c] = X[r*lda + c]
//   A_EDGECAT  fd EdgeConv input cat(x_j - x_i, x_j) (fd/snn_coder.py:52-68):
//              A[r,c<C] = F[nb(r),c] - F[pt(r),c] ; A[r,c>=C] = F[nb(r),c-C]
//   A_ATTNIN   fn attention input q_i - k_j + pos_ij (fn/snn_coder.py:367-371):
//              A[r,c] = Q[pt(r),c] - Kf[nb(r),c] + X[r*lda + c]
// where edge row r = pt*kk + j, pt = global point row, nb = patch-local neighbour idx[pt*ldi + j].
// The epilogue fuses conv bias, eval-mode BatchNorm (scale/shift), the activation (LeakyReLU, exact
// GELU, or the whole LIF^T recurrence), an optional residual and an optional max over groups of 32
// consecutive rows (EdgeConv max over k=32 neighbours).
//
// Tile 128x128x16, 256 threads, 8x8 register micro-tile, register-prefetch double buffering.
// Roofline: FP32 FFMA issue (148 SM x 128 lanes); not HBM.
#pragma once
#include "common.cuh"
#include "neuron.cuh"

namespace sapcu {

enum AMode : int { A_PLAIN = 0, A_EDGECAT = 1, A_ATTNIN = 2 };

struct GemmArgs {
  // A operand
  const float* A = nullptr; int64_t lda = 0; int64_t R = 0; int K = 0;
  const int32_t* idx = nullptr; int ldi = 0; int kk = 0; int Mpts = 0;   // edge loaders: idx[pt*ldi + j]
  const uint32_t* idx8 = nullptr; int ldi8w = 0;   // optional byte-packed copy of idx (4 indices per word) for the fused attention tail
  const float* F = nullptr; int64_t ldf = 0; int C = 0;       // A_EDGECAT
  const float* Q = nullptr; const float* Kf = nullptr; int64_t ldq = 0;   // A_ATTNIN
  // B operand: W[N,K] row-major
  const float* W = nullptr; int N = 0;
  const float* Whi = nullptr; const float* Wlo = nullptr;   // optional pre-split tf32 (hi, lo) copies for the tensor-core engine
  // epilogue
  const float* bias = nullptr; const float* scale = nullptr; const float* shift = nullptr;
  int act = ACT_NONE; int T = 0; const float* nparams = nullptr;   // nparams: [4][N] = d,a,r,th0
  const float* residual = nullptr; int64_t ldr = 0;
  float* Y = nullptr; int64_t ldc = 0;
  float* Y2 = nullptr;   // 2-CTA tensor-core engine, LIF epilogue writing fp16 planes: optional fp32 copy of the same spikes ([R, N], ld = N)
  int tc_passes = 3;     // tensor-core engine only: 3 = 3xTF32 split, 1 = single-pass TF32
  bool tc2_any_rows = false;   // 2-CTA engine from 1024 rows on (plane-exchanging point-level layers: chunk-size independent arithmetic)
  // tensor-core engine only: fuse softmax_k(Y / at_sqrt) and sum_j a_j (at_v[nb_j] + at_pos[e_j]) into the epilogue; Y becomes [points, N]
  const float* at_pos = nullptr; const float* at_v = nullptr; int64_t at_ldv = 0; float at_sqrt = 1.0f;
  float* pool = nullptr; int pool_T = 0, pool_M = 0;   // 2-CTA tensor-core engine: rows are (point*T + t); instead of Y emit pool[(patch*T + t), c] = max over the patch's pool_M points (buffer pre-filled with -inf)
  // fp16x3 tensor-core path (2-CTA kernel): half (hi, lo) copies of W * 2^e, winv = 2^-e; x_unit = the activations are LIF
  // outputs (soft spikes in (0, 0.7)), so x * 2^13 and its residual are representable in fp16
  const float* Wh = nullptr; const float* Wl = nullptr; float winv = 1.0f; bool x_unit = false;
  // fp16 (hi, lo) plane format of x * 2^13 ([R, K] halfs each, hi plane first): x_h2 = A is stored that way (consumed by the
  // fp16x3 kernel without conversion), out_h2 = the LIF epilogue writes Y that way; both need ld == row length
  bool x_h2 = false, out_h2 = false, pos_h2 = false;   // pos_h2: at_pos (fused attention tail) is stored as planes
  // SAPCU_MODE_FAST (2-CTA tensor-core engine): ONE fp16 product per MAC; x_h2 / out_h2 / pos_h2 then mean a single fp16 plane
  // of x * 2^13; lif_tab: tabulated LIF^T chain of the epilogue's neuron (nullptr: reduced-MUFU recurrence)
  bool fast = false; const float* lif_tab = nullptr; uint32_t lif_tab_stride = 0;
  bool edge_bias = false;   // tensor-core engines, A_PLAIN: add Q[pt,c] - Kf[nb,c] (per-point products) to the accumulator, see tc_ptx.cuh
  // 2-CTA tensor-core engine: rows actually present, in device memory (R is then the capacity the buffers and TMA maps are
  // sized for); at_pid: the fused attention tail reads pos row at_pid[e] for edge e (pos held once per distinct point pair)
  const int* R_dev = nullptr; const int32_t* at_pid = nullptr;
  int group = 0;   // 0 or 32
  const char* label = "gemm";   // kernel label of the live profiler (sapcu_profile_report)
};

constexpr int GBM = 128, GBN = 128, GBK = 16, GTHREADS = 256;

template <int AMODE>
struct ARow {   // per-thread row context of the A loader (one row per thread, fixed over the K loop)
  const float* p0 = nullptr;   // PLAIN: row ptr ; EDGECAT: F[nb] ; ATTNIN: X row
  const float* p1 = nullptr;   // EDGECAT: F[pt] ; ATTNIN: Q[pt]
  const float* p2 = nullptr;   // ATTNIN: Kf[nb]
  bool valid = false;
};

template <int AMODE>
__device__ __forceinline__ void arow_init(ARow<AMODE>& r, const GemmArgs& g, int64_t row) {
  r.valid = row < g.R;
  if (!r.valid) return;
  if (AMODE == A_PLAIN) {
    r.p0 = g.A + row * g.lda;
  } else {
    const int64_t pt = row / g.kk;
    const int64_t patch0 = (pt / g.Mpts) * g.Mpts;
    const int64_t nb = patch0 + g.idx[pt * g.ldi + (row - pt * g.kk)];
    if (AMODE == A_EDGECAT) {
      r.p0 = g.F + nb * g.ldf;
      r.p1 = g.F + pt * g.ldf;
    } else {
      r.p0 = g.A + row * g.lda;
      r.p1 = g.Q + pt * g.ldq;
      r.p2 = g.Kf + nb * g.ldq;
    }
  }
}

// loads 8 consecutive K elements [k0, k0+8) of this thread's row
template <int AMODE>
__device__ __forceinline__ void arow_load8(const ARow<AMODE>& r, const GemmArgs& g, int k0, float (&v)[8]) {
  if (!r.valid) {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.0f;
    return;
  }
  if (AMODE == A_PLAIN) {
    const float4 a = *reinterpret_cast<const float4*>(r.p0 + k0);
    const float4 b = *reinterpret_cast<const float4*>(r.p0 + k0 + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else if (AMODE == A_EDGECAT) {
    // C is a multiple of 8, so an 8-wide K slice never straddles the two halves
    if (k0 < g.C) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 n = *reinterpret_cast<const float4*>(r.p0 + k0 + 4 * h);
        const float4 c = *reinterpret_cast<const float4*>(r.p1 + k0 + 4 * h);
        v[4 * h + 0] = __fsub_rn(n.x, c.x); v[4 * h + 1] = __fsub_rn(n.y, c.y);
        v[4 * h + 2] = __fsub_rn(n.z, c.z); v[4 * h + 3] = __fsub_rn(n.w, c.w);
      }
    } else {
      const float4 a = *reinterpret_cast<const float4*>(r.p0 + k0 - g.C);
      const float4 b = *reinterpret_cast<const float4*>(r.p0 + k0 - g.C + 4);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
  } else {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float4 x = *reinterpret_cast<const float4*>(r.p0 + k0 + 4 * h);
      const float4 q = *reinterpret_cast<const float4*>(r.p1 + k0 + 4 * h);
      const float4 kf = *reinterpret_cast<const float4*>(r.p2 + k0 + 4 * h);
      // (q - k) + pos, the reference's evaluation order
      v[4 * h + 0] = __fadd_rn(__fsub_rn(q.x, kf.x), x.x); v[4 * h + 1] = __fadd_rn(__fsub_rn(q.y, kf.y), x.y);
      v[4 * h + 2] = __fadd_rn(__fsub_rn(q.z, kf.z), x.z); v[4 * h + 3] = __fadd_rn(__fsub_rn(q.w, kf.w), x.w);
    }
  }
}

template <int AMODE, int ACT, int GROUP, bool PRECISE>
__global__ void __launch_bounds__(GTHREADS, 2)
gemm_simt_kernel(const GemmArgs g) {
  __shared__ __align__(16) float As[2][GBK][GBM];
  __shared__ __align__(16) float Bs[2][GBK][GBN];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t row0 = (int64_t)blockIdx.x * GBM;
  const int col0 = blockIdx.y * GBN;

  // loader mapping: one tile row per thread, 8 consecutive K per thread
  const int lrow = tid & 127;
  const int lk = (tid >> 7) * 8;
  ARow<AMODE> ar;
  arow_init<AMODE>(ar, g, row0 + lrow);
  const int wn = col0 + lrow;
  const bool wvalid = wn < g.N;
  const float* wrow = g.W + (int64_t)(wvalid ? wn : 0) * g.K;

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

  float ra[8], rb[8];
  auto gload = [&](int k0) {
    arow_load8<AMODE>(ar, g, k0 + lk, ra);
    if (wvalid) {
      const float4 a = *reinterpret_cast<const float4*>(wrow + k0 + lk);
      const float4 b = *reinterpret_cast<const float4*>(wrow + k0 + lk + 4);
      rb[0] = a.x; rb[1] = a.y; rb[2] = a.z; rb[3] = a.w; rb[4] = b.x; rb[5] = b.y; rb[6] = b.z; rb[7] = b.w;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) rb[i] = 0.0f;
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { As[buf][lk + i][lrow] = ra[i]; Bs[buf][lk + i][lrow] = rb[i]; }
  };

  const int nk = g.K / GBK;
  gload(0);
  sstore(0);
  __syncthreads();
  for (int kt = 0; kt < nk; ++kt) {
    const int cur = kt & 1;
    if (kt + 1 < nk) gload((kt + 1) * GBK);
#pragma unroll
    for (int k = 0; k < GBK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[cur][k][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[cur][k][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[cur][k][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[cur][k][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (kt + 1 < nk) {
      sstore(cur ^ 1);
      __syncthreads();
    }
  }

  // ---------------- epilogue ----------------
  float gmax[2][8];
  if (GROUP) {
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int j = 0; j < 8; ++j) gmax[h][j] = -INFINITY;
  }
#pragma unroll
  for (int jh = 0; jh < 2; ++jh) {
    const int cbase = col0 + jh * 64 + tx * 4;
    float bia[4], sc[4], sh[4];
    NeuronParams np[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = cbase + j;
      const bool cv = c < g.N;
      bia[j] = (g.bias && cv) ? g.bias[c] : 0.0f;
      sc[j] = (g.scale && cv) ? g.scale[c] : 1.0f;
      sh[j] = (g.shift && cv) ? g.shift[c] : 0.0f;
      if (ACT == ACT_LIF) {
        const int cc = cv ? c : 0;
        np[j].d = g.nparams[cc]; np[j].a = g.nparams[g.N + cc];
        np[j].r = g.nparams[2 * g.N + cc]; np[j].th0 = g.nparams[3 * g.N + cc];
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t row = row0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
      const bool rv = row < g.R;
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float y = acc[i][jh * 4 + j];
        if (g.bias) y = __fadd_rn(y, bia[j]);
        if (g.scale) y = __fadd_rn(__fmul_rn(y, sc[j]), sh[j]);
        if (g.residual && rv && (cbase + j) < g.N) y = __fadd_rn(y, g.residual[row * g.ldr + cbase + j]);
        if (ACT == ACT_LEAKY) y = act_leaky(y);
        if (ACT == ACT_GELU) y = act_gelu(y);
        if (ACT == ACT_LIF) y = lif_chain<PRECISE>(y, np[j], g.T);
        v[j] = y;
      }
      if (GROUP) {
        if (rv) {
#pragma unroll
          for (int j = 0; j < 4; ++j) gmax[i >> 2][jh * 4 + j] = fmaxf(gmax[i >> 2][jh * 4 + j], v[j]);
        }
      } else if (rv) {
        float* yp = g.Y + row * g.ldc + cbase;
        if (cbase + 3 < g.N && ((g.ldc & 3) == 0)) {
          *reinterpret_cast<float4*>(yp) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (cbase + j < g.N) yp[j] = v[j];
        }
      }
    }
  }
  if (GROUP) {
    // max over 32 consecutive rows: rows [0,32) <-> ty 0..7 half 0, [32,64) <-> ty 8..15 half 0,
    // [64,96) <-> ty 0..7 half 1, [96,128) <-> ty 8..15 half 1
    __syncthreads();
    float* red = &As[0][0][0];   // [16 ty][2 half][128 cols] = 4096 floats (As holds 4096)
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = (j < 4) ? tx * 4 + j : 64 + tx * 4 + (j - 4);
        red[(ty * 2 + h) * 128 + c] = gmax[h][j];
      }
    __syncthreads();
    for (int o = tid; o < 4 * 128; o += GTHREADS) {
      const int grp = o >> 7, c = o & 127;
      const int h = grp >> 1, tyb = (grp & 1) * 8;
      float m = -INFINITY;
#pragma unroll
      for (int t = 0; t < 8; ++t) m = fmaxf(m, red[((tyb + t) * 2 + h) * 128 + c]);
      const int64_t orow = (row0 >> 5) + grp;
      if (orow * 32 < g.R && col0 + c < g.N) g.Y[orow * g.ldc + col0 + c] = m;
    }
  }
}

template <int AMODE, int ACT, int GROUP, bool PRECISE>
static int launch_gemm_simt_t(const GemmArgs& g, cudaStream_t st) {
  dim3 grid((unsigned)ceil_div(g.R, GBM), (unsigned)ceil_div(g.N, GBN));
  gemm_simt_kernel<AMODE, ACT, GROUP, PRECISE><<<grid, GTHREADS, 0, st>>>(g);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

// runtime dispatch over the combinations the two models use
int launch_gemm_simt(const GemmArgs& g, int amode, bool precise, cudaStream_t st);

}  // namespace sapcu
