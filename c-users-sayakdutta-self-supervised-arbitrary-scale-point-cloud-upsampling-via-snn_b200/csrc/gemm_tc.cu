// tcgen05 tensor-core GEMM engine (SAPCU_MODE_TC):  Y[R,N] = epi( X[R,K] * W[N,K]^T ), fp32 in / fp32 out.
//
// fp32-faithful products on the 5th-gen tensor cores by the 3xTF32 split
//     x = x_hi + x_lo,  w = w_hi + w_lo   (hi = x rounded to tf32, lo = x - hi, exact in fp32)
//     x*w ~= w_hi*x_hi + w_hi*x_lo + w_lo*x_hi        (the dropped w_lo*x_lo term is <= 2^-22 relative)
// accumulated in fp32 in TMEM.  This keeps the "fp32 parity mode" tolerances while moving every large
// contraction off the FFMA pipe.
//
// Orientation: the WEIGHT tile is the UMMA A operand (M = 128 output channels -> TMEM lanes) and the
// ACTIVATION tile is the B operand (N = BN rows -> TMEM columns).  One epilogue thread therefore owns one
// output channel: bias / BatchNorm / neuron parameters live in registers, the LIF^T recurrence runs on
// register-resident accumulators, a max over 32 consecutive rows (EdgeConv k = 32) is thread-local, and
// the 32 lanes of a warp store 32 consecutive channels of one row (one 128-byte line).
//
// Persistent, warp-specialised CTA (1 per SM, 640 threads):
//   warp 0        TMA producer   cp.async.bulk.tensor of the pre-split tf32 W hi/lo tiles and the raw fp32 X tile
//                                (128B swizzle) + cp.async.bulk.prefetch.tensor L2 look-ahead for X
//   warp 1        MMA issuer     tcgen05.mma.kind::tf32 (12 per 32-wide k-block), tcgen05.commit; owns TMEM alloc
//   warps 2..3    splitter       lo = x - trunc_tf32(x) into the second buffer (the raw tile is the hi operand: the
//                                tensor core ignores the low 13 mantissa bits)
//   warps 4..19   epilogue       tcgen05.ld -> bias / BN / activation / LIF^T / fused tails -> 128-byte row stores
// Pipelines: smem ring of 2 stages x 96 KiB (mbarriers raw-full / split-full / empty) and 2 TMEM accumulator buffers of
// 256 columns (mbarriers tmem-full / tmem-empty) so the epilogue of tile i overlaps the MMAs of tile i+1.  Every mbarrier
// wait carries a clock64() watchdog: a protocol error surfaces as an error code, never as a hung GPU.
//
// Epilogue flavours (template EXTRA): 0 plain, 1 + residual, 2 edge bias W q_i - W k_j added before BN + LIF (factorised
// attention input), 3 fused attention tail (softmax over the KK edges of a point and the weighted sum; tc_ptx.cuh).
// The LIF path reads TMEM 8 columns at a time with the next piece in flight.
//
// Roofline: tensor pipe (tf32: 2048 MAC/clk/SM, x3 passes); the LIF epilogue is MUFU bound (3 MUFU per
// element-step, 16/clk/SM) and overlaps the MMA stream.
#include <cuda.h>
#include <stdlib.h>
#include <mutex>
#include "gemm_tc.h"
#include "neuron.cuh"
#include "tc_ptx.cuh"

namespace sapcu {

constexpr int TC_BN = 256;                      // activation rows per tile (UMMA N)
constexpr int TC_STAGES = 2, TC_ACC = 2;        // smem stages, TMEM accumulators of TC_BN columns
constexpr int TC_SPLIT_WARP0 = 2, TC_SPLIT_WARPS = 2;
constexpr int TC_EPI_WARP0 = TC_SPLIT_WARP0 + TC_SPLIT_WARPS, TC_EPI = 16;   // 2 + 2 + 16 warps = 640 threads: 96 registers per thread for the epilogue
constexpr int TC_THREADS = (TC_EPI_WARP0 + TC_EPI) * 32;
constexpr uint32_t TC_X_BYTES = TC_BN * TC_BK * 4;
constexpr uint32_t TC_STAGE_BYTES = 2 * TC_TILE_BYTES + 2 * TC_X_BYTES;       // W_hi, W_lo, X_hi, X_lo
constexpr size_t TC_SMEM_BYTES = (size_t)TC_STAGES * TC_STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;


// ------------------------------------------------------------------------------------------------ kernel
template <int ACT, int EXTRA, int KK = 1>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_wlo,
               const __grid_constant__ CUtensorMap map_x, const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;            // 128B swizzle needs 1024 B alignment
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + TC_STAGES * TC_STAGE_BYTES;
  // barrier map (8 bytes each)
  auto bar_raw = [&](int s) { return bar_base + 8u * s; };
  auto bar_split = [&](int s) { return bar_base + 8u * (TC_STAGES + s); };
  auto bar_empty = [&](int s) { return bar_base + 8u * (2 * TC_STAGES + s); };
  auto bar_tfull = [&](int a) { return bar_base + 8u * (3 * TC_STAGES + a); };
  auto bar_tempty = [&](int a) { return bar_base + 8u * (3 * TC_STAGES + TC_ACC + a); };
  const uint32_t tmem_slot = bar_base + 8u * (3 * TC_STAGES + 2 * TC_ACC);
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + TC_STAGES * TC_STAGE_BYTES + 8 * (3 * TC_STAGES + 2 * TC_ACC));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nk = p.K / TC_BK;
  const int64_t total_tiles = p.n_tiles * p.m_tiles;
  const int TR = p.tile_rows;                                       // rows a tile advances by (TC_BN; whole points only when EXTRA == 3)
  constexpr uint32_t idesc = tc_idesc(TC_BN);                       // the MMA always spans TC_BN rows

  if (threadIdx.x == 0) {
    for (int s = 0; s < TC_STAGES; ++s) { mbar_init(bar_raw(s), 1); mbar_init(bar_split(s), TC_SPLIT_WARPS * 32); mbar_init(bar_empty(s), 1); }
    for (int a = 0; a < TC_ACC; ++a) { mbar_init(bar_tfull(a), 1); mbar_init(bar_tempty(a), TC_EPI); }
    fence_barrier_init();
    tma_prefetch_desc(&map_w);
    tma_prefetch_desc(&map_wlo);
    tma_prefetch_desc(&map_x);
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;

  if (warp == 0) {
    // ======================================================================== TMA producer
    if (lane == 0) {
      int s = 0; uint32_t ph = 0; bool ok = true;
      for (int64_t t = blockIdx.x; t < total_tiles && ok; t += gridDim.x) {
        const int m_t = (int)(t % p.m_tiles);
        const int64_t n_t = t / p.m_tiles;
        for (int kb = 0; kb < nk; ++kb) {
          // pull the activation tile TC_L2_PREFETCH k-blocks ahead (possibly in this CTA's next tile) into L2
          int kp = kb + TC_L2_PREFETCH; int64_t tp = t;
          if (kp >= nk) { kp -= nk; tp += gridDim.x; }
          if (kp < nk && tp < total_tiles) tma_prefetch_l2_2d(&map_x, kp * TC_BK, (int)((tp / p.m_tiles) * TR));
          if (!(ok = mbar_wait(bar_empty(s), ph ^ 1u, p.err))) break;
          const uint32_t st = smem_base + s * TC_STAGE_BYTES;
          mbar_expect_tx(bar_raw(s), ((p.split_w || p.passes == 1) ? 1 : 2) * TC_TILE_BYTES + TC_X_BYTES);
          tma_load_2d(st, &map_w, bar_raw(s), kb * TC_BK, m_t * TC_BM);
          if (!p.split_w && p.passes == 3) tma_load_2d(st + TC_TILE_BYTES, &map_wlo, bar_raw(s), kb * TC_BK, m_t * TC_BM);
          tma_load_2d(st + 2 * TC_TILE_BYTES, &map_x, bar_raw(s), kb * TC_BK, (int)(n_t * TR));
          if (++s == TC_STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ======================================================================== MMA issuer
    if (lane == 0) {
      int s = 0, a = 0; uint32_t ph = 0, aph = 0; bool ok = true;
      for (int64_t t = blockIdx.x; t < total_tiles && ok; t += gridDim.x) {
        if (!(ok = mbar_wait(bar_tempty(a), aph ^ 1u, p.err))) break;
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(a * TC_BN);
        for (int kb = 0; kb < nk; ++kb) {
          if (!(ok = mbar_wait(bar_split(s), ph, p.err))) break;
          tc_fence_after();
          const uint32_t st = smem_base + s * TC_STAGE_BYTES;
          const uint64_t w_hi = umma_desc_sw128(st), w_lo = umma_desc_sw128(st + TC_TILE_BYTES);
          const uint64_t x_hi = umma_desc_sw128(st + 2 * TC_TILE_BYTES), x_lo = umma_desc_sw128(st + 2 * TC_TILE_BYTES + TC_X_BYTES);
#pragma unroll
          for (int k8 = 0; k8 < TC_BK / 8; ++k8) {
            const uint64_t adv = (uint64_t)(k8 * 2);            // 8 tf32 = 32 B = 2 x 16 B along the swizzled row
            if (p.passes == 3) {
              umma_tf32(tmem_d, w_lo + adv, x_hi + adv, idesc, (kb | k8) ? 1u : 0u);
              umma_tf32(tmem_d, w_hi + adv, x_lo + adv, idesc, 1u);
              umma_tf32(tmem_d, w_hi + adv, x_hi + adv, idesc, 1u);
            } else {
              umma_tf32(tmem_d, w_hi + adv, x_hi + adv, idesc, (kb | k8) ? 1u : 0u);
            }
          }
          umma_commit(bar_empty(s));                             // frees the smem stage when these MMAs retire
          if (kb == nk - 1) umma_commit(bar_tfull(a));           // accumulator complete
          if (++s == TC_STAGES) { s = 0; ph ^= 1u; }
        }
        if (++a == TC_ACC) { a = 0; aph ^= 1u; }
      }
    }
  } else if (warp < TC_EPI_WARP0) {
    // ======================================================================== splitter: raw -> (hi, lo)
    const int tid = threadIdx.x - TC_SPLIT_WARP0 * 32;
    int s = 0; uint32_t ph = 0; bool ok = true;
    for (int64_t t = blockIdx.x; t < total_tiles && ok; t += gridDim.x) {
      for (int kb = 0; kb < nk; ++kb) {
        if (!(ok = mbar_wait(bar_raw(s), ph, p.err))) break;
        uint8_t* st = smem_gen + s * TC_STAGE_BYTES;
#pragma unroll
        for (int op = 0; op < 2; ++op) {                          // 0: W tile (only when it arrives raw), 1: X tile
          if (p.passes == 1) continue;                            // single-pass TF32: the raw tiles are the operands
          if (op == 0 && !p.split_w) continue;
          const uint32_t bytes = op ? TC_X_BYTES : TC_TILE_BYTES;
          float4* hi = reinterpret_cast<float4*>(st + op * 2 * TC_TILE_BYTES);
          float4* lo = reinterpret_cast<float4*>(st + op * 2 * TC_TILE_BYTES + bytes);
          const int iters = (int)(bytes / 16) / (TC_SPLIT_WARPS * 32);
#pragma unroll
          for (int i = 0; i < iters; ++i) {
            const int e = tid + i * TC_SPLIT_WARPS * 32;
            const float4 v = hi[e];
            float4 l;
            l.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
            l.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
            l.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
            l.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
            lo[e] = l;
          }
        }
        fence_proxy_async();                                      // generic-proxy writes -> visible to the tensor core
        mbar_arrive(bar_split(s));
        if (++s == TC_STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // ======================================================================== epilogue
    const int q = warp & 3;                                       // TMEM lane quarter this warp may access
    constexpr int CHUNKS = (TC_BN / 32) / (TC_EPI / 4);              // 32-column chunks per warp
    const int part = (warp - TC_EPI_WARP0) >> 2;                  // which slice of the 128-column tile
    int a = 0; uint32_t aph = 0; bool ok = true;
    for (int64_t t = blockIdx.x; t < total_tiles && ok; t += gridDim.x) {
      const int m_t = (int)(t % p.m_tiles);
      const int64_t n_t = t / p.m_tiles;
      const int c = m_t * TC_BM + q * 32 + lane;                  // this thread's output channel
      const bool cv = c < p.N;
      const int cc = cv ? c : 0;
      const float bia = p.bias ? p.bias[cc] : 0.0f;
      const float sc = p.scale ? p.scale[cc] : 1.0f;
      const float sh = p.shift ? p.shift[cc] : 0.0f;
      NeuronParams np{0.9f, 0.01f, 0.5f, 1.0f};
      if (ACT == ACT_LIF) { np.d = p.nparams[cc]; np.a = p.nparams[p.N + cc]; np.r = p.nparams[2 * p.N + cc]; np.th0 = p.nparams[3 * p.N + cc]; }
      if (!(ok = mbar_wait(bar_tfull(a), aph, p.err))) break;
      tc_fence_after();
      if (EXTRA == 3) {
        // fused attention tail (see gemm_tc2.cu): the tile holds TR / KK whole points; a warp takes every `parts`-th
        // point, one channel per lane: logits -> softmax over the KK edges -> sum_j a_j (v[nb_j] + pos[e_j])
        const int npts = TR / KK;
        constexpr int parts = TC_EPI / 4;
        {   // pull the pos rows of this CTA's NEXT tile (its 128-channel slab: 4 lines per row) into L2
          const int64_t tn = t + gridDim.x;
          if (tn < total_tiles) {
            const int64_t row0 = (tn / p.m_tiles) * TR;
            const int cb = (int)(tn % p.m_tiles) * TC_BM;
            for (int i = (warp - TC_EPI_WARP0) * 32 + lane; i < TR * 4; i += TC_EPI * 32) {
              const int64_t row = row0 + (i >> 2);
              if (row < p.R) prefetch_l2(p.at_pos + row * p.N + cb + (i & 3) * 32);
            }
          }
        }
        if (part < parts)
          attn_tail_dispatch<KK>(p, tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * TC_BN), part, parts, npts, n_t, c, bia, sc, sh, 1.0f);
      } else if (ACT == ACT_LIF) {
        // 8 columns at a time with the next piece's TMEM load in flight (see gemm_tc2.cu): keeps all 8 recurrences
        // interleaved instead of 32 live accumulators forcing ptxas to serialise them
        const int colw = part * CHUNKS * 32;
        const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * TC_BN + colw);
        float nxt[8];
        __syncwarp();
        tmem_ld_piece<8>(tbase, nxt);
        int my_qo = 0, my_ko = 0, nx_qo = 0, nx_ko = 0;          // EXTRA == 2: this / the next 32-row group's offsets
        float qv[8], kv[8];
        if (EXTRA == 2) {                                         // edge bias W q_i - W k_j: operands of piece 0
          edge_lane_offsets(p, n_t * TC_BN + colw, lane, my_qo, my_ko);
          edge_fetch8(p, my_qo, my_ko, 0, c, qv, kv);
        }
#pragma unroll 1
        for (int pc = 0; pc < CHUNKS * 4; ++pc) {
          float u[8];
          tmem_wait_ld8(nxt);
#pragma unroll
          for (int j = 0; j < 8; ++j) u[j] = nxt[j];
          if (pc + 1 < CHUNKS * 4) tmem_ld_piece<8>(tbase + (uint32_t)((pc + 1) * 8), nxt);
          const int64_t r0 = n_t * TC_BN + colw + pc * 8;
          const int nrows = (int)((p.R - r0) < 8 ? (p.R - r0) : 8);
          if (EXTRA == 2) {                                       // fold this piece's bias in, fetch the next one under the LIF
#pragma unroll
            for (int j = 0; j < 8; ++j) u[j] += qv[j] - kv[j];
            if ((pc & 3) == 0 && pc + 4 < CHUNKS * 4) edge_lane_offsets(p, n_t * TC_BN + colw + (pc + 4) * 8, lane, nx_qo, nx_ko);
            if (pc + 1 < CHUNKS * 4) {
              if (((pc + 1) & 3) == 0) { my_qo = nx_qo; my_ko = nx_ko; }
              edge_fetch8(p, my_qo, my_ko, (pc + 1) & 3, c, qv, kv);
            }
          }
          if (cv && nrows > 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j) u[j] = fmaf(u[j] + bia, sc, sh);
            lif_chain_vec_fast<8>(u, np, p.T);
            float* yp = p.Y + r0 * p.ldc + c;
            if (nrows == 8) {
#pragma unroll
              for (int j = 0; j < 8; ++j) { *yp = u[j]; yp += p.ldc; }
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j) { if (j < nrows) *yp = u[j]; yp += p.ldc; }
            }
          }
        }
      } else {
#pragma unroll 1
      for (int ch = 0; ch < CHUNKS; ++ch) {
        const int col0 = (part * CHUNKS + ch) * 32;
        float v[32];
        __syncwarp();                                             // tcgen05.ld is warp-collective (.sync.aligned)
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * TC_BN + col0), v);
        const int64_t r0 = n_t * TC_BN + col0;
        const int nrows = (int)((p.R - r0) < 32 ? (p.R - r0) : 32);     // <= 0 for tiles past the end
        if (cv && nrows > 0) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = fmaf(v[j] + bia, sc, sh);
        if (EXTRA == 1) {
          const float* rp = p.residual + r0 * p.ldr + c;
#pragma unroll
          for (int j = 0; j < 32; ++j) { if (j < nrows) v[j] += *rp; rp += p.ldr; }
        }
        if (ACT == ACT_LEAKY) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = act_leaky(v[j]);
        }
        if (ACT == ACT_GELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = act_gelu(v[j]);
        }
        if (ACT == ACT_LIF) {
#pragma unroll
          for (int j0 = 0; j0 < 32; j0 += 8) {
            float u[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) u[j] = v[j0 + j];
            lif_chain_vec_fast<8>(u, np, p.T);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j0 + j] = u[j];
          }
        }
        float* yp = p.Y + r0 * p.ldc + c;
        if (nrows == 32) {
#pragma unroll
          for (int j = 0; j < 32; ++j) { *yp = v[j]; yp += p.ldc; }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) { if (j < nrows) *yp = v[j]; yp += p.ldc; }
        }
        }
      }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty(a));
      if (++a == TC_ACC) { a = 0; aph ^= 1u; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// 2-D fp32 row-major [rows, K] (row stride ld floats) -> boxes of [box_rows, 32] with 128B swizzle, OOB rows/cols read as 0
int tc_make_map(CUtensorMap* m, const float* base, int64_t rows, int K, int64_t ld, int box_rows) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("gemm_tc: cuTensorMapEncodeTiled entry point unavailable"); return -2; }
  cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * sizeof(float)};
  cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("gemm_tc: cuTensorMapEncodeTiled failed (%d) rows=%lld K=%d ld=%lld", (int)r, (long long)rows, K, (long long)ld); return -2; }
  return 0;
}

int tc_make_map_f16(CUtensorMap* m, const void* base, int64_t rows, int K, int box_rows) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("gemm_tc: cuTensorMapEncodeTiled entry point unavailable"); return -2; }
  cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("gemm_tc: cuTensorMapEncodeTiled(f16) failed (%d) rows=%lld K=%d", (int)r, (long long)rows, K); return -2; }
  return 0;
}

// Pipeline-watchdog flag of the CURRENT device: one word of mapped pinned host memory per device (kernels of that device
// write it, the host reads it without touching any stream), allocated on first use.
namespace {
std::mutex g_flag_mu;
int* g_flag_host[64] = {};
int* g_flag_dev[64] = {};
}
int* tc_err_flag() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lk(g_flag_mu);
  if (!g_flag_dev[dev]) {
    int* h = nullptr; int* d = nullptr;
    if (cudaHostAlloc(reinterpret_cast<void**>(&h), sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) return nullptr;
    *h = 0;
    if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&d), h, 0) != cudaSuccess) { cudaFreeHost(h); return nullptr; }
    g_flag_host[dev] = h; g_flag_dev[dev] = d;
  }
  return g_flag_dev[dev];
}

bool gemm_tc_supported(const GemmArgs& g, int amode) {
  if (amode != A_PLAIN) return false;
  if (g.K % TC_BK != 0 || g.K < TC_BK) return false;
  if (g.R < 1024) return false;                                   // small row counts (decoder heads) stay on the SIMT engine
  if ((g.lda % 4) != 0 || (reinterpret_cast<uintptr_t>(g.A) & 15) || (reinterpret_cast<uintptr_t>(g.W) & 15)) return false;
  if (g.group != 0) return false;                                  // row-group max stays on the SIMT engine
  if (g.residual && g.act != ACT_NONE) return false;
  if (g.pool || g.x_h2 || g.out_h2 || g.pos_h2) return false;                  // fused max-pool epilogue, fp16-plane tensors: 2-CTA kernel only
  if (g.at_pos) {                                                  // fused attention tail (EXTRA == 3)
    if (!tc_fuse_attn_out_enabled() || g.act != ACT_NONE || g.residual || g.edge_bias || !g.at_v || !g.idx) return false;
    if (g.Mpts > 256 || tc_fused_tile_rows(g.kk) == 0 || g.R % g.kk != 0 || (g.N % 128) != 0 || !g.Whi || !g.Wlo) return false;
  }
  if (g.edge_bias && (g.act != ACT_LIF || (g.N % 128) != 0 || !g.Q || !g.Kf || !g.idx || g.kk < 1 || g.Mpts < 1)) return false;
  if (g.edge_bias && (g.R / g.kk + g.Mpts) * g.ldq >= ((int64_t)1 << 31)) return false;     // 32-bit gather offsets
  if (g.R >= ((int64_t)1 << 31) || g.N > (1 << 20)) return false;
  return true;
}

int launch_gemm_tc(const GemmArgs& g, int amode, cudaStream_t st) {
  SAPCU_REQUIRE(gemm_tc_supported(g, amode), "gemm_tc: unsupported problem");
  int* err = tc_err_flag();
  SAPCU_REQUIRE(err != nullptr, "gemm_tc: cannot allocate the watchdog flag");
  SAPCU_REQUIRE(!g.R_dev && !g.at_pid, "gemm_tc: device-side row counts and pair-indexed pos are 2-CTA engine features");
  const bool presplit = g.Whi != nullptr && g.Wlo != nullptr;
  CUtensorMap mw, mwlo, mx;
  int rc = tc_make_map(&mw, presplit ? g.Whi : g.W, g.N, g.K, g.K, TC_BM);
  if (rc) return rc;
  rc = tc_make_map(&mwlo, presplit ? g.Wlo : g.W, g.N, g.K, g.K, TC_BM);
  if (rc) return rc;
  const int tile_rows = g.at_pos ? tc_fused_tile_rows(g.kk) : TC_BN;
  rc = tc_make_map(&mx, g.A, g.R, g.K, g.lda, TC_BN);
  if (rc) return rc;
  TcParams p;
  p.R = g.R; p.N = g.N; p.K = g.K; p.bias = g.bias; p.scale = g.scale; p.shift = g.shift; p.act = g.act; p.T = g.T;
  p.nparams = g.nparams; p.residual = g.residual; p.ldr = g.ldr; p.Y = g.Y; p.ldc = g.ldc;
  p.aq = g.Q; p.ak = g.Kf; p.ldq = g.ldq; p.idx = g.idx; p.ldi = g.ldi; p.kk = g.kk; p.Mpts = g.Mpts;
  p.m_tiles = (int)ceil_div(g.N, TC_BM); p.n_tiles = ceil_div(g.R, tile_rows); p.err = err;
  p.pool = nullptr; p.pool_T = 0; p.pool_rows = 0; p.acc_scale = 1.0f; p.x_scale = 1.0f; p.out_h2 = 0; p.pos_h2 = 0;
  p.Y2 = nullptr; p.idx8 = g.idx8; p.ldi8w = g.ldi8w; p.at_pos = g.at_pos; p.at_v = g.at_v; p.at_ldv = g.at_ldv; p.at_sqrt = g.at_sqrt; p.tile_rows = tile_rows;
  p.split_w = presplit ? 0 : 1; p.passes = g.tc_passes == 1 ? 1 : 3;
  p.at_pid = nullptr; p.R_dev = nullptr;   // pair-indexed pos and device-side row counts: 2-CTA engine only
  const int64_t total = p.n_tiles * p.m_tiles;
  const int grid = (int)(total < kNumSMs ? total : kNumSMs);
  if (g.at_pos)
    return with_kk(g.kk, [&](auto KQ) { return tc_launch<gemm_tc_kernel<ACT_NONE, 3, decltype(KQ)::value>>(grid, TC_THREADS, TC_SMEM_BYTES, st, mw, mwlo, mx, p); });
  if (g.act == ACT_LIF && g.edge_bias) return tc_launch<gemm_tc_kernel<ACT_LIF, 2>>(grid, TC_THREADS, TC_SMEM_BYTES, st, mw, mwlo, mx, p);
  if (g.act == ACT_LIF) return tc_launch<gemm_tc_kernel<ACT_LIF, 0>>(grid, TC_THREADS, TC_SMEM_BYTES, st, mw, mwlo, mx, p);
  if (g.act == ACT_LEAKY) return tc_launch<gemm_tc_kernel<ACT_LEAKY, 0>>(grid, TC_THREADS, TC_SMEM_BYTES, st, mw, mwlo, mx, p);
  if (g.act == ACT_GELU) return tc_launch<gemm_tc_kernel<ACT_GELU, 0>>(grid, TC_THREADS, TC_SMEM_BYTES, st, mw, mwlo, mx, p);
  if (g.residual) return tc_launch<gemm_tc_kernel<ACT_NONE, 1>>(grid, TC_THREADS, TC_SMEM_BYTES, st, mw, mwlo, mx, p);
  return tc_launch<gemm_tc_kernel<ACT_NONE, 0>>(grid, TC_THREADS, TC_SMEM_BYTES, st, mw, mwlo, mx, p);
}

// Watchdog status of the current device (0 = fine).  The flag is host-visible, so this never touches a stream unless
// SAPCU_TC_SYNC_CHECK=1 asks for the old behaviour (synchronise `st` first: the check then covers the launches just
// enqueued, at the price of serialising the caller).  Without it a stall of THIS call's kernels is reported by the next
// entry point (or by sapcu_device_status after the caller synchronised).
int gemm_tc_check(cudaStream_t st) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
  if (settings().sync_check) SAPCU_CUDA_CHECK(cudaStreamSynchronize(st));
  int* h;
  { std::lock_guard<std::mutex> lk(g_flag_mu); h = g_flag_host[dev]; }
  if (h && *reinterpret_cast<volatile int*>(h)) {
    const int v = *reinterpret_cast<volatile int*>(h);
    *reinterpret_cast<volatile int*>(h) = 0;
    // bit 1: a pair table met a patch point index outside its cloud (edge_pairs.cu); else the pipeline watchdog (value 1)
    if (v & 2) { set_error("fn_forward_indexed / pair_table: a patch point index lies outside the cloud"); return -1; }   // SAPCU_EINVAL
    set_error("gemm_tc: pipeline watchdog fired (mbarrier protocol stall)");
    return -2;
  }
  return 0;
}

}  // namespace sapcu
