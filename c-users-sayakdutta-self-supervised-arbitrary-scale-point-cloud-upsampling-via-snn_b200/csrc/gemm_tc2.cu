// 2-CTA (cta_group::2) tcgen05 GEMM engine, used when N (output channels) % 256 == 0 -- and, as a single-CTA flavour of the
// same pipeline (template CG = 1), for the 128-channel layers whose operands arrive ready-made.
//
// Operand formats (template HM) and what each mode uses them for:
//   0  fp32 rows, 3xTF32 split in the kernel (or single-pass TF32)      point-level layers, every mode (+ LT: fc1 of the wide blocks, SAPCU_MODE_TC)
//   1  fp32 rows converted to fp16 (hi, lo) by the splitter warps        spike-tensor layers without plane hand-over: fd's per-point P|Q (SAPCU_MODE_TC)
//   2  fp16 (hi, lo) planes written by the producer, fp16x3 products     SAPCU_MODE_TC: fc_delta2, fc_gamma, fc_gamma2 + tail, q/k/v of the wide blocks, fd conv5
//   3  ONE fp16 plane, ONE product per MAC, 32 KiB stages                SAPCU_MODE_FAST: the same layers
//   4  fp32 rows, single-pass TF32, compact stages                       SAPCU_MODE_FAST: point-level LIF layers
// Template LT = 1: the LIF^T chain of the epilogue comes from the layer's table in shared memory (lif_table.cuh); the stage
// count shrinks so that pipeline + table fit 227 KiB.
// LIF epilogues store whole 8-row pieces through lif_store_piece<LD>: the model's row strides are compile-time constants there, so
// every store is an immediate offset from one base address per output tensor (the run-time-stride form is the fallback).
//
// A CTA pair (thread-block cluster of 2, same TPC) computes a 256-channel x 256-row tile with ONE
// tcgen05.mma.cta_group::2 stream issued by the leader CTA: each CTA stages only ITS 128 weight rows and ITS
// 128 activation rows (64 KiB per stage instead of 96 KiB for the same per-SM MMA work), so the shared-memory
// operand traffic per FLOP -- the limiter of the 1-CTA kernel (ncu: tensor pipe 57 % active, smem-bound) -- is
// halved.  Accumulators: each CTA's TMEM holds its 128 channels x 256 rows (2 buffers of 256 columns).
//
// Cross-CTA protocol (all waits are watchdogged):
//   raw[s]    local   TMA bytes of this CTA landed                       -> this CTA's splitter              (HM 0, 1)
//             LEADER  TMA bytes of BOTH CTAs (cp.async.bulk.tensor.cta_group::2 counts the follower's loads on the leader's
//                     barrier)                                          -> leader's MMA issuer, no splitter  (HM >= 2)
//   split[s]  LEADER  one arrival per splitter thread of both CTAs (the follower arrives remotely via mapa)   (HM 0, 1)
//   empty[s]  both    tcgen05.commit.cta_group::2 ... multicast::cluster (mask 0b11) -> each CTA's TMA producer
//   tfull[a]  both    multicast commit after the last k-block           -> each CTA's epilogue
//   tempty[a] LEADER  2 x EPI arrivals (epilogue warps of both CTAs)    -> leader's MMA issuer
// Roles per CTA: warp 0 TMA, warp 1 MMA (leader only; both CTAs allocate TMEM with cta_group::2), warps 2..3
// splitter (lo = x - trunc_tf32(x); the raw tile is the hi operand), warps 4..19 epilogue (same flavours as
// gemm_tc.cu, plus EXTRA == 4: max over the patch's points fused into the conv5 epilogue).
// ncu: on the K = 512 layers the MMA issuer never waits on a barrier -- the MMA stream is the limiter (tensor pipe
// ~71 % active = ~790 TFLOP/s of issued tf32 math under the board's power cap); K <= 256 LIF layers are MUFU-bound.
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdlib.h>
#include "gemm_tc.h"
#include "neuron.cuh"
#include "tc_ptx.cuh"
#include "lif_table.cuh"

namespace sapcu {

constexpr int T2_STAGES_MAX = 3;
constexpr int T2_ACC = 2;                       // 2 x 256 TMEM columns
constexpr int T2_BN = 256;                      // rows per pair tile (128 staged by each CTA)
constexpr int T2_SPLIT_WARP0 = 2, T2_SPLIT_WARPS = 2;
constexpr int T2_EPI_WARP0 = T2_SPLIT_WARP0 + T2_SPLIT_WARPS, T2_EPI = 16;   // 2 + 2 + 16 warps = 640 threads: 96 registers per thread for the epilogue
constexpr int T2_THREADS = (T2_EPI_WARP0 + T2_EPI) * 32;
constexpr int T2_FAST_STAGES = 4;               // pair flavour on compact (32 KiB) stages without a LIF table: stages in flight
constexpr size_t T2_SMEM_BYTES = (size_t)T2_STAGES_MAX * 4 * TC_TILE_BYTES + 1024 + 256;   // 3 x 64 KiB (tf32) = 2 x 96 KiB (fp16x3)

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 remAddr32;\n\t"
      "mapa.shared::cluster.u32 remAddr32, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [remAddr32];\n\t}"
      ::"r"(bar), "r"(cta)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_f16_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2cta(uint32_t bar) {      // arrives on `bar` in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3)
               : "memory");
}

// cta_group::1 flavours (CG == 1: the same kernel as a single-CTA "pair" for 128-channel layers, fast mode only)
__device__ __forceinline__ void umma_f16_1cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TMA load into THIS CTA's shared memory whose transaction bytes are counted on the barrier at the same offset in the pair's
// LEADER CTA (shared::cluster addresses carry the CTA's rank inside the pair in bit 24: cleared = the even CTA)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
template <int CG> __device__ __forceinline__ void tma_load_2d_cg(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  if (CG == 2) tma_load_2d_pair(dst, map, bar, c0, c1); else tma_load_2d(dst, map, bar, c0, c1);
}
template <int CG> __device__ __forceinline__ void umma_commit_cg(uint32_t bar) {
  if (CG == 2) umma_commit_2cta(bar); else umma_commit(bar);
}
template <int CG> __device__ __forceinline__ void cta_group_sync() {
  if (CG == 2) cluster_sync_all(); else __syncthreads();
}

// tile t -> (channel tile m_t, row tile n_t); 32-bit divide when the tile index fits
__device__ __forceinline__ void tile_split(int64_t t, int m_tiles, int& m_t, int64_t& n_t) {
  if (t < (1ll << 31)) { const uint32_t q = (uint32_t)t / (uint32_t)m_tiles; n_t = q; m_t = (int)((uint32_t)t - q * (uint32_t)m_tiles); }
  else { n_t = t / m_tiles; m_t = (int)(t - n_t * m_tiles); }
}
// one lane of the (converged) warp, chosen by the hardware: ptxas knows that exactly one thread runs the guarded region and
// issues its uniform-datapath instructions (UTMALDG, UTCHMMA, UTCBAR) without a per-operand uniformisation loop
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P_el;\n\t"
      "elect.sync _|P_el, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P_el;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// whole-warp wait: every lane polls, the outcome is voted so that it (and what depends on it) stays warp-uniform
__device__ __forceinline__ bool mbar_wait_warp(uint32_t bar, uint32_t parity, int* err) {
  return __all_sync(0xffffffffu, mbar_wait(bar, parity, err));
}

// Store one 8-row piece of a LIF epilogue (one channel per thread): fmt 0 = fp32 rows, 1 = fp16 (hi, lo) planes of y * 2^13 (+ the
// fp32 copy p.Y2 when set), 2 = one fp16 plane (fast mode).  LD > 0: compile-time row stride, whole piece (STG [base + imm]); LD == 0:
// run-time stride, `nrows` valid rows.
template <int LD>
__device__ __forceinline__ void lif_store_piece(const TcParams& p, const float (&u)[8], int64_t r0, int c, int fmt, int nrows = 8) {
  const uint32_t ld = LD ? (uint32_t)LD : (uint32_t)p.ldc;
  const int64_t off = r0 * (LD ? (int64_t)LD : p.ldc) + c;
  if (fmt == 2) {
    __half* hp = reinterpret_cast<__half*>(p.Y) + off;
#pragma unroll
    for (int j = 0; j < 8; ++j) if (LD || j < nrows) hp[(uint32_t)j * ld] = __float2half_rn(u[j] * 8192.0f);
  } else if (fmt == 1) {
    if (p.Y2) {
      float* y2p = p.Y2 + off;
#pragma unroll
      for (int j = 0; j < 8; ++j) if (LD || j < nrows) y2p[(uint32_t)j * ld] = u[j];
    }
    __half* hp = reinterpret_cast<__half*>(p.Y) + off;
    __half* lp = hp + p.R * (LD ? (int64_t)LD : p.ldc);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (LD || j < nrows) {
        const float ys = u[j] * 8192.0f;
        const __half h = __float2half_rn(ys);
        hp[(uint32_t)j * ld] = h;
        lp[(uint32_t)j * ld] = __float2half_rn(ys - __half2float(h));
      }
    }
  } else {
    float* yp = p.Y + off;
#pragma unroll
    for (int j = 0; j < 8; ++j) if (LD || j < nrows) yp[(uint32_t)j * ld] = u[j];
  }
}

// H16 = fp16x3 operand format (activations known to be LIF outputs): W arrives as pre-split fp16 (hi, lo) of W * 2^e, the
// splitter turns the raw fp32 activation tile into fp16 (hi, lo) of x * x_scale, and 12 kind::f16 MMAs per 64-wide
// k-block (hi*hi + hi*lo + lo*hi, fp32 accumulate) replace 24 kind::tf32 ones: the same 22-bit products at twice the
// tensor-pipe rate and 2/3 of the operand bytes.  Stage = W_hi, W_lo, X_hi, X_lo (16 KiB each) + 32 KiB raw X; 2 stages.
// HM == 3 (SAPCU_MODE_FAST): ONE fp16 product per MAC.  W = the hi half of the fp16 split, activations = a single fp16 plane of
// x * 2^13 written by the producing epilogue: two TMA loads and 4 kind::f16 MMAs per 64-wide k-block, 32 KiB per stage.
// LT (with ACT_LIF): the LIF^T chain of the epilogue is read from the per-channel piecewise-cubic table (lif_table.cuh) that
// the epilogue warps copy into shared memory once per CTA (a CTA pair keeps its channel block for its whole life).
// CG: CTAs per tile.  2 = the CTA pair described above (256 channels per tile).  1 = the same pipeline in one CTA (128
// channels x 256 rows per tile, cta_group::1 MMAs, no cluster): the 128-channel layers of the first fn block in the fast
// mode, which then share the single-plane operands, the LIF tables and the fused attention tail with the wide layers.
template <int ACT, int EXTRA, int KK, int HM = 0, int LT = 0, int CG = 2>
__global__ void __cluster_dims__(CG, 1, 1) __launch_bounds__(T2_THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_wlo,
                const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_x2, const TcParams p) {
  // HM: 0 = 3xTF32; 1 = fp16x3, raw fp32 activations converted by the splitter warps; 2 = fp16x3, activations already
  // stored as fp16 (hi, lo) planes of x * 2^13 by the kernel that produced them (map_x = hi plane, map_x2 = lo plane): four
  // TMA loads per stage, no conversion, no raw staging -- a third less shared-memory traffic per k-block
  static_assert(CG == 2 || HM >= 2, "the single-CTA flavour takes ready-made operands only (fp16 planes, or the fast mode's formats)");
  constexpr bool H16 = HM == 1 || HM == 2 || HM == 3;        // fp16 operands (HM == 4: single-pass TF32 on fp32 activations)
  constexpr int CW = CG * 128;                               // output channels per tile
  constexpr bool FASTOP = HM == 3 || HM == 4;               // compact stages: one weight tile + one activation tile
  // stages: HM 2 (two fp16 planes per operand, 64 KiB per stage for a pair, 96 KiB single-CTA): 3 / 2 plain, 2 / 1 next to a LIF table
  constexpr int T2_STAGES = HM == 1 ? 2 : (FASTOP && !LT) ? (CG == 2 ? T2_FAST_STAGES : 4) : (FASTOP && CG == 1) ? 2 : FASTOP ? 3 : (CG == 2 ? (LT ? 2 : 3) : (LT ? 1 : 2));
  constexpr uint32_t T2_STAGE_BYTES = (HM == 1 ? 6 : FASTOP ? (CG == 2 ? 2 : 3) : (CG == 2 ? 4 : 6)) * TC_TILE_BYTES;   // HM 3/4: W tile + 128 (pair) or 256 activation rows
  constexpr uint32_t X_TILE = FASTOP ? 1 : 2;               // position of the activation (hi) tile inside a stage
  constexpr uint32_t X_LO_OFF = (CG == 2 ? 3 : 4) * TC_TILE_BYTES;   // lo activation tile (HM 0..2): behind the hi tile of 128 / 256 rows
  constexpr int BKE = H16 ? 64 : TC_BK;                    // k elements per stage
  constexpr bool DIRECT = HM >= 2;                          // operands arrive ready-made: no splitter hop (see the protocol above)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + T2_STAGES * T2_STAGE_BYTES;
  auto bar_raw = [&](int s) { return bar_base + 8u * s; };
  auto bar_split = [&](int s) { return bar_base + 8u * (T2_STAGES + s); };
  auto bar_empty = [&](int s) { return bar_base + 8u * (2 * T2_STAGES + s); };
  auto bar_tfull = [&](int a) { return bar_base + 8u * (3 * T2_STAGES + a); };
  auto bar_tempty = [&](int a) { return bar_base + 8u * (3 * T2_STAGES + T2_ACC + a); };
  const uint32_t tmem_slot = bar_base + 8u * (3 * T2_STAGES + 2 * T2_ACC);
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + T2_STAGES * T2_STAGE_BYTES + 8 * (3 * T2_STAGES + 2 * T2_ACC));

  // warp index, pair rank and (below) the TMEM base go through a shuffle so that the compiler can prove them warp-uniform: the
  // single-thread roles (TMA producer, MMA issuer) then keep their loop state, coordinates and descriptors in uniform
  // registers instead of re-uniformising every operand of every UTMALDG / UTCHMMA (ncu: those two warps, not the tensor
  // pipe, bounded the 32 KiB-stage flavours at ~850 clocks per k-block)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const uint32_t rank = CG == 2 ? __shfl_sync(0xffffffffu, cluster_ctarank(), 0) : 0u;  // 0 = leader
  const int64_t pair = blockIdx.x / CG, npairs = gridDim.x / CG;
  const int nk = p.K / BKE;
  const int64_t total_tiles = p.n_tiles * p.m_tiles;       // m_tiles = N / 256 (channel pairs), n_tiles = ceil(R / tile_rows)
  const int TR = p.tile_rows;                              // rows a tile advances by (256; whole points only when EXTRA == 3)
  constexpr int HALF = T2_BN / CG;                         // rows staged by each CTA: the MMA always spans 256 rows
  // instruction descriptor: D = F32, A = B = TF32 (2) or F16 (0), K-major, M = 256 (pair), N = 256
  constexpr uint32_t idesc = (1u << 4) | ((H16 ? 0u : 2u) << 7) | ((H16 ? 0u : 2u) << 10) | ((uint32_t)(T2_BN >> 3) << 17) | ((uint32_t)(CW >> 4) << 24);

  if (threadIdx.x == 0) {
    for (int s = 0; s < T2_STAGES; ++s) { mbar_init(bar_raw(s), 1); mbar_init(bar_split(s), CG * T2_SPLIT_WARPS * 32); mbar_init(bar_empty(s), 1); }
    for (int a = 0; a < T2_ACC; ++a) { mbar_init(bar_tfull(a), 1); mbar_init(bar_tempty(a), CG * T2_EPI); }
    fence_barrier_init();
    tma_prefetch_desc(&map_w); tma_prefetch_desc(&map_wlo); tma_prefetch_desc(&map_x);
  }
  if (warp == 1) {
    if (CG == 2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  cta_group_sync<CG>();                                     // barriers of both CTAs initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_gen, 0);

  if (warp == 0) {
    // ======================================================================== TMA producer (each CTA: its own halves)
    // the whole warp walks the loop (waits are voted warp-uniform), one elected lane issues
    int s = 0; uint32_t ph = 0; bool ok = true;
    for (int64_t t = pair; t < total_tiles && ok; t += npairs) {
      int m_t; int64_t n_t;
      tile_split(t, p.m_tiles, m_t, n_t);
      const int wrow = m_t * CW + (int)rank * 128;
      const int xrow = (int)(n_t * TR) + (int)rank * HALF;
      int xrow_nx = -1;                                          // activation rows of this pair's next tile (L2 prefetch target)
      if (t + npairs < total_tiles) {
        int m_n; int64_t n_n;
        tile_split(t + npairs, p.m_tiles, m_n, n_n);
        xrow_nx = (int)(n_n * TR) + (int)rank * HALF;
      }
      for (int kb = 0; kb < nk; ++kb) {
        int kp = kb + TC_L2_PREFETCH, xr = xrow;
        if (kp >= nk) { kp -= nk; xr = xrow_nx; }
        if (kp < nk && xr >= 0 && elect_one()) {
          tma_prefetch_l2_2d(&map_x, kp * BKE, xr);
          if (HM == 1) tma_prefetch_l2_2d(&map_x, kp * BKE + 32, xr);
          if (HM == 2) tma_prefetch_l2_2d(&map_x2, kp * BKE, xr);
        }
        if (!(ok = mbar_wait_warp(bar_empty(s), ph ^ 1u, p.err))) break;
        const uint32_t st = smem_base + s * T2_STAGE_BYTES;
        if (elect_one()) {
          if (FASTOP) {
            // DIRECT flavours: only the leader arms its barrier, for the bytes of BOTH CTAs; each CTA's loads report there
            if (rank == 0) mbar_expect_tx(bar_raw(s), CG * T2_STAGE_BYTES);
            tma_load_2d_cg<CG>(st, &map_w, bar_raw(s), kb * BKE, wrow);                // fp16 tiles: 64 halfs x 128 weight rows, x HALF activation rows
            tma_load_2d_cg<CG>(st + TC_TILE_BYTES, &map_x, bar_raw(s), kb * BKE, xrow);
          } else if (HM == 2) {
            if (rank == 0) mbar_expect_tx(bar_raw(s), CG * T2_STAGE_BYTES);
            tma_load_2d_cg<CG>(st, &map_w, bar_raw(s), kb * BKE, wrow);                // four fp16 tiles: 64 halfs x 128 (256 single-CTA) rows
            tma_load_2d_cg<CG>(st + TC_TILE_BYTES, &map_wlo, bar_raw(s), kb * BKE, wrow);
            tma_load_2d_cg<CG>(st + 2 * TC_TILE_BYTES, &map_x, bar_raw(s), kb * BKE, xrow);
            tma_load_2d_cg<CG>(st + X_LO_OFF, &map_x2, bar_raw(s), kb * BKE, xrow);
          } else if (H16) {
            mbar_expect_tx(bar_raw(s), 4 * TC_TILE_BYTES);
            tma_load_2d(st, &map_w, bar_raw(s), kb * BKE, wrow);                       // fp16 tiles: 64 halfs x 128 rows
            tma_load_2d(st + TC_TILE_BYTES, &map_wlo, bar_raw(s), kb * BKE, wrow);
            tma_load_2d(st + 4 * TC_TILE_BYTES, &map_x, bar_raw(s), kb * BKE, xrow);    // raw fp32: two 32-float boxes
            tma_load_2d(st + 5 * TC_TILE_BYTES, &map_x, bar_raw(s), kb * BKE + 32, xrow);
          } else {
            mbar_expect_tx(bar_raw(s), (p.passes == 3 ? 3 : 2) * TC_TILE_BYTES);
            tma_load_2d(st, &map_w, bar_raw(s), kb * TC_BK, wrow);
            if (p.passes == 3) tma_load_2d(st + TC_TILE_BYTES, &map_wlo, bar_raw(s), kb * TC_BK, wrow);
            tma_load_2d(st + 2 * TC_TILE_BYTES, &map_x, bar_raw(s), kb * TC_BK, xrow);
          }
        }
        __syncwarp();
        if (++s == T2_STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ======================================================================== MMA issuer (leader CTA only; one elected lane issues)
    if (rank == 0) {
      int s = 0, a = 0; uint32_t ph = 0, aph = 0; bool ok = true;
      for (int64_t t = pair; t < total_tiles && ok; t += npairs) {
        if (!(ok = mbar_wait_warp(bar_tempty(a), aph ^ 1u, p.err))) break;
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(a * T2_BN);
        for (int kb = 0; kb < nk; ++kb) {
          if (!(ok = mbar_wait_warp(DIRECT ? bar_raw(s) : bar_split(s), ph, p.err))) break;
          tc_fence_after();
          const uint32_t st = smem_base + s * T2_STAGE_BYTES;
          const uint64_t w_hi = umma_desc_sw128(st), w_lo = umma_desc_sw128(st + TC_TILE_BYTES);
          const uint64_t x_hi = umma_desc_sw128(st + X_TILE * TC_TILE_BYTES), x_lo = umma_desc_sw128(st + X_LO_OFF);
          if (elect_one()) {
          if (HM == 4) {                                         // single-pass TF32 on raw fp32 activations (8 floats = 32 B per MMA)
#pragma unroll
            for (int k8 = 0; k8 < TC_BK / 8; ++k8) {
              if (CG == 2) umma_tf32_2cta(tmem_d, w_hi + (uint64_t)(k8 * 2), x_hi + (uint64_t)(k8 * 2), idesc, (kb | k8) ? 1u : 0u);
              else umma_tf32(tmem_d, w_hi + (uint64_t)(k8 * 2), x_hi + (uint64_t)(k8 * 2), idesc, (kb | k8) ? 1u : 0u);
            }
          } else if (HM == 3) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              if (CG == 2) umma_f16_2cta(tmem_d, w_hi + (uint64_t)(ks * 2), x_hi + (uint64_t)(ks * 2), idesc, (kb | ks) ? 1u : 0u);
              else umma_f16_1cta(tmem_d, w_hi + (uint64_t)(ks * 2), x_hi + (uint64_t)(ks * 2), idesc, (kb | ks) ? 1u : 0u);
            }
          } else if (H16) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {                       // 16 halfs = 32 B = 2 x 16 B along the swizzled row
              const uint64_t adv = (uint64_t)(ks * 2);
              if (CG == 2) {
                umma_f16_2cta(tmem_d, w_lo + adv, x_hi + adv, idesc, (kb | ks) ? 1u : 0u);
                umma_f16_2cta(tmem_d, w_hi + adv, x_lo + adv, idesc, 1u);
                umma_f16_2cta(tmem_d, w_hi + adv, x_hi + adv, idesc, 1u);
              } else {
                umma_f16_1cta(tmem_d, w_lo + adv, x_hi + adv, idesc, (kb | ks) ? 1u : 0u);
                umma_f16_1cta(tmem_d, w_hi + adv, x_lo + adv, idesc, 1u);
                umma_f16_1cta(tmem_d, w_hi + adv, x_hi + adv, idesc, 1u);
              }
            }
          } else {
#pragma unroll
            for (int k8 = 0; k8 < TC_BK / 8; ++k8) {
              const uint64_t adv = (uint64_t)(k8 * 2);
              if (p.passes == 3) {
                umma_tf32_2cta(tmem_d, w_lo + adv, x_hi + adv, idesc, (kb | k8) ? 1u : 0u);
                umma_tf32_2cta(tmem_d, w_hi + adv, x_lo + adv, idesc, 1u);
                umma_tf32_2cta(tmem_d, w_hi + adv, x_hi + adv, idesc, 1u);
              } else {
                umma_tf32_2cta(tmem_d, w_hi + adv, x_hi + adv, idesc, (kb | k8) ? 1u : 0u);
              }
            }
          }
          umma_commit_cg<CG>(bar_empty(s));
          if (kb == nk - 1) umma_commit_cg<CG>(bar_tfull(a));
          }
          __syncwarp();
          if (++s == T2_STAGES) { s = 0; ph ^= 1u; }
        }
        if (++a == T2_ACC) { a = 0; aph ^= 1u; }
      }
    }
  } else if (warp < T2_EPI_WARP0) {
    // ======================================================================== splitter: X_lo = x - trunc_tf32(x)
    const int tid = threadIdx.x - T2_SPLIT_WARP0 * 32;
    int s = 0; uint32_t ph = 0; bool ok = !DIRECT;            // ready-made operands: the TMA engine signals the issuer itself
    for (int64_t t = pair; t < total_tiles && ok; t += npairs) {
      for (int kb = 0; kb < nk; ++kb) {
        if (!(ok = mbar_wait(bar_raw(s), ph, p.err))) break;
        uint8_t* st = smem_gen + s * T2_STAGE_BYTES;
        if (H16) {
          // raw fp32 boxes (128B-swizzled rows of 32 floats) -> fp16 hi / lo tiles in the same swizzled K-major layout:
          // item (r, c) = 8 consecutive k of row r: two 16-byte raw chunks in, one 16-byte chunk out per tile
          const uint8_t* raw = st + 4 * TC_TILE_BYTES;
          uint8_t* xh = st + 2 * TC_TILE_BYTES;
          uint8_t* xl = st + 3 * TC_TILE_BYTES;
          const float xs = p.x_scale;
#pragma unroll 4
          for (int i = tid; i < 128 * 8; i += T2_SPLIT_WARPS * 32) {
            const int r = i >> 3, c = i & 7, sw = r & 7;
            const uint8_t* src = raw + (c >> 2) * TC_TILE_BYTES + r * 128;
            const int f0 = (c & 3) * 2;
            const float4 a = *reinterpret_cast<const float4*>(src + ((f0 ^ sw) << 4));
            const float4 b = *reinterpret_cast<const float4*>(src + (((f0 + 1) ^ sw) << 4));
            const float v[8] = {a.x * xs, a.y * xs, a.z * xs, a.w * xs, b.x * xs, b.y * xs, b.z * xs, b.w * xs};
            uint32_t ho[4], lo4[4];
#pragma unroll
            for (int q2 = 0; q2 < 4; ++q2) {
              const __half2 h = __floats2half2_rn(v[2 * q2], v[2 * q2 + 1]);
              const float2 hf = __half22float2(h);
              const __half2 l = __floats2half2_rn(v[2 * q2] - hf.x, v[2 * q2 + 1] - hf.y);
              ho[q2] = *reinterpret_cast<const uint32_t*>(&h);
              lo4[q2] = *reinterpret_cast<const uint32_t*>(&l);
            }
            const int dst = r * 128 + ((c ^ sw) << 4);
            *reinterpret_cast<uint4*>(xh + dst) = make_uint4(ho[0], ho[1], ho[2], ho[3]);
            *reinterpret_cast<uint4*>(xl + dst) = make_uint4(lo4[0], lo4[1], lo4[2], lo4[3]);
          }
          fence_proxy_async();
          if (rank == 0) mbar_arrive(bar_split(s)); else mbar_arrive_cluster(bar_split(s), 0);
          if (++s == T2_STAGES) { s = 0; ph ^= 1u; }
          continue;
        }
        const float4* hi = reinterpret_cast<const float4*>(st + 2 * TC_TILE_BYTES);
        float4* lo = reinterpret_cast<float4*>(st + 3 * TC_TILE_BYTES);
#pragma unroll
        for (int i = 0; i < (int)(TC_TILE_BYTES / 16) / (T2_SPLIT_WARPS * 32); ++i) {
          if (p.passes == 1) break;                               // single-pass TF32: nothing to split
          const int e = tid + i * T2_SPLIT_WARPS * 32;
          const float4 v = hi[e];
          float4 l;
          l.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
          l.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
          l.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
          l.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
          lo[e] = l;
        }
        fence_proxy_async();
        if (rank == 0) mbar_arrive(bar_split(s)); else mbar_arrive_cluster(bar_split(s), 0);
        if (++s == T2_STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // ======================================================================== epilogue (this CTA's 128 channels x 256 rows)
    const int q = warp & 3;
    constexpr int CHUNKS = (T2_BN / 32) / (T2_EPI / 4);
    const int part = (warp - T2_EPI_WARP0) >> 2;
    int a = 0; uint32_t aph = 0; bool ok = true;
    // LT: this CTA's 128-channel block of the tabulated LIF^T chain -> shared memory (behind the barriers), once
    uint32_t lt_desc = 0;                                        // shared-memory address of this lane's descriptor column
    if (LT) {
      const int blk = (int)(pair % p.m_tiles) * CG + (int)rank;       // the host keeps npairs a multiple of m_tiles: fixed channel block
      uint8_t* tsm = smem_gen + T2_STAGES * T2_STAGE_BYTES + 256;
      lif_table_load(p.lif_tab + (size_t)blk * p.lif_tab_stride, tsm, p.lif_tab_stride, threadIdx.x - T2_EPI_WARP0 * 32, T2_EPI * 32);
      asm volatile("bar.sync 1, %0;" ::"r"(T2_EPI * 32) : "memory");
      lt_desc = smem_u32(tsm) + (uint32_t)(q * 32 + lane) * 8u;
    }
    for (int64_t t = pair; t < total_tiles && ok; t += npairs) {
      int m_t; int64_t n_t;
      tile_split(t, p.m_tiles, m_t, n_t);
      const int c = m_t * CW + (int)rank * 128 + q * 32 + lane;
      const float bia = p.bias ? p.bias[c] : 0.0f;
      const float sc = p.scale ? p.scale[c] : 1.0f;
      const float sh = p.shift ? p.shift[c] : 0.0f;
      NeuronParams np{0.9f, 0.01f, 0.5f, 1.0f};
      if (ACT == ACT_LIF) { np.d = p.nparams[c]; np.a = p.nparams[p.N + c]; np.r = p.nparams[2 * p.N + c]; np.th0 = p.nparams[3 * p.N + c]; }
      if (!(ok = mbar_wait(bar_tfull(a), aph, p.err))) break;
      tc_fence_after();
      if (EXTRA == 3) {
        // fused attention tail: this tile holds TR / KK whole points; a warp takes every `parts`-th point, one
        // channel per lane: logits -> softmax over the KK edges -> sum_j a_j (v[nb_j] + pos[e_j])
        const int npts = TR / KK;
        constexpr int parts = T2_EPI / 4;
        {   // pull the pos rows of this pair's NEXT tile (this CTA's 128-channel slab: 4 lines per row) into L2
          const int64_t tn = t + npairs;
          if (tn < total_tiles) {
            const int64_t row0 = (tn / p.m_tiles) * TR;
            const int cb = (int)(tn % p.m_tiles) * CW + (int)rank * 128;
            for (int i = (warp - T2_EPI_WARP0) * 32 + lane; i < TR * 4; i += T2_EPI * 32) {
              const int64_t row = row0 + (i >> 2);
              if (row >= p.R) continue;
              if (p.pos_h2 == 2) { if (!(i & 2)) prefetch_l2(reinterpret_cast<const __half*>(p.at_pos) + row * p.N + cb + (i & 1) * 64); }
              else if (p.pos_h2) prefetch_l2(reinterpret_cast<const __half*>(p.at_pos) + ((i & 2) ? p.R * (int64_t)p.N : 0) + row * p.N + cb + (i & 1) * 64);
              else prefetch_l2(p.at_pos + row * p.N + cb + (i & 3) * 32);
            }
          }
        }
        if (part < parts)
          attn_tail_dispatch<KK>(p, tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * T2_BN), part, parts, npts, n_t, c, bia, sc, sh, H16 ? p.acc_scale : 1.0f);
      } else if (ACT == ACT_LIF) {
        // 8 columns (= rows of Y) at a time: 24 state + 24 temporary registers leave ptxas room to interleave all 8
        // recurrences (with 32 accumulators live it serialised half of them); the next piece is loaded under the math
        const int colw = part * CHUNKS * 32;
        const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * T2_BN + colw);
        float nxt[8];
        __syncwarp();
        tmem_ld_piece<8>(tbase, nxt);
        int my_qo = 0, my_ko = 0, nx_qo = 0, nx_ko = 0;          // EXTRA == 2: this / the next 32-row group's offsets
        float qv[8], kv[8];
        if (EXTRA == 2) {                                         // edge bias W q_i - W k_j: operands of piece 0
          edge_lane_offsets(p, n_t * T2_BN + colw, lane, my_qo, my_ko);
          edge_fetch8(p, my_qo, my_ko, 0, c, qv, kv);
        }
#pragma unroll 1
        for (int pc = 0; pc < CHUNKS * 4; ++pc) {
          float u[8];
          tmem_wait_ld8(nxt);
          // LT: the accumulator's power-of-two scale is folded into the BatchNorm scale below (exact), no multiply here
#pragma unroll
          for (int j = 0; j < 8; ++j) u[j] = (H16 && !LT) ? nxt[j] * p.acc_scale : nxt[j];
          if (pc + 1 < CHUNKS * 4) tmem_ld_piece<8>(tbase + (uint32_t)((pc + 1) * 8), nxt);
          const int64_t r0 = n_t * T2_BN + colw + pc * 8;
          const int nrows = (int)((p.R - r0) < 8 ? (p.R - r0) : 8);
          float eb[8];                                            // LT: the edge bias joins the table coordinate's multiply-add
          if (EXTRA == 2) {                                       // fold this piece's bias in, fetch the next one under the LIF
#pragma unroll
            for (int j = 0; j < 8; ++j) { if (LT) eb[j] = qv[j] - kv[j]; else u[j] += qv[j] - kv[j]; }
            if ((pc & 3) == 0 && pc + 4 < CHUNKS * 4) edge_lane_offsets(p, n_t * T2_BN + colw + (pc + 4) * 8, lane, nx_qo, nx_ko);
            if (pc + 1 < CHUNKS * 4) {
              if (((pc + 1) & 3) == 0) { my_qo = nx_qo; my_ko = nx_ko; }
              edge_fetch8(p, my_qo, my_ko, (pc + 1) & 3, c, qv, kv);
            }
          }
          if (nrows > 0) {
            if (LT) {
              // one multiply-add from the (scaled) accumulator straight to the table coordinate x = BN(acc + bias) - theta0
              const float bx = fmaf(bia, sc, sh) - np.th0;
              const float sca = H16 ? sc * p.acc_scale : sc;       // acc_scale is a power of two: acc * (scale * 2^-n) is exact
#pragma unroll
              for (int j = 0; j < 8; ++j) u[j] = fmaf(u[j], sca, EXTRA == 2 ? fmaf(eb[j], sc, bx) : bx);
              float x0[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) x0[j] = u[j];
              if (lif_table_eval_vec<8>(u, lt_desc)) {   // some |x| >= 255 (or NaN): the exact chain for those
#pragma unroll
                for (int j = 0; j < 8; ++j) if (lif_table_oob(x0[j])) u[j] = lif_chain<false>(x0[j] + np.th0, np, p.T);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j) u[j] = fmaf(u[j] + bia, sc, sh);
              if (FASTOP) lif_chain_vec_fast2<8>(u, np, p.T);
              else lif_chain_vec_fast<8>(u, np, p.T);
            }
            // whole pieces (all but the tensor's last rows) with one of the model's row strides: the stride becomes a compile-time
            // constant and every store of the piece an immediate offset from ONE base address per output tensor
            const int fmt = (HM == 3 && p.out_h2 == 2) ? 2 : p.out_h2 ? 1 : 0;
            const int64_t ld = p.ldc;
            if (nrows == 8 && ld == 512) lif_store_piece<512>(p, u, r0, c, fmt);
            else if (nrows == 8 && ld == 256) lif_store_piece<256>(p, u, r0, c, fmt);
            else if (nrows == 8 && ld == 128) lif_store_piece<128>(p, u, r0, c, fmt);
            else if (nrows == 8 && ld == 1536) lif_store_piece<1536>(p, u, r0, c, fmt);
            else if (nrows == 8 && ld == 768) lif_store_piece<768>(p, u, r0, c, fmt);
            else lif_store_piece<0>(p, u, r0, c, fmt, nrows);
          }
        }
      } else {
      // EXTRA == 4 (conv5 + max over the patch's points): the epilogue function f = act(BN(acc * acc_scale + bias)) is a chain of
      // monotone roundings, non-decreasing in acc * sgn(BN scale), so max_j f(acc_j) == f(sgn * max_j(sgn * acc_j)) exactly: the
      // RAW oriented accumulators are pooled (one multiply + a share of a max per element) and f runs once per (patch, step,
      // channel) at the flush.  mx[q8] = running max of step q8 of patch mx_patch.
      static_assert(EXTRA != 4 || ACT == ACT_NONE || ACT == ACT_LEAKY, "the pooled epilogue needs a monotone activation");
      float mx[8];
      int64_t mx_patch = -1;
      const float sgn = sc < 0.0f ? -1.0f : 1.0f;
#pragma unroll
      for (int q8 = 0; q8 < 8; ++q8) mx[q8] = -INFINITY;
      auto pool_flush = [&]() {
        if (mx_patch >= 0) {
#pragma unroll
          for (int q8 = 0; q8 < 8; ++q8)
            if (q8 < p.pool_T && mx[q8] > -INFINITY) {
              const float m = mx[q8] * sgn;
              float y = fmaf((H16 ? m * p.acc_scale : m) + bia, sc, sh);
              if (ACT == ACT_LEAKY) y = act_leaky(y);
              atomic_max_float(p.pool + (mx_patch * p.pool_T + q8) * p.N + c, y);
            }
        }
#pragma unroll
        for (int q8 = 0; q8 < 8; ++q8) mx[q8] = -INFINITY;
      };
#pragma unroll 1
      for (int ch = 0; ch < CHUNKS; ++ch) {
        const int col0 = (part * CHUNKS + ch) * 32;
        float v[32];
        __syncwarp();
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * T2_BN + col0), v);
        const int64_t r0 = n_t * T2_BN + col0;
        const int nrows = (int)((p.R - r0) < 32 ? (p.R - r0) : 32);
        if (nrows > 0) {
          if (EXTRA == 4) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= sgn;
            int64_t patch; uint32_t prow;                         // r0 = patch * pool_rows + prow (32-bit divide when it fits)
            if ((uint64_t)r0 <= 0xffffffffull && (uint64_t)p.pool_rows <= 0xffffffffull) {
              const uint32_t pq = (uint32_t)r0 / (uint32_t)p.pool_rows;
              patch = pq; prow = (uint32_t)r0 - pq * (uint32_t)p.pool_rows;
            } else { patch = r0 / p.pool_rows; prow = (uint32_t)(r0 - patch * p.pool_rows); }
            const int lim1 = (int)((p.pool_rows - prow) < nrows ? (p.pool_rows - prow) : nrows);   // rows still in `patch`
            if (patch != mx_patch) { pool_flush(); mx_patch = patch; }
            int tt = p.pool_T == 7 ? (int)(prow % 7u) : (int)(prow % (uint32_t)p.pool_T);
            if (p.pool_T == 7 && lim1 == 32) {
              // whole chunk inside one patch, rows = (point, step) with 7 steps: the rows of residue s (mod 7) share a step
              float a7[7];
#pragma unroll
              for (int s7 = 0; s7 < 7; ++s7) {
                a7[s7] = v[s7];
#pragma unroll
                for (int j = s7 + 7; j < 32; j += 7) a7[s7] = fmaxf(a7[s7], v[j]);
              }
#pragma unroll
              for (int r7 = 0; r7 < 7; ++r7)
                if (tt == r7) {
#pragma unroll
                  for (int s7 = 0; s7 < 7; ++s7) mx[(r7 + s7) % 7] = fmaxf(mx[(r7 + s7) % 7], a7[s7]);
                }
            } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (j < lim1) {
#pragma unroll
                for (int q8 = 0; q8 < 8; ++q8) if (q8 == tt) mx[q8] = fmaxf(mx[q8], v[j]);
              }
              tt = (tt + 1 == p.pool_T) ? 0 : tt + 1;
            }
            if (lim1 < nrows) {                                 // the chunk straddles a patch boundary (pool_rows % T == 0)
              pool_flush(); mx_patch = patch + 1;
              tt = 0;
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                if (j >= lim1 && j < nrows) {
#pragma unroll
                  for (int q8 = 0; q8 < 8; ++q8) if (q8 == tt) mx[q8] = fmaxf(mx[q8], v[j]);
                  tt = (tt + 1 == p.pool_T) ? 0 : tt + 1;
                }
              }
            }
            }
          } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaf((H16 ? v[j] * p.acc_scale : v[j]) + bia, sc, sh);
          if (EXTRA == 1) {
            const float* rp = p.residual + r0 * p.ldr + c;
#pragma unroll
            for (int j = 0; j < 32; ++j) { if (j < nrows) v[j] += *rp; rp += p.ldr; }
          }
          if (ACT == ACT_LEAKY) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = act_leaky(v[j]);
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
      if (EXTRA == 4) pool_flush();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { if (rank == 0) mbar_arrive(bar_tempty(a)); else mbar_arrive_cluster(bar_tempty(a), 0); }
      if (++a == T2_ACC) { a = 0; aph ^= 1u; }
    }
  }
  tc_fence_before();
  cta_group_sync<CG>();                                     // nobody leaves while the peer may still touch its smem / barriers
  if (warp == 1) {
    tc_fence_after();
    if (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

__global__ void fill_kernel(float* __restrict__ p, int64_t n, float v) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
int launch_fill(float* p, int64_t n, float v, cudaStream_t st) {
  if (n <= 0) return 0;
  fill_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(p, n, v);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------------ host side
bool gemm_tc2_supported(const GemmArgs& g, int amode) {
  const bool fuse = tc_fuse_attn_out_enabled();
  GemmArgs base = g;
  base.at_pos = nullptr; base.pool = nullptr; base.x_h2 = false; base.out_h2 = false; base.pos_h2 = false;
  if (!gemm_tc_supported(base, amode)) return false;
  if (g.act == ACT_GELU) return false;
  // 128-channel layers: the single-CTA flavour takes ready-made operands only (fp16 planes of the parity-grade mode, fast-mode formats)
  if (g.N % 256 != 0 && !(g.N % 128 == 0 && (gemm_tc2_fast(g) || gemm_tc2_fast_tf32(g) || (g.x_h2 && gemm_tc2_fp16x3(g))))) return false;
  if (!g.Whi || !g.Wlo) return false;                       // pre-split weights only
  // point-level layers that exchange fp16 planes keep their arithmetic (fp16x3 products) for every chunk size the tensor-core
  // engines take at all (>= 1024 rows), so that the result does not depend on how a forward is chunked
  if (g.R < (g.tc2_any_rows ? 1024 : 4096)) return false;
  if (g.pool) {
    if (g.at_pos || g.residual || g.edge_bias || g.act != ACT_LEAKY || g.pool_T < 1 || g.pool_T > 8 || g.pool_M < 1) return false;
    if (g.R % ((int64_t)g.pool_T * g.pool_M) != 0) return false;
  }
  if (g.at_pos) {
    if (!fuse || g.act != ACT_NONE || g.residual || !g.at_v || !g.idx || g.Mpts > 256 || tc_fused_tile_rows(g.kk) == 0) return false;
    if (g.R % g.kk != 0) return false;
  }
  return true;
}

// fp16x3 operands: only where the activations are LIF outputs, the weights carry their half split and the epilogue
// flavour is instantiated
bool gemm_tc2_fp16x3(const GemmArgs& g) {
  return g.x_unit && g.Wh && g.Wl && g.K % 64 == 0 && g.tc_passes != 1 && !g.residual &&
         (g.at_pos || g.act == ACT_LIF || (g.act == ACT_LEAKY && g.pool) || g.act == ACT_NONE);
}

// SAPCU_MODE_FAST operands: one fp16 product per MAC on a single fp16 plane (the producer wrote x * 2^13 as halfs)
bool gemm_tc2_fast(const GemmArgs& g) {
  return g.fast && g.x_h2 && g.x_unit && g.Wh && g.K % 64 == 0 && !g.residual &&
         (g.at_pos || g.act == ACT_LIF || (g.act == ACT_LEAKY && g.pool));
}
// SAPCU_MODE_FAST, point-level LIF layers (fp32 activations in and out): single-pass TF32 with compact stages, so that the
// layer's LIF table fits next to the pipeline (HM = 4)
bool gemm_tc2_fast_tf32(const GemmArgs& g) {
  // LIF layers (any width the engine takes) and plain 256-channel-multiple layers: the operands need no splitter, so they ride
  // the direct TMA -> issuer protocol of the compact-stage flavour
  return g.fast && !g.x_h2 && !g.out_h2 && (g.act == ACT_LIF || (g.act == ACT_NONE && g.N % 256 == 0)) && !g.edge_bias && !g.residual &&
         !g.at_pos && !g.pool && g.Whi && g.K % TC_BK == 0;
}

namespace {
constexpr size_t t2_smem_fast(bool lt, uint32_t tab_stride, int cg) {
  return (size_t)(lt ? (cg == 2 ? 3 : 2) : (cg == 2 ? T2_FAST_STAGES : 4)) * (cg == 2 ? 2 : 3) * TC_TILE_BYTES + 1024 + 256 + (lt ? tab_stride : 0);
}
}  // namespace

int launch_gemm_tc2(const GemmArgs& g, cudaStream_t st) {
  SAPCU_REQUIRE(gemm_tc2_supported(g, A_PLAIN), "gemm_tc2: unsupported problem");
  int* err = tc_err_flag();
  SAPCU_REQUIRE(err != nullptr, "gemm_tc2: cannot allocate the watchdog flag");
  const int tile_rows = g.at_pos ? tc_fused_tile_rows(g.kk) : T2_BN;
  const bool fast = gemm_tc2_fast(g), fast_tf32 = !fast && gemm_tc2_fast_tf32(g);
  const int cg = (g.N % 256 == 0) ? 2 : 1;                   // CTAs per tile: 1 = the single-CTA flavour for 128-channel layers (fast mode)
  SAPCU_REQUIRE(!fast || (g.x_h2 && g.lda == g.K && (!g.out_h2 || (g.act == ACT_LIF && g.ldc == g.N))), "gemm_tc2(fast): needs a single-plane fp16 input with lda == K");
  const bool h16 = fast || gemm_tc2_fp16x3(g);
  const bool pre = h16 && g.x_h2;                            // activations already stored as fp16 (hi, lo) planes
  SAPCU_REQUIRE(fast || !g.x_h2 || (h16 && g.lda == g.K && (g.at_pos || g.act == ACT_LIF || (g.act == ACT_LEAKY && g.pool))), "gemm_tc2: fp16-plane input needs the fp16x3 path and lda == K");
  SAPCU_REQUIRE(!g.out_h2 || (g.act == ACT_LIF && g.ldc == g.N), "gemm_tc2: fp16-plane output is a LIF epilogue with ldc == N");
  CUtensorMap mw, mwlo, mx, mx2;
  int rc = h16 ? tc_make_map_f16(&mw, g.Wh, g.N, g.K, 128) : tc_make_map(&mw, g.Whi, g.N, g.K, g.K, 128);
  if (rc) return rc;
  rc = h16 ? tc_make_map_f16(&mwlo, g.Wl, g.N, g.K, 128) : tc_make_map(&mwlo, g.Wlo, g.N, g.K, g.K, 128);
  if (rc) return rc;
  if (pre) {
    const uint16_t* hp = reinterpret_cast<const uint16_t*>(g.A);
    rc = tc_make_map_f16(&mx, hp, g.R, g.K, T2_BN / cg);
    if (rc) return rc;
    rc = fast ? 0 : tc_make_map_f16(&mx2, hp + g.R * g.K, g.R, g.K, T2_BN / cg);
    if (rc) return rc;
    if (fast) mx2 = mx;
  } else {
    rc = tc_make_map(&mx, g.A, g.R, g.K, g.lda, T2_BN / cg);
    if (rc) return rc;
    mx2 = mx;
  }
  TcParams p;
  p.R = g.R; p.N = g.N; p.K = g.K; p.bias = g.bias; p.scale = g.scale; p.shift = g.shift; p.act = g.act; p.T = g.T;
  p.nparams = g.nparams; p.residual = g.residual; p.ldr = g.ldr; p.Y = g.Y; p.ldc = g.ldc; p.Y2 = g.Y2;
  p.aq = g.Q; p.ak = g.Kf; p.ldq = g.ldq; p.idx = g.idx; p.ldi = g.ldi; p.kk = g.kk; p.Mpts = g.Mpts;
  p.pool = g.pool; p.pool_T = g.pool_T; p.pool_rows = (int64_t)g.pool_T * g.pool_M;
  p.idx8 = g.idx8; p.ldi8w = g.ldi8w;
  p.at_pos = g.at_pos; p.at_v = g.at_v; p.at_ldv = g.at_ldv; p.at_sqrt = g.at_sqrt; p.tile_rows = tile_rows;
  p.m_tiles = g.N / (128 * cg); p.n_tiles = ceil_div(g.R, tile_rows); p.err = err; p.split_w = 0; p.passes = g.tc_passes == 1 ? 1 : 3;
  p.out_h2 = g.out_h2 ? 1 : 0; p.pos_h2 = g.pos_h2 ? 1 : 0;
  p.lif_tab = nullptr; p.lif_tab_stride = 0;
  p.x_scale = h16 ? 8192.0f : 1.0f;                         // soft spikes lie in (0, 0.7): x * 2^13 < 2^13, residual * 2^13 >= fp16's normal range
  p.acc_scale = h16 ? g.winv / 8192.0f : 1.0f;
  const int64_t total = p.n_tiles * p.m_tiles;
  int pairs = (int)(total < kNumSMs / cg ? total : kNumSMs / cg);
  if (fast_tf32) {
    const bool lt = g.act == ACT_LIF && g.lif_tab != nullptr && g.lif_tab_stride > 0 && g.lif_tab_stride <= LT_SMEM_BUDGET;
    if (lt) pairs = (pairs / p.m_tiles) * p.m_tiles;
    SAPCU_REQUIRE(pairs >= 1, "gemm_tc2(fast tf32): empty grid");
    p.lif_tab = reinterpret_cast<const uint8_t*>(g.lif_tab); p.lif_tab_stride = g.lif_tab_stride;
    p.passes = 1; p.x_scale = 1.0f; p.acc_scale = 1.0f;
    const size_t smem = t2_smem_fast(lt, g.lif_tab_stride, cg);
    const int gridf = cg * pairs;
    if (g.act == ACT_NONE) return tc_launch<gemm_tc2_kernel<ACT_NONE, 0, 1, 4, 0, 2>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
    if (cg == 2) return lt ? tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 4, 1, 2>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p) : tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 4, 0, 2>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
    return lt ? tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 4, 1, 1>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p) : tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 4, 0, 1>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
  }
  if (fast) {
    // one fp16 product per MAC: map_w = the hi half of the fp16 weight split, map_x = the single activation plane
    const bool lt = g.act == ACT_LIF && g.lif_tab != nullptr && g.lif_tab_stride > 0 && g.lif_tab_stride <= LT_SMEM_BUDGET;
    if (lt) pairs = (pairs / p.m_tiles) * p.m_tiles;          // a pair keeps one channel block: its table is loaded once
    SAPCU_REQUIRE(pairs >= 1, "gemm_tc2(fast): empty grid");
    p.lif_tab = reinterpret_cast<const uint8_t*>(g.lif_tab); p.lif_tab_stride = g.lif_tab_stride;
    p.out_h2 = g.out_h2 ? 2 : 0; p.pos_h2 = g.pos_h2 ? 2 : 0;
    p.x_scale = 8192.0f; p.acc_scale = g.winv / 8192.0f;
    const size_t smem = t2_smem_fast(lt, g.lif_tab_stride, cg);
    const int gridf = cg * pairs;
    if (g.at_pos)
      return with_kk(g.kk, [&](auto KQ) {
        constexpr int kq = decltype(KQ)::value;
        return cg == 2 ? tc_launch<gemm_tc2_kernel<ACT_NONE, 3, kq, 3, 0>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p) : tc_launch<gemm_tc2_kernel<ACT_NONE, 3, kq, 3, 0, 1>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
      });
    if (g.act == ACT_LEAKY) {
      SAPCU_REQUIRE(cg == 2, "gemm_tc2(fast): the pooled conv5 epilogue needs N %% 256 == 0");
      return tc_launch<gemm_tc2_kernel<ACT_LEAKY, 4, 1, 3, 0>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
    }
    if (g.edge_bias) {
      if (cg == 2) return lt ? tc_launch<gemm_tc2_kernel<ACT_LIF, 2, 1, 3, 1>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p) : tc_launch<gemm_tc2_kernel<ACT_LIF, 2, 1, 3, 0>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
      return lt ? tc_launch<gemm_tc2_kernel<ACT_LIF, 2, 1, 3, 1, 1>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p) : tc_launch<gemm_tc2_kernel<ACT_LIF, 2, 1, 3, 0, 1>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
    }
    if (cg == 2) return lt ? tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 3, 1>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p) : tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 3, 0>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
    return lt ? tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 3, 1, 1>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p) : tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 3, 0, 1>>(gridf, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
  }
  if (pre && cg == 1) {
    // 128-channel layer on (hi, lo) planes: the single-CTA flavour (fp16x3 products; LIF table next to ONE 96 KiB stage)
    SAPCU_REQUIRE(g.at_pos || g.act == ACT_LIF, "gemm_tc2: the single-CTA plane path serves the LIF layers and the attention tail");
    const bool lt = g.act == ACT_LIF && g.lif_tab && g.lif_tab_stride > 0 && g.lif_tab_stride <= LT_SMEM_BUDGET;
    if (lt) { pairs = (pairs / p.m_tiles) * p.m_tiles; p.lif_tab = reinterpret_cast<const uint8_t*>(g.lif_tab); p.lif_tab_stride = g.lif_tab_stride; }
    SAPCU_REQUIRE(pairs >= 1, "gemm_tc2(single-CTA planes): empty grid");
    const size_t smem = (size_t)(lt ? 1 : 2) * 6 * TC_TILE_BYTES + 1024 + 256 + (lt ? g.lif_tab_stride : 0);
    if (g.at_pos)
      return with_kk(g.kk, [&](auto KQ) { return tc_launch<gemm_tc2_kernel<ACT_NONE, 3, decltype(KQ)::value, 2, 0, 1>>(pairs, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p); });
    if (g.edge_bias) return lt ? tc_launch<gemm_tc2_kernel<ACT_LIF, 2, 1, 2, 1, 1>>(pairs, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p) : tc_launch<gemm_tc2_kernel<ACT_LIF, 2, 1, 2, 0, 1>>(pairs, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
    return lt ? tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 2, 1, 1>>(pairs, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p) : tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 2, 0, 1>>(pairs, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
  }
  if (pre && g.act == ACT_LIF && g.lif_tab && g.lif_tab_stride > 0 && g.lif_tab_stride <= LT_SMEM_BUDGET_TC) {
    // fp16x3 products on (hi, lo) planes + the layer's tabulated LIF^T chain: 2 stages of 64 KiB leave room for the table
    pairs = (pairs / p.m_tiles) * p.m_tiles;
    SAPCU_REQUIRE(pairs >= 1, "gemm_tc2(tables): empty grid");
    p.lif_tab = reinterpret_cast<const uint8_t*>(g.lif_tab); p.lif_tab_stride = g.lif_tab_stride;
    const size_t smem = 2 * 4 * (size_t)TC_TILE_BYTES + 1024 + 256 + g.lif_tab_stride;
    if (g.edge_bias) return tc_launch<gemm_tc2_kernel<ACT_LIF, 2, 1, 2, 1>>(2 * pairs, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
    return tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 2, 1>>(2 * pairs, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
  }
  const int grid = 2 * pairs;
  if (pre) {
    if (g.at_pos) return with_kk(g.kk, [&](auto KQ) { return tc_launch<gemm_tc2_kernel<ACT_NONE, 3, decltype(KQ)::value, 2>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p); });
    if (g.act == ACT_LEAKY) return tc_launch<gemm_tc2_kernel<ACT_LEAKY, 4, 1, 2>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
    if (g.edge_bias) return tc_launch<gemm_tc2_kernel<ACT_LIF, 2, 1, 2>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
    return tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 2>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
  }
  if (h16) {
    if (g.at_pos) return with_kk(g.kk, [&](auto KQ) { return tc_launch<gemm_tc2_kernel<ACT_NONE, 3, decltype(KQ)::value, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p); });
    if (g.act == ACT_LIF && g.edge_bias) return tc_launch<gemm_tc2_kernel<ACT_LIF, 2, 1, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
    if (g.act == ACT_LIF) return tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
    if (g.act == ACT_LEAKY) return tc_launch<gemm_tc2_kernel<ACT_LEAKY, 4, 1, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
    return tc_launch<gemm_tc2_kernel<ACT_NONE, 0, 1, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
  }
  if (g.act == ACT_LIF && !g.edge_bias && g.lif_tab && g.lif_tab_stride > 0 && g.lif_tab_stride <= LT_SMEM_BUDGET_TC) {
    // 3xTF32 products (splitter path) + the layer's tabulated LIF^T chain: two 64 KiB stages next to the table
    pairs = (pairs / p.m_tiles) * p.m_tiles;
    SAPCU_REQUIRE(pairs >= 1, "gemm_tc2(3xTF32 + table): empty grid");
    p.lif_tab = reinterpret_cast<const uint8_t*>(g.lif_tab); p.lif_tab_stride = g.lif_tab_stride;
    const size_t smem = 2 * 4 * (size_t)TC_TILE_BYTES + 1024 + 256 + g.lif_tab_stride;
    return tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1, 0, 1>>(2 * pairs, T2_THREADS, smem, st, mw, mwlo, mx, mx2, p);
  }
  if (g.at_pos) return with_kk(g.kk, [&](auto KQ) { return tc_launch<gemm_tc2_kernel<ACT_NONE, 3, decltype(KQ)::value>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p); });
  if (g.act == ACT_LIF && g.edge_bias) return tc_launch<gemm_tc2_kernel<ACT_LIF, 2, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
  if (g.act == ACT_LIF) return tc_launch<gemm_tc2_kernel<ACT_LIF, 0, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
  if (g.act == ACT_LEAKY && g.pool) return tc_launch<gemm_tc2_kernel<ACT_LEAKY, 4, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
  if (g.act == ACT_LEAKY) return tc_launch<gemm_tc2_kernel<ACT_LEAKY, 0, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
  if (g.residual) return tc_launch<gemm_tc2_kernel<ACT_NONE, 1, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
  return tc_launch<gemm_tc2_kernel<ACT_NONE, 0, 1>>(grid, T2_THREADS, T2_SMEM_BYTES, st, mw, mwlo, mx, mx2, p);
}

}  // namespace sapcu
