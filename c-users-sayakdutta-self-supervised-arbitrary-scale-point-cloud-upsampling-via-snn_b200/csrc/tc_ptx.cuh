// PTX wrappers shared by the tcgen05 GEMM engines (sm_100a): mbarrier, TMA, UMMA descriptors, tcgen05 mma/ld/commit.
#pragma once
#include <cstdlib>
#include <type_traits>
#include <cuda_fp16.h>
#include "neuron.cuh"
#include <cuda.h>
#include <stdint.h>
#include "common.cuh"

namespace sapcu {

constexpr int TC_BM = 128;        // output channels per CTA tile (UMMA M per CTA)
constexpr int TC_BK = 32;         // fp32 elements per k-block = one 128-byte swizzle row
constexpr uint32_t TC_TILE_BYTES = TC_BM * TC_BK * 4;          // 16 KiB: a 128-row operand tile
constexpr long long TC_WATCHDOG_CLOCKS = 6000000000LL;         // ~3 s at 1.9 GHz
constexpr int TC_L2_PREFETCH = 4;                              // k-blocks of look-ahead for the activation tile's L2 prefetch

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
// returns false after the watchdog fired (here or in another role)
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, int* err) {
  if (mbar_try_wait(bar, parity)) return true;
  const long long t0 = clock64();
  int spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 1023) == 0) {
      if (*reinterpret_cast<volatile int*>(err) != 0) return false;
      if (clock64() - t0 > TC_WATCHDOG_CLOCKS) { *reinterpret_cast<volatile int*>(err) = 1; __threadfence_system(); return false; }
    }
  }
  return true;
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* map, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, 128-byte swizzled operand tile (rows of 32 fp32 = 128 B, 8-row groups 1024 B apart)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);     // start address        bits [0,14)
  d |= (uint64_t)1 << 16;                        // leading byte offset  bits [16,30) (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset   bits [32,46)
  d |= (uint64_t)1 << 46;                        // descriptor version 1 (sm_100)
  d |= (uint64_t)2 << 61;                        // layout type: SWIZZLE_128B
  return d;
}
// instruction descriptor: D = F32, A = B = TF32, both K-major, M = 128, N = BN
__host__ __device__ constexpr uint32_t tc_idesc(int bn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
}

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// tcgen05.ld.32x32b.xN for N in {1,2,4,8,16}: N consecutive columns of this thread's lane into dst[0..N)
template <int NCOL> __device__ __forceinline__ void tmem_ld_piece(uint32_t taddr, float* dst);
template <> __device__ __forceinline__ void tmem_ld_piece<1>(uint32_t taddr, float* dst) {
  uint32_t r0;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r0) : "r"(taddr) : "memory");
  dst[0] = __uint_as_float(r0);
}
template <> __device__ __forceinline__ void tmem_ld_piece<2>(uint32_t taddr, float* dst) {
  uint32_t r0, r1;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(taddr) : "memory");
  dst[0] = __uint_as_float(r0); dst[1] = __uint_as_float(r1);
}
template <> __device__ __forceinline__ void tmem_ld_piece<4>(uint32_t taddr, float* dst) {
  uint32_t r[4];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
#pragma unroll
  for (int i = 0; i < 4; ++i) dst[i] = __uint_as_float(r[i]);
}
template <> __device__ __forceinline__ void tmem_ld_piece<8>(uint32_t taddr, float* dst) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr) : "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) dst[i] = __uint_as_float(r[i]);
}
template <> __device__ __forceinline__ void tmem_ld_piece<16>(uint32_t taddr, float* dst) {
  uint32_t r[16];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                 "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(taddr) : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) dst[i] = __uint_as_float(r[i]);
}
// tcgen05.wait::ld that also "produces" the 8 registers of a pending tmem_ld_piece<8>, so no use of them can be
// scheduled ahead of the wait (lets the load of the next piece fly under the arithmetic on the current one)
// float atomic max through the integer ALU of the L2 (exact, order-independent); *addr starts at -inf
__device__ __forceinline__ void atomic_max_float(float* addr, float x) {
  if (x >= 0.0f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(x));
  else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(x));
}
__device__ __forceinline__ void tmem_wait_ld8(float (&x)[8]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+f"(x[0]), "+f"(x[1]), "+f"(x[2]), "+f"(x[3]), "+f"(x[4]), "+f"(x[5]), "+f"(x[6]), "+f"(x[7])::"memory");
}
// KK columns (KK <= 31) as a sum of power-of-two pieces, then one tcgen05.wait::ld
template <int KK> __device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, float (&v)[KK]) {
  int o = 0;
  if (KK & 16) { tmem_ld_piece<16>(taddr + o, v + o); o += 16; }
  if (KK & 8) { tmem_ld_piece<8>(taddr + o, v + o); o += 8; }
  if (KK & 4) { tmem_ld_piece<4>(taddr + o, v + o); o += 4; }
  if (KK & 2) { tmem_ld_piece<2>(taddr + o, v + o); o += 2; }
  if (KK & 1) { tmem_ld_piece<1>(taddr + o, v + o); o += 1; }
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}


struct TcParams {
  int64_t R; int N, K;
  const float* bias; const float* scale; const float* shift;
  int act, T; const float* nparams;
  const float* residual; int64_t ldr;
  float* Y; int64_t ldc;
  float* Y2;                  // LIF epilogue with out_h2: optional fp32 copy of the spikes for a second reader that gathers them ([R, N])
  // EXTRA == 2 (fn fc_gamma on the factorised attention input): row e = pt*kk + j of the activation is pos_ij only, and
  // the epilogue adds aq[pt,c] - ak[nb,c] (= W q_i - W k_j, per-POINT products) to the accumulator before the affine
  const float* aq; const float* ak; int64_t ldq; const int32_t* idx; int ldi, kk, Mpts;
  // EXTRA == 3 (fn fc_gamma2, 2-CTA kernel): the epilogue applies softmax over the kk edges of a point to the logits
  // (/ at_sqrt) and writes Y[pt,c] = sum_j a_j (at_v[nb_j,c] + at_pos[e_j,c]) instead of the logits
  const float* at_pos; const float* at_v; int64_t at_ldv; float at_sqrt;
  const uint32_t* idx8; int ldi8w;   // optional byte-packed copy of the graph (4 patch-local indices per word, ldi8w words per point)
  // EXTRA == 4 (fd conv5, 2-CTA kernel): rows are (point*T + t); the epilogue keeps one running maximum per step and
  // merges them into pool[(patch*T + t), c] with float atomic max -- the [P*T, N] activation never reaches HBM
  float* pool; int pool_T; int64_t pool_rows;     // pool_rows = points per patch * T
  int pos_h2;                 // EXTRA == 3: at_pos is stored as fp16 (hi, lo) planes of pos * 2^13 ([R, N] halfs each); 2 = hi plane only (fast mode)
  int out_h2;                 // LIF epilogue of the 2-CTA kernel: write Y as fp16 (hi, lo) planes of y * 2^13 (ldc == N, [R, N] each); 2 = hi plane only (fast mode)
  // SAPCU_MODE_FAST, LIF epilogue: tabulated chain (lif_table.cuh): image of the 128-channel block b at lif_tab + b * lif_tab_stride
  const uint8_t* lif_tab; uint32_t lif_tab_stride;
  float acc_scale, x_scale;   // fp16x3 path: operands are W * 2^e and x * x_scale, acc_scale = 2^-e / x_scale undoes both (exact)
  int tile_rows;              // rows a tile advances by: the MMA tile height, or the whole points inside it when EXTRA == 3
  int m_tiles; int64_t n_tiles;
  int split_w;                // 1: W arrives raw and is split in shared memory; 0: map_w / map_wlo hold pre-split (hi, lo)
  int passes;                 // 3: w_lo*x_hi + w_hi*x_lo + w_hi*x_hi (fp32-grade); 1: w_hi*x_hi only (plain TF32)
  int* err;
};

// Edge bias operands (EXTRA == 2).  The row -> (point, neighbour) resolution is the same for every lane of a warp, so it
// is done once per 32 rows with lane L resolving row e0 + L (rows past the end re-use the last row; offsets fit 32 bits,
// checked on the host): qo = pt * ldq, ko = nb * ldq.
__device__ __forceinline__ void edge_lane_offsets(const TcParams& p, int64_t e0, int lane, int& qo, int& ko) {
  int64_t e64 = e0 + lane;
  if (e64 > p.R - 1) e64 = p.R - 1;
  const uint32_t e = (uint32_t)e64;
  const uint32_t pt = e / (uint32_t)p.kk, j = e - pt * (uint32_t)p.kk;
  const uint32_t patch0 = (pt / (uint32_t)p.Mpts) * (uint32_t)p.Mpts;
  const int nb = (int)patch0 + p.idx[(int64_t)pt * p.ldi + j];
  qo = (int)pt * (int)p.ldq; ko = nb * (int)p.ldq;
}
// qv[r] = aq[pt_r, c], kv[r] = ak[nb_r, c] for rows 8*sub .. 8*sub+7 of the warp's current 32-row group: 16 independent
// loads, consumed by the caller only after its arithmetic on the previous piece (which hides their latency)
__device__ __forceinline__ void edge_fetch8(const TcParams& p, int my_qo, int my_ko, int sub, int c, float (&qv)[8], float (&kv)[8]) {
  // unsigned 32-bit element offsets from the two uniform bases: one 64-bit multiply-add (IMAD.WIDE, fma pipe) per address
  // instead of a LEA / LEA.HI.X pair on the ALU pipe, which the LIF-table epilogue saturates
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int qo = __shfl_sync(0xffffffffu, my_qo, sub * 8 + r), ko = __shfl_sync(0xffffffffu, my_ko, sub * 8 + r);
    qv[r] = p.aq[(uint32_t)(qo + c)]; kv[r] = p.ak[(uint32_t)(ko + c)];
  }
}


// Fused attention tail (EXTRA == 3) for the points pp = part, part + parts, ... of one tile: logits (TMEM columns
// pp*KK .. pp*KK+KK-1 of this thread's channel c) -> /sqrt(d_h) -> softmax over the KK edges -> sum_j a_j (v[nb_j] + pos[e_j]).
// Latency plan per point: the neighbour indices were fetched one point ahead; the 2*KK operand loads are issued first,
// the TMEM read and the softmax run under them, the weighted sum consumes them last.
// NC > 0: the channel count (row stride of pos and of the output) as a compile-time constant -- the KK pos loads of a point
// become immediate offsets from one base address; NC == 0: run-time p.N.
template <int KK, int NC = 0>
__device__ __forceinline__ void attn_tail_points(const TcParams& p, uint32_t tmem_cols, int part, int parts, int npts,
                                                 int64_t n_t, int c, float bia, float sc, float sh, float acc_scale) {
  const int64_t Nn = NC ? (int64_t)NC : (int64_t)p.N;
  const int64_t P_total = p.R / KK;
  const float inv_s = 1.0f / p.at_sqrt;
  const float* vc = p.at_v + c;
  uint32_t nbn[(KK + 3) / 4];                                    // graph row of the next point, 4 patch-local indices (< 256) per word
  auto fetch_row = [&](int64_t ptq) {
    if (p.idx8) {                                                // byte-packed graph: (KK + 3) / 4 word loads, nothing to shift
      const uint32_t* ip = p.idx8 + (ptq < P_total ? ptq : P_total - 1) * p.ldi8w;
#pragma unroll
      for (int w = 0; w < (KK + 3) / 4; ++w) nbn[w] = ip[w];
      return;
    }
    const int32_t* ip = p.idx + (ptq < P_total ? ptq : P_total - 1) * p.ldi;
#pragma unroll
    for (int w = 0; w < (KK + 3) / 4; ++w) nbn[w] = 0u;
#pragma unroll
    for (int j = 0; j < KK; ++j) nbn[j >> 2] |= (uint32_t)ip[j] << (8 * (j & 3));
  };
  fetch_row(n_t * npts + part);
  // first point of the patch that holds this warp's current point: one division per tile, then advanced with the point
  int64_t patch0 = ((n_t * npts + part) / p.Mpts) * p.Mpts;
  int prem = (int)(n_t * npts + part - patch0);
  for (int pp = part; pp < npts; pp += parts, prem += parts) {
    const int64_t pt = n_t * npts + pp;
    if (pt >= P_total) break;                                    // warp-uniform
    while (prem >= p.Mpts) { prem -= p.Mpts; patch0 += p.Mpts; }
    const float* ps = p.at_pos + (pt * KK) * Nn + c;
    float vr[KK], pr[KK];
    __half prh[KK];                                              // fast mode: the raw halves, converted only where they are consumed
    // v[nb_j]: one 64-bit base per point, then byte extract (PRMT) + one 32 x 32 -> 64-bit multiply-add (IMAD.WIDE) per neighbour
    uint64_t vb = (uint64_t)__cvta_generic_to_global(vc) + (uint64_t)(patch0 * p.at_ldv * 4);
    asm volatile("" : "+l"(vb));                                 // ONE 64-bit base value: the per-neighbour address is a single IMAD.WIDE
    uint32_t ldvb = (uint32_t)p.at_ldv * 4u;
    asm volatile("" : "+r"(ldvb));
#pragma unroll
    for (int j = 0; j < KK; ++j) {
      const uint32_t nb = __byte_perm(nbn[j >> 2], 0u, 0x4440u + (uint32_t)(j & 3));
      const uint64_t a = vb + (uint64_t)nb * ldvb;
      asm("ld.global.f32 %0, [%1];" : "=f"(vr[j]) : "l"(a));     // v was written by an earlier kernel of the stream
    }
    if (p.pos_h2 == 2) {                                         // fast mode: one fp16 plane of pos * 2^13
      const __half* ph = reinterpret_cast<const __half*>(p.at_pos) + (pt * KK) * Nn + c;
#pragma unroll
      for (int j = 0; j < KK; ++j) prh[j] = ph[(int64_t)j * Nn];
    } else if (p.pos_h2) {
      const __half* ph = reinterpret_cast<const __half*>(p.at_pos) + (pt * KK) * Nn + c;
      const __half* pl = ph + p.R * Nn;
#pragma unroll
      for (int j = 0; j < KK; ++j) pr[j] = (__half2float(ph[(int64_t)j * Nn]) + __half2float(pl[(int64_t)j * Nn])) * (1.0f / 8192.0f);
    } else {
#pragma unroll
      for (int j = 0; j < KK; ++j) pr[j] = ps[(int64_t)j * Nn];
    }
    fetch_row(pt + parts);                                       // indices of this warp's next point (clamped at the end)
    float av[KK];
    __syncwarp();
    tmem_ld_cols<KK>(tmem_cols + (uint32_t)(pp * KK), av);
    // softmax over the point's KK logits l_j = t_j / sqrt(d_h), t = BN(acc + bias): exp(l_j - max l) = 2^(t_j * k - max(t) * k) with
    // k = log2(e) / sqrt(d_h) > 0 -- one multiply-add per edge; the normalisation is applied once to the weighted sum
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < KK; ++j) { av[j] = fmaf(fmaf(av[j], acc_scale, bia), sc, sh); mx = fmaxf(mx, av[j]); }
    const float kexp = inv_s * 1.4426950408889634f, mxk = -mx * kexp;
    float sum = 0.0f;
#pragma unroll
    for (int j = 0; j < KK; ++j) { av[j] = exp2f_approx(fmaf(av[j], kexp, mxk)); sum += av[j]; }
    float res = 0.0f;
#pragma unroll
    for (int j = 0; j < KK; ++j) res = fmaf(av[j], p.pos_h2 == 2 ? fmaf(__half2float(prh[j]), 1.0f / 8192.0f, vr[j]) : vr[j] + pr[j], res);   // 2^-13 * half is exact: same sum
    p.Y[pt * (NC ? (int64_t)NC : p.ldc) + c] = res * (1.0f / sum);
  }
}

// the yaml model pairs each neighbour count with one width (24 / 128, 18 / 256, 12 / 512): those get the compile-time stride
template <int KK>
__device__ __forceinline__ void attn_tail_dispatch(const TcParams& p, uint32_t tmem_cols, int part, int parts, int npts,
                                                   int64_t n_t, int c, float bia, float sc, float sh, float acc_scale) {
  constexpr int NY = KK == 24 ? 128 : KK == 18 ? 256 : KK == 12 ? 512 : 0;
  if (NY != 0 && p.N == NY && p.ldc == NY) attn_tail_points<KK, NY>(p, tmem_cols, part, parts, npts, n_t, c, bia, sc, sh, acc_scale);
  else attn_tail_points<KK, 0>(p, tmem_cols, part, parts, npts, n_t, c, bia, sc, sh, acc_scale);
}

// host helpers (gemm_tc.cu)
int tc_make_map(CUtensorMap* m, const float* base, int64_t rows, int K, int64_t ld, int box_rows);
int* tc_err_flag();
// Kern<<<grid, threads, smem, st>>>(args...).  The first launch of each kernel on a device raises its dynamic shared-memory
// limit to what the device allows next to the kernel's static shared memory, so the byte count computed at the launch site
// is the only one written down.
template <auto Kern, typename... A>
int tc_launch(int grid, int threads, size_t smem, cudaStream_t st, const A&... args) {
  static PerDeviceOnce once;
  const int rc = once.run([]() -> int {
    int dev = 0, optin = 0;
    cudaFuncAttributes fa;
    SAPCU_CUDA_CHECK(cudaGetDevice(&dev));
    SAPCU_CUDA_CHECK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    SAPCU_CUDA_CHECK(cudaFuncGetAttributes(&fa, Kern));
    SAPCU_CUDA_CHECK(cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes));
    return 0;
  });
  if (rc) return rc;
  Kern<<<grid, threads, smem, st>>>(args...);
  SAPCU_LAUNCH_CHECK();
  return 0;
}
// 2-D fp16 row-major [rows, K] -> boxes of [box_rows, 64 halfs] with 128B swizzle
int tc_make_map_f16(CUtensorMap* m, const void* base, int64_t rows, int K, int box_rows);
// rows a tile advances by in the fused attention epilogue (EXTRA == 3): the whole points that fit in the 256-row MMA tile
// (the few rows behind them are loaded and multiplied but belong to the next tile); 0 = neighbour count not instantiated
inline int tc_fused_tile_rows(int kk) {
  if (kk == 12 || kk == 18 || kk == 24) return (256 / kk) * kk;
  return 0;
}
// f(std::integral_constant<int, kk>{}) for the neighbour counts of tc_fused_tile_rows: the fused attention tail's instantiations
template <class F> int with_kk(int kk, F&& f) {
  if (kk == 12) return f(std::integral_constant<int, 12>{});
  if (kk == 18) return f(std::integral_constant<int, 18>{});
  return f(std::integral_constant<int, 24>{});
}
inline bool tc_fuse_attn_out_enabled() { return settings().fuse_attnout; }

}  // namespace sapcu
