// K1: exact brute-force seed -> input-cloud kNN (replaces sklearn KDTree.query, generation.py:127,153,178).
//
// Large clouds (N >= 2^20): one THREAD owns one seed.  The fp32 copy of the cloud is stored SoA (x[], y[], z[]) and streams
// through shared memory in double-buffered tiles moved by the TMA engine (cp.async.bulk + mbarrier: the copy of tile t+1
// runs under the arithmetic on tile t); every lane of a warp reads the SAME four points (three broadcast LDS.128) and
// tests them against its own seed with a CONSERVATIVE fp32 filter written with Blackwell's packed fp32 instructions
// (FADD2 / FMUL2 / FFMA2: two cloud points per instruction, seed coordinate as the broadcast scalar operand) and a
// 3-input minimum: 3 packed arithmetic + ~1 compare + 0.75 LDS issue slots per pair instead of 8.  Only survivors pay for the exact fp64 squared
// distance ((dx*dx + dy*dy) + dz*dz, no contraction -- the KDTree's reduced distance) and an O(log K) update of the
// thread's private max-heap of (fp64 distance, index) keys; the heap is heap-sorted at the end, so the result is the
// exact fp64 ordering with ties broken by the lowest cloud index, independent of tiling.
//
// Filter soundness: with p~,q~ the fp32 roundings of p,q and Rmax >= every |coordinate|,
// |sqrt(d32) - sqrt(d)| <= 2^-22 Rmax + 2^-21 sqrt(d); a point with d <= tau therefore always has
// d32 <= ((1+2^-20) sqrt(tau) + 2^-21 Rmax)^2 (1+2^-20) =: tau32, recomputed whenever tau changes.
//
// Roofline: FP32 issue, quoted against the scalar formulation's 8 lane-ops per pair (148 SM x 128 lanes x clk / 8 =
// 4.65e12 pairs/s) so that rounds compare; the cloud comes from L2 once per CTA (256 seeds); HBM traffic is only
// S*(24 + 4K) bytes.
#include "common.cuh"
#include "kernels.h"
#include "tc_ptx.cuh"
#include <float.h>
#include <algorithm>
#include <vector>

namespace sapcu {

constexpr int KNN_KMAX = 128;
constexpr int KNN_THREADS = 256;     // seeds per CTA
constexpr int KNN_TILE = 2048;       // cloud points per shared-memory tile (32 KiB)

// fp32 SoA copy (x[npad], y[npad], z[npad]) of a [n,3] fp64 array and the running max |coordinate|; rows n .. npad-1 are
// padding far outside any cloud.  The thread-per-seed kernel copies whole 16-byte groups of rows, so a tile may also hold
// rows outside the seed's cloud: the padding, and in batched launches up to 3 rows of the previous cloud before it and
// rows of the next cloud after it.  They can pass the filter; `consider` drops them by index.
constexpr float KNN_PAD = 3.0e18f;
__host__ __device__ inline int64_t knn_npad(int64_t n) { return (n + 3) / 4 * 4 + 4; }
__global__ void cloud_to_f32_kernel(const double* __restrict__ cloud, int64_t n, float* __restrict__ out, float* __restrict__ rmax) {
  float m = 0.0f;
  const int64_t npad = knn_npad(n);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < (out ? npad : n); i += (int64_t)gridDim.x * blockDim.x) {
    if (i >= n) { out[i] = KNN_PAD; out[npad + i] = KNN_PAD; out[2 * npad + i] = KNN_PAD; continue; }
    const double x = cloud[3 * i], y = cloud[3 * i + 1], z = cloud[3 * i + 2];
    if (out) { out[i] = (float)x; out[npad + i] = (float)y; out[2 * npad + i] = (float)z; }
    m = fmaxf(m, (float)fmax(fmax(fabs(x), fabs(y)), fabs(z)) * 1.0000002f);
  }
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(rmax), __float_as_int(m));   // m >= 0
}

// packed fp32 (two cloud points per instruction; sm_100: FADD2 / FMUL2 / FFMA2)
__device__ __forceinline__ float2 f2_sub(float2 a, float b) {
  float2 r;
  asm("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%4}; sub.f32x2 rc, ra, rb; mov.b64 {%0,%1}, rc;}"
      : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b));
  return r;
}
__device__ __forceinline__ float2 f2_mul(float2 a, float2 b) {
  float2 r;
  asm("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mul.f32x2 rc, ra, rb; mov.b64 {%0,%1}, rc;}"
      : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return r;
}
__device__ __forceinline__ float2 f2_fma(float2 a, float2 b, float2 c) {
  float2 r;
  asm("{.reg .b64 ra, rb, rc, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mov.b64 rc, {%6,%7}; fma.rn.f32x2 rd, ra, rb, rc; mov.b64 {%0,%1}, rd;}"
      : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return r;
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// Batched launches (sapcu_knn_batched): the grid is the concatenation of per-cloud block ranges.  blk_off / cloud_off /
// seed_off are [B+1] prefix tables (device); a CTA finds its cloud by binary search and works on that cloud's rows and
// its own seeds only.  B == 0: the single-cloud launch (whole arrays).  Emitted indices are rows of the CONCATENATED
// cloud array, so the gather that follows needs no per-cloud bookkeeping.  A cloud may start at any row c0: the bulk
// copies of the thread-per-seed kernel need 16-byte-aligned sources, so its tiles start at the aligned row c0 & ~3 and
// the first c0 & 3 rows they hold belong to the previous cloud.
struct KnnSegs { const int64_t* blk_off; const int64_t* cloud_off; const int64_t* seed_off; int B; };
__device__ __forceinline__ void knn_resolve(const KnnSegs& g, int per_block, int64_t& c0, int64_t& N, int64_t& s0, int64_t& s_end) {
  if (g.B == 0) { c0 = 0; s0 = (int64_t)blockIdx.x * per_block; return; }      // N, s_end stay as passed
  int lo = 0, hi = g.B;                                      // last b with blk_off[b] <= blockIdx.x
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (g.blk_off[mid] <= (int64_t)blockIdx.x) lo = mid; else hi = mid; }
  c0 = g.cloud_off[lo]; N = g.cloud_off[lo + 1] - c0;
  s0 = g.seed_off[lo] + ((int64_t)blockIdx.x - g.blk_off[lo]) * per_block; s_end = g.seed_off[lo + 1];
}

__device__ __forceinline__ bool key_less(double da, int ia, double db, int ib) {
  return da < db || (da == db && ia < ib);
}

constexpr size_t KNN_SMEM = 2 * 3 * (size_t)KNN_TILE * sizeof(float) + 16;      // two SoA tiles + two mbarriers
__global__ void __launch_bounds__(KNN_THREADS)
knn_seed_kernel(const double* __restrict__ cloud, const float* __restrict__ cloud32, int64_t N,
                const double* __restrict__ seeds, int64_t S, int K, const float* __restrict__ rmax_p,
                int32_t* __restrict__ out_idx, const KnnSegs segs, int64_t npad_all) {
  extern __shared__ __align__(16) uint8_t knn_sm[];
  float* tile = reinterpret_cast<float*>(knn_sm);                       // [2][3][KNN_TILE]
  const uint32_t bar0 = smem_u32(knn_sm + 2 * 3 * KNN_TILE * sizeof(float));
  int64_t c0, sb;
  knn_resolve(segs, KNN_THREADS, c0, N, sb, S);
  // the bulk copies need 16-byte-aligned sources: tiles start at the aligned row c0 & ~3 and rows are numbered from there,
  // so this cloud's rows are lead .. lead + N - 1 (lead == 0 in the single-cloud launch); the shift is the same for every
  // row, so the heap's (distance, index) order is the cloud-local one
  const int lead = (int)(c0 & 3);
  c0 -= lead;
  const int64_t NT = N + lead;
  cloud += 3 * c0;
  const float* cx = cloud32 + c0; const float* cy = cx + npad_all; const float* cz = cy + npad_all;
  const int64_t s = sb + threadIdx.x;
  const bool active = s < S;
  const float rmax = *rmax_p;
  double sx = 0, sy = 0, sz = 0;
  if (active) { sx = seeds[3 * s]; sy = seeds[3 * s + 1]; sz = seeds[3 * s + 2]; }
  const float fx = (float)sx, fy = (float)sy, fz = (float)sz;

  // private max-heap (root = current K-th best = tau); lives in local memory, touched only by filter survivors
  double hd[KNN_KMAX]; int hi[KNN_KMAX];
  for (int j = 0; j < K; ++j) { hd[j] = DBL_MAX; hi[j] = INT_MAX; }
  double tau = DBL_MAX; int tau_i = INT_MAX;
  float tau32 = FLT_MAX;

  auto consider = [&](int gi) {
    if ((uint32_t)(gi - lead) >= (uint32_t)N) return;                   // padding row or another cloud's row
    const double ex = cloud[3 * (int64_t)gi] - sx, ey = cloud[3 * (int64_t)gi + 1] - sy, ez = cloud[3 * (int64_t)gi + 2] - sz;
    const double d = __dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez));
    if (!key_less(d, gi, tau, tau_i)) return;
    // replace the root and sift down
    int pos = 0;
    while (true) {
      const int l = 2 * pos + 1, r = l + 1;
      if (l >= K) break;
      int c = l;
      if (r < K && key_less(hd[l], hi[l], hd[r], hi[r])) c = r;      // larger child
      if (!key_less(d, gi, hd[c], hi[c])) break;
      hd[pos] = hd[c]; hi[pos] = hi[c];
      pos = c;
    }
    hd[pos] = d; hi[pos] = gi;
    tau = hd[0]; tau_i = hi[0];
    if (tau < DBL_MAX) {
      const float rt = sqrtf((float)tau) * 1.000002f;   // >= (1+2^-20) sqrt(tau) incl. rounding of the cast/sqrt
      const float b = rt + 4.76837158e-7f * rmax;       // 2^-21 Rmax
      tau32 = b * b * 1.000002f;
    }
  };

  // double-buffered SoA tiles: thread 0 asks the TMA engine for tile t+1 while the CTA works on tile t
  if (threadIdx.x == 0) { mbar_init(bar0, 1); mbar_init(bar0 + 8, 1); fence_barrier_init(); }
  __syncthreads();
  const int64_t ntiles = (NT + KNN_TILE - 1) / KNN_TILE;
  auto issue = [&](int64_t t) {
    const int64_t base = t * KNN_TILE;
    const int64_t rows = (NT - base) < KNN_TILE ? ((NT - base + 3) / 4 * 4) : KNN_TILE;   // the padding rows make every copy 16-byte granular
    const uint32_t bytes = (uint32_t)rows * 4u, bar = bar0 + 8u * (uint32_t)(t & 1);
    const uint32_t dst = smem_u32(tile + (t & 1) * 3 * KNN_TILE);
    mbar_expect_tx(bar, 3 * bytes);
    bulk_g2s(dst, cx + base, bytes, bar);
    bulk_g2s(dst + KNN_TILE * 4, cy + base, bytes, bar);
    bulk_g2s(dst + 2 * KNN_TILE * 4, cz + base, bytes, bar);
  };
  if (threadIdx.x == 0 && ntiles > 0) issue(0);
  for (int64_t t = 0; t < ntiles; ++t) {
    if (threadIdx.x == 0 && t + 1 < ntiles) issue(t + 1);               // its buffer was released by the barrier that ended tile t-1
    while (!mbar_try_wait(bar0 + 8u * (uint32_t)(t & 1), (uint32_t)((t >> 1) & 1))) { }
    const int64_t base = t * KNN_TILE;
    const int tn = (NT - base) < KNN_TILE ? (int)((NT - base + 3) / 4 * 4) : KNN_TILE;
    if (active) {
      const float4* xs = reinterpret_cast<const float4*>(tile + (t & 1) * 3 * KNN_TILE);
      const float4* ys = xs + KNN_TILE / 4;
      const float4* zs = ys + KNN_TILE / 4;
#pragma unroll 2
      for (int j = 0; j < tn / 4; ++j) {
        const float4 X = xs[j], Y = ys[j], Z = zs[j];
        const float2 dx0 = f2_sub(make_float2(X.x, X.y), fx), dx1 = f2_sub(make_float2(X.z, X.w), fx);
        const float2 dy0 = f2_sub(make_float2(Y.x, Y.y), fy), dy1 = f2_sub(make_float2(Y.z, Y.w), fy);
        const float2 dz0 = f2_sub(make_float2(Z.x, Z.y), fz), dz1 = f2_sub(make_float2(Z.z, Z.w), fz);
        const float2 d0 = f2_fma(dz0, dz0, f2_fma(dy0, dy0, f2_mul(dx0, dx0)));       // fmaf(dz, dz, fmaf(dy, dy, dx * dx)) per point
        const float2 d1 = f2_fma(dz1, dz1, f2_fma(dy1, dy1, f2_mul(dx1, dx1)));
        if (fminf(fminf(d0.x, d0.y), fminf(d1.x, d1.y)) <= tau32) {
          const int g0 = (int)(base + 4 * j);
          if (d0.x <= tau32) consider(g0);                                           // tau32 only shrinks: re-testing is still sound
          if (d0.y <= tau32) consider(g0 + 1);
          if (d1.x <= tau32) consider(g0 + 2);
          if (d1.y <= tau32) consider(g0 + 3);
        }
      }
    }
    __syncthreads();                                                     // everyone is done with this buffer
  }
  if (!active) return;
  // heap sort: pop the maximum into the tail
  for (int n = K; n > 1; --n) {
    const double md = hd[0]; const int mi = hi[0];
    const double d = hd[n - 1]; const int gi = hi[n - 1];
    int pos = 0;
    while (true) {
      const int l = 2 * pos + 1, r = l + 1;
      if (l >= n - 1) break;
      int c = l;
      if (r < n - 1 && key_less(hd[l], hi[l], hd[r], hi[r])) c = r;
      if (!key_less(d, gi, hd[c], hi[c])) break;
      hd[pos] = hd[c]; hi[pos] = hi[c];
      pos = c;
    }
    hd[pos] = d; hi[pos] = gi;
    hd[n - 1] = md; hi[n - 1] = mi;
  }
  for (int j = 0; j < K; ++j) out_idx[s * K + j] = hi[j] + (int)c0;
}

// ---- small clouds: one WARP per seed.  Each lane tests one cloud point per iteration; survivors are queued and merged
// by rank into a sorted shared-memory list 32 at a time, which amortises the exact fp64 work far better than the
// thread-per-seed kernel when every seed still sees many survivors (K ln(N/K) of N points).
constexpr int KNNW_WARPS = 8;
constexpr int KNNW_TILE = 1024;
constexpr int KNNW_QCAP = 64;


__global__ void __launch_bounds__(KNNW_WARPS * 32)
knn_seed_warp_kernel(const double* __restrict__ cloud, const float* __restrict__ cloud32, int64_t N,
                const double* __restrict__ seeds, int64_t S, int K, const float* __restrict__ rmax_p,
                int32_t* __restrict__ out_idx, const KnnSegs segs, int64_t npad_all) {
  __shared__ float tx[KNNW_TILE], ty[KNNW_TILE], tz[KNNW_TILE];
  __shared__ double ld[KNNW_WARPS][2][KNN_KMAX];
  __shared__ int li[KNNW_WARPS][2][KNN_KMAX];
  __shared__ double qd[KNNW_WARPS][KNNW_QCAP];
  __shared__ int qi[KNNW_WARPS][KNNW_QCAP];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int64_t c0, sb;
  knn_resolve(segs, KNNW_WARPS, c0, N, sb, S);
  cloud += 3 * c0;
  const float* cx = cloud32 + c0; const float* cy = cx + npad_all; const float* cz = cy + npad_all;
  const int64_t s = sb + warp;
  const bool active = s < S;
  const float rmax = *rmax_p;

  double sx = 0, sy = 0, sz = 0;
  if (active) { sx = seeds[3 * s]; sy = seeds[3 * s + 1]; sz = seeds[3 * s + 2]; }
  const float fx = (float)sx, fy = (float)sy, fz = (float)sz;

  int cur = 0;
  for (int j = lane; j < KNN_KMAX; j += 32) { ld[warp][0][j] = DBL_MAX; li[warp][0][j] = INT_MAX; }
  __syncwarp();
  double tau = DBL_MAX; int tau_i = INT_MAX;
  float tau32 = FLT_MAX;
  int qn = 0;

  auto flush = [&]() {
    // merge queue (qn unsorted, unique keys) into the sorted list by rank
    double* L = ld[warp][cur]; int* LI = li[warp][cur];
    double* Lo = ld[warp][cur ^ 1]; int* LIo = li[warp][cur ^ 1];
    for (int e = lane; e < qn; e += 32) {
      const double d = qd[warp][e]; const int id = qi[warp][e];
      int rank = 0;
      for (int j = 0; j < qn; ++j) rank += key_less(qd[warp][j], qi[warp][j], d, id) ? 1 : 0;
      int lo = 0, hi = K;   // first list position whose key is not less than (d,id)
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (key_less(L[mid], LI[mid], d, id)) lo = mid + 1; else hi = mid; }
      const int pos = rank + lo;
      if (pos < K) { Lo[pos] = d; LIo[pos] = id; }
    }
    for (int e = lane; e < K; e += 32) {
      const double d = L[e]; const int id = LI[e];
      int rank = 0;
      for (int j = 0; j < qn; ++j) rank += key_less(qd[warp][j], qi[warp][j], d, id) ? 1 : 0;
      const int pos = rank + e;
      if (pos < K) { Lo[pos] = d; LIo[pos] = id; }
    }
    __syncwarp();
    cur ^= 1; qn = 0;
    tau = ld[warp][cur][K - 1]; tau_i = li[warp][cur][K - 1];
    if (tau < DBL_MAX) {
      const float rt = sqrtf((float)tau) * 1.000002f;   // >= (1+2^-20) sqrt(tau) incl. rounding of the cast/sqrt
      const float b = rt + 4.76837158e-7f * rmax;       // 2^-21 Rmax
      tau32 = b * b * 1.000002f;
    }
    __syncwarp();
  };

  for (int64_t base = 0; base < N; base += KNNW_TILE) {
    const int tn = (int)min((int64_t)KNNW_TILE, N - base);
    __syncthreads();
    for (int j = threadIdx.x; j < tn; j += blockDim.x) { tx[j] = cx[base + j]; ty[j] = cy[base + j]; tz[j] = cz[base + j]; }
    __syncthreads();
    if (!active) continue;
    for (int j0 = 0; j0 < tn; j0 += 32) {
      const int j = j0 + lane;
      bool pass = false;
      if (j < tn) {
        const float dx = tx[j] - fx, dy = ty[j] - fy, dz = tz[j] - fz;
        const float d32 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
        pass = d32 <= tau32;
      }
      if (__any_sync(0xffffffffu, pass)) {
        double d = 0; const int gi = (int)(base + j);
        if (pass) {
          const double ex = cloud[3 * (int64_t)gi] - sx, ey = cloud[3 * (int64_t)gi + 1] - sy, ez = cloud[3 * (int64_t)gi + 2] - sz;
          d = __dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez));
          pass = key_less(d, gi, tau, tau_i);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, pass);
        if (bal) {
          if (pass) {
            const int pos = qn + __popc(bal & ((1u << lane) - 1u));
            qd[warp][pos] = d; qi[warp][pos] = gi;
          }
          qn += __popc(bal);
          __syncwarp();
          if (qn > KNNW_QCAP - 32) flush();
        }
      }
    }
  }
  if (active) {
    if (qn) flush();
    for (int j = lane; j < K; j += 32) out_idx[s * K + j] = li[warp][cur][j] + (int)c0;
  }
}

static int knn_set_attr() {
  static PerDeviceOnce once;
  return once.run([]() -> int {
    SAPCU_CUDA_CHECK(cudaFuncSetAttribute(knn_seed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)KNN_SMEM));
    return 0;
  });
}

int launch_knn_seed(const double* cloud, int64_t N, const double* seeds, int64_t S, int K, int32_t* idx,
                    float* cloud32_scratch, float* rmax_scratch, cudaStream_t st) {
  SAPCU_REQUIRE(K >= 1 && K <= KNN_KMAX, "sapcu_knn: K=%d outside [1,%d]", K, KNN_KMAX);
  SAPCU_REQUIRE(N >= K, "sapcu_knn: K=%d > N=%lld", K, (long long)N);
  SAPCU_REQUIRE(N < (int64_t)INT32_MAX / 3, "sapcu_knn: N too large for int32 indices");
  if (S == 0) return 0;
  SAPCU_CUDA_CHECK(cudaMemsetAsync(rmax_scratch, 0, sizeof(float), st));
  const int blocks = (int)std::min<int64_t>(ceil_div(N, 256), 148 * 8);
  cloud_to_f32_kernel<<<blocks, 256, 0, st>>>(cloud, N, cloud32_scratch, rmax_scratch);
  SAPCU_LAUNCH_CHECK();
  const int sblocks = (int)std::min<int64_t>(ceil_div(S, 256), 148 * 8);
  cloud_to_f32_kernel<<<sblocks, 256, 0, st>>>(seeds, S, nullptr, rmax_scratch);
  SAPCU_LAUNCH_CHECK();
  { const int rc = knn_set_attr(); if (rc) return rc; }
  if (N < (1 << 20))  // measured on B200 (N=1e5: 11 vs 30 ms; N=2e6: 165 vs 114 ms) (tools/knn_microbench.py): survivors dominate below, the scan above
    knn_seed_warp_kernel<<<(unsigned)ceil_div(S, KNNW_WARPS), KNNW_WARPS * 32, 0, st>>>(cloud, cloud32_scratch, N,
                                                                                       seeds, S, K, rmax_scratch, idx, KnnSegs{nullptr, nullptr, nullptr, 0}, knn_npad(N));
  else
    knn_seed_kernel<<<(unsigned)ceil_div(S, KNN_THREADS), KNN_THREADS, KNN_SMEM, st>>>(cloud, cloud32_scratch, N,
                                                                               seeds, S, K, rmax_scratch, idx, KnnSegs{nullptr, nullptr, nullptr, 0}, knn_npad(N));
  SAPCU_LAUNCH_CHECK();
  return 0;
}

// B independent (cloud, seed set) problems in ONE launch.  h_cloud_off / h_seed_off: [B+1] host prefix tables over the
// concatenated arrays; tab: device scratch for 3*(B+1) int64.  The kernel flavour is chosen from the largest cloud.
int launch_knn_seed_batched(const double* clouds, const int64_t* h_cloud_off, const double* seeds, const int64_t* h_seed_off,
                            int B, int K, int32_t* idx, float* cloud32_scratch, float* rmax_scratch, int64_t* tab,
                            cudaStream_t st) {
  SAPCU_REQUIRE(K >= 1 && K <= KNN_KMAX, "sapcu_knn_batched: K=%d outside [1,%d]", K, KNN_KMAX);
  SAPCU_REQUIRE(B >= 1 && h_cloud_off && h_seed_off && h_cloud_off[0] == 0 && h_seed_off[0] == 0, "sapcu_knn_batched: bad offset tables");
  const int64_t Ntot = h_cloud_off[B], Stot = h_seed_off[B];
  SAPCU_REQUIRE(Ntot < (int64_t)INT32_MAX / 3, "sapcu_knn_batched: too many cloud rows for int32 indices");
  int64_t nmax = 0;
  for (int b = 0; b < B; ++b) {
    const int64_t n = h_cloud_off[b + 1] - h_cloud_off[b], s = h_seed_off[b + 1] - h_seed_off[b];
    SAPCU_REQUIRE(s >= 0 && n >= 0, "sapcu_knn_batched: offsets must be non-decreasing");
    SAPCU_REQUIRE(s == 0 || n >= K, "sapcu_knn_batched: cloud %d has %lld points < K=%d", b, (long long)n, K);
    nmax = n > nmax ? n : nmax;
  }
  if (Stot == 0) return 0;
  const bool warp_kernel = nmax < (1 << 20);
  const int per_block = warp_kernel ? KNNW_WARPS : KNN_THREADS;
  std::vector<int64_t> h(3 * (size_t)(B + 1));
  int64_t* blk = h.data(); int64_t* co = blk + (B + 1); int64_t* so = co + (B + 1);
  blk[0] = 0;
  for (int b = 0; b < B; ++b) blk[b + 1] = blk[b] + ceil_div(h_seed_off[b + 1] - h_seed_off[b], per_block);
  for (int b = 0; b <= B; ++b) { co[b] = h_cloud_off[b]; so[b] = h_seed_off[b]; }
  SAPCU_REQUIRE(blk[B] < (int64_t)INT32_MAX, "sapcu_knn_batched: grid too large");
  SAPCU_CUDA_CHECK(cudaMemcpyAsync(tab, h.data(), h.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  SAPCU_CUDA_CHECK(cudaStreamSynchronize(st));               // `h` is a pageable temporary
  SAPCU_CUDA_CHECK(cudaMemsetAsync(rmax_scratch, 0, sizeof(float), st));
  const int blocks = (int)std::min<int64_t>(ceil_div(Ntot, 256), 148 * 8);
  cloud_to_f32_kernel<<<blocks, 256, 0, st>>>(clouds, Ntot, cloud32_scratch, rmax_scratch);
  SAPCU_LAUNCH_CHECK();
  const int sblocks = (int)std::min<int64_t>(ceil_div(Stot, 256), 148 * 8);
  cloud_to_f32_kernel<<<sblocks, 256, 0, st>>>(seeds, Stot, nullptr, rmax_scratch);
  SAPCU_LAUNCH_CHECK();
  { const int rc = knn_set_attr(); if (rc) return rc; }
  const KnnSegs segs{tab, tab + (B + 1), tab + 2 * (B + 1), B};
  if (warp_kernel)
    knn_seed_warp_kernel<<<(unsigned)blk[B], KNNW_WARPS * 32, 0, st>>>(clouds, cloud32_scratch, 0, seeds, 0, K,
                                                                      rmax_scratch, idx, segs, knn_npad(Ntot));
  else
    knn_seed_kernel<<<(unsigned)blk[B], KNN_THREADS, KNN_SMEM, st>>>(clouds, cloud32_scratch, 0, seeds, 0, K,
                                                                    rmax_scratch, idx, segs, knn_npad(Ntot));
  SAPCU_LAUNCH_CHECK();
  return 0;
}

}  // namespace sapcu
