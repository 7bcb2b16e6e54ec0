// Pair table of an fn chunk: the distinct global point pairs (gidx[s,pt], gidx[s,nb]) behind the edges of the intra-patch
// graphs, so that fn's positional encoding (a pure function of the offset p_i - p_j) is evaluated once per pair.
//
//   key     e = pt*kmax + j -> ((gi * N + gj) << jb) | j   (jb bits hold the neighbour rank j < kmax)
//   sort    LSD radix sort (CUB, caller-provided temporary storage) over the bits N^2 * 2^jb needs, carrying e
//   scan    head of a run of equal pairs = its smallest rank j; block b keeps the pairs whose smallest rank is < kk_b
//           (the k = 12 / 18 graphs are prefixes of the top-kmax one), numbered in key order by an inclusive scan
//   emit    pid_b[pt*kk_b + j] = pair row of edge (pt, j), delta_b[u] = (float)(cloud[gi] - cloud[gj]) (fp64 difference,
//           one rounding), U_b = pair count (device memory: the forward never reads it back)
// Every buffer is sized for U = E, so the workspace bound does not depend on the cloud.  The key takes 2 * ceil(log2 N) +
// ceil(log2 kmax) bits (pair_key_fits; 22 + 5 = 27 for the 2,048-point cloud of configs[1]: four 8-bit radix passes).
#include <cub/cub.cuh>
#include "common.cuh"
#include "kernels.h"

namespace sapcu {

namespace {

// bits that hold every value below n
int bits_for(uint64_t n) { int b = 0; while (b < 64 && ((n - 1) >> b) != 0) ++b; return b; }

__global__ void pair_keys_kernel(const int32_t* __restrict__ idx, int kmax, int M, int64_t E, const int32_t* __restrict__ gidx,
                                 int64_t ldg, int64_t N, int jb, uint64_t* __restrict__ key, int32_t* __restrict__ val, int* err) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int64_t pt = e / kmax;
  const int j = (int)(e - pt * kmax);
  const int64_t s = pt / M;
  const int i = (int)(pt - s * M);
  const int nb = idx[e];
  int64_t gi = gidx[s * ldg + i], gj = gidx[s * ldg + nb];
  if (gi < 0 || gi >= N || gj < 0 || gj >= N) {        // never read outside the cloud: flag the forward as failed
    atomicOr(err, 2);
    gi = 0; gj = 0;
  }
  key[e] = ((uint64_t)(gi * N + gj) << jb) | (uint64_t)j;
  val[e] = (int32_t)e;
}

__global__ void pair_flags_kernel(const uint64_t* __restrict__ key, int64_t E, int jb, int3 kk, int* __restrict__ f0,
                                  int* __restrict__ f1, int* __restrict__ f2) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= E) return;
  const uint64_t k = key[i];
  const bool head = i == 0 || (k >> jb) != (key[i - 1] >> jb);
  const int j = (int)(k & ((1ull << jb) - 1));
  f0[i] = head && j < kk.x; f1[i] = head && j < kk.y; f2[i] = head && j < kk.z;
}

__global__ void pair_emit_kernel(const uint64_t* __restrict__ key, const int32_t* __restrict__ val, int64_t E, int jb, int kmax,
                                 const double* __restrict__ cloud, int64_t N, int3 kk, const int* __restrict__ s0,
                                 const int* __restrict__ s1, const int* __restrict__ s2, int32_t* pid0, int32_t* pid1, int32_t* pid2,
                                 float4* d0, float4* d1, float4* d2, int* __restrict__ U) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= E) return;
  const uint64_t k = key[i];
  const bool head = i == 0 || (k >> jb) != (key[i - 1] >> jb);
  const int64_t e = val[i];
  const int64_t pt = e / kmax;
  const int j = (int)(e - pt * kmax);
  float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
  if (head) {
    const uint64_t g = k >> jb;
    const int64_t gi = (int64_t)(g / (uint64_t)N), gj = (int64_t)(g - (uint64_t)gi * (uint64_t)N);
    d = make_float4((float)(cloud[3 * gi] - cloud[3 * gj]), (float)(cloud[3 * gi + 1] - cloud[3 * gj + 1]),
                    (float)(cloud[3 * gi + 2] - cloud[3 * gj + 2]), 0.f);
  }
  const int kb[3] = {kk.x, kk.y, kk.z};
  const int* sc[3] = {s0, s1, s2};
  int32_t* pid[3] = {pid0, pid1, pid2};
  float4* dl[3] = {d0, d1, d2};
#pragma unroll
  for (int b = 0; b < 3; ++b) {
    if (j >= kb[b]) continue;
    const int u = sc[b][i] - 1;
    pid[b][pt * kb[b] + j] = u;
    if (head) dl[b][u] = d;
  }
  if (i == E - 1) { U[0] = s0[i]; U[1] = s1[i]; U[2] = s2[i]; }
}

}  // namespace

bool pair_key_fits(int64_t N, int kmax) {
  return N >= 1 && kmax >= 1 && N <= (1ll << 31) && 2 * bits_for((uint64_t)N) + bits_for((uint64_t)kmax) <= 64;
}

PairBufs pair_plan(int64_t P, int kmax, const int kk[3], int64_t N, void* base) {
  PairBufs q;
  const int64_t E = P * kmax;
  char* b = reinterpret_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) { off = align_up(off, 256); char* p = b + off; off += bytes; return p; };
  q.E = E; q.kmax = kmax;
  q.jb = bits_for((uint64_t)kmax);
  q.bits = bits_for((uint64_t)N * (uint64_t)N) + q.jb;
  if (q.bits < 1) q.bits = 1;
  for (int i = 0; i < 2; ++i) { q.key[i] = reinterpret_cast<uint64_t*>(take(E * 8)); q.val[i] = reinterpret_cast<int32_t*>(take(E * 4)); }
  for (int i = 0; i < 3; ++i) {
    q.kk[i] = kk[i];
    q.flag[i] = reinterpret_cast<int*>(take(E * 4));
    q.pid[i] = reinterpret_cast<int32_t*>(take(P * kk[i] * 4));
    q.delta[i] = reinterpret_cast<float4*>(take(P * kk[i] * 16));
  }
  q.U = reinterpret_cast<int*>(take(3 * sizeof(int)));
  size_t t_sort = 0, t_scan = 0;
  cub::DoubleBuffer<uint64_t> kd(nullptr, nullptr);
  cub::DoubleBuffer<int32_t> vd(nullptr, nullptr);
  cub::DeviceRadixSort::SortPairs(nullptr, t_sort, kd, vd, E, 0, q.bits);
  cub::DeviceScan::InclusiveSum(nullptr, t_scan, (int*)nullptr, (int*)nullptr, E);
  q.tmp_bytes = t_sort > t_scan ? t_sort : t_scan;
  q.tmp = take(q.tmp_bytes);
  q.bytes = align_up(off, 256);
  return q;
}

int build_pairs(const PairBufs& q, const int32_t* idx, int M, const int32_t* gidx, int64_t ldg, const double* cloud, int64_t N,
                int* err, cudaStream_t st) {
  const int64_t E = q.E;
  if (E == 0) return 0;
  SAPCU_REQUIRE(E < (1ll << 31), "edge_pairs: %lld edges in one chunk exceed the 32-bit edge ids", (long long)E);
  const unsigned g = (unsigned)ceil_div(E, 256);
  pair_keys_kernel<<<g, 256, 0, st>>>(idx, q.kmax, M, E, gidx, ldg, N, q.jb, q.key[0], q.val[0], err);
  SAPCU_LAUNCH_CHECK();
  cub::DoubleBuffer<uint64_t> kd(q.key[0], q.key[1]);
  cub::DoubleBuffer<int32_t> vd(q.val[0], q.val[1]);
  size_t tb = q.tmp_bytes;
  SAPCU_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(q.tmp, tb, kd, vd, E, 0, q.bits, st));
  const int3 kk = make_int3(q.kk[0], q.kk[1], q.kk[2]);
  pair_flags_kernel<<<g, 256, 0, st>>>(kd.Current(), E, q.jb, kk, q.flag[0], q.flag[1], q.flag[2]);
  SAPCU_LAUNCH_CHECK();
  for (int b = 0; b < 3; ++b) {     // in place: flag -> pair number + 1
    tb = q.tmp_bytes;
    SAPCU_CUDA_CHECK(cub::DeviceScan::InclusiveSum(q.tmp, tb, q.flag[b], q.flag[b], E, st));
  }
  pair_emit_kernel<<<g, 256, 0, st>>>(kd.Current(), vd.Current(), E, q.jb, q.kmax, cloud, N, kk, q.flag[0], q.flag[1], q.flag[2],
                                      q.pid[0], q.pid[1], q.pid[2], q.delta[0], q.delta[1], q.delta[2], q.U);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

}  // namespace sapcu
