// "Next" rows 2 and 3 of SURVEY.md section 8(f): the two steps that follow the hot path in the reference.
//   outlier filter  generation.py:176-183  self-kNN (k = 30, fp64, sapcu_knn) -> per-point mean neighbour distance ->
//                   keep points whose mean is below threshold x the global mean
//   FPS             generate.py:56-74      farthest point sampling in fp32, start index N/2, distances initialised to
//                   1e32, `dist < distance` update, arg-max with the lowest index on ties
// Roofline: outlier statistics are HBM-bound (S*K*4 B of indices + L2-resident point gathers); FPS is latency-bound by
// one grid-wide barrier per selected point (a cooperative persistent kernel keeps the running distances in registers).
#include <cooperative_groups.h>
#include <float.h>
#include "../../include/sapcu_b200.h"
#include "common.cuh"

namespace cg = cooperative_groups;

namespace sapcu {

// avg[i] = mean_j sqrt(|p_i - p_idx[i][j]|^2), numpy's pairwise summation order for a row of K <= 128 doubles (numpy
// halves longer rows recursively, an order this kernel does not restate)
// qry: the S query points (== pts for the single-GPU filter; a rank's own rows of the gathered points when sharded)
__global__ void knn_mean_dist_kernel(const double* __restrict__ pts, const double* __restrict__ qry, const int32_t* __restrict__ idx,
                                     int64_t S, int K, double* __restrict__ avg) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= S) return;
  const double x = qry[3 * i], y = qry[3 * i + 1], z = qry[3 * i + 2];
  auto dist = [&](int j) {
    const int64_t p = idx[i * K + j];
    const double dx = pts[3 * p] - x, dy = pts[3 * p + 1] - y, dz = pts[3 * p + 2] - z;
    return sqrt(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
  };
  double sum;
  if (K < 8) {
    sum = 0.0;
    for (int j = 0; j < K; ++j) sum = __dadd_rn(sum, dist(j));
  } else {        // numpy pairwise_sum, n <= 128: eight strided accumulators, tree combine, sequential tail
    double r[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) r[t] = dist(t);
    int j = 8;
    for (; j + 8 <= K; j += 8) {
#pragma unroll
      for (int t = 0; t < 8; ++t) r[t] = __dadd_rn(r[t], dist(j + t));
    }
    sum = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; j < K; ++j) sum = __dadd_rn(sum, dist(j));
  }
  avg[i] = sum / (double)K;
}

// deterministic fp64 sum of n values into *out (single block; n is ~1e5..1e6)
__global__ void sum_f64_kernel(const double* __restrict__ a, int64_t n, double* __restrict__ out) {
  __shared__ double sh[1024];
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += a[i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = blockDim.x >> 1; o; o >>= 1) {
    if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = sh[0];
}

// rows [lo, lo + n) of the S row means -> keep[0..n)
__global__ void outlier_mask_kernel(const double* __restrict__ avg, int64_t S, int64_t lo, int64_t n, const double* __restrict__ total,
                                    double threshold, uint8_t* __restrict__ keep) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double avgtotal = *total / (double)S;           // mean over all S*K distances == mean of the row means
  keep[i] = avg[lo + i] < avgtotal * threshold ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------- FPS
constexpr int FPS_THREADS = 512;
constexpr int FPS_PER_THREAD = 8;          // points owned by one thread (registers); capacity = grid * 512 * 8

__global__ void __launch_bounds__(FPS_THREADS)
fps_kernel(const float* __restrict__ xyz, int N, int npoint, int start, int32_t* __restrict__ out,
           unsigned long long* __restrict__ keys /* [3], zero-initialised */) {
  cg::grid_group grid = cg::this_grid();
  __shared__ unsigned long long wkey[FPS_THREADS / 32];
  const int tid = blockIdx.x * FPS_THREADS + threadIdx.x;
  const int stride = gridDim.x * FPS_THREADS;
  float px[FPS_PER_THREAD], py[FPS_PER_THREAD], pz[FPS_PER_THREAD], dmin[FPS_PER_THREAD];
#pragma unroll
  for (int k = 0; k < FPS_PER_THREAD; ++k) {
    const int p = tid + k * stride;
    const bool v = p < N;
    px[k] = v ? xyz[3 * p] : 0.f; py[k] = v ? xyz[3 * p + 1] : 0.f; pz[k] = v ? xyz[3 * p + 2] : 0.f;
    dmin[k] = 1e32f;
  }
  int far = start;
  for (int it = 0; it < npoint; ++it) {
    if (tid == 0) out[it] = far;
    const float cx = xyz[3 * far], cy = xyz[3 * far + 1], cz = xyz[3 * far + 2];
    unsigned long long best = 0ull;
#pragma unroll
    for (int k = 0; k < FPS_PER_THREAD; ++k) {
      const int p = tid + k * stride;
      if (p < N) {
        const float dx = __fsub_rn(px[k], cx), dy = __fsub_rn(py[k], cy), dz = __fsub_rn(pz[k], cz);
        const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
        if (d < dmin[k]) dmin[k] = d;
        const unsigned long long key = ((unsigned long long)__float_as_uint(dmin[k]) << 32) | (unsigned)(0xFFFFFFFFu - (unsigned)p);
        best = key > best ? key : best;
      }
    }
    for (int o = 16; o; o >>= 1) { const unsigned long long t = __shfl_xor_sync(0xffffffffu, best, o); best = t > best ? t : best; }
    if ((threadIdx.x & 31) == 0) wkey[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x < 32) {
      unsigned long long b = threadIdx.x < FPS_THREADS / 32 ? wkey[threadIdx.x] : 0ull;
      for (int o = 16; o; o >>= 1) { const unsigned long long t = __shfl_xor_sync(0xffffffffu, b, o); b = t > b ? t : b; }
      if (threadIdx.x == 0) atomicMax(&keys[it % 3], b);
    }
    grid.sync();
    const unsigned long long g = *reinterpret_cast<volatile unsigned long long*>(&keys[it % 3]);
    far = (int)(0xFFFFFFFFu - (unsigned)(g & 0xFFFFFFFFull));
    if (tid == 0) keys[(it + 2) % 3] = 0ull;     // used again two iterations (and one more grid barrier) from now
  }
}

}  // namespace sapcu

using namespace sapcu;

extern "C" {

size_t sapcu_outlier_workspace_bytes(int64_t S) { return S < 0 ? 0 : align_up((size_t)S * 8, 256) + 256; }

int sapcu_outlier_mask(const double* d_points, int64_t S, const int32_t* d_idx, int K, double threshold, uint8_t* d_keep,
                       void* d_ws, size_t ws_bytes, void* stream) {
  SAPCU_REQUIRE(S >= 0 && K >= 1 && (S == 0 || (d_points && d_idx && d_keep && d_ws)), "outlier_mask: bad argument");
  SAPCU_REQUIRE(K <= 128, "outlier_mask: K=%d > 128", K);
  if (ws_bytes < sapcu_outlier_workspace_bytes(S)) { set_error("outlier_mask: workspace too small"); return SAPCU_EWORKSPACE; }
  if (S == 0) return 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  double* avg = reinterpret_cast<double*>(d_ws);
  double* total = reinterpret_cast<double*>(reinterpret_cast<char*>(d_ws) + align_up((size_t)S * 8, 256));
  knn_mean_dist_kernel<<<(unsigned)ceil_div(S, 128), 128, 0, st>>>(d_points, d_points, d_idx, S, K, avg);
  SAPCU_LAUNCH_CHECK();
  sum_f64_kernel<<<1, 1024, 0, st>>>(avg, S, total);
  SAPCU_LAUNCH_CHECK();
  outlier_mask_kernel<<<(unsigned)ceil_div(S, 256), 256, 0, st>>>(avg, S, 0, S, total, threshold, d_keep);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

int sapcu_knn_mean_dist(const double* d_points, int64_t S, const double* d_query, int64_t rows, const int32_t* d_idx, int K,
                        double* d_mean, void* stream) {
  SAPCU_REQUIRE(S >= 1 && rows >= 0 && K >= 1 && d_points && (rows == 0 || (d_query && d_idx && d_mean)), "knn_mean_dist: bad argument");
  SAPCU_REQUIRE(K <= 128, "knn_mean_dist: K=%d > 128", K);
  if (rows == 0) return 0;
  knn_mean_dist_kernel<<<(unsigned)ceil_div(rows, 128), 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(d_points, d_query, d_idx, rows, K, d_mean);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

int sapcu_outlier_mask_from_means(const double* d_mean_all, int64_t S, int64_t row_lo, int64_t rows, double threshold, uint8_t* d_keep,
                                  void* d_ws, size_t ws_bytes, void* stream) {
  SAPCU_REQUIRE(S >= 1 && row_lo >= 0 && rows >= 0 && row_lo + rows <= S && d_mean_all && d_ws && (rows == 0 || d_keep), "outlier_mask_from_means: bad argument");
  SAPCU_REQUIRE(ws_bytes >= 256, "outlier_mask_from_means: workspace of 256 bytes needed");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  double* total = reinterpret_cast<double*>(d_ws);
  sum_f64_kernel<<<1, 1024, 0, st>>>(d_mean_all, S, total);          // the same fixed summation order on every rank
  SAPCU_LAUNCH_CHECK();
  if (rows == 0) return 0;
  outlier_mask_kernel<<<(unsigned)ceil_div(rows, 256), 256, 0, st>>>(d_mean_all, S, row_lo, rows, total, threshold, d_keep);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

int sapcu_fps(const float* d_xyz, int64_t N, int64_t npoint, int64_t start, int32_t* d_out, void* d_ws, size_t ws_bytes,
              void* stream) {
  SAPCU_REQUIRE(d_xyz && d_out && d_ws && N >= 1 && npoint >= 0 && start >= 0 && start < N, "fps: bad argument");
  SAPCU_REQUIRE(ws_bytes >= 32, "fps: workspace of 32 bytes needed");
  SAPCU_REQUIRE(reinterpret_cast<uintptr_t>(d_ws) % 8 == 0, "fps: workspace %p is not 8-byte aligned", d_ws);
  SAPCU_REQUIRE(N < ((int64_t)1 << 31) && npoint < ((int64_t)1 << 31), "fps: sizes must fit 32 bits");
  if (npoint == 0) return 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int per_sm = 0;
  SAPCU_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fps_kernel, FPS_THREADS, 0));
  int dev = 0, sms = 0;
  SAPCU_CUDA_CHECK(cudaGetDevice(&dev));
  SAPCU_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int64_t max_blocks = (int64_t)per_sm * sms;
  int64_t blocks = ceil_div(N, (int64_t)FPS_THREADS * FPS_PER_THREAD);
  if (blocks > max_blocks) { set_error("fps: N=%lld exceeds the co-resident capacity %lld", (long long)N, (long long)(max_blocks * FPS_THREADS * FPS_PER_THREAD)); return SAPCU_EINVAL; }
  if (blocks < sms && N > (int64_t)FPS_THREADS) blocks = ceil_div(N, FPS_THREADS) < sms ? ceil_div(N, FPS_THREADS) : sms;   // spread small clouds
  SAPCU_CUDA_CHECK(cudaMemsetAsync(d_ws, 0, 32, st));
  int n = (int)N, np_ = (int)npoint, s0 = (int)start;
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(d_ws);
  void* args[] = {(void*)&d_xyz, (void*)&n, (void*)&np_, (void*)&s0, (void*)&d_out, (void*)&keys};
  SAPCU_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)fps_kernel, dim3((unsigned)blocks), dim3(FPS_THREADS), args, 0, st));
  count_launch();
  return 0;
}

}  // extern "C"
