// GPU seed generator: SURVEY.md section 8(f) "next" row 1 -- replaces the reference's separate `./dense` process
// (dense.cpp:175-252, file IPC through test.xyz / target.xyz) with a device-resident, level-synchronous version of the
// same voxel flood fill:
//   queue <- voxel of every input point (input order); pop v: skip if evaluated; d(v) = min over the 8 triangles
//   (p_i, p_8, p_9), i < 8, of the distance from the voxel centre to the triangle, where p_0..p_9 are the centre's 10
//   nearest input points in DESCENDING distance (p_9 nearest); emit the centre if 0.011 <= d <= 0.015; if d <= 0.015
//   push the 6 face neighbours that are not evaluated yet.
// A FIFO flood fill pops all of level L before level L+1, so processing whole levels in queue order with a
// keep-first de-duplication reproduces the reference's evaluation AND output order exactly.
//
// Faithful quirks (dense.cpp line numbers): the kd-tree is built over po[0..pnumber] INCLUSIVE (:193), i.e. with one
// extra all-zero point (`quirk_origin`); voxel ids use int arithmetic that may alias at the grid border (:189,:203-208,
// :237-240); comparisons against 0.0f / 1.0f literals; the emitted coordinates pass through "%lf" (6 decimals,
// :232) before generation.py reads them back (`round6`).  The reference's 5000-point cap (po[5001], :64) does not apply.
// All geometry is fp64 and this file is compiled with -fmad=false so every product/sum rounds as in the g++ build.
// Roofline: FP64 issue for the brute-force 10-NN (N+1 pair evaluations per visited voxel); HBM traffic negligible.
#include <float.h>
#include <math.h>
#include "../../include/sapcu_b200.h"
#include "common.cuh"
#include "geom.cuh"

namespace sapcu {

__device__ __forceinline__ V3 voxel_center(int id, int B, double cell) {
  int t = id;
  const int z = t % B; t /= B;
  const int y = t % B; t /= B;
  const int x = t;
  return {x * cell + 0.5 * cell - 0.5, y * cell + 0.5 * cell - 0.5, z * cell + 0.5 * cell - 0.5};
}

__device__ __forceinline__ bool bit_get(const unsigned* bm, int64_t i) { return (bm[i >> 5] >> (i & 31)) & 1u; }

// initial queue: voxel id of every input point (dense.cpp:186-191)
__global__ void seed_init_kernel(const double* __restrict__ cloud, int64_t N, double cell, int B, int* __restrict__ q) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double v = floor((cloud[3 * i] + 0.5) / cell) * B * B + floor((cloud[3 * i + 1] + 0.5) / cell) * B +
                   floor((cloud[3 * i + 2] + 0.5) / cell);
  q[i] = (int)v;
}

// keep-first claim: claim[id - id_lo] = smallest queue position holding id (only for ids not evaluated yet)
__global__ void seed_claim_kernel(const int* __restrict__ q, int n, const unsigned* __restrict__ evaluated, int64_t id_lo,
                                  int64_t id_hi, int* __restrict__ claim) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t id = q[i];
  if (id < id_lo || id >= id_hi) return;          // cannot be decoded consistently: never evaluated (see launcher note)
  if (bit_get(evaluated, id - id_lo)) return;
  atomicMin(&claim[id - id_lo], i);
}

// evaluate the claimed voxels: 10-NN by brute force over the (N + quirk) points, min triangle distance, flags
__global__ void __launch_bounds__(128)
seed_eval_kernel(const int* __restrict__ q, int n, const int* __restrict__ claim, int64_t id_lo, int64_t id_hi,
                 const double* __restrict__ cloud, int64_t N, int quirk_origin, double cell, int B,
                 int* __restrict__ flags /* bit0 evaluated-here, bit1 emit, bit2 expand */) {
  __shared__ double sx[256], sy[256], sz[256];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool mine = false; int id = 0;
  if (i < n) {
    id = q[i];
    mine = id >= id_lo && id < id_hi && claim[id - id_lo] == i;
  }
  const V3 c = voxel_center(id, B, cell);
  double bd[10]; int bi[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) { bd[k] = DBL_MAX; bi[k] = -1; }
  const int64_t NT = N + (quirk_origin ? 1 : 0);
  for (int64_t base = 0; base < NT; base += 256) {
    __syncthreads();
    for (int j = threadIdx.x; j < 256; j += blockDim.x) {
      const int64_t pidx = base + j;
      const bool real = pidx < N;
      sx[j] = real ? cloud[3 * pidx] : 0.0; sy[j] = real ? cloud[3 * pidx + 1] : 0.0; sz[j] = real ? cloud[3 * pidx + 2] : 0.0;
    }
    __syncthreads();
    if (!mine) continue;
    const int cnt = (int)((NT - base) < 256 ? (NT - base) : 256);
    for (int j = 0; j < cnt; ++j) {
      // dense.cpp:96-97: d = ((0 + dx^2) + dy^2) + dz^2 with (pt - p)
      const double dx = sx[j] - c.x, dy = sy[j] - c.y, dz = sz[j] - c.z;
      const double d = (dx * dx + dy * dy) + dz * dz;
      if (d < bd[9]) {                             // strict: an equal candidate does not replace (dense.cpp:106)
        int k = 9;
#pragma unroll
        for (int s = 9; s > 0; --s) {
          if (k == s && d < bd[s - 1]) { bd[s] = bd[s - 1]; bi[s] = bi[s - 1]; k = s - 1; }
        }
        bd[k] = d; bi[k] = (int)(base + j);
      }
    }
  }
  if (i >= n) return;
  int f = 0;
  if (mine) {
    // bd ascending: bd[0] nearest.  Reference order: pt[9] = nearest, pt[8] = second nearest, pt[0..7] the rest.
    auto P = [&](int k) -> V3 {
      const int64_t pi = bi[k];
      if (pi < 0 || pi >= N) return V3{0.0, 0.0, 0.0};          // the spurious origin point (or fewer than 10 points)
      return V3{cloud[3 * pi], cloud[3 * pi + 1], cloud[3 * pi + 2]};
    };
    const V3 p9 = P(0), p8 = P(1);
    double td = 99999999999999.0;
    for (int k = 2; k < 10; ++k) {
      const V3 t = point_tri(P(k), p8, p9, c);
      const double dd = vdist(t, c);
      if (dd < td) td = dd;
    }
    f = 1;
    if (td >= 0.0110 && td <= 0.0150) f |= 2;
    if (td <= 0.0150) f |= 4;
  }
  flags[i] = f;
}

// scans: exclusive prefix sums of (emit) and (expand) flags -> stable output positions
__global__ void seed_flag_counts_kernel(const int* __restrict__ flags, int n, int* __restrict__ emit, int* __restrict__ expand) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  emit[i] = (flags[i] >> 1) & 1;
  expand[i] = (flags[i] >> 2) & 1;
}

constexpr int SCAN_T = 256, SCAN_ITEMS = 8, SCAN_TILE = SCAN_T * SCAN_ITEMS;
// in-place exclusive scan of one tile per block; block totals to `sums`
__global__ void scan_tile_kernel(int* __restrict__ a, int n, int* __restrict__ sums) {
  __shared__ int wsum[SCAN_T / 32];
  const int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  int v[SCAN_ITEMS]; int tot = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) { v[k] = (base + k < n) ? a[base + k] : 0; tot += v[k]; }
  int inc = tot;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = lane < SCAN_T / 32 ? wsum[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
    if (lane < SCAN_T / 32) wsum[lane] = w;
  }
  __syncthreads();
  int run = inc - tot + (warp ? wsum[warp - 1] : 0);
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) { if (base + k < n) a[base + k] = run; run += v[k]; }
  if (threadIdx.x == SCAN_T - 1) sums[blockIdx.x] = run;
}
__global__ void scan_sums_kernel(int* __restrict__ sums, int nb, int* __restrict__ total) {   // single block, serial over chunks
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int b0 = 0; b0 < nb; b0 += blockDim.x) {
    const int i = b0 + threadIdx.x;
    int v = i < nb ? sums[i] : 0;
    int inc = v;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ int ws[32];
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) ws[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      int w = lane < (int)(blockDim.x >> 5) ? ws[lane] : 0;
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
      ws[lane] = w;
    }
    __syncthreads();
    const int excl = inc - v + (warp ? ws[warp - 1] : 0) + carry;
    if (i < nb) sums[i] = excl;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}
__global__ void scan_add_kernel(int* __restrict__ a, int n, const int* __restrict__ sums) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] += sums[i / SCAN_TILE];
}

// mark evaluated, write emitted centres (BFS order) and the children of expanding voxels (parent order, then direction)
__global__ void seed_commit_kernel(const int* __restrict__ q, int n, const int* __restrict__ flags, const int* __restrict__ emit_pos,
                                   const int* __restrict__ expand_pos, int64_t id_lo, unsigned* __restrict__ evaluated, double cell,
                                   int B, int round6, double* __restrict__ seeds, int64_t seeds_base, int64_t cap,
                                   int* __restrict__ children) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int f = flags[i];
  if (!(f & 1)) return;
  const int id = q[i];
  atomicOr(&evaluated[(id - id_lo) >> 5], 1u << ((id - id_lo) & 31));
  if (f & 2) {
    const int64_t o = seeds_base + emit_pos[i];
    if (o < cap) {
      V3 c = voxel_center(id, B, cell);
      if (round6) {   // fprintf("%lf") + np.loadtxt: nearest double to the 6-decimal rendering
        c.x = nearbyint(c.x * 1e6) / 1e6; c.y = nearbyint(c.y * 1e6) / 1e6; c.z = nearbyint(c.z * 1e6) / 1e6;
      }
      seeds[3 * o] = c.x; seeds[3 * o + 1] = c.y; seeds[3 * o + 2] = c.z;
    }
  }
  if (f & 4) {
    int t = id;
    const int z = t % B; t /= B;
    const int y = t % B; t /= B;
    const int x = t;
    const int go[6][3] = {{1, 0, 0}, {-1, 0, 0}, {0, 1, 0}, {0, -1, 0}, {0, 0, 1}, {0, 0, -1}};
    int* ch = children + 6 * (int64_t)expand_pos[i];
#pragma unroll
    for (int d = 0; d < 6; ++d) ch[d] = (x + go[d][0]) * B * B + (y + go[d][1]) * B + (z + go[d][2]);
  }
}
__global__ void seed_reset_claim_kernel(const int* __restrict__ q, int n, int64_t id_lo, int64_t id_hi, int* __restrict__ claim) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t id = q[i];
  if (id >= id_lo && id < id_hi) claim[id - id_lo] = 0x7fffffff;
}
__global__ void fill_i32_kernel(int* __restrict__ a, int64_t n, int v) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) a[i] = v;
}

struct SeedPlan {
  int B; int64_t id_lo, id_hi, nvox;
  size_t off_eval, off_claim, off_q0, off_q1, off_flags, off_emit, off_expand, off_sums, off_total, bytes;
  int64_t qcap;
};
static SeedPlan seed_plan(int64_t N, double cell, int64_t cap) {
  SeedPlan p;
  p.B = (int)round(1.0 / cell);
  const int64_t B = p.B;
  // x is the top "digit" of a voxel id, so the flood fill legitimately runs past x = B when the cloud touches the +x
  // face (the band reaches 0.015 + one cell beyond the surface); y/z overflow and negative indices alias exactly as in
  // the reference.  Ids outside [id_lo, id_hi) cannot be produced by an expanding voxel.
  const int64_t xpad = (int64_t)ceil(0.015 / cell) + 4;
  p.id_lo = -(B * B + B + 1);
  p.id_hi = (B + xpad + 1) * B * B + 2 * (B * B + B + 1);
  p.nvox = p.id_hi - p.id_lo;
  // a level holds 6 children per expanding voxel; a level is a thin shell of the band around the surface, bounded here
  // by 64 B^2 voxels (a unit-box surface has <= 6 B^2 cells per layer) independently of the output capacity
  int64_t lvl = 64 * B * B;
  if (cap > lvl) lvl = cap;
  if (N > lvl) lvl = N;
  p.qcap = 6 * lvl + 1024;
  size_t o = 0;
  auto take = [&](size_t b) { size_t r = o; o = align_up(o + b, 256); return r; };
  p.off_eval = take(((size_t)p.nvox + 31) / 32 * 4);
  p.off_claim = take((size_t)p.nvox * 4);
  p.off_q0 = take((size_t)p.qcap * 4); p.off_q1 = take((size_t)p.qcap * 4);
  p.off_flags = take((size_t)p.qcap * 4); p.off_emit = take((size_t)p.qcap * 4); p.off_expand = take((size_t)p.qcap * 4);
  p.off_sums = take(((size_t)p.qcap / SCAN_TILE + 2) * 4 * 2);
  p.off_total = take(256);
  p.bytes = o;
  return p;
}

static int scan_exclusive(int* a, int n, int* sums, int* total_dev, cudaStream_t st) {
  const int nb = (int)ceil_div(n, SCAN_TILE);
  scan_tile_kernel<<<nb, SCAN_T, 0, st>>>(a, n, sums);
  SAPCU_LAUNCH_CHECK();
  scan_sums_kernel<<<1, 1024, 0, st>>>(sums, nb, total_dev);
  SAPCU_LAUNCH_CHECK();
  scan_add_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(a, n, sums);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

}  // namespace sapcu

using namespace sapcu;

extern "C" {

size_t sapcu_seedgen_workspace_bytes(int64_t N, double cell, int64_t cap) {
  if (N < 1 || !(cell > 0.0) || cap < 1 || 1.0 / cell > 1000.0) return 0;
  return seed_plan(N, cell, cap).bytes;
}

int sapcu_seedgen(const double* d_cloud, int64_t N, double cell, int quirk_origin, int round6, double* d_seeds, int64_t cap,
                  int64_t* h_count, void* d_ws, size_t ws_bytes, void* stream) {
  SAPCU_REQUIRE(d_cloud && d_seeds && h_count && d_ws && N >= 1 && cap >= 1 && cell > 0.0, "seedgen: bad argument");
  SAPCU_REQUIRE(1.0 / cell <= 1000.0, "seedgen: cell %g gives a grid above 1000^3", cell);
  SAPCU_REQUIRE(N < (1 << 30), "seedgen: too many points");
  const SeedPlan p = seed_plan(N, cell, cap);
  if (ws_bytes < p.bytes) { set_error("seedgen: workspace %zu < %zu bytes", ws_bytes, p.bytes); return SAPCU_EWORKSPACE; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* ws = reinterpret_cast<char*>(d_ws);
  unsigned* evaluated = reinterpret_cast<unsigned*>(ws + p.off_eval);
  int* claim = reinterpret_cast<int*>(ws + p.off_claim);
  int* q[2] = {reinterpret_cast<int*>(ws + p.off_q0), reinterpret_cast<int*>(ws + p.off_q1)};
  int* flags = reinterpret_cast<int*>(ws + p.off_flags);
  int* emit = reinterpret_cast<int*>(ws + p.off_emit);
  int* expand = reinterpret_cast<int*>(ws + p.off_expand);
  int* sums = reinterpret_cast<int*>(ws + p.off_sums);
  int* totals = reinterpret_cast<int*>(ws + p.off_total);
  SAPCU_CUDA_CHECK(cudaMemsetAsync(evaluated, 0, ((size_t)p.nvox + 31) / 32 * 4, st));
  fill_i32_kernel<<<1184, 256, 0, st>>>(claim, p.nvox, 0x7fffffff);
  SAPCU_LAUNCH_CHECK();
  seed_init_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, st>>>(d_cloud, N, cell, p.B, q[0]);
  SAPCU_LAUNCH_CHECK();
  int64_t n = N, emitted = 0;
  int cur = 0;
  for (int level = 0; n > 0; ++level) {
    SAPCU_REQUIRE(level < 100000, "seedgen: flood fill did not terminate");
    const unsigned g = (unsigned)ceil_div(n, 256);
    seed_claim_kernel<<<g, 256, 0, st>>>(q[cur], (int)n, evaluated, p.id_lo, p.id_hi, claim);
    SAPCU_LAUNCH_CHECK();
    seed_eval_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, st>>>(q[cur], (int)n, claim, p.id_lo, p.id_hi, d_cloud, N, quirk_origin,
                                                                cell, p.B, flags);
    SAPCU_LAUNCH_CHECK();
    seed_flag_counts_kernel<<<g, 256, 0, st>>>(flags, (int)n, emit, expand);
    SAPCU_LAUNCH_CHECK();
    int rc = scan_exclusive(emit, (int)n, sums, totals, st);
    if (rc) return rc;
    rc = scan_exclusive(expand, (int)n, sums, totals + 1, st);
    if (rc) return rc;
    int h_tot[2];
    SAPCU_CUDA_CHECK(cudaMemcpyAsync(h_tot, totals, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
    SAPCU_CUDA_CHECK(cudaStreamSynchronize(st));
    const int64_t n_next = 6 * (int64_t)h_tot[1];
    if (n_next > p.qcap) { set_error("seedgen: frontier of %lld voxels exceeds the workspace (raise cap)", (long long)n_next); return SAPCU_EWORKSPACE; }
    seed_commit_kernel<<<g, 256, 0, st>>>(q[cur], (int)n, flags, emit, expand, p.id_lo, evaluated, cell, p.B, round6, d_seeds, emitted,
                                          cap, q[cur ^ 1]);
    SAPCU_LAUNCH_CHECK();
    seed_reset_claim_kernel<<<g, 256, 0, st>>>(q[cur], (int)n, p.id_lo, p.id_hi, claim);
    SAPCU_LAUNCH_CHECK();
    emitted += h_tot[0];
    n = n_next;
    cur ^= 1;
  }
  SAPCU_CUDA_CHECK(cudaStreamSynchronize(st));
  *h_count = emitted;                  // may exceed cap: only the first `cap` seeds were stored
  return 0;
}

}  // extern "C"
