// Exact point-to-triangle-mesh distance over a linear BVH built on the device (Karras 2012), one tree per call.
//   keys    per face the 30-bit Morton code of its centroid (10 bits per axis, quantised in the centroids' bounding box),
//           then the face index: the 64-bit key (morton << 32) | face is unique, so the tree is well defined
//   sort    stable LSD radix sort of the Morton codes, 5 bits per pass (6 passes), carrying the face index; starting from
//           face order, a stable sort by the code alone is the sort by the full (code, face) key
//   build   internal nodes by Karras's split search over the sorted keys; boxes fitted bottom-up, one atomic arrival
//           counter per internal node (the second child to arrive fits its parent); box bounds are exact fp64 min/max of
//           vertex coordinates
//   query   one thread per point, nearest child first, a child pruned only when its box bound is STRICTLY greater than the
//           best D so far, so a face whose D equals the best (and may carry a lower index) is never pruned
// Per face the distance is D(p, f) of face_dist2 below; the result is min over faces of (D, face index), i.e. bitwise the
// brute-force minimum, whatever the tree, the launch configuration or the order of the query points.
// This file is compiled with -fmad=false (_native._FILE_FLAGS), like seedgen.cu.
#include <float.h>
#include <math.h>
#include "../../include/sapcu_b200.h"
#include "common.cuh"
#include "geom.cuh"

namespace sapcu {

constexpr int MD_THREADS = 256;
constexpr int MD_QUERY_THREADS = 128;
constexpr int RADIX_BITS = 5, RADIX = 1 << RADIX_BITS, RADIX_PASSES = 6;    // 6 x 5 bits cover the 30-bit Morton code
constexpr int RADIX_ITEMS = 8, RADIX_TILE = MD_THREADS * RADIX_ITEMS;
// Tree depth: along a root-to-leaf path the common-prefix length of the internal nodes' key ranges strictly increases.
// Distinct keys below 2^62 share between 2 and 63 leading bits, so a path holds at most 62 internal nodes, and the
// traversal stack (one pushed sibling per internal node of the current path) never holds more than 62 entries.
constexpr int MD_STACK = 64;

struct Box { double lo[3], hi[3]; };

struct MeshWs {
  unsigned long long* cbox;   // [6] ordered keys: min x,y,z then max x,y,z of the face centroids
  unsigned* code[2];          // [2][F] Morton codes, radix ping-pong
  int32_t* face[2];           // [2][F] face indices, radix ping-pong; face[0] is the sorted order after the 6 passes
  int* counts;                // [RADIX * nb] per-digit, per-tile counts, then their exclusive scan
  int* left;                  // [F-1] children of internal node i: c >= 0 internal node c, c < 0 the leaf ~c (sorted position)
  int* right;                 // [F-1]
  int* inner_parent;          // [F-1] -1 at the root (internal node 0)
  int* leaf_parent;           // [F]
  int* arrive;                // [F-1] arrival counters of the bottom-up box fit
  Box* inner_box;             // [F-1]
  Box* leaf_box;              // [F]
  double* tri;                // [F][9] the leaf's triangle a, b, c (sorted order)
  int32_t* leaf_face;         // [F] the leaf's face index, -1 for a face with an index outside [0, V)
};

static int64_t radix_tiles(int64_t F) { return ceil_div(F, RADIX_TILE); }

static size_t mesh_bytes(int64_t F, MeshWs* w, char* base) {
  size_t o = 0;
  auto take = [&](size_t b) { const size_t r = o; o = align_up(o + b, 256); return base + r; };
  const size_t f = (size_t)F, inner = f > 1 ? f - 1 : 1;
  MeshWs x;
  x.cbox = reinterpret_cast<unsigned long long*>(take(6 * 8));
  x.code[0] = reinterpret_cast<unsigned*>(take(f * 4));
  x.code[1] = reinterpret_cast<unsigned*>(take(f * 4));
  x.face[0] = reinterpret_cast<int32_t*>(take(f * 4));
  x.face[1] = reinterpret_cast<int32_t*>(take(f * 4));
  x.counts = reinterpret_cast<int*>(take((size_t)RADIX * radix_tiles(F) * 4));
  x.left = reinterpret_cast<int*>(take(inner * 4));
  x.right = reinterpret_cast<int*>(take(inner * 4));
  x.inner_parent = reinterpret_cast<int*>(take(inner * 4));
  x.leaf_parent = reinterpret_cast<int*>(take(f * 4));
  x.arrive = reinterpret_cast<int*>(take(inner * 4));
  x.inner_box = reinterpret_cast<Box*>(take(inner * sizeof(Box)));
  x.leaf_box = reinterpret_cast<Box*>(take(f * sizeof(Box)));
  x.tri = reinterpret_cast<double*>(take(f * 9 * 8));
  x.leaf_face = reinterpret_cast<int32_t*>(take(f * 4));
  if (w) *w = x;
  return o;
}

__device__ __forceinline__ unsigned long long ord_key(double v) {       // unsigned key with the order of the doubles
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | (1ull << 63));
}
__device__ __forceinline__ double ord_val(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & ~(1ull << 63)) : ~k));
}

__device__ __forceinline__ bool face_verts(const double* __restrict__ vtx, int64_t V, const int32_t* __restrict__ faces, int64_t f,
                                           V3* a, V3* b, V3* c) {
  const int32_t i = faces[3 * f], j = faces[3 * f + 1], k = faces[3 * f + 2];
  if (i < 0 || i >= V || j < 0 || j >= V || k < 0 || k >= V) return false;
  *a = V3{vtx[3 * (int64_t)i], vtx[3 * (int64_t)i + 1], vtx[3 * (int64_t)i + 2]};
  *b = V3{vtx[3 * (int64_t)j], vtx[3 * (int64_t)j + 1], vtx[3 * (int64_t)j + 2]};
  *c = V3{vtx[3 * (int64_t)k], vtx[3 * (int64_t)k + 1], vtx[3 * (int64_t)k + 2]};
  return true;
}

__device__ __forceinline__ V3 centroid(V3 a, V3 b, V3 c) { return vdiv(vadd(vadd(a, b), c), 3.0); }

// ---------------------------------------------------------------------------------------------------- per-face distance
__device__ __forceinline__ double dist2(V3 p, V3 q) {
  const double dx = p.x - q.x, dy = p.y - q.y, dz = p.z - q.z;
  return ((dx * dx) + (dy * dy)) + (dz * dz);
}

// closest point of segment ab: t = ((p-a).e) / (e.e) with e = b - a (t = 0 when e.e == 0), clamped to [0, 1]; a + e*t
__device__ __forceinline__ V3 seg_closest(V3 a, V3 b, V3 p) {
  const V3 e = vsub(b, a);
  const double ee = vdot(e, e);
  double t = ee > 0.0 ? vdot(vsub(p, a), e) / ee : 0.0;
  t = t < 0.0 ? 0.0 : (t > 1.0 ? 1.0 : t);
  return vadd(a, vmul(e, t));
}

__device__ __forceinline__ double clampd(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }

// D(p, f): q = point_tri(a, b, c, p) (geom.cuh); when a coordinate of q is not finite (the 0/0 of a degenerate face) q is
// instead the closest of the three segment points ab, bc, ca (seg_closest; the first of equal distances).  q is then
// clamped coordinate-wise into the face's box [min, max of the vertex coordinates] and D = ((dx*dx)+(dy*dy))+(dz*dz).
// The exact closest point lies in that box, so the clamp only moves q towards it (by a few ulp on a well-shaped face).
__device__ __forceinline__ double face_dist2(V3 a, V3 b, V3 c, V3 p) {
  V3 q = point_tri(a, b, c, p);
  if (!(isfinite(q.x) && isfinite(q.y) && isfinite(q.z))) {
    q = seg_closest(a, b, p);
    double d = dist2(p, q);
    const V3 q1 = seg_closest(b, c, p);
    const double d1 = dist2(p, q1);
    if (d1 < d) { q = q1; d = d1; }
    const V3 q2 = seg_closest(c, a, p);
    if (dist2(p, q2) < d) q = q2;
  }
  q.x = clampd(q.x, fmin(fmin(a.x, b.x), c.x), fmax(fmax(a.x, b.x), c.x));
  q.y = clampd(q.y, fmin(fmin(a.y, b.y), c.y), fmax(fmax(a.y, b.y), c.y));
  q.z = clampd(q.z, fmin(fmin(a.z, b.z), c.z), fmax(fmax(a.z, b.z), c.z));
  return dist2(p, q);
}

// Pruning soundness.  For a box [lo, hi] the bound is B = ((gx*gx)+(gy*gy))+(gz*gz) with gx = lo.x - p.x when p.x < lo.x,
// p.x - hi.x when p.x > hi.x, else 0 (each operation rounded, as in D).  Every face below a node has its clamped q inside
// its own box, which lies inside the node's box.  When p.x < lo.x <= q.x, |dx| = fl(q.x - p.x) >= fl(lo.x - p.x) = gx
// because rounding to nearest is monotone and odd; the case p.x > hi.x is the mirror image and gx = 0 otherwise.  Squares
// of non-negative values and sums are monotone under rounding too, so B <= D for every such face, with no slack at all.
// (A margin instead of the clamp would not be sound: on a near-degenerate face the barycentric branch divides by a
// va + vb + vc that can be tiny, and the unclamped point can land arbitrarily far outside the face's box.)  A node is
// pruned only when B > best, so no face with D <= best -- ties included -- is ever skipped.
__device__ __forceinline__ double box_bound(const Box& b, V3 p) {
  const double gx = p.x < b.lo[0] ? b.lo[0] - p.x : (p.x > b.hi[0] ? p.x - b.hi[0] : 0.0);
  const double gy = p.y < b.lo[1] ? b.lo[1] - p.y : (p.y > b.hi[1] ? p.y - b.hi[1] : 0.0);
  const double gz = p.z < b.lo[2] ? b.lo[2] - p.z : (p.z > b.hi[2] ? p.z - b.hi[2] : 0.0);
  return ((gx * gx) + (gy * gy)) + (gz * gz);
}

// ---------------------------------------------------------------------------------------------------- keys
__global__ void mesh_centroid_box_kernel(const double* __restrict__ vtx, int64_t V, const int32_t* __restrict__ faces, int64_t F,
                                         MeshWs w) {
  const int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (f >= F) return;
  V3 a, b, c;
  if (!face_verts(vtx, V, faces, f, &a, &b, &c)) return;
  const V3 m = centroid(a, b, c);
  const double v[3] = {m.x, m.y, m.z};
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const unsigned long long k = ord_key(v[d]);
    if (k < w.cbox[d]) atomicMin(&w.cbox[d], k);
    if (k > w.cbox[3 + d]) atomicMax(&w.cbox[3 + d], k);
  }
}

__device__ __forceinline__ unsigned spread10(unsigned x) {      // 10 bits -> every third bit of 30
  x &= 0x3ffu;
  x = (x | (x << 16)) & 0x030000ffu;
  x = (x | (x << 8)) & 0x0300f00fu;
  x = (x | (x << 4)) & 0x030c30c3u;
  x = (x | (x << 2)) & 0x09249249u;
  return x;
}

__device__ __forceinline__ unsigned quant10(double v, double lo, double hi) {    // NaN and out-of-box values clamp
  const double t = (v - lo) / (hi - lo) * 1023.0;
  return t > 0.0 ? (t < 1023.0 ? (unsigned)t : 1023u) : 0u;
}

__global__ void mesh_morton_kernel(const double* __restrict__ vtx, int64_t V, const int32_t* __restrict__ faces, int64_t F,
                                   MeshWs w) {
  const int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (f >= F) return;
  unsigned code = 0;
  V3 a, b, c;
  if (face_verts(vtx, V, faces, f, &a, &b, &c)) {
    const V3 m = centroid(a, b, c);
    code = (spread10(quant10(m.x, ord_val(w.cbox[0]), ord_val(w.cbox[3]))) << 2) |
           (spread10(quant10(m.y, ord_val(w.cbox[1]), ord_val(w.cbox[4]))) << 1) |
           spread10(quant10(m.z, ord_val(w.cbox[2]), ord_val(w.cbox[5])));
  }
  w.code[0][f] = code;
  w.face[0][f] = (int32_t)f;
}

// ---------------------------------------------------------------------------------------------------- stable LSD radix sort
// Tile b (RADIX_TILE keys) is owned by block b; thread t owns its RADIX_ITEMS consecutive keys.  counts[d * nb + b] = keys of
// tile b with digit d; its exclusive scan (digit-major) is each (digit, tile) pair's first output slot.
__global__ void __launch_bounds__(MD_THREADS) mesh_radix_count_kernel(const unsigned* __restrict__ code, int64_t F, int shift,
                                                                      int* __restrict__ counts, int nb) {
  __shared__ int h[RADIX];
  if (threadIdx.x < RADIX) h[threadIdx.x] = 0;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * RADIX_TILE + (int64_t)threadIdx.x * RADIX_ITEMS;
#pragma unroll
  for (int k = 0; k < RADIX_ITEMS; ++k)
    if (base + k < F) atomicAdd(&h[(code[base + k] >> shift) & (RADIX - 1)], 1);
  __syncthreads();
  if (threadIdx.x < RADIX) counts[threadIdx.x * nb + blockIdx.x] = h[threadIdx.x];
}

// in-place exclusive scan of n ints by one block of 1024 threads, serial over chunks (as seedgen.cu's scan_sums_kernel)
__global__ void __launch_bounds__(1024) mesh_radix_scan_kernel(int* __restrict__ a, int n) {
  __shared__ int ws[32];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int b0 = 0; b0 < n; b0 += blockDim.x) {
    const int i = b0 + threadIdx.x;
    const int v = i < n ? a[i] : 0;
    int inc = v;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) ws[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      int x = ws[lane];
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += t; }
      ws[lane] = x;
    }
    __syncthreads();
    const int excl = inc - v + (warp ? ws[warp - 1] : 0) + carry;
    if (i < n) a[i] = excl;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = excl + v;
    __syncthreads();
  }
}

// Stable scatter: local[d * MD_THREADS + t] = keys of digit d held by threads < t of this tile (plus, before the scan, the
// thread's own count); a key's slot = offs[d * nb + b] + local rank of its digit in tile order.
__global__ void __launch_bounds__(MD_THREADS) mesh_radix_scatter_kernel(const unsigned* __restrict__ code_in,
                                                                        const int32_t* __restrict__ face_in,
                                                                        unsigned* __restrict__ code_out,
                                                                        int32_t* __restrict__ face_out, int64_t F, int shift,
                                                                        const int* __restrict__ offs, int nb) {
  constexpr int PER = RADIX * MD_THREADS / MD_THREADS;          // scan entries per thread (= RADIX)
  __shared__ int local[RADIX * MD_THREADS];
  __shared__ int wsum[MD_THREADS / 32];
  __shared__ int first[RADIX];
  const int t = threadIdx.x;
  const int64_t base = (int64_t)blockIdx.x * RADIX_TILE + (int64_t)t * RADIX_ITEMS;
  for (int e = t; e < RADIX * MD_THREADS; e += MD_THREADS) local[e] = 0;
  __syncthreads();
  unsigned key[RADIX_ITEMS];
  int fc[RADIX_ITEMS];
#pragma unroll
  for (int k = 0; k < RADIX_ITEMS; ++k) {
    const bool in = base + k < F;
    key[k] = in ? code_in[base + k] : 0u;
    fc[k] = in ? face_in[base + k] : 0;
    if (in) ++local[((key[k] >> shift) & (RADIX - 1)) * MD_THREADS + t];     // only thread t touches column t
  }
  __syncthreads();
  // exclusive scan of local[] (digit-major): thread t owns entries [t * PER, (t + 1) * PER)
  int v[PER], tot = 0;
#pragma unroll
  for (int k = 0; k < PER; ++k) { v[k] = local[t * PER + k]; tot += v[k]; }
  const int lane = t & 31, warp = t >> 5;
  int inc = tot;
  for (int o = 1; o < 32; o <<= 1) { const int x = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += x; }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int x = lane < MD_THREADS / 32 ? wsum[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane < MD_THREADS / 32) wsum[lane] = x;
  }
  __syncthreads();
  int run = inc - tot + (warp ? wsum[warp - 1] : 0);
#pragma unroll
  for (int k = 0; k < PER; ++k) { local[t * PER + k] = run; run += v[k]; }
  __syncthreads();
  if (t < RADIX) first[t] = local[t * MD_THREADS];
  __syncthreads();
#pragma unroll
  for (int k = 0; k < RADIX_ITEMS; ++k) {
    if (base + k >= F) break;
    const int d = (key[k] >> shift) & (RADIX - 1);
    const int64_t o = (int64_t)offs[d * nb + blockIdx.x] + (local[d * MD_THREADS + t]++ - first[d]);
    code_out[o] = key[k];
    face_out[o] = fc[k];
  }
}

// ---------------------------------------------------------------------------------------------------- tree
__device__ __forceinline__ unsigned long long leaf_key(const MeshWs& w, int64_t i) {
  return ((unsigned long long)w.code[0][i] << 32) | (unsigned)w.face[0][i];
}
__device__ __forceinline__ int delta(const MeshWs& w, int64_t F, int64_t i, unsigned long long ki, int64_t j) {
  if (j < 0 || j >= F) return -1;
  return __clzll(ki ^ leaf_key(w, j));
}

// Karras 2012, Figure 4: the range [min(i, j), max(i, j)] of internal node i and its split gamma
__global__ void mesh_karras_kernel(int64_t F, MeshWs w) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= F - 1) return;
  const unsigned long long ki = leaf_key(w, i);
  const int d = delta(w, F, i, ki, i + 1) > delta(w, F, i, ki, i - 1) ? 1 : -1;
  const int dmin = delta(w, F, i, ki, i - d);
  int64_t lmax = 2;
  while (delta(w, F, i, ki, i + lmax * d) > dmin) lmax *= 2;
  int64_t l = 0;
  for (int64_t t = lmax / 2; t >= 1; t /= 2)
    if (delta(w, F, i, ki, i + (l + t) * d) > dmin) l += t;
  const int64_t j = i + l * d;
  const int dnode = delta(w, F, i, ki, j);
  int64_t s = 0, t = l;
  do {
    t = (t + 1) / 2;
    if (delta(w, F, i, ki, i + (s + t) * d) > dnode) s += t;
  } while (t > 1);
  const int64_t g = i + s * d + (d < 0 ? -1 : 0);
  const int64_t lo = i < j ? i : j, hi = i < j ? j : i;
  const int L = lo == g ? ~(int)g : (int)g, R = hi == g + 1 ? ~(int)(g + 1) : (int)(g + 1);
  w.left[i] = L;
  w.right[i] = R;
  (L < 0 ? w.leaf_parent[~L] : w.inner_parent[L]) = (int)i;
  (R < 0 ? w.leaf_parent[~R] : w.inner_parent[R]) = (int)i;
  if (i == 0) w.inner_parent[0] = -1;
}

__device__ __forceinline__ Box ldcg_box(const MeshWs& w, int c) {
  const Box* p = c < 0 ? &w.leaf_box[~c] : &w.inner_box[c];
  Box b;
#pragma unroll
  for (int d = 0; d < 3; ++d) { b.lo[d] = __ldcg(&p->lo[d]); b.hi[d] = __ldcg(&p->hi[d]); }
  return b;
}

// leaves: the sorted face's triangle and box; then up the tree, the second child to arrive at a node fits its box
__global__ void mesh_fit_kernel(const double* __restrict__ vtx, int64_t V, const int32_t* __restrict__ faces, int64_t F, MeshWs w) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= F) return;
  const int32_t f = w.face[0][i];
  V3 a, b, c;
  Box bx;
  if (face_verts(vtx, V, faces, f, &a, &b, &c)) {
    const double t[9] = {a.x, a.y, a.z, b.x, b.y, b.z, c.x, c.y, c.z};
#pragma unroll
    for (int k = 0; k < 9; ++k) w.tri[9 * i + k] = t[k];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      bx.lo[d] = fmin(fmin(t[d], t[3 + d]), t[6 + d]);
      bx.hi[d] = fmax(fmax(t[d], t[3 + d]), t[6 + d]);
    }
    w.leaf_face[i] = f;
  } else {                                                  // skipped face: an empty box, never tested
#pragma unroll
    for (int d = 0; d < 3; ++d) { bx.lo[d] = INFINITY; bx.hi[d] = -INFINITY; }
    w.leaf_face[i] = -1;
  }
  w.leaf_box[i] = bx;
  if (F == 1) return;
  for (int p = w.leaf_parent[i]; p >= 0; p = w.inner_parent[p]) {
    __threadfence();
    if (atomicAdd(&w.arrive[p], 1) == 0) return;           // the sibling's box is not written yet: it fits the parent
    __threadfence();
    const Box l = ldcg_box(w, w.left[p]), r = ldcg_box(w, w.right[p]);
#pragma unroll
    for (int d = 0; d < 3; ++d) { bx.lo[d] = fmin(l.lo[d], r.lo[d]); bx.hi[d] = fmax(l.hi[d], r.hi[d]); }
    w.inner_box[p] = bx;
  }
}

#ifdef SAPCU_MESH_COUNTERS
__device__ unsigned long long g_mesh_counts[2];       // nodes whose box bound was computed, point-triangle tests
#endif

// ---------------------------------------------------------------------------------------------------- query
__device__ __forceinline__ void test_leaf(const MeshWs& w, int64_t leaf, V3 p, double* best, int* bf, unsigned long long* ntests) {
  const int f = w.leaf_face[leaf];
  if (f < 0) return;
  const double* t = w.tri + 9 * leaf;
  const double D = face_dist2(V3{t[0], t[1], t[2]}, V3{t[3], t[4], t[5]}, V3{t[6], t[7], t[8]}, p);
  ++*ntests;
  if (D < *best || (D == *best && f < *bf)) { *best = D; *bf = f; }
}

__global__ void __launch_bounds__(MD_QUERY_THREADS) mesh_query_kernel(const double* __restrict__ pts, int64_t S, int64_t F, MeshWs w,
                                                                      double* __restrict__ dist2_out, int32_t* __restrict__ face_out) {
  const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (s >= S) return;
  const V3 p{pts[3 * s], pts[3 * s + 1], pts[3 * s + 2]};
  double best = INFINITY;
  int bf = 0x7fffffff;
  unsigned long long nodes = 0, tests = 0;
  if (F == 1) {
    test_leaf(w, 0, p, &best, &bf, &tests);
  } else {
    int stack_node[MD_STACK];
    double stack_bound[MD_STACK];
    int sp = 0;
    int node = 0;
    while (true) {
      if (node < 0) {
        test_leaf(w, ~node, p, &best, &bf, &tests);
      } else {
        const int l = w.left[node], r = w.right[node];
        const double bl = box_bound(l < 0 ? w.leaf_box[~l] : w.inner_box[l], p);
        const double br = box_bound(r < 0 ? w.leaf_box[~r] : w.inner_box[r], p);
        nodes += 2;
        const bool lnear = bl <= br;
        const int nn = lnear ? l : r, fn = lnear ? r : l;
        const double bn = lnear ? bl : br, bfar = lnear ? br : bl;
        if (!(bfar > best)) { stack_node[sp] = fn; stack_bound[sp] = bfar; ++sp; }
        if (!(bn > best)) { node = nn; continue; }
      }
      bool more = false;
      while (sp > 0) {
        --sp;
        if (!(stack_bound[sp] > best)) { node = stack_node[sp]; more = true; break; }
      }
      if (!more) break;
    }
  }
  dist2_out[s] = best;
  if (face_out) face_out[s] = bf == 0x7fffffff ? -1 : bf;
#ifdef SAPCU_MESH_COUNTERS
  atomicAdd(&g_mesh_counts[0], nodes);
  atomicAdd(&g_mesh_counts[1], tests);
#else
  (void)nodes;
#endif
}

static bool mesh_limits(int64_t V, int64_t F) { return V >= 1 && F >= 1 && F < ((int64_t)1 << 31); }

}  // namespace sapcu

using namespace sapcu;

extern "C" {

size_t sapcu_mesh_distance_workspace_bytes(int64_t V, int64_t F) {
  if (!mesh_limits(V, F)) return 0;
  return mesh_bytes(F, nullptr, nullptr);
}

int sapcu_mesh_distance(const double* d_vertices, int64_t V, const int32_t* d_faces, int64_t F, const double* d_points, int64_t S,
                        double* d_dist2, int32_t* d_face, void* d_ws, size_t ws_bytes, void* stream) {
  SAPCU_REQUIRE(mesh_limits(V, F), "mesh_distance: V=%lld, F=%lld outside V >= 1, 1 <= F < 2^31", (long long)V, (long long)F);
  SAPCU_REQUIRE(S >= 0, "mesh_distance: S=%lld < 0", (long long)S);
  if (S == 0) return 0;
  SAPCU_REQUIRE(d_vertices && d_faces && d_points && d_dist2 && d_ws, "mesh_distance: null pointer");
  const size_t need = mesh_bytes(F, nullptr, nullptr);
  if (ws_bytes < need) {
    set_error("mesh_distance: workspace of %zu bytes, %zu needed", ws_bytes, need);
    return SAPCU_EWORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  MeshWs w;
  mesh_bytes(F, &w, reinterpret_cast<char*>(d_ws));
  const unsigned fb = (unsigned)ceil_div(F, MD_THREADS);
  const int nb = (int)radix_tiles(F);
  // build
  SAPCU_CUDA_CHECK(cudaMemsetAsync(w.cbox, 0xff, 3 * 8, st));
  SAPCU_CUDA_CHECK(cudaMemsetAsync(w.cbox + 3, 0, 3 * 8, st));
  if (F > 1) SAPCU_CUDA_CHECK(cudaMemsetAsync(w.arrive, 0, (size_t)(F - 1) * 4, st));
  mesh_centroid_box_kernel<<<fb, MD_THREADS, 0, st>>>(d_vertices, V, d_faces, F, w);
  SAPCU_LAUNCH_CHECK();
  mesh_morton_kernel<<<fb, MD_THREADS, 0, st>>>(d_vertices, V, d_faces, F, w);
  SAPCU_LAUNCH_CHECK();
  for (int pass = 0; pass < RADIX_PASSES; ++pass) {
    const int in = pass & 1, shift = pass * RADIX_BITS;
    mesh_radix_count_kernel<<<nb, MD_THREADS, 0, st>>>(w.code[in], F, shift, w.counts, nb);
    SAPCU_LAUNCH_CHECK();
    mesh_radix_scan_kernel<<<1, 1024, 0, st>>>(w.counts, RADIX * nb);
    SAPCU_LAUNCH_CHECK();
    mesh_radix_scatter_kernel<<<nb, MD_THREADS, 0, st>>>(w.code[in], w.face[in], w.code[in ^ 1], w.face[in ^ 1], F, shift, w.counts, nb);
    SAPCU_LAUNCH_CHECK();
  }
  if (F > 1) {
    mesh_karras_kernel<<<(unsigned)ceil_div(F - 1, MD_THREADS), MD_THREADS, 0, st>>>(F, w);
    SAPCU_LAUNCH_CHECK();
  }
  mesh_fit_kernel<<<fb, MD_THREADS, 0, st>>>(d_vertices, V, d_faces, F, w);
  SAPCU_LAUNCH_CHECK();
  // query
  mesh_query_kernel<<<(unsigned)ceil_div(S, MD_QUERY_THREADS), MD_QUERY_THREADS, 0, st>>>(d_points, S, F, w, d_dist2, d_face);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

#ifdef SAPCU_MESH_COUNTERS
// work counters of the instrumented build (tools/metrics_bench.py): reset, or read {nodes bounded, point-triangle tests}
int sapcu_mesh_counters(unsigned long long* h_counts, int reset) {
  if (reset) {
    const unsigned long long z[2] = {0, 0};
    SAPCU_CUDA_CHECK(cudaMemcpyToSymbol(g_mesh_counts, z, sizeof(z)));
  }
  if (h_counts) SAPCU_CUDA_CHECK(cudaMemcpyFromSymbol(h_counts, g_mesh_counts, 2 * sizeof(unsigned long long)));
  return 0;
}
#endif

}  // extern "C"
