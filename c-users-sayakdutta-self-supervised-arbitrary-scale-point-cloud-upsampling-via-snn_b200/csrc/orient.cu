// Consistent normal orientation over a kNN graph (the Hoppe et al. spanning-tree propagation) on the device.
//   graph   edges {i, idx[i*k + j]} of the self-kNN, self entries skipped; one fp64 dot per directed entry, computed once
//   forest  Boruvka rounds under the strict edge order (larger |dot|, then the smaller (min, max) pair): every component
//           picks its best outgoing edge with two atomic passes (max of |dot|'s bits, then min of the packed pair among
//           the ties), hooks onto its partner (a mutual pair keeps the lower id as the root) and the hook forest is
//           compressed by synchronous pointer jumping: each step reads one buffer and writes the other, so no kernel
//           reads a word another thread of it writes, and at most ceil(log2 S) + 1 steps run.  Each vertex carries the
//           parity of flip edges (dot < 0) on its tree path to its component's representative, so the orientation needs no
//           traversal of the final tree.
//   roots   largest z (ordered 64-bit key), then the lowest index, with the same two-pass pattern
// At most ceil(log2 S) + 1 rounds are enqueued; a per-round device flag ends the work once a round merged nothing, and a
// per-step flag ends a round's pointer jumping once no pointer moved, so nothing waits on the host.  Every loop is bounded
// and every graph entry outside [0, S) is skipped, so no input can make a kernel run unbounded or read outside its
// arrays.  Every pass is a flat grid over the S*k entries or the S vertices (L2-resident state).
#include "../../include/sapcu_b200.h"
#include "common.cuh"

namespace sapcu {

constexpr int ORIENT_THREADS = 256;
constexpr int ORIENT_KMAX = 128;
constexpr unsigned long long NO_EDGE = ~0ull;

// (parity << 32) | id: a vertex's component and its parity relative to it, or a representative's hook target and the
// parity relative to that target.  One 64-bit word, so a reader never sees one half of an update.
__device__ __forceinline__ unsigned long long pack(unsigned par, unsigned id) { return ((unsigned long long)par << 32) | id; }
__device__ __forceinline__ unsigned id_of(unsigned long long w) { return (unsigned)w; }
__device__ __forceinline__ unsigned par_of(unsigned long long w) { return (unsigned)(w >> 32); }

// ((nx_i*nx_j) + (ny_i*ny_j)) + nz_i*nz_j in fp64 from the fp32 components, no contraction
__device__ __forceinline__ double normal_dot(const float* __restrict__ n, int64_t i, int64_t j) {
  return __dadd_rn(__dadd_rn(__dmul_rn((double)n[3 * i], (double)n[3 * j]), __dmul_rn((double)n[3 * i + 1], (double)n[3 * j + 1])),
                   __dmul_rn((double)n[3 * i + 2], (double)n[3 * j + 2]));
}

struct OrientWs {
  double* dot;                  // [S*k] dot of every directed entry
  unsigned long long* vert;     // [S]   pack(parity to component, component)
  unsigned long long* hook[2];  // [2][S] per representative: pack(parity to target, target); pointer-jumping ping-pong
  unsigned long long* key;      // [S]   per component: max of the primary key (|dot| bits; later z key)
  unsigned long long* arg;      // [S]   per component: min of the tie-break (packed pair; later vertex index)
  unsigned* root_neg;           // [S]   per component: the root's sign relative to the representative
  int* active;                  // [rounds + 1] round r runs when active[r] != 0
  int* moved;                   // [rounds][rounds] jump step j of round r runs when j == 0 or moved[r][j - 1] != 0
};

static int orient_rounds(int64_t S) {
  int r = 0;
  while (((int64_t)1 << r) < S) ++r;
  return r + 1;
}

static OrientWs orient_carve(void* ws, int64_t S, int k) {
  char* p = reinterpret_cast<char*>(ws);
  OrientWs w;
  w.dot = reinterpret_cast<double*>(p);                   p += align_up((size_t)S * k * 8, 256);
  w.vert = reinterpret_cast<unsigned long long*>(p);      p += align_up((size_t)S * 8, 256);
  w.hook[0] = reinterpret_cast<unsigned long long*>(p);   p += align_up((size_t)S * 8, 256);
  w.hook[1] = reinterpret_cast<unsigned long long*>(p);   p += align_up((size_t)S * 8, 256);
  w.key = reinterpret_cast<unsigned long long*>(p);       p += align_up((size_t)S * 8, 256);
  w.arg = reinterpret_cast<unsigned long long*>(p);       p += align_up((size_t)S * 8, 256);
  w.root_neg = reinterpret_cast<unsigned*>(p);            p += align_up((size_t)S * 4, 256);
  w.active = reinterpret_cast<int*>(p);                   p += align_up((size_t)(orient_rounds(S) + 1) * 4, 256);
  w.moved = reinterpret_cast<int*>(p);
  return w;
}

static size_t orient_bytes(int64_t S, int k) {
  const size_t r = (size_t)orient_rounds(S);
  return align_up((size_t)S * k * 8, 256) + 5 * align_up((size_t)S * 8, 256) + align_up((size_t)S * 4, 256) +
         align_up((r + 1) * 4, 256) + align_up(r * r * 4, 256);
}

__global__ void orient_init_kernel(const float* __restrict__ n, const int32_t* __restrict__ idx, int64_t S, int k, OrientWs w,
                                   int rounds) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < S * k) {
    const int64_t j = idx[e];
    w.dot[e] = j >= 0 && j < S ? normal_dot(n, e / k, j) : 0.0;       // out-of-range entries are skipped by every pass
  }
  if (e < S) {
    w.vert[e] = pack(0u, (unsigned)e);
    w.key[e] = 0ull;
    w.arg[e] = NO_EDGE;
  }
  if (e <= rounds) w.active[e] = e == 0;
  if (e < (int64_t)rounds * rounds) w.moved[e] = 0;
}

// pass 1 of a round: the largest |dot| leaving each component (non-negative doubles order like their bit patterns)
__global__ void orient_best_weight_kernel(const int32_t* __restrict__ idx, int64_t S, int k, OrientWs w, int round) {
  if (!w.active[round]) return;
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= S * k) return;
  const int64_t i = e / k, j = idx[e];
  if (j == i || j < 0 || j >= S) return;
  const unsigned ci = id_of(w.vert[i]), cj = id_of(w.vert[j]);
  if (ci == cj) return;
  const unsigned long long b = (unsigned long long)__double_as_longlong(fabs(w.dot[e]));
  if (b > w.key[ci]) atomicMax(&w.key[ci], b);
  if (b > w.key[cj]) atomicMax(&w.key[cj], b);
}

// pass 2: among the edges of that weight, the smallest (min, max) pair
__global__ void orient_best_pair_kernel(const int32_t* __restrict__ idx, int64_t S, int k, OrientWs w, int round) {
  if (!w.active[round]) return;
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= S * k) return;
  const int64_t i = e / k, j = idx[e];
  if (j == i || j < 0 || j >= S) return;
  const unsigned ci = id_of(w.vert[i]), cj = id_of(w.vert[j]);
  if (ci == cj) return;
  const unsigned long long b = (unsigned long long)__double_as_longlong(fabs(w.dot[e]));
  const unsigned long long pr = i < j ? pack((unsigned)i, (unsigned)j) : pack((unsigned)j, (unsigned)i);
  if (b == w.key[ci] && pr < w.arg[ci]) atomicMin(&w.arg[ci], pr);
  if (b == w.key[cj] && pr < w.arg[cj]) atomicMin(&w.arg[cj], pr);
}

// every representative hooks onto the component across its best edge; of a mutual pair the lower id stays the root
__global__ void orient_hook_kernel(const float* __restrict__ n, int64_t S, OrientWs w, int round) {
  if (!w.active[round]) return;
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= S || id_of(w.vert[c]) != (unsigned)c) return;
  const unsigned long long best = w.arg[c];
  unsigned long long h = pack(0u, (unsigned)c);
  if (best != NO_EDGE) {
    const unsigned a = (unsigned)(best >> 32), b = (unsigned)best;
    const unsigned long long va = w.vert[a], vb = w.vert[b];
    const unsigned p = id_of(va) == (unsigned)c ? id_of(vb) : id_of(va);
    if (!(w.arg[p] == best && (unsigned)c < p)) {
      const unsigned flip = normal_dot(n, a, b) < 0.0 ? 1u : 0u;
      h = pack(flip ^ par_of(va) ^ par_of(vb), p);
      w.active[round + 1] = 1;
    }
  }
  w.hook[0][c] = h;
}

// one synchronous pointer-jumping step over the hook forest, XOR-accumulating the parity: hook[j & 1] -> hook[~j & 1].
// A step that moves no pointer leaves both buffers equal on every representative and ends the round's jumping.
__global__ void orient_jump_kernel(int64_t S, OrientWs w, int round, int step, int rounds) {
  if (!w.active[round] || (step > 0 && !w.moved[round * rounds + step - 1])) return;
  const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= S || id_of(w.vert[c]) != (unsigned)c) return;
  const unsigned long long* in = (step & 1) ? w.hook[1] : w.hook[0];
  const unsigned long long h = in[c], hp = in[id_of(h)];
  unsigned long long out = h;
  if (id_of(hp) != id_of(h)) {
    out = pack(par_of(h) ^ par_of(hp), id_of(hp));
    w.moved[round * rounds + step] = 1;
  }
  ((step & 1) ? w.hook[0] : w.hook[1])[c] = out;
}

// every vertex moves to its new representative; the per-component best-edge state is cleared for the next round
__global__ void orient_relabel_kernel(int64_t S, OrientWs w, int round, int rounds) {
  if (!w.active[round]) return;
  const int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (v >= S) return;
  const unsigned long long x = w.vert[v], h = ((rounds & 1) ? w.hook[1] : w.hook[0])[id_of(x)];     // the output of the last jump step
  w.vert[v] = pack(par_of(x) ^ par_of(h), id_of(h));
  w.key[v] = 0ull;
  w.arg[v] = NO_EDGE;
}

// z as an unsigned key with the order of the doubles (-0.0 counts as +0.0)
__device__ __forceinline__ unsigned long long z_key(const double* __restrict__ pts, int64_t v) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(__dadd_rn(pts[3 * v + 2], 0.0));
  return (b >> 63) ? ~b : (b | (1ull << 63));
}

__global__ void orient_root_z_kernel(const double* __restrict__ pts, int64_t S, OrientWs w) {
  const int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (v >= S) return;
  atomicMax(&w.key[id_of(w.vert[v])], z_key(pts, v));
}

__global__ void orient_root_index_kernel(const double* __restrict__ pts, int64_t S, OrientWs w) {
  const int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (v >= S) return;
  const unsigned c = id_of(w.vert[v]);
  if (z_key(pts, v) == w.key[c]) atomicMin(&w.arg[c], (unsigned long long)v);
}

// the root's sign relative to the representative: negated when its nz < 0, XOR its own parity
__global__ void orient_root_sign_kernel(const float* __restrict__ n, int64_t S, OrientWs w) {
  const int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (v >= S) return;
  const unsigned long long x = w.vert[v];
  if (w.arg[id_of(x)] == (unsigned long long)v) w.root_neg[id_of(x)] = (n[3 * v + 2] < 0.f ? 1u : 0u) ^ par_of(x);
}

__global__ void orient_apply_kernel(float* __restrict__ n, int64_t S, OrientWs w, int32_t* __restrict__ root) {
  const int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (v >= S) return;
  const unsigned long long x = w.vert[v];
  if (w.root_neg[id_of(x)] ^ par_of(x)) {
#pragma unroll
    for (int d = 0; d < 3; ++d) n[3 * v + d] = __int_as_float(__float_as_int(n[3 * v + d]) ^ (int)0x80000000);
  }
  if (root) root[v] = (int32_t)w.arg[id_of(x)];
}

}  // namespace sapcu

using namespace sapcu;

extern "C" {

size_t sapcu_orient_normals_workspace_bytes(int64_t S, int k) {
  if (S < 1 || k < 1 || k > ORIENT_KMAX || S * k >= ((int64_t)1 << 31)) return 0;
  return orient_bytes(S, k);
}

int sapcu_orient_normals(const double* d_points, int64_t S, const int32_t* d_idx, int k, float* d_normals, int32_t* d_root,
                         void* d_ws, size_t ws_bytes, void* stream) {
  SAPCU_REQUIRE(k >= 1 && k <= ORIENT_KMAX, "orient_normals: k=%d outside [1,%d]", k, ORIENT_KMAX);
  SAPCU_REQUIRE(S >= 1 && S * k < ((int64_t)1 << 31), "orient_normals: S=%lld with k=%d outside 1 <= S, S*k < 2^31",
                (long long)S, k);
  SAPCU_REQUIRE(d_points && d_idx && d_normals && d_ws, "orient_normals: null pointer");
  if (ws_bytes < orient_bytes(S, k)) {
    set_error("orient_normals: workspace of %zu bytes, %zu needed", ws_bytes, orient_bytes(S, k));
    return SAPCU_EWORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const OrientWs w = orient_carve(d_ws, S, k);
  const int rounds = orient_rounds(S);
  const unsigned eb = (unsigned)ceil_div(S * k, ORIENT_THREADS), vb = (unsigned)ceil_div(S, ORIENT_THREADS);
  const unsigned ib = (unsigned)ceil_div(S * k > (int64_t)rounds * rounds ? S * k : (int64_t)rounds * rounds + 1, ORIENT_THREADS);
  orient_init_kernel<<<ib, ORIENT_THREADS, 0, st>>>(d_normals, d_idx, S, k, w, rounds);
  SAPCU_LAUNCH_CHECK();
  for (int r = 0; r < rounds; ++r) {
    orient_best_weight_kernel<<<eb, ORIENT_THREADS, 0, st>>>(d_idx, S, k, w, r);
    SAPCU_LAUNCH_CHECK();
    orient_best_pair_kernel<<<eb, ORIENT_THREADS, 0, st>>>(d_idx, S, k, w, r);
    SAPCU_LAUNCH_CHECK();
    orient_hook_kernel<<<vb, ORIENT_THREADS, 0, st>>>(d_normals, S, w, r);
    SAPCU_LAUNCH_CHECK();
    for (int j = 0; j < rounds; ++j) {        // a hook chain is shorter than S, so ceil(log2 S) steps reach every root
      orient_jump_kernel<<<vb, ORIENT_THREADS, 0, st>>>(S, w, r, j, rounds);
      SAPCU_LAUNCH_CHECK();
    }
    orient_relabel_kernel<<<vb, ORIENT_THREADS, 0, st>>>(S, w, r, rounds);
    SAPCU_LAUNCH_CHECK();
  }
  orient_root_z_kernel<<<vb, ORIENT_THREADS, 0, st>>>(d_points, S, w);
  SAPCU_LAUNCH_CHECK();
  orient_root_index_kernel<<<vb, ORIENT_THREADS, 0, st>>>(d_points, S, w);
  SAPCU_LAUNCH_CHECK();
  orient_root_sign_kernel<<<vb, ORIENT_THREADS, 0, st>>>(d_normals, S, w);
  SAPCU_LAUNCH_CHECK();
  orient_apply_kernel<<<vb, ORIENT_THREADS, 0, st>>>(d_normals, S, w, d_root);
  SAPCU_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
