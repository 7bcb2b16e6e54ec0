// Earth Mover's Distance between two clouds of n points each: the min-cost perfect matching under Euclidean costs
//   EMD(a, b) = min over permutations s of (1/n) sum_i |a_i - b_s(i)|,
// solved by Bertsekas's forward auction with eps-scaling in one cooperative persistent kernel (grid barriers, no host
// round trip).  Persons are the rows of a, objects the rows of b; c_ij = sqrt(((dx*dx)+(dy*dy))+(dz*dz)) in fp64,
// recomputed from the coordinates on every use (no n x n matrix).  This file is compiled with -fmad=false
// (_native._FILE_FLAGS), so a numpy restatement of c gives the same bits.
//   phase    at one eps, from an empty assignment and the prices of the previous phase, Jacobi rounds until every person
//            owns an object.  Each unassigned person finds the lowest v = c_ij + p_j (lowest j on ties) and the second lowest
//            value, and bids p_j1 + (v2 - v1) + eps for j1 (p + eps when n = 1).  An object goes to its highest bid, ties
//            to the lowest person; its previous owner becomes unassigned.
//   bound    after a phase, primal = sum_i c_i,s(i) and dual = sum_i min_j (c_ij + p_j) - sum_j p_j; dual <= optimum for any
//            prices.  The solve stops when primal - dual <= rel_tol * primal + n * eps_min; otherwise eps /= 5 (not below
//            eps_min) and a new phase starts.  A phase at eps_min that misses the certificate is returned unconverged.
//   order    a bid is a 128-bit key (bid bits, person) raised with a 128-bit CAS: the highest bid, then the lowest person, is
//            the winner whatever order the CASes land in.  Positive doubles order like their bits, and every bid exceeds
//            the object's price, which the key already holds, so the keys never need a reset.  Sums run over fixed
//            256-element chunks in a fixed tree, independent of the grid.  The list of bidders is appended with atomics;
//            its order only decides which warp computes which bid, never a result.
//   bounded  at most `cap` rounds in all (emd_round_cap); phases end when eps reaches eps_min.  A pair whose squared
//            distance overflows fp64 makes c_max infinite: the kernel then returns before the first round.  A bid that is
//            not finite, or a scan that finds no finite value, raises a device flag, and every thread returns after that
//            round's barrier; both leave the outputs of the last completed phase (or "no phase completed"), converged = 0.
#include <cooperative_groups.h>
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include "../../include/sapcu_b200.h"
#include "common.cuh"

namespace cg = cooperative_groups;

namespace sapcu {

constexpr int EMD_THREADS = 256;
constexpr int EMD_WARPS = EMD_THREADS / 32;
constexpr int64_t EMD_MAX_N = 131072;
constexpr int EMD_MIN_CHUNK = 128;        // fewest objects one warp scans when a bidder's scan is split
constexpr int EMD_MAX_UNITS = 16384;      // partial-result slots of split scans (bidders x pieces)
constexpr int EMD_SUM_CHUNK = 256;        // fixed summation chunk
constexpr int EMD_POINTS_PER_BLOCK = 64;  // grid size: ceil(n / 64) blocks, at most the co-resident count
constexpr double EMD_THETA = 5.0;

struct alignas(16) BidKey {
  unsigned long long bid;      // bits of a positive double
  unsigned long long person;
};

struct EmdWs {
  unsigned long long* cmax;    // [1] bits of max c_ij
  int* count;                  // [3] bidder-list lengths, rotating: read in round r, appended in r, reset in r
  int* abort;                  // [1] set when a bid cannot be placed in finite arithmetic
  BidKey* key;                 // [n] highest (bid, person) so far of every object
  double* price;               // [n] == key.bid at the start of every round
  int* kwin;                   // [n] == key.person at the start of every round (-1: ~0, no bid yet)
  int* owner;                  // [n] person owning object j, -1 none
  int* assign;                 // [n] object of person i, -1 none (the working assignment of the current phase)
  int* list[2];                // [2][n] bidders of a round, ping-pong
  double* sbid;                // [n] bid of the k-th bidder of the round
  int* sj;                     // [n] object it bid for
  int* scnt;                   // [n] pieces of the k-th bidder's split scan that have finished
  double* rowmin;              // [n] min_j (c_ij + p_j)
  double* cost;                // [n] c_i,assign(i)
  double* pv1;                 // [EMD_MAX_UNITS] partial (v1, v2, j1) of split scans
  double* pv2;
  int* pj;
  double* sums;                // [3][nch] chunk sums of cost, rowmin, price
};

struct EmdArgs {
  const double* a;
  const double* b;
  int n;
  double rel_tol;
  long long cap;
  int32_t* out_assign;
  double* out_cost;
  double* out_stats;
  EmdWs w;
};

static int64_t emd_chunks(int64_t n) { return ceil_div(n, EMD_SUM_CHUNK); }

static size_t emd_layout(int64_t n, EmdWs* w, char* base) {
  size_t o = 0;
  auto take = [&](size_t b) { const size_t r = o; o = align_up(o + b, 256); return base + r; };
  const size_t m = (size_t)n, nch = (size_t)emd_chunks(n);
  EmdWs x;
  char* hdr = take(64);
  x.cmax = reinterpret_cast<unsigned long long*>(hdr);
  x.count = reinterpret_cast<int*>(hdr + 8);
  x.abort = reinterpret_cast<int*>(hdr + 20);
  x.key = reinterpret_cast<BidKey*>(take(m * sizeof(BidKey)));
  x.price = reinterpret_cast<double*>(take(m * 8));
  x.kwin = reinterpret_cast<int*>(take(m * 4));
  x.owner = reinterpret_cast<int*>(take(m * 4));
  x.assign = reinterpret_cast<int*>(take(m * 4));
  x.list[0] = reinterpret_cast<int*>(take(m * 4));
  x.list[1] = reinterpret_cast<int*>(take(m * 4));
  x.sbid = reinterpret_cast<double*>(take(m * 8));
  x.sj = reinterpret_cast<int*>(take(m * 4));
  x.scnt = reinterpret_cast<int*>(take(m * 4));
  x.rowmin = reinterpret_cast<double*>(take(m * 8));
  x.cost = reinterpret_cast<double*>(take(m * 8));
  x.pv1 = reinterpret_cast<double*>(take((size_t)EMD_MAX_UNITS * 8));
  x.pv2 = reinterpret_cast<double*>(take((size_t)EMD_MAX_UNITS * 8));
  x.pj = reinterpret_cast<int*>(take((size_t)EMD_MAX_UNITS * 4));
  x.sums = reinterpret_cast<double*>(take(3 * nch * 8));
  if (w) *w = x;
  return o;
}

__device__ __forceinline__ double emd_cost(double ax, double ay, double az, const double* __restrict__ b, int j) {
  const double dx = __dsub_rn(ax, __ldg(b + 3 * j)), dy = __dsub_rn(ay, __ldg(b + 3 * j + 1)), dz = __dsub_rn(az, __ldg(b + 3 * j + 2));
  return __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
}

// lowest value v1 (at the lowest object index j1 among equal values) and the second lowest value v2 of a set of objects
struct Best {
  double v1, v2;
  int j1;
};

__device__ __forceinline__ Best best_merge(Best x, Best y) {
  if (y.v1 < x.v1 || (y.v1 == x.v1 && y.j1 < x.j1)) { y.v2 = fmin(y.v2, x.v1); return y; }
  x.v2 = fmin(x.v2, y.v1);
  return x;
}

__device__ __forceinline__ Best warp_best(Best s) {
  for (int o = 16; o; o >>= 1) {
    Best t;
    t.v1 = __shfl_xor_sync(0xffffffffu, s.v1, o);
    t.v2 = __shfl_xor_sync(0xffffffffu, s.v2, o);
    t.j1 = __shfl_xor_sync(0xffffffffu, s.j1, o);
    s = best_merge(s, t);
  }
  return s;
}

// objects [lo, hi) for person (ax, ay, az), one warp; every lane returns the warp's result
__device__ __forceinline__ Best scan_objects(double ax, double ay, double az, const double* __restrict__ b,
                                             const double* price, int lo, int hi, int lane) {
  Best s{INFINITY, INFINITY, 0x7fffffff};
  for (int j = lo + lane; j < hi; j += 32) {              // j increases along a lane: strict < keeps the lowest index
    const double v = __dadd_rn(emd_cost(ax, ay, az, b, j), __ldcg(price + j));
    if (v < s.v1) { s.v2 = s.v1; s.v1 = v; s.j1 = j; }
    else if (v < s.v2) s.v2 = v;
  }
  return warp_best(s);
}

// fixed-order sum of x[lo, hi) (hi - lo <= 32 * k): lane-strided sequential sums, then a xor butterfly; every lane holds it
__device__ __forceinline__ double warp_sum(const double* x, int lo, int hi, int lane) {
  double s = 0.0;
  for (int i = lo + lane; i < hi; i += 32) s = __dadd_rn(s, __ldcg(x + i));
  for (int o = 16; o; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
  return s;
}

__device__ __forceinline__ bool key_less(const BidKey& x, const BidKey& y) {      // x loses to y
  return x.bid < y.bid || (x.bid == y.bid && x.person > y.person);
}

__device__ void place_bid(const EmdArgs& A, int i, int k, const Best& r, double eps) {
  const EmdWs& w = A.w;
  if (r.j1 >= A.n) { atomicExch(w.abort, 1); return; }     // no finite value in the scan
  const double p = __ldcg(w.price + r.j1);
  const double gain = A.n > 1 ? __dsub_rn(r.v2, r.v1) : 0.0;
  const double bid = __dadd_rn(__dadd_rn(p, gain), eps);
  if (!(bid <= DBL_MAX)) { atomicExch(w.abort, 1); return; }
  w.sbid[k] = bid;
  w.sj[k] = r.j1;
  const BidKey mine{(unsigned long long)__double_as_longlong(bid), (unsigned long long)i};
  // The key as the round started: the first CAS succeeds unless another bidder of this round got there first.
  BidKey cur{(unsigned long long)__double_as_longlong(p), (unsigned long long)(long long)__ldcg(w.kwin + r.j1)};
  // Each failed CAS returns a strictly larger key, and only this round's bidders of the object write it: bounded.
  while (key_less(cur, mine)) {
    BidKey old;
    asm volatile("{\n\t.reg .b128 c, v, o;\n\tmov.b128 c, {%2, %3};\n\tmov.b128 v, {%4, %5};\n\t"
                 "atom.global.cas.b128 o, [%6], c, v;\n\tmov.b128 {%0, %1}, o;\n\t}"
                 : "=l"(old.bid), "=l"(old.person)
                 : "l"(cur.bid), "l"(cur.person), "l"(mine.bid), "l"(mine.person), "l"(w.key + r.j1) : "memory");
    if (old.bid == cur.bid && old.person == cur.person) break;
    cur = old;
  }
}

__global__ void __launch_bounds__(EMD_THREADS, 2) emd_auction_kernel(EmdArgs A) {
  cg::grid_group grid = cg::this_grid();
  const EmdWs& w = A.w;
  const int n = A.n;
  const int lane = threadIdx.x & 31;
  const int gw = blockIdx.x * EMD_WARPS + (threadIdx.x >> 5), W = gridDim.x * EMD_WARPS;
  const int tid = blockIdx.x * EMD_THREADS + threadIdx.x, T = gridDim.x * EMD_THREADS;
  const int nch = (n + EMD_SUM_CHUNK - 1) / EMD_SUM_CHUNK;

  // start: zero prices, empty keys, every row a bidder, outputs that say "no phase completed", the largest cost (the
  // workspace arrives uninitialised, apart from the 64-byte header the host clears)
  for (int i = tid; i < n; i += T) {
    w.price[i] = 0.0;
    w.kwin[i] = -1;
    w.key[i] = BidKey{0ull, ~0ull};
    w.owner[i] = -1;
    w.assign[i] = -1;
    w.list[0][i] = i;
    w.scnt[i] = 0;
    A.out_assign[i] = -1;
    A.out_cost[i] = INFINITY;
  }
  for (int i = gw; i < n; i += W) {
    const double ax = __ldg(A.a + 3 * i), ay = __ldg(A.a + 3 * i + 1), az = __ldg(A.a + 3 * i + 2);
    double m = 0.0;
    for (int j = lane; j < n; j += 32) m = fmax(m, emd_cost(ax, ay, az, A.b, j));
    for (int o = 16; o; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) atomicMax(w.cmax, (unsigned long long)__double_as_longlong(m));
  }
  if (tid == 0) {
    w.count[0] = n;
    A.out_stats[0] = INFINITY;
    for (int t = 1; t < 6; ++t) A.out_stats[t] = 0.0;
  }
  grid.sync();
  const double cmax = __longlong_as_double((long long)__ldcg(w.cmax));
  if (!(cmax <= DBL_MAX)) return;                          // a squared distance overflowed: no phase can complete
  const double eps_min = (cmax > 0.0 ? cmax : 1.0) * 0x1p-40;
  const double floor_gap = __dmul_rn((double)n, eps_min);
  double eps = fmax(cmax * 0.25, eps_min);
  long long rounds = 0;
  int phases = 0;
  long long rr = 0;                                        // round slot: list rr & 1, count rr % 3

  for (;;) {
    const int* L = w.list[rr & 1];
    const int nb = __ldcg(w.count + rr % 3);
    if (nb == 0) {
      // ---- phase complete: bounds of the assignment, keep or stop
      for (int i = gw; i < n; i += W) {
        const double ax = __ldg(A.a + 3 * i), ay = __ldg(A.a + 3 * i + 1), az = __ldg(A.a + 3 * i + 2);
        const Best r = scan_objects(ax, ay, az, A.b, w.price, 0, n, lane);
        if (lane == 0) {
          w.rowmin[i] = r.v1;
          w.cost[i] = emd_cost(ax, ay, az, A.b, __ldcg(w.assign + i));
        }
      }
      grid.sync();
      for (int c = gw; c < nch; c += W) {
        const int lo = c * EMD_SUM_CHUNK, hi = min(n, lo + EMD_SUM_CHUNK);
        const double s0 = warp_sum(w.cost, lo, hi, lane), s1 = warp_sum(w.rowmin, lo, hi, lane), s2 = warp_sum(w.price, lo, hi, lane);
        if (lane == 0) { w.sums[c] = s0; w.sums[nch + c] = s1; w.sums[2 * nch + c] = s2; }
      }
      grid.sync();
      // every warp reduces the chunk sums itself, in the same order, and takes the same decision
      const double primal = warp_sum(w.sums, 0, nch, lane);
      const double dual = __dsub_rn(warp_sum(w.sums + nch, 0, nch, lane), warp_sum(w.sums + 2 * nch, 0, nch, lane));
      ++phases;
      const bool converged = __dsub_rn(primal, dual) <= __dadd_rn(__dmul_rn(A.rel_tol, primal), floor_gap);
      const bool stop = converged || eps <= eps_min;
      for (int i = tid; i < n; i += T) {
        A.out_assign[i] = __ldcg(w.assign + i);
        A.out_cost[i] = __ldcg(w.cost + i);
        if (!stop) { w.assign[i] = -1; w.owner[i] = -1; w.list[rr & 1][i] = i; }
      }
      if (tid == 0) {
        A.out_stats[0] = primal; A.out_stats[1] = dual; A.out_stats[2] = eps;
        A.out_stats[3] = (double)phases; A.out_stats[4] = (double)rounds; A.out_stats[5] = converged ? 1.0 : 0.0;
        if (!stop) w.count[rr % 3] = n;
      }
      if (stop) return;
      eps = fmax(eps / EMD_THETA, eps_min);
      grid.sync();
      continue;
    }
    if (rounds >= A.cap) return;                           // the outputs hold the last completed phase
    ++rounds;

    // ---- bids: nb bidders, each scan split into S pieces when the bidders are fewer than the warps
    int S = 1;
    if (nb < W) {
      S = min(W / nb, (n + EMD_MIN_CHUNK - 1) / EMD_MIN_CHUNK);
      S = max(1, min(S, EMD_MAX_UNITS / nb));
    }
    const int units = nb * S;
    for (int u = gw; u < units; u += W) {
      const int k = u / S, s = u - k * S;
      const int i = __ldcg(L + k);
      const double ax = __ldg(A.a + 3 * i), ay = __ldg(A.a + 3 * i + 1), az = __ldg(A.a + 3 * i + 2);
      const int lo = (int)((int64_t)n * s / S), hi = (int)((int64_t)n * (s + 1) / S);
      Best r = scan_objects(ax, ay, az, A.b, w.price, lo, hi, lane);
      if (S == 1) {
        if (lane == 0) place_bid(A, i, k, r, eps);
        continue;
      }
      int last = 0;
      if (lane == 0) {
        w.pv1[u] = r.v1; w.pv2[u] = r.v2; w.pj[u] = r.j1;
        __threadfence();
        last = atomicAdd(w.scnt + k, 1) == S - 1;
      }
      last = __shfl_sync(0xffffffffu, last, 0);
      if (!last) continue;
      __threadfence();
      Best m{INFINITY, INFINITY, 0x7fffffff};
      for (int t = lane; t < S; t += 32) {
        const Best p{__ldcg(w.pv1 + k * S + t), __ldcg(w.pv2 + k * S + t), __ldcg(w.pj + k * S + t)};
        m = best_merge(m, p);
      }
      m = warp_best(m);
      if (lane == 0) {
        w.scnt[k] = 0;
        place_bid(A, i, k, m, eps);
      }
    }
    if (tid == 0) w.count[(rr + 2) % 3] = 0;               // read in round rr - 1, appended from round rr + 1 on
    grid.sync();
    if (__ldcg(w.abort)) return;                           // the outputs hold the last completed phase

    // ---- resolution: the key of each object names its winner
    int* next = w.list[(rr + 1) & 1];
    int* next_count = w.count + (rr + 1) % 3;
    for (int k = tid; k < nb; k += T) {
      const int i = __ldcg(L + k), j = __ldcg(w.sj + k);
      const double bid = __ldcg(w.sbid + k);
      const unsigned long long kb = __ldcg(&w.key[j].bid), kp = __ldcg(&w.key[j].person);
      if (kp == (unsigned long long)i && kb == (unsigned long long)__double_as_longlong(bid)) {
        w.price[j] = bid;
        w.kwin[j] = i;
        const int prev = __ldcg(w.owner + j);
        w.owner[j] = i;
        w.assign[i] = j;
        if (prev >= 0) {
          w.assign[prev] = -1;
          next[atomicAdd(next_count, 1)] = prev;
        }
      } else {
        next[atomicAdd(next_count, 1)] = i;
      }
    }
    ++rr;
    grid.sync();
  }
}

static long long emd_round_cap(int64_t n) {
  static const long long env = [] {                       // read once per process, like the Settings switches
    const char* e = getenv("SAPCU_EMD_MAX_ROUNDS");
    return e ? atoll(e) : 0LL;
  }();
  if (env > 0) return env;
  const long long d = 256LL * n;
  return d > (1LL << 20) ? d : (1LL << 20);
}

}  // namespace sapcu

using namespace sapcu;

extern "C" {

size_t sapcu_emd_workspace_bytes(int64_t n) {
  if (n < 1 || n > EMD_MAX_N) return 0;
  return emd_layout(n, nullptr, nullptr);
}

int sapcu_emd(const double* d_a, const double* d_b, int64_t n, double rel_tol, int32_t* d_assign, double* d_cost,
              double* d_stats, void* d_ws, size_t ws_bytes, void* stream) {
  SAPCU_REQUIRE(n >= 1 && n <= EMD_MAX_N, "emd: n=%lld outside 1 <= n <= %lld", (long long)n, (long long)EMD_MAX_N);
  SAPCU_REQUIRE(rel_tol >= 0.0, "emd: rel_tol must be >= 0");
  SAPCU_REQUIRE(d_a && d_b && d_assign && d_cost && d_stats && d_ws, "emd: null pointer");
  const size_t need = emd_layout(n, nullptr, nullptr);
  if (ws_bytes < need) {
    set_error("emd: workspace of %zu bytes, %zu needed", ws_bytes, need);
    return SAPCU_EWORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int per_sm = 0, dev = 0, sms = 0;
  SAPCU_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, emd_auction_kernel, EMD_THREADS, 0));
  SAPCU_CUDA_CHECK(cudaGetDevice(&dev));
  SAPCU_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (per_sm < 1) { set_error("emd: the auction kernel cannot be resident"); return SAPCU_ECUDA; }
  const int64_t max_blocks = (int64_t)per_sm * sms;
  int64_t blocks = ceil_div(n, EMD_POINTS_PER_BLOCK);
  if (blocks > max_blocks) blocks = max_blocks;
  EmdArgs args;
  args.a = d_a; args.b = d_b; args.n = (int)n; args.rel_tol = rel_tol; args.cap = emd_round_cap(n);
  args.out_assign = d_assign; args.out_cost = d_cost; args.out_stats = d_stats;
  emd_layout(n, &args.w, reinterpret_cast<char*>(d_ws));
  SAPCU_CUDA_CHECK(cudaMemsetAsync(d_ws, 0, 64, st));     // cmax and the list counts
  void* kargs[] = {(void*)&args};
  SAPCU_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)emd_auction_kernel, dim3((unsigned)blocks), dim3(EMD_THREADS), kargs, 0, st));
  count_launch();
  return 0;
}

}  // extern "C"
