// C ABI glue: error string, launch counter, and the stand-alone operator entry points.
#include <atomic>
#include <mutex>
#include <string>
#include <vector>
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include <cmath>
#include "lif_table.cuh"
#include "../../include/sapcu_b200.h"
#include "gemm_simt.cuh"
#include "gemm_tc.h"
#include "kernels.h"

namespace sapcu {

thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

static int env_int(const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; }
const Settings& settings() {
  static const Settings s = [] {
    Settings t;
    t.fuse_attnout = env_int("SAPCU_TC_FUSE_ATTNOUT", 1) != 0;
    t.factor_attnin = env_int("SAPCU_TC_FACTOR_ATTNIN", 1) != 0;
    t.fuse_pool = env_int("SAPCU_TC_FUSE_POOL", 1) != 0;
    t.fast_tables = env_int("SAPCU_FAST_LIF_TABLES", 1) != 0;
    t.sync_check = env_int("SAPCU_TC_SYNC_CHECK", 0) != 0;
    return t;
  }();
  return s;
}

static_assert(sizeof(std::mutex) <= 64, "PerDeviceOnce::mu_ too small");
int PerDeviceOnce::run(int (*f)()) {
  static std::mutex init_mu;                       // guards the placement of the per-object mutex
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { set_error("cudaGetDevice failed"); return -2; }
  if (dev < 0 || dev >= 64) return f();
  std::lock_guard<std::mutex> lk(init_mu);         // attribute setup is rare: one global lock is enough
  if (done_[dev]) return 0;
  const int rc = f();
  if (rc == 0) done_[dev] = true;
  return rc;
}

// ---- optional live timing of the contraction kernels (bench.py roofline)
static std::mutex g_prof_mu;
static bool g_prof_on = false;
struct ProfEntry { cudaEvent_t a, b; const char* label; ProfWork w; };
static std::vector<ProfEntry> g_prof_ev;

bool prof_begin(cudaStream_t st, const char* label, const ProfWork& w, int* slot) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_prof_on) return false;
  cudaEvent_t a, b;
  if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return false;
  cudaEventRecord(a, st);
  g_prof_ev.push_back(ProfEntry{a, b, label, w});
  *slot = (int)g_prof_ev.size() - 1;
  return true;
}
void prof_end(cudaStream_t st, int slot) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (slot >= 0 && slot < (int)g_prof_ev.size()) cudaEventRecord(g_prof_ev[slot].b, st);
}

}  // namespace sapcu

using namespace sapcu;

extern "C" {

const char* sapcu_last_error(void) { return g_err; }
int sapcu_abi_version(void) { return 1; }
int64_t sapcu_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int sapcu_profile(int enable) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (auto& e : g_prof_ev) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
  g_prof_ev.clear();
  g_prof_on = enable != 0;
  return 0;
}

int64_t sapcu_profile_report(char* buf, size_t cap) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  struct Agg { double ms = 0, flops = 0, elsteps = 0, bytes = 0; int64_t n = 0; };
  std::vector<std::pair<std::string, Agg>> agg;                 // first-seen order
  for (auto& e : g_prof_ev) {
    if (cudaEventSynchronize(e.b) != cudaSuccess) { set_error("profile_report: event sync failed"); return SAPCU_ECUDA; }
    float t = 0.f;
    if (cudaEventElapsedTime(&t, e.a, e.b) != cudaSuccess) { set_error("profile_report: elapsed time failed"); return SAPCU_ECUDA; }
    size_t i = 0;
    for (; i < agg.size(); ++i) if (agg[i].first == e.label) break;
    if (i == agg.size()) agg.emplace_back(std::string(e.label), Agg());
    Agg& a = agg[i].second;
    a.ms += t; a.flops += e.w.flops; a.elsteps += e.w.elsteps; a.bytes += e.w.bytes; a.n += 1;
  }
  std::string js = "[";
  char line[512];
  for (size_t i = 0; i < agg.size(); ++i) {
    const Agg& a = agg[i].second;
    snprintf(line, sizeof(line), "%s{\"label\": \"%s\", \"launches\": %lld, \"ms\": %.6f, \"flops\": %.6e, \"lif_elsteps\": %.6e, \"bytes\": %.6e}",
             i ? ", " : "", agg[i].first.c_str(), (long long)a.n, a.ms, a.flops, a.elsteps, a.bytes);
    js += line;
  }
  js += "]";
  if (buf && cap > 0) { const size_t n = js.size() < cap - 1 ? js.size() : cap - 1; memcpy(buf, js.data(), n); buf[n] = 0; }
  return (int64_t)js.size() + 1;
}

int sapcu_profile_read(double* gemm_ms, double* gemm_flops, int64_t* gemm_launches) {
  SAPCU_REQUIRE(gemm_ms && gemm_flops && gemm_launches, "profile_read: null pointer");
  std::lock_guard<std::mutex> lk(g_prof_mu);
  double ms = 0.0, flops = 0.0; int64_t n = 0;
  for (auto& e : g_prof_ev) {
    if (!e.w.gemm) continue;
    SAPCU_CUDA_CHECK(cudaEventSynchronize(e.b));
    float t = 0.f;
    SAPCU_CUDA_CHECK(cudaEventElapsedTime(&t, e.a, e.b));
    ms += t; flops += e.w.flops; ++n;
  }
  *gemm_ms = ms; *gemm_flops = flops; *gemm_launches = n;
  return 0;
}

// fp32 SoA copy of the cloud (3 arrays of round_up(N, 4) + 4 floats, see knn_seed.cu) + one scalar
static size_t knn_c32_bytes(int64_t N) { return align_up((size_t)(3 * ((N + 3) / 4 * 4 + 4)) * sizeof(float), 256); }
size_t sapcu_knn_workspace_bytes(int64_t N) {
  if (N < 0) return 0;
  return knn_c32_bytes(N) + 256;
}

int sapcu_knn(const double* d_cloud, int64_t N, const double* d_seeds, int64_t S, int K, int32_t* d_idx,
              void* d_ws, size_t ws_bytes, void* stream) {
  SAPCU_REQUIRE(N >= 1 && S >= 0, "sapcu_knn: bad sizes N=%lld S=%lld", (long long)N, (long long)S);
  SAPCU_REQUIRE(d_cloud && (S == 0 || (d_seeds && d_idx)) && d_ws, "sapcu_knn: null pointer");
  SAPCU_REQUIRE(reinterpret_cast<uintptr_t>(d_ws) % 16 == 0, "sapcu_knn: workspace %p is not 16-byte aligned", d_ws);
  if (ws_bytes < sapcu_knn_workspace_bytes(N)) {
    set_error("sapcu_knn: workspace %zu < %zu bytes", ws_bytes, sapcu_knn_workspace_bytes(N));
    return SAPCU_EWORKSPACE;
  }
  float* c32 = reinterpret_cast<float*>(d_ws);
  float* rmax = reinterpret_cast<float*>(reinterpret_cast<char*>(d_ws) + knn_c32_bytes(N));
  return launch_knn_seed(d_cloud, N, d_seeds, S, K, d_idx, c32, rmax, reinterpret_cast<cudaStream_t>(stream));
}

size_t sapcu_knn_batched_workspace_bytes(int64_t N_total, int B) {
  if (N_total < 0 || B < 0) return 0;
  return knn_c32_bytes(N_total) + 256 + align_up(3 * (size_t)(B + 1) * sizeof(int64_t), 256);
}

int sapcu_knn_batched(const double* d_clouds, const int64_t* h_cloud_off, const double* d_seeds, const int64_t* h_seed_off,
                      int B, int K, int32_t* d_idx, void* d_ws, size_t ws_bytes, void* stream) {
  SAPCU_REQUIRE(B >= 1 && h_cloud_off && h_seed_off, "sapcu_knn_batched: bad batch description");
  const int64_t N = h_cloud_off[B], S = h_seed_off[B];
  SAPCU_REQUIRE(N >= 1 && S >= 0, "sapcu_knn_batched: bad sizes N=%lld S=%lld", (long long)N, (long long)S);
  SAPCU_REQUIRE(d_clouds && (S == 0 || (d_seeds && d_idx)) && d_ws, "sapcu_knn_batched: null pointer");
  SAPCU_REQUIRE(reinterpret_cast<uintptr_t>(d_ws) % 16 == 0, "sapcu_knn_batched: workspace %p is not 16-byte aligned", d_ws);
  if (ws_bytes < sapcu_knn_batched_workspace_bytes(N, B)) {
    set_error("sapcu_knn_batched: workspace %zu < %zu bytes", ws_bytes, sapcu_knn_batched_workspace_bytes(N, B));
    return SAPCU_EWORKSPACE;
  }
  char* w = reinterpret_cast<char*>(d_ws);
  float* c32 = reinterpret_cast<float*>(w);
  float* rmax = reinterpret_cast<float*>(w + knn_c32_bytes(N));
  int64_t* tab = reinterpret_cast<int64_t*>(w + knn_c32_bytes(N) + 256);
  return launch_knn_seed_batched(d_clouds, h_cloud_off, d_seeds, h_seed_off, B, K, d_idx, c32, rmax, tab,
                                 reinterpret_cast<cudaStream_t>(stream));
}

int sapcu_gather_center_rotate(const double* d_cloud, int64_t N, const double* d_seeds, const int32_t* d_idx,
                               int64_t S, int K, const float* d_normals, float* d_patches, void* stream) {
  SAPCU_REQUIRE(N >= 1 && S >= 0 && K >= 1, "gather_center_rotate: bad sizes");
  SAPCU_REQUIRE(d_cloud && (S == 0 || (d_seeds && d_idx && d_patches)), "gather_center_rotate: null pointer");
  return launch_gather_center_rotate(d_cloud, d_seeds, d_idx, S, K, d_normals, d_patches,
                                     reinterpret_cast<cudaStream_t>(stream));
}

int sapcu_renormalize(float* d_normals, int64_t S, void* stream) {
  SAPCU_REQUIRE(S >= 0 && (S == 0 || d_normals), "renormalize: bad argument");
  return launch_renormalize(d_normals, S, reinterpret_cast<cudaStream_t>(stream));
}

int sapcu_displace(const double* d_seeds, const float* d_normals, const float* d_dist, int64_t S, double* d_out,
                   void* stream) {
  SAPCU_REQUIRE(S >= 0 && (S == 0 || (d_seeds && d_normals && d_dist && d_out)), "displace: bad argument");
  return launch_displace(d_seeds, d_normals, d_dist, S, d_out, reinterpret_cast<cudaStream_t>(stream));
}

int sapcu_lif_chain(const float* d_x, int64_t rows, int C, int T, const float* d_params4, const float* d_eif2,
                    int all_steps, float* d_out, void* stream) {
  SAPCU_REQUIRE(rows >= 0 && C >= 1 && T >= 1 && d_params4 && (rows == 0 || (d_x && d_out)), "lif_chain: bad argument");
  // parameters arrive raw: clamp them on the fly into a small device scratch?  The ABI keeps this operator
  // allocation-free by requiring the caller to pass CLAMPED parameters (the Python shim clamps).
  return launch_neuron_unroll(d_eif2 != nullptr, true, d_x, C, rows, C, T, d_params4, d_eif2, all_steps, d_out, C,
                              reinterpret_cast<cudaStream_t>(stream));
}

int sapcu_lif_table_selftest(const float* h_params4, int C, int T, int samples, double* max_err, double* fit_err, uint32_t* max_block_bytes) {
  SAPCU_REQUIRE(h_params4 && C >= 1 && T >= 1 && T <= 16 && samples >= 1 && max_err && fit_err && max_block_bytes, "lif_table_selftest: bad argument");
  LifTableHost t;
  lif_table_build(h_params4, C, T, &t);
  *fit_err = t.max_err; *max_block_bytes = t.max_block_bytes;
  double worst = 0.0;
  for (int c = 0; c < C; ++c) {
    const double d = h_params4[c], a = h_params4[C + c], r = h_params4[2 * C + c], th0 = h_params4[3 * C + c];
    auto probe = [&](float x) {
      const float got = lif_table_eval_host(t, c, x);
      const double want = lif_chain_exact_host((double)th0 + (double)x, d, a, r, th0, T);
      const double e = std::isnan(got) ? 1e30 : std::fabs((double)got - want);
      worst = e > worst ? e : worst;
    };
    for (int i = 0; i < samples; ++i) {            // geometric spread over both sides, 2^-12 .. 254.9
      const float mag = std::ldexp(1.0f, -12) * std::pow(254.9f / std::ldexp(1.0f, -12), (float)(i + 0.5f) / (float)samples);
      probe(mag); probe(-mag);
    }
    probe(0.0f); probe(-0.0f); probe(1e-30f); probe(-1e-30f); probe(254.99998f); probe(-254.99998f);
    for (int e = 0; e < LT_NB; ++e) {              // both neighbours of every cell boundary y = 2^(e+1): |x| = 2^e - 1
      const float xb = std::ldexp(1.0f, e) - 1.0f;
      for (float s : {1.0f, -1.0f}) { probe(s * xb); probe(s * std::nextafter(xb, 1e9f)); if (xb > 0.0f) probe(s * std::nextafter(xb, 0.0f)); }
    }
  }
  *max_err = worst;
  return 0;
}

int sapcu_intra_knn(const float* d_feat, int64_t ld, int64_t S, int M, int C, int k, int32_t* d_idx, void* stream) {
  SAPCU_REQUIRE(S >= 0 && C >= 1 && ld >= C && (S == 0 || (d_feat && d_idx)), "intra_knn: bad argument");
  return launch_intra_knn(d_feat, ld, S, M, C, k, d_idx, reinterpret_cast<cudaStream_t>(stream));
}

int sapcu_gemm(const float* d_x, int64_t R, int K, const float* d_w, int N, const float* d_bias, float* d_y, int mode,
               void* stream) {
  SAPCU_REQUIRE(R >= 0 && K >= 1 && N >= 1 && d_w && (R == 0 || (d_x && d_y)), "gemm: bad argument");
  GemmArgs g;
  g.A = d_x; g.lda = K; g.R = R; g.K = K; g.W = d_w; g.N = N; g.bias = d_bias; g.Y = d_y; g.ldc = N;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (mode == SAPCU_MODE_TC || mode == SAPCU_MODE_TF32) {
    g.tc_passes = mode == SAPCU_MODE_TF32 ? 1 : 3;
    if (!gemm_tc_supported(g, A_PLAIN)) { set_error("gemm: shape R=%lld K=%d N=%d not supported by the tensor-core engine", (long long)R, K, N); return SAPCU_EINVAL; }
    int rc = launch_gemm_tc(g, A_PLAIN, st);
    return rc ? rc : gemm_tc_check(st);
  }
  SAPCU_REQUIRE(mode == SAPCU_MODE_FP32, "gemm: unknown mode %d", mode);
  return launch_gemm_simt(g, A_PLAIN, true, st);
}

}  // extern "C"
