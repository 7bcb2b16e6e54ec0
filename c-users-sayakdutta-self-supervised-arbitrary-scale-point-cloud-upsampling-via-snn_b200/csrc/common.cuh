// Shared helpers for the sapcu_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

namespace sapcu {

// ---- error plumbing (thread-local message, negative return codes; never throws over the ABI)
void set_error(const char* fmt, ...);
extern thread_local char g_err[512];
void count_launch(int n = 1);
// live per-launch timing (bench.py's roofline entries): algorithmic work of one launch, by the roofline it is graded on
struct ProfWork {
  double flops = 0.0;      // tensor / FFMA: 2*R*K*N of a contraction
  double elsteps = 0.0;    // MUFU: LIF / EIF element-steps (elements x T)
  double bytes = 0.0;      // HBM: algorithmic bytes read + written
  bool gemm = false;       // member of the contraction family (sapcu_profile_read's aggregate)
};
bool prof_begin(cudaStream_t st, const char* label, const ProfWork& w, int* slot);
void prof_end(cudaStream_t st, int slot);
#define SAPCU_PROF(st, label, work, expr)                                             \
  do {                                                                                \
    int _slot = -1;                                                                   \
    const bool _p = sapcu::prof_begin(st, label, work, &_slot);                       \
    const int _rc = (expr);                                                           \
    if (_p) sapcu::prof_end(st, _slot);                                               \
    if (_rc) return _rc;                                                              \
  } while (0)

#define SAPCU_CUDA_CHECK(expr)                                                        \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      sapcu::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return -2;                                                                      \
    }                                                                                 \
  } while (0)

#define SAPCU_LAUNCH_CHECK()                                                          \
  do {                                                                                \
    sapcu::count_launch();                                                            \
    cudaError_t _e = cudaGetLastError();                                              \
    if (_e != cudaSuccess) {                                                          \
      sapcu::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return -2;                                                                      \
    }                                                                                 \
  } while (0)

#define SAPCU_REQUIRE(cond, ...)                                                      \
  do {                                                                                \
    if (!(cond)) { sapcu::set_error(__VA_ARGS__); return -1; }                        \
  } while (0)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

constexpr int kNumSMs = 148;   // B200

// Process-wide switches (environment, DESIGN.md section 5), read ONCE under C++11 static-initialisation locking and
// immutable afterwards: concurrent forwards from several threads / streams all see the same values.
//   fuse_attnout, factor_attnin, fuse_pool  the unfused tensor-core schedule, reference of the fused-epilogue tests
//   fast_tables                             the fast mode's 2-MUFU recurrence instead of the LIF tables
//   sync_check                              every forward synchronises its stream before checking the watchdog flag
struct Settings {
  bool fuse_attnout, factor_attnin, fuse_pool, fast_tables, sync_check;
};
const Settings& settings();

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: run `f` once per CUDA device (thread-safe)
struct PerDeviceOnce {
  int run(int (*f)());
 private:
  bool done_[64] = {};
  char mu_[64] = {};     // storage for a std::mutex (kept opaque so this header stays light); see api.cu
};

// ---- activation codes shared by the GEMM epilogues
enum Act : int { ACT_NONE = 0, ACT_LEAKY = 1, ACT_GELU = 2, ACT_LIF = 3 };

}  // namespace sapcu
