// tcgen05 tensor-core GEMM engine (SAPCU_MODE_TC): interface used by forward.cu.
#pragma once
#include "gemm_simt.cuh"

namespace sapcu {
// true when the tensor-core engine implements this (loader, epilogue, shape) combination;
// everything else stays on the fp32 SIMT engine.
bool gemm_tc_supported(const GemmArgs& g, int amode);
int launch_gemm_tc(const GemmArgs& g, int amode, cudaStream_t st);
// pipeline watchdog status of every launch_gemm_tc since the last check (0 = fine); synchronises the stream
int gemm_tc_check(cudaStream_t st);
// 2-CTA (cta_group::2) variant for N % 256 == 0 problems (gemm_tc2.cu)
bool gemm_tc2_supported(const GemmArgs& g, int amode);
int launch_gemm_tc2(const GemmArgs& g, cudaStream_t st);
// true when launch_gemm_tc2 would run this problem on the fp16x3 operand path (needed to agree on the fp16-plane
// activation format between the kernel that writes a tensor and the one that reads it)
bool gemm_tc2_fp16x3(const GemmArgs& g);
// true when launch_gemm_tc2 would run this problem on the single-product fp16 path of SAPCU_MODE_FAST (input and, for LIF
// layers, output are single fp16 planes of x * 2^13)
bool gemm_tc2_fast(const GemmArgs& g);
bool gemm_tc2_fast_tf32(const GemmArgs& g);
int* tc_err_flag();   // the device's mapped error flag (pipeline watchdog, pair-table index check)
}  // namespace sapcu
