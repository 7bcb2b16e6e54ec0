// Internal launcher prototypes (host side).  Every launcher returns 0 or a negative SAPCU_E* code
// after recording the message with sapcu::set_error.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sapcu {

// knn_seed.cu
int launch_knn_seed(const double* cloud, int64_t N, const double* seeds, int64_t S, int K, int32_t* idx,
                    float* cloud32_scratch, float* rmax_scratch, cudaStream_t st);
int launch_knn_seed_batched(const double* clouds, const int64_t* h_cloud_off, const double* seeds, const int64_t* h_seed_off,
                            int B, int K, int32_t* idx, float* cloud32_scratch, float* rmax_scratch, int64_t* tab,
                            cudaStream_t st);
// patch_ops.cu
int launch_gather_center_rotate(const double* cloud, const double* seeds, const int32_t* idx, int64_t S, int K,
                                const float* normals, float* patches, cudaStream_t st);
int launch_renormalize(float* n, int64_t S, cudaStream_t st);
int launch_displace(const double* seeds, const float* n, const float* d, int64_t S, double* out, cudaStream_t st);
// intra_knn.cu
int launch_intra_knn(const float* feat, int64_t ld, int64_t S, int M, int C, int k, int32_t* idx, cudaStream_t st);
// fn_kernels.cu
int launch_pointwise3_lif(bool edge, bool precise, const float* xyz, const int32_t* idx, int kk, int ldi, int Mpts,
                          int64_t rows, int C, const float* W, const float* bias, const float* scale,
                          const float* shift, const float* np, int T, float* out, cudaStream_t st, int nsplit = 1, bool out_h2 = false);
int launch_edge_pos_lif_fast(const float* xyz, const int32_t* idx, int kk, int ldi, int Mpts, int64_t rows, int C,
                             const float* W, const float* bias, const float* scale, const float* shift, const float* np, int T,
                             float* out_h, const float* tab, uint32_t tab_stride, cudaStream_t st, bool two_planes = false);
// fc_delta + BN + tabulated LIF^T on the offsets delta[u] of the first *U_dev pair rows, (hi, lo) planes out (capacity `rows`:
// the lo plane's offset)
int launch_pair_pos_lif(const float4* delta, const int* U_dev, int64_t rows, int C, const float* W, const float* bias,
                        const float* scale, const float* shift, const float* np, int T, float* out_h, const float* tab,
                        uint32_t tab_stride, cudaStream_t st);
// fc_gamma's BN + tabulated LIF^T per edge from the per-pair product WP[pid[e]] and the per-point edge bias QK (= [W q | W k])
int launch_edge_gamma_lif(const float* WP, const int32_t* pid, const float* QK, const int32_t* idx, int kk, int ldi, int Mpts,
                          int64_t rows, int C, const float* bias, const float* scale, const float* shift, const float* np, int T,
                          float* out_h, const float* tab, uint32_t tab_stride, cudaStream_t st);
// edge_pairs.cu: the pair table of an fn chunk (views into the workspace; pair_plan(.., nullptr) only sizes it)
struct PairBufs {
  int64_t E = 0; int kmax = 0, jb = 0, bits = 0, kk[3] = {0, 0, 0};
  uint64_t* key[2] = {nullptr, nullptr}; int32_t* val[2] = {nullptr, nullptr};
  int* flag[3] = {nullptr, nullptr, nullptr};
  int32_t* pid[3] = {nullptr, nullptr, nullptr};       // [P * kk_b] pair row of every edge of block b
  float4* delta[3] = {nullptr, nullptr, nullptr};      // [U_b] offsets cloud[gi] - cloud[gj]
  int* U = nullptr;                                    // [3] pair counts (device)
  void* tmp = nullptr; size_t tmp_bytes = 0, bytes = 0;
};
PairBufs pair_plan(int64_t P, int kmax, const int kk[3], int64_t N, void* base);
bool pair_key_fits(int64_t N, int kmax);     // the key ((gi * N + gj) << bits(kmax)) | j fits 64 bits
int build_pairs(const PairBufs& q, const int32_t* idx, int M, const int32_t* gidx, int64_t ldg, const double* cloud, int64_t N,
                int* err, cudaStream_t st);
int launch_pack_idx_u8(const int32_t* idx, int ldi, int64_t P, uint32_t* out, cudaStream_t st);
int launch_attn_out(bool precise, const float* logits, const float* pos, const float* V, int64_t ldv,
                    const int32_t* idx, int ldi, int kk, int Mpts, int64_t P, int D, float sqrt_hd, float* out,
                    cudaStream_t st);
int launch_attn_in(const float* Q, const float* Kf, int64_t ldq, const float* pos, const int32_t* idx, int ldi, int kk,
                   int Mpts, int64_t E, int D, float* out, cudaStream_t st);
int launch_fill(float* p, int64_t n, float v, cudaStream_t st);
int launch_group_max(const float* X, int64_t S, int M, int Tt, int C, float* out, cudaStream_t st);
int launch_fn_head(const float* H, int K, int64_t S, const float* W, const float* b, const float* lnw,
                   const float* lnb, float* out, cudaStream_t st);
// fd_kernels.cu
int launch_fd_block0(const float* xyz, const int32_t* idx, int ldi, int Mpts, int64_t P, int nscales, const int* ks,
                     const float* const* W, const float* const* scale, const float* const* shift, float* out,
                     cudaStream_t st);
int launch_edge_gather_unroll(bool eif, const float* PQ, int C, const int32_t* idx, int kk, int Mpts, int64_t S,
                              const float* scale, const float* shift, const float* np, const float* ep, int T, float* U,
                              float* spk, int64_t ldspk_row, int ldo, cudaStream_t st, bool h2 = false, float* spk0 = nullptr, int64_t plane = 0, int choff = 0);
int launch_neuron_unroll(bool eif, bool precise, const float* U, int64_t ldu, int64_t rows, int C, int T,
                         const float* np, const float* ep, int all_steps, float* out, int64_t ldo, cudaStream_t st,
                         bool h2 = false, float* out0 = nullptr, int64_t plane = 0, int choff = 0);
int launch_temporal_lif(bool precise, const float* pool, int64_t S, int Tt, int C, const float* wsm, const float* np,
                        float* out, cudaStream_t st);
int launch_head_attention(const float* qkv, int64_t S, int H, int hd, float scale, float* out, cudaStream_t st);
int launch_layernorm_rows(const float* X, int64_t S, int C, const float* w, const float* b, float* out, cudaStream_t st);
int launch_fd_tail(const float* H, int64_t S, int K, const float* w, const float* b, float* out, cudaStream_t st);

}  // namespace sapcu
