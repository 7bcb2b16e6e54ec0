/*
 * sapcu_b200 -- C ABI of the B200-native inference hot path of the SNN point-cloud
 * upsampler (reference: generation.py:122-172 + fn/snn_coder.py + fd/snn_coder.py).
 *
 * The reference has no FFI of its own (SURVEY.md section 8b): its boundary is the
 * Python level (Generator3D6, fn/fd nn.Modules).  Every entry point below names the
 * reference call site it replaces; the Python shims in the package bind them with
 * ctypes (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in signatures (a stream is `void*`,
 *     i.e. a cudaStream_t; NULL = legacy default stream).
 *   - pointers named d_* are DEVICE pointers borrowed from the caller (never freed,
 *     never retained after the call returns); h_* are HOST pointers.
 *   - every function returns 0 on success or a negative SAPCU_E* code and never
 *     throws; sapcu_last_error() returns a thread-local description.
 *   - nothing here allocates device memory except sapcu_model_finalize (the model's
 *     own weights); scratch space is always a caller-provided workspace.
 *   - there is NO CPU fallback: without a CUDA device every compute entry fails.
 */
#ifndef SAPCU_B200_H
#define SAPCU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAPCU_OK            0
#define SAPCU_EINVAL       -1   /* bad argument (shape, null pointer, unsupported size) */
#define SAPCU_ECUDA        -2   /* a CUDA runtime call or kernel launch failed */
#define SAPCU_EWORKSPACE   -3   /* workspace too small for even one patch */
#define SAPCU_ESTATE       -4   /* model not finalized / missing tensor / handle used on another device */

#define SAPCU_MODEL_FN      0   /* ImprovedSNNNormalEstimation   (fn/snn_coder.py:627) */
#define SAPCU_MODEL_FD      1   /* EnhancedSNNDistanceEstimation (fd/snn_coder.py:805) */

/* arithmetic modes of the dense contractions */
#define SAPCU_MODE_FP32     0   /* fp32 FFMA everywhere: the "fp32 parity mode" */
#define SAPCU_MODE_TC       1   /* tcgen05 tensor-core contractions with 3 split products per MAC (fp16 hi/lo planes where the
                                   input is a spike tensor, tf32 hi/lo elsewhere; fp32-grade products, fp32 accumulate):
                                   meets the fp32-parity tolerances; the mode configs[1] is benchmarked in */
#define SAPCU_MODE_TF32     2   /* tcgen05 single-pass TF32 contractions (10-bit mantissa operands), fp32-grade neuron;
                                   deviation reported separately */
#define SAPCU_MODE_FAST     3   /* the fast tensor-core mode: ONE fp16 product per MAC on fp16 spike tensors (single-pass
                                   TF32 where the input is not a spike tensor), reduced-MUFU / tabulated LIF^T chains;
                                   deviation reported separately (profiles/, tests/test_gpu_parity.py) */

const char* sapcu_last_error(void);
int         sapcu_abi_version(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
int64_t     sapcu_launch_count(void);

/* Live kernel timing for bench.py's roofline line: when enabled, every contraction launch (the dominant kernel
 * family) is bracketed by CUDA events on its launch stream.  sapcu_profile_read synchronises those events and
 * returns their summed duration, the algorithmic FLOPs (2*R*K*N per launch) and the launch count since enable. */
/* Pipeline-watchdog status of the CURRENT CUDA device.  Every mbarrier wait of the tensor-core kernels carries a clock
 * watchdog: a protocol stall makes the kernel exit and raises a host-visible flag instead of hanging the GPU.  The
 * forwards poll that flag (no stream synchronisation) on entry and exit, so a stall is reported at the latest by the next
 * call; after synchronising the stream the caller can ask directly: 0 = fine, SAPCU_ECUDA = a kernel stalled since the
 * last query (results of the affected call are invalid).  SAPCU_TC_SYNC_CHECK=1 restores a synchronising check inside
 * every forward. */
int sapcu_device_status(void);

int sapcu_profile(int enable);
int sapcu_profile_read(double* gemm_ms, double* gemm_flops, int64_t* gemm_launches);
/* Per-kernel report of the same recording as JSON text: [{"label", "launches", "ms", "flops", "lif_elsteps", "bytes"}, ...]
 * (one entry per kernel label of the fn / fd forwards; algorithmic work per label, summed durations).  Writes at most
 * cap bytes (NUL-terminated) and returns the size needed, or a negative error code. */
int64_t sapcu_profile_report(char* h_buf, size_t cap);

/* ------------------------------------------------------------------------------------
 * K1  seed -> input-cloud kNN.  Replaces sklearn KDTree(data).query(chunk, K)
 *     (generation.py:110,127,153).  Exact: ordering by fp64 squared distance
 *     accumulated as ((dx*dx)+(dy*dy))+(dz*dz) without contraction, ties broken by the lowest
 *     cloud index; d_idx[s*K + j] ascending in distance.  K <= 128, K <= N.
 * ---------------------------------------------------------------------------------- */
size_t sapcu_knn_workspace_bytes(int64_t N);   /* fp32 SoA copy of the cloud + one scalar */
int sapcu_knn(const double* d_cloud, int64_t N, const double* d_seeds, int64_t S, int K,
              int32_t* d_idx, void* d_ws, size_t ws_bytes, void* stream);

/* Batched form: B independent (cloud, seed set) problems in ONE launch -- the per-file loop of generate.py:135-160
 * (one KDTree per input file) for a batch of small clouds.  d_clouds / d_seeds are the concatenated [N_total,3] /
 * [S_total,3] fp64 arrays, h_cloud_off / h_seed_off HOST prefix tables of B+1 entries (first 0, last the total).
 * Seeds of problem b see only cloud b; d_idx[s*K + j] is a row of the CONCATENATED cloud array (cloud-local index +
 * h_cloud_off[b]), so sapcu_gather_center_rotate runs on the concatenated arrays unchanged.  Same exactness and
 * tie-break as sapcu_knn; every non-empty problem needs N_b >= K.  Synchronises the stream once (offset upload). */
size_t sapcu_knn_batched_workspace_bytes(int64_t N_total, int B);
int sapcu_knn_batched(const double* d_clouds, const int64_t* h_cloud_off, const double* d_seeds,
                      const int64_t* h_seed_off, int B, int K, int32_t* d_idx,
                      void* d_ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * K2  gather + centre (+ rotate).  Replaces data[idx] - seed and the per-seed Rodrigues
 *     loop (generation.py:128-129,154-160, rotation_matrix_from_vectors :30-47).
 *     d_patches[s][j][:] = (float) R_s * (cloud[idx[s][j]] - seed[s])   (fp64 until the cast)
 *     d_normals == NULL  -> R_s = I (the fn pass); otherwise R_s rotates normal_s onto +x.
 * ---------------------------------------------------------------------------------- */
int sapcu_gather_center_rotate(const double* d_cloud, int64_t N, const double* d_seeds,
                               const int32_t* d_idx, int64_t S, int K,
                               const float* d_normals, float* d_patches, void* stream);

/* F.normalize(n, dim=-1) of generation.py:139, in place on [S,3] fp32. */
int sapcu_renormalize(float* d_normals, int64_t S, void* stream);

/* displacement, generation.py:171-172: out = seed + (double)(n * d)  (product in fp32). */
int sapcu_displace(const double* d_seeds, const float* d_normals, const float* d_dist,
                   int64_t S, double* d_out, void* stream);

/* ------------------------------------------------------------------------------------
 * Seed generator ("next" row 1).  Replaces the `./dense <cell> <N>` process + test.xyz/target.xyz file IPC of
 * generation.py:113-118 (dense.cpp:175-252): voxel flood fill from the occupied cells, a voxel centre is a seed when
 * its distance to the local triangle fan of its 10 nearest input points lies in [0.011, 0.015].  Same seeds in the
 * same (FIFO) order as the reference binary.  quirk_origin != 0 keeps the reference's extra all-zero point in the
 * 10-NN search (dense.cpp:193); round6 != 0 rounds coordinates to 6 decimals like the "%lf" text round trip.
 * d_seeds: [cap,3] f64 (first min(count, cap) seeds are stored); *h_count (HOST) receives the total count.
 * Synchronises the stream once per flood-fill level.
 * ---------------------------------------------------------------------------------- */
size_t sapcu_seedgen_workspace_bytes(int64_t N, double cell, int64_t cap);
int sapcu_seedgen(const double* d_cloud, int64_t N, double cell, int quirk_origin, int round6,
                  double* d_seeds, int64_t cap, int64_t* h_count, void* d_ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Outlier filter ("next" row 2), generation.py:176-183: with d_idx = the k = 30 self-neighbours of every output point
 * (sapcu_knn with cloud == seeds == points), keep[i] = mean_j |p_i - p_idx[i][j]| < threshold * (global mean).
 * ---------------------------------------------------------------------------------- */
size_t sapcu_outlier_workspace_bytes(int64_t S);
int sapcu_outlier_mask(const double* d_points, int64_t S, const int32_t* d_idx, int K, double threshold,
                       uint8_t* d_keep, void* d_ws, size_t ws_bytes, void* stream);

/* The same filter over seeds sharded across GPUs (SURVEY.md section 8f-2: "needs a global mean"): after the all-gather
 * of the displaced points every rank holds all S points; it queries the kNN of ITS rows (sapcu_knn with cloud = all
 * points, seeds = its rows), computes their mean neighbour distances with sapcu_knn_mean_dist, the row means are
 * all-gathered (S doubles), and sapcu_outlier_mask_from_means sums them in one fixed order -- the order of the
 * single-GPU filter -- and masks the rank's rows [row_lo, row_lo + rows): the survivors are bit-identical to
 * sapcu_outlier_mask for any number of ranks.  d_ws: 256 bytes. */
int sapcu_knn_mean_dist(const double* d_points, int64_t S, const double* d_query, int64_t rows,
                        const int32_t* d_idx, int K, double* d_mean, void* stream);
int sapcu_outlier_mask_from_means(const double* d_mean_all, int64_t S, int64_t row_lo, int64_t rows, double threshold,
                                  uint8_t* d_keep, void* d_ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Farthest point sampling ("next" row 3), generate.py:56-74: fp32, start index `start` (the reference uses N/2),
 * running distances initialised to 1e32, ties -> lowest index.  d_out: int32 [npoint] selected indices in order.
 * One cooperative persistent kernel (a grid barrier per selected point); workspace: 32 bytes.
 * ---------------------------------------------------------------------------------- */
int sapcu_fps(const float* d_xyz, int64_t N, int64_t npoint, int64_t start, int32_t* d_out,
              void* d_ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Normal orientation (no reference counterpart; the spanning-tree propagation of Hoppe et al., Open3D's
 * orient_normals_consistent_tangent_plane): flips the signs of unit normals so that neighbours agree (csrc/orient.cu).
 *   graph   undirected, edges {i, d_idx[i*k + j]} for j < k; entries equal to i are skipped (with duplicated points the
 *           self entry is not always in column 0), and so are entries outside [0, S).  Intended input: sapcu_knn with cloud = seeds =
 *           d_points and K = k.  1 <= k <= 128, S >= 1, S*k < 2^31, else SAPCU_EINVAL; a short workspace: SAPCU_EWORKSPACE.
 *   edge    dot = ((nx_i*nx_j) + (ny_i*ny_j)) + nz_i*nz_j in fp64 from the fp32 components, without contraction (a numpy
 *           restatement gives the same bits); a flip edge has dot < 0; its weight is |dot|.
 *   forest  the maximum spanning forest under the strict order: larger |dot| first, then the smaller (min(i,j), max(i,j))
 *           pair -- unique, independent of the launch configuration and of the order in which atomics land.
 *   root    per connected component the point with the largest z (ties -> lowest index); it keeps its normal when
 *           nz >= 0 and is negated when nz < 0 (outward at the topmost point of a closed surface).
 *   others  negated when the root was negated XOR the tree path from the root holds an odd number of flip edges.
 * d_normals: [S,3] fp32, oriented in place -- every output is bitwise its input or the exact negation of it (sign bit).
 * d_root (nullable): int32 [S], each point's root index.  d_points: [S,3] f64 (only z is read).  Allocates nothing and
 * does not synchronise the stream.
 * ---------------------------------------------------------------------------------- */
size_t sapcu_orient_normals_workspace_bytes(int64_t S, int k);   /* 0 for arguments outside the limits above */
int sapcu_orient_normals(const double* d_points, int64_t S, const int32_t* d_idx, int k,
                         float* d_normals, int32_t* d_root, void* d_ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Point-to-mesh distance (no reference counterpart; the P2F metric of the upsampling literature, computed there on the
 * host with CGAL): the exact squared distance from every query point to a triangle mesh (csrc/mesh_dist.cu).
 *   distance  d_dist2[s] = min over faces f of D(p_s, f).  D is ((dx*dx)+(dy*dy))+(dz*dz) in fp64 without contraction,
 *             from p_s to q, where q is the closest point on the triangle (a, b, c) = d_vertices[d_faces[f]] of the shared
 *             routine (csrc/geom.cuh, Ericson's region test in the operation order of the reference's dense.cpp), with
 *             two additions: when a coordinate of that point is not finite (the 0/0 of a degenerate face: two coincident
 *             vertices, or a zero normal) q is the closest of the three segment points of ab, bc, ca, each
 *             a + e*t with e = b - a, t = ((p-a).e)/(e.e) clamped to [0, 1] (t = 0 when e.e == 0), the first of equal
 *             distances; and q is then clamped coordinate-wise into the face's box [min, max of the vertex coordinates]
 *             (which holds the exact closest point, so the clamp only moves q towards it).  No input gives NaN.
 *   face      d_face[s] (nullable): the face attaining the minimum; ties (bitwise-equal D) go to the lowest face index.
 *             -1 (and d_dist2 = +inf) when no face is valid.
 *   order     the result does not depend on the tree, the launch configuration or the order of the query points: it is
 *             bitwise the brute-force minimum of (D, face index).
 *   limits    V >= 1, 1 <= F < 2^31, S >= 0, else SAPCU_EINVAL; S == 0 is a no-op; a short workspace: SAPCU_EWORKSPACE.
 *             Faces with an index outside [0, V) are skipped, so no input makes a kernel read outside its arrays.
 *   method    one linear BVH per call (Karras 2012) over the faces' centroid Morton codes, built and queried on the device.
 * d_vertices: [V,3] f64, d_faces: [F,3] int32, d_points: [S,3] f64, d_dist2: [S] f64.  Allocates nothing and does not
 * synchronise the stream.  The workspace size is a closed form of F (about 200 bytes per face), computed without a device.
 * ---------------------------------------------------------------------------------- */
size_t sapcu_mesh_distance_workspace_bytes(int64_t V, int64_t F);   /* 0 for arguments outside the limits above */
int sapcu_mesh_distance(const double* d_vertices, int64_t V, const int32_t* d_faces, int64_t F,
                        const double* d_points, int64_t S, double* d_dist2, int32_t* d_face,
                        void* d_ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Models.  A handle is built from the same hyper-parameters get_model() consumes
 * (fn/config.py:183-210, fd/config.py:89-117) and the tensors of the module's
 * state_dict (host fp32 pointers, names = state_dict keys, SURVEY.md section 8b).
 *   fn cfg ints : { k0, k1, k2, emb_dims, time_steps_enc, num_heads }
 *   fd cfg ints : { k, emb_dims, time_steps_enc, num_heads, n_scales, k_scale_0 .. }
 * After finalize the handle is immutable (weights, folded parameters, LIF tables) and may be used from several host
 * threads / streams concurrently, each call with its own workspace; per-device kernel attributes and the watchdog flag are
 * set up under a lock on first use of a device, the A/B environment switches are read once per process.  A handle's
 * weights live on the CUDA device that was current at finalize, and the handle records that device:
 * sapcu_fn_forward / sapcu_fd_forward return SAPCU_ESTATE, before any launch, when another device is current, and
 * sapcu_model_destroy frees on the recorded device and leaves the caller's current device unchanged.  One handle per
 * device: finalize a separate handle for every GPU that runs the model.
 * ---------------------------------------------------------------------------------- */
typedef struct sapcu_model sapcu_model;

sapcu_model* sapcu_model_create(int kind, const int32_t* cfg, int ncfg);
int  sapcu_model_set_tensor(sapcu_model* m, const char* name, const float* h_data, int64_t numel);
int  sapcu_model_finalize(sapcu_model* m);       /* folds eval-mode BN, clamps neuron params, uploads */
void sapcu_model_destroy(sapcu_model* m);

/* workspace needed to run `S` patches of M points in ONE internal chunk (forward accepts
 * less and chunks internally; it needs at least the size for S = 1). */
size_t sapcu_model_workspace_bytes(const sapcu_model* m, int64_t S, int M);

/* fn: ImprovedSNNNormalEstimation.forward([S,M,3]) -> [S,3] unit normals (fn/snn_coder.py:670-699).
 * `mode`: bits 0-7 = SAPCU_MODE_*; bits 8-11 (tests only) = b in 1..3: stop after transformer block b, leaving ITS
 * intermediates in the workspace for sapcu_model_tap ("trans<b>.*") -- the normals are then not written. */
int sapcu_fn_forward(const sapcu_model* m, const float* d_patches, int64_t S, int M,
                     float* d_normals, void* d_ws, size_t ws_bytes, int mode, void* stream);

/* fd: EnhancedSNNDistanceEstimation.forward([S,M,3]) -> [S] distances (fd/snn_coder.py:853-871).
 * d_forced_idx (nullable): int32 [3][S][M][k] feature-space neighbour lists for blocks 1..3 taken
 * from the oracle ("teacher-forced" parity runs, SURVEY.md section 7 hard-part 4). */
int sapcu_fd_forward(const sapcu_model* m, const float* d_patches, int64_t S, int M,
                     float* d_dist, const int32_t* d_forced_idx,
                     void* d_ws, size_t ws_bytes, int mode, void* stream);

/* Debug taps for the parity tests: location of a named intermediate inside the workspace of the
 * LAST chunk a forward call of the given `mode` processed (valid when S fits one chunk).  Element (row r, col c) is at
 * float offset  off + r*ld + c.  Returns SAPCU_EINVAL for an unknown name.  fn: "idx", "snn_init", "fcat", "trans<b>.{snn1,
 * snn_qkv,snn_delta2,snn_gamma,logits,res}" (b = the last block the forward executed), "snn_final", "gmax", "enc_out", "dec_h3";
 * fd: "idx0", "idxf1".."idxf3" (feature-space graphs of blocks 1..3), "f0", "u0".."u3", "spikes", "pool", "z", "dec_d2", "dec_hidden". */
int sapcu_model_tap(const sapcu_model* m, const char* name, int64_t S, int M, int mode,
                    int64_t* off_floats, int64_t* rows, int64_t* cols, int64_t* ld);
/* Storage format the most recent forward used for a tap: 0 = fp32 [rows, ld]; 1 = two consecutive fp16 planes
 * [rows, cols] (hi, then lo) of x * 2^13, i.e. x = (hi + lo) / 8192 -- the hand-over format between an epilogue and the
 * fp16x3 contraction that consumes its spikes (MODE_TC, 'trans3.snn_gamma'); 2 = ONE fp16 plane [rows, cols] of x * 2^13
 * (MODE_FAST).  Negative: error code. */
int sapcu_model_tap_format(const sapcu_model* m, const char* name);

/* ------------------------------------------------------------------------------------
 * Stand-alone operators exported for unit parity tests (each is used by the forwards above).
 * ---------------------------------------------------------------------------------- */
/* LIF^T / EIF^T chain from the zero state (fn/snn_coder.py:87-153, fd/snn_coder.py:198-275 applied T
 * times, each step's soft spike fed back as the next step's input):
 * d_params4 = [4][C] rows {decay, adapt, refr_decay, theta0}, ALREADY CLAMPED to the reference's ranges;
 * d_eif2 (nullable -> LIF) = [2][C] rows {delta_T, theta_rh}, clamped.
 * x: [rows, C] row-major.  all_steps == 0 -> out [rows, C] = last step's spikes;
 * all_steps != 0 -> out [rows, T, C] holds every step's spikes. */
int sapcu_lif_chain(const float* d_x, int64_t rows, int C, int T, const float* d_params4,
                    const float* d_eif2 /*nullable {delta_T, theta_rh}*/, int all_steps,
                    float* d_out, void* stream);
/* HOST-ONLY self-test of the tabulated LIF^T chains (no GPU, no stream): builds the table for h_params4 = [4][C] rows {decay, adapt,
 * refr_decay, theta0} (HOST memory, already clamped) and T steps exactly as sapcu_model_finalize does, evaluates the host restatement
 * of the kernels' lookup at `samples` magnitudes per side and channel (geometric over 2^-12 .. 254.9) plus zero, the cell boundaries
 * and their fp32 neighbours, and reports max_err = the largest |table - exact fp64 chain| (the reference's recurrence,
 * fn/snn_coder.py:87-153), fit_err = the builder's own acceptance figure and the largest 128-channel block image in bytes. */
int sapcu_lif_table_selftest(const float* h_params4, int C, int T, int samples, double* max_err, double* fit_err,
                             uint32_t* max_block_bytes);
/* intra-patch kNN of fn/fd `knn()` (fn/snn_coder.py:31-39, fd/snn_coder.py:25-32): features
 * [S*M, C] rows (ld floats apart), top-k of -|xi-xj|^2 in the reference's expanded form, ties -> lowest
 * index.  d_idx: int32 [S*M, k] patch-local indices. */
int sapcu_intra_knn(const float* d_feat, int64_t ld, int64_t S, int M, int C, int k,
                    int32_t* d_idx, void* stream);
/* Y[R,N] = X[R,K] * W[N,K]^T  (+bias) in the selected mode; exported to test the GEMM engines. */
int sapcu_gemm(const float* d_x, int64_t R, int K, const float* d_w, int N, const float* d_bias,
               float* d_y, int mode, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SAPCU_B200_H */
