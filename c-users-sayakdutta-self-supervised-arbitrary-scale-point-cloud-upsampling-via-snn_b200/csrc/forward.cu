// fn / fd forward orchestration: workspace plans, chunking over patches, the layer schedule.
//
// Schedule notes (exactness-preserving, see DESIGN.md):
//  * every `for t in range(T): x, *st = lif(x, *st)` chain of fn is evaluated as one element-wise function
//    fused into the epilogue of the contraction that produces its input (the fed-back spike is gated
//    to zero by the refractory term after step 0, but the gate is still evaluated literally);
//  * fd's time loop (fd/snn_coder.py:408-480) feeds each block's conv output through a gate that is
//    closed for t >= 1, so the graph convolutions and feature-space kNN are evaluated once (t = 0) and
//    only the neuron recurrences + the 960 -> emb contraction + max-pool run for all T steps.
#include <stdlib.h>
#include "../../include/sapcu_b200.h"
#include "gemm_simt.cuh"
#include "gemm_tc.h"
#include "kernels.h"
#include "model.h"
#include "lif_table.cuh"

using namespace sapcu;

namespace {

struct Bump {
  char* base; size_t off = 0;
  explicit Bump(void* b) : base(reinterpret_cast<char*>(b)) {}
  template <class T> T* take(size_t n) {
    off = align_up(off, 256);
    T* p = reinterpret_cast<T*>(base + off);
    off += n * sizeof(T);
    return p;
  }
};

struct FnPlan {
  int32_t* idx; uint32_t* idx8; float *F0, *FCAT, *X, *QKV, *QK, *E1, *E2, *E3, *RES, *R1, *G, *GM, *H0, *H1, *H2, *H3;
  size_t bytes; int kmax; int Dl, kl;
  PairBufs pairs;        // sapcu_fn_forward_indexed: the chunk's pair table (Ncloud > 0)
};
// Ncloud > 0: also the pair table of a chunk whose patch points are rows of a cloud of Ncloud points
FnPlan fn_plan(const FnNet& f, int64_t s, int M, void* base, int64_t Ncloud = 0) {
  FnPlan p; Bump b(base);
  const int64_t P = s * M;
  p.kmax = 0; size_t emax = 0;
  for (int i = 0; i < 3; ++i) {
    const int k = f.blk[i].k < M ? f.blk[i].k : M;
    p.kmax = k > p.kmax ? k : p.kmax;
    emax = (size_t)k * f.blk[i].D > emax ? (size_t)k * f.blk[i].D : emax;
  }
  p.idx = b.take<int32_t>(P * p.kmax);
  p.idx8 = b.take<uint32_t>(P * ((p.kmax + 3) / 4));       // byte-packed copy of the graph for the fused attention tails
  p.F0 = b.take<float>(P * 64); p.FCAT = b.take<float>(P * 192);
  p.X = b.take<float>(P * 512); p.QKV = b.take<float>(P * 1536);
  p.QK = b.take<float>(P * 1024);              // [W q | W k] per point (factorised attention input)
  p.E1 = b.take<float>(P * emax); p.E2 = b.take<float>(P * emax); p.E3 = b.take<float>(P * emax);
  p.RES = b.take<float>(P * 512); p.R1 = b.take<float>(P * 512);
  p.G = b.take<float>(P * f.emb); p.GM = b.take<float>(s * f.emb);
  p.H0 = b.take<float>(s * 2048); p.H1 = b.take<float>(s * 1024); p.H2 = b.take<float>(s * 512); p.H3 = b.take<float>(s * 256);
  if (Ncloud > 0) {
    int kk[3];
    for (int i = 0; i < 3; ++i) kk[i] = f.blk[i].k < M ? f.blk[i].k : M;
    char* pb = b.take<char>(0);
    p.pairs = pair_plan(P, p.kmax, kk, Ncloud, base ? pb : nullptr);
    b.off += p.pairs.bytes;
  }
  p.bytes = align_up(b.off, 256);
  p.Dl = f.blk[2].D; p.kl = f.blk[2].k < M ? f.blk[2].k : M;
  return p;
}

struct FdPlan {
  int32_t *idx0, *idxf[3]; float *F0, *U0, *U1, *U2, *U3, *PQ, *SPK, *SPK0, *AGG, *EDGE, *POOL, *Z, *D0, *T1, *R, *D1, *D2, *QKV, *O, *AO, *LN, *HH;
  size_t bytes; int k, kmax0;
};
FdPlan fd_plan(const FdNet& f, int64_t s, int M, void* base) {
  FdPlan p; Bump b(base);
  const int64_t P = s * M;
  p.k = f.k < M ? f.k : M;
  p.kmax0 = f.kscales[f.nscales - 1] < M ? f.kscales[f.nscales - 1] : M;
  p.idx0 = b.take<int32_t>(P * p.kmax0);
  for (int i = 0; i < 3; ++i) p.idxf[i] = b.take<int32_t>(P * p.k);     // the feature-space graph of every block stays available (parity taps)
  p.F0 = b.take<float>(P * 64 * f.nscales);
  p.U0 = b.take<float>(P * 64); p.U1 = b.take<float>(P * 128); p.U2 = b.take<float>(P * 256); p.U3 = b.take<float>(P * 512);
  p.PQ = b.take<float>(P * 1024);          // factorised EdgeConv (P | Q) rows, tensor-core mode
  p.SPK = b.take<float>(P * f.T * 960);
  p.SPK0 = b.take<float>(P * 960);         // fp32 copy of the step-0 spikes when SPK holds fp16 planes (tensor-core modes)
  p.AGG = b.take<float>(P * f.T * f.emb);
  // MODE_FP32 with a neighbour count other than 32 (the fused 32-row max of the SIMT engine): per-edge EdgeConv activations
  p.EDGE = p.k != 32 ? b.take<float>(P * (int64_t)p.k * 512) : nullptr;
  p.POOL = b.take<float>(s * f.T * f.emb); p.Z = b.take<float>(s * f.emb);
  p.D0 = b.take<float>(s * 256); p.T1 = b.take<float>(s * 128); p.R = b.take<float>(s * 128);
  p.D1 = b.take<float>(s * 128); p.D2 = b.take<float>(s * 64); p.QKV = b.take<float>(s * 192);
  p.O = b.take<float>(s * 64); p.AO = b.take<float>(s * 64); p.LN = b.take<float>(s * 64); p.HH = b.take<float>(s * 32);
  p.bytes = align_up(b.off, 256);
  return p;
}

int64_t pick_chunk(const sapcu_model* m, int64_t S, int M, size_t ws_bytes, int64_t Ncloud = 0) {
  auto need = [&](int64_t s) {
    return m->kind == SAPCU_MODEL_FN ? fn_plan(m->fn, s, M, nullptr, Ncloud).bytes : fd_plan(m->fd, s, M, nullptr).bytes;
  };
  if (need(S) <= ws_bytes) return S;
  int64_t lo = 0, hi = S;   // need(lo) fits (lo = 0 trivially), need(hi) does not
  while (hi - lo > 1) { const int64_t mid = (lo + hi) / 2; if (need(mid) <= ws_bytes) lo = mid; else hi = mid; }
  return lo;
}

// ---- GEMM helper: dispatch on the arithmetic mode
struct G {
  int mode; cudaStream_t st;
  mutable const char* lab = nullptr;                       // profiler label of the next launch: g.L("fn.fc1").layer(...)
  const G& L(const char* l) const { lab = l; return *this; }
  int passes() const { return mode == SAPCU_MODE_TF32 || mode == SAPCU_MODE_FAST ? 1 : 3; }   // tensor-core products per MAC
  int run(GemmArgs g, int amode) const {
    if (lab) { g.label = lab; lab = nullptr; }
    int slot = -1;
    ProfWork w;
    w.gemm = true;
    w.flops = 2.0 * (double)g.R * g.K * g.N;
    if (g.act == ACT_LIF) w.elsteps = (double)g.R * g.N * g.T;
    {   // algorithmic HBM bytes: the activation read once, the result written once (fp16 planes keep the fp32 byte count), the weights once
      const double out_rows = g.at_pos ? (double)g.R / (g.kk > 0 ? g.kk : 1) : (g.pool ? (double)g.R / (g.pool_M > 0 ? g.pool_M : 1) : (double)g.R);
      w.bytes = (double)g.R * g.K * 4.0 + out_rows * g.N * 4.0 + (double)g.N * g.K * 4.0;
      if (g.at_pos) w.bytes += (double)g.R * g.N * 4.0;             // pos rows read by the fused attention tail
    }
    if (g.R_dev) { w = ProfWork{}; w.gemm = true; }          // rows counted on the device: no algorithmic work recorded
    const bool prof = prof_begin(st, g.label, w, &slot);
    int rc;
    g.tc_passes = passes();
    // fast mode, plain point-level contractions: single-pass TF32 needs no operand split -> the compact-stage flavour
    if (mode == SAPCU_MODE_FAST && amode == A_PLAIN && g.act == ACT_NONE && !g.residual && !g.at_pos && !g.pool && !g.x_h2 && !g.out_h2 && !g.edge_bias) g.fast = true;
    if (mode != SAPCU_MODE_FP32 && gemm_tc2_supported(g, amode)) rc = launch_gemm_tc2(g, st);
    else if (mode != SAPCU_MODE_FP32 && gemm_tc_supported(g, amode)) rc = launch_gemm_tc(g, amode, st);
    else rc = launch_gemm_simt(g, amode, mode == SAPCU_MODE_FP32, st);
    if (prof) prof_end(st, slot);
    return rc;
  }
  // plain layer: Y[R, L.N] (ldc) = act(affine(X[R, L.K] (lda)))
  GemmArgs args(const Layer& L, const float* X, int64_t lda, int64_t R, float* Y, int64_t ldc, int act,
                const Neuron* nr = nullptr, int T = 0, const float* res = nullptr, int64_t ldr = 0, bool x_unit = false) const {
    GemmArgs g;
    g.A = X; g.lda = lda; g.R = R; g.K = L.K; g.W = L.W; g.Whi = L.Whi; g.Wlo = L.Wlo; g.N = L.N; g.bias = L.bias; g.scale = L.scale; g.shift = L.shift;
    g.Wh = L.Wh; g.Wl = L.Wl; g.winv = L.winv; g.x_unit = x_unit;
    g.act = act; g.T = T; g.nparams = nr ? nr->np : nullptr; g.residual = res; g.ldr = ldr; g.Y = Y; g.ldc = ldc;
    g.tc_passes = passes();
    if (mode == SAPCU_MODE_FAST && act == ACT_LIF && nr) {     // point-level LIF layers: compact single-pass TF32 stages + the layer's LIF table
      g.fast = true;
      if (settings().fast_tables && nr->tab_ok && nr->tab_T == T) { g.lif_tab = nr->tab; g.lif_tab_stride = nr->tab_stride; }
    }
    return g;
  }
  int layer(const Layer& L, const float* X, int64_t lda, int64_t R, float* Y, int64_t ldc, int act,
            const Neuron* nr = nullptr, int T = 0, const float* res = nullptr, int64_t ldr = 0, bool x_unit = false) const {
    GemmArgs g = args(L, X, lda, R, Y, ldc, act, nr, T, res, ldr, x_unit);
    return run(g, A_PLAIN);
  }
};

// The storage format of the tapped spike tensors (0 fp32, 1 fp16 (hi, lo) planes of x * 2^13, 2 one fp16 plane) is recorded
// in the handle by every forward (sapcu_model::tap_*): debug information for the parity tests, relaxed atomics.

#define SAPCU_TRY(expr) do { int _rc = (expr); if (_rc) return _rc; } while (0)

// One fn block's hand-over formats, in the tap codes above, and the LIF tables and fusions that go with them. plan() in
// fn_chunk fills it before the block's first launch; the launch sequence reads nothing else.
struct BlockPlan {
  int x_planes = 0;      // fc1 -> q/k/v
  int delta = 0;         // pos-enc layer 1 -> fc_delta2
  int pos = 0;           // pos (fc_delta2's spikes) -> fc_gamma and the attention tail
  bool pos32 = false;    // fc_delta2 also writes pos in fp32 (E3), and the attention tail reads that copy
  int gamma = 0;         // fc_gamma -> fc_gamma2
  // LIF chains read from the layer's table (in the fast mode fc1 and q/k/v take theirs in G::args, as every point-level layer)
  bool tab_fc1 = false, tab_qkv = false, tab_delta = false, tab_delta2 = false, tab_gamma = false;
  bool attn_in = false;  // factorised attention input: [W q | W k] per point + fc_gamma's edge-bias epilogue
  bool attn_out = false; // fc_gamma2 with the fused softmax + weighted-sum tail
};

// Where the chunk's patch points come from (sapcu_fn_forward_indexed): gidx[s*ldg + i] = cloud row of patch point i
struct PatchSource { const double* cloud = nullptr; int64_t N = 0; const int32_t* gidx = nullptr; int64_t ldg = 0; };

int fn_chunk(const sapcu_model* mdl, const float* xyz, int64_t s, int M, float* normals, const FnPlan& p, int mode, int stop_block, cudaStream_t st,
             const PatchSource* src = nullptr) {
  const FnNet& f = mdl->fn;
  const int64_t P = s * M;
  const bool precise = mode == SAPCU_MODE_FP32;
  const G g{mode, st};
  { ProfWork w; w.flops = (double)s * M * M * 3; w.bytes = (double)P * (12 + 4.0 * p.kmax);
    SAPCU_PROF(st, "fn.intra_knn(xyz)", w, launch_intra_knn(xyz, 3, s, M, 3, p.kmax, p.idx, st)); }
  if (mode != SAPCU_MODE_FP32 && M <= 256) SAPCU_TRY(launch_pack_idx_u8(p.idx, p.kmax, P, p.idx8, st));
  // the pair table serves the blocks that evaluate pos once per distinct point pair (see `pairs` below), built by the first
  // of them (parity-grade mode only: in the fast mode the per-edge schedule measured faster, 112 vs 115 ms per 8,192 seeds)
  const bool indexed = src && mode == SAPCU_MODE_TC;
  bool table_built = false;
  { ProfWork w; w.elsteps = (double)P * 64 * f.T_enc; w.bytes = (double)P * (12 + 256);
    SAPCU_PROF(st, "fn.conv1+lif", w, launch_pointwise3_lif(false, precise, xyz, nullptr, 0, 0, M, P, 64, f.conv1.W, f.conv1.bias, f.conv1.scale,
                                  f.conv1.shift, f.snn_init.np, f.T_enc, p.F0, st)); }
  const bool use_tables = settings().fast_tables;       // 0: reduced-MUFU chains (A/B)
  auto fits = [](const Neuron& n, uint32_t budget) { return n.tab_ok && n.tab_T == 4 && n.tab_stride <= budget; };
  auto sup2 = [](const GemmArgs& a) { return gemm_tc2_supported(a, A_PLAIN); };
  for (int b = 0; b < 3; ++b) {
    if (stop_block && b >= stop_block) return 0;            // debug: leave block `stop_block`'s intermediates in the workspace
    const FnBlock& k = f.blk[b];
    const int D = k.D, kk = k.k < M ? k.k : M;
    const float* fin = b == 0 ? p.F0 : p.FCAT + 64 * (b - 1);
    const int64_t ldin = b == 0 ? 64 : 192;
    const int64_t E = P * kk;
    const float sq = sqrtf((float)(D / f.heads));           // torch divides the logits by the python scalar sqrt(head_dim)
    // ---- the contractions whose operand formats the plan chooses: one builder each, used to probe and to launch
    auto fc1_args = [&](const BlockPlan& q) {
      GemmArgs a = g.args(k.fc1, fin, ldin, P, p.X, D, ACT_LIF, &k.snn1, 4);
      a.out_h2 = a.tc2_any_rows = q.x_planes != 0;
      if (q.tab_fc1) { a.lif_tab = k.snn1.tab; a.lif_tab_stride = k.snn1.tab_stride; }
      return a;
    };
    auto qkv_args = [&](const BlockPlan& q) {
      GemmArgs a = g.args(k.qkv, p.X, D, P, p.QKV, 3 * D, ACT_LIF, &k.snn_qkv, 4, nullptr, 0, q.x_planes != 0);
      a.x_h2 = a.tc2_any_rows = q.x_planes != 0;
      if (q.tab_qkv) { a.lif_tab = k.snn_qkv.tab; a.lif_tab_stride = k.snn_qkv.tab_stride; }
      return a;
    };
    // per-edge contractions on LIF outputs: input format `in` (2 = the fast mode's single-product path), LIF output format `out`
    auto edge = [](GemmArgs a, int in, int out, const Neuron* n, bool tab) {
      a.x_h2 = in != 0; a.out_h2 = out != 0; a.fast = in == 2;
      a.lif_tab = tab ? n->tab : nullptr; a.lif_tab_stride = tab ? n->tab_stride : 0;
      return a;
    };
    auto delta2_args = [&](const BlockPlan& q) {
      GemmArgs a = edge(g.args(k.fc_delta2, p.E1, D, E, p.E2, D, ACT_LIF, &k.snn_delta2, 4, nullptr, 0, true), q.delta, q.pos,
                        &k.snn_delta2, q.tab_delta2);
      a.Y2 = q.pos32 ? p.E3 : nullptr;
      return a;
    };
    // fc_gamma's first layer is linear, so W(q_i - k_j + pos_ij) = W q_i - W k_j + W pos_ij: the edge contraction runs on
    // pos (E2) alone and its epilogue adds the two per-POINT products [W q | W k] (QK, [P, 2D]) gathered through the graph
    // before BN + LIF; fc_gamma2's epilogue does the softmax over k and the weighted sum.  Neither the attention input nor
    // the logits are materialised.
    auto gamma_args = [&](const BlockPlan& q) {
      GemmArgs a = edge(g.args(k.fc_gamma, p.E2, D, E, p.E1, D, ACT_LIF, &k.snn_gamma, 4, nullptr, 0, true), q.pos, q.gamma,
                        &k.snn_gamma, q.tab_gamma);
      a.Q = p.QK; a.Kf = p.QK + D; a.ldq = 2 * D; a.idx = p.idx; a.ldi = p.kmax; a.kk = kk; a.Mpts = M; a.edge_bias = true;
      return a;
    };
    auto gamma2_args = [&](const BlockPlan& q, float* gin = nullptr) {
      GemmArgs a = edge(g.args(k.fc_gamma2, gin ? gin : p.E1, D, E, p.RES, D, ACT_NONE, nullptr, 0, nullptr, 0, true), q.gamma, 0, nullptr, false);
      a.idx = p.idx; a.ldi = p.kmax; a.kk = kk; a.Mpts = M; a.idx8 = p.idx8; a.ldi8w = (p.kmax + 3) / 4;
      a.at_pos = q.pos32 ? p.E3 : p.E2; a.pos_h2 = q.pos != 0 && !q.pos32;
      a.at_v = p.QKV + 2 * D; a.at_ldv = 3 * D; a.at_sqrt = sq;
      return a;
    };
    // ---- the plan: asks the engines, in dependency order, which formats each producer / consumer pair takes; launches nothing
    auto plan = [&]() {
      BlockPlan q;
      if (mode == SAPCU_MODE_FP32) return q;
      if (mode == SAPCU_MODE_TC) {
        // Parity-grade mode, wide blocks: fc1's spikes have ONE reader, the q/k/v contraction -> handed over as fp16 (hi, lo)
        // planes in the bytes of the fp32 tensor; q/k/v then runs fp16x3 products (the 22-bit products of 3xTF32 at twice the
        // tensor rate, no splitter pass) and reads its LIF^T chains from the layer's table when it fits next to two stages.
        // fc1 itself keeps 3xTF32 products (its input is not a spike tensor) and reads its chain from the table as well.
        q.x_planes = 1;
        const GemmArgs a1 = fc1_args(q), a2 = qkv_args(q);
        q.x_planes = D % 256 == 0 && sup2(a1) && sup2(a2) && gemm_tc2_fp16x3(a2);
        q.tab_fc1 = q.x_planes && fits(k.snn1, LT_SMEM_BUDGET_TC);
        q.tab_qkv = q.x_planes && fits(k.snn_qkv, LT_SMEM_BUDGET_TC);
      }
      const bool factorise = settings().factor_attnin && kk >= 2;
      if (mode == SAPCU_MODE_FAST && factorise) {
        // Fast schedule: every per-edge spike tensor of the block is ONE fp16 plane of x * 2^13, every edge contraction one fp16
        // product per MAC (2-CTA kernel, HM = 3), every LIF^T chain a table lookup where the layer's table fits shared memory.
        BlockPlan t = q;
        t.delta = t.pos = t.gamma = 2;
        t.attn_in = t.attn_out = true;
        t.tab_delta = use_tables && fits(k.snn_delta, LT_SMEM_BUDGET);
        t.tab_delta2 = use_tables && fits(k.snn_delta2, LT_SMEM_BUDGET);
        t.tab_gamma = use_tables && fits(k.snn_gamma, LT_SMEM_BUDGET);
        const GemmArgs a = delta2_args(t), a1 = gamma_args(t), a2 = gamma2_args(t);
        if (sup2(a) && gemm_tc2_fast(a) && sup2(a1) && gemm_tc2_fast(a1) && sup2(a2) && gemm_tc2_fast(a2)) return t;
      }
      // Parity-grade mode with tabulated LIF^T chains: the three per-edge LIF layers of a block whose tables fit next to two
      // pipeline stages read their chains from the tables (lif_table.cuh, |error| <= 4e-5, far inside the spike tolerance); all
      // three edge tensors are then handed over as fp16 (hi, lo) planes.  Without the tables pos stays fp32 (measured slower as
      // planes: the attention tail then issues two 2-byte loads per operand instead of one 4-byte load).
      const bool blk_tab = mode == SAPCU_MODE_TC && factorise && fits(k.snn_delta, LT_SMEM_BUDGET) &&
                           fits(k.snn_delta2, LT_SMEM_BUDGET_TC) && fits(k.snn_gamma, LT_SMEM_BUDGET_TC);
      // fc_delta2 on the pos-enc layer-1 spikes: planes of x * 2^13 (same bytes as fp32) when it runs on the fp16x3 path,
      // which loads them without converting (128-channel layers run on the 2-CTA engine only from planes)
      q.delta = 1;
      const GemmArgs a = delta2_args(q);
      q.delta = sup2(a) && gemm_tc2_fp16x3(a);
      // pos has two readers, fc_gamma's contraction and the fused attention tail: planes when both take them
      q.pos = q.gamma = 1;
      const GemmArgs a1 = gamma_args(q), a2 = gamma2_args(q);
      q.pos = blk_tab && q.delta && sup2(a1) && gemm_tc2_fp16x3(a1) && sup2(a2) && gemm_tc2_fp16x3(a2);
      // the whole chain of plane hand-overs is in place: its producers read their tables, and the attention tail, which gathers
      // pos per edge, prefers one 4-byte load over two 2-byte loads -- with the table-driven (ALU-bound) epilogue the extra
      // fp32 store is free
      q.pos32 = q.tab_delta = q.tab_delta2 = q.pos;
      // fc_gamma's spikes go to fc_gamma2 only: planes when both run on the 2-CTA fp16x3 path
      const GemmArgs b1 = gamma_args(q), b2 = gamma2_args(q);
      q.gamma = factorise && sup2(b1) && sup2(b2) && gemm_tc2_fp16x3(b2);
      q.tab_gamma = blk_tab && q.pos && q.gamma;
      const GemmArgs c1 = gamma_args(q), c2 = gamma2_args(q);
      q.attn_in = factorise && (sup2(c1) || gemm_tc_supported(c1, A_PLAIN));
      q.attn_out = sup2(c2) || gemm_tc_supported(c2, A_PLAIN);
      return q;
    };
    const BlockPlan q = plan();
    // Pair schedule (indexed entry): pos = LIF(BN(W_d2 LIF(BN(W_d (p_i - p_j))))) is a function of the offset alone, and fc_gamma's
    // first layer is linear, so fc_delta, fc_delta2 and W_gamma pos run once per distinct point pair of the chunk (U_b rows,
    // counted on the device) on the engines and flavours the per-edge launches use; per edge remain the table-flavour
    // epilogue of fc_gamma (edge_gamma_lif) and the attention tail, which reads pos through pid.  Buffers: h -> E1, pos ->
    // E2 (+ its fp32 copy in E3 when the tail reads that), W_gamma pos -> whichever of E1 / E3 is free, fc_gamma's spikes ->
    // the other free one.
    Layer Lwp = k.fc_gamma;
    Lwp.bias = nullptr; Lwp.scale = nullptr; Lwp.shift = nullptr;
    float* const WPbuf = q.pos32 ? p.E1 : p.E3;
    float* const GAbuf = q.pos32 ? p.E2 : p.E1;
    auto wp_args = [&]() {
      GemmArgs a = edge(g.args(Lwp, p.E2, D, E, WPbuf, D, ACT_NONE, nullptr, 0, nullptr, 0, true), q.pos, 0, nullptr, false);
      a.R_dev = p.pairs.U + b;
      return a;
    };
    const bool pairs = indexed && q.attn_in && q.attn_out && q.tab_gamma &&
                       q.pos == 1 && q.gamma == 1 && q.pos32 && sup2(wp_args()) && gemm_tc2_fp16x3(wp_args());
    mdl->tap_snn1.store(q.x_planes, std::memory_order_relaxed);
    mdl->tap_delta2.store(q.pos, std::memory_order_relaxed);
    mdl->tap_gamma.store(q.gamma, std::memory_order_relaxed);
    // ---- the block's launches
    SAPCU_TRY(g.L("fn.fc1+lif").run(fc1_args(q), A_PLAIN));
    SAPCU_TRY(g.L("fn.qkv+lif").run(qkv_args(q), A_PLAIN));
    if (pairs && !table_built) {
      int* err = tc_err_flag();
      SAPCU_REQUIRE(err != nullptr, "fn_forward_indexed: cannot allocate the error flag");
      ProfWork w; w.bytes = (double)P * p.kmax * 40.0;
      SAPCU_PROF(st, "fn.edge_pairs", w, build_pairs(p.pairs, p.idx, M, src->gidx, src->ldg, src->cloud, src->N, err, st));
      table_built = true;
    }
    if (pairs) {
      const Neuron& n = k.snn_delta;
      ProfWork w0;                                       // pair rows: counted on the device only, no algorithmic work recorded
      SAPCU_PROF(st, "fn.fc_delta(K=3)+lif (pairs)", w0,
                 launch_pair_pos_lif(p.pairs.delta[b], p.pairs.U + b, E, D, k.fc_delta.W, k.fc_delta.bias, k.fc_delta.scale,
                                     k.fc_delta.shift, n.np, 4, p.E1, n.tab, n.tab_stride, st));
      GemmArgs d2 = delta2_args(q);
      d2.R_dev = p.pairs.U + b;
      SAPCU_TRY(g.L("fn.fc_delta2+lif (pairs)").run(d2, A_PLAIN));
      Layer Lw = k.fc_gamma;
      Lw.bias = nullptr; Lw.scale = nullptr; Lw.shift = nullptr;
      for (int h = 0; h < 2; ++h)   // [W q | W k], [P, 2D]
        SAPCU_TRY(g.L("fn.fc_gamma(Wq|Wk per point)").layer(Lw, p.QKV + h * D, 3 * D, P, p.QK + h * D, 2 * D, ACT_NONE));
      SAPCU_TRY(g.L("fn.fc_gamma(W pos per pair)").run(wp_args(), A_PLAIN));
      const Neuron& ng = k.snn_gamma;
      ProfWork w1; w1.elsteps = (double)E * D * 4; w1.bytes = (double)E * D * (q.gamma == 2 ? 2.0 : 4.0);
      SAPCU_PROF(st, "fn.edge_gamma+lif", w1,
                 launch_edge_gamma_lif(WPbuf, p.pairs.pid[b], p.QK, p.idx, kk, p.kmax, M, E, D, k.fc_gamma.bias, k.fc_gamma.scale,
                                       k.fc_gamma.shift, ng.np, 4, GAbuf, ng.tab, ng.tab_stride, st));
      GemmArgs a2 = gamma2_args(q, GAbuf);
      a2.at_pid = p.pairs.pid[b];
      SAPCU_TRY(g.L("fn.fc_gamma2+softmax+sum(attention tail)").run(a2, A_PLAIN));
      SAPCU_TRY(g.L("fn.out_proj").layer(k.out_proj, p.RES, D, P, p.R1, D, ACT_NONE));
      SAPCU_TRY(g.L("fn.fc2+residual").layer(k.fc2, p.R1, D, P, p.FCAT + 64 * b, 192, ACT_NONE, nullptr, 0, fin, ldin));
      continue;
    }
    {   // pos-enc layer 1 (fc_delta, K = 3) into E1: edge_pos_lif_fast writes one plane, or (hi, lo) planes from the table
      const Neuron& n = k.snn_delta;
      ProfWork w; w.elsteps = (double)E * D * 4; w.bytes = (double)E * D * (q.delta == 2 ? 2.0 : 4.0);
      SAPCU_PROF(st, "fn.fc_delta(K=3)+lif (edge_pos_lif)", w, q.delta == 2 || q.tab_delta
          ? launch_edge_pos_lif_fast(xyz, p.idx, kk, p.kmax, M, E, D, k.fc_delta.W, k.fc_delta.bias, k.fc_delta.scale, k.fc_delta.shift,
                                     n.np, 4, p.E1, q.tab_delta ? n.tab : nullptr, q.tab_delta ? n.tab_stride : 0, st, q.delta == 1)
          : launch_pointwise3_lif(true, precise, xyz, p.idx, kk, p.kmax, M, E, D, k.fc_delta.W, k.fc_delta.bias, k.fc_delta.scale,
                                  k.fc_delta.shift, n.np, 4, p.E1, st, 1, q.delta == 1));
    }
    if (mode == SAPCU_MODE_FP32) {   // the literal schedule: attention input and logits materialised
      SAPCU_TRY(g.L("fn.fc_delta2+lif").layer(k.fc_delta2, p.E1, D, E, p.E2, D, ACT_LIF, &k.snn_delta2, 4));
      GemmArgs a;
      a.A = p.E2; a.lda = D; a.R = E; a.K = D; a.idx = p.idx; a.ldi = p.kmax; a.kk = kk; a.Mpts = M;
      a.Q = p.QKV; a.Kf = p.QKV + D; a.ldq = 3 * D;
      a.W = k.fc_gamma.W; a.N = D; a.bias = k.fc_gamma.bias; a.scale = k.fc_gamma.scale; a.shift = k.fc_gamma.shift;
      a.act = ACT_LIF; a.T = 4; a.nparams = k.snn_gamma.np; a.Y = p.E3; a.ldc = D;
      SAPCU_TRY(g.L("fn.fc_gamma+lif").run(a, A_ATTNIN));
      SAPCU_TRY(g.L("fn.fc_gamma2").layer(k.fc_gamma2, p.E3, D, E, p.E1, D, ACT_NONE));
      SAPCU_TRY(launch_attn_out(precise, p.E1, p.E2, p.QKV + 2 * D, 3 * D, p.idx, p.kmax, kk, M, P, D, sq, p.RES, st));
    } else {
      SAPCU_TRY(g.L("fn.fc_delta2+lif").run(delta2_args(q), A_PLAIN));
      if (q.attn_in) {
        Layer Lw = k.fc_gamma;
        Lw.bias = nullptr; Lw.scale = nullptr; Lw.shift = nullptr;
        for (int h = 0; h < 2; ++h)   // [W q | W k], [P, 2D]
          SAPCU_TRY(g.L("fn.fc_gamma(Wq|Wk per point)").layer(Lw, p.QKV + h * D, 3 * D, P, p.QK + h * D, 2 * D, ACT_NONE));
        SAPCU_TRY(g.L("fn.fc_gamma+edge_bias+lif").run(gamma_args(q), A_PLAIN));
      } else {
        SAPCU_TRY(launch_attn_in(p.QKV, p.QKV + D, 3 * D, p.E2, p.idx, p.kmax, kk, M, E, D, p.E3, st));
        SAPCU_TRY(g.L("fn.fc_gamma+lif").layer(k.fc_gamma, p.E3, D, E, p.E1, D, ACT_LIF, &k.snn_gamma, 4));
      }
      if (q.attn_out) {
        SAPCU_TRY(g.L("fn.fc_gamma2+softmax+sum(attention tail)").run(gamma2_args(q), A_PLAIN));
      } else {
        SAPCU_TRY(g.L("fn.fc_gamma2").layer(k.fc_gamma2, p.E1, D, E, p.E3, D, ACT_NONE));
        SAPCU_TRY(launch_attn_out(precise, p.E3, p.E2, p.QKV + 2 * D, 3 * D, p.idx, p.kmax, kk, M, P, D, sq, p.RES, st));
      }
    }
    SAPCU_TRY(g.L("fn.out_proj").layer(k.out_proj, p.RES, D, P, p.R1, D, ACT_NONE));
    SAPCU_TRY(g.L("fn.fc2+residual").layer(k.fc2, p.R1, D, P, p.FCAT + 64 * b, 192, ACT_NONE, nullptr, 0, fin, ldin));
  }
  if (stop_block) return 0;
  SAPCU_TRY(g.L("fn.conv_final+lif").layer(f.conv_final, p.FCAT, 192, P, p.G, f.emb, ACT_LIF, &f.snn_final, f.T_enc));
  SAPCU_TRY(launch_group_max(p.G, s, M, 1, f.emb, p.GM, st));
  SAPCU_TRY(g.L("fn.decoder").layer(f.fc_out, p.GM, f.emb, s, p.H0, 2048, ACT_NONE));
  SAPCU_TRY(g.L("fn.decoder").layer(f.mlp[0], p.H0, 2048, s, p.H1, 1024, ACT_GELU));
  SAPCU_TRY(g.L("fn.decoder").layer(f.mlp[1], p.H1, 1024, s, p.H2, 512, ACT_GELU));
  SAPCU_TRY(g.L("fn.decoder").layer(f.mlp[2], p.H2, 512, s, p.H3, 256, ACT_GELU));
  SAPCU_TRY(launch_fn_head(p.H3, 256, s, f.head.W, f.head.bias, f.ln_w, f.ln_b, normals, st));
  return 0;
}

int fd_chunk(const sapcu_model* mdl, const float* xyz, int64_t s, int M, float* dist, const int32_t* const forced[3],
             const FdPlan& p, int mode, cudaStream_t st) {
  const FdNet& f = mdl->fd;
  const int64_t P = s * M;
  const bool precise = mode == SAPCU_MODE_FP32;
  const G g{mode, st};
  const int T = f.T;
  { ProfWork w; w.flops = (double)s * M * M * 3; w.bytes = (double)P * (12 + 4.0 * p.kmax0);
    SAPCU_PROF(st, "fd.intra_knn(xyz)", w, launch_intra_knn(xyz, 3, s, M, 3, p.kmax0, p.idx0, st)); }
  {
    int ks[8]; const float* W[8]; const float* sc[8]; const float* sh[8];
    for (int i = 0; i < f.nscales; ++i) {
      ks[i] = f.kscales[i] < M ? f.kscales[i] : M; W[i] = f.first[i].W; sc[i] = f.first[i].scale; sh[i] = f.first[i].shift;
    }
    ProfWork w; for (int i = 0; i < f.nscales; ++i) w.flops += 2.0 * P * ks[i] * 6 * 64; w.bytes = (double)P * (12 + 4.0 * p.kmax0 + 256.0 * f.nscales);
    SAPCU_PROF(st, "fd.block0(4-scale EdgeConv)", w, launch_fd_block0(xyz, p.idx0, p.kmax0, M, P, f.nscales, ks, W, sc, sh, p.F0, st));
  }
  SAPCU_TRY(g.L("fd.scale_fusion").layer(f.fusion, p.F0, 64 * f.nscales, P, p.U0, 64, ACT_LEAKY));
  const int64_t ldspk = (int64_t)T * 960;
  // conv5 (multi-scale fusion) + LeakyReLU + max over the patch's points: in the tensor-core modes the 2-CTA kernel
  // reduces in its epilogue (per-thread running maxima, then float atomic max) and AGG is never written.  `spk` is the
  // spike tensor's format (tap code): conv5 loads it as it is stored.
  auto c5_args = [&](int spk, bool pooled) {
    GemmArgs a = g.args(f.msc, p.SPK, 960, P * T, p.AGG, f.emb, ACT_LEAKY, nullptr, 0, nullptr, 0, true);   // the spike tensor
    a.pool = pooled ? p.POOL : nullptr; a.pool_T = T; a.pool_M = M;
    a.x_h2 = spk != 0; a.fast = spk == 2;
    return a;
  };
  const bool pooled = mode != SAPCU_MODE_FP32 && settings().fuse_pool && gemm_tc2_supported(c5_args(0, true), A_PLAIN);
  // When conv5 runs on the fast or the fp16x3 path the spike tensor is stored as one fp16 plane or as fp16 (hi, lo) planes
  // of s * 2^13 (rows = point*T + t); the step-0 spikes, which the graphs and EdgeConvs of the next block read, are also
  // kept in fp32 (SPK0, [P, 960]).
  const int spk = !pooled ? 0 : (mode == SAPCU_MODE_FAST && gemm_tc2_fast(c5_args(2, true))) ? 2 : gemm_tc2_fp16x3(c5_args(1, true)) ? 1 : 0;
  mdl->tap_spk.store(spk, std::memory_order_relaxed);
  const bool spk_h2 = spk != 0;
  const int64_t plane = spk == 2 ? 0 : P * T * 960;         // fast mode: hi plane only
  const float* S0 = spk_h2 ? p.SPK0 : p.SPK;                     // step-0 spikes: row stride ld0
  const int64_t ld0 = spk_h2 ? 960 : ldspk;
  if (spk_h2) SAPCU_TRY(launch_neuron_unroll(true, precise, p.U0, 64, P, 64, T, f.blk[0].np, f.blk[0].ep, 1, p.SPK, 960, st, true, p.SPK0, plane, 0));
  else SAPCU_TRY(launch_neuron_unroll(true, precise, p.U0, 64, P, 64, T, f.blk[0].np, f.blk[0].ep, 1, p.SPK, 960, st));
  const int cin[3] = {64, 128, 256}, cout[3] = {128, 256, 512};
  const int off_in[3] = {0, 64, 192}, off_out[3] = {64, 192, 448};
  float* U[3] = {p.U1, p.U2, p.U3};
  for (int b = 0; b < 3; ++b) {
    const int32_t* idx = forced[b];
    if (!idx) {
      ProfWork w; w.flops = (double)s * M * M * cin[b]; w.bytes = (double)P * (4.0 * cin[b] + 4.0 * p.k);
      SAPCU_PROF(st, "fd.intra_knn(features)", w, launch_intra_knn(S0 + off_in[b], ld0, s, M, cin[b], p.k, p.idxf[b], st));
      idx = p.idxf[b];
    }
    if (mode != SAPCU_MODE_FP32) {
      // factorised EdgeConv: one per-POINT contraction [P, Cin] x [2 Cout, Cin]^T, then gather / BN / LeakyReLU / max_k
      Layer L = f.convf[b];
      {
        // the input is a slice of the step-0 spike tensor: parity-grade mode -> fp16x3 products (the splitter converts the fp32
        // rows), on the 2-CTA engine from 1,024 rows on so that the arithmetic does not depend on the chunking
        GemmArgs a = g.args(L, S0 + off_in[b], ld0, P, p.PQ, 2 * cout[b], ACT_NONE);
        if (mode == SAPCU_MODE_TC) {
          GemmArgs t = a; t.x_unit = true; t.tc2_any_rows = true;
          if (gemm_tc2_supported(t, A_PLAIN) && gemm_tc2_fp16x3(t)) a = t;
        }
        SAPCU_TRY(g.L("fd.edgeconv(per-point P|Q)").run(a, A_PLAIN));
      }
      ProfWork w; w.elsteps = (double)P * cout[b] * T; w.bytes = (double)P * cout[b] * (8.0 + 4.0 * T) + (double)P * p.k * 4.0;
      SAPCU_PROF(st, "fd.edgeconv gather+max+neuron unroll", w,
                 launch_edge_gather_unroll(b == 0, p.PQ, cout[b], idx, p.k, M, s, f.conv[b].scale, f.conv[b].shift,
                                           f.blk[b + 1].np, f.blk[b + 1].ep, T, U[b], spk_h2 ? p.SPK : p.SPK + off_out[b], ldspk, 960, st,
                                           spk_h2, p.SPK0, plane, off_out[b]));
      continue;
    } else {
      GemmArgs a;
      a.R = P * p.k; a.K = 2 * cin[b]; a.idx = idx; a.ldi = p.k; a.kk = p.k; a.Mpts = M;
      a.F = p.SPK + off_in[b]; a.ldf = ldspk; a.C = cin[b];
      a.W = f.conv[b].W; a.N = cout[b]; a.scale = f.conv[b].scale; a.shift = f.conv[b].shift;
      a.act = ACT_LEAKY; a.group = 32; a.Y = U[b]; a.ldc = cout[b];
      if (p.k != 32) {     // e.g. the constructor default k = 20, or patches of fewer than 32 points: max over k in a second pass
        a.group = 0; a.Y = p.EDGE;
        SAPCU_TRY(g.L("fd.edgeconv(per-edge)").run(a, A_EDGECAT));
        SAPCU_TRY(launch_group_max(p.EDGE, P, p.k, 1, cout[b], U[b], st));
      } else
      SAPCU_TRY(g.L("fd.edgeconv(per-edge)").run(a, A_EDGECAT));
    }
    SAPCU_TRY(launch_neuron_unroll(b == 0, precise, U[b], cout[b], P, cout[b], T, f.blk[b + 1].np, f.blk[b + 1].ep, 1,
                                   p.SPK + off_out[b], 960, st));
  }
  if (pooled) {
    SAPCU_TRY(launch_fill(p.POOL, s * T * f.emb, -INFINITY, st));
    SAPCU_TRY(g.L("fd.conv5+maxpool").run(c5_args(spk, true), A_PLAIN));
  } else {
    SAPCU_TRY(g.L("fd.conv5").run(c5_args(0, false), A_PLAIN));
    SAPCU_TRY(launch_group_max(p.AGG, s, M, T, f.emb, p.POOL, st));
  }
  SAPCU_TRY(launch_temporal_lif(precise, p.POOL, s, T, f.emb, f.tw, f.snn_fc.np, p.Z, st));
  // StandardDistanceDecoder
  SAPCU_TRY(g.layer(f.fc_in, p.Z, f.emb, s, p.D0, 256, ACT_GELU));
  const float* x = p.D0; int xin = 256;
  float* outs[2] = {p.D1, p.D2};
  for (int r = 0; r < 2; ++r) {
    const int ho = f.rb_fc1[r].N;
    SAPCU_TRY(g.layer(f.rb_res[r], x, xin, s, p.R, ho, ACT_NONE));
    SAPCU_TRY(g.layer(f.rb_fc0[r], x, xin, s, p.T1, ho, ACT_GELU));
    SAPCU_TRY(g.layer(f.rb_fc1[r], p.T1, ho, s, outs[r], ho, ACT_GELU, nullptr, 0, p.R, ho));
    x = outs[r]; xin = ho;
  }
  SAPCU_TRY(g.layer(f.to_qkv, p.D2, 64, s, p.QKV, 192, ACT_NONE));
  const int hd = 64 / f.heads;
  SAPCU_TRY(launch_head_attention(p.QKV, s, f.heads, hd, 1.0f / sqrtf((float)hd), p.O, st));
  SAPCU_TRY(g.layer(f.to_out, p.O, 64, s, p.AO, 64, ACT_NONE, nullptr, 0, p.D2, 64));
  SAPCU_TRY(launch_layernorm_rows(p.AO, s, 64, f.ln_w, f.ln_b, p.LN, st));
  SAPCU_TRY(g.layer(f.fc_hidden, p.LN, 64, s, p.HH, 32, ACT_GELU));
  SAPCU_TRY(launch_fd_tail(p.HH, s, 32, f.fc_dist.W, f.fc_dist.bias, dist, st));
  return 0;
}

int check_common(const sapcu_model* m, int kind, const float* patches, int64_t S, int M, const void* out,
                 const void* ws, int mode) {
  SAPCU_REQUIRE(m, "forward: null model");
  SAPCU_REQUIRE(m->kind == kind, "forward: model kind %d used with the wrong entry point", m->kind);
  if (!m->finalized) { set_error("forward: model not finalized"); return SAPCU_ESTATE; }
  int cur = -1;
  SAPCU_CUDA_CHECK(cudaGetDevice(&cur));
  if (cur != m->device) {     // the weights are another GPU's memory: refuse before any launch
    set_error("forward: model handle was finalized on CUDA device %d, but device %d is current", m->device, cur);
    return SAPCU_ESTATE;
  }
  SAPCU_REQUIRE(S >= 0 && M >= 1 && M <= 128, "forward: need S >= 0 and 1 <= M <= 128 (got S=%lld M=%d)", (long long)S, M);
  SAPCU_REQUIRE(S == 0 || (patches && out && ws), "forward: null pointer");
  const int amode = mode & 0xFF;
  SAPCU_REQUIRE(amode == SAPCU_MODE_FP32 || amode == SAPCU_MODE_TC || amode == SAPCU_MODE_TF32 || amode == SAPCU_MODE_FAST, "forward: unknown mode %d", mode);
  SAPCU_REQUIRE((mode >> 8) == 0 || (kind == SAPCU_MODEL_FN && (mode >> 8) <= 3), "forward: bad debug field in mode 0x%x", mode);
  return 0;
}

}  // namespace

extern "C" {

size_t sapcu_model_workspace_bytes(const sapcu_model* m, int64_t S, int M) {
  if (!m || S < 0 || M < 1) return 0;
  if (S == 0) S = 1;
  return m->kind == SAPCU_MODEL_FN ? fn_plan(m->fn, S, M, nullptr).bytes : fd_plan(m->fd, S, M, nullptr).bytes;
}

int sapcu_fn_forward(const sapcu_model* m, const float* d_patches, int64_t S, int M, float* d_normals, void* d_ws,
                     size_t ws_bytes, int mode, void* stream) {
  SAPCU_TRY(check_common(m, SAPCU_MODEL_FN, d_patches, S, M, d_normals, d_ws, mode));
  if (S == 0) return 0;
  // the reference reads a [B,3,M] input whenever shape[1]==3 (fn/snn_coder.py:441): M==3 is ambiguous there
  SAPCU_REQUIRE(M != 3, "fn_forward: M == 3 is ambiguous in the reference ([B,3,N] layout) and unsupported");
  const int64_t chunk = pick_chunk(m, S, M, ws_bytes);
  if (chunk < 1) { set_error("fn_forward: workspace of %zu bytes cannot hold one patch (need %zu)", ws_bytes, sapcu_model_workspace_bytes(m, 1, M)); return SAPCU_EWORKSPACE; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  for (int64_t s0 = 0; s0 < S; s0 += chunk) {
    const int64_t s = (S - s0) < chunk ? (S - s0) : chunk;
    const FnPlan p = fn_plan(m->fn, s, M, d_ws);
    SAPCU_TRY(fn_chunk(m, d_patches + s0 * M * 3, s, M, d_normals + s0 * 3, p, mode & 0xFF, mode >> 8, st));
  }
  if ((mode & 0xFF) != SAPCU_MODE_FP32) SAPCU_TRY(gemm_tc_check(st));
  return 0;
}

size_t sapcu_fn_indexed_workspace_bytes(const sapcu_model* m, int64_t S, int M, int64_t N, int mode) {
  if (!m || m->kind != SAPCU_MODEL_FN || S < 0 || M < 1 || N < 1) return 0;
  if (S == 0) S = 1;
  return fn_plan(m->fn, S, M, nullptr, mode == SAPCU_MODE_TC ? N : 0).bytes;    // the pair table serves SAPCU_MODE_TC only
}

// Test hook: the pair table of `graph` ([S*M, kmax] patch-local neighbour lists, as intra_knn writes them) for neighbour counts
// kk[3], written into d_ws; h_off[0..6] = byte offsets of pid_0..2 ([S*M*kk_b] int32), delta_0..2 ([U_b] float4), U ([3] int32).
size_t sapcu_pair_table_workspace_bytes(int64_t S, int M, int kmax, const int* kk, int64_t N) {
  if (S < 1 || M < 1 || kmax < 1 || !kk || N < 1) return 0;
  return pair_plan(S * M, kmax, kk, N, nullptr).bytes;
}
int sapcu_pair_table(const int32_t* d_graph, int64_t S, int M, int kmax, const int* kk, const int32_t* d_gidx, int64_t ld_gidx,
                     const double* d_cloud, int64_t N, void* d_ws, size_t ws_bytes, int64_t* h_off, void* stream) {
  SAPCU_REQUIRE(d_graph && kk && d_gidx && d_cloud && d_ws && h_off && S >= 1 && M >= 1 && kmax >= 1 && kmax <= M && ld_gidx >= M && N >= 1,
                "pair_table: bad argument");
  for (int b = 0; b < 3; ++b) SAPCU_REQUIRE(kk[b] >= 1 && kk[b] <= kmax, "pair_table: need 1 <= kk <= kmax");
  SAPCU_REQUIRE(pair_key_fits(N, kmax), "pair_table: %lld points x %d ranks do not fit a 64-bit pair key", (long long)N, kmax);
  const PairBufs q = pair_plan(S * M, kmax, kk, N, d_ws);
  SAPCU_REQUIRE(q.bytes <= ws_bytes, "pair_table: workspace of %zu bytes, need %zu", ws_bytes, q.bytes);
  int* err = tc_err_flag();
  SAPCU_REQUIRE(err != nullptr, "pair_table: cannot allocate the error flag");
  SAPCU_TRY(build_pairs(q, d_graph, M, d_gidx, ld_gidx, d_cloud, N, err, reinterpret_cast<cudaStream_t>(stream)));
  const char* base = reinterpret_cast<const char*>(d_ws);
  for (int b = 0; b < 3; ++b) {
    h_off[b] = reinterpret_cast<const char*>(q.pid[b]) - base;
    h_off[3 + b] = reinterpret_cast<const char*>(q.delta[b]) - base;
  }
  h_off[6] = reinterpret_cast<const char*>(q.U) - base;
  return gemm_tc_check(reinterpret_cast<cudaStream_t>(stream));
}

int sapcu_fn_forward_indexed(const sapcu_model* m, const float* d_patches, int64_t S, int M, const double* d_cloud, int64_t N,
                             const int32_t* d_gidx, int64_t ld_gidx, float* d_normals, void* d_ws, size_t ws_bytes, int mode,
                             void* stream) {
  SAPCU_TRY(check_common(m, SAPCU_MODEL_FN, d_patches, S, M, d_normals, d_ws, mode));
  SAPCU_REQUIRE((mode >> 8) == 0, "fn_forward_indexed: no debug field");
  if (S == 0) return 0;
  SAPCU_REQUIRE(M != 3, "fn_forward_indexed: M == 3 is ambiguous in the reference ([B,3,N] layout) and unsupported");
  SAPCU_REQUIRE(d_cloud && d_gidx && N >= 1 && ld_gidx >= M, "fn_forward_indexed: need the cloud, N >= 1 and a gidx row stride >= M");
  SAPCU_REQUIRE(N <= (1ll << 31), "fn_forward_indexed: cloud of %lld points exceeds 32-bit point indices", (long long)N);
  {
    int kmax = 0;
    for (int b = 0; b < 3; ++b) { const int kb = m->fn.blk[b].k < M ? m->fn.blk[b].k : M; kmax = kb > kmax ? kb : kmax; }
    SAPCU_REQUIRE(pair_key_fits(N, kmax), "fn_forward_indexed: a cloud of %lld points needs more than the 64 bits of a pair key", (long long)N);
  }
  // the pair table serves the parity-grade schedule only: the other modes run exactly as sapcu_fn_forward
  const int64_t Nc = mode == SAPCU_MODE_TC ? N : 0;
  const int64_t chunk = pick_chunk(m, S, M, ws_bytes, Nc);
  if (chunk < 1) { set_error("fn_forward_indexed: workspace of %zu bytes cannot hold one patch (need %zu)", ws_bytes, sapcu_fn_indexed_workspace_bytes(m, 1, M, N, mode)); return SAPCU_EWORKSPACE; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  for (int64_t s0 = 0; s0 < S; s0 += chunk) {
    const int64_t s = (S - s0) < chunk ? (S - s0) : chunk;
    const FnPlan p = fn_plan(m->fn, s, M, d_ws, Nc);
    PatchSource src;
    src.cloud = d_cloud; src.N = N; src.gidx = d_gidx + s0 * ld_gidx; src.ldg = ld_gidx;
    SAPCU_TRY(fn_chunk(m, d_patches + s0 * M * 3, s, M, d_normals + s0 * 3, p, mode, 0, st, Nc ? &src : nullptr));
  }
  if (mode != SAPCU_MODE_FP32) SAPCU_TRY(gemm_tc_check(st));
  return 0;
}

int sapcu_fd_forward(const sapcu_model* m, const float* d_patches, int64_t S, int M, float* d_dist,
                     const int32_t* d_forced_idx, void* d_ws, size_t ws_bytes, int mode, void* stream) {
  SAPCU_TRY(check_common(m, SAPCU_MODEL_FD, d_patches, S, M, d_dist, d_ws, mode));
  if (S == 0) return 0;
  const int k = m->fd.k < M ? m->fd.k : M;
  const int64_t chunk = pick_chunk(m, S, M, ws_bytes);
  if (chunk < 1) { set_error("fd_forward: workspace of %zu bytes cannot hold one patch (need %zu)", ws_bytes, sapcu_model_workspace_bytes(m, 1, M)); return SAPCU_EWORKSPACE; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  for (int64_t s0 = 0; s0 < S; s0 += chunk) {
    const int64_t s = (S - s0) < chunk ? (S - s0) : chunk;
    const FdPlan p = fd_plan(m->fd, s, M, d_ws);
    const int32_t* forced[3] = {nullptr, nullptr, nullptr};
    if (d_forced_idx)
      for (int b = 0; b < 3; ++b) forced[b] = d_forced_idx + ((int64_t)b * S + s0) * M * k;
    SAPCU_TRY(fd_chunk(m, d_patches + s0 * M * 3, s, M, d_dist + s0, forced, p, mode, st));
  }
  if (mode != SAPCU_MODE_FP32) SAPCU_TRY(gemm_tc_check(st));
  return 0;
}

}  // extern "C"

// Test hook: one contraction through G::run.  Workspace: W, its tf32 and fp16 splits, bias / scale / shift, the neuron rows,
// the LIF table and the byte-packed graph of the attention tail, each 256-byte aligned.
namespace {
struct CaseWs { float *W, *Whi, *Wlo, *bias, *scale, *shift, *np, *tab; uint16_t *Wh, *Wl; uint32_t* idx8; size_t bytes; };
CaseWs case_plan(const sapcu_gemm_case_args& a, size_t tab_bytes, void* base) {
  CaseWs w; Bump b(base);
  const size_t nk = (size_t)a.N * a.K;
  w.W = b.take<float>(nk); w.Whi = b.take<float>(nk); w.Wlo = b.take<float>(nk);
  w.Wh = b.take<uint16_t>((nk + 1) & ~(size_t)1); w.Wl = b.take<uint16_t>((nk + 1) & ~(size_t)1);
  w.bias = b.take<float>(a.h_bias ? a.N : 0); w.scale = b.take<float>(a.h_scale ? a.N : 0); w.shift = b.take<float>(a.h_shift ? a.N : 0);
  w.np = b.take<float>(a.h_params4 ? 4 * (size_t)a.N : 0);
  w.tab = b.take<float>(tab_bytes / 4);
  const bool pack = a.d_at_pos && a.d_idx && a.kk > 0;
  w.idx8 = b.take<uint32_t>(pack ? (size_t)(a.R / a.kk) * ((a.ldi + 3) / 4) : 0);
  w.bytes = align_up(b.off, 256);
  return w;
}
bool case_table(const sapcu_gemm_case_args& a) { return a.use_table && a.act == ACT_LIF && a.h_params4 && a.T >= 1 && a.T <= 16; }
}  // namespace

extern "C" {

size_t sapcu_gemm_case_workspace_bytes(const sapcu_gemm_case_args* a) {
  if (!a || a->N < 1 || a->K < 1 || a->R < 0 || (a->d_at_pos && a->kk < 1)) return 0;
  LifTablePacked t;
  if (case_table(*a)) lif_table_pack(a->h_params4, a->N, a->T, &t);
  return case_plan(*a, t.img.size() * 4, nullptr).bytes;
}

int sapcu_gemm_case(const sapcu_gemm_case_args* a, void* d_ws, size_t ws_bytes, int mode, void* stream) {
  SAPCU_REQUIRE(a && d_ws && a->R >= 1 && a->K >= 1 && a->N >= 1 && a->h_w && a->d_y && (a->amode == A_EDGECAT ? a->d_f != nullptr : a->d_x != nullptr),
                "gemm_case: bad argument");
  SAPCU_REQUIRE(a->amode >= A_PLAIN && a->amode <= A_ATTNIN && a->act >= ACT_NONE && a->act <= ACT_LIF && a->x_format >= 0 && a->x_format <= 2,
                "gemm_case: bad amode / act / x_format");
  SAPCU_REQUIRE(a->act != ACT_LIF || (a->h_params4 && a->T >= 1), "gemm_case: a LIF epilogue needs its parameters and T >= 1");
  SAPCU_REQUIRE(mode >= SAPCU_MODE_FP32 && mode <= SAPCU_MODE_FAST, "gemm_case: unknown mode %d", mode);
  SAPCU_REQUIRE(!(a->d_idx || a->d_at_pos) || (a->kk >= 1 && a->R % a->kk == 0 && a->ldi >= a->kk && a->mpts >= 1),
                "gemm_case: edge rows need kk >= 1 dividing R, ldi >= kk and mpts >= 1");
  LifTablePacked t;
  if (case_table(*a)) lif_table_pack(a->h_params4, a->N, a->T, &t);
  const CaseWs w = case_plan(*a, t.img.size() * 4, d_ws);
  SAPCU_REQUIRE(w.bytes <= ws_bytes, "gemm_case: workspace of %zu bytes, need %zu", ws_bytes, w.bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const size_t nk = (size_t)a->N * a->K;
  WeightSplit s;
  split_weights(a->h_w, nk, &s);
  // pageable sources: each copy returns once its bytes are staged, so the host vectors may go out of scope afterwards
  auto up = [&](void* dst, const void* src, size_t bytes) { return src && bytes ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st) : cudaSuccess; };
  SAPCU_CUDA_CHECK(up(w.W, a->h_w, nk * 4));
  SAPCU_CUDA_CHECK(up(w.Whi, s.hi.data(), nk * 4)); SAPCU_CUDA_CHECK(up(w.Wlo, s.lo.data(), nk * 4));
  SAPCU_CUDA_CHECK(up(w.Wh, s.h.data(), s.h.size() * 2)); SAPCU_CUDA_CHECK(up(w.Wl, s.l.data(), s.l.size() * 2));
  SAPCU_CUDA_CHECK(up(w.bias, a->h_bias, (size_t)a->N * 4)); SAPCU_CUDA_CHECK(up(w.scale, a->h_scale, (size_t)a->N * 4));
  SAPCU_CUDA_CHECK(up(w.shift, a->h_shift, (size_t)a->N * 4)); SAPCU_CUDA_CHECK(up(w.np, a->h_params4, (size_t)a->N * 16));
  SAPCU_CUDA_CHECK(up(w.tab, t.img.data(), t.img.size() * 4));
  GemmArgs g;
  g.A = a->d_x; g.lda = a->lda; g.R = a->R; g.K = a->K; g.N = a->N;
  g.W = w.W; g.Whi = w.Whi; g.Wlo = w.Wlo; g.Wh = reinterpret_cast<const float*>(w.Wh); g.Wl = reinterpret_cast<const float*>(w.Wl); g.winv = s.winv;
  g.bias = a->h_bias ? w.bias : nullptr; g.scale = a->h_scale ? w.scale : nullptr; g.shift = a->h_shift ? w.shift : nullptr;
  g.act = a->act; g.T = a->T; g.nparams = a->h_params4 ? w.np : nullptr;
  g.residual = a->d_residual; g.ldr = a->ldr; g.Y = a->d_y; g.ldc = a->ldc; g.Y2 = a->d_y2;
  g.F = a->d_f; g.ldf = a->ldf; g.C = a->C;
  g.Q = a->d_q; g.Kf = a->d_kf; g.ldq = a->ldq; g.idx = a->d_idx; g.ldi = a->ldi; g.kk = a->kk; g.Mpts = a->mpts;
  g.edge_bias = a->edge_bias != 0;
  g.x_h2 = a->x_format != 0; g.x_unit = a->x_unit != 0; g.out_h2 = a->out_h2 != 0; g.fast = a->fast != 0;
  if (case_table(*a) && t.usable) { g.lif_tab = w.tab; g.lif_tab_stride = t.stride; }
  g.pool = a->d_pool; g.pool_T = a->pool_T; g.pool_M = a->pool_M;
  g.at_pos = a->d_at_pos; g.at_v = a->d_at_v; g.at_ldv = a->at_ldv; g.at_sqrt = a->at_sqrt; g.at_pid = a->d_at_pid; g.pos_h2 = a->pos_h2 != 0;
  if (a->d_at_pos && a->d_idx && mode != SAPCU_MODE_FP32 && a->mpts <= 256) {          // as fn_chunk: the byte-packed graph
    SAPCU_TRY(launch_pack_idx_u8(a->d_idx, a->ldi, a->R / a->kk, w.idx8, st));
    g.idx8 = w.idx8; g.ldi8w = (a->ldi + 3) / 4;
  }
  g.R_dev = a->d_R_dev; g.tc2_any_rows = a->tc2_any_rows != 0; g.group = a->group;
  const G run{mode, st};
  return run.L("gemm_case").run(g, a->amode);
}

int sapcu_device_status(void) {
  // watchdog flag of the current device, read from host-visible memory (no stream is touched): call after synchronising
  return gemm_tc_check(nullptr) ? SAPCU_ECUDA : 0;
}

int sapcu_model_tap_format(const sapcu_model* m, const char* name) {
  SAPCU_REQUIRE(m && name, "model_tap_format: bad argument");
  const std::string nm(name);
  const bool blk = nm.size() > 7 && nm.compare(0, 5, "trans") == 0 && nm[6] == '.';     // format of the last block the forward executed
  if (m->kind == SAPCU_MODEL_FN && blk && nm.substr(7) == "snn_gamma") return m->tap_gamma.load(std::memory_order_relaxed);
  if (m->kind == SAPCU_MODEL_FN && blk && nm.substr(7) == "snn_delta2") return m->tap_delta2.load(std::memory_order_relaxed);
  if (m->kind == SAPCU_MODEL_FN && blk && nm.substr(7) == "snn1") return m->tap_snn1.load(std::memory_order_relaxed);
  if (m->kind == SAPCU_MODEL_FD && std::string(name) == "spikes") return m->tap_spk.load(std::memory_order_relaxed);
  return 0;
}

int sapcu_model_tap(const sapcu_model* m, const char* name, int64_t S, int M, int mode, int64_t* off_floats,
                    int64_t* rows, int64_t* cols, int64_t* ld) {
  SAPCU_REQUIRE(m && name && off_floats && rows && cols && ld && S >= 1 && M >= 1, "model_tap: bad argument");
  const std::string n(name);
  const int64_t P = S * M;
  auto set = [&](const void* p, int64_t r, int64_t c, int64_t l) {
    *off_floats = (int64_t)(reinterpret_cast<const char*>(p) - (const char*)nullptr) / 4; *rows = r; *cols = c; *ld = l; return 0;
  };
  if (m->kind == SAPCU_MODEL_FN) {
    const FnPlan p = fn_plan(m->fn, S, M, nullptr);
    if (n == "idx") return set(p.idx, P, p.kmax, p.kmax);            // int32 payload
    if (n == "snn_init") return set(p.F0, P, 64, 64);
    if (n == "fcat") return set(p.FCAT, P, 192, 192);
    if (n.size() > 7 && n.compare(0, 5, "trans") == 0 && n[5] >= '1' && n[5] <= '3' && n[6] == '.') {
      // intermediates of block b live in buffers every block reuses: valid for the LAST block the forward executed
      // (block 3, or block b after a forward with the debug field `stop after block b` in its mode argument)
      const int b = n[5] - '1';
      const int D = m->fn.blk[b].D, kl = m->fn.blk[b].k < M ? m->fn.blk[b].k : M;
      const int64_t E = P * kl;
      const std::string t = n.substr(7);
      if (t == "snn1") return set(p.X, P, D, D);
      if (t == "snn_qkv") return set(p.QKV, P, 3 * D, 3 * D);
      if (t == "snn_delta2") return set(p.E2, E, D, D);
      // tensor-core modes rotate the edge buffers (fc_gamma's spikes land in E1)
      if (t == "snn_gamma") return set((mode & 0xFF) != SAPCU_MODE_FP32 ? p.E1 : p.E3, E, D, D);
      if (t == "logits") {   // the tensor-core modes fuse the softmax into the fc_gamma2 epilogue: no logits buffer
        SAPCU_REQUIRE((mode & 0xFF) == SAPCU_MODE_FP32, "model_tap: '%s' is only materialised in SAPCU_MODE_FP32", name);
        return set(p.E1, E, D, D);
      }
      if (t == "res") return set(p.RES, P, D, D);
    }
    if (n == "snn_final") return set(p.G, P, m->fn.emb, m->fn.emb);
    if (n == "gmax") return set(p.GM, S, m->fn.emb, m->fn.emb);
    if (n == "enc_out") return set(p.H0, S, 2048, 2048);
    if (n == "dec_h3") return set(p.H3, S, 256, 256);
  } else {
    const FdPlan p = fd_plan(m->fd, S, M, nullptr);
    const int T = m->fd.T;
    if (n == "idx0") return set(p.idx0, P, p.kmax0, p.kmax0);        // int32 payload
    if (n == "idxf" || n == "idxf3") return set(p.idxf[2], P, p.k, p.k);     // int32 payload: feature-space graph of block 3
    if (n == "idxf1") return set(p.idxf[0], P, p.k, p.k);
    if (n == "idxf2") return set(p.idxf[1], P, p.k, p.k);
    if (n == "f0") return set(p.F0, P, 64 * m->fd.nscales, 64 * m->fd.nscales);
    if (n == "u0") return set(p.U0, P, 64, 64);
    if (n == "u1") return set(p.U1, P, 128, 128);
    if (n == "u2") return set(p.U2, P, 256, 256);
    if (n == "u3") return set(p.U3, P, 512, 512);
    if (n == "spikes") return set(p.SPK, P * T, 960, 960);           // row = point*T + t
    if (n == "pool") return set(p.POOL, S * T, m->fd.emb, m->fd.emb);
    if (n == "z") return set(p.Z, S, m->fd.emb, m->fd.emb);
    if (n == "dec_d2") return set(p.D2, S, 64, 64);
    if (n == "dec_hidden") return set(p.HH, S, 32, 32);
  }
  set_error("model_tap: unknown tap '%s'", name);
  return SAPCU_EINVAL;
}

}  // extern "C"
