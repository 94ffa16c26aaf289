// SET network executor: sequences the kernels of one forward / backward pass of nb
// identical-shape networks (nb=2: twin critics sharing their input, SECritic.py:86-87;
// nb=2K: the twin critics of K seeds, net z reading seed z % K's batch) over a packed batch
// of limb graphs.  Host C++ only; every launch goes to ctx.stream.
//
// Forward follows TransformerModel.forward (SEActor.py:237-287) / SURVEY.md Appendix A/G;
// backward follows SURVEY.md Appendix H.  Activations needed by the backward live in the
// caller-owned stash (layout.h); gradients w.r.t. parameters accumulate into the caller's
// flat gradient arena, which mirrors the parameter arena.
#pragma once
#include "attention.cuh"
#include "common.cuh"
#include "feature.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc_api.h"
#include "layout.h"
#include "misc.cuh"

namespace sgrl {

// ---- backward workspace (floats per token, per net instance) --------------------------
// One FRAME of buffers per backward stage (frame l = encoder layer l, frame n_layers = the heads + final norm), no
// buffer is reused inside a frame: the weight-gradient GEMMs run on side streams (see Side below) and may read a dY
// buffer long after the data-gradient chain has moved on.  Gradients carried between stages (dVg, dh) are written
// out of place into the consuming stage's frame.
enum WS {
  W_DVG, W_DH, W_DH1, W_DUA, W_DUB, W_DQKV, W_DVGP, W_DO, W_DOG, W_DX, W_DDV, W_DZ1, W_DZ2, W_DZ3, W_DG,
  W_DF1, W_DF2, W_DA, W_DA2, W_DA3, W_DT31, W_DT4, W_DR, W_DFF, W_DUH, W_DSH, W_DQ, WS_COUNT
};
inline const int* ws_sizes() {
  static const int s[WS_COUNT] = {384, 128, 128, 256, 256, 768, 756, 256, 768, 128, 384, 96, 96, 96, GP_K,
                                  1, 1, 256, 256, 128, 512, 1024, 96, 128, 256, 148, 3};
  return s;
}
struct WsLayout { long long o[MAX_LAYERS + 1][WS_COUNT]; long long gf /* gradients of the folded vec(G) weights */; long long total; };
inline WsLayout make_ws(int n_layers, long long T) {
  WsLayout w; long long off = 0;
  for (int f = 0; f <= n_layers; ++f)
    for (int i = 0; i < WS_COUNT; ++i) { w.o[f][i] = off; off = align_up(off + (long long)ws_sizes()[i] * T, 64); }
  w.gf = off; off += fold_floats(n_layers);
  w.total = off;
  return w;
}

// ---- side streams: weight-gradient work (dW GEMMs, bias column sums) forks off the data-gradient chain ----------
// fork = record an event on the main stream, make a side stream wait for it, launch there; join = main waits for
// every side stream.  Under CUDA-graph capture this becomes plain fork/join edges of the graph.
// Measured on B200 (CUDA 12.9 / driver 580, tests/test_backward_gpu.py, humanoid B=100): with programmatic dependent launch
// on, a cross-stream dependency built from cudaEventRecord (timing-disabled event) right after a kernel launched with the
// programmatic attribute + cudaStreamWaitEvent does NOT reliably order the waiting stream after that kernel in EAGER
// execution — a forked weight-gradient GEMM occasionally read a dY the data-gradient chain was still writing (errors of
// 1e-4..6e-2 in a few layer-1 gradients, 3 runs out of 4; without PDL or without side streams it did not happen).  A plain, non-programmatic
// launch between the kernel and the event restores the ordering (0 failures in 4), so outside stream capture every fork /
// join event is preceded by this empty kernel.  Inside a captured graph the same record/wait pairs become explicit full
// dependency edges and no fence is needed (Agent.update's hot path is the replayed graph).
__global__ void fence_kernel() {}
inline int stream_fence(cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  SGRL_CUDA(cudaStreamIsCapturing(st, &cs));
  if (cs == cudaStreamCaptureStatusNone) fence_kernel<<<1, 1, 0, st>>>();
  return 0;
}
struct SideSet {
  static constexpr int N = 4;              // lane 0: independent branch of the dependency chain; lanes 1..3: dW / bias-gradient work
  cudaStream_t s[N]; cudaEvent_t fork_ev; cudaEvent_t join_ev[N];
  bool used[N]; int rr; cudaStream_t owner;
};
struct Side {
  static constexpr int NSETS = 8;          // one set per distinct main stream seen (main, the agent's two forward streams, a capture stream, ...)
  SideSet set[NSETS];
  bool made = false; int nowners = 0;
  int dev = -1;                            // device the lanes were created on: one process drives one GPU (DESIGN.md §6)
  int init() {
    int cur = -1;
    SGRL_CUDA(cudaGetDevice(&cur));
    if (!made) dev = cur;
    SGRL_CHECK(cur == dev, "the library's side streams belong to another CUDA device: one process per GPU (set the device before the first call)");
    if (!made) {                         // everything is created up front: nothing but event record/wait happens later (capture-safe)
      for (int k = 0; k < NSETS; ++k) {
        for (int i = 0; i < SideSet::N; ++i) {
          SGRL_CUDA(cudaStreamCreateWithFlags(&set[k].s[i], cudaStreamNonBlocking));
          SGRL_CUDA(cudaEventCreateWithFlags(&set[k].join_ev[i], cudaEventDisableTiming));
          set[k].used[i] = false;
        }
        SGRL_CUDA(cudaEventCreateWithFlags(&set[k].fork_ev, cudaEventDisableTiming));
        set[k].rr = 0; set[k].owner = nullptr;
      }
      made = true;
    }
    return 0;
  }
  SideSet& of(cudaStream_t main) {
    for (int k = 0; k < nowners; ++k) if (set[k].owner == main) return set[k];
    if (nowners < NSETS) {
      SideSet& ss = set[nowners++];
      ss.owner = main;
      return ss;
    }
    return set[(reinterpret_cast<uintptr_t>(main) >> 6) % NSETS];      // more mains than sets: share (only costs overlap)
  }
};
extern Side g_side;
// no forks: the bench's per-class timing pass, or deterministic mode (program order on one stream)
inline bool side_off() { return g_prof.on || det_enabled(); }

struct NetCtx {
  int kind, L, nb, T;
  int in_nets;                            // net z reads input block z % in_nets (1..nb; only the embedding reads the inputs)
  int keep;                               // 0: inference pass (nothing kept for a backward)
  NetLayout lay;
  const float* params; long long zsP;     // live arena; z-stride = lay.live_floats
  const float* phi; const float* plo;     // optional tf32 hi/lo split of the live arena (same layout) for the tcgen05 GEMMs
  float* grads; long long zsG;            // gradient arena (same layout) or nullptr
  StashLayout st; float* stash; long long zsS;
  WsLayout wl; float* ws; long long zsW;
  AttnGraphs gr; const int* rank3;
  float max_action;
  int use_tc;                             // 0: fp32 SIMT; 1: eligible GEMMs on the tcgen05 kernel (3xTF32, fp32 parity); 2: tcgen05 in BF16-input mode
  cudaStream_t stream;

  const float* P(long long off) const { return params + off; }
  float* Gr(long long off) const { return grads + off; }
  float* S(int id) const { return stash + st.gs[id]; }
  float* SL(int l, int id) const { return stash + st.ls[l][id]; }
  float* W(int f, int id) const { return ws + wl.o[f][id]; }
  int ng() const { return kind == ACTOR ? 17 : 20; }
  int ks() const { return D + ng(); }
};

inline int run_gemm(const NetCtx& c, const GemmP& g, cudaStream_t st = nullptr) {
  if (!st) st = c.stream;
  if (c.use_tc && gemm_tc_eligible(g)) {
    GemmP gi = g;
    gi.sm2_ok = c.keep ? 0 : 1;
    gi.prec = c.use_tc == 2 ? 1 : 0;      // use_tc 2: BF16-input mode (reported separately, never the default)
    return gemm_tc(gi, st);
  }
  SGRL_TRY(gemm_simt(g, st));
  if (g.rowsum) {      // the SIMT kernel has no fused row sum: rowsum[m] += alpha * sum_k A(m,k) as a column sum of dY (A = dY^T)
    SGRL_CHECK(g.transA, "rowsum: only for weight-gradient GEMMs (A = dY^T)");
    SGRL_TRY(colsum_launch(g.A, g.lda, g.zsA, g.rowsum, g.zsRowsum, g.K, g.M, g.alpha, g.nb, st));
  }
  return 0;
}
// 1..4 independent projections hanging off the same point of the dependency chain.  Small passes (launch-bound: every
// projection of a 2 304-token step is a 18..144-CTA launch) run them as ONE grouped tcgen05 launch; large passes, where each
// projection fills the machine by itself, as one launch each on the same stream (the two-CTAs-per-SM variant stays available).
inline int run_group(const NetCtx& c, const GemmP* gs, int n, cudaStream_t st = nullptr) {
  if (!st) st = c.stream;
  constexpr long long GROUP_MAXT = 32768;      // tokens x nets
  bool all_tc = c.use_tc && n > 1 && (long long)c.T * c.nb <= GROUP_MAXT;
  for (int i = 0; i < n && all_tc; ++i) all_tc = gemm_tc_eligible(gs[i]);
  if (all_tc) {
    GemmP gp[TC_MAXG];
    for (int i = 0; i < n; ++i) { gp[i] = gs[i]; gp[i].prec = c.use_tc == 2 ? 1 : 0; }
    return gemm_tc_group(gp, n, st);
  }
  for (int i = 0; i < n; ++i) SGRL_TRY(run_gemm(c, gs[i], st));
  return 0;
}
// stream for the next piece of weight-gradient work: a side stream that has been made to wait for everything
// enqueued on the main stream so far (or the main stream itself when side streams are off: side_off)
// `from`: the stream whose work so far the forked stream must wait for (default: the main stream)
inline int side_fork(const NetCtx& c, cudaStream_t* out, int lane = -1, cudaStream_t from = nullptr) {
  Side& sd = g_side;
  if (side_off()) { *out = c.stream; return 0; }
  SideSet& ss = sd.of(c.stream);
  int i = lane;
  if (i < 0) { i = 1 + ss.rr; ss.rr = (ss.rr + 1) % (SideSet::N - 1); }
  if (!from) from = c.stream;
  if (from == ss.s[i]) { *out = from; return 0; }      // same queue: already ordered
  SGRL_TRY(stream_fence(from));
  SGRL_CUDA(cudaEventRecord(ss.fork_ev, from));
  SGRL_CUDA(cudaStreamWaitEvent(ss.s[i], ss.fork_ev, 0));
  ss.used[i] = true;
  *out = ss.s[i];
  return 0;
}
// lane < 0: every lane; else only that lane
inline int side_join(const NetCtx& c, int lane = -1) {
  Side& sd = g_side;
  if (side_off()) return 0;
  SideSet& ss = sd.of(c.stream);
  for (int i = 0; i < SideSet::N; ++i) {
    if (!ss.used[i] || (lane >= 0 && i != lane)) continue;
    SGRL_TRY(stream_fence(ss.s[i]));
    SGRL_CUDA(cudaEventRecord(ss.join_ev[i], ss.s[i]));
    SGRL_CUDA(cudaStreamWaitEvent(c.stream, ss.join_ev[i], 0));
    ss.used[i] = false;
  }
  return 0;
}

// Y[M,N] = X[M,K] W^T (+b): X is stash-like, W/b parameters
inline GemmP lin(const NetCtx& c, const float* X, int ldx, long long zsX, long long w_off, long long b_off,
                 float* Y, int ldy, long long zsY, int M, int N, int K) {
  GemmP g = gemm_defaults();
  g.A = X; g.zsA = zsX; g.lda = ldx; g.transA = 0;
  g.B = c.P(w_off); g.zsB = c.zsP; g.ldb = K; g.transB = 0;
  if (c.phi) { g.Bhi = c.phi + w_off; g.Blo = c.plo + w_off; }
  g.C = Y; g.zsC = zsY; g.ldc = ldy;
  g.M = M; g.N = N; g.K = K; g.nb = c.nb;
  if (b_off >= 0) { g.bias = c.P(b_off); g.zsBias = c.zsP; }
  return g;
}
// dX[M,Kw] = dY[M,Nw] W[Nw,Kw]  (ldw = row stride of W, w_col0 = first column used)
inline GemmP dgrad(const NetCtx& c, const float* dY, int lddy, long long w_off, int ldw, float* dX, int lddx, int M, int Nw, int Kw) {
  GemmP g = gemm_defaults();
  g.A = dY; g.zsA = c.zsW; g.lda = lddy; g.transA = 0;
  g.B = c.P(w_off); g.zsB = c.zsP; g.ldb = ldw; g.transB = 1;
  if (c.phi) { g.Bhi = c.phi + w_off; g.Blo = c.plo + w_off; }
  g.C = dX; g.zsC = c.zsW; g.ldc = lddx;
  g.M = M; g.N = Kw; g.K = Nw; g.nb = c.nb;
  return g;
}
// dW[Nw,Kw] += dY[M,Nw]^T X[M,Kw]
inline GemmP wgrad(const NetCtx& c, const float* dY, int lddy, const float* X, int ldx, long long zsX,
                   long long dw_off, int ldw, int M, int Nw, int Kw) {
  GemmP g = gemm_defaults();
  g.A = dY; g.zsA = c.zsW; g.lda = lddy; g.transA = 1;
  g.B = X; g.zsB = zsX; g.ldb = ldx; g.transB = 1;
  g.C = c.Gr(dw_off); g.zsC = c.zsG; g.ldc = ldw;
  g.M = Nw; g.N = Kw; g.K = M; g.nb = c.nb;
  g.accumulate = 1;
  g.splitk = pick_splitk(Nw, Kw, M, c.nb);
  return g;
}
// ---- the three vec(G) consumers run against their triangle-folded copies (layout.h): K = GP_K instead of 1024 ----
inline FoldDesc fold_desc(const NetCtx& c) {
  FoldDesc d; d.n = 0;
  for (int l = 0; l < c.L; ++l)
    for (int w = 0; w < 2; ++w) { d.src[d.n] = c.lay.lp[l][w ? L_FG1_W : L_G1_W]; d.dst[d.n] = fold_offset(c.L, l, w); d.rows[d.n] = HID; ++d.n; }
  d.src[d.n] = c.lay.gp[G_H1G_W]; d.dst[d.n] = fold_offset(c.L, c.L, 0); d.rows[d.n] = D; ++d.n;
  return d;
}
inline void use_fold(const NetCtx& c, GemmP& g, long long fold_off) {
  const float* w = c.stash + c.st.wf + fold_off;
  g.B = w; g.zsB = c.zsS; g.ldb = GP_K;
  g.Bhi = c.phi ? w + c.st.wf_plane : nullptr; g.Blo = c.phi ? w + 2 * c.st.wf_plane : nullptr;
}
// Y[M,N] = Gp[M,GP_K] W'^T + b
inline GemmP lin_fold(const NetCtx& c, const float* Gp, long long fold_off, long long b_off, float* Y, int ldy, int M, int N) {
  GemmP g = lin(c, Gp, GP_K, c.zsS, 0, b_off, Y, ldy, c.zsS, M, N, GP_K);
  use_fold(c, g, fold_off);
  return g;
}
// dGp[M,GP_K] = dY[M,Nw] W'
inline GemmP dgrad_fold(const NetCtx& c, const float* dY, int lddy, long long fold_off, float* dGp, int M, int Nw) {
  GemmP g = dgrad(c, dY, lddy, 0, GP_K, dGp, GP_K, M, Nw, GP_K);
  use_fold(c, g, fold_off);
  return g;
}
// dW'[Nw,GP_K] += dY^T Gp   (into the workspace; unfolded into the gradient arena at the end of the backward)
inline GemmP wgrad_fold(const NetCtx& c, const float* dY, int lddy, const float* Gp, long long fold_off, int M, int Nw) {
  GemmP g = wgrad(c, dY, lddy, Gp, GP_K, c.zsS, 0, GP_K, M, Nw, GP_K);
  g.C = c.ws + c.wl.gf + fold_off; g.zsC = c.zsW;
  return g;
}
inline int fold_weights(const NetCtx& c, cudaStream_t st) {
  return fold_sym_launch(c.params, c.zsP, c.stash + c.st.wf, c.zsS, c.st.wf_plane, c.phi ? 1 : 0, fold_desc(c), c.nb, st);
}

inline int block_copy(const NetCtx& c, float* dst, int ldd, long long zsD, const float* src, int lds, long long zsSrc, int M, int N, int add,
                      const float* src2 = nullptr, int lds2 = 0, long long zsSrc2 = 0, cudaStream_t st = nullptr) {
  if (!st) st = c.stream;
  return block_copy_launch(dst, ldd, zsD, src, lds, zsSrc, src2, lds2, zsSrc2, M, N, add, c.nb, st);
}
inline int layernorm_fwd(const NetCtx& c, const float* a, int lda, const float* b, int ldb, long long g_off, long long b_off,
                         float* x, float* y, int ldy, float* stats, cudaStream_t st = nullptr) {
  if (!st) st = c.stream;
  return layernorm_fwd_launch(a, lda, b, ldb, c.P(g_off), c.P(b_off), c.zsP, x, y, ldy, nullptr, 0, stats, c.zsS, c.T, c.nb, st);
}
inline int layernorm_bwd(const NetCtx& c, const float* dy1, int ld1, const float* dy2, int ld2, const float* x, int ldx,
                         const float* stats, long long g_off, long long b_off, float* dx, int lddx, bool wg, cudaStream_t st = nullptr,
                         LnRowdiv rd = LnRowdiv{nullptr, nullptr, nullptr, nullptr, 0, 0}) {
  if (!st) st = c.stream;
  return layernorm_bwd_launch(dy1, ld1, dy2, ld2, x, ldx, stats, c.zsS, c.P(g_off), c.zsP, dx, lddx, c.zsW, wg ? c.Gr(g_off) : nullptr,
                              wg ? c.Gr(b_off) : nullptr, c.zsG, rd, c.T, c.nb, st);
}
inline int rowdiv_bwd(const NetCtx& c, float* dy, int lddy, const float* y, int ldy, const float* Fn, float* dF, int N, float cs, int cs_n,
                      cudaStream_t st = nullptr, const float* src = nullptr, int ldsrc = 0, long long zsSrc = 0) {
  if (!st) st = c.stream;
  return rowdiv_bwd_launch(dy, lddy, c.zsW, y, ldy, Fn, c.zsS, dF, N, cs, cs_n, c.T, src, ldsrc, zsSrc, c.nb, st);
}
// the dF accumulators (||G||_F gradients, T floats each) of EVERY frame in one launch at the start of the backward
// (they were 2 * nb memset nodes per layer on the data-gradient chain)
struct ZeroDesc { long long off[2 * (MAX_LAYERS + 1)]; int n; };
__global__ void __launch_bounds__(256) zero_frames_kernel(float* __restrict__ ws, long long zsW, ZeroDesc d, int T) {
  SGRL_PDL_ENTER();
  float* p = ws + blockIdx.z * zsW + d.off[blockIdx.y];
  for (int i = blockIdx.x * 256 + threadIdx.x; i < T; i += gridDim.x * 256) p[i] = 0.f;
}
inline int zero_df_frames(const NetCtx& c) {
  ZeroDesc d; d.n = 0;
  for (int f = 0; f <= c.L; ++f) { d.off[d.n++] = c.wl.o[f][W_DF1]; if (f < c.L) d.off[d.n++] = c.wl.o[f][W_DF2]; }
  int gx = ceil_div(c.T, 256); if (gx > 16) gx = 16; if (gx < 1) gx = 1;
  launch_k(zero_frames_kernel, dim3(gx, d.n, c.nb), 256, 0, c.stream, c.ws, c.zsW, d, c.T);
  SGRL_LAUNCH_OK();
  return 0;
}

inline int unfold_grads(const NetCtx& c, const FoldDesc& d, cudaStream_t st) {
  return unfold_sym_launch(c.ws + c.wl.gf, c.zsW, c.grads, c.zsG, d, c.nb, st);
}

constexpr float QSCALE = 0.08838834764831845f;   // (2*head_dim)^-0.5 = 128^-0.5, subequivariant_attentions.py:88
constexpr float SQRT_D = 11.313708498984761f;    // sqrt(128), SEActor.py:247,249

// ======================================================================================
// forward
// ======================================================================================
inline int net_forward(const NetCtx& c, const float* obs, long long zsObs, const float* act, long long zsAct,
                       float* out, long long zsOut) {
  const int T = c.T, T3 = 3 * c.T, ng = c.ng(), KS = c.ks();
  const NetLayout& Y = c.lay;
  cudaStream_t st = c.stream;
  const long long zS = c.zsS;
  SGRL_CHECK(c.kind == ACTOR || act != nullptr, "critic forward needs actions");
  SGRL_TRY(g_side.init());
  cudaStream_t sb;                 // side stream of the independent branch of the moment (== st when side streams are off)
  // fused schedule: needs the pre-split weights (tcgen05 path) and enough rows for the N = 32 projections to be worth a tile
  const bool fused = c.use_tc && c.phi != nullptr && (long long)T3 * 32 * 128 >= (1 << 21);
  // triangle-folded vec(G) consumers of every layer: on the branch lane next to the embedding and the first projection, joined
  // before the first Gram-generating GEMM reads them
  if (fused) { SGRL_TRY(side_fork(c, &sb, 0)); SGRL_TRY(fold_weights(c, sb)); }
  SGRL_TRY(embed_fwd_launch(obs, zsObs, c.kind == CRITIC ? act : nullptr, zsAct, c.rank3, c.P(Y.gp[G_GENC_W]), c.P(Y.gp[G_ENC_W]),
                            c.P(Y.gp[G_ENC_B]), c.P(Y.gp[G_POS0]), c.P(Y.gp[G_POS1]), c.P(Y.gp[G_POS2]), c.zsP, c.S(T_V0), c.S(T_GD), c.S(T_SH),
                            KS, c.SL(0, S_VGIN), c.SL(0, S_UA) + 128, 256, zS, T, ng, c.nb, c.in_nets, st));
  for (int l = 0; l < c.L; ++l) {
    const long long* lp = Y.lp[l];
    float* Vg = c.SL(l, S_VGIN);
    float* ua = c.SL(l, S_UA);
    float* ub = c.SL(l, S_UB);
    const bool last = l + 1 == c.L;
    float* Vg_next = last ? c.S(T_VGF) : c.SL(l + 1, S_VGIN);
    float* h_next = last ? c.S(T_HL) : c.SL(l + 1, S_UA) + 128;
    const int ld_hn = last ? 128 : 256;
    if (fused) {
      // ---- fused schedule (tcgen05 path): 12 launches per layer on the main stream, the LayerNorms on the branch lane (SURVEY.md Appendix G) ----
      //  Z1 = [Vg g_proj^T | gd]                                  projection on the tensor pipe, gd columns in the epilogue
      //  a1 = relu(linear_g1(tri(Z1^T Z1)))  (+ F1, + G1 if kept)  Gram rows generated inside the GEMM as its A operand
      //  [ u[:, :128] = linear_g2(a1)  ||  vg = vg_proj(Vg) ]      grouped launch
      //  q|k|v = (W u + b)/F1                                      one N = 768 GEMM
      //  attention core
      //  [ x1 = ng_out(o)  ||  dV = g_out(og) ]                   grouped; h1 = LN1(h + x1) on the branch lane
      //  [ Z2 = [dV g_proj2^T | gd]  ||  Z3 = [dV g_proj3^T | gd] ] grouped
      //  a2 = relu(linear_g1'(tri(Z2^T Z2)))  (+ F2, + G2)
      //  u'[:, :128] = linear_g2'(a2)
      //  t31 = relu([linear3 | linear1](u'))
      //  [ f = linear2(t1)/F2  ||  M = linear4(t3)/F2 ]           grouped; h' = LN2(h1 + f) (+ final norm) on the branch lane
      //  Vg' = Vg + dV + linear5(Z3 . M)                           matrix apply + linear5 + residuals
      GemmP gz = lin(c, Vg, 128, zS, lp[L_GPROJ], -1, c.SL(l, S_Z1), 32, zS, T3, 32, 128);
      gz.gdcols = c.S(T_GD); gz.zsGd = zS;
      SGRL_TRY(run_gemm(c, gz));
      if (l == 0) SGRL_TRY(side_join(c, 0));
      GemmP g1 = lin_fold(c, nullptr, fold_offset(c.L, l, 0), lp[L_G1_B], c.SL(l, S_A1), 256, T, 256); g1.relu = 1;
      g1.gramZ = c.SL(l, S_Z1); g1.zsGramZ = zS; g1.gramF = c.SL(l, S_F1); g1.gramG = c.keep ? c.SL(l, S_G1) : nullptr;
      SGRL_TRY(run_gemm(c, g1));
      GemmP pr[2];
      pr[0] = lin(c, c.SL(l, S_A1), 256, zS, lp[L_G2_W], lp[L_G2_B], ua, 256, zS, T, 128, 256);
      pr[1] = lin(c, Vg, 128, zS, lp[L_VG_W], -1, c.SL(l, S_VGP), 252, zS, T3, 252, 128);
      SGRL_TRY(run_group(c, pr, 2));
      GemmP g = lin(c, ua, 256, zS, lp[L_Q_W], lp[L_Q_B], c.SL(l, S_QKV), 768, zS, T, 768, 256);
      g.rowdiv = c.SL(l, S_F1); g.zsRow = zS; g.colscale = QSCALE; g.colscale_n = 256;
      SGRL_TRY(run_gemm(c, g));
      SGRL_TRY(attention_fwd(c.SL(l, S_QKV), c.SL(l, S_VGP), c.S(T_GD), c.SL(l, S_O), c.SL(l, S_OG), c.keep ? c.SL(l, S_P) : nullptr, zS,
                             l == 0 ? c.P(Y.gp[G_REL_W]) : nullptr, l == 0 ? c.P(Y.gp[G_REL_B]) : nullptr, c.zsP, c.gr, c.nb, st));
      pr[0] = lin(c, c.SL(l, S_O), 256, zS, lp[L_NGO_W], lp[L_NGO_B], c.SL(l, S_X1), 128, zS, T, 128, 256);
      pr[1] = lin(c, c.SL(l, S_OG), 256, zS, lp[L_GO_W], -1, c.SL(l, S_DV), 128, zS, T3, 128, 256);
      SGRL_TRY(run_group(c, pr, 2));
      // h1 = LN1(h + ng_out(o)) on the branch lane: first needed by [linear3 | linear1]
      SGRL_TRY(side_fork(c, &sb, 0));
      SGRL_TRY(layernorm_fwd(c, ua + 128, 256, c.SL(l, S_X1), 128, lp[L_N1_W], lp[L_N1_B], c.SL(l, S_X1), ub + 128, 256, c.SL(l, S_ST1), sb));
      pr[0] = lin(c, c.SL(l, S_DV), 128, zS, lp[L_GP2], -1, c.SL(l, S_Z2), 32, zS, T3, 32, 128);
      pr[0].gdcols = c.S(T_GD); pr[0].zsGd = zS;
      pr[1] = lin(c, c.SL(l, S_DV), 128, zS, lp[L_GP3], -1, c.SL(l, S_Z3), 32, zS, T3, 32, 128);
      pr[1].gdcols = c.S(T_GD); pr[1].zsGd = zS;
      SGRL_TRY(run_group(c, pr, 2));
      g1 = lin_fold(c, nullptr, fold_offset(c.L, l, 1), lp[L_FG1_B], c.SL(l, S_A2), 256, T, 256); g1.relu = 1;
      g1.gramZ = c.SL(l, S_Z2); g1.zsGramZ = zS; g1.gramF = c.SL(l, S_F2); g1.gramG = c.keep ? c.SL(l, S_G2) : nullptr;
      SGRL_TRY(run_gemm(c, g1));
      g = lin(c, c.SL(l, S_A2), 256, zS, lp[L_FG2_W], lp[L_FG2_B], ub, 256, zS, T, 128, 256);
      SGRL_TRY(run_gemm(c, g));
      SGRL_TRY(side_join(c, 0));
      g = lin(c, ub, 256, zS, lp[L_L3_W], lp[L_L3_B], c.SL(l, S_T31), 512, zS, T, 512, 256); g.relu = 1;   // [linear3 | linear1]
      SGRL_TRY(run_gemm(c, g));
      pr[0] = lin(c, c.SL(l, S_T31) + 256, 512, zS, lp[L_L2_W], lp[L_L2_B], c.SL(l, S_FF), 128, zS, T, 128, 256);
      pr[0].rowdiv = c.SL(l, S_F2); pr[0].zsRow = zS;
      pr[1] = lin(c, c.SL(l, S_T31), 512, zS, lp[L_L4_W], lp[L_L4_B], c.SL(l, S_MM), 1024, zS, T, 1024, 256);
      pr[1].rowdiv = c.SL(l, S_F2); pr[1].zsRow = zS;
      SGRL_TRY(run_group(c, pr, 2));
      // h' = LN2(h1 + linear2(..)/F2) (+ the encoder's final norm) on the branch lane, next to the matrix apply
      SGRL_TRY(side_fork(c, &sb, 0));
      SGRL_TRY(layernorm_fwd(c, ub + 128, 256, c.SL(l, S_FF), 128, lp[L_N2_W], lp[L_N2_B], c.SL(l, S_X2), h_next, ld_hn, c.SL(l, S_ST2), sb));
      if (last) SGRL_TRY(layernorm_fwd(c, c.S(T_HL), 128, nullptr, 0, Y.gp[G_NORM_W], Y.gp[G_NORM_B], nullptr, c.S(T_SH) + ng, KS, c.S(T_STF), sb));
      SGRL_TRY(matapply_l5_fwd_launch(c.SL(l, S_Z3), c.SL(l, S_MM), c.P(lp[L_L5_W]), c.zsP, Vg, c.SL(l, S_DV), c.keep ? c.SL(l, S_R) : nullptr,
                                      Vg_next, zS, T, c.nb, st));
      SGRL_TRY(side_join(c, 0));
      continue;
    }
    // -- attention block: invariant features of Vg -> u = [g-mlp | h]
    FeatFwdP f{}; f.Xg = Vg; f.zsXg = zS; f.gd = c.S(T_GD); f.zsGd = zS; f.P1 = c.P(lp[L_GPROJ]); f.zsP = c.zsP;
    f.Z = c.SL(l, S_Z1); f.G = c.SL(l, S_G1); f.Fn = c.SL(l, S_F1); f.zsAct = zS; f.T = T; f.nb = c.nb;
    // branch: vg = vg_proj(Vg) only needs the layer input
    SGRL_TRY(side_fork(c, &sb, 0));
    if (l == 0) SGRL_TRY(fold_weights(c, sb));       // triangle-folded vec(G) consumers of every layer, off the main chain
    GemmP g = lin(c, Vg, 128, zS, lp[L_VG_W], -1, c.SL(l, S_VGP), 252, zS, T3, 252, 128);
    SGRL_TRY(run_gemm(c, g, sb));
    SGRL_TRY(inv_feature_fwd(f, st));
    if (l == 0) SGRL_TRY(side_join(c, 0));
    g = lin_fold(c, c.SL(l, S_G1), fold_offset(c.L, l, 0), lp[L_G1_B], c.SL(l, S_A1), 256, T, 256); g.relu = 1;
    SGRL_TRY(run_gemm(c, g));
    g = lin(c, c.SL(l, S_A1), 256, zS, lp[L_G2_W], lp[L_G2_B], ua, 256, zS, T, 128, 256);
    SGRL_TRY(run_gemm(c, g));
    g = lin(c, ua, 256, zS, lp[L_Q_W], lp[L_Q_B], c.SL(l, S_QKV), 768, zS, T, 768, 256);
    g.rowdiv = c.SL(l, S_F1); g.zsRow = zS; g.colscale = QSCALE; g.colscale_n = 256;
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(side_join(c));
    SGRL_TRY(attention_fwd(c.SL(l, S_QKV), c.SL(l, S_VGP), c.S(T_GD), c.SL(l, S_O), c.SL(l, S_OG), c.keep ? c.SL(l, S_P) : nullptr, zS,
                           l == 0 ? c.P(Y.gp[G_REL_W]) : nullptr, l == 0 ? c.P(Y.gp[G_REL_B]) : nullptr, c.zsP, c.gr, c.nb, st));
    // branch: scalar stream h = LN1(h + ng_out(o)) while the vector stream continues on the main stream
    SGRL_TRY(side_fork(c, &sb, 0));
    g = lin(c, c.SL(l, S_O), 256, zS, lp[L_NGO_W], lp[L_NGO_B], c.SL(l, S_X1), 128, zS, T, 128, 256);
    SGRL_TRY(run_gemm(c, g, sb));
    SGRL_TRY(layernorm_fwd(c, ua + 128, 256, c.SL(l, S_X1), 128, lp[L_N1_W], lp[L_N1_B], c.SL(l, S_X1), ub + 128, 256, c.SL(l, S_ST1), sb));
    g = lin(c, c.SL(l, S_OG), 256, zS, lp[L_GO_W], -1, c.SL(l, S_DV), 128, zS, T3, 128, 256);
    SGRL_TRY(run_gemm(c, g));
    // -- feed-forward block: invariant features of dV
    FeatFwdP f2{}; f2.Xg = c.SL(l, S_DV); f2.zsXg = zS; f2.gd = c.S(T_GD); f2.zsGd = zS;
    f2.P1 = c.P(lp[L_GP2]); f2.P2 = c.P(lp[L_GP3]); f2.zsP = c.zsP;
    f2.Z = c.SL(l, S_Z2); f2.Z2 = c.SL(l, S_Z3); f2.G = c.SL(l, S_G2); f2.Fn = c.SL(l, S_F2); f2.zsAct = zS; f2.T = T; f2.nb = c.nb;
    SGRL_TRY(inv_feature_fwd(f2, st));
    g = lin_fold(c, c.SL(l, S_G2), fold_offset(c.L, l, 1), lp[L_FG1_B], c.SL(l, S_A2), 256, T, 256); g.relu = 1;
    SGRL_TRY(run_gemm(c, g));
    g = lin(c, c.SL(l, S_A2), 256, zS, lp[L_FG2_W], lp[L_FG2_B], ub, 256, zS, T, 128, 256);
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(side_join(c));
    g = lin(c, ub, 256, zS, lp[L_L3_W], lp[L_L3_B], c.SL(l, S_T31), 512, zS, T, 512, 256); g.relu = 1;   // [linear3 | linear1]
    SGRL_TRY(run_gemm(c, g));
    // branch: h' = LN2(h + linear2(relu(linear1 u'))/F2) while M = linear4(..)/F2 -> matrix apply -> linear5 runs on the main stream
    SGRL_TRY(side_fork(c, &sb, 0));
    g = lin(c, c.SL(l, S_T31) + 256, 512, zS, lp[L_L2_W], lp[L_L2_B], c.SL(l, S_FF), 128, zS, T, 128, 256);
    g.rowdiv = c.SL(l, S_F2); g.zsRow = zS;
    SGRL_TRY(run_gemm(c, g, sb));
    SGRL_TRY(layernorm_fwd(c, ub + 128, 256, c.SL(l, S_FF), 128, lp[L_N2_W], lp[L_N2_B], c.SL(l, S_X2), h_next, ld_hn, c.SL(l, S_ST2), sb));
    g = lin(c, c.SL(l, S_T31), 512, zS, lp[L_L4_W], lp[L_L4_B], c.SL(l, S_MM), 1024, zS, T, 1024, 256);
    g.rowdiv = c.SL(l, S_F2); g.zsRow = zS;
    SGRL_TRY(run_gemm(c, g));
    // Vg' = Vg + dV + linear5(Z3 . M): matrix apply, the K = 32 projection and both residuals in one launch (misc.cuh)
    SGRL_TRY(matapply_l5_fwd_launch(c.SL(l, S_Z3), c.SL(l, S_MM), c.P(lp[L_L5_W]), c.zsP, Vg, c.SL(l, S_DV), c.keep ? c.SL(l, S_R) : nullptr,
                                    Vg_next, zS, T, c.nb, st));
    SGRL_TRY(side_join(c));
  }
  // final LayerNorm -> right part of SH = [s0 | h]
  if (!fused) SGRL_TRY(layernorm_fwd(c, c.S(T_HL), 128, nullptr, 0, Y.gp[G_NORM_W], Y.gp[G_NORM_B], nullptr, c.S(T_SH) + ng, KS, c.S(T_STF)));
  // -- heads
  FeatFwdP fh{}; fh.head = 1; fh.Xg = c.S(T_VGF); fh.zsXg = zS; fh.V0 = c.S(T_V0); fh.zsV0 = zS; fh.gd = c.S(T_GD); fh.zsGd = zS;
  fh.P1 = c.P(Y.gp[G_GG_W]); fh.P2 = c.kind == ACTOR ? c.P(Y.gp[G_GPH_W]) : nullptr; fh.zsP = c.zsP;
  fh.Z = c.S(T_ZH); fh.Z2 = c.kind == ACTOR ? c.S(T_ZH2) : nullptr; fh.G = c.S(T_GH); fh.Fn = c.S(T_FH); fh.zsAct = zS; fh.T = T; fh.nb = c.nb;
  // the scalar branch u[:, 128:] = linear2_ng(relu(linear1_ng([s0 | h]))) only needs the final norm: on the branch lane, next to
  // the invariant branch K1 -> linear1_g -> linear2_g (3 instead of 5 dependent launches)
  SGRL_TRY(side_fork(c, &sb, 0));
  GemmP g = lin(c, c.S(T_SH), KS, zS, Y.gp[G_H1NG_W], Y.gp[G_H1NG_B], c.S(T_BH), 128, zS, T, 128, KS); g.relu = 1;
  SGRL_TRY(run_gemm(c, g, sb));
  g = lin(c, c.S(T_BH), 128, zS, Y.gp[G_H2NG_W], Y.gp[G_H2NG_B], c.S(T_UH) + 128, 256, zS, T, 128, 128);
  SGRL_TRY(run_gemm(c, g, sb));
  SGRL_TRY(inv_feature_fwd(fh, st));
  g = lin_fold(c, c.S(T_GH), fold_offset(c.L, c.L, 0), Y.gp[G_H1G_B], c.S(T_AH), 128, T, 128); g.relu = 1;
  SGRL_TRY(run_gemm(c, g));
  g = lin(c, c.S(T_AH), 128, zS, Y.gp[G_H2G_W], Y.gp[G_H2G_B], c.S(T_UH), 256, zS, T, 128, 128);
  SGRL_TRY(run_gemm(c, g));
  SGRL_TRY(side_join(c, 0));
  if (c.kind == CRITIC) {
    g = lin(c, c.S(T_UH), 256, zS, Y.gp[G_DNG_W], Y.gp[G_DNG_B], c.S(T_OUT), 1, zS, T, 1, 256);
    g.rowdiv = c.S(T_FH); g.zsRow = zS;
    SGRL_TRY(run_gemm(c, g));
  } else {
    g = lin(c, c.S(T_UH), 256, zS, Y.gp[G_H1M_W], Y.gp[G_H1M_B], c.S(T_M1), 256, zS, T, 256, 256); g.relu = 1;
    SGRL_TRY(run_gemm(c, g));
    g = lin(c, c.S(T_M1), 256, zS, Y.gp[G_H2M_W], Y.gp[G_H2M_B], c.S(T_MH), 1024, zS, T, 1024, 256);
    g.rowdiv = c.S(T_FH); g.zsRow = zS;
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(matapply_fwd_launch(c.S(T_ZH2), c.S(T_MH), c.S(T_RH), zS, T, c.nb, st));
    SGRL_TRY(actor_out_fwd_launch(c.S(T_RH), c.S(T_V0), c.P(Y.gp[G_DG_W]), c.zsP, c.S(T_W3), c.S(T_OUT), zS, c.max_action, T, c.nb, st));
  }
  const int od = c.kind == ACTOR ? 3 : 1;
  if (out) SGRL_TRY(block_copy(c, out, od, zsOut, c.S(T_OUT), od, zS, T, od, 0));
  return 0;
}

// ======================================================================================
// backward.  dOut: gradient w.r.t. the forward output (T x 3 actor, T x 1 critic), per
// instance stride zsDo.  need_wgrad=0 skips parameter gradients (actor step through
// critic1: only d/d(action) is needed, agent.py:167).  dact (critic only, nullable)
// receives d/d(action) (T x 3), overwritten.
// The data-gradient chain runs on c.stream; every dW GEMM / bias column sum forks to a side
// stream (side_fork) right after the dY it consumes has been produced.
// dobs (nullable): receives d/d(obs) (T x 41), overwritten, per instance stride zsDobs — one extra launch at the very end,
// once every frame it reads is complete (input_grad below); nullptr leaves the pass exactly as it is without it.
// ======================================================================================
// d/d(obs) from the stash, the finished workspace frames and the parameters (misc.cuh input_grad_kernel); main stream, after
// the final join.  Algorithmic bytes per token: see tools/obs_grad_bench.py.
inline int input_grad(const NetCtx& c, const float* dOut, long long zsDo, float* dobs, long long zsDobs) {
  const NetLayout& Y = c.lay;
  InGradP p{};
  p.dvg0 = c.W(0, W_DVG); p.dh0 = c.W(0, W_DH);
  p.dzh = c.W(c.L, W_DZ1); p.dzh2 = c.kind == ACTOR ? c.W(c.L, W_DZ3) : nullptr;
  p.dsh = c.W(c.L, W_DSH); p.ldsh = c.ks();
  for (int l = 0; l < c.L; ++l) {
    p.dz[3 * l] = c.W(l, W_DZ1); p.dz[3 * l + 1] = c.W(l, W_DZ2); p.dz[3 * l + 2] = c.W(l, W_DZ3);
    p.dog[l] = c.W(l, W_DOG); p.P[l] = c.SL(l, S_P);
  }
  p.Wg = c.P(Y.gp[G_GENC_W]); p.We = c.P(Y.gp[G_ENC_W]); p.gg = c.P(Y.gp[G_GG_W]);
  p.gph = c.kind == ACTOR ? c.P(Y.gp[G_GPH_W]) : nullptr;
  p.ng = c.ng();
  if (c.kind == ACTOR) { p.dout = dOut; p.zsDo = zsDo; p.out = c.S(T_OUT); p.w3 = c.S(T_W3); }
  p.max_action = c.max_action;
  p.dobs = dobs; p.zsDobs = zsDobs;
  p.cu_limbs = c.gr.cu_limbs; p.G = c.gr.G; p.T = c.T; p.L = c.L;
  p.zsW = c.zsW; p.zsS = c.zsS; p.zsP = c.zsP;
  return input_grad_launch(p, c.nb, c.stream);
}

inline int net_backward(const NetCtx& c, const float* dOut, long long zsDo, int need_wgrad, float* dact, long long zsDact,
                        float* dobs = nullptr, long long zsDobs = 0) {
  const int T = c.T, T3 = 3 * c.T, ng = c.ng(), KS = c.ks();
  const NetLayout& Y = c.lay;
  cudaStream_t st = c.stream;
  const long long zS = c.zsS, zW = c.zsW;
  const bool wg = need_wgrad != 0;
  SGRL_CHECK(!wg || c.grads != nullptr, "backward with need_wgrad requires a gradient arena");
  SGRL_TRY(g_side.init());
  GemmP g;
  int f = c.L, fin = c.L;                               // frame written by this stage / frame holding the incoming dVg, dh
  auto W = [&](int id) { return c.W(f, id); };
  auto Wn = [&](int id) { return c.W(fin, id); };
  // dW[Nw,Kw] += dY^T X (+ db[Nw] += alpha * colsum(dY)) on a side stream
  auto side_w = [&](const float* dY, int lddy, const float* X, int ldx, long long zsX, long long dw_off, int ldw, int M, int Nw, int Kw,
                    long long db_off = -1, float alpha = 1.f, cudaStream_t from = nullptr) -> int {
    if (!wg) return 0;
    cudaStream_t ss;
    SGRL_TRY(side_fork(c, &ss, -1, from));
    GemmP w = wgrad(c, dY, lddy, X, ldx, zsX, dw_off, ldw, M, Nw, Kw);
    w.alpha = alpha;
    if (db_off >= 0) { w.rowsum = c.Gr(db_off); w.zsRowsum = c.zsG; }      // bias gradient rides on the dW GEMM
    SGRL_TRY(run_gemm(c, w, ss));
    return 0;
  };

  // dW of a vec(G) consumer: dW'[Nw,GP_K] += dY^T Gp (+ bias column sum) on a side stream, unfolded at the end
  auto side_w_fold = [&](const float* dY, int lddy, const float* Gp, long long fold_off, int M, int Nw, long long db_off) -> int {
    if (!wg) return 0;
    cudaStream_t ss;
    SGRL_TRY(side_fork(c, &ss, -1, nullptr));
    GemmP w = wgrad_fold(c, dY, lddy, Gp, fold_off, M, Nw);
    w.rowsum = c.Gr(db_off); w.zsRowsum = c.zsG;
    SGRL_TRY(run_gemm(c, w, ss));
    return 0;
  };
  if (wg)
    for (int z = 0; z < c.nb; ++z) SGRL_CUDA(cudaMemsetAsync(c.ws + c.wl.gf + z * c.zsW, 0, sizeof(float) * (size_t)fold_floats(c.L), st));

  // ---------------------------------------------------------------- heads + final norm (frame L)
  SGRL_TRY(zero_df_frames(c));      // dF accumulators of the head block and of every layer
  float* dFh = W(W_DF1);
  if (c.kind == CRITIC) {
    SGRL_TRY(rowdiv_bwd(c, W(W_DQ), 1, c.S(T_OUT), 1, c.S(T_FH), dFh, 1, 1.f, 0, nullptr, dOut, 1, zsDo));      // reads dOut, writes dQ
    SGRL_TRY(side_w(W(W_DQ), 1, c.S(T_UH), 256, zS, Y.gp[G_DNG_W], 256, T, 1, 256, Y.gp[G_DNG_B]));
    g = dgrad(c, W(W_DQ), 1, Y.gp[G_DNG_W], 256, W(W_DUH), 256, T, 1, 256);
    SGRL_TRY(run_gemm(c, g));
  } else {
    SGRL_TRY(actor_out_bwd_launch(dOut, zsDo, c.S(T_OUT), c.S(T_RH), c.S(T_V0), zS, c.P(Y.gp[G_DG_W]), c.zsP, W(W_DR), zW,
                                  wg ? c.Gr(Y.gp[G_DG_W]) : W(W_DQ) /*discarded*/, wg ? c.zsG : zW, wg, c.max_action, T, c.nb, st));
    SGRL_TRY(matapply_bwd_launch(W(W_DR), c.S(T_ZH2), c.S(T_MH), c.S(T_FH), zS, W(W_DZ3), W(W_DT4), dFh, zW, T, c.nb, st));
    SGRL_TRY(side_w(W(W_DT4), 1024, c.S(T_M1), 256, zS, Y.gp[G_H2M_W], 256, T, 1024, 256, Y.gp[G_H2M_B]));
    g = dgrad(c, W(W_DT4), 1024, Y.gp[G_H2M_W], 256, W(W_DA), 256, T, 1024, 256);
    g.mask = c.S(T_M1); g.zsMask = zS; g.ldmask = 256;
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(side_w(W(W_DA), 256, c.S(T_UH), 256, zS, Y.gp[G_H1M_W], 256, T, 256, 256, Y.gp[G_H1M_B]));
    g = dgrad(c, W(W_DA), 256, Y.gp[G_H1M_W], 256, W(W_DUH), 256, T, 256, 256);
    SGRL_TRY(run_gemm(c, g));
  }
  // ---- branch lane (hb): the scalar branch u[:, 128:] = linear2_ng(relu(linear1_ng([s0 | h]))) and the final LayerNorm, next to
  // the invariant branch below (both start from dUH)
  cudaStream_t hb;
  SGRL_TRY(side_fork(c, &hb, 0));
  SGRL_TRY(side_w(W(W_DUH) + 128, 256, c.S(T_BH), 128, zS, Y.gp[G_H2NG_W], 128, T, 128, 128, Y.gp[G_H2NG_B]));
  g = dgrad(c, W(W_DUH) + 128, 256, Y.gp[G_H2NG_W], 128, W(W_DA3), 128, T, 128, 128);
  g.mask = c.S(T_BH); g.zsMask = zS; g.ldmask = 128;
  SGRL_TRY(run_gemm(c, g, hb));
  SGRL_TRY(side_w(W(W_DA3), 128, c.S(T_SH), KS, zS, Y.gp[G_H1NG_W], KS, T, 128, KS, Y.gp[G_H1NG_B], 1.f, hb));
  g = dgrad(c, W(W_DA3), 128, Y.gp[G_H1NG_W], KS, W(W_DSH), KS, T, 128, KS);
  SGRL_TRY(run_gemm(c, g, hb));
  if (dact) SGRL_TRY(block_copy(c, dact, 3, zsDact, W(W_DSH) + 17, KS, zW, T, 3, 0, nullptr, 0, 0, hb));
  // final LayerNorm
  SGRL_TRY(layernorm_bwd(c, W(W_DSH) + ng, KS, nullptr, 0, c.S(T_HL), 128, c.S(T_STF), Y.gp[G_NORM_W], Y.gp[G_NORM_B], W(W_DH), 128, wg, hb));
  // ---- main: u[:, :128] = linear2_g(relu(linear1_g(vec G)))
  SGRL_TRY(side_w(W(W_DUH), 256, c.S(T_AH), 128, zS, Y.gp[G_H2G_W], 128, T, 128, 128, Y.gp[G_H2G_B]));
  g = dgrad(c, W(W_DUH), 256, Y.gp[G_H2G_W], 128, W(W_DA2), 128, T, 128, 128);
  g.mask = c.S(T_AH); g.zsMask = zS; g.ldmask = 128;
  SGRL_TRY(run_gemm(c, g));
  SGRL_TRY(side_w_fold(W(W_DA2), 128, c.S(T_GH), fold_offset(c.L, c.L, 0), T, 128, Y.gp[G_H1G_B]));
  g = dgrad_fold(c, W(W_DA2), 128, fold_offset(c.L, c.L, 0), W(W_DG), T, 128);
  SGRL_TRY(run_gemm(c, g));
  SGRL_TRY(inv_feature_bwd(W(W_DG), dFh, c.S(T_ZH), c.S(T_FH), W(W_DZ1), zS, zW, T, c.nb, st));
  // dVgF = dZh[:, :30] gg_proj[:, 8:] (+ dZh2[:, :30] g_proj[:, 8:])
  g = dgrad(c, W(W_DZ1), 32, Y.gp[G_GG_W] + GN, D + GN, W(W_DVG), 128, T3, NPJ, 128);
  SGRL_TRY(run_gemm(c, g));
  if (c.kind == ACTOR) {
    g = dgrad(c, W(W_DZ3), 32, Y.gp[G_GPH_W] + GN, D + GN, W(W_DVG), 128, T3, NPJ, 128); g.accumulate = 1;
    SGRL_TRY(run_gemm(c, g));
  }
  SGRL_TRY(side_w(W(W_DZ1), 32, c.S(T_V0), 8, zS, Y.gp[G_GG_W], D + GN, T3, NPJ, GN));
  SGRL_TRY(side_w(W(W_DZ1), 32, c.S(T_VGF), 128, zS, Y.gp[G_GG_W] + GN, D + GN, T3, NPJ, 128));
  if (c.kind == ACTOR) {
    SGRL_TRY(side_w(W(W_DZ3), 32, c.S(T_V0), 8, zS, Y.gp[G_GPH_W], D + GN, T3, NPJ, GN));
    SGRL_TRY(side_w(W(W_DZ3), 32, c.S(T_VGF), 128, zS, Y.gp[G_GPH_W] + GN, D + GN, T3, NPJ, 128));
  }
  SGRL_TRY(side_join(c, 0));

  // ---------------------------------------------------------------- encoder layers (frame l reads frame l+1)
  for (int l = c.L - 1; l >= 0; --l) {
    fin = l + 1; f = l;
    const long long* lp = Y.lp[l];
    float* Vg = c.SL(l, S_VGIN);
    float* ua = c.SL(l, S_UA);
    float* ub = c.SL(l, S_UB);
    float* T31 = c.SL(l, S_T31);
    cudaStream_t sb;      // branch lane (== st when side streams are off: the program order below is a valid serial order)
    // ---- branch (sb): LN2 and f = linear2(relu(linear1(u')))/F2
    SGRL_TRY(side_fork(c, &sb, 0));
    // incoming dh: the final norm's output for the last layer; below it, dx1 + du[:, 128:] of the layer above, summed here
    // instead of by a copy kernel at the end of that layer
    // ... with the backward of f = linear2(..)/F2 on the same rows: dFF = dx / F2, dF2 -= <dx, f> / F2 (dx itself stays: LN1's residual)
    const LnRowdiv rd{c.SL(l, S_FF), c.SL(l, S_F2), W(W_DF2), W(W_DFF), 128, 128};
    if (l == c.L - 1)
      SGRL_TRY(layernorm_bwd(c, Wn(W_DH), 128, nullptr, 0, c.SL(l, S_X2), 128, c.SL(l, S_ST2), lp[L_N2_W], lp[L_N2_B], W(W_DX), 128, wg, sb, rd));
    else
      SGRL_TRY(layernorm_bwd(c, Wn(W_DH1), 128, Wn(W_DUA) + 128, 256, c.SL(l, S_X2), 128, c.SL(l, S_ST2), lp[L_N2_W], lp[L_N2_B], W(W_DX), 128, wg, sb, rd));
    SGRL_TRY(side_w(W(W_DFF), 128, T31 + 256, 512, zS, lp[L_L2_W], 256, T, 128, 256, lp[L_L2_B], 1.f, sb));
    g = dgrad(c, W(W_DFF), 128, lp[L_L2_W], 256, W(W_DT31) + 256, 512, T, 128, 256);
    g.mask = T31 + 256; g.zsMask = zS; g.ldmask = 512;
    SGRL_TRY(run_gemm(c, g, sb));
    // ---- main: Vg' = Vg + dV + linear5([g_proj3(dV)|gd] . M)
    SGRL_TRY(side_w(Wn(W_DVG), 128, c.SL(l, S_R), 32, zS, lp[L_L5_W], 32, T3, 128, 32));
    // dR = dVg' W5 and the matrix-apply backward in one launch (misc.cuh)
    SGRL_TRY(matapply_l5_bwd_launch(Wn(W_DVG), c.P(lp[L_L5_W]), c.zsP, c.SL(l, S_Z3), c.SL(l, S_MM), c.SL(l, S_F2), zS, W(W_DZ3), W(W_DT4),
                                    W(W_DF2), zW, T, c.nb, st));
    SGRL_TRY(side_w(W(W_DT4), 1024, T31, 512, zS, lp[L_L4_W], 256, T, 1024, 256, lp[L_L4_B]));
    g = dgrad(c, W(W_DT4), 1024, lp[L_L4_W], 256, W(W_DT31), 512, T, 1024, 256);
    g.mask = T31; g.zsMask = zS; g.ldmask = 512;
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(side_join(c, 0));
    // [linear3 | linear1](u')
    SGRL_TRY(side_w(W(W_DT31), 512, ub, 256, zS, lp[L_L3_W], 256, T, 512, 256, lp[L_L3_B]));
    g = dgrad(c, W(W_DT31), 512, lp[L_L3_W], 256, W(W_DUB), 256, T, 512, 256);
    SGRL_TRY(run_gemm(c, g));
    // ---- branch (sb): LN1: dy = dx2 (residual of LN2) + du'[:, 128:];  dh = ng_out(o)
    SGRL_TRY(side_fork(c, &sb, 0));
    SGRL_TRY(layernorm_bwd(c, W(W_DX), 128, W(W_DUB) + 128, 256, c.SL(l, S_X1), 128, c.SL(l, S_ST1), lp[L_N1_W], lp[L_N1_B], W(W_DH1), 128, wg, sb));
    SGRL_TRY(side_w(W(W_DH1), 128, c.SL(l, S_O), 256, zS, lp[L_NGO_W], 256, T, 128, 256, lp[L_NGO_B], 1.f, sb));
    g = dgrad(c, W(W_DH1), 128, lp[L_NGO_W], 256, W(W_DO), 256, T, 128, 256);
    SGRL_TRY(run_gemm(c, g, sb));
    // d(dV) = dVg' + dZ3[:, :30] g_proj3 (+ dZ2[:, :30] g_proj2, added on the main stream once dZ2 exists): dZ3 has been there since
    // the matrix-apply backward, so this term leaves the main chain
    g = dgrad(c, W(W_DZ3), 32, lp[L_GP3], 128, W(W_DDV), 128, T3, NPJ, 128);
    g.res1 = Wn(W_DVG); g.zsR1 = zW; g.ldr1 = 128;
    SGRL_TRY(run_gemm(c, g, sb));
    // ---- main: u'[:, :128] = linear_g2(relu(linear_g1(vec G2)))
    SGRL_TRY(side_w(W(W_DUB), 256, c.SL(l, S_A2), 256, zS, lp[L_FG2_W], 256, T, 128, 256, lp[L_FG2_B]));
    g = dgrad(c, W(W_DUB), 256, lp[L_FG2_W], 256, W(W_DA), 256, T, 128, 256);
    g.mask = c.SL(l, S_A2); g.zsMask = zS; g.ldmask = 256;
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(side_w_fold(W(W_DA), 256, c.SL(l, S_G2), fold_offset(c.L, l, 1), T, 256, lp[L_FG1_B]));
    g = dgrad_fold(c, W(W_DA), 256, fold_offset(c.L, l, 1), W(W_DG), T, 256);
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(inv_feature_bwd(W(W_DG), W(W_DF2), c.SL(l, S_Z2), c.SL(l, S_F2), W(W_DZ2), zS, zW, T, c.nb, st));
    // d(dV) += dZ2[:, :30] g_proj2   (the branch lane wrote dVg' + dZ3 g_proj3, and dO for the attention backward below)
    SGRL_TRY(side_join(c, 0));
    g = dgrad(c, W(W_DZ2), 32, lp[L_GP2], 128, W(W_DDV), 128, T3, NPJ, 128); g.accumulate = 1;
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(side_w(W(W_DZ2), 32, c.SL(l, S_DV), 128, zS, lp[L_GP2], 128, T3, NPJ, 128));
    SGRL_TRY(side_w(W(W_DZ3), 32, c.SL(l, S_DV), 128, zS, lp[L_GP3], 128, T3, NPJ, 128));
    // dV = g_out(og)
    SGRL_TRY(side_w(W(W_DDV), 128, c.SL(l, S_OG), 256, zS, lp[L_GO_W], 256, T3, 128, 256));
    g = dgrad(c, W(W_DDV), 128, lp[L_GO_W], 256, W(W_DOG), 256, T3, 128, 256);
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(attention_bwd(c.SL(l, S_QKV), c.SL(l, S_VGP), c.S(T_GD), c.SL(l, S_P), zS, W(W_DO), W(W_DOG), W(W_DQKV), W(W_DVGP), zW,
                           (l == 0 && wg) ? c.Gr(Y.gp[G_REL_W]) : nullptr, c.zsG, c.gr, c.nb, st,
                           W(W_DG) /* deterministic mode's partial-sum scratch: free between the two vec(G) halves of the stage */));
    // ---- branch (sb): vg = vg_proj(Vg): dVg(in) = dVg' + dvg vg_proj   (out of place: this frame's dVg)
    SGRL_TRY(side_w(W(W_DVGP), 252, Vg, 128, zS, lp[L_VG_W], 128, T3, 252, 128));
    SGRL_TRY(side_fork(c, &sb, 0));
    g = dgrad(c, W(W_DVGP), 252, lp[L_VG_W], 128, W(W_DVG), 128, T3, 252, 128);
    g.res1 = Wn(W_DVG); g.zsR1 = zW; g.ldr1 = 128;
    SGRL_TRY(run_gemm(c, g, sb));
    // ---- main: q|k|v = (W u + b)/F1 (q also * scale)
    SGRL_TRY(rowdiv_bwd(c, W(W_DQKV), 768, c.SL(l, S_QKV), 768, c.SL(l, S_F1), W(W_DF1), 768, QSCALE, 256));
    SGRL_TRY(side_w(W(W_DQKV), 768, ua, 256, zS, lp[L_Q_W], 256, T, 768, 256, lp[L_Q_B]));
    g = dgrad(c, W(W_DQKV), 768, lp[L_Q_W], 256, W(W_DUA), 256, T, 768, 256);
    SGRL_TRY(run_gemm(c, g));
    // u[:, :128] = linear_g2(relu(linear_g1(vec G1)))
    SGRL_TRY(side_w(W(W_DUA), 256, c.SL(l, S_A1), 256, zS, lp[L_G2_W], 256, T, 128, 256, lp[L_G2_B]));
    g = dgrad(c, W(W_DUA), 256, lp[L_G2_W], 256, W(W_DA2), 256, T, 128, 256);
    g.mask = c.SL(l, S_A1); g.zsMask = zS; g.ldmask = 256;
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(side_w_fold(W(W_DA2), 256, c.SL(l, S_G1), fold_offset(c.L, l, 0), T, 256, lp[L_G1_B]));
    g = dgrad_fold(c, W(W_DA2), 256, fold_offset(c.L, l, 0), W(W_DG), T, 256);
    SGRL_TRY(run_gemm(c, g));
    SGRL_TRY(inv_feature_bwd(W(W_DG), W(W_DF1), c.SL(l, S_Z1), c.SL(l, S_F1), W(W_DZ1), zS, zW, T, c.nb, st));
    SGRL_TRY(side_w(W(W_DZ1), 32, Vg, 128, zS, lp[L_GPROJ], 128, T3, NPJ, 128));
    SGRL_TRY(side_join(c, 0));
    g = dgrad(c, W(W_DZ1), 32, lp[L_GPROJ], 128, W(W_DVG), 128, T3, NPJ, 128); g.accumulate = 1;
    SGRL_TRY(run_gemm(c, g));
    // dh(in) = dx1 + du[:, 128:]: materialised only for the embedding stage (three readers); the layer below sums the two itself
    if (l == 0) SGRL_TRY(block_copy(c, W(W_DH), 128, zW, W(W_DH1), 128, zW, T, 128, 0, W(W_DUA) + 128, 256, zW));
  }
  // ---------------------------------------------------------------- embedding (reads frame 0)
  f = 0; fin = 0;
  if (wg) {
    SGRL_TRY(side_w(W(W_DVG), 128, c.S(T_V0), 8, zS, Y.gp[G_GENC_W], GN, T3, 128, GN, -1, SQRT_D));
    SGRL_TRY(side_w(W(W_DH), 128, c.S(T_SH), KS, zS, Y.gp[G_ENC_W], ng, T, 128, ng, Y.gp[G_ENC_B], SQRT_D));
    SGRL_TRY(pos_embed_bwd_launch(W(W_DH), 128, zW, c.rank3, c.Gr(Y.gp[G_POS0]), c.Gr(Y.gp[G_POS1]), c.Gr(Y.gp[G_POS2]), c.zsG, T, c.nb, st));
  }
  if (dact) {   // + sqrt(128) * dh0 . encoder.weight[:, 17:20]
    SGRL_CHECK(c.kind == CRITIC, "d/d(action) only exists for critics");
    g = dgrad(c, W(W_DH), 128, Y.gp[G_ENC_W] + 17, ng, dact, 3, T, 128, 3);
    g.zsC = zsDact; g.alpha = SQRT_D; g.accumulate = 1;
    SGRL_TRY(run_gemm(c, g));
  }
  SGRL_TRY(side_join(c));
  if (wg) {      // gradients of the folded weights -> (rows,1024) gradient tensors
    SGRL_TRY(unfold_grads(c, fold_desc(c), st));
  }
  if (dobs) SGRL_TRY(input_grad(c, dOut, zsDo, dobs, zsDobs));
  return 0;
}

}  // namespace sgrl
