// C-ABI translation unit of libsgrl_b200.so (see include/sgrl_b200.h).
#include "../../include/sgrl_b200.h"

#include "net.cuh"
#include "replay.cuh"
#include "td3.cuh"

namespace sgrl {
thread_local char g_err[512] = "";
long long g_launches = 0;
Prof g_prof;
long long* g_gemm_trace = nullptr;
int g_pdl = -1;
int g_det = -1;
cudaStream_t g_nopdl_streams[32];
int g_nopdl_count = 0;
Side g_side;
}
using namespace sgrl;

#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" {

int sgrl_version(void) { return 3; }
const char* sgrl_last_error(void) { return g_err; }

long long sgrl_launch_count(void) { return g_launches; }

int sgrl_profile(int enable) {
  g_prof.on = enable != 0;
  g_prof.n = 0;
  return 0;
}

/* after a stream/device synchronize: per class c, ms[c] = summed device time, work[c] = summed
 * flops (GEMM classes) or algorithmic bytes (feature/attention), count[c] = launches */
int sgrl_profile_collect(double* ms, double* work, long long* count, int ncls) {
  SGRL_CHECK(ncls >= PC_COUNT, "need room for every class");
  for (int c = 0; c < ncls; ++c) { ms[c] = 0; work[c] = 0; count[c] = 0; }
  for (int i = 0; i < g_prof.n; ++i) {
    float t = 0.f;
    SGRL_CUDA(cudaEventElapsedTime(&t, g_prof.ev[2 * i], g_prof.ev[2 * i + 1]));
    ms[g_prof.cls[i]] += t; work[g_prof.cls[i]] += g_prof.work[i]; count[g_prof.cls[i]] += 1;
  }
  g_prof.n = 0;
  return 0;
}

int sgrl_gemm_trace(long long* buf64) { g_gemm_trace = buf64; return 0; }

int sgrl_param_count(int kind, int n_layers) {
  if (n_layers < 1 || n_layers > MAX_LAYERS || (kind != ACTOR && kind != CRITIC)) return fail(-2, "bad kind/n_layers", __FILE__, __LINE__);
  return enumerate_params(kind, n_layers, nullptr, 0);
}

int sgrl_param_info(int kind, int n_layers, int index, char* name, int name_cap, int* rows, int* cols, int64_t* offset, int* live) {
  SGRL_CHECK(n_layers >= 1 && n_layers <= MAX_LAYERS && (kind == ACTOR || kind == CRITIC), "bad kind/n_layers");
  static thread_local ParamInfo buf[512];
  const int n = enumerate_params(kind, n_layers, buf, 512);
  SGRL_CHECK(index >= 0 && index < n && n <= 512, "param index out of range");
  snprintf(name, name_cap, "%s", buf[index].name);
  *rows = buf[index].rows; *cols = buf[index].cols; *offset = buf[index].offset; *live = buf[index].live;
  return 0;
}

int sgrl_arena_floats(int kind, int n_layers, int64_t* live_floats, int64_t* dead_floats) {
  SGRL_CHECK(n_layers >= 1 && n_layers <= MAX_LAYERS && (kind == ACTOR || kind == CRITIC), "bad kind/n_layers");
  NetLayout L = make_layout(kind, n_layers);
  *live_floats = L.live_floats; *dead_floats = L.dead_floats;
  return 0;
}

int64_t sgrl_stash_floats(int kind, int n_layers, int64_t T, int keep) { return make_stash(kind, n_layers, T, keep).total; }
int64_t sgrl_ws_floats(int n_layers, int64_t T) { return make_ws(n_layers < 1 ? 1 : n_layers > MAX_LAYERS ? MAX_LAYERS : n_layers, T).total; }

int sgrl_stash_info(int kind, int n_layers, int64_t T, int keep, const char* name, int layer, int64_t* offset, int* per_token) {
  StashLayout S = make_stash(kind, n_layers, T, keep);
  if (layer >= 0) {
    SGRL_CHECK(layer < n_layers, "layer out of range");
    for (int i = 0; i < LS_COUNT; ++i)
      if (!strcmp(name, layer_stash_names()[i])) { *offset = S.ls[layer][i]; *per_token = layer_stash_sizes()[i]; return 0; }
  } else {
    for (int i = 0; i < GS_COUNT; ++i)
      if (!strcmp(name, global_stash_names()[i])) { *offset = S.gs[i]; *per_token = global_stash_size(kind, i); return 0; }
  }
  return fail(-2, "unknown stash buffer", __FILE__, __LINE__);
}

static int make_ctx(const SgrlNetCall* k, cudaStream_t st, NetCtx& c) {
  SGRL_CHECK(k != nullptr, "null call");
  SGRL_CHECK(k->kind == ACTOR || k->kind == CRITIC, "kind must be SGRL_ACTOR or SGRL_CRITIC");
  SGRL_CHECK(k->n_layers >= 1 && k->n_layers <= MAX_LAYERS, "n_layers out of range");
  SGRL_CHECK(k->nb >= 1 && k->nb <= 4, "nb out of range");
  SGRL_CHECK(k->T >= 1 && k->G >= 1, "empty batch");
  SGRL_CHECK(k->params && k->stash && k->cu_limbs && k->relation && k->rank3, "null device pointer");
  c.kind = k->kind; c.L = k->n_layers; c.nb = k->nb; c.T = k->T; c.keep = k->keep;
  c.lay = make_layout(k->kind, k->n_layers);
  c.params = k->params; c.zsP = c.lay.live_floats;
  SGRL_CHECK((k->params_hi == nullptr) == (k->params_lo == nullptr), "params_hi and params_lo go together");
  c.phi = k->params_hi; c.plo = k->params_lo;
  c.grads = k->grads; c.zsG = c.lay.live_floats;
  c.st = make_stash(k->kind, k->n_layers, k->T, k->keep);
  SGRL_CHECK(k->stash_stride >= c.st.total, "stash_stride smaller than sgrl_stash_floats()");
  c.stash = k->stash; c.zsS = k->stash_stride;
  c.wl = make_ws(k->n_layers, k->T);
  c.ws = k->ws; c.zsW = k->ws_stride;
  c.gr.cu_limbs = k->cu_limbs; c.gr.rel_off = k->rel_off; c.gr.relation = k->relation; c.gr.G = k->G; c.gr.T = k->T; c.gr.nmax = k->max_limbs;
  c.rank3 = k->rank3; c.max_action = k->max_action; c.use_tc = k->use_tc; c.stream = st;
  return 0;
}

int sgrl_set_forward(const SgrlNetCall* call, const float* obs, int64_t obs_stride, const float* act, int64_t act_stride,
                     float* out, int64_t out_stride, sgrl_stream_t stream) {
  NetCtx c;
  SGRL_TRY(make_ctx(call, ST(stream), c));
  SGRL_CHECK(obs != nullptr, "null obs");
  return net_forward(c, obs, obs_stride, act, act_stride, out, out_stride);
}

int sgrl_set_backward(const SgrlNetCall* call, const float* dout, int64_t dout_stride, int need_wgrad, float* dact,
                      int64_t dact_stride, sgrl_stream_t stream) {
  NetCtx c;
  SGRL_TRY(make_ctx(call, ST(stream), c));
  SGRL_CHECK(call->keep == 1, "backward needs a forward that ran with keep=1");
  SGRL_CHECK(call->ws != nullptr && call->ws_stride >= c.wl.total, "workspace missing or smaller than sgrl_ws_floats()");
  SGRL_CHECK(dout != nullptr, "null dout");
  return net_backward(c, dout, dout_stride, need_wgrad, dact, dact_stride);
}

int sgrl_inv_feature_fwd(const float* X, const float* v0, const float* gd, const float* P1, const float* P2, float* Z, float* Z2,
                         float* G, float* F, int T, sgrl_stream_t stream) {
  SGRL_CHECK(X && gd && P1 && Z && G && F, "null pointer");
  SGRL_CHECK((P2 == nullptr) == (Z2 == nullptr), "P2 and Z2 go together");
  FeatFwdP f{};
  f.Xg = X; f.V0 = v0; f.gd = gd; f.P1 = P1; f.P2 = P2; f.Z = Z; f.Z2 = Z2; f.G = G; f.Fn = F; f.T = T; f.nb = 1; f.head = v0 != nullptr;
  return inv_feature_fwd(f, ST(stream));
}

int sgrl_inv_feature_bwd(const float* dG, const float* dF, const float* Z, const float* F, float* dZ, int T, sgrl_stream_t stream) {
  SGRL_CHECK(dG && dF && Z && F && dZ, "null pointer");
  return inv_feature_bwd(dG, dF, Z, F, dZ, 0, 0, T, 1, ST(stream));
}

int sgrl_attention_fwd(const float* qkv, const float* vgp, const float* gd, const float* rel_w, const float* rel_b,
                       const int32_t* cu_limbs, const int32_t* rel_off, const float* relation, int G, int max_limbs, float* o, float* og,
                       float* p, sgrl_stream_t stream) {
  SGRL_CHECK(qkv && vgp && gd && cu_limbs && o && og && p, "null pointer");
  SGRL_CHECK((rel_w == nullptr) || (rel_b && relation), "bias needs rel_b and relation");
  AttnGraphs gr{cu_limbs, rel_off, relation, G, 0, max_limbs};
  return attention_fwd(qkv, vgp, gd, o, og, p, 0, rel_w, rel_b, 0, gr, 1, ST(stream));
}

int sgrl_attention_bwd(const float* qkv, const float* vgp, const float* gd, const float* p, const float* d_o, const float* d_og,
                       const int32_t* cu_limbs, const int32_t* rel_off, const float* relation, int G, int max_limbs, float* dqkv,
                       float* dvgp, float* drel_w, sgrl_stream_t stream) {
  SGRL_CHECK(qkv && vgp && gd && p && d_o && d_og && cu_limbs && dqkv && dvgp, "null pointer");
  AttnGraphs gr{cu_limbs, rel_off, relation, G, 0, max_limbs};
  return attention_bwd(qkv, vgp, gd, p, 0, d_o, d_og, dqkv, dvgp, 0, drel_w, 0, gr, 1, ST(stream));
}

int sgrl_gemm(const float* A, int lda, int trans_a, const float* B, int ldb, int trans_b, float* C, int ldc, int M, int N, int K,
              float alpha, const float* bias, const float* rowdiv, int relu, int accumulate, int splitk, int use_tc,
              sgrl_stream_t stream) {
  SGRL_CHECK(A && B && C, "null pointer");
  GemmP g = gemm_defaults();
  g.A = A; g.lda = lda; g.transA = trans_a; g.B = B; g.ldb = ldb; g.transB = trans_b; g.C = C; g.ldc = ldc;
  g.M = M; g.N = N; g.K = K; g.alpha = alpha; g.bias = bias; g.rowdiv = rowdiv; g.relu = relu; g.accumulate = accumulate;
  g.splitk = (splitk < 1 || det_enabled()) ? 1 : splitk;
  if (use_tc) {
    SGRL_CHECK(gemm_tc_eligible(g), "shape/epilogue not eligible for the tcgen05 path");
    g.prec = use_tc == 2 ? 1 : 0;
    return gemm_tc(g, ST(stream));
  }
  return gemm_simt(g, ST(stream));
}

int sgrl_gemm_presplit(const float* A, int lda, int trans_a, const float* B_hi, const float* B_lo, int ldb, int trans_b, float* C, int ldc,
                       int M, int N, int K, float alpha, const float* bias, const float* rowdiv, int relu, int accumulate, int splitk,
                       sgrl_stream_t stream) {
  SGRL_CHECK(A && B_hi && B_lo && C, "null pointer");
  GemmP g = gemm_defaults();
  g.A = A; g.lda = lda; g.transA = trans_a; g.B = B_hi; g.Bhi = B_hi; g.Blo = B_lo; g.ldb = ldb; g.transB = trans_b; g.C = C; g.ldc = ldc;
  g.M = M; g.N = N; g.K = K; g.alpha = alpha; g.bias = bias; g.rowdiv = rowdiv; g.relu = relu; g.accumulate = accumulate;
  g.splitk = (splitk < 1 || det_enabled()) ? 1 : splitk;
  SGRL_CHECK(gemm_tc_eligible(g), "shape/epilogue not eligible for the tcgen05 path");
  return gemm_tc(g, ST(stream));
}

int sgrl_gemm_gram(const float* Z, const float* W_hi, const float* W_lo, const float* bias, float* C, int ldc, float* F, float* G,
                   int T, int N, int relu, sgrl_stream_t stream) {
  SGRL_CHECK(Z && W_hi && W_lo && C, "null pointer");
  GemmP g = gemm_defaults();
  g.gramZ = Z; g.gramF = F; g.gramG = G;
  g.B = W_hi; g.Bhi = W_hi; g.Blo = W_lo; g.ldb = GP_K; g.C = C; g.ldc = ldc;
  g.M = T; g.N = N; g.K = GP_K; g.bias = bias; g.relu = relu;
  SGRL_CHECK(gemm_tc_eligible(g), "shape not eligible for the tcgen05 path");
  return gemm_tc(g, ST(stream));
}

int sgrl_gemm_gd(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw, const float* gd, float* Z, int T3, int K,
                 sgrl_stream_t stream) {
  SGRL_CHECK(A && W_hi && W_lo && gd && Z, "null pointer");
  GemmP g = gemm_defaults();
  g.A = A; g.lda = lda; g.B = W_hi; g.Bhi = W_hi; g.Blo = W_lo; g.ldb = ldw; g.C = Z; g.ldc = 32;
  g.M = T3; g.N = 32; g.K = K; g.gdcols = gd;
  SGRL_CHECK(gemm_tc_eligible(g), "shape not eligible for the tcgen05 path");
  return gemm_tc(g, ST(stream));
}

int sgrl_gemm_pair(const float* A0, int lda0, const float* W0_hi, const float* W0_lo, const float* b0, float* C0, int ldc0, int M0, int N0,
                   int K0, const float* A1, int lda1, const float* W1_hi, const float* W1_lo, const float* b1, float* C1, int ldc1, int M1,
                   int N1, int K1, int relu, sgrl_stream_t stream) {
  SGRL_CHECK(A0 && W0_hi && W0_lo && C0 && A1 && W1_hi && W1_lo && C1, "null pointer");
  GemmP g[2];
  g[0] = gemm_defaults();
  g[0].A = A0; g[0].lda = lda0; g[0].B = W0_hi; g[0].Bhi = W0_hi; g[0].Blo = W0_lo; g[0].ldb = K0; g[0].C = C0; g[0].ldc = ldc0;
  g[0].M = M0; g[0].N = N0; g[0].K = K0; g[0].bias = b0; g[0].relu = relu;
  g[1] = gemm_defaults();
  g[1].A = A1; g[1].lda = lda1; g[1].B = W1_hi; g[1].Bhi = W1_hi; g[1].Blo = W1_lo; g[1].ldb = K1; g[1].C = C1; g[1].ldc = ldc1;
  g[1].M = M1; g[1].N = N1; g[1].K = K1; g[1].bias = b1; g[1].relu = relu;
  SGRL_CHECK(gemm_tc_eligible(g[0]) && gemm_tc_eligible(g[1]), "shape not eligible for the tcgen05 path");
  return gemm_tc_group(g, 2, ST(stream));
}

int sgrl_td3_smooth_action(const float* pi_target, const float* noise, float* next_action, float noise_clip, float max_action,
                           int64_t n, sgrl_stream_t stream) {
  SGRL_CHECK(pi_target && noise && next_action, "null pointer");
  launch_k(td3_smooth_action_kernel, grid_for_flat(n * 4), 256, 0, ST(stream), pi_target, noise, next_action, noise_clip, max_action, n);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_td3_smooth_action_rng(const float* pi_target, float* next_action, float* noise_out, float policy_noise, float noise_clip,
                               float max_action, int64_t n, uint64_t seed, const int32_t* draw, sgrl_stream_t stream) {
  SGRL_CHECK(pi_target && next_action && draw, "null pointer");
  launch_k(td3_smooth_action_rng_kernel, grid_for_flat(n), 256, 0, ST(stream), pi_target, next_action, noise_out, policy_noise, noise_clip,
           max_action, (long long)n, (unsigned long long)seed, draw);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_td3_critic_loss(const float* q1, const float* q2, const float* tq1, const float* tq2, const float* reward, const float* done,
                         const int32_t* tok_graph, const float* tok_weight, float* target, float* dq1, float* dq2, float* loss, float discount,
                         float reward_scale, int T, double* reward_stats, int G, sgrl_stream_t stream) {
  SGRL_CHECK(q1 && q2 && tq1 && tq2 && reward && done && tok_graph && target && dq1 && dq2 && loss, "null pointer");
  int gx = ceil_div(T, 256); if (gx > NUM_SMS) gx = NUM_SMS;
  if (det_enabled()) gx = 1;      // the loss scalar: one add
  launch_k(td3_critic_loss_kernel, gx, 256, 0, ST(stream), q1, q2, tq1, tq2, reward, done, tok_graph, tok_weight, target, dq1, dq2, loss, discount, reward_scale, T, reward_stats, G);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_td3_actor_loss(const float* q1, const float* tok_weight, float* dq1, float* loss, int T, sgrl_stream_t stream) {
  SGRL_CHECK(q1 && dq1 && loss, "null pointer");
  int gx = ceil_div(T, 256); if (gx > NUM_SMS) gx = NUM_SMS;
  if (det_enabled()) gx = 1;      // the loss scalar: one add
  launch_k(td3_actor_loss_kernel, gx, 256, 0, ST(stream), q1, tok_weight, dq1, loss, T);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_sumsq(const float* g, int64_t n, float* out, sgrl_stream_t stream) {
  SGRL_CHECK(g && out, "null pointer");
  SGRL_CHECK(aligned16(g), "gradient arena must be 16-byte aligned");
  // scratch for the per-block partial sums: one slot per destination scalar (hashed), so the optimizers of different modules
  // never share one; allocated on first use (an eager call: Agent.update runs each plan eagerly before capturing it)
  constexpr int SLOTS = 16;
  static float* scratch[64] = {nullptr};      // per device
  int dev = 0;
  SGRL_CUDA(cudaGetDevice(&dev));
  SGRL_CHECK(dev >= 0 && dev < 64, "device index");
  if (!scratch[dev]) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    SGRL_CUDA(cudaStreamIsCapturing(ST(stream), &cs));
    SGRL_CHECK(cs == cudaStreamCaptureStatusNone, "sgrl_sumsq: first call on a device must not be inside a stream capture");
    SGRL_CUDA(cudaMalloc(&scratch[dev], sizeof(float) * SLOTS * SUMSQ_MAX_BLOCKS));
  }
  float* part = scratch[dev] + ((reinterpret_cast<uintptr_t>(out) >> 2) * 2654435761u % SLOTS) * SUMSQ_MAX_BLOCKS;
  int nb = grid_for_flat(n); if (nb > SUMSQ_MAX_BLOCKS) nb = SUMSQ_MAX_BLOCKS;
  launch_k(sumsq_partial_kernel, nb, 256, 0, ST(stream), g, (long long)n, part);
  SGRL_LAUNCH_OK();
  launch_k(sumsq_final_kernel, 1, 256, 0, ST(stream), (const float*)part, nb, out);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_split_tf32(const float* w, float* hi, float* lo, int64_t n, sgrl_stream_t stream) {
  SGRL_CHECK(w && hi && lo, "null pointer");
  SGRL_CHECK((n & 3) == 0 && aligned16(w) && aligned16(hi) && aligned16(lo), "arenas must be 16-byte aligned, n % 4 == 0");
  launch_k(split_tf32_kernel, grid_for_flat(n), 256, 0, ST(stream), w, hi, lo, n);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_adam_clip(float* p, const float* g, float* m, float* v, int64_t n, const float* sumsq, const int32_t* step, double lr,
                   double beta1, double beta2, double eps, float max_norm, float grad_scale, float* p_hi, float* p_lo,
                   sgrl_stream_t stream) {
  SGRL_CHECK(p && g && m && v && sumsq && step, "null pointer");
  SGRL_CHECK((p_hi == nullptr) == (p_lo == nullptr) && (!p_hi || (aligned16(p_hi) && aligned16(p_lo))), "p_hi/p_lo go together, 16-byte aligned");
  SGRL_CHECK((n & 3) == 0 && aligned16(p) && aligned16(g) && aligned16(m) && aligned16(v), "arenas must be 16-byte aligned, n % 4 == 0");
  AdamCfg c{lr, beta1, beta2, (float)beta1, (float)beta2, (float)(1.0 - beta1), (float)(1.0 - beta2), (float)eps, max_norm, grad_scale};
  launch_k(adam_clip_kernel, grid_for_flat(n), 256, 0, ST(stream), p, g, m, v, n, sumsq, step, c, p_hi, p_lo);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_bump_step(int32_t* step, sgrl_stream_t stream) {
  SGRL_CHECK(step, "null pointer");
  launch_k(bump_step_kernel, 1, 1, 0, ST(stream), step);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_polyak(float* target, const float* source, int64_t n, float tau, float* t_hi, float* t_lo, int64_t n_split,
                sgrl_stream_t stream) {
  SGRL_CHECK(target && source, "null pointer");
  SGRL_CHECK((t_hi == nullptr) == (t_lo == nullptr) && (!t_hi || (aligned16(t_hi) && aligned16(t_lo) && (n_split & 3) == 0 && n_split <= n)),
             "t_hi/t_lo go together, 16-byte aligned, n_split % 4 == 0");
  SGRL_CHECK((n & 3) == 0 && aligned16(target) && aligned16(source), "arenas must be 16-byte aligned, n % 4 == 0");
  launch_k(polyak_kernel, grid_for_flat(n), 256, 0, ST(stream), target, source, n, tau, (float)(1.0 - (double)tau), t_hi, t_lo, n_split);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_stream_fence(sgrl_stream_t stream) { return stream_fence(ST(stream)); }

int sgrl_deterministic(int enable) {
  const int prev = det_enabled() ? 1 : 0;
  if (enable >= 0) g_det = enable ? 1 : 0;
  return prev;
}

static int replay_part(ReplayPart& q, const float* rows, int64_t row_floats, int64_t capacity, int obs_dim, int act_dim, int batch) {
  SGRL_CHECK(rows != nullptr, "null pointer");
  SGRL_CHECK(obs_dim > 0 && act_dim > 0 && row_floats == 2LL * obs_dim + act_dim + 2 && capacity > 0 && batch >= 0, "bad replay row geometry");
  q.rows = rows; q.rw = row_floats; q.cap = capacity; q.od = obs_dim; q.ad = act_dim;
  return 0;
}

int sgrl_replay_gather(const float* rows, int64_t row_floats, int64_t capacity, const int64_t* idx, int batch, int obs_dim, int act_dim,
                       float* obs, float* action, float* next_obs, float* reward, float* done, sgrl_stream_t stream) {
  SGRL_CHECK(idx && obs && action && next_obs && reward && done, "null pointer");
  ReplayParts P;
  P.n = 1;
  SGRL_TRY(replay_part(P.p[0], rows, row_floats, capacity, obs_dim, act_dim, batch));
  ReplayOut o{obs, action, next_obs, reward, done};
  return replay_gather(P, &batch, reinterpret_cast<const long long*>(idx), o, ST(stream));
}

int sgrl_replay_gather_packed(const SgrlReplayPart* parts, int n_parts, const int64_t* idx, float* obs, float* action, float* next_obs,
                              float* reward, float* done, sgrl_stream_t stream) {
  SGRL_CHECK(parts && idx && obs && action && next_obs && reward && done, "null pointer");
  SGRL_CHECK(n_parts >= 1 && n_parts <= SGRL_REPLAY_MAX_PARTS, "n_parts must be 1..64");
  ReplayParts P;
  P.n = n_parts;
  int B[SGRL_REPLAY_MAX_PARTS];
  for (int i = 0; i < n_parts; ++i) {
    const SgrlReplayPart& s = parts[i];
    SGRL_TRY(replay_part(P.p[i], s.rows, s.row_floats, s.capacity, s.obs_dim, s.act_dim, s.batch));
    B[i] = s.batch;
  }
  ReplayOut o{obs, action, next_obs, reward, done};
  return replay_gather(P, B, reinterpret_cast<const long long*>(idx), o, ST(stream));
}

int sgrl_replay_scatter(float* rows, int64_t row_floats, int64_t capacity, const int64_t* dst, const float* staged, int n, sgrl_stream_t stream) {
  SGRL_CHECK(rows && dst && staged, "null pointer");
  SGRL_CHECK(row_floats > 0 && capacity > 0 && n >= 0, "bad replay row geometry");
  return replay_scatter(rows, row_floats, reinterpret_cast<const long long*>(dst), staged, n, capacity, ST(stream));
}

}  // extern "C"
