// C-ABI translation unit of libsgrl_b200.so (see include/sgrl_b200.h).
#include "../../include/sgrl_b200.h"

#include "net.cuh"
#include "replay.cuh"
#include "seed_copy.cuh"
#include "td3.cuh"

namespace sgrl {
thread_local char g_err[512] = "";
long long g_launches = 0;
Prof g_prof;
long long* g_gemm_trace = nullptr;
int g_det = -1;
Side g_side;
}
using namespace sgrl;

#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" {

int sgrl_version(void) { return 12; }
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
  SGRL_CHECK(k->nb >= 1 && k->nb <= MAX_NETS, "nb out of range (1..16)");
  SGRL_CHECK(k->in_nets >= 0 && k->in_nets <= k->nb, "in_nets out of range (0..nb)");
  SGRL_CHECK(k->T >= 1 && k->G >= 1, "empty batch");
  SGRL_CHECK(k->params && k->stash && k->cu_limbs && k->relation && k->rank3, "null device pointer");
  c.kind = k->kind; c.L = k->n_layers; c.nb = k->nb; c.T = k->T; c.keep = k->keep;
  c.in_nets = k->in_nets ? k->in_nets : k->nb;
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

int sgrl_set_backward_dobs(const SgrlNetCall* call, const float* dout, int64_t dout_stride, int need_wgrad, float* dact,
                           int64_t dact_stride, float* dobs, int64_t dobs_stride, sgrl_stream_t stream) {
  NetCtx c;
  SGRL_TRY(make_ctx(call, ST(stream), c));
  SGRL_CHECK(call->keep == 1, "backward needs a forward that ran with keep=1");
  SGRL_CHECK(call->ws != nullptr && call->ws_stride >= c.wl.total, "workspace missing or smaller than sgrl_ws_floats()");
  SGRL_CHECK(dout != nullptr, "null dout");
  SGRL_CHECK(dobs == nullptr || c.nb == 1 || dobs_stride >= 41LL * c.T, "dobs_stride smaller than 41 * T: the nets' d/d(obs) would overlap");
  return net_backward(c, dout, dout_stride, need_wgrad, dact, dact_stride, dobs, dobs_stride);
}

int sgrl_set_backward(const SgrlNetCall* call, const float* dout, int64_t dout_stride, int need_wgrad, float* dact,
                      int64_t dact_stride, sgrl_stream_t stream) {
  return sgrl_set_backward_dobs(call, dout, dout_stride, need_wgrad, dact, dact_stride, nullptr, 0, stream);
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
  SGRL_CHECK(qkv && vgp && gd && cu_limbs && o && og, "null pointer");      // p == NULL: inference pass, no probability store
  SGRL_CHECK((rel_w == nullptr) || (rel_b && relation), "bias needs rel_b and relation");
  AttnGraphs gr{cu_limbs, rel_off, relation, G, 0, max_limbs};
  return attention_fwd(qkv, vgp, gd, o, og, p, 0, rel_w, rel_b, 0, gr, 1, ST(stream));
}

int sgrl_attention_bwd(const float* qkv, const float* vgp, const float* gd, const float* p, const float* d_o, const float* d_og,
                       const int32_t* cu_limbs, const int32_t* rel_off, const float* relation, int G, int max_limbs, float* dqkv,
                       float* dvgp, float* drel_w, sgrl_stream_t stream) {
  SGRL_CHECK(qkv && vgp && gd && p && d_o && d_og && cu_limbs && dqkv && dvgp, "null pointer");
  SGRL_CHECK((drel_w == nullptr) || relation, "drel_w needs relation");
  AttnGraphs gr{cu_limbs, rel_off, relation, G, 0, max_limbs};
  return attention_bwd(qkv, vgp, gd, p, 0, d_o, d_og, dqkv, dvgp, 0, drel_w, 0, gr, 1, ST(stream));
}

// ---- the small kernels around the GEMMs (misc.cuh) and the triangle fold (feature.cuh), one entry point per launcher.  Every
// refusal happens before anything is enqueued; a 16-byte check guards each operand a kernel accesses as float4 (float2 for d og)
// unconditionally.
static bool al16(const void* p, long long ld = 0, long long zs = 0) { return aligned16(p) && (ld & 3) == 0 && (zs & 3) == 0; }
#define SGRL_NETS(nb) SGRL_CHECK((nb) >= 1 && (nb) <= MAX_NETS, "nb must be 1..16")
#define SGRL_TOKENS(T) SGRL_CHECK((T) >= 0, "T must be >= 0")

int sgrl_embed_fwd(const float* obs, int64_t zs_obs, const float* act, int64_t zs_act, const int32_t* rank3, const float* Wg, const float* We,
                   const float* be, const float* E0, const float* E1, const float* E2, int64_t zs_p, float* V0, float* GD, float* SH, int ldsh,
                   float* VG, float* H, int ldh, int64_t zs_s, int T, int ng, int nb, int in_nets, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(obs && rank3 && Wg && We && be && E0 && E1 && E2 && V0 && GD && SH && VG && H, "null pointer");
  SGRL_CHECK(ng == 17 || ng == 20, "ng must be 17 (actor) or 20 (critic)");
  SGRL_CHECK((act != nullptr) == (ng == 20), "act is read by critics (ng = 20) only");
  SGRL_NETS(nb);
  SGRL_CHECK(in_nets >= 1 && in_nets <= nb, "in_nets must be 1..nb");
  SGRL_TOKENS(T);
  SGRL_CHECK(ldsh >= ng && ldh >= D, "ldsh < ng or ldh < 128");
  return embed_fwd_launch(obs, zs_obs, act, zs_act, rank3, Wg, We, be, E0, E1, E2, zs_p, V0, GD, SH, ldsh, VG, H, ldh, zs_s, T, ng, nb, in_nets,
                          ST(stream), grid);
}

int sgrl_input_grad(const float* dvg0, const float* dh0, const float* dzh, const float* dzh2, const float* dsh, int ldsh,
                    const float* const* dz, const float* const* dog, const float* const* P, const float* Wg, const float* We, const float* gg,
                    const float* gph, int ng, const float* dout, int64_t zs_do, const float* out, const float* w3, float max_action,
                    float* dobs, int64_t zs_dobs, const int32_t* cu_limbs, int G, int T, int L, int64_t zs_w, int64_t zs_s, int64_t zs_p, int nb,
                    int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(dvg0 && dh0 && dzh && dsh && dz && dog && P && Wg && We && gg && dobs && cu_limbs, "null pointer");
  SGRL_CHECK(ng == 17 || ng == 20, "ng must be 17 (actor) or 20 (critic)");
  SGRL_CHECK(L >= 1 && L <= MAX_LAYERS, "L must be 1..8");
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  SGRL_CHECK(G >= 1, "G must be >= 1");
  SGRL_CHECK(ldsh >= 17, "ldsh < 17");
  const bool actor = dzh2 != nullptr;
  SGRL_CHECK(actor == (ng == 17), "dzh2 (the head's dZ3) is the actor's (ng = 17) and only the actor's");
  SGRL_CHECK(!actor || (gph && dout && out && w3), "the actor variant needs gph, dout, out and w3");
  InGradP p{};
  for (int l = 0; l < L; ++l) {
    SGRL_CHECK(dz[3 * l] && dz[3 * l + 1] && dz[3 * l + 2] && dog[l] && P[l], "null pointer in dz / dog / P");
    SGRL_CHECK((reinterpret_cast<uintptr_t>(dog[l]) & 7u) == 0 && (zs_w & 1) == 0, "dog must be 8-byte aligned with an even zs_w (float2 loads)");
    p.dz[3 * l] = dz[3 * l]; p.dz[3 * l + 1] = dz[3 * l + 1]; p.dz[3 * l + 2] = dz[3 * l + 2]; p.dog[l] = dog[l]; p.P[l] = P[l];
  }
  p.dvg0 = dvg0; p.dh0 = dh0; p.dzh = dzh; p.dzh2 = dzh2; p.dsh = dsh; p.ldsh = ldsh;
  p.Wg = Wg; p.We = We; p.gg = gg; p.gph = actor ? gph : nullptr; p.ng = ng;
  if (actor) { p.dout = dout; p.zsDo = zs_do; p.out = out; p.w3 = w3; }
  p.max_action = max_action; p.dobs = dobs; p.zsDobs = zs_dobs;
  p.cu_limbs = cu_limbs; p.G = G; p.T = T; p.L = L; p.zsW = zs_w; p.zsS = zs_s; p.zsP = zs_p;
  return input_grad_launch(p, nb, ST(stream), grid);
}

int sgrl_pos_embed_bwd(const float* dH, int ldh, int64_t zs_w, const int32_t* rank3, float* dE0, float* dE1, float* dE2, int64_t zs_g, int T, int nb,
                       int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(dH && rank3 && dE0 && dE1 && dE2, "null pointer");
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  SGRL_CHECK(ldh >= D, "ldh < 128");
  return pos_embed_bwd_launch(dH, ldh, zs_w, rank3, dE0, dE1, dE2, zs_g, T, nb, ST(stream), grid);
}

int sgrl_layernorm_fwd(const float* a, int lda, const float* b, int ldb, const float* gamma, const float* beta, int64_t zs_p, float* x, float* y,
                       int ldy, float* y2, int ldy2, float* stats, int64_t zs_s, int T, int nb, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(a && gamma && beta && y && stats, "null pointer");
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  SGRL_CHECK(lda >= D && (!b || ldb >= D) && ldy >= D && (!y2 || ldy2 >= D), "a leading dimension < 128");
  SGRL_CHECK(al16(gamma, 0, zs_p) && al16(beta), "gamma, beta and zs_p must be 16-byte aligned (float4 loads)");
  SGRL_CHECK(!x || al16(x, 0, zs_s), "x and zs_s must be 16-byte aligned (float4 stores)");
  return layernorm_fwd_launch(a, lda, b, ldb, gamma, beta, zs_p, x, y, ldy, y2, ldy2, stats, zs_s, T, nb, ST(stream), grid);
}

int sgrl_layernorm_bwd(const float* dy1, int ld1, const float* dy2, int ld2, const float* x, int ldx, const float* stats, int64_t zs_s,
                       const float* gamma, int64_t zs_p, float* dx, int lddx, int64_t zs_w, float* dgamma, float* dbeta, int64_t zs_g,
                       const float* rd_y, int rd_ldy, const float* rd_F, float* rd_dF, float* rd_out, int rd_ldout, int T, int nb,
                       int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(dy1 && x && stats && gamma && dx, "null pointer");
  SGRL_CHECK((dgamma == nullptr) == (dbeta == nullptr), "dgamma and dbeta go together");
  const int nrd = (rd_y != nullptr) + (rd_F != nullptr) + (rd_dF != nullptr) + (rd_out != nullptr);
  SGRL_CHECK(nrd == 0 || nrd == 4, "rd_y, rd_F, rd_dF and rd_out go together");
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  SGRL_CHECK(ld1 >= D && (!dy2 || ld2 >= D) && ldx >= D && lddx >= D && (!nrd || (rd_ldy >= D && rd_ldout >= D)), "a leading dimension < 128");
  SGRL_CHECK(al16(gamma, 0, zs_p), "gamma and zs_p must be 16-byte aligned (float4 loads)");
  return layernorm_bwd_launch(dy1, ld1, dy2, ld2, x, ldx, stats, zs_s, gamma, zs_p, dx, lddx, zs_w, dgamma, dbeta, zs_g,
                              LnRowdiv{rd_y, rd_F, rd_dF, rd_out, rd_ldy, rd_ldout}, T, nb, ST(stream), grid);
}

int sgrl_matapply_fwd(const float* Z, const float* M, float* R, int64_t zs_s, int T, int nb, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(Z && M && R, "null pointer");
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  return matapply_fwd_launch(Z, M, R, zs_s, T, nb, ST(stream), grid);
}

int sgrl_matapply_bwd(const float* dR, const float* Z, const float* M, const float* F, int64_t zs_s, float* dZ, float* dT, float* dF, int64_t zs_w,
                      int T, int nb, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(dR && Z && M && F && dZ && dT && dF, "null pointer");
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  return matapply_bwd_launch(dR, Z, M, F, zs_s, dZ, dT, dF, zs_w, T, nb, ST(stream), grid);
}

int sgrl_matapply_l5_fwd(const float* Z, const float* M, const float* W5, int64_t zs_p, const float* Vg, const float* dV, float* R, float* Vn,
                         int64_t zs_s, int T, int nb, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(Z && M && W5 && Vg && dV && Vn, "null pointer");      // R == NULL: inference pass
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  return matapply_l5_fwd_launch(Z, M, W5, zs_p, Vg, dV, R, Vn, zs_s, T, nb, ST(stream), grid);
}

int sgrl_matapply_l5_bwd(const float* dVn, const float* W5, int64_t zs_p, const float* Z, const float* M, const float* F, int64_t zs_s, float* dZ,
                         float* dT, float* dF, int64_t zs_w, int T, int nb, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(dVn && W5 && Z && M && F && dZ && dT && dF, "null pointer");
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  SGRL_CHECK(al16(dVn, 0, zs_w), "dVn and zs_w must be 16-byte aligned (float4 loads)");
  return matapply_l5_bwd_launch(dVn, W5, zs_p, Z, M, F, zs_s, dZ, dT, dF, zs_w, T, nb, ST(stream), grid);
}

int sgrl_actor_out_fwd(const float* R, const float* V0, const float* wd, int64_t zs_p, float* W3, float* out, int64_t zs_s, float max_action, int T,
                       int nb, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(R && V0 && wd && W3 && out, "null pointer");
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  return actor_out_fwd_launch(R, V0, wd, zs_p, W3, out, zs_s, max_action, T, nb, ST(stream), grid);
}

int sgrl_actor_out_bwd(const float* dout, int64_t zs_do, const float* out, const float* R, const float* V0, int64_t zs_s, const float* wd,
                       int64_t zs_p, float* dR, int64_t zs_w, float* dwd, int64_t zs_g, float max_action, int T, int nb, int32_t* grid,
                       sgrl_stream_t stream) {
  SGRL_CHECK(dout && out && R && V0 && wd && dR && dwd, "null pointer");
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  return actor_out_bwd_launch(dout, zs_do, out, R, V0, zs_s, wd, zs_p, dR, zs_w, dwd, zs_g, true, max_action, T, nb, ST(stream), grid);
}

int sgrl_rowdiv_bwd(float* dy, int lddy, int64_t zs_w, const float* y, int ldy, const float* F, int64_t zs_s, float* dF, int N, float colscale,
                    int cs_n, const float* src, int ldsrc, int64_t zs_src, int T, int nb, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(dy && y && F && dF, "null pointer");      // src == NULL: dy is read in place
  SGRL_NETS(nb);
  SGRL_TOKENS(T);
  SGRL_CHECK(N >= 1 && lddy >= N && ldy >= N && (!src || ldsrc >= N), "N must be >= 1 and no leading dimension < N");
  SGRL_CHECK(cs_n >= 0 && cs_n <= N, "cs_n must be 0..N");
  return rowdiv_bwd_launch(dy, lddy, zs_w, y, ldy, F, zs_s, dF, N, colscale, cs_n, T, src, ldsrc, zs_src, nb, ST(stream), grid);
}

int sgrl_colsum(const float* X, int ldx, int64_t zs_x, float* out, int64_t zs_o, int M, int N, float alpha, int nb, int32_t* grid,
                sgrl_stream_t stream) {
  SGRL_CHECK(X && out, "null pointer");
  SGRL_NETS(nb);
  SGRL_CHECK(M >= 0 && N >= 1 && ldx >= N, "M must be >= 0, N >= 1 and ldx >= N");
  return colsum_launch(X, ldx, zs_x, out, zs_o, M, N, alpha, nb, ST(stream), grid);
}

int sgrl_block_copy(float* dst, int ldd, int64_t zs_d, const float* src, int lds, int64_t zs_src, const float* src2, int lds2, int64_t zs_src2,
                    int M, int N, int add, int nb, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(dst && src, "null pointer");
  SGRL_NETS(nb);
  SGRL_CHECK(M >= 0 && N >= 1 && ldd >= N && lds >= N && (!src2 || lds2 >= N), "M must be >= 0, N >= 1 and no leading dimension < N");
  return block_copy_launch(dst, ldd, zs_d, src, lds, zs_src, src2, lds2, zs_src2, M, N, add ? 1 : 0, nb, ST(stream), grid);
}

static int fold_desc_of(const int64_t* src, const int64_t* dst, const int32_t* rows, int n, FoldDesc& d) {
  SGRL_CHECK(src && dst && rows, "null pointer");
  SGRL_CHECK(n >= 1 && n <= 2 * MAX_LAYERS + 1, "n must be 1..17");
  d.n = n;
  for (int i = 0; i < n; ++i) {
    SGRL_CHECK(src[i] >= 0 && dst[i] >= 0 && rows[i] >= 1, "offsets must be >= 0, rows >= 1");
    SGRL_CHECK((dst[i] & 3) == 0, "folded matrices must start 16-byte aligned (the tcgen05 GEMMs read them by TMA)");
    d.src[i] = src[i]; d.dst[i] = dst[i]; d.rows[i] = rows[i];
  }
  return 0;
}

int sgrl_fold_sym(const float* params, int64_t zs_p, float* wf, int64_t zs_s, int64_t plane, int with_split, const int64_t* src, const int64_t* dst,
                  const int32_t* rows, int n, int nb, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(params && wf, "null pointer");
  SGRL_NETS(nb);
  SGRL_CHECK(al16(wf, 0, zs_s) && (!with_split || (plane & 3) == 0), "the fold planes (wf, zs_s, plane) must be 16-byte aligned (TMA operands)");
  FoldDesc d;
  SGRL_TRY(fold_desc_of(src, dst, rows, n, d));
  return fold_sym_launch(params, zs_p, wf, zs_s, plane, with_split ? 1 : 0, d, nb, ST(stream), grid);
}

int sgrl_unfold_sym(const float* gf, int64_t zs_w, float* grads, int64_t zs_g, const int64_t* src, const int64_t* dst, const int32_t* rows, int n,
                    int nb, int32_t* grid, sgrl_stream_t stream) {
  SGRL_CHECK(gf && grads, "null pointer");
  SGRL_NETS(nb);
  FoldDesc d;
  SGRL_TRY(fold_desc_of(src, dst, rows, n, d));
  return unfold_sym_launch(gf, zs_w, grads, zs_g, d, nb, ST(stream), grid);
}

int sgrl_gemm(const float* A, int lda, int trans_a, const float* B, int ldb, int trans_b, float* C, int ldc, int M, int N, int K,
              float alpha, const float* bias, const float* rowdiv, int relu, int accumulate, int splitk, int use_tc,
              sgrl_stream_t stream) {
  SGRL_CHECK(A && B && C, "null pointer");
  GemmP g = gemm_defaults();
  g.A = A; g.lda = lda; g.transA = trans_a; g.B = B; g.ldb = ldb; g.transB = trans_b; g.C = C; g.ldc = ldc;
  g.M = M; g.N = N; g.K = K; g.alpha = alpha; g.bias = bias; g.rowdiv = rowdiv; g.relu = relu; g.accumulate = accumulate;
  SGRL_CHECK(splitk <= 1 || (accumulate && !bias), "splitk > 1 needs accumulate = 1 and no bias");
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
  SGRL_CHECK(splitk <= 1 || (accumulate && !bias), "splitk > 1 needs accumulate = 1 and no bias");
  g.splitk = (splitk < 1 || det_enabled()) ? 1 : splitk;
  SGRL_CHECK(gemm_tc_eligible(g), "shape/epilogue not eligible for the tcgen05 path");
  return gemm_tc(g, ST(stream));
}

int sgrl_gemm_desc(const SgrlGemmDesc* d, SgrlGemmPlanInfo* info, sgrl_stream_t stream) {
  SGRL_CHECK(d != nullptr, "null descriptor");
  SGRL_CHECK(d->n >= 1 && d->n <= TC_MAXG, "gemm_desc: 1..4 problems");
  SGRL_CHECK(d->use_tc >= 0 && d->use_tc <= 2, "gemm_desc: use_tc must be 0, 1 or 2");
  GemmP g[TC_MAXG];
  for (int i = 0; i < d->n; ++i) {
    const SgrlGemmProblem& s = d->pr[i];
    SGRL_CHECK((s.A || s.gram_z) && s.B && s.C, "gemm_desc: null A, B or C");
    SGRL_CHECK(s.M >= 0 && s.N >= 0 && s.K >= 1 && s.nb >= 1 && s.nb <= 64, "gemm_desc: M, N >= 0, K >= 1, nb 1..64");
    SGRL_CHECK(s.splitk >= 1 && s.splitk <= 64, "gemm_desc: splitk 1..64");
    SGRL_CHECK(s.splitk == 1 || (s.accumulate && !s.bias), "gemm_desc: splitk > 1 needs accumulate = 1 and no bias");
    SGRL_CHECK((s.B_hi == nullptr) == (s.B_lo == nullptr), "gemm_desc: B_hi and B_lo go together");
    SGRL_CHECK(!s.gram_z || !s.A, "gemm_desc: A and gram_z exclude each other");
    SGRL_CHECK(s.gram_z || (!s.gram_f && !s.gram_g), "gemm_desc: gram_f / gram_g need gram_z");
    GemmP& p = g[i];
    p = gemm_defaults();
    p.A = s.A; p.zsA = s.zs_a; p.lda = s.lda; p.transA = s.trans_a != 0;
    p.B = s.B_hi ? s.B_hi : s.B; p.Bhi = s.B_hi; p.Blo = s.B_lo; p.zsB = s.zs_b; p.ldb = s.ldb; p.transB = s.trans_b != 0;
    p.C = s.C; p.zsC = s.zs_c; p.ldc = s.ldc; p.M = s.M; p.N = s.N; p.K = s.K; p.nb = s.nb;
    p.alpha = s.alpha; p.relu = s.relu != 0; p.bias = s.bias; p.zsBias = s.zs_bias; p.rowdiv = s.rowdiv; p.zsRow = s.zs_rowdiv;
    p.colscale = s.colscale; p.colscale_n = s.colscale_n;
    p.mask = s.mask; p.zsMask = s.zs_mask; p.ldmask = s.ldmask;
    p.res1 = s.res1; p.zsR1 = s.zs_res1; p.ldr1 = s.ldres1; p.res2 = s.res2; p.zsR2 = s.zs_res2; p.ldr2 = s.ldres2;
    p.accumulate = s.accumulate != 0; p.splitk = det_enabled() ? 1 : s.splitk;
    p.rowsum = s.rowsum; p.zsRowsum = s.zs_rowsum; p.gdcols = s.gd; p.zsGd = s.zs_gd;
    p.gramZ = s.gram_z; p.zsGramZ = s.zs_gram_z; p.gramF = s.gram_f; p.gramG = s.gram_g;
    p.sm2_ok = d->sm2_ok != 0; p.prec = d->use_tc == 2 ? 1 : 0;
  }
  TcPlanInfo rep[TC_MAXG];
  memset(rep, 0, sizeof(rep));
  int launches = 1;
  if (d->use_tc == 0) {
    const GemmP& p = g[0];
    SGRL_CHECK(d->n == 1, "gemm_desc: the SIMT kernels take one problem");
    SGRL_CHECK(!p.Bhi && !p.rowsum && !p.gdcols && !p.gramZ, "gemm_desc: B_hi/B_lo, rowsum, gd and gram_z need the tcgen05 path");
    SGRL_CHECK(d->bn == -1 && d->split == -1 && d->csk == -1 && d->sm2 == -1 && d->persist == -1 && d->tma_store == -1 && d->group == -1,
               "gemm_desc: planner overrides need the tcgen05 path");
    rep[0] = TcPlanInfo{gemm_skinny_eligible(p) ? 1 : 0, GB_N, p.transA, p.transB, 0, 0, 0, 0, p.splitk, 0, 1, 0, -1};
    SGRL_TRY(gemm_simt(p, ST(stream)));
  } else {
    for (int i = 0; i < d->n; ++i)
      SGRL_CHECK(g[i].M == 0 || g[i].N == 0 || gemm_tc_eligible(g[i]), "gemm_desc: shape/operands not eligible for the tcgen05 path");
    TcForce f;
    f.bn = d->bn; f.split = d->split; f.csk = d->csk; f.sm2 = d->sm2; f.persist = d->persist; f.tma_store = d->tma_store; f.group = d->group;
    if (d->n == 1) SGRL_TRY(gemm_tc_ex(g[0], f, rep, ST(stream)));
    else SGRL_TRY(gemm_tc_group_ex(g, d->n, f, rep, &launches, ST(stream)));
  }
  if (info) {
    memset(info, 0, sizeof(*info));
    for (int i = 0; i < d->n; ++i) memcpy(&info->pr[i], &rep[i], sizeof(SgrlGemmPlan));
    info->launches = launches;
  }
  return 0;
}
static_assert(sizeof(SgrlGemmPlan) == sizeof(TcPlanInfo), "SgrlGemmPlan mirrors TcPlanInfo");
static_assert(sizeof(SgrlGemmDesc) == 4 * sizeof(SgrlGemmProblem) + 40, "SgrlGemmDesc: the layout _lib.GemmDesc mirrors");

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
  launch_k(td3_smooth_action_kernel, grid_for_flat(n * 4), 256, 0, ST(stream), pi_target, noise, next_action, noise_clip, max_action,
           (long long)n, (const SgrlTd3Hparams*)nullptr, 1LL);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_td3_smooth_action_hp(const float* pi_target, const float* noise, float* next_action, const SgrlTd3Hparams* hp,
                              int64_t per_seed, float max_action, int64_t n, sgrl_stream_t stream) {
  SGRL_CHECK(pi_target && noise && next_action && hp, "null pointer");
  SGRL_CHECK(per_seed >= 1 && n % per_seed == 0, "n must be a multiple of per_seed");
  launch_k(td3_smooth_action_kernel, grid_for_flat(n * 4), 256, 0, ST(stream), pi_target, noise, next_action, 0.f, max_action,
           (long long)n, hp, (long long)per_seed);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_td3_smooth_action_rng(const float* pi_target, float* next_action, float* noise_out, float policy_noise, float noise_clip,
                               float max_action, int64_t n, uint64_t seed, const int32_t* draw, sgrl_stream_t stream) {
  SGRL_CHECK(pi_target && next_action && draw, "null pointer");
  launch_k(td3_smooth_action_rng_kernel, grid_for_flat(n), 256, 0, ST(stream), pi_target, next_action, noise_out, policy_noise, noise_clip,
           max_action, (long long)n, (unsigned long long)seed, draw, (const SgrlTd3Hparams*)nullptr, 1LL);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_td3_smooth_action_rng_hp(const float* pi_target, float* next_action, float* noise_out, const SgrlTd3Hparams* hp,
                                  int64_t per_seed, float max_action, int64_t n, uint64_t seed, const int32_t* draw,
                                  sgrl_stream_t stream) {
  SGRL_CHECK(pi_target && next_action && draw && hp, "null pointer");
  SGRL_CHECK(per_seed >= 1 && n % per_seed == 0, "n must be a multiple of per_seed");
  launch_k(td3_smooth_action_rng_kernel, grid_for_flat(n), 256, 0, ST(stream), pi_target, next_action, noise_out, 0.f, 0.f, max_action,
           (long long)n, (unsigned long long)seed, draw, hp, (long long)per_seed);
  SGRL_LAUNCH_OK();
  return 0;
}

// grid.y = seed: the kernels offset every per-seed operand by blockIdx.y (td3.cuh); one seed is the single-agent entry point
static int critic_loss(const float* q1, const float* q2, const float* tq1, const float* tq2, const float* reward, const float* done,
                       const int32_t* tok_graph, const float* tok_weight, float* target, float* dq1, float* dq2, float* loss, float discount,
                       float reward_scale, int T, double* reward_stats, int G, int K, const SgrlTd3Hparams* hp, cudaStream_t st) {
  SGRL_CHECK(q1 && q2 && tq1 && tq2 && reward && done && tok_graph && target && dq1 && dq2 && loss, "null pointer");
  SGRL_CHECK(K >= 1 && K <= MAX_NETS / 2 && T >= 1 && G >= 1, "bad seed count or batch");
  int gx = ceil_div(T, 256); if (gx > NUM_SMS) gx = NUM_SMS;
  if (det_enabled()) gx = 1;      // the loss scalar: one add
  launch_k(td3_critic_loss_kernel, dim3(gx, K), 256, 0, st, q1, q2, tq1, tq2, reward, done, tok_graph, tok_weight, target, dq1, dq2, loss, discount, reward_scale, T, reward_stats, G, hp);
  SGRL_LAUNCH_OK();
  return 0;
}

static int actor_loss(const float* q1, const float* tok_weight, float* dq1, float* loss, int T, int K, cudaStream_t st) {
  SGRL_CHECK(q1 && dq1 && loss, "null pointer");
  SGRL_CHECK(K >= 1 && K <= MAX_NETS && T >= 1, "bad seed count or batch");
  int gx = ceil_div(T, 256); if (gx > NUM_SMS) gx = NUM_SMS;
  if (det_enabled()) gx = 1;      // the loss scalar: one add
  launch_k(td3_actor_loss_kernel, dim3(gx, K), 256, 0, st, q1, tok_weight, dq1, loss, T);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_td3_critic_loss(const float* q1, const float* q2, const float* tq1, const float* tq2, const float* reward, const float* done,
                         const int32_t* tok_graph, const float* tok_weight, float* target, float* dq1, float* dq2, float* loss, float discount,
                         float reward_scale, int T, double* reward_stats, int G, sgrl_stream_t stream) {
  return critic_loss(q1, q2, tq1, tq2, reward, done, tok_graph, tok_weight, target, dq1, dq2, loss, discount, reward_scale, T, reward_stats,
                     G, 1, nullptr, ST(stream));
}

int sgrl_td3_critic_loss_seeds(const float* q, const float* tq, const float* reward, const float* done, const int32_t* tok_graph,
                               const float* tok_weight, float* target, float* dq, float* loss, float discount, float reward_scale, int T,
                               double* reward_stats, int G, int K, sgrl_stream_t stream) {
  SGRL_CHECK(q && tq && dq, "null pointer");
  const long long h = (long long)K * T;      // critic2 of seed k is net K + k
  return critic_loss(q, q + h, tq, tq + h, reward, done, tok_graph, tok_weight, target, dq, dq + h, loss, discount, reward_scale, T,
                     reward_stats, G, K, nullptr, ST(stream));
}

int sgrl_td3_critic_loss_seeds_hp(const float* q, const float* tq, const float* reward, const float* done, const int32_t* tok_graph,
                                  const float* tok_weight, float* target, float* dq, float* loss, const SgrlTd3Hparams* hp, int T,
                                  double* reward_stats, int G, int K, sgrl_stream_t stream) {
  SGRL_CHECK(q && tq && dq && hp, "null pointer");
  const long long h = (long long)K * T;
  return critic_loss(q, q + h, tq, tq + h, reward, done, tok_graph, tok_weight, target, dq, dq + h, loss, 0.f, 0.f, T,
                     reward_stats, G, K, hp, ST(stream));
}

int sgrl_td3_actor_loss(const float* q1, const float* tok_weight, float* dq1, float* loss, int T, sgrl_stream_t stream) {
  return actor_loss(q1, tok_weight, dq1, loss, T, 1, ST(stream));
}

int sgrl_td3_actor_loss_seeds(const float* q1, const float* tok_weight, float* dq1, float* loss, int T, int K, sgrl_stream_t stream) {
  return actor_loss(q1, tok_weight, dq1, loss, T, K, ST(stream));
}

int sgrl_td3_part_stats(const float* q, const float* target, const float* q1, const float* reward, const int32_t* parts, int P, int T,
                        int G, int K, const SgrlTd3Hparams* hp, double* out, sgrl_stream_t stream) {
  SGRL_CHECK(q && target && reward && parts && hp && out, "null pointer");
  SGRL_CHECK(P >= 1 && P <= 64, "P must be 1..64");
  SGRL_CHECK(K >= 1 && K <= MAX_NETS / 2, "K must be 1..8");
  SGRL_CHECK(T >= 1 && G >= 1, "empty batch");
  launch_k(td3_part_stats_kernel, dim3(P, K), 256, 0, ST(stream), q, target, q1, reward, parts, T, G, K, hp, out);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_sumsq(const float* g, int64_t n, float* out, sgrl_stream_t stream) { return sgrl_sumsq_nets(g, n, 1, out, stream); }

int sgrl_sumsq_nets(const float* g, int64_t n, int nets, float* out, sgrl_stream_t stream) {
  SGRL_CHECK(g && out, "null pointer");
  SGRL_CHECK(aligned16(g), "gradient arena must be 16-byte aligned");
  SGRL_CHECK(nets >= 1 && nets <= MAX_NETS && (nets == 1 || (n & 3) == 0), "nets must be 1..16, n % 4 == 0 for several nets");
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
  int nb = grid_for_flat(n); if (nb > SUMSQ_MAX_BLOCKS / nets) nb = SUMSQ_MAX_BLOCKS / nets;      // blocks per net
  launch_k(sumsq_partial_kernel, dim3(nb, nets), 256, 0, ST(stream), g, (long long)n, part);
  SGRL_LAUNCH_OK();
  launch_k(sumsq_final_kernel, nets, 256, 0, ST(stream), (const float*)part, nb, out);
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
  return sgrl_adam_clip_groups(p, g, m, v, n, 1, 1, sumsq, step, lr, beta1, beta2, eps, max_norm, grad_scale, p_hi, p_lo, stream);
}

// one body for sgrl_adam_clip_groups (hp == NULL: lr and max_norm for every group) and sgrl_adam_clip_groups_hp
static int adam_clip(float* p, const float* g, float* m, float* v, int64_t n_net, int nets, int groups, const float* sumsq,
                     const int32_t* step, double lr, const SgrlTd3Hparams* hp, int lr_of, double beta1, double beta2, double eps,
                     float max_norm, float grad_scale, float* p_hi, float* p_lo, cudaStream_t st) {
  SGRL_CHECK(p && g && m && v && sumsq && step, "null pointer");
  SGRL_CHECK(nets >= 1 && nets <= MAX_NETS && groups >= 1 && groups <= nets && nets % groups == 0, "nets must be 1..16, a multiple of groups");
  SGRL_CHECK((p_hi == nullptr) == (p_lo == nullptr) && (!p_hi || (aligned16(p_hi) && aligned16(p_lo))), "p_hi/p_lo go together, 16-byte aligned");
  SGRL_CHECK((n_net & 3) == 0 && aligned16(p) && aligned16(g) && aligned16(m) && aligned16(v), "arenas must be 16-byte aligned, n % 4 == 0");
  const int64_t n = n_net * nets;
  AdamCfg c{lr, beta1, beta2, (float)beta1, (float)beta2, (float)(1.0 - beta1), (float)(1.0 - beta2), (float)eps, max_norm, grad_scale};
  launch_k(adam_clip_kernel, grid_for_flat(n), 256, 0, st, p, g, m, v, (long long)n, sumsq, step, c, p_hi, p_lo, (long long)n_net, nets, groups,
           hp, lr_of);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_adam_clip_groups(float* p, const float* g, float* m, float* v, int64_t n_net, int nets, int groups, const float* sumsq,
                          const int32_t* step, double lr, double beta1, double beta2, double eps, float max_norm, float grad_scale,
                          float* p_hi, float* p_lo, sgrl_stream_t stream) {
  return adam_clip(p, g, m, v, n_net, nets, groups, sumsq, step, lr, nullptr, 0, beta1, beta2, eps, max_norm, grad_scale, p_hi, p_lo,
                   ST(stream));
}

int sgrl_adam_clip_groups_hp(float* p, const float* g, float* m, float* v, int64_t n_net, int nets, int groups, const float* sumsq,
                             const int32_t* step, const SgrlTd3Hparams* hp, int lr_of, double beta1, double beta2, double eps,
                             float grad_scale, float* p_hi, float* p_lo, sgrl_stream_t stream) {
  SGRL_CHECK(hp != nullptr, "null pointer");
  SGRL_CHECK(lr_of == SGRL_ACTOR || lr_of == SGRL_CRITIC, "lr_of must be SGRL_ACTOR or SGRL_CRITIC");
  return adam_clip(p, g, m, v, n_net, nets, groups, sumsq, step, 0.0, hp, lr_of, beta1, beta2, eps, 0.f, grad_scale, p_hi, p_lo,
                   ST(stream));
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
  launch_k(polyak_kernel, grid_for_flat(n), 256, 0, ST(stream), target, source, (long long)n, tau, (float)(1.0 - (double)tau), t_hi, t_lo,
           (long long)n_split, (const SgrlTd3Hparams*)nullptr, 1, 0LL, 0LL);
  SGRL_LAUNCH_OK();
  return 0;
}

int sgrl_polyak_hp(float* target, const float* source, int nets, int64_t live_net, int64_t dead_net, const SgrlTd3Hparams* hp, int K,
                   float* t_hi, float* t_lo, sgrl_stream_t stream) {
  SGRL_CHECK(target && source && hp, "null pointer");
  SGRL_CHECK(K >= 1 && nets >= K && nets <= MAX_NETS && nets % K == 0, "nets must be 1..16, a multiple of K");
  SGRL_CHECK(live_net > 0 && dead_net >= 0 && live_net % 64 == 0 && dead_net % 64 == 0, "per-net sizes must be multiples of 64 floats");
  SGRL_CHECK((t_hi == nullptr) == (t_lo == nullptr) && (!t_hi || (aligned16(t_hi) && aligned16(t_lo))), "t_hi/t_lo go together, 16-byte aligned");
  SGRL_CHECK(aligned16(target) && aligned16(source), "arenas must be 16-byte aligned");
  const long long n_live = (long long)nets * live_net, n = n_live + (long long)nets * dead_net;
  launch_k(polyak_kernel, grid_for_flat(n), 256, 0, ST(stream), target, source, n, 0.f, 0.f, t_hi, t_lo, n_live, hp, K,
           (long long)live_net, (long long)dead_net);
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
  ReplayParts<SGRL_REPLAY_MAX_PARTS> P;
  P.n = 1;
  SGRL_TRY(replay_part(P.p[0], rows, row_floats, capacity, obs_dim, act_dim, batch));
  ReplayOut o{obs, action, next_obs, reward, done};
  return replay_gather(P, &batch, reinterpret_cast<const long long*>(idx), o, ST(stream));
}

// parts[0..n) (n <= CAP, checked by the caller) -> one gather launch with CAP descriptors in its parameter bank
extern "C++" {
template <int CAP>
static int replay_gather_parts(const SgrlReplayPart* parts, int n, const int64_t* idx, float* obs, float* action, float* next_obs,
                               float* reward, float* done, cudaStream_t st) {
  ReplayParts<CAP> P;
  P.n = n;
  int B[CAP];
  for (int i = 0; i < n; ++i) {
    const SgrlReplayPart& s = parts[i];
    SGRL_TRY(replay_part(P.p[i], s.rows, s.row_floats, s.capacity, s.obs_dim, s.act_dim, s.batch));
    B[i] = s.batch;
  }
  ReplayOut o{obs, action, next_obs, reward, done};
  return replay_gather(P, B, reinterpret_cast<const long long*>(idx), o, st);
}
}  // extern "C++"

int sgrl_replay_gather_packed(const SgrlReplayPart* parts, int n_parts, const int64_t* idx, float* obs, float* action, float* next_obs,
                              float* reward, float* done, sgrl_stream_t stream) {
  SGRL_CHECK(parts && idx && obs && action && next_obs && reward && done, "null pointer");
  SGRL_CHECK(n_parts >= 1 && n_parts <= SGRL_REPLAY_MAX_PARTS, "n_parts must be 1..64");
  return replay_gather_parts<SGRL_REPLAY_MAX_PARTS>(parts, n_parts, idx, obs, action, next_obs, reward, done, ST(stream));
}

int sgrl_replay_gather_seeds(const SgrlReplayPart* parts, int n_parts, int n_seeds, const int64_t* idx, float* obs, float* action,
                             float* next_obs, float* reward, float* done, sgrl_stream_t stream) {
  SGRL_CHECK(parts && idx && obs && action && next_obs && reward && done, "null pointer");
  SGRL_CHECK(n_seeds >= 1 && n_seeds <= SGRL_REPLAY_MAX_SEEDS, "n_seeds must be 1..8");
  SGRL_CHECK(n_parts >= n_seeds && n_parts % n_seeds == 0 && n_parts / n_seeds <= SGRL_REPLAY_MAX_PARTS,
             "n_parts must be n_seeds x (1..64 parts per seed)");
  const int M = n_parts / n_seeds;
  for (int k = 1; k < n_seeds; ++k)        // every seed's part i has seed 0's geometry: seed k's rows land at k x the per-seed totals
    for (int i = 0; i < M; ++i) {
      const SgrlReplayPart &a = parts[i], &b = parts[k * M + i];
      if (b.obs_dim != a.obs_dim || b.act_dim != a.act_dim || b.batch != a.batch) {
        char m[200];
        snprintf(m, sizeof(m), "seed %d part %d: obs_dim, act_dim, batch (%d, %d, %d) differ from seed 0's (%d, %d, %d)", k, i,
                 (int)b.obs_dim, (int)b.act_dim, (int)b.batch, (int)a.obs_dim, (int)a.act_dim, (int)a.batch);
        return fail(-2, m, __FILE__, __LINE__);
      }
    }
  return replay_gather_parts<SGRL_REPLAY_MAX_SEED_PARTS>(parts, n_parts, idx, obs, action, next_obs, reward, done, ST(stream));
}

int sgrl_seed_copy(const SgrlSeedPlane* planes, int n_planes, int K, const int32_t* dst, const int32_t* src, int n_pairs,
                   sgrl_stream_t stream) {
  SGRL_CHECK(planes && dst && src, "null pointer");
  SGRL_CHECK(n_planes >= 1 && n_planes <= SGRL_SEED_COPY_MAX_PLANES, "n_planes must be 1..32");
  SGRL_CHECK(n_pairs >= 1 && n_pairs <= SGRL_SEED_COPY_MAX_PAIRS, "n_pairs must be 1..7");
  SGRL_CHECK(K >= 1 && K <= MAX_NETS / 2, "K must be 1..8");
  SeedCopyArgs a;
  memset(&a, 0, sizeof(a));
  int nps[SGRL_SEED_COPY_MAX_PLANES];
  for (int i = 0; i < n_planes; ++i) {
    const SgrlSeedPlane& q = planes[i];
    SGRL_CHECK(q.base != nullptr, "null plane base");
    SGRL_CHECK(aligned16(q.base), "plane base must be 16-byte aligned");
    SGRL_CHECK(q.n_net > 0 && (q.n_net & 3) == 0, "n_net must be a positive multiple of 4");
    SGRL_CHECK(q.nets_per_seed >= 1 && q.nets_per_seed <= 2, "nets_per_seed must be 1..2");
    a.base[i] = q.base; a.n4[i] = q.n_net / 4; nps[i] = q.nets_per_seed;
  }
  for (int p = 0; p < n_pairs; ++p) {
    SGRL_CHECK(dst[p] >= 0 && dst[p] < K && src[p] >= 0 && src[p] < K, "seed index outside [0, K)");
    SGRL_CHECK(dst[p] != src[p], "dst == src");
    for (int q = 0; q < n_pairs; ++q) {
      SGRL_CHECK(q == p || dst[q] != dst[p], "repeated dst");
      SGRL_CHECK(dst[p] != src[q], "a seed is both a dst and a src");
    }
    a.dst[p] = dst[p]; a.src[p] = src[p];
  }
  a.n_planes = n_planes; a.K = K;
  return seed_copy(a, nps, n_pairs, ST(stream));
}

int sgrl_replay_scatter(float* rows, int64_t row_floats, int64_t capacity, const int64_t* dst, const float* staged, int n, sgrl_stream_t stream) {
  SGRL_CHECK(rows && dst && staged, "null pointer");
  SGRL_CHECK(row_floats > 0 && capacity > 0 && n >= 0, "bad replay row geometry");
  return replay_scatter(rows, row_floats, reinterpret_cast<const long long*>(dst), staged, n, capacity, ST(stream));
}

}  // extern "C"
