/* sgrl_b200 — C ABI of the B200-native SET (subequivariant transformer) hot path.
 *
 * The reference (alpc91/SGRL) has no FFI layer: its hot path sits behind Python nn.Module
 * objects.  Each entry point below names the reference code it replaces (file:line relative
 * to the reference's src/).  The Python modules in sgrl_b200/ (same class names, constructor
 * signatures, state_dict keys as the reference) bind these with ctypes; INTEGRATION.md shows
 * the stub a reference maintainer would add.
 *
 * Conventions: every pointer is a DEVICE pointer to contiguous row-major fp32 (int32 for
 * indices) owned by the caller (exceptions: the HOST descriptor arrays of
 * sgrl_replay_gather_packed, sgrl_replay_gather_seeds, sgrl_seed_copy, sgrl_input_grad and sgrl_fold_sym / sgrl_unfold_sym); the library allocates nothing, never synchronises and never
 * throws.  Every call enqueues work on the given cudaStream_t (pass
 * torch.cuda.current_stream().cuda_stream) and returns 0, or a negative code with a
 * thread-local message in sgrl_last_error().  Calls are re-entrant per stream.
 * Tokens are packed limb-major per graph: token t = limb (t - cu_limbs[g]) of graph g.
 */
#ifndef SGRL_B200_H
#define SGRL_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* sgrl_stream_t; /* cudaStream_t */

enum { SGRL_ACTOR = 0, SGRL_CRITIC = 1 };

int sgrl_version(void);
const char* sgrl_last_error(void);
/* kernels launched by the library so far in this process (bench.py reports the per-step delta) */
long long sgrl_launch_count(void);
/* bench-only device timing of kernel classes [simt gemm, tcgen05 gemm, feature (K1), attention (K2), other]:
 * sgrl_profile(1) brackets every launch of the first four classes with CUDA events on its stream (adds
 * ~2 us per launch: never enabled inside a timed throughput pass); sgrl_profile_collect() after a
 * synchronize returns per class the summed milliseconds, work (flops or algorithmic bytes) and launches. */
int sgrl_profile(int enable);
int sgrl_profile_collect(double* ms, double* work, long long* count, int ncls);
/* developer aid (tools/gemm_trace.py): while buf64 (device, 64 x int64) is set, CTA 0 of every tcgen05 GEMM writes
 * SM-clock timestamps of its pipeline phases there; NULL switches it off */
int sgrl_gemm_trace(long long* buf64);

/* ---- layouts ------------------------------------------------------------------------
 * One "net" = one reference TransformerModel (SEActor.py:170-287).  A module's arena holds
 * nb nets: [live net0 | live net1 | .. | dead net0 | ..]; tensor i of net z lives at
 * z*live_floats + offset (live) or nb*live_floats + z*dead_floats + offset (dead =
 * nn.MultiheadAttention leftovers kept only for state_dict compatibility, SEActor.py:34-36). */
int sgrl_param_count(int kind, int n_layers);
int sgrl_param_info(int kind, int n_layers, int index, char* name, int name_cap,
                    int* rows, int* cols /*0 => 1-D*/, int64_t* offset, int* live);
int sgrl_arena_floats(int kind, int n_layers, int64_t* live_floats, int64_t* dead_floats);
/* floats of forward stash per net instance for T tokens (keep=1: training, every layer kept;
 * keep=0: rollout, layers alias) and of backward workspace */
int64_t sgrl_stash_floats(int kind, int n_layers, int64_t T, int keep);
int64_t sgrl_ws_floats(int n_layers, int64_t T);
/* offset (floats) and floats-per-token of a named stash buffer (layer<0: global buffer); for tests */
int sgrl_stash_info(int kind, int n_layers, int64_t T, int keep, const char* name, int layer,
                    int64_t* offset, int* per_token);

/* ---- whole-network passes -------------------------------------------------------------- */
typedef struct {
  int32_t kind;        /* SGRL_ACTOR: TransformerModel(41 -> 3), SGRL_CRITIC: (44 -> 1) */
  int32_t n_layers;    /* attention_layers (3) */
  int32_t nb;          /* nets evaluated together, 1..16 (2 = twin critics; 2K = the twin critics of K seeds) */
  int32_t T;           /* limb-tokens in the packed batch */
  int32_t G;           /* graphs (samples) in the batch */
  int32_t keep;        /* 1: keep every layer's activations for backward */
  int32_t use_tc;      /* 1: tcgen05 tensor-core projections (3xTF32, fp32 parity), 0: fp32 SIMT, 2: tcgen05 with BF16-rounded
                        * inputs and one MMA pass (fp32 accumulate) — the separately reported reduced-precision mode */
  int32_t max_limbs;   /* largest graph of the batch (2..16), 0 = unknown: sizes the attention kernel's shared-memory staging */
  const float* params; /* live arena of the module (nb * live_floats) */
  float* grads;        /* gradient arena, same layout; may be NULL for forward / data-only backward */
  float* stash;        /* nb * stash_stride floats */
  int64_t stash_stride;
  float* ws;           /* nb * ws_stride floats (backward only) */
  int64_t ws_stride;
  const int32_t* cu_limbs; /* (G+1) token offsets of the graphs */
  const int32_t* rel_off;  /* (G) float offset of each graph's (n,n,3) relation table, NULL = all 0 */
  const float* relation;   /* packed relation tables, utils.py:476-481 */
  const int32_t* rank3;    /* (T,3) traversal ranks of each token's limb, utils.py:368-409 */
  float max_action;
  int32_t in_nets;     /* net z reads its obs / act at obs + (z % in_nets) * obs_stride (act likewise); 0 = nb.  Seed-batched
                        * twin critics (nets [critic1 of seeds 0..K-1 | critic2 of seeds 0..K-1]) use nb = 2K, in_nets = K */
  /* optional (both or neither): tf32 hi/lo split of `params` (same layout; sgrl_split_tf32, or kept fresh by
   * sgrl_adam_clip / sgrl_polyak) so the tcgen05 projections stream pre-split weights by TMA */
  const float* params_hi;
  const float* params_lo;
} SgrlNetCall;

/* SEPolicy.forward (SEActor.py:334-347) / SECritic.forward, Q1 (SECritic.py:66-104), all of
 * TransformerModel.forward (SEActor.py:237-287), MyTransformerEncoderLayer.forward (:82-125)
 * and multi_head_attention_forward (subequivariant_attentions.py:82-154).
 * obs (T,41); act (T,3) for critics (NULL for actors); obs_stride/act_stride = floats between
 * consecutive input blocks (0: shared), net z reading block z % in_nets.  out: nb x (T x 3) tanh-squashed actions scaled by
 * max_action, or nb x (T x 1) per-limb Q. */
int sgrl_set_forward(const SgrlNetCall* call, const float* obs, int64_t obs_stride, const float* act,
                     int64_t act_stride, float* out, int64_t out_stride, sgrl_stream_t stream);

/* loss.backward() through the same modules (agent.py:151,171).  dout: nb x (T x 3|1) gradient
 * w.r.t. `out`.  need_wgrad=1 accumulates parameter gradients into call->grads (zero it first);
 * dact (critics, nullable): nb x (T x 3) gradient w.r.t. the action input (agent.py:167).
 * sgrl_set_backward is sgrl_set_backward_dobs with dobs = NULL. */
int sgrl_set_backward(const SgrlNetCall* call, const float* dout, int64_t dout_stride, int need_wgrad,
                      float* dact, int64_t dact_stride, sgrl_stream_t stream);
/* The same pass, plus (dobs non-NULL) the gradient w.r.t. the observation input: nb x (T x 41), dobs_stride floats
 * between the nets' blocks (>= 41 * T when nb > 1), overwritten.  Works with need_wgrad = 0 too.  It costs one extra
 * launch at the end of the pass, which reads the finished backward workspace and the forward stash; with dobs = NULL
 * the pass launches and computes exactly what sgrl_set_backward does.  Deterministic (no atomics). */
int sgrl_set_backward_dobs(const SgrlNetCall* call, const float* dout, int64_t dout_stride, int need_wgrad,
                           float* dact, int64_t dact_stride, float* dobs, int64_t dobs_stride, sgrl_stream_t stream);

/* ---- single kernels (unit tests, profiling) ---------------------------------------------- */
/* K1: Z=[X P^T | gd], G=Z^T Z, F=||G||+1 (subequivariant_attentions.py:90-96; SEActor.py:93-100,
 * 256-262).  X (T,3,128); v0 (T,3,8) or NULL (head variant, C=136); P1,P2 (30,C) (P2/Z2 NULL for
 * one projection); outputs Z,Z2 (T,3,32), F (T) and G (T,544): G is symmetric, so vec(G) is kept as its upper
 * triangle (528 entries, row-major i<=j, zero-padded to 544 = 17 k-blocks) and contracted against triangle-folded
 * weights W'[o][p(i,j)] = W[o][32i+j] + W[o][32j+i].  The backward takes dG in the same packed form. */
int sgrl_inv_feature_fwd(const float* X, const float* v0, const float* gd, const float* P1, const float* P2,
                         float* Z, float* Z2, float* G, float* F, int T, sgrl_stream_t stream);
int sgrl_inv_feature_bwd(const float* dG, const float* dF, const float* Z, const float* F, float* dZ, int T,
                         sgrl_stream_t stream);
/* K2: attention core (subequivariant_attentions.py:109-151) on packed graphs.  qkv (T,768) holds
 * the already /F-divided and scaled q|k|v; vgp (T,3,252); gd (T,3,2); rel_w (2,3), rel_b (2) or NULL.
 * Outputs o (T,256), og (T,3,256), p (T,2,16) (p[t, h, j] = 0 for j >= the graph's limbs); p NULL: inference pass, no
 * probability store.  The backward's drel_w (2,3) needs relation (the tables the forward's bias was formed from). */
int sgrl_attention_fwd(const float* qkv, const float* vgp, const float* gd, const float* rel_w, const float* rel_b,
                       const int32_t* cu_limbs, const int32_t* rel_off, const float* relation, int G,
                       int max_limbs /* largest graph (2..16), 0 = unknown: sizes the shared-memory staging */,
                       float* o, float* og, float* p, sgrl_stream_t stream);
int sgrl_attention_bwd(const float* qkv, const float* vgp, const float* gd, const float* p,
                       const float* d_o, const float* d_og, const int32_t* cu_limbs, const int32_t* rel_off,
                       const float* relation, int G, int max_limbs, float* dqkv, float* dvgp, float* drel_w /*nullable, accumulates*/,
                       sgrl_stream_t stream);
/* K3: C[M,N] = epi(alpha * A B^T): every nn.Linear call site (SURVEY.md Appendix G).
 * trans_a/trans_b as in csrc/gemm_simt.cuh; bias/rowdiv nullable; relu 0/1; use_tc as above.
 * splitk > 1 lets K be split with atomic adds into C: it requires accumulate = 1 and no bias (refused otherwise). */
int sgrl_gemm(const float* A, int lda, int trans_a, const float* B, int ldb, int trans_b, float* C, int ldc,
              int M, int N, int K, float alpha, const float* bias, const float* rowdiv, int relu, int accumulate,
              int splitk, int use_tc, sgrl_stream_t stream);

/* same with the weight operand B pre-split into its tf32 hi/lo parts (tcgen05 path only) */
int sgrl_gemm_presplit(const float* A, int lda, int trans_a, const float* B_hi, const float* B_lo, int ldb, int trans_b, float* C,
                       int ldc, int M, int N, int K, float alpha, const float* bias, const float* rowdiv, int relu, int accumulate,
                       int splitk, sgrl_stream_t stream);
/* The fused projections of the tcgen05 forward schedule (csrc/net.cuh; unit tests and micro-benchmarks call them here).
 * All take the weight pre-split (W_hi / W_lo, sgrl_split_tf32) and run one tcgen05 launch.
 *  sgrl_gemm_gram: C (T,N) = epi( tri(Z_t^T Z_t) W'^T + b ), the vec(G) consumers linear_g1 / linear1_g
 *    (subequivariant_attentions.py:93-97, SEActor.py:96-101, 259-263) with the Gram rows generated inside the GEMM from
 *    Z (T,3,32) instead of being read from HBM; W' (N,544) is the triangle-folded weight.  F (T, nullable) = ||G||_F + 1,
 *    G (T,544, nullable) = the generated rows (what sgrl_inv_feature_fwd writes).
 *  sgrl_gemm_gd: Z (T3,32) = [A W^T | gd]: the invariant projections g_proj / g_proj2 / g_proj3 (W (30,K) inside a matrix of
 *    row stride ldw whose two following rows are readable) with columns 30,31 of row 3t+r taken from gd (T,3,2)
 *    (subequivariant_attentions.py:91-92, SEActor.py:94-95, 109-110).
 *  sgrl_gemm_pair: two independent projections C_i = A_i W_i^T + b_i [relu] in ONE grouped launch. */
int sgrl_gemm_gram(const float* Z, const float* W_hi, const float* W_lo, const float* bias, float* C, int ldc, float* F, float* G,
                   int T, int N, int relu, sgrl_stream_t stream);
int sgrl_gemm_gd(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw, const float* gd, float* Z, int T3, int K,
                 sgrl_stream_t stream);
int sgrl_gemm_pair(const float* A0, int lda0, const float* W0_hi, const float* W0_lo, const float* b0, float* C0, int ldc0, int M0, int N0,
                   int K0, const float* A1, int lda1, const float* W1_hi, const float* W1_lo, const float* b1, float* C1, int ldc1, int M1,
                   int N1, int K1, int relu, sgrl_stream_t stream);
/* The whole GEMM contract of the library's projections in one descriptor (kernel tests: every variant, epilogue and
 * instance layout that csrc/net.cuh launches can be reached and checked from here).  One problem, per instance z < nb
 * (z-stride 0 = the operand is shared by every instance; every pointer but A, B and C is nullable):
 *   v = alpha * sum_k A(m,k) B(n,k) (+ bias[n]) -> relu -> / rowdiv[m] -> * colscale (n < colscale_n) -> mask[m][n] > 0 ? v : 0
 *       -> + res1[m][n] + res2[m][n] -> C[m][n] = v, or C[m][n] += v (accumulate)
 *   rowsum[m] += alpha * sum_k A(m,k); gd: columns 30, 31 of row m = 3t+r replaced by gd[t][r][0..1] (N = 32);
 *   gram_z (M,96) set: row m of A is the packed Gram triangle of Z_m (K = 544, B pre-split), gram_f[m] = ||G_m||_F + 1,
 *   gram_g (M,544) = the generated rows.  A(m,k), B(n,k) as in sgrl_gemm.  splitk > 1 lets the tcgen05 model split K
 *   with atomics (requires accumulate = 1 and no bias).  B_hi/B_lo (both or neither): B pre-split, tcgen05 only. */
typedef struct {
  const float* A; int64_t zs_a; int32_t lda, trans_a;
  const float* B; const float* B_hi; const float* B_lo; int64_t zs_b; int32_t ldb, trans_b;
  float* C; int64_t zs_c; int32_t ldc, M, N, K;
  float alpha; int32_t relu;
  const float* bias; int64_t zs_bias;
  const float* rowdiv; int64_t zs_rowdiv;
  float colscale; int32_t colscale_n;
  const float* mask; int64_t zs_mask;
  const float* res1; int64_t zs_res1;
  const float* res2; int64_t zs_res2;
  int32_t ldmask, ldres1, ldres2, accumulate;
  float* rowsum; int64_t zs_rowsum;
  const float* gd; int64_t zs_gd;
  const float* gram_z; int64_t zs_gram_z;   /* zs_gram_z also strides gram_f and gram_g */
  float* gram_f; float* gram_g;
  int32_t splitk, nb;
} SgrlGemmProblem;
/* n = 1..4 problems; n > 1 runs them like the networks' grouped projections (one launch when their kernel variants agree).
 * use_tc: 0 fp32 SIMT (n = 1, no rowsum / gd / gram), 1 tcgen05 3xTF32, 2 tcgen05 BF16-input.  sm2_ok: the hint the
 * networks give the tile model (inference pass).  Overrides of the tcgen05 planner, -1 = its model (every
 * field -1: exactly the plan sgrl_gemm and the networks get): bn 64 | 128; split = atomic split-K factor (needs splitk > 1);
 * csk 0 | 2 | 3 cluster split-K ranks; sm2, persist, tma_store, group 0 | 1.  An override the shape or epilogue cannot take
 * is refused with nothing enqueued. */
typedef struct {
  SgrlGemmProblem pr[4];
  int32_t n, use_tc, sm2_ok;
  int32_t bn, split, csk, sm2, persist, tma_store, group;
} SgrlGemmDesc;
/* What was launched, per problem.  path: 0 SIMT tile kernel, 1 skinny kernel, 2 tcgen05.  split: atomic split-K factor
 * (sk_x: folded into blockIdx.x); cluster: cluster split-K ranks (1 = none); tma_c: TMA-store epilogue; epi: the epilogue
 * class the tcgen05 tile kernel selects (0 plain, 1 /rowdiv (+colscale), 2 relu mask, 3 residuals, 4 accumulate, 5 split-K
 * atomics, 6 generic, 7 [X P^T | gd]), -1 where that choice is not made (SIMT, TMA-store and persistent epilogues). */
typedef struct { int32_t path, bn, amn, bmn, bpre, sm2, gram, persist, split, sk_x, cluster, tma_c, epi; } SgrlGemmPlan;
typedef struct { SgrlGemmPlan pr[4]; int32_t launches, pad_; } SgrlGemmPlanInfo;
int sgrl_gemm_desc(const SgrlGemmDesc* d, SgrlGemmPlanInfo* info /* nullable */, sgrl_stream_t stream);
/* ---- the kernels around the projections (csrc/misc.cuh) and the triangle fold (csrc/feature.cuh), one entry point each ----
 * Each launches exactly what the network passes launch: the same host launcher picks the grid (its caps, the deterministic-mode
 * override) and, for the LayerNorms, the float4 / scalar access of every operand from its pointer, leading dimension and z-stride.
 * nb = 1..16 instances on the grid, instance z of an operand at pointer + z * its z-stride (zs_s: forward stash, zs_w: backward
 * workspace, zs_p: parameters, zs_g: gradients, as in csrc/net.cuh).  grid (nullable, 3 ints) receives the grid launched.  T >= 0
 * tokens.  Outputs marked "+=" accumulate; everything else is overwritten.  Refused with nothing enqueued: NULL required pointers,
 * nb outside 1..16, T < 0, and each operand a kernel reads or writes as float4 (float2: dog) that is not 16-byte (8-byte) aligned
 * together with its leading dimension and z-stride.
 *  sgrl_embed_fwd: the input stage (SEActor.py:237-251): obs (T,41) of block z % in_nets (zs_obs), act (T,3) of critics (ng = 20;
 *    NULL for actors, ng = 17), rank3 (T,3) rows 0..14 of the positional tables E0 (15,42), E1 (15,42), E2 (15,44); Wg (128,8),
 *    We (128,ng), be (128).  V0 (T,24), GD (T,6), SH[:, :ng] (row stride ldsh) copies of obs / act; VG (T,3,128) and H (row stride ldh).
 *  sgrl_input_grad: d obs (T,41) (zs_dobs) as sgrl_set_backward_dobs gathers it; dz (3L), dog (L), P (L) are HOST arrays of device
 *    pointers, L = 1..8; dzh2, gph, dout, out, w3 for actors (ng = 17) only.  Deterministic.
 *  sgrl_pos_embed_bwd: dE0, dE1, dE2 += scatter of dH (T,128, row stride ldh) over rank3.
 *  sgrl_layernorm_fwd: x = a + b (b nullable), y = LN(x) gamma + beta (row stride ldy; y2 nullable, a second copy), stats (T,2) =
 *    mean, rstd; x (nullable) is stored with row stride 128.
 *  sgrl_layernorm_bwd: dx = LN backward of dy1 + dy2 (dy2 nullable); dgamma, dbeta (both or neither) +=; with rd_* (all or none)
 *    also rd_out = dx / rd_F and rd_dF[t] += -<dx, rd_y> / rd_F (rd_y, rd_F in the stash, rd_dF, rd_out in the workspace).
 *  sgrl_matapply_fwd / _bwd: R = Z (3x32) M (32x32) per token; backward dZ = dR M^T, dT = Z^T dR / F, dF[t] += -<Z^T dR, M> / F.
 *  sgrl_matapply_l5_fwd / _bwd: the same fused with linear5 and the residuals: Vn = Vg + dV + (Z M) W5^T (W5 (128,32)), R = Z M
 *    kept unless NULL; backward from dVn with dR = dVn W5.
 *  sgrl_actor_out_fwd / _bwd: w = R (3,32) wd, out_i = max_action tanh(sum_r V0[r][5+i] w_r), W3 = w; backward dR and dwd +=.
 *  sgrl_rowdiv_bwd: backward of y = t / F (* colscale on the first cs_n <= N columns): dy = g cs / F with g = src (or dy in place),
 *    dF[t] += -<g, y> / F.
 *  sgrl_colsum: out[n] += alpha * sum_m X[m][n] (zs_x, zs_o).
 *  sgrl_block_copy: dst = (add ? dst : 0) + src (+ src2) on an (M, N) block.
 *  sgrl_fold_sym / sgrl_unfold_sym: n = 1..17 folds W'[o][p(i,j)] = W[o][32i+j] + W[o][32j+i] of the (rows[m],1024) matrix at
 *    params + src[m] into wf + dst[m] (row stride 544; with_split: tf32 hi / lo planes at + plane, + 2 plane), and the gradient
 *    grads + src[m] += unfold of gf + dst[m].  src, dst, rows are HOST arrays. */
int sgrl_embed_fwd(const float* obs, int64_t zs_obs, const float* act, int64_t zs_act, const int32_t* rank3, const float* Wg, const float* We,
                   const float* be, const float* E0, const float* E1, const float* E2, int64_t zs_p, float* V0, float* GD, float* SH, int ldsh,
                   float* VG, float* H, int ldh, int64_t zs_s, int T, int ng, int nb, int in_nets, int32_t* grid, sgrl_stream_t stream);
int sgrl_input_grad(const float* dvg0, const float* dh0, const float* dzh, const float* dzh2, const float* dsh, int ldsh,
                    const float* const* dz, const float* const* dog, const float* const* P, const float* Wg, const float* We, const float* gg,
                    const float* gph, int ng, const float* dout, int64_t zs_do, const float* out, const float* w3, float max_action,
                    float* dobs, int64_t zs_dobs, const int32_t* cu_limbs, int G, int T, int L, int64_t zs_w, int64_t zs_s, int64_t zs_p, int nb,
                    int32_t* grid, sgrl_stream_t stream);
int sgrl_pos_embed_bwd(const float* dH, int ldh, int64_t zs_w, const int32_t* rank3, float* dE0, float* dE1, float* dE2, int64_t zs_g, int T, int nb,
                       int32_t* grid, sgrl_stream_t stream);
int sgrl_layernorm_fwd(const float* a, int lda, const float* b, int ldb, const float* gamma, const float* beta, int64_t zs_p, float* x, float* y,
                       int ldy, float* y2, int ldy2, float* stats, int64_t zs_s, int T, int nb, int32_t* grid, sgrl_stream_t stream);
int sgrl_layernorm_bwd(const float* dy1, int ld1, const float* dy2, int ld2, const float* x, int ldx, const float* stats, int64_t zs_s,
                       const float* gamma, int64_t zs_p, float* dx, int lddx, int64_t zs_w, float* dgamma, float* dbeta, int64_t zs_g,
                       const float* rd_y, int rd_ldy, const float* rd_F, float* rd_dF, float* rd_out, int rd_ldout, int T, int nb,
                       int32_t* grid, sgrl_stream_t stream);
int sgrl_matapply_fwd(const float* Z, const float* M, float* R, int64_t zs_s, int T, int nb, int32_t* grid, sgrl_stream_t stream);
int sgrl_matapply_bwd(const float* dR, const float* Z, const float* M, const float* F, int64_t zs_s, float* dZ, float* dT, float* dF, int64_t zs_w,
                      int T, int nb, int32_t* grid, sgrl_stream_t stream);
int sgrl_matapply_l5_fwd(const float* Z, const float* M, const float* W5, int64_t zs_p, const float* Vg, const float* dV, float* R, float* Vn,
                         int64_t zs_s, int T, int nb, int32_t* grid, sgrl_stream_t stream);
int sgrl_matapply_l5_bwd(const float* dVn, const float* W5, int64_t zs_p, const float* Z, const float* M, const float* F, int64_t zs_s, float* dZ,
                         float* dT, float* dF, int64_t zs_w, int T, int nb, int32_t* grid, sgrl_stream_t stream);
int sgrl_actor_out_fwd(const float* R, const float* V0, const float* wd, int64_t zs_p, float* W3, float* out, int64_t zs_s, float max_action, int T,
                       int nb, int32_t* grid, sgrl_stream_t stream);
int sgrl_actor_out_bwd(const float* dout, int64_t zs_do, const float* out, const float* R, const float* V0, int64_t zs_s, const float* wd,
                       int64_t zs_p, float* dR, int64_t zs_w, float* dwd, int64_t zs_g, float max_action, int T, int nb, int32_t* grid,
                       sgrl_stream_t stream);
int sgrl_rowdiv_bwd(float* dy, int lddy, int64_t zs_w, const float* y, int ldy, const float* F, int64_t zs_s, float* dF, int N, float colscale,
                    int cs_n, const float* src, int ldsrc, int64_t zs_src, int T, int nb, int32_t* grid, sgrl_stream_t stream);
int sgrl_colsum(const float* X, int ldx, int64_t zs_x, float* out, int64_t zs_o, int M, int N, float alpha, int nb, int32_t* grid,
                sgrl_stream_t stream);
int sgrl_block_copy(float* dst, int ldd, int64_t zs_d, const float* src, int lds, int64_t zs_src, const float* src2, int lds2, int64_t zs_src2,
                    int M, int N, int add, int nb, int32_t* grid, sgrl_stream_t stream);
int sgrl_fold_sym(const float* params, int64_t zs_p, float* wf, int64_t zs_s, int64_t plane, int with_split, const int64_t* src, const int64_t* dst,
                  const int32_t* rows, int n, int nb, int32_t* grid, sgrl_stream_t stream);
int sgrl_unfold_sym(const float* gf, int64_t zs_w, float* grads, int64_t zs_g, const int64_t* src, const int64_t* dst, const int32_t* rows, int n,
                    int nb, int32_t* grid, sgrl_stream_t stream);
/* hi = tf32_rna(w), lo = tf32_rna(w - hi): the operand split of the 3xTF32 tensor-core projections, done once per
 * optimizer step for weights instead of once per tile load */
int sgrl_split_tf32(const float* w, float* hi, float* lo, int64_t n, sgrl_stream_t stream);

/* ---- K5: TD3 glue (agent.py:127-148,167) -------------------------------------------------- */
/* The per-step TD3 scalars of one seed.  The _hp entry points below take a DEVICE table of such rows, one per seed (seed k =
 * row k), and their kernels read it when they run: a captured CUDA graph applies the values the table holds at replay, so a
 * caller changes hyper-parameters between updates by rewriting the table in stream order, without recapturing.  Adam's betas
 * and eps, max_action, policy_freq and grad_scale stay by-value arguments shared by all seeds. */
typedef struct {
  double actor_lr, critic_lr;      /* Adam learning rates (doubles, like the Python floats torch.optim.Adam forms its step from) */
  float discount, reward_scale;    /* critic target r * reward_scale + (1 - done) * discount * min(Q1', Q2') */
  float policy_noise, noise_clip;  /* target-policy smoothing: eps ~ N(0, policy_noise^2) clipped to +-noise_clip */
  float tau, one_minus_tau;        /* Polyak; one_minus_tau = (float)(1.0 - (double)tau), as sgrl_polyak forms it */
  float max_norm, pad_;            /* clip_grad_norm_ threshold, <= 0: no clipping */
} SgrlTd3Hparams;                  /* 48 bytes */
int sgrl_td3_smooth_action(const float* pi_target, const float* noise, float* next_action, float noise_clip,
                           float max_action, int64_t n, sgrl_stream_t stream);
/* The same with the target-policy noise drawn inside the kernel: eps ~ N(0, policy_noise^2) (agent.py:128,
 * torch.randn_like(action) * policy_noise) from Philox4x32-10 keyed by `seed`, counter = {element / 4, 0, *draw, 0}
 * (Box-Muller, 4 normals per call).  `draw` is a device counter bumped once per update (sgrl_bump_step), so a replayed
 * CUDA graph draws fresh noise.  noise_out (nullable) receives eps before clipping. */
int sgrl_td3_smooth_action_rng(const float* pi_target, float* next_action, float* noise_out, float policy_noise,
                               float noise_clip, float max_action, int64_t n, uint64_t seed, const int32_t* draw,
                               sgrl_stream_t stream);
/* Both smoothing kernels with per-seed scalars: n = K * per_seed elements, element i belongs to seed i / per_seed (3T for K
 * seeds of T tokens) and takes row i / per_seed's noise_clip (and policy_noise).  The Philox counter and key are those of
 * sgrl_td3_smooth_action_rng, so one seed with the same seed and draw gives the same noise. */
int sgrl_td3_smooth_action_hp(const float* pi_target, const float* noise, float* next_action, const SgrlTd3Hparams* hp,
                              int64_t per_seed, float max_action, int64_t n, sgrl_stream_t stream);
int sgrl_td3_smooth_action_rng_hp(const float* pi_target, float* next_action, float* noise_out, const SgrlTd3Hparams* hp,
                                  int64_t per_seed, float max_action, int64_t n, uint64_t seed, const int32_t* draw,
                                  sgrl_stream_t stream);
/* target = r*scale + (1-done)*discount*min(tq1,tq2) broadcast over limbs; loss (1 float, accumulates)
 * = mse(q1,target)+mse(q2,target); dq1,dq2 = dloss/dq. tok_graph (T) maps token -> sample.
 * tok_weight (T, nullable): weight of each token in the loss for packed mixed-morphology batches
 * (1/(#morphologies * tokens of the token's morphology): the mean over morphologies of the reference's
 * per-morphology loss, src/trainer.py:245-250); NULL = 1/T (one morphology, exactly agent.py:146-148). */
int sgrl_td3_critic_loss(const float* q1, const float* q2, const float* tq1, const float* tq2, const float* reward,
                         const float* done, const int32_t* tok_graph, const float* tok_weight, float* target, float* dq1,
                         float* dq2, float* loss, float discount, float reward_scale, int T,
                         double* reward_stats /*nullable: {sum, sum of squares} of reward*reward_scale over the G graphs, agent.py:158-161*/,
                         int G, sgrl_stream_t stream);
int sgrl_td3_actor_loss(const float* q1, const float* tok_weight, float* dq1, float* loss, int T, sgrl_stream_t stream);
/* The same for K = 1..8 independent seeds sharing the tables (agent.py:136-148, 167 once per seed; sgrl_td3_critic_loss /
 * sgrl_td3_actor_loss are the K = 1 case).  Nets in the seed-batched order: q, tq, dq (2K, T) = [critic1 of seeds 0..K-1 |
 * critic2 of seeds 0..K-1]; reward, done (K, G); target (K, T); loss (K, accumulates); reward_stats (K, 2) or NULL.
 * Actor: q1, dq1 (K, T) (critic1 of each seed), loss (K, accumulates).  One launch each. */
int sgrl_td3_critic_loss_seeds(const float* q, const float* tq, const float* reward, const float* done, const int32_t* tok_graph,
                               const float* tok_weight, float* target, float* dq, float* loss, float discount, float reward_scale, int T,
                               double* reward_stats, int G, int K, sgrl_stream_t stream);
int sgrl_td3_actor_loss_seeds(const float* q1, const float* tok_weight, float* dq1, float* loss, int T, int K, sgrl_stream_t stream);
/* sgrl_td3_critic_loss_seeds with seed k's discount and reward_scale from hp[k] (K rows), the reward statistics included. */
int sgrl_td3_critic_loss_seeds_hp(const float* q, const float* tq, const float* reward, const float* done, const int32_t* tok_graph,
                                  const float* tok_weight, float* target, float* dq, float* loss, const SgrlTd3Hparams* hp, int T,
                                  double* reward_stats, int G, int K, sgrl_stream_t stream);
/* Per-morphology TD3 statistics of a packed (seed-batched) update: for seed k (grid y) and part i (grid x),
 * out[(k*P + i)*4 + 0..3] = critic loss, actor loss (NaN when q1 == NULL), reward mean, reward variance (unbiased; NaN
 * for one sample) over part i's tokens [t0,t1) and graphs [g0,g1) of seed k's block.  parts: DEVICE (P,4) int32
 * {t0,t1,g0,g1} within one seed's block; q (2K,T) [critic1 of seeds | critic2 of seeds], target (K,T), q1 (K,T) or NULL,
 * reward (K,G); hp (K rows) supplies each seed's reward_scale.  fp64 accumulation, fixed-order reductions, no atomics.
 * Critic loss = sum over the part's tokens of (q1-y)^2 + (q2-y)^2 over its token count, actor loss = -sum(q1) over its token
 * count (src/agent.py:146-148, 167 restricted to the part), rewards = reward * reward_scale rounded to fp32 as the critic-loss
 * kernel forms them.  A part that is empty or lies outside [0,T) x [0,G) gets four NaNs.  One launch of P x K CTAs. */
int sgrl_td3_part_stats(const float* q, const float* target, const float* q1, const float* reward, const int32_t* parts,
                        int P, int T, int G, int K, const SgrlTd3Hparams* hp, double* out, sgrl_stream_t stream);

/* ---- K6: optimizer (agent.py:150-156,170-178; common/functional.py:7-10) -------------------- */
int sgrl_sumsq(const float* g, int64_t n, float* out /*accumulates*/, sgrl_stream_t stream);
/* clip_grad_norm_(max_norm) + Adam(lr,b1,b2,eps) in one pass over the flat live arena.  sumsq: device
 * scalar with sum(g^2) (after the all-reduce); step: device int, the 1-based step count to apply;
 * grad_scale multiplies g first (1/world_size).  lr / betas / eps are doubles, like the Python floats torch.optim.Adam
 * derives 1 - beta and the bias corrections from. */
int sgrl_adam_clip(float* p, const float* g, float* m, float* v, int64_t n, const float* sumsq, const int32_t* step,
                   double lr, double beta1, double beta2, double eps, float max_norm, float grad_scale,
                   float* p_hi /*nullable: refreshed tf32 split of p*/, float* p_lo, sgrl_stream_t stream);
/* Per-seed clip_grad_norm_ + Adam over an arena of `nets` nets of n_net floats each (agent.py:150-156,170-178 once per seed).
 * sgrl_sumsq_nets writes (accumulates) one sum of squares per net into out[nets]; sgrl_adam_clip_groups clips net z by the norm
 * over its group {z' : z' % groups == z % groups} (seed-batched twin critics: nets k and K + k, groups = K).  One launch each
 * (sumsq: two); sgrl_sumsq / sgrl_adam_clip are the one-net, one-group case. */
int sgrl_sumsq_nets(const float* g, int64_t n_net, int nets, float* out, sgrl_stream_t stream);
int sgrl_adam_clip_groups(float* p, const float* g, float* m, float* v, int64_t n_net, int nets, int groups, const float* sumsq,
                          const int32_t* step, double lr, double beta1, double beta2, double eps, float max_norm, float grad_scale,
                          float* p_hi, float* p_lo, sgrl_stream_t stream);
/* sgrl_adam_clip_groups with group g's learning rate and clip threshold from hp[g] (`groups` rows): actor_lr when
 * lr_of = SGRL_ACTOR, critic_lr when SGRL_CRITIC, and max_norm (<= 0: group g is not clipped).  sumsq must hold every net's
 * sum of squares, whatever the thresholds. */
int sgrl_adam_clip_groups_hp(float* p, const float* g, float* m, float* v, int64_t n_net, int nets, int groups, const float* sumsq,
                             const int32_t* step, const SgrlTd3Hparams* hp, int lr_of, double beta1, double beta2, double eps,
                             float grad_scale, float* p_hi, float* p_lo, sgrl_stream_t stream);
int sgrl_bump_step(int32_t* step, sgrl_stream_t stream);
int sgrl_polyak(float* target, const float* source, int64_t n, float tau,
                float* t_hi /*nullable: refreshed tf32 split of target[0:n_split]*/, float* t_lo, int64_t n_split, sgrl_stream_t stream);
/* sgrl_polyak over a module arena of `nets` nets ([live nets | dead nets], live_net and dead_net floats per net, multiples of
 * 64: sgrl_arena_floats) with net z, live or dead, updated by the tau / one_minus_tau of seed z % K (hp: K rows, nets % K == 0).
 * t_hi / t_lo (nullable) cover the live nets. */
int sgrl_polyak_hp(float* target, const float* source, int nets, int64_t live_net, int64_t dead_net, const SgrlTd3Hparams* hp, int K,
                   float* t_hi, float* t_lo, sgrl_stream_t stream);

/* Call before recording an event on `stream` that another stream will wait on when the last work on `stream` was a
 * kernel of this library and the stream is not being captured: enqueues an empty non-programmatic launch (see
 * csrc/net.cuh, stream_fence: events recorded right after a programmatic-launch kernel did not reliably order the
 * waiting stream in eager execution).  No-op during stream capture. */
int sgrl_stream_fence(sgrl_stream_t stream);

/* Deterministic mode: enable = 1 / 0 switches it, -1 only queries; returns the previous state (default: environment
 * variable SGRL_DETERMINISTIC, off).  While on, two runs of sgrl_set_backward / the TD3 glue kernels on the same inputs give
 * BIT-IDENTICAL gradients, like the reference's CPU autograd (src/agent.py:151,171): weight-gradient GEMMs are not split
 * over K, the small cross-CTA reductions sum in a fixed order and no work is forked to side streams (csrc/common.cuh).
 * The mode is read when work is enqueued: captured CUDA graphs keep the mode they were captured in. */
int sgrl_deterministic(int enable);

/* ---- K7: device-resident replay storage (common/buffer.py:35-126; SURVEY.md 8f rank 2) --------
 * One transition = one packed row [obs (obs_dim) | action (act_dim) | next_obs (obs_dim) | reward | done] of
 * row_floats = 2*obs_dim + act_dim + 2 floats; `rows` holds `capacity` of them in HBM.
 * sgrl_replay_gather replaces ReplayBuffer.sample / get_batch's five fancy-index gathers + five H2D copies
 * (buffer.py:103-145): idx (batch) int64 row numbers (device) -> obs (batch,obs_dim), action (batch,act_dim),
 * next_obs, reward (batch), done (batch).  The outputs may be the static input buffers of a TD3 update.
 * sgrl_replay_scatter writes n staged rows to rows[dst[i]] (add_transition for transitions already on the device,
 * buffer.py:74-84). */
int sgrl_replay_gather(const float* rows, int64_t row_floats, int64_t capacity, const int64_t* idx, int batch, int obs_dim, int act_dim,
                       float* obs, float* action, float* next_obs, float* reward, float* done, sgrl_stream_t stream);
int sgrl_replay_scatter(float* rows, int64_t row_floats, int64_t capacity, const int64_t* dst, const float* staged, int n,
                        sgrl_stream_t stream);

/* One gather over up to 64 replay buffers (one per morphology of a packed multi-morphology update, src/trainer.py:239-253).
 * `parts` is a HOST array (the one exception to the device-pointer convention), read while the call enqueues the launch and
 * free to reuse when it returns.  Part i contributes parts[i].batch rows; idx (device, sum of batch) holds the row numbers of
 * all parts one after the other (negative ones wrap like numpy's).  The outputs are the parts' batches concatenated: sample b
 * of part i goes to obs / next_obs + (O_i + b*obs_dim_i), action + (A_i + b*act_dim_i) and reward / done [R_i + b], where O_i,
 * A_i and R_i sum obs_dim*batch, act_dim*batch and batch over the parts before i.  With obs_dim = 41*n and act_dim = 3*n this is
 * the packed token layout of Agent.update_packed.  Each part's geometry is checked like sgrl_replay_gather's. */
typedef struct {
  const float* rows;   /* the part's buffer: capacity rows of row_floats = 2*obs_dim + act_dim + 2 */
  int64_t row_floats, capacity;
  int32_t obs_dim, act_dim, batch, pad_;
} SgrlReplayPart;
int sgrl_replay_gather_packed(const SgrlReplayPart* parts, int n_parts, const int64_t* idx, float* obs, float* action,
                              float* next_obs, float* reward, float* done, sgrl_stream_t stream);

/* The packed gather of n_seeds independent agents (a seed-batched packed update): `parts` (HOST, as above) holds n_seeds x M
 * descriptors seed-major, M = n_parts / n_seeds parts (one per morphology) per seed; n_seeds 1..8, M 1..64.  Part i of every
 * seed must have the obs_dim, act_dim and batch of seed 0's part i (the seeds share the morphologies; their buffers, capacities
 * and indices are their own), anything else is refused.  The layout is sgrl_replay_gather_packed's over all n_parts parts, so
 * seed k's rows start at k x the per-seed totals: the block of seed k in a seed-batched update's inputs. */
int sgrl_replay_gather_seeds(const SgrlReplayPart* parts, int n_parts, int n_seeds, const int64_t* idx, float* obs, float* action,
                             float* next_obs, float* reward, float* done, sgrl_stream_t stream);

/* ---- population-based training (SeedBatchedAgent.exploit) ------------------------------------ */
/* One per-seed state array of a seed-batched agent: nets of n_net floats, net z at base + z * n_net.  Seed k of K owns the
 * nets k + j*K for j < nets_per_seed (1: actors; 2: twin critics [critic1 of seeds | critic2 of seeds]). */
typedef struct { float* base; int64_t n_net; int32_t nets_per_seed, pad_; } SgrlSeedPlane;
/* For every pair p, copy seed src[p]'s nets onto seed dst[p]'s nets in every plane.  One launch.
 * planes, dst and src are HOST arrays, read while the call enqueues.  Limits: 1..32 planes, 1..7 pairs.
 * Refused with nothing enqueued: a seed index outside [0, K); dst[p] == src[p]; a repeated dst; a seed that is both a dst
 * and a src in one call; n_net not a multiple of 4; a base that is not 16-byte aligned.  Also refused: NULL arrays or bases,
 * K outside 1..8, n_net <= 0, nets_per_seed outside 1..2. */
int sgrl_seed_copy(const SgrlSeedPlane* planes, int n_planes, int K, const int32_t* dst, const int32_t* src, int n_pairs,
                   sgrl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif
