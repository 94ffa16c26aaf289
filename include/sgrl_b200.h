/* sgrl_b200 — C ABI of the B200-native SET (subequivariant transformer) hot path.
 *
 * The reference (alpc91/SGRL) has no FFI layer: its hot path sits behind Python nn.Module
 * objects.  Each entry point below names the reference code it replaces (file:line relative
 * to the reference's src/).  The Python modules in sgrl_b200/ (same class names, constructor
 * signatures, state_dict keys as the reference) bind these with ctypes; INTEGRATION.md shows
 * the stub a reference maintainer would add.
 *
 * Conventions: every pointer is a DEVICE pointer to contiguous row-major fp32 (int32 for
 * indices) owned by the caller (one exception: the HOST descriptor array of
 * sgrl_replay_gather_packed); the library allocates nothing, never synchronises and never
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
  int32_t nb;          /* nets evaluated together on the same input (2 = twin critics) */
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
  float pad_;
  /* optional (both or neither): tf32 hi/lo split of `params` (same layout; sgrl_split_tf32, or kept fresh by
   * sgrl_adam_clip / sgrl_polyak) so the tcgen05 projections stream pre-split weights by TMA */
  const float* params_hi;
  const float* params_lo;
} SgrlNetCall;

/* SEPolicy.forward (SEActor.py:334-347) / SECritic.forward, Q1 (SECritic.py:66-104), all of
 * TransformerModel.forward (SEActor.py:237-287), MyTransformerEncoderLayer.forward (:82-125)
 * and multi_head_attention_forward (subequivariant_attentions.py:82-154).
 * obs (T,41); act (T,3) for critics (NULL for actors); obs_stride/act_stride = floats between
 * the inputs of consecutive nets (0: shared).  out: nb x (T x 3) tanh-squashed actions scaled by
 * max_action, or nb x (T x 1) per-limb Q. */
int sgrl_set_forward(const SgrlNetCall* call, const float* obs, int64_t obs_stride, const float* act,
                     int64_t act_stride, float* out, int64_t out_stride, sgrl_stream_t stream);

/* loss.backward() through the same modules (agent.py:151,171).  dout: nb x (T x 3|1) gradient
 * w.r.t. `out`.  need_wgrad=1 accumulates parameter gradients into call->grads (zero it first);
 * dact (critics, nullable): nb x (T x 3) gradient w.r.t. the action input (agent.py:167). */
int sgrl_set_backward(const SgrlNetCall* call, const float* dout, int64_t dout_stride, int need_wgrad,
                      float* dact, int64_t dact_stride, sgrl_stream_t stream);

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
 * Outputs o (T,256), og (T,3,256), p (T,2,16). */
int sgrl_attention_fwd(const float* qkv, const float* vgp, const float* gd, const float* rel_w, const float* rel_b,
                       const int32_t* cu_limbs, const int32_t* rel_off, const float* relation, int G,
                       int max_limbs /* largest graph (2..16), 0 = unknown: sizes the shared-memory staging */,
                       float* o, float* og, float* p, sgrl_stream_t stream);
int sgrl_attention_bwd(const float* qkv, const float* vgp, const float* gd, const float* p,
                       const float* d_o, const float* d_og, const int32_t* cu_limbs, const int32_t* rel_off,
                       const float* relation, int G, int max_limbs, float* dqkv, float* dvgp, float* drel_w /*nullable, accumulates*/,
                       sgrl_stream_t stream);
/* K3: C[M,N] = epi(alpha * A B^T): every nn.Linear call site (SURVEY.md Appendix G).
 * trans_a/trans_b as in csrc/gemm_simt.cuh; bias/rowdiv nullable; relu 0/1; use_tc as above. */
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
/* hi = tf32_rna(w), lo = tf32_rna(w - hi): the operand split of the 3xTF32 tensor-core projections, done once per
 * optimizer step for weights instead of once per tile load */
int sgrl_split_tf32(const float* w, float* hi, float* lo, int64_t n, sgrl_stream_t stream);

/* ---- K5: TD3 glue (agent.py:127-148,167) -------------------------------------------------- */
int sgrl_td3_smooth_action(const float* pi_target, const float* noise, float* next_action, float noise_clip,
                           float max_action, int64_t n, sgrl_stream_t stream);
/* The same with the target-policy noise drawn inside the kernel: eps ~ N(0, policy_noise^2) (agent.py:128,
 * torch.randn_like(action) * policy_noise) from Philox4x32-10 keyed by `seed`, counter = {element / 4, 0, *draw, 0}
 * (Box-Muller, 4 normals per call).  `draw` is a device counter bumped once per update (sgrl_bump_step), so a replayed
 * CUDA graph draws fresh noise.  noise_out (nullable) receives eps before clipping. */
int sgrl_td3_smooth_action_rng(const float* pi_target, float* next_action, float* noise_out, float policy_noise,
                               float noise_clip, float max_action, int64_t n, uint64_t seed, const int32_t* draw,
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

/* ---- K6: optimizer (agent.py:150-156,170-178; common/functional.py:7-10) -------------------- */
int sgrl_sumsq(const float* g, int64_t n, float* out /*accumulates*/, sgrl_stream_t stream);
/* clip_grad_norm_(max_norm) + Adam(lr,b1,b2,eps) in one pass over the flat live arena.  sumsq: device
 * scalar with sum(g^2) (after the all-reduce); step: device int, the 1-based step count to apply;
 * grad_scale multiplies g first (1/world_size).  lr / betas / eps are doubles, like the Python floats torch.optim.Adam
 * derives 1 - beta and the bias corrections from. */
int sgrl_adam_clip(float* p, const float* g, float* m, float* v, int64_t n, const float* sumsq, const int32_t* step,
                   double lr, double beta1, double beta2, double eps, float max_norm, float grad_scale,
                   float* p_hi /*nullable: refreshed tf32 split of p*/, float* p_lo, sgrl_stream_t stream);
int sgrl_bump_step(int32_t* step, sgrl_stream_t stream);
int sgrl_polyak(float* target, const float* source, int64_t n, float tau,
                float* t_hi /*nullable: refreshed tf32 split of target[0:n_split]*/, float* t_lo, int64_t n_split, sgrl_stream_t stream);

/* Call before recording an event on `stream` that another stream will wait on when the last work on `stream` was a
 * kernel of this library and the stream is not being captured: enqueues an empty non-programmatic launch (see
 * csrc/net.cuh, stream_fence: events recorded right after a programmatic-launch kernel did not reliably order the
 * waiting stream in eager execution).  No-op during stream capture or with SGRL_PDL=0. */
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

#ifdef __cplusplus
}
#endif
#endif
