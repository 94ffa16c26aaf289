// K5/K6 — TD3 glue and the fused optimizer pass (src/agent.py:127-187, functional.py:7-10).
#pragma once
#include "../../include/sgrl_b200.h"
#include "common.cuh"

namespace sgrl {

// Per-seed TD3 scalars (SgrlTd3Hparams, one row per seed) reach the kernels below as a device table that they read when they
// run, so a captured CUDA graph applies whatever the table holds at replay.  hp == NULL: the by-value scalars (the entry points
// without _hp), with the same arithmetic.

// next_action = clamp(pi_target(s') + clamp(noise, +-c), +-max_action)        agent.py:128-133
// hp: element i belongs to seed i / per_seed and is clipped by that seed's noise_clip
__global__ void td3_smooth_action_kernel(const float* __restrict__ a, const float* __restrict__ noise, float* __restrict__ out,
                                         float noise_clip, float max_action, long long n, const SgrlTd3Hparams* __restrict__ hp,
                                         long long per_seed) {
  SGRL_PDL_ENTER();
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
    const float c = hp ? hp[i / per_seed].noise_clip : noise_clip;
    const float nz = fminf(fmaxf(noise[i], -c), c);
    out[i] = fminf(fmaxf(a[i] + nz, -max_action), max_action);
  }
}

// Philox4x32-10 (Salmon et al., SC'11; the counter-based generator behind torch.cuda's and cuRAND's default streams),
// checked against the Random123 known-answer vectors in tests/test_td3_glue.py through the numpy restatement.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
  }
  return c;
}
// Same smoothing with the noise drawn in the kernel: eps ~ N(0, policy_noise^2) (agent.py:128 torch.randn_like * policy_noise),
// four normals per Philox call (counter = {element / 4, 0, draw, 0}, key = seed; Box-Muller).  `draw` is a device counter the
// caller bumps once per update (sgrl_bump_step), so a replayed CUDA graph draws fresh noise every replay.
// hp: element i belongs to seed i / per_seed and takes that seed's policy_noise and noise_clip; the draws themselves (counter,
// key) do not depend on the seed's row.
__global__ void td3_smooth_action_rng_kernel(const float* __restrict__ a, float* __restrict__ out, float* __restrict__ noise_out,
                                             float policy_noise, float noise_clip, float max_action, long long n,
                                             unsigned long long seed, const int* __restrict__ draw,
                                             const SgrlTd3Hparams* __restrict__ hp, long long per_seed) {
  SGRL_PDL_ENTER();
  const unsigned d = (unsigned)*draw;
  const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
  const long long n4 = (n + 3) >> 2;
  for (long long q = blockIdx.x * 256LL + threadIdx.x; q < n4; q += gridDim.x * 256LL) {
    const uint4 r = philox4x32_10(make_uint4((unsigned)q, (unsigned)(q >> 32), d, 0u), key);
    const float u0 = ((float)r.x + 0.5f) * 2.3283064365386963e-10f, u1 = ((float)r.y + 0.5f) * 2.3283064365386963e-10f;
    const float u2 = ((float)r.z + 0.5f) * 2.3283064365386963e-10f, u3 = ((float)r.w + 0.5f) * 2.3283064365386963e-10f;
    const float r0 = sqrtf(-2.f * logf(fminf(u0, 0.99999994f))), r1 = sqrtf(-2.f * logf(fminf(u2, 0.99999994f)));
    float s0, c0, s1, c1;
    sincospif(2.f * u1, &s0, &c0);
    sincospif(2.f * u3, &s1, &c1);
    const float z[4] = {r0 * c0, r0 * s0, r1 * c1, r1 * s1};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long i = q * 4 + k;
      if (i >= n) break;
      float sigma = policy_noise, c = noise_clip;
      if (hp) { const SgrlTd3Hparams& h = hp[i / per_seed]; sigma = h.policy_noise; c = h.noise_clip; }
      const float e = z[k] * sigma;
      if (noise_out) noise_out[i] = e;
      out[i] = fminf(fmaxf(a[i] + fminf(fmaxf(e, -c), c), -max_action), max_action);
    }
  }
}

// target[t] = r[g(t)] * reward_scale + (1 - done[g(t)]) * discount * min(q1t[t], q2t[t])   agent.py:136-139
// dq1 = 2 (q1 - target)/T, dq2 likewise; loss += sum((q1-y)^2 + (q2-y)^2)/T               agent.py:146-148
__global__ void __launch_bounds__(256) td3_critic_loss_kernel(
    const float* __restrict__ q1, const float* __restrict__ q2, const float* __restrict__ tq1, const float* __restrict__ tq2,
    const float* __restrict__ reward, const float* __restrict__ done, const int* __restrict__ tok_graph,
    const float* __restrict__ tok_w,
    float* __restrict__ target, float* __restrict__ dq1, float* __restrict__ dq2, float* __restrict__ loss,
    float discount, float reward_scale, int T, double* __restrict__ rstats, int G, const SgrlTd3Hparams* __restrict__ hp) {
  SGRL_PDL_ENTER();
  __shared__ float red[8];
  {      // seed k = blockIdx.y (sgrl_td3_critic_loss_seeds): its own (T) outputs, (G) rewards, loss and reward statistics,
         // and (hp) its own discount and reward scale
    const long long k = blockIdx.y;
    if (hp) { discount = hp[k].discount; reward_scale = hp[k].reward_scale; }
    q1 += k * T; q2 += k * T; tq1 += k * T; tq2 += k * T; target += k * T; dq1 += k * T; dq2 += k * T;
    reward += k * G; done += k * G; loss += k;
    if (rstats) rstats += 2 * k;
  }
  if (rstats && blockIdx.x == 0 && threadIdx.x < 32) {
    // sum and sum of squares of the scaled rewards (agent.py:158-161 logs their mean / variance): fp64, one warp
    double s1 = 0.0, s2 = 0.0;
    for (int g = threadIdx.x; g < G; g += 32) { const double x = (double)(reward[g] * reward_scale); s1 += x; s2 += x * x; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
    if (threadIdx.x == 0) { rstats[0] = s1; rstats[1] = s2; }
  }
  float acc = 0.f;
  const float invT = 1.f / (float)T;
  for (int t = blockIdx.x * 256 + threadIdx.x; t < T; t += gridDim.x * 256) {
    const int g = tok_graph[t];
    const float y = reward[g] * reward_scale + (1.f - done[g]) * discount * fminf(tq1[t], tq2[t]);
    target[t] = y;
    const float e1 = q1[t] - y, e2 = q2[t] - y;
    // tok_w (packed mixed-morphology batches): weight of token t in the loss = 1 / (#morphologies * tokens of its morphology),
    // i.e. the mean over morphologies of the reference's per-morphology mse; single morphology: 1/T
    const float w = tok_w ? tok_w[t] : invT;
    dq1[t] = 2.f * e1 * w; dq2[t] = 2.f * e2 * w;
    acc += (e1 * e1 + e2 * e2) * (tok_w ? w * (float)T : 1.f);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 8) {
    float s = red[threadIdx.x];
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffu, s, o);
    if (threadIdx.x == 0) atomicAdd(loss, s * invT);
  }
}

// actor loss = -mean(Q1):  dq = -1/T, loss += -sum(q)/T                                    agent.py:167
__global__ void __launch_bounds__(256) td3_actor_loss_kernel(const float* __restrict__ q1, const float* __restrict__ tok_w, float* __restrict__ dq,
                                                             float* __restrict__ loss, int T) {
  SGRL_PDL_ENTER();
  __shared__ float red[8];
  q1 += (long long)blockIdx.y * T; dq += (long long)blockIdx.y * T; loss += blockIdx.y;      // seed blockIdx.y
  float acc = 0.f;
  const float invT = 1.f / (float)T;
  for (int t = blockIdx.x * 256 + threadIdx.x; t < T; t += gridDim.x * 256) {
    const float w = tok_w ? tok_w[t] : invT;
    dq[t] = -w; acc += q1[t] * (tok_w ? w * (float)T : 1.f);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 8) {
    float s = red[threadIdx.x];
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffu, s, o);
    if (threadIdx.x == 0) atomicAdd(loss, -s * invT);
  }
}

// Per-morphology statistics of a packed update (src/agent.py:146-148, 158-162, 167 restricted to one morphology): CTA (i, k) =
// (part, seed) reduces part i's tokens [t0,t1) and graphs [g0,g1) of seed k's block into out[(k*P + i)*4 + 0..3] = {critic loss,
// actor loss (NaN without q1), reward mean, unbiased reward variance (NaN for one sample)}.  fp64 throughout; every thread sums
// a fixed stride and the block combines warps in index order, so the result does not depend on timing.  A part outside the
// block (or empty) gives four NaNs.
__device__ __forceinline__ double block_sum_fixed(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();                                    // red may still be read by the previous call
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < 8; ++w) s += red[w];
  return s;
}

__global__ void __launch_bounds__(256) td3_part_stats_kernel(const float* __restrict__ q, const float* __restrict__ target,
                                                             const float* __restrict__ q1, const float* __restrict__ reward,
                                                             const int* __restrict__ parts, int T, int G, int K,
                                                             const SgrlTd3Hparams* __restrict__ hp, double* __restrict__ out) {
  SGRL_PDL_ENTER();
  __shared__ double red[8];
  const int i = blockIdx.x, k = blockIdx.y;
  const int t0 = parts[4 * i], t1 = parts[4 * i + 1], g0 = parts[4 * i + 2], g1 = parts[4 * i + 3];
  out += ((long long)k * gridDim.x + i) * 4;
  if (t0 < 0 || t1 > T || t0 >= t1 || g0 < 0 || g1 > G || g0 >= g1) {
    if (threadIdx.x < 4) out[threadIdx.x] = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  const float* c1 = q + (long long)k * T;             // critic1 of seed k is net k, critic2 net K + k
  const float* c2 = q + (long long)(K + k) * T;
  const float* y = target + (long long)k * T;
  const float* r = reward + (long long)k * G;
  const float scale = hp[k].reward_scale;
  double sc = 0.0, sa = 0.0, sr = 0.0;
  for (int t = t0 + threadIdx.x; t < t1; t += 256) {
    const double yt = (double)y[t], e1 = (double)c1[t] - yt, e2 = (double)c2[t] - yt;
    sc += e1 * e1 + e2 * e2;
    if (q1) sa += (double)q1[(long long)k * T + t];
  }
  for (int g = g0 + threadIdx.x; g < g1; g += 256) sr += (double)(r[g] * scale);
  sc = block_sum_fixed(sc, red);
  sa = block_sum_fixed(sa, red);
  sr = block_sum_fixed(sr, red);
  const double nt = (double)(t1 - t0), ng = (double)(g1 - g0), mean = sr / ng;
  double sd = 0.0;                                    // second pass: squared deviations from the mean
  for (int g = g0 + threadIdx.x; g < g1; g += 256) { const double d = (double)(r[g] * scale) - mean; sd += d * d; }
  sd = block_sum_fixed(sd, red);
  if (threadIdx.x == 0) {
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    out[0] = sc / nt;
    out[1] = q1 ? -sa / nt : nan;
    out[2] = mean;
    out[3] = g1 - g0 > 1 ? sd / (ng - 1.0) : nan;
  }
}

// sum of squares of a flat gradient buffer                                                  clip_grad_norm_, agent.py:152-155
// Deterministic (no atomics): every block leaves its partial sum in a scratch slot, a second launch adds the partials in
// index order.  The norm feeds the clip coefficient of every data-parallel replica: with an atomic reduction the ranks
// disagreed in its last bit and the replicas drifted apart after ~40 steps (tools/dp_debug.py, bench.py --check-replicas).
// blockIdx.y / the final kernel's blockIdx.x = net: one sum per net of n floats (sgrl_sumsq_nets; one net = sgrl_sumsq).
constexpr int SUMSQ_MAX_BLOCKS = 2048;
__global__ void __launch_bounds__(256) sumsq_partial_kernel(const float* __restrict__ g, long long n, float* __restrict__ partial) {
  SGRL_PDL_ENTER();
  g += blockIdx.y * n; partial += blockIdx.y * gridDim.x;
  __shared__ float red[8];
  float acc = 0.f;
  const long long n4 = n >> 2;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n4; i += gridDim.x * 256LL) {
    const float4 v = ldg4(g + i * 4);
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) { const float v = g[n4 * 4 + threadIdx.x]; acc += v * v; }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 8) {
    float s = red[threadIdx.x];
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffu, s, o);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
  }
}
__global__ void __launch_bounds__(256) sumsq_final_kernel(const float* __restrict__ partial, int nb, float* __restrict__ out) {
  SGRL_PDL_ENTER();
  partial += blockIdx.x * nb; out += blockIdx.x;
  __shared__ double red[8];
  double acc = 0.0;
  for (int i = threadIdx.x; i < nb; i += 256) acc += (double)partial[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w];
    *out += (float)s;
  }
}

// lr / betas arrive as doubles, like the Python floats torch.optim.Adam computes its scalars from: 1 - beta2 is 0.001
// rounded once to fp32 (torch), not 1.f - 0.999f = 0.00099998713 (1.3e-5 off: visible in exp_avg_sq, tests/test_k6_gpu.py)
struct AdamCfg { double lr, beta1d, beta2d; float beta1, beta2, omb1, omb2, eps, max_norm; float grad_scale; };

// One pass over the live arena: clip coefficient from the global norm, Adam moment update,
// parameter step.  `step` lives on the device so the pass can be replayed from a CUDA graph.
//   coef = min(1, max_norm / (||g|| + 1e-6))     (torch.nn.utils.clip_grad_norm_)
//   m = m + (1-b1)(g - m);  v = b2 v + (1-b2) g^2;  p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
// grad_scale pre-multiplies g (1/world_size after a sum all-reduce).
// Per-group clipping (sgrl_adam_clip_groups): the arena holds `nets` nets of n_net floats and sumsq one sum per net; net z is
// clipped by the norm over its group {z' : z' % groups == z % groups}.  One net, one group: the single global norm.
// hp (sgrl_adam_clip_groups_hp): group g takes its step size from row g's actor_lr (lr_of = SGRL_ACTOR) or critic_lr and its
// clip threshold from row g's max_norm; NULL: c.lr and c.max_norm for every group.
// hi/lo (nullable): the refreshed tf32 split of the parameters for the tcgen05 projections (csrc/gemm_tc.cuh).
__device__ __forceinline__ void split_store4(float4 pv, float* hi, float* lo, long long i4) {
  float4 h, l;
  const float* x = &pv.x; float* hh = &h.x; float* ll = &l.x;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const unsigned hb = (__float_as_uint(x[k]) + 0x1000u) & 0xFFFFE000u;
    hh[k] = __uint_as_float(hb);
    ll[k] = __uint_as_float((__float_as_uint(x[k] - hh[k]) + 0x1000u) & 0xFFFFE000u);
  }
  stg4(hi + i4 * 4, h); stg4(lo + i4 * 4, l);
}

__global__ void __launch_bounds__(256) split_tf32_kernel(const float* __restrict__ w, float* __restrict__ hi, float* __restrict__ lo, long long n) {
  SGRL_PDL_ENTER();
  const long long n4 = n >> 2;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n4; i += gridDim.x * 256LL) split_store4(ldg4(w + i * 4), hi, lo, i);
}

__global__ void __launch_bounds__(256) adam_clip_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                        float* __restrict__ v, long long n, const float* __restrict__ sumsq,
                                                        const int* __restrict__ step, AdamCfg c, float* __restrict__ hi, float* __restrict__ lo,
                                                        long long n_net, int nets, int groups,
                                                        const SgrlTd3Hparams* __restrict__ hp, int lr_of) {
  SGRL_PDL_ENTER();
  __shared__ float sh[1 + 2 * MAX_NETS];  // sqrt of the second bias correction; per group: clip coef * grad_scale, step size
  if (threadIdx.x < groups) {
    const int gi = threadIdx.x;
    double lr = c.lr;
    float max_norm = c.max_norm;
    if (hp) { lr = lr_of == SGRL_ACTOR ? hp[gi].actor_lr : hp[gi].critic_lr; max_norm = hp[gi].max_norm; }
    float s = sumsq[gi];
    for (int z = gi + groups; z < nets; z += groups) s += sumsq[z];
    const float nrm = sqrtf(s) * c.grad_scale;
    float coef = 1.f;
    if (max_norm > 0.f) { coef = max_norm / (nrm + 1e-6f); coef = coef > 1.f ? 1.f : coef; }
    sh[1 + gi] = coef * c.grad_scale;
    const double t = (double)(*step);
    sh[1 + MAX_NETS + gi] = (float)(lr / (1.0 - pow(c.beta1d, t)));
    if (gi == 0) sh[0] = (float)sqrt(1.0 - pow(c.beta2d, t));
  }
  __syncthreads();
  const float bc2s = sh[0];
  const long long n4 = n >> 2;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n4; i += gridDim.x * 256LL) {
    const int gi = groups == 1 ? 0 : (int)((i * 4) / n_net) % groups;
    const float gs = sh[1 + gi], step_size = sh[1 + MAX_NETS + gi];
    float4 pv = *reinterpret_cast<float4*>(p + i * 4);
    const float4 gv = ldg4(g + i * 4);
    float4 mv = *reinterpret_cast<float4*>(m + i * 4), vv = *reinterpret_cast<float4*>(v + i * 4);
    float* pp = &pv.x; const float* gg = &gv.x; float* mm = &mv.x; float* vq = &vv.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gk = gg[k] * gs;
      mm[k] = mm[k] + (gk - mm[k]) * c.omb1;
      vq[k] = vq[k] * c.beta2 + c.omb2 * gk * gk;
      pp[k] -= step_size * (mm[k] / (sqrtf(vq[k]) / bc2s + c.eps));
    }
    stg4(p + i * 4, pv); stg4(m + i * 4, mv); stg4(v + i * 4, vv);
    if (hi) split_store4(pv, hi, lo, i);
  }
}

__global__ void bump_step_kernel(int* step) {
  SGRL_PDL_ENTER(); *step += 1; }

// theta_t <- tau*theta + (1-tau)*theta_t                                                    functional.py:7-10
// Rounded exactly like the reference's three fp32 tensor ops (mul, mul, add — no FMA contraction):
// the per-step change tau*(theta-theta_t) ~ 5e-7 is a few ulps of O(1) weights, so op order is visible.
// hi/lo (nullable) cover the first n_split floats (the live prefix of the arena).
// hp (sgrl_polyak_hp): the arena is [live nets | dead nets], n_split floats of live nets of live_net floats, then dead nets of
// dead_net floats; net z (in either part) belongs to seed z % K and takes that seed's tau / one_minus_tau.  Both per-net sizes
// are multiples of 64 floats (layout.h), so a float4 never straddles two nets.
__global__ void __launch_bounds__(256) polyak_kernel(float* __restrict__ tgt, const float* __restrict__ src, long long n,
                                                     float tau, float one_minus_tau, float* __restrict__ hi, float* __restrict__ lo, long long n_split,
                                                     const SgrlTd3Hparams* __restrict__ hp, int K, long long live_net, long long dead_net) {
  SGRL_PDL_ENTER();
  const long long n4 = n >> 2;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n4; i += gridDim.x * 256LL) {
    if (hp) {
      const long long e = i * 4;
      const int k = K == 1 ? 0 : (int)((e < n_split ? e / live_net : (e - n_split) / dead_net) % K);
      tau = hp[k].tau; one_minus_tau = hp[k].one_minus_tau;
    }
    float4 t = *reinterpret_cast<float4*>(tgt + i * 4);
    const float4 s = ldg4(src + i * 4);
    t.x = __fadd_rn(__fmul_rn(tau, s.x), __fmul_rn(one_minus_tau, t.x));
    t.y = __fadd_rn(__fmul_rn(tau, s.y), __fmul_rn(one_minus_tau, t.y));
    t.z = __fadd_rn(__fmul_rn(tau, s.z), __fmul_rn(one_minus_tau, t.z));
    t.w = __fadd_rn(__fmul_rn(tau, s.w), __fmul_rn(one_minus_tau, t.w));
    stg4(tgt + i * 4, t);
    if (hi && i * 4 < n_split) split_store4(t, hi, lo, i);
  }
}

inline int grid_for_flat(long long n) {
  long long b = (n / 4 + 255) / 256;
  if (b > 8LL * NUM_SMS) b = 8LL * NUM_SMS;
  return b < 1 ? 1 : (int)b;
}

}  // namespace sgrl
