// Small fused kernels around the GEMMs: input embedding, residual+LayerNorm, the per-token
// 3x32 . 32x32 matrix apply (K4), the actor head, and backward helpers.
#pragma once
#include "common.cuh"
#include "layout.h"

namespace sgrl {

// =====================================================================================
// Embedding (TransformerModel.forward input stage, SEActor.py:237-251,153):
//   V0[t][r][c] = x[t][3c+r] (c<8), gd = V0[..,1:3], s0 = x[t][24:] (| action for critics)
//   Vg0 = sqrt(128) * V0 Wg^T,   h0 = sqrt(128) * (We s0 + be) + pos(limb)
// One CTA of 128 threads (thread = output channel, weights held in registers) walks
// 8-token groups staged in shared memory.
// =====================================================================================
constexpr int E_TOK = 8;

__global__ void __launch_bounds__(128) embed_fwd_kernel(
    const float* __restrict__ obs, long long zsObs, const float* __restrict__ act, long long zsAct,
    const int* __restrict__ rank3,
    const float* __restrict__ Wg, const float* __restrict__ We, const float* __restrict__ be,
    const float* __restrict__ E0, const float* __restrict__ E1, const float* __restrict__ E2, long long zsP,
    float* __restrict__ V0, float* __restrict__ GD, float* __restrict__ SH, int ldsh,
    float* __restrict__ VG, float* __restrict__ H, int ldh, long long zsS, int T, int ng, int in_nets) {
  SGRL_PDL_ENTER();
  __shared__ float xs[E_TOK][48];
  __shared__ int rk[E_TOK][3];
  const int c = threadIdx.x, z = blockIdx.y;
  obs += (z % in_nets) * zsObs; if (act) act += (z % in_nets) * zsAct;     // nets z, z + in_nets, ... share one input block
  Wg += z * zsP; We += z * zsP; be += z * zsP; E0 += z * zsP; E1 += z * zsP; E2 += z * zsP;
  V0 += z * zsS; GD += z * zsS; SH += z * zsS; VG += z * zsS; H += z * zsS;
  float wg[GN], we[20];
#pragma unroll
  for (int j = 0; j < GN; ++j) wg[j] = Wg[c * GN + j];
#pragma unroll
  for (int k = 0; k < 20; ++k) we[k] = k < ng ? We[c * ng + k] : 0.f;
  const float bc = be[c];
  const float s128 = 11.313708498984761f;  // sqrt(128)
  const int nin = 24 + ng;   // 41 (actor) | 44 (critic: obs | action)
  for (int t0 = blockIdx.x * E_TOK; t0 < T; t0 += gridDim.x * E_TOK) {
    __syncthreads();
    for (int i = c; i < E_TOK * 48; i += 128) {
      const int tk = i / 48, k = i % 48, t = t0 + tk;
      float v = 0.f;                                   // columns >= nin stay zero (we[k>=ng] == 0 too)
      if (t < T && k < nin) v = k < 41 ? obs[(long long)t * 41 + k] : act[(long long)t * 3 + (k - 41)];
      xs[tk][k] = v;
    }
    if (c < E_TOK * 3) { const int t = t0 + c / 3; rk[c / 3][c % 3] = t < T ? rank3[(long long)t * 3 + c % 3] : 0; }
    __syncthreads();
#pragma unroll
    for (int tk = 0; tk < E_TOK; ++tk) {
      const int t = t0 + tk;
      if (t >= T) break;
      const float* x = xs[tk];
      float hv = 0.f;
#pragma unroll
      for (int k = 0; k < 20; ++k) hv = fmaf(we[k], x[24 + k], hv);   // we[k>=ng] == 0 and xs tail is finite
      const float pos = c < 42 ? E0[rk[tk][0] * 42 + c] : c < 84 ? E1[rk[tk][1] * 42 + (c - 42)] : E2[rk[tk][2] * 44 + (c - 84)];
      H[(long long)t * ldh + c] = (hv + bc) * s128 + pos;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        float v = 0.f;
#pragma unroll
        for (int j = 0; j < GN; ++j) v = fmaf(wg[j], x[3 * j + r], v);
        VG[((long long)t * 3 + r) * 128 + c] = v * s128;
      }
      if (c < 24) V0[(long long)t * 24 + c] = x[3 * (c % 8) + c / 8];          // (r=c/8, j=c%8)
      if (c >= 32 && c < 38) { const int i = c - 32; GD[(long long)t * 6 + i] = x[3 * (1 + i % 2) + i / 2]; }
      if (c >= 64 && c < 64 + ng) SH[(long long)t * ldsh + (c - 64)] = x[24 + (c - 64)];
    }
  }
}

// =====================================================================================
// Gradient w.r.t. the observation input, d obs (T,41), gathered at the end of the backward from what the data-gradient
// chain has already produced (oracle/set_oracle.py::transformer_model).  With x = obs[t], V0[r][j] = x[3j+r], s0 = x[24:41]:
//   d V0[r][j] += sqrt(128) * sum_c dVg0[r][c] Wg[c][j]                       g_encoder          (frame 0 dVg)
//   d s0[k]    += sqrt(128) * sum_c dh0[c] We[c][k]                           encoder            (frame 0 dh)
//   d V0[r][j] += sum_{p<30} dZh[r][p] gg_proj[p][j]   (+ dZh2 . g_proj, actor) head invariants (head frame dZ1 | dZ3)
//   d s0[k]    += dSH[k]                                                      linear1_ng([s0 | h]) (head frame dSH)
//   d V0[r][5+i] += dy_i w_r, dy_i = dOut_i max_action (1 - tanh^2)          actor output axes
// and gd = V0[..., 1:3] (obs vectors 1, 2) enters as columns 30, 31 of every Z (each layer's Z1, Z2, Z3 and the head's) and as
// channels 126, 127 of the attention values of both heads:
//   d gd_j[r][k] += sum_Z dZ[r][30+k] + sum_l sum_h sum_{i in graph(j)} P_l[i][h][j] dOG_l[i][r][128h + 126 + k].
// One warp per token: every lane accumulates its share of the 41 outputs (embedding terms: lane = channel c + 32q; Z terms:
// lane = Z column p; attention terms: lane = (query i, head h)), then 41 butterfly sums.  No atomics, no order that depends
// on timing: bit-identical across runs.  The token's graph comes from a binary search over cu_limbs (ragged packed tables).
// =====================================================================================
struct InGradP {
  const float* dvg0; const float* dh0;             // frame 0: dVg (T,3,128), dh (T,128)                     z-stride zsW
  const float* dzh; const float* dzh2;             // head frame: dZ1 (T,3,32); actor: dZ3 (T,3,32), else nullptr
  const float* dsh; int ldsh;                      // head frame: d[s0 | (act) | h] (T,ldsh)
  const float* dz[3 * MAX_LAYERS];                 // layer frames: dZ1, dZ2, dZ3 of layer l at 3l..3l+2 (only columns 30, 31 read)
  const float* dog[MAX_LAYERS];                    // layer frames: d og (T,3,256)
  const float* P[MAX_LAYERS];                      // stash: attention probabilities (T,2,16)                  z-stride zsS
  const float* Wg; const float* We; const float* gg; const float* gph;   // parameters (gph: actor only)  z-stride zsP
  int ng;                                          // columns of encoder.weight (17 actor | 20 critic)
  const float* dout; long long zsDo;               // actor only: dOut (T,3), out (T,3), w (T,3)
  const float* out; const float* w3; float max_action;
  float* dobs; long long zsDobs;
  const int* cu_limbs; int G, T, L;
  long long zsW, zsS, zsP;
};

__global__ void __launch_bounds__(256) input_grad_kernel(InGradP p) {
  SGRL_PDL_ENTER();
  __shared__ float sWg[GN][128];           // sqrt(128) * g_encoder.weight, transposed
  __shared__ float sWe[17][128];           // sqrt(128) * encoder.weight[:, :17], transposed
  __shared__ float sZh[2][GN][32];         // [gg_proj | g_proj][:, :8] transposed; columns 30, 31 route to V0 vectors 1, 2
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, z = blockIdx.y;
  const bool actor = p.dzh2 != nullptr;
  const float s128 = 11.313708498984761f;
  {
    const float* Wg = p.Wg + z * p.zsP; const float* We = p.We + z * p.zsP; const float* gg = p.gg + z * p.zsP;
    const float* gph = actor ? p.gph + z * p.zsP : nullptr;
    for (int i = threadIdx.x; i < GN * 128; i += 256) { const int j = i >> 7, c = i & 127; sWg[j][c] = s128 * __ldg(Wg + c * GN + j); }
    for (int i = threadIdx.x; i < 17 * 128; i += 256) { const int k = i >> 7, c = i & 127; sWe[k][c] = s128 * __ldg(We + c * p.ng + k); }
    for (int i = threadIdx.x; i < 2 * GN * 32; i += 256) {
      const int m = i / (GN * 32), j = (i >> 5) % GN, q = i & 31;
      const float* W = m ? gph : gg;
      sZh[m][j][q] = q < NPJ ? (W ? __ldg(W + q * (D + GN) + j) : 0.f) : (q - NPJ + 1 == j ? 1.f : 0.f);
    }
  }
  __syncthreads();
  const float e1 = lane == 30 ? 1.f : 0.f, e2 = lane == 31 ? 1.f : 0.f;
  const long long zW = z * p.zsW, zS = z * p.zsS;
  for (int t = blockIdx.x * 8 + warp; t < p.T; t += gridDim.x * 8) {
    float pv[3][GN], ps[17];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int j = 0; j < GN; ++j) pv[r][j] = 0.f;
#pragma unroll
    for (int k = 0; k < 17; ++k) ps[k] = 0.f;
    // ---- embedding: Vg0 = sqrt(128) V0 Wg^T, h0 = sqrt(128) (We s0 + be) + pos
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int c = lane + 32 * q;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float d = __ldg(p.dvg0 + zW + ((long long)t * 3 + r) * 128 + c);
#pragma unroll
        for (int j = 0; j < GN; ++j) pv[r][j] = fmaf(d, sWg[j][c], pv[r][j]);
      }
      const float dh = __ldg(p.dh0 + zW + (long long)t * 128 + c);
#pragma unroll
      for (int k = 0; k < 17; ++k) ps[k] = fmaf(dh, sWe[k][c], ps[k]);
    }
    // ---- head invariants: Zh = [[V0 | Vg] gg_proj^T | gd] (actor: also Zh2 with g_proj), lane = column of Z
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      const float* dz = m ? p.dzh2 : p.dzh;
      if (!dz) continue;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float d = __ldg(dz + zW + ((long long)t * 3 + r) * 32 + lane);
#pragma unroll
        for (int j = 0; j < GN; ++j) pv[r][j] = fmaf(d, sZh[m][j][lane], pv[r][j]);
      }
    }
    // ---- gd columns 30, 31 of every encoder layer's Z1, Z2, Z3
    for (int s = 0; s < 3 * p.L; ++s) {
      if (lane < NPJ) continue;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float d = __ldg(p.dz[s] + zW + ((long long)t * 3 + r) * 32 + lane);
        pv[r][1] = fmaf(d, e1, pv[r][1]);
        pv[r][2] = fmaf(d, e2, pv[r][2]);
      }
    }
    // ---- attention values: gd rides in channels 126, 127 of every (r, head); lane = (query i, head h) of the token's graph
    {
      int lo = 0, hi = p.G;                   // cu_limbs[lo] <= t < cu_limbs[hi]
      while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (__ldg(p.cu_limbs + mid) <= t) lo = mid; else hi = mid; }
      const int t0 = __ldg(p.cu_limbs + lo), n = __ldg(p.cu_limbs + lo + 1) - t0;
      const int i = lane >> 1, h = lane & 1;
      if (i < n) {
        const long long ti = t0 + i;
        for (int l = 0; l < p.L; ++l) {
          const float pr = __ldg(p.P[l] + zS + ti * 32 + h * 16 + (t - t0));
          const float* dog = p.dog[l] + zW + ti * 768 + h * 128 + 126;
#pragma unroll
          for (int r = 0; r < 3; ++r) {
            const float2 v = __ldg(reinterpret_cast<const float2*>(dog + r * 256));
            pv[r][1] = fmaf(pr, v.x, pv[r][1]);
            pv[r][2] = fmaf(pr, v.y, pv[r][2]);
          }
        }
      }
    }
    // ---- reduce over the warp; lane o (and 32 + o) owns obs column o
    float v0 = 0.f, v1 = 0.f;
#pragma unroll
    for (int j = 0; j < GN; ++j)
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float s = warp_sum(pv[r][j]);
        if (lane == 3 * j + r) v0 = s;
      }
#pragma unroll
    for (int k = 0; k < 17; ++k) {
      const float s = warp_sum(ps[k]);
      if (24 + k < 32) { if (lane == 24 + k) v0 = s; }
      else if (lane == 24 + k - 32) v1 = s;
    }
    // head scalar branch [s0 | h] -> linear1_ng: columns 0..16 of dSH
    if (lane >= 24) v0 += __ldg(p.dsh + zW + (long long)t * p.ldsh + (lane - 24));
    if (lane < 9) v1 += __ldg(p.dsh + zW + (long long)t * p.ldsh + (lane + 8));
    // actor output: out_i = max_action tanh(sum_r V0[r][5+i] w_r)  ->  d V0[r][5+i] += dy_i w_r  (obs columns 15..23)
    if (actor && lane >= 15 && lane < 24) {
      const int i = lane / 3 - 5, r = lane % 3;
      const float a = __ldg(p.out + zS + (long long)t * 3 + i) / p.max_action;
      const float dy = __ldg(p.dout + z * p.zsDo + (long long)t * 3 + i) * p.max_action * (1.f - a * a);
      v0 = fmaf(dy, __ldg(p.w3 + zS + (long long)t * 3 + r), v0);
    }
    float* o = p.dobs + z * p.zsDobs + (long long)t * 41;
    o[lane] = v0;
    if (lane < 9) o[32 + lane] = v1;
  }
}

// scatter-add of dh0 into the three positional tables
__global__ void __launch_bounds__(128) pos_embed_bwd_kernel(
    const float* __restrict__ dH, int ldh, long long zsW, const int* __restrict__ rank3,
    float* __restrict__ dE0, float* __restrict__ dE1, float* __restrict__ dE2, long long zsG, int T) {
  SGRL_PDL_ENTER();
  __shared__ float acc[MAX_NODE][128];
  const int c = threadIdx.x, z = blockIdx.y;
  dH += z * zsW; dE0 += z * zsG; dE1 += z * zsG; dE2 += z * zsG;
  for (int r = 0; r < MAX_NODE; ++r) acc[r][c] = 0.f;
  const int which = c < 42 ? 0 : c < 84 ? 1 : 2;
  const int per = (T + gridDim.x - 1) / gridDim.x;
  const int t1 = min(T, (int)(blockIdx.x + 1) * per);
  for (int t = blockIdx.x * per; t < t1; ++t) {
    const int rk = rank3[(long long)t * 3 + which];
    acc[rk][c] += dH[(long long)t * ldh + c];   // column c is private to thread c: no race
  }
  for (int r = 0; r < MAX_NODE; ++r) {
    const float v = acc[r][c];
    if (v != 0.f) {
      if (which == 0) atomicAdd(dE0 + r * 42 + c, v);
      else if (which == 1) atomicAdd(dE1 + r * 42 + (c - 42), v);
      else atomicAdd(dE2 + r * 44 + (c - 84), v);
    }
  }
}

// =====================================================================================
// Residual + LayerNorm over 128 features, one warp per token (eps 1e-5, SEActor.py:90-91,
// 122-123,164-165).   x = a + b;  y = (x-mean)*rstd*gamma + beta
// =====================================================================================
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(
    const float* __restrict__ a, int lda, const float* __restrict__ b, int ldb,
    const float* __restrict__ gamma, const float* __restrict__ beta, long long zsP,
    float* __restrict__ x, float* __restrict__ y, int ldy, float* __restrict__ y2, int ldy2,
    float* __restrict__ stats, long long zsS, int T, int vflags) {
  SGRL_PDL_ENTER();
  const int lane = threadIdx.x & 31, z = blockIdx.y;
  a += z * zsS; if (b) b += z * zsS; if (x) x += z * zsS; y += z * zsS; if (y2) y2 += z * zsS; stats += z * zsS;
  gamma += z * zsP; beta += z * zsP;
  const float4 g = ldg4(gamma + lane * 4), be = ldg4(beta + lane * 4);
  const bool va = vflags & 1, vb = vflags & 2, vy = vflags & 4, vy2 = vflags & 8;
  for (int t = blockIdx.x * 8 + (threadIdx.x >> 5); t < T; t += gridDim.x * 8) {
    float4 v = load4(a + (long long)t * lda + lane * 4, va);
    if (b) {
      const float4 w = load4(b + (long long)t * ldb + lane * 4, vb);
      v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
    }
    if (x) stg4(x + (long long)t * 128 + lane * 4, v);
    const float mean = warp_sum(v.x + v.y + v.z + v.w) * (1.f / 128.f);
    const float d0 = v.x - mean, d1 = v.y - mean, d2 = v.z - mean, d3 = v.w - mean;
    const float var = warp_sum(d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3) * (1.f / 128.f);
    const float rstd = rsqrtf(var + 1e-5f);
    const float4 o = make_float4(d0 * rstd * g.x + be.x, d1 * rstd * g.y + be.y, d2 * rstd * g.z + be.z, d3 * rstd * g.w + be.w);
    store4(y + (long long)t * ldy + lane * 4, o, vy);
    if (y2) store4(y2 + (long long)t * ldy2 + lane * 4, o, vy2);
    if (lane == 0) { stats[(long long)t * 2] = mean; stats[(long long)t * 2 + 1] = rstd; }
  }
}

//   dy = dy1 + dy2;  dx = rstd * (g*dy - mean(g*dy) - xhat * mean(g*dy*xhat));  dgamma += dy*xhat; dbeta += dy
// Optional tail (LayerNorm-2 of an encoder layer, whose input branch is f = linear2(..)/F2): the backward of that row division on
// the same rows, dff = dx / F (-> rd.out), dF[t] -= sum_n dx*f / F — what rowdiv_bwd_kernel did in a launch of its own.
struct LnRowdiv { const float* y; const float* Fn; float* dF; float* out; int ldy, ldout; };    // y, Fn: stash (zsS); dF, out: workspace (zsW)
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(
    const float* __restrict__ dy1, int ld1, const float* __restrict__ dy2, int ld2,
    const float* __restrict__ x, int ldx, const float* __restrict__ stats, long long zsS,
    const float* __restrict__ gamma, long long zsP,
    float* __restrict__ dx, int lddx, long long zsW, float* __restrict__ dgamma, float* __restrict__ dbeta, long long zsG, int T, int vflags,
    LnRowdiv rd) {
  SGRL_PDL_ENTER();
  __shared__ float red[2][8][128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, z = blockIdx.y;
  dy1 += z * zsW; if (dy2) dy2 += z * zsW; dx += z * zsW;
  x += z * zsS; stats += z * zsS; gamma += z * zsP;
  if (rd.y) { rd.y += z * zsS; rd.Fn += z * zsS; rd.dF += z * zsW; rd.out += z * zsW; }
  if (dgamma) { dgamma += z * zsG; dbeta += z * zsG; }
  const float4 g = ldg4(gamma + lane * 4);
  float ag[4] = {0, 0, 0, 0}, ab[4] = {0, 0, 0, 0};
  const bool v1 = vflags & 1, v2 = vflags & 2, vx = vflags & 4, vo = vflags & 8;
  for (int t = blockIdx.x * 8 + warp; t < T; t += gridDim.x * 8) {
    float4 d = load4(dy1 + (long long)t * ld1 + lane * 4, v1);
    if (dy2) {
      const float4 e = load4(dy2 + (long long)t * ld2 + lane * 4, v2);
      d.x += e.x; d.y += e.y; d.z += e.z; d.w += e.w;
    }
    const float4 xv = load4(x + (long long)t * ldx + lane * 4, vx);
    const float mean = stats[(long long)t * 2], rstd = stats[(long long)t * 2 + 1];
    const float xh[4] = {(xv.x - mean) * rstd, (xv.y - mean) * rstd, (xv.z - mean) * rstd, (xv.w - mean) * rstd};
    const float dv[4] = {d.x, d.y, d.z, d.w}, gv[4] = {g.x, g.y, g.z, g.w};
    float s1 = 0.f, s2 = 0.f, gd[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { gd[i] = gv[i] * dv[i]; s1 += gd[i]; s2 += gd[i] * xh[i]; ag[i] += dv[i] * xh[i]; ab[i] += dv[i]; }
    s1 = warp_sum(s1) * (1.f / 128.f); s2 = warp_sum(s2) * (1.f / 128.f);
    float4 o;
    o.x = rstd * (gd[0] - s1 - xh[0] * s2); o.y = rstd * (gd[1] - s1 - xh[1] * s2);
    o.z = rstd * (gd[2] - s1 - xh[2] * s2); o.w = rstd * (gd[3] - s1 - xh[3] * s2);
    store4(dx + (long long)t * lddx + lane * 4, o, vo);
    if (rd.y) {
      const float invF = 1.f / rd.Fn[t];
      const float4 yv = load4(rd.y + (long long)t * rd.ldy + lane * 4, vflags & 16);
      const float s = warp_sum(o.x * yv.x + o.y * yv.y + o.z * yv.z + o.w * yv.w);
      store4(rd.out + (long long)t * rd.ldout + lane * 4, make_float4(o.x * invF, o.y * invF, o.z * invF, o.w * invF), vflags & 32);
      if (lane == 0) atomicAdd(rd.dF + t, -s * invF);     // the other divisions by the same F add their term from a concurrent lane
    }
  }
  if (!dgamma) return;   // data-only backward
#pragma unroll
  for (int i = 0; i < 4; ++i) { red[0][warp][lane * 4 + i] = ag[i]; red[1][warp][lane * 4 + i] = ab[i]; }
  __syncthreads();
  const int c = threadIdx.x & 127, which = threadIdx.x >> 7;
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) s += red[which][w][c];
  atomicAdd((which ? dbeta : dgamma) + c, s);
}

// =====================================================================================
// K4 — per-token matrix apply  R_t = Z_t (3x32) . M_t (32x32)   (SEActor.py:107-112, 271-276)
// one warp per token, lane = output column; M rows stream as coalesced 128 B loads.
// =====================================================================================
__global__ void __launch_bounds__(256) matapply_fwd_kernel(
    const float* __restrict__ Z, const float* __restrict__ M, float* __restrict__ R, long long zsS, int T) {
  SGRL_PDL_ENTER();
  const int lane = threadIdx.x & 31, z = blockIdx.y;
  Z += z * zsS; M += z * zsS; R += z * zsS;
  for (int t = blockIdx.x * 8 + (threadIdx.x >> 5); t < T; t += gridDim.x * 8) {
    const float z0 = Z[(long long)t * 96 + lane], z1 = Z[(long long)t * 96 + 32 + lane], z2 = Z[(long long)t * 96 + 64 + lane];
    const float* m = M + (long long)t * 1024 + lane;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      const float mv = __ldg(m + i * 32);
      a0 = fmaf(__shfl_sync(0xffffffffu, z0, i), mv, a0);
      a1 = fmaf(__shfl_sync(0xffffffffu, z1, i), mv, a1);
      a2 = fmaf(__shfl_sync(0xffffffffu, z2, i), mv, a2);
    }
    float* r = R + (long long)t * 96;
    r[lane] = a0; r[32 + lane] = a1; r[64 + lane] = a2;
  }
}

// backward:  dZ = dR M^T;  dM = Z^T dR;  M = Tm/F  =>  dTm = dM/F (written to dT),  dF -= sum(dM.M)/F
__global__ void __launch_bounds__(256) matapply_bwd_kernel(
    const float* __restrict__ dR, const float* __restrict__ Z, const float* __restrict__ M, const float* __restrict__ Fn,
    long long zsS, float* __restrict__ dZ, float* __restrict__ dT, float* __restrict__ dF, long long zsW, int T) {
  SGRL_PDL_ENTER();
  __shared__ float Ms[8][32][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, z = blockIdx.y;
  Z += z * zsS; M += z * zsS; Fn += z * zsS; dR += z * zsW; dZ += z * zsW; dT += z * zsW; dF += z * zsW;
  for (int t = blockIdx.x * 8 + warp; t < T; t += gridDim.x * 8) {
    const float z0 = Z[(long long)t * 96 + lane], z1 = Z[(long long)t * 96 + 32 + lane], z2 = Z[(long long)t * 96 + 64 + lane];
    const float r0 = dR[(long long)t * 96 + lane], r1 = dR[(long long)t * 96 + 32 + lane], r2 = dR[(long long)t * 96 + 64 + lane];
    const float invF = 1.f / Fn[t];
    const float* m = M + (long long)t * 1024 + lane;
    float* dt = dT + (long long)t * 1024 + lane;
    float facc = 0.f;
    __syncwarp();
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      const float mv = __ldg(m + i * 32);
      Ms[warp][i][lane] = mv;
      const float dm = __shfl_sync(0xffffffffu, z0, i) * r0 + __shfl_sync(0xffffffffu, z1, i) * r1 + __shfl_sync(0xffffffffu, z2, i) * r2;
      dt[i * 32] = dm * invF;
      facc = fmaf(dm, mv, facc);
    }
    facc = warp_sum(facc);
    __syncwarp();
    // lane = i now: dZ[r][i] = sum_j dR[r][j] * M[i][j]
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 8
    for (int j = 0; j < 32; ++j) {
      const float mv = Ms[warp][lane][j];
      a0 = fmaf(__shfl_sync(0xffffffffu, r0, j), mv, a0);
      a1 = fmaf(__shfl_sync(0xffffffffu, r1, j), mv, a1);
      a2 = fmaf(__shfl_sync(0xffffffffu, r2, j), mv, a2);
    }
    float* o = dZ + (long long)t * 96;
    o[lane] = a0; o[32 + lane] = a1; o[64 + lane] = a2;
    if (lane == 0) atomicAdd(dF + t, -facc * invF);     // the other divisions by the same F add their term from a concurrent lane (net.cuh)
  }
}

// =====================================================================================
// K4 fused with linear5 and the two residuals (SEActor.py:107-114):
//   R_t = Z3_t (3x32) . M_t (32x32);   Vg'_t = Vg_t + dV_t + R_t W5^T      (W5 = linear5.weight (128,32), no bias)
// One warp per token.  Phase 1 as matapply_fwd_kernel (lane = column j of R); phase 2: lane owns the four output
// channels c = lane + 32 q, R's columns are broadcast with shuffles and W5 is read transposed from shared memory
// (W5t[j][c]: conflict-free).  12 K MACs per token: far below one tcgen05 tile, and it removes the K = 32 GEMM launch
// (8 us at 2 304 tokens) that used to follow the matrix apply on the critical path of every layer.
// R is written only when the caller keeps activations for a backward (dW5 = dVg'^T R).
// =====================================================================================
__global__ void __launch_bounds__(256) matapply_l5_fwd_kernel(
    const float* __restrict__ Z, const float* __restrict__ M, const float* __restrict__ W5, long long zsP,
    const float* __restrict__ Vg, const float* __restrict__ dV, float* __restrict__ R, float* __restrict__ Vn, long long zsS, int T) {
  SGRL_PDL_ENTER();
  __shared__ float W5t[32 * 128];
  const int lane = threadIdx.x & 31, z = blockIdx.y;
  Z += z * zsS; M += z * zsS; Vg += z * zsS; dV += z * zsS; Vn += z * zsS; W5 += z * zsP;
  if (R) R += z * zsS;
  // W5t[j][c] = W5[c][j]: consecutive threads take consecutive c (conflict-free writes; the strided reads are independent and L2-resident)
  for (int i = threadIdx.x; i < 32 * 128; i += 256) W5t[i] = __ldg(W5 + (i & 127) * 32 + (i >> 7));
  __syncthreads();
  for (int t = blockIdx.x * 8 + (threadIdx.x >> 5); t < T; t += gridDim.x * 8) {
    const float z0 = Z[(long long)t * 96 + lane], z1 = Z[(long long)t * 96 + 32 + lane], z2 = Z[(long long)t * 96 + 64 + lane];
    const float* m = M + (long long)t * 1024 + lane;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      const float mv = __ldg(m + i * 32);
      a0 = fmaf(__shfl_sync(0xffffffffu, z0, i), mv, a0);
      a1 = fmaf(__shfl_sync(0xffffffffu, z1, i), mv, a1);
      a2 = fmaf(__shfl_sync(0xffffffffu, z2, i), mv, a2);
    }
    if (R) { float* r = R + (long long)t * 96; r[lane] = a0; r[32 + lane] = a1; r[64 + lane] = a2; }
    float o[3][4];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const long long at = ((long long)t * 3 + r) * 128 + lane + 32 * q;
        o[r][q] = Vg[at] + dV[at];
      }
    float s[3][4];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int q = 0; q < 4; ++q) s[r][q] = 0.f;
#pragma unroll 8
    for (int j = 0; j < 32; ++j) {
      const float r0 = __shfl_sync(0xffffffffu, a0, j), r1 = __shfl_sync(0xffffffffu, a1, j), r2 = __shfl_sync(0xffffffffu, a2, j);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float w = W5t[j * 128 + lane + 32 * q];
        s[0][q] = fmaf(r0, w, s[0][q]); s[1][q] = fmaf(r1, w, s[1][q]); s[2][q] = fmaf(r2, w, s[2][q]);
      }
    }
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int q = 0; q < 4; ++q) Vn[((long long)t * 3 + r) * 128 + lane + 32 * q] = o[r][q] + s[r][q];
  }
}

// backward of the fused pair:  dR = dVg' W5  (3x128 . 128x32), then matapply_bwd_kernel's math:
//   dZ3 = dR M^T;  dM = Z3^T dR;  M = Tm/F  =>  dTm = dM/F,  dF -= sum(dM.M)/F.   dR is also written (dW5's operand is dVg', R).
__global__ void __launch_bounds__(256) matapply_l5_bwd_kernel(
    const float* __restrict__ dVn, const float* __restrict__ W5, long long zsP, const float* __restrict__ Z, const float* __restrict__ M,
    const float* __restrict__ Fn, long long zsS, float* __restrict__ dZ, float* __restrict__ dT, float* __restrict__ dF, long long zsW, int T) {
  SGRL_PDL_ENTER();
  __shared__ float Ms[8][32][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, z = blockIdx.y;
  Z += z * zsS; M += z * zsS; Fn += z * zsS; dVn += z * zsW; dZ += z * zsW; dT += z * zsW; dF += z * zsW; W5 += z * zsP;
  for (int t = blockIdx.x * 8 + warp; t < T; t += gridDim.x * 8) {
    // dR[r][lane] = sum_c dVg'[r][c] W5[c][lane]; lane holds dVg'[r][4*lane .. 4*lane+3]
    float r0 = 0.f, r1 = 0.f, r2 = 0.f;
    {
      const float4 d0 = *reinterpret_cast<const float4*>(dVn + ((long long)t * 3 + 0) * 128 + lane * 4);
      const float4 d1 = *reinterpret_cast<const float4*>(dVn + ((long long)t * 3 + 1) * 128 + lane * 4);
      const float4 d2 = *reinterpret_cast<const float4*>(dVn + ((long long)t * 3 + 2) * 128 + lane * 4);
#pragma unroll 4
      for (int cl = 0; cl < 32; ++cl) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float w = __ldg(W5 + (cl * 4 + e) * 32 + lane);      // natural layout W5[c][j], lane = j: one coalesced 128 B line, L1-resident (16 KB)
          const float v0 = e == 0 ? d0.x : e == 1 ? d0.y : e == 2 ? d0.z : d0.w;
          const float v1 = e == 0 ? d1.x : e == 1 ? d1.y : e == 2 ? d1.z : d1.w;
          const float v2 = e == 0 ? d2.x : e == 1 ? d2.y : e == 2 ? d2.z : d2.w;
          r0 = fmaf(__shfl_sync(0xffffffffu, v0, cl), w, r0);
          r1 = fmaf(__shfl_sync(0xffffffffu, v1, cl), w, r1);
          r2 = fmaf(__shfl_sync(0xffffffffu, v2, cl), w, r2);
        }
      }
    }
    const float z0 = Z[(long long)t * 96 + lane], z1 = Z[(long long)t * 96 + 32 + lane], z2 = Z[(long long)t * 96 + 64 + lane];
    const float invF = 1.f / Fn[t];
    const float* m = M + (long long)t * 1024 + lane;
    float* dt = dT + (long long)t * 1024 + lane;
    float facc = 0.f;
    __syncwarp();
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      const float mv = __ldg(m + i * 32);
      Ms[warp][i][lane] = mv;
      const float dm = __shfl_sync(0xffffffffu, z0, i) * r0 + __shfl_sync(0xffffffffu, z1, i) * r1 + __shfl_sync(0xffffffffu, z2, i) * r2;
      dt[i * 32] = dm * invF;
      facc = fmaf(dm, mv, facc);
    }
    facc = warp_sum(facc);
    __syncwarp();
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 8
    for (int j = 0; j < 32; ++j) {
      const float mv = Ms[warp][lane][j];
      a0 = fmaf(__shfl_sync(0xffffffffu, r0, j), mv, a0);
      a1 = fmaf(__shfl_sync(0xffffffffu, r1, j), mv, a1);
      a2 = fmaf(__shfl_sync(0xffffffffu, r2, j), mv, a2);
    }
    float* o = dZ + (long long)t * 96;
    o[lane] = a0; o[32 + lane] = a1; o[64 + lane] = a2;
    if (lane == 0) atomicAdd(dF + t, -facc * invF);     // the other divisions by the same F add their term from a concurrent lane (net.cuh)
  }
}

// =====================================================================================
// Actor head tail (SEActor.py:275-285, :341):  w_r = sum_c R[r][c] wd[c];
//   a_i = max_action * tanh( sum_r V0[r][5+i] w_r )
// =====================================================================================
__global__ void __launch_bounds__(256) actor_out_fwd_kernel(
    const float* __restrict__ R, const float* __restrict__ V0, const float* __restrict__ wd, long long zsP,
    float* __restrict__ W3, float* __restrict__ out, long long zsS, float max_action, int T) {
  SGRL_PDL_ENTER();
  const int lane = threadIdx.x & 31, z = blockIdx.y;
  R += z * zsS; V0 += z * zsS; W3 += z * zsS; out += z * zsS; wd += z * zsP;
  const float w = wd[lane];
  for (int t = blockIdx.x * 8 + (threadIdx.x >> 5); t < T; t += gridDim.x * 8) {
    const float* r = R + (long long)t * 96;
    const float w0 = warp_sum(r[lane] * w), w1 = warp_sum(r[32 + lane] * w), w2 = warp_sum(r[64 + lane] * w);
    if (lane < 3) {
      const float* v = V0 + (long long)t * 24;           // V0[r][c] at r*8+c
      const float p = v[0 * 8 + 5 + lane] * w0 + v[1 * 8 + 5 + lane] * w1 + v[2 * 8 + 5 + lane] * w2;
      out[(long long)t * 3 + lane] = max_action * tanhf(p);
      W3[(long long)t * 3 + lane] = lane == 0 ? w0 : lane == 1 ? w1 : w2;
    }
  }
}

__global__ void __launch_bounds__(256) actor_out_bwd_kernel(
    const float* __restrict__ dOut, long long zsDo, const float* __restrict__ out, const float* __restrict__ R, const float* __restrict__ V0,
    long long zsS, const float* __restrict__ wd, long long zsP, float* __restrict__ dR, long long zsW,
    float* __restrict__ dwd, long long zsG, float max_action, int T) {
  SGRL_PDL_ENTER();
  __shared__ float red[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, z = blockIdx.y;
  dOut += z * zsDo; out += z * zsS; R += z * zsS; V0 += z * zsS; wd += z * zsP; dR += z * zsW; dwd += z * zsG;
  const float w = wd[lane];
  float acc = 0.f;
  for (int t = blockIdx.x * 8 + warp; t < T; t += gridDim.x * 8) {
    const float* v = V0 + (long long)t * 24;
    float dp[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const float a = out[(long long)t * 3 + i] / max_action;       // tanh(p)
      dp[i] = dOut[(long long)t * 3 + i] * max_action * (1.f - a * a);
    }
    float* o = dR + (long long)t * 96;
    const float* r = R + (long long)t * 96;
#pragma unroll
    for (int rr = 0; rr < 3; ++rr) {
      const float dw = dp[0] * v[rr * 8 + 5] + dp[1] * v[rr * 8 + 6] + dp[2] * v[rr * 8 + 7];
      o[rr * 32 + lane] = dw * w;
      acc = fmaf(dw, r[rr * 32 + lane], acc);
    }
  }
  red[warp][lane] = acc;
  __syncthreads();
  if (warp == 0) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += red[k][lane];
    atomicAdd(dwd + lane, s);
  }
}

// =====================================================================================
// Backward helpers
// =====================================================================================
// y = t/F (* colscale on the first cs_n columns):  dt = dy * cs / F,  dF[t] -= sum_n dy*y / F.  dt is written to `dy`; the incoming
// gradient is read from `src` (row stride ldsrc, z-stride zsSrc) when given — no separate copy kernel in front — else from `dy` (in place)
__global__ void __launch_bounds__(256) rowdiv_bwd_kernel(
    float* dy, int lddy, long long zsW, const float* __restrict__ y, int ldy, const float* __restrict__ Fn, long long zsS,
    float* __restrict__ dF, int N, float colscale, int cs_n, int T, const float* src, int ldsrc, long long zsSrc) {
  SGRL_PDL_ENTER();
  const int lane = threadIdx.x & 31, z = blockIdx.y;
  dy += z * zsW; dF += z * zsW; y += z * zsS; Fn += z * zsS;
  if (src) src += z * zsSrc; else { src = dy; ldsrc = lddy; }
  for (int t = blockIdx.x * 8 + (threadIdx.x >> 5); t < T; t += gridDim.x * 8) {
    const float invF = 1.f / Fn[t];
    float s = 0.f;
    for (int n = lane; n < N; n += 32) {
      const float d = src[(long long)t * ldsrc + n];
      s = fmaf(d, y[(long long)t * ldy + n], s);
      dy[(long long)t * lddy + n] = d * invF * (n < cs_n ? colscale : 1.f);
    }
    s = warp_sum(s);
    if (lane == 0) atomicAdd(dF + t, -s * invF);
  }
}

// out[n] += alpha * sum_m X[m][n]
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ X, int ldx, long long zsX,
                                                     float* __restrict__ out, long long zsO, int M, int N, float alpha) {
  SGRL_PDL_ENTER();
  __shared__ float red[8][32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5, z = blockIdx.z;
  X += z * zsX; out += z * zsO;
  const int n = blockIdx.x * 32 + tx;
  float s = 0.f;
  if (n < N)
    for (int m = blockIdx.y * 8 + ty; m < M; m += gridDim.y * 8) s += X[(long long)m * ldx + n];
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && n < N) {
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) v += red[k][tx];
    atomicAdd(out + n, alpha * v);
  }
}

// strided copy / add of a (T x N) block:  dst = (add ? dst : 0) + src (+ src2)
__global__ void __launch_bounds__(256) block_copy_kernel(float* __restrict__ dst, int ldd, long long zsD,
                                                         const float* __restrict__ src, int lds, long long zsSrc,
                                                         const float* __restrict__ src2, int lds2, long long zsSrc2, int M, int N, int add) {
  SGRL_PDL_ENTER();
  const int z = blockIdx.y;
  dst += z * zsD; src += z * zsSrc;
  if (src2) src2 += z * zsSrc2;
  const long long total = (long long)M * N;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += gridDim.x * 256LL) {
    const int m = (int)(i / N), n = (int)(i % N);
    float v = src[(long long)m * lds + n];
    if (src2) v += src2[(long long)m * lds2 + n];
    float* d = dst + (long long)m * ldd + n;
    *d = add ? *d + v : v;
  }
}

inline int grid_for_warps(int T) { int g = ceil_div(T, 8); return g > 8 * NUM_SMS ? 8 * NUM_SMS : (g < 1 ? 1 : g); }

// =====================================================================================
// Host launchers: the grid of each kernel above (its caps, the deterministic-mode override) and the vector flags of the
// LayerNorms, in one place for the network passes (net.cuh) and the single-kernel entry points (sgrl_b200.cu).  Arguments
// are the kernel's own; nb net instances on the grid's y (z for colsum); grid (nullable) receives the grid launched.
// =====================================================================================

inline int embed_fwd_launch(const float* obs, long long zsObs, const float* act, long long zsAct, const int* rank3, const float* Wg,
                            const float* We, const float* be, const float* E0, const float* E1, const float* E2, long long zsP, float* V0,
                            float* GD, float* SH, int ldsh, float* VG, float* H, int ldh, long long zsS, int T, int ng, int nb, int in_nets,
                            cudaStream_t st, int* grid = nullptr) {
  int gx = ceil_div(T, E_TOK); if (gx > 4 * NUM_SMS) gx = 4 * NUM_SMS; if (gx < 1) gx = 1;     // above 4 736 tokens CTAs walk groups
  const dim3 g(gx, nb);
  launch_k(embed_fwd_kernel, g, 128, 0, st, obs, zsObs, act, zsAct, rank3, Wg, We, be, E0, E1, E2, zsP, V0, GD, SH, ldsh, VG, H, ldh, zsS, T, ng,
           in_nets);
  return launched(g, grid);
}

inline int input_grad_launch(const InGradP& p, int nb, cudaStream_t st, int* grid = nullptr) {
  int gx = grid_for_warps(p.T); if (gx > 2 * NUM_SMS) gx = 2 * NUM_SMS;
  const dim3 g(gx, nb);
  launch_k(input_grad_kernel, g, 256, 0, st, p);
  return launched(g, grid);
}

inline int pos_embed_bwd_launch(const float* dH, int ldh, long long zsW, const int* rank3, float* dE0, float* dE1, float* dE2, long long zsG,
                                int T, int nb, cudaStream_t st, int* grid = nullptr) {
  int gx = ceil_div(T, 64); if (gx > NUM_SMS) gx = NUM_SMS; if (gx < 1) gx = 1;
  if (det_enabled()) gx = 1;
  const dim3 g(gx, nb);
  launch_k(pos_embed_bwd_kernel, g, 128, 0, st, dH, ldh, zsW, rank3, dE0, dE1, dE2, zsG, T);
  return launched(g, grid);
}

inline int layernorm_fwd_launch(const float* a, int lda, const float* b, int ldb, const float* gamma, const float* beta, long long zsP, float* x,
                                float* y, int ldy, float* y2, int ldy2, float* stats, long long zsS, int T, int nb, cudaStream_t st,
                                int* grid = nullptr) {
  const int vf = host_vec_ok(a, lda, zsS) | (host_vec_ok(b, ldb, zsS) << 1) | (host_vec_ok(y, ldy, zsS) << 2) | (host_vec_ok(y2, ldy2, zsS) << 3);
  const dim3 g(grid_for_warps(T), nb);
  launch_k(layernorm_fwd_kernel, g, 256, 0, st, a, lda, b, ldb, gamma, beta, zsP, x, y, ldy, y2, ldy2, stats, zsS, T, vf);
  return launched(g, grid);
}

// dgamma == nullptr: data-only backward (dbeta ignored)
inline int layernorm_bwd_launch(const float* dy1, int ld1, const float* dy2, int ld2, const float* x, int ldx, const float* stats, long long zsS,
                                const float* gamma, long long zsP, float* dx, int lddx, long long zsW, float* dgamma, float* dbeta, long long zsG,
                                LnRowdiv rd, int T, int nb, cudaStream_t st, int* grid = nullptr) {
  int gx = grid_for_warps(T); if (gx > 2 * NUM_SMS) gx = 2 * NUM_SMS;
  if (dgamma && det_enabled()) gx = 1;      // dgamma / dbeta: one add per address
  const int vf = host_vec_ok(dy1, ld1, zsW) | (host_vec_ok(dy2, ld2, zsW) << 1) | (host_vec_ok(x, ldx, zsS) << 2) | (host_vec_ok(dx, lddx, zsW) << 3) |
                 ((rd.y && host_vec_ok(rd.y, rd.ldy, zsS)) << 4) | ((rd.out && host_vec_ok(rd.out, rd.ldout, zsW)) << 5);
  const dim3 g(gx, nb);
  launch_k(layernorm_bwd_kernel, g, 256, 0, st, dy1, ld1, dy2, ld2, x, ldx, stats, zsS, gamma, zsP, dx, lddx, zsW, dgamma, dbeta, zsG, T,
           vf, rd);
  return launched(g, grid);
}

inline int matapply_fwd_launch(const float* Z, const float* M, float* R, long long zsS, int T, int nb, cudaStream_t st, int* grid = nullptr) {
  const dim3 g(grid_for_warps(T), nb);
  launch_k(matapply_fwd_kernel, g, 256, 0, st, Z, M, R, zsS, T);
  return launched(g, grid);
}

inline int matapply_bwd_launch(const float* dR, const float* Z, const float* M, const float* Fn, long long zsS, float* dZ, float* dT, float* dF,
                               long long zsW, int T, int nb, cudaStream_t st, int* grid = nullptr) {
  const dim3 g(grid_for_warps(T), nb);
  launch_k(matapply_bwd_kernel, g, 256, 0, st, dR, Z, M, Fn, zsS, dZ, dT, dF, zsW, T);
  return launched(g, grid);
}

inline int matapply_l5_fwd_launch(const float* Z, const float* M, const float* W5, long long zsP, const float* Vg, const float* dV, float* R,
                                  float* Vn, long long zsS, int T, int nb, cudaStream_t st, int* grid = nullptr) {
  const dim3 g(grid_for_warps(T), nb);
  launch_k(matapply_l5_fwd_kernel, g, 256, 0, st, Z, M, W5, zsP, Vg, dV, R, Vn, zsS, T);
  return launched(g, grid);
}

inline int matapply_l5_bwd_launch(const float* dVn, const float* W5, long long zsP, const float* Z, const float* M, const float* Fn, long long zsS,
                                  float* dZ, float* dT, float* dF, long long zsW, int T, int nb, cudaStream_t st, int* grid = nullptr) {
  const dim3 g(grid_for_warps(T), nb);
  launch_k(matapply_l5_bwd_kernel, g, 256, 0, st, dVn, W5, zsP, Z, M, Fn, zsS, dZ, dT, dF, zsW, T);
  return launched(g, grid);
}

inline int actor_out_fwd_launch(const float* R, const float* V0, const float* wd, long long zsP, float* W3, float* out, long long zsS,
                                float max_action, int T, int nb, cudaStream_t st, int* grid = nullptr) {
  const dim3 g(grid_for_warps(T), nb);
  launch_k(actor_out_fwd_kernel, g, 256, 0, st, R, V0, wd, zsP, W3, out, zsS, max_action, T);
  return launched(g, grid);
}

// wgrad: dwd is a parameter gradient (one CTA in deterministic mode), else scratch whose sums are discarded
inline int actor_out_bwd_launch(const float* dOut, long long zsDo, const float* out, const float* R, const float* V0, long long zsS, const float* wd,
                                long long zsP, float* dR, long long zsW, float* dwd, long long zsG, bool wgrad, float max_action, int T, int nb,
                                cudaStream_t st, int* grid = nullptr) {
  int gx = grid_for_warps(T); if (gx > 2 * NUM_SMS) gx = 2 * NUM_SMS;
  if (wgrad && det_enabled()) gx = 1;
  const dim3 g(gx, nb);
  launch_k(actor_out_bwd_kernel, g, 256, 0, st, dOut, zsDo, out, R, V0, zsS, wd, zsP, dR, zsW, dwd, zsG, max_action, T);
  return launched(g, grid);
}

inline int rowdiv_bwd_launch(float* dy, int lddy, long long zsW, const float* y, int ldy, const float* Fn, long long zsS, float* dF, int N,
                             float colscale, int cs_n, int T, const float* src, int ldsrc, long long zsSrc, int nb, cudaStream_t st,
                             int* grid = nullptr) {
  const dim3 g(grid_for_warps(T), nb);
  launch_k(rowdiv_bwd_kernel, g, 256, 0, st, dy, lddy, zsW, y, ldy, Fn, zsS, dF, N, colscale, cs_n, T, src, ldsrc, zsSrc);
  return launched(g, grid);
}

inline int colsum_launch(const float* X, int ldx, long long zsX, float* out, long long zsO, int M, int N, float alpha, int nb, cudaStream_t st,
                         int* grid = nullptr) {
  int gy = ceil_div(M, 64); if (gy > 32) gy = 32; if (gy < 1) gy = 1;
  if (det_enabled()) gy = 1;
  const dim3 g(ceil_div(N, 32), gy, nb);
  launch_k(colsum_kernel, g, 256, 0, st, X, ldx, zsX, out, zsO, M, N, alpha);
  return launched(g, grid);
}

inline int block_copy_launch(float* dst, int ldd, long long zsD, const float* src, int lds, long long zsSrc, const float* src2, int lds2,
                             long long zsSrc2, int M, int N, int add, int nb, cudaStream_t st, int* grid = nullptr) {
  int gx = ceil_div((long long)M * N, 256); if (gx > 4 * NUM_SMS) gx = 4 * NUM_SMS; if (gx < 1) gx = 1;
  const dim3 g(gx, nb);
  launch_k(block_copy_kernel, g, 256, 0, st, dst, ldd, zsD, src, lds, zsSrc, src2, lds2, zsSrc2, M, N, add);
  return launched(g, grid);
}

}  // namespace sgrl
