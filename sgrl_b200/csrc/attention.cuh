// K2 — masked multi-head SET attention over packed variable-size limb graphs
// (subequivariant_attentions.py:109-151).  H=2 heads of width 128, <= 16 limbs per graph.
//
// One CTA (a warp-group of 4 warps forward, 8 warps backward) per graph: the graph's
// q|k|v rows and its vector-stream values [vg_proj(Vg) | gravity | direction] are staged in
// shared memory once, scores for both heads are formed there, the softmax over the
// graph's own limbs runs on 16-lane shuffle groups (padding never enters: each graph
// only ever sees its cu_limbs[g]..cu_limbs[g+1] rows, which is what "masking padded keys
// with -inf" reduces to for a packed layout), and the same probabilities weight the
// scalar values (-> o, T x 256) and the three spatial rows of the vector values
// (-> og, T x 3 x 256).  Layer 0 adds the relational bias W_rel . relation[i][j] + b_rel
// (SEActor.py:156-158) computed on the fly from the per-morphology relation table.
#pragma once
#include "common.cuh"
#include "layout.h"

namespace sgrl {

constexpr int A_RS = 772;       // padded smem row stride for 768-float rows (bank offset 4/row)
constexpr int A_DS = 1028;      // padded stride for do|dog rows (256+768)
constexpr int A_FWD_THREADS = 128;
constexpr int A_BWD_THREADS = 256;

struct AttnGraphs {
  const int* cu_limbs;    // (G+1) token offsets
  const int* rel_off;     // (G) float offset of each graph's (n,n,3) relation table, or nullptr (all 0)
  const float* relation;  // packed relation tables
  int G;
  int T;                  // total tokens (profiling/bookkeeping only)
  int nmax;               // largest graph of the batch (limbs), 0 = unknown (MAXN): sizes the shared-memory staging, i.e. CTAs per SM
};
inline int attn_rows(const AttnGraphs& gr) { return (gr.nmax >= 2 && gr.nmax <= MAXN) ? gr.nmax : MAXN; }

// Ampere-style asynchronous copies global -> shared (LDGSTS): a thread issues all of its copies back to back and waits
// once, instead of one exposed global-load latency per loop iteration (the first version staged a 9-limb graph with ~40
// dependent load->store round trips per thread: 25 us per graph and CTA, 27 % of HBM at 147 K tokens).
__device__ __forceinline__ void cp_async16(float* dst, const float* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(float* dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

__device__ __forceinline__ void attn_stage_common(float* qs, float* vs, const float* __restrict__ QKV,
                                                  const float* __restrict__ VGP, const float* __restrict__ GD,
                                                  int t0, int n, int tid, int nthr) {
  for (int i = tid; i < n * 192; i += nthr) {
    const int tk = i / 192, c4 = (i % 192) * 4;
    cp_async16(qs + tk * A_RS + c4, QKV + (long long)(t0 + tk) * 768 + c4);
  }
  // vg rows: (t, r, h) -> 126 learned channels, 8-byte aligned
  for (int i = tid; i < n * 6 * 63; i += nthr) {
    const int c2 = i % 63, rh = (i / 63) % 6, tk = i / (63 * 6);
    const int r = rh >> 1, h = rh & 1;
    cp_async8(vs + tk * A_RS + r * 256 + h * 128 + c2 * 2, VGP + (long long)(t0 + tk) * 756 + r * 252 + h * 126 + c2 * 2);
  }
  for (int i = tid; i < n * 6; i += nthr) {
    const int tk = i / 6, r = (i % 6) >> 1, k = i & 1;
    const float v = __ldg(GD + (long long)(t0 + tk) * 6 + (i % 6));
    vs[tk * A_RS + r * 256 + 126 + k] = v;
    vs[tk * A_RS + r * 256 + 128 + 126 + k] = v;
  }
}

__global__ void __launch_bounds__(A_FWD_THREADS) attention_fwd_kernel(
    const float* __restrict__ QKV, const float* __restrict__ VGP, const float* __restrict__ GD,
    float* __restrict__ O, float* __restrict__ OG, float* __restrict__ P, long long zsS,
    const float* __restrict__ Wrel, const float* __restrict__ brel, long long zsP,   // nullptr unless layer 0
    AttnGraphs gr) {
  SGRL_PDL_ENTER();
  extern __shared__ __align__(16) float smem[];
  const int nr = (gr.nmax >= 2 && gr.nmax <= MAXN) ? gr.nmax : MAXN;
  // (a second staging buffer with the next graph's copies in flight under the arithmetic was measured SLOWER: it halves
  //  the CTAs per SM to 2 x 4 warps and the arithmetic phases are latency-bound: 1 506 vs 3 156 GB/s at 147 K tokens)
  float* qs = smem;                     // [nr][A_RS]   q | k | v
  float* vs = qs + nr * A_RS;           // [nr][A_RS]   vgx: [r][h][128]
  float* S = vs + nr * A_RS;            // [2][16][16]  scores
  float* PT = S + 512;                  // [2][16][16]  probabilities, transposed: [h][j][i]
  const int tid = threadIdx.x, z = blockIdx.y;
  QKV += z * zsS; VGP += z * zsS; GD += z * zsS; O += z * zsS; OG += z * zsS;
  if (P) P += z * zsS;
  float wr[HEADS][3] = {{0, 0, 0}, {0, 0, 0}}, br[HEADS] = {0, 0};
  const bool has_bias = Wrel != nullptr;
  if (has_bias) {
    Wrel += z * zsP; brel += z * zsP;
#pragma unroll
    for (int h = 0; h < HEADS; ++h) { br[h] = brel[h]; for (int c = 0; c < 3; ++c) wr[h][c] = Wrel[h * 3 + c]; }
  }
  for (int g = blockIdx.x; g < gr.G; g += gridDim.x) {
    const int t0 = gr.cu_limbs[g], n = gr.cu_limbs[g + 1] - t0;
    const float* rel = has_bias ? gr.relation + (gr.rel_off ? gr.rel_off[g] : 0) : nullptr;
    __syncthreads();
    attn_stage_common(qs, vs, QKV, VGP, GD, t0, n, tid, A_FWD_THREADS);
    cp_async_wait_all();
    __syncthreads();
    // ---- scores S[h][i][j] = q_i . k_j (+ bias)
    for (int idx = tid; idx < HEADS * n * n; idx += A_FWD_THREADS) {
      const int h = idx / (n * n), ij = idx % (n * n), i = ij / n, j = ij % n;
      const float* q = qs + i * A_RS + h * 128;
      const float* k = qs + j * A_RS + 256 + h * 128;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
      for (int c = 0; c < 128; c += 4) {
        const float4 qv = *reinterpret_cast<const float4*>(q + c), kv = *reinterpret_cast<const float4*>(k + c);
        a0 = fmaf(qv.x, kv.x, a0); a1 = fmaf(qv.y, kv.y, a1); a2 = fmaf(qv.z, kv.z, a2); a3 = fmaf(qv.w, kv.w, a3);
      }
      float s = (a0 + a1) + (a2 + a3);
      if (has_bias) {
        const float* rr = rel + (i * n + j) * 3;
        s += wr[h][0] * rr[0] + wr[h][1] * rr[1] + wr[h][2] * rr[2] + br[h];
      }
      S[(h * 16 + i) * 16 + j] = s;
    }
    __syncthreads();
    // ---- softmax over the graph's own limbs: 16-lane shuffle groups, one row each.  The probabilities are kept
    // TRANSPOSED in shared memory (S[h][j][i]) so that the weighted sums below fetch P[0..15][j] with four 128-bit loads.
    for (int row = tid >> 4; row < HEADS * 16; row += A_FWD_THREADS / 16) {
      const int h = row >> 4, i = row & 15, j = tid & 15;
      const bool valid = (i < n) && (j < n);          // uniform per 16-lane group in i
      float v = valid ? S[row * 16 + j] : -INFINITY;
      float m = v;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o, 16));
      float e = valid ? expf(v - m) : 0.f;
      float sum = e;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o, 16);
      const float p = valid ? e / sum : 0.f;
      PT[(h * 16 + j) * 16 + i] = p;
      if (P && i < n) P[(long long)(t0 + i) * 32 + h * 16 + j] = p;
    }
    __syncthreads();
    // ---- weighted sums: 256 scalar-stream + 768 vector-stream columns.  A thread owns 4 consecutive columns x all rows
    // (64 accumulators): per key j one 128-bit load of the values and up to four of P^T[j][.] feed 64 FMAs (the first
    // version re-read P from shared memory for every column: 17 loads per 16 FMAs, shared-memory bound at 27 % of HBM).
    const int ng4 = (n + 3) >> 2;
    for (int col4 = tid * 4; col4 < 1024; col4 += A_FWD_THREADS * 4) {
      const bool sc = col4 < 256;
      const int cc = sc ? col4 : col4 - 256;
      const int h = (cc & 255) >> 7;
      const float* src = sc ? qs + 512 + cc : vs + cc;
      const float* Ph = PT + h * 256;
      float acc[4][MAXN];
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int i = 0; i < MAXN; ++i) acc[c][i] = 0.f;
      for (int j = 0; j < n; ++j) {
        const float4 vv = *reinterpret_cast<const float4*>(src + j * A_RS);
#pragma unroll
        for (int g4 = 0; g4 < MAXN / 4; ++g4) {
          if (g4 < ng4) {
            const float4 p4 = *reinterpret_cast<const float4*>(Ph + j * 16 + g4 * 4);
            const float pv[4] = {p4.x, p4.y, p4.z, p4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              acc[0][g4 * 4 + k] = fmaf(pv[k], vv.x, acc[0][g4 * 4 + k]);
              acc[1][g4 * 4 + k] = fmaf(pv[k], vv.y, acc[1][g4 * 4 + k]);
              acc[2][g4 * 4 + k] = fmaf(pv[k], vv.z, acc[2][g4 * 4 + k]);
              acc[3][g4 * 4 + k] = fmaf(pv[k], vv.w, acc[3][g4 * 4 + k]);
            }
          }
        }
      }
      float* dst = sc ? O + (long long)t0 * 256 + cc : OG + (long long)t0 * 768 + cc;
      const int ldo = sc ? 256 : 768;
#pragma unroll
      for (int i = 0; i < MAXN; ++i)
        if (i < n) stg4(dst + (long long)i * ldo, make_float4(acc[0][i], acc[1][i], acc[2][i], acc[3][i]));
    }
  }
}

// ---- forward, second version: only q | k are staged.
// Every value element (v, vg, gd) is used by exactly ONE thread of the weighted-sum phase, once per graph, so staging the values
// in shared memory bought nothing and cost two thirds of the 60 KB that limited the first version to 3 CTAs (12 warps) per SM —
// with serialised phases per graph (stage -> scores -> softmax -> sums) that is what kept it at 0.48 of HBM at 147 K tokens.
// Here a thread reads its four value columns straight from global memory (a warp = 512 contiguous bytes of a row), with the
// first rows' loads issued BEFORE the scores phase so that their latency hides behind it; shared memory per CTA drops to
// 19 KB + 4 KB (9-limb graphs) and the register file becomes the occupancy limit (NR = 12 or 16 accumulator rows).
constexpr int A_QS = 516;       // padded smem row stride for the 512 staged floats (q | k) of a token
#ifndef ATTN_JB
#define ATTN_JB 8               // value rows a thread keeps in flight (float4 each)
#endif
#ifndef ATTN_MINB
#define ATTN_MINB 4             // CTAs per SM the register allocation is bounded for
#endif
template <int NR>
__device__ __forceinline__ void attn_load_vals(float4 (&vv)[ATTN_JB], const float* __restrict__ QKV, const float* __restrict__ VGP, const float* __restrict__ GD,
                                               int t0, int j0, int j1, int col4) {
#pragma unroll
  for (int jj = 0; jj < ATTN_JB; ++jj) {
    const int j = j0 + jj;
    if (j >= j1) break;
    const long long t = t0 + j;
    if (col4 < 256) vv[jj] = __ldg(reinterpret_cast<const float4*>(QKV + t * 768 + 512 + col4));
    else {
      const int cc = col4 - 256, r = cc >> 8, h = (cc >> 7) & 1, c = cc & 127;
      const float* src = VGP + t * 756 + r * 252 + h * 126 + c;
      const float2 a = __ldg(reinterpret_cast<const float2*>(src));
      const float2 b = c < 124 ? __ldg(reinterpret_cast<const float2*>(src + 2)) : __ldg(reinterpret_cast<const float2*>(GD + t * 6 + r * 2));
      vv[jj] = make_float4(a.x, a.y, b.x, b.y);
    }
  }
}

template <int NR>
__global__ void __launch_bounds__(A_FWD_THREADS, ATTN_MINB) attention_fwd_v2_kernel(
    const float* __restrict__ QKV, const float* __restrict__ VGP, const float* __restrict__ GD,
    float* __restrict__ O, float* __restrict__ OG, float* __restrict__ P, long long zsS,
    const float* __restrict__ Wrel, const float* __restrict__ brel, long long zsP,   // nullptr unless layer 0
    AttnGraphs gr) {
  SGRL_PDL_ENTER();
  extern __shared__ __align__(16) float smem[];
  const int nr = (gr.nmax >= 2 && gr.nmax <= MAXN) ? gr.nmax : MAXN;
  float* qs = smem;                     // [nr][A_QS]   q | k
  float* S = qs + nr * A_QS;            // [2][16][16]  scores
  float* PT = S + 512;                  // [2][16][16]  probabilities, transposed: [h][j][i]
  const int tid = threadIdx.x, z = blockIdx.y;
  QKV += z * zsS; VGP += z * zsS; GD += z * zsS; O += z * zsS; OG += z * zsS;
  if (P) P += z * zsS;
  float wr[HEADS][3] = {{0, 0, 0}, {0, 0, 0}}, br[HEADS] = {0, 0};
  const bool has_bias = Wrel != nullptr;
  if (has_bias) {
    Wrel += z * zsP; brel += z * zsP;
#pragma unroll
    for (int h = 0; h < HEADS; ++h) { br[h] = brel[h]; for (int c = 0; c < 3; ++c) wr[h][c] = Wrel[h * 3 + c]; }
  }
  for (int g = blockIdx.x; g < gr.G; g += gridDim.x) {
    const int t0 = gr.cu_limbs[g], n = gr.cu_limbs[g + 1] - t0;
    const float* rel = has_bias ? gr.relation + (gr.rel_off ? gr.rel_off[g] : 0) : nullptr;
    __syncthreads();                    // the previous graph's scores / probabilities have been consumed
    for (int i = tid; i < n * 128; i += A_FWD_THREADS) {
      const int tk = i >> 7, c4 = (i & 127) * 4;
      cp_async16(qs + tk * A_QS + c4, QKV + (long long)(t0 + tk) * 768 + c4);
    }
    // value rows 0..7 of this thread's first column group: in flight during the scores and softmax phases
    float4 vv[ATTN_JB];
    attn_load_vals<NR>(vv, QKV, VGP, GD, t0, 0, n, tid * 4);
    cp_async_wait_all();
    __syncthreads();
    // ---- scores S[h][i][j] = q_i . k_j (+ bias)
    for (int idx = tid; idx < HEADS * n * n; idx += A_FWD_THREADS) {
      const int h = idx / (n * n), ij = idx % (n * n), i = ij / n, j = ij % n;
      const float* q = qs + i * A_QS + h * 128;
      const float* k = qs + j * A_QS + 256 + h * 128;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
      for (int c = 0; c < 128; c += 4) {
        const float4 qv = *reinterpret_cast<const float4*>(q + c), kv = *reinterpret_cast<const float4*>(k + c);
        a0 = fmaf(qv.x, kv.x, a0); a1 = fmaf(qv.y, kv.y, a1); a2 = fmaf(qv.z, kv.z, a2); a3 = fmaf(qv.w, kv.w, a3);
      }
      float s = (a0 + a1) + (a2 + a3);
      if (has_bias) {
        const float* rr = rel + (i * n + j) * 3;
        s += wr[h][0] * rr[0] + wr[h][1] * rr[1] + wr[h][2] * rr[2] + br[h];
      }
      S[(h * 16 + i) * 16 + j] = s;
    }
    __syncthreads();
    // ---- softmax (same arithmetic as the first version), probabilities kept transposed: PT[h][j][i]
    for (int row = tid >> 4; row < HEADS * 16; row += A_FWD_THREADS / 16) {
      const int h = row >> 4, i = row & 15, j = tid & 15;
      const bool valid = (i < n) && (j < n);
      float v = valid ? S[row * 16 + j] : -INFINITY;
      float m = v;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o, 16));
      float e = valid ? expf(v - m) : 0.f;
      float sum = e;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o, 16);
      const float p = valid ? e / sum : 0.f;
      PT[(h * 16 + j) * 16 + i] = p;
      if (P && i < n) P[(long long)(t0 + i) * 32 + h * 16 + j] = p;
    }
    __syncthreads();
    // ---- weighted sums: thread = 4 consecutive columns x all rows; same accumulation order over j as the first version
    constexpr int NG4 = NR / 4;
    const int ng4 = (n + 3) >> 2;
#pragma unroll 1
    for (int rd = 0; rd < 2; ++rd) {
      const int col4 = rd * 512 + tid * 4;
      const bool sc = col4 < 256;
      const int cc = sc ? col4 : col4 - 256;
      const int h = (cc & 255) >> 7;
      const float* Ph = PT + h * 256;
      float acc[4][NR];
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int i = 0; i < NR; ++i) acc[c][i] = 0.f;
#pragma unroll 1
      for (int j0 = 0; j0 < n; j0 += ATTN_JB) {
        if (rd > 0 || j0 > 0) attn_load_vals<NR>(vv, QKV, VGP, GD, t0, j0, n, col4);
#pragma unroll
        for (int jj = 0; jj < ATTN_JB; ++jj) {
          const int j = j0 + jj;
          if (j >= n) break;
          const float4 x = vv[jj];
#pragma unroll
          for (int g4 = 0; g4 < NG4; ++g4) {
            if (g4 < ng4) {
              const float4 p4 = *reinterpret_cast<const float4*>(Ph + j * 16 + g4 * 4);
              const float pv[4] = {p4.x, p4.y, p4.z, p4.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                acc[0][g4 * 4 + k] = fmaf(pv[k], x.x, acc[0][g4 * 4 + k]);
                acc[1][g4 * 4 + k] = fmaf(pv[k], x.y, acc[1][g4 * 4 + k]);
                acc[2][g4 * 4 + k] = fmaf(pv[k], x.z, acc[2][g4 * 4 + k]);
                acc[3][g4 * 4 + k] = fmaf(pv[k], x.w, acc[3][g4 * 4 + k]);
              }
            }
          }
        }
      }
      float* dst = sc ? O + (long long)t0 * 256 + cc : OG + (long long)t0 * 768 + cc;
      const int ldo = sc ? 256 : 768;
#pragma unroll
      for (int i = 0; i < NR; ++i)
        if (i < n) stg4(dst + (long long)i * ldo, make_float4(acc[0][i], acc[1][i], acc[2][i], acc[3][i]));
    }
  }
}
constexpr size_t attn_fwd_v2_smem(int nr = MAXN) { return sizeof(float) * (nr * A_QS + 1024); }

constexpr size_t attn_fwd_smem(int nr = MAXN) { return sizeof(float) * (2 * nr * A_RS + 1024); }
constexpr size_t attn_bwd_smem(int nr = MAXN) { return sizeof(float) * (2 * nr * A_RS + nr * A_DS + 1536 + 64); }

// Backward.  Inputs dO (T,256), dOG (T,768) [workspace], saved P, QKV, VGP, GD [stash].
// Outputs dQKV (T,768) — gradient w.r.t. the *stored* (post /F, post-scale) q|k|v — and
// dVGP (T,756); layer 0 also accumulates d rel_encoder.weight (bias gradient is exactly 0).
__global__ void __launch_bounds__(A_BWD_THREADS) attention_bwd_kernel(
    const float* __restrict__ QKV, const float* __restrict__ VGP, const float* __restrict__ GD, const float* __restrict__ P, long long zsS,
    const float* __restrict__ dO, const float* __restrict__ dOG, float* __restrict__ dQKV, float* __restrict__ dVGP, long long zsW,
    float* __restrict__ dWrel, long long zsG, AttnGraphs gr, float* __restrict__ wpart) {
  SGRL_PDL_ENTER();
  extern __shared__ __align__(16) float smem[];
  const int nr = (gr.nmax >= 2 && gr.nmax <= MAXN) ? gr.nmax : MAXN;
  float* qs = smem;
  float* vs = qs + nr * A_RS;
  float* ds = vs + nr * A_RS;            // [nr][A_DS]  dO | dOG
  float* Ps = ds + nr * A_DS;            // [2][16][16]
  float* dS = Ps + 512;                  // [2][16][16]
  float* dST = dS + 512;                 // [2][16][16]  transposed: [h][j][i]
  float* wacc = dST + 512;               // [8 warps][6]
  const int tid = threadIdx.x, z = blockIdx.y;
  QKV += z * zsS; VGP += z * zsS; GD += z * zsS; P += z * zsS;
  dO += z * zsW; dOG += z * zsW; dQKV += z * zsW; dVGP += z * zsW;
  const bool has_bias = dWrel != nullptr;
  if (has_bias) dWrel += z * zsG;
  float wloc[6] = {0, 0, 0, 0, 0, 0};
  for (int g = blockIdx.x; g < gr.G; g += gridDim.x) {
    const int t0 = gr.cu_limbs[g], n = gr.cu_limbs[g + 1] - t0;
    const float* rel = has_bias ? gr.relation + (gr.rel_off ? gr.rel_off[g] : 0) : nullptr;
    __syncthreads();
    attn_stage_common(qs, vs, QKV, VGP, GD, t0, n, tid, A_BWD_THREADS);
    for (int i = tid; i < n * 256; i += A_BWD_THREADS) {
      const int tk = i >> 8, c4 = (i & 255) * 4;
      cp_async16(ds + tk * A_DS + c4, c4 < 256 ? dO + (long long)(t0 + tk) * 256 + c4 : dOG + (long long)(t0 + tk) * 768 + (c4 - 256));
    }
    for (int i = tid; i < 512; i += A_BWD_THREADS) {
      const int h = i >> 8, ii = (i >> 4) & 15, j = i & 15;
      Ps[i] = (ii < n) ? __ldg(P + (long long)(t0 + ii) * 32 + h * 16 + j) : 0.f;
    }
    cp_async_wait_all();
    __syncthreads();
    // ---- dP[h][i][j] = dO_i . v_j + sum_r dOG_i,r . vgx_j,r
    for (int idx = tid; idx < HEADS * n * n; idx += A_BWD_THREADS) {
      const int h = idx / (n * n), ij = idx % (n * n), i = ij / n, j = ij % n;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      const float* d0 = ds + i * A_DS + h * 128;
      const float* v0 = qs + j * A_RS + 512 + h * 128;
#pragma unroll 8
      for (int c = 0; c < 128; c += 4) {
        const float4 a = *reinterpret_cast<const float4*>(d0 + c), b = *reinterpret_cast<const float4*>(v0 + c);
        a0 = fmaf(a.x, b.x, a0); a1 = fmaf(a.y, b.y, a1); a2 = fmaf(a.z, b.z, a2); a3 = fmaf(a.w, b.w, a3);
      }
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float* d1 = ds + i * A_DS + 256 + r * 256 + h * 128;
        const float* v1 = vs + j * A_RS + r * 256 + h * 128;
#pragma unroll 8
        for (int c = 0; c < 128; c += 4) {
          const float4 a = *reinterpret_cast<const float4*>(d1 + c), b = *reinterpret_cast<const float4*>(v1 + c);
          a0 = fmaf(a.x, b.x, a0); a1 = fmaf(a.y, b.y, a1); a2 = fmaf(a.z, b.z, a2); a3 = fmaf(a.w, b.w, a3);
        }
      }
      dS[(h * 16 + i) * 16 + j] = (a0 + a1) + (a2 + a3);
    }
    __syncthreads();
    // ---- dS = P * (dP - sum_j dP*P), 16-lane groups per row
    for (int row = tid >> 4; row < HEADS * 16; row += A_BWD_THREADS / 16) {
      const int i = row & 15, j = tid & 15;
      const bool valid = (i < n) && (j < n);
      const float p = valid ? Ps[row * 16 + j] : 0.f;
      const float dp = valid ? dS[row * 16 + j] : 0.f;
      float s = p * dp;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, 16);
      const float v = p * (dp - s);
      dS[row * 16 + j] = v;
      dST[((row >> 4) * 16 + j) * 16 + i] = v;
      if (has_bias && valid) {
        const int h = row >> 4;
        const float* rr = rel + (i * n + j) * 3;
        wloc[h * 3 + 0] = fmaf(v, rr[0], wloc[h * 3 + 0]);
        wloc[h * 3 + 1] = fmaf(v, rr[1], wloc[h * 3 + 1]);
        wloc[h * 3 + 2] = fmaf(v, rr[2], wloc[h * 3 + 2]);
      }
    }
    __syncthreads();
    // ---- column sweeps: 256 dq + 256 dk + 256 dv + 768 dvg columns.  A thread owns 4 consecutive columns x all rows
    // (64 accumulators); per source row one 128-bit load of the operand and up to four of the weight row feed 64 FMAs
    // (same restructuring as the forward's weighted sums: the first version re-read the weights for every column).
    const int ng4 = (n + 3) >> 2;
    for (int task = tid; task < 384; task += A_BWD_THREADS) {
      const int col4 = task * 4;
      const int kind = col4 < 768 ? col4 >> 8 : 3;
      const int col = kind < 3 ? (col4 & 255) : col4 - 768;
      const int h = (col & 255) >> 7;
      // kind 0: dq_i = sum_j dS[i][j] k_j (weights dS^T[j][.]); 1: dk_j = sum_i dS[i][j] q_i; 2: dv_j = sum_i P[i][j] dO_i; 3: dvg_j = sum_i P[i][j] dOG_i
      const float* W = (kind == 0 ? dST : kind == 1 ? dS : Ps) + h * 256;
      const float* src = kind == 0 ? qs + 256 + col : kind == 1 ? qs + col : kind == 2 ? ds + col : ds + 256 + col;
      const int stride = kind < 2 ? A_RS : A_DS;
      float acc[4][MAXN];
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int i = 0; i < MAXN; ++i) acc[c][i] = 0.f;
      for (int sr = 0; sr < n; ++sr) {
        const float4 xv = *reinterpret_cast<const float4*>(src + sr * stride);
#pragma unroll
        for (int g4 = 0; g4 < MAXN / 4; ++g4) {
          if (g4 < ng4) {
            const float4 w4 = *reinterpret_cast<const float4*>(W + sr * 16 + g4 * 4);
            const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              acc[0][g4 * 4 + k] = fmaf(wv[k], xv.x, acc[0][g4 * 4 + k]);
              acc[1][g4 * 4 + k] = fmaf(wv[k], xv.y, acc[1][g4 * 4 + k]);
              acc[2][g4 * 4 + k] = fmaf(wv[k], xv.z, acc[2][g4 * 4 + k]);
              acc[3][g4 * 4 + k] = fmaf(wv[k], xv.w, acc[3][g4 * 4 + k]);
            }
          }
        }
      }
      if (kind < 3) {
        float* dst = dQKV + (long long)t0 * 768 + kind * 256 + col;
#pragma unroll
        for (int i = 0; i < MAXN; ++i)
          if (i < n) stg4(dst + (long long)i * 768, make_float4(acc[0][i], acc[1][i], acc[2][i], acc[3][i]));
      } else {
        const int c = col & 127, r = col >> 8;      // channels 126,127 of each (r, h) are inputs (gravity, direction): no gradient
        if (c < 126) {
          float* dst = dVGP + (long long)t0 * 756 + r * 252 + h * 126 + c;   // 8-byte aligned
#pragma unroll
          for (int i = 0; i < MAXN; ++i)
            if (i < n) {
              *reinterpret_cast<float2*>(dst + (long long)i * 756) = make_float2(acc[0][i], acc[1][i]);
              if (c + 2 < 126) *reinterpret_cast<float2*>(dst + (long long)i * 756 + 2) = make_float2(acc[2][i], acc[3][i]);
            }
        }
      }
    }
  }
  if (has_bias) {
    // per-warp sums added in warp order (a fixed order: the CTA's contribution does not depend on timing)
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const float s = warp_sum(wloc[k]);
      if ((tid & 31) == 0) wacc[(tid >> 5) * 6 + k] = s;
    }
    __syncthreads();
    if (tid < 6) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < A_BWD_THREADS / 32; ++w) s += wacc[w * 6 + tid];
      // deterministic mode: the CTA's partial goes to a scratch row, rel_wgrad_reduce_kernel adds the rows in index order
      if (wpart) wpart[(long long)z * zsW + (long long)blockIdx.x * 6 + tid] = s;
      else atomicAdd(dWrel + tid, s);
    }
  }
}

inline int attention_fwd(const float* QKV, const float* VGP, const float* GD, float* O, float* OG, float* P, long long zsS,
                         const float* Wrel, const float* brel, long long zsP, const AttnGraphs& gr, int nb, cudaStream_t st) {
  if (gr.G <= 0) return 0;
  static bool attr_done = false;
  if (!attr_done) {
    SGRL_CUDA(cudaFuncSetAttribute(attention_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_fwd_smem()));
    attr_done = true;
  }
  const int nr = attn_rows(gr);
  if (gr.G >= 4 * NUM_SMS) {      // few graphs: one graph's latency is what counts and the first version's is shorter (18.4 vs 19.5 us at 256 graphs)
    static int occ12 = 0, occ16 = 0;
    if (!occ12) {
      SGRL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ12, attention_fwd_v2_kernel<12>, A_FWD_THREADS, attn_fwd_v2_smem(12)));
      SGRL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ16, attention_fwd_v2_kernel<16>, A_FWD_THREADS, attn_fwd_v2_smem(16)));
      if (occ12 < 1) occ12 = 1;
      if (occ16 < 1) occ16 = 1;
    }
    const int per_sm = nr <= 12 ? occ12 : occ16;
    const int gx = gr.G < per_sm * NUM_SMS ? gr.G : per_sm * NUM_SMS;
    prof_begin(PC_ATTENTION, (double)gr.T * nb * (3072.0 + 3024 + 24 + 1024 + 3072 + (P ? 128 : 0)), st);
    if (nr <= 12) launch_k(attention_fwd_v2_kernel<12>, dim3(gx, nb), A_FWD_THREADS, attn_fwd_v2_smem(nr), st, QKV, VGP, GD, O, OG, P, zsS, Wrel, brel, zsP, gr);
    else launch_k(attention_fwd_v2_kernel<16>, dim3(gx, nb), A_FWD_THREADS, attn_fwd_v2_smem(nr), st, QKV, VGP, GD, O, OG, P, zsS, Wrel, brel, zsP, gr);
    prof_end(st);
    SGRL_LAUNCH_OK();
    return 0;
  }
  const int per_sm = (int)((227 * 1024) / (attn_fwd_smem(nr) + 1024)) < 8 ? (int)((227 * 1024) / (attn_fwd_smem(nr) + 1024)) : 8;
  const int gx = gr.G < per_sm * NUM_SMS ? gr.G : per_sm * NUM_SMS;
  // algorithmic bytes per token (SURVEY.md 8d): read q|k|v 3072 + vg 3024 + gd 24, write o 1024 + og 3072 (+ P 128)
  prof_begin(PC_ATTENTION, (double)gr.T * nb * (3072.0 + 3024 + 24 + 1024 + 3072 + 128), st);
  launch_k(attention_fwd_kernel, dim3(gx, nb), A_FWD_THREADS, attn_fwd_smem(nr), st, QKV, VGP, GD, O, OG, P, zsS, Wrel, brel, zsP, gr);
  prof_end(st);
  SGRL_LAUNCH_OK();
  return 0;
}

// d rel_encoder.weight += sum over the CTAs' partial rows, in index order (deterministic mode)
__global__ void __launch_bounds__(32) rel_wgrad_reduce_kernel(const float* __restrict__ wpart, long long zsW, int nparts, float* __restrict__ dWrel, long long zsG) {
  SGRL_PDL_ENTER();
  const int z = blockIdx.y;
  if (threadIdx.x < 6) {
    float s = 0.f;
    for (int b = 0; b < nparts; ++b) s += wpart[(long long)z * zsW + (long long)b * 6 + threadIdx.x];
    dWrel[(long long)z * zsG + threadIdx.x] += s;
  }
}

// scratch (deterministic mode, layer 0 only): >= 6 * min(G, 4 * NUM_SMS) floats per net instance, z-stride zsW; nullptr otherwise
inline int attention_bwd(const float* QKV, const float* VGP, const float* GD, const float* P, long long zsS,
                         const float* dO, const float* dOG, float* dQKV, float* dVGP, long long zsW,
                         float* dWrel, long long zsG, const AttnGraphs& gr, int nb, cudaStream_t st, float* scratch = nullptr) {
  if (gr.G <= 0) return 0;
  static bool attr_done = false;
  if (!attr_done) {
    SGRL_CUDA(cudaFuncSetAttribute(attention_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_bwd_smem()));
    attr_done = true;
  }
  const int nr = attn_rows(gr);
  const int per_sm = (int)((227 * 1024) / (attn_bwd_smem(nr) + 1024)) < 4 ? (int)((227 * 1024) / (attn_bwd_smem(nr) + 1024)) : 4;
  int gx = gr.G < per_sm * NUM_SMS ? gr.G : per_sm * NUM_SMS;
  float* wpart = (dWrel && det_enabled()) ? scratch : nullptr;
  if (dWrel && det_enabled() && !scratch) gx = 1;      // no scratch (stand-alone call): one CTA walks every graph, one add per address
  launch_k(attention_bwd_kernel, dim3(gx, nb), A_BWD_THREADS, attn_bwd_smem(nr), st, QKV, VGP, GD, P, zsS, dO, dOG, dQKV, dVGP, zsW, dWrel, zsG, gr, wpart);
  SGRL_LAUNCH_OK();
  if (wpart) {
    launch_k(rel_wgrad_reduce_kernel, dim3(1, nb), 32, 0, st, (const float*)wpart, zsW, gx, dWrel, zsG);
    SGRL_LAUNCH_OK();
  }
  return 0;
}

}  // namespace sgrl
