// K1 — per-limb invariant feature construction (SURVEY.md §2 K1, Appendix A.3).
//
// For every limb-token t with vector-stream features X_t (3 x C):
//     Z_t = [ X_t P^T | gd_t ]            (3 x 32)   30 learned channels + gravity + target dir
//     G_t = Z_t^T Z_t                     (32 x 32)  O(3)-invariant Gram; column 30 = projection
//                                                    of every channel onto the gravity axis
//     F_t = ||G_t||_F + 1
// replaces  g_proj -> cat gdir -> bmm(Z^T,Z) -> norm+1  of
// subequivariant_attentions.py:90-96, SEActor.py:93-100 and SEActor.py:256-262.
// Optionally a second projection P' gives Z'_t = [X_t P'^T | gd_t] (the operand of the
// per-token matrix apply, SEActor.py:108-110 / :273-274) from the same staged X tile.
//
// G is symmetric: only its upper triangle (528 entries, row-major i<=j, zero-padded to GP_K = 544) is written, and the
// consumers contract it against triangle-folded weights (layout.h, fold_sym_kernel below).
// HBM-bound: reads 12*C+24 B, writes 2176+4+384 B per token.  One CTA stages P once and
// walks 32-token tiles: coalesced float4 loads -> padded smem -> 3x4 register micro-tiles
// for the projection -> per-warp Gram rows written as 512 B coalesced float4 stores.
#pragma once
#include "common.cuh"
#include "layout.h"

namespace sgrl {

// p -> (i << 8 | j) of the packed upper triangle (layout.h tri_index); 0xFFFF for the zero padding slots
struct TriLut { unsigned short v[GP_K]; };
constexpr TriLut make_tri_lut() {
  TriLut t{};
  for (int p = 0; p < GP_K; ++p) t.v[p] = 0xFFFFu;
  for (int i = 0; i < CH; ++i)
    for (int j = i; j < CH; ++j) t.v[tri_index(i, j)] = (unsigned short)((i << 8) | j);
  return t;
}
__constant__ TriLut c_tri = make_tri_lut();
// the 144 four-column chunks (i, jq) of the 32x32 Gram that touch the upper triangle (4*jq + 3 >= i), row-major; code = i << 8 | jq
constexpr int GCH = 144, GCH_PAD = 160;
struct ChunkLut { unsigned short v[GCH_PAD]; };
constexpr ChunkLut make_chunk_lut() {
  ChunkLut t{};
  int n = 0;
  for (int i = 0; i < CH; ++i)
    for (int jq = 0; jq < CH / 4; ++jq)
      if (4 * jq + 3 >= i) t.v[n++] = (unsigned short)((i << 8) | jq);
  for (; n < GCH_PAD; ++n) t.v[n] = 0xFFFFu;
  return t;
}
__constant__ ChunkLut c_chunk = make_chunk_lut();

__device__ __forceinline__ void feat_cp_async16(float* dst, const float* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

constexpr int F_TT = 32;        // tokens per tile (16-token tiles at 4 CTAs/SM measured slower: 2 204 vs 2 783 GB/s at 147 K tokens)
constexpr int F_THREADS = 256;

template <int CE, int NPROJ>
struct FeatSmem {
  static constexpr int C = 128 + CE;
  static constexpr int PJ = 32 * NPROJ;
  static constexpr int XS = 3 * C + 4;  // padded token stride (floats)
  // Ps | Xs (the projected Z tile later overwrites the head of Xs) | gd | chunk table
  static constexpr size_t bytes = sizeof(float) * ((size_t)C * PJ + (size_t)F_TT * XS + F_TT * 8 + GCH_PAD / 2);
  static_assert(F_TT * 3 * PJ <= F_TT * XS, "Z tile must fit into the X staging it replaces");
};

// X = [V0 (T,3,8) if CE==8 | Xg (T,3,128)], P1/P2 (30,C) row-major, gd (T,3,2)
template <int CE, int NPROJ>
__global__ void __launch_bounds__(F_THREADS) inv_feature_fwd_kernel(
    const float* __restrict__ Xg, long long zsXg, const float* __restrict__ V0, long long zsV0,
    const float* __restrict__ gd, long long zsGd,
    const float* __restrict__ P1, const float* __restrict__ P2, long long zsP,
    float* __restrict__ Z, float* __restrict__ Z2, float* __restrict__ G, float* __restrict__ Fn, long long zsAct,
    int T) {
  SGRL_PDL_ENTER();
  using S = FeatSmem<CE, NPROJ>;
  constexpr int C = S::C, PJ = S::PJ, XS = S::XS, JQ = PJ / 4;
  extern __shared__ __align__(16) float smem[];
  float* Ps = smem;                       // [C][PJ]
  float* Xs = Ps + C * PJ;                // [TT][XS]
  float* Zs = Xs;                         // [TT][3][PJ]: written over the X tile once every thread has finished projecting
  float* gds = Xs + F_TT * XS;            // [TT][8] (6 used)
  unsigned short* chk = reinterpret_cast<unsigned short*>(gds + F_TT * 8);   // [GCH_PAD] (divergent lookups: not from constant memory)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, z = blockIdx.y;
  Xg += z * zsXg; gd += z * zsGd; P1 += z * zsP;
  if (CE) V0 += z * zsV0;
  if (NPROJ == 2) P2 += z * zsP;
  Z += z * zsAct; G += z * zsAct; Fn += z * zsAct;
  if (NPROJ == 2) Z2 += z * zsAct;

  for (int i = tid; i < GCH_PAD; i += F_THREADS) chk[i] = c_chunk.v[i];
  // stage P transposed: Ps[c][j] = P[j][c]; columns 30,31 (and 62,63) are zero.  Consecutive threads take consecutive j:
  // the shared-memory writes are conflict-free and the 16 strided (L2-resident, 15 KB) loads of a thread are independent;
  // the coalesced-read order made every write a 32-way bank conflict: 6 us of a 22 us launch at 2 304 tokens.
  for (int i = tid; i < C * PJ; i += F_THREADS) {
    const int c = i / PJ, j = i % PJ;
    const int jj = j & 31;
    float v = 0.f;
    if (jj < 30) v = __ldg((j < 32 ? P1 : P2) + jj * C + c);
    Ps[i] = v;
  }

  const int ntiles = (T + F_TT - 1) / F_TT;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int t0 = tile * F_TT;
    __syncthreads();   // previous tile fully consumed (and Ps staged on first pass)
    // ---- stage X tile: asynchronous 16-byte copies, all of a thread's 12 in flight at once
    for (int i = tid; i < F_TT * 3 * 32; i += F_THREADS) {
      const int tk = i / 96, rem = i % 96, r = rem / 32, c4 = (rem % 32) * 4;
      float* dst = &Xs[tk * XS + r * C + CE + c4];
      if (t0 + tk < T) feat_cp_async16(dst, Xg + ((long long)(t0 + tk) * 3 + r) * 128 + c4);
      else *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (CE) {
      for (int i = tid; i < F_TT * 24; i += F_THREADS) {
        const int tk = i / 24, rem = i % 24, r = rem / 8, c = rem % 8;
        Xs[tk * XS + r * C + c] = (t0 + tk < T) ? __ldg(V0 + (long long)(t0 + tk) * 24 + rem) : 0.f;
      }
    }
    for (int i = tid; i < F_TT * 6; i += F_THREADS) {
      const int tk = i / 6;
      gds[tk * 8 + i % 6] = (t0 + tk < T) ? __ldg(gd + (long long)(t0 + tk) * 6 + i % 6) : 0.f;
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    // ---- projection: each thread owns (token, 4 output channels) x 3 spatial rows, NW of them; results stay in registers.
    // lane = token, warp = channel quad: the P loads are warp-uniform (one broadcast wavefront) and the X loads are
    // conflict-free (token rows 4 banks apart); with lanes = 8 channel quads x 4 tokens every 128-bit load cost four
    // wavefronts and the phase ran at the shared-memory limit (7 loads per 48 FMAs).
    constexpr int NW = F_TT * JQ / F_THREADS;
    static_assert(NW * F_THREADS == F_TT * JQ && F_TT == 32, "work items per thread; lane = token");
    float acc[NW][3][4];
#pragma unroll
    for (int u = 0; u < NW; ++u) {
      const int w = tid + u * F_THREADS;
      const int tk = w & 31, jq = w >> 5;
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[u][r][j] = 0.f;
      const float* xr = Xs + tk * XS;
      const float* pj = Ps + jq * 4;
#pragma unroll 2
      for (int c = 0; c < C; c += 4) {
        float4 x[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) x[r] = *reinterpret_cast<const float4*>(xr + r * C + c);
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          const float4 pv = *reinterpret_cast<const float4*>(pj + (c + cc) * PJ);
#pragma unroll
          for (int r = 0; r < 3; ++r) {
            const float xv = cc == 0 ? x[r].x : cc == 1 ? x[r].y : cc == 2 ? x[r].z : x[r].w;
            acc[u][r][0] = fmaf(xv, pv.x, acc[u][r][0]);
            acc[u][r][1] = fmaf(xv, pv.y, acc[u][r][1]);
            acc[u][r][2] = fmaf(xv, pv.z, acc[u][r][2]);
            acc[u][r][3] = fmaf(xv, pv.w, acc[u][r][3]);
          }
        }
      }
      if ((jq & 7) == 7) {   // channels 30,31 of each Z are [gravity, direction]
#pragma unroll
        for (int r = 0; r < 3; ++r) { acc[u][r][2] = gds[tk * 8 + r * 2 + 0]; acc[u][r][3] = gds[tk * 8 + r * 2 + 1]; }
      }
    }
    __syncthreads();   // every thread is done with the X tile: Z may overwrite it
#pragma unroll
    for (int u = 0; u < NW; ++u) {
      const int w = tid + u * F_THREADS;
      const int tk = w & 31, jq = w >> 5;
#pragma unroll
      for (int r = 0; r < 3; ++r)
        *reinterpret_cast<float4*>(&Zs[(tk * 3 + r) * PJ + jq * 4]) = make_float4(acc[u][r][0], acc[u][r][1], acc[u][r][2], acc[u][r][3]);
    }
    __syncthreads();
    // ---- write Z (and Z') coalesced
    for (int i = tid; i < F_TT * 3 * 8 * NPROJ; i += F_THREADS) {
      const int which = i / (F_TT * 24), rem = i % (F_TT * 24), row = rem / 8, q = rem % 8;
      const int tk = row / 3;
      if (t0 + tk < T) {
        const float4 v = *reinterpret_cast<const float4*>(&Zs[row * PJ + which * 32 + q * 4]);
        stg4((which ? Z2 : Z) + ((long long)t0 * 3 + row) * 32 + q * 4, v);
      }
    }
    // ---- Gram (upper triangle) + Frobenius norm: one warp per token.  The 144 four-column chunks (i, jq) that touch
    // the triangle are dealt to the lanes in row-major order: 3 scalar + 3 128-bit loads and 12 FMAs per chunk
    // (the per-element table walk of the first packed version cost 7 shared loads per output).
    for (int tk = warp; tk < F_TT; tk += F_THREADS / 32) {
      if (t0 + tk >= T) break;
      const float* zr = Zs + tk * 3 * PJ;
      float ss = 0.f;
      float* g = G + (long long)(t0 + tk) * GP_K;
#pragma unroll
      for (int n = 0; n < GCH_PAD / 32; ++n) {
        const unsigned code = chk[n * 32 + lane];
        if (code == 0xFFFFu) continue;
        const int i = code >> 8, jq = code & 255;
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const float zi = zr[r * PJ + i];
          const float4 zj = *reinterpret_cast<const float4*>(zr + r * PJ + jq * 4);
          o.x = fmaf(zi, zj.x, o.x); o.y = fmaf(zi, zj.y, o.y); o.z = fmaf(zi, zj.z, o.z); o.w = fmaf(zi, zj.w, o.w);
        }
        const int j0 = jq * 4;
        // the chunk's valid entries (j >= i) are contiguous in the packed order: a row of a 4x4 block (layout.h)
        float* gr = g + tri_index(i, max(i, j0)) - max(i - j0, 0);
        const float ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (j0 + k >= i) {
            gr[k] = ov[k];
            ss = fmaf(j0 + k == i ? ov[k] : 2.f * ov[k], ov[k], ss);     // ||G||_F^2 over the full symmetric matrix
          }
        }
      }
      if (lane < 16) {     // zero padding slots of the packed layout: 30, 31 of k-blocks 14 and 15, 20..31 of k-block 16
        const int pz = lane < 2 ? GP_OFF + 30 + lane : lane < 4 ? GP_OFF + 62 + (lane - 2) : GP_OFF + 84 + (lane - 4);
        g[pz] = 0.f;
      }
      ss = warp_sum(ss);
      if (lane == 0) Fn[t0 + tk] = sqrtf(ss) + 1.0f;
    }
  }
}

// ---- tiny-batch variant: one warp per token, no block-level barrier ---------------------------------------------
// For the 9..128 tokens of an acting forward (Agent.select_action) the tiled kernel above is one or two CTAs walking
// block-wide phases.  Here lane = output channel: the token's X row sits in the warp's slice of shared memory (128-bit
// broadcast loads), each lane streams its own row of P from L1/L2, keeps Z in registers, and the Gram column j is formed
// from shuffled z_i.  Measured: select_action 416 -> 393 us.  NOT a win at 2 304 tokens (20.5 us per launch like the tiled
// kernel, and the update slowed from 5.38 to 5.79 ms: 2 304 warps each streaming 16 KB of P rows, uncoalesced), so it is
// used for T <= 128 only.
template <int CE, int NPROJ>
__global__ void __launch_bounds__(256) inv_feature_small_fwd_kernel(
    const float* __restrict__ Xg, long long zsXg, const float* __restrict__ V0, long long zsV0,
    const float* __restrict__ gd, long long zsGd,
    const float* __restrict__ P1, const float* __restrict__ P2, long long zsP,
    float* __restrict__ Z, float* __restrict__ Z2, float* __restrict__ G, float* __restrict__ Fn, long long zsAct,
    int T) {
  SGRL_PDL_ENTER();
  constexpr int C = 128 + CE;
  __shared__ __align__(16) float Xw[8][3 * C];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, z = blockIdx.y;
  Xg += z * zsXg; gd += z * zsGd; P1 += z * zsP;
  if (CE) V0 += z * zsV0;
  if (NPROJ == 2) P2 += z * zsP;
  Z += z * zsAct; G += z * zsAct; Fn += z * zsAct;
  if (NPROJ == 2) Z2 += z * zsAct;
  const int t = blockIdx.x * 8 + warp;
  if (t >= T) return;                          // warp-uniform; nothing below synchronises across warps
  float* xw = Xw[warp];
  for (int i = lane; i < 96; i += 32) {
    const int r = i >> 5, c4 = (i & 31) * 4;
    *reinterpret_cast<float4*>(&xw[r * C + CE + c4]) = ldg4(Xg + ((long long)t * 3 + r) * 128 + c4);
  }
  if (CE && lane < 24) xw[(lane >> 3) * C + (lane & 7)] = __ldg(V0 + (long long)t * 24 + lane);
  __syncwarp();
  const int j = lane;
  const bool learned = j < 30;                 // channels 30, 31 are [gravity, direction]
  const float* p1 = P1 + (learned ? j : 0) * C;
  const float* p2 = NPROJ == 2 ? P2 + (learned ? j : 0) * C : nullptr;
  float z1[3] = {0.f, 0.f, 0.f}, z2[3] = {0.f, 0.f, 0.f};
#pragma unroll 2
  for (int c = 0; c < C; c += 4) {
    const float4 pa = ldg4(p1 + c);
    float4 pb = make_float4(0.f, 0.f, 0.f, 0.f);
    if (NPROJ == 2) pb = ldg4(p2 + c);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const float4 x = *reinterpret_cast<const float4*>(&xw[r * C + c]);
      z1[r] = fmaf(x.x, pa.x, fmaf(x.y, pa.y, fmaf(x.z, pa.z, fmaf(x.w, pa.w, z1[r]))));
      if (NPROJ == 2) z2[r] = fmaf(x.x, pb.x, fmaf(x.y, pb.y, fmaf(x.z, pb.z, fmaf(x.w, pb.w, z2[r]))));
    }
  }
  if (!learned) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      z1[r] = __ldg(gd + (long long)t * 6 + r * 2 + (j - 30));
      z2[r] = z1[r];
    }
  }
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    Z[((long long)t * 3 + r) * 32 + j] = z1[r];
    if (NPROJ == 2) Z2[((long long)t * 3 + r) * 32 + j] = z2[r];
  }
  float ss = 0.f;
  float* g = G + (long long)t * GP_K;
#pragma unroll 4
  for (int i = 0; i < CH; ++i) {
    const float a0 = __shfl_sync(0xffffffffu, z1[0], i), a1 = __shfl_sync(0xffffffffu, z1[1], i), a2 = __shfl_sync(0xffffffffu, z1[2], i);
    float o = a0 * z1[0];
    o = fmaf(a1, z1[1], o);
    o = fmaf(a2, z1[2], o);
    if (j >= i) {
      g[tri_index(i, j)] = o;
      ss = fmaf(j == i ? o : 2.f * o, o, ss);
    }
  }
  if (lane < 16) {
    const int pz = lane < 2 ? GP_OFF + 30 + lane : lane < 4 ? GP_OFF + 62 + (lane - 2) : GP_OFF + 84 + (lane - 4);
    g[pz] = 0.f;
  }
  ss = warp_sum(ss);
  if (lane == 0) Fn[t] = sqrtf(ss) + 1.0f;
}

struct FeatFwdP {
  const float* Xg; long long zsXg; const float* V0; long long zsV0; const float* gd; long long zsGd;
  const float* P1; const float* P2; long long zsP;
  float* Z; float* Z2; float* G; float* Fn; long long zsAct;
  int T; int nb; int head;   // head=1: X = [V0 | Xg] (C=136)
};

template <int CE, int NPROJ>
inline int inv_feature_fwd_launch(const FeatFwdP& p, cudaStream_t st) {
  using S = FeatSmem<CE, NPROJ>;
  auto kern = inv_feature_fwd_kernel<CE, NPROJ>;
  static bool attr_done = false;
  if (!attr_done) {
    SGRL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::bytes));
    attr_done = true;
  }
  const int ntiles = ceil_div(p.T, F_TT);
  if (p.T <= 128) {      // a handful of graphs (acting): one warp per token (see inv_feature_small_fwd_kernel)
    prof_begin(PC_FEATURE, (double)p.T * p.nb * (12.0 * S::C + 24 + 4.0 * GP_K + 4 + 384.0 * NPROJ), st);
    launch_k(inv_feature_small_fwd_kernel<CE, NPROJ>, dim3(ceil_div(p.T, 8), p.nb), 256, 0, st, p.Xg, p.zsXg, p.V0, p.zsV0, p.gd, p.zsGd,
             p.P1, p.P2, p.zsP, p.Z, p.Z2, p.G, p.Fn, p.zsAct, p.T);
    prof_end(st);
    SGRL_LAUNCH_OK();
    return 0;
  }
  const int per_sm = (int)((227 * 1024) / (S::bytes + 1024)) < 4 ? (int)((227 * 1024) / (S::bytes + 1024)) : 4;
  const int gx = ntiles < per_sm * NUM_SMS ? ntiles : per_sm * NUM_SMS;
  // algorithmic bytes per token: read X (12*C) + gd (24), write G (4*GP_K = 2176: packed triangle) + F (4) + Z (384 per projection)
  prof_begin(PC_FEATURE, (double)p.T * p.nb * (12.0 * S::C + 24 + 4.0 * GP_K + 4 + 384.0 * NPROJ), st);
  launch_k(kern, dim3(gx, p.nb), F_THREADS, S::bytes, st, p.Xg, p.zsXg, p.V0, p.zsV0, p.gd, p.zsGd, p.P1, p.P2, p.zsP,
                                                   p.Z, p.Z2, p.G, p.Fn, p.zsAct, p.T);
  prof_end(st);
  SGRL_LAUNCH_OK();
  return 0;
}

inline int inv_feature_fwd(const FeatFwdP& p, cudaStream_t st) {
  if (p.T <= 0) return 0;
  const bool two = p.P2 != nullptr;
  if (p.head) return two ? inv_feature_fwd_launch<8, 2>(p, st) : inv_feature_fwd_launch<8, 1>(p, st);
  return two ? inv_feature_fwd_launch<0, 2>(p, st) : inv_feature_fwd_launch<0, 1>(p, st);
}

// ---- backward ------------------------------------------------------------------------
// Inputs: dGp (T,GP_K) gradient w.r.t. the packed triangle from the consumer GEMM (against the folded weights, so
// dGp[p(i,j)] = dL/dG_ij + dL/dG_ji for i<j and dL/dG_ii on the diagonal), dF (T) accumulated gradient w.r.t. F from
// every division by F, Z (T,3,32), F (T).
//   S      = dG + dG^T + 2 dF G / (F-1)   (G recomputed from Z; F-1 = ||G||_F, 0 -> subgradient 0)
//   dZ     = Z S                          (T,3,32); columns 30,31 (inputs) are ignored downstream
__global__ void __launch_bounds__(256) inv_feature_bwd_kernel(
    const float* __restrict__ dG, const float* __restrict__ dF, const float* __restrict__ Z,
    const float* __restrict__ Fn, float* __restrict__ dZ, long long zsAct, long long zsWs, int T) {
  SGRL_PDL_ENTER();
  __shared__ float Sg[8][GP_K];
  __shared__ float Zw[8][3][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, z = blockIdx.y;
  dG += z * zsWs; dF += z * zsWs; dZ += z * zsWs; Z += z * zsAct; Fn += z * zsAct;
  for (int t = blockIdx.x * 8 + warp; t < T; t += gridDim.x * 8) {
    __syncwarp();
#pragma unroll
    for (int r = 0; r < 3; ++r) Zw[warp][r][lane] = Z[(long long)t * 96 + r * 32 + lane];
    const float* dg = dG + (long long)t * GP_K;
#pragma unroll
    for (int n = 0; n < GP_K / 32; ++n) Sg[warp][n * 32 + lane] = __ldg(dg + n * 32 + lane);
    const float nrm = Fn[t] - 1.0f;
    const float coef = nrm > 0.f ? dF[t] / nrm : 0.f;
    __syncwarp();
    const float zj0 = Zw[warp][0][lane], zj1 = Zw[warp][1][lane], zj2 = Zw[warp][2][lane];
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 4
    for (int i = 0; i < 32; ++i) {
      const float zi0 = Zw[warp][0][i], zi1 = Zw[warp][1][i], zi2 = Zw[warp][2][i];
      const float g = zi0 * zj0 + zi1 * zj1 + zi2 * zj2;
      const int lo = min(i, lane), hi = max(i, lane);
      const float d = Sg[warp][tri_index(lo, hi)];
      const float s = (i == lane) ? 2.f * (d + coef * g) : d + 2.f * coef * g;
      a0 = fmaf(zi0, s, a0); a1 = fmaf(zi1, s, a1); a2 = fmaf(zi2, s, a2);
    }
    float* o = dZ + (long long)t * 96;
    o[lane] = a0; o[32 + lane] = a1; o[64 + lane] = a2;
  }
}

inline int inv_feature_bwd(const float* dG, const float* dF, const float* Z, const float* Fn, float* dZ,
                           long long zsAct, long long zsWs, int T, int nb, cudaStream_t st) {
  if (T <= 0) return 0;
  int gx = ceil_div(T, 8);
  if (gx > 8 * NUM_SMS) gx = 8 * NUM_SMS;
  launch_k(inv_feature_bwd_kernel, dim3(gx, nb), 256, 0, st, dG, dF, Z, Fn, dZ, zsAct, zsWs, T);
  SGRL_LAUNCH_OK();
  return 0;
}

// ---- triangle fold of the vec(G) consumers (layout.h) -----------------------------------------------------------
struct FoldDesc {
  long long src[2 * MAX_LAYERS + 1];   // offset of the (rows,1024) weight inside the parameter / gradient arena
  long long dst[2 * MAX_LAYERS + 1];   // offset of the (rows,GP_K) folded matrix inside a fold plane
  int rows[2 * MAX_LAYERS + 1];
  int n;
};

// W'[o][p(i,j)] = W[o][32i+j] + W[o][32j+i] (i<j) | W[o][33i]; planes: fp32, and (with_split) tf32 hi / lo for the tcgen05 path
__global__ void __launch_bounds__(256) fold_sym_kernel(const float* __restrict__ params, long long zsP, float* __restrict__ wf, long long zsS,
                                                       long long plane, int with_split, FoldDesc d) {
  SGRL_PDL_ENTER();
  __shared__ unsigned short tri[GP_K];
  for (int i = threadIdx.x; i < GP_K; i += 256) tri[i] = c_tri.v[i];
  __syncthreads();
  const int m = blockIdx.y, z = blockIdx.z;
  const float* W = params + z * zsP + d.src[m];
  float* o0 = wf + z * zsS + d.dst[m];
  const int total = d.rows[m] * GP_K;
  for (int idx = blockIdx.x * 256 + threadIdx.x; idx < total; idx += gridDim.x * 256) {
    const int o = idx / GP_K, p = idx - o * GP_K;
    const unsigned code = tri[p];
    float v = 0.f;
    if (code != 0xFFFFu) {
      const int i = code >> 8, j = code & 255;
      const float* w = W + (long long)o * (CH * CH);
      v = __ldg(w + i * CH + j);
      if (i != j) v += __ldg(w + j * CH + i);
    }
    o0[idx] = v;
    if (with_split) {
      const unsigned hb = (__float_as_uint(v) + 0x1000u) & 0xFFFFE000u;
      const float h = __uint_as_float(hb);
      o0[plane + idx] = h;
      o0[2 * plane + idx] = __uint_as_float((__float_as_uint(v - h) + 0x1000u) & 0xFFFFE000u);
    }
  }
}

// gradient of the fold: dW[o][32a+b] += dW'[o][p(min(a,b), max(a,b))]  (G symmetric: both orderings get the same value).
// One thread per element of the (rows,1024) gradient: coalesced read-modify-write, the triangle is gathered (L2-resident).
__global__ void __launch_bounds__(256) unfold_sym_kernel(const float* __restrict__ gf, long long zsW, float* __restrict__ grads, long long zsG, FoldDesc d) {
  SGRL_PDL_ENTER();
  const int m = blockIdx.y, z = blockIdx.z;
  const float* src = gf + z * zsW + d.dst[m];
  float* G = grads + z * zsG + d.src[m];
  const int total = d.rows[m] * (CH * CH);
  for (int idx = blockIdx.x * 256 + threadIdx.x; idx < total; idx += gridDim.x * 256) {
    const int o = idx >> 10, a = (idx >> 5) & 31, b = idx & 31;
    const int lo = min(a, b), hi = max(a, b);
    G[idx] += __ldg(src + (long long)o * GP_K + tri_index(lo, hi));
  }
}

// host launchers of the two (network passes and sgrl_fold_sym / sgrl_unfold_sym; grid nullable, as misc.cuh's)
inline int fold_sym_launch(const float* params, long long zsP, float* wf, long long zsS, long long plane, int with_split, const FoldDesc& d, int nb,
                           cudaStream_t st, int* grid = nullptr) {
  const dim3 g(48, d.n, nb);
  launch_k(fold_sym_kernel, g, 256, 0, st, params, zsP, wf, zsS, plane, with_split, d);
  return launched(g, grid);
}
inline int unfold_sym_launch(const float* gf, long long zsW, float* grads, long long zsG, const FoldDesc& d, int nb, cudaStream_t st,
                             int* grid = nullptr) {
  const dim3 g(64, d.n, nb);
  launch_k(unfold_sym_kernel, g, 256, 0, st, gf, zsW, grads, zsG, d);
  return launched(g, grid);
}

}  // namespace sgrl
