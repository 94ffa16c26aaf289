// Generic fp32 SIMT GEMM with fused epilogue.  Used for every contraction whose shape is
// too small or too ragged for the tcgen05 path (K = 8/17/20/30/32/145/148, N = 1/3/30)
// and, in round 1, for the backward contractions (dX = dY W, dW = dY^T X).
//
//   C[z][m][n] (op)= epi( alpha * sum_k A(m,k) * B(n,k) )
//   A(m,k) = transA ? A[k*lda+m] : A[m*lda+k]      B(n,k) = transB ? B[k*ldb+n] : B[n*ldb+k]
//
// so  Y = X W^T        -> transA=0, transB=0   (nn.Linear weight is (N,K) row-major)
//     dX = dY W        -> transA=0, transB=1
//     dW = dY^T X      -> transA=1, transB=1   (contraction over tokens; split-K + atomics)
#pragma once
#include "common.cuh"

namespace sgrl {

struct GemmP {
  const float* A; long long zsA; int lda; int transA;
  const float* B; long long zsB; int ldb; int transB;
  float* C; long long zsC; int ldc;
  int M, N, K;
  float alpha;
  const float* bias; long long zsBias;      // + bias[n]
  int relu;                                 // max(v,0)
  const float* rowdiv; long long zsRow;     // v / rowdiv[m]
  float colscale; int colscale_n;           // v * colscale for n < colscale_n
  const float* mask; long long zsMask; int ldmask;  // v = mask[m][n] > 0 ? v : 0
  const float* res1; long long zsR1; int ldr1;      // + res1[m][n]
  const float* res2; long long zsR2; int ldr2;      // + res2[m][n]
  int accumulate;                           // C += v instead of C = v
  int splitk;                               // >1: K may be split, partial sums atomically added into C (needs accumulate, no bias)
  int nb;                                   // instances (blockIdx.z)
  int vecA, vecB;                           // set by the launcher: operand rows may be fetched as float4
  const float* Bhi; const float* Blo;       // tcgen05 path only, optional: B pre-split into tf32 hi/lo parts (same layout/strides as B)
  int vecE;                                 // set by the tcgen05 launcher: C/mask/res rows allow float4 access
  int csk;                                  // tcgen05 path, set by the launcher: K is split over a (1, splitk, 1) cluster, rank 0 reduces through DSMEM
  int sm2_ok;                               // tcgen05 path: the single-accumulator two-CTAs-per-SM variant may be used (inference passes only)
  long long* dbg;                           // optional (tools/gemm_trace.py): SM-clock timestamps of one CTA's pipeline phases
  int dbg_cta;                              // which CTA (blockIdx.x) writes them (SGRL_TRACE_CTA, default 0)
  int tma_c;                                // tcgen05 path, set by the launcher: plain / rowdiv store epilogue leaves through a TMA tensor store (TcProblem::mapC)
  // ---- tcgen05 path only (gemm_tc.cuh) ----
  int prec;                                 // 0: 3xTF32 error-compensated (fp32 parity); 1: BF16-INPUT mode — both operands rounded (RN-even) to bf16 in
                                            //    the operand path, ONE tf32 MMA pass (bf16 values are exact in tf32), fp32 accumulate: numerically what
                                            //    kind::f16 bf16 x bf16 -> f32 computes.  Never the default; reported separately (north_star).
  int sk_x;                                 // set by the launcher: the split-K index is folded into blockIdx.x (grouped launches)
  // A operand generated on the fly: row m of A is the packed upper triangle (GP_K = 544 floats, layout.h) of G_m = Z_m^T Z_m,
  // Z_m (3 x 32) read from gramZ (T, 96).  K must be GP_K, transA = 0, splitk = 1.  Replaces the Gram phase of the
  // invariant-feature kernel and its 2.2 KB/token round trip (subequivariant_attentions.py:93-97, SEActor.py:96-101, 259-263).
  const float* gramZ; long long zsGramZ;
  float* gramF;                             // out (nullable): F_m = ||G_m||_F + 1     (z-stride zsGramZ)
  float* gramG;                             // out (nullable): the generated rows (T, GP_K), kept for the weight-gradient GEMM (z-stride zsGramZ)
  // epilogue: columns 30, 31 of row m (= 3 t + r) are REPLACED by gd[t][r][0..1] (gdcols (T, 3, 2)): Z = [X P^T | gd] with N = 32
  const float* gdcols; long long zsGd;
  float* rowsum; long long zsRowsum;        // optional: rowsum[m] += alpha * sum_k A(m,k)  (bias gradient of a weight-gradient GEMM, A = dY^T); tcgen05 path
                                            // fuses it into the operand conversion, elsewhere a column-sum kernel follows the GEMM (run_gemm, net.cuh)
};

inline GemmP gemm_defaults() {
  GemmP p;
  memset(&p, 0, sizeof(p));
  p.alpha = 1.f; p.colscale = 1.f; p.splitk = 1; p.nb = 1;
  return p;
}

#ifndef SGRL_TC_TU      // the SIMT kernels belong to the main translation unit; the tcgen05 units (gemm_tc.cu) only need GemmP
constexpr int GB_M = 64, GB_N = 64, GB_K = 16, G_THREADS = 256, G_PAD = 4;

__device__ __forceinline__ void gemm_fetch(float (&r)[4], const float* __restrict__ src, int ld, int trans,
                                           int r0, int k0, int rlim, int klim, bool vec, int tid) {
  if (!trans) {
    const int row = r0 + (tid >> 2), k = k0 + (tid & 3) * 4;
    if (row < rlim && vec && k + 3 < klim) {
      float4 v = ldg4(src + (long long)row * ld + k);
      r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) r[i] = (row < rlim && k + i < klim) ? __ldg(src + (long long)row * ld + k + i) : 0.f;
    }
  } else {
    const int k = k0 + (tid >> 4), row = r0 + (tid & 15) * 4;
    if (k < klim && vec && row + 3 < rlim) {
      float4 v = ldg4(src + (long long)k * ld + row);
      r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) r[i] = (k < klim && row + i < rlim) ? __ldg(src + (long long)k * ld + row + i) : 0.f;
    }
  }
}

__device__ __forceinline__ void gemm_stash(float (*s)[GB_M + G_PAD], const float (&r)[4], int trans, int tid) {
  if (!trans) {
    const int row = tid >> 2, k = (tid & 3) * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) s[k + i][row] = r[i];
  } else {
    const int k = tid >> 4, row = (tid & 15) * 4;
    *reinterpret_cast<float4*>(&s[k][row]) = make_float4(r[0], r[1], r[2], r[3]);
  }
}

__global__ void __launch_bounds__(G_THREADS) gemm_simt_kernel(GemmP p) {
  SGRL_PDL_ENTER();
  __shared__ __align__(16) float As[GB_K][GB_M + G_PAD];
  __shared__ __align__(16) float Bs[GB_K][GB_N + G_PAD];
  const int tid = threadIdx.x, z = blockIdx.z;
  const int tiles_n = (p.N + GB_N - 1) / GB_N;
  const int m0 = (blockIdx.x / tiles_n) * GB_M, n0 = (blockIdx.x % tiles_n) * GB_N;
  const float* A = p.A + z * p.zsA;
  const float* B = p.B + z * p.zsB;
  // K range of this split
  const int ktiles = (p.K + GB_K - 1) / GB_K;
  const int per = (ktiles + p.splitk - 1) / p.splitk;
  const int kt0 = blockIdx.y * per, kt1 = min(ktiles, kt0 + per);
  const bool vecA = p.vecA != 0, vecB = p.vecB != 0;
  const int tx = tid & 15, ty = tid >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  float ra[4], rb[4];
  if (kt0 < kt1) {
    gemm_fetch(ra, A, p.lda, p.transA, m0, kt0 * GB_K, p.M, p.K, vecA, tid);
    gemm_fetch(rb, B, p.ldb, p.transB, n0, kt0 * GB_K, p.N, p.K, vecB, tid);
    gemm_stash(As, ra, p.transA, tid);
    gemm_stash(Bs, rb, p.transB, tid);
  }
  __syncthreads();
  for (int kt = kt0; kt < kt1; ++kt) {
    const bool more = kt + 1 < kt1;
    if (more) {
      gemm_fetch(ra, A, p.lda, p.transA, m0, (kt + 1) * GB_K, p.M, p.K, vecA, tid);
      gemm_fetch(rb, B, p.ldb, p.transB, n0, (kt + 1) * GB_K, p.N, p.K, vecB, tid);
    }
#pragma unroll
    for (int k = 0; k < GB_K; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
    if (more) {
      gemm_stash(As, ra, p.transA, tid);
      gemm_stash(Bs, rb, p.transB, tid);
    }
    __syncthreads();
  }
  if (kt0 >= kt1 && p.splitk > 1) return;

  // ---- epilogue
  float* C = p.C + z * p.zsC;
  const float* bias = p.bias ? p.bias + z * p.zsBias : nullptr;
  const float* rowdiv = p.rowdiv ? p.rowdiv + z * p.zsRow : nullptr;
  const float* mask = p.mask ? p.mask + z * p.zsMask : nullptr;
  const float* res1 = p.res1 ? p.res1 + z * p.zsR1 : nullptr;
  const float* res2 = p.res2 ? p.res2 + z * p.zsR2 : nullptr;
  const bool first_split = blockIdx.y == 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= p.M) continue;
    const float rd = rowdiv ? rowdiv[m] : 1.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= p.N) continue;
      float v = p.alpha * acc[i][j];
      if (bias && first_split) v += bias[n];
      if (p.relu) v = fmaxf(v, 0.f);
      if (rowdiv) v = v / rd;
      if (n < p.colscale_n) v *= p.colscale;
      if (mask) v = mask[(long long)m * p.ldmask + n] > 0.f ? v : 0.f;
      if (res1) v += res1[(long long)m * p.ldr1 + n];
      if (res2) v += res2[(long long)m * p.ldr2 + n];
      float* c = C + (long long)m * p.ldc + n;
      if (p.splitk > 1) atomicAdd(c, v);
      else if (p.accumulate) *c += v;
      else *c = v;
    }
  }
}

// ---- skinny GEMM: C[M<=32, N] = epi(alpha * A[M,K] B[N,K]^T) — the projections of a B=1..3 rollout forward
// (Agent.select_action, src/agent.py:189-198: 9..27 token rows).  The 64x64-tile kernel above spends ~23 us per launch there
// (4-16 CTAs walking K in 16-wide steps with two barriers each: 75 % of a 0.87 ms select_action).  Here the whole A panel
// sits in shared memory, one warp owns one output column, lanes stride over K with 128-bit loads of the weight row
// (coalesced, each weight read exactly once per CTA) and the M partial sums are reduced with shuffles.  Weight-read bound.
constexpr int SK_MAXM = 32, SK_WARPS = 8;
constexpr size_t SK_MAX_SMEM = 160 * 1024;

__global__ void __launch_bounds__(32 * SK_WARPS) gemm_skinny_kernel(GemmP p) {
  SGRL_PDL_ENTER();
  extern __shared__ __align__(16) float sk_As[];          // [M][K]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, z = blockIdx.z;
  const float* A = p.A + z * p.zsA;
  const float* B = p.B + z * p.zsB;
  const int M = p.M, K4 = p.K >> 2;
  float4* As4 = reinterpret_cast<float4*>(sk_As);
  for (int i = tid; i < M * K4; i += 32 * SK_WARPS) {
    const int m = i / K4, k4 = i - m * K4;
    As4[i] = ldg4(A + (long long)m * p.lda + 4 * k4);
  }
  __syncthreads();
  float* C = p.C + z * p.zsC;
  const float* bias = p.bias ? p.bias + z * p.zsBias : nullptr;
  const float* rowdiv = p.rowdiv ? p.rowdiv + z * p.zsRow : nullptr;
  const float* res1 = p.res1 ? p.res1 + z * p.zsR1 : nullptr;
  const float* res2 = p.res2 ? p.res2 + z * p.zsR2 : nullptr;
  for (int n = blockIdx.x * SK_WARPS + warp; n < p.N; n += gridDim.x * SK_WARPS) {
    float acc[SK_MAXM];
#pragma unroll
    for (int m = 0; m < SK_MAXM; ++m) acc[m] = 0.f;
    const float4* brow = reinterpret_cast<const float4*>(B + (long long)n * p.ldb);
    for (int k4 = lane; k4 < K4; k4 += 32) {
      const float4 b = __ldg(brow + k4);
#pragma unroll
      for (int m = 0; m < SK_MAXM; ++m) {
        if (m < M) {
          const float4 a = As4[m * K4 + k4];
          acc[m] = fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, fmaf(a.w, b.w, acc[m]))));
        }
      }
    }
    float mine = 0.f;                                     // lane m keeps the total of row m
#pragma unroll
    for (int m = 0; m < SK_MAXM; ++m) {
      if (m < M) {
        const float t = warp_sum(acc[m]);
        if (lane == m) mine = t;
      }
    }
    if (lane < M) {
      const int m = lane;
      float v = p.alpha * mine;
      if (bias) v += bias[n];
      if (p.relu) v = fmaxf(v, 0.f);
      if (rowdiv) v = v / rowdiv[m];
      if (n < p.colscale_n) v *= p.colscale;
      if (res1) v += res1[(long long)m * p.ldr1 + n];
      if (res2) v += res2[(long long)m * p.ldr2 + n];
      C[(long long)m * p.ldc + n] = v;
    }
  }
}

inline bool gemm_skinny_eligible(const GemmP& p) {
  return p.M >= 1 && p.M <= SK_MAXM && !p.transA && !p.transB && !p.accumulate && p.splitk <= 1 && !p.mask && (p.K & 3) == 0 &&
         host_vec_ok(p.A, p.lda, p.zsA) && host_vec_ok(p.B, p.ldb, p.zsB) && (size_t)p.M * p.K * sizeof(float) <= SK_MAX_SMEM;
}

inline int gemm_skinny(const GemmP& p, cudaStream_t st) {
  static bool attr_done = false;
  if (!attr_done) {
    SGRL_CUDA(cudaFuncSetAttribute(gemm_skinny_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SK_MAX_SMEM));
    attr_done = true;
  }
  int gx = ceil_div(p.N, SK_WARPS); if (gx > 4 * NUM_SMS) gx = 4 * NUM_SMS;
  prof_begin(PC_GEMM, 2.0 * p.M * p.N * (double)p.K * p.nb, st);
  launch_k(gemm_skinny_kernel, dim3(gx, 1, p.nb), 32 * SK_WARPS, (size_t)p.M * p.K * sizeof(float), st, p);
  prof_end(st);
  SGRL_LAUNCH_OK();
  return 0;
}

inline int gemm_simt(const GemmP& p_in, cudaStream_t st) {
  GemmP p = p_in;
  p.vecA = host_vec_ok(p.A, p.lda, p.zsA);
  p.vecB = host_vec_ok(p.B, p.ldb, p.zsB);
  if (p.M <= 0 || p.N <= 0 || p.nb <= 0) return 0;
  SGRL_CHECK(p.K > 0, "gemm: K must be positive");
  SGRL_CHECK(p.splitk >= 1, "gemm: splitk");
  SGRL_CHECK(p.splitk == 1 || (!p.relu && !p.rowdiv && !p.mask && !p.res1 && !p.res2 && p.colscale_n == 0),
             "gemm: split-K only with a linear epilogue");
  SGRL_CHECK(p.splitk == 1 || (p.accumulate && !p.bias), "gemm: split-K needs accumulate = 1 and no bias");   // as the tcgen05 path
  if (gemm_skinny_eligible(p)) return gemm_skinny(p, st);
  const int tiles = ceil_div(p.M, GB_M) * ceil_div(p.N, GB_N);
  dim3 grid(tiles, p.splitk, p.nb);
  prof_begin(PC_GEMM, 2.0 * p.M * p.N * (double)p.K * p.nb, st);
  launch_k(gemm_simt_kernel, grid, G_THREADS, 0, st, p);
  prof_end(st);
  SGRL_LAUNCH_OK();
  return 0;
}

// choose a split-K factor for token-contraction GEMMs (dW): fill ~2 waves of the SMs
inline int pick_splitk(int M, int N, int K, int nb) {
  if (det_enabled()) return 1;          // deterministic mode: no fp32 atomics over K
  const int tiles = ceil_div(M, GB_M) * ceil_div(N, GB_N) * nb;
  const int ktiles = ceil_div(K, GB_K);
  int s = (2 * NUM_SMS + tiles - 1) / tiles;
  if (s > ktiles / 4) s = ktiles / 4;   // at least 4 k-tiles (64 tokens) per split
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  return s;
}

#endif

}  // namespace sgrl
