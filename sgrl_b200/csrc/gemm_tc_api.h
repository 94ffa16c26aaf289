// Entry points of the tcgen05 GEMM translation unit (gemm_tc.cu: gemm_tc.cuh + gemm_tc_persist.cuh).
// The tensor-core kernels are compiled on their own: their code generation (22 instantiations of 160–260 KB each) must not
// move when an unrelated kernel of the library changes.  Measured: built in ONE translation unit with nvcc -split-compile, the
// same gemm_tc.cuh came out as 260 KB or 298 KB per kernel depending on what else was in the module, and the B=256 update ran
// 4.41 or 4.96 ms (profiles/r05p_ln_rowdiv.txt, r05q_timeline_ln.txt: every GEMM launch ~15 % slower, nothing else changed;
// DESIGN.md section 5 "Code generation is part of the measurement").
#pragma once
#include "gemm_simt.cuh"

namespace sgrl {
constexpr int TC_MAXG = 4;      // problems per grouped launch
// shape / alignment / epilogue combination the tcgen05 path can run
bool gemm_tc_eligible(const GemmP& p);
// one problem: tile width, split-K, kernel variant and tensor maps are chosen here
int gemm_tc(const GemmP& p, cudaStream_t st);
// 1..4 independent problems in ONE launch when their kernel variants agree, otherwise one launch each on the same stream
int gemm_tc_group(const GemmP* ps, int n, cudaStream_t st);

// Kernel tests (sgrl_gemm_desc): planner overrides, -1 = the cost model / knobs.  An override the problem cannot take is an error.
struct TcForce { int bn = -1, split = -1, csk = -1, sm2 = -1, persist = -1, tma_store = -1, group = -1; };
// what was launched for one problem (the fields of SgrlGemmPlan, include/sgrl_b200.h)
struct TcPlanInfo { int path, bn, amn, bmn, bpre, sm2, gram, persist, split, sk_x, cluster, tma_c, epi; };
// gemm_tc / gemm_tc_group with overrides and a report (info: 1 / n entries, nullable); every problem is planned before anything
// is enqueued
int gemm_tc_ex(const GemmP& p, const TcForce& f, TcPlanInfo* info, cudaStream_t st);
int gemm_tc_group_ex(const GemmP* ps, int n, const TcForce& f, TcPlanInfo* info, int* launches, cudaStream_t st);

// The epilogue class the tile kernel specialises on (all warp-uniform): 0 plain, 1 /F (+column scale), 2 relu-mask,
// 3 residuals, 4 accumulate, 5 split-K atomics, 6 anything else, 7 [X P^T | gd].  csk: this CTA reduces a cluster split-K
// tile; vec: C / mask / residual rows allow float4 access (GemmP::vecE).  Shared by the kernel and the plan report.
__host__ __device__ __forceinline__ int tc_epi_class(const GemmP& p, bool csk, bool vec) {
  const bool lin = !p.rowdiv && !p.mask && !p.res1 && !p.res2 && p.colscale_n == 0;
  if (p.gdcols) return (lin && !p.accumulate && !p.bias && !p.relu && p.splitk == 1 && vec && p.N == 32) ? 7 : 6;
  if (p.splitk > 1 && !csk) return 5;
  if (p.accumulate) return (lin && !p.relu && !p.bias) ? 4 : 6;
  if (lin) return 0;
  if (p.rowdiv && !p.mask && !p.res1 && !p.res2) return 1;
  if (p.mask && !p.rowdiv && !p.res1 && !p.res2 && p.colscale_n == 0 && !p.relu && !p.bias) return 2;
  if (p.res1 && !p.rowdiv && !p.mask && p.colscale_n == 0 && !p.relu && !p.bias) return 3;
  return 6;
}
}  // namespace sgrl
