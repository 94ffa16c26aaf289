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
}  // namespace sgrl
