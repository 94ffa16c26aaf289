// Shared device/host helpers for the sgrl_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cstdlib>

namespace sgrl {

// ---- error plumbing: C-ABI calls return 0 or a negative code, message kept thread-local
extern thread_local char g_err[512];
inline int fail(int code, const char* what, const char* file, int line) {
  snprintf(g_err, sizeof(g_err), "%s (%s:%d)", what, file, line);
  return code;
}
#define SGRL_CHECK(cond, msg) do { if (!(cond)) return ::sgrl::fail(-2, msg, __FILE__, __LINE__); } while (0)
#define SGRL_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return ::sgrl::fail(-3, cudaGetErrorString(e__), __FILE__, __LINE__); } while (0)
extern long long g_launches;   // kernels launched by this library (bench.py's gpu_launches)
#define SGRL_LAUNCH_OK() do { ++::sgrl::g_launches; cudaError_t e__ = cudaPeekAtLastError(); if (e__ != cudaSuccess) return ::sgrl::fail(-4, cudaGetErrorString(e__), __FILE__, __LINE__); } while (0)
#define SGRL_TRY(call) do { int r__ = (call); if (r__ != 0) return r__; } while (0)

constexpr int NUM_SMS = 148;  // B200
// nets of one module call (SgrlNetCall.nb) and of one grouped optimizer pass: K seeds of twin critics are 2K nets.  Nothing
// else bounds nb: grids put it on gridDim.y / gridDim.z and the GEMM cost model, split-K and tensor maps take it as a count.
constexpr int MAX_NETS = 16;

// ---- launches: every kernel of the library is launched with programmatic dependent launch (PDL) allowed, and begins
// with SGRL_PDL_ENTER(): "my dependents may start launching" + "wait until the kernel before me has completed and its
// memory is visible".  A kernel's CTAs therefore get scheduled (and the tcgen05 GEMM runs its barrier/TMEM/tensor-map
// prologue) while its predecessor is still draining, instead of paying the ~3 us kernel-to-kernel launch gap after it.
// Nothing is read or written before the wait, so stream order semantics are unchanged.  The tcgen05 GEMM alone releases its
// dependents later, once its accumulators are complete (gemm_tc_kernel).
// ---- deterministic mode (SGRL_DETERMINISTIC=1 or sgrl_deterministic(1)): run-to-run bit-identical gradients.  The default
// backward sums in an order that depends on timing in three places: split-K weight-gradient GEMMs (fp32 atomics), small
// cross-CTA reductions (LayerNorm / positional / decoder / relative-bias weight gradients, the loss scalars) and the dF
// accumulators that kernels of concurrent lanes add into.  Deterministic mode removes all three: no split-K (and no cluster
// split-K), one CTA (or per-CTA partials summed in index order) for the small reductions, and no side lanes, so every
// address is added to in program order.  Slower (the weight-gradient GEMMs lose their parallelism over K); the forward was
// deterministic already (tools/determinism_probe.py).
extern int g_det;
inline bool det_enabled() {
  if (g_det < 0) { const char* e = getenv("SGRL_DETERMINISTIC"); g_det = e ? (atoi(e) != 0) : 0; }
  return g_det != 0;
}
#define SGRL_PDL_TRIGGER() asm volatile("griddepcontrol.launch_dependents;" ::: "memory")
#define SGRL_PDL_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")
#define SGRL_PDL_ENTER() do { SGRL_PDL_TRIGGER(); SGRL_PDL_WAIT(); } while (0)
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
// after a launch_k of the host launchers (misc.cuh, feature.cuh): count it, report its grid (grid nullable) and its launch error
inline int launched(dim3 g, int* grid) {
  if (grid) { grid[0] = (int)g.x; grid[1] = (int)g.y; grid[2] = (int)g.z; }
  SGRL_LAUNCH_OK();
  return 0;
}

// ---- optional per-kernel-class device timing (bench.py roofline pass): CUDA events around
// the launches of one class on the launching stream, collected after a synchronize.
enum ProfClass { PC_GEMM = 0, PC_GEMM_TC, PC_FEATURE, PC_ATTENTION, PC_OTHER, PC_COUNT };
struct Prof {
  bool on = false;
  static constexpr int CAP = 8192;
  cudaEvent_t ev[2 * CAP];
  int cls[CAP]; double work[CAP];
  int n = 0; bool made = false;
};
extern Prof g_prof;
inline void prof_begin(int cls, double work, cudaStream_t st) {
  Prof& p = g_prof;
  if (!p.on || p.n >= Prof::CAP) return;
  if (!p.made) { for (int i = 0; i < 2 * Prof::CAP; ++i) cudaEventCreate(&p.ev[i]); p.made = true; }
  p.cls[p.n] = cls; p.work[p.n] = work;
  cudaEventRecord(p.ev[2 * p.n], st);
}
inline void prof_end(cudaStream_t st) {
  Prof& p = g_prof;
  if (!p.on || p.n >= Prof::CAP) return;
  cudaEventRecord(p.ev[2 * p.n + 1], st);
  ++p.n;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void stg4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// 4 consecutive floats with one vector access when (pointer, leading dimension, z-stride) allow it.
// The decision is taken on the HOST and passed in as a kernel argument: when it is derived from the
// pointer bits inside the kernel nvcc folds the scalar path away and emits an unconditional 128-bit access.
inline int host_vec_ok(const void* p, long long ld, long long zs = 0) {
  return p != nullptr && ((reinterpret_cast<uintptr_t>(p) & 15u) == 0) && ((ld & 3) == 0) && ((zs & 3) == 0);
}
__device__ __forceinline__ float4 load4(const float* p, bool vec) {
  if (vec) return *reinterpret_cast<const float4*>(p);
  return make_float4(p[0], p[1], p[2], p[3]);
}
__device__ __forceinline__ void store4(float* p, float4 v, bool vec) {
  if (vec) { *reinterpret_cast<float4*>(p) = v; return; }
  p[0] = v.x; p[1] = v.y; p[2] = v.z; p[3] = v.w;
}

inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace sgrl
