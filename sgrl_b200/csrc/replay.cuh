// K7 — device-resident replay storage (src/common/buffer.py:35-126; SURVEY.md §8f rank 2).
//
// The reference keeps five numpy arrays on the host and, per TD3 update, fancy-indexes each
// of them and pushes five tensors through pageable H2D copies (buffer.py:103-120).  Here
// one transition is ONE packed row in HBM,
//     row = [ obs (od) | action (ad) | next_obs (od) | reward | done ],   rw = 2*od + ad + 2
// so sampling is a single gather: one warp per sampled row streams the row's 4*rw
// contiguous bytes and scatters them into the five batch tensors (which may be the static
// input buffers of Agent.update's plan).  HBM-bound: 8*rw bytes per sampled row.
#pragma once
#include "common.cuh"

namespace sgrl {

struct ReplayOut {
  float* obs; float* act; float* nobs; float* rew; float* done;
};

// Up to SGRL_REPLAY_MAX_PARTS buffers gathered by one launch (Agent.update_packed_from_buffers: one buffer per morphology).
// Part p owns the batch rows [g0, g0 + B_p) of the launch; its samples are written contiguously from float obs0 of obs /
// next_obs and act0 of action, so part after part the outputs are the packed token layout of a mixed-morphology update
// (obs0 = 41 * first token of the part).  The descriptors travel by value as a kernel parameter (64 x 56 B).
#define SGRL_REPLAY_MAX_PARTS 64
struct ReplayPart {
  const float* rows; long long rw, cap, obs0, act0;
  int od, ad, g0, pad_;
};
struct ReplayParts {
  ReplayPart p[SGRL_REPLAY_MAX_PARTS];
  int n, G;        // parts, batch rows of all parts
};

// idx (G) int64 row numbers, part after part.  Rows are 4-byte aligned only (rw is odd for most morphologies), so the copy is
// scalar but fully coalesced: lane k reads float k, k+32, ...
__global__ void __launch_bounds__(256) replay_gather_kernel(const __grid_constant__ ReplayParts P, const long long* __restrict__ idx,
                                                            ReplayOut o) {
  SGRL_PDL_ENTER();
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int b = blockIdx.x * wpb + (threadIdx.x >> 5); b < P.G; b += gridDim.x * wpb) {
    int lo = 0, hi = P.n - 1;                  // the part of row b: the last one with g0 <= b (empty parts share their g0)
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (P.p[mid].g0 <= b) lo = mid; else hi = mid - 1;
    }
    const ReplayPart& q = P.p[lo];
    const long long cap = q.cap, j = b - q.g0;
    const int od = q.od, ad = q.ad;
    long long r = idx[b];
    if (r < 0) r += cap;                       // numpy negative indexing
    if (r < 0 || r >= cap) r = 0;              // host validated the indices; never read out of bounds
    const float* src = q.rows + r * q.rw;
    float* d0 = o.obs + q.obs0 + j * od;
    float* d1 = o.act + q.act0 + j * ad;
    float* d2 = o.nobs + q.obs0 + j * od;
    const int e1 = od, e2 = od + ad, e3 = 2 * od + ad;
    for (int k = lane; k < e3 + 2; k += 32) {
      const float v = __ldg(src + k);
      if (k < e1) d0[k] = v;
      else if (k < e2) d1[k - e1] = v;
      else if (k < e3) d2[k - e2] = v;
      else if (k == e3) o.rew[b] = v;
      else o.done[b] = v;
    }
  }
}

// rows[dst[i]] = staged[i] for i < n: flush of device-side transitions (vectorised envs that
// already live on the GPU); host-side add_transition goes through plain contiguous copies.
__global__ void __launch_bounds__(256) replay_scatter_kernel(float* __restrict__ rows, long long rw, const long long* __restrict__ dst,
                                                             const float* __restrict__ staged, int n, long long cap) {
  SGRL_PDL_ENTER();
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int i = blockIdx.x * wpb + (threadIdx.x >> 5); i < n; i += gridDim.x * wpb) {
    const long long r = dst[i];
    if (r < 0 || r >= cap) continue;
    float* d = rows + r * rw;
    const float* s = staged + (long long)i * rw;
    for (int k = lane; k < rw; k += 32) d[k] = __ldg(s + k);
  }
}

// P.p[i].g0 / obs0 / act0 and P.G are filled in here from the parts' batch sizes (B[i]) in order.
inline int replay_gather(ReplayParts& P, const int* B, const long long* idx, const ReplayOut& o, cudaStream_t st) {
  long long obs0 = 0, act0 = 0, G = 0;
  double bytes = 0;
  for (int i = 0; i < P.n; ++i) {
    ReplayPart& q = P.p[i];
    q.g0 = (int)G; q.obs0 = obs0; q.act0 = act0; q.pad_ = 0;
    G += B[i]; obs0 += (long long)B[i] * q.od; act0 += (long long)B[i] * q.ad;
    bytes += 8.0 * q.rw * B[i];
  }
  if (G > 0x7fffffff) return fail(-2, "more than 2^31 - 1 sampled rows", __FILE__, __LINE__);
  P.G = (int)G;
  if (G == 0) return 0;
  int gx = ceil_div(P.G, 8); if (gx > 8 * NUM_SMS) gx = 8 * NUM_SMS;
  prof_begin(PC_OTHER, bytes, st);
  launch_k(replay_gather_kernel, gx, 256, 0, st, P, idx, o);
  prof_end(st);
  SGRL_LAUNCH_OK();
  return 0;
}

inline int replay_scatter(float* rows, long long rw, const long long* dst, const float* staged, int n, long long cap, cudaStream_t st) {
  if (n <= 0) return 0;
  int gx = ceil_div(n, 8); if (gx > 8 * NUM_SMS) gx = 8 * NUM_SMS;
  launch_k(replay_scatter_kernel, gx, 256, 0, st, rows, rw, dst, staged, n, cap);
  SGRL_LAUNCH_OK();
  return 0;
}

}  // namespace sgrl
