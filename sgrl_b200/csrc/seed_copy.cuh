// Seed copy of a seed-batched agent (SeedBatchedAgent.exploit, population-based training): for every pair p, the nets of seed
// src[p] overwrite those of seed dst[p] in every per-seed state array (plane) of the agent, in one launch.
//
// A plane holds nets of n_net floats, net z at base + z * n_net, and seed k of K owns the nets k + j*K (j < nets_per_seed).
// One (pair, plane, net of the seed) is one segment: a contiguous run of n_net floats read from src's net and written to dst's.
// The work is cut into tiles of SEED_COPY_TILE float4s that never straddle two segments; block b copies tiles b, b + grid, ...
// and finds a tile's segment from the per-plane tile counts (division for the pair and the net, a binary search over the
// planes).  Each thread keeps SEED_COPY_U independent 16-byte loads in flight.  HBM-bound: 8 bytes moved per copied float.
// The plane descriptors and the pairs travel by value as a kernel parameter (about 1.2 KB).
#pragma once
#include "common.cuh"

namespace sgrl {

#define SGRL_SEED_COPY_MAX_PLANES 32
#define SGRL_SEED_COPY_MAX_PAIRS 7
constexpr int SEED_COPY_U = 4;
constexpr int SEED_COPY_TILE = 256 * SEED_COPY_U;

struct SeedCopyArgs {
  float* base[SGRL_SEED_COPY_MAX_PLANES];
  long long n4[SGRL_SEED_COPY_MAX_PLANES];           // float4s per net
  long long tpn[SGRL_SEED_COPY_MAX_PLANES];          // tiles per net
  long long tile0[SGRL_SEED_COPY_MAX_PLANES + 1];    // first tile of plane i within one pair's tiles; tile0[n_planes] = tiles per pair
  int dst[SGRL_SEED_COPY_MAX_PAIRS], src[SGRL_SEED_COPY_MAX_PAIRS];
  int n_planes, K;
  long long tiles;                                   // of all pairs
};

// No seed is both a dst and a src (checked on the host), so no tile reads what another tile writes.
__global__ void __launch_bounds__(256) seed_copy_kernel(const __grid_constant__ SeedCopyArgs a) {
  SGRL_PDL_ENTER();
  const long long per_pair = a.tile0[a.n_planes];      // tiles of one pair
  for (long long t = blockIdx.x; t < a.tiles; t += gridDim.x) {
    const int p = (int)(t / per_pair);
    long long r = t - p * per_pair;
    int lo = 0, hi = a.n_planes - 1;                 // the plane of tile r: the last one with tile0 <= r (no plane is empty)
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (a.tile0[mid] <= r) lo = mid; else hi = mid - 1;
    }
    r -= a.tile0[lo];
    const long long tpn = a.tpn[lo], n4 = a.n4[lo];
    const int j = (int)(r / tpn);
    const long long e0 = (r - j * tpn) * SEED_COPY_TILE + threadIdx.x;
    const float4* s = reinterpret_cast<const float4*>(a.base[lo]) + (long long)(j * a.K + a.src[p]) * n4;
    float4* d = reinterpret_cast<float4*>(a.base[lo]) + (long long)(j * a.K + a.dst[p]) * n4;
    float4 v[SEED_COPY_U];
#pragma unroll
    for (int u = 0; u < SEED_COPY_U; ++u)
      if (e0 + u * 256 < n4) v[u] = __ldcs(s + e0 + u * 256);
#pragma unroll
    for (int u = 0; u < SEED_COPY_U; ++u)
      if (e0 + u * 256 < n4) __stcs(d + e0 + u * 256, v[u]);
  }
}

// a: base, n4, n_planes, K, dst and src filled and checked by the caller (nps[i]: nets per seed of plane i, n_pairs entries of
// dst / src); the tile table is filled here.
inline int seed_copy(SeedCopyArgs& a, const int* nps, int n_pairs, cudaStream_t st) {
  long long t = 0, f4 = 0;
  for (int i = 0; i < a.n_planes; ++i) {
    a.tpn[i] = (a.n4[i] + SEED_COPY_TILE - 1) / SEED_COPY_TILE;
    a.tile0[i] = t;
    t += nps[i] * a.tpn[i];
    f4 += nps[i] * a.n4[i];
  }
  a.tile0[a.n_planes] = t;
  a.tiles = t * n_pairs;
  long long grid = a.tiles < 8LL * NUM_SMS ? a.tiles : 8LL * NUM_SMS;
  prof_begin(PC_OTHER, 32.0 * f4 * n_pairs, st);      // bytes: 16 read + 16 written per float4
  launch_k(seed_copy_kernel, (int)grid, 256, 0, st, a);
  prof_end(st);
  SGRL_LAUNCH_OK();
  return 0;
}

}  // namespace sgrl
