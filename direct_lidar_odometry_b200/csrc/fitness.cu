// fitness.cu — pcl::Registration::getFitnessScore(max_range) for one or many (source, target, T) pairs in two launches.
//
// PCL (registration.hpp, getFitnessScore): transformPointCloud(*input_, T) in float, then per point
//   tree_->nearestKSearch(pt, 1) over the target;  if (nn_dists[0] <= max_range) { score += nn_dists[0]; ++nr; }
//   return nr > 0 ? score / nr : DBL_MAX
// The SQUARED float distance is compared with max_range as given (not with max_range^2), as a double, with <=.
//
// K1 fitness_chunks_kernel: one block per chunk of FITNESS_CHUNK consecutive source points of one pair.  Per point the
//    float transform in Eigen's operation order, the finite check (a non-finite point has a NaN distance in PCL and is
//    never counted), then the exact 1-NN of the registration kernels: the radius-1 cube by a group of LPP lanes, and the
//    queries it cannot settle finished by a warp (grid_search_warp resumed at radius 1), which also crosses empty space
//    when the search is unbounded.  The chunk's (sum, count) is reduced in a fixed order (lane butterfly, then warps).
// K2 fitness_finalize_kernel: one warp per pair sums that pair's chunk partials in chunk order and stores score and
//    count straight into mapped host memory.
// A pair's result depends only on its own points, target and T — not on the launch shape or on the other pairs — so a
// pair scored in a batch has the bits of the same pair scored alone.
#include <cmath>
#include "internal.h"
#include "grid_search.cuh"

namespace ngicp {

constexpr int FIT_THREADS = FITNESS_CHUNK;
constexpr int FIT_WARPS = FIT_THREADS / 32;

// same operation order as xform_row in align.cu and transform_points_kernel in api.cu (never fused)
__device__ __forceinline__ float fit_xform_row(const float* m, float x, float y, float z) {
  return __fadd_rn(__fadd_rn(__fmul_rn(m[0], x), __fmul_rn(m[1], y)), __fadd_rn(__fmul_rn(m[2], z), m[3]));
}

// queries the radius-1 cube could not settle, by chunk-local index; finished by whole warps (as in align.cu's
// linearize_block)
struct FitTailQueue {
  float qx[FIT_THREADS], qy[FIT_THREADS], qz[FIT_THREADS], d[FIT_THREADS];
  int p[FIT_THREADS];
  unsigned short list[FIT_THREADS];
  int n, next;
};

// nearest-neighbour squared distance of the chunk's points -> s_d[local] (NaN: past the end, non-finite, or nothing
// within the cap).  With LPP lanes per point the radius-1 cubes take LPP passes; the queries none of them settled are
// then finished together, by all warps of the block, so that one pass's far-field searches do not wait for the other's.
template <int LPP>
__device__ __forceinline__ void fitness_search(const FitnessPair& pr, const GridParams& gp, int i0, float cap_d2, FitTailQueue& tq, float* s_d) {
  const int lane = threadIdx.x & 31;
  const int sub = threadIdx.x & (LPP - 1), gi = threadIdx.x / LPP;
  const unsigned gmask = (LPP == 1) ? 0u : (((1u << LPP) - 1u) << (lane & ~(LPP - 1)));
  constexpr int PPP = FIT_THREADS / LPP;   // points per pass
  if (threadIdx.x == 0) { tq.n = 0; tq.next = 0; }
  __syncthreads();
#pragma unroll 1
  for (int pass = 0; pass < LPP; ++pass) {
    const int local = pass * PPP + gi;
    const int i = i0 + local;
    float best_d = FLT_MAX;
    int best_p = -1;
    if (i < pr.ns) {   // group-uniform, as is everything up to the queueing
      const float4 p = __ldg(pr.src + i);
      const float qx = fit_xform_row(pr.T + 0, p.x, p.y, p.z), qy = fit_xform_row(pr.T + 4, p.x, p.y, p.z),
                  qz = fit_xform_row(pr.T + 8, p.x, p.y, p.z);
      if (isfinite(qx) && isfinite(qy) && isfinite(qz)) {
        const bool more = grid_nn1_cube1_group<LPP>(pr.tgt, gp, sub, gmask, qx, qy, qz, cap_d2, best_d, best_p);
        if (more && sub == 0) {
          tq.qx[local] = qx; tq.qy[local] = qy; tq.qz[local] = qz; tq.d[local] = best_d; tq.p[local] = best_p;
          tq.list[atomicAdd(&tq.n, 1)] = (unsigned short)local;
        }
      }
    }
    if (sub == 0) s_d[local] = best_p >= 0 ? best_d : NAN;   // a queued point's entry is replaced below
  }
  __syncthreads();
  const int nq = tq.n;
  for (;;) {
    int e = 0;
    if (lane == 0) e = atomicAdd(&tq.next, 1);
    e = __shfl_sync(FULL, e, 0);
    if (e >= nq) break;
    const int s = tq.list[e];
    WarpBest1 rs;
    rs.d = tq.d[s]; rs.p = tq.p[s];
    grid_search_warp<WarpBest1, true, 4>(pr.tgt, gp, tq.qx[s], tq.qy[s], tq.qz[s], cap_d2, rs, false, 1);
    rs.finalize();
    if (lane == 0) s_d[s] = rs.p >= 0 ? rs.d : NAN;
  }
}

__global__ void __launch_bounds__(FIT_THREADS) fitness_chunks_kernel(const FitnessPair* __restrict__ pairs, int n_pairs, float cap_d2,
                                                                      double max_range, double2* __restrict__ partials) {
  __shared__ FitTailQueue s_tq;
  __shared__ float s_d[FIT_THREADS];
  __shared__ double s_sum[FIT_WARPS];
  __shared__ int s_cnt[FIT_WARPS];
  __shared__ int s_pair;
  const int c = blockIdx.x;
  if (threadIdx.x == 0) {   // the last pair whose first chunk is <= c (pairs without chunks share their successor's chunk0)
    int lo = 0, hi = n_pairs - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (pairs[mid].chunk0 <= c) lo = mid; else hi = mid - 1;
    }
    s_pair = lo;
  }
  __syncthreads();
  const FitnessPair& pr = pairs[s_pair];
  const GridParams gp = load_grid(pr.tgt.desc);
  const int i0 = (c - pr.chunk0) * FITNESS_CHUNK;
  if (pr.lpp == 2) fitness_search<2>(pr, gp, i0, cap_d2, s_tq, s_d);
  else fitness_search<1>(pr, gp, i0, cap_d2, s_tq, s_d);
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const float d = s_d[threadIdx.x];
  const bool in = (double)d <= max_range;   // PCL's test; NaN never passes
  const double s = warp_sum(in ? (double)d : 0.0);
  const int n = __popc(__ballot_sync(FULL, in));
  if (lane == 0) { s_sum[w] = s; s_cnt[w] = n; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double bs = 0.0;
    int bn = 0;
#pragma unroll
    for (int k = 0; k < FIT_WARPS; ++k) { bs += s_sum[k]; bn += s_cnt[k]; }
    partials[c] = make_double2(bs, (double)bn);
  }
}

__global__ void fitness_finalize_kernel(const FitnessPair* __restrict__ pairs, int n_pairs, const double2* __restrict__ partials,
                                        FitnessResult* __restrict__ out) {
  const int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (j >= n_pairs) return;   // warp-uniform
  const int c0 = pairs[j].chunk0, nc = pairs[j].nchunks;
  double s = 0.0, n = 0.0;
  for (int c = 0; c < nc; c += 32) {   // the warp loads 32 partials at once; every lane adds them in chunk order
    const double2 v = c + lane < nc ? partials[c0 + c + lane] : make_double2(0.0, 0.0);
    const int m = min(32, nc - c);
    for (int u = 0; u < m; ++u) {
      s += __shfl_sync(FULL, v.x, u);
      n += __shfl_sync(FULL, v.y, u);
    }
  }
  if (lane == 0) {
    FitnessResult r;
    r.score = n > 0.0 ? s / n : DBL_MAX;
    r.n = (unsigned long long)n;
    out[j] = r;
  }
}

// The search is capped at the smallest float above max_range (never below it, so the bounded search finds every point
// the exact double test can accept: same count and sum as PCL's unbounded search followed by the filter); unbounded
// from FLT_MAX on.
cudaError_t launch_fitness(const FitnessPair* pairs_dev, int n_pairs, int total_chunks, double max_range, double2* partials,
                           FitnessResult* out, cudaStream_t st) {
  float cap = FLT_MAX;
  if (max_range < (double)FLT_MAX) {
    cap = nextafterf((float)max_range, INFINITY);
    if (!(cap <= FLT_MAX)) cap = FLT_MAX;
  }
  if (total_chunks > 0) {
    fitness_chunks_kernel<<<total_chunks, FIT_THREADS, 0, st>>>(pairs_dev, n_pairs, cap, max_range, partials);
    note_launches(1);
  }
  fitness_finalize_kernel<<<(n_pairs + 3) / 4, 128, 0, st>>>(pairs_dev, n_pairs, partials, out);   // a warp per pair
  note_launches(1);
  return cudaGetLastError();
}

}  // namespace ngicp
