// align.cu — K4/K5 and the Levenberg-Marquardt driver.
//
// K4  linearize        = NanoGICP::update_correspondences + NanoGICP::linearize fused
//                        (reference include/nano_gicp/impl/nano_gicp_impl.hpp:173-211, :213-270):
//                        per source point (one thread, or a pair of lanes against large targets):
//                        q = float(T) * p  ->  bounded 1-NN on the target grid (3x3x3 cells row by row; searches that
//                        must go farther are finished warp-cooperatively from a shared-memory queue)  ->
//                        M = (C_B + R C_A R^T)^-1  ->  J^T M J / J^T M e / e^T M e, reduced with a transposed warp
//                        butterfly per pass and per-block partials into one packed {H(21), b(6), err} per call.
// K5  compute_error    = NanoGICP::compute_error (:272-296) with correspondences and M frozen.
// LM  align_fused      = LsqRegistration::computeTransformation / step_lm / step_gn / is_converged
//                        (include/nano_gicp/impl/lsq_registration_impl.hpp:89-208) as ONE persistent
//                        cooperative kernel: K4 and K5 phases separated by a grid barrier, the 6x6
//                        LDL^T solve and the accept/reject logic done redundantly by every block from the
//                        same fixed-order sum of partials (every block sums them itself on one GPU; with a
//                        sharded submap the last block sums and exchanges with the peers) — bit-deterministic,
//                        no host round trip: the result is stored straight into mapped host memory.
//
// Per source point K4 touches p_A 16 B + C_A 48 B + p_B 16 B + C_B 48 B + corr 4 B = 132 B of
// compulsory traffic (+48 B M +16 B p_B stored for K5, which then reads 16+48+16+4 = 84 B).
#include <cstdlib>
#include <cstring>
#include <cooperative_groups.h>
#include "internal.h"
#include "grid_search.cuh"
#include "gicp_math.cuh"

namespace ngicp {

constexpr int AL_THREADS = 256;
constexpr int AL_WARPS = AL_THREADS / 32;
constexpr int ALIGN_BATCH_CLUSTER = 8;   // blocks per pair in the batched kernel (portable cluster size)

struct XformF { float m[12]; };   // rows: m[r*4+c], c=3 is translation; float cast of the double state
struct AlignArgs {
  const float4* src_pts; const double* src_cov; int ns;
  GridView tgt; const double* tgt_cov;
  double* mahal; int* corr; float* sqd; float4* tgt_pt;
  double* partials;  // [max_blocks][NRED]
  int max_blocks;
  // sharded-submap mode: this handle only counts source points whose transformed position falls in
  // [slab_lo, slab_hi) along slab_axis (-1 = no filter); see direct_lidar_odometry_b200/sharded.py
  int slab_axis;
  float slab_lo, slab_hi;
};

__device__ __forceinline__ void make_xforms(const Iso3& x, XformF& f) {
#pragma unroll
  for (int r = 0; r < 3; r++) {
#pragma unroll
    for (int c = 0; c < 3; c++) f.m[r * 4 + c] = (float)x.R[r * 3 + c];
    f.m[r * 4 + 3] = (float)x.t[r];
  }
}

// Eigen's Isometry3f * Vector4f: per row a balanced-tree sum of four float products, never fused (SURVEY App. B6)
__device__ __forceinline__ float xform_row(const float* m, float x, float y, float z) {
  return __fadd_rn(__fadd_rn(__fmul_rn(m[0], x), __fmul_rn(m[1], y)), __fadd_rn(__fmul_rn(m[2], z), __fmul_rn(m[3], 1.0f)));
}

// The 1-NN of most source points is settled inside the 3x3x3 cells around them by their own thread.  The rest — points
// whose nearest neighbour may lie farther than one cell (cell edge < max-correspondence distance, or no neighbour
// nearby at all) — used to walk up to 5^3 cells alone and the whole grid waited at the reduction for that one thread.
// They are queued in shared memory instead and the block's warps pull them one by one and finish the search
// cooperatively (grid_search_warp resumed at radius 1, 32 candidates per step).
struct TailQuery { float qx, qy, qz, d; int p; };
struct TailQueue {
  TailQuery q[AL_THREADS];          // slot = threadIdx.x of the owning thread (results are written back in place)
  unsigned short list[AL_THREADS];  // owning threads, in arrival order (the order does not influence any result)
  int n, next;
};

// after the search: Mahalanobis + H/b/err contribution of source point i with nearest sorted slot my_p at my_d
__device__ __forceinline__ void finish_point(const AlignArgs& a, const Iso3& Td, double thr2, int i, const float4 p, float my_d, int my_p, double* acc) {
  int corr = -1;
  if (my_p >= 0 && (double)my_d < thr2) {
    const float4 tp = __ldg(a.tgt.sorted + my_p);
    corr = __float_as_int(tp.w);
    double CA[6], CB[6], RCR[6], M[6];
    const double* ca = a.src_cov + (size_t)i * 6;
    const double* cb = a.tgt_cov + (size_t)corr * 6;
#pragma unroll
    for (int j = 0; j < 6; j++) { CA[j] = __ldg(ca + j); CB[j] = __ldg(cb + j); }
    sym3_rcr(CB, Td.R, CA, RCR);
    sym3_inverse(RCR, M);
    const double px = (double)p.x, py = (double)p.y, pz = (double)p.z;
    double tA[3], e[3];
    tA[0] = Td.R[0] * px + Td.R[1] * py + Td.R[2] * pz + Td.t[0];
    tA[1] = Td.R[3] * px + Td.R[4] * py + Td.R[5] * pz + Td.t[1];
    tA[2] = Td.R[6] * px + Td.R[7] * py + Td.R[8] * pz + Td.t[2];
    e[0] = (double)tp.x - tA[0]; e[1] = (double)tp.y - tA[1]; e[2] = (double)tp.z - tA[2];
    gicp_accumulate(tA, e, M, acc);
    double* md = a.mahal + (size_t)i * 6;
#pragma unroll
    for (int j = 0; j < 6; j++) md[j] = M[j];
    a.tgt_pt[i] = tp;
  }
  a.corr[i] = corr;
  // without a correspondence the search may have stopped at the cap with any candidate: report none, not that one
  a.sqd[i] = corr >= 0 ? my_d : FLT_MAX;
}

__device__ __forceinline__ double error_point(const AlignArgs& a, const Iso3& Td, int i) {
  if (a.corr[i] < 0) return 0.0;
  const float4 p = __ldg(a.src_pts + i);
  const float4 tp = a.tgt_pt[i];
  const double* md = a.mahal + (size_t)i * 6;
  const double px = (double)p.x, py = (double)p.y, pz = (double)p.z;
  const double e0 = (double)tp.x - (Td.R[0] * px + Td.R[1] * py + Td.R[2] * pz + Td.t[0]);
  const double e1 = (double)tp.y - (Td.R[3] * px + Td.R[4] * py + Td.R[5] * pz + Td.t[1]);
  const double e2 = (double)tp.z - (Td.R[6] * px + Td.R[7] * py + Td.R[8] * pz + Td.t[2]);
  const double m0 = md[0] * e0 + md[1] * e1 + md[2] * e2;
  const double m1 = md[1] * e0 + md[3] * e1 + md[4] * e2;
  const double m2 = md[2] * e0 + md[4] * e1 + md[5] * e2;
  return e0 * m0 + e1 * m1 + e2 * m2;
}

// One block's share of a linearize pass.  LPP = lanes per source point: 1 = one thread per point; 2 / 4 = a group of
// adjacent lanes shares the point's candidate scans (a 20k-point scan cannot fill the GPU with one thread per point,
// and the search is a chain of dependent round trips — a group reads LPP x 8 candidates per round trip) and lane 0
// of the group does the fp64 part.
// Which points a block gets: the cloud is cut into chunks of 32 / LPP consecutive points (one warp's worth) and the
// chunks are dealt out round-robin — warp w of block blk takes chunks (pass * AL_WARPS + w) * nblk + blk.  A warp's
// points stay neighbours in space (voxel-filter output is in voxel order: its lanes scan the same target cells), but
// a block's eight warps sit in eight different places of the scan, so no block ends up with only far-field points
// whose searches are all long: with contiguous blocks of 256 points the slowest block took twice as long as the
// fastest (C2: 12 vs 27 us per linearisation) and the grid barrier waits for the slowest.  The trip count is the same
// for every block (the loop contains barriers).
template <int LPP>
__device__ __forceinline__ void linearize_block(const AlignArgs& a, const GridParams& gp, const XformF& Tf, const Iso3& Td,
                                                float cap_d2, double thr2, int blk, int nblk, TailQueue& tq, double& wtot) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = threadIdx.x & (LPP - 1), gi = threadIdx.x / LPP;
  const unsigned gmask = (LPP == 1) ? 0u : (((1u << LPP) - 1u) << (lane & ~(LPP - 1)));
  constexpr int PPW = 32 / LPP;                                   // points per warp and pass
  const int nchunks = (a.ns + PPW - 1) / PPW;
  const int npass = (nchunks + AL_WARPS * nblk - 1) / (AL_WARPS * nblk);
  for (int pass = 0; pass < npass; ++pass) {
    if (threadIdx.x == 0) { tq.n = 0; tq.next = 0; }
    __syncthreads();
    const int chunk = (pass * AL_WARPS + warp) * nblk + blk;
    const int i = chunk * PPW + lane / LPP;
    const bool active = chunk < nchunks && i < a.ns;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    float my_d = FLT_MAX;
    int my_p = -1;
    bool queued = false;
    if (active) {
      p = __ldg(a.src_pts + i);
      const float qx = xform_row(Tf.m + 0, p.x, p.y, p.z), qy = xform_row(Tf.m + 4, p.x, p.y, p.z), qz = xform_row(Tf.m + 8, p.x, p.y, p.z);
      bool mine = isfinite(qx) && isfinite(qy) && isfinite(qz);
      if (a.slab_axis >= 0) {
        const float qa = a.slab_axis == 0 ? qx : (a.slab_axis == 1 ? qy : qz);
        mine = mine && qa >= a.slab_lo && qa < a.slab_hi;
      }
      bool more = false;
      if (mine) {
        if (LPP == 1) more = grid_nn1_cube1(a.tgt, gp, qx, qy, qz, cap_d2, my_d, my_p);
        else more = grid_nn1_cube1_group<LPP>(a.tgt, gp, sub, gmask, qx, qy, qz, cap_d2, my_d, my_p);
      }
      if (more && sub == 0) {
        queued = true;
        TailQuery& t = tq.q[gi];
        t.qx = qx; t.qy = qy; t.qz = qz; t.d = my_d; t.p = my_p;
        tq.list[atomicAdd(&tq.n, 1)] = (unsigned short)gi;
      }
    }
    __syncthreads();
    const int nq = tq.n;
    if (nq > 0) {
      for (;;) {
        int e = 0;
        if (lane == 0) e = atomicAdd(&tq.next, 1);
        e = __shfl_sync(FULL, e, 0);
        if (e >= nq) break;
        TailQuery& t = tq.q[tq.list[e]];
        WarpBest1 rs;
        rs.d = t.d; rs.p = t.p;
        grid_search_warp<WarpBest1, true>(a.tgt, gp, t.qx, t.qy, t.qz, cap_d2, rs, false, 1);
        rs.finalize();
        if (lane == 0) { t.d = rs.d; t.p = rs.p; }
      }
      __syncthreads();
      if (queued) { my_d = tq.q[gi].d; my_p = tq.q[gi].p; }
    }
    // The 28 sums of this pass are reduced over the warp right away (lane j keeps the running total of value j):
    // one live register across the search instead of 28 accumulators.
    double contrib[NRED];
#pragma unroll
    for (int j = 0; j < NRED; j++) contrib[j] = 0.0;
    if (active && sub == 0) finish_point(a, Td, thr2, i, p, my_d, my_p, contrib);
    wtot += warp_sum_transposed<NRED>(contrib);
    __syncthreads();
  }
}

// block-level fixed-order reduction of NV values per thread -> out[0..NV) (written by threads < NV)
// NV == 1: acc[0] is a per-thread value; NV > 1: acc[0] of lane j is already the warp's total of value j
template <int NV>
__device__ __forceinline__ void block_reduce_store(double* acc, double (*s_red)[NRED], double* out) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (NV == 1) {
    const double s = warp_sum(acc[0]);
    if (lane == 0) s_red[w][0] = s;
  } else {
    if (lane < NV) s_red[w][lane] = acc[0];
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double s = 0.0;
#pragma unroll
    for (int ww = 0; ww < AL_WARPS; ww++) s += s_red[ww][threadIdx.x];
    out[threadIdx.x] = s;
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------------
// stepped mode: one launch per phase
// ------------------------------------------------------------------------------------------
struct IsoArg { Iso3 x; };

__global__ void __launch_bounds__(AL_THREADS) linearize_kernel(AlignArgs a, IsoArg T, float cap_d2, double thr2) {
  __shared__ double s_red[AL_WARPS][NRED];
  __shared__ TailQueue s_tq;
  const GridParams gp = load_grid(a.tgt.desc);
  XformF Tf;
  make_xforms(T.x, Tf);
  double acc[1] = {0.0};
  linearize_block<1>(a, gp, Tf, T.x, cap_d2, thr2, blockIdx.x, gridDim.x, s_tq, acc[0]);
  block_reduce_store<NRED>(acc, s_red, a.partials + (size_t)blockIdx.x * NRED);
}

__global__ void __launch_bounds__(AL_THREADS) compute_error_kernel(AlignArgs a, IsoArg T) {
  __shared__ double s_red[AL_WARPS][NRED];
  double acc[1] = {0.0};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.ns; i += gridDim.x * blockDim.x) acc[0] += error_point(a, T.x, i);
  block_reduce_store<1>(acc, s_red, a.partials + (size_t)blockIdx.x * NRED);
}

// ------------------------------------------------------------------------------------------
// sharded submap with an UNBOUNDED correspondence distance (the library default corr_dist_threshold_ = FLT_MAX,
// nano_gicp_impl.hpp:59): slabs + halo are only exact for a finite distance, so the ranks exchange the nearest
// neighbours themselves — every rank finds the nearest point of ITS part of the target for every source point and
// packs (bits of the squared distance) << 32 | rank; a min-all-reduce over the ranks names the rank that holds the global
// nearest neighbour (non-negative floats order like their bit patterns; equal distances go to the lowest rank), and
// that rank alone adds the point's H / b / error terms (SURVEY 8e, fallback row).
// ------------------------------------------------------------------------------------------
constexpr unsigned long long NN1_NONE = 0x7f800000ffffffffull;   // +inf distance: loses against every real neighbour

__global__ void __launch_bounds__(AL_THREADS) nn1_packed_kernel(AlignArgs a, IsoArg T, float cap_d2, double thr2, unsigned rank,
                                                                 unsigned long long* __restrict__ out) {
  const GridParams gp = load_grid(a.tgt.desc);
  XformF Tf;
  make_xforms(T.x, Tf);
  // one WARP per source point: the growing-cube search of the registration tail, from scratch (a source point may lie
  // far outside this rank's part of the target: the search has to be able to cross empty space)
  const int lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const bool any_target = a.tgt.desc->n > 0;
  for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < a.ns; i += nwarps) {
    const float4 p = __ldg(a.src_pts + i);
    const float qx = xform_row(Tf.m + 0, p.x, p.y, p.z), qy = xform_row(Tf.m + 4, p.x, p.y, p.z), qz = xform_row(Tf.m + 8, p.x, p.y, p.z);
    WarpBest1 rs;
    rs.init();
    if (isfinite(qx) && isfinite(qy) && isfinite(qz) && any_target) {
      grid_search_warp<WarpBest1, true, 4>(a.tgt, gp, qx, qy, qz, cap_d2, rs, true);
      rs.finalize();
    }
    if (lane == 0) {
      const bool hit = rs.p >= 0 && (double)rs.d < thr2;
      a.corr[i] = hit ? rs.p : -1;          // parked for linearize_won_kernel: the SORTED SLOT, not yet the original index
      a.sqd[i] = rs.d;
      out[i] = hit ? (((unsigned long long)__float_as_uint(rs.d) << 32) | (unsigned long long)rank) : NN1_NONE;
    }
  }
}

__global__ void __launch_bounds__(AL_THREADS) linearize_won_kernel(AlignArgs a, IsoArg T, double thr2, unsigned rank,
                                                                    const unsigned long long* __restrict__ won) {
  __shared__ double s_red[AL_WARPS][NRED];
  double wtot = 0.0;
  const int npass = (a.ns + gridDim.x * blockDim.x - 1) / (gridDim.x * blockDim.x);      // block-uniform trip count
  for (int pass = 0; pass < npass; ++pass) {
    const int i = (pass * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
    double contrib[NRED];
#pragma unroll
    for (int j = 0; j < NRED; j++) contrib[j] = 0.0;
    if (i < a.ns) {
      const int slot = a.corr[i];
      const float d = a.sqd[i];
      const unsigned long long w = won[i];
      const bool mine = slot >= 0 && (unsigned)(w & 0xffffffffull) == rank && (unsigned)(w >> 32) == __float_as_uint(d);
      if (mine) finish_point(a, T.x, thr2, i, __ldg(a.src_pts + i), d, slot, contrib);
      else a.corr[i] = -1;
    }
    wtot += warp_sum_transposed<NRED>(contrib);
  }
  double acc[1] = {wtot};
  block_reduce_store<NRED>(acc, s_red, a.partials + (size_t)blockIdx.x * NRED);
}

__global__ void reduce_partials_kernel(const double* __restrict__ partials, int nblocks, int nv, double* __restrict__ out) {
  const int t = threadIdx.x;
  if (t < nv) {
    double s = 0.0;
    for (int b = 0; b < nblocks; b++) s += partials[(size_t)b * NRED + t];
    out[t] = s;
  }
}

static inline float cap_from(double max_corr_dist) {
  const double c2 = max_corr_dist * max_corr_dist;
  return c2 >= (double)FLT_MAX ? FLT_MAX : (float)c2 * 1.000001f + 1e-30f;
}

static AlignArgs make_args(const AlignBuffers& ab, int blocks_hint) {
  AlignArgs a;
  a.src_pts = ab.src_pts; a.src_cov = ab.src_cov; a.ns = ab.ns;
  a.tgt = ab.tgt; a.tgt_cov = ab.tgt_cov;
  a.mahal = ab.mahal; a.corr = ab.corr; a.sqd = ab.sqd; a.tgt_pt = ab.tgt_pt;
  a.partials = ab.partials; a.max_blocks = ab.max_blocks;
  a.slab_axis = ab.slab_axis; a.slab_lo = ab.slab_lo; a.slab_hi = ab.slab_hi;
  (void)blocks_hint;
  return a;
}

static int stepped_blocks(const AlignBuffers& ab) {
  int blocks = (ab.ns + AL_THREADS - 1) / AL_THREADS;
  if (blocks < 1) blocks = 1;
  if (blocks > ab.max_blocks) blocks = ab.max_blocks;
  return blocks;
}

cudaError_t launch_linearize(const AlignBuffers& ab, const double* T16, double max_corr_dist, cudaStream_t st) {
  const int blocks = stepped_blocks(ab);
  AlignArgs a = make_args(ab, blocks);
  IsoArg T;
  iso_from_colmajor16(T16, T.x);
  linearize_kernel<<<blocks, AL_THREADS, 0, st>>>(a, T, cap_from(max_corr_dist), max_corr_dist * max_corr_dist);
  reduce_partials_kernel<<<1, 32, 0, st>>>(a.partials, blocks, NRED, ab.reduced);
  note_launches(2);
  return cudaGetLastError();
}

cudaError_t launch_nn1_packed(const AlignBuffers& ab, const double* T16, double max_corr_dist, unsigned rank, unsigned long long* out, cudaStream_t st) {
  int blocks = (ab.ns + AL_WARPS - 1) / AL_WARPS;       // one warp per source point
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 16) blocks = 148 * 16;
  AlignArgs a = make_args(ab, blocks);
  IsoArg T;
  iso_from_colmajor16(T16, T.x);
  nn1_packed_kernel<<<blocks, AL_THREADS, 0, st>>>(a, T, cap_from(max_corr_dist), max_corr_dist * max_corr_dist, rank, out);
  note_launches(1);
  return cudaGetLastError();
}

cudaError_t launch_linearize_won(const AlignBuffers& ab, const double* T16, double max_corr_dist, unsigned rank, const unsigned long long* won,
                                 cudaStream_t st) {
  const int blocks = stepped_blocks(ab);
  AlignArgs a = make_args(ab, blocks);
  IsoArg T;
  iso_from_colmajor16(T16, T.x);
  linearize_won_kernel<<<blocks, AL_THREADS, 0, st>>>(a, T, max_corr_dist * max_corr_dist, rank, won);
  reduce_partials_kernel<<<1, 32, 0, st>>>(a.partials, blocks, NRED, ab.reduced);
  note_launches(2);
  return cudaGetLastError();
}

cudaError_t launch_compute_error(const AlignBuffers& ab, const double* T16, cudaStream_t st) {
  const int blocks = stepped_blocks(ab);
  AlignArgs a = make_args(ab, blocks);
  IsoArg T;
  iso_from_colmajor16(T16, T.x);
  compute_error_kernel<<<blocks, AL_THREADS, 0, st>>>(a, T);
  reduce_partials_kernel<<<1, 32, 0, st>>>(a.partials, blocks, 1, ab.reduced);
  note_launches(2);
  return cudaGetLastError();
}

__global__ void export_mahal_kernel(const double* __restrict__ mahal, const int* __restrict__ corr, int n, double* __restrict__ out16) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double* o = out16 + (size_t)i * 16;
    for (int j = 0; j < 16; j++) o[j] = 0.0;
    if (corr[i] >= 0) {
      const double* m = mahal + (size_t)i * 6;
      o[0] = m[0]; o[1] = m[1]; o[2] = m[2];
      o[4] = m[1]; o[5] = m[3]; o[6] = m[4];
      o[8] = m[2]; o[9] = m[4]; o[10] = m[5];
    }
  }
}
cudaError_t launch_export_mahal(const AlignBuffers& ab, double* out16, cudaStream_t st) {
  if (ab.ns <= 0) return cudaSuccess;
  export_mahal_kernel<<<(ab.ns + 255) / 256, 256, 0, st>>>(ab.mahal, ab.corr, ab.ns, out16);
  note_launches(1);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// fused mode: the whole optimisation in one persistent cooperative kernel
// ------------------------------------------------------------------------------------------
struct LmParams {
  unsigned long long* trace;   // optional device buffer of %globaltimer stamps (debug, NGICP_ALIGN_TRACE=1)
  int max_iterations, lm_max_iterations, optimizer;
  double rot_eps, trans_eps, lm_init_lambda_factor, thr2;
  float cap_d2;
};
struct Guess16 { float g[16]; };

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Grid-wide reduction of per-block partials, all blocks co-resident (cooperative launch).
// Every block stores its partial, then arrives on a monotonic counter; the LAST block to arrive sums
// all partials in a fixed order (so the result does not depend on which block that is), publishes the
// totals and releases a phase flag the other blocks wait on.  One barrier latency per phase, O(blocks)
// traffic, bit-deterministic.
struct GridSync {
  unsigned* arrive;   // bar[0]
  unsigned* flag;     // bar[1]
  unsigned* comm_err; // bar[3]: set by the reducing block when the peer exchange failed (sharded mode), read by all blocks
  double* totals;     // [2][NRED] in global memory
  unsigned phase;     // phases completed so far
  unsigned max_blocks;  // stride between the two phase-parity halves of the partials buffer
};

__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ---- sharded-submap mode: the exchange step fused into the grid reduction -------------------------------------
// Every rank (one process per GPU) owns one slab of the target; the block that finishes this rank's fixed-order sum
// writes the totals straight into EVERY rank's exchange buffer over NVLink (peer stores to IPC-mapped memory), raises
// a sequence flag there, waits until all ranks' flags for this exchange have arrived in its own buffer and adds the
// contributions in rank order.  All ranks therefore hold bit-identical sums and take identical LM decisions; there is
// no host round trip and no separate collective launch.  Slots are double-buffered by the parity of the exchange
// number: a rank can only be one exchange ahead of the slowest one, because finishing exchange s needs every rank's
// flag s.  A rank that does not show up within pc.timeout_ns trips a sticky error flag instead of hanging the GPU.
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// called by all AL_THREADS threads of the reducing block; s = this rank's total of column threadIdx.x (threads < NV)
template <int NV>
__device__ __forceinline__ double peer_exchange_sum(double s, const PeerComm& pc) {
  __shared__ unsigned long long s_seq;
  if (threadIdx.x == 0) s_seq = *pc.seq + 1ull;
  __syncthreads();
  const unsigned long long seq = s_seq;
  const int par = (int)(seq & 1ull);
  if (threadIdx.x < NV) {
    for (int p = 0; p < pc.world; ++p) {
      volatile double* dst = pc.data[p] + (size_t)(par * NGICP_MAX_RANKS + pc.rank) * PEER_SLOT_DOUBLES + threadIdx.x;
      *dst = s;
    }
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < pc.world) {
    st_release_sys_u64(pc.flag[threadIdx.x] + par * NGICP_MAX_RANKS + pc.rank, seq);
    const unsigned long long* mine = pc.flag[pc.rank] + par * NGICP_MAX_RANKS + threadIdx.x;
    const unsigned long long t0 = global_timer_ns();
    while (ld_acquire_sys_u64(mine) < seq) {
      if (*(volatile int*)pc.error) break;
      __nanosleep(200);
      if (global_timer_ns() - t0 > pc.timeout_ns) { *(volatile int*)pc.error = 1; break; }
    }
  }
  __threadfence_system();
  __syncthreads();
  double t = s;
  if (threadIdx.x < NV) {
    t = 0.0;
    for (int r = 0; r < pc.world; ++r)
      t += __ldcv(pc.data[pc.rank] + (size_t)(par * NGICP_MAX_RANKS + r) * PEER_SLOT_DOUBLES + threadIdx.x);
  }
  if (threadIdx.x == 0) *pc.seq = seq;
  return t;
}

// Sharded mode: *s_fail (shared memory) is set when the peer exchange failed (a rank did not show up in time) — the same
// value in every block of the grid, so that all of them leave the LM loop together instead of iterating on partial sums.
// (A word in shared memory, read at the two places that need it: a returned flag kept alive in a register cost the
// 80-register variant 25 % on dense scans.)
template <int NV>
__device__ __forceinline__ void grid_reduce(double* acc, double (*s_red)[NRED], double* s_tot, double* partials, GridSync& gs,
                                            const PeerComm& pc, unsigned* s_fail) {
  __shared__ int s_last;
  if (pc.world == 1) {
    // Single GPU: every block waits until all partials of this phase are published, then sums them ITSELF in the same
    // fixed order (identical totals everywhere, bit-deterministic) — no "last block sums, publishes, the others read
    // back" relay: two L2 round trips less per barrier.  Partials are double-buffered by phase parity: a fast block may
    // already be writing phase p+1 while a slow one still reads phase p (it cannot reach p+2 before that one arrives).
    double* mine = partials + ((size_t)(gs.phase & 1u) * gs.max_blocks + blockIdx.x) * NRED;
    block_reduce_store<NV>(acc, s_red, mine);
    if (threadIdx.x == 0) {
      __threadfence();
      atomicAdd(gs.arrive, 1u);
      const unsigned target = (gs.phase + 1u) * gridDim.x;
      while (ld_relaxed_u32(gs.arrive) < target) __nanosleep(20);
      __threadfence();
    }
    __syncthreads();
    const double* all = partials + (size_t)(gs.phase & 1u) * gs.max_blocks * NRED;
    const int v = threadIdx.x & 31, seg = threadIdx.x >> 5;
    if (v < NV) {
      double part[8];
#pragma unroll
      for (int u = 0; u < 8; u++) part[u] = 0.0;
      const unsigned nb = gridDim.x;
      for (unsigned b0 = seg; b0 < nb; b0 += AL_WARPS * 8) {
        double x[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
          const unsigned bk = b0 + u * AL_WARPS;
          x[u] = bk < nb ? __ldcg(all + (size_t)bk * NRED + v) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 8; u++) part[u] += x[u];
      }
      s_red[seg][v] = ((part[0] + part[1]) + (part[2] + part[3])) + ((part[4] + part[5]) + (part[6] + part[7]));
    }
    __syncthreads();
    if (threadIdx.x < NV) {
      double s = 0.0;
#pragma unroll
      for (int sg = 0; sg < AL_WARPS; sg++) s += s_red[sg][threadIdx.x];
      s_tot[threadIdx.x] = s;
    }
    gs.phase++;
    __syncthreads();
    return;
  }
  block_reduce_store<NV>(acc, s_red, partials + (size_t)blockIdx.x * NRED);
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned prev = atomicAdd(gs.arrive, 1u);
    s_last = (prev == (gs.phase + 1u) * gridDim.x - 1u) ? 1 : 0;
  }
  __syncthreads();
  double* tot = gs.totals + (size_t)(gs.phase & 1u) * NRED;
  if (s_last) {
    __threadfence();
    // warp `seg` sums blocks seg, seg+W, seg+2W, ... for column v = lane; 8 independent loads in flight,
    // combined in a fixed order (the result does not depend on which block happens to arrive last)
    const int v = threadIdx.x & 31, seg = threadIdx.x >> 5;
    if (v < NV) {
      double part[8];
#pragma unroll
      for (int u = 0; u < 8; u++) part[u] = 0.0;
      const unsigned nb = gridDim.x;
      for (unsigned b0 = seg; b0 < nb; b0 += AL_WARPS * 8) {
        double x[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
          const unsigned bk = b0 + u * AL_WARPS;
          x[u] = bk < nb ? __ldcg(partials + (size_t)bk * NRED + v) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 8; u++) part[u] += x[u];
      }
      s_red[seg][v] = ((part[0] + part[1]) + (part[2] + part[3])) + ((part[4] + part[5]) + (part[6] + part[7]));
    }
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x < NV) {
#pragma unroll
      for (int sg = 0; sg < AL_WARPS; sg++) s += s_red[sg][threadIdx.x];
    }
    if (pc.world > 1) s = peer_exchange_sum<NV>(s, pc);
    if (threadIdx.x < NV) __stcg(tot + threadIdx.x, s);
    if (threadIdx.x == 0 && pc.world > 1 && *(volatile int*)pc.error) *(volatile unsigned*)gs.comm_err = 1u;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
      asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(gs.flag), "r"(gs.phase + 1u) : "memory");
    }
  } else if (threadIdx.x == 0) {
    // poll with a relaxed load (no L1 invalidation per probe) and back off so that the reducing block is
    // not starved of L2 bandwidth; one acquire fence once the flag is seen
    while (ld_relaxed_u32(gs.flag) < gs.phase + 1u) __nanosleep(40);
    __threadfence();
  }
  __syncthreads();
  if (threadIdx.x < NV) s_tot[threadIdx.x] = __ldcg(tot + threadIdx.x);
  if (threadIdx.x == 0) *s_fail = __ldcg(gs.comm_err);
  gs.phase++;
  __syncthreads();
}

__device__ __forceinline__ void trace_stamp(const LmParams& prm, int& slot) {
  if (prm.trace && blockIdx.x == 0 && threadIdx.x == 0 && slot < 250) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    prm.trace[1 + slot] = t;
    slot++;
    prm.trace[0] = (unsigned long long)slot;
  }
}

// MINB = resident blocks per SM the kernel is compiled for.  1: 255 registers, the scalar LM state of thread 0 lives in
// registers (shortest critical path; scans up to ~38k points have one point per thread anyway).  2 / 3: 128 / 80
// registers, that state spills to local memory but twice / three times as many source points are in flight — the
// better trade for dense scans (C5).
template <int MINB, int LPP>
__global__ void __launch_bounds__(AL_THREADS, MINB) align_fused_kernel(AlignArgs a, LmParams prm, Guess16 guess, ngicp_result* __restrict__ res, unsigned* bar, double* totals, PeerComm pc) {
  int tslot = 0;
  trace_stamp(prm, tslot);
  __shared__ double s_red[AL_WARPS][NRED];
  __shared__ double s_tot[NRED];
  __shared__ TailQueue s_tq;
  __shared__ Iso3 s_x;        // transform used by the next phase
  __shared__ int s_decision;
  const GridParams gp = load_grid(a.tgt.desc);
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
  const int gstride = gridDim.x * blockDim.x;
  GridSync gs;
  gs.arrive = bar; gs.flag = bar + 1; gs.comm_err = bar + 3; gs.totals = totals; gs.phase = 0; gs.max_blocks = (unsigned)a.max_blocks;

  // scalar LM state, kept by thread 0 of every block (identical everywhere)
  // thread 0's matrices and transforms live in shared memory: in registers they cost the 128-register variants 2 KB of
  // spills (local-memory round trips on the serial solve path between two grid barriers)
  __shared__ double s_lm[3 * 36 + 12];
  __shared__ Iso3 s_iso[3];
  Iso3 &x0 = s_iso[0], &xi = s_iso[1], &delta = s_iso[2];
  double* const H36 = s_lm;
  double* const final_H = s_lm + 36;
  double* const A = s_lm + 72;
  double* const b6 = s_lm + 108;
  double* const d6 = s_lm + 114;
  double lambda = -1.0, y0 = 0.0, nu = 2.0;
  int nr_iterations = 0, n_lin = 0, n_err = 0, lm_failed = 0;
  bool converged = false;
  __shared__ unsigned s_comm_fail;
  if (threadIdx.x == 0) {
    s_comm_fail = 0u;
    double g16[16];
    for (int i = 0; i < 16; i++) g16[i] = (double)guess.g[i];
    iso_from_colmajor16(g16, x0);
    iso_identity(delta);
    for (int i = 0; i < 36; i++) final_H[i] = (i % 7 == 0) ? 1.0 : 0.0;
    for (int i = 0; i < 6; i++) d6[i] = 0.0;
    s_x = x0;
  }
  __syncthreads();

  for (int it = 0; it < prm.max_iterations; ++it) {
    // ---------------- linearize at s_x ----------------
    {
      const Iso3 T = s_x;
      XformF Tf;
      make_xforms(T, Tf);
      double acc[1] = {0.0};
      linearize_block<LPP>(a, gp, Tf, T, prm.cap_d2, prm.thr2, blockIdx.x, gridDim.x, s_tq, acc[0]);
      trace_stamp(prm, tslot);
      if (prm.trace && it == 1 && threadIdx.x == 0 && blockIdx.x < 1024) prm.trace[256 + blockIdx.x] = global_timer_ns();
      grid_reduce<NRED>(acc, s_red, s_tot, a.partials, gs, pc, &s_comm_fail);
      trace_stamp(prm, tslot);
    }
    int outcome = 0;  // 1: step returned true, 0: LM failed
    if (threadIdx.x == 0) {
      nr_iterations = it;
      n_lin++;
      unpack_H(s_tot, H36);
      for (int i = 0; i < 6; i++) b6[i] = s_tot[21 + i];
      y0 = s_tot[27];
    }
    if (prm.optimizer == NGICP_OPT_GAUSS_NEWTON) {
      if (threadIdx.x == 0) {
        double nb[6];
        for (int i = 0; i < 6; i++) nb[i] = -b6[i];
        lm_solve(H36, nb, d6);
        delta_from_step(d6, delta);
        iso_mul(delta, x0, xi);
        x0 = xi;
        for (int i = 0; i < 36; i++) final_H[i] = H36[i];
        converged = lm_is_converged(delta, prm.rot_eps, prm.trans_eps);
        s_x = x0;
        s_decision = (pc.world > 1 && s_comm_fail) ? 0 : (converged ? 2 : 1);
      }
      __syncthreads();
      outcome = 1;
    } else {
      if (threadIdx.x == 0) {
        if (lambda < 0.0) {
          double mx = 0.0;
          for (int i = 0; i < 6; i++) mx = fmax(mx, fabs(H36[i * 7]));
          lambda = prm.lm_init_lambda_factor * mx;
        }
        nu = 2.0;
      }
      for (int j = 0; j < prm.lm_max_iterations; ++j) {
        if (threadIdx.x == 0) {
          double nb[6];
          for (int i = 0; i < 36; i++) A[i] = H36[i];
          for (int i = 0; i < 6; i++) { A[i * 7] += lambda; nb[i] = -b6[i]; }
          lm_solve(A, nb, d6);
          delta_from_step(d6, delta);
          iso_mul(delta, x0, xi);
          s_x = xi;
        }
        __syncthreads();
        // ---------------- compute_error at xi ----------------
        {
          const Iso3 T = s_x;
          double acc[1] = {0.0};
          trace_stamp(prm, tslot);
          for (int i = gtid; i < a.ns; i += gstride) acc[0] += error_point(a, T, i);
          trace_stamp(prm, tslot);
          grid_reduce<1>(acc, s_red, s_tot, a.partials, gs, pc, &s_comm_fail);
          trace_stamp(prm, tslot);
        }
        if (threadIdx.x == 0) {
          n_err++;
          const double yi = s_tot[0];
          double denom = 0.0;
          for (int i = 0; i < 6; i++) denom += d6[i] * (lambda * d6[i] - b6[i]);
          const double rho = (y0 - yi) / denom;
          int dec;
          if (rho < 0) {
            if (lm_is_converged(delta, prm.rot_eps, prm.trans_eps)) dec = 3;  // return true without moving x0
            else { lambda = nu * lambda; nu = 2 * nu; dec = 0; }
          } else {
            x0 = xi;
            // std::max(1/3, v) returns 1/3 unless 1/3 < v (same NaN behaviour)
            const double w3 = 2.0 * rho - 1.0;
            const double v = 1.0 - w3 * w3 * w3;
            lambda = lambda * ((1.0 / 3.0 < v) ? v : 1.0 / 3.0);
            for (int i = 0; i < 36; i++) final_H[i] = H36[i];
            dec = 1;
          }
          // sharded mode, a peer missed an exchange (the same flag in every block): stop through the existing decision
          // word as a failed LM step — the sums of this iteration are partial, the caller gets NGICP_E_COMM
          if (pc.world > 1 && s_comm_fail) dec = 4;
          s_decision = dec;
        }
        __syncthreads();
        const int dec = s_decision;
        __syncthreads();
        if (dec != 0) { outcome = dec == 4 ? 0 : 1; break; }
      }
      if (threadIdx.x == 0) {
        if (outcome == 0) lm_failed = 1;
        else converged = lm_is_converged(delta, prm.rot_eps, prm.trans_eps);
        s_x = x0;
        s_decision = (outcome == 0) ? 0 : (converged ? 2 : 1);
      }
      __syncthreads();
    }
    const int dec = s_decision;
    __syncthreads();
    if (dec == 0 || dec == 2) break;
  }

  if (blockIdx.x == 0 && threadIdx.x == 0) {
    double T16[16];
    iso_to_colmajor16(x0, T16);
    for (int i = 0; i < 16; i++) { res->final_x[i] = T16[i]; res->final_transformation[i] = (float)T16[i]; }
    for (int i = 0; i < 36; i++) res->final_hessian[i] = final_H[i];
    res->lm_lambda = lambda;
    res->last_error = y0;
    res->nr_iterations = nr_iterations;
    res->converged = converged ? 1 : 0;
    res->n_linearize = n_lin;
    res->n_compute_error = n_err;
    res->lm_failed = lm_failed;
    res->reserved = (pc.world > 1) ? *(volatile int*)pc.error : 0;   // 1: a peer did not show up in time
  }
  // leave the barrier words zeroed for the next launch: the last block to depart does it (nobody polls any more)
  if (threadIdx.x == 0) {
    const unsigned prev = atomicAdd(bar + 2, 1u);
    if (prev == gridDim.x - 1u) { bar[0] = 0u; bar[1] = 0u; bar[2] = 0u; bar[3] = 0u; }
  }
}

// ------------------------------------------------------------------------------------------
// batched mode: B independent registrations in ONE launch (ngicp_align_batch; BASELINE config C4).
// One thread-block CLUSTER per pair: the cluster's CTAs work through the pair's "virtual blocks" — exactly the blocks
// (same points, same warps, same lanes) a single align_fused launch of that pair would run — and publish one partial per
// virtual block; a hardware cluster barrier replaces the grid barrier, and every CTA then sums the partials in the
// single launch's fixed order.  Every sum therefore has the single launch's bits and every LM decision is the same:
// a batch result is bit-identical to the B single calls.  Clusters never wait for one another, so the launch is an
// ordinary one with any number of pairs (no co-residency requirement).
// ------------------------------------------------------------------------------------------
namespace cg = cooperative_groups;

struct BatchPair {
  AlignArgs a;
  LmParams prm;
  Guess16 guess;
  ngicp_result* res;
  int vblocks;      // blocks of the equivalent single launch
};

// fixed-order sum of nb per-block partials (the single-GPU branch of grid_reduce): totals -> s_tot[0..NV)
template <int NV>
__device__ __forceinline__ void sum_partials(const double* __restrict__ all, unsigned nb, double (*s_red)[NRED], double* s_tot) {
  const int v = threadIdx.x & 31, seg = threadIdx.x >> 5;
  if (v < NV) {
    double part[8];
#pragma unroll
    for (int u = 0; u < 8; u++) part[u] = 0.0;
    for (unsigned b0 = seg; b0 < nb; b0 += AL_WARPS * 8) {
      double x[8];
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const unsigned bk = b0 + u * AL_WARPS;
        x[u] = bk < nb ? __ldcg(all + (size_t)bk * NRED + v) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 8; u++) part[u] += x[u];
    }
    s_red[seg][v] = ((part[0] + part[1]) + (part[2] + part[3])) + ((part[4] + part[5]) + (part[6] + part[7]));
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double s = 0.0;
#pragma unroll
    for (int sg = 0; sg < AL_WARPS; sg++) s += s_red[sg][threadIdx.x];
    s_tot[threadIdx.x] = s;
  }
  __syncthreads();
}

template <int LPP>
__global__ void __launch_bounds__(AL_THREADS, 2) align_batch_kernel(const BatchPair* __restrict__ pairs) {
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned crank = cluster.block_rank(), csize = cluster.num_blocks();
  __shared__ double s_red[AL_WARPS][NRED];
  __shared__ double s_tot[NRED];
  __shared__ TailQueue s_tq;
  __shared__ Iso3 s_x;
  __shared__ int s_decision;
  __shared__ BatchPair s_pair;
  {
    const int* src = reinterpret_cast<const int*>(pairs + blockIdx.x / csize);
    int* dst = reinterpret_cast<int*>(&s_pair);
    for (int i = threadIdx.x; i < (int)(sizeof(BatchPair) / sizeof(int)); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const AlignArgs& a = s_pair.a;
  const LmParams& prm = s_pair.prm;
  const int VB = s_pair.vblocks;
  const GridParams gp = load_grid(a.tgt.desc);
  unsigned phase = 0;

  // thread 0's matrices and transforms live in shared memory: in registers they cost the 128-register variants 2 KB of
  // spills (local-memory round trips on the serial solve path between two grid barriers)
  __shared__ double s_lm[3 * 36 + 12];
  __shared__ Iso3 s_iso[3];
  Iso3 &x0 = s_iso[0], &xi = s_iso[1], &delta = s_iso[2];
  double* const H36 = s_lm;
  double* const final_H = s_lm + 36;
  double* const A = s_lm + 72;
  double* const b6 = s_lm + 108;
  double* const d6 = s_lm + 114;
  double lambda = -1.0, y0 = 0.0, nu = 2.0;
  int nr_iterations = 0, n_lin = 0, n_err = 0, lm_failed = 0;
  bool converged = false;
  if (threadIdx.x == 0) {
    double g16[16];
    for (int i = 0; i < 16; i++) g16[i] = (double)s_pair.guess.g[i];
    iso_from_colmajor16(g16, x0);
    iso_identity(delta);
    for (int i = 0; i < 36; i++) final_H[i] = (i % 7 == 0) ? 1.0 : 0.0;
    for (int i = 0; i < 6; i++) d6[i] = 0.0;
    s_x = x0;
  }
  __syncthreads();

  for (int it = 0; it < prm.max_iterations; ++it) {
    // ---------------- linearize at s_x: this CTA's virtual blocks ----------------
    {
      const Iso3 T = s_x;
      XformF Tf;
      make_xforms(T, Tf);
      double* mine = a.partials + (size_t)(phase & 1u) * a.max_blocks * NRED;
      for (int vb = (int)crank; vb < VB; vb += (int)csize) {
        double acc[1] = {0.0};
        linearize_block<LPP>(a, gp, Tf, T, prm.cap_d2, prm.thr2, vb, VB, s_tq, acc[0]);
        block_reduce_store<NRED>(acc, s_red, mine + (size_t)vb * NRED);
      }
      __threadfence();
      cluster.sync();
      sum_partials<NRED>(mine, (unsigned)VB, s_red, s_tot);
      phase++;
    }
    int outcome = 0;
    if (threadIdx.x == 0) {
      nr_iterations = it;
      n_lin++;
      unpack_H(s_tot, H36);
      for (int i = 0; i < 6; i++) b6[i] = s_tot[21 + i];
      y0 = s_tot[27];
    }
    if (prm.optimizer == NGICP_OPT_GAUSS_NEWTON) {
      if (threadIdx.x == 0) {
        double nb[6];
        for (int i = 0; i < 6; i++) nb[i] = -b6[i];
        lm_solve(H36, nb, d6);
        delta_from_step(d6, delta);
        iso_mul(delta, x0, xi);
        x0 = xi;
        for (int i = 0; i < 36; i++) final_H[i] = H36[i];
        converged = lm_is_converged(delta, prm.rot_eps, prm.trans_eps);
        s_x = x0;
        s_decision = converged ? 2 : 1;
      }
      __syncthreads();
      outcome = 1;
    } else {
      if (threadIdx.x == 0) {
        if (lambda < 0.0) {
          double mx = 0.0;
          for (int i = 0; i < 6; i++) mx = fmax(mx, fabs(H36[i * 7]));
          lambda = prm.lm_init_lambda_factor * mx;
        }
        nu = 2.0;
      }
      for (int j = 0; j < prm.lm_max_iterations; ++j) {
        if (threadIdx.x == 0) {
          double nb[6];
          for (int i = 0; i < 36; i++) A[i] = H36[i];
          for (int i = 0; i < 6; i++) { A[i * 7] += lambda; nb[i] = -b6[i]; }
          lm_solve(A, nb, d6);
          delta_from_step(d6, delta);
          iso_mul(delta, x0, xi);
          s_x = xi;
        }
        __syncthreads();
        // ---------------- compute_error at xi ----------------
        {
          const Iso3 T = s_x;
          double* mine = a.partials + (size_t)(phase & 1u) * a.max_blocks * NRED;
          for (int vb = (int)crank; vb < VB; vb += (int)csize) {
            double acc[1] = {0.0};
            for (int i = vb * AL_THREADS + threadIdx.x; i < a.ns; i += VB * AL_THREADS) acc[0] += error_point(a, T, i);
            block_reduce_store<1>(acc, s_red, mine + (size_t)vb * NRED);
          }
          __threadfence();
          cluster.sync();
          sum_partials<1>(mine, (unsigned)VB, s_red, s_tot);
          phase++;
        }
        if (threadIdx.x == 0) {
          n_err++;
          const double yi = s_tot[0];
          double denom = 0.0;
          for (int i = 0; i < 6; i++) denom += d6[i] * (lambda * d6[i] - b6[i]);
          const double rho = (y0 - yi) / denom;
          int dec;
          if (rho < 0) {
            if (lm_is_converged(delta, prm.rot_eps, prm.trans_eps)) dec = 3;
            else { lambda = nu * lambda; nu = 2 * nu; dec = 0; }
          } else {
            x0 = xi;
            const double w3 = 2.0 * rho - 1.0;
            const double v = 1.0 - w3 * w3 * w3;
            lambda = lambda * ((1.0 / 3.0 < v) ? v : 1.0 / 3.0);
            for (int i = 0; i < 36; i++) final_H[i] = H36[i];
            dec = 1;
          }
          s_decision = dec;
        }
        __syncthreads();
        const int dec = s_decision;
        __syncthreads();
        if (dec != 0) { outcome = 1; break; }
      }
      if (threadIdx.x == 0) {
        if (outcome == 0) lm_failed = 1;
        else converged = lm_is_converged(delta, prm.rot_eps, prm.trans_eps);
        s_x = x0;
        s_decision = (outcome == 0) ? 0 : (converged ? 2 : 1);
      }
      __syncthreads();
    }
    const int dec = s_decision;
    __syncthreads();
    if (dec == 0 || dec == 2) break;
  }

  if (crank == 0 && threadIdx.x == 0) {
    ngicp_result* res = s_pair.res;
    double T16[16];
    iso_to_colmajor16(x0, T16);
    for (int i = 0; i < 16; i++) { res->final_x[i] = T16[i]; res->final_transformation[i] = (float)T16[i]; }
    for (int i = 0; i < 36; i++) res->final_hessian[i] = final_H[i];
    res->lm_lambda = lambda;
    res->last_error = y0;
    res->nr_iterations = nr_iterations;
    res->converged = converged ? 1 : 0;
    res->n_linearize = n_lin;
    res->n_compute_error = n_err;
    res->lm_failed = lm_failed;
    res->reserved = 0;
  }
  cluster.sync();   // no CTA of the cluster exits while another may still read its partials / shared memory
}

// compiled variants: (resident blocks per SM, lanes per source point)
static const void* fused_variant(int minb, int lpp) {
  if (lpp == 2) return minb <= 2 ? (const void*)align_fused_kernel<2, 2> : (const void*)align_fused_kernel<3, 2>;
  return minb == 1 ? (const void*)align_fused_kernel<1, 1> : (minb == 2 ? (const void*)align_fused_kernel<2, 1> : (const void*)align_fused_kernel<3, 1>);
}
static int fused_blocks_per_sm(int device, int minb, int lpp = 1) {
  static int cached[64][4][5] = {};
  if (device >= 0 && device < 64 && cached[device][minb][lpp]) return cached[device][minb][lpp];
  int per_sm = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fused_variant(minb, lpp), AL_THREADS, 0);
  if (per_sm < 1) per_sm = 1;
  if (device >= 0 && device < 64) cached[device][minb][lpp] = per_sm;
  return per_sm;
}
static int sm_count_of(int device) {
  static int cached[64] = {};
  if (device >= 0 && device < 64 && cached[device]) return cached[device];
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (sms < 1) sms = 1;
  if (device >= 0 && device < 64) cached[device] = sms;
  return sms;
}
// The first launch of a kernel variant is expensive: CUDA loads kernels lazily and, worse, a variant with a larger
// stack frame than anything launched before makes the driver re-size the context's local-memory pool (measured:
// 165-414 ms in the middle of an odometry stream, when the submap first became large enough for the
// two-lanes-per-point variant).  Launch every variant once on an empty problem at ngicp_create time instead.
void align_prime_kernels(int device) {
  unsigned char* buf = nullptr;
  if (cudaMalloc(&buf, 8192) != cudaSuccess) { cudaGetLastError(); return; }
  cudaMemset(buf, 0, 8192);
  AlignArgs a;
  memset(&a, 0, sizeof a);
  a.tgt.desc = reinterpret_cast<GridDesc*>(buf);          // zeroed descriptor: never searched, ns = 0
  a.partials = reinterpret_cast<double*>(buf + 4096);
  a.max_blocks = 4;
  a.slab_axis = -1;
  LmParams prm;
  memset(&prm, 0, sizeof prm);                            // max_iterations = 0: the LM loop is not entered
  Guess16 g;
  for (int i = 0; i < 16; i++) g.g[i] = (i % 5 == 0) ? 1.0f : 0.0f;
  ngicp_result* res = reinterpret_cast<ngicp_result*>(buf + 1024);
  unsigned* bar = reinterpret_cast<unsigned*>(buf + 2048);
  double* totals = reinterpret_cast<double*>(buf + 3072);
  PeerComm pc;
  memset(&pc, 0, sizeof pc);
  pc.world = 1;
  void* args[] = {(void*)&a, (void*)&prm, (void*)&g, (void*)&res, (void*)&bar, (void*)&totals, (void*)&pc};
  for (int lpp = 1; lpp <= 2; ++lpp)
    for (int minb = (lpp == 2 ? 2 : 1); minb <= 3; ++minb) {
      fused_blocks_per_sm(device, minb, lpp);
      cudaLaunchCooperativeKernel(fused_variant(minb, lpp), dim3(1), dim3(AL_THREADS), args, 0, 0);
    }
  cudaDeviceSynchronize();
  cudaFree(buf);
  cudaFuncAttributes fa;
  cudaFuncGetAttributes(&fa, linearize_kernel);
  cudaFuncGetAttributes(&fa, compute_error_kernel);
  cudaFuncGetAttributes(&fa, reduce_partials_kernel);
  cudaFuncGetAttributes(&fa, align_batch_kernel<1>);
  cudaFuncGetAttributes(&fa, align_batch_kernel<2>);
  cudaGetLastError();
}

int align_fused_max_blocks(int device) { return fused_blocks_per_sm(device, 1) * sm_count_of(device); }

// Launch shape of the fused LM kernel for one registration.  Lanes per source point: 2 when the target is much larger
// than the scan (scan-to-map against a submap of overlapping keyframes: hundreds of candidates per query, the pair
// halves the chain of round trips; measured on C2: align 0.207 -> 0.178 ms) and the grid can still give every point its
// own pair; 1 otherwise (scan-to-scan: 0.092 vs 0.096 ms, the 255-register variant wins).  4 lanes per point need the
// 80-register variant and lose (0.123 ms).  Then the fewest resident blocks per SM (= most registers) that hold the
// grid.  NGICP_ALIGN_LPP / _MINB override.  The batched kernel reproduces the same blocks as virtual blocks.
static void fused_shape(const AlignBuffers& ab, int device, int& lpp, int& minb, int& blocks) {
  static const int minb_env = getenv("NGICP_ALIGN_MINB") ? atoi(getenv("NGICP_ALIGN_MINB")) : 0;
  static const int lpp_env = getenv("NGICP_ALIGN_LPP") ? atoi(getenv("NGICP_ALIGN_LPP")) : 0;
  const int sms = sm_count_of(device);
  lpp = 1; minb = 1;
  if (lpp_env == 1 || lpp_env == 2) lpp = lpp_env;
  else if ((long long)ab.nt >= 4ll * ab.ns) {
    const int need = (ab.ns + AL_THREADS / 2 - 1) / (AL_THREADS / 2);
    if (need <= fused_blocks_per_sm(device, 2, 2) * sms && need <= ab.max_blocks) lpp = 2;
  }
  const int ppb = AL_THREADS / lpp;                      // source points per block and pass
  blocks = (ab.ns + ppb - 1) / ppb;
  minb = lpp == 2 ? 2 : 1;
  while (minb < 3 && blocks > fused_blocks_per_sm(device, minb, lpp) * sms) ++minb;
  if (minb_env >= 1 && minb_env <= 3) minb = minb_env;
  if (lpp == 2 && minb < 2) minb = 2;
  const int lim = fused_blocks_per_sm(device, minb, lpp) * sms;
  if (blocks > lim) blocks = lim;
  if (blocks > ab.max_blocks) blocks = ab.max_blocks;
  if (blocks < 1) blocks = 1;
}

static LmParams make_lm_params(const ngicp_params& p, unsigned long long* trace) {
  LmParams prm;
  prm.trace = trace;
  prm.max_iterations = p.max_iterations;
  prm.lm_max_iterations = p.lm_max_iterations;
  prm.optimizer = p.optimizer;
  prm.rot_eps = p.rotation_epsilon;
  prm.trans_eps = p.transformation_epsilon;
  prm.lm_init_lambda_factor = p.lm_init_lambda_factor;
  prm.thr2 = p.max_correspondence_distance * p.max_correspondence_distance;
  prm.cap_d2 = cap_from(p.max_correspondence_distance);
  return prm;
}

size_t align_batch_pair_bytes() { return sizeof(BatchPair); }

// fill one BatchPair record (host staging memory) for launch_align_batch; returns the lanes per point it needs
int align_batch_fill(void* dst, const AlignBuffers& ab, const ngicp_params& p, const float* guess16, ngicp_result* res_dev, int device) {
  int lpp, minb, blocks;
  fused_shape(ab, device, lpp, minb, blocks);
  BatchPair bp;
  memset(&bp, 0, sizeof bp);
  bp.a = make_args(ab, blocks);
  bp.prm = make_lm_params(p, nullptr);
  for (int i = 0; i < 16; i++) bp.guess.g[i] = guess16 ? guess16[i] : ((i % 5 == 0) ? 1.0f : 0.0f);
  bp.res = res_dev;
  bp.vblocks = blocks;
  memcpy(dst, &bp, sizeof bp);
  return lpp;
}

// one cluster of ALIGN_BATCH_CLUSTER blocks per pair; pairs_dev = n_pairs BatchPair records in device memory, all with
// the same lanes-per-point
cudaError_t launch_align_batch(const void* pairs_dev, int n_pairs, int lpp, cudaStream_t st) {
  if (n_pairs <= 0) return cudaSuccess;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = dim3((unsigned)n_pairs * ALIGN_BATCH_CLUSTER);
  cfg.blockDim = dim3(AL_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = ALIGN_BATCH_CLUSTER;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const BatchPair* pp = static_cast<const BatchPair*>(pairs_dev);
  note_launches(1);
  if (lpp == 2) return cudaLaunchKernelEx(&cfg, align_batch_kernel<2>, pp);
  return cudaLaunchKernelEx(&cfg, align_batch_kernel<1>, pp);
}

cudaError_t launch_align_fused(const AlignBuffers& ab, const ngicp_params& p, const float* guess16, ngicp_result* res_dev,
                               unsigned* barrier, int device, cudaStream_t st, unsigned long long* trace, const PeerComm* comm) {
  int lpp, minb, blocks;
  fused_shape(ab, device, lpp, minb, blocks);
  AlignArgs a = make_args(ab, blocks);
  LmParams prm = make_lm_params(p, trace);
  Guess16 g;
  for (int i = 0; i < 16; i++) g.g[i] = guess16 ? guess16[i] : ((i % 5 == 0) ? 1.0f : 0.0f);
  double* totals = ab.reduced;  // [2][NRED]
  note_launches(1);
  PeerComm pc;
  memset(&pc, 0, sizeof pc);
  pc.world = 1;
  if (comm && comm->world > 1) pc = *comm;
  void* args[] = {(void*)&a, (void*)&prm, (void*)&g, (void*)&res_dev, (void*)&barrier, (void*)&totals, (void*)&pc};
  const void* fn = fused_variant(minb, lpp);
  return cudaLaunchCooperativeKernel(fn, dim3(blocks), dim3(AL_THREADS), args, 0, st);
}

}  // namespace ngicp
