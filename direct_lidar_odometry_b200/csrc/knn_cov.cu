// knn_cov.cu — K2+K3: k-nearest-neighbour search fused with the plane-regularised covariance
// estimate (reference include/nano_gicp/impl/nano_gicp_impl.hpp:298-357), plus the raw kNN query
// entry used by the parity tests (KdTreeFLANN::nearestKSearch, include/nano_gicp/nanoflann.hpp:141-152).
//
// Two launches: knn_lists_kernel — one WARP per point for the search (coalesced candidate scans,
// warp-distributed top-k list, few registers so that many warps hide the gather latency), neighbour
// slots parked in HBM (4k B/point of scratch, L2 resident); cov_from_lists_kernel — one THREAD per
// point for the fp64 statistics + 3x3 Jacobi SVD.  Algorithmic bytes of the pair: 16 B point read +
// 48 B covariance write = 64 B/point.
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include "internal.h"
#include "grid_search.cuh"
#include "gicp_math.cuh"
#include "sort_networks.inc"

namespace ngicp {

constexpr int KC_THREADS = 256;
constexpr int KC_WARPS = KC_THREADS / 32;
#ifndef KNN_MIN_BLOCKS
#define KNN_MIN_BLOCKS 5
#endif

// queries: arbitrary points (float4 xyz), results in ORIGINAL index order of the cloud
__global__ void __launch_bounds__(KC_THREADS) knn_query_kernel(GridView g, const float4* __restrict__ queries, int nq, int k,
                                                               int* __restrict__ idx, float* __restrict__ d2) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const GridParams gp = load_grid(g.desc);
  for (int q = warp; q < nq; q += nwarps) {
    const float4 qp = queries[q];
    WarpTopK rs;
    rs.init(k, lane);
    if (isfinite(qp.x) && isfinite(qp.y) && isfinite(qp.z)) grid_search_warp(g, gp, qp.x, qp.y, qp.z, FLT_MAX, rs);
    if (lane < k) {
      int o = -1;
      float dd = -1.f;
      if (rs.p >= 0) { o = __float_as_int(__ldg(g.sorted + rs.p).w); dd = rs.d; }
      idx[(size_t)q * k + lane] = o;
      d2[(size_t)q * k + lane] = dd;
    }
  }
}

// K2: neighbour lists of the cloud's own points, one warp per point, visited in cell order so that
// concurrently running warps read the same cells.  nbr[q*k + j] = sorted slot of the j-th neighbour.
// Only the sorted slots [q_lo, q_hi) are answered (the whole cloud by default; a part of it when the covariances of one
// cloud are split over several GPUs, ngicp_calc_source_covs_part).
__global__ void __launch_bounds__(KC_THREADS, KNN_MIN_BLOCKS) knn_lists_kernel(GridView g, int n, int k, int* __restrict__ nbr, int q_lo, int q_hi) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const GridParams gp = load_grid(g.desc);
  for (int q = q_lo + warp; q < q_hi; q += nwarps) {
    const float4 qp = __ldg(g.sorted + q);
    WarpTopK rs;
    rs.init(k, lane);
    if (isfinite(qp.x) && isfinite(qp.y) && isfinite(qp.z)) grid_search_warp(g, gp, qp.x, qp.y, qp.z, FLT_MAX, rs, k >= 4);
    if (lane < k) nbr[(size_t)q * k + lane] = rs.p;
  }
}

// k in (KNN_MAX_K, KNN_WIDE_MAX_K]: the same growing-cube search with the result set in shared memory (WarpTopKWide)
__global__ void __launch_bounds__(KC_THREADS) knn_query_wide_kernel(GridView g, const float4* __restrict__ queries, int nq, int k,
                                                                    int* __restrict__ idx, float* __restrict__ d2) {
  __shared__ float s_d[KC_WARPS][KNN_WIDE_MAX_K];
  __shared__ int s_p[KC_WARPS][KNN_WIDE_MAX_K];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const GridParams gp = load_grid(g.desc);
  for (int q = warp; q < nq; q += nwarps) {
    const float4 qp = queries[q];
    WarpTopKWide rs;
    rs.init(k, lane, s_d[wib], s_p[wib]);
    if (isfinite(qp.x) && isfinite(qp.y) && isfinite(qp.z)) grid_search_warp(g, gp, qp.x, qp.y, qp.z, FLT_MAX, rs);
    __syncwarp();
    for (int j = lane; j < k; j += 32) {
      const int p = s_p[wib][j];
      idx[(size_t)q * k + j] = p >= 0 ? __float_as_int(__ldg(g.sorted + p).w) : -1;
      d2[(size_t)q * k + j] = p >= 0 ? s_d[wib][j] : -1.f;
    }
  }
}
__global__ void __launch_bounds__(KC_THREADS) knn_lists_wide_kernel(GridView g, int n, int k, int* __restrict__ nbr, int q_lo, int q_hi) {
  __shared__ float s_d[KC_WARPS][KNN_WIDE_MAX_K];
  __shared__ int s_p[KC_WARPS][KNN_WIDE_MAX_K];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const GridParams gp = load_grid(g.desc);
  for (int q = q_lo + warp; q < q_hi; q += nwarps) {
    const float4 qp = __ldg(g.sorted + q);
    WarpTopKWide rs;
    rs.init(k, lane, s_d[wib], s_p[wib]);
    if (isfinite(qp.x) && isfinite(qp.y) && isfinite(qp.z)) grid_search_warp<WarpTopKWide, false, 4>(g, gp, qp.x, qp.y, qp.z, FLT_MAX, rs, true);
    __syncwarp();
    for (int j = lane; j < k; j += 32) nbr[(size_t)q * k + j] = s_p[wib][j];
  }
}

// K2, tile variant (the one launch_covariances uses) — cell-major, one THREAD per query.
// The cell grid is cut into boxes of TQ_CORE^3 cells.  knn_plan_kernel walks the boxes (skipping empty space 8 boxes at
// a time), splits boxes whose surroundings would not fit a tile (dense cells) into 8 children, down to single cells,
// and emits work items: (box, up to 64 of its points).  knn_lists_tile_kernel is persistent; a warp pulls an item,
// copies the cells within radius s (1, then 2, then 4 for the points that need it) around the box into shared memory
// ONCE — one coalesced x-run per (y,z) row, thanks to the x-fastest lower-bound table — and then answers the item's
// points from that tile, 32 at a time, every lane working on ITS OWN query:
//   threshold-and-verify   collect the tile points closer than a guessed T^2 into the lane's column of a
//                          shared-memory list; accept when between k and TQ_LCAP were collected, otherwise rescale
//                          T^2 by (k+8)/count (counts grow ~linearly in T^2 on surfaces) inside a bisection bracket;
//   exactness              T^2 never exceeds the squared, margin-shrunk distance from the query to the nearest face
//                          of the tile that still has cells behind it, so an accepted list contains every point that
//                          can be among the k nearest (same stop rule as grid_search_warp);
//   selection              the covariance only needs the SET of the k nearest, so the lane tightens the threshold on
//                          its short list (secant steps on the count) until exactly k remain — no sorting network,
//                          no dependent shuffles.  An exact tie at the k-th distance has no such threshold: those
//                          (rare) points take the warp search.
// One distance evaluation therefore costs one instruction slot per 32 queries instead of one per query.  Points that
// cannot be decided inside a radius-TQ_SMAX tile (isolated points, ties at the k-th distance) are appended to a list
// that knn_lists_rest_kernel — the next launch on the stream — answers with the growing-cube warp search.  (Round 1
// drained that list inside this kernel and waited for every warp of the launch to finish producing; two such launches
// sharing a GPU could then wait for blocks of their own that were not resident.  No kernel here waits on another block.)
#ifndef TQ_WARPS
#define TQ_WARPS 2
#endif
#define TQ_POS_BITS 9
#define TQ_POS_MASK 0x1ffu
#ifndef TQ_CMAX
#define TQ_CMAX 448      // tile capacity (slots: rows are padded to even lengths); measured on C2: 320 0.69, 384 0.72, 448 0.67 ms for the covariance phase
#endif
#ifndef TQ_LCAP
#define TQ_LCAP 40       // per-query collection capacity
#endif
#ifndef TQ_CORE
#define TQ_CORE KNN_BRICK   // box edge in cells
#endif
#ifndef TQ_PACKED
#define TQ_PACKED 1      // 1: packed f32x2 distance arithmetic (two candidates per instruction); 0: scalar
#endif
#ifndef TQ_UNROLL
#define TQ_UNROLL 1   // measured on C2 (benchmarks/ab_knn.py): 1: 0.752 ms, 2: 0.764, 4: 0.869 for the covariance phase
#endif
#define NG_PRAGMA_(x) _Pragma(#x)
#define NG_UNROLL(n) NG_PRAGMA_(unroll n)
#ifndef TQ_SMAX
#define TQ_SMAX 16       // largest tile radius tried before a point goes to the warp search
#endif
constexpr int TQ_ITEM = 64;  // points per work item
struct TileSmem {
  // staged candidates, structure of arrays: two neighbouring candidates are one 64-bit shared load per coordinate and go
  // through the packed f32x2 pipe together (FADD2 / FMUL2 / FFMA2, sm_100).  Every (y,z) row of the tile starts at an
  // even position and is padded to an even length with a point at +infinity (its distance is +inf: never collected).
  float xs[TQ_CMAX], ys[TQ_CMAX], zs[TQ_CMAX];
  int slot[TQ_CMAX];                     // sorted slot of the candidate
  // collected candidates, one column per lane, last row = dump: ONE 32-bit word per entry = the squared distance with
  // its 9 low mantissa bits replaced by the tile position (TQ_CMAX <= 512).  All thresholds live on the same lattice
  // (low 9 bits zero), so "d < T" and "entry < bits(T)" are the same test; two entries closer than 2^-14 relative cannot be
  // told apart — when that happens exactly at the k-th place the point takes the warp search, like an exact tie.
  unsigned lst[TQ_LCAP + 1][32];
  int cur[TQ_ITEM];                      // sorted slots of the points being answered from the current tile
  float cur_t[TQ_ITEM];                  // their threshold guesses (0 = none yet) ...
  float cur_lo[TQ_ITEM], cur_hi[TQ_ITEM];  // ... inside this bracket (hi < 0 = open)
  int nxt[TQ_ITEM];                      // points that need a larger tile
  int rowoff[68];                        // first tile position of every (y,z) row (radius <= 2 tiles: up to 64 rows)
};

// distance from q to the nearest face of the cell box [x0,x1]x[y0,y1]x[z0,z1] that still has cells behind it
__device__ __forceinline__ float box_face_distance(const GridParams& gp, int x0, int x1, int y0, int y1, int z0, int z1,
                                                   float qx, float qy, float qz) {
  float m = FLT_MAX;
  if (x0 > 0) m = fminf(m, qx - (gp.ox + (float)x0 * gp.cell));
  if (x1 + 1 < gp.dx) m = fminf(m, (gp.ox + (float)(x1 + 1) * gp.cell) - qx);
  if (y0 > 0) m = fminf(m, qy - (gp.oy + (float)y0 * gp.cell));
  if (y1 + 1 < gp.dy) m = fminf(m, (gp.oy + (float)(y1 + 1) * gp.cell) - qy);
  if (z0 > 0) m = fminf(m, qz - (gp.oz + (float)z0 * gp.cell));
  if (z1 + 1 < gp.dz) m = fminf(m, (gp.oz + (float)(z1 + 1) * gp.cell) - qz);
  return m == FLT_MAX ? FLT_MAX : m - gp.margin;
}

#ifdef TQ_DEBUG
#define TQ_CHECK(cond, what, a, b) do { if (!(cond)) { printf("TQ_CHECK %s failed: %d %d (block %d thread %d)\n", what, (int)(a), (int)(b), blockIdx.x, threadIdx.x); __trap(); } } while (0)
#else
#define TQ_CHECK(cond, what, a, b) do { } while (0)
#endif
enum { ST_FALLBACK = 0, ST_TIES, ST_TILES, ST_PASSES, ST_LANES, ST_ITEMS, ST_DEC1, ST_DEC2, ST_DECHI, ST_PASS1, ST_PASS2, ST_PASSHI, ST_CAND, ST_TSUM, ST_TEND, ST_TSTART, ST_TWARPS, ST_N };
// control words shared by the plan and tile launches
enum { CT_ITEMS = 0, CT_NEXT, CT_REST, CT_REST_NEXT, CT_DONE, CT_FIX, CT_SLOW, CT_N = 8 };

// warp-aggregated append of the lanes in `mask` to the warp-search list
__device__ __forceinline__ void fb_append(unsigned mask, int slot, int lane, int* __restrict__ fb_list, int* __restrict__ fb_count,
                                          unsigned char* __restrict__ fb_flags) {
  if (!mask) return;
  if ((mask >> lane) & 1u) fb_flags[slot] = 1;     // the main covariance launch skips it; cov_rest_kernel does it after the warp search
  const int leader = __ffs(mask) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(fb_count, __popc(mask));
  base = __shfl_sync(FULL, base, leader);
  if ((mask >> lane) & 1u) fb_list[base + __popc(mask & ((1u << lane) - 1u))] = slot;
}

// Points whose list the tile kernel delivered but could not ORDER exactly (two of the k kept entries share a lattice
// value): flagged like the warp-search ones so that the main covariance launch (which trusts the order) skips them, and
// listed from the BACK of the same array (the two lists are disjoint and hold at most n points together); cov_rest_kernel
// re-derives their order from exact distances.
__device__ __forceinline__ void fix_append(unsigned mask, int slot, int lane, int n, int* __restrict__ fb_list, int* __restrict__ fix_count,
                                           unsigned char* __restrict__ fb_flags) {
  if (!mask) return;
  if ((mask >> lane) & 1u) fb_flags[slot] = 1;
  const int leader = __ffs(mask) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(fix_count, __popc(mask));
  base = __shfl_sync(FULL, base, leader);
  if ((mask >> lane) & 1u) fb_list[n - 1 - (base + __popc(mask & ((1u << lane) - 1u)))] = slot;
}

__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, v, o); if (lane >= o) v += t; }
  return v;
}
// index of the run that holds flattened position t, given the inclusive scan of the run lengths over the lanes
__device__ __forceinline__ int run_of(int inc, int t) {
  int j = 0;
#pragma unroll
  for (int step = 16; step > 0; step >>= 1) {
    const int v = __shfl_sync(FULL, inc, j + step - 1);
    if (v <= t) j += step;
  }
  return j;
}

// number of points in the cells [x0-s, x0+sz-1+s] x [y0-s, ..] x [z0-s, ..], computed by a group of `nsub` adjacent
// lanes (power of two; `sub` = lane index inside the group); the result is uniform across the group
__device__ __forceinline__ int box_population(const GridView& g, const GridParams& gp, int x0, int y0, int z0, int sz, int s, int sub, int nsub) {
  const int ny = sz + 2 * s, nrows = ny * ny;
  const int xl = max(x0 - s, 0), xr = min(x0 + sz - 1 + s, gp.dx - 1) + 1;
  int c = 0;
  for (int r = sub; r < nrows; r += nsub) {
    const int y = y0 - s + (r % ny), z = z0 - s + (r / ny);
    if (y >= 0 && y < gp.dy && z >= 0 && z < gp.dz && xl < xr) {
      const int* row = g.cell_start + (z * gp.dy + y) * gp.dx;
      c += __ldg(row + xr) - __ldg(row + xl);
    }
  }
  for (int o = nsub >> 1; o > 0; o >>= 1) c += __shfl_xor_sync(FULL, c, o);
  return c;
}

// emit the work items of the boxes held by the lanes with q > 0 (one box per such lane)
// Two lists in one array of n entries (an item holds at least one point): the LONG items from the front — boxes in
// sparse surroundings (`slow`: they will need larger tiles, up to 41 rounds of dependent row lookups at radius 16) and
// items with more than TQ_BIG points (two or more batches per tile) — and the short ones from the back.  The tile kernel
// takes the front list first: a warp handles only ~6 items per launch, so the launch ends with a tail about one item
// long (warps were busy 85 % of the kernel's span) — it should be a short item.
#ifndef TQ_BIG
#define TQ_BIG 32
#endif
__device__ __forceinline__ void emit_items(bool emit, bool slow, int x0, int y0, int z0, int sz, int q, int lane, int n, int4* __restrict__ items,
                                           int* __restrict__ ctrl) {
  const int nit = emit ? (q + TQ_ITEM - 1) / TQ_ITEM : 0;
  // only the last item of a box can be short
  const int nfront = (slow || nit == 0 || q - (nit - 1) * TQ_ITEM > TQ_BIG) ? nit : nit - 1;
  const int nback = nit - nfront;
  if (__any_sync(FULL, nfront > 0)) {
    const int inc = warp_incl_scan(nfront, lane);
    const int total = __shfl_sync(FULL, inc, 31);
    int base = 0;
    if (lane == 0) base = atomicAdd(ctrl + CT_SLOW, total);
    base = __shfl_sync(FULL, base, 0) + inc - nfront;
    for (int i = 0; i < nfront; ++i) items[base + i] = make_int4(x0, y0, z0, sz | (i << 8));
  }
  const unsigned bm = __ballot_sync(FULL, nback > 0);
  if (bm) {
    int base = 0;
    if (lane == 0) base = atomicAdd(ctrl + CT_ITEMS, __popc(bm));
    base = __shfl_sync(FULL, base, 0) + __popc(bm & ((1u << lane) - 1u));
    if (nback > 0) items[n - 1 - base] = make_int4(x0, y0, z0, sz | ((nit - 1) << 8));
  }
}

// one warp per run of x-adjacent boxes (8 on big grids, 1 on small ones): emits the work items of knn_lists_tile_kernel.
// A box whose radius-1 tile would not fit is split into its 8 children (evaluated 4 lanes each, in parallel), and a
// child that still does not fit into its 8 single cells.
// Brick occupancy flags (one byte per box of TQ_CORE^3 cells), so that the plan does not have to walk the dense cell
// table to find out that most of space is empty: 64 MB of table reads for the 16 M-cell grid of the 500k-point C2 submap
// became 0.25 MB of flag reads.  brick_clear zeroes the flags of this grid's boxes, brick_mark sets the flag of every
// point's box (plain stores of the same value: no atomics needed).
__global__ void __launch_bounds__(256) brick_clear_kernel(GridView g, unsigned char* __restrict__ flags, long long flag_cap) {
  const GridParams gp = load_grid(g.desc);
  const long long nb = (long long)((gp.dx + TQ_CORE - 1) / TQ_CORE) * ((gp.dy + TQ_CORE - 1) / TQ_CORE) * ((gp.dz + TQ_CORE - 1) / TQ_CORE);
  if (nb > flag_cap) return;                           // the plan then falls back to table lookups
  const long long nw = (nb + 3) / 4;
  unsigned* f4 = reinterpret_cast<unsigned*>(flags);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += (long long)gridDim.x * blockDim.x) f4[i] = 0u;
}
// control words and warp-search flags to zero (one launch instead of two memset nodes)
__global__ void __launch_bounds__(256) knn_zero_kernel(int* __restrict__ ctrl, unsigned* __restrict__ fb_flags4, int nwords) {
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
  if (gtid < CT_N) ctrl[gtid] = 0;
  for (int i = gtid; i < nwords; i += gridDim.x * blockDim.x) fb_flags4[i] = 0u;
}
__global__ void __launch_bounds__(256) brick_mark_kernel(GridView g, int n, unsigned char* __restrict__ flags, long long flag_cap) {
  const GridParams gp = load_grid(g.desc);
  const int nbx = (gp.dx + TQ_CORE - 1) / TQ_CORE, nby = (gp.dy + TQ_CORE - 1) / TQ_CORE, nbz = (gp.dz + TQ_CORE - 1) / TQ_CORE;
  if ((long long)nbx * nby * nbz > flag_cap) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = __ldg(g.sorted + i);
    const int bx = cell_coord(p.x, gp.ox, gp.inv, gp.dx) / TQ_CORE, by = cell_coord(p.y, gp.oy, gp.inv, gp.dy) / TQ_CORE,
              bz = cell_coord(p.z, gp.oz, gp.inv, gp.dz) / TQ_CORE;
    flags[((long long)bz * nby + by) * nbx + bx] = 1;
  }
}

#ifndef TQ_SLOW_FACTOR
#define TQ_SLOW_FACTOR 2      // a box is "slow" when its radius-1 tile holds fewer than this many times k points
#endif
__global__ void __launch_bounds__(256) knn_plan_kernel(GridView g, int n, int k, int4* __restrict__ items, int* __restrict__ ctrl,
                                                       const unsigned char* __restrict__ flags, long long flag_cap) {
  const int lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const GridParams gp = load_grid(g.desc);
  const int nbx = (gp.dx + TQ_CORE - 1) / TQ_CORE, nby = (gp.dy + TQ_CORE - 1) / TQ_CORE, nbz = (gp.dz + TQ_CORE - 1) / TQ_CORE;
  const int run = ((long long)nbx * nby * nbz > 32768) ? 8 : 1;
  const int nrx = (nbx + run - 1) / run;
  const int nruns = nrx * nby * nbz;
  // the launch covers the usual run count; the stride loop covers flat grids, whose per-axis rounding makes more boxes
  for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < nruns; w += nwarps) {
    const int rbx = (w % nrx) * run, rby = (w / nrx) % nby, rbz = w / (nrx * nby);
    unsigned occ = FULL;                                   // boxes of the run that hold points
    if (run > 1 && (long long)nbx * nby * nbz <= flag_cap) {
      // whole run empty?  (one flag byte per box, the run's boxes are consecutive)
      int e = 0;
      if (lane < run && rbx + lane < nbx) e = flags[((long long)rbz * nby + rby) * nbx + rbx + lane];
      occ = __ballot_sync(FULL, e != 0);
      if (occ == 0u) continue;
    } else if (run > 1) {
      // (grids with more boxes than flag bytes) whole run empty?  (16 core rows, one lane each)
      int e = 0;
      if (lane < TQ_CORE * TQ_CORE) {
        const int y = rby * TQ_CORE + (lane % TQ_CORE), z = rbz * TQ_CORE + (lane / TQ_CORE);
        if (y < gp.dy && z < gp.dz) {
          const int* row = g.cell_start + (z * gp.dy + y) * gp.dx;
          e = __ldg(row + min((rbx + run) * TQ_CORE, gp.dx)) - __ldg(row + rbx * TQ_CORE);
        }
      }
      if (!__any_sync(FULL, e != 0)) continue;
    }
    // the run's boxes side by side, 4 lanes each (a dense run used to be 8 x 2 dependent rounds of table lookups by one
    // warp: the plan kernel's critical path); boxes that fit go out at once, the others are split one after the other
    const int y0 = rby * TQ_CORE, z0 = rbz * TQ_CORE;
    unsigned deep_boxes;
    {
      const int bi = lane >> 2, sub = lane & 3;
      const bool valid = bi < run && rbx + bi < nbx && ((occ >> bi) & 1u);
      const int bx0 = valid ? (rbx + bi) * TQ_CORE : -(1 << 20);       // far outside: box_population touches nothing
      const int Qb = box_population(g, gp, bx0, y0, z0, TQ_CORE, 0, sub, 4);
      const int Cb = box_population(g, gp, Qb > 0 ? bx0 : -(1 << 20), y0, z0, TQ_CORE, 1, sub, 4);
      const bool fits = Qb > 0 && Cb <= TQ_CMAX;
      emit_items(sub == 0 && fits, Cb < TQ_SLOW_FACTOR * k, bx0, y0, z0, TQ_CORE, Qb, lane, n, items, ctrl);
      deep_boxes = __ballot_sync(FULL, sub == 0 && Qb > 0 && !fits);
    }
    for (; deep_boxes; deep_boxes &= deep_boxes - 1) {
      const int bi = (__ffs(deep_boxes) - 1) >> 2;
      const int x0 = (rbx + bi) * TQ_CORE;
      // 8 children of edge TQ_CORE/2, 4 lanes each
      const int h = TQ_CORE / 2;
      const int ch = lane >> 2, sub = lane & 3;
      const int cx0 = x0 + (ch & 1) * h, cy0 = y0 + ((ch >> 1) & 1) * h, cz0 = z0 + (ch >> 2) * h;
      const int Qc = box_population(g, gp, cx0, cy0, cz0, h, 0, sub, 4);
      const int Cc = box_population(g, gp, cx0, cy0, cz0, h, 1, sub, 4);
      const bool fits = Cc <= TQ_CMAX;
      emit_items(sub == 0 && Qc > 0 && fits, false, cx0, cy0, cz0, h, Qc, lane, n, items, ctrl);
      unsigned deep = __ballot_sync(FULL, sub == 0 && Qc > 0 && !fits);
      for (; deep; deep &= deep - 1) {
        const int l = __ffs(deep) - 1;
        const int px = __shfl_sync(FULL, cx0, l), py = __shfl_sync(FULL, cy0, l), pz = __shfl_sync(FULL, cz0, l);
        // 8 single cells of that child; whether their radius-1 tile fits is left to the tile kernel
        const int gx = px + (ch & 1), gy = py + ((ch >> 1) & 1), gz = pz + (ch >> 2);
        const int Qg = box_population(g, gp, gx, gy, gz, 1, 0, sub, 4);
        emit_items(sub == 0 && Qg > 0, false, gx, gy, gz, 1, Qg, lane, n, items, ctrl);
      }
    }
  }
}

// one pass over the tile positions [c, cend): every point closer than T2 goes into the lane's list column (branch-free:
// non-passing candidates land in the dump row).  When a lane's list is about to fill up it LOWERS its own threshold and
// keeps the entries below it — everything dropped, and everything rejected from then on, is farther than the final T2,
// so the list still holds every tile point below the threshold the lane ends with.  T2 < 0 switches a lane off.
#ifndef TQ_TARGET_EXTRA
#define TQ_TARGET_EXTRA 14     // first guesses aim at k + this many collected points (C2, with the warp-wide shrink: 10 0.572, 12 0.517, 14 0.483, 16 0.481, 18 0.495, 20 0.512 ms)
#endif
// thresholds are kept on the lattice of the list entries: 9 low mantissa bits zero (rounded towards zero)
__device__ __forceinline__ float lattice_floor(float t) { return __uint_as_float(__float_as_uint(t) & ~TQ_POS_MASK); }
struct Shrunk { float T2; int cnt; };
#ifndef TQ_SHRINK_F
#define TQ_SHRINK_F 0.75f
#endif
#ifndef TQ_COOP_SHRINK
#define TQ_COOP_SHRINK 1
#endif
#if TQ_COOP_SHRINK
// The lists of the lanes in `om` are about to fill up: each of them LOWERS its threshold (x 3/4 until at most LCAP-4
// entries survive) and keeps the entries below it.  Done by the whole warp, one list at a time, the list's (at most 40)
// entries spread over the lanes: two loads, two ballots, two stores per round — the lane-by-lane version (one lane
// walking its 36 entries while the other 31 wait) was 12 % of the kernel's instructions, two calls per pass.
// Every lane gets back its own (threshold, count): unchanged unless it was in `om`.
__device__ __noinline__ Shrunk shrink_lists(TileSmem& S, unsigned om, float T2, int cnt) {
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  Shrunk r;
  r.T2 = T2; r.cnt = cnt;
  for (; om; om &= om - 1) {
    const int L = __ffs(om) - 1;
    float t = __shfl_sync(FULL, T2, L);
    int n = __shfl_sync(FULL, cnt, L);
    do {
      t = lattice_floor(t * TQ_SHRINK_F);           // counts grow ~linearly in T^2 on surfaces: about 3/4 survive
      const unsigned tb = __float_as_uint(t);
      const unsigned e0 = lane < n ? S.lst[lane][L] : 0xffffffffu;
      const unsigned e1 = lane + 32 < n ? S.lst[lane + 32][L] : 0xffffffffu;
      const bool k0 = e0 < tb, k1 = e1 < tb;
      const unsigned m0 = __ballot_sync(FULL, k0), m1 = __ballot_sync(FULL, k1);
      __syncwarp();
      if (k0) S.lst[__popc(m0 & lt)][L] = e0;                 // order kept, like the sequential compaction
      if (k1) S.lst[__popc(m0) + __popc(m1 & lt)][L] = e1;
      __syncwarp();
      n = __popc(m0) + __popc(m1);
    } while (n > TQ_LCAP - 4);
    if (lane == L) { r.T2 = t; r.cnt = n; }
  }
  return r;
}
#else
__device__ __noinline__ Shrunk shrink_list(unsigned* col, float T2, int cnt) {
  do {
    T2 = lattice_floor(T2 * 0.75f);           // counts grow ~linearly in T^2 on surfaces: about 3/4 survive
    const unsigned tb = __float_as_uint(T2);
    int pos = 0;
    for (int i = 0; i < cnt; ++i) {
      const unsigned e = col[i * 32];
      if (e < tb) { col[pos * 32] = e; ++pos; }
    }
    cnt = pos;
  } while (cnt > TQ_LCAP - 4);
  Shrunk r;
  r.T2 = T2; r.cnt = cnt;
  return r;
}
#endif
// packed f32x2 arithmetic (sm_100): one instruction works on two candidates.  Every operation is the IEEE round-to-nearest
// one of nanoflann's metric, in the same order — d = ((dx*dx) + dy*dy) + dz*dz with every product and sum rounded on its
// own.  ptxas contracts a packed multiply followed by a packed add into FFMA2 even under -fmad=false, so the sums are
// written as fma(a, 1, b) with a ONE the compiler cannot see through (a kernel argument): round(a * 1 + b) == round(a + b).
__device__ __forceinline__ unsigned long long f2_pack(float lo, float hi) { unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void f2_unpack(unsigned long long v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ unsigned long long f2_sub(unsigned long long a, unsigned long long b) { unsigned long long r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ unsigned long long f2_mul(unsigned long long a, unsigned long long b) { unsigned long long r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ unsigned long long f2_fma(unsigned long long a, unsigned long long b, unsigned long long c) { unsigned long long r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
struct Query2 { unsigned long long x, y, z, one; };   // the query's coordinates and 1.0f, each duplicated into both halves
__device__ __forceinline__ unsigned long long sqdist2_unfused(const Query2& q, unsigned long long px, unsigned long long py, unsigned long long pz) {
#if TQ_PACKED
  const unsigned long long dx = f2_sub(q.x, px), dy = f2_sub(q.y, py), dz = f2_sub(q.z, pz);
  return f2_fma(f2_fma(f2_mul(dx, dx), q.one, f2_mul(dy, dy)), q.one, f2_mul(dz, dz));
#else
  float qx, qy, qz, t, x0, x1, y0, y1, z0, z1;
  f2_unpack(q.x, qx, t); f2_unpack(q.y, qy, t); f2_unpack(q.z, qz, t);
  f2_unpack(px, x0, x1); f2_unpack(py, y0, y1); f2_unpack(pz, z0, z1);
  return f2_pack(sqdist_unfused(qx, qy, qz, x0, y0, z0), sqdist_unfused(qx, qy, qz, x1, y1, z1));
#endif
}

// "write, then advance if it passed": the slot after the last accepted entry is simply overwritten by the next
// candidate, so an offer is one 32-bit shared store plus one predicated pointer bump (row stride 128 B).
// c and cend are even (rows are padded to even lengths).
__device__ __forceinline__ int collect_pass(TileSmem& S, unsigned* const col, int c, int cend, float qx, float qy, float qz, float one, float& T2_io, int cnt) {
  float T2 = T2_io;
  Query2 q;
  q.x = f2_pack(qx, qx); q.y = f2_pack(qy, qy); q.z = f2_pack(qz, qz); q.one = f2_pack(one, one);
  // 32-bit shared-window addresses: the bump is one predicated integer add
  const unsigned a0 = (unsigned)__cvta_generic_to_shared(col);
  unsigned p = a0 + (unsigned)cnt * 128u;
  const unsigned plim = a0 + (unsigned)(TQ_LCAP - 4) * 128u;
#define TQ_OFFER(D, CI)                                                                                      \
  {                                                                                                          \
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(p), "r"((__float_as_uint(D) & ~TQ_POS_MASK) | (unsigned)(CI)) : "memory"); \
    if ((D) < T2) p += 128u;                                                                                 \
  }
#if TQ_COOP_SHRINK
#define TQ_MAYBE_SHRINK()                                                       \
  {                                                                             \
    const unsigned om_ = __ballot_sync(FULL, p > plim);                         \
    if (om_) {                                                                  \
      const Shrunk r = shrink_lists(S, om_, T2, (int)((p - a0) >> 7));          \
      T2 = r.T2;                                                                \
      p = a0 + (unsigned)r.cnt * 128u;                                          \
    }                                                                           \
  }
#else
#define TQ_MAYBE_SHRINK()                                                       \
  if (p > plim) {                                                               \
    const Shrunk r = shrink_list(col, T2, (int)((p - a0) >> 7));                \
    T2 = r.T2;                                                                  \
    p = a0 + (unsigned)r.cnt * 128u;                                            \
  }
#endif
#define TQ_PAIR(CI)                                                                                                     \
  {                                                                                                                     \
    const unsigned long long d01 = sqdist2_unfused(q, *reinterpret_cast<const unsigned long long*>(S.xs + (CI)),        \
                                                   *reinterpret_cast<const unsigned long long*>(S.ys + (CI)),           \
                                                   *reinterpret_cast<const unsigned long long*>(S.zs + (CI)));          \
    float da, db;                                                                                                       \
    f2_unpack(d01, da, db);                                                                                             \
    TQ_OFFER(da, (CI)) TQ_OFFER(db, (CI) + 1)                                                                           \
  }
  if ((c & 2) && c < cend) { TQ_PAIR(c) TQ_MAYBE_SHRINK() c += 2; }   // up to a multiple of four: 128-bit loads from here on
NG_UNROLL(TQ_UNROLL)
  for (; c + 4 <= cend; c += 4) {
    const ulonglong2 X = *reinterpret_cast<const ulonglong2*>(S.xs + c);
    const ulonglong2 Y = *reinterpret_cast<const ulonglong2*>(S.ys + c);
    const ulonglong2 Z = *reinterpret_cast<const ulonglong2*>(S.zs + c);
    const unsigned long long d01 = sqdist2_unfused(q, X.x, Y.x, Z.x), d23 = sqdist2_unfused(q, X.y, Y.y, Z.y);
    float d0, d1, d2, d3;
    f2_unpack(d01, d0, d1);
    f2_unpack(d23, d2, d3);
    TQ_OFFER(d0, c) TQ_OFFER(d1, c + 1) TQ_OFFER(d2, c + 2) TQ_OFFER(d3, c + 3)
    TQ_MAYBE_SHRINK()                                           // room for the next four is guaranteed
  }
  if (c < cend) { TQ_PAIR(c) TQ_MAYBE_SHRINK() }
#undef TQ_PAIR
#undef TQ_OFFER
#undef TQ_MAYBE_SHRINK
  T2_io = T2;
  return (int)((p - a0) >> 7);
}

// v[k-1], v[k] of a register array with a run-time k (forces the array through local memory; generic-k path only)
__device__ __noinline__ uint2 pick_kth(const unsigned* v, int k) { return make_uint2(v[k - 1], v[k]); }

template <int KT>
__global__ void __launch_bounds__(TQ_WARPS * 32) knn_lists_tile_kernel(GridView g, int n, int k_rt, int* __restrict__ nbr,
                                                                        const int4* __restrict__ items, int* __restrict__ ctrl,
                                                                        int* __restrict__ fb_list, unsigned char* __restrict__ fb_flags,
                                                                        unsigned long long* __restrict__ stats,
                                                                        int q_lo, int q_hi, float one /* 1.0f, see sqdist2_unfused */) {
  extern __shared__ __align__(16) unsigned char tq_smem_raw[];
  const int k = KT > 0 ? KT : k_rt;
  TileSmem& S = reinterpret_cast<TileSmem*>(tq_smem_raw)[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  const GridParams gp = load_grid(g.desc);
  const int nslow = ctrl[CT_SLOW];
  const int nitems = nslow + ctrl[CT_ITEMS];
  unsigned st_fb = 0, st_ties = 0, st_tiles = 0, st_passes = 0, st_lanes = 0, st_items = 0;
#ifdef TQ_STATS_DETAIL      // per-radius counters (variants/ build only: they cost 30 registers)
  unsigned st_dec[3] = {0, 0, 0}, st_pass[3] = {0, 0, 0};
  unsigned long long st_cand = 0;
  unsigned long long st_t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(st_t0));
#endif

  for (;;) {
    int w = 0;
    if (lane == 0) w = atomicAdd(ctrl + CT_NEXT, 1);
    w = __shfl_sync(FULL, w, 0);
    if (w >= nitems) break;
    st_items++;
    const int4 item = __ldg(items + (w < nslow ? w : n - 1 - (w - nslow)));
    TQ_CHECK(nitems <= n, "nitems", nitems, n);
    const int x0 = item.x, y0 = item.y, z0 = item.z, sz = item.w & 255, first = (item.w >> 8) * TQ_ITEM;
    // ---- the item's points: positions [first, first + TQ_ITEM) of the box's sz*sz contiguous slot ranges ----
    int ncur = 0;
    {
      int qa = 0, qlen = 0;
      if (lane < sz * sz) {
        const int y = y0 + (lane % sz), z = z0 + (lane / sz);
        if (y < gp.dy && z < gp.dz && x0 < gp.dx) {
          const int* row = g.cell_start + (z * gp.dy + y) * gp.dx;
          qa = __ldg(row + x0);
          qlen = __ldg(row + min(x0 + sz, gp.dx)) - qa;
        }
      }
      const int qinc = warp_incl_scan(qlen, lane);
      const int Q = __shfl_sync(FULL, qinc, 31);
      const int qexcl = qinc - qlen;
      ncur = min(TQ_ITEM, Q - first);
      int nkept = 0;                                       // of those, the ones inside the slot range this launch answers
      for (int t0 = 0; t0 < ncur; t0 += 32) {
        const int t = first + t0 + lane;
        const int j = run_of(qinc, t);
        const int ja = __shfl_sync(FULL, qa, j), je = __shfl_sync(FULL, qexcl, j);
        const int slot = ja + (t - je);
        const bool keep = t0 + lane < ncur && slot >= q_lo && slot < q_hi;
        const unsigned km = __ballot_sync(FULL, keep);
        if (keep) {
          const int pos = nkept + __popc(km & lt);
          S.cur[pos] = slot; S.cur_t[pos] = 0.f; S.cur_lo[pos] = 0.f; S.cur_hi[pos] = -1.f;
        }
        nkept += __popc(km);
      }
      ncur = nkept;
      __syncwarp();
    }
    for (int s = 1; s <= TQ_SMAX && ncur > 0; s *= 2) {
      // ---- stage the tile: cells [x0-s, x0+sz-1+s] x [y0-s, ..] x [z0-s, ..], 32 rows per round ----
      const int ny = sz + 2 * s, nrows = ny * ny;
      const int xl = max(x0 - s, 0), xr = min(x0 + sz - 1 + s, gp.dx - 1) + 1;
      int C = 0;
      bool overflow = false;
      for (int r0 = 0; r0 < nrows; r0 += 32) {
        const int r = r0 + lane;
        int a = 0, b = 0;
        if (r < nrows) {
          const int y = y0 - s + (r % ny), z = z0 - s + (r / ny);
          if (y >= 0 && y < gp.dy && z >= 0 && z < gp.dz) {
            const int* row = g.cell_start + (z * gp.dy + y) * gp.dx;
            a = __ldg(row + xl); b = __ldg(row + xr);
          }
        }
        if (!__any_sync(FULL, b != a)) {
          if (s <= 2 && r < nrows) S.rowoff[r] = C;
          continue;
        }
        const int len = b - a, plen = (len + 1) & ~1;           // rows are padded to even lengths
        const int inc = warp_incl_scan(plen, lane);
        const int Cr = __shfl_sync(FULL, inc, 31);
        if (C + Cr > TQ_CMAX) { overflow = true; break; }
        const int excl = inc - plen;
        if (s <= 2 && r < nrows) S.rowoff[r] = C + excl;
        for (int t0 = 0; t0 < Cr; t0 += 32) {
          const int t = t0 + lane;
          const int j = run_of(inc, t);
          const int ja = __shfl_sync(FULL, a, j), je = __shfl_sync(FULL, excl, j), jl = __shfl_sync(FULL, len, j);
          if (t < Cr) {
            const int off = t - je;
            float4 c = make_float4(INFINITY, 0.f, 0.f, 0.f);    // the padding slot of an odd row
            int p = -1;
            if (off < jl) { p = ja + off; c = __ldg(g.sorted + p); }
            S.xs[C + t] = c.x; S.ys[C + t] = c.y; S.zs[C + t] = c.z; S.slot[C + t] = p;
          }
        }
        C += Cr;
      }
      if (overflow) break;                                    // the tile does not fit: warp search for what is left
      if (C < k) continue;                                    // too sparse at this radius
      if (s <= 2 && lane == 0) S.rowoff[nrows] = C;
      __syncwarp();
      st_tiles++;
      // ---- answer the points from the tile, 32 at a time, one collection pass each; a point whose count misses
      //      the window re-queues itself with a rescaled threshold, so retries share passes with other points ----
      const float guess0 = (float)(k + TQ_TARGET_EXTRA) * (float)(ny * ny) * gp.cell * gp.cell / (3.14159265f * (float)C);
      int nnxt = 0;
      float prevT = 0.f;
      for (int round = 0; round < 8 && ncur > 0; ++round) {
        int nre = 0;
        for (int t0 = 0; t0 < ncur; t0 += 32) {
          const int t = t0 + lane;
          const bool has = t < ncur;
          int slot = has ? S.cur[t] : -1;
          float T2 = has ? S.cur_t[t] : 0.f;
          float lo = has ? S.cur_lo[t] : 0.f, hi = has ? S.cur_hi[t] : -1.f;
          float4 qp = make_float4(0.f, 0.f, 0.f, 0.f);
          if (has) qp = __ldg(g.sorted + slot);
          const bool me = has && isfinite(qp.x) && isfinite(qp.y) && isfinite(qp.z);
          if (has && !me)
            for (int j = 0; j < k; ++j) nbr[(size_t)slot * k + j] = -1;
          // the (y,z) rows of cells this batch's points lie in: only tile rows within s of them can hold neighbours
          // closer than the provable radius, so the pass scans that sub-tile (whole tile above radius 2)
          int ylo = 0, yhi = ny - 1, zlo = 0, zhi = ny - 1;
          if (s <= 2) {
            const int yy = cell_coord(qp.y, gp.oy, gp.inv, gp.dy) - (y0 - s), zz = cell_coord(qp.z, gp.oz, gp.inv, gp.dz) - (z0 - s);
            ylo = max(__reduce_min_sync(FULL, me ? yy : ny) - s, 0);
            yhi = min(__reduce_max_sync(FULL, me ? yy : -1) + s, ny - 1);
            zlo = max(__reduce_min_sync(FULL, me ? zz : ny) - s, 0);
            zhi = min(__reduce_max_sync(FULL, me ? zz : -1) + s, ny - 1);
          }
          float m2 = FLT_MAX;
          {
            const float m = box_face_distance(gp, x0 - s, x0 + sz - 1 + s, y0 - s + ylo, y0 - s + yhi, z0 - s + zlo, z0 - s + zhi, qp.x, qp.y, qp.z);
            if (m != FLT_MAX) m2 = m > 0.f ? m * m * 0.999999f : 0.f;
            m2 = lattice_floor(m2);
          }
          // first guess: 1.4 x the k-th distance this lane found last in this tile, else the radius holding k+8
          // points at the tile's surface density (a planar cut through the tile covers ~ny*ny cells)
          if (!(T2 > 0.f)) T2 = prevT > 0.f ? prevT * (float)(k + TQ_TARGET_EXTRA) / (float)k : guess0;
          T2 = lattice_floor(fminf(T2, m2));
          const bool active = me && m2 > 0.f && T2 > 0.f;
          st_passes++;
          st_lanes += __popc(__ballot_sync(FULL, active));
#ifdef TQ_STATS_DETAIL
          st_pass[s == 1 ? 0 : (s == 2 ? 1 : 2)]++;
          if (stats != nullptr) st_cand += s <= 2 ? (unsigned)max(S.rowoff[zhi * ny + yhi + 1] - S.rowoff[zlo * ny + ylo], 0) : (unsigned)C;
#endif
          int c_now = 0;
          const float T2_asked = T2;
          {
            float Tc = active ? T2 : -1.f;      // may come back lower: the lane shrank its list on the way
            if (s <= 2) {
              for (int zr = zlo; zr <= zhi && yhi >= ylo; ++zr)
                c_now = collect_pass(S, &S.lst[0][lane], S.rowoff[zr * ny + ylo], S.rowoff[zr * ny + yhi + 1], qp.x, qp.y, qp.z, one, Tc, c_now);
            } else {
              c_now = collect_pass(S, &S.lst[0][lane], 0, C, qp.x, qp.y, qp.z, one, Tc, 0);
            }
            if (active) T2 = Tc;
          }
          const bool good = active && c_now >= k && c_now <= TQ_LCAP;
          // too few even at the largest provable radius (or no provable radius at all): needs a larger tile
          const bool grow = me && (!active || (c_now < k && T2 >= m2));
          const bool retry = active && !good && !grow;
          // ---- exactly k of the collected points: the lane sorts its list entries in registers (a fixed
          //      compare-exchange network: no data-dependent loop, every lane of the warp does the same work) and keeps
          //      those up to the k-th.  Entries compare by distance down to the lattice; when the k-th and the (k+1)-th
          //      fall on the same lattice value (an exact tie, or two points closer than 2^-14 relative) the set cannot
          //      be decided here: those (rare) points take the warp search ----
          bool decided = good;
          bool tie = false;
          bool needs_fix = false;
          float kth = T2;
          {
            // generic k keeps the old rule (select only when more than k were collected, deliver in list order; the
            // covariance kernel orders them); k = 10 / 20 always go through the network and deliver SORTED lists
            const bool searching = good && (KT > 0 || c_now > k);
            const bool any_search = __any_sync(FULL, searching);
            if (any_search) {
              static_assert(TQ_LCAP == 40 || TQ_LCAP == 32, "the selection networks are generated for 32 and 40 wires");
              unsigned v[TQ_LCAP];
#pragma unroll
              for (int i = 0; i < TQ_LCAP; ++i) v[i] = (searching && i < c_now) ? S.lst[i][lane] : 0xffffffffu;
#define NG_UCAS(A, B) { const unsigned lo_ = min(v[A], v[B]), hi_ = max(v[A], v[B]); v[A] = lo_; v[B] = hi_; }
#if TQ_LCAP == 40
              NGICP_SORTNET_40(NG_UCAS)
#else
              NGICP_SORTNET_32(NG_UCAS)
#endif
#undef NG_UCAS
              // the k-th and (k+1)-th smallest: static register indices when k is a template argument (10 and 20, what
              // DLO uses); a run-time k goes through a small local array (one copy of the network either way — indexing
              // the registers with a run-time k made the compiler clone the whole network per value of k)
              unsigned vk, vk1;
              if (KT > 0) { vk = v[KT > 0 ? KT - 1 : 0]; vk1 = v[KT > 0 ? KT : 0]; }
              else { const uint2 pk = pick_kth(v, k); vk = pk.x; vk1 = pk.y; }
              unsigned bound = 0u;
              if (searching) {
                if ((vk >> TQ_POS_BITS) == (vk1 >> TQ_POS_BITS)) { tie = true; decided = false; st_ties++; }
                else { bound = ((vk >> TQ_POS_BITS) + 1u) << TQ_POS_BITS; kth = __uint_as_float(vk & ~TQ_POS_MASK); }
              }
              if (KT > 0) {
                // the k nearest back into the lane's column in ascending lattice order = ascending exact distance, unless
                // two neighbours share a lattice value (an exact tie or closer than 2^-14 relative): those points are
                // delivered too but flagged, and the covariance fix-up orders them by exact (distance, slot)
                // Written out by the lane itself, straight from the registers (KT/4 128-bit stores into its own row of
                // nbr; the rows of a batch's queries are neighbours in memory most of the time) — the earlier write-out
                // went back through the shared list and took one dependent round per decided query.
                bool near = false;
                constexpr int KW = KT > 0 ? KT : 4;
                int o[KW];
#pragma unroll
                for (int i = 0; i < KW; ++i) {
                  o[i] = S.slot[v[i] & TQ_POS_MASK];
                  if (i > 0) near = near || ((v[i - 1] >> TQ_POS_BITS) == (v[i] >> TQ_POS_BITS));
                }
                needs_fix = searching && !tie && near;
                if (searching && !tie) {
                  int* row = nbr + (size_t)slot * KW;
                  if (KW % 4 == 0) {
#pragma unroll
                    for (int i = 0; i < KW / 4; ++i) reinterpret_cast<int4*>(row)[i] = make_int4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
                  } else if (KW % 2 == 0) {
#pragma unroll
                    for (int i = 0; i < KW / 2; ++i) reinterpret_cast<int2*>(row)[i] = make_int2(o[2 * i], o[2 * i + 1]);
                  } else {
#pragma unroll
                    for (int i = 0; i < KW; ++i) row[i] = o[i];
                  }
                }
              } else {
                const bool compact = searching && !tie;
                int pos = 0;
#pragma unroll
                for (int i = 0; i < TQ_LCAP; ++i) {
                  const unsigned e = S.lst[i][lane];
                  if (compact && i < c_now && e < bound) { S.lst[pos][lane] = e; ++pos; }
                }
              }
            }
          }
          if (decided) prevT = kth;
          const unsigned dmask = __ballot_sync(FULL, decided);
#ifdef TQ_STATS_DETAIL
          st_dec[s == 1 ? 0 : (s == 2 ? 1 : 2)] += __popc(dmask);
#endif
          __syncwarp();
          // ---- generic k: coalesced write-out through the shared list, one query per step, lane j writes the j-th neighbour ----
          for (unsigned mm = KT > 0 ? 0u : dmask; mm; mm &= mm - 1) {
            const int l = __ffs(mm) - 1;
            const int sl = __shfl_sync(FULL, slot, l);
            TQ_CHECK(lane >= k || ((S.lst[lane][l] & TQ_POS_MASK) < (unsigned)C && S.slot[S.lst[lane][l] & TQ_POS_MASK] >= 0), "tilepos", (int)(S.lst[lane][l] & TQ_POS_MASK), C);
            if (lane < k) nbr[(size_t)sl * k + lane] = S.slot[S.lst[lane][l] & TQ_POS_MASK];
          }
          __syncwarp();
          fix_append(__ballot_sync(FULL, needs_fix), slot, lane, n, fb_list, ctrl + CT_FIX, fb_flags);
          // ---- the rest: ties to the warp search, growers to the next radius, retries back into the queue ----
          const unsigned tm = __ballot_sync(FULL, tie);
          st_fb += __popc(tm);
          fb_append(tm, slot, lane, fb_list, ctrl + CT_REST, fb_flags);
          const unsigned gm = __ballot_sync(FULL, grow);
          if (grow) S.nxt[nnxt + __popc(gm & lt)] = slot;
          nnxt += __popc(gm);
          const unsigned rm = __ballot_sync(FULL, retry);
          if (retry) {
            // counts grow ~linearly in T^2 on surfaces: aim at k+8 again, inside the bracket; never above the provable radius
            // the count at T2 was too small; if the lane lowered its threshold on the way, the asked one was too large
            if (c_now < k) { lo = T2; if (T2 < T2_asked) hi = hi > 0.f ? fminf(hi, T2_asked) : T2_asked; } else hi = T2;
            float Tn = T2 * (float)(k + TQ_TARGET_EXTRA) / (float)max(c_now, 2);
            if (Tn <= lo || (hi > 0.f && Tn >= hi)) Tn = hi > 0.f ? 0.5f * (lo + hi) : T2 * 2.f;
            Tn = lattice_floor(fminf(Tn, m2));
            const int pos = nre + __popc(rm & lt);          // nre <= t0: never overtakes the reads
            S.cur[pos] = slot;
            S.cur_t[pos] = Tn;
            S.cur_lo[pos] = lo;
            S.cur_hi[pos] = hi;
          }
          nre += __popc(rm);
          __syncwarp();
        }
        ncur = nre;
      }
      // still retrying after 8 rounds (pathological distributions): let the next radius / the warp search decide
      for (int t0 = 0; t0 < ncur; t0 += 32) {
        const bool has = t0 + lane < ncur;
        const int slot = has ? S.cur[t0 + lane] : -1;
        const unsigned m = __ballot_sync(FULL, has);
        if (has) S.nxt[nnxt + __popc(m & lt)] = slot;
        nnxt += __popc(m);
      }
      __syncwarp();
      for (int t = lane; t < nnxt; t += 32) { S.cur[t] = S.nxt[t]; S.cur_t[t] = 0.f; S.cur_lo[t] = 0.f; S.cur_hi[t] = -1.f; }
      ncur = nnxt;
      __syncwarp();
    }
    // could not be decided inside a tile: warp search
    for (int t0 = 0; t0 < ncur; t0 += 32) {
      const bool has = t0 + lane < ncur;
      const int slot = has ? S.cur[t0 + lane] : -1;
      const unsigned m = __ballot_sync(FULL, has);
      st_fb += __popc(m);
      fb_append(m, slot, lane, fb_list, ctrl + CT_REST, fb_flags);
    }
    __syncwarp();
  }
  if (stats != nullptr && lane == 0) {
    atomicAdd(stats + ST_FALLBACK, (unsigned long long)st_fb);
    atomicAdd(stats + ST_TIES, (unsigned long long)st_ties);
    atomicAdd(stats + ST_TILES, (unsigned long long)st_tiles);
    atomicAdd(stats + ST_PASSES, (unsigned long long)st_passes);
    atomicAdd(stats + ST_LANES, (unsigned long long)st_lanes);
    atomicAdd(stats + ST_ITEMS, (unsigned long long)st_items);
#ifdef TQ_STATS_DETAIL
    atomicAdd(stats + ST_DEC1, (unsigned long long)st_dec[0]); atomicAdd(stats + ST_DEC2, (unsigned long long)st_dec[1]);
    atomicAdd(stats + ST_DECHI, (unsigned long long)st_dec[2]);
    atomicAdd(stats + ST_PASS1, (unsigned long long)st_pass[0]); atomicAdd(stats + ST_PASS2, (unsigned long long)st_pass[1]);
    atomicAdd(stats + ST_PASSHI, (unsigned long long)st_pass[2]);
    atomicAdd(stats + ST_CAND, st_cand);
    unsigned long long st_t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(st_t1));
    atomicAdd(stats + ST_TSUM, st_t1 - st_t0);
    atomicMax(stats + ST_TEND, st_t1);
    atomicMin(stats + ST_TSTART, st_t0);      // the host presets this word to all ones
    atomicAdd(stats + ST_TWARPS, 1ull);
#endif
  }
}

// the points the tile kernel could not decide: one warp per listed point, growing-cube search (same result definition)
__global__ void __launch_bounds__(64) knn_lists_rest_kernel(GridView g, int k, int* __restrict__ nbr, const int* __restrict__ ctrl,
                                                                                     const int* __restrict__ fb_list) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const GridParams gp = load_grid(g.desc);
  const int total = ctrl[CT_REST];
  for (int i = warp; i < total; i += nwarps) {
    const int q = fb_list[i];
    const float4 qp = __ldg(g.sorted + q);
    WarpTopK rs;
    rs.init(k, lane);
    if (isfinite(qp.x) && isfinite(qp.y) && isfinite(qp.z)) grid_search_warp<WarpTopK, false, 4>(g, gp, qp.x, qp.y, qp.z, FLT_MAX, rs, k >= 4);
    if (lane < k) nbr[(size_t)q * k + lane] = rs.p;
  }
}

// K3: one thread per point — mean, covariance / k, regularisation, all fp64 (nano_gicp_impl.hpp:315-353).
// The sums run over the k neighbours in ascending (squared distance, sorted slot) order: nearestKSearch returns them
// ascending (nanoflann_impl.hpp:184-211) and the reference adds them up in that order (:315-321), so on neighbourhoods
// without exact distance ties the fp64 mean and covariance reproduce the reference's bits whichever kNN kernel made the
// list (the tile kernel delivers the SET in slot order; the warp search delivers it sorted, ties in visiting order).
// KT > 0: k known at compile time (10 and 20, the values DLO uses) — keys in registers, k^2 unrolled rank computation.
// SORTED: the list is already in summation order (the tile kernel's k = 10 / 20 lists; points it could not order exactly
// are flagged and left to cov_rest_kernel) — no distances, no keys, no sorting network.
template <int KT, bool SORTED>
__device__ __forceinline__ void cov_point(const GridView& g, int n, int k_rt, int method, const int* __restrict__ nbr, double* __restrict__ covs6,
                                          int q, int* __restrict__ idx_out, float* __restrict__ d2_out) {
  constexpr int KA = KT > 0 ? KT : (KT == 0 ? KNN_MAX_K : KNN_WIDE_MAX_K);   // KT = -1: the wide lists (k up to 128, local-memory keys)
  const int k = KT > 0 ? KT : k_rt;
  const int* my = nbr + (size_t)q * k;
  const float4 qp = __ldg(g.sorted + q);
  const int orig = __float_as_int(qp.w);
  int ord[KA];          // neighbour slots in summation order (dynamically indexed: local memory, L1 resident)
  if (KT > 0 && SORTED) {
#pragma unroll
    for (int j = 0; j < KA; ++j) ord[j] = __ldg(my + j);
  } else if (KT > 0) {
    // keys = (bits of the squared distance) << 32 | sorted slot: non-negative floats order like their bit patterns, the
    // slot breaks exact ties (slots follow (cell, original index), the same for every kNN kernel and every slicing)
    unsigned long long key[KA];
    bool in_order = true;
#pragma unroll
    for (int j = 0; j < KA; ++j) {
      const int p = __ldg(my + j);
      TQ_CHECK(p < n, "nbr", p, q);
      key[j] = 0xffffffff00000000ull | (unsigned)j;           // no neighbour: sorts last, decodes to -1
      if (p >= 0) {
        const float4 c = __ldg(g.sorted + p);
        key[j] = ((unsigned long long)__float_as_uint(sqdist_unfused(qp.x, qp.y, qp.z, c.x, c.y, c.z)) << 32) | (unsigned)p;
      }
      if (j > 0) in_order = in_order && key[j - 1] <= key[j];
    }
    if (!in_order) {
#define NG_CAS(A, B) { const unsigned long long ka = key[A], kb = key[B]; const bool sw = kb < ka; key[A] = sw ? kb : ka; key[B] = sw ? ka : kb; }
      if (KT == 10) { NGICP_SORTNET_10(NG_CAS) }
      else { NGICP_SORTNET_20(NG_CAS) }
#undef NG_CAS
    }
#pragma unroll
    for (int j = 0; j < KA; ++j) ord[j] = (key[j] >> 32) == 0xffffffffull ? -1 : (int)(unsigned)key[j];
  } else {
    unsigned long long key[KA];
    for (int j = 0; j < k; ++j) {
      const int p = __ldg(my + j);
      key[j] = 0xffffffff00000000ull | (unsigned)j;
      if (p >= 0) {
        const float4 c = __ldg(g.sorted + p);
        key[j] = ((unsigned long long)__float_as_uint(sqdist_unfused(qp.x, qp.y, qp.z, c.x, c.y, c.z)) << 32) | (unsigned)p;
      }
    }
    for (int j = 0; j < k; ++j) {       // rank by counting (keys are distinct)
      int r = 0;
      for (int i = 0; i < k; ++i) r += key[i] < key[j] ? 1 : 0;
      ord[r] = __ldg(my + j);
    }
  }
  if (idx_out != nullptr) {   // test hook (ngicp_cov_neighbors): the list as it is summed, original indices, caller's point order
    for (int r = 0; r < k; ++r) {
      const int p = ord[r];
      int oi = -1;
      float dd = -1.f;
      if (p >= 0) { const float4 c = __ldg(g.sorted + p); oi = __float_as_int(c.w); dd = sqdist_unfused(qp.x, qp.y, qp.z, c.x, c.y, c.z); }
      idx_out[(size_t)orig * k + r] = oi;
      d2_out[(size_t)orig * k + r] = dd;
    }
    return;
  }
  double mx = 0.0, my_ = 0.0, mz = 0.0;
  for (int r = 0; r < k; ++r) {
    const int p = ord[r];
    if (p >= 0) { const float4 c = __ldg(g.sorted + p); mx += (double)c.x; my_ += (double)c.y; mz += (double)c.z; }
  }
  const double kd = (double)k;
  mx /= kd; my_ /= kd; mz /= kd;
  double c[6] = {0, 0, 0, 0, 0, 0};
  for (int r = 0; r < k; ++r) {
    const int p = ord[r];
    double x = -mx, y = -my_, z = -mz;   // a missing neighbour is a zero column minus the mean, like the reference's zero-initialised matrix would be
    if (p >= 0) { const float4 v = __ldg(g.sorted + p); x += (double)v.x; y += (double)v.y; z += (double)v.z; }
    c[0] += x * x; c[1] += x * y; c[2] += x * z; c[3] += y * y; c[4] += y * z; c[5] += z * z;
  }
#pragma unroll
  for (int i = 0; i < 6; i++) c[i] /= kd;
  double out[6];
  regularize_cov(c, method, out);
  double* dst = covs6 + (size_t)orig * 6;
#pragma unroll
  for (int i = 0; i < 6; i++) dst[i] = out[i];
}

// main launch: one thread per sorted slot of [q_lo, q_hi); points flagged for the warp search are left to cov_rest_kernel
#ifndef K3_MINB
#define K3_MINB 4      // resident blocks per SM the covariance kernel is compiled for (registers: 4 -> 128, 5 -> 96, 6 -> 80)
#endif
template <int KT, bool SORTED>
__global__ void __launch_bounds__(128, K3_MINB) cov_from_lists_kernel(GridView g, int n, int k_rt, int method, const int* __restrict__ nbr,
                                                             double* __restrict__ covs6, int q_lo, int q_hi,
                                                             const unsigned char* __restrict__ skip_flags,
                                                             int* __restrict__ idx_out, float* __restrict__ d2_out) {
  const int q = q_lo + blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= q_hi || q >= n) return;
  if (skip_flags != nullptr && skip_flags[q]) return;
  cov_point<KT, SORTED>(g, n, k_rt, method, nbr, covs6, q, idx_out, d2_out);
}
// the listed points only (after knn_lists_rest_kernel has answered them); runs beside the main launch on a side stream
template <int KT>
__global__ void __launch_bounds__(128) cov_rest_kernel(GridView g, int n, int k_rt, int method, const int* __restrict__ nbr,
                                                       double* __restrict__ covs6, const int* __restrict__ ctrl, const int* __restrict__ fb_list) {
  const int nrest = ctrl[CT_REST], total = nrest + ctrl[CT_FIX];     // warp-search list from the front, order fix-ups from the back
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x)
    cov_point<KT, false>(g, n, k_rt, method, nbr, covs6, i < nrest ? fb_list[i] : fb_list[n - 1 - (i - nrest)], nullptr, nullptr);
}

static void launch_cov_kernel(const DevCloud& c, int k, int method, const int* nbr, double* covs6, int q_lo, int q_hi, const unsigned char* skip,
                              int* idx_out, float* d2_out, cudaStream_t st, bool sorted = false) {
  const int nq = q_hi - q_lo;
  const dim3 grid((nq + 127) / 128), block(128);
  if (k == 10 && sorted) cov_from_lists_kernel<10, true><<<grid, block, 0, st>>>(c.view(), c.n, k, method, nbr, covs6, q_lo, q_hi, skip, idx_out, d2_out);
  else if (k == 20 && sorted) cov_from_lists_kernel<20, true><<<grid, block, 0, st>>>(c.view(), c.n, k, method, nbr, covs6, q_lo, q_hi, skip, idx_out, d2_out);
  else if (k == 10) cov_from_lists_kernel<10, false><<<grid, block, 0, st>>>(c.view(), c.n, k, method, nbr, covs6, q_lo, q_hi, skip, idx_out, d2_out);
  else if (k == 20) cov_from_lists_kernel<20, false><<<grid, block, 0, st>>>(c.view(), c.n, k, method, nbr, covs6, q_lo, q_hi, skip, idx_out, d2_out);
  else if (k > KNN_MAX_K) cov_from_lists_kernel<-1, false><<<grid, block, 0, st>>>(c.view(), c.n, k, method, nbr, covs6, q_lo, q_hi, skip, idx_out, d2_out);
  else cov_from_lists_kernel<0, false><<<grid, block, 0, st>>>(c.view(), c.n, k, method, nbr, covs6, q_lo, q_hi, skip, idx_out, d2_out);
  note_launches(1);
}
static void launch_cov_rest_kernel(const DevCloud& c, int k, int method, const int* nbr, double* covs6, const int* ctrl, const int* fb_list, int blocks,
                                   cudaStream_t st) {
  if (k == 10) cov_rest_kernel<10><<<blocks, 128, 0, st>>>(c.view(), c.n, k, method, nbr, covs6, ctrl, fb_list);
  else if (k == 20) cov_rest_kernel<20><<<blocks, 128, 0, st>>>(c.view(), c.n, k, method, nbr, covs6, ctrl, fb_list);
  else cov_rest_kernel<0><<<blocks, 128, 0, st>>>(c.view(), c.n, k, method, nbr, covs6, ctrl, fb_list);
  note_launches(1);
}

cudaError_t launch_export_neighbors(const DevCloud& c, int k, const int* nbr_scratch, int* idx_out, float* d2_out, cudaStream_t st) {
  if (c.n <= 0) return cudaSuccess;
  launch_cov_kernel(c, k, 0, nbr_scratch, nullptr, 0, c.n, nullptr, idx_out, d2_out, st);
  return cudaGetLastError();
}

void knn_prime_kernels() {
  cudaFuncAttributes fa;
  cudaFuncGetAttributes(&fa, knn_query_kernel);
  cudaFuncGetAttributes(&fa, knn_lists_kernel);
  cudaFuncGetAttributes(&fa, knn_plan_kernel);
  cudaFuncGetAttributes(&fa, brick_clear_kernel);
  cudaFuncGetAttributes(&fa, brick_mark_kernel);
  cudaFuncGetAttributes(&fa, knn_zero_kernel);
  cudaFuncGetAttributes(&fa, knn_lists_tile_kernel<0>);
  cudaFuncGetAttributes(&fa, knn_lists_tile_kernel<10>);
  cudaFuncGetAttributes(&fa, knn_lists_tile_kernel<20>);
  cudaFuncGetAttributes(&fa, knn_lists_rest_kernel);
  cudaFuncGetAttributes(&fa, knn_query_wide_kernel);
  cudaFuncGetAttributes(&fa, knn_lists_wide_kernel);
  cudaFuncGetAttributes(&fa, cov_from_lists_kernel<-1, false>);
  cudaFuncGetAttributes(&fa, cov_from_lists_kernel<0, false>);
  cudaFuncGetAttributes(&fa, cov_from_lists_kernel<10, false>);
  cudaFuncGetAttributes(&fa, cov_from_lists_kernel<20, false>);
  cudaFuncGetAttributes(&fa, cov_from_lists_kernel<10, true>);
  cudaFuncGetAttributes(&fa, cov_from_lists_kernel<20, true>);
  cudaFuncGetAttributes(&fa, cov_rest_kernel<0>);
  cudaFuncGetAttributes(&fa, cov_rest_kernel<10>);
  cudaFuncGetAttributes(&fa, cov_rest_kernel<20>);
  cudaGetLastError();
}

cudaError_t launch_knn_queries(const DevCloud& c, const float4* queries, int nq, int k, int* idx, float* d2, cudaStream_t st) {
  if (nq <= 0) return cudaSuccess;
  int blocks = (nq + KC_WARPS - 1) / KC_WARPS;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (k > KNN_MAX_K) knn_query_wide_kernel<<<blocks, KC_THREADS, 0, st>>>(c.view(), queries, nq, k, idx, d2);
  else knn_query_kernel<<<blocks, KC_THREADS, 0, st>>>(c.view(), queries, nq, k, idx, d2);
  note_launches(1);
  return cudaGetLastError();
}

// scratch layout (ints): nbr[n*k] | control words[8] | warp-search list[n] | (16-byte aligned) work items int4[n] | warp-search flags (n bytes)
static inline size_t items_offset_ints(int n, int k) { return (((size_t)n * k + CT_N + (size_t)n) + 3) & ~(size_t)3; }
static inline size_t flags_offset_ints(int n, int k) { return items_offset_ints(n, k) + 4 * (size_t)n + 16; }
static inline size_t brick_offset_ints(int n, int k) { return flags_offset_ints(n, k) + ((size_t)n + 3) / 4 + 4; }
size_t covariance_scratch_ints(int n, int k, int table_cap) { return brick_offset_ints(n, k) + (size_t)(brick_flag_bytes(table_cap) / 4) + 4; }

cudaError_t launch_covariances(const DevCloud& c, int k, int method, int* nbr_scratch, double* covs6, int table_cap, cudaStream_t st,
                               int part, int nparts, int knn_path, int tile_min_points, const CovSideStream* side) {
  if (c.n <= 0) return cudaSuccess;
  // the sorted slots this launch answers: everything, or part `part` of `nparts` equal slices (the rest of covs6 is zeroed
  // so that the slices of all parts add up to the full result)
  int q_lo = 0, q_hi = c.n;
  if (nparts > 1) {
    q_lo = (int)((long long)c.n * part / nparts);
    q_hi = (int)((long long)c.n * (part + 1) / nparts);
    cudaError_t ez = cudaMemsetAsync(covs6, 0, sizeof(double) * 6 * (size_t)c.n, st);
    if (ez != cudaSuccess) return ez;
  }
  const int nq = q_hi - q_lo;
  if (nq <= 0) return cudaSuccess;
  // Two exact paths (ngicp_params::knn_path).  One warp per point (knn_lists_kernel): massively parallel, best for scans.
  // Cell-major tiles (plan + tile + rest launches): half the instructions per point but a longer serial path per warp,
  // best for submaps — measured on the C2 submap (500k points, k=20) 0.63 ms against 0.82 ms, on a 22k-point scan 0.19 ms
  // against 0.10 ms (DESIGN.md section 3).  AUTO takes the tiles from knn_tile_min_points (131072) points on.
  // k > 32 has one path, whatever knn_path says: the warp search with the shared-memory result set.
  const bool warp_only = k > KNN_MAX_K || knn_path == NGICP_KNN_WARP || (knn_path != NGICP_KNN_TILE && c.n < tile_min_points);
  static const bool want_stats = getenv("NGICP_KNN_STATS") != nullptr;
  if (warp_only) {
    if (k > KNN_MAX_K) knn_lists_wide_kernel<<<(nq + KC_WARPS - 1) / KC_WARPS, KC_THREADS, 0, st>>>(c.view(), c.n, k, nbr_scratch, q_lo, q_hi);
    else knn_lists_kernel<<<(nq + KC_WARPS - 1) / KC_WARPS, KC_THREADS, 0, st>>>(c.view(), c.n, k, nbr_scratch, q_lo, q_hi);
    note_launches(1);
  } else {
    static std::mutex attr_mutex;
    static bool attr_set[64] = {};
    static int blocks_per_sm[64] = {};
    static int sm_count[64] = {};
    const size_t smem = sizeof(TileSmem) * TQ_WARPS;
    int dev = 0;
    cudaGetDevice(&dev);
    const int di = dev & 63;
    {
      std::lock_guard<std::mutex> lock(attr_mutex);
      if (!attr_set[di]) {
        cudaError_t e = cudaFuncSetAttribute(knn_lists_tile_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(knn_lists_tile_kernel<10>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(knn_lists_tile_kernel<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        int occ[3] = {0, 0, 0};
        if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[0], knn_lists_tile_kernel<0>, TQ_WARPS * 32, smem)) != cudaSuccess) return e;
        if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[1], knn_lists_tile_kernel<10>, TQ_WARPS * 32, smem)) != cudaSuccess) return e;
        if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[2], knn_lists_tile_kernel<20>, TQ_WARPS * 32, smem)) != cudaSuccess) return e;
        blocks_per_sm[di] = occ[0] < occ[1] ? (occ[0] < occ[2] ? occ[0] : occ[2]) : (occ[1] < occ[2] ? occ[1] : occ[2]);
        if ((e = cudaDeviceGetAttribute(&sm_count[di], cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
        if (blocks_per_sm[di] < 1) blocks_per_sm[di] = 1;
        attr_set[di] = true;
      }
    }
    int* ctrl = nbr_scratch + (size_t)c.n * k;
    int* fb_list = ctrl + CT_N;
    int4* items = reinterpret_cast<int4*>(nbr_scratch + items_offset_ints(c.n, k));
    items = reinterpret_cast<int4*>((reinterpret_cast<uintptr_t>(items) + 15) & ~(uintptr_t)15);
    unsigned char* fb_flags = reinterpret_cast<unsigned char*>(nbr_scratch + flags_offset_ints(c.n, k));
    cudaError_t e = cudaSuccess;
    knn_zero_kernel<<<148, 256, 0, st>>>(ctrl, reinterpret_cast<unsigned*>(fb_flags), (c.n + 3) / 4);
    note_launches(1);
    unsigned long long* stats = nullptr;
    if (want_stats) {
      if (cudaMalloc(&stats, ST_N * sizeof(unsigned long long)) != cudaSuccess) return cudaGetLastError();
      cudaMemsetAsync(stats, 0, ST_N * sizeof(unsigned long long), st);
      cudaMemsetAsync(stats + ST_TSTART, 0xff, sizeof(unsigned long long), st);
    }
    // plan: one warp per run of boxes; the grid dimensions live on the device, so cover the table capacity
    // (runs of 8 boxes above 32768 boxes, single boxes below)
    const long long max_boxes = ((long long)table_cap + 63) / 64;
    long long plan_warps = max_boxes > 32768 ? (max_boxes + 7) / 8 + 1024 : max_boxes + 1024;
    unsigned char* bricks = reinterpret_cast<unsigned char*>(nbr_scratch + brick_offset_ints(c.n, k));
    const long long brick_cap = brick_flag_bytes(table_cap);
    if (c.bricks.p && c.bricks.bytes >= (size_t)brick_cap) {
      bricks = c.bricks.as<unsigned char>();            // filled by the fused index kernel
    } else {
      brick_clear_kernel<<<148 * 2, 256, 0, st>>>(c.view(), bricks, brick_cap);
      brick_mark_kernel<<<(c.n + 1023) / 1024, 256, 0, st>>>(c.view(), c.n, bricks, brick_cap);
      note_launches(2);
    }
    knn_plan_kernel<<<(unsigned)((plan_warps + 7) / 8), 256, 0, st>>>(c.view(), c.n, k, items, ctrl, bricks, brick_cap);
    note_launches(1);
    // persistent grid: every resident warp pulls work items until the counter runs out; no block waits for another one,
    // so it does not matter how many of the blocks are resident at a time (other handles may share the GPU)
    int tblocks = sm_count[di] * blocks_per_sm[di];
    const int tneed = (nq + 16 * TQ_WARPS - 1) / (16 * TQ_WARPS);     // small clouds: a few items per warp are enough
    if (tblocks > tneed) tblocks = tneed;
    const dim3 tgrid(tblocks), tblock(TQ_WARPS * 32);
    if (k == 10) knn_lists_tile_kernel<10><<<tgrid, tblock, smem, st>>>(c.view(), c.n, k, nbr_scratch, items, ctrl, fb_list, fb_flags, stats, q_lo, q_hi, 1.0f);
    else if (k == 20) knn_lists_tile_kernel<20><<<tgrid, tblock, smem, st>>>(c.view(), c.n, k, nbr_scratch, items, ctrl, fb_list, fb_flags, stats, q_lo, q_hi, 1.0f);
    else knn_lists_tile_kernel<0><<<tgrid, tblock, smem, st>>>(c.view(), c.n, k, nbr_scratch, items, ctrl, fb_list, fb_flags, stats, q_lo, q_hi, 1.0f);
    note_launches(2);
    // The points the tiles could not decide (isolated ones: a long tail of deep searches by few warps) and their
    // covariances run on a high-priority side stream BESIDE the main covariance launch, which skips them.
    const bool overlap = side != nullptr && side->stream != nullptr && !want_stats;
    cudaStream_t rs = overlap ? side->stream : st;
    if (overlap) {
      if ((e = cudaEventRecord(side->fork, st)) != cudaSuccess) return e;
      if ((e = cudaStreamWaitEvent(rs, side->fork, 0)) != cudaSuccess) return e;
    }
    knn_lists_rest_kernel<<<sm_count[di] * 16, 64, 0, rs>>>   // small blocks: the few long searches must not hold the SMs the main covariance launch needs
       (c.view(), k, nbr_scratch, ctrl, fb_list);
    note_launches(1);
    launch_cov_rest_kernel(c, k, method, nbr_scratch, covs6, ctrl, fb_list, sm_count[di], rs);
    if (overlap && (e = cudaEventRecord(side->join, rs)) != cudaSuccess) return e;
    if (want_stats) {
      unsigned long long h[ST_N] = {};
      cudaMemcpyAsync(h, stats, sizeof(h), cudaMemcpyDeviceToHost, st);
      cudaStreamSynchronize(st);
      cudaFree(stats);
      fprintf(stderr, "[ngicp knn] n=%d k=%d warp-search=%llu (%.1f%%, ties %llu) items=%llu tiles=%llu passes=%llu lanes/pass=%.1f\n",
              c.n, k, h[ST_FALLBACK], 100.0 * (double)h[ST_FALLBACK] / (double)c.n, h[ST_TIES], h[ST_ITEMS], h[ST_TILES], h[ST_PASSES],
              h[ST_PASSES] ? (double)h[ST_LANES] / (double)h[ST_PASSES] : 0.0);
      fprintf(stderr, "[ngicp knn]   decided at radius 1 / 2 / >2: %llu / %llu / %llu, passes %llu / %llu / %llu, candidates per pass %.0f\n",
              h[ST_DEC1], h[ST_DEC2], h[ST_DECHI], h[ST_PASS1], h[ST_PASS2], h[ST_PASSHI],
              h[ST_PASSES] ? (double)h[ST_CAND] / (double)h[ST_PASSES] : 0.0);
      if (h[ST_TWARPS])
        fprintf(stderr, "[ngicp knn]   tile kernel: %llu warps, span %.1f us, mean warp busy %.1f us (%.0f%% of the span)\n", h[ST_TWARPS],
                1e-3 * (double)(h[ST_TEND] - h[ST_TSTART]), 1e-3 * (double)h[ST_TSUM] / (double)h[ST_TWARPS],
                100.0 * (double)h[ST_TSUM] / (double)h[ST_TWARPS] / (double)(h[ST_TEND] - h[ST_TSTART]));
      // the control words of the plan / tile / rest launches, and the plan's work items by box edge (how far it split)
      int hc[CT_N] = {};
      cudaMemcpyAsync(hc, ctrl, sizeof(hc), cudaMemcpyDeviceToHost, st);
      cudaStreamSynchronize(st);
      const int nslow = hc[CT_SLOW], nall = nslow + hc[CT_ITEMS];
      long long by_edge[3] = {0, 0, 0};      // box edge TQ_CORE, TQ_CORE / 2, 1 cells
      if (nall > 0 && nall <= c.n) {
        int4* hi = static_cast<int4*>(malloc(sizeof(int4) * (size_t)c.n));
        if (hi != nullptr && cudaMemcpy(hi, items, sizeof(int4) * (size_t)c.n, cudaMemcpyDeviceToHost) == cudaSuccess) {
          for (int w = 0; w < nall; ++w) {
            const int sz = hi[w < nslow ? w : c.n - 1 - (w - nslow)].w & 255;
            by_edge[sz == TQ_CORE ? 0 : (sz == 1 ? 2 : 1)]++;
          }
        }
        free(hi);
      }
      fprintf(stderr, "[ngicp knn]   control: rest=%d fix=%d slow=%d items=%d, items by box edge %d / %d / 1: %lld / %lld / %lld\n",
              hc[CT_REST], hc[CT_FIX], nslow, hc[CT_ITEMS], TQ_CORE, TQ_CORE / 2, by_edge[0], by_edge[1], by_edge[2]);
    }
    launch_cov_kernel(c, k, method, nbr_scratch, covs6, q_lo, q_hi, fb_flags, nullptr, nullptr, st, k == 10 || k == 20);
    if (overlap && (e = cudaStreamWaitEvent(st, side->join, 0)) != cudaSuccess) return e;
    return cudaGetLastError();
  }
  launch_cov_kernel(c, k, method, nbr_scratch, covs6, q_lo, q_hi, nullptr, nullptr, nullptr, st);
  return cudaGetLastError();
}

}  // namespace ngicp
