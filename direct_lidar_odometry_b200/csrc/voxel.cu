// voxel.cu — K0: pcl::VoxelGrid<PointXYZI>::filter as a sort-based voxel reduce
// (third-party code in the reference; call sites src/dlo/odom.cc:460-463, 487-490, 1160-1163;
// algorithm restated in SURVEY.md App. B1):
//   bbox -> min_b = floor(min * inv), div_b -> per point idx = i + j*dx + k*dx*dy (int32) ->
//   stable radix sort of (idx, point) -> one centroid per run of equal idx, emitted in ascending idx.
// The within-voxel accumulation order is ascending input index (the sort is stable), float32 running
// sums of x,y,z,intensity divided by the float count — the order the CPU oracle fixes as well.
// Algorithmic bytes: 16 N read + 16 M written (BASELINE.md §4; records are 32 B at the boundary).
#include <mutex>
#include <cooperative_groups.h>
#include "internal.h"

namespace ngicp {

// non-finite points get the key one past the last voxel (sorted to the end, never emitted)

__global__ void vox_desc_init_kernel(GridDesc* d) {
  for (int i = 0; i < 3; i++) { d->bb_min[i] = f2ord(FLT_MAX); d->bb_max[i] = f2ord(-FLT_MAX); }
  d->nfinite = 0; d->vcount = 0; d->voverflow = 0;
}

// pcl::CropBox with setNegative(true) (reference odom.cc:122-124,454-457): a point with min <= p <= max on all three
// axes is dropped.  Fused here as "treat it like a non-finite point", which is also how removeNaNFromPointCloud
// (odom.cc:451) is honoured: such points never enter the bounding box, get the invalid key and are never emitted.
struct CropBox { int on; float lo[3], hi[3]; };
// pcl::transformPointCloud(*cloud, *cloud, T) in front of the submap voxel grid (odom.cc:484-490,1157-1163), fused into the
// same pass: x' = ((m00 x + m01 y) + m02 z) + m03, float, unfused — the order the CPU oracle fixes (synth.transform_xyzi)
struct RigidXf { int on; float m[12]; };

// a FLOAT32 field at any byte address (sensor_msgs::PointCloud2 layouts need not be 4-byte aligned: Velodyne's
// point_step is 22)
__device__ __forceinline__ float load_f32(const unsigned char* p, bool aligned) {
  if (aligned) return *reinterpret_cast<const float*>(p);
  const unsigned u = (unsigned)p[0] | ((unsigned)p[1] << 8) | ((unsigned)p[2] << 16) | ((unsigned)p[3] << 24);
  return __uint_as_float(u);
}

// raw records -> float4 {x,y,z,intensity}; bbox over finite points (pcl::getMinMax3D on a non-dense cloud).
// Record i lives at (i / width) * row_step + (i % width) * point_step; its fields at the byte offsets of `lay`
// (plain PointXYZI arrays: one row, offsets 0/4/8/16) — pcl::fromROSMsg's field mapping done on the fly.
__global__ void __launch_bounds__(256) vox_pack_kernel(const unsigned char* __restrict__ raw, RecordLayout lay, int n,
                                                       float4* __restrict__ pts, GridDesc* __restrict__ d, CropBox crop, RigidXf xf) {
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  int finite = 0;
  const bool al = lay.aligned != 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int row = lay.width >= n ? 0 : i / lay.width;
    const unsigned char* r = raw + (size_t)row * lay.row_step + (size_t)(i - row * lay.width) * lay.point_step;
    float x = load_f32(r + lay.off[0], al), y = load_f32(r + lay.off[1], al), z = load_f32(r + lay.off[2], al);
    const float it = lay.off[3] >= 0 ? load_f32(r + lay.off[3], al) : 0.f;
    if (xf.on) {
      const float tx = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(xf.m[0], x), __fmul_rn(xf.m[1], y)), __fmul_rn(xf.m[2], z)), xf.m[3]);
      const float ty = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(xf.m[4], x), __fmul_rn(xf.m[5], y)), __fmul_rn(xf.m[6], z)), xf.m[7]);
      const float tz = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(xf.m[8], x), __fmul_rn(xf.m[9], y)), __fmul_rn(xf.m[10], z)), xf.m[11]);
      x = tx; y = ty; z = tz;
    }
    if (crop.on && x >= crop.lo[0] && x <= crop.hi[0] && y >= crop.lo[1] && y <= crop.hi[1] && z >= crop.lo[2] && z <= crop.hi[2])
      x = __int_as_float(0x7fc00000);   // cropped away
    pts[i] = make_float4(x, y, z, it);
    if (isfinite(x) && isfinite(y) && isfinite(z)) {
      finite++;
      mn[0] = fminf(mn[0], x); mn[1] = fminf(mn[1], y); mn[2] = fminf(mn[2], z);
      mx[0] = fmaxf(mx[0], x); mx[1] = fmaxf(mx[1], y); mx[2] = fmaxf(mx[2], z);
    }
  }
#pragma unroll
  for (int a = 0; a < 3; a++)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(FULL, mn[a], o));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(FULL, mx[a], o));
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) finite += __shfl_xor_sync(FULL, finite, o);
  // one set of atomics per BLOCK (7 same-address atomics per warp serialise in L2: 109k of them for a 500k-point cloud)
  __shared__ float s_mn[8][3], s_mx[8][3];
  __shared__ int s_fin[8];
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int a = 0; a < 3; a++) { s_mn[w][a] = mn[a]; s_mx[w][a] = mx[a]; }
    s_fin[w] = finite;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    for (int ww = 1; ww < nw; ww++) {
#pragma unroll
      for (int a = 0; a < 3; a++) { mn[a] = fminf(mn[a], s_mn[ww][a]); mx[a] = fmaxf(mx[a], s_mx[ww][a]); }
      finite += s_fin[ww];
    }
    if (finite > 0) {
#pragma unroll
      for (int a = 0; a < 3; a++) { atomicMin(&d->bb_min[a], f2ord(mn[a])); atomicMax(&d->bb_max[a], f2ord(mx[a])); }
      atomicAdd(&d->nfinite, finite);
    }
  }
}

// PCL's index-range guard (dx = (int64)((max - min) * inverse_leaf) + 1 per axis; dx*dy*dz > INT32_MAX -> warn, output =
// input), made exact.  The cloud passes through (returns 1) wherever PCL's own arithmetic is not defined or would wrap:
//   * an axis extent (max - min) * inv that is not finite or >= 2^31 (the int64 conversion, then dx*dy*dz, would overflow);
//   * dx*dy*dz > INT32_MAX, computed without wrapping;
//   * floor(min * inv) or floor(max * inv) outside int32, or div_b = max_b - min_b + 1 beyond INT32_MAX;
//   * floor(max * inv) - (float)min_b rounding past max_b - min_b (axes wider than 2^24 cells): the last cell's index
//     would reach div_b and alias the next row, or the invalid key;
//   * a div_b product >= 2^32.
// Otherwise min_b / div_b are PCL's, every float -> int conversion of the key computation is in range on any hardware,
// every finite point's key is below div_b[0]*div_b[1]*div_b[2], and that product is the key of non-finite points.
// SURVEY.md App. B1 states the same rule.
__device__ int vox_grid_setup(const float lo[3], const float hi[3], float inv, int minb[3], int div[3]) {
  long long dxyz = 1;
  unsigned long long cells = 1;
  for (int a = 0; a < 3; a++) { minb[a] = 0; div[a] = 1; }
  int mnb[3], dv[3];
  for (int a = 0; a < 3; a++) {
    const float ext = __fmul_rn(__fsub_rn(hi[a], lo[a]), inv);
    if (!(ext < 2147483648.f)) return 1;
    dxyz *= (long long)ext + 1;                                   // each factor <= 2^31: no wrap before the test below
    if (dxyz > 2147483647ll) return 1;
    const float flo = floorf(__fmul_rn(lo[a], inv)), fhi = floorf(__fmul_rn(hi[a], inv));
    if (!(flo >= -2147483648.f) || !(fhi < 2147483648.f)) return 1;
    const long long span = (long long)fhi - (long long)flo;
    if (span >= 2147483647ll || (long long)__fsub_rn(fhi, flo) > span) return 1;
    cells *= (unsigned long long)(span + 1);
    if (cells >= (1ull << 32)) return 1;
    mnb[a] = (int)flo;
    dv[a] = (int)(span + 1);
  }
  for (int a = 0; a < 3; a++) { minb[a] = mnb[a]; div[a] = dv[a]; }
  return 0;
}

__global__ void vox_setup_kernel(GridDesc* d, float inv) {
  if (d->nfinite == 0) { d->voverflow = 0; for (int a = 0; a < 3; a++) { d->vmin_b[a] = 0; d->vdiv[a] = 1; } return; }
  float lo[3], hi[3];
  for (int a = 0; a < 3; a++) { lo[a] = ord2f(d->bb_min[a]); hi[a] = ord2f(d->bb_max[a]); }
  int minb[3], div[3];
  d->voverflow = vox_grid_setup(lo, hi, inv, minb, div);
  for (int a = 0; a < 3; a++) { d->vmin_b[a] = minb[a]; d->vdiv[a] = div[a]; }
}

__global__ void __launch_bounds__(256) vox_keys_kernel(const float4* __restrict__ pts, int n, const GridDesc* __restrict__ d, float inv,
                                                       unsigned* __restrict__ keys, unsigned* __restrict__ vals) {
  const int m0 = d->vmin_b[0], m1 = d->vmin_b[1], m2 = d->vmin_b[2];
  const unsigned mul1 = (unsigned)d->vdiv[0], mul2 = (unsigned)d->vdiv[0] * (unsigned)d->vdiv[1];
  const bool bad = d->voverflow != 0;
  const unsigned VOX_INVALID = d->voverflow ? 0u : (unsigned)d->vdiv[0] * (unsigned)d->vdiv[1] * (unsigned)d->vdiv[2];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    unsigned key = VOX_INVALID;
    if (!bad && isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) {
      const int i0 = (int)(__fsub_rn(floorf(__fmul_rn(p.x, inv)), (float)m0));
      const int i1 = (int)(__fsub_rn(floorf(__fmul_rn(p.y, inv)), (float)m1));
      const int i2 = (int)(__fsub_rn(floorf(__fmul_rn(p.z, inv)), (float)m2));
      key = (unsigned)i0 + (unsigned)i1 * mul1 + (unsigned)i2 * mul2;   // < div_b product < 2^32 (vox_grid_setup)
    }
    keys[i] = key;
    vals[i] = (unsigned)i;
  }
}

// flags[i] = 1 at the first element of every run of equal valid keys; flags[n] = 0 (sentinel for the total)
__global__ void __launch_bounds__(256) vox_heads_kernel(const unsigned* __restrict__ keys, int n, int* __restrict__ flags, GridDesc* __restrict__ d) {
  const unsigned VOX_INVALID = d->voverflow ? 0u : (unsigned)d->vdiv[0] * (unsigned)d->vdiv[1] * (unsigned)d->vdiv[2];
  if (blockIdx.x == 0 && threadIdx.x == 0) d->n = n + 1;   // length of the scan that follows
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += gridDim.x * blockDim.x) {
    int f = 0;
    if (i < n) {
      const unsigned k = keys[i];
      f = (k != VOX_INVALID && (i == 0 || keys[i - 1] != k)) ? 1 : 0;
    }
    flags[i] = f;
  }
}

// one thread per run head: sequential float accumulation in sorted (= ascending input index) order
__global__ void __launch_bounds__(128) vox_centroid_kernel(const unsigned* __restrict__ keys, const unsigned* __restrict__ perm, int n,
                                                           const int* __restrict__ slots, const float4* __restrict__ pts,
                                                           float* __restrict__ out, int* __restrict__ slot_of_point, const GridDesc* __restrict__ d) {
  const unsigned VOX_INVALID = d->voverflow ? 0u : (unsigned)d->vdiv[0] * (unsigned)d->vdiv[1] * (unsigned)d->vdiv[2];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned k = keys[i];
    if (k == VOX_INVALID) { slot_of_point[perm[i]] = -1; continue; }
    if (i > 0 && keys[i - 1] == k) continue;
    const int slot = slots[i];
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
    int j = i;
    for (; j < n && keys[j] == k; ++j) {
      const unsigned o = perm[j];
      const float4 p = pts[o];
      sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, p.z); si = __fadd_rn(si, p.w);
      slot_of_point[o] = slot;
    }
    const float cnt = (float)(j - i);
    float4* o4 = reinterpret_cast<float4*>(out + (size_t)slot * 8);
    o4[0] = make_float4(__fdiv_rn(sx, cnt), __fdiv_rn(sy, cnt), __fdiv_rn(sz, cnt), 1.0f);
    o4[1] = make_float4(__fdiv_rn(si, cnt), 0.f, 0.f, 0.f);
  }
}

// no voxel grid (vf_scan_use_ = false, odom.cc:460) or PCL's "leaf too small" pass-through: the surviving points in input
// order.  flags = exclusive scan of "kept".
__global__ void __launch_bounds__(256) vox_keep_flags_kernel(const float4* __restrict__ pts, int n, int* __restrict__ flags) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += gridDim.x * blockDim.x) {
    int f = 0;
    if (i < n) { const float4 p = pts[i]; f = (isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) ? 1 : 0; }
    flags[i] = f;
  }
}
__global__ void __launch_bounds__(256) vox_compact_kernel(const float4* __restrict__ pts, int n, const int* __restrict__ slots,
                                                          float* __restrict__ out, int* __restrict__ slot_of_point) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    const bool keep = isfinite(p.x) && isfinite(p.y) && isfinite(p.z);
    slot_of_point[i] = keep ? slots[i] : -1;
    if (keep) {
      float4* o4 = reinterpret_cast<float4*>(out + (size_t)slots[i] * 8);
      o4[0] = make_float4(p.x, p.y, p.z, 1.0f);
      o4[1] = make_float4(p.w, 0.f, 0.f, 0.f);
    }
  }
}

static inline int vgrid(int n, int threads) {
  int g = (n + threads - 1) / threads;
  if (g < 1) g = 1;
  return g > 148 * 16 ? 148 * 16 : g;
}

// the pipeline's outcome for the host: {m, overflow, key bits this cloud needs}, stored into mapped pinned memory
__global__ void vox_result_kernel(const GridDesc* __restrict__ d, const int* __restrict__ total, int* __restrict__ result) {
  const unsigned long long cells = (unsigned long long)d->vdiv[0] * (unsigned long long)d->vdiv[1] * (unsigned long long)d->vdiv[2];
  int bits = 1;
  while (bits < 32 && (1ull << bits) <= cells) bits++;
  result[0] = *total;
  result[1] = d->voverflow;
  result[2] = bits;
}

// records -> the caller's DEVICE buffer, count read on the device (no host round trip before the copy)
__global__ void __launch_bounds__(256) vox_copy_out_kernel(const float4* __restrict__ src, const int* __restrict__ total, size_t cap,
                                                           float4* __restrict__ dst) {
  const size_t m = (size_t)*total;
  if (m > cap) return;                                    // reported by the host after the synchronisation
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * m; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}


// ---------------------------------------------------------------------------------------------------------------
// K0 in ONE persistent cooperative launch (clouds up to VF_CH points per block x one block per SM = 606k points on a
// B200): pack / transform / crop + bounding box -> voxel keys -> stable LSD radix sort (9-bit digits, as many passes as
// THIS cloud's voxel-index range needs: decided on the device, nothing speculated) -> run heads -> centroids, separated
// by grid barriers instead of kernel boundaries.  The multi-kernel pipeline below needs ~20 dependent launches for the
// same work (6 us each at 53k points: launch latency, not bandwidth); here a 53k-point scan is 8 barriers.
// Every block owns one contiguous chunk of the cloud; a radix pass ranks the chunk's items in order warp by warp
// (match_any, as rs_scatter), publishes its digit histogram, and after the barrier every block derives ITS offsets
// itself from the whole (digit-major) histogram table — one digit per thread, no single-block scan kernel in between.
// Same arithmetic and the same stable order as the multi-kernel path: outputs are bit-identical (tests compare both).
// ---------------------------------------------------------------------------------------------------------------
constexpr int VF_THREADS = 512;
constexpr int VF_WARPS = VF_THREADS / 32;
constexpr int VF_CH = 4096;                 // points per block
constexpr int VF_BITS = 9;
constexpr int VF_BINS = 1 << VF_BITS;       // == VF_THREADS: one digit per thread in the offset step
static_assert(VF_BINS == VF_THREADS, "one digit per thread");

struct VoxFusedArgs {
  const unsigned char* raw; RecordLayout lay; int n; float inv;
  CropBox crop; RigidXf xf;
  float4* pts;
  unsigned *keys_a, *vals_a, *keys_b, *vals_b;
  unsigned short* hist;       // [G][VF_BINS] block-major: a block's digit counts (<= VF_CH) are one 1 KB row
  unsigned* bar;              // grid barrier words {arrivals, -, departures}; zero between launches
  float* part;                // [G][8]: per-block bbox min[3], max[3], finite count (as int bits)
  int* blk_heads;             // [G]
  float* out; int* slot_of_point; GridDesc* d;
  int* result;                // mapped pinned {m, overflow, key bits}
  float4* user_out; size_t user_cap;   // optional device destination of the records (nullptr = none)
};

struct VoxFusedSmem {
  unsigned key[VF_CH];
  unsigned val[VF_CH];
  unsigned short rank[VF_CH];
  int wcnt[VF_WARPS][VF_BINS];
  int base[VF_BINS];
  int tot8[8][VF_BINS], bef8[8][VF_BINS];   // partial column sums of the histogram table (offset step)
  int scan[VF_WARPS + 1];
  float red[VF_WARPS][8];
  int minb[3], div[3], overflow, nfinite, bits;
  unsigned invalid;
};

__device__ __forceinline__ int vf_block_exclusive_scan(int v, int* scan /* VF_WARPS + 1 */, int& total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, inc, o); if (lane >= o) inc += t; }
  if (lane == 31) scan[w] = inc;
  __syncthreads();
  if (w == 0) {
    const int ws = lane < VF_WARPS ? scan[lane] : 0;
    int wi = ws;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, wi, o); if (lane >= o) wi += t; }
    if (lane < VF_WARPS) scan[lane] = wi - ws;
    if (lane == 31) scan[VF_WARPS] = wi;
  }
  __syncthreads();
  const int r = scan[w] + inc - v;
  total = scan[VF_WARPS];
  __syncthreads();
  return r;
}

// Grid barrier for the cooperative launch (all blocks co-resident): one arrival counter that only grows within a launch;
// thread 0 of every block arrives and polls with relaxed loads, the block waits on it.  ~half the cost of
// cooperative_groups' grid.sync() at 50-150 blocks.
__device__ __forceinline__ void vf_grid_barrier(unsigned* bar, unsigned& phase) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(bar, 1u);
    const unsigned target = (phase + 1u) * gridDim.x;
    unsigned v;
    do { asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory"); } while (v < target);
    __threadfence();
  }
  phase++;
  __syncthreads();
}

__global__ void __launch_bounds__(VF_THREADS, 1) vox_fused_kernel(VoxFusedArgs a) {
  extern __shared__ __align__(16) unsigned char vf_smem_raw[];
  VoxFusedSmem& S = *reinterpret_cast<VoxFusedSmem*>(vf_smem_raw);
  unsigned phase = 0;
  const int G = gridDim.x, blk = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int n = a.n;
  const int chunk = (n + G - 1) / G;                       // <= VF_CH (host guarantees)
  const int lo = min(blk * chunk, n), hi = min(lo + chunk, n), cnt = hi - lo;

  // ---- pack (+ transform, crop), bounding box of the finite points ----
  {
    float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    int finite = 0;
    const bool al = a.lay.aligned != 0;
    for (int i = lo + tid; i < hi; i += VF_THREADS) {
      const int row = a.lay.width >= n ? 0 : i / a.lay.width;
      const unsigned char* r = a.raw + (size_t)row * a.lay.row_step + (size_t)(i - row * a.lay.width) * a.lay.point_step;
      float x = load_f32(r + a.lay.off[0], al), y = load_f32(r + a.lay.off[1], al), z = load_f32(r + a.lay.off[2], al);
      const float it = a.lay.off[3] >= 0 ? load_f32(r + a.lay.off[3], al) : 0.f;
      if (a.xf.on) {
        const float* m = a.xf.m;
        const float tx = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], x), __fmul_rn(m[1], y)), __fmul_rn(m[2], z)), m[3]);
        const float ty = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[4], x), __fmul_rn(m[5], y)), __fmul_rn(m[6], z)), m[7]);
        const float tz = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[8], x), __fmul_rn(m[9], y)), __fmul_rn(m[10], z)), m[11]);
        x = tx; y = ty; z = tz;
      }
      if (a.crop.on && x >= a.crop.lo[0] && x <= a.crop.hi[0] && y >= a.crop.lo[1] && y <= a.crop.hi[1] && z >= a.crop.lo[2] && z <= a.crop.hi[2])
        x = __int_as_float(0x7fc00000);   // cropped away
      a.pts[i] = make_float4(x, y, z, it);
      if (isfinite(x) && isfinite(y) && isfinite(z)) {
        finite++;
        mn[0] = fminf(mn[0], x); mn[1] = fminf(mn[1], y); mn[2] = fminf(mn[2], z);
        mx[0] = fmaxf(mx[0], x); mx[1] = fmaxf(mx[1], y); mx[2] = fmaxf(mx[2], z);
      }
    }
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        mn[c] = fminf(mn[c], __shfl_xor_sync(FULL, mn[c], o));
        mx[c] = fmaxf(mx[c], __shfl_xor_sync(FULL, mx[c], o));
      }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) finite += __shfl_xor_sync(FULL, finite, o);
    if (lane == 0) {
#pragma unroll
      for (int c = 0; c < 3; c++) { S.red[w][c] = mn[c]; S.red[w][3 + c] = mx[c]; }
      S.red[w][6] = __int_as_float(finite);
    }
    __syncthreads();
    if (tid == 0) {
      for (int ww = 1; ww < VF_WARPS; ww++) {
#pragma unroll
        for (int c = 0; c < 3; c++) { mn[c] = fminf(mn[c], S.red[ww][c]); mx[c] = fmaxf(mx[c], S.red[ww][3 + c]); }
        finite += __float_as_int(S.red[ww][6]);
      }
      float* p = a.part + (size_t)blk * 8;
#pragma unroll
      for (int c = 0; c < 3; c++) { p[c] = mn[c]; p[3 + c] = mx[c]; }
      p[6] = __int_as_float(finite);
    }
  }
  vf_grid_barrier(a.bar, phase);

  // ---- every block: bbox of all blocks -> PCL's min_b / div_b / overflow (vox_setup_kernel's arithmetic) ----
  if (w == 0) {
    float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    int finite = 0;
    for (int b = lane; b < G; b += 32) {
      const float* p = a.part + (size_t)b * 8;
#pragma unroll
      for (int c = 0; c < 3; c++) { mn[c] = fminf(mn[c], __ldcg(p + c)); mx[c] = fmaxf(mx[c], __ldcg(p + 3 + c)); }
      finite += __float_as_int(__ldcg(p + 6));
    }
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        mn[c] = fminf(mn[c], __shfl_xor_sync(FULL, mn[c], o));
        mx[c] = fmaxf(mx[c], __shfl_xor_sync(FULL, mx[c], o));
      }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) finite += __shfl_xor_sync(FULL, finite, o);
    if (lane == 0) {
      S.nfinite = finite;
      int over = 0;
      unsigned long long cells = 1ull;
      if (finite > 0) {
        over = vox_grid_setup(mn, mx, a.inv, S.minb, S.div);
        cells = (unsigned long long)S.div[0] * (unsigned long long)S.div[1] * (unsigned long long)S.div[2];
      } else {
        for (int c = 0; c < 3; c++) { S.minb[c] = 0; S.div[c] = 1; }
      }
      S.overflow = over;
      S.invalid = over ? 0u : (unsigned)cells;
      int bits = 1;
      while (bits < 32 && (1ull << bits) <= cells) bits++;
      S.bits = bits;
      if (blk == 0) {
        GridDesc* d = a.d;
        for (int c = 0; c < 3; c++) { d->bb_min[c] = f2ord(mn[c]); d->bb_max[c] = f2ord(mx[c]); d->vmin_b[c] = S.minb[c]; d->vdiv[c] = S.div[c]; }
        d->nfinite = finite; d->voverflow = over; d->vcount = 0;
      }
    }
  }
  __syncthreads();
  if (S.overflow || S.nfinite == 0) {                      // uniform over the grid: PCL passes the input through / nothing to do
    if (blk == 0 && tid == 0) { a.result[0] = 0; a.result[1] = S.overflow; a.result[2] = S.bits; }
    if (S.nfinite == 0 && !S.overflow)
      for (int i = lo + tid; i < hi; i += VF_THREADS) a.slot_of_point[i] = -1;
    if (tid == 0 && atomicAdd(a.bar + 2, 1u) == gridDim.x - 1u) { a.bar[0] = 0u; a.bar[2] = 0u; }
    return;
  }

  // ---- voxel keys of the own chunk (vox_keys_kernel's arithmetic) ----
  {
    const int m0 = S.minb[0], m1 = S.minb[1], m2 = S.minb[2];
    const unsigned mul1 = (unsigned)S.div[0], mul2 = (unsigned)S.div[0] * (unsigned)S.div[1];
    for (int j = tid; j < cnt; j += VF_THREADS) {
      const float4 p = a.pts[lo + j];
      unsigned key = S.invalid;
      if (isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) {
        const int i0 = (int)(__fsub_rn(floorf(__fmul_rn(p.x, a.inv)), (float)m0));
        const int i1 = (int)(__fsub_rn(floorf(__fmul_rn(p.y, a.inv)), (float)m1));
        const int i2 = (int)(__fsub_rn(floorf(__fmul_rn(p.z, a.inv)), (float)m2));
        key = (unsigned)i0 + (unsigned)i1 * mul1 + (unsigned)i2 * mul2;   // < div_b product < 2^32 (vox_grid_setup)
      }
      S.key[j] = key;
      S.val[j] = (unsigned)(lo + j);
    }
  }
  __syncthreads();

  // ---- stable LSD radix sort ----
  const int passes = (S.bits + VF_BITS - 1) / VF_BITS;
  const int seg = ((cnt + VF_WARPS - 1) / VF_WARPS + 31) & ~31;     // items per warp, whole groups of 32
  const unsigned lt = (1u << lane) - 1u;
  unsigned *kin = a.keys_a, *vin = a.vals_a, *kout = a.keys_b, *vout = a.vals_b;
  for (int p = 0; p < passes; ++p) {
    const int shift = p * VF_BITS;
    if (p > 0) {
      for (int j = tid; j < cnt; j += VF_THREADS) { S.key[j] = __ldcg(kin + lo + j); S.val[j] = __ldcg(vin + lo + j); }
    }
    for (int i = tid; i < VF_WARPS * VF_BINS; i += VF_THREADS) (&S.wcnt[0][0])[i] = 0;
    __syncthreads();
    // rank the warp's items in order (rank among equal digits of this warp)
    for (int j0 = w * seg; j0 < min((w + 1) * seg, cnt); j0 += 32) {
      const int j = j0 + lane;
      const bool valid = j < cnt;
      const unsigned dgt = valid ? ((S.key[j] >> shift) & (VF_BINS - 1)) : (unsigned)VF_BINS;
      const unsigned peers = __match_any_sync(FULL, dgt);
      const int leader = __ffs(peers) - 1;
      int before = 0;
      if (valid && lane == leader) { before = S.wcnt[w][dgt]; S.wcnt[w][dgt] = before + __popc(peers); }
      before = __shfl_sync(FULL, before, leader);
      if (valid) S.rank[j] = (unsigned short)(before + __popc(peers & lt));
      __syncwarp();
    }
    __syncthreads();
    {
      // digit `tid`: block total -> table; per-warp counts -> exclusive over the warps
      int run = 0;
#pragma unroll
      for (int ww = 0; ww < VF_WARPS; ww++) { const int t = S.wcnt[ww][tid]; S.wcnt[ww][tid] = run; run += t; }
      a.hist[(size_t)blk * VF_BINS + tid] = (unsigned short)run;
    }
    vf_grid_barrier(a.bar, phase);
    {
      // column sums of the table (all blocks / the blocks before this one) for every digit: thread = (8 consecutive digits,
      // every 8th block row), one 16-byte load per row — all loads independent, one round of latency
      const int dg = tid & 63, bsub = tid >> 6;
      int tot[8], bef[8];
#pragma unroll
      for (int u = 0; u < 8; u++) { tot[u] = 0; bef[u] = 0; }
      for (int b = bsub; b < G; b += 8) {
        const uint4 q = __ldcg(reinterpret_cast<const uint4*>(a.hist + (size_t)b * VF_BINS) + dg);
        const unsigned wv[4] = {q.x, q.y, q.z, q.w};
        const bool mine = b < blk;
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int c0 = (int)(wv[u] & 0xffffu), c1 = (int)(wv[u] >> 16);
          tot[2 * u] += c0; tot[2 * u + 1] += c1;
          if (mine) { bef[2 * u] += c0; bef[2 * u + 1] += c1; }
        }
      }
#pragma unroll
      for (int u = 0; u < 8; u++) { S.tot8[bsub][dg * 8 + u] = tot[u]; S.bef8[bsub][dg * 8 + u] = bef[u]; }
      __syncthreads();
      int total = 0, before = 0;
#pragma unroll
      for (int r = 0; r < 8; r++) { total += S.tot8[r][tid]; before += S.bef8[r][tid]; }
      int all;
      const int excl = vf_block_exclusive_scan(total, S.scan, all);
      S.base[tid] = excl + before;
    }
    __syncthreads();
    for (int j = tid; j < cnt; j += VF_THREADS) {
      const unsigned key = S.key[j];
      const unsigned dgt = (key >> shift) & (VF_BINS - 1);
      const int pos = S.base[dgt] + S.wcnt[j / seg][dgt] + (int)S.rank[j];
      kout[pos] = key;
      vout[pos] = S.val[j];
    }
    vf_grid_barrier(a.bar, phase);
    unsigned* t = kin; kin = kout; kout = t;
    t = vin; vin = vout; vout = t;
  }
  if (passes == 0) {       // cannot happen (bits >= 1); keeps kin/vin meaningful for the reader
    for (int j = tid; j < cnt; j += VF_THREADS) { kin[lo + j] = S.key[j]; vin[lo + j] = S.val[j]; }
    vf_grid_barrier(a.bar, phase);
  }
  const unsigned* keys = kin;       // sorted keys, permutation
  const unsigned* perm = vin;

  // ---- run heads of the own chunk, their local ranks ----
  {
    constexpr int IPT = VF_CH / VF_THREADS;                // 8 consecutive items per thread
    int flags = 0, c = 0;
#pragma unroll
    for (int u = 0; u < IPT; u++) {
      const int j = tid * IPT + u;
      if (j < cnt) {
        const int i = lo + j;
        const unsigned k = __ldcg(keys + i);
        S.key[j] = k;
        const bool head = k != S.invalid && (i == 0 || __ldcg(keys + i - 1) != k);
        if (head) { flags |= 1 << u; c++; }
      }
    }
    int total;
    int r = vf_block_exclusive_scan(c, S.scan, total);
#pragma unroll
    for (int u = 0; u < IPT; u++) {
      const int j = tid * IPT + u;
      if (j < cnt) {
        S.rank[j] = (unsigned short)r;
        S.val[j] = (flags >> u) & 1;
        r += (flags >> u) & 1;
      }
    }
    if (tid == 0) a.blk_heads[blk] = total;
  }
  vf_grid_barrier(a.bar, phase);
  int slot_base = 0, m_total = 0;
  {
    int before = 0, all = 0;
    for (int b = tid; b < G; b += VF_THREADS) { const int v = __ldcg(a.blk_heads + b); all += v; before += b < blk ? v : 0; }
    // G <= VF_THREADS: one value per thread, block sums through the scan helper
    int t1, t2;
    vf_block_exclusive_scan(before, S.scan, t1);
    vf_block_exclusive_scan(all, S.scan, t2);
    slot_base = t1; m_total = t2;
  }
  // ---- centroids: one thread per run head, sequential float accumulation in sorted (= ascending input index) order ----
  for (int j = tid; j < cnt; j += VF_THREADS) {
    const int i = lo + j;
    const unsigned k = S.key[j];
    if (k == S.invalid) { a.slot_of_point[__ldcg(perm + i)] = -1; continue; }
    if (!S.val[j]) continue;
    const int slot = slot_base + (int)S.rank[j];
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
    int e = i;
    for (; e < n && __ldcg(keys + e) == k; ++e) {
      const unsigned o = __ldcg(perm + e);
      const float4 p = a.pts[o];
      sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, p.z); si = __fadd_rn(si, p.w);
      a.slot_of_point[o] = slot;
    }
    const float c = (float)(e - i);
    const float4 r0 = make_float4(__fdiv_rn(sx, c), __fdiv_rn(sy, c), __fdiv_rn(sz, c), 1.0f);
    const float4 r1 = make_float4(__fdiv_rn(si, c), 0.f, 0.f, 0.f);
    float4* o4 = reinterpret_cast<float4*>(a.out + (size_t)slot * 8);
    o4[0] = r0; o4[1] = r1;
    if (a.user_out != nullptr && (size_t)slot < a.user_cap) { a.user_out[2 * (size_t)slot] = r0; a.user_out[2 * (size_t)slot + 1] = r1; }
  }
  if (blk == 0 && tid == 0) { a.result[0] = m_total; a.result[1] = 0; a.result[2] = S.bits; a.d->vcount = m_total; }
  // leave the barrier words zeroed for the next launch: the last block to depart does it (nobody polls any more)
  if (tid == 0 && atomicAdd(a.bar + 2, 1u) == gridDim.x - 1u) { a.bar[0] = 0u; a.bar[2] = 0u; }
}

static int vox_fused_grid(int device, int n) {
  static std::mutex mu;
  static int sms[64] = {};
  static bool ok[64] = {};
  const int di = device & 63;
  {
    std::lock_guard<std::mutex> lock(mu);
    if (!sms[di]) {
      int v = 0, coop = 0;
      cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device);
      cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
      sms[di] = v > 0 ? v : 1;
      ok[di] = coop != 0 && cudaFuncSetAttribute(vox_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(VoxFusedSmem)) == cudaSuccess;
      cudaGetLastError();
    }
  }
  if (!ok[di]) return 0;
  int g = (n + 1023) / 1024;               // small clouds: fewer blocks, cheaper barriers
  if (g > sms[di]) g = sms[di];
  if (g < 1) g = 1;
  if ((long long)g * VF_CH < (long long)n) return 0;      // too large for one chunk per block: multi-kernel pipeline
  return g;
}

void voxel_prime_kernels() {
  cudaFuncAttributes fa;
  cudaFuncGetAttributes(&fa, vox_fused_kernel);
  cudaGetLastError();
}

cudaError_t voxel_filter_device(const void* in, size_t n, size_t stride_bytes, float leaf, Scratch& sc, const StreamPtr& st,
                                size_t* m_out, int* overflow, const float* crop6, bool compact_on_overflow, const float* T16,
                                void* out, size_t out_cap, bool* copied) {
  RecordLayout lay;
  lay.width = (int)(n < 0x7fffffffu ? n : 0x7fffffffu);
  lay.point_step = stride_bytes;
  lay.row_step = 0;
  lay.off[0] = 0; lay.off[1] = 4; lay.off[2] = 8;
  lay.off[3] = stride_bytes >= 20 ? 16 : (stride_bytes >= 16 ? 12 : -1);
  lay.aligned = 1;
  return voxel_filter_records(in, n, lay, leaf, sc, st, m_out, overflow, crop6, compact_on_overflow, T16, out, out_cap, copied);
}

cudaError_t voxel_filter_records(const void* in, size_t n, RecordLayout lay, float leaf, Scratch& sc, const StreamPtr& st,
                                 size_t* m_out, int* overflow, const float* crop6, bool compact_on_overflow, const float* T16,
                                 void* out, size_t out_cap, bool* copied, bool allow_speculation) {
  cudaError_t e;
  *m_out = 0;
  *overflow = 0;
  if (copied) *copied = false;
  if (n == 0) return cudaSuccess;
  const int ni = (int)n;
  const bool use_grid = leaf > 0.f;
  const float inv = use_grid ? 1.0f / leaf : 1.0f;  // PCL: inverse_leaf_size_ = 1 / leaf_size_ in float
  CropBox crop;
  crop.on = crop6 != nullptr;
  for (int a = 0; a < 3; a++) { crop.lo[a] = crop6 ? crop6[a] : 0.f; crop.hi[a] = crop6 ? crop6[3 + a] : 0.f; }
  RigidXf xf;
  xf.on = T16 != nullptr;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 4; c++) xf.m[r * 4 + c] = T16 ? T16[c * 4 + r] : 0.f;   // column-major 4x4 in
  int last = 0;
  for (int f = 0; f < 4; f++) last = lay.off[f] + 4 > last ? lay.off[f] + 4 : last;
  const size_t rows = (n + (size_t)lay.width - 1) / (size_t)lay.width;
  const size_t cols_last = n - (rows - 1) * (size_t)lay.width;
  const size_t raw_bytes = (rows - 1) * lay.row_step + (cols_last - 1) * lay.point_step + (size_t)last;
  if ((e = sc.staging.reserve(raw_bytes + 16, st)) != cudaSuccess) return e;
  if ((e = sc.queries.reserve(sizeof(float4) * n, st)) != cudaSuccess) return e;
  if ((e = sc.vox_desc.reserve(sizeof(GridDesc), st)) != cudaSuccess) return e;
  const size_t nb = sizeof(unsigned) * n;
  if ((e = sc.keys_a.reserve(nb, st)) != cudaSuccess) return e;
  if ((e = sc.keys_b.reserve(nb, st)) != cudaSuccess) return e;
  if ((e = sc.vals_a.reserve(nb, st)) != cudaSuccess) return e;
  if ((e = sc.vals_b.reserve(nb, st)) != cudaSuccess) return e;
  if ((e = sc.hist.reserve(sizeof(int) * radix_sort_scratch_ints(ni), st)) != cudaSuccess) return e;
  if ((e = sc.flags.reserve(sizeof(int) * (n + 1), st)) != cudaSuccess) return e;
  if ((e = sc.tile_sums.reserve(sizeof(int) * scan_scratch_ints(ni + 1), st)) != cudaSuccess) return e;
  if ((e = sc.vox_out.reserve(32 * n, st)) != cudaSuccess) return e;
  if ((e = sc.vox_slot.reserve(sizeof(int) * n, st)) != cudaSuccess) return e;
  if ((e = cudaMemcpyAsync(sc.staging.p, in, raw_bytes, cudaMemcpyDefault, st->s)) != cudaSuccess) return e;
  GridDesc* d = sc.vox_desc.as<GridDesc>();
  float4* pts = sc.queries.as<float4>();
  // ---- one persistent cooperative launch for everything behind the staging copy (NGICP_VOXEL_FUSED=0: the
  //      multi-kernel pipeline below, kept for clouds beyond 4096 points per SM and as the A/B twin in the tests) ----
  static const bool fused_on = !(getenv("NGICP_VOXEL_FUSED") && atoi(getenv("NGICP_VOXEL_FUSED")) == 0);
  int dev_id = 0;
  cudaGetDevice(&dev_id);
  const int fg = (use_grid && fused_on && allow_speculation && sc.vox_path != 1) ? vox_fused_grid(dev_id, ni) : 0;
  if (fg > 0) {
    if (!sc.vox_result) {
      if (cudaHostAlloc(&sc.vox_result, 8 * sizeof(int), cudaHostAllocMapped) != cudaSuccess ||
          cudaHostGetDevicePointer(&sc.vox_result_dev, sc.vox_result, 0) != cudaSuccess) { cudaGetLastError(); sc.vox_result = nullptr; }
    }
    if (sc.vox_result) {
      if ((e = sc.hist.reserve(sizeof(int) * ((size_t)VF_BINS * fg + 9 * (size_t)fg + 64), st)) != cudaSuccess) return e;
      if (!sc.vox_bar.p) {
        if ((e = sc.vox_bar.reserve(64, st)) != cudaSuccess) return e;
        if ((e = cudaMemsetAsync(sc.vox_bar.p, 0, 64, st->s)) != cudaSuccess) return e;
      }
      bool out_dev = false;
      if (out && copied) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, out) == cudaSuccess) out_dev = attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged;
        else cudaGetLastError();
        out_dev = out_dev && (reinterpret_cast<uintptr_t>(out) & 15u) == 0;
      }
      VoxFusedArgs fa;
      fa.raw = sc.staging.as<unsigned char>(); fa.lay = lay; fa.n = ni; fa.inv = inv; fa.crop = crop; fa.xf = xf;
      fa.pts = pts;
      fa.keys_a = sc.keys_a.as<unsigned>(); fa.vals_a = sc.vals_a.as<unsigned>();
      fa.keys_b = sc.keys_b.as<unsigned>(); fa.vals_b = sc.vals_b.as<unsigned>();
      fa.hist = reinterpret_cast<unsigned short*>(sc.hist.as<int>());
      fa.bar = sc.vox_bar.as<unsigned>();
      fa.part = reinterpret_cast<float*>(sc.hist.as<int>() + (size_t)VF_BINS * fg);
      fa.blk_heads = sc.hist.as<int>() + (size_t)VF_BINS * fg + 8 * (size_t)fg;
      fa.out = sc.vox_out.as<float>(); fa.slot_of_point = sc.vox_slot.as<int>(); fa.d = d;
      fa.result = sc.vox_result_dev;
      fa.user_out = out_dev ? reinterpret_cast<float4*>(out) : nullptr; fa.user_cap = out_cap;
      void* kargs[] = {(void*)&fa};
      if ((e = cudaLaunchCooperativeKernel((const void*)vox_fused_kernel, dim3(fg), dim3(VF_THREADS), kargs, sizeof(VoxFusedSmem), st->s)) != cudaSuccess) return e;
      note_launches(1);
      if ((e = cudaStreamSynchronize(st->s)) != cudaSuccess) return e;
      const int r_m = sc.vox_result[0], r_over = sc.vox_result[1];
      if (!r_over) {
        sc.vox_bits_hint = sc.vox_result[2];
        *m_out = (size_t)r_m;
        if (out_dev && (size_t)r_m <= out_cap) *copied = true;
        return cudaGetLastError();
      }
      // PCL's index-range overflow (leaf far too small for the cloud's extent): handled by the exact path below
    }
  }
  vox_desc_init_kernel<<<1, 1, 0, st->s>>>(d);
  vox_pack_kernel<<<vgrid(ni, 256), 256, 0, st->s>>>(sc.staging.as<unsigned char>(), lay, ni, pts, d, crop, xf);
  note_launches(2);
  int* flags = sc.flags.as<int>();
  auto compact = [&]() -> cudaError_t {
    vox_keep_flags_kernel<<<vgrid(ni + 1, 256), 256, 0, st->s>>>(pts, ni, flags);
    int len = ni + 1;
    cudaError_t ce;
    if ((ce = cudaMemcpyAsync(&d->n, &len, sizeof(int), cudaMemcpyHostToDevice, st->s)) != cudaSuccess) return ce;
    exclusive_scan_inplace(flags, &d->n, 0, ni + 1, sc.tile_sums.as<int>(), st->s);
    vox_compact_kernel<<<vgrid(ni, 256), 256, 0, st->s>>>(pts, ni, flags, sc.vox_out.as<float>(), sc.vox_slot.as<int>());
    note_launches(2);
    int host_m = 0;
    if ((ce = cudaMemcpyAsync(&host_m, flags + ni, sizeof(int), cudaMemcpyDeviceToHost, st->s)) != cudaSuccess) return ce;
    if ((ce = cudaStreamSynchronize(st->s)) != cudaSuccess) return ce;
    *m_out = (size_t)host_m;
    return cudaGetLastError();
  };
  if (!use_grid) return compact();
  vox_setup_kernel<<<1, 1, 0, st->s>>>(d, inv);
  vox_keys_kernel<<<vgrid(ni, 256), 256, 0, st->s>>>(pts, ni, d, inv, sc.keys_a.as<unsigned>(), sc.vals_a.as<unsigned>());
  // ---- speculative path: queue everything behind the key pass with the number of radix passes the PREVIOUS cloud
  //      needed (consecutive scans have nearly the same extent), let the last kernel report {m, overflow, bits needed}
  //      through mapped memory and synchronise ONCE.  More passes than needed are harmless; if this cloud needed more,
  //      or overflowed PCL's index range, the call is redone on the exact path below (rare). ----
  if (allow_speculation && sc.vox_bits_hint > 0) {
    if (!sc.vox_result) {
      if (cudaHostAlloc(&sc.vox_result, 8 * sizeof(int), cudaHostAllocMapped) != cudaSuccess ||
          cudaHostGetDevicePointer(&sc.vox_result_dev, sc.vox_result, 0) != cudaSuccess) { cudaGetLastError(); sc.vox_result = nullptr; }
    }
    if (sc.vox_result) {
      const int bits = sc.vox_bits_hint;
      const int where = radix_sort_pairs(sc.keys_a.as<unsigned>(), sc.vals_a.as<unsigned>(), sc.keys_b.as<unsigned>(), sc.vals_b.as<unsigned>(),
                                         ni, bits, sc.hist.as<int>(), st->s);
      const unsigned* keys = where ? sc.keys_b.as<unsigned>() : sc.keys_a.as<unsigned>();
      const unsigned* perm = where ? sc.vals_b.as<unsigned>() : sc.vals_a.as<unsigned>();
      vox_heads_kernel<<<vgrid(ni + 1, 256), 256, 0, st->s>>>(keys, ni, flags, d);
      exclusive_scan_inplace(flags, &d->n, 0, ni + 1, sc.tile_sums.as<int>(), st->s);
      vox_centroid_kernel<<<vgrid(ni, 128), 128, 0, st->s>>>(keys, perm, ni, flags, pts, sc.vox_out.as<float>(), sc.vox_slot.as<int>(), d);
      vox_result_kernel<<<1, 1, 0, st->s>>>(d, flags + ni, sc.vox_result_dev);
      note_launches(4);
      bool out_dev = false;
      if (out && copied) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, out) == cudaSuccess) out_dev = attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged;
        else cudaGetLastError();
        out_dev = out_dev && (reinterpret_cast<uintptr_t>(out) & 15u) == 0;
        if (out_dev) {
          vox_copy_out_kernel<<<vgrid(ni, 256), 256, 0, st->s>>>(sc.vox_out.as<float4>(), flags + ni, out_cap, reinterpret_cast<float4*>(out));
          note_launches(1);
        }
      }
      if ((e = cudaStreamSynchronize(st->s)) != cudaSuccess) return e;
      const int r_m = sc.vox_result[0], r_over = sc.vox_result[1], r_bits = sc.vox_result[2];
      if (!r_over && r_bits <= bits) {
        sc.vox_bits_hint = r_bits;
        *m_out = (size_t)r_m;
        if (out_dev && (size_t)r_m <= out_cap) *copied = true;
        return cudaGetLastError();
      }
      // mis-speculated: redo exactly (the staging copy and the packed points are still in place, but keep it simple)
      sc.vox_bits_hint = 0;
      return voxel_filter_records(in, n, lay, leaf, sc, st, m_out, overflow, crop6, compact_on_overflow, T16, out, out_cap, copied, false);
    }
  }
  // the voxel grid dimensions decide how many radix passes are needed: one small read-back (the call has to
  // synchronise for the output count anyway) instead of always sorting 32 bits
  int dims[4] = {1, 1, 1, 0};
  if ((e = cudaMemcpyAsync(dims, d->vdiv, 3 * sizeof(int), cudaMemcpyDeviceToHost, st->s)) != cudaSuccess) return e;
  if ((e = cudaMemcpyAsync(dims + 3, &d->voverflow, sizeof(int), cudaMemcpyDeviceToHost, st->s)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(st->s)) != cudaSuccess) return e;
  *overflow = dims[3];
  if (dims[3]) {                                     // PCL passes the input through
    if (compact_on_overflow) return compact();       // ... which, after removeNaN + CropBox, is the surviving points
    *m_out = 0;
    return cudaSuccess;                              // plain voxel filter: the caller copies the raw input
  }
  const unsigned invalid_key = (unsigned)((long long)dims[0] * dims[1] * dims[2]);
  int bits = 1;
  while (bits < 32 && (1ull << bits) <= (unsigned long long)invalid_key) bits++;
  const int where = radix_sort_pairs(sc.keys_a.as<unsigned>(), sc.vals_a.as<unsigned>(), sc.keys_b.as<unsigned>(), sc.vals_b.as<unsigned>(),
                                     ni, bits, sc.hist.as<int>(), st->s);
  const unsigned* keys = where ? sc.keys_b.as<unsigned>() : sc.keys_a.as<unsigned>();
  const unsigned* perm = where ? sc.vals_b.as<unsigned>() : sc.vals_a.as<unsigned>();
  sc.vox_bits_hint = bits;
  vox_heads_kernel<<<vgrid(ni + 1, 256), 256, 0, st->s>>>(keys, ni, flags, d);   // also parks the scan length n+1 in the descriptor
  exclusive_scan_inplace(flags, &d->n, 0, ni + 1, sc.tile_sums.as<int>(), st->s);
  vox_centroid_kernel<<<vgrid(ni, 128), 128, 0, st->s>>>(keys, perm, ni, flags, pts, sc.vox_out.as<float>(), sc.vox_slot.as<int>(), d);
  note_launches(4);
  int host_m = 0;
  if ((e = cudaMemcpyAsync(&host_m, flags + ni, sizeof(int), cudaMemcpyDeviceToHost, st->s)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(st->s)) != cudaSuccess) return e;
  *m_out = (size_t)host_m;
  return cudaGetLastError();
}

}  // namespace ngicp
