// api.cu — the C ABI of libnanogicp_b200.so (include/nanogicp_c.h) and the host side of a handle:
// device-resident clouds / covariances with O(1) sharing and swapping, the stepped LM driver, and
// the import/export of Eigen::Matrix4d covariance records.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "internal.h"
#include "gicp_math.cuh"

using namespace ngicp;

struct ngicp_handle {
  int device = 0;
  // Two streams per handle.  `stream` carries the target side (setInputTarget, target covariances), the registration
  // itself and everything else; `stream_src` carries the SOURCE side (setInputSource / registerInputSource, source
  // covariances) with its own scratch, so that the scan's index + covariances run beside the submap's instead of behind
  // them (C2: 0.18 ms of small, latency-bound kernels).  Every entry point that needs the source on the main stream joins
  // first (join_source).  A caller-supplied stream (ngicp_set_stream) serves both sides: no concurrency, plain stream order.
  StreamPtr stream, stream_src;
  ngicp_params prm;
  std::string err;
  CloudPtr src, tgt;
  CovsPtr src_cov, tgt_cov;
  Scratch sc, sc_src;
  cudaEvent_t ev_join = nullptr, ev_retire = nullptr;
  bool src_pending = false;             // work queued on stream_src that the main stream has not waited for yet
  int nbr_side = NGICP_TARGET;          // which scratch holds the neighbour lists of nbr_cloud
  ngicp_result* res_pinned = nullptr;   // pinned + mapped host memory the fused kernel writes its result to
  ngicp_result* res_mapped = nullptr;   // device-side address of res_pinned
  double* red_pinned = nullptr;         // pinned host mirror of reduced[]
  cudaEvent_t ev[6][2] = {};            // one begin/end pair per timed phase
  bool ev_used[6] = {false, false, false, false, false, false};
  ngicp_timings tm;
  bool lin_valid = false;               // correspondences_/mahalanobis_ valid for compute_error
  std::weak_ptr<DevCloud> nbr_cloud;    // the cloud whose neighbour lists sc.nbr holds (ngicp_cov_neighbors), and their k
  int nbr_k = 0;
  int align_max_blocks = 2048;
  int slab_axis = -1;
  float slab_lo = 0.f, slab_hi = 0.f;
  // sharded-submap mode: exchange buffers of all ranks (own one allocated here, peers IPC-mapped or in-process)
  void* comm_buf = nullptr;
  void* comm_peer[NGICP_MAX_RANKS] = {};
  bool comm_peer_ipc[NGICP_MAX_RANKS] = {};
  PeerComm comm;
  bool comm_on = false;
  // results of ngicp_fitness_batch when this handle leads the batch: pinned + mapped, written by the finalize kernel
  FitnessResult* fit_pinned = nullptr;
  FitnessResult* fit_mapped = nullptr;
  size_t fit_cap = 0;
};

// N1: device-resident keyframe store (SURVEY §8f).  A keyframe is the pair DLO keeps on the host — the voxelised
// world-frame cloud (keyframes[i].second, odom.cc:503,1177) and its covariances (keyframe_normals[i], :500,1174) — held
// here as references to the immutable device buffers the S2S object already made for them.
struct ngicp_kfstore {
  int device = 0;
  // points are copied (16 B each) so that the keyframe does not pin the S2S object's search index (a 128 MiB cell
  // table per cloud); the covariance buffer is immutable and simply shared
  struct Keyframe { std::shared_ptr<DevBuf> pts; int n = 0; CovsPtr covs; cudaEvent_t ready = nullptr; };
  std::vector<Keyframe> kf;
  std::string err;
};

namespace ngicp {
static unsigned long long g_launches = 0;
void note_launches(int n) { __atomic_fetch_add(&g_launches, (unsigned long long)n, __ATOMIC_RELAXED); }
}  // namespace ngicp

namespace {

int fail(ngicp_t* h, int code, const char* what, cudaError_t e = cudaSuccess) {
  if (h) {
    char buf[512];
    if (e != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
    else snprintf(buf, sizeof buf, "%s", what);
    h->err = buf;
  }
  return code;
}

#define NG_CUDA(h, call)                                              \
  do {                                                                \
    cudaError_t _e = (call);                                          \
    if (_e != cudaSuccess) return fail(h, NGICP_E_CUDA, #call, _e);   \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

enum Phase { PH_SET_SRC = 0, PH_SET_TGT, PH_COV_SRC, PH_COV_TGT, PH_ALIGN, PH_VOXEL, PH_COUNT };
inline StreamPtr& side_stream(ngicp_t* h, int which) { return which == NGICP_SOURCE ? h->stream_src : h->stream; }
inline Scratch& side_scratch(ngicp_t* h, int which) { return which == NGICP_SOURCE ? h->sc_src : h->sc; }
inline cudaStream_t ph_stream(ngicp_t* h, int ph);
inline void ph_begin(ngicp_t* h, int ph) { cudaEventRecord(h->ev[ph][0], ph_stream(h, ph)); }
inline void ph_end(ngicp_t* h, int ph) { cudaEventRecord(h->ev[ph][1], ph_stream(h, ph)); h->ev_used[ph] = true; }

// the main stream waits for everything queued on the source-side stream so far
inline void join_source(ngicp_t* h) {
  if (h->src_pending && h->stream_src->s != h->stream->s) {
    cudaEventRecord(h->ev_join, h->stream_src->s);
    cudaStreamWaitEvent(h->stream->s, h->ev_join, 0);
  }
  h->src_pending = false;
}
inline void sync_both(ngicp_t* h) {
  if (h->stream_src && h->stream_src->s && h->stream_src->s != h->stream->s) cudaStreamSynchronize(h->stream_src->s);
  if (h->stream && h->stream->s) cudaStreamSynchronize(h->stream->s);
  h->src_pending = false;
}
// Device buffers are freed in the order of the stream that allocated them.  A buffer that leaves role `which` (source /
// target) after a swap may have been allocated on the OTHER side's stream while this side's stream still reads it:
// make the allocating stream wait for this side before the release is queued.
inline void order_free_after(ngicp_t* h, const StreamPtr& alloc_st, int which) {
  const StreamPtr& role = side_stream(h, which);
  if (!alloc_st || !alloc_st->s || !role || alloc_st->s == role->s) return;
  cudaEventRecord(h->ev_retire, role->s);
  cudaStreamWaitEvent(alloc_st->s, h->ev_retire, 0);
}
inline void drop_cloud(ngicp_t* h, int which) {
  CloudPtr& c = which == NGICP_SOURCE ? h->src : h->tgt;
  if (c && c.use_count() == 1) order_free_after(h, c->pts.st, which);
  c.reset();
}
inline void drop_covs(ngicp_t* h, int which) {
  CovsPtr& c = which == NGICP_SOURCE ? h->src_cov : h->tgt_cov;
  if (c && c.use_count() == 1) order_free_after(h, c->c.st, which);
  c.reset();
}

__global__ void mat4_to_sym6_kernel(const double* __restrict__ m, int n, double* __restrict__ c) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double* s = m + (size_t)i * 16;
    double* d = c + (size_t)i * 6;
    // column-major 4x4: (r,c) at [c*4+r]; upper triangle of the 3x3 block
    d[0] = s[0]; d[1] = s[4]; d[2] = s[8]; d[3] = s[5]; d[4] = s[9]; d[5] = s[10];
  }
}
__global__ void sym6_to_mat4_kernel(const double* __restrict__ c, int n, double* __restrict__ m) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double* s = c + (size_t)i * 6;
    double* d = m + (size_t)i * 16;
    d[0] = s[0]; d[1] = s[1]; d[2] = s[2]; d[3] = 0.0;
    d[4] = s[1]; d[5] = s[3]; d[6] = s[4]; d[7] = 0.0;
    d[8] = s[2]; d[9] = s[4]; d[10] = s[5]; d[11] = 0.0;
    d[12] = 0.0; d[13] = 0.0; d[14] = 0.0; d[15] = 0.0;
  }
}
struct Mat16f { float m[16]; };
__global__ void transform_points_kernel(const float4* __restrict__ pts, int n, Mat16f T, float4* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    float r[3];
#pragma unroll
    for (int k = 0; k < 3; k++)
      r[k] = __fadd_rn(__fadd_rn(__fmul_rn(T.m[0 * 4 + k], p.x), __fmul_rn(T.m[1 * 4 + k], p.y)), __fadd_rn(__fmul_rn(T.m[2 * 4 + k], p.z), T.m[3 * 4 + k]));
    out[i] = make_float4(r[0], r[1], r[2], 1.0f);
  }
}
__global__ void vox_passthrough_kernel(const float4* __restrict__ pts, int n, float* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    float4* o = reinterpret_cast<float4*>(out + (size_t)i * 8);
    o[0] = make_float4(p.x, p.y, p.z, 1.0f);
    o[1] = make_float4(p.w, 0.f, 0.f, 0.f);
  }
}

inline cudaStream_t ph_stream(ngicp_t* h, int ph) { return (ph == PH_SET_SRC || ph == PH_COV_SRC) ? h->stream_src->s : h->stream->s; }

inline int blocks_for(int n) { int g = (n + 255) / 256; return g < 1 ? 1 : (g > 148 * 8 ? 148 * 8 : g); }

int set_cloud(ngicp_t* h, int which, const void* pts, size_t n, size_t stride, bool index) {
  if (!h) return NGICP_E_INVALID;
  if ((!pts && n) || stride < 12 || (stride & 3) || n > 0x7fffff00u) return fail(h, NGICP_E_INVALID, "bad cloud arguments");
  DeviceGuard g(h->device);
  CloudPtr c(new (std::nothrow) DevCloud());
  if (!c) return fail(h, NGICP_E_INVALID, "out of host memory");
  const int ph = which == NGICP_SOURCE ? PH_SET_SRC : PH_SET_TGT;
  StreamPtr& st = side_stream(h, which);
  Scratch& sc = side_scratch(h, which);
  ph_begin(h, ph);
  bool fused = false;
  if (index) NG_CUDA(h, upload_and_index_fused(*c, pts, n, stride, h->prm.grid_cell_size, h->prm.grid_table_cells, sc, st, h->device, &fused));
  if (!fused) {
    NG_CUDA(h, upload_cloud(*c, pts, n, stride, sc, st));
    if (index) NG_CUDA(h, build_index(*c, h->prm.grid_cell_size, h->prm.grid_table_cells, sc, st, h->device));
  }
  ph_end(h, ph);
  drop_cloud(h, which);
  if (which == NGICP_SOURCE) { h->src = c; if (index) drop_covs(h, NGICP_SOURCE); h->src_pending = true; }
  else { h->tgt = c; drop_covs(h, NGICP_TARGET); }
  h->lin_valid = false;
  return NGICP_OK;
}

int ensure_index(ngicp_t* h, CloudPtr& c, int which) {
  if (c->indexed) return NGICP_OK;
  NG_CUDA(h, build_index(*c, h->prm.grid_cell_size, h->prm.grid_table_cells, side_scratch(h, which), side_stream(h, which), h->device));
  return NGICP_OK;
}

int calc_covs(ngicp_t* h, int which, int part = 0, int nparts = 1) {
  if (!h) return NGICP_E_INVALID;
  if (nparts < 1 || part < 0 || part >= nparts) return fail(h, NGICP_E_INVALID, "calculate covariances: bad part / nparts");
  DeviceGuard g(h->device);
  CloudPtr& c = which == NGICP_SOURCE ? h->src : h->tgt;
  if (!c) return fail(h, NGICP_E_STATE, "calculate covariances: cloud not set");
  const int k = h->prm.k_correspondences;
  if (k < 1 || k > KNN_WIDE_MAX_K) return fail(h, NGICP_E_UNSUPPORTED, "k_correspondences must be in [1,128]");
  if (c->n < k) return fail(h, NGICP_E_TOO_FEW_POINTS, "cloud has fewer points than k_correspondences");
  StreamPtr& st = side_stream(h, which);
  Scratch& sc = side_scratch(h, which);
  int rc = ensure_index(h, c, which);  // calculate_covariances re-targets the kd-tree when needed (nano_gicp_impl.hpp:304-306)
  if (rc) return rc;
  CovsPtr cv(new (std::nothrow) DevCovs());
  if (!cv) return fail(h, NGICP_E_INVALID, "out of host memory");
  cv->n = c->n;
  NG_CUDA(h, cv->c.alloc(sizeof(double) * 6 * (size_t)c->n, st));
  const int ph = which == NGICP_SOURCE ? PH_COV_SRC : PH_COV_TGT;
  ph_begin(h, ph);
  NG_CUDA(h, sc.nbr.reserve(sizeof(int) * covariance_scratch_ints(c->n, k, c->table_cap), st));
  h->nbr_cloud.reset();
  if (!sc.cov_side.stream) {
    int lo_pri = 0, hi_pri = 0;
    cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri);
    NG_CUDA(h, cudaStreamCreateWithPriority(&sc.cov_side.stream, cudaStreamNonBlocking, hi_pri));
    NG_CUDA(h, cudaEventCreateWithFlags(&sc.cov_side.fork, cudaEventDisableTiming));
    NG_CUDA(h, cudaEventCreateWithFlags(&sc.cov_side.join, cudaEventDisableTiming));
  }
  // AUTO chooses by cloud size (tiles from knn_tile_min_points on: fewer instructions per point, but a long serial path
  // per warp — worse LATENCY for a scan).  One exception: the source of a handle whose target is a large submap.  Its
  // work runs on the second stream BESIDE the submap's, so what counts is the GPU time it takes away from the target
  // side, not its own latency: tiles (measured on C2: 22k-point scan, step 0.884 -> 0.853 ms).  Both paths give the same
  // neighbour sets and the same summation order.
  int knn_path = h->prm.knn_path;
  if (knn_path == NGICP_KNN_AUTO && which == NGICP_SOURCE && nparts == 1 && c->n >= 8192 && h->tgt &&
      h->tgt->n >= h->prm.knn_tile_min_points && h->stream_src->s != h->stream->s)
    knn_path = NGICP_KNN_TILE;
  NG_CUDA(h, launch_covariances(*c, k, h->prm.regularization_method, sc.nbr.as<int>(), cv->c.as<double>(), c->table_cap, st->s,
                                part, nparts, knn_path, h->prm.knn_tile_min_points, &sc.cov_side));
  ph_end(h, ph);
  if (nparts == 1) { h->nbr_cloud = c; h->nbr_k = k; h->nbr_side = which; }
  drop_covs(h, which);
  (which == NGICP_SOURCE ? h->src_cov : h->tgt_cov) = cv;
  if (which == NGICP_SOURCE) h->src_pending = true;
  h->lin_valid = false;
  return NGICP_OK;
}

int set_covs(ngicp_t* h, int which, const double* covs, size_t n) {
  if (!h || (!covs && n)) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  CovsPtr cv(new (std::nothrow) DevCovs());
  if (!cv) return fail(h, NGICP_E_INVALID, "out of host memory");
  cv->n = (int)n;
  StreamPtr& st = side_stream(h, which);
  Scratch& sc = side_scratch(h, which);
  NG_CUDA(h, cv->c.alloc(sizeof(double) * 6 * (n ? n : 1), st));
  if (n) {
    NG_CUDA(h, sc.cov_stage.reserve(sizeof(double) * 16 * n, st));
    NG_CUDA(h, cudaMemcpyAsync(sc.cov_stage.p, covs, sizeof(double) * 16 * n, cudaMemcpyDefault, st->s));
    NG_CUDA(h, host_source_consumed(covs, sc, st->s));
    mat4_to_sym6_kernel<<<blocks_for((int)n), 256, 0, st->s>>>(sc.cov_stage.as<double>(), (int)n, cv->c.as<double>());
    note_launches(1);
    NG_CUDA(h, cudaGetLastError());
  }
  drop_covs(h, which);
  (which == NGICP_SOURCE ? h->src_cov : h->tgt_cov) = cv;
  if (which == NGICP_SOURCE) h->src_pending = true;
  h->lin_valid = false;
  return NGICP_OK;
}

int get_covs(ngicp_t* h, int which, double* out, size_t n) {
  if (!h || !out) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  CovsPtr& cv = which == NGICP_SOURCE ? h->src_cov : h->tgt_cov;
  if (!cv || (size_t)cv->n != n) return fail(h, NGICP_E_COV_SIZE, "get covariances: size mismatch");
  if (n == 0) return NGICP_OK;
  join_source(h);
  NG_CUDA(h, h->sc.cov_stage.reserve(sizeof(double) * 16 * n, h->stream));
  sym6_to_mat4_kernel<<<blocks_for((int)n), 256, 0, h->stream->s>>>(cv->c.as<double>(), (int)n, h->sc.cov_stage.as<double>());
  note_launches(1);
  NG_CUDA(h, cudaGetLastError());
  NG_CUDA(h, cudaMemcpyAsync(out, h->sc.cov_stage.p, sizeof(double) * 16 * n, cudaMemcpyDefault, h->stream->s));
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  return NGICP_OK;
}

// everything align/linearize need; also performs the lazy covariance computation of
// NanoGICP::computeTransformation (nano_gicp_impl.hpp:163-168) when `lazy` is set
int prepare_align(ngicp_t* h, bool lazy, AlignBuffers& ab) {
  if (!h->src || !h->tgt) return fail(h, NGICP_E_STATE, "align: source/target not set");
  if (h->src->n == 0 || h->tgt->n == 0) return fail(h, NGICP_E_STATE, "align: empty cloud");
  if (!h->tgt->indexed) return fail(h, NGICP_E_STATE, "align: target has no search index");
  if (!h->src_cov || h->src_cov->n != h->src->n) {
    if (!lazy) return fail(h, NGICP_E_COV_SIZE, "source covariances missing");
    int rc = calc_covs(h, NGICP_SOURCE);
    if (rc) return rc;
  }
  if (!h->tgt_cov || h->tgt_cov->n != h->tgt->n) {
    if (!lazy) return fail(h, NGICP_E_COV_SIZE, "target covariances missing");
    int rc = calc_covs(h, NGICP_TARGET);
    if (rc) return rc;
  }
  join_source(h);   // the source's index and covariances are queued on the source-side stream
  const size_t ns = (size_t)h->src->n;
  Scratch& sc = h->sc;
  NG_CUDA(h, sc.mahal.reserve(sizeof(double) * 6 * ns, h->stream));
  NG_CUDA(h, sc.corr.reserve(sizeof(int) * ns, h->stream));
  NG_CUDA(h, sc.sqd.reserve(sizeof(float) * ns, h->stream));
  NG_CUDA(h, sc.tgt_pt.reserve(sizeof(float4) * ns, h->stream));
  NG_CUDA(h, sc.partials.reserve(sizeof(double) * NRED * (size_t)h->align_max_blocks * 2, h->stream));   // two phase-parity halves
  NG_CUDA(h, sc.reduced.reserve(sizeof(double) * 64, h->stream));
  if (!sc.barrier.p) {   // zeroed once; the fused kernel leaves it zeroed (last departing block)
    NG_CUDA(h, sc.barrier.reserve(64, h->stream));
    NG_CUDA(h, cudaMemsetAsync(sc.barrier.p, 0, 64, h->stream->s));
  }
  ab.src_pts = h->src->pts.as<float4>(); ab.src_cov = h->src_cov->c.as<double>(); ab.ns = h->src->n;
  ab.tgt = h->tgt->view(); ab.tgt_cov = h->tgt_cov->c.as<double>(); ab.nt = h->tgt->n;
  ab.mahal = sc.mahal.as<double>(); ab.corr = sc.corr.as<int>(); ab.sqd = sc.sqd.as<float>(); ab.tgt_pt = sc.tgt_pt.as<float4>();
  ab.partials = sc.partials.as<double>(); ab.reduced = sc.reduced.as<double>(); ab.max_blocks = h->align_max_blocks;
  ab.slab_axis = h->slab_axis; ab.slab_lo = h->slab_lo; ab.slab_hi = h->slab_hi;
  return NGICP_OK;
}

int fetch_reduced(ngicp_t* h, int count) {
  NG_CUDA(h, cudaMemcpyAsync(h->red_pinned, h->sc.reduced.p, sizeof(double) * count, cudaMemcpyDeviceToHost, h->stream->s));
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  return NGICP_OK;
}

// host-stepped LM: identical decisions to the fused kernel, one launch per phase
int align_stepped(ngicp_t* h, const AlignBuffers& ab, const float* guess16, ngicp_result* out) {
  const ngicp_params& p = h->prm;
  Iso3 x0, xi, delta;
  double g16[16];
  for (int i = 0; i < 16; i++) g16[i] = guess16 ? (double)guess16[i] : ((i % 5 == 0) ? 1.0 : 0.0);
  iso_from_colmajor16(g16, x0);
  iso_identity(delta);
  double H36[36], b6[6], d6[6] = {0, 0, 0, 0, 0, 0}, final_H[36];
  for (int i = 0; i < 36; i++) final_H[i] = (i % 7 == 0) ? 1.0 : 0.0;
  double lambda = -1.0, y0 = 0.0;
  int nr_iterations = 0, n_lin = 0, n_err = 0, lm_failed = 0;
  bool converged = false;
  double T16[16];
  for (int it = 0; it < p.max_iterations && !converged; ++it) {
    nr_iterations = it;
    iso_to_colmajor16(x0, T16);
    NG_CUDA(h, launch_linearize(ab, T16, p.max_correspondence_distance, h->stream->s));
    int rc = fetch_reduced(h, NRED);
    if (rc) return rc;
    n_lin++;
    unpack_H(h->red_pinned, H36);
    for (int i = 0; i < 6; i++) b6[i] = h->red_pinned[21 + i];
    y0 = h->red_pinned[27];
    bool ok = false;
    if (p.optimizer == NGICP_OPT_GAUSS_NEWTON) {
      double nb[6];
      for (int i = 0; i < 6; i++) nb[i] = -b6[i];
      lm_solve(H36, nb, d6);
      delta_from_step(d6, delta);
      iso_mul(delta, x0, xi);
      x0 = xi;
      memcpy(final_H, H36, sizeof final_H);
      ok = true;
    } else {
      if (lambda < 0.0) {
        double mx = 0.0;
        for (int i = 0; i < 6; i++) mx = fmax(mx, fabs(H36[i * 7]));
        lambda = p.lm_init_lambda_factor * mx;
      }
      double nu = 2.0;
      for (int j = 0; j < p.lm_max_iterations; ++j) {
        double A[36], nb[6];
        memcpy(A, H36, sizeof A);
        for (int i = 0; i < 6; i++) { A[i * 7] += lambda; nb[i] = -b6[i]; }
        lm_solve(A, nb, d6);
        delta_from_step(d6, delta);
        iso_mul(delta, x0, xi);
        iso_to_colmajor16(xi, T16);
        NG_CUDA(h, launch_compute_error(ab, T16, h->stream->s));
        rc = fetch_reduced(h, 1);
        if (rc) return rc;
        n_err++;
        const double yi = h->red_pinned[0];
        double denom = 0.0;
        for (int i = 0; i < 6; i++) denom += d6[i] * (lambda * d6[i] - b6[i]);
        const double rho = (y0 - yi) / denom;
        if (rho < 0) {
          if (lm_is_converged(delta, p.rotation_epsilon, p.transformation_epsilon)) { ok = true; break; }
          lambda = nu * lambda;
          nu = 2 * nu;
          continue;
        }
        x0 = xi;
        const double w3 = 2.0 * rho - 1.0;
            const double v = 1.0 - w3 * w3 * w3;
        lambda = lambda * ((1.0 / 3.0 < v) ? v : 1.0 / 3.0);
        memcpy(final_H, H36, sizeof final_H);
        ok = true;
        break;
      }
    }
    if (!ok) { lm_failed = 1; break; }
    converged = lm_is_converged(delta, p.rotation_epsilon, p.transformation_epsilon);
  }
  iso_to_colmajor16(x0, T16);
  for (int i = 0; i < 16; i++) { out->final_x[i] = T16[i]; out->final_transformation[i] = (float)T16[i]; }
  memcpy(out->final_hessian, final_H, sizeof final_H);
  out->lm_lambda = lambda;
  out->last_error = y0;
  out->nr_iterations = nr_iterations;
  out->converged = converged ? 1 : 0;
  out->n_linearize = n_lin;
  out->n_compute_error = n_err;
  out->lm_failed = lm_failed;
  out->reserved = 0;
  return NGICP_OK;
}

}  // namespace

extern "C" {

int ngicp_grid_info(ngicp_t* h, int which, float* cell, int* dims3, int* ncells) {
  if (!h) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  CloudPtr& c = which == NGICP_SOURCE ? h->src : h->tgt;
  if (!c || !c->indexed) return fail(h, NGICP_E_STATE, "grid info: no search index");
  join_source(h);
  GridDesc d;
  NG_CUDA(h, cudaMemcpyAsync(&d, c->desc.p, sizeof d, cudaMemcpyDeviceToHost, h->stream->s));
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  if (cell) *cell = d.cell;
  if (dims3) { dims3[0] = d.dim[0]; dims3[1] = d.dim[1]; dims3[2] = d.dim[2]; }
  if (ncells) *ncells = d.ncells;
  return NGICP_OK;
}

unsigned long long ngicp_launch_count(void) { return __atomic_load_n(&ngicp::g_launches, __ATOMIC_RELAXED); }

const char* ngicp_version(void) { return "nanogicp-b200 0.1 sm_100a"; }

void ngicp_params_default(ngicp_params* p) {
  if (!p) return;
  p->k_correspondences = 20;
  p->max_correspondence_distance = (double)FLT_MAX;
  p->max_iterations = 64;
  p->transformation_epsilon = 5e-4;
  p->rotation_epsilon = 2e-3;
  p->optimizer = NGICP_OPT_LEVENBERG_MARQUARDT;
  p->lm_max_iterations = 10;
  p->lm_init_lambda_factor = 1e-9;
  p->regularization_method = NGICP_REG_PLANE;
  p->grid_cell_size = 0.f;
  p->grid_table_cells = 1 << 25;
  p->align_mode = NGICP_ALIGN_FUSED;
  p->knn_path = NGICP_KNN_AUTO;
  p->knn_tile_min_points = 131072;
  p->voxel_path = 0;
  p->index_path = 0;
}

int ngicp_create(int device, ngicp_t** out) {
  if (!out) return NGICP_E_INVALID;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return NGICP_E_CUDA;  // no CPU fallback, by design
  if (device < 0 || device >= count) return NGICP_E_INVALID;
  DeviceGuard g(device);
  ngicp_handle* h = new (std::nothrow) ngicp_handle();
  if (!h) return NGICP_E_INVALID;
  h->device = device;
  ngicp_params_default(&h->prm);
  memset(&h->tm, 0, sizeof h->tm);
  h->stream.reset(new StreamRef());
  if (cudaStreamCreateWithFlags(&h->stream->s, cudaStreamNonBlocking) != cudaSuccess) { delete h; return NGICP_E_CUDA; }
  h->stream->owned = true;
  h->stream_src.reset(new StreamRef());
  if (cudaStreamCreateWithFlags(&h->stream_src->s, cudaStreamNonBlocking) != cudaSuccess) { h->stream_src.reset(); delete h; return NGICP_E_CUDA; }
  h->stream_src->owned = true;
  // (device memory comes from the library's own stream-ordered pool, pool_alloc_async: freed blocks stay there instead of
  //  going back to the driver, and the application's default pool is left alone)
  // mapped: the fused kernel stores its 496-byte result straight into host memory (no D2H copy node after it)
  bool ok = cudaHostAlloc(&h->res_pinned, sizeof(ngicp_result), cudaHostAllocMapped) == cudaSuccess &&
            cudaHostGetDevicePointer(&h->res_mapped, h->res_pinned, 0) == cudaSuccess &&
            cudaMallocHost(&h->red_pinned, sizeof(double) * 64) == cudaSuccess;
  for (int i = 0; ok && i < PH_COUNT; i++)
    ok = cudaEventCreate(&h->ev[i][0]) == cudaSuccess && cudaEventCreate(&h->ev[i][1]) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) == cudaSuccess &&
       cudaEventCreateWithFlags(&h->ev_retire, cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    ngicp_destroy(h);
    return NGICP_E_CUDA;
  }
  // Working-set priming, once per device and process: grow the stream-ordered pool to NGICP_POOL_PRIME_MB (default 512)
  // and park NGICP_TABLE_PRIME (default 5) cell tables in the free list, so that the first scans of a stream do not pay
  // for driver-level allocations (a fresh 128 MiB cudaMalloc costs 0.6-25 ms, pool growth ~10 ms per step; measured
  // with benchmarks/configs.py c3).  Both are one-time costs of ngicp_create.
  {
    static std::mutex prime_mutex;
    static bool primed[64] = {};
    std::lock_guard<std::mutex> prime_lock(prime_mutex);
    if (device < 64 && !primed[device]) {
      primed[device] = true;
      const char* e1 = getenv("NGICP_POOL_PRIME_MB");
      const long mb = e1 ? atol(e1) : 512;
      if (mb > 0) {
        void* p = nullptr;
        if (pool_alloc_async(&p, (size_t)mb << 20, h->stream->s) == cudaSuccess) cudaFreeAsync(p, h->stream->s);
        cudaGetLastError();
      }
      const char* e2 = getenv("NGICP_TABLE_PRIME");
      const int nt = e2 ? atoi(e2) : 5;
      const size_t tb = sizeof(int) * ((size_t)h->prm.grid_table_cells + 8);
      std::vector<TableBuf*> tmp;
      for (int i = 0; i < nt && i < 8; i++) {
        TableBuf* t = new (std::nothrow) TableBuf();
        if (!t || t->acquire(tb, device, h->stream) != cudaSuccess) { delete t; cudaGetLastError(); break; }
        tmp.push_back(t);
      }
      for (TableBuf* t : tmp) delete t;   // release() parks them in the free list
      align_prime_kernels(device);
      knn_prime_kernels();
      voxel_prime_kernels();
      index_prime_kernels();
      cudaStreamSynchronize(h->stream->s);
    }
  }
  // NGICP_ALIGN_MAX_BLOCKS caps the persistent LM kernel's grid (default: whatever is co-resident); needed when
  // several handles run their cooperative kernels on ONE GPU at the same time (sharded-mode tests)
  if (const char* e = getenv("NGICP_ALIGN_MAX_BLOCKS")) { const int v = atoi(e); if (v > 0 && v < h->align_max_blocks) h->align_max_blocks = v; }
  *out = h;
  return NGICP_OK;
}

void ngicp_destroy(ngicp_t* h) {
  if (!h) return;
  DeviceGuard g(h->device);
  if (h->stream && h->stream_src) sync_both(h);
  else if (h->stream && h->stream->s) cudaStreamSynchronize(h->stream->s);
  h->src.reset(); h->tgt.reset(); h->src_cov.reset(); h->tgt_cov.reset();
  ngicp_comm_close(h);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->ev_retire) cudaEventDestroy(h->ev_retire);
  if (h->comm_buf) cudaFree(h->comm_buf);
  if (h->res_pinned) cudaFreeHost(h->res_pinned);
  if (h->red_pinned) cudaFreeHost(h->red_pinned);
  if (h->fit_pinned) cudaFreeHost(h->fit_pinned);
  for (int i = 0; i < PH_COUNT; i++)
    for (int j = 0; j < 2; j++)
      if (h->ev[i][j]) cudaEventDestroy(h->ev[i][j]);
  delete h;
}

const char* ngicp_last_error(const ngicp_t* h) { return h ? h->err.c_str() : "null handle"; }

int ngicp_set_stream(ngicp_t* h, void* cuda_stream) {
  if (!h) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  sync_both(h);
  StreamPtr s(new StreamRef()), s2;
  if (cuda_stream) { s->s = (cudaStream_t)cuda_stream; s->owned = false; s2 = s; }   // the caller's stream serves both sides
  else {
    if (cudaStreamCreateWithFlags(&s->s, cudaStreamNonBlocking) != cudaSuccess) return fail(h, NGICP_E_CUDA, "cudaStreamCreate");
    s->owned = true;
    s2.reset(new StreamRef());
    if (cudaStreamCreateWithFlags(&s2->s, cudaStreamNonBlocking) != cudaSuccess) return fail(h, NGICP_E_CUDA, "cudaStreamCreate");
    s2->owned = true;
  }
  h->stream = s;
  h->stream_src = s2;
  return NGICP_OK;
}
void* ngicp_get_stream(const ngicp_t* h) { return h ? (void*)h->stream->s : nullptr; }

int ngicp_sync(ngicp_t* h) {
  if (!h) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  if (h->stream_src->s != h->stream->s) NG_CUDA(h, cudaStreamSynchronize(h->stream_src->s));
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  h->src_pending = false;
  return NGICP_OK;
}

int ngicp_get_timings(ngicp_t* h, ngicp_timings* out) {
  if (!h || !out) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  if (h->stream_src->s != h->stream->s) NG_CUDA(h, cudaStreamSynchronize(h->stream_src->s));
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  h->src_pending = false;
  float* slots[PH_COUNT] = {&h->tm.set_source_ms, &h->tm.set_target_ms, &h->tm.source_covs_ms, &h->tm.target_covs_ms, &h->tm.align_ms, &h->tm.voxel_ms};
  for (int i = 0; i < PH_COUNT; i++)
    if (h->ev_used[i]) cudaEventElapsedTime(slots[i], h->ev[i][0], h->ev[i][1]);
  *out = h->tm;
  return NGICP_OK;
}

int ngicp_set_params(ngicp_t* h, const ngicp_params* p) {
  if (!h || !p) return NGICP_E_INVALID;
  if (p->k_correspondences < 1 || p->k_correspondences > KNN_WIDE_MAX_K) return fail(h, NGICP_E_UNSUPPORTED, "k_correspondences must be in [1,128]");
  if (p->regularization_method < 0 || p->regularization_method > 4) return fail(h, NGICP_E_INVALID, "unknown regularization method");  // the reference abort()s here (nano_gicp_impl.hpp:336-338)
  if (p->grid_table_cells < 64) return fail(h, NGICP_E_INVALID, "grid_table_cells too small");
  if (p->knn_path < NGICP_KNN_AUTO || p->knn_path > NGICP_KNN_TILE) return fail(h, NGICP_E_INVALID, "unknown knn_path");
  if (p->voxel_path < 0 || p->voxel_path > 2) return fail(h, NGICP_E_INVALID, "unknown voxel_path");
  if (p->index_path < 0 || p->index_path > 3) return fail(h, NGICP_E_INVALID, "unknown index_path");
  if (p->align_mode != NGICP_ALIGN_FUSED && p->align_mode != NGICP_ALIGN_STEPPED) return fail(h, NGICP_E_INVALID, "unknown align_mode");
  if (p->optimizer != NGICP_OPT_GAUSS_NEWTON && p->optimizer != NGICP_OPT_LEVENBERG_MARQUARDT) return fail(h, NGICP_E_INVALID, "unknown optimizer");
  h->prm = *p;
  h->sc.vox_path = p->voxel_path;
  h->sc.index_path = p->index_path;
  h->sc_src.index_path = p->index_path;
  h->sc_src.vox_path = p->voxel_path;
  return NGICP_OK;
}
int ngicp_get_params(const ngicp_t* h, ngicp_params* p) {
  if (!h || !p) return NGICP_E_INVALID;
  *p = h->prm;
  return NGICP_OK;
}

int ngicp_set_source(ngicp_t* h, const void* pts, size_t n, size_t stride) { return set_cloud(h, NGICP_SOURCE, pts, n, stride, true); }
int ngicp_set_target(ngicp_t* h, const void* pts, size_t n, size_t stride) { return set_cloud(h, NGICP_TARGET, pts, n, stride, true); }
int ngicp_register_source(ngicp_t* h, const void* pts, size_t n, size_t stride) { return set_cloud(h, NGICP_SOURCE, pts, n, stride, false); }

int ngicp_share_source(ngicp_t* dst, const ngicp_t* src) {
  if (!dst || !src) return NGICP_E_INVALID;
  if (dst->device != src->device) return fail(dst, NGICP_E_INVALID, "handles live on different devices");
  if (!src->src) return fail(dst, NGICP_E_STATE, "share: source not set");
  DeviceGuard g(dst->device);             // dropping the previous cloud frees stream-ordered memory of that device
  sync_both(const_cast<ngicp_t*>(src));   // the index must be complete before another handle's streams read it
  drop_cloud(dst, NGICP_SOURCE);
  dst->src = src->src;
  dst->lin_valid = false;
  return NGICP_OK;
}
int ngicp_share_source_covs(ngicp_t* dst, const ngicp_t* src) {
  if (!dst || !src) return NGICP_E_INVALID;
  if (dst->device != src->device) return fail(dst, NGICP_E_INVALID, "handles live on different devices");
  DeviceGuard g(dst->device);
  sync_both(const_cast<ngicp_t*>(src));
  drop_covs(dst, NGICP_SOURCE);
  dst->src_cov = src->src_cov;
  dst->lin_valid = false;
  return NGICP_OK;
}

int ngicp_swap(ngicp_t* h) {
  if (!h) return NGICP_E_INVALID;
  {
    // the clouds change sides, i.e. streams: nothing may be in flight on either (in OdomNode this follows an align(),
    // which has just synchronised anyway — odom.cc:818)
    DeviceGuard g(h->device);
    sync_both(h);
  }
  h->src.swap(h->tgt);
  h->src_cov.swap(h->tgt_cov);
  h->lin_valid = false;
  return NGICP_OK;
}
// (releasing a cloud frees stream-ordered memory and records events: the handle's device must be current)
int ngicp_clear_source(ngicp_t* h) { if (!h) return NGICP_E_INVALID; DeviceGuard g(h->device); drop_cloud(h, NGICP_SOURCE); drop_covs(h, NGICP_SOURCE); h->lin_valid = false; return NGICP_OK; }
int ngicp_clear_target(ngicp_t* h) { if (!h) return NGICP_E_INVALID; DeviceGuard g(h->device); drop_cloud(h, NGICP_TARGET); drop_covs(h, NGICP_TARGET); h->lin_valid = false; return NGICP_OK; }
size_t ngicp_cloud_size(const ngicp_t* h, int which) {
  if (!h) return 0;
  const CloudPtr& c = which == NGICP_SOURCE ? h->src : h->tgt;
  return c ? (size_t)c->n : 0;
}

int ngicp_calc_source_covs(ngicp_t* h) { return calc_covs(h, NGICP_SOURCE); }
int ngicp_calc_target_covs(ngicp_t* h) { return calc_covs(h, NGICP_TARGET); }
int ngicp_calc_source_covs_part(ngicp_t* h, int part, int nparts) { return calc_covs(h, NGICP_SOURCE, part, nparts); }
int ngicp_covs_device(ngicp_t* h, int which, double** covs6, size_t* n) {
  if (!h || !covs6 || !n) return NGICP_E_INVALID;
  const CovsPtr& cv = which == NGICP_SOURCE ? h->src_cov : h->tgt_cov;
  { DeviceGuard g(h->device); join_source(h); }   // callers continue on the main stream (ngicp_get_stream)
  *covs6 = cv ? cv->c.as<double>() : nullptr;
  *n = cv ? (size_t)cv->n : 0;
  return cv ? NGICP_OK : fail(h, NGICP_E_STATE, "no covariances");
}
int ngicp_cov_neighbors(ngicp_t* h, int which, int* idx, float* d2) {
  if (!h || !idx || !d2) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  CloudPtr& c = which == NGICP_SOURCE ? h->src : h->tgt;
  if (!c || h->nbr_cloud.lock() != c || h->nbr_k < 1) return fail(h, NGICP_E_STATE, "cov_neighbors: the last covariance computation on this handle was not for this cloud");
  const size_t cnt = (size_t)c->n * h->nbr_k;
  join_source(h);
  NG_CUDA(h, h->sc.knn_idx.reserve(sizeof(int) * cnt, h->stream));
  NG_CUDA(h, h->sc.knn_d2.reserve(sizeof(float) * cnt, h->stream));
  NG_CUDA(h, launch_export_neighbors(*c, h->nbr_k, side_scratch(h, h->nbr_side).nbr.as<int>(), h->sc.knn_idx.as<int>(), h->sc.knn_d2.as<float>(), h->stream->s));
  NG_CUDA(h, cudaMemcpyAsync(idx, h->sc.knn_idx.p, sizeof(int) * cnt, cudaMemcpyDefault, h->stream->s));
  NG_CUDA(h, cudaMemcpyAsync(d2, h->sc.knn_d2.p, sizeof(float) * cnt, cudaMemcpyDefault, h->stream->s));
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  return NGICP_OK;
}
int ngicp_set_source_covs(ngicp_t* h, const double* covs, size_t n) { return set_covs(h, NGICP_SOURCE, covs, n); }
int ngicp_set_target_covs(ngicp_t* h, const double* covs, size_t n) { return set_covs(h, NGICP_TARGET, covs, n); }
int ngicp_clear_covs(ngicp_t* h, int which) {
  if (!h) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  drop_covs(h, which);
  h->lin_valid = false;
  return NGICP_OK;
}
size_t ngicp_covs_size(const ngicp_t* h, int which) {
  if (!h) return 0;
  const CovsPtr& c = which == NGICP_SOURCE ? h->src_cov : h->tgt_cov;
  return c ? (size_t)c->n : 0;
}
int ngicp_get_source_covs(ngicp_t* h, double* out, size_t n) { return get_covs(h, NGICP_SOURCE, out, n); }
int ngicp_get_target_covs(ngicp_t* h, double* out, size_t n) { return get_covs(h, NGICP_TARGET, out, n); }

int ngicp_align(ngicp_t* h, const float* guess16, ngicp_result* out) {
  if (!h || !out) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  AlignBuffers ab;
  int rc = prepare_align(h, true, ab);
  if (rc) return rc;
  ph_begin(h, PH_ALIGN);
  if (h->prm.align_mode == NGICP_ALIGN_STEPPED) {
    rc = align_stepped(h, ab, guess16, out);
    if (rc) return rc;
  } else {
    ngicp_result* res_dev = h->res_mapped;
    static const bool want_trace = getenv("NGICP_ALIGN_TRACE") != nullptr;
    unsigned long long* trace = nullptr;
    if (want_trace) {
      NG_CUDA(h, h->sc.trace.reserve(sizeof(unsigned long long) * 1280, h->stream));
      trace = h->sc.trace.as<unsigned long long>();
      NG_CUDA(h, cudaMemsetAsync(trace, 0, sizeof(unsigned long long) * 1280, h->stream->s));
    }
    NG_CUDA(h, launch_align_fused(ab, h->prm, guess16, res_dev, h->sc.barrier.as<unsigned>(), h->device, h->stream->s, trace,
                                  h->comm_on ? &h->comm : nullptr));
    NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
    *out = *h->res_pinned;
    if (h->comm_on && out->reserved != 0) return fail(h, NGICP_E_COMM, "sharded align: a peer rank did not reach the exchange in time");
    if (trace) {
      static unsigned long long t[1280];
      NG_CUDA(h, cudaMemcpy(t, trace, sizeof t, cudaMemcpyDeviceToHost));
      fprintf(stderr, "[align trace, us since start]");
      for (unsigned long long i = 1; i <= t[0] && i < 255; i++) fprintf(stderr, " %.1f", (double)(t[i] - t[1]) * 1e-3);
      fprintf(stderr, "\n[second linearize done per block, us since start]");
      for (int b = 0; b < 1024; b++) if (t[256 + b]) fprintf(stderr, " %.1f", (double)(t[256 + b] - t[1]) * 1e-3);
      fprintf(stderr, "\n");
    }
  }
  ph_end(h, PH_ALIGN);
  h->lin_valid = true;
  if (out->lm_failed) fprintf(stderr, "lm not converged!!\n");  // lsq_registration_impl.hpp:106
  return NGICP_OK;
}

// B independent registrations in one launch: every handle is prepared like a single ngicp_align (lazy covariances,
// per-handle state buffers), the handles' streams are joined into the first one's, and ONE kernel with a thread-block
// cluster per pair runs all the LM loops (align.cu: align_batch_kernel).  Bit-identical to the single calls.
int ngicp_align_batch(ngicp_t* const* hs, size_t n, const float* guesses16, ngicp_result* results) {
  if (!hs || !results || n == 0 || !hs[0]) return NGICP_E_INVALID;
  ngicp_t* h0 = hs[0];
  for (size_t i = 0; i < n; ++i) {
    if (!hs[i]) return fail(h0, NGICP_E_INVALID, "align_batch: null handle");
    if (hs[i]->device != h0->device) return fail(h0, NGICP_E_INVALID, "align_batch: handles live on different devices");
    if (hs[i]->comm_on) return fail(h0, NGICP_E_UNSUPPORTED, "align_batch: a handle is in sharded mode");
    for (size_t j = 0; j < i; ++j)
      if (hs[j] == hs[i]) return fail(h0, NGICP_E_INVALID, "align_batch: the same handle appears twice");
  }
  DeviceGuard g(h0->device);
  const size_t rec = align_batch_pair_bytes();
  std::vector<unsigned char> stage(n * rec), ordered(n * rec);
  std::vector<int> lpp(n);
  ph_begin(h0, PH_ALIGN);
  for (size_t i = 0; i < n; ++i) {
    ngicp_t* h = hs[i];
    AlignBuffers ab;
    int rc = prepare_align(h, true, ab);
    if (rc) { if (h != h0) h0->err = "align_batch: pair " + std::to_string(i) + ": " + h->err; return rc; }
    lpp[i] = align_batch_fill(stage.data() + i * rec, ab, h->prm, guesses16 ? guesses16 + 16 * i : nullptr, h->res_mapped, h->device);
    if (h != h0) {   // everything queued on this handle's stream (index, covariances) precedes the batch kernel
      if (!h->sc.copy_done) NG_CUDA(h0, cudaEventCreateWithFlags(&h->sc.copy_done, cudaEventDisableTiming));
      NG_CUDA(h0, cudaEventRecord(h->sc.copy_done, h->stream->s));
      NG_CUDA(h0, cudaStreamWaitEvent(h0->stream->s, h->sc.copy_done, 0));
    }
  }
  // pairs that need two lanes per source point (target >= 4x the scan) go into a launch of their own
  size_t n1 = 0;
  for (size_t i = 0; i < n; ++i) if (lpp[i] != 2) memcpy(ordered.data() + (n1++) * rec, stage.data() + i * rec, rec);
  size_t n2 = 0;
  for (size_t i = 0; i < n; ++i) if (lpp[i] == 2) memcpy(ordered.data() + (n1 + n2++) * rec, stage.data() + i * rec, rec);
  NG_CUDA(h0, h0->sc.batch_args.reserve(n * rec, h0->stream));
  NG_CUDA(h0, cudaMemcpyAsync(h0->sc.batch_args.p, ordered.data(), n * rec, cudaMemcpyHostToDevice, h0->stream->s));
  NG_CUDA(h0, launch_align_batch(h0->sc.batch_args.p, (int)n1, 1, h0->stream->s));
  NG_CUDA(h0, launch_align_batch(h0->sc.batch_args.as<unsigned char>() + n1 * rec, (int)n2, 2, h0->stream->s));
  ph_end(h0, PH_ALIGN);
  NG_CUDA(h0, cudaStreamSynchronize(h0->stream->s));
  for (size_t i = 0; i < n; ++i) {
    results[i] = *hs[i]->res_pinned;
    hs[i]->lin_valid = true;
    if (results[i].lm_failed) fprintf(stderr, "lm not converged!!\n");  // lsq_registration_impl.hpp:106
  }
  return NGICP_OK;
}

int ngicp_transform_source(ngicp_t* h, const float* T16, float* out_xyz1, size_t n) {
  if (!h || !T16 || !out_xyz1) return NGICP_E_INVALID;
  if (!h->src || (size_t)h->src->n != n) return fail(h, NGICP_E_STATE, "transform: source size mismatch");
  if (n == 0) return NGICP_OK;
  DeviceGuard g(h->device);
  join_source(h);
  NG_CUDA(h, h->sc.queries.reserve(sizeof(float4) * n, h->stream));
  Mat16f T;
  memcpy(T.m, T16, sizeof T.m);
  transform_points_kernel<<<blocks_for((int)n), 256, 0, h->stream->s>>>(h->src->pts.as<float4>(), (int)n, T, h->sc.queries.as<float4>());
  NG_CUDA(h, cudaGetLastError());
  NG_CUDA(h, cudaMemcpyAsync(out_xyz1, h->sc.queries.p, sizeof(float4) * n, cudaMemcpyDefault, h->stream->s));
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  return NGICP_OK;
}

// pcl::Registration::getFitnessScore for n handles, each with its own source, target and T (fitness.cu): the handles'
// streams are joined into the first one's, which runs the two launches and lands the results in its mapped host buffer.
// The registration state (correspondences, lin_valid, results) is left alone.
int ngicp_fitness_batch(ngicp_t* const* hs, size_t n, const float* T16s, double max_range, double* scores, size_t* n_inliers) {
  if (!hs || n == 0 || !hs[0]) return NGICP_E_INVALID;
  ngicp_t* h0 = hs[0];
  if (!T16s || !scores) return fail(h0, NGICP_E_INVALID, "fitness: null argument");
  if (std::isnan(max_range)) return fail(h0, NGICP_E_INVALID, "fitness: max_range is NaN");
  if (n > 0x7fffffffu) return fail(h0, NGICP_E_INVALID, "fitness: too many handles");
  for (size_t i = 0; i < n; ++i) {
    ngicp_t* h = hs[i];
    if (!h) return fail(h0, NGICP_E_INVALID, "fitness: null handle");
    if (h->device != h0->device) return fail(h0, NGICP_E_INVALID, "fitness: handles live on different devices");
    for (size_t j = 0; j < i; ++j)
      if (hs[j] == h) return fail(h0, NGICP_E_INVALID, "fitness: the same handle appears twice");
    const std::string pre = n > 1 ? "fitness: pair " + std::to_string(i) + ": " : "fitness: ";
    // a sharded handle holds one slab of the submap: its nearest neighbours are not the submap's
    if (h->comm_on || h->slab_axis >= 0) return fail(h0, NGICP_E_UNSUPPORTED, (pre + "handle is in sharded mode").c_str());
    if (!h->src || !h->tgt) return fail(h0, NGICP_E_STATE, (pre + "source/target not set").c_str());
    if (h->tgt->n > 0 && !h->tgt->indexed) return fail(h0, NGICP_E_STATE, (pre + "target has no search index").c_str());
  }
  DeviceGuard g(h0->device);
  std::vector<FitnessPair> pairs(n);
  long long chunks = 0;
  for (size_t i = 0; i < n; ++i) {
    ngicp_t* h = hs[i];
    join_source(h);   // the source was uploaded on the source-side stream
    if (h != h0) {    // everything queued on this handle's stream (target index) precedes the launches
      if (!h->sc.copy_done) NG_CUDA(h0, cudaEventCreateWithFlags(&h->sc.copy_done, cudaEventDisableTiming));
      NG_CUDA(h0, cudaEventRecord(h->sc.copy_done, h->stream->s));
      NG_CUDA(h0, cudaStreamWaitEvent(h0->stream->s, h->sc.copy_done, 0));
    }
    FitnessPair& p = pairs[i];
    memset(&p, 0, sizeof p);
    const float* T = T16s + 16 * i;   // column-major: (r,c) at [c*4+r]
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 4; ++c) p.T[r * 4 + c] = T[c * 4 + r];
    p.src = h->src->pts.as<float4>();
    p.ns = h->src->n;
    p.chunk0 = (int)chunks;
    if (h->src->n > 0 && h->tgt->n > 0) {
      p.tgt = h->tgt->view();
      p.nchunks = (h->src->n + FITNESS_CHUNK - 1) / FITNESS_CHUNK;
      // two lanes per point against a target much larger than the scan (the registration kernels' rule)
      p.lpp = (long long)h->tgt->n >= 4ll * h->src->n ? 2 : 1;
    }
    chunks += p.nchunks;
  }
  if (chunks > 0x7fffffff) return fail(h0, NGICP_E_INVALID, "fitness: too many source points");
  if (h0->fit_cap < n) {
    if (h0->fit_pinned) cudaFreeHost(h0->fit_pinned);
    h0->fit_pinned = h0->fit_mapped = nullptr;
    h0->fit_cap = 0;
    NG_CUDA(h0, cudaHostAlloc((void**)&h0->fit_pinned, sizeof(FitnessResult) * n, cudaHostAllocMapped));
    NG_CUDA(h0, cudaHostGetDevicePointer((void**)&h0->fit_mapped, h0->fit_pinned, 0));
    h0->fit_cap = n;
  }
  Scratch& sc = h0->sc;
  NG_CUDA(h0, sc.fit_args.reserve(sizeof(FitnessPair) * n, h0->stream));
  NG_CUDA(h0, sc.fit_partials.reserve(sizeof(double2) * (size_t)(chunks > 0 ? chunks : 1), h0->stream));
  NG_CUDA(h0, cudaMemcpyAsync(sc.fit_args.p, pairs.data(), sizeof(FitnessPair) * n, cudaMemcpyHostToDevice, h0->stream->s));
  NG_CUDA(h0, launch_fitness(sc.fit_args.as<FitnessPair>(), (int)n, (int)chunks, max_range, sc.fit_partials.as<double2>(), h0->fit_mapped,
                             h0->stream->s));
  NG_CUDA(h0, cudaStreamSynchronize(h0->stream->s));
  for (size_t i = 0; i < n; ++i) {
    scores[i] = h0->fit_pinned[i].score;
    if (n_inliers) n_inliers[i] = (size_t)h0->fit_pinned[i].n;
  }
  return NGICP_OK;
}

int ngicp_fitness_score(ngicp_t* h, const float* T16, double max_range, double* score, size_t* n_inliers) {
  if (!h) return NGICP_E_INVALID;
  return ngicp_fitness_batch(&h, 1, T16, max_range, score, n_inliers);
}

int ngicp_voxel_filter(ngicp_t* h, const void* in, size_t n, size_t stride, float leaf, void* out, size_t cap, size_t* m) {
  if (!h || !m || (!in && n) || stride < 12 || (stride & 3) || !(leaf > 0.f) || n > 0x7fffff00u) return h ? fail(h, NGICP_E_INVALID, "bad voxel filter arguments") : NGICP_E_INVALID;
  DeviceGuard g(h->device);
  *m = 0;
  ph_begin(h, PH_VOXEL);
  size_t mm = 0;
  int overflow = 0;
  bool copied = false;
  NG_CUDA(h, voxel_filter_device(in, n, stride, leaf, h->sc, h->stream, &mm, &overflow, nullptr, false, nullptr, out, cap, &copied));
  int status = NGICP_OK;
  if (overflow) {
    // PCL: "Leaf size is too small for the input dataset. Integer indices would overflow." and output = input
    vox_passthrough_kernel<<<blocks_for((int)n), 256, 0, h->stream->s>>>(h->sc.queries.as<float4>(), (int)n, h->sc.vox_out.as<float>());
    NG_CUDA(h, cudaGetLastError());
    mm = n;
    status = NGICP_W_VOXEL_OVERFLOW;
  }
  if (mm > cap) return fail(h, NGICP_E_INVALID, "voxel filter: output capacity too small");
  if (mm && out && !copied) NG_CUDA(h, cudaMemcpyAsync(out, h->sc.vox_out.p, 32 * mm, cudaMemcpyDefault, h->stream->s));
  ph_end(h, PH_VOXEL);
  if (!copied) NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  *m = mm;
  return status;
}

int ngicp_transform_voxel_filter(ngicp_t* h, const void* in, size_t n, size_t stride, const float* T16, float leaf, void* out, size_t cap,
                                 size_t* m) {
  if (!h || !m || !T16 || (!in && n) || stride < 12 || (stride & 3) || n > 0x7fffff00u)
    return h ? fail(h, NGICP_E_INVALID, "bad transform+voxel arguments") : NGICP_E_INVALID;
  DeviceGuard g(h->device);
  *m = 0;
  ph_begin(h, PH_VOXEL);
  size_t mm = 0;
  int overflow = 0;
  bool copied = false;
  NG_CUDA(h, voxel_filter_device(in, n, stride, leaf, h->sc, h->stream, &mm, &overflow, nullptr, true, T16, out, cap, &copied));
  if (mm > cap) return fail(h, NGICP_E_INVALID, "transform+voxel: output capacity too small");
  if (mm && out && !copied) NG_CUDA(h, cudaMemcpyAsync(out, h->sc.vox_out.p, 32 * mm, cudaMemcpyDefault, h->stream->s));
  ph_end(h, PH_VOXEL);
  if (!copied) NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  *m = mm;
  return overflow ? NGICP_W_VOXEL_OVERFLOW : NGICP_OK;
}

int ngicp_preprocess(ngicp_t* h, const void* in, size_t n, size_t stride, const float* crop_min, const float* crop_max, float leaf,
                     void* out, size_t cap, size_t* m) {
  if (!h || !m || (!in && n) || stride < 12 || (stride & 3) || n > 0x7fffff00u || ((crop_min == nullptr) != (crop_max == nullptr)))
    return h ? fail(h, NGICP_E_INVALID, "bad preprocess arguments") : NGICP_E_INVALID;
  DeviceGuard g(h->device);
  *m = 0;
  float crop6[6];
  if (crop_min) for (int a = 0; a < 3; a++) { crop6[a] = crop_min[a]; crop6[3 + a] = crop_max[a]; }
  ph_begin(h, PH_VOXEL);
  size_t mm = 0;
  int overflow = 0;
  bool copied = false;
  NG_CUDA(h, voxel_filter_device(in, n, stride, leaf, h->sc, h->stream, &mm, &overflow, crop_min ? crop6 : nullptr, true, nullptr, out, cap, &copied));
  if (mm > cap) return fail(h, NGICP_E_INVALID, "preprocess: output capacity too small");
  if (mm && out && !copied) NG_CUDA(h, cudaMemcpyAsync(out, h->sc.vox_out.p, 32 * mm, cudaMemcpyDefault, h->stream->s));
  ph_end(h, PH_VOXEL);
  if (!copied) NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  *m = mm;
  return overflow ? NGICP_W_VOXEL_OVERFLOW : NGICP_OK;
}

int ngicp_preprocess_pointcloud2(ngicp_t* h, const void* data, const ngicp_pc2_layout* L, const float* crop_min, const float* crop_max,
                                 float leaf, void* out, size_t cap, size_t* m) {
  if (!h || !m || !L) return h ? fail(h, NGICP_E_INVALID, "bad PointCloud2 arguments") : NGICP_E_INVALID;
  *m = 0;
  const unsigned long long n64 = (unsigned long long)L->width * (unsigned long long)L->height;
  if ((!data && n64) || n64 > 0x7fffff00ull || ((crop_min == nullptr) != (crop_max == nullptr)))
    return fail(h, NGICP_E_INVALID, "bad PointCloud2 arguments");
  if (L->is_bigendian) return fail(h, NGICP_E_UNSUPPORTED, "PointCloud2: big-endian data (PCL reinterprets the bytes as they are; refuse instead)");
  if (L->offset_x < 0 || L->offset_y < 0 || L->offset_z < 0)
    return fail(h, NGICP_E_INVALID, "PointCloud2: no FLOAT32 x/y/z fields");      // pcl::fromROSMsg leaves them unset and warns
  const int offs[4] = {L->offset_x, L->offset_y, L->offset_z, L->offset_intensity};
  for (int f = 0; f < 4; f++)
    if (offs[f] >= 0 && (unsigned long long)offs[f] + 4ull > (unsigned long long)L->point_step)
      return fail(h, NGICP_E_INVALID, "PointCloud2: field beyond point_step");
  if (n64 && (unsigned long long)L->row_step < (unsigned long long)L->width * L->point_step && L->height > 1)
    return fail(h, NGICP_E_INVALID, "PointCloud2: row_step smaller than width * point_step");
  if (n64 == 0) return NGICP_OK;
  DeviceGuard g(h->device);
  RecordLayout lay;
  lay.width = (int)L->width;
  lay.point_step = L->point_step;
  lay.row_step = L->row_step;
  lay.aligned = ((L->point_step | L->row_step) & 3u) == 0;
  for (int f = 0; f < 4; f++) { lay.off[f] = offs[f] >= 0 ? offs[f] : -1; if (offs[f] >= 0 && (offs[f] & 3)) lay.aligned = 0; }
  float crop6[6];
  if (crop_min) for (int a = 0; a < 3; a++) { crop6[a] = crop_min[a]; crop6[3 + a] = crop_max[a]; }
  ph_begin(h, PH_VOXEL);
  size_t mm = 0;
  int overflow = 0;
  bool copied = false;
  NG_CUDA(h, voxel_filter_records(data, (size_t)n64, lay, leaf, h->sc, h->stream, &mm, &overflow, crop_min ? crop6 : nullptr, true, nullptr, out, cap, &copied));
  if (mm > cap) return fail(h, NGICP_E_INVALID, "preprocess: output capacity too small");
  if (mm && out && !copied) NG_CUDA(h, cudaMemcpyAsync(out, h->sc.vox_out.p, 32 * mm, cudaMemcpyDefault, h->stream->s));
  ph_end(h, PH_VOXEL);
  if (!copied) NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  *m = mm;
  return overflow ? NGICP_W_VOXEL_OVERFLOW : NGICP_OK;
}

int ngicp_voxel_assignment(ngicp_t* h, int* slot_of_point, size_t n) {
  if (!h || !slot_of_point) return NGICP_E_INVALID;
  if (!h->sc.vox_slot.p || h->sc.vox_slot.bytes < sizeof(int) * n) return fail(h, NGICP_E_STATE, "no voxel filter result");
  DeviceGuard g(h->device);
  NG_CUDA(h, cudaMemcpyAsync(slot_of_point, h->sc.vox_slot.p, sizeof(int) * n, cudaMemcpyDefault, h->stream->s));
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  return NGICP_OK;
}

int ngicp_knn(ngicp_t* h, int which, const float* queries, size_t nq, size_t q_stride, int k, int* idx, float* d2) {
  if (!h || (!queries && nq) || !idx || !d2 || q_stride < 12 || (q_stride & 3)) return NGICP_E_INVALID;
  if (k < 1 || k > KNN_WIDE_MAX_K) return fail(h, NGICP_E_UNSUPPORTED, "k must be in [1,128]");
  DeviceGuard g(h->device);
  CloudPtr& c = which == NGICP_SOURCE ? h->src : h->tgt;
  if (!c) return fail(h, NGICP_E_STATE, "knn: cloud not set");
  if (!c->indexed) return fail(h, NGICP_E_STATE, "knn: no search index (nanoflann throws here, nanoflann_impl.hpp:1235-1237)");
  if (nq == 0) return NGICP_OK;
  join_source(h);
  DevCloud qc;
  NG_CUDA(h, upload_cloud(qc, queries, nq, q_stride, h->sc, h->stream));
  NG_CUDA(h, h->sc.knn_idx.reserve(sizeof(int) * nq * k, h->stream));
  NG_CUDA(h, h->sc.knn_d2.reserve(sizeof(float) * nq * k, h->stream));
  NG_CUDA(h, launch_knn_queries(*c, qc.pts.as<float4>(), (int)nq, k, h->sc.knn_idx.as<int>(), h->sc.knn_d2.as<float>(), h->stream->s));
  NG_CUDA(h, cudaMemcpyAsync(idx, h->sc.knn_idx.p, sizeof(int) * nq * k, cudaMemcpyDefault, h->stream->s));
  NG_CUDA(h, cudaMemcpyAsync(d2, h->sc.knn_d2.p, sizeof(float) * nq * k, cudaMemcpyDefault, h->stream->s));
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  return NGICP_OK;
}

int ngicp_linearize_partial(ngicp_t* h, const double* T16, double* out43) {
  if (!h || !T16 || !out43) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  AlignBuffers ab;
  int rc = prepare_align(h, false, ab);
  if (rc) return rc;
  NG_CUDA(h, launch_linearize(ab, T16, h->prm.max_correspondence_distance, h->stream->s));
  rc = fetch_reduced(h, NRED);
  if (rc) return rc;
  double tmp[43];
  unpack_H(h->red_pinned, tmp);
  for (int i = 0; i < 6; i++) tmp[36 + i] = h->red_pinned[21 + i];
  tmp[42] = h->red_pinned[27];
  NG_CUDA(h, cudaMemcpy(out43, tmp, sizeof tmp, cudaMemcpyDefault));
  h->lin_valid = true;
  return NGICP_OK;
}

int ngicp_nn1_packed(ngicp_t* h, const double* T16, unsigned rank, unsigned long long* packed_out) {
  if (!h || !T16 || !packed_out) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  AlignBuffers ab;
  int rc = prepare_align(h, false, ab);
  if (rc) return rc;
  const size_t ns = (size_t)ab.ns;
  NG_CUDA(h, h->sc.nn1_packed.reserve(sizeof(unsigned long long) * (ns ? ns : 1), h->stream));
  NG_CUDA(h, launch_nn1_packed(ab, T16, h->prm.max_correspondence_distance, rank, h->sc.nn1_packed.as<unsigned long long>(), h->stream->s));
  NG_CUDA(h, cudaMemcpyAsync(packed_out, h->sc.nn1_packed.p, sizeof(unsigned long long) * ns, cudaMemcpyDefault, h->stream->s));
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  h->lin_valid = false;
  return NGICP_OK;
}

int ngicp_linearize_won(ngicp_t* h, const double* T16, unsigned rank, const unsigned long long* packed_min, double* out43) {
  if (!h || !T16 || !packed_min || !out43) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  AlignBuffers ab;
  int rc = prepare_align(h, false, ab);
  if (rc) return rc;
  const size_t ns = (size_t)ab.ns;
  NG_CUDA(h, h->sc.nn1_won.reserve(sizeof(unsigned long long) * (ns ? ns : 1), h->stream));
  NG_CUDA(h, cudaMemcpyAsync(h->sc.nn1_won.p, packed_min, sizeof(unsigned long long) * ns, cudaMemcpyDefault, h->stream->s));
  NG_CUDA(h, launch_linearize_won(ab, T16, h->prm.max_correspondence_distance, rank, h->sc.nn1_won.as<unsigned long long>(), h->stream->s));
  rc = fetch_reduced(h, NRED);
  if (rc) return rc;
  double tmp[43];
  unpack_H(h->red_pinned, tmp);
  for (int i = 0; i < 6; i++) tmp[36 + i] = h->red_pinned[21 + i];
  tmp[42] = h->red_pinned[27];
  NG_CUDA(h, cudaMemcpy(out43, tmp, sizeof tmp, cudaMemcpyDefault));
  h->lin_valid = true;
  return NGICP_OK;
}

int ngicp_linearize(ngicp_t* h, const double* T16, double* H36, double* b6, double* err, int* corr, float* sqd, double* mahal) {
  if (!h || !T16) return NGICP_E_INVALID;
  double tmp[43];
  int rc = ngicp_linearize_partial(h, T16, tmp);
  if (rc) return rc;
  DeviceGuard g(h->device);
  if (H36) memcpy(H36, tmp, sizeof(double) * 36);
  if (b6) memcpy(b6, tmp + 36, sizeof(double) * 6);
  if (err) *err = tmp[42];
  const size_t ns = (size_t)h->src->n;
  if (corr) NG_CUDA(h, cudaMemcpyAsync(corr, h->sc.corr.p, sizeof(int) * ns, cudaMemcpyDefault, h->stream->s));
  if (sqd) NG_CUDA(h, cudaMemcpyAsync(sqd, h->sc.sqd.p, sizeof(float) * ns, cudaMemcpyDefault, h->stream->s));
  if (mahal) {
    AlignBuffers ab;
    rc = prepare_align(h, false, ab);
    if (rc) return rc;
    NG_CUDA(h, h->sc.cov_stage.reserve(sizeof(double) * 16 * ns, h->stream));
    NG_CUDA(h, launch_export_mahal(ab, h->sc.cov_stage.as<double>(), h->stream->s));
    NG_CUDA(h, cudaMemcpyAsync(mahal, h->sc.cov_stage.p, sizeof(double) * 16 * ns, cudaMemcpyDefault, h->stream->s));
  }
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  return NGICP_OK;
}

int ngicp_correspondences(ngicp_t* h, int* corr, float* sqd, double* mahal16) {
  if (!h) return NGICP_E_INVALID;
  if (!h->lin_valid || !h->src) return fail(h, NGICP_E_STATE, "correspondences: no linearisation on the current clouds");
  DeviceGuard g(h->device);
  const size_t ns = (size_t)h->src->n;
  if (corr) NG_CUDA(h, cudaMemcpyAsync(corr, h->sc.corr.p, sizeof(int) * ns, cudaMemcpyDefault, h->stream->s));
  if (sqd) NG_CUDA(h, cudaMemcpyAsync(sqd, h->sc.sqd.p, sizeof(float) * ns, cudaMemcpyDefault, h->stream->s));
  if (mahal16) {
    AlignBuffers ab;
    memset(&ab, 0, sizeof ab);
    ab.ns = (int)ns; ab.mahal = h->sc.mahal.as<double>(); ab.corr = h->sc.corr.as<int>();
    NG_CUDA(h, h->sc.cov_stage.reserve(sizeof(double) * 16 * ns, h->stream));
    NG_CUDA(h, launch_export_mahal(ab, h->sc.cov_stage.as<double>(), h->stream->s));
    NG_CUDA(h, cudaMemcpyAsync(mahal16, h->sc.cov_stage.p, sizeof(double) * 16 * ns, cudaMemcpyDefault, h->stream->s));
  }
  NG_CUDA(h, cudaStreamSynchronize(h->stream->s));
  return NGICP_OK;
}

int ngicp_compute_error_partial(ngicp_t* h, const double* T16, double* out1) {
  if (!h || !T16 || !out1) return NGICP_E_INVALID;
  if (!h->lin_valid) return fail(h, NGICP_E_STATE, "compute_error needs a preceding linearize on the same clouds");
  DeviceGuard g(h->device);
  AlignBuffers ab;
  int rc = prepare_align(h, false, ab);
  if (rc) return rc;
  NG_CUDA(h, launch_compute_error(ab, T16, h->stream->s));
  rc = fetch_reduced(h, 1);
  if (rc) return rc;
  NG_CUDA(h, cudaMemcpy(out1, h->red_pinned, sizeof(double), cudaMemcpyDefault));
  return NGICP_OK;
}
int ngicp_compute_error(ngicp_t* h, const double* T16, double* err) { return ngicp_compute_error_partial(h, T16, err); }

int ngicp_set_owner_slab(ngicp_t* h, int axis, float lo, float hi) {
  if (!h || axis < -1 || axis > 2) return NGICP_E_INVALID;
  h->slab_axis = axis; h->slab_lo = lo; h->slab_hi = hi;
  h->lin_valid = false;
  return NGICP_OK;
}

// host-only scalar side of one LM / GN trial, the same code the fused kernel runs on the device
int ngicp_lm_trial(const double* H36, const double* b6, double lambda, const double* x0_16, double* d6, double* delta16, double* xi16) {
  if (!H36 || !b6 || !x0_16 || !d6 || !delta16 || !xi16) return NGICP_E_INVALID;
  double A[36], nb[6];
  memcpy(A, H36, sizeof A);
  for (int i = 0; i < 6; i++) { A[i * 7] += lambda; nb[i] = -b6[i]; }
  lm_solve(A, nb, d6);
  Iso3 x0, delta, xi;
  iso_from_colmajor16(x0_16, x0);
  delta_from_step(d6, delta);
  iso_mul(delta, x0, xi);
  iso_to_colmajor16(delta, delta16);
  iso_to_colmajor16(xi, xi16);
  return NGICP_OK;
}
int ngicp_lm_is_converged(const double* delta16, double rot_eps, double trans_eps) {
  if (!delta16) return 0;
  Iso3 d;
  iso_from_colmajor16(delta16, d);
  return lm_is_converged(d, rot_eps, trans_eps) ? 1 : 0;
}

// ---- N4: OdomNode::integrateIMU (odom.cc:859-919), host arithmetic -------------------------------------------------------
int ngicp_imu_prior(const double* stamps, const double* av, size_t n, double prev_stamp, double curr_stamp, float* out_T16) {
  if (!out_T16 || ((!stamps || !av) && n)) return NGICP_E_INVALID;
  struct Sample { double t, x, y, z; };
  std::vector<Sample> frame;
  for (size_t i = 0; i < n; ++i)
    if (curr_stamp - stamps[i] >= 0. && prev_stamp - stamps[i] <= 0.) frame.push_back(Sample{stamps[i], av[3 * i], av[3 * i + 1], av[3 * i + 2]});
  std::sort(frame.begin(), frame.end(), [](const Sample& a, const Sample& b) { return a.t < b.t; });
  float w = 1.f, x = 0.f, y = 0.f, z = 0.f;
  double prev_t = 0.;
  for (const Sample& m : frame) {
    if (prev_t == 0.) { prev_t = m.t; continue; }   // the first sample (and any sample stamped exactly 0) only sets the clock
    const double dt = m.t - prev_t;
    prev_t = m.t;
    const float qw = w, qx = x, qy = y, qz = z;
    w -= 0.5 * (qx * m.x + qy * m.y + qz * m.z) * dt;
    x += 0.5 * (qw * m.x - qz * m.y + qy * m.z) * dt;
    y += 0.5 * (qz * m.x + qw * m.y - qx * m.z) * dt;
    z += 0.5 * (qx * m.y - qy * m.x + qw * m.z) * dt;
  }
  const double norm = sqrt((double)(w * w + x * x + y * y + z * z));   // float sum of float products, sqrt in double
  w /= norm; x /= norm; y /= norm; z /= norm;
  // Eigen::Quaternionf::toRotationMatrix
  const float tx = 2.f * x, ty = 2.f * y, tz = 2.f * z;
  const float twx = tx * w, twy = ty * w, twz = tz * w;
  const float txx = tx * x, txy = ty * x, txz = tz * x;
  const float tyy = ty * y, tyz = tz * y, tzz = tz * z;
  float R[3][3] = {{1.f - (tyy + tzz), txy - twz, txz + twy}, {txy + twz, 1.f - (txx + tzz), tyz - twx}, {txz - twy, tyz + twx, 1.f - (txx + tyy)}};
  for (int i = 0; i < 16; ++i) out_T16[i] = 0.f;
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) out_T16[c * 4 + r] = R[r][c];
  out_T16[15] = 1.f;
  return NGICP_OK;
}

// ---- sharded-submap exchange (align.cu: peer_exchange_sum) ----------------------------------------------------
static int comm_alloc(ngicp_t* h) {
  if (h->comm_buf) return NGICP_OK;
  NG_CUDA(h, cudaMalloc(&h->comm_buf, PEER_BUF_BYTES));   // plain cudaMalloc: IPC cannot export pool memory
  NG_CUDA(h, cudaMemset(h->comm_buf, 0, PEER_BUF_BYTES));
  return NGICP_OK;
}
static void comm_fill(ngicp_t* h, int rank, int world) {
  PeerComm& pc = h->comm;
  memset(&pc, 0, sizeof pc);
  pc.world = world; pc.rank = rank;
  for (int p = 0; p < world; ++p) {
    unsigned char* base = static_cast<unsigned char*>(h->comm_peer[p]);
    pc.data[p] = reinterpret_cast<double*>(base);
    pc.flag[p] = reinterpret_cast<unsigned long long*>(base + PEER_DATA_BYTES);
  }
  unsigned char* own = static_cast<unsigned char*>(h->comm_buf);
  pc.seq = reinterpret_cast<unsigned long long*>(own + PEER_DATA_BYTES + PEER_FLAG_BYTES);
  pc.error = reinterpret_cast<int*>(own + PEER_DATA_BYTES + PEER_FLAG_BYTES + 8);
  const char* e = getenv("NGICP_COMM_TIMEOUT_MS");
  const double ms = e ? atof(e) : 2000.0;
  pc.timeout_ns = (unsigned long long)((ms > 0.0 ? ms : 2000.0) * 1e6);
  h->comm_on = world > 1;
}

int ngicp_comm_export(ngicp_t* h, void* handle64) {
  if (!h || !handle64) return NGICP_E_INVALID;
  static_assert(sizeof(cudaIpcMemHandle_t) <= NGICP_COMM_HANDLE_BYTES, "IPC handle does not fit");
  DeviceGuard g(h->device);
  int rc = comm_alloc(h);
  if (rc) return rc;
  NG_CUDA(h, cudaMemset(h->comm_buf, 0, PEER_BUF_BYTES));
  cudaIpcMemHandle_t ipc;
  NG_CUDA(h, cudaIpcGetMemHandle(&ipc, h->comm_buf));
  memset(handle64, 0, NGICP_COMM_HANDLE_BYTES);
  memcpy(handle64, &ipc, sizeof ipc);
  return NGICP_OK;
}

int ngicp_comm_close(ngicp_t* h) {
  if (!h) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  if (h->stream && h->stream_src) sync_both(h);
  for (int p = 0; p < NGICP_MAX_RANKS; ++p) {
    if (h->comm_peer[p] && h->comm_peer_ipc[p]) cudaIpcCloseMemHandle(h->comm_peer[p]);
    h->comm_peer[p] = nullptr;
    h->comm_peer_ipc[p] = false;
  }
  h->comm_on = false;
  return NGICP_OK;
}

int ngicp_comm_reset(ngicp_t* h) {
  if (!h) return NGICP_E_INVALID;
  if (!h->comm_buf) return fail(h, NGICP_E_STATE, "comm_reset: no exchange buffer (ngicp_comm_export / connect first)");
  DeviceGuard g(h->device);
  if (h->stream && h->stream_src) sync_both(h);
  NG_CUDA(h, cudaMemset(h->comm_buf, 0, PEER_BUF_BYTES));      // slots, sequence flags, own sequence number, sticky error
  return NGICP_OK;
}

int ngicp_comm_connect(ngicp_t* h, int rank, int world, const void* handles) {
  if (!h || !handles || world < 1 || world > NGICP_MAX_RANKS || rank < 0 || rank >= world) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  int rc = comm_alloc(h);
  if (rc) return rc;
  ngicp_comm_close(h);
  for (int p = 0; p < world; ++p) {
    if (p == rank) { h->comm_peer[p] = h->comm_buf; continue; }
    cudaIpcMemHandle_t ipc;
    memcpy(&ipc, static_cast<const unsigned char*>(handles) + (size_t)p * NGICP_COMM_HANDLE_BYTES, sizeof ipc);
    NG_CUDA(h, cudaIpcOpenMemHandle(&h->comm_peer[p], ipc, cudaIpcMemLazyEnablePeerAccess));
    h->comm_peer_ipc[p] = true;
  }
  comm_fill(h, rank, world);
  return NGICP_OK;
}

int ngicp_comm_connect_local(ngicp_t* h, int rank, int world, ngicp_t* const* peers) {
  if (!h || !peers || world < 1 || world > NGICP_MAX_RANKS || rank < 0 || rank >= world) return NGICP_E_INVALID;
  DeviceGuard g(h->device);
  int rc = comm_alloc(h);
  if (rc) return rc;
  ngicp_comm_close(h);
  for (int p = 0; p < world; ++p) {
    ngicp_t* o = peers[p];
    if (!o) return fail(h, NGICP_E_INVALID, "comm_connect_local: null peer");
    if (p == rank) { h->comm_peer[p] = h->comm_buf; continue; }
    { DeviceGuard go(o->device); rc = comm_alloc(o); if (rc) return fail(h, NGICP_E_CUDA, "comm_connect_local: peer buffer"); }
    if (o->device != h->device) {
      int can = 0;
      NG_CUDA(h, cudaDeviceCanAccessPeer(&can, h->device, o->device));
      if (!can) return fail(h, NGICP_E_UNSUPPORTED, "comm_connect_local: no peer access between the devices");
      cudaError_t e = cudaDeviceEnablePeerAccess(o->device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(h, NGICP_E_CUDA, "cudaDeviceEnablePeerAccess", e);
      cudaGetLastError();
    }
    h->comm_peer[p] = o->comm_buf;
  }
  comm_fill(h, rank, world);
  return NGICP_OK;
}

// ---- N1: device-resident keyframes / submap assembly -------------------------------------------------------------
int ngicp_kfstore_create(int device, ngicp_kfstore_t** out) {
  if (!out) return NGICP_E_INVALID;
  ngicp_kfstore* s = new (std::nothrow) ngicp_kfstore();
  if (!s) return NGICP_E_INVALID;
  s->device = device;
  *out = s;
  return NGICP_OK;
}

void ngicp_kfstore_destroy(ngicp_kfstore_t* s) {
  if (!s) return;
  DeviceGuard g(s->device);
  for (auto& k : s->kf) if (k.ready) { cudaEventSynchronize(k.ready); cudaEventDestroy(k.ready); }
  delete s;
}

size_t ngicp_kfstore_size(const ngicp_kfstore_t* s) { return s ? s->kf.size() : 0; }

size_t ngicp_kfstore_points(const ngicp_kfstore_t* s, size_t index) {
  return (s && index < s->kf.size()) ? (size_t)s->kf[index].n : 0;
}

int ngicp_kfstore_push(ngicp_kfstore_t* s, ngicp_t* from, size_t* index_out) {
  if (!s || !from) return NGICP_E_INVALID;
  if (from->device != s->device) return fail(from, NGICP_E_INVALID, "keyframe store lives on another device");
  if (!from->src || !from->src_cov || from->src_cov->n != from->src->n)
    return fail(from, NGICP_E_STATE, "keyframe push: source cloud and its covariances must be set (setInputSource + calculateSourceCovariances)");
  DeviceGuard g(s->device);
  join_source(from);
  ngicp_kfstore::Keyframe k;
  k.n = from->src->n;
  k.pts.reset(new (std::nothrow) DevBuf());
  if (!k.pts) return fail(from, NGICP_E_INVALID, "out of host memory");
  NG_CUDA(from, k.pts->alloc(sizeof(float4) * (size_t)(k.n ? k.n : 1), from->stream));
  if (k.n) NG_CUDA(from, cudaMemcpyAsync(k.pts->p, from->src->pts.p, sizeof(float4) * (size_t)k.n, cudaMemcpyDeviceToDevice, from->stream->s));
  k.covs = from->src_cov;
  NG_CUDA(from, cudaEventCreateWithFlags(&k.ready, cudaEventDisableTiming));
  NG_CUDA(from, cudaEventRecord(k.ready, from->stream->s));
  s->kf.push_back(k);
  if (index_out) *index_out = s->kf.size() - 1;
  return NGICP_OK;
}

int ngicp_kfstore_set_target(ngicp_kfstore_t* s, ngicp_t* to, const int* indices, size_t n_indices) {
  if (!s || !to || (!indices && n_indices)) return NGICP_E_INVALID;
  if (to->device != s->device) return fail(to, NGICP_E_INVALID, "keyframe store lives on another device");
  size_t total = 0;
  for (size_t i = 0; i < n_indices; ++i) {
    if (indices[i] < 0 || (size_t)indices[i] >= s->kf.size()) return fail(to, NGICP_E_INVALID, "keyframe index out of range");
    total += (size_t)s->kf[indices[i]].n;
  }
  if (total == 0) return fail(to, NGICP_E_STATE, "submap without points");
  if (total > 0x7fffff00u) return fail(to, NGICP_E_INVALID, "submap too large");
  DeviceGuard g(to->device);
  cudaStream_t st = to->stream->s;
  CloudPtr c(new (std::nothrow) DevCloud());
  CovsPtr cv(new (std::nothrow) DevCovs());
  if (!c || !cv) return fail(to, NGICP_E_INVALID, "out of host memory");
  ph_begin(to, PH_SET_TGT);
  // submap_cloud += *keyframes[k].second; submap_normals.insert(...) (odom.cc:1315-1328), device to device
  NG_CUDA(to, to->sc.staging.reserve(sizeof(float4) * total + 16, to->stream));
  cv->n = (int)total;
  NG_CUDA(to, cv->c.alloc(sizeof(double) * 6 * total, to->stream));
  size_t off = 0;
  for (size_t i = 0; i < n_indices; ++i) {
    const ngicp_kfstore::Keyframe& k = s->kf[indices[i]];
    const size_t n = (size_t)k.n;
    if (n == 0) continue;
    NG_CUDA(to, cudaStreamWaitEvent(st, k.ready, 0));
    NG_CUDA(to, cudaMemcpyAsync(to->sc.staging.as<float4>() + off, k.pts->p, sizeof(float4) * n, cudaMemcpyDeviceToDevice, st));
    NG_CUDA(to, cudaMemcpyAsync(cv->c.as<double>() + 6 * off, k.covs->c.p, sizeof(double) * 6 * n, cudaMemcpyDeviceToDevice, st));
    off += n;
  }
  // gicp.setInputTarget(submap_cloud) (:830): snapshot + bounding box + search index
  bool fused = false;
  NG_CUDA(to, upload_and_index_fused(*c, to->sc.staging.p, total, sizeof(float4), to->prm.grid_cell_size, to->prm.grid_table_cells, to->sc, to->stream, to->device, &fused));
  if (!fused) {
    NG_CUDA(to, upload_cloud(*c, to->sc.staging.p, total, sizeof(float4), to->sc, to->stream));
    NG_CUDA(to, build_index(*c, to->prm.grid_cell_size, to->prm.grid_table_cells, to->sc, to->stream, to->device));
  }
  ph_end(to, PH_SET_TGT);
  drop_cloud(to, NGICP_TARGET);
  drop_covs(to, NGICP_TARGET);
  to->tgt = c;
  to->tgt_cov = cv;            // gicp.setTargetCovariances(submap_normals) (:833)
  to->lin_valid = false;
  return NGICP_OK;
}

}  // extern "C"


