/* nanogicp_c.h — C ABI of libnanogicp_b200.so: the NanoGICP registration hot path of
 * Direct LiDAR Odometry re-built as hand-written sm_100a CUDA kernels.
 *
 * This is the drop-in boundary.  The reference has no FFI: OdomNode uses the C++ class
 * nano_gicp::NanoGICP<PointXYZI,PointXYZI> directly (reference include/dlo/odom.h:119-120).
 * include/nano_gicp/nano_gicp.hpp in this repo re-creates that class surface and forwards every
 * call to the functions below; each entry point cites the reference member it replaces
 * (paths relative to the reference tree).
 *
 * Conventions
 *   - plain pointers and sizes only; no CUDA/torch types.  `pts` arguments point at n records of
 *     `stride_bytes` each whose first three floats are x,y,z (stride 32 for pcl::PointXYZI, 16 for
 *     float4, 12 for packed xyz).  They may be HOST or DEVICE pointers (unified addressing decides);
 *     the call snapshots them into HBM, the caller keeps ownership.  HOST buffers (pageable or pinned) may be
 *     freed or overwritten as soon as the call returns; DEVICE buffers are read in stream order on the handle's
 *     stream, so the caller must not overwrite them before ngicp_sync() / a later synchronising call (align).
 *   - 4x4 matrices are column-major like Eigen (element (r,c) at [c*4+r]); covariances are
 *     Eigen::Matrix4d records (16 doubles, 128 B) of which only the symmetric upper-left 3x3 is used.
 *   - every function returns an int status: 0 ok, <0 error (ngicp_last_error() has the text),
 *     >0 warning.  Nothing throws or aborts across the boundary.  "LM did not converge" is not an
 *     error: it is reported in ngicp_result like the reference reports it via hasConverged().
 *   - a handle owns one CUDA stream and is not thread-safe; different handles may be used from
 *     different threads / devices concurrently.
 *   - there is NO CPU fallback: every compute entry point launches CUDA kernels on the handle's
 *     device and fails with NGICP_E_CUDA if that is impossible.
 */
#ifndef NANOGICP_C_H
#define NANOGICP_C_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ngicp_handle ngicp_t;

enum {
  NGICP_OK = 0,
  NGICP_E_INVALID = -1,          /* bad argument */
  NGICP_E_STATE = -2,            /* missing source/target/index (PCL prints an error and returns) */
  NGICP_E_TOO_FEW_POINTS = -3,   /* cloud has fewer than k points (UB in the reference, nano_gicp_impl.hpp:315-318) */
  NGICP_E_COV_SIZE = -4,         /* covariance count != point count (assert at nano_gicp_impl.hpp:175-176) */
  NGICP_E_CUDA = -5,
  NGICP_E_UNSUPPORTED = -6,
  NGICP_E_COMM = -7,             /* sharded align: a peer rank did not reach the exchange in time */
  NGICP_W_VOXEL_OVERFLOW = 1     /* voxel index would overflow int32: input passed through, like PCL */
};

/* RegularizationMethod, include/nano_gicp/gicp/gicp_settings.hpp:47 */
enum { NGICP_REG_NONE = 0, NGICP_REG_MIN_EIG = 1, NGICP_REG_NORMALIZED_MIN_EIG = 2, NGICP_REG_PLANE = 3, NGICP_REG_FROBENIUS = 4 };
/* LSQ_OPTIMIZER_TYPE, include/nano_gicp/lsq_registration.hpp:54 */
enum { NGICP_OPT_GAUSS_NEWTON = 0, NGICP_OPT_LEVENBERG_MARQUARDT = 1 };
enum { NGICP_SOURCE = 0, NGICP_TARGET = 1 };
/* how ngicp_align drives the LM loop */
/* which exact kNN kernel family calculate*Covariances runs (both give the same neighbour sets and, since the
 * covariance kernel accumulates in ascending (distance, index) order, the same covariance bits) */
enum {
  NGICP_KNN_AUTO = 0,   /* tiles for clouds of knn_tile_min_points or more, one warp per query below */
  NGICP_KNN_WARP = 1,   /* one warp per query: growing-cube search with a warp-distributed sorted top-k list */
  NGICP_KNN_TILE = 2    /* cell-major tiles staged in shared memory, one thread per query, threshold selection */
};
enum {
  NGICP_ALIGN_FUSED = 0,   /* one persistent cooperative kernel runs the whole LM loop, state stays in HBM/registers */
  NGICP_ALIGN_STEPPED = 1  /* one launch per linearize/compute_error, LM decisions on the host (debug + sharded mode) */
};

typedef struct {
  /* reference parameters and their defaults */
  int k_correspondences;               /* setCorrespondenceRandomness; nano_gicp_impl.hpp:57 (20); 1..128 (above 32: warp search with a
                                          shared-memory result set, untuned); larger values: NGICP_E_UNSUPPORTED */
  double max_correspondence_distance;  /* setMaxCorrespondenceDistance; nano_gicp_impl.hpp:59 (FLT_MAX) */
  int max_iterations;                  /* setMaximumIterations; lsq_registration_impl.hpp:52 (64) */
  double transformation_epsilon;       /* setTransformationEpsilon; lsq_registration_impl.hpp:54 (5e-4) */
  double rotation_epsilon;             /* setRotationEpsilon; lsq_registration_impl.hpp:53 (2e-3) */
  int optimizer;                       /* lsq_registration_impl.hpp:56 (LM) */
  int lm_max_iterations;               /* lsq_registration_impl.hpp:58 (10) */
  double lm_init_lambda_factor;        /* setInitialLambdaFactor; lsq_registration_impl.hpp:59 (1e-9) */
  int regularization_method;           /* setRegularizationMethod; nano_gicp_impl.hpp:61 (PLANE) */
  /* B200-side knobs without a reference counterpart */
  float grid_cell_size;                /* uniform-grid cell edge in metres; 0 = choose from the data */
  int grid_table_cells;                /* capacity of the dense cell table (cells); the cell edge grows to fit */
  int align_mode;                      /* NGICP_ALIGN_FUSED / NGICP_ALIGN_STEPPED */
  int knn_path;                        /* NGICP_KNN_AUTO / _WARP / _TILE */
  int knn_tile_min_points;             /* NGICP_KNN_AUTO switches to the tile kernels at this cloud size (131072) */
  int voxel_path;                      /* voxel filter / preprocess: 0 = one persistent cooperative launch when the cloud fits
                                          (4096 points per SM), 1 = always the multi-kernel pipeline, 2 = as 0 */
  int index_path;                      /* setInputSource / setInputTarget: 0 = snapshot + search index in one persistent cooperative
                                          launch (lowest latency for one stream), 1 = the multi-kernel pipeline, 2 = as 0,
                                          3 = one thread-block cluster per cloud (ordinary launch: best when many handles share
                                          the GPU with small voxelised clouds; clouds above 32k points take 0) */
} ngicp_params;

/* what pcl::Registration / LsqRegistration expose after align() */
typedef struct {
  float final_transformation[16];  /* getFinalTransformation(): double state cast to float, lsq_registration_impl.hpp:113 */
  double final_x[16];              /* the double state itself */
  double final_hessian[36];        /* getFinalHessian(), lsq_registration_impl.hpp:84-86 */
  double lm_lambda;
  double last_error;               /* y0 of the last linearisation */
  int nr_iterations;               /* index of the last outer iteration, lsq_registration_impl.hpp:102 */
  int converged;                   /* hasConverged() */
  int n_linearize;                 /* calls of linearize() */
  int n_compute_error;             /* calls of compute_error() (LM trials) */
  int lm_failed;                   /* 1 when "lm not converged!!" (lsq_registration_impl.hpp:105-108) */
  int reserved;
} ngicp_result;

/* device time of the phases of the last calls on this handle, milliseconds (CUDA events) */
typedef struct {
  float set_source_ms, set_target_ms, source_covs_ms, target_covs_ms, align_ms, voxel_ms;
  float reserved[10];
} ngicp_timings;

/* ---- lifetime ------------------------------------------------------------------------------- */
/* NanoGICP::NanoGICP(), nano_gicp_impl.hpp:49-64 */
int ngicp_create(int device, ngicp_t** out);
void ngicp_destroy(ngicp_t* h);
const char* ngicp_last_error(const ngicp_t* h);
/* run this handle's work on an existing cudaStream_t (e.g. the caller's current stream); NULL = own stream */
int ngicp_set_stream(ngicp_t* h, void* cuda_stream);
void* ngicp_get_stream(const ngicp_t* h);
int ngicp_sync(ngicp_t* h);
int ngicp_get_timings(ngicp_t* h, ngicp_timings* out);

/* ---- parameters: the setters at odom.cc:100-114 and nano_gicp.hpp:82-84 ----------------------- */
void ngicp_params_default(ngicp_params* p);
int ngicp_set_params(ngicp_t* h, const ngicp_params* p);
int ngicp_get_params(const ngicp_t* h, ngicp_params* p);

/* ---- clouds ----------------------------------------------------------------------------------- */
/* NanoGICP::setInputSource, nano_gicp_impl.hpp:120-129: snapshot + build the search index, drop source covariances */
int ngicp_set_source(ngicp_t* h, const void* pts, size_t n, size_t stride_bytes);
/* NanoGICP::setInputTarget, nano_gicp_impl.hpp:131-139 */
int ngicp_set_target(ngicp_t* h, const void* pts, size_t n, size_t stride_bytes);
/* NanoGICP::registerInputSource, nano_gicp_impl.hpp:112-118: snapshot only, no index, covariances kept */
int ngicp_register_source(ngicp_t* h, const void* pts, size_t n, size_t stride_bytes);
/* `gicp.source_kdtree_ = gicp_s2s.source_kdtree_` (odom.cc:525): dst's source cloud+index alias src's, no copy */
int ngicp_share_source(ngicp_t* dst, const ngicp_t* src);
/* `gicp.source_covs_ = gicp_s2s.source_covs_` (odom.cc:815) without leaving HBM */
int ngicp_share_source_covs(ngicp_t* dst, const ngicp_t* src);
/* NanoGICP::swapSourceAndTarget, nano_gicp_impl.hpp:90-98: O(1) role swap of device buffers */
int ngicp_swap(ngicp_t* h);
/* NanoGICP::clearSource / clearTarget, nano_gicp_impl.hpp:100-110 */
int ngicp_clear_source(ngicp_t* h);
int ngicp_clear_target(ngicp_t* h);
size_t ngicp_cloud_size(const ngicp_t* h, int which);

/* ---- covariances ------------------------------------------------------------------------------ */
/* NanoGICP::calculateSourceCovariances / calculateTargetCovariances, nano_gicp_impl.hpp:151-159,298-357 */
int ngicp_calc_source_covs(ngicp_t* h);
int ngicp_calc_target_covs(ngicp_t* h);
/* One cloud's covariances split over several GPUs (dense scans against a sharded submap, SURVEY section 8e): every
 * rank holds the same source cloud (same index, the build is deterministic) and computes the covariances of slice
 * `part` of `nparts` of it (equal slices of the cell-sorted order, i.e. spatially coherent); the entries of the other
 * slices are zero, so an element-wise SUM over the ranks (one all-reduce of 48 B/point over NVLink, exact: x + 0) gives
 * every rank the complete set.  ngicp_covs_device exposes the device buffer (n x 6 doubles: xx,xy,xz,yy,yz,zz in the
 * cloud's own point order) for that collective; it stays owned by the handle. */
int ngicp_calc_source_covs_part(ngicp_t* h, int part, int nparts);
int ngicp_covs_device(ngicp_t* h, int which, double** covs6, size_t* n);
/* test hook: the k neighbours (nearestKSearch result at nano_gicp_impl.hpp:313) the LAST calculate*Covariances call on
 * this handle used for every point of that cloud, in the order the covariance sums ran over them — ascending
 * squared distance, exact ties in (cell, original index) order: idx[n*k] original point indices (-1 = none), d2[n*k] squared distances.  Valid
 * until the next covariance / kNN call on the handle. */
int ngicp_cov_neighbors(ngicp_t* h, int which, int* idx, float* d2);
/* NanoGICP::setSourceCovariances / setTargetCovariances, nano_gicp_impl.hpp:141-149 (n Matrix4d records, host or device) */
int ngicp_set_source_covs(ngicp_t* h, const double* covs, size_t n);
int ngicp_set_target_covs(ngicp_t* h, const double* covs, size_t n);
/* `source_covs_.clear()` (odom.cc:526) */
int ngicp_clear_covs(ngicp_t* h, int which);
/* NanoGICP::getSourceCovariances / getTargetCovariances, nano_gicp.hpp:100-106: writes n*16 doubles */
size_t ngicp_covs_size(const ngicp_t* h, int which);
int ngicp_get_source_covs(ngicp_t* h, double* out, size_t n);
int ngicp_get_target_covs(ngicp_t* h, double* out, size_t n);

/* ---- registration ----------------------------------------------------------------------------- */
/* pcl::Registration::align(output, guess) -> NanoGICP::computeTransformation (nano_gicp_impl.hpp:161-171)
 * -> LsqRegistration::computeTransformation (lsq_registration_impl.hpp:89-115).  Lazily computes missing
 * covariances like the reference.  `guess` NULL = identity (align(output)). */
int ngicp_align(ngicp_t* h, const float* guess16, ngicp_result* out);
/* Batched registration (BASELINE config "10k independent scan pairs"; no reference counterpart — the reference loops
 * over align()): n handles, each set up like for ngicp_align (source, target, parameters; covariances are computed
 * lazily where missing), registered by ONE kernel launch — a thread-block cluster per pair runs that pair's whole LM loop
 * (nano_gicp_impl.hpp:173-296, lsq_registration_impl.hpp:89-208) with exactly the sums of the single-pair kernel, so
 * results[i] is bit-identical to what ngicp_align(handles[i], guess_i, ..) returns.  guesses16: n x 16 floats
 * (column-major 4x4 each) or NULL for identity.  All handles on one device, each at most once; the index / covariance
 * work of different handles runs concurrently on their own streams. */
int ngicp_align_batch(ngicp_t* const* handles, size_t n, const float* guesses16, ngicp_result* results);
/* pcl::transformPointCloud(*input_, output, final) at lsq_registration_impl.hpp:114: writes n packed
 * {x,y,z,1} float4 records (host or device); the facade merges them into the output cloud's records */
int ngicp_transform_source(ngicp_t* h, const float* T16, float* out_xyz1, size_t n);
/* pcl::Registration::getFitnessScore(max_range): mean squared distance from the source, transformed by T (float,
 * column-major, as pcl::transformPointCloud), to its nearest target point, over the points whose SQUARED distance is
 * <= max_range (PCL's comparison).  *score = DBL_MAX and *n_inliers = 0 when no point qualifies.  n_inliers may be NULL.
 * Empty source or target: DBL_MAX / 0.  NGICP_E_INVALID: null arguments or a NaN max_range; NGICP_E_STATE: no source, no
 * target, or a target without a search index; NGICP_E_UNSUPPORTED: a handle in sharded mode (it holds one slab of the
 * target).  Touches no registration state. */
int ngicp_fitness_score(ngicp_t* h, const float* T16, double max_range, double* score, size_t* n_inliers);
/* the same for n handles (own source + target each, one device, each at most once) in a constant number of launches;
 * T16s: n x 16 floats; bit-identical to n single calls */
int ngicp_fitness_batch(ngicp_t* const* handles, size_t n, const float* T16s, double max_range, double* scores, size_t* n_inliers);

/* ---- voxel grid ------------------------------------------------------------------------------- */
/* pcl::VoxelGrid<PointXYZI>::filter with leaf (l,l,l) (odom.cc:126-127,460-463,487-490,1160-1163).
 * in: n PointXYZI-like records (x,y,z at floats 0..2, intensity at float 4 when stride_bytes >= 20);
 * out: up to out_capacity 32-byte PointXYZI records {x,y,z,1,intensity,0,0,0}, ordered by voxel index;
 * *m = number written.  in/out may be host or device memory. */
int ngicp_voxel_filter(ngicp_t* h, const void* in, size_t n, size_t stride_bytes, float leaf, void* out,
                       size_t out_capacity, size_t* m);
/* OdomNode::preprocessPoints (odom.cc:443-465) in one pass over the raw scan: pcl::removeNaNFromPointCloud (:451),
 * the negative pcl::CropBox (:122-124,454-457; a point with crop_min <= p <= crop_max on all axes is dropped; pass NULL
 * for both to skip it) and the scan voxel grid (:460-463; leaf <= 0 skips it, as vf_scan_use_ = false does).  Output
 * records as ngicp_voxel_filter; without a voxel grid the surviving points keep their input order. */
int ngicp_preprocess(ngicp_t* h, const void* in, size_t n, size_t stride_bytes, const float* crop_min, const float* crop_max,
                     float leaf, void* out, size_t out_capacity, size_t* m);
/* The keyframe path: pcl::transformPointCloud(*cloud, *cloud, T) followed by vf_submap.filter (odom.cc:484-490,
 * 1157-1163) in one pass; T16 = column-major float 4x4; leaf <= 0 only transforms.  With non-finite inputs or PCL's
 * index overflow the surviving transformed points are emitted in input order. */
int ngicp_transform_voxel_filter(ngicp_t* h, const void* in, size_t n, size_t stride_bytes, const float* T16, float leaf,
                                 void* out, size_t out_capacity, size_t* m);
/* pcl::fromROSMsg (odom.cc:636-637) + preprocessPoints in the same pass: `data` is the byte array of a
 * sensor_msgs::PointCloud2 (host or device), the layout carries the message's geometry and the byte offsets of its
 * FLOAT32 fields named "x", "y", "z", "intensity" (what pcl::fromROSMsg's field mapping matches for pcl::PointXYZI:
 * same name, datatype FLOAT32, count 1; offset_intensity = -1 when the message has no such field — PCL then leaves
 * intensity 0).  Offsets and steps need not be 4-byte aligned.  Output as ngicp_preprocess. */
typedef struct ngicp_pc2_layout {
  unsigned width, height;        /* points per row, rows (n = width * height) */
  unsigned point_step, row_step; /* bytes per point / per row */
  int offset_x, offset_y, offset_z, offset_intensity;
  int is_bigendian;              /* must be 0 */
} ngicp_pc2_layout;
int ngicp_preprocess_pointcloud2(ngicp_t* h, const void* data, const ngicp_pc2_layout* layout, const float* crop_min,
                                 const float* crop_max, float leaf, void* out, size_t out_capacity, size_t* m);
/* test hook: the output slot every input point was averaged into (-1 for non-finite points) */
int ngicp_voxel_assignment(ngicp_t* h, int* slot_of_point, size_t n);

/* ---- introspection used by the parity tests --------------------------------------------------- */
/* KdTreeFLANN::nearestKSearch (nanoflann.hpp:141-152) for nq queries against the source/target index:
 * idx[nq*k] (original point order, -1 padded), d2[nq*k] ascending */
int ngicp_knn(ngicp_t* h, int which, const float* queries, size_t nq, size_t q_stride_bytes, int k, int* idx, float* d2);
/* NanoGICP::linearize (nano_gicp_impl.hpp:213-270): H 6x6 col-major, b, sum of errors; optional per-point
 * correspondences_ (target index or -1), sq_distances_, and mahalanobis_ (n*16 doubles) */
int ngicp_linearize(ngicp_t* h, const double* T16, double* H36, double* b6, double* err, int* corr, float* sqd, double* mahal);
/* test hook: the per-point state the LAST linearisation on this handle left behind — ngicp_linearize, a fused or stepped
 * ngicp_align (its last linearisation; with max_iterations = 1 the one at the guess) or ngicp_align_batch — in
 * ngicp_linearize's layout: corr[n] target index or -1, sqd[n] nearest squared distance (FLT_MAX without a
 * correspondence), mahal16[n*16] col-major 4x4 (zero without a correspondence).  Any output may be NULL.
 * NGICP_E_STATE when no linearisation is valid for the current clouds. */
int ngicp_correspondences(ngicp_t* h, int* corr, float* sqd, double* mahal16);
/* NanoGICP::compute_error (nano_gicp_impl.hpp:272-296) with the correspondences frozen by the last linearize */
int ngicp_compute_error(ngicp_t* h, const double* T16, double* err);
/* sharded-submap building block: like ngicp_linearize but returns the raw partial sums
 * out43 = {H (36, col-major), b (6), err (1)} so that ranks can all-reduce them; out43 may be device memory */
int ngicp_linearize_partial(ngicp_t* h, const double* T16, double* out43);
/* sharded submap with an UNBOUNDED correspondence distance (the library default corr_dist_threshold_ = FLT_MAX,
 * nano_gicp_impl.hpp:59; slabs + halo are only exact for a finite one): the ranks exchange nearest neighbours.
 *   ngicp_nn1_packed     every source point's nearest neighbour in THIS handle's target under T, as
 *                        (bits of the squared distance) << 32 | rank, 0x7f800000ffffffff = none within the
 *                        max-correspondence distance; packed_out: n_source entries, host or device
 *   (min-all-reduce the arrays over the ranks as int64: the lowest value names the rank holding the global nearest
 *    neighbour; equal distances go to the lowest rank)
 *   ngicp_linearize_won  the partial sums {H, b, err} (layout of ngicp_linearize_partial) over the source points this
 *                        rank won; ngicp_compute_error_partial then works on the same points */
int ngicp_nn1_packed(ngicp_t* h, const double* T16, unsigned rank, unsigned long long* packed_out);
int ngicp_linearize_won(ngicp_t* h, const double* T16, unsigned rank, const unsigned long long* packed_min, double* out43);
int ngicp_compute_error_partial(ngicp_t* h, const double* T16, double* out1);

/* sharded-submap mode (one handle per GPU holds one spatial slab of the target plus a halo of the max-correspondence
 * distance): count only source points whose transformed position lies in [lo, hi) along `axis` (0/1/2; -1 = off) */
int ngicp_set_owner_slab(ngicp_t* h, int axis, float lo, float hi);
/* The exchange step of the sharded mode, fused into ngicp_align: once connected, the persistent LM kernel of every rank
 * writes its partial {H, b, err} (and each trial's error) into every rank's exchange buffer over NVLink / NVSwitch peer
 * memory, waits for the others' flags and sums in rank order — the reference's serial merge of per-thread partials
 * (nano_gicp_impl.hpp:260-267) stretched across GPUs, with no host round trip and no separate collective launch.
 * All ranks must call ngicp_align with the same source, parameters and guess; they take identical LM decisions.
 *   ngicp_comm_export        allocates this rank's exchange buffer and returns its 64-byte CUDA IPC handle
 *   ngicp_comm_connect       maps the buffers of all `world` ranks (handles = world x 64 bytes, indexed by rank; one
 *                            process per GPU); callers must barrier between connect and the first align
 *   ngicp_comm_connect_local the same for handles living in THIS process (several GPUs, or one GPU for tests)
 *   ngicp_comm_close         unmaps; ngicp_align is single-GPU again
 * A rank that does not arrive within NGICP_COMM_TIMEOUT_MS (environment, default 2000) makes ngicp_align return
 * NGICP_E_COMM on the waiting ranks instead of hanging the GPU; reconnect before the next align. */
#define NGICP_COMM_HANDLE_BYTES 64
int ngicp_comm_export(ngicp_t* h, void* handle64);
int ngicp_comm_connect(ngicp_t* h, int rank, int world, const void* handles);
int ngicp_comm_connect_local(ngicp_t* h, int rank, int world, ngicp_t* const* peers);
int ngicp_comm_close(ngicp_t* h);
/* After NGICP_E_COMM the ranks' sequence numbers are out of step and the error flag is sticky: EVERY rank calls this
 * (no align in flight anywhere; put a barrier of the host's process group behind it), which zeroes the rank's own exchange
 * buffer — slots, flags, sequence number, error — and keeps the connections.  The failed align stopped its LM loop at the
 * failed exchange (all blocks of the kernel leave together); its result is not meaningful. */
int ngicp_comm_reset(ngicp_t* h);
/* host-only: the scalar side of one LM trial (lsq_registration_impl.hpp:172-179): d = solve(H + lambda I, -b),
 * delta = [so3_exp(d[0:3]) | d[3:6]], xi = delta * x0 — the same code the fused kernel runs; lambda = 0 gives the
 * Gauss-Newton step (:147-154).  4x4 matrices column-major. */
int ngicp_lm_trial(const double* H36, const double* b6, double lambda, const double* x0_16, double* d6, double* delta16, double* xi16);
/* LsqRegistration::is_converged (lsq_registration_impl.hpp:118-127) */
int ngicp_lm_is_converged(const double* delta16, double rot_eps, double trans_eps);

/* ---- the guess of the S2S align when an IMU is used (SURVEY §8f N4, second half) --------------------------------
 * OdomNode::integrateIMU (odom.cc:859-919): of the n gyro samples (stamps[i] seconds, ang_vel[3*i..] rad/s) those with
 * prev_frame_stamp <= stamp <= curr_frame_stamp are sorted by time and integrated from the identity with the first-order
 * quaternion update q += 0.5 * q (x) (0, w) dt (float quaternion, double products, the first sample only sets the clock),
 * the result is normalised and written as the rotation block of a column-major 4x4 float matrix with zero translation
 * — the `imu_SE3` that getNextPose hands to gicp_s2s.align (odom.cc:801-803).  Host arithmetic, like in the reference;
 * needs no handle and no GPU.  Fewer than two usable samples give the identity. */
int ngicp_imu_prior(const double* stamps, const double* ang_vel_xyz, size_t n, double prev_frame_stamp, double curr_frame_stamp,
                    float* out_T16);

/* ---- device-resident keyframes (additive; SURVEY §8f N1) ------------------------------------------------------
 * OdomNode keeps every keyframe's voxelised world-frame cloud and covariances on the host (keyframes / keyframe_normals,
 * include/dlo/odom.h:80-82), concatenates the selected ones into submap_cloud / submap_normals (odom.cc:1315-1328) and
 * hands both back through setInputTarget + setTargetCovariances (:830-833) — 160 bytes per submap point over PCIe each
 * time the submap changes.  The store keeps the device buffers instead:
 *   ngicp_kfstore_push        right after gicp_s2s.setInputSource(keyframe_cloud) + calculateSourceCovariances()
 *                             (:498-500,1172-1174): keeps a device copy of that cloud's points and shares its covariance buffer
 *   ngicp_kfstore_set_target  target of `to` = the selected keyframes concatenated in the given order (device-to-device)
 *                             + search index; equivalent to the host concatenation followed by :830-833 */
typedef struct ngicp_kfstore ngicp_kfstore_t;
int ngicp_kfstore_create(int device, ngicp_kfstore_t** out);
void ngicp_kfstore_destroy(ngicp_kfstore_t* s);
size_t ngicp_kfstore_size(const ngicp_kfstore_t* s);
size_t ngicp_kfstore_points(const ngicp_kfstore_t* s, size_t index);
int ngicp_kfstore_push(ngicp_kfstore_t* s, ngicp_t* from, size_t* index_out);
int ngicp_kfstore_set_target(ngicp_kfstore_t* s, ngicp_t* to, const int* indices, size_t n_indices);

/* ---- submap keyframe selection (SURVEY §8f N3; host arithmetic in the host language, no GPU, no handle) ------------
 * OdomNode::getSubmapKeyframes (odom.cc:1240-1293) picks the keyframes of the scan-to-map target: the knn keyframes
 * nearest to the current pose, the kcv nearest among the vertices of the 3-D convex hull of all keyframe positions
 * (computeConvexHull, :1017-1050, pcl::ConvexHull -> qhull) and the kcc nearest among the vertices of their 3-D alpha
 * shape (computeConcaveHull, :1057-1090, pcl::ConcaveHull with alpha = keyframe threshD, :95-98).  PCL and qhull do not
 * exist here: csrc/submap_select.cpp builds both hulls from their definitions (incremental hull; Bowyer-Watson Delaunay
 * + PCL's alpha filter).  Positions are n x 3 floats.  Functions returning a count return NGICP_E_INVALID when out_cap
 * is too small.
 *   ngicp_submap_push_indices   pushSubmapIndices (:1210-1233): frames[i] with dists[i] <= the k-th smallest distance
 *   ngicp_submap_convex_hull    indices of the input points that are convex-hull vertices (ascending); none for flat input
 *   ngicp_submap_concave_hull   indices of the input points on the alpha shape (ascending)
 *   ngicp_submap_select         the whole selection with OdomNode's state between scans (hulls kept while there are too
 *                               few keyframes, *changed = submap_hasChanged); out = sorted unique keyframe indices
 *   ngicp_submap_selector_hulls keyframe_convex (which = 0) / keyframe_concave (which = 1) after the last select
 *   ngicp_keyframe_wanted       updateKeyframes' decision (:1102-1153): 1 = add a keyframe at the current pose; quaternions
 *                               are (w, x, y, z) floats */
typedef struct ngicp_submap_selector ngicp_submap_selector_t;
int ngicp_submap_push_indices(const float* dists, const int* frames, int n, int k, int* out, int out_cap);
int ngicp_submap_convex_hull(const float* xyz, int n, int* out, int out_cap);
int ngicp_submap_concave_hull(const float* xyz, int n, double alpha, int* out, int out_cap);
int ngicp_submap_selector_create(int knn, int kcv, int kcc, double alpha, ngicp_submap_selector_t** out);
void ngicp_submap_selector_destroy(ngicp_submap_selector_t* s);
int ngicp_submap_select(ngicp_submap_selector_t* s, const float* kf_xyz, int n, const float* cur_xyz, int* out, int out_cap, int* changed);
int ngicp_submap_selector_hulls(ngicp_submap_selector_t* s, int which, int* out, int out_cap);
int ngicp_keyframe_wanted(const float* kf_xyz, const float* kf_quat_wxyz, int n, const float* cur_xyz, const float* cur_quat_wxyz,
                          double thresh_dist, double thresh_rot_deg);

/* diagnostics: the uniform grid chosen for a cloud's search index (cell edge in metres, dims[3], cell count) */
int ngicp_grid_info(ngicp_t* h, int which, float* cell, int* dims3, int* ncells);

/* number of CUDA kernels this library has launched since it was loaded (all handles; diagnostics for bench.py) */
unsigned long long ngicp_launch_count(void);

/* library identification: "nanogicp-b200 <version> sm_100a" */
const char* ngicp_version(void);

#ifdef __cplusplus
}
#endif
#endif /* NANOGICP_C_H */
