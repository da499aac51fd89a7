// internal.h — host-side declarations shared by the translation units of libnanogicp_b200.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "../../include/nanogicp_c.h"
#include "common.cuh"

namespace ngicp {

// ---- streams and device memory -----------------------------------------------------------------
struct StreamRef {
  cudaStream_t s = nullptr;
  bool owned = false;
  ~StreamRef() {
    if (owned && s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
  }
};
typedef std::shared_ptr<StreamRef> StreamPtr;

cudaError_t pool_alloc_async(void** p, size_t nbytes, cudaStream_t s);   // from the library's private memory pool
// stream-ordered device buffer (the library's own pool on an owned stream, plain cudaMalloc/cudaFree otherwise)
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  StreamPtr st;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  cudaError_t alloc(size_t nbytes, const StreamPtr& stream);
  // grow-only: keeps the allocation when it is already large enough
  cudaError_t reserve(size_t nbytes, const StreamPtr& stream);
  void release();
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// The dense cell table is by far the largest per-cloud buffer (capacity x 4 B, 128 MiB by default) and clouds come
// and go once per scan, so tables are recycled through a small per-process free list instead of the allocator
// (a fresh 128 MiB cudaMallocAsync costs 0.6-25 ms, measured; see benchmarks/exp_setsrc.py).
struct TableBuf {
  void* p = nullptr;
  size_t bytes = 0;
  int device = 0;
  StreamPtr st;
  TableBuf() {}
  TableBuf(const TableBuf&) = delete;
  TableBuf& operator=(const TableBuf&) = delete;
  ~TableBuf() { release(); }
  cudaError_t acquire(size_t nbytes, int dev, const StreamPtr& stream);
  void release();
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// ---- device-resident cloud + index ---------------------------------------------------------------
// Brick occupancy flags of the tile kNN path: one byte per box of KNN_BRICK^3 cells says whether the box holds points
// (the plan kernel then need not walk the dense cell table).  The fused index kernel fills them as a by-product of its
// last pass for clouds that may take the tile path; otherwise launch_covariances does (brick_clear / brick_mark).
constexpr int KNN_BRICK = 4;
inline long long brick_flag_bytes(int table_cap) { return ((long long)table_cap / 16 + 4096) & ~3ll; }   // 4x the boxes of a cubic grid
constexpr int KNN_BRICK_MIN_POINTS = 8192;      // smaller clouds never take the tile path by themselves

struct DevCloud {
  int n = 0;
  DevBuf pts;         // float4[n], original order, w = 1
  bool indexed = false;
  DevBuf desc;        // GridDesc
  TableBuf cell_start;  // int[table_cap + 8], recycled
  DevBuf sorted;      // float4[n], cell order, w = original index bits
  DevBuf bricks;      // brick occupancy flags (see KNN_BRICK) when the index build produced them, else empty
  int table_cap = 0;
  GridView view() const {
    GridView v;
    v.cell_start = cell_start.as<int>() + 3;   // see build_index: 3 ints of alignment padding
    v.sorted = sorted.as<float4>();
    v.desc = desc.as<GridDesc>();
    return v;
  }
};
typedef std::shared_ptr<DevCloud> CloudPtr;

struct DevCovs {
  int n = 0;
  DevBuf c;  // double[n*6], original point order, {xx,xy,xz,yy,yz,zz}
};
typedef std::shared_ptr<DevCovs> CovsPtr;

// side stream (high priority) + fork/join events on which the tile path answers its warp-search rest beside the main
// covariance launch; nullptr = everything on the one stream
struct CovSideStream { cudaStream_t stream = nullptr; cudaEvent_t fork = nullptr, join = nullptr; };

// grow-only scratch owned by a handle
struct Scratch {
  Scratch() {}
  Scratch(const Scratch&) = delete;
  Scratch& operator=(const Scratch&) = delete;
  ~Scratch() {
    if (vox_result) cudaFreeHost(vox_result);
    if (copy_done) cudaEventDestroy(copy_done);
    if (cov_side.stream) { cudaStreamSynchronize(cov_side.stream); cudaStreamDestroy(cov_side.stream); }
    if (cov_side.fork) cudaEventDestroy(cov_side.fork);
    if (cov_side.join) cudaEventDestroy(cov_side.join);
  }
  CovSideStream cov_side;            // created on first use by calc_covs
  cudaEvent_t copy_done = nullptr;   // see host_source_consumed()
  DevBuf staging;    // raw bytes of caller records
  DevBuf keys_a, keys_b, vals_a, vals_b;
  DevBuf hist, tile_sums;
  DevBuf flags;      // voxel head flags / scanned slots
  DevBuf vox_desc;   // GridDesc for the voxel filter
  DevBuf vox_bar;    // grid barrier words of the fused voxel kernel (zero between launches)
  DevBuf index_bar;  // ... of the fused index kernel
  int index_path = 0;  // ngicp_params::index_path of the owning handle (1 = multi-kernel upload + index build only)
  int vox_path = 0;             // ngicp_params::voxel_path of the owning handle (1 = multi-kernel pipeline only)
  int vox_bits_hint = 0;        // key bits the last voxel filter needed (0 = unknown): lets the next call queue its radix
                                // passes without a mid-pipeline read-back of the grid dimensions
  int* vox_result = nullptr;    // mapped pinned {m, overflow, key bits needed}: written by the pipeline's last kernel
  int* vox_result_dev = nullptr;
  DevBuf nn1_packed, nn1_won;   // min-exchange mode of the sharded submap (ngicp_nn1_packed / ngicp_linearize_won)
  DevBuf vox_out;    // PointXYZI records
  DevBuf vox_slot;   // int per input point
  DevBuf knn_idx, knn_d2, queries;
  DevBuf nbr;        // int[n*k] neighbour slots between the kNN and covariance kernels
  DevBuf cov_stage;  // Matrix4d staging for import/export
  // align state
  DevBuf mahal;      // double[ns*6]
  DevBuf corr;       // int[ns]   target ORIGINAL index or -1
  DevBuf sqd;        // float[ns]
  DevBuf tgt_pt;     // float4[ns] matched target point
  DevBuf partials;   // double[blocks*NRED]
  DevBuf reduced;    // double[64]
  DevBuf lm_state;   // device-resident LM state / result of the fused kernel
  DevBuf barrier;    // unsigned counters for the grid barrier
  DevBuf trace;      // debug: %globaltimer stamps of the fused kernel
  DevBuf batch_args; // BatchPair records of ngicp_align_batch
  DevBuf fit_args, fit_partials;   // FitnessPair records and per-chunk {sum, count} of ngicp_fitness_batch
};

// number of kernels launched by this library since load (diagnostics; ngicp_launch_count())
void note_launches(int n);

// ---- sort_scan.cu ---------------------------------------------------------------------------------
void exclusive_scan_inplace(int* data, const int* n_dev, int n_add, int max_n, int* tile_sums, cudaStream_t st);
size_t scan_scratch_ints(int max_n);
size_t radix_sort_scratch_ints(int n);
int radix_sort_pairs(unsigned* keys_a, unsigned* vals_a, unsigned* keys_b, unsigned* vals_b, int n, int bits, int* hist, cudaStream_t st);

// ---- cloud_index.cu -------------------------------------------------------------------------------
// snapshot caller records into cloud.pts (float4) and compute the bounding box into cloud.desc
cudaError_t upload_cloud(DevCloud& c, const void* pts, size_t n, size_t stride_bytes, Scratch& sc, const StreamPtr& st);
// build the uniform grid index of an uploaded cloud
cudaError_t build_index(DevCloud& c, float cell_req, int table_cap, Scratch& sc, const StreamPtr& st, int device);
// both of the above in one persistent cooperative launch; *done = false: not applicable, take the two calls
cudaError_t upload_and_index_fused(DevCloud& c, const void* pts, size_t n, size_t stride_bytes, float cell_req, int table_cap, Scratch& sc,
                                   const StreamPtr& st, int device, bool* done);

// ---- knn_cov.cu -----------------------------------------------------------------------------------
cudaError_t launch_knn_queries(const DevCloud& c, const float4* queries, int nq, int k, int* idx, float* d2, cudaStream_t st);
size_t covariance_scratch_ints(int n, int k, int table_cap);   // neighbour lists + the work lists / flags of the kNN kernels
cudaError_t launch_covariances(const DevCloud& c, int k, int method, int* nbr_scratch /* covariance_scratch_ints() */, double* covs6, int table_cap, cudaStream_t st,
                               int part = 0, int nparts = 1, int knn_path = NGICP_KNN_AUTO, int tile_min_points = 131072,
                               const CovSideStream* side = nullptr);
// test hook: the neighbour lists left in nbr_scratch by launch_covariances, in summation order, as original indices
cudaError_t launch_export_neighbors(const DevCloud& c, int k, const int* nbr_scratch, int* idx_out, float* d2_out, cudaStream_t st);
constexpr int KNN_MAX_K = 32;        // warp-distributed result set (one entry per lane): every tuned kNN kernel
constexpr int KNN_WIDE_MAX_K = 128;  // shared-memory result set of the wide warp search: what the library accepts

// ---- align.cu -------------------------------------------------------------------------------------
struct AlignBuffers {
  const float4* src_pts; const double* src_cov; int ns;
  GridView tgt; const double* tgt_cov; int nt;
  double* mahal; int* corr; float* sqd; float4* tgt_pt;
  double* partials; double* reduced; int max_blocks;
  int slab_axis = -1; float slab_lo = 0.f, slab_hi = 0.f;
};
// one linearisation at T (row-major R + t as Iso3 passed by value inside); reduced[0..NRED) <- packed H,b,err
cudaError_t launch_linearize(const AlignBuffers& ab, const double* T16_colmajor, double max_corr_dist, cudaStream_t st);
cudaError_t launch_nn1_packed(const AlignBuffers& ab, const double* T16, double max_corr_dist, unsigned rank, unsigned long long* out, cudaStream_t st);
cudaError_t launch_linearize_won(const AlignBuffers& ab, const double* T16, double max_corr_dist, unsigned rank, const unsigned long long* won,
                                 cudaStream_t st);
cudaError_t launch_compute_error(const AlignBuffers& ab, const double* T16_colmajor, cudaStream_t st);
cudaError_t launch_export_mahal(const AlignBuffers& ab, double* out16, cudaStream_t st);
// sharded-submap mode: where every rank's exchange buffer is mapped in this process (see align.cu, peer_exchange_sum)
constexpr int NGICP_MAX_RANKS = 8;
constexpr int PEER_SLOT_DOUBLES = 32;                       // >= NRED
constexpr size_t PEER_DATA_BYTES = sizeof(double) * 2 * NGICP_MAX_RANKS * PEER_SLOT_DOUBLES;
constexpr size_t PEER_FLAG_BYTES = sizeof(unsigned long long) * 2 * NGICP_MAX_RANKS;
constexpr size_t PEER_BUF_BYTES = PEER_DATA_BYTES + PEER_FLAG_BYTES + 64;   // + local exchange counter and error flag
struct PeerComm {
  int world, rank;
  double* data[NGICP_MAX_RANKS];               // [2][NGICP_MAX_RANKS][PEER_SLOT_DOUBLES] on each rank
  unsigned long long* flag[NGICP_MAX_RANKS];   // [2][NGICP_MAX_RANKS] on each rank
  unsigned long long* seq;                     // local: exchanges completed
  int* error;                                  // local: sticky "peer timed out"
  unsigned long long timeout_ns;
};
// the whole LM loop in one persistent cooperative kernel; result written to *res_dev (ngicp_result layout)
cudaError_t launch_align_fused(const AlignBuffers& ab, const ngicp_params& prm, const float* guess16, ngicp_result* res_dev,
                               unsigned* barrier, int device, cudaStream_t st, unsigned long long* trace = nullptr,
                               const PeerComm* comm = nullptr);
int align_fused_max_blocks(int device);
// batched registration (ngicp_align_batch): one cluster per pair, see align.cu
size_t align_batch_pair_bytes();
int align_batch_fill(void* dst, const AlignBuffers& ab, const ngicp_params& p, const float* guess16, ngicp_result* res_dev, int device);
cudaError_t launch_align_batch(const void* pairs_dev, int n_pairs, int lpp, cudaStream_t st);
void align_prime_kernels(int device);
void knn_prime_kernels();
void voxel_prime_kernels();
void index_prime_kernels();

// ---- fitness.cu -----------------------------------------------------------------------------------
// pcl::Registration::getFitnessScore over n pairs (ngicp_fitness_score / ngicp_fitness_batch), two launches in all
constexpr int FITNESS_CHUNK = 256;   // source points per work item: fixed, so a pair's summation order never changes
struct FitnessPair {
  const float4* src; int ns;
  GridView tgt;
  float T[12];      // rows of the float transform: T[r*4+c], c = 3 the translation
  int lpp;          // lanes per source point in the radius-1 cube search (1 or 2)
  int chunk0;       // first chunk of this pair in the launch
  int nchunks;      // 0 for an empty source or target
};
struct FitnessResult { double score; unsigned long long n; };
// partials: double2[total_chunks]; out: n_pairs results (mapped host memory)
cudaError_t launch_fitness(const FitnessPair* pairs_dev, int n_pairs, int total_chunks, double max_range, double2* partials,
                           FitnessResult* out, cudaStream_t st);

// ---- voxel.cu -------------------------------------------------------------------------------------
// returns cudaSuccess; *m_out and *overflow are valid after the call (it synchronises once to learn m)
// crop6 = {min xyz, max xyz} of a negative pcl::CropBox or nullptr; leaf <= 0 skips the voxel grid (compaction only);
// compact_on_overflow: on PCL's index-overflow pass-through emit the surviving points instead of leaving it to the caller
// "The caller keeps ownership and may free the buffer on return": a staging copy from PAGEABLE host memory has left the
// caller's buffer when cudaMemcpyAsync returns, one from PINNED host memory has not — wait for it (the copy only, not
// the kernels queued behind it).  Device-resident inputs are read in stream order and documented as such.
cudaError_t host_source_consumed(const void* src, Scratch& sc, cudaStream_t st);

// where record i of a raw cloud lives and where its FLOAT32 fields are (byte offsets; off[3] = intensity, -1 = absent)
struct RecordLayout {
  int width;                 // records per row (>= n: one row)
  size_t point_step, row_step;
  int off[4];
  int aligned;               // every field address is 4-byte aligned (offsets, steps; the staging copy itself is)
};
// out/out_cap/copied: when given, the routine may deliver the records to the caller's buffer itself (device buffers:
// by a kernel that reads the count on the device, so that the whole call needs ONE synchronisation) and says so.
cudaError_t voxel_filter_records(const void* in, size_t n, RecordLayout lay, float leaf, Scratch& sc, const StreamPtr& st,
                                 size_t* m_out, int* overflow, const float* crop6 = nullptr, bool compact_on_overflow = false,
                                 const float* T16 = nullptr, void* out = nullptr, size_t out_cap = 0, bool* copied = nullptr,
                                 bool allow_speculation = true);
cudaError_t voxel_filter_device(const void* in, size_t n, size_t stride_bytes, float leaf, Scratch& sc, const StreamPtr& st,
                                size_t* m_out, int* overflow, const float* crop6 = nullptr, bool compact_on_overflow = false,
                                const float* T16_colmajor = nullptr /* transformPointCloud first */, void* out = nullptr,
                                size_t out_cap = 0, bool* copied = nullptr);

}  // namespace ngicp
