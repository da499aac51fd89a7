// oracle/gicp_oracle.cpp — CPU ORACLE for the NanoGICP hot path.  TEST INFRASTRUCTURE ONLY.
//
// This file is a plain-C++ restatement of the reference's algorithm for the path this
// repo accelerates.  It is NOT part of the product: only tests/, __graft_entry__.smoke()
// and bench.py's cpu_baseline / --impl reference legs may load it.  The product library
// (direct_lidar_odometry_b200/csrc) never links, loads or calls anything in oracle/.
//
// What it follows (all paths relative to /root/reference):
//   voxel filter      pcl::VoxelGrid<PointXYZI>::applyFilter (PCL >=1.10, NOT in the tree; call
//                     sites src/dlo/odom.cc:460-463,487-490,1160-1163) — restated from the published
//                     algorithm, see SURVEY.md App. B1; where PCL's index arithmetic is undefined or wraps
//                     (voxel_grid_setup) the cloud passes through, as in the GPU kernels
//   kd-tree           include/nano_gicp/impl/nanoflann_impl.hpp:867-1012 (build), :1230-1250,
//                     :1355-1418 (query), :149-214 (result set), :441-449 (metric);
//                     wrapper include/nano_gicp/nanoflann.hpp:113-152 (leaf size 100, int index)
//   covariances       include/nano_gicp/impl/nano_gicp_impl.hpp:298-357
//   correspondences   include/nano_gicp/impl/nano_gicp_impl.hpp:173-211
//   linearize         include/nano_gicp/impl/nano_gicp_impl.hpp:213-270
//   compute_error     include/nano_gicp/impl/nano_gicp_impl.hpp:272-296
//   LM / GN driver    include/nano_gicp/impl/lsq_registration_impl.hpp:89-208
//   so3_exp, skewd    include/nano_gicp/gicp/so3.hpp:62-72,99-118
//
// PARITY PIN STATUS
//   * kd-tree kNN: PINNED.  When built with -DORACLE_WITH_REF_NANOFLANN (oracle/_ref/), the
//     kNN backend is the reference's own vendored nanoflann header compiled as-is from
//     /root/reference; tests/golden/knn_ref_*.npz were produced by that build
//     (tests/golden/make_golden.py) and the restated tree below must reproduce them bit-for-bit.
//   * everything that lives in Eigen / PCL (JacobiSVD, Matrix4d::inverse, LDLT, VoxelGrid,
//     Isometry3f*Vector4f evaluation order): PARITY UNPINNED — the reference has no tests,
//     no golden vectors, and Eigen/PCL are not installed here, so those pieces are restated
//     from the libraries' published algorithms and checked by property tests only
//     (tests/test_oracle_*.py).
//
// Build flags mirror the reference's CMakeLists.txt:13-14,24-28 (-std=c++14 -O3 -fopenmp,
// no -march=native) plus -ffp-contract=off so no FMA is ever formed.

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <limits>
#include <memory>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

#ifdef ORACLE_WITH_REF_NANOFLANN
#include <nanoflann_impl.hpp>  // from -I/root/reference/include/nano_gicp/impl (never copied into this repo)
#endif

namespace orc {

// ------------------------------------------------------------------------------------------
// tiny column-major fixed-size matrices (Eigen is not available in this image)
// ------------------------------------------------------------------------------------------
template <int R, int C>
struct Mat {
  double v[R * C];
  Mat() { for (int i = 0; i < R * C; i++) v[i] = 0.0; }
  double& operator()(int r, int c) { return v[c * R + r]; }
  double operator()(int r, int c) const { return v[c * R + r]; }
  static Mat identity() { Mat m; for (int i = 0; i < (R < C ? R : C); i++) m(i, i) = 1.0; return m; }
};
template <int R, int K, int C>
static Mat<R, C> mul(const Mat<R, K>& a, const Mat<K, C>& b) {
  Mat<R, C> o;
  for (int c = 0; c < C; c++)
    for (int r = 0; r < R; r++) {
      double s = 0.0;
      for (int k = 0; k < K; k++) s += a(r, k) * b(k, c);
      o(r, c) = s;
    }
  return o;
}
template <int R, int C>
static Mat<C, R> tr(const Mat<R, C>& a) {
  Mat<C, R> o;
  for (int c = 0; c < C; c++) for (int r = 0; r < R; r++) o(c, r) = a(r, c);
  return o;
}
template <int R, int C>
static Mat<R, C> add(const Mat<R, C>& a, const Mat<R, C>& b) {
  Mat<R, C> o;
  for (int i = 0; i < R * C; i++) o.v[i] = a.v[i] + b.v[i];
  return o;
}
typedef Mat<4, 4> M4;
typedef Mat<3, 3> M3;
typedef Mat<6, 6> M6;
typedef Mat<6, 1> V6;
typedef Mat<4, 1> V4;

// General 4x4 inverse by cofactors (stands in for Eigen's fixed-size-4 inverse kernel used at
// nano_gicp_impl.hpp:208; SURVEY App. B4 — tolerance-level parity only).
static M4 inverse4(const M4& A) {
  const double* m = A.v;  // column-major, but the cofactor formula is transpose-symmetric
  double inv[16];
  inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
  inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
  inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
  inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
  inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
  inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
  inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
  inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
  inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
  inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
  inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
  inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
  inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
  inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
  inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
  inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
  double det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
  double id = 1.0 / det;
  M4 o;
  for (int i = 0; i < 16; i++) o.v[i] = inv[i] * id;
  return o;
}

static M3 inverse3(const M3& a) {
  M3 c;
  c(0, 0) = a(1, 1) * a(2, 2) - a(1, 2) * a(2, 1);
  c(0, 1) = a(0, 2) * a(2, 1) - a(0, 1) * a(2, 2);
  c(0, 2) = a(0, 1) * a(1, 2) - a(0, 2) * a(1, 1);
  c(1, 0) = a(1, 2) * a(2, 0) - a(1, 0) * a(2, 2);
  c(1, 1) = a(0, 0) * a(2, 2) - a(0, 2) * a(2, 0);
  c(1, 2) = a(0, 2) * a(1, 0) - a(0, 0) * a(1, 2);
  c(2, 0) = a(1, 0) * a(2, 1) - a(1, 1) * a(2, 0);
  c(2, 1) = a(0, 1) * a(2, 0) - a(0, 0) * a(2, 1);
  c(2, 2) = a(0, 0) * a(1, 1) - a(0, 1) * a(1, 0);
  double det = a(0, 0) * c(0, 0) + a(0, 1) * c(1, 0) + a(0, 2) * c(2, 0);
  M3 o;
  for (int i = 0; i < 9; i++) o.v[i] = c.v[i] / det;
  return o;
}

// ------------------------------------------------------------------------------------------
// Eigen::JacobiSVD<Matrix3d>(ComputeFullU|ComputeFullV), two-sided Jacobi, restated from the
// published algorithm (SURVEY App. B3).  Used at nano_gicp_impl.hpp:332.
// ------------------------------------------------------------------------------------------
struct Rot { double c, s; };
static Rot rot_mul(Rot a, Rot b) { return Rot{a.c * b.c - a.s * b.s, a.c * b.s + a.s * b.c}; }
static Rot rot_T(Rot a) { return Rot{a.c, -a.s}; }
// x' = c x + s y ; y' = -s x + c y
static void rot_rows(M3& m, int p, int q, Rot j) {
  for (int i = 0; i < 3; i++) { double x = m(p, i), y = m(q, i); m(p, i) = j.c * x + j.s * y; m(q, i) = -j.s * x + j.c * y; }
}
static void rot_cols(M3& m, int p, int q, Rot j) {  // applyOnTheRight(p,q,j): rotation j^T on the column pair
  Rot t = rot_T(j);
  for (int i = 0; i < 3; i++) { double x = m(i, p), y = m(i, q); m(i, p) = t.c * x + t.s * y; m(i, q) = -t.s * x + t.c * y; }
}
static Rot make_jacobi(double x, double y, double z) {
  double deno = 2.0 * std::fabs(y);
  if (deno < DBL_MIN) return Rot{1.0, 0.0};
  double tau = (x - z) / deno;
  double w = std::sqrt(tau * tau + 1.0);
  double t = tau > 0.0 ? 1.0 / (tau + w) : 1.0 / (tau - w);
  double sign_t = t > 0.0 ? 1.0 : -1.0;
  double n = 1.0 / std::sqrt(t * t + 1.0);
  Rot r;
  r.s = -sign_t * (y / std::fabs(y)) * std::fabs(t) * n;
  r.c = n;
  return r;
}
static void real_2x2_jacobi_svd(const M3& W, int p, int q, Rot* jl, Rot* jr) {
  double m00 = W(p, p), m01 = W(p, q), m10 = W(q, p), m11 = W(q, q);
  Rot rot1;
  double t = m00 + m11, d = m10 - m01;
  if (std::fabs(d) < DBL_MIN) { rot1.s = 0.0; rot1.c = 1.0; }
  else { double u = t / d; double tmp = std::sqrt(1.0 + u * u); rot1.s = 1.0 / tmp; rot1.c = u / tmp; }
  // m.applyOnTheLeft(0,1,rot1)
  double a00 = rot1.c * m00 + rot1.s * m10, a01 = rot1.c * m01 + rot1.s * m11;
  double a11 = -rot1.s * m01 + rot1.c * m11;
  *jr = make_jacobi(a00, a01, a11);
  *jl = rot_mul(rot1, rot_T(*jr));
}
static void jacobi_svd3(const M3& A, M3& U, double sv[3], M3& V) {
  double scale = 0.0;
  for (int i = 0; i < 9; i++) scale = std::max(scale, std::fabs(A.v[i]));
  if (scale == 0.0) scale = 1.0;
  M3 W;
  for (int i = 0; i < 9; i++) W.v[i] = A.v[i] / scale;
  U = M3::identity();
  V = M3::identity();
  const double precision = 2.0 * DBL_EPSILON, considerAsZero = DBL_MIN;
  double maxDiag = std::max(std::fabs(W(0, 0)), std::max(std::fabs(W(1, 1)), std::fabs(W(2, 2))));
  bool finished = false;
  int guard = 0;
  while (!finished && guard++ < 1000) {
    finished = true;
    for (int p = 1; p < 3; ++p)
      for (int q = 0; q < p; ++q) {
        double thr = std::max(considerAsZero, precision * maxDiag);
        if (std::fabs(W(p, q)) > thr || std::fabs(W(q, p)) > thr) {
          finished = false;
          Rot jl, jr;
          real_2x2_jacobi_svd(W, p, q, &jl, &jr);
          rot_rows(W, p, q, jl);
          rot_cols(U, p, q, rot_T(jl));
          rot_cols(W, p, q, jr);
          rot_cols(V, p, q, jr);
          maxDiag = std::max(maxDiag, std::max(std::fabs(W(p, p)), std::fabs(W(q, q))));
        }
      }
  }
  for (int i = 0; i < 3; i++) {
    double a = W(i, i);
    sv[i] = std::fabs(a);
    if (a < 0.0) for (int r = 0; r < 3; r++) U(r, i) = -U(r, i);
  }
  for (int i = 0; i < 3; i++) sv[i] *= scale;
  for (int i = 0; i < 3; i++) {
    int pos = i;
    for (int j = i + 1; j < 3; j++) if (sv[j] > sv[pos]) pos = j;
    if (sv[pos] == 0.0) break;
    if (pos != i) {
      std::swap(sv[i], sv[pos]);
      for (int r = 0; r < 3; r++) { std::swap(U(r, i), U(r, pos)); std::swap(V(r, i), V(r, pos)); }
    }
  }
}

// ------------------------------------------------------------------------------------------
// Eigen::LDLT<Matrix<double,6,6>> (lower, symmetric pivoting on the largest remaining diagonal)
// and its solve, restated (SURVEY App. B5).  Used at lsq_registration_impl.hpp:147,172.
// ------------------------------------------------------------------------------------------
static V6 ldlt6_solve(const M6& Ain, const V6& rhs) {
  const int n = 6;
  M6 A = Ain;
  int perm[6];
  for (int k = 0; k < n; k++) {
    int piv = k;
    double big = std::fabs(A(k, k));
    for (int i = k + 1; i < n; i++) if (std::fabs(A(i, i)) > big) { big = std::fabs(A(i, i)); piv = i; }
    perm[k] = piv;
    if (piv != k) {
      // symmetric swap of rows/cols k and piv, touching only the lower triangle
      for (int j = 0; j < k; j++) std::swap(A(k, j), A(piv, j));
      for (int i = piv + 1; i < n; i++) std::swap(A(i, k), A(i, piv));
      std::swap(A(k, k), A(piv, piv));
      for (int i = k + 1; i < piv; i++) std::swap(A(i, k), A(piv, i));
    }
    // A(k,k) -= sum_j L(k,j)^2 D_j ; column update
    if (k > 0) {
      double tmp[6];
      for (int j = 0; j < k; j++) tmp[j] = A(j, j) * A(k, j);
      double s = 0.0;
      for (int j = 0; j < k; j++) s += A(k, j) * tmp[j];
      A(k, k) -= s;
      for (int i = k + 1; i < n; i++) {
        double t = 0.0;
        for (int j = 0; j < k; j++) t += A(i, j) * tmp[j];
        A(i, k) -= t;
      }
    }
    double d = A(k, k);
    if (std::fabs(d) > 0.0)
      for (int i = k + 1; i < n; i++) A(i, k) /= d;
  }
  // solve: x = P^T L^-T D^-1 L^-1 P b
  double x[6];
  for (int i = 0; i < n; i++) x[i] = rhs.v[i];
  for (int k = 0; k < n; k++) std::swap(x[k], x[perm[k]]);
  for (int i = 0; i < n; i++) for (int j = 0; j < i; j++) x[i] -= A(i, j) * x[j];
  const double tol = 1.0 / DBL_MAX;
  for (int i = 0; i < n; i++) x[i] = std::fabs(A(i, i)) > tol ? x[i] / A(i, i) : 0.0;
  for (int i = n - 1; i >= 0; i--) for (int j = i + 1; j < n; j++) x[i] -= A(j, i) * x[j];
  for (int k = n - 1; k >= 0; k--) std::swap(x[k], x[perm[k]]);
  V6 o;
  for (int i = 0; i < n; i++) o.v[i] = x[i];
  return o;
}

// so3_exp (gicp/so3.hpp:99-118) followed by Quaterniond::toRotationMatrix (SURVEY App. B7)
static M3 so3_exp_matrix(double ox, double oy, double oz) {
  double theta_sq = ox * ox + oy * oy + oz * oz;
  double imag_factor, real_factor;
  if (theta_sq < 1e-10) {
    double theta_quad = theta_sq * theta_sq;
    imag_factor = 0.5 - 1.0 / 48.0 * theta_sq + 1.0 / 3840.0 * theta_quad;
    real_factor = 1.0 - 1.0 / 8.0 * theta_sq + 1.0 / 384.0 * theta_quad;
  } else {
    double theta = std::sqrt(theta_sq);
    double half_theta = 0.5 * theta;
    imag_factor = std::sin(half_theta) / theta;
    real_factor = std::cos(half_theta);
  }
  double w = real_factor, x = imag_factor * ox, y = imag_factor * oy, z = imag_factor * oz;
  double tx = 2.0 * x, ty = 2.0 * y, tz = 2.0 * z;
  double twx = tx * w, twy = ty * w, twz = tz * w;
  double txx = tx * x, txy = ty * x, txz = tz * x;
  double tyy = ty * y, tyz = tz * y, tzz = tz * z;
  M3 R;
  R(0, 0) = 1.0 - (tyy + tzz); R(0, 1) = txy - twz;         R(0, 2) = txz + twy;
  R(1, 0) = txy + twz;         R(1, 1) = 1.0 - (txx + tzz); R(1, 2) = tyz - twx;
  R(2, 0) = txz - twy;         R(2, 1) = tyz + twx;         R(2, 2) = 1.0 - (txx + tyy);
  return R;
}

// ------------------------------------------------------------------------------------------
// kNN index interface + two backends
// ------------------------------------------------------------------------------------------
struct CloudView {
  const float* base = nullptr;  // first float of point 0
  size_t n = 0;
  size_t stride = 8;            // floats between consecutive points (8 for pcl::PointXYZI)
  inline const float* pt(size_t i) const { return base + i * stride; }
};

struct KnnIndex {
  virtual ~KnnIndex() {}
  // returns number found (== min(k, n)); idx/d2 ascending by distance
  virtual int knn(const float* q, int k, int* idx, float* d2) const = 0;
};

// nanoflann KNNResultSet semantics (nanoflann_impl.hpp:149-214): insertion keeps the earlier
// visited entry first on exact ties (strict '>' shift test), worst = dists[capacity-1].
struct ResultSet {
  int* indices; float* dists; int capacity; int count;
  ResultSet(int cap, int* i, float* d) : indices(i), dists(d), capacity(cap), count(0) {
    if (capacity) dists[capacity - 1] = std::numeric_limits<float>::max();
  }
  inline float worst() const { return dists[capacity - 1]; }
  inline void add(float dist, int index) {
    int i;
    for (i = count; i > 0; --i) {
      if (dists[i - 1] > dist) {
        if (i < capacity) { dists[i] = dists[i - 1]; indices[i] = indices[i - 1]; }
      } else break;
    }
    if (i < capacity) { dists[i] = dist; indices[i] = index; }
    if (count < capacity) count++;
  }
};

// Restated single-index kd-tree (same split rule, same traversal order, same float bounds as
// nanoflann v1.3.2 so that results — including which of two equidistant points wins — agree
// with the reference build).  Own data layout: flat node array + flat permutation.
class RestatedKdTree : public KnnIndex {
 public:
  RestatedKdTree(const CloudView& c, int leaf_max = 100) : cloud_(c), leaf_max_(leaf_max) {
    const size_t n = c.n;
    order_.resize(n);
    for (size_t i = 0; i < n; i++) order_[i] = (int)i;
    root_ = -1;
    if (n == 0) return;
    for (int d = 0; d < 3; d++) lo_[d] = hi_[d] = coord(0, d);
    for (size_t k = 1; k < n; k++)
      for (int d = 0; d < 3; d++) {
        float v = coord(k, d);
        if (v < lo_[d]) lo_[d] = v;
        if (v > hi_[d]) hi_[d] = v;
      }
    nodes_.reserve(2 * n / (size_t)leaf_max_ + 16);
    float blo[3] = {lo_[0], lo_[1], lo_[2]}, bhi[3] = {hi_[0], hi_[1], hi_[2]};
    root_ = build(0, (int)n, blo, bhi);
    for (int d = 0; d < 3; d++) { lo_[d] = blo[d]; hi_[d] = bhi[d]; }
  }

  int knn(const float* q, int k, int* idx, float* d2) const override {
    ResultSet rs(k, idx, d2);
    if (cloud_.n == 0) return 0;
    float side[3] = {0.f, 0.f, 0.f};
    float dsq = 0.f;
    for (int d = 0; d < 3; d++) {
      if (q[d] < lo_[d]) { side[d] = (q[d] - lo_[d]) * (q[d] - lo_[d]); dsq += side[d]; }
      if (q[d] > hi_[d]) { side[d] = (q[d] - hi_[d]) * (q[d] - hi_[d]); dsq += side[d]; }
    }
    descend(rs, q, root_, dsq, side);
    return rs.count;
  }

 private:
  struct Node { int child1, child2; int a, b; int feat; float divlow, divhigh; };
  CloudView cloud_;
  int leaf_max_;
  std::vector<int> order_;
  std::vector<Node> nodes_;
  int root_;
  float lo_[3], hi_[3];

  inline float coord(size_t i, int d) const { return cloud_.pt(i)[d]; }

  void minmax(const int* ind, int count, int d, float& mn, float& mx) const {
    mn = mx = coord(ind[0], d);
    for (int i = 1; i < count; i++) {
      float v = coord(ind[i], d);
      if (v < mn) mn = v;
      if (v > mx) mx = v;
    }
  }

  // three-way partition around cutval along dimension d: [<cut | ==cut | >cut]
  void partition(int* ind, int count, int d, float cutval, int& lim1, int& lim2) const {
    int left = 0, right = count - 1;
    for (;;) {
      while (left <= right && coord(ind[left], d) < cutval) ++left;
      while (right && left <= right && coord(ind[right], d) >= cutval) --right;
      if (left > right || !right) break;
      std::swap(ind[left], ind[right]);
      ++left; --right;
    }
    lim1 = left;
    right = count - 1;
    for (;;) {
      while (left <= right && coord(ind[left], d) <= cutval) ++left;
      while (right && left <= right && coord(ind[right], d) > cutval) --right;
      if (left > right || !right) break;
      std::swap(ind[left], ind[right]);
      ++left; --right;
    }
    lim2 = left;
  }

  int build(int left, int right, float* blo, float* bhi) {
    int me = (int)nodes_.size();
    nodes_.push_back(Node());
    if ((right - left) <= leaf_max_) {
      Node nd; nd.child1 = nd.child2 = -1; nd.a = left; nd.b = right; nd.feat = 0; nd.divlow = nd.divhigh = 0.f;
      for (int d = 0; d < 3; d++) blo[d] = bhi[d] = coord(order_[left], d);
      for (int k = left + 1; k < right; k++)
        for (int d = 0; d < 3; d++) {
          float v = coord(order_[k], d);
          if (blo[d] > v) blo[d] = v;
          if (bhi[d] < v) bhi[d] = v;
        }
      nodes_[me] = nd;
      return me;
    }
    int* ind = order_.data() + left;
    const int count = right - left;
    // choose the cut dimension: among dims whose bbox span is within (1-1e-5) of the widest,
    // the one with the largest actual spread of the points
    const float EPS = 0.00001f;
    float max_span = bhi[0] - blo[0];
    for (int d = 1; d < 3; d++) { float s = bhi[d] - blo[d]; if (s > max_span) max_span = s; }
    float max_spread = -1.f;
    int cutfeat = 0;
    for (int d = 0; d < 3; d++) {
      float s = bhi[d] - blo[d];
      if (s > (1 - EPS) * max_span) {
        float mn, mx;
        minmax(ind, count, d, mn, mx);
        float spread = mx - mn;
        if (spread > max_spread) { cutfeat = d; max_spread = spread; }
      }
    }
    float split_val = (blo[cutfeat] + bhi[cutfeat]) / 2;
    float mn, mx;
    minmax(ind, count, cutfeat, mn, mx);
    float cutval;
    if (split_val < mn) cutval = mn;
    else if (split_val > mx) cutval = mx;
    else cutval = split_val;
    int lim1, lim2, idx;
    partition(ind, count, cutfeat, cutval, lim1, lim2);
    if (lim1 > count / 2) idx = lim1;
    else if (lim2 < count / 2) idx = lim2;
    else idx = count / 2;

    float llo[3] = {blo[0], blo[1], blo[2]}, lhi[3] = {bhi[0], bhi[1], bhi[2]};
    lhi[cutfeat] = cutval;
    int c1 = build(left, left + idx, llo, lhi);
    float rlo[3] = {blo[0], blo[1], blo[2]}, rhi[3] = {bhi[0], bhi[1], bhi[2]};
    rlo[cutfeat] = cutval;
    int c2 = build(left + idx, right, rlo, rhi);
    Node nd; nd.child1 = c1; nd.child2 = c2; nd.a = nd.b = 0; nd.feat = cutfeat;
    nd.divlow = lhi[cutfeat];
    nd.divhigh = rlo[cutfeat];
    nodes_[me] = nd;
    for (int d = 0; d < 3; d++) { blo[d] = std::min(llo[d], rlo[d]); bhi[d] = std::max(lhi[d], rhi[d]); }
    return me;
  }

  void descend(ResultSet& rs, const float* q, int ni, float mindistsq, float* side) const {
    const Node& nd = nodes_[ni];
    if (nd.child1 < 0 && nd.child2 < 0) {
      float worst = rs.worst();  // captured once per leaf, like the reference
      for (int i = nd.a; i < nd.b; ++i) {
        const int index = order_[i];
        const float* p = cloud_.pt(index);
        float dist = 0.f;
        for (int d = 0; d < 3; d++) { const float diff = q[d] - p[d]; dist += diff * diff; }
        if (dist < worst) rs.add(dist, index);
      }
      return;
    }
    int f = nd.feat;
    float val = q[f];
    float diff1 = val - nd.divlow, diff2 = val - nd.divhigh;
    int best, other;
    float cut;
    if ((diff1 + diff2) < 0) { best = nd.child1; other = nd.child2; cut = (val - nd.divhigh) * (val - nd.divhigh); }
    else { best = nd.child2; other = nd.child1; cut = (val - nd.divlow) * (val - nd.divlow); }
    descend(rs, q, best, mindistsq, side);
    float saved = side[f];
    mindistsq = mindistsq + cut - saved;
    side[f] = cut;
    if (mindistsq * 1.0f <= rs.worst()) descend(rs, q, other, mindistsq, side);
    side[f] = saved;
  }
};

#ifdef ORACLE_WITH_REF_NANOFLANN
// The reference's own kd-tree, instantiated exactly as include/nano_gicp/nanoflann.hpp:100-117 does
// (SO3_Adaptor<float>, DIM=3, int index, leaf_max_size 100).
struct RefAdaptor {
  CloudView c;
  inline size_t kdtree_get_point_count() const { return c.n; }
  inline float kdtree_get_pt(const size_t idx, int dim) const { return c.pt(idx)[dim]; }
  template <class BBOX> bool kdtree_get_bbox(BBOX&) const { return false; }
};
class RefNanoflannTree : public KnnIndex {
  typedef nanoflann::KDTreeSingleIndexAdaptor<nanoflann::SO3_Adaptor<float, RefAdaptor>, RefAdaptor, 3, int> Tree;
  RefAdaptor ad_;
  std::unique_ptr<Tree> tree_;
 public:
  RefNanoflannTree(const CloudView& c) {
    ad_.c = c;
    tree_.reset(new Tree(3, ad_, nanoflann::KDTreeSingleIndexAdaptorParams(100)));
    tree_->buildIndex();
  }
  int knn(const float* q, int k, int* idx, float* d2) const override {
    if (ad_.c.n == 0) return 0;
    nanoflann::KNNResultSet<float, int> rs(k);
    rs.init(idx, d2);
    tree_->findNeighbors(rs, q, nanoflann::SearchParams());
    return (int)rs.size();
  }
};
#endif

// brute force with the same float metric; ties resolved towards the lower index
class BruteForce : public KnnIndex {
  CloudView c_;
 public:
  BruteForce(const CloudView& c) : c_(c) {}
  int knn(const float* q, int k, int* idx, float* d2) const override {
    ResultSet rs(k, idx, d2);
    for (size_t i = 0; i < c_.n; i++) {
      const float* p = c_.pt(i);
      float dist = 0.f;
      for (int d = 0; d < 3; d++) { const float diff = q[d] - p[d]; dist += diff * diff; }
      if (dist < rs.worst()) rs.add(dist, (int)i);
    }
    return rs.count;
  }
};

enum Backend { BACKEND_DEFAULT = 0, BACKEND_RESTATED = 1, BACKEND_REF = 2, BACKEND_BRUTE = 3 };

static KnnIndex* make_index(const CloudView& c, int backend) {
  if (backend == BACKEND_BRUTE) return new BruteForce(c);
#ifdef ORACLE_WITH_REF_NANOFLANN
  if (backend == BACKEND_REF || backend == BACKEND_DEFAULT) return new RefNanoflannTree(c);
#else
  if (backend == BACKEND_REF) return nullptr;
#endif
  return new RestatedKdTree(c);
}

// a cloud owned by the oracle: copies the caller's records (stride preserved) + its index
struct Cloud {
  std::vector<float> data;
  CloudView view;
  std::unique_ptr<KnnIndex> index;
  Cloud(const float* pts, size_t n, size_t stride, int backend, bool build_index) {
    data.assign(pts, pts + n * stride);
    view.base = data.data(); view.n = n; view.stride = stride;
    if (build_index) index.reset(make_index(view, backend));
  }
};

// ------------------------------------------------------------------------------------------
// covariances — nano_gicp_impl.hpp:298-357
// ------------------------------------------------------------------------------------------
enum RegMethod { REG_NONE = 0, REG_MIN_EIG = 1, REG_NORMALIZED_MIN_EIG = 2, REG_PLANE = 3, REG_FROBENIUS = 4 };

static int calc_covariances(const Cloud& cloud, int k, int method, int nthreads, double* out /* n x 16 col-major */,
                            int* knn_idx_out /* optional n x k */, float* knn_d2_out /* optional */) {
  const int n = (int)cloud.view.n;
  if (!cloud.index) return -2;
  if (n < k) return -3;  // the reference reads uninitialised columns here (UB, :315-318)
#pragma omp parallel for num_threads(nthreads) schedule(guided, 8)
  for (int i = 0; i < n; i++) {
    std::vector<int> k_indices(k);
    std::vector<float> k_sq(k);
    int found = cloud.index->knn(cloud.view.pt(i), k, k_indices.data(), k_sq.data());
    if (knn_idx_out) for (int j = 0; j < k; j++) { knn_idx_out[(size_t)i * k + j] = j < found ? k_indices[j] : -1; knn_d2_out[(size_t)i * k + j] = j < found ? k_sq[j] : -1.f; }
    std::vector<double> nb(4 * (size_t)k, 0.0);
    for (int j = 0; j < found; j++) {
      const float* p = cloud.view.pt(k_indices[j]);
      for (int r = 0; r < 4; r++) nb[4 * j + r] = (double)p[r];
    }
    double mean[4] = {0, 0, 0, 0};
    for (int j = 0; j < k; j++) for (int r = 0; r < 4; r++) mean[r] += nb[4 * j + r];
    for (int r = 0; r < 4; r++) mean[r] /= (double)k;
    for (int j = 0; j < k; j++) for (int r = 0; r < 4; r++) nb[4 * j + r] -= mean[r];
    M4 cov;
    for (int r = 0; r < 4; r++)
      for (int c = 0; c < 4; c++) {
        double s = 0.0;
        for (int j = 0; j < k; j++) s += nb[4 * j + r] * nb[4 * j + c];
        cov(r, c) = s / (double)k;
      }
    M4 res;
    if (method == REG_NONE) {
      res = cov;
    } else if (method == REG_FROBENIUS) {
      const double lambda = 1e-3;
      M3 C;
      for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) C(r, c) = cov(r, c) + (r == c ? lambda : 0.0);
      M3 Ci = inverse3(C);
      double nrm = 0.0;
      for (int t = 0; t < 9; t++) nrm += Ci.v[t] * Ci.v[t];
      nrm = std::sqrt(nrm);
      M3 Cn;
      for (int t = 0; t < 9; t++) Cn.v[t] = Ci.v[t] / nrm;
      M3 R = inverse3(Cn);
      for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) res(r, c) = R(r, c);
    } else {
      M3 C, U, V;
      for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) C(r, c) = cov(r, c);
      double sv[3];
      jacobi_svd3(C, U, sv, V);
      double values[3];
      if (method == REG_PLANE) { values[0] = 1.0; values[1] = 1.0; values[2] = 1e-3; }
      else if (method == REG_MIN_EIG) { for (int t = 0; t < 3; t++) values[t] = std::max(sv[t], 1e-3); }
      else { double mx = std::max(sv[0], std::max(sv[1], sv[2])); for (int t = 0; t < 3; t++) values[t] = std::max(sv[t] / mx, 1e-3); }
      M3 UD = U;
      for (int c = 0; c < 3; c++) for (int r = 0; r < 3; r++) UD(r, c) = U(r, c) * values[c];
      M3 R = mul(UD, tr(V));
      for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) res(r, c) = R(r, c);
    }
    std::memcpy(out + (size_t)i * 16, res.v, sizeof(double) * 16);
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// the registration object — NanoGICP + LsqRegistration state
// ------------------------------------------------------------------------------------------
struct Params {
  int k_correspondences = 20;                 // nano_gicp_impl.hpp:57
  double corr_dist_threshold = (double)FLT_MAX;  // :59
  int regularization = REG_PLANE;             // :61
  int max_iterations = 64;                    // lsq_registration_impl.hpp:52
  double rotation_epsilon = 2e-3;             // :53
  double transformation_epsilon = 5e-4;       // :54
  int optimizer = 1;                          // 1 = LevenbergMarquardt (:56), 0 = GaussNewton
  int lm_max_iterations = 10;                 // :58
  double lm_init_lambda_factor = 1e-9;        // :59
  int num_threads = 1;
  int backend = BACKEND_DEFAULT;
};

struct Iso { M3 R; double t[3]; };  // Eigen::Isometry3d
static M4 iso_matrix(const Iso& x) {
  M4 m;
  for (int r = 0; r < 3; r++) { for (int c = 0; c < 3; c++) m(r, c) = x.R(r, c); m(r, 3) = x.t[r]; }
  m(3, 3) = 1.0;
  return m;
}
static Iso iso_from16(const double* T) {
  Iso x;
  for (int r = 0; r < 3; r++) { for (int c = 0; c < 3; c++) x.R(r, c) = T[c * 4 + r]; x.t[r] = T[12 + r]; }
  return x;
}
static Iso iso_mul(const Iso& a, const Iso& b) {
  Iso o;
  o.R = mul(a.R, b.R);
  for (int r = 0; r < 3; r++) o.t[r] = a.R(r, 0) * b.t[0] + a.R(r, 1) * b.t[1] + a.R(r, 2) * b.t[2] + a.t[r];
  return o;
}

struct AlignResult {
  float final_transformation[16];
  double final_x[16];
  double final_hessian[36];
  double lm_lambda;
  double last_error;
  int nr_iterations;
  int converged;
  int n_linearize;
  int n_compute_error;
  int lm_failed;
  int reserved;
};

struct Gicp {
  Params prm;
  std::shared_ptr<Cloud> source, target;
  std::vector<M4> source_covs, target_covs;
  std::vector<M4> mahalanobis;
  std::vector<int> correspondences;
  std::vector<float> sq_distances;
  double lm_lambda = -1.0;
  M6 final_hessian = M6::identity();
  int n_linearize = 0, n_compute_error = 0;

  // nano_gicp_impl.hpp:173-211
  void update_correspondences(const Iso& trans) {
    const int n = (int)source->view.n;
    float tf[16];
    M4 tm = iso_matrix(trans);
    for (int i = 0; i < 16; i++) tf[i] = (float)tm.v[i];
    correspondences.assign(n, -1);
    sq_distances.assign(n, 0.f);
    mahalanobis.resize(n);
    const double thr2 = prm.corr_dist_threshold * prm.corr_dist_threshold;
    M4 tmT = tr(tm);
#pragma omp parallel for num_threads(prm.num_threads) schedule(guided, 8)
    for (int i = 0; i < n; i++) {
      const float* p = source->view.pt(i);
      float q[4];
      // Isometry3f * Vector4f: per-row balanced-tree sum, float, unfused (SURVEY App. B6)
      for (int r = 0; r < 3; r++) {
        float a = tf[0 * 4 + r] * p[0], b = tf[1 * 4 + r] * p[1], c = tf[2 * 4 + r] * p[2], d = tf[3 * 4 + r] * p[3];
        q[r] = (a + b) + (c + d);
      }
      q[3] = p[3];
      int ki; float kd;
      target->index->knn(q, 1, &ki, &kd);
      sq_distances[i] = kd;
      correspondences[i] = ((double)kd < thr2) ? ki : -1;
      if (correspondences[i] < 0) continue;
      const M4& cov_A = source_covs[i];
      const M4& cov_B = target_covs[ki];
      M4 RCR = add(cov_B, mul(mul(tm, cov_A), tmT));
      RCR(3, 3) = 1.0;
      M4 Mi = inverse4(RCR);
      Mi(3, 3) = 0.0;
      mahalanobis[i] = Mi;
    }
  }

  // nano_gicp_impl.hpp:213-270 (H,b may be null) and :272-296
  double accumulate(const Iso& trans, M6* H, V6* b) {
    const int n = (int)source->view.n;
    const int nt = std::max(1, prm.num_threads);
    std::vector<M6> Hs(nt);
    std::vector<V6> bs(nt);
    double sum_errors = 0.0;
#pragma omp parallel for num_threads(nt) reduction(+ : sum_errors) schedule(guided, 8)
    for (int i = 0; i < n; i++) {
      int ti = correspondences[i];
      if (ti < 0) continue;
      const float* pa = source->view.pt(i);
      const float* pb = target->view.pt(ti);
      double mean_A[4] = {(double)pa[0], (double)pa[1], (double)pa[2], (double)pa[3]};
      double mean_B[4] = {(double)pb[0], (double)pb[1], (double)pb[2], (double)pb[3]};
      double tA[4];
      for (int r = 0; r < 3; r++) tA[r] = trans.R(r, 0) * mean_A[0] + trans.R(r, 1) * mean_A[1] + trans.R(r, 2) * mean_A[2] + trans.t[r] * mean_A[3];
      tA[3] = mean_A[3];
      V4 e;
      for (int r = 0; r < 4; r++) e.v[r] = mean_B[r] - tA[r];
      const M4& Mi = mahalanobis[i];
      V4 Me = mul(Mi, e);
      sum_errors += e.v[0] * Me.v[0] + e.v[1] * Me.v[1] + e.v[2] * Me.v[2] + e.v[3] * Me.v[3];
      if (!H || !b) continue;
      Mat<4, 6> J;
      // skewd(transed_mean_A.head<3>()) | -I
      J(0, 1) = -tA[2]; J(0, 2) = tA[1];
      J(1, 0) = tA[2];  J(1, 2) = -tA[0];
      J(2, 0) = -tA[1]; J(2, 1) = tA[0];
      J(0, 3) = -1.0; J(1, 4) = -1.0; J(2, 5) = -1.0;
      Mat<6, 4> Jt = tr(J);
      M6 Hi = mul(mul(Jt, Mi), J);
      V6 bi = mul(mul(Jt, Mi), e);
#ifdef _OPENMP
      int th = omp_get_thread_num();
#else
      int th = 0;
#endif
      Hs[th] = add(Hs[th], Hi);
      bs[th] = add(bs[th], bi);
    }
    if (H && b) {
      *H = M6(); *b = V6();
      for (int t = 0; t < nt; t++) { *H = add(*H, Hs[t]); *b = add(*b, bs[t]); }
    }
    return sum_errors;
  }

  double linearize(const Iso& trans, M6* H, V6* b) {
    n_linearize++;
    update_correspondences(trans);
    return accumulate(trans, H, b);
  }
  double compute_error(const Iso& trans) {
    n_compute_error++;
    return accumulate(trans, nullptr, nullptr);
  }

  // lsq_registration_impl.hpp:118-127
  bool is_converged(const Iso& delta) const {
    double rmax = 0.0, tmax = 0.0;
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) rmax = std::max(rmax, 1.0 / prm.rotation_epsilon * std::fabs(delta.R(r, c) - (r == c ? 1.0 : 0.0)));
    for (int r = 0; r < 3; r++) tmax = std::max(tmax, 1.0 / prm.transformation_epsilon * std::fabs(delta.t[r]));
    return std::max(rmax, tmax) < 1;
  }

  static Iso delta_from(const V6& d) {
    Iso delta;
    delta.R = so3_exp_matrix(d.v[0], d.v[1], d.v[2]);
    delta.t[0] = d.v[3]; delta.t[1] = d.v[4]; delta.t[2] = d.v[5];
    return delta;
  }

  // lsq_registration_impl.hpp:141-158
  bool step_gn(Iso& x0, Iso& delta) {
    M6 H; V6 b;
    linearize(x0, &H, &b);
    V6 nb; for (int i = 0; i < 6; i++) nb.v[i] = -b.v[i];
    V6 d = ldlt6_solve(H, nb);
    delta = delta_from(d);
    x0 = iso_mul(delta, x0);
    final_hessian = H;
    return true;
  }

  // lsq_registration_impl.hpp:160-208
  bool step_lm(Iso& x0, Iso& delta, double* y0_out) {
    M6 H; V6 b;
    double y0 = linearize(x0, &H, &b);
    *y0_out = y0;
    if (lm_lambda < 0.0) {
      double mx = 0.0;
      for (int i = 0; i < 6; i++) mx = std::max(mx, std::fabs(H(i, i)));
      lm_lambda = prm.lm_init_lambda_factor * mx;
    }
    double nu = 2.0;
    for (int i = 0; i < prm.lm_max_iterations; i++) {
      M6 A = H;
      for (int t = 0; t < 6; t++) A(t, t) += lm_lambda;
      V6 nb; for (int t = 0; t < 6; t++) nb.v[t] = -b.v[t];
      V6 d = ldlt6_solve(A, nb);
      delta = delta_from(d);
      Iso xi = iso_mul(delta, x0);
      double yi = compute_error(xi);
      double denom = 0.0;
      for (int t = 0; t < 6; t++) denom += d.v[t] * (lm_lambda * d.v[t] - b.v[t]);
      double rho = (y0 - yi) / denom;
      if (rho < 0) {
        if (is_converged(delta)) return true;
        lm_lambda = nu * lm_lambda;
        nu = 2 * nu;
        continue;
      }
      x0 = xi;
      lm_lambda = lm_lambda * std::max(1.0 / 3.0, 1 - std::pow(2 * rho - 1, 3));
      final_hessian = H;
      return true;
    }
    return false;
  }

  // lsq_registration_impl.hpp:89-115 (+ lazy covariances, nano_gicp_impl.hpp:161-171)
  int align(const float* guess16, AlignResult* res) {
    if (!source || !target || !target->index) return -2;
    if (source_covs.size() != source->view.n) {
      if (!source->index) return -2;
      std::vector<double> tmp(source->view.n * 16);
      int rc = calc_covariances(*source, prm.k_correspondences, prm.regularization, prm.num_threads, tmp.data(), nullptr, nullptr);
      if (rc) return rc;
      source_covs.resize(source->view.n);
      for (size_t i = 0; i < source->view.n; i++) std::memcpy(source_covs[i].v, &tmp[i * 16], 128);
    }
    if (target_covs.size() != target->view.n) {
      std::vector<double> tmp(target->view.n * 16);
      int rc = calc_covariances(*target, prm.k_correspondences, prm.regularization, prm.num_threads, tmp.data(), nullptr, nullptr);
      if (rc) return rc;
      target_covs.resize(target->view.n);
      for (size_t i = 0; i < target->view.n; i++) std::memcpy(target_covs[i].v, &tmp[i * 16], 128);
    }
    double g[16];
    for (int i = 0; i < 16; i++) g[i] = (double)guess16[i];
    Iso x0 = iso_from16(g);
    lm_lambda = -1.0;
    n_linearize = n_compute_error = 0;
    bool converged = false;
    int nr_iterations = 0, lm_failed = 0;
    double y0 = 0.0;
    for (int i = 0; i < prm.max_iterations && !converged; i++) {
      nr_iterations = i;
      Iso delta;
      bool ok = prm.optimizer == 1 ? step_lm(x0, delta, &y0) : step_gn(x0, delta);
      if (!ok) { lm_failed = 1; break; }
      converged = is_converged(delta);
    }
    M4 xm = iso_matrix(x0);
    for (int i = 0; i < 16; i++) { res->final_x[i] = xm.v[i]; res->final_transformation[i] = (float)xm.v[i]; }
    std::memcpy(res->final_hessian, final_hessian.v, sizeof(double) * 36);
    res->lm_lambda = lm_lambda;
    res->last_error = y0;
    res->nr_iterations = nr_iterations;
    res->converged = converged ? 1 : 0;
    res->n_linearize = n_linearize;
    res->n_compute_error = n_compute_error;
    res->lm_failed = lm_failed;
    res->reserved = 0;
    return 0;
  }
};

// ------------------------------------------------------------------------------------------
// pcl::VoxelGrid<PointXYZI>::applyFilter restated (SURVEY App. B1).  Within-voxel accumulation
// order is fixed to ascending input index (PCL's own sort is unstable => implementation-defined).
// Voxel indices are sorted as PCL's cloud_point_index_idx::idx is: unsigned int.
// returns 0 ok, 1 = index would overflow int32 (PCL warns and passes the input through)
//
// Deviation from PCL: its guard only tests dx*dy*dz > INT32_MAX, in int64 that can itself wrap.  Here (and in the
// GPU kernels, csrc/voxel.cu vox_grid_setup) the cloud also passes through where PCL's arithmetic is undefined or
// wraps distinct voxels together: an axis extent (max - min) * inv that is not finite or >= 2^31; floor(min * inv) or
// floor(max * inv) outside int32, or div_b beyond INT32_MAX; floor(max * inv) - (float)min_b rounding past
// max_b - min_b; a div_b product >= 2^32.  Everywhere else the result is PCL's.
// ------------------------------------------------------------------------------------------
static int voxel_grid_setup(const float mn[3], const float mx[3], float inv, int min_b[3], int div_b[3]) {
  int64_t dxyz = 1;
  uint64_t cells = 1;
  for (int d = 0; d < 3; d++) {
    const float ext = (mx[d] - mn[d]) * inv;
    if (!(ext < 2147483648.f)) return 1;
    dxyz *= (int64_t)ext + 1;
    if (dxyz > (int64_t)INT32_MAX) return 1;
    const float flo = std::floor(mn[d] * inv), fhi = std::floor(mx[d] * inv);
    if (!(flo >= -2147483648.f) || !(fhi < 2147483648.f)) return 1;
    const int64_t span = (int64_t)fhi - (int64_t)flo;
    const float fspan = fhi - flo;
    if (span >= (int64_t)INT32_MAX || (int64_t)fspan > span) return 1;
    cells *= (uint64_t)(span + 1);
    if (cells >= (1ull << 32)) return 1;
    min_b[d] = (int)flo;
    div_b[d] = (int)(span + 1);
  }
  return 0;
}

static int voxel_filter(const float* pts, size_t n, size_t stride, float leaf, float* out, size_t* m_out,
                        int* voxel_of_point /* optional, n ints: output slot per input point, -1 if skipped */) {
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  size_t finite = 0;
  for (size_t i = 0; i < n; i++) {
    const float* p = pts + i * stride;
    if (!std::isfinite(p[0]) || !std::isfinite(p[1]) || !std::isfinite(p[2])) continue;
    finite++;
    for (int d = 0; d < 3; d++) { mn[d] = std::min(mn[d], p[d]); mx[d] = std::max(mx[d], p[d]); }
  }
  if (finite == 0) { *m_out = 0; return 0; }
  const float inv = 1.0f / leaf;
  int min_b[3], div_b[3];
  if (voxel_grid_setup(mn, mx, inv, min_b, div_b)) {
    for (size_t i = 0; i < n; i++) std::memcpy(out + i * 8, pts + i * stride, 32);
    *m_out = n;
    return 1;
  }
  const uint32_t mul0 = 1, mul1 = (uint32_t)div_b[0], mul2 = (uint32_t)div_b[0] * (uint32_t)div_b[1];
  struct Rec { uint32_t idx; int pt; };
  std::vector<Rec> recs;
  recs.reserve(n);
  for (size_t i = 0; i < n; i++) {
    const float* p = pts + i * stride;
    if (!std::isfinite(p[0]) || !std::isfinite(p[1]) || !std::isfinite(p[2])) continue;
    int i0 = (int)(std::floor(p[0] * inv) - (float)min_b[0]);
    int i1 = (int)(std::floor(p[1] * inv) - (float)min_b[1]);
    int i2 = (int)(std::floor(p[2] * inv) - (float)min_b[2]);
    recs.push_back(Rec{(uint32_t)i0 * mul0 + (uint32_t)i1 * mul1 + (uint32_t)i2 * mul2, (int)i});
  }
  std::stable_sort(recs.begin(), recs.end(), [](const Rec& a, const Rec& b) { return a.idx < b.idx; });
  if (voxel_of_point) for (size_t i = 0; i < n; i++) voxel_of_point[i] = -1;
  size_t m = 0;
  size_t i = 0;
  while (i < recs.size()) {
    size_t j = i;
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
    while (j < recs.size() && recs[j].idx == recs[i].idx) {
      const float* p = pts + (size_t)recs[j].pt * stride;
      sx += p[0]; sy += p[1]; sz += p[2]; si += p[4];
      if (voxel_of_point) voxel_of_point[recs[j].pt] = (int)m;
      ++j;
    }
    const float cnt = (float)(j - i);
    float* o = out + m * 8;
    o[0] = sx / cnt; o[1] = sy / cnt; o[2] = sz / cnt; o[3] = 1.0f;
    o[4] = si / cnt; o[5] = o[6] = o[7] = 0.f;
    ++m;
    i = j;
  }
  *m_out = m;
  return 0;
}

}  // namespace orc

// ------------------------------------------------------------------------------------------
// C ABI (driven from Python by oracle/oracle.py)
// ------------------------------------------------------------------------------------------
extern "C" {

int orc_has_ref_nanoflann() {
#ifdef ORACLE_WITH_REF_NANOFLANN
  return 1;
#else
  return 0;
#endif
}

int orc_max_threads() {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

int orc_voxel_filter(const float* pts, size_t n, size_t stride_floats, float leaf, float* out, size_t* m, int* voxel_of_point) {
  return orc::voxel_filter(pts, n, stride_floats, leaf, out, m, voxel_of_point);
}

void* orc_cloud_create(const float* pts, size_t n, size_t stride_floats, int backend, int build_index) {
  auto* c = new std::shared_ptr<orc::Cloud>(new orc::Cloud(pts, n, stride_floats, backend, build_index != 0));
  if (build_index && !(*c)->index) { delete c; return nullptr; }
  return c;
}
void orc_cloud_destroy(void* c) { delete (std::shared_ptr<orc::Cloud>*)c; }

int orc_cloud_knn(void* c, const float* q, size_t nq, size_t q_stride_floats, int k, int* idx, float* d2, int nthreads) {
  auto& cl = *(std::shared_ptr<orc::Cloud>*)c;
  if (!cl->index) return -2;
#pragma omp parallel for num_threads(nthreads) schedule(guided, 8)
  for (long i = 0; i < (long)nq; i++) {
    int found = cl->index->knn(q + i * q_stride_floats, k, idx + i * k, d2 + i * k);
    for (int j = found; j < k; j++) { idx[i * k + j] = -1; d2[i * k + j] = -1.f; }
  }
  return 0;
}

int orc_cloud_covariances(void* c, int k, int method, int nthreads, double* covs, int* knn_idx, float* knn_d2) {
  auto& cl = *(std::shared_ptr<orc::Cloud>*)c;
  return orc::calc_covariances(*cl, k, method, nthreads, covs, knn_idx, knn_d2);
}

void* orc_gicp_create() { return new orc::Gicp(); }
void orc_gicp_destroy(void* g) { delete (orc::Gicp*)g; }

void orc_gicp_set_params(void* g, int k, double max_corr_dist, int max_iter, double trans_eps, double rot_eps,
                         int lm_max_iter, double lm_init_lambda_factor, int reg_method, int optimizer, int num_threads) {
  auto* G = (orc::Gicp*)g;
  G->prm.k_correspondences = k;
  G->prm.corr_dist_threshold = max_corr_dist;
  G->prm.max_iterations = max_iter;
  G->prm.transformation_epsilon = trans_eps;
  G->prm.rotation_epsilon = rot_eps;
  G->prm.lm_max_iterations = lm_max_iter;
  G->prm.lm_init_lambda_factor = lm_init_lambda_factor;
  G->prm.regularization = reg_method;
  G->prm.optimizer = optimizer;
  G->prm.num_threads = num_threads > 0 ? num_threads : orc_max_threads();
}

void orc_gicp_set_source(void* g, void* cloud) { auto* G = (orc::Gicp*)g; G->source = *(std::shared_ptr<orc::Cloud>*)cloud; G->source_covs.clear(); }
void orc_gicp_set_target(void* g, void* cloud) { auto* G = (orc::Gicp*)g; G->target = *(std::shared_ptr<orc::Cloud>*)cloud; G->target_covs.clear(); }

static void set_covs(std::vector<orc::M4>& dst, const double* covs, size_t n) {
  dst.resize(n);
  for (size_t i = 0; i < n; i++) std::memcpy(dst[i].v, covs + i * 16, 128);
}
void orc_gicp_set_source_covs(void* g, const double* covs, size_t n) { set_covs(((orc::Gicp*)g)->source_covs, covs, n); }
void orc_gicp_set_target_covs(void* g, const double* covs, size_t n) { set_covs(((orc::Gicp*)g)->target_covs, covs, n); }

static int calc_into(orc::Gicp* G, std::shared_ptr<orc::Cloud>& cl, std::vector<orc::M4>& dst) {
  if (!cl) return -2;
  std::vector<double> tmp(cl->view.n * 16);
  int rc = orc::calc_covariances(*cl, G->prm.k_correspondences, G->prm.regularization, G->prm.num_threads, tmp.data(), nullptr, nullptr);
  if (rc) return rc;
  set_covs(dst, tmp.data(), cl->view.n);
  return 0;
}
int orc_gicp_calc_source_covs(void* g) { auto* G = (orc::Gicp*)g; return calc_into(G, G->source, G->source_covs); }
int orc_gicp_calc_target_covs(void* g) { auto* G = (orc::Gicp*)g; return calc_into(G, G->target, G->target_covs); }
size_t orc_gicp_get_source_covs(void* g, double* out) {
  auto* G = (orc::Gicp*)g;
  if (out) for (size_t i = 0; i < G->source_covs.size(); i++) std::memcpy(out + i * 16, G->source_covs[i].v, 128);
  return G->source_covs.size();
}
size_t orc_gicp_get_target_covs(void* g, double* out) {
  auto* G = (orc::Gicp*)g;
  if (out) for (size_t i = 0; i < G->target_covs.size(); i++) std::memcpy(out + i * 16, G->target_covs[i].v, 128);
  return G->target_covs.size();
}
void orc_gicp_swap(void* g) {
  auto* G = (orc::Gicp*)g;
  G->source.swap(G->target);
  G->source_covs.swap(G->target_covs);
  G->correspondences.clear();
  G->sq_distances.clear();
}

// one linearisation at T (col-major 4x4 double): H 6x6 col-major, b, error; optional per-point outputs
int orc_gicp_linearize(void* g, const double* T16, double* H36, double* b6, double* err, int* corr, float* sqd, double* mahal16) {
  auto* G = (orc::Gicp*)g;
  if (!G->source || !G->target || !G->target->index) return -2;
  if (G->source_covs.size() != G->source->view.n || G->target_covs.size() != G->target->view.n) return -4;
  orc::Iso x = orc::iso_from16(T16);
  orc::M6 H; orc::V6 b;
  double e = G->linearize(x, &H, &b);
  if (H36) std::memcpy(H36, H.v, sizeof(double) * 36);
  if (b6) std::memcpy(b6, b.v, sizeof(double) * 6);
  if (err) *err = e;
  const size_t n = G->source->view.n;
  if (corr) std::memcpy(corr, G->correspondences.data(), n * sizeof(int));
  if (sqd) std::memcpy(sqd, G->sq_distances.data(), n * sizeof(float));
  if (mahal16) for (size_t i = 0; i < n; i++) {
    if (G->correspondences[i] >= 0) std::memcpy(mahal16 + i * 16, G->mahalanobis[i].v, 128);
    else std::memset(mahal16 + i * 16, 0, 128);
  }
  return 0;
}
int orc_gicp_compute_error(void* g, const double* T16, double* err) {
  auto* G = (orc::Gicp*)g;
  if (G->correspondences.size() != G->source->view.n) return -4;
  orc::Iso x = orc::iso_from16(T16);
  *err = G->compute_error(x);
  return 0;
}
int orc_gicp_align(void* g, const float* guess16, orc::AlignResult* res) { return ((orc::Gicp*)g)->align(guess16, res); }

// exposed small kernels for property tests
void orc_svd3(const double* A9, double* U9, double* S3, double* V9) {
  orc::M3 A, U, V;
  std::memcpy(A.v, A9, 72);
  orc::jacobi_svd3(A, U, S3, V);
  std::memcpy(U9, U.v, 72);
  std::memcpy(V9, V.v, 72);
}
void orc_ldlt6_solve(const double* A36, const double* b6, double* x6) {
  orc::M6 A; orc::V6 b;
  std::memcpy(A.v, A36, 288);
  std::memcpy(b.v, b6, 48);
  orc::V6 x = orc::ldlt6_solve(A, b);
  std::memcpy(x6, x.v, 48);
}
void orc_so3_exp(const double* w3, double* R9) {
  orc::M3 R = orc::so3_exp_matrix(w3[0], w3[1], w3[2]);
  std::memcpy(R9, R.v, 72);
}
void orc_inverse4(const double* A16, double* out16) {
  orc::M4 A;
  std::memcpy(A.v, A16, 128);
  orc::M4 o = orc::inverse4(A);
  std::memcpy(out16, o.v, 128);
}

}  // extern "C"
