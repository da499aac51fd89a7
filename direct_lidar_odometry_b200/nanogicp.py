"""Python host-side mirror of `nano_gicp::NanoGICP<PointXYZI,PointXYZI>` over the C ABI.

Same member names, argument meaning and error behaviour as the reference class
(reference include/nano_gicp/nano_gicp.hpp:58-137, include/nano_gicp/lsq_registration.hpp:54-116 and
the pcl::Registration setters OdomNode calls at src/dlo/odom.cc:100-120), so that the parity tests
read like OdomNode's call sites.  The C++ facade with the identical surface is
include/nano_gicp/nano_gicp.hpp.  All compute goes to libnanogicp_b200.so; nothing here computes.

Clouds are (n,8) float32 pcl::PointXYZI records (numpy, or a CUDA torch tensor — the library
accepts host and device pointers alike); (n,3)/(n,4) float32 arrays are accepted too.
Matrices are numpy [row, col]; the ABI's column-major layout is handled here.
"""
from __future__ import annotations

import ctypes as C
import sys
import numpy as np

from . import _lib
from ._lib import Params, Result, Timings


class NanoGICPError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[{code}] {msg}")
        self.code = code


def _ptr_n_stride(cloud):
    """(pointer, n, stride_bytes, keepalive) of a 2-D float32 cloud given as numpy array or torch tensor."""
    if hasattr(cloud, "data_ptr"):  # torch tensor (host or CUDA)
        t = cloud
        if t.dim() != 2 or t.element_size() != 4 or t.stride(1) != 1:
            raise ValueError("cloud tensor must be 2-D float32 with unit inner stride")
        return t.data_ptr(), int(t.shape[0]), int(t.stride(0)) * 4 if t.shape[0] > 1 else int(t.shape[1]) * 4, t
    a = np.asarray(cloud)
    if a.dtype != np.float32 or a.ndim != 2 or a.shape[1] < 3:
        raise ValueError("cloud must be a float32 array of shape (n, >=3)")
    if a.strides[1] != 4:
        a = np.ascontiguousarray(a)
    stride = a.strides[0] if a.shape[0] > 1 else a.shape[1] * 4
    return a.ctypes.data, int(a.shape[0]), int(stride), a


def _mat_to_abi(T, dtype):
    return np.ascontiguousarray(np.asarray(T, dtype=dtype).T).reshape(16)


class CovarianceView:
    """What `source_covs_` / `target_covs_` evaluate to: a device-resident vector of Matrix4d that turns
    into a numpy (n,4,4) array on demand and can be assigned to another NanoGICP without leaving HBM."""

    def __init__(self, owner: "NanoGICP", which: int):
        self.owner, self.which = owner, which

    def __len__(self):
        return int(self.owner._L.ngicp_covs_size(self.owner._h, self.which))

    size = __len__

    def __array__(self, dtype=None, copy=None):
        a = self.owner._get_covs(self.which)
        return a if dtype is None else a.astype(dtype)

    def numpy(self):
        return self.owner._get_covs(self.which)

    def clear(self):
        self.owner._check(self.owner._L.ngicp_clear_covs(self.owner._h, self.which))


class NanoGICP:
    def __init__(self, device: int = 0):
        self._L = _lib.load()
        h = C.c_void_p()
        rc = self._L.ngicp_create(device, C.byref(h))
        if rc != 0 or not h:
            raise NanoGICPError(rc, "ngicp_create failed: no usable CUDA device (this library has no CPU fallback)")
        self._h = h
        self.device = device
        self._p = Params()
        self._L.ngicp_get_params(self._h, C.byref(self._p))
        self._p_ok = Params()
        C.memmove(C.byref(self._p_ok), C.byref(self._p), C.sizeof(self._p))
        self._input = None
        self._target = None
        self._res = Result()
        self._final = np.eye(4, dtype=np.float32)
        self._converged = False
        self.nr_iterations_ = 0

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._L.ngicp_destroy(h)
            self._h = None

    # ------------------------------------------------------------------ helpers
    def _check(self, rc: int):
        if rc < 0:
            raise NanoGICPError(rc, self._L.ngicp_last_error(self._h).decode())
        return rc

    def _push_params(self):
        # a rejected value must not stay in the struct (every later setter would fail with it): restore the last
        # accepted parameters before raising
        rc = self._L.ngicp_set_params(self._h, C.byref(self._p))
        if rc < 0:
            C.memmove(C.byref(self._p), C.byref(self._p_ok), C.sizeof(self._p))
        else:
            C.memmove(C.byref(self._p_ok), C.byref(self._p), C.sizeof(self._p))
        self._check(rc)

    # ------------------------------------------------------------------ parameters (odom.cc:100-120)
    def setNumThreads(self, n: int):  # OpenMP knob of the reference; the GPU path has no use for it
        pass

    def setCorrespondenceRandomness(self, k: int):
        self._p.k_correspondences = int(k)
        self._push_params()

    def setRegularizationMethod(self, method: int):
        self._p.regularization_method = int(method)
        self._push_params()

    def setMaxCorrespondenceDistance(self, d: float):
        self._p.max_correspondence_distance = float(d)
        self._push_params()

    def setMaximumIterations(self, n: int):
        self._p.max_iterations = int(n)
        self._push_params()

    def setTransformationEpsilon(self, eps: float):
        self._p.transformation_epsilon = float(eps)
        self._push_params()

    def setRotationEpsilon(self, eps: float):
        self._p.rotation_epsilon = float(eps)
        self._push_params()

    def setInitialLambdaFactor(self, f: float):
        self._p.lm_init_lambda_factor = float(f)
        self._push_params()

    def setOptimizer(self, opt: int):
        self._p.optimizer = int(opt)
        self._push_params()

    def setLMMaxIterations(self, n: int):
        self._p.lm_max_iterations = int(n)
        self._push_params()

    def setDebugPrint(self, flag: bool):
        pass

    # accepted, and without effect on NanoGICP in the reference as well (SURVEY A8)
    def setEuclideanFitnessEpsilon(self, eps: float):
        pass

    def setRANSACIterations(self, n: int):
        pass

    def setRANSACOutlierRejectionThreshold(self, t: float):
        pass

    def setSearchMethodSource(self, tree=None, force_no_recompute: bool = False):
        pass

    def setSearchMethodTarget(self, tree=None, force_no_recompute: bool = False):
        pass

    # B200-side knobs
    def setGridCellSize(self, cell: float):
        self._p.grid_cell_size = float(cell)
        self._push_params()

    def setGridTableCells(self, cells: int):
        self._p.grid_table_cells = int(cells)
        self._push_params()

    def setAlignMode(self, mode: int):
        self._p.align_mode = int(mode)
        self._push_params()

    def setKnnPath(self, path: int, tile_min_points: int | None = None):
        """Which exact kNN kernel family the covariance computation runs: _lib.KNN_AUTO / KNN_WARP / KNN_TILE."""
        self._p.knn_path = int(path)
        if tile_min_points is not None:
            self._p.knn_tile_min_points = int(tile_min_points)
        self._push_params()

    def setVoxelPath(self, path: int):
        """voxel filter / preprocess: 0 = one persistent cooperative launch when the cloud fits, 1 = multi-kernel pipeline."""
        self._p.voxel_path = int(path)
        self._push_params()

    def setIndexPath(self, path: int):
        """setInputSource / setInputTarget: 0 = snapshot + index in one persistent cooperative launch, 1 = multi-kernel pipeline."""
        self._p.index_path = int(path)
        self._push_params()

    # ------------------------------------------------------------------ clouds
    def setInputSource(self, cloud):
        if self._input is cloud:  # pointer-identity early-out, nano_gicp_impl.hpp:122
            return
        p, n, st, keep = _ptr_n_stride(cloud)
        if n == 0:
            print("[pcl::Registration::setInputSource] Invalid or empty point cloud dataset given!", file=sys.stderr)
            return
        self._check(self._L.ngicp_set_source(self._h, p, n, st))
        self._input = cloud

    def registerInputSource(self, cloud):
        if self._input is cloud:
            return
        p, n, st, keep = _ptr_n_stride(cloud)
        if n == 0:
            print("[pcl::Registration::setInputSource] Invalid or empty point cloud dataset given!", file=sys.stderr)
            return
        self._check(self._L.ngicp_register_source(self._h, p, n, st))
        self._input = cloud

    def setInputTarget(self, cloud):
        if self._target is cloud:
            return
        p, n, st, keep = _ptr_n_stride(cloud)
        if n == 0:
            print("[pcl::Registration::setInputTarget] Invalid or empty point cloud dataset given!", file=sys.stderr)
            return
        self._check(self._L.ngicp_set_target(self._h, p, n, st))
        self._target = cloud

    def swapSourceAndTarget(self):
        self._input, self._target = self._target, self._input
        self._check(self._L.ngicp_swap(self._h))

    def clearSource(self):
        self._input = None
        self._check(self._L.ngicp_clear_source(self._h))

    def clearTarget(self):
        self._target = None
        self._check(self._L.ngicp_clear_target(self._h))

    # `gicp.source_kdtree_ = gicp_s2s.source_kdtree_` (odom.cc:525)
    @property
    def source_kdtree_(self):
        return ("source_index", self)

    @source_kdtree_.setter
    def source_kdtree_(self, other):
        owner = other[1] if isinstance(other, tuple) else other
        self._check(self._L.ngicp_share_source(self._h, owner._h))
        self._input = owner._input

    # ------------------------------------------------------------------ covariances
    def calculateSourceCovariances(self) -> bool:
        self._check(self._L.ngicp_calc_source_covs(self._h))
        return True

    def calculateTargetCovariances(self) -> bool:
        self._check(self._L.ngicp_calc_target_covs(self._h))
        return True

    def calculateSourceCovariancesPart(self, part: int, nparts: int) -> bool:
        """Covariances of slice `part` of `nparts` of the source cloud, zeros elsewhere (ngicp_calc_source_covs_part);
        summing the buffers of all parts (covs_device_tensor + all-reduce) gives the complete set."""
        self._check(self._L.ngicp_calc_source_covs_part(self._h, int(part), int(nparts)))
        return True

    def covs_device_tensor(self, which: int):
        """The handle's covariance buffer as a (n, 6) float64 CUDA tensor WITHOUT copying (xx,xy,xz,yy,yz,zz per point);
        valid until the covariances are replaced.  The kernels that fill it run on the handle's stream: call sync() first,
        or use the tensor under torch.cuda.stream(ExternalStream(handle stream)) as sharded.set_source_sharded does."""
        import torch
        ptr, n = C.c_void_p(0), C.c_size_t(0)
        self._check(self._L.ngicp_covs_device(self._h, which, C.byref(ptr), C.byref(n)))

        class _View:
            __cuda_array_interface__ = {"shape": (int(n.value), 6), "typestr": "<f8", "data": (int(ptr.value), False), "version": 2}
        return torch.as_tensor(_View(), device=torch.device("cuda", self.device))

    def _set_covs(self, which: int, covs):
        if isinstance(covs, CovarianceView):
            if which == _lib.SOURCE and covs.which == _lib.SOURCE:
                self._check(self._L.ngicp_share_source_covs(self._h, covs.owner._h))
                return
            covs = covs.numpy()
        if hasattr(covs, "data_ptr"):  # device tensor of (n,16) column-major Matrix4d records
            n = int(covs.shape[0])
            fn = self._L.ngicp_set_source_covs if which == _lib.SOURCE else self._L.ngicp_set_target_covs
            self._check(fn(self._h, covs.data_ptr(), n))
            return
        a = np.asarray(covs, dtype=np.float64)
        n = a.shape[0]
        abi = np.ascontiguousarray(a.reshape(n, 4, 4).transpose(0, 2, 1)).reshape(n, 16) if n else np.zeros((0, 16))
        fn = self._L.ngicp_set_source_covs if which == _lib.SOURCE else self._L.ngicp_set_target_covs
        self._check(fn(self._h, abi.ctypes.data, n))

    def _get_covs(self, which: int) -> np.ndarray:
        n = int(self._L.ngicp_covs_size(self._h, which))
        out = np.zeros((n, 16), dtype=np.float64)
        if n:
            fn = self._L.ngicp_get_source_covs if which == _lib.SOURCE else self._L.ngicp_get_target_covs
            self._check(fn(self._h, out.ctypes.data, n))
        return out.reshape(n, 4, 4).transpose(0, 2, 1).copy()

    def setSourceCovariances(self, covs):
        self._set_covs(_lib.SOURCE, covs)

    def setTargetCovariances(self, covs):
        self._set_covs(_lib.TARGET, covs)

    def getSourceCovariances(self) -> np.ndarray:
        return self._get_covs(_lib.SOURCE)

    def getTargetCovariances(self) -> np.ndarray:
        return self._get_covs(_lib.TARGET)

    @property
    def source_covs_(self):
        return CovarianceView(self, _lib.SOURCE)

    @source_covs_.setter
    def source_covs_(self, covs):
        self._set_covs(_lib.SOURCE, covs)

    @property
    def target_covs_(self):
        return CovarianceView(self, _lib.TARGET)

    @target_covs_.setter
    def target_covs_(self, covs):
        self._set_covs(_lib.TARGET, covs)

    # ------------------------------------------------------------------ registration
    def align(self, guess=None, want_output: bool = False):
        """pcl::Registration::align(output[, guess]).  Returns the transformed source cloud (n,4) when
        `want_output` (DLO never reads it, odom.cc:799-837), else None."""
        if self._target is None:
            print("[pcl::Registration::align] No input target dataset was given!", file=sys.stderr)
            return None
        g = None
        if guess is not None:
            ga = _mat_to_abi(guess, np.float32)
            g = ga.ctypes.data_as(C.POINTER(C.c_float))
        self._converged = False
        self._check(self._L.ngicp_align(self._h, g, C.byref(self._res)))
        self._final = np.array(self._res.final_transformation, dtype=np.float32).reshape(4, 4).T.copy()
        self._converged = bool(self._res.converged)
        self.nr_iterations_ = int(self._res.nr_iterations)
        if want_output:
            n = int(self._L.ngicp_cloud_size(self._h, _lib.SOURCE))
            out = np.zeros((n, 4), dtype=np.float32)
            Tf = _mat_to_abi(self._final, np.float32)
            self._check(self._L.ngicp_transform_source(self._h, Tf.ctypes.data_as(C.POINTER(C.c_float)), out.ctypes.data, n))
            return out
        return None

    def getFinalTransformation(self) -> np.ndarray:
        return self._final.copy()

    def getFitnessScore(self, max_range: float = sys.float_info.max, T=None) -> float:
        """pcl::Registration::getFitnessScore(max_range): the mean SQUARED distance from the source, transformed by T
        (default: getFinalTransformation()), to its nearest target point, over the points whose squared distance is
        <= max_range (PCL compares the squared distance with max_range as given).  sys.float_info.max when no point
        qualifies.  Searches the device index, so it also works on a target set by KeyframeStore.set_target."""
        return self.fitness(T, max_range)[0]

    def fitness(self, T=None, max_range: float = sys.float_info.max):
        """(score, number of points that entered it) of getFitnessScore — ngicp_fitness_score."""
        Tf = _mat_to_abi(self._final if T is None else T, np.float32)
        score, n = C.c_double(0), C.c_size_t(0)
        self._check(self._L.ngicp_fitness_score(self._h, Tf.ctypes.data_as(C.POINTER(C.c_float)), float(max_range),
                                                C.byref(score), C.byref(n)))
        return score.value, int(n.value)

    def hasConverged(self) -> bool:
        return self._converged

    def getFinalHessian(self) -> np.ndarray:
        return np.array(self._res.final_hessian, dtype=np.float64).reshape(6, 6).T.copy()

    @property
    def result(self) -> Result:
        return self._res

    def final_state(self) -> np.ndarray:
        """The double-precision SE(3) state behind getFinalTransformation()."""
        return np.array(self._res.final_x, dtype=np.float64).reshape(4, 4).T.copy()

    # ------------------------------------------------------------------ introspection (parity tests)
    def knn(self, which: int, queries, k: int):
        p, nq, st, keep = _ptr_n_stride(queries)
        idx = np.zeros((nq, k), dtype=np.int32)
        d2 = np.zeros((nq, k), dtype=np.float32)
        self._check(self._L.ngicp_knn(self._h, which, p, nq, st, k, idx.ctypes.data_as(C.POINTER(C.c_int)),
                                      d2.ctypes.data_as(C.POINTER(C.c_float))))
        return idx, d2

    def cov_neighbors(self, which: int):
        """(idx (n,k) original indices, d2 (n,k)) of the neighbours the last calculate*Covariances call on this handle
        summed over, in summation order (ascending distance, ties by index) — ngicp_cov_neighbors."""
        n = int(self._L.ngicp_cloud_size(self._h, which))
        k = int(self._p.k_correspondences)
        idx = np.zeros((n, k), dtype=np.int32)
        d2 = np.zeros((n, k), dtype=np.float32)
        self._check(self._L.ngicp_cov_neighbors(self._h, which, idx.ctypes.data_as(C.POINTER(C.c_int)),
                                                d2.ctypes.data_as(C.POINTER(C.c_float))))
        return idx, d2

    def linearize(self, T, per_point: bool = False):
        Tc = _mat_to_abi(T, np.float64)
        H, b, e = np.zeros(36), np.zeros(6), C.c_double(0)
        n = int(self._L.ngicp_cloud_size(self._h, _lib.SOURCE))
        corr = np.zeros(n, dtype=np.int32)
        sqd = np.zeros(n, dtype=np.float32)
        mah = np.zeros((n, 16)) if per_point else None
        dp = C.POINTER(C.c_double)
        self._check(self._L.ngicp_linearize(self._h, Tc.ctypes.data_as(dp), H.ctypes.data_as(dp), b.ctypes.data_as(dp),
                                            C.byref(e), corr.ctypes.data_as(C.POINTER(C.c_int)),
                                            sqd.ctypes.data_as(C.POINTER(C.c_float)),
                                            mah.ctypes.data_as(dp) if per_point else None))
        out = dict(H=H.reshape(6, 6).T.copy(), b=b, err=e.value, corr=corr, sqd=sqd)
        if per_point:
            out["mahalanobis"] = mah.reshape(n, 4, 4).transpose(0, 2, 1).copy()
        return out

    def compute_error(self, T) -> float:
        Tc = _mat_to_abi(T, np.float64)
        e = C.c_double(0)
        self._check(self._L.ngicp_compute_error(self._h, Tc.ctypes.data_as(C.POINTER(C.c_double)), C.byref(e)))
        return e.value

    def linearize_partial(self, T, out43=None) -> np.ndarray:
        """Raw {H(36, col-major), b(6), err} partial sums of this handle's target shard (sharded-submap mode)."""
        Tc = _mat_to_abi(T, np.float64)
        if out43 is None:
            out43 = np.zeros(43)
        ptr = out43.data_ptr() if hasattr(out43, "data_ptr") else out43.ctypes.data
        self._check(self._L.ngicp_linearize_partial(self._h, Tc.ctypes.data_as(C.POINTER(C.c_double)), ptr))
        return out43

    def nn1_packed(self, T, rank: int) -> np.ndarray:
        """Every source point's nearest neighbour in THIS handle's target under T as (float bits of d^2) << 32 | rank
        (uint64; 0x7f800000ffffffff = none within the max-correspondence distance) — ngicp_nn1_packed."""
        Tc = _mat_to_abi(T, np.float64)
        n = int(self._L.ngicp_cloud_size(self._h, _lib.SOURCE))
        out = np.zeros(max(n, 1), dtype=np.uint64)
        self._check(self._L.ngicp_nn1_packed(self._h, Tc.ctypes.data_as(C.POINTER(C.c_double)), int(rank), out.ctypes.data))
        return out[:n]

    def linearize_won(self, T, rank: int, packed_min: np.ndarray) -> np.ndarray:
        """{H(36, col-major), b(6), err} over the source points whose global nearest neighbour this rank holds
        (packed_min = element-wise minimum of all ranks' nn1_packed arrays) — ngicp_linearize_won."""
        Tc = _mat_to_abi(T, np.float64)
        pm = np.ascontiguousarray(packed_min, dtype=np.uint64)
        out43 = np.zeros(43)
        self._check(self._L.ngicp_linearize_won(self._h, Tc.ctypes.data_as(C.POINTER(C.c_double)), int(rank), pm.ctypes.data, out43.ctypes.data))
        return out43

    def compute_error_partial(self, T, out1=None):
        Tc = _mat_to_abi(T, np.float64)
        if out1 is None:
            out1 = np.zeros(1)
        ptr = out1.data_ptr() if hasattr(out1, "data_ptr") else out1.ctypes.data
        self._check(self._L.ngicp_compute_error_partial(self._h, Tc.ctypes.data_as(C.POINTER(C.c_double)), ptr))
        return out1

    # ------------------------------------------------------------------ pcl::VoxelGrid
    def _host_records(self, n: int) -> np.ndarray:
        """Reusable host landing buffer for (n, 8) float32 records: a fresh np.zeros per call costs more than the whole
        device pipeline (1.7 MB of page faults for a 53k-point scan); callers get a copy of the m rows that were written."""
        buf = getattr(self, "_rec_buf", None)
        if buf is None or buf.shape[0] < max(n, 1):
            buf = np.empty((max(n + n // 4, 1024), 8), dtype=np.float32)
            self._rec_buf = buf
        return buf

    def voxel_filter(self, cloud, leaf: float, out=None, return_status: bool = False):
        """pcl::VoxelGrid<PointXYZI> with leaf (l,l,l): returns (m,8) float32 records (numpy unless `out`
        is a preallocated CUDA tensor of shape (>=n,8), in which case a view of it is returned)."""
        p, n, st, keep = _ptr_n_stride(cloud)
        m = C.c_size_t(0)
        if out is None:
            buf = self._host_records(n)
            optr, cap = buf.ctypes.data, buf.shape[0]
        else:
            buf = out
            optr, cap = out.data_ptr(), int(out.shape[0])
        rc = self._check(self._L.ngicp_voxel_filter(self._h, p, n, st, C.c_float(leaf), optr, cap, C.byref(m)))
        res = buf[: m.value]
        if out is None:
            res = res.copy()
        return (res, rc) if return_status else res

    def preprocess(self, cloud, crop_size: float | None = 1.0, leaf: float = 0.25, out=None, return_status: bool = False):
        """OdomNode::preprocessPoints (odom.cc:443-465) in one device pass: removeNaN + negative CropBox(+-crop_size,
        None = no crop) + scan voxel grid (leaf <= 0 = no voxel grid).  Same output convention as voxel_filter."""
        p, n, st, keep = _ptr_n_stride(cloud)
        m = C.c_size_t(0)
        if out is None:
            buf = self._host_records(n)
            optr, cap = buf.ctypes.data, buf.shape[0]
        else:
            buf = out
            optr, cap = out.data_ptr(), int(out.shape[0])
        lo = hi = None
        if crop_size is not None:
            lo = (C.c_float * 3)(-crop_size, -crop_size, -crop_size)
            hi = (C.c_float * 3)(crop_size, crop_size, crop_size)
        rc = self._check(self._L.ngicp_preprocess(self._h, p, n, st, lo, hi, C.c_float(leaf), optr, cap, C.byref(m)))
        res = buf[: m.value]
        if out is None:
            res = res.copy()
        return (res, rc) if return_status else res

    def preprocess_pointcloud2(self, msg, crop_size: float | None = 1.0, leaf: float = 0.25, out=None, data_ptr: int | None = None,
                               return_status: bool = False):
        """pcl::fromROSMsg (odom.cc:636-637) + preprocessPoints (:443-465) in one device pass over the message bytes.
        msg: anything with sensor_msgs/PointCloud2's members (see pointcloud2.PointCloud2); data_ptr: address of the
        byte array when it already sits in pinned or device memory (msg.data is then not touched)."""
        from .pointcloud2 import xyzi_layout
        lay = xyzi_layout(msg)
        n = int(msg.width) * int(msg.height)
        keep = None
        if data_ptr is None:
            keep = np.frombuffer(msg.data, dtype=np.uint8)
            data_ptr = keep.ctypes.data if keep.size else None
        m = C.c_size_t(0)
        if out is None:
            buf = self._host_records(n)
            optr, cap = buf.ctypes.data, buf.shape[0]
        else:
            buf = out
            optr, cap = out.data_ptr(), int(out.shape[0])
        lo = hi = None
        if crop_size is not None:
            lo = (C.c_float * 3)(-crop_size, -crop_size, -crop_size)
            hi = (C.c_float * 3)(crop_size, crop_size, crop_size)
        rc = self._check(self._L.ngicp_preprocess_pointcloud2(self._h, data_ptr, C.byref(lay), lo, hi, C.c_float(leaf), optr, cap, C.byref(m)))
        res = buf[: m.value]
        if out is None:
            res = res.copy()
        return (res, rc) if return_status else res

    def transform_voxel_filter(self, cloud, T, leaf: float, out=None):
        """pcl::transformPointCloud(cloud, T) + pcl::VoxelGrid(leaf) in one device pass (keyframes, odom.cc:484-490)."""
        p, n, st, keep = _ptr_n_stride(cloud)
        m = C.c_size_t(0)
        if out is None:
            buf = self._host_records(n)
            optr, cap = buf.ctypes.data, buf.shape[0]
        else:
            buf = out
            optr, cap = out.data_ptr(), int(out.shape[0])
        Tc = _mat_to_abi(T, np.float32)
        self._check(self._L.ngicp_transform_voxel_filter(self._h, p, n, st, Tc.ctypes.data_as(C.POINTER(C.c_float)), C.c_float(leaf),
                                                         optr, cap, C.byref(m)))
        res = buf[: m.value]
        return res.copy() if out is None else res

    def voxel_assignment(self, n: int) -> np.ndarray:
        a = np.zeros(n, dtype=np.int32)
        self._check(self._L.ngicp_voxel_assignment(self._h, a.ctypes.data_as(C.POINTER(C.c_int)), n))
        return a

    def set_owner_slab(self, axis: int, lo: float = 0.0, hi: float = 0.0):
        self._check(self._L.ngicp_set_owner_slab(self._h, axis, C.c_float(lo), C.c_float(hi)))

    # ------------------------------------------------------------------ sharded-submap exchange (fused into align)
    def comm_export(self) -> bytes:
        """This rank's exchange buffer as a 64-byte CUDA IPC handle (allocates it on first use)."""
        buf = (C.c_ubyte * 64)()
        self._check(self._L.ngicp_comm_export(self._h, buf))
        return bytes(buf)

    def comm_connect(self, rank: int, world: int, handles) -> None:
        """Map the exchange buffers of all ranks (`handles[r]` = comm_export() of rank r, one process per GPU).
        Barrier between this call and the first align()."""
        blob = b"".join(bytes(h) for h in handles)
        assert len(blob) == 64 * world
        arr = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        self._check(self._L.ngicp_comm_connect(self._h, rank, world, arr))

    def comm_connect_local(self, rank: int, peers) -> None:
        """Same for NanoGICP objects living in this process (several GPUs, or one GPU in tests)."""
        arr = (C.c_void_p * len(peers))(*[p._h for p in peers])
        self._check(self._L.ngicp_comm_connect_local(self._h, rank, len(peers), arr))

    def comm_close(self) -> None:
        self._check(self._L.ngicp_comm_close(self._h))

    def comm_reset(self) -> None:
        """After NGICP_E_COMM: every rank resets its exchange buffer (then a host-side barrier), connections stay."""
        self._check(self._L.ngicp_comm_reset(self._h))

    def grid_info(self, which: int) -> dict:
        cell, dims, nc = C.c_float(0), (C.c_int * 3)(), C.c_int(0)
        self._check(self._L.ngicp_grid_info(self._h, which, C.byref(cell), dims, C.byref(nc)))
        return {"cell": cell.value, "dims": list(dims), "ncells": nc.value}

    # ------------------------------------------------------------------ plumbing
    def set_stream(self, cuda_stream_ptr: int | None):
        self._check(self._L.ngicp_set_stream(self._h, cuda_stream_ptr))

    def sync(self):
        self._check(self._L.ngicp_sync(self._h))

    def timings(self) -> dict:
        t = Timings()
        self._check(self._L.ngicp_get_timings(self._h, C.byref(t)))
        return {k: getattr(t, k) for k, _ in Timings._fields_ if k != "reserved"}


def imu_prior(stamps, ang_vel, prev_frame_stamp: float, curr_frame_stamp: float) -> np.ndarray:
    """OdomNode::integrateIMU (odom.cc:859-919): the 4x4 float `imu_SE3` guess from the gyro samples between two scans
    (ngicp_imu_prior; host arithmetic, no GPU needed).  stamps (n,) seconds, ang_vel (n,3) rad/s."""
    L = _lib.load()
    st = np.ascontiguousarray(stamps, dtype=np.float64)
    av = np.ascontiguousarray(ang_vel, dtype=np.float64).reshape(-1, 3)
    out = np.zeros(16, dtype=np.float32)
    dp = C.POINTER(C.c_double)
    rc = L.ngicp_imu_prior(st.ctypes.data_as(dp), av.ctypes.data_as(dp), st.shape[0], float(prev_frame_stamp), float(curr_frame_stamp),
                           out.ctypes.data_as(C.POINTER(C.c_float)))
    if rc < 0:
        raise NanoGICPError(rc, "ngicp_imu_prior: bad arguments")
    return out.reshape(4, 4).T.copy()


def align_batch(handles, guesses=None):
    """ngicp_align_batch: register len(handles) independent pairs (each NanoGICP object holds its own source and target)
    in ONE kernel launch; every object ends up exactly as if its own align(guess) had been called.  guesses: sequence
    of 4x4 matrices (None entries = identity) or None.  Returns the list of Result structs."""
    n = len(handles)
    if n == 0:
        return []
    L = handles[0]._L
    arr = (C.c_void_p * n)(*[h._h for h in handles])
    g = None
    if guesses is not None:
        ga = np.zeros((n, 16), dtype=np.float32)
        for i, G in enumerate(guesses):
            ga[i] = _mat_to_abi(np.eye(4) if G is None else G, np.float32)
        g = ga.ctypes.data_as(C.POINTER(C.c_float))
    res = (Result * n)()
    for h in handles:
        if h._target is None:
            raise NanoGICPError(_lib.E_STATE, "align_batch: a handle has no target")
        h._converged = False
    handles[0]._check(L.ngicp_align_batch(arr, n, g, res))
    out = []
    for i, h in enumerate(handles):
        C.memmove(C.byref(h._res), C.byref(res[i]), C.sizeof(Result))
        h._final = np.array(h._res.final_transformation, dtype=np.float32).reshape(4, 4).T.copy()
        h._converged = bool(h._res.converged)
        h.nr_iterations_ = int(h._res.nr_iterations)
        out.append(h._res)
    return out


def fitness_batch(handles, transforms=None, max_range: float = sys.float_info.max):
    """ngicp_fitness_batch: getFitnessScore(max_range) of len(handles) independent pairs (each NanoGICP object with its
    own source and target) in a constant number of launches, bit-identical to the single calls.  transforms: sequence
    of 4x4 matrices (None entries = that handle's getFinalTransformation()) or None.  Returns (scores, counts) as
    float64 / int64 arrays."""
    n = len(handles)
    if n == 0:
        return np.zeros(0), np.zeros(0, dtype=np.int64)
    L = handles[0]._L
    arr = (C.c_void_p * n)(*[h._h for h in handles])
    ta = np.zeros((n, 16), dtype=np.float32)
    for i, h in enumerate(handles):
        T = None if transforms is None else transforms[i]
        ta[i] = _mat_to_abi(h._final if T is None else T, np.float32)
    scores = np.zeros(n)
    counts = np.zeros(n, dtype=np.uint64)
    handles[0]._check(L.ngicp_fitness_batch(arr, n, ta.ctypes.data_as(C.POINTER(C.c_float)), float(max_range),
                                            scores.ctypes.data_as(C.POINTER(C.c_double)),
                                            counts.ctypes.data_as(C.POINTER(C.c_size_t))))
    return scores, counts.astype(np.int64)


class KeyframeStore:
    """Device-resident keyframes (include/nanogicp_c.h, ngicp_kfstore_*): what OdomNode keeps in `keyframes` /
    `keyframe_normals` on the host, and the submap concatenation of getSubmapKeyframes, without leaving the GPU."""

    def __init__(self, device: int = 0):
        self._L = _lib.load()
        h = C.c_void_p()
        rc = self._L.ngicp_kfstore_create(device, C.byref(h))
        if rc != _lib.OK:
            raise NanoGICPError(rc, "ngicp_kfstore_create failed")
        self._h = h

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._L.ngicp_kfstore_destroy(h)
            self._h = None

    def __len__(self):
        return int(self._L.ngicp_kfstore_size(self._h))

    def points(self, index: int) -> int:
        return int(self._L.ngicp_kfstore_points(self._h, index))

    def push(self, gicp: NanoGICP) -> int:
        """keyframes.push_back / keyframe_normals.push_back: the current SOURCE cloud + covariances of `gicp`."""
        idx = C.c_size_t(0)
        gicp._check(self._L.ngicp_kfstore_push(self._h, gicp._h, C.byref(idx)))
        return int(idx.value)

    def set_target(self, gicp: NanoGICP, indices) -> None:
        """submap concat + setInputTarget + setTargetCovariances for the selected keyframes, on the device."""
        arr = (C.c_int * len(indices))(*[int(i) for i in indices])
        gicp._check(self._L.ngicp_kfstore_set_target(self._h, gicp._h, arr, len(indices)))
        gicp._target = object()    # a cloud no caller holds: the next setInputTarget(cloud) is never an identity hit
