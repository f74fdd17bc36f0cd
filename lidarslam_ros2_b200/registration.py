"""Python mirror of the reference's registration surface, bound to the CUDA C-ABI (include/b200reg.h).

The class and method names follow pcl::Registration / pclomp exactly as the lidarslam_ros2 nodes call them
(scanmatcher/src/scanmatcher_component.cpp:103-124, 262-387; graph_based_slam/src/graph_based_slam_component.cpp:
63-86, 145-260; Thirdparty/ndt_omp_ros2/apps/align.cpp:18-40), so a parity test reads like the reference's own
benchmark: setInputTarget / setInputSource / align / getFinalTransformation / getFitnessScore / hasConverged.

Host code here is plumbing only: every numeric result comes from the sm_100a kernels in csrc/. There is no CPU
fallback; constructing an engine without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi
from ._capi import DIRECT1, DIRECT7, DIRECT26, GICP, KDTREE, NDT

__all__ = ["NormalDistributionsTransform", "GeneralizedIterativeClosestPoint", "voxel_grid_filter", "align_batch",
           "B200RegError", "KDTREE", "DIRECT26", "DIRECT7", "DIRECT1"]


class B200RegError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"b200reg error {code}: {msg}")
        self.code = code


def _as_cloud(points) -> np.ndarray:
    a = np.ascontiguousarray(points, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] < 3:
        raise ValueError("cloud must be (N, >=3) float32")
    return a


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _colmajor(T) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(T, dtype=np.float32).T).reshape(16)


def _from_colmajor(buf: np.ndarray) -> np.ndarray:
    return buf.reshape(4, 4).T.copy()


class _Registration:
    """pcl::Registration<PointXYZI, PointXYZI> surface shared by both engines."""

    _kind = NDT

    def __init__(self, device: int = 0):
        self._lib = _capi.lib()
        h = C.c_void_p()
        rc = self._lib.b200reg_create(self._kind, int(device), C.byref(h))
        if rc != 0:
            raise B200RegError(rc, "b200reg_create failed (no CUDA device? there is no CPU fallback)")
        self._h = h
        self.device = device
        self._n_source = 0

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.b200reg_destroy(h)
            self._h = None

    # ---- helpers ----
    def _check(self, rc: int, soft=()):
        if rc != 0 and rc not in soft:
            raise B200RegError(rc, self._lib.b200reg_last_error(self._h).decode())
        return rc

    # ---- pcl::Registration ----
    def setInputTarget(self, cloud):
        """Registration::setInputTarget (+ NDT init(), ndt_omp.h:117-122). Empty clouds are ignored like PCL does."""
        c = _as_cloud(cloud)
        if len(c) == 0:
            return
        self._check(self._lib.b200reg_set_input_target(self._h, _ptr(c), len(c), c.strides[0]))

    def setInputSource(self, cloud):
        c = _as_cloud(cloud)
        if len(c) == 0:
            return
        self._n_source = len(c)
        self._check(self._lib.b200reg_set_input_source(self._h, _ptr(c), len(c), c.strides[0]))

    def setInputTargetDevice(self, dev_ptr: int, n: int):
        """Target already resident in HBM as n float4 (e.g. a torch CUDA tensor's data_ptr())."""
        self._check(self._lib.b200reg_set_input_target_device(self._h, C.c_void_p(dev_ptr), n))

    def setInputSourceDevice(self, dev_ptr: int, n: int):
        self._n_source = n
        self._check(self._lib.b200reg_set_input_source_device(self._h, C.c_void_p(dev_ptr), n))

    def setTransformationEpsilon(self, eps: float):
        self._check(self._lib.b200reg_set_transformation_epsilon(self._h, float(eps)))

    def setMaximumIterations(self, n: int):
        self._check(self._lib.b200reg_set_maximum_iterations(self._h, int(n)))

    def setMaxCorrespondenceDistance(self, d: float):
        self._check(self._lib.b200reg_set_max_correspondence_distance(self._h, float(d)))

    def setEuclideanFitnessEpsilon(self, eps: float):
        self._check(self._lib.b200reg_set_euclidean_fitness_epsilon(self._h, float(eps)))

    def setRANSACIterations(self, n: int):
        self._check(self._lib.b200reg_set_ransac_iterations(self._h, int(n)))

    def align(self, guess=None) -> np.ndarray:
        """Registration::align(output, guess). Returns getFinalTransformation() as a row-major 4x4 numpy array.

        Like PCL this soft-fails when no target/source is set (hasConverged() stays False)."""
        g = _colmajor(guess) if guess is not None else None
        out = np.empty(16, dtype=np.float32)
        self._check(self._lib.b200reg_align(self._h, _ptr(g) if g is not None else None, _ptr(out)),
                    soft=(_capi.ERR_NO_TARGET, _capi.ERR_NO_SOURCE))
        return _from_colmajor(out)

    def getFinalTransformation(self) -> np.ndarray:
        out = np.empty(16, dtype=np.float32)
        self._check(self._lib.b200reg_get_final_transformation(self._h, _ptr(out)))
        return _from_colmajor(out)

    def hasConverged(self) -> bool:
        v = C.c_int(0)
        self._check(self._lib.b200reg_has_converged(self._h, C.byref(v)))
        return bool(v.value)

    def getFitnessScore(self, max_range: float = np.finfo(np.float64).max) -> float:
        v = C.c_double(0)
        self._check(self._lib.b200reg_get_fitness_score(self._h, float(max_range), C.byref(v)))
        return v.value

    def getAligned(self) -> np.ndarray:
        """The `output` cloud of align(): the source transformed by the final transformation, (N, 4) float32."""
        out = np.zeros((self._n_source, 4), dtype=np.float32)
        self._check(self._lib.b200reg_get_aligned(self._h, _ptr(out), 16))
        return out

    # ---- introspection ----
    def stats(self) -> dict:
        s = _capi.Stats()
        self._check(self._lib.b200reg_get_stats(self._h, C.byref(s)))
        return {name: getattr(s, name) for name, _ in s._fields_}

    def nearest(self, queries):
        q = _as_cloud(queries)
        idx = np.empty(len(q), dtype=np.int32)
        d2 = np.empty(len(q), dtype=np.float32)
        self._check(self._lib.b200reg_nn1(self._h, _ptr(q), len(q), q.strides[0], _ptr(idx), _ptr(d2)))
        return idx, d2


class NormalDistributionsTransform(_Registration):
    """pclomp::NormalDistributionsTransform (ndt_omp.h:70-497) on B200."""

    _kind = NDT

    def setResolution(self, resolution: float):
        self._check(self._lib.b200reg_ndt_set_resolution(self._h, float(resolution)))

    def setStepSize(self, step: float):
        self._check(self._lib.b200reg_ndt_set_step_size(self._h, float(step)))

    def setOulierRatio(self, ratio: float):  # sic — the reference's spelling (ndt_omp.h:180)
        self._check(self._lib.b200reg_ndt_set_outlier_ratio(self._h, float(ratio)))

    def setNeighborhoodSearchMethod(self, method: int):
        self._check(self._lib.b200reg_ndt_set_neighborhood_search_method(self._h, int(method)))

    def setNumThreads(self, n: int):
        self._check(self._lib.b200reg_ndt_set_num_threads(self._h, int(n)))

    def getTransformationProbability(self) -> float:
        v = C.c_double(0)
        self._check(self._lib.b200reg_ndt_get_transformation_probability(self._h, C.byref(v)))
        return v.value

    def getFinalNumIteration(self) -> int:
        v = C.c_int(0)
        self._check(self._lib.b200reg_ndt_get_final_num_iteration(self._h, C.byref(v)))
        return v.value

    def calculateScore(self, cloud) -> float:
        c = _as_cloud(cloud)
        v = C.c_double(0)
        self._check(self._lib.b200reg_ndt_calculate_score(self._h, _ptr(c), len(c), c.strides[0], C.byref(v)))
        return v.value

    # ---- batched registrations against the current target (one persistent launch, two in flight) ----
    # b200reg_batch_result as a numpy record: the K results are unpacked with a handful of vectorised field reads
    _BATCH_DTYPE = np.dtype([("final_T", np.float32, (16,)), ("trans_probability", np.float64), ("converged", np.int32),
                             ("iterations", np.int32), ("evaluations", np.int32), ("status", np.int32), ("hits_total", np.int64)])

    def _batch_out(self, res, K):
        assert self._BATCH_DTYPE.itemsize == C.sizeof(_capi.BatchResult)
        if K == 0:
            z = np.zeros(0, dtype=self._BATCH_DTYPE)
            return {"pose": np.zeros((0, 4, 4), dtype=np.float32), **{k: z[k] for k in ("converged", "iterations", "evaluations",
                                                                                       "trans_probability", "hits_total", "status")}}
        a = np.frombuffer(res, dtype=self._BATCH_DTYPE, count=K)
        return {"pose": a["final_T"].reshape(K, 4, 4).transpose(0, 2, 1).copy(),  # column-major -> row-major
                "converged": a["converged"].copy(), "iterations": a["iterations"].copy(), "evaluations": a["evaluations"].copy(),
                "trans_probability": a["trans_probability"].copy(), "hits_total": a["hits_total"].copy(), "status": a["status"].copy()}

    def alignBatch(self, clouds, guesses=None) -> dict:
        """K independent align() calls against the current target, sources in HOST memory (b200reg_ndt_align_batch).
        clouds: list of (N_k, >=3) float32 arrays with equal row stride; guesses: list of 4x4 or None (identity)."""
        K = len(clouds)
        cs = [_as_cloud(c) for c in clouds]
        stride = cs[0].strides[0] if K else 16
        if any(c.strides[0] != stride for c in cs):
            raise ValueError("alignBatch: all clouds must share one row stride")
        ptrs = (C.c_void_p * K)(*[c.ctypes.data for c in cs])
        ns = (C.c_size_t * K)(*[len(c) for c in cs])
        g = np.ascontiguousarray(np.stack([_colmajor(x) for x in guesses])) if guesses is not None else None
        res = (_capi.BatchResult * max(K, 1))()
        rc = self._lib.b200reg_ndt_align_batch(self._h, K, ptrs, ns, stride, _ptr(g) if g is not None else None, res)
        self._check(rc, soft=(_capi.ERR_NO_TARGET,))
        return self._batch_out(res, K)

    def alignBatchDevice(self, dev_ptrs, counts, guesses=None) -> dict:
        """Same with the sources already in HBM as float4 buffers (b200reg_ndt_align_batch_device), read in place."""
        return self.prepareBatchDevice(dev_ptrs, counts, guesses)()

    def prepareBatchDevice(self, dev_ptrs, counts, guesses=None):
        """The argument marshalling of alignBatchDevice done once: returns a callable that performs the C call (a caller
        that registers the same device buffers repeatedly — bench.py's timed region — pays the ctypes packing once)."""
        K = len(dev_ptrs)
        ptrs = (C.c_void_p * K)(*[int(p) for p in dev_ptrs])
        ns = (C.c_size_t * K)(*[int(n) for n in counts])
        g = np.ascontiguousarray(np.stack([_colmajor(x) for x in guesses])) if guesses is not None else None
        gp = _ptr(g) if g is not None else None
        res = (_capi.BatchResult * max(K, 1))()

        gather = self._prepared_gather()

        def call():
            rc = self._lib.b200reg_ndt_align_batch_device(self._h, K, ptrs, ns, gp, res)
            self._check(rc, soft=(_capi.ERR_NO_TARGET,))
            return gather(self._batch_out(res, K))

        call.keepalive = (ptrs, ns, g, res)
        return call

    def prepareBatch(self, clouds, guesses=None):
        """alignBatch (host sources) with the marshalling done once; the arrays in `clouds` must stay alive and unchanged in
        place between calls."""
        K = len(clouds)
        cs = [_as_cloud(c) for c in clouds]
        stride = cs[0].strides[0] if K else 16
        if any(c.strides[0] != stride for c in cs):
            raise ValueError("prepareBatch: all clouds must share one row stride")
        ptrs = (C.c_void_p * K)(*[c.ctypes.data for c in cs])
        ns = (C.c_size_t * K)(*[len(c) for c in cs])
        g = np.ascontiguousarray(np.stack([_colmajor(x) for x in guesses])) if guesses is not None else None
        gp = _ptr(g) if g is not None else None
        res = (_capi.BatchResult * max(K, 1))()

        gather = self._prepared_gather()

        def call():
            rc = self._lib.b200reg_ndt_align_batch(self._h, K, ptrs, ns, stride, gp, res)
            self._check(rc, soft=(_capi.ERR_NO_TARGET,))
            return gather(self._batch_out(res, K))

        call.keepalive = (cs, ptrs, ns, g, res)
        return call

    def sweep(self, sources, targets, guesses=None, fitness_max_range: float = np.finfo(np.float64).max) -> dict:
        """The loop-closure candidate sweep on this GPU (b200reg_ndt_sweep): K independent (source, target) pairs through
        setInputTarget + setInputSource + align + getFitnessScore, pipelined over up to four internal engines."""
        K = len(sources)
        ss = [_as_cloud(c) for c in sources]
        ts = [_as_cloud(c) for c in targets]
        stride = ss[0].strides[0] if K else 16
        if any(c.strides[0] != stride for c in ss + ts):
            raise ValueError("sweep: all clouds must share one row stride")
        sp = (C.c_void_p * K)(*[c.ctypes.data for c in ss])
        tp = (C.c_void_p * K)(*[c.ctypes.data for c in ts])
        sn = (C.c_size_t * K)(*[len(c) for c in ss])
        tn = (C.c_size_t * K)(*[len(c) for c in ts])
        g = np.ascontiguousarray(np.stack([_colmajor(x) for x in guesses])) if guesses is not None else None
        res = (_capi.SweepResult * max(K, 1))()
        self._check(self._lib.b200reg_ndt_sweep(self._h, K, sp, sn, tp, tn, stride, _ptr(g) if g is not None else None,
                                                float(fitness_max_range), res))
        if K == 0:
            return {"pose": np.zeros((0, 4, 4), np.float32), "fitness": np.zeros(0), "converged": np.zeros(0, np.int32),
                    "iterations": np.zeros(0, np.int32), "status": np.zeros(0, np.int32)}
        a = np.frombuffer(res, dtype=self._SWEEP_DTYPE, count=K)
        return {"pose": a["final_T"].reshape(K, 4, 4).transpose(0, 2, 1).copy(), "fitness": a["fitness"].copy(),
                "converged": a["converged"].copy(), "iterations": a["iterations"].copy(), "status": a["status"].copy()}

    _SWEEP_DTYPE = np.dtype([("final_T", np.float32, (16,)), ("fitness", np.float64), ("trans_probability", np.float64),
                             ("converged", np.int32), ("iterations", np.int32), ("status", np.int32), ("pad", np.int32)])

    def attachPoseBoard(self, board):
        """Multi-GPU batch calls (b200reg_ndt_attach_pose_board): with a batch.PoseBoard attached, alignBatch /
        alignBatchDevice become collective over the board's ranks and gatheredPoses() returns every rank's poses of the
        last call. None detaches."""
        self._check(self._lib.b200reg_ndt_attach_pose_board(self._h, board._h if board is not None else None))
        self._board = board

    def _prepared_gather(self):
        """For the prepared batch calls: with a pose board attached (at preparation time) the call's result also carries
        every rank's poses — "gathered" [world, max_rows, 4, 4] (a view into a buffer reused by the next call; rows beyond
        "gathered_counts"[r] are stale) — copied out of the board by b200reg_ndt_gathered_poses into preallocated arrays."""
        b = getattr(self, "_board", None)
        if b is None:
            return lambda out: out
        counts = np.zeros(b.world, dtype=np.int32)
        buf = np.zeros((b.world, b.max_rows, 16), dtype=np.float32)
        view = buf.reshape(b.world, b.max_rows, 4, 4).transpose(0, 1, 3, 2)  # column-major -> row-major, no copy
        pb, pc, fn, h, rows = buf.ctypes.data, counts.ctypes.data, self._lib.b200reg_ndt_gathered_poses, self._h, b.max_rows

        def gather(out):
            self._check(fn(h, pb, pc, rows))
            out["gathered"], out["gathered_counts"] = view, counts
            return out

        return gather

    def gatheredPoses(self):
        """(poses [world, max_count, 4, 4] float32 — rows beyond a rank's count are identity — and counts [world])."""
        b = getattr(self, "_board", None)
        if b is None:
            raise RuntimeError("gatheredPoses: no pose board attached")
        counts = np.zeros(b.world, dtype=np.int32)
        buf = np.zeros((b.world, b.max_rows, 16), dtype=np.float32)
        self._check(self._lib.b200reg_ndt_gathered_poses(self._h, buf.ctypes.data, counts.ctypes.data, b.max_rows))
        m = int(counts.max()) if b.world else 0
        out = buf[:, :m].reshape(b.world, m, 4, 4).transpose(0, 1, 3, 2).copy()
        for r in range(b.world):
            out[r, counts[r]:] = np.eye(4, dtype=np.float32)
        return out, counts

    def setBatchSlots(self, slots: int):
        self._check(self._lib.b200reg_ndt_set_batch_slots(self._h, int(slots)))

    # ---- parity hooks ----
    def derivatives(self, T, p6, compute_hessian: bool = True):
        """One fused derivative pass (computeDerivatives, ndt_omp_impl.hpp:179-284) → (score, g[6], H[6,6])."""
        Tc = _colmajor(T)
        p = np.ascontiguousarray(p6, dtype=np.float64)
        s = C.c_double(0)
        g = np.zeros(6)
        H = np.zeros((6, 6))
        self._check(self._lib.b200reg_ndt_derivatives(self._h, _ptr(Tc), _ptr(p), int(compute_hessian), C.byref(s),
                                                      _ptr(g), _ptr(H)))
        return s.value, g, H

    def hessian_radius(self, T, p6) -> np.ndarray:
        Tc = _colmajor(T)
        p = np.ascontiguousarray(p6, dtype=np.float64)
        H = np.zeros((6, 6))
        self._check(self._lib.b200reg_ndt_hessian_radius(self._h, _ptr(Tc), _ptr(p), _ptr(H)))
        return H

    def voxels(self) -> dict:
        n = C.c_size_t(0)
        self._check(self._lib.b200reg_ndt_num_voxels(self._h, C.byref(n)))
        V = n.value
        idx = np.empty(V, dtype=np.int32)
        npts = np.empty(V, dtype=np.int32)
        mean = np.empty((V, 3))
        icov = np.empty((V, 3, 3))
        cen = np.empty((V, 3), dtype=np.float32)
        if V:
            self._check(self._lib.b200reg_ndt_get_voxels(self._h, _ptr(idx), _ptr(npts), _ptr(mean), _ptr(icov), _ptr(cen)))
        return dict(idx=idx, npts=npts, mean=mean, icov=icov, centroid=cen)


class GeneralizedIterativeClosestPoint(_Registration):
    """pclomp::GeneralizedIterativeClosestPoint (gicp_omp.h:60-369) on B200."""

    _kind = GICP

    def setRotationEpsilon(self, eps: float):
        self._check(self._lib.b200reg_gicp_set_rotation_epsilon(self._h, float(eps)))

    def setCorrespondenceRandomness(self, k: int):
        self._check(self._lib.b200reg_gicp_set_correspondence_randomness(self._h, int(k)))

    def setMaximumOptimizerIterations(self, n: int):
        self._check(self._lib.b200reg_gicp_set_maximum_optimizer_iterations(self._h, int(n)))

    # ---- batched registrations against the current target (lock-step outer loops, inner solves share a launch) ----
    # b200reg_gicp_batch_result as a numpy record
    _BATCH_DTYPE = np.dtype([("final_T", np.float32, (16,)), ("converged", np.int32), ("iterations", np.int32),
                             ("evaluations", np.int32), ("correspondences", np.int32), ("status", np.int32), ("pad", np.int32)])
    _BATCH_FIELDS = ("converged", "iterations", "evaluations", "correspondences", "status")

    def _batch_out(self, res, K):
        assert self._BATCH_DTYPE.itemsize == C.sizeof(_capi.GicpBatchResult)
        if K == 0:
            z = np.zeros(0, dtype=self._BATCH_DTYPE)
            return {"pose": np.zeros((0, 4, 4), dtype=np.float32), **{k: z[k] for k in self._BATCH_FIELDS}}
        a = np.frombuffer(res, dtype=self._BATCH_DTYPE, count=K)
        return {"pose": a["final_T"].reshape(K, 4, 4).transpose(0, 2, 1).copy(),  # column-major -> row-major
                **{k: a[k].copy() for k in self._BATCH_FIELDS}}

    def alignBatch(self, clouds, guesses=None) -> dict:
        """K independent align() calls against the current target, sources in HOST memory (b200reg_gicp_align_batch).
        clouds: list of (N_k, >=3) float32 arrays with equal row stride; guesses: list of 4x4 or None (identity).
        Each result is bitwise what setInputSource + align(guess) gives; the handle's own source is not touched."""
        K = len(clouds)
        cs = [_as_cloud(c) for c in clouds]
        stride = cs[0].strides[0] if K else 16
        if any(c.strides[0] != stride for c in cs):
            raise ValueError("alignBatch: all clouds must share one row stride")
        ptrs = (C.c_void_p * K)(*[c.ctypes.data for c in cs])
        ns = (C.c_size_t * K)(*[len(c) for c in cs])
        g = np.ascontiguousarray(np.stack([_colmajor(x) for x in guesses])) if guesses is not None else None
        res = (_capi.GicpBatchResult * max(K, 1))()
        rc = self._lib.b200reg_gicp_align_batch(self._h, K, ptrs, ns, stride, _ptr(g) if g is not None else None, res)
        self._check(rc, soft=(_capi.ERR_NO_TARGET,))
        return self._batch_out(res, K)

    def alignBatchDevice(self, dev_ptrs, counts, guesses=None) -> dict:
        """Same with the sources already in HBM as float4 buffers (b200reg_gicp_align_batch_device), read in place."""
        K = len(dev_ptrs)
        ptrs = (C.c_void_p * K)(*[int(p) for p in dev_ptrs])
        ns = (C.c_size_t * K)(*[int(n) for n in counts])
        g = np.ascontiguousarray(np.stack([_colmajor(x) for x in guesses])) if guesses is not None else None
        res = (_capi.GicpBatchResult * max(K, 1))()
        rc = self._lib.b200reg_gicp_align_batch_device(self._h, K, ptrs, ns, _ptr(g) if g is not None else None, res)
        self._check(rc, soft=(_capi.ERR_NO_TARGET,))
        return self._batch_out(res, K)

    def setBatchSlots(self, slots: int):
        """Registrations in flight per batched inner-loop launch (1..3; larger values act as 3)."""
        self._check(self._lib.b200reg_ndt_set_batch_slots(self._h, int(slots)))

    # ---- parity hooks ----
    def covariances(self, which: str) -> np.ndarray:
        w = 1 if which == "target" else 0
        n = C.c_size_t(0)
        self._check(self._lib.b200reg_gicp_get_covariances(self._h, w, None, C.byref(n)))
        out = np.empty((n.value, 3, 3))
        if n.value:
            self._check(self._lib.b200reg_gicp_get_covariances(self._h, w, _ptr(out), C.byref(n)))
        return out

    def numCorrespondences(self) -> int:
        v = C.c_int(0)
        self._check(self._lib.b200reg_gicp_num_correspondences(self._h, C.byref(v)))
        return v.value


def align_batch(engines, guesses=None) -> np.ndarray:
    """Batched loop-closure sweep on one GPU: all solves are enqueued before any is awaited. Returns (K,4,4)."""
    K = len(engines)
    if K == 0:
        return np.zeros((0, 4, 4), dtype=np.float32)
    lib = _capi.lib()
    arr = (C.c_void_p * K)(*[e._h for e in engines])
    g = None
    if guesses is not None:
        g = np.ascontiguousarray(np.stack([_colmajor(x) for x in guesses]))
    out = np.empty((K, 16), dtype=np.float32)
    rc = lib.b200reg_align_batch(arr, K, _ptr(g) if g is not None else None, _ptr(out))
    if rc not in (0, _capi.ERR_NO_TARGET, _capi.ERR_NO_SOURCE):
        raise B200RegError(rc, "align_batch failed")
    return np.stack([_from_colmajor(out[i]) for i in range(K)])


def voxel_grid_filter(points, leaf: float, device: int = 0) -> np.ndarray:
    """pcl::VoxelGrid<PointXYZI>::filter with setLeafSize(leaf, leaf, leaf) on the GPU.

    points: (N,3) xyz or (N,4) xyz+intensity → (M,4) float32 in ascending leaf index."""
    p = _as_cloud(points)
    n, w = p.shape
    if w < 4:
        p = np.concatenate([p[:, :3], np.zeros((n, 1), dtype=np.float32)], axis=1)
    p = np.ascontiguousarray(p[:, :4])
    out = np.empty((max(n, 1), 4), dtype=np.float32)
    m = C.c_size_t(0)
    rc = _capi.lib().b200reg_voxelgrid(int(device), _ptr(p), n, 16, 12, float(leaf), _ptr(out), n, C.byref(m))
    if rc != 0:
        raise B200RegError(rc, "b200reg_voxelgrid failed")
    return out[:m.value].copy()
