"""ctypes binding of oracle/_ref/libbadslam_ref.so: the reference's OWN CUDA kernels (unmodified,
compiled by oracle/build_ref.sh) behind oracle/ref_driver.cu.

TEST / BASELINE INFRASTRUCTURE ONLY.  Needs a GPU; `available()` tells whether it can be used.

The GPU tests do not need the library: `reference(scene, ...)` replays what RefDirectBA returned, call by call, when the
test ran against the reference's kernels with BADBA_RECORD_REFERENCE=<dir> set (tests/golden/reference/, one file per
test).  A large output is recorded in part (`Sample`), with the digest of the whole array.
"""
from __future__ import annotations

import base64
import ctypes as C
import hashlib
import json
import os
import re

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libbadslam_ref.so")
RECORDED = os.path.join(os.path.dirname(_HERE), "tests", "golden", "reference")


class Config(C.Structure):
    _fields_ = [("depth_w", C.c_int), ("depth_h", C.c_int), ("color_w", C.c_int), ("color_h", C.c_int),
                ("depth_K", C.c_float * 4), ("color_K", C.c_float * 4),
                ("raw_to_float_depth", C.c_float), ("baseline_fx", C.c_float), ("cell", C.c_int),
                ("use_depth_residuals", C.c_int), ("use_descriptor_residuals", C.c_int)]


class BAOptions(C.Structure):
    _fields_ = [("optimize_poses", C.c_int), ("optimize_geometry", C.c_int),
                ("min_iterations", C.c_int), ("max_iterations", C.c_int),
                ("active_keyframe_window_start", C.c_int), ("active_keyframe_window_end", C.c_int),
                ("optimize_depth_intrinsics", C.c_int), ("optimize_color_intrinsics", C.c_int), ("end_tasks", C.c_int)]


class BAResult(C.Structure):
    _fields_ = [("iterations_done", C.c_int), ("converged", C.c_int), ("n_count", C.c_ulonglong), ("cost", C.c_double),
                ("pose_iterations_total", C.c_int), ("ms_surfel_activation", C.c_float),
                ("ms_geometry_optimization", C.c_float), ("ms_pose_optimization", C.c_float),
                ("kernel_launches", C.c_ulonglong), ("surfels_deleted", C.c_uint), ("surfels_size", C.c_uint),
                ("n_depth_count", C.c_ulonglong)]


class PCGOptions(C.Structure):
    _fields_ = [("optimize_poses", C.c_int), ("optimize_geometry", C.c_int), ("optimize_depth_intrinsics", C.c_int),
                ("optimize_color_intrinsics", C.c_int), ("min_iterations", C.c_int), ("max_iterations", C.c_int),
                ("max_inner_iterations", C.c_int), ("gauge_keyframe", C.c_int), ("end_tasks", C.c_int)]


class PCGResult(C.Structure):
    _fields_ = [("iterations_done", C.c_int), ("converged", C.c_int), ("inner_iterations_total", C.c_int),
                ("last_r_norm", C.c_float), ("ms_pcg", C.c_float), ("kernel_launches", C.c_ulonglong),
                ("surfels_deleted", C.c_uint), ("surfels_size", C.c_uint)]


class OdometryResult(C.Structure):
    _fields_ = [("iterations", C.c_int * 8), ("chose_initial", C.c_int * 8), ("residual_count", C.c_uint),
                ("residual_sum", C.c_float), ("kernel_launches", C.c_ulonglong), ("ms", C.c_float)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        l = C.CDLL(LIB_PATH)
        l.ref_create.restype = C.c_void_p
        l.ref_create.argtypes = [C.POINTER(Config), C.c_uint]
        l.ref_destroy.argtypes = [C.c_void_p]
        l.ref_set_surfels.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint]
        l.ref_get_surfels.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
        l.ref_get_active.argtypes = [C.c_void_p, C.c_void_p]
        l.ref_set_active.argtypes = [C.c_void_p, C.c_void_p]
        l.ref_set_depth_params.argtypes = [C.c_void_p, C.c_float, C.c_void_p]
        l.ref_set_intrinsics.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        l.ref_add_keyframe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_float, C.c_float]
        l.ref_get_pose.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        l.ref_set_pose.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        l.ref_get_activation.argtypes = [C.c_void_p, C.c_int]
        l.ref_set_activation.argtypes = [C.c_void_p, C.c_int, C.c_int]
        l.ref_launch_count.restype = C.c_ulonglong
        l.ref_launch_count.argtypes = [C.c_void_p]
        l.ref_pose_coeffs.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        l.ref_estimate_frame_pose.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        l.ref_update_activation.argtypes = [C.c_void_p]
        l.ref_optimize_intrinsics.argtypes = [C.c_void_p, C.c_int, C.c_int]
        l.ref_get_intrinsics.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        l.ref_get_cfactor.argtypes = [C.c_void_p, C.c_void_p]
        l.ref_optimize_geometry_iteration.argtypes = [C.c_void_p]
        l.ref_bundle_adjust.argtypes = [C.c_void_p, C.POINTER(BAOptions), C.POINTER(BAResult), C.c_int]
        l.ref_bundle_adjust_pcg.argtypes = [C.c_void_p, C.POINTER(PCGOptions), C.POINTER(PCGResult)]
        l.ref_pcg_debug.restype = C.c_uint
        l.ref_pcg_debug.argtypes = [C.c_void_p, C.POINTER(PCGOptions), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        l.ref_end_tasks.restype = C.c_uint
        l.ref_end_tasks.argtypes = [C.c_void_p]
        l.ref_surfels_size.restype = C.c_uint
        l.ref_surfels_size.argtypes = [C.c_void_p]
        l.ref_set_min_observation_counts.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        l.ref_create_surfels_for_keyframe.restype = C.c_uint
        l.ref_create_surfels_for_keyframe.argtypes = [C.c_void_p, C.c_int, C.c_int]
        l.ref_merge_surfels_for_keyframe.restype = C.c_uint
        l.ref_merge_surfels_for_keyframe.argtypes = [C.c_void_p, C.c_int]
        l.ref_compact_surfels.restype = C.c_uint
        l.ref_compact_surfels.argtypes = [C.c_void_p, C.c_uint, C.c_int]
        l.ref_set_surfels_size.argtypes = [C.c_void_p, C.c_uint]
        l.ref_preprocess_frame.restype = C.c_int
        l.ref_preprocess_frame.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        l.ref_track_frame_pairwise.restype = C.c_int
        l.ref_track_frame_pairwise.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                               C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(OdometryResult)]
        l.ref_odometry_get_level.restype = C.c_int
        l.ref_odometry_get_level.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int),
                                             C.POINTER(C.c_int)]
        l.ref_odometry_coeffs.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.POINTER(C.c_uint), C.POINTER(C.c_float), C.c_void_p, C.c_void_p]
        l.ref_snapshot.argtypes = [C.c_void_p]
        l.ref_restore.argtypes = [C.c_void_p]
        l.ref_sync.argtypes = [C.c_void_p]
        l.ref_last_cuda_error.restype = C.c_char_p
        _lib = l
    return _lib


def available() -> bool:
    if not os.path.exists(LIB_PATH):
        return False
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


class RefDirectBA:
    """The reference's CUDA DirectBA hot path on a synthetic scene."""

    def __init__(self, scene, use_depth=True, use_descriptor=True, poses=None):
        self.l = lib()
        cfg = scene.cfg
        c = Config()
        c.depth_w, c.depth_h, c.color_w, c.color_h = cfg.width, cfg.height, cfg.width, cfg.height
        c.depth_K[:] = [float(v) for v in scene.depth_K]
        c.color_K[:] = [float(v) for v in scene.color_K]
        c.raw_to_float_depth, c.baseline_fx, c.cell = cfg.raw_to_float_depth, cfg.baseline_fx, cfg.cell
        c.use_depth_residuals, c.use_descriptor_residuals = int(use_depth), int(use_descriptor)
        self.h = self.l.ref_create(C.byref(c), max(scene.pitch, 1))
        if not self.h:
            raise RuntimeError("ref_create failed (no GPU?)")
        self.K = cfg.num_keyframes
        self.n = scene.num_surfels
        self.cf_shape = tuple(scene.cfactor.shape)
        poses = scene.poses_init if poses is None else poses
        for k in range(self.K):
            p = np.ascontiguousarray(poses[k], np.float32)
            rid = self.l.ref_add_keyframe(self.h, np.ascontiguousarray(scene.depth[k]).ctypes.data,
                                          np.ascontiguousarray(scene.normals[k]).ctypes.data,
                                          np.ascontiguousarray(scene.radius[k]).ctypes.data,
                                          np.ascontiguousarray(scene.color[k]).ctypes.data, p.ctypes.data,
                                          float(scene.min_depth[k]), float(scene.max_depth[k]))
            assert rid == k, rid
        s = np.ascontiguousarray(scene.surfels, np.float32)
        assert self.l.ref_set_surfels(self.h, s.ctypes.data, s.strides[0], self.n) == 0
        if scene.depth_a != 0.0 or np.any(scene.cfactor != 0):
            cf = np.ascontiguousarray(scene.cfactor, np.float32)
            self.l.ref_set_depth_params(self.h, float(scene.depth_a), cf.ctypes.data)

    def close(self):
        if self.h:
            self.l.ref_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def pose(self, k):
        p = np.zeros(7, np.float32)
        self.l.ref_get_pose(self.h, k, p.ctypes.data)
        return p

    def poses(self):
        return np.stack([self.pose(k) for k in range(self.K)])

    def set_pose(self, k, pose):
        p = np.ascontiguousarray(pose, np.float32)
        self.l.ref_set_pose(self.h, k, p.ctypes.data)

    def activation(self):
        return np.array([self.l.ref_get_activation(self.h, k) for k in range(self.K)], np.int32)

    def set_activation(self, k, a):
        self.l.ref_set_activation(self.h, k, int(a))

    def create_surfels_for_keyframe(self, k, filter_new_surfels=True):
        return int(self.l.ref_create_surfels_for_keyframe(self.h, int(k), int(filter_new_surfels)))

    def merge_surfels_for_keyframe(self, k):
        return int(self.l.ref_merge_surfels_for_keyframe(self.h, int(k)))

    def compact_surfels(self, free_count, with_active=True):
        return int(self.l.ref_compact_surfels(self.h, int(free_count), int(with_active)))

    def preprocess_frame(self, raw_depth, rgb, sigma_xy=1.5, sigma_inv_depth=0.005, radius_factor=2.0, max_depth=3.0):
        """BadSlam::PreprocessFrame + ComputeMinMaxDepthCUDA with the reference's kernels:
        (depth, normals, radius, rgba, min_depth, max_depth)."""
        raw = np.ascontiguousarray(raw_depth, np.uint16)
        depth, normals, radius = (np.zeros_like(raw) for _ in range(3))
        rgba = None
        if rgb is not None:
            rgb = np.ascontiguousarray(rgb, np.uint8)
            rgba = np.zeros(rgb.shape[:2] + (4,), np.uint8)
        mn, mx = C.c_float(), C.c_float()
        rc = self.l.ref_preprocess_frame(self.h, sigma_xy, sigma_inv_depth, radius_factor, max_depth, raw.ctypes.data,
                                         None if rgb is None else rgb.ctypes.data, depth.ctypes.data, normals.ctypes.data,
                                         radius.ctypes.data, None if rgba is None else rgba.ctypes.data,
                                         C.addressof(mn), C.addressof(mx))
        assert rc > 0, self.l.ref_last_cuda_error()
        return depth, normals, radius, rgba, mn.value, mx.value

    def track_frame_pairwise(self, base_kf, depth, normals, color_rgba, init1, init2=None, num_scales=5, use_pyramid_level_0=True,
                             use_gradmag=False, test_different_initial_estimates=True):
        """BadSlam::RunOdometry + TrackFramePairwise on the reference's own kernels (restated host loop, ref_driver.cu):
        (base_T_frame_estimate, OdometryResult)."""
        d = np.ascontiguousarray(depth, np.uint16)
        n = np.ascontiguousarray(normals, np.uint16)
        c = np.ascontiguousarray(color_rgba, np.uint8)
        p1 = np.ascontiguousarray(init1, np.float32)
        p2 = p1 if init2 is None else np.ascontiguousarray(init2, np.float32)
        out = np.zeros(7, np.float32)
        res = OdometryResult()
        rc = self.l.ref_track_frame_pairwise(self.h, int(base_kf), d.ctypes.data, n.ctypes.data, c.ctypes.data, int(num_scales),
                                             int(use_pyramid_level_0), int(use_gradmag), int(test_different_initial_estimates),
                                             p1.ctypes.data, p2.ctypes.data, out.ctypes.data, C.byref(res))
        assert rc == 0, self.l.ref_last_cuda_error()
        return out, res

    def odometry_level(self, which, scale):
        w, h = C.c_int(), C.c_int()
        assert self.l.ref_odometry_get_level(self.h, which, scale, None, None, None, C.byref(w), C.byref(h)) == 0
        d = np.zeros((h.value, w.value), np.float32)
        n = np.zeros((h.value, w.value), np.uint16)
        c = np.zeros((h.value, w.value), np.uint8)
        assert self.l.ref_odometry_get_level(self.h, which, scale, d.ctypes.data, n.ctypes.data, c.ctypes.data, C.byref(w), C.byref(h)) == 0
        return d, n, c

    def odometry_coeffs(self, scale, pose_a, pose_b=None, use_gradmag=False):
        pa = np.ascontiguousarray(pose_a, np.float32)
        pb = pa if pose_b is None else np.ascontiguousarray(pose_b, np.float32)
        H, b = np.zeros(21, np.float32), np.zeros(6, np.float32)
        cnt, sm = C.c_uint(), C.c_float()
        counts, costs = np.zeros(2, np.uint32), np.zeros(2, np.float32)
        self.l.ref_odometry_coeffs(self.h, int(scale), int(use_gradmag), pa.ctypes.data, pb.ctypes.data, H.ctypes.data, b.ctypes.data,
                                   C.byref(cnt), C.byref(sm), counts.ctypes.data, costs.ctypes.data)
        return H, b, cnt.value, sm.value, counts, costs

    def set_surfels_size(self, n):
        self.l.ref_set_surfels_size(self.h, int(n))

    def surfels_size(self):
        return int(self.l.ref_surfels_size(self.h))

    def end_tasks(self):
        """PerformBASchemeEndTasks (delete + radius update + compaction); returns the number of deleted surfels."""
        return int(self.l.ref_end_tasks(self.h))

    def surfels(self, rows=8):
        n = self.surfels_size()
        out = np.zeros((rows, max(n, 1)), np.float32)
        assert self.l.ref_get_surfels(self.h, out.ctypes.data, out.strides[0], rows) == 0
        return out[:, :n]

    def active(self):
        out = np.zeros(max(self.surfels_size(), self.n, 1), np.uint8)
        assert self.l.ref_get_active(self.h, out.ctypes.data) == 0
        return out[:self.surfels_size()]

    def set_active(self, flags):
        f = np.ascontiguousarray(flags, np.uint8)
        assert self.l.ref_set_active(self.h, f.ctypes.data) == 0

    def pose_coeffs(self, k, pose):
        p = np.ascontiguousarray(pose, np.float32)
        H = np.zeros(21, np.float32)
        b = np.zeros(6, np.float32)
        cnt = C.c_uint()
        cost = C.c_float()
        self.l.ref_pose_coeffs(self.h, k, p.ctypes.data, H.ctypes.data, b.ctypes.data, C.byref(cnt), C.byref(cost))
        return H, b, cnt.value, cost.value

    def estimate_frame_pose(self, k, init):
        p = np.ascontiguousarray(init, np.float32)
        out = np.zeros(7, np.float32)
        conv = C.c_int()
        its = self.l.ref_estimate_frame_pose(self.h, k, p.ctypes.data, out.ctypes.data, C.byref(conv))
        return out, its, bool(conv.value)

    def update_activation(self):
        self.l.ref_update_activation(self.h)

    def optimize_geometry_iteration(self):
        self.l.ref_optimize_geometry_iteration(self.h)

    def optimize_intrinsics(self, depth=True, color=True):
        self.l.ref_optimize_intrinsics(self.h, int(depth), int(color))

    def intrinsics(self):
        d = np.zeros(4, np.float32)
        c = np.zeros(4, np.float32)
        a = C.c_float()
        self.l.ref_get_intrinsics(self.h, d.ctypes.data, c.ctypes.data, C.byref(a))
        return d, c, a.value

    def cfactor(self):
        out = np.zeros(self.cf_shape, np.float32)
        self.l.ref_get_cfactor(self.h, out.ctypes.data)
        return out

    def set_intrinsics(self, depth_K, color_K):
        d = np.ascontiguousarray(depth_K, np.float32)
        c = np.ascontiguousarray(color_K, np.float32)
        self.l.ref_set_intrinsics(self.h, d.ctypes.data, c.ctypes.data)

    def set_depth_params(self, a, cfactor):
        cf = np.ascontiguousarray(cfactor, np.float32)
        self.l.ref_set_depth_params(self.h, float(a), cf.ctypes.data)

    def bundle_adjust(self, optimize_poses=True, optimize_geometry=True, min_iterations=1, max_iterations=10,
                      window_start=0, window_end=None, count_residuals=True, optimize_depth_intrinsics=False,
                      optimize_color_intrinsics=False, end_tasks=True):
        o = BAOptions(int(optimize_poses), int(optimize_geometry), min_iterations, max_iterations, window_start,
                      self.K - 1 if window_end is None else window_end, int(optimize_depth_intrinsics),
                      int(optimize_color_intrinsics), int(end_tasks))
        r = BAResult()
        self.l.ref_bundle_adjust(self.h, C.byref(o), C.byref(r), int(count_residuals))
        return r

    def bundle_adjust_pcg(self, optimize_poses=True, optimize_geometry=True, optimize_depth_intrinsics=False,
                          optimize_color_intrinsics=False, min_iterations=1, max_iterations=1, max_inner_iterations=30,
                          gauge_keyframe=0, end_tasks=True):
        o = PCGOptions(int(optimize_poses), int(optimize_geometry), int(optimize_depth_intrinsics),
                       int(optimize_color_intrinsics), min_iterations, max_iterations, max_inner_iterations, gauge_keyframe,
                       int(end_tasks))
        r = PCGResult()
        self.l.ref_bundle_adjust_pcg(self.h, C.byref(o), C.byref(r))
        return r

    def pcg_debug(self, optimize_poses=True, optimize_geometry=True, optimize_depth_intrinsics=False,
                  optimize_color_intrinsics=False, gauge_keyframe=0):
        o = PCGOptions(int(optimize_poses), int(optimize_geometry), int(optimize_depth_intrinsics),
                       int(optimize_color_intrinsics), 1, 1, 30, gauge_keyframe, 0)
        n = self.l.ref_pcg_debug(self.h, C.byref(o), None, None, None, None, None)
        r, M, p, g = (np.zeros(n, np.float32) for _ in range(4))
        sc = np.zeros(2, np.float32)
        self.l.ref_pcg_debug(self.h, C.byref(o), r.ctypes.data, M.ctypes.data, p.ctypes.data, g.ctypes.data, sc.ctypes.data)
        return r, M, p, g, sc.astype(np.float64)

    def snapshot(self):
        self.l.ref_snapshot(self.h)

    def restore(self):
        self.l.ref_restore(self.h)

    def sync(self):
        self.l.ref_sync(self.h)

    def launch_count(self):
        return int(self.l.ref_launch_count(self.h))


# ---- recorded runs of RefDirectBA ---------------------------------------------------------------------------------------

WHOLE = 256      # arrays up to this many elements are recorded whole
# outputs (method: tuple positions) that the tests only compare bit for bit (`identical`): recorded as their digest alone
DIGEST_ONLY = {"odometry_level": (0, 2), "preprocess_frame": (3,)}


class Sample(np.ndarray):
    """The recorded part of a reference output: `part` indexes it out of an array of `full_shape` whose bytes hash to
    `digest` (sha1)."""


def _part(shape):
    """The fixed, seeded part of an array of `shape` that a recording keeps: an 8 x 32 window of an image, 128 columns of a
    few-row array (the surfel rows: the first and last 16 and 96 between), 192 entries of a vector (32, 128, 32)."""
    if len(shape) >= 2 and shape[0] > 16:
        h, w = shape[:2]
        return np.arange(h // 3, min(h, h // 3 + 8))[:, None], np.arange(w // 3, min(w, w // 3 + 32))[None, :]
    n, edge, mid = shape[-1], (32, 16)[len(shape) > 1], (128, 96)[len(shape) > 1]
    pick = np.random.default_rng(0).choice(np.arange(edge, n - edge), min(n - 2 * edge, mid), replace=False)
    return (slice(None),) * (len(shape) - 1) + (np.concatenate([np.arange(edge), np.sort(pick), np.arange(n - edge, n)]),)


def same_sample(a, b):
    """(a, b) restricted to what the reference output `b` holds of the whole: unchanged unless `b` is a recorded Sample."""
    if not isinstance(b, Sample):
        return a, b
    a = np.asarray(a)
    assert a.shape == b.full_shape, (a.shape, b.full_shape)
    assert b.part is not None, "this reference output is recorded as its digest only (DIGEST_ONLY)"
    return a[b.part], b.view(np.ndarray)


def identical(a, b):
    """Bitwise equality of `a` and the reference output `b` (over the whole array through the digest of a recorded Sample)."""
    a = np.ascontiguousarray(a)
    if not isinstance(b, Sample):
        b = np.ascontiguousarray(b)
        return a.shape == b.shape and a.itemsize == b.itemsize and a.tobytes() == b.tobytes()
    return a.shape == b.full_shape and a.itemsize == b.itemsize and hashlib.sha1(a.tobytes()).hexdigest() == b.digest


def shape_of(b):
    return b.full_shape if isinstance(b, Sample) else np.shape(b)


def _test_id():
    t = os.environ.get("PYTEST_CURRENT_TEST", "no_test").rsplit(" (", 1)[0]
    return re.sub(r"[^A-Za-z0-9_.-]+", "_", t.split("/")[-1].replace(".py::", "__"))


def _pack(a):
    a = np.ascontiguousarray(a)
    return [a.dtype.str, list(a.shape), base64.b64encode(a.tobytes()).decode()]


def _unpack(p):
    return np.frombuffer(base64.b64decode(p[2]), np.dtype(p[0])).reshape(p[1]).copy()


def _encode(v, digest_only=False):
    if v is None:
        return ["n"]
    if isinstance(v, (bool, np.bool_)):
        return ["b", bool(v)]
    if isinstance(v, (int, np.integer)):
        return ["i", int(v)]
    if isinstance(v, (float, np.floating)):
        return ["f", float(v)]
    if isinstance(v, tuple):
        return ["t", [_encode(x) for x in v]]
    if isinstance(v, C.Structure):
        fields = {f: getattr(v, f) for f, _ in v._fields_}
        return ["s", {f: _encode(np.array(x) if isinstance(x, C.Array) else x) for f, x in fields.items()}]
    v = np.ascontiguousarray(v)
    if v.size <= WHOLE:
        return ["a", _pack(v)]
    if digest_only:
        return ["d", v.dtype.str, list(v.shape), hashlib.sha1(v.tobytes()).hexdigest()]
    part = _part(v.shape)
    return ["p", _pack(v[part]), list(v.shape), hashlib.sha1(v.tobytes()).hexdigest(),
            [None if isinstance(i, slice) else _pack(i) for i in part]]


def _decode(spec):
    kind = spec[0]
    if kind == "n":
        return None
    if kind in ("b", "i", "f"):
        return spec[1]
    if kind == "t":
        return tuple(_decode(s) for s in spec[1])
    if kind == "s":
        import types
        return types.SimpleNamespace(**{k: _decode(s) for k, s in spec[1].items()})
    if kind == "a":
        return _unpack(spec[1])
    if kind == "d":
        out = np.zeros(0, np.dtype(spec[1])).view(Sample)
        out.full_shape, out.digest, out.part = tuple(spec[2]), spec[3], None
        return out
    out = _unpack(spec[1]).view(Sample)
    out.full_shape, out.digest = tuple(spec[2]), spec[3]
    out.part = tuple(slice(None) if i is None else _unpack(i) for i in spec[4])
    return out


class _Recording:
    """One test's calls: per RefDirectBA (in construction order), [method, encoded result] per call, as JSON."""
    current = None

    def __init__(self, test_id, directory, replay):
        self.test_id, self.path = test_id, os.path.join(directory, test_id + ".npz")
        self.calls, self.used = [], []
        if replay:
            if not os.path.exists(self.path):
                raise FileNotFoundError(f"no recorded reference run {self.path}: run the test once against the reference's kernels "
                                        "(oracle/build_ref.sh) with BADBA_RECORD_REFERENCE=<dir> and store <dir>/*.npz there")
            with np.load(self.path) as f:
                self.calls = json.loads(f["calls"].tobytes())

    @classmethod
    def get(cls, directory, replay):
        if cls.current is None or cls.current.test_id != _test_id():
            cls.current = cls(_test_id(), directory, replay)
        return cls.current

    def save(self):
        np.savez_compressed(self.path, calls=np.frombuffer(json.dumps(self.calls).encode(), np.uint8))


class _Recorder:
    def __init__(self, live, rec):
        self._live, self._rec, self._i = live, rec, len(rec.calls)
        rec.calls.append([])

    def __getattr__(self, name):
        fn = getattr(self._live, name)

        def call(*args, **kw):
            out = fn(*args, **kw)
            log = self._rec.calls[self._i]
            digest = DIGEST_ONLY.get(name, ())
            log.append([name, ["t", [_encode(x, j in digest) for j, x in enumerate(out)]] if digest else _encode(out)])
            self._rec.save()
            return out
        return call


class _Replay:
    def __init__(self, rec):
        self._rec, self._i, self._n = rec, len(rec.used), 0
        rec.used.append(None)
        assert self._i < len(rec.calls), f"{rec.path}: the recording has {len(rec.calls)} reference instances, the test makes more"

    def __getattr__(self, name):
        def call(*args, **kw):
            log = self._rec.calls[self._i]
            assert self._n < len(log) and log[self._n][0] == name, \
                f"{self._rec.path}: call {self._n} of reference instance {self._i} is {name}, recorded: {log[self._n][0] if self._n < len(log) else 'none'}"
            out = _decode(log[self._n][1])
            self._n += 1
            return out
        return call


def reference(scene, *args, **kw):
    """RefDirectBA(scene, ...) for a test: recorded into $BADBA_RECORD_REFERENCE when that is set (needs the library and a
    GPU), otherwise replayed from tests/golden/reference/<test>.npz."""
    out_dir = os.environ.get("BADBA_RECORD_REFERENCE")
    if out_dir:
        assert available(), f"{LIB_PATH} missing or no GPU (oracle/build_ref.sh)"
        os.makedirs(out_dir, exist_ok=True)
        return _Recorder(RefDirectBA(scene, *args, **kw), _Recording.get(out_dir, replay=False))
    return _Replay(_Recording.get(RECORDED, replay=True))
