"""ctypes binding of libkvfe.so (include/kvfe.h).  There is no fallback: if the library is missing or
no CUDA device is usable, loading / context creation raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

from .params import CameraParams, FrontendParams

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkvfe.so")


class KvfeError(RuntimeError):
    pass


class DepthParams(C.Structure):
    """kvfe_depth_params == CameraParams::DepthParams (include/kimera-vio/frontend/CameraParams.h:131-155)."""
    _fields_ = [("depth_type", C.c_int32), ("virtual_baseline", C.c_float), ("depth_to_meters", C.c_float),
                ("min_depth", C.c_float), ("max_depth", C.c_float)]


class Config(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("batch", C.c_int32), ("max_keypoints", C.c_int32),
        ("klt_win_size", C.c_int32), ("klt_max_iter", C.c_int32), ("klt_max_level", C.c_int32),
        ("klt_eps", C.c_double),
        ("max_feature_track_age", C.c_int32),
        ("min_nr_mono_inliers", C.c_int32), ("min_nr_stereo_inliers", C.c_int32),
        ("ransac_threshold_mono", C.c_double), ("ransac_threshold_stereo", C.c_double),
        ("ransac_max_iterations", C.c_int32),
        ("ransac_probability", C.c_double),
        ("ransac_randomize", C.c_int32),
        ("ransac_use_1point_stereo", C.c_int32), ("ransac_use_2point_mono", C.c_int32),
        ("pose_2d2d_algorithm", C.c_int32),
        ("optical_flow_predictor_type", C.c_int32),
        ("disparity_threshold", C.c_double),
        ("rnd_libstdcxx", C.c_int32),
        ("max_features_per_frame", C.c_int32),
        ("enable_subpixel_corner_refinement", C.c_int32),
        ("subpix_max_iters", C.c_int32),
        ("subpix_epsilon", C.c_double),
        ("subpix_window_size", C.c_int32), ("subpix_zero_zone", C.c_int32),
        ("enable_non_max_suppression", C.c_int32),
        ("non_max_suppression_type", C.c_int32),
        ("min_distance", C.c_int32),
        ("max_nr_keypoints_before_anms", C.c_int32),
        ("nr_horizontal_bins", C.c_int32), ("nr_vertical_bins", C.c_int32),
        ("binning_mask", C.c_uint8 * 64),
        ("quality_level", C.c_double),
        ("block_size", C.c_int32),
        ("use_harris_detector", C.c_int32),
        ("k", C.c_double),
        ("sobel_cpu_tail_start", C.c_int32),
        ("tolerance_template_matching", C.c_double),
        ("templ_cols", C.c_int32), ("templ_rows", C.c_int32), ("stripe_extra_rows", C.c_int32),
        ("min_point_dist", C.c_double), ("max_point_dist", C.c_double),
        ("subpixel_refinement_stereo", C.c_int32),
        ("min_intra_keyframe_time_ns", C.c_int64), ("max_intra_keyframe_time_ns", C.c_int64),
        ("min_number_features", C.c_int32),
        ("use_stereo_tracking", C.c_int32), ("use_ransac", C.c_int32),
        ("max_disparity_since_lkf", C.c_double),
        ("mesh_2d", C.c_int32), ("subdiv_bounding_factor", C.c_float),
        ("optimize_2d2d_pose_from_inliers", C.c_int32), ("optimize_3d3d_pose_from_inliers", C.c_int32),
        ("frontend_type", C.c_int32),
        ("equalize_image", C.c_int32),
        ("depth", DepthParams),
    ]


DISTORTION_MODELS = {"radtan": 0, "equidistant": 1}   # KVFE_DISTORTION_*


class Rig(C.Structure):
    _fields_ = [("K_left", C.c_double * 9), ("K_right", C.c_double * 9),
                ("D_left", C.c_double * 4), ("D_right", C.c_double * 4),
                ("R1", C.c_double * 9), ("R2", C.c_double * 9),
                ("P1", C.c_double * 12), ("P2", C.c_double * 12),
                ("baseline", C.c_double), ("distortion_model", C.c_int32), ("reserved", C.c_int32)]


def make_depth_params(depth_dtype, virtual_baseline=1.0e-2, depth_to_meters=1.0, min_depth=0.0, max_depth=10.0) -> DepthParams:
    """Defaults are the struct defaults of the reference (CameraParams.h:136-145)."""
    dt = np.dtype(depth_dtype)
    if dt not in (np.dtype(np.uint16), np.dtype(np.float32)):
        raise ValueError("depth images are CV_16UC1 or CV_32FC1 (DepthFrame.cpp:29)")
    return DepthParams(1 if dt == np.dtype(np.float32) else 0, float(virtual_baseline), float(depth_to_meters), float(min_depth),
                       float(max_depth))


class PacketHeader(C.Structure):
    _fields_ = [("n", C.c_int32), ("is_keyframe", C.c_int32), ("mono_status", C.c_int32),
                ("stereo_status", C.c_int32), ("n_smart", C.c_int32), ("nr_tracked", C.c_int32),
                ("nr_mono_putatives", C.c_int32), ("nr_mono_inliers", C.c_int32),
                ("nr_stereo_putatives", C.c_int32), ("nr_stereo_inliers", C.c_int32),
                ("nr_valid_rkp", C.c_int32), ("nr_no_left_rect_rkp", C.c_int32),
                ("nr_no_right_rect_rkp", C.c_int32), ("nr_no_depth_rkp", C.c_int32),
                ("nr_failed_arun_rkp", C.c_int32), ("mode", C.c_int32),
                ("frame_id", C.c_int64), ("timestamp", C.c_int64),
                ("lkf_T_k_mono", C.c_double * 12), ("lkf_T_k_stereo", C.c_double * 12),
                ("info_stereo", C.c_double * 9), ("median_disparity", C.c_double),
                ("n_mesh_triangles", C.c_int32), ("reserved", C.c_int32)]


class StereoOut(C.Structure):
    _fields_ = [("left_status", C.c_void_p), ("left_rect_x", C.c_void_p), ("left_rect_y", C.c_void_p),
                ("right_status", C.c_void_p), ("right_rect_x", C.c_void_p), ("right_rect_y", C.c_void_p),
                ("depth", C.c_void_p), ("points_3d", C.c_void_p), ("right_x", C.c_void_p),
                ("right_y", C.c_void_p)]


# packet array names in kvfe_packet_offsets() order, with dtype and per-keypoint width
PACKET_FIELDS = [("kp_x", np.float32, 1), ("kp_y", np.float32, 1), ("landmark", np.int64, 1),
                 ("age", np.int32, 1), ("score", np.float64, 1), ("versor", np.float64, 3),
                 ("left_status", np.int32, 1), ("left_rect_x", np.float32, 1), ("left_rect_y", np.float32, 1),
                 ("right_status", np.int32, 1), ("right_rect_x", np.float32, 1), ("right_rect_y", np.float32, 1),
                 ("depth", np.float64, 1), ("point3d", np.float64, 3), ("right_x", np.float32, 1),
                 ("right_y", np.float32, 1), ("smart_lmk", np.int64, 1), ("smart_uL", np.float64, 1),
                 ("smart_uR", np.float64, 1), ("smart_v", np.float64, 1), ("mesh_tri", np.float32, 6)]
N_PACKET_ARRAYS = len(PACKET_FIELDS)

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise KvfeError("libkvfe.so not built (run `python -m kimera_vio_b200.build`); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    lib.kvfe_last_error.restype = C.c_char_p
    lib.kvfe_last_error.argtypes = [C.c_void_p]
    lib.kvfe_packet_bytes.restype = C.c_size_t
    lib.kvfe_packet_bytes.argtypes = [C.c_void_p]
    lib.kvfe_cuda_stream.restype = C.c_void_p
    lib.kvfe_upload_destroy.restype = None
    lib.kvfe_upload_destroy.argtypes = [C.c_void_p]
    lib.kvfe_frontend_packets_view.restype = C.c_void_p
    lib.kvfe_frontend_packets_view.argtypes = [C.c_void_p]
    lib.kvfe_cuda_stream.argtypes = [C.c_void_p]
    lib.kvfe_config_default.argtypes = [C.POINTER(Config)]
    lib.kvfe_config_default.restype = None
    lib.kvfe_destroy.argtypes = [C.c_void_p]
    lib.kvfe_destroy.restype = None
    _lib = lib
    return lib


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def make_config(p: FrontendParams, width: int, height: int, batch: int = 1, max_keypoints: int = 0,
                rnd_libstdcxx: str = "lemire", sobel_cpu_tail_start: int = -1, mesh_2d: bool = False, mono: bool = False,
                depth: Optional[DepthParams] = None) -> Config:
    """`depth` (make_depth_params): the RGB-D front-end (frontend_type 2) with this depth block."""
    if depth is not None and mono:
        raise ValueError("mono and depth select different front-ends")
    if depth is not None and getattr(p, "use_pnp_tracking", False):
        # PnP (Tracker.cpp:1064-1288) is not built and its status and pose have no place in the packet: refused, not ignored
        raise ValueError("use_pnp_tracking is not supported by the RGB-D front-end")
    c = Config()
    load().kvfe_config_default(C.byref(c))
    c.width, c.height, c.batch, c.max_keypoints = width, height, batch, max_keypoints
    c.klt_win_size, c.klt_max_iter, c.klt_max_level, c.klt_eps = p.klt_win_size, p.klt_max_iter, p.klt_max_level, p.klt_eps
    c.max_feature_track_age = p.max_feature_track_age
    c.min_nr_mono_inliers, c.min_nr_stereo_inliers = p.min_nr_mono_inliers, p.min_nr_stereo_inliers
    c.ransac_threshold_mono, c.ransac_threshold_stereo = p.ransac_threshold_mono, p.ransac_threshold_stereo
    c.ransac_max_iterations, c.ransac_probability = p.ransac_max_iterations, p.ransac_probability
    c.ransac_randomize = int(p.ransac_randomize)
    c.ransac_use_1point_stereo, c.ransac_use_2point_mono = int(p.ransac_use_1point_stereo), int(p.ransac_use_2point_mono)
    c.pose_2d2d_algorithm = p.pose_2d2d_algorithm
    c.optical_flow_predictor_type = p.optical_flow_predictor_type
    c.disparity_threshold = p.disparity_threshold
    c.rnd_libstdcxx = 0 if rnd_libstdcxx == "lemire" else 1
    c.max_features_per_frame = p.max_features_per_frame
    c.enable_subpixel_corner_refinement = int(p.enable_subpixel_corner_refinement)
    c.subpix_max_iters, c.subpix_epsilon = p.subpix_max_iters, p.subpix_epsilon
    c.subpix_window_size, c.subpix_zero_zone = p.subpix_window_size, p.subpix_zero_zone
    c.enable_non_max_suppression = int(p.enable_non_max_suppression)
    c.non_max_suppression_type = p.non_max_suppression_type
    c.min_distance = p.min_distance
    c.max_nr_keypoints_before_anms = p.max_nr_keypoints_before_anms
    c.nr_horizontal_bins, c.nr_vertical_bins = p.nr_horizontal_bins, p.nr_vertical_bins
    m = np.asarray(p.binning_mask, np.float64).reshape(-1)
    for i in range(64):
        c.binning_mask[i] = int(m[i]) if i < m.size else 0
    c.quality_level, c.block_size = p.quality_level, p.block_size
    c.use_harris_detector, c.k = int(p.use_harris_detector), p.k
    c.sobel_cpu_tail_start = sobel_cpu_tail_start
    c.tolerance_template_matching = p.tolerance_template_matching
    c.templ_cols, c.templ_rows, c.stripe_extra_rows = p.templ_cols, p.templ_rows, p.stripe_extra_rows
    c.min_point_dist, c.max_point_dist = p.min_point_dist, p.max_point_dist
    c.subpixel_refinement_stereo = int(p.subpixel_refinement_stereo)
    c.min_intra_keyframe_time_ns, c.max_intra_keyframe_time_ns = p.min_intra_keyframe_time_ns, p.max_intra_keyframe_time_ns
    c.min_number_features = p.min_number_features
    c.use_stereo_tracking, c.use_ransac = int(p.use_stereo_tracking), int(p.use_ransac)
    c.max_disparity_since_lkf = p.max_disparity_since_lkf
    c.mesh_2d = int(mesh_2d)
    c.optimize_2d2d_pose_from_inliers = int(getattr(p, "optimize_2d2d_pose_from_inliers", 0))
    c.optimize_3d3d_pose_from_inliers = int(getattr(p, "optimize_3d3d_pose_from_inliers", 0))
    c.equalize_image = int(p.equalize_image)
    c.frontend_type = 2 if depth is not None else (1 if mono else 0)
    if depth is not None:
        c.depth = depth
    return c


def make_rig(left: CameraParams, right: CameraParams, R1, R2, P1, P2, baseline: float) -> Rig:
    r = Rig()
    r.K_left[:] = list(np.asarray(left.K, np.float64).reshape(-1))
    r.K_right[:] = list(np.asarray(right.K, np.float64).reshape(-1))
    r.D_left[:] = list(np.asarray(left.distortion, np.float64)[:4])
    r.D_right[:] = list(np.asarray(right.distortion, np.float64)[:4])
    r.R1[:] = list(np.asarray(R1, np.float64).reshape(-1))
    r.R2[:] = list(np.asarray(R2, np.float64).reshape(-1))
    r.P1[:] = list(np.asarray(P1, np.float64).reshape(-1))
    r.P2[:] = list(np.asarray(P2, np.float64).reshape(-1))
    r.baseline = float(baseline)
    if left.distortion_model not in DISTORTION_MODELS or right.distortion_model != left.distortion_model:
        raise ValueError("unsupported distortion model %r / %r" % (left.distortion_model, right.distortion_model))
    r.distortion_model = DISTORTION_MODELS[left.distortion_model]
    return r


class Context:
    """Owns a kvfe_ctx*.  All methods map 1:1 onto the C-ABI entry points."""

    def __init__(self, cfg: Config, rig: Rig):
        self.lib = load()
        self.cfg = cfg
        h = C.c_void_p()
        rc = self.lib.kvfe_create(C.byref(cfg), C.byref(rig), C.byref(h))
        if rc != 0:
            raise KvfeError("kvfe_create failed (%d): %s" % (rc, self.lib.kvfe_last_error(None).decode()))
        self.h = h
        self.W, self.H, self.B = cfg.width, cfg.height, cfg.batch
        self.cap = self.lib.kvfe_max_keypoints(self.h)
        self.packet_bytes = int(self.lib.kvfe_packet_bytes(self.h))
        offs = (C.c_size_t * N_PACKET_ARRAYS)()
        self.lib.kvfe_packet_offsets(self.h, offs, N_PACKET_ARRAYS)
        self.packet_offsets = [int(o) for o in offs]

    def close(self):
        if getattr(self, "h", None):
            self.lib.kvfe_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc: int):
        if rc != 0:
            raise KvfeError("libkvfe error %d: %s" % (rc, self.lib.kvfe_last_error(self.h).decode()))

    @property
    def launches(self) -> int:
        return int(self.lib.kvfe_kernel_launches(self.h))

    # ---- stage level --------------------------------------------------------------------------
    def rectify_pair(self, left: np.ndarray, right: np.ndarray):
        left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
        ol, orr = np.empty_like(left), np.empty_like(right)
        self._chk(self.lib.kvfe_rectify_pair(self.h, _p(left), _p(right), C.c_size_t(left.strides[0]), _p(ol), _p(orr),
                                             C.c_size_t(ol.strides[0])))
        return ol, orr

    def rectify_maps(self, cam: int):
        mx, my = np.empty((self.H, self.W), np.float32), np.empty((self.H, self.W), np.float32)
        self._chk(self.lib.kvfe_rectify_maps(self.h, cam, _p(mx), _p(my)))
        return mx, my

    def pyramid(self, img: np.ndarray):
        img = np.ascontiguousarray(img)
        buf = np.empty(self.W * self.H, np.uint8)
        n = C.c_int()
        self._chk(self.lib.kvfe_pyramid(self.h, _p(img), C.c_size_t(img.strides[0]), _p(buf), C.c_size_t(buf.size), C.byref(n)))
        out, o, w, h = [], 0, self.W, self.H
        for _ in range(1, n.value):
            w, h = (w + 1) // 2, (h + 1) // 2
            out.append(buf[o:o + w * h].reshape(h, w).copy())
            o += w * h
        return out

    def min_eigen_response(self, img: np.ndarray) -> np.ndarray:
        img = np.ascontiguousarray(img)
        out = np.empty((self.H, self.W), np.float32)
        self._chk(self.lib.kvfe_min_eigen_response(self.h, _p(img), C.c_size_t(img.strides[0]), _p(out)))
        return out

    def _existing(self, kps, lmks):
        n = len(lmks)
        ex = np.ascontiguousarray(np.asarray([k[0] for k in kps], np.float32)) if n else np.zeros(1, np.float32)
        ey = np.ascontiguousarray(np.asarray([k[1] for k in kps], np.float32)) if n else np.zeros(1, np.float32)
        el = np.ascontiguousarray(np.asarray(lmks, np.int64)) if n else np.zeros(1, np.int64)
        return ex, ey, el, n

    def detect(self, img: np.ndarray, kps=(), lmks=(), need: int = 0):
        img = np.ascontiguousarray(img)
        ex, ey, el, n = self._existing(kps, lmks)
        ox, oy = np.empty(self.cap, np.float32), np.empty(self.cap, np.float32)
        m = C.c_int()
        self._chk(self.lib.kvfe_detect(self.h, _p(img), C.c_size_t(img.strides[0]), _p(ex), _p(ey), _p(el), n, need,
                                       _p(ox), _p(oy), C.byref(m)))
        return np.stack([ox[:m.value], oy[:m.value]], 1)

    def detect_raw(self, img: np.ndarray, kps=(), lmks=()):
        img = np.ascontiguousarray(img)
        ex, ey, el, n = self._existing(kps, lmks)
        cap = self.cfg.max_nr_keypoints_before_anms
        ox, oy, orr = np.empty(cap, np.float32), np.empty(cap, np.float32), np.empty(cap, np.float32)
        m = C.c_int()
        self._chk(self.lib.kvfe_detect_raw(self.h, _p(img), C.c_size_t(img.strides[0]), _p(ex), _p(ey), _p(el), n,
                                           _p(ox), _p(oy), _p(orr), C.byref(m)))
        return np.stack([ox[:m.value], oy[:m.value]], 1), orr[:m.value].copy()

    def track(self, ref_img, cur_img, ref_R_cur, ref_xy):
        ref_img, cur_img = np.ascontiguousarray(ref_img), np.ascontiguousarray(cur_img)
        xy = np.asarray(ref_xy, np.float32).reshape(-1, 2)
        n = len(xy)
        rx, ry = np.ascontiguousarray(xy[:, 0]), np.ascontiguousarray(xy[:, 1])
        R = np.ascontiguousarray(np.asarray(ref_R_cur, np.float64).reshape(9))
        px, py, cx, cy = (np.zeros(max(n, 1), np.float32) for _ in range(4))
        st = np.zeros(max(n, 1), np.uint8)
        self._chk(self.lib.kvfe_track(self.h, _p(ref_img), _p(cur_img), C.c_size_t(ref_img.strides[0]), _p(R), _p(rx),
                                      _p(ry), n, _p(px), _p(py), _p(cx), _p(cy), _p(st)))
        return np.stack([px[:n], py[:n]], 1), np.stack([cx[:n], cy[:n]], 1), st[:n].copy()

    def undistort_keypoints(self, cam: int, use_R: bool, use_P: bool, xy):
        xy = np.asarray(xy, np.float32).reshape(-1, 2)
        n = len(xy)
        x, y = np.ascontiguousarray(xy[:, 0]), np.ascontiguousarray(xy[:, 1])
        ox, oy = np.zeros(max(n, 1), np.float32), np.zeros(max(n, 1), np.float32)
        self._chk(self.lib.kvfe_undistort_keypoints(self.h, cam, int(use_R), int(use_P), _p(x), _p(y), n, _p(ox), _p(oy)))
        return np.stack([ox[:n], oy[:n]], 1)

    def bearing_vectors(self, xy):
        xy = np.asarray(xy, np.float32).reshape(-1, 2)
        n = len(xy)
        x, y = np.ascontiguousarray(xy[:, 0]), np.ascontiguousarray(xy[:, 1])
        v = np.zeros((max(n, 1), 3), np.float64)
        self._chk(self.lib.kvfe_bearing_vectors(self.h, _p(x), _p(y), n, _p(v)))
        return v[:n]

    def sparse_stereo(self, left, right, kps_xy, versors):
        left, right = np.ascontiguousarray(left), np.ascontiguousarray(right)
        xy = np.asarray(kps_xy, np.float32).reshape(-1, 2)
        n = len(xy)
        x, y = np.ascontiguousarray(xy[:, 0]), np.ascontiguousarray(xy[:, 1])
        vs = np.ascontiguousarray(np.asarray(versors, np.float64).reshape(-1, 3))
        res = dict(left_status=np.zeros(n, np.int32), left_rect_x=np.zeros(n, np.float32),
                   left_rect_y=np.zeros(n, np.float32), right_status=np.zeros(n, np.int32),
                   right_rect_x=np.zeros(n, np.float32), right_rect_y=np.zeros(n, np.float32),
                   depth=np.zeros(n, np.float64), points_3d=np.zeros((n, 3), np.float64),
                   right_x=np.zeros(n, np.float32), right_y=np.zeros(n, np.float32))
        so = StereoOut(*[res[k].ctypes.data for k, _ in StereoOut._fields_])
        rl, rr = np.empty_like(left), np.empty_like(right)
        self._chk(self.lib.kvfe_sparse_stereo(self.h, _p(left), _p(right), C.c_size_t(left.strides[0]), _p(x), _p(y),
                                              _p(vs), n, C.byref(so), _p(rl), _p(rr), C.c_size_t(rl.strides[0])))
        res["left_rect"], res["right_rect"] = rl, rr
        return res

    # ---- boundary completion (include/kvfe.h) ----
    def check_rectified_keypoints(self, cam: int, distorted_xy, rectified_xy, tol: float = 2.0):
        d, u = np.ascontiguousarray(distorted_xy, np.float32).reshape(-1, 2), np.ascontiguousarray(rectified_xy, np.float32).reshape(-1, 2)
        n = len(d)
        st, ox, oy = np.zeros(n, np.int32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        dx, dy, ux, uy = (np.ascontiguousarray(a) for a in (d[:, 0], d[:, 1], u[:, 0], u[:, 1]))
        self._chk(self.lib.kvfe_check_rectified_keypoints(self.h, cam, _p(dx), _p(dy), _p(ux), _p(uy), n, C.c_float(tol), _p(st), _p(ox), _p(oy)))
        return st, np.stack([ox, oy], 1)

    def distort_unrectify_keypoints(self, cam: int, status, xy):
        st = np.ascontiguousarray(status, np.int32)
        a = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        n = len(st)
        x, y = np.ascontiguousarray(a[:, 0]), np.ascontiguousarray(a[:, 1])
        ox, oy = np.zeros(n, np.float32), np.zeros(n, np.float32)
        self._chk(self.lib.kvfe_distort_unrectify_keypoints(self.h, cam, _p(st), _p(x), _p(y), n, _p(ox), _p(oy)))
        return np.stack([ox, oy], 1)

    def undistort_rectify_left_keypoints(self, xy):
        a = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        n = len(a)
        x, y = np.ascontiguousarray(a[:, 0]), np.ascontiguousarray(a[:, 1])
        st, ox, oy = np.zeros(n, np.int32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        self._chk(self.lib.kvfe_undistort_rectify_left_keypoints(self.h, _p(x), _p(y), n, _p(st), _p(ox), _p(oy)))
        return st, np.stack([ox, oy], 1)

    def right_keypoints_rectified(self, left_rect: np.ndarray, right_rect: np.ndarray, left_status, left_xy):
        L, R = np.ascontiguousarray(left_rect, np.uint8), np.ascontiguousarray(right_rect, np.uint8)
        ls = np.ascontiguousarray(left_status, np.int32)
        a = np.ascontiguousarray(left_xy, np.float32).reshape(-1, 2)
        n = len(ls)
        x, y = np.ascontiguousarray(a[:, 0]), np.ascontiguousarray(a[:, 1])
        rs, rx, ry = np.zeros(n, np.int32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        self._chk(self.lib.kvfe_right_keypoints_rectified(self.h, _p(L), _p(R), C.c_size_t(L.shape[1]), _p(ls), _p(x), _p(y), n,
                                                          _p(rs), _p(rx), _p(ry)))
        return rs, np.stack([rx, ry], 1)

    def depth_from_rectified_matches(self, left_status, left_x, right_status, right_x):
        ls, rs = np.ascontiguousarray(left_status, np.int32), np.array(right_status, np.int32)
        lx, rx = np.ascontiguousarray(left_x, np.float32), np.ascontiguousarray(right_x, np.float32)
        n = len(ls)
        depth = np.zeros(n, np.float64)
        self._chk(self.lib.kvfe_depth_from_rectified_matches(self.h, _p(ls), _p(lx), _p(rs), _p(rx), n, _p(depth)))
        return rs, depth

    def compute_median_disparity(self, ref_xy, cur_xy, matches):
        r, c = np.ascontiguousarray(ref_xy, np.float32).reshape(-1, 2), np.ascontiguousarray(cur_xy, np.float32).reshape(-1, 2)
        m = np.ascontiguousarray(matches, np.int32).reshape(-1, 2)
        mr, mc = np.ascontiguousarray(m[:, 0]), np.ascontiguousarray(m[:, 1])
        rx, ry, cx, cy = (np.ascontiguousarray(a) for a in (r[:, 0], r[:, 1], c[:, 0], c[:, 1]))
        med, ok = C.c_double(), C.c_int()
        self._chk(self.lib.kvfe_compute_median_disparity(self.h, _p(rx), _p(ry), len(r), _p(cx), _p(cy), len(c), _p(mr), _p(mc), len(m),
                                                         C.byref(med), C.byref(ok)))
        return bool(ok.value), med.value

    def point3_and_covariance(self, left_xy, right_xy, points_3d, R=None):
        l, r = np.ascontiguousarray(left_xy, np.float32).reshape(-1, 2), np.ascontiguousarray(right_xy, np.float32).reshape(-1, 2)
        p = np.ascontiguousarray(points_3d, np.float64).reshape(-1, 3)
        n = len(p)
        lx, rx, ly = np.ascontiguousarray(l[:, 0]), np.ascontiguousarray(r[:, 0]), np.ascontiguousarray(l[:, 1])
        Rm = None if R is None else np.ascontiguousarray(R, np.float64).reshape(9)
        op, oc = np.zeros((n, 3)), np.zeros((n, 3, 3))
        self._chk(self.lib.kvfe_point3_and_covariance(self.h, _p(lx), _p(rx), _p(ly), _p(p), n, _p(Rm), _p(op), _p(oc)))
        return op, oc

    def equalize_hist(self, img: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(img, np.uint8)
        out = np.empty_like(a)
        self._chk(self.lib.kvfe_equalize_hist(self.h, _p(a), C.c_size_t(a.shape[1]), _p(out), C.c_size_t(a.shape[1])))
        return out

    def depth_detection_mask(self, depth: np.ndarray, dp: DepthParams) -> np.ndarray:
        d = np.ascontiguousarray(depth)
        mask = np.empty(d.shape, np.uint8)
        self._chk(self.lib.kvfe_depth_detection_mask(self.h, _p(d), C.c_size_t(d.strides[0]), C.byref(dp), _p(mask), C.c_size_t(mask.shape[1])))
        return mask

    def rgbd_fill_stereo_frame(self, depth: np.ndarray, dp: DepthParams, kps_xy, left_status, left_xy, versors):
        """RgbdFrame::fillStereoFrame: returns (right_status, right_xy, keypoints_depth, keypoints_3d, right_keypoints)."""
        d = np.ascontiguousarray(depth)
        k = np.ascontiguousarray(kps_xy, np.float32).reshape(-1, 2)
        l = np.ascontiguousarray(left_xy, np.float32).reshape(-1, 2)
        st = np.ascontiguousarray(left_status, np.int32)
        v = np.ascontiguousarray(versors, np.float64).reshape(-1, 3)
        n = len(k)
        assert len(l) == n and len(st) == n and len(v) == n
        kx, ky, lx, ly = (np.ascontiguousarray(a) for a in (k[:, 0], k[:, 1], l[:, 0], l[:, 1]))
        rs, rx, ry = np.zeros(n, np.int32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        dep, p3, rkx, rky = np.zeros(n), np.zeros((n, 3)), np.zeros(n, np.float32), np.zeros(n, np.float32)
        self._chk(self.lib.kvfe_rgbd_fill_stereo_frame(self.h, _p(d), C.c_size_t(d.strides[0]), C.byref(dp), _p(kx), _p(ky), _p(st), _p(lx),
                                                       _p(ly), _p(v), n, _p(rs), _p(rx), _p(ry), _p(dep), _p(p3), _p(rkx), _p(rky)))
        return rs, np.stack([rx, ry], 1), dep, p3, np.stack([rkx, rky], 1)

    def mesh_2d(self, kps_xy):
        xy = np.asarray(kps_xy, np.float32).reshape(-1, 2)
        n = len(xy)
        x, y = np.ascontiguousarray(xy[:, 0]), np.ascontiguousarray(xy[:, 1])
        tri = np.zeros((2 * n + 8, 6), np.float32)
        m = C.c_int()
        self._chk(self.lib.kvfe_mesh_2d(self.h, _p(x), _p(y), n, _p(tri), len(tri), C.byref(m)))
        return tri[:min(m.value, len(tri))].copy()

    def ransac_mono(self, f_ref, f_cur, R12=None):
        a = np.ascontiguousarray(np.asarray(f_ref, np.float64).reshape(-1, 3))
        b = np.ascontiguousarray(np.asarray(f_cur, np.float64).reshape(-1, 3))
        n = len(a)
        R = None if R12 is None else np.ascontiguousarray(np.asarray(R12, np.float64).reshape(9))
        inl = np.zeros(max(n, 1), np.int32)
        m, st = C.c_int(), C.c_int()
        pose = np.zeros(12)
        self._chk(self.lib.kvfe_ransac_mono(self.h, _p(a), _p(b), n, _p(R), _p(inl), C.byref(m), _p(pose), C.byref(st)))
        return st.value, pose.reshape(3, 4), inl[:m.value].tolist()

    def ransac_stereo_3pt(self, p_ref, p_cur):
        a = np.ascontiguousarray(np.asarray(p_ref, np.float64).reshape(-1, 3))
        b = np.ascontiguousarray(np.asarray(p_cur, np.float64).reshape(-1, 3))
        n = len(a)
        inl = np.zeros(max(n, 1), np.int32)
        m, st = C.c_int(), C.c_int()
        pose = np.zeros(12)
        self._chk(self.lib.kvfe_ransac_stereo_3pt(self.h, _p(a), _p(b), n, _p(inl), C.byref(m), _p(pose), C.byref(st)))
        return st.value, pose.reshape(3, 4), inl[:m.value].tolist()

    def ransac_stereo_1pt(self, ref_left, ref_right, cur_left, cur_right, p_ref, p_cur, R):
        arrs = [np.ascontiguousarray(np.asarray(v, np.float32).reshape(-1, 2)) for v in (ref_left, ref_right, cur_left, cur_right)]
        a = np.ascontiguousarray(np.asarray(p_ref, np.float64).reshape(-1, 3))
        b = np.ascontiguousarray(np.asarray(p_cur, np.float64).reshape(-1, 3))
        n = len(a)
        Rm = np.ascontiguousarray(np.asarray(R, np.float64).reshape(9))
        inl = np.zeros(max(n, 1), np.int32)
        m, st = C.c_int(), C.c_int()
        pose, info = np.zeros(12), np.zeros(9)
        self._chk(self.lib.kvfe_ransac_stereo_1pt(self.h, _p(arrs[0]), _p(arrs[1]), _p(arrs[2]), _p(arrs[3]), _p(a), _p(b),
                                                  n, _p(Rm), _p(inl), C.byref(m), _p(pose), _p(info), C.byref(st)))
        return st.value, pose.reshape(3, 4), inl[:m.value].tolist(), info.reshape(3, 3)

    # ---- frame level --------------------------------------------------------------------------
    def reset(self):
        self._chk(self.lib.kvfe_frontend_reset(self.h))

    def bind_packets(self, dev_ptr: int):
        """finalize_kernel writes the packets straight into this device buffer (0 / None: the internal one)."""
        self._chk(self.lib.kvfe_frontend_bind_packets(self.h, C.c_void_p(dev_ptr or None)))

    def force_keyframe(self, flags):
        f = np.ascontiguousarray(flags, np.int32)
        assert f.size == self.B
        self._chk(self.lib.kvfe_frontend_force_keyframe(self.h, _p(f)))

    def detect_masked(self, img: np.ndarray, mask: np.ndarray, kps=(), lmks=(), need: int = 0):
        a, m = np.ascontiguousarray(img, np.uint8), np.ascontiguousarray(mask, np.uint8)
        ex, ey, el, ne = self._existing(kps, lmks)
        ox, oy = np.zeros(self.cap, np.float32), np.zeros(self.cap, np.float32)
        n = C.c_int()
        self._chk(self.lib.kvfe_detect_masked(self.h, _p(a), C.c_size_t(a.shape[1]), _p(m), C.c_size_t(m.shape[1]), _p(ex), _p(ey), _p(el),
                                              ne, need, _p(ox), _p(oy), C.byref(n)))
        return np.stack([ox[:n.value], oy[:n.value]], 1)

    def step(self, lefts: Sequence[np.ndarray], rights: Sequence[np.ndarray], timestamps, kf_R_cur,
             want_rectified: bool = False):
        """Host-buffer step (kvfe_frontend_step).  Returns the parsed packets (list of dicts)."""
        B = self.B
        assert len(lefts) == B and len(rights) == B
        lp = (C.c_void_p * B)(*[l.ctypes.data for l in lefts])
        rp = (C.c_void_p * B)(*[r.ctypes.data for r in rights])
        ts = np.ascontiguousarray(np.asarray(timestamps, np.int64))
        Rm = np.ascontiguousarray(np.asarray(kf_R_cur, np.float64).reshape(B, 9))
        buf = np.empty(B * self.packet_bytes, np.uint8)
        rl = rr = None
        rlp = rrp = None
        if want_rectified:
            rl = [np.zeros((self.H, self.W), np.uint8) for _ in range(B)]
            rr = [np.zeros((self.H, self.W), np.uint8) for _ in range(B)]
            rlp = (C.c_void_p * B)(*[a.ctypes.data for a in rl])
            rrp = (C.c_void_p * B)(*[a.ctypes.data for a in rr])
        self._chk(self.lib.kvfe_frontend_step(self.h, lp, rp, C.c_size_t(lefts[0].strides[0]), _p(ts), _p(Rm), _p(buf),
                                              rlp, rrp, C.c_size_t(self.W)))
        pk = self.parse_packets(buf)
        if want_rectified:
            for b in range(B):
                pk[b]["left_rect"], pk[b]["right_rect"] = rl[b], rr[b]
        return pk

    def step_rgbd(self, imgs: Sequence[np.ndarray], depths: Sequence[np.ndarray], timestamps, kf_R_cur):
        """Host-buffer RGB-D step (kvfe_frontend_step_rgbd): intensity images and registered depth images (uint16 or float32,
        the context's depth_type).  Returns the parsed packets."""
        B = self.B
        assert len(imgs) == B and len(depths) == B
        imgs = [np.ascontiguousarray(a, np.uint8) for a in imgs]
        depths = [np.ascontiguousarray(d) for d in depths]
        ip = (C.c_void_p * B)(*[a.ctypes.data for a in imgs])
        dp = (C.c_void_p * B)(*[d.ctypes.data for d in depths])
        ts = np.ascontiguousarray(np.asarray(timestamps, np.int64))
        Rm = np.ascontiguousarray(np.asarray(kf_R_cur, np.float64).reshape(B, 9))
        buf = np.empty(B * self.packet_bytes, np.uint8)
        self._chk(self.lib.kvfe_frontend_step_rgbd(self.h, ip, C.c_size_t(imgs[0].strides[0]), dp, C.c_size_t(depths[0].strides[0]),
                                                   _p(ts), _p(Rm), _p(buf)))
        return self.parse_packets(buf)

    def step_raw(self, lp, rp, pitch, ts, Rm, buf):
        """Zero-overhead variant for benchmarking: pre-built ctypes pointer arrays / numpy buffers."""
        return self.lib.kvfe_frontend_step(self.h, lp, rp, C.c_size_t(pitch), _p(ts), _p(Rm), _p(buf), None, None,
                                           C.c_size_t(0))

    def step_dev(self, left_dev_ptr: int, right_dev_ptr: int, pitch: int, ts: np.ndarray, Rm: np.ndarray):
        return self.lib.kvfe_frontend_step_dev(self.h, C.c_void_p(left_dev_ptr), C.c_void_p(right_dev_ptr),
                                               C.c_size_t(pitch), _p(ts), _p(Rm))

    def step_dev_timed(self, left_dev_ptr: int, right_dev_ptr: int, pitch: int, ts: np.ndarray, Rm: np.ndarray):
        ms = np.zeros(9, np.float32)
        self._chk(self.lib.kvfe_frontend_step_dev_timed(self.h, C.c_void_p(left_dev_ptr), C.c_void_p(right_dev_ptr),
                                                        C.c_size_t(pitch), _p(ts), _p(Rm), _p(ms)))
        return ms

    def submit_raw(self, lp, rp, pitch: int, ts: np.ndarray, Rm: np.ndarray, packets: np.ndarray):
        """kvfe_frontend_submit with prebuilt pointer arrays; `packets` must stay alive until wait()."""
        return self.lib.kvfe_frontend_submit(self.h, lp, rp, C.c_size_t(pitch), _p(ts), _p(Rm), _p(packets))

    def wait(self):
        return self.lib.kvfe_frontend_wait(self.h)

    def packets_view(self) -> np.ndarray:
        """Packets of the last waited step, in place in the context's pinned I/O block (no copy)."""
        ptr = self.lib.kvfe_frontend_packets_view(self.h)
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(self.B * self.packet_bytes,))

    def sync(self):
        self._chk(self.lib.kvfe_sync(self.h))

    def read_packets(self):
        buf = np.empty(self.B * self.packet_bytes, np.uint8)
        self._chk(self.lib.kvfe_frontend_read_packets(self.h, _p(buf)))
        return self.parse_packets(buf)

    def parse_packets(self, buf: np.ndarray):
        out = []
        for b in range(self.B):
            raw = buf[b * self.packet_bytes:(b + 1) * self.packet_bytes]
            h = PacketHeader.from_buffer_copy(raw[:C.sizeof(PacketHeader)].tobytes())
            d = {k: getattr(h, k) for k, _ in PacketHeader._fields_ if not k.startswith("lkf") and k != "info_stereo"}
            d["lkf_T_k_mono"] = np.array(h.lkf_T_k_mono).reshape(3, 4)
            d["lkf_T_k_stereo"] = np.array(h.lkf_T_k_stereo).reshape(3, 4)
            d["info_stereo"] = np.array(h.info_stereo).reshape(3, 3)
            n = h.n
            for (name, dt, w), off in zip(PACKET_FIELDS, self.packet_offsets):
                cnt = (h.n_mesh_triangles if name == "mesh_tri" else h.n_smart if name.startswith("smart") else n) * w
                a = np.frombuffer(raw.tobytes(), dtype=dt, count=cnt, offset=off).copy()
                d[name] = a.reshape(-1, w) if w > 1 else a
            out.append(d)
        return out

    def debug_lk(self, stream: int = 0):
        px, py, nx, ny = (np.zeros(self.cap, np.float32) for _ in range(4))
        st = np.zeros(self.cap, np.uint8)
        n = C.c_int()
        self._chk(self.lib.kvfe_debug_lk(self.h, stream, _p(px), _p(py), _p(nx), _p(ny), _p(st), C.byref(n)))
        m = n.value
        return np.stack([px[:m], py[:m]], 1), np.stack([nx[:m], ny[:m]], 1), st[:m].copy()


# ---- pipeline (kvfe_pipeline_*) ---------------------------------------------------------------------
class PipelineConfig(C.Structure):
    _fields_ = [("n_streams", C.c_int32), ("n_workers", C.c_int32), ("queue_depth", C.c_int32),
                ("output_slots", C.c_int32), ("want_rectified", C.c_int32), ("rotation_mode", C.c_int32),
                ("checksum_outputs", C.c_int32), ("max_in_flight", C.c_int32), ("prefetch", C.c_int32), ("split_graphs", C.c_int32)]


class PipelineOutput(C.Structure):
    _fields_ = [("stream", C.c_int32), ("slot", C.c_int32), ("tag", C.c_uint64),
                ("is_keyframe", C.c_int32), ("n_keypoints", C.c_int32), ("checksum", C.c_uint64),
                ("packet", C.c_void_p), ("rect_left", C.c_void_p), ("rect_right", C.c_void_p)]


class PipelineStats(C.Structure):
    _fields_ = [("frames_pushed", C.c_int64), ("frames_done", C.c_int64), ("graph_launches", C.c_int64),
                ("kernel_launches", C.c_int64), ("launch_seconds", C.c_double), ("staged_copies", C.c_int64)]


def _pipeline_protos(lib):
    if getattr(lib, "_kvfe_pipe_protos", False):
        return
    lib.kvfe_pipeline_create.argtypes = [C.POINTER(Config), C.POINTER(Rig), C.POINTER(PipelineConfig), C.POINTER(C.c_void_p)]
    lib.kvfe_pipeline_destroy.argtypes = [C.c_void_p]
    lib.kvfe_pipeline_destroy.restype = None
    lib.kvfe_pipeline_last_error.argtypes = [C.c_void_p]
    lib.kvfe_pipeline_last_error.restype = C.c_char_p
    lib.kvfe_pipeline_packet_bytes.argtypes = [C.c_void_p]
    lib.kvfe_pipeline_packet_bytes.restype = C.c_size_t
    lib.kvfe_pipeline_packet_offsets.argtypes = [C.c_void_p, C.POINTER(C.c_size_t), C.c_int]
    lib.kvfe_pipeline_max_keypoints.argtypes = [C.c_void_p]
    lib.kvfe_pipeline_push.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int64, C.c_void_p, C.c_uint64]
    lib.kvfe_pipeline_push_rgbd.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int64, C.c_void_p,
                                            C.c_uint64]
    lib.kvfe_pipeline_push_many.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
    lib.kvfe_pipeline_pop.argtypes = [C.c_void_p, C.POINTER(PipelineOutput), C.c_int, C.c_int]
    lib.kvfe_pipeline_release.argtypes = [C.c_void_p, C.POINTER(PipelineOutput), C.c_int]
    lib.kvfe_pipeline_reset.argtypes = [C.c_void_p]
    lib.kvfe_pipeline_force_keyframe.argtypes = [C.c_void_p, C.c_int]
    lib.kvfe_pipeline_get_stats.argtypes = [C.c_void_p, C.POINTER(PipelineStats)]
    lib._kvfe_pipe_protos = True


class Pipeline:
    """kvfe_pipeline: n_streams camera streams behind input / output queues (include/kvfe.h)."""

    def __init__(self, cfg: Config, rig: Rig, n_streams: int, n_workers: int = 0, queue_depth: int = 4,
                 output_slots: int = 4, want_rectified: bool = True, rotation_mode: int = 0,
                 checksum_outputs: bool = False, max_in_flight: int = 0, prefetch: int = 0, split_graphs: int = 0):
        self.lib = load()
        _pipeline_protos(self.lib)
        self.pc = PipelineConfig(n_streams, n_workers, queue_depth, output_slots, int(want_rectified), rotation_mode,
                                 int(checksum_outputs), max_in_flight, prefetch, split_graphs)
        h = C.c_void_p()
        rc = self.lib.kvfe_pipeline_create(C.byref(cfg), C.byref(rig), C.byref(self.pc), C.byref(h))
        if rc != 0:
            raise KvfeError("kvfe_pipeline_create failed (%d): %s" % (rc, self.lib.kvfe_pipeline_last_error(None).decode()))
        self.h = h
        self.n_streams, self.W, self.H = n_streams, cfg.width, cfg.height
        self.B = 1
        self.cap = self.lib.kvfe_pipeline_max_keypoints(self.h)
        self.packet_bytes = int(self.lib.kvfe_pipeline_packet_bytes(self.h))
        offs = (C.c_size_t * N_PACKET_ARRAYS)()
        self.lib.kvfe_pipeline_packet_offsets(self.h, offs, N_PACKET_ARRAYS)
        self.packet_offsets = [int(o) for o in offs]
        self._outs = (PipelineOutput * max(64, 2 * n_streams))()

    def close(self):
        if getattr(self, "h", None):
            self.lib.kvfe_pipeline_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc: int):
        if rc < 0:
            raise KvfeError("kvfe_pipeline error %d: %s" % (rc, self.lib.kvfe_pipeline_last_error(self.h).decode()))
        return rc

    def push(self, stream: int, left_ptr: int, right_ptr: int, pitch: int, timestamp: int, R: np.ndarray, tag: int = 0) -> bool:
        """Returns False when the stream's input queue is full."""
        R = np.ascontiguousarray(np.asarray(R, np.float64).reshape(9))
        rc = self.lib.kvfe_pipeline_push(self.h, stream, left_ptr, right_ptr, pitch, int(timestamp), R.ctypes.data, int(tag))
        if rc == -4:
            return False
        self._chk(rc)
        return True

    def push_rgbd(self, stream: int, img_ptr: int, pitch: int, depth_ptr: int, depth_pitch: int, timestamp: int, R: np.ndarray,
                  tag: int = 0) -> bool:
        """kvfe_pipeline_push_rgbd (pointers to pageable, pinned or device memory).  Returns False when the queue is full."""
        R = np.ascontiguousarray(np.asarray(R, np.float64).reshape(9))
        rc = self.lib.kvfe_pipeline_push_rgbd(self.h, stream, img_ptr, pitch, depth_ptr, depth_pitch, int(timestamp), R.ctypes.data,
                                              int(tag))
        if rc == -4:
            return False
        self._chk(rc)
        return True

    def pop(self, max_n: int = 0, timeout_ms: int = 1000):
        """Raw outputs (ctypes structs, valid until release)."""
        max_n = min(max_n or len(self._outs), len(self._outs))
        n = self._chk(self.lib.kvfe_pipeline_pop(self.h, self._outs, max_n, timeout_ms))
        return [self._outs[i] for i in range(n)]

    def release(self, outs):
        if not outs:
            return
        arr = (PipelineOutput * len(outs))(*outs)
        self._chk(self.lib.kvfe_pipeline_release(self.h, arr, len(outs)))

    def parse(self, out: PipelineOutput, copy_rect: bool = True):
        """Packet of one output as a dict (same fields as Context.parse_packets), plus the rectified pair."""
        raw = np.ctypeslib.as_array(C.cast(out.packet, C.POINTER(C.c_uint8)), shape=(self.packet_bytes,)).copy()
        d = Context.parse_packets(self, raw)[0]
        d["stream"], d["tag"], d["checksum"] = out.stream, out.tag, out.checksum
        if out.rect_left and copy_rect:
            d["left_rect"] = np.ctypeslib.as_array(C.cast(out.rect_left, C.POINTER(C.c_uint8)), shape=(self.H, self.W)).copy()
            d["right_rect"] = np.ctypeslib.as_array(C.cast(out.rect_right, C.POINTER(C.c_uint8)), shape=(self.H, self.W)).copy()
        return d

    def reset(self):
        self._chk(self.lib.kvfe_pipeline_reset(self.h))

    def force_keyframe(self, stream: int):
        self._chk(self.lib.kvfe_pipeline_force_keyframe(self.h, stream))

    def stats(self) -> dict:
        st = PipelineStats()
        self._chk(self.lib.kvfe_pipeline_get_stats(self.h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in PipelineStats._fields_}
