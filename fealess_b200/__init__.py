"""fealess_b200 - B200-native LINE-MOD + ICP hot path of rlvc/FEALESS behind the reference's call surface.

The product is ``libfealess_b200.so`` (hand-written CUDA for sm_100a + a C ABI, ``include/fealess_b200.h``).
This package is the thin Python host side used by the tests and the benchmark: a ctypes binding plus mirrors
of the reference's interface for this path (same names and argument meaning):

    Detector.match                 cup_linemod::Detector::match          linemod/linemod.hpp:324-327
    Detector.addSyntheticTemplate  Detector::addSyntheticTemplate        linemod/linemod.cpp:1636-1642
    detection                      detection()                           ICP/detection.h:9-11
    icpCloudToCloud_Ex             icpCloudToCloud_Ex                    ICP/ICP.h:165-172
    depthTo3d                      cup_d2pc::depthTo3d                   ICP/depth_to_3d.h:12-13
    nonMaximumSuppression          nonMaximumSuppression                 ICP/NMS.h:14-16

There is NO CPU fallback: importing works anywhere, but creating a handle raises unless the CUDA library is
built and a GPU is present.  Nothing here imports ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

from . import synth  # noqa: F401  (synthetic inputs; numpy only)

__all__ = ["lib", "Handle", "Detector", "Match", "detection", "icpCloudToCloud_Ex", "depthTo3d",
           "nonMaximumSuppression", "FealessError", "MATCH_DTYPE", "ICP_RESULT_DTYPE", "library_path"]

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libfealess_b200.so")

FL_OK, FL_ERR_SIZE, FL_ERR_GEOMETRY, FL_ERR_ROI, FL_ERR_FEATURES = 0, -1, -2, -3, -4
FL_ERR_ARG, FL_ERR_CAPACITY, FL_ERR_CUDA, FL_ERR_STATE, FL_ERR_TRAIN = -5, -6, -7, -8, -9
FL_OPT_FE_WAVES, FL_OPT_SPLIT_REFINE, FL_OPT_TRACE, FL_OPT_FE_DEP_TIMEOUT_TEST, FL_OPT_FE_FORCED_WAVES, FL_OPT_SIM_NO_PRUNE = 0, 1, 2, 3, 4, 5
FL_OPT_SIM_ROTATE = 6
FL_DBG_QUANTIZED, FL_DBG_SPREAD, FL_DBG_LINEAR_MEMORY, FL_DBG_SIMILARITY, FL_DBG_STAGED_TRACE, FL_DBG_LAST_COUNTS, FL_DBG_FE_TRACE = 0, 1, 2, 3, 4, 5, 6
FL_DBG_STAGED_ORDER = 7

MATCH_DTYPE = np.dtype([("x", "<i4"), ("y", "<i4"), ("similarity", "<f4"), ("class_idx", "<i4"), ("template_id", "<i4")])
ICP_RESULT_DTYPE = np.dtype([("R", "<f4", (9,)), ("T", "<f4", (3,)), ("dist_mean", "<f4"), ("inlier_ratio", "<f4"),
                             ("iterations", "<i4"), ("n_points", "<i4"), ("status", "<i4")])
# fl_reco_result_t: one recognised object of fl_recognize* (the match it came from, its hypothesis index, [R | T; 0 0 0 1], the ICP record)
RECO_RESULT_DTYPE = np.dtype([("class_idx", "<i4"), ("template_id", "<i4"), ("x", "<i4"), ("y", "<i4"), ("similarity", "<f4"),
                              ("hypothesis", "<i4"), ("world2cam", "<f4", (16,)), ("icp", ICP_RESULT_DTYPE)])
RECO_MAX_HYP = 256                                                # FL_RECO_MAX_HYP

# every symbol include/fealess_b200.h declares (tests check that the built library exports all of them)
EXPORTED_SYMBOLS = [
    "fl_default_params", "fl_create", "fl_destroy", "fl_last_error", "fl_version", "fl_sync", "fl_stream",
    "fl_upload_templates", "fl_set_template_ids", "fl_num_templates", "fl_get_pose_info", "fl_match", "fl_match_device", "fl_match_device_async", "fl_match_wait", "fl_match_fetch",
    "fl_resize_linear", "fl_match_rescaled", "fl_match_shard_device", "fl_sort_unique_device", "fl_sort_unique_blocks_device", "fl_exchange_buffer_bytes", "fl_exchange_sort_unique_device", "fl_exchange_sort_unique_device_async", "fl_match_shard_exchange_device_async", "fl_depth_to_3d", "fl_icp_cloud_to_cloud_ex",
    "fl_detection_batch", "fl_upload_model_depths", "fl_detection_batch_resident", "fl_detection_batch_resident_device", "fl_detection", "fl_nms", "fl_nms_ex", "fl_debug_option", "fl_debug_keep_spread", "fl_debug_force_baseline", "fl_debug_uses_staged", "fl_debug_plan_staged", "fl_debug_get", "fl_debug_icp_trace", "fl_launch_count",
    "fl_profile", "fl_last_stage_ms", "fl_last_icp_ms",
    "fl_group_create", "fl_group_destroy", "fl_group_size", "fl_group_handle", "fl_group_upload_templates", "fl_group_match",
    "fl_match_async", "fl_set_blocking_wait", "fl_match_shard_exchange_async", "fl_pipe_create", "fl_pipe_destroy", "fl_pipe_depth", "fl_pipe_in_flight", "fl_pipe_handle", "fl_pipe_upload_templates",
    "fl_pipe_submit", "fl_pipe_collect", "fl_pipe_match_batch", "fl_pipe_set_exchange", "fl_default_train_params", "fl_add_template",
    "fl_default_reco_params", "fl_set_recognition", "fl_recognize_async", "fl_recognize_wait", "fl_recognize", "fl_pipe_upload_model_depths",
    "fl_pipe_set_recognition", "fl_pipe_submit_recognition", "fl_pipe_collect_recognition",
    "fl_group_create_pipe", "fl_group_depth", "fl_group_in_flight", "fl_group_upload_model_depths", "fl_group_set_recognition",
    "fl_group_submit_recognition", "fl_group_collect_recognition", "fl_group_recognize",
    "fl_pipe_submit_masked", "fl_group_match_masked", "fl_match_shard_exchange_masked_async", "fl_match_shard_exchange_device_masked_async",
    "fl_pipe_set_recognition_sharded",
]


class FealessError(RuntimeError):
    def __init__(self, rc: int, where: str, detail: str = ""):
        super().__init__("%s failed with status %d%s" % (where, rc, (": " + detail) if detail else ""))
        self.rc = rc


class Params(C.Structure):
    _fields_ = [("n_levels", C.c_int32), ("T", C.c_int32 * 8), ("n_modalities", C.c_int32), ("modality_kind", C.c_int32 * 4),
                ("weak_threshold", C.c_float), ("distance_threshold", C.c_int32), ("difference_threshold", C.c_int32),
                ("max_width", C.c_int32), ("max_height", C.c_int32), ("max_candidates", C.c_int32), ("device", C.c_int32)]


class Intrinsics(C.Structure):
    _fields_ = [("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float)]


class Rect(C.Structure):
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("width", C.c_int32), ("height", C.c_int32)]


class IcpParams(C.Structure):
    _fields_ = [("icp_it_thr", C.c_int32), ("dist_mean_thr", C.c_float), ("dist_diff_thr", C.c_float)]


class RecoParams(C.Structure):
    _fields_ = [("threshold", C.c_float), ("icp", IcpParams), ("top_k", C.c_int32), ("per_class", C.c_int32), ("th_obj_dist", C.c_float)]


class RecoSummary(C.Structure):
    _fields_ = [("n_matches", C.c_int32), ("n_hypotheses", C.c_int32), ("n_roi", C.c_int32), ("n_results", C.c_int32)]


def reco_params(threshold: float = 75.0, icp=(10, 0.5, 0.01), top_k: int = 1, per_class: bool = False, th_obj_dist: float = 0.0) -> RecoParams:
    """fl_reco_params_t; the defaults are fl_default_reco_params (the reference's Recognition)."""
    return RecoParams(float(threshold), IcpParams(*icp), int(top_k), int(bool(per_class)), float(th_obj_dist))


def _reco_args(bgr, depth, W, H):
    """(bgr, depth, src_W, src_H, W, H) of fl_recognize*: dense numpy frames; W x H defaults to the frame's own size."""
    b = None if bgr is None else np.ascontiguousarray(bgr, np.uint8)
    d = np.ascontiguousarray(depth, np.uint16)
    sH, sW = d.shape[:2]
    return b, d, sW, sH, int(W or sW), int(H or sH)


def _summary(s: RecoSummary) -> dict:
    return dict(n_matches=s.n_matches, n_hypotheses=s.n_hypotheses, n_roi=s.n_roi, n_results=s.n_results)


def library_path() -> str:
    return _SO


_lib = None


def lib():
    """The loaded C-ABI library.  Raises if it has not been built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise FealessError(FL_ERR_STATE, "load", "%s is missing - run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(nvcc, sm_100a).  fealess_b200 has no CPU fallback." % _SO)
        L = C.CDLL(_SO)
        L.fl_last_error.restype = C.c_char_p
        L.fl_version.restype = C.c_char_p
        L.fl_stream.restype = C.c_void_p
        L.fl_launch_count.restype = C.c_int64
        L.fl_stream.argtypes = [C.c_void_p]
        L.fl_launch_count.argtypes = [C.c_void_p]
        L.fl_exchange_buffer_bytes.restype = C.c_size_t
        _lib = L
    return _lib


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _check(rc: int, where: str, ok=(FL_OK,)):
    if rc not in ok:
        raise FealessError(rc, where, lib().fl_last_error().decode(errors="replace"))
    return rc


def host_masks(masks, M: int, W: int, H: int):
    """``masks=`` of the calls that take a frame in host memory: None / empty = unmasked, else M entries, each None or an H x W array
    (nonzero = keep).  Returns (ctypes array of M pointers or None, the arrays it points into).  A count other than M or a mask of
    another size raises FealessError(FL_ERR_SIZE) - the -1 of Detector::match (linemod.cpp:1374-1377)."""
    if masks is None or len(masks) == 0:
        return None, []
    if len(masks) != M:
        raise FealessError(FL_ERR_SIZE, "masks", "%d masks for %d modalities" % (len(masks), M))
    keep = [None if m is None else np.ascontiguousarray(m, np.uint8) for m in masks]
    for k in keep:
        if k is not None and k.shape != (H, W):
            raise FealessError(FL_ERR_SIZE, "masks", "a mask of shape %s for a %d x %d frame" % (k.shape, W, H))
    return (C.c_void_p * M)(*[None if k is None else k.ctypes.data for k in keep]), keep


def device_masks(masks, M: int):
    """``masks=`` of the calls that take a frame in device memory: None / empty = unmasked, else M device pointers (0 / None = that
    modality unmasked), each a dense W x H u8 image that stays valid until the frame has been waited for.  A count other than M raises
    FealessError(FL_ERR_SIZE)."""
    if masks is None or len(masks) == 0:
        return None
    if len(masks) != M:
        raise FealessError(FL_ERR_SIZE, "masks", "%d masks for %d modalities" % (len(masks), M))
    return (C.c_void_p * M)(*[int(p) if p else None for p in masks])


STAGED_PLAN_FIELDS = ("nw_template", "tpw", "tpc", "n_cta", "block_threads", "phase_rows", "n_rowblocks", "labels_per_phase",
                      "n_phases", "n_buf", "buf_bytes", "halo_bytes", "smem_bytes")


def plan_staged(W: int, H: int, T: int, n_modalities: int, n_templates: int, max_positions: int, n_sm: int) -> Optional[dict]:
    """fl_debug_plan_staged: the staged similarity kernel's plan for a W x H coarsest level with step T (a dict keyed by
    STAGED_PLAN_FIELDS), or None where the planner refuses the geometry and the baseline kernel runs.  No device needed."""
    out = (C.c_int32 * 16)()
    rc = lib().fl_debug_plan_staged(int(W), int(H), int(T), int(n_modalities), int(n_templates), int(max_positions), int(n_sm), out)
    _check(rc, "fl_debug_plan_staged", ok=(0, 1))
    return dict(zip(STAGED_PLAN_FIELDS, out)) if rc == 1 else None


class Handle:
    """Owns one ``fl_handle`` (one GPU, one stream)."""

    def __init__(self, T: Sequence[int] = (5, 8), modality_kind: Sequence[int] = (0, 1), max_width=640, max_height=480,
                 max_candidates=1 << 16, device=0, weak_threshold=10.0, distance_threshold=2000, difference_threshold=50):
        L = lib()
        p = Params()
        L.fl_default_params(C.byref(p))
        p.n_levels = len(T)
        for i, t in enumerate(T):
            p.T[i] = int(t)
        p.n_modalities = len(modality_kind)
        for i, k in enumerate(modality_kind):
            p.modality_kind[i] = int(k)
        p.weak_threshold = weak_threshold
        p.distance_threshold = distance_threshold
        p.difference_threshold = difference_threshold
        p.max_width, p.max_height, p.max_candidates, p.device = max_width, max_height, max_candidates, device
        self.params = p
        self.T = tuple(int(t) for t in T)
        self.L = len(T)
        self._match_out = {}                                      # capacity -> reusable result buffer of match()
        self.M = len(modality_kind)
        self._h = C.c_void_p()
        rc = L.fl_create(C.byref(p), C.byref(self._h))
        if rc != FL_OK:
            self._h = None
            raise FealessError(rc, "fl_create", L.fl_last_error().decode(errors="replace"))

    def close(self):
        if getattr(self, "_h", None):
            lib().fl_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- templates -------------------------------------------------------------------------------
    def upload_templates(self, tset) -> None:
        hdr = np.ascontiguousarray(tset.headers, np.int32)
        ft = np.ascontiguousarray(tset.features, np.int32)
        co = np.ascontiguousarray(tset.class_of, np.int32)
        pose = None if tset.pose13 is None else np.ascontiguousarray(tset.pose13, np.float32)
        _check(lib().fl_upload_templates(self._h, int(tset.n_templates), _p(hdr), _p(ft), int(ft.shape[0]), _p(co), _p(pose)),
               "fl_upload_templates")

    def set_template_ids(self, ids) -> None:
        a = np.ascontiguousarray(ids, np.int32)
        _check(lib().fl_set_template_ids(self._h, _p(a)), "fl_set_template_ids")

    def num_templates(self) -> int:
        return lib().fl_num_templates(self._h)

    def get_pose_info(self, class_idx: int, template_id: int) -> np.ndarray:
        out = np.zeros(13, np.float32)
        _check(lib().fl_get_pose_info(self._h, class_idx, template_id, _p(out)), "fl_get_pose_info")
        return out

    # ---- match -----------------------------------------------------------------------------------
    def match(self, bgr: Optional[np.ndarray], depth: Optional[np.ndarray], threshold: float,
              class_filter: Optional[Sequence[int]] = None, masks: Optional[Sequence[Optional[np.ndarray]]] = None,
              want_quantized: bool = False, capacity: int = 1 << 16):
        """fl_match with host buffers.  Returns (rc, matches[, quantized list]); rc -1 / -2 mirror the reference's
        ``return -1`` / CV_Assert cases instead of raising."""
        ref = depth if depth is not None else bgr
        H, W = ref.shape[:2]
        bgr_c = None if bgr is None else np.ascontiguousarray(bgr, np.uint8)
        dep_c = None if depth is None else np.ascontiguousarray(depth, np.uint16)
        out = self._match_out.get(capacity)                     # result buffer reused across calls (the returned list is a copy)
        if out is None:
            out = self._match_out[capacity] = np.zeros(capacity, MATCH_DTYPE)
        cnt = C.c_int32(0)
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        marr = None
        keep = []
        if masks:
            if len(masks) != self.M:
                return (FL_ERR_SIZE, out[:0]) + (([],) if want_quantized else ())   # linemod.cpp:1374-1377
            keep = [None if m is None else np.ascontiguousarray(m, np.uint8) for m in masks]
            marr = (C.c_void_p * self.M)(*[None if m is None else m.ctypes.data for m in keep])
        qarr, qbufs = None, []
        if want_quantized:
            qbufs = [np.zeros(((H >> l), (W >> l)), np.uint8) for l in range(self.L) for _ in range(self.M)]
            qarr = (C.c_void_p * (self.L * self.M))(*[q.ctypes.data for q in qbufs])
        rc = lib().fl_match(self._h, _p(bgr_c), C.c_size_t(0 if bgr_c is None else W * 3), _p(dep_c),
                            C.c_size_t(0 if dep_c is None else W * 2), W, H, marr, C.c_float(threshold), _p(cf),
                            0 if cf is None else int(cf.size), _p(out), capacity, C.byref(cnt), qarr)
        if rc not in (FL_OK, FL_ERR_SIZE, FL_ERR_GEOMETRY, FL_ERR_CAPACITY):
            _check(rc, "fl_match")
        res = out[:min(cnt.value, capacity)].copy()
        return (rc, res, qbufs) if want_quantized else (rc, res)

    def resize_linear(self, img: np.ndarray, W: int, H: int) -> np.ndarray:
        """fl_resize_linear: ``cv::resize(img, Size(W, H), INTER_LINEAR)`` on the device for an 8UC3 or 16UC1 image."""
        if img.ndim == 3 and img.shape[2] == 3:
            src, kind, out = np.ascontiguousarray(img, np.uint8), 0, np.zeros((H, W, 3), np.uint8)
        elif img.ndim == 2:
            src, kind, out = np.ascontiguousarray(img, np.uint16), 1, np.zeros((H, W), np.uint16)
        else:
            raise ValueError("resize_linear takes H x W x 3 uint8 or H x W uint16 images")
        _check(lib().fl_resize_linear(self._h, _p(src), C.c_size_t(src.strides[0]), src.shape[1], src.shape[0], kind, _p(out), W, H), "fl_resize_linear")
        return out

    def match_rescaled(self, bgr: Optional[np.ndarray], depth: Optional[np.ndarray], W: int, H: int, threshold: float,
                       class_filter: Optional[Sequence[int]] = None, want_depth: bool = False, capacity: int = 1 << 16):
        """fl_match_rescaled: upload the frame at its own size, rescale it to W x H on the device (INTER_LINEAR), match.
        Returns (rc, matches[, rescaled depth])."""
        ref = depth if depth is not None else bgr
        sH, sW = ref.shape[:2]
        bgr_c = None if bgr is None else np.ascontiguousarray(bgr, np.uint8)
        dep_c = None if depth is None else np.ascontiguousarray(depth, np.uint16)
        out = self._match_out.get(capacity)
        if out is None:
            out = self._match_out[capacity] = np.zeros(capacity, MATCH_DTYPE)
        cnt = C.c_int32(0)
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        dout = np.zeros((H, W), np.uint16) if (want_depth and dep_c is not None) else None
        rc = lib().fl_match_rescaled(self._h, _p(bgr_c), C.c_size_t(0 if bgr_c is None else sW * 3), _p(dep_c),
                                     C.c_size_t(0 if dep_c is None else sW * 2), sW, sH, W, H, C.c_float(threshold), _p(cf),
                                     0 if cf is None else int(cf.size), _p(out), capacity, C.byref(cnt), _p(dout))
        if rc not in (FL_OK, FL_ERR_SIZE, FL_ERR_GEOMETRY, FL_ERR_CAPACITY):
            _check(rc, "fl_match_rescaled")
        res = out[:min(cnt.value, capacity)].copy()
        return (rc, res, dout) if want_depth else (rc, res)

    def match_device(self, d_bgr: int, d_depth: int, W: int, H: int, threshold: float, class_filter=None, masks=None) -> None:
        """Frame already in device memory (raw device pointers, dense rows); results stay on the device.  ``masks``: see device_masks."""
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        _check(lib().fl_match_device(self._h, C.c_void_p(d_bgr), C.c_void_p(d_depth), W, H, device_masks(masks, self.M), C.c_float(threshold), _p(cf),
                                     0 if cf is None else int(cf.size)), "fl_match_device")

    def match_device_async(self, d_bgr: int, d_depth: int, W: int, H: int, threshold: float, class_filter=None, masks=None) -> None:
        """Enqueue-only half of ``match_device`` (finish with ``match_wait``): nothing but kernel launches on the handle's stream."""
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        _check(lib().fl_match_device_async(self._h, C.c_void_p(d_bgr), C.c_void_p(d_depth), W, H, device_masks(masks, self.M), C.c_float(threshold), _p(cf),
                                           0 if cf is None else int(cf.size)), "fl_match_device_async")

    def match_async(self, bgr, depth, threshold: float, class_filter=None, masks=None) -> None:
        """fl_match_async: enqueue-only half of ``match`` for a frame in host memory (dense numpy arrays; page-locked ones are read
        by DMA and have to stay alive until ``match_wait``; masks, see host_masks, are copied before this returns)."""
        H, W = (depth if depth is not None else bgr).shape[:2]
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        marr, _keep = host_masks(masks, self.M, W, H)
        _check(lib().fl_match_async(self._h, _p(bgr), C.c_size_t(W * 3), _p(depth), C.c_size_t(W * 2), W, H, marr, C.c_float(threshold), _p(cf),
                                    0 if cf is None else int(cf.size)), "fl_match_async")

    def add_template(self, bgr, depth, mask=None, num_features=None, strong_threshold: float = 55.0, extract_threshold: int = 2,
                     feature_capacity: int = 4096):
        """fl_add_template = Detector::addTemplate on one view (linemod.cpp:1579-1615).  Returns (rc, headers[L*M, 7], features[n, 3],
        bbox[4]); rc is FL_OK or FL_ERR_TRAIN (too few candidates on a level: the reference returns -1)."""
        H, W = (depth if depth is not None else bgr).shape[:2]
        b = None if bgr is None else np.ascontiguousarray(bgr, np.uint8)
        d = None if depth is None else np.ascontiguousarray(depth, np.uint16)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)

        class TrainParams(C.Structure):
            _fields_ = [("num_features", C.c_int32 * 4), ("strong_threshold", C.c_float), ("extract_threshold", C.c_int32)]
        tp = TrainParams()
        lib().fl_default_train_params(C.byref(tp))
        if num_features is not None:
            for i, v in enumerate(num_features):
                tp.num_features[i] = int(v)
        tp.strong_threshold, tp.extract_threshold = float(strong_threshold), int(extract_threshold)
        n_entries = self.L * self.M
        hdr = np.zeros((n_entries, 7), np.int32)
        ft = np.zeros((feature_capacity, 3), np.int32)
        nf = C.c_int32(0)
        bb = np.zeros(4, np.int32)
        rc = lib().fl_add_template(self._h, _p(b), C.c_size_t(W * 3), _p(d), C.c_size_t(W * 2), _p(m), C.c_size_t(W), W, H, C.byref(tp), _p(hdr), _p(ft),
                                   feature_capacity, C.byref(nf), _p(bb))
        if rc not in (FL_OK, FL_ERR_TRAIN):
            _check(rc, "fl_add_template")
        return rc, hdr, ft[:nf.value].copy(), bb

    def match_wait(self) -> None:
        _check(lib().fl_match_wait(self._h), "fl_match_wait")

    def set_blocking_wait(self, enable: bool = True) -> None:
        """fl_set_blocking_wait: sleep instead of spinning while waiting for the GPU (many host threads on few cores)."""
        _check(lib().fl_set_blocking_wait(self._h, int(enable)), "fl_set_blocking_wait")

    def match_fetch(self, capacity: int = 1 << 16, allow_truncated: bool = False) -> np.ndarray:
        """The merged match list of the last frame.  An overflow (a candidate buffer, an exchange block or ``capacity`` too small)
        raises ``FealessError(FL_ERR_CAPACITY)`` unless ``allow_truncated``; ``last_fetch_rc`` keeps the status either way."""
        out = self._match_out.get(capacity)                     # reused across calls (a fresh 1.3 MB buffer per frame costs more than the fetch)
        if out is None:
            out = self._match_out[capacity] = np.zeros(capacity, MATCH_DTYPE)
        cnt = C.c_int32(0)
        ok = (FL_OK, FL_ERR_CAPACITY) if allow_truncated else (FL_OK,)      # FL_ERR_CAPACITY: more candidates than a buffer holds, list incomplete
        self.last_fetch_rc = lib().fl_match_fetch(self._h, _p(out), capacity, C.byref(cnt))
        _check(self.last_fetch_rc, "fl_match_fetch", ok=ok)
        return out[:min(cnt.value, capacity)].copy()

    def match_shard_device(self, d_bgr: int, d_depth: int, W: int, H: int, threshold: float, d_candidates: int, capacity: int,
                           d_count: int, class_filter=None, masks=None) -> None:
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        _check(lib().fl_match_shard_device(self._h, C.c_void_p(d_bgr), C.c_void_p(d_depth), W, H, device_masks(masks, self.M), C.c_float(threshold), _p(cf),
                                           0 if cf is None else int(cf.size), C.c_void_p(d_candidates), capacity, C.c_void_p(d_count)),
               "fl_match_shard_device")

    def sort_unique_device(self, d_in: int, n_lists: int, list_capacity: int, d_n_in: int, d_out: int, out_capacity: int,
                           d_out_count: int) -> None:
        _check(lib().fl_sort_unique_device(self._h, C.c_void_p(d_in), n_lists, list_capacity, C.c_void_p(d_n_in), C.c_void_p(d_out),
                                           out_capacity, C.c_void_p(d_out_count)), "fl_sort_unique_device")

    def sort_unique_blocks_device(self, d_blocks: int, n_blocks: int, capacity: int) -> None:
        _check(lib().fl_sort_unique_blocks_device(self._h, C.c_void_p(d_blocks), n_blocks, capacity), "fl_sort_unique_blocks_device")

    def exchange_sort_unique_device(self, rank: int, world: int, peer_buffers: Sequence[int], capacity: int, d_local_block: int, epoch: int) -> None:
        arr = (C.c_void_p * world)(*[int(p) for p in peer_buffers])
        _check(lib().fl_exchange_sort_unique_device(self._h, rank, world, arr, capacity, C.c_void_p(d_local_block), C.c_uint32(epoch)),
               "fl_exchange_sort_unique_device")

    def exchange_sort_unique_device_async(self, rank: int, world: int, peer_buffers: Sequence[int], capacity: int, d_local_block: int, epoch: int) -> None:
        arr = (C.c_void_p * world)(*[int(p) for p in peer_buffers])
        _check(lib().fl_exchange_sort_unique_device_async(self._h, rank, world, arr, capacity, C.c_void_p(d_local_block), C.c_uint32(epoch)),
               "fl_exchange_sort_unique_device_async")

    def match_shard_exchange_device_async(self, d_bgr: int, d_depth: int, W: int, H: int, threshold: float, rank: int, world: int,
                                          peer_buffers: Sequence[int], capacity: int, d_local_block: int, epoch: int, class_filter=None,
                                          masks=None) -> None:
        """fl_match_shard_exchange_device_masked_async (``masks``: device pointers, see device_masks; None = unmasked)."""
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        arr = peer_buffers if isinstance(peer_buffers, C.Array) else (C.c_void_p * world)(*[int(p) for p in peer_buffers])
        _check(lib().fl_match_shard_exchange_device_masked_async(self._h, C.c_void_p(d_bgr), C.c_void_p(d_depth), W, H, device_masks(masks, self.M),
                                                                 C.c_float(threshold), _p(cf), 0 if cf is None else int(cf.size), rank, world, arr,
                                                                 capacity, C.c_void_p(d_local_block), C.c_uint32(epoch)),
               "fl_match_shard_exchange_device_masked_async")

    def match_shard_exchange_async(self, bgr, depth, threshold: float, rank: int, world: int, peer_buffers: Sequence[int], capacity: int,
                                   d_local_block: int, epoch: int, class_filter=None, masks=None) -> None:
        """fl_match_shard_exchange_masked_async: the frame in HOST memory (numpy arrays, dense rows; page-locked ones are read by DMA and
        have to stay alive until ``match_wait``; masks, see host_masks, are copied before this returns)."""
        H, W = (depth if depth is not None else bgr).shape[:2]
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        marr, _keep = host_masks(masks, self.M, W, H)
        arr = peer_buffers if isinstance(peer_buffers, C.Array) else (C.c_void_p * world)(*[int(p) for p in peer_buffers])
        _check(lib().fl_match_shard_exchange_masked_async(self._h, _p(bgr), C.c_size_t(W * 3), _p(depth), C.c_size_t(W * 2), W, H, marr, C.c_float(threshold),
                                                          _p(cf), 0 if cf is None else int(cf.size), rank, world, arr, capacity, C.c_void_p(d_local_block),
                                                          C.c_uint32(epoch)), "fl_match_shard_exchange_masked_async")

    def sync(self):
        _check(lib().fl_sync(self._h), "fl_sync")

    def stream_ptr(self) -> int:
        return int(lib().fl_stream(self._h) or 0)

    def launch_count(self) -> int:
        return int(lib().fl_launch_count(self._h))

    def profile(self, enable=True):
        _check(lib().fl_profile(self._h, int(enable)), "fl_profile")

    def last_stage_ms(self) -> np.ndarray:
        out = np.zeros(4, np.float32)
        _check(lib().fl_last_stage_ms(self._h, _p(out)), "fl_last_stage_ms")
        return out

    def last_icp_ms(self) -> float:
        v = C.c_float(0)
        _check(lib().fl_last_icp_ms(self._h, C.byref(v)), "fl_last_icp_ms")
        return float(v.value)

    # ---- debug exports ---------------------------------------------------------------------------
    def icp_trace(self, n_hyp: int) -> np.ndarray:
        """fl_debug_icp_trace: [n_hyp, 20] uint64 phase clock of the last ICP batch (after ``profile(True)``)."""
        out = np.zeros((n_hyp, 20), np.uint64)
        _check(lib().fl_debug_icp_trace(self._h, _p(out), n_hyp), "fl_debug_icp_trace")
        return out

    def debug_option(self, option: int, value: int = 1) -> int:
        """fl_debug_option (FL_OPT_*): developer switches of this handle; returns the call's value (query options) or 0."""
        rc = lib().fl_debug_option(self._h, int(option), int(value))
        if rc < 0:
            _check(rc, "fl_debug_option")
        return rc

    def staged_trace(self):
        """FL_DBG_STAGED_TRACE: [n_cta, 8] int64 timeline of the staged similarity kernel of the last frame (needs FL_OPT_TRACE)."""
        buf = np.zeros(1024 * 136 + 8, np.uint64)
        n = lib().fl_debug_get(self._h, FL_DBG_STAGED_TRACE, 0, 0, 0, C.c_void_p(buf.ctypes.data), C.c_size_t(buf.nbytes))
        if n < 0:
            _check(n, "fl_debug_get(FL_DBG_STAGED_TRACE)")
        return buf[:n * 8].reshape(n, 8).astype(np.int64)

    def staged_order(self):
        """FL_DBG_STAGED_ORDER: (order, mass) of the last staged similarity launch: order[q] = the phase CTA 0 visited at step q,
        mass[8 m + l] = the coarsest level's response sum of (modality m, label l) the order was derived from."""
        buf = np.zeros(32 * 4 + 256, np.uint8)
        n = lib().fl_debug_get(self._h, FL_DBG_STAGED_ORDER, 0, 0, 0, C.c_void_p(buf.ctypes.data), C.c_size_t(buf.nbytes))
        if n < 0:
            _check(n, "fl_debug_get(FL_DBG_STAGED_ORDER)")
        return buf[128:128 + n].astype(np.int64), buf[:128].view(np.uint32).astype(np.int64)

    def fe_trace(self):
        """FL_DBG_FE_TRACE: [n_jobs, 6] int64 {kind, CTAs, first start ns, last end ns, summed CTA spans in SM cycles, the same in ns}
        of the front end of the last frame."""
        buf = np.zeros(6 * 64, np.uint64)
        n = lib().fl_debug_get(self._h, FL_DBG_FE_TRACE, 0, 0, 0, C.c_void_p(buf.ctypes.data), C.c_size_t(buf.nbytes))
        if n < 0:
            _check(n, "fl_debug_get(FL_DBG_FE_TRACE)")
        return buf[:n * 6].reshape(n, 6).astype(np.int64)

    def keep_spread(self, enable=True):
        _check(lib().fl_debug_keep_spread(self._h, int(enable)), "fl_debug_keep_spread")

    def force_baseline(self, enable=True):
        _check(lib().fl_debug_force_baseline(self._h, int(enable)), "fl_debug_force_baseline")

    def uses_staged(self) -> bool:
        return lib().fl_debug_uses_staged(self._h) == 1

    def debug_quantized(self, level, modality, W, H, spread=False) -> np.ndarray:
        out = np.zeros((H >> level, W >> level), np.uint8)
        _check(lib().fl_debug_get(self._h, FL_DBG_SPREAD if spread else FL_DBG_QUANTIZED, level, modality, 0, _p(out),
                                  C.c_size_t(out.nbytes)), "fl_debug_get")
        return out

    def debug_lm(self, level, modality, label, W, H) -> np.ndarray:
        T = self.T[level]
        out = np.zeros((T * T, ((W >> level) // T) * ((H >> level) // T)), np.uint8)
        _check(lib().fl_debug_get(self._h, FL_DBG_LINEAR_MEMORY, level, modality, label, _p(out), C.c_size_t(out.nbytes)), "fl_debug_get")
        return out

    def debug_similarity(self, t, W, H) -> np.ndarray:
        l = self.L - 1
        T = self.T[l]
        out = np.zeros(((H >> l) // T, (W >> l) // T), np.uint16)
        _check(lib().fl_debug_get(self._h, FL_DBG_SIMILARITY, t, 0, 0, _p(out), C.c_size_t(out.nbytes)), "fl_debug_get")
        return out

    # ---- ICP -------------------------------------------------------------------------------------
    def depth_to_3d(self, depth: np.ndarray, K) -> np.ndarray:
        d = np.ascontiguousarray(depth, np.uint16)
        H, W = d.shape
        out = np.zeros((H, W, 3), np.float32)
        _check(lib().fl_depth_to_3d(self._h, _p(d), C.c_size_t(W * 2), W, H, Intrinsics(*[float(v) for v in K]), _p(out)), "fl_depth_to_3d")
        return out

    def icp_cloud_to_cloud_ex(self, pts_ref, pts_model, icp_it_thr=4, dist_mean_thr=0.0, dist_diff_thr=0.0) -> np.ndarray:
        pr = np.ascontiguousarray(pts_ref, np.float32).reshape(-1, 3)
        pm = np.ascontiguousarray(pts_model, np.float32).reshape(-1, 3)
        out = np.zeros(1, ICP_RESULT_DTYPE)
        _check(lib().fl_icp_cloud_to_cloud_ex(self._h, _p(pr), pr.shape[0], _p(pm), pm.shape[0],
                                              IcpParams(icp_it_thr, dist_mean_thr, dist_diff_thr), _p(out)), "fl_icp_cloud_to_cloud_ex")
        return out[0]

    def detection_batch(self, ref_depth, K_ref, model_depths: Sequence[np.ndarray], rects_model, rects_ref, r_match=None, t_match=None,
                        icp_it_thr=10, dist_mean_thr=0.5, dist_diff_thr=0.01) -> np.ndarray:
        ref = np.ascontiguousarray(ref_depth, np.uint16)
        H, W = ref.shape
        n = len(model_depths)
        mds = [np.ascontiguousarray(m, np.uint16) for m in model_depths]
        ptrs = (C.c_void_p * max(n, 1))(*[m.ctypes.data for m in mds])
        strides = (C.c_size_t * max(n, 1))(*[m.strides[0] for m in mds])
        rm = np.ascontiguousarray(rects_model, np.int32).reshape(-1, 4)
        rr = np.ascontiguousarray(rects_ref, np.int32).reshape(-1, 4)
        rmat = None if r_match is None else np.ascontiguousarray(r_match, np.float32).reshape(-1, 9)
        tvec = None if t_match is None else np.ascontiguousarray(t_match, np.float32).reshape(-1, 3)
        out = np.zeros(max(n, 1), ICP_RESULT_DTYPE)
        _check(lib().fl_detection_batch(self._h, _p(ref), C.c_size_t(W * 2), W, H, Intrinsics(*[float(v) for v in K_ref]), ptrs, strides,
                                        _p(rm), _p(rr), _p(rmat), _p(tvec), None, n, IcpParams(icp_it_thr, dist_mean_thr, dist_diff_thr),
                                        _p(out)), "fl_detection_batch")
        return out[:n]

    def upload_model_depths(self, model_depths: Sequence[np.ndarray], rects_model) -> None:
        """fl_upload_model_depths: the templates' rendered depth images (u16 mm, all W x H), cropped to rects_model, stay on the device."""
        n = len(model_depths)
        mds = [np.ascontiguousarray(m, np.uint16) for m in model_depths]
        H, W = mds[0].shape if n else (1, 1)
        ptrs = (C.c_void_p * max(n, 1))(*[m.ctypes.data for m in mds])
        strides = (C.c_size_t * max(n, 1))(*[m.strides[0] for m in mds])
        rm = np.ascontiguousarray(rects_model, np.int32).reshape(-1, 4)
        _check(lib().fl_upload_model_depths(self._h, n, ptrs, strides, _p(rm), W, H), "fl_upload_model_depths")

    def detection_batch_resident(self, ref_depth, K_ref, model_index, rects_ref, r_match=None, t_match=None, icp_it_thr=10,
                                 dist_mean_thr=0.5, dist_diff_thr=0.01, frame_size=None) -> np.ndarray:
        """fl_detection_batch_resident.  ``ref_depth=None`` (with ``frame_size=(W, H)``): the depth frame of the last ``match``."""
        if ref_depth is None:
            W, H = frame_size
            ref, stride = None, 0
        else:
            ref = np.ascontiguousarray(ref_depth, np.uint16)
            H, W = ref.shape
            stride = W * 2
        idx = np.ascontiguousarray(model_index, np.int32).reshape(-1)
        n = len(idx)
        rr = np.ascontiguousarray(rects_ref, np.int32).reshape(-1, 4)
        rmat = None if r_match is None else np.ascontiguousarray(r_match, np.float32).reshape(-1, 9)
        tvec = None if t_match is None else np.ascontiguousarray(t_match, np.float32).reshape(-1, 3)
        out = np.zeros(max(n, 1), ICP_RESULT_DTYPE)
        _check(lib().fl_detection_batch_resident(self._h, _p(ref), C.c_size_t(stride), W, H, Intrinsics(*[float(v) for v in K_ref]), _p(idx),
                                                 _p(rr), _p(rmat), _p(tvec), n, IcpParams(icp_it_thr, dist_mean_thr, dist_diff_thr), _p(out)),
               "fl_detection_batch_resident")
        return out[:n]

    def detection_batch_resident_device(self, d_ref_depth: int, W: int, H: int, K_ref, model_index, rects_ref, r_match=None, t_match=None,
                                        icp_it_thr=10, dist_mean_thr=0.5, dist_diff_thr=0.01) -> np.ndarray:
        """fl_detection_batch_resident_device: the reference depth frame is a device pointer (dense W x H u16)."""
        idx = np.ascontiguousarray(model_index, np.int32).reshape(-1)
        n = len(idx)
        rr = np.ascontiguousarray(rects_ref, np.int32).reshape(-1, 4)
        rmat = None if r_match is None else np.ascontiguousarray(r_match, np.float32).reshape(-1, 9)
        tvec = None if t_match is None else np.ascontiguousarray(t_match, np.float32).reshape(-1, 3)
        out = np.zeros(max(n, 1), ICP_RESULT_DTYPE)
        _check(lib().fl_detection_batch_resident_device(self._h, C.c_void_p(d_ref_depth), W, H, Intrinsics(*[float(v) for v in K_ref]), _p(idx),
                                                        _p(rr), _p(rmat), _p(tvec), n, IcpParams(icp_it_thr, dist_mean_thr, dist_diff_thr), _p(out)),
               "fl_detection_batch_resident_device")
        return out[:n]

    def nms(self, t3, n_model_pts, icp_dist, th_obj_dist) -> np.ndarray:
        t = np.ascontiguousarray(t3, np.float32).reshape(-1, 3)
        nm = np.ascontiguousarray(n_model_pts, np.int32)
        dd = np.ascontiguousarray(icp_dist, np.float32)
        out = np.zeros(max(len(nm), 1), np.int32)
        n = lib().fl_nms(self._h, _p(t), _p(nm), _p(dd), len(nm), C.c_float(th_obj_dist), _p(out))
        if n < 0:
            _check(n, "fl_nms")
        return out[:n].copy()

    # ---- Recognition on the device ---------------------------------------------------------------
    def set_recognition(self, crop_of_template, pose12=None, params: Optional[RecoParams] = None) -> None:
        """fl_set_recognition: crop index per uploaded template (-1 = none), pose table (n_templates x 12, None = the uploaded pose13)."""
        crop = np.ascontiguousarray(crop_of_template, np.int32)
        pose = None if pose12 is None else np.ascontiguousarray(pose12, np.float32).reshape(-1, 12)
        _check(lib().fl_set_recognition(self._h, C.byref(params or reco_params()), _p(crop), _p(pose)), "fl_set_recognition")

    def recognize_async(self, bgr, depth, K, W: Optional[int] = None, H: Optional[int] = None) -> None:
        """fl_recognize_async: the frame (rescaled on the device to W x H when that differs) is matched, refined and suppressed in one
        enqueue.  The arrays must stay alive until ``recognize_wait`` (page-locked ones are read by DMA)."""
        b, d, sW, sH, W, H = _reco_args(bgr, depth, W, H)
        _check(lib().fl_recognize_async(self._h, _p(b), C.c_size_t(sW * 3), _p(d), C.c_size_t(sW * 2), sW, sH, W, H,
                                        Intrinsics(*[float(v) for v in K])), "fl_recognize_async")
        self._reco_keep = (b, d)

    def recognize_wait(self, capacity: int = RECO_MAX_HYP):
        """(rc, results RECO_RESULT_DTYPE, summary dict); rc is FL_OK or FL_ERR_CAPACITY (truncated, or a candidate overflow: no results)."""
        out = np.zeros(max(capacity, 1), RECO_RESULT_DTYPE)
        s = RecoSummary()
        rc = lib().fl_recognize_wait(self._h, _p(out), int(capacity), C.byref(s))
        self._reco_keep = None
        if rc not in (FL_OK, FL_ERR_CAPACITY):
            _check(rc, "fl_recognize_wait")
        return rc, out[:min(s.n_results, capacity)].copy(), _summary(s)

    def recognize(self, bgr, depth, K, W: Optional[int] = None, H: Optional[int] = None, capacity: int = RECO_MAX_HYP):
        self.recognize_async(bgr, depth, K, W, H)
        return self.recognize_wait(capacity)


class Group:
    """fl_group: Detector::match over N handles of this process (``devices`` may repeat a device), templates sharded gid % N.  With
    ``depth`` > 1 (fl_group_create_pipe) up to ``depth`` recognition frames are in flight; handle i = slot * N + member."""

    def __init__(self, devices: Sequence[int], T: Sequence[int] = (5, 8), modality_kind: Sequence[int] = (0, 1), max_width=640, max_height=480,
                 exchange_capacity: int = 2048, depth: int = 1):
        L = lib()
        p = Params()
        L.fl_default_params(C.byref(p))
        p.n_levels = len(T)
        for i, t in enumerate(T):
            p.T[i] = int(t)
        p.n_modalities = len(modality_kind)
        for i, k in enumerate(modality_kind):
            p.modality_kind[i] = int(k)
        p.max_width, p.max_height = max_width, max_height
        self._g = C.c_void_p()
        dv = np.ascontiguousarray(devices, np.int32)
        rc = L.fl_group_create_pipe(C.byref(p), _p(dv), len(dv), exchange_capacity, int(depth), C.byref(self._g))
        if rc != FL_OK:
            self._g = None
            raise FealessError(rc, "fl_group_create_pipe", L.fl_last_error().decode(errors="replace"))
        self.n, self.depth, self.M = len(dv), int(depth), len(modality_kind)
        self._keep = {}                                          # frames in flight: the arrays the DMA reads stay referenced
        self._seq = 0

    def close(self):
        if getattr(self, "_g", None):
            lib().fl_group_destroy(self._g)
            self._g = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def _handle(self, i: int) -> C.c_void_p:
        L = lib()
        L.fl_group_handle.restype = C.c_void_p
        hp = L.fl_group_handle(self._g, int(i))
        if not hp:
            raise FealessError(FL_ERR_ARG, "fl_group_handle")
        return C.c_void_p(hp)

    def member_option(self, i: int, option: int, value: int = 1) -> int:
        """fl_debug_option on handle ``i`` (fl_group_handle: slot * N + member)."""
        rc = lib().fl_debug_option(self._handle(i), int(option), int(value))
        if rc < 0:
            _check(rc, "fl_debug_option")
        return rc

    def launch_counts(self) -> np.ndarray:
        """fl_launch_count of every handle, shape (depth, N)."""
        return np.array([int(lib().fl_launch_count(self._handle(i))) for i in range(self.n * self.depth)], np.int64).reshape(self.depth, self.n)

    def in_flight(self) -> int:
        return int(lib().fl_group_in_flight(self._g))

    def upload_templates(self, tset) -> None:
        hdr = np.ascontiguousarray(tset.headers, np.int32)
        ft = np.ascontiguousarray(tset.features, np.int32)
        co = np.ascontiguousarray(tset.class_of, np.int32)
        pose = np.ascontiguousarray(tset.pose13, np.float32)
        _check(lib().fl_group_upload_templates(self._g, tset.n_templates, _p(hdr), _p(ft), ft.shape[0], _p(co), _p(pose)), "fl_group_upload_templates")

    def match(self, bgr, depth, threshold: float, class_filter=None, capacity: int = 1 << 16, masks=None):
        """fl_group_match_masked: (rc, merged list); ``masks`` as in ``Handle.match`` (a wrong count or size gives rc FL_ERR_SIZE)."""
        H, W = depth.shape[:2]
        b = np.ascontiguousarray(bgr, np.uint8)
        d = np.ascontiguousarray(depth, np.uint16)
        out = np.zeros(capacity, MATCH_DTYPE)
        try:
            marr, _keep = host_masks(masks, self.M, W, H)
        except FealessError as e:
            return e.rc, out[:0]
        cnt = C.c_int32(0)
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        rc = lib().fl_group_match_masked(self._g, _p(b), C.c_size_t(W * 3), _p(d), C.c_size_t(W * 2), W, H, marr, C.c_float(threshold), _p(cf),
                                         0 if cf is None else int(cf.size), _p(out), capacity, C.byref(cnt))
        if rc not in (FL_OK, FL_ERR_CAPACITY):
            _check(rc, "fl_group_match_masked")
        return rc, out[:min(cnt.value, capacity)].copy()

    # ---- Recognition over the group ---------------------------------------------------------------
    def upload_model_depths(self, model_depths: Sequence[np.ndarray], rects_model) -> None:
        """fl_group_upload_model_depths: ``Handle.upload_model_depths`` on every slot of every member."""
        n = len(model_depths)
        mds = [np.ascontiguousarray(m, np.uint16) for m in model_depths]
        H, W = mds[0].shape if n else (1, 1)
        ptrs = (C.c_void_p * max(n, 1))(*[m.ctypes.data for m in mds])
        strides = (C.c_size_t * max(n, 1))(*[m.strides[0] for m in mds])
        rm = np.ascontiguousarray(rects_model, np.int32).reshape(-1, 4)
        _check(lib().fl_group_upload_model_depths(self._g, n, ptrs, strides, _p(rm), W, H), "fl_group_upload_model_depths")

    def set_recognition(self, crop_of_template, pose12=None, params: Optional[RecoParams] = None) -> None:
        """fl_group_set_recognition: crop index and pose of every template of the whole set (order of ``upload_templates``)."""
        crop = np.ascontiguousarray(crop_of_template, np.int32)
        pose = None if pose12 is None else np.ascontiguousarray(pose12, np.float32).reshape(-1, 12)
        _check(lib().fl_group_set_recognition(self._g, C.byref(params or reco_params()), _p(crop), _p(pose)), "fl_group_set_recognition")

    def submit_recognition(self, bgr, depth, K, W: Optional[int] = None, H: Optional[int] = None) -> None:
        """fl_group_submit_recognition (host frame; page-locked arrays are read by DMA while in flight, so they are kept referenced)."""
        b, d, sW, sH, W, H = _reco_args(bgr, depth, W, H)
        _check(lib().fl_group_submit_recognition(self._g, _p(b), C.c_size_t(sW * 3), _p(d), C.c_size_t(sW * 2), sW, sH, W, H,
                                                 Intrinsics(*[float(v) for v in K])), "fl_group_submit_recognition")
        self._keep[self._seq % self.depth] = (b, d)
        self._seq += 1

    def collect_recognition(self, capacity: int = RECO_MAX_HYP):
        """(rc, results, summary) of the oldest frame in flight, as ``Handle.recognize_wait``."""
        out = np.zeros(max(capacity, 1), RECO_RESULT_DTYPE)
        s = RecoSummary()
        rc = lib().fl_group_collect_recognition(self._g, _p(out), int(capacity), C.byref(s))
        if rc not in (FL_OK, FL_ERR_CAPACITY):
            _check(rc, "fl_group_collect_recognition")
        return rc, out[:min(s.n_results, capacity)].copy(), _summary(s)

    def recognize(self, bgr, depth, K, W: Optional[int] = None, H: Optional[int] = None, capacity: int = RECO_MAX_HYP):
        """fl_group_recognize: one frame, submitted and collected (nothing else may be in flight)."""
        b, d, sW, sH, W, H = _reco_args(bgr, depth, W, H)
        out = np.zeros(max(capacity, 1), RECO_RESULT_DTYPE)
        s = RecoSummary()
        rc = lib().fl_group_recognize(self._g, _p(b), C.c_size_t(sW * 3), _p(d), C.c_size_t(sW * 2), sW, sH, W, H,
                                      Intrinsics(*[float(v) for v in K]), _p(out), int(capacity), C.byref(s))
        if rc not in (FL_OK, FL_ERR_CAPACITY):
            _check(rc, "fl_group_recognize")
        return rc, out[:min(s.n_results, capacity)].copy(), _summary(s)


class Pipe:
    """fl_pipe: Detector::match over a stream of frames with ``depth`` frames in flight on one GPU; lists come back in submission
    order and equal ``Handle.match``'s."""

    def __init__(self, depth: int = 3, T: Sequence[int] = (5, 8), modality_kind: Sequence[int] = (0, 1), max_width=640, max_height=480, device: int = 0,
                 max_candidates: Optional[int] = None):
        L = lib()
        p = Params()
        L.fl_default_params(C.byref(p))
        p.n_levels = len(T)
        for i, t in enumerate(T):
            p.T[i] = int(t)
        p.n_modalities = len(modality_kind)
        for i, k in enumerate(modality_kind):
            p.modality_kind[i] = int(k)
        p.max_width, p.max_height, p.device = max_width, max_height, device
        if max_candidates:
            p.max_candidates = int(max_candidates)
        self._p = C.c_void_p()
        rc = L.fl_pipe_create(C.byref(p), int(depth), C.byref(self._p))
        if rc != FL_OK:
            self._p = None
            raise FealessError(rc, "fl_pipe_create", L.fl_last_error().decode(errors="replace"))
        self.depth, self.M = int(depth), len(modality_kind)
        self._keep = {}                                          # frames in flight: the arrays the DMA reads stay referenced
        self._seq = 0
        self._out = {}

    def close(self):
        if getattr(self, "_p", None):
            lib().fl_pipe_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def in_flight(self) -> int:
        return int(lib().fl_pipe_in_flight(self._p))

    def upload_templates(self, tset) -> None:
        hdr = np.ascontiguousarray(tset.headers, np.int32)
        ft = np.ascontiguousarray(tset.features, np.int32)
        co = np.ascontiguousarray(tset.class_of, np.int32)
        pose = np.ascontiguousarray(tset.pose13, np.float32)
        _check(lib().fl_pipe_upload_templates(self._p, tset.n_templates, _p(hdr), _p(ft), ft.shape[0], _p(co), _p(pose)), "fl_pipe_upload_templates")

    def set_template_ids(self, template_ids) -> None:
        """fl_set_template_ids on every slot's handle (global per-class ids of a template shard)."""
        ids = np.ascontiguousarray(template_ids, np.int32)
        L = lib()
        L.fl_pipe_handle.restype = C.c_void_p
        for i in range(self.depth):
            _check(L.fl_set_template_ids(C.c_void_p(L.fl_pipe_handle(self._p, i)), _p(ids)), "fl_set_template_ids")

    def set_exchange(self, rank: int, world: int, capacity: int, peer_buffers: Sequence[Sequence[int]], local_blocks: Sequence[int]) -> None:
        """fl_pipe_set_exchange: ``peer_buffers[i][r]`` = address of rank r's exchange buffer of slot i in this process,
        ``local_blocks[i]`` = slot i's candidate block (device memory, capacity + 1 records)."""
        flat = [int(peer_buffers[i][r]) for i in range(self.depth) for r in range(world)]
        pa = (C.c_void_p * len(flat))(*flat)
        ba = (C.c_void_p * self.depth)(*[int(b) for b in local_blocks])
        _check(lib().fl_pipe_set_exchange(self._p, int(rank), int(world), int(capacity), pa, ba), "fl_pipe_set_exchange")

    def launch_count(self) -> int:
        L = lib()
        L.fl_pipe_handle.restype = C.c_void_p
        L.fl_launch_count.restype = C.c_int64
        return sum(int(L.fl_launch_count(C.c_void_p(L.fl_pipe_handle(self._p, i)))) for i in range(self.depth))

    def submit(self, bgr, depth, threshold: float, class_filter=None, masks=None) -> None:
        """Host frame (numpy arrays; page-locked ones are read by DMA while in flight).  ``masks``: see host_masks (copied before this
        returns)."""
        H, W = (depth if depth is not None else bgr).shape[:2]
        b = None if bgr is None else np.ascontiguousarray(bgr, np.uint8)
        d = None if depth is None else np.ascontiguousarray(depth, np.uint16)
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        marr, _keep = host_masks(masks, self.M, W, H)
        _check(lib().fl_pipe_submit_masked(self._p, _p(b), C.c_size_t(W * 3), _p(d), C.c_size_t(W * 2), W, H, marr, C.c_float(threshold), _p(cf),
                                           0 if cf is None else int(cf.size), 0), "fl_pipe_submit_masked")
        self._keep[self._seq % self.depth] = (b, d)
        self._seq += 1

    def submit_device(self, d_bgr: int, d_depth: int, W: int, H: int, threshold: float, class_filter=None, d_masks=None) -> None:
        """Device frame (dense rows); ``d_masks``: see device_masks."""
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        _check(lib().fl_pipe_submit_masked(self._p, C.c_void_p(d_bgr), C.c_size_t(W * 3), C.c_void_p(d_depth), C.c_size_t(W * 2), W, H,
                                           device_masks(d_masks, self.M), C.c_float(threshold), _p(cf), 0 if cf is None else int(cf.size), 1),
               "fl_pipe_submit_masked")
        self._seq += 1

    def collect(self, capacity: int = 1 << 14, copy: bool = True):
        """(rc, matches) of the oldest frame in flight; rc is FL_OK or FL_ERR_CAPACITY (truncated list)."""
        out = self._out.get(capacity)
        if out is None:
            out = self._out[capacity] = np.zeros(capacity, MATCH_DTYPE)
        cnt = C.c_int32(0)
        rc = lib().fl_pipe_collect(self._p, _p(out), capacity, C.byref(cnt))
        if rc not in (FL_OK, FL_ERR_CAPACITY):
            _check(rc, "fl_pipe_collect")
        m = out[:min(cnt.value, capacity)]
        return rc, (m.copy() if copy else m)

    def match_batch(self, frames, threshold: float, class_filter=None, capacity_per_frame: int = 1 << 12, out=None, copy: bool = True):
        """``frames``: sequence of (bgr, depth) numpy pairs of one geometry.  Returns (rc, [matches per frame]).  ``out`` (optional):
        a reusable MATCH_DTYPE array of at least len(frames) * capacity_per_frame records; ``copy=False`` returns views into it."""
        n = len(frames)
        if n == 0:
            return FL_OK, []
        H, W = frames[0][1].shape[:2]
        bs = [np.ascontiguousarray(f[0], np.uint8) for f in frames]
        ds = [np.ascontiguousarray(f[1], np.uint16) for f in frames]
        pb = (C.c_void_p * n)(*[x.ctypes.data for x in bs])
        pd = (C.c_void_p * n)(*[x.ctypes.data for x in ds])
        if out is None:
            out = np.zeros(n * capacity_per_frame, MATCH_DTYPE)
        elif out.dtype != MATCH_DTYPE or out.size < n * capacity_per_frame or not out.flags.c_contiguous:
            raise ValueError("match_batch: `out` must be a contiguous MATCH_DTYPE array of at least len(frames) * capacity_per_frame records")
        counts = np.zeros(n, np.int32)
        cf = None if not class_filter else np.ascontiguousarray(class_filter, np.int32)
        rc = lib().fl_pipe_match_batch(self._p, n, pb, C.c_size_t(W * 3), pd, C.c_size_t(W * 2), W, H, C.c_float(threshold), _p(cf), 0 if cf is None else int(cf.size), 0,
                                       _p(out), capacity_per_frame, _p(counts))
        if rc not in (FL_OK, FL_ERR_CAPACITY):
            _check(rc, "fl_pipe_match_batch")
        views = [out[f * capacity_per_frame:f * capacity_per_frame + min(int(counts[f]), capacity_per_frame)] for f in range(n)]
        return rc, ([v.copy() for v in views] if copy else views)

    # ---- Recognition over the pipe ----------------------------------------------------------------
    def upload_model_depths(self, model_depths: Sequence[np.ndarray], rects_model) -> None:
        """fl_pipe_upload_model_depths: ``Handle.upload_model_depths`` on every slot."""
        n = len(model_depths)
        mds = [np.ascontiguousarray(m, np.uint16) for m in model_depths]
        H, W = mds[0].shape if n else (1, 1)
        ptrs = (C.c_void_p * max(n, 1))(*[m.ctypes.data for m in mds])
        strides = (C.c_size_t * max(n, 1))(*[m.strides[0] for m in mds])
        rm = np.ascontiguousarray(rects_model, np.int32).reshape(-1, 4)
        _check(lib().fl_pipe_upload_model_depths(self._p, n, ptrs, strides, _p(rm), W, H), "fl_pipe_upload_model_depths")

    def set_recognition(self, crop_of_template, pose12=None, params: Optional[RecoParams] = None) -> None:
        """fl_pipe_set_recognition: ``Handle.set_recognition`` on every slot."""
        crop = np.ascontiguousarray(crop_of_template, np.int32)
        pose = None if pose12 is None else np.ascontiguousarray(pose12, np.float32).reshape(-1, 12)
        _check(lib().fl_pipe_set_recognition(self._p, C.byref(params or reco_params()), _p(crop), _p(pose)), "fl_pipe_set_recognition")

    def set_recognition_sharded(self, tset, crop_of_template, pose12=None, params: Optional[RecoParams] = None) -> None:
        """fl_pipe_set_recognition_sharded (a template-sharded pipe): ``tset`` = the WHOLE set the shards were cut from, crop index and
        pose of every template of it (order of the set; pose12 None = the first 12 floats of the set's pose13)."""
        hdr = np.ascontiguousarray(tset.headers, np.int32)
        co = np.ascontiguousarray(tset.class_of, np.int32)
        crop = np.ascontiguousarray(crop_of_template, np.int32)
        pose = np.ascontiguousarray(np.asarray(tset.pose13, np.float32).reshape(-1, 13)[:, :12] if pose12 is None else pose12, np.float32).reshape(-1, 12)
        _check(lib().fl_pipe_set_recognition_sharded(self._p, C.byref(params or reco_params()), int(tset.n_templates), _p(hdr), _p(co), _p(crop), _p(pose)),
               "fl_pipe_set_recognition_sharded")

    def submit_recognition(self, bgr, depth, K, W: Optional[int] = None, H: Optional[int] = None) -> None:
        """fl_pipe_submit_recognition (host frame; page-locked arrays are read by DMA while in flight, so they are kept referenced)."""
        b, d, sW, sH, W, H = _reco_args(bgr, depth, W, H)
        _check(lib().fl_pipe_submit_recognition(self._p, _p(b), C.c_size_t(sW * 3), _p(d), C.c_size_t(sW * 2), sW, sH, W, H,
                                                Intrinsics(*[float(v) for v in K])), "fl_pipe_submit_recognition")
        self._keep[self._seq % self.depth] = (b, d)
        self._seq += 1

    def collect_recognition(self, capacity: int = RECO_MAX_HYP):
        """(rc, results, summary) of the oldest frame in flight, as ``Handle.recognize_wait``."""
        out = self._out.get(("reco", capacity))
        if out is None:
            out = self._out[("reco", capacity)] = np.zeros(max(capacity, 1), RECO_RESULT_DTYPE)
        s = RecoSummary()
        rc = lib().fl_pipe_collect_recognition(self._p, _p(out), int(capacity), C.byref(s))
        if rc not in (FL_OK, FL_ERR_CAPACITY):
            _check(rc, "fl_pipe_collect_recognition")
        return rc, out[:min(s.n_results, capacity)].copy(), _summary(s)


# --------------------------------------------------------------------------------------------------
# mirrors of the reference interface
# --------------------------------------------------------------------------------------------------
class Match:
    """cup_linemod::Match (linemod/linemod.hpp:253-286)."""
    __slots__ = ("x", "y", "similarity", "class_id", "template_id")

    def __init__(self, x, y, similarity, class_id, template_id):
        self.x, self.y, self.similarity, self.class_id, self.template_id = int(x), int(y), float(similarity), class_id, int(template_id)

    def __repr__(self):
        return "Match(x=%d, y=%d, similarity=%.4f, class_id=%r, template_id=%d)" % (self.x, self.y, self.similarity, self.class_id, self.template_id)


_MODALITY_KIND = {"ColorGradient": 0, "DepthNormal": 1}


class Detector:
    """Host-side mirror of ``cup_linemod::Detector`` for the matching path (linemod/linemod.hpp:292-412).

    Templates are added with ``addSyntheticTemplate`` (one TemplatePyramid = list of (width, height, offset_x,
    offset_y, pyramid_level, features[(x, y, label)]) in the order L0-M0, L0-M1, L1-M0 ...) or in bulk from a
    ``synth.TemplateSet``; classes iterate in sorted name order like the reference's ``std::map``.
    """

    def __init__(self, modalities: Sequence[str] = ("ColorGradient", "DepthNormal"), T_pyramid: Sequence[int] = (5, 8),
                 max_width=640, max_height=480, device=0, max_candidates=1 << 16):
        self.modalities = list(modalities)
        self.T_at_level = [int(t) for t in T_pyramid]
        self._handle_args = (self.T_at_level, [_MODALITY_KIND[m] for m in modalities], max_width, max_height, max_candidates, device)
        self._handle_obj = None     # created on first use so that argument checks behave like the reference without a GPU
        self._classes = {}          # class_id -> list of template pyramids
        self._poses = {}            # class_id -> list of 13-float arrays
        self._dirty = True
        self._revision = 0          # bumped by every template change (consumers with their own copy of the templates compare it)
        self._class_order: List[str] = []

    @property
    def _handle(self) -> Handle:
        if self._handle_obj is None:
            self._handle_obj = Handle(*self._handle_args)
        return self._handle_obj

    # -- accessors (linemod.hpp:357-381) --
    def getModalities(self):
        return self.modalities

    def getT(self, pyramid_level):
        return self.T_at_level[pyramid_level]

    def pyramidLevels(self):
        return len(self.T_at_level)

    def numClasses(self):
        return len(self._classes)

    def numTemplates(self, class_id=None):
        if class_id is None:
            return sum(len(v) for v in self._classes.values())
        return len(self._classes.get(class_id, []))

    def classIds(self):
        return sorted(self._classes)

    def getTemplates(self, class_id, template_id):
        return self._classes[class_id][template_id]

    def getPoseInfo(self, template_id, class_id=None):
        cid = class_id if class_id is not None else self.classIds()[0]
        return self._poses[cid][template_id]

    def addTemplate(self, sources, class_id, object_mask=None, pose_info=None):
        """Detector::addTemplate (linemod.hpp:338-339, linemod.cpp:1579-1615): extract a template pyramid from one view (``sources`` in
        modality order) and append it to ``class_id``.  Returns (template_id, bounding_box (x, y, w, h)); template_id is -1 when a
        pyramid level has too few candidate features (nothing is added)."""
        if len(sources) != len(self.modalities):
            return -1, None
        bgr = depth = None
        for name, src in zip(self.modalities, sources):
            if name == "ColorGradient":
                bgr = src
            else:
                depth = src
        rc, hdr, ft, bb = self._handle.add_template(bgr, depth, object_mask)
        if rc != FL_OK:
            return -1, None
        pyr = [(int(h[0]), int(h[1]), int(h[2]), int(h[3]), int(h[4]), [tuple(int(v) for v in f) for f in ft[h[5]:h[5] + h[6]]]) for h in hdr]
        return self.addSyntheticTemplate(pyr, class_id, pose_info), tuple(int(v) for v in bb)

    def addSyntheticTemplate(self, templates, class_id, pose_info=None) -> int:
        lst = self._classes.setdefault(class_id, [])
        self._poses.setdefault(class_id, []).append(np.zeros(13, np.float32) if pose_info is None else np.asarray(pose_info, np.float32))
        lst.append(templates)
        self._dirty = True
        self._revision += 1
        return len(lst) - 1

    def add_template_set(self, tset) -> None:
        LM = tset.n_levels * tset.n_modalities
        for t in range(tset.n_templates):
            pyr = []
            for e in range(LM):
                h = tset.headers[t * LM + e]
                pyr.append((int(h[0]), int(h[1]), int(h[2]), int(h[3]), int(h[4]), tset.features[h[5]:h[5] + h[6]].copy()))
            self.addSyntheticTemplate(pyr, tset.class_names[int(tset.class_of[t])], tset.pose13[t])

    def _upload(self):
        self._handle.upload_templates(self.template_set())
        self._class_order = self.classIds()
        self._dirty = False

    def template_set(self):
        """The flattened template database in upload order (classes sorted by name, templates by id) as a ``synth.TemplateSet``."""
        names = self.classIds()
        hdrs, feats, class_of, poses, pos = [], [], [], [], 0
        for ci, name in enumerate(names):
            for tid, pyr in enumerate(self._classes[name]):
                for (w, h, ox, oy, lvl, f) in pyr:
                    f = np.asarray(f, np.int32).reshape(-1, 3)
                    hdrs.append((w, h, ox, oy, lvl, pos, len(f)))
                    feats.append(f)
                    pos += len(f)
                class_of.append(ci)
                poses.append(self._poses[name][tid])
        return synth.TemplateSet(len(self.T_at_level), len(self.modalities), tuple(self.T_at_level), names,
                                 np.array(hdrs, np.int32).reshape(-1, 7),
                                 np.concatenate(feats).astype(np.int32) if feats else np.zeros((0, 3), np.int32),
                                 np.array(class_of, np.int32), np.array(poses, np.float32).reshape(-1, 13))

    def match(self, sources: Sequence[np.ndarray], threshold: float, class_ids: Sequence[str] = (),
              quantized_images: Optional[list] = None, masks: Sequence[Optional[np.ndarray]] = ()):
        """Returns (status, matches): status 0 or -1 exactly where the reference returns them (linemod.cpp:1364-1378);
        geometry violations that are CV_Asserts in the reference raise ``FealessError``."""
        if len(sources) != len(self.modalities):
            return -1, []
        if masks and len(masks) != len(self.modalities):
            return -1, []
        if self._dirty:
            self._upload()
        bgr = depth = None
        for m, s in zip(self.modalities, sources):
            if m == "ColorGradient":
                bgr = s
            else:
                depth = s
        filt = None
        if class_ids:
            filt = [self._class_order.index(c) for c in class_ids if c in self._class_order]
            if not filt:
                return 0, []
        r = self._handle.match(bgr, depth, threshold, filt, list(masks) if masks else None, want_quantized=quantized_images is not None)
        rc, recs = r[0], r[1]
        if rc in (FL_ERR_GEOMETRY, FL_ERR_CAPACITY):
            raise FealessError(rc, "Detector.match", "geometry (W%T, H%T, W*H%16) or capacity")
        if rc != FL_OK:
            return -1, []
        if quantized_images is not None:
            quantized_images[:] = r[2]
        return 0, [Match(m["x"], m["y"], m["similarity"], self._class_order[m["class_idx"]], m["template_id"]) for m in recs]


def _detector_match_rescaled(self, sources: Sequence[np.ndarray], W: int, H: int, threshold: float, want_depth: bool = False):
    """``PrepareInputData`` + ``Detector::match`` (obj_reco_lmicp.cpp:216-259, :101): the sources keep their own size on the host and
    are rescaled to W x H on the device.  Returns (status, matches[, rescaled depth])."""
    if len(sources) != len(self.modalities):
        return (-1, [], None) if want_depth else (-1, [])
    if self._dirty:
        self._upload()
    bgr = depth = None
    for m, s in zip(self.modalities, sources):
        if m == "ColorGradient":
            bgr = s
        else:
            depth = s
    r = self._handle.match_rescaled(bgr, depth, W, H, threshold, want_depth=want_depth)
    rc, recs = r[0], r[1]
    if rc in (FL_ERR_GEOMETRY, FL_ERR_CAPACITY):
        raise FealessError(rc, "Detector.match_rescaled", "geometry (W%T, H%T, W*H%16) or capacity")
    ms = [] if rc != FL_OK else [Match(m["x"], m["y"], m["similarity"], self._class_order[m["class_idx"]], m["template_id"]) for m in recs]
    st = 0 if rc == FL_OK else -1
    return (st, ms, r[2]) if want_depth else (st, ms)


Detector.match_rescaled = _detector_match_rescaled

_default_handle = None


def _handle() -> Handle:
    global _default_handle
    if _default_handle is None:
        _default_handle = Handle()
    return _default_handle


def depthTo3d(depth, K, handle: Optional[Handle] = None) -> np.ndarray:
    """cup_d2pc::depthTo3d for a 16UC1 image; K = 3x3 matrix or (fx, fy, cx, cy).  Metres, 0 -> NaN."""
    K = np.asarray(K, np.float64)
    if K.shape == (3, 3):
        K = (K[0, 0], K[1, 1], K[0, 2], K[1, 2])
    return (handle or _handle()).depth_to_3d(depth, K)


def icpCloudToCloud_Ex(pts_ref, pts_model, icp_it_thr=4, dist_mean_thr=0.0, dist_diff_thr=0.0, handle: Optional[Handle] = None):
    """Returns (dist_mean, R 3x3, T 3, px_inliers_ratio) like the reference's return value + out-params."""
    r = (handle or _handle()).icp_cloud_to_cloud_ex(pts_ref, pts_model, icp_it_thr, dist_mean_thr, dist_diff_thr)
    return float(r["dist_mean"]), r["R"].reshape(3, 3).copy(), r["T"].copy(), float(r["inlier_ratio"])


def detection(depImg_model_raw, depImg_ref_raw, tCamIntrinsic, rect_model_final, rect_ref_final, icp_it_thr, dist_mean_thr,
              dist_diff_thr, r_match, t_match, d_match=0.0, handle: Optional[Handle] = None):
    """detection() (ICP/detection.h:9-11): returns (T_final, R_final); raises on a rect outside the image
    (the reference throws a cv::Exception there, detection.cpp:43-44)."""
    r = (handle or _handle()).detection_batch(depImg_ref_raw, tCamIntrinsic, [depImg_model_raw], [rect_model_final], [rect_ref_final],
                                              [r_match], [t_match], icp_it_thr, dist_mean_thr, dist_diff_thr)[0]
    if r["status"] != FL_OK:
        raise FealessError(int(r["status"]), "detection", "rect outside the image")
    return r["T"].copy(), r["R"].reshape(3, 3).copy()


def nonMaximumSuppression(objs: List[dict], th_obj_dist: float, handle: Optional[Handle] = None) -> List[dict]:
    """objs: dicts with match_class, match_sim, r, t, pts_model (array or count), icp_dist; sets 'check_done' like the
    reference mutates obj_data, returns the emitted pose results (object id, confidence, R, T)."""
    if not objs:
        return []
    t3 = np.array([np.asarray(o["t"], np.float32).reshape(3) for o in objs], np.float32)
    nm = [int(o["pts_model"]) if np.isscalar(o["pts_model"]) else len(o["pts_model"]) for o in objs]
    idx = (handle or _handle()).nms(t3, nm, [o["icp_dist"] for o in objs], th_obj_dist)
    return [dict(object_id=objs[i]["match_class"], confidence=objs[i]["match_sim"], R=objs[i]["r"], T=objs[i]["t"], index=int(i)) for i in idx]
