"""Host-side mirror of ``CObjRecoLmICP`` - the immediate caller of the hot path (reference CadReco/obj_reco_lmicp.cpp:47-259,
``SURVEY.md`` section 8f ranks 1 and 3).  Same entry points, argument meaning and status codes:

* ``AddObj(feature_path)``   :67-74   reads ``<path>/linemod_templates.yml`` (``readLinemod``) - and, unlike the reference, ALSO loads
                                       every rendered template depth image ``<path>/depth/<template_id>.png`` once, converted to
                                       millimetres (``convertTo(CV_16UC1, 0.1)``, :187).  The reference decodes that PNG from disk
                                       inside every ``Recognition`` call (:156-157), which would dominate once LINE-MOD + ICP take
                                       tens of microseconds.  On the first ``Recognition`` the images, cropped to their template
                                       boxes, move to the device for good (``fl_upload_model_depths``); from then on a frame's ICP
                                       sends only the hypothesis records and reads the depth frame ``match`` already uploaded
                                       (``fl_detection_batch_resident`` with ``ref_depth == NULL``).
* ``Recognition(rgb, depth, K)`` :86-204  ``PrepareInputData`` (:216-259: size checks, INTER_LINEAR rescale to 640 columns, intrinsics
                                       zoom), ``Detector::match`` at 75 %, then ``detection()`` (ICP, <= 10 iterations, 0.5 / 0.01 mm
                                       thresholds :52-55) on ``matches[0]`` with the template's box as model rect and the box moved to
                                       the match position as reference rect (:127-132), pose packed as a 4x4 world-to-camera matrix
                                       (``Convert`` :20-30).

``top_k`` / ``th_obj_dist`` wire what the reference left unwired (section 8f rank 3): the K best matches are refined in ONE batched ICP
launch (``fl_detection_batch``) and filtered by the reference's ``nonMaximumSuppression`` (ICP/NMS.cpp:6-39).  The defaults
(``top_k=1``, no NMS) are exactly the reference's behaviour.

``submit`` / ``collect`` (not in the reference) are the same Recognition as a stream: each frame is ONE enqueue on the device
(``fl_pipe_submit_recognition``: rescale, match, hypothesis selection, ICP and suppression with no host round trip in between), up to
``frames_in_flight`` frames are in flight from the calling thread, and ``collect`` returns what ``Recognition`` returns for the
oldest one.

Kept from the reference on purpose (``SURVEY.md`` A.6 v): ``detection`` receives the CALLER's intrinsics, not the zoomed ones.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

ERROR_INVALID_PARAM = 0x80000001        # CadReco/lotus_common.h:5-10
ERROR_OPEN_FILE_FAILED = 0x80000002
PROC_IMG_WIDTH = 640                    # obj_reco_lmicp.cpp:16


def model_depth_to_mm(depth_png: np.ndarray) -> np.ndarray:
    """``depImg_model_raw.convertTo(depImg_model_raw_1, CV_16UC1, 0.1)`` (:187): fp32 scale, round half to even, saturate."""
    v = np.rint(depth_png.astype(np.float32) * np.float32(0.1))
    return np.clip(v, 0, 65535).astype(np.uint16)


def select_hypotheses(matches, top_k: int = 1, per_class: bool = False):
    """The matches that go to ICP, in list order: the first ``top_k``, or the first ``top_k`` of every class (test/linemod_acq.cpp:165-184)."""
    top_k = max(1, int(top_k))
    if not per_class:
        return list(matches[:top_k])
    taken, out = {}, []
    for m in matches:
        if taken.get(m.class_id, 0) < top_k:
            taken[m.class_id] = taken.get(m.class_id, 0) + 1
            out.append(m)
    return out


class ObjRecoLmICP:
    def __init__(self, device: int = 0, max_width: int = 640, max_height: int = 480, frames_in_flight: int = 1):
        self.m_matching_threshold = 75.0                             # :52-55
        self.m_icp_it_thr, self.m_dist_mean_thr, self.m_dist_diff_thr = 10, 0.5, 0.01
        self._args = (device, max_width, max_height)
        self.m_lm_detector = None
        self._model_depth: Dict[Tuple[Optional[str], int], np.ndarray] = {}
        self._resident: Optional[Tuple[tuple, Dict[Tuple[str, int], int]]] = None     # (frame shape, crop index) once uploaded
        self.m_cam = None
        self.last_icp_path = None                                    # "resident" / "per-call": which ICP entry the last Recognition took
        self.frames_in_flight = int(frames_in_flight)                # submit / collect: frames one thread keeps on the device
        self._pipe = None
        self._stream_key = None                                      # what the pipe is set up for (_stream_setup)
        self.last_summary = None

    # ---- AddObj ----
    def AddObj(self, str_feature_path: str) -> int:
        from . import linemod_io
        import cv2
        try:
            det = linemod_io.read_linemod(os.path.join(str_feature_path, "linemod_templates.yml"), max_width=self._args[1],
                                          max_height=self._args[2], device=self._args[0])
        except (IOError, ValueError):
            return ERROR_OPEN_FILE_FAILED
        if det.numClasses() == 0:
            return ERROR_OPEN_FILE_FAILED
        depths = {}
        for cid in det.classIds():
            for tid in range(det.numTemplates(cid)):
                if (None, tid) in depths:
                    continue
                img = cv2.imread(os.path.join(str_feature_path, "depth", "%d.png" % tid), cv2.IMREAD_UNCHANGED)
                if img is not None:
                    depths[(None, tid)] = model_depth_to_mm(img)     # the reference keys the file by template_id alone (:156)
        self.m_lm_detector, self._model_depth, self._resident = det, depths, None
        self._close_stream()
        return 0

    def add_detector(self, detector, model_depths_mm: Dict[Tuple[Optional[str], int], np.ndarray]) -> None:
        """Programmatic alternative to ``AddObj``: a ready detector + model depth images in mm keyed by (class_id or None, template_id)."""
        self.m_lm_detector, self._model_depth, self._resident = detector, dict(model_depths_mm), None
        self._close_stream()

    def _upload_model_crops(self, frame_shape) -> Dict[Tuple[str, int], int]:
        """(class_id, template_id) -> index of the template's depth crop on the device; uploaded once per detector."""
        index, images, rects = self._crop_table(frame_shape)
        if images:
            self.m_lm_detector._handle.upload_model_depths(images, rects)
        return index

    def _crop_table(self, frame_shape):
        """(class_id, template_id) -> crop index, and the crops' images and rects (the templates' level-0 boxes)."""
        det, index, images, rects = self.m_lm_detector, {}, [], []
        for cid in det.classIds():
            for tid in range(det.numTemplates(cid)):
                md = self._model_depth.get((cid, tid))
                if md is None:
                    md = self._model_depth.get((None, tid))
                w, h, ox, oy = [int(v) for v in det.getTemplates(cid, tid)[0][:4]]
                if md is None or md.shape != tuple(frame_shape) or ox < 0 or oy < 0 or ox + w > md.shape[1] or oy + h > md.shape[0]:
                    continue                                          # such a hypothesis takes the per-call path (and its ROI error)
                index[(cid, tid)] = len(images)
                images.append(md); rects.append((ox, oy, w, h))
        return index, images, rects

    # ---- PrepareInputData ----
    def _prepare(self, rgb, depth, K) -> Optional[Tuple[np.ndarray, np.ndarray]]:
        if rgb is None or depth is None or rgb.ndim != 3 or depth.ndim != 2 or rgb.shape[0] <= 0 or rgb.shape[1] <= 0:
            return None
        if rgb.shape[:2] != depth.shape[:2] or int(K["width"]) != rgb.shape[1] or int(K["height"]) != rgb.shape[0]:
            return None                                              # :223-227
        zoom = np.float32(PROC_IMG_WIDTH * 1.0 / rgb.shape[1])
        w, h = PROC_IMG_WIDTH, rgb.shape[0] * PROC_IMG_WIDTH // rgb.shape[1]
        self.m_cam = dict(fx=K["fx"] * zoom, fy=K["fy"] * zoom, cx=K["cx"] * zoom, cy=K["cy"] * zoom, width=w, height=h)   # :238-246
        # TImage2Mat(..., true) rescales with INTER_LINEAR when the width differs (:42); that happens on the DEVICE inside
        # Detector.match_rescaled (fl_match_rescaled), so the frame crosses PCIe once at its own size and is never resized on the host
        return np.ascontiguousarray(rgb, np.uint8), np.ascontiguousarray(depth, np.uint16)

    # ---- Recognition ----
    def Recognition(self, rgb: np.ndarray, depth: np.ndarray, K: dict, top_k: int = 1, th_obj_dist: Optional[float] = None, per_class: bool = False):
        """Returns (status, results); results = list of dicts {strObjTag, tWorld2Cam (4x4 fp32), similarity, template_id, icp}.

        Hypotheses: the reference refines ``matches[0]`` only (obj_reco_lmicp.cpp:111) = the default ``top_k=1``; ``top_k`` takes the first
        top_k matches of the sorted list, ``per_class=True`` the first top_k matches of EVERY class (top_k=1: the "best match per class"
        walk of the reference's demo, test/linemod_acq.cpp:165-184); ``th_obj_dist`` (mm) runs nonMaximumSuppression over the refined objects."""
        from . import nonMaximumSuppression
        if self.m_lm_detector is None:
            return ERROR_INVALID_PARAM, []
        prep = self._prepare(rgb, depth, K)
        if prep is None:
            return ERROR_INVALID_PARAM, []
        m_rgb, m_depth = prep
        det = self.m_lm_detector
        fw, fh = self.m_cam["width"], self.m_cam["height"]          # processing size (640 columns)
        rescaled = m_rgb.shape[1] != fw
        if rescaled:
            by_name = {"ColorGradient": m_rgb, "DepthNormal": m_depth}
            rc, matches = det.match_rescaled([by_name[m] for m in det.getModalities()], fw, fh, self.m_matching_threshold)
        else:
            rc, matches = det.match([m_rgb, m_depth], self.m_matching_threshold)
        if rc != 0:
            return ERROR_INVALID_PARAM, []
        if not matches:
            return 0, []
        hyps = []
        for m in select_hypotheses(matches, top_k, per_class):
            tmpl = det.getTemplates(m.class_id, m.template_id)[0]            # current_template[0] (:111, :127-132)
            w, h, ox, oy = int(tmpl[0]), int(tmpl[1]), int(tmpl[2]), int(tmpl[3])
            md = self._model_depth.get((m.class_id, m.template_id))
            if md is None:
                md = self._model_depth.get((None, m.template_id))
            if md is None:
                continue
            pose = np.asarray(det.getPoseInfo(m.template_id, m.class_id), np.float32).reshape(-1)
            P = pose[:12].reshape(3, 4)
            hyps.append(dict(match=m, model_depth=md, rect_model=(ox, oy, w, h), rect_ref=(ox + (m.x - ox), oy + (m.y - oy), w, h),
                             r_match=P[:, :3].copy(), t_match=P[:, 3].copy(), d_match=float(pose[12])))
        if not hyps:
            return 0, []
        Kc = (float(K["fx"]), float(K["fy"]), float(K["cx"]), float(K["cy"]))   # the caller's intrinsics, as the reference passes them (:188)
        if self._resident is None or self._resident[0] != (fh, fw):
            self._resident = ((fh, fw), self._upload_model_crops((fh, fw)))
        crop = [self._resident[1].get((hy["match"].class_id, hy["match"].template_id)) for hy in hyps]
        if all(c is not None for c in crop):                          # crops resident, depth frame already on the device from match()
            ref = None                                                # the (rescaled) depth frame match() left on the device
            if "DepthNormal" not in det.getModalities():              # a colour-only detector never uploaded the depth frame
                ref = det._handle.resize_linear(m_depth, fw, fh) if rescaled else m_depth
            self.last_icp_path = "resident"
            res = det._handle.detection_batch_resident(ref, Kc, crop, [hy["rect_ref"] for hy in hyps], [hy["r_match"] for hy in hyps],
                                                       [hy["t_match"] for hy in hyps], self.m_icp_it_thr, self.m_dist_mean_thr,
                                                       self.m_dist_diff_thr, frame_size=(fw, fh))
        else:
            if rescaled:
                m_depth = det._handle.resize_linear(m_depth, fw, fh)
            self.last_icp_path = "per-call"
            res = det._handle.detection_batch(m_depth, Kc, [hy["model_depth"] for hy in hyps], [hy["rect_model"] for hy in hyps],
                                              [hy["rect_ref"] for hy in hyps], [hy["r_match"] for hy in hyps], [hy["t_match"] for hy in hyps],
                                              self.m_icp_it_thr, self.m_dist_mean_thr, self.m_dist_diff_thr)
        out = []
        for hyp, r in zip(hyps, res):
            if int(r["status"]) != 0:                                 # rect outside the frame: the reference throws (detection.cpp:43-44)
                continue
            pose4 = np.zeros((4, 4), np.float32)                      # Convert (:20-30)
            pose4[:3, :3] = r["R"].reshape(3, 3); pose4[:3, 3] = r["T"]; pose4[3, 3] = 1.0
            out.append(dict(strObjTag=hyp["match"].class_id, tWorld2Cam=pose4, similarity=float(hyp["match"].similarity),
                            template_id=int(hyp["match"].template_id), icp=r.copy()))
        if th_obj_dist is not None and len(out) > 1:                  # nonMaximumSuppression over the refined objects (NMS.cpp:6-39)
            objs = [dict(match_class=o["strObjTag"], match_sim=o["similarity"], r=o["tWorld2Cam"][:3, :3], t=o["tWorld2Cam"][:3, 3],
                         pts_model=int(o["icp"]["n_points"]), icp_dist=float(o["icp"]["dist_mean"])) for o in out]
            keep = nonMaximumSuppression(objs, th_obj_dist, det._handle)
            out = [out[k["index"]] for k in keep]
        return 0, out

    # ---- Recognition as a stream (submit / collect) ----
    def submit(self, rgb: np.ndarray, depth: np.ndarray, K: dict, top_k: int = 1, th_obj_dist: Optional[float] = None, per_class: bool = False) -> int:
        """Queues ``Recognition(rgb, depth, K, top_k, th_obj_dist, per_class)`` as one enqueue on the device and returns 0 (the result
        comes from ``collect``), or ERROR_INVALID_PARAM without queueing where ``Recognition`` returns it before matching.  The arrays
        must not change until the frame has been collected (page-locked ones are read by DMA).  Changing the hypothesis settings, the
        matching threshold or ICP attributes, the detector's templates or the frame size needs an empty stream.
        One difference from ``Recognition``: a template whose depth image does not have the processing size (or does not hold the
        template's level-0 box) has no crop on the device and its hypothesis is dropped; ``Recognition`` refines such a template through
        the per-call ``detection_batch`` path instead."""
        if self.m_lm_detector is None:
            return ERROR_INVALID_PARAM
        prep = self._prepare(rgb, depth, K)
        if prep is None:
            return ERROR_INVALID_PARAM
        m_rgb, m_depth = prep
        fw, fh = self.m_cam["width"], self.m_cam["height"]
        if m_rgb.shape[1] == fw and len(self.m_lm_detector.getModalities()) != 2:
            return ERROR_INVALID_PARAM                                # Recognition's match() gets two sources: -1 (linemod.cpp:1364-1367)
        self._stream_setup((fh, fw), max(1, int(top_k)), bool(per_class), th_obj_dist)
        from . import FL_ERR_SIZE, FealessError
        Kc = (float(K["fx"]), float(K["fy"]), float(K["cx"]), float(K["cy"]))   # the caller's intrinsics (:188)
        bgr = m_rgb if "ColorGradient" in self.m_lm_detector.getModalities() else None
        try:
            self._pipe.submit_recognition(bgr, m_depth, Kc, fw, fh)
        except FealessError as e:
            if e.rc == FL_ERR_SIZE:                                   # match() returns -1 (linemod.cpp:1364-1378)
                return ERROR_INVALID_PARAM
            raise
        return 0

    def collect(self):
        """(status, results) of the oldest submitted frame: what ``Recognition`` returns for it, result for result and bit for bit."""
        from . import FL_ERR_STATE, FL_OK, FealessError
        if self._pipe is None:
            raise FealessError(FL_ERR_STATE, "ObjRecoLmICP.collect", "no frame in flight")
        rc, recs, self.last_summary = self._pipe.collect_recognition()   # {n_matches, n_hypotheses, n_roi, n_results} of that frame
        if rc != FL_OK:                                               # more candidates than the device buffers hold: Detector.match raises too
            raise FealessError(rc, "ObjRecoLmICP.collect", "capacity")
        names = self.m_lm_detector.classIds()
        return 0, [dict(strObjTag=names[int(r["class_idx"])], tWorld2Cam=r["world2cam"].reshape(4, 4).copy(), similarity=float(r["similarity"]),
                        template_id=int(r["template_id"]), icp=r["icp"].copy()) for r in recs]

    def in_flight(self) -> int:
        return 0 if self._pipe is None else self._pipe.in_flight()

    def _stream_setup(self, frame_shape, top_k: int, per_class: bool, th_obj_dist: Optional[float]) -> None:
        """The pipe behind submit / collect: the detector's templates, the crops of ``frame_shape`` and the recognition setup on every slot.
        Crop index and pose table are Recognition's: crops keyed by (class, template_id), pose = getPoseInfo(template_id, class_id)."""
        from . import FL_ERR_STATE, FealessError, Pipe, reco_params
        det = self.m_lm_detector
        key = (frame_shape, det._revision, top_k, per_class, th_obj_dist, float(self.m_matching_threshold), int(self.m_icp_it_thr),
               float(self.m_dist_mean_thr), float(self.m_dist_diff_thr))
        if self._pipe is not None and self._stream_key == key:
            return
        if self.in_flight():
            raise FealessError(FL_ERR_STATE, "ObjRecoLmICP.submit", "frame size, templates or recognition settings changed with frames in flight")
        if self._pipe is None:
            T, kinds, max_w, max_h, max_cand, device = det._handle_args
            self._pipe = Pipe(self.frames_in_flight, T, kinds, max_w, max_h, device, max_cand)
        new_templates = self._stream_key is None or self._stream_key[1] != det._revision
        if new_templates:
            self._pipe.upload_templates(det.template_set())
        if new_templates or self._stream_key[0] != frame_shape:
            index, images, rects = self._crop_table(frame_shape)
            self._pipe.upload_model_depths(images, rects)
            self._stream_crop = np.array([index.get((cid, tid), -1) for cid in det.classIds() for tid in range(det.numTemplates(cid))], np.int32)
        th = 0.0 if th_obj_dist is None else float(th_obj_dist)       # <= 0: no suppression, what NMS over distance th <= 0 keeps anyway
        self._pipe.set_recognition(self._stream_crop, None, reco_params(self.m_matching_threshold, (self.m_icp_it_thr, self.m_dist_mean_thr,
                                                                                                     self.m_dist_diff_thr), top_k, per_class, th))
        self._stream_key = key

    def _close_stream(self) -> None:
        if self._pipe is not None:
            self._pipe.close()
        self._pipe, self._stream_key = None, None
