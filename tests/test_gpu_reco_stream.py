"""GPU: Recognition on the device (fl_set_recognition, fl_recognize*, fl_pipe_*_recognition and the stream methods of both mirrors),
checked bit for bit against ObjRecoLmICP.Recognition on the same frames - tWorld2Cam bits, class tags, template ids and ICP records.
That mirror is checked against the oracle by test_recognition_mirror_end_to_end and test_recognition_rescales_on_the_device; the C++
stream methods are checked against the C++ Recognition (tests/cpp/reco_test.cpp), which test_cpp_reco.py checks against the Python one."""
import os
import struct
import subprocess

import numpy as np
import pytest

import fealess_b200 as fb
from fealess_b200 import build as fbuild
from fealess_b200 import linemod_io, reco, synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT_DIR = os.path.join(ROOT, "tests", "cpp", "_build")
W, H, T = 640, 480, (5, 8)
K = (608.0, 608.0, 320.0, 240.0)
MODES = [(1, False, 0.0), (4, False, 0.0), (1, True, 0.0), (2, True, 25.0), (6, False, 40.0)]


def _kdict(img):
    return dict(fx=K[0], fy=K[1], cx=K[2], cy=K[3], width=img.shape[1], height=img.shape[0])


def _planted(n, n_classes, seed, planted=0.5):
    import fl_oracle_py as F
    b, d = synth.make_frame(W, H, 0)
    det = F.Detector(T)
    assert det.process(b, d) == 0
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    return b, d, synth.make_templates(n, W, H, T, n_classes=n_classes, seed=seed, quantized=q, planted_fraction=planted)


def _feature_dir(path, ts, depth_mm, n_depth=None):
    import cv2
    D0 = fb.Detector()
    D0.add_template_set(ts)
    linemod_io.write_linemod(D0, str(path / "linemod_templates.yml"))
    (path / "depth").mkdir()
    png = (depth_mm.astype(np.uint32) * 10).clip(0, 65535).astype(np.uint16)       # the reference stores 0.1 mm units
    for tid in range(ts.n_templates if n_depth is None else n_depth):
        cv2.imwrite(str(path / "depth" / ("%d.png" % tid)), png)


def _big(b, d):
    import cv2
    return cv2.resize(b, (1280, 960), interpolation=cv2.INTER_CUBIC), cv2.resize(d, (1280, 960), interpolation=cv2.INTER_NEAREST)


def _pair(path, frames_in_flight=1):
    sync, stream = reco.ObjRecoLmICP(), reco.ObjRecoLmICP(frames_in_flight=frames_in_flight)
    assert sync.AddObj(str(path)) == 0 and stream.AddObj(str(path)) == 0
    return sync, stream


def _same(got, want):
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g["strObjTag"] == w["strObjTag"] and g["template_id"] == w["template_id"]
        assert g["tWorld2Cam"].tobytes() == w["tWorld2Cam"].tobytes()
        assert g["icp"].tobytes() == w["icp"].tobytes()
        assert np.float32(g["similarity"]) == np.float32(w["similarity"])


def _stream(obj, frames, **hyp):
    """every frame through submit / collect from this thread, at most obj.frames_in_flight in flight; results in submission order"""
    out, queued = [], 0
    for fb_, fd_ in frames:
        if queued == obj.frames_in_flight:
            out.append(obj.collect())
            queued -= 1
        assert obj.submit(fb_, fd_, _kdict(fb_), **hyp) == 0
        queued += 1
        assert obj.in_flight() == queued
    while queued:
        out.append(obj.collect())
        queued -= 1
    return out


@pytest.fixture(scope="module")
def cpp():
    fbuild.build()
    os.makedirs(OUT_DIR, exist_ok=True)
    libdir = os.path.dirname(fb.library_path())
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    exes = {}
    for name in ("reco_test", "reco_stream_test"):
        exe = os.path.join(OUT_DIR, name + "_s")
        cmd = [cxx, "-std=c++11", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", name + ".cpp"),
               "-o", exe, fb.library_path(), "-lz", "-Wl,-rpath," + libdir]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        exes[name] = exe
    return exes


def _write_frame(path, bgr, depth):
    with open(path, "wb") as f:
        f.write(struct.pack("<ii4d", bgr.shape[1], bgr.shape[0], *K))
        f.write(np.ascontiguousarray(bgr, np.uint8).tobytes())
        f.write(np.ascontiguousarray(depth, np.uint16).tobytes())


def test_recognize_equals_recognition_at_both_sizes(tmp_path):
    """fl_recognize on one handle and the stream at 640 x 480 and with the 1280 x 960 input rescaled on the device; in the common path
    the frame is exactly [resize x 2] + front end + similarity + refinement / sort + selection + ICP + finish."""
    b, d, ts = _planted(24, 1, 61)
    _feature_dir(tmp_path, ts, d)
    sync, stream = _pair(tmp_path)
    det = sync.m_lm_detector
    h = fb.Handle(T, (0, 1))
    h.upload_templates(det.template_set())
    index, images, rects = sync._crop_table((H, W))
    h.upload_model_depths(images, rects)
    h.set_recognition([index.get((c, t), -1) for c in det.classIds() for t in range(det.numTemplates(c))])
    for fb_, fd_ in [(b, d), _big(b, d)]:
        rc, want = sync.Recognition(fb_, fd_, _kdict(fb_))
        assert rc == 0 and len(want) == 1 and sync.last_icp_path == "resident"
        rc, recs, summ = h.recognize(fb_, fd_, K, W, H)
        assert rc == fb.FL_OK and summ["n_results"] == len(recs) == 1 and summ["n_hypotheses"] == 1 and summ["n_matches"] >= 1
        assert recs[0]["world2cam"].tobytes() == want[0]["tWorld2Cam"].tobytes() and recs[0]["icp"].tobytes() == want[0]["icp"].tobytes()
        assert det.classIds()[recs[0]["class_idx"]] == want[0]["strObjTag"] and recs[0]["template_id"] == want[0]["template_id"]
        for rep in range(2):
            n0 = stream._pipe.launch_count() if stream._pipe else 0
            (rc, got), = _stream(stream, [(fb_, fd_)])
            assert rc == 0
            _same(got, want)
            if rep == 1:                                             # steady state (the first frame packs the templates for the geometry)
                assert stream._pipe.launch_count() - n0 == (6 if fb_.shape[1] == W else 8)


@pytest.mark.parametrize("top_k,per_class,th", MODES)
def test_modes_equal_recognition_python_and_cpp(cpp, tmp_path, top_k, per_class, th):
    b, d, ts = _planted(36, 3, 62)
    _feature_dir(tmp_path, ts, d)
    frames = [(b, d), _big(b, d)]
    sync, stream = _pair(tmp_path, 2)
    hyp = dict(top_k=top_k, per_class=per_class, th_obj_dist=th if th > 0 else None)
    got = _stream(stream, frames, **hyp)
    for (fb_, fd_), (rc, res) in zip(frames, got):
        rc_w, want = sync.Recognition(fb_, fd_, _kdict(fb_), **hyp)
        assert rc == rc_w == 0 and len(want) >= 1
        _same(res, want)
    if per_class and th == 0:
        tags = [x["strObjTag"] for x in got[0][1]]
        assert all(tags.count(t) <= top_k for t in set(tags)) and len(set(tags)) > 1
    # C++: SubmitRecognition / CollectRecognition with two frames in flight == CObjRecoLmICP::Recognition (SetHypotheses), bit for bit
    for i, (fb_, fd_) in enumerate(frames):
        _write_frame(str(tmp_path / ("frame%d.bin" % i)), fb_, fd_)
    fr = [str(tmp_path / ("frame%d.bin" % i)) for i in range(len(frames))]
    args = [str(top_k), "1" if per_class else "0", str(th)]
    r_sync = subprocess.run([cpp["reco_test"], "hyp", str(tmp_path)] + args + fr, capture_output=True, text=True)
    r_stream = subprocess.run([cpp["reco_stream_test"], str(tmp_path), "2"] + args + fr, capture_output=True, text=True)
    assert r_sync.returncode == 0 and r_stream.returncode == 0, r_sync.stdout + r_stream.stdout + r_stream.stderr
    want = r_sync.stdout.strip().split("\n")
    assert r_stream.stdout.strip().split("\n") == [want[0]] + want[1::2]


def test_no_matches_and_templates_without_crops(tmp_path):
    b, d, ts = _planted(24, 1, 61)
    _feature_dir(tmp_path, ts, d, n_depth=ts.n_templates // 2)      # the upper half of the templates has no depth image
    sync, stream = _pair(tmp_path, 2)
    blank = (np.zeros_like(b), np.zeros_like(d))
    frames = [blank, (b, d), blank]
    got = _stream(stream, frames, top_k=8)
    summaries = []
    for (fb_, fd_), (rc, res) in zip(frames, got):
        rc_w, want = sync.Recognition(fb_, fd_, _kdict(fb_), top_k=8)
        assert rc == rc_w == 0
        _same(res, want)
    _stream(stream, [(b, d)], top_k=8)
    summaries.append(stream.last_summary)
    rc, ms = sync.m_lm_detector.match([b, d], 75.0)
    assert rc == 0 and summaries[0]["n_matches"] == len(ms) >= 8
    assert summaries[0]["n_hypotheses"] == sum(m.template_id < ts.n_templates // 2 for m in ms[:8])   # selected without a crop: dropped
    assert len(got[0][1]) == 0 and len(got[2][1]) == 0 and len(got[1][1]) >= 1
    _stream(stream, [blank], top_k=8)
    assert stream.last_summary == dict(n_matches=0, n_hypotheses=0, n_roi=0, n_results=0)


def _edge_templates():
    """Planted templates whose level-0 box spans the whole frame width from x = 0, level-0 features moved with the box.  Refinement
    clamps the level-0 search to x <= W - width - 8 T (similarityLocal, linemod.cpp:1525-1534): with width = W the search starts at
    x = -16 T and every match of these templates ends at x < 0 (the C oracle puts them at x = -3 with similarity 100), so every
    reference rect leaves the frame."""
    b, d, ts = _planted(16, 1, 64, planted=1.0)
    LM = ts.n_levels * ts.n_modalities
    keep = [t for t in range(ts.n_templates) if ts.headers[t * LM][2] >= 16 * T[0]]   # features stay inside the shifted search window
    hdrs, feats, pos = [], [], 0
    for t in keep:
        for e in range(LM):
            h = ts.headers[t * LM + e].copy()
            f = ts.features[h[5]:h[5] + h[6]].copy()
            if h[4] == 0:
                f[:, 0] += h[2] + T[0]                                   # at x = -T (the last column of the search) on the planted pixels
                h[0], h[2] = W, 0
            h[5] = pos
            pos += len(f)
            hdrs.append(h)
            feats.append(f)
    return b, d, synth.TemplateSet(ts.n_levels, ts.n_modalities, ts.T, ts.class_names, np.array(hdrs, np.int32), np.concatenate(feats).astype(np.int32),
                                   np.zeros(len(keep), np.int32), ts.pose13[keep])


def test_box_outside_the_frame(cpp, tmp_path):
    """A reference rect outside the frame is FL_ERR_ROI for that hypothesis and gives no result; with ONE hypothesis the C++
    Recognition throws (the cv::Mat ROI assert of detection.cpp:43-44) and so does CollectRecognition."""
    b, d, ts = _edge_templates()
    _feature_dir(tmp_path, ts, d)
    sync, stream = _pair(tmp_path, 2)
    rc, ms = sync.m_lm_detector.match([b, d], 75.0)
    assert rc == 0 and len(ms) >= 4 and all(m.x < 0 for m in ms)
    for top_k in (1, 4):
        (rc, got), = _stream(stream, [(b, d)], top_k=top_k)
        rc_w, want = sync.Recognition(b, d, _kdict(b), top_k=top_k)
        assert rc == rc_w == 0 and got == want == []
        assert stream.last_summary == dict(n_matches=len(ms), n_hypotheses=top_k, n_roi=top_k, n_results=0)
    _write_frame(str(tmp_path / "frame.bin"), b, d)
    r_sync = subprocess.run([cpp["reco_test"], "hyp", str(tmp_path), "1", "0", "0", str(tmp_path / "frame.bin")], capture_output=True, text=True)
    r_stream = subprocess.run([cpp["reco_stream_test"], str(tmp_path), "2", "1", "0", "0", str(tmp_path / "frame.bin")], capture_output=True, text=True)
    assert r_sync.returncode == 3 and "cv::Exception" in r_sync.stdout, r_sync.stdout
    assert r_stream.returncode == 3 and "cv::Exception" in r_stream.stdout and "status -3" in r_stream.stdout, r_stream.stdout
    # with four hypotheses the C++ mirrors return no object instead of throwing
    r_sync = subprocess.run([cpp["reco_test"], "hyp", str(tmp_path), "4", "0", "0", str(tmp_path / "frame.bin")], capture_output=True, text=True)
    r_stream = subprocess.run([cpp["reco_stream_test"], str(tmp_path), "2", "4", "0", "0", str(tmp_path / "frame.bin")], capture_output=True, text=True)
    assert r_sync.returncode == r_stream.returncode == 0, r_sync.stdout + r_stream.stdout
    assert r_stream.stdout.strip().split("\n") == r_sync.stdout.strip().split("\n")[::2] == ["addobj 00000000", "frame 0 status 00000000 results 0"]


def test_settings_and_templates_changed_between_frames(tmp_path):
    """The stream follows the mirror's attributes and its detector: a new matching threshold, new ICP parameters and a template added
    between two frames take effect on the next submit, as they do for Recognition."""
    b, d, ts = _planted(24, 1, 61)
    _feature_dir(tmp_path, ts, d)
    sync, stream = _pair(tmp_path, 2)
    summaries = []
    for step in range(4):
        if step == 1:
            sync.m_matching_threshold = stream.m_matching_threshold = 40.0       # 60 matches instead of 12 (C oracle)
        if step == 2:
            sync.m_icp_it_thr = stream.m_icp_it_thr = 3
            sync.m_dist_mean_thr = stream.m_dist_mean_thr = 0.25
        if step == 3:                                                   # one more template, planted elsewhere on the frame
            extra = _planted(1, 1, 99, planted=1.0)[2]
            pyr = [tuple(int(v) for v in h[:5]) + (extra.features[h[5]:h[5] + h[6]].copy(),) for h in extra.headers]
            for o in (sync, stream):
                o.m_lm_detector.addSyntheticTemplate(pyr, "obj00", extra.pose13[0])
        (rc, got), = _stream(stream, [(b, d)], top_k=6)
        rc_w, want = sync.Recognition(b, d, _kdict(b), top_k=6)
        assert rc == rc_w == 0 and len(want) >= 1
        _same(got, want)
        summaries.append(stream.last_summary)
    assert summaries[1]["n_matches"] > summaries[0]["n_matches"] and summaries[3]["n_matches"] > summaries[2]["n_matches"]
    with pytest.raises(fb.FealessError) as e:                           # a setting changed with a frame in flight
        assert stream.submit(b, d, _kdict(b), top_k=6) == 0
        stream.m_matching_threshold = 80.0
        stream.submit(b, d, _kdict(b), top_k=6)
    assert e.value.rc == fb.FL_ERR_STATE
    stream.collect()



def _many_matches_detector(max_candidates=1 << 16):
    b, d, ts = _planted(400, 2, 2, planted=0.05)
    det = fb.Detector(max_candidates=max_candidates)
    det.add_template_set(ts)
    return b, d, det


def test_deferred_list_and_candidate_overflow():
    """A unique list of more than 1,024 records is sorted after the first wait and selection, ICP and finish run again on it; more
    candidates than the device buffers hold is FL_ERR_CAPACITY, as Recognition's match raises it."""
    b, d, det = _many_matches_detector()
    sync, stream = reco.ObjRecoLmICP(), reco.ObjRecoLmICP(frames_in_flight=2)
    sync.add_detector(det, {(None, t): d for t in range(400)})
    stream.add_detector(det, {(None, t): d for t in range(400)})
    sync.m_matching_threshold = stream.m_matching_threshold = 25.0
    for hyp in (dict(top_k=3), dict(top_k=2, per_class=True, th_obj_dist=25.0)):
        got = _stream(stream, [(b, d), (b, d)], **hyp)
        rc_w, want = sync.Recognition(b, d, _kdict(b), **hyp)
        assert stream.last_summary["n_matches"] > 1024 and rc_w == 0 and len(want) >= 1
        for rc, res in got:
            assert rc == 0
            _same(res, want)
    b, d, det = _many_matches_detector(max_candidates=512)
    sync, stream = reco.ObjRecoLmICP(), reco.ObjRecoLmICP()
    sync.add_detector(det, {(None, t): d for t in range(400)})
    stream.add_detector(det, {(None, t): d for t in range(400)})
    sync.m_matching_threshold = stream.m_matching_threshold = 25.0
    with pytest.raises(fb.FealessError) as e:
        sync.Recognition(b, d, _kdict(b))
    assert e.value.rc == fb.FL_ERR_CAPACITY
    assert stream.submit(b, d, _kdict(b)) == 0
    with pytest.raises(fb.FealessError) as e:
        stream.collect()
    assert e.value.rc == fb.FL_ERR_CAPACITY and stream.in_flight() == 0


@pytest.mark.parametrize("depth", [1, 2, 4, 8])
def test_pipe_depths_over_mixed_frames(tmp_path, depth):
    b, d, ts = _planted(36, 3, 62)
    _feature_dir(tmp_path, ts, d)
    big = _big(b, d)
    frames = []
    for i in range(24):
        k = i % 4
        frames.append((b, d) if k == 0 else big if k == 1 else synth.make_frame(W, H, 100 + i) if k == 2 else (np.zeros_like(b), np.zeros_like(d)))
    sync, stream = _pair(tmp_path, depth)
    hyp = dict(top_k=2, per_class=True, th_obj_dist=25.0)
    want = [sync.Recognition(fb_, fd_, _kdict(fb_), **hyp) for fb_, fd_ in frames]
    got = _stream(stream, frames, **hyp)
    assert len(got) == len(frames)
    for (rc, res), (rc_w, res_w) in zip(got, want):
        assert rc == rc_w == 0
        _same(res, res_w)
    assert sum(len(r) for _, r in got) >= 12


def test_state_errors():
    b, d, ts = _planted(24, 1, 61)
    crops, rects = [d] * ts.n_templates, [tuple(int(v) for v in ts.headers[t * 4][[2, 3, 0, 1]]) for t in range(ts.n_templates)]
    p = fb.Pipe(2)
    p.upload_templates(ts)
    p.upload_model_depths(crops, rects)
    p.set_recognition(np.arange(ts.n_templates))
    with pytest.raises(fb.FealessError) as e:
        p.collect_recognition()
    assert e.value.rc == fb.FL_ERR_STATE
    p.submit_recognition(b, d, K)
    p.submit_recognition(b, d, K)
    for call in (lambda: p.submit_recognition(b, d, K), lambda: p.set_recognition(np.arange(ts.n_templates)),
                 lambda: p.upload_model_depths(crops, rects), lambda: p.upload_templates(ts)):
        with pytest.raises(fb.FealessError) as e:
            call()
        assert e.value.rc == fb.FL_ERR_STATE
    r0, r1 = p.collect_recognition(), p.collect_recognition()
    assert r0[0] == r1[0] == fb.FL_OK and r0[1].tobytes() == r1[1].tobytes() and len(r0[1]) == 1
    p.submit(b, d, 75.0)                                                # a match frame: collect_recognition leaves it to collect
    with pytest.raises(fb.FealessError) as e:
        p.collect_recognition()
    assert e.value.rc == fb.FL_ERR_STATE and p.in_flight() == 1
    rc, ms = p.collect()
    assert rc == fb.FL_OK and len(ms) >= 1 and p.in_flight() == 0
    p.submit_recognition(b, d, K)                                       # the slot takes recognition frames again
    assert p.collect_recognition()[1].tobytes() == r0[1].tobytes()
    p.close()
    h = fb.Handle(T, (0, 1))
    with pytest.raises(fb.FealessError) as e:
        h.recognize(b, d, K)                                            # no templates / no setup
    assert e.value.rc == fb.FL_ERR_STATE
    h.upload_templates(ts)
    h.upload_model_depths(crops, rects)
    with pytest.raises(fb.FealessError) as e:
        h.set_recognition(np.arange(ts.n_templates), params=fb.reco_params(top_k=fb.RECO_MAX_HYP + 1))
    assert e.value.rc == fb.FL_ERR_CAPACITY
    bad = list(rects[0]); bad[2] -= 2
    h2 = fb.Handle(T, (0, 1))
    h2.upload_templates(ts)
    h2.upload_model_depths(crops, [tuple(bad)] + rects[1:])
    with pytest.raises(fb.FealessError) as e:                           # crop 0 is not template 0's level-0 box
        h2.set_recognition(np.arange(ts.n_templates))
    assert e.value.rc == fb.FL_ERR_ARG
    h.set_recognition(np.arange(ts.n_templates))
    assert h.recognize(b, d, K)[0] == fb.FL_OK
    h.upload_model_depths(crops, rects)                                 # a new crop set clears the setup
    with pytest.raises(fb.FealessError) as e:
        h.recognize(b, d, K)
    assert e.value.rc == fb.FL_ERR_STATE
    h.set_template_ids(np.zeros(ts.n_templates, np.int32))
    with pytest.raises(fb.FealessError) as e:
        h.set_recognition(np.arange(ts.n_templates))
    assert e.value.rc == fb.FL_ERR_STATE
    # template-sharded pipe (fl_pipe_set_exchange): recognition is not available there
    p = fb.Pipe(1)
    p.upload_templates(ts)
    p.set_exchange(0, 2, 16, [[1 << 20, 2 << 20]], [3 << 20])           # only stored: no frame is submitted through them
    with pytest.raises(fb.FealessError) as e:
        p.set_recognition(np.arange(ts.n_templates))
    assert e.value.rc == fb.FL_ERR_STATE
    with pytest.raises(fb.FealessError) as e:
        p.submit_recognition(b, d, K)
    assert e.value.rc == fb.FL_ERR_STATE
    p.close()
