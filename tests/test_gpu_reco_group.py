"""GPU: Recognition over a template-sharded group (fl_group_create_pipe, fl_group_*_recognition and CObjRecoLmICP::SetDevices), checked
against a single handle's fl_recognize over the whole set: result records compared as bytes (fl_reco_result_t) and the summaries too.
Members repeat device 0, so every case runs on one GPU; the cases over distinct devices skip where there are too few."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import fealess_b200 as fb
from fealess_b200 import build as fbuild
from fealess_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT_DIR = os.path.join(ROOT, "tests", "cpp", "_build")
W, H, T = 640, 480, (5, 8)
K = (608.0, 608.0, 320.0, 240.0)
MODES = [(1, False, 0.0), (4, False, 0.0), (1, True, 0.0), (2, True, 25.0), (6, False, 40.0)]
TAIL_LAUNCHES = 3                                                # k_reco_select, k_icp_fused, k_reco_finish


def _planted(n, n_classes, seed, planted=0.5):
    import fl_oracle_py as F
    b, d = synth.make_frame(W, H, 0)
    det = F.Detector(T)
    assert det.process(b, d) == 0
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    return b, d, synth.make_templates(n, W, H, T, n_classes=n_classes, seed=seed, quantized=q, planted_fraction=planted)


def _big(b, d):
    import cv2
    return cv2.resize(b, (1280, 960), interpolation=cv2.INTER_CUBIC), cv2.resize(d, (1280, 960), interpolation=cv2.INTER_NEAREST)


def _crops(ts, d):
    """the frame's depth as every template's rendered depth image, cropped to the template's level-0 box"""
    LM = ts.n_levels * ts.n_modalities
    return [d] * ts.n_templates, [tuple(int(v) for v in ts.headers[t * LM][[2, 3, 0, 1]]) for t in range(ts.n_templates)]


def _mixed(b, d, n=24):
    big = _big(b, d)
    return [(b, d) if i % 4 == 0 else big if i % 4 == 1 else synth.make_frame(W, H, 100 + i) if i % 4 == 2 else (np.zeros_like(b), np.zeros_like(d))
            for i in range(n)]


class _Ref:
    """a single handle over the whole set: the reference of every comparison"""

    def __init__(self, ts, crops, rects, crop_of, max_candidates=None):
        self.h = fb.Handle(T, (0, 1), max_candidates=max_candidates) if max_candidates else fb.Handle(T, (0, 1))
        self.h.upload_templates(ts)
        self.h.upload_model_depths(crops, rects)
        self.crop_of = crop_of

    def run(self, frames, params):
        self.h.set_recognition(self.crop_of, params=params)
        return [self.h.recognize(fb_, fd_, K, W, H) for fb_, fd_ in frames]


def _group(ts, crops, rects, crop_of, n, depth, params, cap=4096):
    g = fb.Group([0] * n, depth=depth, exchange_capacity=cap)
    g.upload_templates(ts)
    g.upload_model_depths(crops, rects)
    g.set_recognition(crop_of, params=params)
    return g


def _stream(g, frames, on_submit=None):
    out, queued = [], 0
    for i, (fb_, fd_) in enumerate(frames):
        if queued == g.depth:
            out.append(g.collect_recognition())
            queued -= 1
        if on_submit:
            on_submit(i)
        g.submit_recognition(fb_, fd_, K, W, H)
        queued += 1
        assert g.in_flight() == queued
    while queued:
        out.append(g.collect_recognition())
        queued -= 1
    return out


def _same(got, want):
    assert len(got) == len(want)
    for f, ((rc, recs, summ), (rc_w, recs_w, summ_w)) in enumerate(zip(got, want)):
        assert rc == rc_w, f
        assert summ == summ_w, (f, summ, summ_w)
        assert recs.tobytes() == recs_w.tobytes(), f


@pytest.fixture(scope="module")
def mixed_case():
    b, d, ts = _planted(37, 3, 62)                                   # 37: a multiple of none of the member counts
    crops, rects = _crops(ts, d)
    frames = _mixed(b, d)
    ref = _Ref(ts, crops, rects, np.arange(ts.n_templates))
    want = {m: ref.run(frames, fb.reco_params(top_k=m[0], per_class=m[1], th_obj_dist=m[2])) for m in MODES}
    assert sum(len(r[1]) for r in want[MODES[3]]) >= 6
    return ts, crops, rects, frames, want


@pytest.mark.parametrize("depth", [1, 2, 4, 8])
@pytest.mark.parametrize("n", [2, 3, 4, 8])
def test_members_and_depths_over_mixed_frames(mixed_case, n, depth):
    """24 mixed frames (640 x 480, the 1280 x 960 input rescaled on the device, a random scene, a blank frame) in the five hypothesis
    modes: every frame's records and summary equal the single handle's, in submission order."""
    ts, crops, rects, frames, want = mixed_case
    g = _group(ts, crops, rects, np.arange(ts.n_templates), n, depth, fb.reco_params())
    assert int(fb.lib().fl_group_depth(g._g)) == depth
    for m in MODES:
        g.set_recognition(np.arange(ts.n_templates), params=fb.reco_params(top_k=m[0], per_class=m[1], th_obj_dist=m[2]))
        _same(_stream(g, frames), want[m])
    g.close()


def test_fewer_templates_than_members_and_group_recognize():
    """Five templates over eight members: three members hold none and still take part in the exchange (and own frames)."""
    b, d, ts = _planted(5, 1, 61, planted=1.0)
    crops, rects = _crops(ts, d)
    frames = [(b, d), _big(b, d)] * 4
    params = fb.reco_params(top_k=4)
    want = _Ref(ts, crops, rects, np.arange(ts.n_templates)).run(frames, params)
    assert sum(len(r[1]) for r in want) >= 4
    g = _group(ts, crops, rects, np.arange(ts.n_templates), 8, 2, params)
    _same(_stream(g, frames), want)
    _same([g.recognize(fb_, fd_, K, W, H) for fb_, fd_ in frames], want)
    g.close()


def _edge_templates():
    """planted templates whose level-0 box spans the whole frame width from x = 0 (test_gpu_reco_stream.py): every match ends at x < 0,
    so every reference rect leaves the frame"""
    b, d, ts = _planted(16, 1, 64, planted=1.0)
    LM = ts.n_levels * ts.n_modalities
    keep = [t for t in range(ts.n_templates) if ts.headers[t * LM][2] >= 16 * T[0]]
    hdrs, feats, pos = [], [], 0
    for t in keep:
        for e in range(LM):
            h = ts.headers[t * LM + e].copy()
            f = ts.features[h[5]:h[5] + h[6]].copy()
            if h[4] == 0:
                f[:, 0] += h[2] + T[0]
                h[0], h[2] = W, 0
            h[5] = pos
            pos += len(f)
            hdrs.append(h)
            feats.append(f)
    return b, d, synth.TemplateSet(ts.n_levels, ts.n_modalities, ts.T, ts.class_names, np.array(hdrs, np.int32), np.concatenate(feats).astype(np.int32),
                                   np.zeros(len(keep), np.int32), ts.pose13[keep])


def test_no_matches_missing_crops_boxes_outside_and_deferred_sort():
    b, d, ts = _planted(24, 1, 61)
    crops, rects = _crops(ts, d)
    crop_of = np.where(np.arange(ts.n_templates) < ts.n_templates // 2, np.arange(ts.n_templates), -1)   # upper half: no crop
    blank = (np.zeros_like(b), np.zeros_like(d))
    frames = [blank, (b, d), blank, _big(b, d)]
    params = fb.reco_params(top_k=8)
    want = _Ref(ts, crops, rects, crop_of).run(frames, params)
    assert want[0][2] == dict(n_matches=0, n_hypotheses=0, n_roi=0, n_results=0) and want[1][2]["n_hypotheses"] < 8
    for n, depth in ((3, 2), (2, 4)):
        g = _group(ts, crops, rects, crop_of, n, depth, params)
        _same(_stream(g, frames), want)
        g.close()
    # reference boxes leaving the frame: FL_ERR_ROI hypotheses, no result
    b, d, ts = _edge_templates()
    crops, rects = _crops(ts, np.zeros_like(d))
    for top_k in (1, 4):
        params = fb.reco_params(top_k=top_k)
        want = _Ref(ts, crops, rects, np.arange(ts.n_templates)).run([(b, d)] * 3, params)
        assert want[0][2]["n_roi"] == top_k and want[0][2]["n_results"] == 0
        g = _group(ts, crops, rects, np.arange(ts.n_templates), 3, 2, params)
        _same(_stream(g, [(b, d)] * 3), want)
        g.close()
    # a union of more than 1,024 records: the owner's tail runs once more on the list sorted after the first wait
    b, d, ts = _planted(400, 2, 2, planted=0.05)
    crops, rects = _crops(ts, d)
    frames = [(b, d), _big(b, d), (b, d)]
    for hyp in (dict(top_k=3), dict(top_k=2, per_class=True, th_obj_dist=25.0)):
        params = fb.reco_params(threshold=25.0, **hyp)
        want = _Ref(ts, crops, rects, np.arange(ts.n_templates)).run(frames, params)
        assert want[0][2]["n_matches"] > 1024 and len(want[0][1]) >= 1
        for n, depth in ((2, 2), (4, 3)):
            g = _group(ts, crops, rects, np.arange(ts.n_templates), n, depth, params, cap=8192)
            _same(_stream(g, frames), want)
            g.close()


def test_only_the_owner_runs_the_tail():
    """fl_launch_count of every (slot, member) handle: a frame adds the same match launches on every member of its slot and the three
    tail launches on its owner (member f % n) alone; no other handle moves."""
    b, d, ts = _planted(37, 3, 62)
    crops, rects = _crops(ts, d)
    n, depth = 3, 2
    g = _group(ts, crops, rects, np.arange(ts.n_templates), n, depth, fb.reco_params(top_k=2))
    frames = [(b, d)] * 8
    _stream(g, frames[:depth])                                    # the first frame of every slot packs the templates for the geometry
    per_member = {}
    for f in range(depth, len(frames)):
        before = g.launch_counts()
        g.submit_recognition(b, d, K, W, H)
        rc, recs, _ = g.collect_recognition()
        assert rc == fb.FL_OK and len(recs) >= 1
        delta = g.launch_counts() - before
        s, owner = f % depth, f % n
        assert (np.delete(delta, s, axis=0) == 0).all(), delta
        for m in range(n):
            match = delta[s, m] - (TAIL_LAUNCHES if m == owner else 0)
            assert match >= 3, delta
            assert per_member.setdefault((s, m), match) == match, (f, delta)
    # with every slot busy the totals add up the same way
    before, f0 = g.launch_counts(), len(frames)                   # frames 0 .. 7 went through above
    _stream(g, frames)
    delta = g.launch_counts() - before
    for s in range(depth):
        for m in range(n):
            on_slot = [f for f in range(f0, f0 + len(frames)) if f % depth == s]
            owned = sum(1 for f in on_slot if f % n == m)
            assert delta[s, m] == per_member[(s, m)] * len(on_slot) + TAIL_LAUNCHES * owned, (s, m, delta)
    g.close()


def _raw_counts(g, i=0):
    """FL_DBG_LAST_COUNTS of handle i: raw candidates every member emitted into its exchange block for the last frame"""
    out = np.zeros(16, np.int32)
    fb.lib().fl_debug_get(g._handle(i), fb.FL_DBG_LAST_COUNTS, 0, 0, 0, out.ctypes.data_as(C.c_void_p), C.c_size_t(64))
    return out[3:3 + g.n]


def test_recovery_with_frames_in_flight():
    """A member's front end that times out on an in-grid dependency (FL_OPT_FE_DEP_TIMEOUT_TEST, a bounded wait) re-runs that frame on
    every member of its slot while the other slots hold frames; an exchange block too small for one frame is FL_ERR_CAPACITY for that
    frame alone."""
    b, d, ts = _planted(37, 3, 62)
    crops, rects = _crops(ts, d)
    frames = _mixed(b, d, 12)
    params = fb.reco_params(top_k=2, per_class=True, th_obj_dist=25.0)
    want = _Ref(ts, crops, rects, np.arange(ts.n_templates)).run(frames, params)
    n, depth = 3, 4
    g = _group(ts, crops, rects, np.arange(ts.n_templates), n, depth, params)
    victim = 2 * n + 1                                            # slot 2, member 1: frame 2 (owner: member 2) and later frames of slot 2

    def arm(i):
        if i == 2:
            g.member_option(victim, fb.FL_OPT_FE_DEP_TIMEOUT_TEST, 1)
    _same(_stream(g, frames, arm), want)
    forced = [g.member_option(i, fb.FL_OPT_FE_FORCED_WAVES) for i in range(n * depth)]
    assert forced == [1 if i == victim else 0 for i in range(n * depth)]
    _same(_stream(g, frames), want)
    g.close()
    # exchange capacity: find a frame that one member's block cannot hold at the capacity another frame fits in
    b2, d2, ts2 = _planted(400, 2, 2, planted=0.05)
    crops2, rects2 = _crops(ts2, d2)
    params = fb.reco_params(threshold=60.0, top_k=3)
    probe = fb.Group([0, 0], exchange_capacity=8192)
    probe.upload_templates(ts2)
    many, few = (b2, d2), synth.make_frame(W, H, 7)
    assert probe.match(*many, 60.0)[0] == fb.FL_OK
    c_many = _raw_counts(probe).max()
    assert probe.match(*few, 60.0)[0] == fb.FL_OK
    c_few = _raw_counts(probe).max()
    probe.close()
    assert c_many > c_few, (c_many, c_few)
    frames = [few, many, few, few]
    want = _Ref(ts2, crops2, rects2, np.arange(ts2.n_templates)).run(frames, params)
    g = _group(ts2, crops2, rects2, np.arange(ts2.n_templates), 2, 4, params, cap=max(int(c_few), 1))
    got = _stream(g, frames)
    assert got[1][0] == fb.FL_ERR_CAPACITY and len(got[1][1]) == 0
    _same([got[0]] + got[2:], [want[0]] + want[2:])
    g.close()


def test_state_errors():
    b, d, ts = _planted(24, 1, 61)
    crops, rects = _crops(ts, d)
    g = fb.Group([0, 0], depth=2)
    for call in (lambda: g.collect_recognition(), lambda: g.submit_recognition(b, d, K)):   # nothing in flight / no set-up
        with pytest.raises(fb.FealessError) as e:
            call()
        assert e.value.rc == fb.FL_ERR_STATE
    with pytest.raises(fb.FealessError) as e:                       # no templates
        g.set_recognition(np.arange(ts.n_templates))
    assert e.value.rc == fb.FL_ERR_STATE
    g.upload_templates(ts)
    g.upload_model_depths(crops, rects)
    with pytest.raises(fb.FealessError) as e:
        g.set_recognition(np.arange(ts.n_templates), params=fb.reco_params(top_k=fb.RECO_MAX_HYP + 1))
    assert e.value.rc == fb.FL_ERR_CAPACITY
    bad = list(rects[0]); bad[2] -= 2
    g.upload_model_depths(crops, [tuple(bad)] + rects[1:])
    with pytest.raises(fb.FealessError) as e:                       # crop 0 is not template 0's level-0 box
        g.set_recognition(np.arange(ts.n_templates))
    assert e.value.rc == fb.FL_ERR_ARG
    g.upload_model_depths(crops, rects)
    g.set_recognition(np.arange(ts.n_templates))
    g.submit_recognition(b, d, K)
    g.submit_recognition(b, d, K)
    for call in (lambda: g.submit_recognition(b, d, K), lambda: g.set_recognition(np.arange(ts.n_templates)),
                 lambda: g.upload_model_depths(crops, rects), lambda: g.upload_templates(ts), lambda: g.match(b, d, 75.0),
                 lambda: g.recognize(b, d, K)):
        with pytest.raises(fb.FealessError) as e:
            call()
        assert e.value.rc == fb.FL_ERR_STATE
    r0, r1 = g.collect_recognition(), g.collect_recognition()
    assert r0[0] == r1[0] == fb.FL_OK and r0[1].tobytes() == r1[1].tobytes() and len(r0[1]) == 1 and g.in_flight() == 0
    assert g.match(b, d, 75.0)[0] == fb.FL_OK                        # matching again once nothing is in flight
    g.upload_model_depths(crops, rects)                              # a new crop set clears the set-up
    with pytest.raises(fb.FealessError) as e:
        g.submit_recognition(b, d, K)
    assert e.value.rc == fb.FL_ERR_STATE
    g.set_recognition(np.arange(ts.n_templates))
    g.upload_templates(ts)                                           # ... and so does a template upload
    with pytest.raises(fb.FealessError) as e:
        g.submit_recognition(b, d, K)
    assert e.value.rc == fb.FL_ERR_STATE
    g.close()


@pytest.mark.parametrize("devices", ["0,1", "0,1,2,3"])
def test_distinct_devices(mixed_case, devices):
    import torch
    dv = [int(x) for x in devices.split(",")]
    if torch.cuda.device_count() < max(dv) + 1:
        pytest.skip("%d GPU(s) visible, the case needs %d" % (torch.cuda.device_count(), max(dv) + 1))
    ts, crops, rects, frames, want = mixed_case
    g = fb.Group(dv, depth=4)
    g.upload_templates(ts)
    g.upload_model_depths(crops, rects)
    m = MODES[3]
    g.set_recognition(np.arange(ts.n_templates), params=fb.reco_params(top_k=m[0], per_class=m[1], th_obj_dist=m[2]))
    _same(_stream(g, frames), want[m])
    g.close()


# ---- C++: CObjRecoLmICP::SetDevices ------------------------------------------------------------------------------------------------
def _feature_dir(path, ts, depth_mm):
    import cv2
    from fealess_b200 import linemod_io
    D0 = fb.Detector()
    D0.add_template_set(ts)
    linemod_io.write_linemod(D0, str(path / "linemod_templates.yml"))
    (path / "depth").mkdir()
    png = (depth_mm.astype(np.uint32) * 10).clip(0, 65535).astype(np.uint16)       # the reference stores 0.1 mm units
    for tid in range(ts.n_templates):
        cv2.imwrite(str(path / "depth" / ("%d.png" % tid)), png)


def _write_frame(path, bgr, depth):
    with open(path, "wb") as f:
        f.write(struct.pack("<ii4d", bgr.shape[1], bgr.shape[0], *K))
        f.write(np.ascontiguousarray(bgr, np.uint8).tobytes())
        f.write(np.ascontiguousarray(depth, np.uint16).tobytes())


@pytest.fixture(scope="module")
def cpp_exe():
    fbuild.build()
    os.makedirs(OUT_DIR, exist_ok=True)
    libdir = os.path.dirname(fb.library_path())
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    exe = os.path.join(OUT_DIR, "reco_group_test")
    r = subprocess.run([cxx, "-std=c++11", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "reco_group_test.cpp"), "-o", exe, fb.library_path(), "-lz", "-Wl,-rpath," + libdir],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return exe


def _cpp_passes(out):
    lines = out.strip().split("\n")
    one = [l[len("one "):] for l in lines if l.startswith("one frame")]
    sync = [l[len("sync "):] for l in lines if l.startswith("sync frame")]
    stream = [l[len("stream "):] for l in lines if l.startswith("stream frame")]
    return lines, one, sync, stream


@pytest.mark.parametrize("devices", ["0,0", "0,0,0"])
@pytest.mark.parametrize("depth", [1, 4])
def test_cpp_set_devices_equals_one_gpu(cpp_exe, tmp_path, devices, depth):
    """SetDevices({0,0}) / ({0,0,0}): Recognition and the stream return the single-GPU class's tags and tWorld2Cam bits in every
    hypothesis mode, and throw where it throws (one hypothesis whose box leaves the frame)."""
    b, d, ts = _planted(36, 3, 62)
    _feature_dir(tmp_path, ts, d)
    frames = [(b, d), _big(b, d), synth.make_frame(W, H, 5), (np.zeros_like(b), np.zeros_like(d)), (b, d)]
    paths = []
    for i, (fb_, fd_) in enumerate(frames):
        paths.append(str(tmp_path / ("frame%d.bin" % i)))
        _write_frame(paths[-1], fb_, fd_)
    for top_k, per_class, th in MODES:
        r = subprocess.run([cpp_exe, str(tmp_path), devices, str(depth), str(top_k), "1" if per_class else "0", str(th)] + paths,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        lines, one, sync, stream = _cpp_passes(r.stdout)
        assert "one addobj 00000000" in lines and "multi addobj 00000000" in lines
        assert len(one) == len(frames) and one == sync == stream, r.stdout
        assert sum(" results 0" not in l for l in one) >= 2
        bad = [l for l in lines if l.startswith("badparams")][0].split()[1:]
        assert bad == ["80000001"] * 3
    # boxes outside the frame: Recognition throws at one hypothesis, on one GPU and over the group alike
    edge = tmp_path / "edge"
    edge.mkdir()
    b, d, ts = _edge_templates()
    _feature_dir(edge, ts, d)
    _write_frame(str(edge / "frame.bin"), b, d)
    for top_k in (1, 4):
        r = subprocess.run([cpp_exe, str(edge), devices, str(depth), str(top_k), "0", "0", str(edge / "frame.bin"), str(edge / "frame.bin")],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        lines, one, sync, stream = _cpp_passes(r.stdout)
        assert one == sync == stream, r.stdout
        assert all(l.endswith("exception") for l in one) == (top_k == 1) and len(one) == 2, r.stdout
