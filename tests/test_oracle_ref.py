"""CPU: pins the oracle on the REFERENCE ITSELF.

oracle/_ref/libfl_ref.so is /root/reference/linemod/linemod.cpp + ICP/{ICP,NMS,common,detection,depth_to_3d}.cpp compiled
unmodified (oracle/build_ref.py) against a stand-in for the OpenCV API (oracle/ref_shim).  These tests show, on the golden
fixture and on VGA / 720p inputs:

  (1) oracle/fl_oracle.c == the reference's own code, bit for bit, for every integer stage of Detector::match
      (quantised images, spread images, response maps, linear memories, similarity / similarityLocal maps, the pre-sort match
      list of matchClass, class filters, masks, the CV_Assert cases) and for depthTo3d, matToVec pairing, NMS and the ICP
      poses (icpCloudToCloud_Ex / detection: bit-identical R, T, dist_mean and inlier ratio);
  (2) the real Detector::match (with its own std::sort / std::unique) returns the oracle's canonical list as a set, with
      the same top-1 match;
  (3) the stand-in's image / maths primitives == the real cv2 4.13 of this image, and the reference's code run ON cv2's
      primitives (plugged in through callbacks) gives byte-identical results to the run on the stand-in's.
"""
import os

import numpy as np
import pytest

import fl_oracle_py as F
import fl_ref_py as R
from fealess_b200 import synth
from helpers import canonical, rot_err, tset_from_npz

pytestmark = pytest.mark.skipif(not R.available(), reason="oracle/_ref/libfl_ref.so neither built nor buildable here")


def _pair(T=(5, 8)):
    return F.Detector(tuple(T)), R.Detector(tuple(T))


def _frame_with_templates(W, H, n, T=(5, 8), frame_idx=0, n_classes=2, planted=0.03, seed=3):
    bgr, depth = synth.make_frame(W, H, frame_idx)
    fo, fr = _pair(T)
    assert fo.process(bgr, depth) == 0
    L = len(T)
    quant = [fo.quantized(l, m) for l in range(L) for m in range(2)]
    ts = synth.make_templates(n, W, H, T, n_classes=n_classes, seed=seed, quantized=quant, planted_fraction=planted)
    fo.set_templates(ts)
    fr.set_templates(ts)
    assert fo.process(bgr, depth) == 0 and fr.process(bgr, depth) == 0
    return bgr, depth, ts, fo, fr


def test_library_is_the_reference_build():
    assert b"compiled unmodified" in R.lib().flr_version()
    info = os.path.join(os.path.dirname(R.build_ref.SO), "BUILD_INFO.txt")
    if os.path.exists(info):
        txt = open(info).read()
        for f in ("linemod/linemod.cpp", "ICP/ICP.cpp", "ICP/NMS.cpp", "ICP/detection.cpp", "ICP/depth_to_3d.cpp", "ICP/common.cpp"):
            assert f in txt


# ------------------------------------------------------------------------------------------------ stage functions
@pytest.mark.parametrize("size,idx", [((640, 480), 0), ((640, 480), 3), ((320, 160), 1), ((1280, 720), 2)])
def test_stage_functions_equal_reference(size, idx):
    W, H = size
    bgr, depth = synth.make_frame(W, H, idx)
    qo, mo = F.color_quantize(bgr, want_mag=True)
    qr, mr = R.color_quantize(bgr, want_mag=True)                      # quantizedOrientations + hysteresisGradient, :230-385
    assert np.array_equal(qo, qr) and np.array_equal(mo, mr)
    assert (qo != 0).mean() > 0.02
    do, dr = F.depth_quantize(depth), R.depth_quantize(depth)          # quantizedNormals, :595-685
    assert np.array_equal(do, dr)
    for q in (qo, do):
        for T in (5, 8, 4):
            so, sr = F.spread(q, T), R.spread(q, T)                    # spread / orUnaligned8u, :882-965
            assert np.array_equal(so, sr)
        ro, rr = F.response_maps(so), R.response_maps(so)              # computeResponseMaps (SSSE3 branch), :979-1048
        assert np.array_equal(ro, rr)
        for T in (5, 8):
            for lab in (0, 5):
                assert np.array_equal(F.linearize(ro[lab], T), R.linearize(ro[lab], T))   # linearize, :1060-1088


def test_stage_functions_on_edge_inputs():
    rng = np.random.default_rng(5)
    W, H = 160, 80
    flat = np.full((H, W, 3), 128, np.uint8)
    assert not R.color_quantize(flat).any() and np.array_equal(F.color_quantize(flat), R.color_quantize(flat))
    noise = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    assert np.array_equal(F.color_quantize(noise), R.color_quantize(noise))
    far = np.full((H, W), 2500, np.uint16)                              # beyond distance_threshold -> all zero (:628)
    assert not R.depth_quantize(far).any()
    d = rng.integers(400, 3000, (H, W)).astype(np.uint16)
    d[rng.random((H, W)) < 0.1] = 0                                     # holes
    assert np.array_equal(F.depth_quantize(d), R.depth_quantize(d))
    q = (1 << rng.integers(0, 8, (H, W))).astype(np.uint8) * (rng.random((H, W)) < 0.2)
    for T in (1, 2, 5, 8, 16):
        assert np.array_equal(F.spread(q.astype(np.uint8), T), R.spread(q.astype(np.uint8), T))
    with pytest.raises(ValueError):                                     # (rows * cols) % 16 != 0 -> CV_Assert (:981)
        R.response_maps(np.zeros((3, 5), np.uint8))
    with pytest.raises(ValueError):                                     # cols % T != 0 -> CV_Assert (:1062-1063)
        R.linearize(np.zeros((80, 162), np.uint8), 5)


# ------------------------------------------------------------------------------------------------ golden fixture
@pytest.fixture(scope="module")
def small(golden_dir):
    z = np.load(os.path.join(golden_dir, "linemod_small.npz"))
    T = tuple(int(t) for t in z["T"])
    fo, fr = _pair(T)
    ts = tset_from_npz(z, synth)
    fo.set_templates(ts)
    fr.set_templates(ts)
    assert fo.process(z["bgr"], z["depth"]) == 0 and fr.process(z["bgr"], z["depth"]) == 0
    return z, fo, fr, ts


def test_reference_reproduces_the_golden_fixture(small):
    """The fixture was written by oracle/oracle_cv2.py (cited lines on cv2 primitives); the reference's own code agrees."""
    z, fo, fr, ts = small
    for l in range(2):
        for m in range(2):
            i = l * 2 + m
            assert np.array_equal(fr.quantized(l, m), z["quantized_%d" % i])
            assert np.array_equal(fr.spread(l, m), z["spread_%d" % i])
            for lab in range(8):
                assert np.array_equal(fr.lm(l, m, lab), fo.lm(l, m, lab))
    assert np.array_equal(fr.lm(1, 0, 3), z["lm_L1_M0_label3"])
    for thr in (75, 55):
        raw = fr.match(float(thr))
        assert np.array_equal(raw, z["raw_%d" % thr])                   # matchClass emission order, bit for bit
        assert np.array_equal(canonical(raw), z["final_%d" % thr])
        rc, full = fr.match_full(z["bgr"], z["depth"], float(thr))      # the REAL Detector::match incl. std::sort / std::unique
        assert rc == 0
        assert set(map(tuple, full.tolist())) == set(map(tuple, z["final_%d" % thr].tolist()))
        assert tuple(full[0]) [:4] == tuple(z["final_%d" % thr][0])[:4]
        for i in range(4):
            assert np.array_equal(fr.match_quantized(i // 2, i % 2), z["quantized_%d" % i])   # `quantized_images` output (:1411-1412)
    assert np.array_equal(canonical(fr.match(55.0, class_filter=[1])), z["final_55_class1"])
    rc, full = fr.match_full(z["bgr"], z["depth"], 55.0, class_filter=[1])
    assert rc == 0 and set(map(tuple, full.tolist())) == set(map(tuple, z["final_55_class1"].tolist()))
    # masks (:1366-1378, 455-459, 741-745)
    masks = [z["mask_0"], z["mask_1"]]
    assert fr.process(z["bgr"], z["depth"], masks=masks) == 0
    for i in range(4):
        assert np.array_equal(fr.quantized(i // 2, i % 2), z["mquantized_%d" % i])
    assert np.array_equal(canonical(fr.match(60.0)), z["mfinal_60"])
    rc, full = fr.match_full(z["bgr"], z["depth"], 60.0, masks=masks)
    assert rc == 0 and set(map(tuple, full.tolist())) == set(map(tuple, z["mfinal_60"].tolist()))
    assert fr.process(z["bgr"], z["depth"]) == 0


def test_similarity_maps_equal_reference(small):
    z, fo, fr, ts = small
    nz = 0
    for t in range(ts.n_templates):
        a, b = fo.similarity(t), fr.similarity(t)                       # similarity + addSimilarities (:1130-1214, 1322-1338)
        assert np.array_equal(a, b), t
        nz += int(b.any())
    assert nz == ts.n_templates


# ------------------------------------------------------------------------------------------------ VGA / 720p, many templates
@pytest.mark.parametrize("cfg", [dict(W=640, H=480, n=1500, T=(5, 8), classes=3), dict(W=1280, H=720, n=400, T=(5, 8), classes=15),
                                 dict(W=640, H=480, n=300, T=(4, 8, 8), classes=2)])
def test_match_lists_equal_reference(cfg):
    bgr, depth, ts, fo, fr = _frame_with_templates(cfg["W"], cfg["H"], cfg["n"], cfg["T"], n_classes=cfg["classes"])
    L = len(cfg["T"])
    for l in range(L):
        for m in range(2):
            assert np.array_equal(fo.quantized(l, m), fr.quantized(l, m))
            assert np.array_equal(fo.spread(l, m), fr.spread(l, m))
            for lab in range(8):
                assert np.array_equal(fo.lm(l, m, lab), fr.lm(l, m, lab))
    n_seen = 0
    for thr in (75.0, 60.0):
        raw_o, raw_r = fo.match(thr, canonical=False), fr.match(thr)
        assert np.array_equal(raw_o, raw_r)                             # pre-sort list of matchClass (:1451-1577), every template
        n_seen += len(raw_r)
        fin = fo.match(thr, canonical=True)
        rc, full = fr.match_full(bgr, depth, thr)
        assert rc == 0
        assert set(map(tuple, full.tolist())) == set(map(tuple, fin.tolist()))
        if len(fin):
            assert tuple(full[0])[:4] == tuple(fin[0])[:4]              # x, y, similarity, class of the best match
            assert np.array_equal(full["similarity"], np.sort(full["similarity"])[::-1])
    assert n_seen > 20
    cf = [cfg["classes"] - 1]
    assert np.array_equal(fo.match(60.0, class_filter=cf, canonical=False), fr.match(60.0, class_filter=cf))


def test_similarity_local_equals_reference_through_refinement():
    """similarityLocal (:1226-1300) is reached through matchClass' refinement; its 16x16 maps are also compared directly with
    a numpy evaluation of the linear memories the oracle holds."""
    bgr, depth, ts, fo, fr = _frame_with_templates(640, 480, 200, planted=0.1)
    raw = fr.match(60.0)
    assert len(raw) > 0
    T0, Wc = 5, 640 // 5
    for rec in raw[:6]:
        t = int(np.nonzero((ts.class_of == rec["class_idx"]))[0][rec["template_id"]])
        x, y = int(rec["x"]), int(rec["y"])
        got = fr.similarity_local(t, 0, x, y)
        want = np.zeros((16, 16), np.uint16)
        ox, oy = (x // T0 - 8) * T0, (y // T0 - 8) * T0
        for m in range(2):
            acc = np.zeros((16, 16), np.uint8)
            _, feats = ts.template(t, 0, m)
            for fx, fy, lab in feats:
                px, py = fx + ox, fy + oy
                if px < 0 or py < 0 or px >= 640 or py >= 480:
                    continue
                lmem = fo.lm(0, m, int(lab))[(py % T0) * T0 + px % T0]
                base = (py // T0) * Wc + px // T0
                for r in range(16):
                    acc[r] += lmem[base + r * Wc: base + r * Wc + 16]
            want += acc
        assert np.array_equal(got, want)


def test_error_behaviour_equals_reference():
    fo, fr = _pair((5, 8))
    b, d = synth.make_frame(640, 488, 1)                                # 244 % 8 != 0 at level 1 -> CV_Assert (:1062-1063)
    assert fo.process(b, d) == -2 and fr.process(b, d) == -2
    rc, _ = fr.match_full(b, d)
    assert rc == -2 and "response_map" in fr.last_error()
    # an empty template set: the front end runs, the list is empty
    b, d = synth.make_frame(320, 160, 1)
    rc, full = R.Detector((5, 8)).match_full(b, d)
    assert rc == 0 and len(full) == 0


# ------------------------------------------------------------------------------------------------ ICP side
def test_backprojection_and_pairing_equal_reference():
    _, depth = synth.make_frame(640, 480, 2)
    a, b = F.depth_to_3d_mm(depth, 608, 608, 320, 240), R.depth_to_3d_mm(depth, 608, 608, 320, 240)   # depth_to_3d.cpp:99-137, 244-269
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    a2, b2 = F.depth_to_3d_mm(depth, 611.5, 609.25, 317.3, 242.9), R.depth_to_3d_mm(depth, 611.5, 609.25, 317.3, 242.9)
    assert np.array_equal(a2.view(np.uint32), b2.view(np.uint32))
    assert np.isnan(b[depth == 0]).all()
    n, pr, pm = R.pair_points(a, a2, (100, 80, 120, 90), (140, 60, 120, 90))                           # matToVec, common.cpp:395-416
    pr_o = np.zeros((120 * 90, 3), np.float32)
    pm_o = np.zeros((120 * 90, 3), np.float32)
    n_o = F.lib().flo_pair_points(F._p(np.ascontiguousarray(a)), F._p(np.ascontiguousarray(a2)), 640, 480,
                                  F._p(np.array([100, 80, 120, 90], np.int32)), F._p(np.array([140, 60, 120, 90], np.int32)), F._p(pr_o), F._p(pm_o))
    assert n == n_o and np.array_equal(pr, pr_o[:n]) and np.array_equal(pm, pm_o[:n])
    assert R.pair_points(a, a2, (600, 80, 120, 90), (140, 60, 120, 90))[0] == -3                       # ROI outside the frame


def test_icp_equals_reference(golden_dir):
    z = np.load(os.path.join(golden_dir, "icp_small.npz"))
    K = tuple(float(v) for v in z["K"])
    worst_r, worst_t = 0.0, 0.0
    for i in range(int(z["n_cases"])):
        p = z["rt_match_%d" % i]
        R0, t0 = p[:12].reshape(3, 4)[:, :3], p[:12].reshape(3, 4)[:, 3]
        rm, rr = z["rects_%d" % i]
        o = F.detection(z["model_%d" % i], z["ref_%d" % i], K, rm, rr, r_match=R0, t_match=t0)
        r = R.detection(z["model_%d" % i], z["ref_%d" % i], K, rm, rr, r_match=R0, t_match=t0)          # detection.cpp:11-254
        assert o["rc"] == 0 and r["rc"] == 0
        worst_r = max(worst_r, rot_err(o["R"], r["R"]))
        worst_t = max(worst_t, float(np.abs(o["T"] - r["T"]).max()))
        # and against the cv2-evaluated fixture, at the task's tolerance (1e-4 rad, 0.1 mm)
        assert rot_err(r["R"], z["R_%d" % i]) < 1e-4 and np.abs(r["T"] - z["T_%d" % i]).max() < 0.1
    assert worst_r == 0.0 and worst_t == 0.0, (worst_r, worst_t)        # bit-identical poses on all eight cases (2..5 iterations)
    # the cloud API, with more iterations (synthetic pairs with a larger offset)
    for seed in range(3):
        model, ref, rm, rr, _ = synth.make_icp_pair(640, 480, seed, max_shift_mm=15.0, max_rot_deg=7.0)
        a = F.depth_to_3d_mm(model, 608, 608, 320, 240)
        b = F.depth_to_3d_mm(ref, 608, 608, 320, 240)
        n, pr, pm = R.pair_points(b, a, rr, rm)
        o = F.icp_cloud_to_cloud_ex(pr, pm, 10, 0.05, 0.0001)
        r = R.icp_cloud_to_cloud_ex(pr, pm, 10, 0.05, 0.0001)                                           # ICP.cpp:617-809
        assert o["iterations"] >= 2
        assert np.array_equal(o["R"], r["R"]) and np.array_equal(o["T"], r["T"])
        assert float(o["dist_mean"]) == float(r["dist_mean"]) and float(o["inlier_ratio"]) == float(r["inlier_ratio"])


def test_icp_degenerate_inputs_equal_reference():
    r = R.icp_cloud_to_cloud_ex(np.zeros((2, 3), np.float32), np.zeros((2, 3), np.float32))
    o = F.icp_cloud_to_cloud_ex(np.zeros((2, 3), np.float32), np.zeros((2, 3), np.float32))
    assert r["dist_mean"] == -1 and o["dist_mean"] == -1                                                # ICP.cpp:633-638
    depth = np.full((48, 64), 700, np.uint16)
    assert R.detection(depth, depth, (608, 608, 32, 24), (50, 10, 30, 30), (0, 0, 30, 30))["rc"] == -3   # detection.cpp:43-44
    # every point invalid (z > 900): no pairs -> ICP refuses (< 3 points), pose = r_match / garbage-free
    far = np.full((48, 64), 950, np.uint16)
    ro = F.detection(far, far, (608, 608, 32, 24), (5, 5, 30, 30), (5, 5, 30, 30))
    rr = R.detection(far, far, (608, 608, 32, 24), (5, 5, 30, 30), (5, 5, 30, 30))
    assert ro["rc"] == 0 and rr["rc"] == 0 and ro["n_points"] == 0


def test_nms_equals_reference(golden_dir):
    z = np.load(os.path.join(golden_dir, "icp_small.npz"))
    assert np.array_equal(R.nms(z["nms_t3"], z["nms_n"], z["nms_dist"], 25.0), z["nms_out_th25"])       # NMS.cpp:6-39
    assert np.array_equal(R.nms(z["nms_t3"], z["nms_n"], z["nms_dist"], 8.0), z["nms_out_th8"])
    rng = np.random.default_rng(11)
    for n in (0, 1, 2, 17, 300):
        t3 = rng.uniform(-60, 60, (n, 3)).astype(np.float32)
        nm = rng.integers(50, 12000, n).astype(np.int32)
        dd = rng.uniform(0, 3, n).astype(np.float32)
        for th in (5.0, 30.0, 500.0):
            assert np.array_equal(F.nms(t3, nm, dd, th), R.nms(t3, nm, dd, th))


# ------------------------------------------------------------------------------------------------ the stand-in's primitives vs cv2
cv2 = pytest.importorskip("cv2")


def test_shim_primitives_equal_cv2():
    try:
        cv2.ipp.setUseIPP(False)
    except Exception:
        pass
    rng = np.random.default_rng(2)
    for (W, H, idx) in ((640, 480, 4), (322, 162, 5)):
        bgr, depth = synth.make_frame(W, H, idx)
        sm = R.prim_gaussian7(bgr)
        assert np.array_equal(sm, cv2.GaussianBlur(bgr, (7, 7), 0, 0, borderType=cv2.BORDER_REPLICATE))
        dx, dy = R.prim_sobel(sm)
        assert np.array_equal(dx, cv2.Sobel(sm, cv2.CV_16S, 1, 0, ksize=3, borderType=cv2.BORDER_REPLICATE))
        assert np.array_equal(dy, cv2.Sobel(sm, cv2.CV_16S, 0, 1, ksize=3, borderType=cv2.BORDER_REPLICATE))
        fx, fy = dx[..., 0].astype(np.float32), dy[..., 0].astype(np.float32)
        ang, q = R.prim_phase_q(fx, fy)
        ref_ang = cv2.phase(fx, fy, angleInDegrees=True).ravel()
        assert np.abs(ang - ref_ang).max() < 1e-4                         # <= 1 ulp of a degree value
        ref_q = cv2.convertScaleAbs(ref_ang.reshape(1, -1), alpha=16.0 / 360.0).ravel()
        assert np.array_equal(q, ref_q)
        lab = (1 << rng.integers(0, 8, (H, W))).astype(np.uint8) * (rng.random((H, W)) < 0.6).astype(np.uint8)
        assert np.array_equal(R.prim_median5(lab), cv2.medianBlur(lab, 5))
        if W % 2 == 0 and H % 2 == 0:
            assert np.array_equal(R.prim_pyrdown(bgr), cv2.pyrDown(bgr, dstsize=(W // 2, H // 2)))
            assert np.array_equal(R.prim_resize_nn_half(lab), cv2.resize(lab, (W // 2, H // 2), interpolation=cv2.INTER_NEAREST))
    ref = rng.uniform(0, 200, (4000, 3)).astype(np.float32)
    qs = rng.uniform(0, 200, (1500, 3)).astype(np.float32)
    idx, dist = R.prim_knn1(ref, qs)
    index = cv2.flann_Index(ref, dict(algorithm=4, leaf_max_size=15))      # KDTREE_SINGLE, as ICP.cpp:658
    i2, d2 = index.knnSearch(qs, 1, params=dict(checks=32, eps=0.0, sorted=True))
    assert np.array_equal(idx, i2.ravel()) and np.array_equal(dist, d2.ravel())
    for _ in range(50):
        c = (rng.normal(size=(3, 3)) * rng.choice([1.0, 1e3, 1e6])).astype(np.float32)
        w, u, vt = cv2.SVDecomp(c)                                        # cv::SVD::compute + Mat(vt.t() * u.t()), ICP.cpp:741-744
        want = cv2.gemm(vt, u, 1.0, None, 0.0, flags=cv2.GEMM_1_T | cv2.GEMM_2_T)
        assert np.array_equal(R.svd3_rot(c), want) and np.array_equal(F.svd3_rot(c), want)


def test_reference_on_real_cv2_primitives_is_identical():
    """Plug cv2's GaussianBlur / Sobel / phase / medianBlur / pyrDown / resize / SVDecomp / flann into the stand-in and run
    the reference's code again: every result is byte-identical to the run on the stand-in's own primitives."""
    bgr, depth, ts, fo, fr = _frame_with_templates(640, 480, 400, planted=0.05, frame_idx=6)
    rc, full0 = fr.match_full(bgr, depth, 65.0)
    lms0 = [fr.lm(l, m, lab) for l in range(2) for m in range(2) for lab in range(8)]
    model, ref, rm, rr, _ = synth.make_icp_pair(640, 480, 1, max_shift_mm=12.0, max_rot_deg=6.0)
    K = (608., 608., 320., 240.)
    d0 = R.detection(model, ref, K, rm, rr)
    R.hook_calls.clear()
    R.install_cv2_hooks()
    try:
        assert fr.process(bgr, depth) == 0
        rc, full1 = fr.match_full(bgr, depth, 65.0)
        lms1 = [fr.lm(l, m, lab) for l in range(2) for m in range(2) for lab in range(8)]
        d1 = R.detection(model, ref, K, rm, rr)
    finally:
        R.remove_hooks()
    assert all(R.hook_calls.get(op, 0) > 0 for op in range(9)), R.hook_calls
    assert len(full0) > 0 and np.array_equal(full0, full1)
    assert all(np.array_equal(a, b) for a, b in zip(lms0, lms1))
    assert np.array_equal(d0["R"], d1["R"]) and np.array_equal(d0["T"], d1["T"])
    assert fr.process(bgr, depth) == 0


def test_training_primitives_of_the_shim_equal_cv2():
    """cv::erode (3x3, BORDER_REPLICATE, 1 and 2 iterations) and cv::distanceTransform(DIST_C, 3) are called by template training only
    (linemod.cpp:466, 753, 765); the stand-ins the reference is compiled against equal the real cv2, including the image without a
    zero pixel (65535 in OpenCV 4.13's own code; with IPP on, Intel's routine returns FLT_MAX there - the stand-in follows OpenCV's code)."""
    cv2 = pytest.importorskip("cv2")
    use_ipp = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        _check_training_primitives(cv2)
    finally:
        cv2.ipp.setUseIPP(use_ipp)


def _check_training_primitives(cv2):
    rng = np.random.default_rng(0)
    for t in range(20):
        H, W = int(rng.integers(8, 90)), int(rng.integers(8, 120))
        m = (rng.random((H, W)) < rng.uniform(0.5, 0.98)).astype(np.uint8) * 255
        if t % 5 == 0:
            m[:] = 255
        for it in (1, 2):
            assert np.array_equal(R.prim_erode3(m, it), cv2.erode(m, None, iterations=it, borderType=cv2.BORDER_REPLICATE))
        assert np.array_equal(R.prim_distance_c3(m), cv2.distanceTransform(m, cv2.DIST_C, 3))


def test_reference_add_template_runs_and_is_deterministic():
    """Detector::addTemplate of the reference through the glue: 63 + 63 features at level 0, 31 + 31 at level 1, boxes cropped to the
    features; a mask too small for 63 features returns -1."""
    from fealess_b200 import synth
    W, H = 640, 480
    b, d = synth.make_frame(W, H, 0)
    yy, xx = np.mgrid[0:H, 0:W]
    mask = ((((xx - 320) / 110.0) ** 2 + ((yy - 240) / 80.0) ** 2) <= 1.0).astype(np.uint8) * 255
    det = R.Detector((5, 8))
    rc, hdr, ft, bb = R.add_template(det, b, d, mask)
    assert rc == 0 and hdr[:, 6].tolist() == [63, 63, 31, 31] and len(ft) == 188
    assert (hdr[:2, 0] == bb[2]).all() and (hdr[:2, 1] == bb[3]).all() and bb[0] % 2 == 0 and bb[1] % 2 == 0
    rc2, hdr2, ft2, bb2 = R.add_template(det, b, d, mask)
    assert rc2 == 0 and np.array_equal(hdr, hdr2) and np.array_equal(ft, ft2)
    tiny = ((((xx - 320) / 6.0) ** 2 + ((yy - 240) / 5.0) ** 2) <= 1.0).astype(np.uint8) * 255
    assert R.add_template(det, b, d, tiny)[0] == -1


def test_training_fixture_is_what_the_reference_returns():
    """tests/golden/train_vga.npz (oracle/make_train_golden.py) = the reference's own addTemplate on four synthetic views; the GPU test
    compares fl_add_template with the fixture, so it also runs where oracle/_ref is not built."""
    from fealess_b200 import synth
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "train_vga.npz"))
    W, H = 640, 480
    det = R.Detector((5, 8))
    yy, xx = np.mgrid[0:H, 0:W]
    for i, c in enumerate(g["cases"]):
        b, d = synth.make_frame(W, H, int(c[0]))
        mask = None if c[3] == 0 else ((((xx - c[1]) / c[3]) ** 2 + ((yy - c[2]) / c[4]) ** 2) <= 1.0).astype(np.uint8) * int(c[5])
        rc, hdr, ft, bb = R.add_template(det, b, d, mask)
        assert rc == int(g["rc%d" % i])
        if rc >= 0:
            assert np.array_equal(hdr, g["hdr%d" % i]) and np.array_equal(ft, g["ft%d" % i]) and np.array_equal(bb, g["bb%d" % i])


def test_reference_cases_fixture_is_what_the_reference_returns(golden_dir):
    """tests/golden/reference_cases.npz (oracle/make_ref_golden.py) = the reference's own code on the inputs of tests/test_gpu_ref.py
    and of the reference cases of tests/test_gpu_train.py, entry for entry; and the real Detector::match (its own std::sort /
    std::unique) returns the stored lists as sets, with the same best match and the stored `quantized_images`."""
    import make_ref_golden as G
    from helpers import sha
    z = np.load(os.path.join(golden_dir, "reference_cases.npz"))
    got = G.compute(R)
    assert sorted(got) == sorted(z.files)
    for k in z.files:
        assert np.array_equal(got[k], z[k]), k
    for k, c in enumerate(G.MATCH_CFGS):
        b, d, ts, det = G.match_setup(R, c["W"], c["H"], c["T"], c["n"], c["classes"])
        for thr in (75, 60):
            want = z["m%d_final_%d" % (k, thr)]
            rc, full = det.match_full(b, d, float(thr))
            assert rc == 0 and set(map(tuple, full.tolist())) == set(map(tuple, want.tolist()))
            if len(want):
                assert tuple(full[0])[:4] == tuple(want[0])[:4]
            L = len(c["T"])
            assert [sha(det.match_quantized(l, m)) for l in range(L) for m in range(2)] == [str(x) for x in z["m%d_quantized_sha" % k]]


def test_c_oracle_training_equals_the_reference():
    """flo_add_template (oracle/fl_oracle.c) == the reference's own Detector::addTemplate: every feature, cropped box and bounding box, for
    masks of several shapes and values, no mask, two and three pyramid levels, and the too-few-candidates case; its erode / distance
    transform equal cv2 (IPP off: OpenCV's own code)."""
    cv2 = pytest.importorskip("cv2")
    from fealess_b200 import synth
    use_ipp = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        rng = np.random.default_rng(1)
        for t in range(12):
            H, W = int(rng.integers(8, 90)), int(rng.integers(8, 120))
            m = (rng.random((H, W)) < rng.uniform(0.5, 0.98)).astype(np.uint8) * 255
            if t % 4 == 0:
                m[:] = 255
            for it in (1, 2):
                assert np.array_equal(F.erode3(m, it), cv2.erode(m, None, iterations=it, borderType=cv2.BORDER_REPLICATE))
            assert np.array_equal(F.distance_c3(m), cv2.distanceTransform(m, cv2.DIST_C, 3))
    finally:
        cv2.ipp.setUseIPP(use_ipp)
    W, H = 640, 480
    yy, xx = np.mgrid[0:H, 0:W]
    n_ok = 0
    for T in ((5, 8), (4, 8, 8)):
        fd, rd = F.Detector(T), R.Detector(T)
        for frame, ell, val in ((0, (320, 240, 110, 80), 255), (0, (300, 250, 120, 90), 1), (2, None, 0), (3, (320, 240, 6, 5), 255)):
            b, d = synth.make_frame(W, H, frame)
            mask = None if ell is None else ((((xx - ell[0]) / ell[2]) ** 2 + ((yy - ell[1]) / ell[3]) ** 2) <= 1.0).astype(np.uint8) * val
            a, r = F.add_template(fd, b, d, mask), R.add_template(rd, b, d, mask)
            assert (a[0] == 0) == (r[0] >= 0), (T, frame)
            if r[0] >= 0:
                assert np.array_equal(a[1], r[1]) and np.array_equal(a[2], r[2]) and np.array_equal(a[3], r[3]), (T, frame)
                n_ok += 1
    assert n_ok == 6
