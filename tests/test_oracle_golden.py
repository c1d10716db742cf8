"""CPU: the C oracle (oracle/fl_oracle.c) against the committed golden fixtures produced by oracle/oracle_cv2.py (cited
reference lines evaluated on real OpenCV primitives) and against the sha256 pins of the reference's two tables."""
import os

import numpy as np
import pytest

import fl_oracle_py as F
from fealess_b200 import synth
from helpers import rot_err, sha, tset_from_npz

NORMAL_LUT_SHA = "729e0305a1f5975a88ebb6a9ffc28013c6bf1a2113ea3c112531f44bee7b2243"   # linemod/normal_lut.i:4 (8000 bytes)
SIMILARITY_LUT_SHA = "c76b2f9271addbf9e2529e23de5b7345185a33aa9c5c29c924d8684c48dc3446"  # linemod/linemod.cpp:970 (256 bytes)


def test_reference_tables_are_reproduced():
    assert sha(F.normal_lut()) == NORMAL_LUT_SHA
    assert sha(F.similarity_lut()) == SIMILARITY_LUT_SHA
    lut = F.normal_lut().reshape(20, 20, 20)
    assert set(np.unique(lut)) == {1, 2, 4, 8, 16, 32, 64, 128}       # one-hot, never 0
    assert set(np.unique(F.similarity_lut())) == {0, 1, 2, 4}


@pytest.fixture(scope="module")
def small(golden_dir):
    z = np.load(os.path.join(golden_dir, "linemod_small.npz"))
    det = F.Detector(tuple(int(t) for t in z["T"]))
    ts = tset_from_npz(z, synth)
    det.set_templates(ts)
    assert det.process(z["bgr"], z["depth"]) == 0
    return z, det, ts


def test_front_end_matches_golden(small):
    z, det, _ = small
    for l in range(2):
        for m in range(2):
            i = l * 2 + m
            assert np.array_equal(det.quantized(l, m), z["quantized_%d" % i]), "quantized L%d M%d" % (l, m)
            assert np.array_equal(det.spread(l, m), z["spread_%d" % i]), "spread L%d M%d" % (l, m)
            for lab in range(8):
                assert sha(det.lm(l, m, lab)) == str(z["lm_sha256"][i * 8 + lab]), "LM L%d M%d label %d" % (l, m, lab)
    assert np.array_equal(det.lm(1, 0, 3), z["lm_L1_M0_label3"])


@pytest.mark.parametrize("thr", [75, 55])
def test_match_lists_match_golden(small, thr):
    z, det, _ = small
    raw = det.match(float(thr), canonical=False)
    fin = det.match(float(thr), canonical=True)
    assert np.array_equal(raw, z["raw_%d" % thr])          # emission order: template-major, then row-major cells
    assert np.array_equal(fin, z["final_%d" % thr])
    assert len(fin) > 0
    assert np.array_equal(det.match(float(thr), n_threads=4), fin)     # OpenMP variant is result-identical


def test_class_filter_and_masks_match_golden(small):
    z, det, ts = small
    assert np.array_equal(det.match(55.0, class_filter=[1]), z["final_55_class1"])
    det2 = F.Detector(tuple(int(t) for t in z["T"]))
    det2.set_templates(ts)
    assert det2.process(z["bgr"], z["depth"], masks=[z["mask_0"], z["mask_1"]]) == 0
    for i in range(4):
        assert np.array_equal(det2.quantized(i // 2, i % 2), z["mquantized_%d" % i])
    assert np.array_equal(det2.match(60.0), z["mfinal_60"])


def test_vga_hashes(golden_dir):
    z = np.load(os.path.join(golden_dir, "linemod_vga_hashes.npz"))
    bgr, depth = synth.make_frame(640, 480, 0)
    if sha(bgr) != str(z["bgr_sha"]) or sha(depth) != str(z["depth_sha"]):
        pytest.skip("numpy RNG stream differs from the one the fixture was generated with")
    det = F.Detector((5, 8))
    assert det.process(bgr, depth) == 0
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    assert [sha(x) for x in q] == [str(s) for s in z["quantized_sha"]]
    assert [sha(det.spread(l, m)) for l in range(2) for m in range(2)] == [str(s) for s in z["spread_sha"]]
    assert [sha(det.lm(l, m, lab)) for l in range(2) for m in range(2) for lab in range(8)] == [str(s) for s in z["lm_sha"]]
    ts = synth.make_templates(120, 640, 480, (5, 8), n_classes=2, seed=4, quantized=q, planted_fraction=0.1)
    assert sha(ts.headers) == str(z["headers_sha"]) and sha(ts.features) == str(z["features_sha"])
    det.set_templates(ts)
    assert np.array_equal(det.match(75.0, canonical=False), z["raw_75"])
    assert np.array_equal(det.match(75.0), z["final_75"])


def test_phase_bins_match_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "phase_bins.npz"))
    q = F.phase_q16(z["dx"].astype(np.float32), z["dy"].astype(np.float32))
    assert np.array_equal(q, z["q"])


def test_geometry_and_feature_limits():
    det = F.Detector((5, 8))
    b, d = synth.make_frame(648, 480, 1)            # 648 % 5 != 0  -> CV_Assert in linearize (linemod.cpp:1062-1063)
    assert det.process(b, d) == -2
    ts = synth.make_templates(2, 640, 480, (5, 8), seed=1)
    ts.headers[0, 6] = 64                           # > 63 features -> CV_Assert (linemod.cpp:1137)
    with pytest.raises(ValueError):
        det.set_templates(ts)


def test_icp_matches_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "icp_small.npz"))
    K = tuple(float(v) for v in z["K"])
    iters = []
    for i in range(int(z["n_cases"])):
        p = z["rt_match_%d" % i]
        R0, t0 = p[:12].reshape(3, 4)[:, :3], p[:12].reshape(3, 4)[:, 3]
        rm, rr = z["rects_%d" % i]
        r = F.detection(z["model_%d" % i], z["ref_%d" % i], K, rm, rr, r_match=R0, t_match=t0)
        dm, ratio, it, npts = z["scalars_%d" % i]
        assert r["rc"] == 0 and r["n_points"] == int(npts)
        assert r["iterations"] == int(it), "case %d: iteration count" % i
        # tolerance of the task (BASELINE.json north_star): 1e-4 rad rotation, 1e-4 m = 0.1 mm translation.  Observed between
        # the two CPU restatements: <= 3.3e-5 rad / 6.5e-3 mm (5-iteration case; the difference is cv2's SVD vs the restated one,
        # amplified ~150x by the reference's uncentred covariance).
        assert rot_err(r["R"], z["R_%d" % i]) < 1e-4
        assert np.abs(r["T"] - z["T_%d" % i]).max() < 0.1
        assert abs(float(r["dist_mean"]) - dm) < 1e-3
        iters.append(int(it))
    assert max(iters) >= 4 and min(iters) <= 2      # the fixture exercises short and long runs


def test_icp_degenerate_inputs():
    r = F.icp_cloud_to_cloud_ex(np.zeros((2, 3), np.float32), np.zeros((2, 3), np.float32))
    assert r["dist_mean"] == -1 and r["iterations"] == 0 and not r["R"].any()    # ICP.cpp:633-638
    depth = np.full((48, 64), 700, np.uint16)
    res = F.detection(depth, depth, (608, 608, 32, 24), (50, 10, 30, 30), (0, 0, 30, 30))
    assert res["rc"] == -3                                                       # rect leaves the image (detection.cpp:43-44)


def test_nms_matches_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "icp_small.npz"))
    assert np.array_equal(F.nms(z["nms_t3"], z["nms_n"], z["nms_dist"], 25.0), z["nms_out_th25"])
    assert np.array_equal(F.nms(z["nms_t3"], z["nms_n"], z["nms_dist"], 8.0), z["nms_out_th8"])
    assert len(F.nms(np.zeros((0, 3)), [], [], 1.0)) == 0


def test_reference_cases_fixture(golden_dir):
    """tests/golden/reference_cases.npz, the reference's results that the GPU reference tests compare with (oracle/make_ref_golden.py):
    the C oracle reproduces every entry, so the oracle stays pinned on the reference's results where oracle/_ref is not built."""
    import make_ref_golden as G
    z = np.load(os.path.join(golden_dir, "reference_cases.npz"))
    got = G.compute(F)
    assert sorted(got) == sorted(z.files)
    for k in z.files:
        assert np.array_equal(got[k], z[k]), k
