"""GPU (-m gpu): fl_add_template = Detector::addTemplate (SURVEY 8f rank 4) against the REFERENCE'S OWN addTemplate
(linemod.cpp:1579-1615 compiled unmodified; its erode / distanceTransform stand-ins are pinned on cv2 by tests/test_oracle_ref.py),
whose results on these views are stored in tests/golden/reference_cases.npz (oracle/make_ref_golden.py).  The template pyramid -
every feature, the cropped boxes, the bounding box - has to be identical."""
import os

import numpy as np
import pytest

import fealess_b200 as fb
import make_ref_golden as G
from fealess_b200 import synth
from helpers import sha

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref(golden_dir):
    return np.load(os.path.join(golden_dir, "reference_cases.npz"))


@pytest.mark.parametrize("case", [0, 1, 2, 3, 5])
def test_add_template_equals_the_c_oracle(case):
    """Against oracle/fl_oracle.c (flo_add_template, which tests/test_oracle_ref.py shows equal to the reference's addTemplate): runs with
    or without oracle/_ref on the box."""
    import fl_oracle_py as F
    c = CASES[case]
    W, H, T = c["W"], c["H"], c["T"]
    b, d = synth.make_frame(W, H, c["frame"])
    mask = G.train_mask(W, H, c["mask"])
    orc, ohdr, oft, obb = F.add_template(F.Detector(T), b, d, mask)
    h = fb.Handle(T, (0, 1), W, H)
    rc, hdr, ft, bb = h.add_template(b, d, mask)
    assert (rc == 0) == (orc == 0), (rc, orc)                    # (case 5, an object on the image border, has too few colour candidates: both say so)
    if orc == 0:
        assert np.array_equal(hdr, ohdr) and np.array_equal(ft, oft) and np.array_equal(bb, obb)
    else:
        assert rc == fb.FL_ERR_TRAIN
    h.close()


def test_add_template_equals_the_committed_fixture():
    """The fixture tests/golden/train_vga.npz holds the reference's own addTemplate results (oracle/make_train_golden.py; pinned by
    tests/test_oracle_ref.py); this comparison needs no oracle/_ref on the GPU box."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "train_vga.npz"))
    W, H = 640, 480
    h = fb.Handle((5, 8), (0, 1), W, H)
    for i, c in enumerate(g["cases"]):
        b, d = synth.make_frame(W, H, int(c[0]))
        mask = None if c[3] == 0 else G.ellipse(W, H, float(c[1]), float(c[2]), float(c[3]), float(c[4]), value=int(c[5]))
        rc, hdr, ft, bb = h.add_template(b, d, mask)
        want_rc = int(g["rc%d" % i])
        assert (rc == 0) == (want_rc >= 0), (i, rc, want_rc)
        if want_rc >= 0:
            assert np.array_equal(hdr, g["hdr%d" % i]) and np.array_equal(ft, g["ft%d" % i]) and np.array_equal(bb, g["bb%d" % i]), i
        else:
            assert rc == fb.FL_ERR_TRAIN
    h.close()


# the views of tests/golden/reference_cases.npz: (W, H, T, frame, mask spec); the mask is make_ref_golden.train_mask(W, H, spec)
CASES = [dict(W=W, H=H, T=T, frame=frame, mask=spec) for W, H, T, frame, spec in G.TRAIN_CASES]


@pytest.mark.parametrize("case", CASES)
def test_add_template_equals_reference(case, ref):
    W, H, T = case["W"], case["H"], case["T"]
    b, d = synth.make_frame(W, H, case["frame"])
    mask = G.train_mask(W, H, case["mask"])
    i = CASES.index(case)
    assert [sha(b), sha(d), sha(np.zeros(0, np.uint8) if mask is None else mask)] == [str(x) for x in ref["train%d_inputs_sha" % i]], \
        "synthetic inputs differ from the fixture's"
    rrc = int(ref["train_rc%d" % i])
    if rrc >= 0:
        rhdr, rft, rbb = ref["train_hdr%d" % i], ref["train_ft%d" % i], ref["train_bb%d" % i]
    h = fb.Handle(T, (0, 1), W, H)
    rc, hdr, ft, bb = h.add_template(b, d, mask)
    assert (rc == 0) == (rrc >= 0), (rc, rrc)
    if rrc >= 0:
        assert np.array_equal(hdr, rhdr), (hdr, rhdr)
        assert np.array_equal(ft, rft)
        assert np.array_equal(bb, rbb)
        assert len(ft) == sum(63 >> l for l in range(len(T))) * 2
    h.close()


def test_too_few_candidates_and_trained_template_matches_its_own_view(ref):
    """addTemplate's failure mode, and the trained pyramid going straight back into fl_upload_templates."""
    W, H, T = 640, 480, (5, 8)
    b, d = synth.make_frame(W, H, 0)
    h = fb.Handle(T, (0, 1), W, H)
    tiny = G.ellipse(W, H, 320, 240, 6, 5)                                   # too small for 63 features: both return "no template"
    assert int(ref["train_tiny_rc"]) == -1
    assert h.add_template(b, d, tiny)[0] == fb.FL_ERR_TRAIN
    # a trained template, uploaded as it comes back, matches the view it was cut from at 100 % at its own position
    mask = G.ellipse(W, H, 320, 240, 110, 80)
    rc, hdr, ft, bb = h.add_template(b, d, mask)
    assert rc == 0
    ts = synth.TemplateSet(n_levels=2, n_modalities=2, T=T, class_names=["obj"], headers=hdr.copy(), features=ft.copy(), class_of=np.zeros(1, np.int32),
                           pose13=np.zeros((1, 13), np.float32))
    h.upload_templates(ts)
    rc, got = h.match(b, d, 90.0)
    assert rc == 0 and len(got) >= 1
    # (positions live on the T = 5 grid of level 0, so the best match sits within one cell of the template's box corner)
    assert abs(int(got[0]["x"]) - int(bb[0])) <= 5 and abs(int(got[0]["y"]) - int(bb[1])) <= 5 and got[0]["similarity"] >= 90.0
    h.close()


def test_python_mirror_add_template_then_match():
    """cup_linemod::Detector mirror: addTemplate -> match on the same view finds the new class; a failed addTemplate adds nothing."""
    W, H = 640, 480
    b, d = synth.make_frame(W, H, 0)
    det = fb.Detector()
    tid, bb = det.addTemplate([b, d], "obj", G.ellipse(W, H, 320, 240, 6, 5))
    assert tid == -1 and det.numTemplates() == 0
    tid, bb = det.addTemplate([b, d], "obj", G.ellipse(W, H, 320, 240, 110, 80), pose_info=np.arange(13, dtype=np.float32))
    assert tid == 0 and det.numTemplates("obj") == 1 and bb[0] % 2 == 0 and bb[1] % 2 == 0
    tid2, _ = det.addTemplate([b, d], "obj", G.ellipse(W, H, 200, 300, 60, 140))
    assert tid2 == 1
    rc, ms = det.match([b, d], 90.0)
    assert rc == 0 and len(ms) >= 2 and {m.template_id for m in ms[:4]} >= {0, 1} and ms[0].class_id == "obj"
