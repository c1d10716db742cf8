"""GPU (-m gpu): the staged similarity kernel visits its phases by the frame's response mass (lightest first) and that changes no result.

Every case compares the whole match list with the C oracle record for record, once in the default order and once with
FL_OPT_SIM_ROTATE (the rotated order of CTA b) on the same handle.  The order the kernel used, and the response sums it derived
it from, are read back (FL_DBG_STAGED_ORDER) and compared with the CPU replay (tools/exp_prune_count.py) on the oracle's linear
memories: the sums must be equal word for word."""
import os
import sys

import numpy as np
import pytest

import fealess_b200 as fb
import fl_oracle_py as F
import staged_cases as sc
import test_gpu_similarity_plans as plans
from fealess_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import exp_prune_count as E  # noqa: E402

pytestmark = pytest.mark.gpu

W, H, T = 640, 480, (5, 8)
CAP = 1 << 19


def _both(h, b, d, thr, masks=None):
    """The match list in the default phase order and in the rotated one (FL_OPT_SIM_ROTATE), from one handle."""
    out = []
    for rot in (0, 1):
        assert h.debug_option(fb.FL_OPT_SIM_ROTATE, rot) == 0
        rc, got = h.match(b, d, thr, masks=masks, capacity=CAP)
        assert rc == 0 and h.uses_staged()
        out.append(got)
    h.debug_option(fb.FL_OPT_SIM_ROTATE, 0)
    return out


def _oracle_mass(det, level):
    return np.array([int(det.lm(level, m, lab).astype(np.int64).sum()) for m in range(2) for lab in range(8)], np.int64)


def _check_order(h, det, level, plan):
    """After a default-order match: the sums the kernel read are the oracle's, and CTA 0 visited the phases in the replay's order
    (the rotation of CTA 0, i.e. 0, 1, 2, ..., for the NW = 15 kernel, which has no early exit)."""
    order, mass = h.staged_order()
    want_mass = _oracle_mass(det, level)
    assert np.array_equal(mass[:16], want_mass) and not mass[16:].any(), (mass, want_mass)
    want = np.arange(plan["n_phases"]) if plan["nw_template"] == 15 else E.phase_order(want_mass, plan)
    assert np.array_equal(order, want), (order, want)
    return order


@pytest.fixture(scope="module")
def c2():
    """bench.py's C2 inputs: 8 frames, 8,000 templates (seed 1, 1 % planted on frame 0's quantised images)."""
    frames = [synth.make_frame(W, H, i) for i in range(8)]
    det = F.Detector(T)
    assert det.process(*frames[0]) == 0
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    ts = synth.make_templates(8000, W, H, T, seed=1, quantized=q, planted_fraction=0.01)
    det.set_templates(ts)
    h = fb.Handle(T, (0, 1), W, H, max_candidates=CAP)
    h.upload_templates(ts)
    yield frames, det, ts, h
    h.close()


def test_c2_all_frames_and_thresholds(c2):
    frames, det, ts, h = c2
    plan = fb.plan_staged(W >> 1, H >> 1, T[-1], 2, 8000, 1117, sc.N_SM)
    orders = set()
    for i, (b, d) in enumerate(frames):
        assert det.process(b, d) == 0
        for thr in (60.0, 75.0, 100.0):
            want = det.match(thr, n_threads=8)
            by_mass, rotated = _both(h, b, d, thr)
            assert np.array_equal(by_mass, want), (i, thr, len(by_mass), len(want))
            assert np.array_equal(rotated, want), (i, thr, len(rotated), len(want))
        rc, _ = h.match(b, d, 75.0, capacity=CAP)
        assert rc == 0
        orders.add(tuple(_check_order(h, det, 1, plan)))
    assert len(orders) >= 2                                    # the order does follow the frame


def test_c2_order_is_per_frame_not_cumulative(c2):
    """The sums restart from zero every frame (the kernel's last CTA clears them): the same frame twice gives the same sums."""
    frames, det, ts, h = c2
    b, d = frames[2]
    assert det.process(b, d) == 0
    for _ in range(3):
        assert h.match(b, d, 75.0, capacity=CAP)[0] == 0
        _, mass = h.staged_order()
        assert np.array_equal(mass[:16], _oracle_mass(det, 1))


def test_c2_masked_frame(c2):
    """Masks take the one-kernel-per-stage front end (k_spread_lm): the sums come from the masked linear memories."""
    frames, det, ts, h = c2
    b, d = frames[1]
    rng = np.random.default_rng(5)
    masks = [(rng.random((H, W)) < 0.8).astype(np.uint8) * 255, np.zeros((H, W), np.uint8)]
    masks[1][60:420, 100:560] = 255
    assert det.process(b, d, masks) == 0
    plan = fb.plan_staged(W >> 1, H >> 1, T[-1], 2, 8000, 1117, sc.N_SM)
    for thr in (60.0, 75.0):
        want = det.match(thr, n_threads=8)
        for got in _both(h, b, d, thr, masks=masks):
            assert np.array_equal(got, want), thr
    assert h.match(b, d, 75.0, masks=masks, capacity=CAP)[0] == 0
    _check_order(h, det, 1, plan)
    assert det.process(b, d) == 0                              # back to unmasked on the same handle
    assert np.array_equal(h.match(b, d, 75.0, capacity=CAP)[1], det.match(75.0, n_threads=8))
    _check_order(h, det, 1, plan)


@pytest.mark.parametrize("case", sc.SINGLE_LEVEL, ids=[c.name for c in sc.SINGLE_LEVEL])
def test_every_single_level_plan(case):
    import torch
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    b, d, det, ts, h, t63, peak = plans._single_level(case, n_sm)
    plan = plans._plan_of(case, ts, n_sm)
    assert sc.plan_matches(case, plan)
    for thr in (60.0, 75.0, 100.0):
        want = det.match(thr)
        for got in _both(h, b, d, thr):
            assert np.array_equal(got, want), (case.name, thr)
    assert h.match(b, d, 75.0, capacity=CAP)[0] == 0
    _check_order(h, det, 0, plan)
    h.close()


@pytest.mark.parametrize("case", sc.MULTI_LEVEL, ids=[c.name for c in sc.MULTI_LEVEL])
def test_every_multi_level_plan(case):
    b, d = synth.make_frame(case.W, case.H, 6)
    det = F.Detector(case.T)
    assert det.process(b, d) == 0
    q = [det.quantized(l, m) for l in range(case.L) for m in range(2)]
    ts = synth.make_templates(case.n_templates, case.W, case.H, case.T, n_classes=4, seed=41, quantized=q, planted_fraction=0.1,
                              min_size=case.size, max_size=case.max_size)
    det.set_templates(ts)
    h = fb.Handle(case.T, (0, 1), case.W, case.H, max_candidates=CAP)
    h.upload_templates(ts)
    for thr in (60.0, 75.0, 100.0):
        want = det.match(thr)
        for got in _both(h, b, d, thr):
            assert np.array_equal(got, want), (case.name, thr)
    import torch
    plan = plans._plan_of(case, ts, torch.cuda.get_device_properties(0).multi_processor_count)
    assert h.match(b, d, 75.0, capacity=CAP)[0] == 0
    _check_order(h, det, case.L - 1, plan)
    h.close()


def test_template_sharded_group(c2):
    """The two-member fl_group path (templates dealt over two handles), on two GPUs when there are, else both on GPU 0."""
    import torch
    frames, det, ts, _ = c2
    devices = [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]
    g = fb.Group(devices, exchange_capacity=8192)
    g.upload_templates(ts)
    for i in (0, 3):
        b, d = frames[i]
        assert det.process(b, d) == 0
        want = det.match(75.0, n_threads=8)
        for rot in (0, 1):
            for m in range(2):
                assert g.member_option(m, fb.FL_OPT_SIM_ROTATE, rot) == 0
            rc, got = g.match(b, d, 75.0)
            assert rc == 0 and np.array_equal(got, want), (i, rot)
    g.close()
