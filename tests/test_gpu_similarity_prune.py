"""GPU (-m gpu): the staged similarity kernel's early exit (a template is dropped once no position can reach the threshold) changes
no result.

Every case compares the whole match list with the C oracle record for record, once with the early exit (the default) and once
with FL_OPT_SIM_NO_PRUNE on the same handle.  The exhaustive plan tests run at a threshold of -300, where the bound never bites, so
the plans are run again here at thresholds where it does."""
import numpy as np
import pytest

import fealess_b200 as fb
import fl_oracle_py as F
import staged_cases as sc
import test_gpu_similarity_plans as plans
from fealess_b200 import synth

pytestmark = pytest.mark.gpu

W, H, T = 640, 480, (5, 8)
CAP = 1 << 19


def _both(h, b, d, thr, class_filter=None, capacity=CAP):
    """The match list with the early exit and without it (FL_OPT_SIM_NO_PRUNE), from one handle."""
    out = []
    for off in (0, 1):
        assert h.debug_option(fb.FL_OPT_SIM_NO_PRUNE, off) == 0
        rc, got = h.match(b, d, thr, class_filter=class_filter, capacity=capacity)
        assert rc == 0
        out.append(got)
    h.debug_option(fb.FL_OPT_SIM_NO_PRUNE, 0)
    return out


def _raw_threshold(nf, thr):
    """The kernel's raw threshold int(2 nf + (thr / 100) 2 nf + 0.5) in fp32 (linemod.cpp:1487)."""
    f = np.float32
    return int(f(f(f(2 * nf) + f(f(f(thr) / f(100.0)) * f(2 * nf))) + f(0.5)))


def _threshold_for(nf, raw):
    """A threshold (fp32-exact) whose raw threshold for nf features is ``raw``."""
    for thr in np.arange(-100.0, 200.0, 0.01, dtype=np.float64):
        t = float(np.float32(thr))
        if _raw_threshold(nf, t) == raw:
            return t
    raise AssertionError("no threshold gives raw %d for %d features" % (raw, nf))


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
    n_nonempty = 0
    for i, (b, d) in enumerate(frames):
        assert det.process(b, d) == 0
        for thr in (60.0, 75.0, 90.0, 100.0):
            want = det.match(thr, n_threads=8)
            pruned, full = _both(h, b, d, thr)
            assert h.uses_staged()
            assert np.array_equal(pruned, want), (i, thr, len(pruned), len(want))
            assert np.array_equal(full, want), (i, thr, len(full), len(want))
            n_nonempty += len(want) > 0
    assert n_nonempty >= 8


def test_c2_disabled_classes_and_dead_ctas(c2):
    """A class filter disables most templates (whole CTAs have no live slot from the start, so their producer stops at once); at a
    threshold of 100 nearly every template is dropped after its first phase (whole CTAs die and stop streaming)."""
    frames, det, ts, h = c2
    b, d = frames[0]
    assert det.process(b, d) == 0
    ncls = int(ts.class_of.max()) + 1
    filters = [None] if ncls == 1 else [[0], [ncls - 1]]
    for thr in (75.0, 100.0):
        for cf in filters:
            want = det.match(thr, class_filter=cf, n_threads=8)
            for got in _both(h, b, d, thr, class_filter=cf):
                assert np.array_equal(got, want), (thr, cf)


def test_c2_single_class_disabled():
    """Two classes, one disabled by the class filter: the disabled class's slots are dead from the prologue on."""
    frames = [synth.make_frame(W, H, i) for i in range(2)]
    det = F.Detector(T)
    assert det.process(*frames[0]) == 0
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    ts = synth.make_templates(2000, W, H, T, n_classes=2, seed=3, quantized=q, planted_fraction=0.05)
    det.set_templates(ts)
    h = fb.Handle(T, (0, 1), W, H, max_candidates=CAP)
    h.upload_templates(ts)
    for b, d in frames:
        assert det.process(b, d) == 0
        for cf in ([0], [1], None):
            want = det.match(80.0, class_filter=cf, n_threads=8)
            for got in _both(h, b, d, 80.0, class_filter=cf):
                assert h.uses_staged() and np.array_equal(got, want), cf
    h.close()


@pytest.mark.parametrize("case", sc.SINGLE_LEVEL, ids=[c.name for c in sc.SINGLE_LEVEL])
def test_every_single_level_plan(case):
    import torch
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    b, d, det, ts, h, t63, peak = plans._single_level(case, n_sm)
    assert sc.plan_matches(case, plans._plan_of(case, ts, n_sm))
    for thr in (50.0, 75.0, 90.0, 99.0):
        want = det.match(thr)
        for got in _both(h, b, d, thr):
            assert h.uses_staged() and np.array_equal(got, want), (case.name, thr)
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
    for thr in (60.0, 75.0, 90.0):
        want = det.match(thr)
        for got in _both(h, b, d, thr):
            assert h.uses_staged() and np.array_equal(got, want), (case.name, thr)
    h.close()


@pytest.mark.parametrize("case", [sc.SINGLE_LEVEL[0], sc.SINGLE_LEVEL[4]], ids=["nw3", "nw9"])
def test_boundary_scores(case):
    """Planted templates whose best total is exactly raw_thr + 1 (reported) or exactly raw_thr (not reported).  For the 63-feature
    template whose every feature responds 4 at one position, a best total of raw_thr + 1 puts its partial sum there exactly on the
    bound after every phase (partial + 4 x features left = raw_thr + 1): it must survive every test."""
    import torch
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    b, d, det, ts, h, t63, peak = plans._single_level(case, n_sm)
    nf_of = ts.headers.reshape(ts.n_templates, ts.n_modalities, 7)[:, :, 6].sum(1)
    first = {c: int(np.flatnonzero(ts.class_of == c)[0]) for c in np.unique(ts.class_of)}
    planted = [t for t in range(ts.n_templates - sc.N_EDGE_TEMPLATES) if det.similarity(t).max() >= 2.6 * nf_of[t]][:3]
    assert len(planted) >= 1
    for t in [t63] + planted:
        best = int(det.similarity(t).max())
        cls = int(ts.class_of[t])
        for raw, reported in ((best - 1, True), (best, False)):
            thr = _threshold_for(int(nf_of[t]), raw)
            raw_list = det.match(thr, class_filter=[cls], canonical=False)   # (before the unique step, which may merge records)
            assert bool(np.any(raw_list["template_id"] == t - first[cls])) == reported, (t, raw, best)
            want = det.match(thr, class_filter=[cls])
            for got in _both(h, b, d, thr, class_filter=[cls]):
                assert np.array_equal(got, want), (case.name, t, raw)
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
        for off in (0, 1):
            for m in range(2):
                assert g.member_option(m, fb.FL_OPT_SIM_NO_PRUNE, off) == 0
            rc, got = g.match(b, d, 75.0)
            assert rc == 0 and np.array_equal(got, want), (i, off)
    g.close()
