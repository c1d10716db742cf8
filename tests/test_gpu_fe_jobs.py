"""GPU (-m gpu): the spread job's instantiations and the front end's per-job SM time.

k_front_end_wave compiles the spread + linear-memory job for T = 5 below the coarsest level and T = 8 at it; every other
(T, level) takes the runtime-T code.  Each pyramid below sends every spread job of a level through one of the three, with and
without the coarsest level's nibble linear memories and response sums, and must stay bit-exact with the C oracle."""
import numpy as np
import pytest

import fealess_b200 as fb
import fl_oracle_py as F
from fealess_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("T", [(4, 8), (8, 5), (4, 4), (8, 8)])
def test_spread_paths_bit_exact(T):
    W, H = 640, 480
    b, d = synth.make_frame(W, H, 2)
    det = F.Detector(T)
    assert det.process(b, d) == 0
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    ts = synth.make_templates(300, W, H, T, n_classes=3, seed=9, quantized=q, planted_fraction=0.05)
    det.set_templates(ts)
    h = fb.Handle(T, (0, 1), W, H)
    h.upload_templates(ts)
    h.keep_spread(True)
    rc, got = h.match(b, d, 70.0)
    assert rc == 0
    for l in range(2):
        for m in range(2):
            assert np.array_equal(h.debug_quantized(l, m, W, H, spread=True), det.spread(l, m)), "spread L%d M%d" % (l, m)
            for lab in range(8):
                assert np.array_equal(h.debug_lm(l, m, lab, W, H), det.lm(l, m, lab)), "LM L%d M%d label %d" % (l, m, lab)
    want = det.match(70.0)
    assert len(want) > 0 and np.array_equal(got, want)
    h.close()


def test_fe_trace_sums_each_jobs_cta_spans():
    """FL_DBG_FE_TRACE columns 4 and 5: the summed CTA spans of a job, in SM cycles and in ns.  No CTA outlives its job's
    first-start-to-last-end window, so a job's sum is at most CTAs x that window."""
    W, H, T = 640, 480, (5, 8)
    b, d = synth.make_frame(W, H, 0)
    h = fb.Handle(T, (0, 1), W, H)
    assert h.debug_option(fb.FL_OPT_TRACE, 1) == 0
    h.upload_templates(synth.make_templates(200, W, H, T, seed=3))
    for _ in range(3):
        assert h.match(b, d, 75.0)[0] == 0
    fe = h.fe_trace()
    assert fe.shape[1] == 6 and len(fe) >= 4
    kind, ctas, start, end, cycles, ns = fe.T
    assert (ctas > 0).all() and (end >= start).all()
    assert (ns > 0).all() and (cycles > 0).all()
    assert (ns <= ctas * (end - start)).all()
    ghz = cycles.sum() / ns.sum()
    assert 0.3 < ghz < 3.5, ghz                          # the SM clock the CTAs ran at
    h.close()
