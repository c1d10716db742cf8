"""GPU (-m gpu): which front-end schedule a frame takes, and what it launches.

A frame's front end is one job list (fe_build in fealess_b200/csrc/frontend.cu), launched as one grid with in-grid waits or cut into
waves.  These tests pin the launches per frame of both schedules over the geometries that choose between them, and the jobs of the C2
single launch, with values measured before the two schedules became one list."""
import numpy as np
import pytest

import fealess_b200 as fb
from fealess_b200 import synth

pytestmark = pytest.mark.gpu


# The front end's launches per frame, and which schedule a frame takes.  Without templates a frame is the front end plus one sort launch:
# one front-end launch for the single launch, L + 1 (more when a wave holds over 16 jobs) per wave.
@pytest.mark.parametrize("T, kinds, W, H, masked, waves, launches", [
    ((5, 8), (0, 1), 640, 480, False, False, 2),
    ((5, 8), (0, 1), 640, 480, True, False, 2),
    ((5, 8), (0, 1), 640, 480, True, True, 4),
    ((4, 8), (0, 1), 640, 480, False, False, 2),
    ((8, 5), (0, 1), 640, 480, False, False, 2),
    ((5, 8), (0, 1), 1280, 720, True, False, 2),
    ((5, 5, 5, 5), (0, 1), 1920, 1080, False, False, 2),
    ((5, 5, 5, 5), (0, 1), 1920, 1080, True, True, 6),
    ((5, 8), (0, 1), 225, 480, False, False, 4),      # a level that does not halve: per wave
    ((5, 8), (0, 1), 225, 480, True, False, 4),
    ((5, 8), (0,), 225, 480, False, False, 4),         # colour only, and still per wave
    ((5,), (1, 1, 1), 640, 480, False, False, 3),      # one level, three depth modalities: per wave
    ((5, 8), (0, 1, 1, 1), 640, 480, False, False, 4),
])
def test_front_end_launches_per_frame(T, kinds, W, H, masked, waves, launches):
    b, d = synth.make_frame(W, H, 0)
    rng = np.random.default_rng(5)
    masks = [(rng.random((H, W)) < 0.7).astype(np.uint8) for _ in kinds] if masked else None
    h = fb.Handle(T, kinds, W, H)
    assert h.debug_option(fb.FL_OPT_FE_WAVES, int(waves)) == 0
    for _ in range(2):
        n0 = h.launch_count()
        assert h.match(b, d, 75.0, masks=masks)[0] == 0
        assert h.launch_count() - n0 == launches
    h.close()


def test_c2_single_launch_jobs_and_the_wave_fallback():
    """bench.py's C2 geometry with 8,000 templates: the single launch's jobs in grid order (six L2 prefetches of the staged kernel's tables,
    pyrDown, depth, colour level 1 and 0, spreads level 1 and 0 of both modalities) with their CTAs, then the launches of a frame per wave,
    of the frame whose in-grid wait times out (its single launch, then the re-run per wave with separate refinement), and after it."""
    W, H, T = 640, 480, (5, 8)
    b, d = synth.make_frame(W, H, 0)
    h = fb.Handle(T, (0, 1), W, H)
    h.upload_templates(synth.make_templates(8000, W, H, T, seed=1))
    assert h.debug_option(fb.FL_OPT_TRACE, 1) == 0

    def launches(**kw):
        n0 = h.launch_count()
        assert h.match(b, d, 75.0, **kw)[0] == 0
        return h.launch_count() - n0

    launches()
    assert launches() == 3
    fe = h.fe_trace()
    assert fe[:, 0].tolist() == [7, 7, 7, 7, 7, 7, 2, 6, 5, 5, 4, 4, 4, 4]
    assert fe[:, 1].tolist() == [63, 3, 4, 1, 1, 1, 300, 600, 150, 600, 150, 150, 384, 384]
    assert h.debug_option(fb.FL_OPT_FE_WAVES, 1) == 0
    assert launches() == 5
    assert h.debug_option(fb.FL_OPT_FE_WAVES, 0) == 0
    assert launches() == 3
    assert h.debug_option(fb.FL_OPT_FE_DEP_TIMEOUT_TEST, 1) == 0
    assert launches() == 9 and h.debug_option(fb.FL_OPT_FE_FORCED_WAVES, 0) == 1
    assert launches() == 5
    h.close()
