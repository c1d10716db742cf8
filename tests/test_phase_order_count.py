"""CPU: the staged similarity kernel's phase order by response mass - its debug option and the CPU replay of the early exit under
that order on bench.py's inputs (tools/exp_prune_count.py)."""
import os
import re
import sys

import numpy as np

import fealess_b200 as fb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import exp_prune_count as E  # noqa: E402


def test_rotate_option_and_order_getter_match_the_header():
    with open(os.path.join(ROOT, "include", "fealess_b200.h")) as f:
        src = f.read()
    m = re.search(r"FL_OPT_SIM_ROTATE\s*=\s*(\d+)", src)
    assert m and int(m.group(1)) == fb.FL_OPT_SIM_ROTATE == 6
    m = re.search(r"FL_DBG_STAGED_ORDER\s*=\s*(\d+)", src)
    assert m and int(m.group(1)) == fb.FL_DBG_STAGED_ORDER == 7


def test_phase_order_rule():
    """Groups of labels by ascending summed mass, ties by index, row blocks of a group in order."""
    plan = {"n_phases": 8, "n_rowblocks": 1, "labels_per_phase": 2}
    mass = np.array([5, 5, 1, 1, 9, 0, 2, 2, 3, 3, 0, 0, 7, 7, 4, 4])
    assert E.phase_order(mass, plan).tolist() == [5, 1, 3, 4, 7, 2, 0, 6]
    plan = {"n_phases": 48, "n_rowblocks": 3, "labels_per_phase": 1}
    mass = np.array([3] * 16)
    assert E.phase_order(mass, plan).tolist() == list(range(48))
    mass[7] = 0
    assert E.phase_order(mass, plan).tolist()[:4] == [21, 22, 23, 0]


def test_frame0_count_by_mass():
    """Frame 0 at threshold 75 with the C2 plan, phases by response mass (3 2 1 0 4 7 5 6): 221,582 of 496,000 (template, feature)
    pairs still needed (55.3 % skipped, against 47.9 % in the rotated order), and the busiest warp per CTA at 74.1 features on
    average (84.8 rotated)."""
    frames, det, ts = E.setup()
    tmpl = E.Templates(ts, E.C2_PLAN)
    det.process(*frames[0])
    lm = E.linear_memories(det, tmpl.cells)
    assert E.phase_order(E.label_mass(lm, tmpl.cells), E.C2_PLAN).tolist() == [3, 2, 1, 0, 4, 7, 5, 6]
    r = E.count_frame(lm, tmpl, E.C2_PLAN, 75.0, "tp", "mass")
    assert (r["needed"], r["total"]) == (221582, 496000)
    assert r["alive"] == [8000, 8000, 7914, 3637, 113, 79, 79, 79, 79]
    assert round(r["busiest_warp_pruned"], 1) == 74.1
