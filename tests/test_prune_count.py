"""CPU: the early exit of the staged similarity kernel - its debug option and the count of the work it skips on bench.py's inputs
(tools/exp_prune_count.py)."""
import os
import re
import sys

import fealess_b200 as fb
import staged_cases as sc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import exp_prune_count as E  # noqa: E402


def test_no_prune_option_matches_the_header():
    with open(os.path.join(ROOT, "include", "fealess_b200.h")) as f:
        m = re.search(r"FL_OPT_SIM_NO_PRUNE\s*=\s*(\d+)", f.read())
    assert m and int(m.group(1)) == fb.FL_OPT_SIM_NO_PRUNE == 5


def test_the_stated_c2_plan_is_the_planners():
    p = fb.plan_staged(E.W >> 1, E.H >> 1, E.T[-1], 2, E.N_TEMPLATES, 1117, sc.N_SM)
    assert p is not None and all(p[k] == v for k, v in E.C2_PLAN.items()), p


def test_frame0_count():
    """Frame 0 at threshold 75 with the C2 plan: 258,226 of 496,000 (template, feature) pairs still needed, templates alive after
    each phase, and the busiest warp per CTA going from 123.6 to 84.8 features on average."""
    frames, det, ts = E.setup()
    tmpl = E.Templates(ts, E.C2_PLAN)
    assert max(it[3] for it in tmpl.items) == 1117
    det.process(*frames[0])
    lm = E.linear_memories(det, tmpl.cells)
    r = E.count_frame(lm, tmpl, E.C2_PLAN, 75.0, "tp")
    assert (r["needed"], r["total"]) == (258226, 496000)
    assert r["alive"] == [8000, 8000, 7908, 5755, 2613, 439, 97, 79, 79]
    assert round(r["busiest_warp_full"], 1) == 123.6 and round(r["busiest_warp_pruned"], 1) == 84.8
    assert E.count_frame(lm, tmpl, E.C2_PLAN, 75.0, "words")["needed"] == 258226   # the kernel's word-granular mask loses nothing here
