"""CPU: the staged similarity kernel's planner (fl_debug_plan_staged, host code only).

Every case of staged_cases.py gets the plan it names at 148 SMs, the cases together reach every plan choice, the planner refuses
what the kernel cannot run, and every plan it returns keeps the conditions the kernel's shared-memory layout and its reads rely on."""
import os
import re

import pytest

import fealess_b200 as fb
import staged_cases as sc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FL_LM_PAD = int(re.search(r"#define FL_LM_PAD (\d+)", open(os.path.join(ROOT, "fealess_b200", "csrc", "fl_internal.cuh")).read()).group(1))
SMEM_LIMIT = 227 * 1024 - 512


def _plan(case, n_sm=sc.N_SM):
    W, H, T = case.coarse()
    p = fb.plan_staged(W, H, T, 2, case.n_templates, case.max_positions(), n_sm)
    if p is not None:
        p["n_templates"] = case.n_templates
    return p


@pytest.mark.parametrize("case", sc.CASES, ids=[c.name for c in sc.CASES])
def test_every_case_gets_the_plan_it_names(case):
    p = _plan(case)
    assert sc.plan_matches(case, p), (case, p)


def test_the_cases_cover_every_plan_choice():
    assert sc.missing_coverage([_plan(c) for c in sc.CASES]) == set()


def test_planner_refusals():
    assert fb.plan_staged(160, 120, 4, 2, 256, 700, 148) is not None
    assert fb.plan_staged(164, 120, 4, 2, 256, 700, 148) is None           # Wd = 41: no 4-bit linear memories
    assert fb.plan_staged(640, 480, 8, 2, 256, sc.MAX_STAGED_POSITIONS, 148) is not None
    assert fb.plan_staged(640, 480, 8, 2, 256, sc.MAX_STAGED_POSITIONS + 1, 148) is None
    assert fb.plan_staged(640, 480, 8, 2, 256, 4800, 148) is None
    assert fb.plan_staged(640, 480, 8, 2, 256, 1 << 30, 148) is None        # clamped to the 4,800 cells: still too many
    for n in (0, -1):
        assert fb.plan_staged(160, 120, 4, 2, n, 700, 148) is None
    for mp in (0, -5):
        assert fb.plan_staged(160, 120, 4, 2, 256, mp, 148) is None


@pytest.mark.parametrize("args", [(161, 120, 4), (160, 122, 4), (160, 120, 0), (160, 120, 17), (2, 120, 4), (160, 2, 4)])
def test_bad_geometry_is_an_argument_error(args):
    with pytest.raises(fb.FealessError) as e:
        fb.plan_staged(*args, 2, 256, 100, 148)
    assert e.value.rc == fb.FL_ERR_ARG


def test_bad_counts_are_argument_errors():
    for M, n_sm in ((0, 148), (5, 148), (2, 0), (2, -1)):
        with pytest.raises(fb.FealessError) as e:
            fb.plan_staged(160, 120, 4, M, 256, 100, n_sm)
        assert e.value.rc == fb.FL_ERR_ARG


def _check_invariants(p, W, H, T, M, n, mp, n_sm):
    Wd, Hd = W // T, H // T
    cells, T2 = Wd * Hd, T * T
    nw, G, pr, nrb = p["nw_template"], p["labels_per_phase"], p["phase_rows"], p["n_rowblocks"]
    label_stride = (T2 * cells + FL_LM_PAD + 31) & ~31                   # level_lm_bytes in api.cu
    assert nw in (3, 5, 7, 9, 11, 13, 15) and p["tpw"] == sc.tpw(nw)
    assert 256 * nw >= min(mp, cells)                                   # 32 lanes x NW words x 8 cells cover every position
    assert p["halo_bytes"] >= 4 * (32 * nw + 1)                          # a lane's window runs over 32 NW + 1 words past its first cell
    assert p["halo_bytes"] + 16 <= FL_LM_PAD // 2                        # ... and stays inside the zero pad behind a label
    assert p["smem_bytes"] <= SMEM_LIMIT
    assert p["n_buf"] in (2, 3, 4) or p["n_buf"] == p["n_phases"]
    assert p["n_buf"] <= p["n_phases"] <= 254
    assert p["n_buf"] * p["buf_bytes"] <= p["smem_bytes"] and p["buf_bytes"] % 128 == 0
    assert p["tpc"] <= 31 * p["tpw"] and p["n_cta"] * p["tpc"] >= n and (p["n_cta"] - 1) * p["tpc"] < n
    warps = -(-p["tpc"] // p["tpw"])
    assert p["block_threads"] == 32 * (warps + 1) <= 1024
    assert G in (1, 2, 4) and (G == 1 or nrb == 1)
    assert 1 <= pr <= T2 and nrb == -(-T2 // pr) and p["n_phases"] == M * (8 // G) * nrb
    assert nrb == 1 or (pr * cells) % 32 == 0                            # a row block starts 16-byte aligned in the 4-bit copy
    for rb in range(nrb):                                                # every bulk copy fits its buffer
        rows = min(pr, T2 - rb * pr)
        assert (((((G - 1) * label_stride + rows * cells) >> 1) + p["halo_bytes"] + 15) & ~15) <= p["buf_bytes"]


@pytest.mark.parametrize("W,H,T", [(160, 120, 4), (160, 920, 10), (960, 240, 8), (440, 160, 4), (760, 280, 5), (640, 360, 8)])
def test_every_plan_keeps_the_kernel_invariants(W, H, T):
    cells = (W // T) * (H // T)
    M = 2
    planned = 0
    for n in (256, 257, 1000, 8000, 32000):
        for n_sm in (148, 132, 1):
            for mp in range(1, cells + 1):
                p = fb.plan_staged(W, H, T, M, n, mp, n_sm)
                if mp > sc.MAX_STAGED_POSITIONS:
                    assert p is None, (n, n_sm, mp)
                    continue
                if p is None:
                    continue
                planned += 1
                _check_invariants(p, W, H, T, M, n, mp, n_sm)
    assert planned > 0
