"""The geometries on which the GPU tests run the staged similarity kernel, and the plan each one is meant to reach.

fl_plan_staged (fealess_b200/csrc/similarity_staged.cu) picks the kernel's instantiation and its shared-memory layout from the
coarsest-level grid, the smallest template, the template count and the SM count.  tests/test_staged_plan.py checks on the
CPU that the real planner gives every case here the plan it names; tests/test_gpu_similarity_plans.py runs the cases on the
device.  Together the cases must reach every plan choice (``missing_coverage``), so a planner change that moves a case off its
plan fails instead of silently dropping a kernel variant from the suite.
"""
from __future__ import annotations

import dataclasses
from typing import Optional, Tuple

N_SM = 148              # B200 multiprocessors: the SM count the plans below are stated for
N_EDGE_TEMPLATES = 5    # templates test_gpu_similarity_plans.py adds to every single-level case
MAX_STAGED_POSITIONS = 32 * 15 * 8   # NW <= 15 words of 8 cells per lane


@dataclasses.dataclass(frozen=True)
class Case:
    name: str
    T: Tuple[int, ...]      # pyramid steps; the last one is the coarsest level's
    W: int                  # frame size at level 0
    H: int
    size: int               # smallest template (width = height) at level 0, in pixels
    max_size: int           # largest random template at level 0
    n_templates: int        # templates on the handle, edge templates included
    nw: int                 # expected plan: accumulator words per lane ...
    labels_per_phase: int   # ... labels per phase (G) ...
    n_rowblocks: int        # ... row blocks per label ...
    n_buf: Optional[int]    # ... and ring depth (None: not part of what the case is for)

    @property
    def L(self) -> int:
        return len(self.T)

    def coarse(self) -> Tuple[int, int, int]:
        """(W, H, T) of the coarsest level."""
        return self.W >> (self.L - 1), self.H >> (self.L - 1), self.T[-1]

    def max_positions(self) -> int:
        """template_positions (linemod.cpp:1155) of the smallest template at the coarsest level."""
        W, H, T = self.coarse()
        s = self.size >> (self.L - 1)
        return template_positions(W, H, T, s, s)


def template_positions(W: int, H: int, T: int, w: int, h: int) -> int:
    """Positions of a w x h template (coarsest-level pixels) on a W x H level with step T (linemod.cpp:1155)."""
    Wd, Hd = W // T, H // T
    wf, hf = (w - 1) // T + 1, (h - 1) // T + 1
    return min((Hd - hf) * Wd + (Wd - wf) + 1, Wd * Hd)


def tpw(nw: int) -> int:
    return 2 if nw <= 5 else 1


# single-level handles: every template's candidates are the final list
SINGLE_LEVEL = [
    Case("nw3_g4_4buf", (4,), 160, 120, 48, 96, 261, 3, 4, 1, 4),
    Case("nw5_g4_3buf", (4,), 160, 160, 48, 96, 261, 5, 4, 1, 3),
    Case("nw7_g1", (10,), 160, 920, 16, 64, 261, 7, 1, 1, 2),
    Case("nw3_split", (8,), 960, 240, 200, 224, 261, 3, 1, 2, 2),
    Case("nw9_g2", (4,), 440, 160, 96, 128, 261, 9, 2, 1, 2),
    Case("nw11_g2", (4,), 440, 160, 64, 128, 261, 11, 2, 1, 2),
    Case("nw13_g2", (4,), 160, 440, 128, 140, 261, 13, 2, 1, 2),
    Case("nw15_split", (5,), 760, 280, 160, 200, 261, 15, 1, 2, 2),
]

# two-level handles: the candidates go through refinement and the fused sort
MULTI_LEVEL = [
    Case("vga_nw3", (5, 8), 640, 480, 192, 240, 300, 3, 2, 1, None),
    Case("720p_nw9_split", (5, 8), 1280, 720, 288, 336, 300, 9, 1, 2, None),
    Case("720p_nw11_split", (5, 8), 1280, 720, 192, 240, 300, 11, 1, 2, None),
    Case("720p_nw13_split", (5, 8), 1280, 720, 96, 144, 300, 13, 1, 2, None),
]

CASES = SINGLE_LEVEL + MULTI_LEVEL


def plan_matches(case: Case, plan: Optional[dict]) -> bool:
    return (plan is not None and plan["nw_template"] == case.nw and plan["tpw"] == tpw(case.nw) and
            plan["labels_per_phase"] == case.labels_per_phase and plan["n_rowblocks"] == case.n_rowblocks and
            (case.n_buf is None or plan["n_buf"] == case.n_buf))


def missing_coverage(plans) -> set:
    """The plan choices no plan of ``plans`` (dicts of fb.plan_staged, with "n_templates" added) reaches."""
    want = ({("nw", nw) for nw in (3, 5, 7, 9, 11, 13, 15)} | {("tpw", 1), ("tpw", 2)} | {("G", g) for g in (1, 2, 4)} |
            {("rowblocks", "1"), ("rowblocks", ">=2")} | {("n_buf", n) for n in (2, 3, 4)} | {("partial_cta", True)})
    got = set()
    for p in plans:
        got |= {("nw", p["nw_template"]), ("tpw", p["tpw"]), ("G", p["labels_per_phase"]), ("n_buf", p["n_buf"]),
                ("rowblocks", "1" if p["n_rowblocks"] == 1 else ">=2"), ("partial_cta", p["n_templates"] % p["tpc"] != 0)}
    return want - got
