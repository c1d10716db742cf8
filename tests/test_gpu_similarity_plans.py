"""GPU (-m gpu): the staged similarity kernel, position for position, at every plan fl_plan_staged can choose.

The cases are the table of staged_cases.py.  A single-level handle's candidates are the final list, so at a threshold of -300 (a
raw threshold below zero for every template) the list holds every cell of every template's similarity map and is compared record
for record with the C oracle, one class at a time, on the staged kernel and on the baseline kernel of the same handle.  Each case
adds edge templates: features on the last grid column and on the last row of a row block and of a label, a 63-feature template
whose every feature responds 4 at one position, a template whose features all fall into one phase, one with no feature inside
the frame, and one larger than the frame."""
import numpy as np
import pytest

import fealess_b200 as fb
import fl_oracle_py as F
import staged_cases as sc
from fealess_b200 import synth

pytestmark = pytest.mark.gpu

N_CLASSES = 8
CAP = 1 << 19                # -300 on the largest grid: 33 templates x 8,512 cells in one class


@pytest.fixture(scope="module")
def n_sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _canonical(recs):
    """Sort + adjacent unique of Detector::match under the canonical order (helpers.canonical, vectorised)."""
    if len(recs) == 0:
        return recs
    s = recs[np.lexsort((recs["x"], recs["y"], recs["class_idx"], recs["template_id"], -recs["similarity"].astype(np.float64)))]
    keep = np.ones(len(s), bool)
    keep[1:] = ~((s["x"][1:] == s["x"][:-1]) & (s["y"][1:] == s["y"][:-1]) & (s["similarity"][1:] == s["similarity"][:-1]) &
                 (s["class_idx"][1:] == s["class_idx"][:-1]))
    return s[keep]


def _append(ts, templates):
    """ts plus single-level templates [(w, h, [features of modality 0, features of modality 1])], all in the last class."""
    hs, fs, pos = [ts.headers], [ts.features], ts.features.shape[0]
    for w, h, per_mod in templates:
        for f in per_mod:
            f = np.asarray(f, np.int32).reshape(-1, 3)
            hs.append(np.array([[w, h, 0, 0, 0, pos, len(f)]], np.int32))
            fs.append(f)
            pos += len(f)
    n = len(templates)
    return synth.TemplateSet(1, 2, ts.T, ts.class_names, np.concatenate(hs), np.concatenate(fs).astype(np.int32),
                             np.concatenate([ts.class_of, np.full(n, N_CLASSES - 1, np.int32)]),
                             np.concatenate([ts.pose13, np.zeros((n, 13), np.float32)]))


def _edge_templates(case, plan, q, rng):
    """The five edge templates of a single-level case; returns them and the (index, x, y) of the 63-feature template's peak
    relative to the set's start of edge templates."""
    W, H, T = case.W, case.H, case.T[0]
    S, pr, T2 = case.size, plan["phase_rows"], T * T
    out = []
    # (1) features on the last row of a row block, the first row of the next one and the last row of a label, each at the
    # largest x (last grid column: the read runs past the row end) and y (last grid row) the box allows
    pts = []
    for r in sorted({0, T - 1, pr - 1, T2 - 1} | ({pr} if pr < T2 else set())):
        rx, ry = r % T, r // T
        xm, ym = S - (S - rx) % T, S - (S - ry) % T
        pts += [(xm, ym), (xm, ry), (rx, ym)]
    pts += [(S, S), (S, 0), (0, S)]
    feats = [[(x, y, (3 * i + m) % 8) for i, (x, y) in enumerate(pts * 4)][:31] for m in range(2)]
    out.append((S, S, feats))
    # (2) 63 features (32 + 31) cut out of the quantised images at a grid-aligned origin: every one responds 4 there
    S2 = max(S, 64)
    for _ in range(1000):
        c = int(rng.integers(0, (W - S2 - 1) // T + 1))
        r = int(rng.integers(0, (H - S2 - 1) // T + 1))
        subs = [qm[r * T:r * T + S2 + 1, c * T:c * T + S2 + 1] for qm in q]
        if all(np.count_nonzero(sub) >= 32 for sub in subs):
            break
    else:
        raise AssertionError("no window with 32 oriented pixels per modality")
    feats = []
    for m, n in ((0, 32), (1, 31)):
        ys, xs = np.nonzero(subs[m])
        sel = rng.choice(len(ys), n, replace=False)
        feats.append(np.stack([xs[sel], ys[sel], np.log2(subs[m][ys[sel], xs[sel]]).astype(np.int32)], 1))
    out.append((S2, S2, feats))
    peak = (c, r)
    # (3) 32 features of one label on rows of the first row block: one phase
    xs = [T - 1 + T * i for i in range(S2 // T) if T - 1 + T * i <= S2]
    ys = [T * j for j in range(S2 // T + 1) if T * j <= S2]
    one = [(x, y, 5) for y in ys for x in xs][:32]
    assert len(one) == 32
    out.append((S2, S2, [one, []]))
    # (4) wider than the frame, every feature right of it: no feature inside the frame, but positions
    w4 = W + T
    out.append((w4, S, [[(W + int(rng.integers(0, T + 1)), int(rng.integers(0, S + 1)), int(rng.integers(0, 8))) for _ in range(31)]
                        for _ in range(2)]))
    # (5) larger than the frame: no position at all
    w5, h5 = W + 2 * T, H + 2 * T
    out.append((w5, h5, [[(int(rng.integers(0, w5 + 1)), int(rng.integers(0, h5 + 1)), int(rng.integers(0, 8))) for _ in range(31)]
                         for _ in range(2)]))
    assert len(out) == sc.N_EDGE_TEMPLATES
    return out, peak


def _max_positions(ts, W, H, T):
    """api.cu max_positions: the largest template_positions over the coarsest-level boxes."""
    L, M = ts.n_levels, ts.n_modalities
    hd = ts.headers[(L - 1) * M::L * M]
    return max(sc.template_positions(W, H, T, int(w), int(h)) for w, h in hd[:, :2])


def _single_level(case, n_sm):
    W, H, T = case.W, case.H, case.T[0]
    b, d = synth.make_frame(W, H, 5)
    det = F.Detector(case.T)
    assert det.process(b, d) == 0
    q = [det.quantized(0, m) for m in range(2)]
    want_plan = fb.plan_staged(W, H, T, 2, case.n_templates, case.max_positions(), sc.N_SM)
    rng = np.random.default_rng(sc.SINGLE_LEVEL.index(case))
    ts = synth.make_templates(case.n_templates - sc.N_EDGE_TEMPLATES, W, H, case.T, n_classes=N_CLASSES, seed=31, quantized=q,
                              planted_fraction=0.1, features_per_level=(31,), min_size=case.size, max_size=case.max_size)
    edge, peak = _edge_templates(case, want_plan, q, rng)
    ts = _append(ts, edge)
    assert ts.n_templates == case.n_templates
    assert _max_positions(ts, W, H, T) == case.max_positions()
    det.set_templates(ts)
    t63 = case.n_templates - sc.N_EDGE_TEMPLATES + 1
    assert det.similarity(t63)[peak[1], peak[0]] == 252          # the byte total of the 63-feature template reaches 63 x 4
    h = fb.Handle(case.T, (0, 1), W, H, max_candidates=CAP)
    h.upload_templates(ts)
    return b, d, det, ts, h, t63, peak


def _plan_of(case, ts, n_sm):
    W, H, T = case.coarse()
    p = fb.plan_staged(W, H, T, 2, ts.n_templates, _max_positions(ts, W, H, T), n_sm)
    assert p is not None
    p["n_templates"] = ts.n_templates
    return p


@pytest.mark.parametrize("case", sc.SINGLE_LEVEL, ids=[c.name for c in sc.SINGLE_LEVEL])
def test_single_level_exhaustive(case, n_sm):
    b, d, det, ts, h, t63, peak = _single_level(case, n_sm)
    p = _plan_of(case, ts, n_sm)
    assert sc.plan_matches(case, p), p
    for baseline in (False, True):
        h.force_baseline(baseline)
        for c in range(N_CLASSES):
            want = det.match(-300.0, class_filter=[c])
            rc, got = h.match(b, d, -300.0, class_filter=[c], capacity=CAP)
            assert rc == 0 and h.uses_staged() == (not baseline)
            assert len(got) == len(want) and np.array_equal(got, want), (case.name, "baseline" if baseline else "staged", c)
        rc, got = h.match(b, d, 60.0, capacity=CAP)
        assert rc == 0 and np.array_equal(got, det.match(60.0))
    h.force_baseline(False)
    # the 63-feature template scores 100 % at its planted position
    rc, got = h.match(b, d, 99.0, class_filter=[N_CLASSES - 1], capacity=CAP)
    T = case.T[0]
    off = T // 2 + (T % 2 - 1)
    tid = t63 - int(np.flatnonzero(ts.class_of == N_CLASSES - 1)[0])
    hit = got[(got["template_id"] == tid) & (got["x"] == peak[0] * T + off) & (got["y"] == peak[1] * T + off)]
    assert rc == 0 and len(hit) == 1 and hit["similarity"][0] == np.float32(100.5)
    h.close()


def test_single_level_caller_template_ids(n_sm):
    """fl_set_template_ids on a single-level handle: the candidates carry the caller's ids, on both kernels."""
    case = sc.SINGLE_LEVEL[0]
    b, d, det, ts, h, _, _ = _single_level(case, n_sm)
    n = ts.n_templates
    ids = (np.random.default_rng(3).permutation(n) + 1000).astype(np.int32)
    h.set_template_ids(ids)
    first = np.array([np.flatnonzero(ts.class_of == c)[0] for c in range(N_CLASSES)])
    for thr, filt in ((60.0, None), (-300.0, [2])):
        raw = det.match(thr, class_filter=filt, canonical=False)
        assert np.array_equal(_canonical(raw), det.match(thr, class_filter=filt))
        raw["template_id"] = ids[first[raw["class_idx"]] + raw["template_id"]]
        want = _canonical(raw)
        for baseline in (False, True):
            h.force_baseline(baseline)
            rc, got = h.match(b, d, thr, class_filter=filt, capacity=CAP)
            assert rc == 0 and h.uses_staged() == (not baseline)
            assert np.array_equal(got, want), (thr, baseline)
    h.close()


@pytest.mark.parametrize("case", sc.MULTI_LEVEL, ids=[c.name for c in sc.MULTI_LEVEL])
def test_multi_level(case, n_sm):
    W, H = case.W, case.H
    b, d = synth.make_frame(W, H, 6)
    det = F.Detector(case.T)
    assert det.process(b, d) == 0
    q = [det.quantized(l, m) for l in range(case.L) for m in range(2)]
    ts = synth.make_templates(case.n_templates, W, H, case.T, n_classes=4, seed=41, quantized=q, planted_fraction=0.1,
                              min_size=case.size, max_size=case.max_size)
    det.set_templates(ts)
    p = _plan_of(case, ts, n_sm)
    assert sc.plan_matches(case, p), p
    h = fb.Handle(case.T, (0, 1), W, H, max_candidates=CAP)
    h.upload_templates(ts)
    for thr in (75.0, 50.0):
        want = det.match(thr)
        rc, got = h.match(b, d, thr, capacity=CAP)
        assert rc == 0 and h.uses_staged() and np.array_equal(got, want), thr
    assert len(want) > 0
    h.close()


def test_grid_above_the_staged_limit_runs_the_baseline_kernel(n_sm):
    W, H, T = 640, 480, (8,)
    b, d = synth.make_frame(W, H, 2)
    det = F.Detector(T)
    assert det.process(b, d) == 0
    q = [det.quantized(0, m) for m in range(2)]
    ts = synth.make_templates(256, W, H, T, n_classes=N_CLASSES, seed=51, quantized=q, planted_fraction=0.1,
                              features_per_level=(31,), min_size=48, max_size=96)
    assert _max_positions(ts, W, H, 8) > sc.MAX_STAGED_POSITIONS
    assert fb.plan_staged(W, H, 8, 2, 256, _max_positions(ts, W, H, 8), n_sm) is None
    det.set_templates(ts)
    h = fb.Handle(T, (0, 1), W, H, max_candidates=CAP)
    h.upload_templates(ts)
    for c in (0, 5):
        rc, got = h.match(b, d, -300.0, class_filter=[c], capacity=CAP)
        assert rc == 0 and not h.uses_staged() and np.array_equal(got, det.match(-300.0, class_filter=[c]))
    h.close()


def test_the_cases_cover_every_plan_choice(n_sm):
    """The plans the cases run on this device reach every NW, templates per warp, labels per phase, row-block count, ring depth
    and a partial last CTA: a planner change that moves a case off its plan fails here instead of dropping coverage."""
    plans = []
    for case in sc.CASES:
        W, H, T = case.coarse()
        p = fb.plan_staged(W, H, T, 2, case.n_templates, case.max_positions(), n_sm)
        assert sc.plan_matches(case, p), (case.name, p)
        p["n_templates"] = case.n_templates
        plans.append(p)
    assert sc.missing_coverage(plans) == set()
