"""Developer count (CPU): how much of k_similarity_staged's feature work the early exit skips on bench.py's C2 inputs.

The staged kernel drops a template slot after a phase when, at every position p it tests, partial(p) + 4 x (features left) <=
raw_thr: no candidate is possible any more (a response is at most 4).  This script replays that rule with the C oracle's linear
memories, on bench.py's frames and 8,000-template set (seed 1, 1 % planted on frame 0), in the kernel's phase order (templates
per CTA, slot -> warp).  Two phase orders (--order, count_frame's visit): "rotation" (CTA b starts at phase 7 b mod phases, what the kernel does without the early
exit or with FL_OPT_SIM_ROTATE) and "mass" (the kernel's default: label groups by ascending response sum of the frame, ties by index,
the same in every CTA; see phase_order).  The plan comes from fl_debug_plan_staged for the SM count of GPU 0 when
a GPU is present, else it is the C2 plan on a 148-SM B200 stated below.

Columns per frame: the share of (template, feature) pairs skipped; templates alive before the first phase and after each phase;
features of the busiest warp of a CTA (mean over CTAs) without and with the exit.  Three position sets for the test:
  tp     positions [0, template_positions) - the cells a candidate can come from;
  words  [0, 8 ceil(template_positions / 8)) - what the kernel tests (whole 32-bit accumulator words);
  grid   every cell of the grid - a test without any mask (cells past template_positions hold sums of real data).
Usage: python tools/exp_prune_count.py [--frames 8] [--threshold 75] [--order rotation|mass]"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np

W, H, T, N_TEMPLATES = 640, 480, (5, 8), 8000
# fl_debug_plan_staged(320, 240, 8, 2, 8000, 1117, 148): 146 CTAs of 55 templates, 28 consumer warps x 2 slots, 8 phases of 2 labels
C2_PLAN = {"tpc": 55, "tpw": 2, "block_threads": 29 * 32, "labels_per_phase": 2, "n_rowblocks": 1, "phase_rows": 64, "n_phases": 8}
MASKS = ("tp", "words", "grid")


def plan_for(max_positions):
    try:
        import torch
        if torch.cuda.is_available():
            import fealess_b200 as fb
            n_sm = torch.cuda.get_device_properties(0).multi_processor_count
            p = fb.plan_staged(W >> 1, H >> 1, T[-1], 2, N_TEMPLATES, max_positions, n_sm)
            if p is not None:
                return p, "fl_debug_plan_staged, %d SMs" % n_sm
    except ImportError:
        pass
    return dict(C2_PLAN), "the C2 plan of a 148-SM B200 (no GPU here)"


def raw_threshold(nf, thr):
    f = np.float32
    return int(f(f(f(2 * nf) + f(f(f(thr) / f(100.0)) * f(2 * nf))) + f(0.5)))


class Templates:
    """Per template: its coarsest-level features (phase, flat index into the level's linear memories), raw feature count, box."""

    def __init__(self, ts, plan):
        Tc, Wd, Hd = T[-1], (W >> 1) // T[-1], (H >> 1) // T[-1]
        self.cells, self.Wd, self.Hd = Wd * Hd, Wd, Hd
        L, M = ts.n_levels, ts.n_modalities
        hdr = ts.headers.reshape(ts.n_templates, L, M, 7)[:, L - 1]
        self.items = []
        for t in range(ts.n_templates):
            ph, base, nf = [], [], 0
            for m in range(M):
                _, _, _, _, _, pos, n = hdr[t, m]
                nf += int(n)
                for x, y, lab in ts.features[pos:pos + n]:
                    if x < 0 or y < 0 or x >= W >> 1 or y >= H >> 1:
                        continue
                    row = (y % Tc) * Tc + x % Tc
                    ph.append(((m * 8 + lab) // plan["labels_per_phase"]) * plan["n_rowblocks"] + row // plan["phase_rows"])
                    base.append(((m * 8 + lab) * Tc * Tc + row) * self.cells + (y // Tc) * Wd + x // Tc)
            wf, hf = (int(hdr[t, 0, 0]) - 1) // Tc + 1, (int(hdr[t, 0, 1]) - 1) // Tc + 1
            tp = min((Hd - hf) * Wd + (Wd - wf) + 1, self.cells)
            self.items.append((np.array(ph, np.int64), np.array(base, np.int64), nf, tp))


def label_mass(lm_flat, cells, n_modalities=2):
    """The response sum of every (modality, label) of the coarsest level: what the front end's spread jobs add up on the device."""
    n = T[-1] * T[-1] * cells
    return np.array([int(lm_flat[i * n:(i + 1) * n].astype(np.int64).sum()) for i in range(8 * n_modalities)], np.int64)


def phase_order(mass, plan):
    """The kernel's visit order by response mass: order[q] = the phase visited at step q.  A group of labels_per_phase labels
    weighs the sum of their masses; groups ascending by weight, ties by index; the row blocks of a group keep their order."""
    nrb, lpp = plan["n_rowblocks"], plan["labels_per_phase"]
    n_groups = plan["n_phases"] // nrb
    w = np.array([int(mass[g * lpp:(g + 1) * lpp].sum()) for g in range(n_groups)], np.int64)
    groups = np.argsort(w, kind="stable")
    return np.array([g * nrb + rb for g in groups for rb in range(nrb)], np.int64)


def count_frame(lm_flat, tmpl, plan, thr, mask, visit="rotation"):
    """lm_flat: the coarsest level's linear memories of all (modality, label, row) laid out flat, zero pad behind."""
    nph, tpc = plan["n_phases"], plan["tpc"]
    if visit == "mass":
        step_of = np.argsort(phase_order(label_mass(lm_flat, tmpl.cells), plan))   # step_of[phase] = visit step
    ncw = plan["block_threads"] // 32 - 1
    n_cta = (len(tmpl.items) + tpc - 1) // tpc
    alive = np.zeros(nph + 1, np.int64)
    total = done = 0
    warp_full = np.zeros((n_cta, ncw), np.int64)
    warp_pr = np.zeros((n_cta, ncw), np.int64)
    for t, (ph, base, nf, tp) in enumerate(tmpl.items):
        b, slot = divmod(t, tpc)
        warp = slot % ncw
        n = len(ph)
        total += n
        warp_full[b, warp] += n
        alive[0] += 1
        if n == 0 or tp <= 0:
            alive[1:] += 1
            continue
        P = {"tp": tp, "words": min(8 * ((tp + 7) // 8), tmpl.cells), "grid": tmpl.cells}[mask]
        key = (ph - (b * 7) % nph) % nph if visit == "rotation" else step_of[ph]   # the step at which this CTA visits each feature's phase
        order = np.argsort(key, kind="stable")
        A = lm_flat[base[order][:, None] + np.arange(P)[None, :]].astype(np.int32)
        cs = np.cumsum(A, axis=0)
        acc_after = np.searchsorted(key[order], np.arange(nph), side="right")   # features accumulated after visiting k + 1 phases
        rt = raw_threshold(nf, thr)
        used = n
        for k in range(nph):
            a = int(acc_after[k])
            best = int(cs[a - 1].max()) if a > 0 else 0
            if best + 4 * (n - a) <= rt:
                used = a
                break
            alive[k + 1] += 1
        done += used
        warp_pr[b, warp] += used
    return {"skipped": 1.0 - done / total, "needed": done, "total": total, "alive": alive.tolist(),
            "busiest_warp_full": float(warp_full.max(1).mean()), "busiest_warp_pruned": float(warp_pr.max(1).mean())}


def setup():
    import fl_oracle_py as F
    from fealess_b200 import synth
    frames = [synth.make_frame(W, H, i) for i in range(8)]
    det = F.Detector(T)
    det.process(*frames[0])
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    ts = synth.make_templates(N_TEMPLATES, W, H, T, seed=1, quantized=q, planted_fraction=0.01)
    return frames, det, ts


def linear_memories(det, cells):
    Tc = T[-1]
    lm = np.zeros(2 * 8 * Tc * Tc * cells + 8192, np.uint8)
    for m in range(2):
        for lab in range(8):
            o = (m * 8 + lab) * Tc * Tc * cells
            lm[o:o + Tc * Tc * cells] = det.lm(1, m, lab).reshape(-1)
    return lm


def run(n_frames=8, thr=75.0, masks=MASKS, out=sys.stdout, order="rotation"):
    frames, det, ts = setup()
    Tc = T[-1]
    Wd, Hd = (W >> 1) // Tc, (H >> 1) // Tc
    hd = ts.headers.reshape(ts.n_templates, 2, 2, 7)[:, 1, 0]
    max_pos = max(min((Hd - ((int(h) - 1) // Tc + 1)) * Wd + (Wd - ((int(w) - 1) // Tc + 1)) + 1, Wd * Hd) for w, h in hd[:, :2])
    plan, src = plan_for(max_pos)
    tmpl = Templates(ts, plan)
    out.write("plan (%s): %d templates per CTA, %d consumer warps, %d phases of %d label(s); threshold %g; phase order: %s\n" % (
        src, plan["tpc"], plan["block_threads"] // 32 - 1, plan["n_phases"], plan["labels_per_phase"], thr, order))
    res = {}
    for fi in range(n_frames):
        det.process(*frames[fi])
        lm = linear_memories(det, tmpl.cells)
        for mask in masks:
            r = count_frame(lm, tmpl, plan, thr, mask, order)
            res[(fi, mask)] = r
            out.write("frame %d  %-5s  skipped %5.1f %%  (needed %d of %d)  alive %s  busiest warp %.1f -> %.1f\n" % (
                fi, mask, 100 * r["skipped"], r["needed"], r["total"], " ".join(map(str, r["alive"])), r["busiest_warp_full"],
                r["busiest_warp_pruned"]))
            out.flush()
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--threshold", type=float, default=75.0)
    ap.add_argument("--order", choices=("rotation", "mass"), default="rotation")
    a = ap.parse_args()
    run(a.frames, a.threshold, order=a.order)
