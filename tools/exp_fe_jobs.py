"""Developer experiment (GPU): SM time per job of the single-launch front end (k_front_end_wave), at 1 and at 4 frames in flight.

bench.py's C2 inputs (640x480, T = (5, 8), 8,000 templates planted on the oracle's quantised images, seed 1, 1 % planted,
threshold 75, synth frames 0-7).  Every handle runs with FL_OPT_TRACE, so every CTA of the front end adds its span (from its
start to its end, dependency waits included) to its job's sum (FL_DBG_FE_TRACE).  Per frame the script prints, averaged over
the frames measured:
  * per job: CTAs, CTA-us (summed CTA spans, globaltimer), SM-us = CTA-us / 8 (k_front_end_wave keeps 8 CTAs on an SM:
    __launch_bounds__(256, 8), and its shared memory allows 8), and the summed SM cycles over the ns (the clock the CTAs ran at);
  * the front end's total, and its span (first CTA start to last CTA end);
  * the staged similarity kernel's summed CTA loop ends (FL_DBG_STAGED_TRACE: t_loop_end - t_start over its CTAs) and CTA ends,
    in SM-us (one CTA per SM);
  * each total over the 148 SMs: the part of a frame's time the kernel would take if it had the whole GPU to itself;
  * the card's name and power limit.
1 in flight: one handle, each frame ends in a wait.  4 in flight: fealess_b200.sharded.ShardedPipe of depth 4 as bench.py drives
it, one handle per slot.  FL_OPT_TRACE synchronises a handle's stream once per frame, so the 4-deep stream is slower than
bench.py's; the sums are what a frame's CTAs hold of the SMs while frames overlap.
Usage: python tools/exp_fe_jobs.py [--frames 200] [--md FILE]"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np
import torch

import fealess_b200 as fb
from fealess_b200 import sharded, synth

W, H, T, THR, DEPTH = 640, 480, (5, 8), 75.0, 4
FE_CTAS_PER_SM, N_SM = 8, 148
KIND = {2: "pyrDown", 3: "resize", 4: "spread+LM", 5: "colour", 6: "depth", 7: "prefetch"}


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                              timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return "nvidia-smi unavailable (%s); torch: %s" % (e, torch.cuda.get_device_name(0))


class Acc:
    """per-frame sums of one setting"""

    def __init__(self):
        self.n = 0
        self.jobs = None            # [n_jobs, 2] kind, CTAs
        self.ns = self.cyc = None   # [n_jobs] summed CTA spans
        self.span = self.sim_loop = self.sim_end = 0.0

    def add(self, h):
        fe, st = h.fe_trace(), h.staged_trace()
        if self.jobs is None:
            self.jobs = fe[:, :2].copy()
            self.ns, self.cyc = np.zeros(len(fe)), np.zeros(len(fe))
        assert np.array_equal(self.jobs, fe[:, :2]), "the front end's job list changed between frames"
        self.ns += fe[:, 5]
        self.cyc += fe[:, 4]
        self.span += float(fe[:, 3].max() - fe[:, 2].min())
        self.sim_loop += float((st[:, 3] - st[:, 0]).sum())
        self.sim_end += float((st[:, 4] - st[:, 0]).sum())
        self.n += 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=200, help="frames measured per setting (after 16 warm-up frames)")
    ap.add_argument("--md", help="also write the tables here (markdown)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("exp_fe_jobs.py needs a GPU")
    import fl_oracle_py as F
    frames = [synth.make_frame(W, H, i) for i in range(8)]
    det = F.Detector(T)
    det.process(*frames[0])
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    tset = synth.make_templates(8000, W, H, T, seed=1, quantized=q, planted_fraction=0.01)
    d_inputs = [(torch.from_numpy(f[0]).cuda(), torch.from_numpy(f[1].view(np.int16)).cuda()) for f in frames]

    def make_handle():
        h = fb.Handle(T, (0, 1), W, H)
        assert h.debug_option(fb.FL_OPT_TRACE, 1) == 0
        return h

    # 1 in flight
    one = Acc()
    h1 = make_handle()
    h1.upload_templates(tset)
    for i in range(16 + args.frames):
        tb, td = d_inputs[i % 8]
        h1.match_device_async(tb.data_ptr(), td.data_ptr(), W, H, THR)
        h1.match_wait()
        if i >= 16:
            one.add(h1)
    h1.close()

    # 4 in flight
    four = Acc()
    pipe = sharded.ShardedPipe(make_handle, tset, 0, 1, depth=DEPTH, capacity=2048, device=0)
    seen = 0
    for i in range(16 + args.frames + DEPTH):
        if pipe.in_flight() == DEPTH or i >= 16 + args.frames:
            s = pipe.collect()
            if seen >= 16:
                four.add(s.h)
            seen += 1
        if i < 16 + args.frames:
            tb, td = d_inputs[i % 8]
            pipe.submit_device(tb.data_ptr(), td.data_ptr(), W, H, THR)
    while pipe.in_flight():
        s = pipe.collect()
        four.add(s.h)
    for s in pipe.slots:
        s.close()

    c = card()

    def sm_us(ns, n, per_sm):
        return ns / n / 1e3 / per_sm

    out = ["card (name, power limit, SM clock, max SM clock): " + c, "",
           "Per frame, mean over %d frames (1 in flight) and %d frames (4 in flight).  CTA-us = summed CTA spans (globaltimer); SM-us = "
           "CTA-us / %d CTAs per SM; GHz = summed clock64 cycles over summed ns." % (one.n, four.n, FE_CTAS_PER_SM), "",
           "| job | kind | CTAs | CTA-us, 1 in flight | SM-us, 1 in flight | SM-us, 4 in flight | GHz |", "|---|---|---|---|---|---|---|"]
    for j, (k, n) in enumerate(one.jobs):
        out.append("| %d | %s | %d | %.1f | %.1f | %.1f | %.2f |" % (j, KIND.get(int(k), "?"), n, one.ns[j] / one.n / 1e3, sm_us(one.ns[j], one.n, FE_CTAS_PER_SM),
                                                                 sm_us(four.ns[j], four.n, FE_CTAS_PER_SM), one.cyc[j] / max(one.ns[j], 1)))
    for name, key in (("spread+LM", 4), ("colour", 5), ("depth", 6), ("pyrDown", 2), ("prefetch", 7)):
        sel = one.jobs[:, 0] == key
        out.append("| all | %s | %d | %.1f | %.1f | %.1f | |" % (name, one.jobs[sel, 1].sum(), one.ns[sel].sum() / one.n / 1e3,
                                                           sm_us(one.ns[sel].sum(), one.n, FE_CTAS_PER_SM), sm_us(four.ns[sel].sum(), four.n, FE_CTAS_PER_SM)))
    fe1, fe4 = sm_us(one.ns.sum(), one.n, FE_CTAS_PER_SM), sm_us(four.ns.sum(), four.n, FE_CTAS_PER_SM)
    out.append("| **front end** | | %d | %.1f | **%.1f** | **%.1f** | |" % (one.jobs[:, 1].sum(), one.ns.sum() / one.n / 1e3, fe1, fe4))
    out += ["", "| per frame | 1 in flight | 4 in flight |", "|---|---|---|",
            "| front end span, first CTA start to last CTA end, us | %.2f | %.2f |" % (one.span / one.n / 1e3, four.span / four.n / 1e3),
            "| front end, SM-us | %.1f | %.1f |" % (fe1, fe4),
            "| front end, SM-us / %d SMs, us | %.2f | %.2f |" % (N_SM, fe1 / N_SM, fe4 / N_SM),
            "| similarity kernel, summed CTA loop ends, SM-us | %.1f | %.1f |" % (sm_us(one.sim_loop, one.n, 1), sm_us(four.sim_loop, four.n, 1)),
            "| similarity kernel, summed CTA ends, SM-us | %.1f | %.1f |" % (sm_us(one.sim_end, one.n, 1), sm_us(four.sim_end, four.n, 1)),
            "| similarity kernel, summed CTA ends / %d SMs, us | %.2f | %.2f |" % (N_SM, sm_us(one.sim_end, one.n, 1) / N_SM, sm_us(four.sim_end, four.n, 1) / N_SM),
            "", "card: " + card()]
    text = "\n".join(out)
    print(text)
    if args.md:
        with open(args.md, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
