"""Developer experiment (GPU): the staged similarity kernel with and without its early exit (--ab prune), or with its phases in
the order of the frame's response mass and in the rotated order of FL_OPT_SIM_ROTATE (--ab order), in one process on the same handles.

bench.py's C2 inputs (640x480, 8,000 templates, seed 1, 1 % planted, threshold 75).  The option FL_OPT_SIM_NO_PRUNE is switched
(or FL_OPT_SIM_ROTATE) is switched
off and on in alternation, ROUNDS times, and each time the script measures
  * the similarity stage (the library's own CUDA events, h.profile) over one frame at a time;
  * the stream: microseconds per frame at 4 frames in flight (fealess_b200.sharded.ShardedPipe, as bench.py drives it), inputs
    cycled over 160 device copies (> L2);
  * the in-kernel timeline (FL_OPT_TRACE, a handle of its own): per CTA the end of the phase loop and of the kernel, in us after
    the first CTA started (as tools/exp_warps.py reads it).
The match list must not depend on the option; the script checks that too.
Usage: python tools/exp_prune.py [--ab prune|order] [--rounds 5] [--json F]"""
import argparse
import ctypes as C
import json
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


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active"
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                              timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return "nvidia-smi unavailable (%s); torch: %s" % (e, torch.cuda.get_device_name(0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--frames", type=int, default=400, help="frames per stream measurement")
    ap.add_argument("--json", help="write the per-round figures here")
    ap.add_argument("--ab", choices=("prune", "order"), default="prune",
                    help="prune: FL_OPT_SIM_NO_PRUNE off / on; order: FL_OPT_SIM_ROTATE off (by response mass) / on (rotated)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("exp_prune.py needs a GPU")
    import fl_oracle_py as F
    frames = [synth.make_frame(W, H, i) for i in range(8)]
    det = F.Detector(T)
    det.process(*frames[0])
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    tset = synth.make_templates(8000, W, H, T, seed=1, quantized=q, planted_fraction=0.01)
    print("card:", card())

    pipe = sharded.ShardedPipe(lambda: fb.Handle(T, (0, 1), W, H), tset, 0, 1, depth=DEPTH, capacity=2048, device=0)
    h0 = pipe.slots[0].h
    d_inputs = [(torch.from_numpy(frames[j % 8][0]).cuda(), torch.from_numpy(frames[j % 8][1].view(np.int16)).cuda()) for j in range(160)]
    htr = fb.Handle(T, (0, 1), W, H)
    htr.debug_option(fb.FL_OPT_TRACE, 1)
    htr.upload_templates(tset)
    torch.cuda.synchronize()
    seq = [0]

    opt = fb.FL_OPT_SIM_NO_PRUNE if args.ab == "prune" else fb.FL_OPT_SIM_ROTATE
    names = ("early exit", "FL_OPT_SIM_NO_PRUNE") if args.ab == "prune" else ("by response mass", "FL_OPT_SIM_ROTATE")

    def set_opt(v):
        for s in pipe.slots:
            assert s.h.debug_option(opt, v) == 0
        assert htr.debug_option(opt, v) == 0

    def stream(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        last = None
        for k in range(n + 2 * DEPTH):
            if pipe.in_flight() == DEPTH:
                pipe.collect()
            tb, td = d_inputs[seq[0] % len(d_inputs)]
            seq[0] += 1
            if k == 2 * DEPTH:
                e0.record(pipe.slots[pipe.submitted % DEPTH].stream)
            pipe.submit_device(tb.data_ptr(), td.data_ptr(), W, H, THR)
        while pipe.in_flight():
            last = pipe.collect()
        e1.record(last.stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / n

    def stage(n=100):
        h0.profile(True)
        acc = np.zeros(4)
        for i in range(n + 3):
            tb, td = d_inputs[i % len(d_inputs)]
            h0.match_device_async(tb.data_ptr(), td.data_ptr(), W, H, THR)
            h0.match_wait()
            if i >= 3:
                acc += h0.last_stage_ms()
        h0.profile(False)
        return acc[1] * 1e3 / n

    def timeline():
        loop_end, end = [], []
        buf = np.zeros(1024 * 136 + 8, np.uint64)
        for i in range(8):
            rc, _ = htr.match(*frames[i], THR)
            assert rc == 0
            n = fb.lib().fl_debug_get(htr._h, 4, 0, 0, 0, C.c_void_p(buf.ctypes.data), C.c_size_t(buf.nbytes))
            tr = buf[:n * 8].reshape(n, 8).astype(np.int64)
            t0 = tr[:, 0].min()
            loop_end.append((tr[:, 3] - t0) / 1e3)
            end.append((tr[:, 4] - t0) / 1e3)
        le, en = np.concatenate(loop_end), np.concatenate(end)
        return float(le.mean()), float(le.max()), float(en.mean()), float(en.max())

    lists = {}
    for v in (0, 1):
        set_opt(v)
        lists[v] = [h0.match(*frames[i], THR)[1] for i in range(8)]
    same = all(np.array_equal(a, b) for a, b in zip(lists[0], lists[1]))
    print("match lists of the 8 frames identical with %s and with %s:" % names, same)

    set_opt(0)
    stream(200)
    stage(20)
    rows = []
    for r in range(args.rounds):
        for v in ((0, 1) if r % 2 == 0 else (1, 0)):
            set_opt(v)
            row = {"round": r, "option": names[v], "early_exit": v == 0, "stage_similarity_us": stage(), "stream_us_per_frame": stream(args.frames)}
            row["cta_loop_end_us_mean"], row["cta_loop_end_us_max"], row["cta_end_us_mean"], row["cta_end_us_max"] = timeline()
            rows.append(row)
            print(json.dumps(row))
            sys.stdout.flush()
    set_opt(0)
    for v, name in enumerate(names):
        sel = [x for x in rows if x["early_exit"] == (v == 0)]
        print("%-20s median: stage %.1f us, stream %.2f us/frame, CTA loop end mean %.1f / max %.1f us, CTA end max %.1f us" % (
            name, *(float(np.median([x[k] for x in sel])) for k in ("stage_similarity_us", "stream_us_per_frame", "cta_loop_end_us_mean",
                                                                     "cta_loop_end_us_max", "cta_end_us_max"))))
    print("card:", card())
    if args.json:
        with open(args.json, "w") as f:
            json.dump({"card": card(), "lists_identical": same, "rows": rows}, f, indent=1)
    for s in pipe.slots:
        s.close()
    htr.close()


if __name__ == "__main__":
    main()
