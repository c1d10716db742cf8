"""Masked against unmasked C2 frames, frame and masks resident in device memory: time per frame with 1 frame in flight (one handle,
fl_match_device_async + fl_match_wait) and with 4 in flight (a depth-4 fl_pipe fed with fl_pipe_submit_masked), launches per frame,
and whether the pipe's masked lists equal one handle's.  Prints one JSON line.

    python tools/exp_masked.py [--root TREE] [--steps N] [--reps R]

--root: the tree whose fealess_b200 package is imported (default: this one).  A tree without fl_pipe_submit_masked (the commit before
masked frames took the single-launch front end) runs the 1-in-flight cases only: its fl_match_device already took device masks.
Times are host wall clock over N frames that each end in a device wait, median of R repetitions; the 8 frames and their masks
(18 MB) stay in the 126 MB L2 between frames, as in a camera loop that matches what it has just uploaded."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--steps", type=int, default=400)
ap.add_argument("--reps", type=int, default=5)
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))
sys.path.insert(0, os.path.join(os.path.abspath(args.root), "oracle"))

import torch  # noqa: E402

import fealess_b200 as fb  # noqa: E402
import fl_oracle_py as F  # noqa: E402
from fealess_b200 import synth  # noqa: E402

W, H, T, THR = 640, 480, (5, 8), 75.0
L = fb.lib()
masked_pipe = hasattr(L, "fl_pipe_submit_masked")


def mask(seed, density=0.8):
    rng = np.random.default_rng(seed)
    m = (rng.random((H, W)) < density).astype(np.uint8) * np.uint8(255)
    m[H // 8:H // 2, W // 6:W // 2] = 255
    m[:, 3 * W // 4:] = 0
    return m


frames = [synth.make_frame(W, H, i) for i in range(8)]
det = F.Detector(T)                                       # bench.py's C2 set: 1 % of the templates planted on frame 0
assert det.process(*frames[0]) == 0
ts = synth.make_templates(8000, W, H, T, seed=1, quantized=[det.quantized(l, m) for l in range(2) for m in range(2)], planted_fraction=0.01)
dev = [(torch.from_numpy(b).cuda(), torch.from_numpy(d.view(np.int16)).cuda()) for b, d in frames]
dmask = [(torch.from_numpy(mask(2 * i)).cuda(), torch.from_numpy(mask(2 * i + 1, 0.6)).cuda()) for i in range(8)]
marr = [(C.c_void_p * 2)(a.data_ptr(), b.data_ptr()) for a, b in dmask]

h = fb.Handle(T, (0, 1), W, H)
h.upload_templates(ts)


def one(i, masked):
    b, d = dev[i % 8]
    rc = L.fl_match_device_async(h._h, C.c_void_p(b.data_ptr()), C.c_void_p(d.data_ptr()), W, H, marr[i % 8] if masked else None,
                                 C.c_float(THR), None, 0)
    assert rc == 0, rc
    h.match_wait()


def timed(fn, n):
    fn(0)
    fn(1)
    torch.cuda.synchronize()
    reps = []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        for i in range(n):
            fn(i)
        reps.append((time.perf_counter() - t0) / n * 1e6)
    return round(statistics.median(reps), 2), [round(r, 2) for r in reps]


out = {"gpu": torch.cuda.get_device_name(0), "root": os.path.abspath(args.root), "steps": args.steps, "reps": args.reps}
one(0, False)                                             # the geometry's one-time set-up (packed features, staged plan) is not a frame's
for masked in (False, True):
    n0 = h.launch_count()
    one(0, masked)
    out["launches_per_frame_" + ("masked" if masked else "unmasked")] = h.launch_count() - n0
    out["us_1_in_flight_" + ("masked" if masked else "unmasked")] = timed(lambda i, m=masked: one(i, m), args.steps)

if masked_pipe:
    p = fb.Pipe(4, T, (0, 1), W, H)
    p.upload_templates(ts)

    def piped(i, masked):
        if p.in_flight() == 4:
            p.collect(copy=False)
        b, d = dev[i % 8]
        p.submit_device(b.data_ptr(), d.data_ptr(), W, H, THR, d_masks=[x.data_ptr() for x in dmask[i % 8]] if masked else None)

    for masked in (False, True):
        us, reps = timed(lambda i, m=masked: piped(i, m), args.steps)
        while p.in_flight():
            p.collect(copy=False)
        out["us_4_in_flight_" + ("masked" if masked else "unmasked")] = (us, reps)
    # every masked list of the pipe equals the single handle's
    want = []
    for i in range(8):
        one(i, True)
        want.append(h.match_fetch())
    got = []
    for i in range(8):
        if p.in_flight() == 4:
            got.append(p.collect()[1])
        piped(i, True)
    while p.in_flight():
        got.append(p.collect()[1])
    out["pipe_lists_equal_single"] = all(np.array_equal(a, b) for a, b in zip(got, want))
    p.close()
h.close()
print(json.dumps(out))
