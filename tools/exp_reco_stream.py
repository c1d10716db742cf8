"""Recognition frames/s: today's synchronous mirror against the device-side Recognition pipe driven by ONE host thread.

The C1 workload exactly as bench.bench_recognition builds it: 1 object x 2,000 templates planted on frame 0 (C oracle's quantised
images), top-5 hypotheses, the 640x480 frame and its pixel-doubled 1280x960 variant (rescaled on the device).  Frames sit in
page-locked memory; every run ends with the poses on the host.  Arms, alternated in the same process for --rounds rounds:
  (a) ObjRecoLmICP.Recognition: one thread with one instance, and 8 threads with 8 instances (what bench.py's stream arm does)
  (b) ObjRecoLmICP.submit / collect (fl_pipe_submit_recognition) from one thread at 1, 2, 4 and 8 frames in flight, with the
      runtime spinning in the wait and with a blocking wait (fl_set_blocking_wait)
Every frame's poses are checked bit for bit against the synchronous mirror's.  Prints one JSON line: frames/s per arm (median over
the rounds), kernel launches per frame of the pipe, GPU name and power limit.
    python tools/exp_reco_stream.py [--frames 200] [--rounds 3]"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]
sys.dont_write_bytecode = True

W, H, T = 640, 480, (5, 8)
N_TEMPLATES, TOP_K = 2000, 5


_PINNED = []              # the torch tensors that own the page-locked blocks


def pinned(a: np.ndarray) -> np.ndarray:
    import torch
    t = torch.empty(a.nbytes, dtype=torch.uint8, pin_memory=True)
    _PINNED.append(t)
    p = t.numpy().view(a.dtype).reshape(a.shape)
    p[...] = a
    return p


def gpu_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().split("\n")[0].split(", ") + ["?"])[:2] if r.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=200, help="timed frames per arm and round")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import fealess_b200 as fb
    import fl_oracle_py as F
    from fealess_b200 import reco, synth

    b, d = synth.make_frame(W, H, 0)
    od = F.Detector(T)
    assert od.process(b, d) == 0
    q = [od.quantized(l, m) for l in range(2) for m in range(2)]
    tset = synth.make_templates(N_TEMPLATES, W, H, T, n_classes=1, seed=7, quantized=q, planted_fraction=0.01)
    big_b, big_d = np.repeat(np.repeat(b, 2, 0), 2, 1), np.repeat(np.repeat(d, 2, 0), 2, 1)
    sizes = {"640x480": (pinned(b), pinned(d)), "1280x960_input": (pinned(big_b), pinned(big_d))}

    def mirror(frames_in_flight=1):
        det = fb.Detector()
        det.add_template_set(tset)
        r = reco.ObjRecoLmICP(frames_in_flight=frames_in_flight)
        r.add_detector(det, {(None, tid): d for tid in range(N_TEMPLATES)})
        return r

    sync = [mirror() for _ in range(8)]
    pipes = {k: mirror(k) for k in (1, 2, 4, 8)}
    L = fb.lib()
    L.fl_pipe_handle.restype = C.c_void_p

    def kdict(img):
        return dict(fx=608.0, fy=608.0, cx=320.0, cy=240.0, width=img.shape[1], height=img.shape[0])

    want = {}
    for tag, (fb_, fd_) in sizes.items():
        rc, res = sync[0].Recognition(fb_, fd_, kdict(fb_), top_k=TOP_K)
        assert rc == 0 and res, "the benchmark frame produced no pose"
        want[tag] = [(x["strObjTag"], x["tWorld2Cam"].tobytes()) for x in res]

    def check(tag, res):
        if [(x["strObjTag"], x["tWorld2Cam"].tobytes()) for x in res] != want[tag]:
            raise RuntimeError("%s: a frame's poses differ from the synchronous mirror's" % tag)

    def run_sync(tag, n_threads, n):
        fb_, fd_ = sizes[tag]
        K = kdict(fb_)
        errors = []

        def loop(r, k):
            try:
                for _ in range(k):
                    rc, res = r.Recognition(fb_, fd_, K, top_k=TOP_K)
                    assert rc == 0
                    check(tag, res)
            except Exception as e:  # noqa: BLE001  (re-raised in the main thread)
                errors.append(e)
        per = max(n // n_threads, 1)
        ths = [threading.Thread(target=loop, args=(sync[i], per)) for i in range(n_threads)]
        t0 = time.perf_counter()
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        dt = time.perf_counter() - t0
        if errors:
            raise errors[0]
        return per * n_threads / dt

    def run_pipe(tag, k, blocking, n):
        r, (fb_, fd_) = pipes[k], sizes[tag]
        K = kdict(fb_)
        assert r.submit(fb_, fd_, K, top_k=TOP_K) == 0                 # sets the pipe up (outside the timed window)
        check(tag, r.collect()[1])
        for i in range(k):
            assert L.fl_set_blocking_wait(C.c_void_p(L.fl_pipe_handle(r._pipe._p, i)), int(blocking)) == 0
        n0 = r._pipe.launch_count()
        t0 = time.perf_counter()
        queued = 0
        for _ in range(n):
            if queued == k:
                rc, res = r.collect()
                check(tag, res)
                queued -= 1
            assert r.submit(fb_, fd_, K, top_k=TOP_K) == 0
            queued += 1
        while queued:
            rc, res = r.collect()
            check(tag, res)
            queued -= 1
        fps = n / (time.perf_counter() - t0)
        return fps, (r._pipe.launch_count() - n0) / n

    results, launches = {}, {}
    for rnd in range(args.rounds + 1):                                  # round 0: warm-up of every arm and shape, not reported
        for tag in sizes:
            arms = [("sync_1thread", lambda: run_sync(tag, 1, args.frames)), ("sync_8threads_8instances", lambda: run_sync(tag, 8, args.frames))]
            for k in (1, 2, 4, 8):
                for blocking in (False, True):
                    arms.append(("pipe_1thread_depth%d_%s" % (k, "blocking" if blocking else "spin"), lambda k=k, bl=blocking: run_pipe(tag, k, bl, args.frames)))
            for name, fn in arms:
                v = fn()
                if isinstance(v, tuple):
                    v, launches[tag] = v
                if rnd > 0:
                    results.setdefault(tag, {}).setdefault(name, []).append(v)
    out = {"workload": "C1: Recognition (match at 75 %% + ICP of the top-%d matches + poses on the host), 1 object x %d templates, L=2, T={5,8}, "
                       "frames in page-locked host memory" % (TOP_K, N_TEMPLATES),
           "unit": "frames/s, host wall clock over %d frames, median of %d rounds" % (args.frames, args.rounds),
           "poses_bit_identical_to_sync_mirror": True,
           "pipe_kernel_launches_per_frame": launches}
    for tag, arms in results.items():
        out[tag] = {name: round(float(np.median(v)), 1) for name, v in arms.items()}
    out.update(gpu_info())
    print(json.dumps(out))


if __name__ == "__main__":
    main()
