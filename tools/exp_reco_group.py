"""Recognition frames/s of a template-sharded group (fl_group_*_recognition) driven by ONE host thread, n members x depth slots,
beside the single-GPU recognition pipe (fl_pipe_*_recognition) at the same depth.

Two workloads, templates planted on frame 0 from the C oracle's quantised images, frames page-locked, poses on the host at the end:
  C1  640 x 480, 2,000 templates, top-1
  C4  1280 x 720, 30,000 templates, top-5, nonMaximumSuppression at 30 mm
Every template's crop is the frame's depth cut to its level-0 box.  The group's members are the first n visible GPUs, or - with fewer
GPUs than members - device 0 repeated.  Members that share a device measure the COST of sharding on one GPU (the exchange and the
per-member front ends), not scaling over GPUs; the output says which it was.  Every frame's records are compared byte for byte with
the pipe's.  Prints one JSON line per (workload, n, depth) and one with the GPU name and power limit.
    python tools/exp_reco_group.py [--frames 100] [--members 2,4] [--depths 1,4,8] [--workloads C1,C4]"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]
sys.dont_write_bytecode = True

T = (5, 8)
WORKLOADS = {"C1": dict(W=640, H=480, n_templates=2000, top_k=1, th=0.0, planted=0.01),
             "C4": dict(W=1280, H=720, n_templates=30000, top_k=5, th=30.0, planted=0.002)}
_PINNED = []


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


def stream(obj, frames, K, W, H, depth):
    """every frame through submit / collect from this thread with up to `depth` in flight: (seconds, [records bytes per frame])"""
    out, queued = [], 0
    t0 = time.perf_counter()
    for fb_, fd_ in frames:
        if queued == depth:
            rc, recs, _ = obj.collect_recognition()
            out.append((rc, recs.tobytes()))
            queued -= 1
        obj.submit_recognition(fb_, fd_, K, W, H)
        queued += 1
    while queued:
        rc, recs, _ = obj.collect_recognition()
        out.append((rc, recs.tobytes()))
        queued -= 1
    return time.perf_counter() - t0, out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=100, help="timed frames per arm")
    ap.add_argument("--members", default="2,4")
    ap.add_argument("--depths", default="1,4,8")
    ap.add_argument("--workloads", default="C1,C4")
    args = ap.parse_args()
    import torch
    import fealess_b200 as fb
    import fl_oracle_py as F
    from fealess_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("exp_reco_group.py measures on the GPU; no device is visible")
    n_gpus = torch.cuda.device_count()
    print(json.dumps(dict(gpu_info(), visible_gpus=n_gpus)), flush=True)
    members = [int(x) for x in args.members.split(",")]
    depths = [int(x) for x in args.depths.split(",")]
    for name in args.workloads.split(","):
        w = WORKLOADS[name]
        W, H = w["W"], w["H"]
        b, d = synth.make_frame(W, H, 0)
        od = F.Detector(T)
        assert od.process(b, d) == 0
        q = [od.quantized(l, m) for l in range(2) for m in range(2)]
        ts = synth.make_templates(w["n_templates"], W, H, T, n_classes=1, seed=7, quantized=q, planted_fraction=w["planted"])
        LM = ts.n_levels * ts.n_modalities
        rects = [tuple(int(v) for v in ts.headers[t * LM][[2, 3, 0, 1]]) for t in range(ts.n_templates)]
        crops = [d] * ts.n_templates
        params = fb.reco_params(top_k=w["top_k"], th_obj_dist=w["th"])
        K = (608.0 * W / 640, 608.0 * W / 640, W / 2.0, H / 2.0)
        frame = (pinned(b), pinned(d))
        frames = [frame] * args.frames
        for depth in depths:
            pipe = fb.Pipe(depth, T, (0, 1), W, H)
            pipe.upload_templates(ts)
            pipe.upload_model_depths(crops, rects)
            pipe.set_recognition(np.arange(ts.n_templates), params=params)
            stream(pipe, frames[:2 * depth], K, W, H, depth)                          # warm-up: packing, module load
            t_pipe, want = stream(pipe, frames, K, W, H, depth)
            pipe.close()
            for n in members:
                devices = list(range(n)) if n_gpus >= n else [0] * n
                g = fb.Group(devices, T, (0, 1), W, H, exchange_capacity=8192, depth=depth)
                g.upload_templates(ts)
                g.upload_model_depths(crops, rects)
                g.set_recognition(np.arange(ts.n_templates), params=params)
                stream(g, frames[:2 * depth * n], K, W, H, depth)
                t_group, got = stream(g, frames, K, W, H, depth)
                g.close()
                print(json.dumps(dict(workload=name, W=W, H=H, templates=ts.n_templates, top_k=w["top_k"], nms_mm=w["th"], members=n, depth=depth,
                                      devices=devices, sharing="members share one GPU: cost of sharding, not scaling" if len(set(devices)) < n else "one GPU per member",
                                      group_fps=round(args.frames / t_group, 1), pipe_fps=round(args.frames / t_pipe, 1),
                                      results_per_frame=len(want[0][1]) // fb.RECO_RESULT_DTYPE.itemsize,
                                      bit_identical=got == want)), flush=True)


if __name__ == "__main__":
    main()
