"""Recognition frames/s on template-sharded pipes, one process per GPU (sharded.NativeShardedPipe: frame f refined by rank f % N alone,
its results pushed to the other ranks over peer memory), beside the current C4 figure of bench.py at the same N.

Workload: the C4 set of bench.py (1280 x 720, 15 classes x 2,000 templates, L = 2, T = {5, 8}, top-5 hypotheses, NMS at 30 mm), every
template's crop = frame 0's depth cut to its level-0 box, host frames page-locked.  One host thread per rank submits and collects with
`depth` frames in flight; frames/s = timed frames over the host wall clock, max over ranks.  At N = 1 the pipe is a plain recognition pipe
(fl_pipe_set_recognition: nothing to exchange).  The first frames of every rank are compared byte for byte with a single handle's
fl_recognize over the whole set.  Prints one JSON line per (N, depth), one per bench.py run, and the GPU name and power limit.
    python tools/exp_sharded_reco.py [--gpus 1,2,4,8] [--depths 4,8] [--frames 200] [--bench-steps 100]"""
from __future__ import annotations

import argparse
import json
import os
import socket
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]
sys.dont_write_bytecode = True
N_CHECK = 6                                                      # frames compared with the single handle


def gpu_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().split("\n")[0].split(", ") + ["?"])[:2] if r.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


def _free_port() -> int:
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _torchrun(n: int, argv) -> list:
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port())] + argv
    r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=3000)
    lines = [l for l in r.stdout.split("\n") if l.startswith("{")]
    if r.returncode != 0 or not lines:
        raise SystemExit("exp_sharded_reco.py: %s failed (%d):\n%s" % (" ".join(argv[:2]), r.returncode, r.stdout[-3000:]))
    return lines


def worker(args) -> None:
    import torch
    import torch.distributed as dist
    import bench
    import fealess_b200 as fb
    from fealess_b200 import sharded, synth

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    cfg = bench.PIPELINES["C4"]
    W, H, T = cfg["W"], cfg["H"], cfg["T"]
    n_total = cfg["classes"] * cfg["per_class"]
    frames = [synth.make_frame(W, H, i) for i in range(2)]
    q = bench.oracle_quantized(frames[0], T)
    ts = synth.make_templates(n_total, W, H, T, n_classes=cfg["classes"], seed=1, quantized=q, planted_fraction=0.004)
    LM = ts.n_levels * ts.n_modalities
    rects = [tuple(int(v) for v in ts.headers[t * LM][[2, 3, 0, 1]]) for t in range(n_total)]
    crops = [frames[0][1]] * n_total
    params = fb.reco_params(threshold=bench.THRESHOLD, top_k=bench.TOP_K, th_obj_dist=30.0)
    K = (608.0 * W / 640, 608.0 * W / 640, W / 2.0, H / 2.0)
    pinned = []
    for b, d in frames:
        pb, pd = torch.from_numpy(b).pin_memory(), torch.from_numpy(d.view(np.int16)).pin_memory()
        pinned.append((pb.numpy(), pd.numpy().view(np.uint16)))
    ref = fb.Handle(T, (0, 1), W, H, device=local)
    ref.upload_templates(ts)
    ref.upload_model_depths(crops, rects)
    ref.set_recognition(np.arange(n_total), params=params)
    want = [ref.recognize(*pinned[i % 2], K, W, H) for i in range(N_CHECK)]
    ref.close()
    for depth in args.depths:
        if world > 1:
            obj = sharded.NativeShardedPipe(ts, rank, world, depth=depth, capacity=4096, device=dev, max_width=W, max_height=H)
            obj.upload_model_depths(crops, rects)
            obj.set_recognition(np.arange(n_total), params=params)
            pipe = obj.pipe
        else:
            pipe = obj = fb.Pipe(depth, T, (0, 1), W, H, device=local)
            pipe.upload_templates(ts)
            pipe.upload_model_depths(crops, rects)
            pipe.set_recognition(np.arange(n_total), params=params)

        def run(n):
            out = []
            for i in range(n):
                if pipe.in_flight() == depth:
                    out.append(pipe.collect_recognition())
                pipe.submit_recognition(*pinned[i % 2], K, W, H)
            while pipe.in_flight():
                out.append(pipe.collect_recognition())
            return out
        got = run(max(N_CHECK, 2 * depth))                             # warm-up + check: packing, module loads, workspaces
        same = all(g[0] == w_[0] and g[2] == w_[2] and g[1].tobytes() == w_[1].tobytes() for g, w_ in zip(got, want))
        torch.cuda.synchronize(); dist.barrier()
        launches0 = pipe.launch_count()
        t0 = time.perf_counter()
        run(args.frames)
        dt = time.perf_counter() - t0
        launches = pipe.launch_count() - launches0
        t = torch.tensor([dt, 0.0 if same else 1.0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        owned = len(range(rank, args.frames, world))
        rows = [None] * world
        dist.all_gather_object(rows, dict(rank=rank, launches_per_frame=round(launches / args.frames, 2), icp_launches=owned))
        if rank == 0:
            print(json.dumps(dict(workload="C4 Recognition on template-sharded pipes", W=W, H=H, templates=n_total, top_k=bench.TOP_K, nms_mm=30.0,
                                  gpus=world, depth=depth, frames=args.frames, frames_per_s=round(args.frames / float(t[0].item()), 1),
                                  timer="host wall clock, max over ranks", per_rank=rows,
                                  equal_to_single_handle_first_frames=bool(t[1].item() == 0.0))), flush=True)
        obj.close()
    dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--depths", default="4,8")
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--bench-steps", type=int, default=100)
    ap.add_argument("--worker", action="store_true")
    args = ap.parse_args()
    args.depths = [int(x) for x in args.depths.split(",")]
    if args.worker:
        worker(args)
        sys.stdout.flush()
        os._exit(0)                                                # (no interpreter teardown: it frees torch tensors in arbitrary order)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("exp_sharded_reco.py measures on the GPU; no device is visible")
    n_gpus = torch.cuda.device_count()
    print(json.dumps(dict(gpu_info(), visible_gpus=n_gpus)), flush=True)
    for n in [int(x) for x in args.gpus.split(",")]:
        if n > n_gpus:
            print(json.dumps(dict(gpus=n, skipped="%d GPU(s) visible" % n_gpus)), flush=True)
            continue
        for line in _torchrun(n, [os.path.abspath(__file__), "--worker", "--depths", ",".join(map(str, args.depths)), "--frames", str(args.frames)]):
            print(line, flush=True)
        for line in _torchrun(n, [os.path.join(ROOT, "bench.py"), "--config", "C4", "--steps", str(args.bench_steps)]):
            print(json.dumps(dict(bench_py_C4_gpus=n, line=json.loads(line))), flush=True)


if __name__ == "__main__":
    main()
