"""Multi-GPU Recognition parity check (run under torch.distributed.run on N GPUs of one box): sharded.NativeShardedPipe with
symmetric-memory exchange buffers, frame f refined by rank f % N and its results pushed to the other ranks; every rank must return a
single handle's fl_recognize results over the whole set (records as bytes, and the summary), frame after frame."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import cv2
import numpy as np
import torch
import torch.distributed as dist
import fealess_b200 as fb
from fealess_b200 import sharded, synth
import fl_oracle_py as F

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
W, H, T = 640, 480, (5, 8)
K = (608.0, 608.0, 320.0, 240.0)
b, d = synth.make_frame(W, H, 0)
det = F.Detector(T); det.process(b, d)
q = [det.quantized(l, m) for l in range(2) for m in range(2)]
ts = synth.make_templates(37, W, H, T, n_classes=3, seed=62, quantized=q, planted_fraction=0.5)
LM = ts.n_levels * ts.n_modalities
crops = [d] * ts.n_templates
rects = [tuple(int(v) for v in ts.headers[t * LM][[2, 3, 0, 1]]) for t in range(ts.n_templates)]
big = (cv2.resize(b, (1280, 960), interpolation=cv2.INTER_CUBIC), cv2.resize(d, (1280, 960), interpolation=cv2.INTER_NEAREST))
frames = [(b, d) if i % 4 == 0 else big if i % 4 == 1 else synth.make_frame(W, H, 100 + i) if i % 4 == 2 else (np.zeros_like(b), np.zeros_like(d))
          for i in range(4 * world + 3)]
modes = [dict(top_k=1), dict(top_k=5, per_class=True, th_obj_dist=30.0)]
ref = fb.Handle(T, (0, 1), W, H, device=local)
ref.upload_templates(ts)
ref.upload_model_depths(crops, rects)
ok_all = True
pipe = sharded.NativeShardedPipe(ts, rank, world, depth=3, capacity=4096, device=dev)
pipe.upload_model_depths(crops, rects)
for mode in modes:
    params = fb.reco_params(**mode)
    ref.set_recognition(np.arange(ts.n_templates), params=params)
    want = [ref.recognize(fb_, fd_, K, W, H) for fb_, fd_ in frames]
    pipe.set_recognition(np.arange(ts.n_templates), params=params)
    torch.cuda.synchronize(); dist.barrier()
    got = []
    for fb_, fd_ in frames:
        if pipe.in_flight() == pipe.depth:
            got.append(pipe.collect_recognition())
        pipe.submit_recognition(fb_, fd_, K, W, H)
    while pipe.in_flight():
        got.append(pipe.collect_recognition())
    got.append(pipe.recognize(*frames[1], K, W, H))
    want.append(want[1])
    ok = len(got) == len(want)
    for f, ((rc, recs, summ), (rc_w, recs_w, summ_w)) in enumerate(zip(got, want)):
        same = rc == rc_w and summ == summ_w and recs.tobytes() == recs_w.tobytes()
        ok &= same
        if not same:
            print("rank", rank, "mode", mode, "frame", f, "MISMATCH", rc, rc_w, summ, summ_w, flush=True)
    print("rank", rank, "mode", mode, "PASS" if ok else "FAIL", "results/frame", [len(w[1]) for w in want], flush=True)
    ok_all &= ok
pipe.close()
ref.close()
t = torch.tensor([1 if ok_all else 0], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0:
    print("MULTI-GPU RECO PARITY", "PASS" if int(t.item()) else "FAIL", flush=True)
code = 0 if int(t.item()) else 1
torch.cuda.synchronize()
dist.destroy_process_group()
sys.stdout.flush(); sys.stderr.flush()
os._exit(code)                                                  # (no interpreter teardown: it frees torch tensors in arbitrary order)
