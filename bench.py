#!/usr/bin/env python
"""bench.py - the hot-path benchmark of fealess_b200 (contract: see the task statement / DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--templates n]

Workload (BASELINE.json configs[1], "C2"): LINE-MOD match-only on a synthetic 640x480 RGB-D frame against 8,000
templates (2 pyramid levels, T = {5, 8}, colour-gradient + depth-normal modalities), threshold 75 %.  A "step" is one
pass of ``Detector::match`` over one frame: front end (quantise, spread, response maps, linear memories), global
similarity of every template at the coarsest level, local refinement of the candidates, sort + duplicate pruning.

* ``value``  : template.px evals/s with the frame already resident in HBM (device-timed, CUDA events on the launching
               stream, L2 flushed between steps).  One eval = one (template, coarsest-level cell) total-similarity
               evaluation (SURVEY.md 8d): 8,000 x 1,200 = 9.6 M per frame per GPU.
* ``e2e``    : the same metric through the reference-facing C-ABI call ``fl_match`` with HOST buffers (host->device
               copy of the frame and device->host read of the match list inside the timed region).
* N > 1      : weak scaling, templates sharded (every rank holds 8,000 templates of an N x 8,000 set and sees the
               same frame), one NCCL all-gather of candidate blocks per frame, sort + unique on every rank.
* ``--impl reference``: the reference's OWN CPU implementation: oracle/_ref/libfl_ref.so = /root/reference/linemod/linemod.cpp
               compiled unmodified (oracle/build_ref.py), its real ``Detector::match`` on one host thread (the reference is
               single-threaded), OpenCV's primitives supplied by the real cv2 of the image where importable.  Without the
               prebuilt library: the C restatement under oracle/ with OpenMP over templates (``kind: port``).
* every run of our arm checks, outside the timed region, that the match list of frame 0 equals the CPU arm's list.
* ``--config C4|C5``: the strong-scaling pipeline benchmark (fixed template set sharded over the GPUs, match + exchange + ICP of
               the top-5 hypotheses + NMS, frames/s); see run_pipeline.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

import numpy as np  # noqa: E402

W, H, T = 640, 480, (5, 8)
THRESHOLD = 75.0
FEATURES_COARSE = 62            # 2 modalities x 31 features at the coarsest of 2 levels
CELLS = (W // 2 // T[1]) * (H // 2 // T[1])     # 40 x 30 = 1,200
FRONT_END_BYTES = 5 * W * H + 2 * 8 * (W * H + (W // 2) * (H // 2))   # 7,680,000 B (SURVEY 8d)
N_FRAMES = 8                    # distinct synthetic frames cycled through the steps
N_INPUT_SLOTS = 160             # device copies of them at distinct addresses: 160 x 1.536 MB = 246 MB > 126 MB L2
METRIC = "template.px evals/s (LINE-MOD match, 640x480, 8k templates/GPU)"
WORKLOAD = "C2: LINE-MOD match-only, 640x480, %d templates per GPU, L=2, T={5,8}, threshold 75"   # same string in both arms


def host_info():
    """nproc and CPU model of the box the CPU legs run on (SURVEY 8d)."""
    model = ""
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    model = ln.split(":", 1)[1].strip()
                    break
    except Exception:  # noqa: BLE001
        pass
    return {"nproc": os.cpu_count() or 1, "cpu_model": model}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p.get("sm_max_mhz", 1965.0)), "measured"
    except Exception:
        return 6650.0, 1965.0, "fallback"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region through NVML (same counters as the nvidia-smi line
    of B200_PROFILING.md, but in-process so that a timed region of tens of milliseconds still gets dozens of samples)."""

    def __init__(self, gpu_index: int, period_s: float = 0.002):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.period = period_s
        self.sm, self.reasons, self.power = [], set(), []
        self.sm_max = None
        self._stop_evt = threading.Event()
        self.err = None
        self._ready = threading.Event()

    def start_and_wait(self, timeout=5.0):
        """Start sampling and return once NVML is initialised and the first sample is in (so short timed regions are covered)."""
        self.start()
        self._ready.wait(timeout)

    def run(self):
        try:
            import pynvml as N
            N.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber the devices: map through the PCI bus id of the CUDA device
            try:
                import torch
                bus = torch.cuda.get_device_properties(self.gpu).pci_bus_id
                dom = torch.cuda.get_device_properties(self.gpu).pci_domain_id
                dev = torch.cuda.get_device_properties(self.gpu).pci_device_id
                hdl = N.nvmlDeviceGetHandleByPciBusId(("%08x:%02x:%02x.0" % (dom, bus, dev)).encode())
            except Exception:
                hdl = N.nvmlDeviceGetHandleByIndex(self.gpu)
            self.sm_max = float(N.nvmlDeviceGetMaxClockInfo(hdl, N.NVML_CLOCK_SM))
            bits = {"hw_slowdown": N.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": N.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": N.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": N.nvmlClocksEventReasonSwPowerCap}
            get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self._stop_evt.is_set():
                self.sm.append(float(N.nvmlDeviceGetClockInfo(hdl, N.NVML_CLOCK_SM)))
                r = int(get_reasons(hdl))
                for k, v in bits.items():
                    if r & v:
                        self.reasons.add(k)
                try:
                    self.power.append(N.nvmlDeviceGetPowerUsage(hdl) / 1e3)
                except Exception:
                    pass
                self._ready.set()
                time.sleep(self.period)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)
            self._ready.set()

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2.0)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
               "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None, "source": "NVML, sampled during the timed region"}
        if self.err:
            out["error"] = self.err
        return out


def oracle_quantized(frame, T_):
    """The quantised images of a frame, every level and modality, from the C oracle: templates are planted on them, so that the
    benchmark's inputs are the same whichever build of the CUDA path runs (that path's own images are bit-identical)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fl_oracle_py as F
    det = F.Detector(T_)
    if det.process(*frame) != 0:
        raise SystemExit("bench.py: the C oracle rejected the synthetic frame")
    return [det.quantized(l, m) for l in range(len(T_)) for m in range(2)]


def make_inputs(n_templates: int, seed: int = 1):
    """Frames + a template set with ~1 % planted templates.  The quantised images used for planting come from the product's
    own front end when a GPU is present (our arm) or from the CPU path (reference arm); both are bit-identical."""
    from fealess_b200 import synth
    frames = [synth.make_frame(W, H, i) for i in range(N_FRAMES)]
    return frames, synth


# ------------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: oracle/ (C restatement of the reference's CPU path)
# ------------------------------------------------------------------------------------------------------------------
def cpu_time_frames(frames, tset, n_threads: int, steps: int, warmup: int):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fl_oracle_py as F
    det = F.Detector(T)
    det.set_templates(tset)
    times = []
    last = None
    for i in range(warmup + steps):
        b, d = frames[i % len(frames)]
        t0 = time.perf_counter()
        det.process(b, d)
        m = det.match(THRESHOLD, n_threads=n_threads)
        t1 = time.perf_counter()
        if i >= warmup:
            times.append(t1 - t0)
            last = m
    return times, last


def ref_time_frames(frames, tset, steps: int, warmup: int):
    """The reference's own Detector::match (oracle/_ref) on one thread; returns (times, matches of the last frame, description)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fl_ref_py as R
    prims = "oracle/ref_shim's restated primitives"
    try:
        import cv2  # noqa: F401
        R.install_cv2_hooks()
        prims = "the image's real cv2 %s primitives (GaussianBlur, Sobel, phase, medianBlur, pyrDown, resize) through callbacks" % cv2.__version__
    except Exception:  # noqa: BLE001
        pass
    det = R.Detector(T)
    det.set_templates(tset)
    times, last = [], None
    for i in range(warmup + steps):
        b, d = frames[i % len(frames)]
        t0 = time.perf_counter()
        rc, m = det.match_full(b, d, THRESHOLD)
        t1 = time.perf_counter()
        if rc != 0:
            raise RuntimeError("reference Detector::match returned %d" % rc)
        if i >= warmup:
            times.append(t1 - t0)
            last = m
    R.remove_hooks()
    return times, last, prims


def dump_outputs(out_dir: str, **outputs) -> None:
    """What a caller receives for the last timed frame, so that two builds can be compared output for output: every field of
    every record array as out_dir/<name>_<field>.npy, a plain array as out_dir/<name>.npy, all float64 (exact for the int32
    and float32 values)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        for f in a.dtype.names or [None]:
            np.save(os.path.join(out_dir, name + ("_" + f if f else "") + ".npy"), np.ascontiguousarray(a[f] if f else a, np.float64))


def match_list_sha(m) -> str:
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(m).tobytes()).hexdigest()[:16]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fl_oracle_py as F
    import fl_ref_py as R
    frames, synth = make_inputs(args.templates)
    det = F.Detector(T)
    det.process(*frames[0])
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    tset = synth.make_templates(args.templates, W, H, T, seed=1, quantized=q, planted_fraction=0.01)
    cores_all = os.cpu_count() or 1
    steps = args.steps
    if R.available():
        times, last, prims = ref_time_frames(frames, tset, steps, min(args.warmup, 3))    # ~0.12 s per step on one thread
        kind, cores = "reference", 1
        sample = ("the reference's own Detector::match (linemod.cpp compiled unmodified, oracle/_ref) on ONE thread - its real execution "
                  "model - over %d whole frames x all %d templates; OpenCV supplied by %s" % (steps, args.templates, prims))
    else:
        times, last = cpu_time_frames(frames, tset, cores_all, steps, args.warmup)
        kind, cores = "port", cores_all
        sample = ("oracle/_ref not in this checkout: the C restatement, %d whole frames x all %d templates; front end single-threaded, "
                  "matchClass OpenMP over templates" % (steps, args.templates))
    n_matches = len(last)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, matches=last)
    tot = float(np.sum(times))
    v = args.templates * CELLS * steps / tot
    # for context: the OpenMP restatement on every host core (NOT the reference's execution model)
    pt, _ = cpu_time_frames(frames, tset, cores_all, 6, 2)
    port_all = args.templates * CELLS * len(pt) / float(np.sum(pt))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "evals/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot / steps, "ms_per_step_p50": 1e3 * float(np.median(times)),
            "ms_per_step_p95": 1e3 * float(np.percentile(times, 95)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD % args.templates, "frames_per_s": steps / tot, "matches_last_frame": n_matches},
            "cpu_baseline": {"value": v, "unit": "evals/s", "cores": cores, "kind": kind, "sample": sample, "host": host_info(),
                             "port_all_cores": {"value": port_all, "unit": "evals/s", "cores": cores_all,
                                                "note": "C restatement with OpenMP over templates on every host core - not the reference's execution model"}},
            "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import fealess_b200 as fb
    from fealess_b200 import sharded

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - fealess_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    if world > 1 and hasattr(os, "sched_setaffinity"):
        # one rank = one GPU = its own slice of the host cores: the ranks busy-wait on their streams, and 8 of them sharing
        # 16 cores with the NCCL / sampler threads otherwise delay each other by hundreds of microseconds in ~10 % of the steps
        try:
            cores = sorted(os.sched_getaffinity(0))
            lw = int(os.environ.get("LOCAL_WORLD_SIZE", world))
            per = max(1, len(cores) // lw)
            os.sched_setaffinity(0, set(cores[local * per:(local + 1) * per]) or set(cores))
        except OSError:
            pass
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    hbm_gbs, sm_max_mhz, peak_src = load_peaks()

    frames, synth = make_inputs(args.templates)
    n_total = args.templates * world                                   # weak scaling: per-GPU work fixed
    cap = 2048                                                          # candidate records per rank in the all-gather block (41 KB)
    depth = args.in_flight if args.in_flight > 0 else 4

    def make_handle():
        return fb.Handle(T, (0, 1), W, H, max_candidates=max(1 << 16, world * (cap + 1) + 16), device=local)
    q = oracle_quantized(frames[0], T)          # the inputs do not depend on the build under test
    tset = synth.make_templates(n_total, W, H, T, seed=1, quantized=q, planted_fraction=0.01)
    # `depth` frames in flight per GPU: depth handles (own stream, linear memories, candidate / result blocks, exchange buffer),
    # frames dealt round-robin, lists collected in order (fealess_b200.sharded.ShardedPipe; fl_pipe is the same schedule in C)
    pipe = sharded.ShardedPipe(make_handle, tset, rank, world, depth=depth, capacity=cap, device=dev, exchange=args.exchange)
    sm = pipe.slots[0]
    h = sm.h
    stream = sm.stream
    # inputs larger than L2: N_INPUT_SLOTS device copies of the frames at distinct addresses (160 x 1.5 MB = 246 MB > 126 MB L2),
    # visited in turn, so that no frame's bytes are L2-resident when its step starts
    d_inputs = [(torch.from_numpy(frames[j % N_FRAMES][0]).to(dev), torch.from_numpy(frames[j % N_FRAMES][1].view(np.int16)).to(dev)) for j in range(N_INPUT_SLOTS)]
    d_frames = d_inputs[:N_FRAMES]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2 (latency-mode pass)
    torch.cuda.synchronize()

    def step(i, timed):
        """latency mode: ONE frame in flight, L2 flushed before it, events around exactly its device work"""
        tb, td = d_frames[i % N_FRAMES]
        with torch.cuda.stream(stream):
            flush.zero_()                                               # L2 flush between steps, outside the timed events
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
        # enqueue the frame, record the end event right behind its last kernel, THEN let the host wait: the events bracket the
        # device work only (the synchronous call would put the host's wake-up + event-enqueue latency, ~20 us, inside them)
        whole = sm.match_device_async(tb.data_ptr(), td.data_ptr(), W, H, THRESHOLD) if world > 1 else (h.match_device_async(tb.data_ptr(), td.data_ptr(), W, H, THRESHOLD) or True)
        if whole:
            e1.record(stream)
        (sm if world > 1 else h).match_wait()
        if not whole:                                                  # NCCL exchange: the collective + merge are issued by match_wait
            e1.record(stream)
        return e0, e1

    seq = [0]

    def stream_frames(n, mark=None):
        """n more frames through the pipe without draining it; mark(slot) is called right before the first of them is enqueued"""
        for k in range(n):
            if pipe.in_flight() == depth:
                pipe.collect()
            tb, td = d_inputs[seq[0] % N_INPUT_SLOTS]
            seq[0] += 1
            if k == 0 and mark is not None:
                mark(pipe.slots[pipe.submitted % depth])
            pipe.submit_device(tb.data_ptr(), td.data_ptr(), W, H, THRESHOLD)

    def drain():
        last = None
        while pipe.in_flight():
            last = pipe.collect()
        return last

    stream_frames(max(args.warmup, 3))
    drain()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start_and_wait()                                        # NVML init takes ~10 ms: before the barrier, or every peer's first step waits for rank 0
    if world > 1:
        dist.barrier()
    launches0 = pipe.launch_count()
    import gc
    gc.collect()
    gc.disable()                                                        # no collector pauses inside the timed region
    wall0 = time.perf_counter()
    # Timed region = EXACTLY args.steps frames of a running stream.  The ranks leave the host barrier up to ~1 ms apart, so the pipe
    # is first filled with 2 x depth untimed frames (the on-device exchange re-aligns the ranks) and NOT drained; the start event
    # is recorded on the stream of the slot that receives the first timed frame, right in front of it (so it fires when that
    # slot's previous frame has finished - up to depth - 1 untimed frames are still running then and their remaining work is
    # counted: the figure errs on the slow side by < depth / steps); the end event is recorded after the host has collected the
    # last timed frame, on an idle stream.
    stream_frames(2 * depth)
    e_start = torch.cuda.Event(enable_timing=True)
    e_end = torch.cuda.Event(enable_timing=True)
    stream_frames(args.steps, mark=lambda slot: e_start.record(slot.stream))
    last = drain()
    e_end.record(last.stream)
    torch.cuda.synchronize()
    gc.enable()
    if world > 1:
        dist.barrier()
    wall1 = time.perf_counter()
    launches = pipe.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    n_matches = len(last.fetch())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, matches=last.fetch())
    dev_ms = float(e_start.elapsed_time(e_end))
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    # ---- latency mode (one frame in flight, L2 flushed before every frame, per-frame events): what a caller that needs each
    # list before it submits the next frame sees; the headline of rounds 1-2a ----
    n_lat = min(args.steps, 300)
    for i in range(3):
        step(i, False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        for i in range(2):
            step(i, False)
    gc.disable()
    evs = [step(args.warmup + i, True) for i in range(n_lat)]
    torch.cuda.synchronize()
    gc.enable()
    per_step = np.array([a.elapsed_time(b) for a, b in evs])
    if args.per_step:
        slow = np.nonzero(per_step > 3 * np.median(per_step))[0]
        sys.stderr.write("rank %d latency-mode per-frame device ms: p10 %.4f p50 %.4f p90 %.4f max %.4f mean %.4f | frames > 3x median: %s\n"
                         % (rank, *np.percentile(per_step, [10, 50, 90]), per_step.max(), per_step.mean(),
                            ", ".join("%d (%.2f ms)" % (i, per_step[i]) for i in slow[:8]) or "none"))
    lat = torch.tensor([float(per_step.sum())], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(lat, op=dist.ReduceOp.MAX)
    lat_ms = float(lat.item()) / n_lat
    # ---- correctness, outside the timed region: the match list of frame 0 must equal the CPU arm's list (every rank holds the
    # merged list; the CPU side is the C restatement over ALL n_total templates, OpenMP over templates, pinned bit for bit on
    # the reference's own code by tests/test_oracle_ref.py) ----
    for _ in range(depth):                                          # frame 0 through EVERY slot of the pipe
        pipe.submit_device(d_frames[0][0].data_ptr(), d_frames[0][1].data_ptr(), W, H, THRESHOLD)
    got_all = []
    while pipe.in_flight():
        got_all.append(pipe.collect().fetch().copy())
    got0 = got_all[0]
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fl_oracle_py as F
    odet = F.Detector(T)
    odet.set_templates(tset)
    odet.process(*frames[0])
    want0 = odet.match(THRESHOLD, n_threads=os.cpu_count() or 1)
    list_ok = all(len(g) == len(want0) and bool(np.array_equal(g, want0)) for g in got_all)
    ok_t = torch.tensor([1 if list_ok else 0], device=dev)
    if world > 1:
        dist.all_reduce(ok_t, op=dist.ReduceOp.MIN)
    if int(ok_t.item()) != 1:
        raise SystemExit("bench.py: rank %d: the match list of frame 0 (%d records) differs from the CPU arm's (%d records)" % (rank, len(got0), len(want0)))
    list_sha = match_list_sha(want0)
    evals_per_step = args.templates * world * CELLS
    # per-stage device times: a second, shorter pass with the library's own CUDA events between the stages (on its stream);
    # kept out of the headline loop because every event record costs the pipeline a few microseconds
    stage, n_stage = np.zeros(4), min(args.steps, 100)
    if world == 1:
        h.profile(True)
        for i in range(n_stage + 3):
            step(i, False)
            if i >= 3:
                stage += h.last_stage_ms()
        torch.cuda.synchronize()
        h.profile(False)
    value = evals_per_step * args.steps / (dev_ms * 1e-3)

    # ---- e2e: HOST buffers in, HOST match lists out, through the C ABI; the same stream of frames with `depth` in flight ----
    # the frames live in page-locked host memory (what a capture pipeline hands over) and are DMA'd from there
    pinned = [(torch.from_numpy(b).pin_memory().numpy(), torch.from_numpy(d.view(np.int16)).pin_memory().numpy().view(np.uint16)) for b, d in frames]
    e2e = None
    if world == 1:
        cpipe = fb.Pipe(depth, T, (0, 1), W, H, device=local)            # fl_pipe_*: the C entry points a host application calls
        cpipe.upload_templates(tset)

        def host_stream(n, src):
            m = None
            for i in range(n):
                if cpipe.in_flight() == depth:
                    rc, m = cpipe.collect(4096, copy=False)
                    assert rc == 0
                cpipe.submit(src[i % N_FRAMES][0], src[i % N_FRAMES][1], THRESHOLD)
            while cpipe.in_flight():
                rc, m = cpipe.collect(4096, copy=False)
                assert rc == 0
            return m
        host_stream(8, pinned)
        t0 = time.perf_counter()
        m = host_stream(args.steps, pinned)
        t1 = time.perf_counter()
        # the synchronous call, one frame in flight (fl_match: what the reference's Detector::match signature gives a caller)
        for i in range(3):
            h.match(pinned[i % N_FRAMES][0], pinned[i % N_FRAMES][1], THRESHOLD, capacity=4096)
        n_sync = min(args.steps, 300)
        ts0 = time.perf_counter()
        for i in range(n_sync):
            rc, m1 = h.match(pinned[i % N_FRAMES][0], pinned[i % N_FRAMES][1], THRESHOLD, capacity=4096)
        ts1 = time.perf_counter()
        # the batch entry (fl_pipe_match_batch: B frames in, B lists out, one call): B = 64 (SURVEY 8d)
        batch = [pinned[i % N_FRAMES] for i in range(64)]
        rcb, lists_b = cpipe.match_batch(batch, THRESHOLD)
        tb0 = time.perf_counter()
        rcb, lists_b = cpipe.match_batch(batch, THRESHOLD)
        tb1 = time.perf_counter()
        if rcb != 0 or any(len(lists_b[k]) != len(lists_b[k % N_FRAMES]) for k in range(64)):
            raise SystemExit("bench.py: fl_pipe_match_batch returned status %d or lists that differ between repeats of a frame" % rcb)
        host_stream(8, frames)
        n_page = min(args.steps, 200)
        tp0 = time.perf_counter()
        host_stream(n_page, frames)
        tp1 = time.perf_counter()
        cpipe.close()
        e2e = {"value": evals_per_step * args.steps / (t1 - t0), "unit": "evals/s", "h2d_bytes_per_step": W * H * 5,
               "d2h_bytes_per_step": 64 + len(m) * 20, "frames_per_s": args.steps / (t1 - t0), "frames_in_flight": depth,
               "timer": "host wall clock around a stream of fl_pipe_submit / fl_pipe_collect calls (C ABI; host frames in page-locked memory, "
                        "H2D and the read-back of every frame's match list inside)",
               "frames_per_s_one_frame_in_flight": n_sync / (ts1 - ts0), "frames_per_s_pageable_input": n_page / (tp1 - tp0),
               "frames_per_s_batch64": 64 / (tb1 - tb0), "latency_ms_one_frame": 1e3 * (ts1 - ts0) / n_sync}
    else:
        def host_stream(n):
            m = None
            for i in range(n):
                if pipe.in_flight() == depth:
                    m = pipe.collect().fetch()
                pipe.submit_host(pinned[i % N_FRAMES][0], pinned[i % N_FRAMES][1], THRESHOLD)
            while pipe.in_flight():
                m = pipe.collect().fetch()
            return m
        host_stream(2 * depth)
        torch.cuda.synchronize(); dist.barrier()
        t0 = time.perf_counter()
        m = host_stream(args.steps)
        torch.cuda.synchronize(); dist.barrier()
        t1 = time.perf_counter()
        tt = torch.tensor([t1 - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        py_fps = args.steps / float(tt.item())
        e2e = {"value": evals_per_step * py_fps, "unit": "evals/s", "h2d_bytes_per_step": W * H * 5,
               "d2h_bytes_per_step": 64 + len(m) * 20, "frames_per_s": py_fps, "frames_in_flight": depth,
               "timer": "host wall clock, max over ranks, around a stream of fl_match_shard_exchange_async / fl_match_wait / fl_match_fetch calls per rank "
                        "(host frames in page-locked memory; H2D and the read-back of every frame's merged list inside)"}
        # the same stream with the per-frame host loop inside the library: one fl_pipe per rank in template-sharded mode
        # (fl_pipe_set_exchange), ONE fl_pipe_match_batch call for all `steps` frames.  Peer-memory exchange only; on any failure the
        # Python-driven figure above stands.
        if pipe.exchange == "p2p":
            def all_ok(flag):                                          # every collective below is entered by all ranks or by none
                t_ = torch.tensor([1 if flag else 0], device=dev)
                dist.all_reduce(t_, op=dist.ReduceOp.MIN)
                return int(t_.item()) == 1
            npipe, err = None, None
            try:
                npipe = sharded.NativeShardedPipe(tset, rank, world, depth=depth, capacity=cap, device=dev, T=T, max_width=W, max_height=H)
            except Exception as e:  # noqa: BLE001
                err = "%s: %s" % (type(e).__name__, e)
            if all_ok(npipe is not None):
                batch = [pinned[i % N_FRAMES] for i in range(args.steps)]
                out_n = np.zeros(args.steps * 2048, fb.MATCH_DTYPE)          # result buffer allocated (and touched) outside the timed call
                lists_n, tn0, tn1 = None, 0.0, 1.0
                try:
                    rcw, _ = npipe.match_batch(batch[:2 * depth], THRESHOLD, capacity_per_frame=2048, out=out_n, copy=False)
                    torch.cuda.synchronize()
                except Exception as e:  # noqa: BLE001
                    rcw, err = -1, "%s: %s" % (type(e).__name__, e)
                if all_ok(rcw == 0):
                    dist.barrier()
                    try:
                        tn0 = time.perf_counter()
                        rcn, lists_n = npipe.match_batch(batch, THRESHOLD, capacity_per_frame=2048, out=out_n, copy=False)
                        tn1 = time.perf_counter()
                    except Exception as e:  # noqa: BLE001
                        rcn, err = -1, "%s: %s" % (type(e).__name__, e)
                    good = rcn == 0 and lists_n is not None and np.array_equal(lists_n[0], want0) and all(len(lists_n[k]) == len(lists_n[k % N_FRAMES]) for k in range(len(lists_n)))
                    if all_ok(good):
                        tn = torch.tensor([tn1 - tn0], dtype=torch.float64, device=dev)
                        dist.all_reduce(tn, op=dist.ReduceOp.MAX)
                        nat_fps = args.steps / float(tn.item())
                        e2e["frames_per_s_python_loop"] = py_fps
                        e2e["frames_per_s_one_batch_call"] = nat_fps
                        if nat_fps > py_fps:                                    # the headline e2e is the faster of the two host loops; both are printed
                            e2e.update({"value": evals_per_step * nat_fps, "frames_per_s": nat_fps, "d2h_bytes_per_step": 64 + len(lists_n[-1]) * 20,
                                        "timer": "host wall clock, max over ranks, around ONE fl_pipe_match_batch call per rank (fl_pipe in template-sharded mode: "
                                                 "fl_pipe_set_exchange; host frames in page-locked memory; H2D, fused match + peer-memory exchange and the "
                                                 "read-back of every frame's merged list inside)"})
                    elif err is None:
                        err = "fl_pipe_match_batch (sharded) returned status %s or a list that differs from the CPU arm's on some rank" % rcn
            if npipe is not None:
                npipe.close()
            if err:
                e2e["native_pipe_error"] = err

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (global similarity) + the HBM-bound front end ----
    roofline = None
    extra = {}
    if world == 1:
        st = stage / n_stage                                             # ms: front end, similarity, refine, sort
        sm_clk = (clocks or {}).get("sm_mhz") or sm_max_mhz
        smem_peak = 148 * 128 * sm_clk * 1e6 / 1e9                       # GB/s: 148 SMs x 128 B/clk x achieved SM clock
        alg_bytes = args.templates * CELLS * FEATURES_COARSE             # 62 B per eval (SURVEY 8d)
        ach = alg_bytes / (st[1] * 1e-3) / 1e9
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f).get("k_similarity_staged")
        except Exception:
            pass
        roofline = {"kernel": "k_similarity_staged (global similarity, all templates, coarsest level)", "bound": "smem", "achieved": ach, "peak": smem_peak, "unit": "GB/s", "frac": ach / smem_peak,
                    "traffic": traffic, "kernel_ms": float(st[1]), "timer": "CUDA events on the library's stream around the stage (counter memset + launch + kernel), mean of %d steps" % n_stage, "peak_source": "148 SM x 128 B/clk x %.0f MHz (SM clock sampled under load); "
                    "MEASURED_PEAKS.json has no shared-memory figure" % sm_clk, "algorithmic_bytes_per_launch": alg_bytes}
        fe = FRONT_END_BYTES / (st[0] * 1e-3) / 1e9
        extra["roofline_front_end"] = {"kernels": "k_front_end_wave: ONE launch (colour + depth quantisers, pyrDown, spread + response maps + linear memories of both levels, in-grid dependencies)", "bound": "hbm",
                                       "achieved": fe, "peak": hbm_gbs, "unit": "GB/s", "frac": fe / hbm_gbs, "stage_ms": float(st[0]),
                                       "algorithmic_bytes": FRONT_END_BYTES, "peak_source": peak_src + " MEASURED_PEAKS.json hbm_gbs",
                                       "note": "7.7 MB per VGA frame = 1.2 us at peak: at VGA this stage is bound by instruction issue and dependency latency (13 M warp instructions), not by bandwidth"}
        extra["stage_ms"] = {"front_end": float(st[0]), "similarity_global": float(st[1]), "refine": float(st[2]), "sort_unique_and_fetch": float(st[3])}

    # ---- CPU baseline (rank 0, N = 1 only): the C restatement, single thread = the reference's execution model ----
    cpu = None
    if world == 1 and not args.no_cpu:
        import fl_ref_py as R
        if R.available():                                       # the reference's own Detector::match on one thread (its execution model)
            n_cpu, w_cpu = 40, 4                                  # ~2.5 s of CPU work: a bounded sample of the same workload
            ct, last, prims = ref_time_frames(frames, tset, n_cpu, w_cpu)
            fi = (w_cpu + n_cpu - 1) % len(frames)               # the frame of the reference's last timed step
            if set(map(tuple, last.tolist())) != set(map(tuple, h.match(frames[fi][0], frames[fi][1], THRESHOLD)[1].tolist())):   # (its std::unique may keep non-adjacent duplicates: compare as sets)
                raise SystemExit("bench.py: the reference's own match list of frame %d differs from the GPU's" % fi)
            kind, sample = "reference", "%d whole frames (after %d warm-up), all %d templates, the reference's own Detector::match (oracle/_ref) on one thread; OpenCV = %s" % (n_cpu, w_cpu, args.templates, prims)
        else:
            ct, _ = cpu_time_frames(frames, tset, 1, 40, 4)
            kind, sample = "port", "40 whole frames (after 4 warm-up) of the same workload, all %d templates, single thread (oracle/_ref not in this checkout)" % args.templates
        cv = args.templates * CELLS * len(ct) / float(np.sum(ct))
        cpu = {"value": cv, "unit": "evals/s", "cores": 1, "kind": kind, "frames_per_s": len(ct) / float(np.sum(ct)), "ms_per_frame_p50": 1e3 * float(np.median(ct)),
               "ms_per_frame_p95": 1e3 * float(np.percentile(ct, 95)), "sample": sample, "host": host_info()}

    # ---- ICP (BASELINE configs[2], C3): 256 hypotheses x ~10k points, reported beside the headline ----
    icp = None
    if world == 1 and not args.no_icp:
        icp = bench_icp(h, synth, cpu=not args.no_cpu)

    line = {"metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "latency_mode": {"what": "ONE frame in flight, L2 flushed (256 MB write) before every frame, CUDA events around each frame's device work; %d frames" % n_lat,
                             "ms_per_frame": lat_ms, "ms_per_frame_p50": float(np.median(per_step)), "ms_per_frame_p90": float(np.percentile(per_step, 90)),
                             "ms_per_frame_p95": float(np.percentile(per_step, 95)), "value": evals_per_step / (lat_ms * 1e-3), "unit": "evals/s"},
            "config": {"workload": WORKLOAD % args.templates, "templates_total": n_total, "frames_in_flight": depth,
                       "l2": "inputs larger than L2: the steps walk over %d device copies of the frames at distinct addresses (%.0f MB > 126 MB L2); "
                             "no flush, the stream of frames is not interrupted" % (N_INPUT_SLOTS, N_INPUT_SLOTS * W * H * 5 / 1e6),
                       "timed_region": "exactly `steps` frames of a running stream with `frames_in_flight` frames in flight per GPU; start event in front of the "
                                       "first timed frame on its stream, end event after the last list has been collected; max over ranks",
                       "frames_per_s": args.steps / (dev_ms * 1e-3),
                       "full_resolution_equivalent_evals_per_s": value * (W * H) / CELLS,     # N_templates x W0 x H0 per frame (SURVEY 8d), NOT the headline unit
                       "matches_last_frame": n_matches, "match_list_frame0": {"records": int(len(want0)), "sha256_16": list_sha,
                                                                              "equals_cpu_arm": True}, "parallelism": ("template-sharded x%d, candidate exchange: %s" % (world, "peer-memory push fused into the sort kernel (NVLink)" if sm.exchange == "p2p" else "1 NCCL all-gather/frame")) if world > 1 else "single GPU"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "wall_s_timed_region": wall1 - wall0}
    line.update(extra)
    if icp:
        line["icp"] = icp
    if world == 1 and not args.no_icp:
        try:                                                    # a side measurement: it must never cost the headline line
            line["recognition"] = bench_recognition(synth, frames, q, cpu=not args.no_cpu)
            # BASELINE.json's first metric, "frames/s (LINE-MOD match+ICP, 640x480)", on configs[0] (C1), host buffers in, poses out
            line["frames_per_s_match_icp_640x480"] = {"value": line["recognition"]["frames_per_s_stream"], "unit": "frames/s",
                                                      "frames_in_flight": line["recognition"]["frames_in_flight"],
                                                      "one_frame_in_flight": line["recognition"]["frames_per_s"],
                                                      "cpu_baseline": (line["recognition"].get("cpu_baseline") or {}).get("frames_per_s"),
                                                      "workload": line["recognition"]["workload"],
                                                      "timer": "host wall clock; host frames in, poses out; `frames_in_flight` host threads, each calling the "
                                                               "synchronous ObjRecoLmICP.Recognition mirror on its own instance"}
        except Exception as e:  # noqa: BLE001
            line["recognition"] = {"error": "%s: %s" % (type(e).__name__, e)}
    if world == 1:
        try:                                                    # the front end where its HBM roofline means something: 1920x1080 (SURVEY 8d)
            Wf, Hf, Tf = 1920, 1080, (5, 5, 5, 5)                 # the C5 geometry (T = {5, 8} does not divide 540)
            hf = fb.Handle(Tf, (0, 1), Wf, Hf, device=local)
            hf.upload_templates(synth.make_templates(0, Wf, Hf, Tf))
            fb_, fd_ = synth.make_frame(Wf, Hf, 0)
            tbf, tdf = torch.from_numpy(fb_).to(dev), torch.from_numpy(fd_.view(np.int16)).to(dev)
            hf.profile(True)
            acc, nfe = 0.0, 30
            for i in range(nfe + 3):
                flush.zero_()
                torch.cuda.synchronize()
                hf.match_device(tbf.data_ptr(), tdf.data_ptr(), Wf, Hf, THRESHOLD)
                if i >= 3:
                    acc += float(hf.last_stage_ms()[0])
            hf.profile(False)
            fe_bytes = 5 * Wf * Hf + 2 * 8 * sum((Wf >> l) * (Hf >> l) for l in range(len(Tf)))
            fe_ms = acc / nfe
            line["roofline_front_end_1080p"] = {"kernels": "k_front_end_wave, one launch, 1920x1080, L=4, T={5,5,5,5} (the C5 geometry)", "bound": "hbm", "algorithmic_bytes": fe_bytes,
                                                "stage_ms": fe_ms, "achieved": fe_bytes / (fe_ms * 1e-3) / 1e9, "peak": hbm_gbs, "unit": "GB/s",
                                                "frac": fe_bytes / (fe_ms * 1e-3) / 1e9 / hbm_gbs, "l2": "flushed before every frame",
                                                "timer": "the library's CUDA events around the stage, mean of %d frames" % nfe}
            hf.close()
        except Exception as e:  # noqa: BLE001
            line["roofline_front_end_1080p"] = {"error": "%s: %s" % (type(e).__name__, e)}
    if world == 1 and not args.no_icp:
        try:                                                    # SURVEY 8f rank 4: template training, one view -> one template pyramid
            yy, xx = np.mgrid[0:H, 0:W]
            tmask = ((((xx - 320) / 110.0) ** 2 + ((yy - 240) / 80.0) ** 2) <= 1.0).astype(np.uint8) * 255
            ht = fb.Handle(T, (0, 1), W, H, device=local)
            rct, hdr_t, ft_t, bb_t = ht.add_template(frames[0][0], frames[0][1], tmask)
            n_views = 20
            tt0 = time.perf_counter()
            for i in range(n_views):
                rct, hdr_t, ft_t, bb_t = ht.add_template(frames[0][0], frames[0][1], tmask)
            tt1 = time.perf_counter()
            ht.close()
            tr = {"workload": "Detector::addTemplate on one 640x480 RGB-D view with an elliptic object mask (63 + 63 + 31 + 31 features)",
                  "views_per_s": n_views / (tt1 - tt0), "ms_per_view": 1e3 * (tt1 - tt0) / n_views, "status": int(rct), "features": int(len(ft_t)),
                  "timer": "host wall clock around fl_add_template (upload, front end, magnitude / erosion / distance-transform kernels, candidate "
                           "read-back, host-side stable sort + scattered selection)"}
            if not args.no_cpu:
                import fl_ref_py as R
                if R.available():
                    rdet = R.Detector(T)
                    R.add_template(rdet, frames[0][0], frames[0][1], tmask)
                    tc0 = time.perf_counter()
                    for i in range(3):
                        rrc, rhdr, rft, rbb = R.add_template(rdet, frames[0][0], frames[0][1], tmask)
                    tc1 = time.perf_counter()
                    tr["cpu_baseline"] = {"views_per_s": 3 / (tc1 - tc0), "cores": 1, "kind": "reference",
                                          "sample": "3 views through the reference's own addTemplate (oracle/_ref)",
                                          "identical_result": bool(rrc >= 0 and rct == 0 and np.array_equal(rhdr, hdr_t) and np.array_equal(rft, ft_t) and np.array_equal(rbb, bb_t))}
                else:                                                    # oracle/_ref not in this checkout: the C restatement
                    sys.path.insert(0, os.path.join(ROOT, "oracle"))
                    import fl_oracle_py as Fo
                    odt = Fo.Detector(T)
                    tc0 = time.perf_counter()
                    for i in range(3):
                        orc, ohdr, oft, obb = Fo.add_template(odt, frames[0][0], frames[0][1], tmask)
                    tc1 = time.perf_counter()
                    tr["cpu_baseline"] = {"views_per_s": 3 / (tc1 - tc0), "cores": 1, "kind": "port", "sample": "3 views through flo_add_template (oracle/fl_oracle.c)",
                                          "identical_result": bool(orc == 0 and rct == 0 and np.array_equal(ohdr, hdr_t) and np.array_equal(oft, ft_t) and np.array_equal(obb, bb_t))}
            line["training"] = tr
        except Exception as e:  # noqa: BLE001
            line["training"] = {"error": "%s: %s" % (type(e).__name__, e)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
# strong-scaling pipeline benchmark: BASELINE.json configs[3] (C4) and configs[4] (C5)
# ------------------------------------------------------------------------------------------------------------------
PIPELINES = {
    "C4": dict(W=1280, H=720, T=(5, 8), classes=15, per_class=2000,
               desc="C4: full obj_reco_lmicp pipeline at 1280x720, 15 objects x 2,000 templates (fixed set, sharded over the GPUs), L=2, T={5,8}: "
                    "match + candidate exchange + ICP of the top-5 hypotheses + NMS"),
    "C5": dict(W=1920, H=1080, T=(5, 5, 5, 5), classes=16, per_class=2000,
               desc="C5: stress, 1920x1080, 32,000 templates x 4 pyramid levels (fixed set, sharded over the GPUs), T={5,5,5,5}: "
                    "match + candidate exchange + ICP of the top-5 hypotheses + NMS"),
}
TOP_K = 5


def run_pipeline(args):
    """Strong scaling: ONE fixed template set dealt over the ranks (gid % world), every rank sees the frame.  A step = one frame
    through front end + matchClass on the local shard, the candidate exchange + merge (peer-memory push fused into the sort
    kernel, or one NCCL all-gather), ICP of the top-5 matches dealt over the ranks (k % world) with one all-gather of the pose
    records, and nonMaximumSuppression on every rank.  Timed on the device (CUDA events on the handle's stream bracket the whole
    frame, host decisions included), max over ranks; frame resident in HBM, template depth crops resident (AddObj time)."""
    import torch
    import torch.distributed as dist
    import fealess_b200 as fb
    from fealess_b200 import sharded, synth

    cfg = PIPELINES[args.config]
    Wp, Hp, Tp = cfg["W"], cfg["H"], cfg["T"]
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - fealess_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_total = cfg["classes"] * cfg["per_class"]
    L = len(Tp)
    frames = [synth.make_frame(Wp, Hp, i) for i in range(2)]
    cap = 4096
    h = fb.Handle(Tp, (0, 1), Wp, Hp, max_candidates=max(1 << 16, world * (cap + 1) + 16), device=local)
    q = oracle_quantized(frames[0], Tp)
    tset = synth.make_templates(n_total, Wp, Hp, Tp, n_classes=cfg["classes"], seed=1, quantized=q, planted_fraction=0.004)
    sm = sharded.ShardedMatcher(h, tset, rank, world, capacity=cap, device=dev, exchange=args.exchange)
    stream = sm.stream
    # the templates' rendered depth crops stay on the device (AddObj time); the synthetic stand-in for a rendered view is frame 0's depth
    hdr0 = tset.headers.reshape(n_total, L * 2, 7)[:, 0, :]
    rects_model = np.stack([hdr0[:, 2], hdr0[:, 3], hdr0[:, 0], hdr0[:, 1]], axis=1).astype(np.int32)
    h.upload_model_depths([frames[0][1]] * n_total, rects_model)
    class_first = np.zeros(cfg["classes"], np.int64)
    for c in range(cfg["classes"]):
        class_first[c] = int(np.argmax(tset.class_of == c))
    d_frames = [(torch.from_numpy(b).to(dev), torch.from_numpy(d.view(np.int16)).to(dev)) for b, d in frames]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    K = (608.0 * Wp / 640, 608.0 * Wp / 640, Wp / 2.0, Hp / 2.0)
    # throughput mode: `depth` frames in flight per GPU, one host thread + handle + exchange buffer each (slot 0 is the handle above)
    # default: 8 frames in flight, but not more host threads than this rank's share of the cores (measured at N = 8 on a 32-core box:
    # 4 spinning threads per rank 812 frames/s, 8 sleeping threads per rank 363)
    cores_all = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    depth = args.in_flight if args.in_flight > 0 else max(2, min(8, cores_all // int(os.environ.get("LOCAL_WORLD_SIZE", world))))
    slots = [(h, sm)]
    for _ in range(depth - 1):
        hk = fb.Handle(Tp, (0, 1), Wp, Hp, max_candidates=max(1 << 16, world * (cap + 1) + 16), device=local)
        smk = sharded.ShardedMatcher(hk, tset, rank, world, capacity=cap, device=dev, exchange=args.exchange)
        hk.upload_model_depths([frames[0][1]] * n_total, rects_model)
        slots.append((hk, smk))
    if world > 1 and any(s_[1].exchange != "p2p" for s_ in slots):
        slots = slots[:1]                                              # the NCCL exchange is issued from one host thread only
    depth = len(slots)
    # more waiting host threads than cores (8 ranks x 8 frames in flight on a 16-core box): sleep on the GPU's interrupt instead of spinning
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    blocking = depth * int(os.environ.get("LOCAL_WORLD_SIZE", world)) > cores
    if blocking:
        for hk, _ in slots:
            hk.set_blocking_wait(True)
    n_in = max(2, int(np.ceil(150e6 / (Wp * Hp * 5))))                 # inputs larger than L2: device copies of the frames at distinct addresses
    d_inputs = [(d_frames[j % 2][0].clone(), d_frames[j % 2][1].clone()) for j in range(n_in)]
    torch.cuda.synchronize()
    stamps = np.zeros(4)

    def refine_top(matches, d_depth_ptr):
        top = matches[:TOP_K]
        n = len(top)
        if n == 0:
            return np.zeros(0, fb.ICP_RESULT_DTYPE), np.zeros(0, np.int32)
        gidx = (class_first[top["class_idx"]] + top["template_id"]).astype(np.int64)
        rr = np.stack([top["x"], top["y"], rects_model[gidx, 2], rects_model[gidx, 3]], axis=1).astype(np.int32)
        P = tset.pose13[gidx][:, :12].reshape(n, 3, 4)
        Rm, tm = np.ascontiguousarray(P[:, :, :3]), np.ascontiguousarray(P[:, :, 3])

        def mine(idx):
            return h.detection_batch_resident_device(d_depth_ptr, Wp, Hp, K, gidx[idx].astype(np.int32), rr[idx], Rm[idx], tm[idx])
        res = sharded.refine_sharded(n, mine, rank, world, device=dev)
        ok = np.nonzero(res["status"] == 0)[0]
        keep = h.nms(res["T"][ok], res["n_points"][ok], res["dist_mean"][ok], 30.0) if len(ok) else np.zeros(0, np.int32)
        return res, ok[keep] if len(ok) else keep

    def step(i, timed):
        tb, td = d_frames[i % len(d_frames)]
        with torch.cuda.stream(stream):
            flush.zero_()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); em = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
        t0 = time.perf_counter()
        sm.match_device(tb.data_ptr(), td.data_ptr(), Wp, Hp, THRESHOLD)
        with torch.cuda.stream(stream):
            em.record(stream)                                         # the merged match list is complete on this rank
        m = sm.fetch()
        t1 = time.perf_counter()
        res, keep = refine_top(m, td.data_ptr())
        t2 = time.perf_counter()
        with torch.cuda.stream(stream):
            e1.record(stream)
        if timed:
            stamps[0] += t1 - t0; stamps[1] += t2 - t1; stamps[2] += 1
        return e0, e1, m, res, keep, em

    for i in range(max(args.warmup, 3)):
        step(i, False)
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start_and_wait()
    if world > 1:
        dist.barrier()
    launches0 = h.launch_count()
    evs = []
    for i in range(args.steps):
        evs.append(step(i, True))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches = h.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    per_step = np.array([a.elapsed_time(b) for a, b, *_ in evs])
    match_ms = float(np.sum([ev[0].elapsed_time(ev[5]) for ev in evs]))
    t = torch.tensor([float(per_step.sum()), match_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, match_ms = float(t[0].item()), float(t[1].item())
    # ---- throughput mode: `depth` frames in flight per GPU.  Host thread k of every rank owns slot k and takes frames k, k + depth,
    # ...: front end + matchClass on the shard, peer-memory exchange, then ICP of ALL top-5 hypotheses and NMS on this rank (a
    # hypothesis is latency-, not throughput-bound, so sharding hypotheses buys nothing once frames overlap; no second collective).
    # The ICP of frame i (5 CTAs, milliseconds) runs beside the match stages of the following frames. ----
    import threading

    def refine_local(hk, matches, d_depth_ptr):
        top = matches[:TOP_K]
        n = len(top)
        if n == 0:
            return np.zeros(0, fb.ICP_RESULT_DTYPE), np.zeros(0, np.int32)
        gidx = (class_first[top["class_idx"]] + top["template_id"]).astype(np.int64)
        rr = np.stack([top["x"], top["y"], rects_model[gidx, 2], rects_model[gidx, 3]], axis=1).astype(np.int32)
        P = tset.pose13[gidx][:, :12].reshape(n, 3, 4)
        res = hk.detection_batch_resident_device(d_depth_ptr, Wp, Hp, K, gidx.astype(np.int32), rr, np.ascontiguousarray(P[:, :, :3]), np.ascontiguousarray(P[:, :, 3]))
        ok = np.nonzero(res["status"] == 0)[0]
        keep = hk.nms(res["T"][ok], res["n_points"][ok], res["dist_mean"][ok], 30.0) if len(ok) else np.zeros(0, np.int32)
        return res, ok[keep] if len(ok) else keep

    last_of = [None] * depth
    errors = []

    def worker(k, first, n_frames, host_frames=None):
        try:
            torch.cuda.set_device(local)
            hk, smk = slots[k]
            for i in range(first + k, first + n_frames, depth):
                if host_frames is not None:
                    pb, pd = host_frames[i % len(host_frames)]
                    smk.match_host_async(pb, pd, THRESHOLD)
                    smk.match_wait()
                    ref_ptr = None
                else:
                    tb, td = d_inputs[i % n_in]
                    smk.match_device(tb.data_ptr(), td.data_ptr(), Wp, Hp, THRESHOLD)
                    ref_ptr = td.data_ptr()
                m = smk.fetch()
                if ref_ptr is None:                                    # the depth frame fl_match*_async left on the device
                    top = m[:TOP_K]
                    if len(top):
                        gidx = (class_first[top["class_idx"]] + top["template_id"]).astype(np.int64)
                        rr = np.stack([top["x"], top["y"], rects_model[gidx, 2], rects_model[gidx, 3]], axis=1).astype(np.int32)
                        P = tset.pose13[gidx][:, :12].reshape(len(top), 3, 4)
                        res = hk.detection_batch_resident(None, K, gidx.astype(np.int32), rr, np.ascontiguousarray(P[:, :, :3]), np.ascontiguousarray(P[:, :, 3]), frame_size=(Wp, Hp))
                        ok = np.nonzero(res["status"] == 0)[0]
                        keep = hk.nms(res["T"][ok], res["n_points"][ok], res["dist_mean"][ok], 30.0) if len(ok) else np.zeros(0, np.int32)
                        last_of[k] = (m, res, ok[keep] if len(ok) else keep)
                else:
                    res, keep = refine_local(hk, m, ref_ptr)
                    last_of[k] = (m, res, keep)
        except Exception as e:  # noqa: BLE001
            errors.append("slot %d: %s: %s" % (k, type(e).__name__, e))

    def run_threads(first, n_frames, host_frames=None):
        ths = [threading.Thread(target=worker, args=(k, first, n_frames, host_frames)) for k in range(depth)]
        for t_ in ths:
            t_.start()
        for t_ in ths:
            t_.join()
        if errors:
            raise SystemExit("bench.py: rank %d: %s" % (rank, "; ".join(errors)))

    # first use of every slot from the main thread, in the same order on every rank: workspaces that grow on first use (a cudaMalloc /
    # cudaFree synchronises the whole device; with another slot's exchange kernel waiting for the peer that would stall both ranks)
    for k in range(depth):
        hk, smk = slots[k]
        for f in range(2):
            smk.match_device(d_frames[f][0].data_ptr(), d_frames[f][1].data_ptr(), Wp, Hp, THRESHOLD)
            refine_local(hk, smk.fetch(), d_frames[f][1].data_ptr())
        hk.sync()
    n_tp = args.steps
    run_threads(0, 2 * depth)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches_tp0 = sum(s_[0].launch_count() for s_ in slots)
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record()
    tw0 = time.perf_counter()
    run_threads(2 * depth, n_tp)
    torch.cuda.synchronize()
    ev1.record(); ev1.synchronize()
    timed_last = last_of[(n_tp - 1) % depth]                         # the slot that took the last timed frame, 2 * depth + n_tp - 1
    tw1 = time.perf_counter()
    launches_tp = sum(s_[0].launch_count() for s_ in slots) - launches_tp0
    tp = torch.tensor([float(ev0.elapsed_time(ev1))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tp, op=dist.ReduceOp.MAX)
    tp_ms = float(tp.item())
    # every slot's last frame against slot 0's result for the same frame content (frames alternate between two images)
    # ---- correctness outside the timed region: merged list of frame 0 == the CPU arm's list over ALL templates ----
    _, _, got0, res0, keep0, _ = step(0, False)
    for k in range(depth):
        hk, smk = slots[k]
        smk.match_device(d_frames[0][0].data_ptr(), d_frames[0][1].data_ptr(), Wp, Hp, THRESHOLD)
        mk = smk.fetch()
        rk, kk = refine_local(hk, mk, d_frames[0][1].data_ptr())
        if not (np.array_equal(mk, got0) and np.array_equal(kk, keep0) and np.array_equal(rk["T"], res0["T"]) and np.array_equal(rk["R"], res0["R"])):
            raise SystemExit("bench.py: rank %d: slot %d's frame-0 result differs from slot 0's" % (rank, k))
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fl_oracle_py as F
    odet = F.Detector(Tp)
    odet.set_templates(tset)
    odet.process(*frames[0])
    want0 = odet.match(THRESHOLD, n_threads=os.cpu_count() or 1)
    ok_t = torch.tensor([1 if (len(got0) == len(want0) and np.array_equal(got0, want0)) else 0], device=dev)
    if world > 1:
        dist.all_reduce(ok_t, op=dist.ReduceOp.MIN)
    if int(ok_t.item()) != 1:
        raise SystemExit("bench.py: rank %d: merged match list of frame 0 (%d) differs from the CPU arm's (%d)" % (rank, len(got0), len(want0)))
    # ---- e2e: every frame starts in page-locked host memory, the poses end on the host; same threads, same frames in flight ----
    pin = [(torch.from_numpy(b).pin_memory().numpy(), torch.from_numpy(d.view(np.int16)).pin_memory().numpy().view(np.uint16)) for b, d in frames]
    n_e2e = n_tp
    run_threads(0, 2 * depth, pin)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    w0 = time.perf_counter()
    run_threads(2 * depth, n_e2e, pin)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    tt = torch.tensor([time.perf_counter() - w0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    m = last_of[0][0] if last_of[0] is not None else got0
    if args.dump_outputs and rank == 0:
        m_last, res_last, keep_last = timed_last
        dump_outputs(args.dump_outputs, matches=m_last, icp=res_last, nms_keep=keep_last)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    fps = n_tp / (tp_ms * 1e-3)
    lat_fps = args.steps / (dev_ms * 1e-3)
    cpu = None
    if world == 1 and not args.no_cpu:                                   # one whole frame on one thread: the reference's own code when oracle/_ref is there
        import fl_ref_py as R
        use_ref = R.available()
        t0 = time.perf_counter()
        if use_ref:
            try:
                import cv2  # noqa: F401
                R.install_cv2_hooks()
            except Exception:  # noqa: BLE001
                pass
            rd = R.Detector(Tp)
            rd.set_templates(tset)
            t0 = time.perf_counter()
            rc, ms = rd.match_full(frames[0][0], frames[0][1], THRESHOLD)
        else:
            odet.process(*frames[0]); ms = odet.match(THRESHOLD)
        for mm in ms[:TOP_K]:
            g = int(class_first[int(mm["class_idx"])] + int(mm["template_id"]))
            P = tset.pose13[g][:12].reshape(3, 4)
            (R if use_ref else F).detection(frames[0][1], frames[0][1], K, tuple(int(v) for v in rects_model[g]),
                                            (int(mm["x"]), int(mm["y"]), int(rects_model[g][2]), int(rects_model[g][3])), r_match=P[:, :3], t_match=P[:, 3])
        ct = time.perf_counter() - t0
        if use_ref:
            R.remove_hooks()
        cpu = {"value": 1.0 / ct, "unit": "frames/s", "cores": 1, "kind": "reference" if use_ref else "port",
               "sample": "ONE whole frame on one thread: %s over all %d templates + %d x detection()" % ("the reference's own Detector::match (oracle/_ref)" if use_ref else "the C restatement", n_total, min(TOP_K, len(ms)))}
    cells_c = ((Wp >> (L - 1)) // Tp[-1]) * ((Hp >> (L - 1)) // Tp[-1])
    line = {"metric": "frames/s (LINE-MOD match + top-%d ICP + NMS, %dx%d, %d templates sharded over the GPUs)" % (TOP_K, Wp, Hp, n_total),
            "value": fps, "unit": "frames/s", "n_gpus": world, "steps": n_tp, "warmup": 2 * depth, "ms_per_step": tp_ms / n_tp,
            "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8 (match) / f32 (ICP)", "data": "synthetic",
            "latency_mode": {"what": "ONE frame in flight: match + exchange, then the top-%d hypotheses dealt over the ranks (k %% world) with one all-gather of the pose records, NMS; "
                                     "L2 flushed before every frame; CUDA events around each frame, max over ranks; %d frames" % (TOP_K, args.steps),
                             "frames_per_s": lat_fps, "ms_per_frame": dev_ms / args.steps, "ms_per_frame_p50": float(np.median(per_step)), "ms_per_frame_p95": float(np.percentile(per_step, 95)),
                             "match_exchange_ms_per_frame": match_ms / args.steps, "icp_nms_ms_per_frame": (dev_ms - match_ms) / args.steps,
                             "limiter": "ICP of the top-%d hypotheses: a hypothesis is three serial fp32 sums per iteration over its 15k..40k paired points (exactness), i.e. milliseconds for "
                                        "100..200-pixel templates; it does not shrink with more GPUs once every hypothesis has its own CTA" % TOP_K,
                             "host_wall_ms_per_frame_rank0": {"match_exchange_fetch": 1e3 * stamps[0] / max(stamps[2], 1), "icp_gather_nms": 1e3 * stamps[1] / max(stamps[2], 1)}},
            "config": {"workload": cfg["desc"], "templates_total": n_total, "templates_per_gpu": sm.n_local, "frames_in_flight": depth,
                       "host_wait": "blocking (cudaEventBlockingSync): %d waiting threads on %d cores" % (depth * int(os.environ.get("LOCAL_WORLD_SIZE", world)), cores) if blocking else "spinning",
                       "l2": "inputs larger than L2: %d device copies of the frames at distinct addresses (%.0f MB); no flush, the stream is not interrupted" % (n_in, n_in * Wp * Hp * 5 / 1e6),
                       "timed_region": "`steps` frames dealt over `frames_in_flight` host threads per rank (one handle, stream and exchange buffer each), between two device-wide "
                                       "synchronisations; CUDA events on the default stream around it, max over ranks (wall clock on rank 0: %.3f s)" % (tw1 - tw0),
                       "evals_per_s": n_total * cells_c * fps,
                       "matches_frame0": int(len(got0)), "poses_frame0": int(len(keep0)), "match_list_frame0_equals_cpu_arm": True, "all_slots_equal_on_frame0": True,
                       "parallelism": ("template-sharded x%d (gid %% world), exchange: %s; every rank refines the top-%d of its merged list" % (world, sm.exchange, TOP_K)) if world > 1 else "single GPU",
                       "limiter": "throughput mode: the match stage (front end replicated on every rank + 1/N of the templates) and the host threads' per-frame calls; "
                                  "the ICP's latency is hidden behind the following frames"},
            "clocks": clocks, "gpu_launches": int(launches_tp),
            "e2e": {"value": n_e2e / float(tt.item()), "unit": "frames/s", "h2d_bytes_per_step": Wp * Hp * 5, "d2h_bytes_per_step": 64 + 20 * int(len(m)) + 68 * TOP_K,
                    "frames_in_flight": depth, "timer": "host wall clock, max over ranks; every frame from page-locked host memory (fl_match*_async), poses to the host"},
            "roofline": None, "cpu_baseline": cpu}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def bench_recognition(synth, frames, q, cpu: bool = True, n_templates: int = 2000, top_k: int = 5, n_timed: int = 100, in_flight: int = 8):
    """C1 (BASELINE configs[0]): the reference's whole ``Recognition`` call - PrepareInputData, match at 75 %, ICP of the top-5
    hypotheses - on a 640x480 frame with 1 object x 2,000 templates, through the product API mirror (fealess_b200.reco), host
    buffers in, poses out.  The templates are planted on frame 0, so frame 0 is the frame every timed call processes (each call
    runs match + 5 ICPs); the 1280x960 variant sends the pixel-doubled frame and rescales it on the device."""
    import fealess_b200 as fb
    from fealess_b200 import reco
    b, d = frames[0]
    tset = synth.make_templates(n_templates, W, H, T, n_classes=1, seed=7, quantized=q, planted_fraction=0.01)
    det = fb.Detector()
    det.add_template_set(tset)
    r = reco.ObjRecoLmICP()
    r.add_detector(det, {(None, tid): d for tid in range(n_templates)})       # synthetic rendered depth: the frame's own depth for every template
    K = dict(fx=608.0, fy=608.0, cx=320.0, cy=240.0, width=W, height=H)
    big_b, big_d = np.repeat(np.repeat(b, 2, 0), 2, 1), np.repeat(np.repeat(d, 2, 0), 2, 1)
    Kbig = dict(K, width=2 * W, height=2 * H)
    out = {}
    for tag, (fb_, fd_, Kd) in (("", (b, d, K)), ("_1280x960_input", (big_b, big_d, Kbig))):
        for _ in range(5):
            rc, res = r.Recognition(fb_, fd_, Kd, top_k=top_k)
        if rc != 0 or not res:
            raise RuntimeError("Recognition benchmark frame produced no pose (rc %d)" % rc)
        t0 = time.perf_counter()
        for _ in range(n_timed):
            rc, res = r.Recognition(fb_, fd_, Kd, top_k=top_k)
        dt = (time.perf_counter() - t0) / n_timed
        out["frames_per_s" + tag] = 1.0 / dt
        out["ms_per_frame" + tag] = 1e3 * dt
        out["poses_per_frame" + tag] = len(res)
    # a stream of frames: `in_flight` instances of the mirror (own detector handle, stream, ICP workspace), one host thread each -
    # the ICP of one frame (5 CTAs, latency-bound serial sums) runs beside the match stages and ICPs of the other frames
    import threading
    recos = [r]
    for _ in range(in_flight - 1):
        dk = fb.Detector()
        dk.add_template_set(tset)
        rk = reco.ObjRecoLmICP()
        rk.add_detector(dk, {(None, tid): d for tid in range(n_templates)})
        recos.append(rk)
    bad = []

    def stream(rk, n):
        for _ in range(n):
            rc_, res_ = rk.Recognition(b, d, K, top_k=top_k)
            if rc_ != 0 or len(res_) != len(res0):
                bad.append((rc_, len(res_)))
    rc, res0 = r.Recognition(b, d, K, top_k=top_k)
    for n_each in (5, max(n_timed // 2, 20)):                      # warm-up round, timed round
        ths = [threading.Thread(target=stream, args=(rk, n_each)) for rk in recos]
        t0 = time.perf_counter()
        for t_ in ths:
            t_.start()
        for t_ in ths:
            t_.join()
        dt = time.perf_counter() - t0
    if bad:
        raise RuntimeError("Recognition stream: %d calls returned another result than the single-threaded call: %s" % (len(bad), bad[:3]))
    out["frames_per_s_stream"] = in_flight * n_each / dt
    out["frames_in_flight"] = in_flight
    out.update({"workload": "C1: Recognition (match at 75 %% + ICP of the top-%d matches) on one 640x480 RGB-D frame, 1 object x %d templates, L=2, T={5,8}" % (top_k, n_templates),
                "icp_path": r.last_icp_path,
                "timer": "host wall clock around ObjRecoLmICP.Recognition (H2D of the frame, 3 match launches, 2 ICP launches, poses back), mean of %d calls" % n_timed})
    if cpu:                                                    # the same call on one CPU thread, 3 frames: the reference's own code when oracle/_ref is there
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import fl_oracle_py as F
        import fl_ref_py as R
        use_ref = R.available()
        Kc = (608.0, 608.0, 320.0, 240.0)
        if use_ref:
            try:
                import cv2  # noqa: F401
                R.install_cv2_hooks()
            except Exception:  # noqa: BLE001
                pass
            odet = R.Detector(T)
        else:
            odet = F.Detector(T)
        odet.set_templates(tset)
        t0 = time.perf_counter()
        for _ in range(3):
            if use_ref:
                rc, ms = odet.match_full(b, d, THRESHOLD)          # Detector::match (linemod.cpp:1356-1441)
            else:
                odet.process(b, d)
                ms = odet.match(THRESHOLD)
            for m in ms[:top_k]:
                hdr, _f = tset.template(int(m["template_id"]), 0, 0)
                P = tset.pose13[int(m["template_id"])][:12].reshape(3, 4)
                (R if use_ref else F).detection(d, d, Kc, (int(hdr[2]), int(hdr[3]), int(hdr[0]), int(hdr[1])), (int(m["x"]), int(m["y"]), int(hdr[0]), int(hdr[1])),
                                                r_match=P[:, :3], t_match=P[:, 3])
        ct = (time.perf_counter() - t0) / 3
        if use_ref:
            R.remove_hooks()
        out["cpu_baseline"] = {"frames_per_s": 1.0 / ct, "cores": 1, "kind": "reference" if use_ref else "port",
                               "sample": "3 whole frames on one thread: %s over %d templates + %d x detection() each"
                                         % ("the reference's own Detector::match (oracle/_ref, cv2 primitives)" if use_ref else "the C restatement's front end + matchClass", n_templates, min(top_k, len(ms)))}
    return out


def make_icp_workload(synth, n_hyp: int = 256, crop: int = 104):
    """C3: one 640x480 reference depth frame tiled with 24 moved surfaces, n_hyp hypotheses whose 100x100-pixel model crops
    (~10k points each) sit on those tiles (hypothesis i uses tile i % 24 with its own initial pose)."""
    nx, ny = W // crop, H // crop
    ref = np.zeros((H, W), np.uint16)
    tiles = []
    for k in range(nx * ny):
        x0, y0 = (k % nx) * crop + 2, (k // nx) * crop + 2
        md, rf, rm, rr, p = synth.make_icp_pair(W, H, seed=100 + k, max_rot_deg=6, max_shift_mm=8, rect_wh=(crop - 4, crop - 4), rect_xy=(x0, y0))
        rr = (x0, y0, crop - 4, crop - 4)                              # pixel-aligned crops, like Recognition aligns a match
        ref[y0:y0 + crop - 4, x0:x0 + crop - 4] = rf[y0:y0 + crop - 4, x0:x0 + crop - 4]
        tiles.append((md, rm, rr, p))
    mds, rms, rrs, Rs, ts = [], [], [], [], []
    for i in range(n_hyp):
        md, rm, rr, p = tiles[i % len(tiles)]
        mds.append(md); rms.append(rm); rrs.append(rr)
        Rs.append(p[:12].reshape(3, 4)[:, :3]); ts.append(p[:12].reshape(3, 4)[:, 3])
    return ref, mds, rms, rrs, Rs, ts


def bench_icp(h, synth, n_hyp: int = 256, cpu: bool = True):
    """C3 (BASELINE configs[2]): n_hyp pose hypotheses x ~10k model points against one 640x480 depth frame."""
    ref, mds, rms, rrs, Rs, ts = make_icp_workload(synth, n_hyp)
    K = (608.0, 608.0, 320.0, 240.0)
    h.detection_batch(ref, K, mds, rms, rrs, Rs, ts)          # warm-up (allocates the workspace)
    times, dev = [], []
    h.profile(True)
    for _ in range(5):
        t0 = time.perf_counter()
        res = h.detection_batch(ref, K, mds, rms, rrs, Rs, ts)
        times.append(time.perf_counter() - t0)
        dev.append(h.last_icp_ms())
    trace = h.icp_trace(n_hyp).astype(np.float64)              # per-hypothesis phase clock of the fused launch (SM cycles)
    h.profile(False)
    # the same batch with the model crops resident on the device (uploaded once, as AddObj would): only the reference frame
    # and the hypothesis records are copied per call
    h.upload_model_depths(mds, rms)
    idx = list(range(n_hyp))
    h.detection_batch_resident(ref, K, idx, rrs, Rs, ts)
    times_res = []
    for _ in range(5):
        t0 = time.perf_counter()
        res2 = h.detection_batch_resident(ref, K, idx, rrs, Rs, ts)
        times_res.append(time.perf_counter() - t0)
    if res2.tobytes() != res.tobytes():
        raise RuntimeError("resident-crop ICP results differ from the per-call upload path")
    its = int(res["iterations"].sum())
    t = float(np.min(times))
    out = {"workload": "C3: %d hypotheses x 10,000-pixel model crops (mean %d paired valid points) vs one 640x480 depth frame, <=10 iterations"
                       % (n_hyp, int(res["n_points"].mean())),
           "icp_iters_per_s": its / t, "hypotheses_per_s": n_hyp / t, "total_iterations": its, "batch_ms": 1e3 * t,
           "device_ms": float(np.min(dev)), "icp_iters_per_s_device": its / (float(np.min(dev)) * 1e-3),
           "timer": "host wall clock around fl_detection_batch (includes H2D of crops and D2H of poses)",
           "batch_ms_resident_crops": 1e3 * float(np.min(times_res)),
           "icp_iters_per_s_resident_crops": its / float(np.min(times_res))}
    # roofline of the ICP launch (SURVEY 8d K10): 36 algorithmic bytes per model point and iteration (12 model + 12 matched
    # reference + 12 index-paired reference).  The launch is NOT bandwidth bound - three serial fp32 sums per iteration that must
    # round like the reference's loops set its floor - so the fraction is reported for completeness, next to the share of the
    # hypothesis time spent inside those sums and in the neighbour search.
    hbm_gbs, sm_mhz, peak_src = load_peaks()
    alg = 36.0 * float((res["n_points"].astype(np.float64) * res["iterations"]).sum())
    ach = alg / (float(np.min(dev)) * 1e-3) / 1e9
    tot = max(float(trace[:, 9].sum()), 1.0)
    out["roofline"] = {"kernel": "k_icp_fused (pairing + the whole icpCloudToCloud_Ex loop, one persistent launch)", "bound": "latency (ordered fp32 sums)",
                       "achieved": ach, "peak": hbm_gbs, "unit": "GB/s", "frac": ach / hbm_gbs, "peak_source": peak_src + " MEASURED_PEAKS.json hbm_gbs (no L2 figure there)",
                       "algorithmic_bytes_per_launch": alg, "traffic": None,
                       "time_shares": {"ordered_sums": float((trace[:, 1] + trace[:, 6] + trace[:, 14]).sum() / tot),
                                       "neighbour_search_beyond_the_distance_sum": float((trace[:, 4] - trace[:, 14]).sum() / tot),
                                       "distances": float(trace[:, 3].sum() / tot), "pairing_and_grid": float((trace[:, 0] + trace[:, 2]).sum() / tot),
                                       "correspondences_svd_rest": float((trace[:, 5] + trace[:, 7] + trace[:, 8]).sum() / tot)},
                       "sm_time_us_per_hypothesis_mean": float(trace[:, 9].mean() / sm_mhz), "sm_time_us_per_iteration_mean": float((trace[:, 9] / np.maximum(trace[:, 10], 1)).mean() / sm_mhz),
                       "ordered_sum_cycles_per_step": float(trace[:, 15].sum() / max(float(((1 + trace[:, 10]) * trace[:, 11]).sum()), 1.0))}
    if cpu:                                                    # CPU baseline leg: the C restatement of detection(), one thread, 8 hypotheses
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import fl_oracle_py as F
        import fl_ref_py as R
        use_ref = R.available()
        cits = int(sum(res["iterations"][:8]))                 # (the reference's detection() does not report its iteration count; the poses are identical)
        t0 = time.perf_counter()
        for i in range(8):
            if use_ref:
                rr_ = R.detection(mds[i], ref, K, rms[i], rrs[i], r_match=Rs[i], t_match=ts[i])
                if not (np.array_equal(rr_["R"], res["R"][i].reshape(3, 3)) and np.array_equal(rr_["T"], res["T"][i])):
                    raise RuntimeError("ICP pose %d differs from the reference's own detection()" % i)
            else:
                F.detection(mds[i], ref, K, rms[i], rrs[i], r_match=Rs[i], t_match=ts[i])
        ct = time.perf_counter() - t0
        out["cpu_baseline"] = {"icp_iters_per_s": cits / ct, "hypotheses_per_s": 8 / ct, "cores": 1, "kind": "reference" if use_ref else "port",
                               "sample": "the first 8 hypotheses of the same batch through %s (back-projection of both frames + KD-tree build + ICP loop each); poses compared bit for bit"
                                         % ("the reference's own detection() (oracle/_ref)" if use_ref else "the C restatement")}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (frames); default 500 for C2, 100 for C4 / C5")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--templates", type=int, default=8000, help="templates per GPU")
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "nccl"], help="candidate exchange of the template-sharded path (N > 1)")
    ap.add_argument("--per-step", action="store_true", help="print the distribution of per-step device times of every rank to stderr")
    ap.add_argument("--in-flight", type=int, default=0, help="frames in flight per GPU (1 = the synchronous Detector::match loop); default 4 for C2, 8 for the C4 / C5 pipelines")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-icp", action="store_true", help="skip the ICP side benchmark")
    ap.add_argument("--config", default="C2", choices=["C2", "C4", "C5"], help="C2: the headline match-only benchmark (weak scaling); C4 / C5: the "
                    "strong-scaling pipeline benchmark (fixed template set sharded over the GPUs, match + top-5 ICP + NMS, frames/s)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed frame returned to DIR as "
                    "float64 .npy files: its match list (matches_<field>.npy) and, for C4 / C5, its ICP results (icp_<field>.npy) "
                    "and the NMS keep-list (nms_keep.npy)")
    args = ap.parse_args()
    pipeline = args.config != "C2" and args.impl == "ours"
    if args.steps is None:
        args.steps = 100 if pipeline else 500
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if pipeline:
        run_pipeline(args)
    elif args.impl == "reference":
        run_reference(args)            # ~0.1 s per step on 8 host threads: the default run ends within seconds
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
