"""GPU (-m gpu): masked frames take the single-launch front end, and masks reach every throughput path - pipes, template-sharded
pipes, groups and the C++ Detector over several devices.

A frame's mask of a modality is applied where the spread jobs read the labels (dev_spread_lm): the level-0 mask at a shift of l
when every level halves exactly, the NN mask pyramid built by the per-wave schedule otherwise.  Every case compares the match list
and the quantised images with the C oracle, or with one handle's fl_match of the same frame, record for record and byte for byte."""
import os
import struct
import subprocess
import time

import numpy as np
import pytest

import fealess_b200 as fb
import fl_oracle_py as F
from fealess_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H, T = 640, 480, (5, 8)
CAP = 1 << 19


def _mask(W, H, seed, value=255, density=0.8):
    """A speckled mask (density of kept pixels) with a solid window: labels are dropped both inside objects and along whole rows."""
    rng = np.random.default_rng(seed)
    m = (rng.random((H, W)) < density).astype(np.uint8) * np.uint8(value)
    m[H // 8:H // 2, W // 6:W // 2] = value
    m[:, 3 * W // 4:] = 0
    return m


def _masks(case, W, H):
    a, b = _mask(W, H, 1), _mask(W, H, 2, density=0.6)
    return {"colour": [a, None], "depth": [None, b], "both": [a, b], "zero": [np.zeros((H, W), np.uint8)] * 2,
            "all": [np.full((H, W), 7, np.uint8)] * 2, "value1": [_mask(W, H, 3, 1), _mask(W, H, 4, 1)],
            "value128": [_mask(W, H, 5, 128), _mask(W, H, 6, 128)]}[case]


def _oracle(det, b, d, masks, thr, L=2):
    assert det.process(b, d, masks) == 0
    return det.match(float(thr), n_threads=8), [det.quantized(l, m) for l in range(L) for m in range(2)]


@pytest.fixture(scope="module")
def c2():
    """bench.py's C2 set: 8,000 templates (seed 1, 1 % planted on frame 0's quantised images), frames 0 - 2."""
    frames = [synth.make_frame(W, H, i) for i in range(3)]
    det = F.Detector(T)
    assert det.process(*frames[0]) == 0
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    ts = synth.make_templates(8000, W, H, T, seed=1, quantized=q, planted_fraction=0.01)
    det.set_templates(ts)
    h = fb.Handle(T, (0, 1), W, H, max_candidates=CAP)
    h.upload_templates(ts)
    yield frames, det, ts, h
    h.close()


@pytest.mark.parametrize("case", ["colour", "depth", "both", "zero", "all", "value1", "value128"])
def test_single_handle_equals_oracle(c2, case):
    frames, det, ts, h = c2
    b, d = frames[0]
    masks = _masks(case, W, H)
    for thr in (60, 75):
        want, wq = _oracle(det, b, d, masks, thr)
        rc, got, q = h.match(b, d, float(thr), masks=masks, want_quantized=True, capacity=CAP)
        assert rc == 0 and h.uses_staged() and np.array_equal(got, want), (case, thr, len(got), len(want))
        for i in range(4):
            assert np.array_equal(q[i], wq[i]), (case, thr, i)
            assert np.array_equal(h.debug_quantized(i // 2, i % 2, W, H), wq[i]), (case, thr, i)
        if case == "zero":
            assert len(got) == 0
        unmasked = h.match(b, d, float(thr), capacity=CAP)[1]
        if case == "all":
            assert np.array_equal(got, unmasked)
        else:                                                    # a mask only takes labels away
            assert len(got) <= len(unmasked) and (case != "both" or len(got) < len(unmasked))
    # a device-resident frame and masks give the same list
    import torch
    db, dd = torch.from_numpy(b).cuda(), torch.from_numpy(d.view(np.int16)).cuda()
    dm = [None if m is None else torch.from_numpy(m).cuda() for m in masks]
    h.match_device(db.data_ptr(), dd.data_ptr(), W, H, 75.0, masks=[0 if m is None else m.data_ptr() for m in dm])
    assert np.array_equal(h.match_fetch(CAP), _oracle(det, b, d, masks, 75)[0])


@pytest.mark.parametrize("geom", [(1280, 720, (5, 8), 600), (1920, 1080, (5, 5, 5, 5), 300), (225, 480, (5, 8), 300)],
                         ids=["720p", "c5_four_levels", "does_not_halve"])
def test_other_geometries_equal_oracle(geom):
    """720p, the C5 geometry with four levels, and 225 x 480, whose level 1 (112 x 240) is not an exact half: there the per-wave
    schedule builds the mask pyramid with NN-resize jobs."""
    Wg, Hg, Tg, n = geom
    L = len(Tg)
    b, d = synth.make_frame(Wg, Hg, 1)
    det = F.Detector(Tg)
    assert det.process(b, d) == 0
    q = [det.quantized(l, m) for l in range(L) for m in range(2)]
    ts = synth.make_templates(n, Wg, Hg, Tg, n_classes=3, seed=7, quantized=q, planted_fraction=0.05)
    det.set_templates(ts)
    h = fb.Handle(Tg, (0, 1), Wg, Hg, max_candidates=CAP)
    h.upload_templates(ts)
    for case in ("colour", "both"):
        masks = _masks(case, Wg, Hg)
        want, wq = _oracle(det, b, d, masks, 60, L)
        rc, got, gq = h.match(b, d, 60.0, masks=masks, want_quantized=True, capacity=CAP)
        assert rc == 0 and np.array_equal(got, want), (geom, case, len(got), len(want))
        assert all(np.array_equal(gq[i], wq[i]) for i in range(2 * L)), (geom, case)
    assert len(want) > 0
    h.close()


def test_every_schedule_and_option(c2):
    frames, det, ts, h = c2
    b, d = frames[1]
    masks = _masks("both", W, H)
    want, wq = _oracle(det, b, d, masks, 75)
    assert len(want) > 0
    for opt in (fb.FL_OPT_FE_WAVES, fb.FL_OPT_SPLIT_REFINE, fb.FL_OPT_SIM_NO_PRUNE, fb.FL_OPT_SIM_ROTATE, "force_baseline"):
        if opt == "force_baseline":
            h.force_baseline(True)
        else:
            assert h.debug_option(opt, 1) == 0
        rc, got, q = h.match(b, d, 75.0, masks=masks, want_quantized=True, capacity=CAP)
        assert rc == 0 and np.array_equal(got, want), opt
        assert all(np.array_equal(q[i], wq[i]) for i in range(4)), opt
        if opt == "force_baseline":
            assert not h.uses_staged()
            h.force_baseline(False)
        else:
            h.debug_option(opt, 0)
    assert h.match(b, d, 75.0, masks=masks, capacity=CAP)[0] == 0 and h.uses_staged()


def test_dependency_time_out_reruns_masked_frames(c2):
    """FL_OPT_FE_DEP_TIMEOUT_TEST: the single launch gives up on an in-grid dependency, the handle re-runs the frame with one launch
    per wave from the masks it kept - staged host masks on one handle, device masks on another."""
    import torch
    frames, det, ts, _ = c2
    b, d = frames[2]
    masks = _masks("both", W, H)
    want = _oracle(det, b, d, masks, 75)[0]
    for device in (False, True):
        h = fb.Handle(T, (0, 1), W, H, max_candidates=CAP)
        h.upload_templates(ts)
        assert h.debug_option(fb.FL_OPT_FE_DEP_TIMEOUT_TEST, 1) == 0
        if device:
            db, dd = torch.from_numpy(b).cuda(), torch.from_numpy(d.view(np.int16)).cuda()
            dm = [torch.from_numpy(m).cuda() for m in masks]
            h.match_device(db.data_ptr(), dd.data_ptr(), W, H, 75.0, masks=[m.data_ptr() for m in dm])
            got = h.match_fetch(CAP)
        else:
            rc, got = h.match(b, d, 75.0, masks=masks, capacity=CAP)
            assert rc == 0
        assert h.debug_option(fb.FL_OPT_FE_FORCED_WAVES, 0) == 1
        assert np.array_equal(got, want), device
        h.close()


def test_masked_frame_launches_like_an_unmasked_one(c2):
    frames, det, ts, h = c2
    b, d = frames[0]
    h.match(b, d, 75.0, capacity=CAP)
    n0 = h.launch_count()
    h.match(b, d, 75.0, capacity=CAP)
    n1 = h.launch_count()
    h.match(b, d, 75.0, masks=_masks("both", W, H), capacity=CAP)
    n2 = h.launch_count()
    h.match(b, d, 75.0, masks=_masks("colour", W, H), capacity=CAP)
    assert n1 - n0 == n2 - n1 == h.launch_count() - n2 == 3


def test_first_masked_frame_allocates_nothing(c2):
    """The staged masks are sized at fl_create: free device memory is the same before and after the first masked frame (host masks,
    then device masks).  Another process on the GPU can move the number, so a difference has to show on three fresh handles."""
    import torch
    frames, det, ts, _ = c2
    b, d = frames[0]
    masks = _masks("both", W, H)
    dm = [torch.from_numpy(m).cuda() for m in masks]
    torch.cuda.synchronize()
    diffs = []
    for attempt in range(3):
        h = fb.Handle(T, (0, 1), W, H)
        h.upload_templates(ts)
        assert h.match(b, d, 75.0)[0] == 0                       # the geometry's own set-up (plan, packed features) happens here
        db, dd = torch.from_numpy(b).cuda(), torch.from_numpy(d.view(np.int16)).cuda()
        torch.cuda.synchronize()
        before = torch.cuda.mem_get_info()[0]
        assert h.match(b, d, 75.0, masks=masks)[0] == 0
        h.match_device(db.data_ptr(), dd.data_ptr(), W, H, 75.0, masks=[m.data_ptr() for m in dm])
        after = torch.cuda.mem_get_info()[0]
        h.close()
        diffs.append(before - after)
        if before == after:
            break
    assert diffs[-1] == 0, diffs


def _single_lists(h, frames, plan, thr=75.0):
    return [h.match(*frames[f], thr, masks=mk, capacity=CAP)[1] for f, mk in plan]


def _plan():
    """16 frames: unmasked, masked and differently masked frames of three images, in an order that puts every kind next to every other."""
    kinds = [None, "both", "colour", "depth", "value128", None, "both", "depth", "zero", "colour", None, "value1", "both", "both", None, "all"]
    return [(i % 3, None if k is None else _masks(k, W, H)) for i, k in enumerate(kinds)]


@pytest.mark.parametrize("depth", [1, 2, 3, 4])
def test_pipe_mixes_masked_and_unmasked_frames(c2, depth):
    import torch
    frames, det, ts, h = c2
    plan = _plan()
    want = _single_lists(h, frames, plan)
    pinned = [(torch.from_numpy(b).pin_memory().numpy(), torch.from_numpy(d.view(np.int16)).pin_memory().numpy().view(np.uint16)) for b, d in frames]
    dev = [(torch.from_numpy(b).cuda(), torch.from_numpy(d.view(np.int16)).cuda()) for b, d in frames]
    dmasks = [None if mk is None else [torch.from_numpy(m).cuda() if m is not None else None for m in mk] for _, mk in plan]
    p = fb.Pipe(depth, T, (0, 1), W, H, max_candidates=CAP)
    p.upload_templates(ts)
    got = []
    for k, (f, mk) in enumerate(plan):
        if p.in_flight() == depth:
            got.append(p.collect(CAP))
        if k % 3 == 0:
            p.submit(*frames[f], 75.0, masks=mk)
        elif k % 3 == 1:
            pm = None if mk is None else [None if m is None else torch.from_numpy(m).pin_memory().numpy() for m in mk]
            p.submit(*pinned[f], 75.0, masks=pm)
        else:
            p.submit_device(dev[f][0].data_ptr(), dev[f][1].data_ptr(), W, H, 75.0,
                            d_masks=None if mk is None else [0 if m is None else m.data_ptr() for m in dmasks[k]])
    while p.in_flight():
        got.append(p.collect(CAP))
    assert len(got) == len(plan)
    for k, (rc, m) in enumerate(got):
        assert rc == 0 and np.array_equal(m, want[k]), k
    p.close()


def test_template_sharded_pipes_on_one_gpu(c2):
    """Two pipes = the two ranks of a template-sharded detector on this GPU (as in test_gpu_pipe.py), masked host and device frames."""
    import torch
    from fealess_b200 import sharded
    frames, det, ts, h = c2
    plan = _plan()
    want = _single_lists(h, frames, plan)
    world, depth, cap = 2, 3, 4096
    nbytes = int(fb.lib().fl_exchange_buffer_bytes(world, cap))
    xbuf = [[torch.zeros(nbytes, dtype=torch.uint8, device="cuda") for _ in range(world)] for _ in range(depth)]
    blocks = [[torch.zeros(sharded.block_ints(cap), dtype=torch.int32, device="cuda") for _ in range(depth)] for _ in range(world)]
    dev = [(torch.from_numpy(b).cuda(), torch.from_numpy(d.view(np.int16)).cuda()) for b, d in frames]
    dmasks = [None if mk is None else [torch.from_numpy(m).cuda() if m is not None else None for m in mk] for _, mk in plan]
    pipes = []
    for r in range(world):
        p = fb.Pipe(depth, T, (0, 1), W, H, max_candidates=CAP)
        shard, gids = sharded.shard_template_set(ts, r, world)
        p.upload_templates(shard)
        p.set_template_ids(gids)
        p.set_exchange(r, world, cap, [[xbuf[i][q].data_ptr() for q in range(world)] for i in range(depth)], [b.data_ptr() for b in blocks[r]])
        pipes.append(p)
    torch.cuda.synchronize()
    got = [[], []]
    for k, (f, mk) in enumerate(plan):
        if pipes[0].in_flight() == depth:
            for r in range(world):
                got[r].append(pipes[r].collect(CAP))
        for r in range(world):
            if k % 2:
                pipes[r].submit_device(dev[f][0].data_ptr(), dev[f][1].data_ptr(), W, H, 75.0,
                                       d_masks=None if mk is None else [0 if m is None else m.data_ptr() for m in dmasks[k]])
            else:
                pipes[r].submit(*frames[f], 75.0, masks=mk)
    while pipes[0].in_flight():
        for r in range(world):
            got[r].append(pipes[r].collect(CAP))
    for r in range(world):
        assert len(got[r]) == len(plan)
        for k, (rc, m) in enumerate(got[r]):
            assert rc == 0 and np.array_equal(m, want[k]), (r, k)
    for p in pipes:
        p.close()


def test_sharded_pipe_mirror_with_one_rank(c2):
    """fealess_b200.sharded.ShardedPipe (one rank): submit_host / submit_device pass the masks through."""
    import torch
    from fealess_b200 import sharded
    frames, det, ts, h = c2
    plan = _plan()[:6]
    want = _single_lists(h, frames, plan)
    sp = sharded.ShardedPipe(lambda: fb.Handle(T, (0, 1), W, H, max_candidates=CAP), ts, 0, 1, depth=2)
    dev = [(torch.from_numpy(b).cuda(), torch.from_numpy(d.view(np.int16)).cuda()) for b, d in frames]
    dmasks = [None if mk is None else [torch.from_numpy(m).cuda() if m is not None else None for m in mk] for _, mk in plan]
    got = []
    for k, (f, mk) in enumerate(plan):
        if sp.in_flight() == 2:
            got.append(sp.collect().h.match_fetch(CAP))
        if k % 2:
            sp.submit_device(dev[f][0].data_ptr(), dev[f][1].data_ptr(), W, H, 75.0, masks=None if mk is None else [0 if m is None else m.data_ptr() for m in dmasks[k]])
        else:
            sp.submit_host(*frames[f], 75.0, masks=mk)
    while sp.in_flight():
        got.append(sp.collect().h.match_fetch(CAP))
    assert all(np.array_equal(got[k], want[k]) for k in range(len(plan)))
    sp.close()


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0], [0, 1]], ids=["0,0", "0,0,0", "0,1"])
def test_group_first_frame_masked(c2, devices):
    """The first frame after fl_group_create is masked: no member allocates while its peers' exchange kernels wait for it, so the
    frame returns in well under the 2 s peer time-out, with one handle's list."""
    import torch
    if torch.cuda.device_count() < max(devices) + 1:
        pytest.skip("%d GPU(s) visible, the case needs %d" % (torch.cuda.device_count(), max(devices) + 1))
    frames, det, ts, h = c2
    plan = _plan()[:5]
    want = _single_lists(h, frames, plan)
    g = fb.Group(devices, exchange_capacity=8192)
    g.upload_templates(ts)
    f, mk = plan[1]
    t0 = time.perf_counter()
    rc, got = g.match(*frames[f], 75.0, masks=mk)
    assert time.perf_counter() - t0 < 1.5
    assert rc == 0 and np.array_equal(got, want[1])
    for k, (f, mk) in enumerate(plan):
        rc, got = g.match(*frames[f], 75.0, masks=mk)
        assert rc == 0 and np.array_equal(got, want[k]), k
    assert g.match(*frames[0], 75.0, masks=_masks("both", W, H)[:1])[0] == fb.FL_ERR_SIZE     # mask count, as Handle.match
    g.close()


def test_cpp_detector_use_devices_with_masks(c2, tmp_path):
    """tests/cpp/masked_group_test.cpp: cup_linemod::Detector::useDevices({0, 0}) with masks equals one device, quantised images
    included."""
    from fealess_b200 import build as fbuild
    frames, det, ts, h = c2
    b, d = frames[0]
    assert det.process(b, d) == 0
    small = synth.make_templates(1500, W, H, T, n_classes=3, seed=1, quantized=[det.quantized(l, m) for l in range(2) for m in range(2)],
                                 planted_fraction=0.05)
    masks = _masks("both", W, H)
    blob = b"".join([
        struct.pack("<ii", W, H), np.ascontiguousarray(b, np.uint8).tobytes(), np.ascontiguousarray(d, np.uint16).tobytes(),
        struct.pack("<ii", 2, 2), np.asarray(T, np.int32).tobytes(),
        struct.pack("<i", small.n_templates), np.ascontiguousarray(small.headers, np.int32).tobytes(),
        struct.pack("<i", len(small.features)), np.ascontiguousarray(small.features, np.int32).tobytes(),
        np.ascontiguousarray(small.class_of, np.int32).tobytes(), struct.pack("<f", 60.0), masks[0].tobytes(), masks[1].tobytes()])
    case = tmp_path / "masked_group_case.bin"
    case.write_bytes(blob)
    fbuild.build()
    exe = str(tmp_path / "masked_group_test")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    r = subprocess.run([cxx, "-std=c++11", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "masked_group_test.cpp"), "-o", exe, fb.library_path(),
                        "-Wl,-rpath," + os.path.dirname(fb.library_path())], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([exe, str(case), "0,0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all checks passed" in r.stdout
