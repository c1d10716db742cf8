"""GPU: Recognition on template-sharded pipes (fl_pipe_set_recognition_sharded, fl_pipe_*_recognition after fl_pipe_set_exchange).  Two,
three or eight fl_pipes of this process are the ranks, with exchange buffers in plain device memory, driven in lock-step from one thread.
The reference of every comparison is a single handle's fl_recognize over the whole set: on EVERY rank the result records are compared as
bytes (fl_reco_result_t) and the summaries too."""
import ctypes as C

import numpy as np
import pytest

import fealess_b200 as fb
from fealess_b200 import sharded
from test_gpu_reco_group import K, T, W, H, _Ref, _big, _crops, _edge_templates, _mixed, _planted, _same

pytestmark = pytest.mark.gpu
MODES = [(1, False, 0.0), (5, True, 30.0)]
TAIL_LAUNCHES = 3                                                # k_reco_select, k_icp_fused, k_reco_finish on the frame's owner
RECEIVE_LAUNCHES = 1                                             # k_reco_receive on every other rank


class _Ranks:
    """`world` pipes of `depth` slots = the ranks of one template-sharded detector; the exchange buffers live as long as the pipes"""

    def __init__(self, ts, crops, rects, world, depth, cap=4096):
        import torch
        self.world, self.depth = world, depth
        nbytes = int(fb.lib().fl_exchange_buffer_bytes(world, cap))
        self.xbuf = [[torch.zeros(nbytes, dtype=torch.uint8, device="cuda") for _ in range(world)] for _ in range(depth)]   # [slot][rank]
        self.blocks = [[torch.zeros(sharded.block_ints(cap), dtype=torch.int32, device="cuda") for _ in range(depth)] for _ in range(world)]
        self.pipes = []
        for r in range(world):
            p = fb.Pipe(depth, T, (0, 1), W, H, max_candidates=max(1 << 16, world * (cap + 1) + 16))
            shard, gids = sharded.shard_template_set(ts, r, world)
            p.upload_templates(shard)
            if shard.n_templates:
                p.set_template_ids(gids)
            p.upload_model_depths(crops, rects)
            p.set_exchange(r, world, cap, [[self.xbuf[i][q].data_ptr() for q in range(world)] for i in range(depth)],
                           [b.data_ptr() for b in self.blocks[r]])
            self.pipes.append(p)
        torch.cuda.synchronize()

    def set_recognition(self, ts, crop_of, params):
        for p in self.pipes:
            p.set_recognition_sharded(ts, crop_of, params=params)

    def stream(self, frames, kinds=None, threshold=75.0, capacity=fb.RECO_MAX_HYP):
        """frames in lock-step: every rank submits frame i before any waits; kinds[i] 'm' = a match frame (fl_pipe_submit).  Returns
        the collected (rc, records, summary) or (rc, matches) of every frame, per rank."""
        out, queued = [[] for _ in self.pipes], []

        def collect():
            k = queued.pop(0)
            for r, p in enumerate(self.pipes):
                out[r].append(p.collect() if k == "m" else p.collect_recognition(capacity))
        for i, (b, d) in enumerate(frames):
            if len(queued) == self.depth:
                collect()
            k = kinds[i] if kinds else "r"
            for p in self.pipes:
                if k == "m":
                    p.submit(b, d, threshold)
                else:
                    p.submit_recognition(b, d, K, W, H)
            queued.append(k)
            assert all(p.in_flight() == len(queued) for p in self.pipes)
        while queued:
            collect()
        return out

    def launch_counts(self):
        """fl_launch_count of every slot's handle, shape (depth, world)"""
        L = fb.lib()
        L.fl_pipe_handle.restype = C.c_void_p
        return np.array([[int(L.fl_launch_count(C.c_void_p(L.fl_pipe_handle(p._p, s)))) for p in self.pipes] for s in range(self.depth)], np.int64)

    def close(self):
        for p in self.pipes:
            p.close()


def _same_on_every_rank(got, want):
    for r, g in enumerate(got):
        try:
            _same(g, want)
        except AssertionError as e:
            raise AssertionError("rank %d: %s" % (r, e)) from None


@pytest.fixture(scope="module")
def mixed_case():
    b, d, ts = _planted(37, 3, 62)
    crops, rects = _crops(ts, d)
    frames = _mixed(b, d, 19)                                      # 640 x 480, 1280 x 960 rescaled on the device, a random scene, a blank frame
    ref = _Ref(ts, crops, rects, np.arange(ts.n_templates))
    want = {m: ref.run(frames, fb.reco_params(top_k=m[0], per_class=m[1], th_obj_dist=m[2])) for m in MODES}
    assert sum(len(r[1]) for r in want[MODES[1]]) >= 6
    return ts, crops, rects, frames, want


@pytest.mark.parametrize("depth", [1, 3])
@pytest.mark.parametrize("world", [2, 3])
def test_ranks_and_depths_over_mixed_frames(mixed_case, world, depth):
    """More frames than depth x world, so that every rank owns frames on every slot; top_k = 1, and top_k = 5 per class with suppression."""
    ts, crops, rects, frames, want = mixed_case
    n = 2 * depth * world + 1
    ranks = _Ranks(ts, crops, rects, world, depth)
    for m in MODES:
        ranks.set_recognition(ts, np.arange(ts.n_templates), fb.reco_params(top_k=m[0], per_class=m[1], th_obj_dist=m[2]))
        _same_on_every_rank(ranks.stream(frames[:n]), want[m][:n])
    ranks.close()


def test_no_matches_missing_crops_boxes_outside_and_deferred_lists():
    b, d, ts = _planted(24, 1, 61)
    crops, rects = _crops(ts, d)
    crop_of = np.where(np.arange(ts.n_templates) < ts.n_templates // 2, np.arange(ts.n_templates), -1)   # upper half: no crop
    blank = (np.zeros_like(b), np.zeros_like(d))
    frames = [blank, (b, d), blank, _big(b, d), (b, d)]
    params = fb.reco_params(top_k=8)
    want = _Ref(ts, crops, rects, crop_of).run(frames, params)
    assert want[0][2] == dict(n_matches=0, n_hypotheses=0, n_roi=0, n_results=0) and want[1][2]["n_hypotheses"] < 8
    ranks = _Ranks(ts, crops, rects, 3, 2)
    ranks.set_recognition(ts, crop_of, params)
    _same_on_every_rank(ranks.stream(frames), want)
    ranks.close()
    # reference boxes leaving the frame: FL_ERR_ROI hypotheses, no result
    b, d, ts = _edge_templates()
    crops, rects = _crops(ts, np.zeros_like(d))
    ranks = _Ranks(ts, crops, rects, 2, 2)
    for top_k in (1, 4):
        params = fb.reco_params(top_k=top_k)
        want = _Ref(ts, crops, rects, np.arange(ts.n_templates)).run([(b, d)] * 3, params)
        assert want[0][2]["n_roi"] == top_k and want[0][2]["n_results"] == 0
        ranks.set_recognition(ts, np.arange(ts.n_templates), params)
        _same_on_every_rank(ranks.stream([(b, d)] * 3), want)
    ranks.close()
    # a union of more than 1,024 records: every rank runs the tail on its own copy of the list sorted after the wait
    b, d, ts = _planted(400, 2, 2, planted=0.05)
    crops, rects = _crops(ts, d)
    frames = [(b, d), _big(b, d), (b, d), (b, d)]
    for hyp in (dict(top_k=3), dict(top_k=2, per_class=True, th_obj_dist=25.0)):
        params = fb.reco_params(threshold=25.0, **hyp)
        want = _Ref(ts, crops, rects, np.arange(ts.n_templates)).run(frames, params)
        assert want[0][2]["n_matches"] > 1024 and len(want[0][1]) >= 1
        for world, depth in ((2, 2), (3, 3)):
            ranks = _Ranks(ts, crops, rects, world, depth, cap=8192)
            ranks.set_recognition(ts, np.arange(ts.n_templates), params)
            _same_on_every_rank(ranks.stream(frames), want)
            ranks.close()


def test_fewer_templates_than_ranks():
    """Five templates over eight ranks: three ranks hold none and still take part in the exchange, own frames and push their results."""
    b, d, ts = _planted(5, 1, 61, planted=1.0)
    crops, rects = _crops(ts, d)
    frames = [(b, d), _big(b, d)] * 5
    params = fb.reco_params(top_k=4)
    want = _Ref(ts, crops, rects, np.arange(ts.n_templates)).run(frames, params)
    assert sum(len(r[1]) for r in want) >= 4
    ranks = _Ranks(ts, crops, rects, 8, 2)
    ranks.set_recognition(ts, np.arange(ts.n_templates), params)
    _same_on_every_rank(ranks.stream(frames), want)
    ranks.close()


def test_match_frames_between_recognition_frames(mixed_case):
    """fl_pipe_submit and fl_pipe_submit_recognition on the same sharded pipe: match frames return the single handle's list, recognition
    frames its results, in submission order."""
    ts, crops, rects, frames, want = mixed_case
    m = MODES[1]
    kinds = "rmrrmmrmrrrm"
    sel = [i for i in range(len(frames)) if frames[i][1].shape[1] == W][:len(kinds)]   # match frames take the pipe's own geometry
    h = fb.Handle(T, (0, 1))
    h.upload_templates(ts)
    want_m = {i: h.match(*frames[i], 75.0) for i in sel}
    h.close()
    ranks = _Ranks(ts, crops, rects, 2, 3)
    ranks.set_recognition(ts, np.arange(ts.n_templates), fb.reco_params(top_k=m[0], per_class=m[1], th_obj_dist=m[2]))
    got = ranks.stream([frames[i] for i in sel], kinds=kinds)
    for r in range(2):
        for k, i in enumerate(sel):
            if kinds[k] == "m":
                assert got[r][k][0] == want_m[i][0] == fb.FL_OK and np.array_equal(got[r][k][1], want_m[i][1]), (r, k)
            else:
                _same([got[r][k]], [want[m][i]])
    ranks.close()


def test_capacity_below_the_results(mixed_case):
    """capacity < n_results: FL_ERR_CAPACITY on every rank with the summary intact and the first `capacity` records."""
    ts, crops, rects, frames, want = mixed_case
    m = MODES[1]
    i = max(range(len(frames)), key=lambda k: len(want[m][k][1]))
    n = len(want[m][i][1])
    assert n >= 2
    ranks = _Ranks(ts, crops, rects, 3, 2)
    ranks.set_recognition(ts, np.arange(ts.n_templates), fb.reco_params(top_k=m[0], per_class=m[1], th_obj_dist=m[2]))
    got = ranks.stream([frames[i]] * 4, capacity=n - 1)
    for r in range(3):
        for rc, recs, summ in got[r]:
            assert rc == fb.FL_ERR_CAPACITY and summ == want[m][i][2] and recs.tobytes() == want[m][i][1][:n - 1].tobytes(), r
    ranks.close()


def test_state_errors():
    b, d, ts = _planted(24, 1, 61)
    crops, rects = _crops(ts, d)
    ranks = _Ranks(ts, crops, rects, 2, 2)
    p = ranks.pipes[0]
    for call in (lambda: p.collect_recognition(), lambda: p.submit_recognition(b, d, K)):     # nothing in flight / no set-up
        with pytest.raises(fb.FealessError) as e:
            call()
        assert e.value.rc == fb.FL_ERR_STATE and p.in_flight() == 0
    with pytest.raises(fb.FealessError) as e:                          # the handle-level set-up of a pipe that holds one shard
        p.set_recognition(np.arange(ts.n_templates))
    assert e.value.rc == fb.FL_ERR_STATE and "fl_pipe_set_recognition_sharded" in str(e.value)
    bad = list(rects[0]); bad[2] -= 2
    p.upload_model_depths(crops, [tuple(bad)] + rects[1:])
    with pytest.raises(fb.FealessError) as e:                          # crop 0 is not template 0's level-0 box
        p.set_recognition_sharded(ts, np.arange(ts.n_templates))
    assert e.value.rc == fb.FL_ERR_ARG
    p.upload_model_depths(crops, rects)
    plain = fb.Pipe(2, T, (0, 1), W, H)                                # not template-sharded
    plain.upload_templates(ts)
    plain.upload_model_depths(crops, rects)
    with pytest.raises(fb.FealessError) as e:
        plain.set_recognition_sharded(ts, np.arange(ts.n_templates))
    assert e.value.rc == fb.FL_ERR_STATE
    plain.close()
    ranks.set_recognition(ts, np.arange(ts.n_templates), fb.reco_params())
    want = _Ref(ts, crops, rects, np.arange(ts.n_templates)).run([(b, d)], fb.reco_params())
    for q in ranks.pipes:
        q.submit_recognition(b, d, K)
    with pytest.raises(fb.FealessError) as e:                          # not while a frame is in flight
        p.set_recognition_sharded(ts, np.arange(ts.n_templates))
    assert e.value.rc == fb.FL_ERR_STATE
    _same_on_every_rank([[q.collect_recognition()] for q in ranks.pipes], want)
    p.upload_model_depths(crops, rects)                                # a new crop set clears the set-up
    with pytest.raises(fb.FealessError) as e:
        p.submit_recognition(b, d, K)
    assert e.value.rc == fb.FL_ERR_STATE and p.in_flight() == 0
    ranks.close()


def test_only_the_owner_runs_the_tail():
    """fl_launch_count of every (slot, rank) handle: a frame adds the same match launches on every rank of its slot, the three tail
    launches on its owner (rank f % world) and the one receive launch on every other rank; no other slot moves."""
    b, d, ts = _planted(37, 3, 62)
    crops, rects = _crops(ts, d)
    world, depth = 3, 2
    ranks = _Ranks(ts, crops, rects, world, depth)
    ranks.set_recognition(ts, np.arange(ts.n_templates), fb.reco_params(top_k=2))
    ranks.stream([(b, d)] * depth)                                 # the first frame of every slot packs the templates for the geometry
    per_rank = {}
    for f in range(depth, depth + 4 * world):
        before = ranks.launch_counts()
        got = ranks.stream([(b, d)])
        assert all(g[0][0] == fb.FL_OK and len(g[0][1]) >= 1 for g in got)
        delta = ranks.launch_counts() - before
        s = f % depth
        assert (np.delete(delta, s, axis=0) == 0).all(), delta
        for r in range(world):
            match = delta[s, r] - (TAIL_LAUNCHES if r == f % world else RECEIVE_LAUNCHES)
            assert match >= 3, delta
            assert per_rank.setdefault((s, r), match) == match, (f, delta)
    ranks.close()
