"""GPU: one frame in flight per handle.  Every entry point that enqueues frame work refuses (FL_ERR_STATE) while a match frame or a
recognition frame is in flight, and leaves that frame intact: it then waits and fetches byte for byte what an undisturbed handle gives.
(fl_reco_shard_stage, the group's staging step, shares fl_recognize_async's start; it is not part of the C ABI.)"""
import ctypes as C

import numpy as np
import pytest

import fealess_b200 as fb
from fealess_b200 import synth

pytestmark = pytest.mark.gpu

W, H, T = 640, 480, (5, 8)
K = (608.0, 608.0, 320.0, 240.0)
CAP = 64


@pytest.fixture(scope="module")
def scene():
    import fl_oracle_py as F
    b, d = synth.make_frame(W, H, 0)
    det = F.Detector(T)
    assert det.process(b, d) == 0
    q = [det.quantized(l, m) for l in range(2) for m in range(2)]
    ts = synth.make_templates(24, W, H, T, n_classes=1, seed=61, quantized=q, planted_fraction=0.5)
    rects = [tuple(int(v) for v in ts.headers[t * 4][[2, 3, 0, 1]]) for t in range(ts.n_templates)]
    h = _handle(ts, d, rects)
    h.match_async(b, d, 75.0)
    h.match_wait()
    want_match = h.match_fetch().tobytes()
    rc, res, summary = h.recognize(b, d, K)
    assert rc == fb.FL_OK and len(res) >= 1
    h.close()
    return b, d, ts, rects, want_match, (res.tobytes(), summary)


def _handle(ts, d, rects):
    h = fb.Handle(T, (0, 1), W, H)
    h.upload_templates(ts)
    h.upload_model_depths([d] * ts.n_templates, rects)
    h.set_recognition(np.arange(ts.n_templates))
    return h


def _intruders(h, b, d, ts):
    """(name, call) of every entry point that enqueues frame work, with arguments it would run on; each call returns its status"""
    import torch
    L, hh = fb.lib(), h._h
    db, dd = torch.from_numpy(b).cuda(), torch.from_numpy(d).cuda()
    xbuf = torch.zeros(int(L.fl_exchange_buffer_bytes(1, CAP)), dtype=torch.uint8, device="cuda")
    recs = torch.zeros((CAP + 1) * 4, dtype=torch.int32, device="cuda")      # fl_match_t = 4 x int32; [count | records] blocks
    outs = torch.zeros((CAP + 1) * 4, dtype=torch.int32, device="cuda")
    keep = (db, dd, xbuf, recs, outs)
    peers = (C.c_void_p * 1)(xbuf.data_ptr())
    dev = lambda t: C.c_void_p(t.data_ptr())
    thr, sb, sd, e = C.c_float(75.0), C.c_size_t(W * 3), C.c_size_t(W * 2), C.c_uint32(1)
    out, cnt = np.zeros(CAP, fb.MATCH_DTYPE), C.c_int32(0)
    crops = np.arange(ts.n_templates, dtype=np.int32)
    calls = [
        ("fl_match_device_async", lambda: L.fl_match_device_async(hh, dev(db), dev(dd), W, H, None, thr, None, 0)),
        ("fl_match_async", lambda: L.fl_match_async(hh, fb._p(b), sb, fb._p(d), sd, W, H, None, thr, None, 0)),
        ("fl_match_rescaled", lambda: L.fl_match_rescaled(hh, fb._p(b), sb, fb._p(d), sd, W, H, W, H, thr, None, 0, fb._p(out), CAP, C.byref(cnt), None)),
        ("fl_match_shard_device", lambda: L.fl_match_shard_device(hh, dev(db), dev(dd), W, H, None, thr, None, 0, dev(recs), CAP, dev(outs))),
        ("fl_sort_unique_device", lambda: L.fl_sort_unique_device(hh, dev(recs), 1, CAP, dev(outs), dev(recs), CAP, dev(outs))),
        ("fl_sort_unique_blocks_device", lambda: L.fl_sort_unique_blocks_device(hh, dev(recs), 1, CAP)),
        ("fl_exchange_sort_unique_device", lambda: L.fl_exchange_sort_unique_device(hh, 0, 1, peers, CAP, dev(recs), e)),
        ("fl_exchange_sort_unique_device_async", lambda: L.fl_exchange_sort_unique_device_async(hh, 0, 1, peers, CAP, dev(recs), e)),
        ("fl_match_shard_exchange_async", lambda: L.fl_match_shard_exchange_async(hh, fb._p(b), sb, fb._p(d), sd, W, H, thr, None, 0, 0, 1, peers, CAP,
                                                                                  dev(recs), e)),
        ("fl_match_shard_exchange_masked_async", lambda: L.fl_match_shard_exchange_masked_async(hh, fb._p(b), sb, fb._p(d), sd, W, H, None, thr, None, 0,
                                                                                                0, 1, peers, CAP, dev(recs), e)),
        ("fl_match_shard_exchange_device_async", lambda: L.fl_match_shard_exchange_device_async(hh, dev(db), dev(dd), W, H, thr, None, 0, 0, 1, peers, CAP,
                                                                                                dev(recs), e)),
        ("fl_match_shard_exchange_device_masked_async", lambda: L.fl_match_shard_exchange_device_masked_async(hh, dev(db), dev(dd), W, H, None, thr, None, 0,
                                                                                                              0, 1, peers, CAP, dev(recs), e)),
        ("fl_recognize_async", lambda: L.fl_recognize_async(hh, fb._p(b), sb, fb._p(d), sd, W, H, W, H, fb.Intrinsics(*K))),
        ("fl_set_recognition", lambda: L.fl_set_recognition(hh, C.byref(fb.reco_params()), fb._p(crops), None)),
    ]
    return calls, keep


INTRUDERS = ["fl_match_device_async", "fl_match_async", "fl_match_rescaled", "fl_match_shard_device", "fl_sort_unique_device",
             "fl_sort_unique_blocks_device", "fl_exchange_sort_unique_device", "fl_exchange_sort_unique_device_async",
             "fl_match_shard_exchange_async", "fl_match_shard_exchange_masked_async", "fl_match_shard_exchange_device_async",
             "fl_match_shard_exchange_device_masked_async", "fl_recognize_async", "fl_set_recognition"]


@pytest.mark.parametrize("in_flight", ["match", "recognition"])
@pytest.mark.parametrize("intruder", INTRUDERS)
def test_entry_points_refuse_while_a_frame_is_in_flight(scene, in_flight, intruder):
    b, d, ts, rects, want_match, want_reco = scene
    h = _handle(ts, d, rects)
    calls, _keep = _intruders(h, b, d, ts)
    call = dict(calls)[intruder]
    n0 = h.launch_count()
    if in_flight == "match":
        h.match_async(b, d, 75.0)
    else:
        h.recognize_async(b, d, K)
    n1 = h.launch_count()
    assert call() == fb.FL_ERR_STATE
    assert h.launch_count() == n1 > n0 and fb.lib().fl_last_error()          # nothing launched, and the refusal says why
    if in_flight == "match":
        h.match_wait()
        assert h.match_fetch().tobytes() == want_match
    else:
        rc, res, summary = h.recognize_wait()
        assert rc == fb.FL_OK and (res.tobytes(), summary) == want_reco
    h.sync()
    h.close()


def test_wait_with_nothing_in_flight_says_why():
    h = fb.Handle(T, (0, 1), W, H)
    L = fb.lib()
    out = np.zeros(1, np.uint64)
    assert L.fl_debug_icp_trace(h._h, fb._p(out), 1) == fb.FL_ERR_STATE        # leaves a message of its own behind
    before = L.fl_last_error()
    assert L.fl_match_wait(h._h) == fb.FL_ERR_STATE
    assert L.fl_last_error() and L.fl_last_error() != before
    h.close()
