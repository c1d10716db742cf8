"""CPU: the ABI of Recognition on the device (fl_set_recognition, fl_recognize*, fl_pipe_*_recognition) - struct layouts against
include/fealess_b200.h, no CPU fallback, and the C++ stream methods of CObjRecoLmICP compile cleanly against the minimal OpenCV shim."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import fealess_b200 as fb
from fealess_b200 import reco, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header():
    return re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "fealess_b200.h")).read(), flags=re.S)


def _struct_fields(name):
    body = re.search(r"typedef struct \{([^{}]*)\}\s*%s;" % name, _header()).group(1)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        typ, names = decl.split(None, 1)
        for n in names.split(","):
            m = re.match(r"\s*(\w+)(?:\[(\w+)\])?", n)
            fields.append((typ, m.group(1), m.group(2)))
    return fields


def test_reco_structs_match_the_header():
    assert [f[1] for f in _struct_fields("fl_reco_result_t")] == list(fb.RECO_RESULT_DTYPE.names)
    assert fb.RECO_RESULT_DTYPE.itemsize == 4 * 6 + 16 * 4 + fb.ICP_RESULT_DTYPE.itemsize == 156
    assert fb.RECO_RESULT_DTYPE["world2cam"].shape == (16,) and fb.RECO_RESULT_DTYPE.fields["icp"][0] == fb.ICP_RESULT_DTYPE
    assert [f[1] for f in _struct_fields("fl_reco_summary_t")] == [f[0] for f in fb.RecoSummary._fields_]
    assert ctypes.sizeof(fb.RecoSummary) == 16
    assert [f[1] for f in _struct_fields("fl_reco_params_t")] == [f[0] for f in fb.RecoParams._fields_]
    assert ctypes.sizeof(fb.RecoParams) == 4 + 12 + 4 + 4 + 4
    assert re.search(r"#define FL_RECO_MAX_HYP (\d+)", _header()).group(1) == str(fb.RECO_MAX_HYP)


def test_default_reco_params_are_the_references():
    p = fb.RecoParams()
    fb.lib().fl_default_reco_params(ctypes.byref(p))
    assert (p.threshold, p.icp.icp_it_thr, p.top_k, p.per_class, p.th_obj_dist) == (75.0, 10, 1, 0, 0.0)
    assert np.float32(p.icp.dist_mean_thr) == np.float32(0.5) and np.float32(p.icp.dist_diff_thr) == np.float32(0.01)
    q = fb.reco_params()
    assert bytes(q) == bytes(p)


def test_recognition_without_a_device_fails_with_cuda_error():
    """fl_recognize needs a handle (or a pipe of handles), and fl_create / fl_pipe_create fail with FL_ERR_CUDA without a device:
    every way to the recognition path - Handle.recognize, Pipe.submit_recognition, ObjRecoLmICP.submit - stops there, with no
    fallback.  The C entry points themselves refuse a missing handle or pipe."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = fb.lib()
    K = fb.Intrinsics(608, 608, 320, 240)
    assert L.fl_recognize(None, None, 0, None, 0, 640, 480, 640, 480, K, None, 0, None) == fb.FL_ERR_ARG
    assert L.fl_set_recognition(None, None, None, None) == fb.FL_ERR_ARG
    assert L.fl_pipe_submit_recognition(None, None, 0, None, 0, 640, 480, 640, 480, K) == fb.FL_ERR_ARG
    assert L.fl_pipe_collect_recognition(None, None, 0, None) == fb.FL_ERR_ARG
    for make in (lambda: fb.Handle(), lambda: fb.Pipe(2)):
        with pytest.raises(fb.FealessError) as e:
            make()
        assert e.value.rc == fb.FL_ERR_CUDA
    o = reco.ObjRecoLmICP(frames_in_flight=2)
    det = fb.Detector()
    det.add_template_set(synth.make_templates(4, n_classes=1, seed=5))
    b, d = synth.make_frame(640, 480, 0)
    K = dict(fx=608.0, fy=608.0, cx=320.0, cy=240.0, width=640, height=480)
    o.add_detector(det, {(None, 0): d})
    with pytest.raises(fb.FealessError) as e:                   # the pipe behind submit cannot be created
        o.submit(b, d, K)
    assert e.value.rc == fb.FL_ERR_CUDA
    with pytest.raises(fb.FealessError) as e:
        o.collect()
    assert e.value.rc == fb.FL_ERR_STATE


def test_stream_submit_rejects_what_recognition_rejects():
    """Argument checks of ObjRecoLmICP.submit before anything reaches the device, as Recognition returns them: sizes that disagree,
    and a one-modality detector at 640 columns (Recognition hands match() two sources there: -1, linemod.cpp:1364-1367)."""
    b, d = synth.make_frame(640, 480, 0)
    K = dict(fx=608.0, fy=608.0, cx=320.0, cy=240.0, width=640, height=480)
    o = reco.ObjRecoLmICP()
    assert o.submit(b, d, K) == reco.ERROR_INVALID_PARAM        # no object
    det = fb.Detector()
    det.add_template_set(synth.make_templates(4, n_classes=1, seed=5))
    o.add_detector(det, {(None, 0): d})
    assert o.submit(b, d[:100], K) == reco.ERROR_INVALID_PARAM
    assert o.submit(b, d, dict(K, width=320)) == reco.ERROR_INVALID_PARAM
    o.add_detector(fb.Detector(modalities=("DepthNormal",)), {(None, 0): d})
    assert o.submit(b, d, K) == reco.ERROR_INVALID_PARAM and o.in_flight() == 0


def test_cpp_stream_driver_compiles_cleanly():
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    r = subprocess.run([cxx, "-std=c++11", "-fsyntax-only", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "reco_stream_test.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
