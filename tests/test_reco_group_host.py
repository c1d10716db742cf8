"""CPU: the ABI of Recognition over a template-sharded group (fl_group_create_pipe, fl_group_*_recognition) - the prototypes in
include/fealess_b200.h against the ctypes binding, the argument checks of fl_group_create_pipe, no CPU fallback, and the C++ driver
of CObjRecoLmICP::SetDevices compiles cleanly against the minimal OpenCV shim."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import fealess_b200 as fb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FL_PIPE_MAX_DEPTH = 8

# the new entry points and the C parameter types the binding passes them
PROTOTYPES = {
    "fl_group_create_pipe": ["const fl_params_t*", "const int32_t*", "int32_t", "int32_t", "int32_t", "fl_group**"],
    "fl_group_depth": ["const fl_group*"],
    "fl_group_in_flight": ["const fl_group*"],
    "fl_group_upload_model_depths": ["fl_group*", "int32_t", "const uint16_t* const*", "const size_t*", "const fl_rect_t*", "int32_t", "int32_t"],
    "fl_group_set_recognition": ["fl_group*", "const fl_reco_params_t*", "const int32_t*", "const float*"],
    "fl_group_submit_recognition": ["fl_group*", "const uint8_t*", "size_t", "const uint16_t*", "size_t", "int32_t", "int32_t", "int32_t", "int32_t",
                                    "fl_intrinsics_t"],
    "fl_group_collect_recognition": ["fl_group*", "fl_reco_result_t*", "int32_t", "fl_reco_summary_t*"],
    "fl_group_recognize": ["fl_group*", "const uint8_t*", "size_t", "const uint16_t*", "size_t", "int32_t", "int32_t", "int32_t", "int32_t",
                           "fl_intrinsics_t", "fl_reco_result_t*", "int32_t", "fl_reco_summary_t*"],
}
RETURNS = {"fl_group_depth": "int32_t", "fl_group_in_flight": "int32_t"}


def _header():
    return re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "fealess_b200.h")).read(), flags=re.S)


def _prototype(name):
    m = re.search(r"(\w+)\s+%s\s*\(([^)]*)\)\s*;" % name, _header())
    assert m, name
    params = [re.sub(r"\s+", " ", p.strip()) for p in m.group(2).split(",")]
    types = [re.sub(r"\s*\b\w+$", "", p).replace(" *", "*") for p in params]
    return m.group(1), types


def test_group_recognition_prototypes_match_the_binding():
    for name, want in PROTOTYPES.items():
        ret, types = _prototype(name)
        assert ret == RETURNS.get(name, "int"), name
        assert types == want, (name, types)
        assert name in fb.EXPORTED_SYMBOLS
        getattr(fb.lib(), name)
    # the shape the Python methods hand over: summary and params structs of the header, Group exposes every entry
    for meth in ("in_flight", "upload_model_depths", "set_recognition", "submit_recognition", "collect_recognition", "recognize"):
        assert callable(getattr(fb.Group, meth))
    assert re.search(r"#define FL_PIPE_MAX_DEPTH (\d+)", _header()).group(1) == str(FL_PIPE_MAX_DEPTH)


def test_group_create_pipe_argument_checks():
    """Checked before anything touches a device: a depth outside 1 .. FL_PIPE_MAX_DEPTH, more than 8 members and NULL pointers are
    FL_ERR_ARG, and the group pointer is left NULL."""
    L = fb.lib()
    p = fb.Params()
    L.fl_default_params(C.byref(p))
    dv = np.zeros(9, np.int32)
    g = C.c_void_p(1234)
    for n, cap, depth in ((2, 64, 0), (2, 64, FL_PIPE_MAX_DEPTH + 1), (2, 64, -1), (9, 64, 1), (0, 64, 1), (2, 0, 1)):
        g.value = 1234
        assert L.fl_group_create_pipe(C.byref(p), dv.ctypes.data_as(C.c_void_p), n, cap, depth, C.byref(g)) == fb.FL_ERR_ARG, (n, cap, depth)
        assert not g.value, (n, cap, depth)
    assert L.fl_group_create_pipe(None, dv.ctypes.data_as(C.c_void_p), 2, 64, 2, C.byref(g)) == fb.FL_ERR_ARG
    assert L.fl_group_create_pipe(C.byref(p), None, 2, 64, 2, C.byref(g)) == fb.FL_ERR_ARG
    assert L.fl_group_create_pipe(C.byref(p), dv.ctypes.data_as(C.c_void_p), 2, 64, 2, None) == fb.FL_ERR_ARG
    # the other entry points refuse a missing group
    K = fb.Intrinsics(608, 608, 320, 240)
    assert L.fl_group_depth(None) == 0 and L.fl_group_in_flight(None) == 0
    assert L.fl_group_upload_model_depths(None, 0, None, None, None, 640, 480) == fb.FL_ERR_ARG
    assert L.fl_group_set_recognition(None, None, None, None) == fb.FL_ERR_ARG
    assert L.fl_group_submit_recognition(None, None, 0, None, 0, 640, 480, 640, 480, K) == fb.FL_ERR_ARG
    assert L.fl_group_collect_recognition(None, None, 0, None) == fb.FL_ERR_ARG
    assert L.fl_group_recognize(None, None, 0, None, 0, 640, 480, 640, 480, K, None, 0, None) == fb.FL_ERR_ARG


def test_group_create_pipe_without_a_device_fails_with_cuda_error():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = fb.lib()
    p = fb.Params()
    L.fl_default_params(C.byref(p))
    for devices in ([0, 0], [0, 1]):
        dv = np.array(devices, np.int32)
        g = C.c_void_p(1234)
        assert L.fl_group_create_pipe(C.byref(p), dv.ctypes.data_as(C.c_void_p), len(devices), 64, 4, C.byref(g)) == fb.FL_ERR_CUDA
        assert not g.value
    with pytest.raises(fb.FealessError) as e:
        fb.Group([0, 0], depth=4)
    assert e.value.rc == fb.FL_ERR_CUDA


def test_cpp_group_driver_compiles_cleanly():
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    r = subprocess.run([cxx, "-std=c++11", "-fsyntax-only", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "reco_group_test.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
