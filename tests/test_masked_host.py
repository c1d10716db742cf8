"""CPU: the ABI of masked frames on the throughput paths (fl_pipe_submit_masked, fl_group_match_masked,
fl_match_shard_exchange_(device_)masked_async) - the prototypes in include/fealess_b200.h against the ctypes binding, the mirrors'
mask checks, the per-stage mask kernels gone from the library, and the C++ group driver compiling against the minimal OpenCV shim."""
import os
import re
import subprocess

import numpy as np
import pytest

import fealess_b200 as fb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SHARD = ["int32_t", "int32_t", "void* const*", "int32_t", "fl_match_t*", "uint32_t"]
PROTOTYPES = {
    "fl_pipe_submit_masked": ["fl_pipe*", "const void*", "size_t", "const void*", "size_t", "int32_t", "int32_t", "const void* const*", "float",
                              "const int32_t*", "int32_t", "int32_t"],
    "fl_group_match_masked": ["fl_group*", "const uint8_t*", "size_t", "const uint16_t*", "size_t", "int32_t", "int32_t", "const uint8_t* const*",
                              "float", "const int32_t*", "int32_t", "fl_match_t*", "int32_t", "int32_t*"],
    "fl_match_shard_exchange_masked_async": ["fl_handle*", "const uint8_t*", "size_t", "const uint16_t*", "size_t", "int32_t", "int32_t",
                                             "const uint8_t* const*", "float", "const int32_t*", "int32_t"] + SHARD,
    "fl_match_shard_exchange_device_masked_async": ["fl_handle*", "const void*", "const void*", "int32_t", "int32_t", "const void* const*", "float",
                                                    "const int32_t*", "int32_t"] + SHARD,
}
# the entry point each masked one extends: the same parameters without the masks
UNMASKED = {"fl_pipe_submit_masked": "fl_pipe_submit", "fl_group_match_masked": "fl_group_match",
            "fl_match_shard_exchange_masked_async": "fl_match_shard_exchange_async",
            "fl_match_shard_exchange_device_masked_async": "fl_match_shard_exchange_device_async"}


def _header():
    return re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "fealess_b200.h")).read(), flags=re.S)


def _prototype(name):
    m = re.search(r"(\w+)\s+%s\s*\(([^)]*)\)\s*;" % name, _header())
    assert m, name
    params = [re.sub(r"\s+", " ", p.strip()) for p in m.group(2).split(",")]
    types = [re.sub(r"\s*\b\w+$", "", p).replace(" *", "*") for p in params]
    return m.group(1), types


def test_masked_prototypes_match_the_binding():
    for name, want in PROTOTYPES.items():
        ret, types = _prototype(name)
        assert ret == "int" and types == want, (name, types)
        assert name in fb.EXPORTED_SYMBOLS
        getattr(fb.lib(), name)
        _, old = _prototype(UNMASKED[name])
        mask_at = [i for i, t in enumerate(types) if t.endswith("* const*") and t != "void* const*"]
        assert len(mask_at) == 1 and types[:mask_at[0]] + types[mask_at[0] + 1:] == old, (name, old)
    src = open(os.path.join(ROOT, "fealess_b200", "__init__.py")).read() + open(os.path.join(ROOT, "fealess_b200", "sharded.py")).read()
    for name in PROTOTYPES:
        assert "lib()." + name + "(" in src, name


def test_mask_argument_checks():
    """host_masks / device_masks: the count must be the number of modalities and a host mask the frame's size (FL_ERR_SIZE, the -1
    of Detector::match); no device is touched before the check."""
    W, H = 64, 48
    ok = np.ones((H, W), np.uint8)
    assert fb.host_masks(None, 2, W, H) == (None, []) and fb.host_masks([], 2, W, H) == (None, [])
    arr, keep = fb.host_masks([ok, None], 2, W, H)
    assert len(arr) == 2 and arr[0] == keep[0].ctypes.data and arr[1] is None
    for bad in ([ok], [ok, ok, ok], [ok, np.ones((H, W + 1), np.uint8)], [np.ones((H - 1, W), np.uint8), None]):
        with pytest.raises(fb.FealessError) as e:
            fb.host_masks(bad, 2, W, H)
        assert e.value.rc == fb.FL_ERR_SIZE
    assert fb.device_masks(None, 2) is None
    assert list(fb.device_masks([0, 4096], 2)) == [None, 4096]
    with pytest.raises(fb.FealessError) as e:
        fb.device_masks([4096], 2)
    assert e.value.rc == fb.FL_ERR_SIZE
    b, d = np.zeros((H, W, 3), np.uint8), np.zeros((H, W), np.uint16)
    pipe = object.__new__(fb.Pipe)                               # the checks run before the pipe is used
    pipe.M, pipe.depth, pipe._p = 2, 1, None
    with pytest.raises(fb.FealessError) as e:
        pipe.submit(b, d, 75.0, masks=[ok])
    assert e.value.rc == fb.FL_ERR_SIZE
    with pytest.raises(fb.FealessError) as e:
        pipe.submit_device(0, 0, W, H, 75.0, d_masks=[0, 0, 0])
    assert e.value.rc == fb.FL_ERR_SIZE
    group = object.__new__(fb.Group)
    group.M, group._g = 2, None
    rc, got = group.match(b, d, 75.0, masks=[ok])
    assert rc == fb.FL_ERR_SIZE and len(got) == 0
    rc, got = group.match(b, d, 75.0, masks=[ok, ok[:, :-1]])
    assert rc == fb.FL_ERR_SIZE and len(got) == 0
    assert fb.Detector().match([b, d], 75.0, masks=[ok]) == (-1, [])


def test_no_per_stage_mask_kernels():
    """A masked frame runs the front end's own schedule: the per-stage kernels of the old masked path are gone, and nothing on the
    frame path grows a mask buffer."""
    csrc = os.path.join(ROOT, "fealess_b200", "csrc")
    text = "".join(open(os.path.join(csrc, f)).read() for f in os.listdir(csrc))
    for gone in ("k_apply_mask", "k_spread_lm", "k_pyrdown_bgr", "fl_launch_apply_mask", "fl_launch_spread_lm", "fl_launch_pyrdown_bgr", "d_qm"):
        assert gone not in text, gone
    api = open(os.path.join(csrc, "api.cu")).read()
    assert not re.search(r"d_mask\[[^\]]*\]\[[^\]]*\]\.grow", api)
    so = fb.library_path()
    if os.path.exists(so):
        syms = subprocess.run(["nm", "-D", "-C", so], capture_output=True, text=True).stdout
        assert "k_apply_mask" not in syms and "k_spread_lm" not in syms and "k_pyrdown_bgr" not in syms


def test_cpp_masked_group_driver_compiles(tmp_path):
    from fealess_b200 import build as fbuild
    fbuild.build()
    exe = str(tmp_path / "masked_group_test")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    r = subprocess.run([cxx, "-std=c++11", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "masked_group_test.cpp"), "-o", exe, fb.library_path(),
                        "-Wl,-rpath," + os.path.dirname(fb.library_path())], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([exe], capture_output=True, text=True)          # no case file: prints usage, touches no GPU
    assert r.returncode == 2 and "usage" in r.stdout
