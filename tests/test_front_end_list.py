"""The front end of a frame is one job list built in fealess_b200/csrc/frontend.cu, launched as one grid or wave by wave from that list,
and its per-handle state (dependency counters and their bases, the time-out flag, the job timeline) belongs to frontend.cu.  api.cu only
describes the frame: a change to a job, or to the in-grid counter protocol, touches one file."""
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "fealess_b200", "csrc")
# the same allocator pattern as tests/test_handle_ownership.py
RESOURCE_CALL = re.compile(r"\b(cudaMalloc\w*|cudaFree\w*|cudaHostAlloc|cudaEvent(?:Create\w*|Destroy)|cudaStream(?:Create\w*|Destroy))\s*\(")


def _code(name):
    with open(os.path.join(CSRC, name)) as f:
        src = f.read()
    return re.sub(r"//[^\n]*", "", re.sub(r"/\*.*?\*/", "", src, flags=re.S))


def _struct_body(code, name):
    start = code.index("struct %s {" % name)
    depth, i = 0, code.index("{", start)
    for j in range(i, len(code)):
        depth += {"{": 1, "}": -1}.get(code[j], 0)
        if depth == 0:
            return code[i:j]
    raise AssertionError("unterminated struct " + name)


def test_api_cu_builds_no_front_end_job():
    code = _code("api.cu")
    for word in ("fl_fe_add_", "fl_launch_fe_wave", "wait_slot", "wait_target", "wait_row_", "row_base", "signal_slot"):
        assert word not in code, word
    assert len(re.findall(r"\bfl_fe_run\s*\(", code)) == 1


def test_handle_has_no_front_end_counters():
    body = _struct_body(_code("api.cu"), "fl_handle")
    for field in ("d_fe_counters", "fe_counter_base", "fe_row_base", "h_fe_err"):
        assert not re.search(r"\b%s\b" % field, body), field


def test_frontend_cu_calls_no_allocator_directly():
    code = _code("frontend.cu")
    assert '#include "fl_owned.cuh"' in code
    calls = sorted(set(RESOURCE_CALL.findall(code)))
    assert calls == [], "frontend.cu calls %s; use an owner from fl_owned.cuh" % ", ".join(calls)
