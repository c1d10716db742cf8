"""The frame in flight on a handle lives in one record (fl_frame in fealess_b200/csrc/api.cu): every entry point that enqueues frame work
starts with the same in-flight check, and the group waits through fl_frame_wait instead of inferring a front-end re-run from the debug
options.  Loose per-frame fields kept in step by hand let entry points overwrite each other's frames."""
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "fealess_b200", "csrc")
IN_FLIGHT = '"a frame is in flight on this handle'


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


def test_handle_has_no_loose_pending_fields():
    code = _code("api.cu")
    assert re.findall(r"\bpend_\w+", _struct_body(code, "fl_handle")) == []
    assert re.findall(r"\bpend_\w+", code) == []
    assert re.search(r"\bfl_frame\s+frame\b", _struct_body(code, "fl_handle"))


def test_group_does_not_infer_reruns_from_debug_options():
    assert "fl_debug_option" not in _code("group.cu")
    assert "fl_recognition_pending" not in _code("pipe.cu")


def test_one_in_flight_message():
    code = _code("api.cu")
    assert code.count(IN_FLIGHT) == 1
    for old in ("has not been called for the previous frame", "has not been waited for", "a frame is in flight on this handle\""):
        assert old not in code, old
