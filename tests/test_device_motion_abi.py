"""h263cu_decode_step_device_motion without a GPU: the ctypes layouts against the header, the constant, the Rust
declarations, the import without torch and the shapes motion=True allocates."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

from h263_rs_b200 import _lib, api, frontend, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header():
    return open(os.path.join(ROOT, "include", "h263cu.h")).read()


def test_layouts_match_the_header():
    h = header()
    assert "typedef struct h263cu_device_motion { /* 120 bytes */" in h
    assert "typedef struct h263cu_device_output { /* 40 bytes */" in h
    assert C.sizeof(_lib.DeviceMotion) == 120 and C.sizeof(_lib.DeviceOutput) == 40
    offsets = {f: getattr(_lib.DeviceMotion, f).offset for f, _ in _lib.DeviceMotion._fields_}
    assert offsets == dict(mv=0, mv_stride=8, mb_flags=40, flags_stride=48, mb_quant=72, quant_stride=80, mb_width=104,
                           mb_height=108, stream=112)
    offsets = {f: getattr(_lib.DeviceOutput, f).offset for f, _ in _lib.DeviceOutput._fields_}
    assert offsets == dict(rgba=0, yuv=8, tensor=16, fit=24, filter=32, reserved=36)
    # the header's field order is the ctypes order
    body = re.search(r"typedef struct h263cu_device_motion \{(.*?)\} h263cu_device_motion;", h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"\*?\s*(\w+)(?:\[\d\])?(?:, (\w+))?;", body)
    flat = [n for pair in names for n in pair if n]
    assert flat == [f for f, _ in _lib.DeviceMotion._fields_]


def test_constant_and_entry_points():
    assert re.search(r"#define H263CU_MOTION_OUTSIDE 0x80u", header())
    assert _lib.MOTION_OUTSIDE == 0x80
    # the outside mark does not collide with the exported flags
    assert _lib.MOTION_OUTSIDE & (_lib.MB_INTER | _lib.MB_FOURMV | _lib.MB_CODED | _lib.MB_WIDE) == 0
    L = _lib.lib()
    for name in ("h263cu_decode_step_device_motion", "h263cu_group_decode_step_device_motion"):
        assert name in _lib.SYMBOLS and name in header() and hasattr(L, name)


def test_rust_declarations():
    rs = open(os.path.join(ROOT, "bindings", "h263cu-sys", "src", "lib.rs")).read()
    assert "pub const H263CU_MOTION_OUTSIDE: u32 = 0x80;" in rs
    assert "pub struct h263cu_device_motion {" in rs and "pub struct h263cu_device_output {" in rs
    assert "pub fn h263cu_decode_step_device_motion(" in rs and "pub fn h263cu_group_decode_step_device_motion(" in rs
    assert "size_of::<h263cu_device_motion>(), 120" in rs and "size_of::<h263cu_device_output>(), 40" in rs
    body = re.search(r"pub struct h263cu_device_motion \{(.*?)\}", rs, re.S).group(1)
    assert re.findall(r"pub (\w+):", body) == [f for f, _ in _lib.DeviceMotion._fields_]


def test_api_imports_without_torch():
    code = ("import sys; sys.modules['torch'] = None\n"
            "from h263_rs_b200 import api\n"
            "print(api.motion_shapes(3, 352, 288))\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Motion(mv=(3, 2, 36, 44), flags=(3, 18, 22), quant=(3, 18, 22))" in r.stdout


@pytest.mark.parametrize("w,h", [(352, 288), (176, 144), (161, 99), (15, 15), (4080, 4080)])
def test_allocation_shapes(w, h):
    mbw, mbh = -(-w // 16), -(-h // 16)
    s = api.motion_shapes(5, w, h)
    assert isinstance(s, api.Motion)
    assert s.mv == (5, 2, 2 * mbh, 2 * mbw) and s.flags == (5, mbh, mbw) and s.quant == (5, mbh, mbw)


def test_methods_refuse_a_bad_keyword_before_any_parser_moves():
    dec = api.BatchDecoder.__new__(api.BatchDecoder)
    dec.n, dec.threads, dec.ctx = 1, 1, None
    dec.parsers = [frontend.Parser(1)]
    pk = synth.make_stream(176, 144, 1, 1)
    for call in (lambda: dec.decode_step_device_motion(pk, parse="gpu"), lambda: dec.decode_step_device(pk, parse="gpu", motion=True),
                 lambda: dec.decode_step_device_tensor(pk, (8, 8), parse="gpu", motion=True)):
        with pytest.raises(ValueError):
            call()
