"""The host side of device plane output, checked without a GPU: the ctypes twins of h263cu_device_plane and
h263cu_device_yuv match the header's layout, the Rust -sys crate declares the entry points and structs, and the
Python API still imports without torch (torch is imported by decode_step_device_yuv only)."""
import ctypes as C
import os
import re
import subprocess
import sys

from h263_rs_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_fields(name):
    text = open(os.path.join(ROOT, "include", "h263cu.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return re.findall(r"\b([a-z_]+)(?:\[\d+\])?\s*[,;]", body)


def test_device_plane_layout():
    P = _lib.DevicePlane
    assert C.sizeof(P) == 24
    assert [(f, getattr(P, f).offset) for f, _ in P._fields_] == [("base", 0), ("row_pitch", 8), ("pic_stride", 16)]
    assert _header_fields("h263cu_device_plane") == [f for f, _ in P._fields_]


def test_device_yuv_layout():
    D = _lib.DeviceYuv
    assert C.sizeof(D) == 96
    assert [(f, getattr(D, f).offset) for f, _ in D._fields_] == [
        ("plane", 0), ("width", 72), ("height", 76), ("format", 80), ("reserved", 84), ("stream", 88)]
    assert _header_fields("h263cu_device_yuv") == [f for f, _ in D._fields_]


def test_format_constants_match_the_header():
    text = open(os.path.join(ROOT, "include", "h263cu.h")).read()
    consts = dict(re.findall(r"#define (H263CU_YUV_\w+) (\d+)u", text))
    assert consts == {"H263CU_YUV_I420": str(_lib.YUV_I420), "H263CU_YUV_NV12": str(_lib.YUV_NV12)}


def test_rust_binding_declares_the_entry_points_and_structs():
    text = open(os.path.join(ROOT, "bindings", "h263cu-sys", "src", "lib.rs")).read()
    for name in ("h263cu_decode_step_device_yuv", "h263cu_group_decode_step_device_yuv", "h263cu_device_yuv",
                 "h263cu_device_plane", "H263CU_YUV_I420", "H263CU_YUV_NV12"):
        assert name in text, name


def test_api_imports_without_torch():
    code = ("import sys; sys.modules['torch'] = None; sys.path.insert(0, %r); from h263_rs_b200 import api; "
            "print(api.BatchDecoder.decode_step_device_yuv.__name__, api.DeviceGroup.decode_step_device_yuv.__name__)" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.split() == ["decode_step_device_yuv"] * 2, out.stderr
