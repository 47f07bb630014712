"""The host side of device-resident output, checked without a GPU: the ctypes twin of h263cu_device_rgba matches the
header's layout, and the Python API still imports without torch (torch is imported by decode_step_device only)."""
import ctypes as C
import os
import re
import subprocess
import sys

from h263_rs_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_device_rgba_layout():
    D = _lib.DeviceRgba
    assert C.sizeof(D) == 40
    assert [(f, getattr(D, f).offset) for f, _ in D._fields_] == [
        ("base", 0), ("row_pitch", 8), ("pic_stride", 16), ("width", 24), ("height", 28), ("stream", 32)]
    text = open(os.path.join(ROOT, "include", "h263cu.h")).read()
    body = re.search(r"typedef struct h263cu_device_rgba \{(.*?)\} h263cu_device_rgba;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"\b([a-z_]+)\s*[,;]", body)
    assert names == [f for f, _ in D._fields_]


def test_rust_binding_declares_the_device_entry_points():
    text = open(os.path.join(ROOT, "bindings", "h263cu-sys", "src", "lib.rs")).read()
    for name in ("h263cu_decode_step_device", "h263cu_group_decode_step_device", "h263cu_device_rgba"):
        assert name in text, name


def test_api_imports_without_torch():
    code = "import sys; sys.modules['torch'] = None; sys.path.insert(0, %r); from h263_rs_b200 import api; print(api.BatchDecoder.decode_step_device.__name__)" % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert out.returncode == 0 and "decode_step_device" in out.stdout, out.stderr
