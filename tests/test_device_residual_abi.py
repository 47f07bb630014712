"""h263cu_decode_step_device_residual without a GPU: the ctypes layout against the header and the Rust declarations,
the entry points, the import without torch, the shapes residual=True allocates and the Python argument rules."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

from h263_rs_b200 import _lib, api, frontend, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["y", "y_stride", "cb", "cb_stride", "cr", "cr_stride", "width", "height", "stream"]


def header():
    return open(os.path.join(ROOT, "include", "h263cu.h")).read()


def test_layout_matches_the_header():
    h = header()
    assert "typedef struct h263cu_device_residual { /* 112 bytes */" in h
    assert C.sizeof(_lib.DeviceResidual) == 112
    offsets = {f: getattr(_lib.DeviceResidual, f).offset for f, _ in _lib.DeviceResidual._fields_}
    assert offsets == dict(y=0, y_stride=8, cb=32, cb_stride=40, cr=64, cr_stride=72, width=96, height=100, stream=104)
    body = re.search(r"typedef struct h263cu_device_residual \{(.*?)\} h263cu_device_residual;", h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"\*?\s*(\w+)(?:\[\d\])?(?:, (\w+))?;", body)
    assert [n for pair in names for n in pair if n] == FIELDS == [f for f, _ in _lib.DeviceResidual._fields_]


def test_entry_points():
    h, L = header(), _lib.lib()
    for name in ("h263cu_decode_step_device_residual", "h263cu_group_decode_step_device_residual"):
        assert name in _lib.SYMBOLS and hasattr(L, name)
        assert re.search(r"int %s\(h263cu_\w+\*, h263cu_parser\* const\* parsers" % name, h)
    # the motion call points at the residual call instead of leaving it out
    assert "the prediction residual. */" not in h and "h263cu_decode_step_device_residual below" in h


def test_rust_declarations():
    rs = open(os.path.join(ROOT, "bindings", "h263cu-sys", "src", "lib.rs")).read()
    assert "pub struct h263cu_device_residual {" in rs and "size_of::<h263cu_device_residual>(), 112" in rs
    assert "pub fn h263cu_decode_step_device_residual(" in rs and "pub fn h263cu_group_decode_step_device_residual(" in rs
    body = re.search(r"pub struct h263cu_device_residual \{(.*?)\}", rs, re.S).group(1)
    assert re.findall(r"pub (\w+):", body) == FIELDS


def test_api_imports_without_torch():
    code = ("import sys; sys.modules['torch'] = None\n"
            "from h263_rs_b200 import api\n"
            "print(api.residual_shapes(3, 352, 288))\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Residual(y=(3, 288, 352), cb=(3, 144, 176), cr=(3, 144, 176))" in r.stdout


@pytest.mark.parametrize("w,h", [(352, 288), (176, 144), (161, 99), (15, 15), (1, 1)])
def test_allocation_shapes(w, h):
    s = api.residual_shapes(5, w, h)
    assert isinstance(s, api.Residual)
    assert s.y == (5, h, w) and s.cb == s.cr == (5, -(-h // 2), -(-w // 2))


def test_methods_refuse_a_bad_keyword_before_any_parser_moves():
    dec = api.BatchDecoder.__new__(api.BatchDecoder)
    dec.n, dec.threads, dec.ctx = 1, 1, None
    dec.parsers = [frontend.Parser(1)]
    pk = synth.make_stream(176, 144, 1, 1)
    for call in (lambda: dec.decode_step_device_residual(pk, parse="gpu"),
                 lambda: dec.decode_step_device(pk, parse="gpu", residual=True),
                 lambda: dec.decode_step_device_yuv(pk, parse="gpu", residual=True),
                 lambda: dec.decode_step_device_tensor(pk, (8, 8), parse="gpu", residual=True, motion=True)):
        with pytest.raises(ValueError):
            call()


def test_python_argument_rules_without_a_gpu():
    torch = pytest.importorskip("torch")
    for bad in (api.Residual(None, None, None), (1, 2), 5, api.Residual(torch.zeros((1, 4, 4), dtype=torch.int16), None, None)):
        with pytest.raises(ValueError):
            api._device_residual(bad, 1, 16, 16, 0)
