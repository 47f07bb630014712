"""H263CU_PARSE_ON_DEVICE without a GPU: the constant and the test hook agree between the header, ctypes and the Rust
crate, the parse= keyword is validated before anything runs, the device parse's table layout matches the host
parser's tables, and there is no CPU fallback."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from h263_rs_b200 import _lib, api, frontend, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header():
    return open(os.path.join(ROOT, "include", "h263cu.h")).read()


def test_constant_and_hook_are_declared_everywhere():
    assert re.search(r"#define H263CU_PARSE_ON_DEVICE 4u", header())
    assert _lib.PARSE_ON_DEVICE == 4
    assert "h263cu_test_device_parse_step" in _lib.SYMBOLS
    assert hasattr(_lib.lib(), "h263cu_test_device_parse_step")
    rs = open(os.path.join(ROOT, "bindings", "h263cu-sys", "src", "lib.rs")).read()
    assert "pub const H263CU_PARSE_ON_DEVICE: u32 = 4;" in rs
    assert "pub fn h263cu_test_device_parse_step(" in rs
    # the new bit does not collide with the output bits
    assert _lib.PARSE_ON_DEVICE & (_lib.OUT_RGBA | _lib.OUT_DEBLOCK) == 0


def test_table_layout_matches_the_host_tables():
    """parse_mb.h's table widths are the longest codes of the host parser's tables (the TCOEF table adds the sign)."""
    text = open(os.path.join(ROOT, "h263_rs_b200", "csrc", "parse_mb.h")).read()
    bits = dict(re.findall(r"PT_(\w+)_BITS = (\d+)", text))
    L = _lib.lib()
    for table, name in ((0, "MCBPC_I"), (1, "MCBPC_P"), (2, "CBPY"), (3, "MVD"), (4, "TCOEF")):
        codes = re.search(r"%s_CODES\[\]\s*=\s*\{(.*?)\};" % name,
                          open(os.path.join(ROOT, "h263_rs_b200", "csrc", "vlc_codes.inc")).read(), re.S).group(1)
        longest = max(len(c) for c in re.findall(r'\{"([01]+)"', codes))
        assert int(bits[name]) == longest + (1 if name == "TCOEF" else 0), name
    words = sum(1 << int(v) for v in bits.values())
    assert words * 4 == 100608  # 98.25 KiB, the figure the kernel's shared-memory budget is built on


@pytest.mark.parametrize("bad", ["gpu", "HOST", "", None, 1, True, b"device"])
def test_parse_keyword_is_validated(bad):
    with pytest.raises(ValueError):
        api._parse_flag(bad)
    assert api._parse_flag("host") == 0 and api._parse_flag("device") == _lib.PARSE_ON_DEVICE


def test_methods_refuse_a_bad_keyword_before_any_parser_moves():
    """A decoder object without a context (no GPU here): the keyword is checked before anything touches it."""
    dec = api.BatchDecoder.__new__(api.BatchDecoder)
    dec.n, dec.threads, dec.ctx = 1, 1, None
    dec.parsers = [frontend.Parser(1)]
    pk = synth.make_stream(176, 144, 1, 1)
    for call in (lambda: dec.decode_step(pk, parse="gpu"), lambda: dec.decode_step_device(pk, parse="gpu"),
                 lambda: dec.decode_step_device_yuv(pk, parse="gpu"), lambda: dec.decode_step_device_tensor(pk, (8, 8), parse="gpu")):
        with pytest.raises(ValueError):
            call()
    grp = api.DeviceGroup.__new__(api.DeviceGroup)
    grp.h = None
    for call in (lambda: grp.decode_step(pk, parse="gpu"), lambda: grp.decode_step_device(pk, parse="gpu"),
                 lambda: grp.decode_step_device_yuv(pk, parse="gpu"), lambda: grp.decode_step_device_tensor(pk, (8, 8), parse="gpu")):
        with pytest.raises(ValueError):
            call()


def test_no_cpu_fallback_without_a_device():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a device is present")
    L = _lib.lib()
    err = C.c_int(0)
    assert not L.h263cu_create(0, 1, 176, 144, 0, C.byref(err)) and err.value == _lib.ERR_NO_DEVICE
    with pytest.raises(_lib.H263Error) as e:
        api.BatchDecoder(1, 176, 144)
    assert e.value.code == _lib.ERR_NO_DEVICE
    # the hook needs a context: without one it parses nothing, and the parser does not move
    p = frontend.Parser(1)
    pk = synth.make_stream(176, 144, 2, 1)
    with pytest.raises(_lib.H263Error) as e:
        frontend.parse_step([p], [pk[0]], ctx=type("NoCtx", (), {"h": None})())
    assert e.value.code == _lib.ERR_BAD_ARGUMENT
    with pytest.raises(_lib.H263Error) as e:
        frontend.Parser(1).parse_picture(pk[1])  # a fresh parser has no reference ...
    pics, mbs, ev, errs, _ = frontend.parse_step([p], [pk[1]])
    assert errs[0] == -15  # ... and neither has this one: the hook did not advance it
