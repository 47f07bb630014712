"""The host side of device tensor output, checked without a GPU: the ctypes twin of h263cu_device_tensor matches the
header's layout, the dtype constants and the Rust -sys crate agree, the Python API still imports without torch; and the
output's definition (include/h263cu.h) is the familiar one: its numpy restatement (resample_ref.py) stays within a few
ulp of torch's bilinear interpolation, and the arithmetic the kernel compiles (device_math.cuh) equals the restatement
bit for bit."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import resample_ref as R
from h263_rs_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))

# (h, w) -> (H, W): downscales, upscales, identities, mixed, and the degenerate 1-sample axes
SIZE_PAIRS = [((288, 352), (224, 224)), ((144, 176), (288, 352)), ((120, 160), (75, 100)), ((15, 15), (1, 1)),
              ((15, 15), (37, 53)), ((99, 161), (99, 161)), ((1, 1), (5, 3)), ((31, 47), (64, 20)), ((7, 300), (13, 2)),
              ((576, 704), (224, 224))]


def _header_fields(name):
    text = open(os.path.join(ROOT, "include", "h263cu.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return re.findall(r"\b([a-z_0-9]+)(?:\[\d+\])?\s*[,;]", body)


def test_device_tensor_layout():
    D = _lib.DeviceTensor
    assert C.sizeof(D) == 88
    assert [(f, getattr(D, f).offset) for f, _ in D._fields_] == [
        ("base", 0), ("stride", 8), ("width", 40), ("height", 44), ("dtype", 48), ("reserved", 52), ("mul", 56),
        ("add", 68), ("stream", 80)]
    assert _header_fields("h263cu_device_tensor") == [f for f, _ in D._fields_]


def test_dtype_constants_match_the_header():
    text = open(os.path.join(ROOT, "include", "h263cu.h")).read()
    consts = dict(re.findall(r"#define (H263CU_TENSOR_\w+) (\d+)u", text))
    assert consts == {"H263CU_TENSOR_U8": str(_lib.TENSOR_U8), "H263CU_TENSOR_F32": str(_lib.TENSOR_F32),
                      "H263CU_TENSOR_F16": str(_lib.TENSOR_F16), "H263CU_TENSOR_BF16": str(_lib.TENSOR_BF16)}


def test_rust_binding_declares_the_entry_points_and_struct():
    text = open(os.path.join(ROOT, "bindings", "h263cu-sys", "src", "lib.rs")).read()
    for name in ("h263cu_decode_step_device_tensor", "h263cu_group_decode_step_device_tensor"):
        assert "pub fn %s(" % name in text, name
    body = re.search(r"pub struct h263cu_device_tensor \{(.*?)\}", text, re.S).group(1)
    assert re.findall(r"pub (\w+):", body) == [f for f, _ in _lib.DeviceTensor._fields_]
    for k, v in (("U8", 0), ("F32", 1), ("F16", 2), ("BF16", 3)):
        assert "pub const H263CU_TENSOR_%s: u32 = %d;" % (k, v) in text


def test_symbols_are_listed():
    assert {"h263cu_decode_step_device_tensor", "h263cu_group_decode_step_device_tensor"} <= set(_lib.SYMBOLS)


def test_api_imports_without_torch():
    code = ("import sys; sys.modules['torch'] = None; sys.path.insert(0, %r); from h263_rs_b200 import api; "
            "print(api.BatchDecoder.decode_step_device_tensor.__name__, api.DeviceGroup.decode_step_device_tensor.__name__)" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.split() == ["decode_step_device_tensor"] * 2, out.stderr


def test_identity_size_is_the_picture():
    rng = np.random.default_rng(1)
    rgb = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    v = R.resample(rgb, 37, 53)
    assert np.array_equal(v, rgb.transpose(2, 0, 1).astype(np.float32))
    assert np.array_equal(R.store(v, u8=True), rgb.transpose(2, 0, 1))


def _taps_contracted(n_in, n_out):
    """axis_taps with s = scale * (X + 0.5) - 0.5 rounded once, as one FMA: torch's CPU kernel contracts it so."""
    F = np.float32
    scale = F(n_in) / F(n_out)
    s = np.maximum((np.float64(scale) * (np.arange(n_out) + 0.5) - 0.5).astype(F), F(0))
    i0 = s.astype(np.int32)
    l1 = s - i0.astype(F)
    return i0, i0 + (i0 < n_in - 1).astype(np.int32), F(1) - l1, l1


@pytest.mark.parametrize("src,dst", SIZE_PAIRS)
def test_restatement_is_torch_bilinear(src, dst):
    """torch's F.interpolate(bilinear, align_corners=False, antialias=False) on the CPU evaluates the same formula, but
    rounds the source coordinate once (an FMA) where the definition rounds twice, and sums in its own order.  With its
    coordinate the restatement agrees within 4 ulp of 255 (6.1e-5); as defined, the one extra rounding of a coordinate
    below max(h, w) adds at most 255 * ulp(max(h, w)) (7.8e-3 for CIF)."""
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    rng = np.random.default_rng(sum(src) * 1000 + sum(dst))
    rgb = rng.integers(0, 256, src + (3,), dtype=np.uint8)
    want = F.interpolate(torch.from_numpy(rgb).permute(2, 0, 1)[None].float(), size=dst, mode="bilinear",
                         align_corners=False, antialias=False)[0].numpy()
    ulp255 = np.spacing(np.float32(255))
    close = R.resample(rgb, *dst, taps=_taps_contracted)
    assert np.abs(close - want).max() <= 4 * ulp255, (src, dst, np.abs(close - want).max())
    got = R.resample(rgb, *dst)
    bound = 4 * ulp255 + 255 * np.spacing(np.float32(max(src)))
    assert np.abs(got - want).max() <= bound, (src, dst, np.abs(got - want).max(), bound)


def test_normalisation_constants():
    mul, add = R.normalisation((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))
    assert mul.dtype == np.float32 and add.dtype == np.float32
    assert np.array_equal(mul, np.float32([1 / (255 * 0.229), 1 / (255 * 0.224), 1 / (255 * 0.225)]))
    assert np.array_equal(add, np.float32([-0.485 / 0.229, -0.456 / 0.224, -0.406 / 0.225]))


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("resample") / "libresample_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", out,
                           os.path.join(HERE, "native", "resample_host.cpp")])
    L = C.CDLL(out)
    L.rs_axis.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.rs_resample.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    return L


def test_device_math_axis_taps_match_the_restatement(host):
    for n_in in list(range(1, 40)) + [99, 120, 144, 161, 176, 288, 352, 576, 704, 4080]:
        for n_out in (1, 2, 3, 7, 13, 37, 53, 75, 100, 224, 288, 352, 1000, 16384):
            i0, i1 = np.zeros(n_out, np.int32), np.zeros(n_out, np.int32)
            l0, l1 = np.zeros(n_out, np.float32), np.zeros(n_out, np.float32)
            host.rs_axis(n_in, n_out, i0.ctypes.data, i1.ctypes.data, l0.ctypes.data, l1.ctypes.data)
            r = R.axis_taps(n_in, n_out)
            assert np.array_equal(i0, r[0]) and np.array_equal(i1, r[1]), (n_in, n_out)
            # bit for bit, the sign of zero included
            assert np.array_equal(l0.view(np.uint32), r[2].view(np.uint32)), (n_in, n_out)
            assert np.array_equal(l1.view(np.uint32), r[3].view(np.uint32)), (n_in, n_out)
            assert i0.min() >= 0 and i1.max() <= n_in - 1


@pytest.mark.parametrize("src,dst", SIZE_PAIRS)
def test_device_math_bilinear_matches_the_restatement(host, src, dst):
    rng = np.random.default_rng(7)
    rgb = np.ascontiguousarray(rng.integers(0, 256, src + (3,), dtype=np.uint8))
    v = np.zeros((3,) + dst, np.float32)
    host.rs_resample(rgb.ctypes.data, src[1], src[0], dst[1], dst[0], v.ctypes.data)
    assert np.array_equal(v.view(np.uint32), R.resample(rgb, *dst).view(np.uint32)), (src, dst)
