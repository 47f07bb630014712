"""The host side of the fit form of device tensor output (h263cu_decode_step_device_tensor_fit), checked without a GPU:
the ctypes twins of h263cu_tensor_crop / h263cu_tensor_fit match the header and the Rust -sys crate; the geometry
restatement (fit_ref.py) is torchvision's Resize(S) + CenterCrop sizing and the library's own geometry (through its
test hook) equals it; the value restatement is torchvision's resize + center_crop, resized_crop, and interpolate + pad
on CPU floats within a few ulp; and the Python layer refuses what the C ABI refuses."""
import ctypes as C
import os
import re
from fractions import Fraction

import numpy as np
import pytest

import fit_ref as FR
import resample_ref as R
from h263_rs_b200 import _lib, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "h263cu.h")).read()
RUST = open(os.path.join(ROOT, "bindings", "h263cu-sys", "src", "lib.rs")).read()

F = np.float32
TOL = 4 * np.spacing(np.float32(255))  # 4 ulp of 255, as for the stretch (test_device_tensor_abi.py)
OUTPUTS = [(224, 224), (64, 48), (48, 64), (1, 1), (7, 13), (640, 640)]  # (W, H)
SHORT_SIDES = [1, 7, 32, 224, 256]
STANDARD = [(128, 96), (176, 144), (352, 288), (704, 576), (1408, 1152), (4080, 4080), (161, 99), (15, 15)]


def _header_fields(name):
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), HEADER, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return re.findall(r"\b([a-z_0-9]+)(?:\[\d+\])?\s*[,;]", body)


def test_struct_layouts_match_the_header_and_rust():
    Cr, Fi = _lib.TensorCrop, _lib.TensorFit
    assert C.sizeof(Cr) == 16 and C.sizeof(Fi) == 32
    assert [(f, getattr(Cr, f).offset) for f, _ in Cr._fields_] == [("x", 0), ("y", 4), ("width", 8), ("height", 12)]
    assert [(f, getattr(Fi, f).offset) for f, _ in Fi._fields_] == [
        ("mode", 0), ("short_side", 4), ("fill", 8), ("reserved", 20), ("crops", 24)]
    for name, st in (("h263cu_tensor_crop", Cr), ("h263cu_tensor_fit", Fi)):
        assert _header_fields(name) == [f for f, _ in st._fields_], name
        body = re.search(r"pub struct %s \{(.*?)\n\}" % name, RUST, re.S).group(1)
        assert re.findall(r"pub (\w+):", body) == [f for f, _ in st._fields_], name


def test_constants_and_declarations():
    consts = dict(re.findall(r"#define (H263CU_FIT_\w+) (\d+)u", HEADER))
    want = {"H263CU_FIT_STRETCH": _lib.FIT_STRETCH, "H263CU_FIT_LETTERBOX": _lib.FIT_LETTERBOX,
            "H263CU_FIT_CENTER_CROP": _lib.FIT_CENTER_CROP}
    assert consts == {k: str(v) for k, v in want.items()}
    assert (FR.STRETCH, FR.LETTERBOX, FR.CENTER_CROP) == (0, 1, 2) == tuple(want.values())
    for k, v in want.items():
        assert "pub const %s: u32 = %d;" % (k, v) in RUST
    for name in ("h263cu_decode_step_device_tensor_fit", "h263cu_group_decode_step_device_tensor_fit", "h263cu_test_fit_geometry"):
        assert name in _lib.SYMBOLS and "pub fn %s(" % name in RUST, name
        assert hasattr(_lib.lib(), name), name


def _torchvision_center_crop(S, cw, ch, W, H):
    """(rw, rh, px, py) as torchvision v2 computes them: resize(S) sizing, then centre-crop padding and anchor."""
    from torchvision.transforms.v2.functional import _geometry as G

    rh, rw = G._compute_resized_output_size((ch, cw), [S])
    left, top, right, bottom = G._center_crop_compute_padding(H, W, rh, rw)
    a_top, a_left = G._center_crop_compute_crop_anchor(H, W, rh + top + bottom, rw + left + right)
    return rw, rh, left - a_left, top - a_top


def _sweep():
    for cw in range(1, 65):
        for ch in range(1, 65):
            yield cw, ch
    for cw, ch in STANDARD:
        yield cw, ch


def test_center_crop_geometry_is_torchvision():
    pytest.importorskip("torchvision")
    for cw, ch in _sweep():
        for W, H in OUTPUTS:
            for S in SHORT_SIDES:
                assert FR.geometry(FR.CENTER_CROP, S, cw, ch, W, H) == _torchvision_center_crop(S, cw, ch, W, H), (S, cw, ch, W, H)


def test_letterbox_geometry_is_the_rounded_aspect_fit():
    for cw, ch in _sweep():
        for W, H in OUTPUTS:
            rw, rh, px, py = FR.geometry(FR.LETTERBOX, 0, cw, ch, W, H)
            r = min(Fraction(W, cw), Fraction(H, ch))  # the scale that fits the whole crop
            assert (rw, rh) == (max(1, int(cw * r + Fraction(1, 2))), max(1, int(ch * r + Fraction(1, 2)))), (cw, ch, W, H)
            assert rw == W or rh == H
            assert 0 <= px == (W - rw) // 2 and 0 <= py == (H - rh) // 2


def _lib_geometry(mode, S, cw, ch, W, H):
    out = (C.c_int32 * 4)()
    assert _lib.lib().h263cu_test_fit_geometry(mode, S, cw, ch, W, H, out) == 0
    return tuple(out)


@pytest.mark.parametrize("mode", ["stretch", "letterbox", "center_crop"])
def test_library_geometry_equals_the_restatement(mode):
    m = FR.MODES[mode]
    for cw, ch in _sweep():
        for W, H in OUTPUTS:
            for S in SHORT_SIDES if m == FR.CENTER_CROP else [0]:
                assert _lib_geometry(m, S, cw, ch, W, H) == FR.geometry(m, S, cw, ch, W, H), (mode, S, cw, ch, W, H)
    # the extremes of the argument ranges
    for args in [(16384, 1, 65535, 16384, 16384), (16384, 65535, 1, 1, 16384), (1, 65535, 65535, 1, 1)]:
        S = args[0] if m == FR.CENTER_CROP else 0
        assert _lib_geometry(m, S, *args[1:]) == FR.geometry(m, S, *args[1:]), (mode, args)


def test_library_geometry_refuses_what_the_call_refuses():
    out = (C.c_int32 * 4)()
    L = _lib.lib()
    for args in [(3, 0, 10, 10, 10, 10), (2, 0, 10, 10, 10, 10), (2, 16385, 10, 10, 10, 10), (1, 5, 10, 10, 10, 10),
                 (0, 0, 0, 10, 10, 10), (0, 0, 10, 0, 10, 10), (0, 0, 10, 10, 0, 10), (0, 0, 10, 10, 10, 16385),
                 (0, 0, 65536, 10, 10, 10)]:
        assert L.h263cu_test_fit_geometry(*args, out) == _lib.ERR_BAD_ARGUMENT, args
    assert L.h263cu_test_fit_geometry(0, 0, 10, 10, 10, 10, None) == _lib.ERR_BAD_ARGUMENT


def _taps_contracted(n_in, n_out):
    """resample_ref.axis_taps with the source coordinate rounded once (an FMA), as torch's CPU kernel computes it."""
    scale = F(n_in) / F(n_out)
    s = np.maximum((np.float64(scale) * (np.arange(n_out) + 0.5) - 0.5).astype(F), F(0))
    i0 = s.astype(np.int32)
    l1 = s - i0.astype(F)
    return i0, i0 + (i0 < n_in - 1).astype(np.int32), F(1) - l1, l1


def _picture(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


@pytest.mark.parametrize("src,S,out", [((288, 352), 256, (224, 224)), ((144, 176), 256, (224, 224)),
                                       ((99, 161), 64, (48, 80)), ((31, 47), 100, (200, 60)), ((288, 352), 232, (224, 300)),
                                       ((15, 15), 7, (9, 5)), ((120, 160), 33, (33, 33))])
def test_center_crop_values_are_torchvision(src, S, out):
    """torchvision v2 resize(S, antialias=False) -> center_crop((H, W)) on the 0-255 float picture (zero padding where
    the resized picture is smaller than the output: fill 0)."""
    torch = pytest.importorskip("torch")
    TF = pytest.importorskip("torchvision.transforms.v2.functional")
    rgb = _picture(*src, seed=sum(src) + S)
    img = torch.from_numpy(rgb).permute(2, 0, 1).float()
    want = TF.center_crop(TF.resize(img, [S], antialias=False), list(out)).numpy()
    H, W = out
    g = FR.geometry(FR.CENTER_CROP, S, src[1], src[0], W, H)
    got = FR.values(rgb, H, W, g, taps=_taps_contracted)
    assert np.abs(got - want).max() <= TOL, (src, S, out, np.abs(got - want).max())


@pytest.mark.parametrize("src,crop,out", [((288, 352), (17, 3, 200, 251), (224, 224)), ((144, 176), (0, 0, 176, 144), (96, 128)),
                                          ((99, 161), (160, 98, 1, 1), (5, 7)), ((99, 161), (1, 1, 160, 98), (99, 161)),
                                          ((31, 47), (5, 9, 30, 11), (64, 64))])
def test_crop_values_are_torchvision_resized_crop(src, crop, out):
    torch = pytest.importorskip("torch")
    TF = pytest.importorskip("torchvision.transforms.v2.functional")
    rgb = _picture(*src, seed=sum(crop))
    x, y, w, h = crop
    img = torch.from_numpy(rgb).permute(2, 0, 1).float()
    want = TF.resized_crop(img, y, x, h, w, list(out), antialias=False).numpy()
    H, W = out
    got = FR.values(rgb, H, W, FR.geometry(FR.STRETCH, 0, w, h, W, H), crop=crop, taps=_taps_contracted)
    assert np.abs(got - want).max() <= TOL, (src, crop, out, np.abs(got - want).max())


@pytest.mark.parametrize("src,crop,out,fill", [((288, 352), None, (640, 640), (114, 114, 114)), ((144, 176), None, (224, 640), (0, 0, 0)),
                                               ((99, 161), (3, 4, 50, 90), (64, 64), (1.5, 200, 255)),
                                               ((31, 47), None, (31, 47), (9, 9, 9)), ((15, 15), None, (1, 7), (0, 10, 20))])
def test_letterbox_values_are_interpolate_and_pad(src, crop, out, fill):
    torch = pytest.importorskip("torch")
    Fn = torch.nn.functional
    rgb = _picture(*src, seed=sum(out))
    x, y, w, h = crop or (0, 0, src[1], src[0])
    H, W = out
    rw, rh, px, py = FR.geometry(FR.LETTERBOX, 0, w, h, W, H)
    img = torch.from_numpy(rgb[y:y + h, x:x + w]).permute(2, 0, 1)[None].float()
    r = Fn.interpolate(img, size=(rh, rw), mode="bilinear", align_corners=False, antialias=False)[0]
    want = torch.stack([Fn.pad(r[c], (px, W - rw - px, py, H - rh - py), value=float(fill[c])) for c in range(3)]).numpy()
    got = FR.values(rgb, H, W, (rw, rh, px, py), crop=crop, fill=fill, taps=_taps_contracted)
    assert np.abs(got - want).max() <= TOL, (src, crop, out, np.abs(got - want).max())


def test_stretch_without_crops_is_the_plain_resample():
    rgb = _picture(99, 161, 3)
    for H, W in [(224, 224), (99, 161), (1, 1), (300, 17)]:
        got = FR.values(rgb, H, W, FR.geometry(FR.STRETCH, 0, 161, 99, W, H), fill=(7, 7, 7))
        assert np.array_equal(got.view(np.uint32), R.resample(rgb, H, W).view(np.uint32))


def test_python_refuses_what_the_abi_refuses():
    ok = api._tensor_fit("letterbox", None, 114, None, 2)
    assert ok.mode == _lib.FIT_LETTERBOX and list(ok.fill) == [114.0] * 3 and not ok.crops
    assert api._tensor_fit("stretch", None, 0, None, 2) is None  # the plain stretch takes the existing entry point
    f = api._tensor_fit("center_crop", 256, (1, 2, 3), [[0, 0, 5, 5], [1, 2, 3, 4]], 2)
    assert f.mode == _lib.FIT_CENTER_CROP and f.short_side == 256 and list(f.fill) == [1.0, 2.0, 3.0]
    assert [(f.crops[i].x, f.crops[i].y, f.crops[i].width, f.crops[i].height) for i in range(2)] == [(0, 0, 5, 5), (1, 2, 3, 4)]
    inf, nan = float("inf"), float("nan")
    for args in [("squash", None, 0, None), ("center_crop", None, 0, None), ("center_crop", 0, 0, None),
                 ("center_crop", 16385, 0, None), ("center_crop", 2.5, 0, None), ("letterbox", 256, 0, None),
                 ("stretch", 3, 0, None), ("letterbox", None, -1, None), ("letterbox", None, 256, None),
                 ("letterbox", None, (0, nan, 0), None), ("letterbox", None, inf, None), ("letterbox", None, (1, 2), None),
                 ("stretch", None, 0, [[0, 0, 1, 1]]), ("stretch", None, 0, [[0, 0, 1, 1], [0, 0, 0, 1]]),
                 ("stretch", None, 0, [[0, 0, 1, 1], [0, 0, 1, 0]]), ("stretch", None, 0, [[0, 0, 1, 1], [-1, 0, 1, 1]]),
                 ("stretch", None, 0, [[0, 0, 1, 1], [2 ** 32 - 1, 0, 1, 1]]), ("stretch", None, 0, [[0, 0, 1, 1], [0, 0.5, 1, 1]]),
                 ("stretch", None, 0, [[0, 0, 1], [0, 0, 1]])]:
        with pytest.raises(ValueError):
            api._tensor_fit(*args, 2)
