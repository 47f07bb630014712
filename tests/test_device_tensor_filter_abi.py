"""The host side of antialiased device tensors (h263cu_decode_step_device_tensor_filter), checked without a GPU: the
filter constants and declarations match across the header, ctypes and the Rust -sys crate; the restatement
(filter_ref.py) agrees with torch's CPU F.interpolate(antialias=True) and torchvision v2's resize + center_crop,
resized_crop and interpolate + pad within a stated bound; the device weight functions, built with g++, equal the
restatement bit for bit; and the Python layer refuses what is not offered.

The bound: torch's CPU kernel computes each tap's center and coordinate in double before rounding the weight to float,
where the definition rounds every step to float, so single weights differ in their last bit or two; a sum of up to
six products (bicubic, 1.13x) of values up to 255 then differs by a few ulp of the largest intermediate.  Bicubic
intermediates reach about 300 (the filter overshoots) and its negative lobes cancel, so its bound is wider."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import filter_ref as FL
import fit_ref as FR
from h263_rs_b200 import _lib, api

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HEADER = open(os.path.join(ROOT, "include", "h263cu.h")).read()
RUST = open(os.path.join(ROOT, "bindings", "h263cu-sys", "src", "lib.rs")).read()

F = np.float32
ULP = np.spacing(F(255))
TOL = {FL.BILINEAR_AA: 8 * ULP, FL.BICUBIC_AA: 32 * ULP}
MODES = {FL.BILINEAR_AA: "bilinear", FL.BICUBIC_AA: "bicubic"}
STANDARD = [(128, 96), (176, 144), (352, 288), (704, 576), (1408, 1152), (161, 99), (15, 15)]  # (w, h)


def _picture(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def _torch_aa(rgb, H, W, filt):
    import torch

    img = torch.from_numpy(np.ascontiguousarray(rgb)).permute(2, 0, 1)[None].float()
    return torch.nn.functional.interpolate(img, size=(H, W), mode=MODES[filt], antialias=True, align_corners=False)[0].numpy()


def test_constants_and_declarations():
    consts = dict(re.findall(r"#define (H263CU_FILTER_\w+) (\d+)u", HEADER))
    want = {"H263CU_FILTER_BILINEAR": _lib.FILTER_BILINEAR, "H263CU_FILTER_BILINEAR_AA": _lib.FILTER_BILINEAR_AA,
            "H263CU_FILTER_BICUBIC_AA": _lib.FILTER_BICUBIC_AA}
    assert consts == {k: str(v) for k, v in want.items()}
    assert (FL.BILINEAR, FL.BILINEAR_AA, FL.BICUBIC_AA) == (0, 1, 2) == tuple(want.values())
    for k, v in want.items():
        assert "pub const %s: u32 = %d;" % (k, v) in RUST
    for name in ("h263cu_decode_step_device_tensor_filter", "h263cu_group_decode_step_device_tensor_filter"):
        assert name in _lib.SYMBOLS and "pub fn %s(" % name in RUST and name + "(" in HEADER, name
        assert hasattr(_lib.lib(), name), name
        # the fit call's arguments plus `filter: u32` before per_pic_err
        fit = re.search(r"pub fn %s\((.*?)\) -> c_int;" % name.replace("filter", "fit"), RUST, re.S).group(1)
        new = re.search(r"pub fn %s\((.*?)\) -> c_int;" % name, RUST, re.S).group(1)
        names = lambda body: re.findall(r"(\w+):", body)
        want_args = names(fit)
        want_args.insert(want_args.index("per_pic_err"), "filter")
        assert names(new) == want_args, name
        argtypes = getattr(_lib.lib(), name).argtypes
        assert len(argtypes) == len(want_args) and argtypes[-3] is C.c_uint32, name


@pytest.mark.parametrize("filt", [FL.BILINEAR_AA, FL.BICUBIC_AA])
def test_standard_formats_to_common_sizes(filt):
    pytest.importorskip("torch")
    for w, h in STANDARD:
        rgb = _picture(h, w, w + h)
        for W, H in [(224, 224), (256, 256), (312, 256), (640, 640), (224, 312)]:
            got = FL.values(rgb, H, W, (W, H, 0, 0), filt=filt)
            d = np.abs(got - _torch_aa(rgb, H, W, filt)).max()
            assert d <= TOL[filt], ((w, h), (W, H), d)


@pytest.mark.parametrize("filt", [FL.BILINEAR_AA, FL.BICUBIC_AA])
def test_every_axis_pair_up_to_64(filt):
    """Every n_in -> n_out of one axis in 1..64 (the other axis at its own size, where the filter is the identity)."""
    pytest.importorskip("torch")
    worst = 0.0
    for n_in in range(1, 65):
        rgb = _picture(3, n_in, n_in)
        for n_out in range(1, 65):
            got = FL.values(rgb, 3, n_out, (n_out, 3, 0, 0), filt=filt)
            d = float(np.abs(got - _torch_aa(rgb, 3, n_out, filt)).max())
            assert d <= TOL[filt], (n_in, n_out, d)
            worst = max(worst, d)
        rgb_t = rgb.transpose(1, 0, 2)  # the vertical axis alike
        got = FL.values(rgb_t, 17, 3, (3, 17, 0, 0), filt=filt)
        assert np.abs(got - _torch_aa(rgb_t, 17, 3, filt)).max() <= TOL[filt], n_in


@pytest.mark.parametrize("filt", [FL.BILINEAR_AA, FL.BICUBIC_AA])
def test_extreme_downscales(filt):
    pytest.importorskip("torch")
    for (w, h), (W, H) in [((704, 576), (1, 1)), ((1408, 1152), (3, 2)), ((352, 288), (16, 16)), ((704, 576), (5, 40)),
                           ((176, 144), (1, 144)), ((4080, 16), (7, 16))]:
        rgb = _picture(h, w, W * H)
        got = FL.values(rgb, H, W, (W, H, 0, 0), filt=filt)
        d = np.abs(got - _torch_aa(rgb, H, W, filt)).max()
        assert d <= TOL[filt], ((w, h), (W, H), d)


@pytest.mark.parametrize("filt", [FL.BILINEAR_AA, FL.BICUBIC_AA])
@pytest.mark.parametrize("src,S,out", [((288, 352), 256, (224, 224)), ((144, 176), 256, (224, 224)), ((576, 704), 232, (224, 224)),
                                       ((99, 161), 64, (48, 80)), ((31, 47), 100, (200, 60)), ((15, 15), 7, (9, 5))])
def test_center_crop_values_are_torchvision(src, S, out, filt):
    """torchvision v2 resize(S, antialias=True) -> center_crop((H, W)) on the 0-255 float picture."""
    torch = pytest.importorskip("torch")
    TF = pytest.importorskip("torchvision.transforms.v2.functional")
    from torchvision.transforms import InterpolationMode as IM

    rgb = _picture(*src, seed=sum(src) + S)
    img = torch.from_numpy(rgb).permute(2, 0, 1).float()
    mode = IM.BILINEAR if filt == FL.BILINEAR_AA else IM.BICUBIC
    want = TF.center_crop(TF.resize(img, [S], interpolation=mode, antialias=True), list(out)).numpy()
    H, W = out
    got = FL.values(rgb, H, W, FR.geometry(FR.CENTER_CROP, S, src[1], src[0], W, H), filt=filt)
    assert np.abs(got - want).max() <= TOL[filt], (src, S, out, np.abs(got - want).max())


@pytest.mark.parametrize("filt", [FL.BILINEAR_AA, FL.BICUBIC_AA])
@pytest.mark.parametrize("src,crop,out", [((288, 352), (17, 3, 200, 251), (224, 224)), ((144, 176), (0, 0, 176, 144), (96, 128)),
                                          ((99, 161), (160, 98, 1, 1), (5, 7)), ((99, 161), (1, 1, 160, 98), (99, 161)),
                                          ((31, 47), (5, 9, 30, 11), (64, 64)), ((576, 704), (3, 5, 701, 570), (20, 30))])
def test_crop_values_are_torchvision_resized_crop(src, crop, out, filt):
    """The crop acts as the whole picture: taps are cut and renormalised at its edge, as in resized_crop."""
    torch = pytest.importorskip("torch")
    TF = pytest.importorskip("torchvision.transforms.v2.functional")
    from torchvision.transforms import InterpolationMode as IM

    rgb = _picture(*src, seed=sum(crop))
    x, y, w, h = crop
    img = torch.from_numpy(rgb).permute(2, 0, 1).float()
    mode = IM.BILINEAR if filt == FL.BILINEAR_AA else IM.BICUBIC
    want = TF.resized_crop(img, y, x, h, w, list(out), interpolation=mode, antialias=True).numpy()
    H, W = out
    got = FL.values(rgb, H, W, FR.geometry(FR.STRETCH, 0, w, h, W, H), crop=crop, filt=filt)
    assert np.abs(got - want).max() <= TOL[filt], (src, crop, out, np.abs(got - want).max())


@pytest.mark.parametrize("filt", [FL.BILINEAR_AA, FL.BICUBIC_AA])
@pytest.mark.parametrize("src,crop,out,fill", [((288, 352), None, (640, 640), (114, 114, 114)), ((144, 176), None, (224, 640), (0, 0, 0)),
                                               ((99, 161), (3, 4, 50, 90), (64, 64), (1.5, 200, 255)),
                                               ((576, 704), None, (64, 64), (9, 9, 9)), ((15, 15), None, (1, 7), (0, 10, 20))])
def test_letterbox_values_are_interpolate_and_pad(src, crop, out, fill, filt):
    torch = pytest.importorskip("torch")
    Fn = torch.nn.functional
    rgb = _picture(*src, seed=sum(out))
    x, y, w, h = crop or (0, 0, src[1], src[0])
    H, W = out
    rw, rh, px, py = FR.geometry(FR.LETTERBOX, 0, w, h, W, H)
    img = torch.from_numpy(rgb[y:y + h, x:x + w]).permute(2, 0, 1)[None].float()
    r = Fn.interpolate(img, size=(rh, rw), mode=MODES[filt], align_corners=False, antialias=True)[0]
    want = torch.stack([Fn.pad(r[c], (px, W - rw - px, py, H - rh - py), value=float(fill[c])) for c in range(3)]).numpy()
    got = FL.values(rgb, H, W, (rw, rh, px, py), crop=crop, fill=fill, filt=filt)
    assert np.abs(got - want).max() <= TOL[filt], (src, crop, out, np.abs(got - want).max())


@pytest.mark.parametrize("filt", [FL.BILINEAR_AA, FL.BICUBIC_AA])
def test_identity_size_is_exact(filt):
    """At rw = cw every weight is exactly 0 or 1: the picture itself, as the bilinear definition gives."""
    for n in [1, 2, 3, 15, 99, 176, 704]:
        xmin, xsize, w = FL.aa_taps(n, n, filt == FL.BICUBIC_AA)
        assert set(np.unique(w).tolist()) <= {0.0, 1.0} and (w.sum(1) == 1).all()
        assert np.array_equal(xmin + np.argmax(w, 1), np.arange(n))
    rgb = _picture(31, 47, 5)
    got = FL.values(rgb, 31, 47, (47, 31, 0, 0), filt=filt)
    assert np.array_equal(got, rgb.transpose(2, 0, 1).astype(F))


@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("filter") / "libfilter_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", out,
                           os.path.join(HERE, "native", "filter_host.cpp")])
    L = C.CDLL(out)
    L.aa_axis.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.aa_axis.restype = None
    return L


@pytest.mark.parametrize("filt", [FL.BILINEAR_AA, FL.BICUBIC_AA])
def test_device_weights_equal_the_restatement(host_lib, filt):
    pairs = [(n_in, n_out) for n_in in range(1, 65) for n_out in range(1, 65)]
    pairs += [(w, W) for w, _ in STANDARD for W in (1, 3, 224, 256, 312, 640)]
    pairs += [(h, H) for _, h in STANDARD for H in (1, 224, 256, 312, 640)]
    for n_in, n_out in pairs:
        xmin, xsize, w = FL.aa_taps(n_in, n_out, filt == FL.BICUBIC_AA)
        k = w.shape[1]
        gm, gs = np.empty(n_out, np.int32), np.empty(n_out, np.int32)
        gw = np.zeros((n_out, k), F)
        host_lib.aa_axis(n_in, n_out, int(filt == FL.BICUBIC_AA), k, gm.ctypes.data, gs.ctypes.data, gw.ctypes.data)
        assert np.array_equal(gm, xmin) and np.array_equal(gs, xsize), (n_in, n_out)
        assert np.array_equal(gw.view(np.uint32), w.view(np.uint32)), (n_in, n_out)


def test_python_filter_rules():
    assert api._tensor_filter(False, "bilinear") is None  # the existing entry points
    assert api._tensor_filter(True, "bilinear") == _lib.FILTER_BILINEAR_AA
    assert api._tensor_filter(True, "bicubic") == _lib.FILTER_BICUBIC_AA
    try:
        from torchvision.transforms import InterpolationMode as IM
    except ImportError:
        IM = None
    if IM is not None:
        assert api._tensor_filter(True, IM.BICUBIC) == _lib.FILTER_BICUBIC_AA
        with pytest.raises(ValueError):
            api._tensor_filter(True, IM.NEAREST)
    for args in [(False, "bicubic"), (True, "nearest"), (True, "area"), (True, "lanczos"), (True, "BILINEAR"), (1, "bilinear"),
                 (None, "bilinear"), (True, None)]:
        with pytest.raises(ValueError):
            api._tensor_filter(*args)
    # the filter call always takes a fit, the plain stretch included
    f = api._tensor_fit("stretch", None, 0, None, 2, always=True)
    assert f.mode == _lib.FIT_STRETCH and not f.crops and list(f.fill) == [0.0] * 3
