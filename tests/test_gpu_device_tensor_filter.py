"""Decoded pictures resized with torch's antialiased bilinear or bicubic filter into caller-owned RGB tensors on the
device (h263cu_decode_step_device_tensor_filter, BatchDecoder / DeviceGroup.decode_step_device_tensor(antialias=True,
interpolation=...)): bit-exact against the restatement of the definition (filter_ref.py) applied to the oracle's RGBA,
for every filter, fit mode, dtype and layout, with guard elements around every slot, on both sides of the kernel's
fast / general threshold; the bilinear filter through the new call is the fit call's output; argument errors are
refused before any parser moves."""
import ctypes as C

import numpy as np
import pytest
import torch

import filter_ref as FL
import fit_ref as FR
import resample_ref as R
from helpers import oracle_decode_stream
from h263_rs_b200 import _lib, api, synth
from test_gpu_device_output import SIZES
from test_gpu_device_tensor import DTYPES, IMAGENET, bits, expected_planes, rgb_of, view_of
from test_gpu_device_tensor_fit import FILL, MODES, _fit_struct, _random_crops, case_streams, check_slots, expected_fit

pytestmark = pytest.mark.gpu

FILTERS = {"bilinear_aa": FL.BILINEAR_AA, "bicubic_aa": FL.BICUBIC_AA}
KW = {FL.BILINEAR_AA: dict(antialias=True), FL.BICUBIC_AA: dict(antialias=True, interpolation="bicubic")}


def expected_filter(ref, size, dtype, mode, filt, short_side=None, crop=None, fill=(0.0, 0.0, 0.0), mean=None, std=None):
    """[3, H, W] torch tensor (CPU) of one decoded picture under a fit and a filter: the restatement, then step 4."""
    H, W = size
    w, h = ref["info"]["width"], ref["info"]["height"]
    cw, ch = (crop[2], crop[3]) if crop is not None else (w, h)
    geom = FR.geometry(FR.MODES[mode], short_side or 0, cw, ch, W, H)
    v = FL.values(rgb_of(ref), H, W, geom, None if crop is None else tuple(int(c) for c in crop), fill, filt)
    if dtype == torch.uint8:
        return torch.from_numpy(FL.store(v, u8=True))
    mul, add = (1.0,) * 3, (0.0,) * 3
    if mean is not None or std is not None:
        mul, add = R.normalisation(mean if mean is not None else (0.0,) * 3, std if std is not None else (1.0,) * 3)
    return torch.from_numpy(FL.store(v, mul, add)).to(dtype)


def decode_filter_case(cid, size, mode, filt, dtype=torch.float32, layout="contiguous", deblock=False, short_side=None,
                       fill=(0.0, 0.0, 0.0), crop_fn=None, **norm):
    """Two streams step by step into a guarded view under a fit and a filter; crop_fn(t, [(w, h) per input]) gives the
    step's crops."""
    case, opt, streams, refs = case_streams(cid, deblock)
    dec = api.BatchDecoder(2, case["w"], case["h"], decoder_options=opt, threads=2)
    flat, view = view_of(2, size, dtype, layout)
    before = flat.cpu()
    for t in range(len(streams[0])):
        crops = crop_fn(t, [(case["w"], case["h"])] * 2) if crop_fn else None
        out, errs = dec.decode_step_device_tensor([s[t] for s in streams], size, out=view, deblock=deblock, fit=mode,
                                                  short_side=short_side, fill=fill, crops=crops, **KW[filt], **norm)
        assert out is view
        pics = []
        for i in range(2):
            ref = refs[i][t]
            assert (errs[i] != 0) == isinstance(ref, int), (cid, t, i, int(errs[i]))
            e = None if isinstance(ref, int) else expected_filter(ref, size, dtype, mode, filt, short_side,
                                                                  None if crops is None else crops[i], fill, **norm)
            pics.append((i, e))
        before = check_slots(flat, before, view, pics)
    return dec


def _call_filter(dec, packets, target, f, filt, deblock=False):
    plan = dec.plan_step(packets)
    nd = C.c_uint32(0)
    rc = _lib.lib().h263cu_decode_step_device_tensor_filter(
        dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, len(packets), 2,
        _lib.OUT_DEBLOCK if deblock else 0, C.byref(target) if target is not None else None, C.byref(f) if f is not None else None,
        filt, plan["errs"].ctypes.data, C.byref(nd))
    return rc, plan["errs"], nd.value


def fast_path_everywhere(geom, cw, ch, W, H, filt):
    """Whether every CTA of a picture takes the kernel's fast path (csrc/resample_filter.cu: 32 x 8 output tiles; a
    footprint of at most 32 rows and 4096 samples, supports of at most 7) -- and whether any does."""
    rw, rh, px, py = geom
    bic = filt == FL.BICUBIC_AA
    xm, xs, _ = FL.aa_taps(cw, rw, bic)
    ym, ys, _ = FL.aa_taps(ch, rh, bic)
    r = np.float32(2 if bic else 1)
    sx, sy = np.float32(cw) / np.float32(rw), np.float32(ch) / np.float32(rh)
    sup_ok = (r * sx if sx >= 1 else r) <= 7 and (r * sy if sy >= 1 else r) <= 7
    kinds = set()
    for X0 in range(0, W, 32):
        xa, xb = max(X0 - px, 0), min(min(X0 + 32, W) - px, rw) - 1
        for Y0 in range(0, H, 8):
            ya, yb = max(Y0 - py, 0), min(min(Y0 + 8, H) - py, rh) - 1
            if xa > xb or ya > yb:
                continue
            fw, fh = xm[xb] + xs[xb] - xm[xa], ym[yb] + ys[yb] - ym[ya]
            kinds.add(bool(sup_ok and fh <= 32 and fw * fh <= 4096))
    return kinds


@pytest.mark.parametrize("deblock", [False, True])
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_bilinear_filter_is_the_fit_call(dtype, deblock):
    """H263CU_FILTER_BILINEAR through the new entry point writes the bytes h263cu_decode_step_device_tensor_fit writes."""
    case, opt, streams, refs = case_streams("unaligned_161x99_odd", deblock)
    size = (70, 90)
    a = api.BatchDecoder(2, case["w"], case["h"], decoder_options=opt, threads=2)
    b = api.BatchDecoder(2, case["w"], case["h"], decoder_options=opt, threads=2)
    flat_a, view_a = view_of(2, size, dtype, "padded")
    flat_b, view_b = view_of(2, size, dtype, "padded")
    crops = [(3, 1, 150, 90), (0, 0, 161, 99)]
    f = _fit_struct(mode=_lib.FIT_LETTERBOX, fill=FILL, crops=crops)
    for t in range(len(streams[0])):
        packets = [s[t] for s in streams]
        a.decode_step_device_tensor(packets, size, out=view_a, deblock=deblock, fit="letterbox", fill=FILL, crops=crops)
        _, target = api._device_tensor(view_b, 2, size, None, None, None, 0)
        rc, errs, nd = _call_filter(b, packets, target, f, _lib.FILTER_BILINEAR, deblock)
        assert rc == 0 and not errs.any() and nd == 2
        assert torch.equal(bits(flat_a.cpu()), bits(flat_b.cpu())), t


@pytest.mark.parametrize("filt", FILTERS.values(), ids=FILTERS.keys())
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_identity_size_equals_the_bilinear_output(filt, dtype):
    """At the picture's own size every weight is 0 or 1: the AA filters write what the antialias=False call writes."""
    case, opt, streams, refs = case_streams("unaligned_161x99_odd", False)
    size = (case["h"], case["w"])
    a = api.BatchDecoder(2, case["w"], case["h"], decoder_options=opt, threads=2)
    b = api.BatchDecoder(2, case["w"], case["h"], decoder_options=opt, threads=2)
    norm = IMAGENET if dtype != torch.uint8 else {}
    for t in range(len(streams[0])):
        packets = [s[t] for s in streams]
        out_a, _ = a.decode_step_device_tensor(packets, size, dtype=dtype, **norm)
        out_b, errs = b.decode_step_device_tensor(packets, size, dtype=dtype, **KW[filt], **norm)
        assert not errs.any()
        assert torch.equal(bits(out_a.cpu()), bits(out_b.cpu())), t


@pytest.mark.parametrize("layout", ["contiguous", "channels_last", "padded"])
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("filt", FILTERS.values(), ids=FILTERS.keys())
@pytest.mark.parametrize("cid", SIZES)
def test_every_filter_mode_dtype_and_layout(cid, filt, mode, dtype, layout):
    norm = IMAGENET if dtype in (torch.float16, torch.bfloat16) else {}
    decode_filter_case(cid, (56, 72), mode, filt, dtype, layout, short_side=64 if mode == "center_crop" else None, fill=FILL, **norm)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("filt", FILTERS.values(), ids=FILTERS.keys())
@pytest.mark.parametrize("cid", ["unaligned_47x31", "cif_halfpel", "4cif"])
def test_deblocked_planes(cid, filt, mode):
    decode_filter_case(cid, (64, 96), mode, filt, torch.float16, "padded", deblock=True, short_side=80 if mode == "center_crop" else None,
                       fill=FILL, **IMAGENET)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("filt", FILTERS.values(), ids=FILTERS.keys())
@pytest.mark.parametrize("cid", ["cif_halfpel", "unaligned_161x99_odd", "unaligned_15x15"])
def test_random_crops(cid, filt, mode):
    for seed in range(2):
        decode_filter_case(cid, (48, 64), mode, filt, torch.float32, "padded", short_side=48 if mode == "center_crop" else None,
                           fill=FILL, crop_fn=_random_crops(seed + len(cid)))


# (case, output size, fit, short side): 4CIF downscales from 1.4x to the whole picture in one sample
THRESHOLD = [("4cif", (288, 352), "stretch", None), ("4cif", (224, 224), "center_crop", 256), ("4cif", (160, 256), "stretch", None),
             ("4cif", (112, 128), "letterbox", None), ("4cif", (40, 48), "stretch", None), ("4cif", (7, 5), "stretch", None),
             ("4cif", (1, 1), "stretch", None), ("cif_halfpel", (96, 100), "stretch", None), ("cif_halfpel", (3, 200), "stretch", None)]


@pytest.mark.parametrize("filt", FILTERS.values(), ids=FILTERS.keys())
def test_downscales_on_both_sides_of_the_fast_path_threshold(filt):
    case = None
    kinds = set()
    for cid, size, mode, S in THRESHOLD:
        case = case_streams(cid, False)[0]
        H, W = size
        kinds |= fast_path_everywhere(FR.geometry(FR.MODES[mode], S or 0, case["w"], case["h"], W, H), case["w"], case["h"], W, H, filt)
        for dtype in (torch.uint8, torch.float32):
            decode_filter_case(cid, size, mode, filt, dtype, "padded", short_side=S, fill=FILL)
    assert kinds == {True, False}


def test_bicubic_overshoot_exercises_the_u8_clamp_at_both_ends():
    """A 4x bicubic upscale of a noisy picture overshoots below 0 and above 255: U8 clamps, floats do not."""
    w, h = 32, 32
    pk = synth.make_stream(w, h, 2, 901, mv_mode=0)
    refs = oracle_decode_stream(pk)
    size = (128, 128)
    v = FL.values(rgb_of(refs[0]), 128, 128, (128, 128, 0, 0), filt=FL.BICUBIC_AA)
    assert v.min() < -0.5 and v.max() > 255.5, (v.min(), v.max())
    for dtype in (torch.uint8, torch.float32):
        dec = api.BatchDecoder(1, w, h, threads=1)
        for t in range(2):
            out, errs = dec.decode_step_device_tensor([pk[t]], size, dtype=dtype, antialias=True, interpolation="bicubic")
            assert not errs.any()
            want = expected_filter(refs[t], size, dtype, "stretch", FL.BICUBIC_AA)
            got = out[0].cpu()
            assert torch.equal(bits(got), bits(want)), (dtype, t)
            if t == 0 and dtype == torch.uint8:
                assert (got == 0).any() and (got == 255).any()
            if t == 0 and dtype == torch.float32:
                assert got.min() < -0.5 and got.max() > 255.5


@pytest.mark.parametrize("filt", FILTERS.values(), ids=FILTERS.keys())
def test_mixed_sizes_a_bad_packet_and_a_crop_outside_its_picture(filt):
    dims = [(176, 144), (47, 31), (161, 99), (128, 96)]
    streams = [synth.make_stream(w, h, 3, 800 + i, mv_mode=2) for i, (w, h) in enumerate(dims)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(4, 176, 144, threads=2)
    ids = [2, 0, 3, 1]  # input i -> slot i, whatever its stream
    size = (72, 88)
    # one box per input, inside the picture of the stream that input carries: 161 x 99, 176 x 144, 128 x 96, 47 x 31
    crops = [(1, 2, 150, 90), (0, 0, 176, 144), (3, 1, 40, 30), (10, 20, 30, 10)]
    kw = dict(fit="center_crop", short_side=60, fill=FILL, **KW[filt], **IMAGENET)
    flat, view = view_of(4, size, torch.float32, "padded")
    before = flat.cpu()
    for t in range(3):
        packets = [streams[s][t] for s in ids]
        bad = t == 1
        if bad:
            packets[1] = packets[1][:3]  # stream 0 fails to parse: its slot stays as it was, its stream untouched
        step_crops = list(crops)
        if t == 2:
            step_crops[3] = (20, 0, 30, 10)  # outside its 47 x 31 picture: a per-picture error
        _, errs = dec.decode_step_device_tensor(packets, size, out=view, stream_ids=ids, crops=step_crops, **kw)
        failed = {1} if bad else {3} if t == 2 else set()
        assert {i for i in range(4) if errs[i]} == failed, errs
        if t == 2:
            assert errs[3] == _lib.ERR_BAD_ARGUMENT
        pics = [(i, None if i in failed else expected_filter(refs[s][t], size, torch.float32, "center_crop", filt, 60, step_crops[i], FILL,
                                                             **IMAGENET)) for i, s in enumerate(ids)]
        before = check_slots(flat, before, view, pics)
        if bad:  # the stream carries on with the packet it failed on
            _, errs = dec.decode_step_device_tensor([streams[0][1]], size, out=view, stream_ids=[0], crops=[crops[1]], **kw)
            assert not errs.any()
            before = check_slots(flat, before, view, [(0, expected_filter(refs[0][1], size, torch.float32, "center_crop", filt, 60, crops[1],
                                                                          FILL, **IMAGENET))])


def test_argument_errors_are_refused_before_any_parser_moves():
    pk = synth.make_stream(176, 144, 2, 831)
    ref = oracle_decode_stream(pk)
    dec = api.BatchDecoder(1, 176, 144, threads=1)
    buf = torch.zeros(3 * 144 * 176, dtype=torch.float32, device="cuda")
    _, target = api._device_tensor(buf.view(1, 3, 144, 176), 1, (144, 176), None, None, None, 0)
    _, bad_target = api._device_tensor(buf.view(1, 3, 144, 176), 1, (144, 176), None, None, None, 0)
    bad_target.reserved = 1
    inf, nan = float("inf"), float("nan")
    ok = _fit_struct(mode=_lib.FIT_LETTERBOX)
    cases = [(target, ok, 3), (target, ok, 0xFFFFFFFF), (target, None, _lib.FILTER_BILINEAR_AA), (None, ok, _lib.FILTER_BICUBIC_AA),
             (bad_target, ok, _lib.FILTER_BILINEAR_AA)]
    for kw in [dict(mode=3), dict(reserved=1), dict(mode=_lib.FIT_CENTER_CROP, short_side=0), dict(mode=_lib.FIT_CENTER_CROP, short_side=16385),
               dict(mode=_lib.FIT_LETTERBOX, short_side=5), dict(short_side=1), dict(fill=(0.0, nan, 0.0)), dict(fill=(inf, 0.0, 0.0)),
               dict(fill=(-0.5, 0.0, 0.0)), dict(fill=(0.0, 0.0, 255.5)), dict(crops=[(0, 0, 0, 10)]), dict(crops=[(0, 0, 10, 0)]),
               dict(crops=[(2 ** 32 - 5, 0, 5, 10)]), dict(crops=[(0, 2 ** 32 - 1, 1, 2)])]:
        cases.append((target, _fit_struct(**kw), _lib.FILTER_BICUBIC_AA))
    for tg, f, filt in cases:
        rc, _, nd = _call_filter(dec, [pk[0]], tg, f, filt)
        assert rc == _lib.ERR_BAD_ARGUMENT and nd == 0, (f and (f.mode, f.short_side, list(f.fill), f.reserved), filt)
    g = api.DeviceGroup([0], 1, 176, 144, threads=1)
    plan = g.plan_step([pk[0]])
    nd = C.c_uint32(0)
    assert g.L.h263cu_group_decode_step_device_tensor_filter(g.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, 1,
                                                             0, (_lib.DeviceTensor * 1)(target), C.byref(ok), 3, plan["errs"].ctypes.data,
                                                             C.byref(nd)) == _lib.ERR_BAD_ARGUMENT
    g.close()
    for kw in [dict(interpolation="bicubic"), dict(antialias=True, interpolation="nearest"), dict(antialias="yes"),
               dict(antialias=True, fit="center_crop"), dict(antialias=True, fit="letterbox", fill=256)]:
        with pytest.raises(ValueError):
            dec.decode_step_device_tensor([pk[0]], (144, 176), **kw)
    # nothing moved: the packets decode bit-exact now
    for t in range(2):
        out, errs = dec.decode_step_device_tensor([pk[t]], (100, 120), dtype=torch.uint8, fit="center_crop", short_side=110,
                                                  antialias=True, interpolation="bicubic")
        assert not errs.any()
        assert torch.equal(out[0].cpu(), expected_filter(ref[t], (100, 120), torch.uint8, "center_crop", FL.BICUBIC_AA, 110)), t


def test_ordering_on_the_consumer_stream_without_host_syncs():
    """One reused tensor, a non-default consumer stream that clones it after every call: each clone holds its own step."""
    n, t_steps = 16, 4
    streams = [synth.make_stream(352, 288, t_steps, 840 + s, mv_mode=s % 3) for s in range(n)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(n, 352, 288, threads=4)
    consumer = torch.cuda.Stream()
    clones = []
    with torch.cuda.stream(consumer):
        out = None
        for t in range(t_steps):
            filt = FL.BICUBIC_AA if t % 2 else FL.BILINEAR_AA
            out, errs = dec.decode_step_device_tensor([s[t] for s in streams], (224, 224), out=out, fit="center_crop", short_side=256,
                                                      **KW[filt], **IMAGENET)
            assert not errs.any()
            clones.append(out.clone())
    torch.cuda.synchronize()
    for t, cl in enumerate(clones):
        got = cl.cpu()
        filt = FL.BICUBIC_AA if t % 2 else FL.BILINEAR_AA
        for s in range(n):
            want = expected_filter(refs[s][t], (224, 224), torch.float16, "center_crop", filt, 256, **IMAGENET)
            assert torch.equal(bits(got[s]), bits(want)), (t, s)


def test_alternates_with_rgba_yuv_and_tensor_steps():
    n, t_steps = 3, 10
    streams = [synth.make_stream(176, 144, t_steps, 760 + s, mv_mode=1) for s in range(n)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(n, 176, 144, threads=2)
    for t in range(t_steps):
        packets = [s[t] for s in streams]
        mode = t % 5
        if mode == 0:
            out, errs = dec.decode_step_device(packets)
            assert not errs.any()
            got = out.cpu().numpy().reshape(n, -1)
            for s in range(n):
                assert np.array_equal(got[s], refs[s][t]["rgba"]), (t, s)
        elif mode == 1:
            out, errs = dec.decode_step_device_yuv(packets, layout="nv12")
            assert not errs.any()
            for s in range(n):
                for k, want in enumerate(expected_planes(refs[s][t], "nv12")):
                    assert np.array_equal(out[k][s].cpu().numpy().reshape(want.shape), want), (t, s, k)
        elif mode == 2:
            out, errs = dec.decode_step_device_tensor(packets, (96, 128), dtype=torch.bfloat16, fit="letterbox", fill=FILL)
            assert not errs.any()
            for s in range(n):
                want = expected_fit(refs[s][t], (96, 128), torch.bfloat16, "letterbox", None, None, FILL)
                assert torch.equal(bits(out[s].cpu()), bits(want)), (t, s)
        else:
            filt = FL.BILINEAR_AA if mode == 3 else FL.BICUBIC_AA
            out, errs = dec.decode_step_device_tensor(packets, (96, 128), dtype=torch.bfloat16, fit="letterbox", fill=FILL, **KW[filt])
            assert not errs.any()
            for s in range(n):
                want = expected_filter(refs[s][t], (96, 128), torch.bfloat16, "letterbox", filt, None, None, FILL)
                assert torch.equal(bits(out[s].cpu()), bits(want)), (t, s)
        for s in range(n):
            y, cb, cr = dec.ctx.read_yuv(s)
            r = refs[s][t]
            assert np.array_equal(y, r["y"]) and np.array_equal(cb, r["cb"]) and np.array_equal(cr, r["cr"]), (t, s)


@pytest.mark.parametrize("devices", [[0, 0, 0], "all"])
def test_device_group_with_crops_by_input_position(devices):
    if devices == "all":
        if torch.cuda.device_count() < 2:
            pytest.skip("one GPU")
        devices = list(range(torch.cuda.device_count()))
    nd, per = len(devices), 2
    n, t_steps = nd * per, 3
    streams = [synth.make_stream(176, 144, t_steps, 860 + s, mv_mode=s % 3) for s in range(n)]
    g = api.DeviceGroup(devices, per, 176, 144, threads=4)
    order = list(range(n))[::-1]  # input i carries global stream order[i]
    for t in range(t_steps):
        deblock = t == 2
        filt = FL.BICUBIC_AA if t % 2 else FL.BILINEAR_AA
        refs = [oracle_decode_stream(s[: t + 1], deblock=deblock)[t] for s in streams]
        crops = [(i, 2 * i + 1, 176 - 3 * i - 1, 144 - 2 * i - 3) for i in range(n)]  # one box per input, all different
        outs, errs = g.decode_step_device_tensor([streams[s][t] for s in order], (100, 120), dtype=torch.float32, deblock=deblock,
                                                 stream_ids=order, fit="letterbox", fill=FILL, crops=crops, **KW[filt], **IMAGENET)
        assert not errs.any() and len(outs) == nd
        for i, s in enumerate(order):
            got = outs[s % nd][s // nd].cpu()
            want = expected_filter(refs[s], (100, 120), torch.float32, "letterbox", filt, None, crops[i], FILL, **IMAGENET)
            assert torch.equal(bits(got), bits(want)), (t, i, s)
    g.close()
