"""Decoded pictures letterboxed, centre-cropped or cut to per-picture crop boxes into caller-owned RGB tensors on the
device (h263cu_decode_step_device_tensor_fit, BatchDecoder / DeviceGroup.decode_step_device_tensor(fit=..., crops=...)):
bit-exact against the restatement of the definition (fit_ref.py) applied to the oracle's RGBA, for every mode, dtype
and layout, with guard elements around every slot; a crop outside its picture is that picture's error and leaves its
stream untouched; argument errors are refused before any parser moves."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

import fit_ref as FR
import resample_ref as R
from helpers import oracle_decode_stream
from h263_rs_b200 import _lib, api, frontend, synth
from test_gpu_device_output import SIZES
from test_gpu_device_tensor import BY_ID, DTYPES, IMAGENET, bits, check_guarded, rgb_of, view_of
from test_gpu_parity import _packets

pytestmark = pytest.mark.gpu

MODES = ["stretch", "letterbox", "center_crop"]
FILL = (114.0, 30.5, 200.0)


def expected_fit(ref, size, dtype, mode, short_side=None, crop=None, fill=(0.0, 0.0, 0.0), mean=None, std=None):
    """[3, H, W] torch tensor (CPU) of one decoded picture under a fit: the restatement, then step 4."""
    H, W = size
    w, h = ref["info"]["width"], ref["info"]["height"]
    cw, ch = (crop[2], crop[3]) if crop is not None else (w, h)
    geom = FR.geometry(FR.MODES[mode], short_side or 0, cw, ch, W, H)
    v = FR.values(rgb_of(ref), H, W, geom, None if crop is None else tuple(int(c) for c in crop), fill)
    if dtype == torch.uint8:
        return torch.from_numpy(R.store(v, u8=True))
    mul, add = (1.0,) * 3, (0.0,) * 3
    if mean is not None or std is not None:
        mul, add = R.normalisation(mean if mean is not None else (0.0,) * 3, std if std is not None else (1.0,) * 3)
    return torch.from_numpy(R.store(v, mul, add)).to(dtype)


def check_slots(flat, before, view, pictures):
    """pictures: (slot, expected [3, H, W] tensor, or None for an input that failed).  The decoded slots hold their
    expected values and every other element of the buffer is unchanged."""
    want = before.clone()
    wv = want.as_strided(view.shape, view.stride(), view.storage_offset())
    for slot, e in pictures:
        if e is not None:
            wv[slot] = e
    got = flat.cpu()
    if not torch.equal(bits(got), bits(want)):
        gv = got.as_strided(view.shape, view.stride(), view.storage_offset())
        for slot, e in pictures:
            if e is not None:
                bad = int((bits(gv[slot]) != bits(wv[slot])).sum())
                assert bad == 0, ("slot", slot, bad, "elements differ")
        raise AssertionError("elements outside the decoded slots were written")
    return got


@functools.lru_cache(maxsize=None)
def case_streams(cid, deblock, n_max=3):
    """The packets of a case and of a reseeded twin, and their oracle pictures."""
    case = dict(BY_ID[cid], deblock_flag=1) if deblock else BY_ID[cid]
    a, opt = _packets(case)
    b, _ = _packets(dict(case, seed=case["seed"] + 100))
    n = min(len(a), n_max)
    streams = [a[:n], b[:n]]
    return case, opt, streams, [oracle_decode_stream(s, opt, deblock=deblock) for s in streams]


def decode_fit_case(cid, size, mode, dtype=torch.float32, layout="contiguous", deblock=False, short_side=None, fill=(0.0, 0.0, 0.0),
                    crop_fn=None, **norm):
    """Two streams step by step into a guarded view under a fit; crop_fn(t, [(w, h) per input]) gives the step's crops."""
    case, opt, streams, refs = case_streams(cid, deblock)
    dec = api.BatchDecoder(2, case["w"], case["h"], decoder_options=opt, threads=2)
    flat, view = view_of(2, size, dtype, layout)
    before = flat.cpu()
    for t in range(len(streams[0])):
        crops = crop_fn(t, [(case["w"], case["h"])] * 2) if crop_fn else None
        out, errs = dec.decode_step_device_tensor([s[t] for s in streams], size, out=view, deblock=deblock, fit=mode,
                                                  short_side=short_side, fill=fill, crops=crops, **norm)
        assert out is view
        pics = []
        for i in range(2):
            ref = refs[i][t]
            assert (errs[i] != 0) == isinstance(ref, int), (cid, t, i, int(errs[i]))
            e = None if isinstance(ref, int) else expected_fit(ref, size, dtype, mode, short_side, None if crops is None else crops[i],
                                                               fill, **norm)
            pics.append((i, e))
        before = check_slots(flat, before, view, pics)
    return dec


def _fit_struct(mode=_lib.FIT_STRETCH, short_side=0, fill=(0.0, 0.0, 0.0), reserved=0, crops=None):
    arr = None
    if crops is not None:
        arr = (_lib.TensorCrop * len(crops))(*[_lib.TensorCrop(*c) for c in crops])
    f = _lib.TensorFit(mode, short_side, (C.c_float * 3)(*fill), reserved, arr)
    f._keep = arr
    return f


@pytest.mark.parametrize("deblock", [False, True])
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_stretch_fit_without_crops_is_the_plain_call(dtype, deblock):
    """The fit entry point with STRETCH and no crops writes the bytes h263cu_decode_step_device_tensor writes."""
    case, opt, streams, refs = case_streams("unaligned_161x99_odd", deblock)
    size = (70, 90)
    L = _lib.lib()
    plain = api.BatchDecoder(2, case["w"], case["h"], decoder_options=opt, threads=2)
    fitted = api.BatchDecoder(2, case["w"], case["h"], decoder_options=opt, threads=2)
    flat_a, view_a = view_of(2, size, dtype, "padded")
    flat_b, view_b = view_of(2, size, dtype, "padded")
    before = flat_a.cpu()
    assert torch.equal(bits(before), bits(flat_b.cpu()))
    f = _fit_struct(fill=(0.0, 0.0, 0.0))
    for t in range(len(streams[0])):
        packets = [s[t] for s in streams]
        plain.decode_step_device_tensor(packets, size, out=view_a, deblock=deblock)
        _, target = api._device_tensor(view_b, 2, size, None, None, None, 0)
        plan = fitted.plan_step(packets)
        nd = C.c_uint32(0)
        _lib.check(L.h263cu_decode_step_device_tensor_fit(
            fitted.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, 2, 2,
            _lib.OUT_DEBLOCK if deblock else 0, C.byref(target), C.byref(f), plan["errs"].ctypes.data, C.byref(nd)))
        assert not plan["errs"].any() and nd.value == 2
        before = check_guarded(flat_b, before, view_b, [(i, refs[i][t]) for i in range(2)], size, dtype)
        assert torch.equal(bits(flat_a.cpu()), bits(flat_b.cpu())), t


@pytest.mark.parametrize("layout", ["contiguous", "channels_last", "padded"])
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cid", SIZES)
def test_every_mode_dtype_and_layout(cid, mode, dtype, layout):
    norm = IMAGENET if dtype in (torch.float16, torch.bfloat16) else {}
    decode_fit_case(cid, (56, 72), mode, dtype, layout, short_side=64 if mode == "center_crop" else None, fill=FILL, **norm)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cid", ["unaligned_47x31", "cif_halfpel", "4cif"])
def test_deblocked_planes_under_every_mode(cid, mode):
    decode_fit_case(cid, (64, 96), mode, torch.float16, "padded", deblock=True, short_side=80 if mode == "center_crop" else None,
                    fill=FILL, **IMAGENET)


def _random_crops(seed):
    """Per step, one box per input: odd offsets (chroma parity), 1 x 1 boxes, boxes touching the right and bottom edges,
    and the whole picture, in turn."""
    def fn(t, dims):
        rng = np.random.default_rng(seed * 100 + t)
        out = []
        for i, (w, h) in enumerate(dims):
            kind = (t * len(dims) + i) % 4
            if kind == 0:
                x, y = 2 * int(rng.integers(0, w // 2)) + 1 if w > 1 else 0, 2 * int(rng.integers(0, h // 2)) + 1 if h > 1 else 0
                x, y = min(x, w - 1), min(y, h - 1)
                out.append((x, y, int(rng.integers(1, w - x + 1)), int(rng.integers(1, h - y + 1))))
            elif kind == 1:
                out.append((int(rng.integers(0, w)), int(rng.integers(0, h)), 1, 1))
            elif kind == 2:
                cw, ch = int(rng.integers(1, w + 1)), int(rng.integers(1, h + 1))
                out.append((w - cw, h - ch, cw, ch))
            else:
                out.append((0, 0, w, h))
        return out
    return fn


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cid", ["cif_halfpel", "unaligned_161x99_odd", "unaligned_15x15"])
def test_random_crops(cid, mode):
    for seed in range(2):
        decode_fit_case(cid, (48, 64), mode, torch.float32, "padded", short_side=48 if mode == "center_crop" else None,
                        fill=FILL, crop_fn=_random_crops(seed + len(cid)))


@pytest.mark.parametrize("mode,short_side", [("letterbox", None), ("center_crop", 60)])
def test_mixed_sizes_in_one_step_and_a_bad_packet(mode, short_side):
    dims = [(176, 144), (47, 31), (161, 99), (128, 96)]
    streams = [synth.make_stream(w, h, 3, 800 + i, mv_mode=2) for i, (w, h) in enumerate(dims)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(4, 176, 144, threads=2)
    ids = [2, 0, 3, 1]  # input i -> slot i, whatever its stream
    size = (72, 88)
    kw = dict(fit=mode, short_side=short_side, fill=FILL, **IMAGENET)
    flat, view = view_of(4, size, torch.float32, "padded")
    before = flat.cpu()
    for t in range(3):
        packets = [streams[s][t] for s in ids]
        bad = t == 1
        if bad:
            packets[1] = packets[1][:3]  # stream 0 fails to parse: its slot stays as it was, its stream untouched
        _, errs = dec.decode_step_device_tensor(packets, size, out=view, stream_ids=ids, **kw)
        assert bool(errs[1]) == bad and not errs[[0, 2, 3]].any()
        pics = [(i, None if bad and i == 1 else expected_fit(refs[s][t], size, torch.float32, mode, short_side, None, FILL, **IMAGENET))
                for i, s in enumerate(ids)]
        before = check_slots(flat, before, view, pics)
        if bad:  # the stream carries on with the packet it failed on
            _, errs = dec.decode_step_device_tensor([streams[0][1]], size, out=view, stream_ids=[0], **kw)
            assert not errs.any()
            before = check_slots(flat, before, view, [(0, expected_fit(refs[0][1], size, torch.float32, mode, short_side, None, FILL,
                                                                       **IMAGENET))])


def test_crop_outside_its_picture_is_a_per_picture_error():
    streams = [synth.make_stream(176, 144, 3, 820 + s, mv_mode=1) for s in range(3)]
    refs = [oracle_decode_stream(s) for s in streams]
    hdr = frontend.peek_picture(streams[0][0])  # how a caller learns the size its boxes must fit
    assert (int(hdr["width"]), int(hdr["height"])) == (176, 144)
    dec = api.BatchDecoder(3, 176, 144, threads=2)
    size = (40, 56)
    flat, view = view_of(3, size, torch.uint8, "padded")
    before = flat.cpu()
    good = [(3, 5, 100, 80), (0, 0, 176, 144), (175, 143, 1, 1)]
    for bad_box in [(1, 0, 176, 144), (0, 0, 176, 145), (170, 100, 7, 1), (0, 144, 1, 1)]:
        crops = [bad_box, good[1], good[2]]
        _, errs = dec.decode_step_device_tensor([s[0] for s in streams], size, out=view, fit="letterbox", fill=FILL, crops=crops)
        assert errs[0] == _lib.ERR_BAD_ARGUMENT and not errs[1:].any(), bad_box
        pics = [(0, None)] + [(i, expected_fit(refs[i][0], size, torch.uint8, "letterbox", None, crops[i], FILL)) for i in (1, 2)]
        before = check_slots(flat, before, view, pics)
        # the failed stream did not move: its first packet, with a box that fits, decodes bit-exact
        _, errs = dec.decode_step_device_tensor([streams[0][0]], size, out=view, stream_ids=[0], fit="letterbox", fill=FILL,
                                                crops=[good[0]])
        assert not errs.any()
        before = check_slots(flat, before, view, [(0, expected_fit(refs[0][0], size, torch.uint8, "letterbox", None, good[0], FILL))])
        # the next round feeds every stream its first picture (an I picture) again
    # the streams carry on with their next pictures
    _, errs = dec.decode_step_device_tensor([s[1] for s in streams], size, out=view, fit="letterbox", fill=FILL, crops=good)
    assert not errs.any()
    check_slots(flat, before, view, [(i, expected_fit(refs[i][1], size, torch.uint8, "letterbox", None, good[i], FILL)) for i in range(3)])


def test_fill_values():
    pk, opt = _packets(BY_ID["config1_qcif"])
    assert opt == 1
    ref = oracle_decode_stream(pk[:1], opt)[0]
    # uint8 with 114: the letterbox bars of a 176 x 144 picture in 640 x 640 are exactly 114
    out, errs = api.BatchDecoder(1, 176, 144, threads=1).decode_step_device_tensor([pk[0]], (640, 640), dtype=torch.uint8,
                                                                                    fit="letterbox", fill=114)
    assert not errs.any()
    got = out[0].cpu()
    rw, rh, px, py = FR.geometry(FR.LETTERBOX, 0, 176, 144, 640, 640)
    assert (rw, rh, px, py) == (640, 524, 0, 58)
    assert (got[:, :py] == 114).all() and (got[:, py + rh:] == 114).all()
    assert torch.equal(got, expected_fit(ref, (640, 640), torch.uint8, "letterbox", None, None, (114.0,) * 3))
    # float16 with ImageNet mean / std: fill 0 normalises to `add`
    out, errs = api.BatchDecoder(1, 176, 144, threads=1).decode_step_device_tensor([pk[0]], (224, 224), dtype=torch.float16,
                                                                                    fit="letterbox", fill=0, **IMAGENET)
    assert not errs.any()
    _, add = R.normalisation(IMAGENET["mean"], IMAGENET["std"])
    got = out[0].cpu()
    rw, rh, px, py = FR.geometry(FR.LETTERBOX, 0, 176, 144, 224, 224)
    for c in range(3):
        assert (got[c, :py] == torch.tensor(float(add[c])).half()).all()
    assert torch.equal(bits(got), bits(expected_fit(ref, (224, 224), torch.float16, "letterbox", None, None, (0.0,) * 3, **IMAGENET)))


def test_argument_errors_are_refused_before_any_parser_moves():
    pk = synth.make_stream(176, 144, 2, 831)
    ref = oracle_decode_stream(pk)
    dec = api.BatchDecoder(1, 176, 144, threads=1)
    L = _lib.lib()
    buf = torch.zeros(3 * 144 * 176, dtype=torch.float32, device="cuda")
    _, target = api._device_tensor(buf.view(1, 3, 144, 176), 1, (144, 176), None, None, None, 0)
    inf, nan = float("inf"), float("nan")
    bad = [
        dict(mode=3),                                                 # unknown mode
        dict(reserved=1),                                             # reserved not zero
        dict(mode=_lib.FIT_CENTER_CROP, short_side=0),                # short side out of range
        dict(mode=_lib.FIT_CENTER_CROP, short_side=16385),
        dict(mode=_lib.FIT_LETTERBOX, short_side=5),                  # short side without CENTER_CROP
        dict(short_side=1),
        dict(fill=(0.0, nan, 0.0)), dict(fill=(inf, 0.0, 0.0)),       # fill not finite
        dict(fill=(-0.5, 0.0, 0.0)), dict(fill=(0.0, 0.0, 255.5)),    # fill outside [0, 255]
        dict(crops=[(0, 0, 0, 10)]), dict(crops=[(0, 0, 10, 0)]),     # empty crop
        dict(crops=[(2 ** 32 - 5, 0, 5, 10)]),                        # x + width overflows 32 bits
        dict(crops=[(0, 2 ** 32 - 1, 1, 2)]),                         # y + height overflows 32 bits
    ]
    plan = dec.plan_step([pk[0]])
    for kw in bad:
        f = _fit_struct(**kw)
        nd = C.c_uint32(0)
        rc = L.h263cu_decode_step_device_tensor_fit(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data,
                                                    1, 1, 0, C.byref(target), C.byref(f), plan["errs"].ctypes.data, C.byref(nd))
        assert rc == _lib.ERR_BAD_ARGUMENT, kw
    nd = C.c_uint32(0)
    ok = _fit_struct(mode=_lib.FIT_LETTERBOX)
    assert L.h263cu_decode_step_device_tensor_fit(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, 1, 1,
                                                  0, C.byref(target), None, plan["errs"].ctypes.data, C.byref(nd)) == _lib.ERR_BAD_ARGUMENT
    assert L.h263cu_decode_step_device_tensor_fit(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, 1, 1,
                                                  0, None, C.byref(ok), plan["errs"].ctypes.data, C.byref(nd)) == _lib.ERR_BAD_ARGUMENT
    for kw in [dict(fit="squash"), dict(fit="center_crop"), dict(fit="center_crop", short_side=0), dict(fit="letterbox", short_side=256),
               dict(fit="letterbox", fill=256), dict(fit="letterbox", fill=(1, 2)), dict(fit="letterbox", fill=nan),
               dict(crops=[(0, 0, 10, 10), (0, 0, 10, 10)]), dict(crops=[(0, 0, 0, 10)]), dict(crops=[(-1, 0, 10, 10)])]:
        with pytest.raises(ValueError):
            dec.decode_step_device_tensor([pk[0]], (144, 176), **kw)
    # nothing moved: the packets decode bit-exact now
    for t in range(2):
        out, errs = dec.decode_step_device_tensor([pk[t]], (144, 176), dtype=torch.uint8, fit="center_crop", short_side=144)
        assert not errs.any()
        assert torch.equal(out[0].cpu(), expected_fit(ref[t], (144, 176), torch.uint8, "center_crop", 144)), t


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
            out, errs = dec.decode_step_device_tensor([s[t] for s in streams], (224, 224), out=out, fit="center_crop", short_side=256,
                                                      **IMAGENET)
            assert not errs.any()
            clones.append(out.clone())
    torch.cuda.synchronize()
    for t, cl in enumerate(clones):
        got = cl.cpu()
        for s in range(n):
            want = expected_fit(refs[s][t], (224, 224), torch.float16, "center_crop", 256, **IMAGENET)
            assert torch.equal(bits(got[s]), bits(want)), (t, s)


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
        refs = [oracle_decode_stream(s[: t + 1], deblock=deblock)[t] for s in streams]
        crops = [(i, 2 * i + 1, 176 - 3 * i - 1, 144 - 2 * i - 3) for i in range(n)]  # one box per input, all different
        outs, errs = g.decode_step_device_tensor([streams[s][t] for s in order], (100, 120), dtype=torch.float32, deblock=deblock,
                                                 stream_ids=order, fit="letterbox", fill=FILL, crops=crops, **IMAGENET)
        assert not errs.any() and len(outs) == nd
        for i, s in enumerate(order):
            got = outs[s % nd][s // nd].cpu()
            want = expected_fit(refs[s], (100, 120), torch.float32, "letterbox", None, crops[i], FILL, **IMAGENET)
            assert torch.equal(bits(got), bits(want)), (t, i, s)
    g.close()
