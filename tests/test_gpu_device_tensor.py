"""Decoded pictures resized and converted into caller-owned RGB tensors on the device (h263cu_decode_step_device_tensor,
BatchDecoder / DeviceGroup.decode_step_device_tensor): bit-exact against the numpy restatement of the definition
(resample_ref.py) applied to the oracle's RGBA, for every dtype and layout; nothing written outside the
[slot, 3, H, W] elements of decoded inputs; argument errors refused before any parser moves; ordering against the
consumer's torch stream without host synchronisation."""
import ctypes as C

import numpy as np
import pytest
import torch

import resample_ref as R
from helpers import oracle_decode_stream
from h263_rs_b200 import _lib, api, synth
from test_gpu_device_output import SIZES
from test_gpu_device_yuv import expected_planes
from test_gpu_parity import STREAMS, _packets

pytestmark = pytest.mark.gpu

BY_ID = {c["id"]: c for c in STREAMS}
DTYPES = [torch.uint8, torch.float32, torch.float16, torch.bfloat16]
IMAGENET = dict(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))


def rgb_of(ref):
    w, h = ref["info"]["width"], ref["info"]["height"]
    return np.asarray(ref["rgba"], np.uint8).reshape(h, w, 4)[..., :3]


def expected(ref, size, dtype, mean=None, std=None):
    """[3, H, W] torch tensor (CPU) of one decoded picture: the restatement of the definition; f16 / bf16 cast by torch
    (round to nearest even) from the restated float32."""
    v = R.resample(rgb_of(ref), *size)
    if dtype == torch.uint8:
        return torch.from_numpy(R.store(v, u8=True))
    mul, add = (1.0,) * 3, (0.0,) * 3
    if mean is not None or std is not None:
        mul, add = R.normalisation(mean if mean is not None else (0.0,) * 3, std if std is not None else (1.0,) * 3)
    return torch.from_numpy(R.store(v, mul, add)).to(dtype)


def bits(t):
    """A tensor's bytes, so that float comparisons are bit for bit (-0.0 and NaN patterns included)."""
    return t.contiguous().view(torch.uint8) if t.dtype != torch.uint8 else t


def view_of(n, size, dtype, layout):
    """A pattern-filled flat buffer and an [n, 3, H, W] view of it: contiguous, channels_last, or padded (rows, channel
    planes and slots with gaps, at an odd element offset)."""
    H, W = size
    if layout == "contiguous":
        st, total, off = (3 * H * W, H * W, W, 1), n * 3 * H * W, 0
    elif layout == "channels_last":
        st, total, off = (3 * H * W, 1, 3 * W, 3), n * 3 * H * W, 0
    else:
        row = W + 5
        plane = H * row + 3
        st, total, off = (3 * plane + 11, plane, row, 1), 13 + n * (3 * plane + 11), 13
    g = torch.Generator(device="cpu").manual_seed(n * 7 + H * 3 + W)
    flat = torch.randint(0, 256, (total + 64,), dtype=torch.uint8, generator=g)
    if dtype != torch.uint8:
        flat = (flat.to(torch.float32) * 0.37 - 20).to(dtype)
    flat = flat.cuda()
    return flat, flat.as_strided((n, 3, H, W), st, off)


def check_guarded(flat, before, view, pictures, size, dtype, **norm):
    """pictures: (slot, ref dict or None for an input that failed).  The decoded slots hold the expected values and every
    other element of the buffer is unchanged."""
    want = before.clone()
    wv = want.as_strided(view.shape, view.stride(), view.storage_offset())
    for slot, ref in pictures:
        if ref is not None:
            wv[slot] = expected(ref, size, dtype, **norm)
    got = flat.cpu()
    if not torch.equal(bits(got), bits(want)):
        gv = got.as_strided(view.shape, view.stride(), view.storage_offset())
        for slot, ref in pictures:
            if ref is not None:
                bad = int((bits(gv[slot]) != bits(wv[slot])).sum())
                assert bad == 0, ("slot", slot, bad, "elements differ")
        raise AssertionError("elements outside the decoded slots were written")
    return got


def decode_case(cid, size, dtype=torch.uint8, deblock=False, layout="contiguous", **norm):
    """Two streams (the case and a reseeded twin), step by step into a guarded view; size None = the picture's own."""
    case = dict(BY_ID[cid], deblock_flag=1) if deblock else BY_ID[cid]
    a, opt = _packets(case)
    b, _ = _packets(dict(case, seed=case["seed"] + 100))
    n = min(len(a), 5)
    streams = [a[:n], b[:n]]
    refs = [oracle_decode_stream(s, opt, deblock=deblock) for s in streams]
    size = size or (case["h"], case["w"])
    dec = api.BatchDecoder(2, case["w"], case["h"], decoder_options=opt, threads=2)
    flat, view = view_of(2, size, dtype, layout)
    before = flat.cpu()
    for t in range(n):
        out, errs = dec.decode_step_device_tensor([s[t] for s in streams], size, out=view, deblock=deblock, **norm)
        assert out is view
        for i in range(2):
            assert (errs[i] != 0) == isinstance(refs[i][t], int), (cid, t, i, int(errs[i]))
        pics = [(i, None if isinstance(refs[i][t], int) else refs[i][t]) for i in range(2)]
        before = check_guarded(flat, before, view, pics, size, dtype, **norm)
    return dec, [r[:n] for r in refs], view


@pytest.mark.parametrize("deblock", [False, True])
@pytest.mark.parametrize("cid", SIZES)
def test_identity_size_u8_is_the_oracle_rgb(cid, deblock):
    """At the picture's own size every weight is 0 or 1: uint8 output is the oracle's RGBA without alpha, deblocked
    through both deblock kernels (aligned and unaligned sizes)."""
    dec, refs, view = decode_case(cid, None, torch.uint8, deblock)
    # the last step's pictures, straight against the oracle's bytes (not only through the restatement)
    for i in range(2):
        if not isinstance(refs[i][-1], int):
            assert np.array_equal(view[i].cpu().numpy(), rgb_of(refs[i][-1]).transpose(2, 0, 1)), (cid, i)


RESIZED = [("cif_halfpel", (224, 224), False), ("config1_qcif", (288, 352), False), ("160x120_4mv_dquant", (75, 100), False),
           ("unaligned_15x15", (1, 1), False), ("unaligned_15x15", (37, 53), False), ("unaligned_161x99_odd", (64, 96), True),
           ("4cif", (224, 224), True)]


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
@pytest.mark.parametrize("cid,size,deblock", RESIZED)
def test_resized_bit_exact_for_every_dtype(cid, size, deblock, dtype):
    decode_case(cid, size, dtype, deblock)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16], ids=str)
def test_normalisation_bit_exact_and_close_to_torch(dtype):
    _, refs, _ = decode_case("cif_halfpel", (224, 224), dtype, **IMAGENET)
    # the familiar formula: (x / 255 - mean) / std on the restated values, within 2e-6 (float32 ulps of the result)
    out, errs = api.BatchDecoder(1, 352, 288, threads=1).decode_step_device_tensor(
        [_packets(BY_ID["cif_halfpel"])[0][0]], (224, 224), dtype=torch.float32, **IMAGENET)
    assert not errs.any()
    v = torch.from_numpy(R.resample(rgb_of(refs[0][0]), 224, 224))
    mean = torch.tensor(IMAGENET["mean"])[:, None, None]
    std = torch.tensor(IMAGENET["std"])[:, None, None]
    torch.testing.assert_close(out[0].cpu(), (v / 255 - mean) / std, rtol=0, atol=2e-6)


@pytest.mark.parametrize("dtype", [torch.uint8, torch.float16], ids=str)
@pytest.mark.parametrize("layout", ["contiguous", "channels_last", "padded"])
def test_layouts_and_guard_elements(layout, dtype):
    decode_case("config1_qcif", (100, 132), dtype, layout=layout)
    decode_case("unaligned_47x31", (31, 47), dtype, deblock=True, layout=layout)


def test_torch_channels_last_tensor():
    pk, opt = _packets(BY_ID["config1_qcif"])
    ref = oracle_decode_stream(pk[:2], opt)
    dec = api.BatchDecoder(1, 176, 144, threads=1)
    out = torch.empty((1, 3, 224, 224), dtype=torch.float16, device="cuda").to(memory_format=torch.channels_last)
    for t in range(2):
        got, errs = dec.decode_step_device_tensor([pk[t]], (224, 224), out=out)
        assert got is out and not errs.any()
        assert torch.equal(bits(out[0].cpu()), bits(expected(ref[t], (224, 224), torch.float16)))


def test_mixed_sizes_in_one_step_and_a_bad_packet():
    dims = [(176, 144), (47, 31), (161, 99), (128, 96)]
    streams = [synth.make_stream(w, h, 3, 700 + i, mv_mode=2) for i, (w, h) in enumerate(dims)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(4, 176, 144, threads=2)
    ids = [2, 0, 3, 1]  # input i -> slot i, whatever its stream
    size = (72, 88)
    flat, view = view_of(4, size, torch.float32, "padded")
    before = flat.cpu()
    for t in range(3):
        packets = [streams[s][t] for s in ids]
        bad = t == 1
        if bad:
            packets[1] = packets[1][:3]  # stream 0 fails to parse: its slot stays as it was, its stream untouched
        _, errs = dec.decode_step_device_tensor(packets, size, out=view, stream_ids=ids, **IMAGENET)
        assert bool(errs[1]) == bad and not errs[[0, 2, 3]].any()
        pics = [(i, refs[s][t]) for i, s in enumerate(ids)]
        if bad:
            pics[1] = (1, None)
        before = check_guarded(flat, before, view, pics, size, torch.float32, **IMAGENET)
        if bad:  # the stream carries on with the packet it failed on
            _, errs = dec.decode_step_device_tensor([streams[0][1]], size, out=view, stream_ids=[0], **IMAGENET)
            assert not errs.any()
            before = check_guarded(flat, before, view, [(0, refs[0][1])], size, torch.float32, **IMAGENET)


def test_picture_larger_than_the_context_is_a_per_picture_capacity_error():
    big, small = synth.make_stream(352, 288, 1, 711), synth.make_stream(176, 144, 1, 712)
    rs = oracle_decode_stream(small)
    dec = api.BatchDecoder(2, 176, 144, threads=2)
    flat, view = view_of(2, (50, 60), torch.uint8, "contiguous")
    before = flat.cpu()
    _, errs = dec.decode_step_device_tensor([big[0], small[0]], (50, 60), out=view)
    assert errs[0] == _lib.ERR_CAPACITY and errs[1] == 0
    check_guarded(flat, before, view, [(0, None), (1, rs[0])], (50, 60), torch.uint8)


def _tensor(base, strides=(3 * 144 * 176, 144 * 176, 176, 1), width=176, height=144, dtype=_lib.TENSOR_F32, reserved=0,
            mul=(1.0, 1.0, 1.0), add=(0.0, 0.0, 0.0), stream=None):
    return _lib.DeviceTensor(base, (C.c_int64 * 4)(*strides), width, height, dtype, reserved, (C.c_float * 3)(*mul),
                             (C.c_float * 3)(*add), stream)


def test_argument_errors_are_refused_before_any_parser_moves():
    pk = synth.make_stream(176, 144, 2, 721)
    ref = oracle_decode_stream(pk)
    dec = api.BatchDecoder(1, 176, 144, threads=1)
    L = _lib.lib()
    buf = torch.zeros(3 * 144 * 176, dtype=torch.float32, device="cuda")
    base = buf.data_ptr()
    pinned = torch.zeros(3 * 144 * 176, dtype=torch.float32, pin_memory=True)
    stream = torch.cuda.current_stream().cuda_stream or None
    inf, nan = float("inf"), float("nan")
    bad = [
        dict(dtype=4),                                       # unknown dtype
        dict(reserved=1),                                    # reserved not zero
        dict(width=0), dict(height=0),                       # empty output
        dict(width=16385), dict(height=16385),               # too large
        dict(strides=(0, 144 * 176, 176, 1)),                # strides <= 0
        dict(strides=(3 * 144 * 176, -1, 176, 1)),
        dict(strides=(3 * 144 * 176, 144 * 176, 0, 1)),
        dict(strides=(3 * 144 * 176, 144 * 176, 176, -1)),
        dict(base=base + 2),                                 # not aligned to the element size (f32)
        dict(base=base + 1, dtype=_lib.TENSOR_F16),          # (f16)
        dict(strides=(1, 1 << 38, 176, 1)),                  # a slot spans 2^40 bytes or more
        dict(strides=(1, 1, 1 << 37, 1)),
        dict(strides=(1, 1, 1, 1 << 62)),
        dict(mul=(1.0, inf, 1.0)), dict(add=(nan, 0.0, 0.0)),  # not finite
        dict(dtype=_lib.TENSOR_U8, mul=(1.0, 1.0, 2.0)),     # U8 takes no scale or offset
        dict(dtype=_lib.TENSOR_U8, add=(0.0, 0.5, 0.0)),
        dict(base=pinned.data_ptr()),                        # pinned host memory
        dict(base=0),                                        # null base
    ]
    plan = dec.plan_step([pk[0]])
    for kw in bad:
        target = _tensor(**dict(dict(base=base, stream=stream), **kw))
        nd = C.c_uint32(0)
        rc = L.h263cu_decode_step_device_tensor(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, 1,
                                                1, 0, C.byref(target), plan["errs"].ctypes.data, C.byref(nd))
        assert rc == _lib.ERR_BAD_ARGUMENT, kw
    nd = C.c_uint32(0)
    assert L.h263cu_decode_step_device_tensor(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, 1, 1,
                                              0, None, plan["errs"].ctypes.data, C.byref(nd)) == _lib.ERR_BAD_ARGUMENT
    # the Python layer refuses bad arguments with ValueError
    t = buf.view(1, 3, 144, 176)
    for kw in [
        dict(size=(144, 176), out=t.to(torch.int16)),                       # dtype
        dict(size=(144, 176), out=t.cpu()),                                 # device
        dict(size=(144, 176), out=t[:, :2]),                                # shape
        dict(size=(144, 170), out=t),
        dict(size=(0, 176)), dict(size=(144, 16385)), dict(size=144),        # size
        dict(size=(144, 176), dtype=torch.float64),
        dict(size=(144, 176), out=t, dtype=torch.float16),                  # out and dtype disagree
        dict(size=(144, 176), out=t.expand(1, 3, 144, 176).as_strided((1, 3, 144, 176), (0, 0, 176, 1))),  # zero stride
        dict(size=(144, 176), dtype=torch.uint8, mean=(0.5, 0.5, 0.5)),     # normalised uint8
        dict(size=(144, 176), dtype=torch.uint8, std=(0.5, 0.5, 0.5)),
        dict(size=(144, 176), mean=(0.5, 0.5)),                             # not three values
        dict(size=(144, 176), std=(0.5, 0.0, 0.5)),                         # std of zero
        dict(size=(144, 176), mean=(nan, 0.5, 0.5)),                        # not finite
    ]:
        with pytest.raises(ValueError):
            dec.decode_step_device_tensor([pk[0]], **kw)
    # nothing moved: the packets decode bit-exact now
    for t in range(2):
        out, errs = dec.decode_step_device_tensor([pk[t]], (144, 176), dtype=torch.uint8)
        assert not errs.any()
        assert np.array_equal(out[0].cpu().numpy(), rgb_of(ref[t]).transpose(2, 0, 1)), t


def test_ordering_on_the_consumer_stream_without_host_syncs():
    """One reused tensor, a non-default consumer stream that clones it after every call: each clone holds its own step."""
    n, t_steps = 24, 6
    streams = [synth.make_stream(352, 288, t_steps, 730 + s, mv_mode=s % 3) for s in range(n)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(n, 352, 288, threads=4)
    consumer = torch.cuda.Stream()
    clones = []
    with torch.cuda.stream(consumer):
        out = None
        for t in range(t_steps):
            out, errs = dec.decode_step_device_tensor([s[t] for s in streams], (224, 224), out=out, **IMAGENET)
            assert not errs.any()
            clones.append(out.clone())
    torch.cuda.synchronize()
    for t, cl in enumerate(clones):
        got = cl.cpu()
        for s in range(n):
            assert torch.equal(bits(got[s]), bits(expected(refs[s][t], (224, 224), torch.float16, **IMAGENET))), (t, s)


def test_host_rgba_yuv_and_tensor_steps_alternate():
    n, t_steps = 3, 12
    streams = [synth.make_stream(176, 144, t_steps, 740 + s, mv_mode=1) for s in range(n)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(n, 176, 144, threads=2)
    for t in range(t_steps):
        packets = [s[t] for s in streams]
        mode = t % 4
        if mode == 0:
            assert not dec.decode_step(packets).any()
            dec.ctx.sync()
            for s in range(n):
                assert np.array_equal(dec.ctx.read_rgba(s), refs[s][t]["rgba"]), (t, s)
        elif mode == 1:
            out, errs = dec.decode_step_device(packets)
            assert not errs.any()
            got = out.cpu().numpy().reshape(n, -1)
            for s in range(n):
                assert np.array_equal(got[s], refs[s][t]["rgba"]), (t, s)
        elif mode == 2:
            out, errs = dec.decode_step_device_yuv(packets, layout="nv12")
            assert not errs.any()
            for s in range(n):
                for k, want in enumerate(expected_planes(refs[s][t], "nv12")):
                    assert np.array_equal(out[k][s].cpu().numpy().reshape(want.shape), want), (t, s, k)
        else:
            out, errs = dec.decode_step_device_tensor(packets, (96, 128), dtype=torch.bfloat16)
            assert not errs.any()
            for s in range(n):
                assert torch.equal(bits(out[s].cpu()), bits(expected(refs[s][t], (96, 128), torch.bfloat16))), (t, s)
        if mode:
            for s in range(n):
                with pytest.raises(_lib.H263Error) as e:
                    dec.ctx.read_rgba(s)
                assert e.value.code == _lib.ERR_NO_PICTURE
        for s in range(n):
            y, cb, cr = dec.ctx.read_yuv(s)
            r = refs[s][t]
            assert np.array_equal(y, r["y"]) and np.array_equal(cb, r["cb"]) and np.array_equal(cr, r["cr"]), (t, s)


@pytest.mark.parametrize("cid,deblock", [("unaligned_161x99_odd", False), ("unaligned_47x31", True), ("cif_halfpel", True)])
def test_generic_kernel_fallback(monkeypatch, cid, deblock):
    """H263CU_KERNEL=mb: the warp-per-macroblock recon kernel, and the generic deblock kernel for every size."""
    monkeypatch.setenv("H263CU_KERNEL", "mb")
    dec, _, _ = decode_case(cid, (70, 90), torch.float16, deblock)
    assert dec.ctx.tiled_launch_count() == 0


@pytest.mark.parametrize("devices", [[0, 0, 0], "all"])
def test_device_group(devices):
    if devices == "all":
        if torch.cuda.device_count() < 2:
            pytest.skip("one GPU")
        devices = list(range(torch.cuda.device_count()))
    nd, per = len(devices), 2
    n, t_steps = nd * per, 3
    streams = [synth.make_stream(176, 144, t_steps, 760 + s, mv_mode=s % 3) for s in range(n)]
    g = api.DeviceGroup(devices, per, 176, 144, threads=4)
    for t in range(t_steps):
        deblock = t == 2
        refs = [oracle_decode_stream(s[: t + 1], deblock=deblock)[t] for s in streams]
        outs, errs = g.decode_step_device_tensor([s[t] for s in streams], (112, 112), dtype=torch.float32, deblock=deblock, **IMAGENET)
        assert not errs.any() and len(outs) == nd
        for s in range(n):
            got = outs[s % nd][s // nd].cpu()
            assert torch.equal(bits(got), bits(expected(refs[s], (112, 112), torch.float32, **IMAGENET))), (t, s)
    g.close()
