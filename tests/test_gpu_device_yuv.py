"""Decoded planes straight into caller-owned device memory (h263cu_decode_step_device_yuv, BatchDecoder / DeviceGroup
.decode_step_device_yuv), in the I420 and NV12 layouts: bit-exact against the oracle's planes (deblocked on request),
nothing written outside the slot rectangles, argument errors refused before any parser moves, and ordering against the
consumer's torch stream without host synchronisation."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle_lib as O
from helpers import oracle_decode_stream
from h263_rs_b200 import _lib, api, synth
from test_gpu_device_output import SIZES
from test_gpu_parity import STREAMS, _packets

pytestmark = pytest.mark.gpu

BY_ID = {c["id"]: c for c in STREAMS}
LAYOUTS = ["i420", "nv12"]


def plane_specs(width, height, layout):
    """(name, rows, samples per row, bytes per sample) of each plane of a width x height slot."""
    ch, cw = (height + 1) // 2, (width + 1) // 2
    if layout == "nv12":
        return [("y", height, width, 1), ("uv", ch, cw, 2)]
    return [("y", height, width, 1), ("cb", ch, cw, 1), ("cr", ch, cw, 1)]


def guarded(n, width, height, layout, row_pad=12, gap=40):
    """One pattern-filled byte buffer per plane, with padded rows (pitch a multiple of 4, not of 16) and a gap between
    slots.  Returns (the views the API takes, the plane records)."""
    views, planes = [], []
    for k, (name, rows, cols, bps) in enumerate(plane_specs(width, height, layout)):
        row_bytes = cols * bps
        pitch = (row_bytes + 3) // 4 * 4 + row_pad
        stride = pitch * rows + gap
        total = stride * n + 64
        flat = ((torch.arange(total, dtype=torch.int64, device="cuda") * (37 + 2 * k) + 11) % 251).to(torch.uint8)
        if bps == 2:
            view = flat.as_strided((n, rows, cols, 2), (stride, pitch, 2, 1))
        else:
            view = flat.as_strided((n, rows, cols), (stride, pitch, 1))
        views.append(view)
        planes.append(dict(flat=flat, pitch=pitch, stride=stride, rows=rows, row_bytes=row_bytes,
                           pattern=flat.cpu().numpy().copy()))
    return tuple(views), planes


def expected_planes(ref, layout, deblock=False):
    """The bytes of each plane of a decoded picture, [rows, row bytes]: the oracle's planes, deblocked on request
    (deblock::deblock(plane, plane_width, QUANT_TO_STRENGTH[pquant]))."""
    w, h = ref["info"]["width"], ref["info"]["height"]
    cw, ch = (w + 1) // 2, (h + 1) // 2
    y, cb, cr = ref["y"], ref["cb"], ref["cr"]
    if deblock:
        s = O.lib().orc_quant_to_strength(ref["info"]["quant"])
        y, cb, cr = O.deblock(y, w, s), O.deblock(cb, cw, s), O.deblock(cr, cw, s)
    y, cb, cr = (np.asarray(p, np.uint8).reshape(r, c) for p, r, c in ((y, h, w), (cb, ch, cw), (cr, ch, cw)))
    if layout == "nv12":
        return [y, np.stack([cb, cr], axis=-1).reshape(ch, 2 * cw)]
    return [y, cb, cr]


def check_guarded(planes, pictures, layout):
    """pictures: (slot, ref dict or None for an input that failed, deblock).  Every plane of every picture is
    bit-exact, and every byte outside the slot rectangles of the decoded pictures (and every byte of a failed input's
    slots) is unchanged.  Then the current contents become the new pattern."""
    for k, pl in enumerate(planes):
        after = pl["flat"].cpu().numpy()
        may_write = np.zeros(after.size, bool)
        pitch, stride, rows = pl["pitch"], pl["stride"], pl["rows"]
        for slot, ref, deblock in pictures:
            if ref is None:
                continue
            want = expected_planes(ref, layout, deblock)[k]
            region = after[slot * stride : slot * stride + rows * pitch].reshape(rows, pitch)
            got = region[: want.shape[0], : want.shape[1]]
            assert np.array_equal(got, want), ("plane", k, "slot", slot, int((got != want).sum()))
            may_write[slot * stride : slot * stride + rows * pitch].reshape(rows, pitch)[:, : pl["row_bytes"]] = True
        changed = (after != pl["pattern"]) & ~may_write
        assert not changed.any(), ("plane", k, "bytes written outside the slot rectangles", np.flatnonzero(changed)[:8])
        pl["pattern"] = after.copy()


def pictures_of(refs, t, deblock=False, slots=None):
    out = []
    for i, r in enumerate(refs):
        slot = i if slots is None else slots[i]
        out.append((slot, None if isinstance(r[t], int) else r[t], deblock))
    return out


def decode_case(cid, layout, deblock=False):
    """Two streams (the case and a reseeded twin), decoded step by step into guarded planes whose slot is exactly the
    picture size.  Returns the number of steps that decoded a picture and the decoder."""
    case = dict(BY_ID[cid], deblock_flag=1) if deblock else BY_ID[cid]
    a, opt = _packets(case)
    b, _ = _packets(dict(case, seed=case["seed"] + 100))
    n = min(len(a), 5)
    streams = [a[:n], b[:n]]
    refs = [oracle_decode_stream(s, opt) for s in streams]
    w, h = case["w"], case["h"]
    dec = api.BatchDecoder(2, w, h, decoder_options=opt, threads=2)
    views, planes = guarded(2, w, h, layout)
    stepped = 0
    for t in range(n):
        out, errs = dec.decode_step_device_yuv([s[t] for s in streams], out=views, layout=layout, deblock=deblock)
        assert len(out) == len(views) and all(o is v for o, v in zip(out, views))
        for i in range(2):
            assert (errs[i] != 0) == isinstance(refs[i][t], int), (cid, t, i, int(errs[i]))
        stepped += int((errs == 0).any())
        check_guarded(planes, pictures_of(refs, t, deblock), layout)
    return stepped, dec


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("cid", SIZES)
def test_planes_bit_exact_and_inside_the_slot(cid, layout):
    stepped, dec = decode_case(cid, layout)
    assert dec.ctx.tiled_launch_count() == stepped, cid


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("cid", ["config1_qcif", "4cif", "200x100_unaligned", "unaligned_161x99_odd", "unaligned_47x31",
                                 "unaligned_17x33"])
def test_deblocked_planes(cid, layout):
    """Both deblock kernels (aligned sizes take the register-resident one), and widths with w % 4 != 0 whose last
    words are cut at the picture's edge."""
    decode_case(cid, layout, deblock=True)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("cid", ["unaligned_161x99_odd", "unaligned_47x31", "cif_halfpel"])
def test_generic_kernel_fallback(monkeypatch, cid, layout):
    """H263CU_KERNEL=mb: the warp-per-macroblock kernel stores the planes cut to the picture."""
    monkeypatch.setenv("H263CU_KERNEL", "mb")
    _, dec = decode_case(cid, layout)
    assert dec.ctx.tiled_launch_count() == 0


@pytest.mark.parametrize("layout", LAYOUTS)
def test_mixed_sizes_in_one_step_guard_bytes_and_a_bad_packet(layout):
    dims = [(176, 144), (47, 31), (161, 99), (128, 96)]
    streams = [synth.make_stream(w, h, 3, 700 + i, mv_mode=2) for i, (w, h) in enumerate(dims)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(4, 176, 144, threads=2)
    ids = [2, 0, 3, 1]  # input i -> slot i, whatever its stream
    views, planes = guarded(4, 176, 144, layout)
    for t in range(3):
        packets = [streams[s][t] for s in ids]
        bad = t == 1
        if bad:
            packets[1] = packets[1][:3]  # stream 0 fails to parse: its slots stay as they were, its stream untouched
        _, errs = dec.decode_step_device_yuv(packets, out=views, layout=layout, stream_ids=ids)
        assert bool(errs[1]) == bad and not errs[[0, 2, 3]].any()
        pics = pictures_of([refs[s] for s in ids], t)
        if bad:
            pics[1] = (1, None, False)
        check_guarded(planes, pics, layout)
        if bad:  # the stream carries on with the packet it failed on
            _, errs = dec.decode_step_device_yuv([streams[0][1]], out=views, layout=layout, stream_ids=[0])
            assert not errs.any()
            check_guarded(planes, [(0, refs[0][1], False)], layout)


def test_picture_larger_than_the_slot_is_a_per_picture_capacity_error():
    big, small = synth.make_stream(352, 288, 2, 711), synth.make_stream(176, 144, 2, 712)
    rb, rs = oracle_decode_stream(big), oracle_decode_stream(small)
    dec = api.BatchDecoder(2, 352, 288, threads=2)
    views, planes = guarded(2, 176, 144, "i420")
    _, errs = dec.decode_step_device_yuv([big[0], small[0]], out=views)
    assert errs[0] == _lib.ERR_CAPACITY and errs[1] == 0
    check_guarded(planes, [(0, None, False), (1, rs[0], False)], "i420")
    with pytest.raises(_lib.H263Error):
        dec.ctx.stream_info(0)  # untouched: no picture yet
    # the same packet with a slot large enough, then the stream goes on
    for t in range(2):
        out, errs = dec.decode_step_device_yuv([big[t]], out=None, layout="nv12")
        assert not errs.any() and tuple(out[0].shape) == (1, 288, 352) and tuple(out[1].shape) == (1, 144, 176, 2)
        want = expected_planes(rb[t], "nv12")
        assert np.array_equal(out[0][0].cpu().numpy(), want[0]) and np.array_equal(out[1][0].cpu().numpy().reshape(144, 352), want[1])


def _yuv(planes, width, height, fmt=_lib.YUV_I420, reserved=0, stream=None):
    return _lib.DeviceYuv((_lib.DevicePlane * 3)(*[_lib.DevicePlane(*p) for p in planes]), width, height, fmt, reserved, stream)


def test_argument_errors_are_refused_before_any_parser_moves():
    pk = synth.make_stream(176, 144, 2, 721)
    ref = oracle_decode_stream(pk)
    dec = api.BatchDecoder(1, 176, 144, threads=1)
    L = _lib.lib()
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    base = buf.data_ptr()
    assert base % 256 == 0
    pinned = torch.zeros(1 << 15, dtype=torch.uint8, pin_memory=True)
    stream = torch.cuda.current_stream().cuda_stream or None
    # QCIF I420, tight: Y rows 176 B, chroma rows 88 B (a multiple of 4, not of 16)
    y, cb, cr = (base, 176, 176 * 144), (base + 176 * 144, 88, 88 * 72), (base + 176 * 144 + 88 * 72, 88, 88 * 72)
    good = dict(planes=[y, cb, cr], width=176, height=144, fmt=_lib.YUV_I420, reserved=0)
    nv = dict(good, planes=[y, (base + 176 * 144, 176, 176 * 72), (0, 0, 0)], fmt=_lib.YUV_NV12)
    bad = [
        dict(good, fmt=2),                                                      # unknown format
        dict(good, reserved=1),                                                 # reserved not zero
        dict(nv, planes=[nv["planes"][0], nv["planes"][1], (0, 4, 0)]),         # NV12 with a plane[2]
        dict(nv, planes=[nv["planes"][0], nv["planes"][1], cr]),                # NV12 with a plane[2]
        dict(good, width=0),                                                    # empty slot
        dict(good, height=0),
        dict(good, planes=[(base + 2, 176, 176 * 144), cb, cr]),                # base not 4-byte aligned
        dict(good, planes=[y, (base + 176 * 144 + 2, 88, 88 * 72), cr]),
        dict(good, planes=[(base, 178, 178 * 144), cb, cr]),                    # pitch not a multiple of 4
        dict(good, planes=[y, cb, (cr[0], 88, 88 * 72 + 2)]),                   # stride not a multiple of 4
        dict(good, planes=[(base, 172, 172 * 144), cb, cr]),                    # pitch below the slot row bytes
        dict(good, planes=[y, (cb[0], 84, 84 * 72), cr]),
        dict(nv, planes=[y, (base + 176 * 144, 172, 172 * 72), (0, 0, 0)]),     # NV12 CbCr rows are 2 * 88 bytes
        dict(good, planes=[(base, 1 << 32, 1 << 39), cb, cr]),                  # pitch >= 2^32
        dict(good, planes=[(base, 176, 176 * 143), cb, cr]),                    # stride below pitch * rows
        dict(good, planes=[y, cb, (cr[0], 88, 88 * 71)]),
        dict(good, planes=[(base, 176, 1 << 40), cb, cr]),                      # stride >= 2^40
        dict(good, planes=[(pinned.data_ptr(), 176, 176 * 144), cb, cr]),       # pinned host memory
        dict(good, planes=[y, cb, (pinned.data_ptr(), 88, 88 * 72)]),
        dict(good, planes=[(0, 176, 176 * 144), cb, cr]),                       # null base
    ]
    plan = dec.plan_step([pk[0]])
    for kw in bad:
        target = _yuv(kw["planes"], kw["width"], kw["height"], kw["fmt"], kw["reserved"], stream)
        nd = C.c_uint32(0)
        rc = L.h263cu_decode_step_device_yuv(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, 1, 1,
                                             0, C.byref(target), plan["errs"].ctypes.data, C.byref(nd))
        assert rc == _lib.ERR_BAD_ARGUMENT, kw
    nd = C.c_uint32(0)
    assert L.h263cu_decode_step_device_yuv(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, 1, 1,
                                           0, None, plan["errs"].ctypes.data, C.byref(nd)) == _lib.ERR_BAD_ARGUMENT
    # the Python layer refuses bad tensors with ValueError
    ty = buf[: 176 * 144].view(1, 144, 176)
    tc = buf[176 * 144 : 176 * 144 + 88 * 72].view(1, 72, 88)
    tr = buf[176 * 144 + 88 * 72 : 176 * 144 + 2 * 88 * 72].view(1, 72, 88)
    tuv = buf[176 * 144 : 176 * 144 + 176 * 72].view(1, 72, 88, 2)
    for out, layout in [
        ((ty.to(torch.int16), tc, tr), "i420"),                                 # dtype
        ((ty.cpu(), tc, tr), "i420"),                                           # device
        ((ty, tc[:, :71], tr), "i420"),                                         # shape
        ((ty, tc, tr[:, :, :87]), "i420"),
        ((ty, tc, tr), "nv12"),                                                 # three planes for NV12
        ((ty, tuv), "i420"),                                                    # two planes for I420
        ((ty, tuv[..., :1]), "nv12"),
        ((ty.transpose(1, 2).contiguous().transpose(1, 2), tc, tr), "i420"),   # samples not tight
        ((buf[2 : 2 + 176 * 144].view(1, 144, 176), tc, tr), "i420"),           # base not 4-byte aligned
        ((buf[: 178 * 144].view(1, 144, 178)[:, :, :176], tc, tr), "i420"),     # pitch not a multiple of 4
        ((ty, buf[:200].as_strided((2, 72, 88), (88 * 70, 88, 1)), tr), "i420"),  # stride below pitch * rows
        ((ty, tc, tr), "yuyv"),                                                 # unknown layout
    ]:
        with pytest.raises(ValueError):
            dec.decode_step_device_yuv([pk[0]], out=out, layout=layout)
    # nothing moved: the packets decode bit-exact now
    for t in range(2):
        out, errs = dec.decode_step_device_yuv([pk[t]])
        assert not errs.any()
        want = expected_planes(ref[t], "i420")
        for k in range(3):
            assert np.array_equal(out[k][0].cpu().numpy(), want[k]), (t, k)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_ordering_on_the_consumer_stream_without_host_syncs(layout):
    """One reused set of planes, a non-default consumer stream that clones them after every call: each clone holds its
    own step, so the library's writes waited for the clone before and the clone waited for the writes."""
    n, t_steps = 24, 6
    streams = [synth.make_stream(352, 288, t_steps, 730 + s, mv_mode=s % 3) for s in range(n)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(n, 352, 288, threads=4)
    consumer = torch.cuda.Stream()
    clones = []
    with torch.cuda.stream(consumer):
        out = None
        for t in range(t_steps):
            out, errs = dec.decode_step_device_yuv([s[t] for s in streams], out=out, layout=layout)
            assert not errs.any()
            clones.append([p.clone() for p in out])
    torch.cuda.synchronize()
    for t, cl in enumerate(clones):
        got = [p.cpu().numpy().reshape(n, p.shape[1], -1) for p in cl]
        for s in range(n):
            for k, want in enumerate(expected_planes(refs[s][t], layout)):
                assert np.array_equal(got[k][s], want), (t, s, k)


def test_host_device_rgba_and_device_yuv_steps_alternate():
    n, t_steps = 3, 9
    streams = [synth.make_stream(176, 144, t_steps, 740 + s, mv_mode=1) for s in range(n)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(n, 176, 144, threads=2)
    for t in range(t_steps):
        packets = [s[t] for s in streams]
        mode = t % 3
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
        else:
            layout = LAYOUTS[(t // 3) % 2]
            out, errs = dec.decode_step_device_yuv(packets, layout=layout)
            assert not errs.any()
            for s in range(n):
                for k, want in enumerate(expected_planes(refs[s][t], layout)):
                    assert np.array_equal(out[k][s].cpu().numpy().reshape(want.shape), want), (t, s, k)
        if mode:
            for s in range(n):
                with pytest.raises(_lib.H263Error) as e:
                    dec.ctx.read_rgba(s)
                assert e.value.code == _lib.ERR_NO_PICTURE
        for s in range(n):
            y, cb, cr = dec.ctx.read_yuv(s)
            r = refs[s][t]
            assert np.array_equal(y, r["y"]) and np.array_equal(cb, r["cb"]) and np.array_equal(cr, r["cr"]), (t, s)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("devices", [[0, 0, 0], "all"])
def test_device_group(devices, layout):
    if devices == "all":
        if torch.cuda.device_count() < 2:
            pytest.skip("one GPU")
        devices = list(range(torch.cuda.device_count()))
    nd, per = len(devices), 2
    n, t_steps = nd * per, 3
    streams = [synth.make_stream(176, 144, t_steps, 760 + s, mv_mode=s % 3) for s in range(n)]
    refs = [oracle_decode_stream(s) for s in streams]
    g = api.DeviceGroup(devices, per, 176, 144, threads=4)
    for t in range(t_steps):
        outs, errs = g.decode_step_device_yuv([s[t] for s in streams], layout=layout, deblock=t == 2)
        assert not errs.any() and len(outs) == nd
        for s in range(n):
            for k, want in enumerate(expected_planes(refs[s][t], layout, deblock=t == 2)):
                got = outs[s % nd][k][s // nd].cpu().numpy().reshape(want.shape)
                assert np.array_equal(got, want), (t, s, k)
    g.close()


@pytest.mark.parametrize("cid", ["cif_halfpel", "unaligned_161x99_odd"])
def test_i420_and_nv12_agree(cid):
    """The two layouts of the same stream hold the same samples: NV12's pairs are I420's Cb and Cr, interleaved."""
    case = BY_ID[cid]
    pk, opt = _packets(case)
    w, h = case["w"], case["h"]
    a = api.BatchDecoder(1, w, h, decoder_options=opt, threads=1)
    b = api.BatchDecoder(1, w, h, decoder_options=opt, threads=1)
    for t in range(min(len(pk), 4)):
        (y1, cb, cr), e1 = a.decode_step_device_yuv([pk[t]], layout="i420")
        (y2, uv), e2 = b.decode_step_device_yuv([pk[t]], layout="nv12")
        assert not e1.any() and not e2.any()
        assert torch.equal(y1, y2)
        assert torch.equal(uv[..., 0], cb) and torch.equal(uv[..., 1], cr)
