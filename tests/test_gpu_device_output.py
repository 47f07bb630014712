"""RGBA straight into caller-owned device memory (h263cu_decode_step_device, BatchDecoder / DeviceGroup
.decode_step_device): bit-exact against the oracle, nothing written outside the slot rectangles, argument errors
refused before any parser moves, and ordering against the consumer's torch stream without host synchronisation."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import oracle_decode_stream
from h263_rs_b200 import _lib, api, synth
from test_gpu_parity import STREAMS, _packets

pytestmark = pytest.mark.gpu

BY_ID = {c["id"]: c for c in STREAMS}
SIZES = ["config1_qcif", "cif_halfpel", "4cif", "160x120_4mv_dquant", "unaligned_161x99_odd", "unaligned_15x15",
         "unaligned_17x33", "unaligned_47x31", "unaligned_480x360"]


def guarded(n, width, height, row_pad=48, gap=80):
    """A [n, height, width, 4] view into a pattern-filled byte buffer with padded rows and a gap between slots.
    Returns (view, flat buffer, row_pitch, pic_stride, pattern)."""
    row_pitch = (4 * width + 15) // 16 * 16 + row_pad
    pic_stride = row_pitch * height + gap
    total = pic_stride * n + 64
    pattern = (torch.arange(total, dtype=torch.int64, device="cuda") * 37 + 11) % 251
    flat = pattern.to(torch.uint8)
    view = flat.as_strided((n, height, width, 4), (pic_stride, row_pitch, 4, 1))
    return view, flat, row_pitch, pic_stride, flat.cpu().numpy().copy()


def check_guarded(flat, row_pitch, pic_stride, width, height, pictures, pattern):
    """pictures: (slot, w, h, rgba or None for an input that failed).  The pictures are bit-exact, and every byte
    outside the slot rectangles of the decoded pictures (and every byte of a failed input's slot) is unchanged."""
    after = flat.cpu().numpy()
    may_write = np.zeros(after.size, bool)
    for slot, w, h, rgba in pictures:
        if rgba is None:
            continue
        region = after[slot * pic_stride : slot * pic_stride + height * row_pitch].reshape(height, row_pitch)
        got = region[:h, : 4 * w].reshape(-1)
        assert np.array_equal(got, rgba), ("slot", slot, int((got != rgba).sum()))
        may_write[slot * pic_stride : slot * pic_stride + height * row_pitch].reshape(height, row_pitch)[:, : 4 * width] = True
    changed = (after != pattern) & ~may_write
    assert not changed.any(), ("bytes written outside the slot rectangles", np.flatnonzero(changed)[:8])


def pictures_of(refs, t, slots=None):
    out = []
    for i, r in enumerate(refs):
        rt = r[t]
        slot = i if slots is None else slots[i]
        if isinstance(rt, int):
            out.append((slot, 0, 0, None))
        else:
            out.append((slot, rt["info"]["width"], rt["info"]["height"], rt["rgba"]))
    return out


def decode_case(ids, deblock=False):
    """Two streams per case (the case and a reseeded twin), decoded step by step into a guarded buffer whose slot is
    exactly the picture size."""
    for cid in ids:
        case = dict(BY_ID[cid], deblock_flag=1) if deblock else BY_ID[cid]
        a, opt = _packets(case)
        b, _ = _packets(dict(case, seed=case["seed"] + 100))
        n = min(len(a), 5)
        streams = [a[:n], b[:n]]
        refs = [oracle_decode_stream(s, opt, deblock=deblock) for s in streams]
        w, h = case["w"], case["h"]
        dec = api.BatchDecoder(2, w, h, decoder_options=opt, threads=2)
        view, flat, pitch, stride, pattern = guarded(2, w, h)
        flags = _lib.OUT_RGBA | (_lib.OUT_DEBLOCK if deblock else 0)
        stepped = 0
        for t in range(n):
            out, errs = dec.decode_step_device([s[t] for s in streams], out=view, out_flags=flags)
            assert out is view
            for i in range(2):
                assert (errs[i] != 0) == isinstance(refs[i][t], int), (cid, t, i, int(errs[i]))
            stepped += int((errs == 0).any())
            check_guarded(flat, pitch, stride, w, h, pictures_of(refs, t), pattern)
            pattern = flat.cpu().numpy().copy()
        assert dec.ctx.tiled_launch_count() == stepped, cid


@pytest.mark.parametrize("cid", SIZES)
def test_device_output_bit_exact_and_inside_the_slot(cid):
    decode_case([cid])


@pytest.mark.parametrize("cid", ["config1_qcif", "4cif", "200x100_unaligned", "unaligned_161x99_odd", "unaligned_47x31",
                                 "unaligned_17x33"])
def test_device_output_deblocked(cid):
    """Both deblock kernels (aligned sizes take the register-resident one) and widths with w % 4 != 0, whose last RGBA
    quad is cut at the picture's edge."""
    decode_case([cid], deblock=True)


def test_mixed_sizes_in_one_step_guard_bytes_and_a_bad_packet():
    dims = [(176, 144), (47, 31), (161, 99), (128, 96)]
    streams = [synth.make_stream(w, h, 3, 500 + i, mv_mode=2) for i, (w, h) in enumerate(dims)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(4, 176, 144, threads=2)
    ids = [2, 0, 3, 1]  # input i -> slot i, whatever its stream
    view, flat, pitch, stride, pattern = guarded(4, 176, 144)
    for t in range(3):
        packets = [streams[s][t] for s in ids]
        bad = t == 1
        if bad:
            packets[1] = packets[1][:3]  # stream 0 fails to parse: its slot stays as it was, its stream untouched
        _, errs = dec.decode_step_device(packets, out=view, stream_ids=ids)
        assert bool(errs[1]) == bad and not errs[[0, 2, 3]].any()
        pics = pictures_of([refs[s] for s in ids], t)
        if bad:
            pics[1] = (1, 0, 0, None)
        check_guarded(flat, pitch, stride, 176, 144, pics, pattern)
        if bad:  # the stream carries on with the packet it failed on
            _, errs = dec.decode_step_device([streams[0][1]], out=view, stream_ids=[0])
            assert not errs.any()
            check_guarded(flat, pitch, stride, 176, 144, [(0, 176, 144, refs[0][1]["rgba"])], flat.cpu().numpy())
        pattern = flat.cpu().numpy().copy()


def test_picture_larger_than_the_slot_is_a_per_picture_capacity_error():
    big, small = synth.make_stream(352, 288, 2, 601), synth.make_stream(176, 144, 2, 602)
    rb, rs = oracle_decode_stream(big), oracle_decode_stream(small)
    dec = api.BatchDecoder(2, 352, 288, threads=2)
    view, flat, pitch, stride, pattern = guarded(2, 176, 144)
    _, errs = dec.decode_step_device([big[0], small[0]], out=view)
    assert errs[0] == _lib.ERR_CAPACITY and errs[1] == 0
    check_guarded(flat, pitch, stride, 176, 144, [(0, 0, 0, None), (1, 176, 144, rs[0]["rgba"])], pattern)
    with pytest.raises(_lib.H263Error):
        dec.ctx.stream_info(0)  # untouched: no picture yet
    # the same packet with a slot large enough, then the stream goes on
    for t in range(2):
        out, errs = dec.decode_step_device([big[t]], out=None)
        assert not errs.any() and tuple(out.shape) == (1, 288, 352, 4)
        assert np.array_equal(out[0].cpu().numpy().reshape(-1), rb[t]["rgba"])


def test_argument_errors_are_refused_before_any_parser_moves():
    pk = synth.make_stream(176, 144, 2, 611)
    ref = oracle_decode_stream(pk)
    dec = api.BatchDecoder(1, 176, 144, threads=1)
    L = _lib.lib()
    buf = torch.zeros(176 * 144 * 4 * 2 + 4096, dtype=torch.uint8, device="cuda")
    base = buf.data_ptr()
    assert base % 256 == 0
    pinned = torch.zeros(176 * 144 * 4 + 64, dtype=torch.uint8, pin_memory=True)
    stream = torch.cuda.current_stream().cuda_stream or None
    good = dict(base=base, row_pitch=704, pic_stride=704 * 144, width=176, height=144)
    bad = [
        dict(good, base=base + 4),                 # misaligned base
        dict(good, row_pitch=712),                 # pitch not a multiple of 16
        dict(good, row_pitch=688),                 # pitch below 4 * width
        dict(good, pic_stride=704 * 143),          # stride below pitch * height
        dict(good, base=pinned.data_ptr()),        # pinned host memory
        dict(good, width=0),                       # empty slot
        dict(good, pic_stride=704 * 144 + 8),      # stride not a multiple of 16
    ]
    plan = dec.plan_step([pk[0]])
    for kw in bad:
        target = _lib.DeviceRgba(kw["base"], kw["row_pitch"], kw["pic_stride"], kw["width"], kw["height"], stream)
        nd = C.c_uint32(0)
        rc = L.h263cu_decode_step_device(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, 1, 1,
                                         _lib.OUT_RGBA, C.byref(target), plan["errs"].ctypes.data, C.byref(nd))
        assert rc == _lib.ERR_BAD_ARGUMENT, kw
    nd = C.c_uint32(0)
    assert L.h263cu_decode_step_device(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, 1, 1,
                                       _lib.OUT_RGBA, None, plan["errs"].ctypes.data, C.byref(nd)) == _lib.ERR_BAD_ARGUMENT
    # the Python layer refuses the same tensors with ValueError
    flat = buf[: 704 * 144 * 2 + 64]
    for shape, strides, off in [((1, 144, 176, 4), (704 * 144, 712, 4, 1), 0), ((1, 144, 176, 4), (704 * 144, 704, 4, 1), 4),
                                ((2, 144, 176, 4), (704 * 100, 704, 4, 1), 0), ((1, 144, 176, 4), (704 * 144, 704, 1, 176), 0)]:
        with pytest.raises(ValueError):
            dec.decode_step_device([pk[0]], out=flat[off:].as_strided(shape, strides))
    with pytest.raises(ValueError):
        dec.decode_step_device([pk[0]], out=torch.zeros((1, 144, 176, 4), dtype=torch.uint8))  # host tensor
    # nothing moved: the packets decode bit-exact now
    for t in range(2):
        out, errs = dec.decode_step_device([pk[t]])
        assert not errs.any()
        assert np.array_equal(out[0].cpu().numpy().reshape(-1), ref[t]["rgba"]), t


def test_ordering_on_the_consumer_stream_without_host_syncs():
    """One reused buffer, a non-default consumer stream that clones it after every call: each clone holds its own
    step, so the library's writes waited for the clone before and the clone waited for the writes."""
    n, t_steps = 24, 6
    streams = [synth.make_stream(352, 288, t_steps, 620 + s, mv_mode=s % 3) for s in range(n)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(n, 352, 288, threads=4)
    consumer = torch.cuda.Stream()
    clones = []
    with torch.cuda.stream(consumer):
        buf = torch.empty((n, 288, 352, 4), dtype=torch.uint8, device="cuda")
        for t in range(t_steps):
            out, errs = dec.decode_step_device([s[t] for s in streams], out=buf)
            assert not errs.any()
            clones.append(out.clone())
    torch.cuda.synchronize()
    for t, cl in enumerate(clones):
        got = cl.cpu().numpy().reshape(n, -1)
        for s in range(n):
            assert np.array_equal(got[s], refs[s][t]["rgba"]), (t, s)


def test_host_and_device_steps_alternate():
    n, t_steps = 3, 6
    streams = [synth.make_stream(176, 144, t_steps, 640 + s, mv_mode=1) for s in range(n)]
    refs = [oracle_decode_stream(s) for s in streams]
    dec = api.BatchDecoder(n, 176, 144, threads=2)
    for t in range(t_steps):
        packets = [s[t] for s in streams]
        if t % 2:
            out, errs = dec.decode_step_device(packets)
            assert not errs.any()
            got = out.cpu().numpy().reshape(n, -1)
            for s in range(n):
                assert np.array_equal(got[s], refs[s][t]["rgba"]), (t, s)
                with pytest.raises(_lib.H263Error) as e:
                    dec.ctx.read_rgba(s)
                assert e.value.code == _lib.ERR_NO_PICTURE
        else:
            assert not dec.decode_step(packets).any()
            dec.ctx.sync()
            for s in range(n):
                assert np.array_equal(dec.ctx.read_rgba(s), refs[s][t]["rgba"]), (t, s)
        for s in range(n):
            y, cb, cr = dec.ctx.read_yuv(s)
            r = refs[s][t]
            assert np.array_equal(y, r["y"]) and np.array_equal(cb, r["cb"]) and np.array_equal(cr, r["cr"]), (t, s)


@pytest.mark.parametrize("cid", ["unaligned_161x99_odd", "unaligned_47x31", "cif_halfpel"])
def test_generic_kernel_fallback(monkeypatch, cid):
    """H263CU_KERNEL=mb: the warp-per-macroblock kernel stores RGBA cut to the picture."""
    monkeypatch.setenv("H263CU_KERNEL", "mb")
    case = BY_ID[cid]
    pk, opt = _packets(case)
    pk = pk[:4]
    ref = oracle_decode_stream(pk, opt)
    w, h = case["w"], case["h"]
    dec = api.BatchDecoder(1, w, h, decoder_options=opt, threads=1)
    view, flat, pitch, stride, pattern = guarded(1, w, h)
    for t in range(len(pk)):
        _, errs = dec.decode_step_device([pk[t]], out=view)
        assert not errs.any()
        check_guarded(flat, pitch, stride, w, h, [(0, w, h, ref[t]["rgba"])], pattern)
        pattern = flat.cpu().numpy().copy()
    assert dec.ctx.tiled_launch_count() == 0


@pytest.mark.parametrize("devices", [[0, 0, 0], "all"])
def test_device_group(devices):
    if devices == "all":
        if torch.cuda.device_count() < 2:
            pytest.skip("one GPU")
        devices = list(range(torch.cuda.device_count()))
    nd, per = len(devices), 2
    n, t_steps = nd * per, 3
    streams = [synth.make_stream(176, 144, t_steps, 660 + s, mv_mode=s % 3) for s in range(n)]
    refs = [oracle_decode_stream(s) for s in streams]
    g = api.DeviceGroup(devices, per, 176, 144, threads=4)
    for t in range(t_steps):
        outs, errs = g.decode_step_device([s[t] for s in streams])
        assert not errs.any() and len(outs) == nd
        for s in range(n):
            got = outs[s % nd][s // nd].cpu().numpy().reshape(-1)
            assert np.array_equal(got, refs[s][t]["rgba"]), (t, s)
    g.close()
