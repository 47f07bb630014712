"""h263cu_decode_step_device_motion on the GPU: the motion fields equal the oracle model (motion_ref.py) exactly, with
the host and the device parse, alone and beside every pixel output (whose bytes stay those of the call without
motion), through padded, gapped and permuted layouts; failed inputs, capacity and argument errors leave buffers and
parsers alone; the work is ordered on the caller's stream."""
import ctypes as C

import numpy as np
import pytest
import torch

import motion_ref as M
from h263_rs_b200 import _lib, api, frontend, synth

pytestmark = pytest.mark.gpu

PAT8, PAT16 = 0x5A, 0x5A5A


def fill(motion):
    for t in motion:
        if t is not None:
            t.fill_(PAT16 if t.dtype == torch.int16 else PAT8)


def host(motion):
    torch.cuda.synchronize()
    return [None if t is None else t.cpu().numpy() for t in motion]


def check_slot(got, k, ref, MBW, MBH, what=""):
    """slot k of the host copies `got` (mv, flags, quant) against the model of one picture"""
    e = M.slot(ref, MBW, MBH)
    mv, flags, quant = got
    if mv is not None:
        assert np.array_equal(mv[k], e["mv"]), (what, "mv")
    if flags is not None:
        assert np.array_equal(flags[k], e["flags"]), (what, "flags")
    if quant is not None:
        assert np.array_equal(quant[k], e["quant"]), (what, "quant")


def untouched(got, k):
    for a, p in zip(got, (PAT16, PAT8, PAT8)):
        if a is not None:
            assert (a[k] == p).all()


def mb_layer_failure(packet, options=1):
    """A copy of an I picture's packet damaged past its header so that the product's parser fails it inside the
    macroblock layer (the device parse then runs pack_mbs_kernel for the survivors of the step)"""
    rng = np.random.default_rng(7)
    for _ in range(400):
        pk = bytearray(packet)
        for _ in range(3):
            pos = int(rng.integers(len(pk) // 3, len(pk)))
            pk[pos] ^= 1 << int(rng.integers(0, 8))
        try:
            frontend.Parser(options).parse_picture(bytes(pk))
        except _lib.H263Error as e:
            if e.code in (-3, -4, -5, -6, -7, -8):
                return bytes(pk)
    raise AssertionError("no macroblock-layer failure found")


@pytest.mark.parametrize("parse", ["host", "device", "alternate"])
def test_motion_only_on_every_stream_case(parse):
    cases = M.CASES
    streams = [M.packets_of(c) for c in cases]
    refs = [M.reference_stream(pk, opt) for pk, opt in streams]
    dec = api.BatchDecoder(len(cases), 704, 576, threads=4)
    dec.parsers = [frontend.Parser(opt) for _, opt in streams]
    MBW, MBH = 44, 36
    motion = api.Motion(*[torch.empty(s, dtype=d, device="cuda") for s, d in
                          zip(api.motion_shapes(len(cases), 704, 576), (torch.int16, torch.uint8, torch.uint8))])
    for t in range(max(len(pk) for pk, _ in streams)):
        ids = [s for s in range(len(cases)) if t < len(streams[s][0])]
        fill(motion)
        p = parse if parse != "alternate" else ("host", "device")[t & 1]
        n0 = dec.ctx.launch_count()
        m, errs = dec.decode_step_device_motion([streams[s][0][t] for s in ids], motion=motion, stream_ids=ids, parse=p)
        assert m is motion
        got = host(motion)
        for k, s in enumerate(ids):
            r = refs[s][t]
            if isinstance(r, int):
                assert errs[k] != 0, (cases[s]["id"], t)
                untouched(got, k)
                continue
            assert errs[k] == 0, (cases[s]["id"], t, int(errs[k]))
            check_slot(got, k, r, MBW, MBH, (cases[s]["id"], t, p))
        # the step's reconstruction and the motion kernel
        assert dec.ctx.launch_count() - n0 == 2


@pytest.mark.parametrize("parse", ["host", "device"])
def test_mixed_sizes_into_padded_gapped_buffers_with_a_failed_input(parse):
    """QCIF, CIF, 161x99 and 15x15 in one call into every other slot of padded buffers: each decoded input's grid holds
    the model (the outside cells 0x80 / 0 / 0), and every other byte -- padding, gaps, the slot of the input that failed
    inside the macroblock layer -- keeps its pattern.  Stream 4 fails at step 0 and decodes one step late; at step 3 it
    is alone in the call, in slot 0 (slot = input index, whatever the stream id)."""
    sizes = [(176, 144), (352, 288), (161, 99), (15, 15), (176, 144)]
    n = len(sizes)
    streams = [synth.make_stream(w, h, 3, 300 + k, mv_mode=2, pct_fourmv=20, pct_intra=10) for k, (w, h) in enumerate(sizes)]
    refs = [M.reference_stream(pk) for pk in streams]
    bad = mb_layer_failure(streams[4][0])
    MBW, MBH = 22, 18
    base = [torch.empty((2 * n, 2, 2 * MBH + 3, 2 * MBW + 5), dtype=torch.int16, device="cuda"),
            torch.empty((2 * n, MBH + 2, MBW + 7), dtype=torch.uint8, device="cuda"),
            torch.empty((2 * n, MBH + 1, MBW + 3), dtype=torch.uint8, device="cuda")]
    motion = api.Motion(base[0][::2, :, : 2 * MBH, : 2 * MBW], base[1][::2, :MBH, :MBW], base[2][::2, :MBH, :MBW])
    dec = api.BatchDecoder(n, 352, 288, threads=4)
    for t in range(4):
        for b in base:
            b.fill_(PAT16 if b.dtype == torch.int16 else PAT8)
        inputs = [(s, t - (s == 4)) for s in range(n) if 0 <= t - (s == 4) < 3]
        if t == 0:
            inputs.append((4, None))
        ids = [s for s, _ in inputs]
        pk = [bad if i is None else streams[s][i] for s, i in inputs]
        _, errs = dec.decode_step_device_motion(pk, motion=motion, stream_ids=ids, parse=parse)
        got = host(motion)
        whole = [b.cpu().numpy() for b in base]
        want = [np.full(b.shape, PAT16, np.int16) if b.dtype == torch.int16 else np.full(b.shape, PAT8, np.uint8) for b in base]
        for k, (s, i) in enumerate(inputs):
            if i is None:
                assert errs[k] in (-3, -4, -5, -6, -7, -8), int(errs[k])
                continue
            assert errs[k] == 0, (t, s, int(errs[k]))
            check_slot(got, k, refs[s][i], MBW, MBH, (t, s))
            e = M.slot(refs[s][i], MBW, MBH)
            want[0][2 * k, :, : 2 * MBH, : 2 * MBW] = e["mv"]
            want[1][2 * k, :MBH, :MBW] = e["flags"]
            want[2][2 * k, :MBH, :MBW] = e["quant"]
        for a, b in zip(whole, want):
            assert np.array_equal(a, b), t  # nothing outside the decoded inputs' grids was written
        if t < 3:  # the 15x15 picture is one macroblock: every other cell of its slot is outside
            f = got[1][3]
            assert f[0, 0] != M.OUTSIDE and (f[1:, :] == M.OUTSIDE).all() and (f[:, 1:] == M.OUTSIDE).all()


def test_picture_larger_than_the_slot_is_a_capacity_error():
    pk = synth.make_stream(352, 288, 2, 41, mv_mode=1)
    ref = M.reference_stream(pk)
    dec = api.BatchDecoder(1, 352, 288, threads=1)
    small = api.Motion(None, torch.zeros((1, 9, 11), dtype=torch.uint8, device="cuda"), None)
    _, errs = dec.decode_step_device_motion([pk[0]], motion=small)
    assert errs[0] == _lib.ERR_CAPACITY
    torch.cuda.synchronize()
    assert (small.flags == 0).all()
    # the stream did not move: the I picture decodes now, then the P picture
    for t in range(2):
        m, errs = dec.decode_step_device_motion([pk[t]], motion=True)
        assert errs[0] == 0
        check_slot(host(m), 0, ref[t], 22, 18)
    # with a pixel output the smaller limit counts: an RGBA slot of QCIF refuses the CIF picture
    dec2 = api.BatchDecoder(1, 352, 288, threads=1)
    out = torch.empty((1, 144, 176, 4), dtype=torch.uint8, device="cuda")
    _, _, errs = dec2.decode_step_device([pk[0]], out=out, motion=True)
    assert errs[0] == _lib.ERR_CAPACITY


PIXELS = {
    "rgba": lambda d, pk, m, p: d.decode_step_device(pk, out_flags=_lib.OUT_RGBA | _lib.OUT_DEBLOCK, motion=m, parse=p),
    "i420": lambda d, pk, m, p: d.decode_step_device_yuv(pk, layout="i420", motion=m, parse=p),
    "tensor": lambda d, pk, m, p: d.decode_step_device_tensor(pk, (96, 128), dtype=torch.float16, mean=(0.5, 0.4, 0.3),
                                                              std=(0.2, 0.3, 0.4), motion=m, parse=p),
    "center_crop_aa": lambda d, pk, m, p: d.decode_step_device_tensor(pk, (112, 112), dtype=torch.float32, fit="center_crop",
                                                                      short_side=128, antialias=True, deblock=True, motion=m, parse=p),
}


def as_list(out):
    return [t.cpu().numpy().copy() for t in (out if isinstance(out, (tuple, list)) else [out])]


@pytest.mark.parametrize("kind", sorted(PIXELS))
@pytest.mark.parametrize("parse", ["host", "device"])
def test_pixel_outputs_beside_motion_are_unchanged(kind, parse):
    """Two decoders in lock step, one with motion and one without: the pixel bytes are equal, and the motion fields are
    the model's, with a failed input in the middle."""
    n = 6
    streams = [synth.make_stream(176, 144, 4, 500 + s, mv_mode=s % 3, pct_fourmv=15, pct_dquant=20) for s in range(n)]
    refs = [M.reference_stream(pk) for pk in streams]
    with_m = api.BatchDecoder(n, 176, 144, threads=4)
    without = api.BatchDecoder(n, 176, 144, threads=4)
    pos = [0] * n
    for t in range(5):
        ks = [k for k in range(n) if pos[k] < 4]
        pk = [streams[k][pos[k]] for k in ks]
        if t == 2:
            pk[1] = b"\x00\x00\x84\x00garbage"  # a failed input: its stream stays where it was
        out_m, motion, errs_m = PIXELS[kind](with_m, pk, True, parse) if len(ks) == n else (None, None, None)
        if out_m is None:
            break
        out_p, errs_p = PIXELS[kind](without, pk, None, parse)
        assert np.array_equal(errs_m, errs_p)
        got = host(motion)
        for a, b in zip(as_list(out_m), as_list(out_p)):
            for k in range(n):
                if errs_m[k] == 0:
                    assert a[k].tobytes() == b[k].tobytes(), (kind, t, k)
        for k in range(n):
            if errs_m[k] == 0:
                check_slot(got, k, refs[k][pos[k]], 11, 9, (kind, t, k))
                pos[k] += 1
            else:
                assert t == 2 and k == 1
    assert pos[0] == 4 and pos[1] == 3


def test_permuted_mv_and_flags_alone():
    pk = synth.make_stream(352, 288, 3, 61, mv_mode=2, pct_fourmv=30)
    ref = M.reference_stream(pk)
    dec = api.BatchDecoder(1, 352, 288, threads=1)
    nhwc = torch.full((1, 36, 44, 2), PAT16, dtype=torch.int16, device="cuda")
    for t in range(2):
        m, errs = dec.decode_step_device_motion([pk[t]], motion=api.Motion(nhwc.permute(0, 3, 1, 2), None, None))
        assert errs[0] == 0
        e = M.slot(ref[t], 22, 18)
        torch.cuda.synchronize()
        assert np.array_equal(nhwc.cpu().numpy()[0], e["mv"].transpose(1, 2, 0))
    # only the flags: the mv memory beside it is not touched
    flags = torch.full((1, 18, 22), PAT8, dtype=torch.uint8, device="cuda")
    m, errs = dec.decode_step_device_motion([pk[2]], motion=api.Motion(None, flags, None))
    assert errs[0] == 0 and m.mv is None and m.quant is None
    got = host(m)
    check_slot(got, 0, ref[2], 22, 18)
    assert np.array_equal(nhwc.cpu().numpy()[0], M.slot(ref[1], 22, 18)["mv"].transpose(1, 2, 0))


def test_argument_errors_are_refused_before_any_parser_moves():
    pk = synth.make_stream(176, 144, 2, 71)
    dec = api.BatchDecoder(1, 176, 144, threads=1)
    L = _lib.lib()
    motion, good = api._device_motion(True, 1, 176, 144, 0)
    plan = dec.plan_step([pk[0]])

    def call(m, pixels=None, c=None):
        nd = C.c_uint32(0)
        return L.h263cu_decode_step_device_motion(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data,
                                                  1, 1, 0, None if m is None else C.byref(m), None if pixels is None else C.byref(pixels),
                                                  plan["errs"].ctypes.data, C.byref(nd))

    def edited(**kw):
        m = _lib.DeviceMotion.from_buffer_copy(good)
        for k, v in kw.items():
            if isinstance(v, tuple):
                getattr(m, k[:-2])[int(k[-1])] = v[0]
            else:
                setattr(m, k, v)
        return m

    host_mem = np.zeros(4096, np.uint8)
    bad = [None, edited(mv=None, mb_flags=None, mb_quant=None), edited(mb_width=0), edited(mb_height=256), edited(mb_width=256),
           edited(mv_stride_2=(0,)), edited(flags_stride_1=(-1,)), edited(quant_stride_0=(0,)), edited(mv=good.mv + 1),
           edited(mv_stride_3=(1 << 40,)), edited(flags_stride_0=(1 << 41,), flags_stride_1=(1 << 39,)),
           edited(mb_quant=host_mem.ctypes.data)]
    for m in bad:
        assert call(m) == _lib.ERR_BAD_ARGUMENT
    out = torch.empty((1, 144, 176, 4), dtype=torch.uint8, device="cuda")
    _, rgba = api._device_rgba(out, 1, 176, 144, 0)
    _, ten = api._device_tensor(None, 1, (8, 8), torch.float16, None, None, 0)
    fit = api._tensor_fit("stretch", None, 0, None, 1, always=True)
    bad_pixels = [api._device_output(rgba=rgba, tensor=ten), api._device_output(rgba=rgba, fit=fit),
                  api._device_output(tensor=ten, filt=1), api._device_output(tensor=ten, fit=fit, filt=3),
                  api._device_output(rgba=_lib.DeviceRgba(out.data_ptr() + 1, 704, 704 * 144, 176, 144, None))]
    o = api._device_output(tensor=ten)
    o.reserved = 1
    bad_pixels.append(o)
    for px in bad_pixels:
        assert call(good, px) == _lib.ERR_BAD_ARGUMENT
    # the parser has not moved: a P picture still finds no reference
    _, errs = dec.decode_step_device_motion([pk[1]], motion=motion)
    assert errs[0] == -15
    _, errs = dec.decode_step_device_motion([pk[0]], motion=motion)
    assert errs[0] == 0
    with pytest.raises(ValueError):
        api._device_motion(api.Motion(None, None, None), 1, 176, 144, 0)
    with pytest.raises(ValueError):  # the fields disagree on the grid
        api._device_motion(api.Motion(motion.mv, motion.flags[:, :8], None), 1, 176, 144, 0)


def test_ordering_on_a_side_stream_without_host_syncs():
    n, steps = 8, 5
    streams = [synth.make_stream(176, 144, steps, 900 + s, mv_mode=2) for s in range(n)]
    refs = [M.reference_stream(pk) for pk in streams]
    dec = api.BatchDecoder(n, 176, 144, threads=4)
    side = torch.cuda.Stream()
    motion = api.Motion(*[torch.empty(s, dtype=d, device="cuda") for s, d in
                          zip(api.motion_shapes(n, 176, 144), (torch.int16, torch.uint8, torch.uint8))])
    copies = []
    with torch.cuda.stream(side):
        for t in range(steps):
            fill(motion)  # queued before the call: the library's writes wait for it
            torch.cuda._sleep(2_000_000)
            _, errs = dec.decode_step_device_motion([pk[t] for pk in streams], motion=motion, parse=("host", "device")[t & 1])
            assert (errs == 0).all()
            copies.append([x.clone() for x in motion])  # queued after the call: sees the fields
    torch.cuda.synchronize()
    for t in range(steps):
        got = [x.cpu().numpy() for x in copies[t]]
        for k in range(n):
            check_slot(got, k, refs[k][t], 11, 9, (t, k))


def test_group_form_on_contexts_of_one_device():
    n_ctx, per, steps = 3, 4, 3
    n = n_ctx * per
    streams = [synth.make_stream(176, 144, steps, 800 + s, mv_mode=s % 3) for s in range(n)]
    refs = [M.reference_stream(pk) for pk in streams]
    grp = api.DeviceGroup([0] * n_ctx, per, 176, 144, threads=3)
    for t in range(steps):
        ids = [s for s in range(n) if not (s == 5 and t == 1)]  # stream 5 sits step 1 out
        idx = {s: t - (1 if (s == 5 and t > 1) else 0) for s in ids}
        pk = [streams[s][idx[s]] for s in ids]
        if t == 0:
            motions, errs = grp.decode_step_device_motion(pk, stream_ids=ids)
        else:
            _, motions, errs = grp.decode_step_device_tensor(pk, (64, 64), stream_ids=ids, fit="center_crop", short_side=64,
                                                             motion=True, parse=("host", "device")[t & 1])
        assert (errs == 0).all()
        got = [host(m) for m in motions]
        for s in ids:
            d, local = s % n_ctx, s // n_ctx  # device-major: global stream s in slot s // n of device s % n
            check_slot(got[d], local, refs[s][idx[s]], 11, 9, (t, s))
    grp.close()
