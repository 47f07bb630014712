"""h263cu_decode_step_device_residual on the GPU: the residual planes equal the oracle model (residual_ref.py) exactly,
with the host and the device parse, under both recon kernels, alone and beside every pixel output and the motion fields
(whose bytes stay those of the call without residual), through padded, gapped, sliced and permuted layouts; failed
inputs, capacity and argument errors leave buffers and parsers alone; the work is ordered on the caller's stream."""
import ctypes as C

import numpy as np
import pytest
import torch

import motion_ref as M
import residual_ref as RR
from h263_rs_b200 import _lib, api, synth
from test_gpu_device_motion import mb_layer_failure

pytestmark = pytest.mark.gpu

PAT = 0x5A5A
PLANES = ("y", "cb", "cr")

_MODELS = {}


def model(key, packets, options=1):
    if key not in _MODELS:
        _MODELS[key] = RR.reference_stream(packets, options)
    return _MODELS[key]


def host(res):
    torch.cuda.synchronize()
    return [None if t is None else t.cpu().numpy() for t in res]


def check_slot(got, k, ref, W, H, what=""):
    e = RR.slot(ref, W, H)
    for name, a in zip(PLANES, got):
        if a is not None:
            assert np.array_equal(a[k], e[name]), (what, name, np.argwhere(a[k] != e[name])[:5])


def fill(res):
    for t in res:
        if t is not None:
            t.fill_(PAT)


@pytest.mark.parametrize("kernel", ["default", "mb"])
@pytest.mark.parametrize("parse", ["host", "device", "alternate"])
def test_residual_only_on_every_stream_case(monkeypatch, parse, kernel):
    if kernel == "mb":  # the warp-per-macroblock recon kernel: references without a replicated border
        monkeypatch.setenv("H263CU_KERNEL", "mb")
    cases = M.CASES
    streams = [M.packets_of(c) for c in cases]
    refs = [model(c["id"], pk, opt) for c, (pk, opt) in zip(cases, streams)]
    dec = api.BatchDecoder(len(cases), 704, 576, threads=4)
    dec.parsers = [api.frontend.Parser(opt) for _, opt in streams]
    res = api.Residual(*[torch.empty(s, dtype=torch.int16, device="cuda") for s in api.residual_shapes(len(cases), 704, 576)])
    for t in range(max(len(pk) for pk, _ in streams)):
        ids = [s for s in range(len(cases)) if t < len(streams[s][0])]
        fill(res)
        p = parse if parse != "alternate" else ("host", "device")[t & 1]
        n0 = dec.ctx.launch_count()
        r, errs = dec.decode_step_device_residual([streams[s][0][t] for s in ids], residual=res, stream_ids=ids, parse=p)
        assert r is res
        got = host(res)
        for k, s in enumerate(ids):
            ref = refs[s][t]
            if isinstance(ref, int):
                assert errs[k] != 0, (cases[s]["id"], t)
                assert all((a[k] == PAT).all() for a in got)
                continue
            assert errs[k] == 0, (cases[s]["id"], t, int(errs[k]))
            check_slot(got, k, ref, 704, 576, (cases[s]["id"], t, p, kernel))
        assert dec.ctx.launch_count() - n0 == 2  # the step's reconstruction and the residual kernel


@pytest.mark.parametrize("parse", ["host", "device"])
def test_mixed_sizes_into_padded_gapped_views_with_a_failed_input(parse):
    """QCIF, CIF, 161x99 and 15x15 in one call into every other slot of padded planes: each decoded input's slot holds
    the model (zeros beyond its picture), and every other element -- padding, gaps, the slot of the input that failed
    inside the macroblock layer -- keeps its guard value."""
    sizes = [(176, 144), (352, 288), (161, 99), (15, 15), (176, 144)]
    n = len(sizes)
    streams = [synth.make_stream(w, h, 3, 300 + k, mv_mode=2, pct_fourmv=20, pct_intra=10) for k, (w, h) in enumerate(sizes)]
    refs = [model(("mixed", k), pk) for k, pk in enumerate(streams)]
    bad = mb_layer_failure(streams[4][0])
    W, H = 352, 288
    base = [torch.empty((2 * n, H + 3, W + 7), dtype=torch.int16, device="cuda"),
            torch.empty((2 * n, H // 2 + 1, W // 2 + 5), dtype=torch.int16, device="cuda"),
            torch.empty((2 * n, H // 2 + 2, W // 2 + 3), dtype=torch.int16, device="cuda")]
    res = api.Residual(base[0][::2, :H, :W], base[1][::2, : H // 2, : W // 2], base[2][::2, : H // 2, : W // 2])
    dec = api.BatchDecoder(n, 352, 288, threads=4)
    for t in range(4):
        for b in base:
            b.fill_(PAT)
        inputs = [(s, t - (s == 4)) for s in range(n) if 0 <= t - (s == 4) < 3]
        if t == 0:
            inputs.append((4, None))
        ids = [s for s, _ in inputs]
        pk = [bad if i is None else streams[s][i] for s, i in inputs]
        _, errs = dec.decode_step_device_residual(pk, residual=res, stream_ids=ids, parse=parse)
        whole = [b.cpu().numpy() for b in base]
        want = [np.full(b.shape, PAT, np.int16) for b in base]
        for k, (s, i) in enumerate(inputs):
            if i is None:
                assert errs[k] in (-3, -4, -5, -6, -7, -8), int(errs[k])
                continue
            assert errs[k] == 0, (t, s, int(errs[k]))
            e = RR.slot(refs[s][i], W, H)
            want[0][2 * k, :H, :W], want[1][2 * k, : H // 2, : W // 2], want[2][2 * k, : H // 2, : W // 2] = e["y"], e["cb"], e["cr"]
        for a, b, name in zip(whole, want, PLANES):
            assert np.array_equal(a, b), (t, name)


def test_picture_larger_than_the_slot_is_a_capacity_error():
    pk = synth.make_stream(352, 288, 2, 41, mv_mode=1)
    ref = model("capacity", pk)
    dec = api.BatchDecoder(1, 352, 288, threads=1)
    small = api.Residual(torch.zeros((1, 287, 352), dtype=torch.int16, device="cuda"), None, None)
    _, errs = dec.decode_step_device_residual([pk[0]], residual=small)
    assert errs[0] == _lib.ERR_CAPACITY
    torch.cuda.synchronize()
    assert (small.y == 0).all()
    for t in range(2):  # the stream did not move: the I picture decodes now, then the P picture
        r, errs = dec.decode_step_device_residual([pk[t]], residual=True)
        assert errs[0] == 0
        check_slot(host(r), 0, ref[t], 352, 288)
    # beside motion and pixels the smallest limit counts
    dec2 = api.BatchDecoder(1, 352, 288, threads=1)
    _, _, errs = dec2.decode_step_device_residual([pk[0]], residual=True, motion=api.Motion(None, torch.zeros((1, 9, 11), dtype=torch.uint8,
                                                                                                          device="cuda"), None))
    assert errs[0] == _lib.ERR_CAPACITY
    out = torch.empty((1, 144, 176, 4), dtype=torch.uint8, device="cuda")
    _, _, errs = dec2.decode_step_device([pk[0]], out=out, residual=True)
    assert errs[0] == _lib.ERR_CAPACITY


PIXELS = {
    "rgba": lambda d, pk, **kw: d.decode_step_device(pk, out_flags=_lib.OUT_RGBA, **kw),
    "rgba_deblock": lambda d, pk, **kw: d.decode_step_device(pk, out_flags=_lib.OUT_RGBA | _lib.OUT_DEBLOCK, **kw),
    "i420": lambda d, pk, **kw: d.decode_step_device_yuv(pk, layout="i420", **kw),
    "nv12_deblock": lambda d, pk, **kw: d.decode_step_device_yuv(pk, layout="nv12", deblock=True, **kw),
    "tensor": lambda d, pk, **kw: d.decode_step_device_tensor(pk, (96, 128), dtype=torch.float16, mean=(0.5, 0.4, 0.3),
                                                              std=(0.2, 0.3, 0.4), **kw),
    "tensor_fit": lambda d, pk, **kw: d.decode_step_device_tensor(pk, (80, 80), dtype=torch.uint8, fit="letterbox", fill=7, **kw),
    "tensor_filter": lambda d, pk, **kw: d.decode_step_device_tensor(pk, (112, 112), dtype=torch.float32, fit="center_crop",
                                                                     short_side=128, antialias=True, deblock=True, **kw),
}


def as_list(out):
    return [t.cpu().numpy().copy() for t in (out if isinstance(out, (tuple, list)) else [out])]


@pytest.mark.parametrize("with_motion", [False, True])
@pytest.mark.parametrize("kind", sorted(PIXELS))
def test_pixel_outputs_and_motion_beside_the_residual_are_unchanged(kind, with_motion):
    """Two decoders in lock step, one with the residual and one without: the pixel bytes and the motion fields are
    equal, and the residual is the model's (deblocking does not touch it), with a failed input in the middle."""
    n = 6
    streams = [synth.make_stream(176, 144, 4, 500 + s, mv_mode=s % 3, pct_fourmv=15, pct_dquant=20) for s in range(n)]
    refs = [model(("pixels", s), pk) for s, pk in enumerate(streams)]
    with_r = api.BatchDecoder(n, 176, 144, threads=4)
    without = api.BatchDecoder(n, 176, 144, threads=4)
    pos = [0] * n
    for t in range(5):
        ks = [k for k in range(n) if pos[k] < 4]
        if len(ks) < n:
            break
        pk = [streams[k][pos[k]] for k in ks]
        if t == 2:
            pk[1] = b"\x00\x00\x84\x00garbage"  # a failed input: its stream stays where it was
        parse = ("host", "device")[t & 1]
        m = True if with_motion else None
        got_r = PIXELS[kind](with_r, pk, motion=m, residual=True, parse=parse)
        got_p = PIXELS[kind](without, pk, motion=m, parse=parse)
        errs_r, errs_p = got_r[-1], got_p[-1]
        assert np.array_equal(errs_r, errs_p)
        assert len(got_r) == len(got_p) + 1
        res = host(got_r[-2])
        for a_out, b_out in zip(got_r[:-2], got_p[:-1]):  # the pixel output, then the motion fields
            for a, b in zip(as_list(a_out), as_list(b_out)):
                for k in range(n):
                    if errs_r[k] == 0:
                        assert a[k].tobytes() == b[k].tobytes(), (kind, t, k)
        for k in range(n):
            if errs_r[k] == 0:
                check_slot(res, k, refs[k][pos[k]], 176, 144, (kind, t, k))
                pos[k] += 1
            else:
                assert t == 2 and k == 1
    assert pos[0] == 4 and pos[1] == 3


def test_strided_views_sliced_permuted_and_luma_only():
    pk = synth.make_stream(352, 288, 3, 61, mv_mode=2, pct_fourmv=30)
    ref = model("strided", pk)
    dec = api.BatchDecoder(1, 352, 288, threads=1)
    # y as a permuted [W, H] buffer, cb as a column-sliced view (column stride 3), cr a row-sliced view
    yt = torch.full((1, 352, 288), PAT, dtype=torch.int16, device="cuda")
    cbb = torch.full((1, 144, 3 * 176), PAT, dtype=torch.int16, device="cuda")
    crb = torch.full((1, 2 * 144, 176), PAT, dtype=torch.int16, device="cuda")
    view = api.Residual(yt.permute(0, 2, 1), cbb[:, :, ::3], crb[:, ::2, :])
    for t in range(2):
        _, errs = dec.decode_step_device_residual([pk[t]], residual=view, parse=("host", "device")[t])
        assert errs[0] == 0
        check_slot(host(view), 0, ref[t], 352, 288, t)
        torch.cuda.synchronize()
        assert (cbb[:, :, 1::3] == PAT).all() and (cbb[:, :, 2::3] == PAT).all() and (crb[:, 1::2, :] == PAT).all()
    # Y alone: the chroma memory keeps the previous picture's values
    y = torch.full((1, 288, 352), PAT, dtype=torch.int16, device="cuda")
    r, errs = dec.decode_step_device_residual([pk[2]], residual=api.Residual(y, None, None))
    assert errs[0] == 0 and r.cb is None and r.cr is None
    check_slot(host(r), 0, ref[2], 352, 288)
    got, e = host(view), RR.slot(ref[1], 352, 288)
    assert np.array_equal(got[1][0], e["cb"]) and np.array_equal(got[2][0], e["cr"])


def test_argument_errors_are_refused_before_any_parser_moves():
    pk = synth.make_stream(176, 144, 2, 71)
    dec = api.BatchDecoder(1, 176, 144, threads=1)
    L = _lib.lib()
    res, good = api._device_residual(True, 1, 176, 144, 0)
    _, motion = api._device_motion(True, 1, 176, 144, 0)
    plan = dec.plan_step([pk[0]])

    def call(r, m=None, pixels=None):
        nd = C.c_uint32(0)
        return L.h263cu_decode_step_device_residual(dec.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data,
                                                    1, 1, 0, None if r is None else C.byref(r), None if m is None else C.byref(m),
                                                    None if pixels is None else C.byref(pixels), plan["errs"].ctypes.data, C.byref(nd))

    def edited(src=good, **kw):
        r = type(src).from_buffer_copy(src)
        for k, v in kw.items():
            if isinstance(v, tuple):
                getattr(r, k[:-2])[int(k[-1])] = v[0]
            else:
                setattr(r, k, v)
        return r

    host_mem = np.zeros(4096, np.uint8)
    bad = [None, edited(y=None, cb=None, cr=None), edited(width=0), edited(height=0), edited(width=16385), edited(height=16385),
           edited(y_stride_2=(0,)), edited(cb_stride_1=(-1,)), edited(cr_stride_0=(0,)), edited(y=good.y + 1),
           edited(cb_stride_2=(1 << 40,)), edited(y_stride_1=(1 << 33,)), edited(cr=host_mem.ctypes.data)]
    for r in bad:
        assert call(r) == _lib.ERR_BAD_ARGUMENT
    assert call(good, edited(motion, mb_width=0)) == _lib.ERR_BAD_ARGUMENT
    _, ten = api._device_tensor(None, 1, (8, 8), torch.float16, None, None, 0)
    o = api._device_output(tensor=ten, filt=1)
    assert call(good, None, o) == _lib.ERR_BAD_ARGUMENT
    # the parser has not moved: a P picture still finds no reference
    _, errs = dec.decode_step_device_residual([pk[1]], residual=res)
    assert errs[0] == -15
    _, errs = dec.decode_step_device_residual([pk[0]], residual=res)
    assert errs[0] == 0
    for bad_py in (api.Residual(None, None, None), api.Residual(res.y, res.cb[:, :70], None),
                   api.Residual(res.y.float(), None, None), api.Residual(res.y[:, :, :0], None, None)):
        with pytest.raises(ValueError):
            api._device_residual(bad_py, 1, 176, 144, 0)


def test_ordering_on_a_side_stream_without_host_syncs():
    n, steps = 8, 5
    streams = [synth.make_stream(176, 144, steps, 900 + s, mv_mode=2) for s in range(n)]
    refs = [model(("order", s), pk) for s, pk in enumerate(streams)]
    dec = api.BatchDecoder(n, 176, 144, threads=4)
    side = torch.cuda.Stream()
    res = api.Residual(*[torch.empty(s, dtype=torch.int16, device="cuda") for s in api.residual_shapes(n, 176, 144)])
    copies = []
    with torch.cuda.stream(side):
        for t in range(steps):
            fill(res)  # queued before the call: the library's writes wait for it
            torch.cuda._sleep(2_000_000)
            _, errs = dec.decode_step_device_residual([pk[t] for pk in streams], residual=res, parse=("host", "device")[t & 1])
            assert (errs == 0).all()
            copies.append([x.clone() for x in res])  # queued after the call: sees the residual
    torch.cuda.synchronize()
    for t in range(steps):
        got = [x.cpu().numpy() for x in copies[t]]
        for k in range(n):
            check_slot(got, k, refs[k][t], 176, 144, (t, k))


def test_group_form_on_contexts_of_one_device():
    n_ctx, per, steps = 3, 4, 3
    n = n_ctx * per
    streams = [synth.make_stream(176, 144, steps, 800 + s, mv_mode=s % 3) for s in range(n)]
    refs = [model(("group", s), pk) for s, pk in enumerate(streams)]
    mrefs = [M.reference_stream(pk) for pk in streams]
    grp = api.DeviceGroup([0] * n_ctx, per, 176, 144, threads=3)
    for t in range(steps):
        ids = [s for s in range(n) if not (s == 5 and t == 1)]  # stream 5 sits step 1 out
        idx = {s: t - (1 if (s == 5 and t > 1) else 0) for s in ids}
        pk = [streams[s][idx[s]] for s in ids]
        motions = None
        if t == 0:
            residuals, errs = grp.decode_step_device_residual(pk, stream_ids=ids)
        elif t == 1:
            motions, residuals, errs = grp.decode_step_device_residual(pk, motions=True, stream_ids=ids, parse="device")
        else:
            _, residuals, errs = grp.decode_step_device_tensor(pk, (64, 64), stream_ids=ids, fit="center_crop", short_side=64,
                                                               residual=True)
        assert (errs == 0).all()
        got = [host(r) for r in residuals]
        gm = None if motions is None else [host(m) for m in motions]
        for s in ids:
            d, local = s % n_ctx, s // n_ctx
            check_slot(got[d], local, refs[s][idx[s]], 176, 144, (t, s))
            if gm is not None:
                assert np.array_equal(gm[d][0][local], M.slot(mrefs[s][idx[s]], 11, 9)["mv"])
    grp.close()
