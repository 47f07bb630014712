"""GPU parity: the CUDA path, called through the C ABI, against the oracle -- bit exact
Y/Cb/Cr planes and bit exact RGBA on the same seeded bitstreams, plus the reference's own
known-answer vectors for the colour conversion and the deblocking filter."""
import json
import os

import numpy as np
import pytest

import oracle_lib as O
from helpers import oracle_decode_stream, recon_from_side_info, weighted_sum
from h263_rs_b200 import _lib, api, frontend, synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    with open(os.path.join(G, name)) as f:
        return json.load(f)


# ------------------------------------------------------------------ yuv::bt601 (K4)
def test_yuv420_to_rgba_reference_kats():
    k = load("kat_yuv.json")
    for v in k["yuv_to_rgb"]:
        y, cb, cr = v["yuv"]
        assert list(api.yuv420_to_rgba([y], [cb], [cr], 1)) == v["rgb"] + [255]
    for p in k["yuv420_to_rgba"]:
        assert list(api.yuv420_to_rgba(p["y"], p["cb"], p["cr"], p["width"])) == p["rgba"], p["width"]


@pytest.mark.parametrize("w,h", [(1, 1), (2, 2), (3, 5), (5, 4), (7, 3), (16, 16), (33, 17), (176, 144), (352, 288), (355, 291)])
def test_yuv420_to_rgba_random_planes(w, h):
    rng = np.random.default_rng(w * 1000 + h)
    cw, ch = (w + 1) // 2, (h + 1) // 2
    y = rng.integers(0, 256, w * h).astype(np.uint8)
    cb = rng.integers(0, 256, cw * ch).astype(np.uint8)
    cr = rng.integers(0, 256, cw * ch).astype(np.uint8)
    assert np.array_equal(api.yuv420_to_rgba(y, cb, cr, w), O.yuv420_to_rgba(y, cb, cr, w))


# ------------------------------------------------------------------ deblock (K3)
def test_deblock_reference_kats():
    p = load("kat_deblock.json")["picture"]
    for c in p["cases"]:
        assert list(api.deblock(p["data"], p["width"], c["strength"])) == c["expected"], c["strength"]
    assert list(api.QUANT_TO_STRENGTH) == load("kat_constants.json")["quant_to_strength"]


@pytest.mark.parametrize("w,h", [(8, 8), (9, 17), (10, 10), (11, 17), (16, 16), (17, 9), (31, 33), (40, 24), (88, 72),
                                 (176, 144), (352, 288), (357, 293)])
def test_deblock_random_planes_including_scalar_tails(w, h):
    rng = np.random.default_rng(w * 977 + h)
    smooth = rng.integers(0, 256, (h // 8 + 1, w // 8 + 1)).astype(np.int32)
    base = np.kron(smooth, np.ones((8, 8), np.int32))[:h, :w]
    for amp in (3, 40):
        data = np.clip(base + rng.integers(-amp, amp + 1, (h, w)), 0, 255).astype(np.uint8).reshape(-1)
        for strength in (1, 4, 9, 12):
            assert np.array_equal(api.deblock(data, w, strength), O.deblock(data, w, strength)), (amp, strength)


# ------------------------------------------------------------------ fused recon (K1+K2+K4)
STREAMS = [
    # BASELINE.json config 1: single QCIF stream, 1 I + 29 P, decoded to RGBA
    dict(id="config1_qcif", w=176, h=144, n=30, seed=1),
    dict(id="cif_halfpel", w=352, h=288, n=8, seed=2, mv_mode=1),
    dict(id="cif_borders_escapes", w=352, h=288, n=6, seed=3, mv_mode=2, pct_escape=20, permille_overflow=30,
         truncate_permille=300),
    dict(id="cif_v0_escapes", w=352, h=288, n=4, seed=4, version=0, pct_escape=30),
    dict(id="qcif_baseline_h263", w=176, h=144, n=6, seed=5, flavour=1, pct_escape=10),
    dict(id="160x120_4mv_dquant", w=160, h=120, n=8, seed=6, pct_fourmv=30, pct_dquant=40, mv_mode=1),
    dict(id="200x100_unaligned", w=200, h=100, n=6, seed=7, intra_period=3, mv_mode=2),
    dict(id="4cif", w=704, h=576, n=3, seed=8, mv_mode=2),
    dict(id="sqcif_many_events", w=128, h=96, n=4, seed=9, mean_events_x10=200, pct_cbp_inter=90),
    dict(id="tiny_24x40", w=24, h=40, n=5, seed=10, mv_mode=1),
    dict(id="qcif_all_intra_dense", w=176, h=144, n=3, seed=11, intra_period=1, pct_cbp_intra=100, mean_events_x10=120),
    # sizes that are not multiples of 16 (the tiled kernel's edge fix-up): odd sizes, a single partial macroblock,
    # partial columns / rows of 1 and 15 pixels, vectors pointing across the partial edge
    dict(id="unaligned_161x99_odd", w=161, h=99, n=6, seed=12, mv_mode=2, pct_fourmv=20),
    dict(id="unaligned_15x15", w=15, h=15, n=5, seed=13, mv_mode=1),
    dict(id="unaligned_17x33", w=17, h=33, n=5, seed=14, mv_mode=2),
    dict(id="unaligned_480x360", w=480, h=360, n=4, seed=15, mv_mode=2, intra_period=3),
    dict(id="unaligned_47x31", w=47, h=31, n=6, seed=16, mv_mode=1, pct_intra=30),
]


def _packets(c):
    kw = {k: v for k, v in c.items() if k not in ("id", "w", "h", "n", "seed")}
    return synth.make_stream(c["w"], c["h"], c["n"], c["seed"], **kw), (0 if kw.get("flavour", 0) == 1 else 1)


# small MB-aligned sizes: the register-resident deblock kernel's border cells, chroma planes too narrow
# for a vertical edge (width 8 < 10, deblock.rs:228), single-row / single-column macroblock grids, and
# every quantiser (= every filter strength of QUANT_TO_STRENGTH)
SMALL_ALIGNED = [
    dict(id="16x16", w=16, h=16, n=4, seed=21, mv_mode=1),
    dict(id="32x16", w=32, h=16, n=4, seed=22, mv_mode=2),
    dict(id="16x48", w=16, h=48, n=4, seed=23, mv_mode=1),
    dict(id="48x32_q31", w=48, h=32, n=5, seed=24, mv_mode=2, qp_min=24, qp_max=31),
    dict(id="64x64_q1", w=64, h=64, n=5, seed=25, mv_mode=1, qp_min=1, qp_max=3, pct_dquant=50),
    dict(id="96x80_dense", w=96, h=80, n=4, seed=26, mean_events_x10=150, pct_cbp_inter=95, pct_cbp_intra=100, pct_intra=40),
]


@pytest.mark.parametrize("case", STREAMS + SMALL_ALIGNED, ids=lambda c: c["id"])
def test_decode_next_picture_bit_exact(case):
    packets, opt = _packets(case)
    ref = oracle_decode_stream(packets, opt)
    st = api.H263State(opt)
    for i, pk in enumerate(packets):
        if isinstance(ref[i], int):
            with pytest.raises(_lib.H263Error):
                st.decode_next_picture(pk)
            continue
        st.decode_next_picture(pk)
        pic = st.get_last_picture()
        y, cb, cr = pic.as_yuv()
        assert (pic.width, pic.height) == (ref[i]["info"]["width"], ref[i]["info"]["height"])
        assert np.array_equal(y, ref[i]["y"]), (case["id"], i, "Y")
        assert np.array_equal(cb, ref[i]["cb"]), (case["id"], i, "Cb")
        assert np.array_equal(cr, ref[i]["cr"]), (case["id"], i, "Cr")
        assert np.array_equal(st.get_last_rgba(), ref[i]["rgba"]), (case["id"], i, "RGBA")
    # every picture took the tiled kernel, whatever its size (the generic kernel is only the A/B partner)
    if st.ctx is not None:
        assert st.ctx.tiled_launch_count() == sum(1 for r in ref if not isinstance(r, int)), case["id"]


@pytest.mark.parametrize("case", [STREAMS[0], STREAMS[2], STREAMS[6], STREAMS[7]] + SMALL_ALIGNED, ids=lambda c: c["id"])
def test_deblocked_rgba_bit_exact(case):
    """recon -> deblock(plane, width, QUANT_TO_STRENGTH[pquant]) per plane -> RGBA; the
    reference frames stay un-deblocked (BASELINE.json config 4 composition)."""
    packets, opt = _packets(dict(case, deblock_flag=1))
    ref = oracle_decode_stream(packets, opt, deblock=True)
    st = api.H263State(opt, deblock=True)
    for i, pk in enumerate(packets):
        if isinstance(ref[i], int):
            with pytest.raises(_lib.H263Error):
                st.decode_next_picture(pk)
            continue
        st.decode_next_picture(pk)
        y, cb, cr = st.get_last_picture().as_yuv()
        assert np.array_equal(y, ref[i]["y"]) and np.array_equal(cb, ref[i]["cb"]) and np.array_equal(cr, ref[i]["cr"])
        assert np.array_equal(st.get_last_rgba(), ref[i]["rgba"]), (case["id"], i)


def test_batch_decoder_many_streams_and_device_checksums():
    """16 independent CIF streams decoded in lock step; per-stream planes, RGBA and the
    on-device checksums all match the oracle (the form configs 3-5 use at full size)."""
    n, t_steps = 16, 5
    streams = [synth.make_stream(352, 288, t_steps, 1000 + s, mv_mode=s % 3, pct_fourmv=5 + s) for s in range(n)]
    refs = [oracle_decode_stream(p) for p in streams]
    dec = api.BatchDecoder(n, 352, 288, threads=4)
    for t in range(t_steps):
        errs = dec.decode_step([streams[s][t] for s in range(n)])
        assert not errs.any()
        dec.ctx.sync()
        sums = dec.ctx.checksums(np.arange(n))
        for s in range(n):
            r = refs[s][t]
            assert [int(v) for v in sums[s]] == [weighted_sum(r["y"]), weighted_sum(r["cb"]), weighted_sum(r["cr"]),
                                                 weighted_sum(r["rgba"])], (s, t)
        for s in (0, 7, 15):
            y, cb, cr = dec.ctx.read_yuv(s)
            assert np.array_equal(y, refs[s][t]["y"]) and np.array_equal(cb, refs[s][t]["cb"])
            assert np.array_equal(cr, refs[s][t]["cr"])
            assert np.array_equal(dec.ctx.read_rgba(s), refs[s][t]["rgba"])


def test_resident_steps_replay_and_mixed_sizes():
    """Side info resident in device memory (step_upload/step_run), streams of different
    picture sizes in one step, and a stream that sits out a step."""
    dims = [(176, 144), (352, 288), (160, 120), (128, 96)]
    t_steps = 4
    streams = [synth.make_stream(w, h, t_steps, 50 + i, mv_mode=1) for i, (w, h) in enumerate(dims)]
    refs = [oracle_decode_stream(p) for p in streams]
    ctx = api.Context(0, len(dims), 352, 288)
    parsers = [frontend.Parser(1) for _ in dims]
    decoded = [0] * len(dims)
    for t in range(t_steps + 1):
        active = [s for s in range(len(dims)) if not (s == 2 and t == 1) and decoded[s] < t_steps]
        if not active:
            break
        pics, mbs, events, errs, _ = frontend.parse_step([parsers[s] for s in active],
                                                         [streams[s][decoded[s]] for s in active], active, 2)
        assert not errs.any()
        step = ctx.step_upload(pics, mbs, events)
        ctx.step_run(step, _lib.OUT_RGBA)
        ctx.sync()
        ctx.step_free(step)
        for s in active:
            r = refs[s][decoded[s]]
            y, cb, cr = ctx.read_yuv(s)
            assert np.array_equal(y, r["y"]) and np.array_equal(cb, r["cb"]) and np.array_equal(cr, r["cr"]), (s, t)
            assert np.array_equal(ctx.read_rgba(s), r["rgba"]), (s, t)
            decoded[s] += 1


def test_readback_pipeline_matches():
    """submit_step_readback: RGBA of every step copied back asynchronously (the e2e path)."""
    import ctypes as C

    n, t_steps = 6, 4
    streams = [synth.make_stream(176, 144, t_steps, 300 + s) for s in range(n)]
    refs = [oracle_decode_stream(p) for p in streams]
    dec = api.BatchDecoder(n, 176, 144, threads=2)
    L = _lib.lib()
    size = 176 * 144 * 4
    bufs = []
    for t in range(t_steps):
        pics, mbs, events, errs, _ = dec.parse_step([streams[s][t] for s in range(n)])
        host = L.h263cu_alloc_pinned(n * size)
        assert host
        bufs.append(host)
        _lib.check(L.h263cu_submit_step_readback(dec.ctx.h, pics.ctypes.data, len(pics), mbs.ctypes.data, len(mbs),
                                                 events.ctypes.data, len(events), _lib.OUT_RGBA, host, None))
    dec.ctx.sync()
    for t in range(t_steps):
        arr = np.ctypeslib.as_array(C.cast(bufs[t], C.POINTER(C.c_uint8)), shape=(n * size,))
        for s in range(n):
            assert np.array_equal(arr[s * size : (s + 1) * size], refs[s][t]["rgba"]), (s, t)
        L.h263cu_free_pinned(bufs[t])


def test_decode_step_from_bitstream_with_readback_and_bad_packet():
    """h263cu_decode_step: bitstream packets in, RGBA in pinned host memory out, parse of step t+1
    overlapping the device work of step t.  A packet that fails to parse is reported, leaves its
    stream untouched (state.rs:120-137) and the stream carries on with the next good packet."""
    import ctypes as C

    n, t_steps = 5, 4
    streams = [synth.make_stream(176, 144, t_steps, 700 + s, mv_mode=s % 3) for s in range(n)]
    refs = [oracle_decode_stream(p) for p in streams]
    dec = api.BatchDecoder(n, 176, 144, threads=3)
    L = _lib.lib()
    size = 176 * 144 * 4
    bufs, errs_all = [], []
    nxt = [0] * n  # next picture of every stream
    sent = []
    for t in range(t_steps + 1):
        packets, which = [], []
        for s in range(n):
            if s == 2 and t == 1:
                packets.append(b"\x12\x34\x56\x78\x9a")  # no picture start code
                which.append(-1)
            elif nxt[s] < t_steps:
                packets.append(streams[s][nxt[s]])
                which.append(nxt[s])
                nxt[s] += 1
            else:
                packets.append(b"")  # stream has ended: empty packet fails to parse, nothing happens
                which.append(-1)
        host = L.h263cu_alloc_pinned(n * size)
        assert host
        bufs.append(host)
        errs = dec.decode_step(packets, host_rgba=host, rgba_stride=size).copy()
        errs_all.append(errs)
        sent.append(which)
    dec.ctx.sync()
    for t in range(t_steps + 1):
        arr = np.ctypeslib.as_array(C.cast(bufs[t], C.POINTER(C.c_uint8)), shape=(n * size,))
        for s in range(n):
            k = sent[t][s]
            if k < 0:
                assert errs_all[t][s] != 0, (t, s)
                continue
            assert errs_all[t][s] == 0, (t, s, int(errs_all[t][s]))
            assert np.array_equal(arr[s * size : (s + 1) * size], refs[s][k]["rgba"]), (s, t)
        L.h263cu_free_pinned(bufs[t])
    for s in range(n):
        y, cb, cr = dec.ctx.read_yuv(s)
        assert np.array_equal(y, refs[s][-1]["y"]) and np.array_equal(cb, refs[s][-1]["cb"]) and np.array_equal(cr, refs[s][-1]["cr"])


def test_h263state_facade_surface():
    """The rest of the reference's H263State / DecodedPicture surface (state.rs:53-111, picture.rs:60-142)."""
    pk = synth.make_stream(176, 144, 3, 21)
    st = api.H263State()
    assert st.is_sorenson() and st.get_last_picture() is None and st.get_reference_picture() is None
    hdr = st.parse_picture(pk[0])
    assert (hdr["width"], hdr["height"], hdr["pic_type"]) == (176, 144, 0)
    assert st.get_last_picture() is None  # the peek changes nothing
    ref = oracle_decode_stream(pk)
    for i, p in enumerate(pk):
        st.decode_next_picture(p)
        st.cleanup_buffers()
        pic = st.get_last_picture()
        assert pic.format() == (176, 144) and pic.luma_samples_per_row() == 176 and pic.chroma_samples_per_row() == 88
        h = pic.as_header()
        assert h["quantizer"] == ref[i]["info"]["quant"] and h["temporal_reference"] == ref[i]["info"]["tr"]
        assert np.array_equal(pic.as_luma(), ref[i]["y"]) and np.array_equal(pic.as_chroma_b(), ref[i]["cb"])
        assert np.array_equal(st.get_reference_picture().as_chroma_r(), ref[i]["cr"])


def test_decode_step_refuses_before_any_parser_advances():
    """A step the device stage would refuse (a stream named twice, a stream id out of range) fails as a whole and
    leaves parsers and streams untouched: the same packets decode afterwards.  A picture larger than the context is
    that picture's error only: it is left out of the step, its parser does not advance, the other streams decode."""
    small = synth.make_stream(176, 144, 3, 31)
    big = synth.make_stream(352, 288, 1, 32)
    ref = oracle_decode_stream(small)
    dec = api.BatchDecoder(2, 176, 144, threads=2)
    with pytest.raises(_lib.H263Error) as e:
        dec.decode_step([small[0], small[0]], stream_ids=[1, 1])
    assert e.value.code == _lib.ERR_BAD_ARGUMENT
    with pytest.raises(_lib.H263Error) as e:
        dec.decode_step([small[0]], stream_ids=[7])
    assert e.value.code == _lib.ERR_CAPACITY
    errs = dec.decode_step([small[0], big[0]])
    assert errs[0] == 0 and errs[1] == _lib.ERR_CAPACITY
    dec.ctx.sync()
    with pytest.raises(_lib.H263Error) as e:  # stream 1 has still not decoded anything
        dec.ctx.read_yuv(1)
    assert e.value.code == _lib.ERR_NO_PICTURE
    for t in range(3):  # stream 0 carries on (its I picture decodes again, then the P pictures)
        assert not dec.decode_step([small[t]], stream_ids=[0]).any()
        dec.ctx.sync()
        y, cb, cr = dec.ctx.read_yuv(0)
        assert np.array_equal(y, ref[t]["y"]) and np.array_equal(cb, ref[t]["cb"]) and np.array_equal(cr, ref[t]["cr"])


def test_decode_step_is_a_transaction_when_the_device_stage_refuses():
    """The parsers move on only when the device stage has accepted the step (state.rs:120-137).  A P picture whose
    stream has no reference on the device (a fresh context behind a parser that has seen the I picture) is refused by
    the device stage with UncodedIFrameBlocks; the parser must not have advanced: the same P picture decodes exactly
    once the I picture has been replayed on the new context."""
    pk = synth.make_stream(176, 144, 3, 41)
    ref = oracle_decode_stream(pk)
    dec = api.BatchDecoder(1, 176, 144, threads=1)
    assert not dec.decode_step([pk[0]]).any()
    dec.ctx.sync()
    fresh = api.Context(0, 1, 176, 144)  # same parser, new device state
    dec.ctx = fresh
    with pytest.raises(_lib.H263Error):
        dec.decode_step([pk[1]])
    # parser unchanged: it still expects picture 1 after picture 0; give the device its reference back and go on
    pic, mbs, ev = frontend.Parser(1).parse_picture(pk[0])
    fresh.submit_step(pic, mbs, ev, _lib.OUT_RGBA)
    for t in (1, 2):
        assert not dec.decode_step([pk[t]]).any()
        fresh.sync()
        y, cb, cr = fresh.read_yuv(0)
        assert np.array_equal(y, ref[t]["y"]) and np.array_equal(cb, ref[t]["cb"]) and np.array_equal(cr, ref[t]["cr"])


def test_malformed_records_are_refused_before_they_reach_the_device():
    """Caller-built side info is checked on the host (h263cu_step_upload / h263cu_submit_step*): a record outside its
    picture's grid, out of raster order, pointing past its picture's events or naming another picture is refused."""
    pk = synth.make_stream(176, 144, 2, 51)
    ps = frontend.Parser(1)
    ctx = api.Context(0, 1, 176, 144)
    pic, mbs, ev = ps.parse_picture(pk[0])
    ctx.submit_step(pic, mbs, ev, _lib.OUT_RGBA)
    pic, mbs, ev = ps.parse_picture(pk[1])

    def refused(edit, side=None):
        p, m, u = side if side is not None else (pic, mbs, ev)
        m = m.copy()
        edit(m)
        with pytest.raises(_lib.H263Error) as e:
            ctx.submit_step(p, m, u, _lib.OUT_RGBA)
        assert e.value.code == _lib.ERR_BAD_ARGUMENT
        with pytest.raises(_lib.H263Error) as e:
            ctx.step_upload(p, m, u)
        assert e.value.code == _lib.ERR_BAD_ARGUMENT

    def one_block(side, k, b, n, code=None):
        """The picture with record k's events replaced by n narrow events (run 0, level +1) in block b, appended to
        the picture's events; `code` sets the block's INTRADC code."""
        p, m, u = side[0].copy(), side[1].copy(), np.concatenate([side[2], np.full(n, 1, np.uint16)])
        m["ev_off"][k], m["nev"][k] = len(u) - n, 0
        m["nev"][k, b] = n
        m["flags"][k] &= np.uint8(~_lib.MB_WIDE & 0xFF)
        if code is not None:
            m["u"][k, b] = code
        p["n_event_units"] = len(u)
        return p, m, u

    # Event counts no block can have, with every event inside the picture's share: the tiled kernel walks at most 64
    # events of a block (and would read past its event buffer), an intra DC takes zig-zag index 0, and INTRADC code 0
    # marks a dropped intra block.
    ipic, imbs, iev = frontend.Parser(1).parse_picture(pk[0])
    k_inter = int(np.flatnonzero(mbs["flags"] & _lib.MB_INTER)[0])
    refused(lambda m: None, one_block((pic, mbs, ev), k_inter, 0, 65))
    refused(lambda m: None, one_block((pic, mbs, ev), k_inter, 5, 65))
    refused(lambda m: None, one_block((pic, mbs, ev), k_inter, 3, 255))
    refused(lambda m: None, one_block((ipic, imbs, iev), 0, 2, 64, code=100))
    refused(lambda m: None, one_block((ipic, imbs, iev), 5, 4, 1, code=0))
    kb = tuple(int(v) for v in np.argwhere(imbs["nev"] > 0)[0])
    refused(lambda m: m["u"].__setitem__(kb, 0), (ipic, imbs, iev))  # code 0 over the parser's own events

    refused(lambda m: m["mbx"].__setitem__(5, 200))
    refused(lambda m: m["mby"].__setitem__(7, 99))
    refused(lambda m: m["pic"].__setitem__(0, 3))
    refused(lambda m: m["ev_off"].__setitem__(len(m) - 1, 1 << 30))
    refused(lambda m: m["nev"].__setitem__(len(m) - 1, [64, 64, 64, 64, 64, 64]))
    refused(lambda m: m.__setitem__(slice(0, 2), m[[1, 0]]))  # two records swapped: not in raster order
    # the untouched records still decode, exactly
    ctx.submit_step(pic, mbs, ev, _lib.OUT_RGBA)
    ctx.sync()
    y, _, _ = ctx.read_yuv(0)
    ref = oracle_decode_stream(pk)[1]
    assert np.array_equal(y, ref["y"])
    # the same records with counts a block can have decode exactly: 64 inter events (the last on index 63), 63 intra
    # events beside a dropped block (code 0, no events)
    prev = (ref["y"], ref["cb"], ref["cr"])
    for p, m, u in (one_block((pic, mbs, ev), k_inter, 5, 64), one_block((pic, mbs, ev), k_inter, 1, 64),
                    one_block((ipic, imbs, iev), 5, 2, 63, code=100)):
        if p["pic_type"][0] == _lib.PIC_I:
            m["u"][5, 4] = 0
        exp = recon_from_side_info(p[0], m, u, prev if p["pic_type"][0] != _lib.PIC_I else None)
        ctx.submit_step(p, m, u, _lib.OUT_RGBA)
        ctx.sync()
        y, cb, cr = ctx.read_yuv(0)
        assert np.array_equal(y, exp[0].reshape(-1)) and np.array_equal(cb, exp[1].reshape(-1)) and np.array_equal(cr, exp[2].reshape(-1))
        prev = (y, cb, cr)


def test_device_errors_are_loud():
    ctx = api.Context(0, 2, 176, 144)
    pk = synth.make_stream(352, 288, 1, 1)
    pic, mbs, ev = frontend.Parser(1).parse_picture(pk[0])
    with pytest.raises(_lib.H263Error) as e:  # picture larger than the context
        ctx.submit_step(pic, mbs, ev, _lib.OUT_RGBA)
    assert e.value.code == _lib.ERR_CAPACITY
    with pytest.raises(_lib.H263Error) as e:
        ctx.read_yuv(0)
    assert e.value.code == _lib.ERR_NO_PICTURE


def test_tiled_and_generic_kernels_agree_and_interleave(monkeypatch):
    """The tiled kernel and the generic warp-per-MB kernel are two independent implementations: both
    must match the oracle, on an aligned and an unaligned stream sharing steps, whichever is forced."""
    n = 8
    a = synth.make_stream(352, 288, n, 77, mv_mode=2, intra_period=4, pct_fourmv=20)
    b = synth.make_stream(200, 100, n, 78, mv_mode=1)
    ra, rb = oracle_decode_stream(a), oracle_decode_stream(b)
    for force in (None, "mb", "tile"):
        if force:
            monkeypatch.setenv("H263CU_KERNEL", force)
        else:
            monkeypatch.delenv("H263CU_KERNEL", raising=False)
        ctx = api.Context(0, 2, 352, 288)
        pa, pb = frontend.Parser(1), frontend.Parser(1)
        tb = 0
        for t in range(n):
            with_b = t in (0, 1, 5)
            parsers, packets, ids = [pa], [a[t]], [0]
            if with_b:
                parsers, packets, ids = [pa, pb], [a[t], b[tb]], [0, 1]
            pics, mbs, events, errs, _ = frontend.parse_step(parsers, packets, ids, 2)
            assert not errs.any()
            ctx.submit_step(pics, mbs, events, _lib.OUT_RGBA)
            ctx.sync()
            y, cb, cr = ctx.read_yuv(0)
            assert np.array_equal(y, ra[t]["y"]) and np.array_equal(cb, ra[t]["cb"]) and np.array_equal(cr, ra[t]["cr"]), (force, t)
            assert np.array_equal(ctx.read_rgba(0), ra[t]["rgba"]), (force, t)
            if with_b:
                y, cb, cr = ctx.read_yuv(1)
                assert np.array_equal(y, rb[tb]["y"]) and np.array_equal(cb, rb[tb]["cb"]), (force, t)
                assert np.array_equal(ctx.read_rgba(1), rb[tb]["rgba"])
                tb += 1
        ctx.close()


def _decode_with_records(monkeypatch, force, packets_by_stream, dims, edit):
    """Decodes the streams in lock step through submit_step; `edit(t, pics, mbs)` may rewrite the side info of a step."""
    if force:
        monkeypatch.setenv("H263CU_KERNEL", force)
    else:
        monkeypatch.delenv("H263CU_KERNEL", raising=False)
    n = len(packets_by_stream)
    ctx = api.Context(0, n, max(d[0] for d in dims), max(d[1] for d in dims))
    parsers = [frontend.Parser(1) for _ in range(n)]
    out = []
    for t in range(len(packets_by_stream[0])):
        pics, mbs, events, errs, _ = frontend.parse_step(parsers, [p[t] for p in packets_by_stream], list(range(n)), 2)
        assert not errs.any()
        edit(t, pics, mbs)
        ctx.submit_step(pics, mbs, events, _lib.OUT_RGBA)
        ctx.sync()
        out.append([(ctx.read_yuv(s), ctx.read_rgba(s)) for s in range(n)])
    launches = (ctx.launch_count(), ctx.tiled_launch_count())
    ctx.close()
    return out, launches


PICFLAG_MV_IN_RANGE = 4


def test_vectors_beyond_the_range_take_the_clamped_path(monkeypatch):
    """Hand-built side info may hold vectors the front end never emits (beyond [-32, 31] half-pel units; the
    parser's own are always inside, mvd_pred.rs:70-117, and it says so with H263CU_PICFLAG_MV_IN_RANGE).  Without the
    flag the tiled kernel runs its instantiation with the clamped per-sample prediction (read_sample,
    gather.rs:16-31) and must agree bit for bit with the generic warp-per-macroblock kernel; aligned and unaligned
    picture sizes.  With the flag set falsely the library clears it (it derives the flag from the records)."""
    dims = [(352, 288), (200, 100)]
    streams = [synth.make_stream(w, h, 4, 900 + i, mv_mode=2, pct_fourmv=20) for i, (w, h) in enumerate(dims)]
    rng = np.random.default_rng(5)
    picks = {}

    def edit(keep_flag):
        def f(t, pics, mbs):
            assert (pics["flags"] & PICFLAG_MV_IN_RANGE).all()  # the parser vouches for its vectors
            if t == 0:
                return
            inter = np.flatnonzero((mbs["flags"] & _lib.MB_INTER) != 0)
            if t not in picks:
                idx = rng.choice(inter, size=min(60, len(inter)), replace=False)
                picks[t] = (idx, rng.integers(-120, 121, size=(len(idx), 8)).astype(np.int8))
            idx, mv = picks[t]
            mbs["u"][idx] = mv.view(np.uint8)
            if not keep_flag:
                pics["flags"] &= np.uint8(~PICFLAG_MV_IN_RANGE & 0xFF)
        return f

    tiled, (n_launch, n_tiled) = _decode_with_records(monkeypatch, None, streams, dims, edit(False))
    assert n_tiled == n_launch  # the tiled kernel ran, in its WIDE_MV instantiation
    generic, _ = _decode_with_records(monkeypatch, "mb", streams, dims, edit(False))
    for t in range(len(tiled)):
        for s in range(len(dims)):
            (ya, ca, ra), rgba_a = tiled[t][s]
            (yb, cb_, rb), rgba_b = generic[t][s]
            assert np.array_equal(ya, yb) and np.array_equal(ca, cb_) and np.array_equal(ra, rb), (t, s)
            assert np.array_equal(rgba_a, rgba_b), (t, s)
    # flag set falsely: the library derives MV_IN_RANGE from the records itself (validate_side_info), so the step
    # still takes the clamped-fetch instantiation and the result is the exact one
    lied, _ = _decode_with_records(monkeypatch, None, streams, dims, edit(True))
    for t in range(len(tiled)):
        for s in range(len(dims)):
            (ya, ca, ra), rgba_a = tiled[t][s]
            (yb, cb_, rb), rgba_b = lied[t][s]
            assert np.array_equal(ya, yb) and np.array_equal(ca, cb_) and np.array_equal(ra, rb) and np.array_equal(rgba_a, rgba_b), (t, s)


def test_pipelined_state_overlaps_and_stays_exact():
    """H263State(pipelined=True): decode_next_picture returns once the picture is queued; picture t is consumed after
    packet t + 1 has been handed in (parse of t + 1 overlaps the device work of t).  Every picture still matches the
    oracle, planes and RGBA, and a bad packet in the middle leaves the stream untouched (state.rs:120-137)."""
    pk = synth.make_stream(352, 288, 8, 61, mv_mode=1, pct_fourmv=10)
    ref = oracle_decode_stream(pk)
    st = api.H263State(pipelined=True)
    st.decode_next_picture(pk[0])
    for t in range(1, len(pk)):
        if t == 4:
            with pytest.raises(_lib.H263Error):
                st.decode_next_picture(b"\x00\x00\x80\x01garbage")
        prev = st.get_last_rgba(copy=False)  # picture t - 1: waits for its read-back only
        assert np.array_equal(prev, ref[t - 1]["rgba"]), t - 1
        st.decode_next_picture(pk[t])        # queued; the buffer of picture t - 1 stays valid
        assert np.array_equal(prev, ref[t - 1]["rgba"]), t - 1
    assert np.array_equal(st.get_last_rgba(), ref[-1]["rgba"])
    y, cb, cr = st.get_last_picture().as_yuv()
    assert np.array_equal(y, ref[-1]["y"]) and np.array_equal(cb, ref[-1]["cb"]) and np.array_equal(cr, ref[-1]["cr"])


def test_device_group_shares_parser_threads_across_contexts():
    """h263cu_group_*: one process, several device contexts (here all on device 0, which exercises the same code as
    several GPUs), one shared pool of parser threads.  Global stream s lives on context s % n, slot s // n; RGBA lands
    device-major in the host buffer.  Bit exact against the oracle, with a failing packet and a stream sitting out."""
    import ctypes as C

    n_ctx, per = 3, 4
    n = n_ctx * per
    t_steps = 4
    streams = [synth.make_stream(176, 144, t_steps, 800 + s, mv_mode=s % 3) for s in range(n)]
    refs = [oracle_decode_stream(p) for p in streams]
    grp = api.DeviceGroup([0] * n_ctx, per, 176, 144, threads=3)
    L = _lib.lib()
    size = 176 * 144 * 4
    host = [L.h263cu_alloc_pinned(n * size) for _ in range(2)]
    assert all(host)
    done = [0] * n
    for t in range(t_steps + 1):
        ids, packets, expect = [], [], []
        for s in range(n):
            if s == 5 and t == 2:
                continue  # stream 5 sits this step out
            if done[s] >= t_steps:
                continue
            if s == 7 and t == 1:
                ids.append(s), packets.append(b"\xff\xff\xff\xff"), expect.append(None)
                continue
            ids.append(s), packets.append(streams[s][done[s]]), expect.append(done[s])
            done[s] += 1
        if not ids:
            break
        errs = grp.decode_step(packets, stream_ids=ids, host_rgba=host[t & 1], rgba_stride=size).copy()
        grp.sync()
        arr = np.ctypeslib.as_array(C.cast(host[t & 1], C.POINTER(C.c_uint8)), shape=(n * size,))
        for k, s in enumerate(ids):
            if expect[k] is None:
                assert errs[k] != 0
                continue
            assert errs[k] == 0, (t, s, int(errs[k]))
            r = refs[s][expect[k]]
            p = grp.position(s)
            assert np.array_equal(arr[p * size : (p + 1) * size], r["rgba"]), (t, s)
            ctx, slot = grp.where(s)
            y, cb, cr = ctx.read_yuv(slot)
            assert np.array_equal(y, r["y"]) and np.array_equal(cb, r["cb"]) and np.array_equal(cr, r["cr"]), (t, s)
    assert all(d == t_steps for d in done)
    for h in host:
        L.h263cu_free_pinned(h)
    grp.close()


def test_resident_steps_as_one_cuda_graph():
    """h263cu_graph_*: the resident steps of one stream captured into ONE CUDA graph (BASELINE.json configs[1]: a
    single stream is a chain of dependent launches).  The graph is bound to the stream state it was built from: it
    runs from there, leaves the bookkeeping where the steps would have, can be launched again when the picture count
    is even, and refuses to run from any other state.  Planes and RGBA match the oracle."""
    pk = synth.make_stream(352, 288, 7, 91, mv_mode=1)
    ref = oracle_decode_stream(pk)
    ctx = api.Context(0, 1, 352, 288)
    ps = frontend.Parser(1)
    steps = []
    for p in pk:
        pic, mbs, ev = ps.parse_picture(p)
        steps.append(ctx.step_upload(pic, mbs, ev))
    ctx.step_run(steps[0], _lib.OUT_RGBA)          # the I picture, the ordinary way
    g = ctx.graph_build(steps[1:7], _lib.OUT_RGBA)  # six P pictures: an even count
    n0 = ctx.launch_count()
    ctx.graph_launch(g)
    ctx.sync()
    assert ctx.launch_count() == n0 + 6 and ctx.tiled_launch_count() == 7
    y, cb, cr = ctx.read_yuv(0)
    assert np.array_equal(y, ref[6]["y"]) and np.array_equal(cb, ref[6]["cb"]) and np.array_equal(cr, ref[6]["cr"])
    assert np.array_equal(ctx.read_rgba(0), ref[6]["rgba"])
    assert ctx.stream_info(0)["tr"] == ref[6]["info"]["tr"]
    # an even number of pictures leaves the plane slots where they started: the same graph runs again (P on top of P:
    # the result differs from the stream's, the call must simply be accepted), an odd-length one would not fit after it
    ctx.graph_launch(g)
    ctx.sync()
    g_odd = ctx.graph_build(steps[1:4], _lib.OUT_RGBA)
    ctx.graph_launch(g_odd)
    with pytest.raises(_lib.H263Error) as e:  # the slots have moved on by three pictures: not the captured state
        ctx.graph_launch(g_odd)
    assert e.value.code == _lib.ERR_BAD_ARGUMENT
    with pytest.raises(_lib.H263Error):
        ctx.graph_launch(g)
    ctx.sync()
    ctx.graph_free(g)
    ctx.graph_free(g_odd)
    for s in steps:
        ctx.step_free(s)
    ctx.close()


def test_disposable_p_pictures_are_shown_but_never_predicted_from():
    """EXTENSION (H263CU_OPT_DECODE_DISPOSABLE): Sorenson disposable P pictures decode like P pictures, become the
    stream's last picture, and the next picture still predicts from the last non-disposable one.  Bit exact against
    the oracle run with the same extension, through the single-stream state, the batch path and a CUDA graph."""
    opt = 1 | 0x100
    pk = synth.make_stream(352, 288, 9, 91, pct_disposable=45, mv_mode=2, pct_fourmv=15)
    types = [int(frontend.peek_picture(p)["pic_type"]) for p in pk]
    assert types.count(_lib.PIC_DISPOSABLE_P) >= 2 and types.count(_lib.PIC_P) >= 2
    # a disposable picture followed by a P picture must be in the stream, else the test shows nothing
    assert any(a == _lib.PIC_DISPOSABLE_P and b == _lib.PIC_P for a, b in zip(types, types[1:]))
    ref = oracle_decode_stream(pk, opt)
    st = api.H263State(opt)
    for i, p in enumerate(pk):
        st.decode_next_picture(p)
        y, cb, cr = st.get_last_picture().as_yuv()
        assert np.array_equal(y, ref[i]["y"]) and np.array_equal(cb, ref[i]["cb"]) and np.array_equal(cr, ref[i]["cr"]), (i, types[i])
        assert np.array_equal(st.get_last_rgba(), ref[i]["rgba"]), (i, types[i])
    # without the extension the product refuses the picture like the reference does, and the stream carries on
    st2 = api.H263State(1)
    first = types.index(_lib.PIC_DISPOSABLE_P)
    for p in pk[:first]:
        st2.decode_next_picture(p)
    with pytest.raises(_lib.H263Error) as e:
        st2.decode_next_picture(pk[first])
    assert e.value.code == -17
    # resident steps + CUDA graph walk the same slot logic
    ctx = api.Context(0, 1, 352, 288)
    ps = frontend.Parser(opt)
    steps = []
    for p in pk:
        pic, mbs, ev = ps.parse_picture(p)
        steps.append(ctx.step_upload(pic, mbs, ev))
    ctx.step_run(steps[0], _lib.OUT_RGBA)
    g = ctx.graph_build(steps[1:], _lib.OUT_RGBA)
    ctx.graph_launch(g)
    ctx.sync()
    y, cb, cr = ctx.read_yuv(0)
    assert np.array_equal(y, ref[-1]["y"]) and np.array_equal(cb, ref[-1]["cb"]) and np.array_equal(cr, ref[-1]["cr"])
    assert np.array_equal(ctx.read_rgba(0), ref[-1]["rgba"])
    ctx.graph_free(g)
    for s in steps:
        ctx.step_free(s)
    ctx.close()
