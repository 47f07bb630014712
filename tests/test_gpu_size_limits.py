"""GPU parity at the ends of the picture-size range: 4080 x 4080 (255 x 255 macroblocks, the largest picture the API
takes), 4065 x 4065 (255 macroblocks of which the last holds one valid luma column and row, 2033 chroma columns),
4080 x 16 and 16 x 4080 (one macroblock row / column), 16CIF in the baseline flavour, and 1 x 1, 2 x 2, 255 x 255 and
256 x 256 (both sides of Sorenson's 8-bit / 16-bit custom size code).  Only these sizes reach some encodings of the
kernels at their limit: the device parse's vector ring full at 255 columns (parse_mb.cu, MV_RING), the slot << 12 |
16 mby row word of the device outputs at 16 mby = 4064 with the picture in a slot >= 1, the run-time pitch instantiation
at pitch 4144, byte-wide mbx / mby / mb_w / mb_h at 254 / 255, resize filters with about 74 taps per axis, and the
deblock kernels and the EDGE fix-up on 4065-wide rows.

Every output is compared bit for bit with its reference: the oracle's planes and RGBA (deblocked on request), the
restatements resample_ref / fit_ref / filter_ref applied to the oracle's RGBA, the motion and residual models
(motion_ref, residual_ref), the host parser's side info for the device parse, and helpers.recon_from_side_info for
hand-built side info.  Contexts hold at most 4 streams of 4080 x 4080 (about 0.74 GB)."""
import numpy as np
import pytest
import torch

import filter_ref as FL
import motion_ref as M
import oracle_lib as O
import recon_cases as R
import residual_ref as RR
from helpers import oracle_decode_stream, recon_from_side_info
from h263_rs_b200 import _lib, api, frontend, synth
from test_gpu_device_parse import lockstep_parse
from test_gpu_device_tensor import IMAGENET, bits, expected
from test_gpu_device_tensor_filter import expected_filter
from test_gpu_device_tensor_fit import expected_fit

pytestmark = pytest.mark.gpu

# vectors pushed across all four borders, 4MV, intra-in-P, DQUANT and escapes in every stream
COMMON = dict(mv_mode=2, pct_fourmv=40, pct_intra=10, pct_dquant=20, pct_escape=5, deblock_flag=1)
# name: (width, height, pictures, seed, decoder options, generator overrides)
STREAMS = {
    "4080": (4080, 4080, 3, 71, 1, {}),
    "4065": (4065, 4065, 3, 72, 1, {}),
    "4080x16": (4080, 16, 4, 73, 1, dict(pct_fourmv=60)),
    "16x4080": (16, 4080, 4, 74, 1, dict(pct_fourmv=60)),
    "16cif": (1408, 1152, 4, 75, 0, dict(flavour=1)),
    "1x1": (1, 1, 4, 76, 1, {}),
    "2x2": (2, 2, 4, 77, 1, {}),
    "255": (255, 255, 4, 78, 1, {}),
    "256": (256, 256, 4, 79, 1, {}),
    # for the device parse's side info: every column's upper-right neighbour read from a full ring
    "4080x48": (4080, 48, 4, 80, 1, dict(pct_fourmv=60, pct_uncoded=5, pct_intra=20)),
}
# The decode steps: (context size, stream names in input order).  Input i goes to slot i of a caller's buffer, so the
# 4080 x 4080 and 4065 x 4065 pictures sit in slots >= 1.  The aligned groups run the run-time-pitch aligned
# instantiation, the edge groups EDGE; every grid is sized by the context while the smallest picture stays exact.
GROUPS = {
    "aligned_4080": ((4080, 4080), ["4080x16", "4080", "16x4080"]),
    "edge_4080": ((4080, 4080), ["1x1", "4065", "4080", "16x4080"]),
    "aligned_16cif": ((1408, 1152), ["256", "16cif"]),
    "edge_16cif": ((1408, 1152), ["2x2", "16cif", "255", "1x1"]),
}
BIG = ("4080", "4065")
PAT = 0x5A


@pytest.fixture(scope="module")
def streams():
    out = {}
    for name, (w, h, n, seed, opt, kw) in STREAMS.items():
        out[name] = (synth.make_stream(w, h, n, seed, **dict(COMMON, **kw)), opt)
    return out


@pytest.fixture(scope="module")
def refs(streams):
    """refs(kind, name): the per-picture references of a stream, computed once: "oracle" (oracle_decode_stream),
    "oracle_db" (RGBA of the deblocked planes), "planes" / "planes_db" ([y, cb, cr] 2-D, deblocked), "motion",
    "residual", "records" (the host parser's (pic, mbs, events))."""
    cache = {}

    def get(kind, name):
        key = (kind, name)
        if key in cache:
            return cache[key]
        pk, opt = streams[name]
        if kind == "oracle":
            v = oracle_decode_stream(pk, opt)
        elif kind == "oracle_db":
            v = oracle_decode_stream(pk, opt, deblock=True)
        elif kind in ("planes", "planes_db"):
            v = []
            for r in get("oracle", name):
                w, h = r["info"]["width"], r["info"]["height"]
                cw, ch = (w + 1) // 2, (h + 1) // 2
                y, cb, cr = r["y"], r["cb"], r["cr"]
                if kind == "planes_db":
                    s = O.lib().orc_quant_to_strength(r["info"]["quant"])
                    y, cb, cr = O.deblock(y, w, s), O.deblock(cb, cw, s), O.deblock(cr, cw, s)
                v.append([np.asarray(y, np.uint8).reshape(h, w), np.asarray(cb, np.uint8).reshape(ch, cw),
                          np.asarray(cr, np.uint8).reshape(ch, cw)])
        elif kind == "motion":
            v = M.reference_stream(pk, opt)
        elif kind == "residual":
            v = RR.reference_stream(pk, opt)
        elif kind == "records":
            ps = frontend.Parser(opt)
            v = [ps.parse_picture(p) for p in pk]
        else:
            raise KeyError(kind)
        for r in v:
            assert not isinstance(r, int), (name, r)  # every picture of every stream decodes
        cache[key] = v
        return v

    return get


def decoder(streams, group):
    (cw, ch), names = GROUPS[group]
    dec = api.BatchDecoder(len(names), cw, ch, threads=4)
    dec.parsers = [frontend.Parser(streams[n][1]) for n in names]
    return dec


def steps(streams, group):
    """(t, stream ids, names, packets) of every step of a group: picture t of every stream that has one"""
    names = GROUPS[group][1]
    for t in range(max(len(streams[n][0]) for n in names)):
        ids = [k for k, n in enumerate(names) if t < len(streams[n][0])]
        yield t, ids, [names[k] for k in ids], [streams[names[k]][0][t] for k in ids]


def _kernel(monkeypatch, kernel):
    # read in h263cu_create: set before the context exists
    if kernel == "mb":
        monkeypatch.setenv("H263CU_KERNEL", "mb")
    else:
        monkeypatch.delenv("H263CU_KERNEL", raising=False)


def test_generated_streams_reach_the_limits(streams, refs):
    """The coverage this file relies on, asserted from the host parser's records so that a change of the generator
    cannot quietly stop reaching it: macroblocks at mbx = 254 and mby = 254, 4MV macroblocks in columns 253 and 254 of
    the 255-column rows, and vectors that leave the picture across each of its four borders."""
    recs = refs("records", "4080")
    assert any((m["mbx"] == 254).any() for _, m, _ in recs) and any((m["mby"] == 254).any() for _, m, _ in recs)
    for name in ("4080", "4065", "4080x16", "4080x48"):
        cols = set()
        for _, m, _ in refs("records", name):
            four = m[((m["flags"] & _lib.MB_INTER) != 0) & ((m["flags"] & _lib.MB_FOURMV) != 0)]
            cols |= {int(x) for x in four["mbx"]}
        assert {253, 254} <= cols, (name, sorted(c for c in cols if c > 250))
    for name in ("4080", "4065", "4080x16", "16x4080", "16cif", "255"):
        w, h = STREAMS[name][:2]
        borders = set()
        for pic, m, _ in refs("records", name):
            for r in m[(m["flags"] & _lib.MB_INTER) != 0]:
                mv = r["u"].view(np.int8).reshape(4, 2).astype(int)
                for k in range(4):
                    x, y = 16 * int(r["mbx"]) + 8 * (k & 1), 16 * int(r["mby"]) + 8 * (k >> 1)
                    if x >= w or y >= h:
                        continue
                    sx, sy = x + (mv[k, 0] >> 1), y + (mv[k, 1] >> 1)
                    borders |= {b for b, hit in (("left", sx < 0), ("top", sy < 0), ("right", sx + 8 + (mv[k, 0] & 1) > w),
                                                 ("bottom", sy + 8 + (mv[k, 1] & 1) > h)) if hit}
        assert borders == {"left", "right", "top", "bottom"}, (name, borders)


# ------------------------------------------------------------------------------------------ (a) planes, host RGBA
@pytest.mark.parametrize("deblock", [False, True], ids=["plain", "deblock"])
@pytest.mark.parametrize("kernel", ["default", "mb"])
@pytest.mark.parametrize("parse", ["host", "device"])
@pytest.mark.parametrize("group", list(GROUPS))
def test_planes_and_host_rgba(monkeypatch, streams, refs, group, parse, kernel, deblock):
    _kernel(monkeypatch, kernel)
    dec = decoder(streams, group)
    flags = _lib.OUT_RGBA | (_lib.OUT_DEBLOCK if deblock else 0)
    n_steps = 0
    for t, ids, names, pk in steps(streams, group):
        errs = dec.decode_step(pk, out_flags=flags, stream_ids=ids, parse=parse)
        assert not errs.any(), (t, names, errs)
        n_steps += 1
        dec.ctx.sync()
        for s, name in zip(ids, names):
            want = refs("planes", name)[t]
            for p, got, pw in zip("YUV", dec.ctx.read_yuv(s), want):
                assert np.array_equal(got, pw.reshape(-1)), (group, t, name, p, int((got != pw.reshape(-1)).sum()))
            rgba = refs("oracle_db" if deblock else "oracle", name)[t]["rgba"]
            got = dec.ctx.read_rgba(s)
            assert np.array_equal(got, rgba), (group, t, name, "RGBA", int((got != rgba).sum()))
    assert dec.ctx.launch_count() >= n_steps
    assert dec.ctx.tiled_launch_count() == (0 if kernel == "mb" else n_steps)
    dec.ctx.close()


# ------------------------------------------------------------------------------------------ (b) device RGBA, I420, NV12
def check_slots(got, cols, pictures, what):
    """got: [slots, rows, padded columns, ...] host copy of a pattern-filled buffer whose slots are `cols` columns wide;
    pictures: (slot, expected [h, w, ...]).  Each picture sits at its slot's top left; the row padding and the slots
    without a picture keep the pattern (the rest of a slot's rectangle may be written, include/h263cu.h)."""
    for k, want in pictures:
        h, w = want.shape[:2]
        region = got[k, :h, :w]
        assert np.array_equal(region, want), (what, "slot", k, int((region != want).sum()))
    assert (got[:, :, cols:] == PAT).all(), (what, "row padding written")
    for k in range(len(pictures), got.shape[0]):
        assert (got[k] == PAT).all(), (what, "slot", k, "written without a picture")


@pytest.mark.parametrize("kind", ["rgba", "rgba_db", "i420", "i420_db", "nv12", "nv12_db"])
@pytest.mark.parametrize("parse", ["host", "device"])
@pytest.mark.parametrize("group", list(GROUPS))
def test_device_rgba_and_yuv(streams, refs, group, parse, kind):
    """Caller-owned tensors with padded rows, pattern-filled before every step."""
    dec = decoder(streams, group)
    (W, H), names = GROUPS[group]
    n = len(names)
    deblock = kind.endswith("_db")
    dev = torch.device("cuda", 0)
    cw, ch = (W + 1) // 2, (H + 1) // 2
    if kind.startswith("rgba"):
        shapes = [((n, H, W + 4, 4), W)]
    elif kind.startswith("nv12"):
        shapes = [((n, H, W + 4), W), ((n, ch, cw + 2, 2), cw)]
    else:
        shapes = [((n, H, W + 4), W), ((n, ch, cw + 4), cw), ((n, ch, cw + 4), cw)]
    bases = [torch.empty(s, dtype=torch.uint8, device=dev) for s, _ in shapes]
    out = [b[:, :, :c] for b, (_, c) in zip(bases, shapes)]  # rows padded past the slot's width
    cols = [c for _, c in shapes]
    for t, ids, names_t, pk in steps(streams, group):
        for b in bases:
            b.fill_(PAT)
        if kind.startswith("rgba"):
            _, errs = dec.decode_step_device(pk, out=out[0], out_flags=_lib.OUT_RGBA | (_lib.OUT_DEBLOCK if deblock else 0),
                                             stream_ids=ids, parse=parse)
        else:
            _, errs = dec.decode_step_device_yuv(pk, out=tuple(out), layout=kind[:4], deblock=deblock, stream_ids=ids, parse=parse)
        assert not errs.any(), (t, names_t, errs)
        torch.cuda.synchronize()
        got = [b.cpu().numpy() for b in bases]
        for k, name in enumerate(names_t):
            if name in BIG:
                assert k >= 1  # the row word's slot bits are above 16 * mby = 4064 (rows 4064..4079 of the slot)
        if kind.startswith("rgba"):
            pics = []
            for k, name in enumerate(names_t):
                r = refs("oracle_db" if deblock else "oracle", name)[t]
                w, h = r["info"]["width"], r["info"]["height"]
                pics.append((k, np.asarray(r["rgba"], np.uint8).reshape(h, w, 4)))
            check_slots(got[0], cols[0], pics, (group, t, kind))
            continue
        planes = [(k, refs("planes_db" if deblock else "planes", name)[t]) for k, name in enumerate(names_t)]
        check_slots(got[0], cols[0], [(k, p[0]) for k, p in planes], (group, t, kind, "Y"))
        if kind.startswith("nv12"):
            check_slots(got[1], cols[1], [(k, np.stack([p[1], p[2]], axis=-1)) for k, p in planes], (group, t, kind, "UV"))
        else:
            check_slots(got[1], cols[1], [(k, p[1]) for k, p in planes], (group, t, kind, "Cb"))
            check_slots(got[2], cols[2], [(k, p[2]) for k, p in planes], (group, t, kind, "Cr"))
    dec.ctx.close()


# ------------------------------------------------------------------------------------------ (c) tensor outputs
# kind: (decode_step_device_tensor keywords, the reference of one picture); downscales from 4080 to 224 (bicubic: about
# 74 taps per axis, the general path) and upscales of 1 x 1 and 16 x 4080 to 224 x 224 (the edge groups)
SIZE = (224, 224)
TENSORS = {
    "stretch_f16": (dict(dtype=torch.float16), lambda r: expected(r, SIZE, torch.float16)),
    "center_crop_f32": (dict(dtype=torch.float32, fit="center_crop", short_side=256),
                        lambda r: expected_fit(r, SIZE, torch.float32, "center_crop", 256)),
    "bicubic_aa_u8": (dict(dtype=torch.uint8, antialias=True, interpolation="bicubic"),
                      lambda r: expected_filter(r, SIZE, torch.uint8, "stretch", FL.BICUBIC_AA)),
    "bicubic_aa_bf16": (dict(dtype=torch.bfloat16, antialias=True, interpolation="bicubic", **IMAGENET),
                        lambda r: expected_filter(r, SIZE, torch.bfloat16, "stretch", FL.BICUBIC_AA, **IMAGENET)),
}


@pytest.fixture(scope="module")
def tensor_refs(refs):
    cache = {}

    def get(kind, name, t):
        if (kind, name, t) not in cache:
            cache[(kind, name, t)] = TENSORS[kind][1](refs("oracle", name)[t])
        return cache[(kind, name, t)]

    return get


@pytest.mark.parametrize("kind", list(TENSORS))
@pytest.mark.parametrize("parse", ["host", "device"])
@pytest.mark.parametrize("group", list(GROUPS))
def test_tensor_outputs(streams, tensor_refs, group, parse, kind):
    dec = decoder(streams, group)
    kw = TENSORS[kind][0]
    for t, ids, names, pk in steps(streams, group):
        out, errs = dec.decode_step_device_tensor(pk, SIZE, stream_ids=ids, parse=parse, **kw)
        assert not errs.any(), (t, names, errs)
        got = out.cpu()
        for k, name in enumerate(names):
            want = tensor_refs(kind, name, t)
            assert torch.equal(bits(got[k]), bits(want)), (group, t, name, kind, int((bits(got[k]) != bits(want)).sum()))
    dec.ctx.close()


# ------------------------------------------------------------------------------------------ (d) motion fields, residuals
@pytest.mark.parametrize("parse", ["host", "device"])
@pytest.mark.parametrize("group", list(GROUPS))
def test_motion_fields_and_residuals(streams, refs, group, parse):
    """Motion fields in slots of the context's grid (255 x 255 macroblocks for the 4080 groups) and int16 residuals in
    slots of the context's size (4080 x 4080), pattern-filled before every step."""
    dec = decoder(streams, group)
    (W, H), names = GROUPS[group]
    n = len(names)
    MBW, MBH = (W + 15) // 16, (H + 15) // 16
    dev = torch.device("cuda", 0)
    motion = api.Motion(*[torch.empty(s, dtype=d, device=dev) for s, d in
                          zip(api.motion_shapes(n, W, H), (torch.int16, torch.uint8, torch.uint8))])
    res = api.Residual(*[torch.empty(s, dtype=torch.int16, device=dev) for s in api.residual_shapes(n, W, H)])
    assert motion.flags.shape[1:] == (MBH, MBW)
    for t, ids, names_t, pk in steps(streams, group):
        for x in motion + res:
            x.fill_(PAT)
        m, r, errs = dec.decode_step_device_residual(pk, residual=res, motion=motion, stream_ids=ids, parse=parse)
        assert m is motion and r is res
        assert not errs.any(), (t, names_t, errs)
        torch.cuda.synchronize()
        gm = [x.cpu().numpy() for x in motion]
        gr = [x.cpu().numpy() for x in res]
        for k, name in enumerate(names_t):
            e = M.slot(refs("motion", name)[t], MBW, MBH)
            for f, a in zip(("mv", "flags", "quant"), gm):
                assert np.array_equal(a[k], e[f]), (group, t, name, f, np.argwhere(a[k] != e[f])[:5])
            e = RR.slot(refs("residual", name)[t], W, H)
            for f, a in zip(("y", "cb", "cr"), gr):
                assert np.array_equal(a[k], e[f]), (group, t, name, f, np.argwhere(a[k] != e[f])[:5])
        for k in range(len(names_t), n):
            assert all((a[k] == PAT).all() for a in gm + gr)
    dec.ctx.close()


# ------------------------------------------------------------------------------------------ side info of the device parse
def test_device_parse_side_info_at_255_columns(streams, refs):
    """The device parse's records and events equal the host parser's byte for byte at mb_w = 255 (the vector ring of
    MV_RING = 256 slots holds R = 256 of them: full), mb_w = 1 (R = 2) and 1 x 1.  4080 x 48 carries 60 % 4MV, so the
    upper-right neighbour of every column is read from the full ring."""
    names = ["4080x48", "4080x16", "16x4080", "1x1"]
    ctx = api.Context(0, len(names), 4080, 4080)
    errs = lockstep_parse(ctx, [streams[n][0] for n in names], [streams[n][1] for n in names])
    assert not any(errs)
    four = set()
    for _, m, _ in refs("records", "4080x48"):
        sel = m[((m["flags"] & _lib.MB_FOURMV) != 0) & (m["mby"] > 0)]
        four |= {int(x) for x in sel["mbx"]}
    assert {253, 254} <= four  # 4MV below the first row in the last two columns: predictions from the ring's far end
    ctx.close()


# ------------------------------------------------------------------------------------------ hand-built side info
def push_out(g, specs, w, h, wide):
    """Every inter macroblock on a border gets vectors that point out of the picture across it: within [-32, 31], or
    with `wide` beyond it (up to +-120 half-pel units: the WIDE_MV instantiations)."""
    mb_w, mb_h = (w + 15) // 16, (h + 15) // 16
    lo, hi = (33, 121) if wide else (1, 32)
    for k, s in enumerate(specs):
        X, Y = k % mb_w, k // mb_w
        if not s["inter"] or not (X in (0, mb_w - 1) or Y in (0, mb_h - 1)):
            continue
        mv = []
        for _ in range(4):
            x, y = (int(v) for v in g.rng.integers(-8, 9, 2))
            if X == 0:
                x = -int(g.rng.integers(lo, hi))
            elif X == mb_w - 1:
                x = int(g.rng.integers(lo, min(hi, 32) if not wide else hi))
            if Y == 0:
                y = -int(g.rng.integers(lo, hi))
            elif Y == mb_h - 1:
                y = int(g.rng.integers(lo, min(hi, 32) if not wide else hi))
            mv.append((x, y))
        s["mv"] = mv
    return specs


def handbuilt_stream(w, h, wide, seed):
    """A textured I picture, then P pictures: with 1020 macroblocks, the first carries every block kind of
    recon_cases.case_mbs (filled up with random tiles); a picture of 255 macroblocks (not a multiple of 4) is drawn
    from recon_cases.Gen tile by tile.  Vectors point out across every border."""
    g = R.Gen(seed)
    n = ((w + 15) // 16) * ((h + 15) // 16)
    pics = [(w, h, R.textured_intra(g, n), 7)]
    parts = []
    if n % 4 == 0:
        tiles = iter([])

        def filler():
            nonlocal tiles
            m = next(tiles, None)
            if m is None:
                tiles = iter(g.random_tile())
                m = next(tiles)
            return m

        parts = R.pictures_from_tiles(R.case_mbs(seed), w, h, filler)
    while len(parts) < 2:
        parts.append([m for _ in range((n + 3) // 4) for m in g.random_tile()][:n])
    for specs in parts:
        pics.append((w, h, push_out(g, specs, w, h, wide), int(g.rng.integers(1, 32))))
    return R.pack_stream(0, pics)


HANDBUILT = {  # name: (width, height, vectors beyond [-32, 31])
    "4080x64": (4080, 64, False), "64x4080": (64, 4080, False), "16x4080": (16, 4080, False),
    "4080x64_wide": (4080, 64, True), "64x4080_wide": (64, 4080, True), "16x4080_wide": (16, 4080, True),
    "4065x64_wide": (4065, 64, True),  # EDGE + WIDE_MV
}


@pytest.mark.parametrize("name", list(HANDBUILT))
def test_handbuilt_side_info_at_the_limits(name):
    w, h, wide = HANDBUILT[name]
    pictures = handbuilt_stream(w, h, wide, 11 + len(name))
    ctx = api.Context(0, 1, w, h)
    prev = None
    for t, (pic, mbs, units) in enumerate(pictures):
        if t:
            mv = mbs["u"][(mbs["flags"] & _lib.MB_INTER) != 0].view(np.int8)
            assert (np.abs(mv.astype(int)).max() > 32) == wide, t
        exp = recon_from_side_info(pic[0], mbs, units, prev)
        ctx.submit_step(*R.concat_step([(pic, mbs, units)]), _lib.OUT_RGBA)
        ctx.sync()
        y, cb, cr = ctx.read_yuv(0)
        assert np.array_equal(y, exp[0].reshape(-1)), (name, t, "Y")
        assert np.array_equal(cb, exp[1].reshape(-1)), (name, t, "Cb")
        assert np.array_equal(cr, exp[2].reshape(-1)), (name, t, "Cr")
        assert np.array_equal(ctx.read_rgba(0), O.yuv420_to_rgba(exp[0], exp[1], exp[2], w)), (name, t, "RGBA")
        prev = exp
    assert ctx.tiled_launch_count() == ctx.launch_count() == len(pictures)
    ctx.close()
