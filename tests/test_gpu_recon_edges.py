"""GPU parity on hand-built side info that reaches the kernels' structural edges by construction (recon_cases.py; the
CPU test test_recon_cases.py asserts that every edge occurs): every instantiation of recon_tile_kernel, the generic
recon_mb_kernel, with and without RGBA, bit for bit against helpers.recon_from_side_info + the oracle's BT.601; and
the two in-step deblocking kernels (deblock_rgba_tile_kernel for aligned steps, deblock_rgba_kernel otherwise) on
pictures of flat 8x8 blocks whose edges take every step in -253..253, at every filter strength."""
import numpy as np
import pytest

import oracle_lib as O
import recon_cases as R
from helpers import recon_from_side_info
from h263_rs_b200 import _lib, api

pytestmark = pytest.mark.gpu
N_STREAMS = 9


@pytest.fixture(scope="module")
def streams():
    return R.edge_streams()


@pytest.fixture(scope="module")
def expected(streams):
    cache = {}

    def get(s):
        if s not in cache:
            out, prev = [], None
            for pic, mbs, units in streams[s]:
                prev = recon_from_side_info(pic[0], mbs, units, prev)
                out.append(prev)
            cache[s] = out
        return cache[s]

    return get


def _kernel(monkeypatch, force):
    if force:
        monkeypatch.setenv("H263CU_KERNEL", force)
    else:
        monkeypatch.delenv("H263CU_KERNEL", raising=False)


def _check_picture(ctx, s, exp, w, rgba, tag):
    y, cb, cr = ctx.read_yuv(s)
    assert np.array_equal(y, exp[0].reshape(-1)), tag + ("Y",)
    assert np.array_equal(cb, exp[1].reshape(-1)), tag + ("Cb",)
    assert np.array_equal(cr, exp[2].reshape(-1)), tag + ("Cr",)
    if rgba is not None:
        assert np.array_equal(ctx.read_rgba(s), rgba), tag + ("RGBA",)


# (context size, streams): the context's pitches select the tiled instantiation (recon_tile.cu, launch_recon_tile);
# an unaligned picture in a step selects EDGE, a vector beyond [-32, 31] WIDE_MV
INSTANTIATIONS = {
    "cif": ((352, 288), [0, 1, 2, 3, 4]),
    "qcif": ((176, 144), [0, 1, 2, 3]),
    "4cif": ((704, 576), [0, 1, 2, 3, 4]),
    "generic_aligned": ((128, 96), [0, 1, 2, 3]),
    "edge": ((128, 96), [0, 1, 2, 3, 5, 6]),
    "wide_mv": ((128, 96), [0, 1, 2, 3, 7]),
    "wide_mv_edge": ((128, 96), [0, 1, 2, 3, 7, 8]),
}


@pytest.mark.parametrize("out_flags", [_lib.OUT_RGBA, 0], ids=["rgba", "planes"])
@pytest.mark.parametrize("name", list(INSTANTIATIONS))
def test_tiled_kernel_on_every_edge(monkeypatch, streams, expected, name, out_flags):
    (cw, ch), ids = INSTANTIATIONS[name]
    _kernel(monkeypatch, None)
    ctx = api.Context(0, N_STREAMS, cw, ch)
    steps = R.steps_of(streams, ids)
    for t, ((pics, mbs, units), members) in enumerate(steps):
        ctx.submit_step(pics, mbs, units, out_flags)
        ctx.sync()
        for s, k in members:
            exp = expected(s)[k]
            w = exp[0].shape[1]
            rgba = O.yuv420_to_rgba(exp[0], exp[1], exp[2], w) if out_flags else None
            _check_picture(ctx, s, exp, w, rgba, (name, t, s, k))
    assert ctx.tiled_launch_count() == len(steps) == ctx.launch_count()
    ctx.close()


@pytest.mark.parametrize("out_flags", [_lib.OUT_RGBA, 0], ids=["rgba", "planes"])
def test_generic_kernel_on_every_edge(monkeypatch, streams, expected, out_flags):
    """recon_mb_kernel (H263CU_KERNEL=mb) on every stream side by side: aligned, unaligned and wide-vector pictures"""
    _kernel(monkeypatch, "mb")
    ctx = api.Context(0, N_STREAMS, 352, 288)
    steps = R.steps_of(streams, list(range(N_STREAMS)))
    for t, ((pics, mbs, units), members) in enumerate(steps):
        ctx.submit_step(pics, mbs, units, out_flags)
        ctx.sync()
        for s, k in members:
            exp = expected(s)[k]
            w = exp[0].shape[1]
            rgba = O.yuv420_to_rgba(exp[0], exp[1], exp[2], w) if out_flags else None
            _check_picture(ctx, s, exp, w, rgba, ("mb", t, s, k))
    assert ctx.tiled_launch_count() == 0 and ctx.launch_count() == len(steps)
    ctx.close()


# ------------------------------------------------------------------------------------------ deblocking
STRENGTH_QUANT = {}
for _q, _s in enumerate(api.QUANT_TO_STRENGTH):
    if _s and _s not in STRENGTH_QUANT:
        STRENGTH_QUANT[_s] = _q
# aligned: chroma 8 wide (narrower than the 10 a vertical chroma edge needs), single-row / single-column grids;
# unaligned: odd luma and chroma widths, chroma 5..10 wide, partial macroblocks
ALIGNED = [(16, 16), (32, 16), (16, 48), (48, 32), (64, 48), (176, 144)]
UNALIGNED = [(17, 9), (15, 31), (19, 35), (21, 17), (45, 27), (100, 70), (161, 99)]


def _flat_picture(rng, w, h, pquant, stream, noise):
    """An intra picture of DC-only blocks: each 8x8 block is flat at its INTRADC level (codes 1..255: 8..2032 / 8 and
    128), so neighbouring blocks step by anything in -253..253.  With `noise`, a small coefficient (QP 1..2, level +-1)
    on top of most blocks."""
    n = ((w + 15) // 16) * ((h + 15) // 16)
    specs = []
    for _ in range(n):
        codes = [int(c) for c in rng.integers(1, 256, 6)]
        blocks = [[] for _ in range(6)]
        if noise:
            for b in range(6):
                if rng.random() < 0.8:
                    blocks[b] = R.events_at([int(rng.integers(1, 64))], [int(rng.choice([-1, 1]))], False)
        specs.append(R.mb_spec(False, int(rng.integers(1, 3)), blocks, codes))
    return R.pack_picture(w, h, specs, pquant=pquant, stream=stream)


@pytest.mark.parametrize("noise", [False, True], ids=["flat", "noisy"])
@pytest.mark.parametrize("kind", ["aligned_tile", "aligned_mb", "unaligned"])
def test_in_step_deblocking_at_every_strength(monkeypatch, kind, noise):
    """OUT_RGBA | OUT_DEBLOCK: RGBA = BT.601 of deblock(plane, width, QUANT_TO_STRENGTH[pquant]) per plane (deblock.rs:
    305-315, the SIMD body's floor and the scalar tails' truncation), the planes stay un-deblocked.  Aligned steps run
    the register-resident kernel; steps with an unaligned picture, or H263CU_KERNEL=mb, run the generic one."""
    sizes = UNALIGNED if kind == "unaligned" else ALIGNED
    _kernel(monkeypatch, "mb" if kind == "aligned_mb" else None)
    rng = np.random.default_rng(len(sizes) * 10 + noise)
    ctx = api.Context(0, len(sizes), 176, 144)
    steps = []
    for strength in range(1, 13):
        pics = [_flat_picture(rng, w, h, STRENGTH_QUANT[strength], s, noise) for s, (w, h) in enumerate(sizes)]
        steps.append((strength, pics))
    # steps with the small pictures' strengths shuffled against each other
    for t in range(3):
        pics = [_flat_picture(rng, w, h, int(rng.integers(1, 32)), s, noise) for s, (w, h) in enumerate(sizes)]
        steps.append((None, pics))
    seen = set()
    for strength, pictures in steps:
        pics, mbs, units = R.concat_step(pictures)
        ctx.submit_step(pics, mbs, units, _lib.OUT_RGBA | _lib.OUT_DEBLOCK)
        ctx.sync()
        for s, (w, h) in enumerate(sizes):
            pic, m, u = pictures[s]
            exp = recon_from_side_info(pic[0], m, u)
            st = api.QUANT_TO_STRENGTH[int(pic["pquant"][0])]
            seen.add(st)
            cw = (w + 1) // 2
            dy, dcb, dcr = O.deblock(exp[0], w, st), O.deblock(exp[1], cw, st), O.deblock(exp[2], cw, st)
            _check_picture(ctx, s, exp, w, O.yuv420_to_rgba(dy, dcb, dcr, w), (kind, noise, strength, w, h))
            if strength is not None and w >= 100:
                assert not np.array_equal(dy, exp[0].reshape(-1)), (w, h, strength)  # the filter did something
    assert seen >= set(range(1, 13))
    assert ctx.tiled_launch_count() == (0 if kind == "aligned_mb" else len(steps))
    ctx.close()
