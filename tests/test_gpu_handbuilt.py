"""GPU parity on HAND-BUILT side info against the oracle's exported pieces (inverse_rle, idct_block, gather_block):
what no generated bitstream reaches -- escape levels whose dequantisation wraps in i16 (rle.rs:130-133), level -1024
(block.rs:716 is dead code: the reference accepts it), vectors beyond the range halfpel_decode produces
(gather.rs:16-31 clamps them per sample)."""
import numpy as np
import pytest

import oracle_lib as O
from helpers import oracle_decode_stream, recon_from_side_info
from recon_cases import mb_spec, pack_picture
from h263_rs_b200 import _lib, api, frontend, synth

pytestmark = pytest.mark.gpu
PICFLAG_HAS_INTER, PICFLAG_MV_IN_RANGE = 2, 4


def _build_picture(rng, w, h, inter, levels_pool, qp_range, stream=0):
    """One picture of hand-built records (recon_cases.pack_picture's layout): every macroblock coded, 1..6 events per
    coded block."""
    specs = []
    for k in range((w // 16) * (h // 16)):
        quant = int(rng.integers(qp_range[0], qp_range[1] + 1))
        blocks = []
        for b in range(6):
            ev = []
            if rng.random() < 0.8:
                idx = 0 if inter else 1
                for _ in range(int(rng.integers(1, 7))):
                    run = int(rng.integers(0, 9))
                    if idx + run >= 64:
                        break
                    ev.append((run, int(rng.choice(levels_pool))))
                    idx += run + 1
            blocks.append(ev)
        codes = None if inter else [int(c) for c in rng.choice([1, 2, 64, 127, 129, 200, 254, 255], 6)]
        specs.append(mb_spec(inter, quant, blocks, codes))
    return pack_picture(w, h, specs, pquant=8, stream=stream)


@pytest.mark.parametrize("w,h", [(64, 48), (352, 288)])
def test_escape_levels_wrap_in_i16_on_the_device(w, h):
    """|level| 529..1023 and -1024 at QP 24..31: QP * (2|level| + 1) exceeds 2^15, and the reference's release build
    wraps (rle.rs:130-133) before it clamps.  An I picture and a P picture (zero vectors, residual on top of the
    prediction) of hand-built wide events, compared with orc_inverse_rle + orc_idct_block block by block."""
    rng = np.random.default_rng(w)
    pool = [-1024, -1023, -1000, -700, -529, -513, -512, -511, -3, -1, 1, 2, 17, 511, 512, 529, 600, 682, 683, 900, 1023]
    ctx = api.Context(0, 1, w, h)
    ref = None
    for t, inter in enumerate([False, True, True]):
        pic, mbs, ev = _build_picture(rng, w, h, inter, pool, (24, 31) if t < 2 else (1, 31))
        assert (mbs["flags"] & _lib.MB_WIDE).any()
        exp = recon_from_side_info(pic[0], mbs, ev, ref)
        ctx.submit_step(pic, mbs, ev, _lib.OUT_RGBA)
        ctx.sync()
        y, cb, cr = ctx.read_yuv(0)
        assert np.array_equal(y, exp[0].reshape(-1)), (t, "Y")
        assert np.array_equal(cb, exp[1].reshape(-1)), (t, "Cb")
        assert np.array_equal(cr, exp[2].reshape(-1)), (t, "Cr")
        assert np.array_equal(ctx.read_rgba(0), O.yuv420_to_rgba(exp[0], exp[1], exp[2], w)), (t, "RGBA")
        ref = exp
    assert ctx.tiled_launch_count() == 3
    ctx.close()


def test_wrap_actually_happens_in_the_oracle():
    """Guard for the test above: at QP 31, level 600 dequantises to a value that differs from the unwrapped formula."""
    cls, coefs = O.inverse_rle(None, [0], [600], 31)
    assert coefs[0][0] != min(31 * (2 * 600 + 1), 2047)


@pytest.mark.parametrize("w,h", [(352, 288), (64, 48)])
def test_vectors_beyond_the_range_against_gather_block(w, h):
    """Hand-edited vectors up to +-60 pixels (the parser never emits them, mvd_pred.rs:70-117): the picture loses
    H263CU_PICFLAG_MV_IN_RANGE, the tiled kernel runs its WIDE_MV instantiation, and every block must match
    orc_gather_block (read_sample's clamp, gather.rs:16-31, 47-126) + the residual path."""
    packets = synth.make_stream(w, h, 4, 4242 + w, mv_mode=2, pct_fourmv=25)
    ref_stream = oracle_decode_stream(packets)
    ctx = api.Context(0, 1, w, h)
    ps = frontend.Parser(1)
    rng = np.random.default_rng(9)
    prev = None
    for t, pk in enumerate(packets):
        pic, mbs, ev = ps.parse_picture(pk)
        if t > 0:
            inter = np.flatnonzero((mbs["flags"] & _lib.MB_INTER) != 0)
            idx = rng.choice(inter, size=max(1, len(inter) // 3), replace=False)
            mbs["u"][idx] = rng.integers(-120, 121, size=(len(idx), 8)).astype(np.int8).view(np.uint8)
            pic["flags"] &= np.uint8(~PICFLAG_MV_IN_RANGE & 0xFF)
            exp = recon_from_side_info(pic[0], mbs, ev, prev)
        else:
            exp = [ref_stream[0]["y"].reshape(h, w), ref_stream[0]["cb"].reshape(h // 2, w // 2), ref_stream[0]["cr"].reshape(h // 2, w // 2)]
        ctx.submit_step(pic, mbs, ev, _lib.OUT_RGBA)
        ctx.sync()
        y, cb, cr = ctx.read_yuv(0)
        assert np.array_equal(y, exp[0].reshape(-1)), (t, "Y")
        assert np.array_equal(cb, exp[1].reshape(-1)) and np.array_equal(cr, exp[2].reshape(-1)), (t, "chroma")
        assert np.array_equal(ctx.read_rgba(0), O.yuv420_to_rgba(exp[0], exp[1], exp[2], w)), (t, "RGBA")
        prev = exp
    assert ctx.tiled_launch_count() == ctx.launch_count()
    ctx.close()
