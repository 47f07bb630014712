"""CPU checks of the hand-built edge cases (recon_cases.py) that test_gpu_recon_edges.py runs on the device: every edge
the kernels' bookkeeping has must occur in the steps, as the scheduling model of recon_cases computes it from the
records alone; the records must be ones the library accepts; the saturation pictures must pin their predictions."""
import numpy as np
import pytest

import oracle_lib as O
import recon_cases as R
from helpers import recon_from_side_info
from h263_rs_b200 import _lib, frontend


@pytest.fixture(scope="module")
def streams():
    return R.edge_streams()


# the streams every instantiation runs (test_gpu_recon_edges.py); the CIF motion stream only fits the larger contexts
BLOCK_IDS = [0, 1, 2, 3]


def test_every_block_structure_edge_occurs(streams):
    f = R.features(R.steps_of(streams, BLOCK_IDS))
    need = set()
    # every zig-zag position as a lone coefficient: inter 0..63, intra 1..63 beside the DC, luma and chroma
    for chroma in (False, True):
        need |= {("lone", True, chroma, k) for k in range(64)} | {("lone", False, chroma, k) for k in range(1, 64)}
        # Full with every row-occupancy mask a Full block can have (mask 0 is the Dc / Zero classes)
        need |= {("full_rows", chroma, mask) for mask in range(1, 256)}
        need |= {("cls", "dc", True, chroma)}
        need |= {("cls", c, inter, chroma) for c in ("vert", "full") for inter in (False, True)}
    # classes: intra DC only (codes 1, 254 and 255 -> 1024), an inter coefficient on index 0, Vert with and without the
    # intra DC, Horiz (row 0 only) inter and intra
    need |= {("dc_only_intra", c) for c in (1, 254, 255)} | {("dc_inter_index0",), ("vert", True), ("vert", False),
                                                             ("horiz", True), ("horiz", False)}
    # passes: mixed sort keys, Vert beside non-Vert, short beside long slots, last passes of 1..3 slots
    need |= {("pass_keys", k) for k in ((0, 1), (1, 2), (0, 2), (0, 1, 2))}
    need |= {("pass_vert_mix",), ("pass_long_short",)} | {("last_pass_size", n) for n in (1, 2, 3)}
    # tiles: 0, 1, 24 coded slots; event totals around the round and the chunk; a tile across two pictures that differ
    # in type and QP
    need |= {("tile_slots", n) for n in (0, 1, 24)} | {("tile_events", n) for n in R.TILE_EVENT_TOTALS}
    need |= {("tile_spans_pictures",)}
    # slots on / across a round, ending at event 64, a 64-event inter slot in its own chunk (first in its tile and
    # after other slots), an intra slot of 63 AC events
    need |= {("slot_on_round",), ("slot_straddles_round",), ("slot_ends_at_64",), ("own_chunk_64", "first"),
             ("own_chunk_64", "after"), ("intra_63",)}
    # overflow: the last event on 63 (kept) or on 64 (dropped); run 63 first (intra drops, inter keeps); in a slot that
    # straddles a round, in a later chunk; an intra overflow drops the DC
    need |= {("last_at_63", i) for i in (False, True)} | {("overflow_on_64", i) for i in (False, True)}
    need |= {("first_run_63", False, True), ("first_run_63", True, False), ("overflow_straddles_round",),
             ("overflow_in_later_chunk",), ("overflow_drops_intra_dc",)}
    # values: every QP, both sides of the narrow / wide level boundary, the +-2048 clamp both ways
    need |= {("qp", q) for q in range(1, 32)} | {("level", v) for v in R.LEVELS} | {("clamp", 1), ("clamp", -1)}
    missing = sorted(need - f, key=str)
    assert not missing, missing[:20]


def test_every_vector_and_chroma_residue_occurs(streams):
    f = R.features(R.steps_of(streams, [4]))
    need = {("mv", x, y) for x in range(-32, 32) for y in range(-32, 32)}
    need |= {("chroma_residue", a, r) for a in "xy" for r in range(16)}
    missing = sorted(need - f)
    assert not missing, missing[:20]


def test_wide_vector_streams_leave_the_range(streams):
    for s in (7, 8):
        mv = np.concatenate([m["u"].view(np.int8)[(m["flags"] & _lib.MB_INTER) != 0] for _, m, _ in streams[s]])
        assert np.abs(mv.astype(int)).max() > 32 and len(streams[s]) >= 2


def test_records_are_ones_the_library_accepts(streams):
    """validate_side_info's counts rule (include/h263cu.h): <= 64 events per block, <= 63 intra, none under code 0"""
    for pics in streams.values():
        for pic, mbs, units in pics:
            inter = (mbs["flags"] & _lib.MB_INTER) != 0
            nev = mbs["nev"].astype(int)
            assert (nev <= 64).all() and (nev[~inter] <= 63).all()
            assert not ((mbs["u"][~inter, :6] == 0) & (nev[~inter] > 0)).any()
            assert int(pic["n_event_units"][0]) == len(units)


def test_saturation_pictures_pin_their_predictions(streams):
    """Stream 3: after its first P picture the left / right halves of the macroblock pairs sit at 255 / 0 in every
    plane, and the next P picture puts transformed residuals of both signs on them with zero vectors."""
    pics = streams[3]
    prev = None
    out = []
    for pic, mbs, units in pics:
        prev = recon_from_side_info(pic[0], mbs, units, prev)
        out.append(prev)
    y, cb, cr = out[1]
    for q, v in enumerate((255, 0, 255, 0)):
        assert (y[:, 16 * q : 16 * q + 16] == v).all() and (cb[:, 8 * q : 8 * q + 8] == v).all() and (cr[:, 8 * q : 8 * q + 8] == v).all()
    pic, mbs, units = pics[2]
    signs = set()
    for q, m in enumerate(mbs):
        assert (m["u"] == 0).all() and m["flags"] & _lib.MB_INTER
        for ev in frontend.decode_events(m, units):
            cls, coefs = O.inverse_rle(None, [r for r, _ in ev], [l for _, l in ev], int(m["quant"]))
            assert cls in (2, 3, 4)  # a transform: Horiz, Vert or Full
            r = O.idct_block(cls, coefs, np.full((8, 8), 128, np.uint8)).astype(int) - 128
            if (r > 0).any():
                signs.add((q % 2, 1))
            if (r < 0).any():
                signs.add((q % 2, -1))
    assert signs == {(0, 1), (0, -1), (1, 1), (1, -1)}
