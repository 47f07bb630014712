"""The motion-field model (motion_ref.py) on two independent parsers: the oracle's parse trace and the product's host
parser records give the same flags, quantisers and vectors on every parity stream, picture for picture."""
import numpy as np
import pytest

import motion_ref as M
from h263_rs_b200 import _lib, frontend


@pytest.mark.parametrize("case", M.CASES, ids=lambda c: c["id"])
def test_trace_model_equals_the_product_records(case):
    packets, opt = M.packets_of(case)
    ref = M.reference_stream(packets, opt)
    ps = frontend.Parser(opt)
    seen = set()
    for i, pk in enumerate(packets):
        if isinstance(ref[i], int):
            with pytest.raises(_lib.H263Error):
                ps.parse_picture(pk)
            continue
        pic, mbs, _ = ps.parse_picture(pk)
        r = ref[i]
        assert (int(pic["mb_w"][0]), int(pic["mb_h"][0])) == (r["mb_w"], r["mb_h"])
        got = M.fields_from_records(mbs, r["mb_w"], r["mb_h"])
        for k in ("flags", "quant", "mv"):
            assert np.array_equal(got[k], r[k]), (case["id"], i, k)
        f = r["flags"]
        seen.update(["inter"] if (f & _lib.MB_INTER).any() else [])
        seen.update(["intra"] if (~f & _lib.MB_INTER).any() else [])
        seen.update(["skipped"] if ((f & _lib.MB_INTER) & ~(f >> 3) & 1).any() else [])
        seen.update(["4mv"] if (f & _lib.MB_FOURMV).any() else [])
    assert "intra" in seen, case["id"]


def test_cases_cover_what_the_definition_distinguishes():
    """Across the cases: 4MV, intra macroblocks in P pictures, skipped macroblocks, quantiser changes inside a
    picture, vectors at both ends of the wrap range, truncated pictures and disposable P pictures."""
    kinds = set()
    for case in M.CASES:
        packets, opt = M.packets_of(case)
        for i, r in enumerate(M.reference_stream(packets, opt)):
            if isinstance(r, int):
                kinds.add("failed")
                continue
            f = r["flags"]
            inter, coded = (f & _lib.MB_INTER) > 0, (f & _lib.MB_CODED) > 0
            if (f & _lib.MB_FOURMV).any():
                kinds.add("4mv")
            if inter.any() and (~inter).any():
                kinds.add("intra_in_p")
            if (inter & ~coded).any():
                kinds.add("skipped")
            if len(np.unique(r["quant"])) > 1:
                kinds.add("dquant")
            if r["mv"].min() == -32 or r["mv"].max() == 31:
                kinds.add("range_edge")
            if (r["width"] % 16) or (r["height"] % 16):
                kinds.add("unaligned")
        if case is M.DISPOSABLE:
            types = [int(frontend.peek_picture(p)["pic_type"]) for p in packets]
            assert types.count(_lib.PIC_DISPOSABLE_P) >= 2
    assert {"4mv", "intra_in_p", "skipped", "dquant", "range_edge", "unaligned"} <= kinds, kinds


def test_slot_placement():
    f = M.grid(np.arange(6) % 16, np.arange(6) + 1, np.arange(48).reshape(6, 4, 2), 3, 2)
    s = M.slot(f, 4, 3)
    assert s["flags"].shape == (3, 4) and s["mv"].shape == (2, 6, 8)
    assert (s["flags"][2] == M.OUTSIDE).all() and (s["flags"][:, 3] == M.OUTSIDE).all()
    assert (s["quant"][2] == 0).all() and (s["mv"][:, 4:] == 0).all() and (s["mv"][:, :, 6:] == 0).all()
    # block (2X + (k & 1), 2Y + (k >> 1)) holds vector k of macroblock (X, Y): macroblock (1, 1) is record 4
    for k in range(4):
        assert tuple(s["mv"][:, 2 + (k >> 1), 2 + (k & 1)]) == (32 + 2 * k, 33 + 2 * k)
