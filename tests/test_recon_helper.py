"""The reconstruction helper the hand-built GPU tests trust (helpers.recon_from_side_info), pinned on the CPU: on the
side info the product's parser produces for the parity streams -- 4MV, vectors across the picture border, dquant,
escapes, dropped (zig-zag overflow) blocks, truncated pictures and every unaligned size there -- it must give the
oracle's planes picture for picture."""
import numpy as np
import pytest

from helpers import oracle_decode_stream, recon_from_side_info
from test_gpu_parity import SMALL_ALIGNED, STREAMS, _packets
from h263_rs_b200 import _lib, frontend


@pytest.mark.parametrize("case", STREAMS + SMALL_ALIGNED, ids=lambda c: c["id"])
def test_recon_from_side_info_equals_the_oracle(case):
    packets, opt = _packets(case)
    ref = oracle_decode_stream(packets, opt)
    ps = frontend.Parser(opt)
    prev = None
    n_ok = 0
    for i, pk in enumerate(packets):
        if isinstance(ref[i], int):
            with pytest.raises(_lib.H263Error):
                ps.parse_picture(pk)
            continue
        pic, mbs, ev = ps.parse_picture(pk)
        w, h = int(pic["width"][0]), int(pic["height"][0])
        has_inter = bool((mbs["flags"] & _lib.MB_INTER).any())
        exp = recon_from_side_info(pic[0], mbs, ev, prev if has_inter else None)
        assert np.array_equal(exp[0].reshape(-1), ref[i]["y"]), (case["id"], i, "Y")
        assert np.array_equal(exp[1].reshape(-1), ref[i]["cb"]), (case["id"], i, "Cb")
        assert np.array_equal(exp[2].reshape(-1), ref[i]["cr"]), (case["id"], i, "Cr")
        assert exp[0].shape == (h, w) and exp[1].shape == ((h + 1) // 2, (w + 1) // 2)
        prev = exp
        n_ok += 1
    assert n_ok >= 2, case["id"]
