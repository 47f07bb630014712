"""numpy model of the motion fields of h263cu_decode_step_device_motion (include/h263cu.h), built from the oracle's
parse trace, and the same fields derived from h263cu_mb records.  test_motion_ref.py pins the two against each other on
the product's host parser; the GPU tests compare the device output with the oracle model."""
import numpy as np

import oracle_lib as O
from h263_rs_b200 import _lib, synth

INTRA_TYPES = (3, 4)   # the oracle's MacroblockType: Intra, IntraQ
FOURMV_TYPES = (2, 5)  # Inter4V, Inter4VQ
EXPORTED = _lib.MB_INTER | _lib.MB_FOURMV | _lib.MB_CODED
OUTSIDE = _lib.MOTION_OUTSIDE

# the parity streams (test_gpu_parity.py's STREAMS + SMALL_ALIGNED) and one with disposable P pictures: 4MV, DQUANT,
# intra-in-P, skipped macroblocks, truncated pictures, the baseline flavour, both Sorenson versions, unaligned sizes
from test_gpu_parity import SMALL_ALIGNED, STREAMS, _packets  # noqa: E402

DISPOSABLE = dict(id="cif_disposable", w=352, h=288, n=9, seed=91, pct_disposable=45, mv_mode=2, pct_fourmv=15)
CASES = STREAMS + SMALL_ALIGNED + [DISPOSABLE]


def packets_of(case):
    """(packets, decoder options) of a case"""
    if case is DISPOSABLE:
        kw = {k: v for k, v in case.items() if k not in ("id", "w", "h", "n", "seed")}
        return synth.make_stream(case["w"], case["h"], case["n"], case["seed"], **kw), 1 | 0x100
    return _packets(case)


def grid(flags, quant, mv, mb_w, mb_h):
    """Per-record fields (raster order; mv [n, 4, 2]) as the picture's grids: flags / quant [mb_h, mb_w] and
    mv [2, 2 * mb_h, 2 * mb_w], block (2X + (k & 1), 2Y + (k >> 1)) holding vector k of macroblock (X, Y)."""
    mv = np.asarray(mv, np.int16).reshape(mb_h, mb_w, 2, 2, 2)  # Y, X, k >> 1, k & 1, component
    return dict(flags=np.asarray(flags, np.uint8).reshape(mb_h, mb_w), quant=np.asarray(quant, np.uint8).reshape(mb_h, mb_w),
                mv=np.ascontiguousarray(mv.transpose(4, 0, 2, 1, 3).reshape(2, 2 * mb_h, 2 * mb_w)))


def fields_from_trace(t, pquant, mb_w, mb_h):
    """The definition on the oracle's trace of one picture: its first mb_w * mb_h macroblocks (the oracle keeps trailing
    uncoded ones beyond the capacity), INTER = not an intra type, CODED = COD 0, FOURMV = a coded 4MV type, the quantiser
    carried forward from the last coded macroblock (PQUANT before the first), intra vectors zero."""
    n = mb_w * mb_h
    ty, coded = t["mb_type"][:n], t["coded"][:n].astype(bool)
    assert len(ty) == n
    inter = ~np.isin(ty, INTRA_TYPES)
    flags = (inter * _lib.MB_INTER) | ((coded & np.isin(ty, FOURMV_TYPES)) * _lib.MB_FOURMV) | (coded * _lib.MB_CODED)
    quant = np.empty(n, np.uint8)
    q = pquant
    for k in range(n):
        if coded[k]:
            q = int(t["quant"][k])
        quant[k] = q
    mv = np.where(inter[:, None, None], t["mv"][:n], 0)
    return grid(flags, quant, mv, mb_w, mb_h)


def fields_from_records(mbs, mb_w, mb_h):
    """The definition on one picture's h263cu_mb records (the product's parse)"""
    flags = mbs["flags"] & EXPORTED
    mv = mbs["u"].view(np.int8).reshape(-1, 4, 2).astype(np.int16)
    mv = np.where((flags & _lib.MB_INTER).astype(bool)[:, None, None], mv, 0)
    return grid(flags, mbs["quant"], mv, mb_w, mb_h)


def reference_stream(packets, options=1):
    """The oracle model of every picture of a stream: a dict (width, height, mb_w, mb_h, flags, quant, mv) per picture,
    or the oracle's error code for a picture that fails."""
    st = O.OracleState(options, trace=True)
    out = []
    for pk in packets:
        try:
            st.decode_next_picture(pk)
        except O.OracleError as e:
            out.append(e.code)
            continue
        info = st.info()
        mb_w, mb_h = (info["width"] + 15) // 16, (info["height"] + 15) // 16
        f = fields_from_trace(st.trace(), info["quant"], mb_w, mb_h)
        f.update(width=info["width"], height=info["height"], mb_w=mb_w, mb_h=mb_h)
        out.append(f)
    return out


def slot(f, MBW, MBH):
    """One picture's fields placed in a slot grid of MBW x MBH macroblocks, the outside values beyond the picture"""
    flags = np.full((MBH, MBW), OUTSIDE, np.uint8)
    quant = np.zeros((MBH, MBW), np.uint8)
    mv = np.zeros((2, 2 * MBH, 2 * MBW), np.int16)
    h, w = f["flags"].shape
    flags[:h, :w], quant[:h, :w], mv[:, : 2 * h, : 2 * w] = f["flags"], f["quant"], f["mv"]
    return dict(flags=flags, quant=quant, mv=mv)
