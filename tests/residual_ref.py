"""numpy model of the prediction residuals of h263cu_decode_step_device_residual (include/h263cu.h), built per stream
with the oracle: its decoded planes, its reference planes (the last non-disposable picture) and, from its parse trace,
each macroblock's type and vectors, with the prediction assembled block by block with the oracle's own gather_block
and average_sum_of_mvs.  test_residual_ref.py pins the model; the GPU tests compare the device output with it."""
import ctypes as C

import numpy as np

import oracle_lib as O
from motion_ref import CASES, INTRA_TYPES, packets_of  # noqa: F401  (the cases of the motion model)

ORC_OPT_DECODE_DISPOSABLE, ORC_PIC_DISPOSABLE_P = 0x100, 2  # oracle/h263_oracle.h


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _lib():
    L = O.lib()
    L.orc_average_sum_of_mvs.argtypes = [C.c_int]
    L.orc_average_sum_of_mvs.restype = C.c_int
    return L


def prediction(ref, inter, mv, w, h):
    """gather (gather.rs:140-204) of one picture: ref = (y, cb, cr) planes of the reference ([h, w], [ch, cw] uint8),
    inter [n] bool and mv [n, 4, 2] per macroblock (raster order) -> the pred planes (uint8, 0 outside INTER
    macroblocks), and whether some block's source window leaves the picture."""
    L = _lib()
    cw, ch = (w + 1) // 2, (h + 1) // 2
    mb_w = (w + 15) // 16
    pred = [np.zeros((h, w), np.uint8), np.zeros((ch, cw), np.uint8), np.zeros((ch, cw), np.uint8)]
    src = [np.ascontiguousarray(p, np.uint8) for p in ref]
    leaves = False
    for i in np.flatnonzero(inter):
        X, Y = int(i) % mb_w, int(i) // mb_w
        v = [(int(mv[i, k, 0]), int(mv[i, k, 1])) for k in range(4)]
        for k in range(4):
            x, y = 16 * X + 8 * (k & 1), 16 * Y + 8 * (k >> 1)
            if x < w and y < h:
                L.orc_gather_block(_ptr(src[0]), w, h, x, y, v[k][0], v[k][1], _ptr(pred[0]))
                sx, sy = x + (v[k][0] >> 1), y + (v[k][1] >> 1)
                leaves |= sx < 0 or sy < 0 or sx + 8 + (v[k][0] & 1) > w or sy + 8 + (v[k][1] & 1) > h
        c = (L.orc_average_sum_of_mvs(sum(a for a, _ in v)), L.orc_average_sum_of_mvs(sum(b for _, b in v)))
        for p in (1, 2):
            L.orc_gather_block(_ptr(src[p]), cw, ch, 8 * X, 8 * Y, c[0], c[1], _ptr(pred[p]))
    return pred, leaves


def reference_stream(packets, options=1):
    """The model of every picture of a stream: a dict per picture (width, height, cur and pred planes as uint8,
    y / cb / cr residual planes as int16, inter [mb_h, mb_w], mv [n, 4, 2], coded [n], nev [n, 6], leaves, disposable) or the
    oracle's
    error code for a picture that fails."""
    st = O.OracleState(options, trace=True)
    ref = None
    out = []
    for pk in packets:
        try:
            st.decode_next_picture(pk)
        except O.OracleError as e:
            out.append(e.code)
            continue
        info = st.info()
        w, h = info["width"], info["height"]
        cw, ch = (w + 1) // 2, (h + 1) // 2
        mb_w, mb_h = (w + 15) // 16, (h + 15) // 16
        n = mb_w * mb_h
        t = st.trace()
        inter = ~np.isin(t["mb_type"][:n], INTRA_TYPES)
        mv = t["mv"][:n]
        y, cb, cr = st.yuv()
        cur = [y.reshape(h, w), cb.reshape(ch, cw), cr.reshape(ch, cw)]
        if inter.any():
            assert ref is not None and ref[0].shape == (h, w)
            pred, leaves = prediction(ref, inter, mv, w, h)
        else:
            pred, leaves = [np.zeros_like(p) for p in cur], False
        res = [c.astype(np.int16) - p.astype(np.int16) for c, p in zip(cur, pred)]
        # the next picture's prediction source: the last picture, unless it is disposable and decoded as one
        disposable = bool(options & ORC_OPT_DECODE_DISPOSABLE) and info["ptype"] == ORC_PIC_DISPOSABLE_P
        out.append(dict(width=w, height=h, cur=cur, pred=pred, y=res[0], cb=res[1], cr=res[2], inter=inter.reshape(mb_h, mb_w),
                        mv=mv, coded=t["coded"][:n].astype(bool), nev=t["nev"][:n], leaves=leaves, disposable=disposable))
        if not disposable:
            ref = cur
    return out


def slot(r, W, H):
    """One picture's residual planes placed in a slot of W x H luma samples (ceil(W/2) x ceil(H/2) chroma), 0 beyond the
    picture: a dict y, cb, cr"""
    cW, cH = (W + 1) // 2, (H + 1) // 2
    out = dict(y=np.zeros((H, W), np.int16), cb=np.zeros((cH, cW), np.int16), cr=np.zeros((cH, cW), np.int16))
    for k in ("y", "cb", "cr"):
        hh, ww = r[k].shape
        out[k][:hh, :ww] = r[k]
    return out
