"""Shared helpers for the parity tests."""
import numpy as np

import oracle_lib as O
from h263_rs_b200 import _lib, frontend, synth

INTER_TYPES = (0, 1, 2, 5)


def oracle_decode_stream(packets, options=1, deblock=False):
    """Reference path on the CPU: decode -> [deblock] -> RGBA, per picture.
    Returns a list of dicts (or the error code for pictures that fail)."""
    st = O.OracleState(options)
    out = []
    for pk in packets:
        try:
            st.decode_next_picture(pk)
        except O.OracleError as e:
            out.append(e.code)
            continue
        info = st.info()
        y, cb, cr = st.yuv()
        w = info["width"]
        cw = (w + 1) // 2
        if deblock:
            s = O.lib().orc_quant_to_strength(info["quant"])
            dy, dcb, dcr = O.deblock(y, w, s), O.deblock(cb, cw, s), O.deblock(cr, cw, s)
            rgba = O.yuv420_to_rgba(dy, dcb, dcr, w)
        else:
            rgba = O.yuv420_to_rgba(y, cb, cr, w)
        out.append(dict(info=info, y=y, cb=cb, cr=cr, rgba=rgba))
    return out


def weighted_sum(a):
    a = np.ascontiguousarray(a, np.uint8).reshape(-1).astype(np.uint64)
    i = np.arange(a.size, dtype=np.uint64)
    w = ((i * np.uint64(2654435761)) & np.uint64(0xFFFFFFFF)) | np.uint64(1)
    with np.errstate(over="ignore"):
        return int(((a + np.uint64(1)) * w).sum(dtype=np.uint64))


def compare_parse_with_oracle(packets, options=1):
    """Product parser vs oracle parse trace, picture by picture. Returns (#mbs, #events, #errors)."""
    st = O.OracleState(options, trace=True)
    ps = frontend.Parser(options)
    nmb = nev = nerr = 0
    for i, p in enumerate(packets):
        oerr = perr = 0
        try:
            st.decode_next_picture(p)
        except O.OracleError as e:
            oerr = e.code
        try:
            pic, mbs, ev = ps.parse_picture(p)
        except _lib.H263Error as e:
            perr = -e.code
        if oerr == 100:
            assert perr == 104, (i, oerr, perr)
        else:
            assert oerr == perr, (i, oerr, perr)
        if oerr:
            nerr += 1
            continue
        t = st.trace()
        info = st.info()
        assert (info["width"], info["height"], info["quant"], info["tr"]) == (
            pic["width"][0], pic["height"][0], pic["pquant"][0], pic["temporal_reference"][0])
        # The oracle, like the reference, keeps trailing COD=1 macroblocks beyond the picture's capacity (harmless:
        # gather writes nothing for them, state.rs:419-427); the product stops at capacity.  Compare the first
        # `capacity` records and require the extras to be uncoded inter macroblocks.
        assert len(mbs) <= len(t["mb_type"])
        for k in range(len(mbs), len(t["mb_type"])):
            assert t["mb_type"][k] in INTER_TYPES and not t["coded"][k], (i, k)
        eoff = 0
        for k in range(len(mbs)):
            m = mbs[k]
            inter = t["mb_type"][k] in INTER_TYPES
            assert bool(m["flags"] & 1) == inter, (i, k)
            if t["coded"][k]:
                assert m["quant"] == t["quant"][k], (i, k)
            if inter:
                assert np.array_equal(m["u"].view(np.int8).reshape(4, 2), t["mv"][k]), (i, k)
            blocks = frontend.decode_events(m, ev)
            for b in range(6):
                ne = int(t["nev"][k][b])
                runs, lv = t["run"][eoff : eoff + ne], t["level"][eoff : eoff + ne]
                eoff += ne
                idx = 0 if inter else 1
                ovf = False
                for r in runs:
                    idx += int(r)
                    ovf |= idx >= 64
                    idx += 1
                if ovf:  # dropped block (rle.rs:125-127)
                    assert blocks[b] == []
                    if not inter:
                        assert m["u"][b] == 0
                else:
                    assert blocks[b] == [(int(a), int(c)) for a, c in zip(runs, lv)], (i, k, b)
                    if not inter:
                        assert m["u"][b] == t["intradc"][k][b]
                nev += ne
        nmb += len(mbs)
    return nmb, nev, nerr


def recon_from_side_info(pic, mbs, events, ref=None):
    """The reference's reconstruction tail (state.rs:419-485) on one picture's side info, put together from the
    oracle's exported pieces: gather_block (gather.rs:47-126) per inter block with the chroma vector of
    gather.rs:182, then inverse_rle (rle.rs:82-172) + idct_channel on one block (idct.rs:82-201).  Works on
    hand-built records, so it checks what no bitstream can reach (vectors beyond the parser's range, escape levels
    at the i16-wrap boundary).  Any picture size: planes are the true size ((w + 1) // 2 chroma columns, state.rs and
    picture.rs:39-58), gather_block cuts the blocks of the last macroblock column / row to the picture and its
    read_sample clamps at the true edge, and the transform of an edge block runs on an 8x8 window of which only the
    in-picture part is kept (idct_channel's xs / ys, idct.rs:91-95).  `ref` = (y, cb, cr) planes or None.
    Returns (y, cb, cr) as 2-D arrays."""
    w, h = int(pic["width"]), int(pic["height"])
    cw, ch = (w + 1) // 2, (h + 1) // 2
    planes = [np.zeros((h, w), np.uint8), np.zeros((ch, cw), np.uint8), np.zeros((ch, cw), np.uint8)]
    L = O.lib()
    if ref is not None:
        ref = [np.asarray(ref[0]).reshape(h, w), np.asarray(ref[1]).reshape(ch, cw), np.asarray(ref[2]).reshape(ch, cw)]
    for m in mbs:
        mbx, mby = int(m["mbx"]), int(m["mby"])
        inter = bool(m["flags"] & _lib.MB_INTER)
        if inter:
            assert ref is not None
            mv = m["u"].view(np.int8).reshape(4, 2).astype(int)
            for b in range(4):
                planes[0] = O.gather_block(ref[0], (mbx * 16 + (b & 1) * 8, mby * 16 + (b >> 1) * 8),
                                           (int(mv[b][0]), int(mv[b][1])), planes[0])
            cmv = (L.orc_average_sum_of_mvs(int(mv[:, 0].sum())), L.orc_average_sum_of_mvs(int(mv[:, 1].sum())))
            for p in (1, 2):
                planes[p] = O.gather_block(ref[p], (mbx * 8, mby * 8), cmv, planes[p])
        blocks = frontend.decode_events(m, events, int(pic["first_event"]))
        for b in range(6):
            dc = None
            if not inter:
                dc = int(m["u"][b])
                if dc == 0:
                    continue  # dropped block (zig-zag overflow): stays Zero, rle.rs:125-127
            runs = [r for r, _ in blocks[b]]
            levels = [l for _, l in blocks[b]]
            cls, coefs = O.inverse_rle(dc, runs, levels, int(m["quant"]))
            if b < 4:
                pl, x0, y0 = planes[0], mbx * 16 + (b & 1) * 8, mby * 16 + (b >> 1) * 8
            else:
                pl, x0, y0 = planes[b - 3], mbx * 8, mby * 8
            ys, xs = min(8, pl.shape[0] - y0), min(8, pl.shape[1] - x0)
            if ys <= 0 or xs <= 0:
                continue  # a block of the last macroblock column / row that lies wholly outside the picture
            win = np.zeros((8, 8), np.uint8)
            win[:ys, :xs] = pl[y0 : y0 + ys, x0 : x0 + xs]
            pl[y0 : y0 + ys, x0 : x0 + xs] = O.idct_block(cls, coefs, win)[:ys, :xs]
    return planes
