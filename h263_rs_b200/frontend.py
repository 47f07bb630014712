"""Host front end: serial bitstream parse into compact side info (ctypes front for
h263cu_parser_* / h263cu_parse_step).  One Parser per stream."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import Mb, Pic, check

MB_DTYPE = np.dtype(
    {
        "names": ["ev_off", "pic", "mbx", "mby", "flags", "quant", "nev", "u"],
        "formats": ["<u4", "<u2", "u1", "u1", "u1", "u1", ("u1", 6), ("u1", 8)],
        "offsets": [0, 4, 6, 7, 8, 9, 10, 16],
        "itemsize": 24,
    }
)
PIC_DTYPE = np.dtype(
    {
        "names": ["stream", "width", "height", "mb_w", "mb_h", "pic_type", "pquant", "flags", "version",
                  "temporal_reference", "first_mb", "n_mbs", "first_event", "n_event_units"],
        "formats": ["<u4", "<u2", "<u2", "u1", "u1", "u1", "u1", "u1", "u1", "<u2", "<u4", "<u4", "<u4", "<u4"],
        "offsets": [0, 4, 6, 8, 9, 10, 11, 12, 13, 14, 16, 20, 24, 28],
        "itemsize": 32,
    }
)


class Parser:
    """Per-stream parser state (the host half of h263::H263State)."""

    def __init__(self, options=_lib.OPT_SORENSON):
        self.L = _lib.lib()
        self.options = options
        self.h = self.L.h263cu_parser_create(options)
        if not self.h:
            raise MemoryError

    def __del__(self):
        if getattr(self, "h", None):
            self.L.h263cu_parser_destroy(self.h)
            self.h = None

    def reset(self):
        self.L.h263cu_parser_reset(self.h)

    def parse_picture(self, packet: bytes, stream=0, pic_index=0, mb_base=0, ev_base=0):
        """Returns (pic ndarray[1], mbs ndarray, events ndarray) for one packet."""
        hdr = Pic()
        check(self.L.h263cu_peek_picture(self.options, packet, len(packet), C.byref(hdr)))
        n_mbs = max(int(hdr.n_mbs), 1)
        mbs = np.zeros(n_mbs, MB_DTYPE)
        ev_cap = len(packet) * 16 // 3 + 16
        events = np.zeros(ev_cap, np.uint16)
        pic = np.zeros(1, PIC_DTYPE)
        check(
            self.L.h263cu_parse_picture(
                self.h, packet, len(packet), stream, pic_index, mb_base, ev_base,
                C.cast(pic.ctypes.data, C.POINTER(Pic)), mbs.ctypes.data, n_mbs, events.ctypes.data, ev_cap,
            )
        )
        return pic, mbs[: int(pic["n_mbs"][0])], events[: int(pic["n_event_units"][0])]


def peek_picture(packet: bytes, options=_lib.OPT_SORENSON):
    pic = np.zeros(1, PIC_DTYPE)
    check(_lib.lib().h263cu_peek_picture(options, packet, len(packet), C.cast(pic.ctypes.data, C.POINTER(Pic))))
    return pic[0]


def decode_events(mb, events, ev_base=0):
    """Expand one MB record's event units into per-block lists of (run, level)."""
    out = []
    off = ev_base + int(mb["ev_off"])
    wide = bool(mb["flags"] & _lib.MB_WIDE)
    for b in range(6):
        blk = []
        for _ in range(int(mb["nev"][b])):
            if wide:
                run = int(events[off]) & 63
                level = int(np.int16(events[off + 1]))
                off += 2
            else:
                u = int(events[off])
                run = u >> 10
                level = u & 0x3FF
                if level >= 512:
                    level -= 1024
                off += 1
            blk.append((run, level))
        out.append(blk)
    return out


def parse_step(parsers, packets, stream_ids=None, threads=0, mb_cap=None, ev_cap=None, pinned=None, ctx=None):
    """Threaded parse of one time step. Returns (pics, mbs, events, errors, pic_of_input).  With ctx (an
    api.Context) the macroblock layer is parsed on its GPU instead (h263cu_test_device_parse_step: the same outputs,
    and the parsers do not advance)."""
    L = _lib.lib()
    n = len(parsers)
    assert len(packets) == n
    hp = (C.c_void_p * n)(*[p.h for p in parsers])
    bufs = [np.frombuffer(pk, np.uint8) for pk in packets]
    pp = (C.c_void_p * n)(*[b.ctypes.data for b in bufs])
    lens = (C.c_size_t * n)(*[len(pk) for pk in packets])
    sid = None
    if stream_ids is not None:
        sid = np.ascontiguousarray(stream_ids, np.uint32)
    if mb_cap is None:
        mb_cap = 0
        for pk, p in zip(packets, parsers):
            try:
                mb_cap += int(peek_picture(pk, p.options)["n_mbs"])
            except _lib.H263Error:
                pass
        mb_cap = max(mb_cap, 1)
    if ev_cap is None:
        ev_cap = sum(len(pk) for pk in packets) * 16 // 3 + 16 * n
    pics = np.zeros(n, PIC_DTYPE)
    mbs = np.zeros(mb_cap, MB_DTYPE)
    events = np.zeros(ev_cap, np.uint16)
    errs = np.zeros(n, np.int32)
    pic_of = np.zeros(n, np.int32)
    npics, nm, nu = C.c_uint32(), C.c_uint32(), C.c_uint32()
    call = L.h263cu_parse_step if ctx is None else (lambda *a: L.h263cu_test_device_parse_step(ctx.h, *a))
    check(
        call(
            hp, pp, lens, sid.ctypes.data if sid is not None else None, n, threads, pics.ctypes.data,
            mbs.ctypes.data, mb_cap, events.ctypes.data, ev_cap, C.byref(npics), C.byref(nm), C.byref(nu),
            errs.ctypes.data, pic_of.ctypes.data,
        )
    )
    return pics[: npics.value], mbs[: nm.value], events[: nu.value], errs, pic_of
