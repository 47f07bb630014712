"""Hand-built side info that reaches the reconstruction kernels' structural edges by construction, and a model of the
tiled kernel's scheduling that says, from the records alone, which of those edges a step reaches.

test_gpu_recon_edges.py decodes the steps built here on the device and compares them with
helpers.recon_from_side_info; test_recon_cases.py asserts on the CPU, through the model below, that every listed edge
occurs, so that a later edit of the generator cannot quietly drop one.  The model is a coverage check, not an oracle.

Scheduling of recon_tile_kernel (recon_tile.cu), as modelled by `schedule`:
- a warp takes a tile of 4 consecutive records of the step's record array (the last tile may hold fewer), whatever
  pictures they belong to;
- the coded blocks (nev > 0) become slots in record order, Y0 Y1 Y2 Y3 Cb Cr inside a record: at most 24;
- the slots' events form one sequence: a slot starts at the number of events of the slots before it;
- the events are walked in chunks: a chunk is the longest run of slots, from the first one not yet walked, whose events
  end at most EV_CAP = 64 events after the chunk's first event (one slot at least); inside a chunk the walk goes in
  rounds of 32 events, and a slot that crosses a round boundary carries its running sum into the next round;
- each slot of a chunk is classified Zero / Dc / Vert / Full (Horiz runs as Full); its rows to transform R are the rows
  that hold an event, plus row 0 when an intra DC is present;
- the slots with R != 0 are stably sorted by key (popcount(R) >= 4, 2..3, 1) and transformed in passes of 4
  consecutive sorted slots; a pass whose slots hold more than 8 events takes the scatter loop.
"""
import numpy as np

import oracle_lib as O
from h263_rs_b200 import _lib, frontend

EV_CAP, ROUND, WARP_MBS = 64, 32, 4
PICFLAG_HAS_INTER, PICFLAG_MV_IN_RANGE = 2, 4
# both sides of the narrow (10-bit) / wide boundary: -512..511 fit the narrow form
LEVELS = (1, -1, 2, -2, 255, -255, 511, -511, -512, 512, -513, 1023, -1023, -1024)
TILE_EVENT_TOTALS = (31, 32, 33, 63, 64, 65, 128, 129)

_ZZ = None


def zigzag():
    """lin = 8 * row + column of every zig-zag index, read off the oracle's inverse_rle"""
    global _ZZ
    if _ZZ is None:
        _ZZ = [int(np.flatnonzero(O.inverse_rle(None, [k], [1], 1)[1].reshape(-1))[0]) for k in range(64)]
    return _ZZ


def dequant_raw(level, quant):
    """rle.rs:130-133 before the clamp (i16 arithmetic, release-mode wrapping)"""
    a = np.int16(abs(level))
    with np.errstate(over="ignore"):
        d = np.int16(np.int16(quant) * np.int16(np.int16(2) * a + np.int16(1)))
        v = np.int16((1 if level > 0 else -1) * np.int16(d + np.int16(0 if quant % 2 else -1)))
    return int(v)


# ---------------------------------------------------------------------------------------------- records
def mb_spec(inter, quant, blocks, codes=None, mv=None):
    """One macroblock: `blocks` = 6 lists of (run, level) events; `codes` = the 6 INTRADC codes (intra);
    `mv` = 4 half-pel vectors (inter)."""
    assert len(blocks) == 6
    return dict(inter=bool(inter), quant=int(quant), blocks=[list(b) for b in blocks],
                codes=[int(c) for c in (codes if codes is not None else [0] * 6)], mv=[tuple(v) for v in (mv or [(0, 0)] * 4)])


def pack_picture(w, h, specs, pquant=8, stream=0, pic_type=None):
    """Records and event units of one picture (h263cu_pic / h263cu_mb / h263cu_event) from macroblock specs in
    raster order.  A record uses the wide event form when one of its levels leaves -512..511."""
    mb_w, mb_h = (w + 15) // 16, (h + 15) // 16
    n = mb_w * mb_h
    assert len(specs) == n, (len(specs), n)
    mbs = np.zeros(n, frontend.MB_DTYPE)
    units = []
    for k, s in enumerate(specs):
        m = mbs[k]
        m["ev_off"] = len(units)
        m["pic"], m["mbx"], m["mby"] = 0, k % mb_w, k // mb_w
        m["quant"] = s["quant"]
        wide = any(level < -512 or level > 511 for ev in s["blocks"] for _, level in ev)
        m["flags"] = _lib.MB_CODED | (_lib.MB_INTER if s["inter"] else 0) | (_lib.MB_WIDE if wide else 0)
        if s["inter"]:
            m["u"] = np.array(s["mv"], np.int8).reshape(8).view(np.uint8)
        else:
            m["u"][:6] = s["codes"]
        for b in range(6):
            m["nev"][b] = len(s["blocks"][b])
        for ev in s["blocks"]:
            for run, level in ev:
                assert 0 <= run < 64 and level != 0
                units += [run, level & 0xFFFF] if wide else [(run << 10) | (level & 0x3FF)]
    any_inter = any(s["inter"] for s in specs)
    pic = np.zeros(1, frontend.PIC_DTYPE)
    pic["stream"], pic["width"], pic["height"], pic["mb_w"], pic["mb_h"] = stream, w, h, mb_w, mb_h
    pic["pic_type"] = (1 if any_inter else 0) if pic_type is None else pic_type
    pic["pquant"] = pquant
    pic["flags"] = (PICFLAG_HAS_INTER if any_inter else 0) | PICFLAG_MV_IN_RANGE
    pic["n_mbs"], pic["n_event_units"] = n, len(units)
    return pic, mbs, np.array(units, np.uint16)


def concat_step(pictures):
    """One step's arrays from (pic, mbs, units) triples: record `pic` fields, first_mb and first_event set."""
    pics = np.concatenate([p for p, _, _ in pictures])
    mbs = np.concatenate([m for _, m, _ in pictures])
    units = np.concatenate([u for _, _, u in pictures]) if pictures else np.zeros(0, np.uint16)
    mb0 = ev0 = 0
    for i, (p, m, u) in enumerate(pictures):
        pics[i]["first_mb"], pics[i]["first_event"] = mb0, ev0
        mbs["pic"][mb0 : mb0 + len(m)] = i
        mb0, ev0 = mb0 + len(m), ev0 + len(u)
    return pics, mbs, units


# ---------------------------------------------------------------------------------------------- events
def events_at(indices, levels, inter):
    """Events that put levels[i] on zig-zag index indices[i] (strictly increasing)"""
    idx, out = (0 if inter else 1), []
    for k, lv in zip(indices, levels):
        assert k >= idx
        out.append((k - idx, lv))
        idx = k + 1
    return out


class Gen:
    """Macroblock specs of every kind the edge list asks for.  Quantisers and levels cycle, so that every QP and every
    level of LEVELS occurs; the rest is drawn from a seeded generator."""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.nq = 0
        self.nl = 0

    def quant(self):
        self.nq += 1
        return 1 + (self.nq - 1) % 31

    def level(self):
        self.nl += 1
        return LEVELS[(self.nl - 1) % len(LEVELS)]

    def code(self):
        return int(self.rng.choice([1, 2, 64, 127, 128, 129, 200, 254, 255]))

    def mv(self):
        return [tuple(int(v) for v in self.rng.integers(-32, 32, 2)) for _ in range(4)]

    def n_events(self, n, inter, last=None):
        """n events that stay inside the block; `last` pins the zig-zag index of the last one (64 and beyond:
        the block overflows on its last event)"""
        start = 0 if inter else 1
        if last is None:
            idx = sorted(self.rng.choice(np.arange(start, 64), n, replace=False).tolist())
        else:
            # the others below min(last, 64), the one before the last close enough for a run of at most 63
            pool = np.arange(max(start, last - 64), min(last, 64)) if n > 1 else np.arange(0)
            assert n == 1 and last - start <= 63 or len(pool) >= n - 1
            head = sorted(self.rng.choice(pool, n - 1, replace=False).tolist()) if n > 1 else []
            idx = head + [last]
        return events_at(idx, [self.level() for _ in idx], inter)

    def full(self, mask, inter):
        """A Full block whose events occupy exactly the rows of `mask` (and some column > 0)"""
        zz = zigzag()
        inv = {lin: k for k, lin in enumerate(zz)}
        rows = [r for r in range(8) if (mask >> r) & 1]
        cols = [int(self.rng.integers(0, 8)) for _ in rows]
        if not inter and rows[0] == 0:
            cols[0] = max(cols[0], 1)  # the intra DC owns (0, 0)
        if all(c == 0 for c in cols):
            cols[-1] = int(self.rng.integers(1, 8))
        idx = sorted(inv[8 * r + c] for r, c in zip(rows, cols))
        return events_at(idx, [self.level() for _ in idx], inter)

    def kind(self, kind, inter, chroma=False):
        """One block of a named kind"""
        zz = zigzag()
        inv = {lin: k for k, lin in enumerate(zz)}
        start = 0 if inter else 1
        r = self.rng
        if kind == "empty":
            return []
        if kind == "lone":
            return events_at([int(r.integers(start, 64))], [self.level()], inter)
        if kind == "dc":  # inter: one coefficient on index 0; intra: nothing but the DC
            return events_at([0], [self.level()], True) if inter else []
        if kind == "vert":
            rows = sorted(r.choice(np.arange(1, 8), int(r.integers(1, 8)), replace=False).tolist())
            if inter and r.random() < 0.5:
                rows = [0] + rows
            idx = sorted(inv[8 * y] for y in rows)
            return events_at(idx, [self.level() for _ in idx], inter)
        if kind == "horiz":
            cols = sorted(r.choice(np.arange(1, 8), int(r.integers(1, 8)), replace=False).tolist())
            if inter and r.random() < 0.5:
                cols = [0] + cols
            idx = sorted(inv[c] for c in cols)
            return events_at(idx, [self.level() for _ in idx], inter)
        if kind == "full":
            return self.full(int(r.integers(1, 256)), inter)
        if kind == "long":
            return self.n_events(int(r.integers(9, 64 - start + 1)), inter)
        if kind == "short":
            return self.n_events(int(r.integers(2, 9)), inter)
        raise ValueError(kind)

    def mb(self, inter, blocks, codes=None):
        return mb_spec(inter, self.quant(), blocks, codes if codes is not None else [self.code() for _ in range(6)],
                       self.mv() if inter else None)

    def counts_tile(self, counts, inter=None):
        """A tile of 4 macroblocks whose 24 blocks hold counts[b] events each (missing = 0), within the block"""
        counts = list(counts) + [0] * (24 - len(counts))
        mbs = []
        for q in range(4):
            it = bool(self.rng.integers(0, 2)) if inter is None else inter
            if not it and max(counts[6 * q : 6 * q + 6]) > 63:
                it = True
            mbs.append(self.mb(it, [self.n_events(c, it) if c else [] for c in counts[6 * q : 6 * q + 6]]))
        return mbs

    def random_tile(self):
        kinds = ["empty", "lone", "dc", "vert", "horiz", "full", "full", "short", "long"]
        p = np.array([3, 2, 1, 2, 1, 3, 3, 3, 1], float)
        out = []
        for _ in range(4):
            inter = self.rng.random() < 0.6
            out.append(self.mb(inter, [self.kind(str(self.rng.choice(kinds, p=p / p.sum())), inter, b >= 4) for b in range(6)]))
        return out


def case_mbs(seed=1):
    """The block-structure cases, in tiles of 4 macroblocks (each tile list is one warp's work when the picture that
    holds it starts on a multiple of 4 records)."""
    g = Gen(seed)
    tiles = []

    def add(mbs):
        assert len(mbs) % 4 == 0
        tiles.extend(mbs[i : i + 4] for i in range(0, len(mbs), 4))

    # every zig-zag position as a lone coefficient: inter 0..63, intra 1..63 (beside its DC), luma and chroma
    for inter in (True, False):
        pos = list(range(0 if inter else 1, 64))
        mbs = []
        for i in range(32):
            blocks = []
            for b in range(6):
                j = 4 * i + b if b < 4 else 2 * i + b - 4
                blocks.append(events_at([pos[j]], [g.level()], inter) if j < len(pos) else g.kind("short", inter))
            mbs.append(g.mb(inter, blocks))
        add(mbs)
    # Full with every non-empty row mask, luma and chroma; inter and intra alternate
    mbs = []
    for j in range(128):
        inter = j % 2 == 0
        blocks = []
        for b in range(6):
            mask = 4 * j + b + 1 if b < 4 else 2 * j + b - 4 + 1
            blocks.append(g.full(mask, inter) if mask <= 255 else g.kind("full", inter))
        mbs.append(g.mb(inter, blocks))
    add(mbs)
    # classes: Dc (intra DC only, INTRADC codes 1, 254, 255; an inter coefficient on index 0), Vert with and without
    # an intra DC, Horiz
    add([g.mb(False, [[]] * 6, [255, 254, 1, 128, 255, 1]), g.mb(True, [g.kind("dc", True) for _ in range(6)]),
         g.mb(False, [g.kind("vert", False) for _ in range(6)]), g.mb(True, [g.kind("vert", True) for _ in range(6)])])
    add([g.mb(False, [g.kind("horiz", False) for _ in range(6)]), g.mb(True, [g.kind("horiz", True) for _ in range(6)]),
         g.mb(False, [[]] * 6, [0, 0, 0, 0, 0, 0]), g.mb(True, [[]] * 6)])
    # tiles with 0, 1 and 24 coded slots
    add([g.mb(True, [[]] * 6) for _ in range(4)])
    add([g.mb(False, [[]] * 6) for _ in range(4)])
    add(g.counts_tile([0, 0, 0, 0, 0, 0, 0, 0, 0, 5], inter=True))
    add(g.counts_tile([int(c) for c in g.rng.integers(1, 3, 24)]))
    add(g.counts_tile([int(c) for c in g.rng.integers(1, 9, 24)], inter=False))
    # tile event totals around the round (32) and the chunk (64)
    for total in TILE_EVENT_TOTALS:
        for inter in (True, False):
            counts, left = [], total
            while left:
                c = min(left, int(g.rng.integers(1, 20)))
                counts.append(c)
                left -= c
            assert len(counts) <= 24
            add(g.counts_tile(counts, inter=inter))
    # a slot starting exactly on a round, one straddling it, one ending exactly at event 64 of its chunk
    add(g.counts_tile([10, 22, 5, 3], inter=True))
    add(g.counts_tile([10, 20, 5, 3], inter=False))
    add(g.counts_tile([30, 34, 4]))
    add(g.counts_tile([20, 12, 32, 1, 2], inter=True))
    # an inter slot of 64 events, every run 0, first in its tile and after other slots: its own chunk either way;
    # an intra slot of 63 AC events
    full64 = [(0, g.level()) for _ in range(64)]
    add([g.mb(True, [full64, g.kind("short", True), [], [], [], g.kind("lone", True)])] + g.counts_tile([3, 4, 2, 1, 6])[:3])
    add([g.mb(True, [g.kind("short", True), g.kind("long", True), full64, [], [(0, g.level()) for _ in range(64)], []]),
         g.mb(False, [[(0, g.level()) for _ in range(63)], [], g.kind("short", False), [], [], []])] + g.counts_tile([5, 5])[:2])
    # overflow: the last event on index 63 (kept) or 64 (dropped), on the first event (run 63: intra drops, inter keeps),
    # in a slot that straddles a round, in a slot of the second chunk; an intra overflow drops its DC too
    add([g.mb(True, [g.n_events(5, True, last=63), g.n_events(5, True, last=64), [(63, g.level())], g.n_events(2, True, last=64),
                     g.n_events(12, True, last=63), g.n_events(12, True, last=70)]),
         g.mb(False, [g.n_events(5, False, last=63), g.n_events(5, False, last=64), [(63, g.level())], [(62, g.level())],
                      g.n_events(30, False, last=64), g.n_events(3, False, last=90)]),
         g.mb(True, [g.n_events(20, True), g.n_events(20, True, last=66), g.n_events(30, True, last=64), [], [], []]),
         g.mb(False, [g.n_events(40, False), g.n_events(30, False), g.n_events(8, False, last=64), [], [], g.n_events(2, False, last=80)])])
    # passes that mix the sort keys and Vert with non-Vert slots, short and long slots in one pass, last passes of
    # 1..3 slots: seeded random tiles (the coverage test checks that each of these occurs)
    for _ in range(48):
        add(g.random_tile())
    return tiles


def pictures_from_tiles(tiles, w, h, filler):
    """Cuts the tiles into pictures of w x h (a multiple of 4 macroblocks); the last one is filled with `filler()`"""
    per = ((w + 15) // 16) * ((h + 15) // 16)
    assert per % 4 == 0
    flat = [m for t in tiles for m in t]
    out = []
    for i in range(0, len(flat), per):
        part = flat[i : i + per]
        while len(part) < per:
            part.append(filler())
        out.append(part)
    return out


def textured_intra(g, n):
    """Intra macroblocks with varied content (DC of every block, some AC) to predict from"""
    return [g.mb(False, [g.kind(str(g.rng.choice(["empty", "full", "short", "vert"])), False) for _ in range(6)]) for _ in range(n)]


# ---------------------------------------------------------------------------------------------- sequences
# Streams of the edge sequence.  A stream's pictures are decoded one per step, from step 0.
BLOCKS_W, BLOCKS_H = 128, 96   # the block-structure cases, 48 macroblocks (12 tiles) per picture


def block_stream(seed=1):
    """Stream 0: a textured I picture, then P pictures that hold every case of case_mbs (mixed inter / intra)."""
    g = Gen(seed + 100)
    n = (BLOCKS_W // 16) * (BLOCKS_H // 16)
    pics = [(BLOCKS_W, BLOCKS_H, textured_intra(g, n), 12)]
    for part in pictures_from_tiles(case_mbs(seed), BLOCKS_W, BLOCKS_H, lambda: g.mb(True, [[]] * 6)):
        pics.append((BLOCKS_W, BLOCKS_H, part, int(g.rng.integers(1, 32))))
    return pics


def mixed_pictures_streams(seed=2):
    """Streams 1 (48x16, 3 macroblocks) and 2 (80x48, 15): record counts that are not multiples of 4, so a warp's tile
    spans both pictures; their types and QPs differ in every step."""
    g = Gen(seed)
    a, b = [], []
    types = [(False, False), (True, False), (False, True), (True, True)]
    quants = [(2, 29), (31, 1), (9, 17), (25, 4)]
    for (ia, ib), (qa, qb) in zip(types, quants):
        for lst, w, h, inter, q in ((a, 48, 16, ia, qa), (b, 80, 48, ib, qb)):
            n = ((w + 15) // 16) * ((h + 15) // 16)
            specs = []
            for _ in range(n):
                blocks = [g.kind(str(g.rng.choice(["empty", "full", "short", "vert", "lone"])), inter) for _ in range(6)]
                s = g.mb(inter, blocks)
                s["quant"] = q
                specs.append(s)
            lst.append((w, h, specs, q))
    return a, b


def saturation_stream(seed=3):
    """Stream 3 (64x16): regions driven to 255 and to 0 by intra DCs plus an inter DC step, then residuals of both
    signs on top of those pinned predictions (zero vectors), so that the saturating add clamps at both ends."""
    g = Gen(seed)
    hi, lo = [254] * 6, [1] * 6
    i_pic = [g.mb(False, [[]] * 6, hi), g.mb(False, [[]] * 6, lo), g.mb(False, [[]] * 6, hi), g.mb(False, [[]] * 6, lo)]
    zero = [(0, 0)] * 4
    up, down = [[(0, 40)] for _ in range(6)], [[(0, -40)] for _ in range(6)]  # +-(40 * 21 - 1) / 8: beyond the range
    p1 = [mb_spec(True, 10, up, mv=zero), mb_spec(True, 10, down, mv=zero), mb_spec(True, 10, up, mv=zero), mb_spec(True, 10, down, mv=zero)]
    p2 = [mb_spec(True, 20, [g.full(int(g.rng.integers(1, 256)), True) for _ in range(6)], mv=zero) for _ in range(4)]
    return [(64, 16, i_pic, 5), (64, 16, p1, 10), (64, 16, p2, 20)]


def motion_stream(seed=4):
    """Stream 4 (CIF, 4MV): every luma vector pair of [-32, 31]^2 across three P pictures, coded residual blocks on
    some macroblocks; chroma vector sums of every residue of average_sum_of_mvs follow."""
    g = Gen(seed)
    n = 22 * 18
    pairs = [(x, y) for x in range(-32, 32) for y in range(-32, 32)]
    order = g.rng.permutation(len(pairs))
    pics = [(352, 288, textured_intra(g, n), 6)]
    k = 0
    for _ in range(3):
        specs = []
        for _ in range(n):
            mv = []
            for _ in range(4):
                mv.append(pairs[order[k % len(pairs)]])
                k += 1
            blocks = [g.kind(str(g.rng.choice(["empty", "empty", "lone", "short", "full"])), True) for _ in range(6)]
            s = g.mb(True, blocks)
            s["mv"] = mv
            specs.append(s)
        pics.append((352, 288, specs, int(g.rng.integers(1, 32))))
    assert k >= len(pairs)
    return pics


def small_stream(w, h, n_pics, seed, wide_mv=False):
    """A stream of random tiles at any size, vectors across the picture's edges; with wide_mv, vectors up to +-120
    half-pel units (beyond the range: the picture takes the clamped-prediction instantiation)"""
    g = Gen(seed)
    n = ((w + 15) // 16) * ((h + 15) // 16)
    pics = [(w, h, textured_intra(g, n), 7)]
    for _ in range(n_pics - 1):
        specs = [m for _ in range((n + 3) // 4) for m in g.random_tile()][:n]
        for s in specs:
            if s["inter"]:
                lo, hi = (-120, 121) if wide_mv else (-32, 32)
                s["mv"] = [tuple(int(v) for v in g.rng.integers(lo, hi, 2)) for _ in range(4)]
        pics.append((w, h, specs, int(g.rng.integers(1, 32))))
    return pics


def pack_stream(stream_id, pics):
    return [pack_picture(w, h, specs, pquant=q, stream=stream_id) for w, h, specs, q in pics]


def edge_streams():
    """stream id -> list of packed pictures (pic, mbs, units), one per step from step 0"""
    a, b = mixed_pictures_streams()
    return {0: pack_stream(0, block_stream()), 1: pack_stream(1, a), 2: pack_stream(2, b), 3: pack_stream(3, saturation_stream()),
            4: pack_stream(4, motion_stream()), 5: pack_stream(5, small_stream(40, 24, 6, 5)),
            6: pack_stream(6, small_stream(23, 9, 6, 6)), 7: pack_stream(7, small_stream(64, 48, 6, 7, wide_mv=True)),
            8: pack_stream(8, small_stream(40, 24, 6, 8, wide_mv=True))}


def steps_of(streams, ids):
    """The steps that decode the streams `ids` side by side: step t holds picture t of every stream that has one, in
    the order of `ids`.  Returns a list of (step arrays, [(stream id, picture index)])."""
    out = []
    n = max(len(streams[s]) for s in ids)
    for t in range(n):
        members = [(s, t) for s in ids if t < len(streams[s])]
        step = concat_step([streams[s][t] for s, _ in members])
        out.append((step, members))
    return out


# ---------------------------------------------------------------------------------------------- the model
def _slot(m, b, blk, code):
    inter = bool(m["flags"] & _lib.MB_INTER)
    zz = zigzag()
    idx = 0 if inter else 1
    rows, col, ovf, ovf_at, last = 0, False, False, None, None
    for run, _ in blk:
        idx += run
        if idx >= 64:
            ovf, ovf_at = True, idx
            break
        lin = zz[idx]
        rows |= 1 << (lin >> 3)
        col |= (lin & 7) != 0
        last = idx
        idx += 1
    has_dc = not inter and code != 0 and not ovf
    if ovf or (not rows and not has_dc):
        cls = "zero"
    elif not (rows & 0xFE) and not col:
        cls = "dc"
    elif col:
        cls = "full"
    else:
        cls = "vert"
    R = (rows | (1 if has_dc else 0)) if cls in ("full", "vert") else 0
    n = bin(R).count("1")
    key = 3 if not R else (0 if n >= 4 else (1 if n >= 2 else 2))
    return dict(inter=inter, chroma=b >= 4, nev=len(blk), ev=blk, rows=rows, col=col, ovf=ovf, ovf_at=ovf_at, last=last,
                has_dc=has_dc, cls=cls, R=R, key=key, code=code, quant=int(m["quant"]))


def schedule(pics, mbs, units):
    """The tiles of one step as the tiled kernel schedules them: per tile its slots (with start / end / chunk / pass
    and class), its chunks and its passes."""
    tiles = []
    for t0 in range(0, len(mbs), WARP_MBS):
        recs = mbs[t0 : t0 + WARP_MBS]
        slots = []
        for m in recs:
            p = pics[int(m["pic"])]
            blocks = frontend.decode_events(m, units, int(p["first_event"]))
            inter = bool(m["flags"] & _lib.MB_INTER)
            for b in range(6):
                if m["nev"][b]:
                    slots.append(_slot(m, b, blocks[b], 0 if inter else int(m["u"][b])))
        e = 0
        for s in slots:
            s["start"], s["end"] = e, e + s["nev"]
            e = s["end"]
        chunks, passes = [], []
        s_lo, e_lo = 0, 0
        while s_lo < len(slots):
            s_hi = s_lo + sum(1 for s in slots[s_lo:] if s["end"] - e_lo <= EV_CAP)
            s_hi = max(s_hi, s_lo + 1)
            ch = slots[s_lo:s_hi]
            for s in ch:
                s["chunk"], s["rel"] = len(chunks), s["start"] - e_lo
            need = sorted([s for s in ch if s["key"] < 3], key=lambda s: s["key"])  # stable
            ps = [need[i : i + 4] for i in range(0, len(need), 4)]
            chunks.append(dict(slots=ch, e_lo=e_lo, passes=ps))
            passes += ps
            s_lo, e_lo = s_hi, ch[-1]["end"]
        tiles.append(dict(recs=recs, pics=[pics[int(m["pic"])] for m in recs], slots=slots, events=e, chunks=chunks, passes=passes))
    return tiles


def features(steps):
    """The set of edges the steps reach, as tags (see test_recon_cases.py for the list that must occur)"""
    f = set()
    for (pics, mbs, units), _ in steps:
        for m in mbs:
            inter = bool(m["flags"] & _lib.MB_INTER)
            if inter:
                mv = m["u"].view(np.int8).reshape(4, 2).astype(int)
                for x, y in mv:
                    f.add(("mv", int(x), int(y)))
                f.add(("chroma_residue", "x", int(mv[:, 0].sum()) & 15))
                f.add(("chroma_residue", "y", int(mv[:, 1].sum()) & 15))
            else:
                for b in range(6):
                    if not m["nev"][b] and m["u"][b]:
                        f.add(("dc_only_intra", int(m["u"][b])))
        for t in schedule(pics, mbs, units):
            f.add(("tile_slots", len(t["slots"])))
            f.add(("tile_events", t["events"]))
            if len({int(m["pic"]) for m in t["recs"]}) > 1:
                ps = t["pics"]
                if len({int(p["pic_type"]) for p in ps}) > 1 and len({int(m["quant"]) for m in t["recs"]}) > 1:
                    f.add(("tile_spans_pictures",))
            for c in t["chunks"]:
                if c["passes"]:
                    f.add(("last_pass_size", len(c["passes"][-1])))
            for p in t["passes"]:
                keys = sorted({s["key"] for s in p})
                if len(keys) > 1:
                    f.add(("pass_keys", tuple(keys)))
                verts = {s["cls"] == "vert" for s in p}
                if verts == {True, False}:
                    f.add(("pass_vert_mix",))
                if any(s["nev"] > 8 for s in p) and any(s["nev"] <= 8 for s in p):
                    f.add(("pass_long_short",))
            for i, s in enumerate(t["slots"]):
                inter, chroma, cls = s["inter"], s["chroma"], s["cls"]
                f.add(("cls", cls, inter, chroma))
                f.add(("qp", s["quant"]))
                for _, lv in s["ev"]:
                    f.add(("level", lv))
                    v = dequant_raw(lv, s["quant"])
                    if v > 2047:
                        f.add(("clamp", 1))
                    if v < -2048:
                        f.add(("clamp", -1))
                if s["nev"] == 1 and not s["ovf"]:
                    f.add(("lone", inter, chroma, s["last"]))
                if cls == "dc" and inter:
                    f.add(("dc_inter_index0",))
                if cls == "vert":
                    f.add(("vert", s["has_dc"]))
                if cls == "full" and not (s["rows"] & 0xFE):
                    f.add(("horiz", inter))
                if cls == "full":
                    f.add(("full_rows", chroma, s["rows"]))
                rel, end = s["rel"], s["rel"] + s["nev"]
                if rel and rel % ROUND == 0:
                    f.add(("slot_on_round",))
                straddle = rel // ROUND != (end - 1) // ROUND
                if straddle:
                    f.add(("slot_straddles_round",))
                if end == EV_CAP:
                    f.add(("slot_ends_at_64",))
                if s["nev"] == 64 and inter and all(r == 0 for r, _ in s["ev"]):
                    own = sum(1 for x in t["slots"] if x["chunk"] == s["chunk"]) == 1
                    if own:
                        f.add(("own_chunk_64", "first" if i == 0 else "after"))
                if not inter and s["nev"] == 63 and not s["ovf"]:
                    f.add(("intra_63",))
                if not s["ovf"] and s["last"] == 63:
                    f.add(("last_at_63", inter))
                if s["ovf"] and s["ovf_at"] == 64 and _overflow_on_last(s):
                    f.add(("overflow_on_64", inter))
                if s["ev"][0][0] == 63:
                    f.add(("first_run_63", inter, s["ovf"]))
                if s["ovf"]:
                    if straddle:
                        f.add(("overflow_straddles_round",))
                    if s["chunk"] > 0:
                        f.add(("overflow_in_later_chunk",))
                    if not inter and s["code"]:
                        f.add(("overflow_drops_intra_dc",))
    return f


def _overflow_on_last(s):
    """the block's index reaches 64 on its last event"""
    idx = 0 if s["inter"] else 1
    for k, (run, _) in enumerate(s["ev"]):
        idx += run
        if idx >= 64:
            return k == len(s["ev"]) - 1
        idx += 1
    return False
