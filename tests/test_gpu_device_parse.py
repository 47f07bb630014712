"""The macroblock layer parsed on the GPU (H263CU_PARSE_ON_DEVICE, parse="device"): the side info equals the host
parser's byte for byte (h263cu_test_device_parse_step against h263cu_parse_step), damaged packets fail with the same
per-picture errors, every output of a decode step is the host-parse step's, whole-call failures change nothing, and
the decoded planes match the oracle."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import oracle_decode_stream
from h263_rs_b200 import _lib, api, frontend, synth
from test_frontend import CASES

pytestmark = pytest.mark.gpu

E = _lib


def same_side_info(host, dev):
    """host / dev: parse_step's (pics, mbs, events, errors, pic_of_input); equal byte for byte."""
    for a, b, name in zip(host, dev, ("pics", "mbs", "events", "errors", "pic_of_input")):
        assert a.shape == b.shape, name
        assert a.tobytes() == b.tobytes(), name


def lockstep_parse(ctx, streams, options, threads=4):
    """Every stream decoded step by step: the device hook first (parsers stay), then the host parser (parsers advance).
    streams: list of packet lists.  Returns the per-picture errors seen."""
    parsers = [frontend.Parser(o) for o in options]
    errs = []
    for t in range(max(len(s) for s in streams)):
        idx = [k for k, s in enumerate(streams) if t < len(s)]
        ps = [parsers[k] for k in idx]
        pk = [streams[k][t] for k in idx]
        ids = np.asarray(idx, np.uint32)
        dev = frontend.parse_step(ps, pk, ids, threads, ctx=ctx)
        host = frontend.parse_step(ps, pk, ids, threads)
        same_side_info(host, dev)
        errs += [int(e) for e in host[3]]
    return errs


@pytest.fixture(scope="module")
def ctx():
    return api.Context(0, 4, 352, 288)


def test_side_info_on_the_frontend_cases(ctx):
    for c in CASES:
        kw = {k: v for k, v in c.items() if k not in ("w", "h", "n", "seed")}
        pk = synth.make_stream(c["w"], c["h"], c["n"], c["seed"], **kw)
        opt = 0 if kw.get("flavour") == 1 else 1
        lockstep_parse(ctx, [pk], [opt])


def test_side_info_baseline_disposable_wide_and_dense():
    ctx = api.Context(0, 4, 352, 288)
    streams, opts = [], []
    streams.append(synth.make_stream(176, 144, 6, 31, flavour=1, pct_escape=15)); opts.append(0)
    for dd in (1, 1 | 0x100):  # disposable P pictures without and with H263CU_OPT_DECODE_DISPOSABLE
        streams.append(synth.make_stream(176, 144, 6, 32, pct_disposable=50)); opts.append(dd)
    streams.append(synth.make_stream(352, 288, 4, 33, version=1, pct_escape=40)); opts.append(1)
    streams.append(synth.make_stream(128, 96, 4, 34, mean_events_x10=300, pct_cbp_inter=95)); opts.append(1)
    lockstep_parse(ctx, streams, opts)
    # wide macroblocks and more than 32 events per macroblock were reached
    p, m, ev, _, _ = frontend.parse_step([frontend.Parser(1)], [streams[3][0]])
    assert (m["flags"] & E.MB_WIDE).any()
    p, m, ev, _, _ = frontend.parse_step([frontend.Parser(1)], [streams[4][0]])
    assert (m["nev"].astype(np.int64).sum(axis=1) > 32).any()


def test_side_info_of_a_bench_step():
    """1024 CIF streams with bench.py's generator parameters, I picture then P picture."""
    import bench

    S = 1024
    blobs = bench.generate_streams(range(S), 2, 8)
    ctx = api.Context(0, S, 352, 288)
    streams = [[bytes(b[int(o[t]) : int(o[t]) + int(l[t])]) for t in range(2)] for b, o, l in blobs]
    errs = lockstep_parse(ctx, streams, [1] * S, threads=16)
    assert not any(errs)


# The GOB resynchronisation stub's exits, by what follows the start code: a GOB number of 0 or 15 ends the picture,
# any other is refused (UNIMPLEMENTED_DECODING), and a number cut off, a start code cut off (EOF) or no start code in
# reach ends the picture too.  Every tail begins with at least 10 zero bits, an invalid MCBPC.
GOB_TAILS = {
    "gn0": [0] * 16 + [1] + [0, 0, 0, 0, 0],
    "gn5": [0] * 16 + [1] + [0, 0, 1, 0, 1],
    "gn15": [0] * 16 + [1] + [0, 1, 1, 1, 1],
    "gn_cut": [0] * 16 + [1] + [0, 1],
    "eof": [0] * 12,
    "no_start_code": [0] * 10 + [1] * 14,
}
# The picture is an I picture of a fresh parser: an exit that ends it leaves it padded with uncoded macroblocks, which
# need a reference it does not have (UNCODED_IFRAME_BLOCKS, -15); the refusal is UNIMPLEMENTED_DECODING (-17).
GOB_EXIT_ERR = {"gn0": -15, "gn5": -17, "gn15": -15, "gn_cut": -15, "eof": -15, "no_start_code": -15}


def gob_cases(base):
    """A baseline I picture cut at every bit of its first 90 and followed by each tail: where the cut lands on a
    macroblock boundary, the invalid header reaches the stub.  Returns (cut, tail name, packet)."""
    bits = np.unpackbits(np.frombuffer(base, np.uint8))
    return [(c, name, np.packbits(np.concatenate([bits[:c], np.asarray(tail, np.uint8)])).tobytes())
            for c in range(30, 90) for name, tail in GOB_TAILS.items()]


def damaged_trials(n_trials=960, seed=5):
    """test_frontend.test_damaged_streams_fail_identically's scheme: bit flips (headers included), truncation and
    garbage tails, one victim picture per trial."""
    rng = np.random.default_rng(seed)
    bases = [(synth.make_stream(176, 144, 4, 21, pct_escape=10), 1), (synth.make_stream(64, 48, 5, 22, pct_fourmv=30, mv_mode=1), 1),
             (synth.make_stream(176, 144, 3, 23, flavour=1), 0), (synth.make_stream(48, 32, 6, 24, version=0, pct_escape=25), 1),
             (synth.make_stream(96, 64, 4, 25, version=1, pct_escape=30), 1)]
    streams, opts = [], []
    for trial in range(n_trials):
        base, opt = bases[trial % len(bases)]
        pk = [bytearray(p) for p in base]
        victim = int(rng.integers(0, len(pk)))
        mode = trial % 3
        if mode == 0:
            for _ in range(int(rng.integers(1, 4))):
                pos = int(rng.integers(0, len(pk[victim])))
                pk[victim][pos] ^= 1 << int(rng.integers(0, 8))
        elif mode == 1:
            pk[victim] = pk[victim][: int(rng.integers(1, len(pk[victim])))]
        else:
            pk[victim] = pk[victim] + bytes(rng.integers(0, 256, int(rng.integers(1, 6)), dtype=np.uint8))
        streams.append([bytes(p) for p in pk])
        opts.append(opt)
    for _, _, pk in gob_cases(bases[2][0][0]):
        streams.append([pk])
        opts.append(0)
    return streams, opts


def test_damaged_packets_fail_identically():
    streams, opts = damaged_trials()
    ctx = api.Context(0, len(streams), 176, 144)
    errs = lockstep_parse(ctx, streams, opts, threads=8)
    seen = set(errs)
    # every macroblock- and block-layer error and the one-macroblock-too-many abort
    for code in (-3, -4, -5, -6, -7, -8, -16, -104):
        assert code in seen, (code, sorted(seen))
    # every exit of the GOB stub: a cut where "gn5" is refused is a macroblock boundary of an I picture of a fresh
    # parser (no format change, a supported type: the refusal is the stub's), so every tail at that cut entered the stub
    # too, and each left it by its own exit with the same outcome on both sides (lockstep_parse compared the records)
    first = errs[: len(streams)]  # step 0 holds every stream, in stream order
    cases = gob_cases(synth.make_stream(176, 144, 3, 23, flavour=1)[0])
    by_cut = {}
    for (c, name, _), e in zip(cases, first[len(streams) - len(cases):]):
        by_cut.setdefault(c, {})[name] = e
    stub_cuts = [c for c, r in by_cut.items() if r["gn5"] == -17]
    assert stub_cuts
    cut_exit = False
    for c in stub_cuts:
        # the packet ends at the next byte boundary: "gn_cut" leaves 2 GOB-number bits plus the zero padding, fewer
        # than 5 only for some cuts (else the padded number is read and refused)
        number_cut = 2 + (-(c + 19)) % 8 < 5
        cut_exit |= number_cut
        want = dict(GOB_EXIT_ERR, gn_cut=-15 if number_cut else -17)
        assert by_cut[c] == want, (c, by_cut[c])
    assert cut_exit


# ---- end to end ----

SIZES = [(176, 144), (352, 288), (160, 120), (200, 100)]


def make_sequences(n_streams, n_steps, seed):
    """Mixed picture sizes; at a few (stream, step) points a damaged packet is sent first and the good one next step."""
    rng = np.random.default_rng(seed)
    streams = []
    for s in range(n_streams):
        w, h = SIZES[s % len(SIZES)]
        streams.append(synth.make_stream(w, h, n_steps, 100 + s, pct_fourmv=20, mv_mode=s % 3, pct_escape=5))
    plan = []  # per step: list of (stream, packet)
    pos = [0] * n_streams
    for t in range(n_steps + 3):
        step = []
        for s in range(n_streams):
            if pos[s] >= n_steps:
                continue
            good = streams[s][pos[s]]
            if pos[s] > 0 and rng.random() < 0.15:
                bad = bytearray(good)
                if rng.random() < 0.5:
                    bad = bad[: max(1, len(bad) // 2)]
                else:
                    bad[int(rng.integers(4, len(bad)))] ^= 0xFF
                step.append((s, bytes(bad)))  # resubmitted next step
            else:
                step.append((s, good))
                pos[s] += 1
        if step:
            plan.append(step)
    return plan


def out_of(dec, kind, pk, ids, parse):
    """One step of output `kind`; returns (comparable arrays, errors)."""
    n = len(pk)
    if kind == "host_rgba":
        size = 352 * 288 * 4
        buf = np.zeros(n * size, np.uint8)
        L = _lib.lib()
        pinned = L.h263cu_alloc_pinned(buf.size)
        C.memset(pinned, 0, buf.size)  # the slots of failed inputs are never written
        try:
            errs = dec.decode_step(pk, stream_ids=ids, host_rgba=pinned, rgba_stride=size, parse=parse).copy()
            dec.ctx.sync()
            C.memmove(buf.ctypes.data, pinned, buf.size)
        finally:
            L.h263cu_free_pinned(pinned)
        return [buf.reshape(n, size)], errs
    if kind == "rgba":
        out = torch.zeros((n, 288, 352, 4), dtype=torch.uint8, device="cuda")
        o, errs = dec.decode_step_device(pk, out=out, stream_ids=ids, parse=parse)
        return [o.cpu().numpy()], errs.copy()
    if kind.startswith("i420") or kind.startswith("nv12"):
        layout = kind[:4]
        # zeroed planes: bytes of a slot outside its picture may or may not be written
        z = lambda *shape: torch.zeros(shape, dtype=torch.uint8, device="cuda")  # noqa: E731
        planes = (z(n, 288, 352), z(n, 144, 176, 2)) if layout == "nv12" else (z(n, 288, 352), z(n, 144, 176), z(n, 144, 176))
        outs, errs = dec.decode_step_device_yuv(pk, out=planes, layout=layout, deblock=kind.endswith("_db"), stream_ids=ids,
                                                parse=parse)
        return [t.cpu().numpy() for t in outs], errs.copy()
    if kind == "stretch":
        o, errs = dec.decode_step_device_tensor(pk, (96, 128), dtype=torch.float16, stream_ids=ids, parse=parse)
    elif kind == "center_crop":
        o, errs = dec.decode_step_device_tensor(pk, (112, 112), dtype=torch.float32, fit="center_crop", short_side=128,
                                                stream_ids=ids, parse=parse)
    else:  # bicubic with antialias
        o, errs = dec.decode_step_device_tensor(pk, (64, 64), dtype=torch.float32, antialias=True, interpolation="bicubic",
                                                deblock=True, stream_ids=ids, parse=parse)
    return [o.cpu().numpy().view(np.uint8)], errs.copy()


def run_pair(kind, plan, n_streams, parses):
    """A host-parse decoder and a decoder whose steps use `parses` in turn, in lock step; every output, error, count
    and plane after every step must agree."""
    ref = api.BatchDecoder(n_streams, 352, 288, threads=4)
    dut = api.BatchDecoder(n_streams, 352, 288, threads=4)
    n_fail = 0
    for t, step in enumerate(plan):
        ids = np.asarray([s for s, _ in step], np.uint32)
        pk = [p for _, p in step]
        a, ea = out_of(ref, kind, pk, ids, "host")
        b, eb = out_of(dut, kind, pk, ids, parses[t % len(parses)])
        assert np.array_equal(ea, eb), (kind, t)
        n_fail += int((ea != 0).sum())
        for x, y in zip(a, b):
            # slots of failed inputs are left alone by both: compare the decoded slots only
            for i in np.nonzero(ea == 0)[0]:
                assert np.array_equal(x[i] if x.ndim > 1 else x, y[i] if y.ndim > 1 else y), (kind, t, i)
        torch.cuda.synchronize()
        ref.ctx.sync(), dut.ctx.sync()
        for s in ids[ea == 0]:
            for pa, pb in zip(ref.ctx.read_yuv(int(s)), dut.ctx.read_yuv(int(s))):
                assert np.array_equal(pa, pb), (kind, t, s)
    assert n_fail > 0  # the damaged packets were seen


@pytest.mark.parametrize("kind", ["host_rgba", "rgba", "i420", "i420_db", "nv12", "nv12_db", "stretch", "center_crop", "bicubic_aa"])
def test_end_to_end_every_output(kind):
    plan = make_sequences(12, 5, 7)
    run_pair(kind, plan, 12, ["device"])


def test_host_and_device_steps_alternate_on_one_context():
    plan = make_sequences(12, 6, 8)
    run_pair("rgba", plan, 12, ["device", "host"])
    run_pair("i420", plan, 12, ["host", "device"])


def test_group_form_on_two_contexts_of_one_device():
    plan = make_sequences(8, 4, 9)
    groups = {p: api.DeviceGroup([0, 0], 4, 352, 288, threads=4) for p in ("host", "device")}
    for t, step in enumerate(plan):
        ids = np.asarray([s for s, _ in step], np.uint32)
        pk = [p for _, p in step]
        res = {}
        for p, g in groups.items():
            zeros = [torch.zeros((4, 288, 352, 4), dtype=torch.uint8, device="cuda") for _ in range(2)]
            outs, errs = g.decode_step_device(pk, outs=zeros, stream_ids=ids, parse=p)
            torch.cuda.synchronize()
            res[p] = ([o.cpu().numpy() for o in outs], errs.copy())
        assert np.array_equal(res["host"][1], res["device"][1])
        for s, e in zip(ids, res["host"][1]):
            if e == 0:
                d, k = int(s) % 2, int(s) // 2
                assert np.array_equal(res["host"][0][d][k], res["device"][0][d][k]), (t, s)


def test_whole_call_failures_change_nothing():
    pk = synth.make_stream(176, 144, 3, 41)
    ref = api.BatchDecoder(2, 176, 144, threads=2)
    dut = api.BatchDecoder(2, 176, 144, threads=2)
    ref.decode_step([pk[0], pk[0]])
    dut.decode_step([pk[0], pk[0]], parse="device")
    with pytest.raises(_lib.H263Error) as e:
        dut.decode_step([pk[1], pk[1]], stream_ids=[1, 1], parse="device")  # a stream named twice
    assert e.value.code == _lib.ERR_BAD_ARGUMENT
    with pytest.raises(_lib.H263Error) as e:
        dut.decode_step([pk[1]], stream_ids=[5], parse="device")  # beyond the context
    assert e.value.code == _lib.ERR_CAPACITY
    with pytest.raises(ValueError):
        dut.decode_step_device_tensor([pk[1], pk[1]], (0, 10), parse="device")  # refused before any parser moves
    for t in (1, 2):
        ea = ref.decode_step([pk[t], pk[t]])
        eb = dut.decode_step([pk[t], pk[t]], parse="device")
        assert not ea.any() and not eb.any()
        ref.ctx.sync(), dut.ctx.sync()
        for s in (0, 1):
            for a, b in zip(ref.ctx.read_yuv(s), dut.ctx.read_yuv(s)):
                assert np.array_equal(a, b)


def test_whole_call_failures_inside_the_device_parse_change_nothing():
    """Failures of the call as a whole once the device parse has begun: a packet of 2^28 bytes (refused by the device
    parse) beside a good one, and the test hook refusing its output capacity after the kernel ran and the host had
    finished the pictures.  Neither moves a parser: the next steps decode as on a decoder that never saw them."""
    pk = synth.make_stream(176, 144, 3, 42)
    ref = api.BatchDecoder(2, 176, 144, threads=2)
    dut = api.BatchDecoder(2, 176, 144, threads=2)
    ref.decode_step([pk[0], pk[0]])
    dut.decode_step([pk[0], pk[0]], parse="device")
    huge = np.zeros(1 << 28, np.uint8)
    huge[: len(pk[1])] = np.frombuffer(pk[1], np.uint8)
    with pytest.raises(_lib.H263Error) as e:
        dut.decode_step([pk[1], huge], parse="device")
    assert e.value.code == _lib.ERR_CAPACITY
    del huge
    # the hook with too small an output: the whole call fails after prepare, kernel and finish
    with pytest.raises(_lib.H263Error) as e:
        frontend.parse_step(dut.parsers, [pk[1], pk[1]], None, 2, mb_cap=10, ctx=dut.ctx)
    assert e.value.code == _lib.ERR_CAPACITY
    for t in (1, 2):
        ea = ref.decode_step([pk[t], pk[t]])
        eb = dut.decode_step([pk[t], pk[t]], parse="device")
        assert not ea.any() and not eb.any()
        ref.ctx.sync(), dut.ctx.sync()
        for s in (0, 1):
            for a, b in zip(ref.ctx.read_yuv(s), dut.ctx.read_yuv(s)):
                assert np.array_equal(a, b)


@pytest.mark.parametrize("w,h,n,seed", [(176, 144, 30, 1), (352, 288, 4, 2)])
def test_oracle_anchor(w, h, n, seed):
    pk = synth.make_stream(w, h, n, seed)
    ref = oracle_decode_stream(pk)
    dec = api.BatchDecoder(1, w, h, threads=1)
    for i, p in enumerate(pk):
        errs = dec.decode_step([p], parse="device")
        assert not errs.any()
        dec.ctx.sync()
        y, cb, cr = dec.ctx.read_yuv(0)
        assert np.array_equal(y, np.asarray(ref[i]["y"]).reshape(-1))
        assert np.array_equal(cb, np.asarray(ref[i]["cb"]).reshape(-1))
        assert np.array_equal(cr, np.asarray(ref[i]["cr"]).reshape(-1))
        assert np.array_equal(dec.ctx.read_rgba(0), np.asarray(ref[i]["rgba"]).reshape(-1))
