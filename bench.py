#!/usr/bin/env python3
"""Headline benchmark: decoded RGBA megapixels/s of the fused reconstruction path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2]; configs[4] at N > 1): S = 1024 concurrent CIF 352x288
synthetic Sorenson-Spark streams PER GPU, one picture per stream per step.  Step 0 is the
I picture; warm-up and timed steps are P pictures with half-pel motion vectors.  A "step"
reconstructs one picture for every stream: inverse RLE + dequant + IDCT + motion
compensation + add/clamp + BT.601 RGBA in ONE kernel launch.  Streams shard by stream over
the GPUs (weak scaling, no collective on the data path; torch.distributed is used only for
the timing barrier and the max-over-ranks reduction).

Numbers in the JSON line:
  value      whole-job MP/s with the side info already resident in HBM (h263cu_step_run),
             timed with CUDA events on the launching stream, max over ranks.
  e2e        same metric through the C ABI with HOST buffers: pinned side info ->
             cudaMemcpyAsync -> kernel -> RGBA copied back to pinned host memory, every
             step, all inside the timed region (h263cu_submit_step_readback).
  roofline   recon kernel: algorithmic bytes per launch / average launch duration
             (per-launch CUDA events) against the measured HBM copy bandwidth.
  cpu_baseline  the oracle (C++ restatement of h263-rs, kind "port": no Rust toolchain
             exists here or on the GPU box) on all host cores, bounded sample, N=1 only.
`--impl reference` times that same CPU restatement step-wise on the same workload.

--dump-outputs DIR writes, after the timed steps, what the timed path computed in its last step for a fixed
sample of DUMP_STREAMS of rank 0's streams: y.npy, cb.npy, cr.npy (planes) and rgba.npy as float32, 36 MB in
all, and stream_ids.npy (float64: each stream's global id, which is its generator seed).  The inputs depend only
on the arguments, so two builds (or the two --impl arms) can be compared array for array.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark runs from a tree that may be read-only and writes nothing into it, bytecode caches included
sys.dont_write_bytecode = True

W, H = 352, 288
MB_PER_PIC = 22 * 18
METRIC = "decoded_rgba_megapixels_per_s"
UNIT = "MP/s"
DUMP_STREAMS = 16  # 16 x (Y + Cb + Cr + RGBA) of a CIF picture in float32: 35.7 MB


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=int(os.environ.get("H263_BENCH_STREAMS", 1024)),
                    help="concurrent streams per GPU")
    ap.add_argument("--unique", type=int, default=int(os.environ.get("H263_BENCH_UNIQUE", 0)),
                    help="unique streams per GPU (0 = all unique); fewer are replicated and disclosed")
    ap.add_argument("--skip-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's planes and RGBA of a fixed sample of streams as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------- workload
def generate_streams(stream_ids, n_pictures, threads, w=W, h=H, **overrides):
    """Returns per-stream (blob, off, len) of synthetic streams, one per GLOBAL stream id (the id
    is the generator seed; every fourth stream uses full-range vectors), generated in parallel
    (ctypes releases the GIL inside the generator)."""
    from h263_rs_b200 import synth

    def one(s):
        kw = dict(mv_mode=0 if s % 4 else 1)
        kw.update(overrides)
        p = synth.default_params(w, h, n_pictures, int(s), **kw)
        return synth.make_stream_blob(p)

    with ThreadPoolExecutor(max_workers=threads) as ex:
        return list(ex.map(one, list(stream_ids)))


def workload_description(streams_per_gpu, unique, n_gpus):
    from h263_rs_b200 import synth

    p = synth.params_dict(synth.default_params(W, H, 0, 0))
    for k in ("width", "height", "n_pictures", "seed"):
        p.pop(k)
    return {
        "workload": "%d concurrent CIF 352x288 synthetic Sorenson Spark streams per GPU, P pictures with half-pel "
                    "MVs, fused MC+IDCT+YUV->RGBA (BASELINE.json configs[2]%s)"
                    % (streams_per_gpu, "; sharded by stream over %d GPUs = configs[4]" % n_gpus if n_gpus > 1 else ""),
        "streams_per_gpu": streams_per_gpu,
        "unique_streams_per_gpu": unique,
        "picture": "%dx%d" % (W, H),
        "l2": "inputs larger than L2: every step touches ~%.0f MB (reference + recon planes + RGBA) per GPU vs 126 MB L2"
              % (streams_per_gpu * W * H * 7 / 1e6),
        "generator": p,
    }


def side_info_stats(pics, mbs, events):
    """Coefficient density of one step (reported with every number, SURVEY.md 7.4-1)."""
    nev = mbs["nev"].astype(np.int64)
    coded_blocks = int((nev > 0).sum())
    inter = (mbs["flags"] & 1) != 0
    coded = (mbs["flags"] & 8) != 0
    return {
        "mbs": int(len(mbs)),
        "events_per_mb": round(float(nev.sum()) / max(len(mbs), 1), 3),
        "blocks_with_coefficients_pct": round(100.0 * coded_blocks / max(len(mbs) * 6, 1), 2),
        "mb_uncoded_pct": round(100.0 * float((inter & ~coded).sum()) / max(len(mbs), 1), 2),
        "mb_intra_pct": round(100.0 * float((~inter).sum()) / max(len(mbs), 1), 2),
        "side_info_bytes": int(len(pics) * 32 + len(mbs) * 24 + len(events) * 2),
    }


def algorithmic_bytes(pics, mbs, events):
    """SURVEY.md 8(d): P picture 7 B/px (1.5 reference read + 1.5 recon write + 4 RGBA write),
    I picture 5.5 B/px, plus the side info actually shipped."""
    px = pics["width"].astype(np.int64) * pics["height"].astype(np.int64)
    is_p = (pics["flags"] & 2) != 0  # HAS_INTER
    return float((px * np.where(is_p, 7.0, 5.5)).sum()) + len(pics) * 32 + len(mbs) * 24 + len(events) * 2


# ---------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t_begin, t_end):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, cmax = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx.append(cmax)
            if t_begin - 0.05 <= ts <= t_end + 0.15:
                sm.append(clk)
                try:
                    power.append(float(f[3]))
                except ValueError:
                    pass
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # region shorter than the sampling period: use the nearest samples
            sm = [float(l.split(",")[1]) for _, l in self.lines[-3:] if len(l.split(",")) > 2]
        return {
            "sm_mhz": float(np.median(sm)) if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "power_w_max": max(power) if power else None,
            "samples_in_region": len(sm),
            "reasons": sorted(reasons),
        }


# ---------------------------------------------------------------------------- CPU arm
def cpu_steps(blobs, step_indices, threads, n_streams, dump_dir=None):
    """Decode the pictures `step_indices` (consecutive, starting at 0) for n_streams streams with
    the oracle, step-wise on `threads` threads.  Returns per-step seconds and pixels; with dump_dir,
    writes the last step's pictures as --dump-outputs does."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O

    L = O.lib()
    batch = L.orc_batch_new(n_streams, 1)
    secs = []
    px = C.c_uint64(0)
    # one contiguous blob per step
    for t in step_indices:
        parts = [blobs[s][0][int(blobs[s][1][t]) : int(blobs[s][1][t]) + int(blobs[s][2][t])] for s in range(n_streams)]
        lens = np.array([len(p) for p in parts], np.uint32)
        offs = np.zeros(n_streams, np.uint64)
        offs[1:] = np.cumsum(lens[:-1], dtype=np.uint64)
        blob = np.concatenate(parts)
        before = px.value
        dt = L.orc_batch_step(batch, blob.ctypes.data, offs.ctypes.data, lens.ctypes.data, 0, threads, C.byref(px), None)
        if dt < 0:
            raise RuntimeError("oracle decode error %d" % int(-dt))
        secs.append((dt, px.value - before))
    if dump_dir:
        def read(s):
            y, cb, cr = np.empty(W * H, np.uint8), np.empty(W * H // 4, np.uint8), np.empty(W * H // 4, np.uint8)
            if L.orc_batch_stream_yuv(batch, s, y.ctypes.data, cb.ctypes.data, cr.ctypes.data):
                raise RuntimeError("oracle has no picture for stream %d" % s)
            return y, cb, cr, O.yuv420_to_rgba(y, cb, cr, W)

        slots = dump_slots(n_streams)
        dump_outputs(dump_dir, slots, slots, read)
    L.orc_batch_free(batch)
    return secs


def run_reference(args, rank):
    """--impl reference: the CPU implementation of the path (the oracle port; the Rust
    reference cannot be built: no toolchain) on all host threads, same workload and metric."""
    if rank != 0:
        return
    threads = host_threads()
    n_streams = args.streams
    total = args.warmup + args.steps + 1
    t0 = time.time()
    blobs = generate_streams(range(n_streams), total, threads)
    gen_s = time.time() - t0
    secs = cpu_steps(blobs, range(total), threads, n_streams, args.dump_outputs)
    timed = secs[1 + args.warmup :]
    t = sum(s for s, _ in timed)
    px = sum(p for _, p in timed)
    value = px / t / 1e6
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32+u8", "data": "synthetic",
        "config": workload_description(n_streams, n_streams, args.gpus),
        "cpu_baseline": {
            "value": value, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d timed steps x %d CIF streams (full parse + recon + RGBA per picture), one stream per task on %d "
                      "host threads; C++ restatement of h263-rs (g++ -O2 -ffp-contract=off), not the Rust build"
                      % (args.steps, n_streams, threads),
        },
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "setup_s": {"generate": round(gen_s, 2)},
    }
    emit(out)


# ---------------------------------------------------------------------------- GPU arm
def run_ours(args, rank, world, local_rank, dist):
    import torch

    from h263_rs_b200 import _lib, api, frontend, shard

    # each rank keeps its parser threads and its pinned staging on the socket its GPU hangs off
    placement = shard.bind_rank_to_gpu_node(local_rank, world) if world > 1 else {"numa_node": None, "cpus": None}
    threads = placement["cpus"] or max(1, host_threads() // max(world, 1))
    S = args.streams
    U = args.unique if args.unique and args.unique < S else S
    total = args.warmup + args.steps + 1  # step 0 = I pictures
    L = _lib.lib()
    torch.cuda.set_device(local_rank)
    ctx = api.Context(local_rank, S, W, H)

    # ---- setup (untimed): generate, parse (threaded), stage in pinned memory, upload
    t0 = time.time()
    # shard by stream: this rank owns the global streams s with s % world == rank (shard.py)
    gids = shard.shard_streams(S * world, world, rank)
    blobs = generate_streams(gids[:U], total, threads)
    gen_s = time.time() - t0
    parsers = [frontend.Parser(1) for _ in range(S)]
    host_steps, steps = [], []
    parse_s = 0.0
    parse_px = 0
    for t in range(total):
        packets = []
        for s in range(S):
            b, off, ln = blobs[s % U]
            packets.append(b[int(off[t]) : int(off[t]) + int(ln[t])].tobytes())
        tp = time.time()
        pics, mbs, events, errs, _ = frontend.parse_step(parsers, packets, np.arange(S, dtype=np.uint32), threads,
                                                         mb_cap=S * MB_PER_PIC)
        parse_s += time.time() - tp
        parse_px += S * W * H
        assert not errs.any(), "synthetic stream failed to parse"
        # pinned copies of the side info (what a streaming caller hands to the C ABI)
        pinned = []
        for arr in (pics, mbs, events):
            nbytes = max(arr.nbytes, 16)
            ptr = L.h263cu_alloc_pinned(nbytes)
            assert ptr, "cudaHostAlloc failed"
            C.memmove(ptr, arr.ctypes.data, arr.nbytes)
            pinned.append(ptr)
        host_steps.append((pinned, len(pics), len(mbs), len(events), pics.copy()))
        err = C.c_int(0)
        st = L.h263cu_step_upload(ctx.h, pinned[0], len(pics), pinned[1], len(mbs), pinned[2], len(events), C.byref(err))
        assert st, "step upload failed: %d" % err.value
        steps.append(st)
        if t == total - 1:
            stats = side_info_stats(pics, mbs, events)
            alg_bytes = algorithmic_bytes(pics, mbs, events)
    ctx.sync()
    setup = {"generate": round(gen_s, 2), "parse": round(parse_s, 2)}

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    def reduce_max(v):
        return shard.reduce_max(dist, v, "cuda")

    def reduce_sum(v):
        return shard.reduce_sum(dist, v, "cuda")

    # ---- value: side info resident in HBM, CUDA-event timed, per-launch kernel timing
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    for t in range(1 + args.warmup):
        ctx.step_run(steps[t], _lib.OUT_RGBA)
    barrier()
    launches_before = ctx.launch_count()
    t_begin = time.time()
    ctx.timer_start()
    for t in range(1 + args.warmup, total):
        ctx.step_run(steps[t], _lib.OUT_RGBA)
    ms = ctx.timer_stop()
    barrier()
    t_end = time.time()
    gpu_launches = ctx.launch_count() - launches_before
    clocks = sampler.stop(t_begin, t_end)
    ms_max = reduce_max(ms)
    px_step_rank = S * W * H
    px_total = reduce_sum(float(px_step_rank * args.steps))
    value = px_total / (ms_max * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:  # before anything below runs more steps on these streams
        slots = dump_slots(S)
        dump_outputs(args.dump_outputs, slots, gids[slots % U], lambda s: (*ctx.read_yuv(s), ctx.read_rgba(s)))

    # parity in the same job, on EVERY rank: device checksums of the final pictures of this rank's first streams vs the
    # oracle; rank 0 gathers the verdicts (shard.gather_to_rank0)
    parity = None
    if not args.skip_extras:
        n_check = min(U, 4 if world == 1 else 2)
        mine = parity_check(ctx, blobs, total, n_check)
        parts = shard.gather_to_rank0(dist, np.array([int(mine["bit_exact_vs_oracle"]), n_check], np.uint64), world, rank, "cuda")
        if rank == 0:
            parity = {"streams_checked_per_rank": n_check, "pictures_each": total, "ranks": world,
                      "bit_exact_vs_oracle_per_rank": [bool(p[0]) for p in parts],
                      "bit_exact_vs_oracle": all(bool(p[0]) for p in parts),
                      "global_stream_ids_checked": [int(g) for r in range(world) for g in shard.shard_streams(S * world, world, r)[:n_check]]}

    # ---- the same steps once more with a pair of CUDA events around every launch: the recon kernel's own duration.
    # Kept out of the timed region above: the event pairs cost ~5 us per step and keep consecutive launches from
    # overlapping at their edges (the timed region runs 2 % faster without them).
    ctx.profile_enable(True)
    ctx.profile_read()
    ctx.timer_start()
    for t in range(1 + args.warmup, total):
        ctx.step_run(steps[t], _lib.OUT_RGBA)
    ms_prof = ctx.timer_stop()
    prof = ctx.profile_read()
    ctx.profile_enable(False)

    # ---- sustained: the same resident steps replayed back to back for >= 2 s with the clock sampler running: does the
    # short timed region above hold at the clocks the part settles at under a long load?
    sustained = None
    if not args.skip_extras:
        timed_steps = list(range(1 + args.warmup, total))
        rounds = max(1, int(2.2 / max(ms * 1e-3, 1e-6)))
        s2 = ClockSampler(local_rank)
        s2.start()
        time.sleep(0.3)
        barrier()
        ts0 = time.time()
        ctx.timer_start()
        for _ in range(rounds):
            for t in timed_steps:
                ctx.step_run(steps[t], _lib.OUT_RGBA)
        ms_sus = ctx.timer_stop()
        barrier()
        ts1 = time.time()
        clk2 = s2.stop(ts0, ts1)
        ms_sus_max = reduce_max(ms_sus)
        n_sus = rounds * len(timed_steps)
        sustained = {"seconds": ms_sus_max * 1e-3, "steps": n_sus, "ms_per_step": ms_sus_max / n_sus,
                     "value": px_step_rank * world * n_sus / (ms_sus_max * 1e-3) / 1e6, "unit": UNIT, "clocks": clk2,
                     "vs_short_region": (ms_max / max(args.steps, 1)) / (ms_sus_max / n_sus),
                     "note": "the timed steps replayed %d times back to back (P pictures on top of P pictures: the same "
                             "work per step); vs_short_region = short-region ms per step / sustained ms per step" % rounds}

    # ---- e2e: host buffers through the C ABI, H2D + kernel + D2H(RGBA) inside the timed region
    rgba_bytes = S * W * H * 4
    host_out = [L.h263cu_alloc_pinned(rgba_bytes) for _ in range(2)]
    assert all(host_out), "cudaHostAlloc for the RGBA read-back failed"

    def e2e_step(t):
        pinned, npics, nmbs, nun, _ = host_steps[t]
        _lib.check(L.h263cu_submit_step_readback(ctx.h, pinned[0], npics, pinned[1], nmbs, pinned[2], nun, _lib.OUT_RGBA,
                                                 host_out[t & 1], None))

    for t in range(1 + args.warmup):
        e2e_step(t)
    barrier()
    te = time.perf_counter()
    for t in range(1 + args.warmup, total):
        e2e_step(t)
    ctx.sync()
    e2e_s = time.perf_counter() - te
    barrier()
    e2e_max = reduce_max(e2e_s)
    e2e_value = px_total / e2e_max / 1e6
    # ---- e2e from the bitstream: packets in host memory -> h263cu_decode_step (threaded VLC parse into pinned
    # staging, H2D of the side info, kernel, D2H of the RGBA), the parse of step t+1 overlapping the device work
    # of step t.  This is the batched form of the reference's decode_next_picture + yuv420_to_rgba.
    dec = api.BatchDecoder(S, W, H, threads=threads, ctx=ctx)
    plans = []
    bitstream_bytes = 0
    for t in range(total):
        views = []
        for s in range(S):
            b, off, ln = blobs[s % U]
            views.append(b[int(off[t]) : int(off[t]) + int(ln[t])])
        plans.append(dec.plan_step(views))
        if t > args.warmup:
            bitstream_bytes += sum(v.size for v in views)
    pic_bytes = W * H * 4
    for t in range(1 + args.warmup):
        assert not dec.decode_planned(plans[t], _lib.OUT_RGBA, host_out[t & 1], pic_bytes).any()
    barrier()
    tb = time.perf_counter()
    for t in range(1 + args.warmup, total):
        dec.decode_planned(plans[t], _lib.OUT_RGBA, host_out[t & 1], pic_bytes)
    ctx.sync()
    bit_s = time.perf_counter() - tb
    barrier()
    bit_max = reduce_max(bit_s)
    bit_value = px_total / bit_max / 1e6
    bit_ok = None
    if rank == 0 and not args.skip_extras:
        last = np.ctypeslib.as_array(C.cast(host_out[(total - 1) & 1], C.POINTER(C.c_uint8)), shape=(rgba_bytes,))
        bit_ok = bool(np.array_equal(last[: W * H * 4], ctx.read_rgba(0)))
    # parse alone (same threads, same packets, fresh parsers): the host side of the pipeline
    dec2 = api.BatchDecoder(S, W, H, threads=threads, ctx=ctx)
    plans2 = [dict(p, parsers=(C.c_void_p * S)(*[q.h for q in dec2.parsers])) for p in plans]
    pinned_parse = [L.h263cu_alloc_pinned(n) for n in (S * 32, S * MB_PER_PIC * 24, 64 * 1024 * 1024)]
    assert all(pinned_parse), "cudaHostAlloc failed"
    npk, nmk, nuk = C.c_uint32(), C.c_uint32(), C.c_uint32()
    tp0 = 0.0
    for t in range(total):
        q = plans2[t]
        t0p = time.perf_counter()
        _lib.check(L.h263cu_parse_step(q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, S, threads, pinned_parse[0],
                                       pinned_parse[1], S * MB_PER_PIC, pinned_parse[2], 32 * 1024 * 1024, C.byref(npk),
                                       C.byref(nmk), C.byref(nuk), None, None))
        if t > args.warmup:
            tp0 += time.perf_counter() - t0p
    for p_ in pinned_parse:
        L.h263cu_free_pinned(p_)
    parse_only = {"value": px_step_rank * args.steps / tp0 / 1e6, "unit": UNIT, "threads": threads,
                  "ms_per_step": 1e3 * tp0 / max(args.steps, 1),
                  "note": "h263cu_parse_step alone on this rank's %d streams: serial VLC parse per stream, threaded across "
                          "streams, output packed into pinned memory" % S}
    h2d = int(np.mean([32 * a + 24 * b + 2 * c for _, a, b, c, _ in host_steps[1 + args.warmup :]]))
    e2e_ok = None
    if rank == 0 and not args.skip_extras:
        # the last read-back buffer holds the final step: compare stream 0 with the device copy
        last = np.ctypeslib.as_array(C.cast(host_out[(total - 1) & 1], C.POINTER(C.c_uint8)), shape=(rgba_bytes,))
        e2e_ok = bool(np.array_equal(last[: W * H * 4], ctx.read_rgba(0)))

    # ---- extras (rank 0, N=1): CPU baseline on a bounded sample, host parse rate, single stream
    cpu_baseline = None
    extras = {}
    if rank == 0 and world == 1:
        n_cpu = host_threads()
        # bounded sample: ~10-20 s of CPU work (one CIF picture costs the port ~1.5 ms of one core); a short run leaves
        # fewer pictures for it, at least one of them timed
        warm = min(2, total - 2)
        timed_steps = min(10, total - 1 - warm)
        sample_steps = 1 + warm + timed_steps  # I + warm + timed
        sample_streams = min(U, 768)
        secs = cpu_steps(blobs, range(sample_steps), n_cpu, sample_streams)
        tt = sum(s for s, _ in secs[1 + warm :])
        pp = sum(p for _, p in secs[1 + warm :])
        cpu_baseline = {
            "value": pp / tt / 1e6, "unit": UNIT, "cores": n_cpu, "kind": "port",
            "sample": "%d timed steps x %d CIF streams of the same workload (full parse + recon + RGBA, %.1f s of CPU "
                      "work), %d host threads; C++ restatement of h263-rs, not the Rust build (no Rust toolchain)"
                      % (timed_steps, sample_streams, tt * n_cpu, n_cpu),
        }
        if not args.skip_extras:
            extras["single_stream_config2"] = single_stream(api, frontend, local_rank)
            extras["config4_4cif_deblock"] = config4_deblock(api, frontend, local_rank, threads)
            extras["stateless_drop_ins"] = stateless_drop_ins(api)

    for st in steps:
        L.h263cu_step_free(ctx.h, st)
    for p in host_out:
        L.h263cu_free_pinned(p)
    for pinned, *_ in host_steps:
        for p in pinned:
            L.h263cu_free_pinned(p)

    if rank != 0:
        return
    peaks = measured_peaks()
    # One recon launch per step and nothing else on the stream: timed region / launches is the kernel's average launch
    # duration including the launch gaps, i.e. an upper bound of what a pair of events around each launch reports.
    kernel_ms = ms / max(int(gpu_launches), 1)
    kernel_ms_events = prof["recon_ms"] / max(prof["recon_launches"], 1)
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32+u8", "data": "synthetic",
        "config": dict(workload_description(S, U, world), side_info=stats),
        "frames_per_s": value * 1e6 / (W * H),
        "e2e": {"value": bit_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": rgba_bytes,
                "ms_per_step": 1e3 * bit_max / max(args.steps, 1), "readback_matches_device": bit_ok,
                "bitstream_bytes_per_step": int(bitstream_bytes / max(args.steps, 1)), "parse_threads": threads, "host_placement": placement,
                "path": "h263cu_decode_step: bitstream packets in host memory -> threaded VLC parse into pinned staging -> "
                        "H2D side info -> recon kernel -> D2H RGBA into pinned host memory, steps pipelined"},
        "e2e_from_side_info": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": rgba_bytes,
                               "ms_per_step": 1e3 * e2e_max / max(args.steps, 1), "readback_matches_device": e2e_ok,
                               "path": "h263cu_submit_step_readback on pre-parsed pinned side info (no host parse in the timed region)"},
        "host_parse": parse_only,
        "gpu_launches": int(gpu_launches),
        "roofline": {
            "bound": "hbm", "kernel": "recon_kernel", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": achieved / peaks["hbm_gbs"], "peak_source": peaks["source"], "traffic": ncu_traffic(),
            "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kernel_ms, "kernel_launches_timed": int(gpu_launches),
            "kernel_ms_source": "CUDA events around the timed region / launches in it (one recon launch per step, nothing "
                                "else on the stream): includes launch gaps",
            "kernel_ms_per_launch_events": kernel_ms_events,
            "kernel_share_of_step": (prof["recon_ms"] / ms_prof) if ms_prof > 0 else None,
            "per_launch_events_note": "second pass over the same steps with an event pair around every launch (%d launches, "
                                      "%.4f ms per step in that pass)" % (prof["recon_launches"], ms_prof / max(args.steps, 1)),
            "frac_of_nominal_8TBs": achieved / 8000.0,
            "frac_sustained": (alg_bytes / (sustained["ms_per_step"] * 1e-3) / 1e9 / peaks["hbm_gbs"]) if sustained else None,
            "traffic_source": "static: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture "
                              "profiles/recon_ncu_summary.json (not measured in this run)",
        },
        "sustained": sustained,
        "cpu_baseline": cpu_baseline,
        "clocks": clocks,
        "parity": parity,
        "setup_s": setup,
    }
    out.update(extras)
    c4 = extras.get("config4_4cif_deblock")
    if c4:
        # SURVEY.md 8(d): deblocking adds 0 algorithmic bytes (ideal fusion): 7 B/px for a P picture + side info
        out["roofline_config4"] = {
            "bound": "hbm", "kernel": "recon_tile_kernel + deblock_rgba_tile_kernel (one step = both launches)",
            "achieved": c4["algorithmic_bytes_per_step"] / (c4["ms_per_step"] * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": c4["algorithmic_bytes_per_step"] / (c4["ms_per_step"] * 1e-3) / 1e9 / peaks["hbm_gbs"], "peak_source": peaks["source"],
            "algorithmic_bytes_per_step": c4["algorithmic_bytes_per_step"], "ms_per_step": c4["ms_per_step"],
            "traffic": None}
    emit(out)


def parity_check(ctx, blobs, total, n_check):
    """Bit-exactness evidence inside the bench job: decode a few of the benchmark's own
    streams with the oracle and compare plane / RGBA checksums of the final picture."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    from helpers import weighted_sum

    ok = True
    sums = ctx.checksums(np.arange(n_check))
    for s in range(n_check):
        st = O.OracleState(1)
        b, off, ln = blobs[s]
        for t in range(total):
            st.decode_next_picture(b[int(off[t]) : int(off[t]) + int(ln[t])].tobytes())
        y, cb, cr = st.yuv()
        rgba = O.yuv420_to_rgba(y, cb, cr, W)
        exp = [weighted_sum(y), weighted_sum(cb), weighted_sum(cr), weighted_sum(rgba)]
        ok &= [int(v) for v in sums[s]] == exp
    return {"streams_checked": n_check, "pictures_each": total, "bit_exact_vs_oracle": bool(ok)}


def dump_slots(n_streams):
    """The streams --dump-outputs writes: a seeded sample that depends only on the number of streams."""
    return np.sort(np.random.default_rng(0).choice(n_streams, size=min(DUMP_STREAMS, n_streams), replace=False))


def dump_outputs(out_dir, slots, stream_ids, read):
    """Writes the last step's pictures of `slots`; read(slot) returns flat uint8 (y, cb, cr, rgba) of a CIF picture."""
    pics = [read(int(s)) for s in slots]
    k = len(pics)
    shapes = {"y": (k, H, W), "cb": (k, H // 2, W // 2), "cr": (k, H // 2, W // 2), "rgba": (k, H, W, 4)}
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "stream_ids.npy"), np.asarray(stream_ids, np.float64))
    for i, (name, shape) in enumerate(shapes.items()):
        np.save(os.path.join(out_dir, name + ".npy"), np.stack([p[i] for p in pics]).reshape(shape).astype(np.float32))


def single_stream(api, frontend, device):
    """BASELINE.json configs[1]: ONE CIF stream, 300 pictures -- launch-latency bound."""
    from h263_rs_b200 import _lib, synth

    n = 300
    packets = synth.make_stream(W, H, n, 2, mv_mode=1)
    ps = frontend.Parser(1)
    ctx = api.Context(device, 1, W, H)
    steps = []
    for pk in packets:
        pic, mbs, ev = ps.parse_picture(pk)
        steps.append(ctx.step_upload(pic, mbs, ev))
    ctx.sync()
    for st in steps[:20]:
        ctx.step_run(st, _lib.OUT_RGBA)
    ctx.sync()
    ctx.timer_start()
    for st in steps[20:]:
        ctx.step_run(st, _lib.OUT_RGBA)
    ms = ctx.timer_stop()
    fps = (n - 20) / (ms * 1e-3)
    # the same 280 resident steps as ONE CUDA graph: one launch call instead of 280
    g = ctx.graph_build(steps[20:], _lib.OUT_RGBA)
    ctx.graph_launch(g)
    ctx.sync()
    ctx.timer_start()
    ctx.graph_launch(g)
    ms_graph = ctx.timer_stop()
    ctx.graph_free(g)
    graph_fps = (n - 20) / (ms_graph * 1e-3)
    for st in steps:
        ctx.step_free(st)
    ctx.close()
    # the same stream the way a player drives the reference: H263State::decode_next_picture per packet, then the RGBA
    # of that picture in host memory before the next packet is touched (parse + upload + kernel + read-back, serial)
    state = api.H263State(device=device)
    for pk in packets[:20]:
        state.decode_next_picture(pk)
        state.get_last_rgba()
    t0 = time.perf_counter()
    for pk in packets[20:]:
        state.decode_next_picture(pk)
        rgba = state.get_last_rgba()
    sync_s = time.perf_counter() - t0
    assert rgba.size == W * H * 4
    # and the CPU port on one core, same packets, planes + RGBA per picture
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O

    ost = O.OracleState(1)
    for pk in packets[:20]:
        ost.decode_next_picture(pk)
    t0 = time.perf_counter()
    for pk in packets[20:]:
        ost.decode_next_picture(pk)
        y, cb, cr = ost.yuv()
        O.yuv420_to_rgba(y, cb, cr, W)
    cpu_s = time.perf_counter() - t0
    # pipelined API: packet t + 1 is handed in before picture t is consumed (parse of t + 1 overlaps the device work of t,
    # the RGBA of t arrives in one of two pinned buffers); every picture's RGBA is still touched on the host
    pst = api.H263State(device=device, pipelined=True)
    for pk in packets[:20]:
        pst.decode_next_picture(pk)
    pst.get_last_rgba(copy=False)
    t0 = time.perf_counter()
    acc = 0
    for pk in packets[20:]:
        prev = pst.get_last_rgba(copy=False)
        pst.decode_next_picture(pk)
        acc += int(prev[0]) + int(prev[-1])
    last = pst.get_last_rgba(copy=False)
    pipe_s = time.perf_counter() - t0
    pipe_ok = bool(np.array_equal(last, rgba))
    pipe_fps = (n - 20) / pipe_s
    # the same through the C ABI from native code (tools/single_stream_bench.cpp): what a Rust / C caller gets
    native = None
    try:
        exe = os.path.join(ROOT, "h263_rs_b200", "single_stream_bench.bin")
        r = subprocess.run([exe, os.path.join(ROOT, "h263_rs_b200"), str(device)], capture_output=True, text=True, timeout=120)
        native = json.loads(r.stdout) if r.returncode == 0 else {"error": r.stderr[-300:]}
    except Exception as e:  # the tool is optional evidence, never a reason to lose the bench line
        native = {"error": repr(e)}
    sync_fps, cpu_fps = (n - 20) / sync_s, (n - 20) / cpu_s
    return {"frames_per_s": fps, "value": fps * W * H / 1e6, "unit": UNIT, "pictures": n,
            "note": "one dependent kernel launch per picture (396 macroblocks): latency bound, not a roofline case",
            "resident_cuda_graph": {"frames_per_s": graph_fps, "value": graph_fps * W * H / 1e6, "unit": UNIT, "us_per_picture": ms_graph * 1e3 / (n - 20),
                                    "note": "the same resident steps captured into one CUDA graph (h263cu_graph_build / _launch)"},
            "synchronous_api": {"frames_per_s": sync_fps, "value": sync_fps * W * H / 1e6, "unit": UNIT,
                                "us_per_picture": sync_s / (n - 20) * 1e6,
                                "path": "H263State.decode_next_picture + get_last_rgba per packet (host parse, H2D, kernel, "
                                        "D2H of 405 504 bytes, all serial), Python caller"},
            "pipelined_api": {"frames_per_s": pipe_fps, "value": pipe_fps * W * H / 1e6, "unit": UNIT, "us_per_picture": pipe_s / (n - 20) * 1e6,
                              "last_picture_matches_synchronous": pipe_ok,
                              "path": "H263State(pipelined=True): decode_next_picture(packet t+1) queued before picture t's RGBA is "
                                      "consumed (h263cu_readback_wait), two pinned buffers alternate, Python caller"},
            "native_c_abi": native,
            "cpu_port_one_core": {"frames_per_s": cpu_fps, "value": cpu_fps * W * H / 1e6, "unit": UNIT,
                                  "note": "oracle (C++ restatement of h263-rs) on one host core, same packets, planes + RGBA"}}


def config4_deblock(api, frontend, device, threads, n_streams=256, n_steps=6):
    """BASELINE.json configs[3]: 256 concurrent 4CIF 704x576 streams, deblocking flag set, vectors
    biased across the picture borders; recon kernel + fused deblock/RGBA kernel per step."""
    from h263_rs_b200 import _lib

    w, h = 704, 576
    blobs = generate_streams(range(n_streams), 1 + n_steps, threads, w, h, mv_mode=2, deblock_flag=1)
    ctx = api.Context(device, n_streams, w, h)
    parsers = [frontend.Parser(1) for _ in range(n_streams)]
    steps = []
    for t in range(1 + n_steps):
        packets = [b[int(off[t]) : int(off[t]) + int(ln[t])].tobytes() for b, off, ln in blobs]
        pics, mbs, events, errs, _ = frontend.parse_step(parsers, packets, np.arange(n_streams, dtype=np.uint32), threads,
                                                         mb_cap=n_streams * 44 * 36)
        assert not errs.any()
        steps.append(ctx.step_upload(pics, mbs, events))
        alg = algorithmic_bytes(pics, mbs, events)
    flags = _lib.OUT_RGBA | _lib.OUT_DEBLOCK
    ctx.sync()
    for st in steps[:3]:
        ctx.step_run(st, flags)
    ctx.profile_enable(True)
    ctx.profile_read()
    ctx.timer_start()
    for st in steps[3:]:
        ctx.step_run(st, flags)
    ms = ctx.timer_stop()
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    # parity: stream 0 against the oracle with the deblocking post-filter
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import oracle_decode_stream

    b, off, ln = blobs[0]
    ref = oracle_decode_stream([b[int(off[t]) : int(off[t]) + int(ln[t])].tobytes() for t in range(1 + n_steps)], deblock=True)
    ok = bool(np.array_equal(ctx.read_rgba(0), ref[-1]["rgba"]))
    for st in steps:
        ctx.step_free(st)
    ctx.close()
    n = n_steps - 2
    px = n_streams * w * h * n
    return {"value": px / (ms * 1e-3) / 1e6, "unit": UNIT, "frames_per_s": n_streams * n / (ms * 1e-3), "streams": n_streams,
            "picture": "704x576", "ms_per_step": ms / n, "algorithmic_bytes_per_step": alg, "recon_ms_per_step": prof["recon_ms"] / max(prof["recon_launches"], 1),
            "deblock_rgba_ms_per_step": prof["deblock_ms"] / max(prof["deblock_launches"], 1),
            "bit_exact_vs_oracle_stream0": ok,
            "note": "P pictures, deblock::deblock on Y/Cb/Cr (QUANT_TO_STRENGTH[PQUANT]) fused with RGBA in a second kernel"}


def stateless_drop_ins(api):
    """The literal replacements of yuv::bt601::yuv420_to_rgba and deblock::deblock (host planes in, host planes out, one
    picture per call: pinned staging, own stream) beside the oracle's versions on one core.  A single CIF picture is a
    latency case, not a throughput case: the numbers say what a caller that swaps the sibling crates alone gets."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O

    rng = np.random.default_rng(3)
    out = {}
    for name, (w, h) in (("cif", (352, 288)), ("4cif", (704, 576))):
        y = rng.integers(0, 256, w * h).astype(np.uint8)
        cb = rng.integers(0, 256, (w // 2) * (h // 2)).astype(np.uint8)
        cr = rng.integers(0, 256, (w // 2) * (h // 2)).astype(np.uint8)
        res = {}
        for label, fy, fd in (("gpu", api.yuv420_to_rgba, api.deblock), ("cpu_port_one_core", O.yuv420_to_rgba, O.deblock)):
            for _ in range(3):
                a = fy(y, cb, cr, w)
                b = fd(y, w, 5)
            n = 30
            t0 = time.perf_counter()
            for _ in range(n):
                a = fy(y, cb, cr, w)
            t1 = time.perf_counter()
            for _ in range(n):
                b = fd(y, w, 5)
            t2 = time.perf_counter()
            res[label] = {"yuv420_to_rgba_us": (t1 - t0) / n * 1e6, "deblock_plane_us": (t2 - t1) / n * 1e6}
            res[label + "_out"] = (a, b)
        res["bit_exact"] = bool(np.array_equal(res["gpu_out"][0], res["cpu_port_one_core_out"][0]) and
                                np.array_equal(res["gpu_out"][1], res["cpu_port_one_core_out"][1]))
        del res["gpu_out"], res["cpu_port_one_core_out"]
        out[name] = res
    return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return {"hbm_gbs": float(json.load(open(p))["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json)"}
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic():
    """dram bytes read+written per recon launch from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", "recon_ncu_summary.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


_REAL_STDOUT = None


def guard_stdout():
    """The contract is ONE JSON line on stdout.  Libraries underneath (NCCL's version banner, CUDA warnings) write to
    file descriptor 1 as well: keep the real stdout aside and point fd 1 at stderr for the rest of the run."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(obj):
    line = json.dumps(obj)
    if _REAL_STDOUT is not None:
        _REAL_STDOUT.write(line + "\n")
        _REAL_STDOUT.flush()
    else:
        print(line)


def main():
    args = parse_args()
    guard_stdout()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod

        torch.cuda.set_device(local_rank)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod
    try:
        run_ours(args, rank, world, local_rank, dist)
    finally:
        if dist is not None:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
