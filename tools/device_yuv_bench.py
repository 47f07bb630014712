#!/usr/bin/env python3
"""End-to-end decode from the bitstream with the decoded planes (I420 / NV12) left on the GPU, against device RGBA.

    python tools/device_yuv_bench.py [--gpus N] [--steps K] [--warmup W] [--rounds R] [--out profiles/<name>.json]

bench.py's workload (1024 CIF 352x288 streams per GPU, the same generator and parameters, its helpers imported), the
same parser thread count (all host cores), P pictures timed.  In one run, alternating round by round on ONE context
(or group), it measures:
  (a) MP/s from the bitstream into preallocated torch tensors on the GPU, for each output:
        rgba          h263cu_decode_step_device (the existing device path: the in-run baseline)
        i420          h263cu_decode_step_device_yuv, I420
        nv12          h263cu_decode_step_device_yuv, NV12
        i420_deblock  h263cu_decode_step_device_yuv, I420 with H263CU_OUT_DEBLOCK
  (b) h263cu_parse_step alone (the host parse, same threads and packets), MP/s
  (c) the recon kernel's ms per launch for each output, and the deblock kernel's for i420_deblock
      (h263cu_profile_enable/read), in separate profiled passes
and writes one JSON with the GPU name and power limit beside the numbers.  --gpus N runs the group form
(h263cu_group_* over N devices, N x 1024 streams).  Exits non-zero without a GPU.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (the workload: generate_streams, host_threads, W, H, MB_PER_PIC)

ARMS = ("rgba", "i420", "nv12", "i420_deblock")


def gpu_facts():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines() if q.returncode == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--streams", type=int, default=1024, help="streams per GPU")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_device_yuv_bench.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available() or torch.cuda.device_count() < args.gpus:
        sys.exit("device_yuv_bench: needs %d CUDA device(s), found %d" % (args.gpus, torch.cuda.device_count() if torch.cuda.is_available() else 0))
    from h263_rs_b200 import _lib, api

    L = _lib.lib()
    W, H = bench.W, bench.H
    G, S = args.gpus, args.streams
    N = G * S
    threads = bench.host_threads()
    total = 1 + args.warmup + args.steps
    blobs = bench.generate_streams(range(N), total, threads)
    if G == 1:
        dec = api.BatchDecoder(S, W, H, threads=threads)
        ctxs, parsers = [dec.ctx], dec.parsers
    else:
        dec = api.DeviceGroup(list(range(G)), S, W, H, threads=threads)
        ctxs, parsers = dec.ctxs, dec.parsers
    plans = []
    for t in range(total):
        views = [blobs[s][0][int(blobs[s][1][t]) : int(blobs[s][1][t]) + int(blobs[s][2][t])] for s in range(N)]
        plans.append(dec.plan_step(views))
    # destinations: preallocated tight tensors per device; the consumer stream is torch's current one
    rgba = [torch.empty((S, H, W, 4), dtype=torch.uint8, device="cuda:%d" % d) for d in range(G)]
    rgba_t = (_lib.DeviceRgba * G)(*[_lib.DeviceRgba(o.data_ptr(), W * 4, W * H * 4, W, H,
                                                     torch.cuda.current_stream(d).cuda_stream or None) for d, o in enumerate(rgba)])
    planes, yuv_t = {}, {}
    for layout in ("i420", "nv12"):
        pairs = [api._device_yuv(None, S, W, H, d, layout) for d in range(G)]
        planes[layout] = [p for p, _ in pairs]
        yuv_t[layout] = (_lib.DeviceYuv * G)(*[t for _, t in pairs])
    nd = C.c_uint32(0)

    def step(t, arm):
        q = plans[t]
        if arm == "rgba":
            if G == 1:
                _lib.check(L.h263cu_decode_step_device(dec.ctx.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, q["n"],
                                                       threads, _lib.OUT_RGBA, rgba_t, q["errs"].ctypes.data, C.byref(nd)))
            else:
                _lib.check(L.h263cu_group_decode_step_device(dec.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, q["n"],
                                                             _lib.OUT_RGBA, rgba_t, q["errs"].ctypes.data, C.byref(nd)))
        else:
            target = yuv_t["nv12" if arm == "nv12" else "i420"]
            flags = _lib.OUT_DEBLOCK if arm == "i420_deblock" else 0
            if G == 1:
                _lib.check(L.h263cu_decode_step_device_yuv(dec.ctx.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, q["n"],
                                                           threads, flags, target, q["errs"].ctypes.data, C.byref(nd)))
            else:
                _lib.check(L.h263cu_group_decode_step_device_yuv(dec.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data,
                                                                 q["n"], flags, target, q["errs"].ctypes.data, C.byref(nd)))
        assert not q["errs"].any()

    def sync():
        for c in ctxs:
            c.sync()
        for d in range(G):
            torch.cuda.synchronize(d)

    def run(arm, profile=False):
        """One pass over the stream from its I picture: untimed warm-up steps, then the timed P steps."""
        for p in parsers:
            p.reset()
        for t in range(1 + args.warmup):
            step(t, arm)
        sync()
        if profile:
            for c in ctxs:
                c.profile_enable(True)
                c.profile_read()
        t0 = time.perf_counter()
        for t in range(1 + args.warmup, total):
            step(t, arm)
        sync()
        sec = time.perf_counter() - t0
        prof = None
        if profile:
            rs = [c.profile_read() for c in ctxs]
            for c in ctxs:
                c.profile_enable(False)
            prof = (sum(r["recon_ms"] for r in rs) / max(sum(r["recon_launches"] for r in rs), 1),
                    sum(r["deblock_ms"] for r in rs) / max(sum(r["deblock_launches"] for r in rs), 1))
        return sec, prof

    px = float(N) * W * H * args.steps
    res = {a: [] for a in ARMS}
    for _ in range(args.rounds):
        for arm in ARMS:
            res[arm].append(px / run(arm)[0] / 1e6)
    # result checks on the last step: NV12 holds I420's samples interleaved, and the I420 planes of a sample of streams
    # equal the context's planes (h263cu_read_yuv)
    run("i420")
    i420 = [[p.clone() for p in planes["i420"][d]] for d in range(G)]
    yuv_same = True
    for s in range(0, S, max(S // 16, 1)):
        for d in range(G):
            y, cb, cr = ctxs[d].read_yuv(s)
            got = [p[s].cpu().numpy().reshape(-1) for p in i420[d]]
            yuv_same &= all(np.array_equal(a, np.asarray(b).reshape(-1)) for a, b in zip(got, (y, cb, cr)))
    run("nv12")
    nv12_same = all(torch.equal(planes["nv12"][d][0], i420[d][0]) and torch.equal(planes["nv12"][d][1][..., 0], i420[d][1])
                    and torch.equal(planes["nv12"][d][1][..., 1], i420[d][2]) for d in range(G))
    # (c) kernels per launch
    kern = {a: [] for a in ARMS}
    deb = []
    for _ in range(args.rounds):
        for arm in ARMS:
            r, db = run(arm, profile=True)[1]
            kern[arm].append(r)
            if arm == "i420_deblock":
                deb.append(db)
    # (b) host parse alone on fresh parsers, same packets and threads
    fresh = [type(parsers[0])(1) for _ in range(N)]
    pinned = [L.h263cu_alloc_pinned(n) for n in (N * 32, N * bench.MB_PER_PIC * 24, 128 * 1024 * 1024)]
    assert all(pinned)
    npk, nmk, nuk = C.c_uint32(), C.c_uint32(), C.c_uint32()
    parser_arr = (C.c_void_p * N)(*[p.h for p in fresh])
    tp = 0.0
    for t in range(total):
        q = plans[t]
        t0 = time.perf_counter()
        _lib.check(L.h263cu_parse_step(parser_arr, q["packets"], q["lens"], q["ids"].ctypes.data, N, threads, pinned[0], pinned[1],
                                       N * bench.MB_PER_PIC, pinned[2], 64 * 1024 * 1024, C.byref(npk), C.byref(nmk), C.byref(nuk),
                                       None, None))
        if t > args.warmup:
            tp += time.perf_counter() - t0
    for p in pinned:
        L.h263cu_free_pinned(p)

    def summ(v):
        return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "runs": [float(x) for x in v]}

    out = {
        "tool": "tools/device_yuv_bench.py", "gpus": G, "streams_per_gpu": S, "picture": "%dx%d" % (W, H),
        "steps_timed": args.steps, "warmup": args.warmup, "rounds": args.rounds, "parse_threads": threads,
        "gpu": [torch.cuda.get_device_name(d) for d in range(G)], "nvidia_smi_index_name_power_limit_max_sm_clock": gpu_facts(),
        "unit": "MP/s (decoded megapixels per second, from the bitstream into preallocated device tensors)",
        "a_end_to_end": {a: summ(res[a]) for a in ARMS},
        "b_host_parse_alone": px / tp / 1e6,
        "c_recon_ms_per_launch": {a: summ(kern[a]) for a in ARMS},
        "c_deblock_ms_per_launch_i420_deblock": summ(deb),
        "i420_equals_read_yuv": bool(yuv_same),
        "nv12_equals_i420_interleaved": bool(nv12_same),
        "note": "The four outputs alternate round by round on the same context(s); each round replays the streams from "
                "their I picture and times the P steps from the first bitstream call to a device synchronise.  (c) is a "
                "separate pass with a CUDA event pair around every recon (and deblock) launch.  For i420_deblock the recon "
                "kernel writes only the context's planes; the deblock kernel writes the caller's.",
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
