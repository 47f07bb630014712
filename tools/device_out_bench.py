#!/usr/bin/env python3
"""End-to-end decode from the bitstream with RGBA left on the GPU vs read back to the host.

    python tools/device_out_bench.py [--gpus N] [--steps K] [--warmup W] [--rounds R] [--out profiles/<name>.json]

bench.py's workload (1024 CIF 352x288 streams per GPU, the same generator and parameters, its helpers imported), the
same parser thread count (all host cores), P pictures timed.  In one run, alternating round by round on ONE context
(or group), it measures:
  (a) h263cu_decode_step with the RGBA read back into pinned host memory, MP/s
  (b) h263cu_decode_step_device into a preallocated torch tensor on the GPU, MP/s
  (c) h263cu_parse_step alone (the host parse, same threads and packets), MP/s
  (d) the recon kernel's ms per launch (h263cu_profile_enable/read) with the RGBA pool (with the read-back of the
      previous step running beside it, and without any read-back) and with the device tensor as the TMA store target,
      in separate profiled passes
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
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_device_out_bench.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available() or torch.cuda.device_count() < args.gpus:
        sys.exit("device_out_bench: needs %d CUDA device(s), found %d" % (args.gpus, torch.cuda.device_count() if torch.cuda.is_available() else 0))
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
    pic = W * H * 4
    host = L.h263cu_alloc_pinned(N * pic)
    assert host, "cudaHostAlloc failed"
    # (b)'s destination: one preallocated tensor per device, tight [S, H, W, 4]; the consumer stream is torch's current one
    outs = [torch.empty((S, H, W, 4), dtype=torch.uint8, device="cuda:%d" % d) for d in range(G)]
    targets = (_lib.DeviceRgba * G)(*[_lib.DeviceRgba(o.data_ptr(), W * 4, W * H * 4, W, H,
                                                      torch.cuda.current_stream(d).cuda_stream or None) for d, o in enumerate(outs)])
    nd = C.c_uint32(0)

    def step(t, arm):
        q = plans[t]
        if arm == "host":
            dec.decode_planned(q, _lib.OUT_RGBA, host, pic)
        elif arm == "pool":  # RGBA into the context's pool, no read-back: the recon kernel alone against the same target
            dec.decode_planned(q, _lib.OUT_RGBA, None, 0)
        elif G == 1:
            _lib.check(L.h263cu_decode_step_device(dec.ctx.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, q["n"],
                                                   threads, _lib.OUT_RGBA, targets, q["errs"].ctypes.data, C.byref(nd)))
        else:
            _lib.check(L.h263cu_group_decode_step_device(dec.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, q["n"],
                                                         _lib.OUT_RGBA, targets, q["errs"].ctypes.data, C.byref(nd)))
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
            prof = sum(r["recon_ms"] for r in rs) / max(sum(r["recon_launches"] for r in rs), 1)
        return sec, prof

    px = float(N) * W * H * args.steps
    res = {"host": [], "device": []}
    for _ in range(args.rounds):
        for arm in ("host", "device"):
            res[arm].append(px / run(arm)[0] / 1e6)
    # device result check: the last step's tensor against the host read-back of the same step
    run("device")
    dev_last = [o.cpu().numpy() for o in outs]
    run("host")
    host_last = np.ctypeslib.as_array(C.cast(host, C.POINTER(C.c_uint8)), shape=(N * pic,)).reshape(G, S, -1)
    same = all(np.array_equal(dev_last[d].reshape(S, -1), host_last[d]) for d in range(G))
    # (d) recon kernel per launch, pool target (with and without the read-back running beside it) vs device target
    kern = {"host": [], "pool": [], "device": []}
    for _ in range(args.rounds):
        for arm in ("host", "pool", "device"):
            kern[arm].append(run(arm, profile=True)[1])
    # (c) host parse alone on fresh parsers, same packets and threads
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
    L.h263cu_free_pinned(host)

    def summ(v):
        return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "runs": [float(x) for x in v]}

    out = {
        "tool": "tools/device_out_bench.py", "gpus": G, "streams_per_gpu": S, "picture": "%dx%d" % (W, H),
        "steps_timed": args.steps, "warmup": args.warmup, "rounds": args.rounds, "parse_threads": threads,
        "gpu": [torch.cuda.get_device_name(d) for d in range(G)], "nvidia_smi_index_name_power_limit_max_sm_clock": gpu_facts(),
        "unit": "MP/s (decoded RGBA megapixels per second, from the bitstream)",
        "a_host_readback": summ(res["host"]), "b_device_output": summ(res["device"]),
        "c_host_parse_alone": px / tp / 1e6,
        "d_recon_ms_per_launch": {"pool_target_with_readback": summ(kern["host"]), "pool_target_no_readback": summ(kern["pool"]),
                                  "device_target": summ(kern["device"])},
        "device_output_equals_host_readback": same,
        "note": "(a) and (b) alternate round by round on the same context(s); each round replays the streams from their I "
                "picture and times the P steps from the first bitstream call to a device synchronise.  (d) is a separate "
                "pass with a CUDA event pair around every recon launch.",
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
