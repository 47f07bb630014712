#!/usr/bin/env python3
"""What the motion fields of h263cu_decode_step_device_motion cost: bench.py's 1024 CIF streams decoded from the
bitstream into the 224 x 224 float16 centre crop (Resize(256) + CenterCrop, ImageNet mean / std), with and without the
motion fields beside it, and into the motion fields alone, each with the host and the device parse.

    python tools/device_motion_bench.py [--steps K] [--warmup W] [--rounds R] [--profile-steps P] [--out <path>.json]

Arms, alternating round by round on one context (bench.py's generator; parser threads: bench.py's count, 16 on the B200
machines): tensor, tensor_motion and motion, each with parse="host" and parse="device".  For each arm: MP/s end to end
(first call to a device synchronise, profiler off, medians of the rounds) and ms per step.  From a separate
torch.profiler pass with CUDA activities: the motion kernel's and the recon kernel's device time per launch, and the
motion kernel's bytes (the records it reads, the fields it writes) over its time.  The GPU's name and power limit go
into the same JSON.  Exits non-zero without a GPU.
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
import bench  # noqa: E402

MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
ARMS = [(o, p) for o in ("tensor", "tensor_motion", "motion") for p in ("host", "device")]


def gpu_facts():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines() if q.returncode == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--profile-steps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_device_motion_bench.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("device_motion_bench: needs a CUDA device")
    from h263_rs_b200 import _lib, api

    L = _lib.lib()
    threads = bench.host_threads()
    dev = torch.device("cuda", 0)
    S, W, H = args.streams, 352, 288
    total = 1 + args.warmup + args.steps
    blobs = bench.generate_streams(range(S), total, threads, w=W, h=H)
    dec = api.BatchDecoder(S, W, H, threads=threads)
    plans = []
    for t in range(total):
        views = [blobs[s][0][int(blobs[s][1][t]) : int(blobs[s][1][t]) + int(blobs[s][2][t])] for s in range(S)]
        plans.append(dec.plan_step(views))
    ten, ten_t = api._device_tensor(None, S, (224, 224), torch.float16, MEAN, STD, 0)
    fit = api._tensor_fit("center_crop", 256, 0, None, S)
    motion, mo_t = api._device_motion(True, S, W, H, 0)
    pixels = api._device_output(tensor=ten_t, fit=fit)
    nd = C.c_uint32(0)

    def step(t, out, parse):
        q = plans[t]
        flags = _lib.PARSE_ON_DEVICE if parse == "device" else 0
        a = (dec.ctx.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, q["n"], threads, flags)
        if out == "tensor":
            _lib.check(L.h263cu_decode_step_device_tensor_fit(*a, ten_t, fit, q["errs"].ctypes.data, C.byref(nd)))
        else:
            _lib.check(L.h263cu_decode_step_device_motion(*a, mo_t, pixels if out == "tensor_motion" else None, q["errs"].ctypes.data,
                                                          C.byref(nd)))
        assert not q["errs"].any()

    def sync():
        dec.ctx.sync()
        torch.cuda.synchronize(dev)

    def run(out, parse, prof=None):
        for p in dec.parsers:
            p.reset()
        for t in range(1 + args.warmup):
            step(t, out, parse)
        sync()
        last = total if prof is None else 1 + args.warmup + args.profile_steps
        if prof is not None:
            prof.start()
        t0 = time.perf_counter()
        for t in range(1 + args.warmup, last):
            step(t, out, parse)
        sync()
        sec = time.perf_counter() - t0
        if prof is not None:
            prof.stop()
        return sec

    px = float(S) * W * H * args.steps
    rec = {"%s/%s" % a: {"mps": [], "ms_per_step": []} for a in ARMS}
    for _ in range(args.rounds):
        for out, parse in ARMS:
            sec = run(out, parse)
            rec["%s/%s" % (out, parse)]["mps"].append(px / sec / 1e6)
            rec["%s/%s" % (out, parse)]["ms_per_step"].append(sec * 1e3 / args.steps)

    # the last step's outputs: the tensor is the same with and without motion, and the motion fields the same with
    # and without the tensor, under both parses
    same = {}
    for parse in ("host", "device"):
        run("tensor", parse)
        ref_t = ten.clone()
        run("motion", parse)
        ref_m = [x.clone() for x in motion]
        ten.zero_()
        for x in motion:
            x.zero_()
        run("tensor_motion", parse)
        same[parse] = bool(torch.equal(ref_t, ten)) and all(torch.equal(a, b) for a, b in zip(ref_m, motion))
    same["host_equals_device"] = all(torch.equal(a, b) for a, b in zip(ref_m, motion))

    kernels = {}
    for parse in ("host", "device"):
        prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA])
        run("tensor_motion", parse, prof)
        per = {}
        for e in prof.key_averages():
            us = getattr(e, "device_time_total", None)
            if us is None:
                us = getattr(e, "cuda_time_total", 0)
            if us and e.key and not e.key.startswith("cuda") and "CUDA" in str(getattr(e, "device_type", "CUDA")):
                per[e.key] = (per.get(e.key, (0.0, 0))[0] + us / 1e3, per.get(e.key, (0.0, 0))[1] + e.count)
        kernels[parse] = {k: {"ms_per_launch": v[0] / max(v[1], 1), "launches": v[1]} for k, v in
                          sorted(per.items(), key=lambda kv: -kv[1][0])[:12]}

    def per_launch(parse, name):
        v = [x["ms_per_launch"] for k, x in kernels[parse].items() if name in k]
        return v[0] if v else None

    cells = S * motion.flags.shape[1] * motion.flags.shape[2]
    n_mbs = S * ((W + 15) // 16) * ((H + 15) // 16)
    motion_bytes = {"records_read": 24 * n_mbs, "fields_written": cells * (2 * 2 * 4 + 1 + 1), "jobs_read": 16 * S}
    motion_bytes["total"] = sum(motion_bytes.values())
    mk = {p: per_launch(p, "motion_field_kernel") for p in ("host", "device")}
    rk = {p: per_launch(p, "recon_tile_kernel") for p in ("host", "device")}

    def summ(v):
        return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}

    out = {
        "tool": "tools/device_motion_bench.py", "streams": S, "picture": "%dx%d" % (W, H), "steps_timed": args.steps,
        "warmup": args.warmup, "rounds": args.rounds, "profile_steps": args.profile_steps, "parse_threads": threads,
        "gpu": torch.cuda.get_device_name(dev), "nvidia_smi_index_name_power_limit_max_sm_clock": gpu_facts(),
        "unit": "MP/s: decoded megapixels per second from the bitstream into preallocated device memory",
        "arms": {k: {kk: summ(vv) for kk, vv in v.items()} for k, v in rec.items()},
        "tensor_motion_over_tensor_mps": {p: float(np.median(rec["tensor_motion/" + p]["mps"]) / np.median(rec["tensor/" + p]["mps"]))
                                          for p in ("host", "device")},
        "motion_kernel_ms_per_launch": mk, "recon_kernel_ms_per_launch": rk,
        "motion_over_recon": {p: (mk[p] / rk[p] if mk[p] and rk[p] else None) for p in ("host", "device")},
        "motion_kernel_bytes_per_launch": motion_bytes,
        "motion_kernel_gb_per_s": {p: (motion_bytes["total"] / (mk[p] * 1e-3) / 1e9 if mk[p] else None) for p in ("host", "device")},
        "outputs_equal": same, "kernels_tensor_motion": kernels,
        "note": "the six arms alternate round by round on one context; each round replays the streams from their I picture "
                "and times the P steps from the first bitstream call to a device synchronise.  Kernel times come from a "
                "separate torch.profiler pass over profile_steps steps of the tensor_motion arm.",
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "nvidia_smi_index_name_power_limit_max_sm_clock", "tensor_motion_over_tensor_mps",
                                          "motion_kernel_ms_per_launch", "recon_kernel_ms_per_launch", "motion_kernel_gb_per_s",
                                          "outputs_equal")}))
    print(json.dumps({k: {kk: vv["median"] for kk, vv in v.items()} for k, v in out["arms"].items()}))


if __name__ == "__main__":
    main()
