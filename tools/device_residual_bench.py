#!/usr/bin/env python3
"""What the prediction residuals of h263cu_decode_step_device_residual cost: bench.py's 1024 CIF streams decoded from
the bitstream into the 224 x 224 float16 centre crop (Resize(256) + CenterCrop, ImageNet mean / std), alone, with the
motion fields, with the motion fields and the residual (CoViAR's three inputs from one parse), and into the residual
alone, each with the host and the device parse; beside them the torch route: the planes and the motion fields from
the library and the residual rebuilt with torch ops from them and the previous step's planes.

    python tools/device_residual_bench.py [--steps K] [--warmup W] [--rounds R] [--profile-steps P] [--out <path>.json]

The arms alternate round by round on one context (bench.py's generator; parser threads: bench.py's count, 16 on the B200
machines).  For each arm: MP/s end to end (first call to a device synchronise, profiler off, medians of the rounds) and
ms per step.  From a separate torch.profiler pass with CUDA activities: the residual kernel's and the recon kernel's
device time per launch, and the residual kernel against its byte floor (the planes it must read and write, computed
here from the shapes).  The GPU's name and power limit go into the same JSON.  Exits non-zero without a GPU.
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
OUTS = ("tensor", "tensor_motion", "tensor_motion_residual", "residual", "torch_route")
ARMS = [(o, p) for o in OUTS for p in ("host", "device")]
HBM_TBPS = {"datasheet": 7.7, "measured_peak": 6.54}  # B200 HBM3e: NVIDIA's figure and this project's measured copy peak


def gpu_facts():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines() if q.returncode == 0 else None


def byte_floor(S, W, H):
    """Bytes residual_kernel cannot avoid per step: every sample of cur and of the reference read once (the reference's
    halo around each block not counted), every int16 output written once, the 24-byte record of every macroblock."""
    cw, ch = (W + 1) // 2, (H + 1) // 2
    per = {"cur_read": W * H + 2 * cw * ch, "ref_read": W * H + 2 * cw * ch, "int16_written": 2 * (W * H + 2 * cw * ch),
           "records_read": 24 * ((W + 15) // 16) * ((H + 15) // 16)}
    per["total"] = sum(per.values())
    step = S * per["total"]
    return {"per_picture": per, "per_step": step, "ms_at": {k: step / (v * 1e12) * 1e3 for k, v in HBM_TBPS.items()}}


def torch_residual(torch, cur, prev, mv, flags):
    """The residual of include/h263cu.h in torch ops, for pictures whose sizes are multiples of 16 (bench.py's CIF):
    cur / prev (y, cb, cr) uint8 [S, h, w] planes, mv int16 [S, 2, 2 MBH, 2 MBW], flags uint8 [S, MBH, MBW]."""
    inter = (flags & 1).bool()
    out = []
    for k in range(3):
        c, r = cur[k].int(), prev[k].int()
        S, h, w = c.shape
        if k == 0:
            vx = mv[:, 0].repeat_interleave(8, 1).repeat_interleave(8, 2).int()
            vy = mv[:, 1].repeat_interleave(8, 1).repeat_interleave(8, 2).int()
            m = inter.repeat_interleave(16, 1).repeat_interleave(16, 2)
        else:
            def avg(s):  # average_sum_of_mvs (types.rs:759-768)
                whole, frac = (s >> 4) * 2, s & 15
                return torch.where(frac <= 2, whole, torch.where(frac >= 14, whole + 2, whole + 1))

            sums = mv.int().unflatten(2, (-1, 2)).unflatten(4, (-1, 2)).sum((3, 5))  # [S, 2, MBH, MBW]
            vx = avg(sums[:, 0]).repeat_interleave(8, 1).repeat_interleave(8, 2)
            vy = avg(sums[:, 1]).repeat_interleave(8, 1).repeat_interleave(8, 2)
            m = inter.repeat_interleave(8, 1).repeat_interleave(8, 2)
        dx, ix, dy, iy = vx >> 1, (vx & 1).bool(), vy >> 1, (vy & 1).bool()
        xs = torch.arange(w, device=c.device).view(1, 1, w) + dx
        ys = torch.arange(h, device=c.device).view(1, h, 1) + dy
        flat = r.flatten(1)

        def at(yy, xx):
            return flat.gather(1, (yy.clamp(0, h - 1) * w + xx.clamp(0, w - 1)).flatten(1)).view(S, h, w)

        a, b, cc, d = at(ys, xs), at(ys, xs + 1), at(ys + 1, xs), at(ys + 1, xs + 1)
        pred = torch.where(ix & iy, (a + b + cc + d + 2) >> 2, torch.where(ix, (a + b + 1) >> 1, torch.where(iy, (a + cc + 1) >> 1, a)))
        out.append((c - torch.where(m, pred, 0)).short())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--profile-steps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_device_residual_bench.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("device_residual_bench: needs a CUDA device")
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
    res, re_t = api._device_residual(True, S, W, H, 0)
    # the torch route: two sets of I420 planes, alternating, so that the previous step's are the reference
    yuvs = [api._device_yuv(None, S, W, H, 0, "i420") for _ in range(2)]
    torch_res = [None]
    pixels = api._device_output(tensor=ten_t, fit=fit)
    nd = C.c_uint32(0)

    def step(t, out, parse):
        q = plans[t]
        flags = _lib.PARSE_ON_DEVICE if parse == "device" else 0
        a = (dec.ctx.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, q["n"], threads, flags)
        e = q["errs"].ctypes.data
        if out == "tensor":
            _lib.check(L.h263cu_decode_step_device_tensor_fit(*a, ten_t, fit, e, C.byref(nd)))
        elif out == "tensor_motion":
            _lib.check(L.h263cu_decode_step_device_motion(*a, mo_t, pixels, e, C.byref(nd)))
        elif out == "tensor_motion_residual":
            _lib.check(L.h263cu_decode_step_device_residual(*a, re_t, mo_t, pixels, e, C.byref(nd)))
        elif out == "residual":
            _lib.check(L.h263cu_decode_step_device_residual(*a, re_t, None, None, e, C.byref(nd)))
        else:
            planes, target = yuvs[t & 1]
            _lib.check(L.h263cu_decode_step_device_motion(*a, mo_t, api._device_output(yuv=target), e, C.byref(nd)))
            torch_res[0] = torch_residual(torch, planes, yuvs[(t & 1) ^ 1][0], motion.mv, motion.flags)
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

    # the last step's outputs: tensor and motion the same with and without the residual, the residual the same alone,
    # beside the others, under both parses and from the torch route
    same = {}
    for parse in ("host", "device"):
        run("tensor_motion", parse)
        ref_t, ref_m = ten.clone(), [x.clone() for x in motion]
        run("residual", parse)
        ref_r = [x.clone() for x in res]
        for x in [ten, *motion, *res]:
            x.zero_()
        run("tensor_motion_residual", parse)
        same[parse] = (bool(torch.equal(ref_t, ten)) and all(torch.equal(a, b) for a, b in zip(ref_m, motion)) and
                       all(torch.equal(a, b) for a, b in zip(ref_r, res)))
        run("torch_route", parse)
        same["torch_route_" + parse] = all(torch.equal(a, b) for a, b in zip(ref_r, torch_res[0]))

    kernels = {}
    for parse in ("host", "device"):
        prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA])
        run("tensor_motion_residual", parse, prof)
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

    floor = byte_floor(S, W, H)
    rk = {p: per_launch(p, "residual_kernel") for p in ("host", "device")}
    ck = {p: per_launch(p, "recon_tile_kernel") for p in ("host", "device")}

    def summ(v):
        return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}

    def med(arm):
        return float(np.median(rec[arm]["mps"]))

    out = {
        "tool": "tools/device_residual_bench.py", "streams": S, "picture": "%dx%d" % (W, H), "steps_timed": args.steps,
        "warmup": args.warmup, "rounds": args.rounds, "profile_steps": args.profile_steps, "parse_threads": threads,
        "gpu": torch.cuda.get_device_name(dev), "nvidia_smi_index_name_power_limit_max_sm_clock": gpu_facts(),
        "unit": "MP/s: decoded megapixels per second from the bitstream into preallocated device memory",
        "arms": {k: {kk: summ(vv) for kk, vv in v.items()} for k, v in rec.items()},
        "over_tensor_mps": {p: {o: med("%s/%s" % (o, p)) / med("tensor/" + p) for o in OUTS[1:]} for p in ("host", "device")},
        "residual_kernel_ms_per_launch": rk, "recon_kernel_ms_per_launch": ck,
        "residual_kernel_byte_floor": floor,
        "residual_kernel_over_floor": {p: {k: (rk[p] / v if rk[p] else None) for k, v in floor["ms_at"].items()} for p in ("host", "device")},
        "residual_kernel_gb_per_s_of_floor_bytes": {p: (floor["per_step"] / (rk[p] * 1e-3) / 1e9 if rk[p] else None)
                                                    for p in ("host", "device")},
        "outputs_equal": same, "kernels_tensor_motion_residual": kernels,
        "note": "the ten arms alternate round by round on one context; each round replays the streams from their I picture "
                "and times the P steps from the first bitstream call to a device synchronise.  Kernel times come from a "
                "separate torch.profiler pass over profile_steps steps of the tensor_motion_residual arm.  torch_route: "
                "decode_step_device_yuv + motion into alternating plane buffers, then torch_residual() on this step's and "
                "the previous step's planes (exact for these CIF streams: no partial macroblocks, no disposable pictures).",
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "nvidia_smi_index_name_power_limit_max_sm_clock", "over_tensor_mps",
                                          "residual_kernel_ms_per_launch", "recon_kernel_ms_per_launch", "residual_kernel_over_floor",
                                          "outputs_equal")}))
    print(json.dumps({k: {kk: vv["median"] for kk, vv in v.items()} for k, v in out["arms"].items()}))


if __name__ == "__main__":
    main()
