#!/usr/bin/env python3
"""End-to-end decode from the bitstream into centre-cropped and letterboxed RGB tensors on the GPU (the fit form,
h263cu_decode_step_device_tensor_fit), against the plain stretch and against decoding to device RGBA and cropping in
torch.

    python tools/device_tensor_fit_bench.py [--steps K] [--warmup W] [--rounds R] [--profile-steps P] [--out profiles/<name>.json]

bench.py's workload (1024 CIF 352x288 streams, the same generator and parameters, its helpers imported), the same
parser thread count (all host cores), P pictures timed, one GPU.  Four arms alternate round by round on ONE context:
    stretch      h263cu_decode_step_device_tensor to [1024, 3, 224, 224] float16 NCHW, ImageNet mean / std
    center_crop  the fit form, CENTER_CROP with short side 256 -> 224 x 224 (torchvision's evaluation transform), float16,
                 ImageNet mean / std
    letterbox    the fit form, LETTERBOX into 640 x 640 float16, fill 114, std 1 (values / 255: the detectors' input)
    torch_crop   h263cu_decode_step_device RGBA, then permute / float / F.interpolate(bilinear, align_corners=False,
                 antialias=False) to the short side 256 / centre slice / normalise / half: center_crop's result in torch
For each arm it reports end-to-end MP/s (first bitstream call to a device synchronise, profiler off; medians of the
alternating rounds), the peak of torch's transient device memory above what was allocated before the run
(torch.cuda.max_memory_allocated), the largest difference between center_crop and torch_crop on the same pictures,
and, from a separate torch.profiler pass with CUDA activities, the device time per step of every kernel by name.  The
GPU's name and power limit go into the same JSON.  Exits non-zero without a GPU.
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
import bench  # noqa: E402  (the workload: generate_streams, host_threads, W, H)

ARMS = ("stretch", "center_crop", "letterbox", "torch_crop")
OUT = 224
SHORT = 256
LB = 640
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_device_tensor_fit_bench.json"))
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F

    if not torch.cuda.is_available():
        sys.exit("device_tensor_fit_bench: needs a CUDA device")
    from h263_rs_b200 import _lib, api

    L = _lib.lib()
    W, H, S = bench.W, bench.H, args.streams
    threads = bench.host_threads()
    total = 1 + args.warmup + args.steps
    blobs = bench.generate_streams(range(S), total, threads)
    dec = api.BatchDecoder(S, W, H, threads=threads)
    plans = []
    for t in range(total):
        views = [blobs[s][0][int(blobs[s][1][t]) : int(blobs[s][1][t]) + int(blobs[s][2][t])] for s in range(S)]
        plans.append(dec.plan_step(views))
    dev = torch.device("cuda", 0)
    # destinations, preallocated; the consumer stream is torch's current one
    rgba = torch.empty((S, H, W, 4), dtype=torch.uint8, device=dev)
    rgba_t = _lib.DeviceRgba(rgba.data_ptr(), W * 4, W * H * 4, W, H, torch.cuda.current_stream(dev).cuda_stream or None)
    stretch, stretch_t = api._device_tensor(None, S, (OUT, OUT), torch.float16, MEAN, STD, 0)
    crop, crop_t = api._device_tensor(None, S, (OUT, OUT), torch.float16, MEAN, STD, 0)
    crop_fit = api._tensor_fit("center_crop", SHORT, 0, None, S)
    lb, lb_t = api._device_tensor(None, S, (LB, LB), torch.float16, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), 0)
    lb_fit = api._tensor_fit("letterbox", None, 114, None, S)
    torch_out = torch.empty((S, 3, OUT, OUT), dtype=torch.float16, device=dev)
    mean = torch.tensor(MEAN, device=dev).view(1, 3, 1, 1)
    std = torch.tensor(STD, device=dev).view(1, 3, 1, 1)
    # torchvision's Resize(256) size of a CIF picture and its CenterCrop(224) window (include/h263cu.h's geometry)
    rh, rw = (SHORT, SHORT * W // H) if W > H else (SHORT * H // W, SHORT)
    top, left = int(round((rh - OUT) / 2.0)), int(round((rw - OUT) / 2.0))
    nd = C.c_uint32(0)

    def step(t, arm):
        q = plans[t]
        args_ = (dec.ctx.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, q["n"], threads, 0)
        if arm == "stretch":
            _lib.check(L.h263cu_decode_step_device_tensor(*args_, stretch_t, q["errs"].ctypes.data, C.byref(nd)))
        elif arm == "center_crop":
            _lib.check(L.h263cu_decode_step_device_tensor_fit(*args_, crop_t, crop_fit, q["errs"].ctypes.data, C.byref(nd)))
        elif arm == "letterbox":
            _lib.check(L.h263cu_decode_step_device_tensor_fit(*args_, lb_t, lb_fit, q["errs"].ctypes.data, C.byref(nd)))
        else:
            _lib.check(L.h263cu_decode_step_device(*args_[:-1], _lib.OUT_RGBA, rgba_t, q["errs"].ctypes.data, C.byref(nd)))
            x = rgba[..., :3].permute(0, 3, 1, 2).float()
            x = F.interpolate(x, size=(rh, rw), mode="bilinear", align_corners=False, antialias=False)
            x = x[:, :, top:top + OUT, left:left + OUT]
            torch_out.copy_(((x / 255 - mean) / std).half())
        assert not q["errs"].any()

    def sync():
        dec.ctx.sync()
        torch.cuda.synchronize(dev)

    def run(arm, prof=None):
        """One pass over the streams from their I picture: untimed warm-up steps, then the timed P steps."""
        for p in dec.parsers:
            p.reset()
        for t in range(1 + args.warmup):
            step(t, arm)
        sync()
        base = torch.cuda.memory_allocated(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        last = total if prof is None else 1 + args.warmup + args.profile_steps
        t0 = time.perf_counter()
        if prof is not None:
            prof.start()
        for t in range(1 + args.warmup, last):
            step(t, arm)
        sync()
        if prof is not None:
            prof.stop()
        sec = time.perf_counter() - t0
        return sec, torch.cuda.max_memory_allocated(dev) - base

    px = float(S) * W * H * args.steps
    res = {a: [] for a in ARMS}
    peak = {a: 0 for a in ARMS}
    for _ in range(args.rounds):
        for arm in ARMS:
            sec, extra = run(arm)
            res[arm].append(px / sec / 1e6)
            peak[arm] = max(peak[arm], extra)

    # result check on the last step of a pass: the fused centre crop against torch's conversion of the same pictures
    run("torch_crop")
    run("center_crop")
    diff = (crop.float() - torch_out.float()).abs()
    crop_vs_torch = {"max_abs": float(diff.max()), "mean_abs": float(diff.mean())}
    run("letterbox")
    # the bars above and below the placed picture hold the fill, 114 / 255 (fill through mul / add like a pixel)
    lrh = (2 * H * LB + W) // (2 * W) if W * LB >= H * LB else LB
    bar = (LB - lrh) // 2
    lb_check = {"bar_rows": bar, "fill_value": [float(v) for v in lb[0, :, 0, 0]],
                "bars_hold_the_fill": bool((lb[:, :, :bar] == lb[0, :, 0, 0].view(1, 3, 1, 1)).all()) if bar else None}

    # device time per step by kernel name, from a torch.profiler pass per arm
    kernels = {}
    for arm in ARMS:
        with_prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA])
        run(arm, with_prof)
        timed = []
        for e in with_prof.key_averages():
            us = getattr(e, "device_time_total", None)
            if us is None:
                us = getattr(e, "cuda_time_total", 0)
            if us and e.key and not e.key.startswith("cuda"):  # runtime API calls carry no device time of their own
                timed.append((e.key, us, "CUDA" in str(getattr(e, "device_type", ""))))
        kern = [(k, us) for k, us, on_dev in timed if on_dev] or [(k, us) for k, us, _ in timed]
        per = {}
        for k, us in kern:
            per[k] = per.get(k, 0.0) + us / 1e3 / args.profile_steps
        kernels[arm] = per

    def pick(per, name):
        return sum(v for k, v in per.items() if name in k)

    def summ(v):
        return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "runs": [float(x) for x in v]}

    device_ms = {}
    for arm in ARMS:
        per = kernels[arm]
        recon, resample = pick(per, "recon_tile_kernel") + pick(per, "recon_mb_kernel"), pick(per, "resample_rgb_kernel")
        device_ms[arm] = {"all_kernels": sum(per.values()), "recon": recon, "resample_rgb_kernel": resample,
                          "other (torch)": sum(per.values()) - recon - resample,
                          "by_kernel": {k: v for k, v in sorted(per.items(), key=lambda kv: -kv[1])[:12]}}

    out = {
        "tool": "tools/device_tensor_fit_bench.py", "streams": S, "picture": "%dx%d" % (W, H),
        "outputs": {"stretch": "%dx%d" % (OUT, OUT), "center_crop": "Resize(%d) -> %dx%d (resized %dx%d, window at x %d, y %d)"
                    % (SHORT, OUT, OUT, rw, rh, left, top), "letterbox": "%dx%d" % (LB, LB), "torch_crop": "as center_crop"},
        "steps_timed": args.steps, "warmup": args.warmup, "rounds": args.rounds, "profile_steps": args.profile_steps,
        "parse_threads": threads, "gpu": torch.cuda.get_device_name(dev),
        "nvidia_smi_index_name_power_limit_max_sm_clock": gpu_facts(),
        "unit": "MP/s (decoded megapixels per second, from the bitstream into preallocated device tensors)",
        "end_to_end": {a: summ(res[a]) for a in ARMS},
        "device_ms_per_step": device_ms,
        "torch_transient_peak_bytes": peak,
        "output_bytes": {"stretch": stretch.numel() * 2, "center_crop": crop.numel() * 2, "letterbox": lb.numel() * 2,
                         "torch_crop": torch_out.numel() * 2 + rgba.numel()},
        "center_crop_vs_torch_crop_f16": crop_vs_torch,
        "letterbox_check": lb_check,
        "note": "The arms alternate round by round on one context; each round replays the streams from their I picture "
                "and times the P steps from the first bitstream call to a device synchronise.  device_ms_per_step comes "
                "from a separate torch.profiler pass (CUDA activities) over profile_steps P steps per arm.  "
                "torch_transient_peak_bytes is what torch allocated above the preallocated destinations during a run "
                "(the float32 intermediates of the torch arm); the library's own context memory is not torch's and not "
                "counted.  center_crop_vs_torch_crop_f16 compares the fused centre crop with torch's conversion of the "
                "same pictures: both are bilinear with align_corners=False, antialias=False and differ by rounding only.",
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
