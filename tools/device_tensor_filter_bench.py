#!/usr/bin/env python3
"""End-to-end decode from the bitstream into antialiased, centre-cropped RGB tensors on the GPU (the filter form,
h263cu_decode_step_device_tensor_filter), against the antialias=False fit call and against decoding to device RGBA and
resizing in torchvision.

    python tools/device_tensor_filter_bench.py [--steps K] [--warmup W] [--rounds R] [--profile-steps P] [--out profiles/<name>.json]

bench.py's workload (1024 CIF 352x288 streams, the same generator and parameters, its helpers imported), the same
parser thread count (all host cores), one GPU.  Every arm is torchvision's evaluation transform Resize(256) +
CenterCrop(224) to [1024, 3, 224, 224] float16 with ImageNet mean / std.  Five arms alternate round by round on ONE
context:
    center_crop   h263cu_decode_step_device_tensor_fit, CENTER_CROP 256 -> 224 (antialias=False bilinear): the baseline
    bilinear_aa   the filter form with H263CU_FILTER_BILINEAR_AA (torchvision Resize's default)
    bicubic_aa    the filter form with H263CU_FILTER_BICUBIC_AA
    torch_bilinear_aa  h263cu_decode_step_device RGBA, then permute / float / torchvision v2 resize(256, antialias=True)
                  on CUDA / center_crop / normalize / half: bilinear_aa's result in torch
    torch_bicubic_aa   the same with interpolation=BICUBIC
For each arm it reports end-to-end MP/s (first bitstream call to a device synchronise, profiler off; medians of the
alternating rounds), the peak of torch's transient device memory above what was allocated before the run, the largest
difference of each fused AA arm from its torch arm in float16 ulp, and, from a separate torch.profiler pass with CUDA
activities, the device time per step of every kernel by name.  The GPU's name and power limit go into the same JSON.
Exits non-zero without a GPU.
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

ARMS = ("center_crop", "bilinear_aa", "bicubic_aa", "torch_bilinear_aa", "torch_bicubic_aa")
OUT = 224
SHORT = 256
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_device_tensor_filter_bench.json"))
    args = ap.parse_args()
    import torch
    import torchvision.transforms.v2.functional as TF
    from torchvision.transforms import InterpolationMode

    if not torch.cuda.is_available():
        sys.exit("device_tensor_filter_bench: needs a CUDA device")
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
    fused = {a: api._device_tensor(None, S, (OUT, OUT), torch.float16, MEAN, STD, 0) for a in ARMS[:3]}
    crop_fit = api._tensor_fit("center_crop", SHORT, 0, None, S)
    filters = {"bilinear_aa": _lib.FILTER_BILINEAR_AA, "bicubic_aa": _lib.FILTER_BICUBIC_AA}
    modes = {"torch_bilinear_aa": InterpolationMode.BILINEAR, "torch_bicubic_aa": InterpolationMode.BICUBIC}
    torch_out = {a: torch.empty((S, 3, OUT, OUT), dtype=torch.float16, device=dev) for a in modes}
    nd = C.c_uint32(0)

    def step(t, arm):
        q = plans[t]
        args_ = (dec.ctx.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, q["n"], threads, 0)
        if arm == "center_crop":
            _lib.check(L.h263cu_decode_step_device_tensor_fit(*args_, fused[arm][1], crop_fit, q["errs"].ctypes.data, C.byref(nd)))
        elif arm in filters:
            _lib.check(L.h263cu_decode_step_device_tensor_filter(*args_, fused[arm][1], crop_fit, filters[arm], q["errs"].ctypes.data,
                                                                 C.byref(nd)))
        else:
            _lib.check(L.h263cu_decode_step_device(*args_[:-1], _lib.OUT_RGBA, rgba_t, q["errs"].ctypes.data, C.byref(nd)))
            x = rgba[..., :3].permute(0, 3, 1, 2).float()
            x = TF.resize(x, [SHORT], interpolation=modes[arm], antialias=True)
            x = TF.center_crop(x, [OUT, OUT])
            torch_out[arm].copy_(TF.normalize(x / 255, MEAN, STD).half())
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

    def f16_ulps(a, b):
        """|a - b| in units of float16's spacing at b (both float16 tensors)."""
        bh = b.abs()
        ulp = (torch.nextafter(bh, torch.full_like(bh, float("inf"))) - bh).float()
        return float(((a.float() - b.float()).abs() / ulp).max())

    # result check on the last step of a pass: each fused AA arm against torch's conversion of the same pictures
    vs_torch = {}
    for arm, tarm in (("bilinear_aa", "torch_bilinear_aa"), ("bicubic_aa", "torch_bicubic_aa")):
        run(tarm)
        run(arm)
        a, b = fused[arm][0], torch_out[tarm]
        vs_torch[arm] = {"max_f16_ulp": f16_ulps(a, b), "max_abs": float((a.float() - b.float()).abs().max()),
                         "elements_differing": int((a != b).sum()), "elements": a.numel()}

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
        recon = pick(per, "recon_tile_kernel") + pick(per, "recon_mb_kernel")
        resample = pick(per, "resample_rgb_kernel") + pick(per, "resample_filter_kernel")
        device_ms[arm] = {"all_kernels": sum(per.values()), "recon": recon, "resample (fused arms)": resample,
                          "other (torch)": sum(per.values()) - recon - resample,
                          "by_kernel": {k: v for k, v in sorted(per.items(), key=lambda kv: -kv[1])[:12]}}

    out_bytes = S * 3 * OUT * OUT * 2
    plane_bytes = S * W * H * 3 // 2
    out = {
        "tool": "tools/device_tensor_filter_bench.py", "streams": S, "picture": "%dx%d" % (W, H),
        "output": "Resize(%d) -> CenterCrop(%d) float16, ImageNet mean / std" % (SHORT, OUT),
        "steps_timed": args.steps, "warmup": args.warmup, "rounds": args.rounds, "profile_steps": args.profile_steps,
        "parse_threads": threads, "gpu": torch.cuda.get_device_name(dev),
        "nvidia_smi_index_name_power_limit_max_sm_clock": gpu_facts(),
        "unit": "MP/s (decoded megapixels per second, from the bitstream into preallocated device tensors)",
        "end_to_end": {a: summ(res[a]) for a in ARMS},
        "device_ms_per_step": device_ms,
        "torch_transient_peak_bytes": peak,
        "fused_bytes_per_step": {"planes_read": plane_bytes, "tensor_written": out_bytes,
                                 "floor_ms_at_7.7TB/s": (plane_bytes + out_bytes) / 7.7e12 * 1e3},
        "fused_vs_torch_f16": vs_torch,
        "note": "The arms alternate round by round on one context; each round replays the streams from their I picture "
                "and times the P steps from the first bitstream call to a device synchronise.  device_ms_per_step comes "
                "from a separate torch.profiler pass (CUDA activities) over profile_steps P steps per arm.  "
                "torch_transient_peak_bytes is what torch allocated above the preallocated destinations during a run; the "
                "library's own context memory is not torch's and not counted.  fused_vs_torch_f16 compares each fused AA "
                "arm with torchvision's conversion of the same pictures on CUDA: the same filter, differing by rounding.",
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
