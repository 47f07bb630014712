#!/usr/bin/env python3
"""End-to-end decode from the bitstream with the macroblock layer parsed on the host (parse="host", the threaded
parser) and on the GPU (parse="device", H263CU_PARSE_ON_DEVICE), alternating round by round on one context.

    python tools/device_parse_bench.py [--steps K] [--warmup W] [--rounds R] [--profile-steps P] [--out profiles/<name>.json]

Workloads (bench.py's generator and parameters, its helpers imported; parser threads: bench.py's count, all host
cores, 16 on the B200 machines):
    cif1024_rgba     1024 CIF 352x288 streams into device RGBA (h263cu_decode_step_device)
    cif1024_tensor   the same into the 224 x 224 float16 centre crop (Resize(256) + CenterCrop, ImageNet mean / std)
    4cif256_rgba     256 4CIF 704x576 streams into device RGBA
    n1_rgba          one CIF stream into device RGBA
For each arm: MP/s end to end (first call to a device synchronise, profiler off, medians of the rounds), ms per step,
host CPU seconds per step (process CPU time over the timed steps), H2D bytes per step (host parse: the side info;
device parse: the padded packets and the job records) and, from a separate torch.profiler pass with CUDA activities,
the parse kernel's device ms per launch.  The GPU's name and power limit go into the same JSON.  Exits non-zero without
a GPU.
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
WORKLOADS = {"cif1024_rgba": (1024, 352, 288, "rgba"), "cif1024_tensor": (1024, 352, 288, "tensor"),
             "4cif256_rgba": (256, 704, 576, "rgba"), "n1_rgba": (1, 352, 288, "rgba")}


def gpu_facts():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines() if q.returncode == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--profile-steps", type=int, default=5)
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_device_parse_bench.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("device_parse_bench: needs a CUDA device")
    from h263_rs_b200 import _lib, api, frontend

    L = _lib.lib()
    threads = bench.host_threads()
    dev = torch.device("cuda", 0)
    total = 1 + args.warmup + args.steps
    names = args.only.split(",") if args.only else list(WORKLOADS)
    results = {}
    for name in names:
        S, W, H, out_kind = WORKLOADS[name]
        blobs = bench.generate_streams(range(S), total, threads, w=W, h=H)
        dec = api.BatchDecoder(S, W, H, threads=threads)
        plans = []
        for t in range(total):
            views = [blobs[s][0][int(blobs[s][1][t]) : int(blobs[s][1][t]) + int(blobs[s][2][t])] for s in range(S)]
            plans.append(dec.plan_step(views))
        stream = torch.cuda.current_stream(dev).cuda_stream or None
        rgba = torch.empty((S, H, W, 4), dtype=torch.uint8, device=dev)
        rgba_t = _lib.DeviceRgba(rgba.data_ptr(), W * 4, W * H * 4, W, H, stream)
        ten, ten_t = api._device_tensor(None, S, (224, 224), torch.float16, MEAN, STD, 0)
        fit = api._tensor_fit("center_crop", 256, 0, None, S)
        nd = C.c_uint32(0)

        def step(t, parse):
            q = plans[t]
            flags = _lib.PARSE_ON_DEVICE if parse == "device" else 0
            a = (dec.ctx.h, q["parsers"], q["packets"], q["lens"], q["ids"].ctypes.data, q["n"], threads)
            if out_kind == "rgba":
                _lib.check(L.h263cu_decode_step_device(*a, _lib.OUT_RGBA | flags, rgba_t, q["errs"].ctypes.data, C.byref(nd)))
            else:
                _lib.check(L.h263cu_decode_step_device_tensor_fit(*a, flags, ten_t, fit, q["errs"].ctypes.data, C.byref(nd)))
            assert not q["errs"].any()

        def sync():
            dec.ctx.sync()
            torch.cuda.synchronize(dev)

        def run(parse, prof=None):
            for p in dec.parsers:
                p.reset()
            for t in range(1 + args.warmup):
                step(t, parse)
            sync()
            last = total if prof is None else 1 + args.warmup + args.profile_steps
            if prof is not None:
                prof.start()
            c0, t0 = time.process_time(), time.perf_counter()
            for t in range(1 + args.warmup, last):
                step(t, parse)
            sync()
            sec, cpu = time.perf_counter() - t0, time.process_time() - c0
            if prof is not None:
                prof.stop()
            return sec, cpu

        px = float(S) * W * H * args.steps
        rec = {p: {"mps": [], "ms_per_step": [], "cpu_s_per_step": []} for p in ("host", "device")}
        for _ in range(args.rounds):
            for parse in ("host", "device"):
                sec, cpu = run(parse)
                rec[parse]["mps"].append(px / sec / 1e6)
                rec[parse]["ms_per_step"].append(sec * 1e3 / args.steps)
                rec[parse]["cpu_s_per_step"].append(cpu / args.steps)
        # outputs of the last step agree between the two parses
        run("host")
        ref = (rgba if out_kind == "rgba" else ten).clone()
        run("device")
        same = bool(torch.equal(ref, rgba if out_kind == "rgba" else ten))

        # H2D bytes per step, from the last step's packets: the side info the host parse uploads against the padded
        # packets and 32-byte jobs the device parse uploads (plus 16 bytes a picture of results back)
        lens = [int(blobs[s][2][total - 1]) for s in range(S)]
        pk = [bytes(blobs[s][0][int(blobs[s][1][total - 1]) : int(blobs[s][1][total - 1]) + lens[s]]) for s in range(S)]
        ps = [frontend.Parser(1) for _ in range(S)]
        for t in range(total - 1):  # bring the parsers to the last step
            frontend.parse_step(ps, [bytes(blobs[s][0][int(blobs[s][1][t]) : int(blobs[s][1][t]) + int(blobs[s][2][t])])
                                     for s in range(S)], None, threads)
        pics, mbs, ev, _, _ = frontend.parse_step(ps, pk, None, threads)
        h2d = {"host": int(pics.nbytes + mbs.nbytes + ev.nbytes),
               "device": int(sum((n + 12 + 15) // 16 * 16 for n in lens) + 32 * S), "device_d2h_results": 16 * S,
               "bitstream": int(sum(lens))}

        kernels = {}
        for parse in ("host", "device"):
            prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA])
            run(parse, prof)
            per = {}
            for e in prof.key_averages():
                us = getattr(e, "device_time_total", None)
                if us is None:
                    us = getattr(e, "cuda_time_total", 0)
                if us and e.key and not e.key.startswith("cuda") and "CUDA" in str(getattr(e, "device_type", "CUDA")):
                    per[e.key] = (per.get(e.key, (0.0, 0))[0] + us / 1e3, per.get(e.key, (0.0, 0))[1] + e.count)
            kernels[parse] = {k: {"ms_per_step": v[0] / args.profile_steps, "launches": v[1]} for k, v in
                              sorted(per.items(), key=lambda kv: -kv[1][0])[:10]}
        pk_ms = [(v["ms_per_step"] * args.profile_steps / max(v["launches"], 1)) for k, v in kernels["device"].items()
                 if "parse_mb_kernel" in k]

        def summ(v):
            return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}

        results[name] = {
            "streams": S, "picture": "%dx%d" % (W, H), "output": "device RGBA" if out_kind == "rgba" else
            "224x224 float16 centre crop (Resize(256))",
            "host": {k: summ(v) for k, v in rec["host"].items()}, "device": {k: summ(v) for k, v in rec["device"].items()},
            "device_over_host_mps": float(np.median(rec["device"]["mps"]) / np.median(rec["host"]["mps"])),
            "parse_kernel_ms_per_launch": pk_ms[0] if pk_ms else None,
            "h2d_bytes_per_step": h2d, "outputs_equal": same, "kernels_by_parse": kernels,
        }
        print(name, json.dumps({k: results[name][k] for k in ("host", "device", "parse_kernel_ms_per_launch",
                                                                "device_over_host_mps", "outputs_equal")}), flush=True)
        del dec, rgba, ten
        torch.cuda.empty_cache()

    out = {
        "tool": "tools/device_parse_bench.py", "steps_timed": args.steps, "warmup": args.warmup, "rounds": args.rounds,
        "profile_steps": args.profile_steps, "parse_threads": threads, "gpu": torch.cuda.get_device_name(dev),
        "nvidia_smi_index_name_power_limit_max_sm_clock": gpu_facts(),
        "unit": "MP/s: decoded megapixels per second from the bitstream into preallocated device memory",
        "workloads": results,
        "note": "host and device parse alternate round by round on one context; each round replays the streams from "
                "their I picture and times the P steps from the first bitstream call to a device synchronise.  "
                "cpu_s_per_step is the process's CPU time (all threads) over the timed steps.  Kernel times come from a "
                "separate torch.profiler pass over profile_steps steps.",
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "nvidia_smi_index_name_power_limit_max_sm_clock")}))


if __name__ == "__main__":
    main()
