"""Migration velocity scan on one GPU against a loop of single-velocity Stolt calls; prints one JSON line.

    python scripts/bench_velocity_scan.py [--steps 10] [--warmup 3] [--shapes 2048x4096,8192x65536] [--nv 32]

Shapes are snum x tnum, 10 ns sampling, 5 m trace spacing, seeded normal noise on the device, tapers 100 / 1000, windows
64 x 64, nv velocities evenly from 1.4e8 to 2.0e8.  Per shape two arms alternate step by step in one process, with a
256 MiB L2 flush before every timed call:
  scan   one stolt_scan_device call: the forward transform once, then per velocity the remap / inverse and the focus
         kernel (no images kept)
  loop   nv one-velocity stolt_scan_device calls: each runs one whole Stolt migration (the passes of stolt_device, bit
         for bit) and the same focus kernel
Step time is the median CUDA-event time of the arm.  The per-velocity increment is (scan - one velocity) / (nv - 1),
with "one velocity" the loop's step over nv.  The focus kernel's rate comes from the kernel timer
(impdar_b200_kernel_timer) in one extra scan call: the image bytes it reads (nv x S2 x T x 4 B) over the summed time of
its two kernels, against the HBM bandwidth bench.py's load_peaks() returns (MEASURED_PEAKS.json if present, else its
fallback; "peak_src" says which).  The GPU name, power limit and SM clock are read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock": clock}
    except Exception as e:  # the numbers still stand; say what is missing
        return {"gpu": "unknown (%r)" % (e,)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="2048x4096,8192x65536")
    ap.add_argument("--nv", type=int, default=32)
    ap.add_argument("--window", default="64x64")
    a = ap.parse_args()
    if a.steps < 10 or a.warmup < 3:
        raise SystemExit("need --steps >= 10 and --warmup >= 3")
    import torch
    from bench import load_peaks
    from impdar_b200 import _lib, migrationlib as ml, synthetic
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU mode")
    lib = _lib.load()
    hbm_gbs, peak_src, _ = load_peaks()
    win = tuple(int(s) for s in a.window.split("x"))
    vels = np.linspace(1.4e8, 2.0e8, a.nv)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    result = {"script": "bench_velocity_scan", "steps": a.steps, "warmup": a.warmup, "l2_flush_mib": 256, "nv": a.nv,
              "window": list(win), "hbm_gbs_peak": hbm_gbs, "peak_src": peak_src, **gpu_info(), "shapes": {}}

    def timed(calls, steps, warmup):
        times = {k: [] for k in calls}
        for it in range(warmup + steps):
            for kind, fn in calls.items():
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                if it >= warmup:
                    times[kind].append(e0.elapsed_time(e1))
        return times

    def kernel_ms(call, names):
        lib.impdar_b200_kernel_timer(1)
        call()
        torch.cuda.synchronize()
        out = {}
        for name in names:
            ms, n = ctypes.c_double(0), ctypes.c_int(0)
            lib.impdar_b200_kernel_timer_read(name.encode(), ctypes.byref(ms), ctypes.byref(n))
            out[name] = (ms.value, n.value)
        lib.impdar_b200_kernel_timer(0)
        return out

    for shape in a.shapes.split(","):
        S, T = (int(s) for s in shape.split("x"))
        S2 = 2 * (S // 2)
        g = torch.Generator(device="cuda").manual_seed(S * 131 + T)
        x = torch.randn((S, T), generator=g, device="cuda", dtype=torch.float32)
        dx = synthetic.DX

        def scan():
            return ml.stolt_scan_device(x, synthetic.DT, dx, vels, 100, 1000, win)

        def loop():
            return [ml.stolt_scan_device(x, synthetic.DT, dx, vels[k:k + 1], 100, 1000, win) for k in range(a.nv)]
        times = timed({"scan": scan, "loop": loop}, a.steps, a.warmup)
        lane = (scan(), ml.stolt_last_pipeline())[1]
        # the two arms' focus panels agree bit for bit (each velocity's image is the same)
        same = bool(torch.equal(scan(), torch.cat(loop(), 0)))
        kt = kernel_ms(scan, ["stolt_focus_kernel", "stolt_focus_windows_kernel"])
        focus_ms = kt["stolt_focus_kernel"][0] + kt["stolt_focus_windows_kernel"][0]
        img_bytes = a.nv * S2 * T * 4
        scan_ms, loop_ms = float(np.median(times["scan"])), float(np.median(times["loop"]))
        one_ms = loop_ms / a.nv
        rec = {"lane": lane,
               "scan_ms": scan_ms, "scan_ms_min": float(np.min(times["scan"])), "scan_ms_max": float(np.max(times["scan"])),
               "loop_ms": loop_ms, "loop_ms_min": float(np.min(times["loop"])), "loop_ms_max": float(np.max(times["loop"])),
               "speedup": loop_ms / scan_ms, "loop_ms_per_velocity": one_ms,
               "scan_ms_per_velocity_increment": (scan_ms - one_ms) / (a.nv - 1) if a.nv > 1 else None,
               "focus_kernel_ms": kt["stolt_focus_kernel"][0], "focus_windows_kernel_ms": kt["stolt_focus_windows_kernel"][0],
               "focus_launches": kt["stolt_focus_kernel"][1], "focus_image_bytes": img_bytes,
               "focus_gbs": img_bytes / (focus_ms * 1e-3) / 1e9 if focus_ms else None,
               "focus_share_of_peak": img_bytes / (focus_ms * 1e-3) / 1e9 / hbm_gbs if focus_ms else None,
               "focus_panels_equal": same}
        result["shapes"]["%dx%d" % (S, T)] = rec
        del x
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
