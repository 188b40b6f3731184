"""Time-to-depth conversion (depth_convert_device, float32) on one GPU; prints one JSON line.

    python scripts/bench_depth_conversion.py [--steps 10] [--warmup 3] [--shapes 2048x4096,8192x65536]

Shapes are snum x tnum, 10 ns sampling, seeded normal data on the device.  Fields (interval velocities):
  constant   P = 1, 1.69e8
  layered    P = 1, getVelocityProfile of synthetic.layered_velocity (2.3e8 at the top to 1.69e8)
  scan       P = tnum / 64: the layered profile scaled by 1 +- 3 % per run of 64 traces (a scan_interval_field shape)
  per_trace  P = tnum: the layered profile scaled per trace (a (v, z, x) table with one column per trace)
The depth grid is z = dz * arange(nz), dz = min(v) dt / 2, reaching the deepest last-sample depth.  Each call is timed
with CUDA events after a 256 MiB L2 flush (median of --steps after --warmup); the events bracket the host validation,
the staged upload and both kernels.  Per-kernel times come from the kernel timer (impdar_b200_kernel_timer) in one extra
call.  HBM bytes of the algorithm, from shapes: 4 snum tnum (image) + 4 nz tnum (section) + 8 P snum (profiles read by
pass 1) + 16 P snum (curves written by pass 1 and read once by pass 2); pass 2 alone moves 4 snum tnum + 4 nz tnum +
8 P snum.  Rates are against bench.py's load_peaks() (MEASURED_PEAKS.json if present, else its fallback; "peak_src" says
which).  The GPU name, power limit and SM clock are read in the same run.
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="2048x4096,8192x65536")
    ap.add_argument("--fields", default="constant,layered,scan,per_trace")
    a = ap.parse_args()
    if a.steps < 10 or a.warmup < 3:
        raise SystemExit("need --steps >= 10 and --warmup >= 3")
    import torch
    from bench import load_peaks
    from bench_velocity_scan import gpu_info
    from impdar_b200 import _lib, migrationlib as ml, synthetic
    from impdar_b200.radardata import RadarData
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU mode")
    lib = _lib.load()
    hbm_gbs, peak_src, _ = load_peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    result = {"script": "bench_depth_conversion", "steps": a.steps, "warmup": a.warmup, "l2_flush_mib": 256,
              "dtype": "float32", "hbm_gbs_peak": hbm_gbs, "peak_src": peak_src, **gpu_info(), "shapes": {}}
    names = ["depth_curve_kernel", "depth_resample_kernel"]

    def kernel_ms(call):
        lib.impdar_b200_kernel_timer(1)
        call()
        torch.cuda.synchronize()
        out = {}
        for name in names:
            ms, n = ctypes.c_double(0), ctypes.c_int(0)
            lib.impdar_b200_kernel_timer_read(name.encode(), ctypes.byref(ms), ctypes.byref(n))
            out[name] = ms.value
        lib.impdar_b200_kernel_timer(0)
        return out

    for shape in a.shapes.split(","):
        S, T = (int(s) for s in shape.split("x"))
        tt = np.arange(S) * synthetic.DT * 1e6
        d = RadarData(np.zeros((S, 1), np.float32), dt=synthetic.DT, travel_time=tt, dist=np.zeros(1))
        layered = ml.getVelocityProfile(d, synthetic.layered_velocity(tt))
        g = torch.Generator(device="cuda").manual_seed(S * 7 + T)
        x = torch.randn((S, T), generator=g, device="cuda", dtype=torch.float32)
        rec = {}
        for field in a.fields.split(","):
            rng = np.random.default_rng(S + T)
            if field == "constant":
                prof, colp = np.full((1, S), 1.69e8), np.zeros(T, np.int32)
            elif field == "layered":
                prof, colp = layered[None, :].copy(), np.zeros(T, np.int32)
            elif field == "scan":
                P = -(-T // 64)
                prof = layered[None, :] * (1 + 0.03 * rng.uniform(-1, 1, (P, 1)))
                colp = (np.arange(T) // 64).astype(np.int32)
            else:
                prof = layered[None, :] * (1 + 0.03 * rng.uniform(-1, 1, (T, 1)))
                colp = np.arange(T, dtype=np.int32)
            P = prof.shape[0]
            vmin, vmax = float(prof.min()), float(prof.max())
            dz = vmin * synthetic.DT / 2
            nz = int(np.ceil(vmax * tt[-1] / 1e6 / 2 / dz)) + 1
            zg = dz * np.arange(nz)
            out = torch.empty((nz, T), dtype=torch.float32, device="cuda")

            def call():
                return ml.depth_convert_device(x, tt, prof, colp, zg, out=out)
            times, host = [], []
            for it in range(a.warmup + a.steps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                h0 = time.perf_counter()
                e0.record()
                call()
                e1.record()
                torch.cuda.synchronize()
                h1 = time.perf_counter()
                if it >= a.warmup:
                    times.append(e0.elapsed_time(e1))
                    host.append((h1 - h0) * 1e3)
            first = out.clone()
            call()
            same = bool(torch.equal(torch.nan_to_num(first, nan=-7.0), torch.nan_to_num(out, nan=-7.0)))
            flush.zero_()
            kt = kernel_ms(call)
            k1, k2 = kt["depth_curve_kernel"], kt["depth_resample_kernel"]
            img_b, sec_b, prof_b, curve_b = 4 * S * T, 4 * nz * T, 8 * P * S, 16 * P * S
            alg = img_b + sec_b + prof_b + curve_b
            pass2 = img_b + sec_b + 8 * P * S
            rec[field] = {"nprof": P, "nz": nz,
                          "call_ms": float(np.median(times)), "call_ms_min": float(np.min(times)),
                          "call_ms_max": float(np.max(times)), "call_host_ms": float(np.median(host)),
                          "curve_kernel_ms": k1, "resample_kernel_ms": k2,
                          "alg_bytes": alg, "pass2_bytes": pass2, "pass1_bytes": prof_b + 8 * P * S,
                          "kernels_gbs": alg / ((k1 + k2) * 1e-3) / 1e9 if k1 + k2 else None,
                          "resample_gbs": pass2 / (k2 * 1e-3) / 1e9 if k2 else None,
                          "resample_share_of_peak": pass2 / (k2 * 1e-3) / 1e9 / hbm_gbs if k2 else None,
                          "curve_gbs": (prof_b + 8 * P * S) / (k1 * 1e-3) / 1e9 if k1 else None,
                          "repeatable": same}
            del out
            torch.cuda.empty_cache()
        result["shapes"]["%dx%d" % (S, T)] = rec
        del x
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
