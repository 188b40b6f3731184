"""Kirchhoff migration, constant against layered (per-sample RMS) velocity, on one GPU; prints one JSON line.

    python scripts/bench_kirchhoff_layered.py [--steps 10] [--warmup 3] [--shapes 2048x4096,8192x65536]

Shapes are snum x tnum (2048 x 4096: config 2; 8192 x 65536: the headline image), 10 ns sampling, 5 m trace spacing,
seeded normal noise on the device.  The layered profile is synthetic.layered_velocity through getVelocityProfile and
rms_velocity (2.2e8 at the top down to 1.7e8).  Per shape the two velocities alternate step by step in one process,
with a 256 MiB L2 flush before every timed call; step time is the median of CUDA-event times.  Pairs come from the
kernel's own counters in one extra untimed call; parity is rel-L2 against the float64 per-row reference on sampled
output traces.  The GPU name, power limit and SM clock are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(1, os.path.join(ROOT, "tests"))


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
    ap.add_argument("--parity-traces", type=int, default=4)
    a = ap.parse_args()
    if a.steps < 10 or a.warmup < 3:
        raise SystemExit("need --steps >= 10 and --warmup >= 3")
    import torch
    import impdar_b200
    from impdar_b200 import migrationlib as ml, synthetic, RadarData
    import kirchhoff_layered_oracle as lo
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU mode")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    result = {"script": "bench_kirchhoff_layered", "steps": a.steps, "warmup": a.warmup, "l2_flush_mib": 256,
              **gpu_info(), "shapes": {}}
    for shape in a.shapes.split(","):
        S, T = (int(s) for s in shape.split("x"))
        tt, dist, tint = synthetic.geometry(S, T)
        dat = RadarData(np.zeros((1, 1), np.float32), dt=synthetic.DT, travel_time=tt, dist=dist, trace_int=tint)
        dat.snum, dat.tnum = S, T
        v_lay = ml.rms_velocity(tt, ml.getVelocityProfile(dat, synthetic.layered_velocity(tt)))
        g = torch.Generator(device="cuda").manual_seed(S * 131 + T)
        x = torch.randn((S, T), generator=g, device="cuda", dtype=torch.float32)
        out = torch.empty((S, T), dtype=torch.float32, device="cuda")
        vels = {"constant": 1.69e8, "layered": v_lay}
        times = {k: [] for k in vels}
        for it in range(a.warmup + a.steps):
            for kind, v in vels.items():
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ml.kirchhoff_device(x, tt, dist, v, False, out=out)
                e1.record()
                torch.cuda.synchronize()
                if it >= a.warmup:
                    times[kind].append(e0.elapsed_time(e1))
        rec = {}
        traces = np.unique(np.linspace(0, T - 1, a.parity_traces).astype(int)).tolist()
        for kind, v in vels.items():
            ml.enable_kirchhoff_stats(True)
            ml.kirchhoff_device(x, tt, dist, v, False, out=out)
            pairs, exact = ml.kirchhoff_stats()
            kernel = ml.kirchhoff_last_kernel()
            ml.enable_kirchhoff_stats(False)
            got = ml.kirchhoff_device(x, tt, dist, v, False, out=out)[:, traces].double().cpu().numpy()
            ref = lo.kirchhoff_sparse(x, tt, dist, v, False, traces)
            ms = float(np.median(times[kind]))
            rec[kind] = {"ms_per_step": ms, "ms_min": float(np.min(times[kind])), "ms_max": float(np.max(times[kind])),
                         "kernel": kernel, "pairs": int(pairs), "exact_pairs": int(exact),
                         "pairs_per_s": pairs / (ms * 1e-3),
                         "parity_rel_l2": float(np.linalg.norm(got - ref) / np.linalg.norm(ref)),
                         "parity_traces": traces}
        rec["v_range"] = [float(v_lay.max()), float(v_lay.min())]
        result["shapes"]["%dx%d" % (S, T)] = rec
        del x, out
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
