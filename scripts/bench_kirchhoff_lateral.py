"""Kirchhoff migration with a laterally varying velocity on one GPU, against the layered (one profile) kernels; prints one
JSON line.

    python scripts/bench_kirchhoff_lateral.py [--steps 10] [--warmup 3] [--shapes 2048x4096,8192x65536]

Shapes are snum x tnum, 10 ns sampling, 5 m trace spacing, seeded normal noise on the device.  Per shape four velocity
fields alternate step by step in one process, with a 256 MiB L2 flush before every timed call:
  layered_tile     the firn profile (synthetic.layered_velocity -> getVelocityProfile -> rms_velocity), automatic path
  layered_general  the same vector through the vz general kernel (KIRCHHOFF_GENERAL)
  grid_runs        a 5-strip rectangular (v, z, x) grid table: wide runs, the per-run table path
  per_trace        the firn profile scaled by 1 + 0.03 x / T: one profile per trace, the lateral general kernel
Step time is the median CUDA-event time of the whole call (host-side validation and the profile upload included);
kernel_ms is the summed kernel time of the far-field sum (impdar_b200_kernel_timer) in one extra call.  Pairs come from
the kernel counters in one extra call; parity is rel-L2 against the per-column float64 reference on sampled traces
(run edges included).  The grid table's field is built on the host once per shape (CPU time, host_field_s); at tnum >
4096 from a 4096-trace copy of the geometry (griddata over every sample of the headline image takes minutes), each
trace taking the profile of the nearest copy trace.  --sweep runs, at the first shape only, fields of four profiles in
blocks of w traces through both sides of the dispatch (forced), which sets the run-width threshold.  The GPU name,
power limit and SM clock are read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

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


def grid_field(ml, RadarData, synthetic, tt, dist, S, T):
    """(profiles, col_profile, host CPU seconds) of the 5-strip grid table (tests/test_kirchhoff_lateral.grid_table)."""
    from test_kirchhoff_lateral import grid_table
    Tc = min(T, 4096)
    sel = np.linspace(0, T - 1, Tc).round().astype(int)
    dat = RadarData(np.zeros((1, 1), np.float32), dt=synthetic.DT, travel_time=tt, dist=dist[sel],
                    trace_int=np.full(Tc, 5.0))
    dat.snum, dat.tnum = S, Tc
    t0 = time.process_time()
    prof, colp_c = ml.lateral_rms_field(dat, grid_table(dat))
    host_s = time.process_time() - t0
    colp = colp_c[np.clip(np.searchsorted(sel, np.arange(T)), 0, Tc - 1)] if Tc < T else colp_c
    return prof, colp, host_s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="2048x4096,8192x65536")
    ap.add_argument("--parity-traces", type=int, default=4)
    ap.add_argument("--sweep", default="4,16,64,256", help="run widths of the dispatch sweep ('' to skip)")
    a = ap.parse_args()
    if a.steps < 10 or a.warmup < 3:
        raise SystemExit("need --steps >= 10 and --warmup >= 3")
    import torch
    import impdar_b200  # noqa: F401
    from impdar_b200 import _lib, migrationlib as ml, synthetic, RadarData
    import kirchhoff_layered_oracle as lo
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU mode")
    lib = _lib.load()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    result = {"script": "bench_kirchhoff_lateral", "steps": a.steps, "warmup": a.warmup, "l2_flush_mib": 256,
              **gpu_info(), "shapes": {}}

    def kernel_ms(call):
        lib.impdar_b200_kernel_timer(1)
        call()
        torch.cuda.synchronize()
        tot = 0.0
        for name in (b"kirch_tile_kernel", b"kirch_table_kernel", b"kirch_general_kernel",
                     b"kirch_general_lateral_kernel"):
            ms, n = ctypes.c_double(0), ctypes.c_int(0)
            lib.impdar_b200_kernel_timer_read(name, ctypes.byref(ms), ctypes.byref(n))
            tot += ms.value
        lib.impdar_b200_kernel_timer(0)
        return tot

    def timed(calls, steps, warmup):
        times = {k: [] for k in calls}
        for it in range(warmup + steps):
            for kind, (mode, fn) in calls.items():
                ml.set_kirchhoff_mode(mode)
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                ml.set_kirchhoff_mode(0)
                if it >= warmup:
                    times[kind].append(e0.elapsed_time(e1))
        return times

    for si, shape in enumerate(a.shapes.split(",")):
        S, T = (int(s) for s in shape.split("x"))
        tt, dist, tint = synthetic.geometry(S, T)
        dat = RadarData(np.zeros((1, 1), np.float32), dt=synthetic.DT, travel_time=tt, dist=dist, trace_int=tint)
        dat.snum, dat.tnum = S, T
        v_lay = ml.rms_velocity(tt, ml.getVelocityProfile(dat, synthetic.layered_velocity(tt)))
        g_prof, g_colp, host_s = grid_field(ml, RadarData, synthetic, tt, dist, S, T)
        p_prof = v_lay[None, :] * (1 + 0.03 * np.arange(T) / T)[:, None]
        p_colp = np.arange(T)
        g = torch.Generator(device="cuda").manual_seed(S * 131 + T)
        x = torch.randn((S, T), generator=g, device="cuda", dtype=torch.float32)
        out = torch.empty((S, T), dtype=torch.float32, device="cuda")
        fields = {
            "layered_tile": (0, lambda: ml.kirchhoff_device(x, tt, dist, v_lay, False, out=out), None),
            "layered_general": (1, lambda: ml.kirchhoff_device(x, tt, dist, v_lay, False, out=out), None),
            "grid_runs": (0, lambda: ml.kirchhoff_lateral_device(x, tt, dist, g_prof, g_colp, False, out=out),
                          (g_prof, g_colp)),
            "per_trace": (0, lambda: ml.kirchhoff_lateral_device(x, tt, dist, p_prof, p_colp, False, out=out),
                          (p_prof, p_colp)),
        }
        times = timed({k: (m, fn) for k, (m, fn, _) in fields.items()}, a.steps, a.warmup)
        rec = {"host_field_s": host_s, "host_field_traces": min(T, 4096), "grid_runs_profiles": int(g_prof.shape[0])}
        for kind, (mode, fn, field) in fields.items():
            ml.set_kirchhoff_mode(mode)
            kms = kernel_ms(fn)
            ml.enable_kirchhoff_stats(True)
            fn()
            pairs, exact = ml.kirchhoff_stats()
            kernel = ml.kirchhoff_last_kernel()
            ml.enable_kirchhoff_stats(False)
            fn()
            ml.set_kirchhoff_mode(0)
            colp = field[1] if field else np.zeros(T, dtype=int)
            edges = np.flatnonzero(np.diff(colp))[:2]
            traces = np.unique(np.r_[np.linspace(0, T - 1, a.parity_traces).astype(int), edges, edges + 1]).tolist()
            got = out[:, traces].double().cpu().numpy()
            # per-column reference: trace t with its own profile
            ref = np.column_stack([lo.kirchhoff_sparse(x, tt, dist, field[0][colp[t]] if field else v_lay, False,
                                                       [t])[:, 0] for t in traces])
            ms = float(np.median(times[kind]))
            rec[kind] = {"ms_per_step": ms, "ms_min": float(np.min(times[kind])), "ms_max": float(np.max(times[kind])),
                         "kernel_ms": kms, "kernel": kernel, "pairs": int(pairs), "exact_pairs": int(exact),
                         "pairs_per_s": pairs / (ms * 1e-3), "pairs_per_s_kernel": pairs / (kms * 1e-3) if kms else None,
                         "parity_rel_l2": float(np.linalg.norm(got - ref) / np.linalg.norm(ref)),
                         "parity_traces": traces}
        if si == 0 and a.sweep:
            base = v_lay[None, :] * np.array([1.0, 0.93, 1.05, 0.97])[:, None]
            sweep = {}
            calls = {}
            for w in (int(s) for s in a.sweep.split(",")):
                colp = (np.arange(T) // w) % 4
                for mode, name in ((1, "general"), (2, "runs")):
                    calls["w%d_%s" % (w, name)] = (mode, lambda c=colp: ml.kirchhoff_lateral_device(
                        x, tt, dist, base, c, False, out=out))
            st = timed(calls, a.steps, a.warmup)
            for k, v in st.items():
                sweep[k] = {"ms_per_step": float(np.median(v)), "ms_min": float(np.min(v))}
            rec["run_width_sweep"] = sweep
        result["shapes"]["%dx%d" % (S, T)] = rec
        del x, out
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
