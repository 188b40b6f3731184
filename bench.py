#!/usr/bin/env python
"""Benchmark of the B200 migration/filtering hot path (contract: task prompt, SURVEY.md 8d).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  Default workload = the north-star target (BASELINE.json): Kirchhoff migration of ONE
65536-trace x 8192-sample radargram (configs[4]), output-trace ranges sharded over the N ranks with the aperture-halo
exchange and the gather of the output blocks INSIDE the timed step ("scaling": "strong"; N = 1 is the same image on
one GPU).  Next to the headline the line carries `records`: Stolt on the same 65536 x 8192 array (1 GPU) and the
config-2 Kirchhoff (4096 x 2048, one independent radargram per GPU).  A "step" is one pass of the path over one
radargram.

  value      migrated samples/s, whole job, inputs resident in HBM, CUDA-event timed (max over ranks)
  e2e        same metric through the reference-facing plugin call (RadarData.migrate on HOST numpy data:
             H2D + kernels + D2H inside the timed region)
  roofline   the workload's bound (SURVEY.md 8d): HBM bytes for Stolt/filters, (sample, trace) pairs for
             Kirchhoff, complex MACs for phase shift
  parity     relative L2 / max-abs of the BENCHMARKED output against the float64 oracle (oracle/) on a sample of
             output traces, computed after the timed region
  cpu_baseline  the reference's own loop (baseline/_ref, kind "reference"; the oracle's reference-cost port when
             baseline/_ref is absent) on a bounded sample, 1 host core
  --impl reference   the reference's CPU implementation on all usable host cores, no GPU involved
  --dump-outputs DIR after the timed steps, rank 0 writes the output its last timed step returned as DIR/<record>.npy
             (headline: DIR/<workload>.npy; sub-records under their `records` key), at most DUMP_BYTES in all: an
             output that does not fit its share is sampled to every row of a fixed, seeded set of output traces
             (output_sample).  The inputs are seeded, so two builds run with the same arguments compare file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

VEL_K = 1.69e8
VEL_S = 1.68e8
DUMP_BYTES = 60 * 1000 * 1000     # --dump-outputs: all arrays together, .npy headers included, stay below 64 MB


def output_sample(t, budget, seed=0):
    """float32 / float64 host copy of the output tensor `t` (..., T) in at most `budget` bytes of data: the whole
    tensor when it fits, else every row at a seeded, sorted choice of the T output traces (the same columns for the
    same shape and budget in every run)."""
    import torch
    if t.dtype not in (torch.float32, torch.float64):
        t = t.float()
    T = t.shape[-1]
    col_bytes = t.numel() // T * t.element_size()
    if col_bytes * T > budget:
        k = budget // col_bytes
        if k < 1:
            raise ValueError("one output trace of a %s tensor is larger than the %d-byte dump budget"
                             % (tuple(t.shape), budget))
        cols = np.sort(np.random.default_rng(seed).choice(T, k, replace=False))
        t = t.index_select(-1, torch.as_tensor(cols, device=t.device))
    return t.detach().cpu().numpy()


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback", 1965.0


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler(object):
    """SM clock / throttle-reason sampling DURING the timed region (NVML, 1 ms period for the first 16 samples, then 20 ms; the nvidia-smi
    query line of B200_PROFILING.md reads the same counters)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.sm = []
        self.reasons = set()
        self.smmax = None
        self.stop_flag = False
        self.collect = False   # the thread starts (and initialises NVML) before the warm-up; samples count only
        self.th = None         # while the timed region runs
        self.err = None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if visible:
                try:
                    idx = int(visible.split(",")[self.gpu])
                except Exception:
                    idx = self.gpu
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.smmax = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown,
                     "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown,
                     "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
            while not self.stop_flag:
                if self.collect:
                    self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    for n, bit in names.items():
                        if r & bit:
                            self.reasons.add(n)
                    # dense at first (the short workloads last a few ms), then 50 Hz: a thread that wakes every
                    # millisecond competes with the enqueueing thread for the interpreter lock
                    time.sleep(0.001 if len(self.sm) < 16 else 0.02)
                else:
                    time.sleep(0.002)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.th is not None:
            self.th.join(timeout=2)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.smmax,
               "reasons": sorted(self.reasons), "samples": len(self.sm)}
        if self.err:
            out["error"] = self.err
        return out


# ------------------------------------------------------------------------------ per-kernel timing
def kernel_times(names):
    """{kernel: (avg ms per launch, launches)} from the library's CUDA-event brackets (recorded on the stream
    the kernel is launched on, inside the timed region)."""
    import ctypes
    from impdar_b200 import _lib
    lib = _lib.load()
    out = {}
    for n in names:
        ms, cnt = ctypes.c_double(0.0), ctypes.c_int(0)
        _lib.check(lib.impdar_b200_kernel_timer_read(n.encode(), ctypes.byref(ms), ctypes.byref(cnt)))
        if cnt.value:
            out[n] = (ms.value / cnt.value, cnt.value)
    return out


def ncu_traffic(kernel, kernel_ms=None):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/traffic.json,
    written by scripts/ncu_summary.py), or None.  The capture is of ONE launch shape per kernel (the workload named
    in scripts/gpu_round.sh): when the launch measured here lasts very differently from the captured one it is a
    different shape and the figure does not apply."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        d = json.load(f)
    e = d.get(kernel)
    if not e:
        return None
    if kernel_ms and e.get("ncu_ms") and not (0.6 < e["ncu_ms"] / kernel_ms < 1.6):
        return None
    return e.get("dram_bytes")


def hbm_kernel_roofline(wl, table, ms_step, bytes_per_sample_step, hbm_gbs):
    """HBM-bound paths: `table` = {kernel: algorithmic bytes per launch}.  The dominant kernel (largest total time
    in the timed region) gives achieved/peak/frac; the whole step on SURVEY 8d's byte model is reported beside it."""
    kt = kernel_times(list(table))
    step_gbs = wl.units * bytes_per_sample_step / (ms_step * 1e-3) / 1e9
    r = {"bound": "hbm", "peak": hbm_gbs, "unit": "GB/s", "step_bytes_per_sample": bytes_per_sample_step,
         "step_achieved": step_gbs, "step_frac": step_gbs / hbm_gbs}
    if not kt:
        r.update({"achieved": step_gbs, "frac": step_gbs / hbm_gbs, "traffic": None, "kernel": "whole step"})
        return r
    dom = max(kt, key=lambda k: kt[k][0] * kt[k][1])
    ms, cnt = kt[dom]
    gbs = table[dom] / (ms * 1e-3) / 1e9
    r.update({"achieved": gbs, "frac": gbs / hbm_gbs, "kernel": dom, "kernel_ms": ms, "kernel_launches": cnt,
              "algorithmic_bytes_per_launch": table[dom], "traffic": ncu_traffic(dom, ms),
              "kernel_share_of_step": ms * cnt / (ms_step * wl.steps_timed),
              "kernels": {k: {"ms": v[0], "launches": v[1], "GBps": table[k] / (v[0] * 1e-3) / 1e9} for k, v in kt.items()}})
    return r


# --------------------------------------------------------------------------------------- workloads
class Workload(object):
    name = ""
    dtype = "f32"
    scaling = "weak"

    def __init__(self, args, rank, world):
        self.args, self.rank, self.world = args, rank, world

    def l2_note(self):
        return "L2 flushed between timed steps (256 MiB write)"

    parallelism = "independent radargrams per GPU, no collective"
    steps_timed = 1

    def parallelism_for(self, world):
        return self.parallelism

    def config(self, world=None):
        """The `config` object of the JSON line - the same for this arm and for `--impl reference` at the same --gpus."""
        world = self.world if world is None else world
        return {"workload": self.name, "snum": self.S, "tnum": getattr(self, "T_full", self.T), "l2": self.l2_note(),
                "parallelism": "1 process per GPU, %s" % self.parallelism_for(world)}

    def exchange_note(self):
        return None

    def parity(self):
        return None

    def output(self):
        """The device tensor the last step() returned to its caller (--dump-outputs)."""
        return self.out

    def teardown(self):
        """Drop every tensor so that the next record starts from an empty device."""
        import torch
        from impdar_b200 import device
        for k in list(self.__dict__):
            if isinstance(self.__dict__[k], torch.Tensor):
                del self.__dict__[k]
        device.free_workspaces()
        from impdar_b200 import parallel
        parallel.free_exchange_buffers()
        torch.cuda.empty_cache()


def ncu_extra(kernel):
    """Pipe counters of the committed `ncu --set full` capture of `kernel` (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        e = json.load(f).get(kernel)
    return e.get("pipes") if e else None


KIRCH_KERNELS = ("kirch_tile_kernel", "kirch_table_kernel", "kirch_general_kernel")
# One 4-byte gather per (output sample, input trace) pair is the floor of the diffraction sum as ImpDAR defines it
# (nearest-sample pick, mig_python.py:49-53).  The SM's shared-memory / L1 data pipe delivers one 128-byte wavefront
# (32 lanes x 4 B) per clock: 148 SM x 32 pair/clk x 1.965 GHz.  The tile kernel reads its operands from shared memory
# (one conflict-free wavefront per warp request whatever the alignment); the table kernel's misaligned global gathers
# cost ~1.28 wavefronts per request (ncu, profiles/), the general kernel is issue-bound well below either.
KIRCH_PIPE_PEAK = 148 * 32 * 1.965e9
KIRCH_SURVEY_PEAK = 4.0e12      # SURVEY.md 8d's issue-model ceiling (9 FP32/INT + 1 MUFU + 1 gather per pair)


def kirchhoff_roofline(wl, ms, hbm_gbs, src, pairs_this_rank, pairs_all, exact_pairs):
    """SURVEY.md 8d: Kirchhoff is not HBM-bound; unit of work = one (output sample, in-aperture input trace) pair."""
    kt = kernel_times(list(KIRCH_KERNELS))
    if kt:
        kname = max(kt, key=lambda k: kt[k][0] * kt[k][1])
        kms, kcnt = kt[kname]
    else:
        kname, kms, kcnt = "whole step", ms, wl.steps_timed
    steps = wl.steps_timed
    kms_step = kms * kcnt / steps                      # the exchange pipeline launches the kernel once per row chunk
    pairs_s = pairs_this_rank / (kms_step * 1e-3)
    hbm = wl.S * wl.T * 8 / (ms * 1e-3) / 1e9
    return {"bound": "sm_data_pipe_wavefronts", "achieved": pairs_s, "peak": KIRCH_PIPE_PEAK, "unit": "pair/s",
            "frac": pairs_s / KIRCH_PIPE_PEAK, "traffic": ncu_traffic(kname, kms),
            "kernel": kname, "kernel_ms": kms, "kernel_ms_per_step": kms_step, "kernel_launches": kcnt,
            "kernel_share_of_step": kms * kcnt / (ms * steps),
            "peak_model": "one 4-byte shared-memory/L1 gather per pair, 128 B per SM per clock: 148 x 32 x 1.965e9",
            "survey_issue_model_peak": KIRCH_SURVEY_PEAK, "frac_of_survey_model": pairs_s / KIRCH_SURVEY_PEAK,
            "pairs_this_rank_per_step": pairs_this_rank, "pairs_whole_image": pairs_all, "exact_fp64_pairs": exact_pairs,
            "step_pairs_per_s_all_ranks": pairs_all / (ms * 1e-3),
            "ncu_pipe_counters": ncu_extra(kname),
            "hbm_compulsory_gbs": hbm, "hbm_frac_of_%s_peak" % src: hbm / hbm_gbs}


def kirchhoff_parity(out_dev, x_dev, tt, dist, vel, nearfield, traces, n_rows):
    """rel-L2 / max-abs of the benchmarked output (device fp32, full image) against oracle.migration.kirchhoff_sparse
    (mig_python.py:35-60 restated; float64, fed the float64 upcast of the same fp32 input) on `traces` x n_rows
    strided output samples."""
    from oracle import migration as om
    S = out_dev.shape[0]
    rows = np.unique(np.concatenate([np.linspace(0, S - 1, n_rows).astype(int), [0, 1, S - 2, S - 1]]))
    traces = sorted(set(int(t) for t in traces))
    t0 = time.perf_counter()
    want = om.kirchhoff_sparse(x_dev, tt, dist, vel, nearfield, traces, rows)
    got = out_dev[rows][:, traces].double().cpu().numpy()
    den = float(np.linalg.norm(want))
    return {"rel_l2": float(np.linalg.norm(got - want)) / den if den else float(np.linalg.norm(got - want)),
            "max_abs": float(np.max(np.abs(got - want))), "ref_max_abs": float(np.max(np.abs(want))),
            "n_traces": len(traces), "n_rows": int(len(rows)), "tolerance_rel_l2": 1e-5,
            "oracle": "oracle.migration.kirchhoff_sparse (float64, mig_python.py:35-60)", "oracle_s": time.perf_counter() - t0}


_REF_INPUT = {}


def reference_kirchhoff_input(S, T_used, seed, vel=VEL_K):
    """Full-size float64 inputs of migrationKirchhoffLoop, prepared the way migrationKirchhoff does (mig_python.py:93-108).
    Cached per process (and shared copy-on-write with forked workers): the preparation is O(N) and not what is timed."""
    key = (S, T_used, seed, vel)
    if key not in _REF_INPUT:
        _REF_INPUT.clear()
        rng = np.random.default_rng(seed)
        data = rng.standard_normal((S, T_used))
        tt_sec = np.arange(S) * 1e-8
        zs = vel * tt_sec / 2.0
        _REF_INPUT[key] = (data, np.gradient(data, tt_sec, axis=0), tt_sec, np.arange(T_used) * 5.0, zs, zs ** 2.)
    return _REF_INPUT[key]


def reference_kirchhoff_sample(S, T_full, T_used, n_out, seed, vel=VEL_K, nearfield=False):
    """Time the reference's own migrationKirchhoffLoop (baseline/_ref, mig_python.py:35-60) - or the oracle's
    reference-cost port when baseline/_ref is absent - for `n_out` output samples of output trace 0 (the reference's
    loop bounds tnum=1, snum=n_out) against an (S, T_used) float64 input.  The loop's cost per output sample is one
    argmin over an (S x tnum) matrix, i.e. linear in tnum, so with T_used < T_full (bounded memory and time) the
    full-width rate is rate * T_used / T_full; the factor is returned.  -> (seconds, n_out, kind, scale)"""
    data, gradD, tt_sec, dist, zs, zs2 = reference_kirchhoff_input(S, T_used, seed, vel)
    mig = np.zeros_like(data)
    from oracle import _refimport
    with _quiet():                                   # the reference prints a progress line per output trace
        if _refimport.vendored_available():
            mp_ref = _refimport.import_vendored_mig_python()
            t0 = time.perf_counter()
            with np.errstate(invalid='ignore', divide='ignore'):
                mp_ref.migrationKirchhoffLoop(data, mig, 1, n_out, dist, zs, zs2, tt_sec, vel, gradD, np.max(tt_sec), nearfield)
            secs = time.perf_counter() - t0
            kind = "reference"
        else:
            from oracle import migration as om
            t0 = time.perf_counter()
            om.kirchhoff_loops(data, tt_sec * 1e6, dist / 1e3, vel, nearfield, tnum=1, snum=n_out)
            secs = time.perf_counter() - t0
            kind = "port"
    return secs, n_out, kind, float(T_used) / float(T_full)


class KirchhoffC2(Workload):
    """configs[1]: Kirchhoff, 4096 traces x 2048 samples, v = 1.69e8; one independent radargram per GPU."""
    name = "kirchhoff_4096tr_x_2048smp_v1.69e8"
    e2e_api = ("impdar_b200.RadarData.migrate(mtype='kirch') on host numpy data (pinned input): "
               "impdar_kirchhoff_host_pipelined_f64, 8 row chunks, upload | kernels | float64 download overlapped")
    S, T = 2048, 4096
    nearfield = False
    parallelism = "independent radargrams per GPU, no collective"

    def setup(self):
        import torch
        from impdar_b200 import synthetic
        self.tt, self.dist, self.trace_int = synthetic.geometry(self.S, self.T)
        self.x = synthetic.diffractor_radargram(self.S, self.T, seed=2 + self.rank, n_diffractors=64)
        self.host = torch.empty((self.S, self.T), dtype=torch.float32).pin_memory()
        self.host.copy_(self.x)
        self.out = torch.empty((self.S, self.T), dtype=torch.float32, device="cuda")
        self.units = self.S * self.T
        from impdar_b200 import migrationlib as ml
        ml.enable_kirchhoff_stats(True)
        ml.kirchhoff_device(self.x, self.tt, self.dist, VEL_K, self.nearfield, out=self.out)
        torch.cuda.synchronize()
        self.pairs, self.exact_pairs = ml.kirchhoff_stats()
        ml.enable_kirchhoff_stats(False)

    def step(self):
        from impdar_b200 import migrationlib as ml
        ml.kirchhoff_device(self.x, self.tt, self.dist, VEL_K, self.nearfield, out=self.out)

    def e2e_step(self):
        import impdar_b200
        d = impdar_b200.RadarData(self.host.numpy(), dt=1e-8, travel_time=self.tt, dist=self.dist,
                                  trace_int=self.trace_int)
        with _quiet():
            d.migrate(mtype='kirch', vel=VEL_K, nearfield=self.nearfield)
        return self.S * self.T * 4, d.data.nbytes, float(d.data[self.S // 2, self.T // 2])

    def roofline(self, ms, hbm_gbs, src):
        return kirchhoff_roofline(self, ms, hbm_gbs, src, self.pairs, self.pairs, self.exact_pairs)

    def parity(self):
        T = self.T
        traces = [0, 1, T // 2, T - 1] + list(np.random.default_rng(11).integers(0, T, 28))
        return kirchhoff_parity(self.out, self.x, self.tt, self.dist, VEL_K, self.nearfield, traces, 512)

    def cpu_sample(self, n_samples):
        secs, n, kind, scale = reference_kirchhoff_sample(self.S, self.T, self.T, n_samples, seed=2)
        return secs, n * scale, kind, ("migrationKirchhoffLoop(tnum=1, snum=%d) of %s against a full %d x %d float64 input"
                                       % (n_samples, "baseline/_ref (mig_python.py:35-60)" if kind == "reference" else
                                          "the oracle port", self.S, self.T))

    cpu_default_n = 48
    ref_T_used = 4096
    ref_n = 2


class KirchhoffC5(KirchhoffC2):
    """configs[4] = the north-star target: ONE radargram of 65536 traces x 8192 samples.  N ranks: equal output-trace
    ranges, every rank receives only the input columns its range can reach (range + one aperture
    each side) from the rank that holds the radargram, and the (snum, range) output blocks are gathered straight into
    the final image - both exchanges inside the timed step, overlapped with the kernels in bottom-up row chunks."""
    name = "kirchhoff_65536tr_x_8192smp"
    S, T = 8192, 65536
    scaling = "strong"
    cpu_default_n = 8
    ref_T_used = 8192
    ref_n = 1
    e2e_api = ("impdar_b200.RadarData.migrate(mtype='kirch') on a host numpy radargram (pinned, rank 0); N > 1: "
               "impdar_b200.parallel.kirchhoff_sharded_host - rank 0 uploads, halo exchange, kernels, gather to rank 0, "
               "float64 download")

    def parallelism_for(self, world):
        if world == 1:
            return "one GPU, whole image"
        return ("one radargram, equal output-trace ranges per GPU; halo exchange of the input columns and gather of the "
                "output blocks on rank 0 inside the timed step")

    def exchange_note(self):
        """How the exchange of the timed steps actually travelled (decided at run time: peer mappings can be refused)."""
        if self.world == 1:
            return None
        if self.parallel.peer_output_active():
            inp = ("rank 0 pushes every rank's input-column window into that rank's peer-mapped buffer (strided 2-D copies "
                   "over NVLink, one-element NCCL broadcast per row chunk as the signal)" if self.parallel.peer_input_active()
                   else "NCCL all_to_all send/recv of the input columns")
            return ("%s; the diffraction-sum kernels store their output blocks straight into rank 0's image through "
                    "peer-mapped memory (CUDA IPC over NVLink), one-element NCCL all_reduce per row chunk as completion "
                    "signal" % inp)
        return "NCCL all_to_all send/recv of the input columns and of the output blocks, one per row chunk"

    def setup(self):
        import torch
        from impdar_b200 import synthetic, parallel
        self.tt, self.dist, self.trace_int = synthetic.geometry(self.S, self.T)
        if self.rank == 0:
            self.x = synthetic.diffractor_radargram(self.S, self.T, seed=5, n_diffractors=1024)
            self.host = torch.empty((self.S, self.T), dtype=torch.float32).pin_memory()
            self.host.copy_(self.x)
        else:
            if self.exchange == "broadcast":
                self.x = torch.empty((self.S, self.T), dtype=torch.float32, device="cuda")
            else:                                      # halo exchange: the other ranks never hold the whole image
                self.x = torch.empty((1, 1), dtype=torch.float32, device="cuda").expand(self.S, self.T)
            self.host = "peer"
        self.units = self.S * self.T / self.world   # per rank share; value is whole-job
        self.parallel = parallel
        self.ranges = parallel.kirchhoff_output_ranges(self.T, self.world, self.tt, self.dist, VEL_K)
        self.xb, self.xe = self.ranges[self.rank]
        self.result = None
        self.count_pairs()

    exchange = os.environ.get("IMPDAR_C5_EXCHANGE", "halo")          # development A/B switch: "halo" | "broadcast"

    def step(self):
        kw = {}
        if os.environ.get("IMPDAR_C5_CHUNKS"):          # development A/B switch for the exchange pipeline: "4" or "1,2,2,1"
            c = os.environ["IMPDAR_C5_CHUNKS"]
            kw["pipeline_chunks"] = [float(v) for v in c.split(",")] if "," in c else int(c)
        self.result = None
        self.result = self.parallel.kirchhoff_sharded_device(
            self.x, self.tt, self.dist, VEL_K, False, rank=self.rank, world=self.world,
            gather=True if self.exchange == "broadcast" else 'src', exchange=self.exchange, **kw)

    def output(self):
        return self.result

    def e2e_step(self):
        if self.world == 1:
            return KirchhoffC2.e2e_step(self)
        h = self.host.numpy() if self.rank == 0 else None
        with _quiet():
            out = self.parallel.kirchhoff_sharded_host(h, self.S, self.T, self.tt, self.dist, VEL_K, False,
                                                       rank=self.rank, world=self.world)
        if self.rank == 0:
            return self.S * self.T * 4, out.nbytes, float(out[self.S // 2, self.T // 2])
        return self.S * self.T * 4, self.S * self.T * 8, 0.0

    def count_pairs(self):
        """(sample, trace) pairs inside the aperture, counted on the device over this rank's output range and
        summed over ranks (one extra untimed call)."""
        import torch
        import torch.distributed as dist
        from impdar_b200 import migrationlib as ml
        ml.enable_kirchhoff_stats(True)
        if self.xe > self.xb:
            # the count depends on the geometry only: run the range on an all-zero input window
            c0, c1 = ml.kirchhoff_input_window(self.S, self.tt, self.dist, VEL_K, self.xb, self.xe)
            win = torch.zeros((self.S, c1 - c0), dtype=torch.float32, device="cuda")
            ml.kirchhoff_window_device(win, c0, self.T, self.tt, self.dist, VEL_K, False, self.xb, self.xe)
            torch.cuda.synchronize()
            pairs, exact = ml.kirchhoff_stats()
            self.kernel_used = ml.kirchhoff_last_kernel()
            del win
        else:
            pairs, exact = 0, 0
            self.kernel_used = "none"
        ml.enable_kirchhoff_stats(False)
        self.pairs_rank = float(pairs)
        t = torch.tensor([float(pairs), float(exact)], dtype=torch.float64, device="cuda")
        if self.world > 1:
            dist.all_reduce(t)
        self.pairs, self.exact_pairs = float(t[0].item()), float(t[1].item())

    def roofline(self, ms, hbm_gbs, src):
        r = kirchhoff_roofline(self, ms, hbm_gbs, src, self.pairs_rank, self.pairs, self.exact_pairs)
        if self.world > 1:
            r["kernel_ms_per_step_by_rank"] = getattr(self, "kernel_ms_by_rank", None)
            r["note"] = ("achieved/peak are per GPU (rank 0's kernel and rank 0's share of the pairs; every rank owns the "
                         "same number of output traces - the table kernels' cost is per trace - so the end ranks, whose "
                         "apertures are cut by the profile ends, count fewer pairs for the same work); the step adds the "
                         "exposed part of the halo exchange")
        return r

    def parity(self):
        if self.rank != 0 or self.result is None:
            return None
        T = self.T
        traces = [0, 1, T - 1]
        for b, e in self.ranges:                       # both sides of every shard boundary
            traces += [min(max(b, 0), T - 1), min(max(e - 1, 0), T - 1)]
        traces += list(np.random.default_rng(12).integers(0, T, 32))
        return kirchhoff_parity(self.result, self.x, self.tt, self.dist, VEL_K, False, traces[:64], 160)

    def cpu_sample(self, n_samples):
        secs, n, kind, scale = reference_kirchhoff_sample(self.S, self.T, self.ref_T_used, n_samples, seed=5)
        return secs, n * scale, kind, (
            "migrationKirchhoffLoop(tnum=1, snum=%d) of %s against an %d x %d float64 input; the loop costs one argmin "
            "over (snum x tnum) per output sample, so the rate at tnum=%d is the measured one x %d/%d"
            % (n_samples, "baseline/_ref (mig_python.py:35-60)" if kind == "reference" else "the oracle port",
               self.S, self.ref_T_used, self.T, self.ref_T_used, self.T))


class StoltC5(Workload):
    """The north-star target shape for Stolt: 65536 traces x 8192 samples on one GPU (replicas for N > 1)."""
    name = "stolt_65536tr_x_8192smp"
    S, T = 8192, 65536

    def setup(self):
        import torch
        from impdar_b200 import synthetic
        self.tt, self.dist, self.trace_int = synthetic.geometry(self.S, self.T)
        self.x = synthetic.diffractor_radargram(self.S, self.T, seed=5 + self.rank, n_diffractors=256)
        self.out = torch.empty((1, 2 * (self.S // 2), self.T), dtype=torch.float32, device="cuda")
        self.units = self.S * self.T
        self.host = torch.empty((self.S, self.T), dtype=torch.float32).pin_memory()
        self.host.copy_(self.x)

    def l2_note(self):
        return "inputs (2 GiB) larger than L2; no flush needed"

    def step(self):
        from impdar_b200 import migrationlib as ml
        self.result = ml.stolt_device(self.x, 1e-8, 5.0, VEL_S, 10, 10, out=self.out)

    def output(self):
        return self.result                             # (2 * (snum // 2), tnum) for a 2-D radargram

    def e2e_step(self):
        import impdar_b200
        d = impdar_b200.RadarData(self.host.numpy(), dt=1e-8, travel_time=self.tt, dist=self.dist,
                                  trace_int=self.trace_int)
        with _quiet():
            d.migrate(mtype='stolt', vel=VEL_S, htaper=10, vtaper=10)
        return self.S * self.T * 4, d.data.nbytes, float(d.data[self.S // 2, self.T // 2])

    def roofline(self, ms, hbm_gbs, src):
        # SURVEY.md 8d: 40 B per real sample = five sweeps that each read and write the (paired-trace complex)
        # image once: rowA fwd (+taper), rowB fwd (+transpose), col (FFT_t, remap, iFFT_t), rowB inv, rowA inv.
        # Every pass kernel therefore moves 8 B per real sample per launch (algorithmic bytes).
        per = float(self.units) * 8
        table = {"stolt_col_kernel": per, "stolt_rowA_kernel": per, "stolt_rowB_kernel": per,
                 "stolt_remap_paired_kernel": per, "stolt_remap_kernel": per}
        r = hbm_kernel_roofline(self, table, ms, 40, hbm_gbs)
        r["compulsory_8B_gbs"] = self.units * 8 / (ms * 1e-3) / 1e9
        return r

    def parity(self):
        """Benchmarked output against oracle.migration.stolt_traces (mig_python.py:126-208 in float64 on the float64
        upcast of the same input; full forward transform, inverse evaluated at the sampled traces)."""
        from oracle import migration as om
        need = self.S * self.T * 8 * 3.5
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = None
        if avail is not None and avail < need:
            return {"skipped": "host has %.0f GB available, the float64 oracle needs %.0f GB at this shape" % (avail / 1e9, need / 1e9)}
        T = self.T
        traces = sorted(set([0, 1, T // 2, T - 2, T - 1] + [int(t) for t in np.random.default_rng(13).integers(0, T, 27)]))
        t0 = time.perf_counter()
        want = om.stolt_traces(self.host.numpy(), 1e-8, self.trace_int, self.dist, VEL_S, 10, 10, traces=traces)
        out = self.out[0] if self.out.dim() == 3 else self.out
        got = out[:, traces].double().cpu().numpy()
        den = float(np.linalg.norm(want))
        return {"rel_l2": float(np.linalg.norm(got - want)) / den, "max_abs": float(np.max(np.abs(got - want))),
                "ref_max_abs": float(np.max(np.abs(want))), "n_traces": len(traces), "n_rows": int(want.shape[0]),
                "tolerance_rel_l2": 1e-5, "oracle": "oracle.migration.stolt_traces (float64, mig_python.py:126-208)",
                "oracle_s": time.perf_counter() - t0}

    def cpu_sample(self, n):
        from oracle import migration as om
        S, T = 1024, 2048   # bounded sample: same per-cell cost (two FITPACK point evaluations per (kz, kx) cell)
        img = self.x if self.x.dim() == 2 else self.x[0]
        x64 = img[:S, :T].double().cpu().numpy()
        stride = max(1, 512 // n)
        rows = len(range(0, S // 2, stride))
        t0 = time.perf_counter()
        om.stolt_loops(x64, 1e-8, np.ones(T) * 5.0, np.arange(T) * 0.005, VEL_S, 10, 10, row_stride=stride)
        return time.perf_counter() - t0, S * T * rows / 512.0, "port", self.cpu_sample_desc % n

    cpu_sample_desc = "oracle.migration.stolt_loops (FITPACK point evaluation per cell) on ~%d of the 512 kz rows of a 1024x2048 crop"
    cpu_default_n = 256


class StoltC4(StoltC5):
    """One configs[3] profile (8192 traces x 2048 samples) through Stolt."""
    name = "stolt_8192tr_x_2048smp"
    S, T = 2048, 8192

    def l2_note(self):
        return "L2 flushed between timed steps (256 MiB write)"


class PipelineC4(Workload):
    """configs[3]: vertical_band_pass(2,10) + hfilt(0,T) + Stolt over profiles of 8192 traces x 2048 samples,
    profiles sharded round-robin over GPUs; one step = `--profiles` profiles per GPU (device resident)."""
    name = "pipeline_vbp_hfilt_stolt_8192tr_x_2048smp"
    e2e_api = "impdar_b200.process.process(dats, vbp=(2,10), hfilt=(0,T), migrate=True) on host numpy profiles (pinned)"
    S, T = 2048, 8192

    def setup(self):
        import torch
        from impdar_b200 import synthetic
        self.P = self.args.profiles
        self.tt, self.dist, self.trace_int = synthetic.geometry(self.S, self.T)
        self.x = torch.stack([synthetic.diffractor_radargram(self.S, self.T, seed=4 + self.rank * self.P + p,
                                                             n_diffractors=16) for p in range(self.P)])
        self.units = self.P * self.S * self.T
        from scipy.signal import butter
        nyq = 0.5 / 1e-8
        self.b, self.a = butter(5, [2e6 / nyq, 10e6 / nyq], 'bandpass')
        self.taper = np.exp(-self.tt * 0.05) / np.exp(-self.tt[0] * 0.05)
        self.host = torch.empty((self.P, self.S, self.T), dtype=torch.float32).pin_memory()
        self.host.copy_(self.x)
        self.e2e_units = self.P * self.S * self.T

    def l2_note(self):
        return "inputs larger than L2" if self.args.profiles * self.S * self.T * 4 > 126e6 else Workload.l2_note(self)

    def step(self):
        from impdar_b200 import filtering as fl, migrationlib as ml
        y = fl.filtfilt_device(self.x, 'f32', self.b, self.a)
        y = fl.horizontalfilt_device(y, 'f32', self.taper, 0, self.T)
        self.out = ml.stolt_device(y, 1e-8, 5.0, VEL_S, 10, 10)

    def e2e_step(self):
        # the call a user of the reference makes for this configuration: process(dats, vbp=(2, 10), hfilt=(0, T),
        # migrate=True) (lib/process.py:151-193) on HOST arrays; impdar_b200.process.process uploads each profile
        # once, runs the three steps device resident and downloads once, several profiles in flight
        import impdar_b200
        h = self.host.numpy()
        dats = [impdar_b200.RadarData(h[p], dt=1e-8, travel_time=self.tt, dist=self.dist, trace_int=self.trace_int)
                for p in range(self.P)]
        with _quiet():
            impdar_b200.process.process(dats, vbp=(2, 10), hfilt=(0, self.T), migrate=True)
        return self.P * self.S * self.T * 4, sum(d.data.nbytes for d in dats), float(dats[-1].data[self.S // 2, self.T // 2])

    def roofline(self, ms, hbm_gbs, src):
        # 8 + 8 + 40 B/sample unfused (SURVEY.md 8d); every kernel of the step moves 8 B/sample algorithmically
        per = float(self.units) * 8
        table = {"filtfilt_kernel": per, "hfilt_kernel": per, "stolt_col_kernel": per, "stolt_rowA_kernel": per,
                 "stolt_rowB_kernel": per, "stolt_remap_paired_kernel": per}
        return hbm_kernel_roofline(self, table, ms, 56, hbm_gbs)

    def cpu_sample(self, n):
        from oracle import filtering as of
        x64 = self.x[0].double().cpu().numpy()
        t0 = time.perf_counter()
        y = of.vertical_band_pass(x64, 1e-8, 2, 10)
        of.horizontalfilt(y, self.tt, 0, self.T)
        t_f = time.perf_counter() - t0
        t_s, cells, _, _ = StoltC5.cpu_sample(self, n)
        # Stolt cost scales with cells: extrapolate it to one full profile, add the measured filters, and report
        # the measured time with the equivalent number of fully processed samples
        t_full = t_f + t_s * (self.S * self.T) / cells
        elapsed = t_f + t_s
        return elapsed, self.S * self.T * elapsed / t_full, "port", self.cpu_sample_desc % n

    cpu_sample_desc = ("oracle vertical_band_pass + horizontalfilt on one full profile (measured) + stolt_loops on ~%d of the "
                       "512 kz rows of a 1024x2048 crop extrapolated by cell count to the profile")
    cpu_default_n = 128


class PhshC3(Workload):
    """configs[2]: phase-shift migration, 16384 traces x 4096 samples; constant velocity (default) or layered."""
    name = "phsh_const_16384tr_x_4096smp"
    S, T = 4096, 16384
    layered = False

    def setup(self):
        import torch
        from impdar_b200 import synthetic, migrationlib as ml
        self.tt, self.dist, self.trace_int = synthetic.geometry(self.S, self.T)
        self.x = synthetic.diffractor_radargram(self.S, self.T, seed=3 + self.rank, n_diffractors=128)
        self.out = torch.empty((self.S, self.T), dtype=torch.float32, device="cuda")
        self.units = self.S * self.T
        self.host = torch.empty((self.S, self.T), dtype=torch.float32).pin_memory()
        self.host.copy_(self.x)
        self.vel_table = synthetic.layered_velocity(self.tt)
        d = type("D", (), {})()
        d.travel_time, d.snum, d.tnum, d.dist = self.tt, self.S, self.T, self.dist
        self.vmig = ml.getVelocityProfile(d, self.vel_table) if self.layered else VEL_K

    def l2_note(self):
        return "inputs (256 MiB) larger than L2; no flush needed"

    def step(self):
        from impdar_b200 import migrationlib as ml
        ml.phase_shift_device(self.x, 1e-8, 5.0, self.tt, self.vmig, 10, 10, out=self.out)

    def e2e_step(self):
        import impdar_b200
        from impdar_b200 import migrationlib as ml
        d = impdar_b200.RadarData(self.host.numpy(), dt=1e-8, travel_time=self.tt, dist=self.dist,
                                  trace_int=self.trace_int)
        with _quiet():
            ml.migrationPhaseShift(d, vel=self.vel_table if self.layered else VEL_K, htaper=10, vtaper=10)
        return self.S * self.T * 4, d.data.nbytes, float(d.data[self.S // 2, self.T // 2])

    def roofline(self, ms, hbm_gbs, src):
        nt = 1 << (self.S - 1).bit_length()
        K = self.T // 2 + 1
        macs = float(nt) * K * self.S   # complex MACs over (w, kx >= 0, tau)
        kt = kernel_times(["phsh_const_tc_kernel", "phsh_const_pair_kernel", "phsh_layered_pair_kernel"])
        if not self.layered and "phsh_const_tc_kernel" in kt:
            # constant velocity on the tensor cores: per-kx complex GEMM, tcgen05 kind::tf32 with the 3xTF32 split.
            # algorithmic work = 8 real flop per complex MAC; the kernel executes 3x that on the tensor pipe.  TF32 runs
            # at half the bf16 rate: peak = the driver-measured dense bf16 figure / 2.
            kms, kcnt = kt["phsh_const_tc_kernel"]
            bf16 = 1635.7
            pth = os.path.join(ROOT, "MEASURED_PEAKS.json")
            if os.path.exists(pth):
                with open(pth) as f:
                    bf16 = float(json.load(f).get("bf16_tflops", bf16))
            tf = 8.0 * macs / (kms * 1e-3) / 1e12
            return {"bound": "tensor", "achieved": tf, "peak": bf16 / 2.0, "unit": "TFLOP/s", "frac": tf / (bf16 / 2.0),
                    "traffic": ncu_traffic("phsh_const_tc_kernel", kms), "kernel": "phsh_const_tc_kernel", "kernel_ms": kms,
                    "kernel_launches": kcnt, "kernel_share_of_step": kms * kcnt / (ms * self.steps_timed),
                    "cmacs_per_launch": macs, "executed_tensor_tflops": 3.0 * tf,
                    "peak_model": "TF32 dense = measured bf16 dense / 2; 3xTF32 executes three products per algorithmic one",
                    "ncu_pipe_counters": ncu_extra("phsh_const_tc_kernel"),
                    "note": "bound by the SIMT operand generation (sincospi seeds, recurrences, hi/lo split, shared-memory "
                            "stores), not by the tensor pipe (sm__pipe_tensor_cycles_active 21 %)"}
        peak = 148 * 128 * 1.965e9 / 6.0   # 6 FP32 issue slots per complex multiply-accumulate
        if self.layered:
            peak = 148 * 16 * 1.965e9 / 3.0   # MUFU bound: rsqrt + sin + cos per (tau, w, k)
        kname = "phsh_layered_pair_kernel" if self.layered else "phsh_const_pair_kernel"
        kms, kcnt = kt.get(kname, (ms, self.steps_timed))
        return {"bound": "fp32_simt" if not self.layered else "mufu", "achieved": macs / (kms * 1e-3), "peak": peak,
                "unit": "cmac/s", "frac": macs / (kms * 1e-3) / peak, "traffic": ncu_traffic(kname, kms),
                "kernel": kname, "kernel_ms": kms, "kernel_launches": kcnt,
                "kernel_share_of_step": kms * kcnt / (ms * self.steps_timed),
                "cmacs_per_launch": macs}

    def cpu_sample(self, n):
        from oracle import migration as om
        S, T = self.S, 256   # bounded: all frequencies, a 256-trace crop, n output taus
        x64 = self.x[:, :T].double().cpu().numpy()
        tap = om.phsh_taper(x64, 10, 10)
        nt, kx, ws, FK = om.phase_shift_spectrum(tap, 1e-8, np.ones(T) * 5.0, None)
        t0 = time.perf_counter()
        if self.layered:
            om.phase_shift_layered_tk(FK, kx, ws, 1e-8, self.tt, np.asarray(self.vmig), tau_end=n)
        else:
            om.phase_shift_const_tk(FK, kx, ws, 1e-8, S, VEL_K, tau_end=n)
        return time.perf_counter() - t0, n * T, "port", self.cpu_sample_desc % n

    cpu_sample_desc = "oracle phase-shift recurrence (vectorised over (w,kx), sequential in tau): %d taus x 256 traces, all frequencies"
    cpu_default_n = 256


class PhshC3Layered(PhshC3):
    name = "phsh_layered_16384tr_x_4096smp"
    layered = True


WORKLOADS = {"kirchhoff": KirchhoffC2, "kirchhoff_c5": KirchhoffC5, "stolt": StoltC5, "stolt_c4": StoltC4,
             "pipeline": PipelineC4, "phsh": PhshC3, "phsh_layered": PhshC3Layered}


class _quiet(object):
    def __enter__(self):
        self._so = sys.stdout
        sys.stdout = open(os.devnull, "w")

    def __exit__(self, *a):
        sys.stdout.close()
        sys.stdout = self._so


# ------------------------------------------------------------------------------------- reference arm
_REF_JOB = None


def _ref_job(i):
    S, T_full, T_used, n_out = _REF_JOB
    return reference_kirchhoff_sample(S, T_full, T_used, n_out, 0)


def _ref_job_generic(i):
    wl, n = _REF_JOB
    return wl.cpu_sample(n)


def cpu_only_setup(wl):
    """Build the workload's synthetic input on the host (no CUDA) for the CPU arm of the non-Kirchhoff workloads."""
    from impdar_b200 import synthetic
    wl.tt, wl.dist, wl.trace_int = synthetic.geometry(wl.S, wl.T)
    S, T = wl.S, wl.T
    if S * T > (1 << 26):   # the CPU sample only touches a crop; keep generation bounded
        T = 4096
    x = synthetic.diffractor_radargram(S, T, seed=2, n_diffractors=64, device="cpu")
    wl.x = x
    if T != wl.T:
        wl.T_full, wl.T = wl.T, T
        wl.tt, wl.dist, wl.trace_int = synthetic.geometry(wl.S, wl.T)
    if isinstance(wl, PipelineC4):
        wl.x = x[None]
    if isinstance(wl, PhshC3):
        from impdar_b200 import migrationlib as ml
        wl.vel_table = synthetic.layered_velocity(wl.tt)
        d = type("D", (), {})()
        d.travel_time, d.snum, d.tnum, d.dist = wl.tt, wl.S, wl.T, wl.dist
        wl.vmig = ml.getVelocityProfile(d, wl.vel_table) if wl.layered else VEL_K


def usable_processes(bytes_per_process):
    cores = os.cpu_count() or 1
    try:
        import psutil
        avail = psutil.virtual_memory().available
        cores = max(1, min(cores, int(avail * 0.6 // max(bytes_per_process, 1))))
    except Exception:
        pass
    return cores


def run_reference(args, rank, world):
    """The reference's CPU implementation of the path on the host cores, no GPU involved.  Kirchhoff workloads: the
    UNMODIFIED reference's migrationKirchhoffLoop from baseline/_ref (`pip install --target` of an ImpDAR checkout by
    build(); the module is loaded standalone from there), one process per usable core because the loop is
    single-threaded numpy.
    Each step = every process computes `ref_n` output samples (the loop bounds tnum=1, snum=ref_n the reference itself
    accepts) against an (snum x ref_T_used) float64 input."""
    if rank != 0:
        return
    import torch
    torch.set_num_threads(1)
    import multiprocessing as mp
    global _REF_JOB
    wl = WORKLOADS[args.workload](args, 0, 1)
    if isinstance(wl, KirchhoffC2):
        S, T_full, T_used, n_out = wl.S, wl.T, wl.ref_T_used, wl.ref_n
        cores = usable_processes(S * T_used * 8 * 6)
        _REF_JOB = (S, T_full, T_used, n_out)
        reference_kirchhoff_input(S, T_used, 0)          # before the fork: the workers share it copy-on-write
        job, jobs = _ref_job, list(range(cores))
        from oracle import _refimport
        kind = "reference" if _refimport.vendored_available() else "port"
        sample = ("%s migrationKirchhoffLoop(tnum=1, snum=%d) against an %d x %d float64 input per process, %d processes; "
                  "cost per output sample is linear in tnum, rate scaled by %d/%d to the %d-trace radargram"
                  % ("baseline/_ref mig_python.py:35-60" if kind == "reference" else "oracle port of", n_out, S, T_used,
                     cores, T_used, T_full, T_full))
    else:
        cpu_only_setup(wl)
        cores = os.cpu_count() or 1
        n = max(1, wl.cpu_default_n // 4)
        _REF_JOB = (wl, n)
        job, jobs = _ref_job_generic, list(range(cores))
        kind = "port"
        sample = (wl.cpu_sample_desc % n) + "; %d concurrent samples (processes), one per core" % cores
    pool = mp.get_context("fork").Pool(cores)

    def one_step():
        t0 = time.perf_counter()
        res = pool.map(job, jobs)
        return time.perf_counter() - t0, float(sum(r[1] * (r[3] if isinstance(r[3], float) else 1.0) for r in res))

    for _ in range(min(args.warmup, 1)):
        one_step()
    tot_t, tot_u = 0.0, 0.0
    for _ in range(args.steps):
        t, u = one_step()
        tot_t += t
        tot_u += u
    pool.close()
    value = tot_u / tot_t
    line = {"impl": "reference", "metric": "migrated samples/s", "value": value, "unit": "samples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot_t / args.steps * 1e3,
            "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": wl.config(world=args.gpus),          # this arm runs on the other arm's config
            "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": kind, "sample": sample,
                             "host_cores_available": os.cpu_count()},
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------- main
class Ctx(object):
    pass


def measure(wl, ctx, steps, warmup, with_e2e=True, with_cpu=False, with_parity=True, n_e2e=None, dump_name=None):
    """Warm up, time `steps` steps with CUDA events (barrier + synchronize both sides, max over ranks), dump the last
    step's output as `dump_name` (--dump-outputs), then e2e, parity and the CPU baseline.  Returns the record (rank 0)
    or None."""
    import torch
    import torch.distributed as dist
    rank, world, lib = ctx.rank, ctx.world, ctx.lib

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    wl.setup()
    wl.steps_timed = steps
    need_flush = "flushed" in wl.l2_note()
    sampler = ClockSampler(ctx.local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(warmup):
        wl.step()
    barrier()
    launches0 = lib.impdar_b200_launch_count()
    evs = []
    lib.impdar_b200_kernel_timer(1)   # CUDA-event brackets around the dominant kernels, on their launch stream
    barrier()
    sampler.collect = True
    torch.cuda.profiler.start()   # ncu --profile-from-start off captures only the timed region
    for _ in range(steps):
        if need_flush:
            ctx.flush.fill_(1)
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        a.record()
        wl.step()
        b.record()
        evs.append((a, b))
    barrier()
    sampler.collect = False
    torch.cuda.profiler.stop()
    lib.impdar_b200_kernel_timer(0)   # stop recording; the records stay readable for roofline()
    launches = lib.impdar_b200_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if ctx.args.dump_outputs and rank == 0:
        np.save(os.path.join(ctx.args.dump_outputs, dump_name + ".npy"), output_sample(wl.output(), ctx.dump_budget))
    total_ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / steps
    value = wl.units * world / (ms_per_step * 1e-3)
    if world > 1 and wl.scaling == "strong":
        # every rank's own kernel time per step (load balance of the output-trace ranges), gathered for rank 0's line
        kt = kernel_times(list(KIRCH_KERNELS))
        mine = max([v[0] * v[1] for v in kt.values()] + [0.0]) / steps
        allk = torch.zeros(world, dtype=torch.float64, device="cuda")
        allk[rank] = mine
        dist.all_reduce(allk)
        wl.kernel_ms_by_rank = [round(float(v), 3) for v in allk.tolist()]
    roof = wl.roofline(ms_per_step, ctx.hbm_gbs, ctx.peak_src) if rank == 0 else None

    parity = None
    if with_parity:
        parity = wl.parity()          # of the output the last timed step left behind

    # ---- end to end through the plugin call with HOST buffers
    e2e = None
    if with_e2e and getattr(wl, "host", None) is not None:
        for _ in range(2):
            wl.e2e_step()
        barrier()
        n_e2e = n_e2e or max(2, min(steps, 5))
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            h2d, d2h, probe = wl.e2e_step()
        torch.cuda.synchronize()
        dt_e2e = (time.perf_counter() - t0) / n_e2e
        te = torch.tensor([dt_e2e], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_units = getattr(wl, "e2e_units", wl.units)
        e2e = {"value": e2e_units * world / float(te.item()), "unit": "samples/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": float(te.item()) * 1e3, "steps": n_e2e,
               "api": getattr(wl, "e2e_api", "impdar_b200.RadarData hot-path methods on host numpy data (pinned input)")}
    rec = None
    if rank == 0:
        rec = {"value": value, "unit": "samples/s", "ms_per_step": ms_per_step, "steps": steps, "warmup": warmup,
               "scaling": wl.scaling, "dtype": wl.dtype,
               "config": wl.config(), "exchange": wl.exchange_note(),
               "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e, "roofline": roof, "parity": parity}
        if with_cpu:
            n = ctx.args.cpu_samples or wl.cpu_default_n
            secs, units, kind, desc = wl.cpu_sample(n)
            rec["cpu_baseline"] = {"value": units / secs, "unit": "samples/s", "cores": 1, "kind": kind,
                                   "sample": desc + "; %.1f s" % secs, "host_cores_available": os.cpu_count()}
    wl.teardown()
    return rec


def sub_records(args, world):
    """[(records key, Workload class)] measured after the headline, each for args.steps timed steps."""
    if args.workload != "kirchhoff_c5" or args.no_records:
        return []
    subs = [("kirchhoff_4096x2048_per_gpu", KirchhoffC2)]
    if world == 1:
        subs.insert(0, ("stolt_65536x8192", StoltC5))
    return subs


def dump_budget(n_records):
    """Data bytes per --dump-outputs array when the line has `n_records` records (4 KiB of each share for the header)."""
    return DUMP_BYTES // n_records - 4096


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="kirchhoff_c5", choices=sorted(WORKLOADS),
                    help="headline workload (default: the north-star target, Kirchhoff 65536 x 8192)")
    ap.add_argument("--profiles", type=int, default=8, help="profiles per GPU per step (pipeline workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-records", action="store_true", help="headline only (no Stolt / config-2 sub-records)")
    ap.add_argument("--cpu-samples", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's output of every record as DIR/<name>.npy (see the module doc)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours (the reference arm times bounded samples, not whole outputs)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from impdar_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = Ctx()
    ctx.args, ctx.rank, ctx.local_rank, ctx.world = args, rank, local_rank, world
    ctx.lib = _lib.load()
    ctx.hbm_gbs, ctx.peak_src, _ = load_peaks()
    ctx.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    if os.environ.get("IMPDAR_KIRCH_MODE"):              # development A/B switch: 2 = table path (tile), 3 = gather kernel only
        from impdar_b200 import migrationlib as ml
        ml.set_kirchhoff_mode(int(os.environ["IMPDAR_KIRCH_MODE"]))

    subs = sub_records(args, world)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
    ctx.dump_budget = dump_budget(1 + len(subs))

    wl = WORKLOADS[args.workload](args, rank, world)
    head = measure(wl, ctx, args.steps, args.warmup, with_e2e=not args.no_e2e,
                   with_cpu=(world == 1 and not args.no_cpu_baseline), with_parity=not args.no_parity,
                   dump_name=args.workload)
    records = {}
    for key, cls in subs:
        sub = cls(args, rank, world)
        r = measure(sub, ctx, args.steps, 3, with_e2e=not args.no_e2e, with_cpu=False,
                    with_parity=not args.no_parity, dump_name=key)
        if rank == 0:
            records[key] = r

    if rank == 0:
        line = {"metric": "migrated samples/s", "value": head["value"], "unit": "samples/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
                "scaling": head["scaling"], "vs_baseline": None, "dtype": head["dtype"], "data": "synthetic",
                "config": head["config"], "exchange": head["exchange"], "clocks": head["clocks"],
                "gpu_launches": head["gpu_launches"],
                "e2e": head["e2e"], "roofline": head["roofline"], "parity": head["parity"], "peak_source": ctx.peak_src}
        if "cpu_baseline" in head:
            line["cpu_baseline"] = head["cpu_baseline"]
        if records:
            line["records"] = records
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
