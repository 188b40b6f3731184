"""Summaries for A/B bench runs (scripts/gpu_kirchhoff_layered.sh ab).

    python scripts/ab_line.py BENCH_JSON LABEL RUN         one line per bench.py result
    python scripts/ab_line.py --compare DUMP_A DUMP_B      bench.py --dump-outputs directories, file by file, bit for bit
"""
import glob
import json
import os
import sys

import numpy as np


def line(path, label, run):
    d = json.loads(open(path).read())
    r, rec = d["roofline"], d["records"]
    return ("%-4s run %s  ms/step %.2f  kernel %s %.2f ms  stolt %.3f ms  config2 %.4f ms  parity %.2e  sm_mhz %s"
            % (label, run, d["ms_per_step"], r["kernel"], r["kernel_ms"], rec["stolt_65536x8192"]["ms_per_step"],
               rec["kirchhoff_4096x2048_per_gpu"]["ms_per_step"], d["parity"]["rel_l2"], d["clocks"]["sm_mhz"]))


def compare(a_dir, b_dir):
    files = sorted(glob.glob(os.path.join(a_dir, "*.npy")))
    if not files:
        return ["no dumped outputs in %s" % a_dir]
    out = []
    for f in files:
        g = os.path.join(b_dir, os.path.basename(f))
        a = np.load(f)
        b = np.load(g) if os.path.exists(g) else None
        same = b is not None and a.shape == b.shape and np.array_equal(a, b, equal_nan=True)
        out.append("bitwise %-36s %-14s %s" % (os.path.basename(f), a.shape, "EQUAL" if same else "DIFFERENT"))
    return out


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        print("\n".join(compare(sys.argv[2], sys.argv[3])))
    else:
        print(line(*sys.argv[1:4]))
