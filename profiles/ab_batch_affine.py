"""A/B of the batched-affine rounds (msm_pair.cuh) on one registered 2^20 MSM per group (BN254; uniform scalars).

Settings, alternated within every repetition so that clock and neighbour drift hits all of them alike:
  xyzz      sb_set_tuning(4, 1): plain segmented XYZZ accumulation
  default   sb_set_tuning(4, 0): what the library selects (rounds for G2)
  R=k       sb_set_tuning(4, 2) + (5, k): rounds forced, at most k of them
Times are the library's CUDA events around the device part of the call (sort + accumulation + fold + reduction) and
around the accumulation (rounds + XYZZ accumulation); one JSON line per (group, setting) with the median and the spread.
Every setting must return the same bytes.

  python profiles/ab_batch_affine.py [--reps 7] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import snarkjs_b200  # noqa: E402
from snarkjs_b200 import synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=7)
ap.add_argument("--log2n", type=int, default=20)
ap.add_argument("--rounds", default="1,2,3,4,5")
ap.add_argument("--out", default=None)
args = ap.parse_args()

c = snarkjs_b200.getCurveFromName("bn128")
lib, h = c.lib, c.handle
n = 1 << args.log2n
rng = np.random.default_rng(1)
sc = rng.integers(0, 256, size=n * 32, dtype=np.uint8)
sc.reshape(n, 32)[:, 31] &= 0x1f
settings = [("xyzz", 1, 0), ("default", 0, 0)] + [(f"R={k}", 2, int(k)) for k in args.rounds.split(",")]
try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
except OSError:
    gpu = "unknown"
lines = []
for grp in (1, 2):
    G = c.G1 if grp == 1 else c.G2
    hb = G.registerBases(synth.gen_points(c, grp, 7, n))
    dev = {s[0]: [] for s in settings}; acc = {s[0]: [] for s in settings}
    ref = None
    for rep in range(args.reps + 1):                      # repetition 0 warms every setting up
        for name, mode, cap in settings:
            lib.sb_set_tuning(4, mode); lib.sb_set_tuning(5, cap)
            out = G.multiExpRegistered(hb, sc).tobytes()
            if ref is None:
                ref = out
            assert out == ref, f"G{grp} {name}: result differs"
            if rep:
                dev[name].append(c.last_ms(2)); acc[name].append(lib.sb_last_stat(h, grp - 1))
    lib.sb_set_tuning(4, 0); lib.sb_set_tuning(5, 0)
    for name, _, _ in settings:
        d, a = np.array(dev[name]), np.array(acc[name])
        rec = {"group": f"G{grp}", "setting": name, "n": n, "reps": args.reps, "gpu": gpu,
               "msm_device_ms": float(np.median(d)), "msm_device_ms_min": float(d.min()), "msm_device_ms_max": float(d.max()),
               "accumulate_ms": float(np.median(a)), "accumulate_ms_min": float(a.min()), "accumulate_ms_max": float(a.max())}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
if args.out:
    with open(args.out, "w") as f:
        f.write("".join(json.dumps(r) + "\n" for r in lines))
c.terminate()
