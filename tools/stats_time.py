#!/usr/bin/env python3
"""Time of k_stats (the marker statistics, vampomi_time_kernel which=2: CUDA events, average of --reps launches) on a generated
block, one JSON line per run:

    python tools/stats_time.py [--N 20000] [--M 106250] [--reps 20] [--tag NAME]

The library is the one vampomi_b200 loads (VAMPOMI_LIB selects another build), so two builds are compared by running this
alternately with each. The default block is 17 GB of FP64, far larger than the L2, so every launch reads HBM. The card's name and
power limit come from a read-only nvidia-smi query."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vampomi_b200 as vb  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--N", type=int, default=20000)
ap.add_argument("--M", type=int, default=106250)
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--tag", default="")
a = ap.parse_args()

q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                   text=True, timeout=60, check=True).stdout.strip().split(",")
with vb.Shard(a.N, a.M) as sh:
    sh.generate_iid(11)
    sh.time_kernel(2, 3)                                  # first launches load the kernel
    ms = [sh.time_kernel(2, a.reps) for _ in range(3)]
print(json.dumps(dict(tag=a.tag, lib=os.environ.get("VAMPOMI_LIB", "default"), N=a.N, M=a.M, reps=a.reps, stats_ms=ms,
                      gb_per_s=[a.N * a.M * 8 / (m * 1e-3) / 1e9 for m in ms], gpu=q[0].strip(), power_limit=q[1].strip())))
