#!/usr/bin/env python3
"""Time of the opt-in NaN imputation (vampomi_impute_missing: k_impute_missing plus the read-back of its counts) on the
headline block, next to k_stats on the same block:

    python tools/impute_time.py [--N 20000] [--Mt 850000] [--rounds 3] [--out FILE]

One GPU holds the whole block (N x Mt FP64, 136 GB at the defaults), generated with generate_iid. Then, per round, every
100th column (1 % of them) is uploaded again from the host with 5 % seeded NaNs, and three things are timed:
  impute_ms         a host clock around the synchronous call that replaces those NaNs (one read of the block, plus the
                    reread and writes of the 1 % of columns that hold a NaN)
  impute_clean_ms   a second call, which finds nothing to replace (the read of the block alone)
  stats_ms          vampomi_time_kernel(which=2): k_stats on the same block, CUDA events, average of --reps launches
The read probe (which=4: one plain streaming read of the block) is recorded as the live ceiling. The block is far larger than
the L2, so every pass reads HBM. The card's name and power limit come from a read-only nvidia-smi query."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vampomi_b200 as vb  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--N", type=int, default=20000)
ap.add_argument("--Mt", type=int, default=850000)
ap.add_argument("--every", type=int, default=100, help="columns re-uploaded with NaNs: every this many-th one")
ap.add_argument("--nan-frac", type=float, default=0.05)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--seed", type=int, default=7)
ap.add_argument("--out", default=None, help="also write the JSON record here")
a = ap.parse_args()


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True,
                         timeout=60, check=True).stdout.strip()
    return dict(zip(("gpu", "power_limit", "sm_clock_max"), (s.strip() for s in out.split(","))))


info = gpu_info()
# the first launch of a kernel loads it: warm both up on a small block first
with vb.Shard(256, 64) as w:
    X = np.random.default_rng(0).standard_normal((64, 256))
    X[:, 3] = np.nan
    w.upload(X)
    w.impute_missing()
    w.compute_stats()

cols = np.arange(0, a.Mt, a.every)
rng = np.random.default_rng(a.seed)
H = rng.standard_normal((cols.size, a.N))
H[rng.random(H.shape) < a.nan_frac] = np.nan
n_nan = int(np.isnan(H).sum())

sh = vb.Shard(a.N, a.Mt)
sh.generate_iid(1)
block_bytes = a.N * a.Mt * 8
rounds = []
for r in range(a.rounds):
    for k, j in enumerate(cols):
        sh.upload(H[k:k + 1], j0=int(j))
    t0 = time.perf_counter()
    counts = sh.impute_missing()
    t1 = time.perf_counter()
    clean = sh.impute_missing()
    t2 = time.perf_counter()
    assert counts == (n_nan, int(np.isnan(H).any(axis=1).sum()), int(np.isnan(H).all(axis=1).sum())), counts
    assert clean == (0, 0, 0), clean
    rounds.append(dict(impute_ms=(t1 - t0) * 1e3, impute_clean_ms=(t2 - t1) * 1e3, counts=list(counts)))
    print(json.dumps(dict(round=r, **rounds[-1])), flush=True)

sh.time_kernel(2, 2)
stats_ms = sh.time_kernel(2, a.reps)
sh.time_kernel(4, 2)
read_ms = sh.time_kernel(4, a.reps)
sh.close()

med = lambda k: statistics.median(x[k] for x in rounds)
rec = dict(
    what="vampomi_impute_missing on one GPU holding the whole block, next to k_stats and the read probe on the same block",
    **info, N=a.N, Mt=a.Mt, block_gb=block_bytes / 1e9, columns_with_nan=int(cols.size), nan_entries=n_nan, nan_frac=a.nan_frac,
    rounds=rounds, impute_ms_median=med("impute_ms"), impute_clean_ms_median=med("impute_clean_ms"), stats_ms=stats_ms,
    read_probe_ms=read_ms, impute_over_stats=med("impute_ms") / stats_ms, impute_over_read_probe=med("impute_ms") / read_ms,
    impute_gbs=block_bytes / (med("impute_ms") * 1e6), stats_gbs=block_bytes / (stats_ms * 1e6), read_probe_gbs=block_bytes / (read_ms * 1e6),
    timing="impute: host clock around the synchronous call (launch, kernel, count read-back); stats / read probe: CUDA events, "
           f"average of {a.reps} back-to-back launches; block >> L2, so each pass reads HBM")
print(json.dumps(rec), flush=True)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")
