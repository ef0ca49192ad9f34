#!/usr/bin/env python3
"""A/B timing of the fused pass under the same thermal state: python tools/gram_ab.py [--K 2] [--reps 20] [--rounds 3] name[:knob=v[,knob=v]] ...
Every round times every configuration once (bursts of `reps` launches after 2 warm-up launches), so slow drifts of the SM clock
hit all configurations alike."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vampomi_b200 as vb  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--N", type=int, default=20000)
ap.add_argument("--M", type=int, default=106250)
ap.add_argument("--K", type=int, default=2)
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("configs", nargs="+")
a = ap.parse_args()
sh = vb.Shard(a.N, a.M)
sh.generate_iid(1)
sh.compute_stats()
which = 9 if a.K == 2 else 10
defaults = {"gram_clusters": 0, "gram_cluster": 0}
res = {c: [] for c in a.configs}
for _ in range(a.rounds):
    for c in a.configs:
        _, _, rest = c.partition(":")
        knobs = dict(defaults)
        for kv in filter(None, rest.split(",")):
            k, v = kv.split("=")
            knobs[k] = int(v)
        for k, v in knobs.items():
            sh.set_tuning(k, v)
        sh.time_kernel(which, 2)
        res[c].append(round(sh.time_kernel(which, a.reps), 4))
for c, v in res.items():
    print(json.dumps({"config": c, "K": a.K, "ms": v, "best_gbs": round(a.N * a.M * 8 / min(v) / 1e6)}), flush=True)
