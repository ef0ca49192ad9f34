#!/usr/bin/env python3
"""Matrix kernels under the SUSTAINED power cap (the state the bench's timed region runs in), with the SM clock sampled next to
every figure: python tools/gram_sustain.py [--reps 400] [--rounds 2] name=which[:knob=v,...] ...
`which` is vampomi_time_kernel's selector (4 read probe, 8 k_ax_multi<3>, 9 / 10 the fused pass for two / one system).
A burst of `reps` launches (~1 s on a 17 GB shard) follows a heat-up burst; clocks are nvidia-smi samples taken during the burst."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vampomi_b200 as vb  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--N", type=int, default=20000)
ap.add_argument("--M", type=int, default=106250)
ap.add_argument("--reps", type=int, default=400)
ap.add_argument("--rounds", type=int, default=2)
ap.add_argument("configs", nargs="+")
a = ap.parse_args()


class Clocks(threading.Thread):
    def __init__(self):
        super().__init__(daemon=True)
        self.samples, self.power, self.on = [], [], True

    def run(self):
        while self.on:
            try:
                out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=clocks.sm,power.draw", "--format=csv,noheader,nounits"],
                                     stdout=subprocess.PIPE, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.power.append(float(out[1]))
            except Exception:
                pass
            time.sleep(0.05)


sh = vb.Shard(a.N, a.M)
sh.generate_iid(1)
sh.compute_stats()
defaults = {"gram_clusters": 0, "gram_cluster": 0}
sh.time_kernel(9, a.reps)                                      # heat-up
for rnd in range(a.rounds):
    for c in a.configs:
        name, _, rest = c.partition("=")
        which, _, kn = rest.partition(":")
        knobs = dict(defaults)
        for kv in filter(None, kn.split(",")):
            k, v = kv.split("=")
            knobs[k] = int(v)
        for k, v in knobs.items():
            sh.set_tuning(k, v)
        sh.time_kernel(int(which), 2)
        ck = Clocks()
        ck.start()
        ms = sh.time_kernel(int(which), a.reps)
        ck.on = False
        ck.join()
        print(json.dumps({"config": name, "which": int(which), "knobs": {k: v for k, v in knobs.items() if defaults[k] != v}, "round": rnd,
                          "ms": round(ms, 4), "gbs": round(a.N * a.M * 8 / ms / 1e6),
                          "sm_mhz_median": statistics.median(ck.samples) if ck.samples else None,
                          "power_w_median": statistics.median(ck.power) if ck.power else None, "clock_samples": len(ck.samples)}), flush=True)
