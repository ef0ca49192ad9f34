#!/usr/bin/env python3
"""Runs the fused A^T q / A A^T q pass a few times on one shard (for ncu captures): python tools/gram_one.py [K] [N] [M] [knob=v ...]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vampomi_b200 as vb  # noqa: E402

K = int(sys.argv[1]) if len(sys.argv) > 1 else 2
N = int(sys.argv[2]) if len(sys.argv) > 2 else 20000
M = int(sys.argv[3]) if len(sys.argv) > 3 else 106250
sh = vb.Shard(N, M)
sh.generate_iid(1)
sh.compute_stats()
for kv in sys.argv[4:]:
    k, v = kv.split("=")
    sh.set_tuning(k, int(v))
ms = sh.time_kernel(9 if K == 2 else 10, 3)
print(f"K {K} {' '.join(sys.argv[4:])}: {ms:.3f} ms, {N * M * 8 / ms / 1e6:.0f} GB/s")
