#!/usr/bin/env python3
"""Times the matrix kernels over their tuning knobs on one GPU (CUDA events inside the library, vampomi_time_kernel)
and prints GB/s per variant. Usage: python tools/sweep.py [--N 20000 --M 106250 --reps 10] > gpurun_out/sweep.txt"""
import argparse
import itertools
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import vampomi_b200 as vb  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--N", type=int, default=20000)
ap.add_argument("--M", type=int, default=106250)
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--quick", action="store_true")
ap.add_argument("--storage", default="f64", choices=["f64", "f32"])
ap.add_argument("--multi", type=int, default=0, help="only the multi-vector kernels (one read of A for K vectors), with this many "
                "back-to-back reps per variant")
ap.add_argument("--sustained", type=int, default=0, help="also time a short list of variants with this many back-to-back reps "
                "(seconds-long, i.e. under the power cap) instead of a burst")
ap.add_argument("--gram", type=int, default=0, help="only the fused A^T q / A A^T q pass (kernels_gram.cu) over its cluster "
                "sizes and cluster counts, with this many back-to-back reps per variant")
a = ap.parse_args()

sh = vb.Shard(a.N, a.M, storage=a.storage)
sh.generate_iid(1)
sh.compute_stats()
rng = np.random.default_rng(0)
sh.Ax(rng.standard_normal(a.M))
sh.ATx(rng.standard_normal(a.N))
gb = a.N * a.M * (8 if a.storage == "f64" else 4) / 1e9
results = []


def t(which, label, reps=None, **knobs):
    for k, v in knobs.items():
        sh.set_tuning(k, v)
    sh.time_kernel(which, 2)
    ms = sh.time_kernel(which, reps or a.reps)
    rec = dict(kernel=label, ms=ms, gbs=gb / (ms * 1e-3), reps=reps or a.reps, **knobs)
    results.append(rec)
    print(json.dumps(rec), flush=True)


if a.gram:
    t(4, "read_probe", a.gram)
    t(5, "ax_multi_K2_default", a.gram)
    t(6, "atx_multi_K2_default", a.gram)
    t(9, "gram_K2", a.gram, gram_cluster=0, gram_clusters=0)
    t(10, "gram_K1", a.gram, gram_cluster=0, gram_clusters=0)
    if not a.quick:
        for ncl in (14, 15, 30, 45, 60):
            t(9, "gram_K2", a.gram, gram_cluster=0, gram_clusters=ncl)
        for cs in range(-(-a.N // 2560), 17):                  # every cluster size that holds a column (2 560 rows per CTA)
            t(9, "gram_K2", a.gram, gram_cluster=cs, gram_clusters=0)
    best = {}
    for r in results:
        if r["kernel"] not in best or r["gbs"] > best[r["kernel"]]["gbs"]:
            best[r["kernel"]] = r
    print("BEST", json.dumps(best))
    sys.exit(0)

if a.multi:
    t(4, "read_probe", a.multi)
    t(0, "ax_single_default", a.multi)
    t(1, "atx_single_default", a.multi)
    for gbal in (0, 1, 0, 1):                         # full-wave grid sizing on / off, twice (order effects)
        t(0, "ax_single_default", a.multi, grid_balance=gbal)
        t(5, "ax_multi_K2_default", a.multi, grid_balance=gbal)
        t(8, "ax_multi_K3_default", a.multi, grid_balance=gbal)
        t(6, "atx_multi_K2_default", a.multi, grid_balance=gbal)
    for occ in (3, 0, 3, 0):
        t(5, "ax_multi_K2_occ", a.multi, multi_ax_occ=occ)
        t(8, "ax_multi_K3_occ", a.multi, multi_ax_occ=occ)
    if a.quick:
        sys.exit(0)
    for rv, u in ((1, 4), (1, 8), (2, 2), (2, 4), (1, 2)):
        t(5, "ax_multi_K2", a.multi, multi_ax_rv=rv, multi_ax_unroll=u)
        t(8, "ax_multi_K3", a.multi, multi_ax_rv=rv, multi_ax_unroll=u)
    for o in (1, 2, 3, 4):
        t(5, "ax_multi_K2", a.multi, multi_ax_rv=1, multi_ax_unroll=4, ax_ctas_per_sm=o)
    sh.set_tuning("ax_ctas_per_sm", 0); sh.set_tuning("multi_ax_rv", 0); sh.set_tuning("multi_ax_unroll", 0)
    t(6, "atx_multi_K2_regtile", a.multi, multi_atx_impl=0)
    t(7, "atx_multi_K1_regtile", a.multi, multi_atx_impl=0)
    for tile in (4096, 2048):
        for c_, u in ((2, 2), (2, 4), (1, 2), (1, 4), (4, 2)):
            if tile != 4096 and (c_, u) not in ((2, 4),):
                continue
            t(6, "atx_multi_K2_smem", a.multi, multi_atx_impl=1, multi_atx_cols=c_, multi_atx_unroll=u, multi_atx_tile=tile)
            t(7, "atx_multi_K1_smem", a.multi, multi_atx_impl=1, multi_atx_cols=c_, multi_atx_unroll=u, multi_atx_tile=tile)
    for o in (1, 2, 3, 4):
        t(6, "atx_multi_K2_smem", a.multi, multi_atx_impl=1, multi_atx_cols=2, multi_atx_unroll=2, multi_atx_tile=4096, atx_ctas_per_sm=o)
    best = {}
    for r in results:
        if r["kernel"] not in best or r["gbs"] > best[r["kernel"]]["gbs"]:
            best[r["kernel"]] = r
    print("BEST", json.dumps(best))
    sys.exit(0)

if a.sustained:
    base = dict(ax_impl=0, atx_impl=0, center_split=0, ax_ctas_per_sm=0, atx_ctas_per_sm=0)
    t(4, "read_probe_sustained", a.sustained)
    t(0, "ax_default", a.sustained)
    t(1, "atx_default", a.sustained)
    for il in (1, 0, 1, 0):
        t(0, "ax_default_interleave", a.sustained, interleave=il)
        t(1, "atx_default_interleave", a.sustained, interleave=il)
    for split in (0,):
        for rv, u in ((2, 4), (4, 2)):
            t(0, "ax_sustained", a.sustained, **dict(base, ax_rv=rv, ax_unroll=u, center_split=split))
        for c_, u in ((2, 4), (1, 2)):
            t(1, "atx_sustained", a.sustained, **dict(base, atx_cols=c_, atx_unroll=u, center_split=split))
    for c_, u in ((1, 2), (1, 4), (1, 8), (2, 2), (2, 4), (2, 8), (4, 2), (4, 4)):
        for o in (0, 4, 8):
            t(1, "atx_cta_sustained", a.sustained, **dict(base, atx_impl=2, atx_cols=c_, atx_unroll=u, atx_ctas_per_sm=o))
    t(0, "ax_sustained", a.sustained, **dict(base, ax_impl=1))
    t(1, "atx_sustained", a.sustained, **dict(base, atx_impl=1))
    t(3, "loo_sustained", a.sustained)
    for k, v in base.items():
        sh.set_tuning(k, v)
    sh.set_tuning("ax_rv", 0); sh.set_tuning("ax_unroll", 0); sh.set_tuning("atx_cols", 0); sh.set_tuning("atx_unroll", 0)
    sh.set_tuning("atx_impl", 3)
    if a.quick:
        sys.exit(0)

ax_variants = [(1, 2), (1, 4), (1, 8), (2, 2), (2, 4), (2, 8), (4, 2), (4, 4)]
atx_variants = [(1, 2), (1, 4), (1, 8), (2, 2), (2, 4), (2, 8), (4, 2), (4, 4)]
occ = [0] if a.quick else [0, 1, 2, 3, 4, 6, 8]
for (rv, u), o in itertools.product(ax_variants, occ):
    t(0, "ax", ax_rv=rv, ax_unroll=u, ax_ctas_per_sm=o)
for (c, u), o in itertools.product(atx_variants, occ):
    t(1, "atx", atx_impl=0, atx_cols=c, atx_unroll=u, atx_ctas_per_sm=o)
for o in ([0] if a.quick else [0, 1, 2, 3]):
    t(0, "ax", ax_impl=1, ax_ctas_per_sm=o)
    t(1, "atx", atx_impl=1, atx_ctas_per_sm=o)
sh.set_tuning("ax_impl", 0)
sh.set_tuning("atx_impl", 0)
t(4, "read_probe")
t(4, "read_probe_sustained", 200)
t(2, "stats")
t(3, "loo")
best = {k: max((r for r in results if r["kernel"] == k), key=lambda r: r["gbs"]) for k in ("ax", "atx")}
print("BEST", json.dumps(best))
