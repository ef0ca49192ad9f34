#!/usr/bin/env python3
"""Ingest path (SURVEY.md §8 row a1): writes a marker-major FP64 file and times vampomi_load_file (pread -> pinned ring ->
HBM) for several reader-thread counts. Usage: python tools/load_bench.py [--N 20000 --M 50000]"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vampomi_b200 as vb  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--N", type=int, default=20000)
ap.add_argument("--M", type=int, default=50000)
ap.add_argument("--big", action="store_true", help="few variants only (for a file of tens of GB): page cache, then O_DIRECT reads that bypass it")
a = ap.parse_args()
d = tempfile.mkdtemp(prefix="vampomi_load_", dir="/tmp")
path = os.path.join(d, "m.bin")
sh = vb.Shard(a.N, a.M)
sh.generate_iid(1)
with open(path, "wb") as f:
    step = max(1, (256 << 20) // (a.N * 8))
    for j0 in range(0, a.M, step):
        sh.download(j0, min(step, a.M - j0)).tofile(f)
gb = a.N * a.M * 8 / 1e9
ref = sh.download(0, 64)
res = []
sh.set_tuning("load_threads", 16)
sh.load_file(path)                      # allocates the context's pinned ring once (16 threads x 3 slots): not part of any timing below
last = sh.download(a.M - 64, 64)

if a.big:
    for label, direct, threads in (("page cache", 0, 8), ("page cache", 0, 16), ("O_DIRECT", 1, 4)):
        sh.set_tuning("load_threads", threads); sh.set_tuning("load_depth", 3); sh.set_tuning("load_direct", direct)
        sh.fill(0, 0.0)
        t = time.time()
        sh.load_file(path)
        dt = time.time() - t
        assert np.array_equal(sh.download(0, 64), ref) and np.array_equal(sh.download(a.M - 64, 64), last)
        res.append(dict(source=label, direct=direct, threads=threads, s=round(dt, 3), gbs=round(gb / dt, 2)))
    print(json.dumps(dict(file_gb=gb, results=res)))
    os.unlink(path)
    os.rmdir(d)
    sys.exit(0)
for direct in (0, 1):
    for threads in (1, 2, 4, 8, 16):
        for depth in ((3,) if direct == 0 else (3, 6)):
            sh.set_tuning("load_threads", threads)
            sh.set_tuning("load_depth", depth)
            sh.set_tuning("load_direct", direct)
            sh.fill(0, 0.0)
            t = time.time()
            sh.load_file(path)
            dt = time.time() - t
            assert np.array_equal(sh.download(0, 64), ref) and np.array_equal(sh.download(a.M - 64, 64), last)
            res.append(dict(direct=direct, threads=threads, depth=depth, s=round(dt, 3), gbs=round(gb / dt, 2)))
print(json.dumps(dict(file_gb=gb, note="file just written: buffered reads (direct=0) come from the page cache; direct=1 is O_DIRECT (falls back to "
                      "buffered reads on file systems without it)", results=res)))
os.unlink(path)
os.rmdir(d)
