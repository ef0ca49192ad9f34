#!/usr/bin/env python3
"""SASS mnemonic counts (cuobjdump -sass, sm_100a) of the default kernels of an iteration, no GPU needed:
python tools/sass_summary.py > profiles/r02_sass_default_kernels.txt"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WANT = [("kernels_gram.o", r"k_gram_wsxILi2ELi8EE"), ("kernels_gram.o", r"k_gram_wsxILi1ELi8EE"),
        ("kernels_multi.o", r"k_ax_multiIdLi3ELi1ELi4ELi0E"), ("kernels_multi.o", r"k_ax_reduce_multiILi8E")]
KEEP = re.compile(r"^(DFMA|DADD|DMUL|LDG|STG|LDS|STS|LDL|STL|SHFL|UBLKCP|UTMALDG|USETMAXREG|SYNCS|BAR|UCGABAR|CCTL|MEMBAR|ATOM|RED|ST\.|STAS|MAPA|UMOV|ERRBAR|FENCE)")
print("# SASS mnemonic counts of the default kernels of an iteration (cuobjdump -sass of vampomi_b200/build/*.o, sm_100a).\n"
      "# k_gram_wsx: UTMALDG.3D = cp.async.bulk.tensor.3d (one per ring stage), USETMAXREG = setmaxnreg, SYNCS.* = mbarrier arrive / expect_tx / try_wait,\n# STAS = st.async into a peer\n"
      "# CTA's shared memory (distributed shared memory), no LDL/STL (no local-memory traffic), LDS.128 conflict-free row pairs.\n")
for obj, pat in WANT:
    out = subprocess.run(["cuobjdump", "-sass", os.path.join(ROOT, "vampomi_b200", "build", obj)], stdout=subprocess.PIPE, text=True).stdout
    cur, counts = None, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            if cur and counts is not None:
                break
            cur = m.group(1) if re.search(pat, m.group(1)) else None
            counts = collections.Counter() if cur else None
            continue
        if cur:
            m = re.search(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
            if m and KEEP.match(m.group(1)):
                counts[m.group(1)] += 1
    if counts:
        print(f"== {cur}")
        for k, v in counts.most_common():
            print(f"{v:7d} {k}")
        print()
ptx = subprocess.run(["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
                      os.path.join(ROOT, "vampomi_b200", "csrc", "kernels_gram.cu"), "-o", "/dev/null"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout
lines = ptx.splitlines()
for i, l in enumerate(lines):
    if "k_gram_wsxILi2ELi8EE" in l or "k_gram_wsxILi1ELi8EE" in l:
        print("ptxas -v:", l.split("function")[-1].strip())
        print("         ", lines[i + 1].strip().replace("ptxas info    : ", ""), "|", lines[i + 2].strip().replace("ptxas info    : ", ""))
