#!/usr/bin/env python3
"""Writes tests/golden/midsize_gam1e-2.npz, the outputs tests/test_gpu_vamp.py::test_mid_size_run_matches_the_reference_binary_on_this_box
holds bin/main_meth to: N = 4 000, Mt = 20 000 (0.64 GB), --gam1 1e-2, 4 iterations, probe seed 11.

Source: the patched reference binary (oracle/_ref/main_meth_ref) where it has been built, otherwise the numpy oracle
(oracle/vamp_oracle.py), the restatement of the reference that tests/test_oracle_vs_golden.py holds to the reference's own
outputs at 1e-9. The fixture records which of the two made it (`source`). Stored: x1_hat and r1 of every iteration at a
seeded sample of markers together with their full-vector norms, the three CSV files as bytes, the (k1, k2) CG counts, and
the parameters and SHA-256 the inputs are rebuilt and checked from. Usage: python tests/tools/make_midsize_golden.py [--oracle]
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from make_golden import cg_counts, run_ref  # noqa: E402
from oracle import build_ref  # noqa: E402
from oracle import vamp_oracle as vo  # noqa: E402
from vampomi_b200 import sim  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "midsize_gam1e-2.npz")
CASE = dict(N=4000, M=20000, lam=0.01, h2=0.5, data_seed=77, probe_seed=11, iterations=4, gam1="1e-2")
SAMPLE = 2048          # markers kept per vector: the whole fixture stays near 150 KB
SAMPLE_SEED = 4000


def main():
    c = CASE
    use_ref = os.path.isfile(build_ref.OUT_BIN) and "--oracle" not in sys.argv
    with tempfile.TemporaryDirectory() as d:
        X, y, beta = sim.write_dataset(d, "mid", c["N"], c["M"], lam=c["lam"], h2=c["h2"], seed=c["data_seed"])
        os.makedirs(os.path.join(d, "out"))
        if use_ref:
            log = run_ref(["--meth-file", f"{d}/mid.bin", "--phen-file", f"{d}/mid.phen", "--N", str(c["N"]), "--Mt", str(c["M"]),
                           "--out-dir", f"{d}/out", "--out-name", "m", "--iterations", str(c["iterations"]), "--true-signal-file",
                           f"{d}/mid_ts.bin", "--stop-criteria-thr", "0", "--gam1", c["gam1"], "--verbosity", "1"],
                          c["probe_seed"], threads=os.cpu_count() or 1)
            cg = cg_counts(log)
            source = "reference binary (oracle/_ref/main_meth_ref)"
        else:
            y_txt = np.array([float("%0.10f" % v) for v in y])                       # the .phen text the reference reads
            y_std = y_txt * np.sqrt((c["N"] - 1) / float(((y_txt - y_txt.sum() / c["N"]) ** 2).sum()))   # data::read_phen
            v = vo.Vamp(vo.Data(X, y_std), gam1=float(c["gam1"]), gamw=1.0 / (1.0 - c["h2"]), max_iter=c["iterations"],
                        true_signal=beta, out_dir=f"{d}/out", out_name="m", seed=c["probe_seed"], stop_criteria_thr=0.0)
            v.infere()
            cg = np.array([[[k for (it, kind, k) in v.cg_iters if it == i and kind == want][0] for want in ("lmmse", "onsager")]
                           for i in range(1, c["iterations"] + 1)], dtype=np.int64)
            source = "numpy oracle (oracle/vamp_oracle.py; the reference binary was not available)"
        idx = np.sort(np.random.default_rng(SAMPLE_SEED).choice(c["M"], SAMPLE, replace=False))
        x1 = [np.fromfile(f"{d}/out/m_it_{k}.bin") for k in range(1, c["iterations"] + 1)]
        r1 = [np.fromfile(f"{d}/out/m_r1_it_{k}.bin") for k in range(1, c["iterations"] + 1)]
        csv = {k: np.frombuffer(open(f"{d}/out/m_{k}.csv", "rb").read(), dtype=np.uint8) for k in ("params", "metrics", "prior")}
        np.savez_compressed(OUT, source=source, sha256_A=hashlib.sha256(X.tobytes()).hexdigest(), sample_index=idx,
                            x1=np.array([a[idx] for a in x1]), r1=np.array([a[idx] for a in r1]),
                            x1_norm=np.array([np.linalg.norm(a) for a in x1]), r1_norm=np.array([np.linalg.norm(a) for a in r1]),
                            cg_iters=cg, **{f"csv_{k}": b for k, b in csv.items()}, **{k: str(v_) if k == "gam1" else v_ for k, v_ in c.items()})
    print(OUT, source, "CG", cg.tolist(), f"{os.path.getsize(OUT)} bytes")


if __name__ == "__main__":
    main()
