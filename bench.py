#!/usr/bin/env python3
"""Benchmark of the VAMP inference hot path (BASELINE.json: VAMP iterations/s at N=20k, M=850k FP64 on 1/2/4/8 B200).

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU; torchrun for N > 1)
  python bench.py --impl reference ...                     the reference's own CPU implementation (oracle/_ref) beside it
  python bench.py ... --dump-outputs DIR                   also writes what the last timed step returned, as DIR/<name>.npy

A "step" is ONE full VAMP iteration (Gaussian-mixture denoiser + EM prior update + LMMSE conjugate-gradient solve +
Onsager solve + noise-precision update + metrics) on the synthetic i.i.d. design of the headline configuration, markers
sharded over the N GPUs (total problem fixed: strong scaling). Two timed legs over the SAME iterations (W+1 .. W+K of
two identically initialised solvers):
  value  device-resident: matrix, phenotype and all vectors already in HBM; only the ~20 CSV scalars leave the device
  e2e    the same iterations through the host-buffer C ABI a main_meth run uses: every step re-uploads the phenotype
         (H2D) and brings x1_hat/sqrt(N) and r1/sqrt(N) — the content of _it_k.bin / _r1_it_k.bin — back to host memory
Timing: CUDA events on the library's own stream, barrier + synchronize on both sides, max over ranks.

Before the timed legs every run replays two committed reference-binary fixtures (tests/golden: linear_wellcond, probit_small)
on the job's OWN ranks and communicator and reports `parity` (relative L2 of x1_hat / r1 per iteration over all shards, CSV
values, CG iteration counts) — the 1-, 2-, 4- and 8-GPU lines each carry their own parity evidence.

CPU baseline (`cpu_baseline`, and the whole `--impl reference` arm): the reference binary (oracle/_ref) is timed on a sample
with the headline's COLUMN LENGTH (N = 20 000 x 8 500 markers = 1.36 GB per pass, streamed from DRAM) over the same
warm-up / steps window; what is measured is its effective GB/s per matrix pass with its own CG counts, and the it/s at the
headline size follows from the passes the reference makes there, 2(k1+k2)+8 per iteration with the (k1,k2) the GPU arm measured on
those very iterations (equal by parity; the reference arm alone reads them from profiles/headline_cg_counts.json).
With --cpu-c2 (default in the in-line leg) BASELINE config 2 (N = 10 000, M = 100 000, 8 GB) is additionally run IN FULL by both
command lines on the same files: a measured, not derived, ratio.
"""
import argparse
import json
import math
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (it may be read-only)
sys.path.insert(0, ROOT)

METRIC = "vamp_iterations_per_s"
UNIT = "it/s"
H2 = 0.5            # CLI default --h2 (src/options.hpp:98) -> gamw = 2
LAM = 0.01          # sparsity of the simulated effects (SURVEY.md §8d, C3)
DATA_SEED = 2026
PROBE_SEED = 17


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--N", type=int, default=20000)
    ap.add_argument("--Mt", type=int, default=850000)
    ap.add_argument("--cpu-sample-M", type=int, default=8500, help="markers of the bounded CPU-baseline sample (N stays the headline's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cpu-c2", action="store_true", help="skip the full run of BASELINE config 2 (8 GB) by both command lines")
    ap.add_argument("--no-parity", action="store_true", help="skip the fixture replay on the job's ranks")
    ap.add_argument("--record-cg-counts", type=int, default=0, metavar="ITERATIONS",
                    help="run this many iterations of the workload, write their CG iteration counts to profiles/headline_cg_counts.json "
                         "(what the reference arm uses to turn its GB/s per pass into it/s at the headline size) and exit")
    ap.add_argument("--schedule", default="onepass", choices=["onepass", "recycled", "fused", "plain"],
                    help="onepass (default): recycled + CG iterations that read the block once (fused A^T q / A A^T q pass); recycled: lock-step LMMSE + Onsager solves sharing every read of the block, products of their "
                         "solutions kept by the solves themselves; fused: the same without that recycling (every product computed "
                         "by a pass, sharing reads); plain: one product per pass in the reference's order")
    ap.add_argument("--tune", action="append", default=[], metavar="KNOB=VALUE", help="vampomi_set_tuning knob for experiments (repeatable)")
    ap.add_argument("--no-ab", action="store_true", help="skip the short device-resident legs of the other schedules")
    ap.add_argument("--storage", default="f64", choices=["f64", "f32"],
                    help="f32 = opt-in mode that holds the matrix rounded to FP32 in HBM (arithmetic FP64); NOT the headline configuration")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed legs, write what their last step returned as DIR/<name>.npy "
                                                          "(float64), so that two builds can be compared output for output")
    return ap.parse_args()


def workload_name(N, Mt):
    return (f"linear VAMP inference, synthetic i.i.d. FP64 design N={N} Mt={Mt} ({N * Mt * 8 / 1e9:.0f} GB), CLI defaults "
            f"(10 mixture components, rho 0.5, gam1 1e-6, CG tol 1e-5, EM 1 it), lam={LAM}, h2={H2}")


def ncu_traffic(kernel, N, M_local, bytes_per_launch):
    """roofline.traffic: DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/ncu_traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            rec = json.load(f)[kernel]
        if isinstance(rec, list):        # several captured launch shapes: the matching one, else the first for scaling
            rec = next((r for r in rec if r["N"] == N and r["M_local"] == M_local), rec[0])
    except Exception:
        return None, None
    if rec["N"] == N and rec["M_local"] == M_local:
        return float(rec["dram_bytes"]), f"ncu capture of this launch shape ({rec['source']})"
    ratio = rec["dram_bytes"] / rec["algorithmic_bytes"]
    return bytes_per_launch * ratio, (f"scaled from the ncu capture at M_local={rec['M_local']} (traffic/algorithmic = {ratio:.5f}, "
                                      f"{rec['source']})")


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def summary(self, windows):
        sm, smax, reasons = [], 0.0, set()
        for t, c in self.rows:
            if not any(a <= t <= b for a, b in windows) or len(c) < 8:
                continue
            try:
                sm.append(float(c[1]))
                smax = max(smax, float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# the reference on the host cores (oracle/_ref), on a bounded sample of the same workload
# ------------------------------------------------------------------------------------------------------------------
HEADLINE_CG = os.path.join(ROOT, "profiles", "headline_cg_counts.json")


def ref_binary():
    """(path, flags) of the reference build to time on this host (oracle/build_ref.py: AVX-512 build when the CPU has it)."""
    v4, v3 = os.path.join(ROOT, "oracle", "_ref", "main_meth_ref_v4"), os.path.join(ROOT, "oracle", "_ref", "main_meth_ref")
    try:
        with open("/proc/cpuinfo") as f:
            flags = set(next(l for l in f if l.startswith("flags")).split(":", 1)[1].split())
    except Exception:
        flags = set()
    if {"avx512f", "avx512bw", "avx512cd", "avx512dq", "avx512vl"} <= flags and os.path.isfile(v4):
        return v4, "g++ -Ofast -march=x86-64-v4 -fopenmp"
    return (v3 if os.path.isfile(v3) else None), "g++ -Ofast -march=x86-64-v3 -fopenmp"


def ref_cg_counts(log):
    """(k1, k2) per VAMP iteration from the reference's --verbosity 1 log (src/vamp.cpp:723-724,747-748)."""
    out = []
    for block in log.split("iteration = ")[1:]:
        lm, _, ons = block.partition("[CG onsager]")
        k1 = len(re.findall(r"\[CG\] it = ", lm))
        n = len(re.findall(r"\[CG\] it = ", ons))
        last = re.findall(r"\|\|r_it\|\| / \|\|RHS\|\| = ([0-9.e+-]+)", ons)
        out.append((k1, n if (last and float(last[-1]) < 1e-5) else n + 1))
    return out


def run_reference_files(binary, d, name, N, M, iterations, threads, out_name="ref"):
    os.makedirs(os.path.join(d, out_name), exist_ok=True)
    env = dict(os.environ, OMP_NUM_THREADS=str(threads), VAMPOMI_SEED=str(PROBE_SEED))
    cmd = [binary, "--meth-file", f"{d}/{name}.bin", "--phen-file", f"{d}/{name}.phen", "--N", str(N), "--Mt", str(M), "--out-dir",
           f"{d}/{out_name}", "--out-name", "s", "--iterations", str(iterations), "--stop-criteria-thr", "0", "--true-signal-file",
           f"{d}/{name}_ts.bin", "--verbosity", "1"]
    res = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        return None, None, "reference binary failed: " + res.stdout[-300:].replace("\n", " ")
    times = [float(x) for x in re.findall(r"Total iteration time = ([0-9.eE+-]+)", res.stdout)]
    return times, ref_cg_counts(res.stdout), None


def headline_passes(warmup, steps, live_cg=None):
    """Matrix passes the REFERENCE makes per iteration at the headline size in the timed window: 2(k1+k2)+8 (SURVEY.md §3.1) with
    the CG counts of iterations W+1..W+K — measured by the GPU arm in this run (equal to the reference's by parity), or, in the
    reference arm, read from the committed record of such a run."""
    if live_cg:
        cg, src = live_cg, "CG counts of the same iterations measured by the GPU arm in this run"
    else:
        try:
            with open(HEADLINE_CG) as f:
                rec = json.load(f)
            table = rec["cg_iters_by_iteration"]
            cg = [table[min(i, len(table) - 1)] for i in range(warmup, warmup + steps)]
            src = f"CG counts of iterations {warmup + 1}..{warmup + steps} from profiles/headline_cg_counts.json ({rec['source']})"
        except Exception:
            cg, src = [[6, 6]] * steps, "no record of the headline CG counts: (6,6) assumed"
    return float(np.mean([2 * (k1 + k2) + 8 for k1, k2 in cg])), cg, src


def cpu_baseline(N, Mt, sample_M, warmup, steps, live_cg=None):
    """Times the reference binary on N x sample_M markers (same column length, same model) over iterations W+1..W+K with its own
    per-iteration timer (src/vamp.cpp:400) and derives the it/s at the headline size from its effective GB/s per pass."""
    binary, flags = ref_binary()
    if binary is None:
        return None, "oracle/_ref/main_meth_ref missing"
    threads = os.cpu_count() or 1
    from vampomi_b200 import sim
    with tempfile.TemporaryDirectory() as d:
        sim.write_dataset(d, "s", N, sample_M, lam=max(LAM, 2.0 / sample_M), h2=H2, seed=DATA_SEED)
        times, cg, err = run_reference_files(binary, d, "s", N, sample_M, warmup + steps, threads)
    if err or not times or len(times) < warmup + steps or len(cg) < warmup + steps:
        return None, err or "reference run too short"
    t_win = times[warmup:warmup + steps]
    cg_win = cg[warmup:warmup + steps]
    passes_win = [2 * (k1 + k2) + 8 for k1, k2 in cg_win]                       # it > 1: SURVEY.md §3.1
    bytes_pass = float(N) * sample_M * 8.0
    gbs = sum(passes_win) * bytes_pass / sum(t_win) / 1e9
    p_head, cg_head, cg_src = headline_passes(warmup, steps, live_cg)
    s_per_it = p_head * float(N) * Mt * 8.0 / (gbs * 1e9)
    desc = (f"oracle/_ref (patched reference, {flags}, 1 rank x {threads} OpenMP threads, its own per-iteration timer) on N={N} x {sample_M} of "
            f"the {Mt} markers ({bytes_pass / 1e9:.2f} GB per pass, full column length), iterations {warmup + 1}..{warmup + steps}: "
            f"{gbs:.1f} GB/s effective per matrix pass at its own CG counts {cg_win}; it/s at the headline size = GB/s / "
            f"({p_head:.1f} passes x {N * Mt * 8 / 1e9:.0f} GB), passes = 2(k1+k2)+8 with the {cg_src}")
    return {"value": 1.0 / s_per_it, "unit": UNIT, "cores": threads, "kind": "reference", "sample": desc,
            "effective_gbs_per_pass": gbs, "sample_s_per_iteration": float(np.mean(t_win)), "sample_cg_iters": cg_win,
            "sample_aspect": {"N": N, "M": sample_M}, "headline_passes_per_iteration": p_head, "headline_cg_iters": cg_head,
            "derived": True}, desc


def c2_full(local_device):
    """BASELINE config 2 (N = 10 000, M = 100 000, 8 GB) run IN FULL by the reference binary and by bin/main_meth on the same
    files (matrix generated on the device, downloaded and written marker-major): a measured ratio on an identical configuration."""
    import shutil
    from vampomi_b200 import build, capi, sim
    binary, flags = ref_binary()
    N, M, its = 10000, 100000, 3
    if binary is None:
        return {"skipped": "oracle/_ref missing"}
    if shutil.disk_usage(tempfile.gettempdir()).free < 12e9:
        return {"skipped": "less than 12 GB free under the temporary directory"}
    threads = os.cpu_count() or 1
    with tempfile.TemporaryDirectory() as d:
        sh = capi.Shard(N, M, device=local_device)
        sh.generate_iid(99)
        sh.compute_stats()
        rng = np.random.default_rng(99)
        CM = max(int(M * LAM), 1)
        beta = np.zeros(M)
        beta[rng.choice(M, CM, replace=False)] = rng.normal(0, math.sqrt(H2 / CM), CM)
        y = sh.Ax(beta * math.sqrt(N)) + rng.normal(0, math.sqrt(1 - H2), N)
        with open(f"{d}/c2.bin", "wb") as f:
            step = max(1, (256 << 20) // (N * 8))
            for j0 in range(0, M, step):
                sh.download(j0, min(step, M - j0)).tofile(f)
        sh.close()
        sim.write_phen(f"{d}/c2.phen", y)
        beta.tofile(f"{d}/c2_ts.bin")
        t_ref, cg_ref, err = run_reference_files(binary, d, "c2", N, M, its, threads)
        if err:
            return {"skipped": err}
        os.makedirs(f"{d}/gpu")
        res = subprocess.run([build.MAIN_METH, "--meth-file", f"{d}/c2.bin", "--phen-file", f"{d}/c2.phen", "--N", str(N), "--Mt", str(M),
                              "--out-dir", f"{d}/gpu", "--out-name", "s", "--iterations", str(its), "--stop-criteria-thr", "0",
                              "--true-signal-file", f"{d}/c2_ts.bin", "--seed", str(PROBE_SEED)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if res.returncode != 0:
            return {"skipped": "main_meth failed: " + res.stdout[-300:].replace("\n", " ")}
        t_gpu = [float(x) for x in re.findall(r"Total iteration time = ([0-9.eE+-]+)", res.stdout)]
        cg_gpu = [(int(a_), int(b_)) for a_, b_ in re.findall(r"\[CG\] LMMSE solve: (\d+) iterations, onsager solve: (\d+)", res.stdout)]
        dev = []
        for k in range(1, its + 1):
            for fn in (f"s_it_{k}.bin", f"s_r1_it_{k}.bin"):
                a_, b_ = np.fromfile(f"{d}/gpu/{fn}"), np.fromfile(f"{d}/ref/{fn}")
                dev.append(float(np.linalg.norm(a_ - b_) / max(np.linalg.norm(b_), 1e-300)))
    return {"config": f"BASELINE config 2 in full: N={N} M={M} (8 GB), CLI defaults, {its} iterations, both command lines on the same files",
            "reference_s_per_iteration": t_ref, "gpu_s_per_iteration": t_gpu, "reference_build": flags, "cores": threads,
            "ratio_iterations_2_to_3": float(sum(t_ref[1:]) / max(sum(t_gpu[1:]), 1e-12)), "cg_iters_reference": cg_ref, "cg_iters_gpu": cg_gpu,
            "cg_counts_identical": [tuple(x) for x in cg_ref] == cg_gpu, "max_rel_x1_r1": max(dev),
            "note": "default --gam1 1e-6: parity floor of this start applies (DESIGN.md §4); per-iteration timers of both programs, load excluded"}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cb, desc = cpu_baseline(args.N, args.Mt, args.cpu_sample_M, args.warmup, args.steps)
    if cb is None:
        print(json.dumps({"impl": "reference", "unavailable": desc}))
        return 0
    line = {"metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 / cb["value"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name(args.N, args.Mt), "sample": desc,
                       "note": "value is DERIVED from the measured GB/s per pass of the reference on a sample with the headline's column "
                               "length; the measured quantities are cpu_baseline.effective_gbs_per_pass and sample_s_per_iteration"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------------
# parity of the job's own ranks against committed reference-binary fixtures
# ------------------------------------------------------------------------------------------------------------------
PARITY_CASES = ("linear_wellcond", "probit_small")
_FLAG_KW = {"--EM-max-iter": ("EM_max_iter", int), "--learn-prior-delay": ("learn_prior_delay", int), "--rho": ("rho", float),
            "--gam1": ("gam1", float), "--CG-err-tol": ("CG_err_tol", float), "--EM-err-thr": ("EM_err_thr", float),
            "--learn-vars": ("learn_vars", int), "--merge-vars-thr": ("merge_vars_thr", float), "--CG-max-iter": ("CG_max_iter", int)}


def _csv_rows(blob):
    rows = {}
    for line in bytes(blob).replace(b"\0", b"").decode().splitlines():
        parts = [p.strip() for p in line.split(",")]
        try:
            rows[int(parts[0])] = [float(p) for p in parts[1:]]
        except ValueError:
            continue
    return rows


def parity_block(world, rank, local, new_comm_id, allsum, schedule):
    """Replays committed fixtures (outputs of the reference binary, tests/golden/*.npz) through Shard(nranks = world) + Solver on
    this job's ranks: the default cross-GPU data plane and schedule, checked at the tolerances of the tests (1e-9 / 1e-8)."""
    import hashlib
    from vampomi_b200 import capi, sim
    out = {"cases": [], "schedule": schedule}
    for name in PARITY_CASES:
        g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
        N, M, model = int(g["N"]), int(g["M"]), str(g["model"])
        X, y, beta = sim.simulate(N, M, float(g["lam"]), float(g["h2"]), int(g["data_seed"]), binary=model == "bin_class")
        if hashlib.sha256(X.tobytes()).hexdigest() != str(g["sha256_A"]):
            out["cases"].append({"case": name, "error": "fixture inputs could not be rebuilt (numpy generator drift)"})
            continue
        y = np.array([float("%0.10f" % v) for v in y])                        # the .phen text format the reference read
        if model == "linear":
            y = y * math.sqrt((N - 1) / float(((y - y.sum() / N) ** 2).sum()))   # data::read_phen, src/data.cpp:97-99
        kw = {}
        ex = [str(e) for e in g["extra"]]
        for k_, v_ in zip(ex[::2], ex[1::2]):
            n_, f_ = _FLAG_KW[k_]
            kw[n_] = f_(v_)
        sh = capi.Shard(N, M, device=local, nranks=world, rank=rank, nccl_id=new_comm_id())
        sh.upload(X[sh.S:sh.S + sh.M])
        sh.compute_stats()
        sol = capi.Solver(sh, y, model=model, true_signal=beta[sh.S:sh.S + sh.M], gamw=2.0, seed=int(g["probe_seed"]),
                          fuse_passes={"onepass": 3, "recycled": 2, "fused": 1, "plain": 0}[schedule], **kw)
        want_p, want_m = _csv_rows(g["csv_params"]), _csv_rows(g["csv_metrics"])
        worst_vec, worst_csv, cg_ok = 0.0, 0.0, True
        for k in range(1, int(g["iterations"]) + 1):
            r = sol.step()
            for got, want in ((r["x1"], g["x1"][k - 1][sh.S:sh.S + sh.M]), (r["r1"], g["r1"][k - 1][sh.S:sh.S + sh.M])):
                num, den = allsum(float(((got - want) ** 2).sum())), allsum(float((want ** 2).sum()))
                worst_vec = max(worst_vec, math.sqrt(num / den) if den > 0 else math.sqrt(num))
            for got, want in ((r["params"], want_p[k]), (r["metrics"], want_m[k])):
                for a_, b_ in zip(got, want):
                    if math.isnan(b_) or math.isinf(b_):
                        cg_ok = cg_ok and ((math.isnan(a_) and math.isnan(b_)) or a_ == b_)
                    elif abs(a_ - b_) > 2e-15:                                   # the CSV print quantum
                        worst_csv = max(worst_csv, abs(a_ - b_) / abs(b_) if b_ != 0 else abs(a_ - b_))
            cg_ok = cg_ok and (r["k1"], r["k2"]) == tuple(int(v_) for v_ in g["cg_iters"][k - 1])
        out["comm_mode"] = {0: "none (1 GPU)", 1: "NCCL all-reduce", 2: "fused NVLink peer-memory all-reduce"}[sh.comm_mode()]
        sol.close()
        sh.close()
        out["cases"].append({"case": name, "N": N, "Mt": M, "iterations": int(g["iterations"]), "max_rel_x1_r1": worst_vec,
                             "max_rel_csv": worst_csv, "cg_counts_identical": bool(cg_ok),
                             "pass": bool(worst_vec < 1e-9 and worst_csv < 1e-8 and cg_ok)})
    out["max_rel_x1_r1"] = max((c.get("max_rel_x1_r1", float("inf")) for c in out["cases"]), default=None)
    out["max_rel_csv"] = max((c.get("max_rel_csv", float("inf")) for c in out["cases"]), default=None)
    out["cg_counts_identical"] = all(c.get("cg_counts_identical", False) for c in out["cases"])
    out["pass"] = all(c.get("pass", False) for c in out["cases"])
    out["note"] = ("fixtures = outputs of the reference binary (tests/golden, tests/tools/make_golden.py); relative L2 over ALL shards "
                   "(sums of squares added over the ranks), tolerances 1e-9 (x1_hat, r1) / 1e-8 (CSV values), CG counts exact")
    return out


# ------------------------------------------------------------------------------------------------------------------
# outputs of the timed path (--dump-outputs)
# ------------------------------------------------------------------------------------------------------------------
DUMP_MAX_VALUES = 1 << 21       # per marker vector: x1_hat, r1 and the sample's index stay under 64 MB in all
DUMP_SAMPLE_SEED = 2027
DUMP_NAMES = ("params", "metrics", "prior_probs", "prior_vars", "cg_iters", "nmse", "sample_index", "x1_hat", "r1")


def dump_outputs(out_dir, last, x1, r1):
    """Writes what the last timed step handed its caller: the scalars returned by the step of the device-resident leg (the
    headline value), and x1_hat/sqrt(N), r1/sqrt(N) as the step of the end-to-end leg copied them to host memory (the same
    iteration W+K of an identically initialised solver), over all markers in global order. A vector longer than
    DUMP_MAX_VALUES is replaced by its entries at a fixed seeded sample of marker indices, written as sample_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    for name in DUMP_NAMES:           # a file of an earlier dump (sample_index.npy of a larger run) must not sit beside this one's
        path = os.path.join(out_dir, name + ".npy")
        if os.path.exists(path):
            os.remove(path)
    arrays = {"params": last["params"], "metrics": last["metrics"], "prior_probs": last["probs"], "prior_vars": last["vars"],
              "cg_iters": [last["k1"], last["k2"]], "nmse": [last["nmse"]]}
    if x1.size > DUMP_MAX_VALUES:
        idx = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(x1.size, DUMP_MAX_VALUES, replace=False))
        x1, r1 = x1[idx], r1[idx]
        arrays["sample_index"] = idx
    arrays.update(x1_hat=x1, r1=r1)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))
    return sorted(arrays)


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def main_ours(args):
    import torch
    import torch.distributed as dist
    from vampomi_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torchrun (one rank per GPU)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def new_comm_id():
        """A fresh NCCL unique id for one more set of contexts (rank 0 creates it, everybody receives it)."""
        if world == 1:
            return None
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt = torch.frombuffer(bytearray(capi.comm_unique_id()), dtype=torch.uint8).cuda()
        dist.broadcast(idt, 0)
        return bytes(idt.cpu().numpy().tobytes())

    def allsum(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t)
        return float(t.item())

    parity = None
    if not args.no_parity:
        try:
            parity = parity_block(world, rank, local, new_comm_id, allsum, args.schedule)
        except Exception as e:        # evidence, not the product: report instead of losing the bench line
            parity = {"error": f"{type(e).__name__}: {e}", "pass": False}
    nccl_id = new_comm_id()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    N, Mt = args.N, args.Mt
    t_setup = time.time()
    sh = capi.Shard(N, Mt, device=local, nranks=world, rank=rank, nccl_id=nccl_id, storage=args.storage)
    for kv in args.tune:
        k_, v_ = kv.split("=")
        sh.set_tuning(k_, int(v_))
    sh.generate_iid(DATA_SEED)
    sh.compute_stats()
    # phenotype of the simulated model y = A beta + noise (simulation/data_sim.py:37-47), built with the device operator
    rng = np.random.default_rng(DATA_SEED)
    CM = max(int(Mt * LAM), 1)
    idx = rng.choice(Mt, size=CM, replace=False)
    beta = np.zeros(Mt)
    beta[idx] = rng.normal(0.0, math.sqrt(H2 / CM), CM)
    noise = rng.normal(0.0, math.sqrt(1.0 - H2), N)
    beta_sh = beta[sh.S:sh.S + sh.M]
    g = sh.Ax(beta_sh * math.sqrt(N))
    y = g + noise
    y = y * math.sqrt((N - 1) / float(((y - y.mean()) ** 2).sum()))         # data::read_phen scaling, src/data.cpp:97-99
    setup_s = time.time() - t_setup

    # live read ceiling of this GPU on this very buffer: plain linear streaming read (vampomi_time_kernel which=4), burst of 5
    sh.time_kernel(4, 2)
    probe_ms = sh.time_kernel(4, 5)
    probe_gbs = sh.M * ((N + 15) // 16 * 16) * (8 if args.storage == "f64" else 4) / (probe_ms * 1e-3) / 1e9

    stream = torch.cuda.ExternalStream(sh.stream(), device=torch.device("cuda", local))
    y_pinned = torch.from_numpy(y.copy()).pin_memory()
    x1_host = torch.empty(sh.M, dtype=torch.float64).pin_memory()
    r1_host = torch.empty(sh.M, dtype=torch.float64).pin_memory()

    if args.record_cg_counts > 0:
        sol = capi.Solver(sh, y, model="linear", true_signal=beta_sh, gamw=1.0 / (1.0 - H2), seed=PROBE_SEED,
                          fuse_passes={"onepass": 3, "recycled": 2, "fused": 1, "plain": 0}[args.schedule])
        table = []
        for _ in range(args.record_cg_counts):
            h = sol.step(want_vectors=False)
            table.append([h["k1"], h["k2"]])
        sol.close()
        sh.close()
        if rank == 0:
            with open(HEADLINE_CG, "w") as f:
                json.dump({"workload": workload_name(N, Mt), "data_seed": DATA_SEED, "probe_seed": PROBE_SEED,
                           "source": f"bench.py --record-cg-counts {args.record_cg_counts} on {world} B200 (CG counts do not depend on the GPU count)",
                           "cg_iters_by_iteration": table}, f, indent=1)
            print(json.dumps({"recorded": HEADLINE_CG, "cg_iters_by_iteration": table}))
        if world > 1:
            dist.destroy_process_group()
        return 0

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    windows = []

    def leg(e2e, schedule=None):
        sol = capi.Solver(sh, y, model="linear", true_signal=beta_sh, gamw=1.0 / (1.0 - H2), seed=PROBE_SEED,
                          fuse_passes={"onepass": 3, "recycled": 2, "fused": 1, "plain": 0}[schedule or args.schedule])
        hist = []
        for _ in range(args.warmup):
            hist.append(sol.step(want_vectors=False))
        barrier()
        sh.counters(reset=True)
        sh.profile(True)
        sh.profile_read(reset=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        e0.record(stream)
        for _ in range(args.steps):
            if e2e:
                sh.set(capi.V_Y, y_pinned.numpy())                        # H2D of the step's input
                hist.append(sol.step(want_vectors=True, out_x1=x1_host.numpy(), out_r1=r1_host.numpy()))   # D2H of its result
            else:
                hist.append(sol.step(want_vectors=False))
        e1.record(stream)
        barrier()
        w1 = time.time()
        windows.append((w0, w1))
        ms = e0.elapsed_time(e1)
        prof = sh.profile_read(reset=True)
        sh.profile(False)
        cnt = sh.counters()
        sol.close()
        if world > 1:
            # per-rank device time of the two matrix kernels and of the exchange tail: tells systematic from random rank skew
            mine = torch.tensor([prof["ax_partial"]["ms"] / max(prof["ax_partial"]["launches"], 1),
                                 prof["atx"]["ms"] / max(prof["atx"]["launches"], 1),
                                 1e3 * prof["ax_reduce"]["ms"] / max(prof["ax_reduce"]["launches"], 1), ms], dtype=torch.float64, device="cuda")
            allr = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allr, mine)
            prof["per_rank"] = {"ax_avg_ms": [round(float(a[0]), 4) for a in allr], "atx_avg_ms": [round(float(a[1]), 4) for a in allr],
                                "ax_exchange_tail_avg_us": [round(float(a[2]), 1) for a in allr],
                                "leg_ms": [round(float(a[3]), 3) for a in allr]}
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            k = torch.tensor([float(cnt["kernels"])], dtype=torch.float64, device="cuda")
            dist.all_reduce(k)
            cnt["kernels"] = int(k.item())
        return ms, hist[args.warmup:], prof, cnt

    ms_dev, hist_dev, prof_dev, cnt_dev = leg(e2e=False)
    ms_e2e, hist_e2e, prof_e2e, cnt_e2e = leg(e2e=True)
    dumped = None
    if args.dump_outputs:
        x1_all, r1_all = x1_host.numpy().copy(), r1_host.numpy().copy()
        if world > 1:                 # shards in rank order are the markers in global order (divide_work)
            parts = [None] * world
            dist.all_gather_object(parts, (x1_all, r1_all))
            x1_all, r1_all = np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
        if rank == 0:
            dumped = dump_outputs(args.dump_outputs, hist_dev[-1], x1_all, r1_all)
    # the other schedules on the same box, same iterations (device-resident leg only): what each level of pass sharing buys
    ab = {}
    if not args.no_ab:
        for sched in ("plain", "fused", "recycled", "onepass"):
            if sched == args.schedule:
                continue
            ms_s, hist_s, _, _ = leg(e2e=False, schedule=sched)
            ab[sched] = {"value": args.steps / (ms_s / 1e3), "ms_per_step": ms_s / args.steps,
                         "passes": sum(h["matrix_passes"] for h in hist_s),
                         "cg_iters_per_step": [[h["k1"], h["k2"]] for h in hist_s]}
    if rank == 0:
        sampler.stop()

    if rank != 0:
        sh.close()
        if world > 1:
            dist.destroy_process_group()
        return 0

    value = args.steps / (ms_dev / 1e3)
    e2e_value = args.steps / (ms_e2e / 1e3)
    peak, peak_src = measured_peak()
    # dominant kernel: the matrix pass with the larger total device time in the timed region (rank 0's shard)
    dom = max(("ax_partial", "atx", "gram"), key=lambda k: prof_dev[k]["ms"])
    pd = prof_dev[dom]
    bytes_per_launch = pd["bytes"] / max(pd["launches"], 1)
    avg_ms = pd["ms"] / max(pd["launches"], 1)
    achieved = bytes_per_launch / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
    passes = sum(h["matrix_passes"] for h in hist_dev)
    iter_bytes = passes * float(N) * float(Mt) * (8.0 if args.storage == "f64" else 4.0)                       # whole job: P * N * Mt * 8 over the timed region
    iter_gbs_per_gpu = iter_bytes / (ms_dev * 1e-3) / 1e9 / world
    per_rank = prof_dev.pop("per_rank", None)
    prof_e2e.pop("per_rank", None)
    matrix_ms = sum(prof_dev[k]["ms"] for k in prof_dev)
    # kernel behind each profiling slot: in the fused schedule every pass of iterations > 1 is a multi-vector kernel
    knames = ({"ax_partial": "k_ax_multi", "atx": "k_atx_smem"} if args.schedule != "plain" else {"ax_partial": "k_ax_partial", "atx": "k_atx_cta"})
    knames["gram"] = "k_gram"
    products = sum(2 * (h["k1"] + h["k2"]) + 6 for h in hist_dev)                # matrix-vector products the iterations need (the reference streams A for each, plus 2 repeats)
    traffic, traffic_src = ncu_traffic(knames[dom], N, sh.M, bytes_per_launch)
    roofline = {"bound": "hbm", "kernel": knames[dom], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "frac_of_8TBs_spec": achieved / 8000.0, "read_probe_gbs": probe_gbs, "frac_of_read_probe": achieved / probe_gbs,
                "read_probe_note": "plain linear LDG.256 streaming read of the same buffer, burst of 5 launches before the timed region",
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "bytes_per_launch": bytes_per_launch, "avg_launch_ms": avg_ms,
                "launches_timed": pd["launches"],
                "other_kernel": {k: (prof_dev[k]["bytes"] / max(prof_dev[k]["ms"], 1e-9) / 1e6) for k in ("ax_partial", "atx", "gram") if prof_dev[k]["launches"]},
                "matrix_kernel_share_of_step": (prof_dev["ax_partial"]["ms"] + prof_dev["atx"]["ms"] + prof_dev["gram"]["ms"]) / ms_dev,
                "phase_ms_per_step": {knames["ax_partial"]: prof_dev["ax_partial"]["ms"] / args.steps,
                                      "k_ax_reduce+allreduce+scale": prof_dev["ax_reduce"]["ms"] / args.steps,
                                      knames["atx"] + ("+k_atx_reduce" if args.schedule != "plain" else ""): prof_dev["atx"]["ms"] / args.steps,
                                      "k_gram": prof_dev["gram"]["ms"] / args.steps,
                                      "everything_else": (ms_dev - matrix_ms) / args.steps,
                                      "ax_reduce_avg_us": 1e3 * prof_dev["ax_reduce"]["ms"] / max(prof_dev["ax_reduce"]["launches"], 1)},
                "whole_iteration": {"passes": passes, "gbs_per_gpu": iter_gbs_per_gpu, "frac_of_peak": iter_gbs_per_gpu / peak,
                                    "frac_of_8TBs_spec": iter_gbs_per_gpu / 8000.0,
                                    "matrix_vector_products": products,
                                    "note": "passes = reads of the whole marker block actually made in the timed steps (bytes = passes x N x Mt x 8); "
                                            "matrix_vector_products = products those steps computed — the one-product-per-pass schedule "
                                            "reads the block once for each"}}
    if dom == "gram":
        # one k_gram_ws launch delivers BOTH products of a CG iteration (A^T q and A A^T q, for both systems): by BASELINE.json's
        # own unit — a CG iteration = 2*N*M*8 bytes — it does the work of two reads while reading the block once
        roofline["cg_iteration_equivalent_gbs"] = 2.0 * achieved
        roofline["achieved_note"] = ("achieved counts ONE read of the block per launch (the bytes the launch needs); the reference's "
                                     "unit for the same work is 2*N*M*8 per CG iteration")
    equiv = products * float(N) * float(Mt) * 8.0 / (ms_dev * 1e-3) / 1e9 / world
    roofline["whole_iteration"]["equivalent_gbs_per_gpu"] = equiv
    roofline["whole_iteration"]["equivalent_frac_of_8TBs_spec"] = equiv / 8000.0
    roofline["whole_iteration"]["equivalent_note"] = ("SURVEY.md §8d / north_star unit: P = 2(k1+k2)+6 necessary passes per iteration, each N*Mt*8 bytes, "
                                                      "over the measured time — what the products delivered would cost read one by one")
    if per_rank:
        roofline["per_rank"] = per_rank
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64" if args.storage == "f64" else "f64 arithmetic on a matrix held as f32 (opt-in mode, not the headline)",
            "data": "synthetic",
            "config": {"workload": workload_name(N, Mt), "N": N, "Mt": Mt, "markers_per_gpu": sh.M, "parallelism": f"marker-shard x{world}", "schedule": args.schedule, **({"tune": args.tune} if args.tune else {}),
                       "l2_note": f"inputs larger than L2: every matrix pass streams {sh.M * N * 8 / 1e9:.1f} GB per GPU",
                       "cg_iters_per_step": [[h["k1"], h["k2"]] for h in hist_dev], "first_timed_iteration": args.warmup + 1, "setup_s": round(setup_s, 2),
                       "cross_gpu_sums": {0: "none (1 GPU)", 1: "NCCL all-reduce", 2: "fused NVLink peer-memory all-reduce"}[sh.comm_mode()]},
            "roofline": roofline,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int(N * 8 + 2 * 32 * 8), "d2h_bytes_per_step": int(2 * sh.M * 8 * world + 64 * 8 * 12),
                    "note": "vampomi_solver_step through the host-buffer C ABI; per step: phenotype H2D, x1_hat and r1 D2H"},
            "gpu_launches": int(cnt_dev["kernels"]),
            "clocks": sampler.summary(windows)}
    if ab:
        ab[args.schedule] = {"value": value, "ms_per_step": ms_dev / args.steps, "passes": passes,
                             "cg_iters_per_step": [[h["k1"], h["k2"]] for h in hist_dev]}
        line["schedules"] = {"unit": UNIT, "note": "same W+1..W+K iterations, device-resident leg, one after the other on this box; "
                             "`value` above is the default schedule's", **ab}
    if parity is not None:
        line["parity"] = parity
    if dumped:
        line["dumped_outputs"] = {"dir": os.path.abspath(args.dump_outputs), "files": [n + ".npy" for n in dumped]}
    live_cg = [[h["k1"], h["k2"]] for h in hist_dev]
    sh.close()
    if not args.no_cpu_baseline and world == 1:
        cb, why = cpu_baseline(N, Mt, args.cpu_sample_M, args.warmup, args.steps, live_cg=live_cg)
        line["cpu_baseline"] = cb if cb else {"unavailable": why}
        if cb and not args.no_cpu_c2:
            try:
                line["cpu_baseline"]["c2_full"] = c2_full(local)
            except Exception as e:
                line["cpu_baseline"]["c2_full"] = {"skipped": f"{type(e).__name__}: {e}"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    a = parse_args()
    sys.exit(main_reference(a) if a.impl == "reference" else main_ours(a))
