"""End-to-end parity of the VAMP loop on the GPU: per-iteration x1_hat / r1, params / metrics rows and CG iteration
counts against fixtures produced by the reference binary (tests/golden) and against the numpy oracle; the main_meth
command line against the same fixtures, byte layout of the CSVs included; plus full-size property checks."""
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import vamp_oracle as vo
from vampomi_b200 import build, capi, sim
from vampomi_b200.capi import V_QINV_BERN, V_USER_M0, V_USER_M1, V_USER_N0, V_USER_N1, V_V, V_X1, V_X2, V_Y
from helpers import (assert_rows_close, csv_rows, extra_kwargs, golden_covariates, golden_inputs, load_golden, oracle_run, rel_l2,
                     standardize_phen, tolerances)

pytestmark = pytest.mark.gpu

CASES = ["linear_large_gam2", "linear_cov", "probit_cov", "linear_wide_default", "linear_small", "linear_readme", "linear_ragged", "linear_wellcond", "linear_two_comp", "linear_alpha_scale",
         "linear_stops_early", "linear_warm_start", "probit_small", "probit_ragged", "linear_wide", "probit_wide", "linear_cg_cap", "linear_tight_cg",
         "linear_em_conv", "linear_h2"]


def solver_for(g, A, y_txt, beta, **over):
    model = g["model"]
    y = standardize_phen(y_txt) if model == "linear" else y_txt
    kw = dict(gamw=2.0, seed=int(g["probe_seed"]))
    kw.update(extra_kwargs(g))
    if "h2" in kw:
        kw["gamw"] = 1.0 / (1.0 - kw.pop("h2"))              # src/main_meth.cpp:52
    kw.update(over)
    sh = capi.Shard(int(g["N"]), int(g["M"]))
    sh.upload(A)
    sh.compute_stats(kw.pop("alpha_scale", 1.0))
    sol = capi.Solver(sh, y, model=model, true_signal=beta, x1hat_init=g.get("x1hat_init"), **kw)
    if "C" in g:                                              # --C / --cov-file: standardised covariates, effects fitted in iteration 1
        sol.set_covariates(golden_covariates(g))
    return sh, sol


# schedules of the matrix passes: "onepass" (recycled + CG iterations that read the block once: fused A^T q / A A^T q pass), "recycled" (fused + A x2_hat, A Q^-1 u and A^T A of both kept by the solves themselves),
# "fused" (products that are known together share one read of the block),
# "plain" (one product per pass, A^T y and A x2_hat cached), "reference" (plain + the passes the reference repeats)
SCHEDULES = {"onepass": dict(fuse_passes=3, redundant_passes=0), "recycled": dict(fuse_passes=2, redundant_passes=0), "fused": dict(fuse_passes=1, redundant_passes=0), "plain": dict(fuse_passes=0, redundant_passes=0),
             "reference": dict(fuse_passes=0, redundant_passes=1)}


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("schedule", list(SCHEDULES))
def test_solver_matches_reference_fixture(name, schedule):
    g = load_golden(name)
    rel_vec, rel_csv = tolerances(g)
    A, y_txt, beta = golden_inputs(g)
    sh, sol = solver_for(g, A, y_txt, beta, **SCHEDULES[schedule])
    want_params, want_metrics = csv_rows(g["csv_params"]), csv_rows(g["csv_metrics"])
    got_params, got_metrics = {}, {}
    gamw_used = sol.cfg.gamw                     # tau of this iteration's solves = gamw after the previous iteration (src/vamp.cpp:308)
    for k in range(1, int(g["iterations"]) + 1):
        r = sol.step()
        assert r["it"] == k
        assert rel_l2(r["x1"], g["x1"][k - 1]) < rel_vec, f"x1_hat it {k}"
        assert rel_l2(r["r1"], g["r1"][k - 1]) < rel_vec, f"r1 it {k}"
        got_params[k], got_metrics[k] = r["params"], r["metrics"]
        assert (r["k1"], r["k2"]) == tuple(g["cg_iters"][k - 1]), f"CG iteration counts it {k}"      # exact, both models
        if g["model"] == "linear":
            base = 2 * (r["k1"] + r["k2"])
            if schedule == "reference":   # the reference's own pass count: 6 (it = 1) / 8 (it > 1) + 2(k1+k2), SURVEY.md §3.1
                assert r["matrix_passes"] == base + (6 if k == 1 else 8)
            elif schedule == "plain":     # A^T y cached, A x2_hat computed once
                assert r["matrix_passes"] == base + (5 if k == 1 else 6)
            elif schedule == "fused":     # A^T y once; both solves in lock-step; A [x2, Q^-1 u] and A^T [.., A x2] one pass each
                assert r["matrix_passes"] == 2 * max(r["k1"], r["k2"]) + (3 if k == 1 else 2)
            elif schedule in ("onepass", "recycled"):
                # recycled: nothing but the lock-step solves (and A^T y once); onepass: A [p0 p1 x1] once, then ONE fused pass per
                # lock-step CG iteration. Both recompute the recycled products by two explicit passes every 16th iteration and
                # whenever gam2/tau > 1e5 (cancellation in (rhs - r - gam2 sol)/tau, host/vamp.cpp)
                refresh = 2 if (k % 16 == 0 or r["params"][3] / gamw_used > 1e5) else 0
                solves = max(r["k1"], r["k2"]) + 1 if schedule == "onepass" else 2 * max(r["k1"], r["k2"])
                assert r["matrix_passes"] == solves + (1 if k == 1 else 0) + refresh
            gamw_used = r["params"][4]
        else:
            if schedule == "fused":       # A^T p2, lock-step solves, A [x2, x2/sqrt(N)]
                assert r["matrix_passes"] == 2 * max(r["k1"], r["k2"]) + 2
            elif schedule == "recycled":  # A^T p2, lock-step solves
                assert r["matrix_passes"] == 2 * max(r["k1"], r["k2"]) + 1
            elif schedule == "onepass":   # A^T p2, A [p0 p1 x1/sqrt(N)], one fused pass per lock-step CG iteration
                assert r["matrix_passes"] == max(r["k1"], r["k2"]) + 2
            else:
                assert r["matrix_passes"] == 2 * (r["k1"] + r["k2"]) + 4
    assert_rows_close(got_params, want_params, rel_csv, "params")
    assert_rows_close(got_metrics, want_metrics, rel_csv, "metrics")
    if float(g.get("stop_thr", 0)) > 0:          # the reference stopped here on its own NMSE test (src/vamp.cpp:419-423)
        assert r["nmse"] < float(g["stop_thr"])
    if "C" in g:                                 # the covariate effects the reference printed (6 significant digits)
        assert np.allclose(sol.cov_eff(), g["cov_eff"], rtol=2e-5, atol=1e-9)
    sol.close()
    sh.close()


@pytest.mark.parametrize("name", ["linear_wellcond", "probit_small"])
def test_solver_matches_oracle_tightly(name):
    """GPU vs the numpy oracle on the well-conditioned fixtures: both restate the same arithmetic, so they agree far
    below the 1e-9 contract."""
    g = load_golden(name)
    A, y_txt, beta = golden_inputs(g)
    v = oracle_run(g, A, y_txt, beta)
    sh, sol = solver_for(g, A, y_txt, beta)
    for k in range(1, int(g["iterations"]) + 1):
        r = sol.step()
        assert rel_l2(r["x1"], v.dump[k][0]) < 1e-10 and rel_l2(r["r1"], v.dump[k][1]) < 1e-10
        assert np.allclose(r["probs"], v.history[k - 1]["probs"], rtol=1e-9)
    sol.close()
    sh.close()


def run_cli(args, **kw):
    res = subprocess.run([build.MAIN_METH] + [str(a) for a in args], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, **kw)
    assert res.returncode == 0, res.stdout[-3000:]
    return res.stdout


@pytest.mark.parametrize("schedule", ["onepass", "recycled", "fused", "plain", "reference"])
def test_main_meth_schedule_flag(schedule, tmp_path):
    """--schedule only changes which products share a read of the block: same files for all three."""
    g = load_golden("linear_wellcond")
    rel_vec, rel_csv = tolerances(g)
    d = str(tmp_path)
    golden_inputs(g, d)
    os.makedirs(tmp_path / "out")
    its = int(g["iterations"])
    out = run_cli(["--meth-file", f"{d}/ex.bin", "--phen-file", f"{d}/ex.phen", "--N", g["N"], "--Mt", g["M"], "--out-dir", f"{d}/out",
                   "--out-name", "g", "--iterations", its, "--true-signal-file", f"{d}/ex_ts.bin", "--stop-criteria-thr", 0,
                   "--seed", g["probe_seed"], "--schedule", schedule] + list(g["extra"]))
    assert f"--schedule {schedule}" in out
    for k in range(1, its + 1):
        assert rel_l2(np.fromfile(f"{d}/out/g_it_{k}.bin"), g["x1"][k - 1]) < rel_vec
        assert rel_l2(np.fromfile(f"{d}/out/g_r1_it_{k}.bin"), g["r1"][k - 1]) < rel_vec
    for kind in ("params", "metrics"):
        assert_rows_close(csv_rows(open(f"{d}/out/g_{kind}.csv", "rb").read()), csv_rows(bytes(g[f"csv_{kind}"])), rel_csv, kind)
    res = subprocess.run([build.MAIN_METH, "--schedule", "sideways"], stdout=subprocess.PIPE, text=True)
    assert res.returncode == 1 and "FATAL" in res.stdout


@pytest.mark.parametrize("name", ["linear_small", "probit_small", "linear_stops_early", "linear_warm_start", "linear_alpha_scale",
                                  "linear_two_comp"])
def test_main_meth_command_line_outputs(name, tmp_path):
    g = load_golden(name)
    rel_vec, rel_csv = tolerances(g)
    d = str(tmp_path)
    golden_inputs(g, d)
    os.makedirs(tmp_path / "out")
    its = int(g["iterations"])
    early = float(g.get("stop_thr", 0)) > 0
    args = ["--meth-file", f"{d}/ex.bin", "--phen-file", f"{d}/ex.phen", "--N", g["N"], "--Mt", g["M"], "--out-dir", f"{d}/out",
            "--out-name", "g", "--iterations", 40 if early else its, "--true-signal-file", f"{d}/ex_ts.bin", "--model", g["model"],
            "--stop-criteria-thr", g.get("stop_thr", 0), "--seed", g["probe_seed"], "--run-mode", "inference"] + list(g["extra"])
    if "x1hat_init" in g:
        g["x1hat_init"].tofile(f"{d}/init_it_3.bin")
        args += ["--estimate-file", f"{d}/init_it_3.bin"]
    out = run_cli(args)
    assert "iteration = 1" in out and "x1_hat NMSE" in out
    if early:
        assert "...stopping criteria fulfilled" in out and not os.path.exists(f"{d}/out/g_it_{its + 1}.bin")
    for k in range(1, its + 1):
        assert rel_l2(np.fromfile(f"{d}/out/g_it_{k}.bin"), g["x1"][k - 1]) < rel_vec
        assert rel_l2(np.fromfile(f"{d}/out/g_r1_it_{k}.bin"), g["r1"][k - 1]) < rel_vec
    for kind in ("params", "metrics", "prior"):
        got = open(f"{d}/out/g_{kind}.csv", "rb").read()
        want = bytes(g[f"csv_{kind}"])
        assert len(got) == len(want), f"{kind}.csv size"
        if kind != "prior" or g["model"] == "linear":
            assert np.array_equal(np.frombuffer(got, np.uint8) == 0, np.frombuffer(want, np.uint8) == 0), f"{kind}.csv NUL layout"
        if kind == "prior" and g["model"] == "linear":
            assert got == want
        if kind != "prior":
            assert_rows_close(csv_rows(got), csv_rows(want), rel_csv, kind)


def test_association_and_test_modes(tmp_path):
    g = load_golden("linear_small")
    d = str(tmp_path)
    golden_inputs(g, d)
    os.makedirs(tmp_path / "out")
    last = int(g["iterations"])
    for k in range(1, last + 1):
        g["x1"][k - 1].tofile(f"{d}/out/g_it_{k}.bin")
        g["r1"][k - 1].tofile(f"{d}/out/g_r1_it_{k}.bin")
    common = ["--meth-file", f"{d}/ex.bin", "--phen-file", f"{d}/ex.phen", "--N", g["N"], "--Mt", g["M"], "--out-dir", f"{d}/out",
              "--out-name", "g"]
    run_cli(common + ["--run-mode", "association_test", "--pval-method", "se", "--r1-file", f"{d}/out/g_r1_it_{last}.bin",
                      "--gam1", repr(float(g["se_gam1"]))])
    assert np.allclose(np.fromfile(f"{d}/out/g_it_{last}_pval_se.bin"), g["pval_se"], rtol=1e-10, atol=1e-300)
    run_cli(common + ["--run-mode", "association_test", "--pval-method", "loo", "--estimate-file", f"{d}/out/g_it_{last}.bin"])
    assert np.allclose(np.fromfile(f"{d}/out/g_it_{last}_pval_loo.bin"), g["pval_loo"], rtol=1e-7, atol=1e-300)
    Nt = int(g["N_test"])
    sim.write_dataset(d, "tst", Nt, int(g["M"]), float(g["lam"]), float(g["h2"]), int(g["data_seed"]) + 1000)
    run_cli(["--meth-file-test", f"{d}/tst.bin", "--phen-file-test", f"{d}/tst.phen", "--N-test", Nt, "--Mt", g["M"], "--out-dir",
             f"{d}/out", "--out-name", "g", "--run-mode", "test", "--estimate-file", f"{d}/out/g_it_1.bin", "--test-iter-range",
             f"1,{last}"])
    got = open(f"{d}/out/g_test.csv", "rb").read()
    want = bytes(g["csv_test"])
    assert len(got) == len(want) and got[:39] == want[:39]
    assert_rows_close(csv_rows(got), csv_rows(want), 1e-8, "test.csv")
    # four saved estimates share one pass over the test matrix (ranges that are not a multiple of four, a missing file:
    # like the reference, an unreadable estimate is a zero vector, src/utilities.cpp:251-267, i.e. R2 = 1 - |y|^2/(sd^2 n))
    os.remove(f"{d}/out/g_test.csv")
    run_cli(["--meth-file-test", f"{d}/tst.bin", "--phen-file-test", f"{d}/tst.phen", "--N-test", Nt, "--Mt", g["M"], "--out-dir",
             f"{d}/out", "--out-name", "g", "--run-mode", "test", "--estimate-file", f"{d}/out/g_it_1.bin", "--test-iter-range",
             f"1,{last + 2}"])
    rows = csv_rows(open(f"{d}/out/g_test.csv", "rb").read())
    assert sorted(rows) == list(range(1, last + 3))
    assert_rows_close({k: rows[k] for k in range(1, last + 1)}, csv_rows(want), 1e-8, "test.csv, longer range")
    assert rows[last + 1][0] == rows[last + 2][0] and rows[last + 1][0] < 0.01
    # README's literal association command (test-file flags) fails like the reference: FATAL, exit 1 (SURVEY.md §3.3)
    res = subprocess.run([build.MAIN_METH, "--meth-file-test", f"{d}/ex.bin", "--phen-file-test", f"{d}/ex.phen", "--N", "300", "--Mt", "800",
                          "--run-mode", "association_test"], stdout=subprocess.PIPE, text=True)
    assert res.returncode == 1 and "FATAL: could not open phenotype file" in res.stdout


def test_full_size_properties():
    """One 8-GPU shard of the headline configuration (N = 20 000, M = 106 250; 17 GB), device-generated: properties that
    do not need a CPU pass over the matrix — adjointness <A x, p> = <x, A^T p>, linearity, statistics of the synthetic
    block, kernel variants agreeing, and the CG solution satisfying its own residual test through independent calls."""
    N, M = 20000, 106250
    sh = capi.Shard(N, M)
    sh.generate_iid(7)
    sh.compute_stats()
    mave, msig = sh.stats()
    assert abs(mave.mean()) < 1e-3 and abs(msig.mean() - 1) < 1e-2
    rng = np.random.default_rng(0)
    x, x2, p = rng.standard_normal(M), rng.standard_normal(M), rng.standard_normal(N)
    Ax, ATp = sh.Ax(x), sh.ATx(p)
    assert abs(Ax @ p - x @ ATp) <= 1e-11 * math.sqrt((Ax @ Ax) * (p @ p))
    assert rel_l2(sh.Ax(0.5 * x - 2 * x2), 0.5 * Ax - 2 * sh.Ax(x2)) < 1e-12
    for knobs in (dict(ax_rv=1, ax_unroll=8), dict(ax_rv=4, ax_unroll=4), dict(atx_impl=0, atx_cols=1, atx_unroll=8), dict(atx_impl=0, atx_cols=4, atx_unroll=4),
                  dict(atx_impl=2, atx_cols=2, atx_unroll=4), dict(ax_impl=1, atx_impl=1)):
        for k, v in knobs.items():
            sh.set_tuning(k, v)
        assert rel_l2(sh.Ax(x), Ax) < 1e-13 and rel_l2(sh.ATx(p), ATp) < 1e-13
    sh.set_tuning("atx_impl", 3); sh.set_tuning("ax_impl", 0)
    for k in ("ax_rv", "ax_unroll", "atx_cols", "atx_unroll"):
        sh.set_tuning(k, 0)
    # the iteration's own kernels at this size — k_ax_multi (2 and 3 vectors), k_atx_smem (2 vectors, 10 row tiles) and the fused
    # k_gram pass (8 CTAs per cluster): agreement with the single-vector kernels and adjointness
    from vampomi_b200.capi import V_R1, V_R2, V_Z1, V_Z2, V_TRUE
    x3 = rng.standard_normal(M)
    p2 = rng.standard_normal(N)
    for vec, val in ((V_X1, x), (V_X2, x2), (V_V, x3)):
        sh.set(vec, val)
    Ax2, Ax3, ATp2 = sh.Ax(x2), sh.Ax(x3), sh.ATx(p2)
    sh.ax_multi_dev([V_X1, V_X2], [V_Z1, V_Z2])
    assert rel_l2(sh.get(V_Z1), Ax) < 1e-13 and rel_l2(sh.get(V_Z2), Ax2) < 1e-13
    sh.ax_multi_dev([V_X1, V_X2, V_V], [V_Z1, V_Z2, V_USER_N0])
    assert rel_l2(sh.get(V_Z1), Ax) < 1e-13 and rel_l2(sh.get(V_Z2), Ax2) < 1e-13 and rel_l2(sh.get(V_USER_N0), Ax3) < 1e-13
    sh.set(V_USER_N0, p); sh.set(V_USER_N1, p2)
    sh.atx_multi_dev([V_USER_N0, V_USER_N1], [V_R1, V_R2])
    assert rel_l2(sh.get(V_R1), ATp) < 1e-13 and rel_l2(sh.get(V_R2), ATp2) < 1e-13
    assert abs(sh.get(V_Z2) @ p2 - x2 @ sh.get(V_R2)) <= 1e-11 * math.sqrt((Ax2 @ Ax2) * (p2 @ p2))
    for shape in (18, 16, 11, 10, 6, 3, 0):
        sh.set_tuning("gram_shape", shape)
        sh.aat_multi_dev([V_USER_N0, V_USER_N1], [V_R1, V_R2], [V_Z1, V_Z2])
        assert rel_l2(sh.get(V_R1), ATp) < 1e-13 and rel_l2(sh.get(V_R2), ATp2) < 1e-13, shape
        assert rel_l2(sh.get(V_Z1), sh.Ax(ATp)) < 1e-13 and rel_l2(sh.get(V_Z2), sh.Ax(ATp2)) < 1e-13, shape
    sh.set_tuning("gram_shape", 18)
    w1 = sh.get(V_Z1)
    assert abs(w1 @ p2 - ATp @ ATp2) <= 1e-11 * math.sqrt((w1 @ w1) * (p2 @ p2))       # <A A^T p, p2> = <A^T p, A^T p2>
    # CG: ||(tau A^T A + gam2) mu - v|| / ||v|| below the tolerance, evaluated with separate operator calls
    tau, gam2 = 1.7, 0.9
    v = rng.standard_normal(M)
    sh.set(V_V, v)
    it, rel, _ = sh.cg_solve(V_V, V_X2, tau, gam2, tol=1e-8, max_iter=200)
    mu = sh.get(V_X2)
    res = v - (tau * sh.ATx(sh.Ax(mu)) + gam2 * mu)
    assert 1 < it < 200 and np.linalg.norm(res) / np.linalg.norm(v) < 2e-8
    assert abs(np.linalg.norm(res) / np.linalg.norm(v) - rel) < 1e-9
    # the one-pass CG (q = A p by recurrence, fused pass) stops after the same number of iterations at the same solution
    sh.set_tuning("cg_onepass", 1)
    it1, rel1, _ = sh.cg_solve(V_V, V_USER_M0, tau, gam2, tol=1e-8, max_iter=200)
    assert it1 == it and rel_l2(sh.get(V_USER_M0), mu) < 1e-11 and abs(rel1 - rel) < 1e-6 * rel
    sh.close()


DEFAULT_GAM1_CASES = ["linear_small", "linear_ragged", "linear_readme", "linear_wide_default"]


@pytest.mark.parametrize("name", DEFAULT_GAM1_CASES)
def test_default_gam1_runs_sit_inside_the_reference_builds_own_spread(name):
    """Runs that start from the CLI default --gam1 1e-6 (the headline benchmark is one): at iteration 1 alpha1 = 1 + sigma *
    pkdd/pk cancels to ~1e-8 (src/vamp.cpp:489), so the reference's README-flag (-Ofast) build and an IEEE-strict (-O2) build of
    the SAME sources differ from each other from iteration 2 on (fixture x1_O2 / r1_O2). The CUDA path is held to that
    measured spread — not to a flat tolerance: per iteration, its distance to the -Ofast build may not exceed 1.5 x the
    distance between the two builds, and its distance to the IEEE-strict -O2 build must stay below 1e-11 (measured on a B200:
    <= 6e-14 on all four fixtures, while the two builds are up to 4.4e-7 apart — the -Ofast binary is the outlier)."""
    g = load_golden(name)
    A, y_txt, beta = golden_inputs(g)
    sh, sol = solver_for(g, A, y_txt, beta)
    rows_fast, rows_o2 = csv_rows(g["csv_params"]), csv_rows(g["csv_params_O2"])
    report = []
    for k in range(1, int(g["iterations"]) + 1):
        r = sol.step()
        for key, fast, o2 in (("x1", g["x1"][k - 1], g["x1_O2"][k - 1]), ("r1", g["r1"][k - 1], g["r1_O2"][k - 1])):
            spread = rel_l2(o2, fast)
            d_fast, d_o2 = rel_l2(r[key], fast), rel_l2(r[key], o2)
            report.append((k, key, spread, d_fast, d_o2))
            if k == 1 and key == "x1":
                continue                                         # x1_hat of iteration 1 is exactly zero in all three
            assert d_fast <= 1.5 * spread + 2e-12, (name, k, key, spread, d_fast, d_o2)
            assert d_o2 <= 1e-11, (name, k, key, spread, d_fast, d_o2)
        # alpha1 of this iteration (params column 0): the quantity whose cancellation sets the floor
        a_gpu, a_fast, a_o2 = r["params"][0], rows_fast[k][0], rows_o2[k][0]
        assert abs(a_gpu - a_o2) <= 1e-10 * abs(a_o2) + 2e-15, (name, k, a_gpu, a_fast, a_o2)      # 15 printed decimals
        assert (r["k1"], r["k2"]) == tuple(g["cg_iters"][k - 1])
    print("\n".join(f"{name} it {k} {key}: builds apart {s:.2e}, gpu-Ofast {a:.2e}, gpu-O2 {b:.2e}" for k, key, s, a, b in report))
    sol.close()
    sh.close()


@pytest.mark.parametrize("name", ["linear_wellcond", "probit_small"])
def test_f32_storage_vamp_matches_oracle_on_rounded_matrix(name, tmp_path):
    """--storage f32 (opt-in, outside the reference's contract): the whole VAMP run equals the oracle's run on the matrix
    rounded to FP32, to the same 1e-9 — the mode changes the data that is held, not the arithmetic."""
    g = load_golden(name)
    A, y_txt, beta = golden_inputs(g)
    A32 = A.astype(np.float32).astype(np.float64)
    v = oracle_run(g, A32, y_txt, beta)
    model = g["model"]
    y = standardize_phen(y_txt) if model == "linear" else y_txt
    sh = capi.Shard(int(g["N"]), int(g["M"]), storage="f32")
    sh.upload(A)
    sh.compute_stats()
    kw = dict(gamw=2.0, seed=int(g["probe_seed"]))
    kw.update(extra_kwargs(g))
    if "h2" in kw:
        kw["gamw"] = 1.0 / (1.0 - kw.pop("h2"))              # src/main_meth.cpp:52
    sol = capi.Solver(sh, y, model=model, true_signal=beta, **kw)
    for k in range(1, int(g["iterations"]) + 1):
        r = sol.step()
        assert rel_l2(r["x1"], v.dump[k][0]) < 1e-9 and rel_l2(r["r1"], v.dump[k][1]) < 1e-9
    sol.close()
    sh.close()
    # and through the command line
    d = str(tmp_path)
    golden_inputs(g, d)
    os.makedirs(tmp_path / "out")
    run_cli(["--meth-file", f"{d}/ex.bin", "--phen-file", f"{d}/ex.phen", "--N", g["N"], "--Mt", g["M"], "--out-dir", f"{d}/out", "--out-name", "g",
             "--iterations", 3, "--true-signal-file", f"{d}/ex_ts.bin", "--model", model, "--stop-criteria-thr", "0", "--seed", g["probe_seed"],
             "--storage", "f32"] + list(g["extra"]))
    for k in range(1, 4):
        assert rel_l2(np.fromfile(f"{d}/out/g_it_{k}.bin"), v.dump[k][0]) < 1e-9


REF_BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "main_meth_ref")


def _ref_cg_counts(log):
    """(k1, k2) per VAMP iteration from the reference's --verbosity 1 log: '[CG] it' lines before / after the first
    '[CG onsager]' line of the iteration (src/vamp.cpp:723-724,747-748); see tests/tools/make_golden.py."""
    import re
    out = []
    for block in log.split("iteration = ")[1:]:
        lm, _, ons = block.partition("[CG onsager]")
        k1 = len(re.findall(r"\[CG\] it = ", lm))
        n = len(re.findall(r"\[CG\] it = ", ons))
        last = re.findall(r"\|\|r_it\|\| / \|\|RHS\|\| = ([0-9.e+-]+)", ons)
        out.append((k1, n if (last and float(last[-1]) < 1e-5) else n + 1))
    return out


@pytest.mark.parametrize("gpus", [1, 2])
def test_mid_size_run_matches_the_reference_binary_on_this_box(gpus, tmp_path):
    """bin/main_meth on mid-size files — N = 4 000, Mt = 20 000 (0.64 GB), --gam1 1e-2 — against the stored outputs of the
    reference for the SAME files (tests/golden/midsize_gam1e-2.npz, written by tests/tools/make_midsize_golden.py; its `source`
    says whether the reference binary or the numpy oracle produced it): 1e-9 on x1_hat / r1 of every iteration (at a seeded
    sample of markers, and on the full-vector norms), 1e-8 on the CSV values, CG iteration counts exact, CSV byte layout
    identical. Where the reference binary itself is present (oracle/_ref/main_meth_ref), the same run is also compared with a
    live run of it, whole vectors. With --gpus 2 all of this goes through the marker-sharded path."""
    if capi.device_count() < gpus:
        pytest.skip(f"needs {gpus} GPUs")
    import hashlib
    import re
    g = load_golden("midsize_gam1e-2")
    N, M, its, seed = int(g["N"]), int(g["M"]), int(g["iterations"]), int(g["probe_seed"])
    d = str(tmp_path)
    X, _, _ = sim.write_dataset(d, "mid", N, M, lam=float(g["lam"]), h2=float(g["h2"]), seed=int(g["data_seed"]))
    assert hashlib.sha256(X.tobytes()).hexdigest() == g["sha256_A"], "numpy generator drifted: regenerate the fixture"
    del X
    common = ["--meth-file", f"{d}/mid.bin", "--phen-file", f"{d}/mid.phen", "--N", N, "--Mt", M, "--out-name", "m", "--iterations", its,
              "--true-signal-file", f"{d}/mid_ts.bin", "--stop-criteria-thr", 0, "--gam1", g["gam1"]]
    os.makedirs(tmp_path / "gpu")
    out = run_cli(common + ["--out-dir", f"{d}/gpu", "--seed", seed, "--gpus", gpus], timeout=900)
    got_cg = [(int(a), int(b)) for a, b in re.findall(r"\[CG\] LMMSE solve: (\d+) iterations, onsager solve: (\d+)", out)]
    assert got_cg == [tuple(int(v) for v in c) for c in g["cg_iters"]], "CG iteration counts"
    idx = g["sample_index"]
    for k in range(1, its + 1):
        for key, f in (("x1", f"m_it_{k}.bin"), ("r1", f"m_r1_it_{k}.bin")):
            a = np.fromfile(f"{d}/gpu/{f}")
            assert a.size == M, f
            assert rel_l2(a[idx], g[key][k - 1]) < 1e-9, f
            assert abs(np.linalg.norm(a) - g[f"{key}_norm"][k - 1]) <= 1e-9 * g[f"{key}_norm"][k - 1], f
    def csvs_match(want_of):
        for kind in ("params", "metrics", "prior"):
            got, want = open(f"{d}/gpu/m_{kind}.csv", "rb").read(), want_of(kind)
            assert len(got) == len(want)
            assert np.array_equal(np.frombuffer(got, dtype=np.uint8) == 0, np.frombuffer(want, dtype=np.uint8) == 0), f"{kind}.csv NUL layout"
            if kind != "prior":
                assert_rows_close(csv_rows(got), csv_rows(want), 1e-8, kind)

    csvs_match(lambda kind: bytes(g[f"csv_{kind}"]))
    if not os.path.isfile(REF_BIN):
        return
    os.makedirs(tmp_path / "ref")
    ref = subprocess.run([REF_BIN] + [str(a) for a in common + ["--out-dir", f"{d}/ref", "--verbosity", 1]], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True, timeout=900, env=dict(os.environ, VAMPOMI_SEED=str(seed), OMP_NUM_THREADS=str(os.cpu_count() or 1)))
    assert ref.returncode == 0, ref.stdout[-2000:]
    assert got_cg == _ref_cg_counts(ref.stdout), "CG iteration counts"
    for k in range(1, its + 1):
        for f in (f"m_it_{k}.bin", f"m_r1_it_{k}.bin"):
            assert rel_l2(np.fromfile(f"{d}/gpu/{f}"), np.fromfile(f"{d}/ref/{f}")) < 1e-9, f
    csvs_match(lambda kind: open(f"{d}/ref/m_{kind}.csv", "rb").read())


def test_main_meth_probit_entry_point(tmp_path):
    """bin/main_meth_probit (BASELINE.json configuration 4; src/main_meth_probit.cpp): the probit model without --model on the
    command line, that driver's `test` run mode (confusion-matrix rows, no header, :104-200) and its `predict` mode (:201-227)."""
    g = load_golden("probit_small")
    d = str(tmp_path)
    A, y_txt, beta = golden_inputs(g, d)
    os.makedirs(tmp_path / "out")
    its, N, M = 3, int(g["N"]), int(g["M"])
    exe = build.MAIN_METH_PROBIT

    def run(args):
        res = subprocess.run([exe] + [str(a) for a in args], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert res.returncode == 0, res.stdout[-3000:]
        return res.stdout

    out = run(["--meth-file", f"{d}/ex.bin", "--phen-file", f"{d}/ex.phen", "--N", N, "--Mt", M, "--out-dir", f"{d}/out", "--out-name", "g",
               "--iterations", its, "--true-signal-file", f"{d}/ex_ts.bin", "--stop-criteria-thr", 0, "--seed", g["probe_seed"]] + list(g["extra"]))
    assert "--model" not in out.split("ardyh command line options:")[1].split("INFO")[0]
    for k in range(1, its + 1):
        assert rel_l2(np.fromfile(f"{d}/out/g_it_{k}.bin"), g["x1"][k - 1]) < 1e-9
        assert rel_l2(np.fromfile(f"{d}/out/g_r1_it_{k}.bin"), g["r1"][k - 1]) < 1e-9
    want = csv_rows(g["csv_params"])
    got = csv_rows(open(f"{d}/out/g_params.csv", "rb").read())
    assert_rows_close(got, {k: want[k] for k in range(1, its + 1)}, 1e-8, "params")
    # probit test mode on an independent draw
    Nt = 150
    Xt, yt, _ = sim.write_dataset(d, "tst", Nt, M, float(g["lam"]), float(g["h2"]), int(g["data_seed"]) + 1000, binary=True)
    run(["--meth-file-test", f"{d}/tst.bin", "--phen-file-test", f"{d}/tst.phen", "--N-test", Nt, "--Mt", M, "--out-dir", f"{d}/out", "--out-name", "g",
         "--run-mode", "test", "--estimate-file", f"{d}/out/g_it_1.bin", "--test-iter-range", f"1,{its}"])
    blob = open(f"{d}/out/g_test.csv", "rb").read()
    rows = csv_rows(blob)
    yt_txt = np.array([float("%0.10f" % v) for v in yt])
    dt = vo.Data(Xt, yt_txt)
    assert set(blob[:len(vo.csv_row(1, [0.0] * 5))]) == {0}                 # no header: the first row-length bytes are a hole
    for k in range(1, its + 1):
        z = dt.Ax(np.fromfile(f"{d}/out/g_it_{k}.bin") * math.sqrt(Nt))
        yhat = (z >= 0).astype(float)                                        # normal_cdf(z) >= 0.5
        TP, TN = int(((yt_txt == 1) & (yhat == 1)).sum()), int(((yt_txt == 0) & (yhat == 0)).sum())
        FP, FN = int(((yt_txt == 0) & (yhat == 1)).sum()), int(((yt_txt == 1) & (yhat == 0)).sum())
        assert rows[k][:4] == [TP, TN, FP, FN] and abs(rows[k][4] - (TP + TN) / Nt) < 1e-14
    run(["--meth-file-test", f"{d}/tst.bin", "--phen-file-test", f"{d}/tst.phen", "--N-test", Nt, "--Mt", M, "--out-dir", f"{d}/out", "--out-name", "g",
         "--run-mode", "predict", "--estimate-file", f"{d}/out/g_it_{its}.bin"])
    zhat = np.loadtxt(f"{d}/out/g_.yhat")
    assert zhat.shape == (Nt,) and np.allclose(zhat, dt.Ax(np.fromfile(f"{d}/out/g_it_{its}.bin") * math.sqrt(Nt)), rtol=2e-5, atol=1e-8)
    # main_meth itself still refuses the probit-only run mode quietly (the reference's main does nothing for unknown modes)
    res = subprocess.run([exe, "--meth-file", "x", "--N", "5"], stdout=subprocess.PIPE, text=True)
    assert res.returncode == 1 and "FATAL" in res.stdout


@pytest.mark.parametrize("name", ["linear_cov", "probit_cov"])
def test_main_meth_covariates_flags(name, tmp_path):
    """--C / --cov-file through the command line (src/options.cpp:30-38,226; data::read_covariates; Newton_method_cov): the files of
    the covariate fixtures, and the reference's FATAL for a covariate count that does not match."""
    g = load_golden(name)
    d = str(tmp_path)
    golden_inputs(g, d)
    os.makedirs(tmp_path / "out")
    its = int(g["iterations"])
    args = ["--meth-file", f"{d}/ex.bin", "--phen-file", f"{d}/ex.phen", "--N", g["N"], "--Mt", g["M"], "--out-dir", f"{d}/out", "--out-name", "g",
            "--iterations", its, "--true-signal-file", f"{d}/ex_ts.bin", "--model", g["model"], "--stop-criteria-thr", 0, "--seed", g["probe_seed"],
            "--cov-file", f"{d}/ex.cov"] + list(g["extra"])
    out = run_cli(args + ["--C", g["C"]])
    effs = [float(v) for v in __import__("re").findall(r"cov_eff\[\d+\] = ([-+0-9.eE]+)", out)][:int(g["C"])]
    assert np.allclose(effs, g["cov_eff"], rtol=2e-5, atol=1e-9)
    for k in range(1, its + 1):
        assert rel_l2(np.fromfile(f"{d}/out/g_it_{k}.bin"), g["x1"][k - 1]) < 1e-9
        assert rel_l2(np.fromfile(f"{d}/out/g_r1_it_{k}.bin"), g["r1"][k - 1]) < 1e-9
    for kind in ("params", "metrics"):
        assert_rows_close(csv_rows(open(f"{d}/out/g_{kind}.csv", "rb").read()), csv_rows(g[f"csv_{kind}"]), 1e-8, kind)
    res = subprocess.run([build.MAIN_METH] + [str(a) for a in args + ["--C", int(g["C"]) + 1]], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 1 and "does not match to the specified number of covariates" in res.stdout


@pytest.mark.parametrize("name,schedule", [("linear_wellcond", "onepass"), ("linear_wellcond", "plain"), ("probit_small", "onepass"),
                                           ("linear_cov", "recycled"), ("probit_cov", "fused")])
def test_checkpoint_and_resume_continue_the_same_run(name, schedule, tmp_path):
    """vampomi_solver_save_state / _load_state (SURVEY.md §8 f2): a run stopped after iteration 3 and resumed in a NEW context
    continues with the iterates, CSV values and CG counts of the uninterrupted run."""
    g = load_golden(name)
    A, y_txt, beta = golden_inputs(g)
    its = int(g["iterations"])
    sh, sol = solver_for(g, A, y_txt, beta, **SCHEDULES[schedule])
    full = [sol.step() for _ in range(its)]
    sol.close(); sh.close()
    stop = 2 if its <= 4 else 3
    sh, sol = solver_for(g, A, y_txt, beta, **SCHEDULES[schedule])
    for _ in range(stop):
        sol.step()
    ck = str(tmp_path / "ck.bin")
    sol.save_state(ck)
    sol.close(); sh.close()
    sh, sol = solver_for(g, A, y_txt, beta, **SCHEDULES[schedule])
    torn = bytearray(open(ck, "rb").read())                                       # a writer that died before its completion record
    torn[2048:2048 + 24] = bytes(24)
    open(tmp_path / "torn.bin", "wb").write(torn)
    with pytest.raises(capi.VampomiError):
        sol.load_state(str(tmp_path / "torn.bin"))
    sol.load_state(ck)                                                            # a refused checkpoint leaves the solver untouched
    for k in range(stop, its):
        r = sol.step()
        assert r["it"] == k + 1 and (r["k1"], r["k2"]) == (full[k]["k1"], full[k]["k2"])
        assert rel_l2(r["x1"], full[k]["x1"]) < 1e-11 and rel_l2(r["r1"], full[k]["r1"]) < 1e-11, k
        assert np.allclose(r["params"], full[k]["params"], rtol=1e-10, atol=1e-300) and np.allclose(r["metrics"], full[k]["metrics"], rtol=1e-10, equal_nan=True)
        assert rel_l2(r["x1"], g["x1"][k]) < 1e-9                                 # and, with that, the reference's
    with pytest.raises(capi.VampomiError):
        sol.load_state(ck)                                                        # only a freshly created solver can be restored
    sol.close(); sh.close()
    sh2 = capi.Shard(int(g["N"]), int(g["M"]) - 1)
    sh2.upload(A[:-1]); sh2.compute_stats()
    other = capi.Solver(sh2, standardize_phen(y_txt) if g["model"] == "linear" else y_txt, model=g["model"])
    with pytest.raises(capi.VampomiError):
        other.load_state(ck)                                                      # written for another problem
    other.close(); sh2.close()


def test_main_meth_checkpoint_every_and_resume_from(tmp_path):
    g = load_golden("linear_wellcond")
    d = str(tmp_path)
    golden_inputs(g, d)
    os.makedirs(tmp_path / "out")
    its = int(g["iterations"])
    base = ["--meth-file", f"{d}/ex.bin", "--phen-file", f"{d}/ex.phen", "--N", g["N"], "--Mt", g["M"], "--out-dir", f"{d}/out", "--out-name", "g",
            "--true-signal-file", f"{d}/ex_ts.bin", "--stop-criteria-thr", 0, "--seed", g["probe_seed"]] + list(g["extra"])
    out = run_cli(base + ["--iterations", 4, "--checkpoint-every", 2])
    assert os.path.isfile(f"{d}/out/g_checkpoint_it_2.bin") and os.path.isfile(f"{d}/out/g_checkpoint_it_4.bin") and "--checkpoint-every 2" in out
    size4 = os.path.getsize(f"{d}/out/g_params.csv")
    out = run_cli(base + ["--iterations", its, "--resume-from", f"{d}/out/g_checkpoint_it_4.bin"])
    assert "resuming after iteration 4" in out and "iteration = 5" in out and "iteration = 4\n" not in out
    assert os.path.getsize(f"{d}/out/g_params.csv") > size4
    for k in range(1, its + 1):
        assert rel_l2(np.fromfile(f"{d}/out/g_it_{k}.bin"), g["x1"][k - 1]) < 1e-9
        assert rel_l2(np.fromfile(f"{d}/out/g_r1_it_{k}.bin"), g["r1"][k - 1]) < 1e-9
    for kind in ("params", "metrics"):
        got = open(f"{d}/out/g_{kind}.csv", "rb").read()
        assert len(got) == len(bytes(g[f"csv_{kind}"]))
        assert_rows_close(csv_rows(got), csv_rows(g[f"csv_{kind}"]), 1e-8, kind)
    res = subprocess.run([build.MAIN_METH] + [str(a) for a in base + ["--iterations", its, "--resume-from", f"{d}/out/nothing.bin"]],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 1 and "could not resume" in res.stdout


def test_several_hutchinson_probes_average_the_single_probe_estimates():
    """cfg.probes = P (SURVEY.md §8 f2; not in the reference): alpha2 = gam2 * mean over P probes of u^T Q^-1 u, with the probes of
    the counter hash under seeds seed + p * golden ratio; P = 1 is the reference-parity run."""
    g = load_golden("linear_wellcond")
    A, y_txt, beta = golden_inputs(g)
    seed = int(g["probe_seed"])
    sh, sol = solver_for(g, A, y_txt, beta, probes=3)
    r = sol.step()
    alpha2, gam2 = r["params"][2], r["params"][3]
    vm = []
    for p in range(3):
        sh.draw_probe((seed + 0x9E3779B97F4A7C15 * p) % 2 ** 64, 1)
        _, _, vmu = sh.cg_solve(capi.V_BERN, V_QINV_BERN, sol.cfg.gamw, gam2, tol=1e-5, onsager_mode=True)
        vm.append(vmu)
    assert abs(alpha2 - gam2 * np.mean(vm)) < 1e-12 * alpha2 and len(set(vm)) == 3
    r2 = sol.step()
    assert 0 < r2["params"][2] < 1 and np.isfinite(r2["x1"]).all()
    sol.close(); sh.close()
    sh, sol = solver_for(g, A, y_txt, beta, probes=3)
    rr = sol.step()
    assert rr["params"] == r["params"]                                            # reproducible
    sol.close(); sh.close()
    gp = load_golden("probit_small")
    Ap, yp, bp = golden_inputs(gp)
    sh, sol = solver_for(gp, Ap, yp, bp, probes=2)
    r = sol.step(); r = sol.step()
    assert 0 < r["params"][4] < 1 and np.isfinite(r["r1"]).all()
    sol.close(); sh.close()
