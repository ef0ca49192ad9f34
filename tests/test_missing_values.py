"""--missing mean / vampomi_impute_missing: every NaN of a marker column is replaced, in HBM, by the mean of the column's other
entries before the marker statistics are computed, so a run on a matrix with NaNs is the run on the imputed matrix. The kernel
is checked against a numpy restatement, the VAMP loop against the oracle on the imputed matrix, and the command line against
a plain run on the imputed file, byte for byte. The CPU tests of this file need no GPU; the others are marked one by one."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from vampomi_b200 import build, capi, sim
from helpers import assert_rows_close, csv_rows, extra_kwargs, golden_inputs, load_golden, oracle_run, rel_l2, standardize_phen, tolerances

NEG_NAN = np.array([0xFFF8000000000001], dtype=np.uint64).view(np.float64)[0]      # sign bit set, non-zero payload


# ---- CPU ---------------------------------------------------------------------------------------------------------------------
def test_missing_flag_is_validated_and_echoed_before_any_gpu_work(lib):
    for argv in (["--missing", "foo"], ["--meth-file", "x", "--missing", "NaN"], ["--missing"]):
        res = subprocess.run([build.MAIN_METH] + argv, stdout=subprocess.PIPE, text=True)
        assert res.returncode == 1 and "FATAL" in res.stdout, argv
    res = subprocess.run([build.MAIN_METH, "--missing", "foo"], stdout=subprocess.PIPE, text=True)
    assert "--missing has to be none or mean" in res.stdout
    for value in ("mean", "none"):                 # --N / --Mt missing: stops after the echo, before any GPU work
        res = subprocess.run([build.MAIN_METH, "--meth-file", "x", "--phen-file", "y", "--missing", value], stdout=subprocess.PIPE, text=True)
        assert res.returncode == 1 and f"--missing {value}" in res.stdout


def test_impute_missing_rejects_null_arguments(lib):
    counts = (C.c_longlong * 3)()
    assert lib.vampomi_impute_missing(None, counts) == 1
    assert "impute_missing" in capi.last_error()
    assert lib.vampomi_impute_missing(None, None) == 1


# ---- numpy restatement -------------------------------------------------------------------------------------------------------
def kernel_order_sum(x, VE):
    """Sum of the non-NaN entries of one column in the kernel's order: lane l of the column's warp adds the 32-byte pieces
    l, l + 32, ... (VE values each, value e into accumulator e % 4), then the scalar tail rows nvec*VE + l, + 32, ...
    into accumulator 0; (s0 + s1) + (s2 + s3) per lane, then the xor-butterfly over the 32 lanes."""
    x = [0.0 if np.isnan(v) else float(v) for v in x]
    N, nvec = len(x), len(x) // VE
    lanes = np.zeros(32)
    for lane in range(32):
        s = [0.0] * 4
        for v in range(lane, nvec, 32):
            for e in range(VE):
                s[e & 3] += x[VE * v + e]
        for i in range(nvec * VE + lane, N, 32):
            s[0] += x[i]
        lanes[lane] = (s[0] + s[1]) + (s[2] + s[3])
    for o in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[np.arange(32) ^ o]
    return float(lanes[0])


def impute_ref(X, storage="f64"):
    """(imputed copy, [entries replaced, columns with a NaN, columns without an observed value]) of a marker-major block:
    each NaN becomes the column's nanmean (exactly the observed value when all observed values are equal), 0 for a column
    without observed values. FP32 storage: X is the block as held (rounded when uploaded) and the mean is rounded to FP32
    too. The mean is summed in the kernel's order, so the comparison does not depend on how much the column's sum cancels."""
    out = X.copy()
    miss = np.isnan(X)
    for j in np.nonzero(miss.any(axis=1))[0]:
        nobs = int((~miss[j]).sum())
        obs = X[j][~miss[j]]
        m = kernel_order_sum(X[j], 8 if storage == "f32" else 4) / nobs if nobs else 0.0
        if nobs and obs.min() == obs.max():
            m = obs[0]                               # all observed values equal: exactly that value
        elif nobs:
            assert not np.isfinite(m) or abs(m - np.nanmean(X[j])) <= 1e-12 * np.nanmean(np.abs(X[j]))
        out[j, miss[j]] = np.float32(m) if storage == "f32" else m
    return out, [int(miss.sum()), int(miss.any(axis=1).sum()), int(miss.all(axis=1).sum())]


def seeded_block(N, M, seed):
    """A (M, N) block with the awkward cases in its first columns and 5 % random NaNs in the rest."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((M, N))
    X[0, 0] = np.nan                                 # one NaN
    X[1, :] = np.nan                                 # no observed value
    X[2, :] = np.nan                                 # one observed value
    X[2, N // 2] = 1.25
    X[3, N - 1] = np.nan                             # last row of a ragged N (the scalar tail of the kernel)
    X[4, N - 1] = NEG_NAN                            # negative NaN with a payload
    X[5, 0] = np.inf                                 # +Inf is observed: the mean, and so the fill, is +Inf
    X[5, N - 1] = np.nan
    X[6, N // 2] = -np.inf                           # -Inf in a column without NaN: untouched
    X[8, :] = np.nan                                 # one observed value that does not sum exactly: 0.1 / 1 = 0.1, but the
    X[8, N // 3] = 0.1                               # mean of a constant column must not depend on how it is summed
    X[9, :] = 0.7                                    # all observed values equal (0.7 + 0.7 + ... can miss 0.7 * n by an ulp)
    X[9, ::3] = np.nan
    mask = rng.random((M - 10, N)) < 0.05            # column 7 has no NaN
    X[10:][mask] = np.nan
    return X


@pytest.mark.gpu
@pytest.mark.parametrize("storage", ["f64", "f32"])
@pytest.mark.parametrize("N", [2, 37, 1000, 4099])     # N = 1 is refused by vampomi_create (a column needs two samples)
def test_impute_kernel_matches_numpy(storage, N):
    M = 45
    X = seeded_block(N, M, seed=N)
    held = X.astype(np.float32).astype(np.float64) if storage == "f32" else X
    want, want_counts = impute_ref(held, storage)
    miss = np.isnan(held)
    with capi.Shard(N, M, storage=storage) as sh:
        sh.upload(X)
        assert list(sh.impute_missing()) == want_counts
        got = sh.download()
        assert not np.isnan(got).any()
        assert np.array_equal(got.view(np.uint64)[~miss], held.view(np.uint64)[~miss])     # observed entries bitwise unchanged
        np.testing.assert_allclose(got[miss], want[miss], rtol=1e-14, atol=0)
        assert got[5, 0] == np.inf and got[5, N - 1] == np.inf and got[6, N // 2] == -np.inf
        assert np.all(got[1] == 0.0) and np.all(got[2] == 1.25)
        # a second call finds nothing to replace and writes nothing
        assert sh.impute_missing() == (0, 0, 0)
        assert np.array_equal(sh.download().view(np.uint64), got.view(np.uint64))
        # the statistics are those of the imputed block; the column without observed values is constant (msig = 1)
        sh.compute_stats()
        mave, msig = sh.stats()
        finite = np.isfinite(want).all(axis=1)
        np.testing.assert_allclose(mave[finite], want[finite].mean(axis=1), rtol=1e-12, atol=1e-13)
        assert mave[1] == 0.0 and msig[1] == 1.0
        for j, c in ((2, 1.25), (8, 0.1), (9, 0.7)):  # imputed columns that are constant: their value and msig = 1, exactly
            c = float(np.float32(c)) if storage == "f32" else c
            assert np.all(got[j] == c) and mave[j] == c and msig[j] == 1.0, (j, mave[j], msig[j])
        const = (want.min(axis=1) == want.max(axis=1)) & finite
        assert np.all(msig[const] == 1.0)
        if N > 2:
            sd = want[finite & ~const].std(axis=1, ddof=1)
            np.testing.assert_allclose(msig[finite & ~const], 1.0 / sd, rtol=1e-11)


@pytest.mark.gpu
@pytest.mark.parametrize("storage", ["f64", "f32"])
def test_block_without_nan_is_left_bitwise_unchanged(storage):
    N, M = 1003, 64
    X = np.random.default_rng(4).standard_normal((M, N))
    X[3, 7] = np.inf
    X[9, 1002] = -np.inf
    with capi.Shard(N, M, storage=storage) as sh:
        sh.upload(X)
        before = sh.download()
        assert sh.impute_missing() == (0, 0, 0)
        assert np.array_equal(sh.download().view(np.uint64), before.view(np.uint64))


@pytest.mark.gpu
def test_imputing_invalidates_the_statistics():
    N, M = 200, 30
    X = seeded_block(N, M, seed=1)
    p = np.ones(N)
    out = np.empty(M)
    with capi.Shard(N, M) as sh:
        sh.upload(X)
        sh.compute_stats()                            # statistics of the block with NaNs: valid as far as the library knows
        sh.impute_missing()
        rc = sh.lib.vampomi_atx(sh.h, p.ctypes.data_as(capi.c_double_p), out.ctypes.data_as(capi.c_double_p))
        assert rc == 5, capi.last_error()             # VAMPOMI_ERR_STATE: ATx before compute_stats
        sh.compute_stats()
        assert np.isfinite(sh.ATx(p)[7:]).all()       # column 5 holds +Inf, column 6 -Inf


# ---- VAMP on the imputed matrix ----------------------------------------------------------------------------------------------
def with_nans(A, frac=0.03, seed=17):
    A = A.copy()
    A[np.random.default_rng(seed).random(A.shape) < frac] = np.nan
    return A


@pytest.mark.gpu
@pytest.mark.parametrize("name,storage", [("linear_ragged", "f64"), ("linear_wellcond", "f64"), ("probit_small", "f64"),
                                          ("linear_wellcond", "f32")])
def test_vamp_on_imputed_matrix_matches_oracle(name, storage):
    """upload -> impute -> statistics -> VAMP equals the oracle run on the imputed matrix (as downloaded from the GPU)."""
    g = load_golden(name)
    rel_vec, _ = tolerances(g)
    A, y_txt, beta = golden_inputs(g)
    An = with_nans(A)
    model = g["model"]
    y = standardize_phen(y_txt) if model == "linear" else y_txt
    kw = dict(gamw=2.0, seed=int(g["probe_seed"]))
    kw.update(extra_kwargs(g))
    if "h2" in kw:
        kw["gamw"] = 1.0 / (1.0 - kw.pop("h2"))              # src/main_meth.cpp:52
    with capi.Shard(int(g["N"]), int(g["M"]), storage=storage) as sh:
        sh.upload(An)
        replaced, cols, empty = sh.impute_missing()
        assert replaced == int(np.isnan(An).sum()) and cols == int(np.isnan(An).any(axis=1).sum()) and empty == 0
        Ai = sh.download()
        assert not np.isnan(Ai).any()
        v = oracle_run(g, Ai, y_txt, beta)
        sh.compute_stats(kw.pop("alpha_scale", 1.0))
        sol = capi.Solver(sh, y, model=model, true_signal=beta, x1hat_init=g.get("x1hat_init"), **kw)
        for k in range(1, int(g["iterations"]) + 1):
            r = sol.step()
            assert rel_l2(r["x1"], v.dump[k][0]) < rel_vec, f"x1_hat it {k}"
            assert rel_l2(r["r1"], v.dump[k][1]) < rel_vec, f"r1 it {k}"
        sol.close()


# ---- command line ------------------------------------------------------------------------------------------------------------
def run_cli(args, exe=None, **kw):
    res = subprocess.run([exe or build.MAIN_METH] + [str(a) for a in args], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                         timeout=600, **kw)
    assert res.returncode == 0, res.stdout[-3000:]
    return res.stdout


def imputed_file(src, dst, N, Mt):
    """Writes the block of `src` as imputed by the GPU (FP64 storage) to `dst`."""
    with capi.Shard(N, Mt) as sh:
        sh.load_file(src)
        sh.impute_missing()
        sh.download().tofile(dst)


def assert_same_files(a, b):
    names = sorted(os.listdir(a))
    assert names and names == sorted(os.listdir(b))
    for f in names:
        assert open(os.path.join(a, f), "rb").read() == open(os.path.join(b, f), "rb").read(), f


def nan_inputs(g, d):
    """The fixture's files under d, with 3 % NaNs in ex.bin (nan.bin) and the GPU-imputed block of it (imp.bin)."""
    A, _, _ = golden_inputs(g, d)
    with_nans(A).tofile(f"{d}/nan.bin")
    imputed_file(f"{d}/nan.bin", f"{d}/imp.bin", int(g["N"]), int(g["M"]))
    return A


@pytest.mark.gpu
@pytest.mark.parametrize("name,exe", [("linear_wellcond", "main_meth"), ("probit_small", "main_meth_probit")])
def test_infere_with_missing_mean_equals_run_on_imputed_file(name, exe, tmp_path):
    g = load_golden(name)
    d = str(tmp_path)
    nan_inputs(g, d)
    exe = build.MAIN_METH if exe == "main_meth" else build.MAIN_METH_PROBIT
    common = ["--phen-file", f"{d}/ex.phen", "--N", g["N"], "--Mt", g["M"], "--out-name", "g", "--iterations", 4,
              "--true-signal-file", f"{d}/ex_ts.bin", "--stop-criteria-thr", 0, "--seed", g["probe_seed"]] + list(g["extra"])
    if exe == build.MAIN_METH:
        common += ["--model", g["model"]]
    for sub in ("a", "b"):
        os.makedirs(f"{d}/{sub}")
    out_a = run_cli(common + ["--meth-file", f"{d}/nan.bin", "--out-dir", f"{d}/a", "--missing", "mean"], exe=exe)
    out_b = run_cli(common + ["--meth-file", f"{d}/imp.bin", "--out-dir", f"{d}/b"], exe=exe)
    assert "--missing mean" in out_a and "INFO  : rank 0 replaced" in out_a and "imputing missing values took" in out_a
    assert "replaced" not in out_b and "imputing" not in out_b
    assert_same_files(f"{d}/a", f"{d}/b")


@pytest.mark.gpu
def test_association_and_test_modes_with_missing_mean(tmp_path):
    g = load_golden("linear_small")
    d = str(tmp_path)
    nan_inputs(g, d)
    N, M, last = int(g["N"]), int(g["M"]), int(g["iterations"])
    os.makedirs(f"{d}/est")
    for k in range(1, last + 1):
        g["x1"][k - 1].tofile(f"{d}/est/g_it_{k}.bin")
        g["r1"][k - 1].tofile(f"{d}/est/g_r1_it_{k}.bin")
    Nt = int(g["N_test"])
    Xt, _, _ = sim.write_dataset(d, "tst", Nt, M, float(g["lam"]), float(g["h2"]), int(g["data_seed"]) + 1000)
    with_nans(Xt, seed=23).tofile(f"{d}/tst_nan.bin")
    imputed_file(f"{d}/tst_nan.bin", f"{d}/tst_imp.bin", Nt, M)
    runs = {
        "se": ["--phen-file", f"{d}/ex.phen", "--N", N, "--run-mode", "association_test", "--pval-method", "se",
               "--r1-file", f"{d}/est/g_r1_it_{last}.bin", "--gam1", repr(float(g["se_gam1"]))],
        "loo": ["--phen-file", f"{d}/ex.phen", "--N", N, "--run-mode", "association_test", "--pval-method", "loo",
                "--estimate-file", f"{d}/est/g_it_{last}.bin"],
        "test": ["--phen-file-test", f"{d}/tst.phen", "--N-test", Nt, "--run-mode", "test", "--estimate-file", f"{d}/est/g_it_1.bin",
                 "--test-iter-range", f"1,{last}"],
    }
    for mode, args in runs.items():
        meth = "--meth-file-test" if mode == "test" else "--meth-file"
        nan, imp = (f"{d}/tst_nan.bin", f"{d}/tst_imp.bin") if mode == "test" else (f"{d}/nan.bin", f"{d}/imp.bin")
        for sub in ("a", "b"):
            os.makedirs(f"{d}/{mode}_{sub}")
        common = args + ["--Mt", M, "--out-name", "g"]
        run_cli(common + [meth, nan, "--out-dir", f"{d}/{mode}_a", "--missing", "mean"])
        run_cli(common + [meth, imp, "--out-dir", f"{d}/{mode}_b"])
        assert_same_files(f"{d}/{mode}_a", f"{d}/{mode}_b")
    # the loo p-values see the imputed raw columns: they differ from those of the matrix without NaNs
    os.makedirs(f"{d}/loo_c")
    run_cli(runs["loo"] + ["--Mt", M, "--out-name", "g", "--meth-file", f"{d}/ex.bin", "--out-dir", f"{d}/loo_c"])
    a = np.fromfile(f"{d}/loo_a/g_it_{last}_pval_loo.bin")
    assert not np.array_equal(a, np.fromfile(f"{d}/loo_c/g_it_{last}_pval_loo.bin"))


@pytest.mark.gpu
def test_missing_mean_on_a_file_without_nan_changes_nothing(tmp_path):
    g = load_golden("linear_wellcond")
    d = str(tmp_path)
    golden_inputs(g, d)
    common = ["--meth-file", f"{d}/ex.bin", "--phen-file", f"{d}/ex.phen", "--N", g["N"], "--Mt", g["M"], "--out-name", "g",
              "--iterations", 4, "--true-signal-file", f"{d}/ex_ts.bin", "--stop-criteria-thr", 0, "--seed", g["probe_seed"]] + list(g["extra"])
    for sub in ("a", "b"):
        os.makedirs(f"{d}/{sub}")
    out_a = run_cli(common + ["--out-dir", f"{d}/a", "--missing", "mean"])
    run_cli(common + ["--out-dir", f"{d}/b"])
    assert "INFO  : rank 0 replaced 0 missing values" in out_a
    assert_same_files(f"{d}/a", f"{d}/b")


@pytest.mark.gpu
def test_missing_mean_is_shard_invariant(tmp_path):
    if capi.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    g = load_golden("linear_wellcond")
    rel_vec, rel_csv = tolerances(g)
    d = str(tmp_path)
    A = nan_inputs(g, d)
    its = int(g["iterations"])
    common = ["--meth-file", f"{d}/nan.bin", "--phen-file", f"{d}/ex.phen", "--N", g["N"], "--Mt", g["M"], "--out-name", "g", "--iterations", its,
              "--true-signal-file", f"{d}/ex_ts.bin", "--stop-criteria-thr", 0, "--seed", g["probe_seed"], "--missing", "mean"] + list(g["extra"])
    outs = {}
    for gpus in (1, 2):
        os.makedirs(f"{d}/g{gpus}")
        outs[gpus] = run_cli(common + ["--out-dir", f"{d}/g{gpus}", "--gpus", gpus])
    total = int(np.isnan(with_nans(A)).sum())
    for gpus, out in outs.items():
        counts = [int(l.split("replaced ")[1].split()[0]) for l in out.splitlines() if " replaced " in l]
        assert len(counts) == gpus and sum(counts) == total
    for k in range(1, its + 1):
        for f in (f"g_it_{k}.bin", f"g_r1_it_{k}.bin"):
            assert rel_l2(np.fromfile(f"{d}/g2/{f}"), np.fromfile(f"{d}/g1/{f}")) < rel_vec, f
    for kind in ("params", "metrics"):
        assert_rows_close(csv_rows(open(f"{d}/g2/g_{kind}.csv", "rb").read()), csv_rows(open(f"{d}/g1/g_{kind}.csv", "rb").read()), rel_csv, kind)
