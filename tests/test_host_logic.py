"""Host-side logic of the C++ driver, checked without a GPU against the oracle (which is pinned to the reference
binary's outputs): CSV row formatting incl. non-finite values, phenotype reader, Student-t p-values, the counter hash
that replaces std::random_device, and the mixture-component merge."""
import ctypes as C
import math

import mpmath
import numpy as np
import pytest
from scipy import stats as spstats

from oracle import vamp_oracle as vo
from vampomi_b200 import capi

c_double_p = C.POINTER(C.c_double)


def arr(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(c_double_p)


@pytest.mark.parametrize("values", [[0.0] * 5, [1.5, -2.25e-7, 123456.789, 1e11, 1e-11, 3.0], [float("nan"), -float("nan"), float("inf"), -float("inf")],
                                    [1e22, -1e22, 0.1], []])
def test_csv_row_bytes_match_reference_format(lib, values):
    buf = C.create_string_buffer(4096)
    a, pa = arr(values) if values else (None, None)
    for it in (1, 7, 12345, 123456):
        n = lib.vampomi_host_csv_row(it, pa, len(values), buf, 4096)
        got = buf.raw[:n].decode()
        assert got == vo.csv_row(it, values)          # the oracle's formatter is held to the reference's CSV bytes
        assert n == len(got)
    # 0.0/0.0 as x86 produces it (sign bit set) prints "-nan", as in row 1 of the reference's _metrics.csv
    with np.errstate(all="ignore"):
        neg_nan = np.float64(0.0) / np.float64(0.0)
    a, pa = arr([neg_nan])
    n = lib.vampomi_host_csv_row(1, pa, 1, buf, 4096)
    assert buf.raw[:n].decode() == vo.csv_row(1, [neg_nan])


def test_read_phen_matches_oracle(lib, tmp_path):
    rng = np.random.default_rng(0)
    y = rng.standard_normal(257) * 3 + 1
    p = tmp_path / "a.phen"
    with open(p, "w") as f:
        for i, v in enumerate(y):
            sep = "\t" if i % 3 == 0 else "  "
            f.write(f"{i}{sep}{i} {v:0.10f}\n")
    out, po = arr(np.zeros(300))
    for std in (1, 0):
        n = lib.vampomi_host_read_phen(str(p).encode(), std, po, 300)
        assert n == 257
        want = vo.read_phen(str(p), standardize=bool(std))
        assert np.allclose(out[:n], want, rtol=1e-15, atol=0)
    if True:   # scaled, not centred (src/data.cpp:97-99)
        lib.vampomi_host_read_phen(str(p).encode(), 1, po, 300)
        assert abs(out[:257].std(ddof=1) - 1) < 1e-12 and abs(out[:257].mean()) > 0.1
    assert lib.vampomi_host_read_phen(b"/nonexistent/file.phen", 1, po, 300) == -1
    with open(p, "a") as f:
        f.write("9 9 NA\n")
    assert lib.vampomi_host_read_phen(str(p).encode(), 1, po, 300) == -2


def test_students_t_pvalues_match_scipy(lib):
    rng = np.random.default_rng(1)
    for n in (10, 300, 20000):
        x = rng.standard_normal(n)
        for slope in (0.0, 0.05, 0.5, 5.0):
            yv = slope * x + rng.standard_normal(n)
            got = lib.vampomi_host_linear_reg1d_pvals(x.sum(), (x * x).sum(), (x * yv).sum(), yv.sum(), (yv * yv).sum(), n)
            want = vo.linear_reg1d_pvals(x.sum(), (x * x).sum(), (x * yv).sum(), yv.sum(), (yv * yv).sum(), n)
            assert got == pytest.approx(want, rel=1e-9, abs=1e-300)


def host_t(sumx, sumsqx, sumxy, sumy, sumsqy, n):
    """The t statistic of host/io.cpp linear_reg1d_pvals, operation by operation in FP64 (the host is built without FP
    contraction, so these are the same roundings); None where the host returns 1 without a t."""
    s2y = (sumsqy - sumy * sumy / n) / (n - 1)
    s2x = (sumsqx - sumx * sumx / n) / (n - 1)
    sxy = (sumxy - sumx * sumy / n) / (n - 1)
    if s2x <= 0 or s2y <= 0 or s2x * s2y == 0:
        return None
    r = min(1.0, max(-1.0, sxy / math.sqrt(s2x * s2y)))
    return abs(r * math.sqrt((n - 2) / (1 - r * r))) if abs(r) < 1 else math.inf


def t_tail(t, dof):
    """2 P(T_dof > |t|) = I_{dof/(dof+t^2)}(dof/2, 1/2), in mpmath (40 digits)."""
    with mpmath.workdps(40):
        t = mpmath.mpf(t)
        return mpmath.betainc(mpmath.mpf(dof) / 2, mpmath.mpf(1) / 2, 0, dof / (dof + t * t), regularized=True)


def test_students_t_tail_against_mpmath(lib):
    """The host's Student-t tail (regularised incomplete beta by a continued fraction, DLMF 8.17.22, with lgamma differences) for
    dof 2 ... 19 998 and p from ~1 down to 1e-300, relative to mpmath at the t the host itself computed. Measured on this
    implementation: <= 1.7e-11 at dof 3 998 and <= 8e-11 at dof 19 998 (worst near p = 1, <= 5e-12 for p < 0.05); the bound is
    1e-10. The sums are chosen so that s2x = s2y = 1 and r = sxy, i.e. t = r sqrt((n-2)/(1-r^2)) for a target t."""
    checked = 0
    for dof in (2, 3, 8, 30, 98, 398, 3998, 19998):
        n = dof + 2
        for t in (0.0, 1e-3, 0.01, 0.5, 1.0, 2.0, 3.0, 5.0, 8.0, 12.0, 20.0, 37.0, 40.0, 100.0, 1e3, 1e5, 1e10, 1e50, 1e149):
            r = t / math.sqrt(t * t + n - 2) if t < 1e100 else 1.0 - 1e-16
            sums = (0.0, float(n - 1), r * (n - 1), 0.0, float(n - 1), n)
            th = host_t(*sums)
            want = t_tail(th, dof)
            if want < mpmath.mpf("1e-300"):
                continue
            got = lib.vampomi_host_linear_reg1d_pvals(*sums)
            assert abs(got - want) <= 1e-10 * want, (dof, t, got, float(want))
            checked += 1
    assert checked > 120, checked


# ---- loo p-values entry by entry ----------------------------------------------------------------------------------------------
LOO_CONSTANTS = [0.1, 0.7, 0.9532, 1 / 3, 0.0]


def loo_columns(N, rng):
    cols = [rng.beta(0.3, 0.3, N) for _ in range(6)]                     # bimodal, methylation-like
    cols += [0.9 + 0.005 * rng.standard_normal(N) for _ in range(6)]      # offset: mean 0.9, sd 0.005
    a = np.full(N, 0.1)
    a[-1] = np.nextafter(0.1, 1.0)                                        # one entry off by an ulp
    cols.append(a)
    a = np.full(N, 0.7)
    a[N // 2] = np.nextafter(0.7, 0.0)
    cols.append(a)
    cols += [np.full(N, c) for c in LOO_CONSTANTS]
    return np.array(cols)


def loo_bounds(x, w, c, n):
    """The exact t of the regression of y = w + c x on x (y_mark of src/data.cpp:404-405, with the FP64 c = x1 / sqrt(N) the host
    uses), from two-pass centred long-double sums, and the bound dt on the host's t from the conditioning of the textbook
    formulas of linear_reg1d_pvals. Each of s2x, s2y, sxy is a difference whose terms sum to T (in absolute value); computed from
    FP64 sums of n terms (this test's inputs) and the host's few operations it is within (n + 16) u T, relative eps = that / its
    exact value. r = sxy / sqrt(s2x s2y) is then within dr = (n + 16) u T_xy / (n - 1) / sqrt(s2x s2y) + |r| (eps_x + eps_y) / 2 +
    4 u |r|, and t = r sqrt((n-2)/(1-r^2)), whose derivative is sqrt(n-2) (1-r^2)^-1.5, within dt = dr sqrt(n-2) / (1 - r'^2)^1.5
    + 4 u |t| (1 + r^2)/(1 - r^2), r' = |r| + dr. Returns (|t|, dt), dt = inf where dr >= (1 - |r|)/2: there the formula cannot
    resolve the column (the r^2/(1-r^2) and T/result factors are >= 1/u), and only a finite p in [0, 1] is required."""
    L = np.longdouble
    u = L(2.0 ** -53)
    xl, wl, cl = x.astype(L), w.astype(L), L(c)
    yl = wl + cl * xl
    dx, dy = xl - xl.mean(), yl - yl.mean()
    sxx_c, syy_c, sxy_c = (dx * dx).sum(), (dy * dy).sum(), (dx * dy).sum()
    ax, aw = np.abs(xl), np.abs(wl)
    Tx = (xl * xl).sum() + ax.sum() ** 2 / n
    Ty = (wl * wl).sum() + 2 * abs(cl) * (ax * aw).sum() + cl * cl * (xl * xl).sum() + (aw.sum() + abs(cl) * ax.sum()) ** 2 / n
    Txy = (ax * aw).sum() + abs(cl) * (xl * xl).sum() + ax.sum() * (aw.sum() + abs(cl) * ax.sum()) / n
    if sxx_c <= 0 or syy_c <= 0:
        return None, math.inf
    k = (n + 16) * u
    eps_x, eps_y = k * Tx / sxx_c, k * Ty / syy_c
    r = sxy_c / np.sqrt(sxx_c * syy_c)
    dr = k * Txy / np.sqrt(sxx_c * syy_c) + abs(r) * ((eps_x + eps_y) / 2 + 4 * u)
    if not dr < (1 - abs(r)) / 2:
        return None, math.inf
    t = abs(r) * np.sqrt(L(n - 2) / (1 - r * r))
    rp = abs(r) + dr
    dt = dr * np.sqrt(L(n - 2)) / (1 - rp * rp) ** L(1.5) + 4 * u * t * (1 + r * r) / (1 - r * r)
    return float(t), float(dt)


@pytest.mark.parametrize("N", [400, 20000])
def test_loo_pvalues_entry_by_entry_against_mpmath(lib, N):
    """vampomi_host_loo_pvals(_flagged) against the exact p-value of each marker's regression: p must lie within
    [p(|t| + dt), p(|t| - dt)] (loo_bounds), widened by 1e-10 relative for the Student-t tail. Inputs are the FP64 sums of
    raw columns (bimodal, offset, one entry off by an ulp, constants 0.1, 0.7, 0.9532, 1/3, 0) with effects from none to
    dominant. Constant columns passed as flagged get exactly 1.0; without flags, and for the nearly constant columns, p must be
    finite and in [0, 1]: no NaN from rounding residue."""
    rng = np.random.default_rng(N)
    A = loo_columns(N, rng)
    M = A.shape[0]
    w = rng.standard_normal(N)
    sqrtN = math.sqrt(N)
    x1 = np.array([(0.0, 0.3, -2.0, 30.0, 1e-3, -400.0)[j % 6] for j in range(M)]) * sqrtN
    sums = np.ascontiguousarray(np.stack([A.sum(1), (A * A).sum(1), A @ w], axis=1))
    const = (A.min(1) == A.max(1)).astype(np.uint8)
    assert const.sum() == len(LOO_CONSTANTS)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    flagged, plain, zeros = np.full(M, -1.0), np.full(M, -1.0), np.full(M, -1.0)
    lib.vampomi_host_loo_pvals_flagged(dp(x1), dp(sums), w.sum(), (w * w).sum(), N, M, const.ctypes.data_as(capi.c_u8_p), dp(flagged), 0)
    lib.vampomi_host_loo_pvals(dp(x1), dp(sums), w.sum(), (w * w).sum(), N, M, dp(plain), 0)
    nof = np.zeros(M, dtype=np.uint8)
    lib.vampomi_host_loo_pvals_flagged(dp(x1), dp(sums), w.sum(), (w * w).sum(), N, M, nof.ctypes.data_as(capi.c_u8_p), dp(zeros), 0)
    assert np.array_equal(zeros, plain)
    lib.vampomi_host_loo_pvals_flagged(dp(x1), dp(sums), w.sum(), (w * w).sum(), N, M, None, dp(zeros), 0)
    assert np.array_equal(zeros, plain)
    assert np.all(np.isfinite(plain) & (plain >= 0) & (plain <= 1)), plain
    assert np.all(flagged[const == 1] == 1.0) and np.array_equal(flagged[const == 0], plain[const == 0])
    resolved = 0
    for j in range(M):
        if const[j]:
            continue
        t, dt = loo_bounds(A[j], w, x1[j] / sqrtN, N)
        if not math.isfinite(dt):
            continue
        lo = float(t_tail(t + dt, N - 2)) * (1 - 1e-10)
        hi = min(1.0, float(t_tail(max(0.0, t - dt), N - 2)) * (1 + 1e-10))
        assert lo <= plain[j] <= hi, (j, plain[j], lo, hi, t, dt)
        resolved += 1
    assert resolved >= 12, resolved                       # the bimodal and offset columns are all resolved


def test_loo_pvalues_of_a_marker_block_are_the_same_on_any_number_of_threads(lib):
    """vampomi_host_loo_pvals: the per-marker tail of data::pvals_loo (src/data.cpp:400-414) for a block of markers — equal to the
    per-marker function (and so to scipy) marker by marker, bit for bit on 1, 3 and all host threads."""
    rng = np.random.default_rng(5)
    n, M = 400, 20000
    A = rng.standard_normal((M, n)) * 0.3 + 0.5                     # raw, unstandardised columns
    w = rng.standard_normal(n)                                      # y_mod
    x1 = rng.standard_normal(M) * (rng.random(M) < 0.1)
    sums = np.ascontiguousarray(np.stack([A.sum(1), (A * A).sum(1), A @ w], axis=1))
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    outs = []
    for threads in (1, 3, 0):
        out = np.full(M, -1.0)
        lib.vampomi_host_loo_pvals(dp(x1), dp(sums), w.sum(), (w * w).sum(), n, M, dp(out), threads)
        outs.append(out)
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
    for j in list(range(0, M, 997)) + [M - 1]:
        c = x1[j] / np.sqrt(n)
        ym = w + A[j] * c
        one = lib.vampomi_host_linear_reg1d_pvals(A[j].sum(), (A[j] * A[j]).sum(), (A[j] * ym).sum(), ym.sum(), (ym * ym).sum(), n)
        assert outs[0][j] == pytest.approx(one, rel=1e-9, abs=1e-300)
        assert outs[0][j] == pytest.approx(spstats.linregress(A[j], ym).pvalue, rel=1e-6, abs=1e-300)


def test_counter_hash_matches_oracle_and_reference_hooks(lib):
    for seed in (0, 7, 2 ** 63 + 5):
        for it in (1, 2, 50):
            want = vo.probe_signs(seed, it, 1000, 64)
            got = np.array([lib.vampomi_host_probe_sign(seed, it, 1000 + j) for j in range(64)])
            assert np.array_equal(got, want)
        out, po = arr(np.zeros(500))
        lib.vampomi_host_probit_p1(seed, 500, po)
        assert np.allclose(out, vo.probit_p1(seed, 500), rtol=0, atol=1e-14)
    s = vo.probe_signs(3, 1, 0, 100000)
    assert abs(s.mean()) < 0.02 and set(np.unique(s)) == {-1.0, 1.0}


@pytest.mark.parametrize("vars_,probs,thr", [([0, 1e-6, 1.4e-6, 1e-3, 1.2e-3, 1.0], [0.9, 0.02, 0.02, 0.02, 0.02, 0.02], 0.5),
                                             ([0, 1e-8, 1e-3], [0.5, 0.25, 0.25], 0.5), ([0, 1, 2, 4, 8], [0.2] * 5, 1.01),
                                             ([1.0, 1.0, 1.0], [0.2, 0.3, 0.5], 0.5), ([0, 5e-8, 1.0], [0.5, 0.2, 0.3], 0.9)])
def test_merge_components_matches_oracle(lib, vars_, probs, thr):
    p_want, v_want = list(probs), list(vars_)
    vo.merge_components(p_want, v_want, thr)
    p, pp = arr(probs)
    v, pv = arr(vars_)
    L = lib.vampomi_host_merge_components(pp, pv, len(probs), thr)
    assert L == len(p_want)
    assert np.allclose(p[:L], p_want, rtol=1e-15) and np.allclose(v[:L], v_want, rtol=1e-15)
    assert math.isclose(sum(p[:L]), sum(probs), rel_tol=1e-14)


def test_grid_planning_fills_whole_waves():
    """vampomi_plan_chunks: (row tile x column chunk) grids use the smallest number of full waves that leaves at most 1 % of
    the resident-CTA slots empty; never fewer than min_cols columns per chunk."""
    slots = 296                                             # 148 SMs x 2 CTAs
    assert capi.plan_chunks(slots, 20, 106250, 16, balance=False) == 14          # one wave: 280 of 296 slots
    n = capi.plan_chunks(slots, 20, 106250, 16)
    assert n == 44 and 20 * n <= 3 * slots and 20 * n >= 0.99 * 3 * slots        # three waves of 880 CTAs on 888 slots
    assert capi.plan_chunks(slots, 5, 106250, 16) == 59                          # 295 of 296: one wave is already full
    assert capi.plan_chunks(slots, 10, 106250, 16) == 59                         # two waves: 590 of 592
    assert capi.plan_chunks(slots, 1, 106250, 16) == 296
    assert capi.plan_chunks(slots, 20, 100, 16) == 7                             # small M: at least 16 columns per chunk
    assert capi.plan_chunks(slots, 400, 106250, 16) >= 1                         # more tiles than slots
    for ntiles in range(1, 64):
        n = capi.plan_chunks(slots, ntiles, 10 ** 6, 1)
        waves = -(-ntiles * n // slots)
        assert ntiles * n >= 0.99 * waves * slots or waves >= 8, (ntiles, n)


def test_recycled_products_are_identities_of_the_cg_recurrences():
    """The `recycled` schedule takes A x2_hat, A Q^-1 u and A^T A of both solutions from the solves instead of computing them
    with passes of their own (DESIGN.md §3a). In numpy, with the oracle's operators: running precondCG_solver's recurrences
    (src/vamp.cpp:671-757) with the two extra updates the device makes — Amu += alpha * (A p) next to mu += alpha * p, and r
    always advanced with mu — leaves Amu = A mu and (v - r - gam2 mu)/tau = A^T A mu to rounding, for a cold and a warm start."""
    rng = np.random.default_rng(11)
    N, M = 300, 700
    A = rng.standard_normal((M, N)) * 0.1 + 0.5
    d = vo.Data(A, rng.standard_normal(N))
    tau, gam2 = 2.3, 1.9
    diag = tau * (N - 1) / N + gam2
    for warm in (False, True):
        v = rng.standard_normal(M)
        mu = rng.standard_normal(M) * 0.1 if warm else np.zeros(M)
        Amu = d.Ax(mu) if warm else np.zeros(N)                 # the previous iteration's A x2_hat (warm) or zero
        r = v - (tau * d.ATx(d.Ax(mu)) + gam2 * mu) if warm else v.copy()
        z = r / diag
        p = z.copy()
        for _ in range(12):
            Ap = d.Ax(p)
            dvec = tau * d.ATx(Ap) + gam2 * p
            alpha = (r @ z) / (dvec @ p)
            mu = mu + alpha * p
            Amu = Amu + alpha * Ap
            rz_old = r @ z
            r = r - dvec * alpha
            z = r / diag
            p = z + (r @ z) / rz_old * p
        assert np.linalg.norm(Amu - d.Ax(mu)) < 1e-13 * np.linalg.norm(Amu)
        ata = (v - r - gam2 * mu) / tau
        want = d.ATx(d.Ax(mu))
        assert np.linalg.norm(ata - want) < 1e-12 * np.linalg.norm(want)


def test_covariate_reader_and_newton_match_oracle(tmp_path):
    """SURVEY.md §8 f3 on the host: data::read_covariates (src/data.cpp:159-227) and vamp::Newton_method_cov
    (src/vamp_probit.cpp:525-617) of libvampomi_cuda's host layer against the numpy restatement — no GPU involved."""
    import ctypes as C
    from vampomi_b200 import capi, sim
    lib = capi.load_library()
    N, Cn = 150, 3
    rng = np.random.default_rng(5)
    cov = sim.simulate_covariates(N, Cn, 9)
    cov[:, 1] = 4.25                                          # a constant covariate -> all zeros after standardisation
    path = str(tmp_path / "c.cov")
    sim.write_covariates(path, cov)
    want = vo.read_covariates(path, Cn, N)
    got = np.empty(N * Cn)
    n = lib.vampomi_host_read_covariates(path.encode(), Cn, N, got.ctypes.data_as(capi.c_double_p))
    assert n == N * Cn and np.array_equal(got.reshape(N, Cn), want) and np.all(want[:, 1] == 0)
    assert abs(want[:, 0].mean()) < 1e-12 and abs(want[:, 0].std() - 1) < 1e-12
    assert lib.vampomi_host_read_covariates(path.encode(), Cn + 1, N, got.ctypes.data_as(capi.c_double_p)) == -1      # wrong --C
    assert lib.vampomi_host_read_covariates(path.encode(), Cn, N + 1, got.ctypes.data_as(capi.c_double_p)) == -1      # wrong --N
    Z = vo.read_covariates(path, Cn, N)[:, [0, 2]].copy()
    for y in ((Z @ np.array([0.8, -0.5]) + rng.standard_normal(N) > 0).astype(float), rng.standard_normal(N)):   # probit and linear use
        gg = np.zeros(N)
        eta_want = vo.newton_method_cov(y, gg, Z, np.zeros(2))
        eta = np.zeros(2)
        rc = lib.vampomi_host_newton_cov(y.ctypes.data_as(capi.c_double_p), gg.ctypes.data_as(capi.c_double_p),
                                         np.ascontiguousarray(Z).ctypes.data_as(capi.c_double_p), N, 2, eta.ctypes.data_as(capi.c_double_p))
        assert rc == 0 and np.allclose(eta, eta_want, rtol=1e-9, atol=1e-12), (eta, eta_want)


def test_onepass_cg_recurrences_reproduce_the_two_pass_iterates():
    """The `onepass` schedule (DESIGN.md §3b) in numpy, with the oracle's operators: carrying q = A p as a vector of its own — one
    fused product pair t = A^T q, w = A t per iteration, then A r -= alpha (tau w + gam2 q) and q = (A r)/diag + beta q — gives the
    iterates, residuals and step lengths of precondCG_solver's own recurrences (src/vamp.cpp:671-757), which apply A and A^T to p in
    every iteration; q stays equal to A p to rounding, with and without the periodic recomputation."""
    rng = np.random.default_rng(12)
    N, M = 250, 900
    A = rng.standard_normal((M, N)) * 0.1 + 0.5
    d = vo.Data(A, rng.standard_normal(N))
    tau, gam2 = 2.3, 0.7
    diag = tau * (N - 1) / N + gam2
    v = rng.standard_normal(M)
    for refresh in (0, 5):
        # two passes per iteration: the reference's recurrences
        mu2, r2 = np.zeros(M), v.copy()
        z2 = r2 / diag
        p2 = z2.copy()
        # one pass per iteration
        mu, r = np.zeros(M), v.copy()
        z = r / diag
        p = z.copy()
        q = d.Ax(p)                                   # the solve's only A* pass
        Ar = diag * q
        for it in range(14):
            d2 = tau * d.ATx(d.Ax(p2)) + gam2 * p2
            a2 = (r2 @ z2) / (d2 @ p2)
            mu2 = mu2 + a2 * p2
            rz2 = r2 @ z2
            r2 = r2 - d2 * a2
            z2 = r2 / diag
            p2 = z2 + (r2 @ z2) / rz2 * p2

            if refresh and it > 0 and it % refresh == 0:            # q and A r afresh from p and z (cg.cu, gram_refresh)
                q, Ar = d.Ax(p), diag * d.Ax(z)
            t = d.ATx(q)                                            # the fused pass: A^T q ...
            w = d.Ax(t)                                             # ... and A A^T q
            dvec = tau * t + gam2 * p
            alpha = (r @ z) / (dvec @ p)
            mu = mu + alpha * p
            rz = r @ z
            r = r - dvec * alpha
            z = r / diag
            beta = (r @ z) / rz
            p = z + beta * p
            Ar = Ar - alpha * (tau * w + gam2 * q)
            q = Ar / diag + beta * q
            assert abs(alpha - a2) < 1e-11 * abs(a2)
            assert np.linalg.norm(mu - mu2) < 1e-11 * np.linalg.norm(mu2) and np.linalg.norm(r - r2) < 1e-9 * np.linalg.norm(v)
            assert np.linalg.norm(q - d.Ax(p)) < 1e-10 * np.linalg.norm(q)


def test_product_library_holds_exactly_the_fused_pass_kernels():
    """The fused pass is one kernel, k_gram_wsx<K, CS>: the library must hold its 32 instantiations (one or two systems,
    clusters of 1 ... 16 CTAs), no other k_gram* kernel, and none of them may use local memory."""
    import os
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib = os.path.join(root, "vampomi_b200", "lib", "libvampomi_cuda.so")
    out = subprocess.run(["cuobjdump", "-res-usage", lib], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout
    usage = dict(re.findall(r"Function (\S*k_gram\S*):\s*\n\s*(.*)", out))
    names = sorted(re.search(r"k_gram\w*", f).group(0) for f in usage)
    assert names == sorted(f"k_gram_wsxILi{k}ELi{cs}EEEvPKdmS3_S3_NS0_7GramVecEiixdPdi14CUtensorMap_st" for k in (1, 2) for cs in range(1, 17)), names
    for f, u in usage.items():
        assert re.search(r"\bLOCAL:0\b", u), (f, u)
