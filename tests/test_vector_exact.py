"""Every output entry of the vector kernels (denoiser, EM sums, probit z-channel, se p-values, the CG vector steps) against the
exact value of the same formula, computed in extended precision (np.longdouble, 64-bit mantissa) or in mpmath where numpy has
no extended function (erfc, erfcx), on the inputs the kernel actually read. test_gpu_ops compares these kernels with the numpy
oracle in the L2 norm; the oracle repeats the kernels' formulas in FP64 and shares their rounding, so an entry that is wrong the
same way in both, or small because its terms cancel, is never seen there. Here each entry has its own bound, derived from the
terms the formula adds and from the arguments of its transcendentals (u = 2^-53):

* a sum of n terms in any order, with each term's own relative error e_k:  |got - exact| <= sum_k |term_k| (e_k + (n + 8) u);
* exp(x) with x carrying a relative error a u:  relative error (a |x| + 2) u (CUDA's exp is within 1 ulp = 2 u);
* erfc / erfcx at x with relative error a u in x:  (8 + a |x f'(x) / f(x)|) u (CUDA documents 4 ulp for both).

The whole-path cases at the end run `association_test --pval-method loo` on blocks with constant columns, and a long one-pass
CG solve whose tracked A mu and q = A p are compared with A applied to the device's own mu and p."""
import math
import os
import subprocess

import mpmath
import numpy as np
import pytest

from vampomi_b200 import build, capi
from vampomi_b200.capi import (V_CG2_D, V_CG2_P, V_CG2_R, V_CG2_Z, V_CG_D, V_CG_P, V_CG_R, V_CG_Z, V_MCOV, V_P1, V_R1, V_TMP_M0,
                               V_TMP_M1, V_TMP_N0, V_USER_M0, V_USER_M1, V_USER_N0, V_USER_N1, V_V, V_X1, V_X1_PREV, V_X2, V_Y,
                               V_Z1HAT)

pytestmark = pytest.mark.gpu

LD = np.longdouble
U = 2.0 ** -53
mpmath.mp.dps = 40
VECTOR_MS = (4000, 75777, 200003)     # the grid-stride loops of the vector kernels wrap from 296 x 256 = 75 776 entries on
MIXTURES = (None, 2, 32)
DEFAULT_PROBS = [0.99, 0.005, 0.0025, 0.00125, 0.000625, 0.0003125, 0.00015625, 7.8125e-05, 3.90625e-05, 3.90625e-05]
DEFAULT_VARS = [0, 1e-06, 6e-06, 3e-05, 0.0002, 0.001, 0.006, 0.03, 0.2, 1.0]


@pytest.fixture(autouse=True)
def _extended_precision():
    if np.finfo(np.longdouble).nmant < 63:
        pytest.skip("np.longdouble has fewer than 63 mantissa bits here: no extended-precision reference")


def mixture(L):
    """(probs, vars) of L components: the reference's defaults, or a spike and L - 1 slabs with geometric variances."""
    if L is None:
        return list(DEFAULT_PROBS), list(DEFAULT_VARS)
    slabs = 0.5 ** np.arange(1, L)
    return [0.9] + list(0.1 * slabs / slabs.sum()), [0.0] + list(np.geomspace(1e-6, 1.0, L - 1))


def check(got, exact, bound, what):
    """|got - exact| <= bound entry by entry (+ 1e-300 for underflow); a NaN fails."""
    got = np.atleast_1d(np.asarray(got, dtype=np.float64))
    err = np.abs(got.astype(LD) - exact)
    bad = ~(err <= bound + LD(1e-300))
    if bad.any():
        i = int(np.argmax(bad))
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} entries outside the bound; entry {i}: got {got[i]!r}, "
                             f"exact {float(exact[i])!r}, error {float(err[i]):.3g}, bound {float(bound[i]):.3g}")


# ---- Gaussian-mixture denoiser (k_denoise) -----------------------------------------------------------------------------------
def denoise_exact(y, gam1, probs, vars_):
    """g1, g1d of src/vamp.cpp:440-492 in long double, with error bounds for the FP64 kernel.

    Term l: z_l = pi_l / sqrt(vs_l) e_l, e_l = exp(x_l), vs_l = v_l + sigma, x_l = -y^2 (eta - v_l) / (2 vs_l (eta + sigma)).
    x_l is formed by 8 roundings (sigma = 1/gam1 and vs_l included), so its relative error is <= 8 u and e_l's is
    <= (10 |x_l| + 2) u; sqrt, the division and the product add 4 u: |dz_l| <= (12 + 10 |x_l|) u z_l. pk = sum z_l and
    pkd = -sum z_l y / vs_l are sums of terms of ONE sign, so their relative errors are the largest term error plus L u:
    rel_pk = sum_l (12 + 10|x_l|) u z_l / pk + L u, rel_pkd likewise with 3 u more per term. Then
        |g - exact| <= u |y| + |sigma pkd / pk| (rel_pk + rel_pkd + 4 u)
    which is (c + 4|x|) u (|y| + |sigma pkd/pk|) per entry: for a tiny gam1, g = y + sigma pkd/pk cancels against y and the
    bound is honest about it entry by entry. pkdd = sum_l (-pi_l vs_l^-1.5 e_l + z_l y^2 / vs_l^2) has terms of both signs: its
    error is bounded by sum_l |terms| (18 + 10 |x_l|) u + L u sum|terms|, and
        |gd - exact| <= u (1 + |gd|) + sigma (|pkdd|/pk (rel_pkdd + rel_pk + 2u) + q^2 (2 rel_q + 2u)) + u sigma (|pkdd/pk| + q^2)
    with q = pkd/pk, rel_q = rel_pk + rel_pkd + u."""
    y = np.asarray(y, dtype=np.float64).astype(LD)[:, None]
    sigma = LD(1) / LD(gam1)
    pr, v = np.array(probs, dtype=np.float64).astype(LD), np.array(vars_, dtype=np.float64).astype(LD)
    eta = v.max()
    vs = v + sigma
    x = -LD(0.5) * (y * y) * (eta - v) / vs / (eta + sigma)
    e = np.exp(x)
    z = pr / np.sqrt(vs) * e
    zd = z / vs * y
    t1, t2 = pr / vs ** LD(1.5) * e, zd / vs * y
    L = len(probs)
    pk, pkd, pkdd = z.sum(1), -zd.sum(1), (-t1 + t2).sum(1)
    ax = np.abs(x)
    rel_pk = ((12 + 10 * ax) * z).sum(1) * LD(U) / pk + L * LD(U)
    rel_pkd = np.where(pkd != 0, ((15 + 10 * ax) * np.abs(zd)).sum(1) * LD(U) / np.where(pkd != 0, np.abs(pkd), 1) + L * LD(U), 0)
    abs_pkdd = ((18 + 10 * ax) * (t1 + np.abs(t2))).sum(1) * LD(U) + L * LD(U) * (t1 + np.abs(t2)).sum(1)
    q = pkd / pk
    g = y[:, 0] + sigma * q
    A = pkdd / pk
    gd = 1 + sigma * (A - q * q)
    yy = np.abs(y[:, 0])
    bg = LD(U) * yy + np.abs(sigma * q) * (rel_pk + rel_pkd + 4 * LD(U))
    rel_q = rel_pk + rel_pkd + LD(U)
    bgd = (LD(U) * (1 + np.abs(gd)) + sigma * (abs_pkdd / pk + np.abs(A) * (rel_pk + 2 * LD(U)) + q * q * (2 * rel_q + 2 * LD(U)))
           + LD(U) * sigma * (np.abs(A) + q * q))
    return g, gd, bg, bgd


DENOISE_R1 = [0.0, 1e-300, -40.0, 40.0, 1e3, -1e3, 0.731, -2.5, 7.0]


@pytest.mark.parametrize("L", MIXTURES)
@pytest.mark.parametrize("gam1", [1e-6, 0.37, 25.0, 1e12])
def test_denoise_exact(gam1, L):
    """x1 (plain and damped), x1_prev (bitwise) and the sum of g1d over M markers; g1d entry by entry through a one-marker shard,
    whose sum is that entry. gam1 = 1e12 takes the kernel's degenerate branch (sigma < 1e-10): g1 = y, g1d = 1 exactly."""
    N = 200
    probs, vars_ = mixture(L)
    vint = list(np.array(vars_) * N)
    rng = np.random.default_rng(int(gam1 * 7) % 1000 + (L or 10))
    degenerate = 1.0 / gam1 < 1e-10
    for M in VECTOR_MS:
        with capi.Shard(N, M) as sh:
            r1 = rng.standard_normal(M) * 3
            r1[:len(DENOISE_R1)] = DENOISE_R1
            prev = rng.standard_normal(M)
            g, gd, bg, bgd = denoise_exact(r1, gam1, probs, vint)
            for damp, rho in ((False, 1.0), (True, 0.3)):
                sh.set(V_R1, r1)
                sh.set(V_X1, prev)
                s = sh.denoise(gam1, np.array(probs), np.array(vint), damp=damp, rho=rho)
                x1 = sh.get(V_X1)
                assert np.array_equal(sh.get(V_X1_PREV).view(np.uint64), prev.view(np.uint64)), (M, damp)
                if degenerate:
                    want = LD(rho) * r1.astype(LD) + (1 - LD(rho)) * prev.astype(LD) if damp else r1.astype(LD)
                    if not damp:
                        assert np.array_equal(x1, r1)
                    assert s == float(M), s
                    bnd = 3 * LD(U) * (np.abs(want) + np.abs(prev.astype(LD)))
                    check(x1, want, bnd, f"x1 degenerate damp={damp}")
                    continue
                if damp:
                    # rho g + (1 - rho) prev: two products, a sum and 1 - rho, each rounded once
                    want = LD(rho) * g + (1 - LD(rho)) * prev.astype(LD)
                    bnd = LD(rho) * bg + 4 * LD(U) * (np.abs(LD(rho) * g) + np.abs((1 - LD(rho)) * prev.astype(LD)))
                else:
                    want, bnd = g, bg
                check(x1, want, bnd, f"x1 M={M} damp={damp}")
                check([s], np.array([gd.sum()]), np.array([bgd.sum() + (M + 8) * LD(U) * np.abs(gd).sum()]), f"sum g1d M={M}")
    vals = np.array(DENOISE_R1 + list(rng.standard_normal(6) * 3))
    g, gd, bg, bgd = denoise_exact(vals, gam1, probs, vint)
    with capi.Shard(N, 1) as sh:
        got = []
        for v in vals:
            sh.set(V_R1, [v])
            got.append(sh.denoise(gam1, np.array(probs), np.array(vint)))
            if degenerate:
                assert sh.get(V_X1)[0] == v and got[-1] == 1.0
    if not degenerate:
        check(np.array(got), gd, bgd, "g1d per entry")


# ---- EM sums (k_em_sums) -----------------------------------------------------------------------------------------------------
def em_exact(r, gam1, lam, omegas, vars_):
    """The 2L - 1 sums of src/vamp.cpp:554-597 in long double and their bounds.

    Per marker: num_j = lam om_j exp(x_j) / sqrt(v_j + nv) / sqrt(2 pi) (j >= 1), x_j = -r^2/2 (vmax - v_j)/(v_j + nv)/(vmax + nv),
    tot = sum num_j, X = (1 - lam) / sqrt(2 pi nv) exp(x_0) / tot, x_0 = -r^2/2 vmax / nv / (nv + vmax), pin = 1 / (1 + X),
    beta_j = num_j / tot, gm_j = beta_j (ng_j^2 + 1/(1/v_j + gam1)), ng_j = gam1 r / (1/v_j + gam1). The exponents carry <= 8 u:
    rel(num_j) <= (14 + 10|x_j|) u; tot is a same-sign sum, rel(tot) <= max_j rel(num_j) + L u; rel(X) <= (12 + 10|x_0|) u +
    rel(tot); pin = 1/(1+X) has rel <= rel(X) X/(1+X) + 3 u; rel(beta_j) <= rel(num_j) + rel(tot) + u; gm_j adds 12 u. Each sum
    of M terms is then within sum_i |term_i| (rel_i + (M + 8) u)."""
    r = np.asarray(r, dtype=np.float64).astype(LD)[:, None]
    gam1 = LD(gam1)
    nv = 1 / gam1
    om, v = np.array(omegas, dtype=np.float64).astype(LD), np.array(vars_, dtype=np.float64).astype(LD)
    vmax = v.max()
    two_pi = 2 * LD(str(mpmath.pi))
    r2h = r * r / 2
    vj, oj = v[1:], om[1:]
    xj = -r2h * (vmax - vj) / (vj + nv) / (vmax + nv)
    num = LD(lam) * oj * np.exp(xj) / np.sqrt(vj + nv) / np.sqrt(two_pi)
    ng = gam1 * r / (1 / vj + gam1)
    tot = num.sum(1, keepdims=True)
    x0 = -r2h[:, 0] * vmax / nv / (nv + vmax)
    X = (1 - LD(lam)) / np.sqrt(two_pi * nv) * np.exp(x0) / tot[:, 0]
    pin = 1 / (1 + X)
    beta = num / tot
    gm = beta * (ng * ng + 1 / (1 / vj + gam1))
    L = len(omegas)
    rel_num = (14 + 10 * np.abs(xj)) * LD(U)
    rel_tot = rel_num.max(1) + L * LD(U)
    rel_pin = ((12 + 10 * np.abs(x0)) * LD(U) + rel_tot) * X / (1 + X) + 3 * LD(U)
    rel_beta = rel_num + rel_tot[:, None] + LD(U)
    terms = [pin] + [beta[:, j] * pin for j in range(L - 1)] + [gm[:, j] * pin for j in range(L - 1)]
    rels = [rel_pin] + [rel_beta[:, j] + rel_pin for j in range(L - 1)] + [rel_beta[:, j] + rel_pin + 12 * LD(U) for j in range(L - 1)]
    M = r.shape[0]
    exact = np.array([t.sum() for t in terms])
    bound = np.array([(np.abs(t) * (e + (M + 8) * LD(U))).sum() for t, e in zip(terms, rels)])
    return exact, bound


@pytest.mark.parametrize("L", MIXTURES)
def test_em_sums_exact(L):
    N = 150
    probs, vars_ = mixture(L)
    vint = list(np.array(vars_) * N)
    lam = 1 - probs[0]
    omegas = [probs[0]] + [p / lam for p in probs[1:]]
    rng = np.random.default_rng(6 + (L or 0))
    for M in VECTOR_MS:
        r1 = rng.standard_normal(M) * 2
        r1[:6] = [0.0, 1e-300, 40.0, -40.0, 1e3, -7.5]
        with capi.Shard(N, M) as sh:
            sh.set(V_R1, r1)
            for gam1 in (0.8, 1e-3, 40.0):
                got = sh.em_sums(gam1, lam, omegas, vint)
                assert got.size == 2 * len(probs) - 1
                exact, bound = em_exact(r1, gam1, lam, omegas, vint)
                check(got, exact, bound, f"EM sums M={M} gam1={gam1}")


# ---- probit z-channel (k_probit_z) -------------------------------------------------------------------------------------------
def erfcx_mp(x):
    x = mpmath.mpf(float(x))
    return mpmath.exp(x * x) * mpmath.erfc(x)


def test_probit_z_exact():
    """z1hat = p + s ratio / tau1 / sroot, ratio = 2/sqrt(2 pi) / erfcx(x), x = -s (p + mcov) / sroot / sqrt(2), s = 2y - 1,
    sroot = sqrt(1 + 1/tau1) (src/vamp_probit.cpp:469-488). x is formed with <= 6 roundings; erfcx(x) then has relative error
    <= (8 + 6 k(x)) u with k(x) = |x erfcx'(x) / erfcx(x)| = |x (2x - 2 / (sqrt(pi) erfcx(x)))|; ratio adds 3 u and z1hat's three
    operations 3 u of the ratio term and u of |z1hat|. Where the reference clamps erfcx (x < -10: +Inf, ratio 0; x > 10:
    -DBL_MAX) z1hat must be exactly the clamp's value, computed in FP64 in the kernel's order. The sum of
    1 - ratio/(1 + tau1) (s cc + ratio) over N entries is bounded by the same ratio error on |ratio| (|s cc| + |ratio|) plus
    (N + 8) u times the sum of |terms|."""
    N = 3000
    rng = np.random.default_rng(7)
    yb = (rng.random(N) > 0.5).astype(float)
    p1 = rng.standard_normal(N) * 4
    mcov = rng.standard_normal(N) * 0.5
    mcov[N // 2:] = 0.0
    # zero, both sides of both clamps (x = -+(p + mcov)/sroot/sqrt 2 = -+10) for every tau1, with and without an offset, and
    # p + mcov cancelling
    p1[:12] = [0.0, 30.0, -30.0, 12.0, -12.0, 14.0, 14.2, -14.0, -14.2, 1e-300, 3.0, -3.0]
    mcov[10], mcov[11] = -3.0, 3.0
    p1[28:32] = [1e3, -1e3, 2e3, -2e3]
    mcov[12:28] = 0.0
    with capi.Shard(N, 4) as sh:
        sh.set(V_Y, yb)
        sh.set(V_MCOV, mcov)
        for tau1 in (1e-2, 1.3, 50.0):
            sroot = math.sqrt(1.0 + 1.0 / tau1)
            for i in range(12, 28):                   # |x| within 8e-3 of the clamp at 10, on both sides of it
                p1[i] = (-1) ** i * (10.0 + (i - 20) * 1e-3) * math.sqrt(2.0) * sroot
            sh.set(V_P1, p1)
            s_dev = sh.probit_zdenoise(tau1)
            z = sh.get(V_Z1HAT)
            c0 = 2.0 / math.sqrt(2.0 * 3.14159265358979323846)
            sgn = 2.0 * yb - 1.0
            cc = (p1 + mcov) / sroot
            xarg = -sgn * cc / math.sqrt(2.0)
            lo, hi = xarg < -10.0, xarg > 10.0
            assert lo.any() and hi.any() and (~(lo | hi)).any()
            # clamped entries, FP64 in the kernel's order
            ratio_hi = c0 / -np.finfo(np.float64).max
            want_hi = p1[hi] + sgn[hi] * ratio_hi / tau1 / sroot
            assert np.array_equal(z[hi], want_hi) and np.array_equal(z[lo], p1[lo] + sgn[lo] * 0.0 / tau1 / sroot)
            mid = np.nonzero(~(lo | hi))[0]
            ex_z = np.empty(mid.size, dtype=LD)
            bz = np.empty(mid.size, dtype=LD)
            terms = np.empty(N, dtype=LD)
            bterm = np.zeros(N, dtype=LD)
            terms[lo] = 1
            terms[hi] = 1 - LD(ratio_hi) / (1 + LD(tau1)) * (LD(sgn[hi] * cc[hi]) + LD(ratio_hi))
            bterm[hi] = 8 * LD(U) * np.abs(terms[hi])
            for k, i in enumerate(mid):
                sr = mpmath.sqrt(1 + 1 / mpmath.mpf(tau1))
                c = (mpmath.mpf(p1[i]) + mpmath.mpf(mcov[i])) / sr
                x = -sgn[i] * c / mpmath.sqrt(2)
                ex = erfcx_mp(x)
                ratio = 2 / mpmath.sqrt(2 * mpmath.pi) / ex
                kx = abs(x * (2 * x - 2 / (mpmath.sqrt(mpmath.pi) * ex)))
                rel = (8 + 6 * kx + 3) * U
                ex_z[k] = LD(str(mpmath.mpf(p1[i]) + sgn[i] * ratio / tau1 / sr))
                rt = abs(ratio / tau1 / sr)
                bz[k] = LD(str(rt * (rel + 3 * U) + U * abs(mpmath.mpf(p1[i]) + sgn[i] * ratio / tau1 / sr)))
                R = ratio / (1 + mpmath.mpf(tau1))
                terms[i] = LD(str(1 - R * (sgn[i] * c + ratio)))
                bterm[i] = LD(str(U * (1 + abs(R * (sgn[i] * c + ratio))) + abs(R) * (abs(c) + abs(ratio)) * (2 * rel + 12 * U)))
            check(z[mid], ex_z, bz, f"z1hat tau1={tau1}")
            check([s_dev], np.array([terms.sum()]), np.array([bterm.sum() + (N + 8) * LD(U) * np.abs(terms).sum()]),
                  f"sum g1d tau1={tau1}")


# ---- se p-values (k_pvals_se) ------------------------------------------------------------------------------------------------
def test_pvals_se_exact():
    """p_j = erfc(|r_j| / (sd sqrt 2)) / 2, the normal tail beyond 0, relative to mpmath at |r|/sd from 0 to 38 for both signs.
    The kernel forms x = |r| / (sd sqrt 2) with 2 roundings and sqrt(2.0) (3 u), so p is within (8 + 3 k(x)) u relative with
    k(x) = |x erfc'(x) / erfc(x)| = 2 x exp(-x^2) / (sqrt(pi) erfc(x)) (about 2 x^2 in the tail). sd is the FP64 value the
    library passes, sqrt(1 / (gam1 N)). r = +-0 gives 0.5 exactly, a NaN stays NaN."""
    N, gam1 = 1000, 3.3
    sd = math.sqrt(1.0 / (gam1 * float(N)))
    k = np.concatenate([np.linspace(0, 38, 381)[1:], [5.9, 6.1, 8.5, 8.6, 20.0, 37.9]])
    r = np.concatenate([k * sd, -k * sd, [0.0, -0.0, np.nan]])
    with capi.Shard(N, r.size) as sh:
        got = sh.pvals_se(r, gam1)
    assert got[-3] == 0.5 and got[-2] == 0.5 and np.isnan(got[-1])
    fin = r[:-3]
    exact = np.empty(fin.size, dtype=LD)
    bound = np.empty(fin.size, dtype=LD)
    for i, v in enumerate(fin):
        x = abs(mpmath.mpf(v)) / (mpmath.mpf(sd) * mpmath.sqrt(2))
        e = mpmath.erfc(x)
        kx = 2 * x * mpmath.exp(-x * x) / (mpmath.sqrt(mpmath.pi) * e)
        exact[i] = LD(str(e / 2))
        bound[i] = LD(str(e / 2 * (8 + 3 * kx) * U))
    check(got[:-3], exact, bound, "se p-values")
    assert np.array_equal(got[:fin.size // 2], got[fin.size // 2:fin.size])     # the sign of r1 does not matter


# ---- CG vector steps (k_cg_init / dp / step / finish) --------------------------------------------------------------------------
def make_block(N, M, seed):
    rng = np.random.default_rng(seed)
    A = rng.beta(0.3, 0.3, size=(M, N))
    A[3] = 0.1                                   # a constant column (msig = 1, a zero row of the operator)
    sh = capi.Shard(N, M)
    sh.upload(A)
    sh.compute_stats()
    return sh, A, rng


SYS = [dict(r=V_CG_R, z=V_CG_Z, p=V_CG_P, d=V_CG_D, t=V_TMP_M0), dict(r=V_CG2_R, z=V_CG2_Z, p=V_CG2_P, d=V_CG2_D, t=V_TMP_M1)]


def cg_step_check(prev, cur, v, tau, gam2, diag, M, what):
    """One CG iteration (src/vamp.cpp:694-739) recomputed in long double from the device's previous mu, r, z, p and its own t:
    d = tau t + gam2 p (2 u of |tau t| + |gam2 p|); alpha = <r,z>/<d,p> from dot products within (M + 8) u sum|terms|;
    mu = mu + alpha p, r = r - alpha d (the error of alpha times |p| or |d|, plus 2 u of both terms); z = r / diag
    exactly rounded from the device's r; beta = <r,z>_new / <r,z>_old and p = z + beta p likewise; <v,mu> within
    (M + 8) u sum|v mu| of the device's own mu."""
    L = lambda a: a.astype(LD)
    u = LD(U)
    t, p0, r0, z0, mu0 = L(cur["t"]), L(prev["p"]), L(prev["r"]), L(prev["z"]), L(prev["mu"])
    d = LD(tau) * t + LD(gam2) * p0
    check(cur["d"], d, 2 * u * (np.abs(LD(tau) * t) + np.abs(LD(gam2) * p0)), f"{what}: d")
    dd = L(cur["d"])
    dp, dp_abs = (dd * p0).sum(), np.abs(dd * p0).sum()
    rz0 = (r0 * z0).sum()
    rel_alpha = (M + 8) * u * (dp_abs / abs(dp) + np.abs(r0 * z0).sum() / abs(rz0)) + 2 * u
    alpha = rz0 / dp
    mu = mu0 + alpha * p0
    check(cur["mu"], mu, np.abs(alpha * p0) * rel_alpha + 2 * u * (np.abs(mu0) + np.abs(alpha * p0)), f"{what}: mu")
    r = r0 - alpha * dd
    check(cur["r"], r, np.abs(alpha * dd) * rel_alpha + 2 * u * (np.abs(r0) + np.abs(alpha * dd)), f"{what}: r")
    assert np.array_equal(cur["z"], cur["r"] / diag), f"{what}: z = r / diag, rounded once"
    rr, zz = L(cur["r"]), L(cur["z"])
    rz1 = (rr * zz).sum()
    beta = rz1 / rz0
    rel_beta = (M + 8) * u * (np.abs(rr * zz).sum() / abs(rz1) + np.abs(r0 * z0).sum() / abs(rz0)) + 2 * u
    check(cur["p"], zz + beta * p0, np.abs(beta * p0) * rel_beta + 2 * u * (np.abs(zz) + np.abs(beta * p0)), f"{what}: p")
    vm = L(v) * L(cur["mu"])
    check([cur["vmu"]], np.array([vm.sum()]), np.array([(M + 8) * u * np.abs(vm).sum()]), f"{what}: <v,mu>")


def snapshot(sh, s, mu_vec, vmu):
    k = SYS[s]
    return dict(r=sh.get(k["r"]), z=sh.get(k["z"]), p=sh.get(k["p"]), d=sh.get(k["d"]), t=sh.get(k["t"]), mu=sh.get(mu_vec), vmu=vmu)


@pytest.mark.parametrize("onepass", [0, 1])
def test_cg_steps_exact(onepass):
    """cg_solve and cg_solve_pair with max_iter = 1 and 2 (a solve is deterministic, so the state after iteration 1 of the
    second solve is the state the first one returns). Iteration 2 uses the other parity slot of <r,z>."""
    N, M = 333, 517
    sh, A, rng = make_block(N, M, 31)
    sh.set_tuning("cg_onepass", onepass)
    tau, gam2 = 2.3, 0.7
    diag = tau * (N - 1) / N + gam2
    v, v2 = rng.standard_normal(M), rng.standard_normal(M)
    sh.set(V_V, v)
    sh.set(V_USER_M1, v2)
    init = dict(r=v, z=v / diag, p=v / diag, mu=np.zeros(M))
    states = [init]
    for k in (1, 2):
        it, _, vmu = sh.cg_solve(V_V, V_X2, tau, gam2, tol=1e-30, max_iter=k)
        assert it == k
        states.append(snapshot(sh, 0, V_X2, vmu))
        cg_step_check(states[k - 1], states[k], v, tau, gam2, diag, M, f"cg_solve onepass={onepass} iteration {k}")
    init2 = dict(r=v2, z=v2 / diag, p=v2 / diag, mu=np.zeros(M))
    pair = [[init], [init2]]
    for k in (1, 2):
        res = sh.cg_solve_pair([V_V, V_USER_M1], [V_X2, V_USER_M0], tau, gam2, tol=1e-30, max_iter=k, onsager_mode=(False, False))
        for s, (vec, rhs) in enumerate(((V_X2, v), (V_USER_M0, v2))):
            assert res[s][0] == k
            pair[s].append(snapshot(sh, s, vec, res[s][2]))
            cg_step_check(pair[s][k - 1], pair[s][k], rhs, tau, gam2, diag, M, f"cg_solve_pair system {s} onepass={onepass} iteration {k}")
    sh.close()


# ---- a long one-pass solve -------------------------------------------------------------------------------------------------
def op_ld(A, mave, msig, N):
    Z = (A.astype(LD) - mave.astype(LD)[:, None]) * msig.astype(LD)[:, None]        # [M, N]
    sq = np.sqrt(LD(N))
    Zt = np.ascontiguousarray(Z.T)
    ax = lambda x: Zt @ x.astype(LD) / sq
    atx = lambda q: Z @ q.astype(LD) / sq
    return ax, atx, np.abs(Zt) / sq


def test_long_onepass_solve_matches_two_pass():
    """N = 2050, M = 3000, gam2 = 1e-2, tol = 1e-10: about 120 CG iterations, so the one-pass solve refreshes q = A p and A r
    three times (every 32 iterations). Both schedules must stop at the same iteration. The true relative residual
    ||v - (tau A^T A + gam2 I) mu|| / ||v||, in long double from the held block and the device's mave / msig, must be below
    2 tol: the recursively updated residual the stopping test reads is below tol, and the two differ by the recurrences'
    rounding, O(u k(Q)) relative (Greenbaum 1997), with k(Q) < 1e4 here. The tracked A mu (track_ax_vecs) and q = A p
    (V_TMP_N0) of the one-pass solve must match A applied to the device's own mu and p entry by entry within
    (j + 1) (M + 16) u sum_k |A_ik| |x_k|, j the iterations since their last recomputation (q: the last refresh; A mu: the
    start of the solve, it is never refreshed), each iteration adding a few roundings per term of the recurrence."""
    N, M = 2050, 3000
    sh, A, rng = make_block(N, M, 21)
    mave, msig = sh.stats()
    tau, gam2, tol = 1.0, 1e-2, 1e-10
    v, u2 = rng.standard_normal(M), rng.standard_normal(M)
    sh.set(V_V, v)
    sh.set(V_USER_M1, u2)
    ax, atx, absA = op_ld(A, mave, msig, N)
    its, mus = {}, {}
    for onepass in (0, 1):
        sh.set_tuning("cg_onepass", onepass)
        res = sh.cg_solve_pair([V_V, V_USER_M1], [V_X2, V_USER_M0], tau, gam2, tol=tol, max_iter=500,
                               onsager_mode=(False, False), track_ax_vecs=(V_USER_N0, V_USER_N1))
        its[onepass] = (res[0][0], res[1][0])
        mus[onepass] = (sh.get(V_X2), sh.get(V_USER_M0))
        for s, (rhs, vec) in enumerate(((v, V_X2), (u2, V_USER_M0))):
            mu = mus[onepass][s]
            Qmu = LD(tau) * atx(ax(mu)) + LD(gam2) * mu.astype(LD)
            rel = np.sqrt(((rhs.astype(LD) - Qmu) ** 2).sum() / (rhs.astype(LD) ** 2).sum())
            assert rel < 2 * tol, (onepass, s, float(rel), res[s])
        if onepass:
            k = max(its[1])
            assert k > 64, its
            p, q = sh.get(V_CG_P), sh.get(V_TMP_N0)
            jq = k % 32
            check(q, ax(p), (jq + 1) * (M + 16) * LD(U) * (absA @ np.abs(p).astype(LD)), f"q = A p, {jq} iterations after a refresh")
            for s, tvec in enumerate((V_USER_N0, V_USER_N1)):
                mu = mus[1][s]
                check(sh.get(tvec), ax(mu), (its[1][s] + 1) * (M + 16) * LD(U) * (absA @ np.abs(mu).astype(LD)),
                      f"tracked A mu, system {s}, {its[1][s]} iterations")
    assert its[0] == its[1], its
    sh.close()


# ---- the whole loo path on constant columns --------------------------------------------------------------------------------
def _write_case(tmp, N, M, rng, nan_probe):
    A = rng.beta(0.3, 0.3, size=(M, N))
    for j, c in enumerate([0.1, 0.7, 0.9532, 1 / 3, 0.0]):
        A[j] = c
    A[5] = 0.1
    A[5, -1] = np.nextafter(0.1, 1.0)                 # nearly constant: not flagged, must still give a finite p in [0, 1]
    if nan_probe:
        A[6] = np.nan                                 # an all-NaN probe: imputed to a constant column
        A[7, ::3] = np.nan
        A[7, 1::3] = 0.7                              # observed values all equal: imputed to a constant column
        A[7, 2::3] = 0.7
    y = rng.standard_normal(N)
    np.ascontiguousarray(A).tofile(os.path.join(tmp, "m.bin"))            # marker-major, N doubles per marker
    with open(os.path.join(tmp, "p.phen"), "w") as f:
        for i, v in enumerate(y):
            f.write(f"{i} {i} {v:.12f}\n")
    np.full(M, 0.01).tofile(os.path.join(tmp, "est_it_1.bin"))
    return A


@pytest.mark.parametrize("missing", ["none", "mean"])
def test_association_loo_on_constant_columns(tmp_path, missing):
    """association_test --pval-method loo through main_meth on a block with constant columns (0.1, 0.7, 0.9532, 1/3, 0), a nearly
    constant one and, under --missing mean, an all-NaN probe and a probe whose observed values are all equal. Constant columns
    get p = 1.0 exactly, every other column a finite p in [0, 1]."""
    N, M = 1000, 40
    rng = np.random.default_rng(12)
    _write_case(str(tmp_path), N, M, rng, missing == "mean")
    argv = ["--run-mode", "association_test", "--pval-method", "loo", "--meth-file", str(tmp_path / "m.bin"), "--phen-file",
            str(tmp_path / "p.phen"), "--estimate-file", str(tmp_path / "est_it_1.bin"), "--N", str(N), "--Mt", str(M), "--out-dir",
            str(tmp_path), "--out-name", "a", "--missing", missing]
    res = subprocess.run([build.MAIN_METH] + argv, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:]
    p = np.fromfile(tmp_path / "a_it_1_pval_loo.bin")
    assert p.size == M
    const = [0, 1, 2, 3, 4] + ([6, 7] if missing == "mean" else [])
    assert np.all(p[const] == 1.0), p[const]
    assert np.all(np.isfinite(p) & (p >= 0) & (p <= 1)), p
