"""Every output entry of the matrix and reduction kernels against the exact value of the same operation, computed in extended
precision (np.longdouble with a 64-bit mantissa) on the inputs the kernel actually read: the block as held (rounded under FP32
storage), the device's own mave / msig and, for w = A t of the fused pass, the device's own t. For an entry y = sum_k term_k of
n terms the kernel must meet

    |got - exact| <= (n + 8) * 2^-53 * sum_k |term_k|   (+ 1e-300 for underflow)

This holds for any summation order and for a few roundings per term, so it does not depend on how a kernel is written. A single
dropped, duplicated or mis-centred term, or an FP32 intermediate, exceeds it. The oracle tests compare whole vectors in the L2
norm, which cannot see an entry that is small because its terms cancel; this bound is per entry.

The blocks put the awkward columns first: constants whose value does not sum exactly in FP64, two nearly constant columns (one
entry off by an ulp or by 1e-3, in the last row, which the kernels read in their scalar tail), a large offset, tiny and huge
magnitudes. The other columns hold bimodal beta values in (0, 1). A constant column must come out exact: mave is its value,
msig is 1, its A^T output is 0.0 and its x_j does not change A x by a single bit."""
import numpy as np
import pytest

from vampomi_b200 import capi
from vampomi_b200.capi import (DIFF2, DOT, SQDEV, V_P1, V_R1, V_R2, V_USER_M0, V_USER_N0, V_USER_N1, V_V, V_X1, V_X2, V_Y, V_Z1,
                               V_Z2)

pytestmark = pytest.mark.gpu

LD = np.longdouble
U = 2.0 ** -53
CONSTANTS = [0.1, 0.7, 0.9532, 1 / 3, 0.25, 0.0]
# N below one 256-bit vector (4 doubles, 8 floats), ragged N, the A^T auto switch (ld >= 4096 from N = 4081), the fused pass's
# steps to a larger cluster (N = 2561, 20481) and its largest N; small M with large N leaves most CTAs and clusters without columns
SHAPES = [(2, 17), (3, 1031), (5, 3), (7, 2), (9, 17), (15, 1031), (16, 1), (33, 17), (2561, 3), (4080, 17), (4081, 1031),
          (20481, 2), (40960, 1)]
XIN, XOUT = [V_X1, V_X2, V_V, V_USER_M0], [V_Z1, V_Z2, V_USER_N0, V_USER_N1]
PIN, POUT = [V_USER_N0, V_USER_N1], [V_R1, V_R2]


@pytest.fixture(autouse=True)
def _extended_precision():
    if np.finfo(np.longdouble).nmant < 63:
        pytest.skip("np.longdouble has fewer than 63 mantissa bits here: no extended-precision reference")


def awkward_columns(N, rng, big):
    cols = [np.full(N, c) for c in CONSTANTS]
    a = np.full(N, 0.1)
    a[-1] = np.nextafter(0.1, 1.0)                    # one ulp off, in the last row
    cols.append(a)
    a = np.full(N, 0.7)
    a[-1] += 1e-3
    cols.append(a)
    cols.append(1e3 + 1e-2 * rng.standard_normal(N))  # mean >> sd
    cols.append(rng.standard_normal(N) / big)
    cols.append(rng.standard_normal(N) * big)
    return cols


def make_block(N, M, storage, seed):
    """(block to upload, block as held). With fewer columns than awkward ones, a seed-dependent window of them. FP32 storage
    cannot hold 1e+-100 (they become 0 and Inf), so its extreme columns are 1e+-30."""
    rng = np.random.default_rng(seed)
    awk = awkward_columns(N, rng, 1e30 if storage == "f32" else 1e100)
    if M < len(awk):
        cols = [awk[(seed + k) % len(awk)] for k in range(M)]
    else:
        cols = awk + list(rng.beta(0.3, 0.3, size=(M - len(awk), N)))
    A = np.array(cols)
    return A, (A.astype(np.float32).astype(np.float64) if storage == "f32" else A)


def constant(held):
    return held.min(axis=1) == held.max(axis=1)


def assert_within(got, exact, absum, n, what):
    """Entry by entry: |got - exact| <= (n + 8) u sum|term| + 1e-300. A NaN fails."""
    err = np.abs(np.asarray(got, dtype=np.float64).astype(LD) - exact)
    bound = (n + 8) * LD(U) * absum + LD(1e-300)
    bad = ~(err <= bound)
    if bad.any():
        i = int(np.argmax(bad))
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} entries outside the bound; entry {i}: got {got[i]!r}, "
                             f"exact {float(exact[i])!r}, error {float(err[i]):.3g}, bound {float(bound[i]):.3g}")


def atx_exact(held, mave, msig, p, split=False):
    """out_j = msig_j * sum_i (a_ij - mave_j) p_i / sqrt(N): exact value and sum of |terms| (scaled alike). split adds the terms
    of the center_split formula sum_i a_ij p_i - mave_j sum_i p_i, whose error grows with |mave_j|, not with the centred
    column: that knob trades accuracy on offset columns for one instruction per element, and the bound shows by how much."""
    N = held.shape[1]
    h, pl = held.astype(LD), p.astype(LD)
    terms = (h - mave.astype(LD)[:, None]) * pl[None, :]
    s = msig.astype(LD) / np.sqrt(LD(N))
    absum = np.abs(terms).sum(axis=1)
    if split:
        absum = absum + np.abs(h * pl[None, :]).sum(axis=1) + np.abs(mave.astype(LD)) * np.abs(pl).sum()
    return s * terms.sum(axis=1), np.abs(s) * absum


def ax_exact(held, mave, msig, x, split=False):
    """out_i = sum_j (a_ij - mave_j) (msig_j x_j) / sqrt(N); split as in atx_exact (sum_j a_ij w_j - sum_j mave_j w_j)."""
    N = held.shape[1]
    h, w = held.astype(LD), msig.astype(LD) * x.astype(LD)
    terms = (h - mave.astype(LD)[:, None]) * w[:, None]
    absum = np.abs(terms).sum(axis=0)
    if split:
        absum = absum + np.abs(h * w[:, None]).sum(axis=0) + np.abs(mave.astype(LD) * w).sum()
    sq = np.sqrt(LD(N))
    return terms.sum(axis=0) / sq, absum / sq


def cancelling(held, mave, p):
    """p with its component along one centred column removed (the large-offset one when present), so that this column's
    A^T output is the residue of a cancellation."""
    idx = [j for j in range(held.shape[0]) if not constant(held[j:j + 1])[0]]
    if not idx:
        return p
    j = 8 if 8 in idx else idx[0]
    c = held[j] - mave[j]
    return p - (c @ p) / (c @ c) * c


def setup(N, M, storage, seed):
    A, held = make_block(N, M, storage, seed)
    sh = capi.Shard(N, M, storage=storage)
    sh.upload(A)
    assert np.array_equal(sh.download(), held)
    sh.compute_stats()
    mave, msig = sh.stats()
    return sh, held, mave, msig, np.random.default_rng(seed + 1)


# ---- statistics --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("alpha", [1.0, 0.5])
@pytest.mark.parametrize("storage", ["f64", "f32"])
@pytest.mark.parametrize("N,M", SHAPES)
def test_stats_exact(N, M, storage, alpha):
    A, held = make_block(N, M, storage, N + M)
    with capi.Shard(N, M, storage=storage) as sh:
        sh.upload(A)
        sh.compute_stats(alpha)
        mave, msig = sh.stats()
    assert_stats_exact(held, mave, msig, alpha)


def assert_stats_exact(held, mave, msig, alpha):
    """mave / msig of the columns of `held` (as held on the device) against their exact values."""
    N = held.shape[1]
    const = constant(held)
    # a constant column: its value and msig = 1, bit for bit (src/data.cpp:275-276 intends sumsqr == 0 for it)
    assert np.array_equal(mave[const], held[const, 0]), (np.nonzero(const)[0], mave[const] - held[const, 0])
    assert np.all(msig[const] == 1.0), msig[const]
    h = held.astype(LD)
    mean = h.sum(axis=1) / N
    delta = (N + 2) * LD(U) * np.abs(h).sum(axis=1) / N
    assert np.all(np.abs(mave.astype(LD) - mean) <= delta), np.abs(mave.astype(LD) - mean) / delta
    nc = ~const
    sd = np.sqrt(((h[nc] - mean[nc, None]) ** 2).sum(axis=1) / (N - 1))
    rel = np.abs(msig[nc].astype(LD) * sd ** LD(alpha) - 1)
    bound = (N + 8) * LD(U) + (delta[nc] / sd) ** 2
    assert np.all(rel <= bound), (np.nonzero(nc)[0], rel / bound)


@pytest.mark.parametrize("storage", ["f64", "f32"])
def test_constant_column_with_a_nan_keeps_nan_statistics(storage):
    """Without --missing mean a NaN spreads into the column's mave and msig, also when all other entries are equal: the exact
    treatment of constant columns must not take such a column for a constant one."""
    N, M = 37, 5
    A = np.full((M, N), 0.1)
    A[0, -1] = np.nan                                 # scalar tail
    A[1, 0] = np.nan                                  # first vector
    A[2, :] = np.nan
    A[3, 5] = -np.nan
    with capi.Shard(N, M, storage=storage) as sh:
        sh.upload(A)
        sh.compute_stats()
        mave, msig = sh.stats()
    assert np.isnan(mave[:4]).all() and np.isnan(msig[:4]).all()
    assert mave[4] == np.float64(np.float32(0.1) if storage == "f32" else 0.1) and msig[4] == 1.0


# ---- A^T p and A x -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", ["f64", "f32"])
@pytest.mark.parametrize("N,M", SHAPES)
def test_atx_exact(N, M, storage):
    sh, held, mave, msig, rng = setup(N, M, storage, N * 3 + M)
    const = constant(held)
    ps = [rng.standard_normal(N)]
    ps.append(cancelling(held, mave, ps[0]))
    want = [atx_exact(held, mave, msig, p) for p in ps]
    for knobs in (dict(), dict(atx_impl=0), dict(atx_impl=1), dict(atx_impl=2)):   # {} = automatic choice; FP32: 1 -> automatic
        for k, v in knobs.items():
            sh.set_tuning(k, v)
        for i, p in enumerate(ps):
            got = sh.ATx(p)
            assert_within(got, *want[i], N, f"ATx {knobs} p{i}")
            assert np.all(got[const] == 0.0), (knobs, got[const])
    sh.set_tuning("atx_impl", 0)
    sh.set_tuning("center_split", 1)
    for i, p in enumerate(ps):
        assert_within(sh.ATx(p), *atx_exact(held, mave, msig, p, split=True), N, f"ATx center_split p{i}")
    sh.close()


@pytest.mark.parametrize("storage", ["f64", "f32"])
@pytest.mark.parametrize("N,M", SHAPES)
def test_ax_exact(N, M, storage):
    sh, held, mave, msig, rng = setup(N, M, storage, N * 5 + M)
    const = constant(held)
    x = rng.standard_normal(M)
    x2 = x.copy()
    x2[const] = rng.standard_normal(int(const.sum())) * 100
    want = ax_exact(held, mave, msig, x)
    for knobs in (dict(ax_impl=0), dict(ax_impl=1)):                                # FP32: 1 runs the LDG kernel
        for k, v in knobs.items():
            sh.set_tuning(k, v)
        got = sh.Ax(x)
        assert_within(got, *want, M, f"Ax {knobs}")
        assert np.array_equal(sh.Ax(x2).view(np.uint64), got.view(np.uint64)), knobs   # a constant column adds exactly 0
    sh.set_tuning("ax_impl", 0)
    sh.set_tuning("center_split", 1)
    assert_within(sh.Ax(x), *ax_exact(held, mave, msig, x, split=True), M, "Ax center_split")
    sh.close()


@pytest.mark.parametrize("storage", ["f64", "f32"])
@pytest.mark.parametrize("N,M", SHAPES)
def test_multi_vector_passes_exact(N, M, storage):
    sh, held, mave, msig, rng = setup(N, M, storage, N * 7 + M)
    const = constant(held)
    xs = [rng.standard_normal(M) * s for s in (1.0, 1e-3, 1e3, 1.0)]
    want = [ax_exact(held, mave, msig, x) for x in xs]
    for K in (1, 2, 3, 4):
        for i in range(K):
            sh.set(XIN[i], xs[i])
        sh.ax_multi_dev(XIN[:K], XOUT[:K])
        for i in range(K):
            assert_within(sh.get(XOUT[i]), *want[i], M, f"ax_multi_dev K={K} vector {i}")
    sh.set(XIN[0], xs[0])
    sh.ax_multi_dev(XIN[:1], XOUT[:1])                # the kernel shape depends on K: compare K = 1 with K = 1
    got = sh.get(XOUT[0])
    x2 = xs[0].copy()
    x2[const] = 7.0
    sh.set(XIN[0], x2)
    sh.ax_multi_dev(XIN[:1], XOUT[:1])
    assert np.array_equal(sh.get(XOUT[0]).view(np.uint64), got.view(np.uint64))
    p = rng.standard_normal(N)
    ps = [p, cancelling(held, mave, p)]
    want = [atx_exact(held, mave, msig, q) for q in ps]
    for K in (1, 2):
        for i in range(K):
            sh.set(PIN[i], ps[i])
        sh.atx_multi_dev(PIN[:K], POUT[:K])
        for i in range(K):
            got = sh.get(POUT[i])
            assert_within(got, *want[i], N, f"atx_multi_dev K={K} vector {i}")
            assert np.all(got[const] == 0.0)
    sh.close()


@pytest.mark.parametrize("N,M", SHAPES)
def test_fused_gram_pass_exact(N, M):
    """t = A^T q and w = A t of vampomi_aat_multi_dev at the default kernel shape and automatic cluster size (FP64 storage
    only); w is checked against A applied to the device's own t."""
    sh, held, mave, msig, rng = setup(N, M, "f64", N * 11 + M)
    assert sh.aat_supported()
    const = constant(held)
    q = rng.standard_normal(N)
    qs = [q, cancelling(held, mave, q)]
    for K in (1, 2):
        for i in range(K):
            sh.set(PIN[i], qs[i])
        sh.aat_multi_dev(PIN[:K], POUT[:K], [V_Z1, V_Z2][:K])
        for i in range(K):
            t = sh.get(POUT[i])
            assert_within(t, *atx_exact(held, mave, msig, qs[i]), N, f"aat t K={K} vector {i}")
            assert np.all(t[const] == 0.0)
            assert_within(sh.get([V_Z1, V_Z2][i]), *ax_exact(held, mave, msig, t), M, f"aat w K={K} vector {i}")
    sh.close()


# ---- reductions --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", ["f64", "f32"])
@pytest.mark.parametrize("N,M", SHAPES)
def test_loo_sums_exact(N, M, storage):
    sh, held, mave, msig, rng = setup(N, M, storage, N * 13 + M)
    w = rng.standard_normal(N)
    sh.set(V_USER_N1, w)
    assert_loo_sums_exact(sh.loo_sums(V_USER_N1), held, w)
    sh.close()


def assert_loo_sums_exact(got, held, w):
    """sum x, sum x^2 and sum x w of the columns of `held` (rows of got) against their exact values."""
    N = held.shape[1]
    h, wl = held.astype(LD), w.astype(LD)
    assert_within(got[:, 0], h.sum(axis=1), np.abs(h).sum(axis=1), N, "sum x")
    assert_within(got[:, 1], (h * h).sum(axis=1), (h * h).sum(axis=1), N, "sum x^2")
    assert_within(got[:, 2], (h * wl).sum(axis=1), np.abs(h * wl).sum(axis=1), N, "sum x w")


@pytest.mark.parametrize("N,M", [(75777, 1), (2, 75776), (33, 1031)])
def test_dots_exact(N, M):
    """16 reductions (MAX_DOTS) of all three kinds in one vampomi_dots call, M- and N-vectors mixed, lengths 1 to 75 777: the
    grid-stride loop of k_dots wraps from 296 x 256 = 75 776 elements on."""
    rng = np.random.default_rng(N + M)
    with capi.Shard(N, M) as sh:
        vals = {}
        for vecs, n in (((V_X1, V_R1, V_R2, V_X2, V_V, V_USER_M0), M), ((V_Y, V_Z1, V_Z2, V_USER_N0, V_USER_N1, V_P1), N)):
            a = rng.standard_normal(n)
            for vec, v in zip(vecs, (a, a + 1e-9 * rng.standard_normal(n), 1e100 * rng.standard_normal(n),
                                     1e-100 * rng.standard_normal(n), 1e3 + rng.standard_normal(n), rng.beta(0.3, 0.3, n))):
                sh.set(vec, v)
                vals[vec] = v
        items = [(DOT, V_X1, V_R1), (DIFF2, V_X1, V_R1), (SQDEV, V_X1, V_R1, 0.7), (DOT, V_Y, V_Z1), (DIFF2, V_Y, V_Z1),
                 (SQDEV, V_Z1, V_Y, 1.3), (DOT, V_R2, V_R2), (DOT, V_X2, V_X2), (DOT, V_R2, V_X2), (DIFF2, V_V, V_USER_M0),
                 (SQDEV, V_V, V_V, 1.0 - 2.0 ** -30), (DOT, V_Z2, V_USER_N0), (DIFF2, V_USER_N0, V_USER_N1),
                 (SQDEV, V_P1, V_USER_N1, -2.0), (DOT, V_V, V_V), (DOT, V_USER_N1, V_P1)]
        got = sh.dots(items)
    for k, it in enumerate(items):
        a, b = vals[it[1]].astype(LD), vals[it[2]].astype(LD)
        if it[0] == DOT:
            exact, absum = (a * b).sum(), np.abs(a * b).sum()
        elif it[0] == DIFF2:
            exact = absum = ((a - b) ** 2).sum()
        else:                                         # (a - s b)^2: the rounding of s b counts against |a| + |s b|
            sb = LD(it[3]) * b
            exact, absum = ((a - sb) ** 2).sum(), ((np.abs(a) + np.abs(sb)) ** 2).sum()
        assert_within(got[k:k + 1], np.array([exact]), np.array([absum]), a.size, f"dots item {k} {it}")
