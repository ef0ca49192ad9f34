"""Parity of every kernel-level entry point of the C ABI against the numpy oracle, on seeded inputs, through ctypes.
Shapes include ragged ones (N not a multiple of 4/16/32, a single marker, fewer markers than CTAs, a constant column)."""
import math

import numpy as np
import pytest

from oracle import vamp_oracle as vo
from vampomi_b200 import capi
from vampomi_b200.capi import (V_ATA_X2, V_USER_M1, V_Z2, DIFF2, DOT, SQDEV, V_ATY, V_BERN, V_P1, V_QINV_BERN, V_R1, V_R2, V_TRUE, V_USER_M0,
                               V_USER_N0, V_USER_N1, V_V, V_X1, V_X1_PREV, V_X2, V_Y, V_Z1, V_Z1HAT)
from helpers import rel_l2

pytestmark = pytest.mark.gpu

SHAPES = [(300, 800), (333, 517), (1000, 64), (64, 1), (2050, 300), (4100, 129), (17, 40)]


def make(N, M, seed=0, offset=0.0, scale=1.0):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((M, N)) * scale + offset
    y = rng.standard_normal(N)
    sh = capi.Shard(N, M)
    sh.upload(A)
    sh.compute_stats()
    return sh, A, y, rng


@pytest.mark.parametrize("N,M", SHAPES)
def test_upload_download_stats_ax_atx(N, M):
    sh, A, y, rng = make(N, M, seed=N + M, offset=0.5, scale=0.1)      # methylation-like: mean 0.5, small spread
    assert np.array_equal(sh.download(), A)
    d = vo.Data(A, y)
    mave, msig = sh.stats()
    assert np.allclose(mave, d.mave, rtol=1e-13, atol=1e-15) and np.allclose(msig, d.msig, rtol=1e-12)
    p, x = rng.standard_normal(N), rng.standard_normal(M)
    assert rel_l2(sh.ATx(p), d.ATx(p)) < 1e-12
    assert rel_l2(sh.Ax(x), d.Ax(x)) < 1e-12
    # run-to-run bitwise reproducibility (fixed-order reductions, no atomics on data)
    assert np.array_equal(sh.Ax(x), sh.Ax(x)) and np.array_equal(sh.ATx(p), sh.ATx(p))
    # every A^T p implementation (warp, CTA-cooperative) and the bulk-copy (cp.async.bulk + mbarrier) pipelines on the
    # same ragged shapes
    for impl in (0, 2):
        sh.set_tuning("atx_impl", impl)
        assert rel_l2(sh.ATx(p), d.ATx(p)) < 1e-12
    sh.set_tuning("ax_impl", 1)
    sh.set_tuning("atx_impl", 1)
    assert rel_l2(sh.ATx(p), d.ATx(p)) < 1e-12
    assert rel_l2(sh.Ax(x), d.Ax(x)) < 1e-12
    assert np.array_equal(sh.Ax(x), sh.Ax(x)) and np.array_equal(sh.ATx(p), sh.ATx(p))
    sh.close()


def test_constant_column_and_alpha_scale():
    N, M = 200, 50
    rng = np.random.default_rng(3)
    A = rng.standard_normal((M, N))
    A[7] = 0.25                                   # constant marker -> msig = 1 (src/data.cpp:275-276)
    sh = capi.Shard(N, M)
    sh.upload(A)
    sh.compute_stats(1.0)
    assert sh.stats()[1][7] == 1.0
    sh.compute_stats(0.5)                         # src/data.cpp:273-274
    want = vo.marker_stats(A, 0.5)[1]
    assert np.allclose(sh.stats()[1], want, rtol=1e-12)
    sh.close()


@pytest.mark.parametrize("knobs", [dict(ax_rv=1, ax_unroll=2), dict(ax_rv=1, ax_unroll=8), dict(ax_rv=2, ax_unroll=2),
                                   dict(ax_rv=2, ax_unroll=8), dict(ax_rv=4, ax_unroll=2), dict(ax_rv=4, ax_unroll=4),
                                   dict(ax_ctas_per_sm=1), dict(ax_ctas_per_sm=7),
                                   dict(atx_impl=0, atx_cols=1, atx_unroll=2), dict(atx_impl=0, atx_cols=1, atx_unroll=8),
                                   dict(atx_impl=0, atx_cols=2, atx_unroll=2), dict(atx_impl=0, atx_cols=2, atx_unroll=8),
                                   dict(atx_impl=0, atx_cols=4, atx_unroll=2), dict(atx_impl=0, atx_cols=4, atx_unroll=4),
                                   dict(atx_impl=0, atx_ctas_per_sm=1), dict(atx_impl=0, atx_ctas_per_sm=9), dict(atx_ctas_per_sm=9),
                                   dict(center_split=1, atx_impl=0), dict(center_split=1, ax_rv=1, ax_unroll=8, atx_impl=0, atx_cols=1, atx_unroll=2),
                                   dict(atx_impl=2), dict(atx_impl=2, atx_cols=1, atx_unroll=8), dict(atx_impl=2, atx_cols=4, atx_unroll=2),
                                   dict(atx_impl=2, atx_cols=2, atx_unroll=2, atx_ctas_per_sm=5),
                                   dict(ld_hint=1), dict(ld_hint=2), dict(ld_hint=3), dict(interleave=1), dict(interleave=1, ax_rv=1, ax_unroll=8, atx_cols=4),
                                   dict(interleave=1, ax_ctas_per_sm=7, atx_ctas_per_sm=5),
                                   dict(ax_impl=1), dict(atx_impl=1), dict(ax_impl=1, ax_ctas_per_sm=1), dict(atx_impl=1, atx_ctas_per_sm=1)])
def test_kernel_variants_agree(knobs):
    N, M = 4100, 1033
    sh, A, y, rng = make(N, M, seed=5)
    d = vo.Data(A, y)
    p, x = rng.standard_normal(N), rng.standard_normal(M)
    for k, v in knobs.items():
        sh.set_tuning(k, v)
    assert rel_l2(sh.ATx(p), d.ATx(p)) < 1e-12
    assert rel_l2(sh.Ax(x), d.Ax(x)) < 1e-12
    sh.close()


def test_generate_iid_is_sharding_invariant_and_matches_restatement():
    N, Mt = 257, 91
    full = capi.Shard(N, Mt)
    full.generate_iid(42)
    A = full.download()
    assert np.allclose(A, vo.generate_iid_block(42, 0, Mt, N), rtol=0, atol=1e-13)
    assert abs(A.mean()) < 0.02 and abs(A.std() - 1) < 0.02
    for rank in range(3):
        part = capi.Shard(N, Mt, nranks=3, rank=rank, nccl_id=False)
        part.generate_iid(42)
        assert np.array_equal(part.download(), A[part.S:part.S + part.M])     # identical bits for any shard count
        part.close()
    full.close()


def test_load_file_reads_the_shard_block(tmp_path):
    N, Mt = 123, 77
    rng = np.random.default_rng(1)
    A = rng.standard_normal((Mt, N))
    A.tofile(tmp_path / "a.bin")
    for rank in range(2):
        sh = capi.Shard(N, Mt, nranks=2, rank=rank, nccl_id=False)
        sh.load_file(str(tmp_path / "a.bin"))
        assert np.array_equal(sh.download(), A[sh.S:sh.S + sh.M])            # byte offset S*N*8, src/data.cpp:134
        sh.close()
    # single reader, many readers and more readers than 32 MB column groups give the same block
    sh = capi.Shard(N, Mt)
    for threads in (1, 3, 16):
        sh.set_tuning("load_threads", threads)
        sh.load_file(str(tmp_path / "a.bin"))
        assert np.array_equal(sh.download(), A)
    sh.close()
    # several 32 MB column groups per reader (the ring wraps around), buffered and O_DIRECT reads (4 KB-aligned spans around
    # columns that are not 4 KB-aligned themselves; falls back to buffered reads where the file system has no O_DIRECT), a
    # shard that starts in the middle of the file, padded (N = 4099) and unpadded (N = 4096) column strides
    for N2, Mt2 in ((4099, 5000), (4096, 3000)):
        B = np.random.default_rng(2).standard_normal((Mt2, N2))
        B.tofile(tmp_path / "b.bin")
        for rank, nranks in ((0, 1), (1, 3)):
            sh = capi.Shard(N2, Mt2, nranks=nranks, rank=rank, nccl_id=False)
            for direct, threads, depth in ((0, 2, 2), (1, 2, 3), (1, 1, 8), (0, 5, 3)):
                sh.set_tuning("load_direct", direct); sh.set_tuning("load_threads", threads); sh.set_tuning("load_depth", depth)
                sh.fill(0, 0.0)
                sh.load_file(str(tmp_path / "b.bin"))
                assert np.array_equal(sh.download(), B[sh.S:sh.S + sh.M]), (N2, rank, direct, threads, depth)
            sh.close()
    sh = capi.Shard(N, Mt + 1)
    with pytest.raises(capi.VampomiError, match="too short"):
        sh.load_file(str(tmp_path / "a.bin"))
    with pytest.raises(capi.VampomiError, match="could not open"):
        sh.load_file(str(tmp_path / "missing.bin"))
    sh.close()


def test_two_shards_sum_to_the_full_product():
    N, Mt = 500, 301
    rng = np.random.default_rng(9)
    A, x = rng.standard_normal((Mt, N)), rng.standard_normal(Mt)
    full = capi.Shard(N, Mt)
    full.upload(A)
    full.compute_stats()
    total = np.zeros(N)
    for r in range(2):
        M, S = capi.divide_work(Mt, 2, r)
        part = capi.Shard(N, M)                       # an independent single-rank context over the shard's columns
        part.upload(A[S:S + M])
        part.compute_stats()
        total += part.Ax(x[S:S + M])
        part.close()
    assert rel_l2(total, full.Ax(x)) < 1e-13
    full.close()


def test_vector_ops_and_dots():
    N, M = 300, 1000
    sh, A, y, rng = make(N, M, seed=2)
    a, b = rng.standard_normal(M), rng.standard_normal(M)
    sh.set(V_X1, a)
    sh.set(V_R1, b)
    sh.set(V_Y, y)
    sh.lincomb(V_R2, 1.7, V_X1, -0.3, V_R1, 2.5)
    assert np.allclose(sh.get(V_R2), (1.7 * a - 0.3 * b) / 2.5, rtol=1e-15)
    assert np.allclose(sh.get(V_X1, divisor=math.sqrt(N)), a / math.sqrt(N), rtol=1e-15)
    sh.copy(V_X2, V_X1)
    assert np.array_equal(sh.get(V_X2), a)
    # asynchronous read-out: the value at begin() is what arrives, whatever happens to the vector afterwards
    sh.dump_begin(0, V_X1, math.sqrt(N))
    sh.dump_begin(1, V_Y)
    sh.fill(V_X1, -1.0)
    with pytest.raises(capi.VampomiError):
        sh.dump_begin(0, V_R1)                     # slot still pending
    assert np.allclose(sh.dump_wait(0), a / math.sqrt(N), rtol=1e-15) and np.array_equal(sh.dump_wait(1), y)
    with pytest.raises(capi.VampomiError):
        sh.dump_wait(0, np.empty(M))               # nothing pending
    sh.set(V_X1, a)
    sh.fill(V_V, 3.0)
    got = sh.dots([(DOT, V_X1, V_R1), (DIFF2, V_X1, V_R1), (SQDEV, V_X1, V_R1, 2.0), (DOT, V_Y, V_Y), (DOT, V_V, V_V)])
    want = [a @ b, ((a - b) ** 2).sum(), ((a - 2 * b) ** 2).sum(), y @ y, 9.0 * M]
    assert np.allclose(got, want, rtol=1e-13)
    sh.close()


def test_probe_matches_counter_hash():
    sh = capi.Shard(100, 997, nranks=3, rank=1, nccl_id=False)
    sh.draw_probe(12345, 4)
    want = vo.probe_signs(12345, 4, sh.S, sh.M) / math.sqrt(997)
    assert np.array_equal(sh.get(V_BERN), want)
    sh.close()


def mixture(L):
    """(probs, vars) of L components: the reference's defaults, or a spike and L - 1 slabs with geometric variances."""
    if L is None:
        return list(vo.DEFAULT_PROBS), list(vo.DEFAULT_VARS)
    slabs = 0.5 ** np.arange(1, L)
    return [0.9] + list(0.1 * slabs / slabs.sum()), [0.0] + list(np.geomspace(1e-6, 1.0, L - 1))


# The vector kernels' grid-stride loops wrap from 296 x 256 = 75 776 elements on, so M = 75 777 and 200 003 give a thread two
# or more markers; L = 32 (MAX_MIX) fills 63 of the 64 packed sums of k_em_sums. The marker block is never read by these kernels
# and the oracle's mixture formulas need N only, so neither side gets a matrix of M columns.
VECTOR_MS = (5000, 75777, 200003)
MIXTURES = (None, 2, 32)


@pytest.mark.parametrize("gam1", [1e-6, 0.37, 25.0, 1e12])
def test_denoiser_matches_oracle(gam1):
    N = 200
    rng = np.random.default_rng(4)
    data = vo.Data(rng.standard_normal((2, N)), rng.standard_normal(N))
    for M in VECTOR_MS:
        sh = capi.Shard(N, M)
        r1 = rng.standard_normal(M) * 3
        r1[:5] = [0.0, 1e-300, -40.0, 40.0, 1e3]
        prev = rng.standard_normal(M)
        for L in MIXTURES:
            probs, vars_ = mixture(L)
            vars_int = np.array(vars_) * N
            o = vo.Vamp(data, vars=vars_, probs=probs)
            for damp in (False, True):
                sh.set(V_R1, r1)
                sh.set(V_X1, prev)
                s = sh.denoise(gam1, np.array(probs), vars_int, damp=damp, rho=0.3)
                g, gd = o.g1(r1, gam1), o.g1d(r1, gam1)
                want = 0.3 * g + 0.7 * prev if damp else g
                # g1 = y + sigma*pkd/pk cancels against y when gam1 is tiny (|g1| ~ 1e-7 |y| at gam1 = 1e-6): the error budget
                # is a few ulps of the INPUT magnitude, not of the output
                err = np.linalg.norm(sh.get(V_X1) - want)
                assert err <= 1e-12 * np.linalg.norm(want) + 2e-15 * np.linalg.norm(r1[np.abs(r1) < 100]), (M, L, damp, err, np.linalg.norm(want))
                assert np.array_equal(sh.get(V_X1_PREV), prev), (M, L, damp)
                assert abs(s - gd.sum()) <= 1e-9 * max(abs(gd).sum(), 1.0), (M, L, damp)   # gd cancels to ~1e-8 per term when gam1 is tiny
        sh.close()


def test_em_sums_match_oracle():
    N = 150
    rng = np.random.default_rng(6)
    data = vo.Data(rng.standard_normal((2, N)), rng.standard_normal(N))
    for M in (4000,) + VECTOR_MS:
        sh = capi.Shard(N, M)
        r1 = rng.standard_normal(M) * 2
        sh.set(V_R1, r1)
        for L in MIXTURES:
            probs, vars_ = mixture(L)
            o = vo.Vamp(data, probs=probs, vars=vars_)
            probs, vars_int = list(o.probs), list(o.vars)
            lam = 1 - probs[0]
            omegas = [probs[0]] + [p / lam for p in probs[1:]]
            s_pin, s_beta, s_gam = o.em_sums(r1, 0.8, lam, omegas, vars_int)
            got = sh.em_sums(0.8, lam, omegas, vars_int)
            L = len(probs)
            assert got.size == 2 * L - 1
            assert np.allclose(got[0], s_pin, rtol=1e-12), (M, L)
            assert np.allclose(got[1:L], s_beta, rtol=1e-11, atol=1e-300), (M, L)
            assert np.allclose(got[L:], s_gam, rtol=1e-11, atol=1e-300), (M, L)
        sh.close()


def test_probit_z_channel_matches_oracle():
    N, M = 3000, 40
    sh, A, y, rng = make(N, M, seed=7)
    yb = (rng.random(N) > 0.5).astype(float)
    p1 = rng.standard_normal(N) * 4
    p1[:4] = [0.0, 30.0, -30.0, 12.0]             # hits both erfcx clamps of src/utilities.cpp:295-298
    sh.set(V_Y, yb)
    sh.set(V_P1, p1)
    for tau1 in (1e-2, 1.3, 50.0):
        s = sh.probit_zdenoise(tau1)
        want_z = vo.g1_bin_class(p1, tau1, yb)
        want_d = vo.g1d_bin_class(p1, tau1, yb)
        got_z = sh.get(V_Z1HAT)
        fin = np.isfinite(want_z)
        assert np.array_equal(np.isfinite(got_z), fin)
        assert np.allclose(got_z[fin], want_z[fin], rtol=1e-12, atol=1e-300)
        if np.isfinite(want_d.sum()):
            assert abs(s - want_d.sum()) <= 1e-11 * abs(want_d).sum()
    sh.close()


@pytest.mark.parametrize("onsager", [False, True])
def test_cg_matches_oracle(onsager):
    N, M = 400, 1000
    sh, A, y, rng = make(N, M, seed=8)
    d = vo.Data(A, y)
    o = vo.Vamp(d, CG_err_tol=1e-7)
    o.gam2 = 1.9
    tau = 2.3
    v = rng.standard_normal(M)
    mu0 = rng.standard_normal(M) * 0.1
    sh.set(V_V, v)
    # cold start
    mu = o.precondCG_solver(v, None, tau, 0 if onsager else 1)
    it, rel, vmu = sh.cg_solve(V_V, V_X2, tau, 1.9, warm_start=False, tol=1e-7, max_iter=500, onsager_mode=onsager)
    assert it == o.cg_iters[-1][2]
    assert rel_l2(sh.get(V_X2), mu) < 1e-11
    assert abs(vmu - v @ mu) < 1e-11 * abs(v @ mu)
    # warm start (src/vamp.cpp:311): same fixed point, fewer iterations
    mu_w = o.precondCG_solver(v, mu0, tau, 1)
    sh.set(V_X2, mu0)
    it_w, rel_w, _ = sh.cg_solve(V_V, V_X2, tau, 1.9, warm_start=True, tol=1e-7, max_iter=500)
    assert it_w == o.cg_iters[-1][2] and rel_l2(sh.get(V_X2), mu_w) < 1e-11
    # iteration cap (CG_max_iter) and different look-ahead depths give the same answer
    it_c, _, _ = sh.cg_solve(V_V, V_X2, tau, 1.9, tol=1e-30, max_iter=3)
    assert it_c == 3
    for depth in (1, 4):
        sh.set_tuning("cg_depth", depth)
        it_d, _, _ = sh.cg_solve(V_V, V_QINV_BERN, tau, 1.9, tol=1e-7, max_iter=500, onsager_mode=onsager)
        assert it_d == it and rel_l2(sh.get(V_QINV_BERN), mu) < 1e-11
    sh.close()


def test_association_pvalues_match_oracle():
    N, M = 300, 700
    sh, A, y, rng = make(N, M, seed=10, offset=0.4, scale=0.2)
    d = vo.Data(A, y)
    r1 = rng.standard_normal(M) * 0.2
    r1[:3] = [0.0, -5.0, 5.0]
    got = sh.pvals_se(r1, 3.3)
    assert np.allclose(got, vo.pvals_se(r1, 3.3, N), rtol=1e-12, atol=1e-300)
    # loo: device sums over the RAW columns, host algebra of src/data.cpp:404-414
    x1 = rng.standard_normal(M) * 0.3
    z1 = d.Ax(x1)
    w = y - z1
    sh.set(V_USER_N1, w)
    sums = sh.loo_sums(V_USER_N1)
    assert np.allclose(sums[:, 0], A.sum(1), rtol=1e-12) and np.allclose(sums[:, 1], (A * A).sum(1), rtol=1e-12)
    assert np.allclose(sums[:, 2], A @ w, rtol=1e-10, atol=1e-10)
    sh.close()


# ---------------------------------------------------------------------------------------------------------------------
MULTI_KNOBS = [dict(), dict(multi_ax_rv=1, multi_ax_unroll=2), dict(multi_ax_rv=1, multi_ax_unroll=8), dict(multi_ax_rv=2, multi_ax_unroll=2),
               dict(multi_ax_rv=2, multi_ax_unroll=4), dict(multi_atx_impl=0), dict(multi_atx_cols=1, multi_atx_unroll=2),
               dict(multi_atx_cols=1, multi_atx_unroll=4), dict(multi_atx_cols=2, multi_atx_unroll=4), dict(multi_atx_cols=4, multi_atx_unroll=2),
               dict(multi_atx_tile=256), dict(multi_atx_tile=1000, atx_ctas_per_sm=3), dict(ax_ctas_per_sm=5)]


@pytest.mark.parametrize("storage", ["f64", "f32"])
@pytest.mark.parametrize("N,M", SHAPES + [(9000, 77)])
def test_multi_vector_passes_match_oracle(N, M, storage):
    """One read of the marker block for K vectors (vampomi_ax_multi_dev / vampomi_atx_multi_dev): every vector must get the
    product the single-vector call (and the oracle) gives, for every kernel shape, on ragged sizes."""
    rng = np.random.default_rng(N * 3 + M)
    A = rng.standard_normal((M, N)) * 0.1 + 0.5
    if storage == "f32":
        A = A.astype(np.float32).astype(np.float64)
    y = rng.standard_normal(N)
    sh = capi.Shard(N, M, storage=storage)
    sh.upload(A)
    sh.compute_stats()
    d = vo.Data(A, y)
    xs = [rng.standard_normal(M) for _ in range(4)]
    ps = [rng.standard_normal(N) for _ in range(2)]
    xin, xout = [V_X1, V_X2, V_V, V_USER_M0], [V_Z1, V_Z2, V_USER_N0, V_USER_N1]
    pin, pout = [V_USER_N0, V_USER_N1], [V_R1, V_R2]
    want_ax = [d.Ax(x) for x in xs]
    want_atx = [d.ATx(p) for p in ps]
    for knobs in MULTI_KNOBS:
        for k, v in knobs.items():
            sh.set_tuning(k, v)
        for K in (1, 2, 3, 4):
            for i in range(4):
                sh.set(xin[i], xs[i])
                sh.fill(xout[i], -7.0)
            sh.ax_multi_dev(xin[:K], xout[:K])
            for i in range(K):
                assert rel_l2(sh.get(xout[i]), want_ax[i]) < 1e-12, (knobs, K, i)
            for i in range(K, 4):
                assert np.all(sh.get(xout[i]) == -7.0)           # untouched
        for K in (1, 2):
            for i in range(2):
                sh.set(pin[i], ps[i])
                sh.fill(pout[i], -7.0)
            sh.atx_multi_dev(pin[:K], pout[:K])
            for i in range(K):
                assert rel_l2(sh.get(pout[i]), want_atx[i]) < 1e-12, (knobs, K, i)
            for i in range(K, 2):
                assert np.all(sh.get(pout[i]) == -7.0)
        for k in knobs:
            sh.set_tuning(k, 1 if k == "multi_atx_impl" else 0)
    # bitwise reproducible from run to run
    sh.ax_multi_dev(xin[:2], xout[:2]); a = sh.get(xout[1]).copy()
    sh.ax_multi_dev(xin[:2], xout[:2]); assert np.array_equal(a, sh.get(xout[1]))
    sh.atx_multi_dev(pin, pout); b = sh.get(pout[1]).copy()
    sh.atx_multi_dev(pin, pout); assert np.array_equal(b, sh.get(pout[1]))
    with pytest.raises(capi.VampomiError):
        sh.ax_multi_dev([V_X1, V_X2], [V_Z1, V_Z1])              # outputs must be distinct
    with pytest.raises(capi.VampomiError):
        sh.atx_multi_dev([V_USER_N0, V_USER_N1, V_Z1], [V_R1, V_R2, V_V])   # at most two
    with pytest.raises(capi.VampomiError):
        sh.ax_multi_dev([V_Z1], [V_X1])                          # wrong kinds
    sh.close()


@pytest.mark.parametrize("N,M", SHAPES + [(9000, 77), (20000, 300), (20480, 40), (20496, 40), (33000, 31), (40960, 10)])
def test_fused_gram_pass_matches_the_two_products_at_every_cluster_size(N, M):
    """vampomi_aat_multi_dev: t = A^T q and w = A t from ONE read of the marker block (kernels_gram.cu). Both must equal what
    the two separate products (and the oracle) give, for the default cluster size and every cluster size that holds N, for
    one and two vectors, on ragged sizes; untouched outputs stay untouched; results are bitwise reproducible."""
    rng = np.random.default_rng(N * 7 + M)
    A = rng.standard_normal((M, N)) * 0.1 + 0.5
    y = rng.standard_normal(N)
    sh = capi.Shard(N, M)
    sh.upload(A)
    sh.compute_stats()
    assert sh.aat_supported()
    d = vo.Data(A, y)
    qs = [rng.standard_normal(N) for _ in range(2)]
    want_t = [d.ATx(q) for q in qs]
    want_w = [d.Ax(t) for t in want_t]
    qin, tout, wout = [V_USER_N0, V_USER_N1], [V_R1, V_R2], [V_Z1, V_Z2]
    ld = (N + 15) // 16 * 16
    smallest = -(-ld // 2560)                                        # a CTA holds 2 560 rows of a column
    ran = 0
    for cs in [0] + list(range(smallest, 17)):                       # 0: the default, the smallest cluster that holds N
        sh.set_tuning("gram_cluster", cs)
        for K in (1, 2):
            for i in range(2):
                sh.set(qin[i], qs[i])
                sh.fill(tout[i], -7.0)
                sh.fill(wout[i], -7.0)
            sh.aat_multi_dev(qin[:K], tout[:K], wout[:K])
            for i in range(K):
                assert rel_l2(sh.get(tout[i]), want_t[i]) < 1e-12, (cs, K, i)
                assert rel_l2(sh.get(wout[i]), want_w[i]) < 1e-12, (cs, K, i)
            for i in range(K, 2):
                assert np.all(sh.get(tout[i]) == -7.0) and np.all(sh.get(wout[i]) == -7.0)
            ran += 1
    assert ran == 2 * (18 - smallest) and ran >= 4
    if smallest > 1:
        sh.set_tuning("gram_cluster", smallest - 1)                  # too few CTAs to hold a column
        with pytest.raises(capi.VampomiError):
            sh.aat_multi_dev(qin, tout, wout)
    sh.set_tuning("gram_cluster", 0)
    for clusters in (1, 3, 1000):                                    # any number of column chunks, more than there are columns included
        sh.set_tuning("gram_clusters", clusters)
        sh.aat_multi_dev(qin, tout, wout)
        assert rel_l2(sh.get(tout[1]), want_t[1]) < 1e-12 and rel_l2(sh.get(wout[1]), want_w[1]) < 1e-12
    sh.set_tuning("gram_clusters", 0)
    sh.aat_multi_dev(qin, tout, wout); a, b = sh.get(tout[1]).copy(), sh.get(wout[0]).copy()
    sh.aat_multi_dev(qin, tout, wout); assert np.array_equal(a, sh.get(tout[1])) and np.array_equal(b, sh.get(wout[0]))
    c0 = sh.counters(reset=True)
    sh.aat_multi_dev(qin, tout, wout)
    assert sh.counters()["matrix_passes"] == 1                       # two products, two vectors: ONE read of the block
    with pytest.raises(capi.VampomiError):
        sh.aat_multi_dev([V_USER_N0, V_USER_N1], [V_R1, V_R2], [V_Z1, V_Z1])
    with pytest.raises(capi.VampomiError):
        sh.aat_multi_dev([V_USER_N0], [V_R1], [V_USER_N0])
    with pytest.raises(capi.VampomiError):
        sh.aat_multi_dev([V_R1], [V_USER_N0], [V_Z1])
    sh.close()
    with capi.Shard(64, 10, storage="f32") as s32:
        assert not s32.aat_supported()


@pytest.mark.parametrize("N,M,cluster", [(400, 1000, 0), (333, 517, 4), (2050, 300, 8), (6000, 200, 0)])
def test_onepass_cg_equals_two_pass_cg(N, M, cluster):
    """Knob cg_onepass: the same solves with ONE read of the block per CG iteration (q = A p advanced by its recurrence, the
    fused pass delivering A^T q and A A^T q). Iteration counts must be the oracle's, solutions and the tracked A sol must
    agree to rounding, and the pass count is max(k0, k1) + 1 (+ the refresh passes of long solves)."""
    sh, A, y, rng = make(N, M, seed=N + 3)
    d = vo.Data(A, y)
    o = vo.Vamp(d, CG_err_tol=1e-7)
    gam2, tau = 1.9, 2.3
    o.gam2 = gam2
    v, u, x1 = rng.standard_normal(M), np.sign(rng.standard_normal(M)) / math.sqrt(M), rng.standard_normal(M)
    mu0 = rng.standard_normal(M) * 0.1
    sh.set(V_V, v); sh.set(V_BERN, u); sh.set(V_X1, x1)
    want0 = o.precondCG_solver(v, None, tau, 1); k0 = o.cg_iters[-1][2]
    want1 = o.precondCG_solver(u, None, tau, 0); k1 = o.cg_iters[-1][2]
    want_w = o.precondCG_solver(v, mu0, tau, 1); kw = o.cg_iters[-1][2]
    sh.set_tuning("cg_onepass", 1)
    sh.set_tuning("gram_cluster", cluster)
    for depth, refresh in ((2, 0), (1, 0), (5, 3)):
        sh.set_tuning("cg_depth", depth)
        sh.set_tuning("gram_refresh", refresh)
        sh.fill(V_Z1, 0.0)
        sh.counters(reset=True)
        res = sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_QINV_BERN], tau, gam2, tol=1e-7, extra=(V_X1, V_Z1), track_ax_vecs=(V_Z2, V_USER_N0))
        assert (res[0][0], res[1][0]) == (k0, k1)
        x2, w = sh.get(V_X2), sh.get(V_QINV_BERN)
        assert rel_l2(x2, want0) < 1e-11 and rel_l2(w, want1) < 1e-11
        assert abs(res[1][2] - u @ want1) < 1e-11 * abs(u @ want1)
        assert rel_l2(sh.get(V_Z1), d.Ax(x1)) < 1e-12
        assert rel_l2(sh.get(V_Z2), d.Ax(x2)) < 1e-12 and rel_l2(sh.get(V_USER_N0), d.Ax(w)) < 1e-12
        kmax = max(k0, k1)
        assert sh.counters()["matrix_passes"] == kmax + 1 + ((kmax - 1) // refresh if refresh else 0)
    sh.set_tuning("gram_refresh", 0)
    # single-system entry point and a warm start (A^T A mu0 computed inside: two more passes)
    it_s, _, _ = sh.cg_solve(V_V, V_USER_M0, tau, gam2, tol=1e-7)
    assert it_s == k0 and rel_l2(sh.get(V_USER_M0), want0) < 1e-11
    sh.set(V_X2, mu0)
    sh.counters(reset=True)
    res = sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_QINV_BERN], tau, gam2, warm_start=(True, False), tol=1e-7)
    assert (res[0][0], res[1][0]) == (kw, k1) and rel_l2(sh.get(V_X2), want_w) < 1e-11
    assert sh.counters()["matrix_passes"] == max(kw, k1) + 3
    res = sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_QINV_BERN], tau, gam2, tol=1e-30, max_iter=3, onsager_mode=(False, False))
    assert (res[0][0], res[1][0]) == (3, 3)
    sh.close()


@pytest.mark.parametrize("N,M", [(400, 1000), (333, 517), (2050, 300)])
def test_paired_solve_equals_two_single_solves(N, M):
    """vampomi_cg_solve_pair: two systems with one operator in lock-step. Each system must stop after exactly the
    iterations the single solve (and the oracle) takes and return the same solution; the rider A x on the first pass and a
    warm start from a cached A^T A x must behave like their separate calls."""
    sh, A, y, rng = make(N, M, seed=N + 1)
    d = vo.Data(A, y)
    o = vo.Vamp(d, CG_err_tol=1e-7)
    gam2, tau = 1.9, 2.3
    o.gam2 = gam2
    v, u, x1 = rng.standard_normal(M), np.sign(rng.standard_normal(M)) / math.sqrt(M), rng.standard_normal(M)
    mu0 = rng.standard_normal(M) * 0.1
    sh.set(V_V, v); sh.set(V_BERN, u); sh.set(V_X1, x1)
    want0 = o.precondCG_solver(v, None, tau, 1); k0 = o.cg_iters[-1][2]
    want1 = o.precondCG_solver(u, None, tau, 0); k1 = o.cg_iters[-1][2]
    for depth in (2, 1, 5):
        sh.set_tuning("cg_depth", depth)
        sh.fill(V_Z1, 0.0)
        c0 = sh.counters(reset=True)
        res = sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_QINV_BERN], tau, gam2, tol=1e-7, extra=(V_X1, V_Z1))
        assert (res[0][0], res[1][0]) == (k0, k1)
        assert rel_l2(sh.get(V_X2), want0) < 1e-11 and rel_l2(sh.get(V_QINV_BERN), want1) < 1e-11
        assert abs(res[1][2] - u @ want1) < 1e-11 * abs(u @ want1)
        assert rel_l2(sh.get(V_Z1), d.Ax(x1)) < 1e-12
        assert sh.counters()["matrix_passes"] == 2 * max(k0, k1)            # one pass per product pair, idle look-ahead not counted
    # the same answers as the single-system entry point, to rounding of the reduction order
    it_s, _, _ = sh.cg_solve(V_V, V_USER_M0, tau, gam2, tol=1e-7)
    assert it_s == k0 and rel_l2(sh.get(V_USER_M0), sh.get(V_X2)) < 1e-12
    # warm start of system 0: (a) A^T A mu0 computed inside, (b) handed in from a multi pass
    want_w = o.precondCG_solver(v, mu0, tau, 1); kw = o.cg_iters[-1][2]
    sh.set(V_X2, mu0)
    res = sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_QINV_BERN], tau, gam2, warm_start=(True, False), tol=1e-7)
    assert (res[0][0], res[1][0]) == (kw, k1) and rel_l2(sh.get(V_X2), want_w) < 1e-11
    sh.set(V_X2, mu0)
    sh.ax_multi_dev([V_X2], [V_Z2])
    sh.atx_multi_dev([V_Z2], [V_ATA_X2])
    c = sh.counters(reset=True)
    res = sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_QINV_BERN], tau, gam2, warm_start=(True, False), warm_ata_vecs=(V_ATA_X2, -1), tol=1e-7)
    assert (res[0][0], res[1][0]) == (kw, k1) and rel_l2(sh.get(V_X2), want_w) < 1e-11
    assert sh.counters()["matrix_passes"] == 2 * max(kw, k1)
    # products of the solutions kept by the solve itself: A sol (track_ax_vecs) and A^T A sol = (rhs - r - gam2 sol)/tau
    sh.set(V_X2, mu0)
    sh.ax_multi_dev([V_X2], [V_Z2])                                             # A mu0 on entry (warm system)
    sh.fill(V_USER_N0, 123.0)                                                   # cold system: zeroed by the solve
    res = sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_QINV_BERN], tau, gam2, warm_start=(True, False), tol=1e-7,
                           track_ax_vecs=(V_Z2, V_USER_N0))
    assert (res[0][0], res[1][0]) == (kw, k1)
    x2, w = sh.get(V_X2), sh.get(V_QINV_BERN)
    assert rel_l2(sh.get(V_Z2), d.Ax(x2)) < 1e-13 and rel_l2(sh.get(V_USER_N0), d.Ax(w)) < 1e-13
    sh.lincomb(V_ATA_X2, 1.0, V_V, -1.0, capi.V_CG_R, 1.0)
    sh.lincomb(V_ATA_X2, 1.0, V_ATA_X2, -gam2, V_X2, tau)
    sh.lincomb(V_USER_M0, 1.0, V_BERN, -1.0, capi.V_CG2_R, 1.0)
    sh.lincomb(V_USER_M0, 1.0, V_USER_M0, -gam2, V_QINV_BERN, tau)
    assert rel_l2(sh.get(V_ATA_X2), d.ATx(d.Ax(x2))) < 1e-12 and rel_l2(sh.get(V_USER_M0), d.ATx(d.Ax(w))) < 1e-12
    with pytest.raises(capi.VampomiError):
        sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_QINV_BERN], tau, gam2, track_ax_vecs=(V_Z2, V_Z2))
    # iteration cap applies to both
    res = sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_QINV_BERN], tau, gam2, tol=1e-30, max_iter=3, onsager_mode=(False, False))
    assert (res[0][0], res[1][0]) == (3, 3)
    # argument validation
    with pytest.raises(capi.VampomiError):
        sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_X2], tau, gam2)
    with pytest.raises(capi.VampomiError):
        sh.cg_solve_pair([V_V, V_BERN], [V_X2, capi.V_CG2_P], tau, gam2)
    with pytest.raises(capi.VampomiError):
        sh.cg_solve_pair([V_V, V_BERN], [V_X2, V_QINV_BERN], tau, gam2, extra=(V_X1, capi.V_TMP_N0))
    sh.close()


# opt-in FP32 storage of the marker block (vampomi_create_ex): every value is rounded once, arithmetic stays FP64, so the
# results must equal the oracle's on the ROUNDED matrix
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,M", [(300, 800), (333, 517), (4100, 1033), (64, 1)])
def test_f32_storage_matches_oracle_on_rounded_matrix(N, M, tmp_path):
    rng = np.random.default_rng(N * 7 + M)
    A = rng.standard_normal((M, N)) * 0.1 + 0.5
    A32 = A.astype(np.float32).astype(np.float64)
    y = rng.standard_normal(N)
    sh = capi.Shard(N, M, storage="f32")
    sh.upload(A)
    assert np.array_equal(sh.download(), A32)
    sh.compute_stats()
    d = vo.Data(A32, y)
    mave, msig = sh.stats()
    assert np.allclose(mave, d.mave, rtol=1e-13, atol=1e-15) and np.allclose(msig, d.msig, rtol=1e-12)
    p, x = rng.standard_normal(N), rng.standard_normal(M)
    for knobs in (dict(), dict(atx_impl=0), dict(atx_impl=2, atx_cols=4, atx_unroll=2), dict(ax_rv=1, ax_unroll=8), dict(ax_rv=4, ax_unroll=2),
                  dict(ax_impl=1, atx_impl=1)):          # the bulk knobs fall back to the LDG kernels for FP32 storage
        for k, v in knobs.items():
            sh.set_tuning(k, v)
        assert rel_l2(sh.ATx(p), d.ATx(p)) < 1e-12
        assert rel_l2(sh.Ax(x), d.Ax(x)) < 1e-12
    w = rng.standard_normal(N)
    sh.set(V_USER_N1, w)
    sums = sh.loo_sums(V_USER_N1)
    assert np.allclose(sums[:, 0], A32.sum(1), rtol=1e-12) and np.allclose(sums[:, 2], A32 @ w, rtol=1e-10, atol=1e-10)
    # file ingest rounds the same way
    A.tofile(tmp_path / "a.bin")
    sh.load_file(str(tmp_path / "a.bin"))
    assert np.array_equal(sh.download(), A32)
    sh.close()


def test_f32_storage_generator_is_the_rounded_f64_generator():
    N, M = 257, 91
    a = capi.Shard(N, M)
    b = capi.Shard(N, M, storage="f32")
    a.generate_iid(42)
    b.generate_iid(42)
    assert np.array_equal(b.download(), a.download().astype(np.float32).astype(np.float64))
    a.close()
    b.close()


def test_instrumentation_and_error_paths():
    N, M = 300, 800
    sh, A, y, rng = make(N, M, seed=12)
    assert sh.comm_mode() == 0 and sh.stream() is not None
    sh.counters(reset=True)
    sh.profile(True)
    sh.profile_read(reset=True)
    x = rng.standard_normal(M)
    sh.set(V_V, x)
    it, _, _ = sh.cg_solve(V_V, V_X2, 2.0, 1.5, tol=1e-6)
    c = sh.counters()
    assert c["matrix_passes"] == 2 * it and c["matrix_bytes"] == 2 * it * N * M * 8 and c["allreduces"] == 0
    pr = sh.profile_read()
    assert pr["ax_partial"]["launches"] == it and pr["atx"]["launches"] == it          # look-ahead no-op launches are not counted
    assert pr["ax_partial"]["bytes"] == it * N * M * 8 and pr["ax_partial"]["ms"] > 0
    sh.profile(False)
    assert sh.time_kernel(0, 3) > 0 and sh.time_kernel(1, 3) > 0 and sh.time_kernel(2, 1) > 0 and sh.time_kernel(3, 1) > 0
    # error paths: codes and messages, never a crash
    for knob in ("no_such_knob", "gram_shape", "gram_prefetch"):    # the last two selected fused-pass variants that no longer exist
        with pytest.raises(capi.VampomiError, match="unknown knob"):
            sh.set_tuning(knob, 1)
    with pytest.raises(capi.VampomiError, match="must be in"):
        sh.set_tuning("ax_rv", 99)
    with pytest.raises(capi.VampomiError, match="distinct M-vectors"):
        sh.cg_solve(V_V, V_V, 1.0, 1.0)
    with pytest.raises(capi.VampomiError, match="bad vector id"):
        sh.get(99)
    with pytest.raises(capi.VampomiError, match="outside the shard"):
        sh.upload(A, j0=10)
    fresh = capi.Shard(N, M)
    with pytest.raises(capi.VampomiError, match="before compute_stats"):
        fresh.Ax(x)
    fresh.close()
    sh.close()


def test_onepass_falls_back_where_the_fused_pass_cannot_run():
    """N > 40 960 rows (more than 16 CTAs x 2 560 rows hold) and FP32 storage: vampomi_aat_supported says no, the fused entry point
    refuses, and a solve with cg_onepass set runs the two-pass iterations with the same answer."""
    N, M = 40976, 24
    sh, A, y, rng = make(N, M, seed=5)
    assert not sh.aat_supported()
    with pytest.raises(capi.VampomiError):
        sh.aat_multi_dev([V_USER_N0], [V_R1], [V_Z1])
    d = vo.Data(A, y)
    o = vo.Vamp(d, CG_err_tol=1e-7)
    o.gam2 = 1.9
    v = rng.standard_normal(M)
    want = o.precondCG_solver(v, None, 2.3, 1)
    sh.set(V_V, v)
    sh.set_tuning("cg_onepass", 1)
    sh.counters(reset=True)
    it, _, _ = sh.cg_solve(V_V, V_X2, 2.3, 1.9, tol=1e-7)
    assert it == o.cg_iters[-1][2] and rel_l2(sh.get(V_X2), want) < 1e-11
    assert sh.counters()["matrix_passes"] == 2 * it
    sh.close()
