"""Every output entry of the kernels at the benchmark's shape, N = 20 000 samples x M = 850 000 markers on one GPU: 136 GB and
1.7e10 elements in FP64, 68 GB in FP32 storage. Such a block passes 2^31, 2^32 and 2^33 elements and 2^32 ... 2^36 bytes,
where a column offset, a tensor-map coordinate or a chunk index kept in 32 bits would wrap. The blocks of test_kernel_exact
and test_vector_exact stay below 2^31 elements, so they cannot see such a wrap; this file checks the same outputs against the
same bounds at the size the kernels are tuned for. Per entry y = sum_k term_k of n terms:

    |got - exact| <= (n + 8) * 2^-53 * sum_k |term_k|   (+ 1e-300 for underflow)

For A x, n may be the number of non-zero terms. A term that is exactly 0 (x_j = 0, or a_ij - mave_j = 0 in a constant column,
whose mave is its value exactly) is formed without a rounding, and adding an exact 0 to a partial sum is exact. On any
summation tree, only an addition whose two operands each hold a non-zero term can round, and there are at most n - 1 of them
on the path of any term; the 8 cover the roundings within a term and the final scaling, as before.

The host cannot hold such a block in long double, so each reference needs a few columns only:
* generated block (vampomi_generate_iid): a sample of columns is downloaded, so the reference reads what the kernels read.
  Statistics, A^T p, t of the fused pass and the loo sums of a column need that column alone; A x is checked with x non-zero
  on the sampled columns only. The CG steps are checked from the device's own t (test_vector_exact.cg_step_check).
* mostly constant block: column j holds c_j = VALUES[j % 997] in every row, and the sampled columns hold random and awkward
  columns (test_kernel_exact.awkward_columns). A constant column is exact by the rules test_kernel_exact checks: mave = c_j,
  msig = 1, its A^T output is 0.0 and it adds exactly 0 to A x. So every entry of every output has an exact reference built
  from the sampled columns, and a read of the wrong column shows up as mave_j != c_j.

The sample: the first and the last 64 columns, every 997th, and 32 columns around each column that holds element 2^k
(k >= 31) or byte 2^k (k >= 32) of the block, for the block's column stride ld (N rounded up to 16) and element size. Each
test holds one context, so one large block at a time is on the device. A test skips only when its block cannot be allocated
(a device shared with other work); the reason gives the size it needed. Each test prints the time of its host-side
uploads and file loads (pytest -rP shows it)."""
import time

import numpy as np
import pytest

from vampomi_b200 import capi
from vampomi_b200.capi import V_USER_N1, V_Z1, V_Z2
from test_kernel_exact import (LD, PIN, POUT, XIN, XOUT, assert_loo_sums_exact, assert_stats_exact, assert_within, atx_exact,
                               awkward_columns, ax_exact, cancelling, constant)
from test_missing_values import impute_ref
from test_vector_exact import assert_cg_steps_exact

pytestmark = pytest.mark.gpu

N_FULL, M_FULL = 20000, 850000
PERIOD = 997
# the constant of column j is VALUES[j % 997]: sums of these do not come out exact in FP64, and neighbouring columns differ
VALUES = np.concatenate([[0.1, 0.7, 1 / 3, 0.0, -0.1, -2 / 3, 1e3, -1e3, 0.9532, 2 / 7, -1 / 3],
                         np.random.default_rng(PERIOD).uniform(-3.0, 3.0, PERIOD - 11)])


@pytest.fixture(autouse=True)
def _extended_precision():
    if np.finfo(np.longdouble).nmant < 63:
        pytest.skip("np.longdouble has fewer than 63 mantissa bits here: no extended-precision reference")


def open_shard(N, M, **kw):
    try:
        return capi.Shard(N, M, **kw)
    except capi.VampomiError as e:
        if "marker block failed" in str(e):
            pytest.skip(f"the block does not fit the device's free memory now: {e}")
        raise


def padded(N):
    return (N + 15) // 16 * 16                        # column stride of the block on the device (128-byte columns)


def crossing_columns(M, ld, elem_bytes):
    """The columns of an [M][ld] block that hold element 2^k (k >= 31) or byte 2^k (k >= 32)."""
    offsets = [2 ** k for k in range(31, 64)] + [2 ** k // elem_bytes for k in range(32, 64)]
    return sorted({o // ld for o in offsets if o // ld < M})


def windows(centres, M, half=16):
    return {j for c in centres for j in range(max(c - half, 0), min(c + half, M))}


def sample_columns(M, ld, elem_bytes):
    cross = crossing_columns(M, ld, elem_bytes)
    s = set(range(64)) | set(range(M - 64, M)) | set(range(PERIOD // 2, M, PERIOD)) | windows(cross, M)
    return np.array(sorted(s)), cross


def runs(cols):
    """(first column, count) of each run of consecutive columns."""
    cuts = np.nonzero(np.diff(cols) != 1)[0] + 1
    return [(int(r[0]), r.size) for r in np.split(cols, cuts)]


def download_columns(sh, cols):
    return np.concatenate([sh.download(j0, n) for j0, n in runs(cols)])


def upload_columns(sh, cols, block):
    k = 0
    for j0, n in runs(cols):
        sh.upload(block[k:k + n], j0)
        k += n


def random_columns(N, n, rng, big):
    """Blocks of 11 awkward columns (the large-offset one at row 8, which `cancelling` picks) and 11 of beta values."""
    awk = awkward_columns(N, rng, big)
    B = rng.beta(0.3, 0.3, size=(n, N))
    for s in range(n):
        if s % 22 < len(awk):
            B[s] = awk[s % 22]
    return B


def dense_split_extra(cv, msig, x, const, N):
    """center_split adds sum_j a_ij w_j and sum_j mave_j w_j: on a constant column both are c_j w_j (w_j = msig_j x_j)."""
    return 2 * np.abs(cv[const].astype(LD) * msig[const].astype(LD) * x[const].astype(LD)).sum() / np.sqrt(LD(N))


# ---- checks shared by the tests ----------------------------------------------------------------------------------------------
def check_stats(sh, held, cols, alpha, const=None, cv=None):
    """Statistics of the sampled columns; with a mostly constant block, every constant column: mave = c_j and msig = 1 bit for
    bit, and constant_columns() marks exactly these."""
    sh.compute_stats(alpha)
    mave, msig = sh.stats()
    if const is not None:
        wrong = np.nonzero(mave.view(np.uint64)[const] != cv.view(np.uint64)[const])[0]
        where = np.nonzero(const)[0]
        assert wrong.size == 0, (f"alpha {alpha}: {wrong.size} of {where.size} constant columns with mave != c_j, first column "
                                 f"{where[wrong[0]]}: mave {mave[where[wrong[0]]]!r}, c_j {cv[where[wrong[0]]]!r}")
        bad = np.nonzero(msig[const] != 1.0)[0]
        assert bad.size == 0, f"alpha {alpha}: {bad.size} constant columns with msig != 1, first column {where[bad[0]]}"
        assert np.array_equal(sh.constant_columns(), const)
    assert_stats_exact(held, mave[cols], msig[cols], alpha)
    return mave, msig


def check_atx(sh, held, cols, mave, msig, ps, const=None, cv=None):
    """A^T p for p and cancelling(p): automatic choice, atx_impl 0, 1, 2 and center_split; atx_multi_dev K = 1, 2 with both
    forms (multi_atx_impl 0: [tile][K][M] partials in registers, 1: p tiles in shared memory). Sampled entries against the
    exact value; a constant column gives exactly 0.0 (under center_split: within the bound of its two cancelling sums)."""
    N = sh.N
    want = [atx_exact(held, mave[cols], msig[cols], p) for p in ps]
    for knobs in (dict(), dict(atx_impl=0), dict(atx_impl=1), dict(atx_impl=2)):
        for k, v in knobs.items():
            sh.set_tuning(k, v)
        for i, p in enumerate(ps):
            got = sh.ATx(p)
            assert_within(got[cols], *want[i], N, f"ATx {knobs} p{i}")
            if const is not None:
                assert np.all(got[const] == 0.0), (knobs, np.nonzero(got[const] != 0.0)[0][:10])
    sh.set_tuning("atx_impl", 0)
    sh.set_tuning("center_split", 1)
    for i, p in enumerate(ps):
        got = sh.ATx(p)
        assert_within(got[cols], *atx_exact(held, mave[cols], msig[cols], p, split=True), N, f"ATx center_split p{i}")
        if const is not None:
            s = np.abs(msig[const].astype(LD)) / np.sqrt(LD(N))
            absum = 2 * np.abs(cv[const].astype(LD)) * np.abs(p.astype(LD)).sum() * s
            assert_within(got[const], np.zeros(int(const.sum()), dtype=LD), absum, N, f"ATx center_split p{i}, constant columns")
    sh.set_tuning("center_split", 0)
    sh.set_tuning("atx_impl", 3)
    for impl in (0, 1):
        sh.set_tuning("multi_atx_impl", impl)
        for K in (1, 2):
            for i in range(K):
                sh.set(PIN[i], ps[i])
            sh.atx_multi_dev(PIN[:K], POUT[:K])
            for i in range(K):
                got = sh.get(POUT[i])
                assert_within(got[cols], *want[i], N, f"atx_multi_dev multi_atx_impl={impl} K={K} vector {i}")
                if const is not None:
                    assert np.all(got[const] == 0.0)
    sh.set_tuning("multi_atx_impl", 1)
    return want


def check_ax(sh, held, cols, mave, msig, xs, const=None, cv=None):
    """A x for x = xs[0] (ax_impl 0 and 1, center_split) and A x_k for the first K of xs (ax_multi_dev, K = 1 ... 4). The
    reference holds the sampled columns whose terms can be non-zero: x is zero outside the sample, or the column outside the
    sample is constant. Under center_split a constant column adds c_j w_j twice with opposite signs, so there n is the number
    of x_j != 0. A constant column adds exactly 0: changing x there leaves A x the same bit for bit."""
    N = sh.N
    live = ~constant(held)
    hl, ml, sl = held[live], mave[cols][live], msig[cols][live]
    n = int(live.sum())
    want = [ax_exact(hl, ml, sl, x[cols][live]) for x in xs]
    x2 = None
    if const is not None:
        x2 = xs[0].copy()
        x2[const] = np.random.default_rng(3).standard_normal(int(const.sum())) * 100
    for impl in (0, 1):
        sh.set_tuning("ax_impl", impl)
        got = sh.Ax(xs[0])
        assert_within(got, *want[0], n, f"Ax ax_impl={impl}")
        if x2 is not None:
            assert np.array_equal(sh.Ax(x2).view(np.uint64), got.view(np.uint64)), f"Ax ax_impl={impl}: a constant column changed A x"
    sh.set_tuning("ax_impl", 0)
    sh.set_tuning("center_split", 1)
    exact, absum = ax_exact(hl, ml, sl, xs[0][cols][live], split=True)
    if const is not None:
        absum = absum + dense_split_extra(cv, msig, xs[0], const, N)
    assert_within(sh.Ax(xs[0]), exact, absum, int(np.count_nonzero(xs[0])), "Ax center_split")
    sh.set_tuning("center_split", 0)
    for K in (1, 2, 3, 4):
        for i in range(K):
            sh.set(XIN[i], xs[i])
        sh.ax_multi_dev(XIN[:K], XOUT[:K])
        for i in range(K):
            assert_within(sh.get(XOUT[i]), *want[i], n, f"ax_multi_dev K={K} vector {i}")
    if x2 is not None:
        sh.set(XIN[0], xs[0])
        sh.ax_multi_dev(XIN[:1], XOUT[:1])
        got = sh.get(XOUT[0])
        sh.set(XIN[0], x2)
        sh.ax_multi_dev(XIN[:1], XOUT[:1])
        assert np.array_equal(sh.get(XOUT[0]).view(np.uint64), got.view(np.uint64)), "ax_multi_dev: a constant column changed A x"


def check_fused(sh, held, cols, mave, msig, ps, want_t, clusters, const=None):
    """t = A^T q and w = A t of the fused pass for K = 1, 2 at each cluster size (0 = automatic). t on the sampled entries; with
    a mostly constant block also t = 0.0 on every constant column and w against A applied to the device's own t."""
    N = sh.N
    live = ~constant(held)
    w_cache = {}
    for cs in clusters:
        sh.set_tuning("gram_cluster", cs)
        for K in (1, 2):
            for i in range(K):
                sh.set(PIN[i], ps[i])
            sh.aat_multi_dev(PIN[:K], POUT[:K], [V_Z1, V_Z2][:K])
            for i in range(K):
                t = sh.get(POUT[i])
                what = f"aat gram_cluster={cs} K={K} vector {i}"
                assert_within(t[cols], *want_t[i], N, f"{what}: t")
                if const is None:
                    continue
                assert np.all(t[const] == 0.0), what
                key = t[cols][live].tobytes()
                if key not in w_cache:
                    w_cache[key] = ax_exact(held[live], mave[cols][live], msig[cols][live], t[cols][live])
                assert_within(sh.get([V_Z1, V_Z2][i]), *w_cache[key], int(live.sum()), f"{what}: w")
    sh.set_tuning("gram_cluster", 0)


def check_loo(sh, held, cols, rng, const=None, cv=None):
    N = sh.N
    w = rng.standard_normal(N)
    sh.set(V_USER_N1, w)
    got = sh.loo_sums(V_USER_N1)
    assert_loo_sums_exact(got[cols], held, w)
    if const is not None:
        other = const.copy()
        other[cols] = False                           # constant columns outside the sample
        c, wl = cv[other].astype(LD), w.astype(LD)
        assert_within(got[other, 0], N * c, N * np.abs(c), N, "sum x, constant columns")
        assert_within(got[other, 1], N * c * c, N * c * c, N, "sum x^2, constant columns")
        assert_within(got[other, 2], c * wl.sum(), np.abs(c) * np.abs(wl).sum(), N, "sum x w, constant columns")


# ---- 1. generated block --------------------------------------------------------------------------------------------------------
def test_generated_block_full_size_exact():
    """FP64, vampomi_generate_iid, N = 20 000, M = 850 000: statistics (alpha 1 and 0.5), A^T p, t of the fused pass and the loo
    sums on the sampled columns, A x on x non-zero on the sampled columns only, and CG iterations 1 and 2 of both solvers."""
    N, M = N_FULL, M_FULL
    cols, cross = sample_columns(M, padded(N), 8)
    assert cross and cross[-1] > M // 2 and cols[-1] == M - 1
    rng = np.random.default_rng(20)
    with open_shard(N, M) as sh:
        sh.generate_iid(11)
        held = download_columns(sh, cols)
        for alpha in (0.5, 1.0):
            mave, msig = check_stats(sh, held, cols, alpha)
        p = rng.standard_normal(N)
        ps = [p, cancelling(held, mave[cols], p)]
        want_t = check_atx(sh, held, cols, mave, msig, ps)
        check_fused(sh, held, cols, mave, msig, ps, want_t, (0,))
        xs = []
        for s in (1.0, 1e-3, 1e3, 1.0):
            x = np.zeros(M)
            x[cols] = rng.standard_normal(cols.size) * s
            xs.append(x)
        check_ax(sh, held, cols, mave, msig, xs)
        check_loo(sh, held, cols, rng)
        for onepass in (0, 1):
            assert_cg_steps_exact(sh, onepass, rng.standard_normal(M), rng.standard_normal(M), 2.3, 0.7)


# ---- 2. and 3. mostly constant blocks ------------------------------------------------------------------------------------------
def mostly_constant_case(storage, N, M):
    """Uploads the mostly constant block, imputes three columns past 2^32 elements, then checks every output entry."""
    f32 = storage == "f32"
    ld, eb = padded(N), (4 if f32 else 8)
    cols, cross = sample_columns(M, ld, eb)
    rng = np.random.default_rng(N + eb)
    B = random_columns(N, cols.size, rng, 1e30 if f32 else 1e100)
    # NaNs in three columns that start past element 2^32: none observed, one observed value (in the last row, the scalar
    # tail of the kernels), scattered
    c32 = 2 ** 32 // ld
    assert c32 in cross
    nan_cols = [c32 + 1, c32 + 2, c32 + 3]
    pos = np.searchsorted(cols, nan_cols)
    assert np.array_equal(cols[pos], nan_cols)
    B[pos[0]] = np.nan
    B[pos[1]] = np.nan
    B[pos[1], N - 1] = 0.3
    B[pos[2]] = rng.beta(0.3, 0.3, N)
    B[pos[2], rng.random(N) < 0.05] = np.nan
    rounded = B.astype(np.float32).astype(np.float64) if f32 else B
    with open_shard(N, M, storage=storage) as sh:
        assert sh.aat_supported() != f32
        t0 = time.perf_counter()
        base = np.repeat(VALUES[:, None], N, axis=1)
        for j0 in range(0, M, PERIOD):
            sh.upload(base[:min(PERIOD, M - j0)], j0)
        t1 = time.perf_counter()
        print(f"{storage}: upload of {M * N * 8 / 1e9:.1f} GB of FP64 columns from pageable host memory in "
              f"{-(-M // PERIOD)} calls: {t1 - t0:.1f} s")
        upload_columns(sh, cols, B)
        got = download_columns(sh, cols)
        assert np.array_equal(np.isnan(got), np.isnan(rounded)) and np.array_equal(got[~np.isnan(got)], rounded[~np.isnan(rounded)])
        miss = np.isnan(got)
        want_imp, want_counts = impute_ref(got[pos], storage)
        assert list(sh.impute_missing()) == want_counts and want_counts[1:] == [3, 1]
        held = download_columns(sh, cols)
        assert np.array_equal(held.view(np.uint64)[~miss], got.view(np.uint64)[~miss])       # observed entries unchanged
        imp = held[pos]
        np.testing.assert_allclose(imp[miss[pos]], want_imp[miss[pos]], rtol=1e-14, atol=0)
        assert np.all(imp[0] == 0.0) and np.all(imp[1] == (float(np.float32(0.3)) if f32 else 0.3))
        cv = VALUES[np.arange(M) % PERIOD]
        if f32:
            cv = cv.astype(np.float32).astype(np.float64)
        cv[cols] = held[:, 0]
        const = np.ones(M, dtype=bool)
        const[cols] = constant(held)
        for alpha in (0.5, 1.0):
            mave, msig = check_stats(sh, held, cols, alpha, const, cv)
        p = rng.standard_normal(N)
        ps = [p, cancelling(held, mave[cols], p)]
        want_t = check_atx(sh, held, cols, mave, msig, ps, const, cv)
        if not f32:
            check_fused(sh, held, cols, mave, msig, ps, want_t, (0, 16), const)
        xs = [rng.standard_normal(M) * s for s in (1.0, 1e-3, 1e3, 1.0)]
        check_ax(sh, held, cols, mave, msig, xs, const, cv)
        check_loo(sh, held, cols, rng, const, cv)


def test_mostly_constant_block_full_size_exact():
    """FP64, N = 20 000, M = 850 000 (136 GB): every entry of the statistics, A^T p, A x, the fused pass (K = 1, 2 at the
    automatic 8-CTA clusters and at 16) and the loo sums; mean imputation of three columns past 2^32 elements."""
    mostly_constant_case("f64", N_FULL, M_FULL)


def test_mostly_constant_block_f32_storage_full_size_exact():
    """FP32 storage, N = 20 003 (ld = 20 016: pad rows, a ragged tail), M = 850 000 (68 GB, past 2^32 elements): as the FP64
    case, without the fused pass, which needs FP64 storage."""
    mostly_constant_case("f32", N_FULL + 3, M_FULL)


# ---- 4. loading a file past 4 GiB ----------------------------------------------------------------------------------------------
def test_load_file_past_4_gib(tmp_path):
    """A sparse file of N = 20 000 x Mt = 60 000 (9.6 GB) with about 200 written columns: around the start and the end, the
    second shard's start (column 30 000, byte 4.8e9), the file's 2^32- and 2^33-byte offsets and the second shard's 2^32-byte
    offset on the device; the rest are holes, which read as 0.0. Loaded as rank 0 of 1 and rank 1 of 2, buffered and with
    O_DIRECT, with 1 and 8 reader threads, each time over a block that holds other values: the written columns come back bit
    for bit, every other column is all zeros (its sum of squares is 0; on the single shard also mave = 0 and msig = 1). A shard
    of two without a communicator runs no collective, and compute_stats ends in one, so there the loo sums alone check it."""
    N, Mt = N_FULL, 60000
    col_bytes = N * 8
    M1, S1 = capi.divide_work(Mt, 2, 1)
    centres = [0, S1, Mt - 1] + crossing_columns(Mt, N, 8) + [S1 + c for c in crossing_columns(M1, padded(N), 8)]
    written = np.array(sorted(windows(centres, Mt)))
    assert {26843, 53687, S1 + 26843} <= set(written.tolist())
    rng = np.random.default_rng(4)
    data = rng.standard_normal((written.size, N))
    path = tmp_path / "sparse.bin"
    with open(path, "wb") as f:
        f.truncate(Mt * col_bytes)
        for j0, n in runs(written):
            k0 = int(np.searchsorted(written, j0))
            f.seek(j0 * col_bytes)
            f.write(data[k0:k0 + n].tobytes())
    timings = []
    for nranks, rank in ((1, 0), (2, 1)):
        with open_shard(N, Mt, nranks=nranks, rank=rank, nccl_id=False) as sh:
            mine = (written >= sh.S) & (written < sh.S + sh.M)
            local = written[mine] - sh.S
            holes = np.ones(sh.M, dtype=bool)
            holes[local] = False
            sh.set(V_USER_N1, np.ones(N))
            for direct in (0, 1):
                for threads in (1, 8):
                    what = f"rank {rank} of {nranks}, load_direct={direct}, load_threads={threads}"
                    sh.set_tuning("load_direct", direct)
                    sh.set_tuning("load_threads", threads)
                    sh.generate_iid(5 + direct + threads)
                    t0 = time.perf_counter()
                    sh.load_file(str(path))
                    timings.append(f"{what}: {sh.M * col_bytes / 1e9:.1f} GB in {time.perf_counter() - t0:.2f} s")
                    got = download_columns(sh, local)
                    assert np.array_equal(got.view(np.uint64), data[mine].view(np.uint64)), what
                    sums = sh.loo_sums(V_USER_N1)
                    bad = np.nonzero(sums[holes, 1] != 0.0)[0]
                    assert bad.size == 0, f"{what}: {bad.size} columns of holes with a non-zero entry, first {np.nonzero(holes)[0][bad[0]]}"
                    if nranks == 1:
                        sh.compute_stats()
                        mave, msig = sh.stats()
                        assert np.all(mave[holes] == 0.0) and np.all(msig[holes] == 1.0), what
    print("\n".join(timings))
