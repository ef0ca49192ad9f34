"""TEST INFRASTRUCTURE ONLY — CPU (numpy/scipy) restatement of the reference's VAMP hot path.

This module is the *checker* for the CUDA implementation in ``vampomi_b200/csrc``; nothing in the product path
imports it (only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline leg may). Every function
cites the reference file:line it restates (paths relative to /root/reference).

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md §4). This restatement is pinned instead
against outputs of the reference itself, compiled here by ``oracle/build_ref.py`` into ``oracle/_ref/main_meth_ref``
(patched only to run and to be deterministic); the fixtures under ``tests/golden/`` were produced by that binary via
``tests/tools/make_golden.py`` and ``tests/test_oracle_vs_golden.py`` holds this module to them. The Boost special
functions (normal cdf, Student-t tail) are *not* in /root/reference; they are restated from their published
definitions and pinned against scipy (parity unpinned at the Boost boundary — see DESIGN.md).

Layout convention: the design matrix is held marker-major, ``A[j, i]`` = marker j, sample i — the order of the
reference's ``.bin`` file (README.md:16) and of ``meth_data[j*N + i]`` (src/data.cpp:297).
"""
import math
import os
import re

import numpy as np
from scipy import special as sps
from scipy import stats as spstats

GAMMA_MIN = 1e-11          # src/vamp.hpp:33
GAMMA_MAX = 1e11           # src/vamp.hpp:34
PROBIT_VAR = 1.0           # src/vamp.hpp:35 (--probit-var is parsed but never forwarded)

DEFAULT_VARS = [0, 1e-06, 6e-06, 3e-05, 2e-04, 1e-03, 6e-03, 3e-02, 2e-01, 1e+00]            # src/options.hpp:102
DEFAULT_PROBS = [9.90000e-01, 5.00000e-03, 2.50000e-03, 1.25000e-03, 6.25000e-04, 3.12500e-04,
                 1.56250e-04, 7.81250e-05, 3.90625e-05, 3.90625e-05]                           # src/options.hpp:103

METRICS_HEADER = ["iteration", "R2 denoising", "x1 correlation denoising", "R2 LMMSE", "x2 correlation LMMSE",
                  "z1 correlation denoising", "z2 correlation LMMSE"]                          # src/vamp.hpp:64-70
PARAMS_HEADER = ["iteration", "alpha1", "gam1", "alpha2", "gam2", "gamw"]                     # src/vamp.hpp:72-77
PRIOR_HEADER = ["iteration", "number of components"]                                          # src/vamp.hpp:79
TEST_HEADER = ["iteration", "R2 test", "z correlation test"]                                  # src/main_meth.cpp:143-145


# ----------------------------------------------------------------------------------------------------------------
# Counter-based randomness shared by oracle/_ref (oracle/ref_shims/oracle_hooks.h) and the product (csrc/rng.h)
# ----------------------------------------------------------------------------------------------------------------
_M64 = (1 << 64) - 1


def splitmix64(x):
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        z = x
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def hash3(seed, stream, a, b):
    with np.errstate(over="ignore"):
        h = splitmix64(np.uint64(seed & _M64) + np.uint64(0x632BE59BD9B4E019) * np.uint64(stream))
        h = splitmix64(h ^ np.asarray(a, dtype=np.uint64))
        h = splitmix64(h ^ np.asarray(b, dtype=np.uint64))
    return h


def probe_signs(seed, it, S, M):
    """±1 Hutchinson probe for VAMP iteration ``it`` and global markers S..S+M-1 (patch P2 of src/vamp.cpp:296)."""
    h = hash3(seed, 1, np.uint64(it), np.arange(S, S + M, dtype=np.uint64))
    return np.where((h >> np.uint64(63)) != 0, 1.0, -1.0)


def _box_muller(h1):
    h2 = splitmix64(h1)
    u1 = ((h1 >> np.uint64(11)).astype(np.float64) + 1.0) * 2.0 ** -53
    u2 = (h2 >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(6.283185307179586476925 * u2)


def probit_p1(seed, N):
    """Deterministic N(0,1) start for the probit z-channel (patch P3 of src/vamp_probit.cpp:53)."""
    return _box_muller(hash3(seed, 2, np.arange(N, dtype=np.uint64), np.uint64(0)))


def generate_iid_block(seed, j0, ncols, N):
    """Restatement of the device-side synthetic matrix generator (csrc/kernels.cu: k_generate_iid): A[j,i] ~ N(0,1)
    keyed by (seed, global marker j, sample i); agrees with the device to ~1 ulp (libm differs), not bitwise."""
    j = np.arange(j0, j0 + ncols, dtype=np.uint64)[:, None]
    i = np.arange(N, dtype=np.uint64)[None, :]
    return _box_muller(hash3(seed, 3, j, i))


# ----------------------------------------------------------------------------------------------------------------
# Work split, file formats
# ----------------------------------------------------------------------------------------------------------------
def divide_work(Mt, nranks, rank):
    """src/utilities.cpp:207-239 — contiguous marker blocks, first Mt % nranks ranks get one extra. Returns (M, S)."""
    modu, size = Mt % nranks, Mt // nranks
    lens = [size + 1 if i < modu else size for i in range(nranks)]
    return lens[rank], sum(lens[:rank])


def read_phen(path, standardize=True):
    """src/data.cpp:58-110 — third whitespace-separated token per line; scaled by sqrt((n-1)/sum((y-mean)^2)),
    NOT centred (:97-99); 'NA' is fatal (:73-74)."""
    vals = []
    with open(path) as f:
        for line in f:
            line = line.rstrip("\n")
            toks = re.split(r"\s+", line)
            if toks[2] == "NA":
                raise ValueError("NAN in data!")
            vals.append(_atof(toks[2]))
    y = np.array(vals, dtype=np.float64)
    if standardize:
        avg = y.sum() / len(y)
        sqn = math.sqrt((len(y) - 1) / float(((y - avg) ** 2).sum()))
        y = y * sqn
    return y


def _atof(s):
    m = re.match(r"\s*[-+]?(\d+\.?\d*([eE][-+]?\d+)?|\.\d+([eE][-+]?\d+)?|inf|nan)", s, re.I)
    return float(m.group(0)) if m else 0.0


def read_vec(path, M, S):
    """src/utilities.cpp:251-267 — M doubles at byte offset S*8."""
    return np.fromfile(path, dtype=np.float64, count=M, offset=S * 8)


def store_vec(path, vec, S):
    """src/utilities.cpp:241-249 — raw FP64 at byte offset S*8; file created if absent, never truncated."""
    fd = os.open(path, os.O_WRONLY | os.O_CREAT, 0o644)
    try:
        os.pwrite(fd, np.ascontiguousarray(vec, dtype=np.float64).tobytes(), S * 8)
    finally:
        os.close(fd)


def _fmt_double(v):
    """C's "%20.15f" including glibc's spelling of non-finite values ("-nan" when the sign bit is set)."""
    v = float(v)
    if math.isnan(v):
        return "%20s" % ("-nan" if math.copysign(1.0, v) < 0 else "nan")
    if math.isinf(v):
        return "%20s" % ("-inf" if v < 0 else "inf")
    return "%20.15f" % v


def csv_row(it, values):
    """src/utilities.cpp:366-385."""
    return "%5d" % it + "".join(", " + _fmt_double(v) for v in values) + "\n"


class CsvFile:
    """CSV with the reference's placement rule: header at 0 (src/utilities.cpp:388-401), the row of iteration ``it``
    at byte offset it*len(row) (:383) — which leaves NUL holes and lets rows overlap the header."""

    def __init__(self, path):
        if os.path.exists(path):
            os.unlink(path)                                    # MPI_File_delete, src/vamp.cpp:857
        self.fd = os.open(path, os.O_WRONLY | os.O_CREAT | os.O_EXCL, 0o644)

    def header(self, names):
        os.pwrite(self.fd, (", ".join(names) + "\n").encode(), 0)

    def row(self, it, values):
        b = csv_row(it, values).encode()
        os.pwrite(self.fd, b, it * len(b))

    def close(self):
        os.close(self.fd)


def read_csv_rows(path):
    """Tolerant reader used by tests (mirrors scripts/p_vals.py:41: strip NULs, skip a header if any)."""
    with open(path, "rb") as f:
        text = f.read().replace(b"\0", b"").decode()
    rows = {}
    for line in text.splitlines():
        parts = [p.strip() for p in line.split(",")]
        try:
            it = int(parts[0])
        except ValueError:
            continue
        rows[it] = [float(p) for p in parts[1:]]
    return rows


# ----------------------------------------------------------------------------------------------------------------
# Communicator stand-ins (marker shards = MPI ranks in the reference = GPUs in the product)
# ----------------------------------------------------------------------------------------------------------------
class SelfComm:
    nranks, rank = 1, 0

    def allreduce(self, x):
        return x


class TorchComm:
    """Sum all-reduce over torch.distributed (gloo on CPU) — used by the world_size-2 tests."""

    def __init__(self):
        import torch.distributed as dist
        self._dist = dist
        self.nranks, self.rank = dist.get_world_size(), dist.get_rank()

    def allreduce(self, x):
        import torch
        t = torch.from_numpy(np.atleast_1d(np.asarray(x, dtype=np.float64)).copy())
        self._dist.all_reduce(t)
        out = t.numpy()
        return float(out[0]) if np.ndim(x) == 0 else out


# ----------------------------------------------------------------------------------------------------------------
# Design-matrix operators (class data)
# ----------------------------------------------------------------------------------------------------------------
class Data:
    """Restates ``class data`` for one marker shard. ``A`` is the [M, N] marker-major block this shard owns."""

    def __init__(self, A, y, Mt=None, S=0, comm=None, alpha_scale=1.0):
        self.A = np.asarray(A, dtype=np.float64)
        self.M, self.N = self.A.shape
        self.Mt = self.M if Mt is None else Mt
        self.S = S
        self.y = np.asarray(y, dtype=np.float64)
        self.comm = comm or SelfComm()
        self.mave, self.msig = marker_stats(self.A, alpha_scale)
        self._Z = None

    @property
    def Z(self):
        if self._Z is None:          # standardised copy, (A - mave) * msig; rounding differs from the reference's
            self._Z = (self.A - self.mave[:, None]) * self.msig[:, None]    # in-loop form only at the 1e-16 level
        return self._Z

    def ATx(self, p):
        """src/data.cpp:294-333 — out[j] = msig[j] * sum_i (A[j,i]-mave[j]) * p[i], then * 1/sqrt(N)."""
        return (self.Z @ np.asarray(p, dtype=np.float64)) * (1.0 / math.sqrt(self.N))

    def Ax(self, x):
        """src/data.cpp:340-373 — sum over this shard's markers, all-reduce over shards (:367), then / sqrt(N) (:369)."""
        tmp = np.asarray(x, dtype=np.float64) @ self.Z
        return self.comm.allreduce(tmp) / math.sqrt(self.N)

    def loo_sums(self, j):
        a = self.A[j]
        return a.sum(), (a * a).sum()

    def pvals_loo(self, z1, y, x1_hat):
        """src/data.cpp:385-417 + src/utilities.cpp:269-282. Uses the RAW (unstandardised) column. A constant column (finite,
        min == max, as marker_stats decides) gets p = 1 instead of the formula's ratio of rounding residues (DESIGN §4)."""
        N = self.N
        y_mod = np.asarray(y) - np.asarray(z1)
        out = np.empty(self.M)
        sqrtN = math.sqrt(N)
        for j in range(self.M):
            a = self.A[j]
            if a.min() == a.max() and np.isfinite(a.min()):
                out[j] = 1.0
                continue
            y_mark = y_mod + a / sqrtN * x1_hat[j]
            out[j] = linear_reg1d_pvals(a.sum(), (a * a).sum(), (a * y_mark).sum(), y_mark.sum(),
                                        (y_mark * y_mark).sum(), N)
        return out


def marker_stats(A, alpha_scale=1.0):
    """src/data.cpp:233-283 — two-pass mean and inverse sample sd; constant column -> msig = 1 (:275-276).
    A constant column (finite, no NaN) gets mave = its value and msig = 1 exactly, as in k_stats: the reference tests
    sumsqr == 0, which a sum that misses a value such as 0.1 by an ulp fails (DESIGN §4)."""
    A = np.asarray(A, dtype=np.float64)
    N = A.shape[1]
    mave = A.sum(axis=1) / N
    sumsqr = ((A - mave[:, None]) ** 2).sum(axis=1)
    with np.errstate(divide="ignore", invalid="ignore"):
        sd = np.sqrt(sumsqr / (N - 1.0))
        msig = 1.0 / sd if alpha_scale == 1.0 else 1.0 / np.power(sd, alpha_scale)
    msig = np.where(sumsqr != 0.0, msig, 1.0)
    lo = A.min(axis=1)                                     # NaN when the column holds one
    const = (lo == A.max(axis=1)) & np.isfinite(lo)
    return np.where(const, lo, mave), np.where(const, 1.0, msig)


def linear_reg1d_pvals(sumx, sumsqx, sumxy, sumy, sumsqy, n):
    """src/utilities.cpp:269-282; boost::math::students_t complement cdf == scipy.stats.t.sf. A variance that rounds to <= 0
    gives p = 1 and |r| > 1 is clamped, so that rounding residue never turns into NaN (host/io.cpp does the same)."""
    s2y = (sumsqy - sumy * sumy / n) / (n - 1)
    s2x = (sumsqx - sumx * sumx / n) / (n - 1)
    sxy = (sumxy - sumx * sumy / n) / (n - 1)
    if s2x <= 0 or s2y <= 0 or s2x * s2y == 0:
        return 1.0
    rxy = min(1.0, max(-1.0, sxy / math.sqrt(s2x * s2y)))
    if abs(rxy) == 1.0:
        return 0.0
    t = rxy * math.sqrt((n - 2) / (1 - rxy * rxy))
    return 2.0 * float(spstats.t.sf(abs(t), n - 2))


def pvals_se(r1, gam1, N):
    """src/main_meth.cpp:229-243 (twin: scripts/p_vals.py:58-62): the tail of normal(r1_j, sd) beyond 0. Taken directly,
    erfc(|r1_j| / (sd sqrt 2)) / 2, instead of the reference's 1 - cdf for r1_j <= 0, which loses a negative effect's tail
    (DESIGN §4)."""
    sd = math.sqrt(1.0 / (gam1 * float(N)))
    return 0.5 * sps.erfc(np.abs(np.asarray(r1, dtype=np.float64)) / (sd * math.sqrt(2.0)))


def calc_stdev(vec):
    """src/utilities.cpp:183-205 (sync=0)."""
    vec = np.asarray(vec)
    n = len(vec)
    mean = vec.sum() / n
    return math.sqrt((float((vec * vec).sum()) - n * mean * mean) / (n - 1))


# ----------------------------------------------------------------------------------------------------------------
# Scalar channel functions
# ----------------------------------------------------------------------------------------------------------------
def erfcx_ref(x):
    """src/utilities.cpp:293-363 — scaled complementary error function with the reference's clamps:
    x < -10 -> +inf, x > 10 -> numeric_limits<double>::lowest() (sic)."""
    x = np.asarray(x, dtype=np.float64)
    out = sps.erfcx(np.clip(x, -10.0, 10.0))
    out = np.where(x < -10.0, np.inf, out)
    out = np.where(x > 10.0, -np.finfo(np.float64).max, out)
    return out


def normal_cdf(v):
    """src/utilities.cpp:284-287."""
    return 0.5 * sps.erfc(-np.asarray(v) * math.sqrt(0.5))


def g1_bin_class(p, tau1, y, m_cov=0.0):
    """src/vamp_probit.cpp:469-478."""
    c = (p + m_cov) / math.sqrt(PROBIT_VAR + 1.0 / tau1)
    ratio = 2.0 / math.sqrt(2 * math.pi) / erfcx_ref(-(2 * y - 1) * c / math.sqrt(2))
    return p + (2 * y - 1) * ratio / tau1 / math.sqrt(PROBIT_VAR + 1.0 / tau1)


def g1d_bin_class(p, tau1, y, m_cov=0.0):
    """src/vamp_probit.cpp:480-488."""
    c = (p + m_cov) / math.sqrt(PROBIT_VAR + 1.0 / tau1)
    ratio = 2.0 / math.sqrt(2 * math.pi) / erfcx_ref(-(2 * y - 1) * c / math.sqrt(2))
    return 1 - ratio / (1 + tau1 * PROBIT_VAR) * ((2 * y - 1) * c + ratio)


def read_covariates(path, C, N):
    """data::read_covariates, src/data.cpp:159-227: header line skipped, two ids skipped, C values per row; every covariate is
    standardised with its population standard deviation (long double sums), a constant one becomes zeros. Returns (N, C)."""
    if C == 0:
        return np.zeros((N, 0))
    rows = []
    with open(path) as f:
        for i, line in enumerate(f):
            if i == 0:
                continue
            tok = line.rstrip("\n").split()
            if line[:1].isspace():
                tok = [""] + tok                     # the reference's regex split yields an empty first token then
            vals = [float(t) for t in tok[2:]]
            if len(vals) != C:
                raise ValueError(f"FATAL: number of covariates = {len(vals)} does not match to the specified number of covariates = {C}")
            rows.append(vals)
    Z = np.array(rows, dtype=np.float64).reshape(len(rows), C)
    assert Z.shape[0] == N
    out = np.empty_like(Z)
    for c in range(C):
        col = Z[:, c].astype(np.longdouble)
        cavg = col.sum() / np.longdouble(N)
        csig = np.sqrt(((col - cavg) * (col - cavg)).sum() / np.longdouble(N))
        out[:, c] = 0.0 if csig < 1e-8 else ((col - cavg) / csig).astype(np.float64)
    return out


def _lu_solve(Mx, b):
    """Partial-pivot LU as uBLAS lu_factorize / lu_substitute are used at src/vamp_probit.cpp:551-558; zero RHS if singular."""
    m, b = np.array(Mx, dtype=np.float64), np.array(b, dtype=np.float64)
    n = len(b)
    pm = list(range(n))
    for k in range(n):
        piv = k + int(np.argmax(np.abs(m[k:, k])))
        pm[k] = piv
        if m[piv, k] == 0.0:
            return np.zeros(n)
        if piv != k:
            m[[k, piv], :] = m[[piv, k], :]
        for i in range(k + 1, n):
            m[i, k] /= m[k, k]
            m[i, k + 1:] -= m[i, k] * m[k, k + 1:]
    for k in range(n):
        if pm[k] != k:
            b[k], b[pm[k]] = b[pm[k]], b[k]
    for i in range(n):
        b[i] -= m[i, :i] @ b[:i]
    for i in range(n - 1, -1, -1):
        b[i] = (b[i] - m[i, i + 1:] @ b[i + 1:]) / m[i, i]
    return b


def mlogL_probit(y, gg, Z, eta):
    """src/vamp_probit.cpp:490-502."""
    arg = (2 * y - 1) / math.sqrt(PROBIT_VAR) * (gg + Z @ eta)
    return float(-np.log(normal_cdf(arg)).sum()) / len(y)


def grad_cov(y, gg, Z, eta):
    """src/vamp_probit.cpp:504-523."""
    arg = (2 * y - 1) / math.sqrt(PROBIT_VAR) * (gg + Z @ eta)
    ratio = 2.0 / math.sqrt(2 * math.pi) / erfcx_ref(-arg / math.sqrt(2))
    return ((-1) * ratio * (2 * y - 1) / math.sqrt(PROBIT_VAR)) @ Z / len(y)


def newton_method_cov(y, gg, Z, eta):
    """vamp::Newton_method_cov, src/vamp_probit.cpp:525-617."""
    eta = np.array(eta, dtype=np.float64)
    for it in range(501):
        g = gg + Z @ eta
        arg = (2 * y - 1) * g
        ratio = 2.0 / math.sqrt(2 * math.pi) / erfcx_ref(-arg / math.sqrt(2))
        lam = ratio * (2 * y - 1)
        W = lam * (lam + g)
        rhs = _lu_solve(Z.T @ (Z * W[:, None]), Z.T @ lam)
        grad = grad_cov(y, gg, Z, eta)
        scale, init_val = 1.0, mlogL_probit(y, gg, Z, eta)
        eta_new = eta.copy()
        for _ in range(1, 300):
            displ = scale * rhs
            eta_new = eta + displ
            if mlogL_probit(y, gg, Z, eta_new) <= init_val + float(displ @ grad) / 2:
                break
            scale *= 0.9
        norm_eta = math.sqrt(float(eta @ eta))
        rel_err = 1.0 if norm_eta == 0 else math.sqrt(float((eta - eta_new) @ (eta - eta_new))) / norm_eta
        if rel_err < 1e-4:
            break
        init_val = mlogL_probit(y, gg, Z, eta)
        eta = eta_new
        if mlogL_probit(y, gg, Z, eta) > init_val:
            break
    return eta


def confusion_matrix(y, yhat):
    """src/vamp_probit.cpp:631-652 — [TP, TN, FP, FN]."""
    y, yhat = np.asarray(y), np.asarray(yhat)
    return [int(((y == 1) & (yhat == 1)).sum()), int(((y == 0) & (yhat == 0)).sum()),
            int(((y == 0) & (yhat == 1)).sum()), int(((y == 1) & (yhat == 0)).sum())]


def _div(a, b):
    """IEEE division on scalars (0/0 -> NaN with the sign x86 produces, x/0 -> inf) instead of a Python exception."""
    with np.errstate(all="ignore"):
        return float(np.float64(a) / np.float64(b))


# ----------------------------------------------------------------------------------------------------------------
# class vamp
# ----------------------------------------------------------------------------------------------------------------
class Vamp:
    """Restates ``class vamp`` (src/vamp.hpp, src/vamp.cpp, src/vamp_probit.cpp) for one marker shard."""

    def __init__(self, data, gam1=1e-6, gamw=2.0, max_iter=50, CG_max_iter=500, CG_err_tol=1e-5, EM_max_iter=1,
                 EM_err_thr=1e-2, rho=0.5, learn_vars=1, learn_prior_delay=1, stop_criteria_thr=0.01,
                 merge_vars_thr=5e-1, vars=None, probs=None, true_signal=None, x1hat_init=None,
                 out_dir=None, out_name="out", model="linear", seed=0, verbosity=0, covs=None):
        d = self.data = data
        self.covs = None if covs is None or np.asarray(covs).shape[1] == 0 else np.asarray(covs, dtype=np.float64)   # (N, C), standardised
        self.cov_eff = None
        self.N, self.M, self.Mt, self.S, self.comm = d.N, d.M, d.Mt, d.S, d.comm
        self.gam1, self.gamw = float(gam1), float(gamw)
        self.max_iter, self.CG_max_iter, self.CG_err_tol = max_iter, CG_max_iter, CG_err_tol
        self.EM_max_iter, self.EM_err_thr, self.rho = EM_max_iter, EM_err_thr, rho
        self.learn_vars, self.learn_prior_delay = learn_vars, learn_prior_delay
        self.stop_criteria_thr, self.merge_vars_thr = stop_criteria_thr, merge_vars_thr
        self.vars = [float(v) * self.N for v in (DEFAULT_VARS if vars is None else vars)]     # src/vamp.cpp:87-88
        self.probs = [float(p) for p in (DEFAULT_PROBS if probs is None else probs)]
        self.true_signal = np.zeros(self.M) if true_signal is None else np.asarray(true_signal, dtype=np.float64)
        init = np.zeros(self.M) if x1hat_init is None else np.asarray(x1hat_init, dtype=np.float64)
        self.x1_hat = init / math.sqrt(self.N)                  # src/vamp.cpp:70-72 (with patch P1)
        self.r1 = init / math.sqrt(self.N)                      # src/vamp.cpp:77-79
        self.x2_hat = np.zeros(self.M)
        self.r2 = np.zeros(self.M)
        self.p1 = np.zeros(self.N)
        self.gam2 = 0.0                                         # src/vamp.hpp:12
        self.alpha1 = 0.0
        self.out_dir, self.out_name, self.model = out_dir, out_name, model
        self.seed, self.verbosity = seed, verbosity
        self.mu_CG_last = None
        self.cg_iters = []          # (VAMP it, kind, iterations) — harness extra (patch P5 equivalent)
        self.history = []           # per-iteration dict of the scalars that land in the CSVs
        self.dump = {}              # it -> (x1_hat/sqrt(N), r1/sqrt(N)) when out_dir is None
        self._it = 0

    # ---- scalar reductions (src/utilities.cpp:138-162) ----
    def dotM(self, u, v):
        return float(self.comm.allreduce(float(np.dot(u, v))))            # inner_prod(u, v, sync=1)

    def dotN_sync(self, u, v):
        return float(np.dot(u, v)) * self.comm.nranks                      # replicated N-vector with sync=1 (:835)

    # ---- Gaussian-mixture denoiser ----
    def g1(self, y, gam1):
        """src/vamp.cpp:440-463."""
        sigma = 1.0 / gam1
        if -1e-10 < sigma < 1e-10:
            return np.array(y, dtype=np.float64)
        eta_max = max(self.vars)
        y = np.asarray(y, dtype=np.float64)
        pk = np.zeros_like(y)
        pkd = np.zeros_like(y)
        with np.errstate(all="ignore"):
            for p_i, v_i in zip(self.probs, self.vars):
                expe = -0.5 * (y * y) * (eta_max - v_i) / (v_i + sigma) / (eta_max + sigma)
                z = p_i / math.sqrt(v_i + sigma) * np.exp(expe)
                pk = pk + z
                z = z / (v_i + sigma) * y
                pkd = pkd - z
            return y + sigma * pkd / pk

    def g1d(self, y, gam1):
        """src/vamp.cpp:465-492."""
        sigma = 1.0 / gam1
        y = np.asarray(y, dtype=np.float64)
        if -1e-10 < sigma < 1e-10:
            return np.ones_like(y)
        eta_max = max(self.vars)
        pk = np.zeros_like(y)
        pkd = np.zeros_like(y)
        pkdd = np.zeros_like(y)
        with np.errstate(all="ignore"):
            for p_i, v_i in zip(self.probs, self.vars):
                expe = -0.5 * (y * y) * (eta_max - v_i) / (v_i + sigma) / (eta_max + sigma)
                e = np.exp(expe)
                z = p_i / math.sqrt(v_i + sigma) * e
                pk = pk + z
                z = z / (v_i + sigma) * y
                pkd = pkd - z
                z2 = z / (v_i + sigma) * y
                pkdd = pkdd - p_i / (v_i + sigma) ** 1.5 * e + z2
            return 1 + sigma * (pkdd / pk - (pkd / pk) ** 2)

    # ---- EM prior update ----
    def em_sums(self, r1, gam1, lam, omegas, vars_):
        """Per-marker part of src/vamp.cpp:554-597 for one EM iteration: returns (sum pin, [sum beta_j pin],
        [sum beta_j (gamma_j^2 + v_j) pin]) over this shard (before the all-reduces)."""
        noise_var = 1.0 / gam1
        max_sigma = max(vars_)
        L = len(vars_)
        r2h = (r1 * r1) / 2
        with np.errstate(all="ignore"):
            num = np.empty((L - 1, len(r1)))
            gam = np.empty((L - 1, len(r1)))
            for j in range(1, L):
                num[j - 1] = (lam * omegas[j] * np.exp(-r2h * (max_sigma - vars_[j]) / (vars_[j] + noise_var)
                                                       / (max_sigma + noise_var))
                              / math.sqrt(vars_[j] + noise_var) / math.sqrt(2 * math.pi))
                gam[j - 1] = gam1 * r1 / (_div(1.0, vars_[j]) + gam1)
            tot = num.sum(axis=0)
            beta = num / tot
            pin = 1 / (1 + (1 - lam) / math.sqrt(2 * math.pi * noise_var)
                       * np.exp(-r2h * max_sigma / noise_var / (noise_var + max_sigma)) / tot)
            v = np.array([1.0 / (_div(1.0, vars_[j]) + gam1) for j in range(1, L)])
            gam = beta * (gam * gam + v[:, None])
            return float(pin.sum()), (beta * pin).sum(axis=1), (gam * pin).sum(axis=1)

    def updatePrior(self):
        """src/vamp.cpp:531-643."""
        gam1, probs, vars_ = self.gam1, self.probs, self.vars
        lam = 1 - probs[0]
        omegas = list(probs)
        for j in range(1, len(omegas)):
            omegas[j] = _div(omegas[j], lam)
        for _ in range(self.EM_max_iter):
            probs_prev, vars_prev = list(probs), list(vars_)
            s_pin, s_beta, s_gam = self.em_sums(self.r1, gam1, lam, omegas, vars_)
            lambda_total = float(self.comm.allreduce(s_pin))
            lam = lambda_total / self.Mt
            for j in range(len(probs) - 1):
                res_gammas_total = float(self.comm.allreduce(float(s_gam[j])))
                res_total = float(self.comm.allreduce(float(s_beta[j])))
                if self.learn_vars == 1:
                    vars_[j + 1] = _div(res_gammas_total, res_total)
                omegas[j + 1] = _div(res_total, lambda_total)
                probs[j + 1] = lam * omegas[j + 1]
            probs[0] = 1 - lam
            dp = sum((a - b) ** 2 for a, b in zip(probs, probs_prev))
            npr = sum(a * a for a in probs)
            dv = sum((a - b) ** 2 for a, b in zip(vars_, vars_prev))
            nv = sum(a * a for a in vars_)
            if math.sqrt(_div(dp, npr)) < self.EM_err_thr and math.sqrt(_div(dv, nv)) < self.EM_err_thr:
                break
        merge_components(probs, vars_, self.merge_vars_thr)

    # ---- LMMSE ----
    def lmmse_mult(self, v, tau):
        """src/vamp.cpp:645-662."""
        if not np.any(v):
            return np.zeros(self.M)
        return tau * self.data.ATx(self.data.Ax(v)) + self.gam2 * v

    def precondCG_solver(self, v, mu_start, tau, denoiser):
        """src/vamp.cpp:664-757. Returns mu; records the number of CG iterations executed."""
        diag = tau * (self.N - 1) / self.N + self.gam2
        mu = np.zeros(self.M) if mu_start is None else np.array(mu_start, dtype=np.float64)
        r = v - self.lmmse_mult(mu, tau)
        z = r / diag
        p = z.copy()
        prev_onsager = 0.0
        iters = 0
        for i in range(self.CG_max_iter):
            iters = i + 1
            d = self.lmmse_mult(p, tau)
            alpha = _div(self.dotM(r, z), self.dotM(d, p))
            mu = mu + alpha * p
            if denoiser == 0:
                onsager = self.gam2 * self.dotM(v, mu)
                rel_err = abs(_div(onsager - prev_onsager, onsager)) if onsager != 0 else 1.0
                if rel_err < 1e-8:
                    break
                prev_onsager = onsager
            beta = _div(1.0, self.dotM(r, z))
            r = r - d * alpha
            z = r / diag
            beta *= self.dotM(r, z)
            p = z + beta * p
            rel_err = _div(math.sqrt(self.dotM(r, r)), math.sqrt(self.dotM(v, v)))
            if rel_err < self.CG_err_tol:
                break
        self.cg_iters.append((self._it, "lmmse" if denoiser == 1 else "onsager", iters))
        if denoiser == 1:
            self.mu_CG_last = mu
        return mu

    def g2d_onsager(self, gam2, tau):
        """src/vamp.cpp:494-501."""
        self.invQ_bern_vec = self.precondCG_solver(self.bern_vec, None, tau, 0)
        return gam2 * self.dotM(self.bern_vec, self.invQ_bern_vec)

    def updateNoisePrec(self):
        """src/vamp.cpp:504-529."""
        temp = self.data.Ax(self.x2_hat) - self.data.y
        temp_norm2 = float(np.dot(temp, temp))
        tc_N = self.data.Ax(self.invQ_bern_vec)
        tc_M = self.data.ATx(tc_N)
        trace_corr = self.dotM(self.bern_vec, tc_M) * self.Mt
        self.gamw = _div(float(self.N), temp_norm2 + trace_corr)

    def err_measures(self, ind, metrics):
        """src/vamp.cpp:760-852 (only the values that reach _metrics.csv)."""
        y = self.data.y
        if ind == 1:
            x, Axest = self.x1_hat, self.z1
        else:
            x, Axest = self.x2_hat, self.data.Ax(self.x2_hat)
        corr = _div(self.dotM(x, self.true_signal),
                    math.sqrt(self.dotM(x, x) * self.dotM(self.true_signal, self.true_signal)))
        res = y - Axest
        l2_pred_err = math.sqrt(_div(float(np.dot(res, res)), float(np.dot(y, y))))
        R2 = 1 - l2_pred_err * l2_pred_err
        corr_y = _div(self.dotN_sync(Axest, y), math.sqrt(self.dotN_sync(Axest, Axest) * self.dotN_sync(y, y)))
        if ind == 1:
            metrics[1], metrics[0], metrics[4] = corr, R2, corr_y * corr_y
        else:
            metrics[3], metrics[2], metrics[5] = corr, R2, corr_y * corr_y

    def _draw_probe(self, it):
        self.bern_vec = probe_signs(self.seed, it, self.S, self.M) / math.sqrt(self.Mt)

    def _store(self, it):
        sqrtN = math.sqrt(self.N)
        if self.out_dir is None:
            self.dump[it] = (self.x1_hat / sqrtN, self.r1 / sqrtN)
        else:
            store_vec(os.path.join(self.out_dir, f"{self.out_name}_it_{it}.bin"), self.x1_hat / sqrtN, self.S)
            store_vec(os.path.join(self.out_dir, f"{self.out_name}_r1_it_{it}.bin"), self.r1 / sqrtN, self.S)

    def _open_csvs(self):
        if self.out_dir is None or self.comm.rank != 0:
            return None
        base = os.path.join(self.out_dir, self.out_name)
        return {k: CsvFile(base + f"_{k}.csv") for k in ("metrics", "params", "prior")}     # src/vamp.cpp:854-882

    def infere(self):
        """src/vamp.cpp:94-107."""
        if self.model == "linear":
            return self.infere_linear()
        if self.model == "bin_class":
            return self.infere_bin_class()
        raise ValueError("Invalid model specification!")

    # ---- linear model ----
    def infere_linear(self):
        """src/vamp.cpp:110-438."""
        N, Mt, rho, d = self.N, self.Mt, self.rho, self.data
        y = d.y
        sqrtN = math.sqrt(N)
        metrics, params = [0.0] * 6, [0.0] * 5
        csv = self._open_csvs()
        if csv:
            csv["metrics"].header(METRICS_HEADER)
            csv["params"].header(PARAMS_HEADER)
            csv["prior"].header(PRIOR_HEADER + [f"prob{i}" for i in range(len(self.probs))]
                                + [f"var{i}" for i in range(len(self.vars))])
        for it in range(1, self.max_iter + 1):
            self._it = it
            if it == 1 and self.covs is not None:                # src/vamp.cpp:155-169
                self.cov_eff = newton_method_cov(y, np.zeros(N), self.covs, np.zeros(self.covs.shape[1]))
                y = y - self.covs @ self.cov_eff
            if it > self.learn_prior_delay:
                self.updatePrior()
            x1_hat_prev = self.x1_hat
            self.x1_hat = self.g1(self.r1, self.gam1)
            if it > 1:
                self.x1_hat = rho * self.x1_hat + (1 - rho) * x1_hat_prev
            sum_d = float(self.g1d(self.r1, self.gam1).sum())
            self.alpha1 = float(self.comm.allreduce(sum_d)) / Mt
            self.eta1 = _div(self.gam1, self.alpha1)
            self.z1 = d.Ax(self.x1_hat)
            self._store(it)
            self.gam2 = min(max(self.eta1 - self.gam1, GAMMA_MIN), GAMMA_MAX)
            self.r2 = (self.eta1 * self.x1_hat - self.gam1 * self.r1) / self.gam2
            self.err_measures(1, metrics)
            params[0], params[1] = self.alpha1, self.gam1
            self._draw_probe(it)
            v = self.gamw * d.ATx(y) + self.gam2 * self.r2
            self.x2_hat = self.precondCG_solver(v, None if it == 1 else self.mu_CG_last, self.gamw, 1)
            self.alpha2 = self.g2d_onsager(self.gam2, self.gamw)
            self.eta2 = _div(self.gam2, self.alpha2)
            gam1_prev = self.gam1
            self.gam1 = min(max(self.eta2 - self.gam2, GAMMA_MIN), GAMMA_MAX)
            self.gam1 = rho * self.gam1 + (1 - rho) * gam1_prev
            self.r1 = (self.eta2 * self.x2_hat - self.gam2 * self.r2) / self.gam1
            self.updateNoisePrec()
            self.err_measures(2, metrics)
            params[2], params[3], params[4] = self.alpha2, self.gam2, self.gamw
            if csv:
                csv["params"].row(it, params)
                csv["metrics"].row(it, metrics)
            diff = x1_hat_prev - self.x1_hat
            NMSE = math.sqrt(_div(self.dotM(diff, diff), self.dotM(x1_hat_prev, x1_hat_prev)))
            self.history.append(dict(it=it, params=list(params), metrics=list(metrics), NMSE=NMSE,
                                     probs=list(self.probs), vars=[v_ / N for v_ in self.vars]))
            if it > 1 and NMSE < self.stop_criteria_thr:
                break
        if csv:
            for f in csv.values():
                f.close()
        return self.x1_hat / sqrtN

    # ---- probit model ----
    def infere_bin_class(self):
        """src/vamp_probit.cpp:19-467."""
        N, M, Mt, rho, d = self.N, self.M, self.Mt, self.rho, self.data
        y = d.y
        sqrtN = math.sqrt(N)
        metrics, params = [0.0] * 12, [0.0] * 8
        csv = self._open_csvs()
        tau1 = self.gam1
        ts_scaled = self.true_signal * sqrtN
        self.p1 = probit_p1(self.seed, N)
        self.r1 = np.zeros(M)
        self.r2 = np.zeros(M)
        self.alpha1 = 0.0
        z1_hat = np.zeros(N)
        m_cov = 0.0
        for it in range(1, self.max_iter + 1):
            self._it = it
            if it == 1 and self.covs is not None:                # src/vamp_probit.cpp:78-95
                self.cov_eff = newton_method_cov(y, z1_hat, self.covs, np.zeros(self.covs.shape[1]))
                m_cov = self.covs @ self.cov_eff                 # :214-217
            x1_hat_prev = self.x1_hat
            alpha1_prev = self.alpha1
            self.x1_hat = self.g1(self.r1, self.gam1)
            sum_d = float(self.g1d(self.r1, self.gam1).sum())
            self.alpha1 = float(self.comm.allreduce(sum_d)) / Mt
            self.eta1 = _div(self.gam1, self.alpha1)
            if it > 1:
                self.updatePrior()
                self.x1_hat = rho * self.x1_hat + (1 - rho) * x1_hat_prev
                self.alpha1 = rho * self.alpha1 + (1 - rho) * alpha1_prev
            self._store(it)
            x1_hat_scaled = self.x1_hat / sqrtN
            x1_corr = _div(self.dotM(self.x1_hat, ts_scaled),
                           math.sqrt(self.dotM(self.x1_hat, self.x1_hat) * self.dotM(ts_scaled, ts_scaled)))
            self.gam2 = min(max(self.eta1 - self.gam1, GAMMA_MIN), GAMMA_MAX)
            self.r2 = (self.eta1 * self.x1_hat - self.gam1 * self.r1) / self.gam2
            # z channel
            z1_hat = g1_bin_class(self.p1, tau1, y, m_cov)
            beta1 = float(g1d_bin_class(self.p1, tau1, y, m_cov).sum())
            if beta1 >= N:
                beta1 = N - 1.0
            beta1 /= N
            p2 = (z1_hat - beta1 * self.p1) / (1 - beta1)
            tau2 = tau1 * (1 - beta1) / beta1
            params[0:4] = [self.alpha1, beta1, self.gam1, tau1]
            cm1 = confusion_matrix(y, (normal_cdf(d.Ax(x1_hat_scaled)) >= 0.5).astype(np.float64))
            metrics[0:6] = [cm1[0], cm1[1], cm1[2], cm1[3], sum(cm1[:2]) / float(sum(cm1)), x1_corr]
            # LMMSE for x
            self._draw_probe(it)
            v = tau2 * d.ATx(p2) + self.gam2 * self.r2
            self.x2_hat = self.precondCG_solver(v, None, tau2, 1)
            alpha2 = self.g2d_onsager(self.gam2, tau2)
            x2_corr = _div(self.dotM(self.x2_hat, ts_scaled),
                           math.sqrt(self.dotM(self.x2_hat, self.x2_hat) * self.dotM(ts_scaled, ts_scaled)))
            self.eta2 = _div(self.gam2, alpha2)
            self.r1 = (self.x2_hat - alpha2 * self.r2) / (1 - alpha2)
            self.gam1 = min(max(self.gam2 * (1 - alpha2) / alpha2, GAMMA_MIN), GAMMA_MAX)
            # LMMSE for z
            z2_hat = d.Ax(self.x2_hat)
            beta2 = float(Mt) / N * (1 - alpha2)
            self.p1 = (z2_hat - beta2 * p2) / (1 - beta2)
            tau1 = min(max(tau2 * (1 - beta2) / beta2, GAMMA_MIN), GAMMA_MAX)
            params[4:8] = [alpha2, beta2, self.gam2, tau2]
            cm2 = confusion_matrix(y, (normal_cdf(d.Ax(self.x2_hat / sqrtN)) >= 0.5).astype(np.float64))
            metrics[6:12] = [cm2[0], cm2[1], cm2[2], cm2[3], sum(cm2[:2]) / float(sum(cm2)), x2_corr]
            prior_params = [float(len(self.probs))] + list(self.probs) + list(self.vars)       # un-rescaled (:428)
            if csv:
                csv["params"].row(it, params)
                csv["metrics"].row(it, metrics)
                csv["prior"].row(it, prior_params)
            diff = x1_hat_prev - self.x1_hat
            NMSE = math.sqrt(_div(self.dotM(diff, diff), self.dotM(x1_hat_prev, x1_hat_prev)))
            self.history.append(dict(it=it, params=list(params), metrics=list(metrics), NMSE=NMSE,
                                     probs=list(self.probs), vars=list(self.vars)))
            if it > 1 and NMSE < self.stop_criteria_thr:
                break
        if csv:
            for f in csv.values():
                f.close()
        return self.x1_hat


def merge_components(probs, vars_, thr):
    """src/vamp.cpp:627-642 — in place; erases component k when |v_j - v_k| / min(v_j, v_k) < thr (denominator 1e-7
    when v_j == 0) and adds its probability to component j."""
    j = 0
    while j < len(vars_):
        k = j + 1
        while k < len(vars_):
            denom = min(vars_[j], vars_[k]) if vars_[j] != 0 else 1e-7
            if _div(abs(vars_[j] - vars_[k]), denom) < thr:
                s = probs[j] + probs[k]
                del vars_[k]
                del probs[k]
                probs[j] = s
                k -= 1
            k += 1
        j += 1


# ----------------------------------------------------------------------------------------------------------------
# Run modes other than inference (src/main_meth.cpp)
# ----------------------------------------------------------------------------------------------------------------
def association_se(r1_file_vec, gam1, N):
    return pvals_se(np.asarray(r1_file_vec, dtype=np.float64), gam1, N)


def association_loo(data, est_file_vec):
    """src/main_meth.cpp:245-264."""
    x1_hat = np.asarray(est_file_vec, dtype=np.float64) * math.sqrt(float(data.N))
    z1 = data.Ax(x1_hat)
    return data.pvals_loo(z1, data.y, x1_hat)


def test_mode_row(data_test, est_file_vec):
    """src/main_meth.cpp:163-202 — returns (R2 test, corr^2) for one saved iteration."""
    N_test = data_test.N
    x = np.asarray(est_file_vec, dtype=np.float64) * math.sqrt(float(N_test))
    z = data_test.Ax(x)
    y = data_test.y
    l2 = float(((y - z) ** 2).sum())
    sd = calc_stdev(y)
    r2 = 1 - l2 / (sd * sd * len(y))
    nr = data_test.comm.nranks
    corr_y = _div(float(np.dot(z, y)) * nr, math.sqrt(float(np.dot(z, z)) * nr * float(np.dot(y, y)) * nr))
    return r2, corr_y * corr_y
