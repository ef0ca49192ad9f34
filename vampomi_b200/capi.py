"""ctypes binding of libvampomi_cuda.so (include/vampomi.h, include/vampomi_host.h).

This is the Python mirror of the reference's `class data` / `class vamp` seam for the VAMP hot path: numpy arrays in,
numpy arrays out, every call forwarded to the C ABI. There is no Python or CPU implementation behind it — if the
shared library is missing, or there is no CUDA device, calls raise.
"""
import ctypes as C
import os

import numpy as np

from .build import LIB_PATH

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)
c_ll_p = C.POINTER(C.c_longlong)
c_u8_p = C.POINTER(C.c_ubyte)

MAX_MIX = 32

# vector ids (include/vampomi.h)
V_X1, V_X1_PREV, V_R1, V_R2, V_X2, V_V, V_BERN, V_QINV_BERN, V_TRUE, V_ATY, V_TMP_M0, V_TMP_M1 = range(12)
V_CG_R, V_CG_Z, V_CG_P, V_CG_D, V_USER_M0, V_USER_M1 = 12, 13, 14, 15, 16, 17
V_CG2_R, V_CG2_Z, V_CG2_P, V_CG2_D, V_ATA_X2 = 18, 19, 20, 21, 22
V_Y, V_Z1, V_Z2, V_P1, V_P2, V_Z1HAT, V_TMP_N0, V_TMP_N1, V_USER_N0, V_USER_N1 = range(32, 42)
V_GRAM_W0, V_GRAM_W1, V_GRAM_AR0, V_GRAM_AR1 = range(42, 46)
V_MCOV = 46
DOT, DIFF2, SQDEV = 0, 1, 2


class SolverConfig(C.Structure):
    _fields_ = [("model", C.c_int), ("gam1", C.c_double), ("gamw", C.c_double), ("rho", C.c_double),
                ("CG_max_iter", C.c_int), ("CG_err_tol", C.c_double), ("EM_max_iter", C.c_int),
                ("EM_err_thr", C.c_double), ("learn_vars", C.c_int), ("learn_prior_delay", C.c_int),
                ("merge_vars_thr", C.c_double), ("L", C.c_int), ("probs", C.c_double * MAX_MIX),
                ("vars", C.c_double * MAX_MIX), ("seed", C.c_ulonglong), ("redundant_passes", C.c_int),
                ("fuse_passes", C.c_int), ("probes", C.c_int)]


class IterResult(C.Structure):
    _fields_ = [("it", C.c_int), ("n_params", C.c_int), ("n_metrics", C.c_int), ("params", C.c_double * 8),
                ("metrics", C.c_double * 12), ("nmse", C.c_double), ("gam1_next", C.c_double),
                ("cg_iters_lmmse", C.c_int), ("cg_iters_onsager", C.c_int), ("L", C.c_int),
                ("probs", C.c_double * MAX_MIX), ("vars", C.c_double * MAX_MIX), ("matrix_passes", C.c_longlong),
                ("true_gam1", C.c_double), ("true_gam2", C.c_double)]


# name -> (restype, argtypes); every symbol declared in include/*.h is listed here (tests check the two agree)
_SIGNATURES = {
    "vampomi_last_error": (C.c_char_p, []),
    "vampomi_abi_version": (C.c_int, []),
    "vampomi_device_count": (C.c_int, [c_int_p]),
    "vampomi_create": (C.c_int, [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "vampomi_create_ex": (C.c_int, [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "vampomi_storage": (C.c_int, [C.c_void_p, c_int_p]),
    "vampomi_destroy": (C.c_int, [C.c_void_p]),
    "vampomi_shard": (C.c_int, [C.c_void_p, c_ll_p, c_ll_p]),
    "vampomi_dims": (C.c_int, [C.c_void_p, c_int_p, c_ll_p, c_int_p, c_int_p]),
    "vampomi_divide_work": (C.c_int, [C.c_longlong, C.c_int, C.c_int, c_ll_p, c_ll_p]),
    "vampomi_comm_get_unique_id": (C.c_int, [C.c_void_p]),
    "vampomi_comm_init": (C.c_int, [C.c_void_p, C.c_void_p]),
    "vampomi_comm_mode": (C.c_int, [C.c_void_p, c_int_p]),
    "vampomi_barrier": (C.c_int, [C.c_void_p]),
    "vampomi_upload_columns": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, c_double_p]),
    "vampomi_download_columns": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, c_double_p]),
    "vampomi_load_file": (C.c_int, [C.c_void_p, C.c_char_p]),
    "vampomi_generate_iid": (C.c_int, [C.c_void_p, C.c_ulonglong]),
    "vampomi_impute_missing": (C.c_int, [C.c_void_p, c_ll_p]),
    "vampomi_compute_stats": (C.c_int, [C.c_void_p, C.c_double]),
    "vampomi_get_stats": (C.c_int, [C.c_void_p, c_double_p, c_double_p]),
    "vampomi_constant_columns": (C.c_int, [C.c_void_p, c_u8_p]),
    "vampomi_atx": (C.c_int, [C.c_void_p, c_double_p, c_double_p]),
    "vampomi_ax": (C.c_int, [C.c_void_p, c_double_p, c_double_p]),
    "vampomi_vec_len": (C.c_int, [C.c_void_p, C.c_int, c_ll_p]),
    "vampomi_vec_set": (C.c_int, [C.c_void_p, C.c_int, c_double_p]),
    "vampomi_vec_get": (C.c_int, [C.c_void_p, C.c_int, c_double_p]),
    "vampomi_vec_get_scaled": (C.c_int, [C.c_void_p, C.c_int, C.c_double, c_double_p]),
    "vampomi_dump_begin": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_double]),
    "vampomi_dump_wait": (C.c_int, [C.c_void_p, C.c_int, c_double_p]),
    "vampomi_vec_fill": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "vampomi_vec_copy": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "vampomi_vec_lincomb": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_double, C.c_int, C.c_double]),
    "vampomi_dots": (C.c_int, [C.c_void_p, C.c_int, c_int_p, c_int_p, c_int_p, c_double_p, c_double_p]),
    "vampomi_draw_probe": (C.c_int, [C.c_void_p, C.c_ulonglong, C.c_int]),
    "vampomi_ax_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "vampomi_atx_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "vampomi_ax_multi_dev": (C.c_int, [C.c_void_p, C.c_int, c_int_p, c_int_p]),
    "vampomi_atx_multi_dev": (C.c_int, [C.c_void_p, C.c_int, c_int_p, c_int_p]),
    "vampomi_aat_multi_dev": (C.c_int, [C.c_void_p, C.c_int, c_int_p, c_int_p, c_int_p]),
    "vampomi_aat_supported": (C.c_int, [C.c_void_p, c_int_p]),
    "vampomi_denoise": (C.c_int, [C.c_void_p, C.c_double, c_double_p, c_double_p, C.c_int, C.c_int, C.c_double, c_double_p]),
    "vampomi_em_sums": (C.c_int, [C.c_void_p, C.c_double, C.c_double, c_double_p, c_double_p, C.c_int, c_double_p]),
    "vampomi_cg_solve": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int,
                                   C.c_int, c_int_p, c_double_p, c_double_p]),
    "vampomi_cg_solve_pair": (C.c_int, [C.c_void_p, c_int_p, c_int_p, c_int_p, c_int_p, C.c_double, C.c_double, C.c_double, C.c_int,
                                        c_int_p, C.c_int, C.c_int, c_int_p, c_int_p, c_double_p, c_double_p]),
    "vampomi_probit_zdenoise": (C.c_int, [C.c_void_p, C.c_double, c_double_p]),
    "vampomi_pvals_se": (C.c_int, [C.c_void_p, c_double_p, C.c_double, c_double_p]),
    "vampomi_loo_sums": (C.c_int, [C.c_void_p, C.c_int, c_double_p]),
    "vampomi_counters": (C.c_int, [C.c_void_p, c_ll_p, C.c_int]),
    "vampomi_time_kernel": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_double_p]),
    "vampomi_set_tuning": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "vampomi_plan_chunks": (C.c_longlong, [C.c_longlong, C.c_int, C.c_longlong, C.c_int, C.c_int]),
    "vampomi_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "vampomi_profile_read": (C.c_int, [C.c_void_p, c_double_p, C.c_int]),
    "vampomi_profile_read_ex": (C.c_int, [C.c_void_p, C.c_int, c_double_p, C.c_int]),
    "vampomi_stream": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    # host driver
    "vampomi_main": (C.c_int, [C.c_int, C.POINTER(C.c_char_p)]),
    "vampomi_main_probit": (C.c_int, [C.c_int, C.POINTER(C.c_char_p)]),
    "vampomi_solver_default_config": (None, [C.POINTER(SolverConfig)]),
    "vampomi_solver_create": (C.c_int, [C.c_void_p, C.POINTER(SolverConfig), c_double_p, c_double_p, c_double_p,
                                        C.POINTER(C.c_void_p)]),
    "vampomi_solver_set_covariates": (C.c_int, [C.c_void_p, C.c_int, c_double_p]),
    "vampomi_solver_get_cov_eff": (C.c_int, [C.c_void_p, C.c_int, c_double_p]),
    "vampomi_host_read_covariates": (C.c_longlong, [C.c_char_p, C.c_int, C.c_int, c_double_p]),
    "vampomi_host_newton_cov": (C.c_int, [c_double_p, c_double_p, c_double_p, C.c_int, C.c_int, c_double_p]),
    "vampomi_solver_save_state": (C.c_int, [C.c_void_p, C.c_char_p]),
    "vampomi_solver_load_state": (C.c_int, [C.c_void_p, C.c_char_p]),
    "vampomi_solver_step": (C.c_int, [C.c_void_p, C.POINTER(IterResult), c_double_p, c_double_p]),
    "vampomi_solver_destroy": (C.c_int, [C.c_void_p]),
    "vampomi_host_csv_row": (C.c_int, [C.c_uint, c_double_p, C.c_int, C.c_char_p, C.c_int]),
    "vampomi_host_read_phen": (C.c_longlong, [C.c_char_p, C.c_int, c_double_p, C.c_longlong]),
    "vampomi_host_linear_reg1d_pvals": (C.c_double, [C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int]),
    "vampomi_host_loo_pvals": (None, [c_double_p, c_double_p, C.c_double, C.c_double, C.c_int, C.c_longlong, c_double_p, C.c_int]),
    "vampomi_host_loo_pvals_flagged": (None, [c_double_p, c_double_p, C.c_double, C.c_double, C.c_int, C.c_longlong, c_u8_p,
                                              c_double_p, C.c_int]),
    "vampomi_host_probe_sign": (C.c_double, [C.c_ulonglong, C.c_int, C.c_ulonglong]),
    "vampomi_host_probit_p1": (None, [C.c_ulonglong, C.c_int, c_double_p]),
    "vampomi_host_merge_components": (C.c_int, [c_double_p, c_double_p, C.c_int, C.c_double]),
}

_lib = None


class VampomiError(RuntimeError):
    pass


def load_library(path=None):
    """Loads the shared library (built by vampomi_b200.build / __graft_entry__.build). Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    path = path or os.environ.get("VAMPOMI_LIB", LIB_PATH)
    if not os.path.isfile(path):
        raise VampomiError(f"{path} not found: build it with `python -m vampomi_b200.build` (nvcc, sm_100a). "
                           "There is no Python/CPU fallback for the VAMP kernels.")
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)


def last_error():
    return load_library().vampomi_last_error().decode(errors="replace")


def _check(rc, what):
    if rc != 0:
        raise VampomiError(f"{what} failed (code {rc}): {last_error()}")


def _in(a, n=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if n is not None and a.size != n:
        raise ValueError(f"expected {n} values, got {a.size}")
    return a, a.ctypes.data_as(c_double_p)


def _out(n):
    a = np.empty(int(n), dtype=np.float64)
    return a, a.ctypes.data_as(c_double_p)


def divide_work(Mt, nranks, rank):
    M, S = C.c_longlong(), C.c_longlong()
    _check(load_library().vampomi_divide_work(Mt, nranks, rank, C.byref(M), C.byref(S)), "divide_work")
    return M.value, S.value


def plan_chunks(slots, ntiles, M, min_cols=1, balance=True):
    """Column chunks of the tiled matrix kernels' grids (include/vampomi.h: vampomi_plan_chunks)."""
    return load_library().vampomi_plan_chunks(slots, ntiles, M, min_cols, int(bool(balance)))


def device_count():
    n = C.c_int()
    rc = load_library().vampomi_device_count(C.byref(n))
    return n.value if rc == 0 else 0


def comm_unique_id():
    buf = C.create_string_buffer(128)
    _check(load_library().vampomi_comm_get_unique_id(buf), "comm_get_unique_id")
    return buf.raw


class Shard:
    """One marker shard on one GPU: the `class data` of the reference (src/data.hpp:47-90) plus the device vectors."""

    def __init__(self, N, Mt, device=0, nranks=1, rank=0, nccl_id=None, storage="f64"):
        """storage: "f64" (the reference's layout) or "f32" (opt-in: the block is rounded to FP32 in HBM, arithmetic stays FP64)."""
        self.lib = load_library()
        h = C.c_void_p()
        self.storage = storage
        _check(self.lib.vampomi_create_ex(device, N, Mt, nranks, rank, {"f64": 0, "f32": 1}[storage], C.byref(h)), "vampomi_create")
        self.h = h
        self.N, self.Mt, self.nranks, self.rank = int(N), int(Mt), nranks, rank
        M, S = C.c_longlong(), C.c_longlong()
        _check(self.lib.vampomi_shard(self.h, C.byref(M), C.byref(S)), "vampomi_shard")
        self.M, self.S = M.value, S.value
        if nranks > 1 and nccl_id is not False:      # nccl_id=False: shard-local work only (no collective is legal)
            if nccl_id is None:
                raise ValueError("nccl_id is required when nranks > 1")
            _check(self.lib.vampomi_comm_init(self.h, C.c_char_p(nccl_id)), "vampomi_comm_init")

    def close(self):
        if getattr(self, "h", None):
            self.lib.vampomi_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def barrier(self):
        _check(self.lib.vampomi_barrier(self.h), "barrier")

    def comm_mode(self):
        """0 single shard, 1 NCCL all-reduce, 2 fused peer-memory all-reduce (include/vampomi.h)."""
        m = C.c_int()
        _check(self.lib.vampomi_comm_mode(self.h, C.byref(m)), "comm_mode")
        return m.value

    # ---- matrix ----
    def upload(self, A, j0=0):
        """A: [ncols, N] marker-major block (rows = markers)."""
        A = np.ascontiguousarray(A, dtype=np.float64)
        assert A.ndim == 2 and A.shape[1] == self.N
        _check(self.lib.vampomi_upload_columns(self.h, j0, A.shape[0], A.ctypes.data_as(c_double_p)), "upload_columns")

    def download(self, j0=0, ncols=None):
        ncols = self.M - j0 if ncols is None else ncols
        out = np.empty((ncols, self.N), dtype=np.float64)
        _check(self.lib.vampomi_download_columns(self.h, j0, ncols, out.ctypes.data_as(c_double_p)), "download_columns")
        return out

    def load_file(self, path):
        _check(self.lib.vampomi_load_file(self.h, os.fsencode(path)), "load_file")

    def generate_iid(self, seed):
        _check(self.lib.vampomi_generate_iid(self.h, seed), "generate_iid")

    def impute_missing(self):
        """Replaces every NaN of a column of this shard's block by the mean of the column's other entries (0 if it has none), in
        HBM, before compute_stats(). Returns (entries replaced, columns with a NaN, columns without an observed value)."""
        c = (C.c_longlong * 3)()
        _check(self.lib.vampomi_impute_missing(self.h, c), "impute_missing")
        return c[0], c[1], c[2]

    def compute_stats(self, alpha_scale=1.0):
        _check(self.lib.vampomi_compute_stats(self.h, alpha_scale), "compute_stats")

    def stats(self):
        (a, pa), (b, pb) = _out(self.M), _out(self.M)
        _check(self.lib.vampomi_get_stats(self.h, pa, pb), "get_stats")
        return a, b

    def constant_columns(self):
        """Boolean per column: compute_stats found it constant (mave = its value, msig = 1)."""
        out = np.zeros(self.M, dtype=np.uint8)
        _check(self.lib.vampomi_constant_columns(self.h, out.ctypes.data_as(c_u8_p)), "constant_columns")
        return out.astype(bool)

    def ATx(self, p):
        p, pp = _in(p, self.N)
        out, po = _out(self.M)
        _check(self.lib.vampomi_atx(self.h, pp, po), "atx")
        return out

    def Ax(self, x):
        x, px = _in(x, self.M)
        out, po = _out(self.N)
        _check(self.lib.vampomi_ax(self.h, px, po), "ax")
        return out

    # ---- vectors ----
    def vlen(self, vec):
        return self.M if vec < 32 else self.N

    def set(self, vec, values):
        a, pa = _in(values, self.vlen(vec))
        _check(self.lib.vampomi_vec_set(self.h, vec, pa), "vec_set")

    def get(self, vec, divisor=None):
        out, po = _out(self.vlen(vec))
        if divisor is None:
            _check(self.lib.vampomi_vec_get(self.h, vec, po), "vec_get")
        else:
            _check(self.lib.vampomi_vec_get_scaled(self.h, vec, divisor, po), "vec_get_scaled")
        return out

    def dump_begin(self, slot, vec, divisor=1.0):
        """Starts an asynchronous read-out of vec/divisor (snapshot now, copy underneath later work)."""
        _check(self.lib.vampomi_dump_begin(self.h, slot, vec, divisor), "dump_begin")
        if not hasattr(self, "_dump_len"):
            self._dump_len = {}
        self._dump_len[slot] = self.vlen(vec)

    def dump_wait(self, slot, out=None):
        out = np.empty(self._dump_len.pop(slot)) if out is None else out
        _check(self.lib.vampomi_dump_wait(self.h, slot, out.ctypes.data_as(c_double_p)), "dump_wait")
        return out

    def fill(self, vec, value):
        _check(self.lib.vampomi_vec_fill(self.h, vec, value), "vec_fill")

    def copy(self, dst, src):
        _check(self.lib.vampomi_vec_copy(self.h, dst, src), "vec_copy")

    def lincomb(self, dst, a, x, b, y, c=1.0):
        _check(self.lib.vampomi_vec_lincomb(self.h, dst, a, x, b, y, c), "vec_lincomb")

    def dots(self, items):
        """items: list of (kind, a, b[, scale]) -> np.array of sums."""
        n = len(items)
        kind = (C.c_int * n)(*[it[0] for it in items])
        a = (C.c_int * n)(*[it[1] for it in items])
        b = (C.c_int * n)(*[it[2] for it in items])
        sc = (C.c_double * n)(*[(it[3] if len(it) > 3 else 1.0) for it in items])
        out, po = _out(n)
        _check(self.lib.vampomi_dots(self.h, n, kind, a, b, sc, po), "dots")
        return out

    def draw_probe(self, seed, it):
        _check(self.lib.vampomi_draw_probe(self.h, seed, it), "draw_probe")

    def ax_dev(self, x_vec, out_vec):
        _check(self.lib.vampomi_ax_dev(self.h, x_vec, out_vec), "ax_dev")

    def atx_dev(self, p_vec, out_vec):
        _check(self.lib.vampomi_atx_dev(self.h, p_vec, out_vec), "atx_dev")

    def ax_multi_dev(self, x_vecs, out_vecs):
        """out_k = A x_k for up to 4 M-vectors in ONE pass over the marker block."""
        K = len(x_vecs)
        _check(self.lib.vampomi_ax_multi_dev(self.h, K, (C.c_int * K)(*x_vecs), (C.c_int * K)(*out_vecs)), "ax_multi_dev")

    def atx_multi_dev(self, p_vecs, out_vecs):
        """out_k = A^T p_k for up to 2 N-vectors in ONE pass over the marker block."""
        K = len(p_vecs)
        _check(self.lib.vampomi_atx_multi_dev(self.h, K, (C.c_int * K)(*p_vecs), (C.c_int * K)(*out_vecs)), "atx_multi_dev")

    def aat_multi_dev(self, q_vecs, t_out_vecs, w_out_vecs):
        """t_k = A^T q_k and w_k = A t_k for up to 2 N-vectors in ONE pass over the marker block (kernels_gram.cu)."""
        K = len(q_vecs)
        _check(self.lib.vampomi_aat_multi_dev(self.h, K, (C.c_int * K)(*q_vecs), (C.c_int * K)(*t_out_vecs), (C.c_int * K)(*w_out_vecs)),
               "aat_multi_dev")

    def aat_supported(self):
        y = C.c_int()
        _check(self.lib.vampomi_aat_supported(self.h, C.byref(y)), "aat_supported")
        return bool(y.value)

    # ---- VAMP pieces ----
    def denoise(self, gam1, probs, vars_internal, damp=False, rho=0.5):
        p, pp = _in(probs)
        v, pv = _in(vars_internal, p.size)
        s = C.c_double()
        _check(self.lib.vampomi_denoise(self.h, gam1, pp, pv, p.size, int(bool(damp)), rho, C.byref(s)), "denoise")
        return s.value

    def em_sums(self, gam1, lam, omegas, vars_internal):
        o, po = _in(omegas)
        v, pv = _in(vars_internal, o.size)
        out, pout = _out(2 * o.size - 1)
        _check(self.lib.vampomi_em_sums(self.h, gam1, lam, po, pv, o.size, pout), "em_sums")
        return out

    def cg_solve(self, rhs_vec, sol_vec, tau, gam2, warm_start=False, tol=1e-5, max_iter=500, onsager_mode=False):
        iters, rel, vmu = C.c_int(), C.c_double(), C.c_double()
        _check(self.lib.vampomi_cg_solve(self.h, rhs_vec, sol_vec, int(bool(warm_start)), tau, gam2, tol, max_iter,
                                         int(bool(onsager_mode)), C.byref(iters), C.byref(rel), C.byref(vmu)), "cg_solve")
        return iters.value, rel.value, vmu.value

    def cg_solve_pair(self, rhs_vecs, sol_vecs, tau, gam2, warm_start=(False, False), warm_ata_vecs=(-1, -1), tol=1e-5,
                      max_iter=500, onsager_mode=(False, True), extra=None, track_ax_vecs=(-1, -1)):
        """Two solves with the same operator in lock-step (one read of the marker block per pass for both).
        extra: optional (x_vec, out_vec) — out = A x computed on the first pass. track_ax_vecs: N-vectors kept equal to
        A sol by the solve's own recurrence. Returns [(iters, rel_err, <rhs,sol>)] * 2."""
        i2 = C.c_int * 2
        iters, rel, vmu = i2(), (C.c_double * 2)(), (C.c_double * 2)()
        ex, eo = extra if extra is not None else (-1, -1)
        _check(self.lib.vampomi_cg_solve_pair(self.h, i2(*rhs_vecs), i2(*sol_vecs), i2(*[int(bool(w)) for w in warm_start]),
                                              i2(*warm_ata_vecs), tau, gam2, tol, max_iter,
                                              i2(*[int(bool(o)) for o in onsager_mode]), ex, eo, i2(*track_ax_vecs), iters, rel, vmu),
               "cg_solve_pair")
        return [(iters[s], rel[s], vmu[s]) for s in range(2)]

    def probit_zdenoise(self, tau1):
        s = C.c_double()
        _check(self.lib.vampomi_probit_zdenoise(self.h, tau1, C.byref(s)), "probit_zdenoise")
        return s.value

    def pvals_se(self, r1, gam1):
        r, pr = _in(r1, self.M)
        out, po = _out(self.M)
        _check(self.lib.vampomi_pvals_se(self.h, pr, gam1, po), "pvals_se")
        return out

    def loo_sums(self, w_vec):
        out, po = _out(3 * self.M)
        _check(self.lib.vampomi_loo_sums(self.h, w_vec, po), "loo_sums")
        return out.reshape(self.M, 3)

    # ---- instrumentation ----
    def counters(self, reset=False):
        c = (C.c_longlong * 4)()
        _check(self.lib.vampomi_counters(self.h, c, int(reset)), "counters")
        return dict(kernels=c[0], matrix_passes=c[1], matrix_bytes=c[2], allreduces=c[3])

    def time_kernel(self, which, reps=10):
        ms = C.c_double()
        _check(self.lib.vampomi_time_kernel(self.h, which, reps, C.byref(ms)), "time_kernel")
        return ms.value

    def profile(self, on=True):
        _check(self.lib.vampomi_profile_enable(self.h, int(on)), "profile_enable")

    def profile_read(self, reset=False):
        out, po = _out(12)
        _check(self.lib.vampomi_profile_read_ex(self.h, 4, po, int(reset)), "profile_read")
        names = ("ax_partial", "ax_reduce", "atx", "gram")
        return {n: dict(launches=int(out[3 * i]), ms=float(out[3 * i + 1]), bytes=float(out[3 * i + 2])) for i, n in enumerate(names)}

    def stream(self):
        p = C.c_void_p()
        _check(self.lib.vampomi_stream(self.h, C.byref(p)), "stream")
        return p.value

    def set_tuning(self, name, value):
        _check(self.lib.vampomi_set_tuning(self.h, name.encode(), int(value)), f"set_tuning({name})")


class Solver:
    """The VAMP loop as a stepping object (`class vamp`, src/vamp.hpp:83-150): one step() = one VAMP iteration."""

    def __init__(self, shard, y, model="linear", true_signal=None, x1hat_init=None, probs=None, vars=None, **kw):
        self.shard = shard
        self.lib = shard.lib
        cfg = SolverConfig()
        self.lib.vampomi_solver_default_config(C.byref(cfg))
        cfg.model = {"linear": 0, "bin_class": 1}[model]
        if probs is not None or vars is not None:
            assert probs is not None and vars is not None and len(probs) == len(vars) <= MAX_MIX
            cfg.L = len(probs)
            for i in range(cfg.L):
                cfg.probs[i] = probs[i]
                cfg.vars[i] = vars[i]
        for k, v in kw.items():
            if not hasattr(cfg, k):
                raise TypeError(f"unknown solver option {k}")
            setattr(cfg, k, v)
        self.cfg = cfg
        y, py = _in(y, shard.N)
        pts = px0 = None
        if true_signal is not None:
            ts, pts = _in(true_signal, shard.M)
        if x1hat_init is not None:
            x0, px0 = _in(x1hat_init, shard.M)
        h = C.c_void_p()
        _check(self.lib.vampomi_solver_create(shard.h, C.byref(cfg), py, pts, px0, C.byref(h)), "solver_create")
        self.h = h

    def set_covariates(self, Z):
        """Z: standardised covariates, shape (N, C) (read_covariates). Before the first step."""
        Z = np.ascontiguousarray(Z, dtype=np.float64)
        assert Z.ndim == 2 and Z.shape[0] == self.shard.N
        self.C = Z.shape[1]
        _check(self.lib.vampomi_solver_set_covariates(self.h, self.C, Z.ctypes.data_as(c_double_p)), "solver_set_covariates")

    def cov_eff(self):
        out, po = _out(self.C)
        _check(self.lib.vampomi_solver_get_cov_eff(self.h, self.C, po), "solver_get_cov_eff")
        return out

    def save_state(self, path):
        _check(self.lib.vampomi_solver_save_state(self.h, str(path).encode()), "solver_save_state")

    def load_state(self, path):
        _check(self.lib.vampomi_solver_load_state(self.h, str(path).encode()), "solver_load_state")

    def step(self, want_vectors=True, out_x1=None, out_r1=None):
        res = IterResult()
        x1 = r1 = None
        px = pr = None
        if want_vectors:
            x1 = out_x1 if out_x1 is not None else np.empty(self.shard.M)
            r1 = out_r1 if out_r1 is not None else np.empty(self.shard.M)
            px, pr = x1.ctypes.data_as(c_double_p), r1.ctypes.data_as(c_double_p)
        _check(self.lib.vampomi_solver_step(self.h, C.byref(res), px, pr), "solver_step")
        return dict(it=res.it, params=list(res.params[:res.n_params]), metrics=list(res.metrics[:res.n_metrics]),
                    nmse=res.nmse, gam1_next=res.gam1_next, k1=res.cg_iters_lmmse, k2=res.cg_iters_onsager,
                    probs=list(res.probs[:res.L]), vars=list(res.vars[:res.L]), matrix_passes=res.matrix_passes,
                    x1=x1, r1=r1)

    def close(self):
        if getattr(self, "h", None):
            self.lib.vampomi_solver_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def main(argv):
    """Runs the main_meth command line in-process (include/vampomi_host.h: vampomi_main)."""
    lib = load_library()
    args = [b"main_meth"] + [os.fsencode(a) for a in argv]
    arr = (C.c_char_p * len(args))(*args)
    return lib.vampomi_main(len(args), arr)
