/*
 * vampomi.h — C ABI of libvampomi_cuda.so: the B200 (sm_100a) implementation of gVAMPomi's VAMP hot path.
 *
 * The reference (medical-genomics-group/VAMPomi) has no FFI or plugin seam; its inner seam is `class data`
 * (src/data.hpp:47-90: Ax, ATx, pvals_loo, getters) called by `class vamp` (src/vamp.hpp:83-150). Each entry point
 * below names the reference interface it replaces (file:line relative to the reference repository root).
 *
 * Conventions
 *   - One context = one marker shard on one GPU (= one MPI rank of the reference, src/utilities.cpp:207-239).
 *   - Every function returns 0 on success, non-zero on failure; vampomi_last_error() describes the last failure
 *     on the calling thread. No exceptions cross this boundary. There is NO CPU fallback: without a CUDA device
 *     every compute entry point fails with VAMPOMI_ERR_CUDA.
 *   - Host buffers are caller-owned, plain `double*` (FP64, little endian), marker-major for matrices
 *     (column j of the N x M design matrix is the j-th run of N doubles — README.md:16 / src/data.cpp:297).
 *   - Device memory is library-owned. Device-resident vectors are addressed by the ids below; ids < 32 have
 *     length M (this shard's markers), ids >= 32 have length N (samples, replicated on every shard).
 *   - Calls on one context must come from one thread at a time. With nranks > 1 every rank must make the same
 *     sequence of calls (collectives inside, exactly like MPI_Allreduce inside data::Ax, src/data.cpp:367).
 */
#ifndef VAMPOMI_H
#define VAMPOMI_H

#ifdef __cplusplus
extern "C" {
#endif

#define VAMPOMI_ABI_VERSION 1

enum {
    VAMPOMI_OK = 0,
    VAMPOMI_ERR_ARG = 1,       /* bad argument */
    VAMPOMI_ERR_CUDA = 2,      /* CUDA runtime/driver failure (includes "no device") */
    VAMPOMI_ERR_NCCL = 3,      /* NCCL failure or libnccl not loadable */
    VAMPOMI_ERR_IO = 4,        /* file could not be opened / short read */
    VAMPOMI_ERR_STATE = 5      /* call made in the wrong state (e.g. Ax before statistics) */
};

/* Device-resident vectors. M-vectors are sharded like the reference's rank-local std::vector<double>(M). */
enum {
    VAMPOMI_V_X1 = 0,          /* x1_hat                      src/vamp.hpp:21 */
    VAMPOMI_V_X1_PREV = 1,     /* x1_hat_prev                 src/vamp.cpp:128 */
    VAMPOMI_V_R1 = 2,          /* r1                          src/vamp.hpp:25 */
    VAMPOMI_V_R2 = 3,          /* r2 */
    VAMPOMI_V_X2 = 4,          /* x2_hat (= CG solution of the LMMSE solve; also mu_CG_last, src/vamp.cpp:753) */
    VAMPOMI_V_V = 5,           /* right-hand side v           src/vamp.cpp:301-306 */
    VAMPOMI_V_BERN = 6,        /* bern_vec (Hutchinson probe) src/vamp.hpp:52 */
    VAMPOMI_V_QINV_BERN = 7,   /* invQ_bern_vec               src/vamp.hpp:53 */
    VAMPOMI_V_TRUE = 8,        /* true_signal                 src/vamp.hpp:21 */
    VAMPOMI_V_ATY = 9,         /* A^T y (iteration-invariant; the reference recomputes it, src/vamp.cpp:303) */
    VAMPOMI_V_TMP_M0 = 10,
    VAMPOMI_V_TMP_M1 = 11,
    VAMPOMI_V_CG_R = 12, VAMPOMI_V_CG_Z = 13, VAMPOMI_V_CG_P = 14, VAMPOMI_V_CG_D = 15,   /* src/vamp.cpp:679-692 */
    VAMPOMI_V_USER_M0 = 16,    /* never touched by the library itself (TMP_* and CG_* are clobbered by its calls) */
    VAMPOMI_V_USER_M1 = 17,
    VAMPOMI_V_CG2_R = 18, VAMPOMI_V_CG2_Z = 19, VAMPOMI_V_CG2_P = 20, VAMPOMI_V_CG2_D = 21,   /* second system of a paired solve */
    VAMPOMI_V_ATA_X2 = 22,     /* A^T A x2_hat, kept from one iteration to the next (the warm start's residual needs it) */
    VAMPOMI_V_NUM_M = 23,

    VAMPOMI_V_Y = 32,          /* phenotype y                 src/vamp.hpp:23 */
    VAMPOMI_V_Z1 = 33,         /* z1 = A x1_hat               src/vamp.hpp:24 */
    VAMPOMI_V_Z2 = 34,         /* A x2_hat */
    VAMPOMI_V_P1 = 35,         /* probit p1                   src/vamp.hpp:26 */
    VAMPOMI_V_P2 = 36,         /* probit p2 */
    VAMPOMI_V_Z1HAT = 37,      /* probit z1_hat               src/vamp.hpp:22 */
    VAMPOMI_V_TMP_N0 = 38,
    VAMPOMI_V_TMP_N1 = 39,
    VAMPOMI_V_USER_N0 = 40,
    VAMPOMI_V_USER_N1 = 41,
    VAMPOMI_V_GRAM_W0 = 42, VAMPOMI_V_GRAM_W1 = 43,     /* work: w = A A^T q of the one-pass CG, one per system */
    VAMPOMI_V_GRAM_AR0 = 44, VAMPOMI_V_GRAM_AR1 = 45,   /* work: A r of the one-pass CG */
    VAMPOMI_V_MCOV = 46,       /* probit: covariate offset m_cov = Z cov_eff (src/vamp_probit.cpp:214-217); zero without covariates */
    VAMPOMI_V_NUM_N = 15
};

/* Kinds for vampomi_dots(): out = sum_i f(a_i, b_i). */
enum {
    VAMPOMI_DOT = 0,           /* a_i * b_i                     inner_prod, src/utilities.cpp:138-158 */
    VAMPOMI_DIFF2 = 1,         /* (a_i - b_i)^2                 e.g. l2_norm2(x1_hat_prev - x1_hat), src/vamp.cpp:409-413 */
    VAMPOMI_SQDEV = 2          /* (a_i - s * b_i)^2, s = scale  e.g. src/vamp.cpp:264-267 */
};

typedef struct vampomi_ctx vampomi_ctx;

/* ---- lifecycle ------------------------------------------------------------------------------------------- */
const char* vampomi_last_error(void);
int vampomi_abi_version(void);
/* Number of visible CUDA devices (0 and VAMPOMI_ERR_CUDA when there is none). */
int vampomi_device_count(int* count);

/* Creates the shard `rank` of `nranks` on CUDA device `device`. The marker split is the reference's divide_work
 * (src/utilities.cpp:214-225): first Mt % nranks shards get floor(Mt/nranks)+1 markers. Allocates the M x N block
 * in HBM (column stride padded to a multiple of 16 doubles) and all work vectors. */
int vampomi_create(int device, int N, long long Mt, int nranks, int rank, vampomi_ctx** out);
/* Same, with a choice of how the marker block is HELD in HBM: VAMPOMI_STORE_F64 (the reference's layout, what
 * vampomi_create uses) or VAMPOMI_STORE_F32 — every value is rounded to FP32 when it is uploaded / loaded / generated and
 * widened back to FP64 inside the kernels, so all arithmetic and every interface stay FP64 while each matrix pass streams
 * half the bytes. This is an opt-in mode outside the reference's contract: results equal those of the reference run on
 * the ROUNDED matrix (to the usual 1e-9), not on the original one. */
#define VAMPOMI_STORE_F64 0
#define VAMPOMI_STORE_F32 1
int vampomi_create_ex(int device, int N, long long Mt, int nranks, int rank, int storage, vampomi_ctx** out);
int vampomi_storage(const vampomi_ctx* ctx, int* storage);
int vampomi_destroy(vampomi_ctx* ctx);
/* M (markers of this shard) and S (global index of its first marker) — divide_work's MS[0], MS[1]. */
int vampomi_shard(const vampomi_ctx* ctx, long long* M, long long* S);
/* Problem dimensions the context was created with (any pointer may be NULL). */
int vampomi_dims(const vampomi_ctx* ctx, int* N, long long* Mt, int* nranks, int* rank);
/* Pure host helper with the same rule, usable without a GPU. */
int vampomi_divide_work(long long Mt, int nranks, int rank, long long* M, long long* S);

/* ---- multi-GPU (replaces MPI_COMM_WORLD; one NCCL rank per context) --------------------------------------- */
/* Rank 0 calls get_unique_id and ships the 128 bytes to the other ranks by any means (torch.distributed, a
 * file, a thread-shared buffer); then every rank calls comm_init. Not needed when nranks == 1. */
int vampomi_comm_get_unique_id(void* id128);
int vampomi_comm_init(vampomi_ctx* ctx, const void* id128);
/* How cross-GPU sums are carried out: 0 = single shard (none), 1 = NCCL all-reduce after the producing kernel,
 * 2 = one-shot all-reduce over NVLink peer memory fused into the producing kernels (A x partial reduce and the CG
 * scalar reductions; csrc/xchg.cuh). Mode 2 is chosen at comm_init when every rank could map every peer (CUDA IPC
 * between processes, peer access between threads); the environment variable VAMPOMI_XCHG=0 forces mode 1. */
int vampomi_comm_mode(const vampomi_ctx* ctx, int* mode);
/* All ranks meet here (MPI_Barrier, src/data.cpp:148 / src/vamp.cpp:434): returns once every rank has called it and this rank's
 * stream has drained. vampomi_compute_stats ends with one, so no rank starts an operator (and with it the wall-clock limit of
 * the device-side peer waits, 120 s or VAMPOMI_XCHG_TIMEOUT_S) while another is still loading its shard. A peer wait that does
 * run out raises a flag instead of faulting; the next synchronising call on that context fails with VAMPOMI_ERR_STATE. */
int vampomi_barrier(vampomi_ctx* ctx);

/* ---- design matrix: data::read_methylation_data, src/data.cpp:116-153 -------------------------------------- */
/* Copies `ncols` columns (each N doubles, contiguous) starting at local column j0 from host memory to HBM. */
int vampomi_upload_columns(vampomi_ctx* ctx, long long j0, long long ncols, const double* host);
int vampomi_download_columns(vampomi_ctx* ctx, long long j0, long long ncols, double* host);
/* Reads this shard's block [S, S+M) of a marker-major FP64 file (byte offset S*N*8, src/data.cpp:134) through a
 * ring of pinned staging buffers, overlapping pread with the host-to-device copies. */
int vampomi_load_file(vampomi_ctx* ctx, const char* path);
/* Synthetic i.i.d. N(0,1) block generated on the device from a counter hash of (seed, global marker, sample):
 * identical for any sharding (the model of simulation/data_sim.py:35). */
int vampomi_generate_iid(vampomi_ctx* ctx, unsigned long long seed);
/* Missing values (opt-in; the reference has no such step): every NaN entry of a column of this shard's block, whatever its
 * sign or payload, is replaced in HBM by the mean of that column's non-NaN entries (0 for a column without any), so the
 * run that follows is the run on the imputed matrix. +-Inf is not missing. In FP32 storage the mean is rounded to FP32.
 * Columns without NaN are not written. Call after load_file / upload_columns / generate_iid and before compute_stats (it
 * invalidates the statistics). No communication: a column lives in one shard. counts, for this shard: [0] entries replaced,
 * [1] columns with at least one NaN, [2] columns without an observed value. */
int vampomi_impute_missing(vampomi_ctx* ctx, long long counts[3]);

/* ---- marker statistics: data::compute_markers_statistics, src/data.cpp:233-283 ----------------------------- */
int vampomi_compute_stats(vampomi_ctx* ctx, double alpha_scale);
int vampomi_get_stats(vampomi_ctx* ctx, double* mave_M, double* msig_M);
/* const_M[j] = 1 if compute_stats found column j constant (no NaN, min == max, finite: mave = its value, msig = 1), else 0. The same
 * decision, not a threshold on a variance; vampomi_host_loo_pvals_flagged gives such a column p = 1. */
int vampomi_constant_columns(vampomi_ctx* ctx, unsigned char* const_M);

/* ---- operators with host buffers: data::ATx (src/data.cpp:315-333) and data::Ax (src/data.cpp:340-373) ------ */
/* out_M[j] = msig[j] * sum_i (A[i,j]-mave[j]) * p[i] * (1/sqrt(N)) */
int vampomi_atx(vampomi_ctx* ctx, const double* p_N, double* out_M);
/* out_N[i] = (sum over ALL shards of sum_j (A[i,j]-mave[j]) * msig[j]*x[j]) / sqrt(N) */
int vampomi_ax(vampomi_ctx* ctx, const double* x_M, double* out_N);

/* ---- device-resident vectors ------------------------------------------------------------------------------- */
int vampomi_vec_len(const vampomi_ctx* ctx, int vec, long long* len);
int vampomi_vec_set(vampomi_ctx* ctx, int vec, const double* host);
int vampomi_vec_get(vampomi_ctx* ctx, int vec, double* host);
/* host[i] = vec[i] / divisor — the x/sqrt(N) dumps of src/vamp.cpp:237-249. */
int vampomi_vec_get_scaled(vampomi_ctx* ctx, int vec, double divisor, double* host);
/* The same read-out without a host round trip in the middle of an iteration (the per-iteration dumps of a running
 * solver): begin() enqueues, on the context's stream, a snapshot of vec/divisor and its copy to pinned host memory and
 * returns at once, so the caller keeps enqueueing work behind it; wait() blocks until that copy has landed and hands it to `host`.
 * Two independent slots (0, 1); a slot must be waited for before it is begun again. */
int vampomi_dump_begin(vampomi_ctx* ctx, int slot, int vec, double divisor);
int vampomi_dump_wait(vampomi_ctx* ctx, int slot, double* host);
int vampomi_vec_fill(vampomi_ctx* ctx, int vec, double value);
int vampomi_vec_copy(vampomi_ctx* ctx, int dst, int src);
/* dst[i] = (a*x[i] + b*y[i]) / c — every message update of src/vamp.cpp:259-261,305-306,348-350 and
 * src/vamp_probit.cpp:197-198,250-251,302-303,337-338,367-368 has this shape. */
int vampomi_vec_lincomb(vampomi_ctx* ctx, int dst, double a, int x, double b, int y, double c);
/* n reductions in one launch + (for M-vectors, nranks>1) one all-reduce + one host sync. `scale` may be NULL. */
int vampomi_dots(vampomi_ctx* ctx, int n, const int* kind, const int* a, const int* b, const double* scale, double* out);
/* bern_vec[j] = +-1/sqrt(Mt) from the counter hash of (seed, it, S+j) — replaces the std::random_device draw of
 * src/vamp.cpp:295-296 / src/vamp_probit.cpp:297-298 (oracle patch P2). */
int vampomi_draw_probe(vampomi_ctx* ctx, unsigned long long seed, int it);
/* Operators on device vectors (no host traffic): out = A x (x: M-vector id, out: N-vector id) and out = A^T p. */
int vampomi_ax_dev(vampomi_ctx* ctx, int x_vec, int out_vec);
int vampomi_atx_dev(vampomi_ctx* ctx, int p_vec, int out_vec);
/* The same operators applied to K vectors in ONE pass over the marker block (K <= 4 for A x, K <= 2 for A^T p): every
 * pass is bound by streaming A from HBM, so K independent products cost one read of A instead of K. Each vector keeps the
 * arithmetic of the single-vector call. out_k = A x_k (x: M-vector ids, out: distinct N-vector ids) / out_k = A^T p_k. */
int vampomi_ax_multi_dev(vampomi_ctx* ctx, int K, const int* x_vecs, const int* out_vecs);
int vampomi_atx_multi_dev(vampomi_ctx* ctx, int K, const int* p_vecs, const int* out_vecs);

/* The FUSED pair of products t_k = A^T q_k (M-vectors) and w_k = A t_k = A A^T q_k (N-vectors, summed over all shards) for
 * K <= 2 vectors in ONE pass over the marker block: each column is kept on chip between its dot product and its axpy
 * (csrc/kernels_gram.cu). This is lmmse_mult's ATx(Ax(.)) (src/vamp.cpp:653-654) re-associated around the N-side vector, and
 * what lets a CG iteration read the block once instead of twice (tuning knob cg_onepass / schedule "onepass"). Every
 * product keeps the per-element arithmetic of vampomi_atx_dev / vampomi_ax_dev. Needs FP64 storage and N <= 40960 (clusters of 8 CTAs up to 20480 rows, of 16 beyond)
 * (vampomi_aat_supported); q_vecs / w_out_vecs name N-vectors, t_out_vecs M-vectors, all distinct. */
int vampomi_aat_multi_dev(vampomi_ctx* ctx, int K, const int* q_vecs, const int* t_out_vecs, const int* w_out_vecs);
int vampomi_aat_supported(const vampomi_ctx* ctx, int* yes);

/* ---- Gaussian-mixture denoiser: vamp::g1 / vamp::g1d, src/vamp.cpp:440-492, as used at :203-223 ------------- */
/* X1_PREV <- X1; X1 <- g1(R1, gam1) (then rho*X1 + (1-rho)*X1_PREV if damp != 0); *sum_g1d = sum over ALL shards of
 * g1d(R1_j, gam1). `vars` are the internal (already multiplied by N, src/vamp.cpp:87-88) variances. L <= 32. */
int vampomi_denoise(vampomi_ctx* ctx, double gam1, const double* probs, const double* vars, int L,
                    int damp, double rho, double* sum_g1d);

/* ---- EM prior update, per-marker part of vamp::updatePrior, src/vamp.cpp:554-597 ---------------------------- */
/* sums[0] = sum pin_i; sums[1..L-1] = sum beta_ij pin_i; sums[L..2L-2] = sum beta_ij (gamma_ij^2 + v_j) pin_i,
 * over ALL shards (one packed all-reduce instead of the reference's 1+2(L-1) scalar ones). */
int vampomi_em_sums(vampomi_ctx* ctx, double gam1, double lambda, const double* omegas, const double* vars, int L,
                    double* sums);

/* ---- LMMSE solve: vamp::precondCG_solver + vamp::lmmse_mult, src/vamp.cpp:645-757 --------------------------- */
/* Solves (tau A^T A + gam2 I) sol = rhs by Jacobi-preconditioned CG, entirely on the device: alpha/beta and the
 * stopping tests are computed by kernels, the host only polls a completion flag.
 *   warm_start != 0: start from the current content of `sol_vec` (src/vamp.cpp:311); else from zero (:309,:668).
 *   onsager_mode != 0 is the reference's denoiser==0 branch (:708-726): additionally stop when the relative change
 *   of gam2*<rhs,sol> drops below 1e-8; *rhs_dot_sol returns <rhs, sol> for the returned sol (src/vamp.cpp:498).
 *   *iters = number of CG iterations executed; *rel_err = last ||r||/||rhs|| (NaN if the onsager test ended it). */
int vampomi_cg_solve(vampomi_ctx* ctx, int rhs_vec, int sol_vec, int warm_start, double tau, double gam2,
                     double tol, int max_iter, int onsager_mode, int* iters, double* rel_err, double* rhs_dot_sol);

/* Two solves with the SAME operator (tau A^T A + gam2 I) advanced in lock-step: system 0 and system 1 share every matrix
 * pass (one read of the marker block per A p and per A^T (A p) for both), while each keeps exactly the scalars, the
 * stopping tests and the iteration count it would have in vampomi_cg_solve — a system that has converged is skipped by
 * all later launches. This is how one VAMP iteration runs its LMMSE solve (src/vamp.cpp:308-311) and its Onsager / trace
 * solve (:494-501) in max(k1, k2) instead of k1 + k2 CG iterations' worth of passes.
 *   warm_ata_vec[s]: only read when warm_start[s] != 0 — id of an M-vector that already holds A^T A sol_s (e.g. from a
 *     vampomi_atx_multi_dev of an earlier A sol_s), or -1 to compute it here with two extra passes.
 *   extra_x_vec / extra_out_vec: if extra_x_vec >= 0, extra_out = A extra_x is computed by the first A p pass of the solve
 *     (a third vector on the same read); pass -1 for none.
 *   track_ax_vec (may be NULL; entries -1 = off): N-vector that the solve keeps equal to A sol_s from its OWN products —
 *     it must hold A sol_s on entry when warm_start[s] (it is zeroed for a zero start) and is advanced by alpha * (A p) in
 *     every iteration, the same recurrence that advances sol_s by alpha * p. After the solve A sol_s is there without a
 *     pass of its own (the reference computes A x2_hat and A Q^-1 u with extra passes, src/vamp.cpp:508,518). Likewise
 *     A^T A sol_s follows from the solve's residual: (rhs - r - gam2 sol)/tau with r in VAMPOMI_V_CG_R / _CG2_R.
 * rhs/sol must be distinct, non-work M-vectors. Outputs are arrays of two. */
int vampomi_cg_solve_pair(vampomi_ctx* ctx, const int rhs_vec[2], const int sol_vec[2], const int warm_start[2],
                          const int warm_ata_vec[2], double tau, double gam2, double tol, int max_iter,
                          const int onsager_mode[2], int extra_x_vec, int extra_out_vec, const int track_ax_vec[2],
                          int iters[2], double rel_err[2], double rhs_dot_sol[2]);

/* ---- probit z-channel: vamp::g1_bin_class / g1d_bin_class, src/vamp_probit.cpp:469-488 as used at :213-236 --- */
/* Z1HAT <- g1_bin_class(P1, tau1, Y, m_cov); *sum_g1d = sum_i g1d_bin_class(P1_i, tau1, Y_i, m_cov_i), m_cov = VAMPOMI_V_MCOV (0 unless set). */
int vampomi_probit_zdenoise(vampomi_ctx* ctx, double tau1, double* sum_g1d);

/* ---- association tests -------------------------------------------------------------------------------------- */
/* se (src/main_meth.cpp:229-243): p_j = cdf(normal(r1_j, sqrt(1/(gam1*N))), 0), 1-p_j when r1_j <= 0. */
int vampomi_pvals_se(vampomi_ctx* ctx, const double* r1_M, double gam1, double* pvals_M);
/* loo (src/data.cpp:385-417): per-marker raw-column sums over the N samples against w = y - z1:
 * sums_3M[3j] = sum x, [3j+1] = sum x^2, [3j+2] = sum x*w. The t statistic and p-value follow on the host. */
int vampomi_loo_sums(vampomi_ctx* ctx, int w_vec, double* sums_3M);

/* ---- instrumentation ---------------------------------------------------------------------------------------- */
/* Counters since creation/reset: [0] kernels launched, [1] full passes over the matrix block (Ax/ATx/loo/stats),
 * [2] bytes those passes streamed, [3] all-reduces issued. */
int vampomi_counters(vampomi_ctx* ctx, long long out[4], int reset);
/* Times `reps` back-to-back launches of one matrix kernel with CUDA events on the context's stream.
 * which: 0 = Ax (partial + reduce), 1 = ATx, 2 = stats, 3 = loo sums, 4 = read-bandwidth probe (a plain linear streaming
 * read of the whole marker block, not part of the VAMP path: the live ceiling the matrix kernels are compared with),
 * 5 = A x for 2 vectors in one pass, 6 = A^T p for 2 vectors in one pass, 7 = the multi-vector A^T p kernel with 1 vector,
 * 8 = A x for 3 vectors in one pass, 9 = the fused A^T q / A A^T q pass for 2 vectors, 10 = the same for 1 vector.
 * Returns average milliseconds per launch. */
int vampomi_time_kernel(vampomi_ctx* ctx, int which, int reps, double* ms_avg);
/* Per-kernel device timing of the matrix passes (CUDA events on the context stream around every launch while enabled).
 * read(): out[3k] = launches, out[3k+1] = total ms, out[3k+2] = bytes of A streamed, for k = 0 (k_ax_partial),
 * 1 (k_ax_reduce + all-reduce + scaling) and 2 (k_atx); synchronises the stream; `reset` clears the accumulators. */
int vampomi_profile_enable(vampomi_ctx* ctx, int on);
int vampomi_profile_read(vampomi_ctx* ctx, double out[9], int reset);
/* The same for the first `nkinds` <= 4 kernel kinds (out[3*nkinds]); kind 3 = the fused A^T q / A A^T q pass (k_gram). */
int vampomi_profile_read_ex(vampomi_ctx* ctx, int nkinds, double* out, int reset);
/* The CUDA stream (cudaStream_t) all work of this context is enqueued on — for callers that time with their own events. */
int vampomi_stream(vampomi_ctx* ctx, void** stream);
/* Pure host helper (no GPU needed): the number of column chunks the (row tile x column chunk) grids of the tiled matrix
 * kernels use for `slots` resident CTAs (SMs x CTAs per SM) and `ntiles` row tiles — the smallest number of full waves that
 * fills the slots to 99 % (balance != 0) or one, possibly partly filled, wave (balance == 0); at least `min_cols` columns
 * per chunk. Returns the chunk count (>= 1). */
long long vampomi_plan_chunks(long long slots, int ntiles, long long M, int min_cols, int balance);
/* Tuning knobs (kernel variants); see DESIGN.md. Unknown names fail with VAMPOMI_ERR_ARG. */
int vampomi_set_tuning(vampomi_ctx* ctx, const char* name, int value);

#ifdef __cplusplus
}
#endif
#endif /* VAMPOMI_H */
