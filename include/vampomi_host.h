/*
 * vampomi_host.h — C entry points of the C++ host driver that sits ABOVE the kernel ABI (vampomi.h).
 *
 * The driver is the B200 counterpart of the reference's main_meth.exe (src/main_meth.cpp:9-270) and of
 * `class vamp` (src/vamp.hpp:83-150): it owns the command line, the phenotype / vector / CSV files and the VAMP
 * iteration logic, and reaches the GPU only through the functions declared in vampomi.h.
 *
 *   vampomi_main          the whole program: same flags, run modes and output files as main_meth.exe
 *   vampomi_solver_*      the VAMP loop as a stepping object (one call = one VAMP iteration, src/vamp.cpp:148-428 or
 *                         src/vamp_probit.cpp:68-463) for callers that hold their data in memory (bench, tests)
 */
#ifndef VAMPOMI_HOST_H
#define VAMPOMI_HOST_H

#include "vampomi.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Runs main_meth's command line (argv[0] is ignored). Returns the process exit status (0 ok, 1 after a FATAL line).
 * With --gpus G > 1 it drives G marker shards from G host threads of this process, one GPU each. */
int vampomi_main(int argc, char** argv);
/* The same program entered as main_meth_probit (src/main_meth_probit.cpp:8-233; BASELINE.json configuration 4): --model is forced to
 * bin_class, `--run-mode test` writes the probit confusion-matrix rows [TP, TN, FP, FN, ACC] of that driver (:104-200) and
 * `--run-mode predict` its z_hat text file "<estimate file up to 'it'>.yhat" (:201-227). */
int vampomi_main_probit(int argc, char** argv);

#define VAMPOMI_MAX_MIX 32

typedef struct vampomi_solver_config {
    /* defaults in comments: src/options.hpp:63-104 / src/main_meth.cpp:51-66 */
    int model;                 /* 0 = linear (src/vamp.cpp:110), 1 = bin_class / probit (src/vamp_probit.cpp:19) */
    double gam1;               /* 1e-6 */
    double gamw;               /* 1/(1-h2), h2 = 0.5 */
    double rho;                /* 0.5 */
    int CG_max_iter;           /* 500 */
    double CG_err_tol;         /* 1e-5 */
    int EM_max_iter;           /* 1 */
    double EM_err_thr;         /* 1e-2 */
    int learn_vars;            /* 1 */
    int learn_prior_delay;     /* 1 */
    double merge_vars_thr;     /* 0.5 */
    int L;                     /* number of mixture components */
    double probs[VAMPOMI_MAX_MIX];
    double vars[VAMPOMI_MAX_MIX];     /* as given on the command line (NOT yet multiplied by N) */
    unsigned long long seed;   /* Hutchinson probe / probit start */
    int redundant_passes;      /* 1 = also recompute A^T y and A x2 where the reference does (src/vamp.cpp:303,826);
                                  0 = reuse them (same results, 2 fewer matrix passes per iteration) */
    int fuse_passes;           /* 1 = matrix products whose inputs are known at the same time share ONE read of
                                  the marker block: the LMMSE and the Onsager solve advance in lock-step
                                  (vampomi_cg_solve_pair), A x1_hat rides on their first pass, A x2_hat / A Q^-1 u and the two
                                  A^T products after the solves are one pass each — 2 max(k1,k2) + 2 passes per iteration
                                  instead of 2 (k1+k2) + 6, same arithmetic per product. 0 = one product per pass, in the
                                  reference's order. 2 (default) = fused, and additionally the products of the solves' SOLUTIONS are
                                  not computed by passes of their own but kept by the solves: A x2_hat and A Q^-1 u advance
                                  by alpha * (A p) next to the solutions (vampomi_cg_solve_pair track_ax_vec), A^T A of
                                  both follows from the solves' residuals — 2 max(k1,k2) passes per iteration; the values
                                  differ from separately computed products by recurrence rounding only (~1e-15 relative).
                                  3 = recycled, and every CG iteration reads the marker block ONCE instead of twice: the solves
                                  keep q = A p as a vector of its own and one fused pass delivers A^T q (= A^T A p) and A A^T q
                                  (what the recurrence of q needs), each column staying on chip between its two uses
                                  (vampomi_aat_multi_dev) — max(k1,k2) + 1 passes per iteration; contexts that cannot run the
                                  fused pass (FP32 storage, N > 40960) silently keep the two-pass iterations.
                                  Ignored (0) when redundant_passes = 1. */
    int probes;                /* Hutchinson probes per iteration (SURVEY.md §8 f2): 1 = the reference's single +-1/sqrt(Mt) probe
                                  (src/vamp.cpp:295-296); P > 1 averages u^T Q^-1 u (alpha2) and u^T A^T A Q^-1 u (noise precision) over P
                                  independent probes — P-1 more Onsager solves per iteration, off the reference's parity (its runs
                                  differ from each other by ~10 % because of this one-probe estimate, SURVEY.md fact 3). 0 reads as 1. */
} vampomi_solver_config;

typedef struct vampomi_iter_result {
    int it;                    /* iteration number just completed (1-based) */
    int n_params, n_metrics;   /* linear: 5 / 6, probit: 8 / 12 — the columns of _params.csv / _metrics.csv */
    double params[8];
    double metrics[12];
    double nmse;               /* sqrt(|x1_prev - x1|^2 / |x1_prev|^2), src/vamp.cpp:413 */
    double gam1_next;          /* gam1 the next iteration will use */
    int cg_iters_lmmse;        /* k1 */
    int cg_iters_onsager;      /* k2 */
    int L;                     /* mixture components after this iteration's prior update */
    double probs[VAMPOMI_MAX_MIX];
    double vars[VAMPOMI_MAX_MIX];     /* internal (x N) variances */
    long long matrix_passes;   /* full passes over the marker block this iteration */
    double true_gam1, true_gam2;      /* diagnostics printed by the reference (src/vamp.cpp:270,359) */
} vampomi_iter_result;

typedef struct vampomi_solver vampomi_solver;

void vampomi_solver_default_config(vampomi_solver_config* cfg);

/* `ctx` must hold the matrix block with statistics computed. y_N: phenotype as the reference's data::get_phen()
 * returns it (already scaled for the linear model). true_signal_M / x1hat_init_M may be NULL (zeros). */
int vampomi_solver_create(vampomi_ctx* ctx, const vampomi_solver_config* cfg, const double* y_N,
                          const double* true_signal_M, const double* x1hat_init_M, vampomi_solver** out);
/* One VAMP iteration. If x1_scaled_M / r1_scaled_M are non-NULL they receive x1_hat/sqrt(N) and r1/sqrt(N) — the
 * content of _it_{k}.bin and _r1_it_{k}.bin (src/vamp.cpp:235-249) — for this shard. */
/* Covariates (src/data.cpp:159-227, src/vamp_probit.cpp:490-617, call sites src/vamp.cpp:155-169 and src/vamp_probit.cpp:78-95,
 * 213-232): Z = the standardised N x C matrix (row-major, e.g. from vampomi_host_read_covariates). Must be called before the first
 * step; iteration 1 then fits the effects by the reference's Newton-Raphson and removes them (linear: from y; probit: as the offset
 * m_cov of the z-channel denoiser, device vector VAMPOMI_V_MCOV). get_cov_eff returns the fitted effects. */
int vampomi_solver_set_covariates(vampomi_solver* s, int C, const double* Z_NxC);
int vampomi_solver_get_cov_eff(vampomi_solver* s, int C, double* out_C);
/* Checkpoint / resume (SURVEY.md §8 f2; the reference's --estimate-file restart is dead code, src/vamp.cpp:71-79): save_state
 * writes everything the next iteration depends on — iteration number, gam1, gamw, the prior, the covariate effects and the vectors
 * r1, x1_hat, x2_hat (and the probit p1, tau1, alpha1) — into ONE file that all ranks share (every rank writes its marker slice at
 * its offset; rank 0 the header; every rank ends, after its data are on disk, with a completion record of the marker block it wrote);
 * load_state on a freshly created solver of the same problem — on any number of GPUs — restores it, so that the following
 * iterations equal those of an uninterrupted run (to rounding of two products that are recomputed instead of recycled). A file
 * whose completion records do not tile all Mt markers at the header's iteration (a writer died) is refused with VAMPOMI_ERR_IO
 * and leaves the solver as it was. */
int vampomi_solver_save_state(vampomi_solver* s, const char* path);
int vampomi_solver_load_state(vampomi_solver* s, const char* path);
int vampomi_solver_step(vampomi_solver* s, vampomi_iter_result* res, double* x1_scaled_M, double* r1_scaled_M);
int vampomi_solver_destroy(vampomi_solver* s);

/* ---- host-only pieces of the reference's driver, exported so that they can be checked without a GPU -------------- */
/* One CSV row exactly as write_ofile_csv formats it (src/utilities.cpp:366-385): "%5d" then ", %20.15f" per value and
 * a newline; returns the row length (the reference places the row at byte offset it * length) or -1 if it does not fit. */
int vampomi_host_csv_row(unsigned it, const double* values, int n, char* buf, int buflen);
/* data::read_phen (src/data.cpp:58-110): third whitespace token per line, scaled by sqrt((n-1)/sum((y-mean)^2)) when
 * `standardize`, never centred. Writes up to `cap` values, returns the number of rows, -1 if the file cannot be opened,
 * -2 on an NA value ("NAN in data!"). */
long long vampomi_host_read_phen(const char* path, int standardize, double* out, long long cap);
/* data::read_covariates (src/data.cpp:159-227): header line skipped, two ids skipped, C values per row, every covariate standardised
 * with its population sd (constant -> 0). Writes N*C values row-major; returns that count, -1 on a malformed file / row count != N. */
long long vampomi_host_read_covariates(const char* path, int C, int N, double* Z_NxC);
/* vamp::Newton_method_cov (src/vamp_probit.cpp:525-617): eta_inout holds the start on entry and the fitted effects on return. */
int vampomi_host_newton_cov(const double* y_N, const double* gg_N, const double* Z_NxC, int N, int C, double* eta_inout_C);
/* linear_reg1d_pvals (src/utilities.cpp:269-282) with boost's Student-t complement restated by a continued fraction. A variance that
 * rounds to <= 0 gives 1 and |r| > 1 is clamped: no NaN from sums without NaN. */
double vampomi_host_linear_reg1d_pvals(double sumx, double sumsqx, double sumxy, double sumy, double sumsqy, int n);
/* The per-marker tail of data::pvals_loo (src/data.cpp:400-414) for M markers at once, on `threads` host threads (0 = all, at most
 * 32): x1_M = x1_hat * sqrt(N), sums_3M = what vampomi_loo_sums returns, sum_w / sumsq_w = sum and sum of squares of y_mod. */
void vampomi_host_loo_pvals(const double* x1_M, const double* sums_3M, double sum_w, double sumsq_w, int N, long long M, double* pvals_M, int threads);
/* The same with the columns vampomi_constant_columns reports (const_M[j] != 0), which get p = 1 exactly; const_M = NULL is
 * vampomi_host_loo_pvals. */
void vampomi_host_loo_pvals_flagged(const double* x1_M, const double* sums_3M, double sum_w, double sumsq_w, int N, long long M,
                                    const unsigned char* const_M, double* pvals_M, int threads);
/* The counter-hash stand-ins for std::random_device (oracle patches P2/P3): probe sign (+1/-1) and probit start p1. */
double vampomi_host_probe_sign(unsigned long long seed, int it, unsigned long long global_marker);
void vampomi_host_probit_p1(unsigned long long seed, int N, double* out);
/* vamp::updatePrior's component merge (src/vamp.cpp:627-642), in place; returns the new number of components. */
int vampomi_host_merge_components(double* probs, double* vars, int L, double thr);

#ifdef __cplusplus
}
#endif
#endif /* VAMPOMI_HOST_H */
