#include "vamp.h"
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <fcntl.h>
#include <unistd.h>
#include <iostream>
#include "cov.h"
#include "io.h"
#include "../rng.h"

namespace vampomi_host {

namespace {
double wall_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
constexpr double kGammaMin = 1e-11, kGammaMax = 1e11;      // src/vamp.hpp:33-34
constexpr double kRecycleMaxRatio = 1e5;                   // gam2/tau above which recycled products are recomputed (eps * 1e5 = 2e-11)
constexpr int kRecycleRefresh = 16;                        // ... and every this many VAMP iterations regardless
inline double clampg(double g) { return std::min(std::max(g, kGammaMin), kGammaMax); }
}  // namespace

#define VH(call)                          \
    do {                                  \
        int rc__ = (call);                \
        if (rc__ != VAMPOMI_OK) return rc__; \
    } while (0)

void merge_components(std::vector<double>& probs, std::vector<double>& vars, double thr) {
    for (size_t j = 0; j < vars.size(); j++) {
        for (size_t k = j + 1; k < vars.size(); k++) {
            double denom = vars[j] != 0 ? std::min(vars[j], vars[k]) : 1e-7;
            if (std::fabs(vars[j] - vars[k]) / denom < thr) {
                double s = probs[j] + probs[k];
                vars.erase(vars.begin() + k);
                probs.erase(probs.begin() + k);
                probs[j] = s;
                k--;
            }
        }
    }
}

Vamp::Vamp(vampomi_ctx* ctx, const vampomi_solver_config& cfg) : ctx_(ctx), cfg_(cfg) {
    gam1_ = cfg.gam1;
    gamw_ = cfg.gamw;
}

int Vamp::init(const double* y, const double* true_signal, const double* x1hat_init) {
    VH(vampomi_dims(ctx_, &N_, &Mt_, &nranks_, &rank_));
    VH(vampomi_shard(ctx_, &M_, &S_));
    if (cfg_.L < 1 || cfg_.L > VAMPOMI_MAX_MIX) return VAMPOMI_ERR_ARG;
    probs_.assign(cfg_.probs, cfg_.probs + cfg_.L);
    vars_.assign(cfg_.vars, cfg_.vars + cfg_.L);
    for (double& v : vars_) v *= N_;                                            // src/vamp.cpp:87-88
    y_host_.assign(y, y + N_);
    zbuf_.assign((size_t)N_, 0.0);
    VH(vampomi_vec_set(ctx_, VAMPOMI_V_Y, y));
    std::vector<double> tmp((size_t)M_, 0.0);
    if (true_signal) VH(vampomi_vec_set(ctx_, VAMPOMI_V_TRUE, true_signal));
    else VH(vampomi_vec_set(ctx_, VAMPOMI_V_TRUE, tmp.data()));
    if (x1hat_init) {                                                           // src/vamp.cpp:71-72,78-79 (with patch P1)
        const double sq = std::sqrt((double)N_);
        for (long long i = 0; i < M_; i++) tmp[i] = x1hat_init[i] / sq;
    }
    VH(vampomi_vec_set(ctx_, VAMPOMI_V_X1, tmp.data()));
    VH(vampomi_vec_set(ctx_, VAMPOMI_V_R1, tmp.data()));
    VH(vampomi_vec_fill(ctx_, VAMPOMI_V_X2, 0.0));
    VH(vampomi_vec_fill(ctx_, VAMPOMI_V_R2, 0.0));
    // schedule "onepass" (fuse_passes >= 3): the recycled schedule with CG iterations that read the marker block once
    // (fused A^T q / A A^T q pass); contexts that cannot run it (FP32 storage, N > 40960) keep the two-pass iterations
    if (cfg_.fuse_passes >= 3 && cfg_.redundant_passes == 0) VH(vampomi_set_tuning(ctx_, "cg_onepass", 1));
    else if (cfg_.fuse_passes >= 0) VH(vampomi_set_tuning(ctx_, "cg_onepass", 0));
    it_ = 0;
    aty_ready_ = false;
    ata_x2_ready_ = false;
    if (cfg_.model == 1) {                                                      // src/vamp_probit.cpp:35-61
        tau1_ = gam1_;
        std::vector<double> p1 = probit_p1(cfg_.seed, N_);
        VH(vampomi_vec_set(ctx_, VAMPOMI_V_P1, p1.data()));
        VH(vampomi_vec_fill(ctx_, VAMPOMI_V_R1, 0.0));
        VH(vampomi_vec_fill(ctx_, VAMPOMI_V_R2, 0.0));
        alpha1_ = 0;
        if (cfg_.redundant_passes) {                                            // true_g = A * true_signal_scaled (:46), unused
            VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_USER_M0, std::sqrt((double)N_), VAMPOMI_V_TRUE, 0.0, VAMPOMI_V_TRUE, 1.0));
            VH(vampomi_ax_dev(ctx_, VAMPOMI_V_USER_M0, VAMPOMI_V_USER_N0));
        }
    }
    return VAMPOMI_OK;
}

int Vamp::set_covariates(int C, const double* Z) {
    if (C < 0 || (C > 0 && !Z) || it_ != 0) return VAMPOMI_ERR_ARG;
    C_ = C;
    Z_.assign(Z, Z + (size_t)C * (size_t)N_);
    cov_eff_.assign((size_t)C, 0.0);
    return VAMPOMI_OK;
}

// iteration 1 of both loops (src/vamp.cpp:155-169, src/vamp_probit.cpp:78-93): probit regression of y on the covariates with the
// genetic predictor gg = z1_hat = 0, then the reference's print-out of the effects
int Vamp::fit_covariates() {
    const double t0 = wall_s();
    cov_eff_ = newton_method_cov(y_host_, std::vector<double>((size_t)N_, 0.0), Z_, N_, C_, cov_eff_, verbose, verbosity);
    if (verbose) {
        for (int i0 = 0; i0 < C_; i0++) {
            std::cout << "cov_eff[" << i0 << "] = " << cov_eff_[i0] << ", ";
            if (i0 % 4 == 3) std::cout << std::endl;
        }
        std::cout << std::endl;
        if (cfg_.model == 1) std::cout << "Computing covariate effects took " << wall_s() - t0 << " seconds." << std::endl;   // src/vamp_probit.cpp:94
    }
    return VAMPOMI_OK;
}

int Vamp::apply_covariates() {
    std::vector<double> v((size_t)N_);
    for (int i = 0; i < N_; i++) {
        double s = 0;
        for (int j = 0; j < C_; j++) s += Z_[(size_t)i * C_ + j] * cov_eff_[j];
        // linear: y -= Z cov_eff (src/vamp.cpp:166-168) changes the loop's LOCAL copy of the phenotype only: it feeds A^T y (:303),
        // while updateNoisePrec (:506) and err_measures (:817) fetch the unadjusted phenotype from the dataset again — so the
        // adjusted vector gets a device vector of its own (VAMPOMI_V_MCOV, otherwise unused by the linear model) and Y stays.
        // probit: m_cov of g1_bin_class / g1d_bin_class (src/vamp_probit.cpp:214-232)
        v[i] = cfg_.model == 0 ? y_host_[i] - s : s;
    }
    VH(vampomi_vec_set(ctx_, VAMPOMI_V_MCOV, v.data()));
    aty_ready_ = false;
    return VAMPOMI_OK;
}

// ---- checkpoint file: 4096-byte header, then r1[Mt], x1_hat[Mt], x2_hat[Mt], p1[N] as FP64 -----------------------------------
namespace {
struct CkptHeader {
    char magic[8];
    int model, it, N, L, C, nranks;
    long long Mt;
    double gam1, gamw, alpha1, tau1, gam2, eta1, eta2, alpha2;
    double probs[VAMPOMI_MAX_MIX], vars[VAMPOMI_MAX_MIX];
    double cov_eff[64];
};
// A checkpoint is written by all ranks into one file with no ordering between them, so a run that dies while writing leaves a file
// that can look whole (holes read as zeros). Every rank therefore ends with a record of the marker block it wrote, after its data are
// on disk; a checkpoint is complete when the records of all h.nranks writers carry the header's iteration and tile [0, Mt).
struct CkptShard {
    long long it, S, M;
};
constexpr long long kCkptShards = 2048, kCkptMaxRanks = 64;
static_assert(sizeof(CkptHeader) <= kCkptShards && kCkptShards + kCkptMaxRanks * sizeof(CkptShard) <= 4096, "checkpoint header");
constexpr long long kCkptData = 4096;
bool pwrite_all(int fd, const void* buf, size_t n, long long off) {
    size_t done = 0;
    while (done < n) {
        ssize_t r = pwrite(fd, (const char*)buf + done, n - done, (off_t)(off + (long long)done));
        if (r <= 0) return false;
        done += (size_t)r;
    }
    return true;
}
bool pread_all(int fd, void* buf, size_t n, long long off) {
    size_t done = 0;
    while (done < n) {
        ssize_t r = pread(fd, (char*)buf + done, n - done, (off_t)(off + (long long)done));
        if (r <= 0) return false;
        done += (size_t)r;
    }
    return true;
}
}  // namespace

int Vamp::save_state(const char* path) {
    if (!path || it_ < 1 || C_ > 64 || nranks_ > kCkptMaxRanks) return VAMPOMI_ERR_ARG;
    int fd = ::open(path, O_WRONLY | O_CREAT, 0644);
    if (fd < 0) return VAMPOMI_ERR_IO;
    CkptShard rec = {0, 0, 0};
    bool ok = pwrite_all(fd, &rec, sizeof(rec), kCkptShards + rank_ * (long long)sizeof(rec));   // a file of this name may be there already
    std::vector<double> buf((size_t)std::max<long long>(M_, N_));
    const int vecs[3] = {VAMPOMI_V_R1, VAMPOMI_V_X1, VAMPOMI_V_X2};
    for (int k = 0; k < 3 && ok; k++) {
        ok = vampomi_vec_get(ctx_, vecs[k], buf.data()) == VAMPOMI_OK &&
             pwrite_all(fd, buf.data(), (size_t)M_ * sizeof(double), kCkptData + ((long long)k * Mt_ + S_) * 8);
    }
    if (ok && rank_ == 0) {
        CkptHeader h;
        std::memset(&h, 0, sizeof(h));
        std::memcpy(h.magic, "VAMPCKP2", 8);
        h.model = cfg_.model; h.it = it_; h.N = N_; h.nranks = nranks_; h.L = (int)probs_.size(); h.C = C_; h.Mt = Mt_;
        h.gam1 = gam1_; h.gamw = gamw_; h.alpha1 = alpha1_; h.tau1 = tau1_; h.gam2 = gam2_; h.eta1 = eta1_; h.eta2 = eta2_; h.alpha2 = alpha2_;
        for (int i = 0; i < h.L; i++) { h.probs[i] = probs_[i]; h.vars[i] = vars_[i]; }
        for (int j = 0; j < C_; j++) h.cov_eff[j] = cov_eff_[j];
        ok = pwrite_all(fd, &h, sizeof(h), 0);
        if (ok && cfg_.model == 1)
            ok = vampomi_vec_get(ctx_, VAMPOMI_V_P1, buf.data()) == VAMPOMI_OK &&
                 pwrite_all(fd, buf.data(), (size_t)N_ * sizeof(double), kCkptData + 3LL * Mt_ * 8);
    }
    if (ok) {
        rec = {it_, S_, M_};
        ok = ::fdatasync(fd) == 0 && pwrite_all(fd, &rec, sizeof(rec), kCkptShards + rank_ * (long long)sizeof(rec)) && ::fdatasync(fd) == 0;
    }
    ::close(fd);
    return ok ? VAMPOMI_OK : VAMPOMI_ERR_IO;
}

int Vamp::load_state(const char* path) {
    if (!path || it_ != 0) return VAMPOMI_ERR_ARG;            // on a freshly initialised solver only
    int fd = ::open(path, O_RDONLY);
    if (fd < 0) return VAMPOMI_ERR_IO;
    CkptHeader h;
    bool ok = pread_all(fd, &h, sizeof(h), 0) && !std::memcmp(h.magic, "VAMPCKP2", 8);
    if (ok && (h.model != cfg_.model || h.N != N_ || h.Mt != Mt_ || h.L < 1 || h.L > VAMPOMI_MAX_MIX || h.C != C_)) { ::close(fd); return VAMPOMI_ERR_ARG; }
    if (ok) {                                                 // every writer finished: their marker blocks tile [0, Mt) (any order of ranks)
        CkptShard recs[kCkptMaxRanks];
        ok = h.nranks >= 1 && h.nranks <= kCkptMaxRanks && pread_all(fd, recs, (size_t)h.nranks * sizeof(CkptShard), kCkptShards);
        long long next = 0;
        for (int found = 1; ok && found && next < Mt_;) {
            found = 0;
            for (int k = 0; k < h.nranks; k++)
                if (recs[k].it == h.it && recs[k].S == next && recs[k].M > 0) { next += recs[k].M; found = 1; break; }
        }
        ok = ok && next == Mt_;
    }
    std::vector<double> buf((size_t)std::max<long long>(M_, N_));
    const int vecs[3] = {VAMPOMI_V_R1, VAMPOMI_V_X1, VAMPOMI_V_X2};
    for (int k = 0; k < 3 && ok; k++)
        ok = pread_all(fd, buf.data(), (size_t)M_ * sizeof(double), kCkptData + ((long long)k * Mt_ + S_) * 8) &&
             vampomi_vec_set(ctx_, vecs[k], buf.data()) == VAMPOMI_OK;
    if (ok && cfg_.model == 1)
        ok = pread_all(fd, buf.data(), (size_t)N_ * sizeof(double), kCkptData + 3LL * Mt_ * 8) && vampomi_vec_set(ctx_, VAMPOMI_V_P1, buf.data()) == VAMPOMI_OK;
    ::close(fd);
    if (!ok) return VAMPOMI_ERR_IO;
    it_ = h.it;
    gam1_ = h.gam1; gamw_ = h.gamw; alpha1_ = h.alpha1; tau1_ = h.tau1; gam2_ = h.gam2; eta1_ = h.eta1; eta2_ = h.eta2; alpha2_ = h.alpha2;
    probs_.assign(h.probs, h.probs + h.L);
    vars_.assign(h.vars, h.vars + h.L);
    if (C_ > 0) {
        cov_eff_.assign(h.cov_eff, h.cov_eff + C_);
        VH(apply_covariates());
    }
    // what an uninterrupted run would carry over by recycling is recomputed: A^T y at its next use, A^T A x2_hat inside the next
    // solve, and Z2 = A x2_hat (the tracked product of the warm system must hold A * start on entry)
    aty_ready_ = false;
    ata_x2_ready_ = false;
    if (cfg_.model == 0) VH(vampomi_ax_dev(ctx_, VAMPOMI_V_X2, VAMPOMI_V_Z2));
    return VAMPOMI_OK;
}

void Vamp::fill_prior(vampomi_iter_result* res) const {
    res->L = (int)probs_.size();
    for (int i = 0; i < VAMPOMI_MAX_MIX; i++) {
        res->probs[i] = i < res->L ? probs_[i] : 0.0;
        res->vars[i] = i < res->L ? vars_[i] : 0.0;
    }
}

// x1_hat/sqrt(N) and r1/sqrt(N) as the reference stores them at this point of the iteration (src/vamp.cpp:237-249). The
// values are snapshotted and copied in stream order without a host round trip; step() collects them before it returns.
int Vamp::dump(double* x1_scaled, double* r1_scaled) {
    const double sq = std::sqrt((double)N_);
    if (x1_scaled) { VH(vampomi_dump_begin(ctx_, 0, VAMPOMI_V_X1, sq)); pending_x1_ = x1_scaled; }   // src/vamp.cpp:237-239
    if (r1_scaled) { VH(vampomi_dump_begin(ctx_, 1, VAMPOMI_V_R1, sq)); pending_r1_ = r1_scaled; }   // :246-249
    return VAMPOMI_OK;
}

int Vamp::collect_dump() {
    int rc = VAMPOMI_OK;
    if (pending_x1_) { int r = vampomi_dump_wait(ctx_, 0, pending_x1_); if (r != VAMPOMI_OK) rc = r; pending_x1_ = nullptr; }
    if (pending_r1_) { int r = vampomi_dump_wait(ctx_, 1, pending_r1_); if (r != VAMPOMI_OK) rc = r; pending_r1_ = nullptr; }
    return rc;
}

// src/vamp.cpp:531-643 — the per-marker sums come from the device, everything else is L-length host arithmetic
int Vamp::update_prior() {
    double lambda = 1 - probs_[0];
    std::vector<double> omegas = probs_;
    for (size_t j = 1; j < omegas.size(); j++) omegas[j] /= lambda;
    int em_it = 0;
    for (em_it = 0; em_it < cfg_.EM_max_iter; em_it++) {
        const int L = (int)probs_.size();
        std::vector<double> probs_prev = probs_, vars_prev = vars_;
        std::vector<double> sums((size_t)(2 * L - 1), 0.0);
        VH(vampomi_em_sums(ctx_, gam1_, lambda, omegas.data(), vars_.data(), L, sums.data()));
        const double lambda_total = sums[0];
        lambda = lambda_total / (double)Mt_;                                    // :579
        const double sum_of_pin = lambda_total;                                 // :587
        for (int j = 0; j < L - 1; j++) {
            const double res_total = sums[1 + j], res_gammas_total = sums[L + j];
            if (cfg_.learn_vars == 1) vars_[j + 1] = res_gammas_total / res_total;   // :598-599
            omegas[j + 1] = res_total / sum_of_pin;
            probs_[j + 1] = lambda * omegas[j + 1];
        }
        probs_[0] = 1 - lambda;
        double dp = 0, np = 0, dv = 0, nv = 0;
        for (int j = 0; j < L; j++) {
            dp += (probs_[j] - probs_prev[j]) * (probs_[j] - probs_prev[j]);
            np += probs_[j] * probs_[j];
            dv += (vars_[j] - vars_prev[j]) * (vars_[j] - vars_prev[j]);
            nv += vars_[j] * vars_[j];
        }
        const double dist_probs = std::sqrt(dp / np), dist_vars = std::sqrt(dv / nv);
        if (verbose && verbosity == 1)
            std::cout << "it = " << em_it << ": dist_probs = " << dist_probs << " & dist_vars = " << dist_vars << std::endl;
        if (dist_probs < cfg_.EM_err_thr && dist_vars < cfg_.EM_err_thr) break;
    }
    if (verbose && verbosity == 1)
        std::cout << "Final number of prior EM iterations = " << std::min(em_it + 1, cfg_.EM_max_iter) << " / "
                  << cfg_.EM_max_iter << std::endl;
    merge_components(probs_, vars_, cfg_.merge_vars_thr);
    return VAMPOMI_OK;
}

int Vamp::step(vampomi_iter_result* res, double* x1_scaled, double* r1_scaled) {
    if (!res) return VAMPOMI_ERR_ARG;
    if (Mt_ == 0) return VAMPOMI_ERR_STATE;
    long long c0[4], c1[4];
    VH(vampomi_counters(ctx_, c0, 0));
    std::memset(res, 0, sizeof(*res));
    it_++;
    res->it = it_;
    int rc = cfg_.model == 0 ? step_linear(res, x1_scaled, r1_scaled) : step_probit(res, x1_scaled, r1_scaled);
    const int rc_dump = collect_dump();                                          // also on failure: leaves no read-out pending
    if (rc != VAMPOMI_OK) return rc;
    if (rc_dump != VAMPOMI_OK) return rc_dump;
    VH(vampomi_counters(ctx_, c1, 0));
    res->matrix_passes = c1[1] - c0[1];
    res->gam1_next = gam1_;
    fill_prior(res);
    return VAMPOMI_OK;
}

// One iteration of src/vamp.cpp:148-428.
int Vamp::step_linear(vampomi_iter_result* res, double* x1_scaled, double* r1_scaled) {
    const int it = it_;
    const double sqrtN = std::sqrt((double)N_), rho = cfg_.rho;
    {                                                                           // covariate effects, :153-173
        const double t_cov0 = wall_s();
        if (it == 1 && C_ > 0) {
            VH(fit_covariates());
            VH(apply_covariates());
        }
        if (verbose) std::cout << "time for covariates effects update = " << wall_s() - t_cov0 << " seconds." << std::endl;   // :173
    }
    if (verbose) std::cout << "->DENOISING" << std::endl;
    if (it > cfg_.learn_prior_delay) VH(update_prior());                        // :186-187
    if (verbose) {
        std::cout << "Prior variances = ";
        for (double v : vars_) std::cout << v / (double)N_ << ' ';
        std::cout << std::endl << "Prior probabilities = ";
        for (double p : probs_) std::cout << p << ' ';
        std::cout << std::endl;
    }
    // fused schedule (cfg.fuse_passes): matrix passes whose inputs are known at the same time share ONE read of the block —
    //   A x1_hat rides on the first A p pass of the solves, the LMMSE and the Onsager solve advance in lock-step,
    //   A x2_hat and A Q^-1 u are one pass, A^T (A Q^-1 u) and A^T (A x2_hat) (next iteration's warm-start residual) another —
    // 2 max(k1,k2) + 2 passes per iteration instead of 2 (k1+k2) + 6; every product keeps its own arithmetic.
    const bool fuse = cfg_.fuse_passes != 0 && cfg_.redundant_passes == 0;
    const bool recycle = fuse && cfg_.fuse_passes >= 2;
    double tau_solved = gamw_;
    double sum_d = 0;
    VH(vampomi_denoise(ctx_, gam1_, probs_.data(), vars_.data(), (int)probs_.size(), it > 1, rho, &sum_d));   // :203-219
    alpha1_ = sum_d / (double)Mt_;                                              // :221-223
    eta1_ = gam1_ / alpha1_;
    if (!fuse) VH(vampomi_ax_dev(ctx_, VAMPOMI_V_X1, VAMPOMI_V_Z1));            // :232
    VH(dump(x1_scaled, r1_scaled));                                             // :235-249
    gam2_ = clampg(eta1_ - gam1_);                                              // :255-256
    VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_R2, eta1_, VAMPOMI_V_X1, -gam1_, VAMPOMI_V_R1, gam2_));   // :259-261

    // err_measures(1) (:760-852), true-gam2 diagnostic (:264-270) and the NMSE sums (:409-413) in one reduction launch;
    // needs z1 = A x1_hat, so in the fused schedule it runs after the first pass of the solves
    const double gam1_used = gam1_;
    auto measures1 = [&]() -> int {
        const int kind[10] = {VAMPOMI_DOT, VAMPOMI_DOT, VAMPOMI_DOT, VAMPOMI_DIFF2, VAMPOMI_DOT, VAMPOMI_DOT, VAMPOMI_DOT,
                              VAMPOMI_SQDEV, VAMPOMI_DIFF2, VAMPOMI_DOT};
        const int a[10] = {VAMPOMI_V_X1, VAMPOMI_V_X1, VAMPOMI_V_TRUE, VAMPOMI_V_Y, VAMPOMI_V_Y, VAMPOMI_V_Z1, VAMPOMI_V_Z1,
                           VAMPOMI_V_R2, VAMPOMI_V_X1_PREV, VAMPOMI_V_X1_PREV};
        const int b[10] = {VAMPOMI_V_TRUE, VAMPOMI_V_X1, VAMPOMI_V_TRUE, VAMPOMI_V_Z1, VAMPOMI_V_Y, VAMPOMI_V_Y, VAMPOMI_V_Z1,
                           VAMPOMI_V_TRUE, VAMPOMI_V_X1, VAMPOMI_V_X1_PREV};
        double scale[10] = {1, 1, 1, 1, 1, 1, 1, sqrtN, 1, 1}, d[10];
        VH(vampomi_dots(ctx_, 10, kind, a, b, scale, d));
        const double corr = d[0] / std::sqrt(d[1] * d[2]);                      // :767
        const double l2_pred_err = std::sqrt(d[3] / d[4]);                      // :832
        const double R2 = 1 - l2_pred_err * l2_pred_err;
        const double corr_y = d[5] / std::sqrt(d[6] * d[4]);                    // :835
        res->metrics[1] = corr; res->metrics[0] = R2; res->metrics[4] = corr_y * corr_y;
        res->true_gam2 = (double)Mt_ / d[7];
        res->nmse = std::sqrt(d[8] / d[9]);
        if (verbose) {
            std::cout << "Corr(x1_hat, x0) = " << corr << std::endl;
            std::cout << "Corr(y_hat, y)^2 = " << corr_y * corr_y << std::endl << "R2 = " << R2 << std::endl
                      << "L2(y_hat, y) = " << l2_pred_err << std::endl;
            std::cout << "alpha1 = " << alpha1_ << std::endl << "gam1 = " << gam1_used << std::endl << "gam2 = " << gam2_ << std::endl
                      << "true gam2 = " << res->true_gam2 << std::endl << "______________________" << std::endl << "->LMMSE" << std::endl;
        }
        return VAMPOMI_OK;
    };
    res->params[0] = alpha1_; res->params[1] = gam1_;                           // :275-276
    if (!fuse) VH(measures1());

    const double t_lmmse0 = wall_s();                                           // start_lmmse_step, :288
    VH(vampomi_draw_probe(ctx_, cfg_.seed, it));                                // :295-296
    if (cfg_.redundant_passes || !aty_ready_) {                                 // v = gamw * A^T y + gam2 * r2, :303-306
        VH(vampomi_atx_dev(ctx_, C_ > 0 ? VAMPOMI_V_MCOV : VAMPOMI_V_Y, VAMPOMI_V_ATY));
        aty_ready_ = true;
    }
    VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_V, gamw_, VAMPOMI_V_ATY, gam2_, VAMPOMI_V_R2, 1.0));
    int k1 = 0, k2 = 0;
    double rel = 0, vmu = 0;
    // the reference's per-phase timing lines (src/vamp.cpp:316,333,399): host wall clock around the solves, which end with a
    // synchronising read-back. In the lock-step schedules both solves run inside ONE call, reported as "CG took"; the Onsager
    // solve then has no time of its own ("onsager took 0").
    const double t_cg0 = wall_s();
    double t_cg1 = t_cg0, t_ons1 = t_cg0;
    if (!fuse) {
        VH(vampomi_cg_solve(ctx_, VAMPOMI_V_V, VAMPOMI_V_X2, it > 1, gamw_, gam2_, cfg_.CG_err_tol, cfg_.CG_max_iter, 0, &k1, &rel,
                            nullptr));                                          // :308-311
        t_cg1 = wall_s();
        VH(vampomi_cg_solve(ctx_, VAMPOMI_V_BERN, VAMPOMI_V_QINV_BERN, 0, gamw_, gam2_, cfg_.CG_err_tol, cfg_.CG_max_iter, 1, &k2,
                            &rel, &vmu));                                       // g2d_onsager, :494-501
        t_ons1 = wall_s();
    } else {
        const int rhs[2] = {VAMPOMI_V_V, VAMPOMI_V_BERN}, sol[2] = {VAMPOMI_V_X2, VAMPOMI_V_QINV_BERN};
        const int warm[2] = {it > 1 ? 1 : 0, 0}, ata[2] = {ata_x2_ready_ ? VAMPOMI_V_ATA_X2 : -1, -1}, ons[2] = {0, 1};
        int its[2] = {0, 0};
        double rels[2], vmus[2];
        // recycled schedule: the solves also keep Z2 = A x2_hat (it holds A x2_hat of the previous iteration, the warm start)
        // and USER_N0 = A Q^-1 u up to date from their own A p products
        const int track[2] = {recycle ? VAMPOMI_V_Z2 : -1, recycle ? VAMPOMI_V_USER_N0 : -1};
        VH(vampomi_cg_solve_pair(ctx_, rhs, sol, warm, ata, gamw_, gam2_, cfg_.CG_err_tol, cfg_.CG_max_iter, ons, VAMPOMI_V_X1,
                                 VAMPOMI_V_Z1, track, its, rels, vmus));
        tau_solved = gamw_;
        k1 = its[0]; k2 = its[1]; vmu = vmus[1];
        t_cg1 = t_ons1 = wall_s();
        VH(measures1());
    }
    // further Hutchinson probes (cfg.probes > 1; not in the reference): one more Onsager solve each, from the same counter hash
    // with the probe index folded into the seed; u^T Q^-1 u and u^T A^T A Q^-1 u are averaged over the probes
    const int P = cfg_.probes > 1 ? cfg_.probes : 1;
    double trace_extra = 0;                                     // sum over the extra probes of <u, A^T A Q^-1 u>
    double trace_first = 0;
    bool ata_x2_recycled = false;
    if (P > 1) {
        // <u_1, A^T A Q^-1 u_1> of the first probe must be taken now: BERN / QINV_BERN and the CG work vectors are about to be
        // reused by the extra solves — and so must the recycled A^T A x2_hat, which lives in the LMMSE solve's residual
        if (recycle) {
            VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_ATA_X2, 1.0, VAMPOMI_V_V, -1.0, VAMPOMI_V_CG_R, 1.0));
            VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_ATA_X2, 1.0, VAMPOMI_V_ATA_X2, -gam2_, VAMPOMI_V_X2, tau_solved));
            ata_x2_recycled = true;
            VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_USER_M0, 1.0, VAMPOMI_V_BERN, -1.0, VAMPOMI_V_CG2_R, 1.0));
            VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_USER_M0, 1.0, VAMPOMI_V_USER_M0, -gam2_, VAMPOMI_V_QINV_BERN, tau_solved));
        } else {
            VH(vampomi_ax_dev(ctx_, VAMPOMI_V_QINV_BERN, VAMPOMI_V_USER_N0));
            VH(vampomi_atx_dev(ctx_, VAMPOMI_V_USER_N0, VAMPOMI_V_USER_M0));
        }
        const int kd[1] = {VAMPOMI_DOT}, ad[1] = {VAMPOMI_V_BERN}, bd[1] = {VAMPOMI_V_USER_M0};
        VH(vampomi_dots(ctx_, 1, kd, ad, bd, nullptr, &trace_first));
        for (int p = 1; p < P; p++) {
            VH(vampomi_draw_probe(ctx_, cfg_.seed + 0x9E3779B97F4A7C15ULL * (unsigned long long)p, it));
            int kp = 0;
            double relp = 0, vmup = 0;
            VH(vampomi_cg_solve(ctx_, VAMPOMI_V_BERN, VAMPOMI_V_QINV_BERN, 0, gamw_, gam2_, cfg_.CG_err_tol, cfg_.CG_max_iter, 1, &kp, &relp, &vmup));
            vmu += vmup;
            VH(vampomi_ax_dev(ctx_, VAMPOMI_V_QINV_BERN, VAMPOMI_V_USER_N0));
            VH(vampomi_atx_dev(ctx_, VAMPOMI_V_USER_N0, VAMPOMI_V_USER_M0));
            double tp = 0;
            VH(vampomi_dots(ctx_, 1, kd, ad, bd, nullptr, &tp));
            trace_extra += tp;
        }
        vmu /= P;
    }
    if (verbose)
        std::cout << "CG took " << t_cg1 - t_cg0 << " seconds." << std::endl                                  // :316
                  << "onsager took " << (P > 1 ? wall_s() - t_cg1 : t_ons1 - t_cg1) << " seconds." << std::endl;   // :333
    alpha2_ = gam2_ * vmu;
    res->cg_iters_lmmse = k1; res->cg_iters_onsager = k2;
    eta2_ = gam2_ / alpha2_;                                                    // :341
    const double gam1_prev = gam1_;
    gam1_ = clampg(eta2_ - gam2_);
    gam1_ = rho * gam1_ + (1 - rho) * gam1_prev;                                // :346
    VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_R1, eta2_, VAMPOMI_V_X2, -gam2_, VAMPOMI_V_R2, gam1_));   // :348-350

    // updateNoisePrec (:504-529) + err_measures(2) share A x2_hat; the reference computes it twice (:508, :826)
    // The recycled products are differences of the solves' own vectors: A^T A sol = (rhs - r - gam2 sol)/tau loses
    // ~eps*gam2/(tau*lambda) to cancellation, and Z2 = A x2_hat is advanced by recurrence from one VAMP iteration to the next.
    // So they are recomputed by explicit passes (the `fused` schedule's two passes) whenever gam2/tau is large enough for the
    // cancellation to matter at the 1e-9 contract, and every kRecycleRefresh iterations to cut the accumulated recurrence.
    const bool refresh_products = recycle && (gam2_ / tau_solved > kRecycleMaxRatio || it % kRecycleRefresh == 0);
    if (!fuse) {
        VH(vampomi_ax_dev(ctx_, VAMPOMI_V_X2, VAMPOMI_V_Z2));
        VH(vampomi_ax_dev(ctx_, VAMPOMI_V_QINV_BERN, VAMPOMI_V_USER_N0));       // :518
        VH(vampomi_atx_dev(ctx_, VAMPOMI_V_USER_N0, VAMPOMI_V_USER_M0));        // :519
        if (cfg_.redundant_passes) VH(vampomi_ax_dev(ctx_, VAMPOMI_V_X2, VAMPOMI_V_Z2));
    } else if (!recycle || refresh_products) {
        const int xin[2] = {VAMPOMI_V_X2, VAMPOMI_V_QINV_BERN}, xout[2] = {VAMPOMI_V_Z2, VAMPOMI_V_USER_N0};
        VH(vampomi_ax_multi_dev(ctx_, 2, xin, xout));
        const int pin[2] = {VAMPOMI_V_USER_N0, VAMPOMI_V_Z2}, pout[2] = {VAMPOMI_V_USER_M0, VAMPOMI_V_ATA_X2};
        VH(vampomi_atx_multi_dev(ctx_, 2, pin, pout));                          // A^T A x2_hat: the next iteration's :681-684
        ata_x2_ready_ = true;
    } else {
        // no pass at all: Z2 = A x2_hat and A Q^-1 u were kept by the solves; A^T A of both solutions follows from the solves'
        // own residuals, r = rhs - (tau A^T A + gam2 I) sol  =>  A^T A sol = (rhs - r - gam2 sol) / tau
        if (!ata_x2_recycled) {
            VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_ATA_X2, 1.0, VAMPOMI_V_V, -1.0, VAMPOMI_V_CG_R, 1.0));
            VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_ATA_X2, 1.0, VAMPOMI_V_ATA_X2, -gam2_, VAMPOMI_V_X2, tau_solved));
            VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_USER_M0, 1.0, VAMPOMI_V_BERN, -1.0, VAMPOMI_V_CG2_R, 1.0));
            VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_USER_M0, 1.0, VAMPOMI_V_USER_M0, -gam2_, VAMPOMI_V_QINV_BERN, tau_solved));
        }
        ata_x2_ready_ = true;
    }
    {
        const int kind[9] = {VAMPOMI_DIFF2, VAMPOMI_DOT, VAMPOMI_SQDEV, VAMPOMI_DOT, VAMPOMI_DOT, VAMPOMI_DOT, VAMPOMI_DOT,
                             VAMPOMI_DOT, VAMPOMI_DOT};
        const int a[9] = {VAMPOMI_V_Z2, VAMPOMI_V_BERN, VAMPOMI_V_R1, VAMPOMI_V_X2, VAMPOMI_V_X2, VAMPOMI_V_TRUE, VAMPOMI_V_Y,
                          VAMPOMI_V_Z2, VAMPOMI_V_Z2};
        const int b[9] = {VAMPOMI_V_Y, VAMPOMI_V_USER_M0, VAMPOMI_V_TRUE, VAMPOMI_V_TRUE, VAMPOMI_V_X2, VAMPOMI_V_TRUE, VAMPOMI_V_Y,
                          VAMPOMI_V_Y, VAMPOMI_V_Z2};
        double scale[9] = {1, 1, sqrtN, 1, 1, 1, 1, 1, 1}, d[9];
        VH(vampomi_dots(ctx_, 9, kind, a, b, scale, d));
        const double temp_norm2 = d[0];
        const double trace_corr = (P > 1 ? (trace_first + trace_extra) / P : d[1]) * (double)Mt_;   // :521
        if (verbose)
            std::cout << "l2_norm2(temp) / N = " << temp_norm2 / N_ << std::endl << "trace_correction / N = " << trace_corr / N_ << std::endl;
        gamw_ = (double)N_ / (temp_norm2 + trace_corr);                         // :528
        res->true_gam1 = (double)Mt_ / d[2];
        const double corr2 = d[3] / std::sqrt(d[4] * d[5]);
        const double l2_pred_err = std::sqrt(d[0] / d[6]);
        const double R2 = 1 - l2_pred_err * l2_pred_err;
        const double corr_y = d[7] / std::sqrt(d[8] * d[6]);
        res->metrics[3] = corr2; res->metrics[2] = R2; res->metrics[5] = corr_y * corr_y;
        if (verbose)
            std::cout << "Corr(x2_hat, x0)= " << corr2 << std::endl << "Corr(y_hat, y)^2 = " << corr_y * corr_y << std::endl
                      << "R2 = " << R2 << std::endl << "L2(y_hat, y) = " << l2_pred_err << std::endl;
    }
    res->params[2] = alpha2_; res->params[3] = gam2_; res->params[4] = gamw_;   // :368-370
    res->n_params = 5; res->n_metrics = 6;
    if (verbose)
        std::cout << "alpha2 = " << alpha2_ << std::endl << "gam2 = " << gam2_ << std::endl << "gam1 = " << gam1_ << std::endl
                  << "true gam1 = " << res->true_gam1 << std::endl << "gamw = " << gamw_ << std::endl
                  << "LMMSE step took " << wall_s() - t_lmmse0 << " seconds." << std::endl;                   // :399
    return VAMPOMI_OK;
}

// One iteration of src/vamp_probit.cpp:68-463.
int Vamp::step_probit(vampomi_iter_result* res, double* x1_scaled, double* r1_scaled) {
    const int it = it_;
    const double sqrtN = std::sqrt((double)N_), rho = cfg_.rho;
    if (verbose) std::cout << "...calculating covariate effects" << std::endl;
    if (it == 1 && C_ > 0) {                                                    // :78-95
        VH(fit_covariates());
        VH(apply_covariates());
    }
    if (verbose) std::cout << "->DENOISING" << std::endl;
    const double alpha1_prev = alpha1_;
    double sum_d = 0;
    // g1 / g1d with the CURRENT prior, no damping yet (:112-130)
    VH(vampomi_denoise(ctx_, gam1_, probs_.data(), vars_.data(), (int)probs_.size(), 0, rho, &sum_d));
    alpha1_ = sum_d / (double)Mt_;
    eta1_ = gam1_ / alpha1_;
    if (it > 1) {
        VH(update_prior());                                                     // :139
        // damping of x1_hat and alpha1 (:160-165): x1 = rho*x1 + (1-rho)*x1_prev
        VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_X1, rho, VAMPOMI_V_X1, 1 - rho, VAMPOMI_V_X1_PREV, 1.0));
        alpha1_ = rho * alpha1_ + (1 - rho) * alpha1_prev;
    }
    if (verbose) {
        std::cout << "Prior variances = ";
        for (double v : vars_) std::cout << v / (double)N_ << ' ';
        std::cout << std::endl << "Prior probabilities = ";
        for (double p : probs_) std::cout << p << ' ';
        std::cout << std::endl;
    }
    VH(dump(x1_scaled, r1_scaled));                                             // :167-186
    gam2_ = clampg(eta1_ - gam1_);                                              // :194
    VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_R2, eta1_, VAMPOMI_V_X1, -gam1_, VAMPOMI_V_R1, gam2_));   // :197-198
    double x1_corr;
    {
        const int kind[5] = {VAMPOMI_DOT, VAMPOMI_DOT, VAMPOMI_DOT, VAMPOMI_DIFF2, VAMPOMI_DOT};
        const int a[5] = {VAMPOMI_V_X1, VAMPOMI_V_X1, VAMPOMI_V_TRUE, VAMPOMI_V_X1_PREV, VAMPOMI_V_X1_PREV};
        const int b[5] = {VAMPOMI_V_TRUE, VAMPOMI_V_X1, VAMPOMI_V_TRUE, VAMPOMI_V_X1, VAMPOMI_V_X1_PREV};
        double d[5];
        VH(vampomi_dots(ctx_, 5, kind, a, b, nullptr, d));
        // Corr(x1_hat, sqrt(N)*true_signal) (:189): the sqrt(N) factors written out as the reference multiplies them in
        x1_corr = (d[0] * sqrtN) / std::sqrt(d[1] * (d[2] * sqrtN * sqrtN));
        res->nmse = std::sqrt(d[3] / d[4]);
    }
    // z channel (:213-253)
    double beta1 = 0;
    VH(vampomi_probit_zdenoise(ctx_, tau1_, &beta1));
    if (beta1 >= N_) beta1 = N_ - 1.0;                                          // :234-235
    beta1 /= N_;
    VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_P2, 1.0, VAMPOMI_V_Z1HAT, -beta1, VAMPOMI_V_P1, 1 - beta1));   // :250-251
    const double tau2 = tau1_ * (1 - beta1) / beta1;                            // :253
    res->params[0] = alpha1_; res->params[1] = beta1; res->params[2] = gam1_; res->params[3] = tau1_;
    if (verbose)
        std::cout << "alpha1 = " << alpha1_ << std::endl << "beta1 = " << beta1 << std::endl << "tau1 = " << tau1_ << std::endl;

    // A (x/sqrt(N)) (:271, :403), then the probit prediction at threshold 0.5 and the confusion matrix on the host (N values)
    auto confusion_eval = [&](int zvec, double* out6, double corr) -> int {     // :272-282 / :404-415
        VH(vampomi_vec_get(ctx_, zvec, zbuf_.data()));
        int TP = 0, TN = 0, FP = 0, FN = 0;
        for (int i = 0; i < N_; i++) {
            const double yhat = normal_cdf(zbuf_[i]) >= 0.5 ? 1.0 : 0.0;       // predict_probit, :619-629
            const double yi = y_host_[i];
            if (yi == 1 && yhat == 1) TP++;
            else if (yi == 0 && yhat == 0) TN++;
            else if (yi == 1 && yhat == 0) FN++;
            else if (yi == 0 && yhat == 1) FP++;
        }
        out6[0] = TP; out6[1] = TN; out6[2] = FP; out6[3] = FN;
        out6[4] = (double)(TP + TN) / (double)(TP + TN + FP + FN);
        out6[5] = corr;
        return VAMPOMI_OK;
    };
    auto confusion = [&](int xvec, double* out6, double corr) -> int {
        VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_USER_M1, 1.0, xvec, 0.0, xvec, sqrtN));
        VH(vampomi_ax_dev(ctx_, VAMPOMI_V_USER_M1, VAMPOMI_V_USER_N0));
        return confusion_eval(VAMPOMI_V_USER_N0, out6, corr);
    };
    const bool fuse = cfg_.fuse_passes != 0 && cfg_.redundant_passes == 0;      // see step_linear
    const bool recycle = fuse && cfg_.fuse_passes >= 2;
    auto report1 = [&]() {
        if (verbose) std::cout << "Corr(x1_hat,x0) = " << x1_corr << std::endl << "Accuracy1 = " << res->metrics[4] << std::endl
                               << std::endl << "->LMMSE" << std::endl;
    };
    if (!fuse) { VH(confusion(VAMPOMI_V_X1, res->metrics, x1_corr)); report1(); }
    else VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_USER_M1, 1.0, VAMPOMI_V_X1, 0.0, VAMPOMI_V_X1, sqrtN));

    // LMMSE for x (:296-349)
    VH(vampomi_draw_probe(ctx_, cfg_.seed, it));
    VH(vampomi_atx_dev(ctx_, VAMPOMI_V_P2, VAMPOMI_V_USER_M0));                 // :300
    VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_V, tau2, VAMPOMI_V_USER_M0, gam2_, VAMPOMI_V_R2, 1.0));   // :302-303
    int k1 = 0, k2 = 0;
    double rel = 0, vmu = 0;
    if (!fuse) {
        VH(vampomi_cg_solve(ctx_, VAMPOMI_V_V, VAMPOMI_V_X2, 0, tau2, gam2_, cfg_.CG_err_tol, cfg_.CG_max_iter, 0, &k1, &rel, nullptr));   // :307
        VH(vampomi_cg_solve(ctx_, VAMPOMI_V_BERN, VAMPOMI_V_QINV_BERN, 0, tau2, gam2_, cfg_.CG_err_tol, cfg_.CG_max_iter, 1, &k2, &rel, &vmu));
    } else {                                                                    // both solves in lock-step; A (x1/sqrt(N)) rides on their first pass
        const int rhs[2] = {VAMPOMI_V_V, VAMPOMI_V_BERN}, sol[2] = {VAMPOMI_V_X2, VAMPOMI_V_QINV_BERN};
        const int warm[2] = {0, 0}, ata[2] = {-1, -1}, ons[2] = {0, 1};
        int its[2] = {0, 0};
        double rels[2], vmus[2];
        const int track[2] = {recycle ? VAMPOMI_V_Z2 : -1, -1};                 // recycled: the solve keeps Z2 = A x2_hat itself
        VH(vampomi_cg_solve_pair(ctx_, rhs, sol, warm, ata, tau2, gam2_, cfg_.CG_err_tol, cfg_.CG_max_iter, ons, VAMPOMI_V_USER_M1,
                                 VAMPOMI_V_USER_N0, track, its, rels, vmus));
        k1 = its[0]; k2 = its[1]; vmu = vmus[1];
        VH(confusion_eval(VAMPOMI_V_USER_N0, res->metrics, x1_corr));
        report1();
    }
    for (int p = 1; p < cfg_.probes; p++) {                                     // further Hutchinson probes (not in the reference), averaged
        VH(vampomi_draw_probe(ctx_, cfg_.seed + 0x9E3779B97F4A7C15ULL * (unsigned long long)p, it));
        int kp = 0;
        double relp = 0, vmup = 0;
        VH(vampomi_cg_solve(ctx_, VAMPOMI_V_BERN, VAMPOMI_V_QINV_BERN, 0, tau2, gam2_, cfg_.CG_err_tol, cfg_.CG_max_iter, 1, &kp, &relp, &vmup));
        vmu += vmup;
    }
    if (cfg_.probes > 1) vmu /= cfg_.probes;
    const double alpha2 = gam2_ * vmu;                                          // :311
    res->cg_iters_lmmse = k1; res->cg_iters_onsager = k2;
    double x2_corr;
    {
        const int kind[3] = {VAMPOMI_DOT, VAMPOMI_DOT, VAMPOMI_DOT};
        const int a[3] = {VAMPOMI_V_X2, VAMPOMI_V_X2, VAMPOMI_V_TRUE};
        const int b[3] = {VAMPOMI_V_TRUE, VAMPOMI_V_X2, VAMPOMI_V_TRUE};
        double d[3];
        VH(vampomi_dots(ctx_, 3, kind, a, b, nullptr, d));
        x2_corr = (d[0] * sqrtN) / std::sqrt(d[1] * (d[2] * sqrtN * sqrtN));    // :324
    }
    eta2_ = gam2_ / alpha2;
    VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_R1, 1.0, VAMPOMI_V_X2, -alpha2, VAMPOMI_V_R2, 1 - alpha2));   // :337-338
    gam1_ = clampg(gam2_ * (1 - alpha2) / alpha2);                              // :345-346
    // LMMSE for z (:352-376)
    if (!fuse) VH(vampomi_ax_dev(ctx_, VAMPOMI_V_X2, VAMPOMI_V_Z2));
    else if (!recycle) {                                                        // A x2_hat and A (x2_hat/sqrt(N)) (:403) in one pass
        VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_USER_M1, 1.0, VAMPOMI_V_X2, 0.0, VAMPOMI_V_X2, sqrtN));
        const int xin[2] = {VAMPOMI_V_X2, VAMPOMI_V_USER_M1}, xout[2] = {VAMPOMI_V_Z2, VAMPOMI_V_USER_N0};
        VH(vampomi_ax_multi_dev(ctx_, 2, xin, xout));
    }
    const double beta2 = (double)Mt_ / N_ * (1 - alpha2);
    VH(vampomi_vec_lincomb(ctx_, VAMPOMI_V_P1, 1.0, VAMPOMI_V_Z2, -beta2, VAMPOMI_V_P2, 1 - beta2));     // :367-368
    tau1_ = clampg(tau2 * (1 - beta2) / beta2);                                 // :375-376
    res->params[4] = alpha2; res->params[5] = beta2; res->params[6] = gam2_; res->params[7] = tau2;
    if (verbose)
        std::cout << "alpha2 = " << alpha2 << std::endl << "beta2 = " << beta2 << std::endl << "gam1 = " << gam1_ << std::endl
                  << "gam2 = " << gam2_ << std::endl << "tau2 = " << tau2 << std::endl;
    if (!fuse) VH(confusion(VAMPOMI_V_X2, res->metrics + 6, x2_corr));
    else if (!recycle) VH(confusion_eval(VAMPOMI_V_USER_N0, res->metrics + 6, x2_corr));
    else VH(confusion_eval(VAMPOMI_V_Z2, res->metrics + 6, x2_corr));          // the 0.5 threshold only needs the sign of A x2_hat: no 1/sqrt(N) pass
    if (verbose) std::cout << "Corr(x2_hat, x0) = " << x2_corr << std::endl << "Accuracy2 = " << res->metrics[10] << std::endl;
    res->n_params = 8; res->n_metrics = 12;
    alpha2_ = alpha2;
    return VAMPOMI_OK;
}

}  // namespace vampomi_host

// ------------------------------------------------------------------------------------------------------------------
// C entry points (include/vampomi_host.h)
// ------------------------------------------------------------------------------------------------------------------
struct vampomi_solver {
    vampomi_host::Vamp* impl;
};

extern "C" {

int vampomi_solver_create(vampomi_ctx* ctx, const vampomi_solver_config* cfg, const double* y_N, const double* true_signal_M,
                          const double* x1hat_init_M, vampomi_solver** out) {
    if (!ctx || !cfg || !y_N || !out) return VAMPOMI_ERR_ARG;
    *out = nullptr;
    vampomi_host::Vamp* v = new vampomi_host::Vamp(ctx, *cfg);
    int rc = v->init(y_N, true_signal_M, x1hat_init_M);
    if (rc != VAMPOMI_OK) { delete v; return rc; }
    *out = new vampomi_solver{v};
    return VAMPOMI_OK;
}

int vampomi_solver_set_covariates(vampomi_solver* s, int C, const double* Z_NxC) {
    if (!s || !s->impl) return VAMPOMI_ERR_ARG;
    return s->impl->set_covariates(C, Z_NxC);
}

int vampomi_solver_get_cov_eff(vampomi_solver* s, int C, double* out) {
    if (!s || !s->impl || !out || (int)s->impl->cov_eff().size() != C) return VAMPOMI_ERR_ARG;
    for (int j = 0; j < C; j++) out[j] = s->impl->cov_eff()[j];
    return VAMPOMI_OK;
}

long long vampomi_host_read_covariates(const char* path, int C, int N, double* Z_NxC) {
    std::vector<double> Z;
    std::string err;
    if (!path || !Z_NxC) return -1;
    try {
        if (!vampomi_host::read_covariates(path, C, N, &Z, &err)) return -1;
    } catch (const std::exception&) {
        return -2;
    }
    for (size_t i = 0; i < Z.size(); i++) Z_NxC[i] = Z[i];
    return (long long)Z.size();
}

int vampomi_host_newton_cov(const double* y, const double* gg, const double* Z_NxC, int N, int C, double* eta_inout) {
    if (!y || !gg || !Z_NxC || !eta_inout || N < 1 || C < 1) return -1;
    std::vector<double> eta = vampomi_host::newton_method_cov(std::vector<double>(y, y + N), std::vector<double>(gg, gg + N),
                                                               std::vector<double>(Z_NxC, Z_NxC + (size_t)N * C), N, C,
                                                               std::vector<double>(eta_inout, eta_inout + C), false, 0);
    for (int j = 0; j < C; j++) eta_inout[j] = eta[j];
    return 0;
}

int vampomi_solver_save_state(vampomi_solver* s, const char* path) {
    if (!s || !s->impl) return VAMPOMI_ERR_ARG;
    return s->impl->save_state(path);
}
int vampomi_solver_load_state(vampomi_solver* s, const char* path) {
    if (!s || !s->impl) return VAMPOMI_ERR_ARG;
    return s->impl->load_state(path);
}

int vampomi_solver_step(vampomi_solver* s, vampomi_iter_result* res, double* x1_scaled_M, double* r1_scaled_M) {
    if (!s || !s->impl) return VAMPOMI_ERR_ARG;
    return s->impl->step(res, x1_scaled_M, r1_scaled_M);
}

int vampomi_solver_destroy(vampomi_solver* s) {
    if (s) { delete s->impl; delete s; }
    return VAMPOMI_OK;
}

int vampomi_host_csv_row(unsigned it, const double* values, int n, char* buf, int buflen) {
    if (!buf || n < 0 || (n > 0 && !values)) return -1;
    std::string row = vampomi_host::CsvFile::format_row(it, std::vector<double>(values, values + n));
    if ((int)row.size() + 1 > buflen) return -1;
    std::memcpy(buf, row.c_str(), row.size() + 1);
    return (int)row.size();
}

long long vampomi_host_read_phen(const char* path, int standardize, double* out, long long cap) {
    std::vector<double> y;
    try {
        if (!path || !vampomi_host::read_phen(path, standardize != 0, &y)) return -1;
    } catch (const std::exception&) {
        return -2;
    }
    for (long long i = 0; i < (long long)y.size() && i < cap; i++) out[i] = y[i];
    return (long long)y.size();
}

double vampomi_host_linear_reg1d_pvals(double sumx, double sumsqx, double sumxy, double sumy, double sumsqy, int n) {
    return vampomi_host::linear_reg1d_pvals(sumx, sumsqx, sumxy, sumy, sumsqy, n);
}

void vampomi_host_loo_pvals(const double* x1_M, const double* sums_3M, double sum_w, double sumsq_w, int N, long long M, double* pvals_M, int threads) {
    vampomi_host::loo_pvals(x1_M, sums_3M, sum_w, sumsq_w, N, M, pvals_M, threads);
}

void vampomi_host_loo_pvals_flagged(const double* x1_M, const double* sums_3M, double sum_w, double sumsq_w, int N, long long M,
                                    const unsigned char* const_M, double* pvals_M, int threads) {
    vampomi_host::loo_pvals(x1_M, sums_3M, sum_w, sumsq_w, N, M, pvals_M, threads, const_M);
}

double vampomi_host_probe_sign(unsigned long long seed, int it, unsigned long long global_marker) {
    return vampomi::probe_sign(seed, it, global_marker);
}

void vampomi_host_probit_p1(unsigned long long seed, int N, double* out) {
    std::vector<double> p = vampomi_host::probit_p1(seed, N);
    for (int i = 0; i < N; i++) out[i] = p[i];
}

int vampomi_host_merge_components(double* probs, double* vars, int L, double thr) {
    std::vector<double> p(probs, probs + L), v(vars, vars + L);
    vampomi_host::merge_components(p, v, thr);
    for (size_t i = 0; i < p.size(); i++) { probs[i] = p[i]; vars[i] = v[i]; }
    return (int)p.size();
}

void vampomi_solver_default_config(vampomi_solver_config* cfg) {
    if (!cfg) return;
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->model = 0;
    cfg->gam1 = 1e-6; cfg->gamw = 2.0; cfg->rho = 0.5;
    cfg->CG_max_iter = 500; cfg->CG_err_tol = 1e-5;
    cfg->EM_max_iter = 1; cfg->EM_err_thr = 1e-2;
    cfg->learn_vars = 1; cfg->learn_prior_delay = 1; cfg->merge_vars_thr = 0.5;
    const double vars[10] = {0, 1e-06, 6e-06, 3e-05, 2e-04, 1e-03, 6e-03, 3e-02, 2e-01, 1e+00};
    const double probs[10] = {9.90000e-01, 5.00000e-03, 2.50000e-03, 1.25000e-03, 6.25000e-04,
                              3.12500e-04, 1.56250e-04, 7.81250e-05, 3.90625e-05, 3.90625e-05};
    cfg->L = 10;
    for (int i = 0; i < 10; i++) { cfg->vars[i] = vars[i]; cfg->probs[i] = probs[i]; }
    cfg->seed = 0;
    cfg->redundant_passes = 0;
    cfg->fuse_passes = 3;
    cfg->probes = 1;
}

}  // extern "C"
