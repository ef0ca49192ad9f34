// main_meth's program logic (reference: src/main_meth.cpp:9-270) over the kernel ABI. One "rank" = one marker shard on
// one GPU; with --gpus G the G ranks run as threads of this process and meet in NCCL collectives, where the reference
// runs G MPI processes. Output files, their byte layout, stdout landmarks and exit codes follow the reference.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <future>
#include <iostream>
#include <mutex>
#include <stdexcept>
#include <exception>
#include <thread>
#include <vector>
#include "../../../include/vampomi_host.h"
#include "cov.h"
#include "io.h"
#include "options.h"
#include "vamp.h"

namespace vampomi_host {
namespace {

double now_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// Host-side agreement of the rank threads of `main_meth --gpus G` BEFORE they enter a collective: where an MPI job would be
// torn down by MPI_Abort (src/utilities.cpp:21-46), a rank thread that failed locally (unreadable file, allocation) tells the
// others here, so that nobody is left waiting in ncclCommInitRank or in a device-side exchange for a peer that has returned.
struct RankGate {
    std::mutex m;
    std::condition_variable cv;
    int n = 1, arrived = 0, gen = 0;
    bool failed = false;
    bool agree(bool ok) {                       // true only if EVERY rank reported ok (now and at every earlier gate)
        std::unique_lock<std::mutex> lk(m);
        if (!ok) failed = true;
        const int g = gen;
        if (++arrived == n) { arrived = 0; gen++; cv.notify_all(); }
        else cv.wait(lk, [&] { return gen != g; });
        return !failed;
    }
};

struct Rank {
    const Options& opt;
    int rank, nranks;
    const void* nccl_id;
    RankGate* gate = nullptr;
    bool agree(bool ok) const { return gate ? gate->agree(ok) : ok; }
    vampomi_ctx* ctx = nullptr;
    long long M = 0, S = 0;
    bool root() const { return rank == 0; }
};

int fatal(const Rank& r, const std::string& msg) {
    if (r.root() || r.nranks > 1) std::cout << "FATAL: " << msg << std::endl;
    return 1;
}
int fatal_abi(const Rank& r, const char* what) {
    std::cout << "FATAL: " << what << " failed on rank " << r.rank << ": " << vampomi_last_error() << std::endl;
    return 1;
}

// `class data` constructor (src/data.cpp:24-47): phenotype, marker block into HBM, marker statistics.
int load_dataset(Rank& r, const std::string& phenfp, const std::string& methfp, int N, std::vector<double>* y) {
    // stage 1, local: phenotype and context (host file I/O, cudaMalloc of the block) — then all rank threads agree
    auto stage1 = [&]() -> int {
        if (!read_phen(phenfp, r.opt.model != "bin_class", y)) return 1;                  // src/data.cpp:40-43
        if ((int)y->size() != N) {
            std::cout << "FATAL: phenotype file " << phenfp << " has " << y->size() << " rows but --N is " << N << std::endl;
            return 1;                                                                      // assert(nas + nonas == N), :85
        }
        int ndev = 0;
        if (vampomi_device_count(&ndev) != VAMPOMI_OK) return fatal_abi(r, "device query");
        if (r.nranks > ndev) return fatal(r, "--gpus " + std::to_string(r.nranks) + " exceeds the " + std::to_string(ndev) + " visible CUDA devices");
        const int storage = r.opt.storage == "f32" ? VAMPOMI_STORE_F32 : VAMPOMI_STORE_F64;
        if (vampomi_create_ex(r.rank, N, (long long)r.opt.Mt, r.nranks, r.rank, storage, &r.ctx) != VAMPOMI_OK) return fatal_abi(r, "vampomi_create");
        if (storage == VAMPOMI_STORE_F32 && r.root())
            std::cout << "INFO  : --storage f32: the marker block is rounded to FP32 in GPU memory (all arithmetic stays FP64)" << std::endl;
        return 0;
    };
    int rc = 1;
    try {
        rc = stage1();
    } catch (const std::exception& e) {                                                    // e.g. an NA phenotype (src/data.cpp:74)
        std::cout << "FATAL: " << e.what() << std::endl;
    } catch (...) {
        std::cout << "FATAL: unknown error while reading the inputs of rank " << r.rank << std::endl;
    }
    if (!r.agree(rc == 0)) return rc ? rc : 1;
    // stage 2: communicator (collective), then the local read of the shard's block — and agreement again before the statistics,
    // which end with the rank barrier
    const int storage = r.opt.storage == "f32" ? VAMPOMI_STORE_F32 : VAMPOMI_STORE_F64;
    rc = (r.nranks > 1 && vampomi_comm_init(r.ctx, r.nccl_id) != VAMPOMI_OK) ? fatal_abi(r, "vampomi_comm_init") : 0;
    if (!r.agree(rc == 0)) return rc ? rc : 1;
    if (r.nranks > 1 && r.root()) {
        int mode = 0;
        vampomi_comm_mode(r.ctx, &mode);
        std::cout << "INFO  : cross-GPU sums over " << (mode == 2 ? "NVLink peer memory (fused one-shot all-reduce)" : "NCCL all-reduce")
                  << " on " << r.nranks << " GPUs" << std::endl;
    }
    if (r.root()) std::cout << "meth file name = " << methfp << std::endl;            // :123
    const size_t raw_bytes = (size_t)r.M * (size_t)N * (storage == VAMPOMI_STORE_F32 ? 4 : 8);
    printf("INFO  : rank %d has allocated %zu bytes (%.3f GB) for raw data.\n", r.rank, raw_bytes, double(raw_bytes) / 1.0E9);   // :131
    double ts = now_s();
    rc = vampomi_load_file(r.ctx, methfp.c_str()) != VAMPOMI_OK ? fatal_abi(r, "loading the methylation data") : 0;
    if (!r.agree(rc == 0)) return rc ? rc : 1;
    double te = now_s();
    if (r.root()) std::cout << "reading methylation data took " << te - ts << " seconds." << std::endl;   // :151
    if (r.opt.missing == "mean") {                       // --missing mean: NaN -> column mean in HBM, before the statistics
        long long counts[3] = {0, 0, 0};
        rc = vampomi_impute_missing(r.ctx, counts) != VAMPOMI_OK ? fatal_abi(r, "imputing missing values") : 0;
        const double ti = now_s();
        if (rc == 0)
            printf("INFO  : rank %d replaced %lld missing values by their marker's mean (%lld markers with missing values, %lld without an observed value).\n",
                   r.rank, counts[0], counts[1], counts[2]);
        if (!r.agree(rc == 0)) return rc ? rc : 1;
        if (r.root()) std::cout << "imputing missing values took " << ti - te << " seconds." << std::endl;
        te = now_s();
    }
    if (vampomi_compute_stats(r.ctx, r.opt.alpha_scale) != VAMPOMI_OK) return fatal_abi(r, "marker statistics");
    if (r.root()) std::cout << "rank = " << r.rank << ": statistics took " << now_s() - te << " seconds to run." << std::endl;   // :281
    return 0;
}

// src/utilities.cpp:104-122 — whitespace-separated text estimates, entries [S, S+M)
std::vector<double> read_text_vec(const std::string& path, long long M, long long S) {
    std::vector<double> v;
    std::ifstream in(path);
    double value;
    long long it = 0;
    while (in >> value) {
        if (it >= S && it < S + M) v.push_back(value);
        else if (it >= S + M) break;
        it++;
    }
    v.resize((size_t)M, 0.0);
    return v;
}

int run_infere(Rank& r) {
    const Options& o = r.opt;
    const int N = (int)o.N;
    std::vector<double> y;
    if (int rc = load_dataset(r, o.phen_file, o.meth_file, N, &y)) return rc;

    std::vector<double> true_signal((size_t)r.M, 0.0), x1hat_init((size_t)r.M, 0.0);
    if (!o.true_signal_file.empty()) true_signal = read_vec(o.true_signal_file, r.M, r.S);     // src/main_meth.cpp:69-73
    if (!o.estimate_file.empty()) x1hat_init = read_vec(o.estimate_file, r.M, r.S);            // :75-80

    vampomi_solver_config cfg;
    vampomi_solver_default_config(&cfg);
    if (o.model == "linear") cfg.model = 0;
    else if (o.model == "bin_class") cfg.model = 1;
    else throw std::runtime_error("Invalid model specification!");                             // src/vamp.cpp:104
    cfg.gam1 = o.gam1;
    cfg.gamw = 1.0 / (1.0 - o.h2);                                                             // src/main_meth.cpp:52
    cfg.rho = o.rho;
    cfg.CG_max_iter = (int)o.CG_max_iter; cfg.CG_err_tol = o.CG_err_tol;
    cfg.EM_max_iter = (int)o.EM_max_iter; cfg.EM_err_thr = o.EM_err_thr;
    cfg.learn_vars = (int)o.learn_vars; cfg.learn_prior_delay = (int)o.learn_prior_delay;
    cfg.merge_vars_thr = o.merge_vars_thr;
    if (o.probs.size() != o.vars.size() || o.probs.empty() || o.probs.size() > VAMPOMI_MAX_MIX)
        return fatal(r, "--probs and --vars must have the same length, between 1 and " + std::to_string(VAMPOMI_MAX_MIX));
    cfg.L = (int)o.probs.size();
    for (int i = 0; i < cfg.L; i++) { cfg.probs[i] = o.probs[i]; cfg.vars[i] = o.vars[i]; }
    cfg.seed = o.seed;
    cfg.probes = o.probes;
    cfg.redundant_passes = o.schedule == "reference" ? 1 : 0;
    cfg.fuse_passes = o.schedule == "onepass" ? 3 : o.schedule == "recycled" ? 2 : o.schedule == "fused" ? 1 : 0;

    Vamp vamp(r.ctx, cfg);
    vamp.verbose = r.root();
    vamp.verbosity = o.verbosity;
    if (vamp.init(y.data(), true_signal.data(), x1hat_init.data()) != VAMPOMI_OK) return fatal_abi(r, "solver initialisation");
    if (o.C > 0) {
        // data::read_covariates (src/data.cpp:159-227). The reference's compiling main never calls it, so `--C > 0` there reads
        // an empty matrix out of bounds (SURVEY.md §2 #12); here --C / --cov-file do what the loops' own covariate code expects.
        std::vector<double> Z;
        std::string err;
        const double tc = now_s();
        bool okc = false;
        try { okc = read_covariates(o.cov_file, (int)o.C, N, &Z, &err); } catch (const std::exception&) { err = "covariate file " + o.cov_file + " holds a value that is not a number"; }
        if (!okc) return fatal(r, err);
        if (r.root()) std::cout << "rank = " << r.rank << ": reading covariates took " << now_s() - tc << " seconds to run." << std::endl;   // :200
        if (vamp.set_covariates((int)o.C, Z.data()) != VAMPOMI_OK) return fatal_abi(r, "covariates");
    }

    // --resume-from: continue from a checkpoint of this very problem (vampomi_solver_load_state); the CSV files are kept and the
    // remaining rows land at their usual offsets
    int first_it = 1;
    const bool resuming = !o.resume_from.empty();
    if (resuming) {
        const int rc_load = vamp.load_state(o.resume_from.c_str());
        if (!r.agree(rc_load == VAMPOMI_OK)) return fatal(r, "could not resume from " + o.resume_from + " (missing, damaged or written for another problem)");
        first_it = vamp.iteration() + 1;
        if (r.root()) std::cout << "INFO  : resuming after iteration " << vamp.iteration() << " from " << o.resume_from << std::endl;
    }
    // setup_io (src/vamp.cpp:854-882): rank 0 owns the three CSVs
    const std::string base = o.out_dir + "/" + o.out_name;
    CsvFile csv_metrics, csv_params, csv_prior;
    if (r.root()) {
        if (!csv_metrics.open(base + "_metrics.csv", resuming) || !csv_params.open(base + "_params.csv", resuming) || !csv_prior.open(base + "_prior.csv", resuming)) {
            fprintf(stderr, "*FATAL*: could not create the CSV files under %s\n", o.out_dir.c_str());   // check_mpi abort
            return 1;
        }
        if (cfg.model == 0 && !resuming) {                                                     // headers only in infere_linear, src/vamp.cpp:115-123
            csv_metrics.header({"iteration", "R2 denoising", "x1 correlation denoising", "R2 LMMSE", "x2 correlation LMMSE",
                                "z1 correlation denoising", "z2 correlation LMMSE"});
            csv_params.header({"iteration", "alpha1", "gam1", "alpha2", "gam2", "gamw"});
            std::vector<std::string> ph{"iteration", "number of components"};
            for (size_t i = 0; i < o.probs.size(); i++) ph.push_back("prob" + std::to_string(i));
            for (size_t i = 0; i < o.vars.size(); i++) ph.push_back("var" + std::to_string(i));
            csv_prior.header(ph);
        }
    }

    // The two per-iteration vector files (src/vamp.cpp:235-249) are written by a helper thread while the next iteration
    // already runs on the GPU: two sets of host buffers, at most one write in flight, joined before a buffer is reused and
    // before leaving.
    std::vector<double> x1buf[2] = {std::vector<double>((size_t)r.M), std::vector<double>((size_t)r.M)};
    std::vector<double> r1buf[2] = {std::vector<double>((size_t)r.M), std::vector<double>((size_t)r.M)};
    std::future<bool> writer;
    std::string writer_file;
    auto join_writer = [&]() -> bool { return !writer.valid() || writer.get(); };
    double total_time = 0;
    const int max_iter = (int)o.iterations;
    for (int it = first_it; it <= max_iter; it++) {
        std::vector<double>&x1s = x1buf[it & 1], &r1s = r1buf[it & 1];
        if (r.root())
            std::cout << std::endl << "********************" << std::endl << "iteration = " << it << std::endl
                      << "********************" << std::endl;
        const double t0 = now_s();
        vampomi_iter_result res;
        if (vamp.step(&res, x1s.data(), r1s.data()) != VAMPOMI_OK) return fatal_abi(r, "VAMP iteration");
        const double t1 = now_s();
        const std::string f_x1 = base + "_it_" + std::to_string(it) + ".bin";                  // src/vamp.cpp:235-249
        const std::string f_r1 = base + "_r1_it_" + std::to_string(it) + ".bin";
        if (!join_writer()) return fatal(r, "could not write " + writer_file);
        writer_file = f_x1;
        writer = std::async(std::launch::async, [f_x1, f_r1, &x1s, &r1s, M = r.M, S = r.S]() {
            return store_vec(f_x1, x1s.data(), M, S) && store_vec(f_r1, r1s.data(), M, S);
        });
        if (r.root()) {
            std::cout << "x1_hat filepath_out is " << f_x1 << std::endl << "r1_hat filepath_out is " << f_r1 << std::endl;
            std::cout << "[CG] LMMSE solve: " << res.cg_iters_lmmse << " iterations, onsager solve: " << res.cg_iters_onsager
                      << " iterations, matrix passes: " << res.matrix_passes << std::endl;
            std::cout << "...storing parameters to CSV files" << std::endl;
            csv_params.row(it, std::vector<double>(res.params, res.params + res.n_params));    // :390-391
            csv_metrics.row(it, std::vector<double>(res.metrics, res.metrics + res.n_metrics));
            if (cfg.model == 1) {                                                              // src/vamp_probit.cpp:423-434
                std::vector<double> prior{(double)res.L};
                prior.insert(prior.end(), res.probs, res.probs + res.L);
                prior.insert(prior.end(), res.vars, res.vars + res.L);
                csv_prior.row(it, prior);
            }
            total_time += t1 - t0;
            std::cout << "Total iteration time = " << t1 - t0 << std::endl;                    // src/vamp.cpp:400-401
            std::cout << "Total computation time so far = " << total_time << std::endl;
            std::cout << "...stopping criteria assessment" << std::endl;
            std::cout << "x1_hat NMSE = " << res.nmse << std::endl;                            // :415-417
            std::cout << "stop_criteria_thr = " << o.stop_criteria_thr << std::endl;
        }
        if (o.checkpoint_every > 0 && it % o.checkpoint_every == 0) {
            const std::string ck = base + "_checkpoint_it_" + std::to_string(it) + ".bin";
            if (!r.agree(vamp.save_state(ck.c_str()) == VAMPOMI_OK)) return fatal(r, "could not write " + ck);
            if (r.root()) std::cout << "checkpoint filepath_out is " << ck << std::endl;
        }
        if (it > 1 && res.nmse < o.stop_criteria_thr) {                                        // :419-423
            if (r.root()) std::cout << "...stopping criteria fulfilled" << std::endl;
            break;
        }
        if (it == max_iter && r.root())
            std::cout << "...maximal number of iterations was achieved. The algorithm might not converge!" << std::endl;
    }
    if (!join_writer()) return fatal(r, "could not write " + writer_file);
    return 0;
}

int run_test(Rank& r) {                                                                        // src/main_meth.cpp:112-205
    const Options& o = r.opt;
    const int N_test = (int)o.N_test;
    std::vector<double> y;
    if (int rc = load_dataset(r, o.phen_file_test, o.meth_file_test, N_test, &y)) return rc;
    CsvFile csv;
    if (r.root()) {
        if (!csv.open(o.out_dir + "/" + o.out_name + "_test.csv")) { fprintf(stderr, "*FATAL*: could not create _test.csv\n"); return 1; }
        csv.header({"iteration", "R2 test", "z correlation test"});
    }
    const std::string est = o.estimate_file;
    const size_t pos_dot = est.find(".");                                                      // :151 (first dot, sic)
    const std::string ext = pos_dot == std::string::npos ? est : est.substr(pos_dot + 1);
    const size_t pos_it = est.rfind("it");
    if (r.root()) std::cout << "est_file_name = " << est << std::endl
                            << "iter range = [" << o.test_iter_range[0] << ", " << o.test_iter_range[1] << "]" << std::endl;
    // The reference applies A to one saved estimate per pass (:178). Every pass is bound by streaming the test matrix, so
    // up to four iteration files share one read of it (vampomi_ax_multi_dev); rows are still written in iteration order,
    // and a file that cannot be read stops the run exactly after the rows of the iterations before it.
    std::vector<double> z((size_t)N_test);
    const int in_vec[4] = {VAMPOMI_V_X1, VAMPOMI_V_X2, VAMPOMI_V_R1, VAMPOMI_V_R2};
    const int out_vec[4] = {VAMPOMI_V_Z1, VAMPOMI_V_Z2, VAMPOMI_V_USER_N0, VAMPOMI_V_USER_N1};
    const double sd = calc_stdev(y);
    double yy = 0;
    for (int i = 0; i < N_test; i++) yy += y[i] * y[i];
    for (int it0 = o.test_iter_range[0]; it0 <= o.test_iter_range[1]; it0 += 4) {
        const int nb = std::min(4, o.test_iter_range[1] - it0 + 1);
        int got = 0;
        std::exception_ptr err;
        for (int b = 0; b < nb; b++) {
            const std::string f = est.substr(0, pos_it) + "it_" + std::to_string(it0 + b) + "." + ext;  // :166
            try {
                std::vector<double> x = ext == "bin" ? read_vec(f, r.M, r.S) : read_text_vec(f, r.M, r.S);
                for (double& v : x) v *= std::sqrt((double)N_test);                            // :174-175
                if (vampomi_vec_set(r.ctx, in_vec[b], x.data()) != VAMPOMI_OK) return fatal_abi(r, "vec_set");
                got++;
            } catch (...) {
                err = std::current_exception();
                break;
            }
        }
        if (got > 0 && vampomi_ax_multi_dev(r.ctx, got, in_vec, out_vec) != VAMPOMI_OK) return fatal_abi(r, "Ax");   // :178
        for (int b = 0; b < got; b++) {
            if (vampomi_vec_get(r.ctx, out_vec[b], z.data()) != VAMPOMI_OK) return fatal_abi(r, "vec_get");
            double l2 = 0, zy = 0, zz = 0;
            for (int i = 0; i < N_test; i++) {
                l2 += (y[i] - z[i]) * (y[i] - z[i]);
                zy += z[i] * y[i]; zz += z[i] * z[i];
            }
            const double r2 = 1 - l2 / (sd * sd * y.size());                                   // :187-188
            const double corr_y = (zy * r.nranks) / std::sqrt((zz * r.nranks) * (yy * r.nranks));  // :191 (sync=1 on replicated vectors)
            if (r.root()) {
                std::cout << r2 << ", ";
                csv.row(it0 + b, {r2, corr_y * corr_y});
            }
        }
        if (err) std::rethrow_exception(err);
    }
    return 0;
}

// `test` as the reference's probit driver means it (src/main_meth_probit.cpp:104-200): per saved iteration the probit
// prediction at threshold 0.5 on the test set, confusion matrix and accuracy -> _test.csv rows [TP, TN, FP, FN, ACC], no header.
int run_test_probit(Rank& r) {
    const Options& o = r.opt;
    const int N_test = (int)o.N_test;
    std::vector<double> y;
    if (int rc = load_dataset(r, o.phen_file_test, o.meth_file_test, N_test, &y)) return rc;
    CsvFile csv;
    if (r.root() && !csv.open(o.out_dir + "/" + o.out_name + "_test.csv")) { fprintf(stderr, "*FATAL*: could not create _test.csv\n"); return 1; }
    const std::string est = o.estimate_file;
    const size_t pos_dot = est.find(".");                                                      // :130 (first dot, sic)
    const std::string ext = pos_dot == std::string::npos ? est : est.substr(pos_dot + 1);
    const size_t pos_it = est.rfind("it");
    if (r.root()) std::cout << "est_file_name = " << est << std::endl
                            << "iter range = [" << o.test_iter_range[0] << ", " << o.test_iter_range[1] << "]" << std::endl;
    std::vector<double> z((size_t)N_test);
    for (int it = o.test_iter_range[0]; it <= o.test_iter_range[1]; it++) {
        const std::string f = est.substr(0, pos_it) + "it_" + std::to_string(it) + "." + ext;  // :146
        std::vector<double> x = ext == "bin" ? read_vec(f, r.M, r.S) : read_text_vec(f, r.M, r.S);
        for (double& v : x) v *= std::sqrt((double)N_test);                                    // :154-155
        if (vampomi_vec_set(r.ctx, VAMPOMI_V_X1, x.data()) != VAMPOMI_OK || vampomi_ax_dev(r.ctx, VAMPOMI_V_X1, VAMPOMI_V_Z1) != VAMPOMI_OK ||
            vampomi_vec_get(r.ctx, VAMPOMI_V_Z1, z.data()) != VAMPOMI_OK)
            return fatal_abi(r, "Ax");                                                         // :158
        int TP = 0, TN = 0, FP = 0, FN = 0;
        for (int i = 0; i < N_test; i++) {
            const double yhat = normal_cdf(z[i]) >= 0.5 ? 1.0 : 0.0;                           // :160-166
            if (y[i] == 1 && yhat == 1) TP++;
            else if (y[i] == 0 && yhat == 0) TN++;
            else if (y[i] == 1 && yhat == 0) FN++;
            else if (y[i] == 0 && yhat == 1) FP++;
        }
        const double ACC = (double)(TP + TN) / (double)(TP + TN + FP + FN);
        if (r.root()) {
            std::cout << "---- Iteration " << it << "----" << std::endl << "TP = " << TP << std::endl << "TN = " << TN << std::endl
                      << "FP = " << FP << std::endl << "FN = " << FN << std::endl << "Accuracy = " << ACC << std::endl;
            csv.row(it, {(double)TP, (double)TN, (double)FP, (double)FN, ACC});                // :198
        }
    }
    return 0;
}

// `predict` (src/main_meth_probit.cpp:201-227): z_hat = A_test (x_est * sqrt(N_test)) -> text file "<estimate up to 'it'>.yhat"
int run_predict(Rank& r) {
    const Options& o = r.opt;
    const int N_test = (int)o.N_test;
    std::vector<double> y;
    if (int rc = load_dataset(r, o.phen_file_test, o.meth_file_test, N_test, &y)) return rc;
    const std::string est = o.estimate_file;
    const size_t pos_it = est.rfind("it");
    const std::string pred = est.substr(0, pos_it) + ".yhat";                                  // :208-209
    std::vector<double> x = read_vec(est, r.M, r.S);
    for (double& v : x) v *= std::sqrt((double)N_test);
    std::vector<double> z((size_t)N_test);
    if (vampomi_vec_set(r.ctx, VAMPOMI_V_X1, x.data()) != VAMPOMI_OK || vampomi_ax_dev(r.ctx, VAMPOMI_V_X1, VAMPOMI_V_Z1) != VAMPOMI_OK ||
        vampomi_vec_get(r.ctx, VAMPOMI_V_Z1, z.data()) != VAMPOMI_OK)
        return fatal_abi(r, "Ax");
    if (r.root()) {                                                                            // store_vec_to_file, src/utilities.cpp:126-135
        std::ofstream file(pred);
        if (!file) return fatal(r, "could not write " + pred);
        for (double v : z) file << v << std::endl;
        std::cout << "Storing predictions to file " << pred << std::endl;
    }
    return 0;
}

int run_association(Rank& r) {                                                                 // src/main_meth.cpp:206-265
    const Options& o = r.opt;
    const int N = (int)o.N;
    std::vector<double> y;
    if (int rc = load_dataset(r, o.phen_file, o.meth_file, N, &y)) return rc;
    auto iter_tag = [](const std::string& name, std::string* tag) -> bool {                    // :223-226
        size_t p1 = name.rfind("it_"), p2 = name.rfind(".bin");
        if (p1 == std::string::npos || p2 == std::string::npos || p2 < p1 + 3) return false;
        *tag = name.substr(p1 + 3, p2 - (p1 + 3));
        try { (void)std::stoi(*tag); } catch (...) { return false; }
        return true;
    };
    std::vector<double> pvals((size_t)r.M, 0.0);
    std::string out, tag;
    if (o.pval_method == "se") {
        if (!iter_tag(o.r1_file, &tag)) return fatal(r, "cannot parse the iteration number from --r1-file " + o.r1_file);
        if (r.root()) std::cout << o.r1_file << std::endl;
        std::vector<double> r1 = read_vec(o.r1_file, r.M, r.S);
        if (vampomi_pvals_se(r.ctx, r1.data(), o.gam1, pvals.data()) != VAMPOMI_OK) return fatal_abi(r, "se p-values");
        out = o.out_dir + "/" + o.out_name + "_it_" + tag + "_pval_se.bin";
    } else if (o.pval_method == "loo") {
        if (!iter_tag(o.estimate_file, &tag)) return fatal(r, "cannot parse the iteration number from --estimate-file " + o.estimate_file);
        std::vector<double> x1 = read_vec(o.estimate_file, r.M, r.S);
        const double sqrtN = std::sqrt((double)N);
        for (double& v : x1) v *= sqrtN;                                                       // :254-255
        // y_mod = y - A x1_hat (src/data.cpp:390-391), then one streaming pass for the per-marker sums
        if (vampomi_vec_set(r.ctx, VAMPOMI_V_Y, y.data()) != VAMPOMI_OK || vampomi_vec_set(r.ctx, VAMPOMI_V_X1, x1.data()) != VAMPOMI_OK ||
            vampomi_ax_dev(r.ctx, VAMPOMI_V_X1, VAMPOMI_V_Z1) != VAMPOMI_OK ||
            vampomi_vec_lincomb(r.ctx, VAMPOMI_V_USER_N1, 1.0, VAMPOMI_V_Y, -1.0, VAMPOMI_V_Z1, 1.0) != VAMPOMI_OK)
            return fatal_abi(r, "loo residual");
        std::vector<double> w((size_t)N), sums((size_t)3 * r.M);
        std::vector<unsigned char> constant((size_t)r.M);
        if (vampomi_vec_get(r.ctx, VAMPOMI_V_USER_N1, w.data()) != VAMPOMI_OK || vampomi_loo_sums(r.ctx, VAMPOMI_V_USER_N1, sums.data()) != VAMPOMI_OK ||
            vampomi_constant_columns(r.ctx, constant.data()) != VAMPOMI_OK)
            return fatal_abi(r, "loo sums");
        double sw = 0, sww = 0;
        for (double v : w) { sw += v; sww += v * v; }
        // Student-t per marker, on the host's threads; a constant column gets p = 1 (DESIGN §4)
        loo_pvals(x1.data(), sums.data(), sw, sww, N, r.M, pvals.data(), 0, constant.data());
        out = o.out_dir + "/" + o.out_name + "_it_" + tag + "_pval_loo.bin";
    } else {
        return 0;                                                                              // the reference silently does nothing
    }
    if (r.root()) std::cout << "Storing p-values to file " + out << std::endl;
    if (!store_vec(out, pvals.data(), r.M, r.S)) return fatal(r, "could not write " + out);
    return 0;
}

int run_rank(const Options& opt, int rank, int nranks, const void* nccl_id, RankGate* gate) {
    Rank r{opt, rank, nranks, nccl_id};
    r.gate = gate;
    if (vampomi_divide_work((long long)opt.Mt, nranks, rank, &r.M, &r.S) != VAMPOMI_OK) return fatal_abi(r, "divide_work");
    const long long Mm = opt.Mt % nranks != 0 ? opt.Mt / nranks + 1 : opt.Mt / nranks;
    printf("INFO   : rank %4d has %lld markers over tot Mt = %u, max Mm = %lld, starting at S = %lld\n", rank, r.M, opt.Mt, Mm, r.S);   // src/utilities.cpp:231
    int rc = 0;
    try {
        if (opt.run_mode == "infere") rc = run_infere(r);
        else if (opt.run_mode == "test" && opt.probit_entry) rc = run_test_probit(r);
        else if (opt.run_mode == "predict" && opt.probit_entry) rc = run_predict(r);
        else if (opt.run_mode == "test") rc = run_test(r);
        else if (opt.run_mode == "association_test") rc = run_association(r);
    } catch (const std::exception& e) {
        std::cout << "FATAL: " << e.what() << std::endl;     // the reference throws string literals and terminates
        rc = 1;
    } catch (const char* what) {
        std::cout << "FATAL: " << what << std::endl;
        rc = 1;
    } catch (...) {
        std::cout << "FATAL: unknown error on rank " << rank << std::endl;
        rc = 1;
    }
    if (r.ctx) vampomi_destroy(r.ctx);
    return rc;
}

}  // namespace
}  // namespace vampomi_host

static int main_impl(int argc, char** argv, bool probit_entry) {
    using namespace vampomi_host;
    Options opt;
    std::string echo;
    if (!opt.parse(argc, argv, &echo)) return 1;
    std::cout << echo << std::endl;                                                            // rank 0 echo, src/options.cpp:288-289
    if (probit_entry) {
        // main_meth_probit (src/main_meth_probit.cpp, BASELINE.json configuration 4): the reference's stale probit driver does not
        // compile against its own vamp.hpp (SURVEY.md fact 2); what it means is main_meth with the probit model, plus its own
        // `test` (confusion matrix) and `predict` run modes
        opt.probit_entry = true;
        opt.model = "bin_class";
    }
    const bool test_like = opt.run_mode == "test" || (probit_entry && opt.run_mode == "predict");
    if (opt.Mt == 0 || (test_like ? opt.N_test == 0 : opt.N == 0)) {
        std::cout << "FATAL  : --Mt and --N (or --N-test in test mode) have to be given" << std::endl;
        return 1;
    }
    const int G = opt.gpus;
    if (G == 1) return run_rank(opt, 0, 1, nullptr, nullptr);
    char id[128];
    if (vampomi_comm_get_unique_id(id) != VAMPOMI_OK) {
        std::cout << "FATAL: NCCL bootstrap failed: " << vampomi_last_error() << std::endl;
        return 1;
    }
    std::vector<int> rcs((size_t)G, 0);
    std::vector<std::thread> th;
    RankGate gate;
    gate.n = G;
    for (int g = 0; g < G; g++) th.emplace_back([&, g]() { rcs[g] = run_rank(opt, g, G, id, &gate); });
    for (auto& t : th) t.join();
    for (int rc : rcs) if (rc) return rc;
    return 0;
}

extern "C" int vampomi_main(int argc, char** argv) { return main_impl(argc, argv, false); }
extern "C" int vampomi_main_probit(int argc, char** argv) { return main_impl(argc, argv, true); }
