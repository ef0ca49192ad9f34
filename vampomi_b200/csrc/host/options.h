// Command-line contract of main_meth.exe (reference: src/options.hpp:5-107, src/options.cpp:13-303).
// Same flags, same defaults (the code's, not the README's), same FATAL messages and exit status. Two additions
// that the reference does not have: --seed (counter-hash seed of the Hutchinson probe / probit start) and --gpus; and two
// that choose HOW the same numbers are computed: --storage (FP32 residency of the block, opt-in) and --schedule (which matrix
// products share a read of the block: recycled (default) / fused / plain / reference, see vampomi_solver_config::fuse_passes).
// --missing mean makes the run read a matrix with NaN entries as the matrix with each NaN replaced by its column's mean.
#pragma once
#include <string>
#include <vector>

namespace vampomi_host {

struct Options {
    std::string meth_file, meth_file_test, phen_file, phen_file_test, true_signal_file, estimate_file, r1_file,
        cov_estimate_file, cov_file, cov_file_test;
    std::string run_mode = "infere", out_dir, out_name, model = "linear", pval_method = "se";
    double stop_criteria_thr = 0.01, merge_vars_thr = 5e-1, EM_err_thr = 1e-2;
    unsigned int EM_max_iter = 1, CG_max_iter = 500;
    double CG_err_tol = 1e-5;
    unsigned int Mt = 0, N = 0, N_test = 0, Mt_test = 0, num_mix_comp = 10, learn_vars = 1, learn_prior_delay = 1;
    double alpha_scale = 1.0;
    unsigned int C = 0;
    double probit_var = 1, rho = 0.5, h2 = 0.5, gam1 = 1e-6;
    int verbosity = 0;
    unsigned int iterations = 50;
    std::vector<double> vars{0, 1e-06, 6e-06, 3e-05, 2e-04, 1e-03, 6e-03, 3e-02, 2e-01, 1e+00};
    std::vector<double> probs{9.90000e-01, 5.00000e-03, 2.50000e-03, 1.25000e-03, 6.25000e-04,
                              3.12500e-04, 1.56250e-04, 7.81250e-05, 3.90625e-05, 3.90625e-05};
    std::vector<int> test_iter_range{1, 50};
    // additions
    unsigned long long seed = 0;
    int gpus = 1;
    int probes = 1;                     // --probes P: Hutchinson probes per iteration (1 = the reference)
    int checkpoint_every = 0;           // --checkpoint-every n: write {out}_checkpoint_it_{k}.bin after every n-th iteration
    std::string resume_from;            // --resume-from file: continue a run from such a checkpoint
    bool probit_entry = false;          // entered through main_meth_probit: model forced to bin_class, probit `test` / `predict` run modes
    std::string schedule = "onepass";   // onepass | recycled | fused | plain | reference (vampomi_solver_config::fuse_passes / redundant_passes)
    std::string storage = "f64";     // "f32": hold the marker block rounded to FP32 in HBM (arithmetic stays FP64)
    std::string missing = "none";    // "mean": replace every NaN of a marker column by the mean of its other entries (vampomi_impute_missing)

    // Parses argv. On error prints the reference's FATAL line to stdout and returns false (caller exits 1).
    // `echo` receives the "ardyh command line options" block the reference prints from rank 0.
    bool parse(int argc, char** argv, std::string* echo);
};

}  // namespace vampomi_host
