#include "options.h"
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <sstream>

namespace vampomi_host {

namespace {
std::vector<double> parse_list(const std::string& s) {
    std::vector<double> out;
    std::stringstream ss(s);
    std::string tok;
    while (std::getline(ss, tok, ',')) out.push_back(atof(tok.c_str()));
    return out;
}
}  // namespace

bool Options::parse(int argc, char** argv, std::string* echo) {
    std::stringstream ss;
    ss << "\nardyh command line options:\n";                                   // src/options.cpp:19
    struct StrOpt { const char* flag; std::string* dst; };
    const StrOpt str_opts[] = {
        {"--meth-file", &meth_file}, {"--cov-file", &cov_file}, {"--cov-file-test", &cov_file_test},
        {"--meth-file-test", &meth_file_test}, {"--estimate-file", &estimate_file}, {"--r1-file", &r1_file},
        {"--cov-estimate-file", &cov_estimate_file}, {"--run-mode", &run_mode}, {"--phen-file", &phen_file},
        {"--true-signal-file", &true_signal_file}, {"--phen-file-test", &phen_file_test}, {"--out-dir", &out_dir},
        {"--out-name", &out_name}, {"--model", &model}, {"--pval-method", &pval_method},
    };
    struct DblOpt { const char* flag; double* dst; };
    const DblOpt dbl_opts[] = {
        {"--stop-criteria-thr", &stop_criteria_thr}, {"--merge-vars-thr", &merge_vars_thr}, {"--EM-err-thr", &EM_err_thr},
        {"--alpha-scale", &alpha_scale}, {"--rho", &rho}, {"--probit-var", &probit_var}, {"--h2", &h2}, {"--gam1", &gam1},
        {"--CG-err-tol", &CG_err_tol},
    };
    // {flag, destination, minimum accepted value, wording of the reference's complaint}
    struct UIntOpt { const char* flag; unsigned int* dst; int min; const char* name_in_msg; };
    const UIntOpt uint_opts[] = {
        {"--learn-vars", &learn_vars, 0, "--learn-vars"}, {"--learn-prior-delay", &learn_prior_delay, 0, "--learn-prior-delay"},
        {"--iterations", &iterations, 1, "--iterations"}, {"--num-mix-comp", &num_mix_comp, 1, "--num-mix-comp"},
        {"--EM-max-iter", &EM_max_iter, 1, "--EM-max-iter"}, {"--Mt", &Mt, 1, "--Mt"}, {"--C", &C, 0, "--C"},
        {"--N", &N, 1, "--N"}, {"--N-test", &N_test, 1, "--N_test"}, {"--Mt-test", &Mt_test, 1, "--Mt_test"},
        {"--CG-max-iter", &CG_max_iter, 1, "--CG-max-iter"},
    };

    for (int i = 1; i < argc; ++i) {
        const char* a = argv[i];
        auto need_value = [&]() -> bool {
            if (i == argc - 1) {                                                 // src/options.cpp:293-296
                std::cout << "FATAL  : missing argument for last option \"" << a
                          << "\". Please check your input and relaunch." << std::endl;
                return false;
            }
            return true;
        };
        bool matched = false;
        for (const auto& o : str_opts)
            if (!strcmp(a, o.flag)) {
                if (!need_value()) return false;
                *o.dst = argv[++i];
                ss << o.flag << " " << *o.dst << "\n";
                matched = true;
                break;
            }
        if (matched) continue;
        for (const auto& o : dbl_opts)
            if (!strcmp(a, o.flag)) {
                if (!need_value()) return false;
                *o.dst = atof(argv[++i]);
                ss << o.flag << (strcmp(o.flag, "--probit-var") ? " " : "") << *o.dst << "\n";   // sic, src/options.cpp:199
                matched = true;
                break;
            }
        if (matched) continue;
        for (const auto& o : uint_opts)
            if (!strcmp(a, o.flag)) {
                if (!need_value()) return false;
                if (atoi(argv[i + 1]) < o.min) {                                 // e.g. src/options.cpp:140-143
                    std::cout << "FATAL  : option " << o.name_in_msg << " has to be a "
                              << (o.min == 0 ? "non-negative" : "strictly positive") << " integer! (" << argv[i + 1]
                              << " was passed)" << std::endl;
                    return false;
                }
                *o.dst = (unsigned int)atoi(argv[++i]);
                ss << o.flag << " " << *o.dst << "\n";
                matched = true;
                break;
            }
        if (matched) continue;
        if (!strcmp(a, "--vars") || !strcmp(a, "--probs")) {
            if (!need_value()) return false;
            std::string list = argv[++i];
            ss << a << " " << list << "\n";
            (!strcmp(a, "--vars") ? vars : probs) = parse_list(list);
        } else if (!strcmp(a, "--test-iter-range")) {
            if (!need_value()) return false;
            std::string list = argv[++i];
            ss << "--test-iter-range " << list << "\n";
            std::vector<double> v = parse_list(list);
            for (size_t k = 0; k < v.size() && k < 2; k++) test_iter_range[k] = (int)v[k];
        } else if (!strcmp(a, "--verbosity")) {
            if (!need_value()) return false;
            verbosity = atoi(argv[++i]);
            ss << "--verbosity " << verbosity << "\n";
        } else if (!strcmp(a, "--seed")) {
            if (!need_value()) return false;
            seed = strtoull(argv[++i], nullptr, 10);
            ss << "--seed " << seed << "\n";
        } else if (!strcmp(a, "--storage")) {
            if (!need_value()) return false;
            storage = argv[++i];
            if (storage != "f64" && storage != "f32") {
                std::cout << "FATAL  : option --storage has to be f64 or f32! (" << storage << " was passed)" << std::endl;
                return false;
            }
            ss << "--storage " << storage << "\n";
        } else if (!strcmp(a, "--missing")) {
            if (!need_value()) return false;
            missing = argv[++i];
            if (missing != "none" && missing != "mean") {
                std::cout << "FATAL  : option --missing has to be none or mean! (" << missing << " was passed)" << std::endl;
                return false;
            }
            ss << "--missing " << missing << "\n";
        } else if (!strcmp(a, "--schedule")) {
            if (!need_value()) return false;
            schedule = argv[++i];
            if (schedule != "fused" && schedule != "plain" && schedule != "reference" && schedule != "recycled" && schedule != "onepass") {
                std::cout << "FATAL  : option --schedule has to be onepass, recycled, fused, plain or reference! (" << schedule << " was passed)" << std::endl;
                return false;
            }
            ss << "--schedule " << schedule << "\n";
        } else if (!strcmp(a, "--probes") || !strcmp(a, "--checkpoint-every")) {
            if (!need_value()) return false;
            const int v = atoi(argv[++i]);
            if (v < (a[2] == 'p' ? 1 : 0)) {
                std::cout << "FATAL  : option " << a << " has to be a " << (a[2] == 'p' ? "strictly positive" : "non-negative") << " integer! (" << argv[i] << " was passed)" << std::endl;
                return false;
            }
            (a[2] == 'p' ? probes : checkpoint_every) = v;
            ss << a << " " << v << "\n";
        } else if (!strcmp(a, "--resume-from")) {
            if (!need_value()) return false;
            resume_from = argv[++i];
            ss << "--resume-from " << resume_from << "\n";
        } else if (!strcmp(a, "--gpus")) {
            if (!need_value()) return false;
            gpus = atoi(argv[++i]);
            if (gpus < 1) {
                std::cout << "FATAL  : option --gpus has to be a strictly positive integer! (" << argv[i] << " was passed)" << std::endl;
                return false;
            }
            ss << "--gpus " << gpus << "\n";
        } else {
            std::cout << "FATAL: option \"" << a << "\" unknown\n";             // src/options.cpp:283
            return false;
        }
    }
    if (run_mode == "inference") run_mode = "infere";   // BASELINE.json spells it out; the reference's string is "infere"
    if (meth_file.empty() && meth_file_test.empty()) {                           // src/options.cpp:299-303
        std::cout << "FATAL  : no meth file provided! Please use the --meth-file option." << std::endl;
        return false;
    }
    if (echo) *echo = ss.str();
    return true;
}

}  // namespace vampomi_host
