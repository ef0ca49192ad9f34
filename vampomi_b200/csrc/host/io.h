// Host-side file formats and special functions of the reference's driver (no GPU work here).
#pragma once
#include <string>
#include <vector>

namespace vampomi_host {

// PLINK-style phenotype file: third whitespace token of each line (src/data.cpp:58-110). When `standardize`, the values
// are scaled by sqrt((n-1)/sum((y-mean)^2)) and NOT centred (:97-99). Returns false with the reference's FATAL line
// printed if the file cannot be opened; throws std::runtime_error("NAN in data!") on an NA value (:73-74).
bool read_phen(const std::string& path, bool standardize, std::vector<double>* out);

// M doubles at byte offset S*8 (src/utilities.cpp:251-267). Like the reference, a missing file is not an error
// here: the vector stays zero. `ok` (optional) reports whether all bytes were read.
std::vector<double> read_vec(const std::string& path, long long M, long long S, bool* ok = nullptr);
// Raw FP64 at byte offset S*8, file created if needed and never truncated (src/utilities.cpp:241-249).
bool store_vec(const std::string& path, const double* v, long long M, long long S);

// CSV files written at computed offsets (src/utilities.cpp:366-401): header at 0, row of iteration `it` at
// it*strlen(row). Created fresh (delete + O_EXCL, src/vamp.cpp:857-863).
class CsvFile {
public:
    CsvFile() = default;
    ~CsvFile() { close(); }
    bool open(const std::string& path, bool keep_existing = false);   // keep_existing: resume — rows land at their usual offsets
    void header(const std::vector<std::string>& names);
    void row(unsigned it, const std::vector<double>& values);
    void close();
    static std::string format_row(unsigned it, const std::vector<double>& values);
private:
    int fd_ = -1;
};

// 2 * P(T_{n-2} > |t|): boost::math::cdf(complement(students_t(n-2), |t|)) * 2 of src/utilities.cpp:277-279.
double students_t_two_sided(double t, double dof);
// src/utilities.cpp:269-282; a variance that rounds to <= 0 gives 1 and |r| > 1 is clamped, so that no NaN comes out of a column
// without NaN
double linear_reg1d_pvals(double sumx, double sumsqx, double sumxy, double sumy, double sumsqy, int n);
// data::pvals_loo's per-marker tail (src/data.cpp:400-414) for M markers from the three streamed sums per raw column (sum x, sum x^2,
// sum x*y_mod; vampomi_loo_sums), the scaled estimate x1 (x1_hat * sqrt(N)) and sum / sum of squares of y_mod, spread over host
// threads (0 = all hardware threads, at most 32). `constant` (optional): the columns k_stats found constant
// (vampomi_constant_columns), which get p = 1 exactly.
void loo_pvals(const double* x1, const double* sums, double sw, double sww, int N, long long M, double* pvals, int threads = 0,
               const unsigned char* constant = nullptr);
// src/utilities.cpp:183-205 with sync = 0
double calc_stdev(const std::vector<double>& v);
// src/utilities.cpp:284-287
double normal_cdf(double v);
// Deterministic N(0,1) probit start (oracle patch P3 of src/vamp_probit.cpp:53)
std::vector<double> probit_p1(unsigned long long seed, int N);

}  // namespace vampomi_host
