#include "io.h"
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <numeric>
#include <stdexcept>
#include <algorithm>
#include <system_error>
#include <thread>
#include <vector>
#include "../rng.h"

namespace vampomi_host {

bool read_phen(const std::string& path, bool standardize, std::vector<double>* out) {
    std::ifstream in(path);
    if (!in.is_open()) {
        std::cout << "FATAL: could not open phenotype file: " << path << std::endl;      // src/data.cpp:107
        return false;
    }
    out->clear();
    std::string line;
    double sum = 0.0;
    while (std::getline(in, line)) {
        // tokens separated by runs of whitespace; a leading run yields an empty first token (regex split semantics)
        std::vector<std::string> tok;
        size_t i = 0, n = line.size();
        std::string cur;
        bool in_ws = false;
        for (i = 0; i < n; i++) {
            char ch = line[i];
            bool ws = ch == ' ' || ch == '\t' || ch == '\r' || ch == '\f' || ch == '\v' || ch == '\n';
            if (ws) {
                if (!in_ws) { tok.push_back(cur); cur.clear(); in_ws = true; }
            } else { cur.push_back(ch); in_ws = false; }
        }
        if (!in_ws) tok.push_back(cur);
        if (tok.size() < 3) throw std::runtime_error("phenotype line with fewer than 3 columns");
        if (tok[2] == "NA") throw std::runtime_error("NAN in data!");
        double v = atof(tok[2].c_str());
        out->push_back(v);
        sum += v;
    }
    if (standardize && out->size() > 1) {
        const double nn = (double)out->size();
        const double avg = sum / nn;
        double sqn = 0.0;
        for (double v : *out) sqn += (v - avg) * (v - avg);
        sqn = std::sqrt((nn - 1.0) / sqn);
        for (double& v : *out) v *= sqn;
    }
    return true;
}

std::vector<double> read_vec(const std::string& path, long long M, long long S, bool* ok) {
    std::vector<double> v((size_t)M, 0.0);
    if (ok) *ok = false;
    int fd = ::open(path.c_str(), O_RDONLY);
    if (fd < 0) return v;
    size_t want = (size_t)M * sizeof(double), got = 0;
    while (got < want) {
        ssize_t r = pread(fd, (char*)v.data() + got, want - got, (off_t)(S * 8 + (long long)got));
        if (r <= 0) break;
        got += (size_t)r;
    }
    ::close(fd);
    if (ok) *ok = got == want;
    return v;
}

bool store_vec(const std::string& path, const double* v, long long M, long long S) {
    int fd = ::open(path.c_str(), O_WRONLY | O_CREAT, 0644);
    if (fd < 0) return false;
    size_t want = (size_t)M * sizeof(double), done = 0;
    while (done < want) {
        ssize_t r = pwrite(fd, (const char*)v + done, want - done, (off_t)(S * 8 + (long long)done));
        if (r <= 0) break;
        done += (size_t)r;
    }
    ::close(fd);
    return done == want;
}

bool CsvFile::open(const std::string& path, bool keep_existing) {
    close();
    if (keep_existing) {
        fd_ = ::open(path.c_str(), O_WRONLY | O_CREAT, 0644);
        return fd_ >= 0;
    }
    unlink(path.c_str());
    fd_ = ::open(path.c_str(), O_WRONLY | O_CREAT | O_EXCL, 0644);
    return fd_ >= 0;
}
void CsvFile::close() {
    if (fd_ >= 0) ::close(fd_);
    fd_ = -1;
}
void CsvFile::header(const std::vector<std::string>& names) {
    if (fd_ < 0 || names.empty()) return;
    std::string s = names[0];
    for (size_t i = 1; i < names.size(); i++) s += ", " + names[i];
    s += "\n";
    if (pwrite(fd_, s.data(), s.size(), 0) < 0) perror("csv header");
}
std::string CsvFile::format_row(unsigned it, const std::vector<double>& values) {
    char buf[64];
    snprintf(buf, sizeof buf, "%5d", it);                                       // src/utilities.cpp:372
    std::string s = buf;
    for (double v : values) {
        char b2[400];
        snprintf(b2, sizeof b2, ", %20.15f", v);                                // :376
        s += b2;
    }
    s += "\n";
    return s;
}
void CsvFile::row(unsigned it, const std::vector<double>& values) {
    if (fd_ < 0) return;
    std::string s = format_row(it, values);
    if (pwrite(fd_, s.data(), s.size(), (off_t)((size_t)it * s.size())) < 0) perror("csv row");   // :383
}

// ---- Student t upper tail through the regularised incomplete beta function (continued fraction, DLMF 8.17.22) ----
namespace {
double betacf(double a, double b, double x) {
    const double tiny = 1e-300, eps = 1e-16;
    const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
    double c = 1.0, d = 1.0 - qab * x / qap;
    if (std::fabs(d) < tiny) d = tiny;
    d = 1.0 / d;
    double h = d;
    for (int m = 1; m <= 20000; m++) {
        const int m2 = 2 * m;
        double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
        d = 1.0 + aa * d; if (std::fabs(d) < tiny) d = tiny;
        c = 1.0 + aa / c; if (std::fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        h *= d * c;
        aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
        d = 1.0 + aa * d; if (std::fabs(d) < tiny) d = tiny;
        c = 1.0 + aa / c; if (std::fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (std::fabs(del - 1.0) < eps) break;
    }
    return h;
}
// ln(Gamma(a+b) / (Gamma(a) Gamma(b))): one (a, b) serves every marker of a run (a = (N-2)/2, b = 1/2), so the last pair is kept
// per thread; lgamma_r because std::lgamma writes the global signgam and the markers are spread over threads (loo_pvals)
double ln_inv_beta(double a, double b) {
    thread_local double ka = -1.0, kb = -1.0, kv = 0.0;
    if (a != ka || b != kb) {
        int sg;
        kv = lgamma_r(a + b, &sg) - lgamma_r(a, &sg) - lgamma_r(b, &sg);
        ka = a; kb = b;
    }
    return kv;
}
double ibeta(double a, double b, double x) {
    if (x <= 0.0) return 0.0;
    if (x >= 1.0) return 1.0;
    const double lnbt = ln_inv_beta(a, b) + a * std::log(x) + b * std::log1p(-x);
    const double bt = std::exp(lnbt);
    if (x < (a + 1.0) / (a + b + 2.0)) return bt * betacf(a, b, x) / a;
    return 1.0 - bt * betacf(b, a, 1.0 - x) / b;
}
}  // namespace

double students_t_two_sided(double t, double dof) {
    if (std::isnan(t)) return t;
    const double x = dof / (dof + t * t);
    return ibeta(0.5 * dof, 0.5, x);            // = 2 * (I_x(v/2, 1/2) / 2)
}

double linear_reg1d_pvals(double sumx, double sumsqx, double sumxy, double sumy, double sumsqy, int n) {
    const double s2y = (sumsqy - sumy * sumy / n) / (n - 1);
    const double s2x = (sumsqx - sumx * sumx / n) / (n - 1);
    const double sxy = (sumxy - sumx * sumy / n) / (n - 1);
    // A variance below the formula's resolution comes out as rounding residue, zero or negative: such a column (or phenotype)
    // explains nothing, p = 1. Residue over residue can also give |r| > 1, clamped to a perfect fit. A NaN fails every
    // comparison and stays NaN.
    if (s2x <= 0 || s2y <= 0 || s2x * s2y == 0) return 1.0;
    double rxy = sxy / std::sqrt(s2x * s2y);
    if (rxy > 1.0) rxy = 1.0;
    if (rxy < -1.0) rxy = -1.0;
    const double t = rxy * std::sqrt((n - 2) / (1 - rxy * rxy));
    return students_t_two_sided(t > 0 ? t : (0 - t), (double)(n - 2));
}

void loo_pvals(const double* x1, const double* sums, double sw, double sww, int N, long long M, double* pvals, int threads,
               const unsigned char* constant) {
    const double sqrtN = std::sqrt((double)N);
    auto work = [&](long long j0, long long j1) {
        for (long long j = j0; j < j1; j++) {
            if (constant != nullptr && constant[j]) { pvals[j] = 1.0; continue; }      // DESIGN §4
            // y_mark = y_mod + x * c, c = x1_hat[j]/sqrt(N) (src/data.cpp:404-405): its sums follow from those of x and y_mod
            const double c = x1[j] / sqrtN, sx = sums[3 * j], sxx = sums[3 * j + 1], sxw = sums[3 * j + 2];
            const double sumy = sw + c * sx, sumxy = sxw + c * sxx, sumsqy = sww + 2 * c * sxw + c * c * sxx;
            pvals[j] = linear_reg1d_pvals(sx, sxx, sumxy, sumy, sumsqy, N);                    // src/data.cpp:414
        }
    };
    if (threads <= 0) threads = (int)std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency()), 32u);
    const long long per = 4096;                              // markers are independent: any split gives the same bits
    threads = (int)std::min<long long>(threads, (M + per - 1) / per);
    if (threads <= 1) { work(0, M); return; }
    std::vector<std::thread> pool;
    const long long chunk = (M + threads - 1) / threads;
    for (int t = 0; t < threads; t++) {
        const long long j0 = t * chunk, j1 = std::min(M, j0 + chunk);
        if (j0 >= j1) continue;
        try { pool.emplace_back(work, j0, j1); }
        catch (const std::system_error&) { work(j0, j1); }   // no more threads to be had: this block on the calling thread
    }
    for (auto& th : pool) th.join();
}

double calc_stdev(const std::vector<double>& v) {
    const double sum = std::accumulate(v.begin(), v.end(), 0.0);
    const double sq = std::inner_product(v.begin(), v.end(), v.begin(), 0.0);
    const int n = (int)v.size();
    const double mean = sum / n;
    return std::sqrt((sq - n * mean * mean) / (n - 1));
}

double normal_cdf(double v) { return 0.5 * std::erfc(-v * M_SQRT1_2); }

std::vector<double> probit_p1(unsigned long long seed, int N) {
    std::vector<double> p((size_t)N);
    for (int i = 0; i < N; i++)
        p[i] = vampomi::normal_from_hash(vampomi::hash3(seed, vampomi::STREAM_P1, (uint64_t)i, 0));
    return p;
}

}  // namespace vampomi_host
