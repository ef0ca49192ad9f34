// Elementwise + reduction kernels over the M-length (sharded) and N-length (replicated) vectors of the VAMP loop.
// They move megabytes, not gigabytes — what matters here is (1) the arithmetic follows the reference's formulas
// operation by operation (parity 1e-9), (2) every reduction is bitwise reproducible: per-block partials are
// combined by the last block to finish, in a fixed order, and (3) scalars stay on the device (CG) or come back
// to the host in ONE packed copy per step.
#include <float.h>
#include <math_constants.h>
#include "common.h"
#include "rng.h"
#include "xchg.cuh"

namespace vampomi {

__device__ __forceinline__ double warp_sum_v(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sums K per-thread values over the whole grid. `partials` is [gridDim.x][K], `ticket` a zero-initialised counter
// that this routine leaves at zero again. Result lands in out[0..K) (written by the last block only). With `x` enabled
// the last block also sums over the GPUs of the job through peer memory (xchg.cuh) before writing out[].
__device__ void grid_reduce(const double* v, int K, double* __restrict__ partials, unsigned int* ticket, double* out,
                            const Xchg* x = nullptr) {
    __shared__ double sm[RED_THREADS / 32][MAX_SUMS];
    __shared__ double fin[MAX_SUMS];
    __shared__ bool is_last;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    for (int k = 0; k < K; k++) {
        double s = warp_sum_v(v[k]);
        if (lane == 0) sm[wid][k] = s;
    }
    __syncthreads();
    if (tid < K) {
        double t = sm[0][tid];
#pragma unroll
        for (int w = 1; w < RED_THREADS / 32; w++) t += sm[w][tid];
        partials[(size_t)blockIdx.x * K + tid] = t;
        __threadfence();
    }
    __syncthreads();
    if (tid == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    for (int k = 0; k < K; k++) {
        double t = 0.0;
        for (unsigned b = tid; b < gridDim.x; b += RED_THREADS) t += __ldcg(partials + (size_t)b * K + k);
        t = warp_sum_v(t);
        __syncthreads();
        if (lane == 0) sm[wid][0] = t;
        __syncthreads();
        if (tid == 0) {
            double r = sm[0][0];
#pragma unroll
            for (int w = 1; w < RED_THREADS / 32; w++) r += sm[w][0];
            fin[k] = r;
        }
    }
    __syncthreads();
    if (x != nullptr && x->enabled) xchg_allreduce_scalars(*x, fin, K, out);
    else if (tid < K) out[tid] = fin[tid];
    if (tid == 0) *ticket = 0u;
}

static inline int vec_blocks(long long n) {
    long long b = (n + RED_THREADS - 1) / RED_THREADS;
    if (b > RED_BLOCKS) b = RED_BLOCKS;
    return b < 1 ? 1 : (int)b;
}

#define GRID_STRIDE(i, n) \
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (long long)gridDim.x * blockDim.x)

// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(RED_THREADS) k_fill(double* __restrict__ dst, long long n, double v) {
    GRID_STRIDE(i, n) dst[i] = v;
}
int launch_fill(vampomi_ctx* c, double* dst, long long n, double v) {
    k_fill<<<vec_blocks(n), RED_THREADS, 0, c->stream>>>(dst, n, v);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}

// dst = (a*x + b*y) / cdiv, evaluated as the reference writes its message updates, e.g. src/vamp.cpp:260:
//   r2[i] = (eta1 * x1_hat[i] - gam1 * r1[i]) / gam2
__global__ void __launch_bounds__(RED_THREADS) k_lincomb(double* __restrict__ dst, double a, const double* __restrict__ x, double b,
                                                         const double* __restrict__ y, double cdiv, long long n) {
    GRID_STRIDE(i, n) dst[i] = (a * x[i] + b * y[i]) / cdiv;
}
int launch_lincomb(vampomi_ctx* c, double* dst, double a, const double* x, double b, const double* y, double cdiv, long long n) {
    k_lincomb<<<vec_blocks(n), RED_THREADS, 0, c->stream>>>(dst, a, x, b, y, cdiv, n);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// batched reductions: blockIdx.y selects the item
// ---------------------------------------------------------------------------------------------------------------
struct DotBatch {
    int n;
    int kind[MAX_DOTS];
    const double* a[MAX_DOTS];
    const double* b[MAX_DOTS];
    long long len[MAX_DOTS];
    double scale[MAX_DOTS];
};

__global__ void __launch_bounds__(RED_THREADS) k_dots(DotBatch batch, double* __restrict__ partials, unsigned int* tickets,
                                                      double* __restrict__ out) {
    const int it = blockIdx.y;
    const double* __restrict__ a = batch.a[it];
    const double* __restrict__ b = batch.b[it];
    const long long n = batch.len[it];
    const int kind = batch.kind[it];
    const double s = batch.scale[it];
    double acc = 0.0;
    if (kind == VAMPOMI_DOT) {
        GRID_STRIDE(i, n) acc = fma(a[i], b[i], acc);
    } else if (kind == VAMPOMI_DIFF2) {
        GRID_STRIDE(i, n) { double d = a[i] - b[i]; acc = fma(d, d, acc); }
    } else {
        GRID_STRIDE(i, n) { double d = a[i] - s * b[i]; acc = fma(d, d, acc); }
    }
    grid_reduce(&acc, 1, partials + (size_t)it * RED_BLOCKS, tickets + it, out + it);
}

int launch_dots(vampomi_ctx* c, int n, const int* kind, const double* const* a, const double* const* b, const long long* len,
                const double* scale, double* sums_dev) {
    DotBatch batch;
    batch.n = n;
    long long maxlen = 1;
    for (int i = 0; i < n; i++) {
        batch.kind[i] = kind[i]; batch.a[i] = a[i]; batch.b[i] = b[i]; batch.len[i] = len[i];
        batch.scale[i] = scale ? scale[i] : 1.0;
        if (len[i] > maxlen) maxlen = len[i];
    }
    dim3 grid(vec_blocks(maxlen), n);
    k_dots<<<grid, RED_THREADS, 0, c->stream>>>(batch, c->red_partials, c->red_tickets, sums_dev);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}

// The per-iteration packed sums outside the CG loop (denoiser, EM, metrics): summed over the GPUs by ONE small block through
// the same peer-memory exchange as the CG scalars, instead of an ncclAllReduce (~4 of them per VAMP iteration).
__global__ void __launch_bounds__(64) k_xchg_sums(double* __restrict__ sums, int n, Xchg xc) {
    __shared__ double v[XCHG_SCALARS];
    if ((int)threadIdx.x < n) v[threadIdx.x] = sums[threadIdx.x];
    __syncthreads();
    xchg_allreduce_scalars(xc, v, n, sums);
}
int launch_xchg_sums(vampomi_ctx* c, double* sums_dev, int n) {
    k_xchg_sums<<<1, 64, 0, c->stream>>>(sums_dev, n, c->xchg);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Hutchinson probe
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(RED_THREADS) k_probe(double* __restrict__ bern, long long M, long long S, uint64_t seed, int it,
                                                       double inv_sqrt_Mt_denom) {
    GRID_STRIDE(j, M) bern[j] = probe_sign(seed, it, (uint64_t)(S + j)) / inv_sqrt_Mt_denom;   // (2*bern-1)/sqrt(Mt), src/vamp.cpp:296
}
int launch_probe(vampomi_ctx* c, uint64_t seed, int it) {
    k_probe<<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(c->mvec[VAMPOMI_V_BERN], c->M, c->S, seed, it, sqrt((double)c->Mt));
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Gaussian-mixture denoiser: g1 (src/vamp.cpp:440-463), g1d (:465-492), damping (:208-211), sum of g1d (:214-219)
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(RED_THREADS) k_denoise(const double* __restrict__ r1, double* __restrict__ x1,
                                                         double* __restrict__ x1_prev, long long M, double gam1, MixParams mp,
                                                         int damp, double rho, double* __restrict__ partials,
                                                         unsigned int* ticket, double* __restrict__ out) {
    const double sigma = 1.0 / gam1;
    double eta_max = mp.vars[0];
    for (int l = 1; l < mp.L; l++) eta_max = fmax(eta_max, mp.vars[l]);
    const bool degenerate = (sigma < 1e-10 && sigma > -1e-10);
    double sum_d = 0.0;
    GRID_STRIDE(i, M) {
        const double y = r1[i];
        double g, gd;
        if (degenerate) {
            g = y; gd = 1.0;
        } else {
            double pk = 0.0, pkd = 0.0, pkdd = 0.0;
            for (int l = 0; l < mp.L; l++) {
                const double vs = mp.vars[l] + sigma;
                const double expe_sum = -0.5 * (y * y) * (eta_max - mp.vars[l]) / vs / (eta_max + sigma);
                const double e = exp(expe_sum);
                double z = mp.probs[l] / sqrt(vs) * e;
                pk = pk + z;
                z = z / vs * y;
                pkd = pkd - z;
                const double z2 = z / vs * y;
                pkdd = pkdd - mp.probs[l] / pow(vs, 1.5) * e + z2;
            }
            g = y + sigma * pkd / pk;
            const double q = pkd / pk;
            gd = 1.0 + sigma * (pkdd / pk - q * q);
        }
        const double prev = x1[i];
        x1_prev[i] = prev;
        x1[i] = damp ? rho * g + (1.0 - rho) * prev : g;
        sum_d += gd;
    }
    grid_reduce(&sum_d, 1, partials, ticket, out);
}

int launch_denoise(vampomi_ctx* c, double gam1, const MixParams& mp, int damp, double rho, double* sums_dev) {
    k_denoise<<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(c->mvec[VAMPOMI_V_R1], c->mvec[VAMPOMI_V_X1], c->mvec[VAMPOMI_V_X1_PREV],
                                                              c->M, gam1, mp, damp, rho, c->red_partials, c->red_tickets, sums_dev);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// EM sums (src/vamp.cpp:554-597). mp.probs carries omegas. 2L-1 accumulators per thread.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(RED_THREADS) k_em_sums(const double* __restrict__ r1, long long M, double gam1, double lambda,
                                                         MixParams mp, double* __restrict__ partials, unsigned int* ticket,
                                                         double* __restrict__ out) {
    const int L = mp.L;
    const double noise_var = 1.0 / gam1;
    double max_sigma = mp.vars[0];
    for (int l = 1; l < L; l++) max_sigma = fmax(max_sigma, mp.vars[l]);
    const double two_pi = 2.0 * 3.14159265358979323846;
    double acc[2 * MAX_MIX];
    for (int k = 0; k < 2 * L - 1; k++) acc[k] = 0.0;
    double num[MAX_MIX], ng[MAX_MIX];
    GRID_STRIDE(i, M) {
        const double r = r1[i];
        const double r2h = (r * r) / 2.0;
        double tot = 0.0;
        for (int j = 1; j < L; j++) {
            const double vj = mp.vars[j];
            num[j] = lambda * mp.probs[j] * exp(-r2h * (max_sigma - vj) / (vj + noise_var) / (max_sigma + noise_var))
                     / sqrt(vj + noise_var) / sqrt(two_pi);
            ng[j] = gam1 * r / (1.0 / vj + gam1);
            tot += num[j];
        }
        const double pin = 1.0 / (1.0 + (1.0 - lambda) / sqrt(two_pi * noise_var)
                                        * exp(-r2h * max_sigma / noise_var / (noise_var + max_sigma)) / tot);
        acc[0] += pin;
        for (int j = 1; j < L; j++) {
            const double beta = num[j] / tot;
            const double v = 1.0 / (1.0 / mp.vars[j] + gam1);
            const double gm = beta * (ng[j] * ng[j] + v);
            acc[j] += beta * pin;
            acc[L - 1 + j] += gm * pin;
        }
    }
    grid_reduce(acc, 2 * L - 1, partials, ticket, out);
}

int launch_em_sums(vampomi_ctx* c, double gam1, double lambda, const MixParams& mp, double* sums_dev) {
    k_em_sums<<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(c->mvec[VAMPOMI_V_R1], c->M, gam1, lambda, mp, c->red_partials,
                                                              c->red_tickets, sums_dev);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// probit z-channel (src/vamp_probit.cpp:469-488); erfcx with the reference's clamps (src/utilities.cpp:295-298)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double erfcx_ref(double x) {
    if (x < -10.0) return CUDART_INF;
    if (x > 10.0) return -DBL_MAX;           // numeric_limits<double>::lowest() (sic)
    return erfcx(x);
}

__global__ void __launch_bounds__(RED_THREADS) k_probit_z(const double* __restrict__ p1, const double* __restrict__ y, const double* __restrict__ mcov,
                                                          double* __restrict__ z1hat, long long N, double tau1,
                                                          double* __restrict__ partials, unsigned int* ticket,
                                                          double* __restrict__ out) {
    const double probit_var = 1.0;           // src/vamp.hpp:35
    const double sroot = sqrt(probit_var + 1.0 / tau1);
    double sum_d = 0.0;
    GRID_STRIDE(i, N) {
        const double p = p1[i], s = 2.0 * y[i] - 1.0;
        const double cc = (p + mcov[i]) / sroot;                               // m_cov = Z cov_eff, 0 without covariates (:471,:482)
        const double ratio = 2.0 / sqrt(2.0 * 3.14159265358979323846) / erfcx_ref(-s * cc / sqrt(2.0));
        z1hat[i] = p + s * ratio / tau1 / sroot;
        sum_d += 1.0 - ratio / (1.0 + tau1 * probit_var) * (s * cc + ratio);
    }
    grid_reduce(&sum_d, 1, partials, ticket, out);
}

int launch_probit_z(vampomi_ctx* c, double tau1, double* sums_dev) {
    k_probit_z<<<vec_blocks(c->N), RED_THREADS, 0, c->stream>>>(c->nvec[VAMPOMI_V_P1 - 32], c->nvec[VAMPOMI_V_Y - 32], c->nvec[VAMPOMI_V_MCOV - 32],
                                                               c->nvec[VAMPOMI_V_Z1HAT - 32], c->N, tau1, c->red_partials,
                                                               c->red_tickets, sums_dev);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}

// se p-values (src/main_meth.cpp:233-239): the tail of normal(r1, sd) beyond 0, erfc(|r1| / (sd*sqrt(2))) / 2. The reference
// evaluates cdf(normal(r1, sd), 0) and flips it to 1 - cdf when r1 <= 0, which subtracts a number close to 1 from 1 for a
// negative effect: p loses its digits from 6 sd on and is 0 from 8.5 sd on. The tail taken directly keeps full precision for
// both signs (DESIGN §4); r1 = 0 still gives 0.5 and a NaN stays NaN.
__global__ void __launch_bounds__(RED_THREADS) k_pvals_se(const double* __restrict__ r1, long long M, double sd, double* __restrict__ out) {
    GRID_STRIDE(j, M) out[j] = 0.5 * erfc(fabs(r1[j]) / (sd * sqrt(2.0)));
}
int launch_pvals_se(vampomi_ctx* c, const double* r1_dev, double sd, double* out_dev) {
    k_pvals_se<<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(r1_dev, c->M, sd, out_dev);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Preconditioned CG vector steps (src/vamp.cpp:671-757). All scalars live in CgScalars on the device.
// Every kernel handles the S <= 2 systems of a batch (cg.cu: the LMMSE solve and the Onsager solve of one VAMP iteration
// share the operator and run in lock-step): one launch, one grid reduction and one cross-GPU exchange for all of them.
// A system whose done flag is set is skipped; the flags are identical on all GPUs, so the skips agree everywhere.
// Packed sums: sums[s] = <d,p>; sums[4 + 3s .. 4 + 3s + 2] = <v,mu>, <r,z>, <r,r> (init: sums[4 + 2s], [4 + 2s + 1] = <r,z>, <v,v>).
// ---------------------------------------------------------------------------------------------------------------
// r = v - (tau*AtA mu + gam2*mu) [warm] or r = v; z = r/diag; p = z   (:679-690)
template <int S>
__global__ void __launch_bounds__(RED_THREADS) k_cg_init(CgBatch b, long long M, int N, double tau, double gam2, double diag,
                                                         double* __restrict__ partials, unsigned int* ticket,
                                                         double* __restrict__ out, Xchg xc) {
    double acc[2 * S];
#pragma unroll
    for (int s = 0; s < S; s++) {
        const CgSys& q = b.s[s];
        double a0 = 0.0, a1 = 0.0;
        GRID_STRIDE(i, M) {
            const double vi = q.v[i];
            double ri;
            if (q.warm) {
                double res = q.atx_out[i] * tau;        // lmmse_mult, :656-659
                res += gam2 * q.mu[i];
                ri = vi - res;
            } else {
                q.mu[i] = 0.0;
                ri = vi;
            }
            const double zi = ri / diag;
            q.r[i] = ri; q.z[i] = zi; q.p[i] = zi;
            a0 = fma(ri, zi, a0);
            a1 = fma(vi, vi, a1);
        }
        if (q.amu != nullptr && !q.warm) GRID_STRIDE(i, N) q.amu[i] = 0.0;      // A mu_start of a zero start
        acc[2 * s] = a0; acc[2 * s + 1] = a1;
    }
    grid_reduce(acc, 2 * S, partials, ticket, out, &xc);
}

__global__ void k_cg_init_finish(CgBatch b, const double* __restrict__ sums) {
    const int s = threadIdx.x;
    if (s >= b.S) return;
    CgScalars* cg = b.s[s].cg;
    cg->rz[0] = sums[2 * s]; cg->rz[1] = sums[2 * s];
    cg->vv = sums[2 * s + 1];
    cg->prev_onsager[0] = 0.0; cg->prev_onsager[1] = 0.0;
    cg->rel_err = CUDART_NAN; cg->vmu = 0.0;
    cg->done = 0; cg->iters = 0;
}

// d = tau * AtA p + gam2 * p (lmmse_mult, :656-659); out[s] = <d,p>
template <int S>
__global__ void __launch_bounds__(RED_THREADS) k_cg_dp(CgBatch b, long long M, double tau, double gam2,
                                                       double* __restrict__ partials, unsigned int* ticket,
                                                       double* __restrict__ out, Xchg xc) {
    bool active[S], any = false;
#pragma unroll
    for (int s = 0; s < S; s++) { active[s] = b.s[s].cg->done == 0; any |= active[s]; }
    if (!any) return;
    double acc[S];
#pragma unroll
    for (int s = 0; s < S; s++) {
        const CgSys& q = b.s[s];
        double a = 0.0;
        if (active[s]) {
            GRID_STRIDE(i, M) {
                const double pi = q.p[i];
                double di = q.atx_out[i] * tau;
                di += gam2 * pi;
                q.d[i] = di;
                a = fma(di, pi, a);
            }
        }
        acc[s] = a;
    }
    grid_reduce(acc, S, partials, ticket, out, &xc);
}

// alpha = <r,z>/<d,p>; mu += alpha p; r -= alpha d; z = r/diag; out[3s..3s+2] = <v,mu>, <r,z>, <r,r>   (:701-706, :728-734)
// A system with `amu` also advances amu += alpha * (A p), so that amu stays A mu without a pass of its own.
// One-pass CG (gar != nullptr; kernels_gram.cu): tmpN holds q = A p and gw holds w = A A^T q, so A d = tau w + gam2 q and
// A r follows r: A r -= alpha * A d — the N-side image of r -= alpha d.
template <int S>
__global__ void __launch_bounds__(RED_THREADS) k_cg_step(CgBatch b, long long M, int N, double tau, double gam2, double diag, int parity,
                                                         const double* __restrict__ dp, double* __restrict__ partials,
                                                         unsigned int* ticket, double* __restrict__ out, Xchg xc) {
    bool active[S], any = false;
#pragma unroll
    for (int s = 0; s < S; s++) { active[s] = b.s[s].cg->done == 0; any |= active[s]; }
    if (!any) return;
    double acc[3 * S];
#pragma unroll
    for (int s = 0; s < S; s++) {
        const CgSys& q = b.s[s];
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;
        if (active[s]) {
            const double alpha = q.cg->rz[parity] / dp[s];
            GRID_STRIDE(i, M) {
                const double mui = q.mu[i] + alpha * q.p[i];
                const double ri = q.r[i] - q.d[i] * alpha;
                const double zi = ri / diag;
                q.mu[i] = mui; q.r[i] = ri; q.z[i] = zi;
                a0 = fma(q.v[i], mui, a0);
                a1 = fma(ri, zi, a1);
                a2 = fma(ri, ri, a2);
            }
            if (q.amu != nullptr) GRID_STRIDE(i, N) q.amu[i] += alpha * q.tmpN[i];
            if (q.gar != nullptr) GRID_STRIDE(i, N) {
                double adi = q.gw[i] * tau;
                adi += gam2 * q.tmpN[i];
                q.gar[i] -= adi * alpha;
            }
        }
        acc[3 * s] = a0; acc[3 * s + 1] = a1; acc[3 * s + 2] = a2;
    }
    grid_reduce(acc, 3 * S, partials, ticket, out, &xc);
}

// scalar logic of one CG iteration (:708-726 onsager test, :731-751 beta and residual test) + p = z + beta p (:738-739).
// Every block recomputes the scalars from read-only inputs (slot `parity`); block 0 publishes slot parity^1.
// cg->done is written by block 0 while later-scheduled blocks of the SAME launch may already read it at their entry: if they
// see it set they skip a p update that nothing will read any more (that solve is over), so the race is benign by construction.
// One-pass CG: q = A p follows p: q = (A r)/diag + beta q — the N-side image of p = z + beta p with z = r/diag.
template <int S>
__global__ void __launch_bounds__(RED_THREADS) k_cg_finish(CgBatch b, long long M, int N, int parity, double gam2, double diag, double tol,
                                                           int max_iter, const double* __restrict__ sums) {
#pragma unroll
    for (int s = 0; s < S; s++) {
        const CgSys& q = b.s[s];
        CgScalars* cg = q.cg;
        if (cg->done) continue;
        const double rz_old = cg->rz[parity];
        const double vmu = sums[3 * s], rz_new = sums[3 * s + 1], rr = sums[3 * s + 2];
        int done = 0;
        double prev_onsager = cg->prev_onsager[parity];
        if (q.onsager_mode) {
            const double onsager = gam2 * vmu;
            double rel = 1.0;
            if (onsager != 0.0) rel = fabs((onsager - prev_onsager) / onsager);
            if (rel < 1e-8) done = 1;
            prev_onsager = onsager;
        }
        double rel_err = CUDART_NAN;
        if (!done) {
            double beta = 1.0 / rz_old;                   // pow(<r,z>, -1), :731
            beta *= rz_new;                               // :736
            GRID_STRIDE(i, M) q.p[i] = q.z[i] + beta * q.p[i];
            if (q.gar != nullptr) GRID_STRIDE(i, N) q.tmpN[i] = q.gar[i] / diag + beta * q.tmpN[i];
            rel_err = sqrt(rr) / sqrt(cg->vv);            // :742-744
            if (rel_err < tol) done = 2;
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            const int iters = cg->iters + 1;
            if (!done && iters >= max_iter) done = 3;
            cg->rz[parity ^ 1] = rz_new;
            cg->prev_onsager[parity ^ 1] = prev_onsager;
            cg->rel_err = rel_err;
            cg->vmu = vmu;
            cg->iters = iters;
            __threadfence();
            cg->done = done;
        }
    }
}

int launch_cg_init(vampomi_ctx* c, const CgBatch& b, double tau, double gam2, double diag, double* sums_dev) {
    if (b.S == 1) k_cg_init<1><<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(b, c->M, c->N, tau, gam2, diag, c->red_partials, c->red_tickets, sums_dev, c->xchg);
    else k_cg_init<2><<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(b, c->M, c->N, tau, gam2, diag, c->red_partials, c->red_tickets, sums_dev, c->xchg);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}
int launch_cg_init_finish(vampomi_ctx* c, const CgBatch& b, const double* sums_dev) {
    k_cg_init_finish<<<1, 32, 0, c->stream>>>(b, sums_dev);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}
int launch_cg_dp(vampomi_ctx* c, const CgBatch& b, double tau, double gam2, double* sums_dev) {
    if (b.S == 1) k_cg_dp<1><<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(b, c->M, tau, gam2, c->red_partials, c->red_tickets, sums_dev, c->xchg);
    else k_cg_dp<2><<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(b, c->M, tau, gam2, c->red_partials, c->red_tickets, sums_dev, c->xchg);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}
int launch_cg_step(vampomi_ctx* c, const CgBatch& b, double tau, double gam2, double diag, int parity, const double* dp_dev, double* sums_dev) {
    if (b.S == 1) k_cg_step<1><<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(b, c->M, c->N, tau, gam2, diag, parity, dp_dev, c->red_partials, c->red_tickets, sums_dev, c->xchg);
    else k_cg_step<2><<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(b, c->M, c->N, tau, gam2, diag, parity, dp_dev, c->red_partials, c->red_tickets, sums_dev, c->xchg);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}
int launch_cg_finish(vampomi_ctx* c, const CgBatch& b, int parity, double gam2, double diag, double tol, int max_iter, const double* sums_dev) {
    if (b.S == 1) k_cg_finish<1><<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(b, c->M, c->N, parity, gam2, diag, tol, max_iter, sums_dev);
    else k_cg_finish<2><<<vec_blocks(c->M), RED_THREADS, 0, c->stream>>>(b, c->M, c->N, parity, gam2, diag, tol, max_iter, sums_dev);
    c->counters[0]++;
    VO_CUDA(cudaGetLastError());
    return VAMPOMI_OK;
}

}  // namespace vampomi
