// Internal declarations of libvampomi_cuda.so (not part of the public ABI; see include/vampomi.h).
#pragma once
#include <cuda_runtime.h>
#include <nccl.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include "../../include/vampomi.h"
#include "xchg.cuh"

namespace vampomi {

void set_error(const char* fmt, ...);

#define VO_CUDA(call)                                                                                   \
    do {                                                                                                \
        cudaError_t e__ = (call);                                                                       \
        if (e__ != cudaSuccess) {                                                                       \
            vampomi::set_error("CUDA error %s at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e__)); \
            return VAMPOMI_ERR_CUDA;                                                                    \
        }                                                                                               \
    } while (0)

#define VO_CHECK(expr)                 \
    do {                               \
        int rc__ = (expr);             \
        if (rc__ != VAMPOMI_OK) return rc__; \
    } while (0)

#define VO_ARG(cond, ...)                      \
    do {                                       \
        if (!(cond)) {                         \
            vampomi::set_error(__VA_ARGS__);   \
            return VAMPOMI_ERR_ARG;            \
        }                                      \
    } while (0)

// NCCL is loaded lazily with dlopen("libnccl.so.2"): inside a torch process that resolves to the already-mapped
// torch-bundled library, in the standalone host binary to the system one. Single-GPU use never touches it.
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
int nccl_load(NcclApi** api);

constexpr int MAX_MIX = 32;          // mixture components the denoiser/EM kernels accept
constexpr int RED_BLOCKS = 296;      // grid size of vector kernels (2 CTAs x 148 SMs)
constexpr int RED_THREADS = 256;
constexpr int MAX_DOTS = 16;         // reductions per vampomi_dots() call
constexpr int MAX_SUMS = 64;         // doubles in the packed scalar all-reduce buffer

struct MultiVec {                    // K vectors handled by one multi-right-hand-side pass (kernels_multi.cu)
    int K;
    const double* in[XCHG_KMAX];
    double* out[XCHG_KMAX];
    const int* done[XCHG_KMAX];      // per-slot "skip me" flag in device memory (nullptr = always active)
};

struct MixParams {                   // passed by value to the denoiser / EM kernels
    int L;
    double probs[MAX_MIX];           // probs (denoiser) or omegas (EM)
    double vars[MAX_MIX];
};

struct CgScalars {                   // device-resident CG scalars (src/vamp.cpp:694-751); slot = iteration parity
    double rz[2];
    double prev_onsager[2];
    double vv;
    double rel_err;
    double vmu;
    int done;                        // 0 running, 1 onsager test, 2 residual test, 3 max_iter
    int iters;
};

struct CgSys {                       // one linear system of a CG batch (cg.cu); all pointers are device memory
    const double* v;                 // right-hand side
    double* mu;                      // solution (start vector when warm)
    double *r, *z, *p, *d;           // CG work vectors
    double* atx_out;                 // A^T A mu_start while the solve is set up (warm), then = atx_work
    double* atx_work;                // A^T A p of the current iteration
    double* tmpN;                    // A p
    double* amu;                     // optional N-vector kept equal to A mu by the solve itself (amu += alpha * A p); nullptr = off
    double* gw;                      // one-pass CG: w = A A^T q of the current iteration (N); nullptr = two-pass CG
    double* gar;                     // one-pass CG: A r, advanced by A r -= alpha (tau w + gam2 q) (N)
    CgScalars* cg;
    int warm;
    int onsager_mode;
};
struct CgBatch {
    int S;
    CgSys s[2];
};

struct Tuning {
    int ax_rv = 0;                   // 256-bit vectors per thread per column in Ax (0 = measured default: 2 for FP64 storage, 1 for FP32)
    int ax_unroll = 0;               // columns in flight per thread (0 = measured default: 4 for FP64 storage, 2 for FP32)
    int ax_ctas_per_sm = 0;              // 0 = one resident wave (occupancy query)
    int atx_cols = 0;                // columns per pass in ATx (0 = default of the chosen implementation)
    int atx_unroll = 0;
    int atx_ctas_per_sm = 0;
    int cg_depth = 2;                // CG iterations kept enqueued ahead of the completion poll
    int ax_impl = 0;                 // 0 = per-thread 256-bit LDG streaming, 1 = bulk-copy (cp.async.bulk + mbarrier) pipeline
    int atx_impl = 3;                // 0 = warp per column group, 1 = bulk-copy pipeline, 2 = CTA per column group, 3 = auto (2 when N >= 4096, else 0)
    int xchg = 1;                    // 1 = fused peer-memory all-reduce (xchg.cuh) when it could be set up, 0 = NCCL collectives
    int xchg_ll = 1;                 // vector exchange: 1 = tagged words (no fence, no flags), 0 = payload + system fence + per-CTA flags
    int load_threads = 8;            // parallel pread -> pinned -> HBM pipelines of vampomi_load_file
    int load_depth = 3;              // pinned 32 MB slots per reader thread (reads in flight behind the one being filled)
    int load_direct = 0;             // 1 = O_DIRECT reads in 4 KB-aligned spans straight into the pinned slots (no page-cache copy)
    int ld_hint = 0;                 // L2 hint on the streaming loads of the default kernel shapes: 0 none, 1 L2::256B, 2 L2::evict_first, 3 both
    int interleave = 0;              // experiment: deal column groups round-robin over the grid instead of one contiguous range per CTA
    int multi_ax_rv = 0;             // multi-vector A x: 32-byte vectors per thread per column (0 = 1)
    int multi_ax_unroll = 0;         // multi-vector A x: columns in flight (0 = 4 for FP64 storage, 2 for FP32)
    int multi_ax_occ = 0;            // multi-vector A x, shape (1, 4): 3 = hold the kernel to 80 registers for three CTAs per SM (0 = two)
    int multi_atx_impl = 1;          // multi-vector A^T p: 0 = p tiles in registers, 1 = p tiles in shared memory
    int multi_atx_cols = 0;          // shared-memory form: columns per warp pass (0 = 2 for two vectors, 1 for one)
    int multi_atx_unroll = 0;        // shared-memory form: 32-byte steps in flight per column (0 = 4)
    int multi_atx_tile = 0;          // shared-memory form: rows of p per tile (0 = 2048)
    int grid_balance = 1;            // 1 = (row tile x column chunk) grids sized to full waves of resident CTAs (balanced_chunks), 0 = one, possibly partly filled, wave
    int dump_stream = 0;             // asynchronous read-outs copy on 0 = the context's stream (stream-ordered), 1 = the copy stream
    int center_split = 0;            // 1 = subtract the column mean once per sum instead of once per element (LDG variants)
    int cg_onepass = 0;              // 1 = CG iterations read the marker block ONCE (fused A^T q / A A^T q pass, kernels_gram.cu) where supported
    int gram_cluster = 0;            // fused pass: CTAs per cluster = row tiles of a column, 1 ... 16 (0 = ceil(ld / 2560), the fewest that hold N)
    int gram_clusters = 0;           // fused pass: clusters in the grid (0 = as many as are co-resident, occupancy query)
    int gram_refresh = 0;            // one-pass CG: recompute q = A p with a pass of its own every this many iterations (0 = 32)
};

}  // namespace vampomi

struct vampomi_ctx {
    int device = 0, N = 0, nranks = 1, rank = 0, num_sms = 148;
    long long Mt = 0, M = 0, S = 0;
    size_t ld = 0;                   // column stride of A in doubles (N rounded up to 16)
    size_t mpad = 0;                 // allocated length of M-vectors
    bool stats_ready = false;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    int storage = 0;                 // 0: A held as FP64 (reference layout), 1: A rounded to FP32 in HBM (opt-in; arithmetic stays FP64)
    int elem_bytes = 8;
    double* A = nullptr;             // [M][ld] column-major block in HBM (storage 0)
    float* A32 = nullptr;            // same layout in FP32 (storage 1)
    double* mave = nullptr;
    double* msig = nullptr;
    unsigned char* mconst = nullptr; // 1 = k_stats found the column constant (mave = its value, msig = 1)
    double* mvec[VAMPOMI_V_NUM_M] = {};
    double* nvec[VAMPOMI_V_NUM_N] = {};
    double* ax_partial = nullptr;    // [K][ax_chunks][ld]
    size_t ax_partial_elems = 0;
    double* atx_partial = nullptr;   // [row tiles][K][M] of the tiled A^T kernels
    size_t atx_partial_elems = 0;
    double* red_partials = nullptr;  // [MAX_DOTS][RED_BLOCKS][MAX_SUMS] scratch of the deterministic reductions
    unsigned int* red_tickets = nullptr;
    double* sums = nullptr;          // [MAX_SUMS] packed scalars (device), all-reduced in place
    double* psum = nullptr;          // sum of the N-vector fed to A^T (center_split form)
    double* sums_host = nullptr;     // pinned mirror
    vampomi::CgScalars* cg = nullptr;
    int* cg_poll_host = nullptr;     // pinned ring of done flags
    double* stage = nullptr;         // pinned staging for host<->device vector traffic (max(M,N,3M) doubles)
    size_t stage_elems = 0;
    // asynchronous vector read-out (vampomi_dump_begin / _wait)
    double* dump_dev[2] = {nullptr, nullptr};
    double* dump_host[2] = {nullptr, nullptr};   // pinned
    size_t dump_elems[2] = {0, 0};
    long long dump_len[2] = {0, 0};              // > 0 while a read-out is pending in the slot
    cudaEvent_t dump_ready[2] = {nullptr, nullptr}, dump_done[2] = {nullptr, nullptr};
    vampomi::Xchg xchg = {};         // peer-memory exchange descriptor (enabled == 0 -> NCCL path)
    bool xchg_ready = false;         // set up successfully at comm_init
    unsigned char* xchg_region = nullptr;
    unsigned int* xchg_local = nullptr;
    void* xchg_ipc_opened[vampomi::XCHG_MAX_RANKS] = {};
    void* load_ring = nullptr;       // pinned staging ring of vampomi_load_file (capi.cu LoadRing), allocated once
    int* xchg_err_host = nullptr;    // pinned, device-mapped: raised by a peer wait that gave up (xchg.cuh XchgDeadline)
    cudaEvent_t cg_events[32] = {};  // completion-poll ring of the CG loop, created once
    ncclComm_t comm = nullptr;
    vampomi::NcclApi* nccl = nullptr;
    vampomi::Tuning tune;
    long long counters[4] = {0, 0, 0, 0};
    int gram_clusters[17][2] = {};   // co-resident clusters of k_gram_wsx per (cluster size 1 ... 16, systems), 0 = not queried yet
    // tensor map of the marker block for the fused pass's one-copy-per-step producer (a CUtensorMap; kernels_gram.cu), with its key
    alignas(64) unsigned char gram_tmap[128] = {};
    const void* gram_tmap_A = nullptr;
    size_t gram_tmap_ld = 0;
    long long gram_tmap_M = 0;
    int gram_tmap_rows = 0, gram_tmap_C = 0;
    bool bulk_attr_ax = false, bulk_attr_atx = false;   // opt-in shared-memory size set for the bulk kernels on this device
    // optional per-launch device timing (vampomi_profile_*)
    bool profile = false;
    struct ProfSpan { int kind; cudaEvent_t e0, e1; double bytes; };
    std::vector<ProfSpan> prof_pending;
    std::vector<cudaEvent_t> prof_free;
    double prof_acc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};   // kinds: 0 A x, 1 A x reduce + exchange, 2 A^T p, 3 fused A^T q / A A^T q
};

namespace vampomi {

inline double* vec_ptr(const vampomi_ctx* c, int id) {
    if (id >= 0 && id < VAMPOMI_V_NUM_M) return c->mvec[id];
    if (id >= 32 && id < 32 + VAMPOMI_V_NUM_N) return c->nvec[id - 32];
    return nullptr;
}
inline long long vec_len(const vampomi_ctx* c, int id) {
    if (id >= 0 && id < VAMPOMI_V_NUM_M) return c->M;
    if (id >= 32 && id < 32 + VAMPOMI_V_NUM_N) return c->N;
    return -1;
}
// Column chunks for a (row tiles x column chunks) grid of a streaming matrix kernel. `slots` = resident CTAs of the device
// (SMs x CTAs per SM). One wave is floor(slots / ntiles) chunks, which leaves slots idle whenever ntiles does not divide
// slots (20 row tiles on 296 slots: 280 CTAs, 5 % of the machine unused for the whole kernel). Take the smallest number of
// waves w for which floor(w * slots / ntiles) chunks fill the w waves to within 1 %: every wave is (almost) full, and with
// w > 1 a CTA that finishes early is replaced at once, so the tail is one smaller CTA long.
inline long long balanced_chunks(long long slots, int ntiles, long long M, int min_cols, bool balance) {
    long long nch = slots / ntiles;
    if (balance) {
        for (int w = 1; w <= 8; w++) {
            const long long n = w * slots / ntiles;
            if (n < 1) continue;
            nch = n;
            if ((double)(n * ntiles) >= 0.99 * (double)(w * slots)) break;
        }
    }
    if (min_cols < 1) min_cols = 1;
    const long long cap = (M + min_cols - 1) / min_cols;        // keep at least min_cols columns per chunk
    if (nch > cap) nch = cap;
    if (nch < 1) nch = 1;
    return nch;
}

inline bool is_mvec(int id) { return id >= 0 && id < VAMPOMI_V_NUM_M; }
// M-vectors the library's own calls clobber (TMP_*, CG_*, CG2_*): not usable as rhs / sol of a solve
inline bool is_work_mvec(int id) {
    return (id >= VAMPOMI_V_TMP_M0 && id <= VAMPOMI_V_CG_D) || (id >= VAMPOMI_V_CG2_R && id <= VAMPOMI_V_CG2_D);
}

// ---- launchers (kernels_matrix.cu) ----
int launch_generate_iid(vampomi_ctx* c, uint64_t seed);
int launch_stats(vampomi_ctx* c, double alpha_scale);
int launch_impute_missing(vampomi_ctx* c, long long* counts_dev, int* nblocks);      // counts_dev: [nblocks][3] per-block counts
int launch_ax(vampomi_ctx* c, const double* x_dev, double* out_dev, const int* done_flag);     // incl. all-reduce and 1/sqrt(N)
int launch_atx(vampomi_ctx* c, const double* p_dev, double* out_dev, const int* done_flag);
int launch_loo_sums(vampomi_ctx* c, const double* w_dev, double* sums_dev);
int launch_read_probe(vampomi_ctx* c);
// ---- launchers (kernels_multi.cu): one pass over A for K vectors ----
int launch_ax_multi(vampomi_ctx* c, const MultiVec& mv);
int launch_atx_multi(vampomi_ctx* c, const MultiVec& mv);
int ensure_ax_partial(vampomi_ctx* c, size_t elems);                              // scratch [K][chunks][ld] of the A x style kernels
int launch_ax_reduce_multi(vampomi_ctx* c, int nchunks, const MultiVec& mv);      // chunk partials -> out_k (+ cross-GPU sum, / sqrt(N))
// ---- launchers (kernels_gram.cu): t = A^T q and w = A t in ONE pass over A (K <= 2 systems) ----
bool gram_supported(const vampomi_ctx* c);
int launch_gram(vampomi_ctx* c, const MultiVec& mq, double* const* w_out);
int launch_f64_to_f32(vampomi_ctx* c, float* dst, const double* src_dense, long long ncols, cudaStream_t st);
int launch_f32_to_f64(vampomi_ctx* c, double* dst_dense, const float* src, long long ncols, cudaStream_t st);
// ---- launchers (kernels_bulk.cu) ----
int launch_atx_bulk(vampomi_ctx* c, const double* p_dev, double* out_dev, const int* done_flag);
int launch_ax_bulk(vampomi_ctx* c, const double* x_dev, const int* done_flag, int* nchunks_out);
// ---- launchers (kernels_vector.cu) ----
int launch_fill(vampomi_ctx* c, double* dst, long long n, double v);
int launch_lincomb(vampomi_ctx* c, double* dst, double a, const double* x, double b, const double* y, double cdiv, long long n);
int launch_scale_div(vampomi_ctx* c, double* dst, const double* src, double divisor, long long n, const int* done_flag);
int launch_dots(vampomi_ctx* c, int n, const int* kind, const double* const* a, const double* const* b, const long long* len,
                const double* scale, double* sums_dev);
int launch_probe(vampomi_ctx* c, uint64_t seed, int it);
int launch_denoise(vampomi_ctx* c, double gam1, const MixParams& mp, int damp, double rho, double* sums_dev);
int launch_em_sums(vampomi_ctx* c, double gam1, double lambda, const MixParams& mp, double* sums_dev);
int launch_probit_z(vampomi_ctx* c, double tau1, double* sums_dev);
int launch_pvals_se(vampomi_ctx* c, const double* r1_dev, double sd, double* out_dev);
int launch_cg_init(vampomi_ctx* c, const CgBatch& b, double tau, double gam2, double diag, double* sums_dev);   // also zeroes amu of cold systems
int launch_cg_init_finish(vampomi_ctx* c, const CgBatch& b, const double* sums_dev);
int launch_cg_dp(vampomi_ctx* c, const CgBatch& b, double tau, double gam2, double* sums_dev);
int launch_cg_step(vampomi_ctx* c, const CgBatch& b, double tau, double gam2, double diag, int parity, const double* dp_dev, double* sums_dev);
int launch_cg_finish(vampomi_ctx* c, const CgBatch& b, int parity, double gam2, double diag, double tol, int max_iter, const double* sums_dev);
int launch_xchg_sums(vampomi_ctx* c, double* sums_dev, int n);   // n <= XCHG_SCALARS packed sums over the GPUs via peer memory
// all-reduce `n` doubles in place on the context stream (no-op for nranks == 1)
int allreduce_inplace(vampomi_ctx* c, double* dev, size_t n);
// VAMPOMI_ERR_STATE if a peer-memory wait on this context has given up (a rank is gone or too far behind); call after a stream sync
int xchg_check(vampomi_ctx* c);
// all ranks meet here (tiny NCCL all-reduce + stream sync); no-op for one rank
int rank_barrier(vampomi_ctx* c);
// profiling spans: begin returns an index (or -1 when profiling is off), end closes it
int prof_begin(vampomi_ctx* c, int kind, double bytes);
void prof_end(vampomi_ctx* c, int idx);
int prof_resolve(vampomi_ctx* c);

}  // namespace vampomi
