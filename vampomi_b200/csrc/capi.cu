// extern "C" layer of libvampomi_cuda.so (declared in include/vampomi.h): context lifetime, HBM upload path,
// NCCL plumbing, and thin wrappers that launch the kernels of kernels_matrix.cu / kernels_vector.cu / cg.cu.
#include <dlfcn.h>
#include <fcntl.h>
#include <stdarg.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>
#include <cmath>
#include <vector>
#include <new>
#include <string>
#include <thread>
#include "common.h"

namespace vampomi {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int nccl_load(NcclApi** out) {
    static NcclApi api;
    static int state = 0;      // 0 untried, 1 ok, -1 failed
    if (state == 0) {
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (!api.handle) { state = -1; }
        else {
            api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.handle, "ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.handle, "ncclCommInitRank");
            api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.handle, "ncclCommDestroy");
            api.AllReduce = (decltype(api.AllReduce))dlsym(api.handle, "ncclAllReduce");
            api.AllGather = (decltype(api.AllGather))dlsym(api.handle, "ncclAllGather");
            api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.handle, "ncclGetErrorString");
            state = (api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce && api.AllGather && api.GetErrorString) ? 1 : -1;
        }
    }
    if (state != 1) {
        set_error("libnccl.so.2 could not be loaded (%s)", dlerror() ? dlerror() : "missing symbols");
        return VAMPOMI_ERR_NCCL;
    }
    *out = &api;
    return VAMPOMI_OK;
}

int allreduce_inplace(vampomi_ctx* c, double* dev, size_t n) {
    if (c->nranks == 1) return VAMPOMI_OK;
    if (!c->comm) { set_error("nranks > 1 but vampomi_comm_init was not called"); return VAMPOMI_ERR_STATE; }
    ncclResult_t r = c->nccl->AllReduce(dev, dev, n, ncclDouble, ncclSum, c->comm, c->stream);
    if (r != ncclSuccess) { set_error("ncclAllReduce: %s", c->nccl->GetErrorString(r)); return VAMPOMI_ERR_NCCL; }
    c->counters[3]++;
    return VAMPOMI_OK;
}

int xchg_check(vampomi_ctx* c) {
    if (c->xchg_err_host && *reinterpret_cast<volatile int*>(c->xchg_err_host) != 0) {
        c->xchg.enabled = 0; c->xchg_ready = false;        // sequence numbers are out of step now: this context's exchange is over
        set_error("cross-GPU exchange timed out on rank %d: a peer rank is gone or more than %.0f s behind (VAMPOMI_XCHG_TIMEOUT_S)",
                  c->rank, (double)c->xchg.timeout_ns * 1e-9);
        return VAMPOMI_ERR_STATE;
    }
    return VAMPOMI_OK;
}

int rank_barrier(vampomi_ctx* c) {
    if (c->nranks == 1) return VAMPOMI_OK;
    if (!c->comm) { set_error("nranks > 1 but vampomi_comm_init was not called"); return VAMPOMI_ERR_STATE; }
    int* d = reinterpret_cast<int*>(c->sums + (MAX_SUMS - 2));      // scratch at the end of the packed-sums buffer (never used by the kernels)
    VO_CUDA(cudaMemsetAsync(d, 0, sizeof(int), c->stream));
    ncclResult_t r = c->nccl->AllReduce(d, d, 1, ncclInt, ncclSum, c->comm, c->stream);
    if (r != ncclSuccess) { set_error("ncclAllReduce (barrier): %s", c->nccl->GetErrorString(r)); return VAMPOMI_ERR_NCCL; }
    VO_CUDA(cudaStreamSynchronize(c->stream));
    return VAMPOMI_OK;
}

// packed scalar sums over the GPUs: the peer-memory exchange when it is up (identically on all ranks), else NCCL
static int sum_over_ranks(vampomi_ctx* c, double* dev, size_t n) {
    if (c->nranks == 1) return VAMPOMI_OK;
    if (c->xchg.enabled && n <= (size_t)XCHG_SCALARS) return launch_xchg_sums(c, dev, (int)n);
    return allreduce_inplace(c, dev, n);
}

int prof_begin(vampomi_ctx* c, int kind, double bytes) {
    if (!c->profile) return -1;
    vampomi_ctx::ProfSpan sp;
    sp.kind = kind; sp.bytes = bytes;
    for (cudaEvent_t* e : {&sp.e0, &sp.e1}) {
        if (!c->prof_free.empty()) { *e = c->prof_free.back(); c->prof_free.pop_back(); }
        else if (cudaEventCreate(e) != cudaSuccess) return -1;
    }
    cudaEventRecord(sp.e0, c->stream);
    c->prof_pending.push_back(sp);
    return (int)c->prof_pending.size() - 1;
}
void prof_end(vampomi_ctx* c, int idx) {
    if (idx < 0 || idx >= (int)c->prof_pending.size()) return;
    cudaEventRecord(c->prof_pending[idx].e1, c->stream);
}
int prof_resolve(vampomi_ctx* c) {
    if (c->prof_pending.empty()) return VAMPOMI_OK;
    VO_CUDA(cudaStreamSynchronize(c->stream));
    for (auto& sp : c->prof_pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, sp.e0, sp.e1) == cudaSuccess) {
            c->prof_acc[3 * sp.kind] += 1.0;
            c->prof_acc[3 * sp.kind + 1] += (double)ms;
            c->prof_acc[3 * sp.kind + 2] += sp.bytes;
        }
        c->prof_free.push_back(sp.e0);
        c->prof_free.push_back(sp.e1);
    }
    c->prof_pending.clear();
    return VAMPOMI_OK;
}

// ---- peer-memory exchange set-up (xchg.cuh) -----------------------------------------------------------------------
struct XchgInfo {            // what every rank tells the others about its exchange region
    long long pid;
    int device, ok;
    unsigned long long ptr;
    cudaIpcMemHandle_t handle;
};

static void xchg_teardown(vampomi_ctx* c) {
    for (int g = 0; g < XCHG_MAX_RANKS; g++)
        if (c->xchg_ipc_opened[g]) { cudaIpcCloseMemHandle(c->xchg_ipc_opened[g]); c->xchg_ipc_opened[g] = nullptr; }
    if (c->xchg_region) cudaFree(c->xchg_region);
    if (c->xchg_local) cudaFree(c->xchg_local);
    if (c->xchg_err_host) cudaFreeHost(c->xchg_err_host);
    c->xchg_region = nullptr; c->xchg_local = nullptr; c->xchg_err_host = nullptr;
    c->xchg_ready = false; c->xchg.enabled = 0;
}

// Maps every rank's exchange region into this rank's address space: CUDA IPC between processes (torchrun, one rank
// per process), plain peer access between the rank threads of one process (main_meth --gpus G). Collective: all ranks
// call it right after ncclCommInitRank; the exchange is enabled only if it could be set up on EVERY rank.
static int xchg_setup(vampomi_ctx* c) {
    auto align = [](size_t v) { return (v + 255) / 256 * 256; };
    int ok = c->nranks <= XCHG_MAX_RANKS ? 1 : 0;
    const char* env = getenv("VAMPOMI_XCHG");
    if (env && env[0] == '0') c->tune.xchg = 0;
    Xchg& x = c->xchg;
    x = Xchg{};
    x.G = c->nranks; x.rank = c->rank; x.ld = (unsigned long long)XCHG_KMAX * c->ld;
    x.maxb = XCHG_KMAX * (int)((c->ld + 31) / 32);
    size_t off = 0;
    x.off_flag_vec = off; off = align(off + (size_t)x.G * x.maxb * sizeof(unsigned int));
    x.off_flag_sc = off;  off = align(off + (size_t)x.G * 32 * sizeof(unsigned int));
    x.off_recv_vec = off; off = align(off + (size_t)2 * x.G * XCHG_KMAX * c->ld * 2 * sizeof(double));    // x 2: tagged words (xchg.cuh)
    x.off_recv_sc = off;  off = align(off + (size_t)2 * x.G * XCHG_SCALARS * 2 * sizeof(double));
    const size_t region_bytes = off;
    XchgInfo mine{};
    mine.pid = (long long)getpid(); mine.device = c->device;
    int* err_dev = nullptr;
    if (ok && (cudaMalloc(&c->xchg_region, region_bytes) != cudaSuccess || cudaMemset(c->xchg_region, 0, region_bytes) != cudaSuccess ||
               cudaMalloc(&c->xchg_local, 4 * sizeof(unsigned int)) != cudaSuccess ||
               cudaMemset(c->xchg_local, 0, 4 * sizeof(unsigned int)) != cudaSuccess ||
               cudaHostAlloc(&c->xchg_err_host, sizeof(int), cudaHostAllocMapped) != cudaSuccess ||
               cudaHostGetDevicePointer(&err_dev, c->xchg_err_host, 0) != cudaSuccess ||
               cudaIpcGetMemHandle(&mine.handle, c->xchg_region) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess))
        ok = 0;
    cudaGetLastError();
    if (c->xchg_err_host) *c->xchg_err_host = 0;
    mine.ok = ok; mine.ptr = (unsigned long long)(uintptr_t)c->xchg_region;
    // all-gather the descriptors through NCCL itself (device staging), so no second bootstrap channel is needed. This function
    // is collective: a LOCAL failure (allocation, copy) must not skip the collectives below — the other ranks would hang in
    // them — so local failures only clear `ok`, both collectives are always reached, and only an NCCL failure returns early.
    std::vector<XchgInfo> all((size_t)c->nranks);
    XchgInfo *d_send = nullptr, *d_recv = nullptr;
    int nccl_rc = VAMPOMI_OK;
    bool staged = cudaMalloc(&d_send, sizeof(XchgInfo) > sizeof(int) * 2 ? sizeof(XchgInfo) : sizeof(int) * 2) == cudaSuccess &&
                  cudaMalloc(&d_recv, sizeof(XchgInfo) * c->nranks) == cudaSuccess;
    if (!staged) { ok = 0; mine.ok = 0; cudaGetLastError(); }
    if (staged) {
        if (cudaMemcpyAsync(d_send, &mine, sizeof(XchgInfo), cudaMemcpyHostToDevice, c->stream) != cudaSuccess) { ok = 0; cudaGetLastError(); }
        ncclResult_t r = c->nccl->AllGather(d_send, d_recv, sizeof(XchgInfo), ncclChar, c->comm, c->stream);
        if (r != ncclSuccess) { set_error("ncclAllGather: %s", c->nccl->GetErrorString(r)); nccl_rc = VAMPOMI_ERR_NCCL; }
        else if (cudaMemcpyAsync(all.data(), d_recv, sizeof(XchgInfo) * c->nranks, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
                 cudaStreamSynchronize(c->stream) != cudaSuccess) { ok = 0; cudaGetLastError(); }
    }
    for (int g = 0; g < c->nranks && ok && nccl_rc == VAMPOMI_OK; g++) {
        if (!all[g].ok) { ok = 0; break; }
        if (g == c->rank) { x.peer[g] = c->xchg_region; continue; }
        if (all[g].pid == mine.pid) {                         // a rank thread of this process: direct peer access
            cudaError_t e = cudaDeviceEnablePeerAccess(all[g].device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) ok = 0;
            cudaGetLastError();
            x.peer[g] = (unsigned char*)(uintptr_t)all[g].ptr;
        } else {
            void* p = nullptr;
            if (cudaIpcOpenMemHandle(&p, all[g].handle, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); }
            else { c->xchg_ipc_opened[g] = p; x.peer[g] = (unsigned char*)p; }
        }
    }
    // enable only if EVERY rank succeeded (a mixed job would deadlock): min-reduce the flag; doubles as the barrier that
    // guarantees every region is zeroed before the first push. A rank whose staging allocation failed cannot take part in a
    // device collective at all: it falls back to a host-side int through the same all-reduce on its packed-sums buffer.
    int all_ok = 0;
    if (nccl_rc == VAMPOMI_OK) {
        int* d_ok = staged ? reinterpret_cast<int*>(d_send) : reinterpret_cast<int*>(c->sums + (MAX_SUMS - 2));
        bool sent = cudaMemcpyAsync(d_ok, &ok, sizeof(int), cudaMemcpyHostToDevice, c->stream) == cudaSuccess;
        ncclResult_t r = c->nccl->AllReduce(d_ok, d_ok, 1, ncclInt, ncclMin, c->comm, c->stream);
        if (r != ncclSuccess) { set_error("ncclAllReduce: %s", c->nccl->GetErrorString(r)); nccl_rc = VAMPOMI_ERR_NCCL; }
        else if (!sent || cudaMemcpyAsync(&all_ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
                 cudaStreamSynchronize(c->stream) != cudaSuccess) { all_ok = 0; cudaGetLastError(); }
    }
    if (d_send) cudaFree(d_send);
    if (d_recv) cudaFree(d_recv);
    if (nccl_rc != VAMPOMI_OK) { xchg_teardown(c); return nccl_rc; }
    if (!all_ok) { xchg_teardown(c); return VAMPOMI_OK; }     // stay on the NCCL collectives
    x.err = err_dev;
    {
        double tmo = 120.0;
        if (const char* t = getenv("VAMPOMI_XCHG_TIMEOUT_S")) { const double v = atof(t); if (v > 0) tmo = v; }
        x.timeout_ns = (unsigned long long)(tmo * 1e9);
    }
    x.seq = c->xchg_local; x.ticket = c->xchg_local + 2;
    c->xchg_ready = true;
    x.enabled = c->tune.xchg ? 1 : 0;
    x.ll = c->tune.xchg_ll ? 1 : 0;
    return VAMPOMI_OK;
}

static int ensure_stage(vampomi_ctx* c, size_t elems) {
    if (elems <= c->stage_elems) return VAMPOMI_OK;
    if (c->stage) VO_CUDA(cudaFreeHost(c->stage));
    c->stage = nullptr; c->stage_elems = 0;
    VO_CUDA(cudaMallocHost(&c->stage, elems * sizeof(double)));
    c->stage_elems = elems;
    return VAMPOMI_OK;
}

// device sums -> pinned host -> caller, after the (optional) packed all-reduce; ONE sync
static int fetch_sums(vampomi_ctx* c, int n, bool reduce, double* out) {
    if (reduce) VO_CHECK(sum_over_ranks(c, c->sums, (size_t)n));
    VO_CUDA(cudaMemcpyAsync(c->sums_host, c->sums, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    VO_CUDA(cudaStreamSynchronize(c->stream));
    VO_CHECK(xchg_check(c));
    for (int i = 0; i < n; i++) out[i] = c->sums_host[i];
    return VAMPOMI_OK;
}

static int h2d_vec(vampomi_ctx* c, double* dev, const double* host, long long n) {
    VO_CHECK(ensure_stage(c, (size_t)n));
    memcpy(c->stage, host, (size_t)n * sizeof(double));
    VO_CUDA(cudaMemcpyAsync(dev, c->stage, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    VO_CUDA(cudaStreamSynchronize(c->stream));      // the staging buffer is reused by the next call
    return VAMPOMI_OK;
}
// buffers and events of the asynchronous read-outs (vampomi_dump_begin): allocated once, at context creation, so that no
// allocation (pinning 2 x 6.8 MB takes tens of milliseconds) ever lands inside an iteration
static int ensure_dump(vampomi_ctx* c) {
    const size_t n = c->mpad > c->ld ? c->mpad : c->ld;
    for (int k = 0; k < 2; k++) {
        if (c->dump_elems[k] >= n) continue;
        if (c->dump_dev[k]) VO_CUDA(cudaFree(c->dump_dev[k]));
        if (c->dump_host[k]) VO_CUDA(cudaFreeHost(c->dump_host[k]));
        c->dump_dev[k] = nullptr; c->dump_host[k] = nullptr; c->dump_elems[k] = 0;
        VO_CUDA(cudaMalloc(&c->dump_dev[k], n * sizeof(double)));
        VO_CUDA(cudaMallocHost(&c->dump_host[k], n * sizeof(double)));
        c->dump_elems[k] = n;
        if (!c->dump_ready[k]) {
            VO_CUDA(cudaEventCreateWithFlags(&c->dump_ready[k], cudaEventDisableTiming));
            VO_CUDA(cudaEventCreateWithFlags(&c->dump_done[k], cudaEventDisableTiming));
        }
    }
    return VAMPOMI_OK;
}

static int d2h_vec(vampomi_ctx* c, double* host, const double* dev, long long n) {
    VO_CHECK(ensure_stage(c, (size_t)n));
    VO_CUDA(cudaMemcpyAsync(c->stage, dev, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    VO_CUDA(cudaStreamSynchronize(c->stream));
    VO_CHECK(xchg_check(c));
    memcpy(host, c->stage, (size_t)n * sizeof(double));
    return VAMPOMI_OK;
}

}  // namespace vampomi

using namespace vampomi;

extern "C" {

static void load_ring_free(vampomi_ctx* c);

const char* vampomi_last_error(void) { return g_err; }
int vampomi_abi_version(void) { return VAMPOMI_ABI_VERSION; }

int vampomi_device_count(int* count) {
    VO_ARG(count != nullptr, "device_count: NULL argument");
    *count = 0;
    cudaError_t e = cudaGetDeviceCount(count);
    if (e != cudaSuccess || *count == 0) {
        *count = 0;
        set_error("no CUDA device available (%s); libvampomi_cuda has no CPU fallback", cudaGetErrorString(e));
        return VAMPOMI_ERR_CUDA;
    }
    return VAMPOMI_OK;
}

int vampomi_divide_work(long long Mt, int nranks, int rank, long long* M, long long* S) {
    VO_ARG(Mt >= 1 && nranks >= 1 && rank >= 0 && rank < nranks && M && S, "divide_work: bad arguments");
    const long long modu = Mt % nranks, size = Mt / nranks;           // src/utilities.cpp:214-225
    *M = rank < modu ? size + 1 : size;
    *S = rank * size + (rank < modu ? rank : modu);
    return VAMPOMI_OK;
}

int vampomi_create(int device, int N, long long Mt, int nranks, int rank, vampomi_ctx** out) {
    return vampomi_create_ex(device, N, Mt, nranks, rank, VAMPOMI_STORE_F64, out);
}

int vampomi_storage(const vampomi_ctx* c, int* storage) {
    VO_ARG(c && storage, "storage: NULL argument");
    *storage = c->storage;
    return VAMPOMI_OK;
}

int vampomi_create_ex(int device, int N, long long Mt, int nranks, int rank, int storage, vampomi_ctx** out) {
    VO_ARG(out != nullptr, "create: out is NULL");
    *out = nullptr;
    VO_ARG(storage == VAMPOMI_STORE_F64 || storage == VAMPOMI_STORE_F32, "create: unknown storage %d", storage);
    VO_ARG(N >= 2 && Mt >= 1, "create: need N >= 2 and Mt >= 1 (got N=%d Mt=%lld)", N, Mt);
    VO_ARG(nranks >= 1 && rank >= 0 && rank < nranks, "create: bad rank %d of %d", rank, nranks);
    VO_ARG(Mt >= nranks, "create: fewer markers (%lld) than shards (%d)", Mt, nranks);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        set_error("no CUDA device available (%s); libvampomi_cuda has no CPU fallback", cudaGetErrorString(e));
        return VAMPOMI_ERR_CUDA;
    }
    VO_ARG(device >= 0 && device < ndev, "create: device %d out of range (%d devices)", device, ndev);
    VO_CUDA(cudaSetDevice(device));
    vampomi_ctx* c = new (std::nothrow) vampomi_ctx();
    VO_ARG(c != nullptr, "create: out of host memory");
    c->device = device; c->N = N; c->Mt = Mt; c->nranks = nranks; c->rank = rank;
    c->storage = storage; c->elem_bytes = storage == VAMPOMI_STORE_F32 ? 4 : 8;
    vampomi_divide_work(Mt, nranks, rank, &c->M, &c->S);
    c->ld = ((size_t)N + 15) / 16 * 16;
    c->mpad = ((size_t)c->M + 15) / 16 * 16;
    int rc = [&]() -> int {
        cudaDeviceProp prop;
        VO_CUDA(cudaGetDeviceProperties(&prop, device));
        c->num_sms = prop.multiProcessorCount;
        VO_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        VO_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        const size_t a_bytes = (size_t)c->M * c->ld * (size_t)c->elem_bytes;
        void* a_ptr = nullptr;
        cudaError_t ea = cudaMalloc(&a_ptr, a_bytes);
        if (ea != cudaSuccess) {
            set_error("cudaMalloc of the %.3f GB marker block failed: %s", a_bytes / 1e9, cudaGetErrorString(ea));
            return VAMPOMI_ERR_CUDA;
        }
        if (c->storage == VAMPOMI_STORE_F32) c->A32 = (float*)a_ptr; else c->A = (double*)a_ptr;
        if (c->ld != (size_t)N) VO_CUDA(cudaMemsetAsync(a_ptr, 0, a_bytes, c->stream));    // pad rows must be zero
        VO_CUDA(cudaMalloc(&c->mave, c->mpad * sizeof(double)));
        VO_CUDA(cudaMalloc(&c->msig, c->mpad * sizeof(double)));
        VO_CUDA(cudaMalloc(&c->mconst, c->mpad));
        for (int i = 0; i < VAMPOMI_V_NUM_M; i++) {
            VO_CUDA(cudaMalloc(&c->mvec[i], c->mpad * sizeof(double)));
            VO_CUDA(cudaMemsetAsync(c->mvec[i], 0, c->mpad * sizeof(double), c->stream));
        }
        for (int i = 0; i < VAMPOMI_V_NUM_N; i++) {
            VO_CUDA(cudaMalloc(&c->nvec[i], c->ld * sizeof(double)));
            VO_CUDA(cudaMemsetAsync(c->nvec[i], 0, c->ld * sizeof(double), c->stream));
        }
        VO_CUDA(cudaMalloc(&c->red_partials, (size_t)RED_BLOCKS * MAX_SUMS * sizeof(double)));
        VO_CUDA(cudaMalloc(&c->red_tickets, MAX_DOTS * sizeof(unsigned int)));
        VO_CUDA(cudaMemsetAsync(c->red_tickets, 0, MAX_DOTS * sizeof(unsigned int), c->stream));
        VO_CUDA(cudaMalloc(&c->sums, MAX_SUMS * sizeof(double)));
        VO_CUDA(cudaMemsetAsync(c->sums, 0, MAX_SUMS * sizeof(double), c->stream));
        VO_CUDA(cudaMallocHost(&c->sums_host, MAX_SUMS * sizeof(double)));
        VO_CUDA(cudaMalloc(&c->psum, sizeof(double)));
        VO_CUDA(cudaMalloc(&c->cg, 2 * sizeof(CgScalars)));          // one per system of a paired solve
        VO_CUDA(cudaMemsetAsync(c->cg, 0, 2 * sizeof(CgScalars), c->stream));
        VO_CUDA(cudaMallocHost(&c->cg_poll_host, 64 * sizeof(int)));
        VO_CHECK(ensure_dump(c));
        size_t st = (size_t)(3 * c->M > (long long)c->ld ? 3 * c->M : (long long)c->ld);
        VO_CHECK(ensure_stage(c, st));
        VO_CUDA(cudaStreamSynchronize(c->stream));
        return VAMPOMI_OK;
    }();
    if (rc != VAMPOMI_OK) { vampomi_destroy(c); return rc; }
    *out = c;
    return VAMPOMI_OK;
}

int vampomi_destroy(vampomi_ctx* c) {
    if (!c) return VAMPOMI_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (auto& sp : c->prof_pending) { cudaEventDestroy(sp.e0); cudaEventDestroy(sp.e1); }
    for (auto e : c->prof_free) cudaEventDestroy(e);
    xchg_teardown(c);
    if (c->comm && c->nccl) c->nccl->CommDestroy(c->comm);
    cudaFree(c->A); cudaFree(c->A32); cudaFree(c->mave); cudaFree(c->msig); cudaFree(c->mconst);
    for (auto p : c->mvec) cudaFree(p);
    for (auto p : c->nvec) cudaFree(p);
    cudaFree(c->psum); cudaFree(c->atx_partial);
    cudaFree(c->ax_partial); cudaFree(c->red_partials); cudaFree(c->red_tickets); cudaFree(c->sums); cudaFree(c->cg);
    if (c->sums_host) cudaFreeHost(c->sums_host);
    if (c->cg_poll_host) cudaFreeHost(c->cg_poll_host);
    if (c->stage) cudaFreeHost(c->stage);
    for (auto e : c->cg_events) if (e) cudaEventDestroy(e);
    load_ring_free(c);
    for (int k = 0; k < 2; k++) {
        if (c->dump_dev[k]) cudaFree(c->dump_dev[k]);
        if (c->dump_host[k]) cudaFreeHost(c->dump_host[k]);
        if (c->dump_ready[k]) cudaEventDestroy(c->dump_ready[k]);
        if (c->dump_done[k]) cudaEventDestroy(c->dump_done[k]);
    }
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    delete c;
    return VAMPOMI_OK;
}

int vampomi_shard(const vampomi_ctx* c, long long* M, long long* S) {
    VO_ARG(c && M && S, "shard: NULL argument");
    *M = c->M; *S = c->S;
    return VAMPOMI_OK;
}

int vampomi_dims(const vampomi_ctx* c, int* N, long long* Mt, int* nranks, int* rank) {
    VO_ARG(c, "dims: NULL context");
    if (N) *N = c->N;
    if (Mt) *Mt = c->Mt;
    if (nranks) *nranks = c->nranks;
    if (rank) *rank = c->rank;
    return VAMPOMI_OK;
}

int vampomi_comm_get_unique_id(void* id128) {
    VO_ARG(id128 != nullptr, "comm_get_unique_id: NULL buffer");
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
    NcclApi* api = nullptr;
    VO_CHECK(nccl_load(&api));
    ncclUniqueId id;
    ncclResult_t r = api->GetUniqueId(&id);
    if (r != ncclSuccess) { set_error("ncclGetUniqueId: %s", api->GetErrorString(r)); return VAMPOMI_ERR_NCCL; }
    memcpy(id128, &id, 128);
    return VAMPOMI_OK;
}

int vampomi_comm_init(vampomi_ctx* c, const void* id128) {
    VO_ARG(c && id128, "comm_init: NULL argument");
    if (c->nranks == 1) return VAMPOMI_OK;
    VO_CHECK(nccl_load(&c->nccl));
    VO_CUDA(cudaSetDevice(c->device));
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclResult_t r = c->nccl->CommInitRank(&c->comm, c->nranks, id, c->rank);
    if (r != ncclSuccess) { set_error("ncclCommInitRank: %s", c->nccl->GetErrorString(r)); c->comm = nullptr; return VAMPOMI_ERR_NCCL; }
    return xchg_setup(c);
}

int vampomi_barrier(vampomi_ctx* c) {
    VO_ARG(c, "barrier: NULL context");
    VO_CUDA(cudaSetDevice(c->device));
    return rank_barrier(c);
}

int vampomi_comm_mode(const vampomi_ctx* c, int* mode) {
    VO_ARG(c && mode, "comm_mode: NULL argument");
    *mode = c->nranks == 1 ? 0 : (c->xchg.enabled ? 2 : 1);
    return VAMPOMI_OK;
}

// ---- design matrix --------------------------------------------------------------------------------------------
int vampomi_upload_columns(vampomi_ctx* c, long long j0, long long ncols, const double* host) {
    VO_ARG(c && host && j0 >= 0 && ncols >= 0 && j0 + ncols <= c->M, "upload_columns: range [%lld,+%lld) outside the shard", j0, ncols);
    VO_CUDA(cudaSetDevice(c->device));
    if (ncols == 0) return VAMPOMI_OK;
    c->stats_ready = false;
    if (c->storage == VAMPOMI_STORE_F32) {                 // FP64 columns -> dense device staging -> rounded into place
        long long chunk = (long long)((64ull << 20) / ((size_t)c->N * sizeof(double)));
        if (chunk < 1) chunk = 1;
        double* tmp = nullptr;
        VO_CUDA(cudaMalloc(&tmp, (size_t)(chunk < ncols ? chunk : ncols) * c->N * sizeof(double)));
        int rc = VAMPOMI_OK;
        for (long long j = 0; j < ncols && rc == VAMPOMI_OK; j += chunk) {
            const long long nc = ncols - j < chunk ? ncols - j : chunk;
            if (cudaMemcpyAsync(tmp, host + (size_t)j * c->N, (size_t)nc * c->N * sizeof(double), cudaMemcpyHostToDevice, c->stream) != cudaSuccess) {
                set_error("upload_columns: host-to-device copy failed"); rc = VAMPOMI_ERR_CUDA; break;
            }
            rc = launch_f64_to_f32(c, c->A32 + (size_t)(j0 + j) * c->ld, tmp, nc, c->stream);
            if (cudaStreamSynchronize(c->stream) != cudaSuccess) { set_error("upload_columns: sync failed"); rc = VAMPOMI_ERR_CUDA; }
        }
        cudaFree(tmp);
        return rc;
    }
    VO_CUDA(cudaMemcpy2DAsync(c->A + (size_t)j0 * c->ld, c->ld * sizeof(double), host, (size_t)c->N * sizeof(double),
                              (size_t)c->N * sizeof(double), (size_t)ncols, cudaMemcpyHostToDevice, c->stream));
    VO_CUDA(cudaStreamSynchronize(c->stream));
    return VAMPOMI_OK;
}

int vampomi_download_columns(vampomi_ctx* c, long long j0, long long ncols, double* host) {
    VO_ARG(c && host && j0 >= 0 && ncols >= 0 && j0 + ncols <= c->M, "download_columns: range outside the shard");
    VO_CUDA(cudaSetDevice(c->device));
    if (ncols == 0) return VAMPOMI_OK;
    if (c->storage == VAMPOMI_STORE_F32) {                 // the rounded values, widened back to FP64
        long long chunk = (long long)((64ull << 20) / ((size_t)c->N * sizeof(double)));
        if (chunk < 1) chunk = 1;
        double* tmp = nullptr;
        VO_CUDA(cudaMalloc(&tmp, (size_t)(chunk < ncols ? chunk : ncols) * c->N * sizeof(double)));
        int rc = VAMPOMI_OK;
        for (long long j = 0; j < ncols && rc == VAMPOMI_OK; j += chunk) {
            const long long nc = ncols - j < chunk ? ncols - j : chunk;
            rc = launch_f32_to_f64(c, tmp, c->A32 + (size_t)(j0 + j) * c->ld, nc, c->stream);
            if (rc == VAMPOMI_OK && (cudaMemcpyAsync(host + (size_t)j * c->N, tmp, (size_t)nc * c->N * sizeof(double), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
                                     cudaStreamSynchronize(c->stream) != cudaSuccess)) {
                set_error("download_columns: device-to-host copy failed"); rc = VAMPOMI_ERR_CUDA;
            }
        }
        cudaFree(tmp);
        return rc;
    }
    VO_CUDA(cudaMemcpy2DAsync(host, (size_t)c->N * sizeof(double), c->A + (size_t)j0 * c->ld, c->ld * sizeof(double),
                              (size_t)c->N * sizeof(double), (size_t)ncols, cudaMemcpyDeviceToHost, c->stream));
    VO_CUDA(cudaStreamSynchronize(c->stream));
    return VAMPOMI_OK;
}

// The ingest path (data::read_methylation_data, src/data.cpp:116-153): T reader threads, each with a ring of `load_depth` pinned
// slots of 32 MB and its own copy stream — a slot is read from the file while the earlier ones are still on their way to HBM —
// column groups dealt round-robin. The pinned ring belongs to the CONTEXT and is allocated once (pinning 64 MB takes tens of
// milliseconds; a ring allocated inside the call, per thread, made the thread scaling erratic). Page-cache reads are a kernel
// memcpy per byte: several threads are needed to feed PCIe gen5 (~50 GB/s). With knob load_direct = 1 the file is opened with
// O_DIRECT and read in 4 KB-aligned spans straight into the pinned slots (no page-cache copy; the span's head and tail
// padding is skipped by the device copy), which is the path for files larger than host memory.
namespace {
constexpr size_t kLoadSlotBytes = 32ull << 20;
constexpr size_t kLoadAlign = 4096;
struct LoadRing {
    int threads = 0, depth = 0;
    std::vector<unsigned char*> slot;          // [threads][depth], each kLoadSlotBytes + 2 * kLoadAlign
    std::vector<double*> dslot;                // FP32 storage: dense FP64 staging on the device, rounded into place
    std::vector<cudaEvent_t> ev;
    std::vector<cudaStream_t> st;
};
}  // namespace

static void load_ring_free(vampomi_ctx* c) {
    LoadRing* r = static_cast<LoadRing*>(c->load_ring);
    if (!r) return;
    for (auto p : r->slot) if (p) cudaFreeHost(p);
    for (auto p : r->dslot) if (p) cudaFree(p);
    for (auto e : r->ev) if (e) cudaEventDestroy(e);
    for (auto s : r->st) if (s) cudaStreamDestroy(s);
    delete r;
    c->load_ring = nullptr;
}

static int load_ring_ensure(vampomi_ctx* c, int T, int depth) {
    LoadRing* r = static_cast<LoadRing*>(c->load_ring);
    if (r && r->threads >= T && r->depth >= depth) return VAMPOMI_OK;
    load_ring_free(c);
    r = new (std::nothrow) LoadRing();
    VO_ARG(r != nullptr, "load_file: out of host memory");
    c->load_ring = r;
    r->threads = T; r->depth = depth;
    r->slot.assign((size_t)T * depth, nullptr);
    r->dslot.assign((size_t)T * depth, nullptr);
    r->ev.assign((size_t)T * depth, nullptr);
    r->st.assign((size_t)T, nullptr);
    for (int t = 0; t < T; t++) VO_CUDA(cudaStreamCreateWithFlags(&r->st[t], cudaStreamNonBlocking));
    for (size_t i = 0; i < r->slot.size(); i++) {
        VO_CUDA(cudaMallocHost(&r->slot[i], kLoadSlotBytes + 2 * kLoadAlign));
        VO_CUDA(cudaEventCreateWithFlags(&r->ev[i], cudaEventDisableTiming));
        if (c->storage == VAMPOMI_STORE_F32) VO_CUDA(cudaMalloc(&r->dslot[i], kLoadSlotBytes));
    }
    return VAMPOMI_OK;
}

int vampomi_load_file(vampomi_ctx* c, const char* path) {
    VO_ARG(c && path, "load_file: NULL argument");
    VO_CUDA(cudaSetDevice(c->device));
    const bool direct = c->tune.load_direct != 0;
    int fd = open(path, direct ? (O_RDONLY | O_DIRECT) : O_RDONLY);
    if (fd < 0 && direct) fd = open(path, O_RDONLY);           // file systems without O_DIRECT (tmpfs): the buffered path
    if (fd < 0) { set_error("could not open methylation file %s", path); return VAMPOMI_ERR_IO; }
    const size_t col_bytes = (size_t)c->N * sizeof(double);
    struct stat sb;
    if (fstat(fd, &sb) != 0 || (size_t)sb.st_size < (size_t)(c->S + c->M) * col_bytes) {
        close(fd);
        set_error("%s is too short for N=%d and markers [%lld,%lld)", path, c->N, c->S, c->S + c->M);
        return VAMPOMI_ERR_IO;
    }
    const size_t file_size = (size_t)sb.st_size;
    long long cols_per_slot = (long long)(kLoadSlotBytes / col_bytes);
    if (cols_per_slot < 1) { close(fd); set_error("load_file: one column (%zu bytes) does not fit a staging slot", col_bytes); return VAMPOMI_ERR_ARG; }
    if (cols_per_slot > c->M) cols_per_slot = c->M;
    const long long nitems = (c->M + cols_per_slot - 1) / cols_per_slot;
    int T = c->tune.load_threads;
    if (T < 1) T = 1;
    if (T > 16) T = 16;
    if ((long long)T > nitems) T = (int)nitems;
    int depth = c->tune.load_depth;
    if (depth < 2) depth = 2;
    if (depth > 8) depth = 8;
    int rc_ring = load_ring_ensure(c, T, depth);
    if (rc_ring != VAMPOMI_OK) { close(fd); return rc_ring; }
    LoadRing* ring = static_cast<LoadRing*>(c->load_ring);
    depth = ring->depth;
    std::vector<int> rcs((size_t)T, VAMPOMI_OK);
    std::vector<std::string> errs((size_t)T);
    auto worker = [&](int t) {
        auto fail = [&](int code, const std::string& msg) { rcs[t] = code; errs[t] = msg; };
        if (cudaSetDevice(c->device) != cudaSuccess) return fail(VAMPOMI_ERR_CUDA, "cudaSetDevice failed in a loader thread");
        cudaStream_t st = ring->st[t];
        int k = 0;
        for (long long item = t; item < nitems; item += T, k = (k + 1) % depth) {
            const size_t si = (size_t)t * ring->depth + k;
            const long long j = item * cols_per_slot;
            const long long nc = c->M - j < cols_per_slot ? c->M - j : cols_per_slot;
            if (cudaEventSynchronize(ring->ev[si]) != cudaSuccess) { fail(VAMPOMI_ERR_CUDA, "event sync failed"); break; }   // slot free again?
            const size_t want = (size_t)nc * col_bytes;
            const size_t off = (size_t)(c->S + j) * col_bytes;                 // byte offset S*N*8, src/data.cpp:134
            // O_DIRECT wants offset, length and buffer aligned: read the enclosing 4 KB-aligned span, copy from inside it
            const size_t a0 = direct ? off / kLoadAlign * kLoadAlign : off;
            size_t a1 = direct ? (off + want + kLoadAlign - 1) / kLoadAlign * kLoadAlign : off + want;
            unsigned char* base = (unsigned char*)(((uintptr_t)ring->slot[si] + kLoadAlign - 1) / kLoadAlign * kLoadAlign);
            size_t got = 0, span = a1 - a0;
            bool ok = true;
            while (got < span) {
                ssize_t r = pread(fd, base + got, span - got, (off_t)(a0 + got));
                if (r < 0) { ok = false; break; }
                if (r == 0) break;                                             // end of file inside the padded tail of the last span
                got += (size_t)r;
            }
            if (!ok || a0 + got < off + want || (got < span && a0 + got < file_size)) { fail(VAMPOMI_ERR_IO, std::string("short read from ") + path); break; }
            const unsigned char* src = base + (off - a0);
            bool copied;
            if (c->storage == VAMPOMI_STORE_F32)
                copied = cudaMemcpyAsync(ring->dslot[si], src, want, cudaMemcpyHostToDevice, st) == cudaSuccess &&
                         launch_f64_to_f32(c, c->A32 + (size_t)j * c->ld, ring->dslot[si], nc, st) == VAMPOMI_OK;
            else if (c->ld == (size_t)c->N)                                    // no pad rows: one linear copy
                copied = cudaMemcpyAsync(c->A + (size_t)j * c->ld, src, want, cudaMemcpyHostToDevice, st) == cudaSuccess;
            else
                copied = cudaMemcpy2DAsync(c->A + (size_t)j * c->ld, c->ld * sizeof(double), src, col_bytes, col_bytes, (size_t)nc,
                                           cudaMemcpyHostToDevice, st) == cudaSuccess;
            if (!copied || cudaEventRecord(ring->ev[si], st) != cudaSuccess) { fail(VAMPOMI_ERR_CUDA, "host-to-device copy failed"); break; }
        }
        cudaStreamSynchronize(st);
    };
    std::vector<std::thread> th;
    for (int t = 1; t < T; t++) th.emplace_back(worker, t);
    worker(0);
    for (auto& x : th) x.join();
    close(fd);
    c->stats_ready = false;
    for (int t = 0; t < T; t++)
        if (rcs[t] != VAMPOMI_OK) { set_error("%s", errs[t].c_str()); return rcs[t]; }
    return VAMPOMI_OK;
}

int vampomi_generate_iid(vampomi_ctx* c, unsigned long long seed) {
    VO_ARG(c, "generate_iid: NULL context");
    VO_CUDA(cudaSetDevice(c->device));
    VO_CHECK(launch_generate_iid(c, seed));
    VO_CUDA(cudaStreamSynchronize(c->stream));
    c->stats_ready = false;
    return VAMPOMI_OK;
}

int vampomi_impute_missing(vampomi_ctx* c, long long counts[3]) {
    VO_ARG(c && counts, "impute_missing: NULL argument");
    VO_CUDA(cudaSetDevice(c->device));
    c->stats_ready = false;
    long long* part = reinterpret_cast<long long*>(c->red_partials);
    int nblocks = 0;
    VO_CHECK(launch_impute_missing(c, part, &nblocks));
    VO_CHECK(ensure_stage(c, (size_t)3 * nblocks));
    VO_CUDA(cudaMemcpyAsync(c->stage, part, (size_t)3 * nblocks * sizeof(long long), cudaMemcpyDeviceToHost, c->stream));
    VO_CUDA(cudaStreamSynchronize(c->stream));
    const long long* h = reinterpret_cast<const long long*>(c->stage);
    counts[0] = counts[1] = counts[2] = 0;
    for (int b = 0; b < nblocks; b++)
        for (int k = 0; k < 3; k++) counts[k] += h[3 * b + k];
    return VAMPOMI_OK;
}

int vampomi_compute_stats(vampomi_ctx* c, double alpha_scale) {
    VO_ARG(c, "compute_stats: NULL context");
    VO_CUDA(cudaSetDevice(c->device));
    VO_CHECK(launch_stats(c, alpha_scale));
    VO_CUDA(cudaStreamSynchronize(c->stream));
    c->stats_ready = true;
    // all ranks meet before the first operator call: the fused peer-memory exchange waits for its peers on the DEVICE with a
    // wall-clock limit, so a rank that loaded its shard much faster than the slowest one (cold disk, uneven blocks) must not
    // start that clock while the others are still reading
    return rank_barrier(c);
}

int vampomi_get_stats(vampomi_ctx* c, double* mave, double* msig) {
    VO_ARG(c && mave && msig, "get_stats: NULL argument");
    if (!c->stats_ready) { set_error("get_stats before compute_stats"); return VAMPOMI_ERR_STATE; }
    VO_CUDA(cudaSetDevice(c->device));
    VO_CHECK(d2h_vec(c, mave, c->mave, c->M));
    VO_CHECK(d2h_vec(c, msig, c->msig, c->M));
    return VAMPOMI_OK;
}

int vampomi_constant_columns(vampomi_ctx* c, unsigned char* const_M) {
    VO_ARG(c && const_M, "constant_columns: NULL argument");
    if (!c->stats_ready) { set_error("constant_columns before compute_stats"); return VAMPOMI_ERR_STATE; }
    VO_CUDA(cudaSetDevice(c->device));
    VO_CHECK(ensure_stage(c, (size_t)(c->M + 7) / 8));
    VO_CUDA(cudaMemcpyAsync(c->stage, c->mconst, (size_t)c->M, cudaMemcpyDeviceToHost, c->stream));
    VO_CUDA(cudaStreamSynchronize(c->stream));
    memcpy(const_M, c->stage, (size_t)c->M);
    return VAMPOMI_OK;
}

#define NEED_STATS(c, what) \
    do { if (!(c)->stats_ready) { set_error(what " before compute_stats"); return VAMPOMI_ERR_STATE; } } while (0)

int vampomi_atx(vampomi_ctx* c, const double* p_N, double* out_M) {
    VO_ARG(c && p_N && out_M, "atx: NULL argument");
    NEED_STATS(c, "atx");
    VO_CUDA(cudaSetDevice(c->device));
    double* p = c->nvec[VAMPOMI_V_TMP_N1 - 32];
    double* o = c->mvec[VAMPOMI_V_TMP_M1];
    VO_CHECK(h2d_vec(c, p, p_N, c->N));
    VO_CHECK(launch_atx(c, p, o, nullptr));
    VO_CHECK(d2h_vec(c, out_M, o, c->M));
    return VAMPOMI_OK;
}

int vampomi_ax(vampomi_ctx* c, const double* x_M, double* out_N) {
    VO_ARG(c && x_M && out_N, "ax: NULL argument");
    NEED_STATS(c, "ax");
    VO_CUDA(cudaSetDevice(c->device));
    double* x = c->mvec[VAMPOMI_V_TMP_M1];
    double* o = c->nvec[VAMPOMI_V_TMP_N1 - 32];
    VO_CHECK(h2d_vec(c, x, x_M, c->M));
    VO_CHECK(launch_ax(c, x, o, nullptr));
    VO_CHECK(d2h_vec(c, out_N, o, c->N));
    return VAMPOMI_OK;
}

// ---- vectors ----------------------------------------------------------------------------------------------------
int vampomi_vec_len(const vampomi_ctx* c, int vec, long long* len) {
    VO_ARG(c && len && vec_len(c, vec) >= 0, "vec_len: bad vector id %d", vec);
    *len = vec_len(c, vec);
    return VAMPOMI_OK;
}
int vampomi_vec_set(vampomi_ctx* c, int vec, const double* host) {
    VO_ARG(c && host && vec_ptr(c, vec), "vec_set: bad vector id %d or NULL buffer", vec);
    VO_CUDA(cudaSetDevice(c->device));
    return h2d_vec(c, vec_ptr(c, vec), host, vec_len(c, vec));
}
int vampomi_vec_get(vampomi_ctx* c, int vec, double* host) {
    VO_ARG(c && host && vec_ptr(c, vec), "vec_get: bad vector id %d or NULL buffer", vec);
    VO_CUDA(cudaSetDevice(c->device));
    return d2h_vec(c, host, vec_ptr(c, vec), vec_len(c, vec));
}
int vampomi_vec_get_scaled(vampomi_ctx* c, int vec, double divisor, double* host) {
    VO_ARG(c && host && vec_ptr(c, vec), "vec_get_scaled: bad vector id %d or NULL buffer", vec);
    VO_CUDA(cudaSetDevice(c->device));
    const bool m = is_mvec(vec);
    double* tmp = m ? c->mvec[VAMPOMI_V_TMP_M1] : c->nvec[VAMPOMI_V_TMP_N1 - 32];
    VO_CHECK(launch_scale_div(c, tmp, vec_ptr(c, vec), divisor, vec_len(c, vec), nullptr));
    return d2h_vec(c, host, tmp, vec_len(c, vec));
}
int vampomi_dump_begin(vampomi_ctx* c, int slot, int vec, double divisor) {
    VO_ARG(c && (slot == 0 || slot == 1) && vec_ptr(c, vec), "dump_begin: bad slot %d or vector id %d", slot, vec);
    if (c->dump_len[slot] > 0) { set_error("dump_begin: slot %d still holds a read-out that was not waited for", slot); return VAMPOMI_ERR_STATE; }
    VO_CUDA(cudaSetDevice(c->device));
    const long long n = vec_len(c, vec);
    VO_CHECK(ensure_dump(c));
    VO_CHECK(launch_scale_div(c, c->dump_dev[slot], vec_ptr(c, vec), divisor, n, nullptr));      // snapshot: vec may change right after
    // Default: the copy is stream-ordered on the context's own stream — it costs its PCIe time there (0.3 ms for 6.8 MB) but
    // no host round trip. Knob dump_stream = 1 puts it on the separate copy stream instead, underneath the following kernels;
    // measured on the 136 GB configuration, one GPU: +1.4 ms (default) vs +2.3 ms (copy stream) per iteration over a run
    // without dumps — next to kernels that saturate HBM the copy engine gains nothing.
    if (c->tune.dump_stream == 1) {
        VO_CUDA(cudaEventRecord(c->dump_ready[slot], c->stream));
        VO_CUDA(cudaStreamWaitEvent(c->copy_stream, c->dump_ready[slot], 0));
        VO_CUDA(cudaMemcpyAsync(c->dump_host[slot], c->dump_dev[slot], (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, c->copy_stream));
        VO_CUDA(cudaEventRecord(c->dump_done[slot], c->copy_stream));
    } else {
        VO_CUDA(cudaMemcpyAsync(c->dump_host[slot], c->dump_dev[slot], (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        VO_CUDA(cudaEventRecord(c->dump_done[slot], c->stream));
    }
    c->dump_len[slot] = n;
    return VAMPOMI_OK;
}
int vampomi_dump_wait(vampomi_ctx* c, int slot, double* host) {
    VO_ARG(c && (slot == 0 || slot == 1) && host, "dump_wait: bad slot %d or NULL buffer", slot);
    if (c->dump_len[slot] <= 0) { set_error("dump_wait: nothing pending in slot %d", slot); return VAMPOMI_ERR_STATE; }
    VO_CUDA(cudaSetDevice(c->device));
    VO_CUDA(cudaEventSynchronize(c->dump_done[slot]));
    memcpy(host, c->dump_host[slot], (size_t)c->dump_len[slot] * sizeof(double));
    c->dump_len[slot] = 0;
    return VAMPOMI_OK;
}
int vampomi_vec_fill(vampomi_ctx* c, int vec, double value) {
    VO_ARG(c && vec_ptr(c, vec), "vec_fill: bad vector id %d", vec);
    VO_CUDA(cudaSetDevice(c->device));
    return launch_fill(c, vec_ptr(c, vec), vec_len(c, vec), value);
}
int vampomi_vec_copy(vampomi_ctx* c, int dst, int src) {
    VO_ARG(c && vec_ptr(c, dst) && vec_ptr(c, src) && is_mvec(dst) == is_mvec(src), "vec_copy: bad vector ids %d <- %d", dst, src);
    VO_CUDA(cudaSetDevice(c->device));
    VO_CUDA(cudaMemcpyAsync(vec_ptr(c, dst), vec_ptr(c, src), (size_t)vec_len(c, dst) * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    return VAMPOMI_OK;
}
int vampomi_vec_lincomb(vampomi_ctx* c, int dst, double a, int x, double b, int y, double cdiv) {
    VO_ARG(c && vec_ptr(c, dst) && vec_ptr(c, x) && vec_ptr(c, y) && is_mvec(dst) == is_mvec(x) && is_mvec(dst) == is_mvec(y),
           "vec_lincomb: bad vector ids %d <- %d, %d", dst, x, y);
    VO_CUDA(cudaSetDevice(c->device));
    return launch_lincomb(c, vec_ptr(c, dst), a, vec_ptr(c, x), b, vec_ptr(c, y), cdiv, vec_len(c, dst));
}

int vampomi_dots(vampomi_ctx* c, int n, const int* kind, const int* a, const int* b, const double* scale, double* out) {
    VO_ARG(c && kind && a && b && out && n >= 1 && n <= MAX_DOTS, "dots: need 1..%d items", MAX_DOTS);
    VO_CUDA(cudaSetDevice(c->device));
    const double* pa[MAX_DOTS]; const double* pb[MAX_DOTS]; long long len[MAX_DOTS];
    bool any_m = false;
    for (int i = 0; i < n; i++) {
        VO_ARG(vec_ptr(c, a[i]) && vec_ptr(c, b[i]) && is_mvec(a[i]) == is_mvec(b[i]) && kind[i] >= 0 && kind[i] <= 2,
               "dots: item %d is malformed", i);
        pa[i] = vec_ptr(c, a[i]); pb[i] = vec_ptr(c, b[i]); len[i] = vec_len(c, a[i]);
        any_m |= is_mvec(a[i]);
    }
    VO_CHECK(launch_dots(c, n, kind, pa, pb, len, scale, c->sums));
    if (c->nranks > 1 && any_m) {
        // N-vector items are replicated: divide them by nranks after the packed sum so that one all-reduce serves all
        VO_CHECK(sum_over_ranks(c, c->sums, (size_t)n));
    }
    VO_CHECK(fetch_sums(c, n, false, out));
    if (c->nranks > 1 && any_m)
        for (int i = 0; i < n; i++) if (!is_mvec(a[i])) out[i] /= (double)c->nranks;
    return VAMPOMI_OK;
}

int vampomi_draw_probe(vampomi_ctx* c, unsigned long long seed, int it) {
    VO_ARG(c, "draw_probe: NULL context");
    VO_CUDA(cudaSetDevice(c->device));
    return launch_probe(c, seed, it);
}

static int fill_multi(vampomi_ctx* c, int K, const int* in_vecs, const int* out_vecs, bool in_is_m, MultiVec* mv) {
    VO_ARG(c && in_vecs && out_vecs && K >= 1 && K <= XCHG_KMAX, "multi: need 1..%d vectors", XCHG_KMAX);
    mv->K = K;
    for (int k = 0; k < XCHG_KMAX; k++) { mv->in[k] = nullptr; mv->out[k] = nullptr; mv->done[k] = nullptr; }
    for (int k = 0; k < K; k++) {
        VO_ARG(vec_ptr(c, in_vecs[k]) && vec_ptr(c, out_vecs[k]) && is_mvec(in_vecs[k]) == in_is_m && is_mvec(out_vecs[k]) != in_is_m,
               "multi: vector %d has the wrong kind", k);
        for (int q = 0; q < k; q++) VO_ARG(out_vecs[q] != out_vecs[k], "multi: output vectors must be distinct");
        mv->in[k] = vec_ptr(c, in_vecs[k]);
        mv->out[k] = vec_ptr(c, out_vecs[k]);
    }
    return VAMPOMI_OK;
}

int vampomi_ax_multi_dev(vampomi_ctx* c, int K, const int* x_vecs, const int* out_vecs) {
    MultiVec mv;
    VO_CHECK(fill_multi(c, K, x_vecs, out_vecs, true, &mv));
    NEED_STATS(c, "ax_multi_dev");
    VO_CUDA(cudaSetDevice(c->device));
    return launch_ax_multi(c, mv);
}

int vampomi_atx_multi_dev(vampomi_ctx* c, int K, const int* p_vecs, const int* out_vecs) {
    MultiVec mv;
    VO_CHECK(fill_multi(c, K, p_vecs, out_vecs, false, &mv));
    NEED_STATS(c, "atx_multi_dev");
    VO_CUDA(cudaSetDevice(c->device));
    return launch_atx_multi(c, mv);
}

int vampomi_aat_multi_dev(vampomi_ctx* c, int K, const int* q_vecs, const int* t_out_vecs, const int* w_out_vecs) {
    MultiVec mq;
    VO_ARG(K >= 1 && K <= 2 && w_out_vecs, "aat_multi_dev: 1 or 2 vectors");
    VO_CHECK(fill_multi(c, K, q_vecs, t_out_vecs, false, &mq));
    double* w_out[2] = {nullptr, nullptr};
    for (int k = 0; k < K; k++) {
        VO_ARG(vec_ptr(c, w_out_vecs[k]) && !is_mvec(w_out_vecs[k]) && w_out_vecs[k] != q_vecs[k] && (k == 0 || w_out_vecs[0] != w_out_vecs[1]),
               "aat_multi_dev: w_out must name distinct N-vectors other than q");
        w_out[k] = vec_ptr(c, w_out_vecs[k]);
    }
    NEED_STATS(c, "aat_multi_dev");
    if (!gram_supported(c)) { set_error("aat_multi_dev: the fused pass needs FP64 storage and N <= 40960"); return VAMPOMI_ERR_STATE; }
    VO_CUDA(cudaSetDevice(c->device));
    return launch_gram(c, mq, w_out);
}

int vampomi_aat_supported(const vampomi_ctx* c, int* yes) {
    VO_ARG(c && yes, "aat_supported: NULL argument");
    *yes = gram_supported(c) ? 1 : 0;
    return VAMPOMI_OK;
}

int vampomi_ax_dev(vampomi_ctx* c, int x_vec, int out_vec) {
    VO_ARG(c && is_mvec(x_vec) && vec_ptr(c, out_vec) && !is_mvec(out_vec), "ax_dev: need M-vector in, N-vector out");
    NEED_STATS(c, "ax_dev");
    VO_CUDA(cudaSetDevice(c->device));
    return launch_ax(c, vec_ptr(c, x_vec), vec_ptr(c, out_vec), nullptr);
}
int vampomi_atx_dev(vampomi_ctx* c, int p_vec, int out_vec) {
    VO_ARG(c && vec_ptr(c, p_vec) && !is_mvec(p_vec) && is_mvec(out_vec), "atx_dev: need N-vector in, M-vector out");
    NEED_STATS(c, "atx_dev");
    VO_CUDA(cudaSetDevice(c->device));
    return launch_atx(c, vec_ptr(c, p_vec), vec_ptr(c, out_vec), nullptr);
}

// ---- denoiser / EM / probit ----------------------------------------------------------------------------------------
static int fill_mix(MixParams& mp, const double* probs, const double* vars, int L) {
    VO_ARG(probs && vars && L >= 1 && L <= MAX_MIX, "mixture: need 1..%d components (got %d)", MAX_MIX, L);
    mp.L = L;
    for (int i = 0; i < MAX_MIX; i++) { mp.probs[i] = i < L ? probs[i] : 0.0; mp.vars[i] = i < L ? vars[i] : 0.0; }
    return VAMPOMI_OK;
}

int vampomi_denoise(vampomi_ctx* c, double gam1, const double* probs, const double* vars, int L, int damp, double rho,
                    double* sum_g1d) {
    VO_ARG(c && sum_g1d, "denoise: NULL argument");
    VO_CUDA(cudaSetDevice(c->device));
    MixParams mp;
    VO_CHECK(fill_mix(mp, probs, vars, L));
    VO_CHECK(launch_denoise(c, gam1, mp, damp, rho, c->sums));
    return fetch_sums(c, 1, true, sum_g1d);                         // MPI_Allreduce of sum_d, src/vamp.cpp:222
}

int vampomi_em_sums(vampomi_ctx* c, double gam1, double lambda, const double* omegas, const double* vars, int L, double* sums) {
    VO_ARG(c && sums, "em_sums: NULL argument");
    VO_ARG(L >= 2, "em_sums: needs at least 2 mixture components");
    VO_CUDA(cudaSetDevice(c->device));
    MixParams mp;
    VO_CHECK(fill_mix(mp, omegas, vars, L));
    VO_CHECK(launch_em_sums(c, gam1, lambda, mp, c->sums));
    return fetch_sums(c, 2 * L - 1, true, sums);                    // src/vamp.cpp:578,596,597 packed into one
}

int vampomi_probit_zdenoise(vampomi_ctx* c, double tau1, double* sum_g1d) {
    VO_ARG(c && sum_g1d, "probit_zdenoise: NULL argument");
    VO_CUDA(cudaSetDevice(c->device));
    VO_CHECK(launch_probit_z(c, tau1, c->sums));
    return fetch_sums(c, 1, false, sum_g1d);                        // N-vectors are replicated: no all-reduce
}

// ---- association tests ------------------------------------------------------------------------------------------
int vampomi_pvals_se(vampomi_ctx* c, const double* r1_M, double gam1, double* pvals_M) {
    VO_ARG(c && r1_M && pvals_M, "pvals_se: NULL argument");
    VO_CUDA(cudaSetDevice(c->device));
    double* r = c->mvec[VAMPOMI_V_TMP_M0];
    double* o = c->mvec[VAMPOMI_V_TMP_M1];
    VO_CHECK(h2d_vec(c, r, r1_M, c->M));
    VO_CHECK(launch_pvals_se(c, r, sqrt(1.0 / (gam1 * (double)c->N)), o));
    return d2h_vec(c, pvals_M, o, c->M);
}

int vampomi_loo_sums(vampomi_ctx* c, int w_vec, double* sums_3M) {
    VO_ARG(c && sums_3M && vec_ptr(c, w_vec) && !is_mvec(w_vec), "loo_sums: need an N-vector id");
    VO_CUDA(cudaSetDevice(c->device));
    double* dsums = nullptr;
    VO_CUDA(cudaMalloc(&dsums, (size_t)3 * c->M * sizeof(double)));
    int rc = launch_loo_sums(c, vec_ptr(c, w_vec), dsums);
    if (rc == VAMPOMI_OK) rc = d2h_vec(c, sums_3M, dsums, 3 * c->M);
    cudaFree(dsums);
    return rc;
}

// ---- instrumentation ---------------------------------------------------------------------------------------------
int vampomi_counters(vampomi_ctx* c, long long out[4], int reset) {
    VO_ARG(c && out, "counters: NULL argument");
    for (int i = 0; i < 4; i++) { out[i] = c->counters[i]; if (reset) c->counters[i] = 0; }
    return VAMPOMI_OK;
}

int vampomi_time_kernel(vampomi_ctx* c, int which, int reps, double* ms_avg) {
    VO_ARG(c && ms_avg && reps >= 1 && which >= 0 && which <= 10, "time_kernel: bad arguments");
    if (which != 2 && which != 4) NEED_STATS(c, "time_kernel");
    VO_CUDA(cudaSetDevice(c->device));
    cudaEvent_t e0, e1;
    VO_CUDA(cudaEventCreate(&e0));
    VO_CUDA(cudaEventCreate(&e1));
    double* dsums = nullptr;
    if (which == 3) VO_CUDA(cudaMalloc(&dsums, (size_t)3 * c->M * sizeof(double)));
    long long saved[4];
    memcpy(saved, c->counters, sizeof(saved));
    int rc = VAMPOMI_OK;
    VO_CUDA(cudaStreamSynchronize(c->stream));
    VO_CUDA(cudaEventRecord(e0, c->stream));
    for (int r = 0; r < reps && rc == VAMPOMI_OK; r++) {
        switch (which) {
            case 0: rc = launch_ax(c, c->mvec[VAMPOMI_V_TMP_M1], c->nvec[VAMPOMI_V_TMP_N1 - 32], nullptr); break;
            case 1: rc = launch_atx(c, c->nvec[VAMPOMI_V_TMP_N1 - 32], c->mvec[VAMPOMI_V_TMP_M1], nullptr); break;
            case 2: rc = launch_stats(c, 1.0); break;
            case 4: rc = launch_read_probe(c); break;
            case 5: case 6: case 7: case 8: {
                MultiVec mv{};
                mv.K = which == 7 ? 1 : which == 8 ? 3 : 2;
                if (which == 5 || which == 8) {
                    mv.in[0] = c->mvec[VAMPOMI_V_TMP_M1]; mv.in[1] = c->mvec[VAMPOMI_V_TMP_M0]; mv.in[2] = c->mvec[VAMPOMI_V_USER_M1];
                    mv.out[0] = c->nvec[VAMPOMI_V_TMP_N1 - 32]; mv.out[1] = c->nvec[VAMPOMI_V_TMP_N0 - 32]; mv.out[2] = c->nvec[VAMPOMI_V_USER_N1 - 32];
                    rc = launch_ax_multi(c, mv);
                } else {
                    mv.in[0] = c->nvec[VAMPOMI_V_TMP_N1 - 32]; mv.in[1] = c->nvec[VAMPOMI_V_TMP_N0 - 32];
                    mv.out[0] = c->mvec[VAMPOMI_V_TMP_M1]; mv.out[1] = c->mvec[VAMPOMI_V_TMP_M0];
                    rc = launch_atx_multi(c, mv);
                }
                break;
            }
            case 9: case 10: {
                MultiVec mq{};
                mq.K = which == 9 ? 2 : 1;
                mq.in[0] = c->nvec[VAMPOMI_V_TMP_N1 - 32]; mq.in[1] = c->nvec[VAMPOMI_V_TMP_N0 - 32];
                mq.out[0] = c->mvec[VAMPOMI_V_TMP_M1]; mq.out[1] = c->mvec[VAMPOMI_V_TMP_M0];
                double* w_out[2] = {c->nvec[VAMPOMI_V_GRAM_W0 - 32], c->nvec[VAMPOMI_V_GRAM_W1 - 32]};
                rc = launch_gram(c, mq, w_out);
                break;
            }
            default: rc = launch_loo_sums(c, c->nvec[VAMPOMI_V_TMP_N1 - 32], dsums); break;
        }
    }
    VO_CUDA(cudaEventRecord(e1, c->stream));
    VO_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    VO_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    *ms_avg = (double)ms / reps;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (dsums) cudaFree(dsums);
    memcpy(c->counters, saved, sizeof(saved));
    return rc;
}

int vampomi_profile_enable(vampomi_ctx* c, int on) {
    VO_ARG(c, "profile_enable: NULL context");
    VO_CUDA(cudaSetDevice(c->device));
    VO_CHECK(prof_resolve(c));
    c->profile = on != 0;
    return VAMPOMI_OK;
}

int vampomi_profile_read(vampomi_ctx* c, double out[9], int reset) {
    VO_ARG(c && out, "profile_read: NULL argument");
    VO_CUDA(cudaSetDevice(c->device));
    VO_CHECK(prof_resolve(c));
    for (int i = 0; i < 9; i++) { out[i] = c->prof_acc[i]; if (reset) c->prof_acc[i] = 0; }
    return VAMPOMI_OK;
}

int vampomi_profile_read_ex(vampomi_ctx* c, int nkinds, double* out, int reset) {
    VO_ARG(c && out && nkinds >= 1 && nkinds <= 4, "profile_read_ex: 1..4 kinds");
    VO_CUDA(cudaSetDevice(c->device));
    VO_CHECK(prof_resolve(c));
    for (int i = 0; i < 3 * nkinds; i++) { out[i] = c->prof_acc[i]; if (reset) c->prof_acc[i] = 0; }
    return VAMPOMI_OK;
}

int vampomi_stream(vampomi_ctx* c, void** stream) {
    VO_ARG(c && stream, "stream: NULL argument");
    *stream = (void*)c->stream;
    return VAMPOMI_OK;
}

long long vampomi_plan_chunks(long long slots, int ntiles, long long M, int min_cols, int balance) {
    if (slots < 1 || ntiles < 1 || M < 1) return 1;
    return balanced_chunks(slots, ntiles, M, min_cols, balance != 0);
}

int vampomi_set_tuning(vampomi_ctx* c, const char* name, int value) {
    VO_ARG(c && name, "set_tuning: NULL argument");
    struct { const char* n; int* p; int lo, hi; } knobs[] = {
        {"ax_rv", &c->tune.ax_rv, 0, 4},           {"ax_unroll", &c->tune.ax_unroll, 0, 8},
        {"ax_ctas_per_sm", &c->tune.ax_ctas_per_sm, 0, 32}, {"atx_cols", &c->tune.atx_cols, 0, 4},
        {"atx_unroll", &c->tune.atx_unroll, 0, 8}, {"atx_ctas_per_sm", &c->tune.atx_ctas_per_sm, 0, 32},
        {"cg_depth", &c->tune.cg_depth, 1, 32},     {"ax_impl", &c->tune.ax_impl, 0, 1},
        {"atx_impl", &c->tune.atx_impl, 0, 3},       {"xchg", &c->tune.xchg, 0, 1},
        {"load_threads", &c->tune.load_threads, 1, 16}, {"load_depth", &c->tune.load_depth, 2, 8}, {"load_direct", &c->tune.load_direct, 0, 1}, {"ld_hint", &c->tune.ld_hint, 0, 3},
        {"interleave", &c->tune.interleave, 0, 1},       {"center_split", &c->tune.center_split, 0, 1},
        {"grid_balance", &c->tune.grid_balance, 0, 1},   {"dump_stream", &c->tune.dump_stream, 0, 1},
        {"xchg_ll", &c->tune.xchg_ll, 0, 1},             {"multi_ax_occ", &c->tune.multi_ax_occ, 0, 3},
        {"multi_ax_rv", &c->tune.multi_ax_rv, 0, 2},     {"multi_ax_unroll", &c->tune.multi_ax_unroll, 0, 8},
        {"multi_atx_impl", &c->tune.multi_atx_impl, 0, 1}, {"multi_atx_cols", &c->tune.multi_atx_cols, 0, 4},
        {"multi_atx_unroll", &c->tune.multi_atx_unroll, 0, 4}, {"multi_atx_tile", &c->tune.multi_atx_tile, 0, 16384},
        {"cg_onepass", &c->tune.cg_onepass, 0, 1},       {"gram_shape", &c->tune.gram_shape, 0, 18},         {"gram_prefetch", &c->tune.gram_prefetch, 0, 64},
        {"gram_cluster", &c->tune.gram_cluster, 0, 16},
        {"gram_clusters", &c->tune.gram_clusters, 0, 4096}, {"gram_refresh", &c->tune.gram_refresh, 0, 100000},
    };
    for (auto& k : knobs)
        if (!strcmp(k.n, name)) {
            VO_ARG(value >= k.lo && value <= k.hi, "set_tuning: %s must be in [%d,%d]", name, k.lo, k.hi);
            *k.p = value;
            c->xchg.enabled = (c->xchg_ready && c->tune.xchg) ? 1 : 0;
            c->xchg.ll = c->tune.xchg_ll ? 1 : 0;
            return VAMPOMI_OK;
        }
    set_error("set_tuning: unknown knob %s", name);
    return VAMPOMI_ERR_ARG;
}

}  // extern "C"
