// ONE read of the marker block per conjugate-gradient iteration: t = A^T q and w = A t in the same pass.
//
// The operator of the LMMSE solve is tau*A^T A + gam2*I (vamp::lmmse_mult, src/vamp.cpp:645-662): the reference applies it
// as ATx(Ax(p)) (:653-654), two sweeps over the marker block, and so does the two-pass schedule here. The same CG can be
// advanced with ONE sweep per iteration: keep q = A p as a vector of its own (its recurrence follows from p = z + beta p,
// cg.cu), and let the sweep deliver both t = A^T q (what the iteration needs as A^T A p) and w = A t = A A^T q (what the
// recurrence of q needs). For a marker-major matrix these two products FUSE column by column:
//
//     t_j = msig_j * <a_j - mave_j, q> / sqrt(N)              data::dot_product, src/data.cpp:294-313
//     w  += (a_j - mave_j) * (msig_j * t_j)                   inner loop of data::Ax, src/data.cpp:349-362
//
// Column j is needed twice, but only a dot product apart — so it is kept ON CHIP between the two uses instead of being read
// from HBM again. One column is N*8 = 160 kB at N = 20 000, too much for one SM next to q and w, so a thread-block CLUSTER of
// CS = ceil(ld / ROWS) CTAs (1 ... 16) owns a chunk of columns: CTA r holds rows [r*tile, (r+1)*tile) of q and of w in
// registers. The chunk is walked in steps of C = 2 columns.
//
// A CTA is three warpgroups (THREADS = 384): two of compute warps (NCW = 8) and one SERVICE warpgroup — the communication warp,
// the producer warp and two warps that only hand their registers over. Registers are allotted at launch as if every warp needed
// the same (168 per thread); `setmaxnreg` then moves them: the service warpgroup drops to 96, the compute warpgroups rise to 200,
// which their 5 row pairs of q, w and two steps of columns need, plus the first PF row pairs of the next step (loaded ahead,
// below). Eight compute warps put two on every scheduler.
//
// The columns arrive through a RING of R = 4 stages in shared memory. Each stage holds one step: ONE cp.async.bulk.tensor.3d
// (SASS UTMALDG) per step brings both column pieces of the CTA's row tile (box 16 x tile/16 x C of the {16, ld/16, M} view of
// the block; rows past the end of a column arrive as zeros), completing on the stage's mbarrier; the producer's lanes < C store
// the step's two column means beside it. One issuing warp gets a bulk copy under way only every ~500-650 cycles, whatever its
// size, so one copy per step — not one per column piece — and a warp of its own that refills a stage the moment every compute
// warp has read it, whatever the exchange is doing.
//
// Step s, u = s % 4 (ring stage, exchange slot and barrier; the step loops are unrolled by four, so u is a compile-time offset
// from one shared-window base register and the barrier parity is one bit flipped per trip):
//   compute warp:        LDS the rest of its row pairs of stage u, centre them, dot with q -> add the lane quadruples {l, l^8,
//                        l^16, l^24} (two shuffle levels) -> red[u & 1], arrive on redbar[u];
//                        wait ringbar[(s+1) & 3] -> LDS the column means and the first PF row pairs of step s + 1 (LOADED AHEAD:
//                        they arrive while the axpy below runs, so the next dot starts on data in registers);
//                        wait wready[(s-1) & 3] -> read the weights -> axpy of step s - 1 on the registers that still hold its
//                        centred columns (the axpy is DEFERRED by one step: a compute warp never waits for the cluster round
//                        trip of the step it just dotted, only for the one before it)
//   producer warp:       wait redbar[u] (every compute warp has read stage u: the arrival follows the dot, which consumed the
//                        loads of step s made one phase earlier as well as its own) -> refill stage u with step s + 4
//   communication warp:  wait redbar[u] -> add the NCW warp sums (fixed tree) and the three shuffle levels left -> st.async the
//                        CTA's partial sums to every CTA of the cluster (slot u) -> wait full[u] -> add the CS ranks' partial
//                        sums by a fixed tree -> t_j (cluster rank 0 stores it) and the weight msig_j * t_j -> wbuf[u], arrive
//                        on wready[u], re-arm full[u] for step s + 4
// Every partial sum travels as ONE st.async: an 8-byte store into the peer's shared memory that also completes 8 bytes on the
// peer's mbarrier, so data and arrival are one message and nothing in the loop is a cluster-wide barrier. Four slots make reuse
// safe: a CTA can only send step s + 4 after it has received step s + 3 from everybody, which every peer sends after it has
// consumed step s. red[] has two slots: a compute warp overwrites the slot of step s (at step s + 2) only after it has waited
// for the weights of step s, which the communication warp publishes after reading the slot. Every CTA adds the same values in
// the same order, so all CTAs of a cluster compute bitwise the same t_j.
//
// Output: t (M-vector, written by cluster rank 0) and the per-chunk partials of w, which go through the same k_ax_reduce_multi
// (fixed-order reduction + fused peer-memory all-reduce + 1/sqrt(N)) as the A x passes.
// Algorithmic bytes per launch: N*M_local*8, for t AND w, for up to two systems.
// How this layout was reached, and the variants it replaced, with their measurements: DESIGN.md §3b.
#include <cuda.h>                                               // CUtensorMap (type only: the encoder is fetched through cudaGetDriverEntryPoint)

#include "common.h"

namespace vampomi {

namespace {

struct GramVec {
    const double* q[2];                // in: N-vectors (zero-padded to ld)
    double* t[2];                      // out: M-vectors, t = A^T q
    const int* done[2];                // "skip me" flags (nullptr = always active)
};

// layout of a CTA, shared by the kernel and its launcher
constexpr int GRAM_NCW = 8;                                      // compute warps: two warpgroups
constexpr int GRAM_RP = 5;                                       // 16-byte row pairs per compute thread
constexpr int GRAM_C = 2;                                        // columns per step
constexpr int GRAM_R = 4;                                        // ring stages
constexpr int GRAM_PF = 4;                                       // row pairs of the next step loaded during the axpy
constexpr int GRAM_THREADS = (GRAM_NCW + 4) * 32;                // + the service warpgroup: 384
constexpr int GRAM_ROWS = GRAM_NCW * 32 * GRAM_RP * 2;           // rows per CTA: 2 560

// Shared-memory operations on 32-bit shared-window addresses: inside a cluster launch the compiler re-derives the window base of
// every __shared__ object from SR_CgaCtaId at each use (S2R + LEA per access), so the kernel computes its addresses once.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t opaque_u32(uint32_t x) {       // keeps the compiler from re-deriving such an address at every use
    asm volatile("" : "+r"(x));
    return x;
}
// address of the same shared-memory location in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
// 8-byte store into a peer CTA's shared memory that also counts 8 bytes on the peer's mbarrier: data and arrival in one message
__device__ __forceinline__ void st_async_f64(uint32_t raddr, double v, uint32_t rbar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];"
                 ::"r"(raddr), "l"(__double_as_longlong(v)), "r"(rbar) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init_u(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_u(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cta_u(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_cta_u(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// one try_wait and one branch on the fast path; the spin counter only exists on the slow path
__device__ __forceinline__ void mbar_spin_cta_u(uint32_t bar, uint32_t parity) {
    if (mbar_try_cta_u(bar, parity)) return;
    uint32_t spins = 0;
    while (!mbar_try_cta_u(bar, parity))
        if (++spins > (1u << 28)) __trap();                      // a protocol bug must fault, not hang the GPU
}
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ double2 lds_f64x2(uint32_t addr) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_f64(uint32_t addr, double v) {
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}

// Pairwise (tree) sum of N values held in registers: depth log2(N) instead of N - 1 dependent additions — what the
// communication warp's latency chain wants; the order is fixed, so every CTA adds the same values the same way.
template <int N>
__device__ __forceinline__ double tree_sum(const double (&v)[N]) {
    if constexpr (N == 1) {
        return v[0];
    } else {
        double h[(N + 1) / 2];
#pragma unroll
        for (int i = 0; i < N / 2; i++) h[i] = v[2 * i] + v[2 * i + 1];
        if constexpr ((N & 1) != 0) h[N / 2] = v[N - 1];
        return tree_sum<(N + 1) / 2>(h);
    }
}

// Sums of NV (2 or 4) values over the lane quadruples {l, l^8, l^16, l^24}: at each level a lane hands half of its values to its
// partner and keeps the sums of the other half, so lane l is left with the quadruple's sum of value l / (32 / NV). The levels
// 4, 2, 1 that remain are the same for every NV; the communication warp adds them.
template <int NV>
__device__ __forceinline__ double quad_sum_multi(const double (&v)[NV], int lane) {
    static_assert(NV == 2 || NV == 4, "2 or 4 values");
    const bool up16 = (lane & 16) != 0;
    if constexpr (NV == 4) {
        const bool up8 = (lane & 8) != 0;
        const double a0 = (up16 ? v[2] : v[0]) + __shfl_xor_sync(0xffffffffu, up16 ? v[0] : v[2], 16);
        const double a1 = (up16 ? v[3] : v[1]) + __shfl_xor_sync(0xffffffffu, up16 ? v[1] : v[3], 16);
        return (up8 ? a1 : a0) + __shfl_xor_sync(0xffffffffu, up8 ? a0 : a1, 8);
    } else {
        const double t = (up16 ? v[1] : v[0]) + __shfl_xor_sync(0xffffffffu, up16 ? v[0] : v[1], 16);
        return t + __shfl_xor_sync(0xffffffffu, t, 8);
    }
}

// K systems (1 or 2), CS CTAs per cluster (1 ... 16). Warps 0 ... NCW-1 compute; warp NCW communicates, warp NCW+1 produces.
template <int K, int CS>
__global__ void __launch_bounds__(GRAM_THREADS, 1) k_gram_wsx(const double* __restrict__ A, size_t ld, const double* __restrict__ mave,
                                                             const double* __restrict__ msig, GramVec gv, int tile_rows, int cols_per_chunk,
                                                             long long M, double scale, double* __restrict__ partial, int nchunks,
                                                             const __grid_constant__ CUtensorMap tmap) {
    constexpr int NCW = GRAM_NCW, RP = GRAM_RP, C = GRAM_C, R = GRAM_R, PF = GRAM_PF;
    static_assert(PF <= C * RP, "at most one step ahead");
    constexpr int CK = C * K, LPV = 32 / CK, CT = NCW * 32, PIECE = CT * RP * 2;
    static_assert(C == 2 && (K == 1 || K == 2), "two columns per step: their means are one 16-byte load, their sums one or two value pairs");
    static_assert(CS <= 2 * LPV, "after the butterfly the LPV lanes that hold value ck send it to the CS ranks, at most two each");
    // one control block, addressed as base register + compile-time offset (bytes)
    constexpr uint32_t XSLOT = CS * CK * 8;                      // xbuf[4][CS][CK]: partial sums of the ranks, per exchange slot
    constexpr uint32_t XBUF_O = 0, WBUF_O = XBUF_O + 4 * XSLOT;  // wbuf[4][CK]: axpy weights of a step
    constexpr uint32_t MST_O = WBUF_O + 4 * CK * 8;              // mst[R][C]: column means of a ring stage
    constexpr uint32_t FULL_O = MST_O + R * C * 8, WREADY_O = FULL_O + 32, REDBAR_O = WREADY_O + 32, RINGBAR_O = REDBAR_O + 32;
    // red[2][NCW][32 lanes]: every compute warp's quadruple sums, as they are
    constexpr uint32_t RED_O = RINGBAR_O + R * 8;
    constexpr uint32_t REDSLOT = NCW * 256, CTL_BYTES = RED_O + 2 * REDSLOT;
    static_assert(RED_O % 16 == 0, "16-byte stores");
    extern __shared__ __align__(128) double ring[];              // [R][C][PIECE]
    __shared__ __align__(16) unsigned char ctl[CTL_BYTES];
    bool active[K];
    bool any = false;
#pragma unroll
    for (int k = 0; k < K; k++) { active[k] = gv.done[k] == nullptr || *gv.done[k] == 0; any |= active[k]; }
    if (!any) return;                                            // identical decision in every CTA of the cluster
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    uint32_t crank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
    const size_t rbase = (size_t)crank * tile_rows;
    const long long c0 = (long long)blockIdx.y * cols_per_chunk;
    long long c1 = c0 + cols_per_chunk;
    if (c1 > M) c1 = M;
    // steps and column offsets are 32-bit: a chunk has far fewer than 2^31 columns
    const int ncols = c1 > c0 ? (int)(c1 - c0) : 0;
    const int nsteps = (ncols + C - 1) / C;
    const double* const mave_c = mave + c0;
    const double* const msig_c = msig + c0;
    auto col_of = [&](int s, int cc) { const int j = s * C + cc; return j < ncols ? j : ncols - 1; };   // ragged last step: its last column again
    // a stage holds the C column pieces back to back, tile_rows rows each; the stage's tail behind them is never written by a copy,
    // so it is zeroed once: every compute thread can then load its row pairs unconditionally — a zero row has q = 0 and its w is
    // never stored
    for (int i = C * tile_rows + tid; i < C * PIECE; i += blockDim.x)
#pragma unroll
        for (int st = 0; st < R; st++) ring[(size_t)st * C * PIECE + i] = 0.0;
    const uint32_t cb = opaque_u32(smem_u32(ctl)), ring_u = opaque_u32(smem_u32(ring));
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            mbar_init_u(cb + FULL_O + 8 * i, 1); mbar_init_u(cb + WREADY_O + 8 * i, 1);
            mbar_init_u(cb + REDBAR_O + 8 * i, NCW); mbar_init_u(cb + RINGBAR_O + 8 * i, 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int i = 0; i < 4; i++) mbar_expect_tx_u(cb + FULL_O + 8 * i, XSLOT);
    }
    __syncthreads();
    cluster_sync_all();                                          // every CTA's mbarriers are armed before anybody sends

    if (wid >= NCW) {
        // ----------------------------------------------- service warpgroup -----------------------------------------------
        asm volatile("setmaxnreg.dec.sync.aligned.u32 96;");
        if (wid == NCW + 1) {
            // producer warp. The column means travel beside the copy: lanes < C fetch them before waiting for the stage and store
            // them before lane 0 arrives on its barrier.
            const int row16 = (int)(rbase >> 4), box_bytes = C * tile_rows * 8;
            auto issue_tensor = [&](int s, int st, double mv) {
                if (lane < C) sts_f64(cb + MST_O + (uint32_t)((st * C + lane) * 8), mv);
                __syncwarp();
                if (lane == 0) {
                    const uint32_t bar = cb + RINGBAR_O + 8 * st;
                    mbar_expect_tx_u(bar, (uint32_t)box_bytes);
                    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                                 ::"r"(ring_u + (uint32_t)(st * C * PIECE * 8)), "l"(&tmap), "r"(0), "r"(row16), "r"((int)(c0 + (long long)s * C)), "r"(bar) : "memory");
                }
            };
            auto mean_of = [&](int s) { return lane < C ? __ldg(mave_c + col_of(s, lane)) : 0.0; };
            for (int s = 0; s < R && s < nsteps; s++) issue_tensor(s, s, mean_of(s));
            uint32_t php = 0;
            for (int s0 = 0; s0 + R < nsteps; s0 += 4, php ^= 1u) {
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int s = s0 + u;
                    if (s + R >= nsteps) break;
                    const double mv = mean_of(s + R);
                    mbar_spin_cta_u(cb + REDBAR_O + 8 * u, php);
                    issue_tensor(s + R, u, mv);
                }
            }
        }
        if (wid <= NCW) {
            // communication warp: wid == NCW (warps NCW + 2 and NCW + 3 only hand their registers over)
            const int ck = lane / LPV, dst = lane % LPV, cc_l = ck / K, k_l = ck % K;   // after the butterfly lanes [ck*LPV, (ck+1)*LPV) hold value ck
            bool act = active[0];
#pragma unroll
            for (int k = 1; k < K; k++) act = k_l == k ? active[k] : act;
            double* tout = K > 1 && k_l == 1 ? gv.t[K - 1] : gv.t[0];
            double sg_next = nsteps > 0 ? __ldg(msig_c + col_of(0, cc_l)) : 0.0;
            const uint32_t peer = (uint32_t)(dst < CS ? dst : 0), peer2 = (uint32_t)(dst + LPV < CS ? dst + LPV : 0);   // 16-CTA clusters: two ranks per lane
            const uint32_t rx = mapa_u32(cb + XBUF_O + (crank * CK + ck) * 8, peer), rf = mapa_u32(cb + FULL_O, peer);
            const uint32_t rx2 = mapa_u32(cb + XBUF_O + (crank * CK + ck) * 8, peer2), rf2 = mapa_u32(cb + FULL_O, peer2);
            const uint32_t xb_l = cb + XBUF_O + (uint32_t)ck * 8u, wb_l = cb + WBUF_O + (uint32_t)ck * 8u;
            uint32_t ph = 0;                                     // (s / 4) & 1: phase parity of every four-deep barrier ring
            for (int s0 = 0; s0 < nsteps; s0 += 4, ph ^= 1u) {
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int s = s0 + u;
                    if (s >= nsteps) break;
                    const double sgl = sg_next;
                    sg_next = __ldg(msig_c + col_of(s + 1 < nsteps ? s + 1 : s, cc_l));
                    mbar_spin_cta_u(cb + REDBAR_O + 8 * u, ph);   // every compute warp has read stage u and stored its partial sums
                    // the CTA's partial sum of value ck: the warps by a fixed tree, then the lane levels 4, 2, 1
                    double pw[NCW];
#pragma unroll
                    for (int w = 0; w < NCW; w++) pw[w] = lds_f64(cb + RED_O + (uint32_t)((u & 1) * REDSLOT + w * 256) + (uint32_t)lane * 8u);
                    double sw = tree_sum<NCW>(pw);
                    sw += __shfl_xor_sync(0xffffffffu, sw, 4);
                    sw += __shfl_xor_sync(0xffffffffu, sw, 2);
                    sw += __shfl_xor_sync(0xffffffffu, sw, 1);
                    if (dst < CS) st_async_f64(rx + u * XSLOT, sw, rf + 8 * u);
                    if (CS > LPV && dst + LPV < CS) st_async_f64(rx2 + u * XSLOT, sw, rf2 + 8 * u);
                    // the ranks' values arrive as st.async transactions ON this barrier (data and count are one message), so the
                    // CTA-scope wait orders them; the cluster-scope acquire form would cost an L1 invalidation (CCTL.IVALL) per step
                    mbar_spin_cta_u(cb + FULL_O + 8 * u, ph);
                    // every lane adds the CS partial sums of its value by the same fixed tree: bitwise the same t_j in every CTA
                    double pr[CS];
#pragma unroll
                    for (int r = 0; r < CS; r++) pr[r] = lds_f64(xb_l + (uint32_t)(u * XSLOT + r * CK * 8));
                    const double tot = tree_sum<CS>(pr);
                    const int j = s * C + cc_l;
                    const double tj = (sgl * tot) * scale;                      // sigma_inv * dpa (:306), then * scale (:330)
                    const bool live = j < ncols && act;
                    if (dst == 0) {
                        if (crank == 0 && live) tout[c0 + j] = tj;
                        sts_f64(wb_l + (uint32_t)(u * CK * 8), live ? sgl * tj : 0.0);   // sig_phen_i = msig * x, src/data.cpp:354
                    }
                    __syncwarp();
                    if (lane == 0) {
                        mbar_arrive_cta_u(cb + WREADY_O + 8 * u);
                        mbar_expect_tx_u(cb + FULL_O + 8 * u, XSLOT);           // re-arm the slot for step s + 4
                    }
                }
            }
        }
    } else {
        // ---------------------------------------------- compute warps ----------------------------------------------
        asm volatile("setmaxnreg.inc.sync.aligned.u32 200;");
        bool valid[RP];
        double qr[K][RP][2], acc[K][RP][2];
#pragma unroll
        for (int i = 0; i < RP; i++) {
            const int off = (i * CT + tid) * 2;
            valid[i] = off < tile_rows && rbase + off < ld;
#pragma unroll
            for (int k = 0; k < K; k++) {
                acc[k][i][0] = acc[k][i][1] = 0.0;
                double2 qv = make_double2(0.0, 0.0);
                if (valid[i] && active[k]) qv = *reinterpret_cast<const double2*>(gv.q[k] + rbase + off);   // pad rows of q are zero
                qr[k][i][0] = qv.x; qr[k][i][1] = qv.y;
            }
        }
        double a[2][C][RP][2];                                   // the step being dotted and the step whose axpy is pending
        const uint32_t rows_u = opaque_u32(ring_u + (uint32_t)tid * 16u);             // this thread's first row pair inside a ring stage
        const uint32_t col_stride = (uint32_t)tile_rows * 8u;                         // bytes between the column pieces of a stage

        // The registers left beside q, w and two steps of columns hold PF row pairs: the next step's first ones and its column
        // means are loaded while the axpy of the step before runs (a full step ahead would need ~240 registers)
        double2 nx[PF], nm;
        auto load_ahead = [&](const int u, const uint32_t par) {   // u: ring stage of the step, par: its barrier parity
            mbar_spin_cta_u(cb + RINGBAR_O + 8 * u, par);
            nm = lds_f64x2(cb + MST_O + (uint32_t)(u * C * 8));
#pragma unroll
            for (int p = 0; p < PF; p++)
                nx[p] = lds_f64x2(rows_u + (uint32_t)((u * C * PIECE + (p % RP) * CT * 2) * 8) + (uint32_t)(p / RP) * col_stride);
        };
        auto dot_step = [&](const int u) {                       // u = s % 4: ring stage, barrier; u & 1: register buffer, red slot
            double pd[C][K][2];
#pragma unroll
            for (int cc = 0; cc < C; cc++)
#pragma unroll
                for (int k = 0; k < K; k++) pd[cc][k][0] = pd[cc][k][1] = 0.0;
            const double m[2] = {nm.x, nm.y};
#pragma unroll
            for (int cc = 0; cc < C; cc++)
#pragma unroll
                for (int i = 0; i < RP; i++) {
                    // rows beyond the tile read zeros or the next column's first rows: they only meet q = 0 and unsaved sums
                    const double2 v = cc * RP + i < PF ? nx[cc * RP + i]
                                                       : lds_f64x2(rows_u + (uint32_t)((u * C * PIECE + i * CT * 2) * 8) + (uint32_t)cc * col_stride);
                    const double d0 = v.x - m[cc], d1 = v.y - m[cc];            // meth[i] - mu, src/data.cpp:304 and :360
                    a[u & 1][cc][i][0] = d0; a[u & 1][cc][i][1] = d1;           // kept centred for the deferred axpy
#pragma unroll
                    for (int k = 0; k < K; k++) {
                        pd[cc][k][0] = fma(d0, qr[k][i][0], pd[cc][k][0]);
                        pd[cc][k][1] = fma(d1, qr[k][i][1], pd[cc][k][1]);
                    }
                }
            double v[CK];
#pragma unroll
            for (int cc = 0; cc < C; cc++)
#pragma unroll
                for (int k = 0; k < K; k++) v[cc * K + k] = pd[cc][k][0] + pd[cc][k][1];
            sts_f64(cb + RED_O + (uint32_t)((u & 1) * REDSLOT + wid * 256) + (uint32_t)lane * 8u, quad_sum_multi<CK>(v, lane));
            __syncwarp();
            if (lane == 0) mbar_arrive_cta_u(cb + REDBAR_O + 8 * u);
        };
        auto axpy_step = [&](const int slot, const uint32_t par, const int b) {
            mbar_spin_cta_u(cb + WREADY_O + 8 * slot, par);
            double wgt[CK];
#pragma unroll
            for (int i = 0; i < CK; i += 2) {
                const double2 w2 = lds_f64x2(cb + WBUF_O + (uint32_t)((slot * CK + i) * 8));
                wgt[i] = w2.x; wgt[i + 1] = w2.y;
            }
#pragma unroll
            for (int cc = 0; cc < C; cc++)
#pragma unroll
                for (int i = 0; i < RP; i++)
#pragma unroll
                    for (int k = 0; k < K; k++) {
                        acc[k][i][0] = fma(a[b][cc][i][0], wgt[cc * K + k], acc[k][i][0]);
                        acc[k][i][1] = fma(a[b][cc][i][1], wgt[cc * K + k], acc[k][i][1]);
                    }
        };
        uint32_t ph = 0;
        if (nsteps > 0) load_ahead(0, 0);
        for (int s0 = 0; s0 <= nsteps; s0 += 4, ph ^= 1u) {
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int s = s0 + u;
                if (s < nsteps) dot_step(u);
                if (s + 1 < nsteps) load_ahead((u + 1) & 3, u == 3 ? ph ^ 1u : ph);                    // step s + 1
                if (s >= 1 && s <= nsteps) axpy_step((u + 3) & 3, u == 0 ? ph ^ 1u : ph, (u + 1) & 1);   // step s - 1
            }
        }
#pragma unroll
        for (int k = 0; k < K; k++) {
            if (!active[k]) continue;
            double* prow = partial + ((size_t)k * nchunks + blockIdx.y) * ld + rbase;
#pragma unroll
            for (int i = 0; i < RP; i++)
                if (valid[i]) *reinterpret_cast<double2*>(prow + (i * CT + tid) * 2) = make_double2(acc[k][i][0], acc[k][i][1]);
        }
    }
    cluster_sync_all();                                          // nobody leaves while a peer may still write into its shared memory
}

// {16, ld/16, M} view of the column-major marker block (a column = ld/16 groups of 16 rows) with a box of one CTA's row tile of C
// columns: 16 x tile_rows/16 x C doubles land in shared memory as C contiguous column pieces. Cached in the context.
int gram_tensor_map(vampomi_ctx* c, int tile_rows, int C, CUtensorMap* out) {
    if (c->gram_tmap_A != (const void*)c->A || c->gram_tmap_ld != c->ld || c->gram_tmap_M != c->M || c->gram_tmap_rows != tile_rows || c->gram_tmap_C != C) {
        typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                     CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
        static const EncodeFn encode = [] {                      // resolved once (thread-safe: the rank threads of main_meth --gpus share it)
            void* fn = nullptr;
            cudaDriverEntryPointQueryResult qres;
            if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess) { cudaGetLastError(); fn = nullptr; }
            return (EncodeFn)fn;
        }();
        if (encode == nullptr) { set_error("gram: cuTensorMapEncodeTiled is not available from this driver"); return VAMPOMI_ERR_CUDA; }
        if (c->ld % 16 != 0 || tile_rows % 16 != 0 || tile_rows / 16 > 256) { set_error("gram: tensor map needs ld and the row tile in multiples of 16 rows, at most 4096 rows per tile"); return VAMPOMI_ERR_ARG; }
        const cuuint64_t dims[3] = {16, (cuuint64_t)(c->ld / 16), (cuuint64_t)c->M};
        const cuuint64_t strides[2] = {16 * sizeof(double), (cuuint64_t)c->ld * sizeof(double)};
        const cuuint32_t box[3] = {16, (cuuint32_t)(tile_rows / 16), (cuuint32_t)C};
        const cuuint32_t estr[3] = {1, 1, 1};
        CUtensorMap tm;
        const CUresult r = encode(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, (void*)c->A, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("gram: cuTensorMapEncodeTiled failed (%d) for ld=%zu M=%lld tile_rows=%d", (int)r, c->ld, c->M, tile_rows); return VAMPOMI_ERR_CUDA; }
        static_assert(sizeof(CUtensorMap) == sizeof(c->gram_tmap), "CUtensorMap is 128 bytes");
        memcpy(c->gram_tmap, &tm, sizeof(tm));
        c->gram_tmap_A = (const void*)c->A; c->gram_tmap_ld = c->ld; c->gram_tmap_M = c->M; c->gram_tmap_rows = tile_rows; c->gram_tmap_C = C;
    }
    memcpy(out, c->gram_tmap, sizeof(*out));
    return VAMPOMI_OK;
}

template <int K, int CS>
int gram_launch(vampomi_ctx* c, const GramVec& gv, const MultiVec& mw) {
    constexpr int C = GRAM_C;
    const size_t smem = (size_t)GRAM_R * C * GRAM_ROWS * sizeof(double);
    const auto kern = k_gram_wsx<K, CS>;
    const size_t tr = (c->ld + CS - 1) / CS;
    const int tile_rows = (int)((tr + 15) / 16 * 16);
    CUtensorMap tm;
    VO_CHECK(gram_tensor_map(c, tile_rows, C, &tm));
    if (tile_rows > GRAM_ROWS) { set_error("gram: N=%d needs more than %d rows per CTA at cluster size %d", c->N, GRAM_ROWS, CS); return VAMPOMI_ERR_ARG; }
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.blockDim = dim3(GRAM_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = c->stream; cfg.attrs = attr; cfg.numAttrs = 1;
    // co-resident clusters of this (cluster size, systems) on this device: queried once per context
    int& ncl = c->gram_clusters[CS][K - 1];
    if (ncl <= 0) {
        VO_CUDA(cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (CS > 8) VO_CUDA(cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));   // 16 CTAs: one cluster per GPC
        cfg.gridDim = dim3(CS, c->num_sms);
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, (const void*)kern, &cfg) != cudaSuccess || n < 1) { cudaGetLastError(); n = c->num_sms / CS; }
        ncl = n < 1 ? 1 : n;
    }
    long long nch = c->tune.gram_clusters > 0 ? c->tune.gram_clusters : ncl;
    const long long cap = (c->M + C - 1) / C;
    if (nch > cap) nch = cap;
    int cols_per_chunk = (int)((c->M + nch - 1) / nch);
    cols_per_chunk = (cols_per_chunk + C - 1) / C * C;
    const int nchunks = (int)((c->M + cols_per_chunk - 1) / cols_per_chunk);
    VO_CHECK(ensure_ax_partial(c, (size_t)K * nchunks * c->ld));
    cfg.gridDim = dim3(CS, nchunks);
    if (c->prof_pending.size() > 8192) VO_CHECK(prof_resolve(c));
    int sp = prof_begin(c, 3, (double)c->M * c->N * (double)c->elem_bytes);
    const double scale = 1.0 / sqrt((double)c->N);
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, (const double*)c->A, c->ld, (const double*)c->mave, (const double*)c->msig, gv, tile_rows,
                                       cols_per_chunk, c->M, scale, c->ax_partial, nchunks, tm);
    prof_end(c, sp);
    if (e != cudaSuccess) { set_error("gram kernel launch failed: %s", cudaGetErrorString(e)); cudaGetLastError(); return VAMPOMI_ERR_CUDA; }
    c->counters[0] += 1; c->counters[1]++; c->counters[2] += (long long)c->M * c->N * c->elem_bytes;
    return launch_ax_reduce_multi(c, nchunks, mw);
}

// The cluster size is the smallest that holds a column (knob gram_cluster overrides it), so that a CTA's row tile — and with it the
// bytes a step moves per exchange — is as full as it can be: N = 12 000 on 5 CTAs x 2 400 rows instead of 8 x 1 500 (a step
// costs about the same number of cycles whatever it carries).
template <int K>
int gram_run(vampomi_ctx* c, const MultiVec& mq, double* const* w_out) {
    GramVec gv{};
    MultiVec mw{};
    mw.K = K;
    for (int k = 0; k < K; k++) {
        gv.q[k] = mq.in[k]; gv.t[k] = mq.out[k]; gv.done[k] = mq.done[k];
        mw.in[k] = nullptr; mw.out[k] = w_out[k]; mw.done[k] = mq.done[k];
    }
    int cs = c->tune.gram_cluster;
    if (cs == 0) cs = (int)((c->ld + GRAM_ROWS - 1) / GRAM_ROWS);
    switch (cs) {
#define VAMPOMI_GRAM_CS(n) case n: return gram_launch<K, n>(c, gv, mw);
        VAMPOMI_GRAM_CS(1) VAMPOMI_GRAM_CS(2) VAMPOMI_GRAM_CS(3) VAMPOMI_GRAM_CS(4) VAMPOMI_GRAM_CS(5) VAMPOMI_GRAM_CS(6) VAMPOMI_GRAM_CS(7) VAMPOMI_GRAM_CS(8)
        VAMPOMI_GRAM_CS(9) VAMPOMI_GRAM_CS(10) VAMPOMI_GRAM_CS(11) VAMPOMI_GRAM_CS(12) VAMPOMI_GRAM_CS(13) VAMPOMI_GRAM_CS(14) VAMPOMI_GRAM_CS(15) VAMPOMI_GRAM_CS(16)
#undef VAMPOMI_GRAM_CS
        default: set_error("gram: cluster size must be 1 ... 16"); return VAMPOMI_ERR_ARG;
    }
}

}  // namespace

bool gram_supported(const vampomi_ctx* c) { return c->storage == 0 && c->ld <= (size_t)16 * GRAM_ROWS; }

// t_k = A^T q_k (M-vectors), w_k = A t_k (N-vectors, summed over the GPUs, / sqrt(N)) for K <= 2 systems in ONE pass.
// mq: in = q_k (N-vectors), out = t_k (M-vectors); w_out: the N-vectors that receive w_k. done flags from mq.
int launch_gram(vampomi_ctx* c, const MultiVec& mq, double* const* w_out) {
    if (mq.K < 1 || mq.K > 2) { set_error("gram: 1 or 2 systems"); return VAMPOMI_ERR_ARG; }
    if (!gram_supported(c)) { set_error("gram: needs FP64 storage and N <= 40960"); return VAMPOMI_ERR_ARG; }
    return mq.K == 1 ? gram_run<1>(c, mq, w_out) : gram_run<2>(c, mq, w_out);
}

}  // namespace vampomi
