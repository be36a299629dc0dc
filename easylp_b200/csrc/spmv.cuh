// spmv.cuh — the PDLP hot kernel: a persistent CSR-stream SpMV with a fused epilogue, built from
// warp-autonomous TMA pipelines.
//
//   out_r = epilogue( sum_k val[k] * vec[idx[k]],  k in [ptr[r], ptr[r+1]) )
//
// The same kernel serves A.x (CSR of A) and A'.y (CSC of A = CSR of A').  It is HBM-bound: per row it
// must move 12 B per entry (val 8 + idx 4), 4 B of row pointer, the epilogue's operand vectors and its
// outputs; the gathered vector (8n or 8m bytes) lives in the 126 MB L2.
//
// Design (sm_100a):
//   * every WARP is its own producer/consumer pipeline: it walks tiles of RW = 32/L rows (persistent grid,
//     warp-strided round-robin) and owns a private ring of NSTW stages in shared memory with one mbarrier
//     each.  No CTA-wide or inter-warp synchronisation exists in the loop;
//   * EVERYTHING that streams — the tile's slice of val/idx, its row pointers and the epilogue's operand
//     vectors (x-bar, c, l, u, x0 / y, rhs, y0 and a sense byte per row) — is brought into the ring by 1-D TMA bulk copies
//     (cp.async.bulk -> mbarrier complete_tx); lane i of the warp issues copy i, NSTW tiles ahead of the
//     tile being consumed, so the HBM latency is covered by the ring and not by the warp's own loads;
//   * the only loads the lanes issue to global memory are the gathers vec[idx[k]] (random 8-byte read-only
//     loads that hit L2; the matrix stream is marked evict-first so it does not push the vector out), U of
//     them in flight per lane; a group of L lanes walks one row (L = 1: one lane per row, the sum is formed strictly in
//     index order with separate multiply and add, i.e. bit-identical to a scalar CPU loop);
//   * rows longer than a stage are walked in pieces with a running sum.
// Array contract: val/idx are over-allocated by SPMV_PAD entries, ptr by 4 ints and every epilogue
// operand by SPMV_VPAD doubles (16-byte-granular copies must stay inside the allocations).
#pragma once
#include "common.cuh"
#include "tma.cuh"
#include <algorithm>
#include <cmath>
#include <cstdlib>

namespace elp {

constexpr int SPMV_PAD = 8;        // extra entries behind val / idx
constexpr int SPMV_PTR_PAD = 4;    // extra ints behind ptr
constexpr int SPMV_VPAD = 2;       // extra doubles behind every epilogue operand vector

constexpr int SPMV_ROUTE_WORDS = 16;   // multi-GPU: one 64-byte routing record per tile (8 base positions + 32 mask bytes)

struct SpmvStageLayout {          // byte offsets inside one stage of one warp
    int cap;                      // entries per stage (multiple of 4)
    int off_idx, off_ptr, off_ops, off_route, bytes;
};
// nin operand vectors of doubles, then ninb of bytes (16-byte copies: only for tiles of a multiple of 16 rows)
__host__ __device__ inline SpmvStageLayout spmv_stage_layout(int cap, int rw, int nin, bool route = false, int ninb = 0) {
    SpmvStageLayout s;
    s.cap = cap;
    s.off_idx = cap * 8;
    s.off_ptr = s.off_idx + cap * 4;
    s.off_ops = s.off_ptr + (rw + 4) * 4;
    s.off_route = s.off_ops + nin * ((rw + 1) & ~1) * 8 + ninb * ((rw + 15) & ~15);
    s.off_route = (s.off_route + 15) & ~15;
    s.bytes = s.off_route + (route ? SPMV_ROUTE_WORDS * 4 : 0);
    s.bytes = (s.bytes + 15) & ~15;
    return s;
}

constexpr int SPMV_WARPS = 4;      // warps per CTA (a CTA is only a container: warps never talk)

template <int L, int RPL, int NSTW, class Epi>
__global__ void __launch_bounds__(SPMV_WARPS * 32, 6 / RPL)
spmv_warp_kernel(int nrows, int ntiles, int cap, const int* __restrict__ ptr, const int* __restrict__ idx,
                 const double* __restrict__ val, const double* __restrict__ vec, Epi epi, int l2flags) {
    // NSTW stages per warp: one being consumed, the others in flight (2; 3 is offered to the scatter epilogues, which
    // hold a stage a little longer)
    constexpr int G = 32 / L;                // lane groups per warp
    constexpr int RW = G * RPL;              // rows per warp tile: group g owns rows g, g + G, ...
    constexpr int NIN = Epi::NIN, NINB = Epi::NINB;
    static_assert(NINB == 0 || RW % 16 == 0, "byte operands are staged in 16-byte pieces: tiles of a multiple of 16 rows");
    constexpr int U = (L <= 2) ? 8 : 4;      // gathers in flight per lane
    constexpr int OPS = (RW + 1) & ~1;       // doubles per staged operand
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const SpmvStageLayout lay = spmv_stage_layout(cap, RW, NIN, Epi::DIST, NINB);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* ring = smem_raw + (size_t)warp * NSTW * lay.bytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)SPMV_WARPS * NSTW * lay.bytes) + warp * NSTW;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < NSTW; ++s) mbar_init(&full[s], 1);
        mbar_fence_init();
    }
    __syncwarp();
    const uint64_t pol_stream = l2_policy_evict_first();
    const L2Hints hints{pol_stream, l2_policy_evict_last(), l2flags};
    // multi-GPU push mode: the last CTAs of the grid run no SpMV — they forward the local outboxes to the peers in aligned
    // full-warp stores as the values land (pdlp.cu: ghost_push_role)
    int nctas = gridDim.x;
    if constexpr (Epi::DIST) {
        const int pc = epi.push_ctas();
        if (pc > 0) {
            nctas -= pc;
            if ((int)blockIdx.x >= nctas) {
                epi.acquire(lane);          // the peers' last readers of what the copies overwrite have finished
                epi.push(((int)blockIdx.x - nctas) * SPMV_WARPS + warp, pc * SPMV_WARPS, lane);
                return;
            }
        }
    }
    const int gw = blockIdx.x * SPMV_WARPS + warp, nw = nctas * SPMV_WARPS;
    // Tile walk: warp-strided round robin, also in the multi-GPU kernels.  (Tried there: a contiguous range of tiles per warp
    // with the outgoing values collected in shared-memory rings and sent as aligned 256-byte stores.  The rings and the
    // extra registers cost two resident CTAs per SM, and losing them cost 38 us per iteration at N = 2 — far more than
    // the fuller NVLink packets could return; profiles/r2_multi_gpu_exchange.md.)
    const int t_first = gw, t_last = ntiles, t_step = nw;

    // ---- producer cursor: the next piece to copy (uniform across the warp) --------------------------------
    int p_tile = t_first, p_piece = 0, p_s = 0, p_e = 0, n_s = 0, n_e = 0;
    auto bounds = [&](int t, int& a, int& b) {
        if (t < t_last) {
            const int r0 = t * RW;
            a = __ldg(ptr + r0);
            b = __ldg(ptr + min(r0 + RW, nrows));
        } else { a = 0; b = 0; }
    };
    auto issue = [&](int stage) {
        if (p_tile >= t_last) return;
        const int a0 = p_s & ~3, a1 = (p_e + 3) & ~3;
        const int pstart = a0 + p_piece * cap;
        const int pcnt = max(0, min(cap, a1 - pstart));
        const bool last = pstart + pcnt >= a1;
        const int r0 = p_tile * RW;
        const int rows = min(RW, nrows - r0);
        const uint32_t ptr_bytes = (uint32_t)((rows + 1 + 3) & ~3) * 4u;
        const uint32_t op_bytes = (uint32_t)((rows + 1) & ~1) * 8u;
        const uint32_t opb_bytes = (uint32_t)((rows + 15) & ~15);
        unsigned char* sb = ring + (size_t)stage * lay.bytes;
        // lane i issues copy i: 0 val, 1 idx, 2 row pointers, 3.. epilogue operands
        const void* src = nullptr;
        unsigned char* dst = sb;
        uint32_t bytes = 0;
        if (lane == 0) { src = val + pstart; bytes = (uint32_t)pcnt * 8u; }
        else if (lane == 1) { src = idx + pstart; dst = sb + lay.off_idx; bytes = (uint32_t)pcnt * 4u; }
        else if (p_piece == 0) {
            if (lane == 2) { src = ptr + r0; dst = sb + lay.off_ptr; bytes = ptr_bytes; }
            else if (lane < 3 + NIN) { src = epi.in(lane - 3) + r0; dst = sb + lay.off_ops + (lane - 3) * OPS * 8; bytes = op_bytes; }
            else if (lane < 3 + NIN + NINB) {
                src = epi.in_b(lane - 3 - NIN) + r0;
                dst = sb + lay.off_ops + NIN * OPS * 8 + (lane - 3 - NIN) * ((RW + 15) & ~15);
                bytes = opb_bytes;
            }
            else if (lane == 3 + NIN + NINB) {
                if constexpr (Epi::DIST) {                // multi-GPU: the tile's routing record travels with its operands
                    if (epi.route_table() != nullptr) {
                        src = epi.route_table() + (size_t)p_tile * SPMV_ROUTE_WORDS; dst = sb + lay.off_route; bytes = SPMV_ROUTE_WORDS * 4;
                    }
                }
            }
        }
        if (lane == 0) {
            uint32_t tx = (uint32_t)pcnt * 12u;
            if (p_piece == 0) tx += ptr_bytes + (uint32_t)NIN * op_bytes + (uint32_t)NINB * opb_bytes;
            if constexpr (Epi::DIST) { if (p_piece == 0 && epi.route_table() != nullptr) tx += SPMV_ROUTE_WORDS * 4u; }
            mbar_expect_tx(&full[stage], tx);
        }
        __syncwarp();
        if (bytes > 0) {
            if (lane < 2) tma_load_1d_hint(dst, src, bytes, &full[stage], pol_stream);
            else if (l2flags & 1) tma_load_1d_hint(dst, src, bytes, &full[stage], pol_stream);
            else tma_load_1d(dst, src, bytes, &full[stage]);
        }
        if (last) {
            p_tile += t_step; p_piece = 0;
            p_s = n_s; p_e = n_e;
            bounds(p_tile + t_step, n_s, n_e);    // needed one tile later: its latency is hidden
        } else {
            ++p_piece;
        }
    };
    bounds(p_tile, p_s, p_e);
    bounds(p_tile + t_step, n_s, n_e);
#pragma unroll
    for (int s = 0; s < NSTW; ++s) issue(s);
    // multi-GPU: the gathered vector is filled by the peers' stores.  The matrix stream is already on its way; wait
    // here — once per warp — until every producer has published the epoch this launch consumes.
    if constexpr (Epi::DIST) epi.acquire(lane);         // (`vec` stays the kernel parameter: uniform address arithmetic in the gathers)

    // ---- consumer ------------------------------------------------------------------------------------------
    const int g = lane / L;                // first row of the tile this lane group owns
    const int sub = lane % L;
    int q = 0;
    bool held = false;                     // scatter epilogues: the tile's only stage is still owned by the consumer
    const double* hv = nullptr;
    const int* hi = nullptr;
    int hstage = 0;
    for (int tile = t_first; tile < t_last; tile += t_step) {
        const int row0 = tile * RW + g;
        int st[RPL], en[RPL], a0 = 0, a1 = 0;
        typename Epi::Pre pre[RPL];
        double acc[RPL];
        // multi-GPU: who reads this tile's outputs and where they go (picked out of the staged routing record)
        [[maybe_unused]] typename Epi::Route route[RPL];
#pragma unroll
        for (int j = 0; j < RPL; ++j) { st[j] = 0; en[j] = 0; acc[j] = 0.0; pre[j] = typename Epi::Pre{}; }
        for (int piece = 0;; ++piece) {
            const int stage = q % NSTW;
            mbar_wait(&full[stage], (uint32_t)(q / NSTW) & 1u);
            const unsigned char* sb = ring + (size_t)stage * lay.bytes;
            if (piece == 0) {
                const int* sp = reinterpret_cast<const int*>(sb + lay.off_ptr);
                const int rows = min(RW, nrows - tile * RW);
                a0 = sp[0] & ~3;
                a1 = (sp[rows] + 3) & ~3;
#pragma unroll
                for (int j = 0; j < RPL; ++j) {
                    if (row0 + j * G < nrows) {
                        st[j] = sp[g + j * G];
                        en[j] = sp[g + j * G + 1];
                        if (sub == 0) pre[j] = epi.preload(reinterpret_cast<const double*>(sb + lay.off_ops), OPS, g + j * G);
                    }
                    if constexpr (Epi::DIST)
                        route[j] = epi.route(reinterpret_cast<const uint32_t*>(sb + lay.off_route), lane,
                                             sub == 0 && row0 + j * G < nrows, g + j * G);
                }
            }
            const int pstart = a0 + piece * cap;
            const int pend = min(pstart + cap, a1);
            // index the stage by global entry id
            const double* sv = reinterpret_cast<const double*>(sb) - pstart;
            const int* si = reinterpret_cast<const int*>(sb + lay.off_idx) - pstart;
            int k[RPL], f[RPL];
            bool more = false;
#pragma unroll
            for (int j = 0; j < RPL; ++j) {
                k[j] = max(st[j], pstart) + sub;
                f[j] = min(en[j], pend);
                more |= k[j] < f[j];
            }
            while (more) {
                // the RPL rows of a lane advance together: their gathers are independent and overlap.
                // indices first, gathers next, the values are read from the stage only when they are consumed.
                // Instruction economy matters here (the kernel is issue-bound): one compare against an immediate per
                // entry, plain read-only loads for the gathers.
                double x[RPL][U];
                int c[RPL][U], cnt[RPL];
                const int* sij[RPL];
                const double* svj[RPL];
#pragma unroll
                for (int j = 0; j < RPL; ++j) { cnt[j] = f[j] - k[j]; sij[j] = si + k[j]; svj[j] = sv + k[j]; }
#pragma unroll
                for (int j = 0; j < RPL; ++j)
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (u * L < cnt[j]) c[j][u] = sij[j][u * L];
#pragma unroll
                for (int j = 0; j < RPL; ++j)
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (u * L < cnt[j]) x[j][u] = (l2flags & 8) ? ldg_hint(vec + c[j][u], hints.last) : __ldg(vec + c[j][u]);
#pragma unroll
                for (int j = 0; j < RPL; ++j)
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (u * L < cnt[j]) acc[j] = __dadd_rn(acc[j], __dmul_rn(svj[j][u * L], x[j][u]));
                more = false;
#pragma unroll
                for (int j = 0; j < RPL; ++j) { k[j] += U * L; more |= k[j] < f[j]; }
            }
            // scatter epilogues re-read a tile that fits one stage from that stage: keep it until they are done
            const bool hold = Epi::SCATTER && piece == 0 && pend >= a1;
            __syncwarp();                      // every lane is done reading the stage
            if (!hold) issue(stage);
            ++q;
            if (pend >= a1) {
                if (Epi::SCATTER) { held = hold; hv = sv; hi = si; hstage = stage; }
                break;
            }
        }
#pragma unroll
        for (int j = 0; j < RPL; ++j) {
            double a = acc[j];
            if (L > 1) a = group_sum<L>(a);
            double mult = 0.0;
            const bool owner = sub == 0 && row0 + j * G < nrows;
            if (owner) mult = epi.apply(row0 + j * G, a, pre[j], hints);
            // multi-GPU: the value just produced goes into the ghost vector of every rank that gathers it (warp-collective)
            if constexpr (Epi::DIST) epi.publish(route[j], lane, row0 + j * G, mult);
            if (Epi::SCATTER) {
                // out[idx[k]] += val[k] * mult over this row's entries (fire-and-forget fp64 reductions: SASS RED.ADD.F64);
                // rows whose multiplier is zero (inactive constraints) send nothing.
                if (L > 1) mult = __shfl_sync(0xffffffffu, mult, lane - sub);
                if (mult != 0.0) {
                    const double* vv = held ? hv : val;
                    const int* ii = held ? hi : idx;
                    for (int e = st[j] + sub; e < en[j]; e += L) atomicAdd(epi.scat + ii[e], __dmul_rn(vv[e], mult));
                }
            }
        }
        if (Epi::SCATTER && held) {
            __syncwarp();
            issue(hstage);
        }
    }
}

// ---- long rows: one warp per row -----------------------------------------------------------------------
// Matrices with few, long rows (the supply/demand rows of a transportation problem: 600 rows of 300 entries) give the
// tile kernel above a handful of tiles for 148 SMs.  Here a warp owns a row (warp-strided, grid sized to the rows), the
// lanes stride over its entries with plain streaming loads, and a butterfly sum (fixed order: deterministic) feeds the
// same epilogue.  These matrices live in L2; the kernel is latency-bound, not bandwidth-bound.
template <class Epi>
__global__ void __launch_bounds__(128)
spmv_rowwarp_kernel(int nrows, const int* __restrict__ ptr, const int* __restrict__ idx, const double* __restrict__ val,
                    const double* __restrict__ vec, Epi epi) {
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * 128 + threadIdx.x) >> 5, nw = (gridDim.x * 128) >> 5;
    const L2Hints hints{0, 0, 0};
    for (int r = gw; r < nrows; r += nw) {
        const int a = __ldg(ptr + r), b = __ldg(ptr + r + 1);
        typename Epi::Pre pre{};
        if (lane == 0) pre = epi.preload_global(r);
        double s0 = 0.0, s1 = 0.0;
        int k = a + lane;
        for (; k + 32 < b; k += 64) {                 // two independent chains per lane
            const int c0 = ld_stream(idx + k), c1 = ld_stream(idx + k + 32);
            const double v0 = ld_stream(val + k), v1 = ld_stream(val + k + 32);
            s0 = fma(v0, __ldg(vec + c0), s0);
            s1 = fma(v1, __ldg(vec + c1), s1);
        }
        if (k < b) s0 = fma(ld_stream(val + k), __ldg(vec + ld_stream(idx + k)), s0);
        const double s = warp_sum(s0 + s1);
        if (lane == 0) epi.apply(r, s, pre, hints);
    }
}

// ---- launch plan ---------------------------------------------------------------------------------
struct SpmvPlan {
    int L = 1, rpl = 1, cap = 256, ctas_per_sm = 6, ntiles = 0, nst = 2;
    bool rowwarp = false;          // long rows: one warp per row (spmv_rowwarp_kernel)
    int rw() const { return 32 / L * rpl; }
};

inline int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}

// lanes per row from the mean row length: about six entries or fewer per lane, at most eight lanes
inline int pick_lanes(int64_t nnz, int64_t nrows) {
    const double avg = nrows > 0 ? (double)nnz / (double)nrows : 0.0;
    int L = 1;
    while (L < 8 && avg > 6.0 * L) L *= 2;         // avg <= 6 -> 1, <= 12 -> 2, <= 24 -> 4, else 8
    return L;
}

inline size_t spmv_smem_bytes(const SpmvPlan& p, int nin, bool route = false, int ninb = 0) {
    return (size_t)SPMV_WARPS * p.nst * (spmv_stage_layout(p.cap, p.rw(), nin, route, ninb).bytes + 8);
}

// nin_max: the largest operand count among the epilogues that will run with this plan
inline SpmvPlan plan_spmv(int64_t nnz, int nrows, int nin_max, int force_lanes = 0, int stages = 2) {
    SpmvPlan p;
    p.nst = stages == 3 ? 3 : 2;
    const double avg = nrows > 0 ? (double)nnz / (double)nrows : 0.0;
    p.L = pick_lanes(nnz, nrows);
    if (force_lanes > 0) p.L = force_lanes;
    if (const int l = env_int("ELP_SPMV_L", 0)) p.L = l;       // debugging / sweeps
    if (p.L != 1 && p.L != 2 && p.L != 4 && p.L != 8) p.L = 1;   // RW = 32/L >= 4 keeps the tile copies 16-byte aligned
    p.rpl = env_int("ELP_SPMV_RPL", 1) == 2 ? 2 : 1;   // measured on C4: two rows per lane (half the warps) is ~12 % slower
    const int rw = p.rw();
    // stage capacity: mean tile + ~1.5 sigma of a Poisson-like spread; the few larger tiles are walked in pieces
    const double mean = avg * rw;
    int64_t cap = (int64_t)(mean + 1.5 * std::sqrt(std::max(mean, 1.0)) * env_int("ELP_SPMV_CAPSIG_PCT", 100) / 100.0) + 8;
    cap = (cap + 31) / 32 * 32;
    cap = std::max<int64_t>(64, std::min<int64_t>(cap, 1024));   // <= 12.3 KB per stage; longer tiles go in pieces
    if (const int c = env_int("ELP_SPMV_CAP", 0)) cap = std::max(16, c / 4 * 4);
    p.cap = (int)cap;
    p.ntiles = ceil_div(nrows, rw);
    // few long rows: the tiles of 32/L rows would not fill the machine; a warp per row does
    p.rowwarp = force_lanes == 0 && avg >= 48.0 && p.ntiles < kNumSMs * 6 * SPMV_WARPS;
    if (const char* e = getenv("ELP_SPMV_ROWWARP")) p.rowwarp = atoi(e) != 0 && force_lanes == 0;
    // residency: as many CTAs as 64 K registers allow (6 CTAs of 4 warps at 80 per thread, 3 at 160 for two rows per lane) inside 196 KB of shared memory.
    // Measured on B200: once the CTAs of an SM take more than the 196 KB carve-out step, the L1 left over
    // for the gathers is too small and the kernel slows down by ~30 %.
    const size_t per_cta = spmv_smem_bytes(p, nin_max) + 1024;      // + the 1 KB the system reserves per CTA
    int ctas = (int)std::min<size_t>(196 * 1024 / per_cta, 6 / p.rpl);
    if (const int c = env_int("ELP_SPMV_CTAS", 0)) ctas = c;
    p.ctas_per_sm = std::max(1, ctas);
    return p;
}

template <int L, int RPL, int NSTW, class Epi>
void launch_spmv_inst(const SpmvPlan& p, int nrows, const int* ptr, const int* idx, const double* val,
                      const double* vec, const Epi& epi, cudaStream_t st) {
    auto kern = spmv_warp_kernel<L, RPL, NSTW, Epi>;
    const size_t smem = spmv_smem_bytes(p, Epi::NIN, Epi::DIST, Epi::NINB);
    ELP_REQUIRE(smem <= 227 * 1024, "spmv: stage ring of %zu bytes does not fit in shared memory", smem);
    // per device and ring size: raise the dynamic shared-memory limit once and ask how many CTAs really fit
    static size_t cfg_smem[16] = {};
    static int cfg_occ[16] = {};
    int dev = 0;
    ELP_CUDA(cudaGetDevice(&dev));
    dev &= 15;
    if (cfg_smem[dev] != smem + 1) {
        ELP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        int occ = 0;
        ELP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, SPMV_WARPS * 32, smem));
        cfg_occ[dev] = std::max(1, occ);
        cfg_smem[dev] = smem + 1;
        if (env_int("ELP_SPMV_DEBUG", 0))
            fprintf(stderr, "[spmv] L=%d rpl=%d nin=%d cap=%d smem/CTA=%zu planned CTAs/SM=%d resident=%d tiles=%d\n", L, RPL,
                    Epi::NIN, p.cap, smem, p.ctas_per_sm, occ, p.ntiles);
    }
    // persistent grid: exactly one wave
    const int per_sm = std::min(p.ctas_per_sm, cfg_occ[dev]);
    int grid = std::max(1, std::min(ceil_div(p.ntiles, SPMV_WARPS), kNumSMs * per_sm));
    if constexpr (Epi::DIST) {      // push mode: the pusher CTAs are part of the one resident wave
        const int pc = epi.push_ctas();
        if (pc > 0) {
            ELP_REQUIRE(pc < kNumSMs * per_sm, "spmv: %d pusher CTAs leave no room for the SpMV (%d CTAs fit)", pc, kNumSMs * per_sm);
            grid = std::max(1, std::min(ceil_div(p.ntiles, SPMV_WARPS), kNumSMs * per_sm - pc)) + pc;
        }
    }
    // L2 residency hints (tma.cuh: L2Hints).  Default 3: the operand streams and the outputs nobody gathers from are
    // evict-first like the matrix stream, so that the vector the NEXT kernel gathers from survives in L2.  Measured in
    // alternation K1,K2,K1,... on C4: 0.2766 ms per iteration vs 0.2823 without (gpurun_out/r3c_hints.log).
    const int l2flags = env_int("ELP_SPMV_L2HINTS", 3);
    ELP_LAUNCH(kern, grid, SPMV_WARPS * 32, smem, st, nrows, p.ntiles, p.cap, ptr, idx, val, vec, epi, l2flags);
}

template <int L, class Epi>
void launch_spmv_l(const SpmvPlan& p, int nrows, const int* ptr, const int* idx, const double* val, const double* vec,
                   const Epi& epi, cudaStream_t st) {
    if constexpr (Epi::SCATTER) {    // scatter epilogues: one row per lane group, 2 or 3 stages
        if (p.nst == 3) launch_spmv_inst<L, 1, 3, Epi>(p, nrows, ptr, idx, val, vec, epi, st);
        else launch_spmv_inst<L, 1, 2, Epi>(p, nrows, ptr, idx, val, vec, epi, st);
    } else {
        if (p.rpl == 1) launch_spmv_inst<L, 1, 2, Epi>(p, nrows, ptr, idx, val, vec, epi, st);
        else launch_spmv_inst<L, 2, 2, Epi>(p, nrows, ptr, idx, val, vec, epi, st);
    }
}

template <class Epi>
void launch_spmv(const SpmvPlan& p, int nrows, const int* ptr, const int* idx, const double* val, const double* vec,
                 const Epi& epi, cudaStream_t st) {
    if (nrows <= 0) return;
    if constexpr (!Epi::SCATTER && !Epi::DIST) {
        if (p.rowwarp) {
            const int grid = std::max(1, std::min(ceil_div(nrows, 4), kNumSMs * 16));
            ELP_LAUNCH((spmv_rowwarp_kernel<Epi>), grid, 128, 0, st, nrows, ptr, idx, val, vec, epi);
            return;
        }
    }
    if constexpr (Epi::NINB > 0) {   // byte operands: tiles of 16 or 32 rows only
        ELP_REQUIRE(p.L <= 2, "spmv: an epilogue with byte operands needs a plan of at most two lanes per row (L = %d)", p.L);
        if (p.L == 1) launch_spmv_l<1, Epi>(p, nrows, ptr, idx, val, vec, epi, st);
        else launch_spmv_l<2, Epi>(p, nrows, ptr, idx, val, vec, epi, st);
    } else {
        switch (p.L) {
            case 1:  launch_spmv_l<1, Epi>(p, nrows, ptr, idx, val, vec, epi, st); break;
            case 2:  launch_spmv_l<2, Epi>(p, nrows, ptr, idx, val, vec, epi, st); break;
            case 4:  launch_spmv_l<4, Epi>(p, nrows, ptr, idx, val, vec, epi, st); break;
            default: launch_spmv_l<8, Epi>(p, nrows, ptr, idx, val, vec, epi, st); break;
        }
    }
}

}  // namespace elp
