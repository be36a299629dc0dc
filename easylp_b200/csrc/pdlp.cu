// pdlp.cu — PDLP-style first-order LP solver for large sparse LPs on one or several B200s.
//
// Replaces `status <- solve(prob)` (/root/reference/R/class.R:276; lp_solve's simplex) for LPs whose
// dense tableau does not fit in shared memory.  Problem form (after mapping the reference's rows,
// R/class.R:271-274):   min c'x   s.t.  lc <= A x <= uc ,  l <= x <= u.
//
// Algorithm: restarted reflected Halpern PDHG (r2HPDHG; Lu & Yang 2024, the cuPDLPx scheme):
//   z' = T(z):  x' = proj_[l,u](x - tau (c - A'y)),   y' = prox(y - sigma A(2x' - x))
//   z+ = (k+1)/(k+2) (2 z' - z) + 1/(k+2) z_anchor          (k = iterations since the last restart)
// with Ruiz + Pock-Chambolle diagonal scaling, constant step eta = 0.998/||A||_2 (tau = eta/w,
// sigma = eta*w), primal weight w re-balanced at restarts, fixed-point-error restarts and PDLP's
// relative KKT termination test.  The CPU restatement of this loop is oracle/pdlp_ref.py.
//
// Kernels per iteration (single GPU) — exactly two, both HBM-bound SpMVs with fused epilogues (spmv.cuh):
//   K1  CSC (transposed) SpMV  g = A'y  + projection + reflection + Halpern combine  -> xbar (x is rebuilt from it)
//   K2  CSR SpMV  A xbar       + dual prox + reflection + Halpern combine            -> y
// Matrix stream, row pointers and the epilogue operands arrive in shared memory by TMA bulk copies;
// the gathered vector (x: 8n bytes, y: 8m bytes) lives in the 126 MB L2.
// Algorithmic bytes per plain iteration (DESIGN.md §4.1): 24 nnz + 4 (m+n+2) + 8 (m+n) + 8 (4 + [l] + [u]) n + 33 m.
//
// Multi-GPU (SURVEY §8e): rank g owns a row block of A (for K2, its slice of y) AND a column block of A over all
// rows (for K1, its slice of x).  Nothing is replicated; per iteration the x-bar blocks and the y blocks are
// all-gathered over NVLink (8 (n + m) bytes received per rank) and the scalar residuals of a check travel in one
// 16-double allreduce.  See `struct Pdlp`.
#include "common.cuh"
#include "primitives.cuh"
#include "comm.cuh"
#include "tma.cuh"
#include "spmv.cuh"
#include "../../include/easylp_abi.h"
#include <cmath>
#include <algorithm>
#include <unistd.h>

namespace elp {

struct PdlpParams {   // device-resident; the host rewrites it between iteration chunks
    double tau, sigma;
    int k_base;       // iterations since restart at the start of the chunk
    int pad;
    long long epoch_base;   // multi-GPU: exchange epochs completed before the chunk (iteration `it` produces epoch_base + it + 1)
};

constexpr int SPMV_THREADS = 256;             // block size of the setup-only helper kernels

// ---- epilogues of the SpMV (spmv.cuh): in(i) names the operand vectors the producer stages next to the
// matrix stream, preload() picks this row's operands out of the stage, apply() runs after the row sum ------
struct NoRoute {};
struct StoreEpi {
    static constexpr int NIN = 0, NINB = 0;
    static constexpr bool SCATTER = false;
    static constexpr bool DIST = false;
    double* scat = nullptr;
    double* out;
    using Route = NoRoute;
    struct Pre {};
    __device__ __forceinline__ const double* in(int) const { return nullptr; }
    __device__ __forceinline__ const int8_t* in_b(int) const { return nullptr; }
    __device__ __forceinline__ Pre preload(const double*, int, int) const { return Pre{}; }
    __device__ __forceinline__ Pre preload_global(int) const { return Pre{}; }
    __device__ __forceinline__ double apply(int r, double s, const Pre&, const L2Hints&) const { out[r] = s; return 0.0; }
};

inline StoreEpi store_epi(double* out) { StoreEpi e; e.out = out; return e; }

// ---- multi-GPU exchange: ghost vectors filled by the producers' own stores -------------------------------------
// Rank r gathers only the entries of x-bar (y) that its row (column) block references.  It keeps them in a COMPACT
// ghost vector — entries in ascending global id, its matrix copy for the plain iterations carries the compact ids — with
// two buffers selected by the parity of the epoch, so a producer may run one kernel ahead of its consumers without a
// write-after-read hazard.  The epilogue of the producing kernel stores each value straight into the ghost vector of
// every rank that reads it (peer access / CUDA IPC over NVLink); the position is the tile's base in that rank's vector
// plus the number of lower lanes that also store there (one ballot per destination), so the stores of a warp are
// contiguous.  Masks and bases of a tile form a 64-byte routing record that is staged with the tile by TMA.
// The hand-off lives in the PROLOGUE of the consuming kernel.  Stream order makes everything this rank launched
// before complete, so thread 0 of the kernel first publishes "my part of epoch E is done" in slot `rank` of every
// rank's flag row (one system fence, N stores; no per-CTA fences, counters or extra launches: measured at N = 2 the
// in-producer variant — fence + last-CTA counter in every CTA — cost 21 us per iteration), and one warp per CTA then
// polls the local flag row until all N slots have reached E while the first matrix tiles are already on their way.
struct GhostOut {
    double* buf[8];                    // rank r's ghost vector
    const uint32_t* route;             // [tiles of my block][SPMV_ROUTE_WORDS]: words 0-7 position of the tile's first entry
                                       // in rank r's ghost vector, bytes 32-63 per row of the tile: bit r = rank r gathers it
    int n, rank;
    int dense, first;                  // dense != 0: no compaction — rank r's ghost vector is the whole vector and my block
                                       // starts at `first` in it (chosen when the ranks read most of everything anyway)
    int self_only;                     // measurement switch (ELP_GHOST_LOCAL_ONLY): nothing leaves the GPU (timing only)
    // push mode (see ghost_push_role): buf[r] of a remote rank is a LOCAL outbox indexed like r's ghost vector, the last
    // `push_ctas` CTAs of the kernel move segments of seg_tiles tiles to remote[r] as soon as their values have landed
    double* remote[8];                 // rank r's ghost vector
    unsigned int* err;                 // bit 1: a segment never completed
    int seg_tiles, nseg, ntiles, push_ctas;      // push_ctas == 0: push mode off
};
struct GhostIn {
    const double* vec;                 // my ghost vector
    unsigned int len;                  // its length in doubles
    const unsigned long long* flags;   // my flag row for it (N slots)
    unsigned long long* go;            // local word: block 0 releases the epoch here for the other CTAs of the kernel
    unsigned long long* peer_flag[8];  // rank r's flag row for the same vector; this rank writes slot `rank`
    unsigned int* err;                 // bit 0: a producer never showed up (the host turns it into an error)
    unsigned long long* trace;         // ELP_GHOST_DEBUG bit 64: [4096][4] globaltimer stamps (entry, signalled, flags seen) per kernel
    int n, rank, kind;                 // kind: 0 the kernel consumes y (K1), 1 it consumes x-bar (K2)
    int dbg;                           // 2 no wait, 4 no signal, 64 trace
};
// flag store AFTER an explicit system fence: relaxed is enough (a st.release would repeat the fence per destination)
__device__ __forceinline__ void st_relaxed_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
// consumer prologue: signal my part of epoch `want`, wait for everybody's; returns the buffer that holds the epoch
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// Consumer prologue.  Block 0: thread 0 publishes this rank's part of epoch `want` to every rank, the first N lanes poll
// the local flag row until every rank's slot reached `want`, ONE system fence orders the gathers behind the flags, and
// a local "go" word is released at GPU scope.  Every other CTA only spins on that go word with GPU-scope acquire loads:
// no system-scope fence per CTA (888 of them at once when the flags flip were the constant cost that kept K2 from
// scaling), no system-scope traffic at all outside block 0.
__device__ __forceinline__ void ghost_acquire(const GhostIn& gi, long long want, int lane) {
    const bool tracer = (gi.dbg & 64) && blockIdx.x == 0 && threadIdx.x == 0;
    unsigned long long* tr = tracer ? gi.trace + (size_t)((2 * want + gi.kind) & 4095) * 4 : nullptr;
    if (tracer) { tr[0] = globaltimer_ns(); tr[3] = (unsigned long long)want; }
    if (blockIdx.x == 0) {
        if (threadIdx.x == 0 && !(gi.dbg & 4)) {
            __threadfence_system();
            for (int r = 0; r < gi.n; ++r) st_relaxed_sys(gi.peer_flag[r] + gi.rank, (unsigned long long)want);
        }
        if (tracer) tr[1] = globaltimer_ns();
        if (!(gi.dbg & 2) && (threadIdx.x >> 5) == 0) {
            if (lane < gi.n) {
                unsigned long long spins = 0;
                while ((long long)ld_volatile_u64(gi.flags + lane) < want) {
                    if (++spins > (1ull << 25)) { atomicOr(gi.err, 1u); break; }      // ~10 s: a peer died; fail, do not hang
                    if (spins > 16) __nanosleep(20);
                }
            }
            __syncwarp();
            if (lane == 0) {
                __threadfence_system();                // acquire at system scope, once
                st_release_gpu(gi.go, (unsigned long long)want);
            }
        }
    } else if (!(gi.dbg & 2) && threadIdx.x == 0) {
        unsigned long long spins = 0;
        while ((long long)ld_acquire_gpu(gi.go) < want) {
            if (++spins > (1ull << 25)) { atomicOr(gi.err, 1u); break; }
            if (spins > 8) __nanosleep(20);
        }
    }
    __syncthreads();
    if (tracer) tr[2] = globaltimer_ns();
    // Experiment kept behind dbg bit 128: pull the whole ghost vector into L2 with sequential prefetches (what the peers
    // stored arrived over NVLink; if it sat in HBM only, the first gather of every sector would be a random HBM access).
    // Measured at N = 2: 181.8 us per iteration with it, 177.7 without — the gathers are not where K2 loses its time.
    if (gi.dbg & 128) {
        const size_t lines = ((size_t)gi.len * 8 + 127) / 128;
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < lines; i += (size_t)gridDim.x * blockDim.x)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(gi.vec) + i * 128));
    }
}
// producer side, per row of a warp tile (all 32 lanes call both; `owner` lanes carry a value).  The destination table is
// a kernel parameter and the loops over the destinations are unrolled (constant-bank operands); reading the table from
// device memory in rolled loops was measured 5 % slower at N = 2 (190 vs 180 us per iteration).
struct GhostRoute { unsigned mk; int base; };
__device__ __forceinline__ GhostRoute ghost_route(const GhostOut& go, const uint32_t* rec, int lane, bool owner, int row_in_tile) {
    GhostRoute g;
    if (go.dense) { g.mk = owner ? 1u : 0u; g.base = 0; }        // no record is staged: everything goes everywhere
    else {
        g.mk = owner ? (unsigned)reinterpret_cast<const unsigned char*>(rec)[32 + row_in_tile] : 0u;
        g.base = (int)rec[lane & 7];
    }
    return g;
}
__device__ __forceinline__ void ghost_publish(const GhostOut& go, const GhostRoute& rt, int lane, int row, double v) {
    if (go.dense) {
        // everybody reads (almost) everything: the ghost vectors are plain copies of the whole vector, the value of row
        // `row` of my block goes to position first + row of every copy — aligned, full 256-byte warp stores
        if (rt.mk) {
            const size_t at = (size_t)(go.first + row);
#pragma unroll
            for (int r = 0; r < 8; ++r)
                if (r < go.n && (!go.self_only || r == go.rank)) go.buf[r][at] = v;
        }
        return;
    }
    const unsigned mk = rt.mk;
    const unsigned lower = (1u << lane) - 1u;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        if (r < go.n) {
            const bool send = ((mk >> r) & 1u) && (!go.self_only || r == go.rank);
            const unsigned b = __ballot_sync(0xffffffffu, send);
            const int br = __shfl_sync(0xffffffffu, rt.base, r);
            if (send) go.buf[r][(uint32_t)br + __popc(b & lower)] = v;
        }
    }
}

// ---- push mode: the NVLink traffic leaves through dedicated CTAs of the same kernel ----------------------------------
// Remote stores issued by the SpMV warps share the SM's load/store path with the gathers, and a warp's compacted run for
// one destination is ~18 doubles at an arbitrary 8-byte phase: 160 K short, misaligned NVLink writes per rank and
// iteration at N = 8.  The kernels are held back by them: bodies of 45 / 50 us for 23 / 19 us of work.  In push mode the
// epilogues write what other ranks read into LOCAL outboxes (same compact layout, same positions); the LAST `push_ctas`
// CTAs of the grid do no SpMV — each of their warps owns (segment, destination) items and forwards them in aligned
// groups of 32 consecutive doubles (256-byte warp stores, 8 groups in flight per warp).
// Readiness travels IN the data: an outbox holds a NaN sentinel wherever this launch has not stored yet; the pusher reads
// a group through L2 (ld.relaxed.gpu), forwards it once no lane sees the sentinel and puts the sentinel back.  Every
// value is one 8-byte store, so a non-sentinel read IS the value: the producers need no fence, no counter, nothing.
// History (config 4 forced compact, N = 2, 173 us per iteration with the epilogues' own peer stores):
//   * companion KERNEL on a second stream + per-segment counters + bulk copies                         320 us
//   * pusher CTAs inside the grid, polling the counters with ld.acquire.gpu (= LDG.STRONG.GPU + CCTL.IVALL: an L1
//     invalidation per poll on every SM takes the gathered vector away from the SpMV CTAs next door)     308 us
//   * relaxed polls, no fence at the pushers' end                                                       252 us (148 CTAs), 239 (74)
//   * what remained was the producers' red.release.gpu per tile (MEMBAR.ALL.GPU under a saturated memory system)
//     -> the sentinel protocol below.
constexpr unsigned long long GHOST_SENTINEL = 0xFFF85EED0BADC0DEull;       // a quiet NaN no iterate ever holds
__device__ __forceinline__ unsigned long long ld_relaxed_gpu_u64(const void* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void ghost_push_role(const GhostOut& go, int pw, int npw, int lane) {
    constexpr int U = 8;
    const int nd = go.n - 1;
    const int nitems = go.nseg * nd;
    for (int item = pw; item < nitems; item += npw) {
        const int seg = item / nd, di = item - seg * nd;
        const int r = di < go.rank ? di : di + 1;
        const int t0 = seg * go.seg_tiles, t1 = min(t0 + go.seg_tiles, go.ntiles);
        const uint32_t a = go.route[(size_t)t0 * SPMV_ROUTE_WORDS + r], b = go.route[(size_t)t1 * SPMV_ROUTE_WORDS + r];
        unsigned long long* src = reinterpret_cast<unsigned long long*>(go.buf[r]);
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(go.remote[r]);
        for (uint32_t p0 = a & ~31u; p0 < b; p0 += 32u * U) {          // groups aligned in the destination's index space
            unsigned long long spins = 0;
            for (;;) {
                unsigned long long v[U];
                bool ok = true;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const uint32_t p = p0 + (uint32_t)u * 32u + (uint32_t)lane;
                    v[u] = (p >= a && p < b) ? ld_relaxed_gpu_u64(src + p) : 0ull;
                    ok &= v[u] != GHOST_SENTINEL;
                }
                if (__all_sync(0xffffffffu, ok)) {
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const uint32_t p = p0 + (uint32_t)u * 32u + (uint32_t)lane;
                        if (p >= a && p < b) { dst[p] = v[u]; src[p] = GHOST_SENTINEL; }
                    }
                    break;
                }
                if (++spins > (1ull << 22)) { if (lane == 0) atomicOr(go.err, 2u); return; }     // seconds: fail, do not hang
                __nanosleep(spins < 64 ? 100 : 400);
            }
        }
    }
}

// Halpern weight after k iterations of the epoch, and the iterate it forms: w xb + (1 - w) x0.  One rounding for every
// place that forms x (the plain primal epilogue, its rebuild of x from the carried x-bar, k_halpern_finish): the rebuilt
// x must be the stored one bit for bit.
__host__ __device__ __forceinline__ double halpern_w(int k) { const double kd = (double)k; return (kd + 1.0) / (kd + 2.0); }
__device__ __forceinline__ double halpern_x(double w, double xb, double x0) {
    return __fma_rn(xb, w, __dmul_rn(__dadd_rn(1.0, -w), x0));
}

// bound kinds of the columns (after scaling), as template argument of the plain primal epilogue: a bound that is the
// same constant in every column is not streamed
constexpr int BND_L0 = 1;        // every l is +0.0 (bitwise: -0.0 keeps the stream)
constexpr int BND_UINF = 2;      // every u is +inf

// primal half of T(z) + reflection + Halpern combine.  g = (A'y)_j
// GHOST (multi-GPU plain iterations): gathers y from this rank's ghost vector and publishes x-bar into the peers'.
// Plain single-GPU iterations (CARRY) carry x-bar instead of x: x = halpern_x(w_prev, x-bar, x0) is rebuilt from the staged
// operands, x-bar is overwritten in place (the dual kernel that gathers it has finished), and x itself is only stored
// when `store_x` is set — by the last iteration of a chunk, for the check kernels that read it.  `from_x`: operand 0 is
// x itself (x-bar does not belong to x, e.g. right after a restart).
template <bool CHECK, bool GHOST = false, int BND = 0>
struct PrimalEpi {
    static constexpr bool CARRY = !CHECK && !GHOST;
    static_assert(BND == 0 || CARRY, "constant bounds are a plain single-GPU specialisation");
    static constexpr bool HAS_L = !(BND & BND_L0), HAS_U = !(BND & BND_UINF);
    static constexpr int NIN = (CHECK ? 4 : 5) - !HAS_L - !HAS_U, NINB = 0;
    static constexpr bool SCATTER = false;
    static constexpr bool DIST = GHOST;
    double* scat;
    const double* __restrict__ c;
    const double* __restrict__ l;
    const double* __restrict__ u;
    const double* __restrict__ x0;
    double* __restrict__ x;
    double* __restrict__ xbar;
    double* __restrict__ xp;
    const PdlpParams* __restrict__ P;
    int it;
    GhostIn gin;        // y ghost (consumed)
    GhostOut gout;      // x-bar ghosts (produced)
    int from_x = 1, store_x = 1;      // CARRY only (see above)
    using Route = GhostRoute;
    struct Pre { double x, c, l, u, x0; };
    __device__ __forceinline__ bool reads_xbar() const { return CARRY && !from_x; }
    // operands: x (x-bar when carried), c, l, u, x0 — without the bounds BND makes constants, without x0 in a check
    __device__ __forceinline__ const double* in(int i) const {
        if (i == 0) return reads_xbar() ? xbar : x;
        if (i == 1) return c;
        if (HAS_L && i == 2) return l;
        if (HAS_U && i == 2 + HAS_L) return u;
        return x0;
    }
    __device__ __forceinline__ const int8_t* in_b(int) const { return nullptr; }
    __device__ __forceinline__ Pre preload(const double* s, int rt, int g) const {
        Pre p;
        p.x = s[g]; p.c = s[rt + g];
        p.l = HAS_L ? s[2 * rt + g] : 0.0;
        p.u = HAS_U ? s[(2 + HAS_L) * rt + g] : INFINITY;
        p.x0 = CHECK ? 0.0 : s[(NIN - 1) * rt + g];
        return p;
    }
    __device__ __forceinline__ Pre preload_global(int j) const {
        Pre p;
        p.x = reads_xbar() ? xbar[j] : x[j]; p.c = c[j];
        p.l = HAS_L ? l[j] : 0.0;
        p.u = HAS_U ? u[j] : INFINITY;
        p.x0 = CHECK ? 0.0 : x0[j];
        return p;
    }
    __device__ __forceinline__ double apply(int j, double g, const Pre& p, const L2Hints& h) const {
        const double tau = P->tau;
        // the previous iteration formed x with the weight of k - 1
        const double xk = reads_xbar() ? halpern_x(halpern_w(P->k_base + it - 1), p.x, p.x0) : p.x;
        const double xpj = fmin(fmax(xk - tau * (p.c - g), p.l), p.u);
        const double xb = 2.0 * xpj - xk;
        if (!GHOST) st_out(xbar + j, xb, h, true);
        if (CHECK) {
            xp[j] = xpj;
        } else if (!CARRY || store_x) {
            st_out(x + j, halpern_x(halpern_w(P->k_base + it), xb, p.x0), h, false);
        }
        return GHOST ? xb : 0.0;
    }
    // y of the previous iteration carries epoch_base + it; this launch produces epoch_base + it + 1
    __device__ __forceinline__ void acquire(int lane) const { ghost_acquire(gin, P->epoch_base + it, lane); }
    __device__ __forceinline__ const uint32_t* route_table() const { return gout.route; }
    __device__ __forceinline__ Route route(const uint32_t* rec, int lane, bool owner, int row_in_tile) const {
        return ghost_route(gout, rec, lane, owner, row_in_tile);
    }
    __device__ __forceinline__ void publish(const Route& rt, int lane, int row, double v) const {
        ghost_publish(gout, rt, lane, row, v);
    }
    __host__ __device__ __forceinline__ int push_ctas() const { return gout.push_ctas; }
    __device__ __forceinline__ void push(int pw, int npw, int lane) const { ghost_push_role(gout, pw, npw, lane); }
};

// dual half.  ax = (A xbar)_i.  SCAT: the kernel then adds val[k] * y_new_i into scat[idx[k]] over the entries of row i,
// i.e. it leaves g = A'y_new behind for the next (gather-free) primal update.
// GHOST (multi-GPU plain iterations): gathers x-bar from this rank's ghost vector and publishes y into the peers'.
// RHS (plain single-GPU iterations): the row bounds are rebuilt from the scaled right-hand side and the sense byte,
// lc = (LE ? -inf : rhs), uc = (GE ? +inf : rhs) — 9 bytes per row instead of 16; only where that gives lc / uc exactly.
template <bool CHECK, bool SCAT = false, bool GHOST = false, bool RHS = false>
struct DualEpi {
    static_assert(!RHS || (!CHECK && !SCAT && !GHOST), "the rhs + sense stream is a plain single-GPU specialisation");
    static constexpr int NIN = CHECK || RHS ? 3 : 4, NINB = RHS ? 1 : 0;
    static constexpr bool SCATTER = SCAT;
    static constexpr bool DIST = GHOST;
    double* scat;
    const double* __restrict__ lc;
    const double* __restrict__ uc;
    const double* __restrict__ y0;
    double* __restrict__ y;
    double* __restrict__ yp;
    double* __restrict__ axbar;
    const PdlpParams* __restrict__ P;
    int it;
    GhostIn gin;        // x-bar ghost (consumed)
    GhostOut gout;      // y ghosts (produced)
    const double* __restrict__ rhs = nullptr;     // RHS only: scaled right-hand side and sense of every row
    const int8_t* __restrict__ sense = nullptr;
    using Route = GhostRoute;
    struct Pre { double y, lc, uc, y0; };
    __device__ __forceinline__ const double* in(int i) const {
        if (RHS) return i == 0 ? y : i == 1 ? rhs : y0;
        return i == 0 ? y : i == 1 ? lc : i == 2 ? uc : y0;
    }
    __device__ __forceinline__ const int8_t* in_b(int) const { return sense; }
    static __device__ __forceinline__ void bounds_of(int sn, double r, Pre& p) {
        p.lc = sn == ELP_LE ? -INFINITY : r;
        p.uc = sn == ELP_GE ? INFINITY : r;
    }
    __device__ __forceinline__ Pre preload(const double* s, int rt, int g) const {
        Pre p;
        p.y = s[g];
        if (RHS) bounds_of(reinterpret_cast<const int8_t*>(s + NIN * rt)[g], s[rt + g], p);
        else { p.lc = s[rt + g]; p.uc = s[2 * rt + g]; }
        p.y0 = CHECK ? 0.0 : s[(NIN - 1) * rt + g];
        return p;
    }
    __device__ __forceinline__ Pre preload_global(int i) const {
        Pre p;
        p.y = y[i];
        if (RHS) bounds_of(sense[i], rhs[i], p);
        else { p.lc = lc[i]; p.uc = uc[i]; }
        p.y0 = CHECK ? 0.0 : y0[i];
        return p;
    }
    __device__ __forceinline__ double apply(int i, double ax, const Pre& p, const L2Hints& h) const {
        const double sigma = P->sigma;
        const double v = p.y - sigma * ax;
        const double lo = v + sigma * p.lc;     // -inf when the row has no lower bound
        const double hi = v + sigma * p.uc;     // +inf when the row has no upper bound
        const double ypi = lo > 0.0 ? lo : (hi < 0.0 ? hi : 0.0);
        if (CHECK) {
            yp[i] = ypi;
            axbar[i] = ax;
        } else {
            const double k = (double)(P->k_base + it);
            const double w = (k + 1.0) / (k + 2.0);
            const double yn = w * (2.0 * ypi - p.y) + (1.0 - w) * p.y0;
            st_out(y + i, yn, h, !GHOST);       // with ghosts nobody gathers from the home block
            return yn;
        }
        return 0.0;
    }
    // the x-bar of this same iteration carries epoch_base + it + 1, and so does the y this launch produces
    __device__ __forceinline__ void acquire(int lane) const { ghost_acquire(gin, P->epoch_base + it + 1, lane); }
    __device__ __forceinline__ const uint32_t* route_table() const { return gout.route; }
    __device__ __forceinline__ Route route(const uint32_t* rec, int lane, bool owner, int row_in_tile) const {
        return ghost_route(gout, rec, lane, owner, row_in_tile);
    }
    __device__ __forceinline__ void publish(const Route& rt, int lane, int row, double v) const {
        ghost_publish(gout, rt, lane, row, v);
    }
    __host__ __device__ __forceinline__ int push_ctas() const { return gout.push_ctas; }
    __device__ __forceinline__ void push(int pw, int npw, int lane) const { ghost_push_role(gout, pw, npw, lane); }
};

// Gather-free primal update of the scatter formulation: g = A'y was accumulated by the previous dual kernel.
// Reads g, x, c, l, u, x0; writes x-bar, x and clears g for the next accumulation.  Two columns per thread (16-byte accesses).
__global__ void __launch_bounds__(256)
k_primal_from_g(int n, double* __restrict__ g, const double* __restrict__ c, const double* __restrict__ l,
                const double* __restrict__ u, const double* __restrict__ x0, double* __restrict__ x,
                double* __restrict__ xbar, const PdlpParams* __restrict__ P, int it) {
    const double tau = P->tau;
    const double k = (double)(P->k_base + it);
    const double w = (k + 1.0) / (k + 2.0);
    const int npair = n >> 1;
    for (int q = blockIdx.x * 256 + threadIdx.x; q < npair; q += gridDim.x * 256) {
        const double2 gv = reinterpret_cast<const double2*>(g)[q];
        const double2 xv = reinterpret_cast<const double2*>(x)[q];
        const double2 cv = reinterpret_cast<const double2*>(c)[q];
        const double2 lv = reinterpret_cast<const double2*>(l)[q];
        const double2 uv = reinterpret_cast<const double2*>(u)[q];
        const double2 av = reinterpret_cast<const double2*>(x0)[q];
        const double p0 = fmin(fmax(xv.x - tau * (cv.x - gv.x), lv.x), uv.x);
        const double p1 = fmin(fmax(xv.y - tau * (cv.y - gv.y), lv.y), uv.y);
        const double b0 = 2.0 * p0 - xv.x, b1 = 2.0 * p1 - xv.y;
        reinterpret_cast<double2*>(xbar)[q] = make_double2(b0, b1);
        reinterpret_cast<double2*>(x)[q] = make_double2(w * b0 + (1.0 - w) * av.x, w * b1 + (1.0 - w) * av.y);
        reinterpret_cast<double2*>(g)[q] = make_double2(0.0, 0.0);
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
        const int j = n - 1;
        const double xj = x[j];
        const double pj = fmin(fmax(xj - tau * (c[j] - g[j]), l[j]), u[j]);
        const double bj = 2.0 * pj - xj;
        xbar[j] = bj;
        x[j] = w * bj + (1.0 - w) * x0[j];
        g[j] = 0.0;
    }
}

// lanes per row for the setup-only helper kernels (row statistics, value scaling, row expansion)
inline int pick_helper_lanes(int64_t nnz, int64_t nrows) {
    const double avg = nrows > 0 ? (double)nnz / (double)nrows : 0.0;
    int L = 1;
    while (L < 32 && (double)(2 * L) <= avg * 0.75 + 1.0) L *= 2;   // avg 10 -> 8, avg 5 -> 4, avg 2 -> 1..2
    return L;
}

// ---- row statistics for the scaling: out[r] = s_self[r] * reduce_k |val[k]| * s_other[idx[k]] ------
template <int L, int MODE /*0 max, 1 sum*/>
__global__ void __launch_bounds__(SPMV_THREADS)
rowstat_kernel(int nrows, const int* __restrict__ ptr, const int* __restrict__ idx, const double* __restrict__ val,
               const double* __restrict__ s_self, const double* __restrict__ s_other, double* __restrict__ out) {
    const int row = (int)(((int64_t)blockIdx.x * SPMV_THREADS + threadIdx.x) / L);
    const int lane = threadIdx.x & (L - 1);
    int start = 0, end = 0;
    if (row < nrows) { start = ptr[row]; end = ptr[row + 1]; }
    double s = 0.0;
    for (int k = start + lane; k < end; k += L) {
        const double a = fabs(val[k]) * s_other[idx[k]];
        s = MODE == 0 ? fmax(s, a) : s + a;
    }
    s = MODE == 0 ? group_max<L>(s) : group_sum<L>(s);
    if (lane == 0 && row < nrows) out[row] = s * s_self[row];
}

template <int L>
__global__ void __launch_bounds__(SPMV_THREADS)
scale_vals_kernel(int nrows, const int* __restrict__ ptr, const int* __restrict__ idx, double* __restrict__ val,
                  const double* __restrict__ s_self, const double* __restrict__ s_other) {
    const int row = (int)(((int64_t)blockIdx.x * SPMV_THREADS + threadIdx.x) / L);
    const int lane = threadIdx.x & (L - 1);
    if (row >= nrows) return;
    const double sr = s_self[row];
    for (int k = ptr[row] + lane; k < ptr[row + 1]; k += L) val[k] *= sr * s_other[idx[k]];
}

template <int L>
__global__ void __launch_bounds__(SPMV_THREADS)
expand_rows_kernel(int nrows, const int* __restrict__ ptr, int* __restrict__ row_of) {
    const int row = (int)(((int64_t)blockIdx.x * SPMV_THREADS + threadIdx.x) / L);
    const int lane = threadIdx.x & (L - 1);
    if (row >= nrows) return;
    for (int k = ptr[row] + lane; k < ptr[row + 1]; k += L) row_of[k] = row;
}

// ---- small elementwise kernels ----------------------------------------------------------------
__global__ void k_ruiz_update(int n, double* __restrict__ d, const double* __restrict__ stat) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { const double s = stat[i]; if (s > 0.0) d[i] *= rsqrt(s); }
}
__global__ void k_fill(int n, double* __restrict__ d, double v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = v;
}
__global__ void k_mul(int n, double* __restrict__ d, const double* __restrict__ s) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] *= s[i];
}
__global__ void k_div(int n, double* __restrict__ d, const double* __restrict__ s) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] /= s[i];
}
__global__ void k_scale_scalar(int n, double* __restrict__ d, double a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] *= a;
}
__global__ void k_row_bounds(int m, const int8_t* __restrict__ sense, const double* __restrict__ rhs,
                             double* __restrict__ lc, double* __restrict__ uc) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int s = sense[i];
    const double r = rhs[i];
    lc[i] = (s == ELP_LE) ? -INFINITY : r;
    uc[i] = (s == ELP_GE) ? INFINITY : r;
}
// setup: bit 0 some l is not +0.0, bit 1 some u is not +inf, bit 2 some row whose lc / uc are not what rhs and sense
// rebuild (DualEpi<RHS>), compared bit for bit
__global__ void k_bound_kinds(int n, const double* __restrict__ l, const double* __restrict__ u, int m,
                              const int8_t* __restrict__ sense, const double* __restrict__ rhs, const double* __restrict__ lc,
                              const double* __restrict__ uc, unsigned int* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int f = 0;
    if (i < n) {
        if (__double_as_longlong(l[i]) != 0) f |= 1u;
        if (__double_as_longlong(u[i]) != __double_as_longlong(INFINITY)) f |= 2u;
    }
    if (i < m) {
        const int s = sense[i];
        const double r = rhs[i];
        if (__double_as_longlong(s == ELP_LE ? -INFINITY : r) != __double_as_longlong(lc[i]) ||
            __double_as_longlong(s == ELP_GE ? INFINITY : r) != __double_as_longlong(uc[i]))
            f |= 4u;
    }
    f = __reduce_or_sync(0xffffffffu, f);
    if ((threadIdx.x & 31) == 0 && f) atomicOr(out, f);
}
__global__ void k_init_x(int n, double* __restrict__ x, const double* __restrict__ l, const double* __restrict__ u) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) x[j] = fmin(fmax(0.0, l[j]), u[j]);
}
__global__ void k_pseudo_random(int n, double* __restrict__ v, uint32_t seed) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    uint32_t h = (uint32_t)j * 2654435761u + seed;
    h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
    v[j] = (double)h / 4294967296.0 - 0.5;
}
// after a check without restart: finish the Halpern step from the stored candidate
__global__ void k_halpern_finish(int n, double* __restrict__ x, const double* __restrict__ xbar,
                                 const double* __restrict__ x0, int m, double* __restrict__ y,
                                 const double* __restrict__ yp, const double* __restrict__ y0, double w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = halpern_x(w, xbar[i], x0[i]);
    if (i < m) y[i] = w * (2.0 * yp[i] - y[i]) + (1.0 - w) * y0[i];
}
// restart: iterate and anchor both jump to the candidate T(z)
__global__ void k_restart(int n, double* __restrict__ x, double* __restrict__ x0, const double* __restrict__ xp, int m,
                          double* __restrict__ y, double* __restrict__ y0, const double* __restrict__ yp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { const double v = xp[i]; x[i] = v; x0[i] = v; }
    if (i < m) { const double v = yp[i]; y[i] = v; y0[i] = v; }
}
__global__ void k_unscale(int n, const double* __restrict__ v, const double* __restrict__ s, double sign,
                          double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = sign * v[i] * s[i];
}

// ---- reductions: per-block partials in fixed order, then one block folds them --------------------
constexpr int RED_THREADS = 256;
constexpr int RED_BLOCKS = kNumSMs * 4;
constexpr int NACC = 8;

__device__ __forceinline__ void block_reduce_store(double (&acc)[NACC], double* __restrict__ partials) {
    __shared__ double sm[RED_THREADS / 32][NACC];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NACC; ++k) {
        const double v = warp_sum(acc[k]);
        if (lane == 0) sm[warp][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < NACC) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < RED_THREADS / 32; ++w) s += sm[w][threadIdx.x];
        partials[blockIdx.x * NACC + threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(RED_THREADS)
k_final_reduce(const double* __restrict__ partials, int nblocks, double* __restrict__ out) {
    __shared__ double sm[RED_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = 0; k < NACC; ++k) {
        double s = 0.0;
        for (int b = threadIdx.x; b < nblocks; b += RED_THREADS) s += partials[b * NACC + k];
        s = warp_sum(s);
        if (lane == 0) sm[warp] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < RED_THREADS / 32; ++w) t += sm[w];
            out[k] = t;
        }
        __syncthreads();
    }
}

// row-side check sums.  acc: 0 pres^2 (unscaled), 1 dy.(A dx), 2 |dy|^2, 3 |yp-y0|^2, 4 dual obj (rows),
//                            5 yp.(A xp - proj): objective error the primal residual can hide, 6 unused,
//                            7 reserved (multi-GPU: wall-clock agreement)
__global__ void __launch_bounds__(RED_THREADS)
k_check_rows(int m, const double* __restrict__ axp, const double* __restrict__ axbar, const double* __restrict__ y,
             const double* __restrict__ yp, const double* __restrict__ y0, const double* __restrict__ lc,
             const double* __restrict__ uc, const double* __restrict__ dr, double* __restrict__ partials) {
    double acc[NACC] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = blockIdx.x * RED_THREADS + threadIdx.x; i < m; i += gridDim.x * RED_THREADS) {
        const double a = axp[i], lo = lc[i], hi = uc[i];
        const double off = a - fmin(fmax(a, lo), hi);
        const double viol = off / dr[i];
        const double ypi = yp[i];
        acc[5] += ypi * off;                       // first-order effect of the primal infeasibility on the objective (scale-invariant)
        const double dy = ypi - y[i];
        const double d0 = ypi - y0[i];
        acc[0] += viol * viol;
        acc[1] += dy * (axbar[i] - a);
        acc[2] += dy * dy;
        acc[3] += d0 * d0;
        acc[4] += ypi > 0.0 ? ypi * lo : (ypi < 0.0 ? ypi * hi : 0.0);
    }
    block_reduce_store(acc, partials);
}

// column-side check sums.  acc: 0 dres^2 (unscaled), 1 |dx|^2, 2 |xp-x0|^2, 3 c'xp, 4 dual obj (bounds),
//                               5 xp.(dual residual): objective error the dual residual can hide
__global__ void __launch_bounds__(RED_THREADS)
k_check_cols(int n, const double* __restrict__ g, const double* __restrict__ c, const double* __restrict__ l,
             const double* __restrict__ u, const double* __restrict__ x, const double* __restrict__ xp,
             const double* __restrict__ x0, const double* __restrict__ dc, double* __restrict__ partials) {
    double acc[NACC] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int j = blockIdx.x * RED_THREADS + threadIdx.x; j < n; j += gridDim.x * RED_THREADS) {
        const double r = c[j] - g[j];
        const double xpj = xp[j], lj = l[j], uj = u[j];
        const bool at_lo = isfinite(lj) && xpj <= lj;
        const bool at_hi = isfinite(uj) && xpj >= uj;
        const double rpos = fmax(r, 0.0), rneg = fmin(r, 0.0);
        const double res = ((at_lo ? 0.0 : rpos) + (at_hi ? 0.0 : rneg)) / dc[j];
        const double dx = xpj - x[j];
        const double d0 = xpj - x0[j];
        acc[0] += res * res;
        acc[1] += dx * dx;
        acc[2] += d0 * d0;
        acc[3] += c[j] * xpj;
        acc[4] += (at_lo ? rpos * lj : 0.0) + (at_hi ? rneg * uj : 0.0);
        acc[5] += ((at_lo ? 0.0 : rpos) + (at_hi ? 0.0 : rneg)) * xpj;   // the same for the dual infeasibility
    }
    block_reduce_store(acc, partials);
}

// generic: acc0 = sum a^2, acc1 = sum a*b (b may alias a), for norms / dot products
__global__ void __launch_bounds__(RED_THREADS)
k_dot2(int n, const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ partials) {
    double acc[NACC] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = blockIdx.x * RED_THREADS + threadIdx.x; i < n; i += gridDim.x * RED_THREADS) {
        const double ai = a[i];
        acc[0] += ai * ai;
        acc[1] += ai * b[i];
    }
    block_reduce_store(acc, partials);
}

// sum of squares of the finite row-bound magnitudes (PDLP's ||b||) -> acc0 ; acc1 = sum c^2 style helper
__global__ void __launch_bounds__(RED_THREADS)
k_bound_norm(int m, const double* __restrict__ lc, const double* __restrict__ uc, double* __restrict__ partials) {
    double acc[NACC] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = blockIdx.x * RED_THREADS + threadIdx.x; i < m; i += gridDim.x * RED_THREADS) {
        const double lo = lc[i], hi = uc[i];
        const double a = fmax(isfinite(lo) ? fabs(lo) : 0.0, isfinite(hi) ? fabs(hi) : 0.0);
        acc[0] += a * a;
    }
    block_reduce_store(acc, partials);
}

// certificate sums on the displacement ray (dx = xp - x0 over columns)
//  cols: 0 c'dx, 1 bound violation^2 of the ray, 2 max|dx| (as sum of squares -> use norm), 3 |dx|^2
__global__ void __launch_bounds__(RED_THREADS)
k_ray_cols(int n, const double* __restrict__ xp, const double* __restrict__ x0, const double* __restrict__ c,
           const double* __restrict__ l, const double* __restrict__ u, const double* __restrict__ gray,
           const double* __restrict__ dc, double* __restrict__ partials) {
    // gray = A'(yp - y0) (scaled).  Unscaled ray quantities: dx_u = dx*dc, (A'dy)_u = gray/dc
    double acc[NACC] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int j = blockIdx.x * RED_THREADS + threadIdx.x; j < n; j += gridDim.x * RED_THREADS) {
        const double dxs = xp[j] - x0[j];
        const double dxu = dxs * dc[j];
        const double lj = l[j], uj = u[j];
        acc[0] += c[j] * dxs;                                   // c'dx (scale-invariant)
        double vb = 0.0;                                        // ray must not push against finite bounds
        if (isfinite(lj) && dxu < 0.0) vb += dxu;
        if (isfinite(uj) && dxu > 0.0) vb += dxu;
        acc[1] += vb * vb;
        acc[3] += dxu * dxu;
        // dual ray: reduced cost of the ray r = -A'dy ; parts no finite bound can absorb are residual
        const double r = -gray[j];
        const double rpos = fmax(r, 0.0), rneg = fmin(r, 0.0);
        const double res = ((isfinite(lj) ? 0.0 : rpos) + (isfinite(uj) ? 0.0 : rneg)) / dc[j];
        acc[4] += res * res;
        acc[5] += (isfinite(lj) ? rpos * lj : 0.0) + (isfinite(uj) ? rneg * uj : 0.0);   // bound part of ray objective
    }
    block_reduce_store(acc, partials);
}
// rows: axray = A (xp - x0) (scaled; unscaled = /dr) ; dy = yp - y0 (unscaled = *dr)
__global__ void __launch_bounds__(RED_THREADS)
k_ray_rows(int m, const double* __restrict__ axray, const double* __restrict__ yp, const double* __restrict__ y0,
           const double* __restrict__ lc, const double* __restrict__ uc, const double* __restrict__ dr,
           double* __restrict__ partials) {
    double acc[NACC] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = blockIdx.x * RED_THREADS + threadIdx.x; i < m; i += gridDim.x * RED_THREADS) {
        const double a = axray[i] / dr[i];
        const double lo = lc[i], hi = uc[i];
        double v = 0.0;                                         // primal ray: A dx must stay inside the recession cone
        if (isfinite(lo) && a < 0.0) v += a;
        if (isfinite(hi) && a > 0.0) v += a;
        acc[0] += v * v;
        const double dys = yp[i] - y0[i];
        const double dyu = dys * dr[i];
        acc[1] += dyu * dyu;
        // dual ray objective (rows): dy+ * lc + dy- * uc (scale-invariant); infinite-side components are violations
        if (dys > 0.0) { if (isfinite(lo)) acc[2] += dys * lo; else acc[3] += dyu * dyu; }
        else if (dys < 0.0) { if (isfinite(hi)) acc[2] += dys * hi; else acc[3] += dyu * dyu; }
    }
    block_reduce_store(acc, partials);
}

// ---- small launch helpers used by build_csc / certificates --
__global__ void k_transpose_keys(const int* __restrict__ col, uint32_t nnz, uint64_t* __restrict__ keys,
                                 uint32_t* __restrict__ perm) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) { keys[i] = (uint64_t)(uint32_t)col[i]; perm[i] = i; }
}
__global__ void k_transpose_gather(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ perm,
                                   const int* __restrict__ row_of, const double* __restrict__ val, uint32_t nnz,
                                   int* __restrict__ csc_idx, double* __restrict__ csc_val, int* __restrict__ cols_sorted,
                                   uint32_t* __restrict__ nnz_d) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *nnz_d = nnz;
    if (i >= nnz) return;
    const uint32_t p = perm[i];
    csc_idx[i] = row_of[p];
    csc_val[i] = val[p];
    cols_sorted[i] = (int)keys[i];
}
__global__ void k_fill_ptr(const int* __restrict__ sorted_ids, const uint32_t* __restrict__ nnz_ptr, uint32_t nseg,
                           int* __restrict__ ptr, uint32_t cap) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t nnz = *nnz_ptr;
    if (i > nnz || i > cap) return;
    const int prev = (i == 0) ? -1 : sorted_ids[i - 1];
    const int cur = (i == nnz) ? (int)nseg : sorted_ids[i];
    for (int r = prev + 1; r <= cur; ++r) ptr[r] = (int)i;
}
__global__ void k_diff(int n, const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = a[i] - b[i];
}
void launch_transpose_keys(const int* col, uint32_t nnz, uint64_t* keys, uint32_t* perm, cudaStream_t st) {
    ELP_LAUNCH(k_transpose_keys, ceil_div(nnz, 256), 256, 0, st, col, nnz, keys, perm);
}
void launch_transpose_gather(const uint64_t* keys, const uint32_t* perm, const int* row_of, const double* val,
                             uint32_t nnz, int* csc_idx, double* csc_val, int* cols_sorted, uint32_t* nnz_d,
                             cudaStream_t st) {
    ELP_LAUNCH(k_transpose_gather, ceil_div(nnz, 256), 256, 0, st, keys, perm, row_of, val, nnz, csc_idx, csc_val,
               cols_sorted, nnz_d);
}
void launch_fill_ptr(const int* sorted_ids, const uint32_t* nnz_ptr, uint32_t nseg, int* ptr, uint32_t cap,
                     cudaStream_t st) {
    ELP_LAUNCH(k_fill_ptr, ceil_div((int64_t)cap + 1, 256), 256, 0, st, sorted_ids, nnz_ptr, nseg, ptr, cap);
}
void launch_diff(int n, const double* a, const double* b, double* out, cudaStream_t st) {
    if (n > 0) ELP_LAUNCH(k_diff, ceil_div(n, 256), 256, 0, st, n, a, b, out);
}

// ---- setup of the ghost exchange (multi-GPU) -----------------------------------------------------------------
__global__ void k_mark_used(uint32_t nnz, const int* __restrict__ idx, unsigned char* __restrict__ used) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) used[idx[i]] = 1;                       // same value from every writer
}
__global__ void k_marks_to_u32(uint32_t count, const unsigned char* __restrict__ used, uint32_t* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= count) out[i] = i < count ? (used[i] ? 1u : 0u) : 0u;     // one extra slot: the scan leaves the total there
}
// compact ids of my matrix copy: position of every referenced global id in my ghost vector
__global__ void k_remap_idx(uint32_t nnz, const int* __restrict__ idx, const uint32_t* __restrict__ pos, int* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) out[i] = (int)pos[idx[i]];
}
__global__ void k_fill_u64(size_t n, unsigned long long* __restrict__ out, unsigned long long v) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = v;
}
// routing record of my tile t, word r = position, in rank r's ghost vector, of the tile's first entry (pos = scan of r's marks)
// (record `ntiles` closes the table: the position just behind my block, `count` rows after `first`)
__global__ void k_tile_base(int ntiles, int rw, int first, int count, const uint32_t* __restrict__ pos, int r, uint32_t* __restrict__ route) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t <= ntiles) route[(size_t)t * SPMV_ROUTE_WORDS + r] = pos[first + min(t * rw, count)];
}
// bytes 32.. of the record: one mask per row of the tile
__global__ void k_route_masks(int count, int rw, const unsigned char* __restrict__ mask, uint32_t* __restrict__ route) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < count) reinterpret_cast<unsigned char*>(route)[(size_t)(j / rw) * (SPMV_ROUTE_WORDS * 4) + 32 + (j % rw)] = mask[j];
}
__global__ void k_ghost_list(uint32_t count, const unsigned char* __restrict__ used, const uint32_t* __restrict__ pos, int* __restrict__ list) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count && used[i]) list[pos[i]] = (int)i;
}
// mask[j] bit r: rank r gathers entry first + j
__global__ void k_ghost_mask(int count, int first, size_t stride, int nranks, const unsigned char* __restrict__ used_all,
                             unsigned char* __restrict__ mask, unsigned long long* __restrict__ sent) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    unsigned mk = 0;
    for (int r = 0; r < nranks; ++r) mk |= (used_all[(size_t)r * stride + first + j] ? 1u : 0u) << r;
    mask[j] = (unsigned char)mk;
    atomicAdd(sent, (unsigned long long)__popc(mk));
}
// ghost[k] = full[list[k]]  (after a collective refreshed the full-layout vector)
__global__ void k_compact(int count, const int* __restrict__ list, const double* __restrict__ full, double* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < count) out[k] = full[list[k]];
}

// a rank without columns (rows) launches no K1 (K2): this stands in for the kernel's prologue
__global__ void k_ghost_signal_only(GhostIn gi, const PdlpParams* __restrict__ P, int plus) {
    if (threadIdx.x == 0) {
        __threadfence_system();
        for (int r = 0; r < gi.n; ++r) st_relaxed_sys(gi.peer_flag[r] + gi.rank, (unsigned long long)(P->epoch_base + plus));
    }
}

// ---- kernels of the one-off exchange that builds each rank's column block of A ---------------------
__global__ void k_shift_idx(uint32_t nnz, int* __restrict__ idx, int offset) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) idx[i] += offset;
}
// lens[j] = length of local CSC column j0 + j (0 beyond the matrix)
__global__ void k_col_lens(const int* __restrict__ ptr, int j0, int count, int ncols, uint32_t* __restrict__ lens) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const int col = j0 + j;
    lens[j] = col < ncols ? (uint32_t)(ptr[col + 1] - ptr[col]) : 0u;
}
__global__ void k_sum_lens(int nranks, int nb, const uint32_t* __restrict__ lens, uint32_t* __restrict__ tot) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j > nb) return;
    uint32_t s = 0;
    if (j < nb) for (int r = 0; r < nranks; ++r) s += lens[(size_t)r * nb + j];
    tot[j] = s;                                      // tot[nb] = 0: the scan leaves the total there
}
// column j of my block = concatenation over the source ranks (ascending = ascending global row) of their pieces
__global__ void k_merge_cols(int nranks, int nb, const uint32_t* __restrict__ lens, const uint32_t* __restrict__ srcptr,
                             const uint32_t* __restrict__ newptr, const uint32_t* __restrict__ roff,
                             const int* __restrict__ in_idx, const double* __restrict__ in_val,
                             int* __restrict__ out_ptr, int* __restrict__ out_idx, double* __restrict__ out_val) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j > nb) return;
    out_ptr[j] = (int)newptr[j];
    if (j == nb) return;
    uint32_t dst = newptr[j];
    for (int r = 0; r < nranks; ++r) {
        const uint32_t len = lens[(size_t)r * nb + j];
        const uint32_t src = roff[r] + srcptr[(size_t)r * nb + j];
        for (uint32_t k = 0; k < len; ++k) { out_idx[dst + k] = in_idx[src + k]; out_val[dst + k] = in_val[src + k]; }
        dst += len;
    }
}

// ------------------------------------------------------------------------------------------------
// host-side solver object
//
// Partition (N ranks; N = 1 is the same code with the collectives compiled out of the picture):
//   rows     rank g owns the row block the caller hands it (balanced by non-zeros): CSR with GLOBAL column ids,
//            the slices of y / lc / uc.  y lives in a padded global layout y_full[N][mb] (mb = largest block).
//   columns  rank g owns the columns [g*nb, (g+1)*nb): the CSC of that column block over ALL rows (built once by
//            a grouped send/recv of the ranks' local CSC slices), the slices of x / c / l / u.
//   K1 (A'y + primal update) runs on the column block and gathers from y_full; it writes its x-bar block into
//   xbar_full, which is then all-gathered.  K2 (A x-bar + dual update) runs on the row block and gathers from
//   xbar_full; it updates its y block inside y_full, which is then all-gathered.  All work is sharded (nothing is
//   replicated), the exchange per iteration is 8 (n + m) bytes received per rank, and the scalar residuals of a
//   check travel in one 16-double allreduce.
// ------------------------------------------------------------------------------------------------
struct Pdlp {
    // single GPU: every persistent buffer of the handle is a piece of `arena` (one cudaMalloc / cudaFree instead of ~40),
    // the temporaries of the setup pieces of `scratch` (freed when the setup is over).  Declared first: destroyed last.
    Arena arena, scratch;
    int N = 1, rank = 0;
    int m = 0, mb = 0;          // local rows, padded rows per rank
    int n = 0, nb = 0, n0 = 0, nl = 0;   // global columns, columns per rank, my first column, my column count
    int64_t nnz = 0, nnzc = 0;  // entries of the row block / of the column block
    bool maximize = false;
    elp_options opt{};
    cudaStream_t st = nullptr;
    // matrix (scaled in place after setup)
    DevBuf<int> csr_ptr, csr_idx, csc_ptr, csc_idx;
    DevBuf<double> csr_val, csc_val;
    int Lr = 8, Lc = 4;          // lanes per row of the setup helper kernels
    SpmvPlan plan_r, plan_c;     // tile plans of the two iteration SpMVs (CSR rows / CSC columns)
    // vectors (scaled); column-side ones have nl entries, row-side ones m
    DevBuf<double> c, l, u, dc, x, x0, xp, gcol;
    DevBuf<double> lc, uc, dr, y0, yp, axbar, axp;
    DevBuf<double> rs;           // scaled right-hand side: lc = (LE ? -inf : rs), uc = (GE ? +inf : rs)
    DevBuf<int8_t> rsense;       // row senses, padded to 16-byte copies
    int pbnd = 0;                // plain iterations: bounds that are constants (BND_L0 | BND_UINF), single GPU
    bool drhs = false;           // plain iterations: the dual epilogue streams rs + rsense instead of lc + uc
    DevBuf<double> xbar_full, y_full, xaux_full, yaux_full;   // [N*nb], [N*mb]: gathered vectors + scratch
    // peer-store exchange (N > 1, CUDA IPC): every rank's xbar_full / y_full / flag rows mapped here
    bool scatter = false;        // plain iterations: g = A'y accumulated by the dual kernel's scatter (single GPU only)
    SpmvPlan plan_s;             // tile plan of the scatter kernel (CSR rows)
    // ghost exchange (N > 1): compact ghost vectors filled by the peers' kernels, see GhostOut / GhostIn
    bool ghost = false;
    DevBuf<int> csr_idx_g, csc_idx_g;    // the matrix copies' ids in the compact numbering of my ghost vectors
    DevBuf<unsigned char> xmask, ymask;  // which ranks gather entry j of my x-bar / y block
    DevBuf<uint32_t> xroute, yroute;     // [tiles][SPMV_ROUTE_WORDS] routing records of what K1 / K2 produce
    DevBuf<int> ylist;                   // global (padded) ids of my y ghost entries, ascending
    DevBuf<unsigned long long> ghost_trace;   // ELP_GHOST_DEBUG bit 64
    DevBuf<unsigned char> ghost_mem;     // flag rows, error word, CTA counters, x-bar ghost x2, y ghost x2 (mapped by the peers)
    int gx = 0, gy = 0;                  // entries of my ghost vectors
    GhostIn xin{}, yin{};
    GhostOut xout{}, yout{};
    long long epoch_base = 0;            // never reset: the flag rows only grow
    // push mode (compact ghosts): local outboxes + pusher CTAs inside the SpMV grids, see ghost_push_role
    bool push = false;
    DevBuf<double> xoutbox, youtbox;
    double exch_frac_x = 1.0, exch_frac_y = 1.0;   // fraction of the dense (N-1)-copy exchange that is actually sent
    std::vector<void*> ipc_opened;
    DevBuf<double> partials, scal;                              // scal: 2*NACC
    DevBuf<PdlpParams> params;
    // scalars
    double eta = 1.0, w = 1.0, w_init = 1.0, norm_b = 0.0, norm_c = 0.0, sigma_max = 0.0;
    int k = 0, total = 0, restarts = 0;
    double fpe0 = -1.0, fpe_prev = -1.0;
    double beta_artificial = 0.36;   // artificial restart once the epoch is this fraction of all iterations so far
    // primal-weight controller.  kp = 0.5 is PDLP's geometric-mean smoothing (round 1); 0.85 measured at full size
    // (profiles/r2_primal_weight.jsonl): config 2 19 408 -> 10 510 iterations, config 5 2 764 -> 1 675, config 4 unchanged
    double w_kp = 0.85, w_ki = 0.0, w_kd = 0.0, w_ismooth = 0.3, w_err_sum = 0.0, w_err_prev = 0.0;
    int gap_rule = 0;                // 0: PDLP's gap test at eps/4; 1: gap + residual-induced objective error bound <= gap_factor * eps
    double gap_factor = 1.0, obj_err = 0.0;
    bool need_fpe0 = true;
    int status = ELP_STATUS_TIMEOUT;
    bool finished = false;
    double pobj = 0, dobj = 0, rel_pres = 0, rel_dres = 0, rel_gap = 0;
    int checks = 0;
    WallTimer run_clock;             // started by the first run() after a reset: lp.control(timeout=) covers the whole solve
    bool clock_running = false, time_up = false, hit_time_limit = false;
    // graph of one chunk of (check_every-1) plain iterations
    cudaGraphExec_t graph = nullptr;
    int graph_len = 0;
    int64_t h2d = 0, d2h = 0;

    // ELP_GHOST_DEBUG bit 64: per-kernel timeline of the last ~2000 iterations (rank 0 prints a summary)
    void dump_trace() {
        if (!ghost_trace.p || rank != 0) return;
        std::vector<unsigned long long> h(4096 * 4);
        if (cudaMemcpy(h.data(), ghost_trace.p, h.size() * 8, cudaMemcpyDeviceToHost) != cudaSuccess) return;
        // consecutive slots: (epoch E, K1) at 2E, (E+?, K2) ... slot index = 2 * want + kind; K1 wants E-1, K2 wants E
        double wait[2] = {0, 0}, sig[2] = {0, 0}, span[2] = {0, 0};
        long cnt[2] = {0, 0}, scnt[2] = {0, 0};
        for (int s = 0; s < 4096; ++s) {
            const unsigned long long* a = &h[(size_t)s * 4];
            if (!a[0] || !a[2]) continue;
            const int kind = s & 1;
            wait[kind] += (double)(a[2] - a[1]); sig[kind] += (double)(a[1] - a[0]); ++cnt[kind];
            // next kernel in program order: K1(want=E-1, slot 2E-2) -> K2(want=E, slot 2E+1) -> K1(want=E, slot 2E)
            const int nxt = kind == 0 ? ((s + 3) & 4095) : ((s - 1) & 4095);
            const unsigned long long* b = &h[(size_t)nxt * 4];
            if (b[0] > a[2] && b[0] - a[2] < 2000000ull) { span[kind] += (double)(b[0] - a[2]); ++scnt[kind]; }
        }
        for (int k = 0; k < 2; ++k)
            if (cnt[k])
                fprintf(stderr, "[pdlp trace] rank 0 %s: signal %.2f us, wait for the peers %.2f us, flags-seen -> next kernel's entry %.2f us (%ld samples)\n",
                        k == 0 ? "K1 (A'y + primal)" : "K2 (A xbar + dual)", sig[k] / cnt[k] * 1e-3, wait[k] / cnt[k] * 1e-3,
                        scnt[k] ? span[k] / scnt[k] * 1e-3 : 0.0, cnt[k]);
    }
    ~Pdlp() {
        const bool dbg = getenv("ELP_PDLP_DEBUG") != nullptr;
        WallTimer t;
        if (graph) cudaGraphExecDestroy(graph);
        const double t_graph = t.ms();
        if (st) cudaStreamSynchronize(st);
        dump_trace();
        for (void* p : ipc_opened) cudaIpcCloseMemHandle(p);
        if (st) cudaStreamDestroy(st);
        const double t_stream = t.ms();
        scratch.release();
        arena.release();                 // (the DevBufs inside are arena pieces: their destructors free nothing)
        if (dbg) fprintf(stderr, "[pdlp destroy] graph %.3f ms, stream %.3f ms, arenas %.3f ms\n", t_graph, t_stream - t_graph, t.ms() - t_stream);
    }

    // Builds the ghost exchange: which entries every rank gathers, their compact numbering, the producers' masks and
    // tile bases, and the peer mappings (same process: peer access; other processes: CUDA IPC).  Falls back to NCCL
    // all-gathers of the full vectors when the GPUs cannot reach each other's memory (or ELP_PDLP_P2P=0).
    static constexpr size_t GH_FLAGS_BYTES = 512;      // x flags [0,64) y flags [64,128) err 128, go words 256 (x) and 384 (y)
    void setup_ghost_exchange() {
        ghost = false;
        if (N <= 1 || N > 8 || env_int("ELP_PDLP_P2P", 1) == 0) return;
        Arena* const keep = arena.base ? &arena : nullptr;
        ArenaScope tmp(scratch.base ? &scratch : nullptr);        // temporaries; what the handle keeps goes to `keep` below
        const size_t sx = (size_t)N * nb, sy = (size_t)N * mb;
        // ---- 1. who reads what -----------------------------------------------------------------------------------
        DevBuf<unsigned char> used_x((size_t)N * sx), used_y((size_t)N * sy);
        used_x.zero(st); used_y.zero(st);
        if (nnz > 0) ELP_LAUNCH(k_mark_used, ceil_div(nnz, 256), 256, 0, st, (uint32_t)nnz, csr_idx.p, used_x.p + (size_t)rank * sx);
        if (nnzc > 0) ELP_LAUNCH(k_mark_used, ceil_div(nnzc, 256), 256, 0, st, (uint32_t)nnzc, csc_idx.p, used_y.p + (size_t)rank * sy);
        comm_allgather_bytes(used_x.p, sx, st);
        comm_allgather_bytes(used_y.p, sy, st);
        // ---- 1b. compact or dense?  Compaction pays when the ranks read a small part of each other's blocks (a
        // structured LP: config 5 keeps 23 % at N = 8 and runs 1.9x faster than with dense stores).  When they read
        // most of everything (a random matrix: config 4 keeps 92 % at N = 2, 71 % at N = 4, 55 % at N = 8) the ballots,
        // the positions and the misaligned short stores of the compact scheme cost more than the bytes they save —
        // measured: N = 2 181 vs 159 us, N = 4 130 vs 110 us per iteration — so the ghost vectors are then plain
        // copies of the whole vector (identity numbering, everything to everybody, aligned full-warp stores).
        bool dense = false;
        double kept_all = 1.0;
        {
            DevBuf<unsigned char> tmask((size_t)std::max(std::max(nl, m), 1));
            DevBuf<unsigned long long> cnt(2);
            cnt.zero(st);
            if (nl > 0) ELP_LAUNCH(k_ghost_mask, grid1(nl), 256, 0, st, nl, n0, sx, N, used_x.p, tmask.p, cnt.p);
            if (m > 0) ELP_LAUNCH(k_ghost_mask, grid1(m), 256, 0, st, m, rank * mb, sy, N, used_y.p, tmask.p, cnt.p + 1);
            unsigned long long hc[2] = {0, 0};
            ELP_CUDA(cudaMemcpyAsync(hc, cnt.p, sizeof hc, cudaMemcpyDeviceToHost, st));
            ELP_CUDA(cudaStreamSynchronize(st));
            double tot[2] = {(double)hc[0] + (double)hc[1], ((double)nl + (double)m) * N};
            ELP_CUDA(cudaMemcpyAsync(scal.p, tot, sizeof tot, cudaMemcpyHostToDevice, st));
            comm_allreduce_sum(scal.p, 2, st);
            ELP_CUDA(cudaMemcpyAsync(tot, scal.p, sizeof tot, cudaMemcpyDeviceToHost, st));
            ELP_CUDA(cudaStreamSynchronize(st));
            const double kept = tot[1] > 0 ? tot[0] / tot[1] : 1.0;
            kept_all = kept;
            const int force = env_int("ELP_PDLP_GHOST_DENSE", -1);
            dense = force >= 0 ? force != 0 : kept >= 0.65;      // measured on config 4: 55 % kept (N = 8) compact 118 vs dense 131 us, 71 % (N = 4) equal
            if (opt.verbose > 0 || env_int("ELP_PDLP_DEBUG", 0))
                fprintf(stderr, "[pdlp] rank %d: the ranks read %.1f %% of each other's blocks -> %s ghost vectors\n", rank, 100.0 * kept,
                        dense ? "dense" : "compact");
            if (dense) {                   // "everybody reads everything": the generic code below then yields identity numbering
                ELP_CUDA(cudaMemsetAsync(used_x.p, 1, (size_t)N * sx, st));
                ELP_CUDA(cudaMemsetAsync(used_y.p, 1, (size_t)N * sy, st));
            }
        }
        // ---- 2. compact numbering per consumer; my ids, my lists, the tile bases of what I produce -----------------
        ELP_REQUIRE(plan_c.rpl == 1 && plan_r.rpl == 1, "pdlp: two rows per lane is a single-GPU option");
        {
            ArenaScope k(keep);
            csr_idx_g.alloc(nnz + SPMV_PAD); csc_idx_g.alloc(nnzc + SPMV_PAD);
            xroute.alloc((size_t)(std::max(plan_c.ntiles, 1) + 1) * SPMV_ROUTE_WORDS + 4);      // + the closing record
            yroute.alloc((size_t)(std::max(plan_r.ntiles, 1) + 1) * SPMV_ROUTE_WORDS + 4);
            xmask.alloc((size_t)std::max(nl, 1)); ymask.alloc((size_t)std::max(m, 1));
            ylist.alloc(sy);                                       // at most every padded row
        }
        csr_idx_g.zero(st); csc_idx_g.zero(st);
        xroute.zero(st); yroute.zero(st);
        DevBuf<uint32_t> pos(std::max(sx, sy) + 1);
        ScanWorkspace sw;
        std::vector<uint32_t> gxs(N), gys(N);
        for (int r = 0; r < N; ++r) {
            ELP_LAUNCH(k_marks_to_u32, ceil_div((int64_t)sx + 1, 256), 256, 0, st, (uint32_t)sx, used_x.p + (size_t)r * sx, pos.p);
            exclusive_scan_u32(pos.p, sx + 1, sw, st);
            ELP_CUDA(cudaMemcpyAsync(&gxs[r], pos.p + sx, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
            if (r == rank && nnz > 0) ELP_LAUNCH(k_remap_idx, ceil_div(nnz, 256), 256, 0, st, (uint32_t)nnz, csr_idx.p, pos.p, csr_idx_g.p);
            if (nl > 0) ELP_LAUNCH(k_tile_base, ceil_div(plan_c.ntiles + 1, 256), 256, 0, st, plan_c.ntiles, plan_c.rw(), n0, nl, pos.p, r, xroute.p);
            ELP_CUDA(cudaStreamSynchronize(st));
        }
        for (int r = 0; r < N; ++r) {
            ELP_LAUNCH(k_marks_to_u32, ceil_div((int64_t)sy + 1, 256), 256, 0, st, (uint32_t)sy, used_y.p + (size_t)r * sy, pos.p);
            exclusive_scan_u32(pos.p, sy + 1, sw, st);
            ELP_CUDA(cudaMemcpyAsync(&gys[r], pos.p + sy, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
            if (r == rank) {
                if (nnzc > 0) ELP_LAUNCH(k_remap_idx, ceil_div(nnzc, 256), 256, 0, st, (uint32_t)nnzc, csc_idx.p, pos.p, csc_idx_g.p);
                ELP_LAUNCH(k_ghost_list, ceil_div((int64_t)sy, 256), 256, 0, st, (uint32_t)sy, used_y.p + (size_t)r * sy, pos.p, ylist.p);
            }
            if (m > 0) ELP_LAUNCH(k_tile_base, ceil_div(plan_r.ntiles + 1, 256), 256, 0, st, plan_r.ntiles, plan_r.rw(), rank * mb, m, pos.p, r, yroute.p);
            ELP_CUDA(cudaStreamSynchronize(st));
        }
        gx = (int)gxs[rank]; gy = (int)gys[rank];
        // ---- 3. masks of what I produce -----------------------------------------------------------------------------
        DevBuf<unsigned long long> sent(2);
        sent.zero(st);
        if (nl > 0) ELP_LAUNCH(k_ghost_mask, grid1(nl), 256, 0, st, nl, n0, sx, N, used_x.p, xmask.p, sent.p);
        if (m > 0) ELP_LAUNCH(k_ghost_mask, grid1(m), 256, 0, st, m, rank * mb, sy, N, used_y.p, ymask.p, sent.p + 1);
        ELP_REQUIRE(plan_c.rw() <= 32 && plan_r.rw() <= 32, "pdlp: routing records hold 32 rows per tile");
        if (nl > 0) ELP_LAUNCH(k_route_masks, grid1(nl), 256, 0, st, nl, plan_c.rw(), xmask.p, xroute.p);
        if (m > 0) ELP_LAUNCH(k_route_masks, grid1(m), 256, 0, st, m, plan_r.rw(), ymask.p, yroute.p);
        unsigned long long h[2] = {0, 0};
        ELP_CUDA(cudaMemcpyAsync(h, sent.p, sizeof h, cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        exch_frac_x = nl > 0 ? (double)h[0] / ((double)nl * N) : 1.0;
        exch_frac_y = m > 0 ? (double)h[1] / ((double)m * N) : 1.0;
        // ---- 4. my ghost memory, mapped by everybody -------------------------------------------------------------------
        auto padded = [](uint32_t g) { return (uint32_t)((g + SPMV_VPAD + 31) & ~31u); };
        auto bytes_of = [&](int r) { return GH_FLAGS_BYTES + (size_t)8 * ((size_t)padded(gxs[r]) + padded(gys[r])); };
        {
            ArenaScope own(nullptr);                                // mapped by the peers: its own allocation
            ghost_mem.alloc(bytes_of(rank));
        }
        ghost_mem.zero(st);
        ELP_CUDA(cudaStreamSynchronize(st));
        struct PeerInfo { cudaIpcMemHandle_t h; unsigned long long ptr; long long pid; long long dev; };
        static_assert(sizeof(PeerInfo) % 8 == 0, "peer record must be a multiple of 8 bytes");
        std::vector<PeerInfo> all(N);
        int ok = 1, dev = 0;
        ELP_CUDA(cudaGetDevice(&dev));
        memset(&all[rank], 0, sizeof(PeerInfo));
        all[rank].ptr = (unsigned long long)(uintptr_t)ghost_mem.p;
        all[rank].pid = (long long)getpid();
        all[rank].dev = dev;
        if (cudaIpcGetMemHandle(&all[rank].h, ghost_mem.p) != cudaSuccess) memset(&all[rank].h, 0, sizeof all[rank].h);
        cudaGetLastError();
        DevBuf<unsigned char> hbuf((size_t)N * sizeof(PeerInfo));
        ELP_CUDA(cudaMemcpyAsync(hbuf.p + (size_t)rank * sizeof(PeerInfo), &all[rank], sizeof(PeerInfo), cudaMemcpyHostToDevice, st));
        comm_allgather_bytes(hbuf.p, sizeof(PeerInfo), st);
        ELP_CUDA(cudaMemcpyAsync(all.data(), hbuf.p, (size_t)N * sizeof(PeerInfo), cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        std::vector<unsigned char*> base(N, nullptr);
        for (int r = 0; r < N && ok; ++r) {
            if (r == rank) { base[r] = ghost_mem.p; continue; }
            if (all[r].pid == all[rank].pid) {                 // a thread of this process drives that GPU: plain peer access
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, dev, (int)all[r].dev) != cudaSuccess || !can) { ok = 0; break; }
                const cudaError_t e = cudaDeviceEnablePeerAccess((int)all[r].dev, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { ok = 0; break; }
                base[r] = (unsigned char*)(uintptr_t)all[r].ptr;
            } else {
                void* q = nullptr;
                if (cudaIpcOpenMemHandle(&q, all[r].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; break; }
                ipc_opened.push_back(q);
                base[r] = (unsigned char*)q;
            }
        }
        cudaGetLastError();
        double okd = (double)ok;                                 // everyone or no one
        ELP_CUDA(cudaMemcpyAsync(scal.p, &okd, sizeof okd, cudaMemcpyHostToDevice, st));
        comm_allreduce_sum(scal.p, 1, st);
        ELP_CUDA(cudaMemcpyAsync(&okd, scal.p, sizeof okd, cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        if ((int)okd != N) {
            if (opt.verbose > 0 && rank == 0) fprintf(stderr, "[pdlp] no peer access between the GPUs: NCCL all-gather exchange\n");
            return;
        }
        const int gdbg = env_int("ELP_GHOST_DEBUG", 0);
        xout = GhostOut{}; yout = GhostOut{};
        xin = GhostIn{}; yin = GhostIn{};
        xout.n = yout.n = xin.n = yin.n = N;
        xout.rank = yout.rank = xin.rank = yin.rank = rank;
        xin.dbg = yin.dbg = gdbg;
        xout.route = dense ? nullptr : xroute.p; yout.route = dense ? nullptr : yroute.p;     // dense: no routing records at all
        xout.dense = yout.dense = dense ? 1 : 0;
        xout.first = n0; yout.first = rank * mb;
        xout.self_only = env_int("ELP_GHOST_LOCAL_ONLY", 0) & 1; yout.self_only = (env_int("ELP_GHOST_LOCAL_ONLY", 0) >> 1) & 1;
        for (int r = 0; r < N; ++r) {
            double* g0 = reinterpret_cast<double*>(base[r] + GH_FLAGS_BYTES);
            // ONE buffer per vector (stride 0).  The hand-off in the consumer's prologue already orders a producer's stores
            // behind the last reader: rank A stores x-bar(i+1) into B only after it has seen B's flag y(i), which B raises
            // at the start of its K1(i+1), i.e. after its K2(i) — the last reader of x-bar(i) — has completed; likewise for
            // y.  A second, alternating buffer (first version) doubled the L2 footprint of the gathered vectors and made
            // the stale copy a dead write-back every iteration.
            xout.buf[r] = g0;
            yout.buf[r] = g0 + (size_t)padded(gxs[r]);
            xin.peer_flag[r] = reinterpret_cast<unsigned long long*>(base[r]);
            yin.peer_flag[r] = reinterpret_cast<unsigned long long*>(base[r] + 64);
        }
        unsigned int* err = reinterpret_cast<unsigned int*>(ghost_mem.p + 128);
        xin.vec = xout.buf[rank]; xin.flags = xin.peer_flag[rank]; xin.err = err; xin.kind = 1; xin.len = (unsigned)gx;
        xin.go = reinterpret_cast<unsigned long long*>(ghost_mem.p + 256);
        yin.vec = yout.buf[rank]; yin.flags = yin.peer_flag[rank]; yin.err = err; yin.kind = 0; yin.len = (unsigned)gy;
        yin.go = reinterpret_cast<unsigned long long*>(ghost_mem.p + 384);
        if (gdbg & 64) {
            ArenaScope own(nullptr);
            ghost_trace.alloc(4096 * 4);
            ghost_trace.zero(st);
            xin.trace = yin.trace = ghost_trace.p;
        }

        // ---- 5. push mode: remote destinations become local outboxes, pusher CTAs move them (ghost_push_role) ----------
        // Pays when a rank sends several copies' worth of its block: config 4 at N = 8 (55 % kept, 3.9 copies) 106 -> 90 us
        // per iteration; config 5 at N = 8 (23 %, 1.6 copies) 67 -> 75 us and everything at N = 2 (stores are free there,
        // the pushers' SM slots are not) lose.  `kept` is the all-reduced fraction, so every rank decides alike.
        push = !dense && env_int("ELP_GHOST_PUSH", kept_all * (N - 1) >= 3.0 ? 1 : 0) != 0;
        if (push) {
            const int SEG = std::max(1, env_int("ELP_GHOST_PUSH_SEG", 32));          // tiles per segment
            std::vector<uint32_t> rec0(2 * SPMV_ROUTE_WORDS), rec1(2 * SPMV_ROUTE_WORDS);   // first / closing records of x and y
            ELP_CUDA(cudaMemcpyAsync(rec0.data(), xroute.p, SPMV_ROUTE_WORDS * 4, cudaMemcpyDeviceToHost, st));
            ELP_CUDA(cudaMemcpyAsync(rec1.data(), xroute.p + (size_t)plan_c.ntiles * SPMV_ROUTE_WORDS, SPMV_ROUTE_WORDS * 4, cudaMemcpyDeviceToHost, st));
            ELP_CUDA(cudaMemcpyAsync(rec0.data() + SPMV_ROUTE_WORDS, yroute.p, SPMV_ROUTE_WORDS * 4, cudaMemcpyDeviceToHost, st));
            ELP_CUDA(cudaMemcpyAsync(rec1.data() + SPMV_ROUTE_WORDS, yroute.p + (size_t)plan_r.ntiles * SPMV_ROUTE_WORDS, SPMV_ROUTE_WORDS * 4, cudaMemcpyDeviceToHost, st));
            ELP_CUDA(cudaStreamSynchronize(st));
            auto layout = [&](const uint32_t* a, const uint32_t* b, size_t* off) {      // outbox offsets with the 256-byte phase of the bases
                size_t at = 0;
                for (int r = 0; r < N; ++r) {
                    if (r == rank) { off[r] = 0; continue; }
                    at = ((at + 31) & ~(size_t)31) + (a[r] & 31u);     // a group of 32 is aligned on both sides of the copy
                    off[r] = at;
                    at += (size_t)(b[r] - a[r]);
                }
                return at + 32;
            };
            size_t offx[8] = {}, offy[8] = {};
            const size_t nx = nl > 0 ? layout(rec0.data(), rec1.data(), offx) : 32;
            const size_t ny = m > 0 ? layout(rec0.data() + SPMV_ROUTE_WORDS, rec1.data() + SPMV_ROUTE_WORDS, offy) : 32;
            const int nsx = ceil_div(std::max(plan_c.ntiles, 1), SEG), nsy = ceil_div(std::max(plan_r.ntiles, 1), SEG);
            {
                ArenaScope k(keep);
                xoutbox.alloc(nx); youtbox.alloc(ny);
            }
            // all bytes 0xFF is not the sentinel: fill with the pattern
            ELP_LAUNCH(k_fill_u64, ceil_div((int64_t)nx, 256), 256, 0, st, (size_t)nx, reinterpret_cast<unsigned long long*>(xoutbox.p), GHOST_SENTINEL);
            ELP_LAUNCH(k_fill_u64, ceil_div((int64_t)ny, 256), 256, 0, st, (size_t)ny, reinterpret_cast<unsigned long long*>(youtbox.p), GHOST_SENTINEL);
            const int pctas = std::max(1, env_int("ELP_GHOST_PUSH_CTAS", kNumSMs));
            for (int r = 0; r < N; ++r) {
                xout.remote[r] = xout.buf[r]; yout.remote[r] = yout.buf[r];
                if (r == rank) continue;
                // the epilogues index an outbox like the destination's ghost vector: shift it by the block's first position
                xout.buf[r] = xoutbox.p + offx[r] - rec0[r];
                yout.buf[r] = youtbox.p + offy[r] - rec0[SPMV_ROUTE_WORDS + r];
            }
            xout.seg_tiles = yout.seg_tiles = SEG;
            xout.nseg = nsx; yout.nseg = nsy;
            xout.ntiles = plan_c.ntiles; yout.ntiles = plan_r.ntiles;
            xout.push_ctas = nl > 0 ? pctas : 0; yout.push_ctas = m > 0 ? pctas : 0;
            xout.err = yout.err = xin.err;
            ELP_CUDA(cudaStreamSynchronize(st));
        }

        ghost = true;
        if (opt.verbose > 0 || env_int("ELP_PDLP_DEBUG", 0))
            fprintf(stderr, "[pdlp] rank %d ghost exchange: gathers %d of %d x-bar entries and %d of %d y entries; sends %.1f %% / %.1f %% of a dense all-gather (%s)\n",
                    rank, gx, n, gy, N * mb, 100.0 * exch_frac_x, 100.0 * exch_frac_y,
                    ipc_opened.empty() ? "peer access" : "CUDA IPC");
    }
    // y changed outside the plain iterations (reset, restart, Halpern finish): every rank gets the new blocks through
    // one all-gather and rebuilds the ghost buffer the next plain iteration reads (parity of epoch_base)
    void refresh_y() {
        gather_y(y_full.p);
        if (ghost && gy > 0)
            ELP_LAUNCH(k_compact, grid1(gy), 256, 0, st, gy, ylist.p, y_full.p, const_cast<double*>(yin.vec));
    }
    void check_device_error() {          // a consumer gave up waiting for a peer: report, do not hang or trap
        if (!ghost) return;
        unsigned int e = 0;
        ELP_CUDA(cudaMemcpyAsync(&e, ghost_mem.p + 128, sizeof e, cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        ELP_REQUIRE(e == 0, "pdlp: rank %d timed out waiting for a peer GPU's block (exchange flag never arrived)", rank);
    }
    void barrier_stream() {              // all ranks have finished everything they queued before this point
        if (N > 1) comm_allreduce_sum(scal.p + NACC, 1, st);
    }

    int grid1(int count) const { return std::max(1, ceil_div(count, 256)); }
    double* xbar() { return xbar_full.p + n0; }              // my block of the gathered x-bar
    double* y() { return y_full.p + (size_t)rank * mb; }     // my block of the gathered y
    void gather_x(double* full) { if (N > 1) comm_allgather(full, (size_t)nb, st); }
    void gather_y(double* full) { if (N > 1) comm_allgather(full, (size_t)mb, st); }

    void reduce_to(double* out_dev) {
        ELP_LAUNCH(k_final_reduce, 1, RED_THREADS, 0, st, partials.p, RED_BLOCKS, out_dev);
    }
    // sum over all ranks of a k_* reduction that was just launched into `partials`; returns NACC values
    void fetch_scalars(double* host) {
        reduce_to(scal.p);
        if (N > 1) comm_allreduce_sum(scal.p, NACC, st);
        ELP_CUDA(cudaMemcpyAsync(host, scal.p, NACC * sizeof(double), cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        d2h += NACC * sizeof(double);
    }

    // out[m] = A_rows * v_full      (my rows; v_full in the flat column layout)
    void spmv_rows(const double* v_full, double* out) {
        launch_spmv(plan_r, m, csr_ptr.p, csr_idx.p, csr_val.p, v_full, store_epi(out), st);
    }
    // out[nl] = (A' * v_full)_mycols  (v_full in the padded row layout)
    void spmv_cols(const double* v_full, double* out) {
        launch_spmv(plan_c, nl, csc_ptr.p, csc_idx.p, csc_val.p, v_full, store_epi(out), st);
    }

    template <int MODE>
    void rowstat(int L, int nrows, const int* ptr, const int* idx, const double* val, const double* s_self,
                 const double* s_other, double* out) {
        if (nrows <= 0) return;
        const int grid = ceil_div((int64_t)nrows * L, SPMV_THREADS);
        switch (L) {
            case 1:  ELP_LAUNCH((rowstat_kernel<1, MODE>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other, out); break;
            case 2:  ELP_LAUNCH((rowstat_kernel<2, MODE>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other, out); break;
            case 4:  ELP_LAUNCH((rowstat_kernel<4, MODE>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other, out); break;
            case 8:  ELP_LAUNCH((rowstat_kernel<8, MODE>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other, out); break;
            case 16: ELP_LAUNCH((rowstat_kernel<16, MODE>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other, out); break;
            default: ELP_LAUNCH((rowstat_kernel<32, MODE>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other, out); break;
        }
    }
    void scale_vals(int L, int nrows, const int* ptr, const int* idx, double* val, const double* s_self,
                    const double* s_other) {
        if (nrows <= 0) return;
        const int grid = ceil_div((int64_t)nrows * L, SPMV_THREADS);
        switch (L) {
            case 1:  ELP_LAUNCH((scale_vals_kernel<1>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other); break;
            case 2:  ELP_LAUNCH((scale_vals_kernel<2>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other); break;
            case 4:  ELP_LAUNCH((scale_vals_kernel<4>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other); break;
            case 8:  ELP_LAUNCH((scale_vals_kernel<8>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other); break;
            case 16: ELP_LAUNCH((scale_vals_kernel<16>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other); break;
            default: ELP_LAUNCH((scale_vals_kernel<32>), grid, SPMV_THREADS, 0, st, nrows, ptr, idx, val, s_self, s_other); break;
        }
    }
    void expand_rows(int L, int nrows, const int* ptr, int* row_of) {
        if (nrows <= 0) return;
        const int grid = ceil_div((int64_t)nrows * L, SPMV_THREADS);
        switch (L) {
            case 1:  ELP_LAUNCH((expand_rows_kernel<1>), grid, SPMV_THREADS, 0, st, nrows, ptr, row_of); break;
            case 2:  ELP_LAUNCH((expand_rows_kernel<2>), grid, SPMV_THREADS, 0, st, nrows, ptr, row_of); break;
            case 4:  ELP_LAUNCH((expand_rows_kernel<4>), grid, SPMV_THREADS, 0, st, nrows, ptr, row_of); break;
            case 8:  ELP_LAUNCH((expand_rows_kernel<8>), grid, SPMV_THREADS, 0, st, nrows, ptr, row_of); break;
            case 16: ELP_LAUNCH((expand_rows_kernel<16>), grid, SPMV_THREADS, 0, st, nrows, ptr, row_of); break;
            default: ELP_LAUNCH((expand_rows_kernel<32>), grid, SPMV_THREADS, 0, st, nrows, ptr, row_of); break;
        }
    }

    // ---- setup ---------------------------------------------------------------------------------
    void setup(int m_, int n_, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
               const int8_t* sense, const double* rhs, const double* c_h, int maximize_, const double* lb,
               const double* ub, const elp_options& o, bool dist_, int64_t nnz_device = -1) {
        // nnz_device >= 0: row_ptr / col_idx / vals are DEVICE arrays (a model assembled by elp_model_assemble)
        m = m_; n = n_; maximize = maximize_ != 0; opt = o;
        WallTimer dbg_t;
        const bool dbg = getenv("ELP_PDLP_DEBUG") != nullptr;
        auto mark = [&](const char* what) {
            if (!dbg) return;
            cudaStreamSynchronize(st);
            fprintf(stderr, "[pdlp setup] %-16s %9.3f ms\n", what, dbg_t.ms());
        };
        const bool dist = dist_ && comm().active;
        N = dist ? comm().nranks : 1;
        rank = dist ? comm().rank : 0;
        ELP_REQUIRE(m >= 0 && n > 0, "pdlp: bad shape %d x %d", m, n);
        nnz = nnz_device >= 0 ? nnz_device : (m > 0 ? row_ptr[m] : 0);
        ELP_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        if (N == 1 && env_int("ELP_PDLP_ARENA", 1)) {
            arena.reserve((size_t)24 * nnz + (size_t)4 * (m + n) + (size_t)8 * ((size_t)10 * n + (size_t)9 * m) + (2u << 20));
            scratch.reserve((size_t)52 * nnz + (size_t)16 * ((size_t)n + m) + (8u << 20));
        } else if (N > 1 && env_int("ELP_PDLP_ARENA", 1)) {
            // Distributed: the same two arenas, sized from what this rank knows (its row block; the column block is
            // taken as 1.3 x as many entries — row blocks are balanced by non-zeros — and anything beyond falls back to
            // cudaMalloc).  Besides the milliseconds, this keeps cudaMalloc / cudaFree — which synchronise the device
            // and serialise on process-wide locks — out of the stretches between two collectives when the ranks are
            // threads of ONE process (elp_solve_lp(devices = N)): a rank stuck in cudaFree behind a collective whose
            // peer is stuck in cudaMalloc before launching its half would never return.  Only the ghost memory that
            // the peers map keeps its own allocation.
            const size_t nbg = (size_t)((ceil_div(n, N) + 3) & ~3), sxg = (size_t)N * nbg;
            const size_t mbg = (size_t)m + m / 8 + 64, syg = (size_t)N * mbg;          // padded rows per rank: a guess
            const size_t nnzc_g = (size_t)(1.3 * (double)nnz) + (1u << 20);
            arena.reserve((size_t)16 * nnz + (size_t)16 * nnzc_g + (size_t)8 * (10 * nbg + 10 * (size_t)m) + (size_t)16 * (sxg + syg) +
                          (size_t)3 * (nbg + m) + (size_t)4 * syg + (4u << 20));
            scratch.reserve((size_t)52 * nnz + (size_t)12 * nnzc_g + (size_t)16 * ((size_t)n + m) + (size_t)N * (sxg + syg) +
                            (size_t)8 * std::max(sxg, syg) + (size_t)16 * sxg + (16u << 20));
        }
        ArenaScope persistent(arena.base ? &arena : nullptr);
        partials.alloc((size_t)RED_BLOCKS * NACC); scal.alloc(2 * NACC); params.alloc(1);
        partials.zero(st);
        // block sizes: multiples of 4 keep every block 32-byte aligned (16-byte-granular bulk copies)
        nb = (ceil_div(n, N) + 3) & ~3;
        n0 = std::min(n, rank * nb);
        nl = std::max(0, std::min(n, (rank + 1) * nb) - n0);
        {
            double mx = (double)m;
            if (N > 1) {
                ELP_CUDA(cudaMemcpyAsync(scal.p, &mx, sizeof mx, cudaMemcpyHostToDevice, st));
                comm_allreduce_max(scal.p, 1, st);
                ELP_CUDA(cudaMemcpyAsync(&mx, scal.p, sizeof mx, cudaMemcpyDeviceToHost, st));
                ELP_CUDA(cudaStreamSynchronize(st));
            }
            mb = (std::max(1, (int)mx) + 3) & ~3;
        }
        ELP_REQUIRE((int64_t)N * mb < 0x7fffffffll && (int64_t)N * nb < 0x7fffffffll, "pdlp: problem too large for int32 ids");

        csr_ptr.alloc(m + 1 + SPMV_PTR_PAD); csr_idx.alloc(nnz + SPMV_PAD); csr_val.alloc(nnz + SPMV_PAD);
        csr_idx.zero(st); csr_val.zero(st); csr_ptr.zero(st);
        // epilogue operands are staged by 16-byte-granular bulk copies: SPMV_VPAD doubles of slack each
        const size_t np = (size_t)std::max(nl, 1) + SPMV_VPAD, mp = (size_t)std::max(m, 1) + SPMV_VPAD;
        c.alloc(np); l.alloc(np); u.alloc(np); dc.alloc(np); x.alloc(np); x0.alloc(np); xp.alloc(np); gcol.alloc(np);
        lc.alloc(mp); uc.alloc(mp); dr.alloc(mp); y0.alloc(mp); yp.alloc(mp); axbar.alloc(mp); axp.alloc(mp); rs.alloc(mp);
        rsense.alloc((size_t)((std::max(m, 1) + 15) & ~15));
        rsense.zero(st);
        xbar_full.alloc((size_t)N * nb + SPMV_VPAD); xaux_full.alloc((size_t)N * nb + SPMV_VPAD);
        y_full.alloc((size_t)N * mb + SPMV_VPAD); yaux_full.alloc((size_t)N * mb + SPMV_VPAD);
        for (DevBuf<double>* b : {&c, &l, &u, &dc, &x, &x0, &xp, &gcol, &lc, &uc, &dr, &y0, &yp, &axbar, &axp, &rs, &xbar_full,
                                  &xaux_full, &y_full, &yaux_full})
            b->zero(st);

        if (nnz_device >= 0) {
            ELP_CUDA(cudaStreamSynchronize(0));           // the assembly ran on the default stream
            ELP_CUDA(cudaMemcpyAsync(csr_ptr.p, row_ptr, ((size_t)m + 1) * sizeof(int), cudaMemcpyDeviceToDevice, st));
            if (nnz) {
                ELP_CUDA(cudaMemcpyAsync(csr_idx.p, col_idx, (size_t)nnz * sizeof(int), cudaMemcpyDeviceToDevice, st));
                ELP_CUDA(cudaMemcpyAsync(csr_val.p, vals, (size_t)nnz * sizeof(double), cudaMemcpyDeviceToDevice, st));
            }
        } else {
            if (m == 0) { int z = 0; csr_ptr.upload(&z, 1, st); }
            else csr_ptr.upload(row_ptr, m + 1, st);
            csr_idx.upload(col_idx, nnz, st);
            csr_val.upload(vals, nnz, st);
            h2d += (int64_t)(m + 1) * 4 + nnz * 12;
        }
        c.upload(c_h + n0, nl, st); l.upload(lb + n0, nl, st); u.upload(ub + n0, nl, st);
        h2d += (int64_t)nl * 24;
        rsense.upload(sense, m, st); rs.upload(rhs, m, st);
        h2d += (int64_t)m * 9;
        if (m > 0) ELP_LAUNCH(k_row_bounds, grid1(m), 256, 0, st, m, rsense.p, rs.p, lc.p, uc.p);
        if (maximize && nl > 0) ELP_LAUNCH(k_scale_scalar, grid1(nl), 256, 0, st, nl, c.p, -1.0);

        mark("upload");
        build_column_block();
        mark("column block");
        Lr = pick_helper_lanes(nnz, m);
        Lc = pick_helper_lanes(nnzc, nl);
        plan_r = plan_spmv(nnz, m, 4);
        plan_c = plan_spmv(nnzc, nl, 5);
        {
            int mode = opt.transpose;
            if (const int e = env_int("ELP_PDLP_TRANSPOSE", 0)) mode = e;      // sweeps / A-B runs
            ELP_REQUIRE(mode >= ELP_TRANSPOSE_AUTO && mode <= ELP_TRANSPOSE_SCATTER, "pdlp: bad transpose mode %d", mode);
            ELP_REQUIRE(!(mode == ELP_TRANSPOSE_SCATTER && N > 1), "pdlp: the scatter formulation is single-GPU only");
            scatter = N == 1 && mode == ELP_TRANSPOSE_SCATTER && m > 0;
            if (const char* e = getenv("ELP_PDLP_BETA_ART")) beta_artificial = atof(e);       // experiments
            if (const char* e = getenv("ELP_PDLP_KP")) w_kp = atof(e);
            if (const char* e = getenv("ELP_PDLP_KI")) w_ki = atof(e);
            if (const char* e = getenv("ELP_PDLP_KD")) w_kd = atof(e);
            if (const char* e = getenv("ELP_PDLP_ISMOOTH")) w_ismooth = atof(e);
            if (const char* e = getenv("ELP_PDLP_GAP_RULE")) gap_rule = atoi(e);
            if (const char* e = getenv("ELP_PDLP_GAP_FACTOR")) gap_factor = atof(e);
            plan_s = plan_spmv(nnz, m, 4, 0, env_int("ELP_SPMV_SCAT_STAGES", 2));
        }

        // unscaled norms for the relative termination test
        double h[NACC];
        ELP_LAUNCH(k_bound_norm, RED_BLOCKS, RED_THREADS, 0, st, m, lc.p, uc.p, partials.p);
        fetch_scalars(h);
        norm_b = std::sqrt(h[0]);
        ELP_LAUNCH(k_dot2, RED_BLOCKS, RED_THREADS, 0, st, nl, c.p, c.p, partials.p);
        fetch_scalars(h);
        norm_c = std::sqrt(h[0]);

        mark("norms");
        scale_problem();
        mark("scaling");
        estimate_sigma_max();
        mark("power iteration");
        eta = sigma_max > 0 ? 0.998 / sigma_max : 1.0;
        // initial primal weight from the scaled data: ||c|| / ||b||
        ELP_LAUNCH(k_bound_norm, RED_BLOCKS, RED_THREADS, 0, st, m, lc.p, uc.p, partials.p);
        fetch_scalars(h);
        const double nbn = std::sqrt(h[0]);
        ELP_LAUNCH(k_dot2, RED_BLOCKS, RED_THREADS, 0, st, nl, c.p, c.p, partials.p);
        fetch_scalars(h);
        const double ncn = std::sqrt(h[0]);
        w_init = (nbn > 1e-10 && ncn > 1e-10) ? ncn / nbn : 1.0;
        choose_streams();
        setup_ghost_exchange();
        reset();
        mark("reset");
        ELP_CUDA(cudaStreamSynchronize(st));
        scratch.release();                           // the setup's temporaries, in one cudaFree
    }

    // CSC of my column block over all rows, row ids in the padded y_full layout.  Every rank transposes its own row
    // block with the stable radix sort that backs the assembly, then the column slices travel to their owners in
    // one grouped send/recv and are merged source by source (= ascending global row).
    void build_column_block() {
        ArenaScope tmp(scratch.base ? &scratch : g_arena);       // temporaries; the CSC arrays below go to the handle's arena
        // ---- local transpose: CSC of my row block over all n columns ----------------------------------
        DevBuf<int> lptr((size_t)n + 1), lidx(std::max<int64_t>(nnz, 1));
        DevBuf<double> lval(std::max<int64_t>(nnz, 1));
        if (nnz == 0) {
            lptr.zero(st);
        } else {
            DevBuf<uint64_t> keys(nnz);
            DevBuf<uint32_t> perm(nnz), nnz_d(1);
            DevBuf<int> row_of(nnz), cols_sorted(nnz);
            RadixSortWorkspace ws;
            expand_rows(pick_helper_lanes(nnz, m), m, csr_ptr.p, row_of.p);
            launch_transpose_keys(csr_idx.p, (uint32_t)nnz, keys.p, perm.p, st);
            radix_sort_pairs(keys.p, perm.p, nnz, bit_length_u64((uint64_t)n - 1), ws, st);
            launch_transpose_gather(keys.p, perm.p, row_of.p, csr_val.p, (uint32_t)nnz, lidx.p, lval.p, cols_sorted.p,
                                    nnz_d.p, st);
            launch_fill_ptr(cols_sorted.p, nnz_d.p, (uint32_t)n, lptr.p, (uint32_t)nnz, st);
            if (rank > 0) ELP_LAUNCH(k_shift_idx, ceil_div(nnz, 256), 256, 0, st, (uint32_t)nnz, lidx.p, rank * mb);
            ELP_CUDA(cudaStreamSynchronize(st));
        }
        if (N == 1) {
            nnzc = nnz;
            ArenaScope keep(arena.base ? &arena : nullptr);
            csc_ptr.alloc((size_t)nl + 1 + SPMV_PTR_PAD); csc_idx.alloc(nnzc + SPMV_PAD); csc_val.alloc(nnzc + SPMV_PAD);
            csc_ptr.zero(st); csc_idx.zero(st); csc_val.zero(st);
            ELP_CUDA(cudaMemcpyAsync(csc_ptr.p, lptr.p, ((size_t)n + 1) * sizeof(int), cudaMemcpyDeviceToDevice, st));
            if (nnz) {
                ELP_CUDA(cudaMemcpyAsync(csc_idx.p, lidx.p, (size_t)nnz * sizeof(int), cudaMemcpyDeviceToDevice, st));
                ELP_CUDA(cudaMemcpyAsync(csc_val.p, lval.p, (size_t)nnz * sizeof(double), cudaMemcpyDeviceToDevice, st));
            }
            ELP_CUDA(cudaStreamSynchronize(st));
            return;
        }
        // ---- how much goes where ----------------------------------------------------------------------
        std::vector<int> cut(N + 1);
        for (int g = 0; g <= N; ++g) {
            const int col = std::min(n, g * nb);
            ELP_CUDA(cudaMemcpyAsync(&cut[g], lptr.p + col, sizeof(int), cudaMemcpyDeviceToHost, st));
        }
        ELP_CUDA(cudaStreamSynchronize(st));
        DevBuf<double> cnt_d((size_t)N * N);
        std::vector<double> cnt((size_t)N * N, 0.0);
        for (int g = 0; g < N; ++g) cnt[(size_t)rank * N + g] = (double)(cut[g + 1] - cut[g]);
        ELP_CUDA(cudaMemcpyAsync(cnt_d.p + (size_t)rank * N, cnt.data() + (size_t)rank * N, N * sizeof(double),
                                 cudaMemcpyHostToDevice, st));
        comm_allgather(cnt_d.p, (size_t)N, st);
        ELP_CUDA(cudaMemcpyAsync(cnt.data(), cnt_d.p, (size_t)N * N * sizeof(double), cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        std::vector<uint32_t> roff(N + 1, 0);
        for (int r = 0; r < N; ++r) roff[r + 1] = roff[r] + (uint32_t)cnt[(size_t)r * N + rank];   // what r sends me
        const int64_t total_in = roff[N];
        // ---- lens of every column slice I send, then the grouped exchange -------------------------------
        DevBuf<uint32_t> lens_out((size_t)N * nb), lens_in((size_t)N * nb + 1), srcptr((size_t)N * nb), newptr((size_t)nb + 1);
        DevBuf<uint32_t> roff_d(N + 1);
        DevBuf<int> in_idx(std::max<int64_t>(total_in, 1));
        DevBuf<double> in_val(std::max<int64_t>(total_in, 1));
        for (int g = 0; g < N; ++g)
            ELP_LAUNCH(k_col_lens, ceil_div(nb, 256), 256, 0, st, lptr.p, g * nb, nb, n, lens_out.p + (size_t)g * nb);
        comm_group_start();
        for (int g = 0; g < N; ++g) {
            const size_t cntg = (size_t)(cut[g + 1] - cut[g]);
            comm_send(lens_out.p + (size_t)g * nb, (size_t)nb * sizeof(uint32_t), g, st);
            comm_send(lidx.p + cut[g], cntg * sizeof(int), g, st);
            comm_send(lval.p + cut[g], cntg * sizeof(double), g, st);
            const size_t cin = (size_t)(roff[g + 1] - roff[g]);
            comm_recv(lens_in.p + (size_t)g * nb, (size_t)nb * sizeof(uint32_t), g, st);
            comm_recv(in_idx.p + roff[g], cin * sizeof(int), g, st);
            comm_recv(in_val.p + roff[g], cin * sizeof(double), g, st);
        }
        comm_group_end();
        // ---- merge ---------------------------------------------------------------------------------------
        ScanWorkspace sw;
        ELP_LAUNCH(k_sum_lens, ceil_div(nb + 1, 256), 256, 0, st, N, nb, lens_in.p, newptr.p);
        exclusive_scan_u32(newptr.p, (size_t)nb + 1, sw, st);
        ELP_CUDA(cudaMemcpyAsync(srcptr.p, lens_in.p, (size_t)N * nb * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
        for (int r = 0; r < N; ++r) exclusive_scan_u32(srcptr.p + (size_t)r * nb, (size_t)nb, sw, st);
        roff_d.upload(roff.data(), N + 1, st);
        nnzc = total_in;
        ArenaScope keep(arena.base ? &arena : nullptr);
        csc_ptr.alloc((size_t)nb + 1 + SPMV_PTR_PAD); csc_idx.alloc(nnzc + SPMV_PAD); csc_val.alloc(nnzc + SPMV_PAD);
        csc_ptr.zero(st); csc_idx.zero(st); csc_val.zero(st);
        ELP_LAUNCH(k_merge_cols, ceil_div(nb + 1, 256), 256, 0, st, N, nb, lens_in.p, srcptr.p, newptr.p, roff_d.p,
                   in_idx.p, in_val.p, csc_ptr.p, csc_idx.p, csc_val.p);
        ELP_CUDA(cudaStreamSynchronize(st));
    }

    void scale_problem() {
        ArenaScope tmp(scratch.base ? &scratch : g_arena);
        const int ruiz = opt.ruiz_iters >= 0 ? opt.ruiz_iters : 10;
        // dr_full = yaux_full (padded row layout), dc_full = xaux_full (flat column layout) during scaling
        double* dr_full = yaux_full.p;
        double* dc_full = xaux_full.p;
        double* drl = dr_full + (size_t)rank * mb;
        double* dcl = dc_full + n0;
        ELP_LAUNCH(k_fill, grid1(N * mb), 256, 0, st, N * mb, dr_full, 1.0);
        ELP_LAUNCH(k_fill, grid1(N * nb), 256, 0, st, N * nb, dc_full, 1.0);
        DevBuf<double> rstat(std::max(m, 1)), cstat(std::max(nl, 1));
        for (int it = 0; it < ruiz + 1; ++it) {
            const bool pc = it == ruiz;   // last pass: Pock-Chambolle (alpha = 1) with L1 norms
            if (!pc) {
                rowstat<0>(Lr, m, csr_ptr.p, csr_idx.p, csr_val.p, drl, dc_full, rstat.p);
                rowstat<0>(Lc, nl, csc_ptr.p, csc_idx.p, csc_val.p, dcl, dr_full, cstat.p);
            } else {
                rowstat<1>(Lr, m, csr_ptr.p, csr_idx.p, csr_val.p, drl, dc_full, rstat.p);
                rowstat<1>(Lc, nl, csc_ptr.p, csc_idx.p, csc_val.p, dcl, dr_full, cstat.p);
            }
            if (m > 0) ELP_LAUNCH(k_ruiz_update, grid1(m), 256, 0, st, m, drl, rstat.p);
            if (nl > 0) ELP_LAUNCH(k_ruiz_update, grid1(nl), 256, 0, st, nl, dcl, cstat.p);
            gather_y(dr_full);
            gather_x(dc_full);
        }
        scale_vals(Lr, m, csr_ptr.p, csr_idx.p, csr_val.p, drl, dc_full);
        scale_vals(Lc, nl, csc_ptr.p, csc_idx.p, csc_val.p, dcl, dr_full);
        if (m > 0) ELP_CUDA(cudaMemcpyAsync(dr.p, drl, (size_t)m * sizeof(double), cudaMemcpyDeviceToDevice, st));
        if (nl > 0) ELP_CUDA(cudaMemcpyAsync(dc.p, dcl, (size_t)nl * sizeof(double), cudaMemcpyDeviceToDevice, st));
        if (nl > 0) {
            ELP_LAUNCH(k_mul, grid1(nl), 256, 0, st, nl, c.p, dc.p);
            ELP_LAUNCH(k_div, grid1(nl), 256, 0, st, nl, l.p, dc.p);
            ELP_LAUNCH(k_div, grid1(nl), 256, 0, st, nl, u.p, dc.p);
        }
        if (m > 0) {
            ELP_LAUNCH(k_mul, grid1(m), 256, 0, st, m, lc.p, dr.p);
            ELP_LAUNCH(k_mul, grid1(m), 256, 0, st, m, uc.p, dr.p);
            ELP_LAUNCH(k_mul, grid1(m), 256, 0, st, m, rs.p, dr.p);
        }
    }

    // Single GPU: which operand streams of the plain iterations the scaled problem can do without (pbnd, drhs)
    void choose_streams() {
        pbnd = 0; drhs = false;
        if (N > 1) return;
        unsigned int hf = 0;
        {
            ArenaScope tmp(scratch.base ? &scratch : nullptr);
            DevBuf<unsigned int> f(1);
            f.zero(st);
            const int span = std::max(nl, m);
            if (span > 0) ELP_LAUNCH(k_bound_kinds, grid1(span), 256, 0, st, nl, l.p, u.p, m, rsense.p, rs.p, lc.p, uc.p, f.p);
            f.download(&hf, 1, st);
            ELP_CUDA(cudaStreamSynchronize(st));
        }
        pbnd = ((hf & 1u) ? 0 : BND_L0) | ((hf & 2u) ? 0 : BND_UINF);
        drhs = !(hf & 4u) && (plan_r.rowwarp || plan_r.L <= 2);     // a sense byte per row needs tiles of >= 16 rows
        if (opt.verbose > 0 || env_int("ELP_PDLP_DEBUG", 0))
            fprintf(stderr, "[pdlp] plain iterations stream %s%s and %s\n", (pbnd & BND_L0) ? "" : "l ",
                    (pbnd & BND_UINF) ? "" : "u", drhs ? "rhs + sense" : "lc + uc");
    }

    void estimate_sigma_max() {
        sigma_max = 0.0;
        double h[NACC];
        // has the matrix any entry at all?
        double tot = (double)nnz;
        if (N > 1) {
            ELP_CUDA(cudaMemcpyAsync(scal.p, &tot, sizeof tot, cudaMemcpyHostToDevice, st));
            comm_allreduce_sum(scal.p, 1, st);
            ELP_CUDA(cudaMemcpyAsync(&tot, scal.p, sizeof tot, cudaMemcpyDeviceToHost, st));
            ELP_CUDA(cudaStreamSynchronize(st));
        }
        if (tot == 0.0) return;
        // power iteration on A'A: v in xaux_full (my block at n0), A v in yaux_full (my block), A'(A v) in gcol
        double* v = xaux_full.p + n0;
        double* av = yaux_full.p + (size_t)rank * mb;
        ELP_CUDA(cudaMemsetAsync(xaux_full.p, 0, (size_t)N * nb * sizeof(double), st));
        ELP_CUDA(cudaMemsetAsync(yaux_full.p, 0, (size_t)N * mb * sizeof(double), st));
        if (nl > 0) ELP_LAUNCH(k_pseudo_random, grid1(nl), 256, 0, st, nl, v, 12345u + 7919u * (uint32_t)n0);
        ELP_LAUNCH(k_dot2, RED_BLOCKS, RED_THREADS, 0, st, nl, v, v, partials.p);
        fetch_scalars(h);
        if (nl > 0) ELP_LAUNCH(k_scale_scalar, grid1(nl), 256, 0, st, nl, v, 1.0 / std::sqrt(h[0]));
        double s = 1.0;
        for (int it = 0; it < 60; ++it) {
            gather_x(xaux_full.p);
            spmv_rows(xaux_full.p, av);
            gather_y(yaux_full.p);
            spmv_cols(yaux_full.p, gcol.p);
            ELP_LAUNCH(k_dot2, RED_BLOCKS, RED_THREADS, 0, st, nl, gcol.p, gcol.p, partials.p);
            fetch_scalars(h);
            const double nrm = std::sqrt(h[0]);
            if (!(nrm > 0.0)) { s = 0.0; break; }
            const double s_new = std::sqrt(nrm);
            if (nl > 0) {
                ELP_CUDA(cudaMemcpyAsync(v, gcol.p, (size_t)nl * sizeof(double), cudaMemcpyDeviceToDevice, st));
                ELP_LAUNCH(k_scale_scalar, grid1(nl), 256, 0, st, nl, v, 1.0 / nrm);
            }
            const bool conv = std::fabs(s_new - s) <= 1e-4 * s_new;
            s = s_new;
            if (conv && it >= 10) break;
        }
        sigma_max = s;
    }

    void reset() {
        if (nl > 0) ELP_LAUNCH(k_init_x, grid1(nl), 256, 0, st, nl, x.p, l.p, u.p);
        ELP_CUDA(cudaMemcpyAsync(x0.p, x.p, (size_t)std::max(nl, 1) * sizeof(double), cudaMemcpyDeviceToDevice, st));
        ELP_CUDA(cudaMemcpyAsync(xp.p, x.p, (size_t)std::max(nl, 1) * sizeof(double), cudaMemcpyDeviceToDevice, st));
        y_full.zero(st); y0.zero(st); yp.zero(st); axbar.zero(st); axp.zero(st); xbar_full.zero(st);
        gcol.zero(st);                             // = A'y for y = 0 (scatter formulation)
        w = w_init; k = 0; total = 0; restarts = 0; fpe0 = -1; fpe_prev = -1; need_fpe0 = true;
        w_err_sum = 0.0; w_err_prev = 0.0; obj_err = 0.0;
        status = ELP_STATUS_TIMEOUT; finished = false; checks = 0;
        clock_running = false; time_up = false; hit_time_limit = false;
        push_params();
        if (ghost) refresh_y();    // (its all-gather also keeps any rank from running ahead into a peer that is still resetting)
        else barrier_stream();
        ELP_CUDA(cudaStreamSynchronize(st));
    }

    void push_params() {
        PdlpParams p{eta / w, eta * w, k, 0, epoch_base};
        // pageable source is copied to a staging buffer before the call returns, so a stack object is fine
        ELP_CUDA(cudaMemcpyAsync(params.p, &p, sizeof p, cudaMemcpyHostToDevice, st));
    }

    // ---- iteration pieces ------------------------------------------------------------------------
    // multi-GPU, a rank without columns / rows still owes its consumers the epoch
    void signal_only(const GhostIn& gi, int plus) {
        ELP_LAUNCH(k_ghost_signal_only, 1, 32, 0, st, gi, params.p, plus);
    }
    template <int BND>
    void launch_primal_plain(int it, int from_x, int store_x) {
        PrimalEpi<false, false, BND> epi{nullptr, c.p, l.p, u.p, x0.p, x.p, xbar(), xp.p, params.p, it, GhostIn{}, GhostOut{},
                                         from_x, store_x};
        launch_spmv(plan_c, nl, csc_ptr.p, csc_idx.p, csc_val.p, y_full.p, epi, st);
    }
    // plain iterations: store_x on the last one before a check or the end of run() (see PrimalEpi), from_x when x-bar
    // does not belong to x
    template <bool CHECK>
    void primal_step(int it, bool store_x = true, bool from_x = false) {
        if (!CHECK && scatter) {            // g = A'y is already in gcol (left there by the dual kernel's scatter)
            const int grid = std::max(1, std::min(ceil_div(nl / 2, 256), kNumSMs * 8));
            ELP_LAUNCH(k_primal_from_g, grid, 256, 0, st, nl, gcol.p, c.p, l.p, u.p, x0.p, x.p, xbar(), params.p, it);
            return;
        }
        if (!CHECK && ghost) {              // gathers y from my ghost vector, publishes x-bar into the consumers' ghost vectors
            PrimalEpi<false, true> epi{nullptr, c.p, l.p, u.p, x0.p, x.p, xbar(), xp.p, params.p, it, yin, xout};
            if (nl > 0) launch_spmv(plan_c, nl, csc_ptr.p, xout.dense ? csc_idx.p : csc_idx_g.p, csc_val.p, yin.vec, epi, st);   // dense ghosts: identity numbering
            else signal_only(yin, it);            // what K1's prologue would have said: my y of the previous epoch is out
            return;
        }
        if constexpr (CHECK) {
            PrimalEpi<true> epi{nullptr, c.p, l.p, u.p, x0.p, x.p, xbar(), xp.p, params.p, it, GhostIn{}, GhostOut{}};
            launch_spmv(plan_c, nl, csc_ptr.p, csc_idx.p, csc_val.p, y_full.p, epi, st);
        } else {
            // N > 1 (all-gather exchange): x stays the stored iterate
            const int fx = N > 1 || from_x, sx = N > 1 || store_x;
            switch (pbnd) {
                case 0: launch_primal_plain<0>(it, fx, sx); break;
                case BND_L0: launch_primal_plain<BND_L0>(it, fx, sx); break;
                case BND_UINF: launch_primal_plain<BND_UINF>(it, fx, sx); break;
                default: launch_primal_plain<BND_L0 | BND_UINF>(it, fx, sx); break;
            }
        }
        gather_x(xbar_full.p);
    }
    template <bool CHECK>
    void dual_step(int it) {
        if (!CHECK && scatter) {            // A x-bar + dual update, then g += val * y_new over the row's entries
            DualEpi<false, true> epi{gcol.p, lc.p, uc.p, y0.p, y(), yp.p, axbar.p, params.p, it, GhostIn{}, GhostOut{}};
            launch_spmv(plan_s, m, csr_ptr.p, csr_idx.p, csr_val.p, xbar_full.p, epi, st);
            return;
        }
        if (!CHECK && ghost) {
            DualEpi<false, false, true> epi{nullptr, lc.p, uc.p, y0.p, y(), yp.p, axbar.p, params.p, it, xin, yout};
            if (m > 0) launch_spmv(plan_r, m, csr_ptr.p, yout.dense ? csr_idx.p : csr_idx_g.p, csr_val.p, xin.vec, epi, st);
            else signal_only(xin, it + 1);        // what K2's prologue would have said: my x-bar of this epoch is out
            return;
        }
        if (!CHECK && drhs) {
            DualEpi<false, false, false, true> epi{nullptr, lc.p, uc.p, y0.p, y(), yp.p, axbar.p, params.p, it, GhostIn{}, GhostOut{},
                                                   rs.p, rsense.p};
            launch_spmv(plan_r, m, csr_ptr.p, csr_idx.p, csr_val.p, xbar_full.p, epi, st);
        } else {
            DualEpi<CHECK> epi{nullptr, lc.p, uc.p, y0.p, y(), yp.p, axbar.p, params.p, it, GhostIn{}, GhostOut{}};
            launch_spmv(plan_r, m, csr_ptr.p, csr_idx.p, csr_val.p, xbar_full.p, epi, st);
        }
        if (!CHECK) gather_y(y_full.p);                      // a check iteration does not change y here
    }
    int kernels_per_iter() const { return ghost ? 2 : (m > 0 ? 1 : 0) + (nl > 0 ? 1 : 0); }

    void plain_iterations(int count) {
        if (count <= 0) return;
        const bool want_graph = opt.use_graph != 0 && count == opt.check_every - 1 && count > 1;
        if (want_graph) {
            if (!graph || graph_len != count) {
                if (graph) { cudaGraphExecDestroy(graph); graph = nullptr; }
                cudaGraph_t g = nullptr;
                const int64_t before = g_launches.load();
                ELP_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
                try {
                    for (int i = 0; i < count; ++i) { primal_step<false>(i, i == count - 1); dual_step<false>(i); }
                } catch (...) {
                    cudaStreamEndCapture(st, &g);
                    if (g) cudaGraphDestroy(g);
                    throw;
                }
                ELP_CUDA(cudaStreamEndCapture(st, &g));
                g_launches.store(before);   // capture does not execute; launches are counted per replay
                ELP_CUDA(cudaGraphInstantiate(&graph, g, 0));
                cudaGraphDestroy(g);
                graph_len = count;
            }
            ELP_CUDA(cudaGraphLaunch(graph, st));
            g_launches.fetch_add((int64_t)count * kernels_per_iter());
        } else {
            for (int i = 0; i < count; ++i) { primal_step<false>(i, i == count - 1); dual_step<false>(i); }
        }
        k += count;
        total += count;
        if (ghost) epoch_base += count;
        push_params();
    }

    // One check iteration: computes T(z) with side products, evaluates KKT + fixed-point error, then
    // either restarts from T(z) or completes the Halpern step.  Returns true when the solve is over.
    bool check_iteration() {
        double h[2 * NACC];
        if (ghost) gather_y(y_full.p);             // the plain iterations only kept the ghost vectors current
        primal_step<true>(0);                      // xbar (gathered), xp
        dual_step<true>(0);                        // yp, axbar; y unchanged
        // A xp on my rows (needs everyone's xp) and A' yp on my columns (needs everyone's yp)
        if (nl > 0) ELP_CUDA(cudaMemcpyAsync(xaux_full.p + n0, xp.p, (size_t)nl * sizeof(double), cudaMemcpyDeviceToDevice, st));
        gather_x(xaux_full.p);
        spmv_rows(xaux_full.p, axp.p);
        if (m > 0) ELP_CUDA(cudaMemcpyAsync(yaux_full.p + (size_t)rank * mb, yp.p, (size_t)m * sizeof(double), cudaMemcpyDeviceToDevice, st));
        gather_y(yaux_full.p);
        spmv_cols(yaux_full.p, gcol.p);
        ELP_LAUNCH(k_check_rows, RED_BLOCKS, RED_THREADS, 0, st, m, axp.p, axbar.p, y(), yp.p, y0.p, lc.p, uc.p, dr.p,
                   partials.p);
        reduce_to(scal.p);
        ELP_LAUNCH(k_check_cols, RED_BLOCKS, RED_THREADS, 0, st, nl, gcol.p, c.p, l.p, u.p, x.p, xp.p, x0.p, dc.p,
                   partials.p);
        reduce_to(scal.p + NACC);
        if (N > 1) {
            // slot 7 of the row sums is free: the ranks agree on a wall-clock exit through the same collective
            const double over = (opt.time_limit_s > 0 && run_clock.ms() > opt.time_limit_s * 1e3) ? 1.0 : 0.0;
            ELP_CUDA(cudaMemcpyAsync(scal.p + 7, &over, sizeof over, cudaMemcpyHostToDevice, st));
            comm_allreduce_sum(scal.p, 2 * NACC, st);       // the scalar residuals: ONE collective
        }
        ELP_CUDA(cudaMemcpyAsync(h, scal.p, 2 * NACC * sizeof(double), cudaMemcpyDeviceToHost, st));
        unsigned int dev_err = 0;
        if (ghost) ELP_CUDA(cudaMemcpyAsync(&dev_err, ghost_mem.p + 128, sizeof dev_err, cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        ELP_REQUIRE(dev_err == 0, "pdlp: rank %d timed out waiting for a peer GPU's block (exchange flag never arrived)", rank);
        d2h += 2 * NACC * sizeof(double);
        time_up = N > 1 ? h[7] > 0.0 : (opt.time_limit_s > 0 && run_clock.ms() > opt.time_limit_s * 1e3);
        ++checks;
        const double* hr = h;
        const double* hc = h + NACC;

        const double tau = eta / w, sigma = eta * w;
        const double fpe2 = hc[1] / tau + 2.0 * hr[1] + hr[2] / sigma;
        const double fpe = std::sqrt(std::max(fpe2, 0.0));
        pobj = hc[3];
        dobj = hr[4] + hc[4];
        rel_pres = std::sqrt(hr[0]) / (1.0 + norm_b);
        rel_dres = std::sqrt(hc[0]) / (1.0 + norm_c);
        rel_gap = std::fabs(pobj - dobj) / (1.0 + std::fabs(pobj) + std::fabs(dobj));
        const double eps = opt.eps_rel;
        if (opt.verbose > 0 && rank == 0)
            fprintf(stderr, "[pdlp] it %7d k %6d pres %.3e dres %.3e gap %.3e pobj %.10e fpe %.3e w %.3e restarts %d\n",
                    total + 1, k, rel_pres, rel_dres, rel_gap, maximize ? -pobj : pobj, fpe, w, restarts);
        ++total;   // this check iteration is a full PDHG iteration
        if (!std::isfinite(fpe) || !std::isfinite(pobj)) {
            status = ELP_STATUS_NUMFAILURE; finished = true; return true;
        }
        // The gap is tested at eps/4: |p - d| <= (eps/4)(1 + |p| + |d|); PDLP's plain gap test allows ~2 eps on the
        // objective.  north_star asks for the OBJECTIVE within eps relative, which none of PDLP's three tests bounds: a
        // primal residual of eps (1 + ||b||) can hide an objective error of up to ||y*|| times that.  obj_err adds the
        // rigorous first-order bounds |yp.(A xp - proj)| and |xp.(dual residual)| (scale-invariant; two spare
        // accumulators of the check kernels) and gap_rule = 1 (ELP_PDLP_GAP_RULE) tests that sum instead.  Measured
        // (profiles/r2_gap_rule.md): the bound overestimates the true error 6-50x — the reduced-cost terms it ignores
        // cancel most of it — and costs 3x (C4 at 50 k rows) to 23x (C4 full size) the iterations, so it is an option
        // for callers who need a certificate, not the default.
        obj_err = (std::fabs(pobj - dobj) + std::fabs(hr[5]) + std::fabs(hc[5])) / (1.0 + std::fabs(pobj) + std::fabs(dobj));
        const bool gap_ok = gap_rule == 0 ? rel_gap <= 0.25 * eps : obj_err <= gap_factor * eps;
        if (rel_pres <= eps && rel_dres <= eps && gap_ok) {
            status = ELP_STATUS_OPTIMAL; finished = true; return true;
        }
        if (k > 0 && (checks % 4 == 0) && detect_infeasible()) { finished = true; return true; }

        if (need_fpe0) { fpe0 = fpe; need_fpe0 = false; }
        bool restart = false;
        if (k > 0) {
            if (fpe <= 0.2 * fpe0) restart = true;
            else if (fpe <= 0.8 * fpe0 && fpe_prev >= 0 && fpe > fpe_prev) restart = true;
            else if ((double)k >= beta_artificial * (double)total) restart = true;
        }
        fpe_prev = fpe;
        const int span = std::max(std::max(nl, m), 1);
        if (restart) {
            const double ddx = std::sqrt(hc[2]), ddy = std::sqrt(hr[3]);
            if (ddx > 1e-10 && ddy > 1e-10) {
                // PID-style controller on log w (cuPDLPx): e = log(w dx / dy) is the imbalance of the two movements;
                // kp = 0.5, ki = kd = 0 is PDLP's geometric-mean smoothing; an integral term (ki > 0) diverged on
                // configs 2 and 5 in the CPU lab, so only the proportional gain is used
                const double e = std::log(w * ddx / ddy);
                w_err_sum = w_ismooth * w_err_sum + e;
                w = std::exp(std::log(w) - (w_kp * e + w_ki * w_err_sum + w_kd * (e - w_err_prev)));
                w_err_prev = e;
            }
            ELP_LAUNCH(k_restart, grid1(span), 256, 0, st, nl, x.p, x0.p, xp.p, m, y(), y0.p, yp.p);
            k = 0; ++restarts; need_fpe0 = true; fpe_prev = -1;
        } else {
            const double wk = halpern_w(k);
            ELP_LAUNCH(k_halpern_finish, grid1(span), 256, 0, st, nl, x.p, xbar(), x0.p, m, y(), yp.p, y0.p, wk);
            ++k;
        }
        refresh_y();                               // y changed: everyone needs the new blocks
        if (scatter) spmv_cols(y_full.p, gcol.p);  // ... and the scatter formulation needs g = A'y of the new y
        push_params();
        return false;
    }

    // Farkas-type certificates from the displacement (xp - x0, yp - y0); see oracle/pdlp_ref.py::_certificate
    bool detect_infeasible() {
        double h[2 * NACC];
        const double tol = 1e-6;
        // ray vectors in the scratch gathered buffers; their images in axp / gcol (both free at this point)
        double* dxl = xaux_full.p + n0;
        double* dyl = yaux_full.p + (size_t)rank * mb;
        launch_diff(nl, xp.p, x0.p, dxl, st);
        launch_diff(m, yp.p, y0.p, dyl, st);
        gather_x(xaux_full.p);
        gather_y(yaux_full.p);
        spmv_rows(xaux_full.p, axp.p);
        spmv_cols(yaux_full.p, gcol.p);
        ELP_LAUNCH(k_ray_rows, RED_BLOCKS, RED_THREADS, 0, st, m, axp.p, yp.p, y0.p, lc.p, uc.p, dr.p, partials.p);
        reduce_to(scal.p);
        ELP_LAUNCH(k_ray_cols, RED_BLOCKS, RED_THREADS, 0, st, nl, xp.p, x0.p, c.p, l.p, u.p, gcol.p, dc.p, partials.p);
        reduce_to(scal.p + NACC);
        if (N > 1) comm_allreduce_sum(scal.p, 2 * NACC, st);
        ELP_CUDA(cudaMemcpyAsync(h, scal.p, 2 * NACC * sizeof(double), cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        d2h += 2 * NACC * sizeof(double);
        const double* hr = h;
        const double* hc = h + NACC;
        // primal infeasibility: dual ray with positive objective and vanishing residual
        const double ray_obj = hr[2] + hc[5];
        const double ny = std::sqrt(hr[1]);
        if (ny > 1e-12 && ray_obj > 0.0) {
            const double res = std::sqrt(hc[4]) + std::sqrt(hr[3]);
            if (res / ray_obj <= tol) { status = ELP_STATUS_INFEASIBLE; return true; }
        }
        // dual infeasibility (primal unbounded): primal ray with negative cost staying feasible
        const double cdx = hc[0];
        const double nx = std::sqrt(hc[3]);
        if (nx > 1e-12 && cdx < 0.0) {
            const double viol = std::sqrt(hr[0]) + std::sqrt(hc[1]);
            if (viol / (-cdx) <= tol) { status = ELP_STATUS_UNBOUNDED; return true; }
        }
        return false;
    }

    void run(int max_new_iters, elp_stats* stats) {
        WallTimer wall;
        if (!clock_running) { run_clock = WallTimer(); clock_running = true; }     // the time limit spans all run() calls of a solve
        const int64_t launches0 = g_launches.load();
        cudaEvent_t e0, e1;
        ELP_CUDA(cudaEventCreate(&e0)); ELP_CUDA(cudaEventCreate(&e1));
        ELP_CUDA(cudaEventRecord(e0, st));
        const int ce = std::max(2, opt.check_every);
        opt.check_every = ce;
        const int limit_total = opt.max_iter > 0 ? opt.max_iter : 2000000;
        int budget = max_new_iters > 0 ? max_new_iters : limit_total;
        if (finished && status != ELP_STATUS_TIMEOUT) budget = 0;
        finished = false;
        while (budget > 0 && total < limit_total) {
            // epoch-relative schedule: a check whenever k % check_every == 0 (k = 0 right after a restart)
            if (k % ce == 0) {
                if (check_iteration()) break;
                --budget;
                if (time_up) { hit_time_limit = true; break; }     // (distributed: agreed on inside the check's allreduce)
                continue;
            }
            int cnt = ce - (k % ce);
            cnt = std::min(cnt, std::min(budget, limit_total - total));
            plain_iterations(cnt);
            budget -= cnt;
        }
        ELP_CUDA(cudaEventRecord(e1, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        float ms = 0;
        ELP_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        if (stats) {
            stats->status = status;
            stats->method_used = ELP_METHOD_PDLP;
            stats->iterations = total;
            stats->restarts = restarts;
            stats->primal_obj = maximize ? -pobj : pobj;
            stats->dual_obj = maximize ? -dobj : dobj;
            stats->rel_primal_res = rel_pres;
            stats->rel_dual_res = rel_dres;
            stats->rel_gap = rel_gap;
            stats->solve_ms = ms;
            stats->total_ms = wall.ms();
            stats->kernel_launches = g_launches.load() - launches0;
            stats->h2d_bytes = h2d;
            stats->d2h_bytes = d2h;
            stats->limit_reached = (status == ELP_STATUS_TIMEOUT) ? (hit_time_limit ? 2 : (total >= limit_total ? 1 : 0)) : 0;
        }
    }

    // x: all n columns (gathered from the ranks' blocks); y: my rows
    // collective_x: take part in the all-gather of x even when this rank does not want the result (x_h == nullptr)
    void solution(double* x_h, double* y_h, double* obj, bool collective_x = false) {
        if (x_h || (collective_x && N > 1)) {
            if (nl > 0) ELP_LAUNCH(k_unscale, grid1(nl), 256, 0, st, nl, xp.p, dc.p, 1.0, xaux_full.p + n0);
            gather_x(xaux_full.p);
            if (x_h) {
                xaux_full.download(x_h, n, st);
                d2h += (int64_t)n * 8;
            }
            ELP_CUDA(cudaStreamSynchronize(st));
        }
        if (y_h && m > 0) {
            ELP_LAUNCH(k_unscale, grid1(m), 256, 0, st, m, yp.p, dr.p, maximize ? -1.0 : 1.0, axp.p);
            axp.download(y_h, m, st);
            ELP_CUDA(cudaStreamSynchronize(st));
            d2h += (int64_t)m * 8;
        }
        if (obj) *obj = maximize ? -pobj : pobj;
    }

    // Times the two iteration kernels as they run in a solve: `reps` iterations (primal kernel, dual kernel, no
    // collective) from a mid-solve iterate, one CUDA event between any two launches, so that the two figures add up to
    // the iteration time.  Leaves the solver reset.
    void probe_step(int reps, double* ms_primal, double* ms_dual) {
        reps = std::max(1, std::min(reps, 512));
        reset();
        run(3 * std::max(2, opt.check_every), nullptr);
        std::vector<cudaEvent_t> ev(2 * (size_t)reps + 1);
        for (auto& e : ev) ELP_CUDA(cudaEventCreate(&e));
        // real iterations, exchange included (multi-GPU: the peers run the same sequence).  run() may have ended with a
        // restart (x-bar stale): the first one reads x itself.
        for (int i = 0; i < 3; ++i) { primal_step<false>(i, false, i == 0); dual_step<false>(i); }
        for (int i = 0; i < reps; ++i) {
            ELP_CUDA(cudaEventRecord(ev[2 * i], st));
            primal_step<false>(3 + i, false);
            ELP_CUDA(cudaEventRecord(ev[2 * i + 1], st));
            dual_step<false>(3 + i);
        }
        ELP_CUDA(cudaEventRecord(ev[2 * reps], st));
        if (ghost) epoch_base += 3 + reps;
        ELP_CUDA(cudaStreamSynchronize(st));
        double tp = 0.0, td = 0.0;
        for (int i = 0; i < reps; ++i) {
            float ms = 0;
            ELP_CUDA(cudaEventElapsedTime(&ms, ev[2 * i], ev[2 * i + 1]));
            tp += ms;
            ELP_CUDA(cudaEventElapsedTime(&ms, ev[2 * i + 1], ev[2 * i + 2]));
            td += ms;
        }
        for (auto& e : ev) cudaEventDestroy(e);
        if (ms_primal) *ms_primal = tp / reps;
        if (ms_dual) *ms_dual = td / reps;
        reset();
    }

    void probe_spmv(int reps, double* ms_csr, double* ms_csc) {
        cudaEvent_t e0, e1;
        ELP_CUDA(cudaEventCreate(&e0)); ELP_CUDA(cudaEventCreate(&e1));
        float ms = 0;
        for (int i = 0; i < 3; ++i) { spmv_rows(xbar_full.p, axp.p); }
        ELP_CUDA(cudaEventRecord(e0, st));
        for (int i = 0; i < reps; ++i) spmv_rows(xbar_full.p, axp.p);
        ELP_CUDA(cudaEventRecord(e1, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        ELP_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (ms_csr) *ms_csr = ms / reps;
        for (int i = 0; i < 3; ++i) spmv_cols(y_full.p, gcol.p);
        ELP_CUDA(cudaEventRecord(e0, st));
        for (int i = 0; i < reps; ++i) spmv_cols(y_full.p, gcol.p);
        ELP_CUDA(cudaEventRecord(e1, st));
        ELP_CUDA(cudaStreamSynchronize(st));
        ELP_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (ms_csc) *ms_csc = ms / reps;
        cudaEventDestroy(e0); cudaEventDestroy(e1);
    }
};

// ---- entry points used by abi.cu -----------------------------------------------------------------
Pdlp* pdlp_create(int m, int n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                  const int8_t* sense, const double* rhs, const double* c, int maximize, const double* lb,
                  const double* ub, const elp_options& opt, bool dist, elp_stats* stats, int64_t nnz_device) {
    WallTimer t;
    auto* p = new Pdlp();
    try {
        p->setup(m, n, row_ptr, col_idx, vals, sense, rhs, c, maximize, lb, ub, opt, dist, nnz_device);
    } catch (...) {
        delete p;
        throw;
    }
    if (stats) { stats->setup_ms = t.ms(); stats->h2d_bytes = p->h2d; }
    return p;
}
void pdlp_run(Pdlp* p, int max_new_iters, elp_stats* stats) { p->run(max_new_iters, stats); }
void pdlp_reset(Pdlp* p) { p->reset(); }
void pdlp_solution(Pdlp* p, double* x, double* y, double* obj, bool collective_x) { p->solution(x, y, obj, collective_x); }
void pdlp_probe(Pdlp* p, int reps, double* a, double* b) { p->probe_spmv(reps, a, b); }
void pdlp_probe_step(Pdlp* p, int reps, double* a, double* b) { p->probe_step(reps, a, b); }
int pdlp_transpose(Pdlp* p) { return p->scatter ? ELP_TRANSPOSE_SCATTER : ELP_TRANSPOSE_GATHER; }
void pdlp_destroy(Pdlp* p) { delete p; }

// plain SpMV + feasibility re-check (S4: /root/reference/R/class.R:533-540, R/utils.R:167-171)
__global__ void k_compare_tol(int m, const double* __restrict__ lhs, const double* __restrict__ rhs,
                              const int8_t* __restrict__ sense, double tol, uint8_t* __restrict__ ok) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const double a = lhs[i], b = rhs[i];
    bool f;
    switch (sense[i]) {
        case 0: f = (a + tol <= b) || (a - tol <= b); break;           // "<="  any(lhs +/- tol <= rhs)
        case 1: f = (a + tol >= b) || (a - tol >= b); break;           // ">="
        case 2: f = fabs(a - b) <= tol; break;                          // "=="
        case 3: f = (a + tol < b) || (a - tol < b); break;             // "<"  stays strict (match.fun(dir))
        default: f = (a + tol > b) || (a - tol > b); break;            // ">"
    }
    ok[i] = f ? 1 : 0;
}

void spmv_host(int m, int n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals, const double* x,
               double* out, const int8_t* sense, const double* rhs, double tol, uint8_t* feasible) {
    cudaStream_t st = 0;
    const int64_t nnz = m > 0 ? row_ptr[m] : 0;
    if (m == 0) return;
    Arena arena;                 // eight buffers, one allocation
    arena.reserve((size_t)12 * (nnz + SPMV_PAD) + (size_t)8 * std::max(n, 1) + (size_t)30 * (m + 8) + 16 * 512);
    ArenaScope scope(arena.base ? &arena : nullptr);
    DevBuf<int> ptr(m + 1 + SPMV_PTR_PAD), idx(nnz + SPMV_PAD);
    DevBuf<double> val(nnz + SPMV_PAD), xd(std::max(n, 1)), od(m);
    idx.zero(st); val.zero(st); ptr.zero(st);
    ptr.upload(row_ptr, m + 1, st); idx.upload(col_idx, nnz, st); val.upload(vals, nnz, st); xd.upload(x, n, st);
    // one thread per row: the row sum is formed in index order, bit-identical to a scalar loop
    launch_spmv(plan_spmv(nnz, m, 0, 1), m, ptr.p, idx.p, val.p, xd.p, store_epi(od.p), st);
    if (out) od.download(out, m, st);
    if (feasible) {
        DevBuf<int8_t> sd(m);
        DevBuf<double> rd(m);
        DevBuf<uint8_t> fd(m);
        sd.upload(sense, m, st); rd.upload(rhs, m, st);
        ELP_LAUNCH(k_compare_tol, ceil_div(m, 256), 256, 0, st, m, od.p, rd.p, sd.p, tol, fd.p);
        fd.download(feasible, m, st);
        ELP_CUDA(cudaStreamSynchronize(st));
        return;
    }
    ELP_CUDA(cudaStreamSynchronize(st));
}

}  // namespace elp
