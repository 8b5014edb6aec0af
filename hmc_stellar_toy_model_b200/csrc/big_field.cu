// Large-field RHMC engine: one crowded field too big for a single CTA (BASELINE configs[2] scaled up and configs[4]),
// optionally one row-strip of a field tiled over several GPUs.
//
// State lives in global memory; one leapfrog step is a fixed sequence of small kernels enqueued on the context's
// stream with no host synchronisation (the only host involvement inside a chain is enqueueing, plus -- when the
// field is tiled over GPUs -- the collectives between phases, which the caller issues on the same stream):
//
//   scatter  one warp per star adds f PSF over its (2r+1)^2 patch into the model image Lambda (FP64 atomics into L2)
//   pixel    rho = D/Lambda - 1 in place, V = sum(Lambda - D ln Lambda) over the OWNED rows (fixed-order partials)
//   gather   one warp per star: the three residual-weighted PSF reductions over its patch (shuffle reductions)
//   scalar   one thread per star: metric, half kicks, both implicit fixed points, reflections, momentum refresh
//
// The reference's field-wide stop rule of the fixed-point loops (sampler_RHMC.py:533,543: max over ALL stars) is kept
// exactly with two phases per loop: phase A iterates every star to its own convergence and takes the maximum count
// (atomicMax; across GPUs an all-reduce(max) by the caller), phase B continues every star to that count.  The
// per-star iterations are contractions, so a star that met the tolerance stays within it (same result as iterating
// all stars together).
//
// Tiling: a rank owns global rows [own_lo, own_hi) and holds data rows [row0, row0+nrows) (strip + halo).  Owned
// stars may drift `halo - patch_radius` rows outside the strip; neighbours' stars that can touch the local rows
// arrive as ghosts (f, x, y) in the gathered boundary buffers and are only rendered, never updated.
#include <cuda.h>   // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint, no -lcuda)
#include <cuda_runtime.h>
#include <math_constants.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "../../include/stellar_rhmc.h"
#include "common.cuh"
#include "fastmath.cuh"
#include "poisson.cuh"

using namespace srhmc;

namespace {

thread_local char g_big_err[512] = "";

int bfail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_big_err, sizeof(g_big_err), fmt, ap);
    va_end(ap);
    return code;
}

#define BCU(expr)                                                                                            \
    do {                                                                                                     \
        cudaError_t e__ = (expr);                                                                            \
        if (e__ != cudaSuccess)                                                                              \
            return bfail(SRHMC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

struct BigParams {
    int Rg, C;              // global rows, columns
    int row0, nrows;        // local data rows [row0, row0 + nrows)
    int own_lo, own_hi;     // owned rows
    int rad;
    int use_prior;
    double inv2s2, inv_s2, norm;
    FieldParams F;          // constants for metric_of (B, g0.., f_low, f_lim, alpha, Vpc)
};

constexpr int kMaxRad = 15;
constexpr int kScalars = 8;   // [0] V partial, [1] T partial, [2] bad count, [3] spare ... (doubles)
constexpr int kVBlocks = 1024;

// ------------------------------------------------------------------------------------------------ pixel kernels
__global__ void big_fill_kernel(double* L, size_t n, double B) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) L[i] = B;
}

// Patch geometry of a star in LOCAL row indices.  Returns false when the star does not touch the local rows.
// `clipped_by_data` is set when the patch is cut by the local data window but not by the global image edge.
__device__ __forceinline__ bool patch_of(const BigParams& P, double x, double y, int& i0, int& i1, int& j0, int& j1,
                                         int& mi, int& mj, bool& clipped_by_data) {
    const double fx = floor(x), fy = floor(y);
    mi = (fx > 0.0) ? ((fx > (double)(P.Rg - 1)) ? P.Rg - 1 : (int)fx) : 0;
    mj = (fy > 0.0) ? ((fy > (double)(P.C - 1)) ? P.C - 1 : (int)fy) : 0;
    const int gi0 = max(0, mi - P.rad), gi1 = min(P.Rg - 1, mi + P.rad);
    j0 = max(0, mj - P.rad);
    j1 = min(P.C - 1, mj + P.rad);
    i0 = max(gi0, P.row0);
    i1 = min(gi1, P.row0 + P.nrows - 1);
    clipped_by_data = (i0 != gi0) || (i1 != gi1);
    return i0 <= i1;
}

// Last-block election for fixed-order two-stage reductions: every block publishes its partials, takes a ticket, and
// the block that draws the last ticket sums all partials in index order (bit-reproducible, one launch).
__device__ __forceinline__ bool last_block_ticket(unsigned int* ticket, bool* flag) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        *flag = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (*flag) __threadfence();
    return *flag;
}

}  // namespace

#include "big_tile.cuh"
#include "big_star.cuh"

namespace {

// One warp per star (own stars first, then the two ghost lists).  ghost list layout: [0] = count, then f,x,y triples.
__global__ void big_scatter_kernel(const BigParams P, const double* q, int n_own, const double* ghost_a,
                                   const double* ghost_b, double* L, int* err) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int na = ghost_a ? (int)ghost_a[0] : 0, nb = ghost_b ? (int)ghost_b[0] : 0;
    const long long total = (long long)n_own + na + nb;
    for (long long s = warp; s < total; s += nwarps) {
        const double* src = s < n_own ? q + 3 * s : (s < n_own + na ? ghost_a + 1 + 3 * (s - n_own) : ghost_b + 1 + 3 * (s - n_own - na));
        const double f = src[0], x = src[1], y = src[2];
        int i0, i1, j0, j1, mi, mj;
        bool clipped;
        if (!patch_of(P, x, y, i0, i1, j0, j1, mi, mj, clipped)) {
            if (s < n_own && lane == 0) atomicExch(err, 1);  // an owned star left the local data window
            continue;
        }
        if (s < n_own && clipped && lane == 0) atomicExch(err, 1);
        // lanes own columns j0 + lane (2 rad + 1 <= 31 columns); row factors by shuffle
        const int j = j0 + lane;
        const bool okc = j <= j1;
        const double dy = ((double)j + 0.5) - y;
        const double ey = okc ? exp(-(dy * dy) * P.inv2s2) * P.norm * f : 0.0;
        const int irow = i0 + lane;
        const double dxl = ((double)(irow + 0) + 0.5) - x;
        const double exl = (irow <= i1) ? exp(-(dxl * dxl) * P.inv2s2) : 0.0;
        for (int i = i0; i <= i1; ++i) {
            const double ex = __shfl_sync(0xffffffffu, exl, i - i0);
            if (okc) atomicAdd(&L[(size_t)(i - P.row0) * P.C + j], ex * ey);
        }
    }
}

// rho = D/Lambda - 1 in place; V over owned rows; per-block partials in fixed order.
__global__ void big_pixel_kernel(const BigParams P, const double* D, double* L, int want_V, double* vpart) {
    __shared__ double red[32];
    const size_t n = (size_t)P.nrows * P.C;
    const size_t own0 = (size_t)(P.own_lo - P.row0) * P.C, own1 = (size_t)(P.own_hi - P.row0) * P.C;
    double v = 0.0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const double lam = L[i], d = D[i];
        L[i] = d / lam - 1.0;
        if (want_V && i >= own0 && i < own1) v += lam - d * log(lam);
    }
    if (want_V) {
        double a[1] = {v};
        block_sum<1>(a, red);
        if (threadIdx.x == 0) vpart[blockIdx.x] = a[0];
    }
}

// sum of the per-block partials in index order (one block) -> scalars[0]
__global__ void big_vsum_kernel(const double* vpart, int nblocks, double* scalars) {
    __shared__ double red[32];
    double v = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += blockDim.x) v += vpart[i];
    double a[1] = {v};
    block_sum<1>(a, red);
    if (threadIdx.x == 0) scalars[0] = a[0];
}

// One warp per OWNED star: g_f = -sum rho PSF, g_x = -(f/s^2) sum rho dx PSF, g_y likewise (sampler_RHMC.py:404-406).
__global__ void big_gather_kernel(const BigParams P, const double* q, int n_own, const double* L, double* g) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long s = warp; s < n_own; s += nwarps) {
        const double f = q[3 * s], x = q[3 * s + 1], y = q[3 * s + 2];
        int i0, i1, j0, j1, mi, mj;
        bool clipped;
        double sf = 0.0, sx = 0.0, sy = 0.0;
        if (patch_of(P, x, y, i0, i1, j0, j1, mi, mj, clipped)) {
            const int j = j0 + lane;
            const bool okc = j <= j1;
            const double dy = ((double)j + 0.5) - y;
            const double ey = okc ? exp(-(dy * dy) * P.inv2s2) * P.norm : 0.0;
            const int irow = i0 + lane;
            const double dxl = ((double)irow + 0.5) - x;
            const double exl = (irow <= i1) ? exp(-(dxl * dxl) * P.inv2s2) : 0.0;
            // the lane's column of the residual patch first, all loads in flight together (one L2 latency instead of one per
            // row: this kernel runs one wave of warps on the small fields it serves, so its time IS that latency chain)
            constexpr int kRows = 2 * kMaxRad + 1;
            double rr[kRows];
            const double* lp = L + (size_t)(i0 - P.row0) * P.C + min(j, j1);
            const int nrow = i1 - i0 + 1;
#pragma unroll
            for (int r = 0; r < kRows; ++r) rr[r] = (r < nrow) ? __ldcg(lp + (size_t)r * P.C) : 0.0;
            double c0 = 0.0, c1 = 0.0;
#pragma unroll
            for (int r = 0; r < kRows; ++r) {
                if (r < nrow) {
                    const double ex = __shfl_sync(0xffffffffu, exl, r);
                    const double dx = ((double)(i0 + r) + 0.5) - x;
                    const double rho = okc ? rr[r] : 0.0;
                    c0 = fma(rho, ex, c0);
                    c1 = fma(rho, ex * dx, c1);
                }
            }
            sf = ey * c0;
            sx = ey * c1;
            sy = ey * dy * c0;
        }
        sf = warp_sum(sf);
        sx = warp_sum(sx);
        sy = warp_sum(sy);
        if (lane == 0) {
            g[3 * s] = -sf;
            g[3 * s + 1] = -sx * f * P.inv_s2;
            g[3 * s + 2] = -sy * f * P.inv_s2;
        }
    }
}

// ------------------------------------------------------------------------------------------------ peer exchange
// Collectives of the tiled field done by our own kernels over peer-mapped memory (NVLink P2P between the GPUs of a node;
// CUDA IPC between their processes) instead of NCCL: every rank owns one PeerBox that all ranks can address.  A
// contribution is `payload, then tag = epoch` (system-scope fence in between); the receiver spins on the tag.  Slots are
// double-buffered by epoch parity: a rank can run at most one exchange ahead of a peer, because finishing exchange k+1
// needs the peer's k+1 contribution, which the peer sends only after it has consumed exchange k.  Epochs live in device
// memory and are advanced by the kernels themselves, so a captured CUDA graph of an iteration can be replayed.
constexpr int kMaxWorld = 16;

struct PeerSlot {                 // one small-vector contribution
    unsigned long long tag;
    double v[8];
    unsigned long long mword;     // max exchange: (epoch << 32) | value in ONE 8-byte store -- value and flag arrive together,
                                  // so the exchange needs no system-scope fence on either side
    double pad[6];                // 128 bytes
};
static_assert(sizeof(PeerSlot) == 128, "PeerSlot layout");

// fence-free exchange of one non-negative int tagged with the epoch
__device__ __forceinline__ void peer_send_word(PeerSlot* s, unsigned long long e, int val) {
    *reinterpret_cast<volatile unsigned long long*>(&s->mword) = (e << 32) | (unsigned long long)(unsigned int)val;
}

struct PeerHeader {
    PeerSlot ar[2][kMaxWorld];    // [epoch parity][source rank]
    unsigned long long gtag[2][2];  // ghost mailboxes [parity][side]: tag
};
// ghost mailbox payloads follow the header: [parity][side][list doubles]

struct PeerPtrs {
    unsigned char* box[kMaxWorld];
};

__device__ __forceinline__ void peer_publish_tag(unsigned long long* tag, unsigned long long e) {
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long*>(tag) = e;
}

// spin until *tag >= e; false (and err flag 4) after ~5 s so that a lost peer cannot hang the GPU; once the flag is up
// every later wait gives up at once
__device__ __forceinline__ bool peer_wait_tag(const unsigned long long* tag, unsigned long long e, int* err) {
    const long long t0 = clock64();
    while (*reinterpret_cast<const volatile unsigned long long*>(tag) < e) {
        if (*reinterpret_cast<volatile int*>(err) == 4) return false;
        if (clock64() - t0 > 10000000000LL) {
            atomicExch(err, 4);
            return false;
        }
        __nanosleep(100);
    }
    __threadfence_system();
    return true;
}


// spin until the packed word of slot `s` carries epoch >= e; its low half is the value.  Same time-out rule as peer_wait_tag.
__device__ __forceinline__ bool peer_wait_word(const PeerSlot* s, unsigned long long e, int* err, int& val) {
    const long long t0 = clock64();
    unsigned long long w;
    while (((w = *reinterpret_cast<const volatile unsigned long long*>(&s->mword)) >> 32) < e) {
        if (*reinterpret_cast<volatile int*>(err) == 4) return false;
        if (clock64() - t0 > 10000000000LL) {
            atomicExch(err, 4);
            return false;
        }
        __nanosleep(40);
    }
    val = (int)(unsigned int)(w & 0xffffffffull);
    return true;
}

// What the kernels that produce a fixed-point count need for its all-reduce (all zero without peer exchange)
struct PeerX {
    PeerPtrs peers;
    int rank, world;
    int prod;   // peer exchange is on: the kernel's last block all-reduces the count (peer_max_epilogue)
    unsigned long long* epoch;
    unsigned int* ticket;
    int* err;
};

// all-reduce(max) of *word over the ranks by the LAST block to leave the kernel that produced it: the word is complete (every
// block's atomicMax precedes its ticket), one block polls the mailbox, and the consumer kernel just reads the word.
__device__ __forceinline__ void peer_max_epilogue(const PeerX& X, int* word) {
    __shared__ int s_last, s_max;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(X.ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const unsigned long long e = X.epoch[0] + 1;
    const int par = (int)(e & 1), t = threadIdx.x;
    const int local = *reinterpret_cast<volatile int*>(word);
    if (t == 0) s_max = local;
    __syncthreads();
    if (t < X.world) {
        peer_send_word(&reinterpret_cast<PeerHeader*>(X.peers.box[t])->ar[par][X.rank], e, local);
        const PeerSlot* mine = &reinterpret_cast<const PeerHeader*>(X.peers.box[X.rank])->ar[par][t];
        int got = 0;
        if (peer_wait_word(mine, e, X.err, got)) atomicMax(&s_max, got);
    }
    __syncthreads();
    if (t == 0) {
        *word = s_max;
        X.epoch[0] = e;
        *X.ticket = 0u;
    }
}

// ------------------------------------------------------------------------------------------------ scalar kernels
struct BigStep {
    double h, delta, g_ff2;
    int counter_max;
    int per_star;   // srhmc_big_step.fixed_point_mode = 1: every star's fixed points stop at the star's own convergence
    MetricK K;      // constants of the division-free metric (metric_fast, common.cuh), computed on the host
};

// The per-star kernels use the metric in its division-free form (metric_fast: rcp_fast reciprocals, 2^-60): an FP64 division
// is ~30 instructions on a dependent path and these kernels are either latency-bound (a strip of a tiled field) or spend most
// of their instructions dividing.  Same iterates to rounding, same fixed-point counts (tests/test_bigfield.py).
__device__ __forceinline__ double dphi_f(const BigParams& P, const MetricFast& m, double gpix_f, double f) {
    double gf = gpix_f;
    if (P.use_prior) gf = fma(P.F.alpha, rcp_fast(f), gf);
    return gf + m.tphi;
}

// (1) p -= h dphi/dq; (2) p fixed point, phase A: iterate to this star's own convergence, record the count
__global__ void big_kick1_kernel(const BigParams P, const BigStep S, int n, const double* q, double* p, const double* g,
                                 double* a1, double* a2, int* cnt, const PeerX X) {
    int local_max = 0;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const double f = q[3 * k];
        const MetricFast m = metric_fast(S.K, f);
        double pf = p[3 * k] - S.h * dphi_f(P, m, g[3 * k], f);
        p[3 * k + 1] -= S.h * g[3 * k + 1];
        p[3 * k + 2] -= S.h * g[3 * k + 2];
        const double rho = pf, kap = m.kap;
        a1[3 * k] = rho;      // anchor
        a2[3 * k] = kap;
        int c = 0;
        while (c < S.counter_max) {
            const double pn = rho - S.h * (((pf * pf) * kap) / 2.0);
            const bool more = fabs(pf - pn) > S.delta;
            pf = pn;
            ++c;
            if (!more) break;
        }
        p[3 * k] = pf;
        a1[3 * k + 1] = (double)c;  // own count
        local_max = max(local_max, c);
    }
    if (local_max) atomicMax(cnt, local_max);
    if (X.prod && !S.per_star) peer_max_epilogue(X, cnt);
}

// p fixed point phase B (continue to the global count), then (3) q fixed point phase A
__global__ void big_pfix_qfix_kernel(const BigParams P, const BigStep S, int n, double* q, double* p, double* a1, double* a2,
                                     const int* cnt_p, int* cnt_q, const PeerX X) {
    const int target = S.per_star ? 0 : *cnt_p;
    int local_max = 0;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        double pf = p[3 * k];
        const double rho = a1[3 * k], kap = a2[3 * k];
        for (int c = (int)a1[3 * k + 1]; c < target; ++c) pf = rho - S.h * (((pf * pf) * kap) / 2.0);
        p[3 * k] = pf;
        // q' = sigma + h (p/H(sigma) + p/H(q))
        const double sf = q[3 * k], sx = q[3 * k + 1], sy = q[3 * k + 2];
        const double px = p[3 * k + 1], py = p[3 * k + 2];
        const double u0 = inv_hff_k(S.K, sf), ih0 = inv_hxx_k(S.K, sf);
        const double bf = pf * u0, bx = px * ih0, by = py * ih0;
        double qf = sf, qx = sx, qy = sy;
        int c = 0;
        while (c < S.counter_max) {
            const double uq = inv_hff_k(S.K, qf), ihq = inv_hxx_k(S.K, qf);
            const double nf = sf + S.h * (bf + pf * uq);
            const double nx = sx + S.h * (bx + px * ihq);
            const double ny = sy + S.h * (by + py * ihq);
            const double d = fmax(fabs(qf - nf), fmax(fabs(qx - nx), fabs(qy - ny)));
            qf = nf; qx = nx; qy = ny;
            ++c;
            if (!(d > S.delta)) break;
        }
        a1[3 * k] = sf; a1[3 * k + 1] = sx; a1[3 * k + 2] = sy;   // sigma
        a2[3 * k] = bf; a2[3 * k + 1] = bx; a2[3 * k + 2] = by;   // p/H(sigma)
        q[3 * k] = qf; q[3 * k + 1] = qx; q[3 * k + 2] = qy;
        local_max = max(local_max, c);
        reinterpret_cast<int*>(a2 + 3 * (size_t)n)[k] = c;   // own count, past the 3n doubles of a2
    }
    if (local_max) atomicMax(cnt_q, local_max);
    if (X.prod && !S.per_star) peer_max_epilogue(X, cnt_q);
}

// q fixed point phase B, then (4) p -= h dtau/dq at the new q
// and -- tile path -- the pair records of the star's final position for the coming evaluation (bin_star, big_tile.cuh)
__global__ void big_qfix_kick_kernel(const BigParams P, const BigStep S, int n, double* q, double* p, const double* a1,
                                     const double* a2, const int* cnt_q, int ntx, int* tcnt, PairRec* tlist, int* err,
                                     int2* pack_counts, double lo_edge, double hi_edge, double* Lfill, size_t npix) {
    // star-parallel evaluation path: the model image of the COMING evaluation is reset to the background here (nobody reads
    // it between the last gather and the next scatter), which saves that path a launch per leapfrog step
    if (Lfill)
        for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < npix; i += (size_t)gridDim.x * blockDim.x) Lfill[i] = P.F.B;
    const int target = S.per_star ? 0 : *cnt_q;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const double sf = a1[3 * k], sx = a1[3 * k + 1], sy = a1[3 * k + 2];
        const double bf = a2[3 * k], bx = a2[3 * k + 1], by = a2[3 * k + 2];
        const double pf = p[3 * k], px = p[3 * k + 1], py = p[3 * k + 2];
        double qf = q[3 * k], qx = q[3 * k + 1], qy = q[3 * k + 2];
        for (int c = reinterpret_cast<const int*>(a2 + 3 * (size_t)n)[k]; c < target; ++c) {
            const double uq = inv_hff_k(S.K, qf), ihq = inv_hxx_k(S.K, qf);
            qf = sf + S.h * (bf + pf * uq);
            qx = sx + S.h * (bx + px * ihq);
            qy = sy + S.h * (by + py * ihq);
        }
        q[3 * k] = qf; q[3 * k + 1] = qx; q[3 * k + 2] = qy;
        const MetricFast m = metric_fast(S.K, qf);
        p[3 * k] = pf - S.h * (((pf * pf) * m.kap) / 2.0);
        if (tcnt) bin_star(P, ntx, k, qf, qx, qy, true, tcnt, tlist, err);
        // boundary-star counts per 1024-star chunk for the ordered ghost packing that follows (integer atomics: exact)
        if (pack_counts) {
            if (qx < lo_edge) atomicAdd(&pack_counts[k >> 10].x, 1);
            if (qx >= hi_edge) atomicAdd(&pack_counts[k >> 10].y, 1);
        }
    }
}

// (5) p -= h dphi/dq at the new q; (6) reflections
__global__ void big_kick2_kernel(const BigParams P, const BigStep S, int n, const double* q, double* p, const double* g) {
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const double f = q[3 * k], x = q[3 * k + 1], y = q[3 * k + 2];
        const MetricFast m = metric_fast(S.K, f);
        double pf = p[3 * k] - S.h * dphi_f(P, m, g[3 * k], f);
        double px = p[3 * k + 1] - S.h * g[3 * k + 1];
        double py = p[3 * k + 2] - S.h * g[3 * k + 2];
        if (f < P.F.f_lim) pf *= -1.0;
        if ((x < 0.0) || (x > P.Rg - 1.0)) px *= -1.0;
        if ((y < 0.0) || (y > P.C - 1.0)) py *= -1.0;
        p[3 * k] = pf; p[3 * k + 1] = px; p[3 * k + 2] = py;
    }
}

// Per-star stop rule (srhmc_big_step.fixed_point_mode = 1): nothing in steps (1)-(4) of a leapfrog step couples the stars any
// more, so everything between two gradient evaluations is ONE per-star kernel and no iteration count crosses the GPUs:
//   [FROM_EVAL: g = sum of the footprint partials, (5) last half kick and (6) reflections of the step that just ended]
//   (1) p -= h dphi/dq, (2) p fixed point, (3) q fixed point -- each to the star's own convergence --,
//   (4) p -= h dtau/dq at the new q, pair records of the new position, boundary-star counts for the ghost packing.
// Same expressions, in the same order, as big_tail_kernel / big_kick1_kernel / big_pfix_qfix_kernel / big_qfix_kick_kernel.
template <bool FROM_EVAL>
__global__ void big_perstar_kernel(const BigParams P, const BigStep S, int n, double* q, double* p, double* g, const double* gpart,
                                   int ntx, int* tcnt, PairRec* tlist, int* err, int2* pack_counts, double lo_edge, double hi_edge,
                                   double* Lfill, size_t npix) {
    if (Lfill)   // as big_qfix_kick_kernel: background reset of the star-parallel path's model image
        for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < npix; i += (size_t)gridDim.x * blockDim.x) Lfill[i] = P.F.B;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const double sf = q[3 * k], sx = q[3 * k + 1], sy = q[3 * k + 2];
        double gf, gx, gy;
        if (FROM_EVAL && gpart) {
            gsum_star(P, k, sf, sx, sy, gpart, gf, gx, gy);
            g[3 * k] = gf; g[3 * k + 1] = gx; g[3 * k + 2] = gy;
        } else {
            gf = g[3 * k]; gx = g[3 * k + 1]; gy = g[3 * k + 2];
        }
        const MetricFast m0 = metric_fast(S.K, sf);
        const double dphi = dphi_f(P, m0, gf, sf);
        double pf = p[3 * k], px = p[3 * k + 1], py = p[3 * k + 2];
        if (FROM_EVAL) {
            pf = pf - S.h * dphi;
            px -= S.h * gx;
            py -= S.h * gy;
            if (sf < P.F.f_lim) pf *= -1.0;
            if ((sx < 0.0) || (sx > P.Rg - 1.0)) px *= -1.0;
            if ((sy < 0.0) || (sy > P.C - 1.0)) py *= -1.0;
        }
        // (1), (2)
        pf = pf - S.h * dphi;
        px -= S.h * gx;
        py -= S.h * gy;
        {
            const double rho = pf, kap = m0.kap;
            int c = 0;
            while (c < S.counter_max) {
                const double pn = rho - S.h * (((pf * pf) * kap) / 2.0);
                const bool more = fabs(pf - pn) > S.delta;
                pf = pn;
                ++c;
                if (!more) break;
            }
        }
        // (3) q' = sigma + h (p/H(sigma) + p/H(q))
        const double bf = pf * m0.u, bx = px * m0.ihxx, by = py * m0.ihxx;
        double qf = sf, qx = sx, qy = sy;
        {
            int c = 0;
            while (c < S.counter_max) {
                const double uq = inv_hff_k(S.K, qf), ihq = inv_hxx_k(S.K, qf);
                const double nf = sf + S.h * (bf + pf * uq);
                const double nx = sx + S.h * (bx + px * ihq);
                const double ny = sy + S.h * (by + py * ihq);
                const double d = fmax(fabs(qf - nf), fmax(fabs(qx - nx), fabs(qy - ny)));
                qf = nf; qx = nx; qy = ny;
                ++c;
                if (!(d > S.delta)) break;
            }
        }
        q[3 * k] = qf; q[3 * k + 1] = qx; q[3 * k + 2] = qy;
        // (4)
        const MetricFast m = metric_fast(S.K, qf);
        p[3 * k] = pf - S.h * (((pf * pf) * m.kap) / 2.0);
        p[3 * k + 1] = px;
        p[3 * k + 2] = py;
        if (tcnt) bin_star(P, ntx, k, qf, qx, qy, true, tcnt, tlist, err);
        if (pack_counts) {
            if (qx < lo_edge) atomicAdd(&pack_counts[k >> 10].x, 1);
            if (qx >= hi_edge) atomicAdd(&pack_counts[k >> 10].y, 1);
        }
    }
}

// Tail of a leapfrog step in ONE per-star kernel: [tile path: g = sum of the footprint partials (gsum_star)] ->
// (5) p -= h dphi/dq at the new q -> (6) reflections -> [NEXT: steps (1) and (2, phase A) of the following leapfrog
// step, which start from the same q and the same gradient].  Same operations in the same order as big_gsum_kernel,
// big_kick2_kernel and big_kick1_kernel run back to back.
template <bool NEXT>
__global__ void big_tail_kernel(const BigParams P, const BigStep S, int n, const double* q, double* p, double* g,
                                const double* gpart, double* a1, double* a2, int* cnt, const PeerX X) {
    int local_max = 0;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const double f = q[3 * k], x = q[3 * k + 1], y = q[3 * k + 2];
        double gf, gx, gy;
        if (gpart) {
            gsum_star(P, k, f, x, y, gpart, gf, gx, gy);
            g[3 * k] = gf; g[3 * k + 1] = gx; g[3 * k + 2] = gy;
        } else {
            gf = g[3 * k]; gx = g[3 * k + 1]; gy = g[3 * k + 2];
        }
        const MetricFast m = metric_fast(S.K, f);
        const double dphi = dphi_f(P, m, gf, f);
        double pf = p[3 * k] - S.h * dphi;
        double px = p[3 * k + 1] - S.h * gx;
        double py = p[3 * k + 2] - S.h * gy;
        if (f < P.F.f_lim) pf *= -1.0;
        if ((x < 0.0) || (x > P.Rg - 1.0)) px *= -1.0;
        if ((y < 0.0) || (y > P.C - 1.0)) py *= -1.0;
        if (NEXT) {
            pf = pf - S.h * dphi;
            px -= S.h * gx;
            py -= S.h * gy;
            const double rho = pf, kap = m.kap;
            a1[3 * k] = rho;
            a2[3 * k] = kap;
            int c = 0;
            while (c < S.counter_max) {
                const double pn = rho - S.h * (((pf * pf) * kap) / 2.0);
                const bool more = fabs(pf - pn) > S.delta;
                pf = pn;
                ++c;
                if (!more) break;
            }
            a1[3 * k + 1] = (double)c;
            local_max = max(local_max, c);
        }
        p[3 * k] = pf; p[3 * k + 1] = px; p[3 * k + 2] = py;
    }
    if (NEXT && local_max) atomicMax(cnt, local_max);
    if (NEXT && X.prod && !S.per_star) peer_max_epilogue(X, cnt);
}

// momentum refresh p = z sqrt(H) (sampler_RHMC.py:1021-1022) with device Philox keyed by the GLOBAL star id, or
// injected normals; saves the iteration's start state
__global__ void big_momentum_kernel(const BigParams P, double g_ff2, int n, const double* q, double* p, const double* g,
                                    double* q0, double* g0, const long long* gid, unsigned long long seed, int iter_host,
                                    const int* iter_dev, const double* normals_all /* [iters,n,3] or nullptr */) {
    const int iter = iter_dev ? *iter_dev : iter_host;
    const double* normals = normals_all ? normals_all + (size_t)iter * n * 3 : nullptr;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const Metric m = metric_of(P.F, q[3 * k], g_ff2);
        double z[3];
        if (normals) {
            z[0] = normals[3 * k]; z[1] = normals[3 * k + 1]; z[2] = normals[3 * k + 2];
        } else {
            philox_normals3(seed, 0u, (uint32_t)iter, (uint32_t)gid[k], z);
        }
        p[3 * k] = z[0] * sqrt(m.Hff);
        p[3 * k + 1] = z[1] * sqrt(m.Hxx);
        p[3 * k + 2] = z[2] * sqrt(m.Hxx);
        for (int c = 0; c < 3; ++c) {
            q0[3 * k + c] = q[3 * k + c];
            g0[3 * k + c] = g[3 * k + c];
        }
    }
}

constexpr int kEnergyBlocks = 256;

// scalars[1] = sum (p^2/H + ln|H|)/2, scalars[2] = # stars outside the support, scalars[3] = prior potential
// (per-block partials, summed in block order by the last block)
__global__ void big_energy_kernel(const BigParams P, double g_ff2, int f_pos, int n, const double* q, const double* p,
                                  double* part /* [gridDim.x][4] */, unsigned int* ticket, double* scalars) {
    __shared__ double red[4 * 32];
    __shared__ bool is_last;
    double v[4] = {0, 0, 0, 0};
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const double f = q[3 * k], x = q[3 * k + 1], y = q[3 * k + 2];
        const Metric m = metric_of(P.F, f, g_ff2);
        const double pf = p[3 * k], px = p[3 * k + 1], py = p[3 * k + 2];
        v[0] += pf * pf / m.Hff + px * px / m.Hxx + py * py / m.Hxx;
        v[1] += log(fabs(m.Hff)) + 2.0 * log(fabs(m.Hxx));
        if (P.use_prior) v[2] += P.F.alpha * log(f) + P.F.Vpc;
        const bool bad = (f_pos && f < P.F.f_lim) || (x < -1.0) || (x > P.Rg + 1.0) || (y < -1.0) || (y > P.C + 1.0);
        v[3] += bad ? 1.0 : 0.0;
    }
    block_sum<4>(v, red);
    if (threadIdx.x == 0)
        for (int c = 0; c < 4; ++c) part[4 * blockIdx.x + c] = v[c];
    if (!last_block_ticket(ticket, &is_last)) return;
    double w[4] = {0, 0, 0, 0};
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x)
        for (int c = 0; c < 4; ++c) w[c] += __ldcg(part + 4 * b + c);
    block_sum<4>(w, red);
    if (threadIdx.x == 0) {
        scalars[1] = (w[0] + w[1]) / 2.0;
        scalars[2] = w[3];
        scalars[3] = w[2];
        *ticket = 0u;
    }
}

// E = V + T from the (all-reduced) scalars: slot 4 <- E (kept as E0 when `first`), accept test otherwise
__global__ void big_accept_kernel(int phase /*0: record E0, 1: accept*/, const double* scalars /* global sums */,
                                  const double* local_scalars, double* state,
                                  unsigned long long seed, int iter_host, const int* iter_dev, const double* lnu_in, int n,
                                  double* q, double* g,
                                  const double* q0, const double* g0, double* E_chain, double* V_chain, double* T_chain,
                                  unsigned char* A_chain) {
    // every thread evaluates the same scalars; thread 0 of block 0 writes the records
    const int iter = iter_dev ? *iter_dev : iter_host;
    const double V = (scalars[2] > 0.0) ? CUDART_INF : scalars[0] + scalars[3];
    const double T = scalars[1];
    const double E = V + T;
    if (phase == 0) {
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            state[0] = E;              // E0
            state[1] = local_scalars[0];  // this rank's pixel potential at the start (restored on rejection)
            if (E_chain) E_chain[iter] = E;
            if (V_chain) V_chain[iter] = V;
            if (T_chain) T_chain[iter] = T;
        }
        return;
    }
    const double dE = E - state[0];
    const double lnu = lnu_in ? lnu_in[iter] : philox_lnu(seed, 0u, (uint32_t)iter);
    const bool accept = (dE < 0.0) || (lnu < -dE);
    if (!accept) {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 3 * n; i += gridDim.x * blockDim.x) {
            q[i] = q0[i];
            g[i] = g0[i];
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (A_chain) A_chain[iter] = accept ? 1 : 0;
        state[2] = accept ? 1.0 : 0.0;
        state[3] += accept ? 1.0 : 0.0;
    }
}
// the pixel potential must follow the state on rejection: separate tiny kernel so that it runs after every block of
// big_accept_kernel has read scalars[0]
__global__ void big_restore_v_kernel(double* local_scalars, const double* state, int* iter_dev) {
    if (state[2] == 0.0) local_scalars[0] = state[1];
    if (iter_dev) *iter_dev += 1;  // the next replay of a captured iteration works on the next chain row
}

// boundary stars for the neighbours: list 0 = stars with x < lo_edge (for the rank below), list 1 = x >= hi_edge.
// Layout per list: [0] = count, then triples.  Order follows the star index (deterministic): block b owns the stars
// [b kPackChunk, (b+1) kPackChunk); a first kernel counts its matches, the second one starts at the sum of the counts of
// the blocks before it and compacts with warp ballots.
constexpr int kPackChunk = 1024;
static_assert(kPackChunk == 1 << 10, "big_qfix_kick_kernel counts boundary stars per chunk with k >> 10");

__global__ void big_pack_count_kernel(int n, const double* q, double lo_edge, double hi_edge, int2* counts) {
    __shared__ int c[2];
    if (threadIdx.x == 0) c[0] = c[1] = 0;
    __syncthreads();
    int lo = 0, hi = 0;
    const int k1 = min(n, (int)(blockIdx.x + 1) * kPackChunk);
    for (int k = blockIdx.x * kPackChunk + threadIdx.x; k < k1; k += blockDim.x) {
        const double x = q[3 * k + 1];
        lo += x < lo_edge;
        hi += x >= hi_edge;
    }
    if (lo) atomicAdd(&c[0], lo);
    if (hi) atomicAdd(&c[1], hi);
    __syncthreads();
    if (threadIdx.x == 0) counts[blockIdx.x] = make_int2(c[0], c[1]);
}

// the compaction of the ordered packing (big_pack_kernel, big_pack_xchg_kernel); the last block writes the two list lengths
__device__ __forceinline__ void pack_chunk(int n, const double* q, double lo_edge, double hi_edge, const int2* counts, double* send,
                                           int cap, int* err) {
    __shared__ int base[2];
    __shared__ int wcount[2][32];
    // exclusive prefix of the block counts
    int plo = 0, phi = 0;
    for (int b = threadIdx.x; b < (int)blockIdx.x; b += blockDim.x) {
        const int2 c = counts[b];
        plo += c.x;
        phi += c.y;
    }
    if (threadIdx.x == 0) base[0] = base[1] = 0;
    __syncthreads();
    if (plo) atomicAdd(&base[0], plo);
    if (phi) atomicAdd(&base[1], phi);
    __syncthreads();
    const int k_begin = blockIdx.x * kPackChunk, k_end = min(n, k_begin + kPackChunk);
    for (int k0 = k_begin; k0 < k_end; k0 += blockDim.x) {
        const int k = k0 + threadIdx.x;
        bool lo = false, hi = false;
        double f = 0, x = 0, y = 0;
        if (k < k_end) {
            f = q[3 * k]; x = q[3 * k + 1]; y = q[3 * k + 2];
            lo = x < lo_edge;
            hi = x >= hi_edge;
        }
        // block-wide ordered compaction: per-warp ballots + serial warp offsets
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
        const unsigned blo = __ballot_sync(0xffffffffu, lo), bhi = __ballot_sync(0xffffffffu, hi);
        if (lane == 0) { wcount[0][w] = __popc(blo); wcount[1][w] = __popc(bhi); }
        __syncthreads();
        int off_lo = base[0], off_hi = base[1];
        for (int i = 0; i < w; ++i) { off_lo += wcount[0][i]; off_hi += wcount[1][i]; }
        const unsigned lt = (1u << lane) - 1u;
        if (lo) {
            const int o = off_lo + __popc(blo & lt);
            if (o < cap) { double* d = send + 1 + 3 * (size_t)o; d[0] = f; d[1] = x; d[2] = y; } else atomicExch(err, 2);
        }
        if (hi) {
            const int o = off_hi + __popc(bhi & lt);
            if (o < cap) { double* d = send + (1 + 3 * (size_t)cap) + 1 + 3 * (size_t)o; d[0] = f; d[1] = x; d[2] = y; } else atomicExch(err, 2);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int i = 0; i < nw; ++i) { base[0] += wcount[0][i]; base[1] += wcount[1][i]; }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0 && blockIdx.x == gridDim.x - 1) {
        send[0] = (double)min(base[0], cap);
        send[1 + 3 * (size_t)cap] = (double)min(base[1], cap);
    }
}

__global__ void big_pack_kernel(int n, const double* q, double lo_edge, double hi_edge, const int2* counts, double* send, int cap,
                                int* err) {
    pack_chunk(n, q, lo_edge, hi_edge, counts, send, cap, err);
}

// all-reduce(sum) of n doubles (in -> out), summed in rank order on every rank
__global__ void big_xchg_small_kernel(const PeerPtrs peers, int rank, int world, int n, const double* din, double* dout,
                                      unsigned long long* epoch, int* err) {
    __shared__ int ok;
    const unsigned long long e = epoch[0] + 1;
    const int par = (int)(e & 1);
    const int t = threadIdx.x;
    if (t == 0) ok = 1;
    __syncthreads();
    if (t < world) {
        PeerSlot* s = &reinterpret_cast<PeerHeader*>(peers.box[t])->ar[par][rank];
        for (int k = 0; k < n; ++k) s->v[k] = din[k];
        peer_publish_tag(&s->tag, e);
        const PeerSlot* mine = &reinterpret_cast<const PeerHeader*>(peers.box[rank])->ar[par][t];
        if (!peer_wait_tag(&mine->tag, e, err)) ok = 0;
    }
    __syncthreads();
    if (t == 0) {
        const PeerHeader* h = reinterpret_cast<const PeerHeader*>(peers.box[rank]);
        if (ok) {
            for (int k = 0; k < n; ++k) {
                double acc = __ldcv(&h->ar[par][0].v[k]);
                for (int r = 1; r < world; ++r) acc += __ldcv(&h->ar[par][r].v[k]);
                dout[k] = acc;
            }
        }
        epoch[0] = e;
    }
}

// boundary-star lists straight into the neighbours' mailboxes, then the received lists into the local `recv` layout
// ([source rank][list][1 + 3 cap]) the evaluation reads: list 1 of rank-1 and list 0 of rank+1
__device__ void ghost_exchange_body(const PeerPtrs peers, int rank, int world, const double* send, double* recv, size_t list,
                                      unsigned long long* epoch, int* err, const BigParams P, int ntx, int n_own, int cap, int* tcnt,
                                      PairRec* tlist) {
    const unsigned long long e = epoch[1] + 1;
    const int par = (int)(e & 1);
    auto mailbox = [&](int r, int side) {
        return reinterpret_cast<double*>(peers.box[r] + sizeof(PeerHeader)) + ((size_t)par * 2 + side) * list;
    };
    auto tagof = [&](int r, int side) { return &reinterpret_cast<PeerHeader*>(peers.box[r])->gtag[par][side]; };
    // my list 0 (stars near my lower edge) -> side 1 of rank-1's box; my list 1 -> side 0 of rank+1's box
    for (int dir = 0; dir < 2; ++dir) {
        const int nb = dir == 0 ? rank - 1 : rank + 1;
        if (nb < 0 || nb >= world) continue;
        const double* src = send + (size_t)dir * list;
        double* dst = mailbox(nb, dir == 0 ? 1 : 0);
        const int cnt = 1 + 3 * (int)src[0];
        for (int k = threadIdx.x; k < cnt; k += blockDim.x) dst[k] = src[k];
    }
    __syncthreads();   // the block's payload stores precede the publishing threads' system-scope fence (cumulativity)
    if (threadIdx.x == 0 && rank > 0) peer_publish_tag(tagof(rank - 1, 1), e);
    if (threadIdx.x == 1 && rank < world - 1) peer_publish_tag(tagof(rank + 1, 0), e);
    __shared__ int ok;
    if (threadIdx.x == 0) ok = 1;
    __syncthreads();
    if (threadIdx.x == 0 && rank > 0 && !peer_wait_tag(tagof(rank, 0), e, err)) ok = 0;
    if (threadIdx.x == 1 && rank < world - 1 && !peer_wait_tag(tagof(rank, 1), e, err)) ok = 0;
    __syncthreads();
    for (int side = 0; side < 2; ++side) {
        const int nb = side == 0 ? rank - 1 : rank + 1;
        if (nb < 0 || nb >= world) continue;
        const double* src = mailbox(rank, side);
        double* dst = recv + ((size_t)nb * 2 + (side == 0 ? 1 : 0)) * list;
        const int cnt = ok ? 1 + 3 * (int)__ldcv(src) : 1;
        for (int k = threadIdx.x; k < cnt; k += blockDim.x) dst[k] = ok ? __ldcv(src + k) : 0.0;
    }
    __syncthreads();
    if (threadIdx.x == 0) epoch[1] = e;
    // the received ghosts go straight into the tile lists (what a separate binning kernel used to do before the evaluation)
    if (tcnt) {
        for (int side = 0; side < 2; ++side) {
            const int nb = side == 0 ? rank - 1 : rank + 1;
            if (nb < 0 || nb >= world) continue;
            const double* g = recv + ((size_t)nb * 2 + (side == 0 ? 1 : 0)) * list;
            const int ng = min((int)g[0], cap);
            for (int k = threadIdx.x; k < ng; k += blockDim.x)
                bin_star(P, ntx, n_own + side * cap + k, g[1 + 3 * k], g[2 + 3 * k], g[3 + 3 * k], false, tcnt, tlist, err);
        }
    }
}

// Ordered ghost packing, the exchange and the binning of the received ghosts in ONE kernel: every block compacts its chunk
// (as big_pack_kernel), the last block to finish runs the exchange body.  The chunk counts come from the position-update
// kernel (big_qfix_kick_kernel) and are zeroed here for the next step.
struct GhostX {
    PeerPtrs peers;
    int rank, world;
    double* recv;
    size_t list;
    unsigned long long* epoch;
    unsigned int* ticket;
    int ntx, n_own;
    int* tcnt;
    PairRec* tlist;
};

__global__ void big_pack_xchg_kernel(int n, const double* q, double lo_edge, double hi_edge, int2* counts, double* send, int cap,
                                     int* err, const BigParams P, const GhostX G) {
    __shared__ int s_last;
    pack_chunk(n, q, lo_edge, hi_edge, counts, send, cap, err);
    // last block out: every chunk (and the two list lengths) is in `send`
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(G.ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) counts[b] = make_int2(0, 0);   // for the next step's counting
    if (threadIdx.x == 0) *G.ticket = 0u;
    ghost_exchange_body(G.peers, G.rank, G.world, send, G.recv, G.list, G.epoch, err, P, G.ntx, G.n_own, cap, G.tcnt, G.tlist);
}

struct BBuf {
    void* ptr = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
        if (cudaMalloc(&ptr, bytes) != cudaSuccess) return bfail(SRHMC_ERR_CUDA, "cudaMalloc(%zu) failed", bytes);
        cap = bytes;
        return 0;
    }
    void release() { if (ptr) cudaFree(ptr); ptr = nullptr; cap = 0; }
    template <typename U> U* as() const { return reinterpret_cast<U*>(ptr); }
};

}  // namespace

struct srhmc_big {
    srhmc_big_config cfg;
    BigParams P;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    int n = 0;  // owned stars
    int sm_count = 0;
    int64_t launches = 0;
    BBuf D, L, q, p, g, a1, a2, q0, g0, gid, vpart, scalars, gscalars, state, counters, send, recv, err, normals, lnu, E, V, T, A;
    // fused tile evaluation (big_tile.cuh): tile grid over the local rows, per-tile star lists, per-star footprint partials
    BBuf tcnt, tlist, gpart;
    bool own_binned = false;
    // peer exchange (our own collectives over P2P / IPC mapped memory)
    BBuf peerbox, xepoch, packcnt, xticket;
    bool ghosts_binned = false;   // the ghost exchange kernel has already put the received ghosts into the tile lists
    // With peer exchange the kernel that produces a fixed-point count all-reduces it in its last block, the position-update
    // kernel counts the boundary stars, and packing + ghost exchange + ghost binning are one kernel: 5 kernels per leapfrog
    // step on N ranks.
    bool pack_counted = false;   // big_qfix_kick_kernel has left this step's chunk counts in packcnt
    PeerPtrs peers{};
    void* ipc_opened[kMaxWorld] = {};
    bool peer_enabled = false;  // the pair records of the owned stars' current positions are already in the tile lists
    BBuf epart, tickets;  // per-block energy partials; last-block tickets [0] energy, [1] tile potential
    int nty = 0, ntx = 0;
    bool use_tiles = false;
    int precision = 64;        // 32: gradient-only evaluations run the FP32 tile kernel on a float copy of the data
    BBuf D32;
    CUtensorMap tmapD32{};
    bool tma = false;          // a tensor map over the data window exists: the tile kernels load their tile by TMA
    bool L_filled = false;     // star-parallel path: the position-update kernel has already reset the model image
    int star_mode = -1;        // gradient-only FP64 evaluations by big_star_kernel: -1 = when the tile lists are short (sparse
                               // field), 0 = never, 1 = always (SRHMC_BIG_STAR)
    CUtensorMap tmapD{};
    int world = 1, rank = 0;
    bool have_data = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

namespace {

typedef CUresult (*TmapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D tensor map over a [nrows, cols] image of `elem_bytes`-wide pixels with kTile x kTile boxes (TMA tile loads)
bool encode_tile_map(CUtensorMap* map, void* base, int nrows, int cols, int elem_bytes) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
        qres != cudaDriverEntryPointSuccess) {
        cudaGetLastError();
        return false;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)nrows};
    const cuuint64_t strides[1] = {(cuuint64_t)cols * elem_bytes};
    const cuuint32_t box[2] = {(cuuint32_t)kTile, (cuuint32_t)kTile};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult cr = reinterpret_cast<TmapEncodeFn>(fn)(
        map, elem_bytes == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr,
        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return cr == CUDA_SUCCESS;
}

// float copy of the data window for the FP32 tile kernel (after every change of the FP64 data)
int refresh_float_data(srhmc_big* b) {
    if (b->precision != 32) return 0;
    const size_t npix = (size_t)b->cfg.nrows * b->cfg.cols;
    big_to_float_kernel<<<(int)std::min<size_t>((npix + 255) / 256, 8192), 256, 0, b->stream>>>(b->D.as<double>(), b->D32.as<float>(), npix);
    b->launches += 1;
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return bfail(SRHMC_ERR_CUDA, "float conversion of the data failed: %s", cudaGetErrorString(e));
    return 0;
}

}  // namespace

extern "C" {

const char* srhmc_big_last_error(void) { return g_big_err; }

int srhmc_big_create(const srhmc_big_config* cfg, srhmc_big** out) {
    if (!cfg || !out) return bfail(SRHMC_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->abi_version != SRHMC_ABI_VERSION) return bfail(SRHMC_ERR_INVALID, "ABI version mismatch");
    if (cfg->rows_global < 1 || cfg->cols < 1 || cfg->nrows < 1 || cfg->max_stars < 1)
        return bfail(SRHMC_ERR_INVALID, "rows_global, cols, nrows, max_stars must be >= 1");
    if (cfg->patch_radius < 1 || cfg->patch_radius > kMaxRad) return bfail(SRHMC_ERR_INVALID, "patch_radius must be 1..15");
    if (cfg->row0 < 0 || cfg->row0 + cfg->nrows > cfg->rows_global || cfg->own_lo < cfg->row0 ||
        cfg->own_hi > cfg->row0 + cfg->nrows || cfg->own_lo >= cfg->own_hi)
        return bfail(SRHMC_ERR_INVALID, "inconsistent row ranges");
    if (cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size) return bfail(SRHMC_ERR_INVALID, "bad rank / world_size");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return bfail(SRHMC_ERR_NO_DEVICE, "no CUDA device visible: this library has no CPU path");
    if (cfg->device < 0 || cfg->device >= ndev) return bfail(SRHMC_ERR_INVALID, "device out of range");
    BCU(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    BCU(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10) return bfail(SRHMC_ERR_NO_DEVICE, "device is sm_%d%d; the kernels are built for sm_100a only", prop.major, prop.minor);
    srhmc_big* b = new (std::nothrow) srhmc_big();
    if (!b) return bfail(SRHMC_ERR_INVALID, "out of host memory");
    b->cfg = *cfg;
    b->sm_count = prop.multiProcessorCount;
    b->world = cfg->world_size;
    b->rank = cfg->rank;
    BigParams& P = b->P;
    std::memset(&P, 0, sizeof(P));
    P.Rg = cfg->rows_global; P.C = cfg->cols; P.row0 = cfg->row0; P.nrows = cfg->nrows;
    P.own_lo = cfg->own_lo; P.own_hi = cfg->own_hi; P.rad = cfg->patch_radius; P.use_prior = cfg->use_prior ? 1 : 0;
    const double sigma = cfg->psf_fwhm_pix / 2.354;
    P.inv2s2 = 1.0 / (2.0 * sigma * sigma);
    P.inv_s2 = 1.0 / (sigma * sigma);
    P.norm = 1.0 / (M_PI * 2.0 * sigma * sigma);
    P.F.B = cfg->B_count; P.F.f_lim = cfg->f_lim; P.F.f_low = cfg->f_low;
    P.F.g0 = cfg->g0; P.F.g1 = cfg->g1; P.F.g2 = cfg->g2; P.F.g_xx = cfg->g_xx; P.F.g_ff = cfg->g_ff;
    P.F.alpha = cfg->alpha; P.F.Vpc = cfg->V_prior_const;
    const size_t npix = (size_t)cfg->nrows * cfg->cols, S = 3 * (size_t)cfg->max_stars;
    const size_t list = 1 + 3 * (size_t)std::max(1, cfg->max_ghosts);
    b->nty = (cfg->nrows + kTile - 1) / kTile;
    b->ntx = (cfg->cols + kTile - 1) / kTile;
    const size_t ntiles = (size_t)b->nty * b->ntx;
    // Path of the EVAL phases: the fused tile kernel needs enough tiles to fill the GPU; small dense fields keep the
    // star-parallel scatter/gather kernels.  SRHMC_BIG_PATH=tile|scatter overrides (read when the context is created).
    b->use_tiles = ntiles >= 2 * (size_t)b->sm_count;
    if (const char* e = std::getenv("SRHMC_BIG_STAR")) b->star_mode = std::atoi(e) > 0 ? 1 : 0;
    if (const char* e = std::getenv("SRHMC_BIG_PATH")) {
        if (!std::strcmp(e, "tile")) b->use_tiles = true;
        else if (!std::strcmp(e, "scatter")) b->use_tiles = false;
    }
    int rc = 0;
    rc |= b->D.ensure(npix * 8);
    if (!b->use_tiles) rc |= b->L.ensure(npix * 8);
    if (b->use_tiles) {
        // fixed-capacity pair lists (kTileMaxList records per tile: 32 KB of address space each, only the live records
        // are ever touched)
        rc |= b->tcnt.ensure(ntiles * 4);
        rc |= b->tlist.ensure(ntiles * (size_t)kTileMaxList * sizeof(PairRec)); rc |= b->gpart.ensure(12 * (size_t)cfg->max_stars * 8);
        if (!rc) cudaMemset(b->tcnt.ptr, 0, ntiles * 4);
        if (!rc && (cudaFuncSetAttribute(big_tile_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TileSmem)) != cudaSuccess ||
                    cudaFuncSetAttribute(big_tile_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TileSmem)) != cudaSuccess))
            rc = 1;
    }
    if (!rc && b->use_tiles) {
        // 2-D tensor map over the FP64 data window [nrows, C] with 64 x 64 boxes for the TMA tile loads
        // (global row stride must be a multiple of 16 bytes; otherwise, or without the driver's encoder, cp.async staging)
        if ((cfg->cols % 2) == 0) b->tma = encode_tile_map(&b->tmapD, b->D.ptr, cfg->nrows, cfg->cols, 8);
    }
    rc |= b->q.ensure(S * 8); rc |= b->p.ensure(S * 8); rc |= b->g.ensure(S * 8);
    rc |= b->a1.ensure(S * 8); rc |= b->a2.ensure(S * 8 + (size_t)cfg->max_stars * 4 + 8);
    rc |= b->q0.ensure(S * 8); rc |= b->g0.ensure(S * 8); rc |= b->gid.ensure((size_t)cfg->max_stars * 8);
    rc |= b->vpart.ensure(std::max<size_t>(kVBlocks, ntiles) * 8); rc |= b->scalars.ensure(kScalars * 8); rc |= b->gscalars.ensure(kScalars * 8); rc |= b->state.ensure(8 * 8);
    rc |= b->counters.ensure(4 * 4); rc |= b->err.ensure(4);
    rc |= b->epart.ensure(kEnergyBlocks * 4 * 8); rc |= b->tickets.ensure(2 * 4);
    rc |= b->packcnt.ensure(((size_t)cfg->max_stars / kPackChunk + 2) * sizeof(int2));
    rc |= b->send.ensure(2 * list * 8); rc |= b->recv.ensure((size_t)cfg->world_size * 2 * list * 8);
    if (rc) { srhmc_big_destroy(b); return SRHMC_ERR_CUDA; }
    cudaMemset(b->scalars.ptr, 0, kScalars * 8);
    cudaMemset(b->gscalars.ptr, 0, kScalars * 8);
    cudaMemset(b->state.ptr, 0, 64);
    cudaMemset(b->counters.ptr, 0, 16);
    cudaMemset(b->err.ptr, 0, 4);
    cudaMemset(b->tickets.ptr, 0, 8);
    cudaMemset(b->send.ptr, 0, 2 * list * 8);
    cudaMemset(b->recv.ptr, 0, (size_t)cfg->world_size * 2 * list * 8);
    if (cudaStreamCreateWithFlags(&b->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&b->ev0) != cudaSuccess || cudaEventCreate(&b->ev1) != cudaSuccess) {
        srhmc_big_destroy(b);
        return bfail(SRHMC_ERR_CUDA, "stream/event creation failed");
    }
    b->stream = b->own_stream;
    *out = b;
    return 0;
}

int srhmc_big_destroy(srhmc_big* b) {
    if (!b) return 0;
    cudaSetDevice(b->cfg.device);
    if (b->stream) cudaStreamSynchronize(b->stream);
    BBuf* all[] = {&b->D, &b->L, &b->q, &b->p, &b->g, &b->a1, &b->a2, &b->q0, &b->g0, &b->gid, &b->vpart, &b->scalars, &b->gscalars, &b->state,
                   &b->counters, &b->send, &b->recv, &b->err, &b->normals, &b->lnu, &b->E, &b->V, &b->T, &b->A,
                   &b->tcnt, &b->tlist, &b->gpart, &b->epart, &b->tickets, &b->xepoch, &b->packcnt, &b->xticket, &b->D32};
    for (BBuf* x : all) x->release();
    for (int r = 0; r < kMaxWorld; ++r)
        if (b->ipc_opened[r]) cudaIpcCloseMemHandle(b->ipc_opened[r]);
    b->peerbox.release();
    if (b->ev0) cudaEventDestroy(b->ev0);
    if (b->ev1) cudaEventDestroy(b->ev1);
    if (b->own_stream) cudaStreamDestroy(b->own_stream);
    delete b;
    return 0;
}

int srhmc_big_set_stream(srhmc_big* b, void* s) {
    if (!b) return bfail(SRHMC_ERR_INVALID, "null context");
    BCU(cudaSetDevice(b->cfg.device));
    BCU(cudaStreamSynchronize(b->stream));
    b->stream = reinterpret_cast<cudaStream_t>(s);  // NULL is the CUDA default stream (torch's default stream)
    return 0;
}

int srhmc_big_adopt_stream(srhmc_big* b, void* s) {
    // like srhmc_big_set_stream but without synchronising the previous stream (legal during CUDA-graph capture)
    if (!b) return bfail(SRHMC_ERR_INVALID, "null context");
    b->stream = reinterpret_cast<cudaStream_t>(s);
    return 0;
}

int srhmc_big_synchronize(srhmc_big* b) {
    if (!b) return bfail(SRHMC_ERR_INVALID, "null context");
    BCU(cudaSetDevice(b->cfg.device));
    BCU(cudaStreamSynchronize(b->stream));
    return 0;
}

int64_t srhmc_big_launch_count(srhmc_big* b) { return b ? b->launches : 0; }

int srhmc_big_set_data(srhmc_big* b, const double* D_local) {
    if (!b || !D_local) return bfail(SRHMC_ERR_INVALID, "null argument");
    BCU(cudaSetDevice(b->cfg.device));
    BCU(cudaMemcpyAsync(b->D.ptr, D_local, (size_t)b->cfg.nrows * b->cfg.cols * 8, cudaMemcpyHostToDevice, b->stream));
    if (int rc = refresh_float_data(b)) return rc;
    BCU(cudaStreamSynchronize(b->stream));
    b->have_data = true;
    return 0;
}

int srhmc_big_set_precision(srhmc_big* b, int32_t precision) {
    // 32: gradient-only evaluations through the FP32 tile kernel (float copy of the data, TMA); 64: everything FP64
    if (!b || (precision != 32 && precision != 64)) return bfail(SRHMC_ERR_INVALID, "precision must be 64 or 32");
    BCU(cudaSetDevice(b->cfg.device));
    if (precision == 32) {
        if (!b->use_tiles || !b->tma)
            return bfail(SRHMC_ERR_STATE, "the FP32 build needs the tile path with TMA (field of >= 2 tiles per SM, even column count)");
        const size_t npix = (size_t)b->cfg.nrows * b->cfg.cols;
        if (int rc = b->D32.ensure(npix * 4)) return rc;
        if (!encode_tile_map(&b->tmapD32, b->D32.ptr, b->cfg.nrows, b->cfg.cols, 4)) return bfail(SRHMC_ERR_CUDA, "cannot encode the FP32 tensor map");
        if (cudaFuncSetAttribute(big_tile32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TileSmemF)) != cudaSuccess)
            return bfail(SRHMC_ERR_CUDA, "cannot configure the FP32 tile kernel");
    }
    b->precision = precision;
    if (b->have_data)
        if (int rc = refresh_float_data(b)) return rc;
    BCU(cudaStreamSynchronize(b->stream));
    return 0;
}

int srhmc_big_mock_data(srhmc_big* b, const double* q_true, int32_t n, uint64_t seed, double* D_local_out) {
    // Device-side gen_mock_data (sampler_RHMC.py:77-99 + utils.poisson_realization, utils.py:488-496) for the local data
    // window: every rank passes the SAME truth list, renders the stars that touch its rows through the tile kernel (fixed
    // summation order) and Poisson-samples with the global pixel index as Philox counter, so overlapping halo rows agree
    // between ranks and with an untiled run bit for bit.
    if (!b || (n > 0 && !q_true) || n < 0) return bfail(SRHMC_ERR_INVALID, "bad argument");
    BCU(cudaSetDevice(b->cfg.device));
    cudaStream_t st = b->stream;
    const size_t ntiles = (size_t)b->nty * b->ntx;
    BBuf truth;
    if (int rc = truth.ensure((1 + 3 * (size_t)std::max(1, n)) * 8)) return rc;
    int rc = 0;
    rc |= b->tcnt.ensure(ntiles * 4);
    rc |= b->tlist.ensure(ntiles * (size_t)kTileMaxList * sizeof(PairRec));
    if (rc) { truth.release(); return SRHMC_ERR_CUDA; }
    if (cudaFuncSetAttribute(big_tile_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TileSmem)) != cudaSuccess) {
        truth.release();
        return bfail(SRHMC_ERR_CUDA, "cannot configure the tile kernel");
    }
    const double cnt = (double)n;
    cudaError_t e = cudaMemcpyAsync(truth.ptr, &cnt, 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(truth.as<double>() + 1, q_true, (size_t)n * 24, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(b->tcnt.ptr, 0, ntiles * 4, st);
    b->own_binned = false;
    if (e == cudaSuccess) {
        TileSrc S;
        S.q = nullptr; S.ga = truth.as<double>(); S.gb = nullptr; S.n_own = 0; S.cap = std::max(1, n);
        if (n)
            big_bin_kernel<<<std::max(1, std::min((n + 255) / 256, 8 * b->sm_count)), 256, 0, st>>>(
                b->P, S, b->ntx, 0, n, b->tcnt.as<int>(), b->tlist.as<PairRec>(), b->err.as<int>());
        big_tile_kernel<2><<<(int)ntiles, kTileThreads, sizeof(TileSmem), st>>>(b->P, S, b->ntx, nullptr, b->tcnt.as<int>(), b->tlist.as<PairRec>(),
                                                                                nullptr, nullptr, nullptr, nullptr, nullptr, b->D.as<double>(), seed,
                                                                                b->tmapD, 0);
        b->launches += 2;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && D_local_out)
        e = cudaMemcpyAsync(D_local_out, b->D.ptr, (size_t)b->cfg.nrows * b->cfg.cols * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && refresh_float_data(b) != 0) e = cudaErrorUnknown;
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    truth.release();
    if (e != cudaSuccess) return bfail(SRHMC_ERR_CUDA, "mock data generation failed: %s", cudaGetErrorString(e));
    int err = 0;
    BCU(cudaMemcpy(&err, b->err.ptr, 4, cudaMemcpyDeviceToHost));
    if (err == 3) {
        BCU(cudaMemset(b->err.ptr, 0, 4));
        return bfail(SRHMC_ERR_TOO_LARGE, "more than %d stars touch one 64x64 tile", kTileMaxList);
    }
    b->have_data = true;
    return 0;
}

int srhmc_big_set_stars(srhmc_big* b, const double* q, const int64_t* global_ids, int32_t n) {
    if (!b || (n > 0 && (!q || !global_ids))) return bfail(SRHMC_ERR_INVALID, "null argument");
    if (n < 0 || n > b->cfg.max_stars) return bfail(SRHMC_ERR_INVALID, "%d stars exceed max_stars = %d", n, b->cfg.max_stars);
    BCU(cudaSetDevice(b->cfg.device));
    if (n) {
        BCU(cudaMemcpyAsync(b->q.ptr, q, (size_t)n * 24, cudaMemcpyHostToDevice, b->stream));
        BCU(cudaMemcpyAsync(b->gid.ptr, global_ids, (size_t)n * 8, cudaMemcpyHostToDevice, b->stream));
    }
    BCU(cudaMemsetAsync(b->p.ptr, 0, 3 * (size_t)b->cfg.max_stars * 8, b->stream));
    if (b->own_binned || b->ghosts_binned) {  // records of the previous positions
        BCU(cudaMemsetAsync(b->tcnt.ptr, 0, (size_t)b->nty * b->ntx * 4, b->stream));
        b->own_binned = false;
        b->ghosts_binned = false;
    }
    if (b->pack_counted) {  // boundary counts of the previous positions
        BCU(cudaMemsetAsync(b->packcnt.ptr, 0, b->packcnt.cap, b->stream));
        b->pack_counted = false;
    }
    BCU(cudaStreamSynchronize(b->stream));
    b->n = n;
    return 0;
}

int srhmc_big_get_stars(srhmc_big* b, double* q, double* p, double* grad) {
    if (!b) return bfail(SRHMC_ERR_INVALID, "null context");
    BCU(cudaSetDevice(b->cfg.device));
    if (b->n) {
        if (q) BCU(cudaMemcpyAsync(q, b->q.ptr, (size_t)b->n * 24, cudaMemcpyDeviceToHost, b->stream));
        if (p) BCU(cudaMemcpyAsync(p, b->p.ptr, (size_t)b->n * 24, cudaMemcpyDeviceToHost, b->stream));
        if (grad) BCU(cudaMemcpyAsync(grad, b->g.ptr, (size_t)b->n * 24, cudaMemcpyDeviceToHost, b->stream));
    }
    BCU(cudaStreamSynchronize(b->stream));
    return 0;
}

int srhmc_big_set_momenta(srhmc_big* b, const double* p) {
    if (!b || !p) return bfail(SRHMC_ERR_INVALID, "null argument");
    BCU(cudaSetDevice(b->cfg.device));
    if (b->n) BCU(cudaMemcpyAsync(b->p.ptr, p, (size_t)b->n * 24, cudaMemcpyHostToDevice, b->stream));
    BCU(cudaStreamSynchronize(b->stream));
    return 0;
}

static size_t peer_box_bytes(const srhmc_big* b) {
    const size_t list = 1 + 3 * (size_t)std::max(1, b->cfg.max_ghosts);
    return sizeof(PeerHeader) + 4 * list * 8;
}

int srhmc_big_comm_export(srhmc_big* b, void* ipc_handle_64, void** raw_ptr) {
    if (!b) return bfail(SRHMC_ERR_INVALID, "null context");
    if (b->world > kMaxWorld) return bfail(SRHMC_ERR_INVALID, "peer exchange supports up to %d ranks", kMaxWorld);
    BCU(cudaSetDevice(b->cfg.device));
    if (!b->peerbox.ptr) {
        // a dedicated allocation: cudaIpcGetMemHandle exports the whole cudaMalloc block
        if (int rc = b->peerbox.ensure(peer_box_bytes(b))) return rc;
        if (int rc = b->xepoch.ensure(16)) return rc;
        if (int rc = b->xticket.ensure(16)) return rc;
        BCU(cudaMemset(b->peerbox.ptr, 0, peer_box_bytes(b)));
        BCU(cudaMemset(b->xepoch.ptr, 0, 16));
        BCU(cudaMemset(b->xticket.ptr, 0, 16));
    }
    if (ipc_handle_64) {
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
        cudaIpcMemHandle_t h;
        BCU(cudaIpcGetMemHandle(&h, b->peerbox.ptr));
        std::memcpy(ipc_handle_64, &h, 64);
    }
    if (raw_ptr) *raw_ptr = b->peerbox.ptr;
    return 0;
}

int srhmc_big_comm_import(srhmc_big* b, const void* ipc_handles, void* const* raw_ptrs) {
    if (!b || (!ipc_handles && !raw_ptrs)) return bfail(SRHMC_ERR_INVALID, "null argument");
    if (!b->peerbox.ptr) return bfail(SRHMC_ERR_STATE, "srhmc_big_comm_export has not been called");
    BCU(cudaSetDevice(b->cfg.device));
    for (int r = 0; r < b->world; ++r) {
        if (r == b->rank) {
            b->peers.box[r] = reinterpret_cast<unsigned char*>(b->peerbox.ptr);
        } else if (raw_ptrs) {
            // same process: plain device pointers.  A strip hosted on another device of this process needs peer access
            // enabled explicitly (the IPC path below gets it from cudaIpcMemLazyEnablePeerAccess).
            cudaPointerAttributes at;
            BCU(cudaPointerGetAttributes(&at, raw_ptrs[r]));
            if (at.type != cudaMemoryTypeDevice) return bfail(SRHMC_ERR_INVALID, "mailbox %d is not device memory", r);
            if (at.device != b->cfg.device) {
                int can = 0;
                BCU(cudaDeviceCanAccessPeer(&can, b->cfg.device, at.device));
                if (!can) return bfail(SRHMC_ERR_CUDA, "device %d cannot access the mailbox of rank %d on device %d", b->cfg.device, r, at.device);
                const cudaError_t pe = cudaDeviceEnablePeerAccess(at.device, 0);
                if (pe == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                else if (pe != cudaSuccess) return bfail(SRHMC_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d) failed: %s", at.device, cudaGetErrorString(pe));
            }
            b->peers.box[r] = reinterpret_cast<unsigned char*>(raw_ptrs[r]);
        } else {
            cudaIpcMemHandle_t h;
            std::memcpy(&h, reinterpret_cast<const unsigned char*>(ipc_handles) + 64 * (size_t)r, 64);
            void* p = nullptr;
            BCU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
            b->ipc_opened[r] = p;
            b->peers.box[r] = reinterpret_cast<unsigned char*>(p);
        }
    }
    b->peer_enabled = true;
    BCU(cudaMemset(b->packcnt.ptr, 0, b->packcnt.cap));
    return 0;
}

int srhmc_big_buffers(srhmc_big* b, srhmc_big_buffers_t* out) {
    if (!b || !out) return bfail(SRHMC_ERR_INVALID, "null argument");
    const size_t list = 1 + 3 * (size_t)std::max(1, b->cfg.max_ghosts);
    out->ghost_send = b->send.ptr;
    out->ghost_send_doubles = (int64_t)(2 * list);
    out->ghost_recv = b->recv.ptr;
    out->ghost_recv_doubles = (int64_t)((size_t)b->world * 2 * list);
    out->scalars = b->scalars.ptr;
    out->global_scalars = b->gscalars.ptr;
    out->n_scalars = kScalars;
    out->counters = b->counters.ptr;
    out->n_counters = 4;
    return 0;
}

int srhmc_big_set_draws(srhmc_big* b, const double* normals, const double* lnu, int32_t n_iters) {
    // normals [n_iters, n, 3] for the owned stars (parity mode) and lnu [n_iters]; either may be NULL (device Philox)
    if (!b || n_iters < 0) return bfail(SRHMC_ERR_INVALID, "bad argument");
    BCU(cudaSetDevice(b->cfg.device));
    b->normals.release();
    b->lnu.release();
    if (normals && b->n && n_iters) {
        if (int rc = b->normals.ensure((size_t)n_iters * b->n * 24)) return rc;
        BCU(cudaMemcpyAsync(b->normals.ptr, normals, (size_t)n_iters * b->n * 24, cudaMemcpyHostToDevice, b->stream));
    }
    if (lnu && n_iters) {
        if (int rc = b->lnu.ensure((size_t)n_iters * 8)) return rc;
        BCU(cudaMemcpyAsync(b->lnu.ptr, lnu, (size_t)n_iters * 8, cudaMemcpyHostToDevice, b->stream));
    }
    BCU(cudaStreamSynchronize(b->stream));
    return 0;
}

int srhmc_big_alloc_chains(srhmc_big* b, int32_t n_iters) {
    if (!b || n_iters < 1) return bfail(SRHMC_ERR_INVALID, "bad argument");
    BCU(cudaSetDevice(b->cfg.device));
    if (int rc = b->E.ensure((size_t)n_iters * 8)) return rc;
    if (int rc = b->V.ensure((size_t)n_iters * 8)) return rc;
    if (int rc = b->T.ensure((size_t)n_iters * 8)) return rc;
    if (int rc = b->A.ensure((size_t)n_iters)) return rc;
    BCU(cudaMemsetAsync(b->E.ptr, 0, (size_t)n_iters * 8, b->stream));
    BCU(cudaMemsetAsync(b->V.ptr, 0, (size_t)n_iters * 8, b->stream));
    BCU(cudaMemsetAsync(b->T.ptr, 0, (size_t)n_iters * 8, b->stream));
    BCU(cudaMemsetAsync(b->A.ptr, 0, (size_t)n_iters, b->stream));
    BCU(cudaMemsetAsync(b->state.ptr, 0, 64, b->stream));
    return 0;
}

int srhmc_big_read_chains(srhmc_big* b, int32_t n_iters, double* E, double* V, double* T, uint8_t* A, double* n_accepted,
                          int32_t* error_flag) {
    if (!b) return bfail(SRHMC_ERR_INVALID, "null context");
    BCU(cudaSetDevice(b->cfg.device));
    if (E) BCU(cudaMemcpyAsync(E, b->E.ptr, (size_t)n_iters * 8, cudaMemcpyDeviceToHost, b->stream));
    if (V) BCU(cudaMemcpyAsync(V, b->V.ptr, (size_t)n_iters * 8, cudaMemcpyDeviceToHost, b->stream));
    if (T) BCU(cudaMemcpyAsync(T, b->T.ptr, (size_t)n_iters * 8, cudaMemcpyDeviceToHost, b->stream));
    if (A) BCU(cudaMemcpyAsync(A, b->A.ptr, (size_t)n_iters, cudaMemcpyDeviceToHost, b->stream));
    double st[8] = {0};
    int err = 0;
    BCU(cudaMemcpyAsync(st, b->state.ptr, 64, cudaMemcpyDeviceToHost, b->stream));
    BCU(cudaMemcpyAsync(&err, b->err.ptr, 4, cudaMemcpyDeviceToHost, b->stream));
    BCU(cudaStreamSynchronize(b->stream));
    if (n_accepted) *n_accepted = st[3];
    if (error_flag) *error_flag = err;
    return 0;
}

int srhmc_big_read_scalars(srhmc_big* b, double* scalars /* [8] local partial sums */) {
    if (!b || !scalars) return bfail(SRHMC_ERR_INVALID, "null argument");
    BCU(cudaSetDevice(b->cfg.device));
    BCU(cudaMemcpyAsync(scalars, b->scalars.ptr, kScalars * 8, cudaMemcpyDeviceToHost, b->stream));
    BCU(cudaStreamSynchronize(b->stream));
    return 0;
}

// Enqueue one phase on the context's stream (no synchronisation).  See srhmc_big_phase_id in the header.
int srhmc_big_phase(srhmc_big* b, int32_t phase, const srhmc_big_step* s) {
    if (!b || !s) return bfail(SRHMC_ERR_INVALID, "null argument");
    if (!b->have_data) return bfail(SRHMC_ERR_STATE, "srhmc_big_set_data has not been called");
    BCU(cudaSetDevice(b->cfg.device));
    const BigParams& P = b->P;
    const int n = b->n;
    BigStep S;
    S.h = s->dt / 2.0; S.delta = s->delta; S.g_ff2 = s->g_ff2; S.counter_max = s->counter_max;
    S.per_star = s->fixed_point_mode != 0 ? 1 : 0;
    S.K.c = (P.F.B / P.F.g0) / P.F.g_ff; S.K.ig2 = 1.0 / s->g_ff2; S.K.ig1 = 1.0 / P.F.g1; S.K.Bg2 = P.F.B / P.F.g2;
    S.K.igxx = 1.0 / P.F.g_xx; S.K.f_low = P.F.f_low;   // make_metric_k (common.cuh) on the host
    const int tb = 128, gs = std::max(1, std::min((n + tb - 1) / tb, 4 * b->sm_count));
    const size_t npix = (size_t)P.nrows * P.C;
    const size_t list = 1 + 3 * (size_t)std::max(1, b->cfg.max_ghosts);
    int* cnt = b->counters.as<int>();
    cudaStream_t st = b->stream;
    PeerX X;
    std::memset(&X, 0, sizeof(X));
    const bool peer_multi = b->peer_enabled && b->world > 1;
    if (peer_multi) {
        X.peers = b->peers; X.rank = b->rank; X.world = b->world;
        X.prod = 1;
        X.epoch = b->xepoch.as<unsigned long long>(); X.ticket = b->xticket.as<unsigned int>(); X.err = b->err.as<int>();
    }
    // per-star stop rule: the whole advance between two evaluations in one kernel (big_perstar_kernel)
    auto launch_perstar = [&](bool from_eval, const double* gpart_in) -> int {
        if (b->use_tiles && (b->own_binned || b->ghosts_binned)) {  // records nobody consumed
            BCU(cudaMemsetAsync(b->tcnt.ptr, 0, (size_t)b->nty * b->ntx * 4, st));
            b->ghosts_binned = false;
        }
        if (peer_multi && b->pack_counted) BCU(cudaMemsetAsync(b->packcnt.ptr, 0, b->packcnt.cap, st));
        const double reach_k = (double)(b->cfg.nrows_halo + P.rad + 1);
        const double lo_edge_k = (b->rank > 0) ? (double)P.own_lo + reach_k : -1e300;
        const double hi_edge_k = (b->rank < b->world - 1) ? (double)P.own_hi - reach_k : 1e300;
        int* tc = b->use_tiles ? b->tcnt.as<int>() : nullptr;
        PairRec* tl = b->use_tiles ? b->tlist.as<PairRec>() : nullptr;
        int2* pc = peer_multi ? b->packcnt.as<int2>() : nullptr;
        double* lf = (!b->use_tiles && n > 0) ? b->L.as<double>() : nullptr;
        if (from_eval)
            big_perstar_kernel<true><<<gs, tb, 0, st>>>(P, S, n, b->q.as<double>(), b->p.as<double>(), b->g.as<double>(), gpart_in,
                                                        b->ntx, tc, tl, b->err.as<int>(), pc, lo_edge_k, hi_edge_k, lf, npix);
        else
            big_perstar_kernel<false><<<gs, tb, 0, st>>>(P, S, n, b->q.as<double>(), b->p.as<double>(), b->g.as<double>(), nullptr,
                                                         b->ntx, tc, tl, b->err.as<int>(), pc, lo_edge_k, hi_edge_k, lf, npix);
        b->L_filled = lf != nullptr;
        b->pack_counted = peer_multi;
        b->own_binned = b->use_tiles;
        b->launches += 1;
        return 0;
    };
    switch (phase) {
        case SRHMC_BIG_PS_ADVANCE:
            if (int rc = launch_perstar(false, nullptr)) return rc;
            break;
        case SRHMC_BIG_PACK: {
            // boundary lists for the neighbours: everything that can touch their data rows
            const double reach = (double)(b->cfg.nrows_halo + P.rad + 1);
            const double lo_edge = (b->rank > 0) ? (double)P.own_lo + reach : -1e300;
            const double hi_edge = (b->rank < b->world - 1) ? (double)P.own_hi - reach : 1e300;
            const int pb = std::max(1, (n + kPackChunk - 1) / kPackChunk);
            if (peer_multi) {
                if (!b->pack_counted) {   // a PACK that does not follow a position update (first evaluation of a run)
                    big_pack_count_kernel<<<pb, 256, 0, st>>>(n, b->q.as<double>(), lo_edge, hi_edge, b->packcnt.as<int2>());
                    b->launches += 1;
                }
                GhostX G;
                G.peers = b->peers; G.rank = b->rank; G.world = b->world; G.recv = b->recv.as<double>(); G.list = list;
                G.epoch = b->xepoch.as<unsigned long long>(); G.ticket = b->xticket.as<unsigned int>() + 1;
                G.ntx = b->ntx; G.n_own = n;
                G.tcnt = b->use_tiles ? b->tcnt.as<int>() : nullptr;
                G.tlist = b->use_tiles ? b->tlist.as<PairRec>() : nullptr;
                big_pack_xchg_kernel<<<pb, 256, 0, st>>>(n, b->q.as<double>(), lo_edge, hi_edge, b->packcnt.as<int2>(), b->send.as<double>(),
                                                         std::max(1, b->cfg.max_ghosts), b->err.as<int>(), P, G);
                b->ghosts_binned = b->use_tiles;
                b->pack_counted = false;
                b->launches += 1;
                break;
            }
            big_pack_count_kernel<<<pb, 256, 0, st>>>(n, b->q.as<double>(), lo_edge, hi_edge, b->packcnt.as<int2>());
            big_pack_kernel<<<pb, 256, 0, st>>>(n, b->q.as<double>(), lo_edge, hi_edge, b->packcnt.as<int2>(), b->send.as<double>(),
                                                 std::max(1, b->cfg.max_ghosts), b->err.as<int>());
            b->launches += 2;
            break;
        }
        case SRHMC_BIG_EVAL:
        case SRHMC_BIG_EVAL_V:
        case SRHMC_BIG_EVAL_KICK2:
        case SRHMC_BIG_EVAL_V_KICK2:
        case SRHMC_BIG_EVAL_KICK2_KICK1:
        case SRHMC_BIG_EVAL_PS_ADVANCE: {
            const int want_V = (phase == SRHMC_BIG_EVAL_V || phase == SRHMC_BIG_EVAL_V_KICK2) ? 1 : 0;
            // tail: 0 none, 1 the step's last half kick + reflections, 2 also the next step's first kick + p fixed point A,
            // 3 (per-star stop rule) the step's end and the whole advance of the next step in one kernel
            const int tail = phase == SRHMC_BIG_EVAL_PS_ADVANCE ? 3 : (phase == SRHMC_BIG_EVAL_KICK2_KICK1 ? 2 :
                             ((phase == SRHMC_BIG_EVAL_KICK2 || phase == SRHMC_BIG_EVAL_V_KICK2) ? 1 : 0));
            const double* ga = (b->world > 1 && b->rank > 0) ? b->recv.as<double>() + ((size_t)(b->rank - 1) * 2 + 1) * list : nullptr;
            const double* gb = (b->world > 1 && b->rank < b->world - 1) ? b->recv.as<double>() + ((size_t)(b->rank + 1) * 2 + 0) * list : nullptr;
            const double* gpart = nullptr;
            if (b->use_tiles) {
                TileSrc S;
                S.q = b->q.as<double>(); S.ga = ga; S.gb = gb; S.n_own = n; S.cap = std::max(1, b->cfg.max_ghosts);
                const int ntiles = b->nty * b->ntx;
                if (!b->own_binned && n > 0) {
                    big_bin_kernel<<<std::max(1, std::min((n + 255) / 256, 8 * b->sm_count)), 256, 0, st>>>(
                        P, S, b->ntx, 0, n, b->tcnt.as<int>(), b->tlist.as<PairRec>(), b->err.as<int>());
                    b->launches += 1;
                }
                if ((ga || gb) && !b->ghosts_binned) {
                    big_bin_kernel<<<std::max(1, std::min((2 * S.cap + 255) / 256, 8 * b->sm_count)), 256, 0, st>>>(
                        P, S, b->ntx, n, n + 2 * S.cap, b->tcnt.as<int>(), b->tlist.as<PairRec>(), b->err.as<int>());
                    b->launches += 1;
                }
                b->own_binned = false;  // the tile kernel consumes the lists and re-zeroes the counters
                b->ghosts_binned = false;
                if (b->precision == 32 && !want_V) {
                    big_tile32_kernel<<<ntiles, kTileThreads, sizeof(TileSmemF), st>>>(P, S, b->ntx, b->tcnt.as<int>(), b->tlist.as<PairRec>(),
                                                                                       b->gpart.as<double>(), cnt, b->tmapD32);
                } else if (!want_V && n > 0 && P.rad <= 15 &&
                           (b->star_mode == 1 || (b->star_mode < 0 && 2.0 * n <= 3.0 * ntiles))) {
                    // very sparse field (mean tile list below ~1.5 records): one warp per owned star, neighbours from the tile lists
                    // (big_star.cuh: only the patches are read, not every pixel); the lists are
                    // consumed here, so their counters are re-zeroed by a memset node instead of by the tile CTAs
                    const int sgrid = std::max(1, std::min((n + kStarWarps - 1) / kStarWarps, 64 * b->sm_count));
                    if (P.rad <= 12)
                        big_star_kernel<25><<<sgrid, 32 * kStarWarps, 0, st>>>(P, n, b->q.as<double>(), b->D.as<double>(), b->ntx,
                                                                               b->tcnt.as<int>(), b->tlist.as<PairRec>(), b->gpart.as<double>(), cnt);
                    else
                        big_star_kernel<31><<<sgrid, 32 * kStarWarps, 0, st>>>(P, n, b->q.as<double>(), b->D.as<double>(), b->ntx,
                                                                               b->tcnt.as<int>(), b->tlist.as<PairRec>(), b->gpart.as<double>(), cnt);
                    BCU(cudaMemsetAsync(b->tcnt.ptr, 0, (size_t)ntiles * 4, st));
                } else if (want_V)
                    big_tile_kernel<1><<<ntiles, kTileThreads, sizeof(TileSmem), st>>>(P, S, b->ntx, b->D.as<double>(), b->tcnt.as<int>(),
                        b->tlist.as<PairRec>(), b->gpart.as<double>(), b->vpart.as<double>(),
                        b->tickets.as<unsigned int>() + 1, b->scalars.as<double>(), cnt, nullptr, 0ull, b->tmapD, b->tma ? 1 : 0);
                else
                    big_tile_kernel<0><<<ntiles, kTileThreads, sizeof(TileSmem), st>>>(P, S, b->ntx, b->D.as<double>(), b->tcnt.as<int>(),
                        b->tlist.as<PairRec>(), b->gpart.as<double>(), b->vpart.as<double>(),
                        b->tickets.as<unsigned int>() + 1, b->scalars.as<double>(), cnt, nullptr, 0ull, b->tmapD, b->tma ? 1 : 0);
                b->launches += 1;
                if (tail == 0) {
                    big_gsum_kernel<<<gs, tb, 0, st>>>(P, b->q.as<double>(), n, b->gpart.as<double>(), b->g.as<double>());
                    b->launches += 1;
                }
                gpart = b->gpart.as<double>();
            } else {
                const int pg = (int)std::min<size_t>((npix + 255) / 256, (size_t)kVBlocks);
                if (!b->L_filled) {
                    big_fill_kernel<<<pg, 256, 0, st>>>(b->L.as<double>(), npix, P.F.B);
                    b->launches += 1;
                }
                b->L_filled = false;
                const int total = n + 2 * std::max(1, b->cfg.max_ghosts);
                const int sg = std::max(1, std::min((total * 32 + 255) / 256, 16 * b->sm_count));
                big_scatter_kernel<<<sg, 256, 0, st>>>(P, b->q.as<double>(), n, ga, gb, b->L.as<double>(), b->err.as<int>());
                big_pixel_kernel<<<pg, 256, 0, st>>>(P, b->D.as<double>(), b->L.as<double>(), want_V, b->vpart.as<double>());
                if (want_V) big_vsum_kernel<<<1, 256, 0, st>>>(b->vpart.as<double>(), pg, b->scalars.as<double>());
                const int gg = std::max(1, std::min((n * 32 + 255) / 256, 16 * b->sm_count));
                big_gather_kernel<<<gg, 256, 0, st>>>(P, b->q.as<double>(), n, b->L.as<double>(), b->g.as<double>());
                b->launches += want_V ? 4 : 3;
                if (tail == 2) BCU(cudaMemsetAsync(cnt, 0, 8, st));  // the tile kernel does this on the tile path
            }
            if (tail == 1)
                big_tail_kernel<false><<<gs, tb, 0, st>>>(P, S, n, b->q.as<double>(), b->p.as<double>(), b->g.as<double>(), gpart,
                                                          b->a1.as<double>(), b->a2.as<double>(), cnt, X);
            else if (tail == 2)
                big_tail_kernel<true><<<gs, tb, 0, st>>>(P, S, n, b->q.as<double>(), b->p.as<double>(), b->g.as<double>(), gpart,
                                                         b->a1.as<double>(), b->a2.as<double>(), cnt, X);
            else if (tail == 3) {
                if (int rc = launch_perstar(true, gpart)) return rc;
            }
            if (tail == 1 || tail == 2) b->launches += 1;
            break;
        }
        case SRHMC_BIG_RESET_ITER:
            BCU(cudaMemsetAsync(cnt + 2, 0, 4, st));
            break;
        case SRHMC_BIG_KICK1:
            BCU(cudaMemsetAsync(cnt, 0, 8, st));
            big_kick1_kernel<<<gs, tb, 0, st>>>(P, S, n, b->q.as<double>(), b->p.as<double>(), b->g.as<double>(),
                                                b->a1.as<double>(), b->a2.as<double>(), cnt, X);
            b->launches += 1;
            break;
        case SRHMC_BIG_PFIX_QFIX:
            // tiled over peers: the field-wide maximum of the p fixed-point counts was all-reduced by the last block of the
            // kernel that produced it
            big_pfix_qfix_kernel<<<gs, tb, 0, st>>>(P, S, n, b->q.as<double>(), b->p.as<double>(), b->a1.as<double>(),
                                                    b->a2.as<double>(), cnt, cnt + 1, X);
            b->launches += 1;
            break;
        case SRHMC_BIG_QFIX_KICK: {
            if (b->use_tiles && (b->own_binned || b->ghosts_binned)) {  // records nobody consumed (two position updates without an evaluation)
                BCU(cudaMemsetAsync(b->tcnt.ptr, 0, (size_t)b->nty * b->ntx * 4, st));
                b->ghosts_binned = false;
            }
            if (peer_multi && b->pack_counted)   // counts nobody consumed (two position updates without a PACK)
                BCU(cudaMemsetAsync(b->packcnt.ptr, 0, b->packcnt.cap, st));
            const double reach_k = (double)(b->cfg.nrows_halo + P.rad + 1);
            const double lo_edge_k = (b->rank > 0) ? (double)P.own_lo + reach_k : -1e300;
            const double hi_edge_k = (b->rank < b->world - 1) ? (double)P.own_hi - reach_k : 1e300;
            big_qfix_kick_kernel<<<gs, tb, 0, st>>>(P, S, n, b->q.as<double>(), b->p.as<double>(), b->a1.as<double>(),
                                                    b->a2.as<double>(), cnt + 1, b->ntx, b->use_tiles ? b->tcnt.as<int>() : nullptr,
                                                    b->use_tiles ? b->tlist.as<PairRec>() : nullptr, b->err.as<int>(),
                                                    peer_multi ? b->packcnt.as<int2>() : nullptr, lo_edge_k, hi_edge_k,
                                                    (!b->use_tiles && n > 0) ? b->L.as<double>() : nullptr, npix);
            b->L_filled = !b->use_tiles && n > 0;
            b->pack_counted = peer_multi;
            b->own_binned = b->use_tiles;
            b->launches += 1;
            break;
        }
        case SRHMC_BIG_KICK2:
            big_kick2_kernel<<<gs, tb, 0, st>>>(P, S, n, b->q.as<double>(), b->p.as<double>(), b->g.as<double>());
            b->launches += 1;
            break;
        case SRHMC_BIG_MOMENTUM: {
            const double* z = b->normals.ptr ? b->normals.as<double>() : nullptr;
            big_momentum_kernel<<<gs, tb, 0, st>>>(P, s->g_ff2, n, b->q.as<double>(), b->p.as<double>(), b->g.as<double>(),
                                                   b->q0.as<double>(), b->g0.as<double>(), b->gid.as<long long>(), s->seed,
                                                   s->iteration, s->iteration < 0 ? cnt + 2 : nullptr, z);
            b->launches += 1;
            break;
        }
        case SRHMC_BIG_ENERGY:
            big_energy_kernel<<<std::max(1, std::min((n + 255) / 256, kEnergyBlocks)), 256, 0, st>>>(
                P, s->g_ff2, s->f_pos, n, b->q.as<double>(), b->p.as<double>(), b->epart.as<double>(),
                b->tickets.as<unsigned int>(), b->scalars.as<double>());
            b->launches += 1;
            break;
        case SRHMC_BIG_RECORD_E0:
        case SRHMC_BIG_ACCEPT: {
            const int ph = phase == SRHMC_BIG_ACCEPT ? 1 : 0;
            // single rank: the global sums are the local ones; otherwise the caller has all-reduced `scalars` into
            // `global_scalars` on this stream before this phase
            if (b->world == 1) {
                BCU(cudaMemcpyAsync(b->gscalars.ptr, b->scalars.ptr, kScalars * 8, cudaMemcpyDeviceToDevice, st));
            } else if (b->peer_enabled) {  // sum of the energy partials over the ranks, in rank order on every rank
                big_xchg_small_kernel<<<1, 32, 0, st>>>(b->peers, b->rank, b->world, kScalars, b->scalars.as<double>(),
                                                        b->gscalars.as<double>(), b->xepoch.as<unsigned long long>(), b->err.as<int>());
                b->launches += 1;
            }
            big_accept_kernel<<<gs, tb, 0, st>>>(ph, b->gscalars.as<double>(), b->scalars.as<double>(), b->state.as<double>(), s->seed, s->iteration,
                                                 s->iteration < 0 ? cnt + 2 : nullptr,
                                                 b->lnu.ptr ? b->lnu.as<double>() : nullptr, n, b->q.as<double>(),
                                                 b->g.as<double>(), b->q0.as<double>(), b->g0.as<double>(),
                                                 b->E.ptr ? b->E.as<double>() : nullptr, b->V.ptr ? b->V.as<double>() : nullptr,
                                                 b->T.ptr ? b->T.as<double>() : nullptr,
                                                 b->A.ptr ? b->A.as<unsigned char>() : nullptr);
            if (ph == 1)
                big_restore_v_kernel<<<1, 1, 0, st>>>(b->scalars.as<double>(), b->state.as<double>(),
                                                      s->iteration < 0 ? cnt + 2 : nullptr);
            b->launches += 1 + ph;
            break;
        }
        default:
            return bfail(SRHMC_ERR_INVALID, "unknown phase %d", phase);
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return bfail(SRHMC_ERR_CUDA, "phase %d launch failed: %s", phase, cudaGetErrorString(e));
    return 0;
}

}  // extern "C"
