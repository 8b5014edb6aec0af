// Shared device helpers for the sm_100a RHMC kernels: parameter blocks, the metric of the reference
// (sampler_RHMC.py:229-292), fast FP64 reciprocal, deterministic reductions and a Philox4x32-10 generator.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace srhmc {

constexpr int kWarp = 32;
// Lanes per chain of the one-star kernel.  Measured on the headline workload: 16 lanes 734, 8 lanes 1104, 4 lanes
// 1210 M star-steps/s -- fewer lanes replicate the per-chain scalar work and the table exponentials less; 2 lanes
// would need more than 255 registers.
constexpr int kChainLPC = 4;
constexpr int kChainGroup = 32 / kChainLPC;   // chains per warp: the unit of its work scheduler

// Shared-memory layout of one single-warp block of the one-star kernel (chain_layout, chain_kernel.cuh); byte offsets are
// from the start of the block's dynamic shared memory.
struct ChainLayout {
    size_t log_bytes;   // log table at offset 0
    size_t img_elems;   // elements of one chain image (R rows of kChainCS, plus the bank padding)
    size_t img_bytes;   // stride of the chain images, which start at log_bytes
    size_t tab_base;    // row table of chain 0
    size_t tab_bytes;   // stride of the row tables (a multiple of 16)
    size_t smem_bytes;  // the whole block
};

// Problem constants snapshot (host fills it from srhmc_config).
struct FieldParams {
    int R, C;          // image rows / cols
    int Nmax;          // star slots per field
    int Kc;            // stars per table chunk
    int rad;           // PSF truncation radius in pixels, 0 = full image
    int sx, sy;        // table strides (rows / cols rounded up to the warp-tile)
    int fp_mode;       // 0 parity (field-wide stop rule), 1 per-star
    int D_shared;      // all fields read image 0
    int use_prior, use_Vc, vc_int;  // vc_int: Vc_r_pow as small non-negative integer, or -1
    int hess;          // shared memory holds a second image for the Hessian path
    // compact-table evaluation of the CTA-per-field kernel (field_kernel.cuh, "v3"): every star keeps a TL-row table of
    // {ex, ex dx} pairs and a (TL+1)-column table of f ey over a window clamped inside the image, so that all stars of a
    // crowded field fit one table build and the gradient pass needs no bounds handling
    int v3;            // 1: enabled (patch-limited PSF, rad <= 12, C even (FP64) / C % 4 == 0 (FP32), R >= TL, C >= TL+1, all tables fit)
    int tl;            // TL = 2 rad + 1
    int rs, cs;        // strides: row table in pairs (odd: conflict-free 16-byte stores), column table in entries (odd)
    double inv2s2;     // 1/(2 sigma^2)
    double inv_s2;     // 1/sigma^2
    double norm;       // 1/(2 pi sigma^2)
    double c2;         // exp(-1/sigma^2): second-order ratio of the Gaussian recurrence
    double B, f_lim, f_low;
    double lnB, invB;  // ln(B), 1/B (chain kernel's separable potential)
    double cL, cLh;    // exp(-L^2/sigma^2) and its square root for the chain kernel's stride-L Gaussian recurrences
                       // (L = lanes per chain, kChainLPC)
    double wcut;       // |i + .5 - x| beyond which exp(-(..)^2/2 sigma^2) < 2^-46
    double g0, g1, g2, g_xx, g_ff;
    double alpha, Vpc, vc_pow;
};

enum Mode : int { MODE_EVAL = 0, MODE_STEP = 1, MODE_RUN = 2, MODE_SINGLE = 3, MODE_RUN_RJ = 4 };
// samplers.lightsource_gym family (ls_kernel.cuh)
enum LsVariant : int { LS_HMC = 0, LS_DIAG = 1, LS_HESS = 2, LS_TRIAL = 3, LS_EVAL_HESS = 4, LS_EVAL_BG = 5 };

struct LsArgs {
    int variant, n_fields, niter;
    const void* D;
    const int* nstars;
    const double* q0;        // [F,S]
    const double* p0;        // [F,S] (LS_EVAL_HESS) or nullptr
    const double* dt;        // [S] per-coordinate steps (LS_HMC, LS_HESS, LS_TRIAL: [3]); LS_DIAG: dt[0] = dt_global
    double f_lim, factor1;
    const double* normals;   // [F, niter+1, S]
    const int* steps;        // [F, niter]
    const double* lnu;       // [F, niter]
    const double* background;  // [F,R,C] (LS_TRIAL) or nullptr
    int zero_xy;             // LS_TRIAL: zero the position momenta (flux-only tuning pass)
    double* q_chain;         // [F, niter+1, S]
    double* E_chain;         // [F, niter+1]
    double* dE_chain;        // [F, niter+1]
    unsigned char* A_chain;  // [F, niter]
    double* q_final;         // [F,S]
    double* accept_count;    // [F]
    // LS_EVAL_HESS outputs
    double* d1; double* d2; double* d3;   // [F,S] dV/dq, d2V/dq2, d3V/dq3 (diagonal)
    double* dqdt; double* dpdt;           // [F,S]
    double* E_out;                        // [F]
    int d2_only;
};

// Per-launch arguments (device pointers).
struct LaunchArgs {
    int mode;
    int n_fields;
    int field_begin, field_end;  // chain kernel: this launch covers fields [field_begin, field_end) (0, 0 = all);
                                 // field_begin is a multiple of the warp group size
    const void* D;          // [n_images, R*C] in the pixel type
    const void* D_int;      // same images as exact unsigned integer counts, or nullptr (chain kernel, lossless)
    int D_int_bytes;        // 4: uint32, 2: uint16 (every count < 65536)
    int pix_f32;            // chain kernel: FP32 pixel arithmetic for the gradient-only evaluations (precision-32 contexts)
    const double2* log_table;   // fastmath.cuh reciprocal/log table [kLogTableSize = 64]
    const int* nstars;      // [F] or nullptr
    // state in / out
    const double* q_in;     // [F,S]
    const double* p_in;     // [F,S] (STEP, SINGLE)
    double* q_out;          // [F,S]
    double* p_out;          // [F,S]
    // integrator
    int niter, nsteps, counter_max, f_pos;
    double dt, delta, g_ff2, beta;
    const double* gff2_sched; int n_gff2;
    const double* beta_sched; int n_beta;
    // draws
    const double* normals;  // [F,L,S] or nullptr -> Philox
    const double* lnu;      // [F,L] or nullptr -> Philox
    unsigned long long seed;
    int fid_base, fid_stride;  // Philox field id of local field i = fid_base + i * fid_stride ...
    const int* field_ids;      // ... unless an explicit id array [F] is given
    __device__ __forceinline__ unsigned int philox_field(int field) const {
        return (unsigned int)(field_ids ? field_ids[field] : fid_base + field * fid_stride);
    }
    // outputs
    int chain_stride;
    int n_rows;             // chain rows kept per field
    double* q_chain; double* p_chain; double* E_chain; double* V_chain; double* T_chain;
    unsigned char* A_chain;
    double* accept_rate;    // [F]
    // EVAL outputs
    double* V_out; double* grad_out; double* H_out; double* Hgrad_out;
    int* fp_counts;         // [F,2]
    // chain-kernel work scheduler (MODE_RUN): iteration chunks per chain, per-group completion counters [ceil(F/kChainGroup)],
    // travelling chain state [F,8], error word
    int n_chunks;            // iteration chunks per chain over the whole run
    int chunk_begin, chunk_count;  // chunks [chunk_begin, chunk_begin + chunk_count) are done by THIS launch (0, 0 = all)
    int* sched_done;
    double* sched_state;
    int* sched_err;
    double* draws_normals;  // philox dump
    double* draws_lnu;
};

// Reversible-jump chains (field_kernel MODE_RUN_RJ, field_rj.cuh).  The block sits at the start of the launch's scratch
// buffer, so that LaunchArgs, and with it every other kernel's parameter space, stays as it is.
constexpr int kRjDraws = 14;   // doubles of one (field, iteration) draw record (rj_draws.cuh)
struct RjParams {
    double cdf0, cdf1;          // (P0, P0 + P1) / (P0 + P1 + P2): np.random.choice's cumulative move probabilities
    double pl_lo, pl_span;      // fmin^(1-alpha) and fmax^(1-alpha) - fmin^(1-alpha) of gen_pow_law_sample
    double K_split, beta_a, beta_b, ln_beta;   // ln_beta = ln B(beta_a, beta_b)
    const double* draws;        // [F, L, kRjDraws] injected records, or nullptr (device Philox)
    int* N_chain;               // [F, n_rows] star count at the start of each kept iteration, or nullptr
    unsigned char* move_chain;  // [F, n_rows] 0 within, 1 birth, 2 death, 3 split, 4 merge (gym.move_types), or nullptr
    int* n_final;               // [F] star count after the last iteration
    int* overflow;              // [F] first iteration whose proposal needed more than Nmax stars, -1 if none
    long long field_stride;     // doubles of per-field scratch that follow the block
};
constexpr size_t kRjHeaderDoubles = (sizeof(RjParams) + 15) / 16 * 2;

// ------------------------------------------------------------------ metric (sampler_RHMC.py:229-292)
struct Metric {
    double Hff, dHff, Hxx, dHxx;
};

__device__ __forceinline__ Metric metric_of(const FieldParams& P, double f, double g_ff2) {
    Metric m;
    const double c = (P.B / P.g0) / P.g_ff;
    m.Hff = 1.0 / (f / g_ff2 + c);
    const double s = f + c;
    m.dHff = -1.0 / (s * s);                 // reference formula: ignores g_ff2 (sampler_RHMC.py:292)
    const bool low = f < P.f_low;            // faint clamp at mag mB+2 (sampler_RHMC.py:267-271)
    const double fh = low ? P.f_low : f;
    const double inner = 1.0 / (P.g1 * fh) + P.B / (P.g2 * fh * fh);
    m.Hxx = P.g_xx * (1.0 / inner);
    m.dHxx = low ? 0.0
                 : P.g_xx * (1.0 / (P.g1 * fh * fh) + 2.0 * P.B / (P.g2 * fh * fh * fh)) * (1.0 / (inner * inner));
    return m;
}

// One star's share of the two sums of T = (sum p^2/H + sum ln|H|)/2 (sampler_RHMC.py:353-363)
__device__ __forceinline__ void kinetic_terms(const Metric& m, double pf, double px, double py, double& quad, double& logdet) {
    quad += pf * pf / m.Hff + px * px / m.Hxx + py * py / m.Hxx;
    logdet += log(fabs(m.Hff)) + 2.0 * log(fabs(m.Hxx));
}

// ------------------------------------------------------------------ arithmetic helpers
// 1/a for normal positive a: MUFU.RCP64H seed (~2^-20) + one cubic step -> ~2^-60 relative error.
__device__ __forceinline__ double rcp_fast(double a) {
    double x0;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x0) : "d"(a));
    const double e = fma(-a, x0, 1.0);
    const double t = fma(e, e, e);
    return fma(x0, t, x0);
}
__device__ __forceinline__ float rcp_fast(float a) { return __frcp_rn(a); }

// Division-free form of the reference metric (sampler_RHMC.py:229-292) for the per-star scalar code of the leapfrog step
// (the FP64 divisions of metric_of are ~30 instructions and ~150 cycles each on a dependent path).  With
//   c = (B/g0)/g_ff, u = f/g_ff2 + c, w = 1/(f + c), fh = max(f, f_low), v = 1/fh, t = 1/g1 + (B/g2) v :
//   H_ff = 1/u,  H_ff' = -w^2,  H_ff'/H_ff = -u w^2,  -H_ff'/H_ff^2 = (u w)^2,
//   1/H_xx = v t / g_xx,  H_xx'/H_xx = v (t + (B/g2) v) / t   (0 below the faint clamp).
// Every reciprocal is rcp_fast (2^-60); metric_of stays the reference-order form for reported H, H' and the energies.
struct MetricK {
    double c, ig2, ig1, Bg2, igxx, f_low;
};
__host__ __device__ __forceinline__ MetricK make_metric_k(const FieldParams& P, double g_ff2) {
    MetricK K;
    K.c = (P.B / P.g0) / P.g_ff;
    K.ig2 = 1.0 / g_ff2;
    K.ig1 = 1.0 / P.g1;
    K.Bg2 = P.B / P.g2;
    K.igxx = 1.0 / P.g_xx;
    K.f_low = P.f_low;
    return K;
}
struct MetricFast {
    double u;      // 1/H_ff
    double kap;    // -H_ff'/H_ff^2
    double ihxx;   // 1/H_xx
    double tphi;   // (H_ff'/H_ff + 2 H_xx'/H_xx)/2
};
__device__ __forceinline__ MetricFast metric_fast(const MetricK& K, double f) {
    MetricFast m;
    const double u = fma(f, K.ig2, K.c);
    const double w = rcp_fast(f + K.c);
    const double uw = u * w;
    const bool low = f < K.f_low;
    const double v = rcp_fast(low ? K.f_low : f);
    const double bv = K.Bg2 * v;
    const double t = bv + K.ig1;
    m.u = u;
    m.kap = uw * uw;
    m.ihxx = (v * t) * K.igxx;
    const double dxx = low ? 0.0 : (v * (t + bv)) * rcp_fast(t);
    m.tphi = fma(-0.5 * uw, w, dxx);
    return m;
}
__device__ __forceinline__ double inv_hff_k(const MetricK& K, double f) { return fma(f, K.ig2, K.c); }
__device__ __forceinline__ double inv_hxx_k(const MetricK& K, double f) {
    const double v = rcp_fast(fmax(f, K.f_low));
    return (v * fma(K.Bg2, v, K.ig1)) * K.igxx;
}

__device__ __forceinline__ double ipow(double b, int n) {  // b^n, small n >= 0
    double r = 1.0;
    while (n > 0) {
        if (n & 1) r *= b;
        b *= b;
        n >>= 1;
    }
    return r;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Deterministic CTA-wide sum of NV doubles; result valid in every thread.  `red` holds >= NV*32 doubles.
template <int NV>
__device__ __forceinline__ void block_sum(double (&v)[NV], double* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
    __syncthreads();  // protect `red` from the previous use
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) red[i * 32 + warp] = v[i];
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        double x = (lane < nw) ? red[i * 32 + lane] : 0.0;
        v[i] = warp_sum(x);
    }
}

// ------------------------------------------------------------------ Philox4x32-10 (Salmon et al. 2011)
struct Philox {
    uint32_t key[2];
    __device__ __forceinline__ static void round(uint32_t (&c)[4], const uint32_t (&k)[2]) {
        const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
        const uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
        const uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k[0], n1 = lo1, n2 = hi0 ^ c[3] ^ k[1], n3 = lo0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    }
    __device__ __forceinline__ static void block(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                 uint32_t (&out)[4]) {
        uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
        uint32_t c[4] = {c0, c1, c2, c3};
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            round(c, k);
            k[0] += 0x9E3779B9u;
            k[1] += 0xBB67AE85u;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) out[i] = c[i];
    }
};

// uniform in (0,1) with 53 random bits from two words
__device__ __forceinline__ double u01(uint32_t a, uint32_t b) {
    const unsigned long long m = ((unsigned long long)(a >> 5) << 26) | (unsigned long long)(b >> 6);
    return ((double)m + 0.5) * (1.0 / 9007199254740992.0);
}

// Three standard normals for (field, iteration, star); counter layout documented in DESIGN.md.
__device__ __forceinline__ void philox_normals3(uint64_t seed, uint32_t field, uint32_t iter, uint32_t star,
                                                double (&z)[3]) {
    uint32_t r[4];
    Philox::block(seed, star, iter, field, 0u, r);
    double u1 = u01(r[0], r[1]), u2 = u01(r[2], r[3]);
    double rad = sqrt(-2.0 * log(u1)), s, c;
    sincospi(2.0 * u2, &s, &c);
    z[0] = rad * c;
    z[1] = rad * s;
    Philox::block(seed, star, iter, field, 1u, r);
    u1 = u01(r[0], r[1]);
    u2 = u01(r[2], r[3]);
    rad = sqrt(-2.0 * log(u1));
    sincospi(2.0 * u2, &s, &c);
    z[2] = rad * c;
}
__device__ __forceinline__ double philox_lnu(uint64_t seed, uint32_t field, uint32_t iter) {
    uint32_t r[4];
    Philox::block(seed, 0xFFFFFFFFu, iter, field, 2u, r);
    return log(u01(r[0], r[1]));
}

}  // namespace srhmc
