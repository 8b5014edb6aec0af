// Warp-resident one-star chain kernel (sm_100a): BASELINE.json configs[0..1] -- thousands of independent
// one-star RHMC chains on small images (C <= 32 columns, R <= 64 rows).
//
// LPC lanes own one chain (LPC = 4: eight chains per warp).  A lane owns the image columns sub, sub+LPC, ...;
// the chain's data image sits in shared memory for the whole launch; the star state, momenta, cached gradient
// and energies live in registers (every lane of the group holds the same copy), so a full
// (niter+1) x nsteps chain runs without any block-level barrier, global traffic (except chain rows written out)
// or host involvement.  Blocks are single warps; the grid is sized to a balanced number of warps per SM and each
// warp walks its share of the chains.
//
// Per gradient evaluation (reference: base_class.dVdq, sampler_RHMC.py:365-425, one star, full-image PSF):
//   lanes compute ex_i = exp(-(i+.5-x)^2/2s^2) for their rows -> shared row table {ex_i, ex_i*(i+.5-x)};
//   lanes compute ey_j/(2 pi s^2) for their columns (registers);
//   row loop: Lambda = B + ex_i * (f ey_j); rho = D/Lambda - 1 (MUFU.RCP64H + cubic Newton step);
//             c0_j += rho ex_i; c1_j += rho ex_i dx_i;      [+ V += Lambda - D ln Lambda on request]
//   g_f = -sum_j ey_j c0_j,  g_x = -(f/s^2) sum_j ey_j c1_j,  g_y = -(f/s^2) sum_j ey_j dy_j c0_j  via shuffles.
#pragma once
#include <math_constants.h>

#include "common.cuh"
#include "fastmath.cuh"

namespace srhmc {

constexpr int kChainCS = 32;  // column stride of a chain image in shared memory
constexpr int kChainTabPad = 16;  // bytes of padding after each chain's row table (bank staggering, see chain_kernel)

struct ChainState {
    double f, x, y, pf, px, py;  // q, p
    double gf, gx, gy;           // pixel part of dV/dq at (f, x, y)
    double Vpix;                 // sum(Lambda - D ln Lambda) at (f, x, y)
    // metric cache at f (see ChainConst): u = 1/H_ff, kap = -H_ff'/H_ff^2, ihxx = 1/H_xx,
    // tphi = (H_ff'/H_ff + 2 H_xx'/H_xx)/2
    double u, kap, ihxx, tphi;
};

// Division-free form of the reference metric (sampler_RHMC.py:229-292) for the hot loop.  With
//   c = (B/g0)/g_ff, u = f/g_ff2 + c, w = 1/(f + c), fh = max(f, f_low), v = 1/fh, t = 1/g1 + (B/g2) v :
//   H_ff = 1/u,  H_ff' = -w^2,  H_ff'/H_ff = -u w^2,  -H_ff'/H_ff^2 = (u w)^2,
//   1/H_xx = v t / g_xx,  H_xx'/H_xx = v (t + (B/g2) v) / t   (0 below the faint clamp).
// Every reciprocal is MUFU.RCP64H + one cubic Newton step (rcp_fast, ~2^-60 relative error).
struct ChainConst {
    double c, ig2, ig1, Bg2, igxx, g_xx, f_low;
    double h, hh, delta;
};

__device__ __forceinline__ ChainConst make_chain_const(const FieldParams& P, double g_ff2, double h, double delta) {
    ChainConst K;
    K.c = (P.B / P.g0) / P.g_ff;
    K.ig2 = 1.0 / g_ff2;
    K.ig1 = 1.0 / P.g1;
    K.Bg2 = P.B / P.g2;
    K.igxx = 1.0 / P.g_xx;
    K.g_xx = P.g_xx;
    K.f_low = P.f_low;
    K.h = h;
    K.hh = h / 2.0;
    K.delta = delta;
    return K;
}

__device__ __forceinline__ double inv_hxx(const ChainConst& K, double f) {
    const double v = rcp_fast(fmax(f, K.f_low));
    return (v * fma(K.Bg2, v, K.ig1)) * K.igxx;
}

// full metric cache at s.f
__device__ __forceinline__ void refresh_metric(const ChainConst& K, ChainState& s) {
    const double f = s.f;
    const double u = fma(f, K.ig2, K.c);
    const double w = rcp_fast(f + K.c);
    const double uw = u * w;
    const bool low = f < K.f_low;
    const double v = rcp_fast(low ? K.f_low : f);
    const double bv = K.Bg2 * v;
    const double t = bv + K.ig1;
    s.u = u;
    s.kap = uw * uw;
    s.ihxx = (v * t) * K.igxx;
    const double dxx = low ? 0.0 : (v * (t + bv)) * rcp_fast(t);
    s.tphi = fma(-0.5 * uw, w, dxx);
}

// data pixel as double: plain load, or exact unsigned count
__device__ __forceinline__ double ld_pix(const double* p) { return *p; }
// integer count -> double: one I2F on the (otherwise idle) conversion unit; measured 9% faster than the 2^52 bias trick
// (a MOV plus a DADD on the FP64 pipe)
__device__ __forceinline__ double ld_pix(const unsigned int* p) { return (double)*p; }
__device__ __forceinline__ double ld_pix(const unsigned short* p) { return (double)(unsigned int)*p; }
// FP32 build (north_star: "<= 1e-4 in the FP32 build"): pixel as float, reciprocal by MUFU.RCP alone
__device__ __forceinline__ float ld_pixf(const double* p) { return (float)*p; }
__device__ __forceinline__ float ld_pixf(const unsigned int* p) { return (float)*p; }
// uint16 count -> float without the conversion unit (the FP32 loop is bound by the XU pipe: MUFU.RCP + I2F per pixel):
// 2^23 + d is exact for d < 2^16, so OR-ing d into the mantissa of 2^23 and subtracting 2^23 converts on the ALU / FP32 pipes
__device__ __forceinline__ float ld_pixf(const unsigned short* p) {
    return __uint_as_float(0x4B000000u | (unsigned int)*p) - 8388608.0f;
}
__device__ __forceinline__ float rcp_pixf(float a) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
    return r;
}
// (Measured and not adopted: the product-tree reciprocal (rcp_row) in the FP32 loop: 1725 against 1738 M star-steps/s.)
// (Measured and not adopted: feeding the count as the double 2^52 + d with fma(X, r, -2^52 r) = round(d r) removes the
// I2F from the pixel loop but costs three integer instructions per pixel: 1422 against 1472 M star-steps/s.)
// (Measured and not adopted: one quadratic Newton step instead of rcp_fast's cubic one is 8% faster, but its 2^-40 error
// grows to 1e-8 in q over 30 Metropolis iterations, beyond the 1e-9 trajectory tolerance of the parity tests.)

// Reciprocals of N pixels from ONE MUFU.RCP64H: 1/a_k = (product of the others) / (product of all).  The FP64 instruction
// count is the same as N separate cubic Newton reciprocals (3 per pixel: products down, one Newton step, products up), but the
// pixel loop was bound by the XU pipe (MUFU.RCP64H + I2F per pixel, 8 issue cycles each per scheduler against 14 cycles of
// DFMA): this leaves one MUFU per 3 (4) pixels.  Each result carries <= 4 roundings (~2^-51 relative).  Lambda = 0 in a group
// gives NaN for its neighbours as well (the reference gives inf at that pixel and a non-finite gradient either way).
template <int N>
__device__ __forceinline__ void rcp_group(const double (&a)[N], double (&r)[N]) {
    static_assert(N == 3 || N == 4, "reciprocal groups are triples or quadruples");
    if constexpr (N == 3) {
        const double p01 = a[0] * a[1];
        const double ip = rcp_fast(p01 * a[2]);
        const double r01 = a[2] * ip;
        r[2] = p01 * ip;
        r[0] = a[1] * r01;
        r[1] = a[0] * r01;
    } else {
        const double p01 = a[0] * a[1], p23 = a[2] * a[3];
        const double ip = rcp_fast(p01 * p23);
        const double r01 = p23 * ip, r23 = p01 * ip;
        r[0] = a[1] * r01;
        r[1] = a[0] * r01;
        r[2] = a[3] * r23;
        r[3] = a[2] * r23;
    }
}
// reciprocals of the NCS pixels a lane owns in one image row: triples when NCS is a multiple of 3 (24-column window: 6 slots),
// quadruples for the full-width variant (8 slots)
template <int NCS>
__device__ __forceinline__ void rcp_row(const double (&lam)[NCS], double (&r)[NCS]) {
    constexpr int GS = (NCS % 3 == 0) ? 3 : 4;
#pragma unroll
    for (int g = 0; g < NCS / GS; ++g) {
        double a[GS], o[GS];
#pragma unroll
        for (int k = 0; k < GS; ++k) a[k] = lam[g * GS + k];
        rcp_group<GS>(a, o);
#pragma unroll
        for (int k = 0; k < GS; ++k) r[g * GS + k] = o[k];
    }
}

// Elements of padding after each chain image so that the chains of one warp sit on disjoint shared-memory banks:
// the LPC lanes of a chain read LPC consecutive pixels, so shifting chain g by g*LPC pixels tiles the banks.
__host__ __device__ constexpr int chain_pad(int lpc) { return lpc; }

// Dynamic shared memory of one single-warp block (kernel and host both take it from here): the log table, then the
// kChainGroup chain images, then the kChainGroup row tables.  A row table is a double2 per image row (plus, in the FP32
// build, a float2 per row after it) and is read and written with 128-bit accesses, so every table must start on a
// 16-byte boundary: the FP32 stride 24 R + 16 is rounded up (it is 8 bytes short for odd R); the double stride 16 R + 16
// and the image block before the tables are multiples of 16 already.
__host__ __device__ constexpr ChainLayout chain_layout(int R, size_t elem, bool f32) {
    ChainLayout L{};
    L.log_bytes = kLogTableSize * sizeof(double2);
    L.img_elems = (size_t)R * kChainCS + chain_pad(kChainLPC);
    L.img_bytes = L.img_elems * elem;
    const size_t tab = (size_t)R * (sizeof(double2) + (f32 ? sizeof(float2) : 0)) + kChainTabPad;
    L.tab_bytes = f32 ? (tab + 15) & ~(size_t)15 : tab;
    L.tab_base = L.log_bytes + kChainGroup * L.img_bytes;
    L.smem_bytes = L.tab_base + kChainGroup * L.tab_bytes;
    return L;
}

template <int LPC>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
    for (int o = LPC / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// log1p(t) for |t| < 2^-7 by the alternating series through t^7 (truncation t^8/8 < 2^-59 absolute).
__device__ __forceinline__ double log1p_small(double t) {
    double p = kFM.log1p_c[7];
#pragma unroll
    for (int k = 6; k >= 1; --k) p = fma(p, t, kFM.log1p_c[k]);
    return p * t;
}

// Image rows [r0, r1), all column slots of the lane (columns sub + LPC c): gradient column sums and, per TIER, the
// D * log1p(t) part of the potential.  TIER 0: table logarithm; 1: 7-term series (|t| < 2^-7).
template <int TIER, int LPC, int NCS, typename DT>
__device__ __forceinline__ void rows_all_slots(int r0, int r1, const DT* __restrict__ sDl, const double2* __restrict__ rt,
                                               const double2* __restrict__ ltab, double B, const double (&fey)[NCS],
                                               const double (&tb)[NCS], double (&c0)[NCS],
                                               double (&c1)[NCS], double& vlog, int& bad) {
    constexpr int CPL = NCS;
    for (int i = r0; i < r1; ++i) {
        const double2 re = rt[i];
        double lam[CPL], il[CPL];
#pragma unroll
        for (int c = 0; c < CPL; ++c) lam[c] = fma(re.x, fey[c], B);
        rcp_row<CPL>(lam, il);
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            const double d = ld_pix(sDl + i * kChainCS + LPC * c);
            const double rho = fma(d, il[c], -1.0);
            c0[c] = fma(rho, re.x, c0[c]);
            c1[c] = fma(rho, re.y, c1[c]);
            if (TIER == 0) {
                const double w = fma(re.x, tb[c], 1.0);
                bad |= (__double2hiint(w) < 0x00100000);  // Lambda <= 0: ln undefined -> NaN
                vlog = fma(d, log_pos(w, ltab), vlog);
            } else {
                vlog = fma(d, log1p_small(re.x * tb[c]), vlog);
            }
        }
    }
}

// Rows i whose Gaussian weight exp(-(i+.5-x)^2/2s^2) can reach `thresh / peak` (peak >= 0): the conservative integer
// window [lo, hi) in float arithmetic, empty (lo = R, hi = 0) when peak < thresh.  NaN-safe.
__device__ __forceinline__ void row_window(float xc, float peak, float thresh, float two_s2, int R, int& lo, int& hi) {
    lo = R;
    hi = 0;
    if (peak >= thresh) {
        const float w = sqrtf(__logf(peak / thresh) * two_s2) + 0.51f;
        lo = (int)fminf(fmaxf(floorf(xc - w), 0.0f), (float)R);
        hi = (int)fminf(fmaxf(ceilf(xc + w) + 1.0f, 0.0f), (float)R);
    }
}

// Pixel part of the gradient (and of V) for one chain; all lanes of the warp must call it together.
//
// Tables: lane `sub` owns rows sub + LPC k and columns sub + LPC c.  Along that stride the Gaussian obeys
//   e(u + L) = e(u) r(u),  r(u + L) = r(u) exp(-L^2/s^2),  r(u) = exp(-(2 L u + L^2)/2s^2)
// so each lane evaluates two exponentials per axis and multiplies its way along (error a few ulp per step).
//
// Rows farther than P.wcut pixels from the star have ex_i < 2^-50: their pixels change neither the gradient sums nor
// V beyond 1e-13 relative, and are skipped (the window is the union over the chains of the warp).
//
// V is evaluated in the separable form (Lambda_ij = B + a_i b_j with a_i = ex_i, b_j = f ey_j):
//   sum(Lambda - D ln Lambda) = [R C B - ln B sum(D)] + (sum_i a_i)(sum_j b_j) - sum_ij D_ij log1p(a_i b_j / B)
// so only the last sum needs per-pixel work; log1p is tiered (two tiers) per row range by the largest |t| = |a_i b_j / B| the
// warp sees there (see rows_all_slots).  Code size matters here: a build that unrolled per-slot tier loops grew the
// kernel to 30k instructions and spent 31% of its issue slots waiting for instruction fetch, so the kernel is
// specialised per mode (template MODE) and the tier loops are kept compact.  `vconst` is the bracketed constant of this chain's image.
// PT = float selects the FP32 pixel arithmetic for the gradient-only evaluations (9 of 10 in a chain): float row table,
// float Lambda / rho / column sums, MUFU.RCP; the star state, the tables' recurrences, the final reductions and every
// evaluation that also returns the potential (WANT_V) stay FP64 -- so the energies of the Metropolis test are exact for
// the state reached, and approximate gradients only change the proposal, not the target distribution.
template <int LPC, int NCS, bool WANT_V, typename DT, typename PT = double>
__device__ __forceinline__ void chain_eval(const FieldParams& P, const DT* __restrict__ sD, double2* __restrict__ rt,
                                           const double2* __restrict__ ltab, int sub, double vconst, ChainState& s) {
    constexpr bool F32 = sizeof(PT) == 4 && !WANT_V;
    float2* __restrict__ rtf = reinterpret_cast<float2*>(rt + P.R);   // FP32 copy of the row table (allocated by the FP32 build)
    constexpr int CPL = NCS;            // column slots per lane
    constexpr int WIN = NCS * LPC;      // columns the chain's lanes cover
    constexpr unsigned FULL = 0xffffffffu;
    const int R = P.R, C = P.C;
    const double f = s.f, x = s.x, y = s.y;
    const double cL = P.cL;  // exp(-LPC^2/s^2)
    // All exponentials of this evaluation up front in one straight-line block (four independent Horner chains).
    // rows: anchor at the lane's row nearest the star and recur outwards in both directions, so the anchor never
    // underflows while the star is within ~55 px of the image (beyond that every weight is 0 in double anyway);
    // columns: at most 32 of them, so the first column's weight cannot underflow for a star near the image.
    // row window of the warp
    int i_lo, i_hi;
    {
        const double xc = x - 0.5;
        const int lo = (int)fmin(fmax(ceil(xc - P.wcut), 0.0), (double)R);
        const int hi = (int)fmin(fmax(floor(xc + P.wcut) + 1.0, 0.0), (double)R);
        i_lo = __reduce_min_sync(FULL, lo);
        i_hi = __reduce_max_sync(FULL, hi);
    }
    const int K = (R - sub + LPC - 1) / LPC;  // rows of this lane
    const double kf = fmin(fmax(rint((x - 0.5 - (double)sub) * (1.0 / LPC)), 0.0), (double)(K > 0 ? K - 1 : 0));
    const int ks = (int)kf;
    const double us = ((double)(sub + LPC * ks) + 0.5) - x;
    // column window: the WIN columns starting at the first one within WIN/2 pixels of the star (kept inside the image)
    int jb = sub;
    if (WIN < kChainCS) {
        const double a = ceil(y - (0.5 + 0.5 * WIN));
        jb += (int)fmin(fmax(a, 0.0), (double)max(C - WIN, 0));
    }
    const double v0 = ((double)jb + 0.5) - y;
    const double arg_r = (us * us) * P.inv2s2, arg_c = (v0 * v0) * P.inv2s2;
    const bool ok_r = arg_r < 690.0, ok_c = arg_c < 690.0;
    const double LL = (double)(LPC * LPC);
    const double e_r = exp_neg(-arg_r);
    const double w_r = exp_neg(-(2.0 * LPC * P.inv2s2) * us);   // r_up = w cLh, r_dn = cLh / w, cLh = exp(-L^2/2s^2)
    const double e_c = exp_neg(-arg_c);
    const double r_c = exp_neg(-fma(2.0 * LPC, v0, LL) * P.inv2s2);
    const double cLh = P.cLh;
    double sa = 0.0;
    if (K > 0) {
        const double es = ok_r ? e_r : 0.0;
        const double r_up = ok_r ? w_r * cLh : 0.0;
        const double r_dn = ok_r ? rcp_fast(w_r) * cLh : 0.0;
        double e = es, r = r_up, u = us;
        for (int k = ks; k < K; ++k) {
            if (F32) rtf[sub + LPC * k] = make_float2((float)e, (float)(e * u));
            else rt[sub + LPC * k] = make_double2(e, e * u);
            if (WANT_V) sa += e;
            e *= r;
            r *= cL;
            u += (double)LPC;
        }
        e = es * r_dn;
        r = r_dn * cL;
        u = us - (double)LPC;
        for (int k = ks - 1; k >= 0; --k) {
            if (F32) rtf[sub + LPC * k] = make_float2((float)e, (float)(e * u));
            else rt[sub + LPC * k] = make_double2(e, e * u);
            if (WANT_V) sa += e;
            e *= r;
            r *= cL;
            u -= (double)LPC;
        }
    }
    double ey[CPL], fey[CPL], eydy[CPL], tb[CPL], sb = 0.0;
    {
        double v = v0;
        double e = ok_c ? e_c * P.norm : 0.0;
        double r = ok_c ? r_c : 0.0;
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            const bool in = jb + LPC * c < C;
            ey[c] = in ? e : 0.0;
            fey[c] = f * ey[c];
            eydy[c] = ey[c] * v;
            if (WANT_V) {
                tb[c] = fey[c] * P.invB;
                sb += fey[c];
            }
            e *= r;
            r *= cL;
            v += (double)LPC;
        }
    }
    __syncwarp();
    double c0[CPL], c1[CPL], vlog = 0.0;
    int bad = 0;
#pragma unroll
    for (int c = 0; c < CPL; ++c) c0[c] = c1[c] = 0.0;
    if (F32) {
        float feyf[CPL], c0f[CPL], c1f[CPL];
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            feyf[c] = (float)fey[c];
            c0f[c] = c1f[c] = 0.0f;
        }
        const float Bf = (float)P.B;
#pragma unroll 2
        for (int i = i_lo; i < i_hi; ++i) {
            const float2 re = rtf[i];
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                const float lam = fmaf(re.x, feyf[c], Bf);
                const float rho = fmaf(ld_pixf(sD + i * kChainCS + jb + LPC * c), rcp_pixf(lam), -1.0f);
                c0f[c] = fmaf(rho, re.x, c0f[c]);
                c1f[c] = fmaf(rho, re.y, c1f[c]);
            }
        }
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            c0[c] = (double)c0f[c];
            c1[c] = (double)c1f[c];
        }
    } else if (!WANT_V) {
        // rows per trip of the gradient-only loop.  With the product-tree reciprocal (one MUFU per three pixels) and a 255-register
        // budget (still 8 single-warp blocks per SM) four rows measured best: x2 1533, x3 1543, x4 1556 M star-steps/s
#pragma unroll 4
        for (int i = i_lo; i < i_hi; ++i) {
            const double2 re = rt[i];
            double lam[CPL], il[CPL];
#pragma unroll
            for (int c = 0; c < CPL; ++c) lam[c] = fma(re.x, fey[c], P.B);
            rcp_row<CPL>(lam, il);
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                const double rho = fma(ld_pix(sD + i * kChainCS + jb + LPC * c), il[c], -1.0);
                c0[c] = fma(rho, re.x, c0[c]);
                c1[c] = fma(rho, re.y, c1[c]);
            }
        }
    } else {
        // rows [n0, n1) where some lane of the warp can see |t| >= 2^-7 take the table logarithm, the others the
        // 7-term series.  (A third tier, t - t^2/2 for |t| < 2^-18, was measured SLOWER: its extra loop bodies cost
        // more in instruction fetch than the shorter series saved.)
        float peak = 0.0f;
#pragma unroll
        for (int c = 0; c < CPL; ++c) peak = fmaxf(peak, fabsf((float)tb[c]));
        peak *= 1.0001f;
        const float xc = (float)(x - 0.5), two_s2 = (float)(1.0 / P.inv2s2);
        int n0, n1;
        row_window(xc, peak, 0.0078125f, two_s2, R, n0, n1);  // |t| >= 2^-7
        n0 = __reduce_min_sync(FULL, n0);
        n1 = __reduce_max_sync(FULL, n1);
        n0 = min(max(n0, i_lo), i_hi);
        n1 = min(max(n1, n0), i_hi);
        rows_all_slots<1, LPC, NCS>(i_lo, n0, sD + jb, rt, ltab, P.B, fey, tb, c0, c1, vlog, bad);
        rows_all_slots<0, LPC, NCS>(n0, n1, sD + jb, rt, ltab, P.B, fey, tb, c0, c1, vlog, bad);
        rows_all_slots<1, LPC, NCS>(n1, i_hi, sD + jb, rt, ltab, P.B, fey, tb, c0, c1, vlog, bad);
    }
    __syncwarp();  // row table is rewritten by the next evaluation
    double sf = 0.0, sx = 0.0, sy = 0.0;
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
        sf = fma(ey[c], c0[c], sf);
        sx = fma(ey[c], c1[c], sx);
        sy = fma(eydy[c], c0[c], sy);
    }
    sf = group_sum<LPC>(sf);
    sx = group_sum<LPC>(sx);
    sy = group_sum<LPC>(sy);
    s.gf = -sf;
    s.gx = -sx * f * P.inv_s2;
    s.gy = -sy * f * P.inv_s2;
    if (WANT_V) {
        if (bad) vlog = CUDART_NAN;
        sa = group_sum<LPC>(sa);
        sb = group_sum<LPC>(sb);
        vlog = group_sum<LPC>(vlog);
        s.Vpix = fma(sa, sb, vconst) - vlog;
    }
}

// The chain kernel's copy of philox_normals3 (common.cuh): same counters and uniforms, Box-Muller radius through the
// kernel's table logarithm and only the cosine branch for the third normal -- a third of the inlined code of the
// libm version, values equal to a few ulp.
__device__ __forceinline__ void philox_normals3_tab(uint64_t seed, uint32_t field, uint32_t iter, uint32_t star,
                                                    const double2* __restrict__ ltab, double (&z)[3]) {
    uint32_t r[4];
    Philox::block(seed, star, iter, field, 0u, r);
    double u1 = u01(r[0], r[1]), u2 = u01(r[2], r[3]);
    double rad = sqrt(-2.0 * log_pos(u1, ltab)), s, c;
    sincospi(2.0 * u2, &s, &c);
    z[0] = rad * c;
    z[1] = rad * s;
    Philox::block(seed, star, iter, field, 1u, r);
    u1 = u01(r[0], r[1]);
    u2 = u01(r[2], r[3]);
    z[2] = sqrt(-2.0 * log_pos(u1, ltab)) * cospi(2.0 * u2);
}

__device__ __forceinline__ double philox_lnu_tab(uint64_t seed, uint32_t field, uint32_t iter,
                                                 const double2* __restrict__ ltab) {
    uint32_t r[4];
    Philox::block(seed, 0xFFFFFFFFu, iter, field, 2u, r);
    return log_pos(u01(r[0], r[1]), ltab);
}

// V(q, f_pos) and T(p, H(q)) of a one-star field from the cached pixel potential and metric
// (sampler_RHMC.py:294-363).
// (Making this and the Philox helpers __noinline__ to shrink the kernel was measured slower: the chain state then
// travels through local memory around every call.)
__device__ __forceinline__ void chain_energies(const FieldParams& P, const ChainConst& K, const ChainState& s, int f_pos,
                                               const double2* __restrict__ ltab, double& V, double& T) {
    const double v0 = (s.pf * s.pf) * s.u + (s.px * s.px + s.py * s.py) * s.ihxx;
    // ln|H_ff| + 2 ln|H_xx| through the kernel's own table logarithm (half the code of two libm calls)
    const double v1 = -(log_pos(fabs(s.u), ltab) + 2.0 * log_pos(fabs(s.ihxx), ltab));
    T = (v0 + v1) / 2.0;
    double v = s.Vpix;
    if (P.use_prior) v += P.alpha * log(s.f) + P.Vpc;
    const bool bad = (f_pos && s.f < P.f_lim) || (s.x < -1.0) || (s.x > P.R + 1.0) || (s.y < -1.0) || (s.y > P.C + 1.0);
    V = bad ? CUDART_INF : v;
}

// base_class.RHMC_single_step for a one-star field, state in registers (sampler_RHMC.py:522-566).
// Requires s.g*, s.u, s.kap, s.ihxx, s.tphi valid at s.f on entry; leaves them valid on exit.
template <int LPC, int NCS, typename DT, typename PT = double>
__device__ __forceinline__ void chain_step(const FieldParams& P, const ChainConst& K, const DT* sD, double2* rt,
                                           const double2* ltab, int sub, double vconst, ChainState& s, int counter_max,
                                           bool want_V, int& cnt_p, int& cnt_q) {
    const double h = K.h;
    // (1) p <- p - h dphi/dq(q)
    {
        double gf = s.gf + s.tphi;
        if (P.use_prior) gf = fma(P.alpha, rcp_fast(s.f), gf);
        s.pf = fma(-h, gf, s.pf);
        s.px = fma(-h, s.gx, s.px);
        s.py = fma(-h, s.gy, s.py);
    }
    // (2) p' = rho - h dtau/dq(q, p): only the flux slot moves, dtau/dq_f = p_f^2 kap / 2
    {
        const double rho = s.pf, hk = K.hh * s.kap;
        double pf = s.pf;
        cnt_p = 0;
        while (cnt_p < counter_max) {
            const double pn = fma(-hk, pf * pf, rho);
            const bool more = fabs(pf - pn) > K.delta;
            pf = pn;
            ++cnt_p;
            if (!more) break;
        }
        s.pf = pf;
    }
    // (3) q' = sigma + h (p/H(sigma) + p/H(q)).  With u = 1/H_ff, ih = 1/H_xx:
    //     f_k = sigma_f + h p_f (u0 + u(f_{k-1})),  x_k = sigma_x + h p_x g_k,  g_k = ih0 + ih(f_{k-1}),  g_0 := 0
    {
        const double sf = s.f, u0 = s.u, ih0 = s.ihxx;
        const double hpf = h * s.pf, hpx = h * s.px, hpy = h * s.py;
        const double hpm = fmax(fabs(hpx), fabs(hpy));
        double qf = sf, uq = u0, ihq = ih0, g = 0.0;
        cnt_q = 0;
        while (cnt_q < counter_max) {
            const double gn = ih0 + ihq;
            const double nf = fma(hpf, u0 + uq, sf);
            const double d = fmax(fabs(qf - nf), hpm * fabs(gn - g));
            qf = nf;
            g = gn;
            ++cnt_q;
            if (!(d > K.delta)) break;
            uq = fma(qf, K.ig2, K.c);
            ihq = inv_hxx(K, qf);
        }
        s.f = qf;
        s.x = fma(hpx, g, s.x);
        s.y = fma(hpy, g, s.y);
    }
    // (4) p <- p - h dtau/dq(q, p) at the new q;  metric cache at the new f
    refresh_metric(K, s);
    s.pf = fma(-(K.hh * s.kap), s.pf * s.pf, s.pf);
    // (5) gradient at the new q and last half kick
    if (want_V)
        chain_eval<LPC, NCS, true, DT, PT>(P, sD, rt, ltab, sub, vconst, s);
    else
        chain_eval<LPC, NCS, false, DT, PT>(P, sD, rt, ltab, sub, vconst, s);
    {
        double gf = s.gf + s.tphi;
        if (P.use_prior) gf = fma(P.alpha, rcp_fast(s.f), gf);
        s.pf = fma(-h, gf, s.pf);
        s.px = fma(-h, s.gx, s.px);
        s.py = fma(-h, s.gy, s.py);
    }
    // (6) reflections
    if (s.f < P.f_lim) s.pf = -s.pf;
    if ((s.x < 0.0) || (s.x > P.R - 1.0)) s.px = -s.px;
    if ((s.y < 0.0) || (s.y > P.C - 1.0)) s.py = -s.py;
}

// register budget: the 255-register maximum (the kernel uses 240 and still keeps 8 single-warp blocks per SM resident)
constexpr int kChainMaxReg = 255;
template <int LPC, typename DT, int MODE, int NCS, int MAXREG = kChainMaxReg, typename PT = double>
__global__ void __maxnreg__(MAXREG) chain_kernel(const __grid_constant__ FieldParams P, const __grid_constant__ LaunchArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int GPW = 32 / LPC;  // chains per warp
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int grp = lane / LPC, sub = lane % LPC;
    const int R = P.R, C = P.C;
    static_assert(GPW == kChainGroup && LPC == kChainLPC, "chain_layout describes kChainGroup chains of kChainLPC lanes");
    // per-chain image stride padded by LPC elements: the GPW chains of a warp then sit on disjoint shared-memory banks.
    // Row tables: 16 bytes of padding per chain, so that entry i of chain g sits 4 (g + i) banks into shared memory and the
    // warp's 8 distinct 16-byte entries of a row fill one 128-byte wavefront (unpadded, the 512-byte table stride put all
    // eight on the same four banks: an 8-way conflict on every row-table load and store)
    const ChainLayout lay = chain_layout(R, sizeof(DT), sizeof(PT) == 4);
    const size_t img_elems = lay.img_elems;
    const size_t tab_bytes = lay.tab_bytes;
    // (GPW * img_elems * sizeof(DT) below is GPW * lay.img_bytes, written as the kernel always computed it)
    const size_t warp_bytes = (size_t)GPW * (img_elems * sizeof(DT) + tab_bytes);
    double2* ltab = reinterpret_cast<double2*>(smem_raw);
    unsigned char* wbase = smem_raw + lay.log_bytes + (size_t)warp * warp_bytes;
    DT* sD = reinterpret_cast<DT*>(wbase) + (size_t)grp * img_elems;
    double2* rt = reinterpret_cast<double2*>(wbase + (size_t)GPW * img_elems * sizeof(DT) + (size_t)grp * tab_bytes);
    const double h = A.dt / 2.0;
    for (int i = threadIdx.x; i < kLogTableSize; i += blockDim.x) ltab[i] = A.log_table[i];
    __syncthreads();

    // Work items are (group of GPW chains, chunk of Metropolis iterations); chunk c of a group may run on a different
    // warp than chunk c-1 (the chain state travels through global memory, ordered by a per-group counter), which
    // lets a batch that is not a multiple of the resident warp count finish without a long under-filled tail.
    const int fb = A.field_begin, fe = A.field_end > 0 ? A.field_end : A.n_fields;
    const int G = (fe - fb + GPW - 1) / GPW;
    const int n_chunks = (MODE == MODE_RUN && A.n_chunks > 1) ? A.n_chunks : 1;
    const int chunk_count = (MODE == MODE_RUN && A.chunk_count > 0) ? A.chunk_count : n_chunks;
    const int chunk_begin = (MODE == MODE_RUN && A.chunk_count > 0) ? A.chunk_begin : 0;
    const long long n_tasks = (long long)G * chunk_count;
    const long long gw = (long long)blockIdx.x * nw + warp, W = (long long)gridDim.x * nw;
    for (long long task = gw; task < n_tasks; task += W) {
        const int chunk = chunk_begin + (int)(task / G);
        const int base = fb + (int)(task % G) * GPW;
        const bool live = base + grp < fe;
        const int field = live ? base + grp : fe - 1;  // idle group shadows a valid chain, writes nothing
        constexpr int n = 1;  // the host routes only exactly-one-star batches to this kernel
        const DT* gD = reinterpret_cast<const DT*>(sizeof(DT) == 8 ? A.D : A.D_int) + (size_t)field * R * C;
        __syncwarp();
        double sumD = 0.0;
        for (int i = 0; i < R; ++i)
            for (int j = sub; j < kChainCS; j += LPC) {
                const DT v = (j < C) ? gD[i * C + j] : (DT)0;
                sD[i * kChainCS + j] = v;
                sumD += (double)v;
            }
        sumD = group_sum<LPC>(sumD);
        const double vconst = fma(-P.lnB, sumD, ((double)R * (double)C) * P.B);
        ChainState s;
        const double* q_in = A.q_in + (size_t)field * 3;
        s.f = n ? q_in[0] : 0.0;
        s.x = n ? q_in[1] : 0.0;
        s.y = n ? q_in[2] : 0.0;
        s.pf = s.px = s.py = 0.0;
        if (A.p_in && n) {
            s.pf = A.p_in[(size_t)field * 3];
            s.px = A.p_in[(size_t)field * 3 + 1];
            s.py = A.p_in[(size_t)field * 3 + 2];
        }
        __syncwarp();
        const bool writer = live && sub == 0;
        double g_ff2 = A.g_ff2;
        ChainConst K = make_chain_const(P, g_ff2, h, A.delta);
        int cp = 0, cq = 0;

        if (MODE == MODE_EVAL) {
            chain_eval<LPC, NCS, true, DT, PT>(P, sD, rt, ltab, sub, vconst, s);
            refresh_metric(K, s);
            double V, T;
            chain_energies(P, K, s, A.f_pos, ltab, V, T);
            const Metric m = metric_of(P, s.f, g_ff2);  // reference-order formulas for the reported H, H'
            if (writer) {
                const size_t o = (size_t)field * 3;
                if (A.V_out) A.V_out[field] = V;
                if (A.grad_out) {
                    A.grad_out[o] = s.gf + (P.use_prior ? P.alpha / s.f : 0.0);
                    A.grad_out[o + 1] = s.gx;
                    A.grad_out[o + 2] = s.gy;
                }
                if (A.H_out) { A.H_out[o] = m.Hff; A.H_out[o + 1] = m.Hxx; A.H_out[o + 2] = m.Hxx; }
                if (A.Hgrad_out) { A.Hgrad_out[o] = m.dHff; A.Hgrad_out[o + 1] = m.dHxx; A.Hgrad_out[o + 2] = m.dHxx; }
            }
        } else if (MODE == MODE_STEP) {
            chain_eval<LPC, NCS, false, DT, PT>(P, sD, rt, ltab, sub, vconst, s);
            refresh_metric(K, s);
            for (int t = 0; t < A.nsteps; ++t) chain_step<LPC, NCS, DT, PT>(P, K, sD, rt, ltab, sub, vconst, s, A.counter_max, false, cp, cq);
            if (writer) {
                const size_t o = (size_t)field * 3;
                A.q_out[o] = s.f; A.q_out[o + 1] = s.x; A.q_out[o + 2] = s.y;
                A.p_out[o] = s.pf; A.p_out[o + 1] = s.px; A.p_out[o + 2] = s.py;
                if (A.fp_counts) { A.fp_counts[2 * field] = cp; A.fp_counts[2 * field + 1] = cq; }
            }
        } else if (MODE == MODE_SINGLE) {
            const size_t rows = (size_t)A.nsteps + 1;
            chain_eval<LPC, NCS, true, DT, PT>(P, sD, rt, ltab, sub, vconst, s);
            refresh_metric(K, s);
            double V0, T0;
            chain_energies(P, K, s, A.f_pos, ltab, V0, T0);
            if (writer) {
                const size_t o = (size_t)field * rows * 3;
                A.q_chain[o] = s.f; A.q_chain[o + 1] = s.x; A.q_chain[o + 2] = s.y;
                A.p_chain[o] = s.pf; A.p_chain[o + 1] = s.px; A.p_chain[o + 2] = s.py;
                A.E_chain[field * rows] = 0.0; A.V_chain[field * rows] = 0.0; A.T_chain[field * rows] = 0.0;
            }
            for (int t = 1; t <= A.nsteps; ++t) {
                chain_step<LPC, NCS, DT, PT>(P, K, sD, rt, ltab, sub, vconst, s, A.counter_max, true, cp, cq);
                double V, T;
                chain_energies(P, K, s, A.f_pos, ltab, V, T);
                if (writer) {
                    const size_t o = ((size_t)field * rows + t) * 3;
                    A.q_chain[o] = s.f; A.q_chain[o + 1] = s.x; A.q_chain[o + 2] = s.y;
                    A.p_chain[o] = s.pf; A.p_chain[o + 1] = s.px; A.p_chain[o + 2] = s.py;
                    const double dV = V - V0, dT = T - T0;
                    A.V_chain[field * rows + t] = dV;
                    A.T_chain[field * rows + t] = dT;
                    A.E_chain[field * rows + t] = dV + dT;
                }
            }
        } else {  // MODE_RUN
            const size_t rows = (size_t)A.n_rows;
            const int L = A.niter + 1;
            const int Lc = (L + n_chunks - 1) / n_chunks;
            const int l0 = chunk * Lc, l1 = min(L, l0 + Lc);
            const int grp_id = base / GPW;
            int n_acc = 0;
            if (chunk == 0) {
                chain_eval<LPC, NCS, true, DT, PT>(P, sD, rt, ltab, sub, vconst, s);
            } else {
                // wait until the previous chunk of this group has published its state (bounded spin: a scheduler
                // fault must not hang the device)
                // (the host caps the grid at the resident warp count, so the producer of chunk-1 is always on the device
                // when this context has the GPU to itself; on a shared GPU the spin is bounded instead)
                int ready = 1;
                if (lane == 0) {
                    const long long t0 = clock64();
                    while (*((volatile int*)A.sched_done + grp_id) < chunk) {
                        if (*((volatile int*)A.sched_err) != 0 || clock64() - t0 > 120000000000LL) {  // ~60 s
                            atomicExch(A.sched_err, 1);
                            ready = 0;
                            break;
                        }
                        __nanosleep(200);
                    }
                }
                ready = __shfl_sync(0xffffffffu, ready, 0);
                // a chunk whose predecessor never arrived is dropped (no stale state is advanced, no rows are written);
                // the host reports the scheduler fault
                if (!ready) continue;
                __threadfence();
                const double* st = A.sched_state + (size_t)field * 8;
                s.f = __ldcg(st); s.x = __ldcg(st + 1); s.y = __ldcg(st + 2);
                s.gf = __ldcg(st + 3); s.gx = __ldcg(st + 4); s.gy = __ldcg(st + 5);
                s.Vpix = __ldcg(st + 6);
                n_acc = (int)__ldcg(st + 7);
            }
            for (int l = l0; l < l1; ++l) {
                if (A.gff2_sched && A.n_gff2 > 0) {
                    g_ff2 = A.gff2_sched[min(l, A.n_gff2 - 1)];  // stays at the last entry once the schedule ends
                    K = make_chain_const(P, g_ff2, h, A.delta);
                }
                refresh_metric(K, s);
                double z[3];
                if (A.normals) {
                    const double* zp = A.normals + ((size_t)field * L + l) * 3;
                    z[0] = zp[0]; z[1] = zp[1]; z[2] = zp[2];
                } else {
                    philox_normals3_tab(A.seed, A.philox_field(field), (uint32_t)l, 0u, ltab, z);
                }
                {
                    const double sxx = sqrt(rcp_fast(s.ihxx));
                    s.pf = z[0] * sqrt(rcp_fast(s.u));
                    s.px = z[1] * sxx;
                    s.py = z[2] * sxx;
                }
                const ChainState s0 = s;
                double V0, T0;
                chain_energies(P, K, s, A.f_pos, ltab, V0, T0);
                const double E0 = V0 + T0;
                const bool keep = (l % A.chain_stride) == 0;
                const size_t row = (size_t)field * rows + (size_t)(l / A.chain_stride);
                if (keep && writer) {
                    if (A.q_chain) { A.q_chain[row * 3] = s.f; A.q_chain[row * 3 + 1] = s.x; A.q_chain[row * 3 + 2] = s.y; }
                    if (A.p_chain) { A.p_chain[row * 3] = s.pf; A.p_chain[row * 3 + 1] = s.px; A.p_chain[row * 3 + 2] = s.py; }
                    if (A.E_chain) A.E_chain[row] = E0;
                    if (A.V_chain) A.V_chain[row] = V0;
                    if (A.T_chain) A.T_chain[row] = T0;
                }
                for (int t = 0; t < A.nsteps; ++t)
                    chain_step<LPC, NCS, DT, PT>(P, K, sD, rt, ltab, sub, vconst, s, A.counter_max, t == A.nsteps - 1, cp, cq);
                double V1, T1;
                chain_energies(P, K, s, A.f_pos, ltab, V1, T1);
                const double dE = (V1 + T1) - E0;
                const double lnu = A.lnu ? A.lnu[(size_t)field * L + l] : philox_lnu_tab(A.seed, A.philox_field(field), (uint32_t)l, ltab);
                const bool accept = (dE < 0.0) || (lnu < -dE);
                if (keep && writer && A.A_chain) A.A_chain[row] = accept ? 1 : 0;
                if (accept) {
                    ++n_acc;
                } else {
                    s.f = s0.f; s.x = s0.x; s.y = s0.y;
                    s.gf = s0.gf; s.gx = s0.gx; s.gy = s0.gy;
                    s.Vpix = s0.Vpix;
                }
            }
            if (l1 >= L) {
                if (writer) {
                    if (A.q_out) { A.q_out[(size_t)field * 3] = s.f; A.q_out[(size_t)field * 3 + 1] = s.x; A.q_out[(size_t)field * 3 + 2] = s.y; }
                    if (A.accept_rate) A.accept_rate[field] = (double)n_acc / (double)L;
                }
            } else {
                if (writer) {
                    double* st = A.sched_state + (size_t)field * 8;
                    __stcg(st, s.f); __stcg(st + 1, s.x); __stcg(st + 2, s.y);
                    __stcg(st + 3, s.gf); __stcg(st + 4, s.gx); __stcg(st + 5, s.gy);
                    __stcg(st + 6, s.Vpix);
                    __stcg(st + 7, (double)n_acc);
                }
                __threadfence();
                __syncwarp();
                if (lane == 0) atomicExch(A.sched_done + grp_id, chunk + 1);
            }
        }
    }
}

}  // namespace srhmc
