// CTA-per-field resident RHMC kernel (sm_100a).
//
// One thread block owns one field (one chain): the data image D and the model/residual image stay in shared
// memory for the whole launch, star state (q, p, cached pixel gradient) too, and every leapfrog step, momentum
// refresh, energy and Metropolis test of the chain runs device-side (no host round trip).
//
// Pixel work per gradient evaluation (reference: base_class.dVdq, sampler_RHMC.py:365-425):
//   sweep 1  tables  ex_k[i] = f_k exp(-(i+.5-x_k)^2/2s^2),  ey_k[j] = exp(-(j+.5-y_k)^2/2s^2)/(2 pi s^2)
//                    (separable PSF; built with the exact two-term Gaussian recurrence, 3 exps per star-axis)
//            render  Lambda = B + sum_k ex_k[i] ey_k[j]     register-tiled gather, MRxMC pixels per thread,
//                    deterministic star order; rho = D/Lambda - 1 written back in place (+ V = sum(L - D ln L))
//   sweep 2  grads   one warp per star: column sums c0_j = sum_i rho_ij ex_i, c1_j = sum_i rho_ij ex_i dx_i,
//                    then g_f = -sum_j ey_j c0_j, g_x = -(f/s^2) sum_j ey_j c1_j, g_y = -(f/s^2) sum_j ey_j dy_j c0_j
//                    finished with warp shuffles.
// Scalar work (metric, implicit fixed points, reflections; sampler_RHMC.py:229-292, 448-492, 522-566) is one
// thread per star with a CTA-wide vote per fixed-point iteration (the reference's field-wide stop rule).
#pragma once
#include <cfloat>
#include <math_constants.h>

#include "common.cuh"

namespace srhmc {

struct SmemLayout {
    size_t q, p, g, a1, a2, red, D, L, L2, tabx, taby, span, total;
};

template <typename T>
__host__ __device__ inline SmemLayout make_layout(const FieldParams& P, bool d_in_smem) {
    SmemLayout s;
    size_t o = 0;
    const size_t S = 3 * (size_t)P.Nmax * sizeof(double);
    auto take = [&](size_t bytes) {
        size_t at = o;
        o += (bytes + 15) & ~(size_t)15;
        return at;
    };
    s.q = take(S);
    s.p = take(S);
    s.g = take(S);
    if (!P.v3) {
        s.a1 = take(S);
        s.a2 = take(S);
    }
    s.red = take(8 * 32 * sizeof(double));
    s.D = take(d_in_smem ? (size_t)P.R * P.C * sizeof(T) : 0);
    s.L = take((size_t)P.R * P.C * sizeof(T));
    s.L2 = take(P.hess ? (size_t)P.R * P.C * sizeof(T) : 0);  // 1/Lambda image of the Hessian path (samplers.py:828-927)
    if (P.v3) {
        // compact tables of ALL stars: rs pairs {ex, ex dx} + cs entries f ey per star.  The fixed-point scratch a1 / a2
        // is only live between two evaluations and the tables only inside one, so they share the space.
        const size_t rows = (size_t)P.Nmax * P.rs * 2 * sizeof(T), cols = (size_t)P.Nmax * P.cs * sizeof(T);
        s.tabx = take(rows > 2 * S ? rows : 2 * S);
        s.taby = take(cols);
        s.span = take((size_t)P.Nmax * 2 * sizeof(int));
        s.a1 = s.tabx;
        s.a2 = s.tabx + S;
    } else {
        s.tabx = take((size_t)P.Kc * P.sx * sizeof(T));
        s.taby = take((size_t)P.Kc * P.sy * sizeof(T));
        s.span = take((size_t)P.Kc * 4 * sizeof(short));
    }
    s.total = o;
    return s;
}

template <typename T>
struct Ctx {
    const FieldParams* P;
    T* sD;         // nullptr when D is read from global / L2
    T* sL;
    T* tabx;
    T* taby;
    const T* gD;   // this field's image in global memory
    T* sL2;        // 1/Lambda image (Hessian path), nullptr otherwise
    const double* bg;  // optional per-pixel background replacing the constant B (HMC_find_best_dt's model_data)
    bool hess_out; // render writes rho0 = D/Lambda to sL and 1/Lambda to sL2 instead of rho = D/Lambda - 1
    double *q, *p, *g, *a1, *a2, *red;
    short* span;
    int N;
    double g_ff2, beta, h;
};

template <typename T, int N> struct VecLoad;
template <> struct VecLoad<double, 1> { static __device__ __forceinline__ void ld(const double* p, double* o) { o[0] = p[0]; } };
template <> struct VecLoad<double, 2> { static __device__ __forceinline__ void ld(const double* p, double* o) {
    const double2 v = *reinterpret_cast<const double2*>(p); o[0] = v.x; o[1] = v.y; } };
template <> struct VecLoad<double, 4> { static __device__ __forceinline__ void ld(const double* p, double* o) {
    const double2 a = *reinterpret_cast<const double2*>(p); const double2 b = *reinterpret_cast<const double2*>(p + 2);
    o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y; } };
template <> struct VecLoad<float, 1> { static __device__ __forceinline__ void ld(const float* p, float* o) { o[0] = p[0]; } };
template <> struct VecLoad<float, 2> { static __device__ __forceinline__ void ld(const float* p, float* o) {
    const float2 v = *reinterpret_cast<const float2*>(p); o[0] = v.x; o[1] = v.y; } };
template <> struct VecLoad<float, 4> { static __device__ __forceinline__ void ld(const float* p, float* o) {
    const float4 v = *reinterpret_cast<const float4*>(p); o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; } };

// ---------------------------------------------------------------------------------------------- tables
// One thread per (star, axis).  Exact recurrence: e(u+1) = e(u) r(u), r(u+1) = r(u) exp(-1/s^2), run outwards
// from the pixel that contains the star so the rounding error stays at a few ulp where the PSF matters.
// Measured alternatives (C4, 592 fields x 204 stars): this serial build leaves 80% of the CTA idle at the barriers
// around it (ncu: 37% of stall samples at the phase boundaries, 8% in the zero fill), but a fully parallel build
// with one direct exponential per in-span entry was SLOWER (437 vs 588 M star-steps/s): the kernel is also
// instruction-bound, and 2300 exponentials per chunk cost more issue slots than the idle time they remove.  The
// next step is a strided recurrence with a few lanes per star-axis (as in chain_kernel.cuh) and a single table
// build per evaluation.
// fmode: where the star's flux goes.  0: nowhere (gradient pass of a multi-chunk field), 1: into the row table (render
// pass), 2: into the COLUMN table -- one build then serves both the render (f ex ey) and the gradient pass, whose sums
// carry the factor f and are divided by it at the end (grad_chunk<T, true>).
template <typename T>
__device__ void build_tables(const Ctx<T>& c, int k0, int nk, int fmode) {
    const FieldParams& P = *c.P;
    for (int t = threadIdx.x; t < 2 * nk; t += blockDim.x) {
        const int kk = t >> 1, axis = t & 1, k = k0 + kk;
        const double coord = c.q[3 * k + 1 + axis];
        const int n = axis ? P.C : P.R;
        const int stride = axis ? P.sy : P.sx;
        T* tab = (axis ? c.taby : c.tabx) + (size_t)kk * stride;
        const double scale = axis ? (fmode == 2 ? P.norm * c.q[3 * k] : P.norm) : (fmode == 1 ? c.q[3 * k] : 1.0);
        const double fl = floor(coord);
        int m = 0;
        if (fl > 0.0) m = (fl > (double)(n - 1)) ? n - 1 : (int)fl;
        int lo = 0, hi = n - 1;
        if (P.rad > 0) {
            lo = max(0, m - P.rad);
            hi = min(n - 1, m + P.rad);
        }
        for (int i = 0; i < lo; ++i) tab[i] = (T)0;
        for (int i = hi + 1; i < stride; ++i) tab[i] = (T)0;
        const double u = ((double)m + 0.5) - coord;
        const double e0 = exp(-(u * u) * P.inv2s2) * scale;
        tab[m] = (T)e0;
        double e = e0, r = exp(-(2.0 * u + 1.0) * P.inv2s2);
        for (int i = m + 1; i <= hi; ++i) {
            e *= r;
            r *= P.c2;
            tab[i] = (T)e;
        }
        e = e0;
        r = exp((2.0 * u - 1.0) * P.inv2s2);
        for (int i = m - 1; i >= lo; --i) {
            e *= r;
            r *= P.c2;
            tab[i] = (T)e;
        }
        c.span[4 * kk + 2 * axis] = (short)lo;
        c.span[4 * kk + 2 * axis + 1] = (short)hi;
    }
}

// ---------------------------------------------------------------------------------------------- render
template <typename T, int MR, int MC>
__device__ void render_chunk(const Ctx<T>& c, int nk, bool first, bool last, bool want_V, double& vacc) {
    const FieldParams& P = *c.P;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    constexpr int TR = 8 * MR, TC = 4 * MC;
    const int ntr = (P.R + TR - 1) / TR, ntc = (P.C + TC - 1) / TC;
    for (int wt = warp; wt < ntr * ntc; wt += nwarps) {
        const int ti = (wt / ntc) * TR, tj = (wt % ntc) * TC;
        const int ib = ti + (lane >> 2) * MR, jb = tj + (lane & 3) * MC;
        T acc[MR][MC];
#pragma unroll
        for (int r = 0; r < MR; ++r)
#pragma unroll
            for (int cc = 0; cc < MC; ++cc) {
                const bool ok = (ib + r < P.R) && (jb + cc < P.C);
                acc[r][cc] = first ? ((c.bg && ok) ? (T)c.bg[(ib + r) * P.C + jb + cc] : (T)P.B)
                                   : (ok ? c.sL[(ib + r) * P.C + jb + cc] : (T)0);
            }
        auto accumulate = [&](int kk) {
            T fx[MR], fy[MC];
            VecLoad<T, MR>::ld(c.tabx + (size_t)kk * P.sx + ib, fx);
            VecLoad<T, MC>::ld(c.taby + (size_t)kk * P.sy + jb, fy);
#pragma unroll
            for (int r = 0; r < MR; ++r)
#pragma unroll
                for (int cc = 0; cc < MC; ++cc) acc[r][cc] = fma(fx[r], fy[cc], acc[r][cc]);
        };
        if (P.rad == 0) {
#pragma unroll 2
            for (int kk = 0; kk < nk; ++kk) accumulate(kk);
        } else {
            for (int kb = 0; kb < nk; kb += 32) {
                const int kk = kb + lane;
                bool hit = false;
                if (kk < nk) {
                    const short4 sp = *reinterpret_cast<const short4*>(c.span + 4 * kk);
                    hit = (sp.x <= ti + TR - 1) && (sp.y >= ti) && (sp.z <= tj + TC - 1) && (sp.w >= tj);
                }
                unsigned mask = __ballot_sync(0xffffffffu, hit);
                while (mask) {
                    const int b = __ffs(mask) - 1;
                    mask &= mask - 1;
                    accumulate(kb + b);
                }
            }
        }
#pragma unroll
        for (int r = 0; r < MR; ++r)
#pragma unroll
            for (int cc = 0; cc < MC; ++cc) {
                const int i = ib + r, j = jb + cc;
                if (i < P.R && j < P.C) {
                    const int pix = i * P.C + j;
                    if (!last) {
                        c.sL[pix] = acc[r][cc];
                    } else {
                        const T lam = acc[r][cc];
                        const T d = c.sD ? c.sD[pix] : c.gD[pix];
                        const T il = rcp_fast(lam);
                        if (c.hess_out) {
                            c.sL[pix] = d * il;  // rho0 = D/Lambda
                            c.sL2[pix] = il;
                        } else {
                            c.sL[pix] = fma(d, il, (T)-1);  // rho = D/Lambda - 1
                        }
                        if (want_V) {
                            const double ld = (double)lam;
                            vacc += ld - (double)d * log(ld);
                        }
                    }
                }
            }
    }
}

// ---------------------------------------------------------------------------------------------- gradients
// FY: the column table holds f ey (build_tables fmode 2)
template <typename T, bool FY = false>
__device__ void grad_chunk(const Ctx<T>& c, int k0, int nk) {
    const FieldParams& P = *c.P;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int kk = warp; kk < nk; kk += nwarps) {
        const int k = k0 + kk;
        const double f = c.q[3 * k], x = c.q[3 * k + 1], y = c.q[3 * k + 2];
        const short4 sp = *reinterpret_cast<const short4*>(c.span + 4 * kk);
        const int i0 = sp.x, i1 = sp.y, j0 = sp.z, j1 = sp.w;
        const T* tx = c.tabx + (size_t)kk * P.sx;
        const T* ty = c.taby + (size_t)kk * P.sy;
        T gf = 0, gx = 0, gy = 0;
        for (int jc = j0; jc <= j1; jc += 32) {
            const int j = jc + lane;
            const bool ok = j <= j1;
            const int jj = ok ? j : j1;
            const T ey = ok ? ty[jj] : (T)0;
            const T eydy = ey * (T)(((double)jj + 0.5) - y);
            const T* Lp = c.sL + jj;
            T c0a = 0, c1a = 0, c0b = 0, c1b = 0;
            int i = i0;
            T dxa = (T)(((double)i0 + 0.5) - x), dxb = (T)(((double)i0 + 1.5) - x);  // row offsets, advanced by 2 per pass
            for (; i + 1 <= i1; i += 2) {
                const T ra = Lp[i * P.C], rb = Lp[(i + 1) * P.C];
                const T ea = tx[i], eb = tx[i + 1];
                c0a = fma(ra, ea, c0a);
                c1a = fma(ra, ea * dxa, c1a);
                c0b = fma(rb, eb, c0b);
                c1b = fma(rb, eb * dxb, c1b);
                dxa += (T)2;
                dxb += (T)2;
            }
            if (i <= i1) {
                const T ra = Lp[i * P.C];
                const T ea = tx[i];
                c0a = fma(ra, ea, c0a);
                c1a = fma(ra, ea * dxa, c1a);
            }
            const T c0 = c0a + c0b, c1 = c1a + c1b;
            gf = fma(ey, c0, gf);
            gx = fma(ey, c1, gx);
            gy = fma(eydy, c0, gy);
        }
        // lanes -> one value; accumulate the final reduction in double for both builds
        double df = warp_sum((double)gf), dx = warp_sum((double)gx), dy = warp_sum((double)gy);
        if (lane == 0) {
            c.g[3 * k] = FY ? -df / f : -df;
            c.g[3 * k + 1] = FY ? -dx * P.inv_s2 : -dx * f * P.inv_s2;
            c.g[3 * k + 2] = FY ? -dy * P.inv_s2 : -dy * f * P.inv_s2;
        }
    }
}

// ---------------------------------------------------------------------------------------------- compact-table path ("v3")
// Patch-limited evaluation for crowded fields (BASELINE configs[2..3]): same sums as above (sampler_RHMC.py:365-425 with
// the PSF cut to (2 rad + 1)^2 pixels), organised so that a 204-star 64x64 field needs ONE table build, three CTA barriers
// and no bounds handling in the hot loops:
//   tables  one thread per (star, axis).  Rows: TL = 2 rad + 1 pairs {ex, ex dx} for the image rows [w0, w0 + TL) with
//           w0 = clamp(m - rad, 0, R - TL) (m = pixel holding the star), zero outside the patch, one zero guard pair on each
//           side.  Columns: TL + 1 entries f ey / (2 pi s^2) for the columns [je, je + TL + 1), je even (16-byte aligned
//           residual pairs), zero outside the patch, three zero guards on each side.  The windows always lie inside the image.
//   render  a warp owns 8 rows x 32 columns of Lambda in registers (2 x 4 pixels per lane); stars whose window meets the
//           block are found with one ballot per 32 stars; rho = D / Lambda - 1 goes to shared memory.
//   gather  16 lanes per star (two stars per warp): a lane owns two adjacent columns and walks the TL rows with one
//           16-byte load of the residual pair and one broadcast load of {ex, ex dx} per row (4 FMAs), then the three
//           sums are folded across the 16 lanes with five shuffles.
template <typename T> struct Pair;
template <> struct Pair<double> { typedef double2 type; static __device__ __forceinline__ double2 make(double a, double b) { return make_double2(a, b); } };
template <> struct Pair<float> { typedef float2 type; static __device__ __forceinline__ float2 make(float a, float b) { return make_float2(a, b); } };

template <typename T>
__device__ void build_tables_v3(const Ctx<T>& c) {
    typedef typename Pair<T>::type P2;
    const FieldParams& P = *c.P;
    const int TL = P.tl, CW = P.tl + 1;
    int2* span = reinterpret_cast<int2*>(c.span);
    for (int t = threadIdx.x; t < 2 * c.N; t += blockDim.x) {
        const int k = t >> 1, axis = t & 1;
        const double coord = c.q[3 * k + 1 + axis];
        const int n = axis ? P.C : P.R;
        const double fl = floor(coord);
        int m = 0;
        if (fl > 0.0) m = (fl > (double)(n - 1)) ? n - 1 : (int)fl;
        const int lo = max(0, m - P.rad), hi = min(n - 1, m + P.rad);
        const double u = ((double)m + 0.5) - coord;
        const double scale = axis ? P.norm * c.q[3 * k] : 1.0;
        const double e0 = exp(-(u * u) * P.inv2s2) * scale;
        double eu = e0, ed = e0, ru = exp(-(2.0 * u + 1.0) * P.inv2s2), rd = exp((2.0 * u - 1.0) * P.inv2s2);
        if (axis == 0) {
            const int w0 = min(lo, P.R - TL);
            P2* rt = reinterpret_cast<P2*>(c.tabx) + (k * P.rs + 1 - w0);  // rt[i]: image row i
            const P2 zero = Pair<T>::make((T)0, (T)0);
            for (int i = w0 - 1; i < lo; ++i) rt[i] = zero;                 // leading guard (+ rows cut by the image edge)
            for (int i = hi + 1; i < w0 - 1 + P.rs; ++i) rt[i] = zero;      // trailing guard(s)
            rt[m] = Pair<T>::make((T)e0, (T)(e0 * u));
            for (int s = 1; s <= P.rad; ++s) {
                eu *= ru; ru *= P.c2;
                ed *= rd; rd *= P.c2;
                if (m + s <= hi) rt[m + s] = Pair<T>::make((T)eu, (T)(eu * (u + (double)s)));
                if (m - s >= lo) rt[m - s] = Pair<T>::make((T)ed, (T)(ed * (u - (double)s)));
            }
            span[k].x = w0 - 1;   // image row of pair 0
        } else {
            const int je = min(lo & ~1, P.C - CW);
            T* ct = c.taby + (k * P.cs + 3 - je);  // ct[j]: image column j
            for (int j = je - 3; j < lo; ++j) ct[j] = (T)0;
            for (int j = hi + 1; j < je - 3 + P.cs; ++j) ct[j] = (T)0;
            ct[m] = (T)e0;
            for (int s = 1; s <= P.rad; ++s) {
                eu *= ru; ru *= P.c2;
                ed *= rd; rd *= P.c2;
                if (m + s <= hi) ct[m + s] = (T)eu;
                if (m - s >= lo) ct[m - s] = (T)ed;
            }
            span[k].y = je - 3;   // image column of entry 0
        }
    }
}

template <typename T>
__device__ void render_v3(const Ctx<T>& c, bool want_V, double& vacc) {
    typedef typename Pair<T>::type P2;
    const FieldParams& P = *c.P;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int TL = P.tl, CW = P.tl + 1;
    const int ntr = (P.R + 7) >> 3, ntc = (P.C + 31) >> 5;
    const P2* rowtab = reinterpret_cast<const P2*>(c.tabx);
    const T* coltab = c.taby;
    const int2* span = reinterpret_cast<const int2*>(c.span);   // (image row of pair 0, image column of entry 0)
    const int rs = P.rs, cs = P.cs;
    for (int wt = warp; wt < ntr * ntc; wt += nwarps) {
        const int ti = (wt / ntc) * 8, tj = (wt % ntc) * 32;
        const int ib = ti + (lane >> 3) * 2, jb = tj + (lane & 7) * 4;
        T acc[2][4];
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) acc[r][cc] = (T)P.B;
        // one hit = one star whose window meets this block: 2 row pairs + 4 column entries -> 8 FMAs per lane
        auto hit_load = [&](int k, bool on, P2& r0, P2& r1, T (&f)[4]) -> bool {
            const int2 sp = span[k];
            const int orow = ib - sp.x, ocol = jb - sp.y;   // pair / entry index of the lane's first row / column
            const bool in = on && (unsigned)orow <= (unsigned)TL && (unsigned)ocol <= (unsigned)(CW + 2);
            if (in) {
                const P2* rp = rowtab + (k * rs + orow);
                const T* cp = coltab + (k * cs + ocol);
                r0 = rp[0]; r1 = rp[1];
                f[0] = cp[0]; f[1] = cp[1]; f[2] = cp[2]; f[3] = cp[3];
            }
            return in;
        };
        auto hit_fma = [&](const P2& r0, const P2& r1, const T (&f)[4]) {
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                acc[0][cc] = fma(r0.x, f[cc], acc[0][cc]);
                acc[1][cc] = fma(r1.x, f[cc], acc[1][cc]);
            }
        };
        for (int kb = 0; kb < c.N; kb += 32) {
            const int kk = kb + lane;
            bool hit = false;
            if (kk < c.N) {
                const int2 sp = span[kk];
                hit = (sp.x < ti + 7) && (sp.x + TL >= ti) && (sp.y + 3 <= tj + 31) && (sp.y + 3 + CW > tj);
            }
            unsigned mask = __ballot_sync(0xffffffffu, hit);
            // two hits per trip: their loads are in flight together
            while (mask) {
                const int k0 = kb + __ffs(mask) - 1;
                mask &= mask - 1;
                const bool two = mask != 0;
                const int k1 = two ? kb + __ffs(mask) - 1 : k0;
                mask &= mask - 1;
                P2 a0, a1, b0, b1;
                T fa[4], fb[4];
                const bool ina = hit_load(k0, true, a0, a1, fa);
                const bool inb = hit_load(k1, two, b0, b1, fb);
                if (ina) hit_fma(a0, a1, fa);
                if (inb) hit_fma(b0, b1, fb);
            }
        }
        // residual (and the pixel potential on request)
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int i = ib + r;
            if (i >= P.R) continue;
            if (jb + 3 < P.C) {
                const int pix = i * P.C + jb;
                T d[4];
                if (c.sD) VecLoad<T, 4>::ld(c.sD + pix, d); else VecLoad<T, 4>::ld(c.gD + pix, d);
                T rho[4];
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    rho[cc] = fma(d[cc], rcp_fast(acc[r][cc]), (T)-1);
                    if (want_V) {
                        const double ld = (double)acc[r][cc];
                        vacc += ld - (double)d[cc] * log(ld);
                    }
                }
                P2* o = reinterpret_cast<P2*>(c.sL + pix);
                o[0] = Pair<T>::make(rho[0], rho[1]);
                o[1] = Pair<T>::make(rho[2], rho[3]);
            } else {
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    const int j = jb + cc;
                    if (j >= P.C) continue;
                    const int pix = i * P.C + j;
                    const T lam = acc[r][cc];
                    const T d = c.sD ? c.sD[pix] : c.gD[pix];
                    c.sL[pix] = fma(d, rcp_fast(lam), (T)-1);
                    if (want_V) {
                        const double ld = (double)lam;
                        vacc += ld - (double)d * log(ld);
                    }
                }
            }
        }
    }
}

// Two stars per warp trip (one per half-warp): lane hl of a half owns the columns je + 2 hl, je + 2 hl + 1 of its star's
// window and walks all TL rows.
template <typename T>
__device__ void gather_v3(const Ctx<T>& c) {
    typedef typename Pair<T>::type P2;
    const FieldParams& P = *c.P;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int half = lane >> 4, hl = lane & 15;
    const int TL = P.tl, CW = P.tl + 1;
    const P2* rowtab = reinterpret_cast<const P2*>(c.tabx);
    const int2* span = reinterpret_cast<const int2*>(c.span);
    const int rstride = P.C >> 1;
    const int cofs = 3 + min(2 * hl, CW);           // lanes 13..15 read the zero guards
    const bool dead = 2 * hl >= CW;
    const int npairs = (c.N + 1) >> 1;
    for (int pr = warp; pr < npairs; pr += nwarps) {
        const int kraw = 2 * pr + half;
        const bool live = kraw < c.N;
        const int k = live ? kraw : c.N - 1;
        const int2 sp = span[k];
        const int w0 = sp.x + 1, je = sp.y + 3;
        const T* cp = c.taby + (k * P.cs + cofs);
        const T fy0 = cp[0], fy1 = cp[1];
        const int col = min(je + 2 * hl, P.C - 2);  // always inside the image, 16-byte aligned
        const P2* rho = reinterpret_cast<const P2*>(c.sL + (w0 * P.C + col));
        const P2* rp = rowtab + (k * P.rs + 1);
        T a0 = 0, a1 = 0, b0 = 0, b1 = 0;
#pragma unroll 5
        for (int r = 0; r < TL; ++r) {
            const P2 e = rp[r];
            const P2 v = rho[r * rstride];
            a0 = fma(v.x, e.x, a0);
            a1 = fma(v.x, e.y, a1);
            b0 = fma(v.y, e.x, b0);
            b1 = fma(v.y, e.y, b1);
        }
        const double f = c.q[3 * k], y = c.q[3 * k + 2];
        const double dy0 = ((double)(je + 2 * hl) + 0.5) - y;
        // per-lane contributions of its two columns (the column table carries f)
        double sf = (double)fy0 * (double)a0 + (double)fy1 * (double)b0;
        double sx = (double)fy0 * (double)a1 + (double)fy1 * (double)b1;
        double sy = ((double)fy0 * dy0) * (double)a0 + ((double)fy1 * (dy0 + 1.0)) * (double)b0;
        if (dead) sf = sx = sy = 0.0;
        // fold the three sums over the 16 lanes of the star: 2 + 1 + 1 + 1 shuffles
        const bool h8 = hl & 8;
        const double k0 = h8 ? sy : sf, k1 = h8 ? 0.0 : sx, t0 = h8 ? sf : sy, t1 = h8 ? sx : 0.0;
        const double x0 = k0 + __shfl_xor_sync(0xffffffffu, t0, 8), x1 = k1 + __shfl_xor_sync(0xffffffffu, t1, 8);
        // lanes 0-7: x0 = sum_f (pairs), x1 = sum_x; lanes 8-15: x0 = sum_y, x1 = 0
        const bool h4 = hl & 4;
        double yv = (h4 ? x1 : x0) + __shfl_xor_sync(0xffffffffu, h4 ? x0 : x1, 4);
        // lanes 0-3: sum_f, lanes 4-7: sum_x, lanes 8-11: sum_y, lanes 12-15: 0
        yv += __shfl_xor_sync(0xffffffffu, yv, 2);
        yv += __shfl_xor_sync(0xffffffffu, yv, 1);
        // g_f = -sum_f / f (reciprocal to 2^-60), g_x = -sum_x / s^2, g_y = -sum_y / s^2
        const double sc = (hl < 4) ? rcp_fast(f) : P.inv_s2;
        if (live && (hl & 3) == 0 && hl < 12) c.g[3 * k + (hl >> 2)] = -(yv * sc);
    }
}

// True in every thread when every star of the field has |f| >= the smallest normal T, so that grad_chunk<T, true> can
// divide the flux sum by f.  A zero flux (0/0) or a subnormal one (tables underflow) needs the two-pass branch.
template <typename T>
__device__ bool fluxes_normal(const Ctx<T>& c) {
    const double fmin = sizeof(T) == 8 ? (double)DBL_MIN : (double)FLT_MIN;
    int tiny = 0;
    for (int k = threadIdx.x; k < c.N; k += blockDim.x) tiny |= !(fabs(c.q[3 * k]) >= fmin);
    return !__syncthreads_or(tiny);
}

// Pixel part of V and dV/dq at the current c.q.  Returns sum(Lambda - D ln Lambda) in every thread when want_V.
// KV3: -1 = follow P.v3 at run time (generic kernels), 1 = the compact-table path only, 0 = the chunked tables only
template <typename T, int MR, int MC, int KV3 = -1>
__device__ double eval_pixels(const Ctx<T>& c, bool want_V) {
    const FieldParams& P = *c.P;
    const int nchunks = c.N > 0 ? (c.N + P.Kc - 1) / P.Kc : 1;
    double vacc = 0.0;
    if (KV3 == 1 || (KV3 < 0 && P.v3)) {
        build_tables_v3<T>(c);
        __syncthreads();
        render_v3<T>(c, want_V, vacc);
        __syncthreads();
        gather_v3<T>(c);
        __syncthreads();
    } else if (KV3 == 1) {
        // unreachable: the specialised kernel is only launched for compact-table contexts
    } else if (nchunks == 1 && c.N > 0 && fluxes_normal(c)) {
        // every star's tables fit at once: ONE build serves the render and the gradient pass (flux in the column table)
        build_tables<T>(c, 0, c.N, 2);
        __syncthreads();
        render_chunk<T, MR, MC>(c, c.N, true, true, want_V, vacc);
        __syncthreads();
        grad_chunk<T, true>(c, 0, c.N);
        __syncthreads();
    } else {
        for (int ch = 0; ch < nchunks; ++ch) {
            const int k0 = ch * P.Kc, nk = min(P.Kc, c.N - k0);
            build_tables<T>(c, k0, nk, 1);
            __syncthreads();
            render_chunk<T, MR, MC>(c, nk, ch == 0, ch == nchunks - 1, want_V, vacc);
            __syncthreads();
        }
        for (int ch = 0; ch < nchunks; ++ch) {
            const int k0 = ch * P.Kc, nk = min(P.Kc, c.N - k0);
            if (nk <= 0) break;
            build_tables<T>(c, k0, nk, 0);
            __syncthreads();
            grad_chunk<T>(c, k0, nk);
            __syncthreads();
        }
    }
    if (want_V) {
        double v[1] = {vacc};
        block_sum<1>(v, c.red);
        return v[0];
    }
    return 0.0;
}

// ---------------------------------------------------------------------------------------------- per-star scalars
// dV/dq of star k = pixel part + prior + repulsion (sampler_RHMC.py:404-418)
template <typename T>
__device__ __forceinline__ void total_grad(const Ctx<T>& c, int k, double& gf, double& gx, double& gy) {
    const FieldParams& P = *c.P;
    gf = c.g[3 * k];
    gx = c.g[3 * k + 1];
    gy = c.g[3 * k + 2];
    if (P.use_prior) gf = fma(P.alpha, rcp_fast(c.q[3 * k]), gf);   // per-step path: no FP64 division (2^-60 reciprocal)
    if (P.use_Vc) {
        const double x = c.q[3 * k + 1], y = c.q[3 * k + 2];
        double sx = 0.0, sy = 0.0;
        for (int j = 0; j < c.N; ++j) {
            const double dx = c.q[3 * j + 1] - x, dy = c.q[3 * j + 2] - y;
            double r = sqrt(dx * dx + dy * dy);
            if (fabs(r) < 1e-10) r = 1e32;
            const double ir = 1.0 / r;
            const double w = (P.vc_int >= 0) ? ipow(ir, P.vc_int + 2) : pow(ir, P.vc_pow + 2.0);
            sx += w * dx;
            sy += w * dy;
        }
        gx += c.beta * sx * P.vc_pow;
        gy += c.beta * sy * P.vc_pow;
    }
}

// sum_j R_kj^-pow for the repulsion potential (sampler_RHMC.py:340-349)
template <typename T>
__device__ __forceinline__ double vc_row(const Ctx<T>& c, int k) {
    const FieldParams& P = *c.P;
    const double x = c.q[3 * k + 1], y = c.q[3 * k + 2];
    double s = 0.0;
    for (int j = 0; j < c.N; ++j) {
        const double dx = c.q[3 * j + 1] - x, dy = c.q[3 * j + 2] - y;
        double r = sqrt(dx * dx + dy * dy);
        if (fabs(r) < 1e-10) r = 1e32;
        const double ir = 1.0 / r;
        s += (P.vc_int >= 0) ? ipow(ir, P.vc_int) : pow(ir, P.vc_pow);
    }
    return s;
}

struct Energies {
    double V, T;
};

// two CTA-wide maxima of the fixed-point iteration counts (rhmc_step): a corner of the reduction scratch that block_sum
// (at most 7 values wide here) never touches
template <typename T>
__device__ __forceinline__ int* fp_count_slots(const Ctx<T>& c) { return reinterpret_cast<int*>(c.red + 7 * 32); }

// V(q, f_pos) and T(p, H(q)) from the cached pixel potential (sampler_RHMC.py:294-363).
template <typename T>
__device__ Energies energies(const Ctx<T>& c, double Vpix, int f_pos, bool with_T) {
    const FieldParams& P = *c.P;
    double v[5] = {0, 0, 0, 0, 0};  // sum p^2/H, sum ln|H|, prior, repulsion, bad-count
    for (int k = threadIdx.x; k < c.N; k += blockDim.x) {
        const double f = c.q[3 * k], x = c.q[3 * k + 1], y = c.q[3 * k + 2];
        if (with_T) {
            kinetic_terms(metric_of(P, f, c.g_ff2), c.p[3 * k], c.p[3 * k + 1], c.p[3 * k + 2], v[0], v[1]);
        }
        if (P.use_prior) v[2] += P.alpha * log(f) + P.Vpc;
        if (P.use_Vc) v[3] += vc_row(c, k);
        bool bad = (f_pos && f < P.f_lim) || (x < -1.0) || (x > P.R + 1.0) || (y < -1.0) || (y > P.C + 1.0);
        v[4] += bad ? 1.0 : 0.0;
    }
    block_sum<5>(v, c.red);
    Energies e;
    e.T = (v[0] + v[1]) / 2.0;
    double V = Vpix;
    if (P.use_prior) V += v[2];
    if (P.use_Vc) V += 0.5 * c.beta * v[3];
    e.V = (v[4] > 0.0) ? CUDART_INF : V;
    return e;
}

// ---------------------------------------------------------------------------------------------- one leapfrog step
// base_class.RHMC_single_step (sampler_RHMC.py:522-566).  Requires c.g == pixel gradient at c.q on entry and
// leaves it so on exit.  All threads of the CTA must call it.
template <typename T, int MR, int MC, int KV3 = -1>
__device__ void rhmc_step(const Ctx<T>& c, double delta, int counter_max, bool want_V, double& Vpix, int* counts) {
    const FieldParams& P = *c.P;
    const double h = c.h;
    const int tid = threadIdx.x, nt = blockDim.x;

    // The per-star scalar code runs on N of the CTA's 512 threads while the others wait: it is pure latency, so the metric is
    // taken in its division-free form (metric_fast, common.cuh; 2^-60 reciprocals -- the iterates agree with the division
    // forms to rounding and the fixed-point counts are unchanged).
    const MetricK K = make_metric_k(P, c.g_ff2);
    // (1) p <- p - h dphi/dq(q); set up the p fixed point: a1[3k] = anchor rho_f, a2[3k] = -H_ff'/H_ff^2
    for (int k = tid; k < c.N; k += nt) {
        const MetricFast m = metric_fast(K, c.q[3 * k]);
        double gf, gx, gy;
        total_grad(c, k, gf, gx, gy);
        gf += m.tphi;
        const double pf = c.p[3 * k] - h * gf;
        c.p[3 * k] = pf;
        c.p[3 * k + 1] -= h * gx;
        c.p[3 * k + 2] -= h * gy;
        c.a1[3 * k] = pf;   // own slots only: the q fixed point below reuses a1 / a2 per component without a barrier
        c.a2[3 * k] = m.kap;
    }
    // (2) p' = rho - h dtau/dq(q, p)  until max|p - p'| <= delta   (only flux slots move)
    // (3) q' = sigma + h (p/H(sigma) + p/H(q))  until max|q - q'| <= delta
    // The reference stops each loop when the maximum over ALL stars meets the tolerance (sampler_RHMC.py:533,543).  The
    // per-star maps are contractions, so that count is the maximum of the per-star counts: every star first iterates to its
    // own convergence (phase A), the CTA takes the maximum (one barrier instead of one vote per iteration), and every star
    // continues to it (phase B) -- the same iterates, bit for bit, as iterating all stars together.
    int cnt_p = 0, cnt_q = 0;
    int* cmax = fp_count_slots(c);  // zero on entry (kernel start / the previous step)
    auto p_iter = [&](int k, double& pf) -> bool {
        const double pn = c.a1[3 * k] - h * (((pf * pf) * c.a2[3 * k]) / 2.0);
        const bool more = fabs(pf - pn) > delta;
        pf = pn;
        return more;
    };
    if (P.fp_mode == 0) {
        int own = 0;
        for (int k = tid; k < c.N; k += nt) {
            double pf = c.p[3 * k];
            int n = 0;
            while (n < counter_max) {
                const bool more = p_iter(k, pf);
                ++n;
                if (!more) break;
            }
            c.p[3 * k] = pf;
            c.g[3 * k] = (double)n;   // the pixel gradient is dead until the evaluation at the end of the step
            own = max(own, n);
        }
        own = __reduce_max_sync(0xffffffffu, own);
        if ((tid & 31) == 0 && own > 0) atomicMax(&cmax[0], own);
        __syncthreads();
        cnt_p = cmax[0];
        for (int k = tid; k < c.N; k += nt) {
            double pf = c.p[3 * k];
            for (int n = (int)c.g[3 * k]; n < cnt_p; ++n) p_iter(k, pf);
            c.p[3 * k] = pf;
        }
    } else {
        for (int k = tid; k < c.N; k += nt) {
            double pf = c.p[3 * k];
            int n = 0;
            while (n < counter_max) {
                const bool more = p_iter(k, pf);
                ++n;
                if (!more) break;
            }
            c.p[3 * k] = pf;
            cnt_p = max(cnt_p, n);
        }
    }
    // a1 = sigma, a2 = p/H(sigma): a thread only touches the slots of its own stars
    for (int k = tid; k < c.N; k += nt) {
        const double u0 = inv_hff_k(K, c.q[3 * k]), ih0 = inv_hxx_k(K, c.q[3 * k]);
        c.a1[3 * k] = c.q[3 * k];
        c.a1[3 * k + 1] = c.q[3 * k + 1];
        c.a1[3 * k + 2] = c.q[3 * k + 2];
        c.a2[3 * k] = c.p[3 * k] * u0;
        c.a2[3 * k + 1] = c.p[3 * k + 1] * ih0;
        c.a2[3 * k + 2] = c.p[3 * k + 2] * ih0;
    }
    auto q_iter = [&](int k, double& qf, double& qx, double& qy) -> bool {
        const double uq = inv_hff_k(K, qf), ihq = inv_hxx_k(K, qf);
        const double nf = c.a1[3 * k] + h * (c.a2[3 * k] + c.p[3 * k] * uq);
        const double nx = c.a1[3 * k + 1] + h * (c.a2[3 * k + 1] + c.p[3 * k + 1] * ihq);
        const double ny = c.a1[3 * k + 2] + h * (c.a2[3 * k + 2] + c.p[3 * k + 2] * ihq);
        const double d = fmax(fabs(qf - nf), fmax(fabs(qx - nx), fabs(qy - ny)));
        qf = nf;
        qx = nx;
        qy = ny;
        return d > delta;
    };
    {
        int own = 0;
        for (int k = tid; k < c.N; k += nt) {
            double qf = c.q[3 * k], qx = c.q[3 * k + 1], qy = c.q[3 * k + 2];
            int n = 0;
            while (n < counter_max) {
                const bool more = q_iter(k, qf, qx, qy);
                ++n;
                if (!more) break;
            }
            c.q[3 * k] = qf;
            c.q[3 * k + 1] = qx;
            c.q[3 * k + 2] = qy;
            c.g[3 * k] = (double)n;
            own = max(own, n);
        }
        if (P.fp_mode == 0) {
            own = __reduce_max_sync(0xffffffffu, own);
            if ((tid & 31) == 0 && own > 0) atomicMax(&cmax[1], own);
            __syncthreads();
            cnt_q = cmax[1];
            if (tid == 0) cmax[0] = 0;  // every thread read it before the barrier above
            for (int k = tid; k < c.N; k += nt) {
                double qf = c.q[3 * k], qx = c.q[3 * k + 1], qy = c.q[3 * k + 2];
                for (int n = (int)c.g[3 * k]; n < cnt_q; ++n) q_iter(k, qf, qx, qy);
                c.q[3 * k] = qf;
                c.q[3 * k + 1] = qx;
                c.q[3 * k + 2] = qy;
            }
        } else {
            cnt_q = own;
        }
    }
    // (4) p <- p - h dtau/dq(q, p) at the new q
    for (int k = tid; k < c.N; k += nt) {
        const MetricFast m = metric_fast(K, c.q[3 * k]);
        const double pf = c.p[3 * k];
        c.p[3 * k] = pf - h * (((pf * pf) * m.kap) / 2.0);
    }
    __syncthreads();
    if (tid == 0) cmax[1] = 0;  // read by every thread before the barrier above; next used after several more
    // (5) gradient at the new q, then p <- p - h dphi/dq(q)
    const double v = eval_pixels<T, MR, MC, KV3>(c, want_V);
    if (want_V) Vpix = v;
    for (int k = tid; k < c.N; k += nt) {
        const double f = c.q[3 * k], x = c.q[3 * k + 1], y = c.q[3 * k + 2];
        const MetricFast m = metric_fast(K, f);
        double gf, gx, gy;
        total_grad(c, k, gf, gx, gy);
        gf += m.tphi;
        double pf = c.p[3 * k] - h * gf, px = c.p[3 * k + 1] - h * gx, py = c.p[3 * k + 2] - h * gy;
        // (6) reflections (sampler_RHMC.py:554-564); positions are not clamped
        if (f < P.f_lim) pf *= -1.0;
        if ((x < 0.0) || (x > P.R - 1.0)) px *= -1.0;
        if ((y < 0.0) || (y > P.C - 1.0)) py *= -1.0;
        c.p[3 * k] = pf;
        c.p[3 * k + 1] = px;
        c.p[3 * k + 2] = py;
    }
    __syncthreads();
    if (counts) {
        counts[0] = cnt_p;
        counts[1] = cnt_q;
    }
}

}  // namespace srhmc

#include "field_rj.cuh"

namespace srhmc {

// ---------------------------------------------------------------------------------------------- kernel
// KMODE: -1 = every mode in one kernel (A.mode decides), otherwise the kernel is compiled for that mode alone; KV3 as in
// eval_pixels.  The specialised <MODE_RUN, 1> build is the hot path of crowded-field chains: a third of the code of the
// generic kernel, no spills.  MODE_RUN_RJ (reversible-jump chains) exists only as its own instantiations.
template <typename T, int MR, int MC, int KMODE = -1, int KV3 = -1>
__global__ void __launch_bounds__(512, 1)
field_kernel(const __grid_constant__ FieldParams P, const __grid_constant__ LaunchArgs A, double* scratch, int d_in_smem) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SmemLayout lay = make_layout<T>(P, d_in_smem != 0);
    const int tid = threadIdx.x, nt = blockDim.x;
    const int S = 3 * P.Nmax;

    for (int field = blockIdx.x; field < A.n_fields; field += gridDim.x) {
        Ctx<T> c;
        c.P = &P;
        c.q = reinterpret_cast<double*>(smem_raw + lay.q);
        c.p = reinterpret_cast<double*>(smem_raw + lay.p);
        c.g = reinterpret_cast<double*>(smem_raw + lay.g);
        c.a1 = reinterpret_cast<double*>(smem_raw + lay.a1);
        c.a2 = reinterpret_cast<double*>(smem_raw + lay.a2);
        c.red = reinterpret_cast<double*>(smem_raw + lay.red);
        c.sD = d_in_smem ? reinterpret_cast<T*>(smem_raw + lay.D) : nullptr;
        c.sL = reinterpret_cast<T*>(smem_raw + lay.L);
        c.tabx = reinterpret_cast<T*>(smem_raw + lay.tabx);
        c.taby = reinterpret_cast<T*>(smem_raw + lay.taby);
        c.span = reinterpret_cast<short*>(smem_raw + lay.span);
        c.gD = reinterpret_cast<const T*>(A.D) + (P.D_shared ? 0 : (size_t)field * P.R * P.C);
        c.sL2 = nullptr;
        c.bg = nullptr;
        c.hess_out = false;
        c.N = A.nstars ? A.nstars[field] : P.Nmax;
        c.g_ff2 = A.g_ff2;
        c.beta = A.beta;
        c.h = A.dt / 2.0;

        __syncthreads();  // previous field done with shared memory
        if (c.sD)
            for (int i = tid; i < P.R * P.C; i += nt) c.sD[i] = c.gD[i];
        const double* q_in = A.q_in + (size_t)field * S;
        for (int i = tid; i < 3 * c.N; i += nt) {
            c.q[i] = q_in[i];
            c.p[i] = (A.p_in != nullptr) ? A.p_in[(size_t)field * S + i] : 0.0;
        }
        if (tid == 0) fp_count_slots(c)[0] = fp_count_slots(c)[1] = 0;
        __syncthreads();

        const int mode = KMODE >= 0 ? KMODE : A.mode;
        if constexpr (KMODE == MODE_RUN_RJ) {
            // compiled into the MODE_RUN_RJ instantiations only (field_rj.cuh)
            run_rj_field<T, MR, MC, KV3>(c, A, scratch, field);
        } else if (mode == MODE_EVAL) {
            const double Vpix = eval_pixels<T, MR, MC, KV3>(c, true);
            const Energies e = energies(c, Vpix, A.f_pos, false);
            for (int k = tid; k < c.N; k += nt) {
                double gf, gx, gy;
                total_grad(c, k, gf, gx, gy);
                const Metric m = metric_of(P, c.q[3 * k], c.g_ff2);
                const size_t o = (size_t)field * S + 3 * k;
                if (A.grad_out) { A.grad_out[o] = gf; A.grad_out[o + 1] = gx; A.grad_out[o + 2] = gy; }
                if (A.H_out) { A.H_out[o] = m.Hff; A.H_out[o + 1] = m.Hxx; A.H_out[o + 2] = m.Hxx; }
                if (A.Hgrad_out) { A.Hgrad_out[o] = m.dHff; A.Hgrad_out[o + 1] = m.dHxx; A.Hgrad_out[o + 2] = m.dHxx; }
            }
            if (tid == 0 && A.V_out) A.V_out[field] = e.V;
        } else if (mode == MODE_STEP) {
            eval_pixels<T, MR, MC, KV3>(c, false);
            double Vpix = 0.0;
            int counts[2] = {0, 0};
            for (int s = 0; s < A.nsteps; ++s) rhmc_step<T, MR, MC, KV3>(c, A.delta, A.counter_max, false, Vpix, counts);
            for (int i = tid; i < 3 * c.N; i += nt) {
                A.q_out[(size_t)field * S + i] = c.q[i];
                A.p_out[(size_t)field * S + i] = c.p[i];
            }
            if (A.fp_counts) {
                // parity mode: every thread already holds the field-wide counts; per-star mode: take the CTA max
                int cp = counts[0], cq = counts[1];
                if (P.fp_mode != 0) {
                    for (int o = 16; o > 0; o >>= 1) {
                        cp = max(cp, __shfl_xor_sync(0xffffffffu, cp, o));
                        cq = max(cq, __shfl_xor_sync(0xffffffffu, cq, o));
                    }
                    __syncthreads();
                    if ((tid & 31) == 0) {
                        c.red[tid >> 5] = (double)cp;
                        c.red[32 + (tid >> 5)] = (double)cq;
                    }
                    __syncthreads();
                    for (int w = 0; w < (nt >> 5); ++w) {
                        cp = max(cp, (int)c.red[w]);
                        cq = max(cq, (int)c.red[32 + w]);
                    }
                }
                if (tid == 0) {
                    A.fp_counts[2 * field] = cp;
                    A.fp_counts[2 * field + 1] = cq;
                }
            }
        } else if (mode == MODE_SINGLE) {
            // single_gym.run_single_RHMC, solver="implicit" (sampler_RHMC.py:649-783)
            const size_t rows = (size_t)A.nsteps + 1;
            double Vpix = eval_pixels<T, MR, MC, KV3>(c, true);
            const Energies e0 = energies(c, Vpix, A.f_pos, true);
            for (int i = tid; i < 3 * c.N; i += nt) {
                A.q_chain[((size_t)field * rows) * S + i] = c.q[i];
                A.p_chain[((size_t)field * rows) * S + i] = c.p[i];
            }
            if (tid == 0) {
                A.E_chain[field * rows] = 0.0;
                A.V_chain[field * rows] = 0.0;
                A.T_chain[field * rows] = 0.0;
            }
            for (int s = 1; s <= A.nsteps; ++s) {
                rhmc_step<T, MR, MC, KV3>(c, A.delta, A.counter_max, true, Vpix, nullptr);
                const Energies e = energies(c, Vpix, A.f_pos, true);
                for (int i = tid; i < 3 * c.N; i += nt) {
                    A.q_chain[((size_t)field * rows + s) * S + i] = c.q[i];
                    A.p_chain[((size_t)field * rows + s) * S + i] = c.p[i];
                }
                if (tid == 0) {
                    const double dV = e.V - e0.V, dT = e.T - e0.T;
                    A.V_chain[field * rows + s] = dV;
                    A.T_chain[field * rows + s] = dT;
                    A.E_chain[field * rows + s] = dV + dT;
                }
            }
        } else {  // MODE_RUN: multi_gym.run_RHMC, move 0 (sampler_RHMC.py:1009-1083)
            double* qs = scratch + (size_t)field * 2 * S;  // q and pixel gradient at the start of the iteration
            double* gs = qs + S;
            const size_t rows = (size_t)A.n_rows;
            const int L = A.niter + 1;
            double Vpix = eval_pixels<T, MR, MC, KV3>(c, true);
            int n_acc = 0;
            for (int l = 0; l < L; ++l) {
                if (A.gff2_sched && l < A.n_gff2) c.g_ff2 = A.gff2_sched[l];
                if (A.beta_sched && l < A.n_beta) c.beta = A.beta_sched[l];
                // momentum refresh p = z sqrt(H)  (sampler_RHMC.py:1021-1022)
                for (int k = tid; k < c.N; k += nt) {
                    const Metric m = metric_of(P, c.q[3 * k], c.g_ff2);
                    double z[3];
                    if (A.normals) {
                        const double* zp = A.normals + ((size_t)field * L + l) * S + 3 * k;
                        z[0] = zp[0]; z[1] = zp[1]; z[2] = zp[2];
                    } else {
                        philox_normals3(A.seed, A.philox_field(field), (uint32_t)l, (uint32_t)k, z);
                    }
                    c.p[3 * k] = z[0] * sqrt(m.Hff);
                    c.p[3 * k + 1] = z[1] * sqrt(m.Hxx);
                    c.p[3 * k + 2] = z[2] * sqrt(m.Hxx);
                    qs[3 * k] = c.q[3 * k]; qs[3 * k + 1] = c.q[3 * k + 1]; qs[3 * k + 2] = c.q[3 * k + 2];
                    gs[3 * k] = c.g[3 * k]; gs[3 * k + 1] = c.g[3 * k + 1]; gs[3 * k + 2] = c.g[3 * k + 2];
                }
                __syncthreads();
                const Energies e0 = energies(c, Vpix, A.f_pos, true);
                const double E0 = e0.V + e0.T;
                const double Vpix0 = Vpix;
                const bool keep = (l % A.chain_stride) == 0;
                const size_t row = (size_t)field * rows + (size_t)(l / A.chain_stride);
                if (keep) {
                    if (A.q_chain)
                        for (int i = tid; i < 3 * c.N; i += nt) A.q_chain[row * S + i] = c.q[i];
                    if (A.p_chain)
                        for (int i = tid; i < 3 * c.N; i += nt) A.p_chain[row * S + i] = c.p[i];
                    if (tid == 0) {
                        if (A.E_chain) A.E_chain[row] = E0;
                        if (A.V_chain) A.V_chain[row] = e0.V;
                        if (A.T_chain) A.T_chain[row] = e0.T;
                    }
                }
                for (int s = 0; s < A.nsteps; ++s)
                    rhmc_step<T, MR, MC, KV3>(c, A.delta, A.counter_max, s == A.nsteps - 1, Vpix, nullptr);
                const Energies e1 = energies(c, Vpix, A.f_pos, true);
                const double dE = (e1.V + e1.T) - E0;
                const double lnu = A.lnu ? A.lnu[(size_t)field * L + l] : philox_lnu(A.seed, A.philox_field(field), (uint32_t)l);
                const bool accept = (dE < 0.0) || (lnu < -dE);
                if (keep && tid == 0 && A.A_chain) A.A_chain[row] = accept ? 1 : 0;
                if (accept) {
                    ++n_acc;
                } else {
                    __syncthreads();
                    for (int i = tid; i < 3 * c.N; i += nt) {
                        c.q[i] = qs[i];
                        c.g[i] = gs[i];
                    }
                    Vpix = Vpix0;
                }
                __syncthreads();
            }
            if (A.q_out)
                for (int i = tid; i < 3 * c.N; i += nt) A.q_out[(size_t)field * S + i] = c.q[i];
            if (tid == 0 && A.accept_rate) A.accept_rate[field] = (double)n_acc / (double)L;
        }
    }
}

}  // namespace srhmc
