// Small utility kernels: Philox dump, image conversion, FMA-chain peak microbenchmark, and the precision
// dispatch of the CTA-per-field launchers.
#include "kernels_api.h"
#include "rj_draws.cuh"

namespace srhmc {

// Device normals / log-uniforms exactly as MODE_RUN consumes them (for replay through another implementation).
__global__ void philox_dump_kernel(unsigned long long seed, int n_fields, int L, int Nmax, int fid_base, int fid_stride,
                                   double* normals, double* lnu) {
    const size_t total = (size_t)n_fields * L * Nmax;
    for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(t % Nmax);
        const int l = (int)((t / Nmax) % L);
        const int f = (int)(t / ((size_t)Nmax * L));
        double z[3];
        const uint32_t fid = (uint32_t)(fid_base + f * fid_stride);
        philox_normals3(seed, fid, (uint32_t)l, (uint32_t)k, z);
        double* o = normals + (((size_t)f * L + l) * Nmax + k) * 3;
        o[0] = z[0]; o[1] = z[1]; o[2] = z[2];
        if (k == 0) lnu[(size_t)f * L + l] = philox_lnu(seed, fid, (uint32_t)l);
    }
}

// Reversible-jump draw records exactly as MODE_RUN_RJ consumes them: one thread per (field, iteration).
__global__ void rj_dump_kernel(unsigned long long seed, int n_fields, int L, int fid_base, int fid_stride, double beta_a,
                               double beta_b, double* draws) {
    const size_t total = (size_t)n_fields * L;
    for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int l = (int)(t % L), f = (int)(t / L);
        rj_record(seed, (uint32_t)(fid_base + f * fid_stride), (uint32_t)l, beta_a, beta_b, draws + t * kRjDraws);
    }
}

int rj_dump_launch(cudaStream_t stream, unsigned long long seed, int n_fields, int L, int fid_base, int fid_stride, double beta_a,
                   double beta_b, double* draws) {
    const size_t total = (size_t)n_fields * L;
    const int blocks = (int)((total + 127) / 128 < 4096 ? (total + 127) / 128 : 4096);
    rj_dump_kernel<<<blocks > 0 ? blocks : 1, 128, 0, stream>>>(seed, n_fields, L, fid_base, fid_stride, beta_a, beta_b, draws);
    return (int)cudaGetLastError();
}

// Kinetic energy and the tau-part derivatives of one field per block (sampler_RHMC.py:353-363, 467-492):
//   T = (sum p^2/H + sum ln|H|)/2,  dtau/dq_f = -p_f^2 H_ff'/H_ff^2 / 2 (flux slots only),  dtau/dp = p/H.
__global__ void kinetic_kernel(const FieldParams P, int n_fields, const double* q, const double* p, const int* nstars,
                               double g_ff2, double* T, double* dtaudq, double* dtaudp) {
    __shared__ double red[2 * 32];
    const int field = blockIdx.x;
    if (field >= n_fields) return;
    const int N = nstars ? nstars[field] : P.Nmax;
    const size_t S = 3 * (size_t)P.Nmax;
    double v[2] = {0.0, 0.0};
    for (int k = threadIdx.x; k < N; k += blockDim.x) {
        const size_t o = (size_t)field * S + 3 * k;
        const Metric m = metric_of(P, q[o], g_ff2);
        const double pf = p[o], px = p[o + 1], py = p[o + 2];
        v[0] += pf * pf / m.Hff + px * px / m.Hxx + py * py / m.Hxx;
        v[1] += log(fabs(m.Hff)) + 2.0 * log(fabs(m.Hxx));
        if (dtaudq) {
            dtaudq[o] = -((pf * pf) * m.dHff / (m.Hff * m.Hff)) / 2.0;
            dtaudq[o + 1] = 0.0;
            dtaudq[o + 2] = 0.0;
        }
        if (dtaudp) {
            dtaudp[o] = pf / m.Hff;
            dtaudp[o + 1] = px / m.Hxx;
            dtaudp[o + 2] = py / m.Hxx;
        }
    }
    block_sum<2>(v, red);
    if (threadIdx.x == 0 && T) T[field] = (v[0] + v[1]) / 2.0;
}

// Diagonal metric and its flux derivative for n flat [f, x, y] triples (sampler_RHMC.py:229-292).
__global__ void metric_kernel(const FieldParams P, size_t n_stars, const double* q, double g_ff2, double* H, double* Hgrad) {
    for (size_t k = blockIdx.x * (size_t)blockDim.x + threadIdx.x; k < n_stars; k += (size_t)gridDim.x * blockDim.x) {
        const Metric m = metric_of(P, q[3 * k], g_ff2);
        if (H) { H[3 * k] = m.Hff; H[3 * k + 1] = m.Hxx; H[3 * k + 2] = m.Hxx; }
        if (Hgrad) { Hgrad[3 * k] = m.dHff; Hgrad[3 * k + 1] = m.dHxx; Hgrad[3 * k + 2] = m.dHxx; }
    }
}

int metric_launch(cudaStream_t stream, const FieldParams& P, size_t n_stars, const double* q, double g_ff2, double* H,
                  double* Hgrad) {
    const int blocks = (int)((n_stars + 127) / 128 < 4096 ? (n_stars + 127) / 128 : 4096);
    metric_kernel<<<blocks > 0 ? blocks : 1, 128, 0, stream>>>(P, n_stars, q, g_ff2, H, Hgrad);
    return (int)cudaGetLastError();
}

// T(p, H_diag) = (sum p^2/H + sum ln|H|)/2 for an explicit diagonal (sampler_RHMC.py:353-363); one block.
__global__ void kinetic_diag_kernel(size_t n, const double* p, const double* H, double* T) {
    __shared__ double red[2 * 32];
    double v[2] = {0.0, 0.0};
    for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
        v[0] += p[i] * p[i] / H[i];
        v[1] += log(fabs(H[i]));
    }
    block_sum<2>(v, red);
    if (threadIdx.x == 0) T[0] = (v[0] + v[1]) / 2.0;
}

int kinetic_diag_launch(cudaStream_t stream, size_t n, const double* p, const double* H, double* T) {
    kinetic_diag_kernel<<<1, 256, 0, stream>>>(n, p, H, T);
    return (int)cudaGetLastError();
}

int kinetic_launch(cudaStream_t stream, const FieldParams& P, int n_fields, const double* q, const double* p,
                   const int* nstars, double g_ff2, double* T, double* dtaudq, double* dtaudp) {
    kinetic_kernel<<<n_fields > 0 ? n_fields : 1, 128, 0, stream>>>(P, n_fields, q, p, nstars, g_ff2, T, dtaudq, dtaudp);
    return (int)cudaGetLastError();
}

template <typename T>
__global__ void convert_image_kernel(const double* src, T* dst, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = (T)src[i];
}


size_t field_layout_total_f64(const FieldParams& P, bool dsm);
size_t field_layout_total_f32(const FieldParams& P, bool dsm);
int field_kernel_configure_f64(int mr, int mc, size_t smem);
int field_kernel_configure_f32(int mr, int mc, size_t smem);
int field_kernel_launch_f64(int, int, int, int, size_t, cudaStream_t, const FieldParams&, const LaunchArgs&, double*, int);
int field_kernel_launch_f32(int, int, int, int, size_t, cudaStream_t, const FieldParams&, const LaunchArgs&, double*, int);

size_t field_layout_total(int precision, const FieldParams& P, bool dsm) {
    return precision == 64 ? field_layout_total_f64(P, dsm) : field_layout_total_f32(P, dsm);
}
int field_kernel_configure(int precision, int mr, int mc, size_t smem) {
    return precision == 64 ? field_kernel_configure_f64(mr, mc, smem) : field_kernel_configure_f32(mr, mc, smem);
}
int field_kernel_launch(int precision, int mr, int mc, int grid, int threads, size_t smem, cudaStream_t stream,
                        const FieldParams& P, const LaunchArgs& A, double* scratch, int dsm) {
    return precision == 64 ? field_kernel_launch_f64(mr, mc, grid, threads, smem, stream, P, A, scratch, dsm)
                           : field_kernel_launch_f32(mr, mc, grid, threads, smem, stream, P, A, scratch, dsm);
}

int philox_dump_launch(cudaStream_t stream, unsigned long long seed, int n_fields, int L, int Nmax, int fid_base,
                       int fid_stride, double* normals, double* lnu) {
    const size_t total = (size_t)n_fields * L * Nmax;
    const int blocks = (int)((total + 255) / 256 < 8192 ? (total + 255) / 256 : 8192);
    philox_dump_kernel<<<blocks > 0 ? blocks : 1, 256, 0, stream>>>(seed, n_fields, L, Nmax, fid_base, fid_stride, normals, lnu);
    return (int)cudaGetLastError();
}

int convert_image_launch(cudaStream_t stream, const double* src, float* dst, size_t n) {
    const int blocks = (int)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
    convert_image_kernel<float><<<blocks > 0 ? blocks : 1, 256, 0, stream>>>(src, dst, n);
    return (int)cudaGetLastError();
}

// FMA-chain microbenchmark: 8 independent dependent chains per thread.
template <typename T>
__global__ void __launch_bounds__(256) fma_peak_kernel(T* out, int iters, T a, T b) {
    T x0 = (T)threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

template <typename T>
static int run_fma_peak(int sms, double* tflops, float* ms) {
    const int blocks = sms * 8, threads = 256, iters = 4096;
    T* out = nullptr;
    cudaError_t e = cudaMalloc(&out, (size_t)blocks * threads * sizeof(T));
    if (e != cudaSuccess) return (int)e;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0, 0);
        fma_peak_kernel<T><<<blocks, threads>>>(out, iters, (T)0.999, (T)0.001);
        cudaEventRecord(e1, 0);
        cudaEventSynchronize(e1);
        float t = 0.f;
        cudaEventElapsedTime(&t, e0, e1);
        if (rep > 0 && t < best) best = t;
    }
    e = cudaGetLastError();
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    if (e != cudaSuccess) return (int)e;
    const double flops = 2.0 * 64.0 * (double)iters * (double)blocks * threads;
    *tflops = flops / (best * 1e-3) / 1e12;
    if (ms) *ms = best;
    return 0;
}

int fma_peak_run(int precision, int sms, double* tflops, float* ms) {
    return precision == 64 ? run_fma_peak<double>(sms, tflops, ms) : run_fma_peak<float>(sms, tflops, ms);
}

}  // namespace srhmc
