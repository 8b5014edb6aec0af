// libstellar_rhmc.so -- C ABI (include/stellar_rhmc.h) over the sm_100a RHMC kernels.
// Host logic only: context / buffer ownership, launch configuration, copies.  No CPU compute path exists.
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
#include "kernels_api.h"

using namespace srhmc;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU_TRY(expr)                                                                                        \
    do {                                                                                                    \
        cudaError_t e__ = (expr);                                                                           \
        if (e__ != cudaSuccess)                                                                             \
            return fail(SRHMC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

struct DevBuf {
    void* ptr = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&ptr, want);
        if (e != cudaSuccess) return fail(SRHMC_ERR_CUDA, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        cap = want;
        return 0;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
    }
    template <typename U> U* as() const { return reinterpret_cast<U*>(ptr); }
};

struct KernelChoice {
    int mr, mc;
};

constexpr int kMaxParts = 8;  // launches a pipelined run is cut into at most

}  // namespace

struct srhmc_ctx {
    srhmc_config cfg;
    FieldParams P;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // pipelined run (run_pipelined): copy stream, per-part completion events
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t part_done[kMaxParts] = {}, copies_done = nullptr;
    bool have_data = false, timed = false;
    int64_t launches = 0;
    int sm_count = 0;
    // launch configuration of the CTA-per-field kernel
    KernelChoice kc{};
    int threads = 256;
    size_t smem = 0;
    int d_in_smem = 1;
    FieldParams P_ls;   // parameters of the lightsource-family kernels (chunked tables, never the compact-table path)
    size_t smem_ls = 0;
    int dsm_ls = 1;
    bool chain_ok = false;          // warp-resident one-star kernel configured for this context
    ChainLaunchPlan chain_plan;
    size_t pix_bytes = 8;
    // device buffers
    DevBuf ls_dt, ls_steps, ls_bg, ls_scratch, ls_d1, ls_d2, ls_d3;
    DevBuf field_ids;
    bool run_has_field_ids = false;
    DevBuf sched_done, sched_state, sched_err;  // chain-kernel work scheduler (see chain_kernel.cuh)
    bool sched_used = false;
    DevBuf D32, D16, logtab, flag;  // exact uint32 / uint16 copies of the images, fastmath log table, scratch flag
    int d_int_bytes = 0;            // 0: float64 images only; 4 / 2: the integer copy the chain kernel should read
    DevBuf D, Dstage, q, p, nstars, normals, lnu, sg, sb, qchain, pchain, E, V, T, A, acc, scratch, qout, pout, Vout,
        grad, H, Hg, counts;
    // sizes of the last uploaded run
    int run_L = 0, run_rows = 0;
    bool run_has_nstars = false, run_has_normals = false, run_has_lnu = false, run_one_star = false;
    bool run_has_qchain = false;  // the last launched run recorded q_chain on the device
    DevBuf st_means, st_R, st_neff;  // chain statistics
};

namespace {

KernelChoice pick_kernel(int R, int C, int nwarps) {
    auto tiles = [&](int mr, int mc) { return ((R + 8 * mr - 1) / (8 * mr)) * ((C + 4 * mc - 1) / (4 * mc)); };
    if (tiles(2, 4) >= nwarps) return {2, 4};
    if (tiles(2, 2) >= nwarps) return {2, 2};
    return {1, 2};
}

constexpr size_t kSmemMax = 232448;  // 227 KB opt-in limit per CTA on sm_100

int configure(srhmc_ctx* c) {
    const int prec = c->cfg.precision;
    const size_t elem = prec == 64 ? 8 : 4;
    const srhmc_config& g = c->cfg;
    FieldParams& P = c->P;
    const int R = g.num_rows, C = g.num_cols, N = g.max_stars;
    int threads = 256;
    if ((size_t)R * C >= 4096 || N > 256) threads = 512;
    if ((size_t)R * C <= 256 && N <= 64) threads = 128;
    if (const char* env = std::getenv("SRHMC_FIELD_THREADS")) {  // tuning / experiments
        const int t = std::atoi(env);
        if (t == 128 || t == 256 || t == 512) threads = t;
    }
    c->threads = threads;
    c->kc = pick_kernel(R, C, threads / 32);
    // table strides: rows / columns rounded up to the warp tile, plus 16 bytes so that the tables of consecutive stars
    // start on different shared-memory banks (one thread builds one table: 64-double strides put 16 stars on one bank)
    const int tab_pad = prec == 64 ? 2 : 4;
    P.sx = ((R + 8 * c->kc.mr - 1) / (8 * c->kc.mr)) * 8 * c->kc.mr + tab_pad;
    P.sy = ((C + 4 * c->kc.mc - 1) / (4 * c->kc.mc)) * 4 * c->kc.mc + tab_pad;
    const int nwant = std::max(1, N);
    auto fit = [&](size_t budget, bool dsm) -> int {
        FieldParams Q = P;
        Q.Kc = 0;
        const size_t base = field_layout_total(prec, Q, dsm);
        const size_t per = (size_t)(P.sx + P.sy) * elem + 4 * sizeof(short);
        if (base + per + 64 > budget) return 0;
        return (int)std::min<size_t>((size_t)nwant, (budget - base - 64) / per);
    };
    size_t budget = 112 * 1024;
    if (const char* env = std::getenv("SRHMC_FIELD_SMEM_KB")) budget = (size_t)std::max(16, std::atoi(env)) * 1024;
    int kc = fit(budget, true);
    bool dsm = true;
    if (const char* env = std::getenv("SRHMC_FIELD_D_GLOBAL")) {
        if (env[0] == '1') { dsm = false; kc = fit(budget, false); }
    }
    if (kc < std::min(nwant, 24)) kc = fit(kSmemMax, true);
    if (kc < std::min(nwant, 8)) {
        const int kg = fit(kSmemMax, false);
        if (kg > kc) {
            kc = kg;
            dsm = false;
        }
    }
    if (kc < 1)
        return fail(SRHMC_ERR_TOO_LARGE, "a %dx%d field with %d stars does not fit the CTA-resident kernel (%zu B shared memory)",
                    R, C, N, kSmemMax);
    P.Kc = kc;
    c->d_in_smem = dsm ? 1 : 0;
    c->smem = field_layout_total(prec, P, dsm);
    // the lightsource family (ls_kernel.cuh) always runs with the chunked tables configured above
    c->P_ls = P;
    c->smem_ls = c->smem;
    c->dsm_ls = c->d_in_smem;
    // compact-table evaluation (field_kernel.cuh "v3") when the PSF is patch-limited and every star's tables fit at once
    {
        const int TL = 2 * g.patch_radius + 1;
        bool want = g.patch_radius > 0 && g.patch_radius <= 12 && (C % 2 == 0) && R >= TL && C >= TL + 1 && !P.hess && N >= 1;
        if (const char* env = std::getenv("SRHMC_FIELD_V3"))
            if (env[0] == '0') want = false;
        if (want) {
            FieldParams Q = P;
            Q.v3 = 1;
            Q.tl = TL;
            Q.rs = (TL + 2) | 1;
            Q.cs = (TL + 7) | 1;
            bool dsm3 = true;
            size_t tot = field_layout_total(prec, Q, true);
            if (tot > kSmemMax) {
                dsm3 = false;
                tot = field_layout_total(prec, Q, false);
            }
            if (tot <= kSmemMax) {
                P = Q;
                c->d_in_smem = dsm3 ? 1 : 0;
                c->smem = std::max(tot, c->smem_ls);
            }
        }
    }
    const int e = field_kernel_configure(prec, c->kc.mr, c->kc.mc, c->smem);
    if (e != 0) return fail(SRHMC_ERR_CUDA, "cudaFuncSetAttribute(%zu B shared) failed: %s", c->smem, cudaGetErrorString((cudaError_t)e));
    if (prec == 64) {
        const int e2 = ls_kernel_configure(c->kc.mr, c->kc.mc, c->smem);
        if (e2 != 0) return fail(SRHMC_ERR_CUDA, "cudaFuncSetAttribute(%zu B shared) failed: %s", c->smem, cudaGetErrorString((cudaError_t)e2));
    }
    return 0;
}

int launch_field(srhmc_ctx* c, const LaunchArgs& A_in, bool one_star_everywhere) {
    LaunchArgs A = A_in;
    // the FP32 build of the one-star kernel reads the uint16 count images only
    const bool chain = c->chain_ok && one_star_everywhere && (c->cfg.precision == 64 || c->d_int_bytes == 2);
    A.pix_f32 = (chain && c->cfg.precision == 32) ? 1 : 0;
    if (chain && A.mode == MODE_RUN) {
        // scheduler state of the chunked chain kernel: completion counters start at 0 for every launch
        const size_t groups = ((size_t)A.n_fields + kChainGroup - 1) / kChainGroup;
        if (int rc = c->sched_done.ensure(groups * sizeof(int))) return rc;
        if (int rc = c->sched_state.ensure((size_t)A.n_fields * 8 * sizeof(double))) return rc;
        if (int rc = c->sched_err.ensure(sizeof(int))) return rc;
        CU_TRY(cudaMemsetAsync(c->sched_done.ptr, 0, groups * sizeof(int), c->stream));
        CU_TRY(cudaMemsetAsync(c->sched_err.ptr, 0, sizeof(int), c->stream));
        A.sched_done = c->sched_done.as<int>();
        A.sched_state = c->sched_state.as<double>();
        A.sched_err = c->sched_err.as<int>();
        c->sched_used = true;
    }
    if (c->timed) CU_TRY(cudaEventRecord(c->ev0, c->stream));
    if (chain) {
        int rc = chain_kernel_launch(c->P, A, c->chain_plan, c->sm_count, c->stream);
        if (rc != 0) return fail(SRHMC_ERR_CUDA, "chain kernel launch failed: %s", cudaGetErrorString((cudaError_t)rc));
    } else {
        const int grid = std::max(1, A.n_fields);
        int rc = field_kernel_launch(c->cfg.precision, c->kc.mr, c->kc.mc, grid, c->threads, c->smem, c->stream, c->P, A,
                                     c->scratch.as<double>(), c->d_in_smem);
        if (rc != 0) return fail(SRHMC_ERR_CUDA, "field kernel launch failed: %s", cudaGetErrorString((cudaError_t)rc));
    }
    if (c->timed) CU_TRY(cudaEventRecord(c->ev1, c->stream));
    c->launches += 1;
    return 0;
}

int upload(srhmc_ctx* c, DevBuf& b, const void* src, size_t bytes) {
    if (int rc = b.ensure(bytes)) return rc;
    CU_TRY(cudaMemcpyAsync(b.ptr, src, bytes, cudaMemcpyHostToDevice, c->stream));
    return 0;
}

int download(srhmc_ctx* c, void* dst, const DevBuf& b, size_t bytes) {
    CU_TRY(cudaMemcpyAsync(dst, b.ptr, bytes, cudaMemcpyDeviceToHost, c->stream));
    return 0;
}

bool chain_kernel_eligible(const srhmc_config& g) {
    const char* off = std::getenv("SRHMC_DISABLE_CHAIN_KERNEL");
    if (off && off[0] == '1') return false;
    // precision 32: FP32 pixel arithmetic on the uint16 count images (data that are not counts < 65536 take the CTA kernel)
    return g.max_stars == 1 && g.num_cols <= 32 && g.num_rows <= 64 && !g.use_Vc && !g.shared_data && g.patch_radius == 0;
}

bool all_one_star(const srhmc_ctx* c, const int32_t* nstars) {
    if (!nstars) return c->cfg.max_stars == 1;
    for (int f = 0; f < c->cfg.n_fields; ++f)
        if (nstars[f] != 1) return false;
    return true;
}

}  // namespace

int srhmc::check_stats_args(int64_t n_chains, int64_t rows, int32_t d, int32_t n_groups, int32_t thin, int32_t warm) {
    if (n_chains < 1 || rows < 1 || d < 1 || n_groups < 1 || thin < 1 || warm < 0) return fail(SRHMC_ERR_INVALID, "bad chain statistics argument");
    if (n_chains % n_groups) return fail(SRHMC_ERR_INVALID, "%lld chains do not split into %d equal groups", (long long)n_chains, n_groups);
    if (n_chains / n_groups < 2) return fail(SRHMC_ERR_INVALID, "convergence statistics need at least two chains per group (utils.py:94)");
    const int64_t Lw = rows - warm, Lc = Lw > 0 ? (Lw + thin - 1) / thin : 0;
    if (Lc / 2 < 2) return fail(SRHMC_ERR_INVALID, "fewer than two samples per split chain after warm-up and thinning");
    if (n_chains / n_groups > (1 << 24)) return fail(SRHMC_ERR_INVALID, "too many chains per group");
    return 0;
}

extern "C" {

int srhmc_abi_version(void) { return SRHMC_ABI_VERSION; }
const char* srhmc_last_error(void) { return g_err; }

int srhmc_chain_group_size(void) { return kChainGroup; }

int srhmc_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

void* srhmc_host_alloc(uint64_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) {
        fail(SRHMC_ERR_CUDA, "cudaMallocHost(%llu) failed", (unsigned long long)bytes);
        return nullptr;
    }
    return p;
}
int srhmc_host_free(void* p) {
    if (p) CU_TRY(cudaFreeHost(p));
    return 0;
}

int srhmc_create(const srhmc_config* cfg, srhmc_ctx** out) {
    if (!cfg || !out) return fail(SRHMC_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->abi_version != SRHMC_ABI_VERSION)
        return fail(SRHMC_ERR_INVALID, "ABI version mismatch: caller %d, library %d", cfg->abi_version, SRHMC_ABI_VERSION);
    if (cfg->precision != 64 && cfg->precision != 32) return fail(SRHMC_ERR_INVALID, "precision must be 64 or 32");
    if (cfg->n_fields < 1 || cfg->num_rows < 1 || cfg->num_cols < 1 || cfg->max_stars < 0)
        return fail(SRHMC_ERR_INVALID, "n_fields, num_rows, num_cols must be >= 1 and max_stars >= 0");
    if (cfg->num_rows > 16384 || cfg->num_cols > 16384) return fail(SRHMC_ERR_INVALID, "image dimension too large");
    if (!(cfg->psf_fwhm_pix > 0.0)) return fail(SRHMC_ERR_INVALID, "psf_fwhm_pix must be positive");
    if (cfg->patch_radius < 0 || cfg->patch_radius > 15)
        return fail(SRHMC_ERR_INVALID, "patch_radius must be 0 (full image) or 1..15");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(SRHMC_ERR_NO_DEVICE, "no CUDA device visible: this library has no CPU path");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(SRHMC_ERR_INVALID, "device %d out of range (%d visible)", cfg->device, ndev);
    CU_TRY(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10)
        return fail(SRHMC_ERR_NO_DEVICE, "device %d is sm_%d%d; the kernels are built for sm_100a only", cfg->device, prop.major, prop.minor);

    srhmc_ctx* c = new (std::nothrow) srhmc_ctx();
    if (!c) return fail(SRHMC_ERR_INVALID, "out of host memory");
    c->cfg = *cfg;
    c->sm_count = prop.multiProcessorCount;
    FieldParams& P = c->P;
    std::memset(&P, 0, sizeof(P));
    P.R = cfg->num_rows;
    P.C = cfg->num_cols;
    P.Nmax = cfg->max_stars;
    P.rad = cfg->patch_radius;
    P.fp_mode = cfg->fixed_point_mode;
    P.D_shared = cfg->shared_data ? 1 : 0;
    P.use_prior = cfg->use_prior ? 1 : 0;
    P.use_Vc = cfg->use_Vc ? 1 : 0;
    P.hess = (cfg->enable_hessian && cfg->precision == 64) ? 1 : 0;
    const double sigma = cfg->psf_fwhm_pix / 2.354;  // utils.py:480
    P.inv2s2 = 1.0 / (2.0 * sigma * sigma);
    P.inv_s2 = 1.0 / (sigma * sigma);
    P.norm = 1.0 / (M_PI * 2.0 * sigma * sigma);
    P.c2 = std::exp(-1.0 / (sigma * sigma));
    P.B = cfg->B_count;
    P.lnB = std::log(cfg->B_count);
    P.invB = 1.0 / cfg->B_count;
    P.cL = std::exp(-(double)(kChainLPC * kChainLPC) / (sigma * sigma));
    P.cLh = std::exp(-(double)(kChainLPC * kChainLPC) / (2.0 * sigma * sigma));
    {
        // rows whose Gaussian weight is below 2^-bits of the peak are skipped by the one-star kernel (its 24-column window
        // cuts at 2^-47 for the default PSF); SRHMC_CHAIN_WCUT_BITS overrides for A/B measurements
        double bits = 46.0;
        if (const char* env = std::getenv("SRHMC_CHAIN_WCUT_BITS")) bits = std::max(20.0, std::min(1000.0, std::atof(env)));
        P.wcut = std::sqrt(bits * M_LN2 * 2.0 * sigma * sigma);
    }
    P.f_lim = cfg->f_lim;
    P.f_low = cfg->f_low;
    P.g0 = cfg->g0; P.g1 = cfg->g1; P.g2 = cfg->g2;
    P.g_xx = cfg->g_xx; P.g_ff = cfg->g_ff;
    P.alpha = cfg->alpha;
    P.Vpc = cfg->V_prior_const;
    P.vc_pow = cfg->Vc_r_pow;
    const double rp = std::floor(cfg->Vc_r_pow);
    P.vc_int = (rp == cfg->Vc_r_pow && rp >= 0.0 && rp <= 32.0) ? (int)rp : -1;
    c->pix_bytes = cfg->precision == 64 ? 8 : 4;

    int rc = configure(c);
    if (rc == 0 && chain_kernel_eligible(*cfg)) {
        const int e = chain_kernel_configure(P, c->chain_plan);
        if (e != 0) rc = fail(SRHMC_ERR_CUDA, "chain kernel configuration failed: %s", cudaGetErrorString((cudaError_t)e));
        c->chain_ok = (e == 0);
    }
    if (rc != 0) {
        delete c;
        return rc;
    }
    cudaError_t e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
    if (e != cudaSuccess) {
        delete c;
        return fail(SRHMC_ERR_CUDA, "stream/event creation failed: %s", cudaGetErrorString(e));
    }
    c->stream = c->own_stream;
    c->timed = true;
    {
        double tab[256] = {0};
        fill_log_table(tab);
        int rc2 = c->logtab.ensure(sizeof(tab));
        if (rc2 == 0 && cudaMemcpy(c->logtab.ptr, tab, sizeof(tab), cudaMemcpyHostToDevice) != cudaSuccess)
            rc2 = fail(SRHMC_ERR_CUDA, "log table upload failed");
        if (rc2 == 0) rc2 = c->flag.ensure(16);
        if (rc2 != 0) {
            srhmc_destroy(c);
            return rc2;
        }
    }
    *out = c;
    return 0;
}

int srhmc_destroy(srhmc_ctx* c) {
    if (!c) return 0;
    cudaSetDevice(c->cfg.device);
    cudaStreamSynchronize(c->stream);
    DevBuf* all[] = {&c->ls_dt, &c->ls_steps, &c->ls_bg, &c->ls_scratch, &c->ls_d1, &c->ls_d2, &c->ls_d3, &c->field_ids, &c->sched_done, &c->sched_state, &c->sched_err, &c->D32, &c->D16, &c->logtab, &c->flag, &c->D, &c->Dstage, &c->q, &c->p, &c->nstars, &c->normals, &c->lnu, &c->sg, &c->sb, &c->qchain,
                     &c->pchain, &c->E, &c->V, &c->T, &c->A, &c->acc, &c->scratch, &c->qout, &c->pout, &c->Vout, &c->st_means, &c->st_R, &c->st_neff,
                     &c->grad, &c->H, &c->Hg, &c->counts};
    for (DevBuf* b : all) b->release();
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    for (int s = 0; s < kMaxParts; ++s)
        if (c->part_done[s]) cudaEventDestroy(c->part_done[s]);
    if (c->copies_done) cudaEventDestroy(c->copies_done);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
    return 0;
}

int srhmc_set_stream(srhmc_ctx* c, void* s) {
    if (!c) return fail(SRHMC_ERR_INVALID, "null context");
    CU_TRY(cudaSetDevice(c->cfg.device));
    CU_TRY(cudaStreamSynchronize(c->stream));
    c->stream = s ? reinterpret_cast<cudaStream_t>(s) : c->own_stream;
    return 0;
}

int srhmc_synchronize(srhmc_ctx* c) {
    if (!c) return fail(SRHMC_ERR_INVALID, "null context");
    CU_TRY(cudaSetDevice(c->cfg.device));
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int srhmc_last_kernel_ms(srhmc_ctx* c, float* ms) {
    if (!c || !ms) return fail(SRHMC_ERR_INVALID, "null argument");
    if (c->launches == 0) return fail(SRHMC_ERR_STATE, "no kernel launched yet");
    CU_TRY(cudaSetDevice(c->cfg.device));
    CU_TRY(cudaEventSynchronize(c->ev1));
    CU_TRY(cudaEventElapsedTime(ms, c->ev0, c->ev1));
    return 0;
}

int64_t srhmc_launch_count(srhmc_ctx* c) { return c ? c->launches : 0; }

// after the float64 images are in place on the device (c->D for the FP64 build, c->Dstage for the FP32 build): the
// reduced-precision / exact-integer copies the kernels read
static int finish_data(srhmc_ctx* c, size_t n) {
    if (c->cfg.precision != 64) {
        if (int rc = c->D.ensure(n * 4)) return rc;
        const int e = convert_image_launch(c->stream, c->Dstage.as<double>(), c->D.as<float>(), n);
        if (e != 0) return fail(SRHMC_ERR_CUDA, "image conversion failed: %s", cudaGetErrorString((cudaError_t)e));
        c->launches += 1;
    }
    c->d_int_bytes = 0;
    if (c->chain_ok) {
        // lossless compact copies for the warp-resident kernel when every pixel is an integer count (Poisson data)
        if (int rc = c->D32.ensure(n * 4)) return rc;
        if (int rc = c->D16.ensure(n * 2)) return rc;
        CU_TRY(cudaMemsetAsync(c->flag.ptr, 0, 4, c->stream));
        const double* d64 = c->cfg.precision == 64 ? c->D.as<double>() : c->Dstage.as<double>();
        const int e = to_counts_launch(c->stream, d64, c->D32.as<unsigned int>(), c->D16.as<unsigned short>(), n, c->flag.as<int>());
        if (e != 0) return fail(SRHMC_ERR_CUDA, "count conversion failed: %s", cudaGetErrorString((cudaError_t)e));
        c->launches += 1;
        int flags = 3;
        CU_TRY(cudaMemcpyAsync(&flags, c->flag.ptr, 4, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaStreamSynchronize(c->stream));
        const char* off = std::getenv("SRHMC_DISABLE_U32_IMAGES");   // both integer layouts off
        const char* off16 = std::getenv("SRHMC_DISABLE_U16_IMAGES");
        if (!(off && off[0] == '1') && (flags & 1) == 0)
            c->d_int_bytes = ((flags & 2) == 0 && !(off16 && off16[0] == '1')) ? 2 : 4;
    }
    CU_TRY(cudaStreamSynchronize(c->stream));
    c->have_data = true;
    return 0;
}

int srhmc_set_data(srhmc_ctx* c, const double* D, int64_t n_images) {
    if (!c || !D) return fail(SRHMC_ERR_INVALID, "null argument");
    const int64_t want = c->cfg.shared_data ? 1 : c->cfg.n_fields;
    if (n_images != want) return fail(SRHMC_ERR_INVALID, "expected %lld image(s), got %lld", (long long)want, (long long)n_images);
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t n = (size_t)n_images * c->P.R * c->P.C;
    if (int rc = upload(c, c->cfg.precision == 64 ? c->D : c->Dstage, D, n * 8)) return rc;
    return finish_data(c, n);
}

static int upload_nstars(srhmc_ctx* c, const int32_t* nstars);

// model images of all fields into `dst` (device, float64 [F,R,C])
static int render_models(srhmc_ctx* c, const double* q, const int32_t* nstars, double* dst) {
    const size_t S = 3 * (size_t)c->cfg.max_stars;
    if (S) {
        if (int rc = upload(c, c->q, q, (size_t)c->cfg.n_fields * S * 8)) return rc;
    } else if (int rc = c->q.ensure(8)) {
        return rc;
    }
    if (int rc = upload_nstars(c, nstars)) return rc;
    const int e = model_launch(c->stream, c->P, c->cfg.n_fields, c->q.as<double>(), nstars ? c->nstars.as<int>() : nullptr, nullptr, dst);
    if (e != 0) return fail(SRHMC_ERR_CUDA, "model kernel failed: %s", cudaGetErrorString((cudaError_t)e));
    c->launches += 1;
    return 0;
}

int srhmc_gen_model(srhmc_ctx* c, const double* q, const int32_t* nstars, double* model) {
    if (!c || !model || (c->cfg.max_stars > 0 && !q)) return fail(SRHMC_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t n = (size_t)c->cfg.n_fields * c->P.R * c->P.C;
    if (int rc = c->scratch.ensure(n * 8)) return rc;
    if (int rc = render_models(c, q, nstars, c->scratch.as<double>())) return rc;
    if (int rc = download(c, model, c->scratch, n * 8)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int srhmc_gen_mock_data(srhmc_ctx* c, const double* q_true, const int32_t* nstars, uint64_t seed, int64_t field_id_base,
                        double* D_out) {
    if (!c || (c->cfg.max_stars > 0 && !q_true)) return fail(SRHMC_ERR_INVALID, "null argument");
    if (c->cfg.shared_data) return fail(SRHMC_ERR_INVALID, "mock data are generated per field: not available with shared_data");
    if (field_id_base < 0) return fail(SRHMC_ERR_INVALID, "field_id_base must be >= 0");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t npx = (size_t)c->P.R * c->P.C, n = (size_t)c->cfg.n_fields * npx;
    if (int rc = c->scratch.ensure(n * 8)) return rc;
    DevBuf& dst = c->cfg.precision == 64 ? c->D : c->Dstage;
    if (int rc = dst.ensure(n * 8)) return rc;
    if (int rc = render_models(c, q_true, nstars, c->scratch.as<double>())) return rc;
    const int e = poisson_launch(c->stream, c->scratch.as<double>(), dst.as<double>(), n, seed, (unsigned long long)field_id_base * npx);
    if (e != 0) return fail(SRHMC_ERR_CUDA, "Poisson kernel failed: %s", cudaGetErrorString((cudaError_t)e));
    c->launches += 1;
    if (D_out) {
        if (int rc = download(c, D_out, dst, n * 8)) return rc;
    }
    return finish_data(c, n);
}

static int upload_nstars(srhmc_ctx* c, const int32_t* nstars) {
    if (!nstars) return 0;
    for (int f = 0; f < c->cfg.n_fields; ++f)
        if (nstars[f] < 0 || nstars[f] > c->cfg.max_stars)
            return fail(SRHMC_ERR_INVALID, "nstars[%d] = %d outside [0, %d]", f, nstars[f], c->cfg.max_stars);
    return upload(c, c->nstars, nstars, (size_t)c->cfg.n_fields * sizeof(int32_t));
}

int srhmc_eval(srhmc_ctx* c, const double* q, const int32_t* nstars, int32_t f_pos, double g_ff2, double beta,
               double* V, double* grad, double* H, double* Hgrad) {
    if (!c || !q) return fail(SRHMC_ERR_INVALID, "null argument");
    if (!c->have_data) return fail(SRHMC_ERR_STATE, "srhmc_set_data has not been called");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, FS = F * S * 8;
    if (int rc = upload(c, c->q, q, std::max<size_t>(FS, 8))) return rc;
    if (int rc = upload_nstars(c, nstars)) return rc;
    if (int rc = c->Vout.ensure(F * 8)) return rc;
    if (int rc = c->grad.ensure(std::max<size_t>(FS, 8))) return rc;
    if (int rc = c->H.ensure(std::max<size_t>(FS, 8))) return rc;
    if (int rc = c->Hg.ensure(std::max<size_t>(FS, 8))) return rc;
    if (int rc = c->scratch.ensure(std::max<size_t>(2 * FS, 8))) return rc;
    LaunchArgs A;
    std::memset(&A, 0, sizeof(A));
    A.mode = MODE_EVAL;
    A.n_fields = (int)F;
    A.D = c->D.ptr;
    A.D_int = c->d_int_bytes == 2 ? c->D16.ptr : (c->d_int_bytes == 4 ? c->D32.ptr : nullptr);
    A.D_int_bytes = c->d_int_bytes;
    A.log_table = reinterpret_cast<const double2*>(c->logtab.ptr);
    A.nstars = nstars ? c->nstars.as<int>() : nullptr;
    A.q_in = c->q.as<double>();
    A.f_pos = f_pos;
    A.g_ff2 = g_ff2;
    A.beta = beta;
    A.chain_stride = 1;
    A.V_out = c->Vout.as<double>();
    A.grad_out = c->grad.as<double>();
    A.H_out = c->H.as<double>();
    A.Hgrad_out = c->Hg.as<double>();
    CU_TRY(cudaMemsetAsync(c->grad.ptr, 0, std::max<size_t>(FS, 8), c->stream));
    CU_TRY(cudaMemsetAsync(c->H.ptr, 0, std::max<size_t>(FS, 8), c->stream));
    CU_TRY(cudaMemsetAsync(c->Hg.ptr, 0, std::max<size_t>(FS, 8), c->stream));
    if (int rc = launch_field(c, A, all_one_star(c, nstars))) return rc;
    if (V) if (int rc = download(c, V, c->Vout, F * 8)) return rc;
    if (grad && FS) if (int rc = download(c, grad, c->grad, FS)) return rc;
    if (H && FS) if (int rc = download(c, H, c->H, FS)) return rc;
    if (Hgrad && FS) if (int rc = download(c, Hgrad, c->Hg, FS)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int srhmc_metric(srhmc_ctx* c, const double* q, int64_t n_stars, double g_ff2, double* H, double* Hgrad) {
    if (!c || !q || n_stars < 0) return fail(SRHMC_ERR_INVALID, "bad argument");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t bytes = std::max<size_t>((size_t)n_stars * 24, 8);
    if (int rc = upload(c, c->q, q, bytes)) return rc;
    if (int rc = c->H.ensure(bytes)) return rc;
    if (int rc = c->Hg.ensure(bytes)) return rc;
    const int e = metric_launch(c->stream, c->P, (size_t)n_stars, c->q.as<double>(), g_ff2, c->H.as<double>(), c->Hg.as<double>());
    if (e != 0) return fail(SRHMC_ERR_CUDA, "metric kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
    c->launches += 1;
    if (H && n_stars) if (int rc = download(c, H, c->H, (size_t)n_stars * 24)) return rc;
    if (Hgrad && n_stars) if (int rc = download(c, Hgrad, c->Hg, (size_t)n_stars * 24)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int srhmc_kinetic(srhmc_ctx* c, const double* q, const double* p, const int32_t* nstars, double g_ff2, double* T,
                  double* dtaudq, double* dtaudp) {
    if (!c || !q || !p) return fail(SRHMC_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, FS = std::max<size_t>(F * S * 8, 8);
    if (int rc = upload(c, c->q, q, FS)) return rc;
    if (int rc = upload(c, c->p, p, FS)) return rc;
    if (int rc = upload_nstars(c, nstars)) return rc;
    if (int rc = c->Vout.ensure(F * 8)) return rc;
    if (int rc = c->grad.ensure(FS)) return rc;
    if (int rc = c->H.ensure(FS)) return rc;
    CU_TRY(cudaMemsetAsync(c->grad.ptr, 0, FS, c->stream));
    CU_TRY(cudaMemsetAsync(c->H.ptr, 0, FS, c->stream));
    const int e = kinetic_launch(c->stream, c->P, (int)F, c->q.as<double>(), c->p.as<double>(),
                                 nstars ? c->nstars.as<int>() : nullptr, g_ff2, c->Vout.as<double>(),
                                 c->grad.as<double>(), c->H.as<double>());
    if (e != 0) return fail(SRHMC_ERR_CUDA, "kinetic kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
    c->launches += 1;
    if (T) if (int rc = download(c, T, c->Vout, F * 8)) return rc;
    if (dtaudq && F * S) if (int rc = download(c, dtaudq, c->grad, F * S * 8)) return rc;
    if (dtaudp && F * S) if (int rc = download(c, dtaudp, c->H, F * S * 8)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int srhmc_kinetic_diag(srhmc_ctx* c, const double* p, const double* H_diag, int64_t n, double* T) {
    if (!c || !p || !H_diag || !T || n < 0) return fail(SRHMC_ERR_INVALID, "bad argument");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t bytes = std::max<size_t>((size_t)n * 8, 8);
    if (int rc = upload(c, c->p, p, bytes)) return rc;
    if (int rc = upload(c, c->H, H_diag, bytes)) return rc;
    if (int rc = c->Vout.ensure(8)) return rc;
    const int e = kinetic_diag_launch(c->stream, (size_t)n, c->p.as<double>(), c->H.as<double>(), c->Vout.as<double>());
    if (e != 0) return fail(SRHMC_ERR_CUDA, "kinetic kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
    c->launches += 1;
    if (int rc = download(c, T, c->Vout, 8)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int srhmc_step(srhmc_ctx* c, double* q, double* p, const int32_t* nstars, int32_t nsteps, double dt, double delta,
               int32_t counter_max, double g_ff2, double beta, int32_t* fp_counts) {
    if (!c || !q || !p) return fail(SRHMC_ERR_INVALID, "null argument");
    if (!c->have_data) return fail(SRHMC_ERR_STATE, "srhmc_set_data has not been called");
    if (nsteps < 0 || counter_max < 0) return fail(SRHMC_ERR_INVALID, "nsteps and counter_max must be >= 0");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, FS = std::max<size_t>(F * S * 8, 8);
    if (int rc = upload(c, c->q, q, FS)) return rc;
    if (int rc = upload(c, c->p, p, FS)) return rc;
    if (int rc = upload_nstars(c, nstars)) return rc;
    if (int rc = c->qout.ensure(FS)) return rc;
    if (int rc = c->pout.ensure(FS)) return rc;
    if (int rc = c->counts.ensure(F * 2 * sizeof(int))) return rc;
    if (int rc = c->scratch.ensure(2 * FS)) return rc;
    CU_TRY(cudaMemcpyAsync(c->qout.ptr, c->q.ptr, FS, cudaMemcpyDeviceToDevice, c->stream));
    CU_TRY(cudaMemcpyAsync(c->pout.ptr, c->p.ptr, FS, cudaMemcpyDeviceToDevice, c->stream));
    LaunchArgs A;
    std::memset(&A, 0, sizeof(A));
    A.mode = MODE_STEP;
    A.n_fields = (int)F;
    A.D = c->D.ptr;
    A.D_int = c->d_int_bytes == 2 ? c->D16.ptr : (c->d_int_bytes == 4 ? c->D32.ptr : nullptr);
    A.D_int_bytes = c->d_int_bytes;
    A.log_table = reinterpret_cast<const double2*>(c->logtab.ptr);
    A.nstars = nstars ? c->nstars.as<int>() : nullptr;
    A.q_in = c->q.as<double>();
    A.p_in = c->p.as<double>();
    A.q_out = c->qout.as<double>();
    A.p_out = c->pout.as<double>();
    A.nsteps = nsteps;
    A.dt = dt;
    A.delta = delta;
    A.counter_max = counter_max;
    A.g_ff2 = g_ff2;
    A.beta = beta;
    A.chain_stride = 1;
    A.fp_counts = c->counts.as<int>();
    if (int rc = launch_field(c, A, all_one_star(c, nstars))) return rc;
    if (F * S) {
        if (int rc = download(c, q, c->qout, F * S * 8)) return rc;
        if (int rc = download(c, p, c->pout, F * S * 8)) return rc;
    }
    if (fp_counts) if (int rc = download(c, fp_counts, c->counts, F * 2 * sizeof(int))) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

static int check_run_args(srhmc_ctx* c, const srhmc_run_args* a) {
    if (!c || !a) return fail(SRHMC_ERR_INVALID, "null argument");
    if (!c->have_data) return fail(SRHMC_ERR_STATE, "srhmc_set_data has not been called");
    if (a->niter < 0 || a->nsteps < 0 || a->counter_max < 0) return fail(SRHMC_ERR_INVALID, "niter, nsteps, counter_max must be >= 0");
    if (a->chain_stride < 1) return fail(SRHMC_ERR_INVALID, "chain_stride must be >= 1");
    if ((a->g_ff2_schedule && a->n_g_ff2 < 0) || (a->beta_schedule && a->n_beta < 0)) return fail(SRHMC_ERR_INVALID, "negative schedule length");
    return 0;
}

int srhmc_run_upload(srhmc_ctx* c, const srhmc_run_args* a) {
    if (int rc = check_run_args(c, a)) return rc;
    if (!a->q0) return fail(SRHMC_ERR_INVALID, "q0 is null");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, L = (size_t)a->niter + 1;
    const size_t FS = std::max<size_t>(F * S * 8, 8);
    if (int rc = upload(c, c->q, a->q0, FS)) return rc;
    if (int rc = upload_nstars(c, a->nstars)) return rc;
    c->run_has_nstars = a->nstars != nullptr;
    c->run_one_star = all_one_star(c, a->nstars);
    c->run_has_normals = a->normals != nullptr;
    c->run_has_lnu = a->lnu != nullptr;
    c->run_has_field_ids = a->field_ids != nullptr;
    if (a->field_ids) if (int rc = upload(c, c->field_ids, a->field_ids, F * sizeof(int32_t))) return rc;
    if (a->normals) if (int rc = upload(c, c->normals, a->normals, std::max<size_t>(F * L * S * 8, 8))) return rc;
    if (a->lnu) if (int rc = upload(c, c->lnu, a->lnu, F * L * 8)) return rc;
    if (a->g_ff2_schedule && a->n_g_ff2 > 0) if (int rc = upload(c, c->sg, a->g_ff2_schedule, (size_t)a->n_g_ff2 * 8)) return rc;
    if (a->beta_schedule && a->n_beta > 0) if (int rc = upload(c, c->sb, a->beta_schedule, (size_t)a->n_beta * 8)) return rc;
    c->run_L = (int)L;
    return 0;
}

static int build_run_launch_args(srhmc_ctx* c, const srhmc_run_args* a, LaunchArgs& A) {
    if (int rc = check_run_args(c, a)) return rc;
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, L = (size_t)a->niter + 1;
    if ((int)L != c->run_L) return fail(SRHMC_ERR_STATE, "srhmc_run_launch: niter differs from the uploaded run");
    const size_t rows = (L + a->chain_stride - 1) / a->chain_stride;
    c->run_rows = (int)rows;
    c->run_has_qchain = a->q_chain != nullptr && S > 0;
    const size_t FS = std::max<size_t>(F * S * 8, 8);
    if (a->q_chain) if (int rc = c->qchain.ensure(std::max<size_t>(F * rows * S * 8, 8))) return rc;
    if (a->p_chain) if (int rc = c->pchain.ensure(std::max<size_t>(F * rows * S * 8, 8))) return rc;
    if (a->E_chain) if (int rc = c->E.ensure(F * rows * 8)) return rc;
    if (a->V_chain) if (int rc = c->V.ensure(F * rows * 8)) return rc;
    if (a->T_chain) if (int rc = c->T.ensure(F * rows * 8)) return rc;
    if (a->A_chain) if (int rc = c->A.ensure(F * rows)) return rc;
    if (int rc = c->acc.ensure(F * 8)) return rc;
    if (int rc = c->qout.ensure(FS)) return rc;
    if (int rc = c->scratch.ensure(2 * FS)) return rc;
    // unused star slots of the chains read back as zeros, like the reference's np.zeros allocation
    if (a->q_chain && c->cfg.max_stars > 0 && c->run_has_nstars) CU_TRY(cudaMemsetAsync(c->qchain.ptr, 0, F * rows * S * 8, c->stream));
    if (a->p_chain && c->cfg.max_stars > 0 && c->run_has_nstars) CU_TRY(cudaMemsetAsync(c->pchain.ptr, 0, F * rows * S * 8, c->stream));
    if (c->run_has_nstars) CU_TRY(cudaMemsetAsync(c->qout.ptr, 0, FS, c->stream));
    std::memset(&A, 0, sizeof(A));
    A.mode = MODE_RUN;
    A.n_fields = (int)F;
    A.D = c->D.ptr;
    A.D_int = c->d_int_bytes == 2 ? c->D16.ptr : (c->d_int_bytes == 4 ? c->D32.ptr : nullptr);
    A.D_int_bytes = c->d_int_bytes;
    A.pix_f32 = (c->cfg.precision == 32 && c->d_int_bytes == 2) ? 1 : 0;   // (launch_field recomputes it for the chain kernel)
    A.log_table = reinterpret_cast<const double2*>(c->logtab.ptr);
    A.nstars = c->run_has_nstars ? c->nstars.as<int>() : nullptr;
    A.q_in = c->q.as<double>();
    A.q_out = c->qout.as<double>();
    A.niter = a->niter;
    A.nsteps = a->nsteps;
    A.counter_max = a->counter_max;
    A.f_pos = a->f_pos;
    A.dt = a->dt;
    A.delta = a->delta;
    A.g_ff2 = a->g_ff2;
    A.beta = a->beta;
    A.gff2_sched = (a->g_ff2_schedule && a->n_g_ff2 > 0) ? c->sg.as<double>() : nullptr;
    A.n_gff2 = a->n_g_ff2;
    A.beta_sched = (a->beta_schedule && a->n_beta > 0) ? c->sb.as<double>() : nullptr;
    A.n_beta = a->n_beta;
    A.normals = c->run_has_normals ? c->normals.as<double>() : nullptr;
    A.lnu = c->run_has_lnu ? c->lnu.as<double>() : nullptr;
    A.seed = a->seed;
    A.fid_base = a->field_id_base;
    A.fid_stride = a->field_id_stride == 0 ? 1 : a->field_id_stride;
    A.field_ids = c->run_has_field_ids ? c->field_ids.as<int>() : nullptr;
    A.chain_stride = a->chain_stride;
    A.n_rows = (int)rows;
    A.q_chain = a->q_chain ? c->qchain.as<double>() : nullptr;
    A.p_chain = a->p_chain ? c->pchain.as<double>() : nullptr;
    A.E_chain = a->E_chain ? c->E.as<double>() : nullptr;
    A.V_chain = a->V_chain ? c->V.as<double>() : nullptr;
    A.T_chain = a->T_chain ? c->T.as<double>() : nullptr;
    A.A_chain = a->A_chain ? c->A.as<unsigned char>() : nullptr;
    A.accept_rate = c->acc.as<double>();
    return 0;
}

int srhmc_run_launch(srhmc_ctx* c, const srhmc_run_args* a) {
    LaunchArgs A;
    if (int rc = build_run_launch_args(c, a, A)) return rc;
    return launch_field(c, A, c->run_one_star);
}

int srhmc_run_download(srhmc_ctx* c, const srhmc_run_args* a) {
    if (int rc = check_run_args(c, a)) return rc;
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, rows = (size_t)c->run_rows;
    if (rows == 0) return fail(SRHMC_ERR_STATE, "srhmc_run_download before srhmc_run_launch");
    if (a->q_chain && S) if (int rc = download(c, a->q_chain, c->qchain, F * rows * S * 8)) return rc;
    if (a->p_chain && S) if (int rc = download(c, a->p_chain, c->pchain, F * rows * S * 8)) return rc;
    if (a->E_chain) if (int rc = download(c, a->E_chain, c->E, F * rows * 8)) return rc;
    if (a->V_chain) if (int rc = download(c, a->V_chain, c->V, F * rows * 8)) return rc;
    if (a->T_chain) if (int rc = download(c, a->T_chain, c->T, F * rows * 8)) return rc;
    if (a->A_chain) if (int rc = download(c, a->A_chain, c->A, F * rows)) return rc;
    if (a->q_final && S) if (int rc = download(c, a->q_final, c->qout, F * S * 8)) return rc;
    if (a->accept_rate) if (int rc = download(c, a->accept_rate, c->acc, F * 8)) return rc;
    int sched_err = 0;
    if (c->sched_used) CU_TRY(cudaMemcpyAsync(&sched_err, c->sched_err.ptr, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    if (sched_err) return fail(SRHMC_ERR_CUDA, "chain kernel scheduler timed out waiting for a predecessor chunk");
    return 0;
}

// Large one-star batches: the run is cut along the ITERATION axis into kParts launches on the compute stream, and the
// chain rows a finished part produced travel device-to-host (one strided 2-D copy per output array, on a second
// stream) while the next part computes.  The chain rows are ~73 B per iteration per chain: 0.8 GB for the headline
// workload, 14.7 ms at the 55 GB/s of the link when copied after a 91.5 ms launch.  (Cutting the batch along the
// CHAIN axis instead was measured slower than no overlap at all -- 136.6 vs 106.0 ms: four concurrent part-filled
// grids defeat the chain kernel's work scheduler.)
// Iteration chunks per part of a pipelined run: the part's (group, chunk) work items should fill whole rounds of the
// resident warps.  The kernel cuts L iterations into n = n_parts * k chunks of ceil(L/n): every chunk must be non-empty,
// or its successor-less predecessor never publishes and the empty chunk waits for it (e.g. L = 385, n = 24: 23 x 17 > 385;
// L = 1001, n = 40).  Returns 0 when even n = n_parts is impossible.
static int pipelined_chunks_per_part(int L, int n_parts, long long groups, long long W) {
    auto chunks_ok = [&](int n) {
        const long long Lc = ((long long)L + n - 1) / n;
        return (long long)(n - 1) * Lc < (long long)L;
    };
    if (n_parts < 1 || !chunks_ok(n_parts)) return 0;
    int cpp = 1;
    double best = -1.0;
    for (int k = 1; k <= 8; ++k) {
        if ((long long)L < 16LL * k * n_parts) break;
        if (!chunks_ok(n_parts * k)) continue;
        const long long tasks = groups * k, rounds = (tasks + W - 1) / W;
        const double eff = (double)tasks / (double)(rounds * W);
        if (eff > best + 0.01) { best = eff; cpp = k; }
    }
    return cpp;
}

static int run_pipelined(srhmc_ctx* c, const srhmc_run_args* a, int n_parts) {
    if (int rc = srhmc_run_upload(c, a)) return rc;
    LaunchArgs A;
    if (int rc = build_run_launch_args(c, a, A)) return rc;
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, rows = (size_t)c->run_rows;
    const int L = a->niter + 1;
    if (!c->copy_stream) {
        CU_TRY(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        for (int s = 0; s < kMaxParts; ++s) CU_TRY(cudaEventCreateWithFlags(&c->part_done[s], cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&c->copies_done, cudaEventDisableTiming));
    }
    const size_t groups = (F + kChainGroup - 1) / kChainGroup;
    if (int rc = c->sched_done.ensure(groups * sizeof(int))) return rc;
    if (int rc = c->sched_state.ensure(F * 8 * sizeof(double))) return rc;
    if (int rc = c->sched_err.ensure(sizeof(int))) return rc;
    CU_TRY(cudaMemsetAsync(c->sched_done.ptr, 0, groups * sizeof(int), c->stream));
    CU_TRY(cudaMemsetAsync(c->sched_err.ptr, 0, sizeof(int), c->stream));
    A.sched_done = c->sched_done.as<int>();
    A.sched_state = c->sched_state.as<double>();
    A.sched_err = c->sched_err.as<int>();
    c->sched_used = true;
    // iteration chunks per part: the part's (group, chunk) work items should fill whole rounds of the resident warps
    const long long W = std::max<long long>(1, chain_kernel_resident_warps(A, c->chain_plan, c->sm_count, (int)F));
    const int cpp = pipelined_chunks_per_part(L, n_parts, (long long)groups, W);
    if (cpp < 1) return fail(SRHMC_ERR_INVALID, "run of %d iterations cannot be cut into %d parts", L, n_parts);
    A.n_chunks = n_parts * cpp;
    const int Lc = (L + A.n_chunks - 1) / A.n_chunks;  // the kernel's chunk length
    if (c->timed) CU_TRY(cudaEventRecord(c->ev0, c->stream));
    for (int part = 0; part < n_parts; ++part) {
        A.chunk_begin = part * cpp;
        A.chunk_count = cpp;
        const int rc = chain_kernel_launch(c->P, A, c->chain_plan, c->sm_count, c->stream);
        if (rc != 0) return fail(SRHMC_ERR_CUDA, "chain kernel launch failed: %s", cudaGetErrorString((cudaError_t)rc));
        c->launches += 1;
        CU_TRY(cudaEventRecord(c->part_done[part], c->stream));
        CU_TRY(cudaStreamWaitEvent(c->copy_stream, c->part_done[part], 0));
        const size_t r0 = std::min<size_t>((size_t)part * cpp * Lc, rows), r1 = std::min<size_t>(r0 + (size_t)cpp * Lc, rows);
        auto d2h_rows = [&](void* dst, const DevBuf& b, size_t row_bytes) -> int {
            if (!dst || row_bytes == 0 || r1 <= r0) return 0;
            CU_TRY(cudaMemcpy2DAsync((char*)dst + r0 * row_bytes, rows * row_bytes, (const char*)b.ptr + r0 * row_bytes,
                                     rows * row_bytes, (r1 - r0) * row_bytes, F, cudaMemcpyDeviceToHost, c->copy_stream));
            return 0;
        };
        if (int rc2 = d2h_rows(a->q_chain, c->qchain, S * 8)) return rc2;
        if (int rc2 = d2h_rows(a->p_chain, c->pchain, S * 8)) return rc2;
        if (int rc2 = d2h_rows(a->E_chain, c->E, 8)) return rc2;
        if (int rc2 = d2h_rows(a->V_chain, c->V, 8)) return rc2;
        if (int rc2 = d2h_rows(a->T_chain, c->T, 8)) return rc2;
    }
    if (c->timed) CU_TRY(cudaEventRecord(c->ev1, c->stream));
    // byte-wide rows and the per-chain results go in one piece after the last part
    if (a->A_chain) CU_TRY(cudaMemcpyAsync(a->A_chain, c->A.ptr, F * rows, cudaMemcpyDeviceToHost, c->copy_stream));
    if (a->q_final && S) CU_TRY(cudaMemcpyAsync(a->q_final, c->qout.ptr, F * S * 8, cudaMemcpyDeviceToHost, c->copy_stream));
    if (a->accept_rate) CU_TRY(cudaMemcpyAsync(a->accept_rate, c->acc.ptr, F * 8, cudaMemcpyDeviceToHost, c->copy_stream));
    CU_TRY(cudaEventRecord(c->copies_done, c->copy_stream));
    CU_TRY(cudaStreamWaitEvent(c->stream, c->copies_done, 0));
    int sched_err = 0;
    CU_TRY(cudaMemcpyAsync(&sched_err, c->sched_err.ptr, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    if (sched_err) return fail(SRHMC_ERR_CUDA, "chain kernel scheduler timed out waiting for a predecessor chunk");
    return 0;
}

int srhmc_plan_chunks(int64_t groups, int64_t resident_warps, int32_t n_iterations, int32_t n_parts) {
    if (groups < 1 || resident_warps < 1 || n_iterations < 1 || n_parts < 0) return 0;
    if (n_parts == 0) return pick_chunks(groups, resident_warps, n_iterations);
    return n_parts * pipelined_chunks_per_part(n_iterations, n_parts, groups, resident_warps);
}

int srhmc_run(srhmc_ctx* c, const srhmc_run_args* a) {
    if (c && a && c->chain_ok && (c->cfg.precision == 64 || c->d_int_bytes == 2) && c->cfg.n_fields >= 4096 &&
        a->niter + 1 >= 256 && a->chain_stride == 1 && all_one_star(c, a->nstars)) {
        int parts = 8;  // measured on the headline batch: 1 part 106.0 ms, 2: 102.6, 4: 98.9, 8: 97.6 (kernel alone 91.7)
        if (const char* e = std::getenv("SRHMC_RUN_PARTS")) parts = std::max(1, std::min(kMaxParts, std::atoi(e)));
        if (parts > 1) return run_pipelined(c, a, parts);
    }
    if (int rc = srhmc_run_upload(c, a)) return rc;
    if (int rc = srhmc_run_launch(c, a)) return rc;
    return srhmc_run_download(c, a);
}

int srhmc_run_single(srhmc_ctx* c, const double* q0, const double* p0, const int32_t* nstars, int32_t nsteps, double dt,
                     double delta, int32_t counter_max, int32_t f_pos, double g_ff2, double beta, double* q_chain,
                     double* p_chain, double* E_chain, double* V_chain, double* T_chain) {
    if (!c || !q0 || !p0) return fail(SRHMC_ERR_INVALID, "null argument");
    if (!c->have_data) return fail(SRHMC_ERR_STATE, "srhmc_set_data has not been called");
    if (nsteps < 0 || counter_max < 0) return fail(SRHMC_ERR_INVALID, "nsteps and counter_max must be >= 0");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, rows = (size_t)nsteps + 1;
    const size_t FS = std::max<size_t>(F * S * 8, 8);
    if (int rc = upload(c, c->q, q0, FS)) return rc;
    if (int rc = upload(c, c->p, p0, FS)) return rc;
    if (int rc = upload_nstars(c, nstars)) return rc;
    if (int rc = c->qchain.ensure(std::max<size_t>(F * rows * S * 8, 8))) return rc;
    if (int rc = c->pchain.ensure(std::max<size_t>(F * rows * S * 8, 8))) return rc;
    if (int rc = c->E.ensure(F * rows * 8)) return rc;
    if (int rc = c->V.ensure(F * rows * 8)) return rc;
    if (int rc = c->T.ensure(F * rows * 8)) return rc;
    if (int rc = c->scratch.ensure(2 * FS)) return rc;
    if (S) {
        CU_TRY(cudaMemsetAsync(c->qchain.ptr, 0, F * rows * S * 8, c->stream));
        CU_TRY(cudaMemsetAsync(c->pchain.ptr, 0, F * rows * S * 8, c->stream));
    }
    LaunchArgs A;
    std::memset(&A, 0, sizeof(A));
    A.mode = MODE_SINGLE;
    A.n_fields = (int)F;
    A.D = c->D.ptr;
    A.D_int = c->d_int_bytes == 2 ? c->D16.ptr : (c->d_int_bytes == 4 ? c->D32.ptr : nullptr);
    A.D_int_bytes = c->d_int_bytes;
    A.log_table = reinterpret_cast<const double2*>(c->logtab.ptr);
    A.nstars = nstars ? c->nstars.as<int>() : nullptr;
    A.q_in = c->q.as<double>();
    A.p_in = c->p.as<double>();
    A.nsteps = nsteps;
    A.counter_max = counter_max;
    A.f_pos = f_pos;
    A.dt = dt;
    A.delta = delta;
    A.g_ff2 = g_ff2;
    A.beta = beta;
    A.chain_stride = 1;
    A.n_rows = (int)rows;
    A.q_chain = c->qchain.as<double>();
    A.p_chain = c->pchain.as<double>();
    A.E_chain = c->E.as<double>();
    A.V_chain = c->V.as<double>();
    A.T_chain = c->T.as<double>();
    if (int rc = launch_field(c, A, all_one_star(c, nstars))) return rc;
    if (q_chain && S) if (int rc = download(c, q_chain, c->qchain, F * rows * S * 8)) return rc;
    if (p_chain && S) if (int rc = download(c, p_chain, c->pchain, F * rows * S * 8)) return rc;
    if (E_chain) if (int rc = download(c, E_chain, c->E, F * rows * 8)) return rc;
    if (V_chain) if (int rc = download(c, V_chain, c->V, F * rows * 8)) return rc;
    if (T_chain) if (int rc = download(c, T_chain, c->T, F * rows * 8)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

static int ls_common(srhmc_ctx* c, LsArgs& A, const double* q0, const double* p0, const int32_t* nstars) {
    if (!c->have_data) return fail(SRHMC_ERR_STATE, "srhmc_set_data has not been called");
    if (c->cfg.precision != 64) return fail(SRHMC_ERR_INVALID, "the lightsource_gym entry points need a precision=64 context");
    if (c->cfg.use_prior || c->cfg.use_Vc) return fail(SRHMC_ERR_INVALID, "lightsource_gym has no prior / repulsion: create the context with use_prior = use_Vc = 0");
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, FS = std::max<size_t>(F * S * 8, 8);
    if (int rc = upload(c, c->q, q0, FS)) return rc;
    if (p0) if (int rc = upload(c, c->p, p0, FS)) return rc;
    if (int rc = upload_nstars(c, nstars)) return rc;
    if (int rc = c->ls_scratch.ensure(5 * FS)) return rc;
    std::memset(&A, 0, sizeof(A));
    A.n_fields = (int)F;
    A.D = c->D.ptr;
    A.nstars = nstars ? c->nstars.as<int>() : nullptr;
    A.q0 = c->q.as<double>();
    A.p0 = p0 ? c->p.as<double>() : nullptr;
    return 0;
}

static int ls_launch(srhmc_ctx* c, const LsArgs& A) {
    if (c->timed) CU_TRY(cudaEventRecord(c->ev0, c->stream));
    const int rc = ls_kernel_launch(c->kc.mr, c->kc.mc, std::max(1, A.n_fields), c->threads, c->smem, c->stream, c->P_ls, A,
                                    c->ls_scratch.as<double>(), c->dsm_ls);
    if (rc != 0) return fail(SRHMC_ERR_CUDA, "lightsource kernel launch failed: %s", cudaGetErrorString((cudaError_t)rc));
    if (c->timed) CU_TRY(cudaEventRecord(c->ev1, c->stream));
    c->launches += 1;
    return 0;
}

int srhmc_ls_run(srhmc_ctx* c, const srhmc_ls_args* a) {
    if (!c || !a || !a->q0 || !a->dt || !a->normals || !a->lnu || !a->steps) return fail(SRHMC_ERR_INVALID, "null argument");
    if (a->variant < SRHMC_LS_HMC || a->variant > SRHMC_LS_TRIAL) return fail(SRHMC_ERR_INVALID, "unknown variant %d", a->variant);
    if (a->niter < 0) return fail(SRHMC_ERR_INVALID, "niter must be >= 0");
    if (a->variant == SRHMC_LS_HESS && !c->P.hess) return fail(SRHMC_ERR_STATE, "context was created without enable_hessian");
    if (a->variant == SRHMC_LS_TRIAL && c->cfg.max_stars != 1) return fail(SRHMC_ERR_INVALID, "the step-size trial is a one-star problem");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, L = (size_t)a->niter + 1, n = (size_t)a->niter;
    const size_t need_dt = a->variant == SRHMC_LS_DIAG ? 1 : S;
    if ((size_t)a->n_dt < need_dt) return fail(SRHMC_ERR_INVALID, "dt has %d entries, %zu needed", a->n_dt, need_dt);
    for (size_t i = 0; i < F * n; ++i)
        if (a->steps[i] < 0) return fail(SRHMC_ERR_INVALID, "negative trajectory length");
    LsArgs A;
    if (int rc = ls_common(c, A, a->q0, nullptr, a->nstars)) return rc;
    if (int rc = upload(c, c->ls_dt, a->dt, std::max<size_t>(need_dt * 8, 8))) return rc;
    if (int rc = upload(c, c->normals, a->normals, std::max<size_t>(F * L * S * 8, 8))) return rc;
    if (int rc = upload(c, c->lnu, a->lnu, std::max<size_t>(F * n * 8, 8))) return rc;
    if (int rc = upload(c, c->ls_steps, a->steps, std::max<size_t>(F * n * 4, 8))) return rc;
    c->run_has_normals = c->run_has_lnu = false;  // staging buffers of srhmc_run were overwritten
    if (a->background) if (int rc = upload(c, c->ls_bg, a->background, F * (size_t)c->P.R * c->P.C * 8)) return rc;
    if (int rc = c->qchain.ensure(std::max<size_t>(F * L * S * 8, 8))) return rc;
    if (int rc = c->E.ensure(F * L * 8)) return rc;
    if (int rc = c->V.ensure(F * L * 8)) return rc;
    if (int rc = c->A.ensure(std::max<size_t>(F * n, 8))) return rc;
    if (int rc = c->qout.ensure(std::max<size_t>(F * S * 8, 8))) return rc;
    if (int rc = c->acc.ensure(F * 8)) return rc;
    CU_TRY(cudaMemsetAsync(c->qchain.ptr, 0, std::max<size_t>(F * L * S * 8, 8), c->stream));
    CU_TRY(cudaMemsetAsync(c->E.ptr, 0, F * L * 8, c->stream));
    CU_TRY(cudaMemsetAsync(c->V.ptr, 0, F * L * 8, c->stream));
    CU_TRY(cudaMemsetAsync(c->A.ptr, 0, std::max<size_t>(F * n, 8), c->stream));
    A.variant = a->variant;
    A.niter = a->niter;
    A.dt = c->ls_dt.as<double>();
    A.f_lim = a->f_lim;
    A.factor1 = a->factor1;
    A.normals = c->normals.as<double>();
    A.steps = c->ls_steps.as<int>();
    A.lnu = c->lnu.as<double>();
    A.background = a->background ? c->ls_bg.as<double>() : nullptr;
    A.zero_xy = a->zero_xy_momentum;
    A.q_chain = c->qchain.as<double>();
    A.E_chain = c->E.as<double>();
    A.dE_chain = c->V.as<double>();
    A.A_chain = c->A.as<unsigned char>();
    A.q_final = c->qout.as<double>();
    A.accept_count = c->acc.as<double>();
    if (int rc = ls_launch(c, A)) return rc;
    if (a->q_chain && S) if (int rc = download(c, a->q_chain, c->qchain, F * L * S * 8)) return rc;
    if (a->E_chain) if (int rc = download(c, a->E_chain, c->E, F * L * 8)) return rc;
    if (a->dE_chain) if (int rc = download(c, a->dE_chain, c->V, F * L * 8)) return rc;
    if (a->A_chain && n) if (int rc = download(c, a->A_chain, c->A, F * n)) return rc;
    if (a->q_final && S) if (int rc = download(c, a->q_final, c->qout, F * S * 8)) return rc;
    if (a->accept_count) if (int rc = download(c, a->accept_count, c->acc, F * 8)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int srhmc_eval_background(srhmc_ctx* c, const double* q, const int32_t* nstars, const double* background, double* V,
                          double* grad) {
    if (!c || !q || !background) return fail(SRHMC_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, FS = std::max<size_t>(F * S * 8, 8);
    LsArgs A;
    if (int rc = ls_common(c, A, q, nullptr, nstars)) return rc;
    if (int rc = upload(c, c->ls_bg, background, F * (size_t)c->P.R * c->P.C * 8)) return rc;
    if (int rc = c->ls_d1.ensure(FS)) return rc;
    if (int rc = c->Vout.ensure(F * 8)) return rc;
    CU_TRY(cudaMemsetAsync(c->ls_d1.ptr, 0, FS, c->stream));
    A.variant = LS_EVAL_BG;
    A.background = c->ls_bg.as<double>();
    A.d1 = c->ls_d1.as<double>();
    A.E_out = c->Vout.as<double>();
    if (int rc = ls_launch(c, A)) return rc;
    if (V) if (int rc = download(c, V, c->Vout, F * 8)) return rc;
    if (grad && F * S) if (int rc = download(c, grad, c->ls_d1, F * S * 8)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int srhmc_hessian(srhmc_ctx* c, const double* q, const double* p, const int32_t* nstars, double f_lim, int32_t d2_only,
                  double* d1, double* d2, double* d3, double* dqdt, double* dpdt, double* E) {
    if (!c || !q) return fail(SRHMC_ERR_INVALID, "null argument");
    if (!d2_only && !p) return fail(SRHMC_ERR_INVALID, "p is required unless d2_only");
    if (!c->P.hess) return fail(SRHMC_ERR_STATE, "context was created without enable_hessian");
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, S = 3 * (size_t)c->cfg.max_stars, FS = std::max<size_t>(F * S * 8, 8);
    LsArgs A;
    if (int rc = ls_common(c, A, q, p, nstars)) return rc;
    DevBuf* outs[] = {&c->ls_d1, &c->ls_d2, &c->ls_d3, &c->grad, &c->H};
    for (DevBuf* b : outs) {
        if (int rc = b->ensure(FS)) return rc;
        CU_TRY(cudaMemsetAsync(b->ptr, 0, FS, c->stream));
    }
    if (int rc = c->Vout.ensure(F * 8)) return rc;
    A.variant = LS_EVAL_HESS;
    A.f_lim = f_lim;
    A.d2_only = d2_only ? 1 : 0;
    A.d1 = c->ls_d1.as<double>();
    A.d2 = c->ls_d2.as<double>();
    A.d3 = c->ls_d3.as<double>();
    A.dqdt = c->grad.as<double>();
    A.dpdt = c->H.as<double>();
    A.E_out = c->Vout.as<double>();
    if (int rc = ls_launch(c, A)) return rc;
    if (F * S) {
        if (d2) if (int rc = download(c, d2, c->ls_d2, F * S * 8)) return rc;
        if (!d2_only) {
            if (d1) if (int rc = download(c, d1, c->ls_d1, F * S * 8)) return rc;
            if (d3) if (int rc = download(c, d3, c->ls_d3, F * S * 8)) return rc;
            if (dqdt) if (int rc = download(c, dqdt, c->grad, F * S * 8)) return rc;
            if (dpdt) if (int rc = download(c, dpdt, c->H, F * S * 8)) return rc;
        }
    }
    if (E && !d2_only) if (int rc = download(c, E, c->Vout, F * 8)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}


int srhmc_convergence_stats(int32_t device, const double* q_chain, int64_t n_chains, int64_t n_iter, int32_t d, int32_t n_groups,
                            int32_t thin_rate, int32_t warm_up_num, double* R, double* n_eff) {
    if (!q_chain || !R || !n_eff) return fail(SRHMC_ERR_INVALID, "null argument");
    if (int rc = check_stats_args(n_chains, n_iter, d, n_groups, thin_rate, warm_up_num)) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(SRHMC_ERR_NO_DEVICE, "no CUDA device visible: this library has no CPU path");
    if (device < 0 || device >= ndev) return fail(SRHMC_ERR_INVALID, "device %d out of range (%d visible)", device, ndev);
    CU_TRY(cudaSetDevice(device));
    const int cpg = (int)(n_chains / n_groups);
    const size_t nx = (size_t)n_chains * n_iter * d, nout = (size_t)n_groups * d;
    DevBuf X, means, out;
    int rc = X.ensure(nx * 8);
    if (!rc) rc = means.ensure(conv_stats_scratch_doubles(n_iter, d, n_groups, cpg, thin_rate, warm_up_num) * 8);
    if (!rc) rc = out.ensure(2 * nout * 8);
    cudaError_t e = cudaSuccess;
    if (!rc) e = cudaMemcpy(X.ptr, q_chain, nx * 8, cudaMemcpyHostToDevice);
    if (!rc && e == cudaSuccess)
        e = (cudaError_t)conv_stats_launch(nullptr, X.as<double>(), n_iter, d, n_groups, cpg, thin_rate, warm_up_num, means.as<double>(),
                                           out.as<double>(), out.as<double>() + nout);
    if (!rc && e == cudaSuccess) e = cudaMemcpy(R, out.ptr, nout * 8, cudaMemcpyDeviceToHost);
    if (!rc && e == cudaSuccess) e = cudaMemcpy(n_eff, out.as<double>() + nout, nout * 8, cudaMemcpyDeviceToHost);
    X.release(); means.release(); out.release();
    if (rc) return rc;
    if (e != cudaSuccess) return fail(SRHMC_ERR_CUDA, "chain statistics failed: %s", cudaGetErrorString(e));
    return 0;
}

int srhmc_run_stats(srhmc_ctx* c, int32_t n_groups, int32_t thin_rate, int32_t warm_up_num, double* R, double* n_eff) {
    if (!c || !R || !n_eff) return fail(SRHMC_ERR_INVALID, "null argument");
    if (!c->run_has_qchain || c->run_rows == 0)
        return fail(SRHMC_ERR_STATE, "no resident q_chain: launch a run with q_chain requested first (srhmc_run_launch)");
    const int d = 3 * c->cfg.max_stars;
    if (int rc = check_stats_args(c->cfg.n_fields, c->run_rows, d, n_groups, thin_rate, warm_up_num)) return rc;
    CU_TRY(cudaSetDevice(c->cfg.device));
    const int cpg = c->cfg.n_fields / n_groups;
    const size_t nout = (size_t)n_groups * d;
    if (int rc = c->st_means.ensure(conv_stats_scratch_doubles(c->run_rows, d, n_groups, cpg, thin_rate, warm_up_num) * 8)) return rc;
    if (int rc = c->st_R.ensure(nout * 8)) return rc;
    if (int rc = c->st_neff.ensure(nout * 8)) return rc;
    const int e = conv_stats_launch(c->stream, c->qchain.as<double>(), c->run_rows, d, n_groups, cpg, thin_rate, warm_up_num,
                                    c->st_means.as<double>(), c->st_R.as<double>(), c->st_neff.as<double>());
    if (e != 0) return fail(SRHMC_ERR_CUDA, "chain statistics kernel failed: %s", cudaGetErrorString((cudaError_t)e));
    c->launches += 1;
    if (int rc = download(c, R, c->st_R, nout * 8)) return rc;
    if (int rc = download(c, n_eff, c->st_neff, nout * 8)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int srhmc_find_peaks_descend(srhmc_ctx* c, double* q_seed, int32_t n, int32_t nstep, double dt_f_coeff, double dt_xy_coeff,
                             double f_lim, uint8_t* alive, int32_t* steps_taken) {
    if (!c || !q_seed || !alive || n < 0 || nstep < 0) return fail(SRHMC_ERR_INVALID, "bad argument");
    if (!c->have_data) return fail(SRHMC_ERR_STATE, "srhmc_set_data has not been called");
    if (c->cfg.precision != 64) return fail(SRHMC_ERR_INVALID, "find_peaks runs on FP64 contexts");
    if (n == 0) return 0;
    CU_TRY(cudaSetDevice(c->cfg.device));
    DevBuf q, a, st;
    int rc = q.ensure((size_t)n * 24);
    if (!rc) rc = a.ensure((size_t)n);
    if (!rc) rc = st.ensure((size_t)n * 4);
    cudaError_t e = cudaSuccess;
    if (!rc) e = cudaMemcpyAsync(q.ptr, q_seed, (size_t)n * 24, cudaMemcpyHostToDevice, c->stream);
    if (!rc && e == cudaSuccess)
        e = (cudaError_t)peaks_launch(c->stream, c->P, c->D.as<double>(), n, nstep, dt_f_coeff, dt_xy_coeff, f_lim, q.as<double>(),
                                      a.as<unsigned char>(), st.as<int>());
    if (!rc && e == cudaSuccess) {
        c->launches += 1;
        e = cudaMemcpyAsync(q_seed, q.ptr, (size_t)n * 24, cudaMemcpyDeviceToHost, c->stream);
    }
    if (!rc && e == cudaSuccess) e = cudaMemcpyAsync(alive, a.ptr, (size_t)n, cudaMemcpyDeviceToHost, c->stream);
    if (!rc && e == cudaSuccess && steps_taken) e = cudaMemcpyAsync(steps_taken, st.ptr, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream);
    if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    q.release(); a.release(); st.release();
    if (rc) return rc;
    if (e != cudaSuccess) return fail(SRHMC_ERR_CUDA, "find_peaks descent failed: %s", cudaGetErrorString(e));
    return 0;
}

int srhmc_philox_draws(srhmc_ctx* c, uint64_t seed, int32_t niter, double* normals, double* lnu) {
    return srhmc_philox_draws_ids(c, seed, niter, 0, 1, normals, lnu);
}

int srhmc_philox_draws_ids(srhmc_ctx* c, uint64_t seed, int32_t niter, int32_t fid_base, int32_t fid_stride, double* normals,
                           double* lnu) {
    if (!c || !normals || !lnu || niter < 0) return fail(SRHMC_ERR_INVALID, "bad argument");
    if (fid_stride == 0) fid_stride = 1;
    CU_TRY(cudaSetDevice(c->cfg.device));
    const size_t F = c->cfg.n_fields, N = (size_t)c->cfg.max_stars, L = (size_t)niter + 1;
    if (N == 0) return fail(SRHMC_ERR_INVALID, "max_stars is 0");
    if (int rc = c->normals.ensure(F * L * N * 3 * 8)) return rc;
    if (int rc = c->lnu.ensure(F * L * 8)) return rc;
    const int e = philox_dump_launch(c->stream, seed, (int)F, (int)L, (int)N, fid_base, fid_stride, c->normals.as<double>(),
                                     c->lnu.as<double>());
    if (e != 0) return fail(SRHMC_ERR_CUDA, "philox dump failed: %s", cudaGetErrorString((cudaError_t)e));
    c->launches += 1;
    if (int rc = download(c, normals, c->normals, F * L * N * 3 * 8)) return rc;
    if (int rc = download(c, lnu, c->lnu, F * L * 8)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    c->run_has_normals = false;  // the staging buffers were overwritten
    c->run_has_lnu = false;
    return 0;
}

int srhmc_test_device_math(srhmc_ctx* c, int32_t which, const double* x, double* y, int32_t n) {
    if (!c || !x || !y || n < 0 || which < 0 || which > 2) return fail(SRHMC_ERR_INVALID, "bad argument");
    CU_TRY(cudaSetDevice(c->cfg.device));
    if (int rc = upload(c, c->Dstage, x, std::max<size_t>((size_t)n * 8, 8))) return rc;
    if (int rc = c->grad.ensure(std::max<size_t>((size_t)n * 8, 8))) return rc;
    const int e = math_test_launch(c->stream, which, c->Dstage.as<double>(), c->grad.as<double>(), n, c->logtab.as<double>());
    if (e != 0) return fail(SRHMC_ERR_CUDA, "math test kernel failed: %s", cudaGetErrorString((cudaError_t)e));
    c->launches += 1;
    if (n) if (int rc = download(c, y, c->grad, (size_t)n * 8)) return rc;
    CU_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int srhmc_measure_fma_peak(int32_t device, int32_t precision, double* tflops, float* ms) {
    if (!tflops) return fail(SRHMC_ERR_INVALID, "null argument");
    if (precision != 64 && precision != 32) return fail(SRHMC_ERR_INVALID, "precision must be 64 or 32");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(SRHMC_ERR_NO_DEVICE, "no CUDA device visible");
    if (device < 0 || device >= ndev) return fail(SRHMC_ERR_INVALID, "device out of range");
    CU_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    const int e = fma_peak_run(precision, prop.multiProcessorCount, tflops, ms);
    if (e != 0) return fail(SRHMC_ERR_CUDA, "FMA peak microbenchmark failed: %s", cudaGetErrorString((cudaError_t)e));
    return 0;
}

}  // extern "C"
