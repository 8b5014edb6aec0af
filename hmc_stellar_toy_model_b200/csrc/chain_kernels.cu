// Warp-resident one-star chain kernel: instantiations, occupancy plan, launcher, and the device-math test hook.
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "chain_kernel.cuh"
#include "kernels_api.h"

namespace srhmc {

namespace {

constexpr int kLPC = kChainLPC;  // lanes per chain: 4 -> 8 chains per warp (measured: 16 lanes 734, 8 lanes 1104, 4 lanes 1210 M star-steps/s)
// Column slots per lane: the full 32-column image, or a 24-column window around the star when the PSF weight of
// every dropped column is below 2^-46 of its peak (sigma <= 1.50 px: |dy| >= 12 px).  SRHMC_CHAIN_WINDOW=0 at run time
// forces the full width, so that the tests can compare the two.
constexpr int kSlotsFull = 32 / kLPC;
constexpr int kWinCols = 24;
constexpr int kSlotsWin = kWinCols / kLPC;

bool use_column_window(const FieldParams& P) {
    if (const char* env = std::getenv("SRHMC_CHAIN_WINDOW"))
        if (std::atoi(env) == 0) return false;
    const double half = 0.5 * kWinCols;
    return half * half * P.inv2s2 >= 46.0 * M_LN2;
}

// one single-warp block: the log table and kChainGroup chains of image copy and row tables
size_t chain_smem_bytes(const FieldParams& P, size_t elem, bool f32) { return chain_layout(P.R, elem, f32).smem_bytes; }

template <typename DT, int MODE, int NCS, typename PT = double>
int configure_mode(size_t smem, int& blocks_per_sm) {
    auto fn = chain_kernel<kLPC, DT, MODE, NCS, kChainMaxReg, PT>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    e = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return (int)e;
    int nb = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, kWarp, smem);
    if (e != cudaSuccess) return (int)e;
    if (nb < 1) return (int)cudaErrorInvalidConfiguration;
    blocks_per_sm = blocks_per_sm == 0 ? nb : std::min(blocks_per_sm, nb);
    return 0;
}

template <typename DT, int NCS, typename PT = double>
int configure_slots(size_t smem, int& blocks_per_sm) {
    if (int rc = configure_mode<DT, MODE_EVAL, NCS, PT>(smem, blocks_per_sm)) return rc;
    if (int rc = configure_mode<DT, MODE_STEP, NCS, PT>(smem, blocks_per_sm)) return rc;
    if (int rc = configure_mode<DT, MODE_RUN, NCS, PT>(smem, blocks_per_sm)) return rc;
    return configure_mode<DT, MODE_SINGLE, NCS, PT>(smem, blocks_per_sm);
}

template <typename DT, typename PT = double>
int configure_one(const FieldParams& P, size_t& smem, int& blocks_per_sm) {
    smem = chain_smem_bytes(P, sizeof(DT), sizeof(PT) == 4);
    blocks_per_sm = 0;
    return use_column_window(P) ? configure_slots<DT, kSlotsWin, PT>(smem, blocks_per_sm)
                                : configure_slots<DT, kSlotsFull, PT>(smem, blocks_per_sm);
}

template <typename DT, int NCS, typename PT = double>
void launch_slots(int grid, size_t smem, cudaStream_t stream, const FieldParams& P, const LaunchArgs& A) {
    switch (A.mode) {
        case MODE_EVAL: chain_kernel<kLPC, DT, MODE_EVAL, NCS, kChainMaxReg, PT><<<grid, kWarp, smem, stream>>>(P, A); break;
        case MODE_STEP: chain_kernel<kLPC, DT, MODE_STEP, NCS, kChainMaxReg, PT><<<grid, kWarp, smem, stream>>>(P, A); break;
        case MODE_SINGLE: chain_kernel<kLPC, DT, MODE_SINGLE, NCS, kChainMaxReg, PT><<<grid, kWarp, smem, stream>>>(P, A); break;
        default: chain_kernel<kLPC, DT, MODE_RUN, NCS, kChainMaxReg, PT><<<grid, kWarp, smem, stream>>>(P, A); break;
    }
}

template <typename DT, typename PT = double>
void launch_mode(int grid, size_t smem, cudaStream_t stream, const FieldParams& P, const LaunchArgs& A) {
    if (use_column_window(P))
        launch_slots<DT, kSlotsWin, PT>(grid, smem, stream, P, A);
    else
        launch_slots<DT, kSlotsFull, PT>(grid, smem, stream, P, A);
}

// Grid = (blocks per SM) x SMs with the per-SM count chosen so that every SM runs the same number of equally long
// rounds (all chains of one launch run the same number of iterations).
int balanced_grid(int max_blocks_per_sm, long long blocks_needed, int sms) {
    const long long cap = (long long)max_blocks_per_sm * sms;
    if (blocks_needed <= cap) return (int)std::max<long long>(1, blocks_needed);
    // k resident warps per SM run ceil(needed / (k sms)) rounds; a round costs ~k (throughput-bound) but never less
    // than ~kSat/2 (latency-bound), so prefer the largest k among near-ties.
    const int k_lo = std::max(1, (3 * max_blocks_per_sm) / 4);
    int best_k = max_blocks_per_sm;
    double best_cost = -1.0;
    for (int k = max_blocks_per_sm; k >= k_lo; --k) {
        const long long rounds = (blocks_needed + (long long)k * sms - 1) / ((long long)k * sms);
        const double cost = (double)rounds * k;
        if (best_cost < 0 || cost < best_cost * 0.97) {
            best_cost = cost;
            best_k = k;
        }
    }
    return best_k * sms;
}

__global__ void math_test_kernel(int which, const double* x, double* y, int n, const double2* log_table) {
    __shared__ double2 tab[kLogTableSize];
    for (int i = threadIdx.x; i < kLogTableSize; i += blockDim.x) tab[i] = log_table[i];
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const double v = x[i];
        y[i] = which == 0 ? exp_neg(v) : (which == 1 ? log_pos(v, tab) : rcp_fast(v));
    }
}

// exact-count image check + conversion.  flags bit 0: a pixel is not a uint32-representable integer; bit 1: a pixel
// exceeds 65535 (the uint16 copy is then unusable).
__global__ void to_counts_kernel(const double* src, unsigned int* dst32, unsigned short* dst16, size_t n, int* flags) {
    int bad = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const double v = src[i];
        const bool ok = (v >= 0.0) && (v <= 4294967295.0) && (v == floor(v));
        bad |= ok ? 0 : 1;
        bad |= (ok && v <= 65535.0) ? 0 : 2;
        dst32[i] = ok ? (unsigned int)v : 0u;
        dst16[i] = (ok && v <= 65535.0) ? (unsigned short)v : (unsigned short)0;
    }
    if (bad) atomicOr(flags, bad);
}

}  // namespace

void fill_log_table(double* host_table /* [kLogTableSize*2] */) {
    for (int k = 0; k < kLogTableSize; ++k) {
        const long double c = 1.0L + ((long double)k + 0.5L) / (long double)kLogTableSize;
        const double rc = (double)(1.0L / c);
        host_table[2 * k] = rc;
        host_table[2 * k + 1] = (double)(-logl((long double)rc));
    }
}

int chain_kernel_window_cols(const FieldParams& P) { return use_column_window(P) ? kWinCols : kLPC * kSlotsFull; }

ChainLayout chain_kernel_layout(int R, size_t elem, bool f32) { return chain_layout(R, elem, f32); }

// chain_eval starts each lane's column table at its first column jb with e = exp(-arg_c), arg_c = v0^2/2s^2, v0 = jb + .5 - y,
// and the ratio r_c = exp(-(2 L v0 + L^2)/2s^2), then multiplies its way along the row.  It zeroes the whole table when
// arg_c >= 690, and exp_neg overflows for arguments above ~709.  The window start jb moves in steps of one column when
// y - 12.5 crosses an integer, so |v0| is extreme at the support's ends or at such a crossing, all of which lie on the
// 1/16-pixel grid of y scanned here.
double chain_column_exponent(const FieldParams& P, int win) {
    double worst = 0.0;
    for (int k = 0; k <= 16 * (P.C + 2); ++k) {
        const double y = -1.0 + k / 16.0;
        for (int sub = 0; sub < kLPC; ++sub) {
            int jb = sub;
            if (win < kChainCS) {
                const double a = std::ceil(y - (0.5 + 0.5 * win));
                jb += (int)std::fmin(std::fmax(a, 0.0), (double)std::max(P.C - win, 0));
            }
            const double v0 = ((double)jb + 0.5) - y;
            worst = std::max(worst, std::max(v0 * v0, -(2.0 * kLPC * v0 + kLPC * kLPC)) * P.inv2s2);
        }
    }
    return worst;
}

bool chain_kernel_psf_ok(const FieldParams& P) { return chain_column_exponent(P, chain_kernel_window_cols(P)) <= kChainExpMax; }

int chain_kernel_configure(const FieldParams& P, ChainLaunchPlan& plan) {
    if (int rc = configure_one<double>(P, plan.smem_f64, plan.blocks_per_sm_f64)) return rc;
    if (int rc = configure_one<unsigned int>(P, plan.smem_u32, plan.blocks_per_sm_u32)) return rc;
    if (int rc = configure_one<unsigned short>(P, plan.smem_u16, plan.blocks_per_sm_u16)) return rc;
    // FP32 pixel arithmetic (precision-32 contexts) on the uint16 count images
    return configure_one<unsigned short, float>(P, plan.smem_u16_f32, plan.blocks_per_sm_u16_f32);
}

// Iteration chunks per chain for a MODE_RUN launch of `groups` warp-sized work items on `warps` resident warps.
// One chunk when everything is resident at once (or the chains are short); otherwise enough chunks that the
// under-filled last round costs a few percent instead of up to half the launch.
// The kernel cuts L iterations into n chunks of ceil(L/n) iterations; every chunk must be non-empty (an empty last chunk
// would wait for a predecessor that, being the real last one, never publishes): largest n' <= n with (n'-1) ceil(L/n') < L.
static int valid_chunks(int n, int L) {
    n = std::max(1, std::min(n, L));
    while (n > 1 && (long long)(n - 1) * (((long long)L + n - 1) / n) >= (long long)L) --n;
    return n;
}

int pick_chunks(long long groups, long long warps, int L) {
    if (const char* env = std::getenv("SRHMC_CHAIN_CHUNKS")) {
        const int c = std::atoi(env);
        if (c >= 1) return valid_chunks(c, L);
    }
    if (groups <= warps || L < 64) return 1;
    return valid_chunks(std::min(16, L / 32), L);
}

// resident single-warp blocks per SM of the image layout a launch with these arguments uses
static int max_blocks_per_sm(const LaunchArgs& A, const ChainLaunchPlan& plan) {
    const bool u16 = A.D_int != nullptr && A.D_int_bytes == 2;
    if (u16) return A.pix_f32 ? plan.blocks_per_sm_u16_f32 : plan.blocks_per_sm_u16;
    return A.D_int != nullptr ? plan.blocks_per_sm_u32 : plan.blocks_per_sm_f64;
}

long long chain_kernel_resident_warps(const LaunchArgs& A, const ChainLaunchPlan& plan, int sms, int n_fields) {
    const long long blocks = ((long long)n_fields + kChainGroup - 1) / kChainGroup;
    return std::min<long long>(blocks, (long long)max_blocks_per_sm(A, plan) * sms);
}

int chain_kernel_launch(const FieldParams& P, const LaunchArgs& A_in, const ChainLaunchPlan& plan, int sms, cudaStream_t stream) {
    LaunchArgs A = A_in;
    const int n_range = (A.field_end > 0 ? A.field_end : A.n_fields) - A.field_begin;
    const long long blocks = ((long long)n_range + kChainGroup - 1) / kChainGroup;
    const bool u16 = A.D_int != nullptr && A.D_int_bytes == 2;
    // 4 lanes per chain: 240 of 255 registers -> 8 resident single-warp blocks per SM (2 per scheduler: the register file is
    // partitioned per scheduler, a third warp would need <= 168 registers and measured slower); residency comes from the
    // occupancy query in chain_kernel_configure.  Register-capped 8-lane builds were measured earlier and are slower
    // (128 registers / 16 warps 1057 M star-steps/s, 112 / 18 warps 892 against 1104 at 168 / 12).
    const int max_k = max_blocks_per_sm(A, plan);
    const int full = (int)std::min<long long>(blocks, (long long)max_k * sms);
    int grid = balanced_grid(max_k, blocks, sms);
    if (!(A.mode == MODE_RUN && A.sched_done != nullptr && A.chunk_count > 0)) A.n_chunks = 1;
    if (A.mode == MODE_RUN && A.sched_done != nullptr && A.chunk_count > 0) {
        // one launch of a run that the host has cut along the iteration axis: the chunking is fixed by the caller
        grid = full;
    } else if (A.mode == MODE_RUN && A.sched_done != nullptr) {
        // with the chunked scheduler a partly filled last round costs little, so run at full residency
        if (pick_chunks(blocks, full, A.niter + 1) > 1) grid = full;
        A.n_chunks = pick_chunks(blocks, grid, A.niter + 1);
    }
    if (u16 && A.pix_f32) {
        launch_mode<unsigned short, float>(grid, plan.smem_u16_f32, stream, P, A);
    } else if (u16) {
        launch_mode<unsigned short>(grid, plan.smem_u16, stream, P, A);
    } else if (A.D_int != nullptr) {
        launch_mode<unsigned int>(grid, plan.smem_u32, stream, P, A);
    } else {
        launch_mode<double>(grid, plan.smem_f64, stream, P, A);
    }
    return (int)cudaGetLastError();
}

int math_test_launch(cudaStream_t stream, int which, const double* x, double* y, int n, const double* log_table) {
    math_test_kernel<<<std::max(1, std::min(1024, (n + 255) / 256)), 256, 0, stream>>>(
        which, x, y, n, reinterpret_cast<const double2*>(log_table));
    return (int)cudaGetLastError();
}

int to_counts_launch(cudaStream_t stream, const double* src, unsigned int* dst32, unsigned short* dst16, size_t n,
                     int* flags) {
    const int blocks = (int)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, 4096));
    to_counts_kernel<<<blocks, 256, 0, stream>>>(src, dst32, dst16, n, flags);
    return (int)cudaGetLastError();
}

}  // namespace srhmc
