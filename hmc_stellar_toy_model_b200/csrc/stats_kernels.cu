// On-device chain statistics (SURVEY.md 8f "next" row 4): split-chain Gelman-Rubin R and effective sample size over
// thousands of chains, so that a batch (BASELINE configs[1], [3]) can return summaries instead of its full chains.
//
// Reference: utils.convergence_stats / utils.variogram, utils.py:86-188 (broken under Python 3 upstream: `n = L_chain/2`
// at utils.py:111 is an integer division in the reference's Python 2).  Its quirks are behaviour and are kept:
//   * W is the mean of the within-chain standard DEVIATIONS (np.std, utils.py:120), not variances;
//   * the autocorrelation sum stops at the first odd t with rho_{t+1} + rho_{t+2} < 0 and sums lags 1..t.
//
// One CTA per (group of chains, variable).  Chain layout X[chain][row][d] (the layout of q_chain).  All reductions are
// fixed-order (block_sum), so the numbers are reproducible run to run.
#include <algorithm>
#include <cstdlib>

#include "kernels_api.h"

namespace srhmc {

namespace {

struct StatsGeom {
    long long rows;   // iterations stored per chain
    int d;            // variables per row
    int cpg;          // chains per group
    int thin, warm;
    int n;            // samples per split chain
};

// sample k of split chain j (j = 2 * chain + half) of group g, variable v
__device__ __forceinline__ const double* sample_ptr(const double* X, const StatsGeom& G, int g, int v, int j) {
    const long long chain = (long long)g * G.cpg + (j >> 1);
    const long long first = (long long)G.warm + (long long)G.thin * ((j & 1) ? G.n : 0);
    return X + (chain * G.rows + first) * G.d + v;
}

// Sum of the autocorrelations that enters n_eff (utils.py:137-165) from the variogram at lag t, `vario(t)`: rho_t = 1 - V_t / (2 var);
// nothing when rho_1 < 0.05, otherwise the sum of rho_1 .. rho_t up to the first odd t with rho_{t+1} + rho_{t+2} < 0 (or
// t = n - 2), clamped at 0.  The reference's rho_t list index i holds lag i + 1.  Every caller thread follows the same control
// flow.  Shared by conv_stats_final_kernel and conv_stats_var_kernel.
template <class Vario>
__device__ __forceinline__ double ess_sum_rho(int n, double var, const Vario& vario) {
    const double rho1 = 1.0 - vario(1) / (2.0 * var);
    const double rho2 = 1.0 - vario(2) / (2.0 * var);
    double sum_rho = 0.0;
    if (!(rho1 < 5e-2)) {
        // loop invariant: prefix = sum(rho_t[:t]), cur = rho_t[t]
        double prefix = rho1, cur = rho2;
        int t = 1;
        while (t < n - 2) {
            const double next = 1.0 - vario(t + 2) / (2.0 * var);  // appended as rho_t[t + 1]
            if ((t & 1) && (cur + next) < 0.0) break;
            prefix += cur;
            cur = next;
            ++t;
        }
        sum_rho = prefix < 0.0 ? 0.0 : prefix;
    }
    return sum_rho;
}

__global__ void __launch_bounds__(256) conv_stats_kernel(const double* __restrict__ X, const StatsGeom G, double* __restrict__ means,
                                                         double* __restrict__ R_out, double* __restrict__ neff_out) {
    __shared__ double red[2 * 32];
    const int g = blockIdx.x / G.d, v = blockIdx.x % G.d;
    const int m = 2 * G.cpg, n = G.n;
    const long long stride = (long long)G.thin * G.d;
    double* mu = means + (size_t)blockIdx.x * m;
    // within-chain mean and sample standard deviation of every split chain (np.mean / np.std(ddof=1), utils.py:118-126)
    double part[2] = {0.0, 0.0};
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        const double* x = sample_ptr(X, G, g, v, j);
        double s = 0.0;
        for (int k = 0; k < n; ++k) s += x[k * stride];
        const double mean = s / (double)n;
        double ss = 0.0;
        for (int k = 0; k < n; ++k) {
            const double dlt = x[k * stride] - mean;
            ss += dlt * dlt;
        }
        mu[j] = mean;
        part[0] += sqrt(ss / (double)(n - 1));
        part[1] += mean;
    }
    block_sum<2>(part, red);
    const double W = part[0] / (double)m, mean_all = part[1] / (double)m;
    __syncthreads();
    double b[1] = {0.0};
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        const double dlt = mu[j] - mean_all;
        b[0] += dlt * dlt;
    }
    block_sum<1>(b, red);
    const double B = b[0] * (double)n / (double)(m - 1);
    const double var = W * (double)(n - 1) / (double)n + B / (double)n;
    const double R = sqrt(var / W);

    // variogram at lag t (utils.py:170-188), valid in every thread
    auto variogram = [&](int t) {
        double a[1] = {0.0};
        for (int j = threadIdx.x; j < m; j += blockDim.x) {
            const double* x = sample_ptr(X, G, g, v, j);
            double s = 0.0;
            for (int k = 0; k + t < n; ++k) {
                const double dlt = x[(k + t) * stride] - x[k * stride];
                s += dlt * dlt;
            }
            a[0] += s;
        }
        block_sum<1>(a, red);
        return a[0] / ((double)m * (double)(n - t));
    };
    // effective sample size (utils.py:137-165); every thread follows the same control flow
    const double rho1 = 1.0 - variogram(1) / (2.0 * var);
    const double rho2 = 1.0 - variogram(2) / (2.0 * var);
    double sum_rho = 0.0;
    if (!(rho1 < 5e-2)) {
        // rho_t list of the reference: index i holds lag i + 1.  Loop invariant: prefix = sum(rho_t[:t]), cur = rho_t[t].
        double prefix = rho1, cur = rho2;
        int t = 1;
        while (t < n - 2) {
            const double next = 1.0 - variogram(t + 2) / (2.0 * var);  // appended as rho_t[t + 1]
            if ((t & 1) && (cur + next) < 0.0) break;
            prefix += cur;
            cur = next;
            ++t;
        }
        sum_rho = prefix < 0.0 ? 0.0 : prefix;
    }
    if (threadIdx.x == 0) {
        R_out[blockIdx.x] = R;
        neff_out[blockIdx.x] = (double)m * (double)n / (1.0 + 2.0 * sum_rho);
    }
}


// ---- chain-parallel variant (the default when a split chain fits shared memory) -----------------------------------------
// Stage 1: one warp per chain, 8 chains per CTA.  The warp stages the thinned samples of both halves of its chain in shared
// memory, computes their means / standard deviations, and every lane takes lags t = lane + 1, lane + 33, ... of the
// variogram sums S_t = sum_k (x_{k+t} - x_k)^2 (no shuffles, fixed order).  The CTA adds its warps' sums in warp order and
// writes one partial per lag.  Stage 2: one CTA per (group, variable) adds the partials in CTA order and applies the
// reference's formulas and cut-off rule.  Same numbers as conv_stats_kernel up to summation order (1e-15).
constexpr int kStatsChainsPerBlock = 8;
constexpr int kStatsMaxN = 768;   // samples per split chain held in shared memory (2 * 768 doubles per warp)

__global__ void __launch_bounds__(32 * kStatsChainsPerBlock)
conv_stats_chain_kernel(const double* __restrict__ X, const StatsGeom G, int blocks_per_group, double* __restrict__ mu,
                        double* __restrict__ sd, double* __restrict__ lagpart) {
    extern __shared__ double stats_smem[];
    const int n = G.n, nl = n - 1;                       // lags 1 .. n-1
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* xs = stats_smem + (size_t)warp * 2 * n;       // [half][k]
    double* wsum = stats_smem + (size_t)kStatsChainsPerBlock * 2 * n + (size_t)warp * nl;   // this warp's lag sums
    const int g = blockIdx.x / blocks_per_group, bg = blockIdx.x % blocks_per_group;
    const int c = bg * kStatsChainsPerBlock + warp;       // chain within the group
    const bool live = c < G.cpg;
    const long long stride = (long long)G.thin * G.d;
    const int m = 2 * G.cpg;
    for (int v = 0; v < G.d; ++v) {
        for (int t = lane; t < nl; t += 32) wsum[t] = 0.0;
        if (live) {
            for (int h = 0; h < 2; ++h) {
                const double* x = sample_ptr(X, G, g, v, 2 * c + h);
                double s = 0.0;
                for (int k = lane; k < n; k += 32) {
                    const double val = x[k * stride];
                    xs[h * n + k] = val;
                    s += val;
                }
                s = warp_sum(s);
                const double mean = s / (double)n;
                __syncwarp();
                double ss = 0.0;
                for (int k = lane; k < n; k += 32) {
                    const double dlt = xs[h * n + k] - mean;
                    ss += dlt * dlt;
                }
                ss = warp_sum(ss);
                if (lane == 0) {
                    const size_t o = ((size_t)g * G.d + v) * m + 2 * c + h;
                    mu[o] = mean;
                    sd[o] = sqrt(ss / (double)(n - 1));
                }
                for (int t = lane + 1; t <= nl; t += 32) {
                    double acc = 0.0;
                    const double* a = xs + h * n;
                    for (int k = 0; k + t < n; ++k) {
                        const double dlt = a[k + t] - a[k];
                        acc += dlt * dlt;
                    }
                    wsum[t - 1] += acc;
                }
            }
        }
        __syncthreads();
        // CTA partial per lag, warps added in order
        for (int t = threadIdx.x; t < nl; t += blockDim.x) {
            double acc = 0.0;
            for (int w = 0; w < kStatsChainsPerBlock; ++w) acc += stats_smem[(size_t)kStatsChainsPerBlock * 2 * n + (size_t)w * nl + t];
            lagpart[(((size_t)g * blocks_per_group + bg) * G.d + v) * nl + t] = acc;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
conv_stats_final_kernel(const StatsGeom G, int blocks_per_group, const double* __restrict__ mu, const double* __restrict__ sd,
                        const double* __restrict__ lagpart, double* __restrict__ vario, double* __restrict__ R_out,
                        double* __restrict__ neff_out) {
    __shared__ double red[2 * 32];
    const int g = blockIdx.x / G.d, v = blockIdx.x % G.d;
    const int m = 2 * G.cpg, n = G.n, nl = n - 1;
    const double* mu_gv = mu + (size_t)blockIdx.x * m;
    const double* sd_gv = sd + (size_t)blockIdx.x * m;
    double part[2] = {0.0, 0.0};
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        part[0] += sd_gv[j];
        part[1] += mu_gv[j];
    }
    block_sum<2>(part, red);
    const double W = part[0] / (double)m, mean_all = part[1] / (double)m;
    __syncthreads();
    double b[1] = {0.0};
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        const double dlt = mu_gv[j] - mean_all;
        b[0] += dlt * dlt;
    }
    block_sum<1>(b, red);
    const double B = b[0] * (double)n / (double)(m - 1);
    const double var = W * (double)(n - 1) / (double)n + B / (double)n;
    const double R = sqrt(var / W);
    // variogram of every lag: CTA partials added in order
    double* V = vario + (size_t)blockIdx.x * nl;
    for (int t = threadIdx.x; t < nl; t += blockDim.x) {
        double acc = 0.0;
        for (int p = 0; p < blocks_per_group; ++p) acc += lagpart[(((size_t)g * blocks_per_group + p) * G.d + v) * nl + t];
        V[t] = acc / ((double)m * (double)(n - (t + 1)));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        // effective sample size (utils.py:137-165)
        const double sum_rho = ess_sum_rho(n, var, [&](int lag) { return V[lag - 1]; });
        R_out[blockIdx.x] = R;
        neff_out[blockIdx.x] = (double)m * (double)n / (1.0 + 2.0 * sum_rho);
    }
}


// ---- variable-parallel variant: few chains, many variables (the chains of the large-field engine) -------------------------
// One thread per variable; the K chains are separate row-major buffers [rows][d] (X[c] in the parameter struct), so a warp
// reads 32 consecutive variables of one row per load.  Every thread loops over the split chains and samples in a fixed
// order (reproducible run to run) and runs its own lag loop to its own cut-off.  Same formulas as conv_stats_kernel.
struct ChainSet {
    const double* x[kMaxStatsChains];
};

__global__ void __launch_bounds__(128) conv_stats_var_kernel(const ChainSet X, const StatsGeom G, double* __restrict__ R_out,
                                                             double* __restrict__ neff_out) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= G.d) return;
    const int m = 2 * G.cpg, n = G.n;
    const long long stride = (long long)G.thin * G.d;
    auto sample0 = [&](int j) {   // first sample of split chain j (j = 2 * chain + half)
        const long long first = (long long)G.warm + (long long)G.thin * ((j & 1) ? n : 0);
        return X.x[j >> 1] + first * G.d + v;
    };
    double mu[2 * kMaxStatsChains];
    double sd_sum = 0.0, mu_sum = 0.0;
    for (int j = 0; j < m; ++j) {
        const double* x = sample0(j);
        double s = 0.0;
        for (int k = 0; k < n; ++k) s += x[k * stride];
        const double mean = s / (double)n;
        double ss = 0.0;
        for (int k = 0; k < n; ++k) {
            const double dlt = x[k * stride] - mean;
            ss += dlt * dlt;
        }
        mu[j] = mean;
        sd_sum += sqrt(ss / (double)(n - 1));
        mu_sum += mean;
    }
    const double W = sd_sum / (double)m, mean_all = mu_sum / (double)m;
    double b = 0.0;
    for (int j = 0; j < m; ++j) {
        const double dlt = mu[j] - mean_all;
        b += dlt * dlt;
    }
    const double B = b * (double)n / (double)(m - 1);
    const double var = W * (double)(n - 1) / (double)n + B / (double)n;
    const double sum_rho = ess_sum_rho(n, var, [&](int t) {
        double a = 0.0;
        for (int j = 0; j < m; ++j) {
            const double* x = sample0(j);
            for (int k = 0; k + t < n; ++k) {
                const double dlt = x[(k + t) * stride] - x[k * stride];
                a += dlt * dlt;
            }
        }
        return a / ((double)m * (double)(n - t));
    });
    R_out[v] = sqrt(var / W);
    neff_out[v] = (double)m * (double)n / (1.0 + 2.0 * sum_rho);
}

}  // namespace

static StatsGeom stats_geom(long long rows, int d, int cpg, int thin, int warm) {
    StatsGeom G;
    G.rows = rows; G.d = d; G.cpg = cpg; G.thin = thin; G.warm = warm;
    const long long Lw = rows - warm;
    const long long Lc = Lw > 0 ? (Lw + thin - 1) / thin : 0;  // len(chain[warm:][::thin])
    G.n = (int)(Lc / 2);                                       // utils.py:111 (Python-2 integer division)
    return G;
}

// scratch the statistics need (doubles): split-chain means and standard deviations, per-CTA lag partials, variograms
size_t conv_stats_scratch_doubles(long long rows, int d, int n_groups, int cpg, int thin, int warm) {
    const StatsGeom G = stats_geom(rows, d, cpg, thin, warm);
    const size_t nout = (size_t)n_groups * d, m = 2 * (size_t)cpg, nl = (size_t)std::max(1, G.n - 1);
    const size_t bpg = ((size_t)cpg + kStatsChainsPerBlock - 1) / kStatsChainsPerBlock;
    return 2 * nout * m + (size_t)n_groups * bpg * d * nl + nout * nl;
}

// X [n_groups * cpg chains][rows][d] on the device; scratch: conv_stats_scratch_doubles() doubles; R, n_eff [n_groups, d].
int conv_stats_launch(cudaStream_t stream, const double* X, long long rows, int d, int n_groups, int cpg, int thin, int warm,
                      double* scratch, double* R, double* neff) {
    const StatsGeom G = stats_geom(rows, d, cpg, thin, warm);
    const size_t nout = (size_t)n_groups * d, m = 2 * (size_t)cpg;
    const char* old = std::getenv("SRHMC_STATS_SINGLE_CTA");
    if (G.n > kStatsMaxN || G.n < 3 || (old && old[0] == '1')) {
        conv_stats_kernel<<<n_groups * d, 256, 0, stream>>>(X, G, scratch, R, neff);   // one CTA per (group, variable)
        return (int)cudaGetLastError();
    }
    const int nl = G.n - 1;
    const int bpg = (cpg + kStatsChainsPerBlock - 1) / kStatsChainsPerBlock;
    double* mu = scratch;
    double* sd = mu + nout * m;
    double* lagpart = sd + nout * m;
    double* vario = lagpart + (size_t)n_groups * bpg * d * nl;
    const size_t smem = ((size_t)kStatsChainsPerBlock * 2 * G.n + (size_t)kStatsChainsPerBlock * nl) * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(conv_stats_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    conv_stats_chain_kernel<<<n_groups * bpg, 32 * kStatsChainsPerBlock, smem, stream>>>(X, G, bpg, mu, sd, lagpart);
    conv_stats_final_kernel<<<n_groups * d, 256, 0, stream>>>(G, bpg, mu, sd, lagpart, vario, R, neff);
    return (int)cudaGetLastError();
}

// K (2..kMaxStatsChains) chains, each its own device buffer [rows][d]; R, n_eff [d] on the device.
int conv_stats_var_launch(cudaStream_t stream, const double* const* chains, int k, long long rows, int d, int thin, int warm,
                          double* R, double* neff) {
    if (k < 2 || k > kMaxStatsChains) return (int)cudaErrorInvalidValue;
    ChainSet X{};
    for (int c = 0; c < k; ++c) X.x[c] = chains[c];
    const StatsGeom G = stats_geom(rows, d, k, thin, warm);
    conv_stats_var_kernel<<<(d + 127) / 128, 128, 0, stream>>>(X, G, R, neff);
    return (int)cudaGetLastError();
}

}  // namespace srhmc
