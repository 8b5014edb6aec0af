// Host-callable launchers of the device kernels; each family is compiled in its own translation unit so the
// in-tree build can run them in parallel.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "common.cuh"

namespace srhmc {

// Dynamic shared memory and resident blocks per SM of the one-star kernel for each image layout.  A block is one warp
// holding kChainGroup chains.
struct ChainLaunchPlan {
    size_t smem_f64 = 0, smem_u32 = 0, smem_u16 = 0, smem_u16_f32 = 0;
    int blocks_per_sm_f64 = 0, blocks_per_sm_u32 = 0, blocks_per_sm_u16 = 0, blocks_per_sm_u16_f32 = 0;
};

// CTA-per-field kernel (field_kernel.cuh); precision 64|32, (mr, mc) in {(2,4), (2,2), (1,2)}
size_t field_layout_total(int precision, const FieldParams& P, bool d_in_smem);
int field_kernel_configure(int precision, int mr, int mc, size_t smem);
int field_kernel_launch(int precision, int mr, int mc, int grid, int threads, size_t smem, cudaStream_t stream,
                        const FieldParams& P, const LaunchArgs& A, double* scratch, int d_in_smem);
// lightsource_gym family (ls_kernel.cuh), FP64
int ls_kernel_configure(int mr, int mc, size_t smem);
int ls_kernel_launch(int mr, int mc, int grid, int threads, size_t smem, cudaStream_t stream, const FieldParams& P,
                     const LsArgs& A, double* scratch, int dsm);
int philox_dump_launch(cudaStream_t stream, unsigned long long seed, int n_fields, int L, int Nmax, int fid_base,
                       int fid_stride, double* normals, double* lnu);
// the draw records of field_kernel MODE_RUN_RJ (rj_draws.cuh): draws [n_fields, L, kRjDraws]
int rj_dump_launch(cudaStream_t stream, unsigned long long seed, int n_fields, int L, int fid_base, int fid_stride, double beta_a,
                   double beta_b, double* draws);
int metric_launch(cudaStream_t stream, const FieldParams& P, size_t n_stars, const double* q, double g_ff2, double* H,
                  double* Hgrad);
int kinetic_diag_launch(cudaStream_t stream, size_t n, const double* p, const double* H, double* T);
int kinetic_launch(cudaStream_t stream, const FieldParams& P, int n_fields, const double* q, const double* p,
                   const int* nstars, double g_ff2, double* T, double* dtaudq, double* dtaudp);
int convert_image_launch(cudaStream_t stream, const double* src, float* dst, size_t n);

// warp-resident one-star kernel (chain_kernel.cuh), FP64
int chain_kernel_configure(const FieldParams& P, ChainLaunchPlan& plan);
// columns a chain's lanes cover in a launch now: 24 (window) or 32 (full width)
int chain_kernel_window_cols(const FieldParams& P);
// shared-memory layout of one block for R image rows of elem-byte pixels (f32: FP32 pixel arithmetic)
ChainLayout chain_kernel_layout(int R, size_t elem, bool f32);
// Largest exponent from which a lane's column table starts, over star positions in the support y in [-1, C+1], for a
// window of `window_cols` columns.  chain_eval drops a lane's whole column table at 690 (and exp_neg overflows above ~709),
// so the host sends a PSF to the kernel only when this stays at or below kChainExpMax, 50 under that cut-off (a star a
// little outside the support, within a trajectory, then still gets its whole table); other PSFs take the CTA kernel.
double chain_column_exponent(const FieldParams& P, int window_cols);
constexpr double kChainExpMax = 640.0;
bool chain_kernel_psf_ok(const FieldParams& P);
int chain_kernel_launch(const FieldParams& P, const LaunchArgs& A, const ChainLaunchPlan& plan, int sms, cudaStream_t stream);
// iteration chunks of the MODE_RUN work scheduler for `groups` warp-sized work items on `warps` resident warps
int pick_chunks(long long groups, long long warps, int L);
// warps a MODE_RUN launch of n_fields chains keeps resident (the denominator of its work scheduler's rounds)
long long chain_kernel_resident_warps(const LaunchArgs& A, const ChainLaunchPlan& plan, int sms, int n_fields);

void fill_log_table(double* host_table /* (rc_k, lc_k) pairs, at most 128 of them */);
int math_test_launch(cudaStream_t stream, int which, const double* x, double* y, int n, const double* log_table);
int to_counts_launch(cudaStream_t stream, const double* src, unsigned int* dst32, unsigned short* dst16, size_t n,
                     int* flags);

// device-side mock data (mock_kernels.cu): model image of every field, Poisson realisation with counter-based Philox
int model_launch(cudaStream_t stream, const FieldParams& P, int n_fields, const double* q, const int* nstars,
                 const double* background, double* out);
int poisson_launch(cudaStream_t stream, const double* lam, double* D, size_t n, unsigned long long seed,
                   unsigned long long index_base);

// on-device chain statistics (stats_kernels.cu)
size_t conv_stats_scratch_doubles(long long rows, int d, int n_groups, int cpg, int thin, int warm);
int conv_stats_launch(cudaStream_t stream, const double* X, long long rows, int d, int n_groups, int cpg, int thin, int warm,
                      double* scratch, double* R, double* neff);
// variable-parallel form for a few chains held in separate buffers (the large-field engine): one thread per variable
constexpr int kMaxStatsChains = 16;
int conv_stats_var_launch(cudaStream_t stream, const double* const* chains, int k, long long rows, int d, int thin, int warm,
                          double* R, double* neff);
// argument checks shared by every statistics entry point (message through srhmc_last_error)
int check_stats_args(int64_t n_chains, int64_t rows, int32_t d, int32_t n_groups, int32_t thin, int32_t warm);

// gradient-descent leg of lightsource_gym.find_peaks (peaks_kernels.cu): one warp per seed, image 0 of the context
int peaks_launch(cudaStream_t stream, const FieldParams& P, const double* D, int n, int nstep, double dt_f_coeff,
                 double dt_xy_coeff, double f_lim, double* q, unsigned char* alive, int* steps);

// FMA-chain roofline microbenchmark
int fma_peak_run(int precision, int sms, double* tflops, float* ms);

}  // namespace srhmc
