// CTA-per-field kernel instantiations, double pixels.
#include "field_kernel.cuh"
#include "kernels_api.h"

namespace srhmc {

typedef void (*FieldKernelFn64)(const FieldParams, const LaunchArgs, double*, int);

// compact-table contexts (P.v3) run their chains through the kernel compiled for MODE_RUN and that path alone
static FieldKernelFn64 pick64(int mr, int mc, bool run_v3 = false) {
    if (run_v3) return field_kernel<double, 2, 4, MODE_RUN, 1>;
    if (mr == 2 && mc == 4) return field_kernel<double, 2, 4>;
    if (mr == 2 && mc == 2) return field_kernel<double, 2, 2>;
    return field_kernel<double, 1, 2>;
}

// reversible-jump chains (MODE_RUN_RJ): one instantiation per tile shape and the compact-table one
static FieldKernelFn64 pick64_rj(int mr, int mc, bool v3) {
    if (v3) return field_kernel<double, 2, 4, MODE_RUN_RJ, 1>;
    if (mr == 2 && mc == 4) return field_kernel<double, 2, 4, MODE_RUN_RJ, 0>;
    if (mr == 2 && mc == 2) return field_kernel<double, 2, 2, MODE_RUN_RJ, 0>;
    return field_kernel<double, 1, 2, MODE_RUN_RJ, 0>;
}

size_t field_layout_total_f64(const FieldParams& P, bool dsm) { return make_layout<double>(P, dsm).total; }

int field_kernel_configure_f64(int mr, int mc, size_t smem) {
    cudaError_t e = cudaFuncSetAttribute(pick64(mr, mc), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pick64(mr, mc, true), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    for (int v3 = 0; v3 < 2 && e == cudaSuccess; ++v3)
        e = cudaFuncSetAttribute(pick64_rj(mr, mc, v3 != 0), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    return (int)e;
}

int field_kernel_launch_f64(int mr, int mc, int grid, int threads, size_t smem, cudaStream_t stream, const FieldParams& P,
                            const LaunchArgs& A, double* scratch, int dsm) {
    const FieldKernelFn64 fn = A.mode == MODE_RUN_RJ ? pick64_rj(mr, mc, P.v3 != 0) : pick64(mr, mc, P.v3 && A.mode == MODE_RUN);
    fn<<<grid, threads, smem, stream>>>(P, A, scratch, dsm);
    return (int)cudaGetLastError();
}

}  // namespace srhmc
