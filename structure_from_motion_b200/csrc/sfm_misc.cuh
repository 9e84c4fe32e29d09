// Small utility kernels: FP64 peak probe (the tail's compaction lives in sfm_tail.cuh).
#pragma once
#include "sfm_device.cuh"

namespace sfm {

// 16 independent DFMA chains per thread: the FP64 pipe's sustained rate.
__global__ void __launch_bounds__(256) k_fp64_peak(double* __restrict__ out, int iters, double m) {
    double a[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = 1.0 + 1e-3 * (threadIdx.x + k);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 16; ++k) a[k] = fma(a[k], m, 1e-9);
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += a[k];
    if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace sfm
