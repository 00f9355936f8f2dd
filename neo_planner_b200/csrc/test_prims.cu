// Test hook kernel: the optimizer's vector primitives (nrm2_x87, blas_ddot, loop_dot of lbfgsb_tile.cuh) as nvcc compiles
// them for the device, one vector per thread. Kept out of neoopt.cu: ptxas compiles a __noinline__ device function
// together with all its callers in a translation unit, and a second caller there changed k_optimize's code.
#include <cuda_runtime.h>

// the header's __noinline__ functions get host symbols with external linkage; a namespace of its own keeps this
// translation unit's copies from colliding with neoopt.cu's at link time
#define neo neo_test_prims
#include "lbfgsb_tile.cuh"

using namespace neo_test_prims;

// out[3 i .. 3 i + 3) = nrm2_x87(a_i), blas_ddot(a_i, b_i), loop_dot(a_i, b_i)
__global__ void k_blas_prims(int count, int n, const double *a, const double *b, double *out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const double *ai = a + (size_t)i * n, *bi = b + (size_t)i * n;
    out[3 * (size_t)i] = nrm2_x87(n, ai);
    out[3 * (size_t)i + 1] = blas_ddot(n, ai, bi);
    out[3 * (size_t)i + 2] = loop_dot(n, ai, bi);
}

void launch_blas_prims(int count, int n, const double *a, const double *b, double *out, cudaStream_t stream)
{
    k_blas_prims<<<(count + 127) / 128, 128, 0, stream>>>(count, n, a, b, out);
}
