// Kernels of the device-resident planning inputs: map_T2tau with glibc's log (libm_log.h) and the initial guesses that
// neo_optimize assembles on the host (guesses.straight_line_guess / retry_guesses, optimize_host's x0 staging). They
// live in a translation unit of their own so that nothing neoopt.cu compiles changes: no shared __noinline__ code, no
// new constant-bank data next to k_optimize's.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/neoopt.h"
#include "libm_log.h"

namespace {

// map_T2tau (EP:468-475) as T2tau_one in neoopt.cu computes it on the host: the same operations, uncontracted
__device__ __forceinline__ int T2tau_dev(double T_min, double T_max, double T, double *tau)
{
    const double den = __dsub_rn(T, T_min);
    if (den == 0.0) return NEO_ST_DOMAIN;
    const double a = __dsub_rn(__ddiv_rn(__dsub_rn(T_max, T_min), den), 1.0);
    if (!(a > 0.0) || isinf(a)) return NEO_ST_DOMAIN;
    *tau = -neo::log_glibc(a);
    return 0;
}

__global__ void k_T2tau(int n, double T_min, double T_max, const double *__restrict__ ts, double *__restrict__ tau,
                        int32_t *__restrict__ status)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)n; i += (size_t)gridDim.x * blockDim.x) {
        double t = 0.0;
        const int st = T2tau_dev(T_min, T_max, ts[i], &t);
        tau[i] = st ? 0.0 : t;
        if (status) status[i] = st;
    }
}

struct InitTs { double v[NEO_MAX_PIECES]; };

// One thread per problem. line: guesses._line(head pos, tail pos, M - 1), numpy.linspace's operations one by one
__global__ void k_prepare(int B, int M, double T_min, double T_max, const double *__restrict__ head,
                          const double *__restrict__ tail, const double *__restrict__ q0, const double *__restrict__ ts0,
                          const InitTs init_ts, int count, const double *__restrict__ noise, double *__restrict__ x0,
                          int32_t *__restrict__ x0_status, double *__restrict__ retry_q)
{
    const int K = M - 1, nq = 2 * K, n = nq + M;
    for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < (size_t)B; b += (size_t)gridDim.x * blockDim.x) {
        double s0[2], step[2], delta[2];
        for (int d = 0; d < 2; d++) {
            const double start = head[b * 6 + d], target = tail[b * 6 + d];
            const double hop = __ddiv_rn(__dsub_rn(target, start), (double)(K + 1));
            s0[d] = __dadd_rn(start, hop);
            delta[d] = __dsub_rn(target, s0[d]);
            step[d] = __ddiv_rn(delta[d], (double)K);
        }
        const bool degenerate = step[0] == 0.0 || step[1] == 0.0;          // numpy's branch when any(step == 0)
        auto line = [&](int i, int d) {
            return degenerate ? __dadd_rn(__dmul_rn(__ddiv_rn((double)i, (double)K), delta[d]), s0[d])
                              : __dadd_rn(__dmul_rn((double)i, step[d]), s0[d]);
        };
        double *x = x0 + b * n;
        for (int d = 0; d < 2; d++)
            for (int i = 0; i < K; i++) x[d * K + i] = q0 ? q0[b * nq + d * K + i] : line(i, d);
        int s = 0;
        for (int k = 0; k < M; k++) {
            double t = 0.0;
            const int s1 = T2tau_dev(T_min, T_max, ts0 ? ts0[b * M + k] : init_ts.v[k], &t);
            x[nq + k] = s1 ? 0.0 : t;
            if (s1) s = s1;
        }
        x0_status[b] = s;
        // retry_q (B, count, 2, M-1) = line + noise, noise (B, count, M-1, 2) (guesses.retry_guesses)
        for (int c = 0; c < count; c++) {
            const double *z = noise + (b * count + c) * (size_t)nq;
            double *r = retry_q + (b * count + c) * (size_t)nq;
            for (int d = 0; d < 2; d++)
                for (int i = 0; i < K; i++) r[d * K + i] = __dadd_rn(line(i, d), z[2 * i + d]);
        }
    }
}

int grid_for(size_t items, int threads)
{
    const size_t g = (items + threads - 1) / threads;
    return (int)(g < 65536 ? g : 65536);
}

}  // namespace

cudaError_t launch_T2tau(int n, double T_min, double T_max, const double *ts, double *tau, int32_t *status,
                         cudaStream_t st)
{
    k_T2tau<<<grid_for(n, 256), 256, 0, st>>>(n, T_min, T_max, ts, tau, status);
    return cudaGetLastError();
}

cudaError_t launch_prepare(int B, int M, double T_min, double T_max, const double *head, const double *tail,
                           const double *q0, const double *ts0, const double *init_ts, int count, const double *noise,
                           double *x0, int32_t *x0_status, double *retry_q, cudaStream_t st)
{
    InitTs it = {};
    if (init_ts)
        for (int k = 0; k < M; k++) it.v[k] = init_ts[k];
    k_prepare<<<grid_for(B, 128), 128, 0, st>>>(B, M, T_min, T_max, head, tail, q0, ts0, it, count, noise, x0, x0_status,
                                                 retry_q);
    return cudaGetLastError();
}
