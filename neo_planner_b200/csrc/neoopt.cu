// neoopt.cu -- libneoopt.so: kernels + the C ABI declared in include/neoopt.h.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC (see build.py).
// There is no CPU fallback: without a usable CUDA device neo_create fails with NEO_ERR_NO_DEVICE.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/neoopt.h"
#include "astar_warp.cuh"
#include "lbfgsb_tile.cuh"
#include "map_kernels.cuh"
#include "minco_tile.cuh"

using namespace neo;

// ---------------------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------------------
constexpr int WARPS_PER_CTA = 4;
#ifndef NEO_GROUPED_MIN_PROBLEMS
#define NEO_GROUPED_MIN_PROBLEMS 2048 // batch size from which one-problem-per-warp kernels run as one CTA per SM with grouped starts
#endif
#ifndef NEO_TILE_MIN_PROBLEMS
#define NEO_TILE_MIN_PROBLEMS 12288 // batch size from which short trajectories (M <= 4) run several problems per warp
                                     // (measured on B200: 16 k problems 11.1 vs 11.2 ms, 65 k 38.8 vs 43.2 ms)
#endif
#ifndef NEO_HOST_THREADS
#define NEO_HOST_THREADS 8            // neo_optimize: host threads that assemble inputs / scatter results of a large batch
#endif

struct OptArgs {
    int B, M, max_attempts;
    const double *x0;            // (B,n) tau form
    const int32_t *x0_status;    // (B) or null: NEO_ST_DOMAIN where map_T2tau failed on the host
    const double *head, *tail;   // (B,3,2)
    const int32_t *map_ids;      // (B) or null
    const double *retry_q;       // (B, A-1, 2(M-1)) or null
    const double *retry_tau;     // (M) or null
    int retry_status;            // NEO_ST_DOMAIN if retry_ts is outside (T_min, T_max)
    const MapView *maps;
    unsigned int *counter;       // work queue head
    // per-task records (task = attempt * B + problem), written by the tile that ran the attempt
    double *t_x;                 // (A*B, n)
    double *t_costs;             // (A*B, 4)
    int32_t *t_info;             // (A*B, 4): status, nit, nfev, completed (minimize() returned)
    long long *t_work;           // (A*B, 4): samples, velocity-violating, colliding, nanoseconds on the SM
    unsigned int *p_state;       // (B): bits 0..7 attempts finished, bits 8..15 attempts accepted
    double *x, *ts, *coeffs, *costs;
    int32_t *status, *ok, *attempt, *nit, *runs, *nfev;
    long long *work;
    // optional evaluation trace (neo_optimize_trace; all null otherwise): per task the first trace_cap evaluations
    int trace_cap;
    int bus_q;                               // SM-wide variant: warps per departing group at the evaluation site
    double *tr_x, *tr_f, *tr_g, *tr_costs;   // (A*B, cap, n), (A*B, cap), (A*B, cap, n), (A*B, cap, 4)
    int32_t *tr_status, *tr_len;             // (A*B, cap), (A*B)
};

// A problem is resolved once its lowest accepted attempt has all earlier attempts finished, or all attempts finished.
__device__ __forceinline__ bool resolved(unsigned st, int A)
{
    const unsigned done = st & 0xffu, okm = (st >> 8) & 0xffu;
    if (okm) { const unsigned lower = (1u << (__ffs(okm) - 1)) - 1u; return (done & lower) == lower; }
    return done == (1u << A) - 1u;
}

// Persistent TILES (TL lanes; 32 / TL per warp) pull TASKS = (attempt, problem) from a global queue in attempt-major
// order and run one plan_once (EP:205-237) per task entirely on chip. warm_start_plan (EP:186-203) semantics are kept
// exactly -- the returned attempt is the lowest-index accepted one and counters are summed over attempts 0..that one --
// but a retry whose predecessor is still running elsewhere is started SPECULATIVELY on an otherwise idle tile (its
// inputs, straight line + host-drawn noise, do not depend on the predecessor). A speculative attempt is skipped or
// cancelled as soon as an earlier attempt of its problem is accepted. The tile whose completion resolves a problem
// assembles its outputs (final coefficients included).
// The loop below is the WARP's loop: every round each running tile evaluates f, g at its trial point (one shared
// evaluation site, so the tiles of a warp walk through the evaluator together) and then advances its own optimizer
// (lbfgsb_tile.cuh: opt_advance); a tile whose task ends takes the next one in the same round.
// TL = 32: one problem per warp -- lowest latency per evaluation (few problems per SM, or M >= 5 where n > 16).
// TL = 8 / 16: 4 / 2 problems per warp for short trajectories (n <= TL, 2M <= TL) -- with n = 7 decision variables and
//   ~20 samples per piece a whole warp is mostly idle lanes; tiles cut the issue slots per evaluation ~2x.
// MC: the number of pieces as a compile-time constant (loops over pieces/nodes unroll, lane maps fold).
// MINB x WPC: CTAs per SM the register allocation is sized for x warps per CTA: 3 x 4 (plain) or 1 x 12 (grouped starts,
// see launch_optimize). The optimizer's line-search record, costs and counters live in shared memory, so 168 registers
// per thread hold the rest without spills.
// Grouped starts: this loop is ~55 KB of code walked once per round by every warp, against a 32 KB instruction cache per
// SM and a GPC-level instruction path that saturates (ncu: gcc__cache_requests_type_instruction 95 % of peak, 53 % of
// the stall samples `no_instruction`). Warps that walk the code TOGETHER share every fetched line (devtools/
// icache_share.cu: 12 warps in step run a 96 KB body at 3.6 IPC per SM, spread out at 2.5), but a barrier over all 12
// warps waits for the slowest search direction every round (40 % barrier stalls). Groups of nine are the measured optimum.
template <int MC, int TL, int MINB, int WPC = WARPS_PER_CTA>
__global__ void __launch_bounds__(WPC * 32, MINB) k_optimize(const DevParams P, const OptArgs a)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Tile<TL> T(lane);
    constexpr int TPW = 32 / TL;
    const int M = MC, n = 3 * M - 2, nq = 2 * (M - 1), N = 6 * M, A = a.max_attempts;
    const TileMem m = carve(smem + (size_t)(warp * TPW + lane / TL) * tile_mem_doubles(M, TL), M, TL);
    const unsigned total = (unsigned)A * (unsigned)a.B;
    const bool mine = T.tl < n;
    OptState o;
    opt_begin(o, 0.0);
    bool running = false, retired = false;
    unsigned tid = 0, lower_ok = 0;
    int at = 0;
    size_t b = 0;
    int map_id = 0;              // the MapView itself (14 registers) is re-read from device memory at every evaluation
    unsigned long long t_start = 0;
    __shared__ unsigned s_arrivals;
    constexpr unsigned BUS_DRAIN = 0x80000000u;
    bool drained = false;
    if constexpr (WPC > WARPS_PER_CTA) {
        if (threadIdx.x == 0) s_arrivals = 0;
        __syncthreads();
    }
    for (;;) {
        if constexpr (WPC > WARPS_PER_CTA) {
            // departures in groups: a warp arriving at the evaluation site takes a ticket and waits on a hardware
            // barrier until the bus_q warps of its group have gathered, so that the group walks the evaluator's code
            // together and shares its instruction fetches. The first warp that runs out of tasks ends the scheme: later
            // tickets carry the drain flag (no waiting any more) and it completes the one partially filled group.
            __syncwarp();
            if (!drained) {
                unsigned k = 0;
                if (lane == 0) k = atomicAdd(&s_arrivals, 1u);
                k = __shfl_sync(FULL, k, 0);
                if (k & BUS_DRAIN) drained = true;
                else asm volatile("bar.sync %0, %1;" ::"r"(1 + (int)((k / (unsigned)a.bus_q) & 7u)), "r"(a.bus_q * 32) : "memory");
            }
        }
        if (__all_sync(FULL, retired)) {
            if constexpr (WPC > WARPS_PER_CTA) {
                if (!drained) {
                    unsigned old = 0;
                    if (lane == 0) old = atomicOr(&s_arrivals, BUS_DRAIN);
                    old = __shfl_sync(FULL, old, 0);
                    if (!(old & BUS_DRAIN)) {          // tickets issued so far: old; the last group holds old % bus_q warps
                        const unsigned waiting = old % (unsigned)a.bus_q, g = old / (unsigned)a.bus_q;
                        if (waiting)
                            for (unsigned i = waiting; i < (unsigned)a.bus_q; i++)
                                asm volatile("bar.arrive %0, %1;" ::"r"(1 + (int)(g & 7u)), "r"(a.bus_q * 32) : "memory");
                    }
                }
            }
            break;
        }
        bool ended = false, report = false;      // this tile's task ended in this round / it has a record to write
        if (!running && !retired) {
            unsigned t0 = 0;
            if (T.tl == 0) t0 = atomicAdd(a.counter, 1u);
            tid = T.shfl(t0, 0);
            if (tid >= total) retired = true;
            else {
                at = (int)(tid / (unsigned)a.B);
                b = tid - (unsigned)at * (unsigned)a.B;
                lower_ok = ((1u << at) - 1u) << 8;
                unsigned seen = 0;
                if (T.tl == 0) seen = *reinterpret_cast<volatile unsigned *>(a.p_state + b);
                seen = T.shfl(seen, 0);
                ended = true;
                if (!(seen & lower_ok)) {         // else: an earlier attempt was already accepted, nothing to run
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_start));
                    begin_problem(T, m, M, a.head + b * 6, a.tail + b * 6);
                    map_id = a.map_ids ? a.map_ids[b] : 0;
                    double x0l = 0.0;
                    int st0 = 0;
                    if (at == 0) {
                        if (mine) x0l = a.x0[b * n + T.tl];
                        st0 = a.x0_status ? a.x0_status[b] : 0;
                    } else {
                        if (T.tl < nq) x0l = a.retry_q[(b * (A - 1) + (at - 1)) * nq + T.tl];
                        else if (mine) x0l = a.retry_tau[T.tl - nq];
                        st0 = a.retry_status;
                    }
                    opt_begin(o, x0l);
                    if (T.tl < 7) m.oc[T.tl] = 0.0;
                    T.sync();
                    report = true;
                    if (st0) { o.status = st0; o.x = 0.0; }       // map_T2tau raised (EP:209)
                    else { running = true; ended = false; }
                }
            }
        }
        if (running) {
            if (!opt_same_point(T, o, n)) {
                // ---- the evaluation site: f, g at x --------------------------------------------------------------
                EvalOut ev;
                eval_fg<MC, TL>(T, P, a.maps[map_id], m, M, o.x, ev);
                if (T.tl == 0) { m.oc[4] += (double)ev.ns; m.oc[5] += (double)ev.nv; m.oc[6] += (double)ev.nc; }   // exact below 2^53
                if (a.tr_x && o.nfev < a.trace_cap) {
                    const size_t k = (size_t)tid * a.trace_cap + o.nfev;
                    if (mine) { a.tr_x[k * n + T.tl] = o.x; a.tr_g[k * n + T.tl] = ev.status ? 0.0 : ev.g; }
                    if (T.tl < 4) a.tr_costs[k * 4 + T.tl] = ev.costs[T.tl];
                    if (T.tl == 0) { a.tr_f[k] = ev.f; a.tr_status[k] = ev.status; a.tr_len[tid] = o.nfev + 1; }
                }
                if (ev.status) { o.status = ev.status; running = false; ended = true; report = true; }
                else {
                    o.f = ev.f; o.g = mine ? ev.g : 0.0; o.nfev++; o.xlast = o.x;
                    if (T.tl < 4) m.oc[T.tl] = ev.costs[T.tl];
                }
            }
            if (running) {
                opt_advance<TL, 3 * MC - 2>(T, m, n, o, a.p_state + b, lower_ok);
                if (o.status != ST_RUNNING) { running = false; ended = true; report = true; }
            }
        }
        if (!ended) continue;

        // ---- the task ended: record it, mark it in the problem's state word -------------------------------------
        unsigned bits = 1u << at;
        if (report && o.status != ST_CANCELLED) {
            const bool completed = o.status < NEO_ST_OVERFLOW;             // minimize() returned (EP:213-233)
            T.sync();
            const bool accepted = completed && !(m.oc[3] * P.w3 > P.collision_cost_tol);      // EP:235-237
            if (mine) a.t_x[(size_t)tid * n + T.tl] = o.x;
            if (T.tl < 4) a.t_costs[(size_t)tid * 4 + T.tl] = m.oc[T.tl];
            if (T.tl == 0) {
                a.t_info[(size_t)tid * 4 + 0] = o.status; a.t_info[(size_t)tid * 4 + 1] = o.nit;
                a.t_info[(size_t)tid * 4 + 2] = o.nfev; a.t_info[(size_t)tid * 4 + 3] = completed ? 1 : 0;
                unsigned long long t_end;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
                a.t_work[(size_t)tid * 4 + 0] = (long long)m.oc[4]; a.t_work[(size_t)tid * 4 + 1] = (long long)m.oc[5];
                a.t_work[(size_t)tid * 4 + 2] = (long long)m.oc[6]; a.t_work[(size_t)tid * 4 + 3] = (long long)(t_end - t_start);
            }
            if (accepted) bits |= 1u << (8 + at);
            __threadfence();
        }
        T.sync();
        unsigned old = 0;
        if (T.tl == 0) old = atomicOr(a.p_state + b, bits);
        old = T.shfl(old, 0);
        const unsigned now = old | bits;
        if (!resolved(now, A) || resolved(old, A)) continue;

        // ---- this tile resolved problem b: assemble warm_start_plan's outputs ---------------------------------
        __threadfence();
        const unsigned okm = (now >> 8) & 0xffu;
        const int last = okm ? __ffs(okm) - 1 : A - 1;      // returned attempt (EP:196-203)
        int nit = 0, runs = 0, nfev = 0, src = -1, status = 0;
        long long ns = 0, nv = 0, nc = 0, nanos = 0;
        for (int k = 0; k <= last; k++) {
            const size_t t = (size_t)k * a.B + b;
            const int st = __ldcg(a.t_info + t * 4 + 0);
            status = st;
            nfev += __ldcg(a.t_info + t * 4 + 2);
            ns += __ldcg(a.t_work + t * 4 + 0); nv += __ldcg(a.t_work + t * 4 + 1); nc += __ldcg(a.t_work + t * 4 + 2);
            nanos += __ldcg(a.t_work + t * 4 + 3);
            if (__ldcg(a.t_info + t * 4 + 3)) { runs++; nit += __ldcg(a.t_info + t * 4 + 1); src = k; }
        }
        if (src >= 0) {      // final (int_wpts, ts) -> ts, coefficients (EP:226-229, TU:182)
            const size_t t = (size_t)src * a.B + b;
            const double xf = mine ? __ldcg(a.t_x + t * n + T.tl) : 0.0;
            begin_problem(T, m, M, a.head + b * 6, a.tail + b * 6);
            double e_unused;
            times_from_tau(T, P, m, M, xf, e_unused);
            load_nodes(T, m, M, xf);
            solve_nodes(T, m, M);
            hermite_coeffs(T, m, M);
            if (mine) a.x[b * n + T.tl] = xf;
            if (T.tl < M) a.ts[b * M + T.tl] = m.ts[T.tl];
            for (int i = T.tl; i < 2 * N; i += TL) a.coeffs[b * 2 * N + i] = m.c[i];
            if (T.tl < 4) a.costs[b * 4 + T.tl] = __ldcg(a.t_costs + t * 4 + T.tl);
        } else {
            if (mine) a.x[b * n + T.tl] = 0.0;
            if (T.tl < M) a.ts[b * M + T.tl] = 0.0;
            for (int i = T.tl; i < 2 * N; i += TL) a.coeffs[b * 2 * N + i] = 0.0;
            if (T.tl < 4) a.costs[b * 4 + T.tl] = 0.0;
        }
        if (T.tl == 0) {
            a.status[b] = status; a.ok[b] = okm ? 1 : 0; a.attempt[b] = last; a.nit[b] = nit; a.runs[b] = runs;
            a.nfev[b] = nfev;
            if (a.work) { a.work[b * 4] = ns; a.work[b * 4 + 1] = nv; a.work[b * 4 + 2] = nc; a.work[b * 4 + 3] = nanos; }
        }
        T.sync();
    }
}

struct EvalArgs {
    int B, M;
    const double *x, *head, *tail;
    const int32_t *map_ids;
    const MapView *maps;
    double *costs, *grad, *coeffs, *ts;
    int32_t *status;
};

// get_cost + get_grad (EP:539-585) fused, one tile per problem
template <int MC, int TL>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 3) k_eval(const DevParams P, const EvalArgs a)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Tile<TL> T(lane);
    constexpr int TPW = 32 / TL, TPC = WARPS_PER_CTA * TPW;
    const int M = MC, n = 3 * M - 2, N = 6 * M;
    const int tile = warp * TPW + lane / TL;
    const TileMem m = carve(smem + (size_t)tile * eval_mem_doubles(M, TL), M, TL, true);
    for (size_t b = (size_t)blockIdx.x * TPC + tile; b < (size_t)a.B; b += (size_t)gridDim.x * TPC) {
        begin_problem(T, m, M, a.head + b * 6, a.tail + b * 6);
        const MapView map = a.maps[a.map_ids ? a.map_ids[b] : 0];
        const double xl = T.tl < n ? a.x[b * n + T.tl] : 0.0;
        EvalOut ev;
        eval_fg<MC, TL, true>(T, P, map, m, M, xl, ev);
        if (T.tl < n) a.grad[b * n + T.tl] = ev.status ? 0.0 : ev.g;
        if (T.tl < 4) a.costs[b * 4 + T.tl] = ev.costs[T.tl];
        if (T.tl == 0) a.status[b] = ev.status;
        if (a.coeffs) for (int i = T.tl; i < 2 * N; i += TL) a.coeffs[b * 2 * N + i] = ev.status == NEO_ST_OVERFLOW ? 0.0 : m.c[i];
        if (a.ts && T.tl < M) a.ts[b * M + T.tl] = m.ts[T.tl];
        T.sync();
    }
}

// get_coeffs (EP:261-336 / TU:8-83): q (B,2,M-1), ts (B,M) -> coeffs (B,6M,2)
__global__ void __launch_bounds__(WARPS_PER_CTA * 32) k_coeffs(int B, int M, const double *q, const double *ts,
                                                               const double *head, const double *tail, double *coeffs)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Tile<32> T(lane);
    const int nq = 2 * (M - 1), N = 6 * M;
    const TileMem m = carve(smem + (size_t)warp * tile_mem_doubles(M), M);
    for (size_t b = (size_t)blockIdx.x * WARPS_PER_CTA + warp; b < (size_t)B; b += (size_t)gridDim.x * WARPS_PER_CTA) {
        begin_problem(T, m, M, head + b * 6, tail + b * 6);
        if (lane < M) {
            const double Tt = ts[b * M + lane];
            m.ts[lane] = Tt;
            const double a = 1.0 / Tt, a2 = a * a;
            double *it = m.iT + 5 * lane;
            it[0] = a; it[1] = a2; it[2] = a2 * a; it[3] = a2 * a2; it[4] = a2 * a2 * a;
        }
        __syncwarp();
        const double xl = lane < nq ? q[b * nq + lane] : 0.0;
        load_nodes(T, m, M, xl);
        solve_nodes(T, m, M);
        hermite_coeffs(T, m, M);
        for (int i = lane; i < 2 * N; i += 32) coeffs[b * 2 * N + i] = m.c[i];
        __syncwarp();
    }
}

// get_full_state_cmd (TU:181-195): thread per (trajectory b, sample k)
__global__ void k_sample(int B, int M, const double *__restrict__ coeffs, const double *__restrict__ ts, double hz,
                         int max_samples, double *__restrict__ states, int32_t *__restrict__ count)
{
    for (int b = blockIdx.y; b < B; b += gridDim.y) {
    const double *T = ts + (size_t)b * M;
    double total = 0.0;
    for (int i = 0; i < M; i++) total += T[i];                    // Python sum(self.ts)
    const double step = 1.0 / hz;
    const int cnt = (int)ceil(total / step);                      // len(np.arange(0, total, 1/hz))
    if (blockIdx.x == 0 && threadIdx.x == 0) count[b] = cnt;
    if (!states) continue;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < cnt && k < max_samples; k += gridDim.x * blockDim.x) {
        const double t = (double)k * step;
        int piece = 0;
        double upto = T[0];                                       // sum(ts[:piece+1]) (TU:97-98)
        while (upto < t && piece < M - 1) { piece++; upto += T[piece]; }
        double before = 0.0;
        for (int i = 0; i < piece; i++) before += T[i];
        const double s = t - before;
        const double s2 = s * s, s3 = s2 * s, s4 = s3 * s, s5 = s4 * s;
        const double *c = coeffs + ((size_t)b * 6 * M + 6 * piece) * 2;
        double *o = states + ((size_t)b * max_samples + k) * 6;
#pragma unroll
        for (int d = 0; d < 2; d++) {
            const double c0 = c[d], c1 = c[2 + d], c2 = c[4 + d], c3 = c[6 + d], c4 = c[8 + d], c5 = c[10 + d];
            o[d] = c0 + c1 * s + c2 * s2 + c3 * s3 + c4 * s4 + c5 * s5;
            o[2 + d] = c1 + c2 * (2.0 * s) + c3 * (3.0 * s2) + c4 * (4.0 * s3) + c5 * (5.0 * s4);
            o[4 + d] = c2 * 2.0 + c3 * (6.0 * s) + c4 * (12.0 * s2) + c5 * (20.0 * s3);
        }
    }
    }
}

// FP64 FMA throughput probe: 8 independent accumulators per thread
__global__ void k_fp64_peak(double *out, int iters)
{
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1.0, a2 = a0 + 2.0, a3 = a0 + 3.0, a4 = a0 + 4.0, a5 = a0 + 5.0,
           a6 = a0 + 6.0, a7 = a0 + 7.0;
    const double m = 1.0000001, c = 1e-7;
    for (int i = 0; i < iters; i++) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

// device-side check of exp_dd against the host build of the same header (tests)
__global__ void k_exp_dd(int n, const double *x, double *y)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { bool o; y[i] = exp_dd(x[i], &o); }
}

// test_prims.cu: the optimizer's vector primitives on the device, in a translation unit of their own so that a second
// caller does not change how k_optimize is compiled
void launch_blas_prims(int count, int n, const double *a, const double *b, double *out, cudaStream_t stream);
// device_api.cu: map_T2tau with glibc's log and the initial guesses on the device (neo_T2tau_dev, neo_prepare_dev)
cudaError_t launch_T2tau(int n, double T_min, double T_max, const double *ts, double *tau, int32_t *status, cudaStream_t st);
cudaError_t launch_prepare(int B, int M, double T_min, double T_max, const double *head, const double *tail,
                           const double *q0, const double *ts0, const double *init_ts, int count, const double *noise,
                           double *x0, int32_t *x0_status, double *retry_q, cudaStream_t st);

// ---------------------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------------------
struct MapSlot {
    Cell *cells = nullptr;
    int8_t *occ = nullptr;       // occupancy grid of the last occupancy / point-cloud build
    size_t occ_cap = 0;
    bool has_occ = false;        // occ holds the grid of the map now in the slot (an ESDF upload has none)
    unsigned char *blocked = nullptr;   // has_collision over the enlarged A* grid (astar_warp.cuh), rebuilt with the map
    size_t blocked_cap = 0;
    int H = 0, W = 0;
    double res = 0, ox = 0, oy = 0;
};

// Persistent host worker threads of one handle (neo_optimize's input assembly and result scatter on large batches):
// created at the first large call, parked on a condition variable in between; spawning threads per call cost ~1 ms of
// the 5 ms the host side of a 65,536-problem call used to take.
class HostPool {
public:
    ~HostPool()
    {
        { std::lock_guard<std::mutex> g(mu_); stop_ = true; }
        wake_.notify_all();
        for (auto &t : workers_) t.join();
    }
    // runs fn(begin, end) over [0, count) split into at most NEO_HOST_THREADS parts; the caller works too
    void run(size_t count, const std::function<void(size_t, size_t)> &fn)
    {
        const size_t min_per = 4096;
        size_t nt = count / min_per;
        if (nt > NEO_HOST_THREADS) nt = NEO_HOST_THREADS;
        if (nt <= 1) { fn((size_t)0, count); return; }
        while (workers_.size() + 1 < nt) workers_.emplace_back([this] { loop(); });
        const size_t per = (count + nt - 1) / nt;
        {
            std::lock_guard<std::mutex> g(mu_);
            fn_ = &fn; count_ = count; per_ = per; parts_ = nt; next_ = 1; pending_ = nt - 1; generation_++;
        }
        wake_.notify_all();
        fn((size_t)0, per < count ? per : count);
        work();                                            // help with whatever has not been taken yet
        std::unique_lock<std::mutex> g(mu_);
        done_.wait(g, [this] { return pending_ == 0; });
        fn_ = nullptr;
    }

private:
    void work()
    {
        for (;;) {
            size_t part;
            const std::function<void(size_t, size_t)> *fn;
            size_t count, per;
            {
                std::lock_guard<std::mutex> g(mu_);
                if (!fn_ || next_ >= parts_) return;
                part = next_++; fn = fn_; count = count_; per = per_;
            }
            const size_t b0 = part * per, b1 = b0 + per < count ? b0 + per : count;
            if (b0 < b1) (*fn)(b0, b1);
            {
                std::lock_guard<std::mutex> g(mu_);
                if (--pending_ == 0) done_.notify_all();
            }
        }
    }
    void loop()
    {
        unsigned long long seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> g(mu_);
                wake_.wait(g, [&] { return stop_ || generation_ != seen; });
                if (stop_) return;
                seen = generation_;
            }
            work();
        }
    }
    std::vector<std::thread> workers_;
    std::mutex mu_;
    std::condition_variable wake_, done_;
    const std::function<void(size_t, size_t)> *fn_ = nullptr;
    size_t count_ = 0, per_ = 0, parts_ = 0, next_ = 0, pending_ = 0;
    unsigned long long generation_ = 0;
    bool stop_ = false;
};

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct neo_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    neo_config cfg;
    std::vector<MapSlot> slots;
    std::vector<MapView> views;      // host copies of the published views (sources of the async uploads)
    MapView *d_maps = nullptr;
    unsigned int *d_counter = nullptr;
    // Grow-only buffers. Every host-pointer entry point synchronises before it returns and runs under mu, so all of
    // them lay out their device arrays in `stage`. The two scratch areas a device-pointer launch still reads after its
    // call has returned have buffers of their own.
    DevBuf stage;
    DevBuf opt_scratch;              // launch_optimize: per-task records and per-problem state words
    DevBuf astar_overflow;           // astar_launch: overflow list of the first pass
    DevBuf pinned;                   // pinned host staging buffer (neo_optimize)
    DevBuf astar;                    // per-warp search scratch of neo_astar (node records all-zero between launches)
    size_t astar_cap = 0;            // cells per warp the scratch is laid out for
    int astar_warps = 0;             // worker warps the scratch is laid out for
    size_t astar_laid_icap = 0;      // inserted nodes per search the first-pass lists are laid out for
    int astar_icap = 0;              // development switch (env NEO_ASTAR_ICAP at neo_create): first-pass list length, 0 = default
    std::string err;
    std::mutex mu;
    float last_ms = 0.f;
    long long launches = 0;
    HostPool pool;                   // host worker threads of neo_optimize
    bool host_timing = false;        // development switch (env NEO_HOST_TIMING): neo_optimize prints its host-side phases
    int grouped = -1, group_warps = 0;   // development switches (env NEO_GROUPED = 0 | 1, NEO_GROUP_WARPS at neo_create; -1 / 0: by batch size)
    int tile = 0;                    // development switch (env NEO_TILE = 8 | 16 | 32 at neo_create; 0: by batch size):
                                     // lanes per problem for M <= 4, see launch_optimize / include/neoopt.h
    int sm_count = 0, cc_major = 0, cc_minor = 0;
    char name[128] = {0};
};

static std::string g_create_err;

#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) {                                                                          \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                  \
            return NEO_ERR_CUDA;                                                                          \
        }                                                                                                 \
    } while (0)

static int fail(neo_handle *h, const std::string &msg)
{
    h->err = msg;
    return NEO_ERR_INVALID;
}

static DevParams dev_params(const neo_config &c)
{
    DevParams P;
    P.v_max2 = c.v_max * c.v_max;      // self.v_max**2 (EP:410)
    P.T_min = c.T_min; P.T_max = c.T_max; P.safe_dis = c.safe_dis; P.dt = c.delta_t;
    P.w0 = c.weights[0]; P.w1 = c.weights[1]; P.w2 = c.weights[2]; P.w3 = c.weights[3];
    P.collision_cost_tol = c.collision_cost_tol;
    return P;
}

// makes b hold at least `bytes`: device memory, or mapped pinned host memory for h->pinned (the optimizer writes its
// results straight into it). A call must not grow a buffer it has already enqueued copies into.
static int grow(neo_handle *h, DevBuf &b, size_t bytes, char **out)
{
    const bool pinned = &b == &h->pinned;
    if (b.cap < bytes) {
        if (b.p) CK(pinned ? cudaFreeHost(b.p) : cudaFree(b.p));
        b.p = nullptr; b.cap = 0;
        const size_t cap = bytes + bytes / 4 + 256;
        CK(pinned ? cudaHostAlloc(&b.p, cap, cudaHostAllocMapped) : cudaMalloc(&b.p, cap));
        b.cap = cap;
    }
    *out = (char *)b.p;
    return NEO_OK;
}

// byte offsets of arrays laid out one after another in one buffer, each 256-byte aligned; end is the total size
struct Layout {
    size_t end = 0;
    size_t add(size_t bytes)
    {
        const size_t at = (end + 255) & ~(size_t)255;
        end = at + bytes;
        return at;
    }
};

static int cfg_check(const neo_config *c)
{
    return c && c->delta_t > 0.0 && c->T_max > c->T_min;
}

extern "C" int neo_create(const neo_config *cfg, int device, int max_maps, neo_handle **out)
{
    if (!out || !cfg_check(cfg) || max_maps < 1) { g_create_err = "neo_create: invalid argument"; return NEO_ERR_INVALID; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) {
        g_create_err = std::string("neo_create: no usable CUDA device (") + cudaGetErrorString(e) +
                       "); libneoopt has no CPU fallback";
        return NEO_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major < 10) {
        g_create_err = "neo_create: device is not sm_100 (Blackwell); this library ships sm_100a code only";
        return NEO_ERR_NO_DEVICE;
    }
    neo_handle *h = new neo_handle();
    h->device = device; h->cfg = *cfg; h->slots.resize(max_maps); h->views.resize(max_maps);
    h->host_timing = getenv("NEO_HOST_TIMING") != nullptr;
    if (const char *e = getenv("NEO_ASTAR_ICAP")) h->astar_icap = atoi(e);
    if (const char *e = getenv("NEO_GROUPED")) h->grouped = atoi(e) ? 1 : 0;
    if (const char *e = getenv("NEO_GROUP_WARPS")) h->group_warps = atoi(e);
    if (const char *e = getenv("NEO_TILE")) { const int t = atoi(e); h->tile = (t == 8 || t == 16 || t == 32) ? t : 0; }
    h->sm_count = prop.multiProcessorCount; h->cc_major = prop.major; h->cc_minor = prop.minor;
    snprintf(h->name, sizeof(h->name), "%s", prop.name);
    bool good = cudaSetDevice(device) == cudaSuccess &&
                cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) == cudaSuccess &&
                cudaEventCreate(&h->ev0) == cudaSuccess && cudaEventCreate(&h->ev1) == cudaSuccess &&
                cudaMalloc(&h->d_maps, sizeof(MapView) * max_maps) == cudaSuccess &&
                cudaMemset(h->d_maps, 0, sizeof(MapView) * max_maps) == cudaSuccess &&
                cudaMalloc(&h->d_counter, sizeof(unsigned int) * 64) == cudaSuccess;
    if (!good) {
        g_create_err = std::string("neo_create: ") + cudaGetErrorString(cudaGetLastError());
        delete h;
        return NEO_ERR_CUDA;
    }
    *out = h;
    return NEO_OK;
}

extern "C" int neo_destroy(neo_handle *h)
{
    if (!h) return NEO_ERR_INVALID;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    for (auto &s : h->slots) { if (s.cells) cudaFree(s.cells); if (s.occ) cudaFree(s.occ); if (s.blocked) cudaFree(s.blocked); }
    for (DevBuf *b : {&h->stage, &h->opt_scratch, &h->astar_overflow, &h->astar}) if (b->p) cudaFree(b->p);
    if (h->pinned.p) cudaFreeHost(h->pinned.p);
    cudaFree(h->d_maps); cudaFree(h->d_counter);
    cudaEventDestroy(h->ev0); cudaEventDestroy(h->ev1);
    cudaStreamDestroy(h->stream);
    delete h;
    return NEO_OK;
}

extern "C" int neo_set_config(neo_handle *h, const neo_config *cfg)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (!cfg_check(cfg)) return fail(h, "neo_set_config: invalid config");
    h->cfg = *cfg;
    return NEO_OK;
}

extern "C" const char *neo_last_error(neo_handle *h) { return h ? h->err.c_str() : g_create_err.c_str(); }

extern "C" int neo_device_info(neo_handle *h, int *sm_count, int *cc_major, int *cc_minor, char *name, int name_len)
{
    if (!h) return NEO_ERR_INVALID;
    if (sm_count) *sm_count = h->sm_count;
    if (cc_major) *cc_major = h->cc_major;
    if (cc_minor) *cc_minor = h->cc_minor;
    if (name && name_len > 0) snprintf(name, name_len, "%s", h->name);
    return NEO_OK;
}

// ---------------------------------------------------------------------------------------------------------
// maps
// ---------------------------------------------------------------------------------------------------------
static int slot_prepare(neo_handle *h, int slot, int H, int W, double res, double ox, double oy)
{
    if (slot < 0 || slot >= (int)h->slots.size()) return fail(h, "map slot out of range");
    if (H < 2 || W < 2 || !(res > 0.0)) return fail(h, "map must be at least 2x2 with positive resolution");
    MapSlot &s = h->slots[slot];
    if (s.cells && (size_t)s.H * s.W != (size_t)H * W) { CK(cudaFree(s.cells)); s.cells = nullptr; }
    if (!s.cells) CK(cudaMalloc(&s.cells, sizeof(Cell) * (size_t)H * W));
    s.H = H; s.W = W; s.res = res; s.ox = ox; s.oy = oy;
    s.has_occ = false;                  // until an occupancy build of this shape completes (build_from_occ)
    return NEO_OK;
}

static MapView map_view(const MapSlot &s)
{
    MapView v;
    v.cells = s.cells; v.H = s.H; v.W = s.W; v.res = s.res; v.ox = s.ox; v.oy = s.oy; v.inv_res = 1.0 / s.res;
    v.blocked = s.blocked;
    return v;
}

static int slot_publish(neo_handle *h, int slot, bool sync = true)
{
    MapSlot &s = h->slots[slot];
    // node-blocked grid of the geometric initializer (AP:130-141), one byte per node of the enlarged grid
    const size_t nodes = astar_grid_cells(s.H, s.W, s.res);
    if (s.blocked_cap < nodes) {
        if (s.blocked) { CK(cudaStreamSynchronize(h->stream)); CK(cudaFree(s.blocked)); s.blocked = nullptr; s.blocked_cap = 0; }
        CK(cudaMalloc(&s.blocked, nodes));
        s.blocked_cap = nodes;
    }
    const MapView v = map_view(s);
    const int pad = (int)(10.0 / s.res);
    dim3 grid((s.W + pad + 127) / 128, s.H + pad);
    k_astar_blocked<<<grid, 128, 0, h->stream>>>(v, s.blocked);
    h->launches++;
    CK(cudaGetLastError());
    h->views[slot] = v;                 // pageable source of an async copy: must outlive the call
    CK(cudaMemcpyAsync(h->d_maps + slot, &h->views[slot], sizeof(v), cudaMemcpyHostToDevice, h->stream));
    if (sync) CK(cudaStreamSynchronize(h->stream));
    return NEO_OK;
}

extern "C" int neo_set_map_esdf(neo_handle *h, int slot, int H, int W, double res, double ox, double oy,
                                const double *esdf, const double *gx, const double *gy)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (!esdf || !gx || !gy) return fail(h, "neo_set_map_esdf: null array");
    CK(cudaSetDevice(h->device));
    int rc = slot_prepare(h, slot, H, W, res, ox, oy);
    if (rc) return rc;
    const size_t n = (size_t)H * W;
    Layout L;
    const size_t o_e = L.add(sizeof(double) * n), o_gx = L.add(sizeof(double) * n), o_gy = L.add(sizeof(double) * n);
    char *d;
    if ((rc = grow(h, h->stage, L.end, &d))) return rc;
    CK(cudaMemcpyAsync(d + o_e, esdf, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d + o_gx, gx, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d + o_gy, gy, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    dim3 grid((W + 127) / 128, H);
    k_pack_cells<<<grid, 128, 0, h->stream>>>((double *)(d + o_e), (double *)(d + o_gx), (double *)(d + o_gy), H, W,
                                              h->slots[slot].cells, nullptr, nullptr);
    h->launches++;
    CK(cudaGetLastError());
    return slot_publish(h, slot);
}

// device arrays of one occupancy -> EDT -> cells build: the binarised grid, the EDT's row pass, its flag, the distances
struct OccArrays { size_t occ, g, any, e; };
static OccArrays occ_arrays(Layout &L, size_t n)
{
    return {L.add(n), L.add(sizeof(int) * n), L.add(sizeof(int)), L.add(sizeof(double) * n)};
}

// occupancy (device, int8, in the staging buffer at base) -> exact EDT -> cells
static int build_from_occ(neo_handle *h, int slot, int H, int W, double res, char *base, const OccArrays &o, bool sync = true)
{
    const int8_t *d_occ = (const int8_t *)(base + o.occ);
    int *d_g = (int *)(base + o.g), *d_any = (int *)(base + o.any);
    double *d_e = (double *)(base + o.e);
    MapSlot &s = h->slots[slot];
    const size_t n = (size_t)H * W;
    if (s.occ && s.occ_cap < n) { CK(cudaFree(s.occ)); s.occ = nullptr; }
    if (!s.occ) { CK(cudaMalloc(&s.occ, n)); s.occ_cap = n; }
    CK(cudaMemcpyAsync(s.occ, d_occ, n, cudaMemcpyDeviceToDevice, h->stream));
    s.has_occ = true;
    CK(cudaMemsetAsync(d_any, 0, sizeof(int), h->stream));
    k_edt_rows<<<(H + 7) / 8, 256, 0, h->stream>>>(d_occ, H, W, d_g, d_any);                 // one warp per row
    dim3 grid((W + 127) / 128, H);
    k_edt_cols<<<grid, 128, 0, h->stream>>>(d_g, H, W, d_any, res, d_e);
    k_pack_cells<<<grid, 128, 0, h->stream>>>(d_e, nullptr, nullptr, H, W, s.cells, nullptr, nullptr);
    h->launches += 3;
    CK(cudaGetLastError());
    return slot_publish(h, slot, sync);
}

extern "C" int neo_set_map_occupancy(neo_handle *h, int slot, int H, int W, double res, double ox, double oy,
                                     const int8_t *occ)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (!occ) return fail(h, "neo_set_map_occupancy: null array");
    if ((long long)H * H + (long long)W * W >= (long long)EDT_INF) return fail(h, "map too large for the int32 EDT");
    CK(cudaSetDevice(h->device));
    int rc = slot_prepare(h, slot, H, W, res, ox, oy);
    if (rc) return rc;
    const size_t n = (size_t)H * W;
    Layout L;
    const OccArrays o = occ_arrays(L, n);
    char *d;
    if ((rc = grow(h, h->stage, L.end, &d))) return rc;
    CK(cudaMemcpyAsync(d + o.occ, occ, n, cudaMemcpyHostToDevice, h->stream));
    return build_from_occ(h, slot, H, W, res, d, o);
}

// K maps of one shape in one call (the 256 generated worlds of the data-generation sweep): one H2D copy per group of
// maps, every build enqueued back to back on the handle's stream, ONE synchronisation at the end.
extern "C" int neo_set_maps_occupancy(neo_handle *h, int K, const int32_t *slots, int H, int W, double res, const double *ox,
                                      const double *oy, const int8_t *occ)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (K < 0 || !slots || !ox || !oy || !occ) return fail(h, "neo_set_maps_occupancy: invalid argument");
    if ((long long)H * H + (long long)W * W >= (long long)EDT_INF) return fail(h, "map too large for the int32 EDT");
    for (int k = 0; k < K; k++) {
        if (slots[k] < 0 || slots[k] >= (int)h->slots.size()) return fail(h, "map slot out of range");
        for (int j = 0; j < k; j++) if (slots[j] == slots[k]) return fail(h, "neo_set_maps_occupancy: a slot is named twice");
    }
    if (K == 0) return NEO_OK;
    CK(cudaSetDevice(h->device));
    const size_t n = (size_t)H * W;
    const int group = K < 32 ? K : 32;                        // staging for 32 maps at a time
    Layout L;
    std::vector<OccArrays> o(group);
    for (auto &a : o) a = occ_arrays(L, n);
    char *d;
    int rc = grow(h, h->stage, L.end, &d);
    if (rc) return rc;
    for (int k0 = 0; k0 < K; k0 += group) {
        const int kn = K - k0 < group ? K - k0 : group;
        if (k0) CK(cudaStreamSynchronize(h->stream));          // the staging block is reused by the next group
        for (int k = 0; k < kn; k++) {
            if ((rc = slot_prepare(h, slots[k0 + k], H, W, res, ox[k0 + k], oy[k0 + k]))) return rc;
            CK(cudaMemcpyAsync(d + o[k].occ, occ + n * (size_t)(k0 + k), n, cudaMemcpyHostToDevice, h->stream));
        }
        for (int k = 0; k < kn; k++)
            if ((rc = build_from_occ(h, slots[k0 + k], H, W, res, d, o[k], false))) return rc;
    }
    CK(cudaStreamSynchronize(h->stream));
    return NEO_OK;
}

extern "C" int neo_set_map_points(neo_handle *h, int slot, int n_points, const float *xyz, double z_min, double z_max,
                                  int H, int W, double res, double ox, double oy)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (n_points < 0 || (n_points > 0 && !xyz)) return fail(h, "neo_set_map_points: invalid argument");
    if ((long long)H * H + (long long)W * W >= (long long)EDT_INF) return fail(h, "map too large for the int32 EDT");
    CK(cudaSetDevice(h->device));
    int rc = slot_prepare(h, slot, H, W, res, ox, oy);
    if (rc) return rc;
    const size_t n = (size_t)H * W;
    Layout L;
    const OccArrays o = occ_arrays(L, n);
    const size_t o_xyz = L.add(sizeof(float) * 3 * (size_t)n_points);
    char *d;
    if ((rc = grow(h, h->stage, L.end, &d))) return rc;
    CK(cudaMemsetAsync(d + o.occ, 0, n, h->stream));
    if (n_points > 0) {
        CK(cudaMemcpyAsync(d + o_xyz, xyz, sizeof(float) * 3 * (size_t)n_points, cudaMemcpyHostToDevice, h->stream));
        k_points_to_occ<<<(n_points + 255) / 256, 256, 0, h->stream>>>((const float *)(d + o_xyz), n_points, z_min, z_max,
                                                                       ox, oy, res, H, W, (int8_t *)(d + o.occ));
        h->launches++;
        CK(cudaGetLastError());
    }
    return build_from_occ(h, slot, H, W, res, d, o);
}

// the caller's (H, W) must be the slot's: read-back writes exactly H * W elements into caller-sized arrays
static int check_shape(neo_handle *h, const MapSlot &s, int H, int W, const char *who)
{
    if (H == s.H && W == s.W) return NEO_OK;
    return fail(h, std::string(who) + ": the slot holds a " + std::to_string(s.H) + " x " + std::to_string(s.W) + " map, not " +
                       std::to_string(H) + " x " + std::to_string(W));
}

extern "C" int neo_get_occupancy(neo_handle *h, int slot, int H, int W, int8_t *occ)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (slot < 0 || slot >= (int)h->slots.size() || !h->slots[slot].has_occ || !occ) return fail(h, "neo_get_occupancy: no occupancy in this slot");
    const MapSlot &s = h->slots[slot];
    int rc = check_shape(h, s, H, W, "neo_get_occupancy");
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(occ, s.occ, (size_t)s.H * s.W, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return NEO_OK;
}

extern "C" int neo_get_map(neo_handle *h, int slot, int H, int W, double *esdf, double *gx, double *gy)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (slot < 0 || slot >= (int)h->slots.size() || !h->slots[slot].cells) return fail(h, "neo_get_map: empty slot");
    const MapSlot &s = h->slots[slot];
    int rc = check_shape(h, s, H, W, "neo_get_map");
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    const size_t n = (size_t)s.H * s.W;
    Layout L;
    const size_t o_e = L.add(sizeof(double) * n), o_gx = L.add(sizeof(double) * n), o_gy = L.add(sizeof(double) * n);
    char *d;
    if ((rc = grow(h, h->stage, L.end, &d))) return rc;
    k_unpack_cells<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(s.cells, n, (double *)(d + o_e), (double *)(d + o_gx),
                                                                       (double *)(d + o_gy));
    h->launches++;
    CK(cudaGetLastError());
    if (esdf) CK(cudaMemcpyAsync(esdf, d + o_e, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    if (gx) CK(cudaMemcpyAsync(gx, d + o_gx, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    if (gy) CK(cudaMemcpyAsync(gy, d + o_gy, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return NEO_OK;
}

extern "C" int neo_query_map(neo_handle *h, int slot, int n, const double *xy, int32_t *idx, double *dis, double *grad)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (slot < 0 || slot >= (int)h->slots.size() || !h->slots[slot].cells) return fail(h, "neo_query_map: empty slot");
    if (n < 0 || !xy || !idx || !dis || !grad) return fail(h, "neo_query_map: invalid argument");
    if (n == 0) return NEO_OK;
    CK(cudaSetDevice(h->device));
    Layout L;
    const size_t o_xy = L.add(sizeof(double) * 2 * n), o_idx = L.add(sizeof(int32_t) * 2 * n),
                 o_dis = L.add(sizeof(double) * n), o_grad = L.add(sizeof(double) * 2 * n);
    char *d;
    int rc = grow(h, h->stage, L.end, &d);
    if (rc) return rc;
    CK(cudaMemcpyAsync(d + o_xy, xy, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, h->stream));
    k_query<<<(n + 127) / 128, 128, 0, h->stream>>>(map_view(h->slots[slot]), n, (const double *)(d + o_xy),
                                                    (int32_t *)(d + o_idx), (double *)(d + o_dis), (double *)(d + o_grad));
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(idx, d + o_idx, sizeof(int32_t) * 2 * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(dis, d + o_dis, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(grad, d + o_grad, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return NEO_OK;
}

// ---------------------------------------------------------------------------------------------------------
// launch helpers
// ---------------------------------------------------------------------------------------------------------
static int check_problem(neo_handle *h, int B, int M)
{
    if (B < 0) return fail(h, "B must be >= 0");
    if (M < 2 || M > NEO_MAX_PIECES) return fail(h, "M must be in [2, NEO_MAX_PIECES]");
    if (!h->slots[0].cells) {
        bool any = false;
        for (auto &s : h->slots) any = any || s.cells;
        if (!any) return fail(h, "no map uploaded (neo_set_map_esdf / neo_set_map_occupancy)");
    }
    return NEO_OK;
}

// host-pointer entry points: every map id must name a slot that holds a map (device-pointer entry points document it
// as a precondition: the ids live in device memory)
static int check_map_ids(neo_handle *h, int B, const int32_t *map_ids, const char *who)
{
    if (!map_ids) {
        if (!h->slots[0].cells) return fail(h, std::string(who) + ": map_ids is NULL and slot 0 holds no map");
        return NEO_OK;
    }
    for (int i = 0; i < B; i++)
        if (map_ids[i] < 0 || map_ids[i] >= (int)h->slots.size() || !h->slots[map_ids[i]].cells)
            return fail(h, std::string(who) + ": map id " + std::to_string(map_ids[i]) + " (problem " + std::to_string(i) +
                               ") refers to an empty slot");
    return NEO_OK;
}

static size_t smem_bytes(int M, int TL = 32, int wpc = WARPS_PER_CTA)
{
    return sizeof(double) * (size_t)tile_mem_doubles(M, TL) * wpc * (32 / TL);
}

// sets the kernel's dynamic shared memory and returns in *grid the CTAs for `items` work items at per_cta a CTA, no
// more than are resident on the device at once (the kernels loop over the rest)
template <typename K>
static int launch_grid(neo_handle *h, K kernel, size_t smem, int wpc, size_t items, size_t per_cta, int *grid)
{
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, wpc * 32, smem));
    if (occ < 1) return fail(h, "kernel does not fit on an SM");
    const size_t need = (items + per_cta - 1) / per_cta, resident = (size_t)occ * h->sm_count;
    *grid = (int)(need < resident ? need : resident);
    return NEO_OK;
}

// lanes per problem when short trajectories share a warp: n = 3M - 2 <= 8 for M <= 3, <= 16 for M = 4
constexpr int shared_lanes(int M) { return M <= 3 ? 8 : 16; }

// lanes per problem: M >= 5 needs the warp (n > 16); short trajectories share a warp once the batch is large enough to
// fill the machine with several problems per warp (below that, one problem per warp has the shorter evaluation)
static int tile_lanes(const neo_handle *h, int B, int M)
{
    if (M > 4) return 32;
    if (h->tile) return h->tile == 32 ? 32 : shared_lanes(M);
    return B >= NEO_TILE_MIN_PROBLEMS ? shared_lanes(M) : 32;
}

// The kernels of one piece count and lane count. One instantiation per supported piece count (loops over pieces/nodes
// unroll: 1.27x); sampling schedule by sample_schedule (minco_tile.cuh). Every k_optimize variant is sized for 12
// warps per SM (168 registers, no spills: config 5 38.7 -> 33.2 ms against 8 warps) and exists twice: three CTAs of 4
// warps per SM (small batches: spread over all SMs, nobody waits) and ONE CTA of 12 warps whose warps leave the
// evaluation site in groups of nine, sharing their instruction fetches (config 4 33.9 -> 26.4 ms, config 5 33.2 -> 30.5
// ms, neutral at 2,048 problems).
struct Variant {
    void (*opt)(const DevParams, const OptArgs) = nullptr;
    int opt_wpc = WARPS_PER_CTA;     // warps per CTA of opt
    void (*eval)(const DevParams, const EvalArgs) = nullptr;
};

template <int MC, int TL>
static Variant kernels(bool grouped)
{
    Variant v;
    v.eval = k_eval<MC, TL>;
    if (grouped) { v.opt = k_optimize<MC, TL, 1, 3 * WARPS_PER_CTA>; v.opt_wpc = 3 * WARPS_PER_CTA; }
    else v.opt = k_optimize<MC, TL, 3, WARPS_PER_CTA>;
    return v;
}

// TL: tile_lanes; only M <= 4 has shared-tile kernels
template <int MC>
static Variant variant(int TL, bool grouped)
{
    if constexpr (MC <= 4)
        if (TL < 32) return kernels<MC, shared_lanes(MC)>(grouped);
    return kernels<MC, 32>(grouped);
}

static Variant pick_variant(int M, int TL, bool grouped)
{
    switch (M) {
#ifndef NEO_FAST_BUILD      // development builds (-DNEO_FAST_BUILD) instantiate M = 3 only
        case 2: return variant<2>(TL, grouped);
        case 4: return variant<4>(TL, grouped);
        case 5: return variant<5>(TL, grouped);
        case 6: return variant<6>(TL, grouped);
        case 7: return variant<7>(TL, grouped);
        case 8: return variant<8>(TL, grouped);
        case 9: return variant<9>(TL, grouped);
        case 10: return variant<10>(TL, grouped);
#endif
        case 3: return variant<3>(TL, grouped);
        default: return Variant();
    }
}

static int launch_optimize(neo_handle *h, OptArgs a, cudaStream_t st)
{
    const int TL = tile_lanes(h, a.B, a.M);
    bool grouped = TL < 32 || a.B >= NEO_GROUPED_MIN_PROBLEMS;
    if (h->grouped >= 0) grouped = h->grouped != 0;
    const Variant v = pick_variant(a.M, TL, grouped);
    if (!v.opt) return fail(h, "M must be in [2, NEO_MAX_PIECES]");
    const int wpc = v.opt_wpc;
    a.bus_q = h->group_warps > 0 ? h->group_warps : 3 * wpc / 4;        // 12 warps: 9 (26.4 ms; 8: 26.5, 10: 26.9, 6: 27.9, 12: 30.2)
    if (a.bus_q > wpc) a.bus_q = wpc;
    const size_t smem = smem_bytes(a.M, TL, wpc);
    const size_t tasks = (size_t)a.B * a.max_attempts, n = 3 * a.M - 2;
    int grid;
    int rc = launch_grid(h, v.opt, smem, wpc, tasks, (size_t)wpc * (32 / TL), &grid);
    if (rc) return rc;
    // per-task scratch records + per-problem state word
    Layout L;
    const size_t o_x = L.add(sizeof(double) * tasks * n), o_c = L.add(sizeof(double) * tasks * 4),
                 o_w = L.add(sizeof(long long) * tasks * 4), o_i = L.add(sizeof(int32_t) * tasks * 4),
                 o_p = L.add(sizeof(unsigned) * a.B);
    char *s;
    if ((rc = grow(h, h->opt_scratch, L.end, &s))) return rc;
    a.t_x = (double *)(s + o_x); a.t_costs = (double *)(s + o_c); a.t_work = (long long *)(s + o_w);
    a.t_info = (int32_t *)(s + o_i); a.p_state = (unsigned *)(s + o_p);
    a.maps = h->d_maps;
    a.counter = h->d_counter;
    CK(cudaMemsetAsync(h->d_counter, 0, sizeof(unsigned int), st));
    CK(cudaMemsetAsync(a.p_state, 0, sizeof(unsigned) * a.B, st));
    v.opt<<<grid, wpc * 32, smem, st>>>(dev_params(h->cfg), a);
    h->launches++;
    CK(cudaGetLastError());
    return NEO_OK;
}

static int launch_eval(neo_handle *h, EvalArgs a, cudaStream_t st)
{
    const int TL = tile_lanes(h, a.B, a.M);
    const auto kern = pick_variant(a.M, TL, false).eval;
    if (!kern) return fail(h, "M must be in [2, NEO_MAX_PIECES]");
    // evaluator-only shared memory (no optimizer state): half of k_optimize's per tile, so registers decide the occupancy
    const size_t smem = sizeof(double) * (size_t)eval_mem_doubles(a.M, TL) * WARPS_PER_CTA * (32 / TL);
    int grid;
    int rc = launch_grid(h, kern, smem, WARPS_PER_CTA, a.B, WARPS_PER_CTA * (32 / TL), &grid);
    if (rc) return rc;
    a.maps = h->d_maps;
    kern<<<grid, WARPS_PER_CTA * 32, smem, st>>>(dev_params(h->cfg), a);
    h->launches++;
    CK(cudaGetLastError());
    return NEO_OK;
}

// ---------------------------------------------------------------------------------------------------------
// eval
// ---------------------------------------------------------------------------------------------------------
// the argument checks of neo_eval and neo_eval_dev; `arrays`: the required arrays are all non-null
static int eval_check(neo_handle *h, const char *who, int B, int M, bool arrays)
{
    const int rc = check_problem(h, B, M);
    if (rc) return rc;
    if (!arrays) return fail(h, std::string(who) + ": null pointer");
    return NEO_OK;
}

extern "C" int neo_eval_dev(neo_handle *h, int B, int M, const double *x, const double *head, const double *tail,
                            const int32_t *map_ids, double *costs, double *grad, int32_t *status, double *coeffs,
                            double *ts, void *stream)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    const int rc = eval_check(h, "neo_eval_dev", B, M, x && head && tail && costs && grad && status);
    if (rc || B == 0) return rc;
    CK(cudaSetDevice(h->device));
    const EvalArgs a = {B, M, x, head, tail, map_ids, nullptr, costs, grad, coeffs, ts, status};
    return launch_eval(h, a, stream ? (cudaStream_t)stream : h->stream);
}

extern "C" int neo_eval(neo_handle *h, int B, int M, const double *x, const double *head, const double *tail,
                        const int32_t *map_ids, double *costs, double *grad, int32_t *status, double *coeffs, double *ts)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = eval_check(h, "neo_eval", B, M, x && head && tail && costs && grad && status);
    if (rc || B == 0) return rc;
    if ((rc = check_map_ids(h, B, map_ids, "neo_eval"))) return rc;
    CK(cudaSetDevice(h->device));
    const size_t n = 3 * M - 2, N2 = 12 * M, b = B;
    Layout L;
    const size_t o_x = L.add(sizeof(double) * b * n), o_head = L.add(sizeof(double) * b * 6),
                 o_tail = L.add(sizeof(double) * b * 6), o_ids = L.add(sizeof(int32_t) * b),
                 o_costs = L.add(sizeof(double) * b * 4), o_grad = L.add(sizeof(double) * b * n),
                 o_coeffs = L.add(sizeof(double) * b * N2), o_ts = L.add(sizeof(double) * b * M),
                 o_status = L.add(sizeof(int32_t) * b);
    char *d;
    if ((rc = grow(h, h->stage, L.end, &d))) return rc;
    cudaStream_t st = h->stream;
    CK(cudaMemcpyAsync(d + o_x, x, sizeof(double) * b * n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d + o_head, head, sizeof(double) * b * 6, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d + o_tail, tail, sizeof(double) * b * 6, cudaMemcpyHostToDevice, st));
    if (map_ids) CK(cudaMemcpyAsync(d + o_ids, map_ids, sizeof(int32_t) * b, cudaMemcpyHostToDevice, st));
    const EvalArgs a = {B, M, (const double *)(d + o_x), (const double *)(d + o_head), (const double *)(d + o_tail),
                        map_ids ? (const int32_t *)(d + o_ids) : nullptr, nullptr, (double *)(d + o_costs),
                        (double *)(d + o_grad), coeffs ? (double *)(d + o_coeffs) : nullptr,
                        ts ? (double *)(d + o_ts) : nullptr, (int32_t *)(d + o_status)};
    CK(cudaEventRecord(h->ev0, st));
    if ((rc = launch_eval(h, a, st))) return rc;
    CK(cudaEventRecord(h->ev1, st));
    CK(cudaMemcpyAsync(costs, d + o_costs, sizeof(double) * b * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(grad, d + o_grad, sizeof(double) * b * n, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(status, d + o_status, sizeof(int32_t) * b, cudaMemcpyDeviceToHost, st));
    if (coeffs) CK(cudaMemcpyAsync(coeffs, d + o_coeffs, sizeof(double) * b * N2, cudaMemcpyDeviceToHost, st));
    if (ts) CK(cudaMemcpyAsync(ts, d + o_ts, sizeof(double) * b * M, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    return NEO_OK;
}

// ---------------------------------------------------------------------------------------------------------
// optimize
// ---------------------------------------------------------------------------------------------------------
// map_T2tau (EP:468-475) with the C library's log() -- the function CPython's math.log calls.
static int T2tau_one(const neo_config *cfg, double T, double *tau)
{
    const double den = T - cfg->T_min;
    if (den == 0.0) return NEO_ST_DOMAIN;
    const double a = (cfg->T_max - cfg->T_min) / den - 1.0;
    if (!(a > 0.0) || isinf(a)) return NEO_ST_DOMAIN;
    *tau = -log(a);
    return 0;
}

extern "C" int neo_T2tau(const neo_config *cfg, int n, const double *ts, double *tau, int32_t *status)
{
    if (!cfg || n < 0 || !ts || !tau) return NEO_ERR_INVALID;
    for (int i = 0; i < n; i++) {
        double t = 0.0;
        const int st = T2tau_one(cfg, ts[i], &t);
        tau[i] = st ? 0.0 : t;
        if (status) status[i] = st;
    }
    return NEO_OK;
}

// neo_T2tau on the device: glibc's log restated (libm_log.h), so the results equal the host's bit for bit
extern "C" int neo_T2tau_dev(neo_handle *h, int n, const double *ts, double *tau, int32_t *status, void *stream)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (n < 0) return fail(h, "neo_T2tau_dev: n must be >= 0");
    if (!ts || !tau) return fail(h, "neo_T2tau_dev: null pointer");
    if (n == 0) return NEO_OK;
    CK(cudaSetDevice(h->device));
    CK(launch_T2tau(n, h->cfg.T_min, h->cfg.T_max, ts, tau, status, stream ? (cudaStream_t)stream : h->stream));
    h->launches++;
    return NEO_OK;
}

// The device inputs of neo_optimize_dev, built as optimize_host builds them: x0 = [q0, T2tau(ts0)] with its status,
// the straight-line guess where q0 is NULL, init_ts where ts0 is NULL, and the retry guesses line + noise. The map ids
// are host data: checked like every host-pointer entry point's, then copied to map_ids_dev.
extern "C" int neo_prepare_dev(neo_handle *h, int B, int M, const double *head, const double *tail, const double *q0,
                               const double *ts0, const double *init_ts, int count, const double *noise,
                               const int32_t *map_ids_host, double *x0, int32_t *x0_status, double *retry_q,
                               int32_t *map_ids_dev, void *stream)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = check_problem(h, B, M);
    if (rc) return rc;
    if (count < 0 || count > NEO_MAX_ATTEMPTS - 1) return fail(h, "neo_prepare_dev: count out of range");
    if (!head || !tail || !x0 || !x0_status || (!ts0 && !init_ts) || (count > 0 && (!noise || !retry_q)) ||
        (map_ids_host && !map_ids_dev))
        return fail(h, "neo_prepare_dev: null pointer");
    if (B == 0) return NEO_OK;
    if ((rc = check_map_ids(h, B, map_ids_host, "neo_prepare_dev"))) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    if (map_ids_host) CK(cudaMemcpyAsync(map_ids_dev, map_ids_host, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
    CK(launch_prepare(B, M, h->cfg.T_min, h->cfg.T_max, head, tail, q0, ts0, init_ts, count, noise, x0, x0_status,
                      retry_q, st));
    h->launches++;
    return NEO_OK;
}

// internal: device pointers, tau-form inputs
// the arrays of a neo_result, each with its bytes per problem of M pieces
template <typename F>
static void result_fields(neo_result &r, int M, F f)
{
    const size_t n = 3 * M - 2;
    f(r.x, sizeof(double) * n); f(r.ts, sizeof(double) * M); f(r.coeffs, sizeof(double) * 12 * M);
    f(r.costs, sizeof(double) * 4); f(r.status, sizeof(int32_t)); f(r.ok, sizeof(int32_t)); f(r.attempt, sizeof(int32_t));
    f(r.nit, sizeof(int32_t)); f(r.runs, sizeof(int32_t)); f(r.nfev, sizeof(int32_t)); f(r.work, sizeof(int64_t) * 4);
}

// the argument checks of neo_optimize_dev and neo_optimize(_trace); `inputs` / `retry`: the caller's required input
// arrays / its retry arrays are all non-null
static int optimize_check(neo_handle *h, const char *who, int B, int M, bool inputs, int max_attempts, bool retry,
                          const neo_result *o)
{
    const int rc = check_problem(h, B, M);
    if (rc) return rc;
    if (!inputs || !o || !o->x || !o->ts || !o->coeffs || !o->costs || !o->status || !o->ok || !o->attempt || !o->nit ||
        !o->runs || !o->nfev)
        return fail(h, std::string(who) + ": null pointer");
    if (max_attempts < 1 || max_attempts > NEO_MAX_ATTEMPTS) return fail(h, "max_attempts out of range");
    if (max_attempts > 1 && !retry) return fail(h, "retry arrays required when max_attempts > 1");
    return NEO_OK;
}

// OptArgs of one launch from device pointers and tau-form inputs; launch_optimize adds its scratch, the maps and the queue
static OptArgs opt_args(int B, int M, const double *x0, const int32_t *x0_status, const double *head, const double *tail,
                        const int32_t *map_ids, const double *retry_q, const double *retry_tau, int retry_status,
                        int max_attempts, const neo_result &out)
{
    OptArgs a = {};
    a.B = B; a.M = M; a.max_attempts = max_attempts;
    a.x0 = x0; a.x0_status = x0_status; a.head = head; a.tail = tail; a.map_ids = map_ids;
    a.retry_q = retry_q; a.retry_tau = retry_tau; a.retry_status = retry_status;
    a.x = out.x; a.ts = out.ts; a.coeffs = out.coeffs; a.costs = out.costs;
    a.status = out.status; a.ok = out.ok; a.attempt = out.attempt; a.nit = out.nit; a.runs = out.runs;
    a.nfev = out.nfev; a.work = (long long *)out.work;
    return a;
}

// Device-pointer entry. Inputs are in tau form (x0 = [q0, map_T2tau(ts0)], retry_tau = map_T2tau(retry_ts)): neo_prepare_dev
// builds them on the device, neo_T2tau on the host.
extern "C" int neo_optimize_dev(neo_handle *h, int B, int M, const double *x0, const int32_t *x0_status,
                                const double *head, const double *tail, const int32_t *map_ids, const double *retry_q,
                                const double *retry_tau, int retry_status, int max_attempts, const neo_result *out,
                                void *stream)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    const int rc = optimize_check(h, "neo_optimize_dev", B, M, x0 && head && tail, max_attempts, retry_q && retry_tau, out);
    if (rc || B == 0) return rc;
    CK(cudaSetDevice(h->device));
    return launch_optimize(h, opt_args(B, M, x0, x0_status, head, tail, map_ids, retry_q, retry_tau, retry_status,
                                       max_attempts, *out),
                           stream ? (cudaStream_t)stream : h->stream);
}

struct TraceHost {
    int cap;
    double *x, *f, *g, *costs;
    int32_t *status, *len;
};

// Host-buffer entry: inputs are assembled in ONE pinned staging buffer that mirrors the device layout
// (x0 = [q0, map_T2tau(ts0)], EP:207-211) in three stages, each copied while the next is assembled; results are written
// by the kernel straight into the same pinned buffer (mapped) and scattered into the caller's arrays once it ends. For
// large batches both host passes run on several threads (at 65,536 problems they move 50 MB and take 196,608 logarithms
// -- a quarter of the kernel's time on one thread).
static int optimize_host(neo_handle *h, int B, int M, const double *q0, const double *ts0, const double *head,
                         const double *tail, const int32_t *map_ids, const double *retry_q, const double *retry_ts,
                         int max_attempts, neo_result *out, const TraceHost *trace)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = optimize_check(h, "neo_optimize", B, M, q0 && ts0 && head && tail, max_attempts, retry_q && retry_ts, out);
    if (rc) return rc;
    if (trace && (trace->cap < 1 || !trace->x || !trace->f || !trace->g || !trace->costs || !trace->status || !trace->len))
        return fail(h, "neo_optimize_trace: null trace array");
    if (B == 0) return NEO_OK;
    if ((rc = check_map_ids(h, B, map_ids, "neo_optimize"))) return rc;
    CK(cudaSetDevice(h->device));
    const size_t n = 3 * M - 2, nq = 2 * (M - 1), b = B, A1 = max_attempts - 1;

    // the inputs sit at the same offsets in the pinned and in the device staging buffer
    Layout L;
    const size_t o_x0 = L.add(sizeof(double) * b * n), o_head = L.add(sizeof(double) * b * 6),
                 o_tail = L.add(sizeof(double) * b * 6), o_st0 = L.add(sizeof(int32_t) * b),
                 o_ids = L.add(sizeof(int32_t) * b), o_rtau = L.add(sizeof(double) * NEO_MAX_PIECES), in_end = L.end;
    // device only: the per-task evaluation trace (test path)
    Layout D = L;
    const size_t tasks = b * max_attempts, cap = trace ? trace->cap : 0;
    const size_t o_tx = D.add(sizeof(double) * tasks * cap * n), o_tg = D.add(sizeof(double) * tasks * cap * n),
                 o_tf = D.add(sizeof(double) * tasks * cap), o_tc = D.add(sizeof(double) * tasks * cap * 4),
                 o_tst = D.add(sizeof(int32_t) * tasks * cap), o_tl = D.add(sizeof(int32_t) * tasks);
    // pinned only: the retry guesses, then the results
    const size_t o_rq = L.add(sizeof(double) * b * A1 * nq);
    size_t o_res[11];
    int fi = 0;
    result_fields(*out, M, [&](auto &, size_t bytes) { o_res[fi++] = L.add(bytes * b); });
    char *dbase, *hbase;
    if ((rc = grow(h, h->stage, D.end, &dbase))) return rc;
    if ((rc = grow(h, h->pinned, L.end, &hbase))) return rc;

    double *hx0 = (double *)(hbase + o_x0);
    int32_t *hst = (int32_t *)(hbase + o_st0);
    const bool timing = h->host_timing;
    auto now = [] { return std::chrono::steady_clock::now(); };
    const auto t_begin = now();
    const neo_config cfg = h->cfg;
    std::atomic<int> any_bad_flag{0};
    // three stages, each copied to the device while the next one is assembled
    cudaStream_t st = h->stream;
    h->pool.run(b, [&](size_t i0, size_t i1) {
        bool bad = false;
        for (size_t i = i0; i < i1; i++) {
            memcpy(&hx0[i * n], q0 + i * nq, sizeof(double) * nq);
            int s0 = 0;
            for (int k = 0; k < M; k++) {
                double t = 0.0;
                const int s1 = T2tau_one(&cfg, ts0[i * M + k], &t);
                hx0[i * n + nq + k] = s1 ? 0.0 : t;
                if (s1) s0 = s1;
            }
            hst[i] = s0;
            bad = bad || s0;
        }
        if (bad) any_bad_flag.store(1);
    });
    CK(cudaMemcpyAsync(dbase + o_x0, hbase + o_x0, o_head - o_x0, cudaMemcpyHostToDevice, st));
    const bool any_bad = any_bad_flag.load() != 0;
    h->pool.run(b, [&](size_t i0, size_t i1) {
        memcpy(hbase + o_head + 48 * i0, head + i0 * 6, 48 * (i1 - i0));
        memcpy(hbase + o_tail + 48 * i0, tail + i0 * 6, 48 * (i1 - i0));
        if (map_ids) memcpy(hbase + o_ids + 4 * i0, map_ids + i0, 4 * (i1 - i0));
    });
    double *rtau = (double *)(hbase + o_rtau);
    int rstatus = 0;
    if (A1)
        for (int k = 0; k < M; k++) { rtau[k] = 0.0; const int s1 = T2tau_one(&h->cfg, retry_ts[k], &rtau[k]); if (s1) rstatus = s1; }
    CK(cudaMemcpyAsync(dbase + o_head, hbase + o_head, in_end - o_head, cudaMemcpyHostToDevice, st));     // head, tail, st0, ids, retry tau
    // the retry guesses (the largest input: 4 per problem) stay in the pinned buffer: only the problems that do retry
    // read theirs, through the mapped pointer, when the retry starts
    if (A1)
        h->pool.run(b, [&](size_t i0, size_t i1) {
            memcpy(hbase + o_rq + 8 * i0 * A1 * nq, retry_q + i0 * A1 * nq, 8 * (i1 - i0) * A1 * nq);
        });
    // results: the kernel writes every resolved problem's record straight into the pinned staging buffer (mapped host
    // memory; 0.46 KB per problem, spread over the whole launch), so no device-to-host copy follows the kernel
    char *rbase = nullptr;
    CK(cudaHostGetDevicePointer((void **)&rbase, hbase, 0));
    neo_result d = *out;
    fi = 0;
    result_fields(d, M, [&](auto &p, size_t) { if (p) p = (std::decay_t<decltype(p)>)(rbase + o_res[fi]); fi++; });
    OptArgs a = opt_args(B, M, (const double *)(dbase + o_x0), any_bad ? (const int32_t *)(dbase + o_st0) : nullptr,
                         (const double *)(dbase + o_head), (const double *)(dbase + o_tail),
                         map_ids ? (const int32_t *)(dbase + o_ids) : nullptr, A1 ? (const double *)(rbase + o_rq) : nullptr,
                         A1 ? (const double *)(dbase + o_rtau) : nullptr, rstatus, max_attempts, d);
    if (trace) {
        a.trace_cap = trace->cap;
        a.tr_x = (double *)(dbase + o_tx); a.tr_g = (double *)(dbase + o_tg); a.tr_f = (double *)(dbase + o_tf);
        a.tr_costs = (double *)(dbase + o_tc); a.tr_status = (int32_t *)(dbase + o_tst); a.tr_len = (int32_t *)(dbase + o_tl);
        CK(cudaMemsetAsync(a.tr_len, 0, sizeof(int32_t) * tasks, st));
    }
    const auto t_staged = now();
    CK(cudaEventRecord(h->ev0, st));
    if ((rc = launch_optimize(h, a, st))) return rc;
    CK(cudaEventRecord(h->ev1, st));
    if (trace) {
        CK(cudaMemcpyAsync(trace->x, a.tr_x, sizeof(double) * tasks * cap * n, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(trace->g, a.tr_g, sizeof(double) * tasks * cap * n, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(trace->f, a.tr_f, sizeof(double) * tasks * cap, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(trace->costs, a.tr_costs, sizeof(double) * tasks * cap * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(trace->status, a.tr_status, sizeof(int32_t) * tasks * cap, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(trace->len, a.tr_len, sizeof(int32_t) * tasks, cudaMemcpyDeviceToHost, st));
    }
    const auto t_launched = now();
    CK(cudaStreamSynchronize(st));
    const auto t_done = now();
    CK(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    h->pool.run(b, [&](size_t i0, size_t i1) {
        int fi = 0;
        result_fields(*out, M, [&](auto &p, size_t bytes) {
            if (p) memcpy((char *)p + bytes * i0, hbase + o_res[fi] + bytes * i0, bytes * (i1 - i0));
            fi++;
        });
    });
    if (timing) {
        auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b2) { return std::chrono::duration<double, std::milli>(b2 - a).count(); };
        fprintf(stderr, "neo_optimize B=%d: stage inputs %.3f ms, launch %.3f ms, wait %.3f ms (kernel %.3f ms), scatter %.3f ms\n", B,
                ms(t_begin, t_staged), ms(t_staged, t_launched), ms(t_launched, t_done), h->last_ms, ms(t_done, now()));
    }
    return NEO_OK;
}

extern "C" int neo_optimize(neo_handle *h, int B, int M, const double *q0, const double *ts0, const double *head,
                            const double *tail, const int32_t *map_ids, const double *retry_q, const double *retry_ts,
                            int max_attempts, neo_result *out)
{
    return optimize_host(h, B, M, q0, ts0, head, tail, map_ids, retry_q, retry_ts, max_attempts, out, nullptr);
}

extern "C" int neo_optimize_trace(neo_handle *h, int B, int M, const double *q0, const double *ts0, const double *head,
                                  const double *tail, const int32_t *map_ids, const double *retry_q, const double *retry_ts,
                                  int max_attempts, neo_result *out, int trace_cap, double *tr_x, double *tr_f, double *tr_g,
                                  double *tr_costs, int32_t *tr_status, int32_t *tr_len)
{
    const TraceHost t = {trace_cap, tr_x, tr_f, tr_g, tr_costs, tr_status, tr_len};
    return optimize_host(h, B, M, q0, ts0, head, tail, map_ids, retry_q, retry_ts, max_attempts, out, &t);
}

// ---------------------------------------------------------------------------------------------------------
// coefficients / sampling
// ---------------------------------------------------------------------------------------------------------
static int coeffs_check(neo_handle *h, const char *who, int B, int M, bool arrays)
{
    if (B < 0 || M < 2 || M > NEO_MAX_PIECES) return fail(h, std::string(who) + ": B or M out of range");
    if (!arrays) return fail(h, std::string(who) + ": null pointer");
    return NEO_OK;
}

static int launch_coeffs(neo_handle *h, int B, int M, const double *q, const double *ts, const double *head,
                         const double *tail, double *coeffs, cudaStream_t st)
{
    int grid;
    const int rc = launch_grid(h, k_coeffs, smem_bytes(M), WARPS_PER_CTA, B, WARPS_PER_CTA, &grid);
    if (rc) return rc;
    k_coeffs<<<grid, WARPS_PER_CTA * 32, smem_bytes(M), st>>>(B, M, q, ts, head, tail, coeffs);
    h->launches++;
    CK(cudaGetLastError());
    return NEO_OK;
}

extern "C" int neo_get_coeffs_dev(neo_handle *h, int B, int M, const double *q, const double *ts, const double *head,
                                  const double *tail, double *coeffs, void *stream)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    const int rc = coeffs_check(h, "neo_get_coeffs_dev", B, M, q && ts && head && tail && coeffs);
    if (rc || B == 0) return rc;
    CK(cudaSetDevice(h->device));
    return launch_coeffs(h, B, M, q, ts, head, tail, coeffs, stream ? (cudaStream_t)stream : h->stream);
}

extern "C" int neo_get_coeffs(neo_handle *h, int B, int M, const double *q, const double *ts, const double *head,
                              const double *tail, double *coeffs)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = coeffs_check(h, "neo_get_coeffs", B, M, q && ts && head && tail && coeffs);
    if (rc || B == 0) return rc;
    CK(cudaSetDevice(h->device));
    const size_t nq = 2 * (M - 1), N2 = 12 * M, b = B;
    Layout L;
    const size_t o_q = L.add(sizeof(double) * b * nq), o_ts = L.add(sizeof(double) * b * M),
                 o_head = L.add(sizeof(double) * b * 6), o_tail = L.add(sizeof(double) * b * 6),
                 o_c = L.add(sizeof(double) * b * N2);
    char *d;
    if ((rc = grow(h, h->stage, L.end, &d))) return rc;
    cudaStream_t st = h->stream;
    CK(cudaMemcpyAsync(d + o_q, q, sizeof(double) * b * nq, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d + o_ts, ts, sizeof(double) * b * M, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d + o_head, head, sizeof(double) * b * 6, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d + o_tail, tail, sizeof(double) * b * 6, cudaMemcpyHostToDevice, st));
    if ((rc = launch_coeffs(h, B, M, (const double *)(d + o_q), (const double *)(d + o_ts), (const double *)(d + o_head),
                            (const double *)(d + o_tail), (double *)(d + o_c), st)))
        return rc;
    CK(cudaMemcpyAsync(coeffs, d + o_c, sizeof(double) * b * N2, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return NEO_OK;
}

static int sample_check(neo_handle *h, const char *who, int B, int M, double hz, bool arrays, const double *states,
                        int max_samples)
{
    if (B < 0 || M < 1 || M > 64 || !(hz > 0.0)) return fail(h, std::string(who) + ": invalid argument");
    if (!arrays || (states && max_samples < 1)) return fail(h, std::string(who) + ": null pointer");
    return NEO_OK;
}

static int launch_sample(neo_handle *h, int B, int M, const double *coeffs, const double *ts, double hz, int max_samples,
                         double *states, int32_t *count, cudaStream_t st)
{
    dim3 grid(states ? (max_samples + 127) / 128 : 1, B < 65535 ? B : 65535);
    k_sample<<<grid, 128, 0, st>>>(B, M, coeffs, ts, hz, max_samples, states, count);
    h->launches++;
    CK(cudaGetLastError());
    return NEO_OK;
}

extern "C" int neo_sample_dev(neo_handle *h, int B, int M, const double *coeffs, const double *ts, double hz,
                              int max_samples, double *states, int32_t *count, void *stream)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    const int rc = sample_check(h, "neo_sample_dev", B, M, hz, coeffs && ts && count, states, max_samples);
    if (rc || B == 0) return rc;
    CK(cudaSetDevice(h->device));
    return launch_sample(h, B, M, coeffs, ts, hz, max_samples, states, count, stream ? (cudaStream_t)stream : h->stream);
}

extern "C" int neo_sample(neo_handle *h, int B, int M, const double *coeffs, const double *ts, double hz, int max_samples,
                          double *states, int32_t *count)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = sample_check(h, "neo_sample", B, M, hz, coeffs && ts && count, states, max_samples);
    if (rc || B == 0) return rc;
    CK(cudaSetDevice(h->device));
    const size_t N2 = 12 * M, b = B, ms = states ? max_samples : 0;
    Layout L;
    const size_t o_c = L.add(sizeof(double) * b * N2), o_ts = L.add(sizeof(double) * b * M),
                 o_s = L.add(sizeof(double) * b * ms * 6), o_cnt = L.add(sizeof(int32_t) * b);
    char *d;
    if ((rc = grow(h, h->stage, L.end, &d))) return rc;
    cudaStream_t st = h->stream;
    CK(cudaMemcpyAsync(d + o_c, coeffs, sizeof(double) * b * N2, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d + o_ts, ts, sizeof(double) * b * M, cudaMemcpyHostToDevice, st));
    if (states) CK(cudaMemcpyAsync(d + o_s, states, sizeof(double) * b * ms * 6, cudaMemcpyHostToDevice, st));
    if ((rc = launch_sample(h, B, M, (const double *)(d + o_c), (const double *)(d + o_ts), hz, max_samples,
                            states ? (double *)(d + o_s) : nullptr, (int32_t *)(d + o_cnt), st)))
        return rc;
    CK(cudaMemcpyAsync(count, d + o_cnt, sizeof(int32_t) * b, cudaMemcpyDeviceToHost, st));
    if (states) CK(cudaMemcpyAsync(states, d + o_s, sizeof(double) * b * ms * 6, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (states) for (size_t i = 0; i < b; i++) if (count[i] > max_samples) return fail(h, "neo_sample: max_samples too small");
    return NEO_OK;
}

// ---------------------------------------------------------------------------------------------------------
// geometric initializer (astar_warp.cuh)
// ---------------------------------------------------------------------------------------------------------
constexpr size_t ASTAR_SCRATCH_BUDGET = (size_t)8 << 30;     // bytes of HBM the per-warp search scratch may take
constexpr int ASTAR_WARPS_PER_SM = 16;
constexpr int ASTAR_INSERT_CAP = 16384;       // inserted nodes per search the first pass has room for (28 B each)
constexpr int ASTAR_PASS1_WARPS = 16;         // warps of the second pass (full-size lists: 28 B per grid cell each)

static int astar_launch(neo_handle *h, int B, const double *start, const double *target, const int32_t *map_ids,
                        int max_closed, int max_path, double *path, int32_t *path_len, double *pruned, int32_t *status,
                        int32_t *closed, cudaStream_t st)
{
    // scratch per worker warp: one 4-byte node record per cell of the largest enlarged grid among the uploaded maps, and
    // insertion list + open-list spill for icap inserted nodes; a few warps of the second pass get full-size lists
    size_t cap = 0;
    for (auto &s : h->slots)
        if (s.cells) { const size_t c = astar_grid_cells(s.H, s.W, s.res); cap = c > cap ? c : cap; }
    if (cap == 0) return fail(h, "neo_astar: no map uploaded");
    for (auto &s : h->slots)
        if (s.cells && (s.W + (int)(10.0 / s.res) > 0xffff || s.H + (int)(10.0 / s.res) > 0x7fff))
            return fail(h, "neo_astar: search grid too large (node coordinates are packed into 16 bits)");
    if (cap >= ((size_t)1 << 27)) return fail(h, "neo_astar: search grid too large (open positions are packed into 28 bits)");
    size_t icap = h->astar_icap > 0 ? (size_t)h->astar_icap : (size_t)ASTAR_INSERT_CAP;
    if (icap > cap) icap = cap;
    const size_t list0 = ASTAR_BYTES_PER_INSERT * icap + sizeof(int) * ASTAR_ORDER_SLACK;
    const size_t list1 = ASTAR_BYTES_PER_INSERT * cap + sizeof(int) * ASTAR_ORDER_SLACK;
    const size_t per_warp = sizeof(AstarNode) * cap + list0;
    size_t warps1 = ASTAR_PASS1_WARPS;
    if (list1 * warps1 > ASTAR_SCRATCH_BUDGET / 4) warps1 = ASTAR_SCRATCH_BUDGET / 4 / list1;
    warps1 = warps1 / ASTAR_WARPS_PER_CTA * ASTAR_WARPS_PER_CTA;
    if (warps1 < (size_t)ASTAR_WARPS_PER_CTA) warps1 = ASTAR_WARPS_PER_CTA;
    const size_t budget0 = ASTAR_SCRATCH_BUDGET - list1 * warps1;
    if (per_warp * ASTAR_WARPS_PER_CTA > budget0) return fail(h, "neo_astar: search grid too large for the scratch budget");
    size_t warps = (size_t)h->sm_count * ASTAR_WARPS_PER_SM;
    if (warps > budget0 / per_warp) warps = budget0 / per_warp;
    if (warps > (size_t)B) warps = B;
    if (warps < 1) warps = 1;
    warps = (warps + ASTAR_WARPS_PER_CTA - 1) / ASTAR_WARPS_PER_CTA * ASTAR_WARPS_PER_CTA;     // whole CTAs
    if (warps < warps1) warps = warps1;                                                         // pass 1 borrows node blocks
    if (h->astar_cap != cap || (size_t)h->astar_warps < warps || h->astar_laid_icap != icap) {
        if (h->astar.p) { CK(cudaStreamSynchronize(st)); CK(cudaFree(h->astar.p)); h->astar.p = nullptr; }
        h->astar_cap = 0; h->astar_warps = 0;
        CK(cudaMalloc(&h->astar.p, per_warp * warps + list1 * warps1));
        CK(cudaMemsetAsync(h->astar.p, 0, sizeof(AstarNode) * cap * warps, st));   // nodes untouched
        CK(cudaFuncSetAttribute(k_astar, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ASTAR_SMEM_BYTES));
        h->astar_cap = cap; h->astar_warps = (int)warps; h->astar_laid_icap = icap;
    }
    char *overflow;
    const int rc = grow(h, h->astar_overflow, sizeof(int32_t) * (size_t)B, &overflow);
    if (rc) return rc;
    AstarArgs a;
    a.maps = h->d_maps; a.map_ids = map_ids; a.start = start; a.target = target;
    a.B = B; a.max_closed = max_closed; a.max_path = max_path;
    a.path = path; a.path_len = path_len; a.status = status; a.closed = closed; a.pruned = pruned;
    const size_t laid = (size_t)h->astar_warps;                 // the layout follows the allocation, not this launch
    // [nodes: laid x cap x 4 B][pass 0: spill laid x icap x 24 B | order laid x (icap + 8) x 4 B][pass 1: spill | order]
    char *p0 = (char *)h->astar.p + sizeof(AstarNode) * cap * laid;
    char *p1 = p0 + list0 * laid;
    a.nodes = (AstarNode *)h->astar.p;
    a.cap = cap;
    a.overflow = (int32_t *)overflow;
    a.overflow_count = h->d_counter + 18;
    CK(cudaMemsetAsync(h->d_counter + 16, 0, 3 * sizeof(unsigned int), st));
    // pass 0
    a.spill = (OpenRec *)p0; a.order = (int *)(p0 + sizeof(OpenRec) * icap * laid);
    a.icap = (int)icap; a.pass = 0; a.counter = h->d_counter + 16;
    k_astar<<<(unsigned)(warps / ASTAR_WARPS_PER_CTA), ASTAR_WARPS_PER_CTA * 32, ASTAR_SMEM_BYTES, st>>>(a);
    h->launches++;
    CK(cudaGetLastError());
    // pass 1: searches that inserted more than icap nodes, on a few warps with lists as long as the grid (usually none:
    // the kernel reads the count on the device and returns)
    if (icap < cap) {
        a.spill = (OpenRec *)p1; a.order = (int *)(p1 + sizeof(OpenRec) * cap * warps1);
        a.icap = (int)cap; a.pass = 1; a.counter = h->d_counter + 17;
        k_astar<<<(unsigned)(warps1 / ASTAR_WARPS_PER_CTA), ASTAR_WARPS_PER_CTA * 32, ASTAR_SMEM_BYTES, st>>>(a);
        h->launches++;
        CK(cudaGetLastError());
    }
    return NEO_OK;
}

static int astar_check(neo_handle *h, int B, const double *start, const double *target, int max_closed, int max_path,
                       const double *path, const int32_t *path_len, const double *pruned, const int32_t *status,
                       const int32_t *closed)
{
    if (B < 0 || max_closed < 0 || max_path < 0) return fail(h, "neo_astar: invalid argument");
    if (!start || !target || !path_len || !pruned || !status || !closed || (path && max_path < 1))
        return fail(h, "neo_astar: null pointer");
    return NEO_OK;
}

extern "C" int neo_astar_dev(neo_handle *h, int B, const double *start, const double *target, const int32_t *map_ids,
                             int max_closed, int max_path, double *path, int32_t *path_len, double *pruned,
                             int32_t *status, int32_t *closed, void *stream)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = astar_check(h, B, start, target, max_closed, max_path, path, path_len, pruned, status, closed);
    if (rc) return rc;
    if (B == 0) return NEO_OK;
    CK(cudaSetDevice(h->device));
    return astar_launch(h, B, start, target, map_ids, max_closed, max_path, path, path_len, pruned, status, closed,
                        stream ? (cudaStream_t)stream : h->stream);
}

extern "C" int neo_astar(neo_handle *h, int B, const double *start, const double *target, const int32_t *map_ids,
                         int max_closed, int max_path, double *path, int32_t *path_len, double *pruned, int32_t *status,
                         int32_t *closed)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = astar_check(h, B, start, target, max_closed, max_path, path, path_len, pruned, status, closed);
    if (rc || B == 0) return rc;
    for (int i = 0; i < 2 * B; i++)
        if (!isfinite(start[i]) || !isfinite(target[i])) return fail(h, "neo_astar: start/target must be finite");
    if ((rc = check_map_ids(h, B, map_ids, "neo_astar"))) return rc;
    CK(cudaSetDevice(h->device));
    const size_t b = B, np = path ? (size_t)max_path : 0;
    Layout L;
    const size_t o_s = L.add(sizeof(double) * 2 * b), o_t = L.add(sizeof(double) * 2 * b),
                 o_pr = L.add(sizeof(double) * 8 * b), o_path = L.add(sizeof(double) * 2 * b * np),
                 o_ids = L.add(sizeof(int32_t) * b), o_len = L.add(sizeof(int32_t) * b), o_st = L.add(sizeof(int32_t) * b),
                 o_cl = L.add(sizeof(int32_t) * b);
    char *d;
    if ((rc = grow(h, h->stage, L.end, &d))) return rc;
    cudaStream_t st = h->stream;
    CK(cudaMemcpyAsync(d + o_s, start, sizeof(double) * 2 * b, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d + o_t, target, sizeof(double) * 2 * b, cudaMemcpyHostToDevice, st));
    if (map_ids) CK(cudaMemcpyAsync(d + o_ids, map_ids, sizeof(int32_t) * b, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(h->ev0, st));
    rc = astar_launch(h, B, (const double *)(d + o_s), (const double *)(d + o_t), map_ids ? (const int32_t *)(d + o_ids) : nullptr,
                      max_closed, max_path, path ? (double *)(d + o_path) : nullptr, (int32_t *)(d + o_len),
                      (double *)(d + o_pr), (int32_t *)(d + o_st), (int32_t *)(d + o_cl), st);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev1, st));
    CK(cudaMemcpyAsync(path_len, d + o_len, sizeof(int32_t) * b, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(status, d + o_st, sizeof(int32_t) * b, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(closed, d + o_cl, sizeof(int32_t) * b, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(pruned, d + o_pr, sizeof(double) * 8 * b, cudaMemcpyDeviceToHost, st));
    if (path) CK(cudaMemcpyAsync(path, d + o_path, sizeof(double) * 2 * b * np, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    return NEO_OK;
}

// ---------------------------------------------------------------------------------------------------------
// measurement helpers
// ---------------------------------------------------------------------------------------------------------
extern "C" int neo_last_kernel_ms(neo_handle *h, float *ms)
{
    if (!h || !ms) return NEO_ERR_INVALID;
    *ms = h->last_ms;
    return NEO_OK;
}

extern "C" int neo_launch_count(neo_handle *h, int64_t *count)
{
    if (!h || !count) return NEO_ERR_INVALID;
    *count = h->launches;
    return NEO_OK;
}

extern "C" int neo_fp64_peak(neo_handle *h, double *tflops)
{
    if (!h || !tflops) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    CK(cudaSetDevice(h->device));
    const int threads = 256, blocks = h->sm_count * 8, iters = 1 << 16;
    char *d;
    const int rc = grow(h, h->stage, sizeof(double) * threads * blocks, &d);
    if (rc) return rc;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CK(cudaEventRecord(h->ev0, h->stream));
        k_fp64_peak<<<blocks, threads, 0, h->stream>>>((double *)d, iters);
        CK(cudaEventRecord(h->ev1, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        float ms;
        CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        if (rep && ms < best) best = ms;
        h->launches++;
    }
    *tflops = 2.0 * 8.0 * (double)iters * threads * blocks / (best * 1e-3) / 1e12;
    return NEO_OK;
}

// test hooks: exp_dd on the device and on the host build of the same header
extern "C" int neo_test_exp_dev(neo_handle *h, int n, const double *x, double *y)
{
    if (!h || n < 0 || !x || !y) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (n == 0) return NEO_OK;
    CK(cudaSetDevice(h->device));
    Layout L;
    const size_t o_x = L.add(sizeof(double) * n), o_y = L.add(sizeof(double) * n);
    char *d;
    const int rc = grow(h, h->stage, L.end, &d);
    if (rc) return rc;
    CK(cudaMemcpyAsync(d + o_x, x, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    k_exp_dd<<<(n + 255) / 256, 256, 0, h->stream>>>(n, (const double *)(d + o_x), (double *)(d + o_y));
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(y, d + o_y, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return NEO_OK;
}

// test hooks: the optimizer's dnrm2 (x87_nrm2.h) and its two inner products as the device build computes them
static int test_blas_prims(neo_handle *h, int count, int n, const double *a, const double *b, double *out)
{
    std::lock_guard<std::mutex> g(h->mu);
    if (count == 0 || n == 0) { for (size_t i = 0; i < 3 * (size_t)count; i++) out[i] = 0.0; return NEO_OK; }
    CK(cudaSetDevice(h->device));
    const size_t len = (size_t)count * n;
    Layout L;
    const size_t o_a = L.add(sizeof(double) * len), o_b = L.add(sizeof(double) * len),
                 o_out = L.add(sizeof(double) * 3 * (size_t)count);
    char *d;
    const int rc = grow(h, h->stage, L.end, &d);
    if (rc) return rc;
    CK(cudaMemcpyAsync(d + o_a, a, sizeof(double) * len, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d + o_b, b ? b : a, sizeof(double) * len, cudaMemcpyHostToDevice, h->stream));
    launch_blas_prims(count, n, (const double *)(d + o_a), (const double *)(d + o_b), (double *)(d + o_out), h->stream);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d + o_out, sizeof(double) * 3 * count, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return NEO_OK;
}

extern "C" int neo_test_nrm2_dev(neo_handle *h, int count, int n, const double *v, double *nrm)
{
    if (!h || count < 0 || n < 0 || !v || !nrm) return NEO_ERR_INVALID;
    std::vector<double> out(3 * (size_t)count);
    const int rc = test_blas_prims(h, count, n, v, nullptr, out.data());
    if (rc) return rc;
    for (int i = 0; i < count; i++) nrm[i] = out[3 * (size_t)i];
    return NEO_OK;
}

extern "C" int neo_test_ddot_dev(neo_handle *h, int count, int n, const double *a, const double *b, double *blas, double *loop)
{
    if (!h || count < 0 || n < 0 || !a || !b || !blas || !loop) return NEO_ERR_INVALID;
    std::vector<double> out(3 * (size_t)count);
    const int rc = test_blas_prims(h, count, n, a, b, out.data());
    if (rc) return rc;
    for (int i = 0; i < count; i++) { blas[i] = out[3 * (size_t)i + 1]; loop[i] = out[3 * (size_t)i + 2]; }
    return NEO_OK;
}

// test hook (no GPU needed): `calls` runs of the host worker pool over [0, count); every index must be visited exactly once
// per run. Returns the number of indices whose visit count is wrong.
extern "C" int neo_test_host_pool(long long count, int calls)
{
    HostPool pool;
    std::vector<unsigned char> hits((size_t)count);
    long long bad = 0;
    for (int c = 0; c < calls; c++) {
        std::fill(hits.begin(), hits.end(), 0);
        pool.run((size_t)count, [&](size_t i0, size_t i1) { for (size_t i = i0; i < i1; i++) hits[i]++; });
        for (size_t i = 0; i < (size_t)count; i++) bad += hits[i] != 1;
    }
    return bad > 0x7fffffff ? 0x7fffffff : (int)bad;
}

extern "C" int neo_test_exp_host(int n, const double *x, double *y)
{
    for (int i = 0; i < n; i++) { bool o; y[i] = neo::exp_dd(x[i], &o); }
    return NEO_OK;
}
