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
#ifdef NEO_ROUND_TRACE
__device__ long long g_round_trace[12 * 2048 * 4];      // development probe: per warp of CTA 0, per round: arrive, go, evaluated, advanced
#endif
template <int MODE, int MC, int TL, int MINB, int WPC = WARPS_PER_CTA>
__global__ void __launch_bounds__(WPC * 32, MINB) k_optimize(const DevParams P, const OptArgs a)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Tile<TL> T(lane);
    constexpr int TPW = 32 / TL;
    const int M = MC > 0 ? MC : a.M, n = 3 * M - 2, nq = 2 * (M - 1), N = 6 * M, A = a.max_attempts;
    constexpr bool ONE_BLOCK = MODE == SAMPLE_BY_PIECE_STAGED;
    const TileMem m = carve(smem + (size_t)(warp * TPW + lane / TL) * tile_mem_doubles(M, TL, ONE_BLOCK), M, TL, ONE_BLOCK);
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
#ifdef NEO_ROUND_TRACE
    int rt_round = 0;
#endif
    for (;;) {
#ifdef NEO_ROUND_TRACE
        if (blockIdx.x == 0 && lane == 0 && rt_round < 2048) g_round_trace[(warp * 2048 + rt_round) * 4 + 0] = clock64();
#endif
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
#ifdef NEO_ROUND_TRACE
        if (blockIdx.x == 0 && lane == 0 && rt_round < 2048) g_round_trace[(warp * 2048 + rt_round) * 4 + 1] = clock64();
        const int rt_now = rt_round++;
#endif
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
                OT_BEGIN;
                eval_fg<MODE, TL>(T, P, a.maps[map_id], m, M, o.x, true, ev);
                OT(16);
#ifdef NEO_ROUND_TRACE
                if (blockIdx.x == 0 && lane == 0 && rt_now < 2048) g_round_trace[(warp * 2048 + rt_now) * 4 + 2] = clock64();
#endif
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
                opt_advance<TL, (MC > 0 ? 3 * MC - 2 : 0)>(T, m, n, o, a.p_state + b, lower_ok);
                if (o.status != ST_RUNNING) { running = false; ended = true; report = true; }
            }
        }
#ifdef NEO_ROUND_TRACE
        __syncwarp();
        if (blockIdx.x == 0 && lane == 0 && rt_now < 2048) g_round_trace[(warp * 2048 + rt_now) * 4 + 3] = clock64();
#endif
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
template <int MODE, int MC, int TL>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 3) k_eval(const DevParams P, const EvalArgs a)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Tile<TL> T(lane);
    constexpr int TPW = 32 / TL, TPC = WARPS_PER_CTA * TPW;
    const int M = MC > 0 ? MC : a.M, n = 3 * M - 2, N = 6 * M;
    const int tile = warp * TPW + lane / TL;
    constexpr bool ONE_BLOCK = MODE == SAMPLE_BY_PIECE_STAGED;
    const TileMem m = carve(smem + (size_t)tile * eval_mem_doubles(M, TL, ONE_BLOCK), M, TL, ONE_BLOCK, true);
    for (size_t b = (size_t)blockIdx.x * TPC + tile; b < (size_t)a.B; b += (size_t)gridDim.x * TPC) {
        begin_problem(T, m, M, a.head + b * 6, a.tail + b * 6);
        const MapView map = a.maps[a.map_ids ? a.map_ids[b] : 0];
        const double xl = T.tl < n ? a.x[b * n + T.tl] : 0.0;
        EvalOut ev;
        eval_fg<MODE, TL, true>(T, P, map, m, M, xl, true, ev);
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

// ---------------------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------------------
struct MapSlot {
    Cell *cells = nullptr;
    int8_t *occ = nullptr;       // binarised grid of the last occupancy / point-cloud build
    size_t occ_cap = 0;
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
    std::vector<DevBuf> bufs;        // reusable device staging buffers for the host-pointer entry points
    DevBuf pinned;                   // reusable pinned host staging buffer (neo_optimize)
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

static int fail(neo_handle *h, const char *msg)
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

// grow-only device staging buffer #i
static int dev_buf(neo_handle *h, size_t i, size_t bytes, void **out)
{
    if (h->bufs.size() <= i) h->bufs.resize(i + 1);
    DevBuf &b = h->bufs[i];
    if (b.cap < bytes) {
        if (b.p) CK(cudaFree(b.p));
        b.p = nullptr; b.cap = 0;
        size_t cap = bytes + bytes / 4 + 256;
        CK(cudaMalloc(&b.p, cap));
        b.cap = cap;
    }
    *out = b.p;
    return NEO_OK;
}

// grow-only pinned host staging buffer
static int pin_buf(neo_handle *h, size_t bytes, void **out)
{
    DevBuf &b = h->pinned;
    if (b.cap < bytes) {
        if (b.p) CK(cudaFreeHost(b.p));
        b.p = nullptr; b.cap = 0;
        const size_t cap = bytes + bytes / 4 + 256;
        CK(cudaHostAlloc(&b.p, cap, cudaHostAllocMapped));      // mapped: the optimizer writes its results straight into it
        b.cap = cap;
    }
    *out = b.p;
    return NEO_OK;
}

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
    for (auto &b : h->bufs) if (b.p) cudaFree(b.p);
    if (h->pinned.p) cudaFreeHost(h->pinned.p);
    if (h->astar.p) cudaFree(h->astar.p);
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
    return NEO_OK;
}

static int slot_publish(neo_handle *h, int slot, bool sync = true)
{
    MapSlot &s = h->slots[slot];
    MapView v;
    v.cells = s.cells; v.H = s.H; v.W = s.W; v.res = s.res; v.ox = s.ox; v.oy = s.oy; v.inv_res = 1.0 / s.res;
    v.blocked = nullptr;
    // node-blocked grid of the geometric initializer (AP:130-141), one byte per node of the enlarged grid
    const size_t nodes = astar_grid_cells(s.H, s.W, s.res);
    if (s.blocked_cap < nodes) {
        if (s.blocked) { CK(cudaStreamSynchronize(h->stream)); CK(cudaFree(s.blocked)); s.blocked = nullptr; s.blocked_cap = 0; }
        CK(cudaMalloc(&s.blocked, nodes));
        s.blocked_cap = nodes;
    }
    const int pad = (int)(10.0 / s.res);
    dim3 grid((s.W + pad + 127) / 128, s.H + pad);
    k_astar_blocked<<<grid, 128, 0, h->stream>>>(v, s.blocked);
    h->launches++;
    CK(cudaGetLastError());
    v.blocked = s.blocked;
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
    double *d;
    if ((rc = dev_buf(h, 0, sizeof(double) * 3 * n, (void **)&d))) return rc;
    CK(cudaMemcpyAsync(d, esdf, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d + n, gx, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d + 2 * n, gy, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    dim3 grid((W + 127) / 128, H);
    k_pack_cells<<<grid, 128, 0, h->stream>>>(d, d + n, d + 2 * n, H, W, h->slots[slot].cells, nullptr, nullptr);
    h->launches++;
    CK(cudaGetLastError());
    return slot_publish(h, slot);
}

// occupancy (device, int8) -> exact EDT -> cells; d_occ lives in staging buffer 0 (offset 0)
static int build_from_occ(neo_handle *h, int slot, int H, int W, double res, char *base, size_t off_g, size_t off_any, size_t off_e,
                          bool sync = true)
{
    const int8_t *d_occ = (const int8_t *)base;
    int *d_g = (int *)(base + off_g), *d_any = (int *)(base + off_any);
    double *d_e = (double *)(base + off_e);
    MapSlot &s = h->slots[slot];
    const size_t n = (size_t)H * W;
    if (s.occ && s.occ_cap < n) { CK(cudaFree(s.occ)); s.occ = nullptr; }
    if (!s.occ) { CK(cudaMalloc(&s.occ, n)); s.occ_cap = n; }
    CK(cudaMemcpyAsync(s.occ, d_occ, n, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemsetAsync(d_any, 0, sizeof(int), h->stream));
    k_edt_rows<<<(H + 7) / 8, 256, 0, h->stream>>>(d_occ, H, W, d_g, d_any);                 // one warp per row
    dim3 grid((W + 127) / 128, H);
    k_edt_cols<<<grid, 128, 0, h->stream>>>(d_g, H, W, d_any, res, d_e);
    k_pack_cells<<<grid, 128, 0, h->stream>>>(d_e, nullptr, nullptr, H, W, s.cells, nullptr, nullptr);
    h->launches += 3;
    CK(cudaGetLastError());
    return slot_publish(h, slot, sync);
}

struct OccLayout { size_t off_g, off_any, off_e, total; };
static OccLayout occ_layout(size_t n)
{
    OccLayout L;
    L.off_g = (n + 255) & ~(size_t)255;
    L.off_any = L.off_g + sizeof(int) * n;
    L.off_e = (L.off_any + 256 + 255) & ~(size_t)255;
    L.total = L.off_e + sizeof(double) * n;
    return L;
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
    const OccLayout L = occ_layout(n);
    char *base;
    if ((rc = dev_buf(h, 0, L.total, (void **)&base))) return rc;
    CK(cudaMemcpyAsync(base, occ, n, cudaMemcpyHostToDevice, h->stream));
    return build_from_occ(h, slot, H, W, res, base, L.off_g, L.off_any, L.off_e);
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
    const OccLayout L = occ_layout(n);
    const size_t stride = (L.total + 255) & ~(size_t)255;
    const int group = K < 32 ? K : 32;                        // staging for 32 maps at a time
    char *base;
    int rc = dev_buf(h, 0, stride * group, (void **)&base);
    if (rc) return rc;
    for (int k0 = 0; k0 < K; k0 += group) {
        const int kn = K - k0 < group ? K - k0 : group;
        if (k0) CK(cudaStreamSynchronize(h->stream));          // the staging block is reused by the next group
        for (int k = 0; k < kn; k++) {
            if ((rc = slot_prepare(h, slots[k0 + k], H, W, res, ox[k0 + k], oy[k0 + k]))) return rc;
            CK(cudaMemcpyAsync(base + stride * k, occ + n * (size_t)(k0 + k), n, cudaMemcpyHostToDevice, h->stream));
        }
        for (int k = 0; k < kn; k++)
            if ((rc = build_from_occ(h, slots[k0 + k], H, W, res, base + stride * k, L.off_g, L.off_any, L.off_e, false))) return rc;
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
    const OccLayout L = occ_layout(n);
    char *base;
    float *d_xyz;
    if ((rc = dev_buf(h, 0, L.total, (void **)&base))) return rc;
    if ((rc = dev_buf(h, 1, sizeof(float) * 3 * (size_t)(n_points > 0 ? n_points : 1), (void **)&d_xyz))) return rc;
    CK(cudaMemsetAsync(base, 0, n, h->stream));
    if (n_points > 0) {
        CK(cudaMemcpyAsync(d_xyz, xyz, sizeof(float) * 3 * (size_t)n_points, cudaMemcpyHostToDevice, h->stream));
        k_points_to_occ<<<(n_points + 255) / 256, 256, 0, h->stream>>>(d_xyz, n_points, z_min, z_max, ox, oy, res, H, W,
                                                                       (int8_t *)base);
        h->launches++;
        CK(cudaGetLastError());
    }
    return build_from_occ(h, slot, H, W, res, base, L.off_g, L.off_any, L.off_e);
}

extern "C" int neo_get_occupancy(neo_handle *h, int slot, int8_t *occ)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (slot < 0 || slot >= (int)h->slots.size() || !h->slots[slot].occ || !occ) return fail(h, "neo_get_occupancy: no occupancy in this slot");
    CK(cudaSetDevice(h->device));
    const MapSlot &s = h->slots[slot];
    CK(cudaMemcpyAsync(occ, s.occ, (size_t)s.H * s.W, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return NEO_OK;
}

extern "C" int neo_get_map(neo_handle *h, int slot, double *esdf, double *gx, double *gy)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (slot < 0 || slot >= (int)h->slots.size() || !h->slots[slot].cells) return fail(h, "neo_get_map: empty slot");
    CK(cudaSetDevice(h->device));
    const MapSlot &s = h->slots[slot];
    const size_t n = (size_t)s.H * s.W;
    double *d;
    int rc = dev_buf(h, 0, sizeof(double) * 3 * n, (void **)&d);
    if (rc) return rc;
    k_unpack_cells<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(s.cells, n, d, d + n, d + 2 * n);
    h->launches++;
    CK(cudaGetLastError());
    if (esdf) CK(cudaMemcpyAsync(esdf, d, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    if (gx) CK(cudaMemcpyAsync(gx, d + n, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    if (gy) CK(cudaMemcpyAsync(gy, d + 2 * n, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
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
    const MapSlot &s = h->slots[slot];
    char *base;
    const size_t o_xy = 0, o_idx = sizeof(double) * 2 * n, o_dis = o_idx + sizeof(double) * n /* 8n >= 2*4n */,
                 o_grad = o_dis + sizeof(double) * n;
    int rc = dev_buf(h, 1, o_grad + sizeof(double) * 2 * n, (void **)&base);
    if (rc) return rc;
    CK(cudaMemcpyAsync(base + o_xy, xy, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, h->stream));
    MapView v;
    v.cells = s.cells; v.H = s.H; v.W = s.W; v.res = s.res; v.ox = s.ox; v.oy = s.oy; v.inv_res = 1.0 / s.res;
    v.blocked = s.blocked;
    k_query<<<(n + 127) / 128, 128, 0, h->stream>>>(v, n, (const double *)(base + o_xy), (int32_t *)(base + o_idx),
                                                    (double *)(base + o_dis), (double *)(base + o_grad));
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(idx, base + o_idx, sizeof(int32_t) * 2 * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(dis, base + o_dis, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(grad, base + o_grad, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost, h->stream));
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
        if (!h->slots[0].cells) { h->err = std::string(who) + ": map_ids is NULL and slot 0 holds no map"; return NEO_ERR_INVALID; }
        return NEO_OK;
    }
    for (int i = 0; i < B; i++)
        if (map_ids[i] < 0 || map_ids[i] >= (int)h->slots.size() || !h->slots[map_ids[i]].cells) {
            h->err = std::string(who) + ": map id " + std::to_string(map_ids[i]) + " (problem " + std::to_string(i) + ") refers to an empty slot";
            return NEO_ERR_INVALID;
        }
    return NEO_OK;
}

static size_t smem_bytes(int M, int TL = 32, bool one_block = false, int wpc = WARPS_PER_CTA)
{
    return sizeof(double) * (size_t)tile_mem_doubles(M, TL, one_block) * wpc * (32 / TL);
}

template <typename K>
static int prep_kernel(neo_handle *h, K kernel, size_t smem, int *ctas_per_sm, int wpc = WARPS_PER_CTA)
{
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, wpc * 32, smem));
    if (occ < 1) return fail(h, "kernel does not fit on an SM");
    *ctas_per_sm = occ;
    return NEO_OK;
}

// lanes per problem: M >= 5 needs the warp (n > 16); short trajectories share a warp once the batch is large enough to
// fill the machine with several problems per warp (below that, one problem per warp has the shorter evaluation)
static int tile_lanes(const neo_handle *h, int B, int M)
{
    if (M > 4) return 32;
    const int small = M <= 3 ? 8 : 16;
    if (h->tile) return h->tile == 32 ? 32 : small;
    return B >= NEO_TILE_MIN_PROBLEMS ? small : 32;
}

typedef void (*OptKernel)(const DevParams, const OptArgs);
template <int MODE, int MC, int TL, int MINB>
static OptKernel pick_optimize(bool grouped, int *wpc)
{
    if (grouped) { *wpc = 4 * MINB; return k_optimize<MODE, MC, TL, 1, 4 * MINB>; }
    return k_optimize<MODE, MC, TL, MINB, WARPS_PER_CTA>;
}

static int launch_optimize(neo_handle *h, OptArgs a, cudaStream_t st)
{
    int occ;
    // kernel variant: lanes per problem (tile_lanes) and sampling schedule (minco_tile.cuh) by trajectory length; one
    // instantiation per supported piece count (loops over pieces/nodes unroll: 1.27x). Every variant is sized for 12 warps
    // per SM (168 registers, no spills: config 5 38.7 -> 33.2 ms against 8 warps) and exists twice: three CTAs of 4 warps
    // per SM (small batches: spread over all SMs, nobody waits) and ONE CTA of 12 warps whose warps leave the evaluation
    // site in groups of nine, sharing their instruction fetches (config 4 33.9 -> 26.4 ms, config 5 33.2 -> 30.5 ms,
    // neutral at 2,048 problems).
    void (*kern)(const DevParams, const OptArgs) = nullptr;
    const int TL = tile_lanes(h, a.B, a.M);
    const bool staged = TL < 32;        // shared tiles: one staging block per tile (shared memory is what limits occupancy)
    bool grouped = TL < 32 || a.B >= NEO_GROUPED_MIN_PROBLEMS;
    if (h->grouped >= 0) grouped = h->grouped != 0;
    int wpc = WARPS_PER_CTA;
#define NEO_PICK(MODE, MC, TLV, MINB) pick_optimize<MODE, MC, TLV, MINB>(grouped, &wpc)
#define NEO_KW(MODE, MC) NEO_PICK(MODE, MC, 32, 3)
    switch (a.M) {
#ifndef NEO_FAST_BUILD      // development builds (-DNEO_FAST_BUILD) instantiate M = 3 only
        case 2: kern = TL == 8 ? NEO_PICK(SAMPLE_BY_PIECE_STAGED, 2, 8, 3) : NEO_KW(SAMPLE_BY_PIECE, 2); break;
        case 4: kern = TL == 16 ? NEO_PICK(SAMPLE_BY_PIECE_STAGED, 4, 16, 3) : NEO_KW(SAMPLE_BY_PIECE, 4); break;
        case 5: kern = NEO_KW(SAMPLE_ALL_PIECES, 5); break;
        case 6: kern = NEO_KW(SAMPLE_ALL_PIECES, 6); break;
        case 7: kern = NEO_KW(SAMPLE_ALL_PIECES, 7); break;
        case 8: kern = NEO_KW(SAMPLE_ALL_PIECES, 8); break;
        case 9: kern = NEO_KW(SAMPLE_ALL_PIECES, 9); break;
        case 10: kern = NEO_KW(SAMPLE_ALL_PIECES, 10); break;
#endif
        case 3: kern = TL == 8 ? NEO_PICK(SAMPLE_BY_PIECE_STAGED, 3, 8, 3) : NEO_KW(SAMPLE_BY_PIECE, 3); break;
        default: return fail(h, "M must be in [2, NEO_MAX_PIECES]");
    }
#undef NEO_KW
#undef NEO_PICK
    a.bus_q = h->group_warps > 0 ? h->group_warps : 3 * wpc / 4;        // 12 warps: 9 (26.4 ms; 8: 26.5, 10: 26.9, 6: 27.9, 12: 30.2)
    if (a.bus_q > wpc) a.bus_q = wpc;
    const size_t smem = smem_bytes(a.M, TL, staged, wpc);
    int rc = prep_kernel(h, kern, smem, &occ, wpc);
    if (rc) return rc;
    const size_t tasks = (size_t)a.B * a.max_attempts, n = 3 * a.M - 2;
    const size_t per_cta = (size_t)wpc * (32 / TL);
    const size_t need = (tasks + per_cta - 1) / per_cta;
    const int grid = (int)(need < (size_t)occ * h->sm_count ? need : (size_t)occ * h->sm_count);
    // per-task scratch records + per-problem state word (library-owned, grow-only)
    char *base;
    const size_t o_x = 0, o_c = o_x + sizeof(double) * tasks * n, o_w = o_c + sizeof(double) * tasks * 4,
                 o_i = o_w + sizeof(long long) * tasks * 4, o_p = o_i + sizeof(int32_t) * tasks * 4,
                 total = o_p + sizeof(unsigned) * a.B;
    if ((rc = dev_buf(h, 6, total, (void **)&base))) return rc;
    a.t_x = (double *)(base + o_x); a.t_costs = (double *)(base + o_c); a.t_work = (long long *)(base + o_w);
    a.t_info = (int32_t *)(base + o_i); a.p_state = (unsigned *)(base + o_p);
    a.maps = h->d_maps;
    a.counter = h->d_counter;
    CK(cudaMemsetAsync(h->d_counter, 0, sizeof(unsigned int), st));
    CK(cudaMemsetAsync(a.p_state, 0, sizeof(unsigned) * a.B, st));
    kern<<<grid, wpc * 32, smem, st>>>(dev_params(h->cfg), a);
    h->launches++;
    CK(cudaGetLastError());
    return NEO_OK;
}

static int launch_eval(neo_handle *h, EvalArgs a, cudaStream_t st)
{
    int occ;
    void (*kern)(const DevParams, const EvalArgs) = nullptr;
    const int TL = tile_lanes(h, a.B, a.M);
    switch (a.M) {
#ifndef NEO_FAST_BUILD
        case 2: kern = TL == 8 ? k_eval<SAMPLE_BY_PIECE_STAGED, 2, 8> : k_eval<SAMPLE_BY_PIECE, 2, 32>; break;
        case 4: kern = TL == 16 ? k_eval<SAMPLE_BY_PIECE_STAGED, 4, 16> : k_eval<SAMPLE_BY_PIECE, 4, 32>; break;
        case 5: kern = k_eval<SAMPLE_ALL_PIECES, 5, 32>; break;
        case 6: kern = k_eval<SAMPLE_ALL_PIECES, 6, 32>; break;
        case 7: kern = k_eval<SAMPLE_ALL_PIECES, 7, 32>; break;
        case 8: kern = k_eval<SAMPLE_ALL_PIECES, 8, 32>; break;
        case 9: kern = k_eval<SAMPLE_ALL_PIECES, 9, 32>; break;
        case 10: kern = k_eval<SAMPLE_ALL_PIECES, 10, 32>; break;
#endif
        case 3: kern = TL == 8 ? k_eval<SAMPLE_BY_PIECE_STAGED, 3, 8> : k_eval<SAMPLE_BY_PIECE, 3, 32>; break;
        default: return fail(h, "M must be in [2, NEO_MAX_PIECES]");
    }
    // evaluator-only shared memory (no optimizer state): half of k_optimize's per tile, so registers decide the occupancy
    const size_t smem = sizeof(double) * (size_t)eval_mem_doubles(a.M, TL, TL < 32) * WARPS_PER_CTA * (32 / TL);
    int rc = prep_kernel(h, kern, smem, &occ);
    if (rc) return rc;
    const int per_cta = WARPS_PER_CTA * (32 / TL);
    const int need = (a.B + per_cta - 1) / per_cta;
    const int grid = need < occ * h->sm_count ? need : occ * h->sm_count;
    a.maps = h->d_maps;
    kern<<<grid, WARPS_PER_CTA * 32, smem, st>>>(dev_params(h->cfg), a);
    h->launches++;
    CK(cudaGetLastError());
    return NEO_OK;
}

// byte-offset bump allocator over one staging buffer
struct Carver {
    char *base;
    size_t off = 0;
    template <typename T>
    T *take(size_t count)
    {
        off = (off + 255) & ~(size_t)255;
        T *p = base ? (T *)(base + off) : nullptr;
        off += sizeof(T) * count;
        return p;
    }
};

// ---------------------------------------------------------------------------------------------------------
// eval
// ---------------------------------------------------------------------------------------------------------
extern "C" int neo_eval_dev(neo_handle *h, int B, int M, const double *x, const double *head, const double *tail,
                            const int32_t *map_ids, double *costs, double *grad, int32_t *status, double *coeffs,
                            double *ts, void *stream)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = check_problem(h, B, M);
    if (rc) return rc;
    if (!x || !head || !tail || !costs || !grad || !status) return fail(h, "neo_eval_dev: null pointer");
    if (B == 0) return NEO_OK;
    CK(cudaSetDevice(h->device));
    EvalArgs a;
    a.B = B; a.M = M; a.x = x; a.head = head; a.tail = tail; a.map_ids = map_ids;
    a.costs = costs; a.grad = grad; a.status = status; a.coeffs = coeffs; a.ts = ts; a.maps = nullptr;
    return launch_eval(h, a, stream ? (cudaStream_t)stream : h->stream);
}

extern "C" int neo_eval(neo_handle *h, int B, int M, const double *x, const double *head, const double *tail,
                        const int32_t *map_ids, double *costs, double *grad, int32_t *status, double *coeffs, double *ts)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = check_problem(h, B, M);
    if (rc) return rc;
    if (!x || !head || !tail || !costs || !grad || !status) return fail(h, "neo_eval: null pointer");
    if (B == 0) return NEO_OK;
    if ((rc = check_map_ids(h, B, map_ids, "neo_eval"))) return rc;
    CK(cudaSetDevice(h->device));
    const size_t n = 3 * M - 2, N2 = 12 * M, b = B;
    for (int pass = 0; pass < 2; pass++) {
        Carver c{pass ? (char *)h->bufs[2].p : nullptr};
        double *d_x = c.take<double>(b * n), *d_head = c.take<double>(b * 6), *d_tail = c.take<double>(b * 6);
        int32_t *d_ids = c.take<int32_t>(b);
        double *d_costs = c.take<double>(b * 4), *d_grad = c.take<double>(b * n), *d_coeffs = c.take<double>(b * N2),
               *d_ts = c.take<double>(b * M);
        int32_t *d_status = c.take<int32_t>(b);
        if (!pass) {
            void *p;
            if ((rc = dev_buf(h, 2, c.off + 256, &p))) return rc;
            continue;
        }
        cudaStream_t st = h->stream;
        CK(cudaMemcpyAsync(d_x, x, sizeof(double) * b * n, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_head, head, sizeof(double) * b * 6, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_tail, tail, sizeof(double) * b * 6, cudaMemcpyHostToDevice, st));
        if (map_ids) CK(cudaMemcpyAsync(d_ids, map_ids, sizeof(int32_t) * b, cudaMemcpyHostToDevice, st));
        EvalArgs a;
        a.B = B; a.M = M; a.x = d_x; a.head = d_head; a.tail = d_tail; a.map_ids = map_ids ? d_ids : nullptr;
        a.costs = d_costs; a.grad = d_grad; a.status = d_status; a.coeffs = coeffs ? d_coeffs : nullptr;
        a.ts = ts ? d_ts : nullptr; a.maps = nullptr;
        CK(cudaEventRecord(h->ev0, st));
        if ((rc = launch_eval(h, a, st))) return rc;
        CK(cudaEventRecord(h->ev1, st));
        CK(cudaMemcpyAsync(costs, d_costs, sizeof(double) * b * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(grad, d_grad, sizeof(double) * b * n, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(status, d_status, sizeof(int32_t) * b, cudaMemcpyDeviceToHost, st));
        if (coeffs) CK(cudaMemcpyAsync(coeffs, d_coeffs, sizeof(double) * b * N2, cudaMemcpyDeviceToHost, st));
        if (ts) CK(cudaMemcpyAsync(ts, d_ts, sizeof(double) * b * M, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    }
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

// internal: device pointers, tau-form inputs
struct TraceDev {
    int cap = 0;
    double *x = nullptr, *f = nullptr, *g = nullptr, *costs = nullptr;
    int32_t *status = nullptr, *len = nullptr;
};

static int optimize_dev_impl(neo_handle *h, int B, int M, const double *x0, const int32_t *x0_status, const double *head,
                             const double *tail, const int32_t *map_ids, const double *retry_q, const double *retry_tau,
                             int retry_status, int max_attempts, const neo_result *out, cudaStream_t st,
                             const TraceDev *tr = nullptr)
{
    OptArgs a;
    a.trace_cap = tr ? tr->cap : 0;
    a.tr_x = tr ? tr->x : nullptr; a.tr_f = tr ? tr->f : nullptr; a.tr_g = tr ? tr->g : nullptr;
    a.tr_costs = tr ? tr->costs : nullptr; a.tr_status = tr ? tr->status : nullptr; a.tr_len = tr ? tr->len : nullptr;
    a.B = B; a.M = M; a.max_attempts = max_attempts;
    a.x0 = x0; a.x0_status = x0_status; a.head = head; a.tail = tail; a.map_ids = map_ids;
    a.retry_q = retry_q; a.retry_tau = retry_tau; a.retry_status = retry_status;
    a.maps = nullptr; a.counter = nullptr;
    a.x = out->x; a.ts = out->ts; a.coeffs = out->coeffs; a.costs = out->costs;
    a.status = out->status; a.ok = out->ok; a.attempt = out->attempt; a.nit = out->nit; a.runs = out->runs;
    a.nfev = out->nfev; a.work = (long long *)out->work;
    return launch_optimize(h, a, st);
}

static int result_complete(const neo_result *o)
{
    return o && o->x && o->ts && o->coeffs && o->costs && o->status && o->ok && o->attempt && o->nit && o->runs && o->nfev;
}

// Device-pointer entry. Inputs are in tau form (x0 = [q0, map_T2tau(ts0)], retry_tau = map_T2tau(retry_ts))
// because map_T2tau must run on the host libm to match the reference bit for bit (see neo_T2tau).
extern "C" int neo_optimize_dev(neo_handle *h, int B, int M, const double *x0, const int32_t *x0_status,
                                const double *head, const double *tail, const int32_t *map_ids, const double *retry_q,
                                const double *retry_tau, int retry_status, int max_attempts, const neo_result *out,
                                void *stream)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = check_problem(h, B, M);
    if (rc) return rc;
    if (!x0 || !head || !tail || !result_complete(out)) return fail(h, "neo_optimize_dev: null pointer");
    if (max_attempts < 1 || max_attempts > NEO_MAX_ATTEMPTS) return fail(h, "max_attempts out of range");
    if (max_attempts > 1 && (!retry_q || !retry_tau)) return fail(h, "retry arrays required when max_attempts > 1");
    if (B == 0) return NEO_OK;
    CK(cudaSetDevice(h->device));
    return optimize_dev_impl(h, B, M, x0, x0_status, head, tail, map_ids, retry_q, retry_tau, retry_status, max_attempts,
                             out, stream ? (cudaStream_t)stream : h->stream);
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
    int rc = check_problem(h, B, M);
    if (rc) return rc;
    if (!q0 || !ts0 || !head || !tail || !result_complete(out)) return fail(h, "neo_optimize: null pointer");
    if (max_attempts < 1 || max_attempts > NEO_MAX_ATTEMPTS) return fail(h, "max_attempts out of range");
    if (max_attempts > 1 && (!retry_q || !retry_ts)) return fail(h, "retry arrays required when max_attempts > 1");
    if (trace && (trace->cap < 1 || !trace->x || !trace->f || !trace->g || !trace->costs || !trace->status || !trace->len))
        return fail(h, "neo_optimize_trace: null trace array");
    if (B == 0) return NEO_OK;
    if ((rc = check_map_ids(h, B, map_ids, "neo_optimize"))) return rc;
    CK(cudaSetDevice(h->device));
    const size_t n = 3 * M - 2, nq = 2 * (M - 1), N2 = 12 * M, b = B, A1 = max_attempts - 1;

    struct Lay {
        size_t x0, head, tail, st0, ids, rq, rtau, in_end, x, ts, coeffs, costs, status, ok, attempt, nit, runs, nfev, work, end;
    } L;
    {
        size_t o = 0;
        auto off = [&](size_t bytes) { o = (o + 255) & ~(size_t)255; const size_t at = o; o += bytes; return at; };
        L.x0 = off(8 * b * n); L.head = off(8 * b * 6); L.tail = off(8 * b * 6); L.st0 = off(4 * b); L.ids = off(4 * b);
        L.rtau = off(8 * NEO_MAX_PIECES); L.in_end = off(0); L.rq = off(8 * (b * A1 * nq + 1));
        L.x = off(8 * b * n); L.ts = off(8 * b * M); L.coeffs = off(8 * b * N2); L.costs = off(8 * b * 4);
        L.status = off(4 * b); L.ok = off(4 * b); L.attempt = off(4 * b); L.nit = off(4 * b); L.runs = off(4 * b);
        L.nfev = off(4 * b); L.work = off(8 * b * 4); L.end = off(0);
    }
    char *dbase, *hbase;
    if ((rc = dev_buf(h, 3, L.end, (void **)&dbase))) return rc;
    if ((rc = pin_buf(h, L.end, (void **)&hbase))) return rc;

    double *hx0 = (double *)(hbase + L.x0);
    int32_t *hst = (int32_t *)(hbase + L.st0);
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
    CK(cudaMemcpyAsync(dbase + L.x0, hbase + L.x0, L.head - L.x0, cudaMemcpyHostToDevice, st));
    const bool any_bad = any_bad_flag.load() != 0;
    h->pool.run(b, [&](size_t i0, size_t i1) {
        memcpy(hbase + L.head + 48 * i0, head + i0 * 6, 48 * (i1 - i0));
        memcpy(hbase + L.tail + 48 * i0, tail + i0 * 6, 48 * (i1 - i0));
        if (map_ids) memcpy(hbase + L.ids + 4 * i0, map_ids + i0, 4 * (i1 - i0));
    });
    double *rtau = (double *)(hbase + L.rtau);
    int rstatus = 0;
    if (A1)
        for (int k = 0; k < M; k++) { rtau[k] = 0.0; const int s1 = T2tau_one(&h->cfg, retry_ts[k], &rtau[k]); if (s1) rstatus = s1; }
    CK(cudaMemcpyAsync(dbase + L.head, hbase + L.head, L.in_end - L.head, cudaMemcpyHostToDevice, st));     // head, tail, st0, ids, retry tau
    // the retry guesses (the largest input: 4 per problem) stay in the pinned buffer: only the problems that do retry
    // read theirs, through the mapped pointer, when the retry starts
    if (A1)
        h->pool.run(b, [&](size_t i0, size_t i1) {
            memcpy(hbase + L.rq + 8 * i0 * A1 * nq, retry_q + i0 * A1 * nq, 8 * (i1 - i0) * A1 * nq);
        });
    // results: the kernel writes every resolved problem's record straight into the pinned staging buffer (mapped host
    // memory; 0.46 KB per problem, spread over the whole launch), so no device-to-host copy follows the kernel
    char *rbase = nullptr;
    CK(cudaHostGetDevicePointer((void **)&rbase, hbase, 0));
    neo_result d;
    d.x = (double *)(rbase + L.x); d.ts = (double *)(rbase + L.ts); d.coeffs = (double *)(rbase + L.coeffs);
    d.costs = (double *)(rbase + L.costs);
    d.status = (int32_t *)(rbase + L.status); d.ok = (int32_t *)(rbase + L.ok); d.attempt = (int32_t *)(rbase + L.attempt);
    d.nit = (int32_t *)(rbase + L.nit); d.runs = (int32_t *)(rbase + L.runs); d.nfev = (int32_t *)(rbase + L.nfev);
    d.work = out->work ? (int64_t *)(rbase + L.work) : nullptr;
    TraceDev td;
    size_t tr_tasks = 0;
    if (trace) {      // test path: the per-task evaluation trace lives in its own device buffer
        tr_tasks = b * max_attempts;
        const size_t cap = trace->cap;
        Carver c{nullptr};
        for (int pass = 0; pass < 2; pass++) {
            c.off = 0;
            td.cap = trace->cap;
            td.x = c.take<double>(tr_tasks * cap * n); td.g = c.take<double>(tr_tasks * cap * n);
            td.f = c.take<double>(tr_tasks * cap); td.costs = c.take<double>(tr_tasks * cap * 4);
            td.status = c.take<int32_t>(tr_tasks * cap); td.len = c.take<int32_t>(tr_tasks);
            if (!pass) { void *p; if ((rc = dev_buf(h, 8, c.off + 256, &p))) return rc; c.base = (char *)p; }
        }
        CK(cudaMemsetAsync(td.len, 0, sizeof(int32_t) * tr_tasks, st));
    }
    const auto t_staged = now();
    CK(cudaEventRecord(h->ev0, st));
    rc = optimize_dev_impl(h, B, M, (const double *)(dbase + L.x0), any_bad ? (const int32_t *)(dbase + L.st0) : nullptr,
                           (const double *)(dbase + L.head), (const double *)(dbase + L.tail),
                           map_ids ? (const int32_t *)(dbase + L.ids) : nullptr, A1 ? (const double *)(rbase + L.rq) : nullptr,
                           A1 ? (const double *)(dbase + L.rtau) : nullptr, rstatus, max_attempts, &d, st, trace ? &td : nullptr);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev1, st));
    if (trace) {
        const size_t cap = trace->cap;
        CK(cudaMemcpyAsync(trace->x, td.x, 8 * tr_tasks * cap * n, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(trace->g, td.g, 8 * tr_tasks * cap * n, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(trace->f, td.f, 8 * tr_tasks * cap, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(trace->costs, td.costs, 8 * tr_tasks * cap * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(trace->status, td.status, 4 * tr_tasks * cap, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(trace->len, td.len, 4 * tr_tasks, cudaMemcpyDeviceToHost, st));
    }
    const auto t_launched = now();
    CK(cudaStreamSynchronize(st));
    const auto t_done = now();
    CK(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    h->pool.run(b, [&](size_t i0, size_t i1) {
        const size_t c = i1 - i0;
        memcpy(out->x + i0 * n, hbase + L.x + 8 * i0 * n, 8 * c * n);
        memcpy(out->ts + i0 * M, hbase + L.ts + 8 * i0 * M, 8 * c * M);
        memcpy(out->coeffs + i0 * N2, hbase + L.coeffs + 8 * i0 * N2, 8 * c * N2);
        memcpy(out->costs + i0 * 4, hbase + L.costs + 32 * i0, 32 * c);
        memcpy(out->status + i0, hbase + L.status + 4 * i0, 4 * c);
        memcpy(out->ok + i0, hbase + L.ok + 4 * i0, 4 * c);
        memcpy(out->attempt + i0, hbase + L.attempt + 4 * i0, 4 * c);
        memcpy(out->nit + i0, hbase + L.nit + 4 * i0, 4 * c);
        memcpy(out->runs + i0, hbase + L.runs + 4 * i0, 4 * c);
        memcpy(out->nfev + i0, hbase + L.nfev + 4 * i0, 4 * c);
        if (out->work) memcpy(out->work + i0 * 4, hbase + L.work + 32 * i0, 32 * c);
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
extern "C" int neo_get_coeffs(neo_handle *h, int B, int M, const double *q, const double *ts, const double *head,
                              const double *tail, double *coeffs)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (B < 0 || M < 2 || M > NEO_MAX_PIECES) return fail(h, "neo_get_coeffs: B or M out of range");
    if (!q || !ts || !head || !tail || !coeffs) return fail(h, "neo_get_coeffs: null pointer");
    if (B == 0) return NEO_OK;
    CK(cudaSetDevice(h->device));
    const size_t nq = 2 * (M - 1), N2 = 12 * M, b = B;
    int rc;
    for (int pass = 0; pass < 2; pass++) {
        Carver c{pass ? (char *)h->bufs[4].p : nullptr};
        double *d_q = c.take<double>(b * nq), *d_ts = c.take<double>(b * M), *d_head = c.take<double>(b * 6),
               *d_tail = c.take<double>(b * 6), *d_c = c.take<double>(b * N2);
        if (!pass) {
            void *p;
            if ((rc = dev_buf(h, 4, c.off + 256, &p))) return rc;
            continue;
        }
        cudaStream_t st = h->stream;
        CK(cudaMemcpyAsync(d_q, q, sizeof(double) * b * nq, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_ts, ts, sizeof(double) * b * M, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_head, head, sizeof(double) * b * 6, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_tail, tail, sizeof(double) * b * 6, cudaMemcpyHostToDevice, st));
        int occ;
        if ((rc = prep_kernel(h, k_coeffs, smem_bytes(M), &occ))) return rc;
        const int need = (B + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
        const int grid = need < occ * h->sm_count ? need : occ * h->sm_count;
        k_coeffs<<<grid, WARPS_PER_CTA * 32, smem_bytes(M), st>>>(B, M, d_q, d_ts, d_head, d_tail, d_c);
        h->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(coeffs, d_c, sizeof(double) * b * N2, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return NEO_OK;
}

extern "C" int neo_sample(neo_handle *h, int B, int M, const double *coeffs, const double *ts, double hz, int max_samples,
                          double *states, int32_t *count)
{
    if (!h) return NEO_ERR_INVALID;
    std::lock_guard<std::mutex> g(h->mu);
    if (B < 0 || M < 1 || M > 64 || !(hz > 0.0)) return fail(h, "neo_sample: invalid argument");
    if (!coeffs || !ts || !count || (states && max_samples < 1)) return fail(h, "neo_sample: null pointer");
    if (B == 0) return NEO_OK;
    CK(cudaSetDevice(h->device));
    const size_t N2 = 12 * M, b = B, ms = states ? max_samples : 0;
    int rc;
    for (int pass = 0; pass < 2; pass++) {
        Carver c{pass ? (char *)h->bufs[4].p : nullptr};
        double *d_c = c.take<double>(b * N2), *d_ts = c.take<double>(b * M), *d_s = c.take<double>(b * ms * 6 + 1);
        int32_t *d_cnt = c.take<int32_t>(b);
        if (!pass) {
            void *p;
            if ((rc = dev_buf(h, 4, c.off + 256, &p))) return rc;
            continue;
        }
        cudaStream_t st = h->stream;
        CK(cudaMemcpyAsync(d_c, coeffs, sizeof(double) * b * N2, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_ts, ts, sizeof(double) * b * M, cudaMemcpyHostToDevice, st));
        if (states) CK(cudaMemcpyAsync(d_s, states, sizeof(double) * b * ms * 6, cudaMemcpyHostToDevice, st));
        dim3 grid(states ? (max_samples + 127) / 128 : 1, B < 65535 ? B : 65535);
        k_sample<<<grid, 128, 0, st>>>(B, M, d_c, d_ts, hz, max_samples, states ? d_s : nullptr, d_cnt);
        h->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(count, d_cnt, sizeof(int32_t) * b, cudaMemcpyDeviceToHost, st));
        if (states) CK(cudaMemcpyAsync(states, d_s, sizeof(double) * b * ms * 6, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (states) for (size_t i = 0; i < b; i++) if (count[i] > max_samples) return fail(h, "neo_sample: max_samples too small");
    }
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
    int rc;
    int32_t *overflow;
    if ((rc = dev_buf(h, 9, sizeof(int32_t) * (size_t)B + 256, (void **)&overflow))) return rc;
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
    a.overflow = overflow;
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
    if (rc) return rc;
    if (B == 0) return NEO_OK;
    for (int i = 0; i < 2 * B; i++)
        if (!isfinite(start[i]) || !isfinite(target[i])) return fail(h, "neo_astar: start/target must be finite");
    if (map_ids)
        for (int i = 0; i < B; i++)
            if (map_ids[i] < 0 || map_ids[i] >= (int)h->slots.size() || !h->slots[map_ids[i]].cells)
                return fail(h, "neo_astar: map id refers to an empty slot");
    if (!map_ids && !h->slots[0].cells) return fail(h, "neo_astar: slot 0 is empty");
    CK(cudaSetDevice(h->device));
    const size_t b = B, np = path ? (size_t)max_path : 0;
    for (int pass = 0; pass < 2; pass++) {
        Carver c{pass ? (char *)h->bufs[7].p : nullptr};
        double *d_s = c.take<double>(2 * b), *d_t = c.take<double>(2 * b), *d_pr = c.take<double>(8 * b),
               *d_path = c.take<double>(2 * b * np + 1);
        int32_t *d_ids = c.take<int32_t>(b), *d_len = c.take<int32_t>(b), *d_st = c.take<int32_t>(b),
                *d_cl = c.take<int32_t>(b);
        if (!pass) {
            void *p;
            if ((rc = dev_buf(h, 7, c.off + 256, &p))) return rc;
            continue;
        }
        cudaStream_t st = h->stream;
        CK(cudaMemcpyAsync(d_s, start, sizeof(double) * 2 * b, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_t, target, sizeof(double) * 2 * b, cudaMemcpyHostToDevice, st));
        if (map_ids) CK(cudaMemcpyAsync(d_ids, map_ids, sizeof(int32_t) * b, cudaMemcpyHostToDevice, st));
        CK(cudaEventRecord(h->ev0, st));
        rc = astar_launch(h, B, d_s, d_t, map_ids ? d_ids : nullptr, max_closed, max_path, path ? d_path : nullptr, d_len,
                          d_pr, d_st, d_cl, st);
        if (rc) return rc;
        CK(cudaEventRecord(h->ev1, st));
        CK(cudaMemcpyAsync(path_len, d_len, sizeof(int32_t) * b, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(status, d_st, sizeof(int32_t) * b, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(closed, d_cl, sizeof(int32_t) * b, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(pruned, d_pr, sizeof(double) * 8 * b, cudaMemcpyDeviceToHost, st));
        if (path) CK(cudaMemcpyAsync(path, d_path, sizeof(double) * 2 * b * np, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    }
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
    double *d;
    int rc = dev_buf(h, 5, sizeof(double) * threads * blocks, (void **)&d);
    if (rc) return rc;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CK(cudaEventRecord(h->ev0, h->stream));
        k_fp64_peak<<<blocks, threads, 0, h->stream>>>(d, iters);
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
    double *d;
    int rc = dev_buf(h, 5, sizeof(double) * 2 * n, (void **)&d);
    if (rc) return rc;
    CK(cudaMemcpyAsync(d, x, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    k_exp_dd<<<(n + 255) / 256, 256, 0, h->stream>>>(n, d, d + n);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(y, d + n, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return NEO_OK;
}

// test hooks: the optimizer's dnrm2 (x87_nrm2.h) and its two inner products as the device build computes them
static int test_blas_prims(neo_handle *h, int count, int n, const double *a, const double *b, double *out)
{
    std::lock_guard<std::mutex> g(h->mu);
    if (count == 0 || n == 0) { for (size_t i = 0; i < 3 * (size_t)count; i++) out[i] = 0.0; return NEO_OK; }
    CK(cudaSetDevice(h->device));
    double *d;
    const size_t len = (size_t)count * n;
    int rc = dev_buf(h, 5, sizeof(double) * (2 * len + 3 * (size_t)count), (void **)&d);
    if (rc) return rc;
    CK(cudaMemcpyAsync(d, a, sizeof(double) * len, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d + len, b ? b : a, sizeof(double) * len, cudaMemcpyHostToDevice, h->stream));
    launch_blas_prims(count, n, d, d + len, d + 2 * len, h->stream);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d + 2 * len, sizeof(double) * 3 * count, cudaMemcpyDeviceToHost, h->stream));
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

#ifdef NEO_ROUND_TRACE
extern "C" int neo_test_round_trace(long long *out)
{
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_round_trace, sizeof(long long) * 12 * 2048 * 4);
    return NEO_OK;
}
#endif

#ifdef NEO_OPT_TICKS
// development probe: read and clear the optimizer's phase counters (cycles [0..32), calls [32..64))
extern "C" int neo_test_opt_ticks(long long *out)
{
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_opt_ticks, sizeof(long long) * 64);
    long long z[64] = {0};
    cudaMemcpyToSymbol(g_opt_ticks, z, sizeof(z));
    return NEO_OK;
}
#endif

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
