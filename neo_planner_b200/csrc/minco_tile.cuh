// minco_tile.cuh -- one TILE of TL lanes (8, 16 or 32; TL >= 2M and TL >= n) = one planning problem: fused get_cost + get_grad of the reference optimizer
// (EP:539-585) in fp64 on sm_100a.
//
// The reference solves the dense 6M x 6M MINCO system A c = b (EP:261-336, numpy.linalg.solve) and its transpose
// A^T G = dW/dc (EP:503). Here both are replaced by their exact node-state ("Hermite") reduction:
//   * each quintic piece is written in terms of its boundary states (p, v, a at both ends) in closed form;
//   * the only unknowns are (v_j, a_j) at the M-1 interior waypoints, fixed by jerk/snap continuity: a block-
//     tridiagonal system K u = r with 2x2 blocks, solved by block elimination (M-1 sequential 2x2 steps);
//   * the adjoint variable G = A^-T dW/dc = dW/db is recovered row by row from the multipliers of K (jerk/snap rows),
//     the boundary-state gradients h_i = H(T_i)^T dW/dc_i and closed-form sensitivities (pos/vel/acc rows, q rows,
//     tail rows), and then fed into the reference's own formulas for grad_q and grad_T (EP:506-533) -- including its
//     re-use of T = ts[M-2] for the last piece.
// This is algebraically identical to the reference (verified to ~1e-13 against numpy in scratch prototypes and to
// <= 1e-12 in tests/test_gpu_parity.py) and turns ~6M sequential pivots into M-1 sequential 2x2 blocks.
//
// A warp holds 32/TL tiles; every shuffle, vote and barrier below names only the tile's own lanes (Tile::mask), so the
// tiles of a warp are independent problems that merely share an instruction stream.
//   tau -> T (EP:477-483, double-double exp)                       lanes 0..M-1
//   node blocks, right-hand sides                                   lanes 1..M-1 (one interior node each)
//   block elimination / back substitution                           lanes 0,1 (one per dimension)
//   Hermite coefficients, energy cost+gradient (EP:345-390)          lanes 0..2M-1 (piece, dimension)
//   sampled feasibility + collision penalties (EP:392-466)           all lanes over samples, ESDF cells from L1/L2,
//                                                                    per-lane partial sums added per (piece, slot) in
//                                                                    lane order through shared memory (no shuffles)
//   adjoint, grad_q, grad_T, grad_tau (EP:485-537)                   lanes (node, dimension) / lanes 0..M-1
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "dd_exp.h"

namespace neo {
constexpr unsigned FULL = 0xffffffffu;

constexpr int HIST = 10;        // L-BFGS memory (maxcor, EP:220)
constexpr int LBW = 2 * HIST;   // order of the middle matrix of the compact representation
constexpr int WN_DOUBLES = LBW * (LBW + 1) / 2 + 2 * LBW + 2;    // packed upper triangle + the subspace vector wv + 1/diagonal

struct DevParams {
    double v_max2, T_min, T_max, safe_dis, dt;
    double w0, w1, w2, w3;
    double collision_cost_tol;
};

// One ESDF cell = one 32-byte L2 sector: {grad_x, grad_y, dist, pad}
struct __align__(32) Cell {
    double gx, gy, d, pad;
};

struct MapView {
    const Cell *cells;
    int H, W;
    double res, ox, oy;
    double inv_res;
    const unsigned char *blocked;   // astar_warp.cuh: has_collision at every node of the enlarged search grid (1 = blocked)
};

// The TL lanes that work on one problem.
template <int TL>
struct Tile {
    int tl;            // lane within the tile
    unsigned mask;     // the tile's lanes within the warp
    int base;          // first lane of the tile
    __device__ __forceinline__ explicit Tile(int lane)
        : tl(lane & (TL - 1)), mask(TL == 32 ? FULL : (((1u << (TL & 31)) - 1u) << (lane & ~(TL - 1)))), base(lane & ~(TL - 1)) {}
    __device__ __forceinline__ void sync() const { __syncwarp(mask); }
    __device__ __forceinline__ double shfl(double v, int src) const { return __shfl_sync(mask, v, src, TL); }
    __device__ __forceinline__ int shfl(int v, int src) const { return __shfl_sync(mask, v, src, TL); }
    __device__ __forceinline__ unsigned shfl(unsigned v, int src) const { return __shfl_sync(mask, v, src, TL); }
    __device__ __forceinline__ bool all(bool p) const { return __all_sync(mask, p); }
    __device__ __forceinline__ bool any(bool p) const { return __any_sync(mask, p); }
    __device__ __forceinline__ int rmax(int v) const { return __reduce_max_sync(mask, v); }
    __device__ __forceinline__ unsigned radd(unsigned v) const { return __reduce_add_sync(mask, v); }
    __device__ __forceinline__ double dmax(double v) const
    {
#pragma unroll
        for (int o = TL / 2; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(mask, v, o, TL));
        return v;
    }
};

// Per-tile shared-memory slice (all doubles). n = 3M-2 decision variables.
struct TileMem {
    double *ts;    // [M]
    double *ex;    // [M]      exp(-tau)
    double *iT;    // [M][5]   1/T, 1/T^2, ... 1/T^5
    double *gT;    // [M]
    double *P;     // [M+1][2] node positions: head, q_0..q_{M-2}, tail
    double *U;     // [M+1][4] node (v_x, v_y, a_x, a_y)
    double *blk;   // [M+1][12] per interior node: L (4), D -> D'^-1 (4), U (4), row-major 2x2
    double *r;     // [M+1][4] rhs / eta, then r' / eta' : (row0_x, row0_y, row1_x, row1_y)
    double *lam;   // [M+1][4] multipliers (jerk_x, jerk_y, snap_x, snap_y)
    double *c;     // [6M][2]  polynomial coefficients
    double *gC;    // [6M][2]  dW/dc
    double *h;     // [M][12]  dW/d(boundary state): (ps, vs, as, pe, ve, ae) x (x, y)
    double *Gs;    // [M+1][10] per interior node: (Gq+Gp, Gv, Ga, lamJ, lamS) x (x, y)
    double *e0;    // [2M]     energy per (piece, dim)
    double *nsd;   // [M][2]   sample count of the piece (as double) and its reciprocal
    double *gout;  // [n]      gradient staging
    double *ht;    // [12]     head (3,2), tail (3,2)
    double *pc;    // [M][2]   per-piece feasibility / collision cost
    // optimizer (lbfgsb_tile.cuh): the limited-memory pairs, oldest first, and the inner products formk keeps
    double *ws;    // [HIST][n]  s pairs, ring: pair k lives in row (head + k) % HIST
    double *wy;    // [HIST][n]  y pairs
    double *yr;    // [HIST][HIST] by ring slots: [newer][older] = y_newer . y_older (formk's Y'Y), [older][newer] =
                   //          s_older . y_newer (formk's R_z, the upper triangle of S'Y), [a][a] = y_a . y_a
    double *rzd;   // [HIST]   s_a . y_a as formk computes it (its own inner product, not matupd's dr)
    double *dr;    // [HIST]   diagonal of S'Y as matupd stores it ((gd - gdold) * stp), by ring slot
    double *gv;    // [n]      g and d as vectors every lane can read (sequential inner products)
    double *dv;    // [n]
    double *ls;    // [16]     line-search state (Dcsrch) between evaluations, f and g'd at the start of the search
    double *oc;    // [7]      costs at the last evaluated point (4), work counters samples / violating / colliding (3)
    // one region, two users: per-lane partial sums of the sample loop (evaluation) / the factored middle matrix (direction)
    double *red;   // [15 or 15*M][TL+1] per-lane partial sums of the sample loop (padded rows)
    double *wn;    // [LBW(LBW+1)/2] packed upper triangle, column j at j(j+1)/2; then wv [LBW]
    double *lw;    // [M][2]   first lane and lane count of each piece (SAMPLE_ALL_PIECES)
    double *nsprev; // [M]     sample counts the cached lane assignment was computed for (-1: none)
    double *asg;   // [32]     cached lane assignment: piece + 16 * width + 1024 * rank
};

// Schedules of the evaluator's sample loop (eval_fg). The piece count and the tile width fix which one runs, and the
// tile's shared-memory layout below depends on it: sample_schedule is the one place that decides.
constexpr int SAMPLE_BY_PIECE = 0;          // M <= 4, one problem per warp
constexpr int SAMPLE_ALL_PIECES = 1;        // M >= 5 (always 32 lanes)
constexpr int SAMPLE_BY_PIECE_STAGED = 2;   // M <= 4, tiles narrower than a warp: one staging block, reduced after every
                                            // piece (4 KB instead of 4 M KB of shared memory per warp -> more L1 for the map)
__host__ __device__ constexpr int sample_schedule(int M, int TL)
{
    return M > 4 ? SAMPLE_ALL_PIECES : (TL < 32 ? SAMPLE_BY_PIECE_STAGED : SAMPLE_BY_PIECE);
}

// staging rows of the sample loop's partial sums: one block of 15 rows per piece when all pieces are parked before the
// owners add them (by-piece schedule, latency-optimised), one block otherwise (see eval_fg)
// rows are padded to TL + 1 for a full warp (conflict-free owner reads); narrow tiles are not padded (their shared memory
// decides how many problems an SM holds)
__host__ __device__ constexpr int red_stride(int TL) { return TL == 32 ? 33 : TL; }
// (the one-block schedules are named rather than tested as != SAMPLE_BY_PIECE: for k_coeffs, whose M is not a constant,
// the compiler then shares one M > 4 test with lane_cache_doubles)
__host__ __device__ inline int red_doubles(int M, int TL)
{
    const int s = sample_schedule(M, TL);
    return (s == SAMPLE_ALL_PIECES || s == SAMPLE_BY_PIECE_STAGED) ? 15 * red_stride(TL) : 15 * red_stride(TL) * M;
}
// the all-pieces schedule's cached lane assignment: lw [2M], nsprev [M], asg [32]
__host__ __device__ inline int lane_cache_doubles(int M, int TL)
{
    return sample_schedule(M, TL) == SAMPLE_ALL_PIECES ? 2 * M + M + 32 : 0;
}

// Layout of a tile's slice. Shared memory is what limits the number of problems in flight per SM, so regions whose
// lifetimes do not overlap share storage:
//   [ht]                                     head / tail states: live for the whole problem
//   [A: ts ex iT gT P U blk c gC e0 nsd gout pc]   evaluation scratch, rewritten by every evaluation
//   [B: red  |  r lam h Gs]                  the sample loop's partial sums, then (same storage) the adjoint's vectors;
//                                            r is also used by the node solve, before the sample loop starts
//   A and B together hold the factored middle matrix wn + wv + 1/diagonal while a search direction is computed
//   (no evaluation is in flight then)
//   [ws wy yr rzd dr] [gv dv]                optimizer state: live across evaluations
//   [lw nsprev asg]                          cached lane assignment of the all-pieces schedule (M > 4)
__host__ __device__ inline int scratch_a_doubles(int M)
{
    const int n = 3 * M - 2, M1 = M + 1;
    return M + M + 5 * M + M + 2 * M1 + 4 * M1 + 12 * (M - 1) + 12 * M + 12 * M + 2 * M + 2 * M + n + 2 * M;
}
__host__ __device__ inline int scratch_b_doubles(int M, int TL)
{
    const int M1 = M + 1, adj = 4 * M1 + 4 * M1 + 12 * M + 10 * M1, red = red_doubles(M, TL);
    return red > adj ? red : adj;
}
__host__ __device__ inline int scratch_doubles(int M, int TL)
{
    const int ab = scratch_a_doubles(M) + scratch_b_doubles(M, TL);
    return ab > WN_DOUBLES ? ab : WN_DOUBLES;
}

__host__ __device__ inline int tile_mem_doubles(int M, int TL = 32)
{
    const int n = 3 * M - 2;
    int tot = 12 + scratch_doubles(M, TL) + 2 * HIST * n + HIST * HIST + 2 * HIST + 2 * n + 16 + 7 + lane_cache_doubles(M, TL);
    return (tot + 1) & ~1;
}

// evaluator only (k_eval): no optimizer state behind the scratch regions
__host__ __device__ inline int eval_mem_doubles(int M, int TL)
{
    const int tot = 12 + scratch_a_doubles(M) + scratch_b_doubles(M, TL) + lane_cache_doubles(M, TL);
    return (tot + 1) & ~1;
}

__device__ inline TileMem carve(double *base, int M, int TL = 32, bool eval_only = false)
{
    const int n = 3 * M - 2, M1 = M + 1;
    TileMem m;
    m.ht = base; base += 12;
    double *const scratch = base;
    m.wn = scratch;
    m.ts = base; base += M;
    m.ex = base; base += M;
    m.iT = base; base += 5 * M;
    m.gT = base; base += M;
    m.P = base; base += 2 * M1;
    m.U = base; base += 4 * M1;
    m.blk = base - 12; base += 12 * (M - 1);        // indexed by interior node 1..M-1
    m.c = base; base += 12 * M;
    m.gC = base; base += 12 * M;
    m.e0 = base; base += 2 * M;
    m.nsd = base; base += 2 * M;
    m.gout = base; base += n;
    m.pc = base; base += 2 * M;
    m.red = base;                                   // B: partial sums of the sample loop ...
    m.r = base;                                     // ... or the adjoint's vectors
    m.lam = m.r + 4 * M1;
    m.h = m.lam + 4 * M1;
    m.Gs = m.h + 12 * M;
    if (eval_only) {
        base = scratch + scratch_a_doubles(M) + scratch_b_doubles(M, TL);
        m.ws = m.wy = m.yr = m.rzd = m.dr = m.gv = m.dv = m.ls = m.oc = nullptr;
        m.lw = base; m.nsprev = base + 2 * M; m.asg = base + 3 * M;
        return m;
    }
    base = scratch + scratch_doubles(M, TL);
    m.ws = base; base += HIST * n;
    m.wy = base; base += HIST * n;
    m.yr = base; base += HIST * HIST;
    m.rzd = base; base += HIST;
    m.dr = base; base += HIST;
    m.gv = base; base += n;
    m.dv = base; base += n;
    m.ls = base; base += 16;
    m.oc = base; base += 7;
    m.lw = base; m.nsprev = base + 2 * M; m.asg = base + 3 * M;      // sized by lane_cache_doubles
    return m;
}

// Called when a tile starts on a new problem: head/tail states into shared memory, cached lane assignment dropped.
template <int TL>
__device__ __forceinline__ void begin_problem(const Tile<TL> &T, const TileMem &m, int M, const double *head, const double *tail)
{
    const int lane = T.tl;
    if (lane < 6) { m.ht[lane] = head[lane]; m.ht[6 + lane] = tail[lane]; }
    if (lane < M) {
        if (sample_schedule(M, TL) == SAMPLE_ALL_PIECES) m.nsprev[lane] = -1.0;
        m.pc[2 * lane] = 0.0; m.pc[2 * lane + 1] = 0.0;
    }
    T.sync();
}

// ---------------------------------------------------------------------------------------------------------
// coefficients: tau -> T was done by the caller (m.ts, m.iT); x component xl in lane l
// ---------------------------------------------------------------------------------------------------------

// Writes node positions / boundary (v,a) from the decision vector and the head/tail states.
template <int TL>
__device__ __forceinline__ void load_nodes(const Tile<TL> &T, const TileMem &m, int M, double xl)
{
    const int lane = T.tl;
    const int nq = 2 * (M - 1);
    if (lane < nq) {   // x = [q_x(0..M-2), q_y(0..M-2), tau] (EP:211): node i+1, dim d
        const int d = lane / (M - 1), i = lane - d * (M - 1);
        m.P[2 * (i + 1) + d] = xl;
    }
    if (lane < 2) {    // head / tail rows (EP:274-275): pos, vel, acc
        m.P[lane] = m.ht[lane];
        m.P[2 * M + lane] = m.ht[6 + lane];
        m.U[lane] = m.ht[2 + lane]; m.U[2 + lane] = m.ht[4 + lane];
        m.U[4 * M + lane] = m.ht[8 + lane]; m.U[4 * M + 2 + lane] = m.ht[10 + lane];
    }
    T.sync();
}

// Block-tridiagonal system of the interior nodes (jerk + snap continuity) and its block elimination. Every lane runs
// the M-1 sequential 2x2 steps for dimension d = lane & 1 with the blocks, right-hand sides and the running inverse in
// registers (the blocks depend on 1/T^k only; nothing on the dependent chain goes through shared memory). Leaves
// L, D'^-1, U per node in m.blk (reused by the adjoint) and the node (v, a) in m.U.
template <int TL>
__device__ __forceinline__ void solve_nodes(const Tile<TL> &T, const TileMem &m, int M)
{
    const int lane = T.tl;
    const int d = lane & 1;
    const double *__restrict__ iT = m.iT;
    const double *__restrict__ P = m.P;
    double *__restrict__ blk = m.blk;
    double *__restrict__ rr = m.r;
    double i00 = 0, i01 = 0, i10 = 0, i11 = 0, u00 = 0, u01 = 0, u10 = 0, u11 = 0, p0 = 0, p1 = 0;
    double a = iT[0], a2 = iT[1], a3 = iT[2], a4 = iT[3];
    double pm = P[d], pc = P[2 + d];
    const double hv = m.U[d], ha = m.U[2 + d], tv = m.U[4 * M + d], ta = m.U[4 * M + 2 + d];
    for (int j = 1; j < M; j++) {
        const double b = iT[5 * j], b2 = iT[5 * j + 1], b3 = iT[5 * j + 2], b4 = iT[5 * j + 3];
        const double pn = P[2 * (j + 1) + d];
        const double l00 = -24.0 * a2, l01 = -3.0 * a, l10 = -168.0 * a3, l11 = l00;                      // L_j
        double d00 = 36.0 * (b2 - a2), d01 = 9.0 * (a + b), d10 = -192.0 * (a3 + b3), d11 = -d00;         // D_j
        const double n00 = 24.0 * b2, n01 = -3.0 * b, n10 = -168.0 * b3, n11 = n00;                       // U_j
        const double dm = pc - pm, dp = pn - pc;
        double r0 = 60.0 * (dp * b3 - dm * a3), r1 = -360.0 * (dm * a4 + dp * b4);
        if (j == 1) { r0 -= l00 * hv + l01 * ha; r1 -= l10 * hv + l11 * ha; }          // known (v,a) of the head node
        if (j == M - 1) { r0 -= n00 * tv + n01 * ta; r1 -= n10 * tv + n11 * ta; }      // known (v,a) of the tail node
        if (j > 1) {
            const double w00 = l00 * i00 + l01 * i10, w01 = l00 * i01 + l01 * i11;     // W = L_j D'^-1_{j-1}
            const double w10 = l10 * i00 + l11 * i10, w11 = l10 * i01 + l11 * i11;
            d00 -= w00 * u00 + w01 * u10; d01 -= w00 * u01 + w01 * u11;
            d10 -= w10 * u00 + w11 * u10; d11 -= w10 * u01 + w11 * u11;
            r0 -= w00 * p0 + w01 * p1; r1 -= w10 * p0 + w11 * p1;
        }
        const double idet = 1.0 / (d00 * d11 - d01 * d10);
        i00 = d11 * idet; i01 = -d01 * idet; i10 = -d10 * idet; i11 = d00 * idet;
        if (lane == 0) {
            double *B = blk + 12 * j;
            B[0] = l00; B[1] = l01; B[2] = l10; B[3] = l11;
            B[4] = i00; B[5] = i01; B[6] = i10; B[7] = i11;
            B[8] = n00; B[9] = n01; B[10] = n10; B[11] = n11;
        }
        if (lane < 2) { rr[4 * j + d] = r0; rr[4 * j + 2 + d] = r1; }
        u00 = n00; u01 = n01; u10 = n10; u11 = n11; p0 = r0; p1 = r1;
        a = b; a2 = b2; a3 = b3; a4 = b4; pm = pc; pc = pn;
    }
    T.sync();
    {
        double v = tv, ac = ta;
        for (int j = M - 1; j >= 1; j--) {
            const double *B = blk + 12 * j;
            double r0 = rr[4 * j + d], r1 = rr[4 * j + 2 + d];
            if (j < M - 1) { r0 -= B[8] * v + B[9] * ac; r1 -= B[10] * v + B[11] * ac; }
            v = B[4] * r0 + B[5] * r1; ac = B[6] * r0 + B[7] * r1;
            if (lane < 2) { m.U[4 * j + d] = v; m.U[4 * j + 2 + d] = ac; }
        }
    }
    T.sync();
}

// Quintic coefficients of piece i, dimension d from its boundary states (closed-form Hermite inverse).
template <int TL>
__device__ __forceinline__ void hermite_coeffs(const Tile<TL> &T, const TileMem &m, int M)
{
    const int lane = T.tl;
    if (lane < 2 * M) {
        const int i = lane >> 1, d = lane & 1;
        const double T = m.ts[i], T2 = T * T;
        const double a3 = m.iT[5 * i + 2], a4 = m.iT[5 * i + 3], a5 = m.iT[5 * i + 4];
        const double ps = m.P[2 * i + d], pe = m.P[2 * (i + 1) + d];
        const double vs = m.U[4 * i + d], as = m.U[4 * i + 2 + d], ve = m.U[4 * (i + 1) + d], ae = m.U[4 * (i + 1) + 2 + d];
        const double dl = pe - ps;
        double *c = m.c + 12 * i + d;
        c[0] = ps; c[2] = vs; c[4] = 0.5 * as;
        c[6] = (20.0 * dl - (8.0 * ve + 12.0 * vs) * T - (3.0 * as - ae) * T2) * (0.5 * a3);
        c[8] = (-30.0 * dl + (14.0 * ve + 16.0 * vs) * T + (3.0 * as - 2.0 * ae) * T2) * (0.5 * a4);
        c[10] = (12.0 * dl - 6.0 * (ve + vs) * T - (as - ae) * T2) * (0.5 * a5);
    }
    T.sync();
}

// ---------------------------------------------------------------------------------------------------------
// fused cost + gradient
// ---------------------------------------------------------------------------------------------------------
struct EvalOut {
    double f;          // dot(costs, weights) (EP:558)
    double costs[4];   // unweighted (EP:339)
    double g;          // lane l < n: grad[l] (EP:581)
    int status;        // 0, NEO_ST_OVERFLOW (4) or NEO_ST_NAN (6)
    unsigned ns, nv, nc;   // samples, velocity-violating samples, colliding samples (work accounting)
};

// Exact quotient (p - origin)/res (ESDF:61-62) for the rare sample whose reciprocal estimate lies within 1e-9 of an
// integer; kept out of line so the fp64 division sequence does not sit in the hot loop's instruction stream.
__device__ __noinline__ double exact_quotient(double num, double res) { return num / res; }

// One sample j of one piece (EP:399-466): position/velocity, ESDF lookup, both penalties and their contributions to
// acc[0..11] = dW/dc (slot 2k+d), acc[12] = dW/dT, acc[13] = feasibility cost, acc[14] = collision cost.
// Order of work: position -> cell index -> distance load issued, THEN the velocity polynomial and the feasibility term
// while the load is in flight. Polynomials are evaluated in Estrin form (three independent FMAs, then two dependent
// ones) instead of a six-deep chain (DFMA latency is 12 cycles on this part).
__device__ __forceinline__ void sample_point(const DevParams &P, const MapView &map, const double (&cx)[6],
                                             const double (&cy)[6], int j, int ns, double inv_ns, double (&acc)[16],
                                             EvalOut &out, int &bad)
{
    // The map's size and cell base are read here, with its origin and 1/res, not where they are used: k_optimize passes
    // the map by reference into global memory, and reads after the out-of-line exact_quotient call could not be issued
    // before it, so they would wait for the position and then for each other -- three dependent L1/L2 round trips per
    // sample instead of one ahead of the distance load.
    const Cell *const cells = map.cells;
    const int H = map.H, W = map.W;
    const double t = (double)j * P.dt;               // np.arange(0, T_max, dt)[j] (EP:251)
    const double t2 = t * t, t4 = t2 * t2;
    const double px = fma(t4, fma(cx[5], t, cx[4]), fma(t2, fma(cx[3], t, cx[2]), fma(cx[1], t, cx[0])));
    const double py = fma(t4, fma(cy[5], t, cy[4]), fma(t2, fma(cy[3], t, cy[2]), fma(cy[1], t, cy[0])));
    // collision lookup (EP:415-417): nearest cell, index = int((p - origin)/res), trunc toward zero (ESDF:61-65).
    // The quotient is first formed with the reciprocal (|estimate - exact| <= 4.5e-16 |q| < 1e-9 for every in-map index,
    // |q| < 2^20); the exact IEEE division is only redone when the estimate is within 1e-9 of an integer, so the
    // truncated index is always the reference's.
    const double dy = py - map.oy, dx = px - map.ox;
    double fr = dy * map.inv_res, fc = dx * map.inv_res;
    double tr = trunc(fr), tc = trunc(fc);
    {
        const double er = fabs(fr - tr), ec = fabs(fc - tc);
        if (er < 1e-9 || er > 1.0 - 1e-9) { fr = exact_quotient(dy, map.res); tr = trunc(fr); }
        if (ec < 1e-9 || ec > 1.0 - 1e-9) { fc = exact_quotient(dx, map.res); tc = trunc(fc); }
    }
    if (fr != fr || fc != fc) bad = 6;                 // int(nan) raises ValueError
    const bool inside = tr >= 0.0 && tr < (double)H && tc >= 0.0 && tc < (double)W;
    double dis = 10000.0;
    const Cell *cell = cells;
    if (inside) {
        cell = cells + ((size_t)(int)tr * W + (int)tc);
        dis = __ldg(&cell->d);
    }
    const double t3 = t2 * t;
    const double b1[6] = {0.0, 1.0, 2.0 * t, 3.0 * t2, 4.0 * t3, 5.0 * t4};
    const double vx = fma(b1[5], cx[5], fma(b1[4], cx[4], cx[1])) + fma(b1[3], cx[3], b1[2] * cx[2]);
    const double vy = fma(b1[5], cy[5], fma(b1[4], cy[4], cy[1])) + fma(b1[3], cy[3], b1[2] * cy[2]);
    const double omg = (j == 0 || j == ns - 1) ? 0.5 : 1.0;   // EP:407
    const double vv = (vx * vx + vy * vy) - P.v_max2;
    out.ns++;
    if (vv > 0.0) {       // feasibility (EP:409-413, EP:441-451)
        const double vv2 = vv * vv, vv3 = vv2 * vv;
        acc[13] += (omg * P.dt) * vv3;
        const double K = (3.0 * P.dt * omg) * vv2;
        const double ax = fma(20.0 * t3, cx[5], 12.0 * t2 * cx[4]) + fma(6.0 * t, cx[3], 2.0 * cx[2]);
        const double ay = fma(20.0 * t3, cy[5], 12.0 * t2 * cy[4]) + fma(6.0 * t, cy[3], 2.0 * cy[2]);
        const double v2t = 2.0 * (ax * vx + ay * vy);
        const double kx = (P.w2 * K) * (2.0 * vx), ky = (P.w2 * K) * (2.0 * vy);
#pragma unroll
        for (int k = 1; k < 6; k++) { acc[2 * k] += b1[k] * kx; acc[2 * k + 1] += b1[k] * ky; }
        acc[12] += P.w2 * ((omg * vv3 + K * v2t * (double)j) * inv_ns);
        out.nv++;
    }
    const double vd = P.safe_dis - dis;
    if (vd > 0.0) {       // collision (EP:418-422, EP:453-466); outside the map dis = 10000 never violates
        const double vd2 = vd * vd, vd3 = vd2 * vd;
        acc[14] += (omg * P.dt) * vd3;
        const double2 g = __ldg(reinterpret_cast<const double2 *>(cell));
        const double K = (3.0 * P.dt * omg) * vd2;
        const double p2t = -(g.x * vx + g.y * vy);
        const double kx = -(P.w3 * K) * g.x, ky = -(P.w3 * K) * g.y;
        const double t5 = t4 * t;
        const double b0[6] = {1.0, t, t2, t3, t4, t5};
#pragma unroll
        for (int k = 0; k < 6; k++) { acc[2 * k] += b0[k] * kx; acc[2 * k + 1] += b0[k] * ky; }
        acc[12] += P.w3 * ((omg * vd3 + K * p2t * (double)j) * inv_ns);
        out.nc++;
    }
}

// tau -> T for all pieces; returns 0 or the status the reference's exception maps to. Also fills 1/T^k.
template <int TL>
__device__ __forceinline__ int times_from_tau(const Tile<TL> &T, const DevParams &P, const TileMem &m, int M, double xl,
                                              double &e_out)
{
    const int lane = T.tl;
    const int nq = 2 * (M - 1);
    const double tau = T.shfl(xl, (nq + lane) & (TL - 1));
    int bad = 0;
    double e = 0.0;
    if (lane < M) {
        bool ovf;
        e = exp_dd(-tau, &ovf);                               // math.exp(-tau) (EP:481)
        const double den = (1.0 + e) * (1.0 + e);             // (1+exp(-tau))**2 raises OverflowError (EP:490)
        if (ovf || den == INFINITY) bad = 4;
        const double T = (P.T_max - P.T_min) / (1.0 + e) + P.T_min;
        if (T != T) bad = 6;                                  // int(nan) raises ValueError (EP:401)
        m.ts[lane] = T;
        m.ex[lane] = e;
        const double a = 1.0 / T, a2 = a * a;
        double *it = m.iT + 5 * lane;
        it[0] = a; it[1] = a2; it[2] = a2 * a; it[3] = a2 * a2; it[4] = a2 * a2 * a;
        const int ns = (int)(T / P.dt);                       // sample_num = int(T/delta_t) (EP:401)
        m.nsd[2 * lane] = (double)ns;
        m.nsd[2 * lane + 1] = 1.0 / (double)ns;
        m.pc[2 * lane] = 0.0; m.pc[2 * lane + 1] = 0.0;        // a piece without samples contributes no penalty
    }
    e_out = e;
    bad = T.rmax(bad);
    T.sync();
    return bad;
}

// COLD: the map cells this evaluation reads are probably not in L2 (a one-shot evaluation of many problems, k_eval):
// before the sample loop every lane walks its samples once, forming only position -> cell address, and issues an L2
// prefetch for each, so that the misses overlap instead of being taken one per loop trip (k_eval is bound by exactly
// that latency: long-scoreboard stalls 43 %). The optimizer's evaluations re-read the same cells ~70 times: not worth it.
// MC: the piece count the kernel is compiled for (M == MC); with TL it fixes the sampling schedule.
template <int MC, int TL, bool COLD = false>
__device__ __forceinline__ void eval_fg(const Tile<TL> &T, const DevParams &P, const MapView &map, const TileMem &m, int M,
                                        double xl, EvalOut &out)
{
    static_assert(TL == 32 || MC <= 4, "the all-pieces schedule (M > 4) assigns the 32 lanes of a warp");
    constexpr int SCHEDULE = sample_schedule(MC, TL);
    const int lane = T.tl;
    const int nq = 2 * (M - 1);
    out.status = 0; out.ns = out.nv = out.nc = 0;
    out.g = 0.0;

    double e;
    int bad = times_from_tau(T, P, m, M, xl, e);
    if (bad) { out.status = bad; out.f = 0.0; out.costs[0] = out.costs[1] = out.costs[2] = out.costs[3] = 0.0; return; }

    // ---- coefficients (EP:261-336) ----------------------------------------------------------------
    load_nodes(T, m, M, xl);
    solve_nodes(T, m, M);
    hermite_coeffs(T, m, M);

    // ---- energy + time (EP:345-390): lane (piece i, dim d) -------------------------------------------
    if (lane < 2 * M) {
        const int i = lane >> 1, d = lane & 1;
        const double Ti = m.ts[i], T2 = Ti * Ti, T3 = T2 * Ti, T4 = T3 * Ti, T5 = T4 * Ti;
        const double *ci = m.c + 12 * i + d;
        const double c3 = ci[6], c4 = ci[8], c5 = ci[10];
        const double r3 = 36.0 * Ti * c3 + 72.0 * T2 * c4 + 120.0 * T3 * c5;     // rows of beta3_mat @ c
        const double r4 = 72.0 * T2 * c3 + 192.0 * T3 * c4 + 360.0 * T4 * c5;
        const double r5 = 120.0 * T3 * c3 + 360.0 * T4 * c4 + 720.0 * T5 * c5;
        m.e0[lane] = c3 * r3 + c4 * r4 + c5 * r5;
        double *g = m.gC + 12 * i + d;
        g[0] = 0.0; g[2] = 0.0; g[4] = 0.0;
        g[6] = (P.w0 * 2.0) * r3; g[8] = (P.w0 * 2.0) * r4; g[10] = (P.w0 * 2.0) * r5;
        const double jend = 6.0 * c3 + 24.0 * Ti * c4 + 60.0 * T2 * c5;         // jerk at the piece end
        const double je2 = P.w0 * (jend * jend);
        const double other = __shfl_xor_sync(((1u << (2 * M)) - 1u) << T.base, je2, 1, TL);
        if (d == 0) m.gT[i] = (je2 + other) + P.w1;
    }
    T.sync();
    double costs0 = 0.0, costs1 = 0.0;
    for (int i = 0; i < M; i++) {          // sequential, like the reference's loops / np.sum
        costs0 += m.e0[2 * i] + m.e0[2 * i + 1];
        costs1 += m.ts[i];
    }

    if constexpr (COLD) {
        for (int i = 0; i < M; i++) {
            const int ns = (int)m.nsd[2 * i];
            const double *ci = m.c + 12 * i;
            double cx[6], cy[6];
#pragma unroll
            for (int k = 0; k < 6; k++) { cx[k] = ci[2 * k]; cy[k] = ci[2 * k + 1]; }
            for (int j = lane; j < ns; j += TL) {
                const double t = (double)j * P.dt, t2 = t * t, t4 = t2 * t2;
                const double px = fma(t4, fma(cx[5], t, cx[4]), fma(t2, fma(cx[3], t, cx[2]), fma(cx[1], t, cx[0])));
                const double py = fma(t4, fma(cy[5], t, cy[4]), fma(t2, fma(cy[3], t, cy[2]), fma(cy[1], t, cy[0])));
                const double tr = trunc((py - map.oy) * map.inv_res), tc = trunc((px - map.ox) * map.inv_res);
                if (tr >= 0.0 && tr < (double)map.H && tc >= 0.0 && tc < (double)map.W)      // a hint: no exact-index fix-up
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(map.cells + ((size_t)(int)tr * map.W + (int)tc)));
            }
        }
    }
    // ---- sampled penalties (EP:392-466) -----------------------------------------------------------------
    double costs2 = 0.0, costs3 = 0.0;
    if constexpr (SCHEDULE == SAMPLE_BY_PIECE || SCHEDULE == SAMPLE_BY_PIECE_STAGED) {
        // few pieces (M <= 4): one piece at a time, lanes over its samples; every lane parks its 15 partial sums of the
        // piece in shared memory (row = (piece, slot), padded to TL + 1 so that the owners below read conflict-free).
        // Owner (piece, slot) adds the TL per-lane partial sums in lane order (four interleaved chains): uniform trip
        // counts, no shuffles, deterministic. SAMPLE_BY_PIECE parks all pieces first and lets 15 M owners work at once
        // (shortest dependent chain); SAMPLE_BY_PIECE_STAGED re-uses one block and reduces after every piece (same
        // additions in the same order, a third of the shared memory).
        constexpr bool STAGED = SCHEDULE == SAMPLE_BY_PIECE_STAGED;
#pragma unroll 1
        for (int i = 0; i < M; i++) {            // not unrolled: ONE copy of the sample body in the instruction stream
            const int ns = (int)m.nsd[2 * i];                    // int(T/delta_t) (EP:401)
            const double inv_ns = m.nsd[2 * i + 1];
            const double *ci = m.c + 12 * i;
            double cx[6], cy[6];
#pragma unroll
            for (int k = 0; k < 6; k++) { cx[k] = ci[2 * k]; cy[k] = ci[2 * k + 1]; }
            double acc[16];
#pragma unroll
            for (int s2 = 0; s2 < 16; s2++) acc[s2] = 0.0;
            for (int j = lane; j < ns; j += TL) sample_point(P, map, cx, cy, j, ns, inv_ns, acc, out, bad);
            double *row = m.red + (STAGED ? 0 : 15 * i) * red_stride(TL) + lane;
#pragma unroll
            for (int s2 = 0; s2 < 15; s2++) row[s2 * red_stride(TL)] = acc[s2];
            if (STAGED) {
                T.sync();
                for (int o = lane; o < 15; o += TL) {
                    const double *p = m.red + o * red_stride(TL);
                    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
                    for (int k = 0; k < TL; k += 4) { a0 += p[k]; a1 += p[k + 1]; a2 += p[k + 2]; a3 += p[k + 3]; }
                    const double tot = (a0 + a1) + (a2 + a3);
                    if (o < 12) m.gC[12 * i + o] += tot;
                    else if (o == 12) m.gT[i] += tot;
                    else m.pc[2 * i + (o - 13)] = tot;
                }
                T.sync();
            }
        }
        if (!STAGED) {
            T.sync();
            for (int o = lane; o < 15 * M; o += TL) {
                const double *p = m.red + o * red_stride(TL);
                double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
                for (int k = 0; k < TL; k += 4) { a0 += p[k]; a1 += p[k + 1]; a2 += p[k + 2]; a3 += p[k + 3]; }
                const double tot = (a0 + a1) + (a2 + a3);
                const int i = o / 15, s2 = o - 15 * i;
                if (s2 < 12) m.gC[12 * i + s2] += tot;
                else if (s2 == 12) m.gT[i] += tot;
                else m.pc[2 * i + (s2 - 13)] = tot;
            }
            T.sync();
        }
        for (int i = 0; i < M; i++) { costs2 += m.pc[2 * i]; costs3 += m.pc[2 * i + 1]; }
    } else {
        // many pieces: the 32 lanes are split among the pieces in proportion to their sample counts (every piece with
        // samples gets at least one lane), so a lane only ever accumulates for ONE piece and all pieces are sampled
        // concurrently: ceil(S/32) rounds instead of sum_i ceil(ns_i/32). Per-lane partial sums go to shared memory
        // and are added per (piece, slot) in a fixed lane order.
        int my_piece = 0, my_rank = 0, my_width = 1;
        const double ns_mine = lane < M ? m.nsd[2 * lane] : 0.0;
        if (__any_sync(FULL, lane < M && ns_mine != m.nsprev[lane])) {
            // (re)assign lanes -- only when a sample count changed since the previous evaluation of this problem.
            // lane i < M owns piece i: every non-empty piece gets one lane up front, the remaining lanes are split in
            // proportion to the cumulative sample counts; boundaries hi_i, piece of a lane = #boundaries <= lane.
            const int ns_i = (int)ns_mine;
            int cum = ns_i, nonempty = ns_i > 0 ? 1 : 0;
#pragma unroll
            for (int o = 1; o < 16; o <<= 1) {                  // inclusive scans over lanes 0..M-1 (M <= 10 < 16)
                const int c2 = __shfl_up_sync(FULL, cum, o), n2 = __shfl_up_sync(FULL, nonempty, o);
                if (lane >= o) { cum += c2; nonempty += n2; }
            }
            const int S = __shfl_sync(FULL, cum, M - 1), pieces = __shfl_sync(FULL, nonempty, M - 1);
            int hi = 0;
            if (lane < M && S > 0) hi = nonempty + (int)floor((double)((32 - pieces) * cum) / (double)S);
            int lo = __shfl_up_sync(FULL, hi, 1);
            if (lane == 0) lo = 0;
            if (lane < M) { m.lw[2 * lane] = (double)lo; m.lw[2 * lane + 1] = (double)(hi - lo); m.nsprev[lane] = ns_mine; }
            for (int i = 0; i < M; i++) my_piece += lane >= __shfl_sync(FULL, hi, i) ? 1 : 0;
            if (my_piece >= M || S == 0) { my_piece = 0; my_rank = 1 << 20; }       // no samples at all: idle lane
            else {
                const int plo = __shfl_sync(FULL, lo, my_piece), phi = __shfl_sync(FULL, hi, my_piece);
                my_rank = lane - plo; my_width = phi - plo;
            }
            m.asg[lane] = (double)(my_piece + 16 * my_width + 1024 * my_rank);
            T.sync();
        } else {
            const int v = (int)m.asg[lane];
            my_piece = v & 15; my_width = (v >> 4) & 63; my_rank = v >> 10;
        }
        {
            const int i = my_piece;
            const int ns = (int)m.nsd[2 * i];
            const double inv_ns = m.nsd[2 * i + 1];
            const double *ci = m.c + 12 * i;
            double cx[6], cy[6];
#pragma unroll
            for (int k = 0; k < 6; k++) { cx[k] = ci[2 * k]; cy[k] = ci[2 * k + 1]; }
            double acc[16];
#pragma unroll
            for (int s2 = 0; s2 < 16; s2++) acc[s2] = 0.0;
            for (int j = my_rank; j < ns; j += my_width) sample_point(P, map, cx, cy, j, ns, inv_ns, acc, out, bad);
#pragma unroll
            for (int s2 = 0; s2 < 15; s2++) m.red[s2 * 33 + lane] = acc[s2];
        }
        T.sync();
        {   // owner (piece i, slot s): slot = lane % 16, two pieces per pass, four interleaved chains in fixed order
            const int s2 = lane & 15;
            for (int i = lane >> 4; i < M; i += 2) {
                const int lo = (int)m.lw[2 * i], w = (int)m.lw[2 * i + 1];
                const double *p = m.red + (s2 < 15 ? s2 : 0) * 33 + lo;
                double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
                for (int k = 0; k < w; k += 4) {
                    a0 += p[k];
                    a1 += k + 1 < w ? p[k + 1] : 0.0;
                    a2 += k + 2 < w ? p[k + 2] : 0.0;
                    a3 += k + 3 < w ? p[k + 3] : 0.0;
                }
                const double tot = (a0 + a1) + (a2 + a3);
                if (s2 < 12) m.gC[12 * i + s2] += tot;
                else if (s2 == 12) m.gT[i] += tot;
                else if (s2 < 15) m.pc[2 * i + (s2 - 13)] = tot;
            }
        }
        T.sync();
        for (int i = 0; i < M; i++) { costs2 += m.pc[2 * i]; costs3 += m.pc[2 * i + 1]; }
    }
    bad = T.rmax(bad);
    out.ns = T.radd(out.ns);
    out.nv = T.radd(out.nv);
    out.nc = T.radd(out.nc);
    out.costs[0] = costs0; out.costs[1] = costs1; out.costs[2] = costs2; out.costs[3] = costs3;
    out.f = costs0 * P.w0 + costs1 * P.w1 + costs2 * P.w2 + costs3 * P.w3;
    if (bad) { out.status = bad; return; }
    T.sync();

    // ---- adjoint (EP:494-537) ------------------------------------------------------------------------
    // h_i = H(T_i)^T dW/dc_i: gradient w.r.t. the boundary states of piece i, lane (i, d)
    if (lane < 2 * M) {
        const int i = lane >> 1, d = lane & 1;
        const double a = m.iT[5 * i], a2 = m.iT[5 * i + 1], a3 = m.iT[5 * i + 2], a4 = m.iT[5 * i + 3], a5 = m.iT[5 * i + 4];
        const double *g = m.gC + 12 * i + d;
        const double g0 = g[0], g1 = g[2], g2 = g[4], g3 = g[6], g4 = g[8], g5 = g[10];
        double *h = m.h + 12 * i + d;
        const double pe = 10.0 * a3 * g3 - 15.0 * a4 * g4 + 6.0 * a5 * g5;
        h[0] = g0 - pe;
        h[2] = g1 - 6.0 * a2 * g3 + 8.0 * a3 * g4 - 3.0 * a4 * g5;
        h[4] = 0.5 * g2 - 1.5 * a * g3 + 1.5 * a2 * g4 - 0.5 * a3 * g5;
        h[6] = pe;
        h[8] = -4.0 * a2 * g3 + 7.0 * a3 * g4 - 3.0 * a4 * g5;
        h[10] = 0.5 * a * g3 - a2 * g4 + 0.5 * a3 * g5;
    }
    T.sync();
    // eta_j = dW/d(v_j, a_j) at the interior nodes, then K^T lam = eta by block elimination (lanes 0/1 per dim);
    // the Schur complements of K^T are the transposes of those of K, so D'^-1 from the forward solve is reused.
    {
        const int d = lane & 1;
        double y0 = 0.0, y1 = 0.0;      // y_{j-1} = D'^-T_{j-1} eta'_{j-1}
        for (int j = 1; j < M; j++) {
            const double *B = m.blk + 12 * j;
            double e0 = m.h[12 * (j - 1) + 8 + d] + m.h[12 * j + 2 + d];
            double e1 = m.h[12 * (j - 1) + 10 + d] + m.h[12 * j + 4 + d];
            if (j > 1) {
                const double *Bp = m.blk + 12 * (j - 1);
                e0 -= Bp[8] * y0 + Bp[10] * y1;          // U_{j-1}^T y
                e1 -= Bp[9] * y0 + Bp[11] * y1;
            }
            y0 = B[4] * e0 + B[6] * e1;                  // D'^-T eta'
            y1 = B[5] * e0 + B[7] * e1;
            if (lane < 2) { m.r[4 * j + d] = y0; m.r[4 * j + 2 + d] = y1; }
        }
        T.sync();
        double l0 = 0.0, l1 = 0.0;
        for (int j = M - 1; j >= 1; j--) {
            const double *B = m.blk + 12 * j;
            double s0 = m.r[4 * j + d], s1 = m.r[4 * j + 2 + d];
            if (j < M - 1) {
                const double *Bn = m.blk + 12 * (j + 1);
                const double t0 = Bn[0] * l0 + Bn[2] * l1, t1 = Bn[1] * l0 + Bn[3] * l1;    // L_{j+1}^T lam_{j+1}
                s0 -= B[4] * t0 + B[6] * t1;             // D'^-T (.)
                s1 -= B[5] * t0 + B[7] * t1;
            }
            l0 = s0; l1 = s1;
            if (lane < 2) { m.lam[4 * j + d] = l0; m.lam[4 * j + 2 + d] = l1; }
        }
        if (lane < 2) { m.lam[d] = 0.0; m.lam[2 + d] = 0.0; m.lam[4 * M + d] = 0.0; m.lam[4 * M + 2 + d] = 0.0; }
    }
    T.sync();
    // G rows of interior node j (reference rows 6(j-1)+3 .. 6(j-1)+8), lane (j, d): grad_q and the T-gradient inputs
    if (lane >= 2 && lane < 2 * M) {
        const int j = lane >> 1, d = lane & 1;
        const double a3 = m.iT[5 * (j - 1) + 2], a4 = m.iT[5 * (j - 1) + 3];
        const double b = m.iT[5 * j], b2 = m.iT[5 * j + 1], b3 = m.iT[5 * j + 2], b4 = m.iT[5 * j + 3];
        const double lJ = m.lam[4 * j + d], lS = m.lam[4 * j + 2 + d];
        const double lJm = m.lam[4 * (j - 1) + d], lSm = m.lam[4 * (j - 1) + 2 + d];        // zero at node 0
        const double lJp = m.lam[4 * (j + 1) + d], lSp = m.lam[4 * (j + 1) + 2 + d];        // zero at node M
        const double *hj = m.h + 12 * j + d, *hm = m.h + 12 * (j - 1) + d;
        const double Gp = -hj[0] - (-60.0 * b3 * lJ + 360.0 * b4 * lS) + (-60.0 * b3 * lJp - 360.0 * b4 * lSp);
        const double Gv = -hj[2] - (-36.0 * b2 * lJ + 192.0 * b3 * lS) + (-24.0 * b2 * lJp - 168.0 * b3 * lSp);
        const double Ga = -hj[4] - (-9.0 * b * lJ + 36.0 * b2 * lS) + (-3.0 * b * lJp - 24.0 * b2 * lSp);
        const double Gq = hm[6] + hj[0] + (60.0 * a3 * lJm - 360.0 * a4 * lSm)
                        - ((60.0 * a3 + 60.0 * b3) * lJ + (360.0 * a4 - 360.0 * b4) * lS)
                        - (-60.0 * b3 * lJp - 360.0 * b4 * lSp);
        double *G = m.Gs + 10 * j + d;
        G[0] = Gq + Gp; G[2] = Gv; G[4] = Ga; G[6] = lJ; G[8] = lS;
        m.gout[d * (M - 1) + (j - 1)] = Gq;              // grad_q[d][j-1] = G[6(j-1)+3][d] (EP:506-508)
    }
    T.sync();
    // grad_T (EP:511-533): piece i < M-1 uses T_i; the last piece re-uses the loop variable T = ts[M-2]
    if (lane < M) {
        const int i = lane;
        const double Tq = (i < M - 1) ? m.ts[i] : m.ts[M - 2];
        const double T2 = Tq * Tq, T3 = T2 * Tq, T4 = T3 * Tq;
        const double *ci = m.c + 12 * i;
        double tr = 0.0;
#pragma unroll
        for (int d = 0; d < 2; d++) {
            const double c1 = ci[2 + d], c2 = ci[4 + d], c3 = ci[6 + d], c4 = ci[8 + d], c5 = ci[10 + d];
            const double vel = c1 + 2.0 * Tq * c2 + 3.0 * T2 * c3 + 4.0 * T3 * c4 + 5.0 * T4 * c5;
            const double ac = 2.0 * c2 + 6.0 * Tq * c3 + 12.0 * T2 * c4 + 20.0 * T3 * c5;
            const double jr = 6.0 * c3 + 24.0 * Tq * c4 + 60.0 * T2 * c5;
            if (i < M - 1) {
                const double sn = 24.0 * c4 + 120.0 * Tq * c5;
                const double cr = 120.0 * c5;
                const double *G = m.Gs + 10 * (i + 1) + d;
                tr += G[0] * vel + G[2] * ac + G[4] * jr + G[6] * sn + G[8] * cr;
            } else {      // tail rows: G[-3:] = dW/d(tail pos, vel, acc)
                const double b = m.iT[5 * i], b2 = m.iT[5 * i + 1], b3 = m.iT[5 * i + 2], b4 = m.iT[5 * i + 3];
                const double lJ = m.lam[4 * i + d], lS = m.lam[4 * i + 2 + d];      // multipliers of node M-1 (0 if M = 1)
                const double *h = m.h + 12 * i + d;
                const double Gtp = h[6] + 60.0 * b3 * lJ - 360.0 * b4 * lS;
                const double Gtv = h[8] - 24.0 * b2 * lJ + 168.0 * b3 * lS;
                const double Gta = h[10] + 3.0 * b * lJ - 24.0 * b2 * lS;
                tr += Gtp * vel + Gtv * ac + Gta * jr;
            }
        }
        const double gTi = m.gT[i] - tr;
        m.gout[nq + i] = gTi * (P.T_max - P.T_min) * e / ((1.0 + e) * (1.0 + e));      // EP:485-492
    }
    T.sync();
    out.g = (lane < nq + M) ? m.gout[lane] : 0.0;
    T.sync();
}

}  // namespace neo
