// lbfgsb_tile.cuh -- scipy.optimize.minimize(method='L-BFGS-B', bounds=None, tol=1e-4, maxcor=10, maxls=20) exactly as
// the reference calls it (EP:213-225), one tile of TL lanes per problem, the whole optimizer state on chip: lane l < n
// owns component l of x, g, d, z and of the saved iterate; the limited-memory matrices live in the tile's shared-memory
// slice; scalar logic (More'-Thuente dcsrch/dcstep of MINPACK-2, as used by L-BFGS-B 3.0's lnsrlb) is executed
// redundantly and identically by all lanes of the tile. No host round trips.
//
// scipy is a third-party dependency of the reference (not vendored; scipy 1.18.1 = C port of L-BFGS-B 3.0 over OpenBLAS).
// What is restated here is its ARITHMETIC, operation by operation, for the unbounded case -- the same restatement as
// oracle/minco_oracle.c (which is bit-identical to scipy when both are fed the same f and g; tests/test_oracle_golden.py):
//   * direction by the compact representation: formk (assemble [Y'Y/theta + D, R_z'; R_z, 0], Cholesky of the (1,1)
//     block, triangular solve, Cholesky of the (2,2) block) and subsm (two triangular solves), then d = (x + step) - x
//     as two rounded operations, and x_new = z when the step length is exactly 1;
//   * the summation orders and fused/unfused multiply-adds of the BLAS kernels behind ddot, dpotrf (potf2 + dgemv_t),
//     dtrtrs (trsv for one right-hand side, the blocked trsm kernel for several), daxpy, and the x87 dnrm2 (x87_nrm2.h);
//     scipy's own loops (formk's inner products, subsm) are unfused multiply + add;
//   * ftol = gtol = 1e-4 (tol), factr = ftol/eps; stop if max|g| <= 1e-4 or (f_old-f) <= 1e-4*max(|f_old|,|f|,1);
//     first step min(1/|d|, 1e10) on iteration 0, else 1; dcsrch(ftol=1e-3, gtol=0.9, xtol=0.1, stpmin=0, stpmax=1e10);
//     CONVERGENCE and WARNING exits are both accepted; a 21st evaluation request fails the search;
//   * on a failed search: restore x, f, g; if the memory is empty -> ABNORMAL, else drop the memory and retry;
//     the pair (s, y) is stored unless s'y <= eps * (-g_old's);
//   * scipy's ScalarFunction does not re-evaluate an x identical to the last evaluated one (nfev bookkeeping).
// Every operation whose rounding matters is written with the __d*_rn / __fma_rn intrinsics, which the compiler never
// contracts or reassociates; tests/test_gpu_lockstep.py replays the device's recorded (x, f, g) sequence through the
// checker's optimizer and requires every requested point to be bit-identical.
#pragma once
#include "minco_tile.cuh"
#include "x87_nrm2.h"

namespace neo {

// ---- exactly rounded, never contracted -----------------------------------------------------------------------------
__device__ __forceinline__ double xmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double xadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double xsub(double a, double b) { return __dsub_rn(a, b); }
// division and square root expand to ~15 instructions plus a slow path each; with some 60 call sites in the optimizer they
// are kept out of line so that the hot loop fits the instruction cache (profiles/r2_summary.md: 50 % of the stall samples
// of the first version of this file were instruction fetches)
__device__ __noinline__ double xdiv(double a, double b) { return __ddiv_rn(a, b); }
__device__ __noinline__ double xsqrt(double a) { return __dsqrt_rn(a); }
__device__ __noinline__ double nrm2_x87(int n, const double *v) { return x87_nrm2(n, v); }
__device__ __forceinline__ double xrcp(double a) { return __drcp_rn(a); }          // RN(1 / a), same value as xdiv(1, a)
__device__ __forceinline__ double xfma(double a, double b, double c) { return __fma_rn(a, b, c); }
// a / b, correctly rounded, given rb = RN(1 / b): q = RN(a rb), then one fused correction with the exact residual
// (Markstein's theorem; operands here are in the normal range; checked against the hardware division on 4e8 random pairs)
__device__ __forceinline__ double xdiv_r(double a, double b, double rb)
{
    const double q = __dmul_rn(a, rb);
    return __fma_rn(__fma_rn(-b, q, a), rb, q);
}

struct Dcsrch {
    bool brackt;
    int stage;
    double finit, ginit, gtest, width, width1, stx, fx, gx, sty, fy, gy, stmin, stmax;
};

#define LS_FTOL 1e-3
#define LS_GTOL 0.9
#define LS_XTOL 0.1
#define LS_STPMIN 0.0
#define LS_STPMAX 1e10

__device__ __forceinline__ double max3(double a, double b, double c) { return fmax(a, fmax(b, c)); }

// MINPACK-2 dcstep. Every quotient below is the correctly rounded quotient the host code computes; divisions that
// share a divisor go through one correctly rounded reciprocal (xdiv_r), x / 2 is written x * 0.5 and dx / |dx| is the
// sign of dx (all exact identities), so the values are bit-identical to a plain transcription.
// The four cases of the routine differ in which points feed the cubic and in a few signs; the expensive part (one
// cubic: two reciprocals, a square root, two divisions) is written ONCE on case-selected operands, so that the tiles
// of a warp that are in different cases still execute it together instead of one case after the other.
__device__ __forceinline__ void dcstep(double &stx, double &fx, double &dx, double &sty, double &fy, double &dy, double &stp,
                                       double fp, double dp, bool &brackt, double stpmin, double stpmax)
{
    const double sgnd = xmul(dp, dx > 0.0 ? 1.0 : (dx < 0.0 ? -1.0 : __longlong_as_double(0x7ff8000000000000LL)));
    const int kase = fp > fx ? 1 : (sgnd < 0.0 ? 2 : (fabs(dp) < fabs(dx) ? 3 : 4));
    const bool cubic = kase < 4 || brackt;
    // the cubic through (a: fa, da) and (stp: fb, dp): theta = 3 (fa - fb) / den + da + dp
    const double fa = kase < 4 ? fx : fp, fb = kase < 4 ? fp : fy, da = kase < 4 ? dx : dy;
    const double den = kase < 4 ? xsub(stp, stx) : xsub(sty, stp);
    double theta = 0.0, gamma = 0.0, rden = 0.0;
    if (cubic) {
        rden = __drcp_rn(den);
        theta = xadd(xadd(xdiv_r(xmul(3.0, xsub(fa, fb)), den, rden), da), dp);
        const double s = max3(fabs(theta), fabs(da), fabs(dp));
        const double rs = __drcp_rn(s);
        const double ts = xdiv_r(theta, s, rs);
        double rad = xsub(xmul(ts, ts), xmul(xdiv_r(da, s, rs), xdiv_r(dp, s, rs)));
        if (kase == 3) rad = fmax(0.0, rad);
        gamma = xmul(s, __dsqrt_rn(rad));
        const bool flip = kase == 1 ? stp < stx : (kase == 4 ? stp > sty : stp > stx);
        if (flip) gamma = -gamma;
    }
    // r = p / q
    const double g1 = xsub(gamma, kase == 1 ? dx : dp);
    const double p = xadd(g1, theta);
    const double q = kase == 3 ? xadd(xadd(gamma, xsub(dx, dp)), gamma) : xadd(xadd(g1, gamma), kase == 1 ? dp : (kase == 2 ? dx : dy));
    const double r = cubic ? __ddiv_rn(p, q) : 0.0;
    // the secant / quadratic step: case 1 dx / ((fx - fp) / den + dx) / 2, cases 2 and 3 dp / (dp - dx)
    const double qn = kase == 1 ? dx : dp;
    const double qd = kase == 1 ? xadd(xdiv_r(xsub(fx, fp), den, rden), dx) : xsub(dp, dx);
    const double qq = kase < 4 ? __ddiv_rn(qn, qd) : 0.0;
    double stpf, stpc, stpq;
    if (kase == 1) {
        stpc = xadd(stx, xmul(r, den));
        stpq = xadd(stx, xmul(xmul(qq, 0.5), den));
        if (fabs(xsub(stpc, stx)) < fabs(xsub(stpq, stx))) stpf = stpc; else stpf = xadd(stpc, xmul(xsub(stpq, stpc), 0.5));
        brackt = true;
    } else if (kase == 2) {
        stpc = xadd(stp, xmul(r, xsub(stx, stp)));
        stpq = xadd(stp, xmul(qq, xsub(stx, stp)));
        if (fabs(xsub(stpc, stp)) > fabs(xsub(stpq, stp))) stpf = stpc; else stpf = stpq;
        brackt = true;
    } else if (kase == 3) {
        if (r < 0.0 && gamma != 0.0) stpc = xadd(stp, xmul(r, xsub(stx, stp)));
        else if (stp > stx) stpc = stpmax;
        else stpc = stpmin;
        stpq = xadd(stp, xmul(qq, xsub(stx, stp)));
        if (brackt) {
            if (fabs(xsub(stpc, stp)) < fabs(xsub(stpq, stp))) stpf = stpc; else stpf = stpq;
            if (stp > stx) stpf = fmin(xadd(stp, xmul(0.66, xsub(sty, stp))), stpf);
            else stpf = fmax(xadd(stp, xmul(0.66, xsub(sty, stp))), stpf);
        } else {
            if (fabs(xsub(stpc, stp)) > fabs(xsub(stpq, stp))) stpf = stpc; else stpf = stpq;
            stpf = fmin(stpmax, stpf); stpf = fmax(stpmin, stpf);
        }
    } else {
        if (brackt) stpf = xadd(stp, xmul(r, xsub(sty, stp)));
        else if (stp > stx) stpf = stpmax;
        else stpf = stpmin;
    }
    if (fp > fx) { sty = stp; fy = fp; dy = dp; }
    else {
        if (sgnd < 0.0) { sty = stx; fy = fx; dy = dx; }
        stx = stp; fx = fp; dx = dp;
    }
    stp = stpf;
}

__device__ __forceinline__ void dcsrch_start(Dcsrch &S, double stp, double f, double g)
{
    S.brackt = false; S.stage = 1; S.finit = f; S.ginit = g; S.gtest = xmul(LS_FTOL, g);
    S.width = LS_STPMAX - LS_STPMIN; S.width1 = xmul(S.width, 2.0);
    S.stx = 0.0; S.fx = f; S.gx = g; S.sty = 0.0; S.fy = f; S.gy = g;
    S.stmin = 0.0; S.stmax = xadd(stp, xmul(4.0, stp));
}

// 0 = evaluate at stp, 1 = CONVERGENCE, 2 = WARNING
__device__ __forceinline__ int dcsrch_step(Dcsrch &S, double &stp, double f, double g)
{
    const double ftest = xadd(S.finit, xmul(stp, S.gtest));
    int task = 0;
    if (S.stage == 1 && f <= ftest && g >= 0.0) S.stage = 2;
    if (S.brackt && (stp <= S.stmin || stp >= S.stmax)) task = 2;
    if (S.brackt && xsub(S.stmax, S.stmin) <= xmul(LS_XTOL, S.stmax)) task = 2;
    if (stp == LS_STPMAX && f <= ftest && g <= S.gtest) task = 2;
    if (stp == LS_STPMIN && (f > ftest || g >= S.gtest)) task = 2;
    if (f <= ftest && fabs(g) <= xmul(LS_GTOL, -S.ginit)) task = 1;
    if (task) return task;
    {   // a modified function is used in stage 1 while the decrease is not yet sufficient
        const bool mod = S.stage == 1 && f <= S.fx && f > ftest;
        const double gt = mod ? S.gtest : 0.0;
        const double fm = xsub(f, xmul(stp, gt)), gm = xsub(g, gt);
        double fxm = xsub(S.fx, xmul(S.stx, gt)), fym = xsub(S.fy, xmul(S.sty, gt)), gxm = xsub(S.gx, gt), gym = xsub(S.gy, gt);
        dcstep(S.stx, fxm, gxm, S.sty, fym, gym, stp, fm, gm, S.brackt, S.stmin, S.stmax);
        S.fx = xadd(fxm, xmul(S.stx, gt)); S.fy = xadd(fym, xmul(S.sty, gt));
        S.gx = xadd(gxm, gt); S.gy = xadd(gym, gt);
    }
    if (S.brackt) {
        if (fabs(xsub(S.sty, S.stx)) >= xmul(0.66, S.width1)) stp = xadd(S.stx, xmul(0.5, xsub(S.sty, S.stx)));
        S.width1 = S.width; S.width = fabs(xsub(S.sty, S.stx));
    }
    if (S.brackt) { S.stmin = fmin(S.stx, S.sty); S.stmax = fmax(S.stx, S.sty); }
    else { S.stmin = xadd(stp, xmul(1.1, xsub(stp, S.stx))); S.stmax = xadd(stp, xmul(4.0, xsub(stp, S.stx))); }
    stp = fmax(stp, LS_STPMIN); stp = fmin(stp, LS_STPMAX);
    if ((S.brackt && (stp <= S.stmin || stp >= S.stmax)) || (S.brackt && xsub(S.stmax, S.stmin) <= xmul(LS_XTOL, S.stmax)))
        stp = S.stx;
    return 0;
}

// ---- BLAS kernels restated (see the header of this file and oracle/minco_oracle.c) ------------------------------------
// ddot: n < 16 fused multiply-adds in index order; 16 <= n < 32: the first 16 products rounded, four lanes, fold, then fma
__device__ __noinline__ double blas_ddot(int n, const double *a, const double *b)
{
    double s = 0.0;
    int i = 0;
    if (n >= 16) {
        double v[4];
#pragma unroll
        for (int l = 0; l < 4; l++)
            v[l] = xadd(xadd(xadd(xmul(a[l], b[l]), xmul(a[4 + l], b[4 + l])), xmul(a[8 + l], b[8 + l])), xmul(a[12 + l], b[12 + l]));
        s = xadd(xadd(v[0], v[2]), xadd(v[1], v[3]));
        i = 16;
    }
#pragma unroll 1
    for (; i < n; i++) s = xfma(a[i], b[i], s);
    return s;
}
// a loop written out in scipy's own C: multiply, then add
__device__ __noinline__ double loop_dot(int n, const double *a, const double *b)
{
    double s = 0.0;
#pragma unroll 1
    for (int i = 0; i < n; i++) s = xadd(s, xmul(a[i], b[i]));
    return s;
}

// the same two inner products for a vector length known at compile time (n = 3M - 2, short trajectories): straight-line
// code instead of a call and a loop -- identical operations in identical order
template <int N>
__device__ __forceinline__ double loop_dot_n(const double *a, const double *b, int n = N)
{
    if constexpr (N <= 10) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < N; i++) s = xadd(s, xmul(a[i], b[i]));
        return s;
    } else return loop_dot(n, a, b);
}
template <int N>
__device__ __forceinline__ double blas_ddot_n(const double *a, const double *b, int n = N)
{
    if constexpr (N <= 10) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < N; i++) s = xfma(a[i], b[i], s);
        return s;
    } else return blas_ddot(n, a, b);
}

// packed upper triangle: element (i, j), i <= j
__device__ __forceinline__ int wn_col(int j) { return j * (j + 1) / 2; }

// dpotrf (OpenBLAS potf2_U) on the n x n diagonal block starting at row/column o. false: not positive definite.
// rd[o + j] receives 1 / u_jj (used again by the triangular solves). Per column: the pivot a_jj - ddot(...) and the row
// sums of this lane's elements are independent chains (issued together); only the final scaling waits for the root.
__device__ __noinline__ bool lb_potf2(int tl, int TL, unsigned mask, double *wn, double *rd, int o, int n)
{
#pragma unroll 1
    for (int j = 0; j < n; j++) {
        double *cj = wn + wn_col(o + j) + o;                         // cj[k] = element (o + k, o + j)
        double dot = 0.0;                                             // ddot, j < 16: fused multiply-adds in index order
#pragma unroll 1
        for (int k = 0; k < j; k++) dot = xfma(cj[k], cj[k], dot);
        const int m1 = j & ~3, k3 = j - m1;
        double v[2];
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const int i = j + 1 + tl + q * TL;
            v[q] = 0.0;
            if (i < n) {
                const double *ci = wn + wn_col(o + i) + o;           // ci[k] = element (o + k, o + i)
                double t = ci[j];
                if (m1) {                                             // dgemv_t kernel: four rows at a time in four lanes
                    double a0 = xmul(ci[0], cj[0]), a1 = xmul(ci[1], cj[1]), a2 = xmul(ci[2], cj[2]), a3 = xmul(ci[3], cj[3]);
                    if (m1 == 8) {
                        a0 = xadd(a0, xmul(ci[4], cj[4])); a1 = xadd(a1, xmul(ci[5], cj[5]));
                        a2 = xadd(a2, xmul(ci[6], cj[6])); a3 = xadd(a3, xmul(ci[7], cj[7]));
                    }
                    t = xsub(t, xadd(xadd(a0, a2), xadd(a1, a3)));
                }
                if (k3 == 1) t = xfma(ci[m1], -cj[m1], t);
                else if (k3 == 2) t = xadd(t, xfma(ci[m1], -cj[m1], xmul(ci[m1 + 1], -cj[m1 + 1])));
                else if (k3 == 3) t = xadd(t, xfma(ci[m1 + 2], -cj[m1 + 2], xfma(ci[m1], -cj[m1], xmul(ci[m1 + 1], -cj[m1 + 1]))));
                v[q] = t;
            }
        }
        double ajj = xsub(cj[j], dot);
        if (!(ajj > 0.0)) return false;                               // same value in every lane of the tile
        ajj = __dsqrt_rn(ajj);
        const double r = __drcp_rn(ajj);
        __syncwarp(mask);
        if (tl == 0) { cj[j] = ajj; rd[o + j] = r; }
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const int i = j + 1 + tl + q * TL;
            if (i < n) wn[wn_col(o + i) + o + j] = xmul(v[q], r);
        }
        __syncwarp(mask);
    }
    return true;
}

// Per-tile limited-memory state that is not in shared memory (identical in every lane of the tile)
struct LbMem {
    int col, head, iupdat;
    double theta;
};

__device__ __forceinline__ int lb_slot(const LbMem &L, int k) { const int s = L.head + k; return s >= HIST ? s - HIST : s; }

// matupd + the bookkeeping formk does for a new pair: s, y are the lane-owned components (tl < n)
template <int TL, int NC>
__device__ __forceinline__ void lb_update(const Tile<TL> &T, const TileMem &m, int n, LbMem &L, double s, double y, double rr, double dr)
{
    L.iupdat++;
    if (L.iupdat <= HIST) L.col = L.iupdat;
    else L.head = L.head + 1 == HIST ? 0 : L.head + 1;                // the oldest pair's slot is reused
    const int col = L.col, slot = lb_slot(L, col - 1);
    if (T.tl < n) { m.ws[slot * n + T.tl] = s; m.wy[slot * n + T.tl] = y; }
    L.theta = xdiv(rr, dr);
    if (T.tl == 0) m.dr[slot] = dr;
    T.sync();
    const double *ynew = m.wy + slot * n;
#pragma unroll 1
    for (int e = T.tl; e < 2 * col; e += TL) {
        if (e < col) {                                                 // row `col` of Y'Y
            const int sj = lb_slot(L, e);
            m.yr[slot * HIST + sj] = loop_dot_n<NC>(ynew, m.wy + sj * n, n);
        } else {                                                       // column `col` of R_z
            const int si = lb_slot(L, e - col);
            const double v = loop_dot_n<NC>(m.ws + si * n, ynew, n);
            if (si == slot) m.rzd[slot] = v; else m.yr[si * HIST + slot] = v;
        }
    }
    T.sync();
}

// formk: assemble the middle matrix and factor it. false: a Cholesky factorisation failed (scipy drops the memory).
template <int TL>
__device__ __forceinline__ bool lb_factor(const Tile<TL> &T, const TileMem &m, const LbMem &L)
{
    const int col = L.col;
    const double theta = L.theta, rtheta = xrcp(theta);
    double *wn = m.wn, *rd = m.wn + wn_col(LBW) + LBW;
#pragma unroll 1
    for (int iy = T.tl; iy < col; iy += TL) {
        const int si = lb_slot(L, iy), is = col + iy;
        double *c1 = wn + wn_col(iy), *c2 = wn + wn_col(is);
#pragma unroll 1
        for (int jy = 0; jy <= iy; jy++) {
            const int sj = lb_slot(L, jy);
            double v = xdiv_r(m.yr[si * HIST + sj], theta, rtheta);                    // Y'Y / theta
            if (jy == iy) v = xadd(v, m.dr[si]);                                         // + D
            c1[jy] = v;
            c2[col + jy] = 0.0;                                                           // S'AA'S * theta (no active set)
        }
#pragma unroll 1
        for (int jy = 0; jy < iy; jy++) c2[jy] = -0.0;                                   // -L_a'
#pragma unroll 1
        for (int jy = iy; jy < col; jy++) {
            const int sj = lb_slot(L, jy);
            c2[jy] = jy == iy ? m.rzd[si] : m.yr[si * HIST + sj];                        // R_z'
        }
    }
    // NOTE the transposition: formk fills wn(jy, is) = R_z(iy, jy) for jy >= iy -- column `is`, rows jy: c2[jy] above.
    T.sync();
    if (!lb_potf2(T.tl, TL, T.mask, wn, rd, 0, col)) return false;
    if (col == 1) {                                                    // one right-hand side: trsv, a true division
        if (T.tl == 0) wn[wn_col(1)] = xdiv_r(wn[wn_col(1)], wn[0], rd[0]);
    } else {                                                           // blocked trsm kernel: 8, 4, 2, 1 rows
#pragma unroll 1
        for (int c = col + T.tl; c < 2 * col; c += TL) {
            double *b = wn + wn_col(c);
            int kk = 0;
#pragma unroll 1
            for (int bs = 8; bs > 0; bs >>= 1) {
                if (!(col & bs)) continue;
                if (kk > 0)
#pragma unroll 1
                    for (int i = kk; i < kk + bs; i++) {
                        const double *ui = wn + wn_col(i);
                        double acc = 0.0;
#pragma unroll 1
                        for (int k = 0; k < kk; k++) acc = xfma(ui[k], b[k], acc);
                        b[i] = xsub(b[i], acc);
                    }
#pragma unroll 1
                for (int i = kk; i < kk + bs; i++) {
                    b[i] = xmul(b[i], rd[i]);
#pragma unroll 1
                    for (int k = i + 1; k < kk + bs; k++) b[k] = xfma(-b[i], wn[wn_col(k) + i], b[k]);
                }
                kk += bs;
            }
        }
    }
    T.sync();
    // (2,2) block: every entry (is <= js) gets its own inner product over the first col rows -- one lane each
#pragma unroll 1
    for (int e = T.tl; e < col * (col + 1) / 2; e += TL) {
        int jj = 0;
        while ((jj + 1) * (jj + 2) / 2 <= e) jj++;                    // column (relative), row = e - jj (jj + 1) / 2
        const int ii = e - jj * (jj + 1) / 2, js = col + jj, is = col + ii;
        wn[wn_col(js) + is] = xadd(wn[wn_col(js) + is], blas_ddot(col, wn + wn_col(is), wn + wn_col(js)));
    }
    T.sync();
    const bool pd = lb_potf2(T.tl, TL, T.mask, wn, rd, col, col);
    return pd;
}

// subsm with r = -g: returns the lane-owned component of the subspace step
template <int TL, int NC>
__device__ __forceinline__ double lb_step(const Tile<TL> &T, const TileMem &m, int n, const LbMem &L, double g)
{
    const int col = L.col, m2 = 2 * col;
    const double theta = L.theta, rtheta = xrcp(theta);
    double *wn = m.wn, *wv = m.wn + wn_col(LBW), *rd = wv + LBW;
    double d = -g;
    if (T.tl < n) m.dv[T.tl] = d;
    T.sync();
#pragma unroll 1
    for (int e = T.tl; e < m2; e += TL)
        wv[e] = e < col ? loop_dot_n<NC>(m.wy + lb_slot(L, e) * n, m.dv, n) : xmul(theta, loop_dot_n<NC>(m.ws + lb_slot(L, e - col) * n, m.dv, n));
    T.sync();
    // trsv, transposed: b_i = (b_i - ddot(i, u(0:i, i), b)) / u_ii. Every row's inner product is a chain of fused
    // multiply-adds in index order, so all rows advance together as each b_k becomes final.
    {
        constexpr int RPL = (LBW + TL - 1) / TL;
        double s[RPL];
#pragma unroll
        for (int q = 0; q < RPL; q++) s[q] = 0.0;
#pragma unroll 1
        for (int k = 0; k < m2; k++) {
            if ((k & (TL - 1)) == T.tl) {
                double v = wv[k];
                if (k > 0) {
                    double sk = s[0];
#pragma unroll
                    for (int q = 1; q < RPL; q++) if (k / TL == q) sk = s[q];
                    v = xsub(v, sk);
                }
                wv[k] = xdiv_r(v, wn[wn_col(k) + k], rd[k]);
            }
            T.sync();
            const double bk = wv[k];
#pragma unroll
            for (int q = 0; q < RPL; q++) {
                const int r = T.tl + q * TL;
                if (r > k && r < m2) {
                    const double *ur = wn + wn_col(r);
                    if (r < 16 || k >= 16) s[q] = xfma(ur[k], bk, s[q]);
                    else if (k == 15) s[q] = blas_ddot(16, ur, wv);    // the kernel's 16-element prefix (four lanes, fold)
                }
            }
        }
    }
    T.sync();
#pragma unroll 1
    for (int i = T.tl; i < col; i += TL) wv[i] = -wv[i];
    T.sync();
    // trsv, not transposed: b_i /= u_ii, then b_k = fma(-b_i, u_ki, b_k)
#pragma unroll 1
    for (int i = m2 - 1; i >= 0; i--) {
        const double *ui = wn + wn_col(i);
        if (T.tl == 0) wv[i] = xdiv_r(wv[i], ui[i], rd[i]);
        T.sync();
        const double t = -wv[i];
#pragma unroll 1
        for (int k = T.tl; k < i; k += TL) wv[k] = xfma(t, ui[k], wv[k]);
        T.sync();
    }
    if (T.tl < n) {
#pragma unroll 1
        for (int jy = 0; jy < col; jy++) {
            const int sj = lb_slot(L, jy);
            d = xadd(xadd(d, xdiv_r(xmul(m.wy[sj * n + T.tl], wv[jy]), theta, rtheta)), xmul(m.ws[sj * n + T.tl], wv[col + jy]));
        }
        d = xmul(d, rtheta);
    }
    T.sync();
    return d;
}

// the line-search state lives in shared memory between evaluations (28 registers that would otherwise stay live
// across the evaluator); every lane of the tile holds the same values, the first lane writes them back
template <int TL>
__device__ __forceinline__ void ls_load(const Tile<TL> &T, const double *p, Dcsrch &S)
{
    S.finit = p[0]; S.ginit = p[1]; S.gtest = p[2]; S.width = p[3]; S.width1 = p[4]; S.stx = p[5]; S.fx = p[6]; S.gx = p[7];
    S.sty = p[8]; S.fy = p[9]; S.gy = p[10]; S.stmin = p[11]; S.stmax = p[12];
    const int flags = (int)p[13];
    S.brackt = (flags & 1) != 0; S.stage = flags >> 1;
}
template <int TL>
__device__ __forceinline__ void ls_store(const Tile<TL> &T, double *p, const Dcsrch &S)
{
    T.sync();
    if (T.tl == 0) {
        p[0] = S.finit; p[1] = S.ginit; p[2] = S.gtest; p[3] = S.width; p[4] = S.width1; p[5] = S.stx; p[6] = S.fx; p[7] = S.gx;
        p[8] = S.sty; p[9] = S.fy; p[10] = S.gy; p[11] = S.stmin; p[12] = S.stmax;
        p[13] = (double)((S.brackt ? 1 : 0) | (S.stage << 1));
    }
    T.sync();
}

// ---- the optimizer as a state machine around ONE evaluation site ------------------------------------------------------
constexpr int ST_CANCELLED = 7;      // a speculative retry stopped because an earlier attempt was accepted (never reported)
constexpr int ST_RUNNING = -1;

struct OptState {
    double x, g, d, t, r, z, xlast;          // lane-owned components
    double f, stp, gd;                       // fold and gd_old of the running search: TileMem::ls[14], ls[15]
    LbMem L;
    int nit, nfev, ifun, status;             // (line-search state, last costs and work counters live in TileMem::ls / oc)
    bool first;
};

__device__ __forceinline__ void opt_begin(OptState &o, double x0l)
{
    o.x = x0l; o.g = 0.0; o.d = 0.0; o.t = 0.0; o.r = 0.0; o.z = 0.0; o.xlast = 0.0;
    o.f = 0.0; o.stp = 0.0; o.gd = 0.0;
    o.L.col = 0; o.L.head = 0; o.L.iupdat = 0; o.L.theta = 1.0;
    o.nit = 0; o.nfev = 0; o.ifun = 0; o.status = ST_RUNNING; o.first = true;
}

// true: x is bit-identical to the last evaluated point (no evaluation, scipy's ScalarFunction cache)
template <int TL>
__device__ __forceinline__ bool opt_same_point(const Tile<TL> &T, const OptState &o, int n)
{
    return !o.first && T.all(T.tl >= n || o.x == o.xlast);
}

// g . d with the BLAS kernel's summation order (both vectors go through shared memory so that every lane can add them)
template <int TL, int NC>
__device__ __forceinline__ double opt_gd(const Tile<TL> &T, const TileMem &m, int n, double g, double d)
{
    T.sync();
    if (T.tl < n) { m.gv[T.tl] = g; m.dv[T.tl] = d; }
    T.sync();
    return blas_ddot_n<NC>(m.gv, m.dv, n);
}

// Called after every evaluation (or cache hit) with f, g in place: one step of plan_once's minimize() (EP:213-225).
// Leaves the next trial point in o.x, or sets o.status (>= 0) when minimize() returns.
// cancel_word/cancel_mask: when (*cancel_word & cancel_mask) becomes non-zero (an earlier attempt of the same problem
// has been accepted, so this speculative attempt can never be the returned one) the run stops with ST_CANCELLED.
template <int TL, int NC>
__device__ __forceinline__ void opt_advance(const Tile<TL> &T, const TileMem &m, int n, OptState &o,
                                            const unsigned *cancel_word, unsigned cancel_mask)
{
    const bool mine = T.tl < n;
    const double pgtol = 1e-4, ftol = 1e-4, epsmch = 2.220446049250313e-16;
    const double tol = (ftol / epsmch) * epsmch;
    const int maxls = 20, maxiter = 15000, maxfun = 15000;
    bool new_dir;
    if (o.first) {
        o.first = false;
        if (T.dmax(mine ? fabs(o.g) : 0.0) <= pgtol) { o.status = 1; return; }
        new_dir = true;
    } else {
        o.gd = opt_gd<TL, NC>(T, m, n, o.g, o.d);
        Dcsrch ls;
        ls_load(T, m.ls, ls);
        const int ls_task = dcsrch_step(ls, o.stp, o.f, o.gd);
        if (ls_task == 0) ls_store(T, m.ls, ls);
        if (ls_task == 0) new_dir = false;                                       // FG: another trial point
        else {
            // ---- the line search accepted the last evaluated point -------------------------------------------------
            o.nit++;
            if (cancel_mask) {
                unsigned w = 0;
                if (T.tl == 0) w = *reinterpret_cast<const volatile unsigned *>(cancel_word);
                if (T.shfl(w, 0) & cancel_mask) { o.status = ST_CANCELLED; return; }
            }
            if (T.dmax(mine ? fabs(o.g) : 0.0) <= pgtol) { o.status = 1; return; }
            const double fold = m.ls[14], gdold = m.ls[15];
            if (xsub(fold, o.f) <= xmul(tol, max3(fabs(fold), fabs(o.f), 1.0))) { o.status = 0; return; }
            if (o.nit >= maxiter || o.nfev > maxfun) { o.status = 3; return; }
            const double y = xsub(o.g, o.r);                                       // matupd
            T.sync();
            if (mine) m.dv[T.tl] = y;
            T.sync();
            const double nr = nrm2_x87(n, m.dv);
            const double rr = xmul(nr, nr);
            double dr, ddum, s;
            if (o.stp == 1.0) { dr = xsub(o.gd, gdold); ddum = -gdold; s = o.d; }
            else { dr = xmul(xsub(o.gd, gdold), o.stp); s = xmul(o.d, o.stp); ddum = xmul(-gdold, o.stp); }
            if (!(dr <= xmul(epsmch, ddum))) lb_update<TL, NC>(T, m, n, o.L, s, y, rr, dr);
            new_dir = true;
        }
    }
    for (;;) {      // (re)start a line search; loops only when a failed search drops the memory
        if (new_dir) {
            // ---- direction: Cauchy point x - g with an empty memory (theta = 1), else the subspace step; d = z - x ---
            if (o.L.col > 0 && !lb_factor(T, m, o.L)) { o.L.col = 0; o.L.head = 0; o.L.iupdat = 0; o.L.theta = 1.0; }
            if (o.L.col == 0) o.z = xsub(o.x, o.g);
            else o.z = xadd(o.x, lb_step<TL, NC>(T, m, n, o.L, o.g));
            o.d = mine ? xsub(o.z, o.x) : 0.0;
            // ---- lnsrlb: set up the search -----------------------------------------------------------------------
            T.sync();
            if (mine) m.dv[T.tl] = o.d;
            T.sync();
            const double dnorm = nrm2_x87(n, m.dv);
            o.stp = (o.nit == 0) ? fmin(xdiv(1.0, dnorm), LS_STPMAX) : 1.0;
            o.t = o.x; o.r = o.g;
            o.gd = opt_gd<TL, NC>(T, m, n, o.g, o.d);
            T.sync();
            if (T.tl == 0) { m.ls[14] = o.f; m.ls[15] = o.gd; }
            o.ifun = 0;
            if (o.gd >= 0.0) o.ifun = maxls + 1;                                // not a descent direction: fail
            else { Dcsrch ls; dcsrch_start(ls, o.stp, o.f, o.gd); ls_store(T, m.ls, ls); }
        }
        o.ifun++;
        if (o.ifun - 1 < maxls) break;                                          // evaluate the trial point
        // ---- failed search: restore the iterate; ABNORMAL if the memory is already empty --------------------------
        T.sync();
        o.x = o.t; o.g = o.r; o.f = m.ls[14];
        if (o.L.col == 0) { o.status = 2; return; }
        o.L.col = 0; o.L.head = 0; o.L.iupdat = 0; o.L.theta = 1.0;
        new_dir = true;
    }
    o.x = (o.stp == 1.0) ? o.z : xadd(xmul(o.stp, o.d), o.t);
}

}  // namespace neo
