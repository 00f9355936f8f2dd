/*
 * minco_oracle.c -- TEST INFRASTRUCTURE ONLY (not shipped, not on the product path).
 *
 * Plain-C, single-threaded CPU restatement of the reference NEO-Planner hot path, written from
 * the behaviour of the reference's Python (paths relative to /root/reference):
 *   EP   = src/planner/scripts/traj_planner/expert_planner.py
 *   TU   = src/planner/scripts/traj_planner/traj_utils.py
 *   ESDF = src/planner/scripts/map_server/esdf.py
 * and of scipy 1.18.1's L-BFGS-B driver (third-party, not vendored by the reference; unbounded
 * case of L-BFGS-B 3.0 + MINPACK-2 dcsrch/dcstep, call site EP:213-225).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load this library, and
 * only as the checker. Parity pin: tests/test_oracle_golden.py checks every function here against
 * tests/golden/ (.npz files), which oracle/gen_golden.py produced by importing and running the unmodified
 * reference in the build container (numpy 2.3.5 / scipy 1.18.1).
 *
 * Conventions: D = 2 (the reference's collision gradient only type-checks for D = 2, EP:459-465),
 * s = 3 (EP:36). Decision vector x = [q_x(0..M-2), q_y(0..M-2), tau(0..M-1)] (EP:211).
 * Coefficient layout: row 6*i+k = coefficient of t^k of piece i, column = dimension (EP:261-336).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#include <float.h>

#define ORC_D 2
#define ORC_MAXM 16
#define ORC_MAXN (ORC_D * (ORC_MAXM - 1) + ORC_MAXM)
#define ORC_MAXR (6 * ORC_MAXM)
#define ORC_HIST 10

/* per-attempt status codes (shared numbering with include/neoopt.h) */
enum {
    ORC_CONV_FTOL = 0,   /* CONVERGENCE: REL_REDUCTION_OF_F <= FACTR*EPSMCH */
    ORC_CONV_PG = 1,     /* CONVERGENCE: NORM_OF_PROJECTED_GRADIENT <= PGTOL */
    ORC_ABNORMAL = 2,    /* ABNORMAL_TERMINATION_IN_LNSRCH */
    ORC_MAXITER = 3,
    ORC_OVERFLOW = 4,    /* OverflowError from math.exp / float pow (EP:474-491) */
    ORC_DOMAIN = 5,      /* ValueError / ZeroDivisionError in map_T2tau (EP:474) */
    ORC_NAN = 6          /* int(nan) in the ESDF lookup (ESDF:61) */
};

typedef struct {
    double v_max, T_min, T_max, safe_dis, delta_t;
    double w[4];
    double collision_cost_tol;
    double init_T;
} orc_params;

typedef struct {
    int H, W;
    double res, ox, oy;
    const double *esdf, *gx, *gy; /* (H, W) row-major, row = y, col = x (ESDF:26) */
} orc_map;

/* ------------------------------------------------------------------------------------------ */
/* ESDF build: ESDF:23-33                                                                      */
/* ------------------------------------------------------------------------------------------ */

/* 1-D pass of Meijster's exact EDT, all-integer: out[u] = min_i (u-i)^2 + G[i].
 * G[i] may be EDT_INF (no feature in that row); at least one finite entry is assumed. */
#define EDT_INF ((int64_t)1000000000000LL)
static inline int64_t edt_f(int64_t x, int64_t i, const int64_t *G) { return (x - i) * (x - i) + G[i]; }
static inline int64_t floordiv(int64_t a, int64_t b) { int64_t q = a / b; if ((a % b != 0) && ((a < 0) != (b < 0))) q--; return q; }
static void edt_1d(const int64_t *G, int n, int64_t *out, int *s, int64_t *t)
{
    int q = 0;
    s[0] = 0; t[0] = 0;
    for (int u = 1; u < n; u++) {
        while (q >= 0 && edt_f(t[q], s[q], G) > edt_f(t[q], u, G)) q--;
        if (q < 0) { q = 0; s[0] = u; }
        else {
            int64_t i = s[q];
            int64_t w = 1 + floordiv((int64_t)u * u - i * i + G[u] - G[i], 2 * ((int64_t)u - i));
            if (w < n) { q++; s[q] = u; t[q] = w; }
        }
    }
    for (int u = n - 1; u >= 0; u--) {
        out[u] = edt_f(u, s[q], G);
        if (u == t[q]) q--;
    }
}

/* occ: raw OccupancyGrid values; occupied iff == 100 (ESDF:23, unknown(-1) is free).
 * esdf = sqrt(min squared cell distance to an occupied cell) * res  (ESDF:29)
 * gy, gx = np.gradient(esdf): central differences, one-sided at the borders, unit spacing (ESDF:33).
 * A map with no occupied cell reproduces scipy's behaviour of a single virtual feature at
 * (row -1, col 0) [probed on scipy 1.18.1]. */
void orc_esdf_build(const int8_t *occ, int H, int W, double res, double *esdf, double *gx, double *gy)
{
    const int64_t INF = EDT_INF;
    int64_t *d2 = (int64_t *)malloc(sizeof(int64_t) * (size_t)H * W);
    int any = 0;
    /* pass 1: along each row, squared distance to nearest occupied cell in that row */
    for (int r = 0; r < H; r++) {
        const int8_t *o = occ + (size_t)r * W;
        int64_t *row = d2 + (size_t)r * W;
        int last = -1;
        for (int c = 0; c < W; c++) {
            if (o[c] == 100) { last = c; any = 1; }
            row[c] = last < 0 ? INF : (int64_t)(c - last) * (c - last);
        }
        last = -1;
        for (int c = W - 1; c >= 0; c--) {
            if (o[c] == 100) last = c;
            if (last >= 0) { int64_t d = (int64_t)(last - c) * (last - c); if (d < row[c]) row[c] = d; }
        }
    }
    if (!any) {
        for (int r = 0; r < H; r++)
            for (int c = 0; c < W; c++)
                d2[(size_t)r * W + c] = (int64_t)(r + 1) * (r + 1) + (int64_t)c * c;
    } else {
        int n = H;
        int64_t *f = (int64_t *)malloc(sizeof(int64_t) * n), *o = (int64_t *)malloc(sizeof(int64_t) * n);
        int *v = (int *)malloc(sizeof(int) * (n + 1));
        int64_t *z = (int64_t *)malloc(sizeof(int64_t) * (n + 2));
        for (int c = 0; c < W; c++) {
            for (int r = 0; r < H; r++) f[r] = d2[(size_t)r * W + c];
            edt_1d(f, n, o, v, z);
            for (int r = 0; r < H; r++) d2[(size_t)r * W + c] = o[r];
        }
        free(f); free(o); free(v); free(z);
    }
    for (size_t i = 0; i < (size_t)H * W; i++) esdf[i] = sqrt((double)d2[i]) * res;
    free(d2);
    for (int r = 0; r < H; r++) {
        for (int c = 0; c < W; c++) {
            size_t i = (size_t)r * W + c;
            if (W == 1) gx[i] = 0.0;
            else if (c == 0) gx[i] = esdf[i + 1] - esdf[i];
            else if (c == W - 1) gx[i] = esdf[i] - esdf[i - 1];
            else gx[i] = (esdf[i + 1] - esdf[i - 1]) / 2.0;
            if (H == 1) gy[i] = 0.0;
            else if (r == 0) gy[i] = esdf[i + W] - esdf[i];
            else if (r == H - 1) gy[i] = esdf[i] - esdf[i - W];
            else gy[i] = (esdf[i + W] - esdf[i - W]) / 2.0;
        }
    }
}

/* Brute-force exact EDT (O(N * occupied)), independent of edt_1d; used to cross-check on small maps. */
void orc_esdf_brute(const int8_t *occ, int H, int W, double res, double *esdf)
{
    for (int r = 0; r < H; r++)
        for (int c = 0; c < W; c++) {
            int64_t best = -1;
            for (int rr = 0; rr < H; rr++)
                for (int cc = 0; cc < W; cc++)
                    if (occ[(size_t)rr * W + cc] == 100) {
                        int64_t d = (int64_t)(r - rr) * (r - rr) + (int64_t)(c - cc) * (c - cc);
                        if (best < 0 || d < best) best = d;
                    }
            if (best < 0) best = (int64_t)(r + 1) * (r + 1) + (int64_t)c * c;
            esdf[(size_t)r * W + c] = sqrt((double)best) * res;
        }
}

/* ESDF:61-65. Python int() truncates toward zero. Returns 1 if inside, 0 if outside, -1 on NaN. */
int orc_cell_index(const orc_map *m, double x, double y, int *row, int *col)
{
    double fr = (y - m->oy) / m->res;
    double fc = (x - m->ox) / m->res;
    if (isnan(fr) || isnan(fc)) return -1;
    double tr = trunc(fr), tc = trunc(fc);
    if (tr < 0 || tr >= m->H || tc < 0 || tc >= m->W) { *row = -1; *col = -1; return 0; }
    *row = (int)tr; *col = (int)tc;
    return 1;
}

/* batched query for the bit-exactness tests: out_idx (n,2) = row,col (-1 if outside), out_d, out_g (n,2) */
void orc_query(const orc_map *m, int n, const double *xy, int32_t *out_idx, double *out_d, double *out_g)
{
    for (int i = 0; i < n; i++) {
        int r, c;
        int in = orc_cell_index(m, xy[2 * i], xy[2 * i + 1], &r, &c);
        out_idx[2 * i] = r; out_idx[2 * i + 1] = c;
        if (in == 1) {
            size_t k = (size_t)r * m->W + c;
            out_d[i] = m->esdf[k]; out_g[2 * i] = m->gx[k]; out_g[2 * i + 1] = m->gy[k];
        } else { out_d[i] = 10000.0; out_g[2 * i] = 0.0; out_g[2 * i + 1] = 0.0; }
    }
}

/* ------------------------------------------------------------------------------------------ */
/* time reparametrisation: EP:468-492                                                          */
/* ------------------------------------------------------------------------------------------ */

/* EP:470-475. math.log domain error / division by zero -> ORC_DOMAIN */
int orc_T2tau(const orc_params *p, int M, const double *ts, double *tau)
{
    for (int i = 0; i < M; i++) {
        double den = ts[i] - p->T_min;
        if (den == 0.0) return ORC_DOMAIN;                 /* ZeroDivisionError */
        double a = (p->T_max - p->T_min) / den - 1.0;
        if (!(a > 0.0)) return ORC_DOMAIN;                 /* math domain error (incl. nan) */
        if (isinf(a)) { tau[i] = -INFINITY; continue; }
        tau[i] = -log(a);
    }
    return 0;
}

/* EP:477-483. math.exp raises OverflowError when the result overflows. */
int orc_tau2T(const orc_params *p, int M, const double *tau, double *ts)
{
    for (int i = 0; i < M; i++) {
        double e = exp(-tau[i]);
        if (isinf(e)) return ORC_OVERFLOW;
        ts[i] = (p->T_max - p->T_min) / (1.0 + e) + p->T_min;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------------ */
/* dense solve with partial pivoting (numpy.linalg.solve -> LAPACK gesv): EP:336, EP:503       */
/* ------------------------------------------------------------------------------------------ */
static int lu_factor(int n, double *A, int *piv)
{
    for (int k = 0; k < n; k++) {
        int p = k; double best = fabs(A[k * n + k]);
        for (int i = k + 1; i < n; i++) { double v = fabs(A[i * n + k]); if (v > best) { best = v; p = i; } }
        piv[k] = p;
        if (best == 0.0) return -1;
        if (p != k) for (int j = 0; j < n; j++) { double t = A[k * n + j]; A[k * n + j] = A[p * n + j]; A[p * n + j] = t; }
        double inv = 1.0 / A[k * n + k];
        for (int i = k + 1; i < n; i++) {
            double l = A[i * n + k] * inv;
            A[i * n + k] = l;
            if (l != 0.0) for (int j = k + 1; j < n; j++) A[i * n + j] -= l * A[k * n + j];
        }
    }
    return 0;
}

/* solve A X = B in place (B is n x nrhs row-major) */
static void lu_solve(int n, const double *LU, const int *piv, double *B, int nrhs)
{
    for (int k = 0; k < n; k++) {          /* B <- P B (all interchanges first, as dgetrs/dlaswp) */
        int p = piv[k];
        if (p != k) for (int c = 0; c < nrhs; c++) { double t = B[k * nrhs + c]; B[k * nrhs + c] = B[p * nrhs + c]; B[p * nrhs + c] = t; }
    }
    for (int k = 0; k < n; k++) {
        for (int i = k + 1; i < n; i++) {
            double l = LU[i * n + k];
            if (l != 0.0) for (int c = 0; c < nrhs; c++) B[i * nrhs + c] -= l * B[k * nrhs + c];
        }
    }
    for (int k = n - 1; k >= 0; k--) {
        for (int c = 0; c < nrhs; c++) {
            double s = B[k * nrhs + c];
            for (int j = k + 1; j < n; j++) s -= LU[k * n + j] * B[j * nrhs + c];
            B[k * nrhs + c] = s / LU[k * n + k];
        }
    }
}

/* solve A^T X = B in place using the factorisation P A = L U:  A^T = U^T L^T P */
static void lu_solve_T(int n, const double *LU, const int *piv, double *B, int nrhs)
{
    for (int k = 0; k < n; k++) {          /* U^T w = b (forward) */
        for (int c = 0; c < nrhs; c++) {
            double s = B[k * nrhs + c];
            for (int j = 0; j < k; j++) s -= LU[j * n + k] * B[j * nrhs + c];
            B[k * nrhs + c] = s / LU[k * n + k];
        }
    }
    for (int k = n - 1; k >= 0; k--) {     /* L^T z = w (backward, unit diagonal) */
        for (int c = 0; c < nrhs; c++) {
            double s = B[k * nrhs + c];
            for (int j = k + 1; j < n; j++) s -= LU[j * n + k] * B[j * nrhs + c];
            B[k * nrhs + c] = s;
        }
    }
    for (int k = n - 1; k >= 0; k--) {     /* x = P^T z */
        int p = piv[k];
        if (p != k) for (int c = 0; c < nrhs; c++) { double t = B[k * nrhs + c]; B[k * nrhs + c] = B[p * nrhs + c]; B[p * nrhs + c] = t; }
    }
}

/* ------------------------------------------------------------------------------------------ */
/* MINCO system: EP:261-336 (== TU:8-83)                                                       */
/* ------------------------------------------------------------------------------------------ */
static void build_A(int M, const double *ts, double *A)
{
    int n = 6 * M;
    memset(A, 0, sizeof(double) * n * n);
#define AE(r, c) A[(r) * n + (c)]
    AE(0, 0) = 1.0; AE(1, 1) = 1.0; AE(2, 2) = 2.0;
    for (int i = 0; i < M - 1; i++) {
        double T1 = ts[i], T2 = T1 * T1, T3 = pow(T1, 3), T4 = pow(T1, 4), T5 = pow(T1, 5);
        int r = 6 * i + 3, c = 6 * i;
        double pw[6] = {1.0, T1, T2, T3, T4, T5};
        for (int k = 0; k < 6; k++) { AE(r, c + k) = pw[k]; AE(r + 1, c + k) = pw[k]; }
        AE(r + 1, c + 6) = -1.0;
        AE(r + 2, c + 1) = 1.0; AE(r + 2, c + 2) = 2 * T1; AE(r + 2, c + 3) = 3 * T2; AE(r + 2, c + 4) = 4 * T3; AE(r + 2, c + 5) = 5 * T4;
        AE(r + 2, c + 7) = -1.0;
        AE(r + 3, c + 2) = 2.0; AE(r + 3, c + 3) = 6 * T1; AE(r + 3, c + 4) = 12 * T2; AE(r + 3, c + 5) = 20 * T3;
        AE(r + 3, c + 8) = -2.0;
        AE(r + 4, c + 3) = 6.0; AE(r + 4, c + 4) = 24.0 * T1; AE(r + 4, c + 5) = 60.0 * T2;
        AE(r + 4, c + 9) = -6.0;
        AE(r + 5, c + 4) = 24.0; AE(r + 5, c + 5) = 120.0 * T1;
        AE(r + 5, c + 10) = -24.0;
    }
    {
        double T1 = ts[M - 1], T2 = T1 * T1, T3 = pow(T1, 3), T4 = pow(T1, 4), T5 = pow(T1, 5);
        int r = n - 3, c = n - 6;
        AE(r, c) = 1.0; AE(r, c + 1) = T1; AE(r, c + 2) = T2; AE(r, c + 3) = T3; AE(r, c + 4) = T4; AE(r, c + 5) = T5;
        AE(r + 1, c + 1) = 1.0; AE(r + 1, c + 2) = 2 * T1; AE(r + 1, c + 3) = 3 * T2; AE(r + 1, c + 4) = 4 * T3; AE(r + 1, c + 5) = 5 * T4;
        AE(r + 2, c + 2) = 2.0; AE(r + 2, c + 3) = 6 * T1; AE(r + 2, c + 4) = 12 * T2; AE(r + 2, c + 5) = 20 * T3;
    }
#undef AE
}

/* head/tail: (3, D) zero-padded states (EP:170-184). q: (D, M-1). coeffs out: (6M, D).
 * LU/piv are kept for the adjoint solve. returns 0 or -1 (singular). */
static int solve_coeffs(int M, const double *head, const double *tail, const double *q, const double *ts,
                        double *LU, int *piv, double *coeffs)
{
    int n = 6 * M;
    build_A(M, ts, LU);
    memset(coeffs, 0, sizeof(double) * n * ORC_D);
    for (int k = 0; k < 3; k++)
        for (int d = 0; d < ORC_D; d++) {
            coeffs[k * ORC_D + d] = head[k * ORC_D + d];
            coeffs[(n - 3 + k) * ORC_D + d] = tail[k * ORC_D + d];
        }
    for (int i = 0; i < M - 1; i++)
        for (int d = 0; d < ORC_D; d++) coeffs[(6 * i + 3) * ORC_D + d] = q[d * (M - 1) + i];
    if (lu_factor(n, LU, piv)) return -1;
    lu_solve(n, LU, piv, coeffs, ORC_D);
    return 0;
}

/* public: TU:8-83 / EP:261-336 */
int orc_get_coeffs(int M, const double *head, const double *tail, const double *q, const double *ts, double *coeffs)
{
    double LU[ORC_MAXR * ORC_MAXR]; int piv[ORC_MAXR];
    if (M < 1 || M > ORC_MAXM) return -2;
    return solve_coeffs(M, head, tail, q, ts, LU, piv, coeffs);
}

/* ------------------------------------------------------------------------------------------ */
/* fused get_cost + get_grad: EP:539-585 with EP:345-466, EP:494-537                           */
/* ------------------------------------------------------------------------------------------ */
static inline double cube(double v) { return pow(v, 3); }

int orc_eval(const orc_params *p, const orc_map *map, int M, const double *head, const double *tail,
             const double *x, double *costs, double *grad, double *coeffs_out, double *ts_out)
{
    int n6 = 6 * M, nq = ORC_D * (M - 1);
    double ts[ORC_MAXM], LU[ORC_MAXR * ORC_MAXR], c[ORC_MAXR * ORC_D], gC[ORC_MAXR * ORC_D], gT[ORC_MAXM];
    int piv[ORC_MAXR];
    const double *q = x, *tau = x + nq;
    if (M < 2 || M > ORC_MAXM) return -2;
    int st = orc_tau2T(p, M, tau, ts);
    if (st) return st;
    if (solve_coeffs(M, head, tail, q, ts, LU, piv, c)) return ORC_NAN;
    costs[0] = costs[1] = costs[2] = costs[3] = 0.0;
    memset(gC, 0, sizeof(double) * n6 * ORC_D);
    memset(gT, 0, sizeof(double) * M);

    /* energy: EP:345-384 */
    for (int i = 0; i < M; i++) {
        const double *ci = c + 6 * i * ORC_D;
        double T = ts[i];
        double B[3][3] = {{36 * T, 72 * pow(T, 2), 120 * pow(T, 3)},
                          {72 * pow(T, 2), 192 * pow(T, 3), 360 * pow(T, 4)},
                          {120 * pow(T, 3), 360 * pow(T, 4), 720 * pow(T, 5)}};
        double b3[3] = {6.0, 24 * T, 60 * pow(T, 2)};
        for (int d = 0; d < ORC_D; d++) {
            double tmp[3];
            for (int b = 0; b < 3; b++) {
                double s = 0.0;
                for (int a = 0; a < 3; a++) s += ci[(3 + a) * ORC_D + d] * B[a][b];
                tmp[b] = s;
            }
            double s = 0.0;
            for (int b = 0; b < 3; b++) s += tmp[b] * ci[(3 + b) * ORC_D + d];
            costs[0] += s;
            for (int a = 0; a < 3; a++) {
                double s2 = 0.0;
                for (int b = 0; b < 3; b++) s2 += (p->w[0] * 2 * B[a][b]) * ci[(3 + b) * ORC_D + d];
                gC[(6 * i + 3 + a) * ORC_D + d] += s2;
            }
            double jd = 0.0;
            for (int a = 0; a < 3; a++) jd += ci[(3 + a) * ORC_D + d] * b3[a];
            gT[i] += p->w[0] * (jd * jd);
        }
    }
    /* time: EP:386-390 */
    { double s = 0.0; for (int i = 0; i < M; i++) s += ts[i]; costs[1] += s; }
    for (int i = 0; i < M; i++) gT[i] += p->w[1];

    /* sampled penalties: EP:392-466 */
    double vmax2 = p->v_max * p->v_max;
    for (int i = 0; i < M; i++) {
        const double *ci = c + 6 * i * ORC_D;
        int sample_num = (int)(ts[i] / p->delta_t);
        for (int j = 0; j < sample_num; j++) {
            double t = j * p->delta_t;              /* np.arange(0, T_max, dt)[j] (EP:251) */
            double t2 = t * t, t3 = pow(t, 3), t4 = pow(t, 4), t5 = pow(t, 5);
            double b0[6] = {1, t, t2, t3, t4, t5};
            double b1[6] = {0, 1, 2 * t, 3 * t2, 4 * t3, 5 * t4};
            double b2[6] = {0, 0, 2, 6 * t, 12 * t2, 20 * t3};
            double pos[ORC_D], vel[ORC_D], acc[ORC_D];
            for (int d = 0; d < ORC_D; d++) {
                double sp = 0, sv = 0, sa = 0;
                for (int k = 0; k < 6; k++) { sp += ci[k * ORC_D + d] * b0[k]; sv += ci[k * ORC_D + d] * b1[k]; sa += b2[k] * ci[k * ORC_D + d]; }
                pos[d] = sp; vel[d] = sv; acc[d] = sa;
            }
            double omg = (j == 0 || j == sample_num - 1) ? 0.5 : 1.0;
            double vv = 0.0;
            for (int d = 0; d < ORC_D; d++) vv += vel[d] * vel[d];
            vv -= vmax2;
            if (vv > 0.0) {
                costs[2] += omg * p->delta_t * cube(vv);
                double K = 3 * p->delta_t * omg * (vv * vv);
                double v2t = 0.0;
                for (int d = 0; d < ORC_D; d++) v2t += acc[d] * vel[d];
                v2t *= 2;
                for (int k = 0; k < 6; k++)
                    for (int d = 0; d < ORC_D; d++)
                        gC[(6 * i + k) * ORC_D + d] += p->w[2] * K * (2 * (b1[k] * vel[d]));
                gT[i] += p->w[2] * (omg * cube(vv) / sample_num + K * v2t * j / sample_num);
            }
            int r, cc;
            int in = orc_cell_index(map, pos[0], pos[1], &r, &cc);
            if (in < 0) return ORC_NAN;
            double dis = in ? map->esdf[(size_t)r * map->W + cc] : 10000.0;
            double vd = p->safe_dis - dis;
            if (vd > 0.0) {
                costs[3] += omg * p->delta_t * cube(vd);
                double g[2] = {map->gx[(size_t)r * map->W + cc], map->gy[(size_t)r * map->W + cc]};
                double K = 3 * p->delta_t * omg * (vd * vd);
                double p2t = -(g[0] * vel[0] + g[1] * vel[1]);
                for (int k = 0; k < 6; k++)
                    for (int d = 0; d < ORC_D; d++)
                        gC[(6 * i + k) * ORC_D + d] += p->w[3] * K * (-(b0[k] * g[d]));
                gT[i] += p->w[3] * (omg * cube(vd) / sample_num + K * p2t * j / sample_num);
            }
        }
    }

    /* adjoint: EP:494-537 */
    if (coeffs_out) memcpy(coeffs_out, c, sizeof(double) * n6 * ORC_D);
    if (ts_out) memcpy(ts_out, ts, sizeof(double) * M);
    if (!grad) return 0;
    double *G = gC;
    lu_solve_T(n6, LU, piv, G, ORC_D);
    for (int i = 0; i < M - 1; i++)
        for (int d = 0; d < ORC_D; d++) grad[d * (M - 1) + i] = G[(6 * i + 3) * ORC_D + d];
    double T = 0.0;
    for (int i = 0; i < M - 1; i++) {
        T = ts[i];
        double T2 = pow(T, 2), T3 = pow(T, 3), T4 = pow(T, 4);
        double E[6][6] = {{0, 1, 2 * T, 3 * T2, 4 * T3, 5 * T4},
                          {0, 1, 2 * T, 3 * T2, 4 * T3, 5 * T4},
                          {0, 0, 2, 6 * T, 12 * T2, 20 * T3},
                          {0, 0, 0, 6, 24 * T, 60 * T2},
                          {0, 0, 0, 0, 24, 120 * T},
                          {0, 0, 0, 0, 0, 120}};
        const double *ci = c + 6 * i * ORC_D;
        double tr = 0.0;
        for (int d = 0; d < ORC_D; d++) {
            double tmp[6];
            for (int k = 0; k < 6; k++) {
                double s = 0.0;
                for (int a = 0; a < 6; a++) s += G[(6 * i + 3 + a) * ORC_D + d] * E[a][k];
                tmp[k] = s;
            }
            double s = 0.0;
            for (int k = 0; k < 6; k++) s += tmp[k] * ci[k * ORC_D + d];
            tr += s;
        }
        gT[i] = gT[i] - tr;
    }
    {   /* "for E_M specially": uses the stale loop variable T = ts[M-2] (EP:527-533) */
        double T2 = pow(T, 2), T3 = pow(T, 3), T4 = pow(T, 4);
        double E[3][6] = {{0, 1, 2 * T, 3 * T2, 4 * T3, 5 * T4},
                          {0, 0, 2, 6 * T, 12 * T2, 20 * T3},
                          {0, 0, 0, 6, 24 * T, 60 * T2}};
        const double *ci = c + 6 * (M - 1) * ORC_D;
        double tr = 0.0;
        for (int d = 0; d < ORC_D; d++) {
            double tmp[6];
            for (int k = 0; k < 6; k++) {
                double s = 0.0;
                for (int a = 0; a < 3; a++) s += G[(n6 - 3 + a) * ORC_D + d] * E[a][k];
                tmp[k] = s;
            }
            double s = 0.0;
            for (int k = 0; k < 6; k++) s += tmp[k] * ci[k * ORC_D + d];
            tr += s;
        }
        gT[M - 1] = gT[M - 1] - tr;
    }
    /* chain rule: EP:485-492; (1+exp(-tau))**2 raises OverflowError when it overflows */
    for (int i = 0; i < M; i++) {
        double e = exp(-tau[i]);
        double den = (1 + e) * (1 + e);
        if (isinf(den)) return ORC_OVERFLOW;
        grad[nq + i] = gT[i] * (p->T_max - p->T_min) * e / den;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------------ */
/* L-BFGS-B (unbounded): scipy.optimize.minimize(method='L-BFGS-B') as called at EP:213-225    */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
    int brackt, stage;
    double finit, ginit, gtest, width, width1, stx, fx, gx, sty, fy, gy, stmin, stmax;
} dcs_state;

/* Optional branch counters of the optimizer (tests: which L-BFGS-B branches a run went through). Integer increments only:
 * the arithmetic is the same with and without them. The order is oracle/c_oracle.py's BRANCHES. */
enum {
    OC_DIR = 0,                       /* [0..10]: search directions computed with memory length col */
    OC_FACTOR_FAIL1 = 11,             /* formk: first Cholesky factorisation failed (memory dropped) */
    OC_FACTOR_FAIL2,                  /* formk: second Cholesky factorisation failed */
    OC_NONDESCENT_COL0,               /* g'd >= 0 with an empty memory */
    OC_NONDESCENT_COL,                /* g'd >= 0 with col > 0 */
    OC_MAXLS,                         /* a 21st evaluation request: the search failed */
    OC_ABNORMAL,                      /* failed search with an empty memory: ABNORMAL */
    OC_RESET_FAILED,                  /* failed search with col > 0: memory dropped, search restarted */
    OC_SKIP_UPDATE,                   /* s'y <= eps * (-g_old's): pair not stored */
    OC_WRAP,                          /* a pair stored with a full memory (iupdat > 10): the oldest is overwritten */
    OC_RESET_AFTER_WRAP,              /* a memory drop (either cause) after at least one wrap */
    OC_ACCEPT_STP1,                   /* search accepted with stp == 1 */
    OC_ACCEPT_STP,                    /* search accepted with stp != 1 */
    OC_CACHE_HIT,                     /* trial point equal to the last evaluated one: not evaluated again */
    OC_DCSTEP,                        /* [24..32): dcstep case 1..4 (2 * (case - 1)) x brackt at entry (+1) */
    OC_EXIT_CONV = OC_DCSTEP + 8,     /* dcsrch: CONVERGENCE */
    OC_EXIT_BOUND,                    /* dcsrch WARNING: brackt and stp outside (stmin, stmax) */
    OC_EXIT_XTOL,                     /* dcsrch WARNING: interval width <= xtol * stmax */
    OC_EXIT_STPMAX,                   /* dcsrch WARNING: stp == stpmax */
    OC_EXIT_STPMIN,                   /* dcsrch WARNING: stp == stpmin */
    OC_STX_FALLBACK,                  /* dcsrch: the new stp fell outside the bracket, stp = stx */
    OC_PG_X0,                         /* projected gradient <= pgtol at x0 */
    OC_PG,                            /* projected gradient <= pgtol after an iteration */
    OC_FTOL,                          /* relative reduction of f <= factr * eps */
    OC_MAXITER,                       /* iteration or evaluation limit */
    OC_EVAL_OVERFLOW,                 /* the run ended on an evaluation status: overflow */
    OC_EVAL_DOMAIN,                   /* ... domain error */
    OC_EVAL_NAN,                      /* ... NaN */
    OC_COUNT
};
static __thread int64_t *orc_count_cur = 0;
#define OC(i) do { if (orc_count_cur) orc_count_cur[i]++; } while (0)

/* counters go to c[0..OC_COUNT) (added to) for the calls this thread makes until it passes NULL */
void orc_count_into(int64_t *c) { orc_count_cur = c; }
int orc_count_size(void) { return OC_COUNT; }

static void dcstep(double *stx, double *fx, double *dx, double *sty, double *fy, double *dy, double *stp,
                   double fp, double dp, int *brackt, double stpmin, double stpmax)
{
    double sgnd = dp * (*dx / fabs(*dx));
    double stpf, stpc, stpq, theta, s, gamma, p, q, r;
    OC(OC_DCSTEP + 2 * (fp > *fx ? 0 : sgnd < 0.0 ? 1 : fabs(dp) < fabs(*dx) ? 2 : 3) + (*brackt ? 1 : 0));
    if (fp > *fx) {
        theta = 3.0 * (*fx - fp) / (*stp - *stx) + *dx + dp;
        s = fmax(fabs(theta), fmax(fabs(*dx), fabs(dp)));
        gamma = s * sqrt((theta / s) * (theta / s) - (*dx / s) * (dp / s));
        if (*stp < *stx) gamma = -gamma;
        p = (gamma - *dx) + theta; q = ((gamma - *dx) + gamma) + dp; r = p / q;
        stpc = *stx + r * (*stp - *stx);
        stpq = *stx + ((*dx / ((*fx - fp) / (*stp - *stx) + *dx)) / 2.0) * (*stp - *stx);
        if (fabs(stpc - *stx) < fabs(stpq - *stx)) stpf = stpc; else stpf = stpc + (stpq - stpc) / 2.0;
        *brackt = 1;
    } else if (sgnd < 0.0) {
        theta = 3.0 * (*fx - fp) / (*stp - *stx) + *dx + dp;
        s = fmax(fabs(theta), fmax(fabs(*dx), fabs(dp)));
        gamma = s * sqrt((theta / s) * (theta / s) - (*dx / s) * (dp / s));
        if (*stp > *stx) gamma = -gamma;
        p = (gamma - dp) + theta; q = ((gamma - dp) + gamma) + *dx; r = p / q;
        stpc = *stp + r * (*stx - *stp);
        stpq = *stp + (dp / (dp - *dx)) * (*stx - *stp);
        if (fabs(stpc - *stp) > fabs(stpq - *stp)) stpf = stpc; else stpf = stpq;
        *brackt = 1;
    } else if (fabs(dp) < fabs(*dx)) {
        theta = 3.0 * (*fx - fp) / (*stp - *stx) + *dx + dp;
        s = fmax(fabs(theta), fmax(fabs(*dx), fabs(dp)));
        gamma = s * sqrt(fmax(0.0, (theta / s) * (theta / s) - (*dx / s) * (dp / s)));
        if (*stp > *stx) gamma = -gamma;
        p = (gamma - dp) + theta; q = (gamma + (*dx - dp)) + gamma; r = p / q;
        if (r < 0.0 && gamma != 0.0) stpc = *stp + r * (*stx - *stp);
        else if (*stp > *stx) stpc = stpmax;
        else stpc = stpmin;
        stpq = *stp + (dp / (dp - *dx)) * (*stx - *stp);
        if (*brackt) {
            if (fabs(stpc - *stp) < fabs(stpq - *stp)) stpf = stpc; else stpf = stpq;
            if (*stp > *stx) stpf = fmin(*stp + 0.66 * (*sty - *stp), stpf);
            else stpf = fmax(*stp + 0.66 * (*sty - *stp), stpf);
        } else {
            if (fabs(stpc - *stp) > fabs(stpq - *stp)) stpf = stpc; else stpf = stpq;
            stpf = fmin(stpmax, stpf); stpf = fmax(stpmin, stpf);
        }
    } else {
        if (*brackt) {
            theta = 3.0 * (fp - *fy) / (*sty - *stp) + *dy + dp;
            s = fmax(fabs(theta), fmax(fabs(*dy), fabs(dp)));
            gamma = s * sqrt((theta / s) * (theta / s) - (*dy / s) * (dp / s));
            if (*stp > *sty) gamma = -gamma;
            p = (gamma - dp) + theta; q = ((gamma - dp) + gamma) + *dy; r = p / q;
            stpc = *stp + r * (*sty - *stp);
            stpf = stpc;
        } else if (*stp > *stx) stpf = stpmax;
        else stpf = stpmin;
    }
    if (fp > *fx) { *sty = *stp; *fy = fp; *dy = dp; }
    else {
        if (sgnd < 0.0) { *sty = *stx; *fy = *fx; *dy = *dx; }
        *stx = *stp; *fx = fp; *dx = dp;
    }
    *stp = stpf;
}

#define LS_FTOL 1e-3
#define LS_GTOL 0.9
#define LS_XTOL 0.1
#define LS_STPMIN 0.0
#define LS_STPMAX 1e10

static void dcsrch_start(dcs_state *S, double stp, double f, double g)
{
    S->brackt = 0; S->stage = 1; S->finit = f; S->ginit = g; S->gtest = LS_FTOL * g;
    S->width = LS_STPMAX - LS_STPMIN; S->width1 = S->width / 0.5;
    S->stx = 0.0; S->fx = f; S->gx = g; S->sty = 0.0; S->fy = f; S->gy = g;
    S->stmin = 0.0; S->stmax = stp + 4.0 * stp;
}

/* returns 0 = FG (evaluate at *stp), 1 = CONVERGENCE, 2 = WARNING (both accepted by lnsrlb) */
static int dcsrch_step(dcs_state *S, double *stp, double f, double g)
{
    double ftest = S->finit + *stp * S->gtest;
    int task = 0;
    if (S->stage == 1 && f <= ftest && g >= 0.0) S->stage = 2;
    if (S->brackt && (*stp <= S->stmin || *stp >= S->stmax)) task = 2;
    if (S->brackt && S->stmax - S->stmin <= LS_XTOL * S->stmax) task = 2;
    if (*stp == LS_STPMAX && f <= ftest && g <= S->gtest) task = 2;
    if (*stp == LS_STPMIN && (f > ftest || g >= S->gtest)) task = 2;
    if (f <= ftest && fabs(g) <= LS_GTOL * (-S->ginit)) task = 1;
    if (task == 1) OC(OC_EXIT_CONV);
    else if (task == 2) {
        if (S->brackt && (*stp <= S->stmin || *stp >= S->stmax)) OC(OC_EXIT_BOUND);
        if (S->brackt && S->stmax - S->stmin <= LS_XTOL * S->stmax) OC(OC_EXIT_XTOL);
        if (*stp == LS_STPMAX && f <= ftest && g <= S->gtest) OC(OC_EXIT_STPMAX);
        if (*stp == LS_STPMIN && (f > ftest || g >= S->gtest)) OC(OC_EXIT_STPMIN);
    }
    if (task) return task;
    if (S->stage == 1 && f <= S->fx && f > ftest) {
        double fm = f - *stp * S->gtest, fxm = S->fx - S->stx * S->gtest, fym = S->fy - S->sty * S->gtest;
        double gm = g - S->gtest, gxm = S->gx - S->gtest, gym = S->gy - S->gtest;
        dcstep(&S->stx, &fxm, &gxm, &S->sty, &fym, &gym, stp, fm, gm, &S->brackt, S->stmin, S->stmax);
        S->fx = fxm + S->stx * S->gtest; S->fy = fym + S->sty * S->gtest;
        S->gx = gxm + S->gtest; S->gy = gym + S->gtest;
    } else {
        dcstep(&S->stx, &S->fx, &S->gx, &S->sty, &S->fy, &S->gy, stp, f, g, &S->brackt, S->stmin, S->stmax);
    }
    if (S->brackt) {
        if (fabs(S->sty - S->stx) >= 0.66 * S->width1) *stp = S->stx + 0.5 * (S->sty - S->stx);
        S->width1 = S->width; S->width = fabs(S->sty - S->stx);
    }
    if (S->brackt) { S->stmin = fmin(S->stx, S->sty); S->stmax = fmax(S->stx, S->sty); }
    else { S->stmin = *stp + 1.1 * (*stp - S->stx); S->stmax = *stp + 4.0 * (*stp - S->stx); }
    *stp = fmax(*stp, LS_STPMIN); *stp = fmin(*stp, LS_STPMAX);
    if ((S->brackt && (*stp <= S->stmin || *stp >= S->stmax)) ||
        (S->brackt && S->stmax - S->stmin <= LS_XTOL * S->stmax)) { *stp = S->stx; OC(OC_STX_FALLBACK); }
    return 0;
}

/* ---- scipy 1.18.1's L-BFGS-B (C port of L-BFGS-B 3.0), unbounded case, restated operation by operation ------------
 * scipy is a third-party dependency of the reference (call site EP:213-225; not vendored, not pinned by the reference:
 * README.md:43). Its compiled module calls BLAS/LAPACK from the bundled OpenBLAS 0.3.31 (SkylakeX kernels on the build
 * machine); the routines below restate the arithmetic of exactly those kernels for the sizes that occur here (vectors of
 * n <= 31, triangular systems of order <= 20), so that -- fed the same (f, g) values -- this file walks through the same
 * iterates as scipy BIT FOR BIT. Pinned by tests/test_oracle_golden.py::test_lbfgsb_restatement_bit_identical_to_scipy
 * (reference-identical Python f/g driven through scipy.optimize.minimize and through orc_lbfgsb_cb).
 * How each rule was established (against scipy.optimize._lbfgsb.setulb's workspace, call by call) is recorded in
 * DESIGN.md section 3. The file is compiled with -ffp-contract=off: every fused multiply-add below is an explicit fma().
 *   ddot   n < 16: s = fma(a_i, b_i, s) in index order. 16 <= n < 32: the first 16 products are rounded, added in four
 *          lanes ((p_l + p_l+4) + p_l+8) + p_l+12, folded (v0 + v2) + (v1 + v3); the rest continues with fma.
 *   dnrm2  x87 kernel: squares and their sum in 80-bit extended precision, fsqrt, rounded to double once at the end.
 *   dpotrf (potf2_U): diagonal a_jj - ddot, sqrt; row to the right y_i -= sum_k a_ki a_kj in the order of the dgemv_t
 *          kernel (blocks of four rows in lanes, (l0 + l2) + (l1 + l3); 1-3 leftover rows folded as below); times 1/a_jj.
 *   dtrtrs one right-hand side -> trsv: transposed: (b_i - ddot) / u_ii; not transposed: b_i / u_ii, then fma axpy.
 *          several right-hand sides -> trsm kernel: blocks of 8, 4, 2, 1 rows; per block first b_i -= sum over the rows
 *          of earlier blocks (fma from zero), then inside the block b_i *= 1/u_ii and b_k = fma(-b_i, u_ik, b_k).
 *   loops written out in scipy's own C (formk's inner products, subsm, the projected gradient) are plain mul + add. */
static double blas_ddot(int n, const double *a, int sa, const double *b, int sb)
{
    double s = 0.0;
    int i = 0;
    if (n >= 16) {
        double v[4];
        for (int l = 0; l < 4; l++)
            v[l] = ((a[l * sa] * b[l * sb] + a[(4 + l) * sa] * b[(4 + l) * sb]) + a[(8 + l) * sa] * b[(8 + l) * sb]) +
                   a[(12 + l) * sa] * b[(12 + l) * sb];
        s = (v[0] + v[2]) + (v[1] + v[3]);
        i = 16;
    }
    for (; i < n; i++) s = fma(a[i * sa], b[i * sb], s);
    return s;
}

/* OpenBLAS 0.3.31 dnrm2_k (x86_64 nrm2.S, the kernel every x86_64 target of scipy's bundled library uses; disassembled
 * from scipy.libs: dnrm2_k_SKYLAKEX): x87 arithmetic in 80-bit extended precision. Four accumulators: blocks of 8
 * elements feed element i to accumulator i mod 4, the remaining n mod 8 elements all go to accumulator 0, and the sum is
 * D + ((C + A) + B) before fsqrt and the rounding to double. For n < 8 this is the plain sequential sum. */
static double blas_dnrm2(int n, const double *a)
{
    long double acc[4] = {0.0L, 0.0L, 0.0L, 0.0L};
    const int nb = n >> 3;
    for (int i = 0; i < 8 * nb; i++) { const long double v = a[i]; acc[i & 3] += v * v; }
    for (int i = 8 * nb; i < n; i++) { const long double v = a[i]; acc[0] += v * v; }
    const long double s = acc[3] + ((acc[2] + acc[0]) + acc[1]);
    return (double)sqrtl(s);
}

#define LB_M ORC_HIST
#define LB_W (2 * LB_M)
/* upper-triangular factor in a[o..o+n)[o..o+n) of the LB_W x LB_W row-major array; 0 if not positive definite */
static int lapack_potf2(double (*a)[LB_W], int o, int n)
{
    for (int j = 0; j < n; j++) {
        double ajj = a[o + j][o + j] - blas_ddot(j, &a[o][o + j], LB_W, &a[o][o + j], LB_W);
        if (!(ajj > 0.0)) return 0;
        ajj = sqrt(ajj);
        a[o + j][o + j] = ajj;
        if (j == n - 1) break;
        const int m1 = j & ~3, k3 = j - m1;
        for (int i = j + 1; i < n; i++) {
#define COL(k) a[o + (k)][o + i]
#define XJ(k) a[o + (k)][o + j]
            double v = a[o + j][o + i];
            if (m1) {
                double acc[4];
                for (int l = 0; l < 4; l++) acc[l] = COL(l) * XJ(l);
                if (m1 == 8) for (int l = 0; l < 4; l++) acc[l] = acc[l] + COL(4 + l) * XJ(4 + l);
                v = v - ((acc[0] + acc[2]) + (acc[1] + acc[3]));
            }
            if (k3 == 1) v = fma(COL(m1), -XJ(m1), v);
            else if (k3 == 2) v = v + fma(COL(m1), -XJ(m1), COL(m1 + 1) * -XJ(m1 + 1));
            else if (k3 == 3) v = v + fma(COL(m1 + 2), -XJ(m1 + 2), fma(COL(m1), -XJ(m1), COL(m1 + 1) * -XJ(m1 + 1)));
            a[o + j][o + i] = v;
#undef COL
#undef XJ
        }
        const double r = 1.0 / ajj;
        for (int i = j + 1; i < n; i++) a[o + j][o + i] = a[o + j][o + i] * r;
    }
    return 1;
}

/* u = a[0..n)[0..n) upper. b: contiguous vector. */
static void blas_trsv_T(double (*u)[LB_W], int n, double *b)
{
    for (int i = 0; i < n; i++) {
        if (i > 0) b[i] = b[i] - blas_ddot(i, &u[0][i], LB_W, b, 1);
        b[i] = b[i] / u[i][i];
    }
}

static void blas_trsv_N(double (*u)[LB_W], int n, double *b)
{
    for (int i = n - 1; i >= 0; i--) {
        b[i] = b[i] / u[i][i];
        const double t = -b[i];
        for (int k = 0; k < i; k++) b[k] = fma(t, u[k][i], b[k]);
    }
}

/* u^T X = B for the nrhs >= 2 columns c0.. of the same array (rows 0..n-1), n <= 15 */
static void blas_trsm_LT(double (*a)[LB_W], int n, int c0, int nrhs)
{
    for (int c = c0; c < c0 + nrhs; c++) {
        int kk = 0;
        for (int bs = 8; bs > 0; bs >>= 1) {
            if (!(n & bs)) continue;
            if (kk > 0)
                for (int i = kk; i < kk + bs; i++) {
                    double acc = 0.0;
                    for (int k = 0; k < kk; k++) acc = fma(a[k][i], a[k][c], acc);
                    a[i][c] = a[i][c] - acc;
                }
            for (int i = kk; i < kk + bs; i++) {
                a[i][c] = a[i][c] * (1.0 / a[i][i]);
                for (int k = i + 1; k < kk + bs; k++) a[k][c] = fma(-a[i][c], a[i][k], a[k][c]);
            }
            kk += bs;
        }
    }
}

/* limited-memory matrices (all variables free): pairs oldest first */
typedef struct {
    int n, col, iupdat;
    double theta;
    double ws[LB_M][ORC_MAXN], wy[LB_M][ORC_MAXN];
    double dr[LB_M];                 /* diagonal of S'Y as stored by matupd: (gd - gdold) * stp */
    double yy[LB_M][LB_M];           /* formk's wn1 block (1,1): Y'Y, lower triangle */
    double rz[LB_M][LB_M];           /* formk's wn1 block (2,1): upper triangle of S'Y (its own inner products) */
    double wn[LB_W][LB_W];           /* the factored middle matrix */
} lb_mem;

static double loop_dot(int n, const double *a, const double *b) { double s = 0.0; for (int i = 0; i < n; i++) s = s + a[i] * b[i]; return s; }

static void lb_reset(lb_mem *C, int n) { C->n = n; C->col = 0; C->iupdat = 0; C->theta = 1.0; }

static void lb_update(lb_mem *C, const double *s, const double *y, double rr, double dr)
{
    const int n = C->n;
    C->iupdat++;
    if (C->iupdat <= LB_M) C->col = C->iupdat;
    else {
        OC(OC_WRAP);
        memmove(C->ws[0], C->ws[1], sizeof(double) * (LB_M - 1) * ORC_MAXN);
        memmove(C->wy[0], C->wy[1], sizeof(double) * (LB_M - 1) * ORC_MAXN);
        for (int j = 0; j < LB_M - 1; j++) {
            C->dr[j] = C->dr[j + 1];
            for (int i = j; i < LB_M - 1; i++) C->yy[i][j] = C->yy[i + 1][j + 1];
            for (int i = 0; i < LB_M - 1; i++) C->rz[i][j] = C->rz[i + 1][j + 1];
        }
    }
    const int col = C->col;
    memcpy(C->ws[col - 1], s, sizeof(double) * n); memcpy(C->wy[col - 1], y, sizeof(double) * n);
    C->theta = rr / dr;
    C->dr[col - 1] = dr;
    for (int j = 0; j < col; j++) C->yy[col - 1][j] = loop_dot(n, C->wy[col - 1], C->wy[j]);
    for (int i = 0; i < col; i++) C->rz[i][col - 1] = loop_dot(n, C->ws[i], C->wy[col - 1]);
}

/* formk: assemble and factor; 0 if a Cholesky factorisation fails (scipy then drops the memory) */
static int lb_factor(lb_mem *C)
{
    const int col = C->col;
    const double theta = C->theta;
    double (*wn)[LB_W] = C->wn;
    for (int iy = 0; iy < col; iy++) {
        const int is = col + iy;
        for (int jy = 0; jy <= iy; jy++) { wn[jy][iy] = C->yy[iy][jy] / theta; wn[col + jy][is] = 0.0 * theta; }
        for (int jy = 0; jy < iy; jy++) wn[jy][is] = -0.0;
        for (int jy = iy; jy < col; jy++) wn[jy][is] = C->rz[iy][jy];
        wn[iy][iy] = wn[iy][iy] + C->dr[iy];
    }
    if (!lapack_potf2(wn, 0, col)) { OC(OC_FACTOR_FAIL1); return 0; }
    if (col == 1) wn[0][1] = wn[0][1] / wn[0][0];        /* one right-hand side: trsv */
    else blas_trsm_LT(wn, col, col, col);
    for (int is = col; is < 2 * col; is++)
        for (int js = is; js < 2 * col; js++)
            wn[is][js] = wn[is][js] + blas_ddot(col, &wn[0][is], LB_W, &wn[0][js], LB_W);
    if (!lapack_potf2(wn, col, col)) { OC(OC_FACTOR_FAIL2); return 0; }
    return 1;
}

/* subsm with r = -g: the subspace step (added to x by the caller) */
static void lb_step(lb_mem *C, const double *g, double *d)
{
    const int col = C->col, n = C->n;
    const double theta = C->theta;
    double wv[LB_W];
    for (int i = 0; i < n; i++) d[i] = -g[i];
    for (int i = 0; i < col; i++) { wv[i] = loop_dot(n, C->wy[i], d); wv[col + i] = theta * loop_dot(n, C->ws[i], d); }
    blas_trsv_T(C->wn, 2 * col, wv);
    for (int i = 0; i < col; i++) wv[i] = -wv[i];
    blas_trsv_N(C->wn, 2 * col, wv);
    for (int jy = 0; jy < col; jy++)
        for (int i = 0; i < n; i++) d[i] = d[i] + C->wy[jy][i] * wv[jy] / theta + C->ws[jy][i] * wv[col + jy];
    const double it = 1.0 / theta;
    for (int i = 0; i < n; i++) d[i] = d[i] * it;
}

typedef struct {
    double x[ORC_MAXN];
    double costs[4];      /* costs at the last evaluated trial point (EP:233 reads self.costs) */
    double f;
    int status, nit, nfev;
} orc_result;

/* f, g (and the four unweighted cost terms) at x; returns 0 or the status the reference's exception maps to */
typedef int (*orc_fg_fn)(void *ctx, int n, const double *x, double *f, double *g, double *costs);
enum { ORC_REPLAY_DIVERGED = 8 };

/* Optional recording of every evaluation (x, f, g) of the running minimize() call, for the lockstep tests. */
typedef struct { int cap, len; double *x, *f, *g; } orc_trace;
static __thread orc_trace *orc_trace_cur = 0;

/* plan_once's minimize() call: tol=1e-4 -> ftol = gtol = 1e-4; maxcor 10; maxls 20; maxiter = maxfun = 15000. */
static int lbfgsb_run(int n, const double *x0, orc_fg_fn fg, void *ctx, orc_result *out)
{
    const int maxls = 20, maxiter = 15000, maxfun = 15000;
    const double pgtol = 1e-4, ftol = 1e-4, epsmch = DBL_EPSILON;
    const double tol = (ftol / epsmch) * epsmch;
    double x[ORC_MAXN], g[ORC_MAXN], d[ORC_MAXN], z[ORC_MAXN], t[ORC_MAXN], r[ORC_MAXN], xl[ORC_MAXN], xn[ORC_MAXN];
    double costs[4] = {0, 0, 0, 0}, f = 0.0, fold;
    int nit = 0, nfev = 0, st;
    static __thread lb_mem C;
    lb_reset(&C, n);
    memcpy(x, x0, sizeof(double) * n);
#define LB_EVAL()                                                                                              \
    do {                                                                                                       \
        st = fg(ctx, n, x, &f, g, costs);                                                                      \
        if (st) {                                                                                              \
            if (st >= ORC_OVERFLOW && st <= ORC_NAN) OC(OC_EVAL_OVERFLOW + st - ORC_OVERFLOW);                  \
            out->status = st; out->nit = nit; out->nfev = nfev; memcpy(out->x, x, sizeof(double) * n); return st; \
        }                                                                                                      \
        nfev++; memcpy(xl, x, sizeof(double) * n); memcpy(out->costs, costs, sizeof(costs));                    \
        if (orc_trace_cur && orc_trace_cur->len < orc_trace_cur->cap) {                                        \
            orc_trace *T = orc_trace_cur;                                                                      \
            memcpy(T->x + (size_t)T->len * n, x, sizeof(double) * n); memcpy(T->g + (size_t)T->len * n, g, sizeof(double) * n); \
            T->f[T->len++] = f;                                                                                \
        }                                                                                                      \
    } while (0)
    LB_EVAL();
    double sbg = 0.0; for (int i = 0; i < n; i++) sbg = fmax(sbg, fabs(g[i]));
    if (sbg <= pgtol) { st = ORC_CONV_PG; OC(OC_PG_X0); goto done; }
    for (;;) {
        /* search direction: Cauchy point x - g with an empty memory (theta = 1), else the subspace step; d = z - x */
        if (C.col == 0) for (int i = 0; i < n; i++) z[i] = x[i] - g[i];
        else {
            if (!lb_factor(&C)) { if (C.iupdat > LB_M) OC(OC_RESET_AFTER_WRAP); lb_reset(&C, n); continue; }
            lb_step(&C, g, d);
            for (int i = 0; i < n; i++) z[i] = x[i] + d[i];
        }
        for (int i = 0; i < n; i++) d[i] = z[i] - x[i];
        OC(OC_DIR + C.col);
        /* lnsrlb */
        const double dnorm = blas_dnrm2(n, d);
        double stp = (nit == 0) ? fmin(1.0 / dnorm, LS_STPMAX) : 1.0;
        memcpy(t, x, sizeof(double) * n); memcpy(r, g, sizeof(double) * n); fold = f;
        double gd = blas_ddot(n, g, 1, d, 1), gdold = gd;
        int fail = 0;
        if (gd >= 0.0) { fail = 1; OC(C.col == 0 ? OC_NONDESCENT_COL0 : OC_NONDESCENT_COL); }
        else {
            dcs_state ls; dcsrch_start(&ls, stp, f, gd);
            int ifun = 0;
            for (;;) {
                ifun++;
                if (ifun - 1 >= maxls) { fail = 1; OC(OC_MAXLS); break; }
                if (stp == 1.0) memcpy(xn, z, sizeof(double) * n);
                else for (int i = 0; i < n; i++) xn[i] = stp * d[i] + t[i];
                int same = 1; for (int i = 0; i < n; i++) if (xn[i] != xl[i]) { same = 0; break; }
                memcpy(x, xn, sizeof(double) * n);
                if (!same) LB_EVAL();          /* scipy's ScalarFunction does not re-evaluate an unchanged x */
                else OC(OC_CACHE_HIT);
                gd = blas_ddot(n, g, 1, d, 1);
                if (dcsrch_step(&ls, &stp, f, gd)) break;
            }
        }
        if (fail) {
            memcpy(x, t, sizeof(double) * n); memcpy(g, r, sizeof(double) * n); f = fold;
            if (C.col == 0) { st = ORC_ABNORMAL; OC(OC_ABNORMAL); goto done; }
            OC(OC_RESET_FAILED);
            if (C.iupdat > LB_M) OC(OC_RESET_AFTER_WRAP);
            lb_reset(&C, n);
            continue;
        }
        nit++;
        OC(stp == 1.0 ? OC_ACCEPT_STP1 : OC_ACCEPT_STP);
        sbg = 0.0; for (int i = 0; i < n; i++) sbg = fmax(sbg, fabs(g[i]));
        if (sbg <= pgtol) { st = ORC_CONV_PG; OC(OC_PG); goto done; }
        { const double dd = fmax(fmax(fabs(fold), fabs(f)), 1.0); if (fold - f <= tol * dd) { st = ORC_CONV_FTOL; OC(OC_FTOL); goto done; } }
        if (nit >= maxiter || nfev > maxfun) { st = ORC_MAXITER; OC(OC_MAXITER); goto done; }
        /* BFGS update (matupd) */
        double rr, dr, ddum;
        for (int i = 0; i < n; i++) r[i] = g[i] - r[i];
        { const double nr = blas_dnrm2(n, r); rr = nr * nr; }
        if (stp == 1.0) { dr = gd - gdold; ddum = -gdold; }
        else { dr = (gd - gdold) * stp; for (int i = 0; i < n; i++) d[i] = d[i] * stp; ddum = -gdold * stp; }
        if (dr <= epsmch * ddum) { OC(OC_SKIP_UPDATE); continue; }   /* skip the update */
        lb_update(&C, d, r, rr, dr);
    }
done:
    memcpy(out->x, x, sizeof(double) * n);
    out->f = f; out->status = st; out->nit = nit; out->nfev = nfev;
    return st;
#undef LB_EVAL
}

/* evaluator = this file's orc_eval */
typedef struct { const orc_params *p; const orc_map *map; int M; const double *head, *tail; } fg_problem;
static int fg_oracle(void *ctx, int n, const double *x, double *f, double *g, double *costs)
{
    (void)n;
    const fg_problem *q = (const fg_problem *)ctx;
    const int st = orc_eval(q->p, q->map, q->M, q->head, q->tail, x, costs, g, 0, 0);
    if (st) return st;
    *f = costs[0] * q->p->w[0] + costs[1] * q->p->w[1] + costs[2] * q->p->w[2] + costs[3] * q->p->w[3];
    return 0;
}

int orc_lbfgsb(const orc_params *p, const orc_map *map, int M, const double *head, const double *tail,
               const double *x0, orc_result *out)
{
    fg_problem q = {p, map, M, head, tail};
    return lbfgsb_run(ORC_D * (M - 1) + M, x0, fg_oracle, &q, out);
}

/* the same optimizer around a caller-supplied evaluator (tests: the reference's own Python get_cost/get_grad) */
int orc_lbfgsb_cb(int n, const double *x0, orc_fg_fn fg, void *ctx, orc_result *out) { return lbfgsb_run(n, x0, fg, ctx, out); }
/* the restated BLAS norm alone (tests/test_x87_nrm2.py pins it to scipy's bundled kernel) */
double orc_dnrm2(int n, const double *a) { return blas_dnrm2(n, a); }
/* ... and the two inner products (the BLAS kernel's order, and scipy's own loops) */
double orc_ddot(int n, const double *a, const double *b) { return blas_ddot(n, a, 1, b, 1); }
double orc_loop_dot(int n, const double *a, const double *b) { return loop_dot(n, a, b); }

/* ... with every evaluation recorded: x (cap, n), f (cap), g (cap, n); returns the number of evaluations recorded */
int orc_lbfgsb_traced(const orc_params *p, const orc_map *map, int M, const double *head, const double *tail,
                      const double *x0, orc_result *out, int cap, double *xs, double *fs, double *gs)
{
    orc_trace T = {cap, 0, xs, fs, gs};
    orc_trace_cur = &T;
    orc_lbfgsb(p, map, M, head, tail, x0, out);
    orc_trace_cur = 0;
    return T.len;
}

/* Lockstep replay: the optimizer above is fed evaluations recorded elsewhere (the device's). Evaluation k must be
 * requested at exactly xs[k] (bitwise); it then returns fs[k], gs[k], costs[k], status[k]. If the requested point
 * differs, the run stops with ORC_REPLAY_DIVERGED and *first_bad = k. Identical requests all the way prove that the
 * recorded run and this optimizer made the same decisions from the same numbers. */
typedef struct { int n_evals, k, bad; const double *xs, *fs, *gs, *costs; const int32_t *status; } fg_replay;
static int fg_from_trace(void *ctx, int n, const double *x, double *f, double *g, double *costs)
{
    fg_replay *q = (fg_replay *)ctx;
    const int k = q->k;
    if (k >= q->n_evals || memcmp(x, q->xs + (size_t)k * n, sizeof(double) * n)) { q->bad = k; return ORC_REPLAY_DIVERGED; }
    q->k++;
    *f = q->fs[k]; memcpy(g, q->gs + (size_t)k * n, sizeof(double) * n); memcpy(costs, q->costs + (size_t)k * 4, sizeof(double) * 4);
    return q->status ? q->status[k] : 0;
}

int orc_lbfgsb_replay(int n, const double *x0, int n_evals, const double *xs, const double *fs, const double *gs,
                      const double *costs, const int32_t *status, orc_result *out, int *first_bad, int *used)
{
    fg_replay q = {n_evals, 0, -1, xs, fs, gs, costs, status};
    const int st = lbfgsb_run(n, x0, fg_from_trace, &q, out);
    *first_bad = q.bad; *used = q.k;
    return st;
}

/* ------------------------------------------------------------------------------------------ */
/* plan_once / warm_start_plan: EP:186-237                                                     */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
    double x[ORC_MAXN];        /* final decision vector of the accepted attempt */
    double ts[ORC_MAXM];
    double coeffs[ORC_MAXR * ORC_D];
    double costs[4];           /* unweighted, at the last evaluated point (EP:233) */
    int status;                /* status of the last attempt run */
    int ok;                    /* 1: an attempt passed the collision test; 0: "No solution" */
    int attempt;               /* index of the accepted (or last) attempt */
    int nit;                   /* sum of nit over attempts whose minimize() returned (EP:230) */
    int runs;                  /* opt_running_times increment (EP:232) */
    int nfev;                  /* total cost+grad evaluations over all attempts */
} orc_plan;

/* one plan_once: returns 1 if accepted, 0 if it raised (any reason). q0 (D, M-1), ts0 (M) */
static int plan_once(const orc_params *p, const orc_map *map, int M, const double *head, const double *tail,
                     const double *q0, const double *ts0, orc_plan *out)
{
    int nq = ORC_D * (M - 1), n = nq + M;
    double x0[ORC_MAXN];
    orc_result res;
    memcpy(x0, q0, sizeof(double) * nq);
    int st = orc_T2tau(p, M, ts0, x0 + nq);
    if (st) { out->status = st; return 0; }
    st = orc_lbfgsb(p, map, M, head, tail, x0, &res);
    out->nfev += res.nfev;
    out->status = st;
    if (st >= ORC_OVERFLOW) return 0;                 /* exception propagated out of minimize() */
    memcpy(out->x, res.x, sizeof(double) * n);
    if (orc_tau2T(p, M, res.x + nq, out->ts)) { out->status = ORC_OVERFLOW; return 0; }
    out->nit += res.nit; out->runs += 1;
    memcpy(out->costs, res.costs, sizeof(res.costs));
    return !(res.costs[3] * p->w[3] > p->collision_cost_tol);
}

/* warm_start_plan (EP:186-203): attempt 0 from (q0, ts0); attempt a >= 1 restarts from retry_q[a-1]
 * (D, M-1) = straight line + host-drawn N(0, 0.5) noise (EP:92-94, EP:200) with ts = retry_ts (EP:97-99). */
int orc_warm_start_plan(const orc_params *p, const orc_map *map, int M, const double *head, const double *tail,
                        const double *q0, const double *ts0, const double *retry_q, const double *retry_ts,
                        int max_attempts, orc_plan *out)
{
    double q[ORC_D * ORC_MAXM], ts[ORC_MAXM];
    memset(out, 0, sizeof(*out));
    memcpy(q, q0, sizeof(double) * ORC_D * (M - 1)); memcpy(ts, ts0, sizeof(double) * M);
    for (int a = 0; a < max_attempts; a++) {
        out->attempt = a;
        if (plan_once(p, map, M, head, tail, q, ts, out)) { out->ok = 1; break; }
        if (a + 1 < max_attempts) {
            memcpy(q, retry_q + (size_t)a * ORC_D * (M - 1), sizeof(double) * ORC_D * (M - 1));
            memcpy(ts, retry_ts, sizeof(double) * M);
        }
    }
    if (out->runs > 0) {   /* coefficients of the final (int_wpts, ts), as get_full_state_cmd recomputes them (TU:182) */
        double LU[ORC_MAXR * ORC_MAXR]; int piv[ORC_MAXR];
        solve_coeffs(M, head, tail, out->x, out->ts, LU, piv, out->coeffs);
    }
    return out->ok;
}

/* batch entry used by the tests and the CPU-baseline timer */
void orc_plan_batch(const orc_params *p, const orc_map *map, int B, int M, const double *head, const double *tail,
                    const double *q0, const double *ts0, const double *retry_q, const double *retry_ts,
                    int max_attempts, double *x, double *ts, double *coeffs, double *costs, int32_t *status, int32_t *ok,
                    int32_t *attempt, int32_t *nit, int32_t *runs, int32_t *nfev)
{
    int nq = ORC_D * (M - 1), n = nq + M;
    for (int b = 0; b < B; b++) {
        orc_plan pl;
        orc_warm_start_plan(p, map, M, head + (size_t)b * 3 * ORC_D, tail + (size_t)b * 3 * ORC_D,
                            q0 + (size_t)b * nq, ts0 + (size_t)b * M,
                            retry_q ? retry_q + (size_t)b * (max_attempts - 1) * nq : 0, retry_ts, max_attempts, &pl);
        memcpy(x + (size_t)b * n, pl.x, sizeof(double) * n);
        memcpy(ts + (size_t)b * M, pl.ts, sizeof(double) * M);
        memcpy(coeffs + (size_t)b * 6 * M * ORC_D, pl.coeffs, sizeof(double) * 6 * M * ORC_D);
        memcpy(costs + (size_t)b * 4, pl.costs, sizeof(double) * 4);
        status[b] = pl.status; ok[b] = pl.ok; attempt[b] = pl.attempt; nit[b] = pl.nit; runs[b] = pl.runs; nfev[b] = pl.nfev;
    }
}

/* the same batch on `threads` host threads (problems are independent; interleaved assignment). Used by the full-size
 * parity sweeps and as the all-core CPU yardstick of bench.py. */
#include <pthread.h>
typedef struct {
    const orc_params *p; const orc_map *const *maps; const int32_t *map_ids; int B, M, first, stride, max_attempts;
    const double *head, *tail, *q0, *ts0, *retry_q, *retry_ts;
    double *x, *ts, *coeffs, *costs; int32_t *status, *ok, *attempt, *nit, *runs, *nfev;
} mt_job;
static void *mt_worker(void *arg)
{
    const mt_job *j = (const mt_job *)arg;
    const int M = j->M, nq = ORC_D * (M - 1), n = nq + M;
    for (int b = j->first; b < j->B; b += j->stride) {
        orc_plan pl;
        const orc_map *map = j->maps[j->map_ids ? j->map_ids[b] : 0];
        orc_warm_start_plan(j->p, map, M, j->head + (size_t)b * 3 * ORC_D, j->tail + (size_t)b * 3 * ORC_D,
                            j->q0 + (size_t)b * nq, j->ts0 + (size_t)b * M,
                            j->retry_q ? j->retry_q + (size_t)b * (j->max_attempts - 1) * nq : 0, j->retry_ts, j->max_attempts, &pl);
        memcpy(j->x + (size_t)b * n, pl.x, sizeof(double) * n);
        memcpy(j->ts + (size_t)b * M, pl.ts, sizeof(double) * M);
        memcpy(j->coeffs + (size_t)b * 6 * M * ORC_D, pl.coeffs, sizeof(double) * 6 * M * ORC_D);
        memcpy(j->costs + (size_t)b * 4, pl.costs, sizeof(double) * 4);
        j->status[b] = pl.status; j->ok[b] = pl.ok; j->attempt[b] = pl.attempt; j->nit[b] = pl.nit; j->runs[b] = pl.runs;
        j->nfev[b] = pl.nfev;
    }
    return 0;
}
void orc_plan_batch_mt(const orc_params *p, const orc_map *const *maps, const int32_t *map_ids, int B, int M,
                       const double *head, const double *tail, const double *q0, const double *ts0, const double *retry_q,
                       const double *retry_ts, int max_attempts, int threads, double *x, double *ts, double *coeffs,
                       double *costs, int32_t *status, int32_t *ok, int32_t *attempt, int32_t *nit, int32_t *runs, int32_t *nfev)
{
    if (threads < 1) threads = 1;
    if (threads > 256) threads = 256;
    pthread_t th[256];
    mt_job jobs[256];
    for (int t = 0; t < threads; t++) {
        mt_job j = {p, maps, map_ids, B, M, t, threads, max_attempts, head, tail, q0, ts0, retry_q, retry_ts,
                    x, ts, coeffs, costs, status, ok, attempt, nit, runs, nfev};
        jobs[t] = j;
        pthread_create(&th[t], 0, mt_worker, &jobs[t]);
    }
    for (int t = 0; t < threads; t++) pthread_join(th[t], 0);
}

/* batched eval used by the parity tests */
void orc_eval_batch(const orc_params *p, const orc_map *map, int B, int M, const double *head, const double *tail,
                    const double *x, double *costs, double *grad, int32_t *status)
{
    int n = ORC_D * (M - 1) + M;
    for (int b = 0; b < B; b++)
        status[b] = orc_eval(p, map, M, head + (size_t)b * 3 * ORC_D, tail + (size_t)b * 3 * ORC_D,
                             x + (size_t)b * n, costs + (size_t)b * 4, grad + (size_t)b * n, 0, 0);
}

/* ------------------------------------------------------------------------------------------ */
/* trajectory sampling: TU:85-195                                                              */
/* ------------------------------------------------------------------------------------------ */
/* get_pos/get_vel/get_acc at absolute time t (TU:85-157): piece located with cumulative sums; t beyond
 * the end clamps to sum(ts). out: (3, D) = pos, vel, acc. */
void orc_state_at(int M, const double *coeffs, const double *ts, double t, double *out)
{
    double total = 0.0;
    for (int i = 0; i < M; i++) total += ts[i];
    if (t > total) t = total;
    int piece = 0;
    double acc_t = ts[0];     /* sum(ts[:piece+1]) */
    while (acc_t < t) { piece++; acc_t += ts[piece]; }
    double before = 0.0;
    for (int i = 0; i < piece; i++) before += ts[i];
    double T = t - before;
    double T2 = T * T, T3 = pow(T, 3), T4 = pow(T, 4), T5 = pow(T, 5);
    double b0[6] = {1, T, T2, T3, T4, T5};
    double b1[6] = {0, 1, 2 * T, 3 * T2, 4 * T3, 5 * T4};
    double b2[6] = {0, 0, 2, 6 * T, 12 * T2, 20 * T3};
    const double *c = coeffs + 6 * piece * ORC_D;
    for (int d = 0; d < ORC_D; d++) {
        double sp = 0, sv = 0, sa = 0;
        for (int k = 0; k < 6; k++) { sp += c[k * ORC_D + d] * b0[k]; sv += c[k * ORC_D + d] * b1[k]; sa += c[k * ORC_D + d] * b2[k]; }
        out[0 * ORC_D + d] = sp; out[1 * ORC_D + d] = sv; out[2 * ORC_D + d] = sa;
    }
}

/* number of samples of np.arange(0, total, 1/hz) = ceil(total / step) (numpy's _arange_safe_ceil_to_intp) */
int orc_sample_count(int M, const double *ts, double hz)
{
    double total = 0.0;
    for (int i = 0; i < M; i++) total += ts[i];
    double step = 1.0 / hz;
    return (int)ceil((total - 0.0) / step);
}

/* get_full_state_cmd (TU:181-195): states (N, 3, D) at t_k = k * (1/hz) */
void orc_sample(int M, const double *coeffs, const double *ts, double hz, int N, double *states)
{
    double step = 1.0 / hz;
    for (int k = 0; k < N; k++) orc_state_at(M, coeffs, ts, k * step, states + (size_t)k * 3 * ORC_D);
}
