/*
 * neoopt.h -- C ABI of libneoopt.so: the B200 (sm_100a) batched MINCO trajectory optimizer that
 * replaces the hot path of NEO-Planner's Python optimizer. Plain pointers and sizes only; no torch
 * types. A reference maintainer binds these with ctypes (see INTEGRATION.md).
 *
 * Reference interfaces replaced (paths relative to the reference repo root):
 *   EP   = src/planner/scripts/traj_planner/expert_planner.py
 *   TU   = src/planner/scripts/traj_planner/traj_utils.py
 *   ESDF = src/planner/scripts/map_server/esdf.py
 *
 * Conventions
 *   D = 2 (planar; EP:416, ESDF:26), s = 3 (minimum jerk; EP:36), 2 <= M <= NEO_MAX_PIECES pieces.
 *   Decision vector x[n], n = 2(M-1)+M: [q_x(0..M-2), q_y(0..M-2), tau(0..M-1)]            (EP:211)
 *   head/tail: (3,2) row-major = pos, vel, acc; callers zero-pad missing rows              (EP:170-184)
 *   q (int_wpts): (2, M-1) row-major; ts: (M); coeffs: (6M, 2) row-major, row 6i+k = t^k of piece i (EP:261-336)
 *   All floating point data is IEEE fp64. All arrays are caller-owned; nothing is retained after
 *   return except uploaded maps (library-owned device copies).
 *   Return value: 0 on success, <0 = NEO_ERR_* (text via neo_last_error). Per-problem outcomes are
 *   reported in `status` arrays (NEO_ST_*), never as a failing return code.
 *   Thread safety: calls on one handle are serialised by an internal mutex; handles are independent.
 *   Functions ending in _dev take DEVICE pointers and enqueue on `stream` (a cudaStream_t passed as
 *   void*; NULL = the handle's own stream, cudaStreamLegacy = the legacy default stream) without synchronising. A handle owns ONE set of scratch buffers
 *   (work-queue counter, per-attempt records): consecutive _dev launches on the same handle must be ordered on the
 *   same stream, and maps must not be re-uploaded while a launch is in flight. Use one handle per concurrent stream.
 *   map_ids passed to host-pointer entry points are validated (every id must name a slot that holds a map, else
 *   NEO_ERR_INVALID); for _dev entry points that is a precondition (the ids are in device memory).
 *   Kernel selection: problems with M <= 4 pieces run one per warp below NEO_TILE_MIN_PROBLEMS (12288) problems per call
 *   and 4 (M <= 3) or 2 (M = 4) per warp from there on (one CTA per SM whose warps start their evaluations in groups);
 *   results of the two schedules differ in the last bits of the sampled sums (different partial-sum order), never in
 *   the algorithm. Development switches read from the environment at neo_create (A/B measurements, parity tests):
 *   NEO_TILE = 8 | 16 | 32 pins the lanes per problem, NEO_GROUPED = 0 turns the grouped starts off, NEO_GROUP_WARPS
 *   sets the group size.
 */
#ifndef NEOOPT_H
#define NEOOPT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NEO_MAX_PIECES 10
#define NEO_MAX_ATTEMPTS 8

/* API errors */
#define NEO_OK 0
#define NEO_ERR_INVALID (-1)     /* bad argument (M out of range, null pointer, no map, ...) */
#define NEO_ERR_CUDA (-2)        /* CUDA runtime error; see neo_last_error */
#define NEO_ERR_NO_DEVICE (-3)   /* no usable sm_100 device: this library has no CPU fallback */

/* per-problem status of the last optimisation attempt (EP:205-237 + scipy L-BFGS-B task messages) */
#define NEO_ST_CONV_FTOL 0   /* CONVERGENCE: REL_REDUCTION_OF_F <= FACTR*EPSMCH */
#define NEO_ST_CONV_PG 1     /* CONVERGENCE: NORM_OF_PROJECTED_GRADIENT <= PGTOL */
#define NEO_ST_ABNORMAL 2    /* ABNORMAL_TERMINATION_IN_LNSRCH (result still used, as scipy returns it) */
#define NEO_ST_MAXITER 3     /* maxiter / maxfun = 15000 reached */
#define NEO_ST_OVERFLOW 4    /* OverflowError raised by math.exp / float pow (EP:481, EP:489-490) */
#define NEO_ST_DOMAIN 5      /* ValueError / ZeroDivisionError in map_T2tau: ts outside (T_min, T_max) (EP:474) */
#define NEO_ST_NAN 6         /* ValueError: int(nan) in the sample loop / ESDF lookup (EP:401, ESDF:61) */

/* a1: parameter struct = DefaultConfig (EP:12-25) / planner_config.yaml:2-13 */
typedef struct {
    double v_max;
    double T_min;
    double T_max;
    double safe_dis;
    double delta_t;
    double weights[4];          /* energy, time, feasibility, collision */
    double collision_cost_tol;
} neo_config;

typedef struct neo_handle neo_handle;

/* lifecycle ---------------------------------------------------------------------------------- */
/* MinJerkPlanner.__init__ (EP:33-60). `device` = CUDA ordinal. `max_maps` = number of map slots. */
int neo_create(const neo_config *cfg, int device, int max_maps, neo_handle **out);
int neo_destroy(neo_handle *h);
int neo_set_config(neo_handle *h, const neo_config *cfg);
const char *neo_last_error(neo_handle *h);   /* h may be NULL: error of the last failed neo_create */
int neo_device_info(neo_handle *h, int *sm_count, int *cc_major, int *cc_minor, char *name, int name_len);

/* maps ----------------------------------------------------------------------------------------- */
/* Upload the three arrays an ESDF object holds (ESDF:29-33): esdf_map, esdf_grad_x, esdf_grad_y, each
 * (H, W) row-major (row = y, col = x). */
int neo_set_map_esdf(neo_handle *h, int slot, int H, int W, double res, double ox, double oy,
                     const double *esdf, const double *gx, const double *gy);
/* ESDF.occupancy_map_cb (ESDF:11-33) on the device: occ = raw OccupancyGrid data (int8, 100 = occupied,
 * everything else free), exact Euclidean distance transform * res, np.gradient central differences.
 * Bit-exact with scipy.ndimage.distance_transform_edt + numpy.gradient. */
int neo_set_map_occupancy(neo_handle *h, int slot, int H, int W, double res, double ox, double oy,
                          const int8_t *occ);
/* The same for K maps of one shape (H, W, res) in one call: slots (K) distinct map slots, ox / oy (K) origins, occ
 * (K, H, W). One synchronisation at the end instead of one per map (the 256 generated worlds of the data-generation
 * sweep, BASELINE.json configs[3]). */
int neo_set_maps_occupancy(neo_handle *h, int K, const int32_t *slots, int H, int W, double res, const double *ox,
                           const double *oy, const int8_t *occ);
/* Map build from a point cloud / voxel-centre list (the step before ESDF.occupancy_map_cb, done by the external
 * octomap_server in the reference: map_server_global.launch:17-31): xyz (n,3) float32 as stored in a .pcd; a cell
 * (row = floor((y-oy)/res), col = floor((x-ox)/res)) is occupied iff a point with z_min <= z <= z_max falls into it;
 * then the same exact EDT + gradient as neo_set_map_occupancy. */
int neo_set_map_points(neo_handle *h, int slot, int n_points, const float *xyz, double z_min, double z_max,
                       int H, int W, double res, double ox, double oy);
/* The occupancy grid the map in this slot was built from: occ (H, W), the values neo_set_map_occupancy /
 * neo_set_maps_occupancy received (100 = occupied, any other value free) or the 0 / 100 grid neo_set_map_points
 * projected. A slot whose map came from neo_set_map_esdf has none (NEO_ERR_INVALID) until the next
 * neo_set_map_occupancy / neo_set_maps_occupancy / neo_set_map_points on it. (H, W) is the size of the caller's array
 * and must be the slot's shape, else NEO_ERR_INVALID and nothing is written. */
int neo_get_occupancy(neo_handle *h, int slot, int H, int W, int8_t *occ);
/* Read a slot back (for checks / for filling a reference ESDF object): each out array (H, W) or NULL; (H, W) must be the
 * slot's shape, as for neo_get_occupancy. */
int neo_get_map(neo_handle *h, int slot, int H, int W, double *esdf, double *gx, double *gy);
/* ESDF.get_edt_dis / get_edt_grad (ESDF:53-82) for n points xy (n,2): idx (n,2) = row, col (-1,-1 when
 * outside), dis (n) (10000 outside), grad (n,2) = [grad_x, grad_y] ([0,0] outside). */
int neo_query_map(neo_handle *h, int slot, int n, const double *xy, int32_t *idx, double *dis, double *grad);

/* cost + gradient ------------------------------------------------------------------------------ */
/* get_cost + get_grad (EP:539-585) fused, for B independent problems.
 * x (B,n); head, tail (B,3,2); map_ids (B) or NULL (= slot 0).
 * costs (B,4) unweighted [energy, time, feasibility, collision]; grad (B,n); status (B): 0 or NEO_ST_OVERFLOW/NAN.
 * coeffs (B,6M,2) and ts (B,M) are optional (may be NULL). */
int neo_eval(neo_handle *h, int B, int M, const double *x, const double *head, const double *tail,
             const int32_t *map_ids, double *costs, double *grad, int32_t *status, double *coeffs, double *ts);

/* optimisation --------------------------------------------------------------------------------- */
/* Outputs of neo_optimize, all (B, ...) and caller-allocated. */
typedef struct {
    double *x;         /* (B,n)   final decision vector of the returned attempt                       */
    double *ts;        /* (B,M)   map_tau2T of its tau part (EP:229)                                  */
    double *coeffs;    /* (B,6M,2) coefficients of the final (int_wpts, ts), as TU:182 recomputes them */
    double *costs;     /* (B,4)   unweighted costs at the LAST EVALUATED point (what EP:233 reads)     */
    int32_t *status;   /* (B)     NEO_ST_* of the last attempt that ran                                */
    int32_t *ok;       /* (B)     1: an attempt passed `collision cost <= tol` (EP:236); 0: the reference
                                  would raise "No solution for the given target" (EP:203)              */
    int32_t *attempt;  /* (B)     index of the returned attempt                                        */
    int32_t *nit;      /* (B)     sum of res.nit over attempts whose minimize() returned (EP:230)      */
    int32_t *runs;     /* (B)     number of such attempts (opt_running_times, EP:232)                  */
    int32_t *nfev;     /* (B)     fused cost+grad evaluations over all attempts                        */
    int64_t *work;     /* (B,4) or NULL: samples, velocity-violating samples, colliding samples summed over all
                                  evaluations of attempts 0..attempt (for the roofline flop count), and the
                                  nanoseconds those attempts occupied a warp (critical-path accounting)      */
} neo_result;

/* warm_start_plan (EP:186-203) for B problems: attempt 0 starts from (q0, ts0) through plan_once
 * (EP:205-237: tau = map_T2tau(ts), L-BFGS-B with scipy's tol=1e-4/maxcor=10/maxls=20 semantics);
 * attempt a >= 1 restarts from retry_q[b][a-1] (2, M-1) with ts = retry_ts (M) -- the straight line plus
 * N(0,0.5) noise the host draws (EP:92-99, EP:200). max_attempts = 5 reproduces the reference;
 * max_attempts = 1 is a bare plan_once. retry_* may be NULL when max_attempts == 1.
 * q0 (B,2,M-1); ts0 (B,M); head, tail (B,3,2); map_ids (B) or NULL. */
int neo_optimize(neo_handle *h, int B, int M, const double *q0, const double *ts0, const double *head,
                 const double *tail, const int32_t *map_ids, const double *retry_q, const double *retry_ts,
                 int max_attempts, neo_result *out);

/* neo_optimize plus a record of what the device evaluated (parity tests: the recorded sequence is replayed through the
 * CPU checker's optimizer, tests/test_gpu_lockstep.py). Per task t = attempt * B + problem the first trace_cap
 * evaluations: tr_x (A*B, cap, n) trial points, tr_f (A*B, cap), tr_g (A*B, cap, n), tr_costs (A*B, cap, 4),
 * tr_status (A*B, cap) 0 or the NEO_ST_* the evaluation raised, tr_len (A*B) evaluations made (0: task never ran).
 * Speculative retries that were cancelled leave a partial record. */
int neo_optimize_trace(neo_handle *h, int B, int M, const double *q0, const double *ts0, const double *head,
                       const double *tail, const int32_t *map_ids, const double *retry_q, const double *retry_ts,
                       int max_attempts, neo_result *out, int trace_cap, double *tr_x, double *tr_f, double *tr_g,
                       double *tr_costs, int32_t *tr_status, int32_t *tr_len);

/* Device-pointer variant: every pointer (inputs, retry_*, and all non-NULL members of *out) is a DEVICE
 * pointer; the launch is enqueued on `stream` and not synchronised. Inputs are in tau form (neo_prepare_dev
 * builds them on the device, neo_T2tau on the host):
 *   x0 (B,n) = [q0, neo_T2tau(ts0)], x0_status (B) or NULL = its per-problem status,
 *   retry_tau (M) = neo_T2tau(retry_ts), retry_status = its status (0 or NEO_ST_DOMAIN). */
int neo_optimize_dev(neo_handle *h, int B, int M, const double *x0, const int32_t *x0_status, const double *head,
                     const double *tail, const int32_t *map_ids, const double *retry_q, const double *retry_tau,
                     int retry_status, int max_attempts, const neo_result *out, void *stream);
int neo_eval_dev(neo_handle *h, int B, int M, const double *x, const double *head, const double *tail,
                 const int32_t *map_ids, double *costs, double *grad, int32_t *status, double *coeffs, double *ts,
                 void *stream);

/* Device-resident inputs: the same values the host-pointer path assembles, computed on the device. DEVICE pointers,
 * enqueued on `stream` (NULL = the handle's own) without synchronising, like the _dev calls above.
 * neo_T2tau_dev: neo_T2tau for n device values -- glibc's log is restated on the device (csrc/libm_log.h), so tau and
 *   status equal neo_T2tau's bit for bit on a host whose C library is glibc on an x86-64 CPU with FMA. status may be NULL.
 * neo_prepare_dev: the inputs of neo_optimize_dev for B problems, as neo_optimize builds them from (q0, ts0):
 *   x0 (B,n) = [q0, T2tau(ts0)] (tau = 0 where the status is set), x0_status (B) = the last nonzero status of the row;
 *   q0 (B,2,M-1) or NULL = the straight line of guesses.straight_line_guess (head pos -> tail pos, M-1 waypoints);
 *   ts0 (B,M) or NULL = the HOST vector init_ts (M) for every problem;
 *   retry_q (B,count,2,M-1) = that straight line + noise (B,count,M-1,2) (guesses.retry_guesses); count in [0, 7];
 *   map_ids_host (B) or NULL: HOST ids, checked like neo_optimize's (NEO_ERR_INVALID before anything is enqueued),
 *   then copied to the device array map_ids_dev (B) that neo_optimize_dev reads.
 *   head, tail (B,3,2) are device arrays. The retry durations are host data: pass neo_T2tau(init_ts) as retry_tau. */
int neo_T2tau_dev(neo_handle *h, int n, const double *ts, double *tau, int32_t *status, void *stream);
int neo_prepare_dev(neo_handle *h, int B, int M, const double *head, const double *tail, const double *q0,
                    const double *ts0, const double *init_ts, int count, const double *noise, const int32_t *map_ids_host,
                    double *x0, int32_t *x0_status, double *retry_q, int32_t *map_ids_dev, void *stream);
/* neo_get_coeffs / neo_sample on device arrays. neo_sample_dev always writes count (the full count, which may exceed
 * max_samples) and never writes a row at or past max_samples; states may be NULL (counts only). */
int neo_get_coeffs_dev(neo_handle *h, int B, int M, const double *q, const double *ts, const double *head,
                       const double *tail, double *coeffs, void *stream);
int neo_sample_dev(neo_handle *h, int B, int M, const double *coeffs, const double *ts, double hz, int max_samples,
                   double *states, int32_t *count, void *stream);

/* host helpers with the reference's libm semantics --------------------------------------------- */
/* map_T2tau (EP:468-475) for n values using the C library's log(), i.e. the same function CPython's
 * math.log calls. status (n): 0 or NEO_ST_DOMAIN. */
int neo_T2tau(const neo_config *cfg, int n, const double *ts, double *tau, int32_t *status);
/* get_coeffs (EP:261-336 / TU:8-83) for B problems on the device: q (B,2,M-1), ts (B,M) -> coeffs (B,6M,2) */
int neo_get_coeffs(neo_handle *h, int B, int M, const double *q, const double *ts, const double *head,
                   const double *tail, double *coeffs);

/* trajectory sampling ---------------------------------------------------------------------------- */
/* get_full_state_cmd(hz) (TU:181-195) for B trajectories: states (B, max_samples, 3, 2) = pos, vel, acc at
 * t_k = k/hz, k < count[b] = len(np.arange(0, sum(ts), 1/hz)); rows beyond count[b] are left untouched.
 * Fails with NEO_ERR_INVALID if any count exceeds max_samples (call with states = NULL to get counts only). */
int neo_sample(neo_handle *h, int B, int M, const double *coeffs, const double *ts, double hz, int max_samples,
               double *states, int32_t *count);

/* geometric initializer ---------------------------------------------------------------------------- */
/* AstarPlanner.plan (astar_planner.py:22-103) followed by GeoPlanner.prune_path_nodes (geo_planner.py:57-101) for B
 * start/target pairs, one warp each: 8-connected A* over the map grid enlarged by int(10 m / res) cells (origin moved by
 * -5 m), nodes tested with ESDF.has_collision (0.5 m), open-set ties resolved like Python's min() over the insertion-
 * ordered dict; then line-of-sight shortcutting (0.1 m samples, 0.4 m clearance) and selection of exactly four key
 * nodes, of which the middle two are the int_wpts GeoPlanner.geo_traj_plan warm-starts from (geo_planner.py:29).
 * start, target (B,2); map_ids (B) or NULL. Outputs: pruned (B,4,2); path_len (B) full path length; path
 * (B,max_path,2) or NULL: the first min(path_len, max_path) path nodes [x, y]; closed (B) number of expanded nodes;
 * status (B): NEO_ASTAR_FOUND, NEO_ASTAR_EXHAUSTED (open set ran empty: path = [target cell], as the reference returns),
 * NEO_ASTAR_START_OUTSIDE (start not on the enlarged grid; the reference's grid index would alias -- rejected here),
 * NEO_ASTAR_LIMIT (more than max_closed > 0 nodes expanded; 0 = no limit, the reference has none). */
#define NEO_ASTAR_FOUND 0
#define NEO_ASTAR_EXHAUSTED 1
#define NEO_ASTAR_START_OUTSIDE 2
#define NEO_ASTAR_LIMIT 3
int neo_astar(neo_handle *h, int B, const double *start, const double *target, const int32_t *map_ids, int max_closed,
              int max_path, double *path, int32_t *path_len, double *pruned, int32_t *status, int32_t *closed);
/* Device-pointer variant, enqueued on `stream` and not synchronised (scratch is grown before the launch). */
int neo_astar_dev(neo_handle *h, int B, const double *start, const double *target, const int32_t *map_ids,
                  int max_closed, int max_path, double *path, int32_t *path_len, double *pruned, int32_t *status,
                  int32_t *closed, void *stream);

/* measurement helpers ---------------------------------------------------------------------------- */
/* Device time in ms of the most recent optimize/eval kernel launched through a host-pointer entry point
 * (CUDA events on the launching stream). */
int neo_last_kernel_ms(neo_handle *h, float *ms);
/* FP64 FMA throughput microbenchmark (dependent-chain-free DFMA loop on all SMs): returns TFLOP/s. */
int neo_fp64_peak(neo_handle *h, double *tflops);
/* Number of kernels this library has launched on this handle since creation. */
int neo_launch_count(neo_handle *h, int64_t *count);

/* test hooks: the double-double exp used for tau -> T, on the device and as compiled for the host */
int neo_test_exp_dev(neo_handle *h, int n, const double *x, double *y);
int neo_test_exp_host(int n, const double *x, double *y);
/* test hooks: the optimizer's vector primitives (lbfgsb_tile.cuh) compiled for the device with the library's flags, one
 * vector per thread. v, a, b: (count, n) row-major. nrm: dnrm2 (x87_nrm2.h); blas: the ddot kernel's summation order (n < 32);
 * loop: scipy's own mul + add loop. */
int neo_test_nrm2_dev(neo_handle *h, int count, int n, const double *v, double *nrm);
int neo_test_ddot_dev(neo_handle *h, int count, int n, const double *a, const double *b, double *blas, double *loop);
/* test hook (no GPU needed): `calls` runs of the host worker pool that neo_optimize uses, over [0, count); returns the number
 * of indices not visited exactly once per run. */
int neo_test_host_pool(long long count, int calls);

#ifdef __cplusplus
}
#endif
#endif /* NEOOPT_H */
