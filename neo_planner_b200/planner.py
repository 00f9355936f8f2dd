"""Host-side mirror of the reference optimizer interface (src/planner/scripts/traj_planner/expert_planner.py and
traj_utils.py) on top of libneoopt.so.

* ``MinJerkPlanner`` -- drop-in for the reference class of the same name: same constructor, methods, attribute
  results and exceptions (SURVEY.md §8b), one problem at a time, every numeric step on the B200.
* ``BatchPlanner``   -- the same operations for B independent problems per call (what the hardware is for):
  ``plan`` / ``warm_start_plan`` / ``batch_plan`` / ``get_cost_grad`` / ``get_full_state_cmd``.

There is no CPU fallback: constructing either class without the built library or without a Blackwell GPU raises.
"""
from __future__ import annotations

import math

import numpy as np

from . import guesses, lib
from .lib import (ST_ABNORMAL, ST_CONV_FTOL, ST_CONV_PG, ST_DOMAIN, ST_MAXITER, ST_NAN, ST_OVERFLOW)  # noqa: F401


class DefaultConfig:
    """Library defaults of the reference (EP:12-25)."""

    def __init__(self):
        self.v_max = 10.0
        self.T_min = 2.0
        self.T_max = 20.0
        self.safe_dis = 0.5
        self.delta_t = 0.1
        self.weights = [1.0, 1.0, 0.001, 10000]
        self.init_wpts_mode = 'fixed'
        self.init_seg_len = 2.0
        self.init_wpts_num = 2
        self.init_T = 2.0
        self.collision_cost_tol = 10
        self.opt_tol = 1e-4


def _raise_for_status(st):
    """Re-create the exception the reference would have propagated (SURVEY.md §8a Q11)."""
    if st == ST_OVERFLOW:
        raise OverflowError('math range error')
    if st == ST_DOMAIN:
        raise ValueError('math domain error')
    if st == ST_NAN:
        raise ValueError('cannot convert float NaN to integer')


class _MapCache:
    """Uploads a duck-typed map object (ESDF:17-33 attributes) into a handle slot once per map version."""

    def __init__(self, handle):
        self.handle = handle
        self.keys = {}
        self.held = {}      # the cached object itself: keeps its id() from being reused by a new map while it is the key

    def ensure(self, slot, m):
        key = (id(m), getattr(m, 'version', None), id(getattr(m, 'esdf_map', None)))
        if self.keys.get(slot) == key:
            return
        if hasattr(m, 'esdf_map'):
            self.handle.set_map_esdf(slot, float(m.map_resolution), float(m.map_origin.x), float(m.map_origin.y),
                                     m.esdf_map, m.esdf_grad_x, m.esdf_grad_y)
        elif hasattr(m, 'occ'):       # neo_planner_b200.worlds.World: build the field on the device
            self.handle.set_map_occupancy(slot, m.H, m.W, m.res, m.ox, m.oy, m.occ)
        else:
            raise TypeError('map must expose esdf_map/esdf_grad_x/esdf_grad_y (ESDF) or be a worlds.World')
        self.keys[slot] = key
        self.held[slot] = (m, getattr(m, 'esdf_map', None))


class TrajUtils:
    """TU:85-250 -- trajectory getters on the final (int_wpts, ts); sampling runs on the device."""

    def __init__(self):
        self.coeffs = []
        self.s = 3

    def _piece(self, t):
        k = 0
        while sum(self.ts[:k + 1]) < t:
            k += 1
        return k, t - sum(self.ts[:k])

    def _deriv(self, t, order):
        if t > sum(self.ts):
            return self._deriv(sum(self.ts), order)
        if isinstance(self.coeffs, list) and self.coeffs == []:
            self.get_coeffs(self.int_wpts, self.ts)
        k, T = self._piece(t)
        blk = self.coeffs[6 * k:6 * (k + 1), :]
        beta = [np.array([1, T, T**2, T**3, T**4, T**5]),
                np.array([0, 1, 2*T, 3*T**2, 4*T**3, 5*T**4]),
                np.array([0, 0, 2, 6*T, 12*T**2, 20*T**3]),
                np.array([0, 0, 0, 6, 24*T, 60*T**2])][order]
        return np.dot(blk.T, np.array([beta]).T).T

    def get_pos(self, t):
        return self._deriv(t, 0)

    def get_vel(self, t):
        return self._deriv(t, 1)

    def get_acc(self, t):
        return self._deriv(t, 2)

    def get_jerk(self, t):
        return self._deriv(t, 3)

    def get_full_state_cmd(self, hz=300):
        """TU:181-195: (N, 3, D) = [pos, vel, acc] at t = k/hz, sampled by the device kernel."""
        self.get_coeffs(self.int_wpts, self.ts)
        states, count = self._handle().sample(self.M, self.coeffs[None], np.asarray(self.ts)[None], hz)
        return states[0, :count[0]]

    def _array(self, order):
        self.get_coeffs(self.int_wpts, self.ts)
        states, count = self._handle().sample(self.M, self.coeffs[None], np.asarray(self.ts)[None], 1.0 / 0.1)
        if order <= 2:
            return states[0, :count[0], order]
        return np.array([self.get_jerk(t)[0] for t in np.arange(0, sum(self.ts), 0.1)])

    def get_pos_array(self):
        return self._array(0)

    def get_vel_array(self):
        return self._array(1)

    def get_acc_array(self):
        return self._array(2)

    def get_jer_array(self):
        return self._array(3)


class MinJerkPlanner(TrajUtils):
    """Minimum-jerk MINCO planner with the reference's interface (EP:28-585), computed on the B200."""

    def __init__(self, config=None, device: int = 0):
        super().__init__()
        config = DefaultConfig() if config is None else config
        self.s = 3
        self.v_max = config.v_max
        self.T_min = config.T_min
        self.T_max = config.T_max
        self.safe_dis = config.safe_dis
        self.collision_cost_tol = config.collision_cost_tol
        self.weights = np.array(config.weights)
        self.delta_t = config.delta_t
        self.opt_tol = config.opt_tol
        self.init_wpts_mode = config.init_wpts_mode
        self.init_seg_len = config.init_seg_len
        self.init_wpts_num = int(config.init_wpts_num)
        self.init_T = config.init_T
        self.batch_num = 3
        self.iter_num = 0
        self.opt_running_times = 0
        self._device = device
        self._h = None
        self._maps = None
        self.D = 2

    # ---- plumbing ---------------------------------------------------------------------------------------------
    def _handle(self):
        if self._h is None:
            self._h = lib.Handle(self, self._device, 1)
            self._maps = _MapCache(self._h)
        return self._h

    def _sync_map(self):
        self._handle()
        self._maps.ensure(0, self.map)

    # ---- entry points (EP:62-203) -------------------------------------------------------------------------------
    def plan(self, map, head_state, tail_state):
        int_wpts, ts = self.generate_init_variables(head_state, tail_state)
        self.warm_start_plan(map, head_state, tail_state, int_wpts, ts)

    def generate_init_variables(self, head_state, tail_state, seed=0):
        M = guesses.pieces_for(self, head_state, tail_state)
        if seed != 0:
            q, ts = guesses.retry_guesses(self, head_state, tail_state, M, 1)     # draws from np.random, as EP:94
            return q[0], ts
        q, ts = guesses.straight_line_guess(self, np.asarray(head_state)[None], np.asarray(tail_state)[None], M)
        return q[0], ts[0]

    def batch_generate_init_variables(self, head_state, tail_state):
        if self.init_wpts_mode != 'fixed':
            print("Error! init_wpts_mode must be 'fixed'")
        c, ts = guesses.lateral_guesses(self, np.asarray(head_state)[None], np.asarray(tail_state)[None],
                                        self.init_wpts_num + 1, self.batch_num)
        return c[0], ts

    def batch_plan(self, map, head_state, tail_state):
        """EP:142-168: three candidates through plan_once; keep the cheapest feasible one, else re-plan."""
        cands, ts = self.batch_generate_init_variables(head_state, tail_state)
        best_w = np.zeros(cands.shape)
        best_t = np.zeros((self.batch_num, len(ts)))
        score = np.zeros(self.batch_num)
        for i in range(self.batch_num):
            try:
                self.read_planning_conditions(map, head_state, tail_state, cands[i], ts)
                self.plan_once()
                best_w[i] = self.int_wpts
                best_t[i] = self.ts
                score[i] = self.weighted_cost.sum()
            except Exception:
                score[i] = np.inf
        if np.min(score) < np.inf:
            j = int(np.argmin(score))
            self.int_wpts = best_w[j]
            self.ts = best_t[j]
            self.final_cost = score[j]
        else:
            self.warm_start_plan(map, head_state, tail_state, cands[0], ts)

    def read_planning_conditions(self, map, head_state, tail_state, int_wpts, ts):
        head_state = np.asarray(head_state, dtype=np.float64)
        tail_state = np.asarray(tail_state, dtype=np.float64)
        self.map = map
        self.D = head_state.shape[1]
        if self.D != 2:
            raise ValueError('only planar problems (D = 2) are supported (the reference node runs D = 2, NODE:593-595)')
        self.M = np.asarray(ts).shape[0]
        self.head_state = lib.pad_state(head_state)
        self.tail_state = lib.pad_state(tail_state)
        self.int_wpts = int_wpts
        self.ts = ts

    def warm_start_plan(self, map, head_state, tail_state, int_wpts, ts):
        self.read_planning_conditions(map, head_state, tail_state, int_wpts, ts)
        seed = 0
        while seed < 5:
            try:
                self.plan_once()
                return
            except Exception as ex:
                print(f"Re-planning for {ex}, current seed: {seed}")
                seed += 1
                self.int_wpts, self.ts = self.generate_init_variables(head_state, tail_state, seed)
        raise Exception("No solution for the given target")

    def plan_once(self):
        """EP:205-237 -- one L-BFGS-B run on the device (neo_optimize with max_attempts = 1)."""
        self._sync_map()
        q0 = np.asarray(self.int_wpts, dtype=np.float64).reshape(1, 2, self.M - 1)
        ts0 = np.asarray(self.ts, dtype=np.float64).reshape(1, self.M)
        out = self._h.optimize(self.M, q0, ts0, self.head_state[None], self.tail_state[None], max_attempts=1)
        st = int(out['status'][0])
        _raise_for_status(st)
        nq = 2 * (self.M - 1)
        self.int_wpts = out['x'][0, :nq].reshape(2, self.M - 1)
        self.tau = out['x'][0, nq:].copy()
        self.ts = out['ts'][0].copy()
        self.coeffs = out['coeffs'][0].copy()
        self.costs = out['costs'][0].copy()
        self.last_status = st
        self.last_nfev = int(out['nfev'][0])
        self.iter_num += int(out['nit'][0])
        self.opt_running_times += 1
        self.weighted_cost = self.costs * self.weights
        self.final_cost = self.weighted_cost.sum()
        if self.weighted_cost[3] > self.collision_cost_tol:
            raise ValueError("collision cost too large")

    def print_results(self):
        print(self.int_wpts.T)
        print(self.ts)
        self.weighted_cost = self.costs * self.weights
        print("Energy cost: %f, Time cost: %f, Feasibility cost: %f, Collision cost: %f" % tuple(self.weighted_cost))

    # ---- pieces of the objective (EP:261-585) ---------------------------------------------------------------------
    def get_coeffs(self, int_wpts, ts):
        h = self._handle()
        q = np.asarray(int_wpts, dtype=np.float64).reshape(1, 2, -1)
        self.coeffs = h.get_coeffs(q.shape[2] + 1, q, np.asarray(ts, dtype=np.float64)[None], self.head_state[None],
                                   self.tail_state[None])[0]

    def map_T2tau(self, ts):
        tau, st = self._handle().T2tau(np.asarray(ts, dtype=np.float64))
        for s in st.reshape(-1):
            _raise_for_status(int(s))
        return tau

    def map_tau2T(self, tau):
        ts = np.zeros(len(tau))
        for i in range(len(tau)):
            ts[i] = (self.T_max - self.T_min) / (1 + math.exp(-tau[i])) + self.T_min
        return ts

    def _eval(self, x):
        self._sync_map()
        x = np.asarray(x, dtype=np.float64)
        out = self._h.eval(self.M, x[None], self.head_state[None], self.tail_state[None], want_coeffs=True)
        _raise_for_status(int(out['status'][0]))
        nq = 2 * (self.M - 1)
        self.int_wpts = np.reshape(x[:nq], (2, self.M - 1))
        self.tau = x[nq:]
        self.ts = out['ts'][0]
        self.coeffs = out['coeffs'][0]
        return out

    def get_cost(self, x):
        out = self._eval(x)
        self.costs = out['costs'][0]
        return np.dot(self.costs, self.weights)

    def get_grad(self, x):
        return self._eval(x)['grad'][0]

    def reset_cost(self):
        self.costs = np.zeros(len(self.weights))

    def _costs_here(self):
        x = np.concatenate((np.reshape(self.int_wpts, (-1,)), self.map_T2tau(self.ts)))
        self._sync_map()
        out = self._h.eval(self.M, x[None], self.head_state[None], self.tail_state[None])
        _raise_for_status(int(out['status'][0]))
        return out['costs'][0]

    def add_energy_cost(self):
        self.costs[0] += self._costs_here()[0]

    def add_time_cost(self):
        self.costs[1] += np.sum(self.ts)

    def add_sampled_cost(self):
        c = self._costs_here()
        self.costs[2] += c[2]
        self.costs[3] += c[3]


class BatchPlanner:
    """B independent planning problems per call. Results are returned as a dict of (B, ...) arrays:
    x, ts, coeffs, costs, status, ok, attempt, nit, runs, nfev, work (see include/neoopt.h: neo_result)."""

    def __init__(self, config=None, device: int = 0, max_maps: int = 1):
        self.cfg = DefaultConfig() if config is None else config
        self.handle = lib.Handle(self.cfg, device, max_maps)
        self.maps = _MapCache(self.handle)
        self.weights = np.array(self.cfg.weights, dtype=np.float64)

    @property
    def M(self):
        return int(self.cfg.init_wpts_num) + 1

    def set_map(self, m, slot: int = 0):
        self.maps.ensure(slot, m)

    def plan(self, head, tail, map_ids=None, rng=None, max_attempts=5, M=None):
        """MinJerkPlanner.plan (EP:62-80) for every problem: straight-line guess, up to 5 attempts."""
        M = self.M if M is None else M
        q0, ts0 = guesses.straight_line_guess(self.cfg, head, tail, M)
        return self.warm_start_plan(head, tail, q0, ts0, map_ids, rng, max_attempts)

    def warm_start_plan(self, head, tail, int_wpts, ts, map_ids=None, rng=None, max_attempts=5):
        """EP:186-203. int_wpts (B,2,M-1), ts (B,M). Retry noise comes from `rng` (np.random.Generator) or, when
        None, from the global np.random stream like the reference."""
        ts = np.asarray(ts, dtype=np.float64)
        M = ts.shape[1]
        rq = rts = None
        if max_attempts > 1:
            rq, rts = guesses.retry_guesses(self.cfg, head, tail, M, max_attempts - 1, rng=rng)
        return self.handle.optimize(M, int_wpts, ts, head, tail, map_ids, rq, rts, max_attempts)

    def batch_plan(self, head, tail, map_ids=None, rng=None):
        """EP:142-168 for every problem: 3 lateral candidates in one launch (3B problems), argmin of the weighted
        cost among the feasible ones; problems with no feasible candidate fall back to warm_start_plan."""
        head = np.asarray(head, dtype=np.float64); tail = np.asarray(tail, dtype=np.float64)
        B = head.shape[0]; M = self.M
        cands, ts = guesses.lateral_guesses(self.cfg, head, tail, M)
        k = cands.shape[1]
        rep = lambda a: np.repeat(a, k, axis=0)                                       # noqa: E731
        ids = None if map_ids is None else rep(np.asarray(map_ids))
        out = self.handle.optimize(M, cands.reshape(B * k, 2, M - 1), np.tile(ts, (B * k, 1)), rep(head), rep(tail), ids,
                                   max_attempts=1)
        score = (out['costs'] * self.weights).sum(axis=1)
        score[out['ok'] == 0] = np.inf
        score = score.reshape(B, k)
        best = np.argmin(score, axis=1)
        pick = np.arange(B) * k + best
        res = {key: (None if v is None else v[pick].copy()) for key, v in out.items()}
        res['final_cost'] = score[np.arange(B), best]
        res['best_idx'] = best.astype(np.int32)
        res['runs'] = out['runs'].reshape(B, k).sum(axis=1).astype(np.int32)
        res['nit'] = out['nit'].reshape(B, k).sum(axis=1).astype(np.int32)
        res['nfev'] = out['nfev'].reshape(B, k).sum(axis=1).astype(np.int32)
        lost = np.nonzero(~np.isfinite(res['final_cost']))[0]
        if len(lost):
            fb = self.warm_start_plan(head[lost], tail[lost], cands[lost, 0], np.tile(ts, (len(lost), 1)),
                                      None if map_ids is None else np.asarray(map_ids)[lost], rng)
            for key in ('x', 'ts', 'coeffs', 'costs', 'status', 'ok', 'attempt'):
                res[key][lost] = fb[key]
            for key in ('runs', 'nit', 'nfev'):
                res[key][lost] += fb[key]
            res['best_idx'][lost] = -1
            res['final_cost'][lost] = (fb['costs'] * self.weights).sum(axis=1)
        return res

    def get_cost_grad(self, x, head, tail, map_ids=None, M=None):
        """get_cost + get_grad (EP:539-585) at B points: dict(costs (B,4), cost (B), grad (B,n), status (B))."""
        M = self.M if M is None else M
        out = self.handle.eval(M, x, head, tail, map_ids)
        out['cost'] = out['costs'] @ self.weights
        return out

    def get_full_state_cmd(self, coeffs, ts, hz=300):
        """TU:181-195 for B trajectories: states (B, Nmax, 3, 2), count (B)."""
        return self.handle.sample(np.asarray(ts).shape[1], coeffs, ts, hz)

    # ---- device-resident variants ------------------------------------------------------------------------------
    # The same operations on torch CUDA tensors: inputs stay on the device, results come back as CUDA tensors on the
    # handle's device, and the work is enqueued on the current torch stream without a host synchronisation. Results are
    # bit-identical to the host methods given the same inputs and retry noise.
    def _dev_states(self, s):
        """(B, k<=3, 2) tensor or array-like -> (B, 3, 2) contiguous float64 tensor on the handle's device, zero padded."""
        import torch
        dev = torch.device('cuda', self.handle.device)
        s = s.to(dev, torch.float64) if torch.is_tensor(s) else torch.from_numpy(np.asarray(s, dtype=np.float64)).to(dev, non_blocking=True)
        if s.shape[-1] != 2:
            raise ValueError('only planar problems (D = 2) are supported, as in the reference node (NODE:593-595)')
        if s.shape[-2] == 3:
            return s.contiguous()
        out = torch.zeros(s.shape[:-2] + (3, 2), dtype=torch.float64, device=dev)
        out[..., :min(3, s.shape[-2]), :] = s[..., :3, :]
        return out

    def plan_dev(self, head, tail, map_ids=None, noise=None, generator=None, max_attempts=5, M=None):
        """plan on the device: straight-line guess, up to max_attempts attempts. See warm_start_plan_dev."""
        return self.warm_start_plan_dev(head, tail, None, None, map_ids, noise, generator, max_attempts,
                                        M=self.M if M is None else M)

    def warm_start_plan_dev(self, head, tail, int_wpts, ts, map_ids=None, noise=None, generator=None, max_attempts=5,
                            M=None):
        """warm_start_plan on the device. head/tail (B,k,2), int_wpts (B,2,M-1) and ts (B,M) are CUDA tensors (or
        array-likes, uploaded); int_wpts = None starts from the straight line, ts = None from the init_T durations.
        map_ids is HOST array-like (B) (checked before anything is enqueued). Retry noise (B, max_attempts-1, M-1, 2) is
        `noise` (a float64 CUDA tensor) or, when None, drawn on the device as N(0, 0.5) with the torch.Generator
        `generator` (None: torch's default CUDA generator). That is not the np.random stream the host method draws
        from: pass the same `noise` to compare the two. Returns the result dict of warm_start_plan as CUDA tensors."""
        import torch
        h = self.handle
        dev = torch.device('cuda', h.device)
        head, tail = self._dev_states(head), self._dev_states(tail)
        B = head.shape[0]
        if M is None:
            M = ts.shape[1] if ts is not None else int_wpts.shape[2] + 1
        up = lambda a: None if a is None else (a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev, non_blocking=True))  # noqa: E731
        init = guesses.init_ts(self.cfg, M)
        count = max_attempts - 1
        if count > 0 and noise is None:
            noise = torch.normal(0.0, 0.5, (B, count, M - 1, 2), generator=generator, dtype=torch.float64, device=dev)
        prep = h.prepare_dev(M, head, tail, up(int_wpts), up(ts), init, noise if count > 0 else None, map_ids)
        rtau, rst = None, 0
        if count > 0:
            tau, st = h.T2tau(init)                  # host data: the host's log, as neo_optimize computes it
            rtau, rst = torch.from_numpy(tau).to(dev, non_blocking=True), int(st.max())
        return h.optimize_dev(M, prep['x0'], head, tail, prep['x0_status'], prep['map_ids'], prep['retry_q'], rtau, rst,
                              max_attempts)

    def get_coeffs_dev(self, int_wpts, ts, head, tail):
        """get_coeffs (EP:261-336) on the device for B problems: int_wpts (B,2,M-1), ts (B,M) -> coeffs (B,6M,2)."""
        return self.handle.get_coeffs_dev(ts.shape[1], int_wpts, ts, self._dev_states(head), self._dev_states(tail))

    def get_full_state_cmd_dev(self, coeffs, ts, hz=300, max_samples=None):
        """get_full_state_cmd on the device: states (B, max_samples, 3, 2), count (B) int32. max_samples defaults to
        ceil(M T_max hz) + 1, which holds every trajectory the optimizer returns; count is the full sample count, and a
        trajectory with more samples than max_samples is cut at max_samples rows."""
        M = ts.shape[1]
        if max_samples is None:
            max_samples = math.ceil(M * self.cfg.T_max * hz) + 1
        return self.handle.sample_dev(M, coeffs, ts, hz, max_samples)
