"""Lockstep replay of the device optimizer (tests/test_gpu_lockstep.py) on problems chosen to reach its rare branches, with
the branches it took counted.

Each case builds one population on the host, seeded: dense and sparse pillar worlds and random pillar maps, starts and
goals touching or inside obstacles, boundary velocities up to 3 v_max with large accelerations, initial durations within
1e-6 of T_min or T_max, and parameter sets with random weights, speed limits and clearances, all weights times 1e-7, or
a large time weight. Every attempt the device ran is replayed through the checker's optimizer (scipy's L-BFGS-B
restated, oracle/minco_oracle.c) and must ask for the recorded points bit for bit and end as the device ended. During
such a replay the checker takes exactly the decisions the device took, so its branch counters
(oracle/c_oracle.BRANCHES) say which branches of lbfgsb_tile.cuh were shown to follow scipy, at which tile width and
piece count. tests/test_lbfgsb_branch_coverage.py shows the same branches in step with scipy itself.

The last test prints the table and asserts: every branch in DEVICE_REQUIRED was taken; search directions with every
memory length 1..10 occurred at each (tile width, M) in COL_KEYS; a memory drop followed a wrap of the ring buffer."""
import os

import numpy as np
import pytest

from neo_planner_b200 import lib
from neo_planner_b200.guesses import retry_guesses, straight_line_guess
from neo_planner_b200.worlds import YamlConfig, make_problems, make_world
from oracle import c_oracle

pytestmark = pytest.mark.gpu

# Branches the device cannot take through neo_optimize:
#   exit_stpmin: stpmin = 0 and an unbracketed search only moves stp up, so stp == stpmin never happens.
#   maxiter: 15000 iterations or 15000 evaluations per attempt.
#   eval_domain: the device evaluator reports DOMAIN only for x0 (T -> tau on the host), never for a trial point.
#   exit_stpmax: the search reaches stp = 1e10 only on objectives that stay linear over that range (the scipy-side test
#     has them); a MINCO cost grows at least quadratically along a search direction.
#   factor_fail1, factor_fail2, nondescent_col: not reached by these populations (nor by the scipy-compared objectives
#     of test_lbfgsb_branch_coverage.py); counted and printed, not required.
DEVICE_REQUIRED = ([f'dir_col{c}' for c in range(11)] +
                   ['nondescent_col0', 'maxls', 'abnormal', 'reset_failed_search', 'skip_update', 'wrap',
                    'reset_after_wrap', 'accept_stp1', 'accept_stp', 'cache_hit'] +
                   [f'dcstep{k}_{b}' for k in range(1, 5) for b in ('open', 'brackt')] +
                   ['exit_conv', 'exit_bound', 'exit_xtol', 'stx_fallback', 'pg_x0', 'pg', 'ftol', 'eval_overflow'])
# floors of the rarer counts, about half of what the first B200 run measured (totals over all cases)
FLOORS = {'abnormal': 500, 'skip_update': 400, 'reset_after_wrap': 200, 'cache_hit': 2000, 'dcstep2_brackt': 300,
          'dcstep3_open': 700, 'dcstep4_open': 600, 'pg_x0': 150, 'pg': 150, 'eval_overflow': 500, 'nondescent_col0': 20}
# (tile lanes, M) at which every memory length 1..10 must occur: 8 lanes at both of its piece counts, 16 lanes, the
# 32-lane tile at a short, a middle (n = 16: the first size on the ddot n >= 16 path) and the longest trajectory
COL_KEYS = [(8, 2), (8, 3), (16, 4), (32, 3), (32, 6), (32, 10)]

# (tile lanes, M, NEO_GROUPED or None, problems per parameter set)
CASES = ([(8, 2, None, 96), (8, 3, None, 96), (8, 3, 0, 48), (16, 4, None, 96)] +
         [(32, M, None, 96 if M <= 5 else 48) for M in range(2, 11)])
FAR_CASES = [(8, 2), (32, 3)]
PARAM_SETS = ['yaml', 'random', 'tiny', 'time']
ATTEMPTS = {'yaml': 8, 'random': 3, 'tiny': 1, 'time': 2}

_COUNTS = {}


def config(kind, rng):
    cfg = YamlConfig()
    if kind == 'random':
        cfg.weights = list(10.0 ** rng.uniform(-2, 2, 4))
        cfg.v_max = float(rng.uniform(0.3, 5.0)); cfg.safe_dis = float(rng.uniform(0.2, 1.5))
        cfg.delta_t = float(rng.choice([0.05, 0.1, 0.2]))
    elif kind == 'tiny':
        cfg.weights = [w * 1e-7 for w in cfg.weights]
    elif kind == 'time':
        cfg.weights = [1.0, 1000.0, 1.0, 10000.0]
    return cfg


def world_for(case_id, kind, rng):
    """dense / sparse synthetic worlds, or a random pillar map as in test_gpu_eval_property.py"""
    if kind == 'random':
        H, W = int(rng.integers(80, 160)), int(rng.integers(80, 160))
        occ = np.zeros((H, W), np.int8)
        for _ in range(int(rng.integers(4, 16))):
            r, c = int(rng.integers(0, H)), int(rng.integers(0, W))
            occ[r:r + int(rng.integers(1, 8)), c:c + int(rng.integers(1, 8))] = 100
        return dict(H=H, W=W, res=0.1, ox=-2.0, oy=-float(H) * 0.05, occ=occ)
    w = make_world(case_id % 3, dense=case_id % 2 == 0)
    return dict(H=w.H, W=w.W, res=w.res, ox=w.ox, oy=w.oy, occ=w.occ, world=w)


def population(cfg, wd, B, M, rng):
    """head, tail (B, 3, 2) and ts0 (B, M): four quarters -- as make_problems draws them; start or goal moved onto an
    occupied cell; boundary velocities up to 3 v_max and accelerations up to ~4 v_max; durations next to T_min / T_max"""
    if 'world' in wd:
        hp, tp = make_problems(wd['world'], B, M=M, v_max=cfg.v_max, safe_dis=cfg.safe_dis, first=int(rng.integers(0, 10**6)))
    else:
        span = np.array([wd['W'], wd['H']]) * wd['res']; o = np.array([wd['ox'], wd['oy']])
        hp = np.zeros((B, 2, 2)); tp = np.zeros((B, 2, 2))
        hp[:, 0] = o + rng.uniform(0.05, 0.45, (B, 2)) * span; tp[:, 0] = o + rng.uniform(0.55, 0.95, (B, 2)) * span
        hp[:, 1] = rng.normal(0, 0.3, (B, 2)); tp[:, 1] = rng.normal(0, 0.3, (B, 2))
    head = np.zeros((B, 3, 2)); tail = np.zeros((B, 3, 2))
    head[:, :2] = hp; tail[:, :2] = tp
    q = B // 4
    rows, cols = np.nonzero(wd['occ'] > 0)
    if rows.size:
        pick = rng.integers(0, rows.size, q)
        cell = np.stack([wd['ox'] + (cols[pick] + rng.uniform(0, 1, q)) * wd['res'],
                         wd['oy'] + (rows[pick] + rng.uniform(0, 1, q)) * wd['res']], axis=1)
        goal = rng.random(q) < 0.5
        head[:q][~goal, 0] = cell[~goal]; tail[:q][goal, 0] = cell[goal]
    s = slice(q, 2 * q)
    for st in (head, tail):
        ang = rng.uniform(0, 2 * np.pi, q)
        st[s, 1] = (rng.uniform(0, 3, q) * cfg.v_max)[:, None] * np.stack([np.cos(ang), np.sin(ang)], axis=1)
        st[s, 2] = rng.normal(0, 2 * cfg.v_max, (q, 2))
    q0, ts0 = straight_line_guess(cfg, head, tail, M)
    t = slice(2 * q, 3 * q)
    near = np.where(rng.random((q, M)) < 0.5, cfg.T_min + rng.uniform(1e-8, 1e-6, (q, M)),
                    cfg.T_max - rng.uniform(1e-8, 1e-6, (q, M)))
    ts0 = ts0.copy(); ts0[t] = near
    return head, tail, q0, ts0


def handle_for(cfg, wd, tile, grouped):
    saved = {k: os.environ.get(k) for k in ('NEO_TILE', 'NEO_GROUPED')}
    os.environ['NEO_TILE'] = str(tile)
    if grouped is not None:
        os.environ['NEO_GROUPED'] = str(grouped)
    try:
        h = lib.Handle(cfg, 0, 1)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    h.set_map_occupancy(0, wd['H'], wd['W'], wd['res'], wd['ox'], wd['oy'], wd['occ'])
    return h


def x0_of(h, M, q0, ts0, rq, rts, b, at):
    if at == 0:
        tau, st = h.T2tau(ts0[b])
        return np.concatenate((q0[b].reshape(-1), tau)), int(st.max())
    tau, st = h.T2tau(rts)
    return np.concatenate((rq[b, at - 1].reshape(-1), tau)), int(st.max())


def cap_for(M, B, A):
    """evaluations recorded per attempt: as many as keep the trace (x and g) under ~0.5 GB"""
    n = 3 * M - 2
    return int(min(6000, 0.5e9 / (B * A * n * 16)))


def replay_all(h, M, B, A, head, tail, q0, ts0, rq, rts, cap, tag):
    """Runs the device with traces and replays every attempt through the checker; returns (counts, attempts, evaluations)
    over the attempts the device really ran."""
    out, tr = h.optimize_trace(M, q0, ts0, head, tail, retry_q=rq if A > 1 else None, retry_ts=rts if A > 1 else None,
                               max_attempts=A, cap=cap)
    counts = c_oracle.new_counts()
    checked = evals = 0
    for b in range(B):
        for at in range(A):
            t = at * B + b
            k = int(tr['len'][t])
            if k == 0:
                continue                          # never ran (an earlier attempt had been accepted) or domain error
            x0, st0 = x0_of(h, M, q0, ts0, rq, rts, b, at)
            assert st0 == 0
            c = c_oracle.new_counts()
            r = c_oracle.lbfgsb_replay(x0, tr['x'][t, :k], tr['f'][t, :k], tr['g'][t, :k], tr['costs'][t, :k],
                                       tr['status'][t, :k], counts=c)
            if at <= out['attempt'][b]:
                assert k < cap, (tag, b, at, 'trace capacity too small')
                assert r['first_bad'] == -1 and r['used'] == k, (tag, b, at, r['first_bad'], k)
                if at == out['attempt'][b] and out['runs'][b] > 0 and r['status'] < 4:
                    assert np.array_equal(r['x'], out['x'][b]), (tag, b, at)
                    assert r['status'] == out['status'][b], (tag, b, at)
                    assert np.array_equal(r['costs'], out['costs'][b]), (tag, b, at)
                counts += c
                checked += 1; evals += k
            else:                                 # speculative retry: complete, or cancelled at the end of its record
                assert r['first_bad'] in (-1, k), (tag, b, at, r['first_bad'], k)
    return counts, checked, evals


@pytest.mark.parametrize('tile,M,grouped,B', CASES)
def test_adversarial_population_replays_bit_for_bit(tile, M, grouped, B):
    counts = c_oracle.new_counts()
    checked = evals = 0
    for pi, kind in enumerate(PARAM_SETS):
        case_id = 1000 * M + 10 * tile + pi + (5 if grouped == 0 else 0)
        rng = np.random.default_rng(case_id)
        cfg = config(kind, rng); cfg.init_wpts_num = M - 1
        wd = world_for(case_id, 'random' if pi % 2 else 'synthetic', rng)
        head, tail, q0, ts0 = population(cfg, wd, B, M, rng)
        A = ATTEMPTS[kind]
        rq, rts = retry_guesses(cfg, head, tail, M, max(A - 1, 1), rng=rng)
        h = handle_for(cfg, wd, tile, grouped)
        c, n_att, n_ev = replay_all(h, M, B, A, head, tail, q0, ts0, rq, rts, cap_for(M, B, A), kind)
        h.close()
        counts += c; checked += n_att; evals += n_ev
    print(f'tile={tile} M={M} grouped={grouped}: {checked} attempts / {evals} evaluations replayed bit for bit')
    assert checked >= B * len(PARAM_SETS)
    _COUNTS[(tile, M, grouped)] = counts


@pytest.mark.parametrize('tile,M', FAR_CASES)
def test_far_from_the_origin_replays_bit_for_bit(tile, M):
    """An empty map 4e12 m from the origin (an ulp of x is ~1e-3 there), start and goal at rest up to 100 m apart and
    every initial duration one ulp below T_max (tau ~ 36, where dT/dtau ~ 1e-15): for short distances the Cauchy step
    x - g rounds back to x in every component although max|g| > pgtol, so g'd = 0 -- a non-descent direction with an
    empty memory, ABNORMAL; for shorter ones the gradient is below pgtol at x0."""
    cfg = YamlConfig(); cfg.init_wpts_num = M - 1
    O, B = 4e12, 192
    wd = dict(H=100, W=100, res=0.1, ox=O, oy=O, occ=np.zeros((100, 100), np.int8))
    rng = np.random.default_rng(77 + M)
    head = np.zeros((B, 3, 2)); tail = np.zeros((B, 3, 2))
    head[:, 0] = O + 5.0
    tail[:, 0] = head[:, 0] + (10 ** rng.uniform(-4, 2, B))[:, None] * np.array([0.6, 0.8])
    q0, ts0 = straight_line_guess(cfg, head, tail, M)
    ts0[:] = np.nextafter(cfg.T_max, 0.0)
    rq, rts = retry_guesses(cfg, head, tail, M, 1, rng=rng)
    h = handle_for(cfg, wd, tile, None)
    counts, checked, evals = replay_all(h, M, B, 1, head, tail, q0, ts0, rq, rts, 4000, 'far')
    h.close()
    print(f'far from the origin, tile={tile} M={M}: {checked} attempts / {evals} evaluations replayed bit for bit')
    assert checked == B
    _COUNTS[('far', tile, M)] = counts


def test_device_branch_coverage():
    """Runs after the cases above (file order) and sums what they recorded."""
    expected = {(t, M, g) for t, M, g, _ in CASES} | {('far', t, M) for t, M in FAR_CASES}
    if set(_COUNTS) != expected:
        pytest.skip('needs the whole file')
    keys = [(t, M, g) for t, M, g, _ in CASES] + [('far', t, M) for t, M in FAR_CASES]
    total = sum(_COUNTS.values())
    label = lambda k: f'f{k[1]}/{k[2]}' if k[0] == 'far' else f'{k[0]}/{k[1]}' + ('/ug' if k[2] == 0 else '')
    print('\ndevice branch counts (tile lanes / M; ug: NEO_GROUPED=0; f: far from the origin), from replays that '
          'matched bit for bit')
    print(f'{"branch":20s}' + ''.join(f'{label(k):>8s}' for k in keys) + f'{"total":>9s}')
    for i, b in enumerate(c_oracle.BRANCHES):
        print(f'{b:20s}' + ''.join(f'{int(_COUNTS[k][i]):8d}' for k in keys) + f'{int(total[i]):9d}')
    counts = c_oracle.counts_dict(total)
    missing = [b for b in DEVICE_REQUIRED if counts[b] == 0]
    assert not missing, missing
    for tile, M in COL_KEYS:
        c = c_oracle.counts_dict(_COUNTS[(tile, M, None)])
        short = [col for col in range(1, 11) if c[f'dir_col{col}'] == 0]
        assert not short, (tile, M, short)
    assert counts['reset_after_wrap'] > 0
    low = {b: (counts[b], f) for b, f in FLOORS.items() if counts[b] < f}
    assert not low, low
