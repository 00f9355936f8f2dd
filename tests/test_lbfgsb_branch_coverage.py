"""Which L-BFGS-B branches the checker's optimizer (oracle/minco_oracle.c) has been shown to take exactly as scipy does.

Every run below is made twice, by scipy.optimize.minimize and by the checker around the same Python f and g. The two must
evaluate the same sequence of points, bit for bit, and end with the same x, nit and nfev (or raise at the same point).
The checker's branch counters (c_oracle.BRANCHES) are summed over those runs. The populations are the random objectives
of test_lbfgsb_property.py, MINCO problems as in test_oracle_golden.py, and objectives built to reach rare branches:
failed line searches, skipped updates, steps too small to move x, huge first steps, overflow and domain errors in the
middle of a search. The last test asserts that each branch in REQUIRED was taken at least once. Together with
tests/test_gpu_lockstep*.py (device run == checker run) this pins the device optimizer to scipy branch by branch."""
import math

import numpy as np
import pytest
import scipy.optimize as sopt

from neo_planner_b200.worlds import make_world, make_problems, YamlConfig
from oracle import c_oracle, minco_ref
from test_lbfgsb_property import openblas_core, random_objective

OPTS = {'maxcor': 10, 'maxfun': 15000, 'maxiter': 15000, 'maxls': 20}

# Branches the scipy-compared runs must reach. Not listed:
#   factor_fail1 / factor_fail2: the middle matrix is positive definite in exact arithmetic (D = s'y > 0 is enforced by
#     the skip test); none of the populations here, nor a search over rotation-dominated, indefinite and anisotropic
#     objectives, made its rounded Cholesky fail. The checker's handling is the same memory drop as a failed search.
#   nondescent_col: reached by no population compared with scipy here (see the device test for the lockstep side).
#   exit_stpmin: stpmin = 0 and an unbracketed search only moves stp up, so stp == stpmin never happens.
#   eval_nan: a Python evaluator raises OverflowError or ValueError; the NaN status exists only in the C evaluator.
REQUIRED = ([f'dir_col{c}' for c in range(11)] +
            ['nondescent_col0', 'maxls', 'abnormal', 'reset_failed_search', 'skip_update', 'wrap', 'reset_after_wrap',
             'accept_stp1', 'accept_stp', 'cache_hit'] +
            [f'dcstep{k}_{b}' for k in range(1, 5) for b in ('open', 'brackt')] +
            ['exit_conv', 'exit_bound', 'exit_xtol', 'exit_stpmax', 'stx_fallback', 'pg_x0', 'pg', 'ftol',
             'maxiter', 'eval_overflow', 'eval_domain'])

_TOTAL = {}


def run_both(f, g, x0):
    """scipy and the checker on one objective; returns the checker's branch counts if the two runs are identical."""
    seen_s, seen_c = [], []

    def fs(x):
        seen_s.append(np.array(x))
        return f(x)

    def fgc(x):
        seen_c.append(np.array(x))
        return f(x), g(x)
    try:
        res = sopt.minimize(fs, x0, method='L-BFGS-B', jac=g, bounds=None, tol=1e-4, options=OPTS)
    except (OverflowError, ValueError, ZeroDivisionError):
        res = None
    counts = c_oracle.new_counts()
    x, nit, nfev, st = c_oracle.lbfgsb_cb(fgc, x0, counts=counts)
    assert len(seen_s) == len(seen_c) and all(np.array_equal(a, b) for a, b in zip(seen_s, seen_c))
    if res is None:
        assert st >= 4
    else:
        assert st < 4 and nit == res.nit and nfev == res.nfev and np.array_equal(x, res.x)
    return counts


def rotation(rng):
    """a symmetric part plus a large rotation in the 'gradient': s'y can be tiny against |y|^2, searches fail"""
    n = int(rng.integers(2, 12))
    Q = np.linalg.qr(rng.normal(size=(n, n)))[0]
    H = Q @ np.diag(10.0 ** rng.uniform(-3, 3, n)) @ Q.T
    A = rng.normal(size=(n, n)); A = (A - A.T) * 10 ** rng.uniform(-1, 3)
    return (lambda x: float(0.5 * x @ H @ x + np.sum(np.cos(x))), lambda x: H @ x - np.sin(x) + A @ x,
            rng.normal(size=n) * 3)


def indefinite(rng):
    """an indefinite quadratic inside a quartic wall: negative curvature along some steps, skipped updates"""
    n = int(rng.integers(2, 12))
    Q = np.linalg.qr(rng.normal(size=(n, n)))[0]
    H = Q @ np.diag(rng.uniform(-1, 1, n) * 10.0 ** rng.uniform(-2, 2, n)) @ Q.T
    q = 10 ** rng.uniform(-4, 0)
    return lambda x: float(0.5 * x @ H @ x + q * np.sum(x ** 4)), lambda x: H @ x + 4 * q * x ** 3, rng.normal(size=n) * 3


def far(rng):
    """a minimum at 1e12..1e17: late steps are below an ulp of x, trial points repeat the last one (cache hits)"""
    n = int(rng.integers(2, 12))
    c = 10.0 ** rng.uniform(12, 17); off = rng.uniform(0.1, 5, n); sc = 10 ** rng.uniform(-2, 2, n)
    return (lambda x: float(np.sum(0.5 * sc * (x - c) ** 2 + off * x)), lambda x: sc * (x - c) + off,
            np.full(n, c) + rng.normal(size=n) * 10 ** rng.uniform(0, 4))


def steep(rng):
    """an exponential wall that raises OverflowError (as the reference's math.exp does) once its exponent passes 60: long
    first steps from a start below the wall land beyond it in the middle of a search"""
    n = int(rng.integers(2, 12))
    a = 10 ** rng.uniform(0, 2.5); c = rng.normal(size=n)

    def ex(x):
        e = a * (x - c)
        if e.max() > 60.0:
            raise OverflowError('math range error')
        return np.exp(e)
    return lambda x: float(np.sum(ex(x)) + np.sum(x ** 2)), lambda x: a * ex(x) + 2 * x, c - rng.uniform(0, 3, n)


def linear_far(rng):
    """f = s'x far from the origin: the Cauchy step x - g rounds back to x, d = 0, g'd = 0 (not a descent direction)"""
    n = int(rng.integers(2, 6)); s = rng.uniform(0.5, 2, n)
    return lambda x: float(s @ x), lambda x: s.copy(), np.full(n, 1e17) * (1 + rng.uniform(0, 1, n))


def flat_start(rng):
    """all weights tiny: the projected gradient at x0 is already below pgtol"""
    n = int(rng.integers(2, 12)); w = 10 ** rng.uniform(-9, -6)
    return lambda x: float(w * np.sum(np.cos(x))), lambda x: -w * np.sin(x), rng.normal(size=n)


def log_barrier(rng):
    """sum -log(x) + k x'x / 2 from near the boundary: the first step (length 1) leaves the domain, math.log raises
    ValueError"""
    n = int(rng.integers(2, 8)); k = 10 ** rng.uniform(1.5, 3)
    return (lambda x: float(sum(-math.log(v) for v in x) + 0.5 * k * x @ x), lambda x: -1.0 / x + k * x,
            rng.uniform(0.05, 0.5, n))


def linear_steep(rng):
    """f = -s'x + tiny curvature from a small x0: the first step (1 / |d|) is far too short, the search extrapolates to
    stp = stpmax (1e10) and stops there; every later pair is skipped and the run ends on the evaluation limit"""
    n = int(rng.integers(2, 6)); s = rng.uniform(0.5, 2, n)
    return lambda x: float(-s @ x + 1e-30 * x @ x), lambda x: -s + 2e-30 * x, rng.normal(size=n) * 1e-3


FAMILIES = {'rotation': (rotation, 40), 'indefinite': (indefinite, 40), 'far': (far, 30), 'steep': (steep, 40),
            'linear_far': (linear_far, 4), 'flat_start': (flat_start, 4), 'log_barrier': (log_barrier, 8),
            'linear_steep': (linear_steep, 4)}


def skip_unless_skylakex():
    if openblas_core() not in (b'SkylakeX', b'?'):
        pytest.skip('scipy rounds differently on this OpenBLAS kernel family (see test_oracle_golden.py)')


@pytest.mark.parametrize('family', ['rotation', 'far', 'steep', 'log_barrier'])
def test_counters_change_no_rounding(family):
    """The same runs with and without counters: same x, nit, nfev and status, bit for bit (no scipy needed)."""
    make, _ = FAMILIES[family]
    for seed in range(6):
        f, g, x0 = make(np.random.default_rng(seed))

        def fg(x):
            return f(x), g(x)
        plain = c_oracle.lbfgsb_cb(fg, x0)
        counts = c_oracle.new_counts()
        counted = c_oracle.lbfgsb_cb(fg, x0, counts=counts)
        assert np.array_equal(plain[0], counted[0]) and plain[1:] == counted[1:]
        assert counts.sum() > 0
        assert c_oracle.lbfgsb_cb(fg, x0)[1:] == plain[1:]          # counting is switched off again


def test_random_objectives_branch_counts():
    skip_unless_skylakex()
    rng = np.random.default_rng(7)
    total = c_oracle.new_counts()
    for _ in range(60):
        n = int(rng.integers(2, 29))
        total += run_both(*random_objective(n, int(rng.integers(0, 2**31 - 1)), rng.uniform(0, 4), rng.uniform(0, 2),
                                            rng.uniform(0, 0.3)))
    _TOTAL['random'] = total


@pytest.mark.parametrize('M,count', [(3, 16), (6, 4), (10, 4)])
def test_minco_objectives_branch_counts(M, count):
    skip_unless_skylakex()
    cfg = YamlConfig(); cfg.init_wpts_num = M - 1
    w = make_world(2)
    grid = minco_ref.GridMap(w.occ, w.H, w.W, w.res, w.ox, w.oy)
    head, tail = make_problems(w, count, M=M)
    opt = minco_ref.RefOptimizer(cfg)
    total = c_oracle.new_counts()
    for k in range(count):
        q0, ts0 = opt.straight_line_guess(head[k], tail[k])
        opt.set_problem(grid, head[k], tail[k], q0, ts0)
        total += run_both(opt.cost, opt.grad, np.concatenate((q0.reshape(-1), opt.T2tau(ts0))))
    _TOTAL[f'minco M={M}'] = total


@pytest.mark.parametrize('family', list(FAMILIES))
def test_crafted_objectives_branch_counts(family):
    skip_unless_skylakex()
    make, count = FAMILIES[family]
    total = c_oracle.new_counts()
    for seed in range(count):
        total += run_both(*make(np.random.default_rng(seed)))
    _TOTAL[family] = total


def test_every_required_branch_was_taken_in_step_with_scipy():
    """Runs after the tests above (file order) and sums what they recorded."""
    skip_unless_skylakex()
    expected = {'random', 'minco M=3', 'minco M=6', 'minco M=10', *FAMILIES}
    if set(_TOTAL) != expected:
        pytest.skip('needs the whole file: ' + ', '.join(sorted(expected - set(_TOTAL))) + ' did not run')
    names = list(_TOTAL)
    total = sum(_TOTAL.values())
    print('\nbranch counts of the checker in runs bit-identical to scipy')
    print(f'{"branch":22s}' + ''.join(f'{k[:11]:>12s}' for k in names) + f'{"total":>12s}')
    for i, b in enumerate(c_oracle.BRANCHES):
        print(f'{b:22s}' + ''.join(f'{int(_TOTAL[k][i]):12d}' for k in names) + f'{int(total[i]):12d}')
    counts = c_oracle.counts_dict(total)
    missing = [b for b in REQUIRED if counts[b] == 0]
    assert not missing, missing
