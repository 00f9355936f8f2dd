"""Property test (hypothesis, SURVEY.md §4): the restated L-BFGS-B (oracle/minco_oracle.c, the arithmetic the device
optimizer shares -- tests/test_gpu_lockstep.py) against scipy.optimize.minimize on random objective functions: random
dimension, conditioning, non-quadratic terms, starting points, including functions whose gradient is deliberately NOT
the gradient of the function (like the reference's, SURVEY.md Q1/Q2) so that line searches fail and the memory is
dropped. Same final x bit for bit, same iteration and evaluation counts."""
import ctypes
import glob
import os

import numpy as np
import pytest
import scipy
import scipy.optimize as sopt
from hypothesis import HealthCheck, example, given, settings, strategies as st

from oracle import c_oracle


def openblas_core():
    for so in glob.glob(os.path.join(os.path.dirname(scipy.__file__), '..', 'scipy.libs', '*openblas*')):
        try:
            f = ctypes.CDLL(so).scipy_openblas_get_corename
            f.restype = ctypes.c_char_p
            return f()
        except Exception:
            pass
    return b'?'


def random_objective(n, seed, cond, quartic, skew):
    rng = np.random.default_rng(seed)
    Q = np.linalg.qr(rng.normal(size=(n, n)))[0]
    H = Q @ np.diag(10.0 ** rng.uniform(-cond / 2, cond / 2, n)) @ Q.T
    c = rng.normal(size=n); S = rng.normal(size=(n, n)) * skew
    x0 = rng.normal(size=n) * 3.0

    def f(x):
        return float(0.5 * x @ H @ x + quartic * np.sum((x - c) ** 4) + np.sum(np.cos(x)))

    def g(x):       # skew > 0: not the gradient of f (a rotation is mixed in), as in the reference
        return H @ x + 4.0 * quartic * (x - c) ** 3 - np.sin(x) + S @ np.sin(x)
    return f, g, x0


@settings(max_examples=120, deadline=None, suppress_health_check=[HealthCheck.too_slow], derandomize=True, database=None)
@given(n=st.integers(2, 28), seed=st.integers(0, 2**31 - 1), cond=st.floats(0.0, 4.0), quartic=st.floats(0.0, 2.0),
       skew=st.floats(0.0, 0.3))
# found by this test in round 2: the last trial point differed in one component by one ulp because the restated norm
# added the squares sequentially; OpenBLAS's x87 kernel uses four accumulators for n >= 8 (tests/test_x87_nrm2.py)
@example(n=25, seed=25, cond=1.582789709559926, quartic=1.582789709559926, skew=0.0)
def test_restated_lbfgsb_walks_scipys_iterates(n, seed, cond, quartic, skew):
    f, g, x0 = random_objective(n, seed, cond, quartic, skew)
    res = sopt.minimize(f, x0, method='L-BFGS-B', jac=g, bounds=None, tol=1e-4,
                        options={'maxcor': 10, 'maxfun': 15000, 'maxiter': 15000, 'maxls': 20})
    x, nit, nfev, status = c_oracle.lbfgsb_cb(lambda v: (f(v), g(v)), x0)
    if openblas_core() not in (b'SkylakeX', b'?'):
        pytest.skip('scipy rounds differently on this OpenBLAS kernel family (see test_oracle_golden.py)')
    assert nit == res.nit and nfev == res.nfev, (nit, res.nit, nfev, res.nfev)
    assert np.array_equal(x, res.x)
