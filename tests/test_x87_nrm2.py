"""csrc/x87_nrm2.h (the device's restatement of OpenBLAS's x87 dnrm2 kernel: 80-bit extended arithmetic on integer pairs,
four accumulators, D + ((C + A) + B), fsqrt, one rounding to double) compiled for the host and compared with the REAL
kernel -- scipy.linalg.blas.dnrm2 calls the bundled OpenBLAS -- and with the checker's `long double` restatement
(oracle/minco_oracle.c: blas_dnrm2), bit for bit, for every n the optimizer uses (1..28) and beyond. Vectors include the
adversarial kind: sums of squares that land next to a rounding boundary of the result, where the summation order and
the extended format decide the last bit."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
from scipy.linalg import blas

from oracle import c_oracle
from test_lbfgsb_property import openblas_core

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, 'devtools', 'x87_host.cpp')
HDR = os.path.join(ROOT, 'neo_planner_b200', 'csrc', 'x87_nrm2.h')
SO = os.path.join(ROOT, 'devtools', '_x87_host.so')


@pytest.fixture(scope='module')
def sim():
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(SRC), os.path.getmtime(HDR)):
        cxx = shutil.which('g++') or shutil.which('c++')
        if cxx is None:
            pytest.skip('no host C++ compiler')
        subprocess.run([cxx, '-O2', '-std=c++17', '-shared', '-fPIC', '-ffp-contract=off', '-o', SO, SRC], check=True)
    lib = ctypes.CDLL(SO)
    dp = ctypes.POINTER(ctypes.c_double)

    def run(v):
        v = np.ascontiguousarray(v, dtype=np.float64)
        count, n = v.shape
        fast = np.zeros(count); exact = np.zeros(count)
        lib.sim_x87_nrm2(count, n, v.ctypes.data_as(dp), fast.ctypes.data_as(dp), exact.ctypes.data_as(dp))
        return fast, exact
    return run


def vectors(rng, count, n):
    """Random vectors of mixed scales, plus vectors whose LAST component is tuned so that the norm lands within a few
    2^-64 of the midpoint between two doubles (the cases the last bit of the x87 result depends on)."""
    v = rng.normal(size=(count, n)) * 10.0 ** rng.uniform(-6, 6, size=(count, 1)) * 10.0 ** rng.uniform(-2, 2, size=(count, n))
    k = count // 2
    if n >= 2:
        import math
        for i in range(k):
            head = v[i, :-1]
            s = math.fsum(float(x) * float(x) for x in head)
            target = math.sqrt(s) * (1.0 + rng.uniform(0.1, 2.0))                  # a norm a bit above the head's
            m, e = math.frexp(target)
            target = math.ldexp(math.floor(m * 2 ** 53) + 0.5, e - 53)             # midpoint between two doubles (as exact as a double can say)
            rest = target * target - s
            if rest > 0:
                v[i, -1] = math.sqrt(rest) * (1.0 + rng.integers(-3, 4) * 2.0 ** -52)
    return v


@pytest.mark.parametrize('n', list(range(1, 33)) + [40, 63])
def test_emulation_equals_the_real_kernel(sim, n):
    rng = np.random.default_rng(1000 + n)
    v = vectors(rng, 4000 if n < 8 else 16000, n)       # n >= 8: four accumulators, the order matters in ~1 of 3000 vectors
    fast, exact = sim(v)
    real = np.array([blas.dnrm2(row) for row in v])
    checker = np.array([c_oracle.dnrm2(row) for row in v])
    assert np.array_equal(exact, real), (n, int((exact != real).sum()))
    assert np.array_equal(fast, real), (n, int((fast != real).sum()))
    assert np.array_equal(checker, real), (n, int((checker != real).sum()))


def test_edge_magnitudes(sim):
    v = np.array([[0.0, 0.0, 0.0], [1e-200, 2e-200, 0.0], [1e150, 1e150, 1e150], [3.0, 4.0, 0.0], [1.0, 0.0, 0.0],
                  [2.0 ** -600, 2.0 ** -600, 2.0 ** -600]])
    fast, exact = sim(v)
    real = np.array([blas.dnrm2(row) for row in v])
    assert np.array_equal(fast, real) and np.array_equal(exact, real)


def dot_vectors(rng, count, n):
    """Pairs whose products span twelve decades and whose sum cancels to a small fraction of its largest term, so that the
    summation order and which products are fused decide the last bits."""
    a = rng.normal(size=(count, n)) * 10.0 ** rng.uniform(-6, 6, size=(count, 1)) * 10.0 ** rng.uniform(-3, 3, size=(count, n))
    b = rng.normal(size=(count, n)) * 10.0 ** rng.uniform(-3, 3, size=(count, n))
    if n >= 2:
        k = count // 2
        p = a[:k, :-1] * b[:k, :-1]
        a[:k, -1] = -p.sum(axis=1) / b[:k, -1] * (1.0 + rng.normal(size=k) * 1e-9)
    return a, b


@pytest.fixture(scope='module')
def dev():
    from neo_planner_b200 import lib
    from neo_planner_b200.worlds import YamlConfig
    h = lib.Handle(YamlConfig(), 0, 1)
    yield h
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize('n', list(range(1, 33)) + [40, 63])
def test_device_build_nrm2_equals_the_real_kernel(dev, n):
    """nrm2_x87 of lbfgsb_tile.cuh compiled by nvcc with the library's flags (--fmad=true: its two-sum is written with
    plain operators that nvcc may contract) on the adversarial vectors above."""
    rng = np.random.default_rng(1000 + n)
    v = vectors(rng, 4000 if n < 8 else 16000, n)
    got = dev.nrm2_dev(v)
    checker = np.array([c_oracle.dnrm2(row) for row in v])
    assert np.array_equal(got, checker), (n, int((got != checker).sum()))
    real = np.array([blas.dnrm2(row) for row in v])
    assert np.array_equal(got, real), (n, int((got != real).sum()))


@pytest.mark.gpu
def test_device_build_nrm2_edge_magnitudes(dev):
    v = np.array([[0.0, 0.0, 0.0], [1e-200, 2e-200, 0.0], [1e150, 1e150, 1e150], [3.0, 4.0, 0.0], [1.0, 0.0, 0.0],
                  [2.0 ** -600, 2.0 ** -600, 2.0 ** -600], [1e-310, 0.0, 5e-324], [1e300, -1e300, 1e-300],
                  [2.0 ** 511, 2.0 ** 511, 0.0], [-7.0, 0.0, -24.0]])
    got = dev.nrm2_dev(v)
    assert np.array_equal(got, np.array([blas.dnrm2(row) for row in v]))
    assert np.array_equal(got, np.array([c_oracle.dnrm2(row) for row in v]))


@pytest.mark.gpu
@pytest.mark.parametrize('n', list(range(1, 32)))
def test_device_build_ddot_equals_the_checker(dev, n):
    """blas_ddot (fused chain; the four-lane prefix from n = 16) and loop_dot (multiply, then add) of lbfgsb_tile.cuh as
    nvcc compiles them for the device, against the checker's restatement and, for the BLAS order, scipy's own ddot."""
    rng = np.random.default_rng(2000 + n)
    a, b = dot_vectors(rng, 4000, n)
    blas_d, loop_d = dev.ddot_dev(a, b)
    ref = np.array([c_oracle.ddot(x, y) for x, y in zip(a, b)])
    assert np.array_equal(blas_d, ref[:, 0]), (n, int((blas_d != ref[:, 0]).sum()))
    assert np.array_equal(loop_d, ref[:, 1]), (n, int((loop_d != ref[:, 1]).sum()))
    if n >= 2:
        assert (ref[:, 0] != ref[:, 1]).sum() >= 100        # the vectors tell the two orders apart
    if openblas_core() in (b'SkylakeX', b'?'):
        real = np.array([blas.ddot(x, y) for x, y in zip(a, b)])
        assert np.array_equal(blas_d, real), (n, int((blas_d != real).sum()))
