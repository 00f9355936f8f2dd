"""csrc/libm_log.h (the device's restatement of glibc's log, the function CPython's math.log calls) compiled for the host
with g++ and compared bit for bit with the C library's own log, called from a helper built with -fno-builtin so that the
compiler cannot fold or replace the call. np.log is not glibc's log and is not used as the reference.

Inputs: random positive finite bit patterns (subnormals included), arguments near 1 (the separate polynomial path), the
map_T2tau arguments (T_max - T_min) / (T - T_min) - 1 of both parameter sets at random T and on the 0.1 grids the
initial guesses use, and the special operands."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'neo_planner_b200', 'csrc')

NEO_SRC = r'''
#include "libm_log.h"
extern "C" void neo_log_arr(long n, const double *x, double *y) { for (long i = 0; i < n; i++) y[i] = neo::log_glibc(x[i]); }
'''
REF_SRC = r'''
#include <math.h>
extern "C" void ref_log_arr(long n, const double *x, double *y) { for (long i = 0; i < n; i++) y[i] = log(x[i]); }
'''
PARAMS = [(2.0, 20.0), (0.5, 5.0)]          # (T_min, T_max): library defaults (EP:12-25) and planner_config.yaml


def _host_has_fma():
    try:
        with open('/proc/cpuinfo') as f:
            flags = next((ln for ln in f if ln.startswith('flags')), '').split()
    except OSError:
        return False
    return 'fma' in flags and 'avx2' in flags


@pytest.fixture(scope='module')
def logs(tmp_path_factory):
    if not _host_has_fma():
        pytest.skip("glibc's log takes its non-FMA variant on this CPU; libm_log.h restates the FMA one")
    cxx = shutil.which('g++') or shutil.which('c++')
    if cxx is None:
        pytest.skip('no host C++ compiler')
    d = tmp_path_factory.mktemp('libm_log')
    (d / 'neo.cpp').write_text(NEO_SRC)
    (d / 'ref.cpp').write_text(REF_SRC)
    so = str(d / 'logs.so')
    subprocess.run([cxx, '-O2', '-std=c++17', '-fPIC', '-ffp-contract=off', '-I', CSRC, '-c', '-o', str(d / 'neo.o'),
                    str(d / 'neo.cpp')], check=True)
    subprocess.run([cxx, '-O2', '-fPIC', '-fno-builtin', '-c', '-o', str(d / 'ref.o'), str(d / 'ref.cpp')], check=True)
    subprocess.run([cxx, '-shared', '-o', so, str(d / 'neo.o'), str(d / 'ref.o'), '-lm'], check=True)
    lib = ctypes.CDLL(so)
    dp = ctypes.POINTER(ctypes.c_double)

    def run(fn, x):
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1)
        y = np.empty_like(x)
        fn(ctypes.c_long(x.size), x.ctypes.data_as(dp), y.ctypes.data_as(dp))
        return y
    return lambda x: (run(lib.neo_log_arr, x), run(lib.ref_log_arr, x))


def assert_same(x, got, want):
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), x[np.isnan(got) != nan][:5]
    bad = (got.view(np.uint64) != want.view(np.uint64)) & ~nan
    assert not bad.any(), f'{bad.sum()} of {x.size} differ, e.g. log({x[bad][0].hex()}) = {got[bad][0].hex()} vs {want[bad][0].hex()}'


def test_random_bit_patterns(logs):
    rng = np.random.default_rng(1)
    u = rng.integers(0, 2**63, size=10_000_000, dtype=np.uint64)              # sign bit clear
    u = u[(u >> np.uint64(52)) != np.uint64(0x7ff)]                             # finite
    sub = rng.integers(1, 2**52, size=100_000, dtype=np.uint64)                # subnormals
    x = np.concatenate([u, sub]).view(np.float64)
    assert_same(x, *logs(x))


def test_near_one(logs):
    rng = np.random.default_rng(2)
    x = 1.0 + rng.uniform(-2.0**-6, 2.0**-6, size=1_000_000)
    assert_same(x, *logs(x))


@pytest.mark.parametrize('T_min,T_max', PARAMS)
def test_map_T2tau_arguments(logs, T_min, T_max):
    rng = np.random.default_rng(3)
    k = np.arange(1, int(round(T_max * 10)) * 2, dtype=np.float64)
    T = np.concatenate([rng.uniform(T_min, T_max, size=1_000_000), k * 0.1, 1.5 * (k * 0.1)])
    with np.errstate(divide="ignore"):
        a = (T_max - T_min) / (T - T_min) - 1.0                                  # T2tau_one's operation order
    a = a[(a > 0) & np.isfinite(a)]
    assert a.size > 1_000_000
    assert_same(a, *logs(a))


def test_special_operands(logs):
    e = np.arange(-1074, 1024, dtype=np.float64)
    k = np.arange(-64, 65, dtype=np.float64)
    one_ulps = np.concatenate([np.nextafter(1.0, 2.0) + 0.0 * k, (1.0 + k * 2.0**-52), (1.0 + k * 2.0**-53)])
    x = np.concatenate([np.ldexp(1.0, e.astype(np.int64)), one_ulps,
                        [np.finfo(np.float64).max, np.finfo(np.float64).tiny, 5e-324, 0.0, -0.0, -1.0, -5e-324,
                         -np.inf, np.inf, np.nan, -np.nan]])
    got, want = logs(x)
    assert_same(x, got, want)
    assert got[-11 + 3] == -np.inf and got[-11 + 4] == -np.inf and got[-11 + 8] == np.inf
