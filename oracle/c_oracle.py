"""ctypes loader for oracle/libminco_oracle.so (the plain-C CPU checker). TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline leg may import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, 'libminco_oracle.so')

STATUS_NAMES = ['CONV_FTOL', 'CONV_PG', 'ABNORMAL', 'MAXITER', 'OVERFLOW', 'DOMAIN', 'NAN']


class Params(C.Structure):
    _fields_ = [('v_max', C.c_double), ('T_min', C.c_double), ('T_max', C.c_double), ('safe_dis', C.c_double),
                ('delta_t', C.c_double), ('w', C.c_double * 4), ('collision_cost_tol', C.c_double),
                ('init_T', C.c_double)]

    @classmethod
    def from_config(cls, cfg):
        p = cls()
        p.v_max, p.T_min, p.T_max, p.safe_dis, p.delta_t = cfg.v_max, cfg.T_min, cfg.T_max, cfg.safe_dis, cfg.delta_t
        for i in range(4):
            p.w[i] = float(cfg.weights[i])
        p.collision_cost_tol = float(cfg.collision_cost_tol)
        p.init_T = float(cfg.init_T)
        return p


class Map(C.Structure):
    _fields_ = [('H', C.c_int), ('W', C.c_int), ('res', C.c_double), ('ox', C.c_double), ('oy', C.c_double),
                ('esdf', C.c_void_p), ('gx', C.c_void_p), ('gy', C.c_void_p)]


def build(force: bool = False) -> str:
    src = os.path.join(HERE, 'minco_oracle.c')
    if force or not os.path.exists(SO) or os.path.getmtime(SO) < os.path.getmtime(src):
        subprocess.check_call(['make', '-C', HERE, '-s', '-B'])
    return SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.orc_get_coeffs.restype = C.c_int
        _lib.orc_sample_count.restype = C.c_int
        _lib.orc_sample_count.argtypes = [C.c_int, C.c_void_p, C.c_double]
        _lib.orc_sample.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p]
        _lib.orc_esdf_build.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.orc_esdf_brute.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p]
        _lib.orc_count_into.argtypes = [C.c_void_p]
        _lib.orc_count_size.restype = C.c_int
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class OracleMap:
    """Owns the three (H, W) fp64 arrays the C checker reads."""

    def __init__(self, occ, H, W, res, ox, oy, arrays=None):
        self.H, self.W, self.res, self.ox, self.oy = int(H), int(W), float(res), float(ox), float(oy)
        if arrays is None:
            occ8 = np.ascontiguousarray(np.asarray(occ).reshape(H, W), dtype=np.int8)
            self.esdf = np.empty((H, W)); self.gx = np.empty((H, W)); self.gy = np.empty((H, W))
            lib().orc_esdf_build(_p(occ8), self.H, self.W, self.res, _p(self.esdf), _p(self.gx), _p(self.gy))
        else:
            self.esdf, self.gx, self.gy = (f64(a) for a in arrays)
        self.c = Map(self.H, self.W, self.res, self.ox, self.oy, self.esdf.ctypes.data, self.gx.ctypes.data,
                     self.gy.ctypes.data)

    @classmethod
    def from_world(cls, w):
        return cls(w.occ, w.H, w.W, w.res, w.ox, w.oy)

    def query(self, xy):
        xy = f64(xy).reshape(-1, 2)
        n = xy.shape[0]
        idx = np.empty((n, 2), np.int32); d = np.empty(n); g = np.empty((n, 2))
        lib().orc_query(C.byref(self.c), C.c_int(n), _p(xy), _p(idx), _p(d), _p(g))
        return idx, d, g


def esdf_brute(occ, H, W, res):
    occ8 = np.ascontiguousarray(np.asarray(occ).reshape(H, W), dtype=np.int8)
    out = np.empty((H, W))
    lib().orc_esdf_brute(_p(occ8), H, W, float(res), _p(out))
    return out


def pad_state(s):
    """(k<=3, 2) -> (3, 2) zero padded, as EP:170-184."""
    s = np.asarray(s, dtype=np.float64)
    out = np.zeros(s.shape[:-2] + (3, 2))
    out[..., :min(3, s.shape[-2]), :] = s[..., :3, :]
    return out


def eval_batch(params, omap, M, head, tail, x):
    x = f64(x); B = x.shape[0]; n = x.shape[1]
    head = f64(pad_state(head)); tail = f64(pad_state(tail))
    costs = np.zeros((B, 4)); grad = np.zeros((B, n)); status = np.zeros(B, np.int32)
    lib().orc_eval_batch(C.byref(params), C.byref(omap.c), C.c_int(B), C.c_int(M), _p(head), _p(tail), _p(x),
                         _p(costs), _p(grad), _p(status))
    return costs, grad, status


def get_coeffs(M, head, tail, q, ts):
    head = f64(pad_state(head)); tail = f64(pad_state(tail)); q = f64(q); ts = f64(ts)
    out = np.zeros((6 * M, 2))
    rc = lib().orc_get_coeffs(C.c_int(M), _p(head), _p(tail), _p(q), _p(ts), _p(out))
    assert rc == 0
    return out


def plan_batch(params, omap, M, head, tail, q0, ts0, retry_q=None, retry_ts=None, max_attempts=1):
    """q0: (B, 2, M-1); ts0: (B, M); retry_q: (B, max_attempts-1, 2, M-1); retry_ts: (M,)."""
    q0 = f64(q0); B = q0.shape[0]; n = 2 * (M - 1) + M
    ts0 = f64(ts0)
    head = f64(pad_state(head)); tail = f64(pad_state(tail))
    if max_attempts > 1:
        retry_q = f64(retry_q); retry_ts = f64(retry_ts)
        assert retry_q.shape == (B, max_attempts - 1, 2, M - 1)
    out = dict(x=np.zeros((B, n)), ts=np.zeros((B, M)), coeffs=np.zeros((B, 6 * M, 2)), costs=np.zeros((B, 4)),
               status=np.zeros(B, np.int32), ok=np.zeros(B, np.int32), attempt=np.zeros(B, np.int32),
               nit=np.zeros(B, np.int32), runs=np.zeros(B, np.int32), nfev=np.zeros(B, np.int32))
    lib().orc_plan_batch(C.byref(params), C.byref(omap.c), C.c_int(B), C.c_int(M), _p(head), _p(tail), _p(q0), _p(ts0),
                         _p(retry_q) if max_attempts > 1 else None, _p(retry_ts) if max_attempts > 1 else None,
                         C.c_int(max_attempts), _p(out['x']), _p(out['ts']), _p(out['coeffs']), _p(out['costs']),
                         _p(out['status']), _p(out['ok']), _p(out['attempt']), _p(out['nit']), _p(out['runs']),
                         _p(out['nfev']))
    return out


class Result(C.Structure):
    _fields_ = [('x', C.c_double * 46), ('costs', C.c_double * 4), ('f', C.c_double), ('status', C.c_int),
                ('nit', C.c_int), ('nfev', C.c_int)]


FG_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                    C.POINTER(C.c_double))


def dnrm2(a):
    """The restated OpenBLAS dnrm2 (x87 extended arithmetic, four accumulators) on one vector."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    f = lib().orc_dnrm2
    f.restype = C.c_double
    f.argtypes = [C.c_int, C.POINTER(C.c_double)]
    return float(f(a.size, a.ctypes.data_as(C.POINTER(C.c_double))))


# the optimizer's branch counters (minco_oracle.c, enum OC_*), in order
BRANCHES = ([f'dir_col{c}' for c in range(11)] +
            ['factor_fail1', 'factor_fail2', 'nondescent_col0', 'nondescent_col', 'maxls', 'abnormal', 'reset_failed_search',
             'skip_update', 'wrap', 'reset_after_wrap', 'accept_stp1', 'accept_stp', 'cache_hit'] +
            [f'dcstep{k}_{"brackt" if b else "open"}' for k in range(1, 5) for b in (0, 1)] +
            ['exit_conv', 'exit_bound', 'exit_xtol', 'exit_stpmax', 'exit_stpmin', 'stx_fallback',
             'pg_x0', 'pg', 'ftol', 'maxiter', 'eval_overflow', 'eval_domain', 'eval_nan'])


def new_counts():
    """A zeroed counter array for the `counts=` argument of lbfgsb_cb / lbfgsb_replay (counts are added to it)."""
    assert lib().orc_count_size() == len(BRANCHES)
    return np.zeros(len(BRANCHES), np.int64)


def counts_dict(c):
    return {k: int(v) for k, v in zip(BRANCHES, c)}


def _counted(counts, call):
    if counts is None:
        return call()
    assert counts.dtype == np.int64 and counts.shape == (len(BRANCHES),) and counts.flags.c_contiguous
    lib().orc_count_into(_p(counts))
    try:
        return call()
    finally:
        lib().orc_count_into(None)


def ddot(a, b):
    """The restated inner products on one pair of vectors: (the BLAS ddot kernel's order, scipy's own mul + add loop)."""
    a = np.ascontiguousarray(a, dtype=np.float64); b = np.ascontiguousarray(b, dtype=np.float64)
    assert a.shape == b.shape and a.ndim == 1
    out = []
    for f in (lib().orc_ddot, lib().orc_loop_dot):
        f.restype = C.c_double
        f.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        out.append(float(f(a.size, _p(a), _p(b))))
    return tuple(out)


def lbfgsb_cb(fg, x0, counts=None):
    """The C restatement of scipy's L-BFGS-B around a Python evaluator fg(x) -> (f, g). Returns (x, nit, nfev, status).
    counts: an array from new_counts() to which the run's branch counters are added."""
    x0 = f64(x0); n = x0.size

    def tramp(_ctx, n_, xp, fp, gp, cp):
        x = np.array([xp[i] for i in range(n_)])
        try:
            f, g = fg(x)
        except OverflowError:
            return 4
        except (ValueError, ZeroDivisionError):
            return 5
        fp[0] = float(f)
        for i in range(n_):
            gp[i] = float(g[i])
        for i in range(4):
            cp[i] = 0.0
        return 0
    res = Result()
    cb = FG_FN(tramp)
    st = _counted(counts, lambda: lib().orc_lbfgsb_cb(C.c_int(n), _p(x0), cb, None, C.byref(res)))
    return np.array(res.x[:n]), res.nit, res.nfev, st


def lbfgsb_traced(params, omap, M, head, tail, x0, cap=4096):
    """One minimize() call of the checker with every evaluation recorded. Returns dict(x, nit, nfev, status, xs, fs, gs)."""
    x0 = f64(x0); n = x0.size
    head = f64(pad_state(head)); tail = f64(pad_state(tail))
    xs = np.zeros((cap, n)); fs = np.zeros(cap); gs = np.zeros((cap, n))
    res = Result()
    k = lib().orc_lbfgsb_traced(C.byref(params), C.byref(omap.c), C.c_int(M), _p(head), _p(tail), _p(x0), C.byref(res),
                                C.c_int(cap), _p(xs), _p(fs), _p(gs))
    return dict(x=np.array(res.x[:n]), nit=res.nit, nfev=res.nfev, status=res.status, costs=np.array(res.costs[:]),
                xs=xs[:k], fs=fs[:k], gs=gs[:k])


def lbfgsb_replay(x0, xs, fs, gs, costs=None, status=None, counts=None):
    """Feeds recorded evaluations (the device's) to the checker's optimizer. Returns dict(x, nit, nfev, status,
    first_bad (-1: every requested point was bit-identical to the recorded one), used). counts: as for lbfgsb_cb; for a
    replay that matched to the end they are the branches the recorded run took."""
    x0 = f64(x0); n = x0.size
    xs = f64(xs).reshape(-1, n); gs = f64(gs).reshape(-1, n); fs = f64(fs)
    k = xs.shape[0]
    costs = np.zeros((k, 4)) if costs is None else f64(costs)
    st = None if status is None else np.ascontiguousarray(status, dtype=np.int32)
    res = Result(); bad = C.c_int(-1); used = C.c_int(0)
    rc = _counted(counts, lambda: lib().orc_lbfgsb_replay(C.c_int(n), _p(x0), C.c_int(k), _p(xs), _p(fs), _p(gs), _p(costs),
                                                          None if st is None else _p(st), C.byref(res), C.byref(bad),
                                                          C.byref(used)))
    return dict(x=np.array(res.x[:n]), nit=res.nit, nfev=res.nfev, status=rc, first_bad=bad.value, used=used.value,
                costs=np.array(res.costs[:]))


def plan_batch_mt(params, maps, M, head, tail, q0, ts0, retry_q=None, retry_ts=None, max_attempts=1, map_ids=None,
                  threads=None):
    """plan_batch over several maps on `threads` host threads (default: all cores). maps: list of OracleMap."""
    threads = threads or os.cpu_count() or 1
    q0 = f64(q0); B = q0.shape[0]; n = 2 * (M - 1) + M
    ts0 = f64(ts0)
    head = f64(pad_state(head)); tail = f64(pad_state(tail))
    if max_attempts > 1:
        retry_q = f64(retry_q); retry_ts = f64(retry_ts)
        assert retry_q.shape == (B, max_attempts - 1, 2, M - 1)
    ids = None if map_ids is None else np.ascontiguousarray(map_ids, dtype=np.int32)
    arr = (C.c_void_p * len(maps))(*[C.addressof(m_.c) for m_ in maps])
    out = dict(x=np.zeros((B, n)), ts=np.zeros((B, M)), coeffs=np.zeros((B, 6 * M, 2)), costs=np.zeros((B, 4)),
               status=np.zeros(B, np.int32), ok=np.zeros(B, np.int32), attempt=np.zeros(B, np.int32),
               nit=np.zeros(B, np.int32), runs=np.zeros(B, np.int32), nfev=np.zeros(B, np.int32))
    lib().orc_plan_batch_mt(C.byref(params), arr, None if ids is None else _p(ids), C.c_int(B), C.c_int(M), _p(head),
                            _p(tail), _p(q0), _p(ts0), _p(retry_q) if max_attempts > 1 else None,
                            _p(retry_ts) if max_attempts > 1 else None, C.c_int(max_attempts), C.c_int(threads),
                            _p(out['x']), _p(out['ts']), _p(out['coeffs']), _p(out['costs']), _p(out['status']),
                            _p(out['ok']), _p(out['attempt']), _p(out['nit']), _p(out['runs']), _p(out['nfev']))
    return out


def sample(M, coeffs, ts, hz):
    coeffs = f64(coeffs); ts = f64(ts)
    N = lib().orc_sample_count(C.c_int(M), _p(ts), float(hz))
    out = np.zeros((N, 3, 2))
    lib().orc_sample(C.c_int(M), _p(coeffs), _p(ts), float(hz), C.c_int(N), _p(out))
    return out
