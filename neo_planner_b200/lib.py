"""ctypes binding of libneoopt.so (include/neoopt.h). This is the only way Python reaches the optimizer:
there is no CPU fallback, and a missing library or device raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.environ.get('NEO_SO') or os.path.join(HERE, 'libneoopt.so')     # NEO_SO: development override

MAX_PIECES = 10
MAX_ATTEMPTS = 8
ST_CONV_FTOL, ST_CONV_PG, ST_ABNORMAL, ST_MAXITER, ST_OVERFLOW, ST_DOMAIN, ST_NAN = range(7)
STATUS_NAMES = ['CONV_FTOL', 'CONV_PG', 'ABNORMAL', 'MAXITER', 'OVERFLOW', 'DOMAIN', 'NAN']
ERR_NO_DEVICE = -3
ASTAR_FOUND, ASTAR_EXHAUSTED, ASTAR_START_OUTSIDE, ASTAR_LIMIT = range(4)


class NeoError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [('v_max', C.c_double), ('T_min', C.c_double), ('T_max', C.c_double), ('safe_dis', C.c_double),
                ('delta_t', C.c_double), ('weights', C.c_double * 4), ('collision_cost_tol', C.c_double)]

    @classmethod
    def from_config(cls, cfg):
        c = cls()
        c.v_max, c.T_min, c.T_max = float(cfg.v_max), float(cfg.T_min), float(cfg.T_max)
        c.safe_dis, c.delta_t = float(cfg.safe_dis), float(cfg.delta_t)
        for i in range(4):
            c.weights[i] = float(cfg.weights[i])
        c.collision_cost_tol = float(cfg.collision_cost_tol)
        return c


class Result(C.Structure):
    _fields_ = [('x', C.c_void_p), ('ts', C.c_void_p), ('coeffs', C.c_void_p), ('costs', C.c_void_p),
                ('status', C.c_void_p), ('ok', C.c_void_p), ('attempt', C.c_void_p), ('nit', C.c_void_p),
                ('runs', C.c_void_p), ('nfev', C.c_void_p), ('work', C.c_void_p)]


EXPORTS = ['neo_create', 'neo_destroy', 'neo_set_config', 'neo_last_error', 'neo_device_info', 'neo_set_map_esdf',
           'neo_set_map_occupancy', 'neo_set_maps_occupancy', 'neo_set_map_points', 'neo_get_occupancy', 'neo_get_map', 'neo_query_map', 'neo_eval', 'neo_eval_dev', 'neo_optimize',
           'neo_optimize_dev', 'neo_optimize_trace', 'neo_T2tau', 'neo_get_coeffs', 'neo_sample', 'neo_last_kernel_ms', 'neo_fp64_peak',
           'neo_launch_count', 'neo_test_exp_dev', 'neo_test_exp_host', 'neo_test_nrm2_dev', 'neo_test_ddot_dev', 'neo_test_host_pool', 'neo_astar', 'neo_astar_dev']

_lib = None


def load():
    """Loads libneoopt.so; raises if it has not been built (python -m neo_planner_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            raise NeoError(f'{SO} not found: build it with `python -m neo_planner_b200.build` '
                           '(there is no CPU fallback)')
        lib = C.CDLL(SO)
        V, I, D = C.c_void_p, C.c_int, C.c_double
        lib.neo_last_error.restype = C.c_char_p
        lib.neo_last_error.argtypes = [V]
        lib.neo_create.argtypes = [C.POINTER(Config), I, I, C.POINTER(V)]
        lib.neo_destroy.argtypes = [V]
        lib.neo_set_config.argtypes = [V, C.POINTER(Config)]
        lib.neo_device_info.argtypes = [V, V, V, V, V, I]
        lib.neo_set_map_esdf.argtypes = [V, I, I, I, D, D, D, V, V, V]
        lib.neo_set_map_occupancy.argtypes = [V, I, I, I, D, D, D, V]
        lib.neo_set_maps_occupancy.argtypes = [V, I, V, I, I, D, V, V, V]
        lib.neo_get_map.argtypes = [V, I, V, V, V]
        lib.neo_set_map_points.argtypes = [V, I, I, V, D, D, I, I, D, D, D]
        lib.neo_get_occupancy.argtypes = [V, I, V]
        lib.neo_query_map.argtypes = [V, I, I, V, V, V, V]
        lib.neo_eval.argtypes = [V, I, I, V, V, V, V, V, V, V, V, V]
        lib.neo_eval_dev.argtypes = [V, I, I, V, V, V, V, V, V, V, V, V, V]
        lib.neo_optimize.argtypes = [V, I, I, V, V, V, V, V, V, V, I, C.POINTER(Result)]
        lib.neo_optimize_dev.argtypes = [V, I, I, V, V, V, V, V, V, V, I, I, C.POINTER(Result), V]
        lib.neo_optimize_trace.argtypes = [V, I, I, V, V, V, V, V, V, V, I, C.POINTER(Result), I, V, V, V, V, V, V]
        lib.neo_T2tau.argtypes = [C.POINTER(Config), I, V, V, V]
        lib.neo_get_coeffs.argtypes = [V, I, I, V, V, V, V, V]
        lib.neo_sample.argtypes = [V, I, I, V, V, D, I, V, V]
        lib.neo_last_kernel_ms.argtypes = [V, V]
        lib.neo_fp64_peak.argtypes = [V, V]
        lib.neo_launch_count.argtypes = [V, V]
        lib.neo_test_exp_dev.argtypes = [V, I, V, V]
        lib.neo_test_exp_host.argtypes = [I, V, V]
        lib.neo_test_nrm2_dev.argtypes = [V, I, I, V, V]
        lib.neo_test_ddot_dev.argtypes = [V, I, I, V, V, V, V]
        lib.neo_astar.argtypes = [V, I, V, V, V, I, I, V, V, V, V, V]
        lib.neo_astar_dev.argtypes = [V, I, V, V, V, I, I, V, V, V, V, V, V]
        _lib = lib
    return _lib


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != tuple(shape):
        raise ValueError(f'expected shape {tuple(shape)}, got {a.shape}')
    return a


def pad_state(s):
    """(..., k<=3, 2) -> (..., 3, 2), zero padded like read_planning_conditions (EP:170-184)."""
    s = np.asarray(s, dtype=np.float64)
    if s.shape[-1] != 2:
        raise ValueError('only planar problems (D = 2) are supported, as in the reference node (NODE:593-595)')
    if s.ndim >= 2 and s.shape[-2] == 3 and s.flags.c_contiguous:
        return s                               # already padded: no copy (3 MB per call at 65,536 problems)
    out = np.zeros(s.shape[:-2] + (3, 2))
    k = min(3, s.shape[-2])
    out[..., :k, :] = s[..., :k, :]
    return out


class Handle:
    """Owns one neo_handle (one CUDA device, one stream, a set of map slots)."""

    def __init__(self, cfg, device: int = 0, max_maps: int = 1):
        self.lib = load()
        self.cfg = Config.from_config(cfg)
        self.h = C.c_void_p()
        rc = self.lib.neo_create(C.byref(self.cfg), int(device), int(max_maps), C.byref(self.h))
        if rc != 0:
            raise NeoError(f'neo_create failed ({rc}): {self.lib.neo_last_error(None).decode()}')
        self.max_maps = max_maps
        self.device = device

    def close(self):
        if getattr(self, 'h', None):
            self.lib.neo_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise NeoError(f'libneoopt error {rc}: {self.lib.neo_last_error(self.h).decode()}')

    def set_config(self, cfg):
        self.cfg = Config.from_config(cfg)
        self._ck(self.lib.neo_set_config(self.h, C.byref(self.cfg)))

    def device_info(self):
        sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
        name = C.create_string_buffer(128)
        self._ck(self.lib.neo_device_info(self.h, C.addressof(sm), C.addressof(ma), C.addressof(mi),
                                          C.addressof(name), 128))
        return dict(sm_count=sm.value, cc=(ma.value, mi.value), name=name.value.decode())

    # ---- maps -----------------------------------------------------------------------------------
    def set_map_esdf(self, slot, res, ox, oy, esdf, gx, gy):
        esdf = f64(esdf); H, W = esdf.shape
        gx = f64(gx, (H, W)); gy = f64(gy, (H, W))
        self._ck(self.lib.neo_set_map_esdf(self.h, slot, H, W, res, ox, oy, ptr(esdf), ptr(gx), ptr(gy)))

    def set_map_occupancy(self, slot, H, W, res, ox, oy, occ):
        occ = np.ascontiguousarray(np.asarray(occ).reshape(H, W), dtype=np.int8)
        self._ck(self.lib.neo_set_map_occupancy(self.h, slot, H, W, res, ox, oy, ptr(occ)))

    def set_maps_occupancy(self, slots, H, W, res, ox, oy, occ):
        """K maps of one shape in one call: slots (K), ox / oy (K), occ (K, H, W)."""
        slots = np.ascontiguousarray(slots, dtype=np.int32); K = slots.size
        occ = np.ascontiguousarray(np.asarray(occ).reshape(K, H, W), dtype=np.int8)
        ox = f64(np.broadcast_to(np.asarray(ox, dtype=np.float64), (K,))); oy = f64(np.broadcast_to(np.asarray(oy, dtype=np.float64), (K,)))
        self._ck(self.lib.neo_set_maps_occupancy(self.h, K, ptr(slots), H, W, float(res), ptr(ox), ptr(oy), ptr(occ)))

    def set_map_points(self, slot, xyz, z_min, z_max, H, W, res, ox, oy):
        xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        self._ck(self.lib.neo_set_map_points(self.h, slot, xyz.shape[0], ptr(xyz), z_min, z_max, H, W, res, ox, oy))

    def get_occupancy(self, slot, H, W):
        occ = np.empty((H, W), np.int8)
        self._ck(self.lib.neo_get_occupancy(self.h, slot, ptr(occ)))
        return occ

    def get_map(self, slot, H, W):
        e = np.empty((H, W)); gx = np.empty((H, W)); gy = np.empty((H, W))
        self._ck(self.lib.neo_get_map(self.h, slot, ptr(e), ptr(gx), ptr(gy)))
        return e, gx, gy

    def query_map(self, slot, xy):
        xy = f64(xy).reshape(-1, 2); n = xy.shape[0]
        idx = np.empty((n, 2), np.int32); d = np.empty(n); g = np.empty((n, 2))
        self._ck(self.lib.neo_query_map(self.h, slot, n, ptr(xy), ptr(idx), ptr(d), ptr(g)))
        return idx, d, g

    # ---- cost / gradient ----------------------------------------------------------------------------
    def eval(self, M, x, head, tail, map_ids=None, want_coeffs=False):
        x = f64(x); B = x.shape[0]; n = 3 * M - 2
        x = f64(x, (B, n)); head = f64(pad_state(head), (B, 3, 2)); tail = f64(pad_state(tail), (B, 3, 2))
        ids = None if map_ids is None else np.ascontiguousarray(map_ids, dtype=np.int32)
        costs = np.zeros((B, 4)); grad = np.zeros((B, n)); status = np.zeros(B, np.int32)
        coeffs = np.zeros((B, 6 * M, 2)) if want_coeffs else None
        ts = np.zeros((B, M)) if want_coeffs else None
        self._ck(self.lib.neo_eval(self.h, B, M, ptr(x), ptr(head), ptr(tail), ptr(ids), ptr(costs), ptr(grad),
                                   ptr(status), ptr(coeffs), ptr(ts)))
        out = dict(costs=costs, grad=grad, status=status)
        if want_coeffs:
            out.update(coeffs=coeffs, ts=ts)
        return out

    # ---- optimisation ---------------------------------------------------------------------------------
    @staticmethod
    def alloc_result(B, M, work=True):
        n = 3 * M - 2
        return dict(x=np.zeros((B, n)), ts=np.zeros((B, M)), coeffs=np.zeros((B, 6 * M, 2)), costs=np.zeros((B, 4)),
                    status=np.zeros(B, np.int32), ok=np.zeros(B, np.int32), attempt=np.zeros(B, np.int32),
                    nit=np.zeros(B, np.int32), runs=np.zeros(B, np.int32), nfev=np.zeros(B, np.int32),
                    work=np.zeros((B, 4), np.int64) if work else None)

    @staticmethod
    def result_struct(out):
        r = Result()
        for k, _ in Result._fields_:
            setattr(r, k, None if out.get(k) is None else out[k].ctypes.data)
        return r

    @staticmethod
    def _plan_inputs(M, q0, ts0, head, tail, map_ids, retry_q, retry_ts, max_attempts):
        """Contiguous arrays of the shapes neo_optimize reads: (B, q0, ts0, head, tail, map_ids, retry_q, retry_ts)."""
        q0 = f64(q0); B = q0.shape[0]
        q0 = f64(q0, (B, 2, M - 1)); ts0 = f64(ts0, (B, M))
        head = f64(pad_state(head), (B, 3, 2)); tail = f64(pad_state(tail), (B, 3, 2))
        ids = None if map_ids is None else np.ascontiguousarray(map_ids, dtype=np.int32)
        if max_attempts > 1:
            retry_q = f64(retry_q, (B, max_attempts - 1, 2, M - 1)); retry_ts = f64(retry_ts, (M,))
        else:
            retry_q = retry_ts = None
        return B, q0, ts0, head, tail, ids, retry_q, retry_ts

    def optimize(self, M, q0, ts0, head, tail, map_ids=None, retry_q=None, retry_ts=None, max_attempts=1, out=None):
        B, *args = self._plan_inputs(M, q0, ts0, head, tail, map_ids, retry_q, retry_ts, max_attempts)
        if out is None:
            out = self.alloc_result(B, M)
        r = self.result_struct(out)
        self._ck(self.lib.neo_optimize(self.h, B, M, *map(ptr, args), max_attempts, C.byref(r)))
        return out

    def optimize_trace(self, M, q0, ts0, head, tail, map_ids=None, retry_q=None, retry_ts=None, max_attempts=1, cap=512):
        """neo_optimize_trace: optimize() plus, per task (attempt * B + problem), the first `cap` evaluations the device
        made: dict(x (A*B, cap, n), f, g, costs, status, len (A*B)). For the lockstep tests."""
        B, *args = self._plan_inputs(M, q0, ts0, head, tail, map_ids, retry_q, retry_ts, max_attempts)
        n = 3 * M - 2
        out = self.alloc_result(B, M)
        r = self.result_struct(out)
        T = B * max_attempts
        tr = dict(x=np.zeros((T, cap, n)), f=np.zeros((T, cap)), g=np.zeros((T, cap, n)), costs=np.zeros((T, cap, 4)),
                  status=np.zeros((T, cap), np.int32), len=np.zeros(T, np.int32))
        self._ck(self.lib.neo_optimize_trace(self.h, B, M, *map(ptr, args), max_attempts, C.byref(r), cap, ptr(tr['x']),
                                             ptr(tr['f']), ptr(tr['g']), ptr(tr['costs']), ptr(tr['status']), ptr(tr['len'])))
        return out, tr

    def T2tau(self, ts):
        ts = f64(ts); tau = np.zeros_like(ts); st = np.zeros(ts.size, np.int32)
        self._ck(self.lib.neo_T2tau(C.byref(self.cfg), ts.size, ptr(ts), ptr(tau), ptr(st)))
        return tau, st.reshape(ts.shape)

    # ---- coefficients / sampling -------------------------------------------------------------------------
    def get_coeffs(self, M, q, ts, head, tail):
        q = f64(q); B = q.shape[0]
        q = f64(q, (B, 2, M - 1)); ts = f64(ts, (B, M))
        head = f64(pad_state(head), (B, 3, 2)); tail = f64(pad_state(tail), (B, 3, 2))
        out = np.zeros((B, 6 * M, 2))
        self._ck(self.lib.neo_get_coeffs(self.h, B, M, ptr(q), ptr(ts), ptr(head), ptr(tail), ptr(out)))
        return out

    def sample(self, M, coeffs, ts, hz):
        coeffs = f64(coeffs); B = coeffs.shape[0]
        coeffs = f64(coeffs, (B, 6 * M, 2)); ts = f64(ts, (B, M))
        count = np.zeros(B, np.int32)
        self._ck(self.lib.neo_sample(self.h, B, M, ptr(coeffs), ptr(ts), float(hz), 0, None, ptr(count)))
        mx = max(int(count.max()), 1)
        states = np.zeros((B, mx, 3, 2))
        self._ck(self.lib.neo_sample(self.h, B, M, ptr(coeffs), ptr(ts), float(hz), mx, ptr(states), ptr(count)))
        return states, count

    # ---- geometric initializer -------------------------------------------------------------------------
    def astar(self, start, target, map_ids=None, max_path=0, max_closed=0):
        """neo_astar: A* + pruning for B start/target pairs -> dict(pruned (B,4,2), path_len, status, closed[, path])."""
        start = f64(start).reshape(-1, 2); B = start.shape[0]
        target = f64(target, (B, 2))
        ids = None if map_ids is None else np.ascontiguousarray(map_ids, dtype=np.int32)
        pruned = np.zeros((B, 4, 2)); plen = np.zeros(B, np.int32); st = np.zeros(B, np.int32); cl = np.zeros(B, np.int32)
        path = np.zeros((B, max_path, 2)) if max_path > 0 else None
        self._ck(self.lib.neo_astar(self.h, B, ptr(start), ptr(target), ptr(ids), int(max_closed), int(max_path), ptr(path),
                                    ptr(plen), ptr(pruned), ptr(st), ptr(cl)))
        out = dict(pruned=pruned, path_len=plen, status=st, closed=cl)
        if path is not None:
            out['path'] = path
        return out

    # ---- measurement -----------------------------------------------------------------------------------
    def last_kernel_ms(self):
        ms = C.c_float()
        self._ck(self.lib.neo_last_kernel_ms(self.h, C.addressof(ms)))
        return ms.value

    def fp64_peak(self):
        t = C.c_double()
        self._ck(self.lib.neo_fp64_peak(self.h, C.addressof(t)))
        return t.value

    def launch_count(self):
        n = C.c_int64()
        self._ck(self.lib.neo_launch_count(self.h, C.addressof(n)))
        return n.value

    def exp_dev(self, x):
        x = f64(x).reshape(-1); y = np.empty_like(x)
        self._ck(self.lib.neo_test_exp_dev(self.h, x.size, ptr(x), ptr(y)))
        return y

    def nrm2_dev(self, v):
        """dnrm2 of each row of v (count, n) by the optimizer's nrm2_x87 on the device"""
        v = f64(v); count, n = v.shape; out = np.empty(count)
        self._ck(self.lib.neo_test_nrm2_dev(self.h, count, n, ptr(v), ptr(out)))
        return out

    def ddot_dev(self, a, b):
        """row-wise a . b (count, n) by the optimizer's two inner products on the device: (blas_ddot, loop_dot)"""
        a = f64(a); count, n = a.shape; b = f64(b, (count, n))
        blas = np.empty(count); loop = np.empty(count)
        self._ck(self.lib.neo_test_ddot_dev(self.h, count, n, ptr(a), ptr(b), ptr(blas), ptr(loop)))
        return blas, loop


def exp_host(x):
    x = f64(x).reshape(-1); y = np.empty_like(x)
    load().neo_test_exp_host(x.size, ptr(x), ptr(y))
    return y
