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
           'neo_launch_count', 'neo_test_exp_dev', 'neo_test_exp_host', 'neo_test_nrm2_dev', 'neo_test_ddot_dev', 'neo_test_host_pool', 'neo_astar', 'neo_astar_dev',
           'neo_T2tau_dev', 'neo_prepare_dev', 'neo_get_coeffs_dev', 'neo_sample_dev']

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
        lib.neo_get_map.argtypes = [V, I, I, I, V, V, V]
        lib.neo_set_map_points.argtypes = [V, I, I, V, D, D, I, I, D, D, D]
        lib.neo_get_occupancy.argtypes = [V, I, I, I, V]
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
        lib.neo_T2tau_dev.argtypes = [V, I, V, V, V, V]
        lib.neo_prepare_dev.argtypes = [V, I, I, V, V, V, V, V, I, V, V, V, V, V, V, V]
        lib.neo_get_coeffs_dev.argtypes = [V, I, I, V, V, V, V, V, V]
        lib.neo_sample_dev.argtypes = [V, I, I, V, V, D, I, V, V, V]
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
        """The (H, W) grid the slot's map was built from; raises NeoError if (H, W) is not the slot's shape or the map
        came from set_map_esdf."""
        occ = np.empty((H, W), np.int8)
        self._ck(self.lib.neo_get_occupancy(self.h, slot, H, W, ptr(occ)))
        return occ

    def get_map(self, slot, H, W):
        """(esdf, gx, gy) of the slot, each (H, W); raises NeoError if (H, W) is not the slot's shape."""
        e = np.empty((H, W)); gx = np.empty((H, W)); gy = np.empty((H, W))
        self._ck(self.lib.neo_get_map(self.h, slot, H, W, ptr(e), ptr(gx), ptr(gy)))
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

    # ---- device tensors ----------------------------------------------------------------------------------
    # The _dev methods take and return torch CUDA tensors on this handle's device, enqueue their work on the current
    # torch stream of that device and do not synchronise. They compute what the host methods above compute.
    def _stream(self):
        import torch
        s = torch.cuda.current_stream(self.device).cuda_stream
        # torch's default stream is the legacy default stream, handle 0, which the C API would read as "the handle's own
        # stream" (a non-blocking one, unordered with torch's work); cudaStreamLegacy (1) names it instead
        return C.c_void_p(s if s else 1)

    def _dev(self, name, t, dtype, shape, optional=False):
        """Device pointer of tensor t after checking its dtype, shape, contiguity and device (None stays None when
        optional)."""
        import torch
        if t is None and optional:
            return None
        if not torch.is_tensor(t):
            raise TypeError(f'{name}: expected a torch tensor, got {type(t).__name__}')
        if t.dtype != dtype:
            raise ValueError(f'{name}: expected dtype {dtype}, got {t.dtype}')
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f'{name}: expected shape {tuple(shape)}, got {tuple(t.shape)}')
        if t.device != torch.device('cuda', self.device):
            raise ValueError(f'{name}: expected a tensor on cuda:{self.device}, got {t.device}')
        if not t.is_contiguous():
            raise ValueError(f'{name}: tensor must be contiguous')
        return t.data_ptr()

    def _empty(self, shape, dtype=None, zero=False):
        import torch
        dtype = torch.float64 if dtype is None else dtype
        return (torch.zeros if zero else torch.empty)(shape, dtype=dtype, device=torch.device('cuda', self.device))

    def T2tau_dev(self, ts):
        """neo_T2tau_dev: T2tau of a float64 CUDA tensor (any shape) -> (tau, status int32), equal to T2tau's bits."""
        import torch
        p = self._dev('ts', ts, torch.float64, ts.shape)
        tau = self._empty(ts.shape); st = self._empty(ts.shape, torch.int32)
        self._ck(self.lib.neo_T2tau_dev(self.h, ts.numel(), p, tau.data_ptr(), st.data_ptr(), self._stream()))
        return tau, st

    def prepare_dev(self, M, head, tail, q0=None, ts0=None, init_ts=None, noise=None, map_ids=None):
        """neo_prepare_dev: the inputs of optimize_dev, built on the device as optimize() builds them on the host.
        head, tail (B,3,2); q0 (B,2,M-1) or None = straight line; ts0 (B,M) or None = init_ts, a HOST array (M);
        noise (B,count,M-1,2) or None; map_ids: HOST array-like (B) or None. Returns dict(x0 (B,n), x0_status (B),
        retry_q (B,count,2,M-1) or None, map_ids (B) int32 CUDA tensor or None)."""
        import torch
        B, n, K = len(head), 3 * M - 2, M - 1
        f = torch.float64
        ph = self._dev('head', head, f, (B, 3, 2)); pt = self._dev('tail', tail, f, (B, 3, 2))
        pq = self._dev('q0', q0, f, (B, 2, K), optional=True); pts = self._dev('ts0', ts0, f, (B, M), optional=True)
        count = 0 if noise is None else noise.shape[1] if noise.dim() == 4 else -1
        pn = self._dev('noise', noise, f, (B, count, K, 2), optional=True)
        its = None if init_ts is None else f64(init_ts, (M,))
        ids = None if map_ids is None else np.ascontiguousarray(map_ids, dtype=np.int32).reshape(-1)
        if ids is not None and ids.size != B:
            raise ValueError(f'map_ids: expected {B} ids, got {ids.size}')
        out = dict(x0=self._empty((B, n)), x0_status=self._empty(B, torch.int32),
                   retry_q=self._empty((B, count, 2, K)) if count > 0 else None,
                   map_ids=self._empty(B, torch.int32) if ids is not None else None)
        self._ck(self.lib.neo_prepare_dev(self.h, B, M, ph, pt, pq, pts, ptr(its), count, pn, ptr(ids),
                                          out['x0'].data_ptr(), out['x0_status'].data_ptr(),
                                          None if out['retry_q'] is None else out['retry_q'].data_ptr(),
                                          None if ids is None else out['map_ids'].data_ptr(), self._stream()))
        return out

    def alloc_result_dev(self, B, M, work=True):
        """alloc_result's fields as CUDA tensors on this handle's device."""
        import torch
        n, i32 = 3 * M - 2, torch.int32
        out = dict(x=self._empty((B, n), zero=True), ts=self._empty((B, M), zero=True),
                   coeffs=self._empty((B, 6 * M, 2), zero=True), costs=self._empty((B, 4), zero=True))
        for k in ('status', 'ok', 'attempt', 'nit', 'runs', 'nfev'):
            out[k] = self._empty(B, i32, zero=True)
        out['work'] = self._empty((B, 4), torch.int64, zero=True) if work else None
        return out

    def optimize_dev(self, M, x0, head, tail, x0_status=None, map_ids=None, retry_q=None, retry_tau=None, retry_status=0,
                     max_attempts=1, out=None):
        """neo_optimize_dev on CUDA tensors: x0 (B,n) in tau form, x0_status (B) int32 or None, head/tail (B,3,2),
        map_ids (B) int32 CUDA tensor or None (a precondition: every id names a slot holding a map -- prepare_dev checks
        them), retry_q (B,A-1,2,M-1), retry_tau (M) and the host int retry_status when max_attempts > 1. Returns the
        result dict of alloc_result_dev (or `out`)."""
        import torch
        B, n, f, i32 = x0.shape[0], 3 * M - 2, torch.float64, torch.int32
        args = [self._dev('x0', x0, f, (B, n)), self._dev('x0_status', x0_status, i32, (B,), True),
                self._dev('head', head, f, (B, 3, 2)), self._dev('tail', tail, f, (B, 3, 2)),
                self._dev('map_ids', map_ids, i32, (B,), True),
                self._dev('retry_q', retry_q, f, (B, max_attempts - 1, 2, M - 1), True),
                self._dev('retry_tau', retry_tau, f, (M,), True)]
        out = self.alloc_result_dev(B, M) if out is None else out
        r = Result()
        shapes = dict(x=(B, n), ts=(B, M), coeffs=(B, 6 * M, 2), costs=(B, 4), work=(B, 4))
        for k, _ in Result._fields_:
            dt = f if k in ('x', 'ts', 'coeffs', 'costs') else torch.int64 if k == 'work' else i32
            setattr(r, k, self._dev(k, out.get(k), dt, shapes.get(k, (B,)), optional=k == 'work'))
        self._ck(self.lib.neo_optimize_dev(self.h, B, M, *args, int(retry_status), int(max_attempts), C.byref(r),
                                           self._stream()))
        return out

    def get_coeffs_dev(self, M, q, ts, head, tail):
        """neo_get_coeffs_dev: q (B,2,M-1), ts (B,M), head/tail (B,3,2) CUDA tensors -> coeffs (B,6M,2)."""
        import torch
        B, f = q.shape[0], torch.float64
        out = self._empty((B, 6 * M, 2))
        self._ck(self.lib.neo_get_coeffs_dev(self.h, B, M, self._dev('q', q, f, (B, 2, M - 1)), self._dev('ts', ts, f, (B, M)),
                                             self._dev('head', head, f, (B, 3, 2)), self._dev('tail', tail, f, (B, 3, 2)),
                                             out.data_ptr(), self._stream()))
        return out

    def sample_dev(self, M, coeffs, ts, hz, max_samples):
        """neo_sample_dev: states (B, max_samples, 3, 2) (zero past each count) and count (B) int32, the full sample
        count even where it exceeds max_samples (those trajectories are cut at max_samples rows)."""
        import torch
        B, f = coeffs.shape[0], torch.float64
        states = self._empty((B, max_samples, 3, 2), zero=True); count = self._empty(B, torch.int32)
        self._ck(self.lib.neo_sample_dev(self.h, B, M, self._dev('coeffs', coeffs, f, (B, 6 * M, 2)),
                                         self._dev('ts', ts, f, (B, M)), float(hz), int(max_samples), states.data_ptr(),
                                         count.data_ptr(), self._stream()))
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
