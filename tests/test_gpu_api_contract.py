"""The argument contract of the C ABI (include/neoopt.h), called through ctypes. Every host-pointer entry point and its
device-pointer twin reject malformed arguments with NEO_ERR_INVALID before they launch anything, B = 0 returns NEO_OK
without a launch, and a rejected call leaves the handle working: a small neo_eval afterwards returns what it returned
before."""
import numpy as np
import pytest

from neo_planner_b200 import lib
from neo_planner_b200.guesses import straight_line_guess
from neo_planner_b200.worlds import YamlConfig, make_problems, make_world

pytestmark = pytest.mark.gpu

OK, INVALID = 0, -1
B, M = 4, 3
LEN = 1 << 12          # elements of every argument array: enough for B problems of M pieces, one attempt, trace_cap 1


class Ctx:
    """A handle with a map in slot 0 (slot 1 stays empty), argument arrays on the host and on the device, and the
    result of a small neo_eval to compare with after each rejected call."""

    def __init__(self):
        import torch
        self.torch = torch
        cfg = YamlConfig()
        w = make_world(0)
        self.h = lib.Handle(cfg, 0, 2)
        self.h.set_map_occupancy(0, w.H, w.W, w.res, w.ox, w.oy, w.occ)
        self.lib = self.h.lib
        self.keep = []
        head, tail = make_problems(w, B, M=M)
        q0, ts0 = straight_line_guess(cfg, head, tail, M)
        tau, _ = self.h.T2tau(ts0)
        self.ref_args = (M, np.concatenate([q0.reshape(B, -1), tau], axis=1), head, tail)
        self.ref = self.h.eval(*self.ref_args)

    def host(self, dtype=np.float64, values=None):
        a = np.zeros(LEN, dtype)
        if values is not None:
            a[:len(values)] = values
        self.keep.append(a)
        return a.ctypes.data

    def dev(self, dtype=np.float64):
        t = self.torch.zeros(LEN * np.dtype(dtype).itemsize, dtype=self.torch.uint8, device='cuda')
        self.keep.append(t)
        return t.data_ptr()

    def result(self, alloc):
        r = lib.Result()
        for k, _ in lib.Result._fields_:
            setattr(r, k, alloc(np.int64 if k == 'work' else np.float64 if k in ('x', 'ts', 'coeffs', 'costs') else np.int32))
        return r

    def launches(self):
        return self.h.launch_count()

    def eval_unchanged(self):
        now = self.h.eval(*self.ref_args)
        for k in ('costs', 'grad', 'status'):
            assert np.array_equal(now[k], self.ref[k]), k


@pytest.fixture(scope='module')
def ctx():
    return Ctx()


# Valid arguments of each entry point (B problems of M pieces, map_ids NULL, one attempt), with the positions of its
# arguments: 'required' pointers, 'm_bad' piece counts out of range, and where they exist the result struct, max_attempts,
# the two retry arrays, map_ids and trace_cap.
def _eval(c, dev):
    a = c.dev if dev else c.host
    args = [c.h.h, B, M, a(), a(), a(), None, a(), a(), a(np.int32), None, None]
    return args + [None] if dev else args


def _optimize(c, trace):
    a = c.host
    args = [c.h.h, B, M, a(), a(), a(), a(), None, None, None, 1, c.result(a)]
    return args + [1, a(), a(), a(), a(), a(np.int32), a(np.int32)] if trace else args


def _optimize_dev(c):
    a = c.dev
    return [c.h.h, B, M, a(), None, a(), a(), None, None, None, 0, 1, c.result(a), None]


def _astar(c, dev):
    a = c.dev if dev else c.host
    args = [c.h.h, B, a(), a(), None, 0, 0, None, a(np.int32), a(), a(np.int32), a(np.int32)]
    return args + [None] if dev else args


ENTRIES = {
    'neo_eval': dict(build=lambda c: _eval(c, False), required=[3, 4, 5, 7, 8, 9], m_bad=[1, 11], map_ids=6),
    'neo_eval_dev': dict(build=lambda c: _eval(c, True), required=[3, 4, 5, 7, 8, 9], m_bad=[1, 11]),
    'neo_optimize': dict(build=lambda c: _optimize(c, False), required=[3, 4, 5, 6], m_bad=[1, 11], out=11, attempts=10,
                         retry=(8, 9), map_ids=7),
    'neo_optimize_trace': dict(build=lambda c: _optimize(c, True), required=[3, 4, 5, 6, 13, 14, 15, 16, 17, 18],
                               m_bad=[1, 11], out=11, attempts=10, retry=(8, 9), map_ids=7, cap=12),
    'neo_optimize_dev': dict(build=_optimize_dev, required=[3, 5, 6], m_bad=[1, 11], out=12, attempts=11, retry=(8, 9)),
    'neo_get_coeffs': dict(build=lambda c: [c.h.h, B, M, c.host(), c.host(), c.host(), c.host(), c.host()],
                           required=[3, 4, 5, 6, 7], m_bad=[1, 11]),
    'neo_sample': dict(build=lambda c: [c.h.h, B, M, c.host(), c.host(), 10.0, 0, None, c.host(np.int32)],
                       required=[3, 4, 8], m_bad=[0, 65]),
    'neo_astar': dict(build=lambda c: _astar(c, False), required=[2, 3, 8, 9, 10, 11], map_ids=4),
    'neo_astar_dev': dict(build=lambda c: _astar(c, True), required=[2, 3, 8, 9, 10, 11]),
}


def _set(i, v):
    def f(c, args):
        args[i] = v(c) if callable(v) else v
    return f


def _null_field(i, field):
    def f(c, args):
        setattr(args[i], field, None)
    return f


def _cases():
    for name, e in ENTRIES.items():
        yield name, 'B<0', _set(1, -1)
        yield name, 'handle NULL', _set(0, None)
        for m in e.get('m_bad', []):
            yield name, f'M={m}', _set(2, m)
        for i in e['required']:
            yield name, f'arg {i} NULL', _set(i, None)
        if 'out' in e:
            yield name, 'out NULL', _set(e['out'], None)
            for field, _ in lib.Result._fields_:
                if field != 'work':
                    yield name, f'out.{field} NULL', _null_field(e['out'], field)
        if 'attempts' in e:
            at, (rq, rt) = e['attempts'], e['retry']
            yield name, 'max_attempts=0', _set(at, 0)
            yield name, 'max_attempts=9', _set(at, 9)
            yield name, 'max_attempts=2 without retry arrays', _set(at, 2)
            for only in (rq, rt):
                def f(c, args, at=at, only=only, dev=name.endswith('_dev')):
                    args[at] = 2
                    args[only] = c.dev() if dev else c.host()
                yield name, f'max_attempts=2 with retry arg {only} only', f
        if 'map_ids' in e:
            for ids in ([0, 1, 0, 0], [0, 0, 2, 0], [-1, 0, 0, 0]):
                yield name, f'map_ids={ids}', _set(e['map_ids'], lambda c, ids=ids: c.host(np.int32, ids))
        if 'cap' in e:
            yield name, 'trace_cap=0', _set(e['cap'], 0)
    for nm in ('neo_astar', 'neo_astar_dev'):
        yield nm, 'max_closed<0', _set(5, -1)
        yield nm, 'max_path<0', _set(6, -1)
        yield nm, 'path without max_path', _set(7, lambda c, dev=nm.endswith('_dev'): c.dev() if dev else c.host())
    for v in (np.nan, np.inf):
        yield 'neo_astar', f'start {v}', _set(2, lambda c, v=v: c.host(values=[0.0, v]))
        yield 'neo_astar', f'target {v}', _set(3, lambda c, v=v: c.host(values=[0.0, 0.0, v]))
    yield 'neo_sample', 'hz=0', _set(5, 0.0)
    yield 'neo_sample', 'states with max_samples=0', _set(7, lambda c: c.host())


CASES = list(_cases())


@pytest.mark.parametrize('name,what,mutate', CASES, ids=[f'{n}-{w}' for n, w, _ in CASES])
def test_rejected_without_launch(ctx, name, what, mutate):
    ctx.keep.clear()
    args = ENTRIES[name]['build'](ctx)
    mutate(ctx, args)
    before = ctx.launches()
    assert getattr(ctx.lib, name)(*args) == INVALID
    assert ctx.launches() == before
    ctx.eval_unchanged()


@pytest.mark.parametrize('name', list(ENTRIES))
def test_empty_batch_is_a_no_op(ctx, name):
    ctx.keep.clear()
    args = ENTRIES[name]['build'](ctx)
    args[1] = 0
    before = ctx.launches()
    assert getattr(ctx.lib, name)(*args) == OK
    assert ctx.launches() == before
    ctx.eval_unchanged()


def test_sample_rejects_too_small_max_samples(ctx):
    # 4 trajectories of 3 one-second pieces sampled at 8 Hz need 24 samples each
    count = np.zeros(B, np.int32)
    states = np.zeros((B, 5, 3, 2))
    rc = ctx.lib.neo_sample(ctx.h.h, B, M, ctx.host(), ctx.host(values=np.ones(B * M)), 8.0, 5, lib.ptr(states),
                            lib.ptr(count))
    assert rc == INVALID and b'max_samples' in ctx.lib.neo_last_error(ctx.h.h)
    assert (count == 24).all()
    ctx.eval_unchanged()


def test_map_read_back_checks_the_shape(ctx):
    """neo_get_map / neo_get_occupancy write H x W elements into the caller's arrays: a shape other than the slot's is
    rejected before anything is copied, and after an ESDF upload the slot has no occupancy grid until the next
    occupancy build -- whether the new map is larger, smaller or of the same shape."""
    w = make_world(0)
    h = lib.Handle(YamlConfig(), 0, 1)
    h.set_map_occupancy(0, w.H, w.W, w.res, w.ox, w.oy, w.occ)
    occ_want = np.where(w.occ == 100, 100, 0).astype(np.int8)
    n = (w.H + 1) * (w.W + 1)                         # room for every shape tried below
    bufs = [np.full(n, 7.0) for _ in range(3)]
    obuf = np.full(n, 7, np.int8)

    def rejected(H, W, what):
        before = h.launch_count()
        assert h.lib.neo_get_map(h.h, 0, H, W, *map(lib.ptr, bufs)) == INVALID, ('get_map', H, W)
        assert what in h.lib.neo_last_error(h.h), h.lib.neo_last_error(h.h)
        assert h.lib.neo_get_occupancy(h.h, 0, H, W, lib.ptr(obuf)) == INVALID, ('get_occupancy', H, W)
        assert h.launch_count() == before
        assert all((b == 7.0).all() for b in bufs) and (obuf == 7).all()

    for H, W in ((w.H, w.W - 1), (w.H + 1, w.W), (150, 600), (0, 0), (-1, w.W)):
        rejected(H, W, b'300 x 300')
        if H >= 0:
            with pytest.raises(lib.NeoError):
                h.get_map(0, H, W)
            with pytest.raises(lib.NeoError):
                h.get_occupancy(0, H, W)
    assert np.array_equal(h.get_occupancy(0, w.H, w.W), occ_want)
    e, gx, gy = h.get_map(0, w.H, w.W)
    # ESDF uploads: smaller, then the same shape as the occupancy build, then larger
    for H, W in ((9, 11), (w.H, w.W), (w.H + 20, w.W + 7)):
        rng = np.random.default_rng(H)
        arrays = [rng.normal(size=(H, W)) for _ in range(3)]
        h.set_map_esdf(0, 0.1, 1.0, -2.0, *arrays)
        before = h.launch_count()
        for args in ((H, W), (w.H, w.W)):
            assert h.lib.neo_get_occupancy(h.h, 0, *args, lib.ptr(obuf)) == INVALID
            assert b'no occupancy' in h.lib.neo_last_error(h.h)
        assert h.launch_count() == before and (obuf == 7).all()
        with pytest.raises(lib.NeoError, match='no occupancy'):
            h.get_occupancy(0, H, W)
        back = h.get_map(0, H, W)
        assert all(np.array_equal(a, b) for a, b in zip(back, arrays))
        if (H, W) != (w.H, w.W):
            rejected(w.H, w.W, f'{H} x {W}'.encode())
    # the next occupancy build brings the grid back
    h.set_map_occupancy(0, w.H, w.W, w.res, w.ox, w.oy, w.occ)
    assert np.array_equal(h.get_occupancy(0, w.H, w.W), occ_want)
    assert all(np.array_equal(a, b) for a, b in zip(h.get_map(0, w.H, w.W), (e, gx, gy)))
    h.close()
    ctx.eval_unchanged()


def test_set_maps_occupancy_argument_checks(ctx):
    H = W = 8
    occ = np.zeros((2, H, W), np.int8)
    ox = np.zeros(2); oy = np.zeros(2)
    good = np.array([1, 0], np.int32)

    def call(K, slots, ox_=ox, oy_=oy, occ_=occ):
        before = ctx.launches()
        rc = ctx.lib.neo_set_maps_occupancy(ctx.h.h, K, lib.ptr(slots), H, W, 0.1, lib.ptr(ox_), lib.ptr(oy_), lib.ptr(occ_))
        return rc, ctx.launches() - before

    for bad in ((2, np.array([1, 1], np.int32)), (2, np.array([0, 2], np.int32)), (2, np.array([-1, 0], np.int32)),
                (-1, good), (2, None)):
        assert call(*bad) == (INVALID, 0), bad
        ctx.eval_unchanged()
    for kw in (dict(ox_=None), dict(oy_=None), dict(occ_=None)):
        assert call(2, good, **kw) == (INVALID, 0), kw
        ctx.eval_unchanged()
    assert call(0, good) == (OK, 0)
    ctx.eval_unchanged()
