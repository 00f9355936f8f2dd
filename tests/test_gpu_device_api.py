"""The device-resident planning API: neo_T2tau_dev, neo_prepare_dev, neo_get_coeffs_dev, neo_sample_dev, the torch
methods of lib.Handle and BatchPlanner built on them, and NeoBatchPlanner.enhanced_traj_plan_dev. Each result is
compared bit for bit with the host path on the same inputs and retry noise (drawn by np.random.default_rng and handed
to both), every call is checked not to wait for the GPU, and argument errors are checked to launch nothing."""

import numpy as np
import pytest

import bench
from neo_planner_b200 import frames, guesses, lib
from neo_planner_b200.planner import BatchPlanner
from neo_planner_b200.worlds import LibraryDefaultConfig, YamlConfig, make_problems, make_world

pytestmark = pytest.mark.gpu

FIELDS = ['x', 'ts', 'coeffs', 'costs', 'status', 'ok', 'attempt', 'nit', 'runs', 'nfev', 'work']


@pytest.fixture(scope='module')
def gpu():
    """torch on cuda:0 with a non-default current stream (the _dev calls must enqueue on it)."""
    import torch
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(device=dev)
    prev = torch.cuda.current_stream(dev)
    torch.cuda.set_stream(stream)
    yield dict(torch=torch, dev=dev, stream=stream)
    torch.cuda.synchronize()
    torch.cuda.set_stream(prev)


def same_bits(a, b):
    """a (NumPy) and b (NumPy or torch) hold the same bits in the same shape."""
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b.cpu().numpy() if hasattr(b, 'cpu') else b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def assert_results_equal(host, dev, what):
    for k in FIELDS:
        h, d = host[k], dev[k]
        if k == 'work':                        # the fourth column is nanoseconds on the SM
            h, d = h[:, :3], d[:, :3].contiguous()
        assert same_bits(h, d), (what, k)


def T_values(T_min, T_max, rng):
    k = np.arange(0, int(round(T_max * 10)) * 2 + 2, dtype=np.float64)
    return np.concatenate([rng.uniform(T_min - 1.0, T_max + 1.0, 1_000_000), k * 0.1, 1.5 * (k * 0.1),
                           [T_min, T_max, np.nextafter(T_min, np.inf), np.nextafter(T_max, -np.inf), np.nan, np.inf,
                            -np.inf, 0.0, -0.0]])


@pytest.mark.parametrize('cfg', [YamlConfig(), LibraryDefaultConfig()], ids=['yaml', 'library'])
def test_T2tau_dev_equals_host(gpu, cfg):
    torch = gpu['torch']
    h = lib.Handle(cfg, 0, 1)
    ts = T_values(cfg.T_min, cfg.T_max, np.random.default_rng(5))
    tau, st = h.T2tau(ts)
    tau_d, st_d = h.T2tau_dev(torch.from_numpy(ts).to(gpu['dev']))
    torch.cuda.synchronize()
    assert (st == lib.ST_DOMAIN).sum() > 100_000 and (st == 0).sum() > 600_000
    assert same_bits(tau, tau_d) and same_bits(st, st_d)


def line_host(head, tail, M):
    return np.transpose(guesses._line(head[:, 0, :], tail[:, 0, :], M - 1), (0, 2, 1))


def test_prepare_dev_equals_host_staging(gpu):
    torch, dev = gpu['torch'], gpu['dev']
    cfg = YamlConfig()
    w = make_world(3)
    B, M = 4096, 4
    h = lib.Handle(cfg, 0, 2)
    for slot in (0, 1):
        h.set_map_occupancy(slot, w.H, w.W, w.res, w.ox, w.oy, w.occ)
    head, tail = make_problems(w, B, M=M)
    tail[::7, 0, 0] = head[::7, 0, 0]                      # start == target in x: numpy's degenerate linspace branch
    tail[::11, 0, 1] = head[::11, 0, 1]
    rng = np.random.default_rng(9)
    q0 = rng.normal(size=(B, 2, M - 1)) * 10.0
    ts0 = rng.uniform(0.3, 5.5, size=(B, M))
    ts0[::13, 1] = np.nan
    ts0[::17, 2] = cfg.T_min
    noise = rng.normal(0, 0.5, (B, 3, M - 1, 2))
    ids = np.ones(B, np.int32)
    init = guesses.init_ts(cfg, M)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)                       # noqa: E731
    hd, tl = T(lib.pad_state(head)), T(lib.pad_state(tail))
    line = line_host(head, tail, M)
    assert same_bits(line, guesses.straight_line_guess(cfg, head, tail, M)[0])
    retry_host = np.ascontiguousarray(np.transpose(np.transpose(line, (0, 2, 1))[:, None] + noise, (0, 1, 3, 2)))

    def host_x0(q, ts):
        tau, st = h.T2tau(ts)
        status = np.array([next((s for s in row[::-1] if s), 0) for row in st], np.int32)
        return np.concatenate([q.reshape(B, -1), tau], axis=1), status

    for q, ts in [(q0, ts0), (None, ts0), (q0, None), (None, None)]:
        out = h.prepare_dev(M, hd, tl, None if q is None else T(q), None if ts is None else T(ts), init, T(noise), ids)
        x0, st = host_x0(line if q is None else q, np.tile(init, (B, 1)) if ts is None else ts)
        torch.cuda.synchronize()
        assert same_bits(x0, out['x0']) and same_bits(st, out['x0_status']), (q is None, ts is None)
        assert same_bits(retry_host, out['retry_q']) and same_bits(ids, out['map_ids'])
    assert (host_x0(q0, ts0)[1] == lib.ST_DOMAIN).sum() > 400
    # retry_q matches the host's own retry guesses when both draw the same noise
    rq, _ = guesses.retry_guesses(cfg, head, tail, M, 3, rng=np.random.default_rng(9))
    out = h.prepare_dev(M, hd, tl, None, None, init, T(np.random.default_rng(9).normal(0, 0.5, (B, 3, M - 1, 2))), None)
    assert same_bits(rq, out['retry_q']) and out['map_ids'] is None


@pytest.fixture(scope='module')
def planners():
    """BatchPlanner per benchmark workload, its maps uploaded."""
    cache = {}

    def get(name):
        if name not in cache:
            wl = bench.workload(name, 0, 1)
            bp = BatchPlanner(wl['cfg'], 0, len(wl['worlds']))
            ws = wl['worlds']
            bp.handle.set_maps_occupancy(np.arange(len(ws)), ws[0].H, ws[0].W, ws[0].res, [x.ox for x in ws],
                                         [x.oy for x in ws], np.stack([np.asarray(x.occ).reshape(x.H, x.W) for x in ws]))
            cache[name] = (wl, bp)
        return cache[name]
    yield get
    cache.clear()


@pytest.mark.parametrize('name', ['c2', 'c4', 'c5'])
def test_plan_dev_equals_plan(gpu, planners, name):
    """c2: 1,024 problems, M = 3; c4: 65,536 problems over 256 worlds (8-lane grouped kernel); c5: 16,384 problems,
    M = 10 on a 1200 x 1200 map."""
    torch, dev = gpu['torch'], gpu['dev']
    wl, bp = planners(name)
    B, M, ids = wl['B'], wl['M'], wl['map_ids']
    host = bp.plan(wl['head'], wl['tail'], ids, rng=np.random.default_rng(11), M=M)
    noise = torch.from_numpy(np.random.default_rng(11).normal(0, 0.5, (B, 4, M - 1, 2))).to(dev)
    res = bp.plan_dev(torch.from_numpy(wl['head']).to(dev), torch.from_numpy(wl['tail']).to(dev), ids, noise=noise, M=M)
    torch.cuda.synchronize()
    assert_results_equal(host, res, name)


def test_plan_dev_on_torch_default_stream(gpu, planners):
    """On torch's default stream (the legacy default stream, handle 0) the work is ordered with torch's own."""
    torch, dev = gpu['torch'], gpu['dev']
    wl, bp = planners('c2')
    B, M = wl['B'], wl['M']
    host = bp.plan(wl['head'], wl['tail'], None, rng=np.random.default_rng(22), M=M)
    with torch.cuda.stream(torch.cuda.default_stream(dev)):
        assert torch.cuda.current_stream(dev).cuda_stream == 0
        noise = torch.from_numpy(np.random.default_rng(22).normal(0, 0.5, (B, 4, M - 1, 2))).to(dev)
        res = bp.plan_dev(wl['head'], wl['tail'], None, noise=noise, M=M)
        got = {k: v.cpu() for k, v in res.items()}           # ordered on the default stream, no explicit synchronise
    assert_results_equal(host, got, 'default stream')


def test_warm_start_plan_dev_equals_host(gpu, planners):
    """warm-start guesses with noisy waypoints, durations out of range and NaN durations (attempt 0 then fails in
    map_T2tau on both paths and the retries start from the straight line)."""
    torch, dev = gpu['torch'], gpu['dev']
    wl, bp = planners('c2')
    B, M = wl['B'], wl['M']
    rng = np.random.default_rng(12)
    q = wl['q0'] + rng.normal(0, 0.3, wl['q0'].shape)
    ts = wl['ts0'] * rng.uniform(0.5, 1.5, wl['ts0'].shape)
    ts[::9, 0] = 7.0
    ts[::10, 2] = np.nan
    host = bp.warm_start_plan(wl['head'], wl['tail'], q, ts, None, rng=np.random.default_rng(13))
    noise = torch.from_numpy(np.random.default_rng(13).normal(0, 0.5, (B, 4, M - 1, 2))).to(dev)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)                       # noqa: E731
    res = bp.warm_start_plan_dev(T(wl['head']), T(wl['tail']), T(q), T(ts), None, noise=noise)
    torch.cuda.synchronize()
    assert (host['attempt'] > 0).sum() >= B // 10
    assert_results_equal(host, res, 'warm start')
    # get_coeffs_dev of the final waypoints and durations gives the optimizer's coefficients
    nq = 2 * (M - 1)
    c = bp.get_coeffs_dev(res['x'][:, :nq].reshape(B, 2, M - 1).contiguous(), res['ts'], T(wl['head']), T(wl['tail']))
    hc = bp.handle.get_coeffs(M, host['x'][:, :nq].reshape(B, 2, M - 1), host['ts'], wl['head'], wl['tail'])
    torch.cuda.synchronize()
    assert same_bits(hc, c)


def test_get_full_state_cmd_dev(gpu, planners):
    """past the 65,535-row grid height, and with max_samples below the counts"""
    torch, dev = gpu['torch'], gpu['dev']
    wl, bp = planners('c2')
    res = bp.plan(wl['head'], wl['tail'], None, rng=np.random.default_rng(14))
    reps = 70_000 // wl['B'] + 1
    coeffs, ts = np.tile(res['coeffs'], (reps, 1, 1)), np.tile(res['ts'], (reps, 1))
    ts[::5] *= 1.0 + 1e-3 * np.random.default_rng(15).uniform(size=ts[::5].shape)
    cd, tsd = torch.from_numpy(coeffs).to(dev), torch.from_numpy(ts).to(dev)
    for hz in (7, 60):
        B = coeffs.shape[0] if hz == 7 else 2_000
        states, count = bp.get_full_state_cmd(coeffs[:B], ts[:B], hz)
        sd, cnt = bp.get_full_state_cmd_dev(cd[:B], tsd[:B], hz)
        torch.cuda.synchronize()
        assert sd.shape[1] == int(np.ceil(wl['M'] * wl['cfg'].T_max * hz)) + 1 >= count.max()
        assert same_bits(count, cnt)
        assert same_bits(states, sd[:, :states.shape[1]]) and not sd[:, states.shape[1]:].any()
    # max_samples below the counts: full counts, rows cut at max_samples
    B, cut = coeffs.shape[0], 8                            # every trajectory lasts >= 3 T_min = 1.5 s: >= 11 samples
    states, count = bp.get_full_state_cmd(coeffs, ts, 7)
    assert (count > cut).all()
    sd, cnt = bp.get_full_state_cmd_dev(cd, tsd, 7, max_samples=cut)
    torch.cuda.synchronize()
    assert sd.shape == (B, cut, 3, 2) and same_bits(count, cnt) and same_bits(states[:, :cut], sd)


def scene(B, seed=0):
    rng = np.random.default_rng(seed)
    w = make_world(7)
    head, tail = make_problems(w, B)
    yaw = np.arctan2(head[:, 1, 1], head[:, 1, 0]) + rng.normal(0, 0.1, B)
    att = np.stack([np.cos(yaw / 2), rng.normal(0, 0.05, B), rng.normal(0, 0.05, B), np.sin(yaw / 2)], axis=1)
    gp = np.concatenate([head[:, 0] - 0.5 * head[:, 1], np.full((B, 1), 2.0)], axis=1)
    gv = np.concatenate([head[:, 1], np.zeros((B, 1))], axis=1)
    lv = frames.rotate_inverse(att, gv)
    depth = rng.integers(1, 256, size=(B, 480, 640), dtype=np.uint8)
    init_pos = np.concatenate([head[:, 0], np.full((B, 1), 2.0)], axis=1)
    return w, tail, att, gp, gv, lv, depth, init_pos


def test_wpts_world_dev_bits(gpu):
    torch, dev = gpu['torch'], gpu['dev']
    rng = np.random.default_rng(16)
    B = 200_000
    att, pos = rng.normal(size=(B, 4)), rng.normal(size=(B, 3)) * 30.0
    net = np.concatenate([rng.normal(size=(B, 6)) * 5.0, rng.uniform(-1.0, 25.0, size=(B, 3))], axis=1)
    q, ts = frames.wpts_world(att, pos, net, M=3)
    T = lambda a: torch.from_numpy(a).to(dev)                                             # noqa: E731
    qd, tsd = frames.wpts_world_dev(T(att), T(pos), T(net), M=3)
    assert same_bits(q, qd) and same_bits(ts, tsd)


@pytest.mark.parametrize('clamp_ts', [False, True])
def test_enhanced_traj_plan_dev_equals_host(gpu, clamp_ts):
    torch, dev = gpu['torch'], gpu['dev']
    from neo_planner_b200.initializer import NeoBatchPlanner
    B = 256
    w, tail, att, gp, gv, lv, depth, init_pos = scene(B, seed=17)
    bp = BatchPlanner(YamlConfig())
    bp.set_map(w)
    neo = NeoBatchPlanner(bp, des_pos_z=2.0, device='cuda', clamp_ts=clamp_ts)
    host = neo.enhanced_traj_plan(depth, lv, att, gp, gv, init_pos, gv, tail, rng=np.random.default_rng(18))
    noise = torch.from_numpy(np.random.default_rng(18).normal(0, 0.5, (B, 4, 2, 2))).to(dev)
    res = neo.enhanced_traj_plan_dev(torch.from_numpy(depth).to(dev), lv, att, gp, gv, init_pos, gv, tail, noise=noise)
    torch.cuda.synchronize()
    assert host['nn_ts_outside_bounds'].any()
    assert_results_equal(host, res, f'clamp_ts={clamp_ts}')
    for k in ('nn_int_wpts', 'nn_ts', 'nn_ts_outside_bounds'):
        assert same_bits(host[k], res[k]), k


def test_dev_calls_do_not_wait(gpu, planners):
    """Queued behind a long kernel on a non-default stream, every _dev call returns while the stream is still busy;
    after a synchronise the results equal those of the same calls made on an idle stream."""
    torch, dev, stream = gpu['torch'], gpu['dev'], gpu['stream']
    from neo_planner_b200.initializer import NeoBatchPlanner
    wl, bp = planners('c2')
    B, M = wl['B'], wl['M']
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)                       # noqa: E731
    head, tail, noise = T(wl['head']), T(wl['tail']), T(np.random.default_rng(19).normal(0, 0.5, (B, 4, M - 1, 2)))
    head3, tail3_d, ts0, q0 = T(lib.pad_state(wl['head'])), T(lib.pad_state(wl['tail'])), T(wl['ts0']), T(wl['q0'])
    w, tail3, att, gp, gv, lv, depth, init_pos = scene(64, seed=20)
    bp3 = BatchPlanner(YamlConfig())
    bp3.set_map(w)
    neo = NeoBatchPlanner(bp3, des_pos_z=2.0, device='cuda')
    noise3 = T(np.random.default_rng(21).normal(0, 0.5, (64, 4, 2, 2)))
    depth_d = T(depth)

    def calls(check):
        out = {}
        out['tau'] = bp.handle.T2tau_dev(ts0)[0]; check('T2tau_dev')
        out['prep'] = bp.handle.prepare_dev(M, head3, tail3_d, None, None, guesses.init_ts(wl['cfg'], M), noise,
                                            np.zeros(B, np.int32))['x0']
        check('prepare_dev')
        out['plan'] = bp.plan_dev(head, tail, None, noise=noise, M=M); check('plan_dev')
        out['warm'] = bp.warm_start_plan_dev(head, tail, q0, ts0, None, noise=noise); check('warm_start_plan_dev')
        nq = 2 * (M - 1)
        out['coeffs'] = bp.get_coeffs_dev(out['plan']['x'][:, :nq].reshape(B, 2, M - 1).contiguous(), out['plan']['ts'],
                                          head, tail)
        check('get_coeffs_dev')
        out['states'] = bp.get_full_state_cmd_dev(out['plan']['coeffs'], out['plan']['ts'], 60); check('get_full_state_cmd_dev')
        out['neo'] = neo.enhanced_traj_plan_dev(depth_d, lv, att, gp, gv, init_pos, gv, tail3, noise=noise3)
        check('enhanced_traj_plan_dev')
        return out

    ref = calls(lambda what: None)                 # warm-up on an idle stream: buffers grown, cuDNN algorithms chosen
    torch.cuda.synchronize()
    assert torch.cuda.current_stream(dev) == stream and stream != torch.cuda.default_stream(dev)
    torch.cuda._sleep(4_000_000_000)

    def busy(what):
        assert not stream.query(), f'{what} waited for the stream'
    got = calls(busy)
    torch.cuda.synchronize()

    def flat(o):
        if isinstance(o, dict):
            return [v for k in sorted(o) for v in flat(o[k])]
        if isinstance(o, (tuple, list)):
            return [v for x in o for v in flat(x)]
        return [] if o is None else [o]
    for a, b in zip(flat(ref), flat(got), strict=True):
        if a.dtype == torch.int64:                 # work: nanoseconds column
            a, b = a[..., :3], b[..., :3]
        assert torch.equal(a, b)


def test_argument_errors_launch_nothing(gpu, planners):
    torch, dev = gpu['torch'], gpu['dev']
    wl, bp = planners('c2')
    h = bp.handle
    L, B, M = h.lib, 8, 3
    buf = [torch.zeros(1 << 14, dtype=torch.float64, device=dev) for _ in range(8)]
    p = [b.data_ptr() for b in buf]
    ids_ok = np.zeros(B, np.int32)
    ids_bad = ids_ok.copy()
    ids_bad[5] = 1                               # the c2 handle holds one map (slot 0)
    init = np.full(M, 2.5)
    INVALID = -1

    def prepare(**kw):
        a = dict(B=B, M=M, head=p[0], tail=p[1], q0=None, ts0=None, init_ts=lib.ptr(init), count=2, noise=p[2],
                 ids=lib.ptr(ids_ok), x0=p[3], x0_status=p[4], retry_q=p[5], ids_dev=p[6])
        a.update(kw)
        return L.neo_prepare_dev(h.h, a['B'], a['M'], a['head'], a['tail'], a['q0'], a['ts0'], a['init_ts'], a['count'],
                                 a['noise'], a['ids'], a['x0'], a['x0_status'], a['retry_q'], a['ids_dev'], None)

    bad_calls = {
        'T2tau_dev n < 0': lambda: L.neo_T2tau_dev(h.h, -1, p[0], p[1], p[2], None),
        'T2tau_dev ts NULL': lambda: L.neo_T2tau_dev(h.h, 4, None, p[1], p[2], None),
        'T2tau_dev tau NULL': lambda: L.neo_T2tau_dev(h.h, 4, p[0], None, p[2], None),
        'prepare_dev M = 1': lambda: prepare(M=1),
        'prepare_dev M = 11': lambda: prepare(M=11),
        'prepare_dev B < 0': lambda: prepare(B=-1),
        'prepare_dev count = 8': lambda: prepare(count=8),
        'prepare_dev head NULL': lambda: prepare(head=None),
        'prepare_dev tail NULL': lambda: prepare(tail=None),
        'prepare_dev x0 NULL': lambda: prepare(x0=None),
        'prepare_dev x0_status NULL': lambda: prepare(x0_status=None),
        'prepare_dev no ts0, no init_ts': lambda: prepare(init_ts=None),
        'prepare_dev noise NULL': lambda: prepare(noise=None),
        'prepare_dev retry_q NULL': lambda: prepare(retry_q=None),
        'prepare_dev map_ids_dev NULL': lambda: prepare(ids_dev=None),
        'prepare_dev bad host map id': lambda: prepare(ids=lib.ptr(ids_bad)),
        'get_coeffs_dev M = 1': lambda: L.neo_get_coeffs_dev(h.h, B, 1, p[0], p[1], p[2], p[3], p[4], None),
        'get_coeffs_dev M = 11': lambda: L.neo_get_coeffs_dev(h.h, B, 11, p[0], p[1], p[2], p[3], p[4], None),
        'get_coeffs_dev q NULL': lambda: L.neo_get_coeffs_dev(h.h, B, M, None, p[1], p[2], p[3], p[4], None),
        'get_coeffs_dev coeffs NULL': lambda: L.neo_get_coeffs_dev(h.h, B, M, p[0], p[1], p[2], p[3], None, None),
        'sample_dev M = 0': lambda: L.neo_sample_dev(h.h, B, 0, p[0], p[1], 10.0, 8, p[2], p[3], None),
        'sample_dev hz = 0': lambda: L.neo_sample_dev(h.h, B, M, p[0], p[1], 0.0, 8, p[2], p[3], None),
        'sample_dev count NULL': lambda: L.neo_sample_dev(h.h, B, M, p[0], p[1], 10.0, 8, p[2], None, None),
        'sample_dev coeffs NULL': lambda: L.neo_sample_dev(h.h, B, M, None, p[1], 10.0, 8, p[2], p[3], None),
        'sample_dev max_samples 0': lambda: L.neo_sample_dev(h.h, B, M, p[0], p[1], 10.0, 0, p[2], p[3], None),
    }
    for what, call in bad_calls.items():
        before = h.launch_count()
        assert call() == INVALID, what
        assert h.launch_count() == before, what
    assert prepare() == 0 and L.neo_T2tau_dev(h.h, 4, p[0], p[1], None, None) == 0
    torch.cuda.synchronize()
    # the torch layer checks dtype, shape, contiguity and device before calling the library
    ts = torch.full((4, M), 2.5, dtype=torch.float64, device=dev)
    for bad in (ts.float(), ts.cpu(), ts.t().contiguous().t(), ts[:, :2]):
        with pytest.raises((TypeError, ValueError)):
            h.get_coeffs_dev(M, torch.zeros(4, 2, M - 1, dtype=torch.float64, device=dev), bad,
                             torch.zeros(4, 3, 2, dtype=torch.float64, device=dev),
                             torch.zeros(4, 3, 2, dtype=torch.float64, device=dev))
    with pytest.raises(lib.NeoError):
        bp.plan_dev(torch.from_numpy(wl['head'][:B]).to(dev), torch.from_numpy(wl['tail'][:B]).to(dev), ids_bad,
                    noise=torch.zeros(B, 4, M - 1, 2, dtype=torch.float64, device=dev))
