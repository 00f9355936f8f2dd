"""What bench.py times, checked for what it computes: k_eval and k_coeffs / k_sample at batches that make every tile loop
over several problems, neo_optimize_dev launched back to back as the timed steps launch it, and the per-problem work
counters the roofline figures are computed from.

The launches run the benchmark's own inputs, buffers and launch sequence (bench.workload, bench.DeviceRun,
bench.timed_steps) on a non-default stream with the 256 MiB L2 flush between launches. Three kinds of evidence:
  * bit-for-bit equality between paths that run the same kernel: repeated launches, the host-pointer entry point
    against the device-pointer one, a problem inside a large batch against the same problem evaluated alone;
  * the CPU checker (oracle/minco_oracle.c) at the tolerances the other tests established -- cost and gradient within
    1e-6 relative, coefficients and sampled states within the 1e-10 of test_gpu_parity.py scaled by the coefficient
    magnitude, whole plans with test_gpu_fullsize.compare_with_checker's thresholds;
  * the work counters recomputed in NumPy from the recorded evaluations.

Batch sizes come from a bound, not from the occupancy the library happens to pick: an SM holds at most 64 warps, so at
most sm_count * 64 * (32 / TL) tiles of TL lanes are resident at once. B = 3 * bound + 5 problems make every tile run at
least three problems and leave a ragged tail.
"""
import ctypes as C
import os
import time

import numpy as np
import pytest

import bench
from neo_planner_b200 import lib, sharding
from neo_planner_b200.worlds import YamlConfig, make_world
from oracle import c_oracle
from test_gpu_fullsize import compare_with_checker

pytestmark = pytest.mark.gpu

RECORD_FIELDS = ('x', 'ts', 'coeffs', 'costs', 'status', 'ok', 'attempt', 'nit', 'runs', 'nfev')
N_MAPS = 16                   # maps of the perturbed batches (random map id per problem)
LAYOUTS = [(2, 8), (2, 32), (3, 8), (3, 32), (4, 16), (4, 32)] + [(M, 32) for M in range(5, 11)]


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def handle_with_tile(cfg, n_maps, tile):
    """A handle whose lanes per problem do not depend on the batch size (NEO_TILE is read at neo_create)."""
    old = os.environ.get('NEO_TILE')
    os.environ['NEO_TILE'] = str(tile)
    try:
        return lib.Handle(cfg, 0, n_maps)
    finally:
        if old is None:
            del os.environ['NEO_TILE']
        else:
            os.environ['NEO_TILE'] = old


# ---------------------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope='module', autouse=True)
def wall_time():
    t0 = time.perf_counter()
    yield
    print(f'\ntest_gpu_bench_paths: wall time {time.perf_counter() - t0:.1f} s')


@pytest.fixture(scope='module')
def gpu():
    """torch on cuda:0 with a non-default stream and the benchmark's L2 flush buffer, as bench.main sets them up."""
    import torch
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(device=dev)
    prev = torch.cuda.current_stream(dev)
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    yield dict(torch=torch, dev=dev, flush=flush, stream=stream)
    torch.cuda.synchronize()
    torch.cuda.set_stream(prev)


@pytest.fixture(scope='module')
def runs(gpu):
    """bench.DeviceRun per workload, built once: maps uploaded, inputs and result records in HBM."""
    cache = {}

    def get(name):
        if name not in cache:
            wl = bench.workload(name, 0, 1)
            cache[name] = bench.DeviceRun(wl, 0, gpu['dev'], gpu['torch'], lib, C)
        return cache[name]
    yield get
    cache.clear()


@pytest.fixture(scope='module')
def sm_count():
    h = lib.Handle(YamlConfig(), 0, 1)
    n = h.device_info()['sm_count']
    h.close()
    return n


def resident_bound(sm_count, TL):
    return sm_count * 64 * (32 // TL)


def batch_for(sm_count, TL):
    bound = resident_bound(sm_count, TL)
    B = 3 * bound + 5
    return B, bound, B // bound


@pytest.fixture(scope='module')
def worlds16():
    ws = [make_world(100 + k) for k in range(N_MAPS)]
    return ws, [c_oracle.OracleMap.from_world(w) for w in ws]


@pytest.fixture(scope='module')
def tiled_handles(worlds16):
    """One handle per forced lane count, each holding the N_MAPS maps."""
    cfg = YamlConfig()
    ws, _ = worlds16
    hs = {}
    for tile in (8, 16, 32):
        h = handle_with_tile(cfg, N_MAPS, tile)
        h.set_maps_occupancy(np.arange(N_MAPS), ws[0].H, ws[0].W, ws[0].res, [w.ox for w in ws], [w.oy for w in ws],
                             np.stack([np.asarray(w.occ).reshape(w.H, w.W) for w in ws]))
        hs[tile] = h
    yield hs
    for h in hs.values():
        h.close()


def perturbed_inputs(cfg, world, M, B, seed):
    """B random problems over N_MAPS maps of the shape of `world`, with interleaved problems that leave the evaluator
    early or diverge. Returns dict(x, head, tail, ids, kind) with kind: 0 plain, 1 tau = -720 (OverflowError), 2 NaN in
    q (int(nan)), 3 / 4 a duration within 1e-3 of T_min / T_max, 5 start and goal far outside the map."""
    rng = np.random.default_rng(seed)
    nq = 2 * (M - 1)
    span = np.array([world.W * world.res, world.H * world.res])
    org = np.array([world.ox, world.oy])
    head = np.zeros((B, 3, 2)); tail = np.zeros((B, 3, 2))
    head[:, 0] = org + rng.uniform(-0.1, 1.1, (B, 2)) * span            # some start outside the map
    ang = rng.uniform(0, 2 * np.pi, B)
    tail[:, 0] = head[:, 0] + (5.0 * M / 3.0) * np.stack([np.cos(ang), np.sin(ang)], axis=1)
    for s in (head, tail):
        s[:, 1] = rng.normal(0, 0.5, (B, 2)); s[:, 2] = rng.normal(0, 0.3, (B, 2))
    kind = np.zeros(B, np.int32)
    kind[1::37] = 1; kind[2::37] = 2; kind[3::37] = 3; kind[4::37] = 4; kind[5::37] = 5
    far = kind == 5
    head[far, 0] = org + np.array([-40.0, -40.0]); tail[far, 0] = org + np.array([-40.0, -40.0 + 5.0 * M / 3.0])
    lam = np.linspace(0, 1, M + 1)[1:-1]
    q = head[:, None, 0, :] + lam[None, :, None] * (tail[:, 0] - head[:, 0])[:, None, :] + rng.normal(0, 0.4, (B, M - 1, 2))
    q = np.transpose(q, (0, 2, 1)).reshape(B, nq)
    tau = rng.normal(0, 1.5, (B, M))
    piece = rng.integers(0, M, B)
    rows = np.arange(B)
    tau[kind == 1, piece[kind == 1]] = -720.0
    q[kind == 2, rng.integers(0, nq, B)[kind == 2]] = np.nan
    for k, T in ((3, cfg.T_min + 1e-3 * rng.uniform(0.01, 1.0, B)), (4, cfg.T_max - 1e-3 * rng.uniform(0.01, 1.0, B))):
        sel = kind == k
        a = (cfg.T_max - cfg.T_min) / (T[sel] - cfg.T_min) - 1.0
        tau[rows[sel], piece[sel]] = -np.log(a)
    ids = rng.integers(0, N_MAPS, B).astype(np.int32)
    return dict(x=np.concatenate([q, tau], axis=1), head=head, tail=tail, ids=ids, kind=kind)


def check_eval_against_checker(cfg, M, omaps, x, head, tail, ids, dev):
    """Device evaluation `dev` vs c_oracle.eval_batch map by map: equal status everywhere, cost
    and gradient within 1e-6 where the status is 0. Returns (worst cost error, worst gradient error, evaluations)."""
    p = c_oracle.Params.from_config(cfg)
    B = x.shape[0]
    ids = np.zeros(B, np.int32) if ids is None else ids
    costs = np.zeros((B, 4)); grad = np.zeros_like(x); status = np.zeros(B, np.int32)
    for s in np.unique(ids):
        sel = np.nonzero(ids == s)[0]
        costs[sel], grad[sel], status[sel] = c_oracle.eval_batch(p, omaps[s], M, head[sel], tail[sel], x[sel])
    bad = np.nonzero(dev['status'] != status)[0]
    assert bad.size == 0, ('status differs from the checker', bad[:10], dev['status'][bad[:10]], status[bad[:10]])
    ok = status == 0
    assert np.allclose(dev['costs'][ok], costs[ok], rtol=1e-6, atol=1e-9)
    cerr = np.max(np.abs(dev['costs'][ok] - costs[ok]) / np.maximum(np.abs(costs[ok]), 1e-3), axis=1)
    scale = np.maximum(np.max(np.abs(grad[ok]), axis=1), 1e-9)
    gerr = np.max(np.abs(dev['grad'][ok] - grad[ok]), axis=1) / scale
    assert (gerr <= 1e-6).all(), gerr.max()
    return float(cerr.max()), float(gerr.max()), int(ok.sum())


def dev_result(torch, dev, B, M):
    """A packed result record buffer (the layout of bench.DeviceRun / sharding.DeviceShard) and its neo_result."""
    out = torch.zeros(sharding.packed_record_bytes(B, M), dtype=torch.uint8, device=dev)
    work = torch.zeros(B * 4, dtype=torch.int64, device=dev)
    res = lib.Result()
    for k, o in sharding.packed_record_offsets(B, M).items():
        setattr(res, k, out.data_ptr() + o)
    res.work = work.data_ptr()
    return out, work, res


def records(out, work, B, M):
    f = sharding.split_packed_records(out.cpu().numpy().reshape(1, -1), B, M)
    f = {k: np.ascontiguousarray(v[0]) for k, v in f.items()}
    f['work'] = work.cpu().numpy().reshape(B, 4).copy()
    return f


def assert_same_records(a, b, what):
    for k in RECORD_FIELDS:
        assert same_bits(a[k], b[k]), (what, k)
    assert same_bits(a['work'][:, :3], b['work'][:, :3]), (what, 'work')


# ---------------------------------------------------------------------------------------------------------- A: k_eval
@pytest.mark.parametrize('name', ['c2', 'c4', 'c5'])
def test_eval_dev_on_bench_inputs(name, gpu, runs):
    """neo_eval_dev exactly as bench.eval_rate launches it (the expert guess of every problem, flush in between): two
    launches identical, equal to neo_eval, and within the established tolerances of the checker."""
    torch, flush = gpu['torch'], gpu['flush']
    run = runs(name)
    wl, h, M, B, n = run.wl, run.h, run.M, run.B, run.n
    st = torch.cuda.current_stream().cuda_stream
    assert st != 0
    outs = []
    for _ in range(2):
        costs = torch.zeros(B * 4, dtype=torch.float64, device=gpu['dev']); grad = torch.zeros(B * n, dtype=torch.float64, device=gpu['dev'])
        status = torch.zeros(B, dtype=torch.int32, device=gpu['dev'])
        flush.zero_()
        h._ck(h.lib.neo_eval_dev(h.h, B, M, run.x0.data_ptr(), run.head.data_ptr(), run.tail.data_ptr(),
                                 None if run.ids_d is None else run.ids_d.data_ptr(), costs.data_ptr(), grad.data_ptr(),
                                 status.data_ptr(), None, None, run.C.c_void_p(st)))
        outs.append((costs, grad, status))
    torch.cuda.synchronize()
    dev = [dict(costs=c.cpu().numpy().reshape(B, 4), grad=g.cpu().numpy().reshape(B, n), status=s.cpu().numpy()) for c, g, s in outs]
    for k in ('costs', 'grad', 'status'):
        assert same_bits(dev[0][k], dev[1][k]), k
    x = run.x0.cpu().numpy(); head = lib.pad_state(wl['head']); tail = lib.pad_state(wl['tail'])
    host = h.eval(M, x, head, tail, wl['map_ids'])
    for k in ('costs', 'grad', 'status'):
        assert same_bits(host[k], dev[0][k]), k
    assert (dev[0]['status'] == 0).all()
    omaps = [c_oracle.OracleMap.from_world(w) for w in wl['worlds']]
    ce, ge, cnt = check_eval_against_checker(wl['cfg'], M, omaps, x, head, tail, wl['map_ids'], dev[0])
    tl = 32 if M > 4 or B < 12288 else (8 if M <= 3 else 16)
    print(f'\n[A] {name}: B={B}, M={M}, {len(omaps)} map(s), {tl} lanes per problem: two neo_eval_dev launches and neo_eval '
          f'identical; vs checker on {cnt} evaluations: worst rel cost err {ce:.2e}, worst rel grad err {ge:.2e}')


@pytest.mark.parametrize('M,tile', LAYOUTS)
def test_eval_many_problems_per_tile(M, tile, sm_count, tiled_handles, worlds16):
    """Perturbed problems over 16 maps at every lane layout the library can pick, sized so that every tile evaluates at
    least three problems, with problems that leave early (overflow, NaN) interleaved; then >= 512 of them evaluated
    alone must give the same bits as inside the large batch."""
    cfg = YamlConfig()
    h = tiled_handles[tile]
    ws, omaps = worlds16
    B, bound, trips = batch_for(sm_count, tile)
    inp = perturbed_inputs(cfg, ws[0], M, B, seed=1000 * M + tile)
    x, head, tail, ids, kind = inp['x'], inp['head'], inp['tail'], inp['ids'], inp['kind']
    big = h.eval(M, x, head, tail, ids, want_coeffs=True)
    assert (big['status'][kind == 1] == lib.ST_OVERFLOW).all()
    assert (big['status'][kind == 2] == lib.ST_NAN).all()
    assert (big['status'][(kind == 3) | (kind == 4) | (kind == 5)] == 0).all()
    ce, ge, cnt = check_eval_against_checker(cfg, M, omaps, x, head, tail, ids, big)
    # position independence: the same problem alone (a batch of one, same lane count) -- every output bit for bit
    rng = np.random.default_rng(M)
    sample = np.unique(np.concatenate([np.nonzero(kind > 0)[0][:60], rng.choice(B, 460, replace=False), [0, B - 1]]))
    assert sample.size >= 512
    for i in sample:
        one = h.eval(M, x[i:i + 1], head[i:i + 1], tail[i:i + 1], ids[i:i + 1], want_coeffs=True)
        for k in ('costs', 'grad', 'status', 'coeffs', 'ts'):
            assert same_bits(one[k][0], big[k][i]), (int(i), k)
    print(f'\n[A] M={M}, {tile} lanes: B={B} = 3 x {bound} + 5 (resident tiles <= {sm_count} SMs x 64 warps x {32 // tile}), '
          f'>= {trips} loop trips per tile; {len(np.unique(ids))} maps; {int((kind > 0).sum())} edge problems; vs checker on '
          f'{cnt} evaluations: worst rel cost err {ce:.2e}, worst rel grad err {ge:.2e}; {sample.size} problems alone identical')


# ------------------------------------------------------------------------------------------------ B: k_coeffs, k_sample
def tau_to_T(cfg, tau):
    """map_tau2T (EP:477-483) as the device computes it: its exp, bit-identical on the host (lib.exp_host)."""
    e = lib.exp_host(-np.asarray(tau, dtype=np.float64)).reshape(np.shape(tau))
    return (cfg.T_max - cfg.T_min) / (1.0 + e) + cfg.T_min


def sample_scale(c, ts):
    """Per trajectory: the largest of sum_k k^2 |c_k| max(1, T_i)^k over its pieces and dimensions -- the magnitude of
    the terms summed for position, velocity and acceleration (sampled states are compared relative to it)."""
    B, M = ts.shape
    c = np.abs(c.reshape(B, M, 6, 2))
    pw = np.maximum(1.0, ts)[:, :, None] ** np.arange(6)[None, None, :] * np.maximum(1, np.arange(6)) ** 2
    return np.maximum(1.0, np.max(np.einsum('bmkd,bmk->bmd', c, pw).reshape(B, -1), axis=1))


def counts_only(h, M, coeffs, ts, hz):
    B = ts.shape[0]
    count = np.zeros(B, np.int32)
    h._ck(h.lib.neo_sample(h.h, B, M, lib.ptr(lib.f64(coeffs)), lib.ptr(lib.f64(ts)), float(hz), 0, None, lib.ptr(count)))
    return count


def arange_len(ts, hz):
    """len(np.arange(0, sum(ts), 1/hz)) per row, with Python's left-to-right sum as the reference (TU:190)."""
    return np.array([len(np.arange(0, sum(row), 1 / hz)) for row in ts.tolist()])


@pytest.mark.parametrize('M', list(range(2, 11)))
def test_coeffs_and_sampling_every_M(M, sm_count, tiled_handles, worlds16):
    """neo_get_coeffs at a batch that loops every warp over three or more problems, against the checker's dense solve;
    a problem alone gives the same bits; neo_sample counts equal numpy's arange length exactly, states match the
    checker's sampling of the same coefficients.
    Tolerance: test_gpu_parity.test_get_coeffs_and_sampling holds M = 3 coefficients and states to 1e-10 m on plans
    whose coefficients are O(1-10); here the bound is 1e-10 times each piece's coefficient magnitude (coefficients) or
    each trajectory's term magnitude (states), which covers durations at T_min / T_max and ten pieces."""
    cfg = YamlConfig()
    h = tiled_handles[32]
    ws, _ = worlds16
    B, bound, trips = batch_for(sm_count, 32)
    inp = perturbed_inputs(cfg, ws[0], M, B, seed=7000 + M)
    nq = 2 * (M - 1)
    x = inp['x']
    q = np.nan_to_num(x[:, :nq]).reshape(B, 2, M - 1)
    ts = tau_to_T(cfg, x[:, nq:])
    # durations whose sum is an exact multiple of 1/hz for every integer hz (the count's knife edge)
    ts[:64] = 1.0
    ts[64:128] = np.where(np.arange(M) % 2 == 0, 1.25, 0.75)
    ts[128:192] = 0.5 * (1 + np.arange(M) % 3)
    head, tail = inp['head'], inp['tail']
    c = h.get_coeffs(M, q, ts, head, tail)
    ref = np.stack([c_oracle.get_coeffs(M, head[b], tail[b], q[b], ts[b]) for b in range(B)])
    err = np.abs(c - ref).reshape(B, M, 12).max(axis=2)
    scale = np.maximum(1.0, np.abs(ref).reshape(B, M, 12).max(axis=2))
    worst_c = float((err / scale).max())
    assert worst_c <= 1e-10, worst_c
    for i in np.unique(np.concatenate([np.arange(0, B, B // 61), [B - 1]])):
        assert same_bits(h.get_coeffs(M, q[i:i + 1], ts[i:i + 1], head[i:i + 1], tail[i:i + 1])[0], c[i]), int(i)
    # sampling
    sub = np.unique(np.concatenate([np.arange(192), np.random.default_rng(M).choice(B, 64, replace=False)]))
    scale_s = sample_scale(c[sub], ts[sub])
    worst_s = 0.0
    exact = sum(float(sum(r)).is_integer() for r in ts.tolist())
    for hz in (7, 10, 30, 60, 100):
        count = counts_only(h, M, c, ts, hz)
        want = arange_len(ts, hz)
        assert np.array_equal(count, want), (hz, np.nonzero(count != want)[0][:10])
        states, cnt = h.sample(M, c[sub], ts[sub], hz)
        assert np.array_equal(cnt, count[sub])
        for j, b in enumerate(sub):
            r = c_oracle.sample(M, c[b], ts[b], hz)
            assert r.shape[0] == cnt[j], (hz, int(b))
            e = float(np.max(np.abs(states[j, :cnt[j]] - r))) / scale_s[j] if cnt[j] else 0.0
            worst_s = max(worst_s, e)
    assert worst_s <= 1e-10, worst_s
    print(f'\n[B] M={M}: neo_get_coeffs B={B} = 3 x {bound} + 5 (32 lanes), >= {trips} loop trips per warp; worst coefficient '
          f'error / piece magnitude {worst_c:.2e}; counts at 7/10/30/60/100 Hz equal to np.arange on all {B} problems '
          f'({exact} of them with an integral sum of durations); worst state error / term magnitude {worst_s:.2e} on {sub.size} x 5')


def test_sample_beyond_the_grid_height(tiled_handles, worlds16):
    """k_sample puts trajectories on gridDim.y (at most 65,535) and loops over the rest: counts for 3 x 65,535 + 5
    trajectories and states for 65,535 + 1,001, the rows past the first grid pass compared with the checker."""
    cfg = YamlConfig(); M = 2
    h = tiled_handles[32]
    ws, _ = worlds16
    B = 3 * 65535 + 5
    inp = perturbed_inputs(cfg, ws[0], M, 4096, seed=55)
    q = np.nan_to_num(inp['x'][:, :2]).reshape(-1, 2, 1)
    rng = np.random.default_rng(56)
    ts = rng.uniform(0.55, 1.0, (4096, M))
    c = h.get_coeffs(M, q, ts, inp['head'], inp['tail'])
    idx = np.arange(B) % 4096
    count = counts_only(h, M, c[idx], ts[idx], 10.0)
    assert np.array_equal(count, arange_len(ts, 10.0)[idx])
    Bs = 65535 + 1001
    states, cnt = h.sample(M, c[idx[:Bs]], ts[idx[:Bs]], 7.0)
    assert np.array_equal(cnt, arange_len(ts, 7.0)[idx[:Bs]])
    worst = 0.0
    for b in list(range(65535, Bs)) + list(range(0, 65535, 997)):
        r = c_oracle.sample(M, c[idx[b]], ts[idx[b]], 7.0)
        assert r.shape[0] == cnt[b]
        worst = max(worst, float(np.max(np.abs(states[b, :cnt[b]] - r))))
    assert worst <= 1e-10 * float(sample_scale(c, ts).max()), worst
    print(f'\n[B] neo_sample past gridDim.y: counts of {B} trajectories exact; states of {Bs}, worst error {worst:.2e} m')


# ------------------------------------------------------------------------------------------- C: neo_optimize_dev timed
@pytest.mark.parametrize('name', ['c2', 'c5', 'c4'])
def test_optimize_dev_as_timed(name, gpu, runs):
    """bench.timed_steps (W = 1, K = 2) on the benchmark's DeviceRun: every step returns the same records, equal bit for
    bit to neo_optimize (host buffers) on the same inputs; c2 and c5 against the checker as in test_gpu_fullsize."""
    torch = gpu['torch']
    run = runs(name)
    wl, h, M, B = run.wl, run.h, run.M, run.B
    snaps = []
    launch = run.launch

    def launch_and_keep():       # stream-ordered copies of every step's records
        launch()
        snaps.append((run.out.clone(), run.work.clone()))
    run.launch = launch_and_keep
    try:
        bench.timed_steps(torch, None, run, 2, 1, gpu['flush'], False, None)
    finally:
        del run.launch
    assert len(snaps) == 3
    recs = [records(o, w, B, M) for o, w in snaps]
    for r in recs[1:]:
        assert_same_records(r, recs[0], 'step')
    head, tail = lib.pad_state(wl['head']), lib.pad_state(wl['tail'])
    host = h.optimize(M, wl['q0'], wl['ts0'], head, tail, wl['map_ids'], wl['retry_q'], wl['retry_ts'], 5)
    assert_same_records(host, recs[0], 'host path')
    rec = recs[0]
    msg = f'\n[C] {name}: B={B}, M={M}: 3 timed-path launches identical and equal to neo_optimize; ok {rec["ok"].mean():.4f}'
    if name == 'c4':
        print(msg)
        return
    sel = np.arange(B) if B <= 4096 else np.sort(np.random.default_rng(0).choice(B, 4096, replace=False))
    print(msg + f'; vs checker on {sel.size} problems:')
    compare_with_checker(wl['cfg'], M, wl['worlds'], wl['map_ids'], head, tail, wl['q0'], wl['ts0'], wl['retry_q'],
                         wl['retry_ts'], rec, sel, 0.975 if M == 3 else 0.97)


@pytest.mark.parametrize('name', ['c2', 'c4'])
def test_optimize_dev_input_statuses(name, gpu, runs):
    """The device entry point's own status inputs: x0_status for ~1 % of problems whose ts0 leaves (T_min, T_max), and
    retry_status = NEO_ST_DOMAIN for a retry guess outside it. Both must equal neo_optimize, which derives the same
    statuses on the host."""
    torch, dev = gpu['torch'], gpu['dev']
    run = runs(name)
    wl, h, M, B, n = run.wl, run.h, run.M, run.B, run.n
    cfg = wl['cfg']
    nq = 2 * (M - 1)
    head, tail = lib.pad_state(wl['head']), lib.pad_state(wl['tail'])
    rng = np.random.default_rng(17)
    bad = np.nonzero(rng.random(B) < 0.01)[0]
    ts_bad = wl['ts0'].copy()
    ts_bad[bad, rng.integers(0, M, bad.size)] = rng.choice([cfg.T_min, cfg.T_max, cfg.T_min - 0.3, cfg.T_max + 2.0, 0.0], bad.size)
    st = torch.cuda.current_stream().cuda_stream

    def device_run(ts0, rts):
        tau, s = h.T2tau(ts0)                      # tau = 0 where map_T2tau raises, as neo_optimize stages it
        x0_status = s.max(axis=1).astype(np.int32)
        rtau, rs = h.T2tau(rts)
        x0 = torch.from_numpy(np.concatenate([wl['q0'].reshape(B, nq), tau], axis=1)).to(dev)
        st_d = torch.from_numpy(x0_status).to(dev) if x0_status.any() else None
        rtau_d = torch.from_numpy(rtau).to(dev)
        out, work, res = dev_result(torch, dev, B, M)
        h._ck(h.lib.neo_optimize_dev(h.h, B, M, x0.data_ptr(), None if st_d is None else st_d.data_ptr(), run.head.data_ptr(),
                                     run.tail.data_ptr(), None if run.ids_d is None else run.ids_d.data_ptr(), run.rq.data_ptr(),
                                     rtau_d.data_ptr(), lib.ST_DOMAIN if rs.any() else 0, 5, C.byref(res), C.c_void_p(st)))
        torch.cuda.synchronize()
        return records(out, work, B, M), x0_status

    d, x0_status = device_run(ts_bad, wl['retry_ts'])
    assert (x0_status[bad] == lib.ST_DOMAIN).all() and x0_status.sum() == lib.ST_DOMAIN * bad.size
    host = h.optimize(M, wl['q0'], ts_bad, head, tail, wl['map_ids'], wl['retry_q'], wl['retry_ts'], 5)
    assert_same_records(host, d, 'x0_status')
    assert (d['attempt'][bad] >= 1).all()          # attempt 0 of those problems never ran
    rts_bad = wl['retry_ts'].copy(); rts_bad[M // 2] = cfg.T_max + 1.0
    d2, _ = device_run(wl['ts0'], rts_bad)
    host2 = h.optimize(M, wl['q0'], wl['ts0'], head, tail, wl['map_ids'], wl['retry_q'], rts_bad, 5)
    assert_same_records(host2, d2, 'retry_status')
    failed0 = d2['attempt'] > 0
    assert (d2['ok'][failed0] == 0).all() and (d2['status'][failed0] == lib.ST_DOMAIN).all() and (d2['runs'] <= 1).all()
    print(f'\n[C] {name}: x0_status on {bad.size} problems and retry_status = NEO_ST_DOMAIN ({int(failed0.sum())} problems '
          f'reach a retry): neo_optimize_dev equal to neo_optimize bit for bit')


# --------------------------------------------------------------------------------------------- D: the work counters
def recount(cfg, M, omaps, ids, head, tail, tr, out, B):
    """For every evaluation of attempts 0..attempt recorded by neo_optimize_trace: samples S, velocity-violating S_v and
    colliding S_c recomputed in NumPy from the recorded decision vector, summed per problem; plus, per problem, the
    number of samples within 1e-9 (relative) of a threshold or of a cell boundary, and the tasks that ended on an
    evaluation error."""
    n, nq = 3 * M - 2, 2 * (M - 1)
    S, Sv, Sc, knife, knife_v, knife_c = (np.zeros(B, np.int64) for _ in range(6))
    raised = np.zeros(B, np.int64); lens = np.zeros(B, np.int64)
    xs, owner, stat = [], [], []
    for b in range(B):
        for k in range(int(out['attempt'][b]) + 1):
            t = k * B + b
            L = int(tr['len'][t])
            lens[b] += L
            if L == 0:
                continue
            st = tr['status'][t, :L]
            assert (st[:-1] == 0).all(), (b, k)          # an evaluation error ends its task
            raised[b] += int(st[-1] != 0)
            xs.append(tr['x'][t, :L]); owner.append(np.full(L, b)); stat.append(st)
    X = np.concatenate(xs); own = np.concatenate(owner); st = np.concatenate(stat)
    T = tau_to_T(cfg, X[:, nq:])
    early = (st == lib.ST_OVERFLOW) | np.isnan(T).any(axis=1)        # left before the sample loop: no samples
    ns = np.where(early[:, None], 0, np.trunc(T / cfg.delta_t)).astype(np.int64)
    np.add.at(S, own, ns.sum(axis=1))
    finite = ~early & np.isfinite(X).all(axis=1)                     # NaN positions: no violation, outside every cell
    v2 = cfg.v_max * cfg.v_max
    idx = np.nonzero(finite)[0]
    for c0 in range(0, idx.size, 1024):
        ev = idx[c0:c0 + 1024]
        cf = np.stack([c_oracle.get_coeffs(M, head[own[e]], tail[own[e]], X[e, :nq].reshape(2, M - 1), T[e]) for e in ev])
        cf = cf.reshape(len(ev), M, 6, 2)
        cnt = ns[ev].reshape(-1)                                      # (evaluation, piece) groups of samples
        grp = np.repeat(np.arange(cnt.size), cnt)
        j = np.arange(grp.size) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        t = j * cfg.delta_t
        cs = cf.reshape(-1, 6, 2)[grp]
        tp = t[:, None] ** np.arange(6)[None, :]
        pos = np.einsum('sk,skd->sd', tp, cs)
        vel = np.einsum('sk,skd->sd', tp[:, :5] * np.arange(1, 6)[None, :], cs[:, 1:])
        vv = (vel[:, 0] * vel[:, 0] + vel[:, 1] * vel[:, 1]) - v2
        e_of = ev[grp // M]
        b_of = own[e_of]
        dis = np.empty(grp.size)
        near = np.zeros(grp.size, bool)
        for s in np.unique(ids[b_of]):
            sel = ids[b_of] == s
            m = omaps[s]
            _, dis[sel], _ = m.query(pos[sel])
            qq = (pos[sel] - np.array([m.ox, m.oy])) / m.res
            near[sel] = (np.abs(qq - np.round(qq)) <= 1e-9 * np.maximum(1.0, np.abs(qq))).any(axis=1)
        vc = cfg.safe_dis - dis
        # the distance is a map value, bit-identical on both sides for the same cell (cells at exactly safe_dis are
        # common and decided alike): only the cell can differ, so the collision test's knife edge is the cell boundary
        kv = np.abs(vv) <= 1e-9 * v2
        np.add.at(Sv, b_of, (vv > 0.0).astype(np.int64))
        np.add.at(Sc, b_of, (vc > 0.0).astype(np.int64))
        np.add.at(knife_v, b_of, kv.astype(np.int64))
        np.add.at(knife_c, b_of, near.astype(np.int64))
        np.add.at(knife, b_of, (kv | near).astype(np.int64))
    return dict(S=S, Sv=Sv, Sc=Sc, knife=knife, knife_v=knife_v, knife_c=knife_c, raised=raised, lens=lens, evals=X.shape[0],
                raised_samples=int(ns[st != 0].sum()))


@pytest.mark.parametrize('name,count,tile', [('c4', 512, 8), ('c5', 128, 32)])
def test_work_counters(name, count, tile):
    """neo_result.work (samples, velocity-violating, colliding samples over the evaluations of attempts 0..attempt) against
    a NumPy recount of every evaluation neo_optimize_trace recorded. A few extra problems start from a NaN waypoint:
    their first evaluation raises (int(nan)) after sampling, which pins the counting definitions -- such an evaluation
    counts in work but not in nfev, so sum(trace lengths) = nfev + tasks that ended on an evaluation error."""
    wl = bench.workload(name, 0, 1)
    cfg, M = wl['cfg'], wl['M']
    ids_all = wl['map_ids'] if wl['map_ids'] is not None else np.zeros(wl['B'], np.int32)
    extra = 16 if name == 'c4' else 8
    sel = np.concatenate([np.arange(count), np.arange(extra)])
    B = sel.size
    q0 = wl['q0'][sel].copy(); q0[count:, 0, 0] = np.nan
    ts0, rq = wl['ts0'][sel], wl['retry_q'][sel]
    head, tail, ids = lib.pad_state(wl['head'][sel]), lib.pad_state(wl['tail'][sel]), ids_all[sel]
    used = np.unique(ids)
    h = handle_with_tile(cfg, int(used.max()) + 1, tile)
    for s in used:
        w = wl['worlds'][s]
        h.set_map_occupancy(int(s), w.H, w.W, w.res, w.ox, w.oy, w.occ)
    plain = h.optimize(M, q0, ts0, head, tail, ids if wl['map_ids'] is not None else None, rq, wl['retry_ts'], 5)
    cap = int(plain['nfev'].max()) + 2            # a task makes at most nfev + 1 evaluations
    out, tr = h.optimize_trace(M, q0, ts0, head, tail, ids if wl['map_ids'] is not None else None, rq, wl['retry_ts'], 5, cap=cap)
    assert_same_records(out, plain, 'trace')
    for b in range(B):
        for k in range(int(out['attempt'][b]) + 1):
            assert tr['len'][k * B + b] < cap
    omaps = {int(s): c_oracle.OracleMap.from_world(wl['worlds'][s]) for s in used}
    r = recount(cfg, M, omaps, ids, head, tail, tr, out, B)
    w = out['work']
    assert np.array_equal(r['S'], w[:, 0]), np.nonzero(r['S'] != w[:, 0])[0][:10]
    dv, dc = np.abs(w[:, 1] - r['Sv']), np.abs(w[:, 2] - r['Sc'])
    assert (dv <= r['knife']).all() and (dc <= r['knife']).all(), (np.nonzero(dv > r['knife'])[0][:10], np.nonzero(dc > r['knife'])[0][:10])
    assert np.array_equal(r['lens'], out['nfev'] + r['raised'])
    assert (r['raised'][count:] >= 1).all() and r['raised_samples'] > 0
    print(f'\n[D] {name}: {B} problems ({extra} starting from a NaN waypoint), {tile} lanes, cap {cap}: {r["evals"]} evaluations '
          f'recounted; samples {int(r["S"].sum())} exact; velocity-violating {int(w[:, 1].sum())} (numpy {int(r["Sv"].sum())}), '
          f'colliding {int(w[:, 2].sum())} (numpy {int(r["Sc"].sum())}); knife-edge samples {int(r["knife"].sum())} '
          f'(speed {int(r["knife_v"].sum())}, cell boundary {int(r["knife_c"].sum())}) '
          f'({r["knife"].sum() / max(r["S"].sum(), 1):.2e} of all); {int(r["raised"].sum())} evaluations raised '
          f'({r["raised_samples"]} samples in work, not in nfev)')
