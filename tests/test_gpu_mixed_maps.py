"""Launches whose problems read maps of different shape, resolution and origin, and slots that change shape.

Every kernel that reads a map picks it per problem (maps[map_ids[b]]) and takes that map's origin, 1 / res, H, W and
cell base inside its loops. The other tests run only maps of one geometry per launch, so a kernel that took the geometry
of slot 0, of the previous problem of its tile, or once per warp or launch, would pass them. Here one handle holds eight
maps chosen so that any mix-up changes results:

  slot  shape      res    origin               upload                why
  0     300x300    0.1    (0, -15)             set_map_occupancy     the benchmark's geometry (make_world(0))
  1     300x300    0.12   (-7.31, 4.05)        set_map_occupancy     slot 0's cells under another geometry (twin)
  2, 3  173x411    0.05   far / near origin    set_maps_occupancy    H != W, W not a multiple of 32, |origin| ~ 1e3
  4     411x173    0.07   (3.3, -2.2)          set_map_occupancy     slot 2's cell count, transposed
  5     1200x1200  0.05   (0, -30)             set_map_occupancy     the largest A* grid (sizes the search scratch)
  6     7x5        0.25   (-2.1, 3.3)          set_map_esdf          tiny: most samples fall outside (distance 10000)
  7     grid_for   0.3    grid_for             set_map_points        1 / res inexact; cloud with edge and NaN points

Batches interleave and shuffle the map ids and hold 3 x (resident tiles) + 5 problems, so every tile moves through at
least three problems, most of them on a map other than the previous one's. Bit-for-bit comparisons are always between
handles created with the same NEO_TILE (different lane counts legitimately differ in the last bits).
"""
import os
import subprocess
import time
from dataclasses import dataclass, field

import numpy as np
import pytest

from neo_planner_b200 import guesses, lib, pointcloud
from neo_planner_b200.esdf import ESDF
from neo_planner_b200.planner import BatchPlanner, MinJerkPlanner
from neo_planner_b200.worlds import World, YamlConfig, make_problems, make_world
from oracle import astar_ref, c_oracle, minco_ref, pointcloud_ref
from test_gpu_bench_paths import LAYOUTS, RECORD_FIELDS, batch_for, same_bits

pytestmark = pytest.mark.gpu

CFG = YamlConfig()
N_SLOTS = 8
SMALL = 6                     # the 7 x 5 map: too small for the spans of M >= 4
POOL = 96                     # start/goal pairs per map and piece count


# ------------------------------------------------------------------------------------------------------------ map set
@dataclass
class Geo:
    slot: int
    H: int
    W: int
    res: float
    ox: float
    oy: float
    kind: str                                  # 'occ' | 'esdf' | 'points'
    occ: np.ndarray                            # the (H, W) occupancy the map is built from
    scale: float = 1.0                         # problem scale relative to slot 0 (the twin's problems are scaled copies)
    pts: np.ndarray = None                     # 'points': the cloud and its slab
    z: tuple = None
    omap: c_oracle.OracleMap = field(default=None, repr=False)
    _grid: object = field(default=None, repr=False)

    def __post_init__(self):
        self.omap = c_oracle.OracleMap(self.occ, self.H, self.W, self.res, self.ox, self.oy)

    @property
    def org(self):
        return np.array([self.ox, self.oy])

    @property
    def span(self):
        return np.array([self.W * self.res, self.H * self.res])

    def grid(self):
        """minco_ref.GridMap (scipy's EDT, which the checker's map is pinned to) for oracle/astar_ref.py."""
        if self._grid is None:
            self._grid = minco_ref.GridMap(self.occ, self.H, self.W, self.res, self.ox, self.oy)
        return self._grid


def pillar_occ(H, W, res, n, seed):
    rng = np.random.default_rng(seed)
    occ = np.zeros((H, W), np.int8)
    for _ in range(n):
        sx, sy = rng.uniform(0.5, 1.5, 2) / res
        c, r = rng.uniform(0, W), rng.uniform(0, H)
        occ[int(max(r - sy / 2, 0)):int(min(r + sy / 2, H - 1)) + 1, int(max(c - sx / 2, 0)):int(min(c + sx / 2, W - 1)) + 1] = 100
    occ[rng.random((H, W)) < 0.002] = -1                        # unknown cells are free (ESDF:23)
    return occ


def point_cloud(res):
    """Pillar columns over a 24 x 14 m area plus a ground plane below the slab, then the adversarial points: on cell
    edges, in the band between -1 and 0 cells (floor gives -1, truncation would give 0), z exactly at the slab's ends in
    float32 and one float32 step beyond them, NaN and infinite coordinates. Returns (xyz float32, z_min, z_max, grid)."""
    rng = np.random.default_rng(77)
    cols = []
    for _ in range(14):
        cx, cy = rng.uniform(-2.0, 20.0), rng.uniform(5.5, 18.5)
        s = rng.uniform(0.3, 1.2)
        k = int(rng.integers(40, 120))
        xy = np.stack([cx + rng.uniform(-s, s, k), cy + rng.uniform(-s, s, k)], 1)
        cols.append(np.concatenate([xy, rng.uniform(0.6, 2.0, (k, 1))], 1))
    gx, gy = np.meshgrid(np.arange(-3.0, 21.0, 0.25), np.arange(5.0, 19.0, 0.25))
    cols.append(np.stack([gx.ravel(), gy.ravel(), np.zeros(gx.size)], 1))           # ground: under the slab
    base = np.concatenate(cols).astype(np.float32)
    ox, oy, H, W = pointcloud.grid_for(base, res)
    z_min, z_max = 0.5, float(np.float32(2.3))
    f32 = np.float32
    adv = []
    for k in range(0, W + 1, 3):                              # x on the cell edges, formed as product and as sum
        adv.append((ox + k * res, oy + 0.5 * res * (k % H + 1), 1.0))
        adv.append((sum([ox] + [res] * k), oy + res * (k % H) + 0.01, 1.0))
    for k in range(0, H + 1, 3):
        adv.append((ox + 0.5 * res * (k % W + 1), oy + k * res, 1.0))
    for u in (1e-9, 0.25, 0.5, 0.999):                        # between -1 and 0 cells
        adv.append((ox - u * res, oy + 3.5 * res, 1.0)); adv.append((ox + 4.5 * res, oy - u * res, 1.0))
    zlo, zhi = f32(z_min), f32(z_max)
    for j, z in enumerate((zlo, zhi, np.nextafter(zlo, f32(-np.inf)), np.nextafter(zhi, f32(np.inf)))):
        adv.append((ox + (7.5 + 2 * j) * res, oy + 2.5 * res, z))
    for bad in ((np.nan, oy + 1.0, 1.0), (ox + 1.0, np.nan, 1.0), (ox + 1.0, oy + 1.0, np.nan), (np.inf, oy + 1.0, 1.0),
                (ox + 1.0, -np.inf, 1.0), (-np.inf, np.inf, 1.0)):
        adv.append(bad)
    xyz = np.concatenate([base, np.array(adv, dtype=np.float64).astype(np.float32)])
    return xyz, z_min, z_max, (ox, oy, H, W)


def build_geos():
    w0, w5 = make_world(0), make_world(3, dense=True)
    tiny = np.zeros((7, 5), np.int8); tiny[2:4, 1:3] = 100; tiny[6, 4] = 100
    xyz, z_min, z_max, (ox7, oy7, H7, W7) = point_cloud(0.3)
    occ7 = pointcloud_ref.project_numpy(xyz, z_min, z_max, H7, W7, 0.3, ox7, oy7)
    return [
        Geo(0, 300, 300, 0.1, 0.0, -15.0, 'occ', w0.occ),
        Geo(1, 300, 300, 0.12, -7.31, 4.05, 'occ', w0.occ, scale=1.2),
        Geo(2, 173, 411, 0.05, 1234.5, -987.25, 'occ', pillar_occ(173, 411, 0.05, 14, 2)),
        Geo(3, 173, 411, 0.05, -0.37, 0.81, 'occ', pillar_occ(173, 411, 0.05, 14, 3)),
        Geo(4, 411, 173, 0.07, 3.3, -2.2, 'occ', pillar_occ(411, 173, 0.07, 22, 4)),
        Geo(5, 1200, 1200, 0.05, 0.0, -30.0, 'occ', w5.occ),
        Geo(6, 7, 5, 0.25, -2.1, 3.3, 'esdf', tiny),
        Geo(7, H7, W7, 0.3, ox7, oy7, 'points', occ7, pts=xyz, z=(z_min, z_max)),
    ]


def upload(h, slot, g):
    """g into slot `slot` of h through g's own upload path (slots 2 and 3 alone: set_map_occupancy)."""
    if g.kind == 'esdf':
        h.set_map_esdf(slot, g.res, g.ox, g.oy, g.omap.esdf, g.omap.gx, g.omap.gy)
    elif g.kind == 'points':
        h.set_map_points(slot, g.pts, g.z[0], g.z[1], g.H, g.W, g.res, g.ox, g.oy)
    else:
        h.set_map_occupancy(slot, g.H, g.W, g.res, g.ox, g.oy, g.occ)


def new_handle(n_maps, **env):
    """A handle created under development switches (NEO_TILE, NEO_GROUPED, NEO_ASTAR_ICAP are read at neo_create);
    a value of None unsets the variable."""
    old = {k: os.environ.get(k) for k in env}
    for k, v in env.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = str(v)
    try:
        return lib.Handle(CFG, 0, n_maps)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def mixed_handle(geos, **env):
    """All eight maps, uploaded as the table in the module docstring says (slots 2 and 3 in one set_maps_occupancy)."""
    h = new_handle(N_SLOTS, **env)
    for g in geos:
        if g.slot not in (2, 3):
            upload(h, g.slot, g)
    g2, g3 = geos[2], geos[3]
    h.set_maps_occupancy([2, 3], g2.H, g2.W, g2.res, [g2.ox, g3.ox], [g2.oy, g3.oy], np.stack([g2.occ, g3.occ]))
    return h


def single_handle(g, **env):
    h = new_handle(1, **env)
    upload(h, 0, g)
    return h


# --------------------------------------------------------------------------------------------------------- problems
def slots_for(M):
    return [s for s in range(N_SLOTS) if M <= 3 or s != SMALL]


def edt_at(g, p):
    """The checker map's distance at points p (n, 2): int() cells as ESDF:61, -1 outside."""
    r = np.trunc((p[:, 1] - g.oy) / g.res); c = np.trunc((p[:, 0] - g.ox) / g.res)
    inside = (r >= 0) & (r < g.H) & (c >= 0) & (c < g.W) & np.isfinite(r) & np.isfinite(c)
    out = np.full(p.shape[0], -1.0)
    out[inside] = g.omap.esdf[r[inside].astype(int), c[inside].astype(int)]
    return out


def pool_for(g, M, seed):
    """POOL start/goal pairs (head, tail (POOL, 3, 2)) of length 5M/3 on free cells of g, both ends on the map when it
    can hold the span; three in four (at least) pass within safe_dis of an obstacle on the straight line, so the
    collision terms are active. A map too small for the span gets pairs around it (it is used at M <= 3 only)."""
    rng = np.random.default_rng(seed)
    L = 5.0 * M / 3.0
    margin = CFG.safe_dis + 0.1
    fits = L < 0.9 * g.span.max()
    heads, tails = [], []
    want_near = np.arange(POOL) % 4 != 3
    for _ in range(400):
        n = 4096
        if fits:
            p0 = g.org + rng.uniform(0.0, 1.0, (n, 2)) * g.span
        else:
            p0 = g.org + rng.uniform(-1.0, 2.0, (n, 2)) * g.span
        th = rng.uniform(0, 2 * np.pi, n)
        d = np.stack([np.cos(th), np.sin(th)], 1)
        p1 = p0 + L * d
        if fits:
            ok = (edt_at(g, p0) > margin) & (edt_at(g, p1) > margin)
        else:
            ok = (edt_at(g, p0) != 0.0) & (edt_at(g, p1) != 0.0)
        lam = np.linspace(0, 1, 24)
        seg = p0[:, None, :] + lam[None, :, None] * (p1 - p0)[:, None, :]
        dd = edt_at(g, seg.reshape(-1, 2)).reshape(n, -1)
        near = ((dd >= 0) & (dd < CFG.safe_dis)).any(axis=1)
        for i in np.nonzero(ok)[0]:
            k = len(heads)
            if k == POOL:
                break
            if fits and want_near[k] and not near[i]:
                continue
            hd = np.zeros((3, 2)); tl = np.zeros((3, 2))
            hd[0], hd[1] = p0[i], 0.5 * d[i]
            tl[0], tl[1] = p1[i], 0.8 * CFG.v_max * d[i]
            heads.append(hd); tails.append(tl)
        if len(heads) == POOL:
            break
    assert len(heads) == POOL, (g.slot, M, len(heads))
    return np.array(heads), np.array(tails)


class Problems:
    """Start/goal pools per (slot, M); the twin's (slot 1) are slot 0's scaled about the origin by res1 / res0."""

    def __init__(self, geos):
        self.geos = geos
        self.cache = {}

    def pool(self, slot, M):
        if (slot, M) not in self.cache:
            if slot == 1:
                h0, t0 = self.pool(0, M)
                g0, g1 = self.geos[0], self.geos[1]
                s = g1.res / g0.res
                h1, t1 = h0.copy(), t0.copy()
                h1[:, 0] = g1.org + (h0[:, 0] - g0.org) * s
                t1[:, 0] = g1.org + (t0[:, 0] - g0.org) * s
                self.cache[(slot, M)] = (h1, t1)
            else:
                self.cache[(slot, M)] = pool_for(self.geos[slot], M, 1000 * slot + M)
        return self.cache[(slot, M)]

    def batch(self, M, B, seed):
        """B problems over slots_for(M): ids interleaved, then shuffled. Returns dict(ids, head, tail, j)."""
        rng = np.random.default_rng(seed)
        slots = np.array(slots_for(M), np.int32)
        ids = rng.permutation(np.resize(slots, B)).astype(np.int32)
        j = rng.integers(0, POOL, B)
        head = np.zeros((B, 3, 2)); tail = np.zeros((B, 3, 2))
        for s in slots:
            sel = ids == s
            hp, tp = self.pool(int(s), M)
            head[sel], tail[sel] = hp[j[sel]], tp[j[sel]]
        return dict(ids=ids, head=head, tail=tail, j=j)

    def eval_inputs(self, M, B, seed):
        """A batch plus decision vectors: waypoints on the straight line + N(0, 0.4 m x scale), tau ~ N(0, 1.5); every
        37th problem overflows (tau = -720) and the next one has a NaN waypoint, so tiles also leave problems early."""
        b = self.batch(M, B, seed)
        rng = np.random.default_rng(seed + 1)
        scale = np.array([g.scale for g in self.geos])[b['ids']]
        lam = np.linspace(0, 1, M + 1)[1:-1]
        h0, t0 = b['head'][:, 0], b['tail'][:, 0]
        q = h0[:, None, :] + lam[None, :, None] * (t0 - h0)[:, None, :] + rng.normal(0, 0.4, (B, M - 1, 2)) * scale[:, None, None]
        q = np.transpose(q, (0, 2, 1)).reshape(B, -1)
        tau = rng.normal(0, 1.5, (B, M))
        kind = np.zeros(B, np.int32); kind[1::37] = 1; kind[2::37] = 2
        tau[kind == 1, 0] = -720.0
        q[kind == 2, 0] = np.nan
        b.update(x=np.concatenate([q, tau], axis=1), kind=kind)
        return b


# ---------------------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope='module', autouse=True)
def wall_time():
    t0 = time.perf_counter()
    try:
        card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                              text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                      # the figure is reported, not needed
        card = f'(nvidia-smi: {e})'
    yield
    print(f'\ntest_gpu_mixed_maps: wall time {time.perf_counter() - t0:.1f} s on {card}')


@pytest.fixture(scope='module')
def geos():
    return build_geos()


@pytest.fixture(scope='module')
def problems(geos):
    return Problems(geos)


@pytest.fixture(scope='module')
def sm_count():
    h = lib.Handle(CFG, 0, 1)
    n = h.device_info()['sm_count']
    h.close()
    return n


@pytest.fixture(scope='module')
def eval_handles(geos):
    """Per NEO_TILE: the mixed handle and one single-map handle per slot."""
    cache = {}

    def get(tile, slot=None):
        key = (tile, slot)
        if key not in cache:
            cache[key] = mixed_handle(geos, NEO_TILE=tile) if slot is None else single_handle(geos[slot], NEO_TILE=tile)
        return cache[key]
    yield get
    for h in cache.values():
        h.close()


def assert_same_records(a, b, what):
    for k in RECORD_FIELDS:
        assert same_bits(a[k], b[k]), (what, k)
    assert same_bits(a['work'][:, :3], b['work'][:, :3]), (what, 'work')


def sub(rec, sel):
    return {k: (None if v is None else v[sel]) for k, v in rec.items()}


# ------------------------------------------------------------------------------------------- B.1 map build, lookups
def adversarial_points(g, rng):
    """Random points over the map and a margin around it, and the points where a cell index is decided by one rounding:
    x = ox + k res formed as a product and as a running sum (likewise y), points between -1 and 0 cells (int() gives
    0, they are outside), ox + W res and oy + H res one ulp either side, and points far away."""
    pts = [g.org + rng.uniform(-0.2, 1.2, (4096, 2)) * g.span]
    ks = np.arange(-2, max(g.W, g.H) + 3)
    xs_p, ys_p = g.ox + ks * g.res, g.oy + ks * g.res
    xs_s, ys_s = np.empty(ks.size), np.empty(ks.size)
    sx = g.ox + ks[0] * g.res; sy = g.oy + ks[0] * g.res
    for i in range(ks.size):
        xs_s[i], ys_s[i] = sx, sy
        sx += g.res; sy += g.res
    mid = g.org + 0.5 * g.span
    other = g.org + rng.uniform(0, 1, (ks.size, 2)) * g.span
    for xs, ys in ((xs_p, ys_p), (xs_s, ys_s)):
        pts += [np.stack([xs, np.full(ks.size, mid[1])], 1), np.stack([np.full(ks.size, mid[0]), ys], 1),
                np.stack([xs, other[:, 1]], 1), np.stack([other[:, 0], ys], 1), np.stack([xs, ys], 1)]
    u = np.concatenate([[1e-12, 1e-9, 0.5, 0.999999], rng.uniform(0, 1, 60)])
    band_x, band_y = g.ox - u * g.res, g.oy - u * g.res
    yy, xx = g.oy + rng.uniform(0, 1, u.size) * g.span[1], g.ox + rng.uniform(0, 1, u.size) * g.span[0]
    pts += [np.stack([band_x, yy], 1), np.stack([xx, band_y], 1), np.stack([band_x, band_y], 1),
            np.stack([np.nextafter(g.ox, -np.inf) + 0 * yy, yy], 1), np.stack([xx, np.nextafter(g.oy, -np.inf) + 0 * xx], 1)]
    ex, ey = g.ox + g.W * g.res, g.oy + g.H * g.res
    for e in (np.nextafter(ex, -np.inf), ex, np.nextafter(ex, np.inf)):
        pts.append(np.stack([np.full(u.size, e), yy], 1))
    for e in (np.nextafter(ey, -np.inf), ey, np.nextafter(ey, np.inf)):
        pts.append(np.stack([xx, np.full(u.size, e)], 1))
    far = np.array([[1e6, 0.0], [-1e6, 0.0], [0.0, 1e6], [0.0, -1e6], [1e12, -1e12], [-3e15, 3e15]]) + g.org
    pts.append(far)
    return np.concatenate(pts)


def test_map_build_and_lookups(geos):
    """get_map of every slot bit-identical to its checker map; query_map bit-identical to OracleMap.query on random and
    adversarial points; the point-cloud grid equal to pointcloud_ref.project_numpy; no occupancy in the ESDF slot."""
    h = mixed_handle(geos)
    rng = np.random.default_rng(5)
    n_pts = 0
    for g in geos:
        e, gx, gy = h.get_map(g.slot, g.H, g.W)
        assert same_bits(e, g.omap.esdf) and same_bits(gx, g.omap.gx) and same_bits(gy, g.omap.gy), g.slot
        if g.kind == 'esdf':
            with pytest.raises(lib.NeoError, match='no occupancy'):
                h.get_occupancy(g.slot, g.H, g.W)
        else:
            assert same_bits(h.get_occupancy(g.slot, g.H, g.W), g.occ), g.slot        # as uploaded, unknown (-1) too
        with pytest.raises(lib.NeoError):
            h.get_map(g.slot, g.W, g.H) if g.W != g.H else h.get_map(g.slot, g.H, g.W + 1)
        p = adversarial_points(g, rng)
        idx, d, gr = h.query_map(g.slot, p)
        ridx, rd, rg = g.omap.query(p)
        assert same_bits(idx, ridx) and same_bits(d, rd) and same_bits(gr, rg), g.slot
        outside = (ridx[:, 0] < 0).sum()
        assert 0 < outside < p.shape[0]
        n_pts += p.shape[0]
    g7 = geos[7]
    raw = g7.pts[:-6].astype(np.float64)                        # the cloud's edge cases really sit on the edges
    assert g7.occ.sum() > 0 and (np.floor((raw[:, 0] - g7.ox) / g7.res) == -1).any()
    h.close()
    print(f'\n[B.1] {len(geos)} maps bit-identical to the checker; {n_pts} lookups identical; point-cloud grid '
          f'{g7.H}x{g7.W}, {int((g7.occ == 100).sum())} occupied cells, equal to project_numpy')


# -------------------------------------------------------------------------------------------------------- B.2 k_eval
def check_against_checker(geos, M, b, out):
    p = c_oracle.Params.from_config(CFG)
    B = b['x'].shape[0]
    costs = np.zeros((B, 4)); grad = np.zeros_like(b['x']); status = np.zeros(B, np.int32)
    for s in np.unique(b['ids']):
        sel = np.nonzero(b['ids'] == s)[0]
        costs[sel], grad[sel], status[sel] = c_oracle.eval_batch(p, geos[s].omap, M, b['head'][sel], b['tail'][sel], b['x'][sel])
    bad = np.nonzero(out['status'] != status)[0]
    assert bad.size == 0, ('status differs from the checker', bad[:10], out['status'][bad[:10]], status[bad[:10]])
    ok = status == 0
    assert np.allclose(out['costs'][ok], costs[ok], rtol=1e-6, atol=1e-9)
    cerr = np.max(np.abs(out['costs'][ok] - costs[ok]) / np.maximum(np.abs(costs[ok]), 1e-3), axis=1)
    gerr = np.max(np.abs(out['grad'][ok] - grad[ok]), axis=1) / np.maximum(np.max(np.abs(grad[ok]), axis=1), 1e-9)
    assert (gerr <= 1e-6).all(), gerr.max()
    return float(cerr.max()), float(gerr.max()), int(ok.sum()), costs


@pytest.mark.parametrize('M,tile', LAYOUTS)
def test_eval_mixed_geometry(M, tile, geos, problems, sm_count, eval_handles):
    """k_eval over all maps in one launch: statuses equal to the checker's and cost / gradient within 1e-6, map by map;
    bit for bit equal to single-map handles evaluating only their map's problems; and, as evidence that this comparison
    sees a geometry mix-up, the same batch with every id moved to a map of another geometry changes the results of most
    problems."""
    B, bound, trips = batch_for(sm_count, tile)
    b = problems.eval_inputs(M, B, seed=31 * M + tile)
    h = eval_handles(tile)
    out = h.eval(M, b['x'], b['head'], b['tail'], b['ids'], want_coeffs=True)
    assert (out['status'][b['kind'] == 1] == lib.ST_OVERFLOW).all() and (out['status'][b['kind'] == 2] == lib.ST_NAN).all()
    ce, ge, cnt, ref_costs = check_against_checker(geos, M, b, out)
    active = int(((ref_costs[:, 3] > 0) & (out['status'] == 0)).sum())
    for s in slots_for(M):
        sel = np.nonzero(b['ids'] == s)[0]
        one = eval_handles(tile, s).eval(M, b['x'][sel], b['head'][sel], b['tail'][sel], None, want_coeffs=True)
        for k in ('costs', 'grad', 'status', 'coeffs', 'ts'):
            assert same_bits(one[k], out[k][sel]), (s, k)
    # sensitivity: each slot's problems evaluated on the next slot (0 -> 1 among them)
    slots = slots_for(M)
    nxt = {s: slots[(i + 1) % len(slots)] for i, s in enumerate(slots)}
    moved = h.eval(M, b['x'], b['head'], b['tail'], np.array([nxt[s] for s in b['ids']], np.int32))
    plain = b['kind'] == 0
    changed = plain & ((moved['costs'] != out['costs']).any(axis=1) | (moved['grad'] != out['grad']).any(axis=1))
    frac = changed.sum() / plain.sum()
    twin = plain & (b['ids'] == 0)
    frac0 = changed[twin].sum() / twin.sum()
    assert frac >= 0.5 and frac0 >= 0.5, (frac, frac0)
    print(f'\n[B.2] M={M}, {tile} lanes: B={B} = 3 x {bound} + 5, >= {trips} loop trips per tile over {len(slots)} maps; '
          f'vs checker on {cnt} evaluations ({active} with collision cost): worst rel cost err {ce:.2e}, grad err {ge:.2e}; '
          f'single-map handles identical; ids moved to another map change {frac:.3f} of the problems (slot 0 -> 1: {frac0:.3f})')


# ---------------------------------------------------------------------------------------------------- B.3 k_optimize
def plan_inputs(problems, M, B, seed):
    b = problems.batch(M, B, seed)
    q0, ts0 = guesses.straight_line_guess(CFG, b['head'], b['tail'], M)
    rq, rts = guesses.retry_guesses(CFG, b['head'], b['tail'], M, 4, rng=np.random.default_rng(seed + 2))
    b.update(q0=q0, ts0=ts0, rq=rq, rts=rts)
    return b


def optimize_dev(h, M, b):
    """neo_optimize_dev on CUDA tensors with the inputs neo_optimize stages on the host (x0 = [q0, T2tau(ts0)])."""
    import torch
    dev = torch.device('cuda', 0)
    B = b['q0'].shape[0]
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)        # noqa: E731
    tau, st = h.T2tau(b['ts0'])
    rtau, rst = h.T2tau(b['rts'])
    out = h.optimize_dev(M, T(np.concatenate([b['q0'].reshape(B, -1), tau], axis=1)), T(b['head']), T(b['tail']),
                         T(st.max(axis=1).astype(np.int32)), T(b['ids']), T(b['rq']), T(rtau), int(rst.max()), 5)
    torch.cuda.synchronize()
    return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}


def replay(h, M, b, rec, sel):
    """neo_optimize_trace on the problems `sel` (their map ids interleaved as in the batch): the records must equal the
    batch's, and every attempt that ran must replay through the checker's L-BFGS-B bit for bit."""
    cap = int(rec['nfev'][sel].max()) + 2
    out, tr = h.optimize_trace(M, b['q0'][sel], b['ts0'][sel], b['head'][sel], b['tail'][sel], b['ids'][sel], b['rq'][sel],
                               b['rts'], 5, cap=cap)
    assert_same_records(out, sub(rec, sel), 'trace of the sample')
    n = sel.size
    tau0, _ = h.T2tau(b['ts0'][sel]); rtau, _ = h.T2tau(b['rts'])
    attempts = evals = 0
    for i in range(n):
        for at in range(int(out['attempt'][i]) + 1):
            t = at * n + i
            k = int(tr['len'][t])
            if k == 0:
                continue
            assert k < cap
            x0 = np.concatenate((b['q0'][sel[i]].reshape(-1), tau0[i])) if at == 0 else \
                np.concatenate((b['rq'][sel[i], at - 1].reshape(-1), rtau))
            r = c_oracle.lbfgsb_replay(x0, tr['x'][t, :k], tr['f'][t, :k], tr['g'][t, :k], tr['costs'][t, :k], tr['status'][t, :k])
            assert r['first_bad'] == -1 and r['used'] == k, (int(sel[i]), at, r['first_bad'], k)
            if at == out['attempt'][i] and out['runs'][i] > 0 and r['status'] < 4:
                assert np.array_equal(r['x'], out['x'][i]) and r['status'] == out['status'][i], (int(sel[i]), at)
            attempts += 1; evals += k
    return attempts, evals


@pytest.mark.parametrize('grouped', [1, 0])
@pytest.mark.parametrize('M,tile', [(3, 8), (3, 32), (4, 16), (6, 32)])
def test_optimize_mixed_geometry(M, tile, grouped, geos, problems, sm_count):
    """k_optimize (5 attempts) over all maps in one launch, through neo_optimize and neo_optimize_dev: every record bit
    for bit equal to single-map handles planning only their map's problems, the device records equal to the host ones;
    64 problems per map replayed through the checker's optimizer; agreement with the checker's own plans printed."""
    B, bound, trips = batch_for(sm_count, tile)
    b = plan_inputs(problems, M, B, seed=100 * M + tile)
    env = dict(NEO_TILE=tile, NEO_GROUPED=grouped)
    h = mixed_handle(geos, **env)
    rec = h.optimize(M, b['q0'], b['ts0'], b['head'], b['tail'], b['ids'], b['rq'], b['rts'], 5)
    for s in slots_for(M):
        sel = np.nonzero(b['ids'] == s)[0]
        one = single_handle(geos[s], **env)
        r1 = one.optimize(M, b['q0'][sel], b['ts0'][sel], b['head'][sel], b['tail'][sel], None, b['rq'][sel], b['rts'], 5)
        one.close()
        assert_same_records(r1, sub(rec, sel), f'slot {s} alone')
    d = optimize_dev(h, M, b)
    assert_same_records(d, rec, 'neo_optimize_dev')
    rng = np.random.default_rng(M + tile)
    sample = np.sort(np.concatenate([rng.choice(np.nonzero(b['ids'] == s)[0], 64, replace=False) for s in slots_for(M)]))
    attempts, evals = replay(h, M, b, rec, sample)
    h.close()
    ref = c_oracle.plan_batch_mt(c_oracle.Params.from_config(CFG), [g.omap for g in geos], M, b['head'][sample],
                                 b['tail'][sample], b['q0'][sample], b['ts0'][sample], b['rq'][sample], b['rts'], 5,
                                 map_ids=b['ids'][sample])
    agree = (ref['ok'] == rec['ok'][sample]) & (np.max(np.abs(ref['coeffs'] - rec['coeffs'][sample]).reshape(sample.size, -1), axis=1) <= 1e-4)
    print(f'\n[B.3] M={M}, {tile} lanes, grouped={grouped}: B={B} = 3 x {bound} + 5 (>= {trips} problems per tile) over '
          f'{len(slots_for(M))} maps; ok {rec["ok"].mean():.4f}; single-map handles and neo_optimize_dev identical; '
          f'{attempts} attempts / {evals} evaluations of {sample.size} problems replayed bit for bit; '
          f'checker plans agree on {agree.mean():.4f} of them')


# ------------------------------------------------------------------------------------------------------- B.4 k_astar
ASTAR_SLOTS = (0, 2, 4, 5, 6)


def astar_inputs(geos, problems):
    """24 start/target pairs per map of ASTAR_SLOTS (3 m apart on slot 6's grid, which is mostly off the map), plus
    starts off slot 6's enlarged grid."""
    starts, targets, ids = [], [], []
    for s in ASTAR_SLOTS:
        if s == SMALL:
            g = geos[s]
            rng = np.random.default_rng(9)
            lo = g.org - astar_ref.EXPAND / 2
            hi = lo + np.array([g.W + int(astar_ref.EXPAND / g.res), g.H + int(astar_ref.EXPAND / g.res)]) * g.res
            p0 = lo + rng.uniform(0.05, 0.95, (24, 2)) * (hi - lo)
            th = rng.uniform(0, 2 * np.pi, 24)
            p1 = np.clip(p0 + 3.0 * np.stack([np.cos(th), np.sin(th)], 1), lo + 0.01, hi - 0.01)
            p0[:4] = [lo - 1.0, hi + 0.5, [lo[0] - 0.3, hi[1] - 1.0], [hi[0] + 2.0, lo[1] + 1.0]]     # off the grid
        else:
            hd, tl = problems.pool(s, 3)
            p0, p1 = hd[:24, 0], tl[:24, 0]
        starts.append(p0); targets.append(p1); ids.append(np.full(24, s, np.int32))
    order = np.random.default_rng(4).permutation(24 * len(ASTAR_SLOTS))
    return np.concatenate(starts)[order], np.concatenate(targets)[order], np.concatenate(ids)[order]


def assert_same_searches(a, b, what):
    """k_astar outputs bit for bit; of `path` the rows before path_len (the rest are not written, include/neoopt.h)."""
    for k in ('status', 'path_len', 'closed', 'pruned'):
        assert same_bits(a[k], b[k]), (what, k)
    for i, n in enumerate(np.minimum(a['path_len'], a['path'].shape[1])):
        assert same_bits(a['path'][i, :n], b['path'][i, :n]), (what, 'path', i)


def astar_oracle(geos, start, target, ids):
    refs = []
    for i in range(start.shape[0]):
        g = geos[ids[i]]
        grid = astar_ref.SearchGrid(g.grid())
        sx, sy = grid.cell_of(*start[i])
        if not (0 <= sx < grid.W and 0 <= sy < grid.H):
            refs.append(None)
            continue
        path, found, nclosed = astar_ref.astar(g.grid(), start[i], target[i])
        four, _, _ = astar_ref.prune(g.grid(), path)
        refs.append((path, found, nclosed, four))
    return refs


def test_astar_mixed_grids(geos, problems):
    """k_astar over five maps whose enlarged grids differ in size (the 1200 x 1200 map sizes the per-warp scratch) in one
    launch, with the default first-pass lists and with NEO_ASTAR_ICAP = 64 (the second pass, on lists as long as the
    largest grid): status, path, key nodes and expansion counts equal to oracle/astar_ref.py and to single-map handles,
    and a second identical launch gives the same results (the scratch is left clean across grids of different size)."""
    start, target, ids = astar_inputs(geos, problems)
    refs = astar_oracle(geos, start, target, ids)
    max_path = 4096
    results = {}
    for icap in (None, 64):
        h = mixed_handle(geos, NEO_ASTAR_ICAP=icap)
        out = h.astar(start, target, ids, max_path=max_path)
        again = h.astar(start, target, ids, max_path=max_path)
        h.close()
        assert_same_searches(again, out, ('again', icap))
        for i, r in enumerate(refs):
            if r is None:
                assert out['status'][i] == lib.ASTAR_START_OUTSIDE and out['path_len'][i] == 0, i
                continue
            path, found, nclosed, four = r
            assert out['status'][i] == (lib.ASTAR_FOUND if found else lib.ASTAR_EXHAUSTED), (i, ids[i])
            assert out['path_len'][i] == len(path) <= max_path and out['closed'][i] == nclosed, (i, ids[i])
            assert np.array_equal(out['path'][i, :len(path)], np.array(path)), (i, ids[i])
            assert np.array_equal(out['pruned'][i], np.array(four)), (i, ids[i])
        for s in ASTAR_SLOTS:
            sel = np.nonzero(ids == s)[0]
            one = single_handle(geos[s], NEO_ASTAR_ICAP=icap)
            o1 = one.astar(start[sel], target[sel], None, max_path=max_path)
            one.close()
            assert_same_searches(o1, {k: v[sel] for k, v in out.items()}, (icap, s))
        results[icap] = out
    second = results[64]['closed'] > 64
    assert second.sum() >= 20, second.sum()                                      # these searches took the second pass
    assert all(second[ids == s].any() for s in (0, 2, 4, 5))
    assert_same_searches(results[64], results[None], 'second pass')
    st = results[None]['status']
    print(f'\n[B.4] A*: {ids.size} searches over slots {ASTAR_SLOTS} in one launch ({int((st == lib.ASTAR_FOUND).sum())} found, '
          f'{int((st == lib.ASTAR_EXHAUSTED).sum())} exhausted, {int((st == lib.ASTAR_START_OUTSIDE).sum())} starts off the '
          f'grid); equal to astar_ref and single-map handles; with NEO_ASTAR_ICAP=64 {int(second.sum())} searches took the '
          f'second pass (max closed {int(results[64]["closed"].max())}); repeated launches identical')


# ---------------------------------------------------------------------------------------------- B.5 slot lifecycle
def lifecycle_steps(geos):
    g2, g4 = geos[2], geos[4]
    small = pillar_occ(24, 31, 0.2, 3, 11)
    return [
        ('300x300 occupancy', Geo(0, 300, 300, 0.1, 0.0, -15.0, 'occ', geos[0].occ)),
        ('173x411 ESDF', Geo(0, 173, 411, 0.05, 2.0, -4.0, 'esdf', g2.occ)),
        ('411x173 occupancy', Geo(0, 411, 173, 0.07, 3.3, -2.2, 'occ', g4.occ)),
        ('411x173 at half the resolution', Geo(0, 411, 173, 0.035, 3.3, -2.2, 'occ', g4.occ)),
        ('24x31 occupancy', Geo(0, 24, 31, 0.2, 5.0, -3.0, 'occ', small)),
    ]


def test_slot_lifecycle(geos, problems):
    """One slot re-uploaded through a sequence of shapes (new allocation, same cell count with a new W, a larger A* grid,
    back to a small map): after each upload get_map, get_occupancy, query_map, eval, optimize and astar equal a fresh
    handle holding that map, bit for bit."""
    M, B = 3, 64
    b = problems.batch(M, B, seed=8)
    b['head'][:, 0] = problems.pool(0, M)[0][:B, 0]; b['tail'][:, 0] = problems.pool(0, M)[1][:B, 0]
    q0, ts0 = guesses.straight_line_guess(CFG, b['head'], b['tail'], M)
    rq, rts = guesses.retry_guesses(CFG, b['head'], b['tail'], M, 4, rng=np.random.default_rng(3))
    rng = np.random.default_rng(12)
    h = new_handle(1, NEO_TILE=32)
    x = np.concatenate([q0.reshape(B, -1), h.T2tau(ts0)[0]], axis=1)
    for what, g in lifecycle_steps(geos):
        upload(h, 0, g)
        f = single_handle(g, NEO_TILE=32)
        pts = adversarial_points(g, rng)
        assert all(same_bits(u, v) for u, v in zip(h.get_map(0, g.H, g.W), f.get_map(0, g.H, g.W))), what
        assert all(same_bits(u, v) for u, v in zip(h.get_map(0, g.H, g.W), (g.omap.esdf, g.omap.gx, g.omap.gy))), what
        if g.kind == 'esdf':
            with pytest.raises(lib.NeoError, match='no occupancy'):
                h.get_occupancy(0, g.H, g.W)
        else:
            assert same_bits(h.get_occupancy(0, g.H, g.W), f.get_occupancy(0, g.H, g.W)), what
        assert all(same_bits(u, v) for u, v in zip(h.query_map(0, pts), f.query_map(0, pts))), what
        e1, e2 = h.eval(M, x, b['head'], b['tail'], want_coeffs=True), f.eval(M, x, b['head'], b['tail'], want_coeffs=True)
        for k in ('costs', 'grad', 'status', 'coeffs', 'ts'):
            assert same_bits(e1[k], e2[k]), (what, k)
        assert_same_records(h.optimize(M, q0, ts0, b['head'], b['tail'], None, rq, rts, 5),
                            f.optimize(M, q0, ts0, b['head'], b['tail'], None, rq, rts, 5), what)
        s1 = h.astar(b['head'][:16, 0], b['tail'][:16, 0], max_path=1024, max_closed=20000)
        s2 = f.astar(b['head'][:16, 0], b['tail'][:16, 0], max_path=1024, max_closed=20000)
        assert_same_searches(s1, s2, what)
        f.close()
    h.close()
    print(f'\n[B.5] one slot through {len(lifecycle_steps(geos))} uploads: maps, lookups, {B} evaluations, {B} plans and '
          f'16 searches equal to a fresh handle after each')


# ----------------------------------------------------------------------------------------------- B.6 Python drop-ins
def growing_esdfs():
    """ESDF objects as octomap_server's projected map grows: make_world(0), the same origin with 30 more rows and 60
    more columns, then 20 columns and 10 rows prepended (the origin moves by -2 m, -1 m)."""
    w = make_world(0)
    grids = [(w.occ, w.ox, w.oy)]
    g1 = np.zeros((w.H + 30, w.W + 60), np.int8); g1[:w.H, :w.W] = w.occ
    grids.append((g1, w.ox, w.oy))
    g2 = np.zeros((g1.shape[0] + 10, g1.shape[1] + 20), np.int8); g2[10:, 20:] = g1
    grids.append((g2, w.ox - 2.0, w.oy - 1.0))
    out = []
    for occ, ox, oy in grids:
        e = ESDF()
        e.occupancy_map_cb(World(0, occ.shape[0], occ.shape[1], w.res, ox, oy, occ, w.pillars).occupancy_msg())
        out.append(e)
    return out


def plan_result(p, esdf, head, tail, seed):
    np.random.seed(seed)
    it, runs = p.iter_num, p.opt_running_times
    try:
        p.plan(esdf, head, tail)
        err = None
    except Exception as ex:
        err = str(ex)
    out = {k: np.asarray(getattr(p, k, np.nan)) for k in ('int_wpts', 'ts', 'coeffs', 'costs')}
    return dict(out, err=err, nit=p.iter_num - it, runs=p.opt_running_times - runs)


def test_minjerk_planner_on_a_growing_map(monkeypatch, geos):
    """MinJerkPlanner.plan re-uploads slot 0 as the ESDF grows and moves: every plan equals a fresh planner's."""
    monkeypatch.setenv('NEO_TILE', '32')
    esdfs = growing_esdfs()
    w = make_world(0)
    head, tail = make_problems(w, 4, M=3)
    p = MinJerkPlanner(YamlConfig())
    n = 0
    for k, e in enumerate(esdfs):
        for i in range(4):
            seed = 10 * k + i
            got = plan_result(p, e, head[i], tail[i], seed)
            want = plan_result(MinJerkPlanner(YamlConfig()), e, head[i], tail[i], seed)
            assert got['err'] == want['err'], (k, i)
            for key in ('int_wpts', 'ts', 'coeffs', 'costs'):
                assert same_bits(got[key], want[key]), (k, i, key)
            assert (got['nit'], got['runs']) == (want['nit'], want['runs']), (k, i)
            n += 1
    print(f'\n[B.6] MinJerkPlanner: {n} plans over {len(esdfs)} growing ESDFs '
          f'({" -> ".join(f"{e.map_height}x{e.map_width}" for e in esdfs)}) equal to fresh planners')


class FixedNoise:
    """Stands in for a np.random.Generator: returns a given array from normal()."""

    def __init__(self, a):
        self.a = a

    def normal(self, loc, scale, size):
        assert tuple(size) == self.a.shape
        return self.a


def test_batch_planner_mixed_slots(monkeypatch, geos, problems):
    """BatchPlanner.plan and plan_dev with map_ids over the eight slots equal per-map BatchPlanners (same retry noise)."""
    import torch
    monkeypatch.setenv('NEO_TILE', '32')
    M, B = 3, 512
    b = problems.batch(M, B, seed=21)
    noise = np.random.default_rng(22).normal(0, 0.5, (B, 4, M - 1, 2))
    bp = BatchPlanner(YamlConfig(), max_maps=N_SLOTS)
    for g in geos:
        upload(bp.handle, g.slot, g)
    host = bp.plan(b['head'], b['tail'], b['ids'], rng=np.random.default_rng(22))
    dev = bp.plan_dev(b['head'], b['tail'], b['ids'], noise=torch.from_numpy(noise).cuda())
    torch.cuda.synchronize()
    dev = {k: (None if v is None else v.cpu().numpy()) for k, v in dev.items()}
    assert_same_records(dev, host, 'plan_dev')
    for g in geos:
        sel = np.nonzero(b['ids'] == g.slot)[0]
        one = BatchPlanner(YamlConfig(), max_maps=1)
        upload(one.handle, 0, g)
        r1 = one.plan(b['head'][sel], b['tail'][sel], rng=FixedNoise(noise[sel]))
        d1 = one.plan_dev(b['head'][sel], b['tail'][sel], noise=torch.from_numpy(noise[sel]).cuda())
        torch.cuda.synchronize()
        assert_same_records(r1, sub(host, sel), f'plan, slot {g.slot}')
        assert_same_records({k: (None if v is None else v.cpu().numpy()) for k, v in d1.items()}, sub(dev, sel),
                            f'plan_dev, slot {g.slot}')
        one.handle.close()
    bp.handle.close()
    print(f'\n[B.6] BatchPlanner: plan and plan_dev of {B} problems over {N_SLOTS} slots equal to per-map planners; '
          f'ok {host["ok"].mean():.3f}')
