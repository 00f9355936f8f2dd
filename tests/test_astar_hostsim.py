"""CPU check of the geometric initializer's device source (csrc/astar_warp.cuh): devtools/astar_host.cu compiles the very
same search/pruning code with a single lane for the host, and this test runs it against the reference's golden paths
(tests/golden/geo_M3.npz). It covers the arithmetic and control flow of the kernel in the GPU-less container; the 32-lane
execution is covered by tests/test_gpu_geo.py. The host build is a test aid only -- the library never loads it."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from neo_planner_b200.build import nvcc_path
from neo_planner_b200.worlds import make_world
from oracle import minco_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, 'devtools', 'astar_host.cu')
SO = os.path.join(ROOT, 'devtools', '_astar_host.so')


@pytest.fixture(scope='module')
def sim():
    deps = [SRC, os.path.join(ROOT, 'neo_planner_b200', 'csrc', 'astar_warp.cuh')]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        nvcc = shutil.which(nvcc_path())
        if nvcc is None:
            pytest.skip('nvcc not available to build the host simulation')
        subprocess.run([nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-O2', '-std=c++17', '-shared', '-Xcompiler',
                        '-fPIC', '-o', SO, SRC], check=True, cwd=ROOT)
    lib = ctypes.CDLL(SO)
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int32)

    def run(gm, start, target, max_path=512, max_closed=0, open_fast=512):
        start = np.ascontiguousarray(start, dtype=np.float64).reshape(-1, 2)
        target = np.ascontiguousarray(target, dtype=np.float64).reshape(-1, 2)
        B = start.shape[0]
        esdf = np.ascontiguousarray(gm.esdf, dtype=np.float64)
        out = dict(path=np.zeros((B, max_path, 2)), path_len=np.zeros(B, np.int32), pruned=np.zeros((B, 4, 2)),
                   status=np.zeros(B, np.int32), closed=np.zeros(B, np.int32))
        rc = lib.sim_astar(gm.H, gm.W, ctypes.c_double(gm.res), ctypes.c_double(gm.ox), ctypes.c_double(gm.oy),
                           esdf.ctypes.data_as(dp), B, start.ctypes.data_as(dp), target.ctypes.data_as(dp), max_closed, max_path, open_fast,
                           out['path'].ctypes.data_as(dp), out['path_len'].ctypes.data_as(ip), out['pruned'].ctypes.data_as(dp),
                           out['status'].ctypes.data_as(ip), out['closed'].ctypes.data_as(ip))
        assert rc == 0, 'search scratch was not restored'
        return out
    return run


@pytest.fixture(params=[None, 40], ids=['lists-fit', 'second-pass'])
def insert_cap(request, monkeypatch):
    """None: the insertion list / open-list spill hold the whole grid. 40: most searches outgrow the first pass's lists and
    are re-run by the second pass, as k_astar does with its ASTAR_INSERT_CAP (results must not depend on it)."""
    if request.param is None:
        monkeypatch.delenv('NEO_ASTAR_ICAP', raising=False)
    else:
        monkeypatch.setenv('NEO_ASTAR_ICAP', str(request.param))
    return request.param


def test_kernel_source_on_host_matches_reference_paths(golden, sim, insert_cap):
    g = golden('geo_M3.npz')
    off = np.concatenate(([0], np.cumsum(g['path_len'])))
    for wid, dn in sorted(set(zip(g['world_id'].tolist(), g['dense'].tolist()))):
        sel = np.nonzero((g['world_id'] == wid) & (g['dense'] == dn))[0]
        w = make_world(wid, dense=bool(dn))
        gm = minco_ref.GridMap(w.occ, w.H, w.W, w.res, w.ox, w.oy)
        for open_fast in (512, 5):           # 5: nearly the whole open list lives in the spill area
            out = sim(gm, g['head'][sel, 0], g['tail'][sel, 0], open_fast=open_fast)
            assert np.all(out['status'] == 0) and np.array_equal(out['path_len'], g['path_len'][sel])
            assert np.array_equal(out['pruned'], g['pruned'][sel])
            for j, i in enumerate(sel):
                assert np.array_equal(out['path'][j, :g['path_len'][i]], g['path'][off[i]:off[i + 1]]), (wid, i)


def test_kernel_source_on_host_edge_cases(golden, sim, insert_cap):
    g = golden('geo_M3.npz')
    gm = minco_ref.GridMap(g['tiny_occ'], 12, 16, 1.0, 0.0, 0.0)
    out = sim(gm, [[2.5, 2.5]], [[10.5, 6.5]], open_fast=16)
    assert out['status'][0] == 1 and out['closed'][0] == int(g['lost_closed'])
    assert np.array_equal(out['path'][0, :1], g['lost_path']) and np.array_equal(out['pruned'][0], g['lost_pruned'])
    out = sim(gm, [[2.5, 2.5], [-20.0, 0.0], [2.5, 2.5]], [[2.6, 2.7], [3.0, 3.0], [10.5, 6.5]], max_closed=10)
    assert out['status'].tolist() == [0, 2, 3] and out['path_len'].tolist() == [1, 0, 0]


def test_kernel_source_on_host_random_maps(sim):
    """Property test (hypothesis): random small maps with random obstacles, resolutions and origins, start/target anywhere
    on or around the map (blocked, unreachable and out-of-grid cases included): the device source run on the host and
    the checker agree on status, path, pruned key nodes and expansion count."""
    from hypothesis import given, settings, strategies as st, HealthCheck
    from oracle import astar_ref

    @settings(max_examples=60, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)
    @given(st.integers(4, 14), st.integers(4, 14), st.sampled_from([0.5, 1.0, 2.0, 0.25]), st.floats(-3, 3), st.floats(-3, 3),
           st.floats(0.0, 0.35), st.integers(0, 10 ** 6))
    def run(H, W, res, ox, oy, density, seed):
        rng = np.random.default_rng(seed)
        occ = np.where(rng.random((H, W)) < density, 100, 0).astype(np.int8)
        gm = minco_ref.GridMap(occ, H, W, res, ox, oy)
        lo = np.array([ox - 6.0, oy - 6.0]); hi = np.array([ox + W * res + 6.0, oy + H * res + 6.0])
        start = rng.uniform(lo, hi, size=(3, 2)); target = rng.uniform(lo, hi, size=(3, 2))
        out = sim(gm, start, target, max_path=2048, open_fast=int(rng.choice([3, 64, 512])))
        grid = astar_ref.SearchGrid(gm)
        for i in range(3):
            sx, sy = grid.cell_of(start[i, 0], start[i, 1])
            if not (0 <= sx < grid.W and 0 <= sy < grid.H):
                assert out['status'][i] == 2 and out['path_len'][i] == 0      # rejected up front (reference: index aliasing)
                continue
            path, found, nclosed = astar_ref.astar(gm, start[i], target[i])
            four, _, _ = astar_ref.prune(gm, path)
            assert out['status'][i] == (0 if found else 1) and out['closed'][i] == nclosed
            assert out['path_len'][i] == len(path) and np.array_equal(out['path'][i, :len(path)], np.array(path))
            assert np.array_equal(out['pruned'][i], np.array(four))
    run()
