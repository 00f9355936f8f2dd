"""bench.py --dump-outputs: the packed result records of the timed path written back as one float64 array per field, in
global problem order, and a fixed seeded sample of problems when the records exceed the size budget."""
import os

import numpy as np

import bench
from neo_planner_b200 import sharding


def packed(rng, ws, B, M):
    """ws rank blocks of B problems each, every field filled with distinct values through the packed layout."""
    n = 3 * M - 2
    raw = np.zeros((ws, sharding.packed_record_bytes(B, M)), np.uint8)
    off = sharding.packed_record_offsets(B, M)
    want = {}
    for r in range(ws):
        f = dict(x=rng.normal(size=(B, n)), ts=rng.uniform(1, 4, size=(B, M)), coeffs=rng.normal(size=(B, 6 * M, 2)),
                 costs=rng.normal(size=(B, 4)))
        for k in sharding.INT_FIELDS:
            f[k] = rng.integers(-5, 500, size=B).astype(np.int32)
        for k, a in f.items():
            b = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
            raw[r, off[k]:off[k] + b.size] = b
            want.setdefault(k, []).append(a)
    return raw.reshape(-1), {k: np.concatenate(v) for k, v in want.items()}


def test_dump_writes_every_field_in_global_order(tmp_path):
    B, M, ws = 37, 3, 2
    raw, want = packed(np.random.default_rng(0), ws, B, M)
    bench.dump_outputs(str(tmp_path), raw, B, M)
    assert sorted(os.listdir(tmp_path)) == sorted(k + '.npy' for k in want)
    for k, a in want.items():
        got = np.load(tmp_path / (k + '.npy'))
        assert got.dtype == np.float64 and np.array_equal(got, a.astype(np.float64)), k


def test_dump_samples_the_same_problems_above_the_budget(tmp_path, monkeypatch):
    B, M = 500, 4
    raw, want = packed(np.random.default_rng(1), 1, B, M)
    monkeypatch.setattr(bench, 'DUMP_BUDGET', 64_000)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), raw, B, M)
    total = sum(os.path.getsize(tmp_path / 'a' / f) for f in os.listdir(tmp_path / 'a'))
    assert 60_000 < total <= 64_000
    idx = np.load(tmp_path / 'a' / 'problem_index.npy').astype(np.int64)
    assert 0 < len(idx) < B and np.all(np.diff(idx) > 0)
    assert np.array_equal(idx, np.load(tmp_path / 'b' / 'problem_index.npy'))
    for k, a in want.items():
        assert np.array_equal(np.load(tmp_path / 'a' / (k + '.npy')), a[idx].astype(np.float64)), k
