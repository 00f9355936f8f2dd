"""The NumPy summation orders that frames.wpts_world_dev restates (NeoBatchPlanner.enhanced_traj_plan_dev): a NumPy
release that sums np.linalg.norm or einsum('...ij,...j->...i') differently fails here first, without a GPU. Also
clamp_durations_dev against clamp_durations on CPU tensors. wpts_world_dev itself is compared on the GPU
(tests/test_gpu_device_api.py): torch's CPU sqrt is not correctly rounded, CUDA's double sqrt is."""
import numpy as np
import torch

from neo_planner_b200 import frames


def inputs(B, seed=0):
    rng = np.random.default_rng(seed)
    att = rng.normal(size=(B, 4))
    pos = rng.normal(size=(B, 3)) * 30.0
    net = np.concatenate([rng.normal(size=(B, 6)) * 5.0, rng.uniform(-1.0, 25.0, size=(B, 3))], axis=1)
    net[::97, 7] = np.nan
    net[::89, 6] = np.inf
    return att, pos, net


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def test_numpy_summation_order():
    """The orders frames.*_dev restate, as NumPy computes them for these shapes."""
    rng = np.random.default_rng(1)
    q = rng.normal(size=(200_000, 1, 4))
    s = q * q
    assert same_bits(np.linalg.norm(q, axis=-1, keepdims=True)[..., 0], np.sqrt(((s[..., 0] + s[..., 1]) + s[..., 2]) + s[..., 3]))
    R = frames.rotation_matrix(q)
    v = rng.normal(size=(200_000, 2, 3)) * 10.0
    p = [R[..., :, j] * v[..., None, j] for j in range(3)]
    assert same_bits(np.einsum('...ij,...j->...i', R, v), (p[0] + p[2]) + p[1])
    assert not same_bits(np.einsum('...ij,...j->...i', R, v), (p[0] + p[1]) + p[2])     # the order is not the obvious one


def test_clamp_durations_dev_bits():
    _, _, net = inputs(100_000, seed=2)
    ts = net[:, 6:]
    for T_min, T_max in [(2.0, 20.0), (0.5, 5.0)]:
        out, touched = frames.clamp_durations(ts, T_min, T_max)
        outd, touchedd = frames.clamp_durations_dev(torch.from_numpy(ts), T_min, T_max)
        assert same_bits(out, outd.numpy()) and np.array_equal(touched, touchedd.numpy())
