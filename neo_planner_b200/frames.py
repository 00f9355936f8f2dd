"""Body/world frame transforms and the network I/O layout of the reference (record_planner.py:13-72,
nn_planner.py:104-134), batched in NumPy. The reference uses pyquaternion objects (`.rotate`, `.inverse`,
`.rotation_matrix`); here the unit-quaternion algebra is restated on arrays (w, x, y, z order). Pinned in
tests/test_host_logic.py against tests/golden/nn_io.npz -- the outputs of the reference's own form_nn_input /
form_nn_output / get_wpts_world, run unmodified by oracle/gen_golden.py with a stand-in for pyquaternion (not
installed here) -- to 1e-13, and against scipy.spatial.transform.Rotation."""
from __future__ import annotations

import numpy as np


def rotation_matrix(q):
    """(..., 4) unit quaternions (w, x, y, z) -> (..., 3, 3), pyquaternion.Quaternion.rotation_matrix."""
    q = np.asarray(q, dtype=np.float64)
    q = q / np.linalg.norm(q, axis=-1, keepdims=True)
    w, x, y, z = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    R = np.empty(q.shape[:-1] + (3, 3))
    R[..., 0, 0] = 1 - 2 * (y * y + z * z); R[..., 0, 1] = 2 * (x * y - z * w); R[..., 0, 2] = 2 * (x * z + y * w)
    R[..., 1, 0] = 2 * (x * y + z * w); R[..., 1, 1] = 1 - 2 * (x * x + z * z); R[..., 1, 2] = 2 * (y * z - x * w)
    R[..., 2, 0] = 2 * (x * z - y * w); R[..., 2, 1] = 2 * (y * z + x * w); R[..., 2, 2] = 1 - 2 * (x * x + y * y)
    return R


def rotate(q, v):
    """Quaternion.rotate(v): world <- body for an attitude quaternion."""
    return np.einsum('...ij,...j->...i', rotation_matrix(q), np.asarray(v, dtype=np.float64))


def rotate_inverse(q, v):
    """Quaternion.inverse.rotate(v): body <- world."""
    return np.einsum('...ji,...j->...i', rotation_matrix(q), np.asarray(v, dtype=np.float64))


def normalize_depth(depth_img):
    """record_planner.py:15: (depth / max(depth) * 255).astype(uint8) per image."""
    depth_img = np.asarray(depth_img)
    B = depth_img.shape[0]
    mx = depth_img.reshape(B, -1).max(axis=1).reshape(B, 1, 1)
    return (depth_img / mx * 255).astype(np.uint8)


def motion_info(local_vel, attitude, global_pos, global_vel, des_pos_z, init_pos, init_vel, target_state):
    """record_planner.py:17-48 for a batch: (B,24) =
    [local_vel 3 | R 9 row-major | init pos 3 | init vel 3 | target pos 3 | target vel 3] (body frame)."""
    attitude = np.asarray(attitude, dtype=np.float64)
    B = attitude.shape[0]
    R = rotation_matrix(attitude)
    p0 = np.zeros((B, 3)); v0 = np.zeros((B, 3))
    p0[:, :2] = np.asarray(init_pos)[:, :2]; p0[:, 2] = des_pos_z
    v0[:, :2] = np.asarray(init_vel)[:, :2]
    tp = np.zeros((B, 3)); tv = np.zeros((B, 3))
    target_state = np.asarray(target_state, dtype=np.float64)
    tp[:, :2] = target_state[:, 0, :]; tp[:, 2] = des_pos_z
    tv[:, :2] = target_state[:, 1, :]
    gp = np.asarray(global_pos, dtype=np.float64); gv = np.asarray(global_vel, dtype=np.float64)
    return np.concatenate([np.asarray(local_vel, dtype=np.float64), R.reshape(B, 9),
                           rotate_inverse(attitude, p0 - gp), rotate_inverse(attitude, v0 - gv),
                           rotate_inverse(attitude, tp - gp), rotate_inverse(attitude, tv - gv)], axis=1)


def form_nn_input(depth_img, local_vel, attitude, global_pos, global_vel, des_pos_z, init_pos, init_vel, target_state):
    """record_planner.py:13-58 for a batch.
    depth_img (B,H,W) float/uint; local_vel, global_pos, global_vel (B,3); attitude (B,4) wxyz;
    init_pos/init_vel (B,>=2) planning start in the map frame; target_state (B,2,2) = [pos; vel].
    Returns depth_norm (B,H,W) uint8 and motion_info (B,24)."""
    return normalize_depth(depth_img), motion_info(local_vel, attitude, global_pos, global_vel, des_pos_z, init_pos,
                                                   init_vel, target_state)


def form_nn_output(attitude, global_pos, des_pos_z, int_wpts):
    """record_planner.py:61-72: int_wpts (B,2,K) in the map frame -> (B,3K) body-frame waypoints, waypoint-major."""
    int_wpts = np.asarray(int_wpts, dtype=np.float64)
    B, _, K = int_wpts.shape
    w3 = np.concatenate([np.transpose(int_wpts, (0, 2, 1)), np.full((B, K, 1), float(des_pos_z))], axis=2)     # (B,K,3)
    local = rotate_inverse(np.asarray(attitude)[:, None, :], w3 - np.asarray(global_pos, dtype=np.float64)[:, None, :])
    return local.reshape(B, 3 * K)


def wpts_world(attitude, global_pos, net_out, M=3):
    """nn_planner.py:104-134: network output (B, 3(M-1)+M) -> int_wpts (B,2,M-1) in the map frame, ts (B,M)."""
    net_out = np.asarray(net_out, dtype=np.float64)
    B = net_out.shape[0]
    local = net_out[:, :3 * (M - 1)].reshape(B, M - 1, 3)
    world = rotate(np.asarray(attitude)[:, None, :], local) + np.asarray(global_pos, dtype=np.float64)[:, None, :]
    return np.ascontiguousarray(np.transpose(world[:, :, :2], (0, 2, 1))), net_out[:, 3 * (M - 1):].copy()


def quat_array(attitude):
    """(w, x, y, z) from what the reference passes as `drone_state.attitude`: a pyquaternion.Quaternion (`.q` /
    `.elements`), or already an array."""
    for attr in ('q', 'elements'):
        v = getattr(attitude, attr, None)
        if v is not None:
            return np.asarray(v, dtype=np.float64)
    return np.asarray(attitude, dtype=np.float64)


def clamp_durations(ts, T_min, T_max, margin=1e-3):
    """SURVEY.md §8d (config 3): network durations outside (T_min, T_max) make map_T2tau raise on entry (EP:209), so the
    reference throws the whole guess away and retries from a noisy straight line. clamp_durations moves them just
    inside the interval instead (and reports which samples it touched) so that the predicted WAYPOINTS still warm-start
    the optimizer. Returns (ts_clamped, touched (B,) bool)."""
    ts = np.asarray(ts, dtype=np.float64)
    lo, hi = T_min + margin * (T_max - T_min), T_max - margin * (T_max - T_min)
    out = np.clip(np.where(np.isfinite(ts), ts, lo), lo, hi)
    return out, np.any(out != ts, axis=-1)


# ---- the same transforms on CUDA tensors (float64), bit-identical to the NumPy functions above -----------------------
# Every product and sum is its own elementwise operation (no fused multiply-add) and the sums run in NumPy 2.x's order
# for these shapes: np.linalg.norm over 4 components adds them left to right, and einsum('...ij,...j->...i') with a
# broadcast (B,1,3,3) matrix forms (R[i,0] v0 + R[i,2] v2) + R[i,1] v1. tests/test_frames_dev_order.py pins both.
def rotation_matrix_dev(q):
    """rotation_matrix for a (..., 4) float64 tensor."""
    s = q * q
    q = q / (((s[..., 0:1] + s[..., 1:2]) + s[..., 2:3]) + s[..., 3:4]).sqrt()
    w, x, y, z = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    rows = [[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
            [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
            [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]]
    import torch
    return torch.stack([torch.stack(r, dim=-1) for r in rows], dim=-2)


def rotate_dev(q, v):
    """rotate for tensors: q (..., 4), v (..., 3) broadcast against it."""
    R = rotation_matrix_dev(q)
    p = [R[..., :, j] * v[..., None, j] for j in range(3)]
    return (p[0] + p[2]) + p[1]


def wpts_world_dev(attitude, global_pos, net_out, M=3):
    """wpts_world on the device: attitude (B,4), global_pos (B,3), net_out (B, 3(M-1)+M) float64 CUDA tensors ->
    int_wpts (B,2,M-1), ts (B,M), both contiguous."""
    B = net_out.shape[0]
    local = net_out[:, :3 * (M - 1)].reshape(B, M - 1, 3)
    world = rotate_dev(attitude[:, None, :], local) + global_pos[:, None, :]
    return world[:, :, :2].transpose(1, 2).contiguous(), net_out[:, 3 * (M - 1):].contiguous()


def clamp_durations_dev(ts, T_min, T_max, margin=1e-3):
    """clamp_durations for a float64 tensor: (ts_clamped, touched (B,) bool)."""
    lo, hi = T_min + margin * (T_max - T_min), T_max - margin * (T_max - T_min)
    out = ts.where(ts.isfinite(), ts.new_tensor(lo)).clamp(lo, hi)
    return out, (out != ts).any(dim=-1)
