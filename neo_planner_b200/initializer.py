"""Learned initializer of NEO-Planner (SURVEY.md §8 a24 / §8f-4): depth image + 24 motion floats -> 2 body-frame
waypoints + 3 durations, which warm-start the MINCO optimizer (neo_planner.py:42-51).

The network is the one dense contraction on the path, so it stays PyTorch (cuDNN/cuBLAS convs, bf16 autocast on the
GPU) as north_star prescribes; no custom kernel. Architecture restated from nn_trainer.py:109-155 (`PlannerNet`,
MLP heads) and nn_trainer_conv.py:108-160 (`PlannerNetConv`, Conv1d heads -- the variant that is saved as
saved_net/planner_net.*, which nn_planner.py:25 loads). The reference's trained weights are not in the repository
(.MISSING_LARGE_BLOBS) and torchvision's ImageNet weights cannot be downloaded here, so weights are seeded random:
throughput and plumbing are real, the paper's iteration savings are not reproducible from this repo alone."""
from __future__ import annotations

import numpy as np
import torch
from torch import nn

from . import frames
from .planner import MinJerkPlanner, TrajUtils

IMG_WIDTH, IMG_HEIGHT, MOTION_INPUT_SIZE, OUTPUT_SIZE = 640, 480, 24, 9
IMG_FEATURE_SIZE = MOTION_FEATURE_SIZE = 24


def _backbone():
    from torchvision import models
    net = models.resnet18(weights=None)
    net.conv1 = nn.Conv2d(1, 64, kernel_size=7, stride=2, padding=3, bias=False)      # 1-channel depth input
    net.fc = nn.Linear(net.fc.in_features, IMG_FEATURE_SIZE)
    return net


class PlannerNet(nn.Module):
    """nn_trainer.py:109-155."""

    def __init__(self):
        super().__init__()
        self.img_backbone = _backbone()
        self.motion_backbone = nn.Sequential(nn.Linear(MOTION_INPUT_SIZE, 48), nn.LeakyReLU(), nn.Linear(48, 24),
                                             nn.LeakyReLU(), nn.Linear(24, 24), nn.LeakyReLU(),
                                             nn.Linear(24, MOTION_FEATURE_SIZE))
        self.mlp = nn.Sequential(nn.Linear(IMG_FEATURE_SIZE + MOTION_FEATURE_SIZE, 48), nn.LeakyReLU(), nn.Linear(48, 96),
                                 nn.LeakyReLU(), nn.Linear(96, 96), nn.LeakyReLU(), nn.Linear(96, OUTPUT_SIZE))

    def forward(self, x):
        img = x[:, :IMG_WIDTH * IMG_HEIGHT].reshape(-1, 1, IMG_HEIGHT, IMG_WIDTH)
        vec = x[:, IMG_WIDTH * IMG_HEIGHT:]
        return self.mlp(torch.cat([self.img_backbone(img), self.motion_backbone(vec)], dim=1))


class PlannerNetConv(nn.Module):
    """nn_trainer_conv.py:108-160."""

    def __init__(self):
        super().__init__()
        self.img_backbone = _backbone()

        def head(width, out):
            return nn.Sequential(nn.Conv1d(1, 16, 3, 1, 1), nn.LeakyReLU(), nn.Conv1d(16, 32, 3, 1, 1), nn.LeakyReLU(),
                                 nn.Conv1d(32, 64, 3, 1, 1), nn.LeakyReLU(), nn.Flatten(), nn.Linear(64 * width, out))
        self.motion_backbone = head(MOTION_INPUT_SIZE, MOTION_FEATURE_SIZE)
        self.mlp = head(IMG_FEATURE_SIZE + MOTION_FEATURE_SIZE, OUTPUT_SIZE)

    def forward(self, x):
        img = x[:, :IMG_WIDTH * IMG_HEIGHT].reshape(-1, 1, IMG_HEIGHT, IMG_WIDTH)
        vec = x[:, IMG_WIDTH * IMG_HEIGHT:].unsqueeze(1)
        feat = torch.cat([self.img_backbone(img), self.motion_backbone(vec)], dim=1)
        return self.mlp(feat.unsqueeze(1))


def process_input(depth_norm, motion_info):
    """nn_trainer.py:51-58 for a batch: (B,H,W) uint8 + (B,24) -> (B, 307224) float32."""
    B = depth_norm.shape[0]
    return np.concatenate([depth_norm.reshape(B, -1).astype(np.float32), np.asarray(motion_info).astype(np.float32)], axis=1)


class NeoBatchPlanner:
    """NeoPlanner.enhanced_traj_plan (neo_planner.py:42-51) for B samples: network guess -> warm_start_plan.

    `planner` is a planner.BatchPlanner. Network guesses with durations outside (T_min, T_max) lose their first
    attempt exactly as in the reference (map_T2tau raises, EP:209 -> re-seeded straight line, EP:197-200)."""

    def __init__(self, planner, des_pos_z=2.0, net=None, device='cuda', dtype=torch.bfloat16, seed=42, clamp_ts=False):
        self.planner, self.des_pos_z, self.device, self.dtype = planner, des_pos_z, torch.device(device), dtype
        self.clamp_ts = clamp_ts      # True: keep the predicted waypoints when a predicted duration is out of range
        if net is None:
            torch.manual_seed(seed)
            net = PlannerNetConv()
        self.net = net.to(self.device).eval()
        if self.device.type == 'cuda':
            self.net = self.net.to(memory_format=torch.channels_last)
            torch.backends.cudnn.benchmark = True        # fixed 480x640 frames: let cuDNN pick its fastest kernels once

    @torch.no_grad()
    def normalize_depth(self, depth_img, chunk=512):
        """record_planner.py:15 on the device: (depth / max(depth) * 255).astype(uint8), evaluated in fp64 like NumPy
        does, so the truncation to uint8 is the reference's. depth_img: (B,H,W) array (any real dtype) or tensor. Returns
        a uint8 CUDA tensor (B,H,W)."""
        if not torch.is_tensor(depth_img):
            depth_img = np.asarray(depth_img)
        out = torch.empty(tuple(depth_img.shape), dtype=torch.uint8, device=self.device)
        for i in range(0, len(depth_img), chunk):
            d = depth_img[i:i + chunk]
            d = (d if torch.is_tensor(d) else torch.from_numpy(np.ascontiguousarray(d))).to(self.device, non_blocking=True).double()
            mx = d.amax(dim=(1, 2), keepdim=True)
            out[i:i + chunk] = (d / mx * 255).to(torch.uint8)
        return out

    @torch.no_grad()
    def predict(self, depth_norm, motion_info, chunk=512):
        """Network forward for B samples. depth_norm: (B,H,W) uint8, NumPy or CUDA tensor (images travel as uint8 and
        are widened on the device; the flattened float vector of nn_trainer.py:51-58 is formed there). Returns (B,9)."""
        return self.predict_dev(depth_norm, motion_info, chunk).cpu().numpy()

    @torch.no_grad()
    def predict_dev(self, depth_norm, motion_info, chunk=512):
        """predict, leaving the (B,9) float64 output on the device."""
        if not torch.is_tensor(depth_norm):
            depth_norm = torch.from_numpy(np.ascontiguousarray(depth_norm))
        motion = torch.from_numpy(np.asarray(motion_info, dtype=np.float32)).to(self.device, non_blocking=True)
        B = depth_norm.shape[0]
        outs = []
        for i in range(0, B, chunk):
            img = depth_norm[i:i + chunk].to(self.device, non_blocking=True).reshape(-1, IMG_WIDTH * IMG_HEIGHT)
            with torch.autocast(self.device.type, dtype=self.dtype, enabled=self.device.type == 'cuda'):
                lowp = self.dtype if self.device.type == 'cuda' else torch.float32      # 0..255 is exact in bf16
                x = torch.cat([img.to(lowp), motion[i:i + chunk].to(lowp)], dim=1)
                outs.append(self.net(x).float())
        return torch.cat(outs).double()

    def enhanced_traj_plan(self, depth_img, local_vel, attitude, global_pos, global_vel, init_pos, init_vel, target_state,
                           map_ids=None, rng=None):
        motion = frames.motion_info(local_vel, attitude, global_pos, global_vel, self.des_pos_z, init_pos, init_vel,
                                    target_state)
        out = self.predict(self.normalize_depth(depth_img), motion)
        int_wpts, ts = frames.wpts_world(attitude, global_pos, out, M=3)
        cfg = self.planner.cfg
        outside = ~np.all((ts > cfg.T_min) & (ts < cfg.T_max), axis=1)
        ts_used = frames.clamp_durations(ts, cfg.T_min, cfg.T_max)[0] if self.clamp_ts else ts
        head = np.stack([np.asarray(init_pos)[:, :2], np.asarray(init_vel)[:, :2]], axis=1)
        res = self.planner.warm_start_plan(head, target_state, int_wpts, ts_used, map_ids, rng)
        res['nn_int_wpts'], res['nn_ts'], res['nn_ts_outside_bounds'] = int_wpts, ts, outside
        return res

    def enhanced_traj_plan_dev(self, depth_img, local_vel, attitude, global_pos, global_vel, init_pos, init_vel,
                               target_state, map_ids=None, noise=None, generator=None):
        """enhanced_traj_plan with the network output kept on the device: the waypoint transform, the duration clamp,
        the initial guesses and the optimizer all run there, and nothing waits for the GPU. depth_img may be a CUDA
        tensor; the per-sample states are host arrays (they also form the motion vector). Retry noise as in
        BatchPlanner.warm_start_plan_dev (`noise` tensor, else N(0, 0.5) from the torch `generator`, not np.random).
        Returns the keys of enhanced_traj_plan as CUDA tensors, bit-identical to it for the same network and noise."""
        motion = frames.motion_info(local_vel, attitude, global_pos, global_vel, self.des_pos_z, init_pos, init_vel,
                                    target_state)
        out = self.predict_dev(self.normalize_depth(depth_img), motion)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(self.device, non_blocking=True)  # noqa: E731
        int_wpts, ts = frames.wpts_world_dev(up(attitude), up(global_pos), out, M=3)
        cfg = self.planner.cfg
        outside = ~((ts > cfg.T_min) & (ts < cfg.T_max)).all(dim=1)
        ts_used = frames.clamp_durations_dev(ts, cfg.T_min, cfg.T_max)[0] if self.clamp_ts else ts
        head = np.stack([np.asarray(init_pos)[:, :2], np.asarray(init_vel)[:, :2]], axis=1)
        res = self.planner.warm_start_plan_dev(head, target_state, int_wpts, ts_used, map_ids, noise, generator)
        res['nn_int_wpts'], res['nn_ts'], res['nn_ts_outside_bounds'] = int_wpts, ts, outside
        return res


class NNPlanner(TrajUtils):
    """Drop-in for the reference's NNPlanner (nn_planner.py:19-134): one sample per call, same method names and result
    attributes (`int_wpts` (2, M-1) in the map frame, `ts` (M,)). The reference runs an exported ONNX file through
    onnxruntime; here the same network (PlannerNetConv, nn_trainer_conv.py:108-160) runs in PyTorch on the GPU --
    pass `net` with loaded weights (`net.load_state_dict(torch.load('planner_net.pth'))`); without it the weights are
    seeded random, because the reference's trained file is not in its repository."""

    def __init__(self, des_pos_z=2.0, net=None, device=None, dtype=torch.bfloat16, seed=42):
        super().__init__()
        self.device = torch.device(device or ('cuda' if torch.cuda.is_available() else 'cpu'))
        self.dtype = dtype
        if net is None:
            torch.manual_seed(seed)
            net = PlannerNetConv()
        self.net = net.to(self.device).eval()
        self.init_planning_params(des_pos_z)

    def init_planning_params(self, des_pos_z):          # nn_planner.py:60-68
        self.M, self.s, self.D, self.nn_output_D = 3, 3, 2, 3
        self.head_state = np.zeros((self.s, self.D))
        self.tail_state = np.zeros((self.s, self.D))
        self.des_pos_z = des_pos_z

    def nn_traj_plan(self, depth_img, drone_state, plan_init_state, target_state):      # nn_planner.py:70-82
        q = frames.quat_array(drone_state.attitude)
        target_state = np.asarray(target_state, dtype=np.float64)
        depth_norm, motion = frames.form_nn_input(np.asarray(depth_img)[None], np.asarray(drone_state.local_vel)[None], q[None],
                                                  np.asarray(drone_state.global_pos)[None], np.asarray(drone_state.global_vel)[None],
                                                  self.des_pos_z, np.asarray(plan_init_state.global_pos)[None],
                                                  np.asarray(plan_init_state.global_vel)[None], target_state[None, :2, :2])
        self.drone_state = drone_state
        self.head_state[0, :self.D] = plan_init_state.global_pos[:2]
        self.head_state[1, :self.D] = plan_init_state.global_vel[:2]
        self.tail_state[0, :self.D] = target_state[0, :2]
        self.tail_state[1, :self.D] = target_state[1, :2]
        self.onnx_predict(depth_norm[0], motion[0])

    @torch.no_grad()
    def onnx_predict(self, depth_image_norm, motion_info):                             # nn_planner.py:87-111
        x = torch.from_numpy(process_input(np.asarray(depth_image_norm)[None], np.asarray(motion_info)[None])).to(self.device)
        with torch.autocast(self.device.type, dtype=self.dtype, enabled=self.device.type == 'cuda'):
            output = self.net(x).float().reshape(1, -1).double().cpu().numpy()
        k = self.nn_output_D * (self.M - 1)
        int_wpts_local = output[0][:k].reshape(self.M - 1, self.nn_output_D).T
        self.ts = output[0][k:]
        self.int_wpts = self.get_wpts_world(int_wpts_local)[:self.D, :]

    def get_wpts_world(self, int_wpts):                                                # nn_planner.py:123-134
        q = frames.quat_array(self.drone_state.attitude)
        return (frames.rotate(q[None], np.asarray(int_wpts, dtype=np.float64).T) + np.asarray(self.drone_state.global_pos)).T


class NeoPlanner(MinJerkPlanner):
    """Drop-in for the reference's NeoPlanner (neo_planner.py:10-51; `selected_planner:=neo`, the shipped default):
    network guess -> warm_start_plan on the device, one problem per call. clamp_ts=True keeps the predicted waypoints
    when a predicted duration falls outside (T_min, T_max) (frames.clamp_durations); False is the reference: map_T2tau
    raises and the first retry starts from a noisy straight line (EP:197-200)."""

    def __init__(self, planner_config, device: int = 0, net=None, clamp_ts=False, dtype=torch.bfloat16):
        super().__init__(planner_config, device)
        self.nn_planner = NNPlanner(planner_config.des_pos_z, net=net, dtype=dtype,
                                    device=f'cuda:{device}' if torch.cuda.is_available() else 'cpu')
        self.clamp_ts = clamp_ts

    def enhanced_traj_plan(self, map, depth_img, drone_state, plan_init_state, target_state):
        self.nn_planner.nn_traj_plan(depth_img, drone_state, plan_init_state, target_state)
        int_wpts, ts = self.nn_planner.int_wpts, self.nn_planner.ts
        if self.clamp_ts:
            ts = frames.clamp_durations(ts[None], self.T_min, self.T_max)[0][0]
        drone_state_2d = np.array([plan_init_state.global_pos[:2], plan_init_state.global_vel[:2]])
        self.warm_start_plan(map, drone_state_2d, target_state, int_wpts, ts)           # 2D planning, z is fixed
