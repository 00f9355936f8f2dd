"""Learned-initializer pipeline, device-resident against the host path: 4,096 depth frames -> CNN -> warm_start_plan ->
60 Hz setpoints (get_full_state_cmd).

    python scripts/gpu_device_pipeline.py [--frames 4096] [--reps 5] [--out DIR]

* host path: NeoBatchPlanner.enhanced_traj_plan (network output copied to the host, waypoint transform and guesses in
  NumPy, neo_optimize through its pinned staging) and BatchPlanner.get_full_state_cmd (neo_sample, twice);
* device path: enhanced_traj_plan_dev and get_full_state_cmd_dev (everything stays on the GPU).

Both start from the same depth frames, already in device memory as uint8, and the same retry noise. The two paths
alternate in one process and each repetition is timed with CUDA events on the current stream, ending in a synchronise.
The host synchronisations each path makes are counted as the synchronising torch operations (torch's sync debug mode)
plus the libneoopt host-pointer calls (each ends in a stream synchronise). The card's name and power limit are printed
with the times. One JSON line on stdout (and DIR/device_pipeline.json with --out)."""
import argparse
import json
import os
import subprocess
import sys
import warnings

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from neo_planner_b200 import frames, lib
from neo_planner_b200.initializer import NeoBatchPlanner
from neo_planner_b200.planner import BatchPlanner
from neo_planner_b200.worlds import YamlConfig, make_problems, make_world

HZ = 60


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ''
    return q or torch.cuda.get_device_name(0)


class HostSyncs:
    """Counts libneoopt host-pointer calls, each of which synchronises its stream before returning."""

    def __init__(self):
        self.n = 0
        for name, calls in (('optimize', 1), ('sample', 2), ('get_coeffs', 1), ('eval', 1)):
            self._wrap(name, calls)

    def _wrap(self, name, calls):
        f = getattr(lib.Handle, name)

        def counted(h, *a, **k):
            self.n += calls
            return f(h, *a, **k)
        setattr(lib.Handle, name, counted)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=4096)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    B = args.frames
    rng = np.random.default_rng(0)
    cfg = YamlConfig()
    w = make_world(0)
    head, tail = make_problems(w, B)
    yaw = np.arctan2(head[:, 1, 1], head[:, 1, 0])
    att = np.stack([np.cos(yaw / 2), np.zeros(B), np.zeros(B), np.sin(yaw / 2)], axis=1)
    gp = np.concatenate([head[:, 0] - 0.5 * head[:, 1], np.full((B, 1), 2.0)], axis=1)
    gv = np.concatenate([head[:, 1], np.zeros((B, 1))], axis=1)
    lv = frames.rotate_inverse(att, gv)
    init_pos = np.concatenate([head[:, 0], np.full((B, 1), 2.0)], axis=1)
    depth = torch.from_numpy(rng.integers(1, 256, size=(B, 480, 640), dtype=np.uint8)).cuda()
    noise_np = rng.normal(0, 0.5, (B, 4, 2, 2))
    noise = torch.from_numpy(noise_np).cuda()
    syncs = HostSyncs()

    bp = BatchPlanner(cfg)
    bp.set_map(w)
    neo = NeoBatchPlanner(bp, des_pos_z=2.0, device='cuda', dtype=torch.bfloat16, clamp_ts=True)

    def host():
        res = neo.enhanced_traj_plan(depth, lv, att, gp, gv, init_pos, gv, tail, rng=np.random.default_rng(1))
        states, count = bp.get_full_state_cmd(res['coeffs'], res['ts'], HZ)
        return res, states, count

    def device():
        res = neo.enhanced_traj_plan_dev(depth, lv, att, gp, gv, init_pos, gv, tail, noise=noise)
        states, count = bp.get_full_state_cmd_dev(res['coeffs'], res['ts'], HZ)
        return res, states, count

    def run(fn):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        return out, a.elapsed_time(b)

    def count_syncs(fn):
        torch.cuda.synchronize()
        before = syncs.n
        torch.cuda.set_sync_debug_mode('warn')
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter('always')
            fn()
        torch.cuda.set_sync_debug_mode('default')
        torch.cuda.synchronize()
        return dict(torch=sum('synchroniz' in str(c.message) for c in caught), libneoopt=syncs.n - before)

    (rh, sh, ch), _ = run(host)                # warm-up: cuDNN algorithm choice, buffers grown
    (rd, sd, cd), _ = run(device)
    # same results (the host path draws its retry noise from default_rng(1): check the device path with that noise)
    nd = torch.from_numpy(np.random.default_rng(1).normal(0, 0.5, (B, 4, 2, 2))).cuda()
    rd1 = neo.enhanced_traj_plan_dev(depth, lv, att, gp, gv, init_pos, gv, tail, noise=nd)
    sd1, cd1 = bp.get_full_state_cmd_dev(rd1['coeffs'], rd1['ts'], HZ)
    differ = [k for k in ('x', 'ts', 'coeffs', 'costs', 'status', 'ok', 'attempt', 'nit', 'runs', 'nfev', 'work',
                          'nn_int_wpts', 'nn_ts', 'nn_ts_outside_bounds')
              if not np.array_equal(np.asarray(rh[k])[:, :3] if k == 'work' else np.asarray(rh[k]),
                                    (rd1[k][:, :3] if k == 'work' else rd1[k]).cpu().numpy(), equal_nan=k != 'nn_ts_outside_bounds')]
    if not np.array_equal(ch, cd1.cpu().numpy()) or not np.array_equal(sh, sd1[:, :sh.shape[1]].cpu().numpy()):
        differ.append('setpoints')
    motion = frames.motion_info(lv, att, gp, gv, 2.0, init_pos, gv, tail)
    dn = neo.normalize_depth(depth)
    repeatable = bool(torch.equal(neo.predict_dev(dn, motion), neo.predict_dev(dn, motion)))
    times = {'host': [], 'device': []}
    for _ in range(args.reps):
        times['host'].append(run(host)[1])
        times['device'].append(run(device)[1])
    line = {'pipeline': f'{B} depth frames -> PlannerNetConv (bf16) -> warm_start_plan (<= 5 attempts) -> {HZ} Hz setpoints',
            'card': card(), 'reps': args.reps,
            'host_path_ms': times['host'], 'device_path_ms': times['device'],
            'host_path_median_ms': float(np.median(times['host'])), 'device_path_median_ms': float(np.median(times['device'])),
            'host_syncs': {'host_path': count_syncs(host), 'device_path': count_syncs(device)},
            'fields_differing_from_host_path': differ, 'network_output_repeatable': repeatable,
            'ok_fraction': float(rh['ok'].mean())}
    print(json.dumps(line))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'device_pipeline.json'), 'w') as f:
            json.dump(line, f, indent=1)


if __name__ == '__main__':
    main()
