#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 MINCO trajectory optimizer (see DESIGN.md §6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c4|c2|c5] [--no-extras]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one pass of the hot path (warm_start_plan semantics: straight-line expert guess, up to 5 L-BFGS-B
attempts, EP:62-80 / EP:186-237) over one batch of synthetic problems. Workloads:
  c4 (default; BASELINE.json configs[3] = the batch north_star quotes the metric on): 65,536 start-goal pairs = 256
     generated worlds x 256 pairs, M = 3, planner_config.yaml parameters. With N ranks the WORLDS are sharded over the
     ranks (strong scaling: the job stays 65,536 problems) and every step ends with ONE NCCL all-gather of the packed
     result records.
  c2 (configs[1]): 1,024 pairs on one shared map per rank (weak scaling).   c5 (configs[4]): 16,384 pairs per rank,
     M = 10, 1200x1200 @0.05 m map.
At N = 1 the line also carries, under "extras", the other configurations measured the same way (c2, c5), the fused
cost+gradient evaluation rate (k_eval, the second half of BASELINE.json's metric) and the latency of ONE plan through the
drop-in MinJerkPlanner.plan (the reference node's call, NODE:490-525), each with its own roofline / CPU figure.
Prints ONE JSON line (rank 0).
--dump-outputs DIR writes the result records of the last timed step as DIR/<field>.npy (see dump_outputs), so that two
builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from neo_planner_b200.worlds import make_world, make_problems, YamlConfig  # noqa: E402
from neo_planner_b200 import guesses  # noqa: E402

METRIC = 'optimized trajectories/sec to convergence'
UNIT = 'traj/s'


def workload(name, rank, world_size=1):
    """Seeded problem set of one rank. Returns dict(worlds, cfg, M, head, tail, map_ids, q0, ts0, retry_q, retry_ts).
    c2: 1,024 problems on one world per rank (weak scaling). c5: 16,384 problems, M = 10, 1200x1200 @0.05 m map per rank.
    c4: 65,536 problems = 256 worlds x 256 pairs in total, worlds sharded over the ranks (strong scaling)."""
    from neo_planner_b200 import sharding
    cfg = YamlConfig()
    if name == 'c5':
        M, per_world, dense, world_ids = 10, 16384, True, [rank]
    elif name == 'c4':
        M, per_world, dense, world_ids = 3, 256, False, sharding.shard_worlds(256, world_size, rank)
    else:
        M, per_world, dense, world_ids = 3, 1024, False, [rank]
    cfg.init_wpts_num = M - 1
    worlds, heads, tails, ids = [], [], [], []
    for slot, wid in enumerate(world_ids):
        w = make_world(wid, dense=dense)
        a, b = make_problems(w, per_world, M=M)
        worlds.append(w); heads.append(a); tails.append(b); ids.append(np.full(per_world, slot, np.int32))
    head, tail, map_ids = np.concatenate(heads), np.concatenate(tails), np.concatenate(ids)
    q0, ts0 = guesses.straight_line_guess(cfg, head, tail, M)
    rq, rts = guesses.retry_guesses(cfg, head, tail, M, 4, rng=np.random.default_rng(77_000 + rank))
    return dict(name=name, world=worlds[0], worlds=worlds, cfg=cfg, M=M, B=len(head), head=head, tail=tail,
                map_ids=map_ids if len(worlds) > 1 else None, q0=q0, ts0=ts0, retry_q=rq, retry_ts=rts,
                scaling='strong' if name == 'c4' else 'weak')


def describe(wl, n_gpus):
    w = wl['world']
    cfgidx = {'c2': 1, 'c4': 3, 'c5': 4}[wl['name']]
    maps = f"{len(wl['worlds'])} {w.H}x{w.W} @{w.res} m random-pillar map(s) per GPU"
    total = f"{wl['B'] * n_gpus} start-goal pairs in total ({wl['B']} per GPU) " if wl['scaling'] == 'strong' else f"{wl['B']} start-goal pairs per GPU "
    return {'workload': total + f"on {maps}, M={wl['M']} pieces, expert straight-line init, "
                        f"warm_start_plan semantics (<=5 attempts), planner_config.yaml parameters (BASELINE.json configs[{cfgidx}])",
            'problems_per_gpu': wl['B'], 'pieces': wl['M'], 'map': f'{w.H}x{w.W}@{w.res}', 'maps_per_gpu': len(wl['worlds']),
            'max_attempts': 5,
            'sharding': f'{n_gpus} rank(s), worlds sharded over ranks, NCCL all-gather of result records' if n_gpus > 1 else 'single GPU',
            'l2': 'flushed between timed steps (256 MiB write)'}


# ------------------------------------------------------------------------------------------------ CPU arms
_W = {}


def cpu_sample_workload(name):
    """The CPU arms time a bounded sample: the problems of the first world of the workload."""
    return workload(name, 0, 256 if name == 'c4' else 1)


def _pool_init(name, rank):
    import warnings
    warnings.filterwarnings('ignore')
    from oracle import minco_ref
    wl = cpu_sample_workload(name)
    w = wl['world']
    _W['wl'] = wl
    _W['grid'] = minco_ref.GridMap(w.occ, w.H, w.W, w.res, w.ox, w.oy)
    _W['opt'] = minco_ref.RefOptimizer(wl['cfg'])


def _pool_plan(k):
    """One reference-equivalent plan() (Python/NumPy + scipy L-BFGS-B, oracle/minco_ref.py) for problem k."""
    wl, opt = _W['wl'], _W['opt']
    np.random.seed(1_000 + k)
    n0, f0 = opt.iter_num, opt.nfev
    try:
        opt.plan(_W['grid'], wl['head'][k], wl['tail'][k])
        ok = 1
    except Exception:
        ok = 0
    return ok, opt.nfev - f0


def cpu_reference_run(name, steps, warmup, per_step=None):
    """Times the reference's own algorithm (Python + scipy, all host cores) on bounded samples of the workload:
    per_step plans per step (>= 128), the value is total plans / total time; the median step is reported beside it."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    per_step = per_step or max(128, 4 * cores)
    ctx = mp.get_context('fork')
    with ctx.Pool(cores, initializer=_pool_init, initargs=(name, 0)) as pool:
        B = {'c2': 1024, 'c4': 256, 'c5': 16384}[name]
        k0 = 0
        for _ in range(warmup):
            pool.map(_pool_plan, [(k0 + i) % B for i in range(per_step)], chunksize=1)
            k0 += per_step
        oks = evals = 0
        step_s = []
        t0 = time.perf_counter()
        for _ in range(steps):
            t1 = time.perf_counter()
            r = pool.map(_pool_plan, [(k0 + i) % B for i in range(per_step)], chunksize=1)
            step_s.append(time.perf_counter() - t1)
            k0 += per_step
            oks += sum(a for a, _ in r); evals += sum(b for _, b in r)
        dt = time.perf_counter() - t0
    n = per_step * steps
    return dict(value=n / dt, seconds=dt, cores=cores, problems=n, ok=oks, evals_per_s=evals / dt, per_step=per_step,
                median_step_value=per_step / float(np.median(step_s)))


def c_port_run(wl, count=256, threads=1):
    """Plain-C port (oracle/minco_oracle.c) on the first `count` problems of the workload, on `threads` host threads
    -- the stricter CPU yardstick (the reference itself is Python)."""
    from oracle import c_oracle
    maps = [c_oracle.OracleMap.from_world(w) for w in wl['worlds'][:max(1, (count + 255) // 256)]] if wl['map_ids'] is not None \
        else [c_oracle.OracleMap.from_world(wl['world'])]
    p = c_oracle.Params.from_config(wl['cfg'])
    sl = slice(0, count)
    ids = None if wl['map_ids'] is None else wl['map_ids'][sl]
    t0 = time.perf_counter()
    out = c_oracle.plan_batch_mt(p, maps, wl['M'], wl['head'][sl], wl['tail'][sl], wl['q0'][sl], wl['ts0'][sl], wl['retry_q'][sl],
                                 wl['retry_ts'], 5, map_ids=ids, threads=threads)
    dt = time.perf_counter() - t0
    return dict(value=count / dt, unit=UNIT, cores=threads, kind='port-c', sample=f'first {count} problems, {threads} thread(s)',
                ok=int(out['ok'].sum()), evals_per_s=float(out['nfev'].sum()) / dt)


def ncu_traffic(name):
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_optimize launch from the committed `ncu --set full` capture
    (profiles/ncu_k_optimize.json), or None when no capture exists for this workload."""
    try:
        d = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_k_optimize.json')))
        return d[name]['dram_bytes_read'] + d[name]['dram_bytes_write']
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8): 'hw_slowdown',
                 getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40): 'hw_thermal_slowdown',
                 getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20): 'sw_thermal_slowdown',
                 getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4): 'sw_power_cap'}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.dev, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.dev)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.dev)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.01)

    def result(self):
        self.stop_flag = True
        if self.is_alive():
            self.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {'sm_mhz': med, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons), 'samples': len(self.samples)}


# ------------------------------------------------------------------------------------------------ device arm
def flop_count(M, evals, work):
    """SURVEY.md §8d: F = 1280 M per evaluation + 50 per sample + 65 per velocity-violating + 56 per colliding sample."""
    return 1280.0 * M * evals + 50.0 * work[0] + 65.0 * work[1] + 56.0 * work[2]


class DeviceRun:
    """One workload resident on one GPU: maps uploaded, inputs in HBM, result record buffer, launch closure."""

    def __init__(self, wl, local_rank, dev, torch, lib, C):
        self.wl, self.torch, self.lib = wl, torch, lib
        cfg, M, B = wl['cfg'], wl['M'], wl['B']
        self.M, self.B = M, B
        n, nq = 3 * M - 2, 2 * (M - 1)
        self.n = n
        self.h = h = lib.Handle(cfg, local_rank, len(wl['worlds']))
        ws = wl['worlds']
        t0 = time.perf_counter()                                                               # device EDT build, all maps
        h.set_maps_occupancy(np.arange(len(ws)), ws[0].H, ws[0].W, ws[0].res, [w_.ox for w_ in ws], [w_.oy for w_ in ws],
                             np.stack([np.asarray(w_.occ).reshape(w_.H, w_.W) for w_ in ws]))
        self.map_build_s = time.perf_counter() - t0
        self.ids_d = None if wl['map_ids'] is None else torch.from_numpy(wl['map_ids']).to(dev)
        tau0, st0 = h.T2tau(wl['ts0'])
        rtau, rst = h.T2tau(wl['retry_ts'])
        assert not st0.any() and not rst.any()
        self.x0 = torch.from_numpy(np.concatenate([wl['q0'].reshape(B, nq), tau0], axis=1)).to(dev)
        self.head = torch.from_numpy(lib.pad_state(wl['head'])).to(dev)
        self.tail = torch.from_numpy(lib.pad_state(wl['tail'])).to(dev)
        self.rq = torch.from_numpy(wl['retry_q'].reshape(B, -1)).to(dev)
        self.rtau = torch.from_numpy(rtau).to(dev)
        # ONE packed result record buffer per rank (bytes): [x | ts | coeffs | costs] doubles, then
        # [status ok attempt nit runs nfev] int32 -- gathered with one collective
        self.rec_d = n + M + 12 * M + 4
        self.nbytes = B * self.rec_d * 8 + B * 6 * 4
        self.out = torch.zeros(self.nbytes, dtype=torch.uint8, device=dev)
        self.work = torch.zeros(B * 4, dtype=torch.int64, device=dev)
        base = self.out.data_ptr()
        off = np.cumsum([0, B * n, B * M, B * 12 * M]) * 8
        res = lib.Result()
        res.x, res.ts, res.coeffs, res.costs = (base + int(o) for o in off)
        ibase = base + B * self.rec_d * 8
        res.status, res.ok, res.attempt, res.nit, res.runs, res.nfev = (ibase + 4 * B * i for i in range(6))
        res.work = self.work.data_ptr()
        self.res, self.C = res, C

    def ints(self):
        return self.out[self.B * self.rec_d * 8:].view(self.torch.int32).view(6, self.B)

    def launch(self):
        st = self.torch.cuda.current_stream().cuda_stream
        assert st != 0
        h = self.h
        h._ck(h.lib.neo_optimize_dev(h.h, self.B, self.M, self.x0.data_ptr(), None, self.head.data_ptr(), self.tail.data_ptr(),
                                     None if self.ids_d is None else self.ids_d.data_ptr(), self.rq.data_ptr(),
                                     self.rtau.data_ptr(), 0, 5, self.C.byref(self.res), self.C.c_void_p(st)))

    def accounting(self):
        ints = self.ints()
        evals = float(ints[5].double().sum().item())
        wk = [float(v) for v in self.work.view(self.B, 4).double().sum(0).tolist()]
        return dict(ok_fraction=float(ints[1].float().mean().item()), evals=evals, work=wk,
                    flops=flop_count(self.M, evals, wk), l2_bytes=8.0 * wk[0] + 16.0 * wk[2])


def timed_steps(torch, dist, run, K, W, flush, distributed, all_bytes):
    """W warm-up + K timed steps (CUDA events on the launching stream, L2 flushed outside the bracket). Returns the
    per-rank sum of the K step times in ms."""
    def step():
        run.launch()
        if distributed:
            dist.all_gather_into_tensor(all_bytes, run.out)
    for _ in range(W):
        flush.zero_()
        step()
    torch.cuda.synchronize()
    if distributed:
        dist.barrier()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for a, b in evs:
        flush.zero_()
        a.record()
        step()
        b.record()
    torch.cuda.synchronize()
    if distributed:
        dist.barrier()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


DUMP_BUDGET = 64_000_000
NPY_HEADER = 128


def dump_outputs(path, raw, B, M):
    """Writes what a caller of the timed path receives -- x, ts, coeffs, costs and the int32 fields status, ok, attempt,
    nit, runs, nfev -- from the packed record buffer(s) `raw` (one block of B problems per rank, global order) as
    path/<field>.npy in float64 (exact for the int32 fields). Above DUMP_BUDGET bytes in all, a fixed seeded sample of
    problems is written instead, with its problem indices as path/problem_index.npy."""
    from neo_planner_b200 import sharding
    f = sharding.split_packed_records(raw.reshape(-1, sharding.packed_record_bytes(B, M)), B, M)
    f = {k: v.reshape((-1,) + v.shape[2:]) for k, v in f.items()}
    total = f['x'].shape[0]
    per_problem = 8 * sum(v[0].size for v in f.values())
    keep = np.arange(total)
    if total * per_problem + NPY_HEADER * len(f) > DUMP_BUDGET:
        rows = (DUMP_BUDGET - NPY_HEADER * (len(f) + 1)) // (per_problem + 8)
        keep = np.sort(np.random.default_rng(0).choice(total, rows, replace=False))
        f['problem_index'] = keep
    os.makedirs(path, exist_ok=True)
    for k, v in f.items():
        np.save(os.path.join(path, k + '.npy'), np.asarray(v if k == 'problem_index' else v[keep], dtype=np.float64))


def roofline_of(acc, M, step_ms, fp64_peak, hbm_peak, peaks_found, hbm_bytes, name):
    ach = acc['flops'] / (step_ms * 1e-3) / 1e12
    return {'bound': 'fp64', 'kernel': 'k_optimize', 'achieved': ach, 'peak': fp64_peak, 'unit': 'TFLOP/s', 'frac': ach / fp64_peak,
            'traffic': ncu_traffic(name),
            'peak_source': 'measured in this run (neo_fp64_peak DFMA microbenchmark; MEASURED_PEAKS.json has no fp64 figure)',
            'flops_per_launch': acc['flops'], 'l2_gather_bytes_per_launch': acc['l2_bytes'],
            'l2_gather_GBps': acc['l2_bytes'] / (step_ms * 1e-3) / 1e9,
            'hbm': {'bound': 'hbm', 'achieved': hbm_bytes / (step_ms * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                    'frac': hbm_bytes / (step_ms * 1e-3) / 1e9 / hbm_peak, 'algorithmic_bytes_per_launch': hbm_bytes,
                    'peak_source': 'MEASURED_PEAKS.json' if peaks_found else 'fallback'}}


def hbm_bytes_of(wl):
    M, B, n, w = wl['M'], wl['B'], 3 * wl['M'] - 2, wl['world']
    return B * (8 * n + 96 + 8 * (12 * M + M + 4) + 12) + len(wl['worlds']) * w.H * w.W * 32


def e2e_run(torch, dist, run, wl, lib, Ke, distributed, world_size, dev):
    """The same step through the host-buffer C ABI call (neo_optimize: H2D + kernel + D2H inside), and -- with several
    ranks -- the gather of the packed records, as ShardedPlanner does it. Wall clock, max over ranks."""
    from neo_planner_b200 import sharding
    h, M, B = run.h, wl['M'], wl['B']
    out_host = lib.Handle.alloc_result(B, M)
    hp, tp = lib.pad_state(wl['head']), lib.pad_state(wl['tail'])

    shard = sharding.DeviceShard(h, M, B, world_size, dev, 5) if distributed else None

    def step():
        if distributed:     # host inputs -> HBM, kernel, ONE all-gather on the device, ONE D2H of the gathered batch on every rank
            shard.plan(wl['q0'], wl['ts0'], hp, tp, wl['map_ids'], wl['retry_q'], wl['retry_ts'])
        else:
            h.optimize(M, wl['q0'], wl['ts0'], hp, tp, wl['map_ids'], wl['retry_q'], wl['retry_ts'], 5, out=out_host)
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    if distributed:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        step()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if distributed:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out_host = {k: v[dist.get_rank()] for k, v in shard.views().items()}      # this rank's block of the gathered batch
    return out_host, float(t.item())


def eval_rate(torch, run, wl, K, W, flush):
    """Fused cost+gradient evaluations per second (k_eval through neo_eval_dev) at the expert guess of every problem."""
    h, M, B, n = run.h, wl['M'], wl['B'], run.n
    dev = run.x0.device
    costs = torch.zeros(B * 4, dtype=torch.float64, device=dev); grad = torch.zeros(B * n, dtype=torch.float64, device=dev)
    status = torch.zeros(B, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    l0 = h.launch_count()

    def launch():
        h._ck(h.lib.neo_eval_dev(h.h, B, M, run.x0.data_ptr(), run.head.data_ptr(), run.tail.data_ptr(),
                                 None if run.ids_d is None else run.ids_d.data_ptr(), costs.data_ptr(), grad.data_ptr(),
                                 status.data_ptr(), None, None, run.C.c_void_p(st)))
    for _ in range(W):
        flush.zero_(); launch()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for a, b in evs:
        flush.zero_(); a.record(); launch(); b.record()
    torch.cuda.synchronize()
    ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    ts = wl['ts0']
    S = float(np.floor(ts / wl['cfg'].delta_t + 1e-9).sum())          # samples per launch at the expert guess
    flops = 1280.0 * M * B + 50.0 * S
    return dict(metric='fused cost+gradient evaluations/sec', value=B / (ms * 1e-3), unit='evals/s', ms_per_launch=ms, evaluations_per_launch=B,
                gpu_launches=int(h.launch_count() - l0 - W), flops_per_launch_lower_bound=flops,
                note='flop count without the violation terms (65 S_v + 56 S_c): k_eval does not export them'), flops / (ms * 1e-3) / 1e12


def single_plan_latency(wl, count=200):
    """ONE plan per call through the drop-in class, host buffers, as the reference node calls it (NODE:490-525):
    MinJerkPlanner(config).plan(map, head_state, tail_state) with an ESDF map object."""
    from neo_planner_b200.planner import MinJerkPlanner
    from neo_planner_b200.esdf import ESDF
    w = wl['world']
    e = ESDF()
    e.occupancy_map_cb(w.occupancy_msg())
    pl = MinJerkPlanner(wl['cfg'])
    ms, fails = [], 0
    import contextlib
    import io
    sink = io.StringIO()                    # the drop-in prints the reference's "Re-planning for ..." messages
    for k in range(count + 5):
        np.random.seed(1_000 + k)
        t0 = time.perf_counter()
        try:
            with contextlib.redirect_stdout(sink):
                pl.plan(e, wl['head'][k % wl['B']][:2], wl['tail'][k % wl['B']][:2])
        except Exception:
            fails += 1
        if k >= 5:
            ms.append(1e3 * (time.perf_counter() - t0))
    ms = np.array(ms)
    return dict(metric='latency of one MinJerkPlanner.plan call (host buffers, map resident)', unit='ms', plans=count,
                p50=float(np.percentile(ms, 50)), p90=float(np.percentile(ms, 90)), p99=float(np.percentile(ms, 99)),
                mean=float(ms.mean()), no_solution=fails)


def cpu_single_plan_latency(name, count=24):
    """The reference's algorithm (Python + scipy port), one process, one plan per call: what the node's 30-100 ms are."""
    _pool_init(name, 0)
    ms = []
    for k in range(count):
        t0 = time.perf_counter()
        _pool_plan(k)
        ms.append(1e3 * (time.perf_counter() - t0))
    return dict(p50=float(np.percentile(ms, 50)), p99=float(np.percentile(ms, 99)), plans=count, unit='ms',
                kind='port (oracle/minco_ref.py, one process)')


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='c4', choices=['c2', 'c4', 'c5'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the result records of the last timed step as DIR/<field>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    rank = int(os.environ.get('RANK', '0'))
    world_size = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    K, W = args.steps, max(args.warmup, 3 if args.impl == 'ours' else 0)

    if args.impl == 'reference':
        if rank != 0:
            return 0
        wl = workload(args.workload, 0, max(args.gpus, 1))
        r = cpu_reference_run(args.workload, K, args.warmup)
        sample = (f"{r['per_step']} plans per step x {K} steps (problems of the first world of the same seeded workload, cycled), "
                  f"multiprocessing.Pool({r['cores']}), Python+scipy restatement of the reference (oracle/minco_ref.py; the "
                  f"reference is pure Python, there is nothing to compile)")
        line = {'impl': 'reference', 'metric': METRIC, 'value': r['value'], 'unit': UNIT, 'n_gpus': args.gpus, 'steps': K,
                'warmup': args.warmup, 'ms_per_step': 1e3 * r['seconds'] / K, 'higher_is_better': True, 'scaling': wl['scaling'],
                'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'config': describe(wl, args.gpus),
                'cpu_baseline': {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'port', 'sample': sample,
                                 'evals_per_s': r['evals_per_s'], 'ok_fraction': r['ok'] / r['problems'],
                                 'median_step_value': r['median_step_value']},
                'e2e': {'value': r['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0}
        print(json.dumps(line))
        return 0

    # CPU baselines first (rank 0, N = 1 only): fork the worker pool before CUDA is initialised in this process
    cpu_base = cpu_lat = None
    if world_size == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(args.workload, steps=2, warmup=1)
        wl0 = workload(args.workload, 0, 1)
        cores = os.cpu_count() or 1
        c1 = c_port_run(wl0, 256, 1)
        call = c_port_run(wl0, min(wl0['B'], 8192 if wl0['M'] <= 4 else 1024), cores)
        cpu_base = {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'port',
                    'sample': f"{r['problems']} plans of the same workload (problems of its first world, cycled), Python+scipy "
                              f"restatement of the reference (oracle/minco_ref.py), multiprocessing.Pool({r['cores']})",
                    'evals_per_s': r['evals_per_s'], 'ok_fraction': r['ok'] / r['problems'], 'median_step_value': r['median_step_value'],
                    'c_port_single_thread': c1, 'c_port_all_cores': call,
                    'note': 'the reference is Python; the plain-C port on all cores is the stricter yardstick -- see gpu_vs_c_port_all_cores'}
        if not args.no_extras:
            cpu_lat = cpu_single_plan_latency('c2')

    import torch
    import torch.distributed as dist
    import ctypes as C
    from neo_planner_b200 import lib

    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl ours needs a CUDA device (there is no CPU fallback)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    distributed = world_size > 1
    if distributed:
        dist.init_process_group('nccl', device_id=dev)

    wl = workload(args.workload, rank, world_size)
    run = DeviceRun(wl, local_rank, dev, torch, lib, C)
    fp64_peak = run.h.fp64_peak()
    map_build_s = run.map_build_s
    all_bytes = torch.zeros(world_size * run.nbytes, dtype=torch.uint8, device=dev) if distributed else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.Stream(device=dev)     # a real (non-default) stream: NULL would mean "the handle's own stream"
    torch.cuda.set_stream(stream)

    launches0 = run.h.launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_wall0 = time.perf_counter()
    step_ms_list = timed_steps(torch, dist, run, K, W, flush, distributed, all_bytes)
    t_wall = time.perf_counter() - t_wall0
    # the clock-sampling launches below rewrite run.out: keep the records of the last timed step
    last_step = (all_bytes if distributed else run.out).clone() if args.dump_outputs and rank == 0 else None
    launches = (run.h.launch_count() - launches0) * K // (K + W)        # kernels of this library inside the timed region
    # keep the GPU under the same load a little longer if the timed region was too short to sample clocks.
    # Kernel launches only: the number of extra iterations differs per rank, so no collective may run here.
    t_extra = time.perf_counter()
    while len(sampler.samples) < 20 and time.perf_counter() - t_extra < 2.0:
        run.launch()
        torch.cuda.synchronize()
    clocks = sampler.result()
    tmax = torch.tensor([sum(step_ms_list)], dtype=torch.float64, device=dev)
    if distributed:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms = float(tmax.item())
    B = wl['B']
    value = world_size * B * K / (total_ms * 1e-3)
    step_ms = total_ms / K
    acc = run.accounting()

    # ---- e2e: host buffers through the C ABI, H2D + D2H (+ the gather) inside the timed region ---------------------
    Ke = max(3, min(K, 20))
    out_host, t_e2e = e2e_run(torch, dist, run, wl, lib, Ke, distributed, world_size, dev)
    e2e_value = world_size * B * Ke / t_e2e
    n, nq, M = run.n, 2 * (wl['M'] - 1), wl['M']
    h2d = world_size * (8 * (B * n + 12 * B + B * 4 * nq + M) + (4 * B if wl['map_ids'] is not None else 0))
    d2h = world_size * (8 * B * (n + M + 12 * M + 4) + 4 * B * 6 + 8 * B * 4)
    if distributed:     # every rank copies the whole gathered batch (world_size blocks) to its host
        d2h = world_size * world_size * (8 * B * (n + M + 12 * M + 4) + 4 * B * 6)
    assert np.array_equal(out_host['ok'], run.ints()[1].cpu().numpy())      # both paths computed the same thing

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = peaks.get('hbm_gbs', 6650.0)

    # ---- the other configurations, the evaluation rate and the single-plan latency (N = 1 only) ---------------------
    extras = None
    if world_size == 1 and not args.no_extras:
        extras = {}
        ev, ev_tflops = eval_rate(torch, run, wl, K, W, flush)
        ev['roofline'] = {'bound': 'fp64', 'kernel': 'k_eval', 'achieved': ev_tflops, 'peak': fp64_peak, 'unit': 'TFLOP/s',
                          'frac': ev_tflops / fp64_peak, 'traffic': None}
        ev['config'] = {'workload': f"{B} evaluations per launch: the expert straight-line guess of every {wl['name']} problem"}
        extras['k_eval'] = ev
        del run
        for name in ('c2', 'c5'):
            if name == args.workload:
                continue
            wl_x = workload(name, 0, 1)
            rx = DeviceRun(wl_x, local_rank, dev, torch, lib, C)
            l0 = rx.h.launch_count()
            ms_list = timed_steps(torch, dist, rx, K, W, flush, False, None)
            sm = float(np.mean(ms_list))
            ax = rx.accounting()
            _, te = e2e_run(torch, dist, rx, wl_x, lib, Ke, False, 1, dev)
            extras[name] = {'metric': METRIC, 'value': wl_x['B'] / (sm * 1e-3), 'unit': UNIT, 'ms_per_step': sm, 'steps': K,
                            'config': describe(wl_x, 1), 'ok_fraction': ax['ok_fraction'], 'mean_evals_per_traj': ax['evals'] / wl_x['B'],
                            'evals_per_s': ax['evals'] / (sm * 1e-3), 'e2e': {'value': wl_x['B'] * Ke / te, 'unit': UNIT},
                            'gpu_launches': int((rx.h.launch_count() - l0) * K // (K + W)), 'map_build_s': rx.map_build_s,
                            'roofline': roofline_of(ax, wl_x['M'], sm, fp64_peak, hbm_peak, bool(peaks), hbm_bytes_of(wl_x), name)}
            if name == 'c2':
                lat = single_plan_latency(wl_x)
                if cpu_lat is not None:
                    lat['cpu_reference_port'] = cpu_lat
                lat['reference_node_reports'] = '30-100 ms per plan (SURVEY.md §8a a10, probed)'
                extras['single_plan_latency'] = lat
            del rx

    if rank == 0:
        line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world_size, 'steps': K, 'warmup': W,
                'ms_per_step': step_ms, 'higher_is_better': True, 'scaling': wl['scaling'], 'vs_baseline': None, 'dtype': 'f64',
                'data': 'synthetic', 'config': describe(wl, world_size),
                'evals_per_s': world_size * acc['evals'] / (step_ms * 1e-3), 'mean_evals_per_traj': acc['evals'] / B,
                'ok_fraction': acc['ok_fraction'], 'clocks': clocks, 'map_build_s': map_build_s,
                'map_build_note': f"{len(wl['worlds'])} occupancy grids -> exact EDT + gradient on the device (neo_set_maps_occupancy: H2D, 5 kernels per map, one sync), outside the timed steps",
                'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'steps': Ke,
                        'includes': 'neo_optimize with host buffers: inputs staged in pinned memory and copied (retry guesses are read over PCIe on demand, counted in full here), kernel, results written by the kernel into mapped pinned memory, scatter into the caller arrays' + (' -- with several ranks: sharding.DeviceShard (inputs staged and copied, neo_optimize_dev, ONE NCCL all-gather of the packed records on the device, ONE D2H of the gathered batch on every rank)' if distributed else '')},
                'gpu_launches': int(launches) * world_size,
                'roofline': roofline_of(acc, M, step_ms, fp64_peak, hbm_peak, bool(peaks), hbm_bytes_of(wl), wl['name']),
                'wall_s_timed_region': t_wall}
        if cpu_base is not None:
            cpu_base['gpu_vs_c_port_all_cores'] = value / cpu_base['c_port_all_cores']['value']
            line['cpu_baseline'] = cpu_base
        if extras is not None:
            line['extras'] = extras
        if last_step is not None:
            dump_outputs(args.dump_outputs, last_step.cpu().numpy(), B, wl['M'])
        print(json.dumps(line))
    if distributed:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
