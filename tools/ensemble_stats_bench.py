#!/usr/bin/env python
"""
Ensemble statistics on the device against member files, at C5 shape: the bench's 7M-reach network
(synth.forest(7_000_000, 5000, seed=4, depth_bias=0.5), muskingum_params(.., 4)), 51 members, float32 lateral
inflows, 48 hourly rows.  Member m's inflows are the view big[m:m+T] of one pinned (T+M, n) array: distinct series
in 2.3 GB instead of 69 GB of host memory.

Prints one JSON line:
  stats_call    wall time of Plan.route_ensemble_stats_host with six statistics (float32 out) and its D2H bytes
  member_call   wall time of Plan.route_ensemble_host with float32 member outputs on the same inputs and its D2H bytes
                (every member's rows land in the same pinned array: same copies, same rate, 1.3 GB of host memory
                instead of 69 GB)
  kernel        the statistics kernel alone over a resident (51, 16, n) fp64 array (46 GB, far past L2), CUDA events,
                GB/s on its M*8 + S*4 bytes per (row, reach) against HBM3e's 7.7 TB/s
  parity        the statistics of 16 routed rows on sampled reaches, fp64, against numpy over the fp64 outputs of
                single-member routes of the same reaches (bit for bit)

    python tools/ensemble_stats_bench.py [--reaches 7000000] [--members 51] [--rows 48] > profiles/....jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import river_route_b200 as rr  # noqa: E402
from river_route_b200 import synth  # noqa: E402
from river_route_b200.plan import ensemble_stats_dev  # noqa: E402

STATS = ['mean', 'std', 'min', 'max', 'p10', 'p90']
HBM_BPS = 7.7e12
DT = 3600


def numpy_statistic(x, name):
    return {'mean': np.mean, 'std': np.std, 'min': np.min, 'max': np.max}[name](x, axis=0) if name[0] != 'p' \
        else np.percentile(x, int(name[1:]), axis=0)


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def kernel_time(n, M, rows, iters):
    import torch
    x = torch.rand((M, rows, n), dtype=torch.float64, device='cuda') * 100.0
    outs = [torch.empty((rows, n), dtype=torch.float32, device='cuda') for _ in STATS]
    stream = torch.cuda.current_stream().cuda_stream
    res = {}
    for label, names in (('six', STATS), ('no_percentile', ['mean', 'std', 'min', 'max'])):
        o = outs[:len(names)]
        call = lambda: ensemble_stats_dev(names, M, x.data_ptr(), rows * n, n, rows, n, [t.data_ptr() for t in o], n, True,
                                          0, stream)
        for _ in range(3):
            call()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            call()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b) / iters
        nbytes = rows * n * (M * 8 + len(names) * 4)
        res[label] = dict(stats=names, ms=round(ms, 3), bytes=nbytes, gbps=round(nbytes / ms / 1e6, 1),
                          frac_hbm=round(nbytes / (ms * 1e-3) / HBM_BPS, 3))
    del x, outs
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reaches', type=int, default=7_000_000)
    ap.add_argument('--members', type=int, default=51)
    ap.add_argument('--rows', type=int, default=48)
    ap.add_argument('--repeats', type=int, default=2)
    ap.add_argument('--kernel-rows', type=int, default=16)
    ap.add_argument('--kernel-iters', type=int, default=10)
    ap.add_argument('--sample', type=int, default=4096)
    args = ap.parse_args()
    if not rr.cuda_available():
        raise SystemExit('needs a CUDA device')
    n, M, T = args.reaches, args.members, args.rows
    rec = dict(tool='ensemble_stats_bench', gpu=gpu_info(), reaches=n, members=M, rows=T, lateral='float32',
               network='synth.forest(n, 5000, seed=4, depth_bias=0.5), muskingum_params(n, 4)')
    rec['kernel'] = kernel_time(n, M, args.kernel_rows, args.kernel_iters)

    down = synth.forest(n, 5000, seed=4, depth_bias=0.5)
    k, x = synth.muskingum_params(n, 4)
    dt_div_k = DT / k
    den = dt_div_k + (2 * (1 - x))
    c1, c2, c3 = (dt_div_k - 2 * x) / den, (dt_div_k + 2 * x) / den, ((2 * (1 - x)) - dt_div_k) / den
    plan = rr.Plan(down)
    plan.set_coefficients(c1, c2, c3, (c1 + c2) / DT)
    big = rr.pinned_empty((T + M, n), np.float32)
    for t0 in range(0, T + M, 8):
        t1 = min(T + M, t0 + 8)
        big[t0:t1] = synth.lateral_volumes(t1 - t0, n, seed=100 + t0)
    lats = [big[m:m + T] for m in range(M)]
    q0 = np.full(n, 5.0)
    stat_out = [rr.pinned_empty((T, n), np.float32) for _ in STATS]
    member_out = rr.pinned_empty((T, n), np.float32)

    def stats_call():
        return plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, STATS, stat_out, 1)

    def member_call():
        return plan.route_ensemble_host(rr.MODE_RAPID, q0, lats, [member_out] * M, 1)

    times = {'stats': [], 'member': []}
    means = {}
    for rep in range(args.repeats + 1):           # rep 0 warms both up (allocations, pinned bounce, modules)
        for name, fn in (('stats', stats_call), ('member', member_call)):
            t0 = time.perf_counter()
            means[name] = fn()
            dt = time.perf_counter() - t0
            if rep:
                times[name].append(round(dt, 3))
    rec['stats_call'] = dict(stats=STATS, seconds=times['stats'], best=min(times['stats']), d2h_bytes=len(STATS) * T * n * 4)
    rec['member_call'] = dict(seconds=times['member'], best=min(times['member']), d2h_bytes=M * T * n * 4)
    rec['stats_over_member'] = round(rec['stats_call']['best'] / rec['member_call']['best'], 3)
    rec['final_state_equal'] = bool(np.array_equal(means['stats'], means['member']))

    # parity: 16 rows, sampled reaches, fp64 out; members one at a time through the single-member call
    rows = 16
    pick = np.sort(np.random.default_rng(0).choice(n, args.sample, replace=False)).astype(np.int32)
    plan.set_output_subset(pick)
    got = [np.empty((rows, pick.shape[0])) for _ in STATS]
    plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, [a[:rows] for a in lats], STATS, got, 1)
    members = np.empty((M, rows, pick.shape[0]))
    for m in range(M):
        q = q0.copy()
        plan.route_host(rr.MODE_RAPID, q, lats[m][:rows], members[m], 1)
    plan.set_output_subset(None)
    rec['parity'] = dict(rows=rows, reaches=int(pick.shape[0]),
                         bitwise={s: bool(np.array_equal(got[i], numpy_statistic(members, s))) for i, s in enumerate(STATS)})
    plan.close()
    print(json.dumps(rec), flush=True)


if __name__ == '__main__':
    main()
