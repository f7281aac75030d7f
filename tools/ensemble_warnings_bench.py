#!/usr/bin/env python
"""
Flood-warning products of an ensemble on the device, at C5 shape: the bench's 7M-reach network
(synth.forest(7_000_000, 5000, seed=4, depth_bias=0.5), muskingum_params(.., 4)), 51 members, float32 lateral
inflows, 48 hourly rows.  Member m's inflows are the view big[m:m+T] of one pinned (T+M, n) array: distinct series
in 2.3 GB instead of 69 GB of host memory.  Six return-period-like thresholds per river (fixed fractions of a routed
reference row), so every exceedance level is hit somewhere.

Prints one JSON line; the three calls run alternately after a warm-up round:
  six_stats        Plan.route_ensemble_stats_host with the six statistics of tools/ensemble_stats_bench.py (float32
                   out): the baseline; wall time and D2H bytes
  warnings_steps   the same six plus six exceed_* statistics, per-step rows
  warnings_peaks   the same twelve statistics with horizon peaks only (outs=None): only the peaks cross PCIe
  kernel           the statistics kernel alone over a resident (51, 16, n) fp64 array (46 GB, far past L2), CUDA
                   events, GB/s on its M*8 + output bytes per (row, reach) against HBM3e's 7.7 TB/s:
                   exceed_only   six exceed_* statistics, float32 rows (the no-sort instantiation)
                   peak_mode     the twelve statistics, peaks only (sorting instantiation, one CTA row; 12 B of peak
                                 state read and written per statistic and (row, reach))
  parity           twelve statistics with peaks on 16 routed rows of sampled reaches, fp64, against numpy over the fp64
                   outputs of single-member routes of the same reaches (bit for bit)

    python tools/ensemble_warnings_bench.py [--reaches 7000000] [--members 51] [--rows 48] > profiles/....jsonl
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
LABELS = ['rp2', 'rp5', 'rp10', 'rp25', 'rp50', 'rp100']
FRACTIONS = [0.6, 0.8, 1.0, 1.2, 1.5, 2.0]    # threshold = fraction * a reference discharge of the reach
EXCEED = [f'exceed_{x}' for x in LABELS]
WARN = STATS + EXCEED
HBM_BPS = 7.7e12
DT = 3600


def numpy_statistic(x, name, thr):
    if name.startswith('exceed_'):
        return np.mean(x > thr[LABELS.index(name[7:])], axis=0)
    return {'mean': np.mean, 'std': np.std, 'min': np.min, 'max': np.max}[name](x, axis=0) if name[0] != 'p' \
        else np.percentile(x, int(name[1:]), axis=0)


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def kernel_time(n, M, rows, iters):
    import torch
    x = torch.rand((M, rows, n), dtype=torch.float64, device='cuda') * 100.0
    thr = torch.tensor(FRACTIONS, dtype=torch.float64, device='cuda')[:, None] * 50.0 * torch.ones((1, n), dtype=torch.float64,
                                                                                                  device='cuda')
    outs = [torch.empty((rows, n), dtype=torch.float32, device='cuda') for _ in EXCEED]
    peak = torch.empty((len(WARN), n), dtype=torch.float64, device='cuda')
    prow = torch.empty((len(WARN), n), dtype=torch.int32, device='cuda')
    stream = torch.cuda.current_stream().cuda_stream
    res = {}
    cases = (('exceed_only', EXCEED, lambda: ensemble_stats_dev(EXCEED, M, x.data_ptr(), rows * n, n, rows, n,
                                                                [t.data_ptr() for t in outs], n, True, 0, stream,
                                                                thresholds=LABELS, thr_ptr=thr.data_ptr(), ldt=n),
              len(EXCEED) * 4),
             ('peak_mode', WARN, lambda: ensemble_stats_dev(WARN, M, x.data_ptr(), rows * n, n, rows, n, None, 0, False, 0,
                                                            stream, thresholds=LABELS, thr_ptr=thr.data_ptr(), ldt=n,
                                                            peak_ptrs=(peak.data_ptr(), prow.data_ptr()), ldk=n),
              len(WARN) * 12))
    for label, names, call, out_bytes in cases:
        for _ in range(3):
            call()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            call()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b) / iters
        nbytes = rows * n * (M * 8 + out_bytes)
        res[label] = dict(stats=names, ms=round(ms, 3), bytes=nbytes, gbps=round(nbytes / ms / 1e6, 1),
                          frac_hbm=round(nbytes / (ms * 1e-3) / HBM_BPS, 3))
    del x, outs, peak, prow, thr
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
    rec = dict(tool='ensemble_warnings_bench', gpu=gpu_info(), reaches=n, members=M, rows=T, lateral='float32',
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
    # thresholds: fractions of member 0's discharge at the middle row
    ref_row = np.empty((T, n), dtype=np.float32)
    q = q0.copy()
    plan.route_host(rr.MODE_RAPID, q, lats[0], ref_row, 1)
    base = ref_row[T // 2].astype(np.float64)
    del ref_row
    thr = np.array([f * base for f in FRACTIONS])
    plan.set_thresholds(dict(zip(LABELS, thr)))
    six_out = [rr.pinned_empty((T, n), np.float32) for _ in STATS]
    warn_out = six_out + [rr.pinned_empty((T, n), np.float32) for _ in EXCEED]
    peaks = (np.empty((len(WARN), n)), np.empty((len(WARN), n), dtype=np.int32))
    calls = {
        'six_stats': (lambda: plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, STATS, six_out, 1),
                      len(STATS) * T * n * 4),
        'warnings_steps': (lambda: plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, WARN, warn_out, 1),
                           len(WARN) * T * n * 4),
        'warnings_peaks': (lambda: plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, WARN, None, 1, peaks=peaks),
                           len(WARN) * n * 12),
    }
    times = {name: [] for name in calls}
    for rep in range(args.repeats + 1):           # rep 0 warms every call up (allocations, modules)
        for name, (fn, _) in calls.items():
            t0 = time.perf_counter()
            fn()
            dt = time.perf_counter() - t0
            if rep:
                times[name].append(round(dt, 3))
    for name, (_, d2h) in calls.items():
        rec[name] = dict(seconds=times[name], best=min(times[name]), d2h_bytes=d2h)
    rec['warnings_steps']['stats'] = rec['warnings_peaks']['stats'] = WARN
    rec['six_stats']['stats'] = STATS
    # the peaks-only call's peaks against the per-step rows of the steps call (float32 rows: value within rounding)
    rec['peaks_vs_rows_max_equal_f32'] = bool(all(np.array_equal(peaks[0][s].astype(np.float32), warn_out[s].max(axis=0))
                                                  for s in range(len(WARN))))

    # parity: 16 rows, sampled reaches, fp64 out and peaks; members one at a time through the single-member call
    rows = 16
    pick = np.sort(np.random.default_rng(0).choice(n, args.sample, replace=False)).astype(np.int32)
    plan.set_output_subset(pick)
    got = [np.empty((rows, pick.shape[0])) for _ in WARN]
    pk = (np.empty((len(WARN), pick.shape[0])), np.empty((len(WARN), pick.shape[0]), dtype=np.int32))
    plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, [a[:rows] for a in lats], WARN, got, 1, peaks=pk)
    members = np.empty((M, rows, pick.shape[0]))
    for m in range(M):
        q = q0.copy()
        plan.route_host(rr.MODE_RAPID, q, lats[m][:rows], members[m], 1)
    plan.set_output_subset(None)
    bitwise = {}
    for i, s in enumerate(WARN):
        want = numpy_statistic(members, s, thr[:, pick])
        bitwise[s] = bool(np.array_equal(got[i], want) and np.array_equal(pk[0][i], want.max(axis=0))
                          and np.array_equal(pk[1][i], want.argmax(axis=0)))
    rec['parity'] = dict(rows=rows, reaches=int(pick.shape[0]), bitwise=bitwise)
    plan.close()
    print(json.dumps(rec), flush=True)


if __name__ == '__main__':
    main()
