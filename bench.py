#!/usr/bin/env python
"""
bench.py -- reach-timesteps/sec of the RapidMuskingum routing hot path (BASELINE.json metric).

Workload (config.workload = "C4"): the GEOGLOWS-scale configuration of BASELINE.json configs[3] --
a synthetic 7M-reach forest in 5000 independent basins (SURVEY.md 8d generator, seed 4), hourly
lateral inflow volumes, dt_routing = dt_runoff = 3600 s, fp64.  One "step" routes one chunk of `--rows`
hourly time steps over the whole network, chained in time through the channel state (a 1-year run is
8760/rows such steps).  The 7M-reach network fits one B200, so it is the N=1 workload; with N GPUs the basins of
the same network are bin-packed over the ranks (no collective in the time loop) and every step routes
N x `--rows` time steps, so the bytes each GPU streams per step stay fixed ("scaling": "weak"; `--scaling strong`
keeps the rows, and so the total work, fixed instead).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...            # the reference itself (numba) on the host cores
    python bench.py ... --dump-outputs DIR                   # + the last timed step's results, sampled, as .npy

Same arguments, same inputs: the network, the parameters and the lateral inflows are generated from fixed seeds, so
the files --dump-outputs writes let two builds be compared output for output.

One JSON line on rank 0:
  value      device-resident launches, CUDA events (max over ranks)
  e2e        the same rows through the host-array API the router classes call: pinned fp64 lateral inflows in,
             float32 discharge out (what the reference hands its writer), H2D + D2H inside the timed region
  roofline   the routing kernel: `frac` on SURVEY 8d's 56 B per reach-timestep (the contract; a model ratio, not
             a bandwidth utilisation, because a 64-step time tile reads coefficients and topology once),
             `traffic` / `frac_dram` on the DRAM bytes ncu measured for this kernel variant (profiles/traffic.json),
             `frac_min` on the bytes a time-tiled kernel must move (16 + 40 / tile_rows); the same three for the
             whole step under `step`
  checks     parity of this run's own results: against the CPU oracle on a whole-basin subset of every rank, and
             (N > 1) the sharded result gathered over NCCL into params-file order against a single-GPU route of the
             whole network on rank 0
The reference arm never imports river_route_b200: it runs river-route's own numba kernels (oracle/refarm.py).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B_ALG = 56.0  # algorithmic bytes per reach-timestep (SURVEY.md 8d): 8 lateral + 8 discharge + 32 coefficients + 8 topology
DT = 3600
PARITY_TOL = 1e-10   # north_star: fp64 discharge within 1e-10 relative


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--reaches', type=int, default=7_000_000)
    ap.add_argument('--basins', type=int, default=5000)
    ap.add_argument('--rows', type=int, default=240, help='hourly time steps per step (per GPU in weak scaling)')
    ap.add_argument('--e2e-rows', type=int, default=0, help='time steps per end-to-end step, per GPU (0 = --rows)')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='weak: N x rows time steps per step on N GPUs (bytes per GPU fixed); strong: rows fixed')
    ap.add_argument('--no-e2e-variants', action='store_true')
    ap.add_argument('--e2e-steps', type=int, default=3)
    ap.add_argument('--check-rows', type=int, default=128, help='rows of the parity checks (two time tiles)')
    ap.add_argument('--no-checks', action='store_true')
    ap.add_argument('--cpu-sample-reaches', type=int, default=1_000_000)
    ap.add_argument('--ref-cores', type=int, default=0, help='reference arm: worker processes (0 = all host cores)')
    ap.add_argument('--depth-bias', type=float, default=0.5)
    ap.add_argument('--time-tile', type=int, default=0)
    ap.add_argument('--tile-stride', type=int, default=0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--staging', default='auto', choices=['auto', 'registers', 'registers-tiled', 'tma', 'out-reach-major', 'lateral-grouped', 'direct', 'direct-nohw'])
    ap.add_argument('--order', default='growth', choices=['growth', 'level'],
                    help='reach order of the synthetic params file: generator order or sorted by topological level')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed to DIR/discharge.npy and '
                         'DIR/channel_state.npy (float64, a fixed sample of the reaches, at most 64 MB in all)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the results of the CUDA arm (--impl b200)')
    return args


def coefficients(k, x, dt_routing, dt_runoff):
    """The reference's exact expressions (routers/Muskingum.py:174-179, TransformMuskingum.py:104)."""
    dt_div_k = dt_routing / k
    denominator = dt_div_k + (2 * (1 - x))
    _2x = 2 * x
    c1 = (dt_div_k - _2x) / denominator
    c2 = (dt_div_k + _2x) / denominator
    c3 = ((2 * (1 - x)) - dt_div_k) / denominator
    return c1, c2, c3, (c1 + c2) / dt_runoff


def workload_config(args):
    """Identical in both arms: the workload, not how one arm happens to run it."""
    return {'workload': 'C4', 'router': 'RapidMuskingum', 'reaches': args.reaches, 'basins': args.basins,
            'scaling_rule': (f'weak: rows_per_step = {args.rows} x n_gpus on the same {args.reaches}-reach network'
                             if args.scaling == 'weak' else 'strong: rows_per_step fixed'),
            'network': f'synthetic forest seed 4 depth_bias {args.depth_bias} (SURVEY.md 8d), reach order: {args.order}',
            'rows_per_step_per_gpu': args.rows, 'dt_runoff_s': DT, 'dt_routing_s': DT, 'substeps': 1,
            'parallelism': f'basin-sharded x{args.gpus}, no collective in the time loop',
            'l2': 'inputs larger than L2: every step streams rows x reaches x 16 B'}


# ---------------------------------------------------------------------------------------------------------------
# reference arm
# ---------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: river-route's own numba path on the host cores -- RapidMuskingum._router ->
    rapid_route (routers/RapidMuskingum.py:19-33, _numba_kernels.py:49-84) from the unmodified copy under
    oracle/_ref, independent watersheds in separate processes as docs/references/parallelism.md:67-112 describes.
    A step routes `--rows` hourly steps of the whole network (the N=1 step of the CUDA arm).  No product code and no
    GPU library is loaded by this arm."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from oracle import refarm
    cores = args.ref_cores or (len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else os.cpu_count() or 1)
    down = refarm.forest(args.reaches, args.basins, seed=4, depth_bias=args.depth_bias)
    k, x = refarm.muskingum_params(args.reaches, 4)
    if args.order != 'growth':
        raise SystemExit('--impl reference runs the generator (growth) order only')
    rows = args.rows
    if refarm.reference_available():
        kind = 'reference'
        pool = refarm.WatershedPool(down, k, x, rows, cores, DT)
        step = pool.step
        how = ('river_route v2.0.1 from oracle/_ref (unmodified): RapidMuskingum._router -> numba rapid_route, '
               f'{cores} worker processes over LPT-packed whole basins (multiprocessing.Pool)')
    else:
        # the copy of the reference did not travel (built without /root/reference): time the C restatement instead
        kind = 'port'
        from oracle import oracle
        part = refarm.basin_parts(down, cores)
        shards = []
        for c in range(cores):
            idx = np.flatnonzero(part == c)
            local = refarm.local_network(down, idx)
            c1, c2, c3, c4 = coefficients(k[idx], x[idx], DT, DT)
            indptr, indices = oracle.csc_from_down(local)
            shards.append(dict(indptr=indptr, indices=indices, lhs_off=oracle.lhs_off_data(c1, indices), c2=c2, c3=c3,
                               c4_dt=c4, q_t=np.zeros(idx.shape[0]), ql=refarm.lateral_volumes(rows, idx.shape[0], 100 + c),
                               out=np.zeros((rows, idx.shape[0]))))
        step = lambda: oracle.rapid_route_sharded(shards, 1, cores)   # noqa: E731
        how = f'oracle/rr_oracle.c rapid_route (C restatement; oracle/_ref absent), {cores} threads over LPT-packed basins'
    for _ in range(args.warmup):
        step()
    t = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t
    if kind == 'reference':
        pool.close()
    value = args.reaches * rows * args.steps / dt
    sample = (f'{args.reaches} reaches x {rows} hourly steps per step (the N=1 step; the CPU does not grow with --gpus), '
              f'state chained between steps; {how}; host has {os.cpu_count()} cores')
    line = {
        'impl': 'reference', 'metric': 'reach-timesteps/sec (RapidMuskingum, fp64)', 'value': value,
        'unit': 'reach-timesteps/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(args),
        'cpu_baseline': {'value': value, 'unit': 'reach-timesteps/s', 'cores': cores, 'kind': kind, 'sample': sample},
        'e2e': {'value': value, 'unit': 'reach-timesteps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline(down, k, x, target_reaches, rows):
    """Rank 0, N=1: the reference's numba rapid_route on ONE core (it is single-threaded by construction) on a bounded
    sample -- the first whole basins of the network x `rows` steps -- plus the C restatement on the same sample."""
    from oracle import refarm
    res = {'unit': 'reach-timesteps/s', 'cores': 1}
    outlets = np.flatnonzero(down < 0)
    m = int(outlets[np.searchsorted(outlets, min(target_reaches, down.shape[0]) - 1)]) + 1
    ql = refarm.lateral_volumes(rows, m, 99)
    if refarm.reference_available():
        r = refarm.single_core(down, k, x, target_reaches, rows, DT, ql=ql)
        res.update(value=r['value'], kind='reference',
                   sample=f"first {r['reaches']} reaches (whole basins) x {rows} hourly steps, river_route v2.0.1 "
                          f"RapidMuskingum._router -> numba rapid_route (oracle/_ref), warm, {r['seconds']:.2f} s; "
                          f"host has {os.cpu_count()} cores; the all-cores figure is the --impl reference arm")
    from oracle import oracle
    c1, c2, c3, c4 = coefficients(k[:m], x[:m], DT, DT)
    indptr, indices = oracle.csc_from_down(down[:m])
    lhs = oracle.lhs_off_data(c1, indices)
    out, q = np.zeros((rows, m)), np.zeros(m)
    oracle.rapid_route(indptr, indices, lhs, c2, c3, c4, q, ql[:2], out[:2], 1)   # page in
    t = time.perf_counter()
    oracle.rapid_route(indptr, indices, lhs, c2, c3, c4, q, ql, out, 1)
    sec = time.perf_counter() - t
    port = {'value': m * rows / sec, 'kind': 'port', 'sample': f'same sample, oracle/rr_oracle.c (-O3, scalar), {sec:.2f} s'}
    if 'value' in res:
        res['port'] = port
    else:
        res.update(port)
    return res


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML polled every few
    milliseconds from a thread (the timed region is only a few hundred ms); nvidia-smi as a fallback."""
    SMI_Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread, self.proc = index, [], False, None, None
        self.max_mhz = None

    def _visible_index(self):
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        if vis:
            try:
                return int(vis.split(',')[self.index])
            except Exception:
                pass
        return self.index

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self._visible_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons = {'hw_slowdown': pynvml.nvmlClocksThrottleReasonHwSlowdown,
                       'hw_thermal_slowdown': pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                       'sw_thermal_slowdown': pynvml.nvmlClocksThrottleReasonSwThermalSlowdown,
                       'sw_power_cap': pynvml.nvmlClocksThrottleReasonSwPowerCap}

            def poll():
                while not self.stop_flag:
                    try:
                        mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        mask = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                        self.samples.append((mhz, [k for k, bit in reasons.items() if mask & bit]))
                    except Exception:
                        pass
                    time.sleep(0.004)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.SMI_Q}', '--format=csv,noheader,nounits',
                                          '-i', str(self._visible_index()), '-lms', '50'], stdout=subprocess.PIPE, text=True)

            def read():
                names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
                for line in self.proc.stdout:
                    f = [x.strip() for x in line.split(',')]
                    try:
                        self.max_mhz = float(f[2])
                        self.samples.append((float(f[1]), [nm for nm, v in zip(names, f[5:9]) if v.lower().startswith('active')]))
                    except Exception:
                        continue
            threading.Thread(target=read, daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=1.0)
        if self.proc:
            time.sleep(0.1)
            self.proc.terminate()
        sm = [x[0] for x in self.samples]
        reasons = sorted({r for x in self.samples for r in x[1]})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': self.max_mhz, 'reasons': reasons,
                'samples': len(sm)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


def pcie_ceiling(world, e2e_value):
    """The measured concurrent pinned H2D + D2H rate of this pool's boxes at this rank count
    (tools/pcie_ceiling_probe.py -> profiles/r02_pcie_ceiling.jsonl) and the e2e value as a fraction of what it allows
    for 8 B in / 4 B out per reach-timestep."""
    try:
        best = None
        with open(os.path.join(ROOT, 'profiles', 'r02_pcie_ceiling.jsonl')) as f:
            for line in f:
                d = json.loads(line)
                if d.get('n_gpus') == world:
                    best = d
        if best is None:
            return None
        h2d = best['h2d_only']['GBps_aggregate_per_direction'] * 1e9 / 8.0      # 8 B enter the GPU per reach-timestep
        both = best['both']['GBps_aggregate_per_direction'] * 1e9 / 8.0         # ... while as many bytes leave it
        return {'GBps_h2d_only': best['h2d_only']['GBps_aggregate_per_direction'],
                'GBps_d2h_only': best['d2h_only']['GBps_aggregate_per_direction'],
                'GBps_each_direction_when_both_run': best['both']['GBps_aggregate_per_direction'],
                'reach_steps_per_s_at_h2d_only_rate': h2d, 'reach_steps_per_s_at_both_directions_rate': both,
                'e2e_frac_of_h2d_only_ceiling': e2e_value / h2d,
                'note': 'e2e moves 8 B in and 4 B out per reach-timestep: its ceiling lies between the two rates',
                'source': 'profiles/r02_pcie_ceiling.jsonl (tools/pcie_ceiling_probe.py, same pool, all ranks at once)'}
    except Exception:
        return None


def ncu_traffic(variant):
    """DRAM bytes per reach-timestep of each kernel class from the committed ncu capture of this kernel variant."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            return json.load(f)['variants'].get(variant)
    except Exception:
        return None


def roofline_block(ktimes, steps, n, rows, tile_rows, value, variant, peak, peak_src, n_in_kernel=None):
    """All fractions are of the measured copy peak.  `frac`: the contract's 56 B (a model ratio: > 1 is possible);
    `frac_dram`: DRAM bytes ncu counted for this variant / CUDA-event time; `frac_min`: bytes a time-tiled kernel must
    move (8 lateral + 8 discharge + 40 B of coefficients / topology once per tile)."""
    units = float(n) * float(rows)
    # reach-timesteps ONE launch of the wavefront kernel processes: with the headwater blocks routed by the staging
    # kernel (pipeline, RapidMuskingum, >= 2^18 reaches) that is the non-headwater share of the network
    k_units = float(n_in_kernel if n_in_kernel is not None else n) * float(rows)
    kernel_ms = ktimes['route']['ms'] / max(ktimes['route']['launches'], 1)
    b_min = 16.0 + 40.0 / max(tile_rows, 1)
    tr = ncu_traffic(variant) or {}

    def gbs(bytes_per_unit, ms, u=None):
        return bytes_per_unit * (units if u is None else u) / (ms * 1e-3) / 1e9
    achieved = gbs(B_ALG, kernel_ms, k_units)
    r_bytes = (tr.get('route') or {}).get('dram_bytes_per_reach_step')     # per reach-timestep of the WHOLE network
    block = {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
             'units_per_launch': k_units, 'units_note': 'reach-timesteps the wavefront launch itself advances',
             'traffic': r_bytes * units if r_bytes else None,
             'frac_dram': gbs(r_bytes, kernel_ms) / peak if r_bytes else None,
             'frac_min': gbs(b_min, kernel_ms, k_units) / peak,
             'kernel': 'rr_direct_kernel<RAPID>' if variant == 'pipeline' else 'rr_wavefront_kernel<RAPID>', 'kernel_ms': kernel_ms,
             'tile_rows': tile_rows,
             'algorithmic_bytes_per_reach_step': B_ALG, 'min_bytes_per_reach_step': b_min,
             'dram_bytes_per_reach_step': r_bytes, 'peak_source': peak_src,
             'traffic_source': (f"{tr.get('source')} ({tr.get('reaches')} reaches x {tr.get('rows')} rows, variant "
                                f"'{variant}'), scaled per reach-timestep") if tr else None,
             'frac_note': "frac = 56 B contract / kernel time (model ratio, can exceed 1); frac_dram = measured DRAM "
                          "bytes / kernel time; frac_min = (16 + 40/tile_rows) B / kernel time; all / measured copy peak",
             'step_ms_by_kernel': {k_: v['ms'] / steps for k_, v in ktimes.items()}}
    step_ms = sum(v['ms'] for v in ktimes.values()) / steps
    s_bytes = None
    if tr and all(c in tr for c in ('route', 'permute_to_working', 'permute_to_user')):
        s_bytes = sum(tr[c]['dram_bytes_per_reach_step'] for c in ('route', 'permute_to_working', 'permute_to_user'))
    block['step'] = {'ms': step_ms, 'frac': gbs(B_ALG, step_ms) / peak,
                     'frac_dram': gbs(s_bytes, step_ms) / peak if s_bytes else None,
                     'frac_min': gbs(b_min, step_ms) / peak, 'dram_bytes_per_reach_step': s_bytes,
                     'traffic': s_bytes * units if s_bytes else None}
    return block


def main():
    args = parse()
    if not args.e2e_rows:
        args.e2e_rows = args.rows
    if args.impl == 'reference':
        return run_reference(args)

    import torch
    import river_route_b200 as rr
    from river_route_b200 import synth
    from river_route_b200.sharding import shard_by_basin

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus and world > 1:
        raise SystemExit(f'--gpus {args.gpus} but WORLD_SIZE={world}')
    if not rr.cuda_available():
        raise SystemExit('bench.py needs a CUDA device: river_route_b200 has no CPU fallback')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    numa_bound = False
    if world > 1:                                   # each rank streams over its own PCIe link from its own NUMA node
        from river_route_b200.sharding import bind_to_gpu_numa
        numa_bound = bind_to_gpu_numa(local_rank)
    dist = None
    real_stdout = None
    if world > 1:
        # stdout carries exactly one JSON line: anything libraries print there meanwhile (NCCL's version banner at
        # communicator creation) goes to stderr instead
        sys.stdout.flush()
        real_stdout = os.dup(1)
        os.dup2(2, 1)
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)

    # ---- network, shard, plan ----
    down = synth.forest(args.reaches, args.basins, seed=4, depth_bias=args.depth_bias)
    k, x = synth.muskingum_params(args.reaches, 4)
    if args.order == 'level':
        down = synth.relabel(down, synth.level_sorted_order(down))
    idx, local_down = shard_by_basin(down, world, rank)
    n = int(idx.shape[0])
    plan = rr.Plan(local_down, time_tile=args.time_tile, tile_stride=args.tile_stride, device=local_rank,
                   staging=args.staging)
    c1, c2, c3, c4 = coefficients(k[idx], x[idx], DT, DT)
    plan.set_coefficients(c1, c2, c3, c4)
    info = plan.info

    # ---- device-resident inputs: lateral volumes gamma(0.3, 5e4 m3) with half exact zeros.  Row t is generated for
    # the WHOLE network from a per-row seed and this rank keeps its own columns, so the input of reach i at step t does
    # not depend on how the basins are sharded (the N > 1 result can be compared with a single-GPU route) ----
    rows = args.rows * (world if args.scaling == 'weak' else 1)
    ld = ((n + 31) // 32) * 32
    gen = torch.Generator(device=dev)
    idx_t = torch.from_numpy(idx).to(dev)
    conc = torch.full((args.reaches,), 0.3, dtype=torch.float64, device=dev)

    def lateral_row(t, cols=None):
        gen.manual_seed(1234 + 7919 * t)
        g = torch._standard_gamma(conc, generator=gen) * 5.0e4
        g[torch.rand(args.reaches, device=dev, generator=gen) < 0.5] = 0.0
        return g if cols is None else g[cols]

    d_lat = torch.zeros((rows, ld), dtype=torch.float64, device=dev)
    for t in range(rows):
        d_lat[t, :n] = lateral_row(t, idx_t if world > 1 else None)
    d_out = torch.empty((rows, ld), dtype=torch.float64, device=dev)
    d_q = torch.zeros(n, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        plan.route_dev(rr.MODE_RAPID, d_q.data_ptr(), d_lat.data_ptr(), ld, d_out.data_ptr(), ld, rows, 1, stream)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    rr.launch_count(reset=True)
    from river_route_b200.plan import timing_enable, timing_read
    timing_enable(True)
    timing_read(reset=True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev[0].record()
    for s in range(args.steps):
        step()
        ev[s + 1].record()
    barrier()
    launches = rr.launch_count()
    ktimes = timing_read(reset=True)
    prof = plan.read_profile()
    timing_enable(False)
    clocks = sampler.stop() if rank == 0 else None
    total_ms = ev[0].elapsed_time(ev[-1])
    t_max = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
    total_ms_max = float(t_max.item())
    value = args.reaches * rows * args.steps / (total_ms_max * 1e-3)
    if args.dump_outputs:                           # before the checks below reuse d_out
        dump_outputs(args.dump_outputs, torch, dist, rank, world, down, idx, d_out, d_q, rows, dev)

    # ---- summary outputs gathered over NVLink (outside the time loop): outlet discharge of the last step ----
    outlets = torch.from_numpy(np.flatnonzero(local_down < 0)).to(dev)
    summary = torch.stack([d_out[rows - 1, outlets].sum(), d_q.sum(), torch.tensor(float(n), device=dev, dtype=torch.float64)])
    if dist is not None:
        parts = [torch.empty_like(summary) for _ in range(world)]
        dist.all_gather(parts, summary)
        summary_all = torch.stack(parts).cpu().numpy()
    else:
        summary_all = summary.cpu().numpy()[None]
    finite = bool(torch.isfinite(d_out[:, :n]).all().item())
    checks = {'finite': finite, 'tolerance': PARITY_TOL,
              'summary_per_rank[outlet_q_last_step, state_sum, reaches]': summary_all.tolist()}

    # ---- parity of this run's own results (outside the timed region) ----
    if not args.no_checks:
        checks.update(parity_checks(args, torch, dist, rr, plan, dev, stream, rank, world, down, k, x, idx, local_down,
                                    d_lat, ld, n, lateral_row))

    # ---- end to end through the host-array API: pinned H2D + route + D2H every step ----
    er = min(args.e2e_rows * (world if args.scaling == 'weak' else 1), rows)
    h_lat = rr.pinned_empty((er, n))
    for t0 in range(0, er, 32):
        h_lat[t0:t0 + 32] = d_lat[t0:min(er, t0 + 32), :n].cpu().numpy()
    h_q = rr.pinned_empty((n,))

    def timed_host(call):
        """max over ranks of the wall time of `e2e_steps` host-array calls (state chained between them)."""
        h_q[:] = 0.0
        call()                                                          # warm-up (allocates the staging buffers)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            call()
        barrier()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return args.reaches * er * args.e2e_steps / float(t.item())

    # headline: what RapidMuskingum.route() does between reading a qlateral file and handing the float32 array to
    # the writer (routers.TransformMuskingum._route_lateral -> rr_route_host_ex)
    h_out32 = rr.pinned_empty((er, n), dtype=np.float32)
    e2e_value = timed_host(lambda: plan.route_host(rr.MODE_RAPID, h_q, h_lat, h_out32, 1))
    # the host path must agree with the device path on the same inputs (zero state)
    d_chk_q = torch.zeros(n, dtype=torch.float64, device=dev)
    h_q[:] = 0.0
    plan.route_host(rr.MODE_RAPID, h_q, h_lat, h_out32, 1)
    plan.route_dev(rr.MODE_RAPID, d_chk_q.data_ptr(), d_lat.data_ptr(), ld, d_out.data_ptr(), ld, er, 1, stream)
    torch.cuda.synchronize()
    host_equals_dev = True
    for t0 in range(0, er, 32):
        host_equals_dev &= bool(np.array_equal(d_out[t0:t0 + 32, :n].cpu().numpy().astype(np.float32), h_out32[t0:t0 + 32]))
    variants = {}
    if not args.no_e2e_variants and world == 1:                        # extra pinned host memory: one GPU only
        variants = e2e_variants(args, rr, plan, timed_host, h_q, h_lat, h_out32, er, n, local_down, local_rank, rank)

    if rank == 0:
        peak, peak_src = measured_peak()
        variant = {'auto': 'pipeline', 'direct': 'pipeline', 'registers-tiled': 'ring'}.get(args.staging, args.staging)
        tile_rows = plan.tile_rows(rows, 1)
        line = {
            'metric': 'reach-timesteps/sec (RapidMuskingum, fp64)', 'value': value, 'unit': 'reach-timesteps/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total_ms_max / args.steps,
            'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(args),
            'run': {'rows_per_step': rows, 'reaches_rank0': n, 'plan': {k_: int(v) for k_, v in info.items()}},
            'roofline': roofline_block(ktimes, args.steps, n, rows, tile_rows, value, variant, peak, peak_src,
                                       n - int(info['n_headwaters']) if (variant == 'pipeline' and args.staging != 'direct-nohw' and
                                                                         (n >= (1 << 18) or args.staging == 'direct')) else n),
            'e2e': {'value': e2e_value, 'unit': 'reach-timesteps/s', 'h2d_bytes_per_step': int(n * er * 8 + n * 8),
                    'd2h_bytes_per_step': int(n * er * 4 + n * 8), 'rows_per_step': er, 'steps': args.e2e_steps,
                    'api': 'Plan.route_host with a float32 output array -> rr_route_host_ex: pinned fp64 lateral inflows '
                           'in, route, float32 cast on the device (TransformMuskingum.py:146), float32 discharge out; '
                           'chunked cudaMemcpyAsync on three streams',
                    'host_equals_device_path': host_equals_dev, 'numa_bound': numa_bound, 'variants': variants,
                    'pcie_ceiling': pcie_ceiling(world, e2e_value)},
            'gpu_launches': int(launches), 'kernel_phase_cycles': prof,
            'clocks': clocks,
            'checks': checks,
        }
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline(down, k, x, args.cpu_sample_reaches, rows)
        if real_stdout is not None:
            sys.stdout.flush()
            os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
    ok = checks.get('parity_ok', True) and finite and host_equals_dev
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if not ok:
        raise SystemExit('bench.py: parity check failed (see "checks" / "e2e.host_equals_device_path")')


DUMP_BYTES = 60 << 20    # --dump-outputs: payload of all files together, below 64 MB with the .npy headers


def dump_sample(down, rows):
    """Reaches (indices in params-file order) whose results --dump-outputs writes: every basin outlet, whose discharge
    carries the whole basin upstream of it, and a seeded uniform sample of the other reaches, as many as keep `rows`
    discharge values and one state value per reach within DUMP_BYTES.  Depends on the network and `rows` only."""
    k = DUMP_BYTES // ((rows + 1) * 8)
    if k < 1:
        raise SystemExit(f'--dump-outputs: {rows} rows of one reach exceed {DUMP_BYTES} bytes')
    rng = np.random.default_rng(20261020)
    outlets = np.flatnonzero(down < 0)
    if outlets.shape[0] >= k:
        return np.sort(rng.choice(outlets, k, replace=False))
    inner = np.flatnonzero(down >= 0)
    extra = rng.choice(inner, min(k - outlets.shape[0], inner.shape[0]), replace=False)
    return np.sort(np.concatenate([outlets, extra]))


def dump_outputs(out_dir, torch, dist, rank, world, down, idx, d_out, d_q, rows, dev):
    """What the timed path handed back after its last step -- the discharge of that step's rows and the channel state
    it left -- at the dump_sample reaches, gathered to rank 0 and written there as DIR/discharge.npy (rows x reaches)
    and DIR/channel_state.npy (reaches), float64, columns in params-file order."""
    sample = dump_sample(down, rows)
    pos = np.flatnonzero(np.isin(idx, sample))                     # this rank's columns of sampled reaches
    pos_t = torch.from_numpy(pos).to(dev)
    cols_t = torch.from_numpy(np.searchsorted(sample, idx[pos])).to(dev)
    buf = torch.zeros((rows + 1, sample.shape[0]), dtype=torch.float64, device=dev)
    buf[:rows, cols_t] = d_out[:rows, pos_t]
    buf[rows, cols_t] = d_q[pos_t]
    if dist is not None:                                           # every sampled reach lives on exactly one rank
        own = torch.zeros(sample.shape[0], dtype=torch.uint8, device=dev)
        own[cols_t] = 1
        parts = [torch.empty_like(buf) for _ in range(world)] if rank == 0 else None
        owners = [torch.empty_like(own) for _ in range(world)] if rank == 0 else None
        dist.gather(buf, parts, dst=0)
        dist.gather(own, owners, dst=0)
        if rank == 0:
            for p, o in zip(parts, owners):
                buf[:, o.bool()] = p[:, o.bool()]
    if rank == 0:
        res = buf.cpu().numpy()
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, 'discharge.npy'), res[:rows])
        np.save(os.path.join(out_dir, 'channel_state.npy'), res[rows])


def parity_error(got, ref):
    """SURVEY.md 8d: smallest tol with |got - ref| <= tol*|ref| + tol*max_t|ref_reach| everywhere."""
    scale = np.abs(ref) + np.max(np.abs(ref), axis=0, keepdims=True)
    err = np.abs(got - ref)
    with np.errstate(divide='ignore', invalid='ignore'):
        ratio = np.where(scale > 0, err / scale, np.where(err > 0, np.inf, 0.0))
    return float(ratio.max()) if ratio.size else 0.0


def parity_checks(args, torch, dist, rr, plan, dev, stream, rank, world, down, k, x, idx, local_down, d_lat, ld, n, lateral_row):
    """(1) every rank: zero-state route of the first `check_rows` rows, compared with the CPU oracle on the rank's first
    whole basins (about 60k reaches).  (2) N > 1: the ranks' results gathered over NCCL into params-file order on rank 0
    and compared with rank 0 routing the whole network on its own GPU."""
    from oracle import oracle                                              # the checker, never the thing measured
    from river_route_b200.sharding import shard_by_basin
    cr = min(args.check_rows, d_lat.shape[0])
    d_chk = torch.empty((cr, ld), dtype=torch.float64, device=dev)
    d_q0 = torch.zeros(n, dtype=torch.float64, device=dev)
    plan.route_dev(rr.MODE_RAPID, d_q0.data_ptr(), d_lat.data_ptr(), ld, d_chk.data_ptr(), ld, cr, 1, stream)
    torch.cuda.synchronize()
    outl = np.flatnonzero(local_down < 0)
    m = int(outl[np.searchsorted(outl, min(60_000, n) - 1)]) + 1
    c1, c2, c3, c4 = coefficients(k[idx[:m]], x[idx[:m]], DT, DT)
    indptr, indices = oracle.csc_from_down(local_down[:m])
    ql = d_lat[:cr, :m].cpu().numpy()
    ref, q_ref = np.zeros((cr, m)), np.zeros(m)
    oracle.rapid_route(indptr, indices, oracle.lhs_off_data(c1, indices), c2, c3, c4, q_ref, np.ascontiguousarray(ql), ref, 1)
    got = d_chk[:, :m].cpu().numpy()
    err = torch.tensor([parity_error(got, ref), parity_error(d_q0[:m].cpu().numpy()[None], q_ref[None]),
                        float(np.count_nonzero((got == 0.0) != (ref == 0.0)))], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
    res = {'oracle_parity_max_rel': float(err[0]), 'oracle_state_parity_max_rel': float(err[1]),
           'oracle_zero_pattern_mismatches': int(err[2]),
           'oracle_sample': f'every rank: its first {m} reaches (whole basins; rank 0 figure) x {cr} rows vs oracle/rr_oracle.c'}
    ok = res['oracle_parity_max_rel'] <= PARITY_TOL and res['oracle_state_parity_max_rel'] <= PARITY_TOL
    if dist is not None:
        sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([n], dtype=torch.int64, device=dev))
        sizes = [int(s.item()) for s in sizes]
        n_max = max(sizes)
        mine = torch.zeros((cr, n_max), dtype=torch.float64, device=dev)
        mine[:, :n] = d_chk[:, :n]
        parts = [torch.empty((cr, n_max), dtype=torch.float64, device=dev) for _ in range(world)] if rank == 0 else None
        dist.gather(mine, parts, dst=0)                                    # NCCL over NVLink: outputs only, after the loop
        del mine
        verdict = torch.zeros(2, dtype=torch.float64, device=dev)
        if rank == 0:
            N = down.shape[0]
            ldf = ((N + 31) // 32) * 32
            full = torch.empty((cr, N), dtype=torch.float64, device=dev)
            for r in range(world):
                idx_r, _ = shard_by_basin(down, world, r)
                full[:, torch.from_numpy(idx_r).to(dev)] = parts[r][:, :sizes[r]]
            del parts
            lat_full = torch.zeros((cr, ldf), dtype=torch.float64, device=dev)
            for t in range(cr):
                lat_full[t, :N] = lateral_row(t)
            plan1 = rr.Plan(down, device=dev.index)
            plan1.set_coefficients(*coefficients(k, x, DT, DT))
            out1 = torch.empty((cr, ldf), dtype=torch.float64, device=dev)
            q1 = torch.zeros(N, dtype=torch.float64, device=dev)
            plan1.route_dev(rr.MODE_RAPID, q1.data_ptr(), lat_full.data_ptr(), ldf, out1.data_ptr(), ldf, cr, 1, stream)
            torch.cuda.synchronize()
            diff = (full - out1[:, :N]).abs()
            scale = out1[:, :N].abs() + out1[:, :N].abs().amax(dim=0, keepdim=True)
            rel = torch.where(scale > 0, diff / scale, torch.where(diff > 0, torch.full_like(diff, float('inf')), torch.zeros_like(diff)))
            verdict[0] = rel.max()
            verdict[1] = float(torch.equal(full, out1[:, :N]))
            plan1.close()
            del full, lat_full, out1, q1, diff, scale, rel
            torch.cuda.empty_cache()
        dist.broadcast(verdict, src=0)
        res['sharded_vs_single_gpu_max_rel'] = float(verdict[0])
        res['sharded_vs_single_gpu_bitwise_equal'] = bool(verdict[1])
        res['sharded_vs_single_gpu_sample'] = (f'{cr} rows x all {down.shape[0]} reaches: {world} ranks gathered with NCCL '
                                               f'into params-file order vs one plan of the whole network on rank 0')
        ok = ok and res['sharded_vs_single_gpu_max_rel'] <= PARITY_TOL
    res['parity_ok'] = bool(ok)
    del d_chk
    return res


def e2e_variants(args, rr, plan, timed_host, h_q, h_lat, h_out32, er, n, local_down, local_rank, rank):
    variants = {}
    # (a) the reference kernel's own contract: fp64 discharge array back to the host (rapid_route drop-in)
    h_out64 = rr.pinned_empty((er, n))
    variants['kernel_level_f64_out'] = {
        'value': timed_host(lambda: plan.route_host(rr.MODE_RAPID, h_q, h_lat, h_out64, 1)),
        'h2d_bytes_per_step': int(n * er * 8 + n * 8), 'd2h_bytes_per_step': int(n * er * 8 + n * 8),
        'api': 'Plan.route_host -> rr_route_host (kernels.rapid_route signature)'}
    del h_out64
    # (b) gridded runoff in (float32, ERA5 0.25 degree grid), float32 discharge out: weight table -> route in
    #     one device residency (routers.TransformMuskingum._route_runoff -> rr_runoff_route_host)
    from river_route_b200.transforms import Transform
    n_cells = 721 * 1440
    rng = np.random.default_rng(77 + rank)
    per = rng.integers(4, 9, n)
    indptr = np.zeros(n + 1, dtype=np.int32)
    np.cumsum(per, out=indptr[1:])
    first = rng.integers(0, n_cells - 8, n)
    indices = (np.repeat(first, per) + (np.arange(indptr[-1]) - np.repeat(indptr[:-1], per))).astype(np.int32)
    w = rng.random(indptr[-1])
    w /= np.repeat(np.add.reduceat(w, indptr[:-1]), per)
    tf = Transform(indptr, indices, w, n_cells, area=rng.uniform(1e5, 5e8, n), device=local_rank)
    h_grid = rr.pinned_empty((er, n_cells), dtype=np.float32)
    for t0 in range(0, er, 16):
        blk = h_grid[t0:t0 + 16]
        blk[:] = (rng.gamma(0.3, 2e-3, blk.shape) * (rng.random(blk.shape) < 0.4)).astype(np.float32)
    variants['grid_runoff_to_discharge_f32'] = {
        'value': timed_host(lambda: plan.runoff_route_host(tf, rr.MODE_RAPID, h_q, h_grid, h_out32, 1, as_volumes=True)),
        'h2d_bytes_per_step': int(n_cells * er * 4 + n * 8), 'd2h_bytes_per_step': int(n * er * 4 + n * 8),
        'api': 'Plan.runoff_route_host -> rr_runoff_route_host (weights SpMM + route + float32 cast on the device)',
        'weight_table': f'{int(indptr[-1])} entries, 4-8 cells per river, {n_cells} grid cells'}
    # (c) the same, copying back only the basin outlets (rr_plan_set_output_subset: the device-side form of the
    #     reference's subset writer, docs/tutorial/advanced.md:147-170): neither PCIe direction is the bound any more
    outlets_idx = np.flatnonzero(local_down < 0).astype(np.int32)
    plan.set_output_subset(outlets_idx)
    h_out_sub = rr.pinned_empty((er, outlets_idx.shape[0]), dtype=np.float32)
    variants['grid_runoff_to_outlet_discharge_f32'] = {
        'value': timed_host(lambda: plan.runoff_route_host(tf, rr.MODE_RAPID, h_q, h_grid, h_out_sub, 1, as_volumes=True)),
        'h2d_bytes_per_step': int(n_cells * er * 4 + n * 8),
        'd2h_bytes_per_step': int(outlets_idx.shape[0] * er * 4 + n * 8), 'outlets': int(outlets_idx.shape[0]),
        'api': 'Plan.set_output_subset + Plan.runoff_route_host (all reaches routed, outlet columns copied back)'}
    plan.set_output_subset(None)
    tf.close()
    del h_grid, h_out_sub
    # (d) lateral inflows stored as float32 (a qlateral variable may be; the reference upcasts on the host,
    #     TransformMuskingum.py:36): the rows cross PCIe as stored and are upcast -- exactly -- by the staging kernel
    h_lat32 = rr.pinned_empty((er, n), dtype=np.float32)
    for t0 in range(0, er, 32):
        h_lat32[t0:t0 + 32] = h_lat[t0:t0 + 32]
    variants['f32_lateral_in_f32_out'] = {
        'value': timed_host(lambda: plan.route_host(rr.MODE_RAPID, h_q, h_lat32, h_out32, 1)),
        'h2d_bytes_per_step': int(n * er * 4 + n * 8), 'd2h_bytes_per_step': int(n * er * 4 + n * 8),
        'api': 'Plan.route_host with a float32 lateral array -> rr_route_host_typed'}
    # (e) the class API on files: RapidMuskingum(config).route() with a float32 qlateral netCDF and the discharge
    #     netCDF on tmpfs.  Slabs go file -> pinned buffer -> GPU -> pinned buffer -> file; the network plan is reused by
    #     the second (timed) route().  On this image the files are classic netCDF through scipy (big-endian on disk, no
    #     netCDF4 / HDF5 stack), so the number is bounded by single-threaded byte swapping, not by PCIe.
    try:
        variants['router_files'] = router_files_variant(args, rr, n, local_down, h_lat32, min(er, 64))
    except Exception as e:                                   # optional variant: never takes the bench line down
        variants['router_files'] = {'error': f'{type(e).__name__}: {e}'}
    return variants


def router_files_variant(args, rr, n, local_down, h_lat32, rows):
    import shutil
    import tempfile
    import pandas as pd
    from river_route_b200 import ncio, synth
    tmp = tempfile.mkdtemp(prefix='rr_bench_', dir='/dev/shm' if os.path.isdir('/dev/shm') else None)
    try:
        ids = np.arange(n, dtype=np.int64) + 1
        k, x = synth.muskingum_params(args.reaches, 4)
        pd.DataFrame({'river_id': ids, 'downstream_river_id': np.where(local_down >= 0, ids[np.where(local_down >= 0, local_down, 0)], -1),
                      'k': k[:n], 'x': x[:n]}).to_parquet(os.path.join(tmp, 'params.parquet'))
        with ncio.open_nc(os.path.join(tmp, 'ql.nc'), 'w') as nc:
            nc.createDimension('time', rows)
            nc.createDimension('river_id', n)
            tv = nc.createVariable('time', 'f8', ('time',))
            tv.units = 'seconds since 2022-01-01 00:00:00'
            tv[:] = np.arange(rows) * float(DT)
            nc.createVariable('river_id', 'i4', ('river_id',))[:] = ids.astype(np.int32)
            nc.createVariable('qlateral', 'f4', ('time', 'river_id'))[:] = h_lat32[:rows]
        r = rr.RapidMuskingum(params_file=os.path.join(tmp, 'params.parquet'), qlateral_files=[os.path.join(tmp, 'ql.nc')],
                              discharge_dir=tmp, log=False)
        t0 = time.perf_counter()
        r.route()                                             # builds the plan, pins the slab buffers
        first = time.perf_counter() - t0
        t0 = time.perf_counter()
        r._set_network_dependent_vectors()
        setup = time.perf_counter() - t0
        t0 = time.perf_counter()
        r._execute_routing()
        execute = time.perf_counter() - t0
        size = os.path.getsize(os.path.join(tmp, 'discharge_ql.nc'))
        return {'value': n * rows / execute, 'rows': rows, 'first_route_s': first, 'params_read_and_plan_reuse_s': setup,
                'execute_routing_s': execute, 'h2d_bytes_per_step': int(n * rows * 4 + n * 8),
                'd2h_bytes_per_step': int(n * rows * 4 + n * 8), 'discharge_file_bytes': int(size), 'netcdf_backend': ncio.backend(),
                'api': 'RapidMuskingum(params_file, qlateral_files, discharge_dir).route(): float32 qlateral netCDF in, '
                       'discharge netCDF out, both on tmpfs; value = reaches x rows / _execute_routing wall time'}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == '__main__':
    main()
