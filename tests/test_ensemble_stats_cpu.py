"""
Ensemble statistics without a GPU: the statistic names, the numpy definitions the device kernel follows (pinned here
against numpy itself for every member count and percentile the kernel accepts), and the host logic of
``TransformMuskingum.set_ensemble_statistics`` with the device calls replaced by oracle-backed stand-ins
(tests/fakes.py plus ``fake_route_ensemble_stats_host`` below).
"""
import os

import numpy as np
import pandas as pd
import pytest

import river_route_b200 as rr
from river_route_b200 import ncio, plan as plan_mod, synth
from river_route_b200.plan import parse_statistics
from oracle import oracle
from tests import fakes
from tests.helpers import network_arrays

STATS = ['mean', 'std', 'min', 'max', 'p0', 'p25', 'p50', 'p75', 'p90', 'p100']


def numpy_statistic(x, name):
    """The statistic over axis 0 of the stacked (members, rows, n) fp64 array, as numpy computes it."""
    return {'mean': np.mean, 'std': np.std, 'min': np.min, 'max': np.max}[name](x, axis=0) if name[0] != 'p' \
        else np.percentile(x, int(name[1:]), axis=0)


def spec_percentile(x, q):
    """np.percentile's 'linear' method as the device computes it (rr_stats.cu): sorted members, lo / hi / g from the
    two IEEE operations numpy uses, then numpy's _lerp."""
    M = x.shape[0]
    v = (M - 1) * (q / 100.0)
    lo = int(np.floor(v))
    hi = min(lo + 1, M - 1)
    g = v - lo
    srt = np.sort(x, axis=0)
    a, b = srt[lo], srt[hi]
    diff = b - a
    return a + diff * g if g < 0.5 else b - diff * (1 - g)


def spec_mean_std(x):
    acc = x[0].copy()
    for m in range(1, x.shape[0]):
        acc = acc + x[m]
    mean = acc / x.shape[0]
    ss = (x[0] - mean) * (x[0] - mean)
    for m in range(1, x.shape[0]):
        d = x[m] - mean
        ss = ss + d * d
    return mean, np.sqrt(ss / x.shape[0])


def test_statistic_names():
    assert parse_statistics(['mean', 'std', 'min', 'max', 'p0', 'p25', 'p100']) == [
        ('mean', 0, 0), ('std', 1, 0), ('min', 2, 0), ('max', 3, 0), ('p0', 4, 0), ('p25', 4, 25), ('p100', 4, 100)]
    assert parse_statistics('p50') == [('p50', 4, 50)]
    for bad, msg in [(['avg'], 'unknown'), (['p101'], 'unknown'), (['p05'], 'unknown'), (['p-1'], 'unknown'),
                     (['P50'], 'unknown'), (['p'], 'unknown'), ([3], 'strings'), (['mean', 'mean'], 'duplicate'),
                     ([], 'between'), ([f'p{q}' for q in range(17)], 'between')]:
        with pytest.raises(ValueError, match=msg):
            parse_statistics(bad)


def test_spec_formulas_are_numpy_bit_for_bit():
    """For every M in 1..64 and every integer q in 0..100, on non-negative data with many ties and zeros."""
    rng = np.random.default_rng(0)
    for M in range(1, 65):
        x = rng.gamma(0.7, 30.0, (M, 4, 50)) * (rng.random((M, 4, 50)) < 0.8)
        x[:, :, :10] = np.round(x[:, :, :10] / 10.0)                      # exact ties
        x[:, 0, 10:20] = x[0, 0, 10:20]                                    # every member equal
        pct = np.percentile(x, np.arange(101), axis=0)
        for q in range(101):
            assert np.array_equal(spec_percentile(x, q), pct[q]), (M, q)
        mean, std = spec_mean_std(x)
        assert np.array_equal(mean, np.mean(x, axis=0)) and np.array_equal(std, np.std(x, axis=0)), M


def fake_route_ensemble_stats_host(self, mode, q_init, laterals, stats, outs, substeps, resample=1, q_final=None):
    """Oracle-backed stand-in for Plan.route_ensemble_stats_host: the members through the oracle, the device's output
    tail (subset, resample), then numpy's statistics over the stacked fp64 member outputs."""
    parsed = parse_statistics(stats)
    M, T = len(laterals), outs[0].shape[0] * resample
    assert len(outs) == len(parsed) and all(o.shape == (T // resample, self.n_out) for o in outs)
    members, finals = np.empty((M, T // resample, self.n_out)), np.empty((M, self.n))
    for m in range(M):
        q = (q_init if q_init.ndim == 1 else q_init[m]).copy()
        fakes._finish(self, fakes._route(self, mode, q, np.ascontiguousarray(laterals[m], dtype=np.float64), T, substeps),
                      members[m], resample)
        finals[m] = q
    for o, (name, _, _) in zip(outs, parsed):
        o[...] = numpy_statistic(members, name).astype(o.dtype)
    if q_final is not None:
        q_final[...] = finals
    return np.array(list(finals)).mean(axis=0)


@pytest.fixture
def host_only(monkeypatch):
    fakes.install(monkeypatch.setattr)
    monkeypatch.setattr(plan_mod.Plan, 'route_ensemble_stats_host', fake_route_ensemble_stats_host)


def _members(tmp_path, n=180, T=40, M=5, f32=False):
    down = synth.forest(n, 3, seed=12, depth_bias=0.6)
    kk, x = synth.muskingum_params(n, 12)
    ids = np.arange(n, dtype=np.int64) + 7
    params = str(tmp_path / 'p.parquet')
    pd.DataFrame({'river_id': ids, 'downstream_river_id': np.where(down >= 0, ids[np.where(down >= 0, down, 0)], -1),
                  'k': kk, 'x': x}).to_parquet(params)
    q0 = np.random.default_rng(5).uniform(0, 25, n)
    pd.DataFrame({'Q': q0}).to_parquet(tmp_path / 'q0.parquet')
    files, laterals = [], []
    base = synth.lateral_volumes(T, n, 60)
    for m in range(M):
        ql = base * np.random.default_rng(70 + m).lognormal(0, 0.3, (1, n))
        if f32:
            ql = ql.astype(np.float32)
        path = str(tmp_path / f'member_{m}.nc')
        with ncio.open_nc(path, 'w') as nc:
            nc.createDimension('time', T)
            nc.createDimension('river_id', n)
            tv = nc.createVariable('time', 'f8', ('time',))
            tv.units = 'seconds since 2023-03-01 00:00:00'
            tv[:] = np.arange(T) * 3600.0
            nc.createVariable('river_id', 'i4', ('river_id',))[:] = ids.astype(np.int32)
            nc.createVariable('qlateral', 'f4' if f32 else 'f8', ('time', 'river_id'))[:] = ql
        files.append(path)
        laterals.append(ql.astype(np.float64))
    out_dir = tmp_path / 'out'
    out_dir.mkdir()
    cfg = dict(params_file=params, qlateral_files=files, discharge_dir=str(out_dir),
               channel_state_init_file=str(tmp_path / 'q0.parquet'), runoff_processing_mode='ensemble',
               channel_state_final_file=str(tmp_path / 'final.parquet'), log=False)
    return dict(cfg=cfg, down=down, k=kk, x=x, ids=ids, q0=q0, laterals=laterals, n=n, T=T, M=M, out_dir=out_dir)


@pytest.mark.parametrize('k,slab_rows,subset,f32', [(1, 0, False, False), (2, 16, True, True), (4, 8, False, False)])
def test_router_writes_one_statistics_file(tmp_path, host_only, monkeypatch, k, slab_rows, subset, f32):
    c = _members(tmp_path, f32=f32)
    if slab_rows:
        monkeypatch.setenv('RR_ROUTER_SLAB_ROWS', str(slab_rows))
    calls = []
    real = plan_mod.Plan.route_ensemble_stats_host

    def spy(self, mode, q_init, lats, stats, outs, substeps, resample=1, q_final=None):
        calls.append((len(lats), lats[0].shape[0], q_init.ndim, resample))
        return real(self, mode, q_init, lats, stats, outs, substeps, resample=resample, q_final=q_final)
    monkeypatch.setattr(plan_mod.Plan, 'route_ensemble_stats_host', spy)
    pick = np.array([c['n'] - 1, 3, 50, 3]) if subset else None
    stats_path = str(tmp_path / 'stats.nc')
    r = rr.RapidMuskingum(**dict(c['cfg'], dt_discharge=3600 * k)).set_ensemble_statistics(stats_path, STATS)
    if subset:
        r.set_output_rivers(c['ids'][pick])
    r.route()
    T, n, M = c['T'], c['n'], c['M']
    # every call routes all members of one time slab; later slabs chain the members' own states
    assert all(cl[0] == M and cl[3] == k for cl in calls) and sum(cl[1] for cl in calls) == T
    assert calls[0][2] == 1 and all(cl[2] == 2 for cl in calls[1:])
    if slab_rows:
        assert len(calls) == -(-T // slab_rows)
    assert not any(f.startswith('discharge') for f in os.listdir(c['out_dir'])), 'member files were written'
    a = network_arrays(c['down'], c['k'], c['x'], 3600, 3600)
    members, finals = [], []
    for ql in c['laterals']:
        q, ref = c['q0'].copy(), np.zeros((T, n))
        oracle.rapid_route(a['indptr'], a['indices'], a['lhs_off'], a['c2'], a['c3'], a['c4_dt'], q, ql, ref, 1)
        finals.append(q)
        ref = ref.reshape(T // k, k, n).mean(axis=1) if k > 1 else ref
        members.append(ref[:, pick] if subset else ref)
    members = np.array(members)
    with ncio.open_nc(stats_path) as ds:
        assert sorted(ds.variables) == sorted(['time', 'river_id'] + [f'Q_{s}' for s in STATS])
        for s in STATS:
            v = ds.variables[f'Q_{s}']
            assert tuple(v.dimensions) == ('time', 'river_id')
            got = ncio.read_array(v)
            assert got.dtype == np.float32 and np.array_equal(got, numpy_statistic(members, s).astype(np.float32)), s
            assert (ncio.attrs_of(v).get('percentile') == int(s[1:])) if s[0] == 'p' else 'percentile' not in ncio.attrs_of(v)
        tv = ds.variables['time']
        dates = ncio.decode_time(ncio.read_array(tv), ncio.attrs_of(tv)['units'])
        rid = ncio.read_array(ds.variables['river_id'])
    assert dates.shape == (T // k,) and np.all(np.diff(dates) == np.timedelta64(3600 * k, 's'))
    assert dates[0] == np.datetime64('2023-03-01T00:00:00')
    assert np.array_equal(rid, c['ids'][pick] if subset else c['ids'])
    assert np.array_equal(r.channel_state, np.array(finals).mean(axis=0))
    assert np.array_equal(pd.read_parquet(tmp_path / 'final.parquet')['Q'].values, r.channel_state)


def test_router_rejects_unsupported_runs(tmp_path, host_only):
    from river_route_b200.distributed import Shard
    c = _members(tmp_path, M=2)
    stats_path = str(tmp_path / 'stats.nc')
    with pytest.raises(ValueError, match='unknown ensemble statistic'):
        rr.RapidMuskingum(**c['cfg']).set_ensemble_statistics(stats_path, ['mean', 'median'])
    cases = [
        (rr.RapidMuskingum(**dict(c['cfg'], runoff_processing_mode='sequential')), "runoff_processing_mode='ensemble'"),
        (rr.UnitMuskingum(**c['cfg']), 'UnitMuskingum'),
        (rr.RapidMuskingum(**c['cfg']).set_write_discharges(lambda *a: None), 'set_write_discharges'),
        (rr.RapidMuskingum(_shard=Shard(0, 2), **c['cfg']), 'basin-sharded'),
    ]
    many = dict(c['cfg'], qlateral_files=[c['cfg']['qlateral_files'][0]] * 65, discharge_dir=None,
                discharge_files=[str(tmp_path / 'out' / f'd{m}.nc') for m in range(65)])
    cases.append((rr.RapidMuskingum(**many), 'at most 64 members'))
    from tests.test_routers_gpu import _grid_case
    g = _grid_case(tmp_path, n=600, T=12, ny=9, nx=14)
    grid_cfg = dict(params_file=g['params'], grid_runoff_files=[x[0] for x in g['grids']],
                    grid_weights_file=str(tmp_path / 'weights.nc'), discharge_dir=str(c['out_dir']), var_x='lon',
                    var_y='lat', runoff_processing_mode='ensemble', log=False)
    cases.append((rr.RapidMuskingum(**grid_cfg), 'qlateral_files'))
    for router, msg in cases:
        with pytest.raises(ValueError, match=msg):
            router.set_ensemble_statistics(stats_path).route()
    assert not os.path.exists(stats_path)
