"""
Flood-warning products without a GPU: the 'exceed_<label>' names, the numpy definitions the device follows for
exceedance and horizon peaks, and the host logic of ``set_ensemble_statistics(..., thresholds=, horizon=)`` -- the
thresholds table, the peak merge across time slabs and the file layout -- with the device calls replaced by the
oracle-backed stand-in ``fake_route_ensemble_stats_host`` below (plus tests/fakes.py).
"""
import numpy as np
import pandas as pd
import pytest

import river_route_b200 as rr
from river_route_b200 import ncio, plan as plan_mod
from river_route_b200.plan import parse_statistics
from oracle import oracle
from tests import fakes
from tests.helpers import network_arrays
from tests.test_ensemble_stats_cpu import _members, numpy_statistic


def exceedance(x, thr):
    """np.mean(x > thr, axis=0): the device's definition."""
    return np.mean(x > thr, axis=0)


def statistic(x, name, thr_by_label):
    return exceedance(x, thr_by_label[name[7:]]) if name.startswith('exceed_') else numpy_statistic(x, name)


def test_exceed_names():
    assert parse_statistics(['mean', 'exceed_rp2', 'p50', 'exceed_rp100'], ('rp2', 'rp10', 'rp100')) == [
        ('mean', 0, 0), ('exceed_rp2', 5, 0), ('p50', 4, 50), ('exceed_rp100', 5, 2)]
    assert parse_statistics('exceed_x', ['x']) == [('exceed_x', 5, 0)]
    for names, labels, msg in [(['exceed_rp2'], (), 'unknown ensemble statistic'),
                               (['exceed_rp5'], ('rp2',), 'unknown ensemble statistic'),
                               (['exceed_'], ('rp2',), 'unknown ensemble statistic'),
                               (['exceed_rp2'], ('rp2', 'rp2'), 'duplicate threshold labels'),
                               (['exceed_rp2', 'exceed_rp2'], ('rp2',), 'duplicate ensemble statistics'),
                               (['mean'] + [f'exceed_l{i}' for i in range(16)], [f'l{i}' for i in range(16)], 'between')]:
        with pytest.raises(ValueError, match=msg):
            parse_statistics(names, labels)
    assert len(parse_statistics([f'exceed_l{i}' for i in range(16)], [f'l{i}' for i in range(16)])) == 16


def test_numpy_definitions():
    """What the kernel reproduces: strict '>' (ties do not count), NaN never exceeded, M = 1, and peaks as max / first
    argmax over the rows."""
    x = np.array([[[1.0, 2.0, 0.0]], [[3.0, 2.0, 0.0]], [[2.0, 5.0, 0.0]]])    # (M=3, rows=1, n=3)
    thr = np.array([2.0, np.nan, 0.0])
    assert np.array_equal(exceedance(x, thr), [[1 / 3, 0.0, 0.0]])
    assert np.array_equal(exceedance(x[:1], np.array([0.5, 2.0, -1.0])), [[1.0, 0.0, 1.0]])   # M = 1
    # count / M with one IEEE division, as the kernel does
    rng = np.random.default_rng(1)
    for M in (1, 2, 5, 51, 64):
        x = np.round(rng.gamma(0.5, 4.0, (M, 6, 40)))
        thr = x[rng.integers(0, M, 40), rng.integers(0, 6, 40), np.arange(40)]
        thr[::5] = np.nan
        cnt = (x > thr).sum(axis=0)
        assert np.array_equal(exceedance(x, thr), cnt.astype(np.float64) / M), M
    rows = np.array([[1.0, 3.0, 0.5], [3.0, 3.0, 0.5], [2.0, 1.0, 0.5], [3.0, 0.0, 0.7]])
    peak, row = np.full(3, -np.inf), np.zeros(3, dtype=np.int64)
    for t, r in enumerate(rows):                                                  # the kernel's running update
        better = r > peak
        peak[better], row[better] = r[better], t
    assert np.array_equal(peak, rows.max(axis=0)) and np.array_equal(row, rows.argmax(axis=0))
    assert np.array_equal(row, [1, 0, 3])


def fake_route_ensemble_stats_host(self, mode, q_init, laterals, stats, outs, substeps, resample=1, q_final=None,
                                   peaks=None):
    """Oracle-backed stand-in for Plan.route_ensemble_stats_host with thresholds and peaks."""
    labels = getattr(self, 'threshold_labels', ())
    parsed = parse_statistics(stats, labels)
    assert outs is not None or peaks is not None
    M = len(laterals)
    T = outs[0].shape[0] * resample if outs is not None else laterals[0].shape[0]
    members, finals = np.empty((M, T // resample, self.n_out)), np.empty((M, self.n))
    for m in range(M):
        q = (q_init if q_init.ndim == 1 else q_init[m]).copy()
        fakes._finish(self, fakes._route(self, mode, q, np.ascontiguousarray(laterals[m], dtype=np.float64), T, substeps),
                      members[m], resample)
        finals[m] = q
    sub = getattr(self, '_fake_subset', None)
    thr = {k: (v if sub is None else v[sub]) for k, v in getattr(self, '_fake_thr', {}).items()}
    for s, (name, _, _) in enumerate(parsed):
        rows = statistic(members, name, thr)
        if outs is not None:
            outs[s][...] = rows.astype(outs[s].dtype)
        if peaks is not None:
            peaks[0][s], peaks[1][s] = rows.max(axis=0), rows.argmax(axis=0)
    if q_final is not None:
        q_final[...] = finals
    return finals.mean(axis=0)


@pytest.fixture
def host_only(monkeypatch):
    fakes.install(monkeypatch.setattr)
    real = plan_mod.Plan.set_thresholds

    def set_thresholds(self, thresholds=None):
        real(self, thresholds)                                                    # host-side: validates, keeps labels
        self._fake_thr = {k: np.asarray(v, dtype=np.float64) for k, v in (thresholds or {}).items()}
    monkeypatch.setattr(plan_mod.Plan, 'set_thresholds', set_thresholds)
    monkeypatch.setattr(plan_mod.Plan, 'route_ensemble_stats_host', fake_route_ensemble_stats_host)


def _reference_members(c, k, pick):
    a = network_arrays(c['down'], c['k'], c['x'], 3600, 3600)
    members, finals = [], []
    for ql in c['laterals']:
        q, ref = c['q0'].copy(), np.zeros((c['T'], c['n']))
        oracle.rapid_route(a['indptr'], a['indices'], a['lhs_off'], a['c2'], a['c3'], a['c4_dt'], q, ql, ref, 1)
        finals.append(q)
        ref = ref.reshape(c['T'] // k, k, c['n']).mean(axis=1) if k > 1 else ref
        members.append(ref if pick is None else ref[:, pick])
    return np.array(members), np.array(finals)


NAMES = ['mean', 'p50', 'exceed_rp2', 'max', 'exceed_rp10']


@pytest.mark.parametrize('horizon', ['steps', 'peaks', 'both'])
@pytest.mark.parametrize('k,slab_rows,subset,as_frame', [(1, 8, False, False), (2, 16, True, True)])
def test_router_writes_warnings(tmp_path, host_only, monkeypatch, horizon, k, slab_rows, subset, as_frame):
    c = _members(tmp_path, T=48)
    T, n, ids = c['T'], c['n'], c['ids']
    monkeypatch.setenv('RR_ROUTER_SLAB_ROWS', str(slab_rows))
    pick = np.array([n - 1, 3, 50, 3, 0]) if subset else None
    members, finals = _reference_members(c, k, pick)
    full_members, _ = _reference_members(c, k, None)
    # thresholds: rp2 from a member (exact ties), rp10 well above; the first 20 rivers missing, one id not in the network
    rp2 = full_members[2, 5].astype(np.float32)
    rp10 = (full_members.max(axis=(0, 1)) * 0.9).astype(np.float32)
    table = pd.DataFrame({'rp10': np.append(rp10[20:], 7.0), 'river_id': np.append(ids[20:], 10 ** 9),
                          'rp2': np.append(rp2[20:], 7.0), 'unused': 1.0})[::-1]
    if not as_frame:
        table.to_parquet(tmp_path / 'rp.parquet')
        table = str(tmp_path / 'rp.parquet')
    thr = {lab: np.where(np.arange(n) < 20, np.nan, v.astype(np.float64)) for lab, v in (('rp2', rp2), ('rp10', rp10))}
    if subset:
        thr = {lab: v[pick] for lab, v in thr.items()}
    path = str(tmp_path / 'warn.nc')
    r = rr.RapidMuskingum(**dict(c['cfg'], dt_discharge=3600 * k)).set_ensemble_statistics(path, NAMES, thresholds=table,
                                                                                         horizon=horizon)
    if subset:
        r.set_output_rivers(ids[pick])
    r.route()
    ref = {s: statistic(members, s, thr) for s in NAMES}
    with ncio.open_nc(path) as ds:
        per_step = [f'Q_{s}' for s in NAMES] if horizon != 'peaks' else []
        peak_vars = [f'Q_{s}_peak{x}' for s in NAMES for x in ('', '_time')] if horizon != 'steps' else []
        assert sorted(ds.variables) == sorted(['time', 'river_id'] + per_step + peak_vars)
        tv = ds.variables['time']
        units = ncio.attrs_of(tv)['units']
        assert units == 'seconds since 2023-03-01 00:00:00' and ncio.read_array(tv).shape == (T // k,)
        for s in NAMES:
            exc = s.startswith('exceed_')
            for v_name in ([f'Q_{s}'] if per_step else []) + ([f'Q_{s}_peak'] if peak_vars else []):
                at = ncio.attrs_of(ds.variables[v_name])
                assert at['units'] == ('1' if exc else 'm3 s-1') and (at.get('threshold') == s[7:] if exc else 'threshold' not in at)
            if per_step:
                v = ds.variables[f'Q_{s}']
                assert tuple(v.dimensions) == ('time', 'river_id')
                assert np.array_equal(ncio.read_array(v), ref[s].astype(np.float32)), s
            if peak_vars:
                pv, tv_ = ds.variables[f'Q_{s}_peak'], ds.variables[f'Q_{s}_peak_time']
                assert tuple(pv.dimensions) == ('river_id',) and tuple(tv_.dimensions) == ('river_id',)
                assert ncio.attrs_of(tv_)['units'] == units
                got_t = ncio.read_array(tv_)
                assert got_t.dtype == np.float64
                assert np.array_equal(ncio.read_array(pv), ref[s].max(axis=0).astype(np.float32)), s
                assert np.array_equal(got_t, ref[s].argmax(axis=0) * 3600.0 * k), s
        assert np.array_equal(ncio.read_array(ds.variables['river_id']), ids[pick] if subset else ids)
    # rivers missing from the table are never above their (NaN) threshold
    if not subset:
        assert (ref['exceed_rp2'][:, :20] == 0).all() and ref['exceed_rp2'][:, 20:].any()
    assert np.array_equal(r.channel_state, finals.mean(axis=0))


def test_peaks_merge_across_slabs_keeps_the_first_tie(tmp_path, host_only, monkeypatch):
    """The per-slab peaks are merged with a strict '>': a maximum reached in two slabs keeps the earlier row."""
    c = _members(tmp_path, T=32)
    monkeypatch.setenv('RR_ROUTER_SLAB_ROWS', '16')
    flat = np.full((32, c['n']), 0.0)
    flat[10] = flat[20] = 5.0                                                     # equal peaks in slab 0 and slab 1
    flat[25, :7] = 9.0                                                            # a later, larger one on a few rivers
    real = fake_route_ensemble_stats_host

    def fixed(self, mode, q_init, laterals, stats, outs, substeps, resample=1, q_final=None, peaks=None):
        mean = real(self, mode, q_init, laterals, stats, outs, substeps, resample, q_final, peaks)
        t0 = fixed.row
        fixed.row += laterals[0].shape[0]
        rows = flat[t0:fixed.row]
        for s in range(len(stats)):
            if outs is not None:
                outs[s][...] = rows
            if peaks is not None:
                peaks[0][s], peaks[1][s] = rows.max(axis=0), rows.argmax(axis=0)
        return mean
    fixed.row = 0
    monkeypatch.setattr(plan_mod.Plan, 'route_ensemble_stats_host', fixed)
    path = str(tmp_path / 'w.nc')
    rr.RapidMuskingum(**c['cfg']).set_ensemble_statistics(path, ['mean'], horizon='both').route()
    with ncio.open_nc(path) as ds:
        got_t = ncio.read_array(ds.variables['Q_mean_peak_time'])
        assert np.array_equal(ncio.read_array(ds.variables['Q_mean_peak']), flat.max(axis=0).astype(np.float32))
    assert np.array_equal(got_t, flat.argmax(axis=0) * 3600.0)
    assert (got_t[:7] == 25 * 3600.0).all() and (got_t[7:] == 10 * 3600.0).all()


def test_router_refusals(tmp_path, host_only):
    c = _members(tmp_path, M=2)
    path = str(tmp_path / 'w.nc')
    ids = c['ids']
    with pytest.raises(ValueError, match='horizon'):
        rr.RapidMuskingum(**c['cfg']).set_ensemble_statistics(path, ['mean'], horizon='peak')
    with pytest.raises(ValueError, match='unknown ensemble statistic'):
        rr.RapidMuskingum(**c['cfg']).set_ensemble_statistics(path, ['exceed_rp2'])
    with pytest.raises(ValueError, match="'river_id' column"):
        rr.RapidMuskingum(**c['cfg']).set_ensemble_statistics(path, ['mean'], thresholds=pd.DataFrame({'rp2': [1.0]}))
    dup = pd.DataFrame({'river_id': [ids[0], ids[0]], 'rp2': [1.0, 2.0]})
    with pytest.raises(ValueError, match='more than once'):
        rr.RapidMuskingum(**c['cfg']).set_ensemble_statistics(path, ['exceed_rp2'], thresholds=dup).route()
    none = pd.DataFrame({'river_id': [10 ** 9, 10 ** 9 + 1], 'rp2': [1.0, 2.0]})
    with pytest.raises(ValueError, match='no river id'):
        rr.RapidMuskingum(**c['cfg']).set_ensemble_statistics(path, ['exceed_rp2'], thresholds=none).route()


def test_plain_statistics_keep_todays_call(tmp_path, host_only, monkeypatch):
    """Without exceed names and with horizon='steps' the plan call has exactly the earlier arguments, even when a
    thresholds table is given."""
    c = _members(tmp_path, M=3)
    seen = []

    def spy(self, mode, q_init, lats, stats, outs, substeps, resample=1, q_final=None):
        seen.append(stats)
        return fake_route_ensemble_stats_host(self, mode, q_init, lats, stats, outs, substeps, resample, q_final)
    monkeypatch.setattr(plan_mod.Plan, 'route_ensemble_stats_host', spy)
    table = pd.DataFrame({'river_id': c['ids'], 'rp2': np.ones(c['n'])})
    r = rr.RapidMuskingum(**c['cfg']).set_ensemble_statistics(str(tmp_path / 'w.nc'), ['mean', 'p50'], thresholds=table)
    r.route()
    assert seen and all(s == ['mean', 'p50'] for s in seen)
    assert r.plan.threshold_labels == ()
