"""
Flood-warning products on the B200: threshold exceedance (RR_STAT_EXCEED) and horizon peaks of the ensemble statistics,
from the kernel (rr_ensemble_stats_dev_ex) through the routed call (Plan.route_ensemble_stats_host(peaks=...)) to the
router's file.  Everything must equal numpy on the stacked fp64 member values bit for bit: np.mean(x > thr, axis=0) for
exceedance, rows.max(axis=0) / rows.argmax(axis=0) for the peaks.
"""
import ctypes as C
import os

import numpy as np
import pandas as pd
import pytest

import river_route_b200 as rr
from river_route_b200 import _lib, ncio, synth
from river_route_b200.plan import ensemble_stats_dev
from tests.conftest import require_cuda
from tests.test_ensemble_stats_cpu import numpy_statistic

pytestmark = pytest.mark.gpu
LABELS = ('a', 'b', 'c')
MIXED = ['mean', 'exceed_a', 'p50', 'max', 'exceed_c', 'std', 'exceed_b', 'p90']   # sorting instantiation
EXCEED_ONLY = ['exceed_b', 'exceed_a', 'min']


@pytest.fixture(autouse=True)
def _cuda():
    require_cuda()


@pytest.fixture
def chunk_rows():
    def set_rows(rows):
        if rows:
            os.environ['RR_STREAM_CHUNK_ROWS'] = str(rows)
        else:
            os.environ.pop('RR_STREAM_CHUNK_ROWS', None)
    yield set_rows
    os.environ.pop('RR_STREAM_CHUNK_ROWS', None)


def reference(x, names, thr):
    """Statistic rows of the stacked (M, rows, n) fp64 array, thr (labels, n)."""
    return [np.mean(x > thr[LABELS.index(s[7:])], axis=0) if s.startswith('exceed_') else numpy_statistic(x, s)
            for s in names]


def _thresholds(x, rng):
    """Thresholds drawn from the member values themselves (exact ties with x), with NaN entries."""
    M, rows, n = x.shape
    thr = np.stack([x[rng.integers(0, M, n), rng.integers(0, rows, n), np.arange(n)] for _ in LABELS])
    thr[1, ::7] = np.nan
    thr[2, 3::11] = 0.0
    return thr


@pytest.mark.parametrize('M', [1, 2, 5, 51, 64])
def test_kernel_exceedance_and_peaks_are_numpy_bit_for_bit(M):
    import torch
    rng = np.random.default_rng(100 + M)
    rows, n = 9, 700 + 13
    ld = n + 29
    x = rng.gamma(0.5, 20.0, (M, rows, ld)) * (rng.random((M, rows, ld)) < 0.7)
    x[:, :, :300] = np.round(x[:, :, :300] / 8.0)                                 # exact ties, repeated maxima
    thr = _thresholds(x[:, :, :n], rng)
    ldt = n + 3
    thr_pad = np.full((len(LABELS), ldt), -1.0)
    thr_pad[:, :n] = thr
    xd, thr_d = torch.from_numpy(x).cuda(), torch.from_numpy(thr_pad).cuda()
    sub = np.array([n - 1, 0, 5, 5, 300, 0, 31, 32], dtype=np.int32)
    sub_d = torch.from_numpy(sub).cuda()
    cuts = [0, 4, 5, rows]                                                        # three launches, row0 offsets
    for names in (MIXED, EXCEED_ONLY):
        ref = reference(x[:, :, :n], names, thr)
        for dt in (torch.float64, torch.float32):
            for subset in (False, True):
                n_out = sub.shape[0] if subset else n
                ldo, ldk = n_out + 5, n_out + 3
                outs = [torch.full((rows, ldo), float('nan'), dtype=dt, device='cuda') for _ in names]
                peak = torch.full((len(names), ldk), float('-inf'), dtype=torch.float64, device='cuda')
                peak[:, n_out:] = float('nan')
                prow = torch.full((len(names), ldk), -7, dtype=torch.int32, device='cuda')
                for r0, r1 in zip(cuts[:-1], cuts[1:]):
                    ensemble_stats_dev(names, M, xd.data_ptr() + r0 * ld * 8, rows * ld, ld, r1 - r0, n_out,
                                       [o.data_ptr() + r0 * ldo * o.element_size() for o in outs], ldo, dt == torch.float32,
                                       sub_d.data_ptr() if subset else 0, thresholds=LABELS, thr_ptr=thr_d.data_ptr(),
                                       ldt=ldt, peak_ptrs=(peak.data_ptr(), prow.data_ptr()), ldk=ldk, row0=r0)
                torch.cuda.synchronize()
                pk, pr = peak.cpu().numpy(), prow.cpu().numpy()
                for s, o in enumerate(outs):
                    want = ref[s][:, sub] if subset else ref[s]
                    got = o.cpu().numpy()
                    assert np.array_equal(got[:, :n_out], want.astype(got.dtype)), (M, names[s], dt, subset)
                    assert np.isnan(got[:, n_out:]).all()
                    assert np.array_equal(pk[s, :n_out], want.max(axis=0)), (M, names[s], subset)
                    assert np.array_equal(pr[s, :n_out], want.argmax(axis=0)), (M, names[s], subset)
                    assert np.isnan(pk[s, n_out:]).all() and (pr[s, n_out:] == -7).all()   # nothing past n_out
        # peaks without per-step rows
        peak = torch.full((len(names), n), float('-inf'), dtype=torch.float64, device='cuda')
        prow = torch.zeros((len(names), n), dtype=torch.int32, device='cuda')
        ensemble_stats_dev(names, M, xd.data_ptr(), rows * ld, ld, rows, n, None, 0, False, thresholds=LABELS,
                           thr_ptr=thr_d.data_ptr(), ldt=ldt, peak_ptrs=(peak.data_ptr(), prow.data_ptr()), ldk=n)
        torch.cuda.synchronize()
        for s in range(len(names)):
            assert np.array_equal(peak[s].cpu().numpy(), ref[s].max(axis=0)) and \
                np.array_equal(prow[s].cpu().numpy(), ref[s].argmax(axis=0)), names[s]


def test_kernel_validation_errors():
    import torch
    M, rows, n = 3, 2, 64
    xd = torch.zeros((M, rows, n), dtype=torch.float64, device='cuda')
    out = torch.empty((rows, n), dtype=torch.float64, device='cuda')
    peak = torch.empty((1, n), dtype=torch.float64, device='cuda')

    def raw(kind, q, thr, outs, pk, pr):
        spec = _lib.StatsSpec()
        spec.n_stats, spec.kind[0], spec.q[0] = 1, kind, q
        arr = (C.c_void_p * 1)(outs) if outs else None
        _lib.check(_lib.lib.rr_ensemble_stats_dev_ex(C.byref(spec), M, C.c_void_p(xd.data_ptr()), rows * n, n, rows, n, None,
                                                     C.c_void_p(thr), n, arr, n, 0, C.c_void_p(pk), C.c_void_p(pr), n, 0,
                                                     None))
    with pytest.raises(RuntimeError, match='needs thresholds'):
        raw(5, 0, None, out.data_ptr(), None, None)
    with pytest.raises(RuntimeError, match='no output'):
        raw(0, 0, None, None, None, None)
    with pytest.raises(RuntimeError, match='peak needs peak_row'):
        raw(0, 0, None, out.data_ptr(), peak.data_ptr(), None)
    with pytest.raises(RuntimeError, match='unknown statistic kind'):
        raw(6, 0, None, out.data_ptr(), None, None)


def _network(n, nbas, seed, dt_routing, dt_runoff):
    from tests.helpers import network_arrays
    down = synth.forest(n, nbas, seed=seed, depth_bias=0.5)
    k, x = synth.muskingum_params(n, seed)
    return down, network_arrays(down, k, x, dt_routing, dt_runoff)


@pytest.mark.parametrize('staging,K', [('auto', 1), ('direct', 1), ('registers-tiled', 1), ('auto', 2)])
@pytest.mark.parametrize('f32,resample,rows', [(False, 1, 0), (True, 3, 16), (False, 3, 0)])
def test_routed_warnings_equal_numpy_on_member_outputs(staging, K, f32, resample, rows, chunk_rows):
    n, T, M = 20000 + 3, 48, 5
    down, a = _network(n, 5, 21, 3600 // K, 3600)
    plan = rr.Plan(down, renumber='always', staging=staging)
    plan.set_coefficients(a['c1'], a['c2'], a['c3'], a['c4_dt'])
    base = synth.lateral_volumes(T, n, 9)
    lats = [base * s for s in np.random.default_rng(3).lognormal(0, 0.3, (M, 1, n))]
    lats[2][:, :500] = lats[1][:, :500]
    if f32:
        lats = [x.astype(np.float32) for x in lats]
    q0 = np.random.default_rng(2).uniform(0, 40, n)
    chunk_rows(rows)
    members = [np.empty((T // resample, n)) for _ in range(M)]
    mean = plan.route_ensemble_host(rr.MODE_RAPID, q0, lats, members, K, resample=resample)
    stacked = np.array(members)
    thr = _thresholds(stacked, np.random.default_rng(4))
    plan.set_thresholds(dict(zip(LABELS, thr)))
    assert plan.threshold_labels == LABELS
    ref = reference(stacked, MIXED, thr)
    S, R = len(MIXED), T // resample
    # the existing statistics alone, then the same with exceedance and peaks in the same call: unchanged
    plain = [s for s in MIXED if not s.startswith('exceed_')]
    outs0 = [np.empty((R, n)) for _ in plain]
    plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, plain, outs0, K, resample=resample)
    outs = [np.full((R, n), np.nan) for _ in MIXED]
    pk = (np.empty((S, n)), np.empty((S, n), dtype=np.int32))
    smean = plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, MIXED, outs, K, resample=resample, peaks=pk)
    assert np.array_equal(smean, mean)
    for s, name in enumerate(MIXED):
        assert np.array_equal(outs[s], ref[s]), name
        assert np.array_equal(pk[0][s], ref[s].max(axis=0)) and np.array_equal(pk[1][s], ref[s].argmax(axis=0)), name
    for o, name in zip(outs0, plain):
        assert np.array_equal(o, outs[MIXED.index(name)]), name
    # peaks only: nothing per step, the same peaks
    pk2 = (np.empty((S, n)), np.empty((S, n), dtype=np.int32))
    m2 = plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, MIXED, None, K, resample=resample, peaks=pk2)
    assert np.array_equal(pk2[0], pk[0]) and np.array_equal(pk2[1], pk[1]) and np.array_equal(m2, mean)
    # output subset: thresholds read at the user index of each column
    pick = np.array([n - 1, 0, 777, 0, 19999, 13], dtype=np.int32)
    plan.set_output_subset(pick)
    sub = [np.empty((R, pick.shape[0]), dtype=np.float32) for _ in MIXED]
    pk3 = (np.empty((S, pick.shape[0])), np.empty((S, pick.shape[0]), dtype=np.int32))
    plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, MIXED, sub, K, resample=resample, peaks=pk3)
    plan.set_output_subset(None)
    for s, name in enumerate(MIXED):
        assert np.array_equal(sub[s], ref[s][:, pick].astype(np.float32)), name
        assert np.array_equal(pk3[0][s], pk[0][s][pick]) and np.array_equal(pk3[1][s], pk[1][s][pick]), name
    plan.close()


def test_routed_validation_errors():
    n, T = 3000, 8
    down, a = _network(n, 2, 5, 3600, 3600)
    plan = rr.Plan(down)
    plan.set_coefficients(a['c1'], a['c2'], a['c3'], a['c4_dt'])
    lats = [synth.lateral_volumes(T, n, 1)] * 2
    q0 = np.zeros(n)
    with pytest.raises(ValueError, match='unknown ensemble statistic'):
        plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, ['exceed_a'], [np.empty((T, n))], 1)
    plan.set_thresholds({'a': np.ones(n)})
    spec = _lib.StatsSpec()
    spec.n_stats, spec.kind[0], spec.q[0] = 1, 5, 1                               # row 1 of one threshold row
    out = np.empty((T, n))
    arr_m, arr_s = C.c_void_p * 2, C.c_void_p * 1
    with pytest.raises(RuntimeError, match='threshold index 1 outside'):
        _lib.check(_lib.lib.rr_route_ensemble_stats_host_ex(
            plan._h, rr.MODE_RAPID, _lib.as_f64p(q0), 0, 2, arr_m(*[x.ctypes.data for x in lats]), 0, n, C.byref(spec),
            arr_s(out.ctypes.data), n, 0, None, n, None, T, 1, 1, None, None, 0))
    spec.q[0] = 0
    with pytest.raises(RuntimeError, match='no output'):
        _lib.check(_lib.lib.rr_route_ensemble_stats_host_ex(
            plan._h, rr.MODE_RAPID, _lib.as_f64p(q0), 0, 2, arr_m(*[x.ctypes.data for x in lats]), 0, n, C.byref(spec),
            None, n, 0, None, n, None, T, 1, 1, None, None, 0))
    plan.set_thresholds(None)
    with pytest.raises(RuntimeError, match='needs thresholds'):
        _lib.check(_lib.lib.rr_route_ensemble_stats_host_ex(
            plan._h, rr.MODE_RAPID, _lib.as_f64p(q0), 0, 2, arr_m(*[x.ctypes.data for x in lats]), 0, n, C.byref(spec),
            arr_s(out.ctypes.data), n, 0, None, n, None, T, 1, 1, None, None, 0))
    plan.close()


@pytest.mark.parametrize('horizon', ['both', 'peaks'])
def test_router_writes_numpy_warnings_of_member_outputs(tmp_path, monkeypatch, horizon):
    from tests.test_routers_gpu import _stream_case
    c = _stream_case(tmp_path, n=4000, T=40, files=6, f32=True, seed=7)
    monkeypatch.setenv('RR_ROUTER_SLAB_ROWS', '16')
    out_dir = tmp_path / 'out'
    out_dir.mkdir()
    members, finals = [], []

    def router():
        return rr.RapidMuskingum(params_file=c['params'], qlateral_files=c['files'], discharge_dir=str(out_dir),
                                 dt_discharge=7200, channel_state_init_file=c['state'], runoff_processing_mode='ensemble',
                                 log=False)
    ids = pd.read_parquet(c['params'])['river_id'].to_numpy()
    names = ['mean', 'p50', 'exceed_rp2', 'exceed_rp10']
    stats_path = str(tmp_path / 'warn.nc')
    r0 = router().set_ensemble_statistics(str(tmp_path / 'mean.nc'), ['mean'])   # its plan routes the single members
    r0.route()
    for ql in c['laterals']:
        q, o = c['q0'].copy(), np.empty((20, c['n']))
        r0.plan.route_host(rr.MODE_RAPID, q, ql, o, 1, resample=2)
        members.append(o)
        finals.append(q)
    # thresholds from the member outputs, for all rivers but the first 100, plus a river outside the network
    members = np.array(members)
    thr = {'rp2': members[1, 3], 'rp10': members[4].max(axis=0)}
    table = pd.DataFrame({'river_id': np.concatenate([ids[100:], [10 ** 9]]),
                          **{k: np.concatenate([v[100:], [1.0]]).astype(np.float32) for k, v in thr.items()}})
    full = {k: np.where(np.arange(c['n']) < 100, np.nan, v.astype(np.float32).astype(np.float64)) for k, v in thr.items()}
    r = router().set_ensemble_statistics(stats_path, names, thresholds=table, horizon=horizon)
    r.route()
    ref = [np.mean(members > full[s[7:]], axis=0) if s.startswith('exceed_') else numpy_statistic(members, s) for s in names]
    with ncio.open_nc(stats_path) as ds:
        for name, want in zip(names, ref):
            if horizon == 'both':
                assert np.array_equal(ncio.read_array(ds.variables[f'Q_{name}']), want.astype(np.float32)), name
            else:
                assert f'Q_{name}' not in ds.variables
            assert np.array_equal(ncio.read_array(ds.variables[f'Q_{name}_peak']), want.max(axis=0).astype(np.float32)), name
            assert np.array_equal(ncio.read_array(ds.variables[f'Q_{name}_peak_time']), want.argmax(axis=0) * 7200.0), name
    assert np.array_equal(r.channel_state, np.array(finals).mean(axis=0))
