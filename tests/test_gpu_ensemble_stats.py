"""
Ensemble statistics on the B200: the statistics kernel (rr_ensemble_stats_dev) and the routed path
(rr_route_ensemble_stats_host) must give numpy's np.mean / np.std / np.min / np.max / np.percentile over the stacked
fp64 member outputs bit for bit, and the router must write them to one file.
"""
import os

import numpy as np
import pytest

import river_route_b200 as rr
from river_route_b200 import ncio, synth
from river_route_b200.plan import ensemble_stats_dev
from oracle import oracle
from tests.conftest import require_cuda
from tests.helpers import network_arrays
from tests.test_ensemble_stats_cpu import numpy_statistic

pytestmark = pytest.mark.gpu
ALL16 = ['mean', 'std', 'min', 'max', 'p0', 'p1', 'p5', 'p10', 'p25', 'p33', 'p50', 'p67', 'p75', 'p90', 'p99', 'p100']
NO_SORT = ['max', 'std', 'min', 'mean']
SEVEN = ['mean', 'std', 'min', 'max', 'p25', 'p50', 'p75']


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


@pytest.mark.parametrize('M', [1, 2, 5, 51, 64])
def test_kernel_is_numpy_bit_for_bit(M):
    import torch
    rng = np.random.default_rng(M)
    rows, n = 7, 1000 + 13
    ld = n + 29
    x = rng.gamma(0.5, 20.0, (M, rows, ld)) * (rng.random((M, rows, ld)) < 0.7)   # many exact zeros
    x[:, :, :300] = np.round(x[:, :, :300] / 8.0)                                 # many exact ties
    x[:, 2, 300:400] = x[0, 2, 300:400]                                           # all members equal
    xd = torch.from_numpy(x).cuda()
    sub = np.array([n - 1, 0, 5, 5, 700, 0, 31, 32], dtype=np.int32)
    sub_d = torch.from_numpy(sub).cuda()
    for names in (ALL16, NO_SORT):
        ref = [numpy_statistic(x[:, :, :n], s) for s in names]
        for dt in (torch.float64, torch.float32):
            for subset in (False, True):
                n_out = sub.shape[0] if subset else n
                ldo = n_out + 5
                outs = [torch.full((rows, ldo), float('nan'), dtype=dt, device='cuda') for _ in names]
                ensemble_stats_dev(names, M, xd.data_ptr(), rows * ld, ld, rows, n_out, [o.data_ptr() for o in outs], ldo,
                                   dt == torch.float32, sub_d.data_ptr() if subset else 0)
                torch.cuda.synchronize()
                for s, o in enumerate(outs):
                    want = ref[s][:, sub] if subset else ref[s]
                    want = want.astype(np.float32) if dt == torch.float32 else want
                    got = o.cpu().numpy()
                    assert np.array_equal(got[:, :n_out], want), (M, names[s], dt, subset)
                    assert np.isnan(got[:, n_out:]).all()                       # nothing written past n_out
    with pytest.raises(RuntimeError, match='percentiles must lie'):
        ensemble_stats_dev_raw_percentile(M, xd, rows, ld, n)


def ensemble_stats_dev_raw_percentile(M, xd, rows, ld, n):
    """The C side validates percentiles itself (the Python parser never produces q > 100)."""
    import ctypes as C
    import torch
    from river_route_b200 import _lib
    spec = _lib.StatsSpec()
    spec.n_stats, spec.kind[0], spec.q[0] = 1, 4, 101
    out = torch.empty((rows, n), dtype=torch.float64, device='cuda')
    arr = (C.c_void_p * 1)(out.data_ptr())
    _lib.check(_lib.lib.rr_ensemble_stats_dev(C.byref(spec), M, C.c_void_p(xd.data_ptr()), rows * ld, ld, rows, n, None, arr,
                                              n, 0, None))


def _network(n, nbas, seed, dt_routing, dt_runoff):
    down = synth.forest(n, nbas, seed=seed, depth_bias=0.5)
    k, x = synth.muskingum_params(n, seed)
    return down, network_arrays(down, k, x, dt_routing, dt_runoff)


@pytest.mark.parametrize('staging,K', [('auto', 1), ('direct', 1), ('registers-tiled', 1), ('auto', 2)])
@pytest.mark.parametrize('f32,resample,rows', [(False, 1, 0), (True, 3, 16), (True, 1, 16), (False, 3, 0)])
def test_routed_statistics_equal_numpy_on_member_outputs(staging, K, f32, resample, rows, chunk_rows):
    n, T, M = 25000 + 3, 48, 5
    down, a = _network(n, 5, 17, 3600 // K, 3600)
    plan = rr.Plan(down, renumber='always', staging=staging)
    plan.set_coefficients(a['c1'], a['c2'], a['c3'], a['c4_dt'])
    base = synth.lateral_volumes(T, n, 9)
    lats = [base * s for s in np.random.default_rng(1).lognormal(0, 0.3, (M, 1, n))]
    lats[2][:, :500] = lats[1][:, :500]                                           # members with equal values
    if f32:
        lats = [x.astype(np.float32) for x in lats]
    q0 = np.random.default_rng(2).uniform(0, 40, n)
    chunk_rows(rows)
    # the existing per-member call, fp64 outputs: what the statistics must reduce to
    members = [np.empty((T // resample, n)) for _ in range(M)]
    finals = np.empty((M, n))
    mean = plan.route_ensemble_host(rr.MODE_RAPID, q0, lats, members, K, resample=resample, q_final=finals)
    stacked = np.array(members)
    ref = [numpy_statistic(stacked, s) for s in SEVEN]
    outs = [np.full((T // resample, n), np.nan) for _ in SEVEN]
    sf = np.empty((M, n))
    smean = plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, SEVEN, outs, K, resample=resample, q_final=sf)
    for s, name in enumerate(SEVEN):
        assert np.array_equal(outs[s], ref[s]), name
    assert np.array_equal(sf, finals) and np.array_equal(smean, mean)
    outs32 = [np.full((T // resample, n), np.nan, dtype=np.float32) for _ in SEVEN]
    plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, SEVEN, outs32, K, resample=resample)
    for s, name in enumerate(SEVEN):
        assert np.array_equal(outs32[s], ref[s].astype(np.float32)), name
    # two time slabs chained through the members' own states == one call
    cut = 24
    oa = [np.empty((cut // resample, n), dtype=np.float32) for _ in SEVEN]
    ob = [np.empty(((T - cut) // resample, n), dtype=np.float32) for _ in SEVEN]
    st = np.empty((M, n))
    plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, [x[:cut] for x in lats], SEVEN, oa, K, resample=resample, q_final=st)
    st2 = np.empty((M, n))
    m2 = plan.route_ensemble_stats_host(rr.MODE_RAPID, np.ascontiguousarray(st), [x[cut:] for x in lats], SEVEN, ob, K,
                                        resample=resample, q_final=st2)
    for s in range(len(SEVEN)):
        assert np.array_equal(np.vstack([oa[s], ob[s]]), outs32[s]), SEVEN[s]
    assert np.array_equal(st2, finals) and np.array_equal(m2, mean)
    # output subset: the columns of the full result
    pick = np.array([n - 1, 0, 777, 0, 24999, 13], dtype=np.int32)
    plan.set_output_subset(pick)
    sub = [np.empty((T // resample, pick.shape[0]), dtype=np.float32) for _ in SEVEN]
    plan.route_ensemble_stats_host(rr.MODE_RAPID, q0, lats, SEVEN, sub, K, resample=resample)
    plan.set_output_subset(None)
    for s in range(len(SEVEN)):
        assert np.array_equal(sub[s], outs32[s][:, pick]), SEVEN[s]
    # the CPU oracle per member, then numpy: the same statistics within float32 rounding
    orc = []
    for m in range(M):
        q, r_ = q0.copy(), np.zeros((T, n))
        oracle.rapid_route(a['indptr'], a['indices'], a['lhs_off'], a['c2'], a['c3'], a['c4_dt'], q, lats[m].astype(np.float64), r_, K)
        orc.append(r_.reshape(T // resample, resample, n).mean(axis=1) if resample > 1 else r_)
    orc = np.array(orc)
    scale = np.abs(orc).max(axis=(0, 1))
    for s, name in enumerate(SEVEN):
        want = numpy_statistic(orc, name)
        assert np.all(np.abs(outs32[s] - want) <= 2e-7 * np.abs(want) + 1e-9 * scale + 1e-30), name
    plan.close()


def test_router_writes_numpy_statistics_of_member_outputs(tmp_path, monkeypatch):
    from tests.test_routers_gpu import _stream_case
    c = _stream_case(tmp_path, n=4000, T=40, files=6, f32=True, seed=7)
    monkeypatch.setenv('RR_ROUTER_SLAB_ROWS', '16')
    out_dir = tmp_path / 'out'
    out_dir.mkdir()
    stats_path = str(tmp_path / 'stats.nc')
    names = ['mean', 'std', 'min', 'max', 'p10', 'p50', 'p90']
    r = rr.RapidMuskingum(params_file=c['params'], qlateral_files=c['files'], discharge_dir=str(out_dir), dt_discharge=7200,
                          channel_state_init_file=c['state'], runoff_processing_mode='ensemble', log=False)
    r.set_ensemble_statistics(stats_path, names).route()
    assert os.listdir(out_dir) == []
    # the members one by one through the same plan, fp64 output resampled on the device
    members, finals = [], []
    for ql in c['laterals']:
        q, o = c['q0'].copy(), np.empty((20, c['n']))
        r.plan.route_host(rr.MODE_RAPID, q, ql, o, 1, resample=2)
        members.append(o)
        finals.append(q)
    members = np.array(members)
    with ncio.open_nc(stats_path) as ds:
        for name in names:
            got = ncio.read_array(ds.variables[f'Q_{name}'])
            assert np.array_equal(got, numpy_statistic(members, name).astype(np.float32)), name
    assert np.array_equal(r.channel_state, np.array(finals).mean(axis=0))
