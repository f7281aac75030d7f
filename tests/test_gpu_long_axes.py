"""
GPU: device calls longer than a CUDA grid has rows in y (65 535).  Every launch whose grid.y counts rows or row groups
-- the weights transform, the permutes, stage_out / stage_out_unit / stage_out_sub and the sentinel fill -- caps grid.y
and strides, so one call of any length must give the bits of the same rows routed as two shorter calls chained
through the state, and agree with the CPU oracle.  Small networks keep the arrays small; T is just past each limit.
"""
import os

import numpy as np
import pytest
import torch

import river_route_b200 as rr
from river_route_b200 import synth
from river_route_b200.transforms import Transform, weights_transform
from oracle import oracle
from tests.conftest import require_cuda
from tests.helpers import network_arrays, parity_error

pytestmark = pytest.mark.gpu
TOL = 1e-10
GRID_Y = 65535


@pytest.fixture(autouse=True)
def _cuda():
    require_cuda()


@pytest.fixture
def chunk_rows():
    def set_rows(rows):
        os.environ['RR_STREAM_CHUNK_ROWS'] = str(rows)
    yield set_rows
    os.environ.pop('RR_STREAM_CHUNK_ROWS', None)


def _network(n, seed, K=1):
    down = synth.forest(n, 2, seed=seed, depth_bias=0.5)
    k, x = synth.muskingum_params(n, seed)
    return down, network_arrays(down, k, x, 3600 // K, 3600)


def _weights(n_rivers, n_points, seed):
    rng = np.random.default_rng(seed)
    per = rng.integers(0, 6, n_rivers)
    ridx = np.repeat(np.arange(n_rivers), per)
    return oracle.weights_csr(ridx, rng.integers(0, n_points, ridx.shape[0]), rng.random(ridx.shape[0]), n_rivers, n_points)


def _cumulative_runoff(T, n_points, seed):
    rng = np.random.default_rng(seed)
    x = (rng.gamma(0.3, 2e-3, (T, n_points)) * (rng.random((T, n_points)) < 0.4)).astype(np.float32)
    return np.cumsum(x, axis=0, dtype=np.float32)


def test_weights_transform_past_grid_y():
    """8 * 65 535 = 524 280 time steps fill grid.y; 524 296 need a second pass of some CTAs."""
    T, n_riv, n_pts = 8 * GRID_Y + 16, 40, 64
    indptr, indices, data = _weights(n_riv, n_pts, 1)
    x = _cumulative_runoff(T, n_pts, 2)
    x[8 * GRID_Y - 1, 3] = np.nan                                  # last step of the first grid pass
    x[8 * GRID_Y, 5] = np.nan                                      # first step of the second pass
    got = weights_transform(indptr, indices, data, x, cumulative=True)
    ref = oracle.weights_transform(indptr, indices, data, x, cumulative=True, fma=True)
    assert np.array_equal(got, ref)
    assert parity_error(got, oracle.weights_transform(indptr, indices, data, x, cumulative=True)) < TOL


def test_runoff_route_host_chunk_past_grid_y(chunk_rows):
    """One streamed chunk of 524 304 rows (past the weights limit), then a shorter one that takes the cumulative lead."""
    n, n_pts, T = 48, 64, 524304 + 40000
    down, a = _network(n, 3)
    indptr, indices, data = _weights(n, n_pts, 4)
    area = np.random.default_rng(5).uniform(1e5, 5e8, n)
    x = _cumulative_runoff(T, n_pts, 6)
    plan = rr.Plan(down)
    plan.set_coefficients(a['c1'], a['c2'], a['c3'], a['c4_dt'])
    tf = Transform(indptr, indices, data, n_pts, area=area)
    q0 = np.random.default_rng(7).uniform(0, 30, n)
    res = {}
    for rows in (524304, 65536):
        chunk_rows(rows)
        q, out = q0.copy(), np.empty((T, n))
        plan.runoff_route_host(tf, rr.MODE_RAPID, q, x, out, 1, cumulative=True, as_volumes=True)
        res[rows] = q, out
    assert np.array_equal(res[524304][1], res[65536][1]) and np.array_equal(res[524304][0], res[65536][0])
    ql = oracle.weights_transform(indptr, indices, data, x, cumulative=True, area=area)
    q_ref, ref = q0.copy(), np.zeros((T, n))
    oracle.rapid_route(a['indptr'], a['indices'], a['lhs_off'], a['c2'], a['c3'], a['c4_dt'], q_ref, ql, ref, 1)
    assert parity_error(res[524304][1], ref) < TOL and parity_error(res[524304][0], q_ref) < TOL
    tf.close()
    plan.close()


def _route_dev(plan, mode, q0, lat, T, K, split=None, qf0=None):
    """Route rows [0, T) in one device call, or in two calls split at row `split`; returns host (out, q, q_full)."""
    n = q0.shape[0]
    dev = torch.device('cuda')
    d_lat = torch.from_numpy(lat).to(dev)
    d_out = torch.full((T, n), float('nan'), dtype=torch.float64, device=dev)
    d_q = torch.from_numpy(q0).to(dev)
    d_qf = torch.from_numpy(qf0).to(dev) if qf0 is not None else None
    qf_ptr = d_qf.data_ptr() if d_qf is not None else 0
    for a, b in ([(0, T)] if split is None else [(0, split), (split, T)]):
        plan.route_dev(mode, d_q.data_ptr(), d_lat[a:].data_ptr(), n, d_out[a:].data_ptr(), n, b - a, K, 0, qf_ptr)
    torch.cuda.synchronize()
    return d_out.cpu().numpy(), d_q.cpu().numpy(), (d_qf.cpu().numpy() if d_qf is not None else None)


# (label, mode, reaches, T, substeps, plan options): each T is just past the grid.y limit of one launch of that path
ROUTE_CASES = [
    # stage_out_kernel and permute_to_user<16>: ceil(T / 16) grid rows
    ('rapid-pipeline', rr.MODE_RAPID, 64, 16 * GRID_Y + 32, 1, dict(renumber='always')),
    # stage_out_unit_kernel and permute_to_working<16> of the lateral inflows
    ('unit-pipeline', rr.MODE_UNIT, 64, 16 * GRID_Y + 32, 1, dict(renumber='always')),
    # stage_out_sub_kernel: 64 // 12 = 5 rows per tile
    ('direct-K12', rr.MODE_RAPID, 64, 5 * GRID_Y + 25, 12, dict(renumber='always', staging='direct')),
    # permute_to_working<8> / permute_to_user<8>: row-major working arrays
    ('registers', rr.MODE_RAPID, 64, 8 * GRID_Y + 16, 1, dict(renumber='always', staging='registers')),
    # params-file order: no permutation at all (control)
    ('registers-never', rr.MODE_RAPID, 64, 8 * GRID_Y + 16, 1, dict(renumber='never', staging='registers')),
    # several substeps on the default staging: row-major working arrays, permute<8>
    ('substeps', rr.MODE_RAPID, 64, 8 * GRID_Y + 16, 2, dict(renumber='always')),
]


@pytest.mark.parametrize('label,mode,n,T,K,opts', ROUTE_CASES, ids=[c[0] for c in ROUTE_CASES])
def test_route_dev_past_grid_y(label, mode, n, T, K, opts):
    down, a = _network(n, 11, K)
    rng = np.random.default_rng(12)
    q0 = rng.uniform(0, 30, n)
    plan = rr.Plan(down, **opts)
    split = (T // 2) // 64 * 64
    if mode == rr.MODE_UNIT:
        lat = synth.lateral_volumes(T, n, 13) / 3600.0
        plan.set_coefficients(a['c1'], a['c2'], a['c3'], None)
        one = _route_dev(plan, mode, q0, lat, T, K, qf0=q0)
        two = _route_dev(plan, mode, q0, lat, T, K, split, qf0=q0)
        sp = oracle.unit_split(down.astype(np.int64))
        inner, hw, ai, ah = sp['inner_idx'], sp['hw_idx'], sp['a_inner'], sp['a_hw']
        c1i, c2i, c3i = a['c1'][inner], a['c2'][inner], a['c3'][inner]
        q_ch, q_full, ref = q0[inner].copy(), q0[inner].copy(), np.zeros((T, n))
        oracle.unit_route(ai[0], ai[1], -c1i[ai[1]], ai[0], ai[1], ai[2], ah[0], ah[1], ah[2], c1i, c2i, c3i, hw, inner,
                          q_ch, q_full, lat, ref, K)
        assert parity_error(one[0], ref) < TOL
        assert parity_error(one[1][inner], q_ch) < TOL and parity_error(one[2][inner], q_full) < TOL
    else:
        lat = synth.lateral_volumes(T, n, 13)
        plan.set_coefficients(a['c1'], a['c2'], a['c3'], a['c4_dt'])
        one = _route_dev(plan, mode, q0, lat, T, K)
        two = _route_dev(plan, mode, q0, lat, T, K, split)
        q_ref, ref = q0.copy(), np.zeros((T, n))
        oracle.rapid_route(a['indptr'], a['indices'], a['lhs_off'], a['c2'], a['c3'], a['c4_dt'], q_ref, lat, ref, K)
        assert parity_error(one[0], ref) < TOL and parity_error(one[1], q_ref) < TOL
    for x, y in zip(one, two):
        assert (x is None and y is None) or np.array_equal(x, y), label
    plan.close()


def test_route_dev_sentinel_fill_past_grid_y():
    """32 reaches: one block, so the pipeline arms its 64-row tiles with the sentinel pattern; 65 537 tiles."""
    n, T = 32, 64 * GRID_Y + 128
    down, a = _network(n, 17)
    plan = rr.Plan(down, renumber='always')
    plan.set_coefficients(a['c1'], a['c2'], a['c3'], a['c4_dt'])
    assert plan.tile_rows(T) == 64
    q0 = np.random.default_rng(18).uniform(0, 30, n)
    lat = synth.lateral_volumes(T, n, 19)
    dev = torch.device('cuda')
    d_lat = torch.from_numpy(lat).to(dev)
    d_one = torch.empty((T, n), dtype=torch.float64, device=dev)
    d_two = torch.empty((T, n), dtype=torch.float64, device=dev)
    d_q1, d_q2 = torch.from_numpy(q0).to(dev), torch.from_numpy(q0).to(dev)
    plan.route_dev(rr.MODE_RAPID, d_q1.data_ptr(), d_lat.data_ptr(), n, d_one.data_ptr(), n, T, 1)
    split = 32 * GRID_Y
    plan.route_dev(rr.MODE_RAPID, d_q2.data_ptr(), d_lat.data_ptr(), n, d_two.data_ptr(), n, split, 1)
    plan.route_dev(rr.MODE_RAPID, d_q2.data_ptr(), d_lat[split:].data_ptr(), n, d_two[split:].data_ptr(), n, T - split, 1)
    torch.cuda.synchronize()
    assert torch.equal(d_one, d_two) and torch.equal(d_q1, d_q2)
    del d_two, d_q2
    out, q = d_one.cpu().numpy(), d_q1.cpu().numpy()
    del d_one, d_lat
    q_ref, ref = q0.copy(), np.zeros((T, n))
    oracle.rapid_route(a['indptr'], a['indices'], a['lhs_off'], a['c2'], a['c3'], a['c4_dt'], q_ref, lat, ref, 1)
    assert parity_error(out, ref) < TOL and parity_error(q, q_ref) < TOL
    plan.close()
