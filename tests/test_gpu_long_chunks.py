"""
GPU: host calls whose time chunk holds more rows than a CUDA grid has in y (65 535).  A small network with a long call
gets such chunks (the chunk length follows the bytes per row); with float32 lateral inflows off the direct pipeline
(two substeps) the inflows are upcast before routing, and a float32 output is cast after it, each over all rows of the
chunk at once.  Both kernels stride over rows, so one 70 000-row chunk must give the bits of 4 096-row chunks.
"""
import os

import numpy as np
import pytest

import river_route_b200 as rr
from river_route_b200 import synth
from oracle import oracle
from tests.conftest import require_cuda
from tests.helpers import network_arrays, parity_error

pytestmark = pytest.mark.gpu
TOL = 1e-10
N, T, K = 200, 70000, 2


@pytest.fixture(autouse=True)
def _cuda():
    require_cuda()


@pytest.fixture
def chunk_rows():
    def set_rows(rows):
        os.environ['RR_STREAM_CHUNK_ROWS'] = str(rows)
    yield set_rows
    os.environ.pop('RR_STREAM_CHUNK_ROWS', None)


def _case(seed):
    down = synth.forest(N, 3, seed=seed, depth_bias=0.5)
    k, x = synth.muskingum_params(N, seed)
    a = network_arrays(down, k, x, 3600 // K, 3600)
    plan = rr.Plan(down)
    plan.set_coefficients(a['c1'], a['c2'], a['c3'], a['c4_dt'])
    return plan, a


def _oracle(a, q0, ql):
    q, ref = q0.copy(), np.zeros((T, N))
    oracle.rapid_route(a['indptr'], a['indices'], a['lhs_off'], a['c2'], a['c3'], a['c4_dt'], q, ql.astype(np.float64), ref, K)
    return q, ref


def test_route_host_one_long_chunk(chunk_rows):
    plan, a = _case(21)
    ql32 = synth.lateral_volumes(T, N, 5).astype(np.float32)
    q0 = np.random.default_rng(3).uniform(0, 40, N)
    chunk_rows(T)
    q64, out64 = q0.copy(), np.full((T, N), np.nan)
    plan.route_host(rr.MODE_RAPID, q64, ql32, out64, K)
    q_o, ref = _oracle(a, q0, ql32)
    assert parity_error(out64, ref) < TOL and parity_error(q64, q_o) < TOL
    q, out32 = q0.copy(), np.full((T, N), np.nan, dtype=np.float32)
    plan.route_host(rr.MODE_RAPID, q, ql32, out32, K)
    assert np.array_equal(out32, out64.astype(np.float32)) and np.array_equal(q, q64)
    chunk_rows(4096)
    q_s, out_s = q0.copy(), np.full((T, N), np.nan, dtype=np.float32)
    plan.route_host(rr.MODE_RAPID, q_s, ql32, out_s, K)
    assert np.array_equal(out_s, out32) and np.array_equal(q_s, q)
    plan.close()


def test_route_ensemble_host_one_long_chunk(chunk_rows):
    M = 2
    plan, a = _case(22)
    base = synth.lateral_volumes(T, N, 6)
    lats = [(base * s).astype(np.float32) for s in (0.8, 1.3)]
    q0 = np.random.default_rng(4).uniform(0, 40, N)
    res = {}
    for rows in (T, 4096):
        chunk_rows(rows)
        outs = [np.full((T, N), np.nan, dtype=np.float32) for _ in range(M)]
        finals = np.empty((M, N))
        mean = plan.route_ensemble_host(rr.MODE_RAPID, q0, lats, outs, K, q_final=finals)
        res[rows] = outs, finals, mean
    (outs, finals, mean), (outs_s, finals_s, mean_s) = res[T], res[4096]
    for m in range(M):
        q_o, ref = _oracle(a, q0, lats[m])
        assert parity_error(finals[m], q_o) < TOL, m
        assert np.allclose(outs[m], ref.astype(np.float32), rtol=3e-7, atol=1e-30), m
        assert np.array_equal(outs_s[m], outs[m]), m
    assert np.array_equal(finals_s, finals) and np.array_equal(mean_s, mean)
    plan.close()
