"""
GPU: every dispatch branch of the unit-hydrograph convolution (rr_uh.cu) and of the grid-weight transform (rr_spmm.cu),
bit for bit against the CPU oracle compiled with FMA contraction.  Each kernel applies one fma per term in the oracle's
order; padded taps and zero inputs are fma(0, x, acc) == acc and a float32 input converted to fp64 is exact, so any
difference in a single bit means a kernel summed in another order, dropped a term or read the wrong element.

Default UH dispatch on n_ks (no RR_UH_REGISTERS):
    1-8     uh_conv_kernel_reg<8,1>  + uh_state_kernel_reg<1>
    9-16    uh_conv_kernel_reg<8,2>  + uh_state_kernel_reg<2>
    17-48   uh_conv_kernel_smem<16>  + uh_state_kernel_reg<3..6>
    49-192  uh_conv_kernel_smem<16>  (up to 12 tap groups) + uh_state_kernel
    > 192   uh_conv_kernel<8>        + uh_state_kernel
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import river_route_b200 as rr
from river_route_b200 import _lib, synth
from river_route_b200.transforms import Transform, uh_convolve, weights_transform
from oracle import oracle
from tests.conftest import require_cuda
from tests.helpers import network_arrays, parity_error

pytestmark = pytest.mark.gpu
TOL = 1e-10
N_KS = [1, 8, 9, 16, 17, 36, 48, 49, 100, 192, 193, 260]


@pytest.fixture(autouse=True)
def _cuda():
    require_cuda()


def _uh_case(n, n_ks, T, seed):
    rng = np.random.default_rng(seed)
    ker = rng.uniform(0, 1, (n_ks, n)) * (rng.random((n_ks, n)) < 0.7)
    lat = rng.gamma(0.3, 2e-3, (T, n)) * (rng.random((T, n)) < 0.5)
    s0 = rng.uniform(0, 1e-3, (n_ks, n))
    return lat, ker, s0


def _check_uh(lat, ker, state_gpu, state_fma, state_plain):
    """One call on both sides; states are updated in place.  Bitwise against the FMA oracle, 1e-10 against the plain one."""
    out = uh_convolve(lat, ker, state_gpu)
    ref = oracle.uh_convolve(lat, ker, state_fma, fma=True)
    plain = oracle.uh_convolve(lat, ker, state_plain)
    assert np.array_equal(out, ref)
    assert np.array_equal(state_gpu, state_fma)
    col = np.max(np.abs(plain), axis=0) + np.max(np.abs(state_plain), axis=0)
    assert parity_error(out, plain, col) < TOL and parity_error(state_gpu, state_plain, col) < TOL
    assert np.all(state_gpu[-1] == 0)


@pytest.mark.parametrize('n_ks', N_KS)
def test_uh_every_dispatch_branch(n_ks):
    n = 300                                                  # not a multiple of the 128-thread CTA
    for T in sorted({1, max(1, n_ks - 1), 7, 301}):
        lat, ker, s0 = _uh_case(n, n_ks, T, 1000 * n_ks + T)
        _check_uh(lat, ker, s0.copy(), s0.copy(), s0.copy())


def _time_chunk(n, n_ks, T):
    """The time chunk rr_uh_convolve_dev gives each grid row (rr_uh.cu), as a multiple of 16 for the smem kernel."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    gx = (n + 127) // 128
    want_y = max(1, (sms * 16 + gx - 1) // gx)
    chunk = max(max(8 * n_ks, 64), (T + want_y - 1) // want_y)
    chunk = min((chunk + 7) // 8 * 8, T)
    if n_ks > 16 and (n_ks + 15) // 16 * 16 * 128 * 8 <= 192 * 1024:
        chunk = min((chunk + 15) // 16 * 16, T)
    return chunk


@pytest.mark.parametrize('n_ks,extra', [(8, 5), (16, 3), (36, 0), (36, 13), (100, 0), (100, 7), (260, 11)])
def test_uh_few_basins_split_time_over_grid_y(n_ks, extra):
    """n <= 128: one CTA column, time split into ~20 grid rows.  extra = 0 ends the last 16-output iteration of the smem
    kernel exactly at T (t0 + 16 == T on the predicate-free path); other values end it on the guarded path."""
    n = 100
    base = max(8 * n_ks, 64)                                 # the chunk floor of rr_uh.cu: a chunk re-reads n_ks - 1 rows
    T = 20 * ((base + 15) // 16 * 16) + extra
    chunk = _time_chunk(n, n_ks, T)
    assert (T + chunk - 1) // chunk >= 20
    lat, ker, s0 = _uh_case(n, n_ks, T, n_ks + extra)
    _check_uh(lat, ker, s0.copy(), s0.copy(), s0.copy())


@pytest.mark.parametrize('n_ks', [100, 260])
def test_uh_chained_calls_shorter_than_kernel(n_ks):
    """Carry-over through the generic state kernel, including calls shorter than the kernel (old state rows ahead)."""
    n = 200
    rng = np.random.default_rng(n_ks)
    ker = rng.uniform(0, 1, (n_ks, n)) * (rng.random((n_ks, n)) < 0.7)
    s_gpu, s_fma, s_plain = np.zeros((n_ks, n)), np.zeros((n_ks, n)), np.zeros((n_ks, n))
    for c, T in enumerate([1, 5, n_ks + 3, 2 * n_ks]):
        lat = rng.gamma(0.3, 2e-3, (T, n)) * (rng.random((T, n)) < 0.5)
        _check_uh(lat, ker, s_gpu, s_fma, s_plain)


def _vp(t):
    return C.c_void_p(t.data_ptr())


@pytest.mark.parametrize('n_ks', [9, 36, 100, 260])
def test_uh_device_call_leading_dimensions(n_ks):
    """rr_uh_convolve_dev with four different leading dimensions; padding columns hold NaN and must stay NaN."""
    n, T = 200, 97
    ldl, ldk, lds, ldo = n + 3, n + 11, n + 19, n + 27
    lat, ker, s0 = _uh_case(n, n_ks, T, 7 * n_ks)
    dev = torch.device('cuda')

    def padded(a, ld):
        b = np.full((a.shape[0], ld), np.nan)
        b[:, :n] = a
        return torch.from_numpy(b).to(dev)

    d_lat, d_ker, d_s = padded(lat, ldl), padded(ker, ldk), padded(s0, lds)
    d_out = torch.full((T, ldo), float('nan'), dtype=torch.float64, device=dev)
    _lib.check(_lib.lib.rr_uh_convolve_dev(n, n_ks, T, _vp(d_lat), ldl, _vp(d_ker), ldk, _vp(d_s), lds, _vp(d_out), ldo,
                                           None))
    torch.cuda.synchronize()
    out, st = d_out.cpu().numpy(), d_s.cpu().numpy()
    s_ref = s0.copy()
    ref = oracle.uh_convolve(lat, ker, s_ref, fma=True)
    assert np.array_equal(out[:, :n], ref) and np.array_equal(st[:, :n], s_ref)
    assert np.isnan(out[:, n:]).all() and np.isnan(st[:, n:]).all()


# ------------------------------------------------------------------------------------------------------
# grid-weight transform
# ------------------------------------------------------------------------------------------------------
def _weight_table(n_rivers, n_points, seed):
    """Empty rows, short rows and one row of several thousand entries."""
    rng = np.random.default_rng(seed)
    per = rng.integers(0, 7, n_rivers)
    per[::11] = 0
    per[n_rivers // 2] = 4000
    ridx = np.repeat(np.arange(n_rivers), per)
    pidx = rng.integers(0, n_points, ridx.shape[0])
    indptr, indices, data = oracle.weights_csr(ridx, pidx, rng.random(ridx.shape[0]), n_rivers, n_points)
    assert (np.diff(indptr) == 0).any() and np.diff(indptr).max() > 2000
    return indptr, indices, data


def _grid(T, n_points, seed, f32, cumulative):
    rng = np.random.default_rng(seed)
    x = rng.gamma(0.3, 2e-3, (T, n_points)) * (rng.random((T, n_points)) < 0.5)
    x -= 1e-4 * rng.random((T, n_points))                    # some negative increments: force_positive has work
    if cumulative:
        x = np.cumsum(x, axis=0)
    for t in (7, 8, T - 1):                                  # time-block boundaries and the last step
        if 0 <= t < T:
            x[t, rng.integers(0, n_points, 40)] = np.nan
    return x.astype(np.float32) if f32 else x


def _check_weights(indptr, indices, data, x, area):
    for cumulative in (False, True):
        xs = np.cumsum(np.nan_to_num(x), axis=0).astype(x.dtype) if cumulative else x
        if cumulative:
            xs[np.isnan(x)] = np.nan
        for clip in (False, True):
            for keep_nan in (False, True):
                kw = dict(cumulative=cumulative, force_positive=clip, area=area, keep_nan=keep_nan)
                got = weights_transform(indptr, indices, data, xs, **kw)
                ref = oracle.weights_transform(indptr, indices, data, xs, fma=True, **kw)
                assert np.array_equal(got, ref, equal_nan=True), kw
                if keep_nan:
                    assert np.array_equal(np.isnan(got), np.isnan(ref)), kw
                else:
                    assert not np.isnan(got).any()
                    assert parity_error(got, oracle.weights_transform(indptr, indices, data, xs, **kw)) < TOL, kw


@pytest.mark.parametrize('T', [1, 7, 8, 9, 37])
@pytest.mark.parametrize('f32', [True, False])
def test_weights_every_option(T, f32):
    n_riv, n_pts = 700, 6000
    indptr, indices, data = _weight_table(n_riv, n_pts, 3)
    x = _grid(T, n_pts, 4 + T, f32, False)
    area = np.random.default_rng(5).uniform(1e5, 5e8, n_riv)
    _check_weights(indptr, indices, data, x, area)
    _check_weights(indptr, indices, data, x, None)


@pytest.mark.parametrize('f32', [True, False])
def test_weights_grid_y_filled(f32):
    """T = 8 * 65 535: the largest call whose time blocks each get a grid row of their own."""
    T, n_riv, n_pts = 524280, 40, 64
    rng = np.random.default_rng(6)
    per = rng.integers(0, 6, n_riv)
    ridx = np.repeat(np.arange(n_riv), per)
    indptr, indices, data = oracle.weights_csr(ridx, rng.integers(0, n_pts, ridx.shape[0]), rng.random(ridx.shape[0]),
                                               n_riv, n_pts)
    x = _grid(T, n_pts, 7, f32, True)
    for clip in (False, True):
        got = weights_transform(indptr, indices, data, x, cumulative=True, force_positive=clip)
        ref = oracle.weights_transform(indptr, indices, data, x, cumulative=True, force_positive=clip, fma=True)
        assert np.array_equal(got, ref)


@pytest.mark.parametrize('f32', [True, False])
def test_weights_device_call_leading_dimensions(f32):
    """rr_weights_transform_dev with ldx > n_points and ldy > n_rivers: NaN padding is never read or written."""
    n_riv, n_pts, T = 300, 6000, 29
    ldx, ldy = n_pts + 5, n_riv + 7
    indptr, indices, data = _weight_table(n_riv, n_pts, 8)
    x = _grid(T, n_pts, 9, f32, True)
    area = np.random.default_rng(10).uniform(1e5, 5e8, n_riv)
    dev = torch.device('cuda')
    xp = np.full((T, ldx), np.nan, dtype=x.dtype)
    xp[:, :n_pts] = x
    d_x = torch.from_numpy(xp).to(dev)
    d_y = torch.full((T, ldy), float('nan'), dtype=torch.float64, device=dev)
    d_ptr, d_idx = torch.from_numpy(indptr).to(dev), torch.from_numpy(indices).to(dev)
    d_w, d_a = torch.from_numpy(data).to(dev), torch.from_numpy(area).to(dev)
    _lib.check(_lib.lib.rr_weights_transform_dev(n_riv, n_pts, T, _vp(d_ptr), _vp(d_idx), _vp(d_w), _vp(d_x), int(f32),
                                                 ldx, _vp(d_y), ldy, 1, 1, _vp(d_a), None))
    torch.cuda.synchronize()
    y = d_y.cpu().numpy()
    ref = oracle.weights_transform(indptr, indices, data, x, cumulative=True, force_positive=True, area=area, fma=True)
    assert np.array_equal(y[:, :n_riv], ref) and np.isnan(y[:, n_riv:]).all()


# ------------------------------------------------------------------------------------------------------
# the generic state kernel inside the streamed pipeline
# ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n_ks,rows', [(60, 7), (60, 16), (200, 16), (200, 40)])
def test_streamed_uh_chunks_shorter_than_kernel(n_ks, rows):
    """runoff_route_host with a UH transform whose kernel is longer than the stream's time chunks: each chunk's
    convolution reads carry-over rows it does not replace.  Chunked == one chunk bit for bit; the UH state equals the
    FMA oracle chain bit for bit; the discharge agrees with the oracle."""
    n, n_pts, T, K = 3000 + 7, 700, 90, 1
    down = synth.forest(n, 4, seed=n_ks, depth_bias=0.5)
    k, xk = synth.muskingum_params(n, n_ks)
    a = network_arrays(down, k, xk, 3600, 3600)
    rng = np.random.default_rng(n_ks + rows)
    per = rng.integers(1, 6, n)
    ridx = np.repeat(np.arange(n), per)
    indptr, indices, data = oracle.weights_csr(ridx, rng.integers(0, n_pts, ridx.shape[0]), rng.random(ridx.shape[0]),
                                               n, n_pts)
    ker = rng.uniform(0, 1, (n_ks, n)) * (rng.random((n_ks, n)) < 0.6)
    s0 = rng.uniform(0, 1e-3, (n_ks, n))
    s0[-1] = 0.0
    q0 = rng.uniform(0, 30, n)
    x = (rng.gamma(0.3, 2e-3, (T, n_pts)) * (rng.random((T, n_pts)) < 0.4)).astype(np.float32)
    plan = rr.Plan(down)
    plan.set_coefficients(a['c1'], a['c2'], a['c3'], None)
    res = {}
    try:
        for r in (0, rows):
            if r:
                os.environ['RR_STREAM_CHUNK_ROWS'] = str(r)
            tf = Transform(indptr, indices, data, n_pts).set_unit_hydrograph(ker, s0)
            q, out = q0.copy(), np.empty((T, n))
            plan.runoff_route_host(tf, rr.MODE_UNIT, q, x, out, K)
            res[r] = q, out, tf.uh_state()
            tf.close()
    finally:
        os.environ.pop('RR_STREAM_CHUNK_ROWS', None)
    for u, v in zip(res[0], res[rows]):
        assert np.array_equal(u, v)
    depths = oracle.weights_transform(indptr, indices, data, x, fma=True)
    s_fma = s0.copy()
    conv_fma = oracle.uh_convolve(depths, ker, s_fma, fma=True)
    assert np.array_equal(res[rows][2], s_fma)
    s_ref = s0.copy()
    conv = oracle.uh_convolve(oracle.weights_transform(indptr, indices, data, x), ker, s_ref)
    sp = oracle.unit_split(down.astype(np.int64))
    inner, hw, ai, ah = sp['inner_idx'], sp['hw_idx'], sp['a_inner'], sp['a_hw']
    c1i, c2i, c3i = a['c1'][inner], a['c2'][inner], a['c3'][inner]
    q_ch, q_full, ref = q0[inner].copy(), q0[inner].copy(), np.zeros((T, n))
    oracle.unit_route(ai[0], ai[1], -c1i[ai[1]], ai[0], ai[1], ai[2], ah[0], ah[1], ah[2], c1i, c2i, c3i, hw, inner,
                      q_ch, q_full, conv, ref, K)
    col = np.max(np.abs(conv), axis=0)
    assert parity_error(res[rows][1], ref, col) < TOL
    assert np.array_equal(conv_fma[-1][hw], res[rows][0][hw])
    plan.close()
