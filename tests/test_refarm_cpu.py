"""The reference arm of bench.py (oracle/refarm.py): it runs river-route's own numba kernels from oracle/_ref, builds
the same synthetic workload as the CUDA arm without loading the product library, and agrees with the C oracle."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle, refarm
from tests.helpers import ROOT, network_arrays, parity_error

needs_ref = pytest.mark.skipif(not refarm.reference_available(),
                               reason='oracle/_ref absent: run `python oracle/ref_install.py` where /root/reference exists')


def test_standalone_generators_match_the_product_generators():
    from river_route_b200 import synth
    for n, nb, seed, bias in ((5000, 7, 4, 0.5), (1234, 1, 0, 0.9)):
        assert np.array_equal(refarm.forest(n, nb, seed=seed, depth_bias=bias), synth.forest(n, nb, seed=seed, depth_bias=bias))
    k0, x0 = synth.muskingum_params(999, 4)
    k1, x1 = refarm.muskingum_params(999, 4)
    assert np.array_equal(k0, k1) and np.array_equal(x0, x1)
    assert np.array_equal(synth.lateral_volumes(7, 333, 99), refarm.lateral_volumes(7, 333, 99))
    import river_route_b200 as rr
    down = refarm.forest(5000, 7, seed=4)
    assert np.array_equal(refarm.basin_parts(down, 3), rr.label_basins(down, 3)[2])


@needs_ref
def test_reference_router_object_matches_oracle():
    """make_router drives the reference's own adjacency_matrix / _set_muskingum_coefficients / _router; the C oracle
    restates the same arithmetic (bit-identical up to numba's fastmath FMA contraction)."""
    n, T = 3000, 20
    down = refarm.forest(n, 4, seed=2, depth_bias=0.6)
    k, x = refarm.muskingum_params(n, 2)
    ql = refarm.lateral_volumes(T, n, 5)
    r = refarm.make_router(down.astype(np.int64), k, x, 3600, 3600, T)
    a = network_arrays(down, k, x, 3600, 3600)
    assert np.array_equal(r._csc_indptr, a['indptr']) and np.array_equal(r._csc_indices, a['indices'])
    assert np.array_equal(r.c1, a['c1']) and np.array_equal(r._lhs_off_data, a['lhs_off'])
    q, ref = np.zeros(n), np.zeros((T, n))
    for _ in range(2):                                       # two chained "files"
        got = refarm.route_once(r, ql)
        oracle.rapid_route(a['indptr'], a['indices'], a['lhs_off'], a['c2'], a['c3'], a['c4_dt'], q, ql, ref, 1)
        assert parity_error(got, ref) < 1e-12
    assert parity_error(r.channel_state[None], q[None]) < 1e-12


def test_reference_arm_line_and_isolation():
    """`bench.py --impl reference` prints the contract's line, runs the reference (kind = "reference") over worker
    processes, uses the CUDA arm's config verbatim and never maps the product library.  Without the reference package
    the arm times the C restatement instead (kind = "port"); line, isolation and config are held to the same checks."""
    code = (
        "import sys, json, runpy\n"
        "sys.argv = ['bench.py', '--impl', 'reference', '--reaches', '40000', '--basins', '30', '--rows', '16',"
        " '--steps', '2', '--warmup', '1', '--ref-cores', '2']\n"
        "runpy.run_path('bench.py', run_name='__main__')\n"
        "maps = open('/proc/self/maps').read()\n"
        "print(json.dumps({'librr_b200': 'librr_b200' in maps, 'cuda': 'libcudart' in maps or 'libcuda.so' in maps,"
        " 'pkg': any(m.startswith('river_route_b200') for m in sys.modules)}))\n")
    out = subprocess.run([sys.executable, '-c', code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith('{')]
    line, iso = lines[0], lines[1]
    assert iso == {'librr_b200': False, 'cuda': False, 'pkg': False}
    kind = 'reference' if refarm.reference_available() else 'port'
    assert line['impl'] == 'reference' and line['cpu_baseline']['kind'] == kind and line['cpu_baseline']['cores'] == 2
    assert line['value'] > 0 and line['e2e']['value'] == line['value'] and line['gpu_launches'] == 0
    sys.path.insert(0, ROOT)
    import bench
    args = bench.parse.__globals__['argparse'].Namespace(reaches=40000, basins=30, rows=16, scaling='weak', depth_bias=0.5,
                                                         order='growth', gpus=1)
    assert line['config'] == bench.workload_config(args)     # the CUDA arm prints exactly this dict
