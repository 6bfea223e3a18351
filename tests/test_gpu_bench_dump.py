"""bench.py --dump-outputs: the last timed step's arrays as float64 .npy files, at most 64 MB in all.  The
c3 workload (50 000 frequencies) is too large to dump whole, so its frequency-resolved arrays come as the
documented seeded sample; what is written must be what the reference computed for the same inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import ff_oracle as oracle
import workloads
from helpers import nerr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ('eigvals', 'eigvecs', 'propagators', 'control_matrix', 'filter_function', 'infidelity',
         'e2e_infidelity')


def bench(steps, *extra):
    proc = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--workload', 'c3', '--extra', 'none',
                           '--no-int8', '--no-cpu-baseline', '--steps', str(steps), '--warmup', '0', *extra],
                          capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-3000:]
    return json.loads(proc.stdout)


def complex_array(a):
    assert a.shape[-1] == 2
    return a[..., 0] + 1j*a[..., 1]


def test_dump_outputs_c3(engine, tmp_path):
    out = tmp_path / 'dump'
    line2 = bench(2, '--dump-outputs', str(out))
    # --steps sets the number of timed steps: the launches of the timed window scale with it
    line3 = bench(3)
    assert line2['steps'] == 2 and line3['steps'] == 3
    assert line2['gpu_launches'] > 0 and 3*line2['gpu_launches'] == 2*line3['gpu_launches']

    assert sorted(os.listdir(out)) == sorted(f'{k}.npy' for k in NAMES)
    assert sum(os.path.getsize(out / f'{k}.npy') for k in NAMES) <= 64_000_000
    got = {k: np.load(out / f'{k}.npy') for k in NAMES}
    assert all(a.dtype == np.float64 for a in got.values())

    wl = workloads.get('c3')
    n_omega, order = len(wl.omega), np.argsort(wl.n_ids)
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'workload_full_c3.npz'))
    np.testing.assert_allclose(got['e2e_infidelity'], g['infidelity'], rtol=1e-10)
    np.testing.assert_allclose(got['infidelity'][order], g['infidelity'], rtol=1e-10)

    # eigensystem and propagators of the whole pulse
    H = oracle.hamiltonian_from_coeffs(wl.c_opers, wl.c_coeffs)
    ev, _, Q = oracle.diagonalize(H, wl.dt)
    V, P = complex_array(got['eigvecs']), complex_array(got['propagators'])
    assert nerr(got['eigvals'], ev) < 1e-10 and nerr(P, Q) < 1e-10
    assert nerr((V*got['eigvals'][:, None, :]) @ V.conj().swapaxes(1, 2), H) < 1e-10
    assert np.allclose(P[0], np.eye(wl.d), rtol=0, atol=1e-15) and nerr(P[-1], g['total_propagator']) < 1e-10

    # control matrix and filter function on the seeded sample of frequencies
    B = complex_array(got['control_matrix'])
    assert B.shape[:2] == (len(wl.n_opers), len(wl.basis)) and 0 < B.shape[2] < n_omega
    keep = np.sort(np.random.default_rng(0).choice(n_omega, B.shape[2], replace=False))
    both, at_keep, at_pick = np.intersect1d(keep, g['pick'], return_indices=True)
    assert len(both) > 100
    for j, k in enumerate(order):
        assert np.abs(B[k][:, at_keep] - g['control_matrix'][j][:, at_pick]).max() < 1e-10*g['scale'][j]
    F = complex_array(got['filter_function'])
    assert F.shape == (len(wl.n_opers),)*2 + (B.shape[2],)
    assert nerr(F, oracle.filter_function(B)) < 1e-12
    assert nerr(F[order][:, order][..., at_keep], g['filter_function'][..., at_pick]) < 1e-10
