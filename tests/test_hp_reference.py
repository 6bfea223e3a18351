"""The extended-precision control-matrix reference (tests/hp_control_matrix.py) and the ledger of kernel
instances (tests/test_gpu_ctrlmat_instances.py), checked without a GPU:

- the reference agrees with a 30-digit mpmath evaluation of the same formula on the special branches;
- the float64 oracle stays within 1 * EPS * M on every ledger case, so the bound is sound, and a relative
  error of 1e-12 on the upper half of the grid breaks KAPPA * EPS * M while the normalised error that the
  older parity tests use does not notice it, so the bound is tight;
- the ledger names exactly the control-matrix kernel instances compiled into libffb200.so.
"""
import os
import re
import shutil
import subprocess

import mpmath
import numpy as np
import pytest

import ff_oracle as oracle
import hp_control_matrix as hp
import test_gpu_ctrlmat_instances as ledger
from helpers import nerr, rand_herm


def _mp_entry(ev, V, Q, w, basis, n_opers, n_coeffs, dt, t, j, k):
    """B_jk(w) in 30-digit arithmetic from the float64 inputs (exact conversions)."""
    mpmath.mp.dps = 30
    G, d = ev.shape
    mat = lambda a: mpmath.matrix([[mpmath.mpc(complex(x)) for x in row] for row in a])  # noqa: E731
    w = mpmath.mpf(float(w))
    total = mpmath.mpc(0)
    for g in range(G):
        Vg = mat(V[g])
        Vh = Vg.H
        QdV = mat(Q[g]).H*Vg
        Bbar = Vh*mat(n_opers[j])*Vg*mpmath.mpf(float(n_coeffs[j, g]))
        Cbar = QdV.H*mat(basis[k])*QdV
        dtg = mpmath.mpf(float(dt[g]))
        step = mpmath.mpc(0)
        for m in range(d):
            for n in range(d):
                x = w + mpmath.mpf(float(ev[g, m])) - mpmath.mpf(float(ev[g, n]))
                y = x*dtg/2
                integral = dtg if y == 0 else dtg*mpmath.expj(y)*mpmath.sin(y)/y
                step += Bbar[m, n]*integral*Cbar[n, m]
        total += mpmath.expj(w*mpmath.mpf(float(t[g])))*step
    return total


def _draw(rng, d, G, dt_scale=1.0):
    H = oracle.hamiltonian_from_coeffs(rand_herm(rng, d, 2), rng.standard_normal((2, G)))
    dt = dt_scale*(1 - rng.random(G))
    ev, V, Q = oracle.diagonalize(H, dt)
    return ev, V, Q, dt, np.concatenate(([0.0], dt.cumsum()))


@pytest.mark.parametrize('d', [2, 3])
def test_reference_against_mpmath(d):
    rng = np.random.default_rng(11 + d)
    G, n_nops, n_basis = 3, 2, 2
    ev, V, Q, dt, t = _draw(rng, d, G)
    n_opers = rand_herm(rng, d, n_nops)
    basis = rng.standard_normal((n_basis, d, d)) + 1j*rng.standard_normal((n_basis, d, d))
    n_coeffs = rng.random((n_nops, G)) + 0.5
    split = ev[1, 1] - ev[1, 0]
    omega = np.array([
        0.0,                                  # x = 0 exactly on the diagonal
        -split,                               # omega on a level splitting: x = 0 up to rounding
        -split + 1e-9/dt[1],                  # |x dt| ~ 1e-9
        -2.7,                                 # negative
        3e6/t[-1], 1e7/t[-1],                 # |omega t| ~ 1e6 - 1e7
    ])
    B, M = hp.control_matrix(ev, V, Q, omega, basis, n_opers, n_coeffs, dt, t)
    for j in range(n_nops):
        for k in range(n_basis):
            for o, w in enumerate(omega):
                ref = _mp_entry(ev, V, Q, w, basis, n_opers, n_coeffs, dt, t, j, k)
                dev = abs(mpmath.mpc(mpmath.mpf(str(B[j, k, o].real)), mpmath.mpf(str(B[j, k, o].imag))) - ref)
                assert dev <= 1e-3*hp.EPS*float(M[j, k, o]), (j, k, w, float(dev), float(M[j, k, o]))


def _oracle(inputs):
    return oracle.control_matrix_from_scratch(*(inputs[k] for k in (
        'eigvals', 'eigvecs', 'propagators', 'omega', 'basis', 'n_opers', 'n_coeffs', 'dt', 't')))


@pytest.mark.parametrize('name', list(ledger.CASES))
def test_oracle_within_bound_and_perturbation_rejected(name):
    inputs = ledger.build_inputs(name)
    B_hp, M = ledger.reference(inputs)
    B = _oracle(inputs)
    assert hp.ratio(B, B_hp, M).max() <= 1.0
    if np.abs(inputs['omega']).max()*inputs['t'][-1] > 2e3:
        return  # long pulses: |omega t| dominates M at the top of the grid
    # short pulses: a relative error of 1e-12 on the upper half of the grid fails the kernels' bound ...
    n_omega = B.shape[-1]
    perturbed = B.copy()
    perturbed[..., n_omega//2:] *= 1 + 1e-12
    assert hp.ratio(perturbed, B_hp, M).max() > ledger.KAPPA
    # ... and passes the normalised tolerance of 1e-10 per noise operator
    assert max(nerr(perturbed[j], B_hp[j].astype(complex)) for j in range(len(B))) < 1e-10


def _compiled_instances():
    import __graft_entry__ as entry
    entry.build()
    from filter_functions_b200 import _lib
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    cxxfilt = shutil.which('c++filt')
    if not os.path.exists(cuobjdump) or cxxfilt is None:
        pytest.skip('cuobjdump / c++filt not available')
    symbols = subprocess.run([cuobjdump, '-symbols', _lib.library_path], capture_output=True, text=True,
                             check=True).stdout
    mangled = sorted(set(re.findall(r'\b(_Z\w*ctrlmat_\w*_kernel\w*)', symbols)))
    names = subprocess.run([cxxfilt], input='\n'.join(mangled), capture_output=True, text=True,
                           check=True).stdout.split('\n')
    # "(anonymous namespace)::ctrlmat_static_kernel<12, 4, 6, 2, true>(...)" -> without namespace / arguments
    return {re.search(r'ctrlmat_\w+_kernel(<[^>]*>)?', n).group(0) for n in names if 'ctrlmat_' in n}


def test_ledger_covers_every_compiled_instance():
    compiled = _compiled_instances()
    assert len(compiled) >= 39
    assert compiled == set(ledger.LEDGER), (
        f'compiled but not in the ledger: {sorted(compiled - set(ledger.LEDGER))}; '
        f'in the ledger but not compiled: {sorted(set(ledger.LEDGER) - compiled)}')
    for kernel, cases in ledger.LEDGER.items():
        if kernel in ledger.UNREACHABLE:
            probe, reason = ledger.UNREACHABLE[kernel]
            assert probe in ledger.CASES and reason
            continue
        splits = [ledger.CASES[c]['S'] for c in cases]
        assert 1 in splits and max(splits) > 1, (kernel, cases)
