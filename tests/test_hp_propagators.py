"""The extended-precision front-end reference (tests/hp_propagators.py) and the ledger of front-end kernel
instances (tests/test_gpu_diag_instances.py), checked without a GPU:

- the reference agrees with 30-digit mpmath (expm, eighe, the sequential product) on the special cases,
  to 1e-3 of the bounds it is used with;
- the float64 oracle (numpy.linalg.eigh and its sequential product) stays within KAPPA of every
  bound on every ledger case, so the bounds are sound;
- the ledger names exactly the diag* / scan* kernel instances compiled into libffb200.so.
"""
import os
import re
import shutil
import subprocess

import mpmath
import numpy as np
import pytest

import ff_oracle as oracle
import hp_propagators as hp
import test_gpu_diag_instances as ledger
from helpers import rand_herm


def _mp(x):
    return mpmath.matrix([[mpmath.mpc(complex(v).real, complex(v).imag) for v in row] for row in x])


def _mpc(z):
    """A clongdouble as mpmath number, exactly (the shortest repr of a long double round-trips)."""
    return mpmath.mpc(mpmath.mpf(str(z.real)), mpmath.mpf(str(z.imag)))


def _special(kind, rng):
    """(H, dt) of a special case of the reference check."""
    if kind == 'diagonal':
        H = np.array([np.diag([0.3, -1.2, 0.3, 2.0])])
        return H, np.array([0.7])
    if kind == 'identity':
        return np.array([-1.7*np.eye(3)]), np.array([0.45])
    if kind == 'kron':
        return np.kron(rand_herm(rng, 2, 2), np.eye(2)), np.array([0.5, 1.3])
    if kind == 'cluster':
        lam = np.array([1.0, 1.0 + 1e-15, -1.0, -1.0 + 2e-15])
        U = np.linalg.qr(rng.standard_normal((4, 4)) + 1j*rng.standard_normal((4, 4)))[0]
        return np.array([(U*lam) @ U.conj().T]), np.array([0.9])
    if kind == 'large':
        H = rand_herm(rng, 2, 2)
        return H, 1e4/hp.spectral_norms(H)
    if kind == 'dt0':
        return rand_herm(rng, 3, 2), np.array([0.0, 0.6])
    if kind == 'd1':
        return np.array([[[2.5]], [[-0.75]], [[1e3]]], dtype=complex), np.array([0.3, 0.2, 0.9])
    return rand_herm(rng, 3, 3), 1 - rng.random(3)


@pytest.mark.parametrize('kind', ['diagonal', 'identity', 'kron', 'cluster', 'large', 'dt0', 'd1', 'random'])
def test_reference_against_mpmath(kind):
    rng = np.random.default_rng(len(kind))
    H, dt = _special(kind, rng)
    G, d, _ = H.shape
    ref = hp.Reference(H, dt)
    m = hp.segment_scale(H, dt)
    with mpmath.workdps(30):
        Q_mp = mpmath.eye(d)
        for g in range(G):
            P_mp = mpmath.expm(-1j*mpmath.mpf(float(dt[g]))*_mp(H[g]))
            dev = max(abs(_mpc(ref.P[g][i, j]) - P_mp[i, j]) for i in range(d) for j in range(d))
            # the bound of one step (depth 1, KAPPA = 1)
            assert dev <= 1e-3*hp.EPS*(m[g] + d), (kind, g, float(dev))
            Q_mp = P_mp*Q_mp
            dev = max(abs(_mpc(ref.Q[g + 1][i, j]) - Q_mp[i, j]) for i in range(d) for j in range(d))
            assert dev <= 1e-3*hp.EPS*(d + m[:g + 1].sum()), (kind, g, float(dev))
            E = sorted(mpmath.eighe(_mp(H[g]), eigvals_only=True))
            dev = max(abs(mpmath.mpf(str(ref.ev[list(ref.idx).index(g), j])) - E[j]) for j in range(d))
            assert dev <= 1e-3*hp.EPS*d*max(ref.norms[g], 1e-300)
    if kind == 'diagonal':  # exact where the answer is known
        assert (ref.ev[0] == np.sort(np.diag(H[0]).real).astype(hp.LD)).all()


def test_reference_rejects_a_small_error():
    """A relative error of 1e-13 in one step's propagator, harmless to a normalised 1e-10 comparison,
    breaks the step bound of the kernels."""
    rng = np.random.default_rng(5)
    H, dt = rand_herm(rng, 4, 50), 1 - rng.random(50)
    ref = hp.Reference(H, dt)
    ev, V, Q = oracle.diagonalize(H, dt)
    assert max(ref.ratios(ev, V, Q, 1).values()) <= ledger.KAPPA
    P = Q[1:] @ np.linalg.inv(Q[:-1])
    P[20] *= 1 + 1e-13
    Q_bad = Q.copy()
    for g in range(20, 50):
        Q_bad[g + 1] = P[g] @ Q_bad[g]
    assert ref.ratios(ev, V, Q_bad, 1)['step'] > ledger.KAPPA
    assert np.abs(Q_bad - Q).max() < 1e-10


_worst = {}


@pytest.mark.parametrize('name', list(ledger.CASES))
def test_oracle_within_bounds(name):
    inputs = ledger.build_inputs(name)
    ev, V, Q = oracle.diagonalize(inputs['H'], inputs['dt'])
    ratios = ledger.reference(inputs).ratios(ev, V, Q, hp.scan_depth('oracle', ev.shape[1], len(ev)))
    for b, r in ratios.items():
        _worst[b] = max(_worst.get(b, 0.0), r)
    bad = {k: v for k, v in ratios.items() if not v <= ledger.KAPPA}
    assert not bad, f'{name}: {bad}'


def test_zz_oracle_report():
    """The float64 oracle's largest error / (EPS scale) per bound over the ledger cases."""
    print('oracle: ' + ', '.join(f'{b} {_worst[b]:.3g}' for b in ledger.BOUNDS if b in _worst))


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
    mangled = sorted(set(re.findall(r'\b(_Z\w*(?:diag|scan)_\w*kernel\w*)', symbols)))
    names = subprocess.run([cxxfilt], input='\n'.join(mangled), capture_output=True, text=True,
                           check=True).stdout.split('\n')
    # "(anonymous namespace)::scan_block_kernel<4, 128>(...)" -> without namespace / arguments
    found = (re.search(r'\b((?:diag|scan)_\w*kernel)(<[^>]*>)?\(', n) for n in names)
    return {m.group(1) + (m.group(2) or '') for m in found if m}


def test_ledger_covers_every_compiled_instance():
    compiled = _compiled_instances()
    assert len(compiled) == 16
    assert compiled == set(ledger.LEDGER), (
        f'compiled but not in the ledger: {sorted(compiled - set(ledger.LEDGER))}; '
        f'in the ledger but not compiled: {sorted(set(ledger.LEDGER) - compiled)}')
    assert all(ledger.LEDGER.values())
