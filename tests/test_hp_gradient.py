"""The extended-precision gradient reference (tests/hp_gradient.py) and the gradient ledger
(tests/test_gpu_gradient.py), checked without a GPU:

- (a) the 80-bit formula agrees with 30-digit mpmath central differences of the whole forward pipeline
  (eigendecomposition, propagators, control matrix, filter function, trapezoid rule) to 1e-14 relative;
- (b) the float64 evaluation of the formula stays within KAPPA * EPS * M on every ledger case;
- (c) the ledger names exactly the gradient kernel instances compiled into libffb200.so.
"""
import os
import re
import shutil
import subprocess

import mpmath
import numpy as np
import pytest

import ff_oracle as oracle
import hp_gradient as hg
import test_gpu_gradient as ledger


def _herm(rng, d, n):
    A = rng.standard_normal((n, d, d)) + 1j*rng.standard_normal((n, d, d))
    return (A + A.conj().transpose(0, 2, 1))/2


def _mp_infidelity(c_opers, c_coeffs, n_opers, n_coeffs, dt, basis, omega, S, norm_d):
    """I_a of every noise operator in 30-digit arithmetic; c_coeffs / n_coeffs are mpf matrices."""
    mat = lambda a: mpmath.matrix([[mpmath.mpc(complex(x)) for x in row] for row in a])  # noqa: E731
    d = c_opers.shape[-1]
    G, n_nops, n_basis, n_omega = len(dt), len(n_opers), len(basis), len(omega)
    A, N, Cb = [mat(a) for a in c_opers], [mat(a) for a in n_opers], [mat(a) for a in basis]
    w = [mpmath.mpf(float(x)) for x in omega]
    Q = mpmath.eye(d)
    t = mpmath.mpf(0)
    B = [[[mpmath.mpc(0)]*n_omega for _ in range(n_basis)] for _ in range(n_nops)]
    for g in range(G):
        H = mpmath.zeros(d, d)
        for h in range(len(A)):
            H += A[h]*c_coeffs[h][g]
        E, V = mpmath.eighe(H)
        dtg = mpmath.mpf(float(dt[g]))
        QdV = Q.H*V
        Cbar = [QdV.H*C*QdV for C in Cb]
        Bbar = [V.H*N[j]*V*n_coeffs[j][g] for j in range(n_nops)]
        for o in range(n_omega):
            phase = mpmath.expj(w[o]*t)
            I = mpmath.matrix(d, d)
            for m in range(d):
                for n in range(d):
                    y = (w[o] + E[m] - E[n])*dtg/2   # no cancellation near a resonance
                    I[m, n] = dtg*mpmath.expj(y)*mpmath.sinc(y)
            for j in range(n_nops):
                BI = mpmath.matrix(d, d)
                for m in range(d):
                    for n in range(d):
                        BI[m, n] = Bbar[j][m, n]*I[m, n]
                for k in range(n_basis):
                    B[j][k][o] += phase*sum(BI[m, n]*Cbar[k][n, m] for m in range(d) for n in range(d))
        P = V*mpmath.diag([mpmath.expj(-e*dtg) for e in E])*V.H
        Q = P*Q
        t += dtg
    out = []
    for j in range(n_nops):
        F = [sum(abs(B[j][k][o])**2 for k in range(n_basis)) for o in range(n_omega)]
        f = [mpmath.mpf(float(S[j][o]))*F[o] for o in range(n_omega)]
        out.append(sum((f[o] + f[o + 1])*(w[o + 1] - w[o]) for o in range(n_omega - 1))/2
                   /(2*mpmath.pi*norm_d))
    return out


def _truth_case(k):
    """Tiny pulses that together hit every special branch of the formula."""
    rng = np.random.default_rng(100 + k)
    d = [1, 2, 3, 2, 3, 2, 3, 2, 3, 3][k]
    G, n_omega = 4 if d == 3 else 5, 5 if d == 3 else 6
    c_opers = _herm(rng, d, 2)
    if d >= 2 and k in (2, 4, 8):
        # control 0 has a degenerate (k = 2, 8) or 1e-10-split (k = 4) spectrum; segment 1 uses it alone
        diag = np.ones(d)
        diag[-1] = -1.0
        if k == 4:
            diag[0] += 1e-10
        c_opers[0] = np.diag(diag)
    c_coeffs = rng.standard_normal((2, G))
    if k in (2, 4, 8):
        c_coeffs[1, 1] = 0.0
    c_coeffs[:, G - 2] = 0.0 if k % 2 == 0 else c_coeffs[:, G - 2]   # an H = 0 segment
    dt = 1 - rng.random(G)
    if k in (3, 6, 9):
        dt[1] = 0.0                                                  # a dt = 0 segment
    n_opers = _herm(rng, d, 2)
    if k in (5, 6, 7, 9):
        n_opers[1] = n_opers[1] + 0.5j*np.triu(np.ones((d, d)), 1)   # not Hermitian
    import filter_functions_b200 as ff
    basis = np.asarray(ff.Basis.ggm(d)) if d > 1 else np.ones((1, 1, 1), dtype=complex)
    if k in (3, 7, 9) and d > 1:
        basis = basis[[0, d*d - 1] if d == 2 else [0, 2, 5, 7]]      # incomplete
    n_coeffs = rng.random((2, G)) + 0.5
    deps = None
    if k >= 5 or d == 1:  # at d = 1 the controls only enter through the sensitivities
        deps = rng.standard_normal((2, 2, G))
        n_coeffs[0, 2] = 0.0                                         # s = 0 on one segment
    H = oracle.hamiltonian_from_coeffs(c_opers, c_coeffs)
    ev = np.linalg.eigvalsh(H)
    split = ev[0, -1] - ev[0, 0] if d > 1 else 0.5
    omega = np.sort(np.array([0.0, -1.1, 0.7, 2.3, split + 1e-9, -split][:n_omega]))
    S = rng.random((2, n_omega)) + 0.2
    return c_opers, c_coeffs, n_opers, n_coeffs, dt, basis, omega, S, deps


@pytest.mark.parametrize('k', range(10))
def test_formula_against_mpmath_differences(k):
    mpmath.mp.dps = 30
    c_opers, c_coeffs, n_opers, n_coeffs, dt, basis, omega, S, deps = _truth_case(k)
    d, G = c_opers.shape[-1], len(dt)
    H = oracle.hamiltonian_from_coeffs(c_opers, c_coeffs)
    ev, V, Q = oracle.diagonalize(H, dt)
    t = np.concatenate(([0.0], dt.cumsum()))
    dI, _ = hg.derivative(ev, V, Q, omega, basis, n_opers, n_coeffs, dt, t, c_opers, S, deps)
    h = mpmath.mpf('1e-12')
    cc = [[mpmath.mpf(float(x)) for x in row] for row in c_coeffs]
    nc = [[mpmath.mpf(float(x)) for x in row] for row in n_coeffs]
    fd = np.zeros(dI.shape)
    for hh in range(2):
        for g in range(G):
            vals = []
            for sign in (1, -1):
                c2 = [row[:] for row in cc]
                n2 = [row[:] for row in nc]
                c2[hh][g] += sign*h
                if deps is not None:
                    for j in range(2):
                        n2[j][g] += sign*h*mpmath.mpf(float(deps[j, hh, g]))
                vals.append(_mp_infidelity(c_opers, c2, n_opers, n2, dt, basis, omega, S, d))
            fd[:, g, hh] = [float((a - b)/(2*h)) for a, b in zip(*vals)]
    err = np.abs(dI.astype(float) - fd).max()/np.abs(fd).max()
    print(f'[gradient truth] case {k} (d={d}): max |dI_hp - dI_mp| / max |dI| = {err:.2e}')
    assert err < 1e-14


@pytest.mark.parametrize('name', list(ledger.CASES))
def test_float64_formula_within_bound(name):
    inputs = ledger.build_inputs(name)
    H = oracle.hamiltonian_from_coeffs(inputs['c_opers'], inputs['c_coeffs'])
    ev, V, Q = oracle.diagonalize(H, inputs['dt'])
    t = np.concatenate(([0.0], np.asarray(inputs['dt']).cumsum()))
    B = oracle.control_matrix_from_scratch(ev, V, Q, inputs['omega'], inputs['basis'], inputs['n_opers'],
                                           inputs['n_coeffs'], inputs['dt'], t)
    dI_hp, M = ledger.reference(inputs, ev, V, Q)
    dI, _ = ledger.reference(inputs, ev, V, Q, hp=False, control_matrix=B)
    r = hg.ratio(dI, dI_hp, M)
    print(f'[gradient] float64 formula, {name}: worst ratio {r.max():.3g}')
    assert r.max() <= ledger.KAPPA


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
    mangled = sorted(set(re.findall(r'\b(_Z\w*grad_\w*_kernel\w*)', symbols)))
    names = subprocess.run([cxxfilt], input='\n'.join(mangled), capture_output=True, text=True,
                           check=True).stdout.split('\n')
    return {re.search(r'grad_\w+_kernel(<[^>]*>)?', n).group(0) for n in names if 'grad_' in n}


def test_ledger_covers_every_compiled_instance():
    compiled = _compiled_instances()
    assert compiled == set(ledger.LEDGER), (
        f'compiled but not in the ledger: {sorted(compiled - set(ledger.LEDGER))}; '
        f'in the ledger but not compiled: {sorted(set(ledger.LEDGER) - compiled)}')
    for kernel, cases in ledger.LEDGER.items():
        chunks = [-(-ledger.CASES[c]['G']//ledger.CASES[c]['L']) for c in cases]
        assert max(chunks) > 1, kernel
        assert any(ledger.CASES[c]['G'] % ledger.CASES[c]['L'] for c in cases if
                   ledger.CASES[c]['G'] > ledger.CASES[c]['L']), kernel   # a ragged last chunk
        if not kernel.startswith('grad_chunk_kernel'):
            assert 1 in chunks, kernel
