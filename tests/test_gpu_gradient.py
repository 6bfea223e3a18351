"""ff.infidelity_derivative on the GPU against the extended-precision reference (tests/hp_gradient.py).

The ledger reaches every compiled gradient kernel instance (d = 1 ... 8) with one case whose segment axis is
one chunk and one with several chunks and a ragged last chunk; grad_chunk_kernel<d> only runs when there
is more than one chunk.  FFB_GRAD_SEGS_PER_CHUNK fixes the split.  Every entry of every case must satisfy
|dI_gpu - dI_hp| <= KAPPA * EPS * M.
"""
import os

import numpy as np
import pytest

import hp_gradient as hg
import workloads

KAPPA = 16

# name -> d, G, n_omega, segments per chunk, noise operators, controls, options
CASES = {}
for _d in range(1, 9):
    CASES[f'd{_d}_one_chunk'] = dict(d=_d, G=5, n_omega=9, L=5, n_nops=2, n_cops=2, seed=10 + _d)
    CASES[f'd{_d}_chunks'] = dict(d=_d, G=11, n_omega=7, L=4, n_nops=2, n_cops=3, seed=30 + _d,
                                  spectrum_2d=True, deps=True)
CASES['d2_subsets'] = dict(d=2, G=9, n_omega=12, L=2, n_nops=3, n_cops=3, seed=51, spectrum_2d=True,
                           controls=[2, 0], nops=[2, 0], deps=True)
CASES['d3_incomplete_nonherm'] = dict(d=3, G=6, n_omega=10, L=6, n_nops=2, n_cops=2, seed=52,
                                      basis_rows=[0, 2, 5, 7], nonherm=True)
CASES['c2'] = dict(workload='c2', G=40, n_omega=64, L=40, seed=0)
CASES['c2_chunks'] = dict(workload='c2', G=40, n_omega=64, L=7, seed=0, spectrum_2d=True)
CASES['d4'] = dict(workload='d4', G=30, n_omega=48, L=30, seed=0, deps=True)
CASES['d4_chunks'] = dict(workload='d4', G=30, n_omega=48, L=8, seed=0, deps=True,
                          controls=[4, 0, 2], nops=[5, 1, 0])

LEDGER = {}
for _d in range(1, 9):
    LEDGER[f'grad_prologue_kernel<{_d}>'] = [f'd{_d}_one_chunk', f'd{_d}_chunks']
    LEDGER[f'grad_sweep_kernel<{_d}>'] = [f'd{_d}_one_chunk', f'd{_d}_chunks']
    LEDGER[f'grad_chunk_kernel<{_d}>'] = [f'd{_d}_chunks']
LEDGER['grad_reduce_kernel'] = list(CASES)


def _herm(rng, d, n):
    A = rng.standard_normal((n, d, d)) + 1j*rng.standard_normal((n, d, d))
    return (A + A.conj().transpose(0, 2, 1))/2


def build_inputs(name):
    """The pulse arrays, frequencies, spectrum and options of a ledger case."""
    case = CASES[name]
    rng = np.random.default_rng(case['seed'])
    if 'workload' in case:
        wl = workloads.get(case['workload'], G=case['G'], n_omega=case['n_omega'])
        inputs = dict(c_opers=wl.c_opers, c_ids=list(wl.c_ids), c_coeffs=wl.c_coeffs, n_opers=wl.n_opers,
                      n_ids=list(wl.n_ids), n_coeffs=wl.n_coeffs, dt=wl.dt,
                      basis=np.asarray(wl.basis, dtype=complex), omega=wl.omega)
        n_nops, n_cops = len(wl.n_opers), len(wl.c_opers)
        deps = None
        if case.get('deps'):  # sensitivities J_i = c_coeffs[i] of the exchange workload
            deps = np.zeros((n_nops, n_cops, case['G']))
            for i in range(3):
                deps[i, i] = 1.0
        base = wl.spectrum
    else:
        d, G, n_omega = case['d'], case['G'], case['n_omega']
        n_nops, n_cops = case['n_nops'], case['n_cops']
        n_opers = _herm(rng, d, n_nops)
        if case.get('nonherm'):
            n_opers[1] = n_opers[1] + 0.4j*np.triu(np.ones((d, d)), 1)
        import filter_functions_b200 as ff
        basis = np.asarray(ff.Basis.ggm(d)) if d > 1 else np.ones((1, 1, 1), dtype=complex)
        if 'basis_rows' in case:
            basis = basis[case['basis_rows']]
        c_coeffs = rng.standard_normal((n_cops, G))
        c_coeffs[:, G//2] = 0.0                               # an H = 0 segment
        dt = 1 - rng.random(G)
        omega = np.sort(np.concatenate(([0.0, -1.3], 6*rng.standard_normal(n_omega - 2))))
        inputs = dict(c_opers=_herm(rng, d, n_cops), c_ids=[f'c{i}' for i in range(n_cops)],
                      c_coeffs=c_coeffs, n_opers=n_opers, n_ids=[f'n{i}' for i in range(n_nops)],
                      n_coeffs=rng.random((n_nops, G)) + 0.5, dt=dt, basis=np.ascontiguousarray(basis),
                      omega=omega)
        deps = rng.standard_normal((n_nops, n_cops if 'controls' not in case else len(case['controls']),
                                    G)) if case.get('deps') else None
        base = 1/(1 + inputs['omega']**2)
    controls = case.get('controls')
    nops = case.get('nops')
    n_sel = len(nops) if nops is not None else n_nops
    if deps is not None and controls is not None and deps.shape[1] != len(controls):
        deps = np.ascontiguousarray(deps[:, controls])
    spectrum = (base[None]*(1 + np.arange(n_sel))[:, None]) if case.get('spectrum_2d') else base
    inputs.update(spectrum=np.ascontiguousarray(spectrum), deps=deps, L=case['L'],
                  control_identifiers=None if controls is None else [inputs['c_ids'][i] for i in controls],
                  n_oper_identifiers=None if nops is None else [inputs['n_ids'][i] for i in nops],
                  ctrl_idx=np.arange(n_cops) if controls is None else np.asarray(controls),
                  nop_idx=np.arange(n_nops) if nops is None else np.asarray(nops))
    return inputs


def make_pulse(ff, inputs):
    return ff.PulseSequence.from_arrays(
        inputs['c_opers'], inputs['c_ids'], inputs['c_coeffs'], inputs['n_opers'], inputs['n_ids'],
        inputs['n_coeffs'], inputs['dt'], basis=inputs['basis'])


def reference(inputs, eigvals, eigvecs, propagators, hp=True, control_matrix=None):
    t = np.concatenate(([0.0], np.asarray(inputs['dt']).cumsum()))
    return hg.derivative(eigvals, eigvecs, propagators, inputs['omega'], inputs['basis'],
                         inputs['n_opers'], inputs['n_coeffs'], inputs['dt'], t, inputs['c_opers'],
                         inputs['spectrum'], inputs['deps'], inputs['ctrl_idx'], inputs['nop_idx'],
                         hp=hp, control_matrix=control_matrix)


def _call(ff, pulse, inputs, **kwargs):
    os.environ['FFB_GRAD_SEGS_PER_CHUNK'] = str(inputs['L'])
    try:
        return ff.infidelity_derivative(pulse, inputs['spectrum'], inputs['omega'],
                                        control_identifiers=inputs['control_identifiers'],
                                        n_oper_identifiers=inputs['n_oper_identifiers'],
                                        n_coeffs_deps=inputs['deps'], **kwargs)
    finally:
        del os.environ['FFB_GRAD_SEGS_PER_CHUNK']


_WORST = {}


@pytest.mark.gpu
@pytest.mark.parametrize('name', list(CASES))
def test_case_within_bound(engine, name):
    ff = engine
    inputs = build_inputs(name)
    pulse = make_pulse(ff, inputs)
    pulse.diagonalize()
    dI = _call(ff, pulse, inputs)
    dI_hp, M = reference(inputs, pulse.eigvals, pulse.eigvecs, pulse.propagators)
    r = hg.ratio(dI, dI_hp, M)
    _WORST[name] = r.max()
    print(f'[gradient] {name}: worst |dI - dI_hp| / (EPS M) = {r.max():.3g}')
    assert r.max() <= KAPPA, (name, r.max(), np.unravel_index(r.argmax(), r.shape))


@pytest.mark.gpu
def test_per_instance_report():
    rows = []
    for kernel, cases in LEDGER.items():
        seen = [_WORST[c] for c in cases if c in _WORST]
        if seen:
            rows.append(f'{kernel}: {max(seen):.3g} over {len(seen)} cases')
    print('[gradient] worst ratio per instance:\n  ' + '\n  '.join(rows))


def _infid(ff, inputs, c_coeffs, n_coeffs):
    pulse = ff.PulseSequence.from_arrays(
        inputs['c_opers'], inputs['c_ids'], c_coeffs, inputs['n_opers'], inputs['n_ids'], n_coeffs,
        inputs['dt'], basis=inputs['basis'])
    S = inputs['spectrum']
    idx = inputs['nop_idx']
    return np.array([ff.infidelity(pulse, S[k] if S.ndim == 2 else S, inputs['omega'],
                                   n_oper_identifiers=[inputs['n_ids'][idx[k]]])[0]
                     for k in range(len(idx))])


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['d2_subsets', 'd3_incomplete_nonherm'])
def test_against_central_differences_of_infidelity(engine, name):
    """float64 central differences of ff.infidelity itself, at 1e-6 relative."""
    ff = engine
    inputs = build_inputs(name)
    dI = _call(ff, make_pulse(ff, inputs), inputs)
    h = 1e-5
    fd = np.zeros_like(dI)
    for col, ci in enumerate(inputs['ctrl_idx']):
        for g in range(len(inputs['dt'])):
            step = np.zeros_like(inputs['c_coeffs'])
            step[ci, g] = h
            dn = np.zeros_like(inputs['n_coeffs'])
            if inputs['deps'] is not None:
                dn[:, g] = inputs['deps'][:, col, g]*h
            fd[:, g, col] = (_infid(ff, inputs, inputs['c_coeffs'] + step, inputs['n_coeffs'] + dn)
                             - _infid(ff, inputs, inputs['c_coeffs'] - step,
                                      inputs['n_coeffs'] - dn))/(2*h)
    err = np.abs(dI - fd).max()/np.abs(fd).max()
    print(f'[gradient] {name}: central differences of ff.infidelity, max rel. deviation {err:.2e}')
    assert err < 1e-6


@pytest.mark.gpu
def test_repeat_is_bit_identical_and_cached_matches_cold(engine):
    ff = engine
    inputs = build_inputs('d4_chunks')
    cold = make_pulse(ff, inputs)
    first = _call(ff, cold, inputs)
    assert cold._is_cold(), 'the call must not cache anything'
    assert np.array_equal(first, _call(ff, cold, inputs))
    cached = make_pulse(ff, inputs)
    cached.get_control_matrix(inputs['omega'])
    warm = _call(ff, cached, inputs)
    print(f'[gradient] cached vs cold: bit-identical {np.array_equal(first, warm)}, '
          f'max |diff| / max |dI| = {np.abs(first - warm).max()/np.abs(first).max():.2e}')
    np.testing.assert_allclose(warm, first, rtol=0, atol=1e-13*np.abs(first).max())


@pytest.mark.gpu
def test_invalid_arguments(engine):
    ff = engine
    inputs = build_inputs('d2_subsets')
    pulse = make_pulse(ff, inputs)
    S, omega = inputs['spectrum'], inputs['omega']
    with pytest.raises(ValueError, match='Spectrum'):
        ff.infidelity_derivative(pulse, np.ones((3, 3, len(omega))), omega)
    with pytest.raises(ValueError, match='Spectrum'):
        ff.infidelity_derivative(pulse, np.ones(len(omega) + 1), omega)
    with pytest.raises(ValueError, match='identifiers'):
        ff.infidelity_derivative(pulse, S[0], omega, control_identifiers=['nope'])
    with pytest.raises(ValueError, match='identifiers'):
        ff.infidelity_derivative(pulse, S[0], omega, n_oper_identifiers=['nope'])
    with pytest.raises(ValueError, match='n_coeffs_deps'):
        ff.infidelity_derivative(pulse, S[0], omega, n_coeffs_deps=np.zeros((3, 2, len(pulse.dt))))
    rng = np.random.default_rng(9)
    big = ff.PulseSequence.from_arrays(_herm(rng, 9, 1), ['a'], rng.standard_normal((1, 3)),
                                       _herm(rng, 9, 1), ['n'], np.ones((1, 3)), np.ones(3))
    with pytest.raises(ValueError, match='d <= 8'):
        ff.infidelity_derivative(big, np.ones(4), np.linspace(0, 1, 4))
