"""The banded route of the control matrix (DESIGN 4.1.1), checked against the extended-precision reference.

Pulses of at least 1024 segments on the tensor path evaluate dense frequency bands by Chebyshev interpolation
of per-chunk partial sums.  Each case draws seeded inputs whose grid holds bands that pay (many targets) and
bands that do not (a sparse tail), plus the special frequencies: 0, a negative one, the level splittings
+-fl(E_m - E_n) of a sampled segment, the edges k W of the band lattice and the end proxies of a band.  It
checks

- the dispatch record: instance, route, chunk length, bands and proxies;
- |B - B_hp| <= KAPPA * EPS * M at up to 128 sampled targets (tests/hp_control_matrix.py), the bound every
  kernel instance meets on the direct route;
- that a second call repeats every bit.
"""
import zlib

import numpy as np
import pytest

import ff_oracle as oracle
import hp_control_matrix as hp
from helpers import rand_herm

pytestmark = pytest.mark.gpu

KAPPA = 8
BAND_P, BAND_SIGMA, QUANTUM = 48, 16.0, 128

_STATIC_SPLIT = 'ctrlmat_static_kernel<12, 4, 6, 2, true>'

CASES = {
    # d = 4 Pauli basis, six noise operators: the identity-split static instance, uniform dt
    'split_uniform': dict(kernel=_STATIC_SPLIT, d=4, G=1500, n_nops=6, dt='const', route='function', blocks=1),
    # every segment its own dt and one long segment (the longest chunk sets the band width)
    'split_ragged_long': dict(kernel=_STATIC_SPLIT, d=4, G=1100, n_nops=6, dt='long', route='function',
                              blocks=1),
    # the pulse pipeline in three frequency blocks
    'pulse_blocks3': dict(kernel=_STATIC_SPLIT, d=4, G=1030, n_nops=6, dt='const', route='pulse', blocks=3),
    # generic tensor kernel, d = 5
    'generic_d5': dict(kernel='ctrlmat_main_kernel<4, 8>', d=5, G=1100, n_nops=2, n_basis=16, dt='rand',
                       route='function', blocks=1),
}


def band_width(dt, L):
    """W = 4 sigma / T_c, T_c the longest chunk of L segments, in the plan kernel's order of operations."""
    t = np.concatenate(([0.0], np.cumsum(dt)))
    G = len(dt)
    T_c = max((t[g1 - 1] + dt[g1 - 1]) - t[g0] for g0, g1 in ((g, min(G, g + L)) for g in range(0, G, L)))
    return 4*BAND_SIGMA/T_c


def build_inputs(name):
    c = CASES[name]
    d, G, n_nops = c['d'], c['G'], c['n_nops']
    n_basis = c.get('n_basis', d*d)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    c_opers = rand_herm(rng, d, 2)
    c_coeffs = rng.standard_normal((2, G))
    if c['dt'] == 'const':
        dt = np.full(G, 0.2)
    elif c['dt'] == 'long':
        dt = 0.2*(1 + 0.5*rng.random(G))
        dt[G//2 + 7] = 4.0
    else:
        dt = 0.15 + 0.1*rng.random(G)
    ev, V, Q = oracle.diagonalize(oracle.hamiltonian_from_coeffs(c_opers, c_coeffs), dt)
    n_opers = rand_herm(rng, d, n_nops)
    if d == 4:
        import filter_functions_b200 as ff
        basis = np.asarray(ff.Basis.pauli(2))        # element 0 is the identity
    else:
        basis = rand_herm(rng, d, n_basis)
    n_coeffs = rng.random((n_nops, G)) + 0.5
    t = np.concatenate(([0.0], dt.cumsum()))
    W = band_width(dt, QUANTUM)
    g = int(rng.integers(G))
    dE = np.subtract.outer(ev[g], ev[g])[np.triu_indices(d, 1)]
    # dense below 3 W (bands that pay), sparse above (bands that do not)
    dense = np.geomspace(1e-3, 3*W, 900)
    sparse = np.geomspace(3.2*W, 60.0, 40)
    special = [0.0, -0.37, -dE[0], dE[0], W, 2*W, 0.5*W + 0.5*W, 1.5*W - 0.5*W, 2.5*W + 0.5*W]
    omega = np.sort(np.concatenate((dense, sparse, special)))
    pick = np.unique(np.concatenate((
        np.searchsorted(omega, special),
        rng.choice(len(omega), 128 - len(special), replace=False))))[:128]
    return dict(eigvals=ev, eigvecs=V, propagators=Q, omega=omega, basis=basis, n_opers=n_opers,
                n_coeffs=n_coeffs, dt=dt, t=t, c_opers=c_opers, c_coeffs=c_coeffs, pick=pick)


def compute(ff, name, inputs):
    from filter_functions_b200 import _lib
    c = CASES[name]
    _lib.dispatch_log()
    if c['route'] == 'pulse':
        pulse = ff.PulseSequence(list(zip(inputs['c_opers'], inputs['c_coeffs'])),
                                 list(zip(inputs['n_opers'], inputs['n_coeffs'])), inputs['dt'],
                                 ff.Basis.pauli(2))
        ff.infidelity(pulse, 1/(1 + inputs['omega']**2), inputs['omega'])
        B = pulse.get_control_matrix(inputs['omega'])
        inputs = dict(inputs, eigvals=pulse.eigvals, eigvecs=pulse.eigvecs, propagators=pulse.propagators,
                      basis=np.asarray(pulse.basis), n_opers=np.asarray(pulse.n_opers),
                      n_coeffs=np.asarray(pulse.n_coeffs), t=pulse.t)
    else:
        B = ff.numeric.calculate_control_matrix_from_scratch(
            *(inputs[k] for k in ('eigvals', 'eigvecs', 'propagators', 'omega', 'basis', 'n_opers',
                                  'n_coeffs', 'dt', 't')))
    return np.array(B), _lib.dispatch_log(), inputs


@pytest.mark.parametrize('name', list(CASES))
def test_banded_case(engine, monkeypatch, name):
    c = CASES[name]
    if c['blocks'] > 1:
        monkeypatch.setenv('FFB_PIPELINE_BLOCKS', str(c['blocks']))
    inputs = build_inputs(name)
    B, records, inputs = compute(engine, name, inputs)
    assert len(records) == c['blocks'], records
    for rec in records:
        assert rec['kernel'] == c['kernel'], rec
        assert (rec['route'], rec['chunk_segs']) == (1, QUANTUM), rec
        assert rec['S'] == -(-c['G']//QUANTUM) and rec['passes_per_chunk'] == QUANTUM//4, rec
        assert rec['n_proxies'] == BAND_P*rec['n_bands'], rec
    assert sum(rec['n_bands'] for rec in records) >= 2, records
    assert sum(rec['n_omega'] for rec in records) == len(inputs['omega'])
    assert np.isfinite(B.view(float)).all()

    pick = inputs['pick']
    sub = dict(inputs, omega=inputs['omega'][pick])
    B_hp, M = hp.control_matrix(*(sub[k] for k in ('eigvals', 'eigvecs', 'propagators', 'omega', 'basis',
                                                   'n_opers', 'n_coeffs', 'dt', 't')))
    r = hp.ratio(B[..., pick], B_hp, M)
    worst = np.unravel_index(r.argmax(), r.shape)
    assert r.max() <= KAPPA, f'{name}: |B - B_hp| / (EPS M) = {r.max():.2f} at omega = ' \
                             f'{inputs["omega"][pick][worst[-1]]!r} {worst}'

    if c['route'] == 'function':   # a second call repeats every bit
        B2, _, _ = compute(engine, name, inputs)
        assert np.array_equal(B.view(np.uint64), B2.view(np.uint64))
