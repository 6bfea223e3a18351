"""Every compiled instance of the control-matrix kernels, reached on purpose and checked entry by entry.

LEDGER maps each ``ctrlmat_*_kernel<...>`` instance of libffb200.so to the cases that reach it, or to the
reason it cannot be reached on a B200.  A case draws seeded inputs, computes the control matrix through
``numeric.calculate_control_matrix_from_scratch`` (or the pulse pipeline), and checks

- that the dispatch record (``_lib.dispatch_log``) names the intended instance, split ``S`` and number of
  frequency blocks -- a dispatch change that moves a case elsewhere fails here by name;
- that every entry is finite and within KAPPA * EPS * M of the extended-precision reference
  (tests/hp_control_matrix.py), M being the per-entry error scale of a float64 evaluation.

The expected instance and ``S`` of each case were read from the record of a B200 run: part of the choice
depends on the occupancy the device reports.  Every reachable instance has a case with S = 1 and one with
S > 1 whose last chunk is ragged (n_pass % passes_per_chunk != 0).
"""
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import ff_oracle as oracle
import hp_control_matrix as hp
from helpers import nerr, rand_herm

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

#: float64 kernels pass when |B - B_hp| <= KAPPA * EPS * M at every entry
KAPPA = 8


def case(kernel, d, G, n_nops, n_basis, S, n_omega=40, herm=(True, True), identity=False, dt='rand',
         omega='plain', env=None, route='function', blocks=1):
    return dict(kernel=kernel, d=d, G=G, n_nops=n_nops, n_basis=n_basis, S=S, n_omega=n_omega, herm=herm,
                identity=identity, dt=dt, omega=omega, env=env or {}, route=route, blocks=blocks)


_DFMA1, _DFMA3 = 'ctrlmat_dfma_kernel<{}, {}, 1>', 'ctrlmat_dfma_kernel<{}, {}, 3>'
_NH = (False, True)      # non-Hermitian noise operators: two parts per operator row
_NHB = (True, False)     # non-Hermitian basis

#: name -> case.  dt: 'rand' (every segment its own dt), 'pass' (dt constant over runs of 4 segments, so
#: it changes exactly at pass, DFMA stage, piece and chunk boundaries), 'const'.  omega: 'plain' (0, a
#: negative frequency, omega = -fl(E_m - E_n) of a sampled segment, one within 1e-9 of a splitting, and a
#: geometric grid), 'wide' (the same up to |omega t| = 1e7).
CASES = {
    # ---- DFMA, thread per frequency (rows <= 16, d = 2, 3); S > 1 from G = 256 on
    'dfma4_d2': case(_DFMA1.format(4, 4), 2, 37, 1, 4, 1, omega='wide'),
    'dfma4_d2_split': case(_DFMA1.format(4, 4), 2, 300, 1, 4, 2, dt='pass'),
    'dfma8_d2_nonherm': case(_DFMA1.format(8, 8), 2, 37, 1, 4, 1, herm=_NH),
    'dfma8_d2_split': case(_DFMA1.format(8, 8), 2, 300, 2, 4, 2, dt='pass'),
    'dfma12_d2': case(_DFMA1.format(12, 12), 2, 45, 3, 4, 1),
    'dfma12_d2_split': case(_DFMA1.format(12, 12), 2, 301, 3, 4, 2, dt='pass'),
    'dfma12_d2_identity_off': case(_DFMA1.format(12, 12), 2, 301, 3, 4, 2, identity=True,
                                   env={'FFB_DFMA_SPLIT_IDENTITY': '0'}),
    'dfma16_d2_nonherm_basis': case(_DFMA1.format(16, 16), 2, 37, 2, 4, 1, herm=_NHB),
    'dfma16_d2_split': case(_DFMA1.format(16, 16), 2, 300, 4, 4, 2, dt='pass'),
    'dfma4_d3': case(_DFMA3.format(4, 4), 3, 37, 1, 4, 1),
    'dfma4_d3_split': case(_DFMA3.format(4, 4), 3, 300, 1, 4, 2, dt='pass'),
    'dfma8_d3_nonherm': case(_DFMA3.format(8, 8), 3, 37, 1, 2, 1, herm=(False, False)),
    'dfma8_d3_split': case(_DFMA3.format(8, 8), 3, 300, 2, 4, 2, dt='pass'),
    'dfma12_d3': case(_DFMA3.format(12, 12), 3, 37, 1, 9, 1),
    'dfma12_d3_split': case(_DFMA3.format(12, 12), 3, 300, 1, 9, 2, dt='pass'),
    'dfma12_d3_identity_off': case(_DFMA3.format(12, 12), 3, 37, 1, 9, 1, identity=True,
                                   env={'FFB_DFMA_SPLIT_IDENTITY': '0'}),
    'dfma16_d3': case(_DFMA3.format(16, 16), 3, 37, 4, 4, 1),
    'dfma16_d3_split': case(_DFMA3.format(16, 16), 3, 300, 2, 4, 2, herm=_NHB, dt='pass'),
    # identity rows split off (basis element 0 = identity / sqrt(d))
    'dfma_id8_d2': case(_DFMA1.format(8, 6), 2, 37, 2, 4, 1, identity=True),
    'dfma_id8_d2_split': case(_DFMA1.format(8, 6), 2, 300, 2, 4, 2, identity=True, dt='pass'),
    'dfma_id12_d2': case(_DFMA1.format(12, 9), 2, 37, 3, 4, 1, identity=True),
    'dfma_id12_d2_split': case(_DFMA1.format(12, 9), 2, 301, 3, 4, 2, identity=True, dt='pass'),
    'dfma_id16_d2': case(_DFMA1.format(16, 12), 2, 37, 4, 4, 1, identity=True),
    'dfma_id16_d2_split': case(_DFMA1.format(16, 12), 2, 300, 4, 4, 2, identity=True, dt='pass'),
    'dfma_id12_d3': case(_DFMA3.format(12, 8), 3, 37, 1, 9, 1, identity=True),
    'dfma_id12_d3_split': case(_DFMA3.format(12, 8), 3, 300, 1, 9, 2, identity=True, dt='pass'),

    # ---- static d = 4 (6 level pairs), one pass per stage
    'static12_split_id': case('ctrlmat_static_kernel<12, 4, 6, 2, true>', 4, 37, 6, 16, 1, identity=True),
    'static12_split_id_S': case('ctrlmat_static_kernel<12, 4, 6, 2, true>', 4, 263, 6, 16, 8, identity=True,
                                dt='pass'),
    'static12_identity_off': case('ctrlmat_static_kernel<12, 4, 6, 2, false>', 4, 263, 6, 16, 8,
                                  identity=True, env={'FFB_CTRLMAT_SPLIT_IDENTITY': '0'}),
    'static12_nonherm': case('ctrlmat_static_kernel<12, 4, 6, 2, false>', 4, 37, 3, 16, 1, herm=_NH),
    'static12_wide_S': case('ctrlmat_static_kernel<12, 4, 6, 2, false>', 4, 263, 6, 16, 8, omega='wide',
                            dt='pass'),
    'static12_rb2_S': case('ctrlmat_static_kernel<12, 4, 6, 2, false>', 4, 263, 12, 16, 8, dt='pass'),
    'static10': case('ctrlmat_static_kernel<10, 4, 6, 1, false>', 4, 37, 5, 16, 1),
    'static10_S': case('ctrlmat_static_kernel<10, 4, 6, 1, false>', 4, 263, 5, 16, 8, dt='pass'),
    'static8': case('ctrlmat_static_kernel<8, 4, 6, 1, false>', 4, 37, 4, 16, 1),
    'static8_S': case('ctrlmat_static_kernel<8, 4, 6, 1, false>', 4, 263, 4, 16, 8, dt='pass'),
    'static6': case('ctrlmat_static_kernel<6, 8, 6, 1, false>', 4, 37, 3, 16, 1),
    'static6_S': case('ctrlmat_static_kernel<6, 8, 6, 1, false>', 4, 263, 3, 16, 8, dt='pass'),
    # ---- static d = 8 (28 level pairs), a pass in pieces
    'static8x28': case('ctrlmat_static_kernel<8, 4, 28, 4, false>', 8, 20, 2, 32, 1),
    'static8x28_S': case('ctrlmat_static_kernel<8, 4, 28, 4, false>', 8, 66, 2, 32, 2, dt='pass'),
    'static12x28': case('ctrlmat_static_kernel<12, 4, 28, 6, false>', 8, 20, 3, 32, 1),
    'static12x28_S': case('ctrlmat_static_kernel<12, 4, 28, 6, false>', 8, 66, 3, 32, 2, dt='pass'),
    # ---- static d = 16, transposed layout (short pulses)
    'static16T': case('ctrlmat_static_kernel<12, 4, 30, 7, false>', 16, 5, 1, 96, 1),
    'static16T_S': case('ctrlmat_static_kernel<12, 4, 30, 7, false>', 16, 17, 1, 96, 2),
    'static16T_nonherm_S': case('ctrlmat_static_kernel<12, 4, 30, 7, false>', 16, 17, 1, 48, 2, herm=_NH),

    # ---- generic tensor kernel, d = 5 (10 level pairs), rows = n_nops * n_basis set the row tiles
    'main1': case('ctrlmat_main_kernel<1, 8>', 5, 37, 1, 8, 1),
    'main1_S': case('ctrlmat_main_kernel<1, 8>', 5, 171, 1, 8, 3, dt='pass'),
    'main2': case('ctrlmat_main_kernel<2, 8>', 5, 37, 1, 16, 1),
    'main2_S': case('ctrlmat_main_kernel<2, 8>', 5, 171, 1, 16, 5, dt='pass'),
    'main3': case('ctrlmat_main_kernel<3, 8>', 5, 37, 1, 24, 1),
    'main3_S': case('ctrlmat_main_kernel<3, 8>', 5, 171, 1, 24, 5, dt='pass'),
    'main4_nonherm': case('ctrlmat_main_kernel<4, 8>', 5, 37, 1, 16, 1, herm=_NH),
    'main4_S': case('ctrlmat_main_kernel<4, 8>', 5, 171, 2, 16, 5, dt='pass'),
    'main5': case('ctrlmat_main_kernel<5, 8>', 5, 37, 2, 20, 1),
    'main5_S': case('ctrlmat_main_kernel<5, 8>', 5, 171, 2, 20, 5, dt='pass'),
    'main6': case('ctrlmat_main_kernel<6, 8>', 5, 37, 3, 16, 1),
    'main6_S': case('ctrlmat_main_kernel<6, 8>', 5, 171, 3, 16, 5, dt='pass'),
    'main7': case('ctrlmat_main_kernel<7, 4>', 5, 37, 4, 14, 1),
    'main7_S': case('ctrlmat_main_kernel<7, 4>', 5, 171, 4, 14, 5, dt='pass'),
    'main8': case('ctrlmat_main_kernel<8, 4>', 5, 37, 4, 16, 1),
    'main8_S': case('ctrlmat_main_kernel<8, 4>', 5, 171, 4, 16, 5, dt='pass'),
    'main10': case('ctrlmat_main_kernel<10, 4>', 5, 37, 5, 16, 1),
    'main10_S': case('ctrlmat_main_kernel<10, 4>', 5, 171, 5, 16, 5, dt='pass'),
    'main12': case('ctrlmat_main_kernel<12, 4>', 5, 37, 6, 16, 1),
    'main12_S': case('ctrlmat_main_kernel<12, 4>', 5, 171, 6, 16, 5, dt='pass'),

    # ---- the pulse pipeline (Pauli basis) in three frequency blocks (widths 64, 64, 22)
    'pulse_static_split_blocks': case('ctrlmat_static_kernel<12, 4, 6, 2, true>', 4, 67, 6, 16, 2,
                                      n_omega=150, identity=True, route='pulse', blocks=3,
                                      env={'FFB_PIPELINE_BLOCKS': '3'}),
    'pulse_dfma_blocks': case(_DFMA1.format(8, 6), 2, 300, 2, 4, 2, n_omega=150, identity=True,
                              route='pulse', blocks=3, env={'FFB_PIPELINE_BLOCKS': '3'}),
    # ---- fixed point on the int8 tensor cores (opt-in); its tolerance is that of its error model
    'int8_short': case('ctrlmat_i8_kernel', 4, 64, 6, 16, 1, identity=True, env={'FFB_CTRLMAT_INT8': '1'}),
    'int8': case('ctrlmat_i8_kernel', 4, 263, 6, 16, 5, identity=True, env={'FFB_CTRLMAT_INT8': '1'}),
}

#: instances no shape reaches on a B200, with the record that shows why
UNREACHABLE = {
    'ctrlmat_static_kernel<12, 4, 6, 1, false>': (
        'static12_wide_S', 'MT = 12 allows 3 CTAs per SM by registers (ctas_by_regs = 3): stage budget '
        '216 KiB / 3 / 2 = 36 KiB < one d = 4 pass of 40.6 KB, so the pass is always staged in two pieces'),
    'ctrlmat_static_kernel<10, 4, 6, 2, false>': (
        'static10_S', 'MT = 10: 3 CTAs per SM, 36 KiB budget >= one d = 4 pass of 33.9 KB: never two pieces'),
    'ctrlmat_static_kernel<8, 4, 6, 2, false>': (
        'static8_S', 'MT = 8: 3 CTAs per SM, 36 KiB budget >= one d = 4 pass of 27.3 KB: never two pieces'),
    'ctrlmat_static_kernel<6, 8, 6, 2, false>': (
        'static6_S', 'MT = 6: 1 CTA per SM (8 warps), 48 KiB budget >= one d = 4 pass of 20.6 KB'),
    'ctrlmat_static_kernel<8, 4, 28, 5, false>': (
        'static8x28_S', 'd = 8, MT = 8: 3 CTAs per SM, a pass of 119.5 KB fits 36 KiB pieces in n_sp = 4'),
    'ctrlmat_static_kernel<8, 4, 28, 6, false>': (
        'static8x28_S', 'd = 8, MT = 8: 3 CTAs per SM, a pass of 119.5 KB fits 36 KiB pieces in n_sp = 4'),
    'ctrlmat_static_kernel<12, 4, 28, 5, false>': (
        'static12x28_S', 'd = 8, MT = 12: 3 CTAs per SM, a pass of 177.9 KB needs n_sp = 6 pieces of 36 KiB'),
    'ctrlmat_static_kernel<12, 4, 28, 7, false>': (
        'static12x28_S', 'd = 8, MT = 12: 3 CTAs per SM, a pass of 177.9 KB needs n_sp = 6 pieces of 36 KiB'),
}

LEDGER = {}
for _name, _c in CASES.items():
    LEDGER.setdefault(_c['kernel'], []).append(_name)
for _kernel, (_probe, _reason) in UNREACHABLE.items():
    assert _kernel not in LEDGER, _kernel
    LEDGER[_kernel] = []


def build_inputs(name):
    """Seeded inputs of a case: dict of the arguments of calculate_control_matrix_from_scratch plus the
    pulse's control Hamiltonian (c_opers, c_coeffs)."""
    c = CASES[name]
    d, G, n_nops, n_basis = c['d'], c['G'], c['n_nops'], c['n_basis']
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    c_opers = rand_herm(rng, d, 2)
    c_coeffs = rng.standard_normal((2, G))
    if c['dt'] == 'rand':
        dt = 1 - rng.random(G)
    elif c['dt'] == 'pass':
        # runs of 4 segments; some consecutive runs share their dt, so not every pass boundary changes it
        dt = np.repeat(rng.choice([0.3, 0.45, 0.7], size=(G + 3)//4), 4)[:G]
    else:
        dt = np.full(G, 0.4)
    ev, V, Q = oracle.diagonalize(oracle.hamiltonian_from_coeffs(c_opers, c_coeffs), dt)

    def operators(n, hermitian):
        if hermitian:
            return rand_herm(rng, d, n)
        return rng.standard_normal((n, d, d)) + 1j*rng.standard_normal((n, d, d))

    n_opers = operators(n_nops, c['herm'][0])
    basis = operators(n_basis, c['herm'][1])
    if c['identity']:
        basis[0] = np.eye(d)/np.sqrt(d)
    n_coeffs = rng.random((n_nops, G)) + 0.5
    t = np.concatenate(([0.0], dt.cumsum()))
    # frequencies on the special branches of the integral, then a geometric grid
    g = int(rng.integers(G))
    dE = np.subtract.outer(ev[g], ev[g])[np.triu_indices(d, 1)]
    special = [0.0, -0.37, -dE[0], dE[-1]*(1 + 1e-9)]
    top = 1e7/t[-1] if c['omega'] == 'wide' else 60.0
    grid = np.geomspace(1e-2, top, c['n_omega'] - len(special))
    omega = np.concatenate((special, grid))
    return dict(eigvals=ev, eigvecs=V, propagators=Q, omega=omega, basis=basis, n_opers=n_opers,
                n_coeffs=n_coeffs, dt=dt, t=t, c_opers=c_opers, c_coeffs=c_coeffs)


def reference(inputs):
    return hp.control_matrix(*(inputs[k] for k in ('eigvals', 'eigvecs', 'propagators', 'omega', 'basis',
                                                   'n_opers', 'n_coeffs', 'dt', 't')))


def compute(ff, name, inputs):
    """The control matrix of a case through its route, with the dispatch records of the call."""
    from filter_functions_b200 import _lib
    c = CASES[name]
    _lib.dispatch_log()
    if c['route'] == 'pulse':
        pulse = ff.PulseSequence(list(zip(inputs['c_opers'], inputs['c_coeffs'])),
                                 list(zip(inputs['n_opers'], inputs['n_coeffs'])), inputs['dt'],
                                 ff.Basis.pauli(int(np.log2(c['d']))))
        ff.infidelity(pulse, 1/(1 + inputs['omega']**2), inputs['omega'])
        B = pulse.get_control_matrix(inputs['omega'])
        # the reference is fed with the pulse's own eigensystem and basis
        inputs = dict(inputs, eigvals=pulse.eigvals, eigvecs=pulse.eigvecs, propagators=pulse.propagators,
                      basis=np.asarray(pulse.basis), n_opers=np.asarray(pulse.n_opers),
                      n_coeffs=np.asarray(pulse.n_coeffs), t=pulse.t)
    else:
        B = ff.numeric.calculate_control_matrix_from_scratch(
            *(inputs[k] for k in ('eigvals', 'eigvecs', 'propagators', 'omega', 'basis', 'n_opers',
                                  'n_coeffs', 'dt', 't')))
    return np.array(B), _lib.dispatch_log(), inputs


def check_record(name, records):
    c = CASES[name]
    assert len(records) == c['blocks'], (name, records)
    for rec in records:
        assert rec['kernel'] == c['kernel'], \
            f"{name}: dispatched to {rec['kernel']}, the ledger expects {c['kernel']} ({rec})"
        assert rec['S'] == c['S'], f"{name}: S = {rec['S']}, the ledger expects {c['S']} ({rec})"
        assert rec['n_blocks'] == c['blocks']
    if c['S'] > 1:
        rec = records[0]
        assert rec['n_pass'] % rec['passes_per_chunk'] != 0, f'{name}: last chunk not ragged ({rec})'
    if c['blocks'] > 1:
        widths = [rec['n_omega'] for rec in records]
        assert sum(widths) == c['n_omega'] and len(set(widths)) > 1, widths


def _env(monkeypatch, name):
    for key, value in CASES[name]['env'].items():
        monkeypatch.setenv(key, value)


_report = {}


@pytest.mark.parametrize('name', list(CASES))
def test_instance_case(engine, monkeypatch, name):
    _env(monkeypatch, name)
    inputs = build_inputs(name)
    B, records, inputs = compute(engine, name, inputs)
    check_record(name, records)
    assert np.isfinite(B.view(float)).all()
    B_hp, M = reference(inputs)
    if CASES[name]['kernel'] == 'ctrlmat_i8_kernel':
        # fixed point: the 1e-10 normalised tolerance of its quantisation error model (DESIGN 4.9)
        worst = max(nerr(B[j], B_hp[j].astype(complex)) for j in range(len(B)))
        assert worst < 1e-10, worst
        _report.setdefault(CASES[name]['kernel'], []).append((name, records[0]['S'], worst))
        return
    else:
        r = hp.ratio(B, B_hp, M)
        ratio = float(r.max())
        assert ratio <= KAPPA, f'{name}: |B - B_hp| / (EPS M) = {ratio:.2f} at {np.unravel_index(r.argmax(), r.shape)}'
    _report.setdefault(CASES[name]['kernel'], []).append((name, records[0]['S'], ratio))


def test_unreachable_instances_recorded(engine):
    """The probe shape of each unreachable instance goes elsewhere, with the occupancy the reason names."""
    from filter_functions_b200 import _lib
    for kernel, (probe, reason) in UNREACHABLE.items():
        _, records, _ = compute(engine, probe, build_inputs(probe))
        assert records[0]['kernel'] != kernel
        assert f"ctas_by_regs = {records[0]['ctas_by_regs']}" in reason or \
            f"{records[0]['ctas_by_regs']} CTA" in reason, (kernel, records[0])
    _lib.dispatch_log()


def test_non_fused_dfma_prologue(engine, tmp_path):
    """FFB_DFMA_FUSED_PROLOGUE=0 is read once per process: run one d = 3 DFMA case in a child process."""
    name = 'dfma12_d3_split'
    out = tmp_path / 'result.npz'
    code = (f'import sys; sys.path[:0] = {[ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]!r}\n'
            'import json, numpy as np, filter_functions_b200 as ff\n'
            'import test_gpu_ctrlmat_instances as t\n'
            f'B, records, _ = t.compute(ff, {name!r}, t.build_inputs({name!r}))\n'
            f'np.savez({str(out)!r}, B=B, records=json.dumps(records))\n')
    env = dict(os.environ, FFB_DFMA_FUSED_PROLOGUE='0')
    subprocess.run([sys.executable, '-c', code], check=True, env=env, cwd=ROOT)
    data = np.load(out)
    records = json.loads(str(data['records']))
    check_record(name, records)
    assert records[0]['prologue'] == 'transform_small_kernel<3>+assemble_dfma_kernel'
    B_hp, M = reference(build_inputs(name))
    assert hp.ratio(data['B'], B_hp, M).max() <= KAPPA


def test_zz_report():
    """One line per instance: its cases, their S, and the largest |B - B_hp| / (EPS M)."""
    for kernel in sorted(_report):
        rows = _report[kernel]
        measure = ('max normalised error' if kernel == 'ctrlmat_i8_kernel' else 'max |B - B_hp| / (EPS M)')
        print(f"{kernel}: {', '.join(f'{n} (S = {s})' for n, s, _ in rows)}; "
              f'{measure} = {max(r for _, _, r in rows):.3g}')
