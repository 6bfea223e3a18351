"""Every compiled instance of the front-end kernels (eigensolver and propagator scan), reached on purpose
and checked segment by segment against an extended-precision reference.

LEDGER maps each ``diag*`` / ``scan*`` kernel instance of libffb200.so to the cases that reach it.  A case
draws a seeded Hamiltonian, diagonalises it through ``numeric.diagonalize`` (H given) or
``numeric._diagonalize_from_coeffs`` (H formed on the device from control operators and coefficients), and
checks

- that the dispatch record (``_lib.diag_dispatch_log``) names the intended diagonaliser, the scan instances in
  order of first launch, the number of scan levels S and the segments per scan block or chunk;
- that eigenvalues, eigenvectors and propagators are finite, the eigenvalues ascending, and every bound of
  tests/hp_propagators.py holds with KAPPA on every segment (eigenvalues on a sample of segments).

The two environment flags that select the non-fused paths are read once per process: their cases run in a
child process.  Exact checks (diagonal H, scale equivariance, repeatability) compare bits.
"""
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import ff_oracle as oracle
import hp_propagators as hp
from helpers import rand_herm

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

#: float64 kernels pass when every error is within KAPPA * EPS * scale (hp_propagators); the float64 oracle
#: (numpy.linalg.eigh and its sequential product) passes the same bounds on every case (test_hp_propagators)
KAPPA = 16
BOUNDS = ('eigvals', 'residual', 'orthonormality', 'step', 'chain')
NO_FUSE, NO_SMALL = {'FFB_DIAG_FUSED': '0'}, {'FFB_DIAG_SMALL': '0'}


def case(d, G, H='rand', dt='rand', route='H', env=None):
    return dict(d=d, G=G, H=H, dt=dt, route=route, env=env or {})


#: name -> case.  H: 'rand' (random Hermitian), 'identity' (c_g 1: every pivot zero), 'kron' (A_g x 1_2),
#: 'cluster10' / 'cluster15' (two clusters of eigenvalues with gaps 1e-10 / 1e-15 of ||H||), 'real'
#: (real symmetric), 'imag' (real diagonal, imaginary off-diagonal), 'graded' (entries 1e-8 ... 1e8),
#: 'zeros' (every third segment H = 0), 'coeffs' (three control operators, formed on the device),
#: 'd4' / 'c2' (the workloads).  dt: 'rand', 'tiny' (0, 1e-12 and random, alternating), 'large'
#: (||H_g|| dt_g = 1e4), 'workload'.
CASES = {
    # ---- fused d = 2 (256 segments per block): block edges, 96 blocks, a second level, its tree product
    'fused_d2_G1': case(2, 1),
    'fused_d2_G255': case(2, 255),
    'fused_d2_G256': case(2, 256),
    'fused_d2_G257': case(2, 257),
    'fused_d2_G24576': case(2, 24576),
    'fused_d2_G24577': case(2, 24577),
    'fused_d2_G65537': case(2, 65537),
    # ---- fused d = 3, 4 (128 segments per block)
    'fused_d3_G10000': case(3, 10000),
    'fused_d3_G8192': case(3, 8192),
    'fused_d3_G12288': case(3, 12288),
    'fused_d3_G12289': case(3, 12289),
    'fused_d3_G16385': case(3, 16385),
    'fused_d4_G10000': case(4, 10000),
    'fused_d4_G8192': case(4, 8192),
    'fused_d4_G12288': case(4, 12288),
    'fused_d4_G12289': case(4, 12289),
    'fused_d4_G16385': case(4, 16385),
    # ---- generic path: chunk length L = 8 ... 256 (L^2 >= G), ragged last chunk
    'generic_d5_G1': case(5, 1),
    'generic_d5_G7': case(5, 7),
    'generic_d5_G64': case(5, 64),
    'generic_d5_G65': case(5, 65),
    'generic_d5_G4097': case(5, 4097),
    'generic_d5_G65537': case(5, 65537),
    'generic_d1': case(1, 37),
    'generic_d8': case(8, 37),
    'generic_d16': case(16, 23),
    'generic_d17': case(17, 9),
    'generic_d31': case(31, 5),
    'generic_d32': case(32, 6),
    # ---- spectra
    'identity_d4': case(4, 300, H='identity'),
    'identity_d8': case(8, 37, H='identity'),
    'kron_d4': case(4, 300, H='kron'),
    'kron_d6': case(6, 37, H='kron'),
    'cluster10_d4': case(4, 300, H='cluster10'),
    'cluster15_d4': case(4, 300, H='cluster15'),
    'cluster15_d8': case(8, 37, H='cluster15'),
    'real_d3': case(3, 300, H='real'),
    'real_d7': case(7, 37, H='real'),
    'imag_d2': case(2, 300, H='imag'),
    'imag_d6': case(6, 37, H='imag'),
    'graded_d4': case(4, 300, H='graded'),
    'graded_d6': case(6, 37, H='graded'),
    'zeros_tiny_d3': case(3, 300, H='zeros', dt='tiny'),
    'zeros_tiny_d5': case(5, 37, H='zeros', dt='tiny'),
    'large_d2': case(2, 300, dt='large'),
    'large_d4': case(4, 300, dt='large'),
    'large_d5': case(5, 37, dt='large'),
    # ---- control operators and coefficients, H formed on the device
    'coeffs_d2': case(2, 1000, H='coeffs', route='coeffs'),
    'coeffs_d4': case(4, 1000, H='coeffs', route='coeffs'),
    'coeffs_d6': case(6, 37, H='coeffs', route='coeffs'),
    'workload_d4': case(4, 10000, H='d4', dt='workload', route='coeffs'),
    'workload_c2': case(2, 10000, H='c2', dt='workload', route='coeffs'),
    # ---- the non-fused paths (flags read once per process: child processes)
    'nofuse_d2_G257': case(2, 257, env=NO_FUSE),
    'nofuse_d3_G12289': case(3, 12289, env=NO_FUSE),
    'nofuse_d4_G10000': case(4, 10000, env=NO_FUSE),
    'nofuse_coeffs_d4': case(4, 1000, H='coeffs', route='coeffs', env=NO_FUSE),
    'nosmall_d2_G257': case(2, 257, env=NO_SMALL),
    'nosmall_d3_G300': case(3, 300, H='real', env=NO_SMALL),
    'nosmall_d4_G10000': case(4, 10000, env=NO_SMALL),
    'nosmall_coeffs_d4': case(4, 1000, H='coeffs', route='coeffs', env=NO_SMALL),
}


def expected(d, G, env):
    """(kernel, prologue, S, passes_per_chunk) of the dispatch record: the dispatch of ffbi_diagonalize.
    d = 2, 3, 4 always scan in blocks; FFB_DIAG_SMALL=0 moves only their diagonalisation to diag_kernel."""
    if 2 <= d <= 4:
        NT = 256 if d == 2 else 128
        levels, n = 1, G
        while -(-n//NT) > 96:
            levels, n = levels + 1, -(-n//NT)
        names = ['scan_block_kernel', 'scan_apply_prefix_kernel'] + ['scan_apply_small_kernel']*(levels > 1)
        prologue = '+'.join(f'{k}<{d}, {NT}>' for k in names)
        if env.get('FFB_DIAG_SMALL') == '0':
            kernel = 'diag_kernel'
        elif env.get('FFB_DIAG_FUSED') == '0':
            kernel = f'diag_small_kernel<{d}>'
        else:
            kernel = f'scan_block_kernel<{d}, {NT}>'
        return kernel, prologue, levels, NT
    L = 8
    while L*L < G and L < 256:
        L *= 2
    return 'diag_kernel', 'scan_local_kernel+scan_totals_kernel+scan_apply_from_kernel', 1, L


def instances(name):
    kernel, prologue, _, _ = expected(CASES[name]['d'], CASES[name]['G'], CASES[name]['env'])
    return [kernel] + [k for k in prologue.split('+') if k != kernel]


LEDGER = {}
for _name in CASES:
    for _kernel in instances(_name):
        LEDGER.setdefault(_kernel, []).append(_name)


def _unitary(rng, G, d):
    Z = rng.standard_normal((G, d, d)) + 1j*rng.standard_normal((G, d, d))
    Q, R = np.linalg.qr(Z)
    return Q*(np.diagonal(R, axis1=1, axis2=2)/np.abs(np.diagonal(R, axis1=1, axis2=2)))[:, None, :]


def _hamiltonian(kind, d, G, rng):
    """(H, c_opers, c_coeffs); the operators are None unless H is formed from them."""
    if kind in ('d4', 'c2'):
        import workloads
        wl = workloads.get(kind)
        return np.einsum('ijk,il->ljk', wl.c_opers, wl.c_coeffs), wl.c_opers, wl.c_coeffs
    if kind == 'coeffs':
        c_opers, c_coeffs = rand_herm(rng, d, 3), rng.standard_normal((3, G))
        return np.einsum('ijk,il->ljk', c_opers, c_coeffs), c_opers, c_coeffs
    if kind == 'identity':
        H = rng.standard_normal(G)[:, None, None]*np.eye(d)
    elif kind == 'kron':
        H = np.kron(rand_herm(rng, d//2, G), np.eye(2))
    elif kind in ('cluster10', 'cluster15'):
        gap = 1e-10 if kind == 'cluster10' else 1e-15
        lam = np.where(np.arange(d) < d//2, -1.0, 1.0) + gap*np.arange(d)
        U = _unitary(rng, G, d)
        H = (U*lam) @ U.conj().transpose(0, 2, 1)
    elif kind == 'real':
        H = rand_herm(rng, d, G).real.astype(complex)
    elif kind == 'imag':
        A = rand_herm(rng, d, G)
        H = 1j*A.imag + np.diagonal(A.real, axis1=1, axis2=2)[:, :, None]*np.eye(d)
    elif kind == 'graded':
        s = np.logspace(-4, 4, d)
        H = s[:, None]*rand_herm(rng, d, G)*s[None, :]
    else:
        H = rand_herm(rng, d, G)
        if kind == 'zeros':
            H[::3] = 0
    return H, None, None


def _dt(kind, H, G, rng):
    if kind == 'workload':
        return None
    dt = 1 - rng.random(G)
    if kind == 'tiny':
        dt[0::3], dt[1::3] = 0.0, 1e-12
    elif kind == 'large':
        dt = 1e4/np.maximum(hp.spectral_norms(H), 1e-300)
    return dt


def build_inputs(name):
    """dict(H, dt, c_opers, c_coeffs) of a case.  Cases that differ only in their flags share the seed."""
    c = CASES[name]
    key = f"{c['H']}/{c['d']}/{c['G']}/{c['dt']}"
    rng = np.random.default_rng(zlib.crc32(key.encode()))
    H, c_opers, c_coeffs = _hamiltonian(c['H'], c['d'], c['G'], rng)
    dt = _dt(c['dt'], H, c['G'], rng)
    if dt is None:
        import workloads
        dt = workloads.get(c['H']).dt
    return dict(key=key, H=H, dt=dt, c_opers=c_opers, c_coeffs=c_coeffs)


_references = {}


def reference(inputs):
    """hp_propagators.Reference of a case's Hamiltonian, shared between the cases that use it."""
    if inputs['key'] not in _references:
        _references[inputs['key']] = hp.Reference(inputs['H'], inputs['dt'])
    return _references[inputs['key']]


def depth(name):
    c = CASES[name]
    return hp.scan_depth('small' if 2 <= c['d'] <= 4 else 'generic', c['d'], c['G'])


def compute(ff, name, inputs):
    """(ev, V, Q) of a case through its route, with the dispatch records of the call."""
    from filter_functions_b200 import _lib
    _lib.diag_dispatch_log()
    if CASES[name]['route'] == 'coeffs':
        out = ff.numeric._diagonalize_from_coeffs(inputs['c_opers'], inputs['c_coeffs'], inputs['dt'])
    else:
        out = ff.numeric.diagonalize(inputs['H'], inputs['dt'])
    return tuple(np.array(x) for x in out), _lib.diag_dispatch_log()


def check_record(name, records):
    c = CASES[name]
    assert len(records) == 1, (name, records)
    rec = records[0]
    kernel, prologue, S, per_chunk = expected(c['d'], c['G'], c['env'])
    assert rec['kernel'] == kernel, f"{name}: diagonalised by {rec['kernel']}, the ledger expects {kernel}"
    assert rec['prologue'] == prologue, f"{name}: scan {rec['prologue']}, the ledger expects {prologue}"
    assert (rec['S'], rec['passes_per_chunk'], rec['n_pass']) == (S, per_chunk, c['G']), (name, rec)


_report = {}


def check_case(name, inputs, result, records):
    """Record, finiteness, order and every bound; returns the worst ratio per bound."""
    check_record(name, records)
    ev, V, Q = result
    c = CASES[name]
    assert ev.shape == (c['G'], c['d']) and V.shape == (c['G'], c['d'], c['d'])
    assert Q.shape == (c['G'] + 1, c['d'], c['d'])
    for x in result:
        assert np.isfinite(x.view(float)).all(), name
    assert (np.diff(ev, axis=1) >= 0).all(), name
    ratios = reference(inputs).ratios(ev, V, Q, depth(name))
    for kernel in instances(name):
        _report.setdefault(kernel, []).append((name, ratios))
    bad = {k: v for k, v in ratios.items() if not v <= KAPPA}
    assert not bad, f'{name}: error / (EPS scale) above {KAPPA}: {bad}'
    return ratios


@pytest.mark.parametrize('name', [n for n in CASES if not CASES[n]['env']])
def test_instance_case(engine, name):
    inputs = build_inputs(name)
    result, records = compute(engine, name, inputs)
    check_case(name, inputs, result, records)


@pytest.mark.parametrize('flag', ['FFB_DIAG_FUSED', 'FFB_DIAG_SMALL'])
def test_flag_cases(engine, tmp_path, flag):
    """The flags are read once per process: the cases of one flag run in a child process."""
    names = [n for n in CASES if flag in CASES[n]['env']]
    out = tmp_path/'result.npz'
    code = (f'import sys; sys.path[:0] = {[ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]!r}\n'
            'import json, numpy as np, filter_functions_b200 as ff\n'
            'import test_gpu_diag_instances as t\n'
            'arrays, records = {}, {}\n'
            f'for name in {names!r}:\n'
            '    (ev, V, Q), rec = t.compute(ff, name, t.build_inputs(name))\n'
            '    arrays.update({name + "/ev": ev, name + "/V": V, name + "/Q": Q})\n'
            '    records[name] = rec\n'
            f'np.savez({str(out)!r}, records=json.dumps(records), **arrays)\n')
    subprocess.run([sys.executable, '-c', code], check=True, env=dict(os.environ, **{flag: '0'}), cwd=ROOT)
    data = np.load(out)
    records = json.loads(str(data['records']))
    failed = []
    for name in names:
        try:
            check_case(name, build_inputs(name), tuple(data[f'{name}/{k}'] for k in ('ev', 'V', 'Q')),
                       records[name])
        except AssertionError as err:
            failed.append(str(err))
    assert not failed, failed


@pytest.mark.parametrize('name', ['workload_d4', 'workload_c2'])
def test_drift(engine, name):
    """Unitarity defect of Q_g at G/4, G/2, G: at most twice the float64 oracle's, or KAPPA EPS d sqrt(g).
    The renormalised eigenvector columns keep it there (DESIGN 4.3)."""
    inputs = build_inputs(name)
    (ev, V, Q), _ = compute(engine, name, inputs)
    _, _, Q_o = oracle.diagonalize(inputs['H'], inputs['dt'])
    G, d = CASES[name]['G'], CASES[name]['d']
    gs = [G//4, G//2, G]
    defect, bound = hp.unitarity_defect(Q, gs), hp.drift_bound(hp.unitarity_defect(Q_o, gs), d, gs, KAPPA)
    print(f'{name}: unitarity defect at g = {gs}: {defect}, oracle {hp.unitarity_defect(Q_o, gs)}')
    assert (defect <= bound).all(), (defect, bound)


@pytest.mark.parametrize('d,G', [(1, 5), (2, 300), (4, 300), (5, 37), (9, 7)])
def test_diagonal_exact(engine, d, G):
    """Diagonal H with repeated entries: eigenvalues are the stably sorted diagonal bit for bit, V the
    matching permutation, and Q_1 = diag(e^{-i h dt}) within the sincos rounding."""
    rng = np.random.default_rng(d*G)
    h = rng.choice([-1.5, 0.25, 0.25, 2.0, -1.5, 3.0], size=(G, d))
    H = h[:, :, None]*np.eye(d)
    dt = 1 - rng.random(G)
    ev, V, Q = engine.numeric.diagonalize(H, dt)
    order = np.argsort(h, axis=1, kind='stable')
    assert np.array_equal(ev, np.take_along_axis(h, order, axis=1))
    perm = np.zeros((G, d, d), dtype=complex)
    perm[np.arange(G)[:, None], order, np.arange(d)[None, :]] = 1
    assert np.array_equal(V, perm)
    phase = np.exp(-1j*h[0]*dt[0])
    assert np.abs(Q[1] - np.diag(phase)).max() <= 4*hp.EPS
    assert np.array_equal(Q[1] - np.diag(np.diag(Q[1])), np.zeros((d, d)))


@pytest.mark.parametrize('k', [-1000, -600, -540, -520, -300, 300, 500, 520, 600, 1000])
@pytest.mark.parametrize('d', [2, 4, 6])
def test_scale_equivariance(engine, d, k):
    """eigvals(2^k H) = 2^k eigvals(H) and identical eigenvectors, bit for bit; with dt scaled by 2^-k the
    propagators are identical too.  Every scaled entry stays a normal double."""
    rng = np.random.default_rng(40 + d)
    G = 37
    H = rand_herm(rng, d, G)
    dt = 1 - rng.random(G)
    ev, V, Q = engine.numeric.diagonalize(H, dt)
    Hk = np.ldexp(H.real, k) + 1j*np.ldexp(H.imag, k)
    dt_k = np.ldexp(dt, -k)
    for x in (Hk.real, Hk.imag, dt_k):
        assert (np.abs(x[x != 0]) >= np.finfo(float).tiny).all() and np.isfinite(x).all()
    ev_k, V_k, Q_k = engine.numeric.diagonalize(Hk, dt_k)
    assert np.array_equal(ev_k, np.ldexp(ev, k))
    assert np.array_equal(V_k, V)
    assert np.array_equal(Q_k, Q)


@pytest.mark.parametrize('name', ['fused_d4_G12289', 'generic_d5_G4097', 'coeffs_d4'])
def test_repeatable(engine, name):
    inputs = build_inputs(name)
    first, _ = compute(engine, name, inputs)
    second, _ = compute(engine, name, inputs)
    for a, b in zip(first, second):
        assert np.array_equal(a, b)


def test_zz_report():
    """One line per instance: its cases and the largest error / (EPS scale) of each bound."""
    for kernel in sorted(_report):
        rows = _report[kernel]
        worst = {b: max(r[b] for _, r in rows) for b in BOUNDS}
        print(f"{kernel}: {', '.join(n for n, _ in rows)}; "
              + ', '.join(f'{b} {v:.3g}' for b, v in worst.items()))
