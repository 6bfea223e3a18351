"""Shared generators and comparison helpers for the parity tests (mirrors tests/testutil.py of the
reference: rand_herm, rand_herm_traceless, rand_pulse_sequence, generate_dd_hamiltonian)."""
import gzip
import os
import pickle
import string
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RAISED = '__ValueError__'


class ReferenceResults:
    """What the unmodified reference (qutech/filter_functions) returns for the seeded inputs of a
    differential test.  ``self(key, fn)`` is ``fn(reference)`` where the reference is staged under
    ``baseline/_ref``, else the value stored under ``key`` in ``tests/golden/<name>.pkl.gz``.  A ValueError
    comes back as ``(RAISED, message)``; ``fn`` returns plain data (arrays, lists, dicts, strings).

    ``FFB_RECORD_REFERENCE=1`` evaluates every ``fn`` and rewrites the file on ``save()``: with the
    reference itself where it is staged, else with this package, whose results on these inputs the same
    comparisons had found equal to the reference's (the file's 'source' entry says which)."""

    def __init__(self, name):
        self.path = os.path.join(ROOT, 'tests', 'golden', f'{name}.pkl.gz')
        self.record = os.environ.get('FFB_RECORD_REFERENCE', '0') not in ('', '0')
        self.module, self.stored = None, {}
        if os.path.isdir(os.path.join(ROOT, 'baseline', '_ref', 'filter_functions')):
            for p in (os.path.join(ROOT, 'oracle', 'shim'), os.path.join(ROOT, 'baseline', '_ref')):
                if p not in sys.path:
                    sys.path.insert(0, p)
            import filter_functions
            self.module, self.source = filter_functions, 'reference'
        elif self.record:
            import filter_functions_b200
            self.module, self.source = filter_functions_b200, 'filter_functions_b200'
        else:
            with gzip.open(self.path, 'rb') as fh:
                self.stored = pickle.load(fh)

    def __call__(self, key, fn):
        if self.module is None:
            return self.stored[key]
        try:
            value = fn(self.module)
        except ValueError as err:
            value = (RAISED, str(err))
        if self.record:
            self.stored[key] = value
        return value

    def save(self):
        if self.record:
            with gzip.open(self.path, 'wb') as fh:
                pickle.dump({**self.stored, 'source': self.source}, fh, protocol=4)


def nerr(x, ref):
    """max|x - ref| / max|ref| -- the normalised error SURVEY.md 8c prescribes."""
    ref = np.asarray(ref)
    scale = np.abs(ref).max()
    return float(np.abs(np.asarray(x) - ref).max()/(scale if scale > 0 else 1.0))


def rand_herm(rng, d, n=1):
    A = rng.standard_normal((n, d, d)) + 1j*rng.standard_normal((n, d, d))
    return (A + A.conj().transpose(0, 2, 1))/2


def rand_herm_traceless(rng, d, n=1):
    A = rand_herm(rng, d, n).transpose()
    A -= A.trace(axis1=0, axis2=1)/d
    return A.transpose()


def rand_pulse_arrays(rng, d, n_dt, n_cops=3, n_nops=3, commensurable=False):
    """Same draw order as reference tests/testutil.py:131-190 (so seeded tests reproduce)."""
    c_opers = rand_herm_traceless(rng, d, n_cops)
    n_opers = rand_herm_traceless(rng, d, n_nops)
    c_coeffs = rng.standard_normal((n_cops, n_dt))
    n_coeffs = rng.random((n_nops, n_dt))
    letters = np.array(list(string.ascii_letters))
    c_ids = rng.choice(letters, n_cops, replace=False)
    n_ids = rng.choice(letters, n_nops, replace=False)
    if commensurable:
        dt = np.full(n_dt, 1 - rng.random())
    else:
        dt = 1 - rng.random(n_dt)
    return c_opers, c_coeffs, c_ids, n_opers, n_coeffs, n_ids, dt


def rand_pulse_sequence(ff, rng, d, n_dt, n_cops=3, n_nops=3, btype='GGM', commensurable=False):
    c_opers, c_coeffs, c_ids, n_opers, n_coeffs, n_ids, dt = rand_pulse_arrays(
        rng, d, n_dt, n_cops, n_nops, commensurable)
    basis = ff.Basis.ggm(d) if btype == 'GGM' else ff.Basis.pauli(int(np.log2(d)))
    return ff.PulseSequence(list(zip(c_opers, c_coeffs, c_ids)), list(zip(n_opers, n_coeffs, n_ids)),
                            dt, basis)


def dd_hamiltonian(n, tau=10, tau_pi=1e-2, dd_type='cpmg'):
    """Primitive-pulse dynamical decoupling sequence (reference tests/testutil.py:82-128)."""
    X = np.array([[0, 1], [1, 0]], dtype=complex)

    def cdd_odd(g, t):
        return np.array([*cdd_even(g - 1, t/2), t/2, *(cdd_even(g - 1, t/2) + t/2)])

    def cdd_even(g, t):
        if g == 0:
            return np.array([])
        return np.array([*cdd_odd(g - 1, t/2), *(cdd_odd(g - 1, t/2) + t/2)])

    if dd_type == 'cpmg':
        delta = np.array([0] + [(g - 0.5)/n for g in range(1, n + 1)])
    elif dd_type == 'udd':
        delta = np.array([0] + [np.sin(np.pi*g/(2*n + 2))**2 for g in range(1, n + 1)])
    elif dd_type == 'pdd':
        delta = np.array([0] + [g/(n + 1) for g in range(1, n + 1)])
    else:
        delta = np.insert(cdd_odd(n, 1) if n % 2 else cdd_even(n, 1), 0, 0)
    s_p = np.pi/tau_pi*np.array([0, 1])
    t_p = tau_pi*np.array([0, 1])
    s, t = np.array([]), np.array([0])
    for i in range(len(delta) - 1):
        s = np.append(s, s_p)
        t = np.append(t, t_p + (delta*tau)[i + 1] - tau_pi/2)
    t = np.append(t, tau)
    s = np.append(s, 0)
    return [[X/2, s]], np.diff(t)
