"""Differential test (CPU) of the host helpers that were added for drop-in completeness against the
UNMODIFIED reference: ``util.tensor``, ``util.remove_float_errors``, ``Basis.from_partial`` / ``pauli`` /
``ggm`` / expansions and predicates, ``superoperator.liouville_to_choi`` / ``liouville_is_CP`` /
``liouville_is_cCP``, ``util.get_sample_frequencies``, ``util.parse_operators`` / ``parse_spectrum`` error
behaviour.  The reference runs where it is staged under ``baseline/_ref``; elsewhere its results on these
seeded inputs come from ``tests/golden/reference_host_helpers.pkl.gz`` (``helpers.ReferenceResults``).  None
of these needs the GPU."""
import warnings

import numpy as np
import pytest

import filter_functions_b200 as ffb
from filter_functions_b200 import superoperator as so_new
from helpers import RAISED, ReferenceResults


@pytest.fixture(scope='module')
def ref():
    results = ReferenceResults('reference_host_helpers')
    yield results
    results.save()


def herm(rng, d, n=1):
    a = rng.standard_normal((n, d, d)) + 1j*rng.standard_normal((n, d, d))
    return a + a.conj().swapaxes(1, 2)


def basis_data(b):
    return {'array': b.view(np.ndarray).copy(), 'labels': list(b.labels), 'btype': b.btype,
            **{pred: bool(getattr(b, pred)) for pred in
               ('isherm', 'isnorm', 'isorthogonal', 'isorthonorm', 'istraceless', 'iscomplete')}}


def test_tensor_and_cleanup(ref):
    rng = np.random.default_rng(0)
    for case in range(60):
        rank = int(rng.integers(1, 4))
        n_args = int(rng.integers(1, 4))
        lead = tuple(rng.integers(1, 4, size=rng.integers(0, 3)))
        args = []
        for _ in range(n_args):
            shape = tuple(rng.integers(1, 4, size=rank))
            my_lead = tuple(1 if rng.random() < 0.3 else n for n in lead)[rng.integers(0, len(lead) + 1):]
            args.append(rng.standard_normal(my_lead + shape) + 1j*rng.standard_normal(my_lead + shape))
        want = ref(f'tensor/{case}', lambda m: m.util.tensor(*args, rank=rank))
        if isinstance(want, tuple) and want[0] == RAISED:
            with pytest.raises(ValueError) as got:
                ffb.util.tensor(*args, rank=rank)
            assert str(got.value) == want[1]
            continue
        got = ffb.util.tensor(*args, rank=rank)
        assert got.shape == want.shape and np.allclose(got, want, rtol=1e-14, atol=0)
    for dtype in (float, complex):
        x = (np.eye(4) + 1e-17*rng.standard_normal((4, 4))).astype(dtype)
        for args in ((), (100,)):
            want = ref(f'remove_float_errors/{dtype.__name__}/{args}',
                       lambda m: m.util.remove_float_errors(x.copy(), *args))
            assert np.array_equal(ffb.util.remove_float_errors(x.copy(), *args), want)


def test_basis_constructors_predicates_and_expansion(ref):
    rng = np.random.default_rng(1)
    for n in (1, 2):
        want = ref(f'pauli/{n}', lambda m: basis_data(m.Basis.pauli(n)))
        assert np.array_equal(ffb.Basis.pauli(n), want['array'])
        assert list(ffb.Basis.pauli(n).labels) == want['labels']
    for d in (2, 3, 4, 5):
        a, b = ffb.Basis.ggm(d), ref(f'ggm/{d}', lambda m: basis_data(m.Basis.ggm(d)))
        assert np.allclose(a.view(np.ndarray), b['array'], atol=1e-16)
        assert list(a.labels) == b['labels'] and a.btype == b['btype']
        M = herm(rng, d, 3)
        for kw in (dict(), dict(hermitian=True), dict(traceless=True), dict(tidyup=True)):
            want = ref(f'ggm/{d}/expand/{sorted(kw)}', lambda m: m.Basis.ggm(d).expand(M, **kw))
            assert np.allclose(a.expand(M, **kw), want, atol=1e-14)
        # partial bases: random orthogonal subsets in a rotated frame, with and without the identity
        g = b['array']
        for trial in range(6):
            n = int(rng.integers(1, d*d))
            q, _ = np.linalg.qr(rng.standard_normal((d*d, d*d)))
            part = (np.einsum('ij,jkl->ikl', q[:n], g) if trial % 2
                    else g[rng.choice(d*d, size=n, replace=False)]*rng.uniform(0.5, 3))
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                want = ref(f'from_partial/{d}/{trial}', lambda m: basis_data(m.Basis.from_partial(part)))
                got = ffb.Basis.from_partial(part)
            assert got.shape == want['array'].shape and got.btype == want['btype']
            assert list(got.labels) == want['labels']
            for pred in ('isherm', 'isnorm', 'isorthogonal', 'isorthonorm', 'istraceless', 'iscomplete'):
                assert bool(getattr(got, pred)) == want[pred], pred
            # both are complete orthonormal bases (the map between them is unitary) and the given elements
            # (plus the identity of a traceless basis) sit at the same positions in both
            gw, gg = want['array'].reshape(d*d, -1), got.view(np.ndarray).reshape(d*d, -1)
            overlap = gw.conj() @ gg.T
            assert np.allclose(np.abs(np.linalg.det(overlap)), 1, atol=1e-9)
            same = [i for i in range(d*d) if np.isclose(abs(overlap[i, i]), 1, atol=1e-9)]
            assert len(same) >= n
    X, Y = ffb.util.paulis[1:3]
    for case, (args, kw) in enumerate((([X, X + Y], {}), ([np.diag([1.0, 0])], dict(traceless=True)),
                                       ([X, Y], dict(labels=['a'])))):
        want = ref(f'from_partial/error/{case}', lambda m: basis_data(m.Basis.from_partial(args, **kw)))
        assert isinstance(want, tuple) and want[0] == RAISED
        with pytest.raises(ValueError) as e_new:
            ffb.Basis.from_partial(args, **kw)
        assert str(e_new.value) == want[1]


def test_choi_and_cp_checks(ref):
    rng = np.random.default_rng(2)
    for d in (2, 3, 4):
        b_new = ffb.Basis.ggm(d)
        S = rng.standard_normal((4, d*d, d*d)) + 1j*rng.standard_normal((4, d*d, d*d))
        want = ref(f'choi/{d}', lambda m: m.superoperator.liouville_to_choi(S, m.Basis.ggm(d)))
        assert np.allclose(so_new.liouville_to_choi(S, b_new), want)
        H = herm(rng, d)[0]
        w, v = np.linalg.eigh(H)
        U = (v*np.exp(-1j*w)) @ v.conj().T
        L = ref(f'liouville/{d}', lambda m: m.superoperator.liouville_representation(U, m.Basis.ggm(d)))
        for fn in ('liouville_is_CP', 'liouville_is_cCP'):
            for i, arg in enumerate((L, -L, S, np.stack([L, -np.eye(d*d)]))):
                def call(m):
                    res = getattr(m.superoperator, fn)(arg, m.Basis.ggm(d), return_eig=True)
                    return np.asarray(res[0]), np.asarray(res[1][0])
                want = ref(f'{fn}/{d}/{i}', call)
                got = getattr(so_new, fn)(arg, b_new, return_eig=True)
                assert np.array_equal(np.asarray(got[0]), want[0]), fn
                assert np.allclose(got[1][0], want[1], atol=1e-10)


def test_sample_frequencies_and_parsers(ref):
    rng = np.random.default_rng(3)
    X, Y, Z = ffb.util.paulis[1:]
    for G in (1, 5, 40):
        dt = rng.uniform(0.1, 2, G)
        coeffs = rng.standard_normal(G)
        b = ffb.PulseSequence([[X/2, coeffs, 'X']], [[Z/2, np.ones(G), 'Z']], dt)
        for i, kw in enumerate((dict(), dict(n_samples=57, spacing='linear'), dict(include_quasistatic=True),
                                dict(omega_min=1e-3, omega_max=7.0))):
            want = ref(f'sample_frequencies/{G}/{i}', lambda m: m.util.get_sample_frequencies(
                m.PulseSequence([[X/2, coeffs, 'X']], [[Z/2, np.ones(G), 'Z']], dt), **kw))
            assert np.array_equal(ffb.util.get_sample_frequencies(b, **kw), want)
        with pytest.raises(ValueError):
            ffb.util.get_sample_frequencies(b, spacing='foo')
    omega = np.linspace(0, 1, 11)
    for i, (S, idx) in enumerate(((np.ones((2, 11)), [0, 1]), (np.ones(11), [0]),
                                  (np.ones((2, 2, 11)) + 0j, [0, 1]))):
        want = ref(f'parse_spectrum/{i}', lambda m: m.util.parse_spectrum(S, omega, np.array(idx)))
        assert np.array_equal(ffb.util.parse_spectrum(S, omega, np.array(idx)), want)
    bad = [(np.ones((3, 11)), [0, 1]), (np.ones((2, 2, 2, 11)), [0, 1]), (np.ones(10), [0]),
           (np.arange(44).reshape(2, 2, 11)*(1 + 1j), [0, 1])]
    for i, (S, idx) in enumerate(bad):
        want = ref(f'parse_spectrum/error/{i}', lambda m: m.util.parse_spectrum(S, omega, np.array(idx)))
        assert isinstance(want, tuple) and want[0] == RAISED
        with pytest.raises(ValueError) as e_new:
            ffb.util.parse_spectrum(S, omega, np.array(idx))
        assert str(e_new.value) == want[1]
