"""Differential test of the Hamiltonian join (``concatenate_without_filter_function``, reference
``pulse_sequence.py:1340-1483, :1599-1665``) against the UNMODIFIED reference staged under
``baseline/_ref`` where it is staged, elsewhere against its results on these seeded inputs stored in
``tests/golden/reference_join.pkl.gz`` (``helpers.ReferenceResults``): random pulse libraries with shared /
partially shared operators, identifier clashes, equal operators under different identifiers and
non-constant noise sensitivities; results, identifier mappings and exception types + messages must agree.
Every library is joined in several random orders, so that the remembered join plans are exercised."""
import numpy as np
import pytest

from helpers import ReferenceResults


@pytest.fixture(scope='module')
def ref():
    results = ReferenceResults('reference_join')
    yield results
    results.save()


X = np.array([[0, 1], [1, 0]], dtype=complex)
Y = np.array([[0, -1j], [1j, 0]])
Z = np.array([[1, 0], [0, -1]], dtype=complex)
OPS = {'X': X/2, 'Y': Y/2, 'Z': Z/2, 'P': (X + Z)/3}


def random_library(rng, n_lib, nasty):
    """Recipes [(c_items, n_items, dt)] -- built by both packages from the same arrays."""
    recipes = []
    for _ in range(n_lib):
        G = int(rng.integers(1, 5))
        names = list(OPS)
        c_names = list(rng.choice(names, rng.integers(1, 3), replace=False))
        n_names = list(rng.choice(names, rng.integers(1, 3), replace=False))
        c_items = [[OPS[k], rng.standard_normal(G), k] for k in c_names]
        n_items = []
        for k in n_names:
            coeff = np.full(G, 1.5) if (not nasty or rng.random() < 0.8) else rng.random(G)
            n_items.append([OPS[k], coeff, 'n' + k])
        if nasty and rng.random() < 0.25:       # identifier names another operator here
            c_items[0][2] = str(rng.choice(names))
        if nasty and rng.random() < 0.15:       # same operator, another identifier
            n_items[0][2] = 'other'
        if len(set(i[2] for i in c_items)) < len(c_items) or len(set(i[2] for i in n_items)) < len(n_items):
            continue
        recipes.append((c_items, n_items, 1 - rng.random(G)*0.5))
    return recipes


def outcome(join, pulses):
    try:
        new, cmap, nmap = join(pulses, return_identifier_mappings=True)
    except Exception as err:        # noqa: BLE001 -- the type and text are what is compared
        return type(err).__name__, str(err)
    return (new.c_opers, list(new.c_oper_identifiers), new.c_coeffs, new.n_opers,
            list(new.n_oper_identifiers), new.n_coeffs, new.dt, new.tau,
            {int(k): dict(v) for k, v in cmap.items()}, {int(k): dict(v) for k, v in nmap.items()})


def joined(package, recipes, idx):
    pulses = [package.PulseSequence(c, n, dt) for c, n, dt in recipes]
    return outcome(package.pulse_sequence.concatenate_without_filter_function, [pulses[i] for i in idx])


@pytest.mark.parametrize('nasty', [False, True])
def test_join_matches_reference(ref, nasty):
    import filter_functions_b200 as ff
    rng = np.random.default_rng(2026 + nasty)
    n_ok = n_err = 0
    for lib in range(60):
        recipes = random_library(rng, int(rng.integers(2, 7)), nasty)
        if len(recipes) < 2:
            continue
        mine = [ff.PulseSequence(c, n, dt) for c, n, dt in recipes]
        for seq in range(4):    # same library, several sequences (plan reuse, other first occurrences)
            idx = rng.integers(0, len(recipes), int(rng.integers(2, 25)))
            got = outcome(ff.pulse_sequence.concatenate_without_filter_function, [mine[i] for i in idx])
            want = ref(f'{nasty}/{lib}/{seq}', lambda m: joined(m, recipes, idx))
            assert len(got) == len(want)
            if len(got) == 2:
                assert got == want
                n_err += 1
                continue
            n_ok += 1
            for g, w in zip(got, want):
                if isinstance(w, np.ndarray):
                    np.testing.assert_array_equal(g, w)
                elif isinstance(w, float):
                    assert g == pytest.approx(w, rel=1e-15)
                else:
                    assert g == w
    assert n_ok > 50 and (n_err > 5 if nasty else n_err == 0)
