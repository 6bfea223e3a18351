"""Concatenation of gates that carry different noise operators through ``ffb_concatenate_pulses``: the rows a
gate lacks are computed from scratch into the atomic stack, the cached rows are copied in, and the stack is
contracted.  Covered here: both stack modes (all P pulse slots, and the two-slot running sum used when the
stack would not fit), and a gate whose missing rows are not one contiguous run, which is filled through a
scratch buffer and scattered into its slot."""
import numpy as np
import pytest

import ff_oracle as oracle
from helpers import nerr

pytestmark = pytest.mark.gpu


def oracle_B(pulse, omega):
    H = oracle.hamiltonian_from_coeffs(pulse.c_opers, pulse.c_coeffs)
    ev, V, Q = oracle.diagonalize(H, pulse.dt)
    return oracle.control_matrix_from_scratch(ev, V, Q, omega, np.asarray(pulse.basis), pulse.n_opers,
                                              pulse.n_coeffs, pulse.dt)


@pytest.mark.parametrize('stack', ['1', '0'], ids=['full_stack', 'two_slots'])
def test_concatenation_fills_missing_rows(engine, monkeypatch, stack):
    ff = engine
    from filter_functions_b200 import pulse_sequence
    monkeypatch.setenv('FFB_CONCAT_STACK', stack)          # read by every ffb_concatenate_pulses call
    monkeypatch.setenv('FFB_CONCAT_ROUTE', 'atomic')       # the route under test, whatever the cost model says
    calls = []
    on_device = pulse_sequence._concatenate_on_device
    monkeypatch.setattr(pulse_sequence, '_concatenate_on_device',
                        lambda *args, **kwargs: calls.append(1) or on_device(*args, **kwargs))
    rng = np.random.default_rng(23)
    d = 4
    omega = np.geomspace(1e-2, 30, 700)
    basis = ff.Basis.pauli(2)

    def herm(n):
        A = rng.standard_normal((n, d, d)) + 1j*rng.standard_normal((n, d, d))
        return (A + A.conj().transpose(0, 2, 1))/2

    ops, noise = herm(2), herm(4)
    level = [0.7, None, 1.3, 0.9]      # an operator some gate lacks needs one constant sensitivity

    def gate(carried):
        G = int(rng.integers(2, 6))
        H_c = [[ops[k], rng.standard_normal(G), f'c{k}'] for k in range(2)]
        H_n = [[noise[k], 0.5 + rng.random(G) if level[k] is None else np.full(G, level[k]), f'n{k}']
               for k in carried]
        pulse = ff.PulseSequence(H_c, H_n, 1 - rng.random(G)*0.5, basis)
        pulse.cache_control_matrix(omega)
        return pulse

    # merged noise operators n0..n3: the first gate lacks rows 0, 2 and 3 (two runs), the second rows 2
    # and 3 (one run, written in place), the third lacks none; the first gate recurs at the end
    a, b, c = gate([1]), gate([0, 1]), gate([0, 1, 2, 3])
    gates = [a, b, c, a]
    total = ff.concatenate(gates, omega=omega)
    assert calls == [1]
    whole = ff.concatenate(gates, calc_filter_function=False)
    B_o = oracle_B(whole, omega)
    assert nerr(total.get_control_matrix(omega), B_o) < 1e-9
    assert nerr(total.get_filter_function(omega), oracle.filter_function(B_o)) < 1e-9
