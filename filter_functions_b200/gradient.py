"""Gradient of the first-order infidelity with respect to the control amplitudes.

:func:`infidelity_derivative` is what pulse optimisation (e.g. GRAPE with qopt) needs: the exact
derivative of :func:`filter_functions_b200.infidelity` with respect to every control amplitude of every
segment, computed on the GPU in one adjoint sweep over the segments (DESIGN.md section 4.11).
"""
import numpy as np
from numpy import ndarray

from . import _lib, util

__all__ = ['infidelity_derivative']

#: largest Hilbert-space dimension the gradient kernels are built for
MAX_DIM = 8


def infidelity_derivative(pulse, spectrum, omega, control_identifiers=None,
                          n_oper_identifiers=None, n_coeffs_deps=None) -> ndarray:
    r"""Derivative of the first-order infidelity with respect to the control amplitudes,
    :math:`\partial\mathcal{I}_\alpha/\partial u_h(t_g)`, of shape (n_nops, G, n_ctrl).

    The infidelity is that of :func:`~filter_functions_b200.numeric.infidelity`,
    :math:`\mathcal{I}_\alpha = \frac{1}{2\pi d}\int S_\alpha(\omega) F_{\alpha\alpha}(\omega)\,d\omega`
    with the same trapezoid rule on ``omega``, for uncorrelated noise.

    Parameters
    ----------
    pulse: PulseSequence
        The pulse; its Hamiltonian is :math:`H_g = \sum_h u_h(g) A_h` with the amplitudes
        ``pulse.c_coeffs``.  Its basis must be traceless (up to one identity element).  A cached
        diagonalisation and a control matrix cached for the same ``omega`` are used; nothing new is
        cached.
    spectrum: array_like, shape (n_omega,) or (n_nops, n_omega)
        One noise spectrum for all, or one per selected noise operator.  Cross spectra are not
        supported.
    omega: array_like, shape (n_omega,)
        The frequencies of the integral.
    control_identifiers: sequence of str, optional
        The controls to differentiate by, in this order (default: ``pulse.c_oper_identifiers``).
    n_oper_identifiers: sequence of str, optional
        The noise operators, in this order (default: all of ``pulse.n_oper_identifiers``).
    n_coeffs_deps: array_like, shape (len(pulse.n_oper_identifiers), n_ctrl, G), optional
        :math:`\partial s_\alpha(g)/\partial u_h(g)` for noise sensitivities that depend on the
        controls, axes in the order of ``pulse.n_oper_identifiers`` and of the chosen controls.

    Returns
    -------
    ndarray, shape (n_nops, G, n_ctrl)
        The derivative for each selected noise operator, segment and control.
    """
    c_idx = util.get_indices_from_identifiers(pulse.c_oper_identifiers, control_identifiers)
    n_idx = util.get_indices_from_identifiers(pulse.n_oper_identifiers, n_oper_identifiers)
    d = pulse.c_opers.shape[-1]
    if d > MAX_DIM:
        raise ValueError(f'infidelity_derivative supports Hilbert-space dimensions d <= {MAX_DIM}, '
                         f'not d = {d} (README: limits)')
    if not pulse.basis.istraceless:
        raise ValueError('infidelity_derivative needs a traceless basis (up to an identity element)')
    omega = _lib.as_f64(np.asarray(omega))
    if omega.ndim != 1 or not len(omega):
        raise ValueError(f'Expected omega of shape (n_omega,), not {omega.shape}')
    G, n_omega, n_sel, n_ctrl = len(pulse.dt), len(omega), len(n_idx), len(c_idx)
    n_nops = len(pulse.n_opers)
    spectrum = np.asarray(spectrum)
    if spectrum.shape not in ((n_omega,), (n_sel, n_omega)):
        raise ValueError(f'Spectrum should be of shape ({n_omega},) or ({n_sel}, {n_omega}), not '
                         f'{spectrum.shape} (infidelity_derivative supports uncorrelated noise only)')
    spectrum = _lib.as_f64(spectrum.real)
    if n_coeffs_deps is not None:
        n_coeffs_deps = _lib.as_f64(n_coeffs_deps)
        if n_coeffs_deps.shape != (n_nops, n_ctrl, G):
            raise ValueError(f'Expected n_coeffs_deps of shape {(n_nops, n_ctrl, G)}, not '
                             f'{n_coeffs_deps.shape}')

    # cached arrays are used as they are (their device mirrors, if any, are not uploaded again);
    # nothing is added to the pulse's caches
    data, freq = pulse._data, pulse._frequency_data
    have_diag = all(key in data for key in ('eigvals', 'eigvecs', 'propagators'))
    eigvals = _lib.as_f64(data['eigvals']) if have_diag else None
    eigvecs = _lib.as_c128(data['eigvecs']) if have_diag else None
    propagators = _lib.as_c128(data['propagators']) if have_diag else None
    B = None
    if have_diag and 'control_matrix' in freq and np.array_equal(pulse.omega, omega):
        B = _lib.as_c128(freq['control_matrix'])
    dt = _lib.as_f64(pulse.dt)
    t = _lib.as_f64(data['t'] if 't' in data else np.concatenate(([0.0], dt.cumsum())))
    c_opers, c_coeffs = _lib.as_c128(pulse.c_opers), _lib.as_f64(pulse.c_coeffs)
    n_opers, n_coeffs = _lib.as_c128(pulse.n_opers), _lib.as_f64(pulse.n_coeffs)
    basis = _lib.as_c128(np.asarray(pulse.basis))
    c_idx32 = np.ascontiguousarray(c_idx, dtype=np.int32)
    n_idx32 = np.ascontiguousarray(n_idx, dtype=np.int32)
    out = np.empty((n_sel, G, n_ctrl), dtype=np.float64)
    p = _lib.ptr
    ctx = _lib.context()
    _lib.check(ctx, _lib.lib().ffb_infidelity_derivative(
        ctx, G, d, len(c_opers), n_nops, len(basis), n_omega, p(c_opers),
        None if have_diag else p(c_coeffs), p(eigvals), p(eigvecs), p(propagators), p(omega),
        p(basis), p(n_opers), p(n_coeffs), p(dt), p(t), p(B), n_ctrl, p(c_idx32), n_sel, p(n_idx32),
        p(spectrum), spectrum.ndim, p(n_coeffs_deps), int(pulse.d), p(out)))
    return out
