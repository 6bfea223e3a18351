"""Extended-precision reference of the first-order control matrix and its per-entry error scale.

    B_jk(w) = sum_g e^{i w t_g} sum_mn Bbar^{(g)}_{j,mn} I^{(g)}_mn(w) Cbar^{(g)}_{k,nm}
    Bbar^{(g)}_j = s_j^{(g)} V_g^+ N_j V_g,   Cbar^{(g)}_k = (Q_g^+ V_g)^+ C_k (Q_g^+ V_g),
    I^{(g)}_mn(w) = dt_g e^{iy} sin(y)/y,  y = x dt_g / 2,  x = w + E_m - E_n  (dt_g where y = 0)

evaluated in np.longdouble / np.clongdouble (64-bit significand on x86-64) from the caller's float64
inputs, promoted exactly.  It does not depend on an eigensolver, so it serves the function route (inputs
drawn by the test) and the pulse route (the pulse's own cached eigensystem) alike.

The phase e^{i w t_g} is evaluated without rounding its argument: t_g is cut into pieces of 11 significant
bits, each product w * piece is exact in the 64-bit significand, and the phase is the product of the
pieces' phases.  This keeps the reference accurate at |w t| ~ 1e7, where a rounded argument would cost
~1e-12 absolute.

Error scale of a float64 evaluation of the same formula, per entry:

    M_jk(w) = sum_g sum_mn |Bbar_j,mn| |I_mn| |Cbar_k,nm| (d + sqrt(G) + |w t_g| + |x_mn dt_g|)

d covers the transforms and the contraction, sqrt(G) the sum over the G segments (its rounding errors add
like a random walk in every order the kernels and the float64 formula use; at omega ~ 0, where the terms
add coherently, the float64 formula reaches 1.2 EPS M at d = 2, G = 300 without it), |w t_g| the rounding
of fl(w t_g) (the kernels round that product exactly as the float64 formula does), |x dt_g| the rounding
of the integral's argument.  A float64 kernel passes when |B - B_hp| <= kappa * EPS * M at every entry.
"""
import numpy as np

LD, CLD = np.longdouble, np.clongdouble
EPS = 2.0**-53

if np.finfo(LD).nmant < 63:  # pragma: no cover - platforms whose long double is float64
    raise ImportError('hp_control_matrix needs an 80-bit long double (x86-64)')


def _pieces(x, n=5, bits=11):
    """float64 array -> n float64 arrays of at most `bits` significant bits that sum to x exactly."""
    out, rest = [], np.asarray(x, dtype=float).copy()
    for _ in range(n):
        m, e = np.frexp(rest)
        hi = np.ldexp(np.trunc(np.ldexp(m, bits)), e - bits)
        out.append(hi)
        rest = rest - hi  # exact: hi holds the leading bits of rest
    assert not rest.any()
    return out


def _cis(a):
    return np.cos(a) + 1j*np.sin(a)


def exact_phase(omega, t_g):
    """e^{i omega t_g} (clongdouble) for float64 omega (array) and t_g (scalar), argument not rounded."""
    w = np.asarray(omega, dtype=float).astype(LD)
    phase = np.ones(w.shape, dtype=CLD)
    for piece in _pieces(np.float64(t_g)):
        if piece:
            phase = phase*_cis(w*LD(piece))  # 53 x 11 bits: exact in the 64-bit significand
    return phase


def transformed_operators(eigvecs, propagators, basis, n_opers, n_coeffs):
    """Bbar (n_nops, G, d, d) and Cbar (G, n_basis, d, d) in clongdouble."""
    V = np.asarray(eigvecs, dtype=complex).astype(CLD)
    Q = np.asarray(propagators, dtype=complex).astype(CLD)
    C = np.asarray(basis, dtype=complex).astype(CLD)
    N = np.asarray(n_opers, dtype=complex).astype(CLD)
    s = np.asarray(n_coeffs, dtype=float).astype(LD)
    Vd = V.conj().swapaxes(-1, -2)
    Bbar = (Vd[None] @ N[:, None] @ V[None])*s[:, :, None, None]
    QdV = Q[:-1].conj().swapaxes(-1, -2) @ V
    Cbar = QdV.conj().swapaxes(-1, -2)[:, None] @ C[None] @ QdV[:, None]
    return Bbar, Cbar


def control_matrix(eigvals, eigvecs, propagators, omega, basis, n_opers, n_coeffs, dt, t=None):
    """(B_hp, M): the control matrix (n_nops, n_basis, n_omega) in clongdouble and its error scale in
    longdouble.  Arguments as numeric.calculate_control_matrix_from_scratch."""
    eigvals = np.asarray(eigvals, dtype=float)
    omega = np.asarray(omega, dtype=float)
    dt = np.asarray(dt, dtype=float)
    t = np.concatenate(([0.0], dt.cumsum())) if t is None else np.asarray(t, dtype=float)
    G, d = eigvals.shape
    Bbar, Cbar = transformed_operators(eigvecs, propagators, basis, n_opers, n_coeffs)
    n_nops, n_basis, n_omega = Bbar.shape[0], Cbar.shape[1], len(omega)
    E = eigvals.astype(LD)
    w = omega.astype(LD)
    B = np.zeros((n_omega, n_nops, n_basis), dtype=CLD)
    M = np.zeros((n_omega, n_nops, n_basis), dtype=LD)
    root_G = np.sqrt(LD(G))
    for g in range(G):
        dtg = LD(dt[g])
        x = w[:, None, None] + (E[g][:, None] - E[g][None, :])            # (n_omega, d, d)
        y = x*dtg/2
        zero = y == 0
        sinc = np.sin(y)/np.where(zero, 1, y)
        sinc[zero] = 1
        integral = dtg*_cis(y)*sinc
        CT = Cbar[g].swapaxes(-1, -2).reshape(n_basis, d*d).T             # (d*d, n_basis)
        X = (integral[:, None]*Bbar[None, :, g]).reshape(n_omega*n_nops, d*d)
        phase = exact_phase(omega, t[g])
        B += (X @ CT).reshape(n_omega, n_nops, n_basis)*phase[:, None, None]
        weight = d + root_G + np.abs(w*LD(t[g]))[:, None, None] + np.abs(x*dtg)
        aX = (np.abs(integral)[:, None]*np.abs(Bbar[None, :, g])*weight[:, None]).reshape(n_omega*n_nops, d*d)
        M += (aX @ np.abs(CT)).reshape(n_omega, n_nops, n_basis)
    return B.transpose(1, 2, 0), M.transpose(1, 2, 0)


def ratio(B, B_hp, M):
    """|B - B_hp| / (EPS M) per entry (float64); entries with M = 0 must match exactly."""
    err = np.abs(np.asarray(B).astype(CLD) - B_hp)
    with np.errstate(divide='ignore', invalid='ignore'):
        r = np.where(M > 0, err/(EPS*M), np.where(err > 0, np.inf, 0))
    return r.astype(float)
