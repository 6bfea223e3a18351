"""Extended-precision reference of the infidelity gradient (ff.infidelity_derivative) and its per-entry
error scale.

    dI_a/du_h(g) = 1/(pi d) sum_w u_w S_a(w) Re[c1 + c2 + c3]          (DESIGN.md section 4.11)
    c1 = e s sum_ij Abar_h,ij R_ij,  R_ij = i dt^2 [sum_n Bbar_jn E3(z_jn, z_in) Wt_ni
                                                   - sum_m Bbar_mi E3(z_mi, z_mj) Wt_jm]
    c2 = sum_ij (Abar_h o I(0))_ij (-i Xt_ji),   Xt = U^+ [W, Y_{>g}] U
    c3 = (ds_a(g)/du_h(g)) e tr((Bbar o I) Wt)

with U = Q_{g-1}^+ V_g, Wt = U^+ W U, W_a = sum_k conj(B_ak) C_k, Y_{>g} the sum of the later segment terms,
z_mn = (w + E_m - E_n) dt and E3(z1, z2) = exp[i z1, i z2, 0] evaluated with the kernels' three branches.

`derivative(..., hp=True)` evaluates it in np.longdouble / np.clongdouble from the float64 inputs (the
control matrix from hp_control_matrix, the phase e^{iwt} without rounding its argument) and returns the
error scale M of a float64 evaluation: the same sum with absolute values of every factor as it is
evaluated (|W| from the control matrix's own error scale, the difference quotients of E3 as
(|f1| + |f2|) / |dz|), weighted by d + sqrt(G) + |w t_g| + max |z|.  `derivative(..., hp=False)` is the
float64 evaluation of the same formula.  A float64 evaluation passes when |dI - dI_hp| <= kappa EPS M.
"""
import numpy as np

import hp_control_matrix as hpc

LD, CLD = np.longdouble, np.clongdouble
EPS = hpc.EPS


def _e2(z, C):
    y = z/2
    half = (np.cos(y) + 1j*np.sin(y)).astype(C)
    sinc = np.sin(y)/np.where(y == 0, 1, y)
    sinc = np.where(y == 0, 1, sinc)
    return half, half*sinc


def _e3(z1, z2, h1, h2, f1, f2, R, C):
    """exp[i z1, i z2, 0] and the absolute-value scale of its evaluation (broadcasting)."""
    z1, z2 = np.broadcast_arrays(z1, z2)
    h1, h2, f1, f2 = np.broadcast_arrays(h1, h2, f1, f2)
    with np.errstate(all='ignore'):
        dz = z1 - z2
        far = np.abs(dz) > 1
        v_far = (f1 - f2)/(1j*np.where(far, dz, 1))
        a_far = (np.abs(f1) + np.abs(f2))/np.abs(np.where(far, dz, 1))
        first = np.abs(z1) >= np.abs(z2)
        y = dz/2
        sinc = np.where(y == 0, 1, np.sin(y)/np.where(y == 0, 1, y))
        pp = h1*h2*sinc
        zz = np.where(first, z1, z2)
        ff = np.where(first, f2, f1)
        near = ~far & (np.maximum(np.abs(z1), np.abs(z2)) > 1)
        zs = np.where(near, zz, 1)
        v_near = (pp - ff)/(1j*zs)
        a_near = (np.abs(pp) + np.abs(ff))/np.abs(zs)
        lo = np.minimum(np.minimum(z1, z2), 0)
        hi = np.maximum(np.maximum(z1, z2), 0)
        cen = (lo + hi)/2
        u0, u1, u2 = z1 - cen, z2 - cen, -cen
        small = ~far & ~near
        u0, u1, u2 = (np.where(small, u, 0) for u in (u0, u1, u2))
        p0 = np.ones_like(u0)
        H2 = np.ones_like(u0)
        H3 = np.ones_like(u0)
        inv_fact = R(1)/2
        total = np.full(u0.shape, inv_fact, dtype=C)
        for n in range(1, 21):
            p0 = p0*u0
            H2 = p0 + u1*H2
            H3 = H2 + u2*H3
            inv_fact = inv_fact/(n + 2)
            total = total + (1j**n)*H3*inv_fact
        v_small = (np.cos(cen) + 1j*np.sin(cen))*total
        val = np.where(far, v_far, np.where(near, v_near, v_small)).astype(C)
        scale = np.where(far, a_far, np.where(near, a_near, np.abs(v_small))).astype(R)
    return val, scale


def derivative(eigvals, eigvecs, propagators, omega, basis, n_opers, n_coeffs, dt, t, c_opers,
               spectrum, n_coeffs_deps=None, ctrl_idx=None, nop_idx=None, norm_d=None, hp=True,
               control_matrix=None):
    """(dI, M): the derivative (n_sel, G, n_ctrl) and, with hp=True, its float64 error scale (else None).
    spectrum is (n_omega,) or (n_sel, n_omega); control_matrix (all noise operators) is computed with
    hp_control_matrix (hp=True) or must be passed (hp=False, e.g. the oracle's)."""
    R, C = (LD, CLD) if hp else (np.float64, np.complex128)
    eigvals = np.asarray(eigvals, dtype=float)
    omega = np.asarray(omega, dtype=float)
    dt = np.asarray(dt, dtype=float)
    t = np.asarray(t, dtype=float)
    G, d = eigvals.shape
    n_nops = len(n_opers)
    ctrl_idx = np.arange(len(c_opers)) if ctrl_idx is None else np.asarray(ctrl_idx)
    nop_idx = np.arange(n_nops) if nop_idx is None else np.asarray(nop_idx)
    norm_d = d if norm_d is None else norm_d
    n_sel, n_ctrl, n_omega = len(nop_idx), len(ctrl_idx), len(omega)
    if hp:
        B, MB = hpc.control_matrix(eigvals, eigvecs, propagators, omega, basis, n_opers, n_coeffs, dt, t)
    else:
        B, MB = np.asarray(control_matrix, dtype=complex), None
    cast = (lambda x: np.asarray(x, dtype=complex).astype(C))
    V, Q, Cb = cast(eigvecs), cast(propagators), cast(basis)
    N, A = cast(n_opers)[nop_idx], cast(c_opers)[ctrl_idx]
    E, w, dtR = eigvals.astype(R), omega.astype(R), dt.astype(R)
    s = np.asarray(n_coeffs, dtype=float)[nop_idx].astype(R)                       # (a, G)
    deps = (np.zeros((n_sel, n_ctrl, G)) if n_coeffs_deps is None
            else np.asarray(n_coeffs_deps, dtype=float)[nop_idx]).astype(R)        # (a, h, G)
    spectrum = np.broadcast_to(np.asarray(spectrum, dtype=float), (n_sel, n_omega)).astype(R)
    u = np.zeros(n_omega, dtype=R)
    if n_omega > 1:
        left = np.concatenate(([0], w[1:] - w[:-1]))
        right = np.concatenate((w[1:] - w[:-1], [0]))
        u = (left + right)/2
    us = u[None]*spectrum                                                          # (a, w)
    Vd = V.conj().swapaxes(-1, -2)
    U = Q[:-1].conj().swapaxes(-1, -2) @ V                                         # (G, d, d)
    Ud = U.conj().swapaxes(-1, -2)
    Bb = Vd[None] @ N[:, None] @ V[None]                                           # (a, G, d, d)
    Ab = Vd[None] @ A[:, None] @ V[None]                                           # (h, G, d, d)
    z0 = (E[:, :, None] - E[:, None, :])*dtR[:, None, None]
    I0 = dtR[:, None, None]*_e2(z0, C)[1]
    AI0 = Ab*I0[None]
    Bsel = np.asarray(B)[nop_idx].astype(C)
    W = np.einsum('akw,kij->awij', Bsel.conj(), Cb)
    Y = np.zeros_like(W)
    out = np.zeros((n_sel, G, n_ctrl), dtype=R)
    if hp:
        aW = np.einsum('akw,kij->awij', np.asarray(MB)[nop_idx].astype(R), np.abs(Cb))
        aY = np.zeros(W.shape, dtype=R)
        M = np.zeros((n_sel, G, n_ctrl), dtype=R)
        root_G = np.sqrt(R(G))
    for g in range(G - 1, -1, -1):
        z = ((w[:, None, None] + E[g][None, :, None]) - E[g][None, None, :])*dtR[g]   # (w, d, d)
        hf, f = _e2(z, C)
        I = dtR[g]*f
        BI = Bb[:, g][:, None]*I[None]                                             # (a, w, d, d)
        Wt = Ud[g] @ W @ U[g]
        Xt = Ud[g] @ (W @ Y - Y @ W) @ U[g]
        tau = np.einsum('awmn,awnm->aw', BI, Wt)
        K1, aK1 = _e3(z[:, None, :, :], z[:, :, None, :], hf[:, None, :, :], hf[:, :, None, :],
                      f[:, None, :, :], f[:, :, None, :], R, C)                     # (w, i, j, n)
        K2, aK2 = _e3(z[:, :, :, None], z[:, :, None, :], hf[:, :, :, None], hf[:, :, None, :],
                      f[:, :, :, None], f[:, :, None, :], R, C)                     # (w, m, i, j)
        Rm = (np.einsum('ajn,wijn,awni->awij', Bb[:, g], K1, Wt)
              - np.einsum('ami,wmij,awjm->awij', Bb[:, g], K2, Wt))
        e = hpc.exact_phase(omega, t[g]) if hp else np.exp(1j*(omega*t[g]))
        C1 = 1j*dtR[g]**2*s[:, g, None, None, None]*e[None, :, None, None]*Rm
        X2 = -1j*Xt.swapaxes(-1, -2)
        val = (np.einsum('hij,awij->ahw', Ab[:, g], C1) + np.einsum('hij,awij->ahw', AI0[:, g], X2)).real
        val = val + deps[:, :, g, None]*(e[None]*tau).real[:, None, :]
        out[:, g, :] = np.einsum('ahw,aw->ah', val, us)
        T = U[g] @ BI @ Ud[g]
        Y = Y + (s[:, g, None, None, None]*e[None, :, None, None])*T
        if hp:
            aU, aUd = np.abs(U[g]), np.abs(Ud[g])
            aBI = np.abs(Bb[:, g])[:, None]*np.abs(I)[None]
            aWt = aUd @ aW @ aU
            aXt = aUd @ (aW @ aY + aY @ aW) @ aU
            atau = np.einsum('awmn,awnm->aw', aBI, aWt)
            aBb = np.abs(Bb[:, g])
            aR = (np.einsum('ajn,wijn,awni->awij', aBb, aK1, aWt)
                  + np.einsum('ami,wmij,awjm->awij', aBb, aK2, aWt))
            aC1 = dtR[g]**2*np.abs(s[:, g, None, None, None])*aR
            mval = (np.einsum('hij,awij->ahw', np.abs(Ab[:, g]), aC1)
                    + np.einsum('hij,awij->ahw', np.abs(AI0[:, g]), aXt.swapaxes(-1, -2)))
            mval = mval + np.abs(deps[:, :, g, None])*atau[:, None, :]
            weight = d + root_G + np.abs(w*R(t[g])) + np.abs(z).max(axis=(1, 2))
            M[:, g, :] = np.einsum('ahw,aw->ah', mval*weight[None, None], np.abs(us))
            aY = aY + np.abs(s[:, g, None, None, None])*(aU @ aBI @ aUd)
    scale = 1/(np.pi*R(norm_d)) if hp else 1/(np.pi*norm_d)
    return out*scale, (M*scale if hp else None)


def ratio(dI, dI_hp, M):
    """|dI - dI_hp| / (EPS M) per entry (float64); entries with M = 0 must match exactly."""
    err = np.abs(np.asarray(dI, dtype=float).astype(LD) - dI_hp)
    with np.errstate(divide='ignore', invalid='ignore'):
        r = np.where(M > 0, err/(EPS*M), np.where(err > 0, np.inf, 0))
    return r.astype(float)
