"""Extended-precision reference of the front end -- eigenvalues, piecewise propagators and their running
product -- and the error scales of a float64 evaluation.

    P_g = exp(-i H_g dt_g),   Q_0 = 1,  Q_{g+1} = P_g Q_g

evaluated in np.longdouble / np.clongdouble (64-bit significand on x86-64) from the caller's float64 inputs,
promoted exactly.  The propagators come from scaling and squaring with a Taylor core, not from an
eigensolver, so they are independent of what they check; the eigenvalues of sampled segments come from
mpmath at 30 digits.

Error scales of a float64 evaluation, with EPS = 2^-53 and per segment m_g = d (1 + ||H_g||_2 dt_g):

- eigenvalues                  |lambda_j - lambda_j^hp|           <= kappa EPS d ||H_g||_2
- eigenvectors                 ||H v_j - lambda_j v_j||_max        <= kappa EPS d ||H_g||_2
                               ||V^+ V - 1||_max                   <= kappa EPS d
- one step                     ||Q_{g+1} Q_g^-1 - P_g^hp||_max     <= kappa EPS (m_g + d depth)
- the chain                    ||Q_g - Q_g^hp||_max                <= kappa EPS (d depth + sum_{h<g} m_h)

depth is the number of matrix products on the path of one Q_g (log2 of the scan block, the levels of the
tree product of the block totals, one apply per scan level).  The step quotient isolates the rounding of
one segment from the drift accumulated before it.  The chain bound is linear in G: a sequential float64
product of near-identity steps drifts almost linearly (the oracle's own chain reaches 1.55 times the
linear scale with kappa = 1), so a sqrt(G) bound is not a property of float64 evaluation.  The unitarity
defect ||Q_g^+ Q_g - 1||_max is checked separately against the float64 oracle's.
"""
import math

import mpmath
import numpy as np

LD, CLD = np.longdouble, np.clongdouble
EPS = 2.0**-53

if np.finfo(LD).nmant < 63:  # pragma: no cover - platforms whose long double is float64
    raise ImportError('hp_propagators needs an 80-bit long double (x86-64)')

_TAYLOR_TERMS = 24  # ||A|| <= 1/2 after scaling: 0.5^24 / 24! < 1e-30


def promote(H):
    return np.asarray(H, dtype=complex).astype(CLD)


def spectral_norms(H):
    """||H_g||_2 per segment (float64)."""
    H = np.asarray(H, dtype=complex)
    return np.linalg.norm(H, 2, axis=(-2, -1)) if H.shape[-1] > 1 else np.abs(H[:, 0, 0])


def propagators(H, dt):
    """exp(-i H_g dt_g) in clongdouble by scaling and squaring with a Taylor core, all segments at once."""
    A = promote(H)*(-1j*np.asarray(dt, dtype=float).astype(LD))[:, None, None]
    G, d, _ = A.shape
    norm1 = np.abs(A).sum(axis=-2).max(axis=-1).astype(float)
    s = np.maximum(0, np.ceil(np.log2(np.maximum(norm1, 1e-300)/0.5))).astype(int)
    A = A*np.ldexp(np.ones(G), -s).astype(LD)[:, None, None]  # exact
    eye = np.broadcast_to(np.eye(d, dtype=CLD), A.shape)
    P = eye.copy()
    for k in range(_TAYLOR_TERMS, 0, -1):  # Horner: 1 + A/1 (1 + A/2 (1 + ...))
        P = eye + (A @ P)/LD(k)
    for r in range(1, int(s.max(initial=0)) + 1):
        sel = s >= r
        P[sel] = P[sel] @ P[sel]
    return P


def chain(P):
    """Q_0 = 1, Q_{g+1} = P_g Q_g by the sequential product in clongdouble."""
    G, d, _ = P.shape
    Q = np.empty((G + 1, d, d), dtype=CLD)
    Q[0] = np.eye(d)
    for g in range(G):
        Q[g + 1] = P[g] @ Q[g]
    return Q


def sample(G, seed=0, n=64):
    """Segments whose eigenvalues are checked: all for G <= n, else a seeded n plus the first and last."""
    if G <= n:
        return np.arange(G)
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate(([0, G - 1], rng.choice(G, n, replace=False))))


def eigvals(H, idx):
    """Eigenvalues (ascending, longdouble) of the segments idx by mpmath.eighe at 30 digits."""
    H = np.asarray(H, dtype=complex)
    out = np.empty((len(idx), H.shape[-1]), dtype=LD)
    with mpmath.workdps(30):
        for i, g in enumerate(idx):
            A = mpmath.matrix([[mpmath.mpc(x.real, x.imag) for x in row] for row in H[g]])
            E = sorted(mpmath.eighe(A, eigvals_only=True))
            out[i] = [LD(mpmath.nstr(e, 30)) for e in E]
    return out


def inverse(Q):
    """Q^-1 in clongdouble for nearly unitary Q: Newton's iteration X <- X (2 - Q X) from X = Q^+."""
    X = Q.conj().swapaxes(-1, -2)
    two = 2*np.eye(Q.shape[-1], dtype=CLD)
    for _ in range(3):
        X = X @ (two - Q @ X)
    return X


def segment_scale(H, dt):
    """m_g = d (1 + ||H_g||_2 dt_g)."""
    d = np.asarray(H).shape[-1]
    return d*(1 + spectral_norms(H)*np.abs(np.asarray(dt, dtype=float)))


def _ratio(err, scale):
    """err / (EPS scale) elementwise; a zero scale admits only a zero error."""
    err = np.asarray(err, dtype=float)
    scale = np.asarray(scale, dtype=float)
    with np.errstate(divide='ignore', invalid='ignore'):
        return np.where(scale > 0, err/(EPS*scale), np.where(err > 0, np.inf, 0.0))


def _maxabs(x):
    return np.abs(x).max(axis=(-2, -1))


class Reference:
    """The reference of one Hamiltonian: propagators, chain, sampled eigenvalues and error scales."""

    def __init__(self, H, dt, seed=0):
        self.H = np.asarray(H, dtype=complex)
        self.dt = np.asarray(dt, dtype=float)
        G, d, _ = self.H.shape
        self.G, self.d = G, d
        self.norms = spectral_norms(self.H)
        self.m = segment_scale(self.H, self.dt)
        self.P = propagators(self.H, self.dt)
        self.Q = chain(self.P)
        self.idx = sample(G, seed)
        self.ev = eigvals(self.H, self.idx)

    def ratios(self, ev, V, Q, depth):
        """Per-bound worst |error| / (EPS scale) of a float64 result (ev, V, Q) whose chain runs through
        `depth` matrix products per Q_g."""
        d = self.d
        ev = np.asarray(ev, dtype=float)
        Hl = promote(self.H)
        Vl = promote(V)
        Ql = promote(Q)
        evl = ev.astype(LD)
        out = {}
        out['eigvals'] = _ratio(np.abs(evl[self.idx] - self.ev).max(axis=-1), d*self.norms[self.idx]).max()
        resid = _maxabs(Hl @ Vl - Vl*evl[:, None, :])
        out['residual'] = _ratio(resid, d*self.norms).max()
        gram = Vl.conj().swapaxes(-1, -2) @ Vl - np.eye(d)
        out['orthonormality'] = _ratio(_maxabs(gram), np.full(self.G, float(d))).max()
        step = _maxabs(Ql[1:] @ inverse(Ql[:-1]) - self.P)
        out['step'] = _ratio(step, self.m + d*depth).max()
        drift = np.concatenate(([0.0], np.cumsum(self.m)))
        out['chain'] = _ratio(_maxabs(Ql - self.Q), d*depth + drift).max()
        return {k: float(v) for k, v in out.items()}


def unitarity_defect(Q, g):
    """||Q_g^+ Q_g - 1||_max (evaluated in long double) of the chain entries g."""
    Qg = promote(np.asarray(Q)[g])
    return _maxabs(Qg.conj().swapaxes(-1, -2) @ Qg - np.eye(Qg.shape[-1])).astype(float)


def drift_bound(defect_oracle, d, g, kappa):
    """What the unitarity defect of Q_g may reach: twice the float64 oracle's, or kappa EPS d sqrt(g)."""
    return np.maximum(2*np.asarray(defect_oracle), kappa*EPS*d*np.sqrt(np.asarray(g, dtype=float)))


def scan_depth(path, d, G):
    """Matrix products on the path of one Q_g.  'small': the block scan of NT = 256 (d = 2) or 128 (d = 3, 4)
    segments, recursive over the block totals while there are more than 96 blocks; 'generic': one product in
    the chunk, one in the chunk totals, one apply."""
    if path == 'generic':
        return 3
    if path == 'oracle':
        return 1
    NT = 256 if d == 2 else 128
    depth, n = 0, G
    while True:
        nb = -(-n//NT)
        depth += int(math.log2(NT)) + 1
        if nb <= 96:
            return depth + math.ceil(math.log2(nb)) if nb > 1 else depth
        n = nb
