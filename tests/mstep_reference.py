"""TEST INFRASTRUCTURE ONLY -- backward-error reference for the M-step solve (csrc/chol.cu, k_chol_solve) on top
of oracle/em_numpy.py (gram_and_rhs, pilot_stats, which stay pinned to the reference goldens).

A forward error bar relerr(theta, solve(G, B)) <= c * cond(G) checks almost nothing once G is ill-conditioned
and, at small cond, cannot tell a backward-stable FP64 solve from one that lost a few digits.  The normwise
backward error

    eta = ||G theta - B||_F / (||G||_F ||theta||_F + ||B||_F)

does not depend on cond(G): a backward-stable Cholesky solve gives eta of order sqrt(L) u whatever G is, and a
solve that loses precision anywhere (a lower-precision factor, a dropped low-order term of an update) gives a
larger eta at any conditioning.  G, B and the residual must then be exact to well below u, so they are formed in
np.clongdouble (64-bit mantissa), or from Gaussian-integer inputs whose every partial sum is an integer below
2^53, for which the FP64 Gram -- the device's DMMA Gram included, in any summation order -- is exact."""
from __future__ import annotations

import numpy as np
import scipy.linalg

from oracle import em_numpy as orc

U = 2.0 ** -53           # unit roundoff of FP64
LD = np.clongdouble


def tau(L):
    """Bound on eta for a backward-stable FP64 Cholesky solve of order L (the typical eta is about sqrt(L) u)."""
    return 8.0 * L * U


def exact_gram_and_rhs(Psi, Y, m, R):
    """G, B of orc.gram_and_rhs with every product and sum in clongdouble."""
    return orc.gram_and_rhs(*(np.asarray(a).astype(LD) for a in (Psi, Y, m, R)))


def system(PsiP, Yp, Xp, PsiD, Yd, m, R, exact_fp64=False):
    """Normal equations of one trial (pilots plus data statistics) -> (G, B).  exact_fp64: the inputs are Gaussian
    integers that pass integer_gram_bound, so the FP64 Gram is exact and is returned as clongdouble."""
    mp, Rp = orc.pilot_stats(Xp)
    if exact_fp64:
        assert integer_gram_bound(PsiP, Yp, mp, Rp) + integer_gram_bound(PsiD, Yd, m, R) < 2.0 ** 53
        Gp, Bp = _gram_fp64(PsiP, Yp, mp, Rp)
        Gd, Bd = _gram_fp64(PsiD, Yd, m, R)
        return (Gp + Gd).astype(LD), (Bp + Bd).astype(LD)
    Gp, Bp = exact_gram_and_rhs(PsiP, Yp, mp, Rp)
    Gd, Bd = exact_gram_and_rhs(PsiD, Yd, m, R)
    return Gp + Gd, Bp + Bd


def _gram_fp64(Psi, Y, m, R):
    """orc.gram_and_rhs as n_tx^2 BLAS products Psi^H diag(R[:, i, j]) Psi (the einsum takes seconds at L > 1000)."""
    T, N1 = Psi.shape
    n_tx = m.shape[1]
    G = np.empty((N1, n_tx, N1, n_tx), dtype=np.result_type(Psi, R))
    for i in range(n_tx):
        for j in range(n_tx):
            G[:, i, :, j] = (Psi.conj().T * R[:, i, j]) @ Psi
    V = (Psi.conj()[:, :, None] * m[:, None, :]).reshape(T, N1 * n_tx)
    return G.reshape(N1 * n_tx, N1 * n_tx), V.T @ Y


def design_system(Psi, X, Y):
    """Pilot normal equations (W^H W, W^H Y) of the design rows W[t, n n_tx + i] = psi[t, n] x[t, i], in clongdouble."""
    W = (np.asarray(Psi).astype(LD)[:, :, None] * np.asarray(X).astype(LD)[:, None, :]).reshape(Psi.shape[0], -1)
    Wh = W.conj().T
    return Wh @ W, Wh @ np.asarray(Y).astype(LD)


def backward_error(G, B, theta):
    """Normwise backward error eta of theta for G theta = B, residual in clongdouble."""
    G, B, th = (np.asarray(a).astype(LD) for a in (G, B, theta))
    nrm = lambda a: np.sqrt(np.sum(a.real ** 2 + a.imag ** 2))
    return float(nrm(G @ th - B) / (nrm(G) * nrm(th) + nrm(B)))


def refined_solve(G, B, max_iter=20):
    """Reference solution (clongdouble): FP64 Cholesky, refined with clongdouble residuals until the correction is
    below 1e-18 relative or stops shrinking (at cond(G) u_ld > 1e-18 the refinement stagnates there)."""
    G, B = np.asarray(G).astype(LD), np.asarray(B).astype(LD)
    cf = scipy.linalg.cho_factor(G.astype(np.complex128), lower=True)
    x = scipy.linalg.cho_solve(cf, B.astype(np.complex128)).astype(LD)
    last = np.inf
    for _ in range(max_iter):
        dx = scipy.linalg.cho_solve(cf, (B - G @ x).astype(np.complex128)).astype(LD)
        x = x + dx
        rel = float(np.linalg.norm(dx.astype(np.complex128)) / np.linalg.norm(x.astype(np.complex128)))
        if rel < 1e-18 or rel > 0.5 * last:
            break
        last = rel
    return x


def relerr(a, b):
    a, b = np.asarray(a).astype(LD), np.asarray(b).astype(LD)
    nrm = lambda v: np.sqrt(np.sum(v.real ** 2 + v.imag ** 2))
    return float(nrm(a - b) / nrm(b))


# ---------------------------------------------------------------------------
# Gaussian-integer inputs
# ---------------------------------------------------------------------------

def _gi(rng, shape, k):
    return (rng.integers(-k, k + 1, shape) + 1j * rng.integers(-k, k + 1, shape)).astype(np.complex128)


def integer_gram_bound(Psi, Y, m, R):
    """Largest magnitude any partial sum of a real or imaginary part of G or B can take, for integer inputs: the
    Gram and right-hand side of the entrywise |re| + |im| (every product and sum of the FP64 Gram, in any order, is
    then an integer below this)."""
    a = lambda z: np.abs(np.asarray(z).real) + np.abs(np.asarray(z).imag)
    G, B = _gram_fp64(a(Psi), a(Y), a(m), a(R))
    return float(max(G.max(initial=0.0), B.max(initial=0.0)))


def integer_inputs(rng, B, N1, n_tx, n_rx, T_p, T_d, cond=None):
    """Gaussian-integer M-step inputs of B trials: dict PsiP, PsiD, Xp, Yp, Yd, m, R (complex128 holding integers;
    R_t = A^H A + I exactly Hermitian with an integer diagonal), and per trial the exact 'G', 'B' (clongdouble) and
    'cond' (cond(G)).

    cond=None: well conditioned.  cond=kappa: RIS columns 0 and 1 are equal in every row except data row 0, where
    they differ by 1, and every other row is weighted by an integer K, so that the n_tx directions (e_0 - e_1) (x) v
    keep an O(1) eigenvalue while the rest of G grows with K^2; K is chosen from the cond at K = 1 so that
    cond(G) ~ kappa.  Every partial sum stays below 2^53 (asserted), so G and B are exact in FP64."""
    out = dict(PsiP=_gi(rng, (B, T_p, N1), 2), PsiD=_gi(rng, (B, T_d, N1), 2), Xp=_gi(rng, (B, T_p, n_tx), 1),
               Yp=_gi(rng, (B, T_p, n_rx), 3), Yd=_gi(rng, (B, T_d, n_rx), 3), m=_gi(rng, (B, T_d, n_tx), 2))
    A = _gi(rng, (B, T_d, n_tx, n_tx), 1)
    out["R"] = A.conj().transpose(0, 1, 3, 2) @ A + np.eye(n_tx)
    out["G"], out["B"], out["cond"] = [], [], []
    for b in range(B):
        def gram():
            return system(*(out[k][b] for k in ("PsiP", "Yp", "Xp", "PsiD", "Yd", "m", "R")), exact_fp64=True)
        if cond is not None:
            assert N1 >= 2 and T_d >= 1
            out["PsiP"][b, :, 1] = out["PsiP"][b, :, 0]
            out["PsiD"][b, :, 1] = out["PsiD"][b, :, 0]
            out["PsiD"][b, 0, 1] += 1
            c1 = np.linalg.cond(gram()[0].astype(np.complex128))
            K = max(1, int(round(np.sqrt(cond / c1))))
            out["PsiP"][b] *= K
            out["PsiD"][b, 1:] *= K
        G, Bm = gram()
        out["G"].append(G)
        out["B"].append(Bm)
        out["cond"].append(float(np.linalg.cond(G.astype(np.complex128))))
    return out
