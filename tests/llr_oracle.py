"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the exact Gray-labelled bit LLRs (include/sbce.h,
sbce_bit_llr), built on the E-step pieces of oracle/em_numpy.py (which stays pinned to the reference goldens).

Every hypothesis's residual is formed directly, as posterior_stats does, and each side of each bit is a
logaddexp reduction of -d2/varn^2 over the hypotheses whose label has that bit; the result is clamped to
+-CLAMP.  A symbol with a non-finite input has NaN LLRs (NaN propagates through the reductions)."""
from __future__ import annotations

import numpy as np

from oracle import em_numpy as orc

CLAMP = 32.0


def bit_labels(M):
    """(M, log2 M) labels: gray(iI) MSB first, then gray(iQ) MSB first, m = iQ*sqrt(M) + iI (restated here
    independently of the package's qam.bit_labels)."""
    sq = int(round(np.sqrt(M)))
    q = sq.bit_length() - 1
    out = np.zeros((M, 2 * q), dtype=np.uint8)
    for m in range(M):
        iI, iQ = m % sq, m // sq
        gI, gQ = iI ^ (iI >> 1), iQ ^ (iQ >> 1)
        for i in range(q):
            out[m, i] = (gI >> (q - 1 - i)) & 1
            out[m, q + i] = (gQ >> (q - 1 - i)) & 1
    return out


def _data_residual_input(Yd, PsiD, Theta, n_tx, Xoff):
    Heff = orc.effective_channels(PsiD, Theta, n_tx)
    Y = Yd if Xoff is None else Yd - np.einsum("trj,tj->tr", Heff, Xoff)   # hypotheses x_k + o_t
    return Y, Heff


def _finish(l0, l1, clamp):
    with np.errstate(invalid="ignore"):
        return np.clip(l0 - l1, -CLAMP, CLAMP) if clamp else l0 - l1


def bit_llr(Yd, PsiD, Theta, cons, n_tx, varn, Xoff=None, clamp=True):
    """(T_d, n_tx, log2 M) float64 bit LLRs of one trial, every hypothesis enumerated (K up to 2^20); clamp=False
    returns the unclamped values."""
    M = len(cons)
    K = M ** n_tx
    lab = bit_labels(M)
    nb = lab.shape[1]
    Y, Heff = _data_residual_input(Yd, PsiD, Theta, n_tx, Xoff)
    s2 = float(varn) ** 2
    dig = orc.hypothesis_digits(np.arange(K), M, n_tx)            # (K, n_tx)
    table = cons[dig]
    T_d = Y.shape[0]
    out = np.empty((T_d, n_tx, nb))
    chunk = max(1, (1 << 21) // K)
    for t0 in range(0, T_d, chunk):
        sl = slice(t0, min(T_d, t0 + chunk))
        with np.errstate(invalid="ignore"):
            a = -orc.hypothesis_distances(Y[sl], Heff[sl], table) / s2   # (t, K)
        for j in range(n_tx):
            for i in range(nb):
                one = lab[dig[:, j], i].astype(bool)
                with np.errstate(invalid="ignore"):
                    l0 = np.logaddexp.reduce(a[:, ~one], axis=1)
                    l1 = np.logaddexp.reduce(a[:, one], axis=1)
                out[sl, j, i] = _finish(l0, l1, clamp)
    return out


def bit_llr_split(Yd, PsiD, Theta, cons, n_tx, varn, Xoff=None, clamp=True):
    """bit_llr for the 2^24-leaf trees: streams split into a leading half A and a trailing half B as in
    posterior_stats_split, residuals formed directly for every (a, b) block by block; the sides of a bit of A
    reduce over b first (per-a logaddexp), those of B over a first."""
    M = len(cons)
    lab = bit_labels(M)
    nb = lab.shape[1]
    nA = n_tx // 2
    dA = orc.hypothesis_digits(np.arange(M ** nA), M, nA)
    dB = orc.hypothesis_digits(np.arange(M ** (n_tx - nA)), M, n_tx - nA)
    XA, XB = cons[dA], cons[dB]
    Y, Heff = _data_residual_input(Yd, PsiD, Theta, n_tx, Xoff)
    s2 = float(varn) ** 2
    T_d = Y.shape[0]
    out = np.empty((T_d, n_tx, nb))
    rows = max(1, (1 << 21) // len(XB))
    for t in range(T_d):
        u = Y[t][None, :] - XA @ Heff[t][:, :nA].T
        v = XB @ Heff[t][:, nA:].T
        a = np.empty((len(XA), len(XB)))
        for a0 in range(0, len(XA), rows):
            r = u[a0:a0 + rows, None, :] - v[None, :, :]
            with np.errstate(invalid="ignore"):
                a[a0:a0 + rows] = -(r.real ** 2 + r.imag ** 2).sum(axis=2) / s2
        with np.errstate(invalid="ignore"):
            la = np.logaddexp.reduce(a, axis=1)     # (KA,)
            lb = np.logaddexp.reduce(a, axis=0)     # (KB,)
            for j in range(n_tx):
                lm, dj = (la, dA[:, j]) if j < nA else (lb, dB[:, j - nA])
                for i in range(nb):
                    one = lab[dj, i].astype(bool)
                    out[t, j, i] = _finish(np.logaddexp.reduce(lm[~one]), np.logaddexp.reduce(lm[one]), clamp)
    return out
