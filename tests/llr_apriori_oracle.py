"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the extrinsic bit LLRs with a-priori input (include/sbce.h,
sbce_bit_llr_apriori), written independently of the kernel's penalty form.

Every hypothesis k gets the log-weight -d2_k/varn^2 - sum_{j,i} b_ji(k) La_ji (the prior's ln P(b) up to a
constant per symbol), with La clamped to +-CLAMP first; each side of each bit is a logaddexp reduction over the
hypotheses whose label has that bit, the bit's La is subtracted and the result is clamped to +-CLAMP.  A NaN in
a symbol's La makes all of its LLRs NaN (0 * NaN reaches every hypothesis), as does a non-finite input."""
from __future__ import annotations

import numpy as np

import llr_oracle as lo
from oracle import em_numpy as orc

CLAMP = lo.CLAMP


def clamp_prior(La):
    with np.errstate(invalid="ignore"):
        return np.clip(np.asarray(La, np.float64), -CLAMP, CLAMP)   # NaN stays NaN, +-inf -> +-32


def _finish(l0, l1, La, clamp):
    with np.errstate(invalid="ignore"):
        v = l0 - l1 - La
        return np.clip(v, -CLAMP, CLAMP) if clamp else v


def bit_llr_apriori(Yd, PsiD, Theta, cons, n_tx, varn, La, Xoff=None, clamp=True):
    """(T_d, n_tx, log2 M) float64 extrinsic LLRs of one trial with priors La (T_d, n_tx, log2 M), every
    hypothesis enumerated (K up to 2^20); clamp=False returns the unclamped values."""
    M = len(cons)
    K = M ** n_tx
    lab = lo.bit_labels(M)
    nb = lab.shape[1]
    La = clamp_prior(La)
    Y, Heff = lo._data_residual_input(Yd, PsiD, Theta, n_tx, Xoff)
    s2 = float(varn) ** 2
    dig = orc.hypothesis_digits(np.arange(K), M, n_tx)            # (K, n_tx)
    table = cons[dig]
    bits = lab[dig].reshape(K, n_tx * nb).astype(np.float64)      # b_ji(k), (K, n_tx * nb)
    T_d = Y.shape[0]
    out = np.empty((T_d, n_tx, nb))
    chunk = max(1, (1 << 21) // K)
    for t0 in range(0, T_d, chunk):
        sl = slice(t0, min(T_d, t0 + chunk))
        with np.errstate(invalid="ignore"):
            a = -orc.hypothesis_distances(Y[sl], Heff[sl], table) / s2 - La[sl].reshape(-1, n_tx * nb) @ bits.T
        for j in range(n_tx):
            for i in range(nb):
                one = lab[dig[:, j], i].astype(bool)
                with np.errstate(invalid="ignore"):
                    l0 = np.logaddexp.reduce(a[:, ~one], axis=1)
                    l1 = np.logaddexp.reduce(a[:, one], axis=1)
                out[sl, j, i] = _finish(l0, l1, La[sl, j, i], clamp)
    return out


def bit_llr_apriori_split(Yd, PsiD, Theta, cons, n_tx, varn, La, Xoff=None, clamp=True):
    """bit_llr_apriori for the 2^24-leaf trees, split as llr_oracle.bit_llr_split: the prior is separable per
    stream, so the leading half's part is added to the rows (a) and the trailing half's to the columns (b)."""
    M = len(cons)
    lab = lo.bit_labels(M)
    nb = lab.shape[1]
    La = clamp_prior(La)
    nA = n_tx // 2
    dA = orc.hypothesis_digits(np.arange(M ** nA), M, nA)
    dB = orc.hypothesis_digits(np.arange(M ** (n_tx - nA)), M, n_tx - nA)
    XA, XB = cons[dA], cons[dB]
    bA = lab[dA].reshape(len(dA), -1).astype(np.float64)
    bB = lab[dB].reshape(len(dB), -1).astype(np.float64)
    Y, Heff = lo._data_residual_input(Yd, PsiD, Theta, n_tx, Xoff)
    s2 = float(varn) ** 2
    T_d = Y.shape[0]
    out = np.empty((T_d, n_tx, nb))
    rows = max(1, (1 << 21) // len(XB))
    for t in range(T_d):
        u = Y[t][None, :] - XA @ Heff[t][:, :nA].T
        v = XB @ Heff[t][:, nA:].T
        with np.errstate(invalid="ignore"):
            pA = -bA @ La[t, :nA].reshape(-1)
            pB = -bB @ La[t, nA:].reshape(-1)
        a = np.empty((len(XA), len(XB)))
        for a0 in range(0, len(XA), rows):
            r = u[a0:a0 + rows, None, :] - v[None, :, :]
            with np.errstate(invalid="ignore"):
                a[a0:a0 + rows] = -(r.real ** 2 + r.imag ** 2).sum(axis=2) / s2 + pA[a0:a0 + rows, None] + pB[None, :]
        with np.errstate(invalid="ignore"):
            la = np.logaddexp.reduce(a, axis=1)     # (KA,)
            lb = np.logaddexp.reduce(a, axis=0)     # (KB,)
            for j in range(n_tx):
                lm, dj = (la, dA[:, j]) if j < nA else (lb, dB[:, j - nA])
                for i in range(nb):
                    one = lab[dj, i].astype(bool)
                    out[t, j, i] = _finish(np.logaddexp.reduce(lm[~one]), np.logaddexp.reduce(lm[one]), La[t, j, i],
                                           clamp)
    return out
