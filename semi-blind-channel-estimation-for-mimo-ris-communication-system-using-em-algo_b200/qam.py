"""Square QAM constellation and joint-hypothesis indexing used by the estimator.

Restates what the reference takes from its vendored modulation module
(/root/reference/Proposed method/QAM.py:310-322): the UN-normalised grid
c[iQ*sqrt(M)+iI] = (2 iI - sqrt(M) + 1) + 1j (2 iQ - sqrt(M) + 1), and the
itertools.product ordering of joint hypotheses (Proposed method/PM.py:25-31):
k = sum_j idx_j * M**(n_tx-1-j), stream 0 most significant.
"""
from __future__ import annotations

import numpy as np

SUPPORTED_M = (4, 16, 64)


def constellation(M: int) -> np.ndarray:
    root = int(round(float(M) ** 0.5))
    if root * root != M or root & (root - 1):
        raise ValueError("constellation order must be a square power of two, got %r" % (M,))
    levels = 2.0 * np.arange(root) - (root - 1)
    grid = levels.reshape(1, root) + 1j * levels.reshape(root, 1)
    return np.ascontiguousarray(grid.reshape(M), dtype=np.complex128)


def digits_of(k, M: int, n_tx: int) -> np.ndarray:
    """(..., n_tx) per-stream constellation indices of joint hypothesis indices k."""
    k = np.asarray(k, dtype=np.int64)
    shifts = M ** np.arange(n_tx - 1, -1, -1, dtype=np.int64)
    return (k[..., None] // shifts) % M


def symbols_of(k, M: int, n_tx: int) -> np.ndarray:
    """(..., n_tx) complex symbol vectors of joint hypothesis indices k."""
    return constellation(M)[digits_of(k, M, n_tx)]


def bit_labels(M: int) -> np.ndarray:
    """(M, log2 M) uint8 Gray labels of the constellation indices (include/sbce.h, sbce_bit_llr): with
    m = iQ*sqrt(M) + iI and gray(a) = a ^ (a >> 1), the bits of m are gray(iI) MSB first, then gray(iQ) MSB
    first -- [iI, iQ] for QPSK, one bit between adjacent PAM levels on each axis.  The reference's vendored
    QAM.py carries a labelling of its own that no script uses, so no reference output pins this convention."""
    constellation(M)   # validates M
    q = int(round(np.log2(M))) // 2
    sq = 1 << q
    m = np.arange(M)
    gi, gq = (m % sq) ^ ((m % sq) >> 1), (m // sq) ^ ((m // sq) >> 1)
    shifts = np.arange(q - 1, -1, -1)
    bits = np.concatenate([(gi[:, None] >> shifts) & 1, (gq[:, None] >> shifts) & 1], axis=1)
    return np.ascontiguousarray(bits, dtype=np.uint8)


def bits_of(k, M: int, n_tx: int) -> np.ndarray:
    """(..., n_tx, log2 M) uint8 labels of joint hypothesis indices k (the layout of the bit LLRs)."""
    return bit_labels(M)[digits_of(k, M, n_tx)]


def constellation_from_table(all_possibleSymbols, M: int) -> np.ndarray:
    """Recover the per-stream constellation from the reference's (K, n_tx) table."""
    tab = np.asarray(all_possibleSymbols)
    n_tx = tab.shape[1]
    return np.ascontiguousarray(tab[:: M ** (n_tx - 1), 0], dtype=np.complex128)
