"""CPU tests of the bit LLRs with a-priori input: the numpy oracle of tests/llr_apriori_oracle.py against the
plain bit-LLR oracle and against scipy logsumexp over the prior-weighted posterior, and the argument checks of
sbce_bit_llr_apriori (no device needed)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
from scipy.special import logsumexp

import sbce
from oracle import em_numpy as orc

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import llr_apriori_oracle as lao  # noqa: E402
import llr_oracle as lo  # noqa: E402


def _trial(n_tx, n_rx, M, T_d, varn, seed):
    t = orc.gen_trial(3, n_tx, n_rx, M, 4, T_d, varn, seed=seed)
    rng = np.random.default_rng(seed)
    theta = t["h"] + 0.05 * (rng.standard_normal(t["h"].shape) + 1j * rng.standard_normal(t["h"].shape))
    return t["Yd"], t["PsiD"], theta


def _prior(T_d, n_tx, M, seed, scale=8.0):
    return scale * np.random.default_rng(seed).standard_normal((T_d, n_tx, int(np.log2(M))))


def _posterior_extrinsic(Yd, PsiD, theta, M, n_tx, varn, La):
    """Independent: log-likelihood plus the log prior probability of every hypothesis's bits,
    ln P(b = 0) = -ln(1 + e^-La), ln P(b = 1) = -ln(1 + e^La); scipy logsumexp over each side; minus La."""
    La = np.clip(La, -32, 32)
    cons = orc.qam_constellation(M)
    table = orc.hypothesis_table(cons, n_tx)
    Heff = orc.effective_channels(PsiD, theta, n_tx)
    res = Yd[:, None, :] - np.einsum("trj,kj->tkr", Heff, table)
    bits = sbce.qam.bits_of(np.arange(M ** n_tx), M, n_tx)          # (K, n_tx, nb)
    lp0, lp1 = -np.logaddexp(0, -La), -np.logaddexp(0, La)         # (T_d, n_tx, nb)
    logprior = np.einsum("kji,tji->tk", 1 - bits, lp0) + np.einsum("kji,tji->tk", bits, lp1)
    logp = -(np.abs(res) ** 2).sum(axis=2) / varn ** 2 + logprior
    out = np.empty((len(Yd), n_tx, bits.shape[2]))
    for j in range(n_tx):
        for i in range(bits.shape[2]):
            one = bits[:, j, i] == 1
            out[:, j, i] = logsumexp(logp[:, ~one], axis=1) - logsumexp(logp[:, one], axis=1) - La[:, j, i]
    return np.clip(out, -32, 32)


@pytest.mark.parametrize("n_tx,n_rx,M,varn", [(1, 2, 16, 0.7), (2, 2, 4, 0.5), (2, 3, 16, 2.0), (3, 3, 4, 0.3)])
def test_zero_prior_is_the_plain_oracle(n_tx, n_rx, M, varn):
    Yd, PsiD, theta = _trial(n_tx, n_rx, M, 5, varn, seed=11 + n_tx)
    cons = orc.qam_constellation(M)
    La = np.zeros((5, n_tx, int(np.log2(M))))
    assert np.array_equal(lao.bit_llr_apriori(Yd, PsiD, theta, cons, n_tx, varn, La),
                          lo.bit_llr(Yd, PsiD, theta, cons, n_tx, varn))
    if n_tx >= 2:
        np.testing.assert_allclose(lao.bit_llr_apriori_split(Yd, PsiD, theta, cons, n_tx, varn, La),
                                   lo.bit_llr_split(Yd, PsiD, theta, cons, n_tx, varn), rtol=0, atol=1e-12)


@pytest.mark.parametrize("n_tx,n_rx,M,varn", [(1, 2, 16, 0.7), (2, 2, 4, 0.5), (2, 3, 16, 2.0), (3, 3, 4, 0.3)])
def test_oracle_matches_logsumexp_over_the_prior_weighted_posterior(n_tx, n_rx, M, varn):
    Yd, PsiD, theta = _trial(n_tx, n_rx, M, 5, varn, seed=7 + n_tx)
    cons = orc.qam_constellation(M)
    La = _prior(5, n_tx, M, seed=3 + n_tx)
    La[0, 0, 0] = 50.0     # beyond the clamp: read as 32
    ref = _posterior_extrinsic(Yd, PsiD, theta, M, n_tx, varn, La)
    np.testing.assert_allclose(lao.bit_llr_apriori(Yd, PsiD, theta, cons, n_tx, varn, La), ref, rtol=0, atol=1e-9)
    if n_tx >= 2:
        np.testing.assert_allclose(lao.bit_llr_apriori_split(Yd, PsiD, theta, cons, n_tx, varn, La), ref, rtol=0,
                                   atol=1e-9)


def test_oracle_nan_prior_marks_only_its_symbol():
    Yd, PsiD, theta = _trial(2, 2, 16, 6, 0.5, seed=5)
    cons = orc.qam_constellation(16)
    La = _prior(6, 2, 16, seed=1)
    clean = lao.bit_llr_apriori(Yd, PsiD, theta, cons, 2, 0.5, La)
    La[3, 1, 2] = np.nan
    bad = lao.bit_llr_apriori(Yd, PsiD, theta, cons, 2, 0.5, La)
    assert np.isnan(bad[3]).all()
    keep = np.arange(6) != 3
    assert np.array_equal(bad[keep], clean[keep])
    assert np.isnan(lao.bit_llr_apriori_split(Yd, PsiD, theta, cons, 2, 0.5, La)[3]).all()


def _cfg(n_tx, n_rx, M, mode, p1=1):
    return sbce.Problem(N=4, n_tx=n_tx, n_rx=n_rx, M=M, T_p=0, T_d=4, itera=1, mode=mode,
                        partition_r=(p1 - 1) * np.log2(M)).cfg(1)


def test_abi_argument_errors_need_no_device():
    lib = sbce._lib.load()
    E_NULL, E_UNSUPPORTED = -1, -3
    dummy = (C.c_double * 4)()
    io = sbce._lib.Io()
    io.Yd = io.PsiD = io.varn = C.addressof(dummy)
    cfg = _cfg(2, 2, 16, "soft")
    f = lib.sbce_bit_llr_apriori
    assert f(None, C.byref(io), dummy, dummy, dummy, dummy, 0, None) == E_NULL
    assert f(C.byref(cfg), None, dummy, dummy, dummy, dummy, 0, None) == E_NULL
    assert f(C.byref(cfg), C.byref(io), None, dummy, dummy, dummy, 0, None) == E_NULL
    assert f(C.byref(cfg), C.byref(io), dummy, None, dummy, dummy, 0, None) == E_NULL      # llr_a is required
    assert f(C.byref(cfg), C.byref(io), dummy, dummy, None, dummy, 0, None) == E_NULL
    for mode in ("pm", "pm_beta", "zf", "mmse"):
        assert f(C.byref(_cfg(2, 2, 16, mode)), C.byref(io), dummy, dummy, dummy, dummy, 0, None) == E_UNSUPPORTED
    for mode in ("soft", "hard"):   # 8x8 16-QAM: 2^32 leaves, beyond the exhaustive tree
        assert f(C.byref(_cfg(8, 8, 16, mode)), C.byref(io), dummy, dummy, dummy, dummy, 0, None) == E_UNSUPPORTED
