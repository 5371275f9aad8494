"""CPU tests of the bit-level layer: Gray labels, the numpy bit-LLR oracle, the argument checks of sbce_bit_llr /
sbce_accumulate_ber (no device needed) and the BER aggregation of the sweep drivers."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
from scipy.special import logsumexp

import sbce
from oracle import em_numpy as orc

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import llr_oracle as lo  # noqa: E402


@pytest.mark.parametrize("M", [4, 16, 64])
def test_labels_are_a_gray_bijection(M):
    lab = sbce.qam.bit_labels(M)
    q = int(np.log2(M)) // 2
    sq = 1 << q
    assert lab.shape == (M, 2 * q) and lab.dtype == np.uint8
    assert len({tuple(r) for r in lab}) == M                      # bijection onto all 2q-bit words
    assert np.array_equal(lab, lo.bit_labels(M))
    grid = lab.reshape(sq, sq, 2 * q)                             # [iQ][iI]
    # adjacent in-phase levels differ in exactly one in-phase bit, and never in a quadrature bit; and vice versa
    dI = np.abs(np.diff(grid.astype(int), axis=1))
    assert (dI[..., :q].sum(axis=-1) == 1).all() and (dI[..., q:] == 0).all()
    dQ = np.abs(np.diff(grid.astype(int), axis=0))
    assert (dQ[..., q:].sum(axis=-1) == 1).all() and (dQ[..., :q] == 0).all()
    k = np.arange(M ** 2)
    assert np.array_equal(sbce.qam.bits_of(k, M, 2), lab[sbce.qam.digits_of(k, M, 2)])


def test_qpsk_labels_are_iI_iQ():
    cons = sbce.qam.constellation(4)
    lab = sbce.qam.bit_labels(4)
    for m in range(4):
        assert lab[m, 0] == (cons[m].real > 0) and lab[m, 1] == (cons[m].imag > 0)   # bit 0 <-> level -1


def _trial(n_tx, n_rx, M, T_d, varn, seed):
    t = orc.gen_trial(3, n_tx, n_rx, M, 4, T_d, varn, seed=seed)
    rng = np.random.default_rng(seed)
    theta = t["h"] + 0.05 * (rng.standard_normal(t["h"].shape) + 1j * rng.standard_normal(t["h"].shape))
    return t["Yd"], t["PsiD"], theta


def _posterior_llr(Yd, PsiD, theta, M, n_tx, varn, Xoff=None):
    """Independent: log-posterior of every hypothesis, scipy logsumexp over each side of each bit."""
    cons = orc.qam_constellation(M)
    table = orc.hypothesis_table(cons, n_tx)
    Heff = orc.effective_channels(PsiD, theta, n_tx)
    X = table[None] if Xoff is None else table[None] + Xoff[:, None, :]
    res = Yd[:, None, :] - np.einsum("trj,tkj->tkr", Heff, np.broadcast_to(X, (len(Yd),) + table.shape))
    logp = -(np.abs(res) ** 2).sum(axis=2) / varn ** 2
    bits = sbce.qam.bits_of(np.arange(M ** n_tx), M, n_tx)          # (K, n_tx, nb)
    out = np.empty((len(Yd), n_tx, bits.shape[2]))
    for j in range(n_tx):
        for i in range(bits.shape[2]):
            one = bits[:, j, i] == 1
            out[:, j, i] = logsumexp(logp[:, ~one], axis=1) - logsumexp(logp[:, one], axis=1)
    return np.clip(out, -32, 32)


@pytest.mark.parametrize("n_tx,n_rx,M,varn", [(1, 2, 16, 0.7), (2, 2, 4, 0.5), (2, 3, 16, 2.0), (3, 3, 4, 0.3)])
def test_oracle_matches_logsumexp_over_the_posterior(n_tx, n_rx, M, varn):
    Yd, PsiD, theta = _trial(n_tx, n_rx, M, 5, varn, seed=7 + n_tx)
    cons = orc.qam_constellation(M)
    ref = _posterior_llr(Yd, PsiD, theta, M, n_tx, varn)
    np.testing.assert_allclose(lo.bit_llr(Yd, PsiD, theta, cons, n_tx, varn), ref, rtol=0, atol=1e-9)
    if n_tx >= 2:
        np.testing.assert_allclose(lo.bit_llr_split(Yd, PsiD, theta, cons, n_tx, varn), ref, rtol=0, atol=1e-9)
    Xoff = cons[np.random.default_rng(1).integers(0, M, (5, n_tx))]
    ref = _posterior_llr(Yd, PsiD, theta, M, n_tx, varn, Xoff)
    np.testing.assert_allclose(lo.bit_llr(Yd, PsiD, theta, cons, n_tx, varn, Xoff=Xoff), ref, rtol=0, atol=1e-9)


def test_oracle_clamps_and_propagates_nan():
    Yd, PsiD, theta = _trial(2, 2, 16, 6, 0.05, seed=3)
    cons = orc.qam_constellation(16)
    llr = lo.bit_llr(Yd, PsiD, theta, cons, 2, 0.05)
    assert np.abs(llr).max() == 32.0 and (np.abs(llr) == 32.0).mean() > 0.5    # peaked: most bits clamp
    Yd[2, 1] = np.nan
    bad = lo.bit_llr(Yd, PsiD, theta, cons, 2, 0.05)
    assert np.isnan(bad[2]).all()
    keep = np.arange(6) != 2
    assert np.array_equal(bad[keep], llr[keep])
    assert np.isnan(lo.bit_llr_split(Yd, PsiD, theta, cons, 2, 0.05)[2]).all()


def _cfg(n_tx, n_rx, M, mode, p1=1):
    return sbce.Problem(N=4, n_tx=n_tx, n_rx=n_rx, M=M, T_p=0, T_d=4, itera=1, mode=mode,
                        partition_r=(p1 - 1) * np.log2(M)).cfg(1)


def test_abi_argument_errors_need_no_device():
    lib = sbce._lib.load()
    E_NULL, E_UNSUPPORTED = -1, -3
    io = sbce._lib.Io()
    cfg = _cfg(2, 2, 16, "soft")
    assert lib.sbce_bit_llr(None, C.byref(io), None, None, None, 0, None) == E_NULL
    assert lib.sbce_bit_llr(C.byref(cfg), None, None, None, None, 0, None) == E_NULL
    assert lib.sbce_bit_llr(C.byref(cfg), C.byref(io), None, None, None, 0, None) == E_NULL
    for mode in ("pm", "pm_beta", "zf", "mmse"):
        assert lib.sbce_bit_llr(C.byref(_cfg(2, 2, 16, mode)), C.byref(io), None, None, None, 0, None) == E_UNSUPPORTED
    assert lib.sbce_bit_llr(C.byref(_cfg(8, 8, 16, "soft")), C.byref(io), None, None, None, 0, None) == E_UNSUPPORTED
    assert lib.sbce_bit_llr(C.byref(_cfg(8, 8, 16, "hard")), C.byref(io), None, None, None, 0, None) == E_UNSUPPORTED

    dummy = (C.c_double * 4)()
    assert lib.sbce_accumulate_ber(None, dummy, dummy, 1, dummy, None) == E_NULL
    assert lib.sbce_accumulate_ber(C.byref(cfg), None, dummy, 1, dummy, None) == E_NULL
    assert lib.sbce_accumulate_ber(C.byref(cfg), dummy, None, 1, dummy, None) == E_NULL
    assert lib.sbce_accumulate_ber(C.byref(cfg), dummy, dummy, 1, None, None) == E_NULL
    # 8x8 16-QAM: 32-bit joint indices, beyond the int32 decisions (the pointers are never dereferenced)
    assert lib.sbce_accumulate_ber(C.byref(_cfg(8, 8, 16, "zf")), dummy, dummy, 1, dummy, None) == E_UNSUPPORTED


def test_finish_aggregates_ber_and_reports_nan_without_bits():
    from sbce.drivers import PointResult, _finish

    a = PointResult(nmse_sum=0.6, n_valid=3.0, n_flagged=1.0, sym_err=5.0, sym_total=50.0, ser_coded_sum=0.9, n_trials=4.0,
                    bit_err=7.0, bit_total=100.0)
    b = PointResult(nmse_sum=0.2, n_valid=4.0, n_flagged=0.0, n_trials=4.0)
    out = _finish([10, 20], [a, b], device=None)
    assert out["ber"][0] == 0.07 and np.isnan(out["ber"][1])
    # the existing keys and values are those of a run without bit counts
    a0 = PointResult(nmse_sum=0.6, n_valid=3.0, n_flagged=1.0, sym_err=5.0, sym_total=50.0, ser_coded_sum=0.9, n_trials=4.0)
    ref = _finish([10, 20], [a0, b], device=None)
    assert set(out) == {"x", "nmse", "n_valid", "n_flagged", "ser", "ser_as_coded", "n_trials", "ber"}
    for k in set(ref) - {"ber"}:
        np.testing.assert_array_equal(out[k], ref[k])
    assert a.vec()[:7].tolist() == a0.vec()[:7].tolist()
