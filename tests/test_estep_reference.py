"""The E-step reference (tests/estep_reference.py) is itself right: the FP64 oracle meets its bound on every case
the GPU tests use, perturbations of the size a subtly wrong kernel would make do not, the split and unsplit
references agree, and the GPU case list reaches every effective-channel and k_enum variant."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import estep_reference as er  # noqa: E402
from test_gpu_batches import enum_instantiated, enum_variant, heff_variant, SQM  # noqa: E402
from test_gpu_estep_accuracy import CASES, VARNS, inputs  # noqa: E402

from oracle import em_numpy as orc  # noqa: E402


def _oracle(Yd, PsiD, theta, cons, n_tx, varn, Xoff, hard):
    if Xoff is not None:   # superimposed offsets: the hypotheses are x + o, i.e. y' = y - Heff o
        Yd = Yd - np.einsum("trj,tj->tr", orc.effective_channels(PsiD, theta, n_tx), Xoff)
    fn = orc.posterior_stats if len(cons) ** n_tx <= (1 << 18) else orc.posterior_stats_split
    m, R, ks, lse = fn(Yd, PsiD, theta, cons, n_tx, varn, hard=hard)
    if Xoff is not None:
        m, R = er.superimpose(m, R, Xoff)
    return m, R, ks, lse


@pytest.mark.parametrize("case", CASES, ids=lambda c: "x".join(map(str, c)))
def test_oracle_meets_the_bound_on_every_gpu_case(case):
    """posterior_stats / posterior_stats_split within tau of the exact statistics, kstar by the gap rule, at every
    varn of the sweep (trees of 2^16 leaves or more at its ends and middle, the 2^24-leaf trees at varn = 1: the
    references take seconds per symbol there)."""
    Yd, PsiD, theta, Xoff = inputs(case)
    n_tx, M = case[1], case[3]
    cons = orc.qam_constellation(M)
    K = M ** n_tx
    varns = list(VARNS) if K < (1 << 16) else [1e-3, 1.0, 100.0] if K < (1 << 24) else [1.0]
    worst = 0.0
    for b in range(Yd.shape[0]):
        xo = None if Xoff is None else Xoff[b]
        refs = er.reference(Yd[b], PsiD[b], theta[b], cons, n_tx, varns, xo)
        for varn, ref in zip(varns, refs):
            m, R, ks, lse = _oracle(Yd[b], PsiD[b], theta[b], cons, n_tx, varn, xo, False)
            assert not er.kstar_bad(ref, ks)
            r, adm = er.ratios(ref, m, R, lse, False)
            assert adm == len(ks), (varn, adm)
            assert r <= 1.0, (varn, r)
            worst = max(worst, r)
    print("largest error/tau of the FP64 oracle on %s: %.3e" % (case, worst))


def _small():
    Yd, PsiD, theta, _ = inputs((8, 2, 2, 16, 7))
    return Yd[1], PsiD[1], theta[1], orc.qam_constellation(16), 2


@pytest.mark.parametrize("varn", [0.7, 3.3, 10.1])
def test_perturbations_fail_the_bound(varn):
    """Errors a subtly wrong kernel would make exceed tau: one hypothesis' d2 rounded to float32, and the exponent
    formed with varn^2 rounded to float32.  The unperturbed statistics meet it."""
    Yd, PsiD, theta, cons, n_tx = _small()
    ref = er.exact_stats(Yd, PsiD, theta, cons, n_tx, varn)
    H = orc.effective_channels(er._ld(PsiD), er._ld(theta), n_tx)
    X = orc.hypothesis_table(cons, n_tx)
    r = er._ld(Yd)[:, None, :] - np.einsum("trj,kj->tkr", H, er._ld(X))
    d2 = np.sum(r.real ** 2 + r.imag ** 2, axis=2)
    exact = er.stats_from_d2(d2, X, varn, ref.rho)
    assert er.ratios(ref, exact.m, exact.R, exact.lse, False)[0] <= 1e-3

    # d2 of the runner-up of every symbol rounded to float32
    d2f = d2.copy()
    for t in range(len(d2f)):
        d2f[t, ref.k2[t]] = np.float32(d2f[t, ref.k2[t]])
    bad = er.stats_from_d2(d2f, X, varn, ref.rho)
    assert er.ratios(ref, bad.m, bad.R, bad.lse, False)[0] > 1.0

    # varn^2 rounded to float32 in the exponent
    v32 = np.sqrt(np.longdouble(np.float32(np.float64(varn) ** 2)))
    bad = er.stats_from_d2(d2, X, v32, ref.rho)
    assert er.ratios(ref, bad.m, bad.R, bad.lse, False)[0] > 1.0


def test_perturbed_kstar_fails_the_gap_rule():
    """Any hypothesis but k* fails where the gap is resolvable; the runner-up passes where it is not."""
    Yd, PsiD, theta, cons, n_tx = _small()
    ref = er.exact_stats(Yd, PsiD, theta, cons, n_tx, 0.3)
    assert not er.kstar_bad(ref, ref.kstar)
    assert np.all(ref.gap > 2 * np.maximum(ref.eps_star, ref.eps2))
    assert len(er.kstar_bad(ref, ref.k2)) == len(ref.k2)
    ref.gap[:] = 0.0
    ref.d2star[:] = [er.d2_at(ref, t, k) - er.eps_at(ref, t, k) for t, k in enumerate(ref.k2)]
    assert not er.kstar_bad(ref, ref.k2)


@pytest.mark.parametrize("shape", [(5, 2, 3, 16, 2), (4, 3, 4, 4, 2), (4, 4, 4, 4, 1)])
def test_split_and_unsplit_references_agree(shape):
    N, n_tx, n_rx, M, T_d = shape
    Yd, PsiD, theta, _ = inputs(shape)
    cons = orc.qam_constellation(M)
    rng = np.random.default_rng(1)
    Xoff = cons[rng.integers(0, M, (T_d, n_tx))]
    for xo in (None, Xoff):
        a = er.exact_stats(Yd[1], PsiD[1], theta[1], cons, n_tx, [0.05, 2.0], xo)
        b = er.exact_stats_split(Yd[1], PsiD[1], theta[1], cons, n_tx, [0.05, 2.0], xo, rows=3)
        for x, y in zip(a, b):
            for name in ("m", "R", "lse", "lnZ", "d2star", "gap", "dbeta", "lse_lin", "eps_star", "eps2"):
                u, v = getattr(x, name), getattr(y, name)
                assert np.all(np.abs(u - v) <= 1e-15 * (1 + np.abs(u))), name
            for name in ("kstar", "k2", "n_win"):
                assert np.array_equal(getattr(x, name), getattr(y, name)), name


def test_accuracy_cases_reach_every_variant():
    """The sweep of tests/test_gpu_estep_accuracy.py reaches every effective-channel branch (the tensor path with
    1..4 column tiles and ragged K among them), every k_enum instantiation, both 2^24-leaf trees, odd T_d and
    superimposed offsets."""
    heff = {heff_variant(*c[:3])[1] for c in CASES}
    assert heff == {"smem", "global", "mma", "rows"}
    mma = [c for c in CASES if heff_variant(*c[:3])[1] == "mma"]
    assert {(c[1] * c[2] + 7) // 8 for c in mma} == {1, 2, 3, 4}
    assert any((c[0] + 1) % 8 for c in mma)
    want = {enum_variant(n, M, h) for n in range(1, 9) for M in (4, 16, 64) for h in (False, True)
            if enum_instantiated(n, SQM[M])}
    assert {enum_variant(c[1], c[3], h) for c in CASES for h in (False, True)} == want
    assert {(c[1], c[3]) for c in CASES if c[3] ** c[1] == 1 << 24} == {(4, 64), (6, 16)}
    assert any(c[4] % 2 for c in CASES if c[1] <= 4)
    assert any("sup" in c for c in CASES)
