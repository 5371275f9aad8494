"""The M-step's pivot threshold at its boundary, mixed batches of flagged and good trials, and invariance under
power-of-two scaling.

The Cholesky of k_chol_solve (csrc/chol.cu) flags a trial with SBCE_ST_NOT_PD when a pivot is not above 1e-13
times the largest pivot so far in that trial (a NaN pivot included); the identity padding of the matrix up to a
multiple of 8 is exempt.  The designs below have known pivots: with the pilot symbols zero the pilot Gram is
exactly 0, and data symbol t = (n, i) has psi_t = row n of a unit upper-triangular Gaussian-integer V and the
statistic R_t = d[n n_tx + i] e_i e_i^T, so that G = (V (x) I)^H diag(d) (V (x) I) and its pivots are exactly d.
With V = I the device computes them exactly too, so a ratio of 2^-43 (1.14e-13) must pass and 2^-44 (5.7e-14)
must be flagged."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mstep_reference as mr  # noqa: E402

pytestmark = pytest.mark.gpu

NOT_PD = 1
# n_tx -> N + 1: L = 45, 44, 42 (not multiples of 16, so padding rows follow the last pivot) on the scalar Gram
# (n_tx = 1), the TMA Gram (n_tx = 4) and the generic tensor-path Gram (n_tx = 6)
N1_OF = {1: 45, 4: 11, 6: 7}
N_RX = 2


@pytest.fixture(scope="module")
def S(cuda_device):
    import sbce

    sbce._lib.require_device()
    return sbce


def pivot_design(rng, N1, n_tx, d, V=None):
    """One trial of the known-pivot design: inputs of DeviceSession.mstep (T_p = 1, T_d = L)."""
    L = N1 * n_tx
    V = np.eye(N1, dtype=np.complex128) if V is None else V
    n, i = np.divmod(np.arange(L), n_tx)
    R = np.zeros((L, n_tx, n_tx), np.complex128)
    R[np.arange(L), i, i] = d
    m = np.zeros((L, n_tx), np.complex128)
    m[np.arange(L), i] = 1.0
    return dict(PsiD=V[n], Yd=mr._gi(rng, (L, N_RX), 3), m=m, R=R, PsiP=np.ones((1, N1), np.complex128),
                Yp=np.zeros((1, N_RX), np.complex128), Xp=np.zeros((1, n_tx), np.complex128))


def run(S, n_tx, trials):
    """M-step of a batch of trials (dicts as pivot_design) -> theta, status (numpy)."""
    import torch

    N1 = trials[0]["PsiD"].shape[1]
    T_p, T_d = trials[0]["PsiP"].shape[0], trials[0]["PsiD"].shape[0]
    prob = S.Problem(N=N1 - 1, n_tx=n_tx, n_rx=N_RX, M=4, T_p=T_p, T_d=T_d, itera=1)
    ses = S.DeviceSession(prob, len(trials))
    t = lambda k: torch.from_numpy(np.ascontiguousarray(np.stack([tr[k] for tr in trials]))).to(ses.device)
    theta, status = ses.mstep(t("Yd"), t("Yp"), t("PsiD"), t("PsiP"), t("Xp"), t("m"), t("R"))
    torch.cuda.synchronize()
    return theta.cpu().numpy(), status.cpu().numpy()


def eta(tr, theta):
    G, B = mr.system(tr["PsiP"], tr["Yp"], tr["Xp"], tr["PsiD"], tr["Yd"], tr["m"], tr["R"])
    return mr.backward_error(G, B, theta)


POSITIONS = [1, 15, 16, 17, 31, 32, -1]


@pytest.mark.parametrize("n_tx", [1, 4, 6])
@pytest.mark.parametrize("log2_ratio, flagged", [(-43, False), (-44, True)])
def test_pivot_threshold_boundary(S, n_tx, log2_ratio, flagged):
    """One pivot 2^-43 / 2^-44 among ones, at panel starts and ends and at the last row before the padding."""
    N1 = N1_OF[n_tx]
    L = N1 * n_tx
    rng = np.random.default_rng(n_tx)
    trials = []
    for p in POSITIONS:
        d = np.ones(L)
        d[p] = 2.0 ** log2_ratio
        trials.append(pivot_design(rng, N1, n_tx, d))
    theta, status = run(S, n_tx, trials)
    assert status.tolist() == [NOT_PD if flagged else 0] * len(POSITIONS), (L, status)
    if not flagged:
        for b, tr in enumerate(trials):
            assert eta(tr, theta[b]) <= mr.tau(L)


@pytest.mark.parametrize("n_tx", [1, 4, 6])
def test_pivot_threshold_uses_the_largest_pivot_of_earlier_panels(S, n_tx):
    """Pivot 2^20 at position 0 (panel 0) and 2^-24 / 2^-23 at position 40 (panel 2): ratios 2^-44 / 2^-43."""
    N1 = N1_OF[n_tx]
    L = N1 * n_tx
    rng = np.random.default_rng(10 + n_tx)
    trials = []
    for small in (2.0 ** -24, 2.0 ** -23):
        d = np.ones(L)
        d[0], d[40] = 2.0 ** 20, small
        trials.append(pivot_design(rng, N1, n_tx, d))
    theta, status = run(S, n_tx, trials)
    assert status.tolist() == [NOT_PD, 0]
    assert eta(trials[1], theta[1]) <= mr.tau(L)


def test_pivot_threshold_compares_with_earlier_pivots_only(S):
    """Tiny pivots before large ones are not flagged (the rule looks at the largest pivot SO FAR): 2^-50 at
    positions 0..19, across the first panel boundary, then ones; and 2^-60 at position 0 only."""
    n_tx, N1 = 4, N1_OF[4]
    L = N1 * n_tx
    rng = np.random.default_rng(3)
    d0, d1 = np.ones(L), np.ones(L)
    d0[:20] = 2.0 ** -50
    d1[0] = 2.0 ** -60
    trials = [pivot_design(rng, N1, n_tx, d0), pivot_design(rng, N1, n_tx, d1)]
    theta, status = run(S, n_tx, trials)
    assert status.tolist() == [0, 0]
    for b, tr in enumerate(trials):
        assert eta(tr, theta[b]) <= mr.tau(L)


def test_uniform_tiny_pivots_with_padding(S):
    """All pivots 2^-60 at L = 17 (seven identity padding rows up to 24): not flagged, the padding's unit pivots
    come after every live one and never count against them; the solve is backward stable at that scale."""
    N1, n_tx = 17, 1
    tr = pivot_design(np.random.default_rng(4), N1, n_tx, np.full(N1, 2.0 ** -60))
    theta, status = run(S, n_tx, [tr])
    assert status.tolist() == [0]
    assert eta(tr, theta[0]) <= mr.tau(N1)


def test_pivot_threshold_with_rounding_factorisation(S):
    """V = I + a Gaussian-integer superdiagonal (the factorisation now rounds): a pivot 2^-36 (1.5e-11) of the
    largest passes with a backward-stable solve, 2^-50 (8.9e-16) is flagged; at positions 17 and 40."""
    n_tx, N1 = 4, N1_OF[4]
    L = N1 * n_tx
    rng = np.random.default_rng(5)
    V = np.eye(N1, dtype=np.complex128)
    V[np.arange(N1 - 1), np.arange(1, N1)] = mr._gi(rng, N1 - 1, 1) + 1
    trials = []
    for small in (2.0 ** -36, 2.0 ** -50):
        for p in (17, 40):
            d = np.ones(L)
            d[p] = small
            trials.append(pivot_design(rng, N1, n_tx, d, V))
    theta, status = run(S, n_tx, trials)
    assert status.tolist() == [0, 0, NOT_PD, NOT_PD]
    for b in (0, 1):
        assert eta(trials[b], theta[b]) <= mr.tau(L)


def test_mixed_batch_flags_only_the_bad_trials(S):
    """A flagged trial (pivot ratio 2^-44) and one with a NaN statistic among good ones: each bad trial gets
    SBCE_ST_NOT_PD (a NaN pivot is not above the threshold), the good trials have status 0 and are bitwise equal to
    the same trials solved without the bad ones."""
    n_tx, N1 = 4, N1_OF[4]
    L = N1 * n_tx
    rng = np.random.default_rng(6)
    inp = mr.integer_inputs(rng, 2, N1, n_tx, N_RX, 1, L)
    good = [{k: inp[k][b] for k in ("PsiP", "PsiD", "Xp", "Yp", "Yd", "m", "R")} for b in range(2)]
    d = np.ones(L)
    d[17] = 2.0 ** -44
    flagged = pivot_design(rng, N1, n_tx, d)
    flagged["PsiP"] = good[0]["PsiP"].copy()      # the pilot Gram stays 0: Xp = 0
    nan = {k: v.copy() for k, v in good[1].items()}
    nan["R"][5, 1, 1] = np.nan
    theta, status = run(S, n_tx, [good[0], flagged, nan, good[1]])
    assert status[[0, 3]].tolist() == [0, 0]
    assert status[1] == NOT_PD and status[2] & NOT_PD, status
    theta_ref, status_ref = run(S, n_tx, good)
    assert status_ref.tolist() == [0, 0]
    assert np.array_equal(theta[[0, 3]], theta_ref)
    for b in range(2):
        assert eta(good[b], theta_ref[b]) <= mr.tau(L)


def test_mstep_is_invariant_under_power_of_two_scaling(S):
    """Statistics, Y and Xp scaled so that G -> 2^(2k) G and B -> 2^(2k) B for 2k = -600 .. 600: theta is
    unchanged (no absolute epsilon in the Gram, the factorisation or the back substitution)."""
    n_tx, N1 = 4, N1_OF[4]
    inp = mr.integer_inputs(np.random.default_rng(7), 1, N1, n_tx, N_RX, 16, 30)
    base = {k: inp[k][0] for k in ("PsiP", "PsiD", "Xp", "Yp", "Yd", "m", "R")}
    ks = (-300, -150, -64, -1, 0, 1, 64, 150, 300)
    trials = []
    for k in ks:
        s = 2.0 ** k
        tr = dict(base, Yd=base["Yd"] * s, Yp=base["Yp"] * s, Xp=base["Xp"] * s, m=base["m"] * s, R=base["R"] * s * s)
        trials.append(tr)
    theta, status = run(S, n_tx, trials)
    assert status.tolist() == [0] * len(ks)
    th0 = theta[ks.index(0)]
    errs = [mr.relerr(theta[j], th0) for j in range(len(ks))]
    assert max(errs) <= 1e-14, errs
    print("power-of-two scaling 2k = %s: bitwise equal to 2k = 0: %s"
          % ([2 * k for k in ks], [bool(np.array_equal(theta[j], th0)) for j in range(len(ks))]))
