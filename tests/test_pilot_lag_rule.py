"""The lag rule of the pilot normal equations (include/sbce.h, "Pilot normal equations") in numpy: which pilot
designs qualify, and that the block-Toeplitz pilot Gram built from the lag table matches the pair formula within
the documented bound at the shapes of the benchmark workloads."""
import re

import numpy as np
import pytest

import sbce

U = 2.0 ** -53
HEADER = open(__import__("os").path.join(__import__("os").path.dirname(__file__), "..", "include", "sbce.h")).read()
TOL_ULPS = int(re.search(r"#define SBCE_PILOT_LAG_TOL_ULPS (\d+)", HEADER).group(1))


def tol(N1):
    return TOL_ULPS * N1 * U


def lag_index(N1, s):
    n, m = np.tril_indices(N1)
    return n, m, np.where((m == 0) & (s == 1), n, n - m + s)


def qualifying_shift(P):
    """The shift the device check picks (1 preferred), None when the design keeps the pair form."""
    N1 = P.shape[1]
    ok = {}
    for s in (0, 1):
        n, m, lag = lag_index(N1, s)
        with np.errstate(invalid="ignore", over="ignore"):
            err = np.abs(np.conj(P[:, n]) * P[:, m] - np.conj(P[:, lag]))
            ok[s] = bool(np.all(err <= tol(N1) * np.abs(P[:, lag])))     # NaN compares false
    return 1 if ok[1] else (0 if ok[0] else None)


def device_top_design(T_p, N, shift=1):
    """The design of sbce_generate_batch (SBCE_PILOTS_TOP): argument reduced exactly in integers, then the phase
    (numpy's cos / sin of pi x stand in for sincospi)."""
    t = np.arange(T_p)[:, None]
    k = np.arange(N + 1 - shift)[None, :]
    x = -2.0 * ((t * k) % T_p) / T_p
    P = np.ones((T_p, N + 1), dtype=np.complex128)
    P[:, shift:] = np.cos(np.pi * x) + 1j * np.sin(np.pi * x)
    return P


SHAPES = sorted({(w.T_p, w.N) for w in sbce.workloads.WORKLOADS.values()})


@pytest.mark.parametrize("T_p,N", SHAPES)
def test_device_designs_qualify_with_their_shift(T_p, N):
    assert qualifying_shift(device_top_design(T_p, N, 1)) == 1
    assert qualifying_shift(device_top_design(T_p, N, 0)) == 0   # no direct link: all columns are DFT columns


@pytest.mark.parametrize("T_p,N", [(320, 64), (40, 16), (320, 256)])
def test_numpy_designs_qualify(T_p, N):
    # the reference's construction: exp(-2j pi t n / T_p) from the unreduced argument, off by O(N) ulp
    assert qualifying_shift(sbce.signal_model.pilot_phases(T_p, N, "top")) == 1


@pytest.mark.parametrize("T_p,N,numpy_made", [(320, 64, False), (40, 16, False), (320, 64, True)])
def test_lag_gram_matches_pair_gram_within_the_bound(T_p, N, numpy_made):
    rng = np.random.default_rng(7)
    n_tx = 4
    P = sbce.signal_model.pilot_phases(T_p, N, "top") if numpy_made else device_top_design(T_p, N)
    x = (rng.integers(0, 4, (T_p, n_tx)) * 2 - 3) + 1j * (rng.integers(0, 4, (T_p, n_tx)) * 2 - 3)
    R = np.conj(x)[:, :, None] * x[:, None, :]
    N1 = N + 1
    F = np.einsum("tl,tij->lij", np.conj(P), R)
    n, m, lag = lag_index(N1, 1)
    pair = np.einsum("tp,tij->pij", np.conj(P[:, n]) * P[:, m], R)
    bound = (tol(N1) + 4 * T_p * U) * np.abs(R).sum(axis=0)   # rule + both sums' rounding
    assert np.all(np.abs(pair - F[lag]) <= bound[None])


def test_perturbation_nan_and_per_trial_designs_fail():
    P = device_top_design(320, 64)
    assert qualifying_shift(P) == 1
    Q = P.copy()
    Q[17, 5] += 2 * tol(65)                 # above the bound
    assert qualifying_shift(Q) is None
    assert qualifying_shift(2.0 ** -50 * P) is None    # the bound is relative: no other modulus passes
    assert qualifying_shift(2.0 * P) is None
    Q = P.copy()
    Q[3, 9] = np.nan
    assert qualifying_shift(Q) is None
    Q = P.copy()
    Q[0, 2] = np.inf
    assert qualifying_shift(Q) is None
    rs = np.random.RandomState(3)
    assert qualifying_shift(sbce.signal_model.data_phases_random(320, 64, rs)) is None


