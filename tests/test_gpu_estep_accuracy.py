"""E-step accuracy on the device against the extended-precision reference (tests/estep_reference.py): an SNR sweep
over every effective-channel and k_enum variant with the derived bound tau and the kstar gap rule, near ties
resolved down to the bound, exact ties of a stream whose channel column is zero, and bitwise equivariance of the
E-step and the bit LLRs under scaling (Yd, theta, varn) by powers of two."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import estep_reference as er  # noqa: E402

import sbce  # noqa: E402
from oracle import em_numpy as orc  # noqa: E402

pytestmark = pytest.mark.gpu

VARNS = (1e-3, 1e-2, 0.1, 1.0, 10.0, 100.0)

# N, n_tx, n_rx, M, T_d[, "sup"] -- effective-channel variants (test_gpu_batches.heff_variant): per lane with theta
# in shared memory ("smem"), per lane with theta in global memory (N = 256), the DMMA tensor path with 1..4 column
# tiles and ragged K (N + 1 not a multiple of 8), 8-lane rows (n_tx >= 5).  E-step variants: every
# k_enum<NTX, SQM, HARD, 4> instantiation, both 2^24-leaf trees (4 x 64-QAM, 6 x 16-QAM, one symbol), flat
# posteriors at varn >= 10 that overflow the candidate queue, odd T_d (an idle half-warp).  "sup": superimposed
# pilot offsets.  Trial 0 has theta near the truth, trial 1 (where there are two) theta = 0.3 h.
CASES = [
    (8, 1, 4, 4, 9), (8, 1, 2, 16, 7), (15, 1, 8, 64, 37),
    (8, 2, 2, 4, 11, "sup"), (17, 2, 4, 16, 33), (6, 2, 3, 64, 9),
    (20, 3, 4, 4, 40), (5, 3, 4, 16, 10, "sup"), (5, 3, 4, 64, 4),
    (23, 4, 6, 4, 19), (31, 4, 8, 16, 5), (4, 4, 4, 64, 1), (256, 4, 4, 4, 6),
    (6, 5, 5, 4, 9), (4, 5, 6, 16, 3), (5, 6, 6, 4, 7), (3, 6, 6, 16, 1), (5, 7, 8, 4, 6), (6, 8, 8, 4, 5),
]
SCALES = (-300, -150, -1, 1, 150, 300)


def inputs(case, seed=0):
    """(Yd, PsiD, theta, Xoff or None) for a case; theta near the truth for trial 0, far for trial 1."""
    N, n_tx, n_rx, M, T_d = case[:5]
    B = 1 if M ** n_tx > (1 << 18) else 2
    tb = sbce.signal_model.generate_batch(N, n_tx, n_rx, M, 4, T_d, 0.1, B, seed=seed + 17 * N + n_tx, legacy=False)
    rng = np.random.default_rng(seed + 5)
    theta = tb.h + 0.05 * (rng.standard_normal(tb.h.shape) + 1j * rng.standard_normal(tb.h.shape))
    if B > 1:
        theta[1] = 0.3 * tb.h[1]
    Xoff = None
    if "sup" in case:
        cons = orc.qam_constellation(M)
        Xoff = cons[rng.integers(0, M, (B, T_d, n_tx))]
        Xoff[:, T_d // 2:] = 0.0      # zero beyond the pilot length
    return tb.Yd, tb.PsiD, theta, Xoff


def case_id(case):
    return "x".join(str(c) for c in case)


def run_estep(S, case, hard, Yd, PsiD, theta, varn, Xoff=None, full_scan=False):
    import torch

    N, n_tx, n_rx, M, T_d = case[:5]
    B = Yd.shape[0]
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=0 if Xoff is not None else 4, T_d=T_d, itera=1,
                     mode="hard" if hard else "soft", superimposed=Xoff is not None, full_scan=full_scan)
    ses = S.DeviceSession(prob, B)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    vn = t(np.broadcast_to(np.asarray(varn, dtype=np.float64), (B,)))
    out = ses.estep(t(Yd), t(PsiD), t(theta), vn, Xp=None if Xoff is None else t(Xoff))
    torch.cuda.synchronize()
    return [o.cpu().numpy() for o in out]


def run_llr(S, case, hard, Yd, PsiD, theta, varn, Xoff=None, La=None):
    import torch

    N, n_tx, n_rx, M, T_d = case[:5]
    B = Yd.shape[0]
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=0 if Xoff is not None else 4, T_d=T_d, itera=1,
                     mode="hard" if hard else "soft", superimposed=Xoff is not None)
    ses = S.DeviceSession(prob, B)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    vn = t(np.broadcast_to(np.asarray(varn, dtype=np.float64), (B,)))
    out = ses.bit_llr(t(Yd), t(PsiD), t(theta), vn, Xp=None if Xoff is None else t(Xoff),
                      llr_a=None if La is None else t(La))
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.fixture(scope="module")
def S(cuda_device):
    sbce._lib.require_device()
    return sbce


_REFS = {}


def references(case):
    """Per trial, the references at every varn of the sweep (cached: soft and hard share them)."""
    if case not in _REFS:
        Yd, PsiD, theta, Xoff = inputs(case)
        cons = orc.qam_constellation(case[3])
        _REFS[case] = [er.reference(Yd[b], PsiD[b], theta[b], cons, case[1], list(VARNS),
                                    None if Xoff is None else Xoff[b]) for b in range(Yd.shape[0])]
    return _REFS[case]


def variant_label(case, hard):
    from test_gpu_batches import enum_variant, heff_variant

    N, n_tx, n_rx, M = case[:4]
    return "%s %s%s" % (heff_variant(N, n_tx, n_rx)[1], enum_variant(n_tx, M, hard), " sup" if "sup" in case else "")


# ---------------------------------------------------------------------------
# SNR sweep
# ---------------------------------------------------------------------------

@pytest.mark.parametrize("hard", [False, True], ids=["soft", "hard"])
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_estep_within_bound_across_snr(S, case, hard):
    """m, R and lse within tau of the exact statistics, kstar by the gap rule, at varn = 1e-3 .. 100."""
    Yd, PsiD, theta, Xoff = inputs(case)
    refs = references(case)
    label = variant_label(case, hard)
    for i, varn in enumerate(VARNS):
        m, R, ks, ls = run_estep(S, case, hard, Yd, PsiD, theta, varn, Xoff)
        worst, adm, total = 0.0, 0, 0
        for b in range(Yd.shape[0]):
            ref = refs[b][i]
            assert not er.kstar_bad(ref, ks[b]), (varn, b, er.kstar_bad(ref, ks[b])[:4])
            r, a = er.ratios(ref, m[b], R[b], ls[b], hard, ks[b])
            worst, adm, total = max(worst, r), adm + a, total + Yd.shape[1]
        print("ESTEP_RATIO %s | varn %g | %.3e | admitted %d/%d" % (label, varn, worst, adm, total))
        assert adm >= (total + 1) // 2, "too few symbols admitted to the first-order bound"
        assert worst <= 1.0, (label, varn, worst)


# ---------------------------------------------------------------------------
# near ties
# ---------------------------------------------------------------------------

def _tie_symbols(H, cons, M, n_tx, streams, factor, rng, eps_of):
    """One received vector per stream j in `streams`: on the bisector of Heff x_a and Heff x_b (x_b = x_a with
    stream j one PAM level over), moved towards x_a so that the exact gap is factor * 2 max(eps_a, eps_b).  x_a is
    drawn until every other hypothesis is clearly farther than x_b (FP64 distances)."""
    sq = int(round(np.sqrt(M)))
    X = orc.hypothesis_table(cons, n_tx) if M ** n_tx <= (1 << 16) else \
        cons[orc.hypothesis_digits(np.arange(M ** n_tx), M, n_tx)]
    Y, pairs = [], []
    for t, j in enumerate(streams):
        for _ in range(200):
            da = rng.integers(0, M, n_tx)
            db = da.copy()
            db[j] = da[j] + (1 if da[j] % sq < sq - 1 else -1)
            xa, xb = cons[da], cons[db]
            D = H[t] @ (xa - xb)
            nD = np.linalg.norm(D)
            mid = H[t] @ (xa + xb) / 2
            y = mid + factor * eps_of(t, mid, nD / 2) / nD * D / nD
            ka = int(sum(int(da[i]) * M ** (n_tx - 1 - i) for i in range(n_tx)))
            kb = int(sum(int(db[i]) * M ** (n_tx - 1 - i) for i in range(n_tx)))
            r = y[None, :] - X @ H[t].T
            d2 = (r.real ** 2 + r.imag ** 2).sum(axis=1)
            d2[[ka, kb]] = np.inf
            if d2.min() > 1.1 * nD * nD / 4:
                break
        else:
            raise AssertionError("no isolated pair found")
        Y.append(y)
        pairs.append((ka, kb))
    return np.array(Y), pairs


TIE_SHAPES = [(8, 2, 4, 16), (6, 3, 4, 64), (6, 4, 8, 16), (5, 6, 8, 4)]


@pytest.mark.parametrize("hard", [False, True], ids=["soft", "hard"])
@pytest.mark.parametrize("shape", TIE_SHAPES, ids=case_id)
def test_near_ties_are_resolved_down_to_the_bound(S, shape, hard):
    """y on the bisector of two hypotheses that differ in stream 0 (closed-form leaves), a middle stream or stream
    n_tx - 1 (a lane-split prefix), offset so that the exact gap is 1000, 10 and 0.5 times 2 eps: the device must
    pick k* whenever the gap is above 2 eps, and a hypothesis within eps of the minimum otherwise."""
    N, n_tx, n_rx, M = shape
    cons = orc.qam_constellation(M)
    streams = sorted({0, n_tx // 2, n_tx - 1})
    rng = np.random.default_rng(N * n_tx + M)
    tb = sbce.signal_model.generate_batch(N, n_tx, n_rx, M, 4, len(streams), 0.1, 1, seed=5, legacy=False)
    theta, PsiD = tb.h[:1], tb.PsiD[:1]
    H = orc.effective_channels(PsiD[0], theta[0], n_tx)
    for factor in (1000.0, 10.0, 0.5):
        def eps_of(t, mid, r):
            # the module's rho_t at y = mid (it depends on ||y|| only weakly), eps at residual norm r
            rt = er.residual_error(mid[None, :], PsiD[0][t:t + 1], theta[0], n_tx, cons)[0]
            return 2 * r * rt + rt * rt
        Y, pairs = _tie_symbols(H, cons, M, n_tx, streams, factor, rng, eps_of)
        Yd = Y[None]
        case = (N, n_tx, n_rx, M, len(streams))
        varn = 0.3
        ref = er.reference(Yd[0], PsiD[0], theta[0], cons, n_tx, varn)
        m, R, ks, ls = run_estep(S, case, hard, Yd, PsiD, theta, varn)
        for t, (ka, kb) in enumerate(pairs):
            assert int(ref.kstar[t]) == ka, "construction: x_a must be the exact arg-min"
            bound = 2 * max(ref.eps_star[t], er.eps_at(ref, t, kb))
            ratio = float(ref.gap[t] / bound)
            assert 0.25 * factor < ratio < 4 * factor, (factor, ratio)
            print("TIE %s stream %d factor %g gap/2eps %.3g kstar %s" % (case_id(shape), streams[t], factor, ratio,
                                                                         "k*" if ks[0, t] == ka else ks[0, t]))
        assert not er.kstar_bad(ref, ks[0]), (factor, er.kstar_bad(ref, ks[0]))
        if factor > 1:
            assert [int(k) for k in ks[0]] == [a for a, _ in pairs]
        r, _ = er.ratios(ref, m[0], R[0], ls[0], hard, ks[0])
        assert r <= 1.0, (factor, r)


# ---------------------------------------------------------------------------
# exact ties: a stream with a zero channel column
# ---------------------------------------------------------------------------

TIE_CASES = [(8, 2, 2, 16, 7), (5, 3, 4, 64, 4), (23, 4, 6, 4, 9), (31, 4, 8, 16, 5), (6, 6, 6, 4, 5),
             (6, 8, 8, 4, 5)]


@pytest.mark.parametrize("hard", [False, True], ids=["soft", "hard"])
@pytest.mark.parametrize("case", TIE_CASES, ids=case_id)
def test_zero_column_stream_ties_exactly(S, case, hard):
    """Rows n' n_tx + j of theta zero for every n': column j of every Heff_t is exactly zero and the M values of
    stream j tie exactly.  kstar takes digit 0 there (first index, the np.argmax rule) and the reduced problem's
    digits elsewhere; soft: m_j = 0, R_jj = 2 (M - 1) / 3, R_ij = 0, and the other streams' statistics are the
    reduced problem's."""
    N, n_tx, n_rx, M, T_d = case
    cons = orc.qam_constellation(M)
    Yd, PsiD, theta0, _ = inputs(case, seed=9)
    Yd, PsiD, theta0 = Yd[:1], PsiD[:1], theta0[:1]
    for j in sorted({0, n_tx // 2, n_tx - 1}):
        theta = theta0.copy()
        theta[0, j::n_tx] = 0.0
        keep = [i for i in range(n_tx) if i != j]
        th_red = theta[0].reshape(N + 1, n_tx, n_rx)[:, keep].reshape(-1, n_rx)
        varn = 0.3
        m, R, ks, ls = run_estep(S, case, hard, Yd, PsiD, theta, varn)
        m, R, ks, ls = m[0], R[0], ks[0], ls[0]
        assert np.all(np.isfinite(m)) and np.all(np.isfinite(R)) and np.all(np.isfinite(ls))
        full = er.reference(Yd[0], PsiD[0], theta[0], cons, n_tx, varn)
        red = er.reference(Yd[0], PsiD[0], th_red, cons, n_tx - 1, varn)
        dig = orc.hypothesis_digits(ks.astype(np.int64), M, n_tx)
        assert np.all(dig[:, j] == 0), ks
        rdig = orc.hypothesis_digits(red.kstar, M, n_tx - 1)
        for t in range(T_d):
            if red.gap[t] > 2 * max(red.eps_star[t], red.eps2[t]):
                assert np.array_equal(dig[t, keep], rdig[t]), (j, t)
        assert not er.kstar_bad(full, ks)
        r, _ = er.ratios(full, m, R, ls, hard, ks)
        assert r <= 1.0, (j, r)
        if hard:
            continue
        tm, tR, _, adm = er.taus(red)
        rnd = er.C_S * er.U * full.n_win
        xm = full.xmax
        assert np.all(np.abs(m[:, j]) <= xm * rnd)
        assert np.all(np.abs(R[:, j, j] - 2 * (M - 1) / 3) <= xm * xm * rnd)
        off = np.abs(np.delete(R[:, j, :], j, axis=1)).max(axis=1)
        assert np.all(off <= er.taus(full)[1])
        sub = np.ix_(range(T_d), keep, keep)
        em = np.abs((er._ld(m[:, keep]) - red.m).astype(complex)).max(axis=1)
        eR = np.abs((er._ld(R[sub]) - red.R).astype(complex)).max(axis=(1, 2))
        # the full problem's window holds M times the reduced problem's hypotheses
        assert np.all((em <= tm + xm * rnd)[adm]) and np.all((eR <= tR + xm * xm * rnd)[adm]), (j, em, eR)


# ---------------------------------------------------------------------------
# scale equivariance
# ---------------------------------------------------------------------------

def _assert_normal_range(Yd, PsiD, theta, varn, n_tx, cons, k, Xoff):
    """Every squared distance, varn^2 and 1/varn^2 of the scaled inputs is a normal FP64 number below the 1e300
    sentinels: bounded from the inputs (d2 <= (||y'|| + ||Heff||_F X)^2, entries of y and theta normal)."""
    tiny, big = 2.0 ** -1022 * 2.0 ** 64, 1e300 * 2.0 ** -64
    s = 2.0 ** k
    for b in range(Yd.shape[0]):
        H = orc.effective_channels(PsiD[b], theta[b], n_tx)
        X = np.abs(cons).max() * np.sqrt(n_tx) + (0.0 if Xoff is None else np.linalg.norm(Xoff[b], axis=1))
        dmax = (np.linalg.norm(Yd[b], axis=1) + np.linalg.norm(H, axis=(1, 2)) * X) ** 2
        assert np.all(dmax * s * s < big)
        for a in (Yd[b], theta[b]):
            v = np.abs(np.concatenate([a.real.ravel(), a.imag.ravel()]))
            v = v[v > 0]
            assert np.all(v * s > tiny) and np.all(v * s < big)
    v2 = (varn * s) ** 2
    assert tiny < v2 < big and tiny < 1 / v2 < big and er.THR * v2 < big


@pytest.mark.parametrize("hard", [False, True], ids=["soft", "hard"])
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_scaling_by_powers_of_two_is_bitwise_equivariant(S, case, hard):
    """(Yd, theta, varn) -> 2^k (Yd, theta, varn) leaves every d2 / varn^2 unchanged; no absolute constant of the
    E-step (the 1e300 sentinels, the 64 varn^2 window, the Babai slicer) and none of the bit LLRs (La unscaled)
    may show through: m, R, kstar, lse and the LLRs must be bitwise those at k = 0."""
    Yd, PsiD, theta, Xoff = inputs(case)
    cons = orc.qam_constellation(case[3])
    rng = np.random.default_rng(3)
    La = rng.uniform(-8, 8, (Yd.shape[0], case[4], case[1], int(np.log2(case[3]))))
    for varn in (0.3, 10.0):
        base = run_estep(S, case, hard, Yd, PsiD, theta, varn, Xoff)
        lbase = run_llr(S, case, hard, Yd, PsiD, theta, varn, Xoff)
        labase = run_llr(S, case, hard, Yd, PsiD, theta, varn, Xoff, La)
        for k in SCALES:
            _assert_normal_range(Yd, PsiD, theta, varn, case[1], cons, k, Xoff)
            s = 2.0 ** k
            got = run_estep(S, case, hard, Yd * s, PsiD, theta * s, varn * s, Xoff)
            for name, a, b in zip(("m", "R", "kstar", "lse"), base, got):
                assert np.array_equal(a, b), (name, varn, k)
            assert np.array_equal(lbase, run_llr(S, case, hard, Yd * s, PsiD, theta * s, varn * s, Xoff)), (varn, k)
            assert np.array_equal(labase, run_llr(S, case, hard, Yd * s, PsiD, theta * s, varn * s, Xoff, La)), \
                (varn, k)
