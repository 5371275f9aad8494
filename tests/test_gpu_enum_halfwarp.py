"""Up to 4 streams, k_enum runs two data symbols per warp, one per 16-lane half.  The halves are independent: each has its own
shared-memory block, votes, shuffles and flushes only within its half, and may take a different path from its
neighbour.  These tests build inputs whose two symbols of a warp behave differently, or whose last warp holds a
single symbol, and check every statistic against the oracle and the pruned scan against the full scan."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

THR = 64.0      # enqueue window of the E-step, in units of varn^2
QCAP_4X4 = 480  # candidate queue of the 4-stream kernels (EnumT::QCAP)


@pytest.fixture(scope="module")
def S(cuda_device):
    import sbce

    sbce._lib.require_device()
    return sbce


@pytest.fixture(scope="module")
def orc():
    from oracle import em_numpy

    return em_numpy


def queued_nodes(orc, Yd, PsiD, theta, M, n_tx, varn):
    """Per symbol: nodes (digits of streams 1..n_tx-1) whose best leaf lies within THR varn^2 of the minimum,
    i.e. the nodes the E-step queues once its incumbent is the arg-min (a lower bound on what it queues)."""
    cons = orc.qam_constellation(M)
    d2 = orc.hypothesis_distances(Yd, orc.effective_channels(PsiD, theta, n_tx), orc.hypothesis_table(cons, n_tx))
    node_min = d2.reshape(len(Yd), M, M ** (n_tx - 1)).min(axis=1)   # stream 0 is the most significant digit
    return (node_min <= d2.min(axis=1)[:, None] + THR * varn ** 2).sum(axis=1)


def run(S, Yd, PsiD, theta, varn, n_tx, M, hard, full_scan=False):
    import torch

    B, T_d, n_rx = Yd.shape
    N = PsiD.shape[2] - 1
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1, mode="hard" if hard else "soft",
                     full_scan=full_scan)
    ses = S.DeviceSession(prob, B)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    outs = ses.estep(t(Yd), t(PsiD), t(theta), t(np.full(B, varn)))
    torch.cuda.synchronize()
    return [o.cpu().numpy() for o in outs]


def check(S, orc, Yd, PsiD, theta, varn, n_tx, M, hard):
    """Oracle at 1e-10 (indices bit-exact), then the pruned scan bitwise against the full scan."""
    m, R, ks, ls = run(S, Yd, PsiD, theta, varn, n_tx, M, hard)
    cons = orc.qam_constellation(M)
    for b in range(Yd.shape[0]):
        mo, Ro, ko, lo = orc.posterior_stats(Yd[b], PsiD[b], theta[b], cons, n_tx, varn, hard=hard)
        assert np.array_equal(ks[b], ko), "hard-decision indices must be bit-exact"
        assert np.abs(m[b] - mo).max() < 1e-10 * max(1.0, np.abs(mo).max())
        assert np.abs(R[b] - Ro).max() < 1e-10 * max(1.0, np.abs(Ro).max())
        if not hard:
            np.testing.assert_allclose(ls[b], lo, rtol=1e-10, atol=1e-8)
    full = run(S, Yd, PsiD, theta, varn, n_tx, M, hard, full_scan=True)
    for a, f in zip((m, R, ks, ls), full):
        assert np.array_equal(a, f), "default and full scan must agree bitwise"


def two_regime_batch(S, orc, T_d, varn, flat_scale):
    """4x4 16-QAM.  Even symbols: y = Heff x + small noise (one node within the window: narrow flush).  Odd
    symbols: the same row with channel and observation scaled by `flat_scale`, so that every hypothesis lies
    within the window and no node is ever dead (general flush with flushes in the middle of the scan).  (y = 0
    would flatten the posterior too, but x and -x then tie exactly and the arg-min is decided by rounding.)"""
    N, n_tx, n_rx, M = 8, 4, 4, 16
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, 4, T_d, 0.02, 2, seed=211, legacy=False)
    Yd, PsiD = tb.Yd.copy(), tb.PsiD.copy()
    Yd[:, 1::2] *= flat_scale
    PsiD[:, 1::2] *= flat_scale
    return Yd, PsiD, tb.h, n_tx, M


@pytest.mark.parametrize("hard", [False, True])
def test_halves_take_different_flush_paths(S, orc, hard):
    varn = 0.3
    Yd, PsiD, theta, n_tx, M = two_regime_batch(S, orc, 16, varn, 0.015)
    for b in range(Yd.shape[0]):
        q = queued_nodes(orc, Yd[b], PsiD[b], theta[b], M, n_tx, varn)
        assert (q[0::2] <= 2).all(), "even symbols should queue one or two nodes (narrow flush)"
        assert (q[1::2] == M ** (n_tx - 1)).all(), "odd symbols should queue every node (general flush)"
        assert (q[1::2] > QCAP_4X4).all()
    check(S, orc, Yd, PsiD, theta, varn, n_tx, M, hard)


# (n_tx, n_rx, M, varn, T_d): 4x4 16-QAM (the headline kernel, half-warps) and 8x8 QPSK (a warp per symbol)
SINGLE_HALF_CASES = [(4, 4, 16, 0.1, T_d) for T_d in (1, 3, 5, 255)] + [(8, 8, 4, 0.3, T_d) for T_d in (1, 3, 5)]


@pytest.mark.parametrize("case", SINGLE_HALF_CASES)
@pytest.mark.parametrize("hard", [False, True])
def test_last_warp_with_a_single_symbol(S, orc, case, hard):
    n_tx, n_rx, M, varn, T_d = case
    tb = S.signal_model.generate_batch(6, n_tx, n_rx, M, 4, T_d, varn, 2, seed=17 + T_d, legacy=False)
    rng = np.random.default_rng(T_d)
    theta = tb.h + 0.05 * (rng.standard_normal(tb.h.shape) + 1j * rng.standard_normal(tb.h.shape))
    check(S, orc, tb.Yd, tb.PsiD, theta, varn, n_tx, M, hard)


@pytest.mark.parametrize("hard", [False, True])
def test_flat_posterior_overflows_the_queue(S, orc, hard):
    """Every symbol flat: all 4096 nodes of a 4x4 16-QAM symbol are queued, more than eight times the queue,
    so each symbol flushes mid-scan on the general path; no node is dead, so the pruned scan still matches the
    full scan bitwise.  With an odd T_d the last warp has one half."""
    varn = 0.5
    N, n_tx, n_rx, M, T_d = 8, 4, 4, 16, 13
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, 4, T_d, 0.02, 2, seed=5, legacy=False)
    Yd, PsiD = 0.03 * tb.Yd, 0.03 * tb.PsiD
    for b in range(2):
        assert (queued_nodes(orc, Yd[b], PsiD[b], tb.h[b], M, n_tx, varn) == M ** (n_tx - 1)).all()
    check(S, orc, Yd, PsiD, tb.h, varn, n_tx, M, hard)
