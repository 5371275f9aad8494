"""On half-warp groups (up to 4 streams) the innermost node level of k_enum is packed: the group takes its live
nodes one after the other and its 16 lanes split the stream-1 symbols below each one.  Which lane visits which
node therefore depends on which nodes are live, i.e. on the pruning.  These tests build batches where many nodes
stay live, where hypotheses tie exactly and where the queue fills in the middle of the walk, and check the pruned
walk bitwise against the full scan and every statistic against the oracle, in soft and hard mode."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

THR = 64.0      # enqueue window of the E-step, in units of varn^2
QCAP_4X4 = 480  # candidate queue of the half-warp kernels (EnumT::QCAP)


@pytest.fixture(scope="module")
def S(cuda_device):
    import sbce

    sbce._lib.require_device()
    return sbce


@pytest.fixture(scope="module")
def orc():
    from oracle import em_numpy

    return em_numpy


def run(S, Yd, PsiD, theta, varn, n_tx, M, hard, full_scan):
    import torch

    B, T_d, n_rx = Yd.shape
    prob = S.Problem(N=PsiD.shape[2] - 1, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1,
                     mode="hard" if hard else "soft", full_scan=full_scan)
    ses = S.DeviceSession(prob, B)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    outs = ses.estep(t(Yd), t(PsiD), t(theta), t(np.full(B, varn)))
    torch.cuda.synchronize()
    return [o.cpu().numpy() for o in outs]


def queued_nodes(orc, Yd, PsiD, theta, M, n_tx, varn):
    """Per symbol: nodes whose best leaf lies within THR varn^2 of the minimum (a lower bound on what is queued)."""
    cons = orc.qam_constellation(M)
    d2 = orc.hypothesis_distances(Yd, orc.effective_channels(PsiD, theta, n_tx), orc.hypothesis_table(cons, n_tx))
    node_min = d2.reshape(len(Yd), M, M ** (n_tx - 1)).min(axis=1)   # stream 0 is the most significant digit
    return (node_min <= d2.min(axis=1)[:, None] + THR * varn ** 2).sum(axis=1)


def make_case(S, n_tx, M, varn, T_d, theta_kind, seed):
    """Batch of two trials observed through the true channel at noise level varn.  theta_kind: "true" estimates
    with the true channel; "zero" with theta = 0 (every hypothesis ties exactly); "tie1" with the channel of stream
    1 zeroed (hypotheses that differ only in stream 1 tie exactly, inside one packed step)."""
    tb = S.signal_model.generate_batch(8, n_tx, n_tx, M, 4, T_d, varn, 2, seed=seed, legacy=False)
    theta = tb.h.copy()
    if theta_kind == "zero":
        theta[:] = 0.0
    elif theta_kind == "tie1":
        theta[:, 1::n_tx, :] = 0.0   # rows n' * n_tx + 1: stream 1 of every RIS element
    return tb.Yd, tb.PsiD, theta


# (name, n_tx, M, varn, T_d, theta): odd T_d everywhere, so the last warp holds a single symbol
CASES = [
    ("4x4_16qam_varn1", 4, 16, 1.0, 13, "true"),   # a few live nodes per round
    ("4x4_16qam_varn3", 4, 16, 3.0, 7, "true"),    # 100-400 queued nodes per symbol
    ("4x4_16qam_varn5", 4, 16, 5.0, 7, "true"),    # more than QCAP queued nodes: flushes mid-walk
    ("4x4_16qam_theta0", 4, 16, 0.3, 5, "zero"),   # all 65536 hypotheses tie; every node queued
    ("4x4_16qam_tie1", 4, 16, 0.1, 9, "tie1"),
    ("3x3_64qam_varn1", 3, 64, 1.0, 7, "true"),    # M = 64: four packed steps per live node
    ("3x3_64qam_tie1", 3, 64, 0.3, 5, "tie1"),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("hard", [False, True], ids=["soft", "hard"])
def test_packed_walk_matches_full_scan_and_oracle(S, orc, case, hard):
    _, n_tx, M, varn, T_d, theta_kind = case
    Yd, PsiD, theta = make_case(S, n_tx, M, varn, T_d, theta_kind, seed=97 + T_d)
    pruned = run(S, Yd, PsiD, theta, varn, n_tx, M, hard, full_scan=False)
    full = run(S, Yd, PsiD, theta, varn, n_tx, M, hard, full_scan=True)
    for a, f in zip(pruned, full):
        assert np.array_equal(a, f, equal_nan=True), "default and full scan must agree bitwise"
    m, R, ks, ls = pruned
    cons = orc.qam_constellation(M)
    for b in range(Yd.shape[0]):
        mo, Ro, ko, lo = orc.posterior_stats(Yd[b], PsiD[b], theta[b], cons, n_tx, varn, hard=hard)
        assert np.array_equal(ks[b], ko), "hard-decision indices must be bit-exact"
        assert np.abs(m[b] - mo).max() < 1e-10 * max(1.0, np.abs(mo).max())
        assert np.abs(R[b] - Ro).max() < 1e-10 * max(1.0, np.abs(Ro).max())
        if not hard:
            np.testing.assert_allclose(ls[b], lo, rtol=1e-10, atol=1e-8)


def test_cases_reach_the_paths_they_name(S, orc):
    """The varn = 5 and theta = 0 batches queue more nodes than the queue holds, so they flush mid-walk; the tie
    batches hold exact ties that the arg-min must break towards the first index."""
    for name, n_tx, M, varn, T_d, theta_kind in CASES:
        Yd, PsiD, theta = make_case(S, n_tx, M, varn, T_d, theta_kind, seed=97 + T_d)
        if name in ("4x4_16qam_varn5", "4x4_16qam_theta0"):
            q = queued_nodes(orc, Yd[0], PsiD[0], theta[0], M, n_tx, varn)
            assert q.max() > QCAP_4X4, name
        if theta_kind != "true":
            cons = orc.qam_constellation(M)
            d2 = orc.hypothesis_distances(Yd[0], orc.effective_channels(PsiD[0], theta[0], n_tx),
                                          cons[orc.hypothesis_digits(np.arange(M ** n_tx), M, n_tx)])
            assert ((d2 == d2.min(axis=1)[:, None]).sum(axis=1) >= M).all(), name
