"""The partitioned and detector E-step (k_pm_stats and k_det_stats, csrc/pm.cu) statistic by statistic.

The two kernels are the whole E-step of the PM, PM-beta (k_pm_stats), ZF and MMSE (k_det_stats) modes.  These tests call the stand-alone E-step and
compare m_t, R_t and the ZF / MMSE decisions with oracle/em_numpy.py's trace variants, over both template
instantiations, partitions from one enumerated stream to all of them, candidate counts below and above the 32 lanes
of a warp, phase rows below, at and above one pass of the warp, shared and per-trial phases, peaked and flat
posteriors and symbol counts that leave a CTA's warps idle.

* Discrete results are bit-exact: ZF / MMSE decisions and statistics, and plain PM's statistics (sums of products of
  integer constellation points, exact in any order).  PM-beta's m and R agree within 1e-10.
* Every margin of the inputs (ordering arg-max, slicer boundaries, the as-coded slicer's best pair) is checked to
  exceed 1e-9 first, so a failure points at the kernel and not at a tie.
* Oracle-free identities: PM-beta with every stream enumerated equals the soft E-step (an independent kernel), and
  plain PM with every stream enumerated has a closed form.
* ZF at cond(H) = 1e4 and 1e8 decides as pinv does.
* The workspace query rejects partitions with more than 2^24 candidates per symbol."""
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_batches import pm_variant  # noqa: E402

import sbce  # noqa: E402

MARGIN = 1e-9
B = 2

# N, n_tx, n_rx, M, p1, T_d, varn, psi_shared.  M^p1 is a power of 4, so a warp's 32 lanes see 4 or 16 candidates
# (idle lanes), 64 (exactly two each) or 256..65536 (many each).  N + 1 = 2, 9, 32 (one pass of the warp), 33 (the
# quirky channel drops the last phase: one pass for it, two for the exact one), 65, 257.
PM_ROWS = [
    (8, 1, 1, 4, 1, 7, 0.02, False),      # n_tx = 1, 4 candidates, nothing zero-forced
    (1, 2, 2, 4, 1, 9, 10.0, True),       # N + 1 = 2, one stream zero-forced
    (31, 3, 4, 4, 2, 10, 0.02, False),    # N + 1 = 32, 16 candidates, n_rx > n_tx
    (32, 3, 3, 4, 3, 13, 10.0, True),     # N + 1 = 33, 64 candidates, p+1 = n_tx
    (64, 4, 6, 16, 2, 11, 0.02, False),   # N + 1 = 65, 256 candidates, two streams zero-forced
    (256, 2, 2, 64, 2, 5, 10.0, False),   # N + 1 = 257, 4096 candidates, p+1 = n_tx
    (8, 4, 4, 4, 4, 6, 0.02, True),       # n_tx = 4 (last of <4>), p+1 = n_tx
    (12, 4, 4, 64, 2, 5, 0.3, False),     # 4096 candidates, two streams zero-forced
    (9, 5, 5, 4, 1, 9, 0.02, False),      # n_tx = 5 (first of <8>), four streams zero-forced
    (16, 5, 6, 16, 2, 7, 10.0, True),     # 256 candidates
    (6, 5, 5, 4, 5, 6, 0.3, False),       # p+1 = n_tx in <8>, 1024 candidates
    (32, 8, 8, 4, 4, 5, 0.02, False),     # n_tx = 8, 256 candidates, N + 1 = 33
    (8, 8, 8, 64, 2, 5, 0.02, True),      # n_tx = 8, 4096 candidates, six streams zero-forced
    (64, 6, 8, 16, 3, 6, 10.0, False),    # 4096 candidates, N + 1 = 65
]

# N, n_tx, n_rx, M, T_d, varn, psi_shared
DET_ROWS = [
    (8, 1, 1, 4, 7, 0.02, False),
    (31, 2, 2, 16, 10, 0.3, True),
    (32, 3, 4, 64, 9, 0.5, False),        # 64-QAM, n_rx > n_tx, N + 1 = 33
    (64, 4, 4, 16, 11, 10.0, False),      # strong MMSE regularisation, N + 1 = 65
    (1, 5, 8, 64, 6, 0.2, True),          # <8>, 64-QAM (2^30 hypotheses), N + 1 = 2
    (256, 8, 8, 4, 5, 0.3, False),        # n_tx = 8, N + 1 = 257
    (8, 6, 6, 16, 7, 1.0, False),
]

PM_MODES = [(mode, q) for mode in ("pm", "pm_beta") for q in (True, False)]
DET_MODES = [(mode, q) for mode in ("zf", "mmse") for q in (True, False)]


def _pr(M, p1):
    """partition_r giving p+1 = p1 enumerated streams (PM.py:74-75: p = int(partition_r / log2 M))."""
    return (p1 - 1) * math.log2(M)


def _inputs(N, n_tx, n_rx, M, T_d, varn, psi_shared, seed):
    """Seeded data and a theta near the truth for trial 0, a poorer one for trial 1."""
    tb = sbce.signal_model.generate_batch(N, n_tx, n_rx, M, 4, T_d, varn, B, seed=seed, legacy=False)
    rng = np.random.default_rng(seed)
    theta = tb.h + 0.05 * (rng.standard_normal(tb.h.shape) + 1j * rng.standard_normal(tb.h.shape))
    theta[1] = 0.7 * tb.h[1] + 0.2 * (rng.standard_normal(tb.h.shape[1:]) + 1j * rng.standard_normal(tb.h.shape[1:]))
    PsiD = np.ascontiguousarray(tb.PsiD[0]) if psi_shared else tb.PsiD
    return tb.Yd, PsiD, theta, np.full(B, float(varn))


def _estep(prob, Yd, PsiD, theta, varn):
    import torch

    ses = sbce.DeviceSession(prob, B)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    out = ses.estep(t(Yd), t(PsiD), t(theta), t(varn))
    torch.cuda.synchronize()
    return [x.cpu().numpy() for x in out]


def _psi(PsiD, b):
    return PsiD if PsiD.ndim == 2 else PsiD[b]


# ---------------------------------------------------------------------------
# CPU: what the tables reach, and the partition cap
# ---------------------------------------------------------------------------

def test_pm_stats_table_reaches_every_branch():
    """The parity rows below reach both instantiations, every mode with quirks on and off, candidate counts below 32
    (idle lanes), a multiple of 32 and many per lane, phase rows within one warp pass and beyond it, and partitions
    with and without zero-forced streams."""
    items = set()
    for (N, n_tx, n_rx, M, p1, T_d, varn, shared) in PM_ROWS:
        K = M ** p1
        items |= {pm_variant(n_tx, "pm"), "nB=0" if p1 == n_tx else "nB>0", "N1<=32" if N + 1 <= 32 else "N1>32",
                  "T_d%4" if T_d % 4 else "T_d", "shared" if shared else "per-trial",
                  "peaked" if varn < 0.1 else "flat" if varn >= 10 else "mid"}
        items.add("K<32" if K < 32 else "K=64" if K == 64 else "K>>32")
        items.add("p1=1" if p1 == 1 else "p1=n_tx" if p1 == n_tx else "p1 mid")
        items.add(("4096", M, n_tx))
    for (N, n_tx, n_rx, M, T_d, varn, shared) in DET_ROWS:
        items |= {("det", pm_variant(n_tx, "zf")), ("det M", M), "det n_rx>n_tx" if n_rx > n_tx else "det square",
                  "det N1<=32" if N + 1 <= 32 else "det N1>32", "det T_d%4" if T_d % 4 else "det T_d"}
    need = {"k_pm_stats<4>", "k_pm_stats<8>", "nB=0", "nB>0", "N1<=32", "N1>32", "T_d%4", "shared", "per-trial",
            "peaked", "flat", "K<32", "K=64", "K>>32", "p1=1", "p1=n_tx", "p1 mid", ("4096", 64, 2),
            ("det", "k_det_stats<4>"), ("det", "k_det_stats<8>"), ("det M", 4), ("det M", 16), ("det M", 64),
            "det n_rx>n_tx", "det square", "det N1<=32", "det N1>32", "det T_d%4"}
    assert not need - items, sorted(map(str, need - items))
    assert {r[1] for r in PM_ROWS} >= {1, 4, 5, 8} and {r[1] for r in DET_ROWS} >= {1, 4, 5, 8}
    assert set(PM_MODES) == {(m, q) for m in ("pm", "pm_beta") for q in (True, False)}
    assert set(DET_MODES) == {(m, q) for m in ("zf", "mmse") for q in (True, False)}
    # the oracle stays cheap: few symbols where every symbol has 4096 candidates
    assert all(r[5] <= 6 for r in PM_ROWS if r[3] ** r[4] >= 4096)


@pytest.mark.parametrize("mode", ["pm", "pm_beta"])
def test_workspace_query_caps_the_partition_at_2_24_candidates(mode):
    """k_pm_stats enumerates M^(p+1) candidates per symbol in an int: the workspace query admits exactly the
    partitions with p1 log2(M) <= 24 (8x8, every constellation and p1) and answers "unsupported" beyond."""
    for M in (4, 16, 64):
        for p1 in range(1, 9):
            prob = sbce.Problem(N=8, n_tx=8, n_rx=8, M=M, T_p=8, T_d=8, itera=1, mode=mode, partition_r=_pr(M, p1))
            assert prob.p1 == p1
            try:
                ok = sbce.engine.workspace_bytes(prob, 1) > 0
            except sbce.SbceError as e:
                assert "unsupported" in str(e), e
                ok = False
            assert ok == (p1 * math.log2(M) <= 24), (M, p1)


# ---------------------------------------------------------------------------
# GPU: against the trace oracle
# ---------------------------------------------------------------------------

@pytest.fixture(scope="module")
def orc(cuda_device):
    sbce._lib.require_device()
    from oracle import em_numpy

    return em_numpy


def _ids(rows):
    return ["N%d-%dx%d-M%d-" % r[:4] + "-".join(str(x) for x in r[4:]) for r in rows]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,quirks", PM_MODES, ids=["%s-q%d" % (m, q) for m, q in PM_MODES])
@pytest.mark.parametrize("row", PM_ROWS, ids=_ids(PM_ROWS))
def test_pm_estep_matches_trace_oracle(orc, row, mode, quirks):
    N, n_tx, n_rx, M, p1, T_d, varn, shared = row
    Yd, PsiD, theta, vn = _inputs(N, n_tx, n_rx, M, T_d, varn, shared, seed=200 + N + n_tx)
    prob = sbce.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1, mode=mode, quirks=quirks,
                        psi_shared=shared, partition_r=_pr(M, p1))
    cons = orc.qam_constellation(M)
    refs = [orc.pm_stats_trace(Yd[b], _psi(PsiD, b), theta[b], cons, n_tx, varn, p1, mode == "pm_beta", quirks)
            for b in range(B)]
    for b, (_, _, tr) in enumerate(refs):
        for t, s in enumerate(tr):
            assert s["order_gap"] > MARGIN and s["slice_gap"] > MARGIN, ("tie in the inputs, change the seed", b, t)
            assert len(s["cands"]) == M ** p1
    m, R, ks, ls = _estep(prob, Yd, PsiD, theta, vn)
    assert (ks == -1).all() and np.isnan(ls).all()
    for b, (mo, Ro, _) in enumerate(refs):
        if mode == "pm":
            assert np.array_equal(m[b], mo), b
            assert np.array_equal(R[b], Ro), b
        else:
            assert np.abs(m[b] - mo).max() < 1e-10 * max(1.0, np.abs(mo).max()), b
            assert np.abs(R[b] - Ro).max() < 1e-10 * max(1.0, np.abs(Ro).max()), b


@pytest.mark.gpu
@pytest.mark.parametrize("mode,quirks", DET_MODES, ids=["%s-q%d" % (m, q) for m, q in DET_MODES])
@pytest.mark.parametrize("row", DET_ROWS, ids=_ids(DET_ROWS))
def test_detector_estep_matches_trace_oracle(orc, row, mode, quirks):
    N, n_tx, n_rx, M, T_d, varn, shared = row
    Yd, PsiD, theta, vn = _inputs(N, n_tx, n_rx, M, T_d, varn, shared, seed=300 + N + n_tx)
    prob = sbce.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1, mode=mode, quirks=quirks,
                        psi_shared=shared)
    cons = orc.qam_constellation(M)
    refs = [orc.detector_stats_trace(Yd[b], _psi(PsiD, b), theta[b], cons, n_tx, varn, mode, quirks)
            for b in range(B)]
    for b, (_, _, _, tr) in enumerate(refs):
        for t, s in enumerate(tr):
            assert s["slice_gap"] > MARGIN and s["pair_gap"] > MARGIN, ("tie in the inputs, change the seed", b, t)
    m, R, ks, ls = _estep(prob, Yd, PsiD, theta, vn)
    assert np.isnan(ls).all()
    for b, (mo, Ro, ko, _) in enumerate(refs):
        assert np.array_equal(ks[b], ko), b
        assert np.array_equal(m[b], mo), b
        assert np.array_equal(R[b], Ro), b


# ---------------------------------------------------------------------------
# GPU: identities that need no oracle
# ---------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("n_tx,M", [(2, 16), (4, 4), (4, 16), (5, 4)])
def test_pm_beta_with_every_stream_enumerated_equals_soft_estep(orc, n_tx, M):
    """With p+1 = n_tx (quirks off) the candidate list is every hypothesis, so PM-beta's posterior is the soft
    E-step's: k_pm_stats against k_enum on the same inputs."""
    N, n_rx, T_d = 9, n_tx + 1 if n_tx < 4 else n_tx, 7
    Yd, PsiD, theta, vn = _inputs(N, n_tx, n_rx, M, T_d, 0.4, False, seed=400 + n_tx + M)
    pm = sbce.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1, mode="pm_beta", quirks=False,
                      partition_r=_pr(M, n_tx))
    soft = sbce.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1, mode="soft")
    m1, R1, _, _ = _estep(pm, Yd, PsiD, theta, vn)
    m0, R0, _, _ = _estep(soft, Yd, PsiD, theta, vn)
    assert np.abs(m1 - m0).max() < 1e-10 * max(1.0, np.abs(m0).max())
    assert np.abs(R1 - R0).max() < 1e-10 * max(1.0, np.abs(R0).max())


@pytest.mark.gpu
@pytest.mark.parametrize("quirks", [True, False])
@pytest.mark.parametrize("n_tx,M", [(1, 64), (2, 16), (3, 4), (4, 16), (5, 4), (8, 4)])
def test_pm_with_every_stream_enumerated_has_closed_form(orc, n_tx, M, quirks):
    """Plain PM with p+1 = n_tx sums weight 1 over all M^n_tx vectors: m_t = 0 and R_t = M^n_tx 2(M-1)/3 I,
    bit-exact."""
    N, n_rx, T_d = 5, n_tx if n_tx != 5 else 6, 6
    Yd, PsiD, theta, vn = _inputs(N, n_tx, n_rx, M, T_d, 0.3, False, seed=500 + n_tx)
    prob = sbce.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1, mode="pm", quirks=quirks,
                        partition_r=_pr(M, n_tx))
    m, R, ks, _ = _estep(prob, Yd, PsiD, theta, vn)
    assert np.array_equal(m, np.zeros_like(m))
    want = np.broadcast_to(M ** n_tx * 2 * (M - 1) / 3 * np.eye(n_tx), R.shape)
    assert np.array_equal(R, want)
    assert (ks == -1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kappa", [1e4, 1e8])
@pytest.mark.parametrize("n_tx,n_rx,M", [(4, 4, 16), (3, 6, 64), (8, 8, 4)])
def test_zf_decides_like_pinv_on_ill_conditioned_channels(orc, n_tx, n_rx, M, kappa):
    """N = 1 with theta_1 = 0: every symbol sees the channel H = U diag(1, ..., 1/kappa) V^H.  On noiseless data
    pinv(H) y returns the transmitted symbols to within kappa * eps, far inside the slicer's margin of 1, so the
    ZF decisions must be exactly the transmitted hypotheses."""
    rng = np.random.default_rng(int(kappa) % 1000 + n_tx)
    unitary = lambda n: np.linalg.qr(rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n)))[0]
    s = np.ones(n_tx)
    s[-1] = 1.0 / kappa
    H = unitary(n_rx)[:, :n_tx] @ np.diag(s) @ unitary(n_tx).conj().T
    assert np.linalg.cond(H) == pytest.approx(kappa, rel=1e-3)
    N, T_d = 1, 33
    theta = np.zeros((B, 2 * n_tx, n_rx), np.complex128)
    theta[:, :n_tx] = H.T                           # Theta[j, r] = H[r, j]: direct link only
    cons = orc.qam_constellation(M)
    idx = rng.integers(0, M, (B, T_d, n_tx))
    Yd = np.einsum("rj,btj->btr", H, cons[idx])
    PsiD = np.ones((B, T_d, 2), np.complex128)
    PsiD[:, :, 1] = np.exp(1j * rng.uniform(0, 2 * np.pi, (B, T_d)))
    prob = sbce.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1, mode="zf", quirks=False)
    _, _, ks, _ = _estep(prob, Yd, PsiD, theta, np.full(B, 0.1))
    want = (idx * M ** np.arange(n_tx - 1, -1, -1)).sum(axis=2)
    assert np.array_equal(ks, want), int((ks != want).sum())
