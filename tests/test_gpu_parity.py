"""GPU parity tests: the CUDA path (through the C ABI) against the numpy oracle on
identical seeded inputs, and against the golden vectors minted from the literal
reference.  Bars (BASELINE.json north_star): theta within 1e-9 relative Frobenius at
equal iteration count, hard-decision indices bit-exact, NMSE to 4 significant figures."""
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import golden_names, load_golden

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import estep_reference as er  # noqa: E402
import mstep_reference as mr  # noqa: E402

pytestmark = pytest.mark.gpu

RTOL = 1e-9


def relerr(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b)))


@pytest.fixture(scope="module")
def S(cuda_device):
    import sbce

    sbce._lib.require_device()
    return sbce


@pytest.fixture(scope="module")
def orc():
    from oracle import em_numpy

    return em_numpy


ESTEP_CASES = [
    # N, n_tx, n_rx, M, T_d, varn
    (8, 1, 1, 4, 20, 0.5), (8, 1, 4, 16, 20, 0.3), (12, 1, 8, 64, 12, 0.4),
    (8, 2, 2, 4, 33, 0.1), (8, 2, 2, 4, 33, 3.0), (8, 2, 4, 16, 17, 0.3), (6, 2, 3, 64, 9, 0.5),
    (7, 3, 3, 4, 21, 0.2), (5, 3, 4, 16, 10, 1.5), (5, 3, 2, 4, 10, 0.7),
    (9, 4, 4, 4, 19, 0.1), (6, 4, 4, 16, 6, 0.5), (6, 4, 4, 16, 6, 30.0), (4, 4, 6, 4, 7, 0.4), (4, 2, 8, 4, 7, 0.4),
    # wide arrays (BASELINE.json configs 4/5: 8x8): row-per-lane QR + deep hypothesis trees
    (6, 5, 5, 4, 9, 0.3), (5, 6, 6, 4, 7, 0.2), (5, 7, 8, 4, 6, 0.4), (6, 8, 8, 4, 9, 0.3), (6, 8, 8, 4, 5, 20.0),
    (4, 5, 6, 16, 3, 0.6), (4, 6, 4, 4, 5, 0.5), (5, 5, 7, 4, 18, 0.2),
    # tensor-path effective-channel kernel (n_tx n_rx >= 8, N >= 15): 1..4 column tiles, ragged K (N + 1 not a
    # multiple of 8), symbol counts that are not multiples of 16 / 32 / 128
    (15, 1, 8, 4, 37, 0.3), (17, 2, 4, 16, 33, 0.4), (20, 3, 4, 4, 40, 0.3), (16, 4, 4, 4, 130, 0.2),
    (23, 4, 6, 4, 19, 0.3), (18, 3, 8, 4, 21, 0.4), (31, 4, 8, 4, 45, 0.3), (40, 2, 6, 16, 29, 0.5),
    # 64-QAM on 3 and 4 streams (16-lane PAM groups of the narrow flush), peaked and flat posteriors (varn >= 4
    # overflows the candidate queue); 6 streams of 16-QAM (2^24 leaves)
    (5, 3, 4, 64, 4, 0.2), (5, 3, 4, 64, 4, 6.0), (4, 4, 4, 64, 1, 0.2), (4, 4, 4, 64, 1, 5.0), (3, 6, 6, 16, 1, 0.4),
    # effective channel too long for shared memory and for the tensor path (BASELINE.json config 3: N = 256)
    (256, 4, 4, 4, 6, 0.3),
]


_ESTEP_REFS = {}


@pytest.mark.parametrize("case", ESTEP_CASES)
@pytest.mark.parametrize("hard", [False, True])
def test_estep_matches_oracle(S, orc, case, hard):
    """m, R and lse within the derived bound tau of the exact (clongdouble) statistics, kstar by the gap rule
    (tests/estep_reference.py): the oracle's FP64 distances are formed directly, the device's through a QR, so
    neither is bit-exact against the other; the extended-precision reference decides."""
    import torch

    N, n_tx, n_rx, M, T_d, varn = case
    B = 3
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, 4, T_d, varn, B, seed=100 + N, legacy=False)
    rng = np.random.default_rng(7)
    # theta near the truth (peaked posteriors) for b=0,1 and far (flat-ish) for b=2
    theta = tb.h + 0.05 * (rng.standard_normal(tb.h.shape) + 1j * rng.standard_normal(tb.h.shape))
    theta[2] = 0.3 * tb.h[2]
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1, mode="hard" if hard else "soft")
    ses = S.DeviceSession(prob, B)
    dev = ses.device
    m, R, ks, ls = ses.estep(torch.from_numpy(tb.Yd).to(dev), torch.from_numpy(tb.PsiD).to(dev),
                             torch.from_numpy(theta).to(dev), torch.from_numpy(tb.varn).to(dev))
    torch.cuda.synchronize()
    m, R, ks, ls = m.cpu().numpy(), R.cpu().numpy(), ks.cpu().numpy(), ls.cpu().numpy()
    cons = orc.qam_constellation(M)
    if case not in _ESTEP_REFS:    # soft and hard share the reference
        _ESTEP_REFS[case] = [er.reference(tb.Yd[b], tb.PsiD[b], theta[b], cons, n_tx, varn) for b in range(B)]
    for b in range(B):
        ref = _ESTEP_REFS[case][b]
        assert not er.kstar_bad(ref, ks[b]), er.kstar_bad(ref, ks[b])[:4]
        r, adm = er.ratios(ref, m[b], R[b], ls[b], hard, ks[b])
        assert r <= 1.0, (b, r)
        assert adm == T_d or hard


@pytest.mark.parametrize("case", [(8, 2, 2, 16, 40, 0.1), (6, 3, 3, 16, 24, 0.4), (8, 4, 4, 16, 24, 0.1),
                                  (8, 4, 4, 16, 12, 5.0), (6, 4, 4, 4, 30, 0.2), (5, 4, 4, 64, 4, 0.3),
                                  (5, 3, 4, 64, 6, 2.0)])
@pytest.mark.parametrize("hard", [False, True])
def test_subtree_skipping_is_bit_identical_to_full_scan(S, case, hard):
    """The default E-step skips subtrees whose partial distance exceeds incumbent + 64 varn^2; such
    nodes can neither improve the arg-min nor enter the posterior sums, so every output must be
    bit-identical to the scan that visits all M^(n_tx-1) nodes (SBCE_FLAG_FULL_SCAN)."""
    import torch

    N, n_tx, n_rx, M, T_d, varn = case
    B = 3
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, 4, T_d, varn, B, seed=31 + N, legacy=False)
    rng = np.random.default_rng(3)
    theta = tb.h + 0.1 * (rng.standard_normal(tb.h.shape) + 1j * rng.standard_normal(tb.h.shape))
    theta[2] = 0.5 * tb.h[2]
    outs = []
    for full in (False, True):
        prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1, mode="hard" if hard else "soft",
                         full_scan=full)
        ses = S.DeviceSession(prob, B)
        dev = ses.device
        outs.append([x.cpu().numpy() for x in ses.estep(torch.from_numpy(tb.Yd).to(dev), torch.from_numpy(tb.PsiD).to(dev),
                                                        torch.from_numpy(theta).to(dev), torch.from_numpy(tb.varn).to(dev))])
    (m0, R0, k0, l0), (m1, R1, k1, l1) = outs
    assert np.array_equal(k0, k1)
    if varn < 1.0 or hard:
        for a, b in ((m0, m1), (R0, R1), (l0, l1)):
            assert np.array_equal(a, b)
    else:
        # flat posteriors overflow the candidate queue mid-scan; the flush points (hence the summation
        # order) may differ between the two scans, the sums agree to rounding
        for a, b in ((m0, m1), (R0, R1), (l0, l1)):
            np.testing.assert_allclose(a, b, rtol=1e-13, atol=1e-13)


def test_estep_zero_theta_is_uniform_posterior(S, orc):
    """theta = 0 (first iteration of the zero-start scripts): every hypothesis ties; posterior
    uniform, arg-max = index 0 (np.argmax first-index rule)."""
    import torch

    N, n_tx, n_rx, M, T_d = 6, 2, 2, 16, 5
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, 4, T_d, 0.1, 2, seed=3, legacy=False)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1)
    ses = S.DeviceSession(prob, 2)
    dev = ses.device
    th = torch.zeros((2, prob.L, n_rx), dtype=torch.complex128, device=dev)
    m, R, ks, ls = ses.estep(torch.from_numpy(tb.Yd).to(dev), torch.from_numpy(tb.PsiD).to(dev), th,
                             torch.from_numpy(tb.varn).to(dev))
    assert int(ks.abs().max()) == 0
    assert float(m.abs().max()) < 1e-12
    eye = 10.0 * np.eye(n_tx)
    assert np.abs(R.cpu().numpy() - eye).max() < 1e-11


MSTEP_CASES = [(8, 2, 2, 4, 12, 30), (32, 2, 2, 4, 40, 50), (6, 1, 4, 16, 8, 20), (5, 3, 3, 4, 14, 16),
               (16, 4, 4, 16, 24, 80), (11, 3, 2, 4, 20, 40), (64, 4, 4, 4, 64, 256),
               # wide arrays: generic tensor-path Gram (n_tx = 5..8)
               (6, 5, 5, 4, 20, 40), (7, 6, 8, 4, 24, 50), (5, 7, 7, 4, 30, 41), (9, 8, 8, 4, 50, 77),
               (12, 8, 8, 16, 60, 120),
               # long channels: n_tx = 4 beyond the fixed-chunk Gram kernel (N = 256), and a solution vector
               # that no longer fits in shared memory (L = 1288, n_rx = 8 -> global scratch); Gaussian-integer inputs
               # ("int"), whose FP64 Gram is exact, so that the exact system stays cheap at L > 300
               (256, 4, 2, 4, 600, 800, "int", None), (256, 2, 2, 4, 300, 400, "int", None),
               (160, 8, 8, 4, 800, 900, "int", None),
               # random Hermitian PD statistics ("pd": no enumeration).  n_tx = 1, L = N + 1 = 2..17: every
               # residue of L mod 16 of the blocked Cholesky, incl. n_rx = 1 (three zero rows under the matrix)
               *[(N, 1, (1, 2, 3, 4, 6, 8)[N % 6], 4, 3, 2 * N + 4, "pd") for N in range(1, 17)],
               # block lengths 1, 15, 16, 17, 64, 65 (ragged chunk, one stage, ring wrap-around) on the scalar,
               # TMA (n_tx = 4, N <= 143) and generic Gram
               *[(N, n_tx, 3, 4, T_p, T_d, "pd") for N, n_tx in ((20, 2), (10, 4), (6, 6))
                 for T_p, T_d in ((1, 65), (65, 1), (15, 64), (64, 15), (16, 17), (17, 16))],
               # n_tx = 4 on both sides of the TMA / generic Gram switch
               (143, 4, 2, 4, 64, 300, "int", None), (144, 4, 2, 4, 64, 300, "int", None),
               # n_rx = 8, Lp = 48 / 56: the solution vector on both sides of the shared / global scratch switch
               (5, 8, 8, 4, 16, 20, "pd"), (6, 8, 8, 4, 16, 20, "pd"),
               # ill-conditioned systems, cond(G) ~ 1e4 / 1e8 / 1e12 from nearly collinear RIS columns (integer
               # inputs with weighted rows, mstep_reference.integer_inputs) on every Gram kernel: scalar n_tx = 1..3,
               # TMA and generic n_tx = 4 at N = 143 / 144, wide n_tx = 5..8; L mod 16 = 0, 1, 15 and the solution
               # vector in shared memory and in global scratch
               *[(N, n_tx, n_rx, 4, T_p, T_d, "int", cond)
                 for N, n_tx, n_rx, T_p, T_d in ((16, 1, 1, 4, 30), (23, 2, 2, 8, 40), (4, 3, 3, 2, 12),
                                                  (143, 4, 2, 16, 170), (144, 4, 2, 16, 170), (6, 5, 5, 4, 12),
                                                  (7, 6, 3, 4, 14), (6, 7, 7, 4, 12), (6, 8, 8, 4, 12))
                 for cond in (1e4, 1e8, 1e12)]]


def random_pd_stats(rng, B, T, n_tx):
    """Per-symbol statistics m (random) and R = (A + A^H)/2 + c I (exactly Hermitian, positive definite)."""
    A = rng.standard_normal((B, T, n_tx, n_tx)) + 1j * rng.standard_normal((B, T, n_tx, n_tx))
    R = 0.5 * (A + A.conj().transpose(0, 1, 3, 2))
    R += (np.linalg.norm(A, ord=2, axis=(2, 3)) + 0.5)[:, :, None, None] * np.eye(n_tx)
    m = rng.standard_normal((B, T, n_tx)) + 1j * rng.standard_normal((B, T, n_tx))
    return m, R


@pytest.mark.parametrize("case", MSTEP_CASES)
def test_mstep_matches_oracle(S, orc, case):
    """Backward error eta of theta against the exact normal equations (clongdouble, or FP64 from integer inputs)
    within tau(L) = 8 L u at any conditioning, and the forward error against the refined reference solution within
    8 L u cond(G)."""
    import torch

    N, n_tx, n_rx, M, T_p, T_d, *kind = case
    B = 2
    if kind[:1] == ["int"]:
        inp = mr.integer_inputs(np.random.default_rng(N * 10 + n_tx), B, N + 1, n_tx, n_rx, T_p, T_d, cond=kind[1])
        tb = SimpleNamespace(**inp)
        sm, sR = inp["m"], inp["R"]
    else:
        tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, 0.1, B, seed=5, legacy=False)
    if kind == ["pd"]:   # random pilot phases: the pilot block observes every RIS element, even when T_d = 1
        tb.PsiP[:] = np.exp(2j * np.pi * np.random.default_rng(N + T_p).random(tb.PsiP.shape))
    cons = orc.qam_constellation(M)
    # (the M-step does not depend on the mode; 8 streams of 16-QAM only exist in the partitioned modes)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=1,
                     mode="soft" if n_tx * np.log2(M) <= 24 else "pm_beta")
    if kind[:1] != ["int"]:
        # soft statistics from a perturbed theta so R_t is full-rank-ish; computed by the oracle
        # (for the 64x4x4 case use rank-one statistics of the true symbols to keep the CPU side fast)
        sm = np.empty((B, T_d, n_tx), np.complex128)
        sR = np.empty((B, T_d, n_tx, n_tx), np.complex128)
        for b in range(B):
            if kind == ["pd"]:
                m_, R_ = random_pd_stats(np.random.default_rng(N * 100 + T_d + b), 1, T_d, n_tx)
                sm[b], sR[b] = m_[0], R_[0]
            elif M ** n_tx <= 4096 or (n_tx > 4 and N < 10 and M == 4):
                sm[b], sR[b], _, _ = orc.posterior_stats(tb.Yd[b], tb.PsiD[b], 0.7 * tb.h[b], cons, n_tx, 2.0)
            else:
                sm[b], sR[b] = orc.pilot_stats(tb.Xd[b])
    ses = S.DeviceSession(prob, B)
    dev = ses.device
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    theta, status = ses.mstep(t(tb.Yd), t(tb.Yp), t(tb.PsiD), t(tb.PsiP), t(tb.Xp), t(sm), t(sR))
    torch.cuda.synchronize()
    theta = theta.cpu().numpy()
    assert status.cpu().numpy().tolist() == [0] * B
    L = prob.L
    for b in range(B):
        if kind[:1] == ["int"]:
            G, Bm, cond = inp["G"][b], inp["B"][b], inp["cond"][b]
        else:
            G, Bm = mr.system(tb.PsiP[b], tb.Yp[b], tb.Xp[b], tb.PsiD[b], tb.Yd[b], sm[b], sR[b])
            cond = np.linalg.cond(G.astype(np.complex128))
        eta = mr.backward_error(G, Bm, theta[b])
        assert eta <= mr.tau(L), (eta, mr.tau(L))
        err = mr.relerr(theta[b], mr.refined_solve(G, Bm))
        assert err <= 8 * L * mr.U * cond, (err, cond)


def test_mstep_flags_singular_system(S):
    """T_p + T_d < L: the normal matrix is singular; the trial must be flagged, not poisoned."""
    import torch

    N, n_tx, n_rx, M, T_p, T_d = 16, 2, 2, 4, 4, 8
    B = 2
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, 0.1, B, seed=5, legacy=False)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=1)
    sm = tb.Xd.conj()
    sR = tb.Xd.conj()[:, :, :, None] * tb.Xd[:, :, None, :]
    ses = S.DeviceSession(prob, B)
    dev = ses.device
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    theta, status = ses.mstep(t(tb.Yd), t(tb.Yp), t(tb.PsiD), t(tb.PsiP), t(tb.Xp), t(sm), t(sR))
    assert (status.cpu().numpy() != 0).all()


# ---------------------------------------------------------------------------
# whole estimator, reference-signature entry points, golden vectors of the literal reference
# ---------------------------------------------------------------------------

def _ref_objects(g, n_rx):
    """Rebuild the reference's Python objects (lists of column vectors, dense Z_p) from a fixture."""
    Y_d = [g["Yd"][t].reshape(-1, 1) for t in range(g["Yd"].shape[0])]
    Y_p = [g["Yp"][t].reshape(-1, 1) for t in range(g["Yp"].shape[0])]
    Z_p = [np.kron(g["Wp"][t][None, :], np.eye(n_rx, dtype=np.complex128)) for t in range(g["Wp"].shape[0])]
    return Y_d, Y_p, Z_p, g["PsiD"].T.copy()


@pytest.mark.parametrize("name", golden_names("soft"))
def test_em_soft_golden(S, orc, name):
    meta, g = load_golden(name)
    n_tx, n_rx, M = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g, n_rx)
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    h0 = None if int(meta.get("zero_start", 0)) else g["theta0"].reshape(-1, 1)
    theta = S.em(Y_d, Y_p, int(meta["T_d"]), int(meta["T_p"]), Z_p, PsiTilde_td, table, M, float(meta["varn"]),
                 int(meta["itera"]), h0)
    assert theta.shape == (g["theta_ref"].size, 1)
    assert relerr(theta.reshape(g["theta_ref"].shape), g["theta_ref"]) < RTOL
    assert abs(S.nmse(theta, g["h"]) - g["nmse_ref"]) <= 1e-8 * max(1.0, g["nmse_ref"])


@pytest.mark.parametrize("name", golden_names("nodirect"))
def test_em_no_direct_link_golden(S, orc, name):
    """No-direct-link layout of `direct vs non direct - T_pv s nmse.py` (SURVEY 8f-4) through the reference-signature
    entry point: N phase rows, L = N n_tx; and the same data with the direct link (`em_direct_in`)."""
    meta, g = load_golden(name)
    n_tx, n_rx, M = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    T_d, T_p, varn, itera = int(meta["T_d"]), int(meta["T_p"]), float(meta["varn"]), int(meta["itera"])
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g, n_rx)
    theta = S.em(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, table, M, varn, itera, None)
    assert theta.shape == (int(meta["N"]) * n_tx * n_rx, 1)
    assert relerr(theta.reshape(g["theta_ref"].shape), g["theta_ref"]) < RTOL
    g1 = {k[4:]: v for k, v in g.items() if k.startswith("din_")}
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g1, n_rx)
    theta = S.em(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, table, M, varn, itera, None)
    assert relerr(theta.reshape(g1["theta_ref"].shape), g1["theta_ref"]) < RTOL


@pytest.mark.parametrize("name", golden_names("parallel"))
def test_em_parallel_golden(S, orc, name):
    """Superimposed pilots (`Parallel/ParallelProtocol_Tp.py:64`) through the reference-signature entry point."""
    meta, g = load_golden(name)
    n_tx, n_rx, M, N = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"]), int(meta["N"])
    T, T_p, T_d = int(meta["T"]), int(meta["T_p"]), int(meta["T_d"])
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    Y = [g["Y"][t].reshape(-1, 1) for t in range(T)]
    X_p = [g["Xp"][t].reshape(-1, 1) for t in range(T_p)]
    X_d = [g["Xd"][t].reshape(-1, 1) for t in range(T_d)]
    theta = S.em_parallel(Y, T, None, X_d, X_p, T_p, T_d, n_tx, g["Psi"].T.copy(), table, M, float(meta["varn"]),
                          int(meta["itera"]), N)
    assert relerr(theta.reshape(g["theta_ref"].shape), g["theta_ref"]) < RTOL


@pytest.mark.parametrize("case", [(8, 2, 2, 16, 12, 40, 4, 0.3, False), (6, 3, 4, 4, 50, 30, 3, 0.5, True),
                                  (10, 4, 4, 4, 20, 60, 3, 0.2, False), (5, 6, 8, 4, 10, 48, 2, 0.4, False)])
def test_em_superimposed_batch_matches_oracle(S, orc, case):
    """Superimposed pilots, batched, incl. the wide-array E-step: decisions bit-exact, theta 1e-9."""
    N, n_tx, n_rx, M, T_p, T_d, itera, varn, hard = case
    B, T = 3, max(T_p, T_d)
    rng = np.random.default_rng(12)
    cons = orc.qam_constellation(M)
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, 2, T, varn, B, seed=8, legacy=False, variant="top_td")
    Xoff = np.zeros((B, T, n_tx), np.complex128)
    Xoff[:, :T_p] = cons[rng.integers(0, M, (B, T_p, n_tx))]
    Xd = np.zeros((B, T, n_tx), np.complex128)
    Xd[:, :T_d] = cons[rng.integers(0, M, (B, T_d, n_tx))]
    W = (tb.PsiD[:, :, :, None] * (Xd + Xoff)[:, :, None, :]).reshape(B, T, -1)
    Y = W @ tb.h + np.sqrt(varn / 2) * (rng.standard_normal((B, T, n_rx)) + 1j * rng.standard_normal((B, T, n_rx)))
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=0, T_d=T, itera=itera, mode="hard" if hard else "soft",
                     zero_start=True, superimposed=True)
    res = S.run_host(prob, Y, np.zeros((B, 0, n_rx), np.complex128), tb.PsiD, np.zeros((B, 0, N + 1), np.complex128),
                     Xoff, tb.varn, h_true=tb.h)
    assert (res.status == 0).all()
    for b in range(B):
        ref, tr = orc.em_superimposed(Y[b], tb.PsiD[b], Xoff[b], M, varn, itera, hard=hard, return_trace=True)
        assert relerr(res.theta[b], ref) < RTOL
        assert np.array_equal(res.kstar[b], tr["kstar"])
        if not hard:   # (hard mode reports -min d2 / varn^2, not the log-sum)
            np.testing.assert_allclose(res.lse[b], np.array(tr["lse"]), rtol=1e-9)


@pytest.mark.parametrize("name", golden_names("hard"))
def test_em_hard_golden(S, orc, name):
    meta, g = load_golden(name)
    n_tx, n_rx, M = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    T_d, T_p, varn, itera = int(meta["T_d"]), int(meta["T_p"]), float(meta["varn"]), int(meta["itera"])
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g, n_rx)
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    X_d = [g["Xd"][t].reshape(-1, 1) for t in range(T_d)]
    if "llf_ref" in g:
        theta, llf = S.em_llf(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, table, M, varn, itera, g["theta0"].reshape(-1, 1),
                              X_d=X_d)
        assert llf.shape == (itera, 1)
        np.testing.assert_allclose(llf.reshape(-1), g["llf_ref"], rtol=1e-9)
    else:
        theta, X_dest = S.em_ser(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, table, M, varn, itera,
                                 g["theta0"].reshape(-1, 1))
        assert np.array_equal(np.vstack(X_dest), g["xdest_ref"])  # bit-exact decisions
        assert S.ser_as_coded(X_d, X_dest) == g["ser_ref"]
    assert relerr(theta.reshape(g["theta_ref"].shape), g["theta_ref"]) < RTOL


@pytest.mark.parametrize("name", golden_names("loglik"))
def test_em_loglik_golden(S, orc, name):
    """`Proposed method/Log_likelihood.py:45` through its own positional signature (Z_d, n_tx as arguments)."""
    meta, g = load_golden(name)
    n_tx, n_rx, M = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    T_d, T_p, varn, itera = int(meta["T_d"]), int(meta["T_p"]), float(meta["varn"]), int(meta["itera"])
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g, n_rx)
    Wd = (g["PsiD"][:, :, None] * g["Xd"][:, None, :]).reshape(T_d, -1)
    Z_d = [np.kron(Wd[t][None, :], np.eye(n_rx, dtype=np.complex128)) for t in range(T_d)]
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    theta, llf = S.em_loglik(Y_d, Y_p, T_d, T_p, Z_p, Z_d, PsiTilde_td, table, M, varn, itera, g["theta0"].reshape(-1, 1), n_tx)
    assert llf.shape == (itera, 1)
    np.testing.assert_allclose(llf.reshape(-1), g["llf_ref"], rtol=1e-9)
    assert relerr(theta.reshape(g["theta_ref"].shape), g["theta_ref"]) < RTOL


@pytest.mark.parametrize("name", golden_names(["soft_td", "iter_llf"]))
def test_em_remaining_soft_scripts_golden(S, orc, name):
    """`Proposed method/Proposed_method_NMSEvsTd.py:44` em and `Proposed method/IterationsvsLLF.py:44` em (soft + LLF)."""
    meta, g = load_golden(name)
    n_tx, n_rx, M = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    T_d, T_p, varn, itera = int(meta["T_d"]), int(meta["T_p"]), float(meta["varn"]), int(meta["itera"])
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g, n_rx)
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    h0 = g["theta0"].reshape(-1, 1)
    if "llf_ref" in g:
        Wd = (g["PsiD"][:, :, None] * g["Xd"][:, None, :]).reshape(T_d, -1)
        Z_d = [np.kron(Wd[t][None, :], np.eye(n_rx, dtype=np.complex128)) for t in range(T_d)]
        theta, llf = S.em_iterations_llf(Y_d, Y_p, T_d, T_p, Z_p, Z_d, PsiTilde_td, table, M, varn, itera, h0, n_tx)
        np.testing.assert_allclose(llf.reshape(-1), g["llf_ref"], rtol=1e-9)
    else:
        theta = S.em(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, table, M, varn, itera, h0)
    assert relerr(theta.reshape(g["theta_ref"].shape), g["theta_ref"]) < RTOL


@pytest.mark.parametrize("name", golden_names("pm_ser"))
def test_em_pm_ser_golden(S, orc, name):
    """`Proposed method/SER/PM_SER.py:55` em_pm: the PM estimator from a random start, all iterations executed."""
    meta, g = load_golden(name)
    n_tx, n_rx, M = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g, n_rx)
    cons = orc.qam_constellation(M)
    th = S.em_pm(Y_d, Y_p, int(meta["T_d"]), int(meta["T_p"]), Z_p, PsiTilde_td, orc.hypothesis_table(cons, n_tx), M,
                 float(meta["varn"]), int(meta["itera"]), g["theta0"].reshape(-1, 1), g["h"].reshape(-1), n_tx,
                 int(meta["partition_r"]), None, cons, genie_stop=False)
    assert relerr(th.reshape(g["theta_ref"].shape), g["theta_ref"]) < RTOL


@pytest.mark.parametrize("name", golden_names("irs"))
def test_em_irs_elements_golden(S, orc, name):
    """BASELINE.json config 3: `Proposed method/IRS_elements.py:268` em(..., h_initial, N) with its genie stop."""
    meta, g = load_golden(name)
    n_tx, n_rx, M, N = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"]), int(meta["N"])
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g, n_rx)
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    theta = S.em(Y_d, Y_p, int(meta["T_d"]), int(meta["T_p"]), Z_p, PsiTilde_td, table, M, float(meta["varn"]),
                 int(meta["itera"]), g["theta0"].reshape(-1, 1), N, h=g["h"], genie_stop=True)
    assert relerr(theta.reshape(g["theta_ref"].shape), g["theta_ref"]) < RTOL


@pytest.mark.parametrize("name", golden_names("multi"))
def test_multi_detector_golden(S, orc, name):
    meta, g = load_golden(name)
    n_tx, n_rx, M = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    T_d, T_p, varn, itera = int(meta["T_d"]), int(meta["T_p"]), float(meta["varn"]), int(meta["itera"])
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g, n_rx)
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    h0 = g["theta0"].reshape(-1, 1)
    stop = "SNR/all_Detectors.py" not in str(meta.get("src", ""))     # that script has no genie stop in em / em_ml
    th = S.em(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, table, M, varn, itera, h0, h=g["h"], genie_stop=stop)
    assert relerr(th.reshape(g["h"].shape), g["theta_em_ref"]) < RTOL
    th = S.em_ml(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, table, M, varn, itera, h0, h=g["h"], genie_stop=stop)
    assert relerr(th.reshape(g["h"].shape), g["theta_ml_ref"]) < RTOL


BATCH_CASES = [
    # N, n_tx, n_rx, M, T_p, T_d, itera, varn, mode   (T_p <= N keeps the "pm" pilot design's LS start
    # well-posed: its DFT rows repeat with period N, see test_garbage_start_stays_finite)
    (32, 2, 2, 4, 32, 58, 10, 0.1, "soft"),      # shipped config 1 shape (N=32, 2x2, QPSK, 10 iterations)
    (32, 1, 8, 4, 16, 60, 6, 0.1, "soft"),       # shipped config 2 shape
    (16, 2, 2, 16, 20, 60, 4, 0.4, "soft"),
    (16, 2, 2, 16, 20, 60, 4, 0.4, "hard"),
    (10, 3, 3, 4, 24, 40, 4, 0.3, "soft"),
    (12, 4, 4, 4, 32, 64, 3, 0.2, "soft"),
    (8, 4, 4, 16, 24, 40, 2, 0.5, "soft"),
    (8, 4, 4, 16, 24, 40, 2, 0.5, "hard"),
    (6, 8, 8, 4, 64, 80, 2, 0.3, "soft"),        # 8x8 QPSK (K = 65536), BASELINE.json config 4
    (6, 8, 8, 4, 64, 80, 2, 0.3, "hard"),
    (5, 6, 8, 4, 40, 50, 3, 0.5, "soft"),
    (4, 5, 5, 16, 30, 10, 2, 0.8, "soft"),       # 5 streams of 16-QAM: K = 2^20
    # small shapes that run the kernels of the headline path end to end (tensor-path effective channel, TMA Gram
    # with its DMMA right-hand-side CTA, task-pipeline Cholesky with the solution vector in shared memory)
    # (T_p = 10 N: the PM.py pilot design repeats with period N and leaves the last RIS element unobserved; every
    # phase row then meets enough independent pilot vectors for pinv() to have a clean rank gap)
    (16, 4, 4, 4, 160, 48, 3, 0.3, "soft"),
    (16, 4, 4, 4, 160, 72, 3, 0.3, "hard"),
    (20, 4, 4, 16, 100, 96, 2, 0.2, "soft"),
    (24, 3, 4, 4, 144, 90, 3, 0.3, "soft"),
    (16, 1, 1, 16, 16, 60, 4, 0.1, "soft"),      # one receive antenna (three zero rows under the Cholesky factor)
    (10, 3, 3, 64, 24, 30, 2, 0.3, "soft"),      # 3 streams of 64-QAM (K = 2^18)
]


@pytest.mark.parametrize("case", BATCH_CASES)
def test_em_batch_matches_oracle(S, orc, case):
    N, n_tx, n_rx, M, T_p, T_d, itera, varn, mode = case
    B = 4 if M ** n_tx <= 4096 else 2      # the oracle enumerates all K hypotheses per symbol
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, B, seed=42, legacy=False)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, mode=mode)
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h,
                     Xd_true=tb.Xd)
    assert (res.status == 0).all() and (res.iters == itera).all()
    for b in range(B):
        ref, tr = orc.em(tb.Yd[b], tb.Yp[b], tb.PsiD[b], tb.PsiP[b], tb.Xp[b], M, varn, itera, theta0=tb.theta0[b],
                         hard=(mode == "hard"), Xd_true=tb.Xd[b], return_trace=True)
        assert relerr(res.theta[b], ref) < RTOL
        assert np.array_equal(res.kstar[b], tr["kstar"])
        nm = orc.nmse(ref, tb.h[b])
        assert abs(res.nmse[b] - nm) <= 5e-5 * nm  # 4 significant figures
        np.testing.assert_allclose(res.llf[b], np.array(tr["llf"]), rtol=1e-8)
        if mode == "soft":
            np.testing.assert_allclose(res.lse[b], np.array(tr["lse"]), rtol=1e-9)


def test_garbage_start_stays_finite(S, orc):
    """N=32, T_p=40 with the Proposed-method pilot design: pinv() of the rank-deficient pilot matrix
    inverts singular values of 3e-14 and the reference's own LS start has norm ~1e13.  The first E-step
    then sees |d2| ~ 1e27 whose rounding error dwarfs varn^2; the posterior must collapse to the
    arg-min hypothesis (as float(beta) underflow does in the reference) instead of producing NaN."""
    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 32, 2, 2, 4, 40, 50, 4, 0.1
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, 4, seed=42, legacy=False)
    assert np.linalg.norm(tb.theta0[0]) > 1e9
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera)
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h)
    assert np.isfinite(res.theta).all() and (res.status == 0).all()
    assert res.nmse.max() < 50.0


def test_zero_start_config1_as_shipped(S, orc):
    """Proposed_method_NMSEvsTp.py as shipped: N=32, 2x2, QPSK, T_d=50, zero start, 10 iterations,
    pilot design exp(-j2pi t n/T_p) + ones row, at its well-posed sweep point T_p=40."""
    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 32, 2, 2, 4, 40, 50, 10, 0.1
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, 3, seed=3, legacy=True, variant="top_tp")
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, zero_start=True)
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, h_true=tb.h)
    for b in range(3):
        ref = orc.em(tb.Yd[b], tb.Yp[b], tb.PsiD[b], tb.PsiP[b], tb.Xp[b], M, varn, itera, theta0=None)
        assert relerr(res.theta[b], ref) < RTOL
        nm = orc.nmse(ref, tb.h[b])
        assert abs(res.nmse[b] - nm) <= 5e-5 * nm


def test_zero_start_and_shared_status(S, orc):
    """theta0 = 0 start of the top-level scripts (Proposed_method_NMSEvsTp.py:45)."""
    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 16, 2, 2, 4, 24, 40, 6, 0.1
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, 3, seed=9, legacy=False, variant="top_tp")
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, zero_start=True)
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, h_true=tb.h)
    for b in range(3):
        ref = orc.em(tb.Yd[b], tb.Yp[b], tb.PsiD[b], tb.PsiP[b], tb.Xp[b], M, varn, itera, theta0=None)
        assert relerr(res.theta[b], ref) < RTOL


@pytest.mark.parametrize("name", golden_names(["pm", "pm_beta"]))
def test_em_pm_golden(S, orc, name):
    """Partitioned EM against the literal PM.py / PM_beta.py (genie stop active, quirks on)."""
    meta, g = load_golden(name)
    n_tx, n_rx, M = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    T_d, T_p, varn, itera = int(meta["T_d"]), int(meta["T_p"]), float(meta["varn"]), int(meta["itera"])
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g, n_rx)
    cons = orc.qam_constellation(M)
    h0 = g["theta0"].reshape(-1, 1)
    pr = int(meta["partition_r"])
    if str(meta["kind"]) == "pm":
        table = orc.hypothesis_table(cons, n_tx)
        th = S.em_pm(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, table, M, varn, itera, h0, g["h"].reshape(-1), n_tx, pr,
                     None, cons)
    else:
        th = S.em_pm_beta(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h0, g["h"].reshape(-1), n_tx, pr,
                          None, cons)
    assert relerr(th.reshape(g["theta_ref"].shape), g["theta_ref"]) < RTOL


PM_CASES = [
    # N, n_tx, n_rx, M, T_p, T_d, itera, varn, mode, partition_r, quirks
    (8, 2, 2, 4, 8, 30, 3, 0.2, "pm", 0, True), (8, 2, 2, 4, 8, 30, 3, 0.2, "pm_beta", 0, True),
    (8, 3, 3, 4, 8, 40, 3, 0.3, "pm_beta", 2, True), (8, 3, 4, 16, 8, 40, 2, 0.5, "pm_beta", 4, False),
    (6, 4, 4, 4, 6, 48, 2, 0.3, "pm", 2, True), (6, 4, 4, 16, 6, 48, 2, 0.6, "pm_beta", 4, False),
    (6, 2, 4, 16, 6, 30, 2, 0.6, "pm_beta", 4, True),   # p+1 = n_tx: no zero-forced streams
    # wide arrays, BASELINE.json configs 4/5: 8x8 16-QAM is only tractable with the partition (p+1 = 2 -> 256 candidates)
    # (T_p >= n_tx: the min-norm LS start has rank <= T_p, below that the zero-forcing matrices are singular)
    (6, 8, 8, 16, 16, 70, 2, 0.6, "pm_beta", 4, False), (6, 8, 8, 16, 16, 70, 2, 0.6, "pm_beta", 4, True),
    (6, 6, 8, 4, 6, 60, 2, 0.4, "pm", 2, True), (5, 5, 5, 64, 5, 40, 2, 0.8, "pm_beta", 6, False),
]


@pytest.mark.parametrize("case", PM_CASES)
def test_em_pm_batch_matches_oracle(S, orc, case):
    N, n_tx, n_rx, M, T_p, T_d, itera, varn, mode, pr, quirks = case
    B = 3
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, B, seed=77, legacy=False)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, mode=mode, partition_r=pr,
                     quirks=quirks, genie_stop=False)
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h)
    for b in range(B):
        ref = orc.em_pm(tb.Yd[b], tb.Yp[b], tb.PsiD[b], tb.PsiP[b], tb.Xp[b], M, varn, itera, tb.theta0[b],
                        h_true=tb.h[b], partition_r=pr, weighted=(mode == "pm_beta"), genie_stop=False,
                        quirks=quirks, how="solve")
        assert relerr(res.theta[b], ref) < 1e-8, (b, relerr(res.theta[b], ref))


@pytest.mark.parametrize("name", golden_names(["multi", "detectors"]))
def test_em_zf_mmse_golden(S, orc, name):
    """em_zf / em_mmse against the literal PMvsMLvsZFvsMMSE.py (genie stop active, all quirks on)."""
    meta, g = load_golden(name)
    n_tx, n_rx, M = int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    T_d, T_p, varn, itera = int(meta["T_d"]), int(meta["T_p"]), float(meta["varn"]), int(meta["itera"])
    Y_d, Y_p, Z_p, PsiTilde_td = _ref_objects(g, n_rx)
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    h0 = g["theta0"].reshape(-1, 1)
    src = str(meta.get("src", ""))
    stop, guard = "SNR/all_Detectors.py" not in src, "all_detectorsvsTd.py" in src   # the scripts differ in the stop rule
    th = S.em_zf(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, table, M, varn, itera, h0, g["h"].reshape(-1), genie_stop=stop,
                 zf_stop_guard=guard)
    assert relerr(th.reshape(g["h"].shape), g["theta_zf_ref"]) < RTOL
    th = S.em_mmse(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, table, M, varn, itera, h0, g["h"].reshape(-1), genie_stop=stop)
    assert relerr(th.reshape(g["h"].shape), g["theta_mmse_ref"]) < RTOL


DETECTOR_CASES = [
    # N, n_tx, n_rx, M, T_p, T_d, itera, varn, mode, quirks
    (8, 2, 2, 4, 8, 30, 3, 0.3, "zf", True), (8, 2, 2, 4, 8, 30, 3, 0.3, "mmse", True),
    (8, 3, 3, 4, 8, 30, 3, 0.5, "zf", False), (6, 4, 4, 16, 6, 40, 2, 0.5, "mmse", False),
    (6, 2, 4, 16, 6, 30, 3, 1.0, "zf", True), (6, 3, 4, 4, 6, 30, 3, 2.0, "mmse", True),
    (6, 8, 8, 4, 16, 70, 2, 0.5, "zf", False), (6, 6, 8, 16, 6, 60, 2, 0.5, "mmse", False),
    (6, 5, 6, 4, 6, 50, 2, 0.5, "mmse", True),
]


@pytest.mark.parametrize("case", DETECTOR_CASES)
def test_em_detector_batch_matches_oracle(S, orc, case):
    N, n_tx, n_rx, M, T_p, T_d, itera, varn, mode, quirks = case
    B = 4
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, B, seed=91, legacy=False)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, mode=mode, quirks=quirks,
                     genie_stop=True)
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h)
    for b in range(B):
        ref, tr = orc.em_detector(tb.Yd[b], tb.Yp[b], tb.PsiD[b], tb.PsiP[b], tb.Xp[b], M, varn, itera, tb.theta0[b],
                                  kind=mode, h_true=tb.h[b], genie_stop=True, quirks=quirks, return_trace=True)
        assert int(res.iters[b]) == tr["iters"]
        assert relerr(res.theta[b], ref) < RTOL


def test_genie_stop_iteration_counts(S, orc):
    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 8, 2, 2, 4, 8, 40, 6, 0.1
    B = 6
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, B, seed=5, legacy=False)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, genie_stop=True)
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h)
    for b in range(B):
        ref, tr = orc.em(tb.Yd[b], tb.Yp[b], tb.PsiD[b], tb.PsiP[b], tb.Xp[b], M, varn, itera, theta0=tb.theta0[b],
                         h_true=tb.h[b], genie_stop=True, return_trace=True)
        assert int(res.iters[b]) == tr["iters"]
        assert relerr(res.theta[b], ref) < RTOL


def test_shared_phase_design_across_batch(S, orc):
    """Deterministic DFT data phases of Proposed_method_NMSEvsTd.py:92-94 are the same for every trial:
    with SBCE_FLAG_PSI_SHARED the phase matrices are passed once ([T][N+1]) and must give the same result
    as the per-trial layout."""
    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 12, 2, 4, 4, 16, 40, 5, 0.2
    B = 5
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, B, seed=4, legacy=False, variant="top_td")
    assert np.array_equal(tb.PsiD[0], tb.PsiD[B - 1]) and np.array_equal(tb.PsiP[0], tb.PsiP[B - 1])
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, zero_start=True)
    full = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, h_true=tb.h)
    import dataclasses

    prob_s = dataclasses.replace(prob, psi_shared=True)
    shared = S.run_host(prob_s, tb.Yd, tb.Yp, tb.PsiD[0].copy(), tb.PsiP[0].copy(), tb.Xp, tb.varn, h_true=tb.h)
    assert np.array_equal(full.theta, shared.theta) and np.array_equal(full.kstar, shared.kstar)
    ref = orc.em(tb.Yd[1], tb.Yp[1], tb.PsiD[1], tb.PsiP[1], tb.Xp[1], M, varn, itera, theta0=None)
    assert relerr(shared.theta[1], ref) < RTOL


def test_shared_pilot_design_only(S, orc):
    """SBCE_FLAG_PSIP_SHARED: the deterministic pilot design is passed once, the random data phases per trial
    (the layout of every `Proposed method/` sweep); must be bit-identical to the per-trial layout, on the host
    route, the device route, the stand-alone M-step and the on-device generator + LS start."""
    import dataclasses

    import torch

    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 12, 4, 4, 16, 60, 48, 3, 0.3
    B = 5
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, B, seed=14, legacy=False, variant="top_tp")
    assert np.array_equal(tb.PsiP[0], tb.PsiP[B - 1]) and not np.array_equal(tb.PsiD[0], tb.PsiD[1])
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera)
    full = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h, Xd_true=tb.Xd)
    prob_s = dataclasses.replace(prob, psip_shared=True)
    sh = S.run_host(prob_s, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP[0].copy(), tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h,
                    Xd_true=tb.Xd)
    for k in ("theta", "kstar", "llf", "lse", "nmse"):
        assert np.array_equal(getattr(full, k), getattr(sh, k)), k
    ref = orc.em(tb.Yd[2], tb.Yp[2], tb.PsiD[2], tb.PsiP[2], tb.Xp[2], M, varn, itera, theta0=tb.theta0[2])
    assert relerr(sh.theta[2], ref) < RTOL
    # device route + generator + LS start with the shared pilot design
    ses, ses_s = S.DeviceSession(prob, B), S.DeviceSession(prob_s, B)
    g, gs = ses.generate(B, varn, seed=3, pilot_design="top"), ses_s.generate(B, varn, seed=3, pilot_design="top")
    assert gs["PsiP"].shape == (T_p, N + 1) and torch.equal(g["PsiP"][3], gs["PsiP"])
    for k in ("Yp", "Yd", "PsiD", "h", "Xp"):
        assert torch.equal(g[k], gs[k]), k
    t0, st = ses.ls_start(g["Yp"], g["PsiP"], g["Xp"])
    t0s, sts = ses_s.ls_start(gs["Yp"], gs["PsiP"], gs["Xp"])
    assert torch.equal(t0, t0s) and int(sts.abs().max()) == 0
    r = ses.run(g["Yd"], g["Yp"], g["PsiD"], g["PsiP"], g["Xp"], g["varn"], theta0=t0, h_true=g["h"])
    rs = ses_s.run(gs["Yd"], gs["Yp"], gs["PsiD"], gs["PsiP"], gs["Xp"], gs["varn"], theta0=t0s, h_true=gs["h"])
    assert torch.equal(r.theta, rs.theta) and torch.equal(r.nmse, rs.nmse)


def test_drivers_on_gpu_match_oracle_runner(S, orc):
    """The sweep drivers through the CUDA library equal the same drivers fed by the oracle."""
    import sys, os

    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_multirank_gloo import oracle_runner

    cfg = S.SweepConfig(N=8, n_tx=2, n_rx=2, M=4, T_p=8, T_d=32, itera=3, monte_iter=6, varn=0.2, mode="hard", seed=3,
                        max_batch=4)
    a = S.nmse_vs_td(cfg, [32, 40])
    b = S.nmse_vs_td(cfg, [32, 40], runner=oracle_runner)
    np.testing.assert_allclose(a["nmse"], b["nmse"], rtol=5e-5)      # 4 significant figures
    np.testing.assert_allclose(a["ser"], b["ser"], rtol=0, atol=0)   # decisions bit-exact -> identical SER
    np.testing.assert_allclose(a["ser_as_coded"], b["ser_as_coded"], rtol=0, atol=0)
    c = S.detectors_vs_snr(S.SweepConfig(N=8, n_tx=2, n_rx=2, M=4, T_p=8, T_d=24, itera=2, monte_iter=4, seed=1,
                                         partition_r=1), [0.0, 10.0])
    assert set(c) == {"pm_beta", "hard", "zf", "mmse", "soft"} and all(np.isfinite(v["nmse"]).all() for v in c.values())


def test_north_star_size_properties(S):
    """N=64, 4x4, 16-QAM (K=65536): too slow for the oracle at full size, so check
    size-independent properties: (a) noiseless data with theta0 = truth is a fixed point of the
    M-step and decisions equal the transmitted symbols; (b) EM does not increase NMSE from the LS start
    at high SNR; (c) hard and soft EM agree when posteriors are collapsed."""
    N, n_tx, n_rx, M, T_p, T_d = 64, 4, 4, 16, 64, 288
    B = 2
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, 1e-4, B, seed=1, legacy=False)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=2, mode="soft")
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, np.full(B, 0.05), theta0=tb.h, h_true=tb.h)
    assert (res.status == 0).all()
    k_true = (tb.idx_d * (M ** np.arange(n_tx - 1, -1, -1))).sum(axis=2)
    assert np.array_equal(res.kstar, k_true.astype(np.int32))
    assert res.nmse.max() < 1e-6
    prob_h = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=2, mode="hard")
    res_h = S.run_host(prob_h, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, np.full(B, 0.05), theta0=tb.h, h_true=tb.h)
    assert relerr(res_h.theta, res.theta) < 1e-9
