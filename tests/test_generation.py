"""On-device input generation + LS start (SURVEY.md section 8f-1).

CPU part: the numpy restatement of the generator (oracle/philox.py) against the Random123
known-answer vectors of Philox4x32-10 and against the signal model's moments.
GPU part: the CUDA generator element by element against that restatement (symbol indices
bit-exact), sharding invariance, the LS start against numpy's pinv, and the fully on-device
sweep driver against the oracle fed with the very same (copied-back) trials."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mstep_reference as mr  # noqa: E402


def relerr(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b)))


def test_philox_known_answers():
    """Random123 kat_vectors, philox4x32 10 rounds."""
    from oracle.philox import philox4x32_10

    def hx(t):
        return ["%08x" % int(v) for v in t]

    assert hx(philox4x32_10(0, 0, 0, 0, 0, 0)) == ["6627e8d5", "e169c58d", "bc57ac4c", "9b00dbd8"]
    f = 0xFFFFFFFF
    assert hx(philox4x32_10(f, f, f, f, f, f)) == ["408f276d", "41c83b0e", "a20bc7c6", "6d5451fd"]
    assert hx(philox4x32_10(0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344, 0xA4093822, 0x299F31D0)) == \
        ["d16cfe09", "94fdcceb", "5001e420", "24126ea1"]


def test_generator_restatement_follows_the_signal_model():
    """Moments and structure of one generated trial (reference: Proposed method/PM.py:11-40,119-148)."""
    from oracle import em_numpy as orc
    from oracle.philox import generate_trial

    N, n_tx, n_rx, M, T_p, T_d, varn = 24, 2, 3, 16, 400, 600, 0.25
    g = generate_trial(N, n_tx, n_rx, M, T_p, T_d, varn, seed=5, trial=11)
    cons = orc.qam_constellation(M)
    assert np.array_equal(g["Xd"], cons[g["idx_d"]]) and np.array_equal(g["Xp"], cons[g["idx_p"]])
    counts = np.bincount(g["idx_d"].reshape(-1), minlength=M)
    assert counts.min() > 0.5 * counts.mean()                                   # all 16 points drawn, roughly uniform
    assert np.allclose(g["PsiD"][:, 0], 1.0) and np.allclose(np.abs(g["PsiD"]), 1.0)
    assert np.allclose(g["PsiP"][:, N], 0.0) and np.allclose(g["PsiP"][:, 0], 1.0)  # quirk Q3: last element off
    nz = np.concatenate((g["noise_p"].reshape(-1), g["noise_d"].reshape(-1)))
    assert abs(np.mean(np.abs(nz) ** 2) / varn - 1.0) < 0.05 and abs(nz.mean()) < 0.03
    assert abs(np.mean(nz.real ** 2) / np.mean(nz.imag ** 2) - 1.0) < 0.1
    # cascaded channel: Theta[(n+1)*n_tx + j, r] = H_BS[n, j] * H_SU[r, n]  => rank-one blocks
    blk = g["h"].reshape(N + 1, n_tx, n_rx)[3]
    assert np.linalg.matrix_rank(blk, tol=1e-10) == 1
    # a different trial index or seed gives different data
    g2 = generate_trial(N, n_tx, n_rx, M, T_p, T_d, varn, seed=5, trial=12)
    assert not np.array_equal(g["idx_d"], g2["idx_d"])


# ---------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def S(cuda_device):
    import sbce

    sbce._lib.require_device()
    return sbce


GEN_CASES = [
    # N, n_tx, n_rx, M, T_p, T_d, varn, pilot_design, data_phases
    (8, 2, 2, 4, 12, 30, 0.1, "pm", "random"), (16, 4, 4, 16, 20, 40, 0.5, "top", "random"),
    (9, 3, 2, 64, 7, 11, 2.0, "top", "dft"), (6, 8, 8, 4, 16, 20, 0.3, "pm", "random"), (33, 1, 6, 16, 5, 9, 1.0, "pm", "dft"),
]


@gpu
@pytest.mark.parametrize("case", GEN_CASES)
def test_device_generator_matches_restatement(S, case):
    from oracle.philox import generate_trial

    N, n_tx, n_rx, M, T_p, T_d, varn, pilot, phases = case
    B, seed, trial0 = 3, 77, 1 << 33          # trial counter beyond 32 bits
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=1, mode="hard")
    ses = S.DeviceSession(prob, B)
    tb = {k: v.cpu().numpy() for k, v in ses.generate(B, varn, seed, trial0=trial0, pilot_design=pilot,
                                                      data_phases=phases).items()}
    for b in range(B):
        g = generate_trial(N, n_tx, n_rx, M, T_p, T_d, varn, seed, trial0 + b, pilot, phases)
        assert np.array_equal(tb["Xd"][b], g["Xd"]) and np.array_equal(tb["Xp"][b], g["Xp"])   # integer work: bit-exact
        for k in ("h", "PsiP", "PsiD", "Yp", "Yd"):
            assert np.abs(tb[k][b] - g[k]).max() < 1e-12 * max(1.0, np.abs(g[k]).max()), k


@gpu
@pytest.mark.parametrize("case", [(8, 2, 2, 4, 12, 30, 0.1, "pm", "random"), (5, 3, 4, 16, 9, 14, 0.4, "top", "dft")])
def test_device_generator_no_direct_link(S, case):
    """All N + 1 phase rows are RIS elements (no ones row, no H_BU): "direct vs non direct - T_pv s nmse.py"."""
    from oracle import em_numpy as orc
    from oracle.philox import generate_trial

    N, n_tx, n_rx, M, T_p, T_d, varn, pilot, phases = case
    B, seed = 2, 5
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=3, zero_start=True)
    ses = S.DeviceSession(prob, B)
    dv = ses.generate(B, varn, seed, pilot_design=pilot, data_phases=phases, direct_link=False)
    tb = {k: v.cpu().numpy() for k, v in dv.items()}
    for b in range(B):
        g = generate_trial(N, n_tx, n_rx, M, T_p, T_d, varn, seed, b, pilot, phases, direct_link=False)
        assert np.array_equal(tb["Xd"][b], g["Xd"]) and np.array_equal(tb["Xp"][b], g["Xp"])
        for k in ("h", "PsiP", "PsiD", "Yp", "Yd"):
            assert np.abs(tb[k][b] - g[k]).max() < 1e-12 * max(1.0, np.abs(g[k]).max()), k
        assert np.allclose(np.abs(tb["PsiD"][b]), 1.0) and np.allclose(np.abs(tb["PsiP"][b]), 1.0)
    res = ses.run(dv["Yd"], dv["Yp"], dv["PsiD"], dv["PsiP"], dv["Xp"], dv["varn"], h_true=dv["h"])
    theta = res.theta.cpu().numpy()
    for b in range(B):
        ref = orc.em(tb["Yd"][b], tb["Yp"][b], tb["PsiD"][b], tb["PsiP"][b], tb["Xp"][b], M, varn, 3, theta0=None)
        assert relerr(theta[b], ref) < 1e-9


@gpu
def test_generation_is_sharding_invariant(S):
    N, n_tx, n_rx, M, T_p, T_d = 8, 2, 2, 16, 12, 20
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=1)
    ses = S.DeviceSession(prob, 6)
    whole = ses.generate(6, 0.2, seed=9, trial0=100)
    a, b = ses.generate(2, 0.2, seed=9, trial0=100), ses.generate(4, 0.2, seed=9, trial0=102)
    for k in ("h", "Xd", "Xp", "PsiD", "Yp", "Yd"):
        both = np.concatenate((a[k].cpu().numpy(), b[k].cpu().numpy()))
        assert np.array_equal(whole[k].cpu().numpy(), both), k


@gpu
@pytest.mark.parametrize("case", [(8, 2, 2, 4, 8, "pm"), (8, 2, 2, 4, 40, "top"), (16, 4, 4, 16, 30, "top"),
                                  (16, 4, 4, 16, 90, "top"), (6, 8, 8, 4, 20, "pm"), (12, 3, 4, 16, 36, "top"),
                                  (64, 4, 4, 16, 320, "top")])
def test_ls_start_matches_pinv(S, case):
    """h_initial = pinv(vstack Z_p) vstack Y_p (PM.py:147), both for T_p < L (min-norm) and T_p >= L."""
    N, n_tx, n_rx, M, T_p, pilot = case
    B = 3
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=8, itera=1)
    ses = S.DeviceSession(prob, B)
    tb = ses.generate(B, 0.1, seed=3, pilot_design=pilot)
    th0, st = ses.ls_start(tb["Yp"], tb["PsiP"], tb["Xp"])
    th0, st = th0.cpu().numpy(), st.cpu().numpy()
    assert (st == 0).all()
    for b in range(B):
        PsiP, Xp, Yp = (tb[k][b].cpu().numpy() for k in ("PsiP", "Xp", "Yp"))
        Wp = (PsiP[:, :, None] * Xp[:, None, :]).reshape(T_p, -1)
        ref = np.linalg.pinv(Wp) @ Yp
        cond = np.linalg.cond(Wp)
        assert relerr(th0[b], ref) < max(1e-9, 1e-14 * cond * cond), (relerr(th0[b], ref), cond)


@gpu
@pytest.mark.parametrize("case", [(8, 2, 2, 40, None), (16, 4, 4, 90, None), (64, 4, 4, 320, None),
                                  (6, 8, 8, 70, None), (16, 4, 4, 90, 1e-6), (6, 8, 8, 70, 1e-6)])
def test_ls_start_primal_route_backward_error(S, case):
    """T_p >= L with distinct, non-zero phase columns: the LS start solves the pilot normal equations
    (W^H W) theta = W^H y_p with k_chol_solve, unscaled.  Backward error against the exact system within
    tau(L) = 8 L u, also with column 2 a near-duplicate of column 1 (relative offset eps: cond ~ 1 / eps^2)."""
    import torch

    N, n_tx, n_rx, T_p, eps = case
    B = 2
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=4, T_p=T_p, T_d=8, itera=1)
    ses = S.DeviceSession(prob, B)
    rng = np.random.default_rng(N + T_p)
    PsiP = np.exp(2j * np.pi * rng.random((B, T_p, N + 1)))
    if eps is not None:
        PsiP[:, :, 2] = PsiP[:, :, 1] * np.exp(1j * eps * rng.standard_normal((B, T_p)))
    Xp = S.qam.constellation(16)[rng.integers(0, 16, (B, T_p, n_tx))]
    Yp = rng.standard_normal((B, T_p, n_rx)) + 1j * rng.standard_normal((B, T_p, n_rx))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    th0, st = ses.ls_start(t(Yp), t(PsiP), t(Xp))
    th0, st = th0.cpu().numpy(), st.cpu().numpy()
    assert st.tolist() == [0] * B
    L = prob.L
    for b in range(B):
        G, Bm = mr.design_system(PsiP[b], Xp[b], Yp[b])
        if eps is not None:
            assert np.linalg.cond(G.astype(np.complex128)) > 1e8
        eta = mr.backward_error(G, Bm, th0[b])
        assert eta <= mr.tau(L), (eta, mr.tau(L))


@gpu
def test_ls_start_structural_rank_deficiency_follows_pinv(S):
    """The reference's pilot designs are rank deficient by construction ("pm": last RIS element off = zero
    column; top-level: the inserted ones row duplicates the n = 0 DFT row).  pinv gives the min-norm solution
    (zero / even split); the device reproduces exactly that by merging identical columns."""
    for pilot, N, n_tx, T_p in (("pm", 8, 2, 24), ("top", 8, 2, 40), ("pm", 16, 3, 60)):
        # 16-QAM: pilot vectors of the repeating "pm" rows are (almost surely) not parallel, so the only rank
        # deficiency is the structural one
        prob = S.Problem(N=N, n_tx=n_tx, n_rx=2, M=16, T_p=T_p, T_d=8, itera=1)
        ses = S.DeviceSession(prob, 2)
        tb = ses.generate(2, 0.1, seed=3, pilot_design=pilot)
        th0, st = ses.ls_start(tb["Yp"], tb["PsiP"], tb["Xp"])
        assert (st.cpu().numpy() == 0).all()
        for b in range(2):
            PsiP, Xp, Yp = (tb[k][b].cpu().numpy() for k in ("PsiP", "Xp", "Yp"))
            Wp = (PsiP[:, :, None] * Xp[:, None, :]).reshape(T_p, -1)
            assert np.linalg.matrix_rank(Wp) == Wp.shape[1] - n_tx       # one zero / duplicated RIS column
            ref = np.linalg.pinv(Wp) @ Yp
            assert relerr(th0[b].cpu().numpy(), ref) < 1e-9
        if pilot == "pm":
            assert float(th0[:, N * n_tx:, :].abs().max()) == 0.0     # switched-off element: exactly zero


@gpu
def test_ls_start_flags_unstructured_rank_deficiency(S):
    """Two identical pilot rows (same phases, same symbols) in a block with T_p < L: K = W W^H is exactly
    singular, numpy's pinv would invert rounding noise (cf. test_garbage_start_stays_finite); the device
    flags the trial (pivot below 1e-13 of the largest one) and leaves the other trial alone."""
    import torch

    prob = S.Problem(N=6, n_tx=2, n_rx=2, M=4, T_p=8, T_d=8, itera=1)
    ses = S.DeviceSession(prob, 2)
    tb = ses.generate(2, 0.1, seed=3, pilot_design="top")
    PsiP, Xp = tb["PsiP"].clone(), tb["Xp"].clone()
    PsiP[0, 5] = PsiP[0, 2]
    Xp[0, 5] = Xp[0, 2]
    _, st = ses.ls_start(tb["Yp"], PsiP, Xp)
    torch.cuda.synchronize()
    assert st.cpu().numpy().tolist() == [1, 0]


@gpu
@pytest.mark.parametrize("mode", ["soft", "hard"])
def test_on_device_pipeline_matches_oracle_on_the_same_trials(S, mode):
    """generate -> LS start -> EM, all on the GPU, against the oracle run on the copied-back inputs."""
    from oracle import em_numpy as orc

    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 12, 2, 2, 16, 30, 50, 4, 0.3
    B = 4
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, mode=mode)
    ses = S.DeviceSession(prob, B)
    tb = ses.generate(B, varn, seed=21, pilot_design="top")
    th0, st = ses.ls_start(tb["Yp"], tb["PsiP"], tb["Xp"])
    res = ses.run(tb["Yd"], tb["Yp"], tb["PsiD"], tb["PsiP"], tb["Xp"], tb["varn"], theta0=th0, h_true=tb["h"])
    h = {k: v.cpu().numpy() for k, v in tb.items()}
    theta, kstar, nm = res.theta.cpu().numpy(), res.kstar.cpu().numpy(), res.nmse.cpu().numpy()
    for b in range(B):
        Wp = (h["PsiP"][b][:, :, None] * h["Xp"][b][:, None, :]).reshape(T_p, -1)
        t0 = np.linalg.pinv(Wp) @ h["Yp"][b]
        ref, tr = orc.em(h["Yd"][b], h["Yp"][b], h["PsiD"][b], h["PsiP"][b], h["Xp"][b], M, varn, itera, theta0=t0,
                         hard=(mode == "hard"), return_trace=True)
        assert relerr(theta[b], ref) < 1e-9
        assert np.array_equal(kstar[b], tr["kstar"])
        assert abs(nm[b] - orc.nmse(ref, h["h"][b])) <= 5e-5 * orc.nmse(ref, h["h"][b])


@gpu
def test_on_device_sweep_driver(S):
    """SweepConfig(on_device=True): the curve equals the one recomputed from the same Philox trials through
    the oracle; SER figures are exact; result does not depend on max_batch."""
    from oracle import em_numpy as orc
    from oracle.philox import generate_trial

    cfg = S.SweepConfig(N=8, n_tx=2, n_rx=2, M=4, T_p=8, T_d=32, itera=3, monte_iter=10, varn=0.5, mode="hard", seed=3,
                        max_batch=4, variant="top_tp", on_device=True)
    xs = [24, 32]
    a = S.nmse_vs_td(cfg, xs)
    import dataclasses

    b = S.nmse_vs_td(dataclasses.replace(cfg, max_batch=7), xs)
    np.testing.assert_allclose(a["nmse"], b["nmse"], rtol=1e-13)
    assert np.array_equal(a["ser"], b["ser"])
    cons = orc.qam_constellation(cfg.M)
    for i, T_d in enumerate(xs):
        nm, err, coded = [], 0, 0.0
        for t in range(cfg.monte_iter):
            g = generate_trial(cfg.N, cfg.n_tx, cfg.n_rx, cfg.M, cfg.T_p, T_d, cfg.varn, cfg.seed * 1000003 + i, t, "top",
                               "random")
            t0 = np.linalg.pinv(g["Wp"]) @ g["Yp"]
            ref, tr = orc.em(g["Yd"], g["Yp"], g["PsiD"], g["PsiP"], g["Xp"], cfg.M, cfg.varn, cfg.itera, theta0=t0,
                             hard=True, return_trace=True)
            nm.append(orc.nmse(ref, g["h"]))
            xest = cons[orc.hypothesis_digits(tr["kstar"], cfg.M, cfg.n_tx)]
            err += np.count_nonzero(g["Xd"] - xest)
            coded += orc.ser_as_coded(g["Xd"], xest)
        assert abs(a["nmse"][i] - np.mean(nm)) <= 5e-5 * np.mean(nm)          # 4 significant figures
        assert a["ser"][i] == err / (cfg.monte_iter * T_d * cfg.n_tx)
        assert abs(a["ser_as_coded"][i] - coded / cfg.monte_iter) < 1e-12


@gpu
def test_baseline_json_configs_through_the_on_device_drivers(S):
    """The sweep shapes BASELINE.json names beyond the bench line, end to end on the GPU (generation, LS start,
    EM, accumulation) at a handful of trials: config 3 (`IRS_elements.py`: N = 16 ... 256, 2x2 QPSK, well-posed
    T_p + T_d >= 1.3 L, SURVEY 8d) and config 4 (`PMvsMLvsZFvsMMSE.py` / `SNR/all_Detectors.py`: 8x8 QPSK with the
    exhaustive tree, 4x4 64-QAM with the PM partition p+1 = 2 -> 4096 candidates, SNR sweep, SER from hard decisions)."""
    import math

    # ---- config 3
    for N in (16, 64, 256):
        L = (N + 1) * 2
        T_p = 20 * math.ceil(N / 15)
        T_d = max(32, int(1.3 * L) - T_p + 8)
        cfg = S.SweepConfig(N=N, n_tx=2, n_rx=2, M=4, T_p=T_p, T_d=T_d, itera=5, monte_iter=6, varn=1.0, mode="soft", seed=1,
                            variant="top_tp", on_device=True)
        r = S.nmse_vs_N(cfg, [N])
        assert r["n_valid"][0] == 6 and np.isfinite(r["nmse"]).all() and r["nmse"][0] < 1.0, (N, r)
    # ---- config 4: 8x8 QPSK, exhaustive 65536-leaf tree, hard decisions -> SER vs SNR
    cfg = S.SweepConfig(N=16, n_tx=8, n_rx=8, M=4, T_p=160, T_d=64, itera=3, monte_iter=4, mode="hard", seed=2,
                        variant="top_tp", on_device=True)
    r = S.ser_vs_snr(cfg, [0.0, 10.0, 20.0])
    assert np.isfinite(r["nmse"]).all() and (r["n_valid"] == 4).all()
    assert r["nmse"][2] < r["nmse"][0] and r["ser"][2] <= r["ser"][0] and r["ser"][2] < 0.05
    # ---- config 4: 4x4 64-QAM with the partition (p = int(6 / log2 64) = 1 -> 64^2 = 4096 candidates per symbol)
    cfg = S.SweepConfig(N=16, n_tx=4, n_rx=4, M=64, T_p=80, T_d=48, itera=2, monte_iter=4, mode="pm_beta", partition_r=6,
                        quirks=False, seed=3, variant="top_tp", on_device=True)
    r = S.nmse_vs_snr(cfg, [10.0, 30.0])
    assert np.isfinite(r["nmse"]).all() and r["nmse"][1] < r["nmse"][0]
    # ---- config 5 shape at toy trial count: 8x8 16-QAM, partitioned (2^32 joint hypotheses are out of reach
    # of any exhaustive method), N = 32
    cfg = S.SweepConfig(N=32, n_tx=8, n_rx=8, M=16, T_p=320, T_d=32, itera=2, monte_iter=3, mode="pm_beta", partition_r=4,
                        quirks=False, seed=4, variant="top_tp", on_device=True)
    r = S.nmse_vs_snr(cfg, [20.0])
    assert np.isfinite(r["nmse"]).all() and r["n_valid"][0] == 3
