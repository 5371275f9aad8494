"""GPU parity at the FULL sizes BASELINE.json names, through the very code paths bench.py times.

* headline (configs[1], N=64, 4x4, 16-QAM, T_p=320, T_d=256, 10 iterations, B=1184, pilot design shared):
  the host-buffer route (two-half pipeline), the device route and the chunked-workspace route must agree
  BITWISE, and trials 0 and 592 (first trial of each half) must match the oracle: theta 1e-9 relative
  Frobenius, decisions bit-exact, NMSE to 4 significant figures, per-iteration log-sums 1e-9.
* the reference's own NMSE curves (unmodified top-level scripts, tests/golden/script_top_*.npz) re-driven
  with sbce.em in place of the reference's em.
* configs[2..4] at their stated sizes (N = 256; 8x8 QPSK; 4x4 64-QAM partition; 8x8 16-QAM at L = 2056).

The oracle needs minutes per trial at these sizes, so its outputs are committed fixtures
(tests/golden/config_*.npz, minted by oracle/make_config_golden.py); every test first proves (SHA-256 of the
integer draws, projections of the floating arrays) that it regenerated the inputs the fixture was minted from.
"""

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

RTOL = 1e-9


def same(a, b):
    """Bitwise-level equality that treats NaN == NaN (lse is NaN in the modes that form no log-sum)."""
    a, b = np.asarray(a), np.asarray(b)
    return np.array_equal(a, b, equal_nan=True) if a.dtype.kind in "fc" else np.array_equal(a, b)


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


def _check_inputs(tb, trials, meta, g):
    from oracle.make_config_golden import check_inputs

    check_inputs(tb, trials, meta["digest"], g["probes"])


def _to_dev(d, dev):
    import torch

    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in d.items()}


def _run_device(S, prob, hin, trials_in_flight, B=None, want_llf=False):
    """Device route on the first B trials of the host dictionary `hin`."""
    import torch

    B = hin["Yd"].shape[0] if B is None else B
    ses = S.DeviceSession(prob, trials_in_flight)
    cut = {k: (v if (k == "PsiP" and v.ndim == 2) else v[:B]) for k, v in hin.items()}
    t = _to_dev(cut, ses.device)
    res = ses.run(t["Yd"], t["Yp"], t["PsiD"], t["PsiP"], t["Xp"], t["varn"],
                  theta0=None if prob.zero_start else t["theta0"], h_true=t["h_true"])
    torch.cuda.synchronize()
    return {k: getattr(res, k).cpu().numpy() for k in ("theta", "kstar", "lse", "nmse", "iters", "status")}


def _check_against_fixture(got_theta, got_kstar, got_nmse, got_lse, g, i, soft, rtol=RTOL):
    assert relerr(got_theta, g["theta_ref"][i]) < rtol, relerr(got_theta, g["theta_ref"][i])
    if g["kstar_ref"].shape[1]:
        assert np.array_equal(got_kstar, g["kstar_ref"][i]), "hard-decision indices must be bit-exact"
    nm = float(g["nmse_ref"][i])
    assert abs(float(got_nmse) - nm) <= 5e-5 * nm, (got_nmse, nm)      # 4 significant figures
    if soft and g["lse_ref"].shape[1]:
        np.testing.assert_allclose(got_lse, g["lse_ref"][i], rtol=1e-9)


# ---------------------------------------------------------------------------
# 1. the configuration bench.py times, through the routes it times
# ---------------------------------------------------------------------------

def test_headline_config_all_routes_bitwise_equal_and_match_oracle(S):
    """Reference: `Proposed method/Proposed_method_NMSEvsTd.py:44-76` (em) scaled to the north-star size."""
    meta, g = load_golden("config_headline_b1184")
    w = S.workloads.HEADLINE
    B, trials = int(meta["B"]), [int(t) for t in meta["trials"]]
    assert B == w.trials_per_step == 1184 and trials == [0, B // 2]
    tb = S.workloads.make_batch(w, B, seed=S.workloads.bench_seed(w, 0))
    _check_inputs(tb, trials, meta, g)
    prob = w.problem(psip_shared=True)
    assert S._lib.load().sbce_host_split_threshold() <= B      # the host route takes its two-half pipeline
    # (a) end-to-end route, pinned host buffers, exactly as bench.py's e2e leg
    hin = S.workloads.host_arrays(w, tb, psip_shared=True, pinned=True)
    hout = S.engine.alloc_host_outputs(prob, B, want=("kstar", "lse", "nmse", "iters", "status"), pinned=True)
    S.engine.run_host(prob, hin["Yd"], hin["Yp"], hin["PsiD"], hin["PsiP"], hin["Xp"], hin["varn"],
                      theta0=hin["theta0"], h_true=hin["h_true"], device=0, out=hout)
    assert (hout.status == 0).all() and (hout.iters == w.itera).all()
    # (b) device route, whole batch in flight, exactly as bench.py's `value` leg
    dev = _run_device(S, prob, hin, B)
    for k in ("theta", "kstar", "lse", "nmse", "iters", "status"):
        assert same(getattr(hout, k), dev[k]), "host route and device route differ in %s" % k
    # (c) chunked workspace: 250 trials through a workspace that holds 100
    chunked = _run_device(S, prob, hin, 100, B=250)
    for k in ("theta", "kstar", "lse", "nmse", "iters", "status"):
        assert same(chunked[k], dev[k][:250]), "chunked workspace differs in %s" % k
    # (d) the oracle, all 10 iterations, first trial of each half
    for i, b in enumerate(trials):
        _check_against_fixture(hout.theta[b], hout.kstar[b], hout.nmse[b], hout.lse[b], g, i, soft=True)
    # EM improved on the LS start (sanity of the operating point)
    nm0 = np.mean([S.nmse(tb.theta0[b], tb.h[b]) for b in range(32)])
    assert hout.nmse[:32].mean() < 0.2 * nm0


def test_bench_dump_outputs_shapes_and_reproducibility(S, tmp_path):
    """`bench.py --dump-outputs` on workload 1 (on-device inputs): two runs with the same arguments write the
    same arrays (same inputs, same results), in the shapes a caller of the device route receives."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    w = S.workloads.WORKLOADS[1]
    B = 64
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--config", "1", "--steps", "2",
                              "--trials-per-step", str(B), "--kernels-only", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
        dumps.append({f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b = dumps
    assert set(a) == {"theta", "kstar", "lse", "nmse", "iters", "status"}
    assert a["theta"].shape == (B, w.L, w.n_rx, 2) and a["kstar"].shape == (B, w.T_d)
    assert all(v.dtype == np.float64 for v in a.values())
    assert (a["status"] == 0).all() and (a["iters"] == w.itera).all()
    for k in a:
        assert same(a[k], b[k]), k


@pytest.mark.parametrize("shared", ["none", "pilots", "all"])
def test_chunked_workspace_small(S, shared):
    """B = 7 trials through a workspace of 3: per-trial, pilot-shared and fully shared phase layouts
    (offset_io must not advance a shared matrix)."""
    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 9, 2, 3, 16, 24, 40, 3, 0.3
    B = 7
    variant = "top_td" if shared == "all" else "top_tp"
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, B, seed=5, legacy=False, variant=variant)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, psi_shared=(shared == "all"),
                     psip_shared=(shared == "pilots"))
    hin = dict(Yd=tb.Yd, Yp=tb.Yp, Xp=tb.Xp, theta0=tb.theta0, h_true=tb.h, varn=tb.varn,
               PsiD=tb.PsiD[0].copy() if shared == "all" else tb.PsiD,
               PsiP=tb.PsiP[0].copy() if shared != "none" else tb.PsiP)

    def run(inflight):
        import torch

        ses = S.DeviceSession(prob, inflight)
        t = _to_dev(hin, ses.device)
        r = ses.run(t["Yd"], t["Yp"], t["PsiD"], t["PsiP"], t["Xp"], t["varn"], theta0=t["theta0"], h_true=t["h_true"])
        torch.cuda.synchronize()
        return {k: getattr(r, k).cpu().numpy() for k in ("theta", "kstar", "lse", "nmse", "iters", "status")}

    full, part = run(B), run(3)
    for k in full:
        assert same(full[k], part[k]), k


def test_host_route_two_half_split_small_problem(S, orc):
    """The two-half pipeline of sbce_em_batch_host at B >= its threshold on a tiny problem: equal to the
    device route bitwise, and to the oracle on the first trial of each half and the last trial."""
    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 4, 2, 2, 4, 12, 16, 2, 0.2
    B = S._lib.load().sbce_host_split_threshold() + 17          # odd count: halves of unequal size
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, B, seed=9, legacy=False, variant="top_tp")
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera)
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h)
    hin = dict(Yd=tb.Yd, Yp=tb.Yp, PsiD=tb.PsiD, PsiP=tb.PsiP, Xp=tb.Xp, theta0=tb.theta0, h_true=tb.h, varn=tb.varn)
    dev = _run_device(S, prob, hin, B)
    for k in ("theta", "kstar", "lse", "nmse", "iters", "status"):
        assert same(getattr(res, k), dev[k]), k
    half = (B + 1) // 2
    for b in (0, half - 1, half, B - 1):
        ref, tr = orc.em(tb.Yd[b], tb.Yp[b], tb.PsiD[b], tb.PsiP[b], tb.Xp[b], M, varn, itera, theta0=tb.theta0[b],
                         return_trace=True)
        assert relerr(res.theta[b], ref) < RTOL and np.array_equal(res.kstar[b], tr["kstar"])


def test_host_route_graph_replay_tracks_new_inputs(S):
    """sbce_em_batch_host replays the kernel schedule of a call from a CUDA graph from the third call with the
    same configuration on (abi.cu: run_half).  The replay must read the CURRENT call's inputs (same pool
    addresses, new data), a changed configuration must not hit a stale graph, and the launch counter must
    report a replayed call like an eager one."""
    engine = S.engine
    N, n_tx, n_rx, M, T_p, T_d, varn, B = 6, 2, 2, 4, 16, 24, 0.3, 48
    sets = [S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn * (1 + i), B, seed=40 + i, legacy=False,
                                          variant="top_tp") for i in range(2)]
    expect = {}
    for itera in (2, 3):
        prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera)
        for i, tb in enumerate(sets):
            hin = dict(Yd=tb.Yd, Yp=tb.Yp, PsiD=tb.PsiD, PsiP=tb.PsiP, Xp=tb.Xp, theta0=tb.theta0, h_true=tb.h,
                       varn=tb.varn)
            expect[(itera, i)] = _run_device(S, prob, hin, B)
    counts = []
    # eager, capture, then replays -- alternating data sets, then a different iteration count, then back
    order = [(2, 0), (2, 1), (2, 0), (2, 1), (2, 0), (3, 1), (3, 0), (3, 1), (2, 1), (3, 0)]
    for itera, i in order:
        tb = sets[i]
        prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera)
        engine.launch_count(reset=True)
        res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h)
        counts.append((itera, engine.launch_count()))
        for k in ("theta", "kstar", "lse", "nmse", "iters", "status"):
            assert same(getattr(res, k), expect[(itera, i)][k]), (itera, i, k)
    for itera in (2, 3):
        c = {n for it, n in counts if it == itera}
        assert len(c) == 1 and min(c) > 0, counts


def test_partitioned_modes_report_no_decisions(S):
    """PM / PM-beta take no joint decision and form no log-sum: kstar must read -1 and lse NaN on every call
    (not whatever the buffers held), and the sweep drivers must not turn them into a symbol error rate."""
    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 8, 2, 2, 4, 8, 30, 2, 0.2
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, 5, seed=77, legacy=False)
    for mode in ("pm", "pm_beta"):
        prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, mode=mode)
        for _ in range(2):
            res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h)
            assert (res.kstar == -1).all() and np.isnan(res.lse).all() and np.isfinite(res.nmse).all()
    cfg = S.SweepConfig(N=8, n_tx=2, n_rx=2, M=4, T_p=8, T_d=24, itera=2, monte_iter=4, seed=1, partition_r=1)
    out = S.detectors_vs_snr(cfg, [0.0, 10.0], modes=("pm_beta", "zf"))
    assert np.isnan(out["pm_beta"]["ser"]).all() and np.isfinite(out["pm_beta"]["nmse"]).all()
    assert np.isfinite(out["zf"]["ser"]).all()
    # detector modes do decide; lse stays NaN there
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, mode="zf")
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h)
    assert (res.kstar >= 0).all() and np.isnan(res.lse).all()


def test_session_on_a_device_that_is_not_current(S):
    """DeviceSession(device=cuda:1) while cuda:0 is current must launch on cuda:1 (needs two GPUs)."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    N, n_tx, n_rx, M, T_p, T_d, itera, varn = 6, 2, 2, 4, 12, 20, 2, 0.3
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, varn, 3, seed=2, legacy=False)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera)
    hin = dict(Yd=tb.Yd, Yp=tb.Yp, PsiD=tb.PsiD, PsiP=tb.PsiP, Xp=tb.Xp, theta0=tb.theta0, h_true=tb.h, varn=tb.varn)
    outs = []
    for d in (0, 1):
        torch.cuda.set_device(0)
        ses = S.DeviceSession(prob, 3, device="cuda:%d" % d)
        t = _to_dev(hin, ses.device)
        r = ses.run(t["Yd"], t["Yp"], t["PsiD"], t["PsiP"], t["Xp"], t["varn"], theta0=t["theta0"], h_true=t["h_true"])
        torch.cuda.synchronize(ses.device)
        assert r.theta.device.index == d and torch.cuda.current_device() == 0
        outs.append(r.theta.cpu().numpy())
    assert np.array_equal(outs[0], outs[1])
    res = S.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=tb.theta0, h_true=tb.h, device=1)
    assert torch.cuda.current_device() == 0 and np.array_equal(res.theta, outs[0])


# ---------------------------------------------------------------------------
# 2. the reference's own curves, re-driven through the GPU estimator
# ---------------------------------------------------------------------------

def _dense_Zp(PsiP, Xp, n_rx):
    Wp = (PsiP[:, :, None] * Xp[:, None, :]).reshape(PsiP.shape[0], -1)
    return [np.kron(Wp[t][None, :], np.eye(n_rx, dtype=np.complex128)) for t in range(Wp.shape[0])]


def _cols(A):
    return [A[t].reshape(-1, 1) for t in range(A.shape[0])]


def test_script_top_td_curve_through_gpu(S, orc):
    """`Proposed_method_NMSEvsTd.py:116-161`, unmodified, np.random.seed(0): its `mse` array is the fixture.
    The loop is re-driven in the script's draw order with sbce.em (reference signature, dense Z_p list, zero
    start, 20 iterations) in place of the reference's em; well-posed points to 4 significant figures."""
    meta, g = load_golden("script_top_td_s0")
    N, n_tx, n_rx, M = int(meta["N"]), int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    T_p, varn, itera = int(meta["T_p"]), float(meta["varn"]), int(meta["itera"])
    rs = np.random.RandomState(int(meta["seed"]))
    h = orc.channel_vector(n_tx, n_rx, N, 1.0, rs, flatten="C")
    _, Xp = orc.draw_symbols(n_tx, M, T_p, rs)
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    mse = []
    for T_d in meta["T_d"]:
        T_d = int(T_d)
        _, Xd = orc.draw_symbols(n_tx, M, T_d, rs)
        PsiP, PsiD = orc.irs_phases(T_p, T_d, N, rs, variant="top_td")
        Yp, Yd, _ = orc.received_signals(PsiP, PsiD, Xp, Xd, h, varn, rs)
        theta = S.em(_cols(Yd), _cols(Yp), T_d, T_p, _dense_Zp(PsiP, Xp, n_rx), PsiD.T.copy(), table, M, varn, itera)
        mse.append(S.nmse(theta, h))
    ref = np.asarray(g["mse_ref"]).reshape(-1)
    L = (N + 1) * n_tx
    ok = np.array([T_p + int(td) >= 1.3 * L for td in meta["T_d"]])
    assert ok.sum() == 8
    np.testing.assert_allclose(np.array(mse)[ok], ref[ok], rtol=5e-5)


def test_script_top_tp_curve_through_gpu(S, orc):
    """`Proposed_method_NMSEvsTp.py:103-151`, unmodified, np.random.seed(0), re-driven with sbce.em; parity on
    the sweep points with T_p + T_d >= 1.3 L (the others solve a numerically singular system by LU,
    SURVEY.md section 7 hard part 1 -- there the GPU must flag or at least stay finite)."""
    meta, g = load_golden("script_top_tp_s0")
    N, n_tx, n_rx, M = int(meta["N"]), int(meta["n_tx"]), int(meta["n_rx"]), int(meta["M"])
    T_d, varn, itera = int(meta["T_d"]), float(meta["varn"]), int(meta["itera"])
    L = (N + 1) * n_tx
    rs = np.random.RandomState(int(meta["seed"]))
    h = orc.channel_vector(n_tx, n_rx, N, 1.0, rs, flatten="C")
    _, Xd = orc.draw_symbols(n_tx, M, T_d, rs)
    table = orc.hypothesis_table(orc.qam_constellation(M), n_tx)
    ref = np.asarray(g["mse_ref"]).reshape(-1)
    checked = 0
    for i, T_p in enumerate(meta["T_p"]):
        T_p = int(T_p)
        PsiP, PsiD = orc.irs_phases(T_p, T_d, N, rs, variant="top_tp")
        _, Xp = orc.draw_symbols(n_tx, M, T_p, rs)
        Yp, Yd, _ = orc.received_signals(PsiP, PsiD, Xp, Xd, h, varn, rs)
        theta = S.em(_cols(Yd), _cols(Yp), T_d, T_p, _dense_Zp(PsiP, Xp, n_rx), PsiD.T.copy(), table, M, varn, itera)
        if T_p + T_d >= 1.3 * L:
            got = S.nmse(theta, h)
            assert abs(got - ref[i]) <= 5e-5 * ref[i], (T_p, got, ref[i])
            checked += 1
    assert checked >= 2


# ---------------------------------------------------------------------------
# 3. BASELINE.json configs[2..4] at their stated sizes
# ---------------------------------------------------------------------------

CONFIG_FIXTURES = [("config_3_n256", 3), ("config_4_8x8qpsk", 4), ("config_41_64qam_pm", 41), ("config_5_l2056", 5)]


@pytest.mark.parametrize("name,key", CONFIG_FIXTURES)
def test_baseline_configs_at_size_match_oracle(S, name, key):
    """config 3: `Proposed method/IRS_elements.py:353-430` at N = 256 (L = 514); config 4:
    `Proposed method/PMvsMLvsZFvsMMSE.py:342-416` 8x8 QPSK (K = 65536, hard decisions) and the 4x4 64-QAM
    partitioned leg (4096 candidates); config 5: 8x8 16-QAM PM-beta at N = 256 (L = 2056, 67 MB normal
    matrix per trial).  Host route and device route, both against the committed oracle output."""
    meta, g = load_golden(name)
    w = S.workloads.WORKLOADS[key]
    assert int(meta["workload"]) == key
    B, trials = int(meta["B"]), [int(t) for t in meta["trials"]]
    tb = S.workloads.make_batch(w, B)
    _check_inputs(tb, trials, meta, g)
    prob = w.problem(psip_shared=True)
    hin = S.workloads.host_arrays(w, tb, psip_shared=True)
    res = S.run_host(prob, hin["Yd"], hin["Yp"], hin["PsiD"], hin["PsiP"], hin["Xp"], hin["varn"],
                     theta0=None if w.zero_start else hin["theta0"], h_true=hin["h_true"])
    assert (res.status == 0).all() and (res.iters == w.itera).all()
    dev = _run_device(S, prob, hin, 1)                      # one trial in flight: chunked when B = 2
    assert np.array_equal(res.theta, dev["theta"]) and np.array_equal(res.kstar, dev["kstar"])
    # partitioned modes: 1e-8, the bar of test_em_pm_batch_matches_oracle (per-symbol ZF solves by Cholesky here,
    # by pinv / inv in the reference; PM.py:66,98)
    rtol = RTOL if w.mode in ("soft", "hard") else 1e-8
    for i, b in enumerate(trials):
        _check_against_fixture(res.theta[b], res.kstar[b], res.nmse[b], res.lse[b], g, i, soft=(w.mode == "soft"),
                               rtol=rtol)
