"""Per-kernel coverage and batch hygiene of the CUDA path.

* A Python mirror of the launch predicates maps a case of the parity tables (test_gpu_parity.py) to the kernel
  instantiation and runtime branch it runs; a CPU test asserts the tables reach every instantiated variant, a GPU
  test checks the mirror against the kernel names torch.profiler records.
* Mixed batches: per-trial noise variances, starts and bad trials (unobserved RIS element, NaN data) in one call;
  every regular trial must be bitwise the trial run alone, match the oracle at its own varn, and the bad ones
  must carry their status bit without leaking into their neighbours.
* Dirty workspaces and output buffers: results must not depend on what the memory held before the call.
* The shape limit: the largest admitted phase rows must launch, and the workspace query must admit exactly the
  shapes whose Gram launch fits in shared memory."""
import os
import re
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_parity import BATCH_CASES, DETECTOR_CASES, ESTEP_CASES, MSTEP_CASES, PM_CASES, relerr  # noqa: E402

import sbce  # noqa: E402

# ---------------------------------------------------------------------------
# mirror of the launchers (csrc/*.cu); sizes in bytes, one complex128 = 16
# ---------------------------------------------------------------------------
CPLX = 16
SMEM_CAP = 227 * 1024
SQM = {4: 2, 16: 4, 64: 8}


def heff_variant(N, n_tx, n_rx):
    """estep.cu launch_heff_qr / run_heff (:1039) / run_heff_rows (:1104) -> (kernel, branch)."""
    N1, L = N + 1, (N + 1) * n_tx
    if n_tx >= 5:
        return "k_heff_qr_rows<%d>" % n_tx, "rows"
    NC = n_tx * n_rx
    NT, KP = (NC + 7) // 8, (N1 + 7) & ~7
    smem_mma = CPLX * (KP * (NT * 8 + 2) + 4 * 32 * (NC + 1))
    if NC >= 8 and N1 >= 16 and smem_mma <= 100 * 1024:
        return "k_heff_qr_mma<%d, %d>" % (n_tx, n_rx), "mma"
    return "k_heff_qr<%d, %d>" % (n_tx, n_rx), ("smem" if CPLX * L * n_rx <= 64 * 1024 else "global")


def enum_instantiated(n_tx, sqm):
    """estep.cu run_enum_ntx (:1126) for n_tx <= 4, run_enum_wide (:1116) for 5..8 (2^24 leaves at most)."""
    return sqm in ((2, 4, 8) if n_tx <= 4 else (2, 4) if n_tx <= 6 else (2,))


def enum_variant(n_tx, M, hard):
    """estep.cu run_enum (:1080): k_enum<NTX, SQM, HARD, 4 warps>."""
    assert enum_instantiated(n_tx, SQM[M])
    return "k_enum<%d, %d, %d, 4>" % (n_tx, SQM[M], int(hard))


def gram_variant(N, n_tx, n_rx):
    """mstep.cu gram_smem (:618), the size computation of run_gram_scalar / run_gram4 / run_gram_wide
    -> (kernel, dynamic shared memory of the launch)."""
    N1 = N + 1
    rhs1 = CPLX * 8 * (N1 + n_tx * n_rx + 2)          # right-hand-side CTA: one 8-symbol MMA step
    rhs_want = 2 * rhs1
    if n_tx <= 3:
        tc = 16
        while tc > 2 and CPLX * 2 * tc * (N1 + n_tx * n_tx) > 100 * 1024:
            tc >>= 1
        pair, rhs_want, kernel = CPLX * 2 * tc * (N1 + n_tx * n_tx), rhs1, "k_gram<%d>" % n_tx
    elif n_tx == 4 and CPLX * 4 * 16 * (N1 + 16) <= 160 * 1024:
        pair, kernel = CPLX * 4 * 16 * (N1 + 16), "k_gram_tma4"
    else:
        tc = 32
        while tc > 8 and CPLX * 2 * tc * (N1 + n_tx * n_tx) > 100 * 1024:
            tc >>= 1
        pair, kernel = CPLX * 2 * tc * (N1 + n_tx * n_tx), "k_gram_mma<%d>" % n_tx
    smem = max(pair, rhs_want)
    if smem > SMEM_CAP:
        smem = max(pair, rhs1)
    return kernel, smem


def chol_variant(N, n_tx, n_rx):
    """chol.cu launch_chol_solve (:441): solution vector in shared memory or in global scratch."""
    L = (N + 1) * n_tx
    Lp = (L + 7) & ~7
    Ltot = Lp + ((n_rx + 3) & ~3)
    npan, nrb = (Lp + 15) // 16, (Ltot + 15) // 16 + 1
    fixed = CPLX * 4 * 16 * 17 + 4 * (nrb + 2 * npan + 2)
    return "k_chol_solve", ("smem" if fixed + CPLX * Lp * n_rx <= 24 * 1024 else "global")


def admitted(N, n_tx, n_rx):
    """abi.cu make_dims (shape part) with mstep.cu gram_supports (:644)."""
    if not (1 <= n_tx <= 8 and 1 <= n_rx <= 8) or (n_tx <= 4 and n_rx not in (1, 2, 3, 4, 6, 8)):
        return False
    return CPLX * 16 * (N + 1 + n_tx * n_tx) <= SMEM_CAP and gram_variant(N, n_tx, n_rx)[1] <= SMEM_CAP


def pm_variant(n_tx, mode):
    """pm.cu launch_pm_stats: k_pm_stats (PM, PM-beta) or k_det_stats (ZF, MMSE), <4> for n_tx <= 4 and <8> for the
    wide arrays."""
    return "%s<%d>" % ("k_det_stats" if mode in ("zf", "mmse") else "k_pm_stats", 4 if n_tx <= 4 else 8)


def covered_items():
    """item -> list of parity-table rows that reach it."""
    items = {}

    def add(key, row):
        items.setdefault(key, []).append(row)

    for c in ESTEP_CASES:
        N, n_tx, n_rx, M = c[:4]
        add(("heff", heff_variant(N, n_tx, n_rx)[1]), ("estep", c))
        for hard in (False, True):
            add(("enum", enum_variant(n_tx, M, hard)), ("estep", c))
    for c in MSTEP_CASES:
        N, n_tx, n_rx = c[:3]
        add(("gram", gram_variant(N, n_tx, n_rx)[0]), ("mstep", c))
        add(("chol", chol_variant(N, n_tx, n_rx)[1]), ("mstep", c))
    for c in BATCH_CASES:
        N, n_tx, n_rx, M, mode = c[0], c[1], c[2], c[3], c[8]
        add(("heff", heff_variant(N, n_tx, n_rx)[1]), ("batch", c))
        add(("enum", enum_variant(n_tx, M, mode == "hard")), ("batch", c))
        add(("gram", gram_variant(N, n_tx, n_rx)[0]), ("batch", c))
        add(("chol", chol_variant(N, n_tx, n_rx)[1]), ("batch", c))
    for c in PM_CASES:
        add(("pm", pm_variant(c[1], c[8])), ("pm", c))
    for c in DETECTOR_CASES:
        add(("pm", pm_variant(c[1], c[8])), ("detector", c))
    return items


def required_items():
    req = {("heff", b) for b in ("smem", "global", "mma", "rows")}
    req |= {("enum", "k_enum<%d, %d, %d, 4>" % (n, q, h)) for n in range(1, 9) for q in (2, 4, 8) for h in (0, 1)
            if enum_instantiated(n, q)}
    req |= {("gram", "k_gram<%d>" % n) for n in (1, 2, 3)} | {("gram", "k_gram_tma4")}
    req |= {("gram", "k_gram_mma<%d>" % n) for n in range(4, 9)}
    req |= {("chol", "smem"), ("chol", "global")}
    req |= {("pm", pm_variant(n, mode)) for n in (4, 8) for mode in ("pm", "zf")}
    return req


def test_parity_tables_reach_every_kernel_variant():
    """Every kernel instantiation and launch branch of the E-step, Gram and Cholesky is compared with the oracle by
    at least one row of the parity tables (a variant only some other test runs can be wrong unnoticed)."""
    items = covered_items()
    missing = sorted(required_items() - set(items))
    assert not missing, "no parity row reaches %s" % missing
    # both sides of the n_tx = 4 TMA / generic Gram switch are compared at its edge (N = 143 / 144)
    n4 = {c[0]: gram_variant(c[0], 4, c[2])[0] for c in MSTEP_CASES if c[1] == 4}
    assert n4.get(143) == "k_gram_tma4" and n4.get(144) == "k_gram_mma<4>"


def test_workspace_query_admits_exactly_the_launchable_shapes():
    """sbce_workspace_bytes (make_dims) answers SBCE_E_UNSUPPORTED exactly where the Gram launch of the shape
    would not fit in shared memory, near the phase-row limit of every (n_tx, n_rx)."""
    for n_tx in range(1, 9):
        for n_rx in range(1, 9):
            edge = 907 - n_tx * n_tx
            for N in list(range(edge - 40, edge + 3)) + [1, 64, 256]:
                prob = sbce.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=4, T_p=8, T_d=8, itera=1)
                try:
                    ok = sbce.engine.workspace_bytes(prob, 1) > 0
                except sbce.SbceError as e:
                    assert "unsupported" in str(e)
                    ok = False
                assert ok == admitted(N, n_tx, n_rx), (N, n_tx, n_rx, ok)


# ---------------------------------------------------------------------------
# GPU: the mirror against the kernels actually launched
# ---------------------------------------------------------------------------

@pytest.fixture(scope="module")
def S(cuda_device):
    sbce._lib.require_device()
    return sbce


@pytest.fixture(scope="module")
def orc():
    from oracle import em_numpy

    return em_numpy


def _kernel_names(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type.name == "CUDA"]


def _pattern(name):
    # bool template arguments print as 0/1 or false/true depending on the demangler
    p = re.escape(name).replace(r"\ ", " ")
    p = re.sub(r"(?<=, )([01])(?=, 4>)", lambda m: "(?:%s|%s)" % (m.group(1), "true" if m.group(1) == "1" else "false"), p)
    return re.compile(r"(?<![A-Za-z0-9_])" + p)


@pytest.mark.gpu
@pytest.mark.parametrize("case,hard", [((5, 3, 4, 64, 4, 0.2), True), ((256, 4, 4, 4, 6, 0.3), False),
                                       ((16, 4, 4, 4, 130, 0.2), False), ((6, 8, 8, 4, 9, 0.3), True)])
def test_estep_launches_the_mirrored_kernels(S, case, hard):
    import torch

    N, n_tx, n_rx, M, T_d, varn = case
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, 4, T_d, varn, 1, seed=1, legacy=False)
    ses = S.DeviceSession(S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1,
                                    mode="hard" if hard else "soft"), 1)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    ses.estep(t(tb.Yd), t(tb.PsiD), t(tb.h), t(tb.varn))      # first launches (attribute opt-ins) outside the trace
    names = _kernel_names(lambda: ses.estep(t(tb.Yd), t(tb.PsiD), t(tb.h), t(tb.varn)))
    for want in (heff_variant(N, n_tx, n_rx)[0], enum_variant(n_tx, M, hard)):
        assert any(_pattern(want).search(n) for n in names), (want, names)
    assert not any("k_heff" in n and not _pattern(heff_variant(N, n_tx, n_rx)[0]).search(n) for n in names), names


@pytest.mark.gpu
@pytest.mark.parametrize("case", [(20, 2, 3, 4, 16, 17), (143, 4, 2, 4, 64, 40), (144, 4, 2, 4, 64, 40),
                                  (6, 8, 8, 4, 16, 20), (5, 8, 8, 4, 16, 20)])
def test_mstep_launches_the_mirrored_kernels(S, orc, case):
    import torch

    N, n_tx, n_rx, M, T_p, T_d = case
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, T_p, T_d, 0.1, 1, seed=2, legacy=False)
    ses = S.DeviceSession(S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=1), 1)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    sm, sR = tb.Xd.conj(), tb.Xd.conj()[..., :, None] * tb.Xd[..., None, :]
    args = [t(a) for a in (tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, sm, sR)]
    ses.mstep(*args)
    names = _kernel_names(lambda: ses.mstep(*args))
    gram = [n for n in names if "k_gram" in n]
    assert gram and all(_pattern(gram_variant(N, n_tx, n_rx)[0]).search(n) for n in gram), names
    assert any("k_chol_solve" in n for n in names), names


@pytest.mark.gpu
@pytest.mark.parametrize("n_tx,mode", [(3, "pm_beta"), (6, "pm"), (2, "zf"), (6, "mmse")])
def test_pm_estep_launches_the_mirrored_kernel(S, n_tx, mode):
    import torch

    N, n_rx, M, T_d = 6, n_tx, 4, 9
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, 4, T_d, 0.3, 1, seed=3, legacy=False)
    ses = S.DeviceSession(S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=4, T_d=T_d, itera=1, mode=mode,
                                    partition_r=2), 1)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    args = [t(a) for a in (tb.Yd, tb.PsiD, tb.h, tb.varn)]
    ses.estep(*args)
    names = _kernel_names(lambda: ses.estep(*args))
    pm = [n for n in names if "k_pm_stats" in n or "k_det_stats" in n]
    assert pm and all(_pattern(pm_variant(n_tx, mode)).search(n) for n in pm), names


# ---------------------------------------------------------------------------
# mixed batches
# ---------------------------------------------------------------------------
B_MIX = 9
LS, TRUTH_NOISE, HUGE, UNOBSERVED, NAN_YD, AT_TRUTH = 0, 1, 2, 3, 4, 5
BAD = (UNOBSERVED, NAN_YD)
REGULAR = [b for b in range(B_MIX) if b not in BAD]

MIX_CASES = [
    # mode, N, n_tx, n_rx, M, T_p, T_d, itera, partition_r
    ("soft", 8, 2, 2, 4, 24, 40, 4, 0),      # scalar Gram, effective channel in shared memory
    ("hard", 16, 4, 4, 4, 80, 48, 3, 0),     # tensor-path effective channel, TMA Gram
    ("soft", 5, 6, 6, 4, 40, 30, 3, 0),      # row-per-lane QR, generic Gram
    ("pm_beta", 8, 3, 3, 16, 40, 40, 3, 4),
    ("zf", 8, 2, 2, 4, 24, 40, 3, 0),
    ("mmse", 8, 3, 3, 4, 30, 40, 3, 0),
    ("superimposed", 8, 2, 2, 4, 0, 48, 3, 0),
]


def _mixed_problem(case):
    mode, N, n_tx, n_rx, M, T_p, T_d, itera, pr = case
    sup = mode == "superimposed"
    return sbce.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, mode="soft" if sup else mode,
                        partition_r=pr, genie_stop=not sup, zero_start=sup, superimposed=sup)


def _mixed_inputs(prob, seed=3):
    """Nine trials of one shape: varn log-spaced over 0.01..10, LS / truth + noise / 1e6-scaled / at-truth starts,
    one trial with an unobserved RIS element and one with a NaN in its data."""
    B, N, n_tx, n_rx, M = B_MIX, prob.N, prob.n_tx, prob.n_rx, prob.M
    varn = np.logspace(-2, 1, B)
    rng = np.random.default_rng(seed)
    if prob.superimposed:
        T = prob.T_d
        tb = sbce.signal_model.generate_batch(N, n_tx, n_rx, M, 2, T, varn, B, seed=seed, legacy=False,
                                              variant="top_td")
        tb.PsiD[:, :, 1:] = np.exp(1j * rng.uniform(0, 2 * np.pi, (B, T, N)))
        from oracle import em_numpy as orc

        cons = orc.qam_constellation(M)
        Xoff = np.zeros((B, T, n_tx), np.complex128)
        Xoff[:, :T // 3] = cons[rng.integers(0, M, (B, T // 3, n_tx))]
        Xd = cons[rng.integers(0, M, (B, T, n_tx))]
        W = (tb.PsiD[:, :, :, None] * (Xd + Xoff)[:, :, None, :]).reshape(B, T, -1)
        Y = W @ tb.h + np.sqrt(varn / 2)[:, None, None] * (rng.standard_normal((B, T, n_rx)) +
                                                            1j * rng.standard_normal((B, T, n_rx)))
        inp = dict(Yd=Y, Yp=np.zeros((B, 0, n_rx), np.complex128), PsiD=tb.PsiD.copy(),
                   PsiP=np.zeros((B, 0, N + 1), np.complex128), Xp=Xoff, varn=varn, theta0=None, h_true=tb.h,
                   Xd_true=None)
    else:
        tb = sbce.signal_model.generate_batch(N, n_tx, n_rx, M, prob.T_p, prob.T_d, varn, B, seed=seed,
                                              legacy=False, variant="top_tp")
        # random pilot phases (T_p >= L): the pilot block alone determines the channel, so every start, however
        # poor its first decisions, leaves a positive definite normal matrix (the deterministic pilot designs
        # leave one RIS element to the data)
        tb.PsiP[:, :, 1:] = np.exp(1j * rng.uniform(0, 2 * np.pi, (B, prob.T_p, N)))
        Wp = (tb.PsiP[:, :, :, None] * tb.Xp[:, :, None, :]).reshape(B, prob.T_p, -1)
        tb.Yp = Wp @ tb.h + np.sqrt(varn / 2)[:, None, None] * (rng.standard_normal(tb.Yp.shape) +
                                                                 1j * rng.standard_normal(tb.Yp.shape))
        WpH = Wp.conj().transpose(0, 2, 1)
        theta0 = np.linalg.solve(WpH @ Wp, WpH @ tb.Yp)
        theta0[TRUTH_NOISE] = tb.h[TRUTH_NOISE] + 0.1 * (rng.standard_normal(tb.h.shape[1:]) +
                                                         1j * rng.standard_normal(tb.h.shape[1:]))
        theta0[HUGE] *= 1e6
        theta0[AT_TRUTH] = tb.h[AT_TRUTH]
        inp = dict(Yd=tb.Yd.copy(), Yp=tb.Yp, PsiD=tb.PsiD.copy(), PsiP=tb.PsiP.copy(), Xp=tb.Xp, varn=varn,
                   theta0=theta0, h_true=tb.h, Xd_true=tb.Xd)
        inp["PsiP"][UNOBSERVED, :, N // 2] = 0.0
    inp["PsiD"][UNOBSERVED, :, N // 2] = 0.0      # RIS element never illuminated: singular normal matrix
    inp["Yd"][NAN_YD, prob.T_d // 2, 0] = np.nan
    return inp


def _take(inp, idx):
    return {k: (None if v is None else np.ascontiguousarray(v[idx])) for k, v in inp.items()}


OUT_KEYS = ("theta", "kstar", "llf", "lse", "nmse", "iters", "status")


def _run_device(ses, inp, out=None):
    import torch

    t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    res = ses.run(*(t(inp[k]) for k in ("Yd", "Yp", "PsiD", "PsiP", "Xp", "varn")), theta0=t(inp["theta0"]),
                  h_true=t(inp["h_true"]), Xd_true=t(inp["Xd_true"]), out=out)
    torch.cuda.synchronize()
    return {k: getattr(res, k).cpu().numpy() for k in OUT_KEYS if getattr(res, k) is not None}


def _run_host(prob, inp):
    res = sbce.run_host(prob, inp["Yd"], inp["Yp"], inp["PsiD"], inp["PsiP"], inp["Xp"], inp["varn"],
                        theta0=inp["theta0"], h_true=inp["h_true"], Xd_true=inp["Xd_true"])
    return {k: getattr(res, k) for k in OUT_KEYS if getattr(res, k) is not None}


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _assert_same(r1, r2, idx=slice(None), what=""):
    assert set(r1) == set(r2)
    for k in r1:
        assert _same_bits(r1[k][idx], r2[k]), (what, k)


def _oracle(orc, prob, inp, b, pr):
    g = lambda k: inp[k][b]
    vb = float(inp["varn"][b])
    mode = prob.mode
    if prob.superimposed:
        th, tr = orc.em_superimposed(g("Yd"), g("PsiD"), g("Xp"), prob.M, vb, prob.itera, return_trace=True)
        tr["iters"] = prob.itera
        return th, tr
    args = (g("Yd"), g("Yp"), g("PsiD"), g("PsiP"), g("Xp"), prob.M, vb, prob.itera)
    if mode in ("soft", "hard"):
        return orc.em(*args, theta0=g("theta0"), hard=mode == "hard", h_true=g("h_true"), genie_stop=True,
                      Xd_true=g("Xd_true"), return_trace=True)
    if mode in ("zf", "mmse"):
        return orc.em_detector(*args, g("theta0"), kind=mode, h_true=g("h_true"), genie_stop=True, quirks=True,
                               return_trace=True)
    return orc.em_pm(*args, g("theta0"), h_true=g("h_true"), partition_r=pr, weighted=True, genie_stop=True,
                     quirks=True, how="solve", return_trace=True)


@pytest.mark.gpu
@pytest.mark.parametrize("case", MIX_CASES, ids=[c[0] + "-%dx%d" % (c[2], c[3]) for c in MIX_CASES])
def test_mixed_batch_trials_are_independent(S, orc, case):
    import torch

    prob = _mixed_problem(case)
    pr = case[8]
    inp = _mixed_inputs(prob)
    ses = S.DeviceSession(prob, 2)                       # the batch runs in chunks of two trials
    full = _run_device(ses, inp)
    # the same batch reversed, through the host route (one chunk, pipelined copies) and trial by trial
    rev = _run_device(ses, _take(inp, slice(None, None, -1)))
    _assert_same(full, rev, slice(None, None, -1), "reversed")
    _assert_same(full, _run_host(prob, inp), what="host route")
    for b in REGULAR:
        _assert_same(full, _run_device(ses, _take(inp, slice(b, b + 1))), slice(b, b + 1), "trial %d alone" % b)
    # bad trials are flagged, regular ones are not
    st = full["status"]
    assert st[UNOBSERVED] & 1, st
    assert st[NAN_YD] != 0, st
    assert (st[REGULAR] == 0).all(), st
    # regular trials against the oracle at their own noise variance
    bar = 1e-8 if prob.mode == "pm_beta" else 1e-9
    for b in REGULAR:
        ref, tr = _oracle(orc, prob, inp, b, pr)
        assert relerr(full["theta"][b], ref) < bar, (b, relerr(full["theta"][b], ref))
        assert int(full["iters"][b]) == tr["iters"], b
        if prob.mode in ("soft", "hard"):
            assert np.array_equal(full["kstar"][b], tr["kstar"]), b
            it = tr["iters"]
            if "llf" in full and tr["llf"]:
                np.testing.assert_allclose(full["llf"][b][:it], tr["llf"], rtol=1e-8)
            if prob.mode == "soft":
                np.testing.assert_allclose(full["lse"][b][:it], tr["lse"], rtol=1e-9)
    if not prob.superimposed:
        assert (full["iters"][REGULAR] < prob.itera).any()    # the genie stop ended some trials early
    # the sweep accumulator drops exactly the flagged trials
    acc = torch.zeros(3, dtype=torch.float64, device=ses.device)
    res = sbce.Result(theta=torch.from_numpy(full["theta"]).to(ses.device), nmse=torch.from_numpy(full["nmse"]).to(ses.device),
                      status=torch.from_numpy(full["status"]).to(ses.device))
    ses.accumulate(res, None, acc)
    a = acc.cpu().numpy()
    ok = full["status"] == 0
    np.testing.assert_allclose(a[0], full["nmse"][ok].sum(), rtol=1e-13)
    assert a[1] == ok.sum() and a[2] == (~ok).sum()


# ---------------------------------------------------------------------------
# dirty workspaces and output buffers
# ---------------------------------------------------------------------------
DIRTY_CASES = [("soft", 8, 2, 2, 4, 24, 40, 3, 0), ("hard", 10, 3, 3, 4, 40, 40, 3, 0),
               ("soft", 5, 6, 6, 4, 40, 30, 3, 0), ("pm_beta", 8, 3, 3, 16, 40, 40, 3, 4)]


def _fill(t, how, seed=0):
    import torch

    v = t.view(torch.uint8) if t.dtype != torch.uint8 else t
    if how == "zeros":
        v.zero_()
    elif how == "ones":
        v.fill_(0xFF)                                    # NaN doubles, -1 int32
    else:
        g = torch.Generator(device=t.device).manual_seed(seed)
        v.copy_(torch.randint(0, 256, v.shape, dtype=torch.uint8, device=t.device, generator=g))


@pytest.mark.gpu
@pytest.mark.parametrize("case", DIRTY_CASES, ids=[c[0] + "-%dx%d" % (c[2], c[3]) for c in DIRTY_CASES])
def test_results_do_not_depend_on_workspace_or_output_contents(S, orc, case):
    """L and n_rx are not multiples of the padding (Lp - L and RP - n_rx padding rows), so every padding row and
    column of G / G_p and every per-trial flag must be rewritten by the call."""
    import torch

    prob = _mixed_problem(case)
    inp = _mixed_inputs(prob)
    B = B_MIX
    ses = S.DeviceSession(prob, B)
    dev = ses.device
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    sm, sR = inp["Xd_true"].conj(), inp["Xd_true"].conj()[..., :, None] * inp["Xd_true"][..., None, :]

    def calls():
        out = {}
        out["run"] = _run_device(ses, inp)
        m, R, ks, ls = ses.estep(t(inp["Yd"]), t(inp["PsiD"]), t(inp["theta0"]), t(inp["varn"]))
        out["estep"] = [x.cpu().numpy() for x in (m, R, ks, ls)]
        out["mstep"] = [x.cpu().numpy() for x in ses.mstep(t(inp["Yd"]), t(inp["Yp"]), t(inp["PsiD"]),
                                                            t(inp["PsiP"]), t(inp["Xp"]), t(sm), t(sR))]
        out["ls"] = [x.cpu().numpy() for x in ses.ls_start(t(inp["Yp"]), t(inp["PsiP"]), t(inp["Xp"]))]
        return out

    results = {}
    for how in ("zeros", "ones", "random"):
        _fill(ses.ws, how, seed=len(results))
        results[how] = calls()
    ref = results["zeros"]
    for how in ("ones", "random"):
        for k in ref:
            if k == "run":
                _assert_same(ref[k], results[how][k], what=how)
            else:
                for i, (a, b) in enumerate(zip(ref[k], results[how][k])):
                    assert _same_bits(a, b), (how, k, i)
    # garbage in the caller's output buffers: skipped iterations read NaN, the PM modes write kstar = -1
    out = ses.alloc_outputs(B, llf=True)
    for k in OUT_KEYS:
        _fill(getattr(out, k), "random", seed=7)
    dirty = _run_device(ses, inp, out=out)
    _assert_same(ref["run"], dirty, what="dirty outputs")
    it = dirty["iters"]
    assert (it[REGULAR] >= 1).all() and (it[REGULAR] < prob.itera).any()
    for b in range(B):
        assert np.isnan(dirty["llf"][b, it[b]:]).all() and np.isnan(dirty["lse"][b, it[b]:]).all(), b
    if prob.mode == "pm_beta":
        assert (dirty["kstar"] == -1).all() and np.isnan(dirty["lse"]).all()
    # the same for the stand-alone E-step: kstar = -1 and lse = NaN where the mode produces neither
    eout = [torch.empty_like(torch.from_numpy(a)).to(dev) for a in ref["estep"]]
    for o in eout:
        _fill(o, "random", seed=8)
    got = [x.cpu().numpy() for x in ses.estep(t(inp["Yd"]), t(inp["PsiD"]), t(inp["theta0"]), t(inp["varn"]),
                                              out=eout)]
    for i, (a, b) in enumerate(zip(ref["estep"], got)):
        assert _same_bits(a, b), ("dirty estep outputs", i)
    if prob.mode == "pm_beta":
        assert (got[2] == -1).all() and np.isnan(got[3]).all()


@pytest.mark.gpu
def test_host_route_large_small_large_equals_device_route(S):
    """The host route keeps one scratch pool and up to four cached graphs per device: a small configuration between
    two large ones (pool kept, graphs recaptured and replayed) must not change any result."""
    big, small = DIRTY_CASES[2], DIRTY_CASES[0]
    fresh = {}
    for c in (big, small):
        prob = _mixed_problem(c)
        fresh[c] = _run_device(S.DeviceSession(prob, B_MIX), _mixed_inputs(prob))
    for c in (big, small, big, big, small):
        prob = _mixed_problem(c)
        _assert_same(fresh[c], _run_host(prob, _mixed_inputs(prob)), what=c[0])


# ---------------------------------------------------------------------------
# the phase-row limit
# ---------------------------------------------------------------------------

def _limit_shape(n_tx):
    n_rx = 8
    N = max(N for N in range(900 - n_tx * n_tx, 910) if admitted(N, n_tx, n_rx))
    return N, n_rx


@pytest.mark.gpu
@pytest.mark.parametrize("n_tx", range(1, 9))
def test_largest_admitted_phase_rows_launch(S, n_tx):
    """The largest N the C ABI admits for each n_tx (n_rx = 8) runs: the stand-alone M-step on a noiseless,
    consistent system (rank-one statistics of the true symbols; the least-squares solution on
    W = [psi_t (x) x_t] is then the channel itself) and one hard-decision EM iteration on the host route."""
    import torch

    N, n_rx = _limit_shape(n_tx)
    N1, L = N + 1, (N + 1) * n_tx
    T_p = T_d = (6 * L + 9) // 10
    rng = np.random.default_rng(n_tx)
    from oracle import em_numpy as orc

    cons = orc.qam_constellation(4)
    Psi = lambda T: np.exp(1j * rng.uniform(0, 2 * np.pi, (1, T, N1)))
    PsiP, PsiD = Psi(T_p), Psi(T_d)
    Xp, Xd = cons[rng.integers(0, 4, (1, T_p, n_tx))], cons[rng.integers(0, 4, (1, T_d, n_tx))]
    h = (rng.standard_normal((1, L, n_rx)) + 1j * rng.standard_normal((1, L, n_rx))) / np.sqrt(2)
    H = h.reshape(N1, n_tx * n_rx)
    Y = lambda P, X: np.einsum("tjr,tj->tr", (P[0] @ H).reshape(-1, n_tx, n_rx), X[0])[None]
    Yp, Yd = Y(PsiP, Xp), Y(PsiD, Xd)
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=4, T_p=T_p, T_d=T_d, itera=1, mode="hard")
    assert S.engine.workspace_bytes(prob, 1) > 0
    ses = S.DeviceSession(prob, 1)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    sm = Xd.conj()
    sR = Xd.conj()[:, :, :, None] * Xd[:, :, None, :]
    theta, status = ses.mstep(t(Yd), t(Yp), t(PsiD), t(PsiP), t(Xp), t(sm), t(sR))
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    assert relerr(theta.cpu().numpy(), h) < 1e-8
    del ses, theta
    vn = 0.01
    noise = lambda Z: np.sqrt(vn / 2) * (rng.standard_normal(Z.shape) + 1j * rng.standard_normal(Z.shape))
    res = S.run_host(prob, Yd + noise(Yd), Yp + noise(Yp), PsiD, PsiP, Xp, np.array([vn]), theta0=h + 0.01 * h,
                     h_true=h)
    assert int(res.status[0]) == 0 and np.isfinite(res.theta).all()
    assert res.nmse[0] < 1e-3
