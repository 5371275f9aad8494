"""Estimator entry points with the reference's names, positional argument order
and return shapes; each call is a batch of one through the C ABI
(sbce_em_batch_host).  The reference's implicit module globals (N, n_tx, h, Z_d)
became keyword arguments or are inferred from the arrays.

  em        /root/reference/Proposed_method_NMSEvsTp.py:43 (theta0 = 0)
            /root/reference/Proposed method/Proposed_method_NMSEvsTp.py:50 (theta0 = h_initial)
            /root/reference/Proposed method/IRS_elements.py:268 (+N)
  em_ml     /root/reference/Proposed method/PMvsMLvsZFvsMMSE.py:135 (hard decisions, genie stop)
  em_llf    /root/reference/Proposed method/ML_detecctor.py:51 (hard decisions, returns LLF per iteration)
  em_ser    /root/reference/Proposed method/SER/log_max_SER.py:51 (hard decisions, returns X_dest)
  em_pm     /root/reference/Proposed method/PM.py:47 (partitioned, weight 1, lstsq)
  em_pm_beta /root/reference/Proposed method/PM_beta.py:42 (partitioned, posterior weights)
  em_zf, em_mmse /root/reference/Proposed method/PMvsMLvsZFvsMMSE.py:95,54 (detector-driven EM)
"""
from __future__ import annotations

import numpy as np

from . import engine
from .qam import SUPPORTED_M, constellation, constellation_from_table, symbols_of


def _stack_cols(lst):
    """list of (n,1) arrays -> (T, n)."""
    return np.hstack([np.asarray(a).reshape(-1, 1) for a in lst]).T.astype(np.complex128)


def _pilot_factors(Z_p, n_rx, n_tx, N1, PsiTilde_tp=None, X_p=None):
    """PsiP (T_p,N+1), Xp (T_p,n_tx).  Exact when the caller passes the phase matrix
    and pilot symbols; otherwise the rank-one design row w_t = psi~_t (x) x_t is read
    from row 0 of the reference's dense Z_p[t] (entries 0::n_rx) and split as
    psi' = W[:, j0] / W[n0, j0], x' = W[n0, :] around its largest entry, which
    reproduces w_t to rounding."""
    if PsiTilde_tp is not None and X_p is not None:
        return np.asarray(PsiTilde_tp, dtype=np.complex128).T.copy(), _stack_cols(X_p)
    T_p = len(Z_p)
    PsiP = np.empty((T_p, N1), dtype=np.complex128)
    Xp = np.empty((T_p, n_tx), dtype=np.complex128)
    for t in range(T_p):
        w = np.asarray(Z_p[t][0, 0::n_rx]).reshape(N1, n_tx)
        n0, j0 = np.unravel_index(int(np.argmax(np.abs(w))), w.shape)
        piv = w[n0, j0]
        if piv == 0:
            PsiP[t], Xp[t] = 0, 0
        else:
            PsiP[t] = w[:, j0] / piv
            Xp[t] = w[n0, :]
    return PsiP, Xp


def _common(Y_d, Y_p, Z_p, PsiTilde_td, M, n_tx, PsiTilde_tp, X_p, cons=None):
    if M not in SUPPORTED_M:
        raise ValueError("M must be one of %s" % (SUPPORTED_M,))
    if cons is not None and not np.array_equal(np.asarray(cons, dtype=np.complex128), constellation(M)):
        raise ValueError("only the reference's un-normalised square QAM constellation is supported")
    Yd = _stack_cols(Y_d)
    Yp = _stack_cols(Y_p)
    n_rx = Yd.shape[1]
    PsiD = np.asarray(PsiTilde_td, dtype=np.complex128).T.copy()
    N1 = PsiD.shape[1]
    PsiP, Xp = _pilot_factors(Z_p, n_rx, n_tx, N1, PsiTilde_tp, X_p)
    return Yd, Yp, PsiD, PsiP, Xp, n_rx, N1


def _theta_arg(h_initial, L, n_rx):
    return None if h_initial is None else np.asarray(h_initial, dtype=np.complex128).reshape(1, L, n_rx)


def _run(mode, Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h_initial, n_tx, *, cons=None, h=None,
         genie_stop=False, Xd_true=None, partition_r=0.0, quirks=True, PsiTilde_tp=None, X_p=None, device=0,
         zf_stop_guard=False):
    Yd, Yp, PsiD, PsiP, Xp, n_rx, N1 = _common(Y_d, Y_p, Z_p, PsiTilde_td, M, n_tx, PsiTilde_tp, X_p, cons)
    if Yd.shape[0] != T_d or Yp.shape[0] != T_p:
        raise ValueError("T_d / T_p do not match the lengths of Y_d / Y_p")
    L = N1 * n_tx
    prob = engine.Problem(N=N1 - 1, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=int(itera), mode=mode,
                          genie_stop=bool(genie_stop and h is not None), quirks=quirks,
                          zero_start=h_initial is None, partition_r=partition_r, zf_stop_guard=zf_stop_guard)
    h_true = None if h is None else np.asarray(h, dtype=np.complex128).reshape(1, L, n_rx)
    xd = None if Xd_true is None else np.asarray(Xd_true, dtype=np.complex128).reshape(1, T_d, n_tx)
    res = engine.run_host(prob, Yd[None], Yp[None], PsiD[None], PsiP[None], Xp[None], float(varn),
                          theta0=_theta_arg(h_initial, L, n_rx), h_true=h_true, Xd_true=xd, device=device)
    return res, prob


def _ntx_from_table(all_possibleSymbols):
    return int(np.asarray(all_possibleSymbols).shape[1])


def em(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial=None, N=None, *,
       h=None, genie_stop=False, **kw):
    """Soft-decision EM, full enumeration.  Returns theta (D,1) complex128."""
    n_tx = _ntx_from_table(all_possibleSymbols)
    cons = constellation_from_table(all_possibleSymbols, M)
    res, prob = _run("soft", Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h_initial, n_tx, cons=cons, h=h,
                     genie_stop=genie_stop, **kw)
    return res.theta.reshape(-1, 1)


def em_ml(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial, *, h=None,
          genie_stop=True, **kw):
    """Hard-decision ("log-max") EM; the genie stop is active when the true h is given
    (the reference reads it from a module global)."""
    n_tx = _ntx_from_table(all_possibleSymbols)
    cons = constellation_from_table(all_possibleSymbols, M)
    res, _ = _run("hard", Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h_initial, n_tx, cons=cons, h=h,
                  genie_stop=genie_stop, **kw)
    return res.theta.reshape(-1, 1)


def em_parallel(Y, T, Z, X_d, X_p, T_p, T_d, n_tx, PsiTilde_t, all_possibleSymbols, M, varn, itera, N, *, hard=False,
                device=0):
    """Parallel protocol with superimposed pilots: the reference's `em` of Parallel/ParallelProtocol_Tp.py:64
    (same positional signature).  Hypotheses of symbol t are x_k + x_p[t] (zero beyond T_p), no separate pilot
    term, zero start.  Z and X_d are accepted for signature compatibility and not used (as in the reference)."""
    cons = constellation_from_table(all_possibleSymbols, M)
    if M not in SUPPORTED_M or not np.array_equal(np.asarray(cons, dtype=np.complex128), constellation(M)):
        raise ValueError("only the reference's un-normalised square QAM constellation is supported")
    Yd = _stack_cols(Y)
    n_rx = Yd.shape[1]
    Psi = np.asarray(PsiTilde_t, dtype=np.complex128).T.copy()
    if Yd.shape[0] != T or Psi.shape != (T, N + 1):
        raise ValueError("T does not match Y / PsiTilde_t")
    Xoff = np.zeros((T, n_tx), dtype=np.complex128)
    if T_p:
        Xoff[:T_p] = _stack_cols(X_p)
    prob = engine.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=0, T_d=T, itera=int(itera), mode="hard" if hard else "soft",
                          zero_start=True, superimposed=True)
    empty = np.zeros((1, 0, n_rx), np.complex128)
    res = engine.run_host(prob, Yd[None], empty, Psi[None], np.zeros((1, 0, N + 1), np.complex128), Xoff[None],
                          float(varn), device=device)
    return res.theta.reshape(-1, 1)


def _true_data_from_Zd(Z_d, PsiTilde_td, n_rx, n_tx):
    Psi = np.asarray(PsiTilde_td)
    T_d = len(Z_d)
    Xd = np.empty((T_d, n_tx), dtype=np.complex128)
    for t in range(T_d):
        w = np.asarray(Z_d[t][0, 0::n_rx]).reshape(-1, n_tx)
        n0 = int(np.argmax(np.abs(Psi[:, t])))
        Xd[t] = w[n0] / Psi[n0, t]
    return Xd


def em_llf(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial, *, Z_d=None,
           X_d=None, soft=False, **kw):
    """Hard-decision (soft=True: soft-decision) EM returning (theta, logLikelihood (itera,1)) -- the LLF exactly as
    coded in ML_detecctor.py:84 (needs the TRUE data: Z_d list or X_d list)."""
    n_tx = _ntx_from_table(all_possibleSymbols)
    cons = constellation_from_table(all_possibleSymbols, M)
    n_rx = np.asarray(Y_d[0]).shape[0]
    if X_d is not None:
        xd = _stack_cols(X_d)
    elif Z_d is not None:
        xd = _true_data_from_Zd(Z_d, PsiTilde_td, n_rx, n_tx)
    else:
        raise ValueError("em_llf needs Z_d or X_d (the reference reads Z_d from a module global)")
    res, _ = _run("soft" if soft else "hard", Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h_initial, n_tx,
                  cons=cons, Xd_true=xd, **kw)
    return res.theta.reshape(-1, 1), res.llf.reshape(int(itera), 1)


def em_loglik(Y_d, Y_p, T_d, T_p, Z_p, Z_d, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial, n_tx=None, **kw):
    """`Proposed method/Log_likelihood.py:45` -- the same estimator as em_llf with the positional signature of that
    script (Z_d and n_tx are arguments there instead of module globals).  Returns (theta, logLikelihood (itera,1))."""
    return em_llf(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial, Z_d=Z_d, **kw)


def em_iterations_llf(Y_d, Y_p, T_d, T_p, Z_p, Z_d, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial, n_tx=None,
                      **kw):
    """`Proposed method/IterationsvsLLF.py:44` -- SOFT-decision EM with the as-coded LLF per iteration, positional
    signature of that script.  Returns (theta, logLikelihood (itera,1))."""
    return em_llf(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial, Z_d=Z_d, soft=True,
                  **kw)


def em_ser(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial, **kw):
    """Hard-decision EM returning (theta, X_dest): X_dest is the list of (1,n_tx) decisions
    of the last iteration, made before its M-step (SER/log_max_SER.py:77-78,89)."""
    n_tx = _ntx_from_table(all_possibleSymbols)
    cons = constellation_from_table(all_possibleSymbols, M)
    res, _ = _run("hard", Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h_initial, n_tx, cons=cons, **kw)
    xs = symbols_of(res.kstar[0], M, n_tx)
    return res.theta.reshape(-1, 1), [xs[t][None, :] for t in range(T_d)]


def em_pm(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial, h, n_tx,
          partition_r, X_d=None, qamCons=None, *, genie_stop=True, quirks=True, **kw):
    """Partitioned EM with un-weighted candidates (PM.py:47-116)."""
    res, _ = _run("pm", Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h_initial, n_tx, cons=qamCons, h=h,
                  genie_stop=genie_stop, partition_r=partition_r, quirks=quirks, **kw)
    return res.theta.reshape(-1, 1)


def em_pm_beta(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h_initial, h, n_tx, partition_r, X_d=None,
               qamCons=None, *, genie_stop=True, quirks=True, **kw):
    """Partitioned EM with posterior-weighted candidates (PM_beta.py:42-112)."""
    res, _ = _run("pm_beta", Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h_initial, n_tx, cons=qamCons,
                  h=h, genie_stop=genie_stop, partition_r=partition_r, quirks=quirks, **kw)
    return res.theta.reshape(-1, 1)


def em_zf(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial, h, *,
          genie_stop=True, quirks=True, **kw):
    """Zero-forcing detector EM (PMvsMLvsZFvsMMSE.py:95-133).  quirks=True reproduces the off-by-one psi slice and
    the table-indexing slicer.  The three scripts that ship this function differ only in the genie stop:
    PMvsMLvsZFvsMMSE.py:128 stops without the `l != 0` guard (default here), all_detectorsvsTd.py:127 has the
    guard (`zf_stop_guard=True`), SNR/all_Detectors.py has no stop at all (`genie_stop=False`)."""
    n_tx = _ntx_from_table(all_possibleSymbols)
    cons = constellation_from_table(all_possibleSymbols, M)
    res, _ = _run("zf", Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h_initial, n_tx, cons=cons, h=h,
                  genie_stop=genie_stop, quirks=quirks, **kw)
    return res.theta.reshape(-1, 1)


def em_mmse(Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, all_possibleSymbols, M, varn, itera, h_initial, h, *,
            genie_stop=True, quirks=True, **kw):
    """MMSE detector EM (PMvsMLvsZFvsMMSE.py:54-93)."""
    n_tx = _ntx_from_table(all_possibleSymbols)
    cons = constellation_from_table(all_possibleSymbols, M)
    res, _ = _run("mmse", Y_d, Y_p, T_d, T_p, Z_p, PsiTilde_td, M, varn, itera, h_initial, n_tx, cons=cons, h=h,
                  genie_stop=genie_stop, quirks=quirks, **kw)
    return res.theta.reshape(-1, 1)


def bit_llr(Y_d, PsiTilde_td, theta, M, varn, n_tx, *, X_p=None, llr_a=None, device=0):
    """Exact Gray-labelled bit LLRs of the data symbols at the estimate `theta` (the (D,1) vector em() returns),
    in the reference's data conventions: Y_d the list of (n_rx,1) observations, PsiTilde_td the (N+1, T_d) phases
    with the direct-link ones row.  X_p (list of (n_tx,1) pilot symbols): the parallel protocol's superimposed
    pilots, added to the data of the first len(X_p) symbols (em_parallel).  Returns (T_d, n_tx * log2 M)
    float64: ln P(bit = 0) - ln P(bit = 1) under the E-step's posterior (exponent d2/varn^2, uniform prior),
    clamped to [-32, 32], bits in the order of qam.bit_labels per stream, stream 0 first.  llr_a: a-priori LLRs
    from a channel decoder in the same (T_d, n_tx * log2 M) layout; then the result is the extrinsic LLR (the
    posterior under that prior minus llr_a, include/sbce.h: sbce_bit_llr_apriori), which equals the a-posteriori
    LLR when there is no prior (llr_a = 0)."""
    import torch

    if M not in SUPPORTED_M:
        raise ValueError("M must be one of %s" % (SUPPORTED_M,))
    Yd = _stack_cols(Y_d)
    T_d, n_rx = Yd.shape
    PsiD = np.asarray(PsiTilde_td, dtype=np.complex128).T.copy()
    if PsiD.shape[0] != T_d:
        raise ValueError("PsiTilde_td has %d columns, Y_d %d symbols" % (PsiD.shape[0], T_d))
    N1 = PsiD.shape[1]
    L = N1 * n_tx
    th = np.asarray(theta, dtype=np.complex128).reshape(1, L, n_rx)
    Xoff = None
    if X_p is not None:
        Xoff = np.zeros((1, T_d, n_tx), dtype=np.complex128)
        if len(X_p):
            Xoff[0, :len(X_p)] = _stack_cols(X_p)
    prob = engine.Problem(N=N1 - 1, n_tx=n_tx, n_rx=n_rx, M=M, T_p=0, T_d=T_d, itera=1,
                          superimposed=Xoff is not None)
    dev = torch.device("cuda", device)
    ses = engine.DeviceSession(prob, 1, device=dev)
    t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    La = None
    if llr_a is not None:
        La = np.asarray(llr_a, dtype=np.float64)
        nb = n_tx * int(np.log2(M))
        if La.shape != (T_d, nb):
            raise ValueError("llr_a has shape %s, expected (%d, %d)" % (La.shape, T_d, nb))
        La = La.reshape(1, T_d, n_tx, -1)
    out = ses.bit_llr(t(Yd[None]), t(PsiD[None]), t(th), torch.full((1,), float(varn), dtype=torch.float64, device=dev),
                      Xp=t(Xoff), llr_a=t(La))
    return out.cpu().numpy().reshape(T_d, -1)


def nmse(theta_hat, h):
    """Proposed_method_NMSEvsTp.py:138."""
    a = np.asarray(theta_hat).reshape(-1)
    b = np.asarray(h).reshape(-1)
    d = a - b
    return float(np.vdot(d, d).real / np.vdot(b, b).real)


def ser_as_coded(X_d, X_dest):
    """SER/log_max_SER.py:162 including its (T_d,n_tx,1)-(T_d,1,n_tx) broadcast."""
    T_d = len(X_d)
    n_tx = np.asarray(X_d[0]).size
    return float(np.count_nonzero(np.array(X_d) - np.array(X_dest)) / (T_d * n_tx))


def ser_true(X_d, X_dest):
    a = np.array([np.asarray(x).reshape(-1) for x in X_d])
    b = np.array([np.asarray(x).reshape(-1) for x in X_dest])
    return float(np.count_nonzero(a - b) / a.size)
