"""TEST INFRASTRUCTURE ONLY -- numpy complex128 restatement of the reference's
semi-blind EM channel-estimation hot path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
reference legs may import this module; the product (the package next to this
directory) never does and fails loudly when its CUDA library is missing.

Parity status: the reference ships NO tests, golden vectors or fixtures
("parity unpinned" by the reference's own tests, SURVEY.md section 8c).  This
restatement is therefore pinned against the reference ITSELF: the literal
reference functions are executed in the build container through
oracle/ref_harness.py on seeded inputs, their inputs/outputs are committed
under tests/golden/ (generator: oracle/make_golden.py) and
tests/test_oracle_golden.py asserts this file reproduces them.

All file:line citations are relative to /root/reference.

Layout used everywhere in this repository (one trial):
    L      = (N+1)*n_tx                      unknowns per receive antenna
    Theta  (L, n_rx)   Theta[n'*n_tx+j, r] = h[(n'*n_tx+j)*n_rx+r]     (PM.py:15)
    PsiD   (T_d, N+1)  row t = psi~_t (ones at n'=0: direct link, PM.py:179)
    PsiP   (T_p, N+1)
    Xp     (T_p, n_tx) pilot symbols,   Xd (T_d, n_tx) true data symbols
    Yp     (T_p, n_rx),                 Yd (T_d, n_rx)
    y_t[r] = sum_{n',j} psi~[t,n'] x_t[j] Theta[n'*n_tx+j, r] + noise   (PM.py:138-146:
             Z_t = psi~_t^T (x) x_t^T (x) I_nrx is never materialised here)
"""
from __future__ import annotations

import itertools
import math

import numpy as np

# --------------------------------------------------------------------------
# constellation and hypothesis order
# --------------------------------------------------------------------------

def qam_constellation(M: int) -> np.ndarray:
    """Un-normalised square QAM grid, in-phase index fastest.
    Follows `Proposed method/QAM.py:310-322` (orders=int, base_amplitude 1,
    phase_offset 0): c[iQ*sqrtM + iI] = (2 iI - sqrtM + 1) + 1j (2 iQ - sqrtM + 1)."""
    s = int(round(math.sqrt(M)))
    if s * s != M or (s & (s - 1)) != 0:
        raise ValueError("M must be a square power of two")
    axis = np.arange(-s + 1, s, 2, dtype=np.float64)
    return (axis[None, :] + 1j * axis[:, None]).reshape(-1).astype(np.complex128)


def hypothesis_table(cons: np.ndarray, n_tx: int) -> np.ndarray:
    """(K, n_tx) table in itertools.product order, stream 0 most significant
    (`Proposed method/PM.py:25-31`): k = sum_j idx_j * M**(n_tx-1-j)."""
    return np.asarray(list(itertools.product(*([cons] * n_tx))), dtype=np.complex128).reshape(-1, n_tx)


def hypothesis_digits(k: np.ndarray, M: int, n_tx: int) -> np.ndarray:
    """Base-M digits of hypothesis indices, shape (..., n_tx), stream 0 first."""
    k = np.asarray(k)
    out = np.empty(k.shape + (n_tx,), dtype=np.int64)
    for j in range(n_tx - 1, -1, -1):
        out[..., j] = k % M
        k = k // M
    return out


# --------------------------------------------------------------------------
# signal model (input generation) -- reference RNG call order, SURVEY App. C
# --------------------------------------------------------------------------

def channel_vector(n_tx, n_rx, N, varh=1.0, rs=np.random, flatten="F"):
    """`Proposed method/PM.py:11-17`.  Returns Theta_true (L, n_rx).
    h = [vec_F(H_BU); vec_F(khatri_rao(H_BS^T, H_SU))]; entry for (n+1, j, r)
    is H_BS[n, j] * H_SU[r, n].
    flatten="C" restates the two top-level scripts, which use C-order
    `.flatten()` (`Proposed_method_NMSEvsTp.py:14`): the entries of h are then a
    scrambled arrangement of the same products, which the estimator -- linear in
    whatever h is -- does not care about."""
    sd = math.sqrt(varh / 2)
    H_BU = rs.normal(0.0, sd, (n_rx, 2 * n_tx)).view(np.complex128)
    H_BS = rs.normal(0.0, sd, (N, 2 * n_tx)).view(np.complex128)
    H_SU = rs.normal(0.0, sd, (n_rx, 2 * N)).view(np.complex128)
    if flatten == "C":
        kr = H_BS.T[:, None, :] * H_SU[None, :, :]          # (n_tx, n_rx, N): row j*n_rx+r, col n
        h = np.concatenate((H_BU.reshape(-1), kr.reshape(-1)))
        return h.reshape((N + 1) * n_tx, n_rx)
    Theta = np.empty((N + 1, n_tx, n_rx), dtype=np.complex128)
    Theta[0] = H_BU.T
    Theta[1:] = H_BS[:, :, None] * H_SU.T[:, None, :]
    return Theta.reshape((N + 1) * n_tx, n_rx)


def draw_symbols(n_tx, M, T, rs=np.random):
    """`Proposed method/PM.py:19-24,34-40`: T draws of n_tx i.i.d. constellation
    indices (one `choice` call per symbol time).  Returns (idx (T,n_tx), X (T,n_tx))."""
    cons = qam_constellation(M)
    idx = np.empty((T, n_tx), dtype=np.int64)
    for t in range(T):
        idx[t] = rs.choice(range(0, M), n_tx, True)
    return idx, cons[idx]


def irs_phases(T_p, T_d, N, rs=np.random, beta_min=0.0, beta_max=2 * math.pi, amp=1.0,
               variant="pm"):
    """RIS phase designs, returned already in the estimator layout
    (PsiP (T_p,N+1), PsiD (T_d,N+1)), i.e. after the driver's np.insert of the
    direct-link ones row.

    variant "pm"  : `Proposed method/PM.py:119-130,179` -- pilots exp(-j2pi t n/N)
                    for n<N written into rows 0..N-1 of an (N+1,T_p) zero array
                    (so row 0 is all-ones and row N stays ZERO: last element off
                    during pilots); data phases exp(j U(0,2pi)) + ones row.
    variant "top_tp": `Proposed_method_NMSEvsTp.py:72-83,129-130` -- pilots
                    exp(-j2pi t n/T_p), n<N, ones row inserted; data as "pm".
    variant "top_td": `Proposed_method_NMSEvsTd.py:80-96` -- pilots as "top_tp";
                    data deterministic exp(-j2pi t n/T_d) over n = 0..N (no RNG)."""
    # phase arguments are formed with Python scalar arithmetic exactly as the
    # reference does ((-1j*2*pi*t*n)/N): numpy's array complex division multiplies
    # by a reciprocal and lands 1 ulp away, which would break byte-identity.
    def dft(T, rows, denom):
        arg = np.array([[(-1j * 2 * np.pi * (t) * (n)) / (denom) for n in range(rows)] for t in range(T)],
                       dtype=np.complex128).reshape(T, rows)
        return np.exp(arg)

    if variant == "pm":
        PsiP = np.zeros((T_p, N + 1), dtype=np.complex128)
        PsiP[:, :N] = dft(T_p, N, N)
    else:
        PsiP = np.ones((T_p, N + 1), dtype=np.complex128)
        PsiP[:, 1:] = dft(T_p, N, T_p)
    if variant == "top_td":
        PsiD = dft(T_d, N + 1, T_d)
    else:
        PsiD = np.ones((T_d, N + 1), dtype=np.complex128)
        for t in range(T_d):
            beta = (beta_max - beta_min) * rs.uniform(0, 1, (N, 1)) + beta_min
            PsiD[t, 1:] = (amp * np.exp(1j * beta))[:, 0]
    return PsiP, PsiD


def design_rows(Psi, X):
    """w_t = psi~_t (x) x_t, shape (T, L): the only non-trivial row of the
    reference's dense Z_t (`Proposed method/PM.py:138`)."""
    T = Psi.shape[0]
    return (Psi[:, :, None] * X[:, None, :]).reshape(T, -1)


def received_signals(PsiP, PsiD, Xp, Xd, Theta_true, varn, rs=np.random):
    """`Proposed method/PM.py:132-148`: Y = Z h + n with n = normal(0, sqrt(varn/2),
    (n_rx,2)).view(complex), pilots first then data, one RNG call per symbol time;
    LS start theta0 = pinv(vstack Z_p) vstack Y_p (:147).  Because
    Z_p = W_p (x) I_nrx, pinv(Z_p) = pinv(W_p) (x) I_nrx exactly."""
    n_rx = Theta_true.shape[1]
    sd = math.sqrt(varn / 2)
    Wp = design_rows(PsiP, Xp)
    Wd = design_rows(PsiD, Xd)
    Yp = Wp @ Theta_true
    for t in range(Wp.shape[0]):
        Yp[t] += rs.normal(0.0, sd, (n_rx, 2)).view(np.complex128)[:, 0]
    Yd = Wd @ Theta_true
    for t in range(Wd.shape[0]):
        Yd[t] += rs.normal(0.0, sd, (n_rx, 2)).view(np.complex128)[:, 0]
    theta0 = np.linalg.pinv(Wp) @ Yp
    return Yp, Yd, theta0


def gen_trial(N, n_tx, n_rx, M, T_p, T_d, varn, seed=None, order="pm", variant="pm", rs=None):
    """One seeded realisation in the reference's draw order.
    order "pm"  : channel, data symbols, RIS phases, pilot symbols, noise
                  (`Proposed method/PM.py:174-183`)
    order "rev4": channel, data symbols, pilot symbols, RIS phases, noise
                  (`Proposed method/Proposed_method_NMSEvsTp.py:155-163`)"""
    if rs is None:
        rs = np.random.RandomState(seed)
    Theta_true = channel_vector(n_tx, n_rx, N, 1.0, rs)
    idx_d, Xd = draw_symbols(n_tx, M, T_d, rs)
    if order == "rev4":
        idx_p, Xp = draw_symbols(n_tx, M, T_p, rs)
        PsiP, PsiD = irs_phases(T_p, T_d, N, rs, variant=variant)
    else:
        PsiP, PsiD = irs_phases(T_p, T_d, N, rs, variant=variant)
        idx_p, Xp = draw_symbols(n_tx, M, T_p, rs)
    Yp, Yd, theta0 = received_signals(PsiP, PsiD, Xp, Xd, Theta_true, varn, rs)
    return dict(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, varn=float(varn),
                h=Theta_true, Xd=Xd, Xp=Xp, idx_d=idx_d, idx_p=idx_p, PsiP=PsiP, PsiD=PsiD,
                Yp=Yp, Yd=Yd, theta0=theta0)


# --------------------------------------------------------------------------
# E-step pieces
# --------------------------------------------------------------------------

def effective_channels(PsiD, Theta, n_tx):
    """Heff[t, r, j] = sum_n' psi~[t,n'] Theta[n'*n_tx+j, r] -- what
    Z(x, psi~_t) theta collapses to (`Proposed_method_NMSEvsTp.py:56`)."""
    T_d, N1 = PsiD.shape
    n_rx = Theta.shape[1]
    Th = Theta.reshape(N1, n_tx, n_rx)
    return np.einsum("tn,njr->trj", PsiD, Th)


def hypothesis_distances(Yd, Heff, table):
    """d2[t,k] = || y_t - Heff_t x_k ||^2   (`Proposed_method_NMSEvsTp.py:56-57`)."""
    pred = np.einsum("trj,kj->tkr", Heff, table)
    res = Yd[:, None, :] - pred
    return (res.real ** 2 + res.imag ** 2).sum(axis=2)


def posterior_stats(Yd, PsiD, Theta, cons, n_tx, varn, hard=False, chunk=None):
    """Per-symbol sufficient statistics of the E-step.

    soft (`Proposed_method_NMSEvsTp.py:53-62`): beta = softmax_k(-d2/varn**2)
    (NOTE varn**2, quirk Q1), m_t = sum beta conj(x_k), R_t = sum beta conj(x_k) x_k^T.
    hard (`Proposed method/ML_detecctor.py:66-77`): k* = argmax_k beta (first index
    on ties == argmin d2), rank-one statistics at x_{k*}.
    Also returns kstar (T_d,) and lse (T_d,) = log sum_k exp(-d2/varn**2)."""
    T_d = Yd.shape[0]
    M = len(cons)
    K = M ** n_tx
    Heff = effective_channels(PsiD, Theta, n_tx)
    s2 = float(varn) ** 2
    m = np.zeros((T_d, n_tx), dtype=np.complex128)
    R = np.zeros((T_d, n_tx, n_tx), dtype=np.complex128)
    kstar = np.zeros(T_d, dtype=np.int64)
    lse = np.zeros(T_d)
    if chunk is None:
        chunk = max(1, min(T_d, (1 << 22) // max(K, 1)))
    if K <= (1 << 16):
        table = hypothesis_table(cons, n_tx)
    else:
        table = cons[hypothesis_digits(np.arange(K), M, n_tx)]
    for t0 in range(0, T_d, chunk):
        sl = slice(t0, min(T_d, t0 + chunk))
        d2 = hypothesis_distances(Yd[sl], Heff[sl], table)
        ks = np.argmin(d2, axis=1)
        dmin = d2[np.arange(d2.shape[0]), ks]
        a = -(d2 - dmin[:, None]) / s2
        e = np.exp(a)
        se = e.sum(axis=1)
        kstar[sl] = ks
        lse[sl] = -dmin / s2 + np.log(se)
        if hard:
            xs = table[ks]
            m[sl] = xs.conj()
            R[sl] = xs.conj()[:, :, None] * xs[:, None, :]
        else:
            beta = e / se[:, None]
            m[sl] = beta @ table.conj()
            R[sl] = np.einsum("tk,ki,kj->tij", beta, table.conj(), table, optimize=True)
    return m, R, kstar, lse


def posterior_stats_split(Yd, PsiD, Theta, cons, n_tx, varn, hard=False):
    """posterior_stats for trees too large for one hypothesis table (2^24 leaves: 4 streams of 64-QAM, 6 of
    16-QAM).  The streams are split into a leading half A and a trailing half B (k = a * K_B + b); the residual
    y - H_A x_a - H_B x_b and its squared norm are still formed directly for every (a, b), block by block, and
    the posterior sums reduce over b (statistics of A), over a (statistics of B) and through one
    conj(X_A)^T beta X_B product (cross terms of R)."""
    T_d = Yd.shape[0]
    M = len(cons)
    nA = n_tx // 2
    XA, XB = hypothesis_table(cons, nA), hypothesis_table(cons, n_tx - nA)
    KA, KB = len(XA), len(XB)
    Heff = effective_channels(PsiD, Theta, n_tx)
    s2 = float(varn) ** 2
    m = np.zeros((T_d, n_tx), dtype=np.complex128)
    R = np.zeros((T_d, n_tx, n_tx), dtype=np.complex128)
    kstar = np.zeros(T_d, dtype=np.int64)
    lse = np.zeros(T_d)
    rows = max(1, (1 << 21) // KB)
    for t in range(T_d):
        u = Yd[t][None, :] - XA @ Heff[t][:, :nA].T            # (KA, n_rx)
        v = XB @ Heff[t][:, nA:].T                             # (KB, n_rx)
        d2 = np.empty((KA, KB))
        for a0 in range(0, KA, rows):
            r = u[a0:a0 + rows, None, :] - v[None, :, :]
            d2[a0:a0 + rows] = (r.real ** 2 + r.imag ** 2).sum(axis=2)
        k = int(np.argmin(d2))
        dmin = d2.flat[k]
        e = np.exp(-(d2 - dmin) / s2)
        se = e.sum()
        kstar[t] = k
        lse[t] = -dmin / s2 + np.log(se)
        if hard:
            x = np.concatenate([XA[k // KB], XB[k % KB]])
            m[t] = x.conj()
            R[t] = x.conj()[:, None] * x[None, :]
            continue
        beta = e / se
        bA, bB = beta.sum(axis=1), beta.sum(axis=0)
        m[t, :nA], m[t, nA:] = bA @ XA.conj(), bB @ XB.conj()
        R[t, :nA, :nA] = np.einsum("a,ai,aj->ij", bA, XA.conj(), XA)
        R[t, nA:, nA:] = np.einsum("b,bi,bj->ij", bB, XB.conj(), XB)
        R[t, :nA, nA:] = XA.conj().T @ beta @ XB
        R[t, nA:, :nA] = R[t, :nA, nA:].conj().T
    assert KA * KB == M ** n_tx
    return m, R, kstar, lse


# --------------------------------------------------------------------------
# M-step pieces
# --------------------------------------------------------------------------

def gram_and_rhs(Psi, Y, m, R):
    """G = sum_t (psi~_t^* psi~_t^T) (x) R_t  (L,L),  B = sum_t (psi~_t^* (x) m_t) y_t^T (L,n_rx).
    Equals the reference's D x D accumulators divided out by the trailing (x) I_nrx
    (`Proposed_method_NMSEvsTp.py:61-62`: Z^H Z = (w^* w^T) (x) I, Z^H y = w^* (x) y)."""
    T, N1 = Psi.shape
    n_tx = m.shape[1]
    L = N1 * n_tx
    G = np.einsum("tn,tp,tij->nipj", Psi.conj(), Psi, R, optimize=True).reshape(L, L)
    V = (Psi.conj()[:, :, None] * m[:, None, :]).reshape(T, L)
    B = V.T @ Y
    return G, B


def pilot_stats(Xp):
    """Pilots are symbols known with probability one: m = conj(x), R = conj(x) x^T
    (`Proposed_method_NMSEvsTp.py:63-65`)."""
    return Xp.conj(), Xp.conj()[:, :, None] * Xp[:, None, :]


def solve_normal(G, B, how="solve"):
    """`np.linalg.solve` (`Proposed_method_NMSEvsTp.py:66`) or `np.linalg.lstsq`
    (`Proposed method/PM.py:108`) on the L x L system (the reference solves the
    Kronecker-expanded D x D system (G (x) I_nrx) theta = vec(B); identical)."""
    if how == "lstsq":
        return np.linalg.lstsq(G, B, rcond=None)[0]
    return np.linalg.solve(G, B)


# --------------------------------------------------------------------------
# metrics
# --------------------------------------------------------------------------

def nmse(Theta_hat, Theta_true):
    """`Proposed_method_NMSEvsTp.py:138`: ||theta^ - h||^2 / ||h||^2."""
    d = Theta_hat - Theta_true
    return float((d.real ** 2 + d.imag ** 2).sum() / (Theta_true.real ** 2 + Theta_true.imag ** 2).sum())


def llf_as_coded(Theta, Yp, Yd, PsiP, PsiD, Xp, Xd_true, M, varn):
    """The thesis "LLF" exactly as coded (`Proposed method/ML_detecctor.py:55-57,84`):
    un-squared Frobenius norms of the stacked residual blocks, Z_d built from the
    TRUE data symbols (quirk Q7)."""
    T_p, T_d = Yp.shape[0], Yd.shape[0]
    n_tx = Xp.shape[1]
    rp = Yp - design_rows(PsiP, Xp) @ Theta
    rd = Yd - design_rows(PsiD, Xd_true) @ Theta
    e1 = T_d * n_tx * math.log(M)
    e2 = (T_d + T_p) * math.log(math.pi * varn ** 2)
    return float(-e1 - e2 - np.linalg.norm(rp) / varn ** 2 - np.linalg.norm(rd) / varn ** 2)


def ser_as_coded(Xd_true, X_est):
    """`Proposed method/SER/log_max_SER.py:162`: count_nonzero over the
    (T_d, n_tx, n_tx) broadcast of (T_d,n_tx,1) - (T_d,1,n_tx) (quirk Q8)."""
    T_d, n_tx = Xd_true.shape
    diff = Xd_true[:, :, None] - X_est[:, None, :]
    return float(np.count_nonzero(diff) / (T_d * n_tx))


def ser_true(Xd_true, X_est):
    return float(np.count_nonzero(Xd_true - X_est) / Xd_true.size)


# --------------------------------------------------------------------------
# estimators
# --------------------------------------------------------------------------

def em(Yd, Yp, PsiD, PsiP, Xp, M, varn, itera, theta0=None, n_tx=None, hard=False,
       h_true=None, genie_stop=False, Xd_true=None, return_trace=False):
    """Soft (`Proposed_method_NMSEvsTp.py:43-69`, theta0 = 0;
    `Proposed method/Proposed_method_NMSEvsTp.py:50-83`, theta0 = LS) or hard
    (`Proposed method/ML_detecctor.py:51-86`) decision EM, full enumeration.

    genie_stop reproduces `Proposed method/PMvsMLvsZFvsMMSE.py:169,288`:
    break when | ||theta|| - ||h|| | < 1 and l != 0.
    Returns Theta (L,n_rx) and a dict: kstar of the LAST executed iteration
    (decisions made before that iteration's M-step, `SER/log_max_SER.py:77-78`),
    llf (as coded, per iteration, if Xd_true given), lse (proper incomplete-data
    log-likelihood sum_t log sum_k per iteration, evaluated at the theta that
    entered the iteration), iters executed."""
    n_tx = Xp.shape[1] if n_tx is None else n_tx
    N1 = PsiD.shape[1]
    L = N1 * n_tx
    n_rx = Yd.shape[1]
    cons = qam_constellation(M)
    Theta = np.zeros((L, n_rx), dtype=np.complex128) if theta0 is None else np.array(theta0, dtype=np.complex128)
    mp_, Rp_ = pilot_stats(Xp)
    Gp, Bp = gram_and_rhs(PsiP, Yp, mp_, Rp_)
    trace = dict(llf=[], lse=[], norm=[], kstar=None, iters=0)
    for l in range(itera):
        m, R, kstar, lse = posterior_stats(Yd, PsiD, Theta, cons, n_tx, varn, hard=hard)
        Gd, Bd = gram_and_rhs(PsiD, Yd, m, R)
        Theta = solve_normal(Gp + Gd, Bp + Bd)
        trace["kstar"] = kstar
        trace["lse"].append(float(lse.sum()))
        trace["norm"].append(float(np.linalg.norm(Theta)))
        trace["iters"] = l + 1
        if Xd_true is not None:
            trace["llf"].append(llf_as_coded(Theta, Yp, Yd, PsiP, PsiD, Xp, Xd_true, M, varn))
        if genie_stop and h_true is not None and l != 0 and abs(np.linalg.norm(Theta) - np.linalg.norm(h_true)) < 1:
            break
    return (Theta, trace) if return_trace else Theta


def em_superimposed(Y, Psi, Xoff, M, varn, itera, n_tx=None, hard=False, return_trace=False):
    """Parallel protocol, `Parallel/ParallelProtocol_Tp.py:64-86`: pilots are superimposed on the data,
    the hypotheses of symbol t are x_k + o_t (o_t = pilot symbol, zero beyond the pilot length, :56-62),
    there is no separate pilot term and theta starts at 0.  With x~ = x + o:
        d2_k = ||(y - Heff o) - Heff x_k||^2,  m~ = m + conj(o),
        R~_ij = R_ij + m_i o_j + conj(o_i) conj(m_j) + conj(o_i) o_j."""
    n_tx = Xoff.shape[1] if n_tx is None else n_tx
    L, n_rx = Psi.shape[1] * n_tx, Y.shape[1]
    cons = qam_constellation(M)
    Theta = np.zeros((L, n_rx), dtype=np.complex128)
    trace = dict(kstar=None, lse=[], iters=0)
    for l in range(itera):
        Heff = effective_channels(Psi, Theta, n_tx)
        Yshift = Y - np.einsum("trj,tj->tr", Heff, Xoff)
        m, R, kstar, lse = posterior_stats(Yshift, Psi, Theta, cons, n_tx, varn, hard=hard)
        Rt = (R + m[:, :, None] * Xoff[:, None, :] + Xoff.conj()[:, :, None] * m.conj()[:, None, :]
              + Xoff.conj()[:, :, None] * Xoff[:, None, :])
        mt = m + Xoff.conj()
        G, B = gram_and_rhs(Psi, Y, mt, Rt)
        Theta = solve_normal(G, B)
        trace["kstar"] = kstar
        trace["lse"].append(float(lse.sum()))
        trace["iters"] = l + 1
    return (Theta, trace) if return_trace else Theta


def _argmax_complex_first(v):
    """np.argmax on a complex vector orders lexicographically (real, then imag),
    first index on ties (`Proposed method/PM.py:67`)."""
    return int(np.argmax(v))


def pm_candidates(y, channel, cons, p1):
    """Candidate list of one data symbol, `Proposed method/PM.py:61-102`.
    channel (n_rx,n_tx) is the (quirky, Q4) effective channel.  Returns the
    (M**p1, n_tx) candidate vectors IN ORDERED POSITION (quirk Q5: never permuted
    back to stream order) and the stream order j."""
    n_tx = channel.shape[1]
    j, j_c, arr = [], list(range(n_tx)), channel
    for _ in range(n_tx):
        yeta = np.diag(np.linalg.pinv(arr.conj().T @ arr))
        k = _argmax_complex_first(yeta)
        j.append(j_c[k])
        arr = np.delete(arr, k, axis=1)
        del j_c[k]
    A = channel[:, j[:p1]]
    Bc = channel[:, j[p1:]]
    nB = n_tx - p1
    tabA = hypothesis_table(cons, p1)
    cands = np.empty((tabA.shape[0], n_tx), dtype=np.complex128)
    if nB > 0:
        pinvB = np.linalg.inv(Bc.conj().T @ Bc) @ Bc.conj().T
    for i in range(tabA.shape[0]):
        cands[i, :p1] = tabA[i]
        if nB > 0:
            z = pinvB @ (y - A @ tabA[i])
            # joint argmin over M**nB vectors of ||z-b||^2 separates per stream
            # (first index on ties in product order == per-stream first index)
            for s in range(nB):
                cands[i, p1 + s] = cons[int(np.argmin(np.abs(z[s] - cons) ** 2))]
    return cands, j


def pm_stats(Yd, PsiD, Theta, cons, n_tx, varn, partition_r, weighted, quirks=True):
    """Per-symbol statistics of the partitioned estimator.
    weighted=False: `Proposed method/PM.py:94-104` (every candidate weight 1, NOT
    normalised); weighted=True: `Proposed method/PM_beta.py:87-95` (posterior over
    the candidate list, evaluated with the FULL psi~_t)."""
    T_d, N1 = PsiD.shape
    N = N1 - 1
    n_rx = Yd.shape[1]
    M = len(cons)
    p1 = int(partition_r / math.log2(M)) + 1
    Th = Theta.reshape(N1, n_tx, n_rx)
    m = np.zeros((T_d, n_tx), dtype=np.complex128)
    R = np.zeros((T_d, n_tx, n_tx), dtype=np.complex128)
    Heff = effective_channels(PsiD, Theta, n_tx)
    for t in range(T_d):
        if quirks:
            # PM.py:63 uses PsiTilde_td[:N,t] AFTER the ones row was inserted (:179):
            # phases [1, psi_0..psi_{N-2}] paired with RIS elements 0..N-1.
            chan = Th[0].T + np.einsum("n,njr->rj", PsiD[t, :N], Th[1:])
        else:
            chan = Heff[t]
        cands, _ = pm_candidates(Yd[t], chan, cons, p1)
        if not quirks:
            # un-permute to stream order
            _, order = pm_candidates(Yd[t], chan, cons, p1)
            fixed = np.empty_like(cands)
            fixed[:, order] = cands
            cands = fixed
        if weighted:
            res = Yd[t][None, :] - cands @ Heff[t].T
            d2 = (res.real ** 2 + res.imag ** 2).sum(axis=1)
            a = -(d2 - d2.min()) / float(varn) ** 2
            w = np.exp(a)
            w /= w.sum()
        else:
            w = np.ones(cands.shape[0])
        m[t] = w @ cands.conj()
        R[t] = np.einsum("k,ki,kj->ij", w, cands.conj(), cands)
    return m, R


def _boundary_margin(z, sqM):
    """Smallest distance of the real and imaginary parts of z to a decision boundary of the per-axis slicer
    (levels at the odd integers -sqM+1..sqM-1, boundaries at the even integers between them)."""
    bounds = np.arange(-sqM + 2, sqM - 1, 2, dtype=np.float64)
    v = np.concatenate([np.ravel(np.real(z)), np.ravel(np.imag(z))])
    if v.size == 0:
        return math.inf
    return float(np.abs(v[:, None] - bounds[None, :]).min())


def _order_trace(channel):
    """Stream order of `Proposed method/PM.py:65-70` and, over its rounds, the smallest relative gap between the
    largest and second-largest diag(pinv(A^H A)) (the arg-max decision of the round)."""
    n_tx = channel.shape[1]
    j, j_c, arr, gap = [], list(range(n_tx)), channel, math.inf
    for _ in range(n_tx):
        yeta = np.diag(np.linalg.pinv(arr.conj().T @ arr))
        k = _argmax_complex_first(yeta)
        if len(yeta) > 1:
            s = np.sort(yeta.real)
            gap = min(gap, float((s[-1] - s[-2]) / abs(s[-1])))
        j.append(j_c[k])
        arr = np.delete(arr, k, axis=1)
        del j_c[k]
    return j, gap


def _fsum_c(v):
    return complex(math.fsum(np.real(v)), math.fsum(np.imag(v)))


def pm_stats_trace(Yd, PsiD, Theta, cons, n_tx, varn, p1, weighted, quirks=True):
    """pm_stats (p1 = p+1 streams enumerated) with a per-symbol trace for kernel tests.  Returns (m, R, trace);
    trace[t] holds the stream `order`, the candidate list `cands` (as the statistics use it), the `weights`
    (normalised for PM-beta, 1 for PM), and the margins of every discrete decision on the way:
        order_gap  relative gap between the largest and second-largest diag(pinv(A^H A)) of each ordering round
        slice_gap  smallest distance of a zero-forced value z of set B to a decision boundary of its axis
    m_t and R_t are summed exactly (math.fsum) over weights normalised in long double."""
    T_d, N1 = PsiD.shape
    N = N1 - 1
    n_rx = Yd.shape[1]
    M = len(cons)
    sqM = int(round(math.sqrt(M)))
    Th = Theta.reshape(N1, n_tx, n_rx)
    Heff = effective_channels(PsiD, Theta, n_tx)
    tabA = hypothesis_table(cons, p1)
    nB = n_tx - p1
    m = np.zeros((T_d, n_tx), dtype=np.complex128)
    R = np.zeros((T_d, n_tx, n_tx), dtype=np.complex128)
    trace = []
    for t in range(T_d):
        chan = Th[0].T + np.einsum("n,njr->rj", PsiD[t, :N], Th[1:]) if quirks else Heff[t]
        order, order_gap = _order_trace(chan)
        cands = np.empty((len(tabA), n_tx), dtype=np.complex128)
        cands[:, :p1] = tabA
        slice_gap = math.inf
        if nB > 0:
            A, Bc = chan[:, order[:p1]], chan[:, order[p1:]]
            z = (np.linalg.inv(Bc.conj().T @ Bc) @ Bc.conj().T @ (Yd[t][:, None] - A @ tabA.T)).T   # (K, nB)
            slice_gap = _boundary_margin(z, sqM)
            cands[:, p1:] = cons[np.argmin(np.abs(z[:, :, None] - cons[None, None, :]) ** 2, axis=2)]
        if not quirks:
            fixed = np.empty_like(cands)
            fixed[:, order] = cands
            cands = fixed
        if weighted:
            res = Yd[t][None, :] - cands @ Heff[t].T
            d2 = (res.real ** 2 + res.imag ** 2).sum(axis=1)
            e = np.exp(-(d2 - d2.min()).astype(np.longdouble) / np.longdouble(varn) ** 2)
            w = (e / e.sum()).astype(np.float64)
        else:
            w = np.ones(len(cands))
        for i in range(n_tx):
            m[t, i] = _fsum_c(w * cands[:, i].conj())
            for k in range(n_tx):
                R[t, i, k] = _fsum_c(w * cands[:, i].conj() * cands[:, k])
        trace.append(dict(order=order, cands=cands, weights=w, order_gap=order_gap, slice_gap=slice_gap))
    return m, R, trace


def detector_stats_trace(Yd, PsiD, Theta, cons, n_tx, varn, kind, quirks=True):
    """detector_stats with the decisions and their margins, for kernel tests.  Returns (m, R, kstar, trace);
    kstar[t] is the joint hypothesis index of the decision, trace[t] holds the estimate `est` (ZF: pinv(H) y in
    float64; MMSE: inv(H^H H + varn^2 I) H^H y) and
        slice_gap  proper slicer (quirks off): smallest distance of est to a decision boundary of its axis
        pair_gap   as-coded slicer (quirks on): gap between the best and second-best (stream, point) distance."""
    T_d, N1 = PsiD.shape
    N = N1 - 1
    n_rx = Yd.shape[1]
    M = len(cons)
    sqM = int(round(math.sqrt(M)))
    Th = Theta.reshape(N1, n_tx, n_rx)
    Heff = effective_channels(PsiD, Theta, n_tx)
    m = np.zeros((T_d, n_tx), dtype=np.complex128)
    R = np.zeros((T_d, n_tx, n_tx), dtype=np.complex128)
    kstar = np.zeros(T_d, dtype=np.int64)
    trace = []
    for t in range(T_d):
        chan = Th[0].T + np.einsum("n,njr->rj", PsiD[t, :N], Th[1:]) if quirks else Heff[t]
        if kind == "zf":
            est = np.linalg.pinv(chan) @ Yd[t]
        else:
            est = np.linalg.inv(chan.conj().T @ chan + (varn ** 2) * np.eye(n_tx)) @ chan.conj().T @ Yd[t]
        tr = dict(est=est, slice_gap=math.inf, pair_gap=math.inf)
        if quirks:
            dig = slicer_as_coded(est, cons, n_tx)
            dist = np.sort(np.abs(est.reshape(-1, 1) - cons.reshape(1, -1)).ravel())
            tr["pair_gap"] = float(dist[1] - dist[0]) if dist.size > 1 else math.inf
        else:
            dig = np.array([int(np.argmin(np.abs(est[j] - cons) ** 2)) for j in range(n_tx)])
            tr["slice_gap"] = _boundary_margin(est, sqM)
        kstar[t] = int(sum(int(dig[j]) * M ** (n_tx - 1 - j) for j in range(n_tx)))
        x = cons[dig]
        m[t] = x.conj()
        R[t] = x.conj()[:, None] * x[None, :]
        trace.append(tr)
    return m, R, kstar, trace


def em_pm(Yd, Yp, PsiD, PsiP, Xp, M, varn, itera, theta0, h_true=None, partition_r=0,
          weighted=False, genie_stop=True, quirks=True, how=None, return_trace=False):
    """Partitioned EM: `Proposed method/PM.py:47-116` (weighted=False, lstsq) and
    `Proposed method/PM_beta.py:42-112` / `PMvsMLvsZFvsMMSE.py:176-246`
    (weighted=True, solve)."""
    n_tx = Xp.shape[1]
    cons = qam_constellation(M)
    Theta = np.array(theta0, dtype=np.complex128)
    mp_, Rp_ = pilot_stats(Xp)
    Gp, Bp = gram_and_rhs(PsiP, Yp, mp_, Rp_)
    how = how or ("solve" if weighted else "lstsq")
    iters = 0
    for l in range(itera):
        m, R = pm_stats(Yd, PsiD, Theta, cons, n_tx, varn, partition_r, weighted, quirks)
        Gd, Bd = gram_and_rhs(PsiD, Yd, m, R)
        Theta = solve_normal(Gp + Gd, Bp + Bd, how)
        iters = l + 1
        if genie_stop and h_true is not None and l != 0 and abs(np.linalg.norm(Theta) - np.linalg.norm(h_true)) < 1:
            break
    return (Theta, dict(iters=iters)) if return_trace else Theta


# --------------------------------------------------------------------------
# detector-driven EM (zero forcing / MMSE), SURVEY section 8f-3
# --------------------------------------------------------------------------

def slicer_as_coded(data_est, cons, n_tx):
    """`Proposed method/PMvsMLvsZFvsMMSE.py:49-52` (nearest_symbol_ecul) as it is CALLED
    (:68,:109): `estimated_symbol` is (n_tx,1), `constellation` is the (K,n_tx) hypothesis table, so
    `estimated_symbol - s` broadcasts to (n_tx,n_tx) and np.argmin runs over the flattened
    (K,n_tx,n_tx) array of |data_est[i] - s_k[j]|; the flat index is then used as a ROW index into the
    table (quirk; SURVEY 8f-3).  Closed form of that flat index: let (i*, c*) minimise
    |data_est[i] - c| over streams and constellation points (first i on ties, first c on ties); the
    first table row containing c* is k = idx(c*), where it sits in the last stream (or in stream 0
    when idx = 0), hence flat = idx * n_tx^2 + i* * n_tx + (n_tx-1 if idx else 0)."""
    M = len(cons)
    dist = np.abs(data_est.reshape(-1, 1) - cons.reshape(1, -1))      # (n_tx, M)
    vmin = dist.min()
    # first (k,i,j) in flat order attaining vmin: smallest idx first, then smallest i
    cand = [(int(c), int(i)) for i in range(n_tx) for c in range(M) if dist[i, c] == vmin]
    idx, i_star = min(cand)
    flat = idx * n_tx * n_tx + i_star * n_tx + ((n_tx - 1) if idx else 0)
    if flat >= M ** n_tx:
        raise IndexError("reference slicer indexes past the hypothesis table")
    return hypothesis_digits(np.array(flat), M, n_tx)


def detector_stats(Yd, PsiD, Theta, cons, n_tx, varn, kind, quirks=True):
    """Per-symbol rank-one statistics of `em_zf` / `em_mmse`
    (`Proposed method/PMvsMLvsZFvsMMSE.py:54-133`): effective channel with the off-by-one psi slice
    (:64,:105, quirk Q4), x = pinv(H) y (ZF, :66) or inv(H^H H + varn^2 I) H^H y (MMSE, :107), then the
    slicer above (quirks) or a proper per-stream nearest-point slicer (quirks off)."""
    T_d, N1 = PsiD.shape
    N = N1 - 1
    n_rx = Yd.shape[1]
    M = len(cons)
    Th = Theta.reshape(N1, n_tx, n_rx)
    Heff = effective_channels(PsiD, Theta, n_tx)
    m = np.zeros((T_d, n_tx), dtype=np.complex128)
    R = np.zeros((T_d, n_tx, n_tx), dtype=np.complex128)
    for t in range(T_d):
        if quirks:
            chan = Th[0].T + np.einsum("n,njr->rj", PsiD[t, :N], Th[1:])
        else:
            chan = Heff[t]
        if kind == "zf":
            est = np.linalg.pinv(chan) @ Yd[t]
        else:
            est = np.linalg.inv(chan.conj().T @ chan + (varn ** 2) * np.eye(n_tx)) @ chan.conj().T @ Yd[t]
        if quirks:
            dig = slicer_as_coded(est, cons, n_tx)
        else:
            dig = np.array([int(np.argmin(np.abs(est[j] - cons) ** 2)) for j in range(n_tx)])
        x = cons[dig]
        m[t] = x.conj()
        R[t] = x.conj()[:, None] * x[None, :]
    return m, R


def em_detector(Yd, Yp, PsiD, PsiP, Xp, M, varn, itera, theta0, kind="zf", h_true=None, genie_stop=True,
                quirks=True, return_trace=False, zf_stop_guard=False):
    """`em_zf` (`PMvsMLvsZFvsMMSE.py:95-133`) / `em_mmse` (:54-93).  NOTE the genie stop of em_zf has no
    `l != 0` guard (:128) while em_mmse's has (:87); `all_detectorsvsTd.py:127` has the guard in em_zf too
    (zf_stop_guard=True) and `SNR/all_Detectors.py` has no stop in em / em_ml / em_zf / em_mmse (genie_stop=False)."""
    n_tx = Xp.shape[1]
    cons = qam_constellation(M)
    Theta = np.array(theta0, dtype=np.complex128)
    mp_, Rp_ = pilot_stats(Xp)
    Gp, Bp = gram_and_rhs(PsiP, Yp, mp_, Rp_)
    iters = 0
    for l in range(itera):
        m, R = detector_stats(Yd, PsiD, Theta, cons, n_tx, varn, kind, quirks)
        Gd, Bd = gram_and_rhs(PsiD, Yd, m, R)
        Theta = solve_normal(Gp + Gd, Bp + Bd)
        iters = l + 1
        if genie_stop and h_true is not None and (l != 0 or (kind == "zf" and not zf_stop_guard)) \
                and abs(np.linalg.norm(Theta) - np.linalg.norm(h_true)) < 1:
            break
    return (Theta, dict(iters=iters)) if return_trace else Theta
