"""TEST INFRASTRUCTURE ONLY -- extended-precision reference for the E-step statistics (csrc/estep.cu: k_heff_qr*,
k_enum) on top of oracle/em_numpy.py (effective_channels, hypothesis_table, which stay pinned to the reference
goldens), and an accuracy bound derived from the kernels' arithmetic, not fitted to their output.

Reference.  Heff_t and every squared distance d2_k = ||y'_t - Heff_t x_k||^2 are formed directly in np.clongdouble
(64-bit mantissa) from the FP64 inputs, with y'_t = y_t - Heff_t o_t for superimposed pilot offsets o_t.  From
them: the posterior beta_k = exp(-(d2_k - d2*)/varn^2) / Z, m = sum beta conj(x), R = sum beta conj(x) x^T,
lse = -d2*/varn^2 + ln Z, the exact arg-min k* (first index on ties), the gap d2_(2) - d2*, and the count n_win of
hypotheses with d2_k <= d2* + 64 varn^2.  The FP64 oracle agrees with this to 2e-13 relative or better; the
device computes its distances differently (Householder QR, then a tree walk), so it is checked against this
reference, not against the oracle.

Bound.  The device evaluates d2_k as ||(y' + dy) - (Heff + dH) x_k||^2 up to rounding in the final sums:
  * the RIS contraction Heff_t = sum_n psi_tn Theta_n (N+1 complex multiply-adds, two real FMAs per part, in the
    lane loop and on the DMMA path alike) is exact up to |dH_rj| <= gamma_{2(N+2)} sum_n |psi_tn| |Theta_{n j, r}|,
    whose effect on the residual is at most c_c u ||(|Psi_t| |Theta|)||_F (x_max sqrt(n_tx) + ||o_t||),
    c_c = 2 (N + 2);
  * the Householder reduction of [Heff_t | y'_t] (NR = max(n_rx, n_tx) rows) and the tree's residual updates are
    backward stable: the distances are those of [Heff + dH | y' + dy] with ||dy|| + ||dH||_F ||x|| bounded by
    c_d u (||y'_t|| + ||Heff_t||_F (x_max sqrt(n_tx) + ||o_t||)).  First order, one reflection per stream, each an
    inner product and an update over at most NR rows, plus one rounding per level of the walk and of the final
    sum of squares, gives c_d of order NR + n_tx + 1; complex arithmetic rounds to within 2u per operation, so
    c_d = 2 (NR + n_tx + 1).  The rounding of the sums of squares themselves is u d2_k = u ||r_k||^2, below
    ||r_k|| rho_t / c_d, so it is covered too.
So the residual vector of every hypothesis is off by at most
    rho_t = u [c_d (||y'_t|| + ||Heff_t||_F X_t) + c_c ||(|Psi_t| |Theta|)||_F X_t],   X_t = x_max sqrt(n_tx) + ||o_t||
and its squared norm by at most eps_k = 2 ||r_k|| rho_t + rho_t^2.

Softmax to first order: with delta_k = -dd2_k / varn^2, d beta_k = beta_k (delta_k - sum_j beta_j delta_j), and
writing delta_k - mean = (delta_k - delta_*) - sum_j beta_j (delta_j - delta_*),
    ||d beta||_1 <= 2 sum_{k != k*} beta_k (eps_k + eps_k*) / varn^2  =: dbeta.
It vanishes as the posterior collapses, so the bound is as tight at high SNR as at low.  Only symbols with
dbeta < 1e-3 are admitted (first order is then accurate).

Rounding of the sums: every weight in the window is an exponential of an argument of magnitude <= 64 (twice:
node weight, leaf weight; once more when the reference distance is rescaled), so its relative error is at most
(2 * 64 + 8) u; normalising doubles that, and the sums over n_win weights add n_win u.  Hence
c_s = 2 (2 * 64 + 8) + 2 = 274 covers c_s u n_win (n_win >= 1).  The bounds are
    tau_m   = x_max   (dbeta + c_s u n_win)
    tau_R   = x_max^2 (dbeta + c_s u n_win)
    tau_lse = sum_k beta_k eps_k / varn^2 + c_s u (d2*/varn^2 + |ln Z| + n_win)
(the lse sums scale d2*/varn^2, the log of the sum and the sum itself).

kstar.  If gap > 2 max(eps_k*, eps_k2) (k2 the runner-up), kstar must be k*.  Otherwise it may be any hypothesis k
whose exact distance is within eps_k + eps_k* of the minimum (both evaluations may err by that much)."""
from __future__ import annotations

import numpy as np

from oracle import em_numpy as orc

U = 2.0 ** -53           # unit roundoff of FP64
LD = np.clongdouble
THR = 64.0               # enqueue window of k_enum, in units of varn^2
C_S = 2 * (2 * THR + 8) + 2
DBETA_MAX = 1e-3         # admission: first-order term below this


def _ld(a):
    return np.asarray(a).astype(LD)


def _nrm(a, axis):
    return np.sqrt(np.sum(np.abs(np.asarray(a, dtype=np.complex128)) ** 2, axis=axis))


def residual_error(Yd, PsiD, theta, n_tx, cons, Xoff=None):
    """rho_t of the module docstring (T_d,): bound on the error of the device's residual vector of any hypothesis."""
    T_d, N1 = PsiD.shape
    n_rx = Yd.shape[1]
    NR = max(n_rx, n_tx)
    c_d = 2.0 * (NR + n_tx + 1)
    c_c = 2.0 * (N1 + 1)
    xmax = float(np.abs(cons).max())
    H = orc.effective_channels(PsiD, theta, n_tx)
    Habs = orc.effective_channels(np.abs(PsiD), np.abs(theta), n_tx)      # sum_n |psi| |Theta|
    X = xmax * np.sqrt(n_tx) + (np.zeros(T_d) if Xoff is None else _nrm(Xoff, 1))
    y = Yd if Xoff is None else Yd - np.einsum("trj,tj->tr", H, Xoff)
    return U * (c_d * (_nrm(y, 1) + _nrm(H, (1, 2)) * X) + c_c * _nrm(Habs, (1, 2)) * X)


class _Sym:
    """Accumulates the per-symbol results."""

    def __init__(self, T_d, n_tx):
        self.m = np.zeros((T_d, n_tx), dtype=LD)
        self.R = np.zeros((T_d, n_tx, n_tx), dtype=LD)
        z = lambda: np.zeros(T_d, dtype=np.longdouble)
        self.lse, self.lnZ, self.d2star, self.gap, self.beta_max = z(), z(), z(), z(), z()
        self.eps_star, self.eps2, self.dbeta, self.lse_lin = z(), z(), z(), z()
        self.kstar = np.zeros(T_d, dtype=np.int64)
        self.k2 = np.zeros(T_d, dtype=np.int64)
        self.n_win = np.zeros(T_d, dtype=np.int64)


def _eps(d2, rho):
    return 2 * np.sqrt(np.maximum(d2, 0)) * rho + rho * rho


def stats_from_d2(d2, X, varn, rho):
    """Posterior statistics and bound terms from exact distances d2 (T, K) (np.longdouble) and the hypothesis
    table X (K, n_tx).  Exposed so that tests can perturb d2 and see the bound react."""
    T, K = d2.shape
    s2 = np.longdouble(varn) ** 2
    out = _Sym(T, X.shape[1])
    Xc, Xl = _ld(X).conj(), _ld(X)
    rho = np.asarray(rho, dtype=np.longdouble)
    for t in range(T):
        d = d2[t]
        k = int(np.argmin(d))
        ds = d[k]
        dm = d.copy()
        dm[k] = np.inf
        k2 = int(np.argmin(dm)) if K > 1 else k
        w = np.exp(-(d - ds) / s2)
        Z = w.sum()
        beta = w / Z
        eps = _eps(d, rho[t])
        out.m[t] = beta @ Xc
        out.R[t] = (Xc * beta[:, None]).T @ Xl
        out.lnZ[t] = np.log(Z)
        out.lse[t] = -ds / s2 + out.lnZ[t]
        out.kstar[t], out.k2[t], out.d2star[t] = k, k2, ds
        out.gap[t] = d[k2] - ds if K > 1 else np.inf
        out.beta_max[t] = beta[k]
        out.eps_star[t], out.eps2[t] = eps[k], eps[k2]
        out.n_win[t] = int(np.count_nonzero(d <= ds + THR * s2))
        out.dbeta[t] = 2 * (np.sum(beta * (eps + eps[k])) - beta[k] * 2 * eps[k]) / s2
        out.lse_lin[t] = np.sum(beta * eps) / s2
    return out


def _finish(out, Yp, H, cons, n_tx, varn, rho, Xoff):
    out.off = None if Xoff is None else _ld(Xoff)
    out.rho = np.asarray(rho, dtype=np.longdouble)
    out.Y, out.H, out.cons, out.n_tx, out.M = Yp, H, np.asarray(cons), n_tx, len(cons)
    out.varn = float(varn)
    out.xmax = float(np.abs(cons).max())
    return out


def exact_stats(Yd, PsiD, theta, cons, n_tx, varn, Xoff=None):
    """Reference of k_enum's outputs and the bound terms for every symbol (see the module docstring); the result
    also holds the exact Heff (.H) and y' (.Y) so that d2_at() can price any hypothesis.  varn may be a sequence:
    the distances are then formed once and a list of results (one per varn) is returned."""
    varns = list(np.atleast_1d(varn))
    T_d = Yd.shape[0]
    M = len(cons)
    K = M ** n_tx
    H = orc.effective_channels(_ld(PsiD), _ld(theta), n_tx)
    Yp = _ld(Yd) if Xoff is None else _ld(Yd) - np.einsum("trj,tj->tr", H, _ld(Xoff))
    X = orc.hypothesis_table(cons, n_tx) if K <= (1 << 16) else cons[orc.hypothesis_digits(np.arange(K), M, n_tx)]
    rho = residual_error(Yd, PsiD, theta, n_tx, cons, Xoff)
    chunk = max(1, (1 << 19) // K)
    parts = [[] for _ in varns]
    for t0 in range(0, T_d, chunk):
        sl = slice(t0, min(T_d, t0 + chunk))
        r = Yp[sl, None, :] - np.einsum("trj,kj->tkr", H[sl], _ld(X))
        d2 = np.sum(r.real ** 2 + r.imag ** 2, axis=2)
        for i, v in enumerate(varns):
            parts[i].append(stats_from_d2(d2, X, v, rho[sl]))
    outs = []
    for v, ps in zip(varns, parts):
        out = _Sym(T_d, n_tx)
        for name in vars(out):
            setattr(out, name, np.concatenate([getattr(p, name) for p in ps]))
        outs.append(_finish(out, Yp, H, cons, n_tx, v, rho, Xoff))
    return outs if np.ndim(varn) else outs[0]


def exact_stats_split(Yd, PsiD, theta, cons, n_tx, varn, Xoff=None, rows=64):
    """exact_stats for the 2^24-leaf trees (4 streams of 64-QAM, 6 of 16-QAM), structured like
    orc.posterior_stats_split: streams split into a leading half A and a trailing half B (k = a K_B + b), the
    residuals formed directly block by block, in two passes (minimum and runner-up, then the sums for every
    varn).  Keep T_d small: several seconds per symbol."""
    T_d = Yd.shape[0]
    M = len(cons)
    nA = n_tx // 2
    XA, XB = orc.hypothesis_table(cons, nA), orc.hypothesis_table(cons, n_tx - nA)
    KA, KB = len(XA), len(XB)
    H = orc.effective_channels(_ld(PsiD), _ld(theta), n_tx)
    Yp = _ld(Yd) if Xoff is None else _ld(Yd) - np.einsum("trj,tj->tr", H, _ld(Xoff))
    rho = np.asarray(residual_error(Yd, PsiD, theta, n_tx, cons, Xoff), dtype=np.longdouble)
    varns = list(np.atleast_1d(varn))
    outs = [_Sym(T_d, n_tx) for _ in varns]
    XAc, XBc, XBl = _ld(XA).conj(), _ld(XB).conj(), _ld(XB)
    for t in range(T_d):
        u = Yp[t][None, :] - _ld(XA) @ H[t][:, :nA].T               # (KA, n_rx)
        v = _ld(XB) @ H[t][:, nA:].T                                 # (KB, n_rx)
        ur, ui, vr, vi = u.real, u.imag, v.real, v.imag

        def block(a0):
            dr = ur[a0:a0 + rows, None, :] - vr[None, :, :]
            di = ui[a0:a0 + rows, None, :] - vi[None, :, :]
            return np.sum(dr * dr + di * di, axis=2)

        best = [np.inf, -1, np.inf, -1]     # d*, k*, runner-up distance, runner-up index
        for a0 in range(0, KA, rows):
            d = block(a0).ravel()
            i1 = int(np.argmin(d))
            v1 = d[i1]
            d[i1] = np.inf
            i2 = int(np.argmin(d))
            for val, kk in ((v1, i1), (d[i2], i2)):
                k = a0 * KB + kk
                if val < best[0] or (val == best[0] and k < best[1]):
                    best[2:] = best[:2]
                    best[:2] = [val, k]
                elif val < best[2] or (val == best[2] and k < best[3]):
                    best[2:] = [val, k]
        ds, k, dsec, k2 = best
        s2 = [np.longdouble(vn) ** 2 for vn in varns]
        Z = [np.longdouble(0) for _ in varns]
        se = [np.longdouble(0) for _ in varns]
        n_win = [0 for _ in varns]
        bA = [np.zeros(KA, dtype=np.longdouble) for _ in varns]
        bB = [np.zeros(KB, dtype=np.longdouble) for _ in varns]
        cross = [np.zeros((nA, n_tx - nA), dtype=LD) for _ in varns]
        for a0 in range(0, KA, rows):
            d = block(a0)
            eps = _eps(d, rho[t])
            for i in range(len(varns)):
                w = np.exp(-(d - ds) / s2[i])
                Z[i] += w.sum()
                bA[i][a0:a0 + rows] = w.sum(axis=1)
                bB[i] += w.sum(axis=0)
                cross[i] += XAc[a0:a0 + rows].T @ (w.astype(LD) @ XBl)
                se[i] += np.sum(w * eps)
                n_win[i] += int(np.count_nonzero(d <= ds + THR * s2[i]))
        eps_s, eps_2 = _eps(ds, rho[t]), _eps(dsec, rho[t])
        for i, out in enumerate(outs):
            bs = 1 / Z[i]                    # the weight of k* is exactly 1
            ba, bb, cr, sei = bA[i] / Z[i], bB[i] / Z[i], cross[i] / Z[i], se[i] / Z[i]
            out.m[t, :nA], out.m[t, nA:] = ba @ XAc, bb @ XBc
            out.R[t, :nA, :nA] = (XAc * ba[:, None]).T @ _ld(XA)
            out.R[t, nA:, nA:] = (XBc * bb[:, None]).T @ XBl
            out.R[t, :nA, nA:] = cr
            out.R[t, nA:, :nA] = cr.conj().T
            out.lnZ[t] = np.log(Z[i])
            out.lse[t] = -ds / s2[i] + out.lnZ[t]
            out.kstar[t], out.k2[t], out.d2star[t], out.gap[t] = k, k2, ds, dsec - ds
            out.beta_max[t] = bs
            out.eps_star[t], out.eps2[t] = eps_s, eps_2
            out.n_win[t] = n_win[i]
            out.dbeta[t] = 2 * (sei + eps_s - bs * 2 * eps_s) / s2[i]
            out.lse_lin[t] = sei / s2[i]
    outs = [_finish(out, Yp, H, cons, n_tx, vn, rho, Xoff) for out, vn in zip(outs, varns)]
    return outs if np.ndim(varn) else outs[0]


def reference(Yd, PsiD, theta, cons, n_tx, varn, Xoff=None):
    """exact_stats, or exact_stats_split for trees of more than 2^18 leaves."""
    fn = exact_stats if len(cons) ** n_tx <= (1 << 18) else exact_stats_split
    return fn(Yd, PsiD, theta, cons, n_tx, varn, Xoff)


# ---------------------------------------------------------------------------
# bounds and checks
# ---------------------------------------------------------------------------

def d2_at(ref, t, k):
    """Exact squared distance of hypothesis k of symbol t."""
    x = ref.cons[orc.hypothesis_digits(np.asarray(k), ref.M, ref.n_tx)]
    r = ref.Y[t] - ref.H[t] @ _ld(x)
    return np.sum(r.real ** 2 + r.imag ** 2)


def eps_at(ref, t, k):
    return _eps(d2_at(ref, t, k), ref.rho[t])


def superimpose(m, R, o):
    """Statistics of x + o from those of x (k_superimpose_stats, oracle.em_numpy.em_superimposed):
    m~ = m + conj(o), R~ = R + m o^T + conj(o) m^H + conj(o) o^T."""
    oc = o.conj()
    return (m + oc, R + m[:, :, None] * o[:, None, :] + oc[:, :, None] * m.conj()[:, None, :]
            + oc[:, :, None] * o[:, None, :])


def taus(ref):
    """(tau_m, tau_R, tau_lse, admitted) per symbol.  With offsets o the statistics are those of x + o, formed
    from m and R with one rounding per term: tau_m gains u (x_max + |o|_max), tau_R gains 2 |o|_max tau_m for the
    propagated error of m and 8 u (x_max + |o|_max)^2 for the roundings."""
    s2 = np.longdouble(ref.varn) ** 2
    rnd = C_S * U * ref.n_win
    tm = ref.xmax * (ref.dbeta + rnd)
    tR = ref.xmax ** 2 * (ref.dbeta + rnd)
    tl = ref.lse_lin + C_S * U * (ref.d2star / s2 + np.abs(ref.lnZ) + ref.n_win)
    if ref.off is not None:
        om = np.abs(ref.off.astype(np.complex128)).max(axis=1)
        tR = tR + 2 * om * tm + 8 * U * (ref.xmax + om) ** 2
        tm = tm + U * (ref.xmax + om)
    return (tm.astype(np.float64), tR.astype(np.float64), tl.astype(np.float64),
            np.asarray(ref.dbeta < DBETA_MAX))


def kstar_bad(ref, kstar):
    """Symbols whose kstar breaks the gap rule (module docstring), as a list of (t, kstar, k*, why)."""
    bad = []
    for t, k in enumerate(np.asarray(kstar)):
        k = int(k)
        if k == ref.kstar[t]:
            continue
        if ref.gap[t] > 2 * max(ref.eps_star[t], ref.eps2[t]):
            bad.append((t, k, int(ref.kstar[t]), "gap %.3e resolvable" % float(ref.gap[t])))
        elif not 0 <= k < ref.M ** ref.n_tx or d2_at(ref, t, k) - ref.d2star[t] > eps_at(ref, t, k) + ref.eps_star[t]:
            bad.append((t, k, int(ref.kstar[t]), "not within eps of the minimum"))
    return bad


def ratios(ref, m, R, lse, hard, kstar=None):
    """Largest error / tau of m, R and lse over the admitted symbols, and the admitted count.  Hard mode: m and R
    must be exactly the rank-one statistics at the returned kstar (ratio 0, else inf); lse is not compared (the
    kernel returns the max-log term there, the reference the log-sum).  With offsets the statistics are those of
    x + o (superimpose)."""
    m, R = np.asarray(m), np.asarray(R)
    if hard:
        x = ref.cons[orc.hypothesis_digits(np.asarray(kstar, dtype=np.int64), ref.M, ref.n_tx)]
        if ref.off is not None:
            x = x + ref.off.astype(np.complex128)     # small integers: exact
        same = np.array_equal(m, x.conj()) and np.array_equal(R, x.conj()[:, :, None] * x[:, None, :])
        return (0.0 if same else np.inf), len(m)
    tm, tR, tl, adm = taus(ref)
    rm, rR = (ref.m, ref.R) if ref.off is None else superimpose(ref.m, ref.R, ref.off)
    em = np.abs((_ld(m) - rm).astype(np.complex128)).max(axis=1)
    eR = np.abs((_ld(R) - rR).astype(np.complex128)).max(axis=(1, 2))
    el = np.abs((np.asarray(lse, dtype=np.longdouble) - ref.lse).astype(np.float64))
    r = np.stack([em / tm, eR / tR, el / tl])[:, adm]
    return (float(r.max()) if r.size else 0.0), int(adm.sum())
