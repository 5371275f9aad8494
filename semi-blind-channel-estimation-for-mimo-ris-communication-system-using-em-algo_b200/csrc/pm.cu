// Partitioned ("PM") reduced-complexity E-step: statistics of one data symbol from
// a short candidate list instead of all M^n_tx hypotheses.
//
// Reference semantics (/root/reference/Proposed method/PM.py:58-104, PM_beta.py:55-95):
//   channel  = h_bu + reshape(prod @ PsiTilde_td[:N,t])        effective n_rx x n_tx channel; the
//              slice is taken AFTER the ones row was inserted, i.e. phases [1,psi_0..psi_{N-2}]
//              are paired with RIS elements 0..N-1 (quirk Q4, reproduced under SBCE_FLAG_QUIRKS)
//   ordering : n_tx rounds of k = argmax diag(pinv(A^H A)), record, delete column k  (PM.py:65-70)
//   p+1 weakest-detected streams (set A) are enumerated exhaustively (M^(p+1) candidates); for each,
//   the remaining streams (set B) are zero-forced, z = inv(B^H B) B^H (y - A x_A), and sliced to the
//   nearest constellation vector (PM.py:94-99)
//   candidate vector X = [x_A, x_B] stays in ORDERED position (quirk Q5, PM.py:102)
//   PM.py     : every candidate has weight 1 (not normalised)                    (PM.py:103-104)
//   PM_beta.py: posterior over the candidates, exp(-||y - Z(X) theta||^2/varn^2) (PM_beta.py:87-95)
//
// One warp per data symbol: lanes cooperate on the two RIS contractions (quirky and exact
// effective channel), every lane repeats the tiny n_tx x n_tx algebra (uniform, no divergence),
// candidates are strided across lanes and the statistics are merged with warp shuffles.
#include <math.h>

#include "common.cuh"

namespace sbce {

constexpr int PM_MAXR = 8;   // receive antennas
// PM_MAXT (template parameter of everything below): 4 for n_tx <= 4, 8 for the wide arrays, so that the
// per-lane scratch of the common small configurations stays small

// Cholesky of the k x k Hermitian matrix A (row-major, stride PM_MAXT) in place (lower); returns false if not PD
template <int PM_MAXT>
__device__ bool small_chol(cplx (*A)[PM_MAXT], int k) {
    bool ok = true;
    for (int c = 0; c < k; ++c) {
        double piv = A[c][c].x;
        for (int q = 0; q < c; ++q) piv -= cnorm2(A[c][q]);
        if (!(piv > 0.0)) { ok = false; piv = 1.0; }
        const double dg = sqrt(piv);
        A[c][c] = mk(dg, 0.0);
        for (int r = c + 1; r < k; ++r) {
            cplx v = A[r][c];
            for (int q = 0; q < c; ++q) cfmsc(v, A[r][q], A[c][q]);
            A[r][c] = cscale(v, 1.0 / dg);
        }
    }
    return ok;
}

// diag of inv(A) given its Cholesky factor Lc (lower): W = Lc^-1, diag_i = sum_{q>=i} |W[q][i]|^2
template <int PM_MAXT>
__device__ void inv_diag_from_chol(cplx (*Lc)[PM_MAXT], int k, double* dg) {
    cplx W[PM_MAXT][PM_MAXT];
    for (int c = 0; c < k; ++c) {
        for (int i = 0; i < k; ++i) {
            if (i < c) W[i][c] = mk(0.0, 0.0);
            else if (i == c) W[i][c] = mk(1.0 / Lc[i][i].x, 0.0);
            else {
                cplx acc = mk(0.0, 0.0);
                for (int q = c; q < i; ++q) cfma(acc, Lc[i][q], W[q][c]);
                W[i][c] = cscale(acc, -1.0 / Lc[i][i].x);
            }
        }
    }
    for (int i = 0; i < k; ++i) {
        double s = 0.0;
        for (int q = i; q < k; ++q) s += cnorm2(W[q][i]);
        dg[i] = s;
    }
}

__device__ __forceinline__ cplx cons_val(int m, int sqM, int hb) {
    return mk((double)(2 * (m & (sqM - 1)) - sqM + 1), (double)(2 * (m >> hb) - sqM + 1));
}

// nearest constellation index to z: separable per axis, first index on ties
__device__ int slice_qam(cplx z, int sqM, int hb) {
    int bi = 0, bq = 0;
    double di = 1e300, dq = 1e300;
    for (int a = 0; a < sqM; ++a) {
        const double lv = (double)(2 * a - sqM + 1);
        const double ei = (z.x - lv) * (z.x - lv), eq = (z.y - lv) * (z.y - lv);
        if (ei < di) { di = ei; bi = a; }
        if (eq < dq) { dq = eq; bq = a; }
    }
    return (bq << hb) | bi;
}

// x = pinv(H) y for an n_rx x n_tx channel of full column rank (n_rx >= n_tx) through a Householder QR of H:
// R x = (Q^H y)[:n_tx].  Normal equations would square cond(H) and lose the last pivot near cond 1e8.
// A and w are overwritten (the factors and Q^H y).
template <int PM_MAXT>
__device__ void zf_solve_qr(cplx (*A)[PM_MAXT], cplx* w, int n_rx, int n_tx, cplx* est) {
    for (int c = 0; c < n_tx; ++c) {
        // reflector v = x - alpha e_0 with alpha = -e^{i arg x_0} ||x||, x = A[c:, c]; P = I - v v^H / (v^H x)
        double nx = 0.0;
        for (int r = c; r < n_rx; ++r) nx += cnorm2(A[r][c]);
        nx = sqrt(nx);
        const double a0 = sqrt(cnorm2(A[c][c]));
        const cplx ph = a0 > 0.0 ? cscale(A[c][c], 1.0 / a0) : mk(1.0, 0.0);
        const cplx alpha = cscale(ph, -nx);
        const double vx = nx * (nx + a0);     // v^H x, real and >= 0
        if (vx > 0.0) {
            A[c][c] = csub(A[c][c], alpha);   // column c now holds v
            for (int j = c + 1; j < n_tx; ++j) {
                cplx s = mk(0, 0);
                for (int r = c; r < n_rx; ++r) cfmac(s, A[r][j], A[r][c]);  // v^H A[c:, j]
                s = cscale(s, 1.0 / vx);
                for (int r = c; r < n_rx; ++r) { const cplx u = cmul(A[r][c], s); A[r][j] = csub(A[r][j], u); }
            }
            cplx s = mk(0, 0);
            for (int r = c; r < n_rx; ++r) cfmac(s, w[r], A[r][c]);          // v^H w[c:]
            s = cscale(s, 1.0 / vx);
            for (int r = c; r < n_rx; ++r) { const cplx u = cmul(A[r][c], s); w[r] = csub(w[r], u); }
        }
        A[c][c] = alpha;
    }
    for (int a = n_tx - 1; a >= 0; --a) {
        cplx v = w[a];
        for (int q = a + 1; q < n_tx; ++q) { cplx nv = cmul(A[a][q], est[q]); v = csub(v, nv); }
        // a zero column (theta = 0 gives H = 0) contributes 0, as pinv(0) = 0 does
        const double dn = cnorm2(A[a][a]);
        est[a] = dn > 0.0 ? cscale(cmulc(v, A[a][a]), 1.0 / dn) : mk(0, 0);
    }
}

// Body of k_pm_stats (DET = false: PM, PM-beta) and k_det_stats (DET = true: ZF, MMSE).  Two kernels, so that the
// detector solve does not change the register allocation of the candidate loop.  Both are bounded to 7 CTAs of 128
// threads per SM (at most 72 registers): left to itself ptxas settles on 64 registers and spills.
template <int PM_MAXT, bool DET>
__device__ __forceinline__ void pm_stats_body(const Dims& d, const cplx* __restrict__ Yd, const cplx* __restrict__ PsiD,
                                              const cplx* __restrict__ theta, const double* __restrict__ varn,
                                              const int32_t* __restrict__ active, cplx* __restrict__ stat_m,
                                              cplx* __restrict__ stat_R, int32_t* __restrict__ kstar) {
    const int b = blockIdx.y;
    if (active != nullptr && active[b] == 0) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t = blockIdx.x * (blockDim.x >> 5) + warp;
    if (t >= d.T_d) return;
    const int n_tx = d.n_tx, n_rx = d.n_rx, N1 = d.N1, N = d.N;
    const int sqM = d.sqM, hb = d.bitsM / 2, M = d.M;
    const bool quirks = (d.flags & SBCE_FLAG_QUIRKS) != 0;
    const bool weighted = d.mode == SBCE_MODE_PM_BETA;
    const cplx* psi = PsiD + ((size_t)(d.psi_shared ? 0 : b) * d.T_d + t) * N1;
    const cplx* th = theta + (size_t)b * d.L * n_rx;

    // exact effective channel He[r][j] and the reference's (quirky) channel Hq[r][j]
    cplx He[PM_MAXR][PM_MAXT], Hq[PM_MAXR][PM_MAXT];
    for (int r = 0; r < n_rx; ++r)
        for (int j = 0; j < n_tx; ++j) { He[r][j] = mk(0, 0); Hq[r][j] = mk(0, 0); }
    for (int n = lane; n < N1; n += 32) {
        const cplx p = psi[n];
        for (int j = 0; j < n_tx; ++j)
            for (int r = 0; r < n_rx; ++r) cfma(He[r][j], p, th[(size_t)(n * n_tx + j) * n_rx + r]);
        if (n < N) {  // phase index n pairs with RIS element n, i.e. theta block n+1 (PM.py:63)
            for (int j = 0; j < n_tx; ++j)
                for (int r = 0; r < n_rx; ++r) cfma(Hq[r][j], p, th[(size_t)((n + 1) * n_tx + j) * n_rx + r]);
        }
    }
    for (int r = 0; r < n_rx; ++r)
        for (int j = 0; j < n_tx; ++j) {
            He[r][j] = mk(warp_sum(He[r][j].x), warp_sum(He[r][j].y));
            Hq[r][j] = mk(warp_sum(Hq[r][j].x), warp_sum(Hq[r][j].y));
            Hq[r][j] = cadd(Hq[r][j], th[(size_t)j * n_rx + r]);  // + h_bu
        }
    cplx (*Hc)[PM_MAXT] = quirks ? Hq : He;  // channel used for ordering / zero forcing

    cplx y[PM_MAXR];
    for (int r = 0; r < n_rx; ++r) y[r] = Yd[((size_t)b * d.T_d + t) * n_rx + r];

    if constexpr (DET) {
        // ---- detector-driven EM (em_zf / em_mmse, PMvsMLvsZFvsMMSE.py:54-133): x = pinv(H) y (ZF) or
        // (H^H H + varn^2 I)^-1 H^H y (MMSE), sliced to one hypothesis, rank-one statistics.  Every lane computes
        // the same tiny solve.
        cplx est[PM_MAXT];
        if (d.mode == SBCE_MODE_ZF) {
            zf_solve_qr(Hc, y, n_rx, n_tx, est);   // last use of Hc and y: factored in place
        } else {
            cplx Gm[PM_MAXT][PM_MAXT];
            const double reg = varn[b] * varn[b];
            for (int a = 0; a < n_tx; ++a)
                for (int c = 0; c <= a; ++c) {
                    cplx sacc = mk(0, 0);
                    for (int r = 0; r < n_rx; ++r) cfmac(sacc, Hc[r][c], Hc[r][a]);
                    if (a == c) sacc.x += reg;
                    Gm[a][c] = sacc;
                }
            small_chol(Gm, n_tx);
            for (int a = 0; a < n_tx; ++a) {
                cplx sacc = mk(0, 0);
                for (int r = 0; r < n_rx; ++r) cfmac(sacc, y[r], Hc[r][a]);
                est[a] = sacc;
            }
            for (int a = 0; a < n_tx; ++a) {
                cplx v = est[a];
                for (int q = 0; q < a; ++q) { cplx nv = cmul(Gm[a][q], est[q]); v = csub(v, nv); }
                est[a] = cscale(v, 1.0 / Gm[a][a].x);
            }
            for (int a = n_tx - 1; a >= 0; --a) {
                cplx v = est[a];
                for (int q = a + 1; q < n_tx; ++q) cfmsc(v, est[q], Gm[q][a]);
                est[a] = cscale(v, 1.0 / Gm[a][a].x);
            }
        }
        int k = 0;
        if (quirks) {
            // nearest_symbol_ecul as called (PMvsMLvsZFvsMMSE.py:49-52,68): argmin over the flattened
            // (K, n_tx, n_tx) array of |est[i] - table[k][j]| used as a ROW index of the table.  With (i*, c*)
            // the closest (stream, constellation point) pair, first c then first i on ties, that flat index is
            // idx(c*) n_tx^2 + i* n_tx + (n_tx-1 if idx(c*) else 0).
            double best = 1e300;
            int bi = 0, bc = 0;
            for (int c = 0; c < M; ++c) {
                const cplx cv = cons_val(c, sqM, hb);
                for (int i = 0; i < n_tx; ++i) {
                    const double dd = cnorm2(csub(est[i], cv));
                    if (dd < best) { best = dd; bc = c; bi = i; }
                }
            }
            k = bc * n_tx * n_tx + bi * n_tx + (bc ? n_tx - 1 : 0);
            int K = 1;
            for (int a = 0; a < n_tx; ++a) K *= M;
            if (k >= K) k = K - 1;  // the reference would raise IndexError here (only when n_tx^2 > M^(n_tx-1))
        } else {
            for (int a = 0; a < n_tx; ++a) k = k * M + slice_qam(est[a], sqM, hb);
        }
        if (lane == 0) {
            const size_t sidx = (size_t)b * d.T_d + t;
            cplx X[PM_MAXT];
            for (int a = n_tx - 1, kk = k; a >= 0; --a) { X[a] = cons_val(kk % M, sqM, hb); kk /= M; }
            for (int i = 0; i < n_tx; ++i) {
                stat_m[sidx * n_tx + i] = cconj(X[i]);
                for (int j = 0; j < n_tx; ++j) stat_R[(sidx * n_tx + i) * n_tx + j] = cmulc(X[j], X[i]);
            }
            if (kstar) kstar[sidx] = k;
        }
        return;
    }

    // ---- ordering (PM.py:65-70)
    int order[PM_MAXT], remaining[PM_MAXT];
    for (int j = 0; j < n_tx; ++j) remaining[j] = j;
    for (int round = 0; round < n_tx; ++round) {
        const int k = n_tx - round;
        cplx A[PM_MAXT][PM_MAXT];
        for (int a = 0; a < k; ++a)
            for (int c = 0; c <= a; ++c) {
                cplx s = mk(0, 0);
                for (int r = 0; r < n_rx; ++r) cfmac(s, Hc[r][remaining[c]], Hc[r][remaining[a]]);  // conj(col a) . col c
                A[a][c] = s;
            }
        small_chol(A, k);
        double dg[PM_MAXT];
        inv_diag_from_chol(A, k, dg);
        int best = 0;
        for (int a = 1; a < k; ++a)
            if (dg[a] > dg[best]) best = a;
        order[round] = remaining[best];
        for (int a = best; a + 1 < k; ++a) remaining[a] = remaining[a + 1];
    }
    const int p1 = d.p1, nB = n_tx - p1;

    // ---- zero forcing of set B: PB = inv(B^H B) B^H (nB x n_rx), v0 = PB y, VA = PB A (nB x p1)
    cplx v0[PM_MAXT], VA[PM_MAXT][PM_MAXT];
    if (nB > 0) {
        cplx Gb[PM_MAXT][PM_MAXT];
        for (int a = 0; a < nB; ++a)
            for (int c = 0; c <= a; ++c) {
                cplx s = mk(0, 0);
                for (int r = 0; r < n_rx; ++r) cfmac(s, Hc[r][order[p1 + c]], Hc[r][order[p1 + a]]);
                Gb[a][c] = s;
            }
        small_chol(Gb, nB);
        // columns to solve for: y and the p1 columns of A
        for (int col = 0; col <= p1; ++col) {
            cplx rhs[PM_MAXT];
            for (int a = 0; a < nB; ++a) {
                cplx s = mk(0, 0);
                for (int r = 0; r < n_rx; ++r) {
                    const cplx v = (col == 0) ? y[r] : Hc[r][order[col - 1]];
                    cfmac(s, v, Hc[r][order[p1 + a]]);  // conj(B col a) * v
                }
                rhs[a] = s;
            }
            // forward L w = rhs, backward L^H x = w
            for (int a = 0; a < nB; ++a) {
                cplx v = rhs[a];
                for (int q = 0; q < a; ++q) { cplx nv = cmul(Gb[a][q], rhs[q]); v = csub(v, nv); }
                rhs[a] = cscale(v, 1.0 / Gb[a][a].x);
            }
            for (int a = nB - 1; a >= 0; --a) {
                cplx v = rhs[a];
                for (int q = a + 1; q < nB; ++q) cfmsc(v, rhs[q], Gb[q][a]);
                rhs[a] = cscale(v, 1.0 / Gb[a][a].x);
            }
            for (int a = 0; a < nB; ++a) {
                if (col == 0) v0[a] = rhs[a]; else VA[a][col - 1] = rhs[a];
            }
        }
    }

    // ---- candidates
    int ncand = 1;
    for (int a = 0; a < p1; ++a) ncand *= M;
    const double vn = varn[b];
    const double inv_s2 = 1.0 / (vn * vn);

    auto build = [&](int c, cplx* X) {
        // x_A from the digits of c (first A stream most significant, itertools.product order)
        cplx xa[PM_MAXT];
        for (int a = p1 - 1, cc = c; a >= 0; --a) { xa[a] = cons_val(cc % M, sqM, hb); cc /= M; }
        cplx Xo[PM_MAXT];
        for (int a = 0; a < p1; ++a) Xo[a] = xa[a];
        for (int s = 0; s < nB; ++s) {
            cplx z = v0[s];
            for (int a = 0; a < p1; ++a) { cplx nv = cmul(VA[s][a], xa[a]); z = csub(z, nv); }
            Xo[p1 + s] = cons_val(slice_qam(z, sqM, hb), sqM, hb);
        }
        if (quirks) {
            for (int a = 0; a < n_tx; ++a) X[a] = Xo[a];
        } else {
            for (int a = 0; a < n_tx; ++a) X[order[a]] = Xo[a];
        }
    };
    auto dist2 = [&](const cplx* X) {
        double s = 0.0;
        for (int r = 0; r < n_rx; ++r) {
            cplx e = y[r];
            for (int j = 0; j < n_tx; ++j) { cplx nv = cmul(He[r][j], X[j]); e = csub(e, nv); }
            s += cnorm2(e);
        }
        return s;
    };

    double dmin = 1e300;
    if (weighted) {
        for (int c = lane; c < ncand; c += 32) {
            cplx X[PM_MAXT];
            build(c, X);
            dmin = fmin(dmin, dist2(X));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dmin = fmin(dmin, shfl_xor_d(dmin, o));
    }
    double S = 0.0;
    cplx mm[PM_MAXT], RR[PM_MAXT][PM_MAXT];
    for (int i = 0; i < n_tx; ++i) {
        mm[i] = mk(0, 0);
        for (int j = 0; j < n_tx; ++j) RR[i][j] = mk(0, 0);
    }
    for (int c = lane; c < ncand; c += 32) {
        cplx X[PM_MAXT];
        build(c, X);
        const double w = weighted ? exp((dmin - dist2(X)) * inv_s2) : 1.0;
        S += w;
        for (int i = 0; i < n_tx; ++i) {
            mm[i].x = fma(w, X[i].x, mm[i].x);
            mm[i].y = fma(-w, X[i].y, mm[i].y);
            for (int j = 0; j < n_tx; ++j) {
                const cplx cx = cmulc(X[j], X[i]);  // conj(X_i) X_j
                RR[i][j].x = fma(w, cx.x, RR[i][j].x);
                RR[i][j].y = fma(w, cx.y, RR[i][j].y);
            }
        }
    }
    S = warp_sum(S);
    const double sc = weighted ? 1.0 / S : 1.0;
    const size_t sidx = (size_t)b * d.T_d + t;
    for (int i = 0; i < n_tx; ++i) {
        const double a = warp_sum(mm[i].x), c = warp_sum(mm[i].y);
        if (lane == 0) stat_m[sidx * n_tx + i] = mk(a * sc, c * sc);
        for (int j = 0; j < n_tx; ++j) {
            const double e = warp_sum(RR[i][j].x), f = warp_sum(RR[i][j].y);
            if (lane == 0) stat_R[(sidx * n_tx + i) * n_tx + j] = mk(e * sc, f * sc);
        }
    }
}

template <int PM_MAXT>
__global__ void __launch_bounds__(128, 7) k_pm_stats(Dims d, const cplx* __restrict__ Yd, const cplx* __restrict__ PsiD,
                                                  const cplx* __restrict__ theta, const double* __restrict__ varn,
                                                  const int32_t* __restrict__ active, cplx* __restrict__ stat_m,
                                                  cplx* __restrict__ stat_R) {
    pm_stats_body<PM_MAXT, false>(d, Yd, PsiD, theta, varn, active, stat_m, stat_R, nullptr);
}

template <int PM_MAXT>
__global__ void __launch_bounds__(128, 7) k_det_stats(Dims d, const cplx* __restrict__ Yd, const cplx* __restrict__ PsiD,
                                                   const cplx* __restrict__ theta, const double* __restrict__ varn,
                                                   const int32_t* __restrict__ active, cplx* __restrict__ stat_m,
                                                   cplx* __restrict__ stat_R, int32_t* __restrict__ kstar) {
    pm_stats_body<PM_MAXT, true>(d, Yd, PsiD, theta, varn, active, stat_m, stat_R, kstar);
}

cudaError_t launch_pm_stats(const Dims& d, int nb, const double* Yd, const double* PsiD, const double* theta,
                            const double* varn, const int32_t* active, double* stat_m, double* stat_R,
                            int32_t* kstar, cudaStream_t s) {
    if (d.n_tx > 8 || d.n_rx > PM_MAXR) return cudaErrorInvalidValue;
    dim3 grid((d.T_d + 3) / 4, nb);
    const cplx *y = (const cplx*)Yd, *psi = (const cplx*)PsiD, *th = (const cplx*)theta;
    cplx *m = (cplx*)stat_m, *R = (cplx*)stat_R;
    if (d.mode == SBCE_MODE_ZF || d.mode == SBCE_MODE_MMSE) {
        if (d.n_tx <= 4) k_det_stats<4><<<grid, 128, 0, s>>>(d, y, psi, th, varn, active, m, R, kstar);
        else k_det_stats<8><<<grid, 128, 0, s>>>(d, y, psi, th, varn, active, m, R, kstar);
    } else {
        if (d.n_tx <= 4) k_pm_stats<4><<<grid, 128, 0, s>>>(d, y, psi, th, varn, active, m, R);
        else k_pm_stats<8><<<grid, 128, 0, s>>>(d, y, psi, th, varn, active, m, R);
    }
    count_launch();
    return cudaGetLastError();
}

}  // namespace sbce
