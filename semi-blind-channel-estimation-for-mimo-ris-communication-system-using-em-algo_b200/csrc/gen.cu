// On-device input generation and least-squares start (SURVEY.md section 8f-1): the step immediately
// before the hot path, moved to the GPU so that a Monte-Carlo sweep needs no host generation and no
// host->device copy of ~300 KB per trial.
//
// Reference semantics (all in /root/reference/Proposed method/PM.py):
//   channelMatrix  :11-17   H_BU (n_rx x n_tx), H_BS (N x n_tx), H_SU (n_rx x N) i.i.d. CN(0, varh);
//                           h = [vec_F(H_BU); vec_F(khatri_rao(H_BS^T, H_SU))]  ->  Theta[n'][j][r]
//   symbols/pilotSymbols :19-40   i.i.d. uniform constellation indices, un-normalised QAM grid (QAM.py:310-322)
//   irsMatrix      :119-130 pilot phases exp(-j 2pi t n / N) for n < N written into rows 0..N-1 of an
//                           (N+1) x T_p zero array (row N stays 0), data phases exp(j U(0, 2pi)); the driver
//                           inserts the direct-link ones row (:179).  Top-level variants:
//                           Proposed_method_NMSEvsTp.py:72-83,129 (ones row + exp(-j 2pi t n / T_p)),
//                           Proposed_method_NMSEvsTd.py:92-94 (deterministic DFT data phases)
//   receivedSignals:132-148 Y_t = Z_t h + n_t, n_t ~ CN(0, varn); h_initial = pinv(vstack Z_p) vstack Y_p
//
// B200 design: counter-based Philox4x32-10 (hand-written, no library RNG) keyed by the sweep seed, with
// the counter = (element index, array id, global trial index): every element of every trial is a pure
// function of (seed, trial, array, element), so a batch can be generated in any sharding across GPUs and
// reproduced bit-exactly by the numpy restatement of the generator in oracle/philox.py.  The Kronecker
// design matrix Z is never formed: Y is contracted straight from (psi, x, Theta), and the LS start is
// the min-norm solution through the T_p x T_p Hadamard-product Gram  K = (Psi Psi^H) o (X X^H)  when
// T_p < L, or through the pilot normal equations (the M-step kernels) when T_p >= L.
#include <math.h>

#include "common.cuh"

namespace sbce {

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11), counter (c0..c3), key (k0,k1)
// ---------------------------------------------------------------------------
struct U4 { uint32_t x, y, z, w; };

__device__ __forceinline__ U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = U4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}

enum GenStream { GS_HBU = 0, GS_HBS = 1, GS_HSU = 2, GS_XD = 3, GS_XP = 4, GS_PHI = 5, GS_NP = 6, GS_ND = 7 };

struct GenKey { uint32_t k0, k1; unsigned long long trial0; };

__device__ __forceinline__ U4 draw(const GenKey& k, int stream, unsigned long long trial, uint32_t elem) {
    const unsigned long long tr = k.trial0 + trial;
    return philox4x32_10(U4{elem, (uint32_t)stream, (uint32_t)tr, (uint32_t)(tr >> 32)}, k.k0, k.k1);
}
// 53-bit uniform in (0,1) from two words
__device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
    const unsigned long long v = ((unsigned long long)a << 21) ^ (unsigned long long)(b >> 11);
    return ((double)v + 0.5) * (1.0 / 9007199254740992.0);
}
// one CN(0, var) sample (Box-Muller on the two uniforms of one Philox block)
__device__ __forceinline__ cplx cn_sample(const U4& r, double var) {
    const double u1 = u53(r.x, r.y), u2 = u53(r.z, r.w);
    const double rad = sqrt(-var * log(u1));
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    return mk(rad * c, rad * s);
}

// ---------------------------------------------------------------------------
// channel: Theta[b][n'][j][r]
// ---------------------------------------------------------------------------
__global__ void k_gen_channel(Dims d, GenKey key, double varh, int nodirect, cplx* __restrict__ h) {
    const int b = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;   // (n', j, r)
    if (e >= d.L * d.n_rx) return;
    const int r = e % d.n_rx, l = e / d.n_rx, j = l % d.n_tx, np = l / d.n_tx;
    cplx v;
    if (np == 0 && !nodirect) {
        v = cn_sample(draw(key, GS_HBU, b, (uint32_t)(r * d.n_tx + j)), varh);             // H_BU[r][j]
    } else {
        const int n = nodirect ? np : np - 1;
        const int nris = nodirect ? d.N1 : d.N;
        const cplx bs = cn_sample(draw(key, GS_HBS, b, (uint32_t)(n * d.n_tx + j)), varh);  // H_BS[n][j]
        const cplx su = cn_sample(draw(key, GS_HSU, b, (uint32_t)(r * nris + n)), varh);   // H_SU[r][n]
        v = cmul(bs, su);
    }
    h[(size_t)b * d.L * d.n_rx + e] = v;
}

// ---------------------------------------------------------------------------
// symbols: X[b][t][j] (complex constellation points), pilots and data
// ---------------------------------------------------------------------------
__global__ void k_gen_symbols(Dims d, GenKey key, cplx* __restrict__ Xp, cplx* __restrict__ Xd) {
    const int b = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int np = d.T_p * d.n_tx, nd = d.T_d * d.n_tx;
    if (e >= np + nd) return;
    const bool pil = e < np;
    const int idx = pil ? e : e - np;
    const uint32_t w = draw(key, pil ? GS_XP : GS_XD, b, (uint32_t)idx).x;
    const int m = (int)(w & (uint32_t)(d.M - 1));          // M is a power of two: unbiased
    const int hb = d.bitsM / 2;
    const cplx v = mk((double)(2 * (m & (d.sqM - 1)) - d.sqM + 1), (double)(2 * (m >> hb) - d.sqM + 1));
    if (pil) { if (Xp) Xp[(size_t)b * np + idx] = v; }
    else if (Xd) Xd[(size_t)b * nd + idx] = v;
}

// ---------------------------------------------------------------------------
// RIS phases in the estimator layout Psi[b|1][t][n'] (ones row already inserted)
// ---------------------------------------------------------------------------
__device__ __forceinline__ cplx dft_phase(long long t, long long n, long long denom) {
    // exp(-j 2 pi t n / denom) with the argument reduced exactly in integers
    const long long q = (t * n) % denom;
    double s, c;
    sincospi(-2.0 * (double)q / (double)denom, &s, &c);
    return mk(c, s);
}

__global__ void k_gen_phases(Dims d, GenKey key, int pilot_design, int data_phases, int nodirect, cplx* __restrict__ PsiP,
                             cplx* __restrict__ PsiD) {
    const int b = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int np = d.T_p * d.N1, nd = d.T_d * d.N1;
    if (e >= np + nd) return;
    if (e < np) {
        if (!PsiP || (d.psiP_shared && b > 0)) return;
        const int t = e / d.N1, n1 = e % d.N1;
        cplx v;
        if (nodirect) v = dft_phase(t, n1, pilot_design == SBCE_PILOTS_PM ? d.N1 : d.T_p);   // all rows are elements
        else if (pilot_design == SBCE_PILOTS_PM) v = (n1 < d.N) ? dft_phase(t, n1, d.N) : mk(0.0, 0.0);
        else v = (n1 == 0) ? mk(1.0, 0.0) : dft_phase(t, n1 - 1, d.T_p);
        PsiP[(size_t)b * np + e] = v;
    } else {
        const int f = e - np;
        const int t = f / d.N1, n1 = f % d.N1;
        if (!PsiD || (d.psi_shared && b > 0)) return;
        cplx v;
        if (data_phases == SBCE_PHASES_DFT) v = dft_phase(t, n1, d.T_d);
        else if (n1 == 0 && !nodirect) v = mk(1.0, 0.0);
        else {
            const U4 r = draw(key, GS_PHI, b, nodirect ? (uint32_t)(t * d.N1 + n1) : (uint32_t)(t * d.N + (n1 - 1)));
            double s, c;
            sincospi(2.0 * u53(r.x, r.y), &s, &c);
            v = mk(c, s);
        }
        PsiD[(size_t)b * nd + f] = v;
    }
}

// ---------------------------------------------------------------------------
// received blocks: Y[b][t][r] = sum_{n',j} psi[t,n'] x_t[j] Theta[n'*n_tx+j][r] + CN(0, varn[b])
// one warp per (b, t): lanes split the RIS index, shuffle-reduce, lanes 0..n_rx-1 add the noise
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_gen_received(Dims d, GenKey key, int T, int noise_stream,
                                                      const cplx* __restrict__ Psi, const cplx* __restrict__ X,
                                                      const cplx* __restrict__ h, const double* __restrict__ varn,
                                                      cplx* __restrict__ Y) {
    const int b = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t = blockIdx.x * (blockDim.x >> 5) + warp;
    if (t >= T) return;
    const int n_tx = d.n_tx, n_rx = d.n_rx;
    const cplx* psi = Psi + ((size_t)(d.psi_shared ? 0 : b) * T + t) * d.N1;
    const cplx* x = X + ((size_t)b * T + t) * n_tx;
    const cplx* th = h + (size_t)b * d.L * n_rx;
    cplx acc[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) acc[r] = mk(0.0, 0.0);
    for (int n = lane; n < d.N1; n += 32) {
        const cplx p = psi[n];
        for (int j = 0; j < n_tx; ++j) {
            const cplx w = cmul(p, x[j]);
            const cplx* row = th + (size_t)(n * n_tx + j) * n_rx;
#pragma unroll
            for (int r = 0; r < 8; ++r)
                if (r < n_rx) cfma(acc[r], w, row[r]);
        }
    }
#pragma unroll
    for (int r = 0; r < 8; ++r)
        if (r < n_rx) acc[r] = mk(warp_sum(acc[r].x), warp_sum(acc[r].y));
    if (lane < n_rx) {
        cplx v = mk(0.0, 0.0);
#pragma unroll
        for (int r = 0; r < 8; ++r)
            if (r == lane) v = acc[r];
        const cplx nz = cn_sample(draw(key, noise_stream, b, (uint32_t)(t * n_rx + lane)), varn[b]);
        Y[((size_t)b * T + t) * n_rx + lane] = cadd(v, nz);
    }
}

// ---------------------------------------------------------------------------
// LS start, dual (min-norm) form for T_p < L:  K = W W^H = (Psi Psi^H) o (X X^H),  K A = Y_p,
// Theta0 = W^H A.  K is written as the lower trapezoid [K ; Y_p^H] the Cholesky kernel expects.
// ---------------------------------------------------------------------------
__global__ void k_ls_dual_build(Dims d, Dims dd, const cplx* __restrict__ PsiP, const cplx* __restrict__ Xp,
                                const cplx* __restrict__ Yp, cplx* __restrict__ Kall) {
    const int b = blockIdx.y;
    const int T = d.T_p, Lp = dd.Lp, Ltot = dd.Ltot;
    const cplx* psi = PsiP + (size_t)(d.psi_shared ? 0 : b) * T * d.N1;
    const cplx* x = Xp + (size_t)b * T * d.n_tx;
    const cplx* y = Yp + (size_t)b * T * d.n_rx;
    cplx* K = Kall + (size_t)b * Ltot * Lp;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < Ltot * Lp; e += gridDim.x * blockDim.x) {
        const int row = e / Lp, col = e % Lp;
        cplx v = mk(0.0, 0.0);
        if (row < T) {
            if (col <= row) {
                cplx a = mk(0.0, 0.0), c = mk(0.0, 0.0);
                for (int n = 0; n < d.N1; ++n) cfmac(a, psi[(size_t)row * d.N1 + n], psi[(size_t)col * d.N1 + n]);
                for (int j = 0; j < d.n_tx; ++j) cfmac(c, x[row * d.n_tx + j], x[col * d.n_tx + j]);
                v = cmul(a, c);
            }
        } else if (row < Lp) {
            v = (col == row) ? mk(1.0, 0.0) : mk(0.0, 0.0);          // identity padding
        } else {
            const int r = row - Lp;
            if (r < d.n_rx && col < T) v = cconj(y[col * d.n_rx + r]);   // B^H rows
        }
        K[e] = v;
    }
}

// Theta0[n'*n_tx+j][r] = sum_t conj(psi[t,n'] x_t[j]) A[t][r]
__global__ void k_ls_dual_expand(Dims d, const cplx* __restrict__ PsiP, const cplx* __restrict__ Xp,
                                 const cplx* __restrict__ A, cplx* __restrict__ theta0) {
    const int b = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;   // (l, r)
    if (e >= d.L * d.n_rx) return;
    const int r = e % d.n_rx, l = e / d.n_rx, j = l % d.n_tx, np = l / d.n_tx;
    const cplx* psi = PsiP + (size_t)(d.psi_shared ? 0 : b) * d.T_p * d.N1;
    const cplx* x = Xp + (size_t)b * d.T_p * d.n_tx;
    const cplx* a = A + (size_t)b * d.T_p * d.n_rx;
    cplx acc = mk(0.0, 0.0);
    for (int t = 0; t < d.T_p; ++t) {
        const cplx w = cmul(psi[(size_t)t * d.N1 + np], x[t * d.n_tx + j]);
        cfmac(acc, a[t * d.n_rx + r], w);   // a * conj(w)
    }
    theta0[(size_t)b * d.L * d.n_rx + e] = acc;
}

// ---------------------------------------------------------------------------
// LS start, primal form for T_p >= L.  The reference's own pilot designs are rank deficient BY
// CONSTRUCTION: "pm" leaves the last RIS element off (a zero column of Psi_p, PM.py:120-124) and the
// top-level scripts insert a ones row next to the n = 0 DFT row, which is also all ones
// (Proposed_method_NMSEvsTp.py:77,129) -- two identical columns.  numpy's pinv returns the min-norm
// solution there: zero for a zero column, an even split between identical columns.  That is reproduced
// exactly: identical columns are merged into one scaled by sqrt(multiplicity) (min |a|^2+|b|^2 subject to
// a+b = s  <=>  min |s'|^2 with column sqrt(2) w, a = b = s'/sqrt(2)), removed columns get a unit diagonal,
// and the solution is spread back.  Any other rank deficiency is flagged by the Cholesky (SBCE_ST_NOT_PD).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_ls_dedup(Dims d, const cplx* __restrict__ PsiP, cplx* __restrict__ PsiW,
                                                  double* __restrict__ scale, int32_t* __restrict__ rep) {
    const int b = blockIdx.x;
    const int T = d.T_p, N1 = d.N1;
    const cplx* psi = PsiP + (size_t)b * T * N1;
    cplx* pw = PsiW + (size_t)b * T * N1;
    double* sc = scale + (size_t)b * N1;
    int32_t* rp = rep + (size_t)b * N1;
    for (int n = threadIdx.x; n < N1; n += blockDim.x) {
        bool zero = true;
        for (int t = 0; t < T && zero; ++t) zero = (psi[(size_t)t * N1 + n].x == 0.0 && psi[(size_t)t * N1 + n].y == 0.0);
        int r = zero ? -1 : n;
        for (int m = 0; m < n && r == n; ++m) {
            bool same = true;
            for (int t = 0; t < T && same; ++t) {
                const cplx a = psi[(size_t)t * N1 + n], c = psi[(size_t)t * N1 + m];
                same = (a.x == c.x && a.y == c.y);
            }
            if (same) r = m;
        }
        rp[n] = r;
    }
    __syncthreads();
    for (int n = threadIdx.x; n < N1; n += blockDim.x) {
        int mult = 0;
        if (rp[n] == n)
            for (int m = n; m < N1; ++m) mult += (rp[m] == n);
        sc[n] = sqrt((double)mult);   // 0 for removed columns
    }
    __syncthreads();
    for (int e = threadIdx.x; e < T * N1; e += blockDim.x) pw[e] = cscale(psi[e], sc[e % N1]);
}

// unit diagonal on the rows of removed columns (their rows / columns of G and of B^H are exactly zero)
__global__ void k_ls_fix_diag(Dims d, const double* __restrict__ scale, cplx* __restrict__ Gall) {
    const int b = blockIdx.y;
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= d.L) return;
    const double sc = scale[(size_t)(d.psi_shared ? 0 : b) * d.N1 + l / d.n_tx];
    if (sc == 0.0) Gall[(size_t)b * d.Ltot * d.Lp + (size_t)l * d.Lp + l] = mk(1.0, 0.0);
}

__global__ void k_ls_spread(Dims d, const double* __restrict__ scale, const int32_t* __restrict__ rep,
                            const cplx* __restrict__ thw, cplx* __restrict__ theta0) {
    const int b = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;   // (l, r)
    if (e >= d.L * d.n_rx) return;
    const int r = e % d.n_rx, l = e / d.n_rx, j = l % d.n_tx, np = l / d.n_tx;
    const size_t pb = (size_t)(d.psi_shared ? 0 : b) * d.N1;
    const int rp = rep[pb + np];
    cplx v = mk(0.0, 0.0);
    if (rp >= 0) v = cscale(thw[(size_t)b * d.L * d.n_rx + (size_t)(rp * d.n_tx + j) * d.n_rx + r], 1.0 / scale[pb + rp]);
    theta0[(size_t)b * d.L * d.n_rx + e] = v;
}

// ---------------------------------------------------------------------------
// symbol-error accumulation on the device (drivers): true per-stream errors and the reference's
// as-coded count (SER/log_max_SER.py:162 broadcasts (T,n,1) - (T,1,n): all n_tx^2 cross pairs)
// acc[0] += per-stream errors, acc[1] += symbols, acc[2] += sum over trials of the as-coded SER
// ---------------------------------------------------------------------------
__global__ void k_accumulate_ser(Dims d, int nb, const int32_t* __restrict__ kstar, const cplx* __restrict__ Xd,
                                 double* __restrict__ acc) {
    const int b = blockIdx.x;
    if (b >= nb) return;
    const int hb = d.bitsM / 2;
    double err = 0.0, coded = 0.0;
    for (int t = threadIdx.x; t < d.T_d; t += blockDim.x) {
        const int k = kstar[(size_t)b * d.T_d + t];
        const cplx* x = Xd + ((size_t)b * d.T_d + t) * d.n_tx;
        for (int i = 0; i < d.n_tx; ++i) {
            const cplx xi = x[i];
            for (int j = 0; j < d.n_tx; ++j) {
                const int m = (k >> (d.bitsM * (d.n_tx - 1 - j))) & (d.M - 1);
                const double re = (double)(2 * (m & (d.sqM - 1)) - d.sqM + 1), im = (double)(2 * (m >> hb) - d.sqM + 1);
                const bool diff = (xi.x != re) || (xi.y != im);
                if (diff) coded += 1.0;
                if (diff && i == j) err += 1.0;
            }
        }
    }
    err = warp_sum(err);
    coded = warp_sum(coded);
    __shared__ double se[32], sc[32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { se[warp] = err; sc[warp] = coded; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double e2 = 0.0, c2 = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { e2 += se[w]; c2 += sc[w]; }
        atomicAdd(&acc[0], e2);
        atomicAdd(&acc[1], (double)d.T_d * d.n_tx);
        atomicAdd(&acc[2], c2 / ((double)d.T_d * d.n_tx));
    }
}

// ---------------------------------------------------------------------------
// bit-error accumulation on the device (BER curves): Gray labels of include/sbce.h, per stream gray(iI) then
// gray(iQ).  acc[0] += bit errors, acc[1] += bits compared.  Counts are integers, so the atomics' order does
// not matter.
// ---------------------------------------------------------------------------
__global__ void k_accumulate_ber(Dims d, int nb, const int32_t* __restrict__ kstar, const cplx* __restrict__ Xd,
                                 double* __restrict__ acc) {
    const int b = blockIdx.x;
    if (b >= nb) return;
    const int hb = d.bitsM / 2, top = d.sqM - 1;
    auto gray = [](int a) { return a ^ (a >> 1); };
    // PAM index of a level 2a - sqrt(M) + 1 (the true symbols are exact constellation points)
    auto level = [&](double v) { return min(max((int)lround(0.5 * (v + top)), 0), top); };
    double err = 0.0;
    for (int t = threadIdx.x; t < d.T_d; t += blockDim.x) {
        const int k = kstar[(size_t)b * d.T_d + t];
        const cplx* x = Xd + ((size_t)b * d.T_d + t) * d.n_tx;
        for (int j = 0; j < d.n_tx; ++j) {
            const int m = (k >> (d.bitsM * (d.n_tx - 1 - j))) & (d.M - 1);
            const int lab = (gray(m >> hb) << hb) | gray(m & top);   // label as an integer, Q bits low
            const int tru = (gray(level(x[j].y)) << hb) | gray(level(x[j].x));
            err += (double)__popc(lab ^ tru);
        }
    }
    err = warp_sum(err);
    __shared__ double se[32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) se[warp] = err;
    __syncthreads();
    if (threadIdx.x == 0) {
        double e2 = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) e2 += se[w];
        atomicAdd(&acc[0], e2);
        atomicAdd(&acc[1], (double)d.T_d * d.n_tx * d.bitsM);
    }
}

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
static GenKey make_key(const sbce_gen* g) {
    GenKey k;
    k.k0 = (uint32_t)(g->seed & 0xffffffffu);
    k.k1 = (uint32_t)(g->seed >> 32);
    k.trial0 = (unsigned long long)g->trial0;
    return k;
}

cudaError_t launch_generate(const Dims& d, int nb, const sbce_gen* g, const sbce_io& io, double* h_out, double* Xp_out,
                            double* Xd_out, double* PsiP_out, double* PsiD_out, double* Yp_out, double* Yd_out,
                            cudaStream_t s) {
    const GenKey key = make_key(g);
    {
        dim3 grid((d.L * d.n_rx + 255) / 256, nb);
        k_gen_channel<<<grid, 256, 0, s>>>(d, key, g->varh, g->no_direct_link ? 1 : 0, (cplx*)h_out);
        count_launch();
    }
    {
        dim3 grid(((d.T_p + d.T_d) * d.n_tx + 255) / 256, nb);
        k_gen_symbols<<<grid, 256, 0, s>>>(d, key, (cplx*)Xp_out, (cplx*)Xd_out);
        count_launch();
    }
    {
        dim3 grid(((d.T_p + d.T_d) * d.N1 + 255) / 256, (d.psi_shared && d.psiP_shared) ? 1 : nb);
        k_gen_phases<<<grid, 256, 0, s>>>(d, key, g->pilot_design, g->data_phases, g->no_direct_link ? 1 : 0, (cplx*)PsiP_out,
                                         (cplx*)PsiD_out);
        count_launch();
    }
    if (d.T_p > 0) {
        dim3 grid((d.T_p + 3) / 4, nb);
        Dims dp = d;
        dp.psi_shared = d.psiP_shared;
        k_gen_received<<<grid, 128, 0, s>>>(dp, key, d.T_p, GS_NP, (const cplx*)PsiP_out, (const cplx*)Xp_out,
                                            (const cplx*)h_out, io.varn, (cplx*)Yp_out);
        count_launch();
    }
    {
        dim3 grid((d.T_d + 3) / 4, nb);
        k_gen_received<<<grid, 128, 0, s>>>(d, key, d.T_d, GS_ND, (const cplx*)PsiD_out, (const cplx*)Xd_out,
                                            (const cplx*)h_out, io.varn, (cplx*)Yd_out);
        count_launch();
    }
    return cudaGetLastError();
}

cudaError_t launch_ls_start(const Dims& d, int nb, const sbce_io& io, double* theta0, int32_t* status, Workspace& ws,
                            cudaStream_t s) {
    cudaError_t e = cudaMemsetAsync(ws.stat, 0, (size_t)nb * 4, s);
    if (e != cudaSuccess) return e;
    if (d.T_p >= d.L) {
        // primal: the pilot normal equations, i.e. an M-step without data
        const int npsi = d.psi_shared ? 1 : nb;
        k_ls_dedup<<<npsi, 128, 0, s>>>(d, (const cplx*)io.PsiP, (cplx*)ws.psiw, ws.ls_scale, ws.ls_rep);
        count_launch();
        e = launch_pilot_stats(d, nb, io.Xp, ws.pil_m, ws.pil_R, s);
        if (e != cudaSuccess) return e;
        e = launch_normal_equations(d, nb, ws.psiw, d.T_p, io.Yp, ws.pil_m, ws.pil_R, nullptr, ws.G, nullptr, s);
        if (e != cudaSuccess) return e;
        {
            dim3 grid((d.L + 127) / 128, nb);
            k_ls_fix_diag<<<grid, 128, 0, s>>>(d, ws.ls_scale, (cplx*)ws.G);
            count_launch();
        }
        double* thw = ws.Gp;   // [nb][L][n_rx] solution of the merged system (the pilot Gram buffer is free here)
        e = launch_chol_solve(d, nb, ws.G, thw, nullptr, ws.stat, ws.thbuf, s);
        if (e != cudaSuccess) return e;
        {
            dim3 grid((d.L * d.n_rx + 127) / 128, nb);
            k_ls_spread<<<grid, 128, 0, s>>>(d, ws.ls_scale, ws.ls_rep, (const cplx*)thw, (cplx*)theta0);
            count_launch();
        }
    } else {
        Dims dd = d;
        dd.L = d.T_p;
        dd.Lp = (d.T_p + 3) & ~3;
        dd.Ltot = dd.Lp + d.RP;
        {
            const int total = dd.Ltot * dd.Lp;
            dim3 grid(min((total + 255) / 256, 64), nb);
            k_ls_dual_build<<<grid, 256, 0, s>>>(d, dd, (const cplx*)io.PsiP, (const cplx*)io.Xp, (const cplx*)io.Yp,
                                                 (cplx*)ws.G);
            count_launch();
        }
        double* A = ws.Gp;   // [nb][T_p][n_rx], the pilot Gram buffer is free here
        e = launch_chol_solve(dd, nb, ws.G, A, nullptr, ws.stat, ws.thbuf, s);
        if (e != cudaSuccess) return e;
        dim3 grid((d.L * d.n_rx + 127) / 128, nb);
        k_ls_dual_expand<<<grid, 128, 0, s>>>(d, (const cplx*)io.PsiP, (const cplx*)io.Xp, (const cplx*)A, (cplx*)theta0);
        count_launch();
    }
    if (status) {
        e = cudaMemcpyAsync(status, ws.stat, (size_t)nb * 4, cudaMemcpyDeviceToDevice, s);
        if (e != cudaSuccess) return e;
    }
    return cudaGetLastError();
}

cudaError_t launch_accumulate_ser(const Dims& d, int nb, const int32_t* kstar, const double* Xd, double* acc,
                                  cudaStream_t s) {
    if (nb == 0) return cudaSuccess;
    k_accumulate_ser<<<nb, 128, 0, s>>>(d, nb, kstar, (const cplx*)Xd, acc);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_accumulate_ber(const Dims& d, int nb, const int32_t* kstar, const double* Xd, double* acc,
                                  cudaStream_t s) {
    if (nb == 0) return cudaSuccess;
    k_accumulate_ber<<<nb, 128, 0, s>>>(d, nb, kstar, (const cplx*)Xd, acc);
    count_launch();
    return cudaGetLastError();
}

}  // namespace sbce
