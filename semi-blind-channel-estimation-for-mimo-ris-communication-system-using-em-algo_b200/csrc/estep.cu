// E-step of the semi-blind EM estimator: posterior over all M^n_tx QAM
// hypotheses of every data symbol.
//
// Reference semantics (one data symbol t, /root/reference/Proposed_method_NMSEvsTp.py:53-62):
//   d2_k   = || y_t - Z(x_k, psi~_t) theta ||^2          for all K = M^n_tx hypotheses
//   beta_k = exp(-d2_k / varn^2) / sum_k' exp(-d2_k'/varn^2)
//   numer += beta_k Z^H y ,  denom += beta_k Z^H Z
// which collapses (SURVEY.md 8a-6) to per-symbol statistics
//   m_t = sum_k beta_k conj(x_k)          R_t = sum_k beta_k conj(x_k) x_k^T
// and, for the hard-decision variant (Proposed method/ML_detecctor.py:66-77),
//   k*  = argmax_k beta_k (first index on ties), rank-one statistics at x_{k*}.
//
// B200 design (not a translation of the double Python loop):
//  1. k_heff_qr: one LANE per data symbol.  The Kronecker design row
//     psi~_t^T (x) x^T (x) I is never formed; the lane contracts theta over the
//     RIS index into the n_rx x n_tx effective channel Heff_t and immediately
//     reduces [Heff_t | y_t] to upper-triangular form with Householder
//     reflections in registers (real non-negative diagonal).  Then
//     d2(x) = c0 + sum_i | ytilde_i - sum_{j>=i} R_ij x_j |^2  exactly.
//  2. k_enum: one HALF-WARP (16 lanes) per data symbol up to 4 streams, two
//     symbols per warp (a whole warp per symbol for 5..8 streams), walks the
//     hypothesis tree stream n_tx-1 -> 1 with partial residuals in registers; the
//     top levels are split across the group's lanes, the inner levels are
//     group-uniform loops fed by shared-memory tables R_ij*c_m (on half-warps the
//     stream-1 level is packed: the lanes split the children of one live node).  Every collective
//     is a group collective, so the two symbols of a warp may take different paths.  Because R_00 is real, the last stream separates into its
//     in-phase and quadrature PAM components, so the sum over the M leaves of a
//     node is a product of two sqrt(M)-term sums: every hypothesis is accounted
//     for exactly, at O(1) work per node when the node's best leaf is more than
//     64 varn^2 above the running minimum (its whole weight is < 2e-28 of the
//     normaliser and rounds away in FP64, exactly as in the reference where
//     float(beta) underflows).  Online max-subtracted accumulation per lane,
//     group-shuffle log-sum-exp merge at the end; the incomplete-data
//     log-likelihood sum_k exp(-d2/varn^2) falls out of the same reduction.
#include <math.h>

#include "common.cuh"
#include "tensor.cuh"
#include "tree.cuh"

namespace sbce {

static __device__ __forceinline__ constexpr int cmax(int a, int b) { return a > b ? a : b; }

// ---------------------------------------------------------------------------
// pilots: symbols known with probability one
// ---------------------------------------------------------------------------
__global__ void k_pilot_stats(int n_tx, int total, const cplx* __restrict__ Xp, cplx* __restrict__ pm,
                              cplx* __restrict__ pR) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;  // flat (b,t)
    if (s >= total) return;
    const cplx* x = Xp + (size_t)s * n_tx;
    for (int i = 0; i < n_tx; ++i) {
        cplx xi = x[i];
        pm[(size_t)s * n_tx + i] = cconj(xi);
        for (int j = 0; j < n_tx; ++j) pR[((size_t)s * n_tx + i) * n_tx + j] = cmulc(x[j], xi);  // conj(x_i) x_j
    }
}

cudaError_t launch_pilot_stats(const Dims& d, int nb, const double* Xp, double* pil_m, double* pil_R, cudaStream_t s) {
    int total = nb * d.T_p;
    if (total == 0) return cudaSuccess;
    k_pilot_stats<<<(total + 127) / 128, 128, 0, s>>>(d.n_tx, total, (const cplx*)Xp, (cplx*)pil_m, (cplx*)pil_R);
    count_launch();
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// 1. effective channel + Householder QR, one lane per symbol
// ---------------------------------------------------------------------------
// Per-lane tail shared by the effective-channel kernels: A = Heff_t (rows >= NRX zero), then
// y' = y - Heff o_t (superimposed pilots), Householder QR of [A | y] in registers, record store.
template <int NTX, int NRX>
__device__ __forceinline__ void heff_qr_finish(const Dims& d, int b, int t, cplx (&A)[cmax(NTX, NRX)][NTX],
                                               const cplx* __restrict__ Yd, const cplx* __restrict__ Xoff,
                                               double* __restrict__ qr) {
    constexpr int NR = cmax(NTX, NRX);
    cplx y[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) y[r] = (r < NRX) ? Yd[((size_t)b * d.T_d + t) * NRX + r] : mk(0.0, 0.0);
    if (Xoff != nullptr) {   // superimposed pilots: hypotheses are x_k + o_t  <=>  y' = y - Heff o_t
        const cplx* o = Xoff + ((size_t)b * d.T_d + t) * NTX;
#pragma unroll
        for (int j = 0; j < NTX; ++j) {
            const cplx oj = o[j], noj = mk(-oj.x, -oj.y);
#pragma unroll
            for (int r = 0; r < NRX; ++r) cfma(y[r], A[r][j], noj);
        }
    }

    // Householder, column k; afterwards row k is rotated so that R_kk = ||x|| >= 0 is real
#pragma unroll
    for (int k = 0; k < NTX; ++k) {
        double nrm2 = 0.0;
#pragma unroll
        for (int i = k; i < NR; ++i) nrm2 += cnorm2(A[i][k]);
        if (nrm2 > 0.0) {
            const double nrm = sqrt(nrm2);
            const cplx a0 = A[k][k];
            const double abs0 = sqrt(cnorm2(a0));
            const cplx phase = abs0 > 0.0 ? mk(a0.x / abs0, a0.y / abs0) : mk(1.0, 0.0);
            // v = x - alpha e_k with alpha = -phase*nrm  =>  v_k = phase*(abs0+nrm)
            const cplx vk = cscale(phase, abs0 + nrm);
            const double beta = 1.0 / (nrm * (nrm + abs0));  // 2 / (v^H v)
#pragma unroll
            for (int c = k + 1; c <= NTX; ++c) {  // c == NTX is the y column
                cplx w = mk(0.0, 0.0);
                if (c < NTX) {
                    cfmac(w, A[k][c], vk);  // conj(v_k) * a
#pragma unroll
                    for (int i = k + 1; i < NR; ++i) cfmac(w, A[i][c], A[i][k]);
                    w = cscale(w, beta);
                    cplx nw = mk(-w.x, -w.y);
                    cfma(A[k][c], nw, vk);
#pragma unroll
                    for (int i = k + 1; i < NR; ++i) cfma(A[i][c], nw, A[i][k]);
                } else {
                    cfmac(w, y[k], vk);
#pragma unroll
                    for (int i = k + 1; i < NR; ++i) cfmac(w, y[i], A[i][k]);
                    w = cscale(w, beta);
                    cplx nw = mk(-w.x, -w.y);
                    cfma(y[k], nw, vk);
#pragma unroll
                    for (int i = k + 1; i < NR; ++i) cfma(y[i], nw, A[i][k]);
                }
            }
            // rotate row k by conj(-phase): diagonal becomes +nrm
            const cplx rot = mk(-phase.x, phase.y);
#pragma unroll
            for (int c = k + 1; c < NTX; ++c) A[k][c] = cmul(A[k][c], rot);
            y[k] = cmul(y[k], rot);
            A[k][k] = mk(nrm, 0.0);
        } else {
            A[k][k] = mk(0.0, 0.0);
        }
    }

    double* rec = qr + ((size_t)b * d.T_d + t) * d.rec;
#pragma unroll
    for (int i = 0; i < NTX; ++i)
#pragma unroll
        for (int j = i; j < NTX; ++j) {
            rec[qr_rec_R(NTX, i, j)] = A[i][j].x;
            rec[qr_rec_R(NTX, i, j) + 1] = (j == i) ? 0.0 : A[i][j].y;
        }
#pragma unroll
    for (int i = 0; i < NTX; ++i) {
        rec[qr_rec_yt(NTX, i)] = y[i].x;
        rec[qr_rec_yt(NTX, i) + 1] = y[i].y;
    }
    double c0 = 0.0;
#pragma unroll
    for (int i = NTX; i < NR; ++i) c0 += cnorm2(y[i]);
    rec[qr_rec_c0(NTX)] = c0;
    rec[qr_rec_c0(NTX) + 1] = 0.0;
}

template <int NTX, int NRX>
__global__ void __launch_bounds__(128) k_heff_qr(Dims d, const cplx* __restrict__ Yd, const cplx* __restrict__ PsiD,
                                                 const cplx* __restrict__ theta, const int32_t* __restrict__ active,
                                                 const cplx* __restrict__ Xoff, double* __restrict__ qr, int use_smem) {
    constexpr int NR = cmax(NTX, NRX);
    extern __shared__ double2 heff_smem[];
    const int b = blockIdx.y;
    if (active != nullptr && active[b] == 0) return;
    // theta of the trial is read by every lane at warp-uniform addresses, 16 values per RIS index: staged in
    // shared memory once per CTA (coalesced) the inner loop issues LDS broadcasts instead of global loads
    // (the global-load queue was the kernel's top stall, profiles/r01m); use_smem = 0: theta too long
    const cplx* th = theta + (size_t)b * d.L * NRX;
    if (use_smem) {
        for (int e = threadIdx.x; e < d.L * NRX; e += blockDim.x) heff_smem[e] = th[e];
        __syncthreads();
        th = heff_smem;
    }
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= d.T_d) return;

    const cplx* psi = PsiD + ((size_t)(d.psi_shared ? 0 : b) * d.T_d + t) * d.N1;

    cplx A[NR][NTX];
#pragma unroll
    for (int r = 0; r < NR; ++r)
#pragma unroll
        for (int j = 0; j < NTX; ++j) A[r][j] = mk(0.0, 0.0);

    // Heff[r][j] = sum_n' psi~[t][n'] Theta[n'*n_tx + j][r]; theta reads are warp-uniform (broadcast)
#pragma unroll 4
    for (int n = 0; n < d.N1; ++n) {
        const cplx p = psi[n];
        const cplx* row = th + (size_t)n * NTX * NRX;
#pragma unroll
        for (int j = 0; j < NTX; ++j)
#pragma unroll
            for (int r = 0; r < NRX; ++r) cfma(A[r][j], p, row[j * NRX + r]);
    }
    heff_qr_finish<NTX, NRX>(d, b, t, A, Yd, Xoff, qr);
}

// ---------------------------------------------------------------------------
// 1a. the same on the FP64 tensor path.  Heff = Psi_d (T_d x N+1) . Theta (N+1 x n_tx n_rx) is a dense complex
// GEMM per trial (the RIS contraction, Proposed_method_NMSEvsTp.py:56 without the Kronecker products); the
// per-lane kernel above streams each lane's psi row with stride-(N+1) 16-byte loads (17 % of HBM peak, the
// load queue is its top stall, profiles/r01m).  Here a warp owns 32 symbols = two 16-row MMA tiles: A
// fragments (psi) are 128-byte row segments per 8-column step straight from global memory, B fragments
// (Theta, shared by the whole CTA) come from a padded shared-memory copy; the 2 x NT x 4 accumulators are
// transposed through shared memory so that lane t ends up with Heff_t in registers and runs the same
// Householder tail.
// ---------------------------------------------------------------------------
template <int NTX, int NRX>
__global__ void __launch_bounds__(128, 4) k_heff_qr_mma(Dims d, const cplx* __restrict__ Yd,
                                                        const cplx* __restrict__ PsiD, const cplx* __restrict__ theta,
                                                        const int32_t* __restrict__ active,
                                                        const cplx* __restrict__ Xoff, double* __restrict__ qr) {
    constexpr int NR = cmax(NTX, NRX);
    constexpr int NC = NTX * NRX;          // complex columns of the GEMM: (j, r) -> j * NRX + r
    constexpr int NT = (NC + 7) / 8;       // 8-column MMA tiles
    constexpr int TS = NT * 8 + 2;         // row stride of the staged Theta: fragment loads are conflict-free
    constexpr int HS = NC + 1;             // row stride of the transposed result
    extern __shared__ double2 heff_smem[];
    const int b = blockIdx.y;
    if (active != nullptr && active[b] == 0) return;
    const int N1 = d.N1, KP = (N1 + 7) & ~7;
    cplx* sTh = heff_smem;                 // [KP][TS], rows >= N1 and columns >= NC zero
    cplx* sH = sTh + KP * TS;              // [4 warps][32][HS]
    {
        const cplx* th = theta + (size_t)b * d.L * NRX;
        for (int e = threadIdx.x; e < KP * TS; e += blockDim.x) {
            const int n = e / TS, c = e % TS;
            sTh[e] = (n < N1 && c < NC) ? th[n * NC + c] : mk(0.0, 0.0);
        }
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
    const int t0 = blockIdx.x * 128 + warp * 32;
    if (t0 >= d.T_d) return;
    const cplx* psi_b = PsiD + (size_t)(d.psi_shared ? 0 : b) * d.T_d * N1;
    const cplx* prow[2][2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int h = 0; h < 2; ++h) prow[mt][h] = psi_b + (size_t)min(t0 + mt * 16 + g + 8 * h, d.T_d - 1) * N1;
    {   // pull this warp's 32 phase rows into L2 before the k loop touches them (lane = row): the fragment loads
        // below are then L2 hits instead of DRAM round trips (0.200 -> 0.174 ms at the north-star size)
        const char* rowp = (const char*)(psi_b + (size_t)min(t0 + lane, d.T_d - 1) * N1);
        for (int o = 0; o < N1 * (int)sizeof(cplx); o += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(rowp + o));
    }
    double cr[2][NT][4], ci[2][NT][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
            for (int e = 0; e < 4; ++e) { cr[mt][nt][e] = 0.0; ci[mt][nt][e] = 0.0; }
#pragma unroll 2
    for (int k0 = 0; k0 < KP; k0 += 8) {
        const int ka = k0 + tig, kb = ka + 4;
        const bool va = ka < N1, vb = kb < N1;
        double ar[2][4], ai[2][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            // A fragment order: (row g, k lo), (row g+8, k lo), (row g, k hi), (row g+8, k hi)
            const cplx a0 = va ? prow[mt][0][ka] : mk(0.0, 0.0), a1 = va ? prow[mt][1][ka] : mk(0.0, 0.0);
            const cplx a2 = vb ? prow[mt][0][kb] : mk(0.0, 0.0), a3 = vb ? prow[mt][1][kb] : mk(0.0, 0.0);
            ar[mt][0] = a0.x; ar[mt][1] = a1.x; ar[mt][2] = a2.x; ar[mt][3] = a3.x;
            ai[mt][0] = a0.y; ai[mt][1] = a1.y; ai[mt][2] = a2.y; ai[mt][3] = a3.y;
        }
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            const cplx b0 = sTh[ka * TS + 8 * nt + g], b1 = sTh[kb * TS + 8 * nt + g];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                // (ar + i ai)(br + i bi): re += ar br - ai bi ; im += ar bi + ai br
                dmma16x8x8(cr[mt][nt], ar[mt], b0.x, b1.x);
                dmma16x8x8(ci[mt][nt], ar[mt], b0.y, b1.y);
                dmma16x8x8(cr[mt][nt], ai[mt], -b0.y, -b1.y);
                dmma16x8x8(ci[mt][nt], ai[mt], b0.x, b1.x);
            }
        }
    }
    // transpose through shared memory: accumulator (row g + 8h, columns 8 nt + 2 tig, + 1) -> H[symbol][column]
    cplx* H = sH + (size_t)warp * 32 * HS;
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int row = mt * 16 + g + 8 * h, c = 8 * nt + 2 * tig;
                if (c < NC) H[row * HS + c] = mk(cr[mt][nt][2 * h], ci[mt][nt][2 * h]);
                if (c + 1 < NC) H[row * HS + c + 1] = mk(cr[mt][nt][2 * h + 1], ci[mt][nt][2 * h + 1]);
            }
    __syncwarp();
    const int t = t0 + lane;
    if (t >= d.T_d) return;
    cplx A[NR][NTX];
#pragma unroll
    for (int r = 0; r < NR; ++r)
#pragma unroll
        for (int j = 0; j < NTX; ++j) A[r][j] = (r < NRX) ? H[lane * HS + j * NRX + r] : mk(0.0, 0.0);
    heff_qr_finish<NTX, NRX>(d, b, t, A, Yd, Xoff, qr);
}

// ---------------------------------------------------------------------------
// 1b. wide arrays (n_tx = 5..8): the (8 x (n_tx+1)) work matrix [Heff_t | y_t] no longer fits the
// registers of one lane, so EIGHT lanes share a symbol, lane r owning receive row r.  The theta reads of
// the RIS contraction are then 8 consecutive complex values per (n', j) -- one 128-byte line per symbol
// group; the Householder inner products become 3-step xor-shuffle sums inside the aligned 8-lane group.
// All lanes execute every shuffle (no group-divergent branches); same record layout as k_heff_qr.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double group8_sum(double v) {
    v += shfl_xor_d(v, 4);
    v += shfl_xor_d(v, 2);
    v += shfl_xor_d(v, 1);
    return v;
}

template <int NTX>
__global__ void __launch_bounds__(128) k_heff_qr_rows(Dims d, const cplx* __restrict__ Yd,
                                                      const cplx* __restrict__ PsiD, const cplx* __restrict__ theta,
                                                      const int32_t* __restrict__ active,
                                                      const cplx* __restrict__ Xoff, double* __restrict__ qr) {
    const int b = blockIdx.y;
    if (active != nullptr && active[b] == 0) return;
    const int r = threadIdx.x & 7;
    const int tq = blockIdx.x * (blockDim.x >> 3) + (threadIdx.x >> 3);
    const bool tv = tq < d.T_d;
    const int t = tv ? tq : d.T_d - 1;   // surplus groups redo the last symbol (they must stay in the shuffles)
    const int nrx = d.n_rx;
    const bool rv = r < nrx;
    const int rr = rv ? r : 0;

    const cplx* psi = PsiD + ((size_t)(d.psi_shared ? 0 : b) * d.T_d + t) * d.N1;
    const cplx* th = theta + (size_t)b * d.L * nrx;

    cplx A[NTX + 1];   // row r of [Heff | y]
#pragma unroll
    for (int j = 0; j <= NTX; ++j) A[j] = mk(0.0, 0.0);
#pragma unroll 2
    for (int n = 0; n < d.N1; ++n) {
        const cplx p = psi[n];
        const cplx* row = th + (size_t)n * NTX * nrx + rr;
#pragma unroll
        for (int j = 0; j < NTX; ++j) cfma(A[j], p, __ldg(&row[j * nrx]));
    }
    A[NTX] = Yd[((size_t)b * d.T_d + t) * nrx + rr];
    if (Xoff != nullptr) {   // superimposed pilots: y' = y - Heff o_t
        const cplx* o = Xoff + ((size_t)b * d.T_d + t) * NTX;
#pragma unroll
        for (int j = 0; j < NTX; ++j) {
            const cplx oj = o[j];
            cfma(A[NTX], A[j], mk(-oj.x, -oj.y));
        }
    }
    if (!rv) {
#pragma unroll
        for (int j = 0; j <= NTX; ++j) A[j] = mk(0.0, 0.0);
    }

#pragma unroll
    for (int k = 0; k < NTX; ++k) {
        const double nrm2 = group8_sum(r >= k ? cnorm2(A[k]) : 0.0);
        const bool ok = nrm2 > 0.0;
        const double nrm = sqrt(nrm2);
        const int src = (threadIdx.x & 24) + k;   // lane that owns row k of this group
        const cplx a0 = mk(shfl_d(A[k].x, src), shfl_d(A[k].y, src));
        const double abs0 = sqrt(cnorm2(a0));
        const cplx phase = abs0 > 0.0 ? mk(a0.x / abs0, a0.y / abs0) : mk(1.0, 0.0);
        const cplx vk = cscale(phase, abs0 + nrm);                      // v_k = phase (|a0| + ||x||)
        const double beta = ok ? 1.0 / (nrm * (nrm + abs0)) : 0.0;      // 2 / (v^H v)
        const cplx vr = (r == k) ? vk : (r > k ? A[k] : mk(0.0, 0.0));  // this lane's entry of v
#pragma unroll
        for (int c = k + 1; c <= NTX; ++c) {
            cplx w = mk(0.0, 0.0);
            cfmac(w, A[c], vr);   // conj(v_r) a_rc
            w = mk(group8_sum(w.x) * beta, group8_sum(w.y) * beta);
            const cplx nw = mk(-w.x, -w.y);
            cfma(A[c], nw, vr);
        }
        if (r == k) {   // rotate row k so that its diagonal entry is +||x||
            const cplx rot = mk(-phase.x, phase.y);
#pragma unroll
            for (int c = k + 1; c <= NTX; ++c) A[c] = cmul(A[c], rot);
            A[k] = mk(ok ? nrm : 0.0, 0.0);
        }
    }
    const double c0 = group8_sum(r >= NTX ? cnorm2(A[NTX]) : 0.0);
    if (!tv) return;
    double* rec = qr + ((size_t)b * d.T_d + t) * d.rec;
    if (r < NTX) {
#pragma unroll
        for (int j = 0; j < NTX; ++j)
            if (j >= r) {
                rec[qr_rec_R(NTX, r, j)] = A[j].x;
                rec[qr_rec_R(NTX, r, j) + 1] = (j == r) ? 0.0 : A[j].y;
            }
        rec[qr_rec_yt(NTX, r)] = A[NTX].x;
        rec[qr_rec_yt(NTX, r) + 1] = A[NTX].y;
    }
    if (r == 0) {
        rec[qr_rec_c0(NTX)] = c0;
        rec[qr_rec_c0(NTX) + 1] = 0.0;
    }
}

// ---------------------------------------------------------------------------
// 2. hypothesis-tree enumeration, one half-warp (n_tx <= 4) or warp per symbol
// ---------------------------------------------------------------------------
constexpr double SBCE_THR = 64.0;  // nodes whose best leaf is > THR*varn^2 above the incumbent weigh < e^-64
__device__ __forceinline__ double shfl_xor_h(unsigned hm, double v, int o) { return __shfl_xor_sync(hm, v, o); }

// Cooperative, out-of-line processing of the queued candidate nodes of one symbol: every lane of the
// symbol's group takes queue entries round-robin, rebuilds the node's residuals from its code, sums its
// M leaves in closed form (separable in-phase / quadrature PAM sums) and the group adds the result to the
// shared accumulators, kept relative to the reference distance `aref` (rescaled when the incumbent improves).
// `count` entries are queued; the caller empties the queue afterwards.
// Only the calling group takes part: the other symbol of a warp may be anywhere else.
template <int NTX, int SQM>
__device__ __noinline__ void enum_flush(double* ws, double warp_best, int count) {
    typedef EnumT<NTX, SQM> E;
    const int lane = E::glane();
    const unsigned hm = E::gmask();
    __syncwarp(hm);
    const int n = min(count, E::QCAP);
    const int* q = (const int*)(ws + E::O_Q);
    const double* g = ws + E::O_G;
    const double inv_s2 = ws[E::O_S2];
    double aref = ws[E::O_AREF];
    if (warp_best < aref) {
        // aref starts at the finite sentinel 1e300, above every admitted d2 (include/sbce.h): the argument is then
        // hugely negative (or -inf), f = 0, and the still-zero accumulators stay zero
        const double f = exp((warp_best - aref) * inv_s2);
        for (int i = lane; i < E::NACC; i += E::G) ws[E::O_ACC + i] *= f;
        aref = warp_best;
    }
    double* A = ws + E::O_ACC;
    // Narrow path.  At operating SNRs the queue almost always holds ONE node (the arg-min node, whose M leaves
    // carry the whole posterior) or two; the general path below would run all 16 lanes through ~700
    // instructions (9 exponentials in sequence per lane) for it.  Here the group shares one entry: the lanes of
    // a 2*SQM subgroup take one PAM level of the in-phase or of the quadrature component each (one exponential
    // per lane, min / sums by xor shuffles), every lane then holds the node's closed-form leaf sums and lane i
    // adds statistic i (mod 16).
    if (n <= 2) {
        constexpr int LG = (SQM == 2 ? 1 : (SQM == 4 ? 2 : 3));
        const int a = lane & (SQM - 1);
        const bool isQ = (lane >> LG) & 1;
        const double pq = E::pam(a);
        for (int e = 0; e < n; ++e) {
            const int code = q[e];
            cplx t0;
            const double base = E::rebuild(ws, code, t0);
            const double ev = (isQ ? t0.y : t0.x) - g[a];
            const double dd = ev * ev;
            double mn = dd;
#pragma unroll
            for (int o = SQM / 2; o > 0; o >>= 1) mn = fmin(mn, shfl_xor_h(hm, mn, o));
            const double w = exp((mn - dd) * inv_s2);
            double s0 = w, s1 = pq * w, s2 = pq * pq * w;
#pragma unroll
            for (int o = SQM / 2; o > 0; o >>= 1) {
                s0 += shfl_xor_h(hm, s0, o);
                s1 += shfl_xor_h(hm, s1, o);
                s2 += shfl_xor_h(hm, s2, o);
            }
            const double o0 = shfl_xor_h(hm, s0, SQM), o1 = shfl_xor_h(hm, s1, SQM), o2 = shfl_xor_h(hm, s2, SQM);
            const double om = shfl_xor_h(hm, mn, SQM);
            const double EI = isQ ? o0 : s0, A1 = isQ ? o1 : s1, A2 = isQ ? o2 : s2, minI = isQ ? om : mn;
            const double EQ = isQ ? s0 : o0, B1 = isQ ? s1 : o1, B2 = isQ ? s2 : o2, minQ = isQ ? mn : om;
            const double W = exp((aref - (base + minI + minQ)) * inv_s2);
            const double E0 = W * EI * EQ;
            const cplx F0 = mk(W * A1 * EQ, -W * EI * B1);  // sum over leaves of e * conj(x_0)
            const double Q0 = W * (A2 * EQ + EI * B2);      // sum over leaves of e * |x_0|^2
            // statistic idx belongs to lane idx & 15: every lane picks its values out of the (group-uniform) results
            // with predicated register moves and then makes ONE shared-memory update per 16 statistics (as ~25
            // single-lane read-modify-writes behind divergent branches this was 14 % of the kernel's stall
            // samples, profiles/r02m); per entry, so the order of the additions is unchanged
            constexpr int NR = (E::NACC + E::G - 1) / E::G;
            double mine[NR];
#pragma unroll
            for (int r = 0; r < NR; ++r) mine[r] = 0.0;
            E::node_stats(code, E0, F0, Q0, [&](int idx, double v) {
                if ((idx & (E::G - 1)) == lane) mine[idx / E::G] = v;
            });
#pragma unroll
            for (int r = 0; r < NR; ++r)
                if (E::G * r + lane < E::NACC) A[E::G * r + lane] += mine[r];
            __syncwarp(hm);
        }
        if (lane == 0) ws[E::O_AREF] = aref;
        __syncwarp(hm);
        return;
    }
    // General path: one queue entry per lane per round; the group reduces every statistic right away (rare
    // path: keep the register footprint small so that it does not limit the occupancy of the scan loop)
    // per round every lane drops the NACC contributions of its queue entry into a shared scratch
    // [NACC][16]; afterwards lane i sums statistic i over the lanes that held an entry (a transpose
    // instead of NACC butterfly reductions: ~25 stores + nround loads per lane, no shuffles)
    double* scr = ws + E::O_SCR;
    int nround = 0;
    for (int e0 = 0; e0 < n; e0 += E::G) {
        const int e = e0 + lane;
        const bool have = e < n;
        nround = min(E::G, n - e0);
        const int code = have ? q[e] : 0;
        cplx t0;
        const double base = E::rebuild(ws, code, t0);
        double minI = 1e300, minQ = 1e300;
#pragma unroll
        for (int a = 0; a < SQM; ++a) {
            const double eI = t0.x - g[a], eQ = t0.y - g[a];
            minI = fmin(minI, eI * eI);
            minQ = fmin(minQ, eQ * eQ);
        }
        const double W = have ? exp((aref - (base + minI + minQ)) * inv_s2) : 0.0;
        double EI = 0, A1 = 0, A2 = 0, EQ = 0, B1 = 0, B2 = 0;
#pragma unroll 1
        for (int a = 0; a < SQM; ++a) {
            const double pq = E::pam(a);
            const double eI = t0.x - g[a], eQ = t0.y - g[a];
            const double wI = exp((minI - eI * eI) * inv_s2), wQ = exp((minQ - eQ * eQ) * inv_s2);
            EI += wI; A1 = fma(pq, wI, A1); A2 = fma(pq * pq, wI, A2);
            EQ += wQ; B1 = fma(pq, wQ, B1); B2 = fma(pq * pq, wQ, B2);
        }
        const double E0 = W * EI * EQ;
        const cplx F0 = mk(W * A1 * EQ, -W * EI * B1);  // sum over leaves of e * conj(x_0)
        const double Q0 = W * (A2 * EQ + EI * B2);      // sum over leaves of e * |x_0|^2
        E::node_stats(code, E0, F0, Q0, [&](int idx, double v) { scr[idx * E::G + lane] = v; });
        __syncwarp(hm);
        for (int i = lane; i < E::NACC; i += E::G) {
            double acc = 0.0;
            for (int e2 = 0; e2 < nround; ++e2) acc += scr[i * E::G + e2];
            A[i] += acc;
        }
        __syncwarp(hm);
    }
    __syncwarp(hm);
    if (lane == 0) ws[E::O_AREF] = aref;
    __syncwarp(hm);
}

template <int NTX, int SQM, bool HARD>
struct Scan {
    typedef EnumT<NTX, SQM> E;
    static constexpr int M = E::M;
    double* ws;
    const cplx* tab;
    const double* g;
    double r0;        // R_00 (real): PAM unit of the leaf stream
    double thr;       // 64 varn^2
    double best, lim; // incumbent distance and enqueue limit best + thr
    int bestk;
    int cnt;          // queued nodes (group-uniform)
    bool prune;       // skip subtrees whose partial distance already exceeds lim (bit-identical results)

    // the M leaves below a node: t0 = residual on row 0, nb = partial distance of the node, code = node digits.
    // Every lane of the group calls it (`live`: the lane holds a node), so that queue slots are handed out in lane
    // order by a ballot: the queue order follows from which lane holds which node, not from the atomics' timing.
    __device__ __forceinline__ void leaf(cplx t0, double nb, int code, bool live) {
        const double fI = E::fold(t0.x, r0), fQ = E::fold(t0.y, r0);
        const double nodemin = fma(fI, fI, fma(fQ, fQ, nb));
        const bool hit = live && nodemin <= lim;   // rare at operating SNRs
        if (hit && nodemin <= best) {
            double dI, dQ;
            const int iI = E::slice(t0.x, g, dI), iQ = E::slice(t0.y, g, dQ);
            const double val = nb + dI + dQ;
            const int k = code + ((iQ * SQM + iI) << (E::BITS * (NTX - 1)));
            if (val < best || (val == best && k < bestk)) {
                best = val;
                bestk = k;
                lim = HARD ? val : val + thr;
            }
        }
        if (!HARD) {
            const unsigned q = __ballot_sync(E::gmask(), hit) >> E::gshift();
            if (q != 0u) {
                if (hit) {
                    const int slot = cnt + __popc(q & ((1u << E::glane()) - 1u));
                    if (slot < E::QCAP) ((int*)(ws + E::O_Q))[slot] = code;
                }
                cnt += __popc(q);
            }
        }
    }

    // group arg-min of (best, bestk), first index on ties; every lane ends with it and the matching limit
    __device__ __forceinline__ void merge_best() {
        const unsigned hm = E::gmask();
#pragma unroll
        for (int o = E::G / 2; o > 0; o >>= 1) {
            const double ob = shfl_xor_h(hm, best, o);
            const int ok = __shfl_xor_sync(hm, bestk, o);
            if (ob < best || (ob == best && ok < bestk)) { best = ob; bestk = ok; }
        }
        lim = HARD ? best : best + thr;
    }

    // PER_LANE: nodes a lane may enqueue before the next call
    template <int PER_LANE>
    __device__ __forceinline__ void maybe_flush() {
        if (!HARD && cnt > E::QCAP - E::G * PER_LANE) {
            const unsigned hm = E::gmask();
            double wb = best;
#pragma unroll
            for (int o = E::G / 2; o > 0; o >>= 1) wb = fmin(wb, shfl_xor_h(hm, wb, o));
            enum_flush<NTX, SQM>(ws, wb, cnt);
            cnt = 0;
        }
    }

    // Branch and bound.  Every leaf below a node has d2 >= the node's partial distance `base`; once
    // base > lim (incumbent + 64 varn^2) none of them can improve the arg-min or pass the enqueue test,
    // so the subtree is "dead": visiting it would change nothing.  Lanes carry a dead flag instead of
    // returning (the loops contain group collectives and must stay convergent within the group); a row
    // or subtree is skipped only when a vote of the group says it is dead for all its lanes.

    // streams S_ ... 1 enumerated with group-uniform loops
    template <int S_>
    __device__ __forceinline__ void inner(const cplx (&acc)[NTX], double base, int code, cplx r01, bool dead) {
        dead = dead || (prune && base > lim);
        if constexpr (S_ == 0) {
            leaf(acc[0], base, code, !dead);
        } else if constexpr (S_ == 1 && M % E::G == 0) {
            // Innermost node level, packed (half-warp groups: M is 16 or 64).  The group takes its live nodes one
            // after the other, in lane order, and its G lanes split the M stream-1 symbols below each one, G per
            // step, a leaf node per lane.  At operating SNRs one or two of 16 lanes are live here, and each costs
            // one step instead of the whole group walking M nodes in lock-step for it.
            // After every step the group merges its incumbent.  So the incumbent, the enqueue limit, the queued
            // nodes, their order (lane order within a step) and the flush points change only in steps that hold a
            // live node, and a step is the same slice of one node's children at the same lanes whether dead nodes
            // are skipped or not: the pruned walk and the full scan run the same live steps in the same order.
            const unsigned hm = E::gmask();
            unsigned todo = __ballot_sync(hm, !dead) >> E::gshift();
            while (todo != 0u) {
                const int src = __ffs(todo) - 1;
                todo &= todo - 1u;
                cplx pacc[NTX];   // the node's residuals; rows above 1 are not read
#pragma unroll
                for (int i = 0; i < NTX; ++i)
                    pacc[i] = i <= 1 ? mk(__shfl_sync(hm, acc[i].x, src, E::G), __shfl_sync(hm, acc[i].y, src, E::G))
                                     : acc[i];
                const double pbase = __shfl_sync(hm, base, src, E::G);
                const int pcode = __shfl_sync(hm, code, src, E::G);
#pragma unroll 1
                for (int m = E::glane(); m < M; m += E::G) {
                    cplx nacc[NTX];
                    const double nb = E::step(pacc, nacc, 1, m, pbase, g, tab);
                    const double b0 = best;
                    inner<0>(nacc, nb, pcode + (m << (E::BITS * (NTX - 2))), r01, false);
                    if (__any_sync(hm, best != b0)) merge_best();
                    maybe_flush<1>();
                }
            }
        } else if constexpr (S_ == 1) {
            if (__all_sync(E::gmask(), dead)) return;
            // innermost node level, every lane its own node (warp groups: M < G).  |u_1|^2 and R_01 x_1 are
            // separable in the in-phase / quadrature indices.
            // The queue is checked once per node (its M leaves per lane) when that fits, else once per row of SQM.
            constexpr bool NODE_FLUSH = E::G * M < E::QCAP;
            const double* g1 = g + SQM;
            double dI1[SQM];
#pragma unroll
            for (int a = 0; a < SQM; ++a) {
                const double eI = acc[1].x - g1[a];
                dI1[a] = eI * eI;
            }
#pragma unroll 1
            for (int iQ = 0; iQ < SQM; ++iQ) {
                // the quadrature term is formed here (a table indexed by the loop counter lived in local memory);
                // product and sum are rounded separately, as the table version did
                const double eQ = acc[1].y - g1[iQ];
                const double bq = base + __dmul_rn(eQ, eQ);
                const bool deadq = dead || (prune && bq > lim);
                if (__all_sync(E::gmask(), deadq)) continue;
                const double pQ = E::pam(iQ);
                // t = acc0 - pQ * (i r01) = acc0 - pQ*(-r01.y + i r01.x)
                const cplx tq = mk(fma(pQ, r01.y, acc[0].x), fma(-pQ, r01.x, acc[0].y));
                const int cq = code + ((iQ * SQM) << (E::BITS * (NTX - 2)));
#pragma unroll
                for (int iI = 0; iI < SQM; ++iI) {
                    const double pI = E::pam(iI);
                    const cplx t0 = mk(fma(-pI, r01.x, tq.x), fma(-pI, r01.y, tq.y));
                    leaf(t0, bq + dI1[iI], cq + (iI << (E::BITS * (NTX - 2))), !deadq);
                }
                if (!NODE_FLUSH) maybe_flush<SQM>();
            }
            if (NODE_FLUSH) maybe_flush<M>();
        } else {
            if (__all_sync(E::gmask(), dead)) return;
#pragma unroll 1
            for (int m = 0; m < M; ++m) {
                cplx nacc[NTX];
                const double nb = E::step(acc, nacc, S_, m, base, g, tab);
                inner<S_ - 1>(nacc, nb, code + (m << (E::BITS * (NTX - 1 - S_))), r01, dead);
            }
        }
    }

    // prefix streams (lane-varying digits taken from p), then the uniform inner levels
    template <int S_, int LEFT>
    __device__ __forceinline__ void prefix(const cplx (&acc)[NTX], double base, int code, int p, cplx r01, bool dead) {
        if constexpr (LEFT == 0) {
            inner<S_>(acc, base, code, r01, dead);
        } else {
            const int m = (p >> (E::BITS * (LEFT - 1))) & (M - 1);
            cplx nacc[NTX];
            const double nb = E::step(acc, nacc, S_, m, base, g, tab);
            prefix<S_ - 1, LEFT - 1>(nacc, nb, code + (m << (E::BITS * (NTX - 1 - S_))), p, r01, dead);
        }
    }
};

// Up to 4 streams, two symbols per warp, one per half-warp (E::G = 16): symbol t = 2 (global warp index) + sub,
// `gl` = lane within the group.  Every phase of a symbol (start-up, prefix rounds, both flush paths, incumbent
// merge, outputs) fits in 16 lanes, so a warp keeps twice the symbols in flight with the same registers per
// thread (4x4 16-QAM: 0.949 -> 0.809 ms per launch).  The halves run independently: they may have different
// live rounds, take different flush paths or collapse; a half without a symbol (odd T_d) leaves at once.
// 5..8 streams: one symbol per warp (E::G = 32), same code.
// (4 CTAs per SM at 128 registers with a few spilled words beat 3 CTAs at 140 registers without: 1.16 vs 1.22 ms)
template <int NTX, int SQM, bool HARD, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, (NTX > 4 ? 2 : 4)) k_enum(Dims d, const double* __restrict__ qr,
                                                     const double* __restrict__ varn,
                                                     const int32_t* __restrict__ active, cplx* __restrict__ stat_m,
                                                     cplx* __restrict__ stat_R, int32_t* __restrict__ kstar,
                                                     double* __restrict__ lse_sym) {
    typedef EnumT<NTX, SQM> E;
    constexpr int M = E::M;
    extern __shared__ __align__(16) double enum_smem[];   // [SPW WARPS][E::WS_DOUBLES]
    const int b = blockIdx.y;
    constexpr int SPW = 32 / E::G;   // symbols per warp
    const int warp = threadIdx.x >> 5, sub = (threadIdx.x & 31) / E::G, gl = E::glane();
    const int t = (blockIdx.x * WARPS + warp) * SPW + sub;
    if (t >= d.T_d) return;
    // the global reads a group starts with -- trial flag, noise variance, the QR record -- are issued together
    // (one after the other they were three DRAM round trips before the first useful instruction, 10 % of the
    // kernel's stall samples in profiles/r02m)
    const double* grec = qr + ((size_t)b * d.T_d + t) * d.rec;
    const int32_t act = (active != nullptr) ? active[b] : 1;
    const double vn = varn[b];
    const double rec0 = (gl < E::REC) ? grec[gl] : 0.0;
    if (act == 0) return;

    double* ws = enum_smem + (size_t)(SPW * warp + sub) * E::WS_DOUBLES;
    cplx* tab = (cplx*)(ws + E::O_TAB);
    double* g = ws + E::O_G;
    // the QR record of the symbol: coalesced loads by the group into the (still idle) flush scratch, then
    // broadcast reads from shared memory (every lane needs all of it; 30+ uniform global loads per lane before)
    const double* rec = ws + E::O_SCR;
    {
        if (gl < E::REC) ws[E::O_SCR + gl] = rec0;
        for (int i = gl + E::G; i < E::REC; i += E::G) ws[E::O_SCR + i] = grec[i];
        __syncwarp(E::gmask());
    }
    cplx yt[NTX];
    cplx r01 = mk(0.0, 0.0);
    double r00;
    {
        cplx Rm[NTX][NTX];
#pragma unroll
        for (int i = 0; i < NTX; ++i)
#pragma unroll
            for (int j = i; j < NTX; ++j) Rm[i][j] = mk(rec[qr_rec_R(NTX, i, j)], rec[qr_rec_R(NTX, i, j) + 1]);
#pragma unroll
        for (int i = 0; i < NTX; ++i) yt[i] = mk(rec[qr_rec_yt(NTX, i)], rec[qr_rec_yt(NTX, i) + 1]);
        r00 = Rm[0][0].x;
        if (NTX > 1) r01 = Rm[0][NTX > 1 ? 1 : 0];
        // tables: R_is * c_m for i<s, and the real PAM levels R_ss * pam_a
#pragma unroll
        for (int s = 1; s < NTX; ++s)
#pragma unroll
            for (int i = 0; i < s; ++i)
                for (int m = gl; m < M; m += E::G) tab[E::pair(i, s) * M + m] = cmul(Rm[i][s], E::cval(m));
        if (gl < SQM) {
#pragma unroll
            for (int s = 0; s < NTX; ++s) g[s * SQM + gl] = Rm[s][s].x * E::pam(gl);
        }
    }
    const double c0 = rec[qr_rec_c0(NTX)];
    const double s2 = vn * vn, inv_s2 = 1.0 / s2;
    if (gl == 0) {
#pragma unroll
        for (int i = 0; i < NTX; ++i) {
            ws[E::O_YT + 2 * i] = yt[i].x;
            ws[E::O_YT + 2 * i + 1] = yt[i].y;
        }
        ws[E::O_C0] = c0;
        ws[E::O_AREF] = 1e300;
        ws[E::O_S2] = inv_s2;
    }
    for (int i = gl; i < E::NACC; i += E::G) ws[E::O_ACC + i] = 0.0;
    __syncwarp(E::gmask());

    Scan<NTX, SQM, HARD> sc;
    sc.ws = ws;
    sc.tab = tab;
    sc.g = g;
    sc.r0 = r00;
    sc.thr = SBCE_THR * s2;
    sc.cnt = 0;
    sc.prune = (d.flags & SBCE_FLAG_FULL_SCAN) == 0;
    // Babai point (successive slicing): a tight upper bound on min d2 -> incumbent
    {
        cplx acc[NTX];
#pragma unroll
        for (int i = 0; i < NTX; ++i) acc[i] = yt[i];
        double base = c0;
        int k = 0;
#pragma unroll
        for (int s = NTX - 1; s >= 0; --s) {
            double dI, dQ;
            const int iI = E::slice(acc[s].x, g + s * SQM, dI), iQ = E::slice(acc[s].y, g + s * SQM, dQ);
            const int m = iQ * SQM + iI;
            base += dI + dQ;
            k += m << (E::BITS * (NTX - 1 - s));
            E::descend(acc, acc, s, m, tab);
        }
        sc.best = base;
        sc.bestk = k;
        sc.lim = HARD ? base : base + sc.thr;
    }

    // Top-level pre-pass (prefixes of two or more streams): lane m tests the FIRST prefix stream's symbol m against
    // the Babai bound once.  A round of 16 prefixes whose top symbols are all dead would only compute its prefix
    // levels to find every lane dead; it is dropped from the group's list of live rounds (16-QAM on 3+ streams and
    // QPSK on 4+: one top symbol per round).  Dead under the initial bound implies dead under any later (tighter)
    // one, and a dead round contributes nothing in either mode, so the sequence of visited live nodes -- hence
    // the queue order and every output bit -- is unchanged (Scan::packed for the levels below the prefixes).
    constexpr int NROUND = (E::NPREF + E::G - 1) / E::G;
    static_assert(NROUND <= 32, "one bit per round");
    unsigned live = NROUND == 32 ? 0xffffffffu : (1u << NROUND) - 1u;
    if (E::PL >= 2 && sc.prune) {
        constexpr int TOP_SHIFT = E::BITS * (E::PL - 1);
        const bool a = gl < M && !(c0 + E::dist(yt, NTX - 1, gl, g) > sc.lim);
        const unsigned top_alive = __ballot_sync(E::gmask(), a) >> E::gshift();   // this group's bits
        live = 0u;
#pragma unroll
        for (int r = 0; r < NROUND; ++r) {
            const int lo = (E::G * r) >> TOP_SHIFT, hi = min(E::G * r + E::G - 1, E::NPREF - 1) >> TOP_SHIFT;
            const unsigned bits = ((2u << hi) - 1u) & ~((1u << lo) - 1u);   // hi < M <= 16
            if (top_alive & bits) live |= 1u << r;
        }
    }
    // The group walks its live rounds in increasing order.  Iteration j of both halves of a warp is their j-th
    // live round, so two symbols with as many live rounds (at operating SNRs: one each) walk their prefixes in
    // step; skipping dead rounds in place would leave the halves in different iterations, one after the other.
    // All lanes of the group iterate the same prefixes (invalid ones carry an infinite partial distance).
    while (live != 0u) {
        const int pb = E::G * (__ffs(live) - 1);
        live &= live - 1u;
        const int p = pb + gl;
        const bool valid = p < E::NPREF;
        // ytilde and c0 come from the shared block: held in registers across the walk, they spilled
        cplx acc[NTX];
#pragma unroll
        for (int i = 0; i < NTX; ++i) acc[i] = mk(ws[E::O_YT + 2 * i], ws[E::O_YT + 2 * i + 1]);
        sc.template prefix<NTX - 1, E::PL>(acc, ws[E::O_C0], 0, valid ? p : 0, r01, !valid);
    }

    sc.merge_best();
    const double best = sc.best;
    const int bestk = sc.bestk;
    const size_t sidx = (size_t)b * d.T_d + t;
    if (kstar != nullptr && gl == 0) kstar[sidx] = bestk;

    bool collapsed = HARD;
    double S = 0.0;
    if (!HARD) {
        enum_flush<NTX, SQM>(ws, best, sc.cnt);
        S = ws[E::O_ACC];
        // Nothing within 64 varn^2 of the incumbent was queued: only happens when |d2| is so large that
        // its rounding error exceeds the window (e.g. a garbage start vector of norm 1e13); every weight
        // but the best one underflows, so the posterior is the one-hot at k*.
        if (!(S > 0.0) || !isfinite(S)) collapsed = true;
    }
    if (collapsed) {
        if (gl == 0) {
            cplx xs[NTX];
#pragma unroll
            for (int s = 0; s < NTX; ++s) xs[s] = E::cval(E::digit(bestk, s));
#pragma unroll
            for (int i = 0; i < NTX; ++i) {
                stat_m[sidx * NTX + i] = cconj(xs[i]);
#pragma unroll
                for (int j = 0; j < NTX; ++j) stat_R[(sidx * NTX + i) * NTX + j] = cmulc(xs[j], xs[i]);
            }
            if (lse_sym != nullptr) lse_sym[sidx] = -best * inv_s2;
        }
        return;
    }
    // outputs: lane l < n_tx^2 writes R[i][j] with (i, j) = (l / n_tx, l % n_tx) (l += 16), lane j < n_tx writes
    // m[j] -- coalesced stores (lane 0 alone issued all n_tx + n_tx^2 of them one after the other before)
    {
        const double invS = 1.0 / S;
        const double* A = ws + E::O_ACC;
        for (int l = gl; l < NTX * NTX; l += E::G) {
            const int i = l / NTX, j = l % NTX;
            cplx v;
            if (i == j) {
                v = mk(A[E::A_RD + j] * invS, 0.0);
            } else {
                const int pr = E::acc_R(min(i, j), max(i, j));
                const double a = A[pr] * invS, c = A[pr + 1] * invS;
                v = mk(a, i < j ? c : -c);
            }
            stat_R[sidx * NTX * NTX + l] = v;
        }
        if (gl < NTX) stat_m[sidx * NTX + gl] = mk(A[E::A_MRE + gl] * invS, A[E::A_MIM + gl] * invS);
        if (lse_sym != nullptr && gl == 0) lse_sym[sidx] = -ws[E::O_AREF] * inv_s2 + log(S);
    }
}

// ---------------------------------------------------------------------------
// superimposed pilots: statistics of x~ = x + o from those of x
//   m~_i = m_i + conj(o_i),   R~_ij = R_ij + m_i o_j + conj(o_i) conj(m_j) + conj(o_i) o_j
// ---------------------------------------------------------------------------
__global__ void k_superimpose_stats(Dims d, int nb, const cplx* __restrict__ Xoff, const int32_t* __restrict__ active,
                                    cplx* __restrict__ stat_m, cplx* __restrict__ stat_R) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;   // flat (b, t)
    if (s >= nb * d.T_d) return;
    if (active != nullptr && active[s / d.T_d] == 0) return;
    const int n = d.n_tx;
    const cplx* o = Xoff + (size_t)s * n;
    cplx* m = stat_m + (size_t)s * n;
    cplx* R = stat_R + (size_t)s * n * n;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            cplx v = R[i * n + j];
            cfma(v, m[i], o[j]);
            v = cadd(v, cconj(cmul(o[i], m[j])));
            v = cadd(v, cmulc(o[j], o[i]));   // conj(o_i) o_j
            R[i * n + j] = v;
        }
    for (int i = 0; i < n; ++i) m[i] = cadd(m[i], cconj(o[i]));
}

cudaError_t launch_superimpose_stats(const Dims& d, int nb, const double* Xoff, const int32_t* active, double* stat_m,
                                     double* stat_R, cudaStream_t s) {
    const int total = nb * d.T_d;
    k_superimpose_stats<<<(total + 127) / 128, 128, 0, s>>>(d, nb, (const cplx*)Xoff, active, (cplx*)stat_m, (cplx*)stat_R);
    count_launch();
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// dispatch
// ---------------------------------------------------------------------------
template <int NTX, int NRX>
static cudaError_t run_heff(const Dims& d, int nb, const double* Yd, const double* PsiD, const double* theta,
                            const int32_t* active, const double* Xoff, double* qr, cudaStream_t s) {
    static SmemOptIn optin_mma, optin;
    dim3 grid((d.T_d + 127) / 128, nb);
    // tensor path once the contraction is a real GEMM: at least one full 8-column tile and two 8-deep steps
    constexpr int NC = NTX * NRX, NT = (NC + 7) / 8;
    const int KP = (d.N1 + 7) & ~7;
    const size_t smem_mma = sizeof(cplx) * ((size_t)KP * (NT * 8 + 2) + 4 * 32 * (NC + 1));
    if (NC >= 8 && d.N1 >= 16 && smem_mma <= 100 * 1024) {
        cudaError_t e = opt_in_smem(optin_mma, (const void*)k_heff_qr_mma<NTX, NRX>, smem_mma);
        if (e != cudaSuccess) return e;
        k_heff_qr_mma<NTX, NRX><<<grid, 128, smem_mma, s>>>(d, (const cplx*)Yd, (const cplx*)PsiD, (const cplx*)theta,
                                                            active, (const cplx*)Xoff, qr);
        count_launch();
        return cudaGetLastError();
    }
    size_t smem = sizeof(cplx) * (size_t)d.L * NRX;
    const int use_smem = smem <= 64 * 1024;
    if (!use_smem) smem = 0;
    cudaError_t e = opt_in_smem(optin, (const void*)k_heff_qr<NTX, NRX>, smem);
    if (e != cudaSuccess) return e;
    k_heff_qr<NTX, NRX><<<grid, 128, smem, s>>>(d, (const cplx*)Yd, (const cplx*)PsiD, (const cplx*)theta, active,
                                                (const cplx*)Xoff, qr, use_smem);
    count_launch();
    return cudaGetLastError();
}

template <int NTX>
static cudaError_t run_heff_ntx(const Dims& d, int nb, const double* Yd, const double* PsiD, const double* theta,
                                const int32_t* active, const double* Xoff, double* qr, cudaStream_t s) {
    switch (d.n_rx) {
        case 1: return run_heff<NTX, 1>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 2: return run_heff<NTX, 2>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 3: return run_heff<NTX, 3>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 4: return run_heff<NTX, 4>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 6: return run_heff<NTX, 6>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 8: return run_heff<NTX, 8>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        default: return cudaErrorInvalidValue;
    }
}

template <int NTX, int SQM>
static cudaError_t run_enum_sqm(const Dims& d, int nb, const double* qr, const double* varn, const int32_t* active,
                                double* stat_m, double* stat_R, int32_t* kstar, double* lse_sym, cudaStream_t s) {
    typedef EnumT<NTX, SQM> E;
    constexpr int WARPS = 4, SYMS = WARPS * 32 / E::G;   // symbols per CTA
    dim3 grid((d.T_d + SYMS - 1) / SYMS, nb);
    constexpr size_t smem = sizeof(double) * SYMS * E::WS_DOUBLES;
    static SmemOptIn optin[2];   // one per kernel: [hard]
    const bool hard = d.mode == SBCE_MODE_HARD;
    const auto kernel = hard ? k_enum<NTX, SQM, true, WARPS> : k_enum<NTX, SQM, false, WARPS>;
    cudaError_t e = opt_in_smem(optin[hard], (const void*)kernel, smem);
    if (e != cudaSuccess) return e;
    kernel<<<grid, WARPS * 32, smem, s>>>(d, qr, varn, active, (cplx*)stat_m, (cplx*)stat_R, kstar, lse_sym);
    count_launch();
    return cudaGetLastError();
}

template <int NTX>
static cudaError_t run_enum(const Dims& d, int nb, const double* qr, const double* varn, const int32_t* active,
                            double* stat_m, double* stat_R, int32_t* kstar, double* lse_sym, cudaStream_t s) {
    switch (d.sqM) {   // enum_instantiated takes log2 M
        case 2:
            if constexpr (enum_instantiated(NTX, 2))
                return run_enum_sqm<NTX, 2>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
            break;
        case 4:
            if constexpr (enum_instantiated(NTX, 4))
                return run_enum_sqm<NTX, 4>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
            break;
        case 8:
            if constexpr (enum_instantiated(NTX, 6))
                return run_enum_sqm<NTX, 8>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
            break;
    }
    return cudaErrorInvalidValue;
}

template <int NTX>
static cudaError_t run_heff_rows(const Dims& d, int nb, const double* Yd, const double* PsiD, const double* theta,
                                 const int32_t* active, const double* Xoff, double* qr, cudaStream_t s) {
    dim3 grid((d.T_d + 15) / 16, nb);   // 8 lanes per symbol, 16 symbols per CTA
    k_heff_qr_rows<NTX><<<grid, 128, 0, s>>>(d, (const cplx*)Yd, (const cplx*)PsiD, (const cplx*)theta, active,
                                             (const cplx*)Xoff, qr);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_heff_qr(const Dims& d, int nb, const double* Yd, const double* PsiD, const double* theta,
                           const int32_t* active, const double* Xoff, double* qr, cudaStream_t s) {
    switch (d.n_tx) {
        case 1: return run_heff_ntx<1>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 2: return run_heff_ntx<2>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 3: return run_heff_ntx<3>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 4: return run_heff_ntx<4>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 5: return run_heff_rows<5>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 6: return run_heff_rows<6>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 7: return run_heff_rows<7>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        case 8: return run_heff_rows<8>(d, nb, Yd, PsiD, theta, active, Xoff, qr, s);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_enum(const Dims& d, int nb, const double* qr, const double* varn, const int32_t* active,
                        double* stat_m, double* stat_R, int32_t* kstar, double* lse_sym, cudaStream_t s) {
    switch (d.n_tx) {
        case 1: return run_enum<1>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
        case 2: return run_enum<2>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
        case 3: return run_enum<3>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
        case 4: return run_enum<4>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
        case 5: return run_enum<5>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
        case 6: return run_enum<6>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
        case 7: return run_enum<7>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
        case 8: return run_enum<8>(d, nb, qr, varn, active, stat_m, stat_R, kstar, lse_sym, s);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace sbce
