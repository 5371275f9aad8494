// M-step of the semi-blind EM estimator: weighted least squares for the channel.
//
// Reference semantics (/root/reference/Proposed_method_NMSEvsTp.py:61-66):
//   denom = sum_p Z_p^H Z_p + sum_{t,k} beta Z^H Z      (D x D, D = L*n_rx)
//   numer = sum_p Z_p^H y_p + sum_{t,k} beta Z^H y_t    (D)
//   theta = np.linalg.solve(denom, numer)
// With Z = (psi~^T (x) x^T) (x) I_nrx every Z^H Z is (w^* w^T) (x) I_nrx, so the
// system is  (G (x) I) theta = vec(B)  with the L x L Hermitian
//   G = sum_t (psi~_t^* psi~_t^T) (x) R_t ,   B = sum_t (psi~_t^* (x) m_t) y_t^T   (L x n_rx)
// (pilots: R = conj(x) x^T, m = conj(x)).  SURVEY.md section 8a-6.
//
// B200 design:
//  * Gram: the Kronecker / Khatri-Rao structure is applied by index arithmetic.  One (n >= n') pair of
//    RIS indices owns the whole n_tx x n_tx block  sum_t conj(psi[t,n]) psi[t,n'] R_t ; because R_t is
//    Hermitian its 2 n_tx^2 real accumulators are [p_r ; p_i] (2 x T) times a real (T x n_tx^2) matrix
//    built from diag(R_t) and the upper entries, i.e. the whole Gram is ONE real GEMM that runs on the
//    FP64 tensor path (k_gram_tma4 for n_tx = 4, k_gram_mma<NTX> for n_tx = 5..8 and long rows; scalar
//    k_gram<NTX> below 4).  Only the lower triangle is produced.  The last CTA of each trial writes B^H as extra
//    rows below the matrix, and the padding.
//  * k_chol: one CTA per trial, LEFT-looking blocked complex Cholesky (panel width 16) on the augmented
//    lower trapezoid [G ; B^H], panel updates and the triangular solve as DMMA products; the B^H rows
//    come out as (C^-1 B)^H for free, so only the back substitution C^H theta = z remains.  A
//    non-positive pivot flags the trial (status bit) instead of poisoning the batch.
#include <math.h>

#include "common.cuh"
#include "tensor.cuh"

namespace sbce {

// ---------------------------------------------------------------------------
// Gram + right-hand side
// ---------------------------------------------------------------------------
constexpr int GR_THREADS = 256;
constexpr int GR_TC = 16;  // symbols per shared-memory chunk (default; shrunk at launch for very long psi rows)


// The last CTA of every trial: right-hand side rows B^H stored under the matrix,
//   row Lp + r, column l = n*n_tx + i :  conj(B[l][r]) = sum_t psi[t,n] conj(m_t[i] y_t[r]),
// plus the identity padding of the trapezoid.  With Zc[t][i n_rx + r] = conj(m_t[i] y_t[r]) this is the complex
// GEMM  Out (N+1 x n_tx n_rx) = Psi^T (N+1 x T) . Zc (T x n_tx n_rx)  and runs on the FP64 tensor path: a warp owns
// one 16-row tile of RIS indices and two 8-column tiles; psi and Zc chunks are staged in shared memory (Zc rows
// padded by two elements: conflict-free B fragments).  Its scalar predecessor -- one thread per column l, n_rx
// complex accumulators, 5 shared loads per 4 complex FMAs -- executed 23 % of the Gram kernel's instructions
// and held 21 % of its resident warp time (profiles/r02d) for 5 % of its arithmetic.
template <int NTX>
__device__ __forceinline__ void gram_rhs_cta(const Dims& d, int T, int b, cplx* sPsi, cplx* /*unused*/, const cplx* psi_b,
                                             const cplx* __restrict__ Y, const cplx* __restrict__ sm, const cplx* Gi,
                                             cplx* Gb) {
    const int N1 = d.N1, n_rx = d.n_rx;
    const int NC = NTX * n_rx;              // complex columns (i, r) -> i * n_rx + r
    const int ZS = NC + 2;                  // padded row stride of the staged Zc
    unsigned dyn_bytes;
    asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn_bytes));
    // chunk length: as many symbols as the CTA's dynamic shared memory holds (the pair CTAs of the same launch
    // size it for their operand ring), a multiple of 8 (one MMA k-step), at most 128
    int TCR = (int)(dyn_bytes / (sizeof(cplx) * (N1 + ZS)));
    TCR = max(8, min(TCR & ~7, 128));
    cplx* sZ = sPsi + (size_t)TCR * N1;
    const cplx* m_b = sm + (size_t)b * T * NTX;
    const cplx* y_b = Y + (size_t)b * T * n_rx;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
    const int MT = (N1 + 15) >> 4, NTP = (NC + 15) >> 4;       // 16-row tiles, pairs of 8-column tiles
    const int units = MT * NTP;
    constexpr int NWARP = GR_THREADS / 32;
    for (int u0 = 0; u0 < units; u0 += NWARP) {
        const int u = u0 + warp;
        const bool live = u < units;                            // warp-uniform
        const int mt = live ? u / NTP : 0, np = live ? u % NTP : 0;
        const int n0 = mt * 16, c0 = np * 16;
        const int ra = min(n0 + g, N1 - 1), rb = min(n0 + g + 8, N1 - 1);     // clamped RIS rows (results discarded)
        double cr[2][4], ci[2][4];
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) { cr[j][e] = 0.0; ci[j][e] = 0.0; }
        for (int t0 = 0; t0 < T; t0 += TCR) {
            const int tc = min(TCR, T - t0);
            const int tc8 = (tc + 7) & ~7;
            __syncthreads();
            for (int e = threadIdx.x; e < tc8 * N1; e += GR_THREADS)
                sPsi[e] = (e < tc * N1) ? psi_b[(size_t)t0 * N1 + e] : mk(0.0, 0.0);
            for (int e = threadIdx.x; e < tc8 * ZS; e += GR_THREADS) {
                const int tt = e / ZS, c = e % ZS;
                cplx v = mk(0.0, 0.0);
                if (tt < tc && c < NC) {
                    const int ii = c / n_rx, r = c % n_rx;
                    v = cconj(cmul(m_b[(size_t)(t0 + tt) * NTX + ii], y_b[(size_t)(t0 + tt) * n_rx + r]));
                }
                sZ[e] = v;
            }
            __syncthreads();
            if (live) {
                for (int ks = 0; ks < tc8; ks += 8) {
                    const cplx* pl = sPsi + (size_t)(ks + tig) * N1;
                    const cplx* ph = sPsi + (size_t)(ks + tig + 4) * N1;
                    // A fragment order: (row g, k lo), (row g+8, k lo), (row g, k hi), (row g+8, k hi)
                    const cplx a0 = pl[ra], a1 = pl[rb], a2 = ph[ra], a3 = ph[rb];
                    const double ar[4] = {a0.x, a1.x, a2.x, a3.x};
                    const double ai[4] = {a0.y, a1.y, a2.y, a3.y};
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int c = min(c0 + 8 * j + g, ZS - 1);           // columns >= NC hold zeros
                        const cplx b0 = sZ[(size_t)(ks + tig) * ZS + c], b1 = sZ[(size_t)(ks + tig + 4) * ZS + c];
                        // (ar + i ai)(br + i bi): re += ar br - ai bi ; im += ar bi + ai br
                        dmma16x8x8(cr[j], ar, b0.x, b1.x);
                        dmma16x8x8(ci[j], ar, b0.y, b1.y);
                        dmma16x8x8(cr[j], ai, -b0.y, -b1.y);
                        dmma16x8x8(ci[j], ai, b0.x, b1.x);
                    }
                }
            }
        }
        if (live) {
            // accumulator (row g + 8h, columns 8 j + 2 tig, + 1) -> G[(Lp + r) * Lp + n * NTX + i]
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int h = 0; h < 2; ++h)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int n = n0 + g + 8 * h, c = c0 + 8 * j + 2 * tig + e;
                        if (n < N1 && c < NC) {
                            const int ii = c / n_rx, r = c % n_rx;
                            const size_t o = (size_t)(d.Lp + r) * d.Lp + (n * NTX + ii);
                            cplx v = mk(cr[j][2 * h + e], ci[j][2 * h + e]);
                            if (Gi) v = cadd(v, Gi[o]);
                            Gb[o] = v;
                        }
                    }
        }
    }
    // padding: identity on the padded diagonal rows L..Lp-1, zero padded columns / rows of B^H
    const int padrows = (d.Lp - d.L) + d.RP;
    for (int e = threadIdx.x; e < padrows * d.Lp; e += GR_THREADS) {
        const int pr = e / d.Lp, c = e % d.Lp;
        if (pr < d.Lp - d.L) {
            const int row = d.L + pr;
            Gb[(size_t)row * d.Lp + c] = (c == row) ? mk(1.0, 0.0) : mk(0.0, 0.0);
        } else {
            const int r = pr - (d.Lp - d.L);
            if (r >= d.n_rx || c >= d.L) Gb[(size_t)(d.Lp + r) * d.Lp + c] = mk(0.0, 0.0);
        }
    }
}

// CTAs 0 .. nP-1: one thread per lower-triangular (n >= n') pair of RIS indices.
// CTA nP (the last one of a trial): the right-hand side rows B^H stored under the matrix,
//   row Lp + r, column l = n*n_tx + i :  conj(B[l][r]) = sum_t psi[t,n] conj(m_t[i] y_t[r]),
// one thread per column l with n_rx accumulators, plus the identity padding of the trapezoid.
// Both kinds of CTA stage the same psi chunks in shared memory.
template <int NTX>
__global__ void __launch_bounds__(GR_THREADS, 2) k_gram(Dims d, int T, int TC, const cplx* __restrict__ Psi,
                                                     const cplx* __restrict__ sR, const cplx* __restrict__ Y,
                                                     const cplx* __restrict__ sm, const cplx* __restrict__ Ginit,
                                                     cplx* __restrict__ Gout, const int32_t* __restrict__ active) {
    extern __shared__ double2 gsm[];
    const int b = blockIdx.y;
    if (active != nullptr && active[b] == 0) return;
    const int N1 = d.N1;
    const int P = N1 * (N1 + 1) / 2;
    cplx* sPsi = gsm;            // [TC][N1]
    cplx* sRr = sPsi + TC * N1;  // [TC][NTX*NTX]  (rhs CTA: sized from the dynamic shared memory it finds)
    const cplx* psi_b = Psi + (size_t)(d.psi_shared ? 0 : b) * T * N1;
    const size_t gstride = (size_t)d.Ltot * d.Lp;
    cplx* Gb = Gout + (size_t)b * gstride;
    const cplx* Gi = Ginit ? Ginit + (size_t)b * gstride : nullptr;

    if (blockIdx.x == gridDim.x - 1) {
        gram_rhs_cta<NTX>(d, T, b, sPsi, sRr, psi_b, Y, sm, Gi, Gb);
        return;
    }

    const int item = blockIdx.x * GR_THREADS + threadIdx.x;
    const bool is_pair = item < P;
    int n = 0, np = 0;
    if (is_pair) {
        n = (int)((sqrtf(8.0f * (float)item + 1.0f) - 1.0f) * 0.5f);   // the two loops below make it exact
        while ((n + 1) * (n + 2) / 2 <= item) ++n;
        while (n * (n + 1) / 2 > item) --n;
        np = item - n * (n + 1) / 2;
    }

    // R_t is Hermitian: only its real diagonal and its upper triangle are used.  For i<j the two block
    // entries  acc[i][j] += p R_ij  and  acc[j][i] += p conj(R_ij)  share their four real products, so we
    // accumulate U = sum pr Rr, V = sum pi Ri, W = sum pr Ri, Z = sum pi Rr (4 FMAs instead of 8) and
    // combine at the end:  acc[i][j] = (U - V, W + Z),  acc[j][i] = (U + V, Z - W).
    constexpr int NPAIR = NTX * (NTX - 1) / 2;
    constexpr int NPAIR1 = NPAIR > 0 ? NPAIR : 1;
    double dg_re[NTX], dg_im[NTX];
    double U[NPAIR1], V[NPAIR1], W[NPAIR1], Z[NPAIR1];
#pragma unroll
    for (int i = 0; i < NTX; ++i) { dg_re[i] = 0.0; dg_im[i] = 0.0; }
#pragma unroll
    for (int q = 0; q < NPAIR1; ++q) { U[q] = 0.0; V[q] = 0.0; W[q] = 0.0; Z[q] = 0.0; }

    const cplx* R_b = sR + (size_t)b * T * NTX * NTX;
    // two-stage cp.async pipeline: chunk c+1 streams into the other buffer while chunk c is consumed
    const int stage_elems = TC * (N1 + NTX * NTX);      // complex elements per stage
    auto issue = [&](int chunk, int buf) {
        const int t0 = chunk * TC;
        const int tc = min(TC, T - t0);
        cplx* dpsi = gsm + buf * stage_elems;
        cplx* dR = dpsi + TC * N1;
        const cplx* spsi = psi_b + (size_t)t0 * N1;
        const cplx* sRg = R_b + (size_t)t0 * NTX * NTX;
        for (int e = threadIdx.x; e < tc * N1; e += GR_THREADS) cp_async16(dpsi + e, spsi + e);
        for (int e = threadIdx.x; e < tc * NTX * NTX; e += GR_THREADS) cp_async16(dR + e, sRg + e);
        cp_async_commit();
    };
    const int nchunk = (T + TC - 1) / TC;
    if (nchunk > 0) issue(0, 0);
    for (int ck = 0; ck < nchunk; ++ck) {
        const int buf = ck & 1;
        if (ck + 1 < nchunk) { issue(ck + 1, buf ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
        __syncthreads();
        const int tc = min(TC, T - ck * TC);
        const cplx* cPsi = gsm + buf * stage_elems;
        const cplx* cR = cPsi + TC * N1;
        if (is_pair) {
#pragma unroll 4
            for (int tt = 0; tt < tc; ++tt) {
                const cplx a = cPsi[tt * N1 + n];
                const cplx c = cPsi[tt * N1 + np];
                const cplx p = cmulc(c, a);  // conj(psi[t,n]) psi[t,n']
                const cplx* Rt = cR + tt * NTX * NTX;
#pragma unroll
                for (int i = 0; i < NTX; ++i) {
                    const double r = Rt[i * NTX + i].x;
                    dg_re[i] = fma(p.x, r, dg_re[i]);
                    dg_im[i] = fma(p.y, r, dg_im[i]);
                }
#pragma unroll
                for (int i = 0; i < NTX; ++i)
#pragma unroll
                    for (int j = i + 1; j < NTX; ++j) {
                        const int q = i * NTX - i * (i + 1) / 2 + (j - i - 1);
                        const cplx r = Rt[i * NTX + j];
                        U[q] = fma(p.x, r.x, U[q]);
                        V[q] = fma(p.y, r.y, V[q]);
                        W[q] = fma(p.x, r.y, W[q]);
                        Z[q] = fma(p.y, r.x, Z[q]);
                    }
            }
        }
        __syncthreads();  // everyone is done with this buffer before it is refilled (chunk ck+2)
    }
    if (is_pair) {
        auto put = [&](int i, int j, cplx v) {
            const size_t o = (size_t)(n * NTX + i) * d.Lp + (np * NTX + j);
            if (Gi) v = cadd(v, Gi[o]);
            Gb[o] = v;
        };
#pragma unroll
        for (int i = 0; i < NTX; ++i) put(i, i, mk(dg_re[i], dg_im[i]));
#pragma unroll
        for (int i = 0; i < NTX; ++i)
#pragma unroll
            for (int j = i + 1; j < NTX; ++j) {
                const int q = i * NTX - i * (i + 1) / 2 + (j - i - 1);
                put(i, j, mk(U[q] - V[q], W[q] + Z[q]));
                put(j, i, mk(U[q] + V[q], Z[q] - W[q]));
            }
    }
}

// ---------------------------------------------------------------------------
// Gram on the FP64 tensor path, n_tx = 4.
// With the Hermitian product sharing above, the 32 real accumulators of a RIS pair are
//   [pr ; pi] (2 x T)  times  Bmat (T x 16 real columns = [Rd0..Rd3, (Rr,Ri) of the 6 upper entries]),
// i.e. the whole Gram is ONE real GEMM with M = 2 x (number of pairs), N = 16, K = T whose A operand
// p_t = conj(psi[t,n]) psi[t,n'] is generated on the fly into the mma.m16n8k8 fragment layout from the
// staged psi chunk.  A warp owns two 16-pair tiles; per 8 symbols it issues 8 MMAs (= 32 DMMA.8x8x4)
// against 20 shared-memory loads, so the kernel is bound by the FP64 pipe, not by shared memory.
// B-matrix column -> double offset inside the raw 4x4 complex R_t (row-major, interleaved):
__device__ __forceinline__ int gram_bcol_offset(int col) {
    // cols 0..3: real diagonal (i,i) ; cols 4+2q, 5+2q: re, im of the q-th upper entry (0,1)(0,2)(0,3)(1,2)(1,3)(2,3)
    const int up[6] = {1, 2, 3, 6, 7, 11};  // 4*i + j
    if (col < 4) return 2 * (5 * col);
    const int q = (col - 4) >> 1;
    return 2 * up[q] + ((col - 4) & 1);
}

// ---------------------------------------------------------------------------
// k_gram_tma4: the FP64 tensor-path Gram fed by the TMA engine.  (A cp.async double-buffered predecessor spent
// only half of its warp time in the DMMA loop, profiles/r01h: 9 % issuing ~10 cp.async per thread and
// chunk, 7 % at the two CTA barriers per chunk that couple all eight warps, 15 % in the epilogue.)  The
// staged operands are CONTIGUOUS in global memory -- 16 symbols of psi ([16][N+1] complex) and of R_t
// ([16][16] complex) -- so one elected lane of a producer warp moves each chunk with two 1-D bulk copies
// (cp.async.bulk ... mbarrier::complete_tx) into a 4-stage ring; the eight DMMA warps never touch the
// staging: each waits on the stage's `full` mbarrier, runs its DMMAs and arrives on `empty` on its own
// -- no __syncthreads in the loop, so a slow warp no longer stalls the other seven.
// ---------------------------------------------------------------------------
constexpr int GT_TC = 16;        // symbols per stage
constexpr int GT_STAGES = 4;     // ring depth
constexpr int GT_THREADS = GR_THREADS;        // 8 DMMA warps; warp 0's elected lane also drives the TMA ring

__global__ void __launch_bounds__(GT_THREADS, 2) k_gram_tma4(Dims d, int T, const cplx* __restrict__ Psi,
                                                            const cplx* __restrict__ sR, const cplx* __restrict__ Y,
                                                            const cplx* __restrict__ sm, const cplx* __restrict__ Ginit,
                                                            cplx* __restrict__ Gout, const int32_t* __restrict__ active) {
    constexpr int NTX = 4;
    extern __shared__ __align__(128) double2 gsm[];
    __shared__ __align__(8) unsigned long long bar_full[GT_STAGES], bar_empty[GT_STAGES];
    const int b = blockIdx.y;
    if (active != nullptr && active[b] == 0) return;
    const int N1 = d.N1;
    const int P = N1 * (N1 + 1) / 2;
    const cplx* psi_b = Psi + (size_t)(d.psi_shared ? 0 : b) * T * N1;
    const size_t gstride = (size_t)d.Ltot * d.Lp;
    cplx* Gb = Gout + (size_t)b * gstride;
    const cplx* Gi = Ginit ? Ginit + (size_t)b * gstride : nullptr;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
    if (blockIdx.x == gridDim.x - 1) {
        gram_rhs_cta<NTX>(d, T, b, gsm, gsm + GR_TC * N1, psi_b, Y, sm, Gi, Gb);
        return;
    }
    const int stage_elems = GT_TC * (N1 + NTX * NTX);   // complex elements per stage: [TC][N1] psi, [TC][16] R
    const cplx* R_b = sR + (size_t)b * T * NTX * NTX;
    const int nchunk = (T + GT_TC - 1) / GT_TC;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < GT_STAGES; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], GR_THREADS / 32); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // producer: fills stage (ck % STAGES) with chunk ck; executed by warp 0 (all lanes for the ragged
    // zero fill, the elected lane for the barrier and the two bulk copies)
    auto produce = [&](int ck) {
        const int s = ck % GT_STAGES;
        const int t0 = ck * GT_TC;
        const int tc = min(GT_TC, T - t0);
        cplx* dpsi = gsm + s * stage_elems;
        cplx* dR = dpsi + GT_TC * N1;
        if (tc < GT_TC) {   // ragged last chunk: symbols beyond T contribute zero
            for (int e = tc * N1 + lane; e < GT_TC * N1; e += 32) dpsi[e] = mk(0.0, 0.0);
            for (int e = tc * NTX * NTX + lane; e < GT_TC * NTX * NTX; e += 32) dR[e] = mk(0.0, 0.0);
            __syncwarp();
        }
        if (lane == 0) {
            const unsigned bpsi = (unsigned)(tc * N1 * sizeof(cplx)), bR = (unsigned)(tc * NTX * NTX * sizeof(cplx));
            mbar_expect_tx(&bar_full[s], bpsi + bR);
            tma_bulk_g2s(dpsi, psi_b + (size_t)t0 * N1, bpsi, &bar_full[s]);
            tma_bulk_g2s(dR, R_b + (size_t)t0 * NTX * NTX, bR, &bar_full[s]);
        }
        __syncwarp();
    };
    if (warp == 0)
        for (int ck = 0; ck < min(GT_STAGES, nchunk); ++ck) produce(ck);

    // ---------------- DMMA warps: pairs of this lane: tile u (0,1), row half h (0,1) -> item
    int pn[2][2], pnp[2][2];
    bool pv[2][2], tile_live[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        tile_live[u] = (blockIdx.x * GR_THREADS + (2 * warp + u) * 16) < P;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int item = blockIdx.x * GR_THREADS + (2 * warp + u) * 16 + g + 8 * h;
            pv[u][h] = item < P;
            item = min(item, P - 1);
            int n = (int)((sqrtf(8.0f * (float)item + 1.0f) - 1.0f) * 0.5f);   // made exact by the loops below
            while ((n + 1) * (n + 2) / 2 <= item) ++n;
            while (n * (n + 1) / 2 > item) --n;
            pn[u][h] = n;
            pnp[u][h] = item - n * (n + 1) / 2;
        }
    }
    const int boff0 = gram_bcol_offset(g), boff1 = gram_bcol_offset(8 + g);
    // The accumulators START from the pilot part G_p instead of adding it in the epilogue: its loads are issued
    // here, before the first wait on the operand ring, where their latency is hidden behind the TMA prologue
    // (in the epilogue they were 8 % of the kernel's stall samples, profiles/r02d).  An upper pair (i<j) is kept
    // as U = sum pr Rr, W = sum pr Ri, Z = sum pi Rr, V = sum pi Ri with out_ij = (U - V, W + Z) and
    // out_ji = (U + V, Z - W): starting from U = (a.x + b.x)/2, V = (b.x - a.x)/2, W = (a.y - b.y)/2,
    // Z = (a.y + b.y)/2 yields a = G_p[ij], b = G_p[ji] (to one rounding of the larger of the two).
    double accr[2][2][4], acci[2][2][4];  // [tile][n-tile][c0..c3]
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const bool on = Gi != nullptr && pv[u][h];
            const cplx* gp = on ? Gi + (size_t)(pn[u][h] * NTX) * d.Lp + pnp[u][h] * NTX : nullptr;
            auto gi = [&](int i, int j) { return on ? gp[(size_t)i * d.Lp + j] : mk(0.0, 0.0); };
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const int col = 8 * nt + 2 * tig;
                double r0, r1, i0, i1;
                if (col < 4) {
                    const cplx a = gi(col, col), c2 = gi(col + 1, col + 1);
                    r0 = a.x; i0 = a.y; r1 = c2.x; i1 = c2.y;
                } else {
                    const int q = (col - 4) >> 1;
                    const int qi = (q < 3) ? 0 : (q < 5 ? 1 : 2);
                    const int qj = (q < 3) ? q + 1 : (q < 5 ? q - 1 : 3);
                    const cplx a = gi(qi, qj), c2 = gi(qj, qi);
                    r0 = 0.5 * (a.x + c2.x); i1 = 0.5 * (c2.x - a.x); r1 = 0.5 * (a.y - c2.y); i0 = 0.5 * (a.y + c2.y);
                }
                accr[u][nt][2 * h] = r0; accr[u][nt][2 * h + 1] = r1;
                acci[u][nt][2 * h] = i0; acci[u][nt][2 * h + 1] = i1;
            }
        }

    for (int ck = 0; ck < nchunk; ++ck) {
        const int s = ck % GT_STAGES;
        // refill the stage of the PREVIOUS chunk (three chunks of look-ahead): by now the other warps have
        // almost always released it, so the wait on its `empty` barrier rarely blocks warp 0
        if (warp == 0 && ck >= 1 && ck - 1 + GT_STAGES < nchunk) {
            mbar_wait(&bar_empty[(ck - 1) % GT_STAGES], ((ck - 1) / GT_STAGES) & 1);
            produce(ck - 1 + GT_STAGES);
        }
        mbar_wait(&bar_full[s], (ck / GT_STAGES) & 1);
        const cplx* cPsi = gsm + s * stage_elems;
        const double* cR = (const double*)(cPsi + GT_TC * N1);
#pragma unroll
        for (int ks = 0; ks < GT_TC / 8; ++ks) {
            const int tlo = ks * 8 + tig, thi = tlo + 4;
            const double b00 = cR[tlo * 32 + boff0], b01 = cR[thi * 32 + boff0];
            const double b10 = cR[tlo * 32 + boff1], b11 = cR[thi * 32 + boff1];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                if (!tile_live[u]) continue;   // warp-uniform: ragged last pair CTA of a trial
                // A fragment order: (row g, t lo), (row g+8, t lo), (row g, t hi), (row g+8, t hi)
                const cplx p0 = cmulc(cPsi[tlo * N1 + pnp[u][0]], cPsi[tlo * N1 + pn[u][0]]);
                const cplx p1 = cmulc(cPsi[tlo * N1 + pnp[u][1]], cPsi[tlo * N1 + pn[u][1]]);
                const cplx p2 = cmulc(cPsi[thi * N1 + pnp[u][0]], cPsi[thi * N1 + pn[u][0]]);
                const cplx p3 = cmulc(cPsi[thi * N1 + pnp[u][1]], cPsi[thi * N1 + pn[u][1]]);
                const double pr[4] = {p0.x, p1.x, p2.x, p3.x};
                const double pi[4] = {p0.y, p1.y, p2.y, p3.y};
                dmma16x8x8(accr[u][0], pr, b00, b01);
                dmma16x8x8(accr[u][1], pr, b10, b11);
                dmma16x8x8(acci[u][0], pi, b00, b01);
                dmma16x8x8(acci[u][1], pi, b10, b11);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_empty[s]);   // this warp is done with the stage
    }
    // epilogue: accumulator (row g + 8h, cols 2 tig, 2 tig + 1 of n-tile nt)
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (!pv[u][h]) continue;
            const int n = pn[u][h], np = pnp[u][h];
            auto put = [&](int i, int j, cplx v) { Gb[(size_t)(n * NTX + i) * d.Lp + (np * NTX + j)] = v; };
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const double r0 = accr[u][nt][2 * h], r1 = accr[u][nt][2 * h + 1];
                const double i0 = acci[u][nt][2 * h], i1 = acci[u][nt][2 * h + 1];
                const int col = 8 * nt + 2 * tig;
                if (col < 4) {  // two diagonal entries: (pr Rd, pi Rd)
                    put(col, col, mk(r0, i0));
                    put(col + 1, col + 1, mk(r1, i1));
                } else {        // one upper pair q: U = pr Rr, W = pr Ri, Z = pi Rr, V = pi Ri
                    const int q = (col - 4) >> 1;
                    const int qi = (q < 3) ? 0 : (q < 5 ? 1 : 2);
                    const int qj = (q < 3) ? q + 1 : (q < 5 ? q - 1 : 3);
                    put(qi, qj, mk(r0 - i1, r1 + i0));
                    put(qj, qi, mk(r0 + i1, i0 - r1));
                }
            }
        }
}

// Generic tensor-path Gram, n_tx = 4..8.  Column layout of the real B matrix (NC columns, padded to a
// multiple of 8): [0, NTX) the real diagonal of R_t; from the even offset PO on, (re, im) of the upper
// entries (i<j) in row-major order.  A warp owns one 16-pair tile and all NT column tiles; the chunk
// length TC (multiple of 8) is chosen at launch so that two cp.async stages fit in shared memory.
template <int NTX>
struct GramCols {
    static constexpr int NPAIR = NTX * (NTX - 1) / 2;
    static constexpr int PO = (NTX + 1) & ~1;
    static constexpr int NC = PO + 2 * NPAIR;
    static constexpr int NT = (NC + 7) / 8;
    __device__ __forceinline__ static void pair_ij(int q, int& i, int& j) {
        i = 0;
        while (q >= NTX - 1 - i) { q -= NTX - 1 - i; ++i; }
        j = i + 1 + q;
    }
    // column -> double offset inside the raw R_t (row-major NTX x NTX interleaved complex); -1: padding
    __device__ __forceinline__ static int offset(int col) {
        if (col < NTX) return 2 * (col * NTX + col);
        if (col < PO || col >= NC) return -1;
        int i, j;
        pair_ij((col - PO) >> 1, i, j);
        return 2 * (i * NTX + j) + ((col - PO) & 1);
    }
};

constexpr int GW_PAIRS = (GR_THREADS / 32) * 16;   // pairs per CTA of the generic kernel

template <int NTX>
__global__ void __launch_bounds__(GR_THREADS, 1) k_gram_mma(Dims d, int T, int TC, const cplx* __restrict__ Psi,
                                                          const cplx* __restrict__ sR, const cplx* __restrict__ Y,
                                                          const cplx* __restrict__ sm, const cplx* __restrict__ Ginit,
                                                          cplx* __restrict__ Gout, const int32_t* __restrict__ active) {
    typedef GramCols<NTX> GC;
    constexpr int NT = GC::NT;
    constexpr int RS = 2 * NTX * NTX;   // doubles per staged R_t
    extern __shared__ double2 gsm[];
    const int b = blockIdx.y;
    if (active != nullptr && active[b] == 0) return;
    const int N1 = d.N1;
    const int P = N1 * (N1 + 1) / 2;
    const cplx* psi_b = Psi + (size_t)(d.psi_shared ? 0 : b) * T * N1;
    const size_t gstride = (size_t)d.Ltot * d.Lp;
    cplx* Gb = Gout + (size_t)b * gstride;
    const cplx* Gi = Ginit ? Ginit + (size_t)b * gstride : nullptr;
    if (blockIdx.x == gridDim.x - 1) {
        gram_rhs_cta<NTX>(d, T, b, gsm, gsm + GR_TC * N1, psi_b, Y, sm, Gi, Gb);
        return;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
    int pn[2], pnp[2];
    bool pv[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        int item = blockIdx.x * GW_PAIRS + warp * 16 + g + 8 * h;
        pv[h] = item < P;
        item = min(item, P - 1);
        int n = (int)((sqrtf(8.0f * (float)item + 1.0f) - 1.0f) * 0.5f);   // made exact by the loops below
        while ((n + 1) * (n + 2) / 2 <= item) ++n;
        while (n * (n + 1) / 2 > item) --n;
        pn[h] = n;
        pnp[h] = item - n * (n + 1) / 2;
    }
    int boff[NT];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) boff[nt] = GC::offset(8 * nt + g);
    double accr[NT][4], acci[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) { accr[nt][e] = 0.0; acci[nt][e] = 0.0; }

    const cplx* R_b = sR + (size_t)b * T * NTX * NTX;
    const int stage_elems = TC * (N1 + NTX * NTX);
    auto issue = [&](int chunk, int buf) {
        const int t0 = chunk * TC;
        const int tc = min(TC, T - t0);
        cplx* dpsi = gsm + buf * stage_elems;
        cplx* dR = dpsi + TC * N1;
        const cplx* spsi = psi_b + (size_t)t0 * N1;
        const cplx* sRg = R_b + (size_t)t0 * NTX * NTX;
        for (int e = threadIdx.x; e < tc * N1; e += GR_THREADS) cp_async16(dpsi + e, spsi + e);
        for (int e = threadIdx.x; e < tc * NTX * NTX; e += GR_THREADS) cp_async16(dR + e, sRg + e);
        if (tc < TC) {  // ragged last chunk: symbols beyond T contribute zero
            for (int e = tc * N1 + threadIdx.x; e < TC * N1; e += GR_THREADS) dpsi[e] = mk(0.0, 0.0);
            for (int e = tc * NTX * NTX + threadIdx.x; e < TC * NTX * NTX; e += GR_THREADS) dR[e] = mk(0.0, 0.0);
        }
        cp_async_commit();
    };
    const int nchunk = (T + TC - 1) / TC;
    if (nchunk > 0) issue(0, 0);
    for (int ck = 0; ck < nchunk; ++ck) {
        const int buf = ck & 1;
        if (ck + 1 < nchunk) { issue(ck + 1, buf ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
        __syncthreads();
        const cplx* cPsi = gsm + buf * stage_elems;
        const double* cR = (const double*)(cPsi + TC * N1);
        for (int ks = 0; ks < TC / 8; ++ks) {
            const int tlo = ks * 8 + tig, thi = tlo + 4;
            // A fragment order: (row g, t lo), (row g+8, t lo), (row g, t hi), (row g+8, t hi)
            const cplx p0 = cmulc(cPsi[tlo * N1 + pnp[0]], cPsi[tlo * N1 + pn[0]]);
            const cplx p1 = cmulc(cPsi[tlo * N1 + pnp[1]], cPsi[tlo * N1 + pn[1]]);
            const cplx p2 = cmulc(cPsi[thi * N1 + pnp[0]], cPsi[thi * N1 + pn[0]]);
            const cplx p3 = cmulc(cPsi[thi * N1 + pnp[1]], cPsi[thi * N1 + pn[1]]);
            const double pr[4] = {p0.x, p1.x, p2.x, p3.x};
            const double pi[4] = {p0.y, p1.y, p2.y, p3.y};
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const double b0 = boff[nt] >= 0 ? cR[tlo * RS + boff[nt]] : 0.0;
                const double b1 = boff[nt] >= 0 ? cR[thi * RS + boff[nt]] : 0.0;
                dmma16x8x8(accr[nt], pr, b0, b1);
                dmma16x8x8(acci[nt], pi, b0, b1);
            }
        }
        __syncthreads();
    }
    // epilogue: accumulator (row g + 8h, cols 8 nt + 2 tig, + 1)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        if (!pv[h]) continue;
        const int n = pn[h], np = pnp[h];
        auto put = [&](int i, int j, cplx v) {
            const size_t o = (size_t)(n * NTX + i) * d.Lp + (np * NTX + j);
            if (Gi) v = cadd(v, Gi[o]);
            Gb[o] = v;
        };
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            const double r0 = accr[nt][2 * h], r1 = accr[nt][2 * h + 1];
            const double i0 = acci[nt][2 * h], i1 = acci[nt][2 * h + 1];
            const int col = 8 * nt + 2 * tig;
            if (col < NTX) {  // diagonal entries: (pr Rd, pi Rd)
                put(col, col, mk(r0, i0));
                if (col + 1 < NTX) put(col + 1, col + 1, mk(r1, i1));
            } else if (col >= GC::PO && col < GC::NC) {  // upper pair: U = pr Rr, W = pr Ri, Z = pi Rr, V = pi Ri
                int qi, qj;
                GC::pair_ij((col - GC::PO) >> 1, qi, qj);
                put(qi, qj, mk(r0 - i1, r1 + i0));
                put(qj, qi, mk(r0 + i1, i0 - r1));
            }
        }
    }
}

// shared memory the right-hand-side CTA needs at least: one 8-symbol MMA step of psi and of the padded Zc rows
static size_t rhs_smem_min(int N1, int ntx, int n_rx) { return sizeof(cplx) * (size_t)(8 * (N1 + ntx * n_rx + 2)); }

constexpr size_t GRAM_SMEM_CAP = 227 * 1024;   // opt-in shared memory per block on sm_100

// Dynamic shared memory of the one Gram launch for a shape, and the pair CTAs' chunk length.  The pair CTAs need
// their operand stages; the right-hand-side CTA of the same launch sizes its chunk from whatever it finds (16
// symbols when they fit under the cap, one 8-symbol MMA step at least).  make_dims() admits a shape through
// gram_supports(), the launchers below request exactly this: an admitted shape is a shape that launches.
static size_t gram_smem(int N1, int ntx, int n_rx, int* tc_out) {
    const size_t rhs1 = rhs_smem_min(N1, ntx, n_rx);
    size_t pair, rhs_want = 2 * rhs1;
    int tc;
    if (ntx <= 3) {           // scalar k_gram: two cp.async stages, chunk shrunk for very long phase rows
        tc = GR_TC;
        while (tc > 2 && sizeof(cplx) * (size_t)(2 * tc * (N1 + ntx * ntx)) > 100 * 1024) tc >>= 1;
        pair = sizeof(cplx) * (size_t)(2 * tc * (N1 + ntx * ntx));
        rhs_want = rhs1;
    } else if (ntx == 4 && sizeof(cplx) * (size_t)(GT_STAGES * GT_TC * (N1 + 16)) <= 160 * 1024) {
        tc = GT_TC;               // k_gram_tma4: four-stage TMA ring (N <= 143)
        pair = sizeof(cplx) * (size_t)(GT_STAGES * GT_TC * (N1 + 16));
    } else {                      // k_gram_mma<NTX>: two stages of the largest chunk under 100 KB, 8 symbols at least
        tc = 32;
        while (tc > 8 && sizeof(cplx) * (size_t)(2 * tc * (N1 + ntx * ntx)) > 100 * 1024) tc >>= 1;
        pair = sizeof(cplx) * (size_t)(2 * tc * (N1 + ntx * ntx));
    }
    if (tc_out) *tc_out = tc;
    size_t smem = pair > rhs_want ? pair : rhs_want;
    if (smem > GRAM_SMEM_CAP) smem = pair > rhs1 ? pair : rhs1;
    return smem;
}

// Admitted phase-row lengths: N + 1 + n_tx^2 <= 908 for every n_tx (two 8-symbol stages of the generic kernel in
// 227 KB; the documented limit, also for the scalar kernel, which would take longer rows), and the launch for
// this shape must fit.  abi.cu's make_dims() answers SBCE_E_UNSUPPORTED otherwise, before any launch.
bool gram_supports(int N1, int n_tx, int n_rx) {
    return sizeof(cplx) * (size_t)(2 * 8 * (N1 + n_tx * n_tx)) <= GRAM_SMEM_CAP &&
           gram_smem(N1, n_tx, n_rx, nullptr) <= GRAM_SMEM_CAP;
}

template <int NTX>
static cudaError_t run_gram_wide(const Dims& d, int nb, const double* Psi, int T, const double* sR, const double* Y,
                                 const double* sm, const double* Ginit, double* Gout, const int32_t* active,
                                 cudaStream_t s) {
    static SmemOptIn optin;
    const int P = d.N1 * (d.N1 + 1) / 2;
    dim3 grid((P + GW_PAIRS - 1) / GW_PAIRS + 1, nb);   // + 1: the right-hand-side / padding CTA
    int tc = 0;
    const size_t smem = gram_smem(d.N1, NTX, d.n_rx, &tc);
    if (smem > GRAM_SMEM_CAP) return cudaErrorInvalidValue;
    cudaError_t e = opt_in_smem(optin, (const void*)k_gram_mma<NTX>, smem);
    if (e != cudaSuccess) return e;
    k_gram_mma<NTX><<<grid, GR_THREADS, smem, s>>>(d, T, tc, (const cplx*)Psi, (const cplx*)sR, (const cplx*)Y,
                                                   (const cplx*)sm, (const cplx*)Ginit, (cplx*)Gout, active);
    count_launch();
    return cudaGetLastError();
}

// n_tx <= 3: scalar Hermitian-shared kernel, chunk length shrunk for very long phase rows
template <int NTX>
static cudaError_t run_gram_scalar(const Dims& d, int nb, const double* Psi, int T, const double* sR, const double* Y,
                                   const double* sm, const double* Ginit, double* Gout, const int32_t* active,
                                   cudaStream_t s) {
    static SmemOptIn optin;
    const int P = d.N1 * (d.N1 + 1) / 2;
    dim3 grid((P + GR_THREADS - 1) / GR_THREADS + 1, nb);   // + 1: the right-hand-side / padding CTA
    int tc = 0;
    const size_t smem = gram_smem(d.N1, NTX, d.n_rx, &tc);
    if (smem > GRAM_SMEM_CAP) return cudaErrorInvalidValue;
    cudaError_t e = opt_in_smem(optin, (const void*)k_gram<NTX>, smem);
    if (e != cudaSuccess) return e;
    k_gram<NTX><<<grid, GR_THREADS, smem, s>>>(d, T, tc, (const cplx*)Psi, (const cplx*)sR, (const cplx*)Y,
                                               (const cplx*)sm, (const cplx*)Ginit, (cplx*)Gout, active);
    count_launch();
    return cudaGetLastError();
}

// n_tx = 4: TMA-fed tensor-path kernel while its four-stage ring fits in 160 KB (N <= 143), else the generic one
static cudaError_t run_gram4(const Dims& d, int nb, const double* Psi, int T, const double* sR, const double* Y,
                             const double* sm, const double* Ginit, double* Gout, const int32_t* active,
                             cudaStream_t s) {
    constexpr int NTX = 4;
    static SmemOptIn optin;
    if (sizeof(cplx) * (size_t)(GT_STAGES * GT_TC * (d.N1 + NTX * NTX)) > 160 * 1024)
        return run_gram_wide<4>(d, nb, Psi, T, sR, Y, sm, Ginit, Gout, active, s);
    const int P = d.N1 * (d.N1 + 1) / 2;
    dim3 grid((P + GR_THREADS - 1) / GR_THREADS + 1, nb);   // + 1: the right-hand-side / padding CTA
    const size_t smem = gram_smem(d.N1, NTX, d.n_rx, nullptr);
    cudaError_t e = opt_in_smem(optin, (const void*)k_gram_tma4, smem);
    if (e != cudaSuccess) return e;
    k_gram_tma4<<<grid, GT_THREADS, smem, s>>>(d, T, (const cplx*)Psi, (const cplx*)sR, (const cplx*)Y,
                                               (const cplx*)sm, (const cplx*)Ginit, (cplx*)Gout, active);
    count_launch();
    return cudaGetLastError();
}

// Normal-equation build: lower triangle of G, B^H rows and padding, one launch.
cudaError_t launch_normal_equations(const Dims& d, int nb, const double* Psi, int T, const double* Y,
                                    const double* sm, const double* sR, const double* Ginit, double* Gout,
                                    const int32_t* active, cudaStream_t s) {
    if (d.n_rx > RH_MAXR) return cudaErrorInvalidValue;
    switch (d.n_tx) {
        case 1: return run_gram_scalar<1>(d, nb, Psi, T, sR, Y, sm, Ginit, Gout, active, s);
        case 2: return run_gram_scalar<2>(d, nb, Psi, T, sR, Y, sm, Ginit, Gout, active, s);
        case 3: return run_gram_scalar<3>(d, nb, Psi, T, sR, Y, sm, Ginit, Gout, active, s);
        case 4: return run_gram4(d, nb, Psi, T, sR, Y, sm, Ginit, Gout, active, s);
        case 5: return run_gram_wide<5>(d, nb, Psi, T, sR, Y, sm, Ginit, Gout, active, s);
        case 6: return run_gram_wide<6>(d, nb, Psi, T, sR, Y, sm, Ginit, Gout, active, s);
        case 7: return run_gram_wide<7>(d, nb, Psi, T, sR, Y, sm, Ginit, Gout, active, s);
        case 8: return run_gram_wide<8>(d, nb, Psi, T, sR, Y, sm, Ginit, Gout, active, s);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace sbce
