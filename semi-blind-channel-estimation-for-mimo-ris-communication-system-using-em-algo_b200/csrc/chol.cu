// Solve step of the M-step: blocked complex Cholesky of the augmented lower trapezoid [G ; B^H] produced by the
// normal-equation kernels (mstep.cu), then the back substitution.
//
// Reference semantics (/root/reference/Proposed_method_NMSEvsTp.py:66):
//   theta = np.linalg.solve(denom, numer)   with denom = G (x) I_nrx  =>  Theta = G^-1 B   (L x n_rx)
//
// k_chol_solve -- one CTA (4 warps) per trial, LEFT-looking blocked factorisation (panel width 16) on the FP64
//   tensor path (mma.sync m16n8k8.f64, SASS DMMA.8x8x4) with look-ahead, organised as a BARRIER-FREE TASK
//   PIPELINE.  Iteration k works on the 16-row tiles below the diagonal block of panel k; a tile is taken
//   through two steps by the warp that claimed it:
//     A. X = S W_k^H           triangular solve of panel k as a GEMM against the inverse of the diagonal block,
//     B. S' = A - C[rows, 0:g0] C[g0:g0+16, 0:g0]^H    update for panel k+1 against ALL previous columns.
//   The (panel, tile) pairs form ONE ordered task list; warps claim tasks from a shared counter and synchronise
//   through flags in shared memory only -- panels completed per 16-row block (s_prog), "block row k+1 is final"
//   (s_rowready), "W_k is available" (s_wready) -- so a warp that runs out of tiles of panel k starts on panel
//   k+1 as soon as its inputs exist.  Every wait is on a task EARLIER in the list and tasks are claimed in
//   order, so the earliest unfinished task can always run: no deadlock.  The warp that owns tile (k, 0) factors
//   the next diagonal block in registers; the inverses W_k live in a 3-deep ring (the writer checks that all
//   tiles of panel k-2 are past their triangular solve).  Operand fragments come straight from global memory,
//   double-buffered in registers (the block row hits L1, the tile rows stream from L2 / DRAM and are pulled
//   into L1 two steps ahead by prefetch.global.L1, which holds no registers); the complex product uses three
//   real DMMA products (Gauss): re = P1 + P2, im = P3 - P1 + P2 with P1 = ar br, P2 = ai bi,
//   P3 = (ar + ai)(br - bi).  The trailing matrix is never touched; the B^H rows carried under the matrix come
//   out as (C^-1 B)^H, i.e. the forward substitution is free.
// The back substitution runs in the same CTA afterwards (17 blocks, W^H applied instead of a serial triangular
// solve).  It holds 18 % of the kernel's resident warp time (profiles/r02d) as serial latency; moving it into a
// kernel of its own (one warp per trial, right-hand sides in shared memory) was measured and is slower
// (1.96 ms for both kernels against 1.84 ms): one warp per trial leaves only 8 warps per SM to hide the
// 17 x ~5 dependent global-load latencies of a trial.
//
// Measured history of this file (B200, N=64 4x4: L=260, 1184 trials per launch; gpurun_out/r02b-r02g):
//   k_chol2 (round 1: look-ahead, one CTA barrier per panel, register-fed operands)                    1.94 ms
//   task pipeline, both operands through a per-warp cp.async ring (2-4 stages, 3-4 CTAs/SM)     2.10 - 2.82 ms
//     (the ring costs L1 capacity: the block-row operand then misses; deeper rings made it worse)
//   task pipeline, register-fed operands                                                               2.03 ms
//   + Gauss 3-multiplication product                                                                   1.89 ms
//   + L1 prefetch two steps ahead                                                                      1.84 ms
//   two panels per pass over the factor (32-column update, halves the operand stream)           2.06 - 2.41 ms
//     (48 accumulator registers + double-buffered block rows spill at 128 and at 168 registers)
//   L2 evict_last on every third trial / evict_first stream (createpolicy + cache_hint)          1.84 ms (+-0)
//   L2 prefetch of the next block's rows in the back substitution                                      +-0
//   back substitution as a separate warp-per-trial kernel                                          1.96 ms
//   next step's fragment loads pinned to the top of the step (volatile asm; ptxas sinks them)   1.86 ms (+-0)
//   CTA shapes at 128 registers (gpurun_out/r02p): 8 warps x 2 CTAs/SM 2.34 ms, 16 warps x 1 CTA/SM 3.80 ms,
//     2 warps x 8 CTAs/SM 1.87 ms -- the factors of 2 resp. 1 resident trial per SM fit in L2, those of 4 do
//     not: the trials in flight per SM matter, L2 residency does not
//   96 registers / 5 CTAs per SM (680 bytes of spills), with or without the Gauss product             2.43 ms
//   back substitution: W row as independent loads before the barrier + L1 prefetch of the next block   1.82 ms
//     (both column rounds of the update fetched up front: spills, 2.02 ms)
//   fragments as 256-bit loads on a permuted contraction index (halves the L1 wavefronts of a load)    1.81 ms
//   L1 prefetch distance 0 / 1 / 2 / 3 steps                                        2.02 / 1.87 / 1.81 / 1.83 ms
//   L1 prefetch of the 16 x 16 block to be updated four steps before the loop ends (its read-modify-write wait
//     held 12.6 % of the warp samples, profiles/r02m) and of the block-row operand by the idle lanes   +-0.5 %
//     -- removing single stall sites no longer moves the kernel: DRAM 40 %, L2->L1 5 TB/s, DMMA pipe 44 %, L1
//     wavefronts 47 % are all half used; what is left is the number of independent trials per SM (registers)
//   no register double buffer (operands read from L1 behind the prefetch): 4 CTAs/SM 1.84 ms; 5 CTAs/SM at 96
//     registers 2.39 ms, 6 at 80 registers 3.20 ms (the register-resident diagonal factor spills 0.8 - 1.6 KB)
//   L1 policies on the fragment loads (ld.global.lu / evict_first for the streamed rows, evict_last for the
//     block rows) and the solution vector moved to global memory (L1 156 -> 224 KB)                     +-0.3 %
#include <math.h>

#include "common.cuh"
#include "tensor.cuh"

namespace sbce {

constexpr int CH_NB = 16;            // panel width
constexpr int CH_DS = CH_NB + 1;     // row stride (complex) of the shared 16x16 blocks
constexpr int CF_WARPS = 4;          // warps of a factorisation CTA

// Diagonal block, register resident (a shared-memory version sat on the critical path for 43 % of an earlier
// kernel, profiles/r01i: LDS -> DFMA -> STS round trips, a DSQRT + DDIV per column, a DDIV per row of the
// inverse).  Lane r (and its mirror r + 16) keeps row r of the block in
// registers; column c is a left-looking dot product against row c, fetched with width-16 shuffles; the
// pivot is broadcast, inverted once with rsqrt (no division anywhere); the inverse W = L^-1 is built column
// per lane from broadcast reads of L in shared memory.  W's strict lower part is parked in the unused
// strict UPPER triangle of the diagonal block in global memory (A[k0+j][k0+i] = W[i][j], i > j) so that
// the back substitution can apply W^H instead of running a serial triangular solve.
__device__ __forceinline__ void chol_diag_factor_reg(const Dims& d, cplx* A, int ld, int k0, int nb, cplx* sD, cplx* sW,
                                                     int lane, double& maxpiv, int* s_bad) {
    const unsigned full = 0xffffffffu;
    const int r = lane & 15;
    cplx a[CH_NB];
    {
        const cplx* rowp = A + (size_t)(k0 + min(r, nb - 1)) * ld + k0;
#pragma unroll
        for (int c = 0; c < CH_NB; ++c) a[c] = (r < nb && c <= r && c < nb) ? rowp[c] : mk(0.0, 0.0);
    }
    double invs[CH_NB];
#pragma unroll
    for (int c = 0; c < CH_NB; ++c) {
        cplx s = a[c];
#pragma unroll
        for (int q = 0; q < c; ++q) {
            const cplx lcq = mk(__shfl_sync(full, a[q].x, c, 16), __shfl_sync(full, a[q].y, c, 16));
            cfmsc(s, a[q], lcq);   // s -= L[r][q] conj(L[c][q])
        }
        double piv = __shfl_sync(full, s.x, c, 16);
        const bool live = c < nb;
        if (live) {
            // numerically singular: not above 1e-13 times the largest pivot so far in the trial (NaN included, and
            // non-positive pivots whatever the maximum); the identity padding (k0 + c >= L) is exempt
            if (!(piv > ((k0 + c < d.L) ? 1e-13 * maxpiv : 0.0))) {
                if (lane == 0) *s_bad = 1;
                piv = 1.0;
            }
            maxpiv = fmax(maxpiv, piv);
        } else {
            piv = 1.0;
        }
        const double inv = rsqrt(piv);
        invs[c] = live ? inv : 0.0;
        a[c] = (!live || r < c) ? mk(0.0, 0.0) : (r == c ? mk(piv * inv, 0.0) : cscale(s, inv));
    }
    if (lane < CH_NB) {
#pragma unroll
        for (int c = 0; c < CH_NB; ++c) sD[r * CH_DS + c] = a[c];
    }
    __syncwarp();
    // W = L^-1, lane = column j:  W[i][j] = -inv_i sum_{q<i} L[i][q] W[q][j]  (W[q][j] = 0 for q < j)
    cplx w[CH_NB];
#pragma unroll
    for (int i = 0; i < CH_NB; ++i) {
        cplx acc0 = mk(0.0, 0.0), acc1 = mk(0.0, 0.0);
#pragma unroll
        for (int q = 0; q < i; ++q) {
            if (q & 1) cfma(acc1, sD[i * CH_DS + q], w[q]); else cfma(acc0, sD[i * CH_DS + q], w[q]);
        }
        w[i] = (i == r) ? mk(invs[i], 0.0) : mk(-invs[i] * (acc0.x + acc1.x), -invs[i] * (acc0.y + acc1.y));
    }
    if (lane < CH_NB) {
#pragma unroll
        for (int i = 0; i < CH_NB; ++i) sW[i * CH_DS + r] = w[i];
        if (r < nb) {   // row k0 + r of the block: L up to the diagonal, then W^T
            cplx* rowp = A + (size_t)(k0 + r) * ld + k0;
#pragma unroll
            for (int c = 0; c < CH_NB; ++c)
                if (c < nb) rowp[c] = (c <= r) ? sD[r * CH_DS + c] : w[c];
        }
    }
    __syncwarp();
}

__device__ __forceinline__ void spin_until_ge(const volatile int* p, int v) {
    while (*p < v) __nanosleep(20);
    __threadfence_block();
}

// ---------------------------------------------------------------------------
// Factorisation
// ---------------------------------------------------------------------------
template <bool GAUSS, int MINB, int PF>
__global__ void __launch_bounds__(CF_WARPS * 32, MINB) k_chol_solve(Dims d, cplx* __restrict__ Gall,
                                                                    cplx* __restrict__ theta,
                                                                    const int32_t* __restrict__ active,
                                                                    int32_t* __restrict__ stat, cplx* th_global) {
    constexpr int CH_THREADS = CF_WARPS * 32;
    extern __shared__ __align__(16) double2 csm[];
    const int b = blockIdx.x;
    if (active != nullptr && active[b] == 0) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, tig = lane & 3;
    const int Lp = d.Lp, Ltot = d.Ltot, ld = d.Lp;
    cplx* A = Gall + (size_t)b * Ltot * Lp;
    const int npan = (Lp + CH_NB - 1) / CH_NB;
    const int nrb = (Ltot + 15) / 16 + 1;
    cplx* sD = csm;                                            // [16][17] diagonal block scratch
    cplx* sWb = sD + CH_NB * CH_DS;                            // [3][16][17] inverses of the diagonal blocks
    cplx* sTh = sWb + 3 * CH_NB * CH_DS;                       // [Lp][n_rx] solution vector (unless in global scratch)
    int* s_prog = (int*)(sTh + (th_global ? 0 : Lp * d.n_rx)); // [nrb] panels completed per aligned 16-row block
    int* s_adone = s_prog + nrb;                               // [npan] tiles of panel k past their triangular solve
    int* s_start = s_adone + npan;                             // [npan + 1] first task id of panel k
    __shared__ int s_next, s_bad;
    __shared__ volatile int s_wready, s_rowready;
    __shared__ double s_maxpiv;

    for (int i = tid; i < nrb + npan; i += CH_THREADS) s_prog[i] = 0;
    if (tid == 0) {
        s_next = 0; s_bad = 0; s_wready = 0; s_rowready = 0; s_maxpiv = 0.0;
        int acc = 0;
        for (int k = 0; k < npan; ++k) {
            s_start[k] = acc;
            const int g0 = min(k * CH_NB + CH_NB, Lp);
            acc += (Ltot - g0 + 15) >> 4;
        }
        s_start[npan] = acc;
    }
    __syncthreads();
    if (warp == 0) {
        double maxpiv = 0.0;
        chol_diag_factor_reg(d, A, ld, 0, min(CH_NB, Lp), sD, sWb, lane, maxpiv, &s_bad);
        __threadfence_block();
        __syncwarp();
        if (lane == 0) { s_maxpiv = maxpiv; s_wready = 1; }
    }
    __syncthreads();
    const int ntasks = s_start[npan];

    int myk = 0;
    for (;;) {
        int id = 0;
        if (lane == 0) id = atomicAdd(&s_next, 1);
        id = __shfl_sync(0xffffffffu, id, 0);
        if (id >= ntasks) break;
        while (id >= s_start[myk + 1]) ++myk;
        const int k = myk, t = id - s_start[myk];
        const int k0 = k * CH_NB;
        const int nb = min(CH_NB, Lp - k0);
        const int g0 = k0 + nb;                                   // first row below the diagonal block = next panel
        const int nbn = (k + 1 < npan) ? min(CH_NB, Lp - g0) : 0;
        const int r0 = g0 + (t << 4);
        const cplx* sW = sWb + (k % 3) * CH_NB * CH_DS;

        if (k > 0) {
            spin_until_ge((const volatile int*)&s_prog[r0 >> 4], k);
            spin_until_ge((const volatile int*)&s_prog[(min(r0 + 16, Ltot) - 1) >> 4], k);
        }
        spin_until_ge(&s_wready, k + 1);

        const int ra = min(r0 + g, Ltot - 1), rb8 = min(r0 + g + 8, Ltot - 1);
        double cr[2][4], ci[2][4];
        // ---- step A: X = S W^H on columns k0 .. k0+nb-1
        {
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int e = 0; e < 4; ++e) { cr[j][e] = 0.0; ci[j][e] = 0.0; }
            const cplx* pa0 = A + (size_t)ra * ld + k0 + tig;
            const cplx* pa1 = A + (size_t)rb8 * ld + k0 + tig;
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                const int q0 = 8 * kk + tig;
                cplx a0 = mk(0, 0), a1 = mk(0, 0), a2 = mk(0, 0), a3 = mk(0, 0);
                if (q0 < nb) { a0 = pa0[8 * kk]; a1 = pa1[8 * kk]; }
                if (q0 + 4 < nb) { a2 = pa0[8 * kk + 4]; a3 = pa1[8 * kk + 4]; }
                const double ar[4] = {a0.x, a1.x, a2.x, a3.x};
                const double ai[4] = {a0.y, a1.y, a2.y, a3.y};
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const cplx w0 = sW[(8 * j + g) * CH_DS + 8 * kk + tig];
                    const cplx w1 = sW[(8 * j + g) * CH_DS + 8 * kk + tig + 4];
                    dmma16x8x8(cr[j], ar, w0.x, w1.x);
                    dmma16x8x8(ci[j], ai, w0.x, w1.x);
                    dmma16x8x8(cr[j], ai, w0.y, w1.y);
                    dmma16x8x8(ci[j], ar, -w0.y, -w1.y);
                }
            }
            __syncwarp();  // all lanes have read S before anyone overwrites it
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int row = r0 + g + 8 * h;
                    const int c = 8 * j + 2 * tig;
                    if (row < Ltot && c < nb) {
                        cplx* p2 = A + (size_t)row * ld + k0 + c;
                        p2[0] = mk(cr[j][2 * h], ci[j][2 * h]);
                        p2[1] = mk(cr[j][2 * h + 1], ci[j][2 * h + 1]);
                    }
                }
        }
        __threadfence_block();
        __syncwarp();
        if (lane == 0) atomicAdd(&s_adone[k], 1);
        if (nbn == 0) continue;                                   // last panel: nothing left to update
        if (t == 0) {
            if (lane == 0) s_rowready = k + 1;                    // block row k+1 is final in columns < g0
        } else {
            spin_until_ge(&s_rowready, k + 1);
        }
        // ---- step B
        {
            if (tig == 0) {   // the blocks to be updated are only needed at the very end: start fetching them now
                asm volatile("prefetch.global.L2 [%0];" ::"l"(A + (size_t)ra * ld + g0));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(A + (size_t)rb8 * ld + g0));
            }
            double p3[GAUSS ? 2 : 1][4];
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int e = 0; e < 4; ++e) { cr[j][e] = 0.0; ci[j][e] = 0.0; if (GAUSS) p3[GAUSS ? j : 0][e] = 0.0; }
            // the contraction index of a step is permuted: lane tig takes columns (2 tig, 2 tig + 1) of the step's 8
            // as its k = tig and k = tig + 4 elements -- for BOTH operands, so the product is unchanged -- and fetches
            // them as one 256-bit load (rows start on 128-byte lines: a fragment load touches 8 lines instead of 16)
            const cplx* pa0 = A + (size_t)ra * ld + 2 * tig;
            const cplx* pa1 = A + (size_t)rb8 * ld + 2 * tig;
            const cplx* pb[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) pb[j] = A + (size_t)min(g0 + 8 * j + g, Ltot - 1) * ld + 2 * tig;
            // fragments are double-buffered in registers: the loads of step q+1 are in flight during the DMMAs of
            // step q (the tile rows stream from L2 / DRAM, the block rows hit L1)
            constexpr int NJ = 2;
            cplx fa[4], fb[NJ][2];
            ldg256(pa0, fa[0], fa[2]);
            ldg256(pa1, fa[1], fa[3]);
#pragma unroll
            for (int j = 0; j < NJ; ++j) ldg256(pb[j], fb[j][0], fb[j][1]);
            auto pair = [&](int j, const double (&ar)[4], const double (&ai)[4], const double (&as)[4], const cplx& b0,
                            const cplx& b1) {
                if (GAUSS) {
                    dmma16x8x8(cr[j], ar, b0.x, b1.x);
                    dmma16x8x8(ci[j], ai, b0.y, b1.y);
                    dmma16x8x8(p3[GAUSS ? j : 0], as, b0.x - b0.y, b1.x - b1.y);
                } else {
                    dmma16x8x8(cr[j], ar, b0.x, b1.x);
                    dmma16x8x8(ci[j], ai, b0.x, b1.x);
                    dmma16x8x8(cr[j], ai, b0.y, b1.y);
                    dmma16x8x8(ci[j], ar, -b0.y, -b1.y);
                }
            };
            // L1 prefetch of the streamed operand PF steps ahead (no registers held): lane r < 16 touches the line
            // that is row r's 8-column step
            const cplx* ppf = A + (size_t)min(r0 + (lane & 15), Ltot - 1) * ld;
#pragma unroll 1
            for (int q0 = 0; q0 < g0; q0 += 8) {
                cplx na[4], nbf[NJ][2];
                const int qn = (q0 + 8 < g0) ? q0 + 8 : q0;   // last step reloads itself (harmless, L1 hit)
                if (PF > 0 && lane < 16 && q0 + 8 * PF < g0)
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(ppf + q0 + 8 * PF));
                ldg256(pa0 + qn, na[0], na[2]);
                ldg256(pa1 + qn, na[1], na[3]);
#pragma unroll
                for (int j = 0; j < NJ; ++j) ldg256(pb[j] + qn, nbf[j][0], nbf[j][1]);
                const double ar[4] = {fa[0].x, fa[1].x, fa[2].x, fa[3].x};
                const double ai[4] = {fa[0].y, fa[1].y, fa[2].y, fa[3].y};
                const double as[4] = {fa[0].x + fa[0].y, fa[1].x + fa[1].y, fa[2].x + fa[2].y, fa[3].x + fa[3].y};
                pair(0, ar, ai, as, fb[0][0], fb[0][1]);
                pair(1, ar, ai, as, fb[1][0], fb[1][1]);
#pragma unroll
                for (int e = 0; e < 4; ++e) fa[e] = na[e];
#pragma unroll
                for (int j = 0; j < NJ; ++j)
                    { fb[j][0] = nbf[j][0]; fb[j][1] = nbf[j][1]; }
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int cbase = g0 + 8 * j;
                const int width = g0 + nbn;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int row = r0 + g + 8 * h;
                    const int c = cbase + 2 * tig;
                    if (row < Ltot && c < width) {
                        cplx* p2 = A + (size_t)row * ld + c;
                        const cplx v0 = p2[0], v1 = p2[1];
                        double re0, im0, re1, im1;
                        if (GAUSS) {
                            re0 = cr[j][2 * h] + ci[j][2 * h];
                            im0 = p3[GAUSS ? j : 0][2 * h] - cr[j][2 * h] + ci[j][2 * h];
                            re1 = cr[j][2 * h + 1] + ci[j][2 * h + 1];
                            im1 = p3[GAUSS ? j : 0][2 * h + 1] - cr[j][2 * h + 1] + ci[j][2 * h + 1];
                        } else {
                            re0 = cr[j][2 * h]; im0 = ci[j][2 * h]; re1 = cr[j][2 * h + 1]; im1 = ci[j][2 * h + 1];
                        }
                        p2[0] = mk(v0.x - re0, v0.y - im0);
                        p2[1] = mk(v1.x - re1, v1.y - im1);
                    }
                }
            }
        }
        __threadfence_block();
        __syncwarp();
        if (lane == 0) *((volatile int*)&s_prog[r0 >> 4]) = k + 1;
        if (t == 0) {
            // next diagonal block: its inverse goes into the ring slot last read by the tiles of panel k-2
            if (k >= 2) spin_until_ge((const volatile int*)&s_adone[k - 2], s_start[k - 1] - s_start[k - 2]);
            double maxpiv = s_maxpiv;
            chol_diag_factor_reg(d, A, ld, g0, nbn, sD, sWb + ((k + 1) % 3) * CH_NB * CH_DS, lane, maxpiv, &s_bad);
            __threadfence_block();
            __syncwarp();
            if (lane == 0) { s_maxpiv = maxpiv; s_wready = k + 2; }
        }
    }
    __syncthreads();
    if (tid == 0 && s_bad && stat) atomicOr(&stat[b], SBCE_ST_NOT_PD);

    // ---- back substitution  C^H theta = z,  z[l][r] = conj(A[Lp + r][l]).  Column-oriented ("right-looking"):
    // blocks of 16 unknowns from the bottom up; x = W^H rhs with W = D^-1 parked in the strict upper triangle of
    // the diagonal block (no serial triangular solve); then every earlier right-hand-side entry c < k0 is updated
    // with the block's 16 factor rows -- contiguous in memory, consecutive threads read consecutive columns
    // (coalesced), 16 independent loads in flight per thread.
    cplx* th = th_global ? th_global + (size_t)b * d.Lp * d.n_rx : sTh;
    const int nrx = d.n_rx;
    for (int e = tid; e < Lp * nrx; e += CH_THREADS) {
        const int l = e / nrx, r = e % nrx;
        th[e] = cconj(A[(size_t)(Lp + r) * ld + l]);
    }
    // A thread's W row is fetched as 15 independent predicated loads BEFORE the barrier that precedes the dependent
    // accumulation (the compiler's own unrolling left up to four serial L2 round trips per block), and the next
    // diagonal block's 2 x 16 lines are pulled into L1 during the update phase of the current block.
    const int kfirst = ((Lp - 1) / CH_NB) * CH_NB;
    auto prefetch_w = [&](int k0) {
        if (tid < 2 * CH_NB && k0 + (tid >> 1) < Lp)
            asm volatile("prefetch.global.L1 [%0];" ::"l"(A + (size_t)(k0 + (tid >> 1)) * ld + k0 + 8 * (tid & 1)));
    };
    prefetch_w(kfirst);
    for (int k0 = kfirst; k0 >= 0; k0 -= CH_NB) {
        const int nb = min(CH_NB, Lp - k0);
        const bool act = tid < nb * nrx;
        const int bc = act ? tid / nrx : 0, br = act ? tid % nrx : 0;
        cplx wv[CH_NB];
        const cplx* wrow = A + (size_t)(k0 + bc) * ld + k0;
        const double wd = wrow[bc].x;
#pragma unroll
        for (int q = 1; q < CH_NB; ++q) wv[q] = (act && q > bc && q < nb) ? wrow[q] : mk(0.0, 0.0);
        __syncthreads();  // th updates of the previous block are complete
        cplx xv = mk(0.0, 0.0);
        if (act) {
            xv = cscale(th[(k0 + bc) * nrx + br], 1.0 / wd);
#pragma unroll
            for (int q = 1; q < CH_NB; ++q)
                if (q > bc && q < nb) cfmac(xv, th[(k0 + q) * nrx + br], wv[q]);
        }
        __syncthreads();
        if (act) th[(k0 + bc) * nrx + br] = xv;
        if (k0 >= CH_NB) prefetch_w(k0 - CH_NB);
        __syncthreads();
        for (int c = tid; c < k0; c += CH_THREADS) {
            cplx cq[CH_NB];
#pragma unroll
            for (int q = 0; q < CH_NB; ++q) cq[q] = (q < nb) ? A[(size_t)(k0 + q) * ld + c] : mk(0.0, 0.0);
            for (int r = 0; r < nrx; ++r) {
                cplx v = th[c * nrx + r];
#pragma unroll
                for (int q = 0; q < CH_NB; ++q)
                    if (q < nb) cfmsc(v, th[(k0 + q) * nrx + r], cq[q]);
                th[c * nrx + r] = v;
            }
        }
    }
    __syncthreads();
    cplx* out = theta + (size_t)b * d.L * nrx;
    bool bad = false;
    for (int e = tid; e < d.L * nrx; e += CH_THREADS) {
        const cplx v = th[e];
        out[e] = v;
        if (!isfinite(v.x) || !isfinite(v.y)) bad = true;
    }
    if (bad && stat) atomicOr(&stat[b], SBCE_ST_NONFINITE);
}

cudaError_t launch_chol_solve(const Dims& d, int nb, double* G, double* theta, const int32_t* active, int32_t* stat,
                              double* th_scratch, cudaStream_t s) {
    static SmemOptIn optin;
    const int npan = (d.Lp + CH_NB - 1) / CH_NB, nrb = (d.Ltot + 15) / 16 + 1;
    const size_t fixed = sizeof(cplx) * (size_t)(4 * CH_NB * CH_DS) + sizeof(int) * (size_t)(nrb + 2 * npan + 2);
    const size_t thb = sizeof(cplx) * (size_t)d.Lp * d.n_rx;
    // the solution vector sits in shared memory only while that leaves most of the SM's L1 to the block-row
    // operand of the four resident trials, else in the caller's global scratch
    double* thg = nullptr;
    size_t smem = fixed + thb;
    if (smem > 24 * 1024) {
        if (!th_scratch) return cudaErrorInvalidValue;
        thg = th_scratch;
        smem = fixed;
    }
    // <Gauss product, 4 CTAs per SM (128 registers), L1 prefetch 2 steps ahead>: CTA shapes measured on B200 at
    // L = 260: 128 threads x 4 CTAs/SM 1.84 ms per 1184 trials, x 3 CTAs/SM (168 registers, no spills) 2.15 ms --
    // latency bound, more resident trials per SM win even though their factors no longer fit in L2
    cudaError_t e = opt_in_smem(optin, (const void*)k_chol_solve<true, 4, 2>, smem);
    if (e != cudaSuccess) return e;
    k_chol_solve<true, 4, 2><<<nb, CF_WARPS * 32, smem, s>>>(d, (cplx*)G, (cplx*)theta, active, stat, (cplx*)thg);
    count_launch();
    return cudaGetLastError();
}

}  // namespace sbce
