// Exact Gray-labelled bit LLRs of every data symbol at a channel estimate (conventions, window and clamp:
// include/sbce.h, sbce_bit_llr).
//
// Input is the E-step's QR record (k_heff_qr*): d2(x) = c0 + sum_i | ytilde_i - sum_{j>=i} R_ij x_j |^2.
// k_bit_llr walks the same hypothesis tree as k_enum (EnumT's tables and level arithmetic, streams n_tx-1 -> 1,
// stream 0 in closed form), one WARP per symbol, in two passes over the same walk:
//   1. the exact minimum d2: Babai incumbent, branch and bound on the partial distance (a lower bound of every
//      leaf below), warp minimum;
//   2. the per-bit sums relative to that minimum (the best hypothesis has weight 1), skipping subtrees whose
//      partial distance exceeds minimum + 96 varn^2.  Per surviving stream-1 node the M leaves are summed in
//      closed form: R_00 is real, so stream 0 separates into in-phase weights w_I[a] and quadrature weights
//      w_Q[b].  Both sides of every bit are accumulated explicitly (never as total minus the other side: that
//      cancels exactly in the cases that matter): the bits of streams >= 1 are fixed by the node code and take
//      the node's total; in-phase bit i of stream 0 takes W (sum_{a: gray(a)_i = v} w_I[a]) (sum_b w_Q[b]) on
//      side v, the quadrature bits likewise.
// The top streams are split across the lanes (the fewest with M^PL >= 32 prefixes), each lane walks its
// prefixes' subtrees alone, and the warp sums the per-lane accumulators in a fixed order: results do not
// depend on timing, chunking or the contents of the output buffer.  This runs once per trial after the EM
// loop, so the mapping favours clarity over the last few percent.
//
// With a-priori LLRs (PRIOR, k_bit_llr<n_tx, sqrt M, true>; include/sbce.h, sbce_bit_llr_apriori) every tree level
// also adds its stream's prior penalty varn^2 P_s(m) >= 0 (tables in the warp's shared block), stream 0's as
// separate in-phase and quadrature terms P_0I(iI) + P_0Q(iQ), so the partial metric stays a lower bound and
// the closed form of stream 0 keeps its I/Q separation.  The window widens by the largest |La| of the symbol
// and the result is the extrinsic LLR, the posterior one minus La.  Each penalty is its own addition: a zero
// prior adds +0.0 everywhere and reproduces the plain kernel bit for bit.
#include <math.h>

#include "common.cuh"
#include "tree.cuh"

namespace sbce {

constexpr double LLR_THR = 96.0;   // window of the sums, in units of varn^2 (error bound: include/sbce.h)

template <int NTX, int SQM, bool PRIOR = false>
struct LlrT {
    typedef EnumT<NTX, SQM> E;
    static constexpr int M = E::M, BITS = E::BITS, HB = E::HB;
    static constexpr int NB = NTX * BITS;   // LLRs per symbol
    static constexpr int NODE_STREAMS = NTX - 1;
    static constexpr int PLWANT = (5 + BITS - 1) / BITS;   // prefix streams so that M^PL >= 32
    static constexpr int PL = NODE_STREAMS < PLWANT ? NODE_STREAMS : PLWANT;
    static constexpr int NPREF = 1 << (BITS * PL);
    // per-warp shared block (doubles): tables R_is c_m, then the PAM levels R_ss pam_a, then with PRIOR the
    // penalties in distance units: P_s[m] for streams 1 .. NTX-1, then P_0I[a] and P_0Q[a]
    static constexpr int O_TAB = 0;
    static constexpr int O_G = O_TAB + 2 * E::NPAIR1 * M;
    static constexpr int O_P = O_G + NTX * SQM;
    static constexpr int O_P0I = O_P + (NTX - 1) * M, O_P0Q = O_P0I + SQM;
    static constexpr int WS_DOUBLES = ((PRIOR ? O_P0Q + SQM : O_P) + 1) & ~1;
    // bit i (MSB first) of the Gray label of PAM index a
    __device__ __forceinline__ static int bit(int a, int i) { return ((a ^ (a >> 1)) >> (HB - 1 - i)) & 1; }
};

// One lane's walk.  SUM = false: pass 1, `best` is the running minimum and the limit follows it.  SUM = true:
// pass 2, `best` is the warp's minimum and s0 / s1 collect both sides of every bit.  PRIOR: partial distances
// include the prior penalties, which follow the PAM levels g in the shared block (LlrT::O_P).
template <int NTX, int SQM, bool SUM, bool PRIOR = false>
struct LlrWalk {
    typedef EnumT<NTX, SQM> E;
    typedef LlrT<NTX, SQM, PRIOR> T;
    const cplx* tab;
    const double* g;
    double inv_s2;
    double best;
    double lim;    // subtrees whose partial distance exceeds lim are skipped
    bool prune;
    double s0[T::NB], s1[T::NB];

    // varn^2 P_s(m) of stream s >= 1; stream 0's in-phase and quadrature terms
    __device__ __forceinline__ double pen_s(int s, int m) const { return g[T::O_P - T::O_G + (s - 1) * T::M + m]; }
    __device__ __forceinline__ const double* pen_I() const { return g + (T::O_P0I - T::O_G); }
    __device__ __forceinline__ const double* pen_Q() const { return g + (T::O_P0Q - T::O_G); }

    // min over the PAM levels a of (v - g_a)^2 + p[a]: stream 0's best leaf on one axis under the prior
    __device__ __forceinline__ double pam_min(double v, const double* p) const {
        double dmin = 1e300;
#pragma unroll
        for (int a = 0; a < SQM; ++a) {
            const double e = v - g[a];
            double da = e * e;
            da += p[a];
            dmin = fmin(dmin, da);
        }
        return dmin;
    }

    __device__ __forceinline__ void leaf(cplx t0, double nb, int code) {
        if (!SUM) {
            double dI, dQ;
            if constexpr (PRIOR) {
                dI = pam_min(t0.x, pen_I());
                dQ = pam_min(t0.y, pen_Q());
            } else {
                E::slice(t0.x, g, dI);
                E::slice(t0.y, g, dQ);
            }
            const double v = nb + dI + dQ;
            if (v < best) { best = v; lim = v; }
            return;
        }
        double eI[SQM], eQ[SQM], minI = 1e300, minQ = 1e300;
#pragma unroll
        for (int a = 0; a < SQM; ++a) {
            const double xI = t0.x - g[a], xQ = t0.y - g[a];
            eI[a] = xI * xI;
            eQ[a] = xQ * xQ;
            if constexpr (PRIOR) {
                eI[a] += pen_I()[a];
                eQ[a] += pen_Q()[a];
            }
            minI = fmin(minI, eI[a]);
            minQ = fmin(minQ, eQ[a]);
        }
        const double W = exp((best - (nb + minI + minQ)) * inv_s2);   // the node's best leaf, <= 1
        if (W == 0.0) return;
        double SI = 0.0, SQ = 0.0, I0[T::HB], I1[T::HB], Q0[T::HB], Q1[T::HB];
#pragma unroll
        for (int i = 0; i < T::HB; ++i) { I0[i] = 0.0; I1[i] = 0.0; Q0[i] = 0.0; Q1[i] = 0.0; }
#pragma unroll
        for (int a = 0; a < SQM; ++a) {
            const double wI = exp((minI - eI[a]) * inv_s2), wQ = exp((minQ - eQ[a]) * inv_s2);
            SI += wI;
            SQ += wQ;
#pragma unroll
            for (int i = 0; i < T::HB; ++i) {
                if (T::bit(a, i)) { I1[i] += wI; Q1[i] += wQ; } else { I0[i] += wI; Q0[i] += wQ; }
            }
        }
        const double WI = W * SQ, WQ = W * SI, total = W * SI * SQ;
#pragma unroll
        for (int i = 0; i < T::HB; ++i) {
            s0[i] += WI * I0[i];
            s1[i] += WI * I1[i];
            s0[T::HB + i] += WQ * Q0[i];
            s1[T::HB + i] += WQ * Q1[i];
        }
#pragma unroll
        for (int s = 1; s < NTX; ++s) {
            const int m = E::digit(code, s), iI = m & (SQM - 1), iQ = m >> T::HB;
#pragma unroll
            for (int i = 0; i < T::HB; ++i) {
                const int bI = T::bit(iI, i), bQ = T::bit(iQ, i);
                s0[s * T::BITS + i] += bI ? 0.0 : total;
                s1[s * T::BITS + i] += bI ? total : 0.0;
                s0[s * T::BITS + T::HB + i] += bQ ? 0.0 : total;
                s1[s * T::BITS + T::HB + i] += bQ ? total : 0.0;
            }
        }
    }

    // streams S_ .. 1 below a node (acc: residuals, base: partial distance, code: digits so far), then the leaves
    template <int S_>
    __device__ __forceinline__ void walk(const cplx (&acc)[NTX], double base, int code) {
        if constexpr (S_ == 0) {
            leaf(acc[0], base, code);
        } else {
#pragma unroll 1
            for (int m = 0; m < T::M; ++m) {
                cplx nacc[NTX];
                double nb = E::step(acc, nacc, S_, m, base, g, tab);
                if constexpr (PRIOR) nb += pen_s(S_, m);
                if (prune && nb > lim) continue;
                walk<S_ - 1>(nacc, nb, code + (m << (T::BITS * (NTX - 1 - S_))));
            }
        }
    }

    // every prefix p = lane, lane + 32, ...: the top PL streams take the digits of p (stream n_tx-1-l the l-th
    // base-M digit), which is also the node code of the prefix
    __device__ __forceinline__ void run(const cplx (&yt)[NTX], double c0, int lane) {
#pragma unroll 1
        for (int p = lane; p < T::NPREF; p += 32) {
            cplx acc[NTX];
#pragma unroll
            for (int i = 0; i < NTX; ++i) acc[i] = yt[i];
            double base = c0;
            bool dead = false;
#pragma unroll
            for (int l = 0; l < T::PL; ++l) {
                const int m = (p >> (T::BITS * l)) & (T::M - 1);
                base = E::step(acc, acc, NTX - 1 - l, m, base, g, tab);
                if constexpr (PRIOR) base += pen_s(NTX - 1 - l, m);
                dead = dead || (prune && base > lim);
            }
            if (!dead) walk<NTX - 1 - T::PL>(acc, base, p);
        }
    }
};

// k_bit_llr's PRIOR_ is a pack: empty for the plain kernel (sbce_bit_llr), which keeps its name
// k_bit_llr<n_tx, sqrt M>, its parameters and its code; `true` for the a-priori kernel k_bit_llr<n_tx, sqrt M, true>
// (sbce_bit_llr_apriori), which also takes la, the a-priori LLRs in llr's layout.  A warp reads its symbol's la
// before it writes anything, so llr may be la: neither is __restrict__ (the plain kernel compiles to the same code
// without it).
template <bool>
using llr_prior = const double*;

template <int NTX, int SQM, bool... PRIOR_>
__global__ void __launch_bounds__(128) k_bit_llr(Dims d, const double* __restrict__ qr, const double* __restrict__ varn,
                                                 double* llr, llr_prior<PRIOR_>... la_) {
    constexpr bool PRIOR = (PRIOR_ || ...);
    typedef EnumT<NTX, SQM> E;
    typedef LlrT<NTX, SQM, PRIOR> T;
    extern __shared__ __align__(16) double llr_smem[];   // [4 warps][T::WS_DOUBLES]
    const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t = blockIdx.x * 4 + warp;
    if (t >= d.T_d) return;   // warp-uniform
    const size_t sidx = (size_t)b * d.T_d + t;
    double* out = llr + sidx * T::NB;
    const double* rec = qr + sidx * d.rec;

    bool finite = true;
    // PRIOR: lane i < NB holds La of bit i clamped to +-SBCE_LLR_CLAMP (+-inf -> +-32), amax the symbol's
    // largest |La|; a NaN prior makes the whole symbol NaN, like a non-finite record
    double lai = 0.0, amax = 0.0;
    if constexpr (PRIOR) {
        if (lane < T::NB) {
            const double* la[] = {la_...};
            const double raw = la[0][sidx * T::NB + lane];
            finite = !isnan(raw);
            lai = fmin(fmax(raw, -(double)SBCE_LLR_CLAMP), (double)SBCE_LLR_CLAMP);
        }
        amax = fabs(lai);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) amax = fmax(amax, shfl_xor_d(amax, o));
    }
    for (int i = lane; i < E::REC; i += 32) finite = finite && isfinite(rec[i]);
    if (!__all_sync(0xffffffffu, finite)) {
        if (lane < T::NB) out[lane] = __longlong_as_double(0x7ff8000000000000ll);   // NaN
        return;
    }

    double* ws = llr_smem + (size_t)warp * T::WS_DOUBLES;
    cplx* tab = (cplx*)(ws + T::O_TAB);
    double* g = ws + T::O_G;
    cplx yt[NTX];
    {
        cplx Rm[NTX][NTX];
#pragma unroll
        for (int i = 0; i < NTX; ++i)
#pragma unroll
            for (int j = i; j < NTX; ++j) Rm[i][j] = mk(rec[qr_rec_R(NTX, i, j)], rec[qr_rec_R(NTX, i, j) + 1]);
#pragma unroll
        for (int i = 0; i < NTX; ++i) yt[i] = mk(rec[qr_rec_yt(NTX, i)], rec[qr_rec_yt(NTX, i) + 1]);
#pragma unroll
        for (int s = 1; s < NTX; ++s)
#pragma unroll
            for (int i = 0; i < s; ++i)
                for (int m = lane; m < T::M; m += 32) tab[E::pair(i, s) * T::M + m] = cmul(Rm[i][s], E::cval(m));
        if (lane < SQM) {
#pragma unroll
            for (int s = 0; s < NTX; ++s) g[s * SQM + lane] = Rm[s][s].x * E::pam(lane);
        }
    }
    if constexpr (PRIOR) {
        // penalty tables, in distance units: varn^2 sum_i max(0, (2 bit_i - 1) La_i) over the bits of a symbol
        // (stream s >= 1) or of one PAM axis (stream 0)
        double* pen = ws + T::O_P;
        const double s2p = varn[b] * varn[b];
#pragma unroll
        for (int s = 0; s < NTX; ++s) {
            double lb[T::BITS];
#pragma unroll
            for (int i = 0; i < T::BITS; ++i) lb[i] = shfl_d(lai, s * T::BITS + i);
            if (s == 0) {
                if (lane < SQM) {
                    double PI = 0.0, PQ = 0.0;
#pragma unroll
                    for (int i = 0; i < T::HB; ++i) {
                        PI += fmax(0.0, T::bit(lane, i) ? lb[i] : -lb[i]);
                        PQ += fmax(0.0, T::bit(lane, i) ? lb[T::HB + i] : -lb[T::HB + i]);
                    }
                    pen[T::O_P0I - T::O_P + lane] = s2p * PI;
                    pen[T::O_P0Q - T::O_P + lane] = s2p * PQ;
                }
            } else {
                for (int m = lane; m < T::M; m += 32) {
                    const int iI = m & (SQM - 1), iQ = m >> T::HB;
                    double P = 0.0;
#pragma unroll
                    for (int i = 0; i < T::HB; ++i) {
                        P += fmax(0.0, T::bit(iI, i) ? lb[i] : -lb[i]);
                        P += fmax(0.0, T::bit(iQ, i) ? lb[T::HB + i] : -lb[T::HB + i]);
                    }
                    pen[(s - 1) * T::M + m] = s2p * P;
                }
            }
        }
    }
    __syncwarp();
    const double c0 = rec[qr_rec_c0(NTX)];
    const double vn = varn[b], s2 = vn * vn;

    // pass 1: exact minimum, from the Babai point (successive slicing) as incumbent
    double dmin;
    {
        LlrWalk<NTX, SQM, false, PRIOR> w;
        w.tab = tab;
        w.g = g;
        w.inv_s2 = 0.0;
        w.prune = true;
        cplx acc[NTX];
#pragma unroll
        for (int i = 0; i < NTX; ++i) acc[i] = yt[i];
        double base = c0;
#pragma unroll
        for (int s = NTX - 1; s >= 0; --s) {
            double dI, dQ;
            const int iI = E::slice(acc[s].x, g + s * SQM, dI), iQ = E::slice(acc[s].y, g + s * SQM, dQ);
            base += dI + dQ;
            if constexpr (PRIOR) {   // the plain Babai point under the full metric: any hypothesis bounds the minimum
                if (s > 0) {
                    base += w.pen_s(s, iQ * SQM + iI);
                } else {
                    base += w.pen_I()[iI];
                    base += w.pen_Q()[iQ];
                }
            }
            E::descend(acc, acc, s, iQ * SQM + iI, tab);
        }
        w.best = base;
        w.lim = base;
        w.run(yt, c0, lane);
        dmin = w.best;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dmin = fmin(dmin, shfl_xor_d(dmin, o));
    }

    // pass 2: both sides of every bit, relative to the minimum
    LlrWalk<NTX, SQM, true, PRIOR> w;
    w.tab = tab;
    w.g = g;
    w.inv_s2 = 1.0 / s2;
    w.best = dmin;
    if constexpr (PRIOR)
        w.lim = dmin + (LLR_THR + amax) * s2;   // window 96 + max |La| (include/sbce.h)
    else
        w.lim = dmin + LLR_THR * s2;
    w.prune = (d.flags & SBCE_FLAG_FULL_SCAN) == 0;
#pragma unroll
    for (int i = 0; i < T::NB; ++i) { w.s0[i] = 0.0; w.s1[i] = 0.0; }
    w.run(yt, c0, lane);

    double mine = 0.0;
#pragma unroll
    for (int i = 0; i < T::NB; ++i) {
        const double a0 = warp_sum(w.s0[i]), a1 = warp_sum(w.s1[i]);
        if (lane == i) {
            double v = log(a0) - log(a1);
            if constexpr (PRIOR) v -= lai;   // extrinsic: the posterior LLR minus the bit's own prior
            // clamp to +-SBCE_LLR_CLAMP (one side empty: +-inf -> +-32); a NaN stays NaN
            mine = v > SBCE_LLR_CLAMP ? (double)SBCE_LLR_CLAMP : (v < -SBCE_LLR_CLAMP ? -(double)SBCE_LLR_CLAMP : v);
        }
    }
    if (lane < T::NB) out[lane] = mine;
}

template <int NTX, int SQM, bool PRIOR>
static cudaError_t run_llr(const Dims& d, int nb, const double* qr, const double* varn, const double* la, double* llr,
                           cudaStream_t s) {
    constexpr int WARPS = 4;   // one symbol per warp (the kernel's launch bound is 128 threads)
    dim3 grid((d.T_d + WARPS - 1) / WARPS, nb);
    constexpr size_t smem = sizeof(double) * WARPS * LlrT<NTX, SQM, PRIOR>::WS_DOUBLES;
    static_assert(smem <= 48 * 1024, "no shared-memory opt-in");
    if constexpr (PRIOR)
        k_bit_llr<NTX, SQM, true><<<grid, WARPS * 32, smem, s>>>(d, qr, varn, llr, la);
    else
        k_bit_llr<NTX, SQM><<<grid, WARPS * 32, smem, s>>>(d, qr, varn, llr);
    count_launch();
    return cudaGetLastError();
}

template <int NTX, bool PRIOR>
static cudaError_t run_llr_ntx(const Dims& d, int nb, const double* qr, const double* varn, const double* la,
                               double* llr, cudaStream_t s) {
    switch (d.sqM) {   // enum_instantiated takes log2 M
        case 2:
            if constexpr (enum_instantiated(NTX, 2)) return run_llr<NTX, 2, PRIOR>(d, nb, qr, varn, la, llr, s);
            break;
        case 4:
            if constexpr (enum_instantiated(NTX, 4)) return run_llr<NTX, 4, PRIOR>(d, nb, qr, varn, la, llr, s);
            break;
        case 8:
            if constexpr (enum_instantiated(NTX, 6)) return run_llr<NTX, 8, PRIOR>(d, nb, qr, varn, la, llr, s);
            break;
    }
    return cudaErrorInvalidValue;
}

template <bool PRIOR>
static cudaError_t launch_llr(const Dims& d, int nb, const double* qr, const double* varn, const double* la,
                              double* llr, cudaStream_t s) {
    switch (d.n_tx) {
        case 1: return run_llr_ntx<1, PRIOR>(d, nb, qr, varn, la, llr, s);
        case 2: return run_llr_ntx<2, PRIOR>(d, nb, qr, varn, la, llr, s);
        case 3: return run_llr_ntx<3, PRIOR>(d, nb, qr, varn, la, llr, s);
        case 4: return run_llr_ntx<4, PRIOR>(d, nb, qr, varn, la, llr, s);
        case 5: return run_llr_ntx<5, PRIOR>(d, nb, qr, varn, la, llr, s);
        case 6: return run_llr_ntx<6, PRIOR>(d, nb, qr, varn, la, llr, s);
        case 7: return run_llr_ntx<7, PRIOR>(d, nb, qr, varn, la, llr, s);
        case 8: return run_llr_ntx<8, PRIOR>(d, nb, qr, varn, la, llr, s);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_bit_llr(const Dims& d, int nb, const double* qr, const double* varn, double* llr, cudaStream_t s) {
    return launch_llr<false>(d, nb, qr, varn, nullptr, llr, s);
}

cudaError_t launch_bit_llr_apriori(const Dims& d, int nb, const double* qr, const double* varn, const double* la,
                                   double* llr, cudaStream_t s) {
    return launch_llr<true>(d, nb, qr, varn, la, llr, s);
}

}  // namespace sbce
