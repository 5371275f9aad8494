// The hypothesis tree of one data symbol, shared by the E-step enumeration (estep.cu) and the bit LLRs
// (llr.cu): constellation and index conventions, the per-symbol shared-memory layout of k_enum, and the tree
// arithmetic on the QR record (one level's partial distance, the residual update, the PAM slicer).
#pragma once

#include "common.cuh"

namespace sbce {

template <int NTX, int SQM>
struct EnumT {
    static constexpr int M = SQM * SQM;
    static constexpr int BITS = (SQM == 2 ? 2 : (SQM == 4 ? 4 : 6));
    static constexpr int HB = BITS / 2;
    static constexpr int NODE_STREAMS = NTX - 1;
    static constexpr int PLWANT = (5 + BITS - 1) / BITS;  // prefix streams so that M^PL >= 32 (two rounds of 16)
    static constexpr int PL = NODE_STREAMS < PLWANT ? NODE_STREAMS : PLWANT;
    static constexpr int NPREF = 1 << (BITS * PL);
    static constexpr int NPAIR = NTX * (NTX - 1) / 2;
    static constexpr int NPAIR1 = NPAIR > 0 ? NPAIR : 1;
    // accumulator block (doubles): S = sum of the weights, Re m_s, Im m_s, R_ss, then (Re, Im) of R_is for i < s
    static constexpr int A_MRE = 1, A_MIM = A_MRE + NTX, A_RD = A_MIM + NTX, A_RU = A_RD + NTX;
    static constexpr int NACC = A_RU + 2 * NPAIR;
    static constexpr int REC = qr_record_doubles(NTX);
    // Lanes per symbol: a half-warp (two symbols per warp) up to 4 streams.  The deep trees of 5..8 streams keep
    // a whole warp: their halves diverge at every level, one after the other (8x8 QPSK hard: 1.04 ms per launch
    // on half-warps against 0.88 ms on warps).
    static constexpr int G = NTX > 4 ? 32 : 16;
    // Candidate queue (node codes) per symbol: 480 entries let eight 4x4 16-QAM blocks (7.1 KB each) share a
    // quarter of the SM's 228 KB (4 CTAs per SM); the warp-per-symbol kernels keep 1024.
    static constexpr int QCAP = G == 32 ? 1024 : 480;
    // the calling lane's group (its symbol's lanes) as a member mask, and the lane's index in it
    __device__ __forceinline__ static unsigned gmask() { return G == 32 ? 0xffffffffu : 0xFFFFu << (threadIdx.x & 16); }
    __device__ __forceinline__ static int glane() { return threadIdx.x & (G - 1); }
    // shift that brings the group's bits of a ballot down to bit 0
    __device__ __forceinline__ static int gshift() { return threadIdx.x & (32 - G); }
    // per-symbol shared block (doubles): tables, PAM levels, ytilde, c0, accumulators, aref, then ints
    static constexpr int O_TAB = 0;
    static constexpr int O_G = O_TAB + 2 * NPAIR1 * M;
    static constexpr int O_YT = O_G + NTX * SQM;
    static constexpr int O_C0 = O_YT + 2 * NTX;
    static constexpr int O_ACC = O_C0 + 1;
    static constexpr int O_AREF = O_ACC + NACC;
    static constexpr int O_S2 = O_AREF + 1;     // inv_s2
    static constexpr int O_Q = O_S2 + 1;        // QCAP ints = QCAP/2 doubles (the count is a group-uniform register)
    static constexpr int O_SCR = O_Q + QCAP / 2;   // [NACC][16] reduction scratch of the flush (QR record at start-up)
    static constexpr int WS_DOUBLES = ((O_SCR + NACC * G) + 1) & ~1;
    static_assert(NACC * G >= REC, "the QR record is staged in the flush scratch");
    // The queue never drops a node (a dropped node is lost silently).  Between two maybe_flush() calls a group
    // enqueues at most G nodes in a packed step (one per lane), and G*M (G*SQM per row) in a stream-1 level walked by
    // every lane for its own node; the threshold leaves room for them.  When every node stream is a prefix stream
    // there is no such call, and at most one node per prefix is queued.
    static_assert(PL < NODE_STREAMS || NPREF <= QCAP, "prefix-only trees must fit the queue without a flush");
    static_assert(G * SQM < QCAP, "maybe_flush threshold");
    // the top-level pre-pass votes with one lane per top symbol
    static_assert(PL < 2 || M <= G, "pre-pass: one lane per top symbol");

    __device__ __forceinline__ static double pam(int a) { return (double)(2 * a - SQM + 1); }
    __device__ __forceinline__ static cplx cval(int m) { return mk(pam(m & (SQM - 1)), pam(m >> HB)); }
    __device__ __forceinline__ static int pair(int i, int s) { return s * (s - 1) / 2 + i; }
    __device__ __forceinline__ static int acc_R(int i, int s) { return A_RU + 2 * pair(i, s); }   // Re R_is; Im at +1
    // symbol index of stream s in a node or hypothesis code
    __device__ __forceinline__ static int digit(int code, int s) { return (code >> (BITS * (NTX - 1 - s))) & (M - 1); }

    // One tree level, stream s taking symbol m: dist = its term of the partial distance; descend = the residuals
    // of the streams below lose R_is c_m (out may be acc); step = both, returning base + dist.
    __device__ __forceinline__ static double dist(const cplx (&acc)[NTX], int s, int m, const double* g) {
        const double* gs = g + s * SQM;
        const double eI = acc[s].x - gs[m & (SQM - 1)];
        const double eQ = acc[s].y - gs[m >> HB];
        return fma(eI, eI, eQ * eQ);
    }
    __device__ __forceinline__ static void descend(const cplx (&acc)[NTX], cplx (&out)[NTX], int s, int m,
                                                   const cplx* tab) {
#pragma unroll
        for (int i = 0; i < NTX; ++i) out[i] = (i < s) ? csub(acc[i], tab[pair(i, s) * M + m]) : acc[i];
    }
    __device__ __forceinline__ static double step(const cplx (&acc)[NTX], cplx (&out)[NTX], int s, int m, double base,
                                                  const double* g, const cplx* tab) {
        const double nb = base + dist(acc, s, m, g);
        descend(acc, out, s, m, tab);
        return nb;
    }

    // A queued node rebuilt from its code and the symbol's shared block: returns its partial distance (streams
    // NTX-1 .. 1), t0 = its residual on row 0.
    __device__ __forceinline__ static double rebuild(const double* ws, int code, cplx& t0) {
        cplx acc[NTX];
#pragma unroll
        for (int i = 0; i < NTX; ++i) acc[i] = mk(ws[O_YT + 2 * i], ws[O_YT + 2 * i + 1]);
        double base = ws[O_C0];
#pragma unroll
        for (int s = NTX - 1; s >= 1; --s)
            base = step(acc, acc, s, digit(code, s), base, ws + O_G, (const cplx*)(ws + O_TAB));
        t0 = acc[0];
        return base;
    }

    // Every statistic of one node, in accumulator order, as sink(index, value).  E0, F0, Q0: the sums over the
    // node's M leaves of the weight, of weight * conj(x_0) and of weight * |x_0|^2; x_1.. are the node's digits.
    template <class Sink>
    __device__ __forceinline__ static void node_stats(int code, double E0, cplx F0, double Q0, Sink&& sink) {
        sink(0, E0);
        sink(A_MRE, F0.x);
        sink(A_MIM, F0.y);
        sink(A_RD, Q0);
#pragma unroll
        for (int s = 1; s < NTX; ++s) {
            const cplx xs = cval(digit(code, s));
            sink(A_MRE + s, E0 * xs.x);
            sink(A_MIM + s, -E0 * xs.y);
            sink(A_RD + s, E0 * cnorm2(xs));
            const cplx v = cmul(F0, xs);  // conj(x_0) x_s summed over the leaves
            sink(acc_R(0, s), v.x);
            sink(acc_R(0, s) + 1, v.y);
#pragma unroll
            for (int i = 1; i < NTX; ++i)
                if (i < s) {
                    const cplx cx = cmulc(xs, cval(digit(code, i)));  // conj(x_i) x_s
                    sink(acc_R(i, s), E0 * cx.x);
                    sink(acc_R(i, s) + 1, E0 * cx.y);
                }
        }
    }

    // nearest PAM level to v among gs[0..SQM) (increasing), first index on ties; dist = squared distance
    __device__ __forceinline__ static int slice(double v, const double* gs, double& dist) {
        int a = 0;
        double e = v - gs[0];
        dist = e * e;
#pragma unroll
        for (int q = 1; q < SQM; ++q) {
            e = v - gs[q];
            const double dq = e * e;
            if (dq < dist) { dist = dq; a = q; }
        }
        return a;
    }

    // distance from v to the nearest level of the symmetric PAM set {+-r, +-3r, ...}: fold |v| around the
    // midpoints (for 4 levels: ||v| - 2r| - r), no comparisons, 1 + log2(SQM/2) subtractions
    __device__ __forceinline__ static double fold(double v, double r) {
        double a = fabs(v);
        if (SQM == 8) a = fabs(a - 4.0 * r);
        if (SQM >= 4) a = fabs(a - 2.0 * r);
        return a - r;
    }
};

}  // namespace sbce
