// Shared device helpers and the internal launcher interface of libsbce.
// Everything here is FP64: the parity bar is 1e-9 relative Frobenius on theta.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/sbce.h"

namespace sbce {

typedef double2 cplx;  // .x = re, .y = im  (numpy complex128 memory)

__host__ __device__ __forceinline__ cplx mk(double re, double im) { return make_double2(re, im); }
__device__ __forceinline__ cplx cadd(cplx a, cplx b) { return mk(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ cplx csub(cplx a, cplx b) { return mk(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ cplx cmul(cplx a, cplx b) {
    return mk(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}
// a * conj(b)
__device__ __forceinline__ cplx cmulc(cplx a, cplx b) {
    return mk(fma(a.x, b.x, a.y * b.y), fma(a.y, b.x, -a.x * b.y));
}
__device__ __forceinline__ cplx cconj(cplx a) { return mk(a.x, -a.y); }
__device__ __forceinline__ cplx cscale(cplx a, double s) { return mk(a.x * s, a.y * s); }
__device__ __forceinline__ double cnorm2(cplx a) { return fma(a.x, a.x, a.y * a.y); }
// acc += a*b
__device__ __forceinline__ void cfma(cplx& acc, cplx a, cplx b) {
    acc.x = fma(a.x, b.x, acc.x);
    acc.x = fma(-a.y, b.y, acc.x);
    acc.y = fma(a.x, b.y, acc.y);
    acc.y = fma(a.y, b.x, acc.y);
}
// acc += a*conj(b)
__device__ __forceinline__ void cfmac(cplx& acc, cplx a, cplx b) {
    acc.x = fma(a.x, b.x, acc.x);
    acc.x = fma(a.y, b.y, acc.x);
    acc.y = fma(a.y, b.x, acc.y);
    acc.y = fma(-a.x, b.y, acc.y);
}
// acc -= a*conj(b)
__device__ __forceinline__ void cfmsc(cplx& acc, cplx a, cplx b) {
    acc.x = fma(-a.x, b.x, acc.x);
    acc.x = fma(-a.y, b.y, acc.x);
    acc.y = fma(-a.y, b.x, acc.y);
    acc.y = fma(a.x, b.y, acc.y);
}

__device__ __forceinline__ double shfl_xor_d(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += shfl_xor_d(v, o);
    return v;
}

constexpr int RH_MAXR = 8;   // receive antennas supported by the normal-equation / solve kernels

// Problem dimensions resolved once on the host and passed by value to kernels.
struct Dims {
    int N, N1, n_tx, n_rx, M, sqM, bitsM, T_p, T_d, itera;
    int L;      // (N+1)*n_tx
    int Lp;     // L rounded up to a multiple of 4 (micro-tile granularity of the Cholesky)
    int RP;     // n_rx rounded up to a multiple of 4 (rows that carry B^H below the matrix)
    int Ltot;   // Lp + RP rows of the augmented lower-trapezoidal normal matrix
    int mode;
    unsigned flags;
    int p1;     // PM: streams enumerated exhaustively
    int psi_shared;   // the phase matrix a kernel is handed has no batch dimension (data phases in the EM loop)
    int psiP_shared;  // ... the pilot phases (launchers of pilot-side kernels copy this into psi_shared)
    int rec;    // doubles per per-symbol QR record
};

// Per-symbol QR record written by the effective-channel kernel and consumed by
// the enumeration kernel (doubles): R upper triangle row-major, real diagonal
// stored as (d,0); then ytilde[n_tx]; then c0 stored as (c0,0).  Offsets of the
// (re, im) pair of R_ij (i <= j), of ytilde_i and of c0:
__host__ __device__ __forceinline__ constexpr int qr_rec_R(int n_tx, int i, int j) {
    return 2 * (i * n_tx - i * (i - 1) / 2 + j - i);
}
__host__ __device__ __forceinline__ constexpr int qr_rec_yt(int n_tx, int i) { return n_tx * (n_tx + 1) + 2 * i; }
__host__ __device__ __forceinline__ constexpr int qr_rec_c0(int n_tx) { return qr_rec_yt(n_tx, n_tx); }
__host__ __device__ __forceinline__ constexpr int qr_record_doubles(int n_tx) { return n_tx * (n_tx + 1) + 2 * n_tx + 2; }
static_assert(qr_rec_yt(8, 0) == qr_rec_R(8, 7, 7) + 2 && qr_rec_c0(8) + 2 == qr_record_doubles(8),
              "QR record: R, ytilde and c0 are packed back to back");

// The exhaustive tree (k_enum) is instantiated for every constellation up to 4 streams, and beyond that while
// the joint hypothesis index has at most 24 bits (8 streams of QPSK, 6 of 16-QAM).
constexpr bool enum_instantiated(int n_tx, int log2M) { return n_tx <= 4 || n_tx * log2M <= 24; }

// workspace carve-up for `nb` trials in flight
struct Workspace {
    double* stat_m;   // [nb][T_d][n_tx] cplx
    double* stat_R;   // [nb][T_d][n_tx][n_tx] cplx
    double* pil_m;    // [nb][T_p][n_tx] cplx
    double* pil_R;    // [nb][T_p][n_tx][n_tx] cplx
    double* qr;       // [nb][T_d][rec]
    double* lse_sym;  // [nb][T_d]
    double* Gp;       // [nb][Ltot][Lp] cplx  pilot part of the augmented normal matrix
    double* G;        // [nb][Ltot][Lp] cplx  working copy, overwritten by its Cholesky factor
    int32_t* active;  // [nb]
    int32_t* stat;    // [nb]
    int32_t* kscratch;// [nb][T_d]
    double* psiw;     // [nb][T_p][N+1] cplx  LS start: pilot phases with identical columns merged
    double* ls_scale; // [nb][N+1]  sqrt(multiplicity) of a kept column, 0 for a removed one
    int32_t* ls_rep;  // [nb][N+1]  representative column (-1: zero column)
    double* thbuf;    // [nb][Lp][n_rx] cplx  back-substitution vector when it does not fit in shared memory
    size_t bytes;
};

size_t carve_workspace(const Dims& d, int nb, void* base, Workspace* ws);

// ---- launchers (one translation unit each) --------------------------------
// E-step side (estep.cu)
cudaError_t launch_pilot_stats(const Dims& d, int nb, const double* Xp, double* pil_m, double* pil_R, cudaStream_t s);
cudaError_t launch_heff_qr(const Dims& d, int nb, const double* Yd, const double* PsiD, const double* theta,
                           const int32_t* active, const double* Xoff, double* qr, cudaStream_t s);
cudaError_t launch_superimpose_stats(const Dims& d, int nb, const double* Xoff, const int32_t* active, double* stat_m,
                                     double* stat_R, cudaStream_t s);
cudaError_t launch_enum(const Dims& d, int nb, const double* qr, const double* varn, const int32_t* active,
                        double* stat_m, double* stat_R, int32_t* kstar, double* lse_sym, cudaStream_t s);
// M-step side (mstep.cu)
cudaError_t launch_normal_equations(const Dims& d, int nb, const double* Psi, int T, const double* Y,
                                    const double* sm, const double* sR, const double* Ginit, double* Gout,
                                    const int32_t* active, cudaStream_t s);
bool gram_supports(int N1, int n_tx, int n_rx);   // the Gram launch of this shape fits in shared memory (mstep.cu)
cudaError_t launch_chol_solve(const Dims& d, int nb, double* G, double* theta, const int32_t* active, int32_t* stat,
                              double* th_scratch, cudaStream_t s);
// metrics (metrics.cu)
cudaError_t launch_init_state(const Dims& d, int nb, const double* theta0, double* theta, int32_t* active,
                              int32_t* stat, int32_t* iters, double* llf, double* lse, cudaStream_t s);
cudaError_t launch_after_iteration(const Dims& d, int nb, int l, const double* theta, const double* h_true,
                                   const double* Yp, const double* Yd, const double* PsiP, const double* PsiD,
                                   const double* Xp, const double* Xd_true, const double* varn, const double* lse_sym,
                                   int32_t* active, int32_t* iters, double* llf, double* lse, cudaStream_t s);
cudaError_t launch_final_metrics(const Dims& d, int nb, const double* theta, const double* h_true, const int32_t* stat,
                                 double* nmse, int32_t* status, cudaStream_t s);
cudaError_t launch_accumulate_nmse(const double* nmse, const int32_t* status, int batch, double* acc, cudaStream_t s);
cudaError_t run_fp64_peak(double* tflops, double* seconds);
// generation + LS start (gen.cu)
cudaError_t launch_generate(const Dims& d, int nb, const sbce_gen* g, const sbce_io& io, double* h_out, double* Xp_out,
                            double* Xd_out, double* PsiP_out, double* PsiD_out, double* Yp_out, double* Yd_out,
                            cudaStream_t s);
cudaError_t launch_ls_start(const Dims& d, int nb, const sbce_io& io, double* theta0, int32_t* status, Workspace& ws,
                            cudaStream_t s);
cudaError_t launch_accumulate_ser(const Dims& d, int nb, const int32_t* kstar, const double* Xd, double* acc,
                                  cudaStream_t s);

void count_launch(int n = 1);


// Opt-in to more than 48 KB of dynamic shared memory, once per (kernel instantiation, device) instead of on
// every launch of the EM loop.  Each launcher keeps one `static SmemOptIn` per kernel it launches.
struct SmemOptIn {
    std::atomic<size_t> have[64];
};
inline cudaError_t opt_in_smem(SmemOptIn& st, const void* kernel, size_t smem) {
    if (smem <= 48 * 1024) return cudaSuccess;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64 && st.have[dev].load(std::memory_order_relaxed) >= smem) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess && dev >= 0 && dev < 64) st.have[dev].store(smem, std::memory_order_relaxed);
    return e;
}

}  // namespace sbce
