/*
 * sbce.h -- C ABI of the B200-native semi-blind EM channel estimator
 * (MIMO-RIS link, pilots + unknown QAM data).
 *
 * The reference (a directory of Python scripts) has no FFI; its de-facto
 * interface for this path is the family of estimator functions every driver
 * calls:
 *     em(Y_d,Y_p,T_d,T_p,Z_p,PsiTilde_td,all_possibleSymbols,M,varn,itera[,h_initial])
 *         /root/reference/Proposed_method_NMSEvsTp.py:43
 *         /root/reference/Proposed method/Proposed_method_NMSEvsTp.py:50
 *     em (hard decisions, + LLF / + decisions)
 *         /root/reference/Proposed method/ML_detecctor.py:51
 *         /root/reference/Proposed method/SER/log_max_SER.py:51
 *     em_ml /root/reference/Proposed method/PMvsMLvsZFvsMMSE.py:135
 *     em_pm /root/reference/Proposed method/PM.py:47, PM_beta.py:42
 * One batched entry point, sbce_em_batch(), replaces the body of all of them;
 * the Python functions with the reference's names and argument order sit on
 * top of it (package estimators.py) and INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - plain pointers and sizes only; every complex array is interleaved
 *     (re,im) float64, i.e. numpy complex128 / torch.complex128 memory, C order.
 *   - L = (N+1)*n_tx unknowns per receive antenna; the channel vector h of the
 *     reference is viewed as Theta[L][n_rx] with Theta[n'*n_tx+j][r] =
 *     h[(n'*n_tx+j)*n_rx+r]  (n'=0: direct link; Proposed method/PM.py:15).
 *   - hypothesis index k = sum_j idx_j * M^(n_tx-1-j) (itertools.product order,
 *     Proposed method/PM.py:25-31), constellation index = iQ*sqrt(M)+iI
 *     (Proposed method/QAM.py:320-322).
 *   - all calls are asynchronous on `stream` unless the name ends in _host.
 *     Process-wide state is limited to: the per-device scratch cache and streams
 *     of the *_host entry points (one mutex per device, so host threads driving
 *     different GPUs run concurrently), the launch counter (atomic) and the
 *     optional phase profiler (atomic switch, mutex-protected span list).  The
 *     *_host entry points restore the caller's current device and drain their
 *     streams on every return path, errors included.
 *   - limits: n_tx, n_rx <= 8; M in {4, 16, 64}; N + 1 + n_tx^2 <= 908 (the
 *     normal-equation kernels stage phase rows in shared memory); trials are
 *     processed in chunks of at most 65535 per launch whatever the workspace.
 *   - return value: 0 ok, <0 argument error (SBCE_E_*), >0 a cudaError_t.
 *     Per-trial numerical status is reported in status[b] (bit mask).
 */
#ifndef SBCE_H
#define SBCE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SBCE_VERSION 100

/* estimator modes */
#define SBCE_MODE_SOFT 0    /* posterior-weighted statistics (em)                         */
#define SBCE_MODE_HARD 1    /* arg-max hypothesis, rank-one statistics (em_ml / log-max)  */
#define SBCE_MODE_PM 2      /* partitioned, candidate weight 1 (Proposed method/PM.py)    */
#define SBCE_MODE_PM_BETA 3 /* partitioned, posterior over candidates (PM_beta.py)        */
#define SBCE_MODE_ZF 4      /* zero-forcing detector EM (em_zf, PMvsMLvsZFvsMMSE.py:95)   */
#define SBCE_MODE_MMSE 5    /* MMSE detector EM (em_mmse, PMvsMLvsZFvsMMSE.py:54)         */

/* flags */
#define SBCE_FLAG_GENIE_STOP 1u /* stop a trial when | ||theta|| - ||h_true|| | < 1 and l != 0 (PM.py:110)   */
#define SBCE_FLAG_QUIRKS 2u     /* PM / ZF / MMSE modes: reproduce the off-by-one psi slice (PM.py:63), the
                                   un-permuted candidate vector (PM.py:102) and the table-indexing slicer
                                   nearest_symbol_ecul (PMvsMLvsZFvsMMSE.py:49-52); cleared = corrected behaviour */
#define SBCE_FLAG_PSI_SHARED 4u /* PsiP / PsiD are shared by all trials of the batch ([T][N+1], no batch dim) */
#define SBCE_FLAG_ZERO_START 8u /* theta0 is ignored, EM starts from 0 (Proposed_method_NMSEvsTp.py:45)      */
#define SBCE_FLAG_FULL_SCAN 16u /* E-step visits every node of the hypothesis tree.  Default (flag clear): subtrees
                                   whose partial distance already exceeds the incumbent + 64 varn^2 are skipped --
                                   they could neither improve the arg-min nor enter the posterior sums, so the
                                   outputs are BIT-IDENTICAL to the full scan (tests/test_gpu_parity.py)              */

#define SBCE_FLAG_SUPERIMPOSED 32u /* parallel protocol (/root/reference/Parallel/ParallelProtocol_Tp.py:64-86): pilots are
                                   SUPERIMPOSED on the data, the hypotheses of symbol t are x_k + o_t with the known offset
                                   o_t (pilot symbol, zero beyond the pilot length), there is no separate pilot block:
                                   T_p must be 0 and io->Xp holds the offsets [B][T_d][n_tx]; soft / hard modes only */

#define SBCE_FLAG_PSIP_SHARED 64u  /* only the PILOT phases PsiP are shared by all trials ([T_p][N+1]); data phases stay per
                                   trial.  The reference's pilot designs are deterministic DFT patterns (PM.py:120-124,
                                   Proposed_method_NMSEvsTp.py:77) while its data phases are redrawn per trial (PM.py:125-129):
                                   passing the pilot design once halves the input volume of a sweep point */

#define SBCE_FLAG_ZF_STOP_GUARD 128u /* ZF mode: the genie stop also requires l != 0, as em_zf of
                                   "Proposed method/all_detectorsvsTd.py":127 has it (PMvsMLvsZFvsMMSE.py:128 does not) */

/* Pilot normal equations.  For T_p > 0 every call first checks on the device, in one pass over the T_p (N+1)(N+2)/2
 * phase products of the pilot design (once when shared, per trial otherwise, so that both layouts of one design
 * give the same bits), whether the design is a DFT design up to the error of its phases: for every t and n >= n',
 *     | conj(psi[t,n]) psi[t,n'] - conj(psi[t,lag]) | <= SBCE_PILOT_LAG_TOL_ULPS * (N+1) * 2^-53 * |psi[t,lag]|,
 *     lag = n - n' + s for n' >= 1,  lag = n for n' = 0,
 * for the shift s = 0 (psi[t,n] = w_t^n) or s = 1 (a ones column in front of w_t^0 .. w_t^(N-1), the design of
 * SBCE_PILOTS_TOP).  A NaN or Inf fails, and so does a design whose entries are not of unit (or zero) modulus, since
 * the bound is relative.  Then block (n, n') of the pilot Gram is F(lag) = sum_t conj(psi[t,lag]) R_t, N+1 distinct
 * n_tx x n_tx blocks built by one GEMM instead of a sum per pair (mstep.cu, k_pilot_lag_gram).  A design that
 * fails keeps the pair form; the choice is made on the device and is invisible to the caller.
 * The bound: a DFT phase w_t^n = exp(-2j pi t n / T_p) has an argument below 2 pi N.  Computed from that argument
 * as it stands (numpy's exp(-2j pi t n / T_p), the reference's own construction), a few roundings of it move the
 * phase by O(N) units of 2^-53: measured, the left side reaches 833 * 2^-53 at T_p = 320, N = 64 and 3329 * 2^-53
 * at T_p = 320, N = 256, i.e. 13 (N+1) units.  With the argument reduced exactly first (sbce_generate_batch:
 * sincospi(-2q/T_p), q = t n mod T_p) it stays under 21 units at any N.  The bound, 32 (N+1) units, admits both
 * constructions and no design that is further from a DFT design than its own phases' rounding makes it.  A term
 * conj(psi[t,n]) psi[t,n'] R_t of the pilot Gram then moves by at most 32 (N+1) 2^-53 |R_t| (4.6e-13 relative at
 * N = 64): the lag form gives the pilot Gram of the DFT design the input stands for, as accurately as the input
 * phases themselves determine it. */
#define SBCE_PILOT_LAG_TOL_ULPS 32

/* per-trial status bits */
/* SBCE_ST_NOT_PD: the Cholesky of the normal matrix met a pivot that is not above 1e-13 times the largest pivot
 * so far in the trial (a NaN pivot included; the identity padding rows are exempt): numerically singular M-step */
#define SBCE_ST_NOT_PD 1
#define SBCE_ST_NONFINITE 2 /* a non-finite value appeared in theta                                      */

/* argument errors */
#define SBCE_E_NULL (-1)
#define SBCE_E_SHAPE (-2)
#define SBCE_E_UNSUPPORTED (-3)
#define SBCE_E_WORKSPACE (-4)
#define SBCE_E_NODEVICE (-5)

typedef struct sbce_cfg {
    int32_t N;            /* RIS elements; phase matrices have N+1 rows (row 0 = direct link) */
    int32_t n_tx, n_rx;   /* transmit / receive antennas                                       */
    int32_t M;            /* constellation order: 4, 16 or 64                                  */
    int32_t T_p, T_d;     /* pilot / data block lengths                                        */
    int32_t itera;        /* EM iterations                                                     */
    int32_t batch;        /* trials B in this call                                             */
    int32_t mode;         /* SBCE_MODE_*                                                       */
    uint32_t flags;       /* SBCE_FLAG_*                                                       */
    int32_t partition_p1; /* PM modes: p+1 = streams enumerated exhaustively (PM.py:74-75);
                             M^(p+1) candidates per symbol, at most 2^24 (p1*log2(M) <= 24)    */
    int32_t reserved[5];
} sbce_cfg;

/* Device (or, for *_host entry points, host) buffers of one batch.  Shapes in
 * elements of complex128 unless stated; nullable ones are marked. */
typedef struct sbce_io {
    const double* Yd;      /* [B][T_d][n_rx]                                                   */
    const double* Yp;      /* [B][T_p][n_rx]                                                   */
    const double* PsiD;    /* [B][T_d][N+1]  (or [T_d][N+1] with SBCE_FLAG_PSI_SHARED)          */
    const double* PsiP;    /* [B][T_p][N+1]  (or [T_p][N+1] with SBCE_FLAG_PSI_SHARED / _PSIP_SHARED) */
    const double* Xp;      /* [B][T_p][n_tx] pilot symbols  ([B][T_d][n_tx] offsets with SBCE_FLAG_SUPERIMPOSED) */
    const double* theta0;  /* [B][L][n_rx]   start point; nullable with SBCE_FLAG_ZERO_START   */
    const double* varn;    /* [B] float64 -- the E-step divides by varn^2 (reference quirk Q1) */
    const double* h_true;  /* [B][L][n_rx]   nullable: needed for nmse[] and the genie stop    */
    const double* Xd_true; /* [B][T_d][n_tx] nullable: needed for llf[] (as-coded LLF)         */
    double* theta;         /* [B][L][n_rx]   out                                               */
    int32_t* kstar;        /* [B][T_d] int32 out, nullable: decisions of the last executed
                              iteration, made before its M-step (SER/log_max_SER.py:77-78);
                              -1 in the PM / PM_BETA modes, which take no joint decision        */
    double* llf;           /* [B][itera] float64 out, nullable: LLF exactly as coded
                              (ML_detecctor.py:84); entries of skipped iterations are NaN      */
    double* lse;           /* [B][itera] float64 out, nullable: sum_t log sum_k exp(-d2/varn^2)
                              at the theta that entered the iteration (SOFT / HARD modes; NaN
                              in the PM, ZF and MMSE modes, which never form the sum)           */
    double* nmse;          /* [B] float64 out, nullable (needs h_true)                         */
    int32_t* iters;        /* [B] int32 out, nullable: iterations executed                     */
    int32_t* status;       /* [B] int32 out, nullable: SBCE_ST_* bit mask                      */
} sbce_io;

/* library / device probes */
int sbce_version(void);
const char* sbce_error_string(int code);
int sbce_device_count(void);

/* Bytes of device workspace needed to keep `trials_in_flight` trials of `cfg`
 * in flight (cfg->batch is ignored).  sbce_em_batch() processes the batch in
 * chunks of as many trials as the workspace it is given can hold. */
int sbce_workspace_bytes(const sbce_cfg* cfg, int32_t trials_in_flight, size_t* bytes);

/* The hot path: `itera` EM iterations for every trial of the batch.
 * All pointers in `io` are DEVICE pointers; `stream` is a cudaStream_t. */
int sbce_em_batch(const sbce_cfg* cfg, const sbce_io* io, void* workspace, size_t workspace_bytes,
                  void* stream);

/* Same, with HOST pointers in `io`: stages through pinned memory, copies
 * host->device, runs sbce_em_batch on an internal stream, copies the outputs
 * back and synchronises.  `device` selects the GPU. */
int sbce_em_batch_host(const sbce_cfg* cfg, const sbce_io* io, int32_t device);

/* Batch size from which sbce_em_batch_host() pipelines a call in two halves (the upload of the
 * second half overlaps the kernels of the first). */
int sbce_host_split_threshold(void);

/* Stand-alone E-step sweep (posterior statistics at a given theta), device
 * pointers.  stat_m [B][T_d][n_tx], stat_R [B][T_d][n_tx][n_tx] complex128,
 * kstar [B][T_d] int32 (nullable), lse_sym [B][T_d] float64 (nullable).
 * Uses cfg->mode exactly as the EM loop does; as there, kstar is -1 in the PM / PM_BETA
 * modes and lse_sym is NaN in the PM, PM_BETA, ZF and MMSE modes.
 * Scale: the soft and hard statistics, kstar and lse_sym depend on (Yd, theta, varn) only through d2/varn^2, and
 * scaling all three by 2^k leaves every output bit unchanged as long as every d2, varn^2 and 1/varn^2 stays a
 * normal FP64 number below 1e300 (the E-step's initial reference distance and slicer sentinels).  The bit LLRs
 * (sbce_bit_llr, sbce_bit_llr_apriori with La unscaled) share that property. */
int sbce_estep(const sbce_cfg* cfg, const sbce_io* io, const double* theta, double* stat_m,
               double* stat_R, int32_t* kstar, double* lse_sym, void* workspace,
               size_t workspace_bytes, void* stream);

/* Stand-alone M-step (normal-equation build + Cholesky solve) from given data
 * statistics; pilots enter with probability-one statistics.  theta_out [B][L][n_rx]. */
int sbce_mstep(const sbce_cfg* cfg, const sbce_io* io, const double* stat_m, const double* stat_R,
               double* theta_out, int32_t* status, void* workspace, size_t workspace_bytes,
               void* stream);

/* Per-sweep-point accumulation used before the cross-GPU sum:
 * acc[0] += sum_b nmse[b] over trials with status==0, acc[1] += their count,
 * acc[2] += count of trials with status!=0.  acc is 3 float64 on the device. */
int sbce_accumulate_nmse(const double* nmse, const int32_t* status, int32_t batch, double* acc,
                         void* stream);

/* ---- on-device input generation and LS start (the step right before the hot path) ------------------
 * Replaces, for Monte-Carlo sweeps, the reference's per-trial host generation
 *     channelMatrix / symbols / pilotSymbols   /root/reference/Proposed method/PM.py:11-40
 *     irsMatrix (+ inserted ones row)          /root/reference/Proposed method/PM.py:119-130,179
 *     receivedSignals (Y = Z h + n, h_initial) /root/reference/Proposed method/PM.py:132-148
 * Counter-based Philox4x32-10 keyed by `seed`; element e of array a of global trial (trial0 + b) is
 * Philox(counter = (e, a, trial), key = seed), so results do not depend on batch size or sharding
 * (oracle/philox.py restates the generator in numpy; symbol indices are bit-exact). */
#define SBCE_PILOTS_PM 0     /* exp(-j2pi t n/N), n<N, in rows 0..N-1, row N zero (PM.py:120-124)                */
#define SBCE_PILOTS_TOP 1    /* ones row + exp(-j2pi t n/T_p) (Proposed_method_NMSEvsTp.py:72-83,129)           */
#define SBCE_PHASES_RANDOM 0 /* ones row + exp(j U(0,2pi)) per (trial, symbol, element) (PM.py:125-129,179)     */
#define SBCE_PHASES_DFT 1    /* exp(-j2pi t n/T_d) over n = 0..N (Proposed_method_NMSEvsTd.py:92-94)            */

typedef struct sbce_gen {
    uint64_t seed;        /* Philox key                                                        */
    int64_t trial0;       /* global index of the first trial of this batch (disjoint per rank) */
    int32_t pilot_design; /* SBCE_PILOTS_*                                                     */
    int32_t data_phases;  /* SBCE_PHASES_*                                                     */
    double varh;          /* channel variance (reference: 1)                                   */
    int32_t no_direct_link; /* 1: every one of the cfg->N + 1 phase rows is a RIS element (no ones row, no H_BU):
                               "Proposed method/direct vs non direct - T_pv s nmse.py":11-18,108-120               */
    int32_t reserved[3];
} sbce_gen;

/* Fills the caller's DEVICE buffers io->h_true, Xp, Xd_true, PsiP, PsiD, Yp, Yd (declared const in
 * sbce_io because the estimator only reads them; here they are written) for cfg->batch trials;
 * reads io->varn [B].  With SBCE_FLAG_PSI_SHARED the phase arrays have no batch dimension. */
int sbce_generate_batch(const sbce_cfg* cfg, const sbce_gen* gen, const sbce_io* io, void* stream);

/* LS start h_initial = pinv(Z_p) y_p (PM.py:147) for every trial: min-norm solution through the
 * T_p x T_p Gram (Psi Psi^H) o (X X^H) when T_p < L, pilot normal equations when T_p >= L.
 * Reads io->Yp, PsiP, Xp; writes theta0 [B][L][n_rx]; status (nullable) gets SBCE_ST_NOT_PD for
 * rank-deficient pilot blocks (where pinv would invert rounding noise): a Cholesky pivot not above 1e-13 times the
 * largest pivot so far, NaN included.  Workspace as sbce_em_batch. */
int sbce_ls_start(const sbce_cfg* cfg, const sbce_io* io, double* theta0, int32_t* status, void* workspace,
                  size_t workspace_bytes, void* stream);

/* Symbol-error accumulation for the SER drivers (SER/log_max_SER.py:162): acc[0] += per-stream symbol
 * errors, acc[1] += symbols compared, acc[2] += sum over trials of the as-coded SER (the reference's
 * (T,n,1)-(T,1,n) broadcast).  kstar [B][T_d] int32, Xd_true [B][T_d][n_tx] complex128, acc 3 float64. */
int sbce_accumulate_ser(const sbce_cfg* cfg, const int32_t* kstar, const double* Xd_true, int32_t batch, double* acc,
                        void* stream);

/* ---- bit level: exact Gray-labelled bit LLRs at a channel estimate, and bit-error counts ----------------
 * Labelling.  Constellation index m = iQ*sqrt(M) + iI; with q = log2 sqrt(M) and gray(a) = a ^ (a >> 1), the
 * log2 M bits of m are gray(iI) MSB first, then gray(iQ) MSB first (QPSK: [iI, iQ], bit 0 <-> level -1).
 * Adjacent PAM levels differ in one bit on each axis.  The reference's vendored QAM.py carries a labelling
 * of its own that no script uses, so no reference output pins this one.
 *
 * LLR.  llr[b][t][j][i] = ln sum_{k: bit i of stream j = 0} exp(-d2_k/varn^2)
 *                       - ln sum_{k: bit i of stream j = 1} exp(-d2_k/varn^2),
 * float64, [B][T_d][n_tx][log2 M]; positive means 0 is more likely, hard bit = (llr < 0).  The prior is
 * uniform and the exponent is the E-step's own d2/varn^2 (quirk Q1), so these are the LLRs of the posterior
 * the EM iterates on; a caller who wants the exponent d2/varn passes sqrt(varn).
 *
 * Window and clamp.  The walk skips subtrees whose partial distance exceeds min_k d2_k + 96 varn^2, and the
 * result is clamped to [-SBCE_LLR_CLAMP, SBCE_LLR_CLAMP].  Weights are measured relative to the best
 * hypothesis (weight 1).  With K <= 2^24 hypotheses the skipped part of either sum is at most K e^-96; the
 * larger side holds at least half the total, so at least 1/2, and whenever the true |llr| < 32 the smaller
 * side holds at least e^-32 / 2.  The relative error of either sum, hence the absolute error of the LLR, is
 * below 2 * 2^24 * e^-64 < 1e-20 -- the same e^-64 margin the E-step's window gives its sums.  Whenever the
 * true |llr| >= 32 the result is exactly +-32.  SBCE_FLAG_FULL_SCAN disables the window.
 *
 * Every LLR of a symbol whose QR record (effective channel and observation) is not finite is NaN, not a
 * clamp; no other symbol or trial changes. */
#define SBCE_LLR_CLAMP 32

/* Bit LLRs of every data symbol at `theta` (device pointers): reads io->Yd, PsiD, varn, and io->Xp (the
 * offsets) with SBCE_FLAG_SUPERIMPOSED, whose LLRs are those of the data bits.  Honours SBCE_FLAG_PSI_SHARED
 * and SBCE_FLAG_FULL_SCAN.  cfg->mode must be SBCE_MODE_SOFT or SBCE_MODE_HARD (both give the same LLRs);
 * the shapes are those of the exhaustive tree (1-4 streams of 4/16/64-QAM, 5-8 of QPSK, 5-6 of 16-QAM: at
 * most 24 LLRs per symbol).  llr [B][T_d][n_tx][log2 M] float64.  Workspace as the E-step's. */
int sbce_bit_llr(const sbce_cfg* cfg, const sbce_io* io, const double* theta, double* llr, void* workspace,
                 size_t workspace_bytes, void* stream);

/* ---- bit LLRs with a-priori input: extrinsic LLRs for iterative detection and decoding -----------------
 * A-priori LLRs.  La[b][t][j][i] = ln P(bit = 0) - ln P(bit = 1) from a channel decoder, in the layout and
 * labelling of llr; on read each is clamped to +-SBCE_LLR_CLAMP (an infinite prior counts as +-32).
 *
 * Metric.  A bit taking value v costs pen(v) = max(0, (2v - 1) La): nothing when it agrees with the prior's
 * hard decision, |La| when it does not.  Stream j's symbol m costs P_j(m) = sum_i pen(bit_i(m)) >= 0, and
 * min_m P_j(m) = 0 since the labelling is a bijection onto all bit patterns.  Hypothesis k has the metric
 *     mu_k = d2_k + varn^2 sum_j P_j(x_j),
 * and exp(-mu_k/varn^2) is its posterior under the prior up to a constant.  The penalties are non-negative and
 * belong to single tree levels, so partial metrics stay lower bounds along the tree; and since the Gray label
 * puts the in-phase bits on iI and the quadrature bits on iQ, P_0(m) = P_0I(iI) + P_0Q(iQ) and stream 0 keeps
 * its closed form as separable in-phase / quadrature PAM weights.
 *
 * Extrinsic LLR.  llr_ext = ln S0 - ln S1 - La (La clamped), clamped to [-SBCE_LLR_CLAMP, SBCE_LLR_CLAMP], where
 * S0, S1 are both sides of the bit under mu, each accumulated explicitly.  An empty side gives +-inf before the
 * clamp, so exactly +-32.  With La = 0 this is sbce_bit_llr bit for bit: extrinsic and a-posteriori LLRs
 * coincide without a prior.
 *
 * Window.  The walk skips subtrees whose partial metric exceeds min_k mu_k + (96 + A) varn^2, A the largest
 * clamped |La| of the symbol (A = 0: sbce_bit_llr's window).  Whenever the true |llr_ext| < 32, the posterior
 * LLR is below 32 + A in magnitude, so the smaller side holds at least e^-(32+A) / 2 of the best hypothesis's
 * weight while the skipped part is at most K e^-(96+A), K <= 2^24: the relative error of either sum, hence the
 * absolute error of llr_ext, is again below 2 * 2^24 * e^-64 < 1e-20.  A side the window leaves empty holds
 * at most K e^-(96+A) against at least 1 on the other, so the posterior LLR exceeds 96 + A - ln 2^24 in
 * magnitude, |llr_ext| > 78, and the clamp makes the result exactly +-32.
 * SBCE_FLAG_FULL_SCAN disables the window.
 *
 * Non-finite input.  A NaN anywhere in a symbol's La, like a non-finite QR record, makes all of that symbol's
 * outputs NaN; no other symbol changes. */

/* sbce_bit_llr with a-priori LLRs llr_a (required) -> extrinsic LLRs llr_ext, both [B][T_d][n_tx][log2 M]
 * float64 on the device.  Checks, shapes, modes, flags (SBCE_FLAG_PSI_SHARED, SBCE_FLAG_FULL_SCAN,
 * SBCE_FLAG_SUPERIMPOSED), chunking and workspace are those of sbce_bit_llr.  llr_ext may be llr_a: each
 * symbol's priors are read before its outputs are written, so a turbo loop can update its LLRs in place. */
int sbce_bit_llr_apriori(const sbce_cfg* cfg, const sbce_io* io, const double* theta, const double* llr_a,
                         double* llr_ext, void* workspace, size_t workspace_bytes, void* stream);

/* Bit-error accumulation for the BER curves: acc[0] += bit errors between the labels of the kstar digits
 * and of Xd_true, acc[1] += bits compared.  Same arguments and limits as sbce_accumulate_ser; acc is 2
 * float64 on the device. */
int sbce_accumulate_ber(const sbce_cfg* cfg, const int32_t* kstar, const double* Xd_true, int32_t batch, double* acc,
                        void* stream);

/* Measured FP64 FMA throughput of the current device (TFLOP/s, 2 flops per
 * FMA), used as the roofline denominator for the FP64-bound kernels. */
int sbce_measure_fp64_peak(double* tflops, double* seconds);

/* Per-phase device timing (CUDA events on the launch stream around every phase of
 * sbce_em_batch), used by bench.py for the per-kernel roofline numbers.
 * sbce_profile_begin() arms it; sbce_profile_end() disarms, synchronises and returns
 * the summed milliseconds and the number of timed launches per phase. */
#define SBCE_PHASE_SETUP 0   /* state init + pilot normal equations (once per call)      */
#define SBCE_PHASE_HEFF_QR 1 /* effective channel + Householder QR (one lane per symbol) */
#define SBCE_PHASE_ENUM 2    /* hypothesis-tree posterior sweep (one warp per symbol)    */
#define SBCE_PHASE_GRAM 3    /* Hermitian normal-matrix build                            */
#define SBCE_PHASE_RHS 4     /* right-hand side rows + padding                           */
#define SBCE_PHASE_CHOL 5    /* blocked Cholesky + triangular solves                     */
#define SBCE_PHASE_METRICS 6 /* per-iteration bookkeeping, LLF, NMSE                     */
#define SBCE_N_PHASES 7
int sbce_profile_begin(void);
int sbce_profile_end(double* ms_per_phase, int64_t* spans_per_phase, int32_t n_phases);

/* Number of kernels this library launched since the last reset (for bench.py's
 * gpu_launches claim). */
int64_t sbce_launch_count(int32_t reset);

#ifdef __cplusplus
}
#endif
#endif /* SBCE_H */
