// C ABI of libsbce (declared in include/sbce.h): argument validation, workspace
// carve-up, chunking of the batch, and the kernel schedule of the EM loop.
#include <atomic>
#include <mutex>
#include <vector>
#include <stdio.h>
#include <string.h>

#include "common.cuh"

namespace sbce {

static std::atomic<long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- optional per-phase CUDA-event timing (bench.py's roofline numbers) --------------------------
// Events are recorded on the launch stream around every phase while profiling is on; the cost is one
// cudaEventRecord pair per phase launch.  sbce_profile_end() synchronises and sums the intervals.
// The switch is an atomic; the span list and the event pool are only touched under g_prof_mu, so concurrent
// callers (one host thread per GPU) may run with profiling armed.
struct PhaseSpan { int phase; cudaEvent_t a, b; };
static std::atomic<bool> g_prof_on{false};
static std::vector<PhaseSpan> g_spans;
static std::vector<cudaEvent_t> g_event_pool;
static std::mutex g_prof_mu;

static cudaEvent_t prof_event() {
    {
        std::lock_guard<std::mutex> lock(g_prof_mu);
        if (!g_event_pool.empty()) { cudaEvent_t e = g_event_pool.back(); g_event_pool.pop_back(); return e; }
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

struct PhaseScope {
    bool on; int phase; cudaStream_t s; cudaEvent_t a;
    PhaseScope(int ph, cudaStream_t st) : on(g_prof_on.load(std::memory_order_relaxed)), phase(ph), s(st), a(nullptr) {
        if (on) { a = prof_event(); cudaEventRecord(a, s); }
    }
    ~PhaseScope() {
        if (on) {
            cudaEvent_t b = prof_event();
            cudaEventRecord(b, s);
            std::lock_guard<std::mutex> lock(g_prof_mu);
            g_spans.push_back({phase, a, b});
        }
    }
};

static int make_dims(const sbce_cfg* c, Dims* d, bool with_estep = true) {
    if (!c) return SBCE_E_NULL;
    if (c->N < 1 || c->n_tx < 1 || c->n_rx < 1 || c->T_p < 0 || c->T_d < 1 || c->itera < 0 || c->batch < 0)
        return SBCE_E_SHAPE;
    int sq = 0;
    if (c->M == 4) sq = 2; else if (c->M == 16) sq = 4; else if (c->M == 64) sq = 8; else return SBCE_E_UNSUPPORTED;
    if (c->n_tx > 8 || c->n_rx > 8) return SBCE_E_UNSUPPORTED;
    // the normal-equation kernels stage chunks of the phase rows in shared memory; gram_supports() is the same
    // size computation the Gram launchers use (mstep.cu: gram_smem)
    if (!gram_supports(c->N + 1, c->n_tx, c->n_rx)) return SBCE_E_UNSUPPORTED;
    if (c->n_tx <= 4 && !(c->n_rx <= 4 || c->n_rx == 6 || c->n_rx == 8)) return SBCE_E_UNSUPPORTED;
    if (c->mode < SBCE_MODE_SOFT || c->mode > SBCE_MODE_MMSE) return SBCE_E_UNSUPPORTED;
    if (with_estep) {
        // joint hypothesis indices are int32 (kstar); the exhaustive tree is instantiated up to 2^24 leaves
        // for the wide arrays (8 streams of QPSK, 6 of 16-QAM) -- beyond that use the partitioned modes
        const int log2M = sq == 2 ? 2 : (sq == 4 ? 4 : 6), bits = c->n_tx * log2M;
        const bool tree = c->mode == SBCE_MODE_SOFT || c->mode == SBCE_MODE_HARD;
        if (tree && !enum_instantiated(c->n_tx, log2M)) return SBCE_E_UNSUPPORTED;
        if ((c->mode == SBCE_MODE_ZF || c->mode == SBCE_MODE_MMSE) && bits > 30) return SBCE_E_UNSUPPORTED;
    }
    d->N = c->N; d->N1 = c->N + 1; d->n_tx = c->n_tx; d->n_rx = c->n_rx; d->M = c->M; d->sqM = sq;
    d->bitsM = (sq == 2 ? 2 : (sq == 4 ? 4 : 6));
    d->T_p = c->T_p; d->T_d = c->T_d; d->itera = c->itera;
    d->L = d->N1 * c->n_tx;
    d->Lp = (d->L + 7) & ~7;   // rows of the factor start on 128-byte lines (chol.cu loads 8-column steps as one line)
    d->RP = (c->n_rx + 3) & ~3;
    d->Ltot = d->Lp + d->RP;
    d->mode = c->mode; d->flags = c->flags; d->p1 = c->partition_p1;
    d->psi_shared = (c->flags & SBCE_FLAG_PSI_SHARED) ? 1 : 0;
    d->psiP_shared = (c->flags & (SBCE_FLAG_PSI_SHARED | SBCE_FLAG_PSIP_SHARED)) ? 1 : 0;
    d->rec = qr_record_doubles(c->n_tx);
    if (c->mode == SBCE_MODE_PM || c->mode == SBCE_MODE_PM_BETA) {
        if (c->partition_p1 < 1 || c->partition_p1 > c->n_tx) return SBCE_E_SHAPE;
        // M^p1 candidates per symbol (an int in k_pm_stats): the same 2^24 bound as the exhaustive tree
        if (with_estep && c->partition_p1 * d->bitsM > 24) return SBCE_E_UNSUPPORTED;
    }
    if (c->mode >= SBCE_MODE_PM && c->n_rx < c->n_tx) return SBCE_E_UNSUPPORTED;
    if (c->flags & SBCE_FLAG_SUPERIMPOSED) {
        if (c->T_p != 0) return SBCE_E_SHAPE;
        if (c->mode != SBCE_MODE_SOFT && c->mode != SBCE_MODE_HARD) return SBCE_E_UNSUPPORTED;
    }
    return 0;
}

static inline size_t al(size_t x) { return (x + 255) & ~(size_t)255; }

size_t carve_workspace(const Dims& d, int nb, void* base, Workspace* ws) {
    size_t off = 0;
    char* p = (char*)base;
    auto take = [&](size_t bytes) { char* r = p ? p + off : nullptr; off += al(bytes); return r; };
    const size_t B = (size_t)nb;
    ws->stat_m = (double*)take(B * d.T_d * d.n_tx * 16);
    ws->stat_R = (double*)take(B * d.T_d * d.n_tx * d.n_tx * 16);
    ws->pil_m = (double*)take(B * d.T_p * d.n_tx * 16 + 16);
    ws->pil_R = (double*)take(B * d.T_p * d.n_tx * d.n_tx * 16 + 16);
    ws->qr = (double*)take(B * d.T_d * d.rec * 8);
    ws->lse_sym = (double*)take(B * d.T_d * 8);
    ws->Gp = (double*)take(B * d.Ltot * d.Lp * 16);
    ws->G = (double*)take(B * d.Ltot * d.Lp * 16);
    ws->active = (int32_t*)take(B * 4);
    ws->stat = (int32_t*)take(B * 4);
    ws->kscratch = (int32_t*)take(B * d.T_d * 4);
    ws->thbuf = (double*)take(B * d.Lp * d.n_rx * 16);
    ws->psiw = (double*)take(B * d.T_p * d.N1 * 16 + 16);
    ws->ls_scale = (double*)take(B * d.N1 * 8);
    ws->ls_rep = (int32_t*)take(B * d.N1 * 4);
    ws->bytes = off;
    return off;
}

#define CK(x)                                  \
    do {                                       \
        cudaError_t _e = (x);                  \
        if (_e != cudaSuccess) return (int)_e; \
    } while (0)

// forward declaration (pm.cu)
cudaError_t launch_pm_stats(const Dims& d, int nb, const double* Yd, const double* PsiD, const double* theta,
                            const double* varn, const int32_t* active, double* stat_m, double* stat_R,
                            int32_t* kstar, cudaStream_t s);

static int estep_dispatch(const Dims& d, int nb, const double* Yd, const double* PsiD, const double* theta,
                          const double* varn, const int32_t* active, Workspace& ws, double* stat_m, double* stat_R,
                          int32_t* kstar, double* lse_sym, const double* Xoff, cudaStream_t s) {
    if (d.mode == SBCE_MODE_SOFT || d.mode == SBCE_MODE_HARD) {
        {
            PhaseScope ps(SBCE_PHASE_HEFF_QR, s);
            CK(launch_heff_qr(d, nb, Yd, PsiD, theta, active, Xoff, ws.qr, s));
        }
        {
            PhaseScope ps(SBCE_PHASE_ENUM, s);
            CK(launch_enum(d, nb, ws.qr, varn, active, stat_m, stat_R, kstar, lse_sym, s));
            if (Xoff) CK(launch_superimpose_stats(d, nb, Xoff, active, stat_m, stat_R, s));
        }
    } else {
        PhaseScope ps(SBCE_PHASE_ENUM, s);
        CK(launch_pm_stats(d, nb, Yd, PsiD, theta, varn, active, stat_m, stat_R, kstar, s));
    }
    return 0;
}

// dims as seen by kernels that are handed the PILOT phase matrix
static inline Dims pilot_dims(const Dims& d) { Dims dp = d; dp.psi_shared = d.psiP_shared; return dp; }

static int em_chunk(const Dims& d, int nb, const sbce_io& io, Workspace& ws, cudaStream_t s) {
    // Only the exhaustive modes produce a per-symbol log-sum (lse) and, with the detector modes, joint decisions
    // (kstar).  The partitioned modes write neither: kstar reads -1 and lse stays NaN instead of leaking whatever
    // the buffers held.
    const bool tree = d.mode == SBCE_MODE_SOFT || d.mode == SBCE_MODE_HARD;
    const bool decides = tree || d.mode == SBCE_MODE_ZF || d.mode == SBCE_MODE_MMSE;
    if (io.kstar && !decides) CK(cudaMemsetAsync(io.kstar, 0xFF, (size_t)nb * d.T_d * sizeof(int32_t), s));
    {
        PhaseScope ps(SBCE_PHASE_SETUP, s);
        CK(launch_init_state(d, nb, io.theta0, io.theta, ws.active, ws.stat, io.iters, io.llf, io.lse, s));
        // pilot part of the normal equations, once (the reference recomputes it every iteration:
        // Proposed_method_NMSEvsTp.py:63-65)
        CK(launch_pilot_stats(d, nb, io.Xp, ws.pil_m, ws.pil_R, s));
        CK(launch_normal_equations(pilot_dims(d), nb, io.PsiP, d.T_p, io.Yp, ws.pil_m, ws.pil_R, nullptr, ws.Gp, nullptr, s));
    }
    for (int l = 0; l < d.itera; ++l) {
        int rc = estep_dispatch(d, nb, io.Yd, io.PsiD, io.theta, io.varn, ws.active, ws, ws.stat_m, ws.stat_R,
                                io.kstar, ws.lse_sym, (d.flags & SBCE_FLAG_SUPERIMPOSED) ? io.Xp : nullptr, s);
        if (rc) return rc;
        {
            PhaseScope ps(SBCE_PHASE_GRAM, s);
            CK(launch_normal_equations(d, nb, io.PsiD, d.T_d, io.Yd, ws.stat_m, ws.stat_R, ws.Gp, ws.G, ws.active,
                                       s));
        }
        {
            PhaseScope ps(SBCE_PHASE_CHOL, s);
            CK(launch_chol_solve(d, nb, ws.G, io.theta, ws.active, ws.stat, ws.thbuf, s));
        }
        {
            PhaseScope ps(SBCE_PHASE_METRICS, s);
            CK(launch_after_iteration(d, nb, l, io.theta, io.h_true, io.Yp, io.Yd, io.PsiP, io.PsiD, io.Xp,
                                      io.Xd_true, io.varn, tree ? ws.lse_sym : nullptr, ws.active, io.iters, io.llf,
                                      io.lse, s));
        }
    }
    {
        PhaseScope ps(SBCE_PHASE_METRICS, s);
        CK(launch_final_metrics(d, nb, io.theta, io.h_true, ws.stat, io.nmse, io.status, s));
    }
    return 0;
}

static sbce_io offset_io(const Dims& d, const sbce_io& io, size_t b0) {
    sbce_io o = io;
    const size_t Ln = (size_t)d.L * d.n_rx * 2;
    auto adv = [](const double* p, size_t n) { return p ? p + n : p; };
    auto advw = [](double* p, size_t n) { return p ? p + n : p; };
    o.Yd = adv(io.Yd, b0 * d.T_d * d.n_rx * 2);
    o.Yp = adv(io.Yp, b0 * d.T_p * d.n_rx * 2);
    if (!d.psi_shared) o.PsiD = adv(io.PsiD, b0 * d.T_d * d.N1 * 2);
    if (!d.psiP_shared) o.PsiP = adv(io.PsiP, b0 * d.T_p * d.N1 * 2);
    o.Xp = adv(io.Xp, b0 * ((d.flags & SBCE_FLAG_SUPERIMPOSED) ? d.T_d : d.T_p) * d.n_tx * 2);
    o.theta0 = adv(io.theta0, b0 * Ln);
    o.varn = adv(io.varn, b0);
    o.h_true = adv(io.h_true, b0 * Ln);
    o.Xd_true = adv(io.Xd_true, b0 * d.T_d * d.n_tx * 2);
    o.theta = advw(io.theta, b0 * Ln);
    o.kstar = io.kstar ? io.kstar + b0 * d.T_d : nullptr;
    o.llf = advw(io.llf, b0 * d.itera);
    o.lse = advw(io.lse, b0 * d.itera);
    o.nmse = advw(io.nmse, b0);
    o.iters = io.iters ? io.iters + b0 : nullptr;
    o.status = io.status ? io.status + b0 : nullptr;
    return o;
}

static int check_io(const Dims& d, const sbce_io* io) {
    if (!io) return SBCE_E_NULL;
    if (!io->Yd || !io->PsiD || !io->varn || !io->theta) return SBCE_E_NULL;
    if (d.T_p > 0 && (!io->Yp || !io->PsiP || !io->Xp)) return SBCE_E_NULL;
    if (!(d.flags & SBCE_FLAG_ZERO_START) && !io->theta0) return SBCE_E_NULL;
    if ((d.flags & SBCE_FLAG_GENIE_STOP) && !io->h_true) return SBCE_E_NULL;
    if ((d.flags & SBCE_FLAG_SUPERIMPOSED) && !io->Xp) return SBCE_E_NULL;
    return 0;
}

}  // namespace sbce

using namespace sbce;

extern "C" {

int sbce_version(void) { return SBCE_VERSION; }

const char* sbce_error_string(int code) {
    switch (code) {
        case 0: return "ok";
        case SBCE_E_NULL: return "required pointer is null";
        case SBCE_E_SHAPE: return "invalid shape parameter";
        case SBCE_E_UNSUPPORTED: return "unsupported configuration (n_tx,n_rx<=8; n_tx<=4: n_rx in {1,2,3,4,6,8}; M in {4,16,64}; N+1+n_tx^2<=908; exhaustive modes with n_tx>4 need n_tx*log2(M)<=24; PM modes need partition_p1*log2(M)<=24)";
        case SBCE_E_WORKSPACE: return "workspace too small for one trial";
        case SBCE_E_NODEVICE: return "no CUDA device";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

int sbce_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int sbce_workspace_bytes(const sbce_cfg* cfg, int32_t trials_in_flight, size_t* bytes) {
    Dims d;
    int rc = make_dims(cfg, &d);
    if (rc) return rc;
    if (!bytes) return SBCE_E_NULL;
    if (trials_in_flight < 1) return SBCE_E_SHAPE;
    Workspace ws;
    *bytes = carve_workspace(d, trials_in_flight, nullptr, &ws);
    return 0;
}

// Trials per chunk: as many as the workspace holds, at most `want`, and at most 65535 -- the chunk size is
// gridDim.y of the Gram / E-step / generator launches.
constexpr int SBCE_MAX_CHUNK = 65535;
static int trials_fitting(const Dims& d, size_t bytes, int want) {
    Workspace ws;
    if (want > SBCE_MAX_CHUNK) want = SBCE_MAX_CHUNK;
    if (carve_workspace(d, 1, nullptr, &ws) > bytes) return 0;
    int lo = 1, hi = want;
    while (lo < hi) {
        int mid = (lo + hi + 1) / 2;
        if (carve_workspace(d, mid, nullptr, &ws) <= bytes) lo = mid; else hi = mid - 1;
    }
    return lo;
}

int sbce_em_batch(const sbce_cfg* cfg, const sbce_io* io, void* workspace, size_t workspace_bytes, void* stream) {
    Dims d;
    int rc = make_dims(cfg, &d);
    if (rc) return rc;
    rc = check_io(d, io);
    if (rc) return rc;
    if (cfg->batch == 0) return 0;
    if (!workspace) return SBCE_E_NULL;
    const int chunk = trials_fitting(d, workspace_bytes, cfg->batch);
    if (chunk < 1) return SBCE_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    for (int b0 = 0; b0 < cfg->batch; b0 += chunk) {
        const int nb = (cfg->batch - b0 < chunk) ? cfg->batch - b0 : chunk;
        Workspace ws;
        carve_workspace(d, nb, workspace, &ws);
        sbce_io o = offset_io(d, *io, (size_t)b0);
        rc = em_chunk(d, nb, o, ws, s);
        if (rc) return rc;
    }
    return 0;
}

int sbce_estep(const sbce_cfg* cfg, const sbce_io* io, const double* theta, double* stat_m, double* stat_R,
               int32_t* kstar, double* lse_sym, void* workspace, size_t workspace_bytes, void* stream) {
    Dims d;
    int rc = make_dims(cfg, &d);
    if (rc) return rc;
    if (!io || !io->Yd || !io->PsiD || !io->varn || !theta || !stat_m || !stat_R || !workspace) return SBCE_E_NULL;
    if (cfg->batch == 0) return 0;
    const int chunk = trials_fitting(d, workspace_bytes, cfg->batch);
    if (chunk < 1) return SBCE_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    // as in em_chunk: the modes that take no joint decision return kstar = -1 and the modes that never form the
    // log-sum return lse_sym = NaN (all-ones bytes), not whatever the caller's buffers held
    const bool tree = d.mode == SBCE_MODE_SOFT || d.mode == SBCE_MODE_HARD;
    const bool decides = tree || d.mode == SBCE_MODE_ZF || d.mode == SBCE_MODE_MMSE;
    for (int b0 = 0; b0 < cfg->batch; b0 += chunk) {
        const int nb = (cfg->batch - b0 < chunk) ? cfg->batch - b0 : chunk;
        Workspace ws;
        carve_workspace(d, nb, workspace, &ws);
        sbce_io o = offset_io(d, *io, (size_t)b0);
        const size_t sb = (size_t)b0 * d.T_d;
        if (kstar && !decides) CK(cudaMemsetAsync(kstar + sb, 0xFF, (size_t)nb * d.T_d * sizeof(int32_t), s));
        if (lse_sym && !tree) CK(cudaMemsetAsync(lse_sym + sb, 0xFF, (size_t)nb * d.T_d * sizeof(double), s));
        rc = estep_dispatch(d, nb, o.Yd, o.PsiD, theta + (size_t)b0 * d.L * d.n_rx * 2, o.varn, nullptr, ws,
                            stat_m + sb * d.n_tx * 2, stat_R + sb * d.n_tx * d.n_tx * 2, kstar ? kstar + sb : nullptr,
                            lse_sym ? lse_sym + sb : nullptr, (d.flags & SBCE_FLAG_SUPERIMPOSED) ? o.Xp : nullptr, s);
        if (rc) return rc;
    }
    return 0;
}

int sbce_mstep(const sbce_cfg* cfg, const sbce_io* io, const double* stat_m, const double* stat_R, double* theta_out,
               int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
    Dims d;
    int rc = make_dims(cfg, &d, false);   // no E-step here: the hypothesis-count limits do not apply
    if (rc) return rc;
    if (!io || !io->Yd || !io->PsiD || !stat_m || !stat_R || !theta_out || !workspace) return SBCE_E_NULL;
    if (d.T_p > 0 && (!io->Yp || !io->PsiP || !io->Xp)) return SBCE_E_NULL;
    if (cfg->batch == 0) return 0;
    const int chunk = trials_fitting(d, workspace_bytes, cfg->batch);
    if (chunk < 1) return SBCE_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    for (int b0 = 0; b0 < cfg->batch; b0 += chunk) {
        const int nb = (cfg->batch - b0 < chunk) ? cfg->batch - b0 : chunk;
        Workspace ws;
        carve_workspace(d, nb, workspace, &ws);
        sbce_io o = offset_io(d, *io, (size_t)b0);
        const size_t sb = (size_t)b0 * d.T_d;
        CK(cudaMemsetAsync(ws.stat, 0, (size_t)nb * 4, s));
        CK(launch_pilot_stats(d, nb, o.Xp, ws.pil_m, ws.pil_R, s));
        CK(launch_normal_equations(pilot_dims(d), nb, o.PsiP, d.T_p, o.Yp, ws.pil_m, ws.pil_R, nullptr, ws.Gp, nullptr, s));
        CK(launch_normal_equations(d, nb, o.PsiD, d.T_d, o.Yd, stat_m + sb * d.n_tx * 2,
                                   stat_R + sb * d.n_tx * d.n_tx * 2, ws.Gp, ws.G, nullptr, s));
        CK(launch_chol_solve(d, nb, ws.G, theta_out + (size_t)b0 * d.L * d.n_rx * 2, nullptr, ws.stat, ws.thbuf, s));
        if (status) CK(cudaMemcpyAsync(status + b0, ws.stat, (size_t)nb * 4, cudaMemcpyDeviceToDevice, s));
    }
    return 0;
}

int sbce_accumulate_nmse(const double* nmse, const int32_t* status, int32_t batch, double* acc, void* stream) {
    if (!nmse || !acc) return SBCE_E_NULL;
    CK(launch_accumulate_nmse(nmse, status, batch, acc, (cudaStream_t)stream));
    return 0;
}

int sbce_generate_batch(const sbce_cfg* cfg, const sbce_gen* gen, const sbce_io* io, void* stream) {
    Dims d;
    int rc = make_dims(cfg, &d, false);
    if (rc) return rc;
    if (!gen || !io) return SBCE_E_NULL;
    if (!io->h_true || !io->Xd_true || !io->PsiD || !io->Yd || !io->varn) return SBCE_E_NULL;
    if (d.T_p > 0 && (!io->Xp || !io->PsiP || !io->Yp)) return SBCE_E_NULL;
    if (gen->pilot_design < SBCE_PILOTS_PM || gen->pilot_design > SBCE_PILOTS_TOP) return SBCE_E_UNSUPPORTED;
    if (gen->data_phases < SBCE_PHASES_RANDOM || gen->data_phases > SBCE_PHASES_DFT) return SBCE_E_UNSUPPORTED;
    if (cfg->batch == 0) return 0;
    // the trial index is gridDim.y of the generator kernels: at most 65535 trials per launch
    for (int b0 = 0; b0 < cfg->batch; b0 += SBCE_MAX_CHUNK) {
        const int nb = (cfg->batch - b0 < SBCE_MAX_CHUNK) ? cfg->batch - b0 : SBCE_MAX_CHUNK;
        sbce_gen g = *gen;
        g.trial0 = gen->trial0 + b0;
        const sbce_io o = offset_io(d, *io, (size_t)b0);
        CK(launch_generate(d, nb, &g, o, (double*)o.h_true, (double*)o.Xp, (double*)o.Xd_true, (double*)o.PsiP,
                           (double*)o.PsiD, (double*)o.Yp, (double*)o.Yd, (cudaStream_t)stream));
    }
    return 0;
}

int sbce_ls_start(const sbce_cfg* cfg, const sbce_io* io, double* theta0, int32_t* status, void* workspace,
                  size_t workspace_bytes, void* stream) {
    Dims d;
    int rc = make_dims(cfg, &d, false);
    if (rc) return rc;
    if (!io || !io->Yp || !io->PsiP || !io->Xp || !theta0 || !workspace) return SBCE_E_NULL;
    if (d.T_p < 1) return SBCE_E_SHAPE;
    if (cfg->batch == 0) return 0;
    const int chunk = trials_fitting(d, workspace_bytes, cfg->batch);
    if (chunk < 1) return SBCE_E_WORKSPACE;
    for (int b0 = 0; b0 < cfg->batch; b0 += chunk) {
        const int nb = (cfg->batch - b0 < chunk) ? cfg->batch - b0 : chunk;
        Workspace ws;
        carve_workspace(d, nb, workspace, &ws);
        sbce_io o = offset_io(d, *io, (size_t)b0);
        CK(launch_ls_start(pilot_dims(d), nb, o, theta0 + (size_t)b0 * d.L * d.n_rx * 2, status ? status + b0 : nullptr, ws,
                           (cudaStream_t)stream));
    }
    return 0;
}

int sbce_accumulate_ser(const sbce_cfg* cfg, const int32_t* kstar, const double* Xd_true, int32_t batch, double* acc,
                        void* stream) {
    Dims d;
    int rc = make_dims(cfg, &d, false);
    if (rc) return rc;
    if (!kstar || !Xd_true || !acc) return SBCE_E_NULL;
    if (d.n_tx * d.bitsM > 30) return SBCE_E_UNSUPPORTED;
    CK(launch_accumulate_ser(d, batch, kstar, Xd_true, acc, (cudaStream_t)stream));
    return 0;
}

int sbce_measure_fp64_peak(double* tflops, double* seconds) {
    CK(run_fp64_peak(tflops, seconds));
    return 0;
}

int sbce_profile_begin(void) {
    std::lock_guard<std::mutex> lock(g_prof_mu);
    for (auto& sp : g_spans) { g_event_pool.push_back(sp.a); g_event_pool.push_back(sp.b); }
    g_spans.clear();
    g_prof_on.store(true);
    return 0;
}

int sbce_profile_end(double* ms_per_phase, int64_t* spans_per_phase, int32_t n_phases) {
    std::lock_guard<std::mutex> lock(g_prof_mu);
    g_prof_on.store(false);
    if (!ms_per_phase || n_phases < 1) return SBCE_E_NULL;
    for (int i = 0; i < n_phases; ++i) { ms_per_phase[i] = 0.0; if (spans_per_phase) spans_per_phase[i] = 0; }
    for (auto& sp : g_spans) {
        CK(cudaEventSynchronize(sp.b));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, sp.a, sp.b));
        if (sp.phase >= 0 && sp.phase < n_phases) {
            ms_per_phase[sp.phase] += ms;
            if (spans_per_phase) spans_per_phase[sp.phase] += 1;
        }
        g_event_pool.push_back(sp.a);
        g_event_pool.push_back(sp.b);
    }
    g_spans.clear();
    return 0;
}

int64_t sbce_launch_count(int32_t reset) {
    long long v = g_launches.load();
    if (reset) g_launches.store(0);
    return (int64_t)v;
}

// ---------------------------------------------------------------------------
// host-pointer convenience path (the end-to-end route the Python estimators use)
// ---------------------------------------------------------------------------
namespace {
// The kernel schedule of one half of a host-route call (~55 launches at 10 EM iterations), captured into a CUDA
// graph the second time the same (configuration, device buffers) pair comes by.  A synchronous call per sweep
// step leaves the GPU waiting on the host thread between launches; on shared hosts a descheduled thread turned
// a 58 ms call into 75-130 ms (profiles/r02m).  A graph replays the whole schedule from one launch.
struct GraphSlot {
    unsigned long long key = 0;
    int seen = 0;                    // eager runs with this key so far
    long long launches = 0;          // kernels in the graph (for sbce_launch_count)
    cudaGraphExec_t exec = nullptr;
    unsigned long long stamp = 0;    // least recently used slot is recycled
};
struct DevPool {
    void* p = nullptr;
    size_t cap = 0;
    cudaStream_t stream = nullptr;   // compute + device->host
    cudaStream_t copy = nullptr;     // host->device, runs ahead of the compute stream
    cudaEvent_t ev[2] = {nullptr, nullptr};
    GraphSlot graphs[4];
    unsigned long long clock = 0;
    std::mutex mu;                   // one caller at a time per device; different devices run concurrently
};

unsigned long long fnv1a(const void* data, size_t n, unsigned long long h) {
    const unsigned char* p = (const unsigned char*)data;
    for (size_t i = 0; i < n; ++i) { h ^= p[i]; h *= 1099511628211ull; }
    return h;
}
constexpr int SBCE_MAX_DEVICES = 64;
DevPool g_pool[SBCE_MAX_DEVICES];

int pool_get(int dev, size_t bytes, DevPool** out) {
    DevPool& P = g_pool[dev];
    if (!P.stream) {
        CK(cudaStreamCreateWithFlags(&P.stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&P.copy, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&P.ev[0], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&P.ev[1], cudaEventDisableTiming));
    }
    if (P.cap < bytes) {
        // the cached graphs hold addresses inside the old allocation (both streams are idle here: every call
        // drains them before it returns)
        for (GraphSlot& g : P.graphs) {
            if (g.exec) cudaGraphExecDestroy(g.exec);
            g = GraphSlot();
        }
        if (P.p) CK(cudaFree(P.p));
        P.p = nullptr;
        P.cap = 0;
        CK(cudaMalloc(&P.p, bytes));
        P.cap = bytes;
    }
    *out = &P;
    return 0;
}

// Restores the calling thread's current device on scope exit (the host route selects `device` itself).
struct DeviceGuard {
    int prev = -1;
    bool armed = false;
    int enter(int dev) {
        CK(cudaGetDevice(&prev));
        armed = true;
        if (prev != dev) CK(cudaSetDevice(dev));
        return 0;
    }
    ~DeviceGuard() {
        if (armed) { int cur = -1; if (cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev); }
    }
};

// Drains both streams of the pool on scope exit: whatever path leaves sbce_em_batch_host (error returns
// included), no DMA is still reading or writing the caller's host buffers afterwards.
struct DrainGuard {
    DevPool* P = nullptr;
    ~DrainGuard() {
        if (P) {
            if (P->copy) cudaStreamSynchronize(P->copy);
            if (P->stream) cudaStreamSynchronize(P->stream);
        }
    }
};

// Batch size from which the host route splits a call in two halves (upload of the second half overlaps the
// kernels of the first); below it the kernels lose more from the smaller launch than the overlap wins
// (measured on B200 at the north-star size).  sbce_host_split_threshold() exposes it to tests.
constexpr int SBCE_HOST_SPLIT_MIN_BATCH = 1184;
}  // namespace

int sbce_host_split_threshold(void) { return SBCE_HOST_SPLIT_MIN_BATCH; }

// One half of a host-route call on the pool's compute stream: eager the first time a (configuration, buffers)
// key is seen, captured into a graph the second time, replayed from then on.  Never while the phase profiler is
// armed (its events must be recorded eagerly).
static int run_half(DevPool* P, const sbce_cfg* c2, const sbce_io* o, void* ws, size_t ws_bytes) {
    cudaStream_t s = P->stream;
    if (g_prof_on.load(std::memory_order_relaxed)) return sbce_em_batch(c2, o, ws, ws_bytes, (void*)s);
    unsigned long long key = fnv1a(c2, sizeof(*c2), 1469598103934665603ull);
    key = fnv1a(o, sizeof(*o), key);
    key = fnv1a(&ws, sizeof(ws), key);
    key = fnv1a(&ws_bytes, sizeof(ws_bytes), key);
    GraphSlot* slot = nullptr;
    GraphSlot* lru = &P->graphs[0];
    for (GraphSlot& g : P->graphs) {
        if (g.key == key && g.seen > 0) slot = &g;
        if (g.stamp < lru->stamp) lru = &g;
    }
    if (!slot) {   // first sight: run eagerly (this also performs every one-time function-attribute opt-in)
        if (lru->exec) { cudaGraphExecDestroy(lru->exec); lru->exec = nullptr; }
        lru->key = key; lru->seen = 1; lru->launches = 0; lru->stamp = ++P->clock;
        return sbce_em_batch(c2, o, ws, ws_bytes, (void*)s);
    }
    slot->stamp = ++P->clock;
    if (!slot->exec) {
        const long long before = g_launches.load();
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
            cudaGetLastError();
            return sbce_em_batch(c2, o, ws, ws_bytes, (void*)s);
        }
        const int rc = sbce_em_batch(c2, o, ws, ws_bytes, (void*)s);
        const cudaError_t ce = cudaStreamEndCapture(s, &graph);
        const long long captured = g_launches.load() - before;
        g_launches.fetch_sub(captured);                           // nothing ran yet
        if (rc != 0 || ce != cudaSuccess || graph == nullptr) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            slot->seen = 0;                                       // do not try again with this key
            slot->key = 0;
            return rc ? rc : sbce_em_batch(c2, o, ws, ws_bytes, (void*)s);
        }
        const cudaError_t ie = cudaGraphInstantiate(&slot->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) {
            cudaGetLastError();
            slot->exec = nullptr; slot->seen = 0; slot->key = 0;
            return sbce_em_batch(c2, o, ws, ws_bytes, (void*)s);
        }
        slot->launches = captured;
    }
    slot->seen += 1;
    CK(cudaGraphLaunch(slot->exec, s));
    count_launch((int)slot->launches);
    return 0;
}

int sbce_em_batch_host(const sbce_cfg* cfg, const sbce_io* io, int32_t device) {
    Dims d;
    int rc = make_dims(cfg, &d);
    if (rc) return rc;
    rc = check_io(d, io);
    if (rc) return rc;
    if (cfg->batch == 0) return 0;
    if (device < 0 || device >= SBCE_MAX_DEVICES || device >= sbce_device_count()) return SBCE_E_NODEVICE;
    std::lock_guard<std::mutex> lock(g_pool[device].mu);
    DeviceGuard dg;
    rc = dg.enter(device);
    if (rc) return rc;
    const size_t B = (size_t)cfg->batch;
    const size_t Ln = (size_t)d.L * d.n_rx * 16;
    const size_t psiB = d.psi_shared ? 1 : B, psiPB = d.psiP_shared ? 1 : B;
    // device mirror of the io block
    struct Seg { const void* h; size_t bytes; size_t off; bool in; void* hout; };
    size_t off = 0;
    auto seg = [&](const void* h, size_t bytes, bool in, void* hout) {
        Seg s{h, bytes, off, in, hout};
        if (h || hout) off += al(bytes);
        return s;
    };
    Seg sYd = seg(io->Yd, B * d.T_d * d.n_rx * 16, true, nullptr);
    Seg sYp = seg(io->Yp, B * d.T_p * d.n_rx * 16, true, nullptr);
    Seg sPd = seg(io->PsiD, psiB * d.T_d * d.N1 * 16, true, nullptr);
    Seg sPp = seg(io->PsiP, psiPB * d.T_p * d.N1 * 16, true, nullptr);
    const size_t xpT = (d.flags & SBCE_FLAG_SUPERIMPOSED) ? d.T_d : d.T_p;   // offsets ride in Xp
    Seg sXp = seg(io->Xp, B * xpT * d.n_tx * 16, true, nullptr);
    Seg sT0 = seg(io->theta0, B * Ln, true, nullptr);
    Seg sVn = seg(io->varn, B * 8, true, nullptr);
    Seg sHt = seg(io->h_true, B * Ln, true, nullptr);
    Seg sXd = seg(io->Xd_true, B * d.T_d * d.n_tx * 16, true, nullptr);
    Seg oTh = seg(nullptr, B * Ln, false, io->theta);
    Seg oKs = seg(nullptr, B * d.T_d * 4, false, io->kstar);
    Seg oLl = seg(nullptr, B * d.itera * 8, false, io->llf);
    Seg oLs = seg(nullptr, B * d.itera * 8, false, io->lse);
    Seg oNm = seg(nullptr, B * 8, false, io->nmse);
    Seg oIt = seg(nullptr, B * 4, false, io->iters);
    Seg oSt = seg(nullptr, B * 4, false, io->status);
    const size_t io_bytes = off;
    // workspace: as many trials in flight as fit in ~1/3 of free memory, at most the batch
    size_t freeb = 0, totalb = 0;
    CK(cudaMemGetInfo(&freeb, &totalb));
    size_t per1 = 0, perB = 0;
    { Workspace w; per1 = carve_workspace(d, 1, nullptr, &w); perB = carve_workspace(d, cfg->batch, nullptr, &w); }
    size_t budget = (freeb + g_pool[device].cap) / 3;
    if (budget < per1) budget = per1;
    size_t ws_bytes = perB < budget ? perB : budget;
    DevPool* P = nullptr;
    rc = pool_get(device, io_bytes + ws_bytes + 256, &P);
    if (rc) return rc;
    DrainGuard drain;
    drain.P = P;
    char* base = (char*)P->p;
    cudaStream_t s = P->stream;
    sbce_io dio;
    memset(&dio, 0, sizeof(dio));
    auto dp = [&](const Seg& q) { return (q.h || q.hout) ? (double*)(base + q.off) : nullptr; };
    dio.Yd = dp(sYd); dio.Yp = dp(sYp); dio.PsiD = dp(sPd); dio.PsiP = dp(sPp); dio.Xp = dp(sXp);
    dio.theta0 = dp(sT0); dio.varn = dp(sVn); dio.h_true = dp(sHt); dio.Xd_true = dp(sXd);
    dio.theta = dp(oTh); dio.kstar = (int32_t*)dp(oKs); dio.llf = dp(oLl); dio.lse = dp(oLs); dio.nmse = dp(oNm);
    dio.iters = (int32_t*)dp(oIt); dio.status = (int32_t*)dp(oSt);

    // Large batches go in two halves: the host->device copy of the second half overlaps the kernels of
    // the first (copy stream runs ahead; the compute stream waits on one event per half).
    const int nhalf = (cfg->batch >= SBCE_HOST_SPLIT_MIN_BATCH) ? 2 : 1;
    const int half = (cfg->batch + nhalf - 1) / nhalf;
    struct Part { Seg* q; size_t per_trial; };
    Part ins[] = {{&sYd, (size_t)d.T_d * d.n_rx * 16}, {&sYp, (size_t)d.T_p * d.n_rx * 16},
                  {&sPd, d.psi_shared ? 0 : (size_t)d.T_d * d.N1 * 16}, {&sPp, d.psiP_shared ? 0 : (size_t)d.T_p * d.N1 * 16},
                  {&sXp, xpT * d.n_tx * 16}, {&sT0, Ln}, {&sVn, 8}, {&sHt, Ln},
                  {&sXd, (size_t)d.T_d * d.n_tx * 16}};
    Part outs[] = {{&oTh, Ln}, {&oKs, (size_t)d.T_d * 4}, {&oLl, (size_t)d.itera * 8}, {&oLs, (size_t)d.itera * 8},
                   {&oNm, 8}, {&oIt, 4}, {&oSt, 4}};
    for (int hf = 0; hf < nhalf; ++hf) {
        const size_t b0 = (size_t)hf * half;
        const size_t nb = (b0 + half <= B) ? (size_t)half : B - b0;
        for (Part& pt : ins) {
            if (!pt.q->h || !pt.q->bytes) continue;
            if (pt.per_trial == 0) {  // shared across the batch: once
                if (hf == 0) CK(cudaMemcpyAsync(base + pt.q->off, pt.q->h, pt.q->bytes, cudaMemcpyHostToDevice, P->copy));
            } else {
                CK(cudaMemcpyAsync(base + pt.q->off + b0 * pt.per_trial, (const char*)pt.q->h + b0 * pt.per_trial,
                                   nb * pt.per_trial, cudaMemcpyHostToDevice, P->copy));
            }
        }
        CK(cudaEventRecord(P->ev[hf], P->copy));
    }
    for (int hf = 0; hf < nhalf; ++hf) {
        const size_t b0 = (size_t)hf * half;
        const size_t nb = (b0 + half <= B) ? (size_t)half : B - b0;
        CK(cudaStreamWaitEvent(s, P->ev[hf], 0));
        sbce_cfg c2 = *cfg;
        c2.batch = (int32_t)nb;
        sbce_io o = offset_io(d, dio, b0);
        rc = run_half(P, &c2, &o, base + al(io_bytes), ws_bytes);
        if (rc) return rc;
        for (Part& pt : outs)
            if (pt.q->hout && pt.q->bytes)
                CK(cudaMemcpyAsync((char*)pt.q->hout + b0 * pt.per_trial, base + pt.q->off + b0 * pt.per_trial,
                                   nb * pt.per_trial, cudaMemcpyDeviceToHost, s));
    }
    CK(cudaStreamSynchronize(s));
    CK(cudaStreamSynchronize(P->copy));
    return 0;
}

}  // extern "C"
