"""Monte-Carlo sweep drivers: the module-level loops of the reference scripts as
functions that RETURN the averaged curves (and the raw per-trial matrix) instead
of plotting them.

  nmse_vs_tp        /root/reference/Proposed method/Proposed_method_NMSEvsTp.py:153-176, PM.py:172-191
  nmse_vs_td        /root/reference/Proposed method/Proposed_method_NMSEvsTd.py:139-154
  nmse_vs_N         /root/reference/Proposed method/IRS_elements.py:373-414
  detectors_vs_snr  /root/reference/Proposed method/SNR/all_Detectors.py:356-395
  ser_vs_snr        /root/reference/Proposed method/SER/log_max_SER.py:147-167

Every (trial, sweep point) is independent, so a sweep point is one batched call
of the CUDA library; trials are sharded across ranks with disjoint seeds and the
per-point accumulators are summed once at the end (dist.allreduce_sum).
"""
from __future__ import annotations

from dataclasses import dataclass, replace
from typing import Callable, List, Sequence

import numpy as np

from . import dist, engine, signal_model
from .qam import bit_labels, bits_of, symbols_of


@dataclass
class SweepConfig:
    N: int = 32
    n_tx: int = 2
    n_rx: int = 2
    M: int = 4
    T_p: int = 20
    T_d: int = 50
    itera: int = 5
    monte_iter: int = 16
    varn: float = 0.1
    mode: str = "soft"            # soft | hard | pm | pm_beta | zf | mmse
    start: str = "ls"             # ls (h_initial, PM.py:147) | zero (Proposed_method_NMSEvsTp.py:45)
    genie_stop: bool = False
    quirks: bool = True
    partition_r: float = 0.0
    variant: str = "pm"           # RIS phase design family (signal_model.pilot_phases / data phases)
    order: str = "pm"             # RNG draw order of a trial
    legacy_rng: bool = True
    seed: int = 0
    max_batch: int = 4096         # trials per library call
    direct_link: bool = True      # False: no BS-user link, L = N n_tx ("direct vs non direct - T_pv s nmse.py"); on_device only
    on_device: bool = False       # generate inputs + LS start on the GPU (Philox; sbce_generate_batch / sbce_ls_start):
                                  # nothing but the per-point accumulators crosses PCIe


@dataclass
class PointResult:
    nmse_sum: float = 0.0
    n_valid: float = 0.0
    n_flagged: float = 0.0
    sym_err: float = 0.0          # true per-stream symbol errors
    sym_total: float = 0.0
    ser_coded_sum: float = 0.0    # sum over trials of the as-coded SER (log_max_SER.py:162)
    n_trials: float = 0.0
    bit_err: float = 0.0          # bit errors between the Gray labels (qam.bit_labels) of decisions and data
    bit_total: float = 0.0

    def vec(self):
        return np.array([self.nmse_sum, self.n_valid, self.n_flagged, self.sym_err, self.sym_total,
                         self.ser_coded_sum, self.n_trials, self.bit_err, self.bit_total], dtype=np.float64)


SER_MODES = ("soft", "hard", "zf", "mmse")


def cuda_runner(prob: engine.Problem, tb: signal_model.TrialBatch, device=0) -> engine.Result:
    """Default runner: the CUDA library through its host-buffer entry point."""
    theta0 = None if prob.zero_start else tb.theta0
    return engine.run_host(prob, tb.Yd, tb.Yp, tb.PsiD, tb.PsiP, tb.Xp, tb.varn, theta0=theta0, h_true=tb.h,
                           device=device)


def _ser_as_coded_batch(Xd, Xest):
    # (B,T,n,1) - (B,T,1,n): the reference's broadcast (quirk Q8)
    diff = Xd[:, :, :, None] - Xest[:, :, None, :]
    return np.count_nonzero(diff, axis=(1, 2, 3)) / (Xd.shape[1] * Xd.shape[2])


def run_point_device(cfg: SweepConfig, point_index: int, device=0, per_trial=None) -> PointResult:
    """run_point with everything on the GPU: Philox generation straight into the SoA layout, LS start,
    EM, NMSE / SER / BER accumulation; one 8-double read-back per sweep point.  Trial b of the point is the
    same whatever the batch size or the number of ranks (counter-based generator)."""
    import torch

    rank, ws = dist.world()
    lo, hi = dist.shard_trials(cfg.monte_iter, rank, ws)
    # without the direct link every phase row is a RIS element: N rows instead of N + 1
    prob = engine.Problem(N=cfg.N if cfg.direct_link else cfg.N - 1, n_tx=cfg.n_tx, n_rx=cfg.n_rx, M=cfg.M, T_p=cfg.T_p,
                          T_d=cfg.T_d, itera=cfg.itera, mode=cfg.mode, genie_stop=cfg.genie_stop, quirks=cfg.quirks,
                          zero_start=(cfg.start == "zero"), partition_r=cfg.partition_r,
                          psip_shared=True)      # the pilot design is deterministic: generated and stored once
    acc = PointResult()
    if hi <= lo:
        return acc
    dev = torch.device("cuda", device)
    pilot = "pm" if cfg.variant == "pm" else "top"
    phases = "dft" if cfg.variant == "top_td" else "random"
    with torch.cuda.device(dev):
        nbmax = min(cfg.max_batch, hi - lo)
        free, _ = torch.cuda.mem_get_info(dev)
        per_trial_bytes = engine.workspace_bytes(prob, 1)
        inflight = int(max(1, min(nbmax, (free // 3) // max(1, per_trial_bytes))))
        ses = engine.DeviceSession(prob, inflight, device=dev)
        acc_n = torch.zeros(3, dtype=torch.float64, device=dev)
        acc_s = torch.zeros(3, dtype=torch.float64, device=dev)
        acc_b = torch.zeros(2, dtype=torch.float64, device=dev)
        for b0 in range(lo, hi, cfg.max_batch):
            nb = min(cfg.max_batch, hi - b0)
            tb = ses.generate(nb, cfg.varn, seed=cfg.seed * 1000003 + point_index, trial0=b0, pilot_design=pilot,
                              data_phases=phases, direct_link=cfg.direct_link)
            theta0, st0 = (None, None) if prob.zero_start else ses.ls_start(tb["Yp"], tb["PsiP"], tb["Xp"])
            res = ses.run(tb["Yd"], tb["Yp"], tb["PsiD"], tb["PsiP"], tb["Xp"], tb["varn"], theta0=theta0,
                          h_true=tb["h"])
            if st0 is not None:
                res.status.bitwise_or_(st0)   # a rank-deficient pilot block flags the trial
            decides = cfg.mode in SER_MODES
            ses.accumulate(res, tb["Xd"], acc_n, acc_s if decides else None, acc_b if decides else None)
            if per_trial is not None:
                per_trial[b0:b0 + nb] = res.nmse.cpu().numpy()
            acc.n_trials += nb
        a, c, e = acc_n.cpu().numpy(), acc_s.cpu().numpy(), acc_b.cpu().numpy()
    acc.nmse_sum, acc.n_valid, acc.n_flagged = float(a[0]), float(a[1]), float(a[2])
    acc.sym_err, acc.sym_total, acc.ser_coded_sum = float(c[0]), float(c[1]), float(c[2])
    acc.bit_err, acc.bit_total = float(e[0]), float(e[1])
    return acc


def run_point(cfg: SweepConfig, point_index: int, runner: Callable = None, device=0, per_trial=None) -> PointResult:
    """All Monte-Carlo trials of one sweep point owned by this rank."""
    if cfg.on_device and runner is None:
        return run_point_device(cfg, point_index, device, per_trial)
    runner = runner or cuda_runner
    rank, ws = dist.world()
    lo, hi = dist.shard_trials(cfg.monte_iter, rank, ws)
    prob = engine.Problem(N=cfg.N, n_tx=cfg.n_tx, n_rx=cfg.n_rx, M=cfg.M, T_p=cfg.T_p, T_d=cfg.T_d, itera=cfg.itera,
                          mode=cfg.mode, genie_stop=cfg.genie_stop, quirks=cfg.quirks,
                          zero_start=(cfg.start == "zero"), partition_r=cfg.partition_r)
    acc = PointResult()
    for b0 in range(lo, hi, cfg.max_batch):
        nb = min(cfg.max_batch, hi - b0)
        seed = cfg.seed + point_index * cfg.monte_iter + b0
        tb = signal_model.generate_batch(cfg.N, cfg.n_tx, cfg.n_rx, cfg.M, cfg.T_p, cfg.T_d, cfg.varn, nb, seed=seed,
                                         legacy=cfg.legacy_rng, order=cfg.order, variant=cfg.variant)
        res = runner(prob, tb, device)
        status = np.zeros(nb, dtype=np.int32) if res.status is None else np.asarray(res.status)
        ok = status == 0
        nm = np.asarray(res.nmse)
        acc.nmse_sum += float(nm[ok].sum())
        acc.n_valid += float(ok.sum())
        acc.n_flagged += float((~ok).sum())
        acc.n_trials += nb
        if per_trial is not None:
            per_trial[b0:b0 + nb] = nm
        # joint decisions exist in the exhaustive and detector modes only: the partitioned estimators
        # (PM.py / PM_beta.py) never decide the whole symbol vector, kstar is -1 there
        if res.kstar is not None and cfg.mode in SER_MODES:
            xest = symbols_of(np.asarray(res.kstar), cfg.M, cfg.n_tx)
            acc.sym_err += float(np.count_nonzero(tb.Xd - xest))
            acc.sym_total += float(tb.Xd.size)
            acc.ser_coded_sum += float(_ser_as_coded_batch(tb.Xd, xest).sum())
            bits_est = bits_of(np.asarray(res.kstar), cfg.M, cfg.n_tx)
            acc.bit_err += float(np.count_nonzero(bits_est != bit_labels(cfg.M)[tb.idx_d]))
            acc.bit_total += float(bits_est.size)
    return acc


def _finish(xs, accs: List[PointResult], per_trial=None, device=None):
    """Cross-rank sum of the per-point accumulators (the one collective of a sweep, SNR/all_Detectors.py:389-395
    averages over trials) and the averaged curves.  Points without symbol decisions report ser = ber = NaN."""
    mat = np.stack([a.vec() for a in accs])
    mat = dist.allreduce_sum(mat, device=device)
    with np.errstate(invalid="ignore", divide="ignore"):
        has_ser = mat[:, 4] > 0
        out = dict(x=list(xs),
                   nmse=mat[:, 0] / np.maximum(mat[:, 1], 1.0),
                   n_valid=mat[:, 1], n_flagged=mat[:, 2],
                   ser=np.where(has_ser, mat[:, 3] / np.maximum(mat[:, 4], 1.0), np.nan),
                   ser_as_coded=np.where(has_ser, mat[:, 5] / np.maximum(mat[:, 6], 1.0), np.nan),
                   n_trials=mat[:, 6],
                   ber=np.where(mat[:, 8] > 0, mat[:, 7] / np.maximum(mat[:, 8], 1.0), np.nan))
    if per_trial is not None:
        out["per_trial"] = per_trial
    return out


def _sweep(cfg: SweepConfig, xs: Sequence, apply: Callable, runner=None, device=0, keep_per_trial=False):
    accs = []
    rank, ws = dist.world()
    per = np.full((cfg.monte_iter, len(xs)), np.nan) if (keep_per_trial and ws == 1) else None
    for i, x in enumerate(xs):
        c = apply(cfg, x)
        col = None if per is None else per[:, i]
        accs.append(run_point(c, i, runner, device, col))
    return _finish(xs, accs, per, device=device)


def nmse_vs_tp(cfg: SweepConfig, T_p_list: Sequence[int], runner=None, device=0, keep_per_trial=False):
    return _sweep(cfg, T_p_list, lambda c, x: replace(c, T_p=int(x)), runner, device, keep_per_trial)


def nmse_vs_td(cfg: SweepConfig, T_d_list: Sequence[int], runner=None, device=0, keep_per_trial=False):
    return _sweep(cfg, T_d_list, lambda c, x: replace(c, T_d=int(x)), runner, device, keep_per_trial)


def nmse_vs_N(cfg: SweepConfig, N_list: Sequence[int], runner=None, device=0, keep_per_trial=False):
    return _sweep(cfg, N_list, lambda c, x: replace(c, N=int(x)), runner, device, keep_per_trial)


def snr_to_varn(snr_db, power=10.0):
    """SNR/all_Detectors.py:350-354: varn = 10 / power**(SNR/10) with power = 10."""
    return 10.0 / (power ** (np.asarray(snr_db, dtype=np.float64) / 10.0))


def nmse_vs_snr(cfg: SweepConfig, snr_db: Sequence[float], runner=None, device=0, keep_per_trial=False):
    return _sweep(cfg, snr_db, lambda c, x: replace(c, varn=float(snr_to_varn(x))), runner, device, keep_per_trial)


def detectors_vs_snr(cfg: SweepConfig, snr_db: Sequence[float], modes=("pm_beta", "hard", "zf", "mmse", "soft"), runner=None,
                     device=0):
    """One NMSE-vs-SNR curve per estimator on identically seeded data (all_Detectors.py:356-395)."""
    out = {}
    for m in modes:
        c = replace(cfg, mode=m)
        out[m] = nmse_vs_snr(c, snr_db, runner, device)
    return out


def ser_vs_snr(cfg: SweepConfig, snr_db: Sequence[float], runner=None, device=0):
    """Hard-decision EM symbol error rate vs SNR (log_max_SER.py:147-167): returns both the
    as-coded figure (with the reference's broadcast) and the true per-stream SER, and the bit error rate
    of the same decisions under the Gray labels of qam.bit_labels (`ber`)."""
    return nmse_vs_snr(replace(cfg, mode="hard"), snr_db, runner, device)
