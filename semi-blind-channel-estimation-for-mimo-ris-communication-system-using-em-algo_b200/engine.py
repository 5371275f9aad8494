"""Batched host-side interface to libsbce: one call = `itera` EM iterations for a
batch of Monte-Carlo trials laid out as structure-of-arrays (one contiguous
complex128 array per quantity, trial index outermost).

Two routes, both through the C ABI (include/sbce.h):
  * run_host(...)   numpy in / numpy out  -> sbce_em_batch_host (H2D, kernels, D2H)
  * run_device(...) torch.cuda tensors    -> sbce_em_batch on the current stream
PyTorch is only the device allocator / stream provider here.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _lib
from ._lib import (FLAG_FULL_SCAN, FLAG_GENIE_STOP, FLAG_PSIP_SHARED, FLAG_PSI_SHARED, FLAG_ZF_STOP_GUARD, FLAG_QUIRKS, FLAG_SUPERIMPOSED, FLAG_ZERO_START, MODE_HARD,
                   MODE_MMSE, MODE_PM, MODE_PM_BETA, MODE_SOFT, MODE_ZF)

MODES = {"soft": MODE_SOFT, "hard": MODE_HARD, "pm": MODE_PM, "pm_beta": MODE_PM_BETA, "zf": MODE_ZF,
         "mmse": MODE_MMSE}


@dataclass
class Problem:
    """Static shape/mode description of a batch (the former module globals of the
    reference scripts: N, n_tx, n_rx, M_symbols, T_p, T_d, itera ...)."""
    N: int
    n_tx: int
    n_rx: int
    M: int
    T_p: int
    T_d: int
    itera: int
    mode: str = "soft"
    genie_stop: bool = False
    quirks: bool = True
    zero_start: bool = False
    psi_shared: bool = False    # PsiP and PsiD are passed once ([T][N+1]) for the whole batch
    psip_shared: bool = False   # only the (deterministic) pilot design PsiP is shared; data phases stay per trial
    partition_r: float = 0.0
    full_scan: bool = False   # E-step visits every tree node instead of skipping provably weightless subtrees
    zf_stop_guard: bool = False  # ZF mode: genie stop only from the second iteration on (all_detectorsvsTd.py:127)
    superimposed: bool = False  # parallel protocol (Parallel/ParallelProtocol_Tp.py): Xp holds per-symbol offsets, T_p = 0

    @property
    def L(self):
        return (self.N + 1) * self.n_tx

    @property
    def p1(self):
        # Proposed method/PM.py:74-75: p = int(partition_r / log2 M), A holds p+1 streams
        return int(self.partition_r / math.log2(self.M)) + 1

    def cfg(self, batch):
        flags = 0
        flags |= FLAG_GENIE_STOP if self.genie_stop else 0
        flags |= FLAG_QUIRKS if self.quirks else 0
        flags |= FLAG_PSI_SHARED if self.psi_shared else 0
        flags |= FLAG_PSIP_SHARED if self.psip_shared else 0
        flags |= FLAG_ZERO_START if self.zero_start else 0
        flags |= FLAG_FULL_SCAN if self.full_scan else 0
        flags |= FLAG_SUPERIMPOSED if self.superimposed else 0
        flags |= FLAG_ZF_STOP_GUARD if self.zf_stop_guard else 0
        c = _lib.Cfg()
        c.N, c.n_tx, c.n_rx, c.M = self.N, self.n_tx, self.n_rx, self.M
        c.T_p, c.T_d, c.itera, c.batch = self.T_p, self.T_d, self.itera, batch
        c.mode, c.flags, c.partition_p1 = MODES[self.mode], flags, self.p1
        return c

    def shapes(self, B):
        pb = () if self.psi_shared else (B,)
        ppb = () if (self.psi_shared or self.psip_shared) else (B,)
        return dict(Yd=(B, self.T_d, self.n_rx), Yp=(B, self.T_p, self.n_rx), PsiD=pb + (self.T_d, self.N + 1),
                    PsiP=ppb + (self.T_p, self.N + 1), Xp=(B, self.T_d if self.superimposed else self.T_p, self.n_tx),
                    theta0=(B, self.L, self.n_rx),
                    h_true=(B, self.L, self.n_rx), Xd_true=(B, self.T_d, self.n_tx))


@dataclass
class Result:
    theta: object
    kstar: object = None
    llf: object = None
    lse: object = None
    nmse: object = None
    iters: object = None
    status: object = None


_IN_C = ("Yd", "Yp", "PsiD", "PsiP", "Xp", "theta0", "h_true", "Xd_true")


def _np_c128(a, shape, name):
    a = np.ascontiguousarray(a, dtype=np.complex128)
    if a.shape != tuple(shape):
        raise ValueError("%s has shape %s, expected %s" % (name, a.shape, tuple(shape)))
    return a


def alloc_host_outputs(prob: Problem, B, want=("kstar", "lse", "nmse", "iters", "status"), pinned=False) -> Result:
    """Output arrays for run_host(out=...); pinned=True allocates page-locked memory through torch."""
    def mk(shape, dtype):
        if pinned:
            import torch

            tdt = {np.complex128: torch.complex128, np.float64: torch.float64, np.int32: torch.int32}[dtype]
            return torch.empty(shape, dtype=tdt).pin_memory().numpy()
        return np.empty(shape, dtype=dtype)

    out = Result(theta=mk((B, prob.L, prob.n_rx), np.complex128))
    if "kstar" in want:
        out.kstar = mk((B, prob.T_d), np.int32)
    if "llf" in want:
        out.llf = mk((B, prob.itera), np.float64)
    if "lse" in want:
        out.lse = mk((B, prob.itera), np.float64)
    if "nmse" in want:
        out.nmse = mk((B,), np.float64)
    if "iters" in want:
        out.iters = mk((B,), np.int32)
    if "status" in want:
        out.status = mk((B,), np.int32)
    return out


def run_host(prob: Problem, Yd, Yp, PsiD, PsiP, Xp, varn, theta0=None, h_true=None, Xd_true=None,
             want=("kstar", "llf", "lse", "nmse", "iters", "status"), device=0, out: Optional[Result] = None) -> Result:
    """numpy route (host buffers; copies are inside the call)."""
    if out is not None:
        return _run_host_into(prob, Yd, Yp, PsiD, PsiP, Xp, varn, theta0, h_true, Xd_true, device, out)
    lib = _lib.require_device()
    B = int(np.asarray(Yd).shape[0])
    sh = prob.shapes(B)
    ins = dict(Yd=Yd, Yp=Yp, PsiD=PsiD, PsiP=PsiP, Xp=Xp, theta0=theta0, h_true=h_true, Xd_true=Xd_true)
    keep = {}
    io = _lib.Io()
    for k in _IN_C:
        v = ins[k]
        if v is None:
            setattr(io, k, None)
            continue
        a = _np_c128(v, sh[k], k)
        keep[k] = a
        setattr(io, k, a.ctypes.data)
    vn = np.ascontiguousarray(np.broadcast_to(np.asarray(varn, dtype=np.float64), (B,)))
    keep["varn"] = vn
    io.varn = vn.ctypes.data
    out = Result(theta=np.empty((B, prob.L, prob.n_rx), dtype=np.complex128))
    io.theta = out.theta.ctypes.data
    if "kstar" in want:
        out.kstar = np.empty((B, prob.T_d), dtype=np.int32)
        io.kstar = out.kstar.ctypes.data
    if "llf" in want and Xd_true is not None:
        out.llf = np.empty((B, prob.itera), dtype=np.float64)
        io.llf = out.llf.ctypes.data
    if "lse" in want:
        out.lse = np.empty((B, prob.itera), dtype=np.float64)
        io.lse = out.lse.ctypes.data
    if "nmse" in want and h_true is not None:
        out.nmse = np.empty((B,), dtype=np.float64)
        io.nmse = out.nmse.ctypes.data
    if "iters" in want:
        out.iters = np.empty((B,), dtype=np.int32)
        io.iters = out.iters.ctypes.data
    if "status" in want:
        out.status = np.empty((B,), dtype=np.int32)
        io.status = out.status.ctypes.data
    cfg = prob.cfg(B)
    _lib.check(lib.sbce_em_batch_host(C.byref(cfg), C.byref(io), device))
    return out


def _run_host_into(prob, Yd, Yp, PsiD, PsiP, Xp, varn, theta0, h_true, Xd_true, device, out: Result) -> Result:
    """run_host with caller-owned (e.g. pinned) input and output arrays: no allocation, no conversion."""
    lib = _lib.require_device()
    B = int(Yd.shape[0])
    sh = prob.shapes(B)
    ins = dict(Yd=Yd, Yp=Yp, PsiD=PsiD, PsiP=PsiP, Xp=Xp, theta0=theta0, h_true=h_true, Xd_true=Xd_true)
    io = _lib.Io()
    for k in _IN_C:
        v = ins[k]
        if v is None:
            continue
        if v.dtype != np.complex128 or not v.flags.c_contiguous or v.shape != tuple(sh[k]):
            raise ValueError("%s must be C-contiguous complex128 of shape %s" % (k, sh[k]))
        setattr(io, k, v.ctypes.data)
    if varn.dtype != np.float64 or varn.shape != (B,):
        raise ValueError("varn must be float64 of shape (B,)")
    io.varn = varn.ctypes.data
    io.theta = out.theta.ctypes.data
    for k in ("kstar", "llf", "lse", "nmse", "iters", "status"):
        a = getattr(out, k)
        if a is not None and not (k == "llf" and Xd_true is None) and not (k == "nmse" and h_true is None):
            setattr(io, k, a.ctypes.data)
    cfg = prob.cfg(B)
    _lib.check(lib.sbce_em_batch_host(C.byref(cfg), C.byref(io), device))
    return out


# ---------------------------------------------------------------------------
# device route (torch tensors as device memory)
# ---------------------------------------------------------------------------

def _t_ptr(t):
    return None if t is None else t.data_ptr()


def workspace_bytes(prob: Problem, trials_in_flight: int) -> int:
    lib = _lib.load()
    n = C.c_size_t(0)
    cfg = prob.cfg(trials_in_flight)
    _lib.check(lib.sbce_workspace_bytes(C.byref(cfg), trials_in_flight, C.byref(n)))
    return int(n.value)


class DeviceSession:
    """Holds the device workspace for a Problem and launches on torch's current stream."""

    def __init__(self, prob: Problem, trials_in_flight: int, device=None):
        import torch

        self.torch = torch
        self.lib = _lib.require_device()
        self.prob = prob
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.trials_in_flight = int(trials_in_flight)
        self.ws_bytes = workspace_bytes(prob, self.trials_in_flight)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=self.device)

    def _on_device(self):
        """libsbce launches on the calling thread's CURRENT device: make it the session's for the call."""
        return self.torch.cuda.device(self.device)

    def _check(self, t, shape, name, dtype):
        torch = self.torch
        if t is None:
            return None
        if t.dtype != dtype or not t.is_cuda or not t.is_contiguous() or tuple(t.shape) != tuple(shape):
            raise ValueError("%s must be a contiguous cuda %s tensor of shape %s (got %s %s)" %
                             (name, dtype, tuple(shape), t.dtype, tuple(t.shape)))
        return t

    def alloc_outputs(self, B, llf=False, lse=True, nmse=True, kstar=True):
        torch, p = self.torch, self.prob
        dev = self.device
        return Result(theta=torch.empty((B, p.L, p.n_rx), dtype=torch.complex128, device=dev),
                      kstar=torch.empty((B, p.T_d), dtype=torch.int32, device=dev) if kstar else None,
                      llf=torch.empty((B, p.itera), dtype=torch.float64, device=dev) if llf else None,
                      lse=torch.empty((B, p.itera), dtype=torch.float64, device=dev) if lse else None,
                      nmse=torch.empty((B,), dtype=torch.float64, device=dev) if nmse else None,
                      iters=torch.empty((B,), dtype=torch.int32, device=dev),
                      status=torch.empty((B,), dtype=torch.int32, device=dev))

    def _io(self, B, Yd, Yp, PsiD, PsiP, Xp, varn, theta0, h_true, Xd_true):
        torch, p = self.torch, self.prob
        sh = p.shapes(B)
        c128 = torch.complex128
        io = _lib.Io()
        io.Yd = _t_ptr(self._check(Yd, sh["Yd"], "Yd", c128))
        io.Yp = _t_ptr(self._check(Yp, sh["Yp"], "Yp", c128))
        io.PsiD = _t_ptr(self._check(PsiD, sh["PsiD"], "PsiD", c128))
        io.PsiP = _t_ptr(self._check(PsiP, sh["PsiP"], "PsiP", c128))
        io.Xp = _t_ptr(self._check(Xp, sh["Xp"], "Xp", c128))
        io.theta0 = _t_ptr(self._check(theta0, sh["theta0"], "theta0", c128))
        io.h_true = _t_ptr(self._check(h_true, sh["h_true"], "h_true", c128))
        io.Xd_true = _t_ptr(self._check(Xd_true, sh["Xd_true"], "Xd_true", c128))
        io.varn = _t_ptr(self._check(varn, (B,), "varn", torch.float64))
        return io

    def run(self, Yd, Yp, PsiD, PsiP, Xp, varn, theta0=None, h_true=None, Xd_true=None, out: Optional[Result] = None):
        """Asynchronous on torch's current stream; returns the (device) Result."""
        torch, p = self.torch, self.prob
        B = int(Yd.shape[0])
        io = self._io(B, Yd, Yp, PsiD, PsiP, Xp, varn, theta0, h_true, Xd_true)
        if out is None:
            out = self.alloc_outputs(B, llf=Xd_true is not None, nmse=h_true is not None)
        io.theta = _t_ptr(out.theta)
        io.kstar = _t_ptr(out.kstar)
        io.llf = _t_ptr(out.llf) if Xd_true is not None else None
        io.lse = _t_ptr(out.lse)
        io.nmse = _t_ptr(out.nmse) if h_true is not None else None
        io.iters = _t_ptr(out.iters)
        io.status = _t_ptr(out.status)
        cfg = p.cfg(B)
        with self._on_device():
            stream = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(self.lib.sbce_em_batch(C.byref(cfg), C.byref(io), self.ws.data_ptr(), self.ws_bytes, stream))
        return out

    def estep(self, Yd, PsiD, theta, varn, Xp=None, out=None):
        """Stand-alone E-step sweep at `theta` -> (m, R, kstar, lse_sym) device tensors, written into
        `out` = (m, R, kstar, lse_sym) when given.  kstar is -1 in the PM modes and lse_sym NaN in the PM, ZF
        and MMSE modes, whatever the buffers held.
        With Problem.superimposed the per-symbol pilot offsets Xp [B][T_d][n_tx] are required."""
        torch, p = self.torch, self.prob
        B = int(Yd.shape[0])
        if p.superimposed and Xp is None:
            raise ValueError("superimposed pilots: estep() needs the offsets Xp [B][T_d][n_tx]")
        io = self._io(B, Yd, None, PsiD, None, Xp if p.superimposed else None, varn, None, None, None)
        dev = self.device
        shapes = ((B, p.T_d, p.n_tx), (B, p.T_d, p.n_tx, p.n_tx), (B, p.T_d), (B, p.T_d))
        dtypes = (torch.complex128, torch.complex128, torch.int32, torch.float64)
        if out is None:
            out = [torch.empty(sh, dtype=dt, device=dev) for sh, dt in zip(shapes, dtypes)]
        m, R, ks, ls = (self._check(o, sh, name, dt)
                        for o, sh, name, dt in zip(out, shapes, ("m", "R", "kstar", "lse_sym"), dtypes))
        self._check(theta, (B, p.L, p.n_rx), "theta", torch.complex128)
        cfg = p.cfg(B)
        with self._on_device():
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(self.lib.sbce_estep(C.byref(cfg), C.byref(io), theta.data_ptr(), m.data_ptr(), R.data_ptr(),
                                           ks.data_ptr(), ls.data_ptr(), self.ws.data_ptr(), self.ws_bytes, stream))
        return m, R, ks, ls

    def bit_llr(self, Yd, PsiD, theta, varn, Xp=None, out=None, llr_a=None):
        """Exact Gray-labelled bit LLRs of every data symbol at `theta` -> (B, T_d, n_tx, log2 M) float64 device
        tensor (written into `out` when given): ln P(bit = 0) - ln P(bit = 1) under the E-step's posterior
        (exponent d2/varn^2, uniform prior), clamped to [-32, 32]; NaN for a symbol whose inputs are not finite.
        Conventions: include/sbce.h (sbce_bit_llr), labels: qam.bit_labels.  Soft and hard modes only (both
        give the same LLRs).  With Problem.superimposed the offsets Xp [B][T_d][n_tx] are required.

        llr_a: a-priori LLRs from a channel decoder, a float64 device tensor of the same shape (clamped to +-32 on
        read; a NaN makes its symbol NaN).  Then the result is the extrinsic LLR, the posterior under that prior
        minus llr_a (sbce_bit_llr_apriori), for iterative detection and decoding; `out` may be llr_a itself.  With
        no prior the extrinsic and a-posteriori LLRs coincide: llr_a = 0 gives the same bits as llr_a=None."""
        torch, p = self.torch, self.prob
        if p.mode not in ("soft", "hard"):
            raise ValueError("bit LLRs are defined for the soft and hard modes, not %r" % (p.mode,))
        B = int(Yd.shape[0])
        if p.superimposed and Xp is None:
            raise ValueError("superimposed pilots: bit_llr() needs the offsets Xp [B][T_d][n_tx]")
        io = self._io(B, Yd, None, PsiD, None, Xp if p.superimposed else None, varn, None, None, None)
        dev = self.device
        shape = (B, p.T_d, p.n_tx, int(math.log2(p.M)))
        if out is None:
            out = torch.empty(shape, dtype=torch.float64, device=dev)
        self._check(out, shape, "out", torch.float64)
        self._check(theta, (B, p.L, p.n_rx), "theta", torch.complex128)
        if llr_a is not None:
            self._check(llr_a, shape, "llr_a", torch.float64)
        cfg = p.cfg(B)
        with self._on_device():
            stream = torch.cuda.current_stream(dev).cuda_stream
            if llr_a is None:
                _lib.check(self.lib.sbce_bit_llr(C.byref(cfg), C.byref(io), theta.data_ptr(), out.data_ptr(),
                                                 self.ws.data_ptr(), self.ws_bytes, stream))
            else:
                _lib.check(self.lib.sbce_bit_llr_apriori(C.byref(cfg), C.byref(io), theta.data_ptr(), llr_a.data_ptr(),
                                                         out.data_ptr(), self.ws.data_ptr(), self.ws_bytes, stream))
        return out

    def mstep(self, Yd, Yp, PsiD, PsiP, Xp, stat_m, stat_R):
        """Stand-alone M-step from given data statistics -> (theta, status)."""
        torch, p = self.torch, self.prob
        B = int(Yd.shape[0])
        dev = self.device
        varn = torch.ones((B,), dtype=torch.float64, device=dev)
        io = self._io(B, Yd, Yp, PsiD, PsiP, Xp, varn, None, None, None)
        self._check(stat_m, (B, p.T_d, p.n_tx), "stat_m", torch.complex128)
        self._check(stat_R, (B, p.T_d, p.n_tx, p.n_tx), "stat_R", torch.complex128)
        theta = torch.empty((B, p.L, p.n_rx), dtype=torch.complex128, device=dev)
        status = torch.empty((B,), dtype=torch.int32, device=dev)
        cfg = p.cfg(B)
        with self._on_device():
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(self.lib.sbce_mstep(C.byref(cfg), C.byref(io), stat_m.data_ptr(), stat_R.data_ptr(),
                                           theta.data_ptr(), status.data_ptr(), self.ws.data_ptr(), self.ws_bytes, stream))
        return theta, status


    # ---- on-device generation + LS start (include/sbce.h: sbce_generate_batch, sbce_ls_start) ----
    def generate(self, B, varn, seed, trial0=0, pilot_design="pm", data_phases="random", varh=1.0, direct_link=True):
        """Philox-generated trials written straight into device tensors (same names as
        signal_model.TrialBatch: h, Xd, Xp, PsiP, PsiD, Yp, Yd, varn).  Trial b of the batch is global
        trial trial0 + b of the sweep keyed by `seed`, independent of batch size and sharding."""
        torch, p = self.torch, self.prob
        dev = self.device
        sh = p.shapes(B)
        c128 = torch.complex128
        tb = {k: torch.empty(sh[k], dtype=c128, device=dev) for k in ("Yd", "Yp", "PsiD", "PsiP", "Xp")}
        tb["h"] = torch.empty(sh["h_true"], dtype=c128, device=dev)
        tb["Xd"] = torch.empty(sh["Xd_true"], dtype=c128, device=dev)
        if torch.is_tensor(varn):
            tb["varn"] = varn.to(device=dev, dtype=torch.float64).expand(B).contiguous()
        else:
            tb["varn"] = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(np.asarray(varn, np.float64), (B,)))).to(dev)
        io = _lib.Io()
        io.Yd, io.Yp, io.PsiD, io.PsiP, io.Xp = (tb[k].data_ptr() for k in ("Yd", "Yp", "PsiD", "PsiP", "Xp"))
        io.h_true, io.Xd_true, io.varn = tb["h"].data_ptr(), tb["Xd"].data_ptr(), tb["varn"].data_ptr()
        g = _lib.Gen()
        g.seed, g.trial0 = int(seed) & (2 ** 64 - 1), int(trial0)
        g.pilot_design, g.data_phases, g.varh = _lib.PILOTS[pilot_design], _lib.PHASES_KIND[data_phases], float(varh)
        g.no_direct_link = 0 if direct_link else 1   # all Problem.N + 1 phase rows are RIS elements
        cfg = p.cfg(B)
        with self._on_device():
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(self.lib.sbce_generate_batch(C.byref(cfg), C.byref(g), C.byref(io), stream))
        return tb

    def ls_start(self, Yp, PsiP, Xp):
        """h_initial = pinv(Z_p) y_p of every trial (PM.py:147) -> (theta0, status) device tensors."""
        torch, p = self.torch, self.prob
        B = int(Yp.shape[0])
        dev = self.device
        sh = p.shapes(B)
        io = _lib.Io()
        io.Yp = _t_ptr(self._check(Yp, sh["Yp"], "Yp", torch.complex128))
        io.PsiP = _t_ptr(self._check(PsiP, sh["PsiP"], "PsiP", torch.complex128))
        io.Xp = _t_ptr(self._check(Xp, sh["Xp"], "Xp", torch.complex128))
        theta0 = torch.empty((B, p.L, p.n_rx), dtype=torch.complex128, device=dev)
        status = torch.empty((B,), dtype=torch.int32, device=dev)
        cfg = p.cfg(B)
        with self._on_device():
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(self.lib.sbce_ls_start(C.byref(cfg), C.byref(io), theta0.data_ptr(), status.data_ptr(),
                                              self.ws.data_ptr(), self.ws_bytes, stream))
        return theta0, status

    def accumulate(self, res: "Result", Xd, acc_nmse, acc_ser=None, acc_ber=None):
        """Adds this batch to the per-point device accumulators: acc_nmse (3 float64: sum NMSE over valid
        trials, valid count, flagged count), acc_ser (3 float64: symbol errors, symbols, sum of as-coded SER),
        acc_ber (2 float64: bit errors between the Gray labels of the decisions and of Xd, bits compared)."""
        torch, p = self.torch, self.prob
        B = int(res.theta.shape[0])
        if res.nmse is None:
            raise ValueError("accumulate() needs Result.nmse: run(..., h_true=...) computes it")
        # joint decisions exist in the exhaustive and detector modes only (PM modes report kstar = -1)
        decides = (res.kstar is not None and p.mode in ("soft", "hard", "zf", "mmse")
                   and p.n_tx * int(math.log2(p.M)) <= 30)
        ser_ok = acc_ser is not None and decides
        with self._on_device():
            stream = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(self.lib.sbce_accumulate_nmse(res.nmse.data_ptr(),
                                                     None if res.status is None else res.status.data_ptr(), B,
                                                     acc_nmse.data_ptr(), stream))
            if ser_ok:
                cfg = p.cfg(B)
                _lib.check(self.lib.sbce_accumulate_ser(C.byref(cfg), res.kstar.data_ptr(), Xd.data_ptr(), B,
                                                        acc_ser.data_ptr(), stream))
            if acc_ber is not None and decides:
                _lib.check(self.lib.sbce_accumulate_ber(C.byref(p.cfg(B)), res.kstar.data_ptr(), Xd.data_ptr(), B,
                                                        acc_ber.data_ptr(), stream))


def fp64_peak_tflops():
    lib = _lib.require_device()
    tf, sec = C.c_double(0), C.c_double(0)
    _lib.check(lib.sbce_measure_fp64_peak(C.byref(tf), C.byref(sec)))
    return float(tf.value)


def launch_count(reset=False):
    return int(_lib.load().sbce_launch_count(1 if reset else 0))


def profile_begin():
    _lib.check(_lib.load().sbce_profile_begin())


def profile_end():
    """-> {phase: (milliseconds, timed launches)} summed since profile_begin()."""
    n = len(_lib.PHASES)
    ms = (C.c_double * n)()
    cnt = (C.c_int64 * n)()
    _lib.check(_lib.load().sbce_profile_end(ms, cnt, n))
    return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(_lib.PHASES)}
