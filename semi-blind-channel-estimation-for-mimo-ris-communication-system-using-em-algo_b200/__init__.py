"""sbce-b200: semi-blind EM channel estimation for MIMO-RIS links on B200.

Drop-in for the hot path of the thesis scripts (em / em_ml / em_pm and the
NMSE / SER sweep drivers); the arithmetic lives in libsbce.so (hand-written
sm_100a CUDA behind the C ABI of include/sbce.h).  No CPU fallback."""
from . import _lib, dist, drivers, engine, estimators, qam, signal_model, workloads  # noqa: F401
from ._lib import SbceError  # noqa: F401
from .engine import DeviceSession, Problem, Result, run_host  # noqa: F401
from .estimators import (bit_llr, em, em_iterations_llf, em_llf, em_loglik, em_ml, em_mmse, em_parallel, em_pm, em_pm_beta, em_ser, em_zf, nmse, ser_as_coded,  # noqa: F401
                         ser_true)
from .signal_model import channelMatrix, irsMatrix, pilotSymbols, receivedSignals, symbols  # noqa: F401
from .drivers import (SweepConfig, detectors_vs_snr, nmse_vs_N, nmse_vs_snr, nmse_vs_td, nmse_vs_tp,  # noqa: F401
                      ser_vs_snr)

__all__ = ["bit_llr", "em", "em_parallel", "em_ml", "em_llf", "em_loglik", "em_iterations_llf", "em_ser", "em_pm", "em_pm_beta", "em_zf", "em_mmse", "Problem", "DeviceSession", "run_host",
           "SweepConfig", "nmse_vs_tp", "nmse_vs_td", "nmse_vs_N", "nmse_vs_snr", "detectors_vs_snr", "ser_vs_snr"]
