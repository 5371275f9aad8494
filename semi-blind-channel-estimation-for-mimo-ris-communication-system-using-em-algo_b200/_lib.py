"""ctypes binding of libsbce.so (C ABI in include/sbce.h).

There is deliberately NO fallback: if the CUDA library is missing or no CUDA
device is visible, every compute entry point raises.  The numpy oracle under
/oracle is test infrastructure and is never imported from here.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsbce.so")

MODE_SOFT, MODE_HARD, MODE_PM, MODE_PM_BETA, MODE_ZF, MODE_MMSE = 0, 1, 2, 3, 4, 5
FLAG_GENIE_STOP, FLAG_QUIRKS, FLAG_PSI_SHARED, FLAG_ZERO_START, FLAG_FULL_SCAN, FLAG_SUPERIMPOSED = 1, 2, 4, 8, 16, 32
FLAG_PSIP_SHARED = 64
FLAG_ZF_STOP_GUARD = 128
ST_NOT_PD, ST_NONFINITE = 1, 2


class SbceError(RuntimeError):
    pass


class Cfg(C.Structure):
    _fields_ = [("N", C.c_int32), ("n_tx", C.c_int32), ("n_rx", C.c_int32), ("M", C.c_int32),
                ("T_p", C.c_int32), ("T_d", C.c_int32), ("itera", C.c_int32), ("batch", C.c_int32),
                ("mode", C.c_int32), ("flags", C.c_uint32), ("partition_p1", C.c_int32),
                ("reserved", C.c_int32 * 5)]


_IO_FIELDS = ["Yd", "Yp", "PsiD", "PsiP", "Xp", "theta0", "varn", "h_true", "Xd_true",
              "theta", "kstar", "llf", "lse", "nmse", "iters", "status"]


class Io(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in _IO_FIELDS]


class Gen(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("trial0", C.c_int64), ("pilot_design", C.c_int32), ("data_phases", C.c_int32),
                ("varh", C.c_double), ("no_direct_link", C.c_int32), ("reserved", C.c_int32 * 3)]


PILOTS = {"pm": 0, "top": 1, "top_tp": 1, "top_td": 1}
PHASES_KIND = {"random": 0, "dft": 1}

# every symbol include/sbce.h declares; tests assert the library exports all of them
EXPORTS = ["sbce_version", "sbce_error_string", "sbce_device_count", "sbce_workspace_bytes", "sbce_em_batch",
           "sbce_em_batch_host", "sbce_estep", "sbce_mstep", "sbce_accumulate_nmse", "sbce_measure_fp64_peak",
           "sbce_launch_count", "sbce_profile_begin", "sbce_profile_end", "sbce_generate_batch", "sbce_ls_start",
           "sbce_accumulate_ser", "sbce_host_split_threshold", "sbce_bit_llr", "sbce_accumulate_ber",
           "sbce_bit_llr_apriori"]

LLR_CLAMP = 32.0   # SBCE_LLR_CLAMP: bit LLRs are clamped to [-32, 32]

PHASES = ["setup", "heff_qr", "enum", "gram", "rhs", "chol", "metrics"]

_lib = None


def load():
    """Load libsbce.so or raise SbceError (never falls back to a CPU path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SbceError("libsbce.so not built at %s -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.sbce_version.restype = C.c_int
    lib.sbce_error_string.restype = C.c_char_p
    lib.sbce_error_string.argtypes = [C.c_int]
    lib.sbce_device_count.restype = C.c_int
    lib.sbce_workspace_bytes.argtypes = [C.POINTER(Cfg), C.c_int32, C.POINTER(C.c_size_t)]
    lib.sbce_em_batch.argtypes = [C.POINTER(Cfg), C.POINTER(Io), C.c_void_p, C.c_size_t, C.c_void_p]
    lib.sbce_em_batch_host.argtypes = [C.POINTER(Cfg), C.POINTER(Io), C.c_int32]
    lib.sbce_estep.argtypes = [C.POINTER(Cfg), C.POINTER(Io), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.sbce_mstep.argtypes = [C.POINTER(Cfg), C.POINTER(Io), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_size_t, C.c_void_p]
    lib.sbce_accumulate_nmse.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.sbce_generate_batch.argtypes = [C.POINTER(Cfg), C.POINTER(Gen), C.POINTER(Io), C.c_void_p]
    lib.sbce_ls_start.argtypes = [C.POINTER(Cfg), C.POINTER(Io), C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                  C.c_void_p]
    lib.sbce_accumulate_ser.argtypes = [C.POINTER(Cfg), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.sbce_bit_llr.argtypes = [C.POINTER(Cfg), C.POINTER(Io), C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                 C.c_void_p]
    lib.sbce_bit_llr_apriori.argtypes = [C.POINTER(Cfg), C.POINTER(Io), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_size_t, C.c_void_p]
    lib.sbce_accumulate_ber.argtypes = [C.POINTER(Cfg), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.sbce_measure_fp64_peak.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.sbce_profile_end.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int32]
    lib.sbce_host_split_threshold.restype = C.c_int
    lib.sbce_launch_count.restype = C.c_int64
    lib.sbce_launch_count.argtypes = [C.c_int32]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise SbceError("libsbce error %d: %s" % (rc, load().sbce_error_string(rc).decode()))


def require_device():
    lib = load()
    if lib.sbce_device_count() < 1:
        raise SbceError("no CUDA device visible: the estimator has no CPU path")
    return lib
