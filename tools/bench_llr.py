#!/usr/bin/env python
"""Time sbce_bit_llr against one sbce_estep call at the same channel estimate (CUDA events, the two calls
alternated in one process), at the headline workload (N = 64, 4x4 16-QAM, T_d = 256, B = 1184), 8x8 QPSK and
2x2 QPSK.  theta is the result of a 10-iteration EM run on on-device generated trials, so the LLRs are taken
where a receiver would take them.  Prints one JSON document with the card's name and power limit.

    python tools/bench_llr.py [--reps 20] [--trials 1184]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sbce  # noqa: E402
from sbce import workloads  # noqa: E402

# (label, workload key): the headline, the 8x8 QPSK detector point, the 2x2 QPSK sweep point
CASES = [("headline 4x4 16-QAM", 2), ("8x8 QPSK", 4), ("2x2 QPSK", 1)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else ("?", "?")
    return name, power


def run_case(label, key, B, reps):
    import torch

    w = workloads.WORKLOADS[key]
    prob = w.problem(itera=10)
    ses = sbce.DeviceSession(prob, B)
    tb = ses.generate(B, w.varn, seed=w.seed, pilot_design="top", data_phases="random")
    theta0 = None if prob.zero_start else ses.ls_start(tb["Yp"], tb["PsiP"], tb["Xp"])[0]
    res = ses.run(tb["Yd"], tb["Yp"], tb["PsiD"], tb["PsiP"], tb["Xp"], tb["varn"], theta0=theta0, h_true=tb["h"])
    theta = res.theta
    dev = ses.device
    outs = [torch.empty(s, dtype=d, device=dev) for s, d in
            (((B, w.T_d, w.n_tx), torch.complex128), ((B, w.T_d, w.n_tx, w.n_tx), torch.complex128),
             ((B, w.T_d), torch.int32), ((B, w.T_d), torch.float64))]
    llr = torch.empty((B, w.T_d, w.n_tx, int(np.log2(w.M))), dtype=torch.float64, device=dev)

    def estep():
        ses.estep(tb["Yd"], tb["PsiD"], theta, tb["varn"], out=outs)

    def bit_llr():
        ses.bit_llr(tb["Yd"], tb["PsiD"], theta, tb["varn"], out=llr)

    for _ in range(3):   # warm-up of both shapes
        estep()
        bit_llr()
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(reps)]
    for r in range(reps):
        ev[r][0].record()
        estep()
        ev[r][1].record()
        ev[r][2].record()
        bit_llr()
        ev[r][3].record()
    torch.cuda.synchronize()
    te = np.array([e[0].elapsed_time(e[1]) for e in ev])
    tl = np.array([e[2].elapsed_time(e[3]) for e in ev])
    # where the time goes: device time per kernel and per pair of calls (one sbce_estep + one sbce_bit_llr; the
    # effective-channel kernel runs in both), from a separate profiled run
    from torch.profiler import ProfilerActivity, profile

    nprof = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(nprof):
            estep()
            bit_llr()
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        name = e.key.split("(")[0].replace("void ", "")
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0 and name.startswith("sbce::"):
            kernels[name] = round(t / 1000.0 / nprof, 4)   # ms per pair of calls
    clamped = float((llr.abs() == sbce._lib.LLR_CLAMP).double().mean().item())
    return dict(case=label, workload=w.as_dict(), trials=B, reps=reps,
                estep_ms_median=float(np.median(te)), estep_ms_min=float(te.min()), estep_ms_max=float(te.max()),
                bit_llr_ms_median=float(np.median(tl)), bit_llr_ms_min=float(tl.min()), bit_llr_ms_max=float(tl.max()),
                ratio_median=float(np.median(tl) / np.median(te)), kernel_ms_per_call_pair=kernels, clamped_fraction=clamped,
                nonfinite=int((~torch.isfinite(llr)).sum().item()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--trials", type=int, default=1184)
    a = ap.parse_args()
    sbce._lib.require_device()
    name, power = card()
    res = [run_case(label, key, a.trials, a.reps) for label, key in CASES]
    print(json.dumps(dict(gpu=name, power_limit=power, note="both calls include the effective-channel + QR kernel",
                          results=res), indent=1))


if __name__ == "__main__":
    main()
