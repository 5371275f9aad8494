#!/usr/bin/env python
"""Time sbce_bit_llr_apriori (random a-priori LLRs) against sbce_bit_llr at the same channel estimate (CUDA
events, the two calls alternated in one process), on the cases and the EM-converged theta of tools/bench_llr.py:
the headline workload (N = 64, 4x4 16-QAM, T_d = 256, B = 1184), 8x8 QPSK and 2x2 QPSK.  The priors are
6 N(0, 1) per bit (both signs, a few beyond the clamp).  Prints one JSON document with the card's name and power
limit, the per-kernel device time of a call pair from a separate torch.profiler run, and whether a zero prior
reproduces sbce_bit_llr bit for bit.

    python tools/bench_llr_apriori.py [--reps 20] [--trials 1184]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import sbce  # noqa: E402
from bench_llr import CASES, card  # noqa: E402
from sbce import workloads  # noqa: E402


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
    shape = (B, w.T_d, w.n_tx, int(np.log2(w.M)))
    gen = torch.Generator(device=dev).manual_seed(w.seed)
    La = 6.0 * torch.randn(shape, dtype=torch.float64, device=dev, generator=gen)
    llr = torch.empty(shape, dtype=torch.float64, device=dev)
    ext = torch.empty(shape, dtype=torch.float64, device=dev)

    def plain():
        ses.bit_llr(tb["Yd"], tb["PsiD"], theta, tb["varn"], out=llr)

    def apriori():
        ses.bit_llr(tb["Yd"], tb["PsiD"], theta, tb["varn"], out=ext, llr_a=La)

    zero = torch.zeros(shape, dtype=torch.float64, device=dev)
    plain()
    ses.bit_llr(tb["Yd"], tb["PsiD"], theta, tb["varn"], out=ext, llr_a=zero)
    torch.cuda.synchronize()
    zero_bitwise = bool(torch.equal(llr, ext))
    for _ in range(3):   # warm-up of both kernels
        plain()
        apriori()
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(reps)]
    for r in range(reps):
        ev[r][0].record()
        plain()
        ev[r][1].record()
        ev[r][2].record()
        apriori()
        ev[r][3].record()
    torch.cuda.synchronize()
    tp = np.array([e[0].elapsed_time(e[1]) for e in ev])
    ta = np.array([e[2].elapsed_time(e[3]) for e in ev])
    # device time per kernel and per pair of calls (one of each; the effective-channel kernel runs in both), from a
    # separate profiled run
    from torch.profiler import ProfilerActivity, profile

    nprof = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(nprof):
            plain()
            apriori()
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        name = e.key.split("(")[0].replace("void ", "")
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0 and name.startswith("sbce::"):
            kernels[name] = round(t / 1000.0 / nprof, 4)   # ms per pair of calls
    return dict(case=label, workload=w.as_dict(), trials=B, reps=reps, prior="6 N(0,1) per bit",
                bit_llr_ms_median=float(np.median(tp)), bit_llr_ms_min=float(tp.min()), bit_llr_ms_max=float(tp.max()),
                apriori_ms_median=float(np.median(ta)), apriori_ms_min=float(ta.min()), apriori_ms_max=float(ta.max()),
                ratio_median=float(np.median(ta) / np.median(tp)), kernel_ms_per_call_pair=kernels,
                zero_prior_bitwise_equal=zero_bitwise,
                clamped_fraction_posterior=float((llr.abs() == sbce._lib.LLR_CLAMP).double().mean().item()),
                clamped_fraction_extrinsic=float((ext.abs() == sbce._lib.LLR_CLAMP).double().mean().item()),
                nonfinite=int((~torch.isfinite(ext)).sum().item()))


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
