"""Lag-form pilot normal equations on the GPU (mstep.cu: k_pilot_lag_check, k_pilot_lag_gram, k_pilot_lag_expand):
a qualifying pilot design gives the results of the pair-form Gram to rounding, matches the oracle, is
bitwise the same on every route, leaves the status bits of non-finite inputs as they were, and the profiler sees
the lag form do the work exactly when the design qualifies."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def S(cuda_device):
    import sbce

    sbce._lib.require_device()
    return sbce


def device_batch(S, N, n_tx, n_rx, M, T_p, T_d, itera, B, seed, varn=0.1):
    """Trials from the on-device generator with the shared top design (which qualifies), as numpy arrays."""
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T_p, T_d=T_d, itera=itera, psip_shared=True)
    ses = S.DeviceSession(prob, B)
    g = ses.generate(B, varn, seed=seed, pilot_design="top")
    tb = {k: v.cpu().numpy() for k, v in g.items()}
    rng = np.random.default_rng(seed)
    tb["theta0"] = tb["h"] + 0.1 * (rng.standard_normal(tb["h"].shape) + 1j * rng.standard_normal(tb["h"].shape))
    return prob, tb


def run_device(S, prob, tb, in_flight, PsiP=None):
    import torch

    ses = S.DeviceSession(prob, in_flight)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ses.device)
    P = tb["PsiP"] if PsiP is None else PsiP
    r = ses.run(t(tb["Yd"]), t(tb["Yp"]), t(tb["PsiD"]), t(P), t(tb["Xp"]), t(tb["varn"]), theta0=t(tb["theta0"]),
                h_true=t(tb["h"]))
    torch.cuda.synchronize()
    return {k: getattr(r, k).cpu().numpy() for k in ("theta", "kstar", "nmse", "iters", "status")}


def rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


@pytest.mark.parametrize("n_tx,n_rx", [(1, 2), (2, 2), (4, 4), (5, 6), (8, 8)])
def test_lag_form_matches_oracle_and_pair_form(S, n_tx, n_rx):
    import dataclasses

    from oracle import em_numpy as orc

    N, M, T_p, T_d, itera, B = 12, 4, 128, 16, 3, 3
    prob, tb = device_batch(S, N, n_tx, n_rx, M, T_p, T_d, itera, B, seed=100 + n_tx)
    lag = run_device(S, prob, tb, B)
    # one phase moved by 1e-11, far above the rule's bound (32 (N+1) ulp): the pair-form Gram builds G_p
    P = tb["PsiP"].copy()
    P[7, 5] += 1e-11
    pair = run_device(S, prob, tb, B, PsiP=P)
    assert rel(lag["theta"], pair["theta"]) < 1e-9
    # the per-trial layout of the same design takes the same path, bit for bit
    per_trial = run_device(S, dataclasses.replace(prob, psip_shared=False), tb, B,
                           PsiP=np.broadcast_to(tb["PsiP"], (B,) + tb["PsiP"].shape))
    assert all(np.array_equal(lag[k], per_trial[k]) for k in lag)
    assert np.array_equal(lag["kstar"], pair["kstar"]) and np.array_equal(lag["iters"], pair["iters"])
    assert np.array_equal(lag["status"], pair["status"]) and not lag["status"].any()
    for b in range(B):
        ref = orc.em(tb["Yd"][b], tb["Yp"][b], tb["PsiD"][b], tb["PsiP"], tb["Xp"][b], M, float(tb["varn"][b]), itera,
                     theta0=tb["theta0"][b])
        assert rel(lag["theta"][b], ref) < 1e-9, b


def test_routes_are_bitwise_equal(S):
    N, n_tx, n_rx, M, T_p, T_d, itera, B = 20, 4, 4, 16, 64, 24, 3, 7
    prob, tb = device_batch(S, N, n_tx, n_rx, M, T_p, T_d, itera, B, seed=5)
    dev = run_device(S, prob, tb, B)
    chunked = run_device(S, prob, tb, 3)
    for _ in range(3):   # eager, captured into a graph, replayed
        host = S.run_host(prob, tb["Yd"], tb["Yp"], tb["PsiD"], tb["PsiP"], tb["Xp"], tb["varn"], theta0=tb["theta0"],
                          h_true=tb["h"])
        for k in ("theta", "kstar", "nmse", "iters", "status"):
            assert np.array_equal(getattr(host, k), dev[k]), k
            assert np.array_equal(chunked[k], dev[k]), k


def test_non_finite_pilots_set_status_bits(S):
    N, n_tx, n_rx, M, T_p, T_d, itera, B = 10, 2, 2, 4, 32, 12, 2, 4
    prob, tb = device_batch(S, N, n_tx, n_rx, M, T_p, T_d, itera, B, seed=9)
    tb["Yp"] = tb["Yp"].copy()
    tb["Yp"][1, 3, 0] = np.nan                 # one trial's pilot block: the design still qualifies
    st = run_device(S, prob, tb, B)["status"]
    assert st[1] != 0 and not st[[0, 2, 3]].any(), st
    P = tb["PsiP"].copy()
    P[5, 3] = np.nan                           # the shared design: the pair form takes over, every trial flagged
    tb["Yp"][1, 3, 0] = 0.0
    st = run_device(S, prob, tb, B, PsiP=P)["status"]
    assert np.all(st != 0), st


# Solve-only M-step calls under torch.profiler, in a fresh interpreter (a process that already ran other profiler
# sessions may deliver no device activity to a later one).  Every call is made once outside the trace.  With the
# shared design the lag kernels run and the pilot launch of the pair-form Gram exits at once; with a perturbed copy
# (above the rule's bound) or a copy scaled by 2^-30 (the bound is relative) the lag kernels exit and the pair-form
# pilot Gram does its full work.
_PROFILE_SCRIPT = r"""
import json
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile
import sbce

N, n_tx, n_rx, M, T, B = 64, 4, 4, 16, 320, 64
out = {}
for case in ("shared", "perturbed", "scaled"):
    prob = sbce.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=T, T_d=T, itera=1, psip_shared=True)
    ses = sbce.DeviceSession(prob, B)
    g = ses.generate(B, 0.1, seed=3, pilot_design="top")
    P = g["PsiP"].clone()
    if case == "perturbed":
        P[7, 9] += 1e-11
    if case == "scaled":
        P *= 2.0 ** -30
    sm = g["Xd"].conj()
    sR = (sm[..., :, None] * g["Xd"][..., None, :]).contiguous()
    args = (g["Yd"], g["Yp"], g["PsiD"], P, g["Xp"], sm.contiguous(), sR)
    ses.mstep(*args)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ses.mstep(*args)
        torch.cuda.synchronize()
    out[case] = [(e.name, e.device_time_total) for e in prof.events() if e.device_type.name == "CUDA"]
print(json.dumps(out))
"""


@pytest.fixture(scope="module")
def traces(S):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-c", _PROFILE_SCRIPT], cwd=root, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def _grams(trace):
    """(pilot, data) durations of the two pair-form Gram launches of a solve-only M-step, in launch order."""
    g = [t for n, t in trace if "k_gram" in n]
    assert len(g) == 2, trace
    return g


def test_profiler_sees_the_lag_form_when_the_design_qualifies(traces):
    names = [n for n, _ in traces["shared"]]
    for k in ("k_pilot_lag_check", "k_pilot_lag_gram", "k_pilot_lag_expand"):
        assert any(k in n for n in names), (k, names)
    pilot, data = _grams(traces["shared"])
    assert pilot < 0.1 * data, traces["shared"]          # the pilot launch of the pair form exited at once


@pytest.mark.parametrize("case", ["perturbed", "scaled"])
def test_profiler_sees_the_pair_form_otherwise(traces, case):
    pilot, data = _grams(traces[case])
    assert pilot > 0.5 * data, traces[case]       # same T for pilots and data: comparable work
    lag = [t for n, t in traces[case] if "k_pilot_lag_gram" in n or "k_pilot_lag_expand" in n]
    assert lag and max(lag) < 0.1 * data, traces[case]
