#!/usr/bin/env python
"""bench.py -- EM channel-estimation trials/s on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C] [--trials-per-step B]
                    [--dump-outputs DIR]

Workload (default --config 2 = BASELINE.json configs[1], the north-star size): one NMSE-vs-T_d sweep point of
Proposed_method_NMSEvsTd.py scaled to N=64 RIS elements, 4x4 MIMO, 16-QAM (K = 65536 joint hypotheses per data
symbol), T_p=320, T_d=256, 10 EM iterations, soft-decision EM from the LS start, varn=0.1 -- an operating point
where the LS start is identifiable (T_p >= L=260) and EM improves the NMSE several-fold; at the reference's
T_p=16 the M-step is singular at this L.  `--config 1|3|4|41|5` times the other BASELINE.json workloads
(sbce/workloads.py) with the same line format.  A "step" is one batched call of the hot path over `B`
independent Monte-Carlo trials per GPU; trials are sharded across ranks (disjoint seeds, no data-path
collective) -> weak scaling.

Prints ONE JSON line (rank 0):
  value          trials/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e            the same through the host-buffer C-ABI entry point sbce_em_batch_host: pinned host memory -> H2D ->
                 kernels -> D2H inside the timed region; with N > 1 ranks the per-point NMSE/SER accumulators are
                 summed over NCCL inside the timed region too (the one collective of a sweep)
  e2e_on_device  a whole sweep point without PCIe traffic: Philox generation, LS start, EM and the NMSE/SER
                 accumulation on the device, one NCCL sum + one 6-double read-back at the end (timed)
  sweep          the GLOBAL (all ranks) NMSE / SER of the timed sweep points and, for N > 1, a check that the
                 NCCL-reduced sums equal a single-rank recomputation of the same Philox trials
  parity         (config 2, B=1184) the timed outputs against the committed oracle fixture
                 tests/golden/config_headline_b1184.npz, and the e2e route against the device route bitwise
  roofline / kernels / cpu_baseline / clocks as the driver contract asks.
`--impl reference` times the CPU restatement of the reference (oracle/em_numpy.py; the literal reference is
Python that cannot travel and takes weeks per trial at this size, BASELINE.md section 4.1) on the host cores,
on the same config/metric/unit.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "EM channel-estimation trials/sec"
UNIT = "trials/s"
NCU_TRAFFIC_FILE = os.path.join(ROOT, "profiles", "ncu_traffic.json")
HEADLINE_FIXTURE = os.path.join(ROOT, "tests", "golden", "config_headline_b1184.npz")


# ---------------------------------------------------------------------------
# algorithmic work models (stated in DESIGN.md section 5)
# ---------------------------------------------------------------------------

def flops_models(w):
    """Per trial-iteration flop counts (add = mul = 1, FMA = 2); stated in DESIGN.md section 5.
    `*_survey` entries are SURVEY.md section 8d's algorithmic figures; the un-suffixed ones count what the
    kernels of this repository execute (used for roofline fractions, so that a cheaper algorithm does
    not read as a higher utilisation)."""
    N1, n_tx, n_rx, M, T_d = w["N"] + 1, w["n_tx"], w["n_rx"], w["M"], w["T_d"]
    L = N1 * n_tx
    P = N1 * (N1 + 1) // 2
    sq = int(round(M ** 0.5))
    lg = int(math.log2(sq // 2)) if sq >= 2 else 0
    # hypothesis tree, FULL scan: every deepest node (M^(n_tx-1) of them) costs the separable update of the
    # row-0 residual (2 FMA), its partial distance (1 add), two folds (1+log2(sqrt(M)/2) subtractions each),
    # the leaf minimum (2 FMA) and one compare; each group of M deepest nodes shares 4 sqrt(M) flops of
    # separable level-1 distances; prefix levels cost ~6+2s flops per node above.
    nodes = float(M) ** (n_tx - 1)
    f_node = 4 + 1 + 2 * (1 + lg) + 4 + 1
    enum = nodes * f_node
    if n_tx >= 2:
        enum += (nodes / M) * 4 * sq
    cnt = 1.0
    for s in range(n_tx - 1, 1, -1):
        cnt *= M
        enum += cnt * (6 + 2 * s)
    nr = max(n_rx, n_tx)
    # Hermitian-shared real GEMM: per (RIS pair, symbol) 2 rows x NC real columns x 2 flops (+ 8 for p_t);
    # NC = n_tx diagonal columns + 2 per upper entry, padded to a multiple of 8 on the tensor path
    nc = n_tx + n_tx * (n_tx - 1)
    if n_tx >= 4:
        nc = ((n_tx + 1) // 2 * 2 + n_tx * (n_tx - 1) + 7) // 8 * 8
    gram_exec = (2.0 * 2.0 * nc + 8.0) * P * T_d
    return dict(
        enum_full_scan=T_d * enum,
        heff_qr=T_d * (8.0 * N1 * n_tx * n_rx + 16.0 * n_tx * n_tx * nr),
        gram=gram_exec + 8.0 * T_d * L * n_rx,          # Hermitian-shared real GEMM + p_t generation + rhs rows
        gram_survey=4.0 * T_d * L * (L + 1) + 8.0 * T_d * L * (n_rx + 1),   # SURVEY 8d F_G + F_B
        chol=4.0 * L ** 3 / 3.0 + 8.0 * n_rx * L * L,   # SURVEY 8d F_S (complex Cholesky + two triangular solves)
        survey_estep=T_d * (float(M) ** n_tx * (2 * n_tx * n_rx + 4 * n_rx + 3 + 4 * n_tx + 2 * n_tx * (n_tx + 1))
                            + 8.0 * N1 * n_tx * n_rx + 8.0 * n_tx * M * n_rx),  # SURVEY 8d F_E (naive enumeration)
    )


def bytes_models(w):
    """Algorithmic DRAM bytes per trial-iteration of the kernels that have an HBM side (DESIGN.md section 5)."""
    N1, n_tx, n_rx, T_d = w["N"] + 1, w["n_tx"], w["n_rx"], w["T_d"]
    L = N1 * n_tx
    Lp = (L + 3) // 4 * 4
    rec = n_tx * (n_tx + 1) + 2 * n_tx + 2
    tri = 16.0 * (Lp * (Lp + 1) / 2 + ((n_rx + 3) // 4 * 4) * Lp)      # packed lower trapezoid [G ; B^H]
    return dict(heff_qr=T_d * (16.0 * (N1 + n_rx) + 8.0 * rec),        # psi row + y in, QR record out
                chol=2.0 * tri,                                        # factor read once + written once
                gram=16.0 * T_d * (N1 + n_tx * n_tx + n_tx + n_rx) + 2.0 * tri)   # operands in, G_p in, G out


# ---------------------------------------------------------------------------
# clocks sampling
# ---------------------------------------------------------------------------

class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.p is None:
            return out
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().strip().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                 parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


DUMP_LIMIT_BYTES = 64 * 10 ** 6
DUMP_SAMPLE_SEED = 20261


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT_BYTES):
    """Writes the per-trial outputs `arrays` (name -> array with the trial index outermost) to
    out_dir/<name>.npy as float64; complex arrays gain a trailing (real, imag) axis.  When the files would exceed
    `limit` bytes in all, the same fixed, seeded sample of trials is written from every array, and its trial
    indices go to out_dir/trial_index.npy.  Returns the number of trials written."""
    import numpy as np

    conv = {}
    for name, a in arrays.items():
        a = np.ascontiguousarray(a)
        conv[name] = a.view(np.float64).reshape(a.shape + (2,)) if a.dtype.kind == "c" else a.astype(np.float64)
    B = next(iter(conv.values())).shape[0]
    per_trial = sum(a.nbytes for a in conv.values()) // max(1, B)
    payload = limit - 256 * (len(conv) + 1)          # room for the .npy headers
    keep = B if per_trial * B <= payload else max(1, payload // (per_trial + 8))
    os.makedirs(out_dir, exist_ok=True)
    idx = None
    if keep < B:
        idx = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(B, size=keep, replace=False))
        np.save(os.path.join(out_dir, "trial_index.npy"), idx.astype(np.float64))
    for name, a in conv.items():
        np.save(os.path.join(out_dir, name + ".npy"), a if idx is None else a[idx])
    return keep


def workload_dict(w):
    d = w.as_dict()
    d.update(partition_r=w.partition_r, quirks=w.quirks, zero_start=w.zero_start)
    return d


def cpu_sample(wd, sample_iters, seed=1234):
    """One bounded sample of the CPU arm (oracle/cpu_bench.py) in a FRESH interpreter: the worker pool is forked
    from a process without a CUDA context or pinned buffers (forking the GPU process cost ~80 s per pool)."""
    out = subprocess.run([sys.executable, "-m", "oracle.cpu_bench", json.dumps(wd), str(int(sample_iters)), str(int(seed))],
                         cwd=ROOT, capture_output=True, text=True, timeout=1800)
    if out.returncode != 0:
        raise RuntimeError("cpu_bench failed: " + out.stderr[-800:])
    return json.loads(out.stdout.strip().splitlines()[-1])


# ---------------------------------------------------------------------------
# reference arm (CPU)
# ---------------------------------------------------------------------------

def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import importlib

    workloads = importlib.import_module("sbce").workloads      # shapes only: nothing of the product runs here

    w = workloads.WORKLOADS[args.config]
    wd = workload_dict(w)
    vals, last = [], None
    # every step is one bounded sample: all host cores, one trial each, `it` EM iterations from the LS start,
    # scaled to the full iteration count.  Long runs (the driver's --steps 20 --warmup 5) use one iteration per
    # sample so that the whole run stays within a few minutes (~7 s per sample at the headline size).
    it_timed = args.cpu_sample_iters if (args.steps + args.warmup) <= 12 else 1
    for i in range(args.warmup + args.steps):
        r = cpu_sample(wd, it_timed if i >= args.warmup else 1, seed=1000 + 97 * i)
        if i >= args.warmup:
            vals.append(r)
        last = r
    tot_slices = sum(r["cores"] * r["sample_iters"] for r in vals) / float(w.itera)     # trial-equivalents processed
    tot_time = sum(r["slowest_worker_s"] for r in vals)
    value = tot_slices / tot_time
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * tot_time / max(1, len(vals)), higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic", impl="reference",
                config=dict(workload=w.describe(), **w.as_dict()),
                cpu_baseline=dict(value=value, unit=UNIT, cores=last["cores"], kind="port", sample=last["sample"]),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------
# our arm (GPU)
# ---------------------------------------------------------------------------

def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as tdist

    import sbce
    from sbce import dist as sdist, engine, workloads

    rank, world, local = sdist.init_from_env("nccl")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sbce._lib.require_device()

    w = workloads.WORKLOADS[args.config]
    wd = w.as_dict()
    B = args.trials_per_step or w.trials_per_step
    prob = w.problem(psip_shared=True)
    tree = w.mode in ("soft", "hard")
    pilot_design = "pm" if w.variant == "pm" else "top"
    data_phases = "dft" if w.variant == "top_td" else "random"
    ses = engine.DeviceSession(prob, B, device=dev)

    # ---- synthetic inputs.  The headline workload is generated once by numpy on the host (disjoint seed per
    # rank; the parity fixture is minted from rank 0's batch); the other workloads come from the on-device
    # Philox generator + LS start (host generation needs an SVD per trial, minutes at L = 2056) and are copied
    # back to pinned host memory for the end-to-end leg.
    host_generated = (w.key == 2) and not args.device_inputs
    if host_generated:
        tb = workloads.make_batch(w, B, seed=workloads.bench_seed(w, rank))
        host_in = workloads.host_arrays(w, tb, psip_shared=True)
        t_dev = {k: torch.from_numpy(v).to(dev) for k, v in host_in.items()}
    else:
        g = ses.generate(B, w.varn, seed=workloads.bench_seed(w, rank), trial0=rank * B, pilot_design=pilot_design,
                         data_phases=data_phases)
        theta0, _ = (None, None) if w.zero_start else ses.ls_start(g["Yp"], g["PsiP"], g["Xp"])
        t_dev = dict(Yd=g["Yd"], Yp=g["Yp"], PsiD=g["PsiD"], PsiP=g["PsiP"], Xp=g["Xp"], h_true=g["h"], varn=g["varn"])
        if theta0 is not None:
            t_dev["theta0"] = theta0
        torch.cuda.synchronize()
        host_in = {k: v.cpu().numpy() for k, v in t_dev.items()}
    input_bytes = sum(v.nbytes for v in host_in.values())
    out = ses.alloc_outputs(B, llf=False, lse=True, nmse=True, kstar=True)

    def step():
        ses.run(t_dev["Yd"], t_dev["Yp"], t_dev["PsiD"], t_dev["PsiP"], t_dev["Xp"], t_dev["varn"],
                theta0=t_dev.get("theta0"), h_true=t_dev["h_true"], out=out)

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    fp64_peak = engine.fp64_peak_tflops()          # live DFMA microbenchmark (no FP64 entry in MEASURED_PEAKS.json)
    barrier()

    sampler = ClockSampler(local)
    sampler.start()
    engine.launch_count(reset=True)
    engine.profile_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    phases = engine.profile_end()
    launches = engine.launch_count()
    clocks = sampler.stop()
    tms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        tdist.all_reduce(tms, op=tdist.ReduceOp.MAX)
    ms_max = float(tms.item())
    value = world * B * args.steps / (ms_max * 1e-3)

    # ---- same workload with the E-step forced to visit every node of the hypothesis tree
    # (SBCE_FLAG_FULL_SCAN; outputs are bit-identical, see tests) -- reported next to the headline
    full = None
    if tree and not (args.no_full_scan or args.kernels_only):
        import dataclasses

        prob_fs = dataclasses.replace(prob, full_scan=True)
        ses_fs = engine.DeviceSession(prob_fs, B, device=dev)
        out_fs = ses_fs.alloc_outputs(B, llf=False, lse=True, nmse=True, kstar=True)

        def step_fs():
            ses_fs.run(t_dev["Yd"], t_dev["Yp"], t_dev["PsiD"], t_dev["PsiP"], t_dev["Xp"], t_dev["varn"],
                       theta0=t_dev.get("theta0"), h_true=t_dev["h_true"], out=out_fs)

        step_fs()
        barrier()
        engine.profile_begin()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nfs = args.steps
        f0.record()
        for _ in range(nfs):
            step_fs()
        f1.record()
        barrier()
        ph_fs = engine.profile_end()
        tfs = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
        if world > 1:
            tdist.all_reduce(tfs, op=tdist.ReduceOp.MAX)
        same = bool(torch.equal(out_fs.theta, out.theta) and torch.equal(out_fs.kstar, out.kstar))
        full = dict(value=world * B * nfs / (float(tfs.item()) * 1e-3), unit=UNIT, steps=nfs,
                    enum_avg_launch_ms=ph_fs["enum"][0] / max(1, ph_fs["enum"][1]),
                    outputs_bit_identical_to_default=same)
        del ses_fs, out_fs

    # sanity: the timed work produced valid estimates
    nm = out.nmse.cpu().numpy()
    st = out.status.cpu().numpy()
    nmse_mean = float(nm[st == 0].mean()) if (st == 0).any() else float("nan")
    th0 = host_in.get("theta0")
    nmse_init = None if th0 is None else float(np.mean([sbce.nmse(th0[i], host_in["h_true"][i]) for i in range(min(B, 64))]))
    dev_out = {k: getattr(out, k).cpu().numpy() for k in ("theta", "kstar", "lse", "nmse", "iters", "status")}

    # ---- end-to-end through the host-buffer C-ABI entry point, pinned host memory; with several ranks the
    # per-point accumulators (sum NMSE, valid trials, flagged trials) are summed over NCCL inside the timed region
    e2e = None
    e2e_equal = None
    if not args.kernels_only:
        pin = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory().numpy() for k, v in host_in.items()}
        hout = engine.alloc_host_outputs(prob, B, want=("kstar", "lse", "nmse", "iters", "status"), pinned=True)
        d2h_bytes = sum(getattr(hout, k).nbytes for k in ("theta", "kstar", "lse", "nmse", "iters", "status"))

        def e2e_step():
            engine.run_host(prob, pin["Yd"], pin["Yp"], pin["PsiD"], pin["PsiP"], pin["Xp"], pin["varn"],
                            theta0=pin.get("theta0"), h_true=pin["h_true"], device=local, out=hout)

        def point_acc():
            ok = hout.status == 0
            return np.array([float(hout.nmse[ok].sum()), float(ok.sum()), float((~ok).sum())])

        # --steps synchronous calls.  Single calls sporadically take 1.3-5x longer on a shared host, so with few
        # steps one such call moves the mean noticeably; e2e.median_step_ms shows the steady state.
        # warm-up: pool allocation and >= 1.5 s of steady calls.  On a shared host single calls sporadically
        # take 1.5-2x longer for ~0.3 s at a time (SM clock and the copy rate unchanged; the device-timed `value`
        # queues its kernels ahead and does not see it): e2e.value is the honest mean over the timed calls,
        # e2e.median_step_ms shows the steady state
        tw, nw = time.perf_counter(), 0
        while nw < max(3, args.warmup) or (w.key == 2 and time.perf_counter() - tw < 1.5):
            e2e_step()
            nw += 1
        e2e_equal = all(np.array_equal(getattr(hout, k), dev_out[k], equal_nan=(dev_out[k].dtype.kind in "fc"))
                        for k in dev_out)
        barrier()
        # plain pinned-host -> device copy rate of this box (explains how far e2e can sit below `value`)
        big = max(pin.values(), key=lambda a: a.nbytes)
        tsrc = torch.from_numpy(big)
        tdst = torch.empty(tsrc.shape, dtype=tsrc.dtype, device=dev)
        tdst.copy_(tsrc, non_blocking=True)
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(3):
            tdst.copy_(tsrc, non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        h2d_gbs = 3 * big.nbytes / (c0.elapsed_time(c1) * 1e-3) / 1e9
        del tdst
        barrier()
        step_ms, accs = [], []
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ta = time.perf_counter()
            e2e_step()          # synchronous: returns after the D2H copies completed
            accs.append(point_acc())
            step_ms.append(1e3 * (time.perf_counter() - ta))
        acc_global = sdist.allreduce_sum(np.stack(accs), device=dev)   # NCCL sum (no-op on one rank)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        te = torch.tensor([t1 - t0], dtype=torch.float64, device=dev)
        if world > 1:
            tdist.all_reduce(te, op=tdist.ReduceOp.MAX)
        e2e = dict(value=world * B * args.steps / float(te.item()), unit=UNIT,
                   h2d_bytes_per_step=int(input_bytes) * world, d2h_bytes_per_step=int(d2h_bytes) * world,
                   bytes_are="whole job (all ranks)", steps=args.steps, warmup_calls=nw,
                   step_ms=[round(x, 2) for x in step_ms], median_step_ms=round(statistics.median(step_ms), 2),
                   h2d_gbs_measured=h2d_gbs,
                   collective="one NCCL sum of %d float64 inside the timed region" % acc_global.size if world > 1 else None,
                   nmse_global=float(acc_global[:, 0].sum() / max(1.0, acc_global[:, 1].sum())),
                   trials_global=float(acc_global[:, 1:].sum()))

    # ---- a sweep on the device only: step i = sweep point i, this rank owns global trials [rank*B, (rank+1)*B)
    # of every point (counter-based generator: the trials do not depend on the sharding)
    ondev = None
    sweep = None
    if not args.kernels_only:
        n_pts = args.steps
        acc_n = torch.zeros((n_pts, 3), dtype=torch.float64, device=dev)
        acc_s = torch.zeros((n_pts, 3), dtype=torch.float64, device=dev)
        sweep_seed = 777000 + 1000 * w.key

        def point(i, trial0, an, as_):
            gg = ses.generate(B, w.varn, seed=sweep_seed + i, trial0=trial0, pilot_design=pilot_design,
                              data_phases=data_phases)
            th0_, st0 = (None, None) if w.zero_start else ses.ls_start(gg["Yp"], gg["PsiP"], gg["Xp"])
            r = ses.run(gg["Yd"], gg["Yp"], gg["PsiD"], gg["PsiP"], gg["Xp"], gg["varn"], theta0=th0_, h_true=gg["h"])
            if st0 is not None:
                r.status.bitwise_or_(st0)
            ses.accumulate(r, gg["Xd"], an, as_)

        for i in range(min(2, n_pts)):                       # warm-up (allocator, generator kernels)
            point(i, rank * B, acc_n[i], acc_s[i])
        acc_n.zero_()
        acc_s.zero_()
        barrier()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw0 = time.perf_counter()
        o0.record()
        for i in range(n_pts):
            point(i, rank * B, acc_n[i], acc_s[i])
        both = torch.cat([acc_n, acc_s], dim=1)
        if world > 1:
            tdist.all_reduce(both, op=tdist.ReduceOp.SUM)    # NCCL: the one collective of the sweep
        o1.record()
        glob = both.cpu().numpy()                             # read-back of n_pts x 6 doubles (synchronises)
        tw1 = time.perf_counter()
        tod = torch.tensor([o0.elapsed_time(o1), 1e3 * (tw1 - tw0)], dtype=torch.float64, device=dev)
        if world > 1:
            tdist.all_reduce(tod, op=tdist.ReduceOp.MAX)
        ondev = dict(value=world * B * n_pts / (float(tod[1].item()) * 1e-3), unit=UNIT, steps=n_pts,
                     device_ms_per_step=float(tod[0].item()) / n_pts, wall_ms_per_step=float(tod[1].item()) / n_pts,
                     h2d_bytes_per_step=0, d2h_bytes_per_step=int(glob.nbytes / n_pts),
                     includes="Philox generation + LS start + EM + NMSE/SER accumulation"
                              + (" + NCCL all-reduce" if world > 1 else "") + " + accumulator read-back; timed by host "
                              "wall clock around the loop (max over ranks)")
        has_ser = glob[:, 4] > 0
        sweep = dict(points=n_pts, trials_per_point=world * B,
                     nmse=[float(a / max(1.0, c)) for a, c in zip(glob[:, 0], glob[:, 1])],
                     flagged=[float(x) for x in glob[:, 2]],
                     ser=[float(e / t) if ok else None for e, t, ok in zip(glob[:, 3], glob[:, 4], has_ser)],
                     reduced_over="NCCL all_reduce(SUM), %d ranks" % world if world > 1 else "single rank")
        if world > 1 and rank == 0:
            # sharding invariance: rank 0 alone recomputes point 0 over ALL world*B trials; the sums must agree
            # up to summation order
            an1 = torch.zeros(3, dtype=torch.float64, device=dev)
            as1 = torch.zeros(3, dtype=torch.float64, device=dev)
            for r_ in range(world):
                point(0, r_ * B, an1, as1)
            one = torch.cat([an1, as1]).cpu().numpy()
            rel = float(abs(one[0] - glob[0, 0]) / max(abs(one[0]), 1e-300))
            sweep["single_rank_check"] = dict(nmse_sum_single_rank=float(one[0]), nmse_sum_reduced=float(glob[0, 0]),
                                              rel_diff=rel, counts_equal=bool(np.array_equal(one[[1, 2, 3, 4]],
                                                                                             glob[0, [1, 2, 3, 4]])),
                                              ok=bool(rel < 1e-12 and np.array_equal(one[[1, 2, 3, 4]], glob[0, [1, 2, 3, 4]])))

    if rank != 0:
        if world > 1:
            tdist.barrier()
            tdist.destroy_process_group()
        return 0

    # ---- parity of the timed outputs against the committed oracle fixture (headline, rank 0, B = 1184)
    parity = None
    if host_generated and os.path.exists(HEADLINE_FIXTURE):
        z = np.load(HEADLINE_FIXTURE, allow_pickle=False)
        if int(z["meta_B"]) == B:
            rel, keq, nrel, lrel = 0.0, True, 0.0, 0.0
            for i, b in enumerate(int(t) for t in z["meta_trials"]):
                ref = z["theta_ref"][i]
                rel = max(rel, float(np.linalg.norm(dev_out["theta"][b] - ref) / np.linalg.norm(ref)))
                keq = keq and bool(np.array_equal(dev_out["kstar"][b], z["kstar_ref"][i]))
                nrel = max(nrel, float(abs(dev_out["nmse"][b] - z["nmse_ref"][i]) / z["nmse_ref"][i]))
                lrel = max(lrel, float(np.max(np.abs(dev_out["lse"][b] - z["lse_ref"][i]) / np.abs(z["lse_ref"][i]))))
            parity = dict(fixture="tests/golden/config_headline_b1184.npz (oracle/make_config_golden.py)",
                          trials_checked=[int(t) for t in z["meta_trials"]], iterations=w.itera, max_rel_theta=rel,
                          kstar_equal=keq, max_rel_nmse=nrel, max_rel_lse=lrel,
                          e2e_route_equals_device_route_bitwise=e2e_equal,
                          ok=bool(rel < 1e-9 and keq and nrel < 5e-5 and (e2e_equal is not False)))
    elif e2e_equal is not None:
        parity = dict(fixture=None, e2e_route_equals_device_route_bitwise=e2e_equal,
                      note="oracle parity of this workload: tests/test_gpu_configs.py")

    # ---- per-kernel roofline from the CUDA-event phase timers recorded inside the timed region
    fm, bm = flops_models(wd), bytes_models(wd)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    total_phase_ms = sum(v[0] for v in phases.values())
    kernels = {}
    for name, (pms, cnt) in phases.items():
        if cnt == 0:
            continue
        avg_s = pms * 1e-3 / cnt
        k = dict(ms_total=pms, launches=cnt, share=pms / total_phase_ms, avg_launch_ms=1e3 * avg_s)
        if name in fm and not (name == "enum"):
            k["tflops"] = fm[name] * B / avg_s / 1e12
            k["frac_fp64_peak"] = k["tflops"] / fp64_peak if fp64_peak > 0 else None
        if name + "_survey" in fm:
            k["tflops_survey_model"] = fm[name + "_survey"] * B / avg_s / 1e12
            k["frac_fp64_peak_survey_model"] = k["tflops_survey_model"] / fp64_peak if fp64_peak > 0 else None
        if name in bm:
            k["gbs"] = bm[name] * B / avg_s / 1e9
            k["frac_hbm_peak"] = k["gbs"] / hbm_peak
        kernels[name] = k
    # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture
    ncu_traffic, ncu_src = {}, None
    try:
        t = json.load(open(NCU_TRAFFIC_FILE))
        ent = t.get("config_%d" % w.key)
        if ent and int(ent["trials_per_launch"]) > 0:
            ncu_traffic = {k: v * (B / float(ent["trials_per_launch"])) for k, v in ent["dram_bytes_per_launch"].items()}
            ncu_src = ent["source"]
    except Exception:
        pass
    for name, v in ncu_traffic.items():
        if name in kernels:
            kernels[name]["dram_bytes_per_launch_ncu"] = v
            if name in bm:
                kernels[name]["dram_over_algorithmic"] = v / (bm[name] * B)
    with_model = [n for n in kernels if "tflops" in kernels[n]]
    roofline = None
    if with_model:
        top = max(with_model, key=lambda n: kernels[n]["ms_total"])
        roofline = dict(bound="tensor", pipe="FP64 tensor path (mma.sync DMMA; tcgen05 has no FP64 kind)", kernel=top,
                        achieved=kernels[top]["tflops"], peak=fp64_peak, unit="TFLOP/s",
                        frac=kernels[top]["frac_fp64_peak"],
                        frac_survey_model=kernels[top].get("frac_fp64_peak_survey_model"),
                        traffic=ncu_traffic.get(top), traffic_unit="bytes per launch (ncu dram read+write, %s)" % ncu_src,
                        share_of_step=kernels[top]["share"],
                        peak_source="live DFMA micro-benchmark in libsbce (2 flop/FMA); MEASURED_PEAKS.json has no FP64 entry",
                        flops_per_launch=fm[top] * B,
                        note="achieved = EXECUTED flops of the kernel (DESIGN.md section 5) / CUDA-event launch time; "
                             "frac_survey_model uses SURVEY 8d's algorithmic figure, which counts the Hermitian-shared "
                             "work the kernel does not do")
        if "heff_qr" in kernels and "gbs" in kernels["heff_qr"]:
            roofline["hbm_side"] = dict(kernel="heff_qr", achieved=kernels["heff_qr"]["gbs"], peak=hbm_peak, unit="GB/s",
                                        frac=kernels["heff_qr"]["frac_hbm_peak"], peak_source=hbm_src)
    if "enum" in kernels and tree:
        kernels["enum"]["note"] = ("default E-step skips provably weightless subtrees: executed work is data "
                                   "dependent, see full_scan.enum_* for the fixed-work variant")
    if full is not None:
        es = full["enum_avg_launch_ms"] * 1e-3
        full["enum_tflops"] = fm["enum_full_scan"] * B / es / 1e12
        full["enum_frac_fp64_peak"] = full["enum_tflops"] / fp64_peak if fp64_peak > 0 else None
        full["enum_survey_model_tflops"] = fm["survey_estep"] * B / es / 1e12

    # ---- CPU baseline (oracle port) on a bounded sample, rank 0, N=1 only
    cpu = None
    if world == 1 and not (args.no_cpu_baseline or args.kernels_only):
        r = cpu_sample(workload_dict(w), args.cpu_sample_iters)
        cpu = dict(value=r["trials_per_s"], unit=UNIT, cores=r["cores"], kind="port", sample=r["sample"],
                   seconds=r["seconds"])

    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms_max / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f64", data="synthetic",
                config=dict(workload=w.describe(), baseline_json_config=w.key, source=w.source,
                            trials_per_step_per_gpu=B, pilot_design=w.variant,
                            inputs="numpy on the host, uploaded once" if host_generated else
                                   "on-device Philox generator + LS start (sbce_generate_batch / sbce_ls_start)",
                            layout="deterministic pilot phases passed once per batch; data phases, symbols, channels per trial",
                            enumeration=("exact posterior over all M^n_tx hypotheses; subtrees that provably carry no "
                                         "weight (partial distance > incumbent + 64 varn^2) are skipped, outputs "
                                         "bit-identical to the full scan (see full_scan)") if tree else
                                        "partitioned candidate lists (PM.py:61-104), p+1 = %d streams enumerated" % prob.p1,
                            l2="inputs (%.0f MB per GPU) %s the 126 MB L2" % (input_bytes / 1e6,
                                                                            "larger than" if input_bytes > 126e6 else
                                                                            "smaller than (workspace per step %.0f MB exceeds it)"
                                                                            % (ses.ws_bytes / 1e6)), **wd),
                e2e=e2e, e2e_on_device=ondev, sweep=sweep, parity=parity,
                gpu_launches=int(launches), clocks=clocks, roofline=roofline, kernels=kernels, cpu_baseline=cpu,
                full_scan=full,
                check=dict(nmse_mean=nmse_mean, nmse_ls_start=nmse_init, flagged_trials=int((st != 0).sum())))
    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, dev_out)
    print(json.dumps(line))
    if world > 1:
        tdist.barrier()
        tdist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6,
                    help="timed steps of every leg (device route, full scan, e2e, on-device sweep points)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 41, 5],
                    help="BASELINE.json workload (sbce/workloads.py); 2 = configs[1], the headline")
    ap.add_argument("--trials-per-step", type=int, default=0, help="trials per GPU per step (0: the workload's default)")
    ap.add_argument("--cpu-sample-iters", type=int, default=2, help="EM iterations each CPU worker runs (bounded sample)")
    ap.add_argument("--device-inputs", action="store_true", help="headline too: generate the inputs on the device")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-scan", action="store_true")
    ap.add_argument("--kernels-only", action="store_true", help="device-resident leg only (kernel tuning runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (theta, kstar, lse, nmse, "
                         "iters, status of rank 0's trials) to DIR/<name>.npy as float64, at most 64 MB in all; "
                         "inputs depend only on the arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
