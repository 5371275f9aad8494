"""CPU tests of the BASELINE.json workload table, the full-size oracle fixtures and bench.py's work models.
(The GPU side of the same fixtures is tests/test_gpu_configs.py.)"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import sbce
from conftest import load_golden
from oracle import em_numpy as orc
from oracle.make_config_golden import check_inputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workload_table_is_well_posed_and_supported():
    """Every workload: T_p + T_d >= 1.3 L (SURVEY 8d), the library accepts its shape (workspace query needs
    no GPU), and the headline is BASELINE.json configs[1] / north_star (N=64, 4x4, 16-QAM)."""
    W = sbce.workloads.WORKLOADS
    assert set(W) == {1, 2, 3, 4, 41, 5}
    for k, w in W.items():
        assert w.T_p + w.T_d >= 1.3 * w.L, k
        assert sbce.engine.workspace_bytes(w.problem(), 1) > 0
    h = sbce.workloads.HEADLINE
    assert (h.N, h.n_tx, h.n_rx, h.M, h.itera, h.mode, h.trials_per_step) == (64, 4, 4, 16, 10, "soft", 1184)
    assert W[5].L == 2056 and W[3].L == 514 and W[4].M ** W[4].n_tx == 65536
    assert W[41].problem().p1 == 2 and W[5].problem().p1 == 2        # p + 1 = 2 streams enumerated (PM.py:74-75)
    # 148 trials of workload 5 in flight fit a B200 (180 GB) with room to spare
    assert sbce.engine.workspace_bytes(W[5].problem(), 148) < 60e9


def test_long_phase_rows_are_rejected_not_launched():
    """N + 1 + n_tx^2 > 908 exceeds the shared-memory staging of the normal-equation kernels: the C ABI must
    answer SBCE_E_UNSUPPORTED (not an opaque launch failure), at the documented limit."""
    ok = sbce.Problem(N=906, n_tx=1, n_rx=1, M=4, T_p=8, T_d=8, itera=1)
    assert sbce.engine.workspace_bytes(ok, 1) > 0
    for bad in (sbce.Problem(N=907, n_tx=1, n_rx=1, M=4, T_p=8, T_d=8, itera=1),
                sbce.Problem(N=850, n_tx=8, n_rx=8, M=4, T_p=8, T_d=8, itera=1)):
        with pytest.raises(sbce.SbceError, match="unsupported"):
            sbce.engine.workspace_bytes(bad, 1)


@pytest.mark.parametrize("name,key", [("config_3_n256", 3), ("config_4_8x8qpsk", 4), ("config_41_64qam_pm", 41)])
def test_config_fixture_inputs_regenerate_bit_identically(name, key):
    """The fixture's SHA-256 pins the inputs; make_batch must reproduce them here exactly as it will on the GPU
    box, and the fixture's NMSE must be the oracle's NMSE of its own theta."""
    meta, g = load_golden(name)
    w = sbce.workloads.WORKLOADS[key]
    B, trials = int(meta["B"]), [int(t) for t in meta["trials"]]
    tb = sbce.workloads.make_batch(w, B)
    check_inputs(tb, trials, meta["digest"], g["probes"])
    for i, b in enumerate(trials):
        assert abs(orc.nmse(g["theta_ref"][i], tb.h[b]) - g["nmse_ref"][i]) <= 1e-12 * g["nmse_ref"][i]
    assert g["theta_ref"].shape == (len(trials), w.L, w.n_rx)


def test_config3_fixture_is_reproduced_by_the_oracle():
    """One fixture is re-derived in full on the CPU (N = 256, 2x2 QPSK: seconds): the committed arrays are the
    oracle's output, not stale files."""
    meta, g = load_golden("config_3_n256")
    w = sbce.workloads.WORKLOADS[3]
    tb = sbce.workloads.make_batch(w, int(meta["B"]))
    th, tr = orc.em(tb.Yd[0], tb.Yp[0], tb.PsiD[0], tb.PsiP[0], tb.Xp[0], w.M, w.varn, w.itera, theta0=tb.theta0[0],
                    return_trace=True)
    assert np.linalg.norm(th - g["theta_ref"][0]) <= 1e-12 * np.linalg.norm(th)
    assert np.array_equal(np.asarray(tr["kstar"]), g["kstar_ref"][0])


def test_headline_fixture_shape():
    meta, g = load_golden("config_headline_b1184")
    w = sbce.workloads.HEADLINE
    assert int(meta["B"]) == 1184 and [int(t) for t in meta["trials"]] == [0, 592]
    assert g["theta_ref"].shape == (2, w.L, w.n_rx) and g["kstar_ref"].shape == (2, w.T_d)
    assert g["lse_ref"].shape == (2, w.itera) and (g["nmse_ref"] < 0.02).all()


def test_host_arrays_layout():
    w = sbce.workloads.WORKLOADS[1]
    tb = sbce.workloads.make_batch(w, 3)
    d = sbce.workloads.host_arrays(w, tb, psip_shared=True)
    sh = w.problem(psip_shared=True).shapes(3)
    for k in ("Yd", "Yp", "PsiD", "PsiP", "Xp", "theta0", "h_true"):
        assert d[k].shape == tuple(sh[k]) and d[k].flags.c_contiguous, k
    assert d["PsiP"].shape == (w.T_p, w.N + 1) and d["varn"].shape == (3,)
    tb.PsiP[1, 0, 0] += 1.0
    with pytest.raises(ValueError):
        sbce.workloads.host_arrays(w, tb, psip_shared=True)


def test_bench_work_models_match_design_section_5():
    import bench

    wd = sbce.workloads.HEADLINE.as_dict()
    f, b = bench.flops_models(wd), bench.bytes_models(wd)
    P, T_d, L = 65 * 66 // 2, 256, 260
    assert f["gram"] == 72.0 * P * T_d + 8.0 * T_d * L * 4                 # 64 real-GEMM + 8 p_t flops per pair and symbol
    assert f["gram_survey"] == 4.0 * T_d * L * (L + 1) + 8.0 * T_d * L * 5
    assert abs(f["chol"] - (4.0 * L ** 3 / 3 + 32.0 * L * L)) < 1e-6
    assert 1.6 < f["gram_survey"] / f["gram"] < 1.9                        # the Hermitian-shared form does ~58 % of it
    assert b["chol"] == 2 * 16.0 * (260 * 261 / 2 + 4 * 260)
    w8 = sbce.workloads.WORKLOADS[5].as_dict()
    f8 = bench.flops_models(w8)
    assert f8["gram"] > 0 and f8["chol"] > 1.1e10                          # SURVEY: ~1.2e10 flops per Cholesky at L = 2056


def test_bench_dump_outputs_format_and_size_limit(tmp_path):
    """bench.py --dump-outputs: every array as float64 (complex ones with a trailing real/imag axis); above the
    size limit the same seeded sample of trials from every array, with its trial indices, within the limit."""
    import bench

    rng = np.random.default_rng(0)
    B = 50
    arrays = dict(theta=rng.standard_normal((B, 6, 2)) + 1j * rng.standard_normal((B, 6, 2)),
                  kstar=rng.integers(0, 16, (B, 7)).astype(np.int32), nmse=rng.random(B))
    assert bench.dump_outputs(str(tmp_path / "all"), arrays) == B
    assert sorted(os.listdir(tmp_path / "all")) == ["kstar.npy", "nmse.npy", "theta.npy"]
    th, ks = np.load(tmp_path / "all" / "theta.npy"), np.load(tmp_path / "all" / "kstar.npy")
    assert th.dtype == np.float64 and np.array_equal(th[..., 0] + 1j * th[..., 1], arrays["theta"])
    assert ks.dtype == np.float64 and np.array_equal(ks, arrays["kstar"])

    limit = 4096
    n = bench.dump_outputs(str(tmp_path / "a"), arrays, limit=limit)
    assert 0 < n < B and bench.dump_outputs(str(tmp_path / "b"), arrays, limit=limit) == n
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["kstar.npy", "nmse.npy", "theta.npy", "trial_index.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    idx = np.load(tmp_path / "a" / "trial_index.npy").astype(np.int64)
    assert len(idx) == n and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "nmse.npy"), arrays["nmse"][idx])


def test_bench_rejects_fewer_than_one_step():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (CPU oracle port) on the smallest workload: same metric / unit / config keys,
    impl = reference, a cpu_baseline describing the run, zero-copy e2e."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "1", "--steps", "1",
                          "--warmup", "0", "--cpu-sample-iters", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "trials/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["value"] > 0
    assert line["config"]["N"] == 32 and line["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    """Launched under torchrun with N > 1 the reference arm runs on rank 0 only: every other rank exits 0 without
    work and without printing a line."""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip() == ""
