"""Exact Gray-labelled bit LLRs (sbce_bit_llr, k_bit_llr) and bit-error counts (sbce_accumulate_ber) on the GPU,
against the numpy oracle of tests/llr_oracle.py and against closed forms, plus the BER curves of the drivers."""
import os
import re
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import llr_oracle as lo  # noqa: E402

pytestmark = pytest.mark.gpu

CLAMP = 32.0


@pytest.fixture(scope="module")
def S(cuda_device):
    import sbce

    sbce._lib.require_device()
    return sbce


@pytest.fixture(scope="module")
def orc():
    from oracle import em_numpy

    return em_numpy


def _t(S, a, dev):
    import torch

    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def gpu_llr(S, Yd, PsiD, theta, varn, n_tx, M, mode="soft", full_scan=False, Xoff=None, psi_shared=False,
            in_flight=None, out=None):
    import torch

    B, T_d, n_rx = Yd.shape
    N = PsiD.shape[-1] - 1
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=0, T_d=T_d, itera=1, mode=mode, full_scan=full_scan,
                     superimposed=Xoff is not None, psi_shared=psi_shared)
    ses = S.DeviceSession(prob, in_flight or B)
    vn = np.broadcast_to(np.asarray(varn, np.float64), (B,))
    r = ses.bit_llr(_t(S, Yd, ses.device), _t(S, PsiD, ses.device), _t(S, theta, ses.device), _t(S, vn, ses.device),
                    Xp=_t(S, Xoff, ses.device), out=out)
    torch.cuda.synchronize()
    return r.cpu().numpy()


def inputs(S, n_tx, n_rx, M, T_d, B, seed, N=2):
    tb = S.signal_model.generate_batch(N, n_tx, n_rx, M, 4, T_d, 0.01, B, seed=seed, legacy=False)
    rng = np.random.default_rng(seed)
    theta = tb.h + 0.05 * (rng.standard_normal(tb.h.shape) + 1j * rng.standard_normal(tb.h.shape))
    return tb, theta


def oracle_llr(orc, Yd, PsiD, theta, M, n_tx, varn, Xoff=None):
    """Unclamped oracle values of one trial; the split enumeration for the 2^24-leaf trees."""
    cons = orc.qam_constellation(M)
    f = lo.bit_llr_split if M ** n_tx > (1 << 20) else lo.bit_llr
    return f(Yd, PsiD, theta, cons, n_tx, varn, Xoff=Xoff, clamp=False)


def check_against_oracle(got, raw):
    """|llr - clamp(oracle)| <= 1e-8; oracle beyond +-(32 + 1e-6): exactly +-32; hard bits agree where |llr| > 1e-6."""
    assert got.shape == raw.shape
    beyond = np.abs(raw) > CLAMP + 1e-6
    assert np.array_equal(got[beyond], np.sign(raw[beyond]) * CLAMP)
    np.testing.assert_allclose(got, np.clip(raw, -CLAMP, CLAMP), rtol=0, atol=1e-8)
    sure = np.abs(raw) > 1e-6
    assert np.array_equal(got[sure] < 0, raw[sure] < 0)


SHAPES = ([(n, M) for n in (1, 2, 3, 4) for M in (4, 16, 64)] + [(n, 4) for n in (5, 6, 7, 8)] + [(5, 16), (6, 16)])


@pytest.mark.parametrize("n_tx,M", SHAPES)
@pytest.mark.parametrize("regime", ["peaked", "flat"])
def test_every_shape_against_the_oracle(S, orc, n_tx, M, regime):
    big = M ** n_tx > (1 << 16)
    T_d = 3 if big else 7
    B = 1 if big else 2
    tb, theta = inputs(S, n_tx, n_tx, M, T_d, B, seed=100 * n_tx + M)
    varn = 0.1 if regime == "peaked" else {4: 3.0, 16: 6.0, 64: 10.0}[M]
    got = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M)
    assert got.shape == (B, T_d, n_tx, int(np.log2(M)))
    clamped = []
    for b in range(B):
        raw = oracle_llr(orc, tb.Yd[b], tb.PsiD[b], theta[b], M, n_tx, varn)
        check_against_oracle(got[b], raw)
        clamped.append(np.abs(got[b]) == CLAMP)
    frac = np.mean(clamped)
    if regime == "peaked":
        assert frac > 0.5
    else:
        assert frac < 0.5


@pytest.mark.parametrize("n_rx", [1, 3])
def test_single_stream_qpsk_closed_form(S, orc, n_rx):
    """n_tx = 1, QPSK: llr_I = -4 Re(h^H y) / varn^2, llr_Q = -4 Im(h^H y) / varn^2 (clamped), no enumeration."""
    tb, theta = inputs(S, 1, n_rx, 4, 33, 2, seed=5)
    clamped = []
    for varn in (1.3, 0.3):   # mostly inside the clamp, mostly clamped
        got = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, 1, 4)
        for b in range(2):
            h = orc.effective_channels(tb.PsiD[b], theta[b], 1)[:, :, 0]          # (T_d, n_rx)
            z = np.einsum("tr,tr->t", h.conj(), tb.Yd[b])
            ref = np.stack([-4 * z.real, -4 * z.imag], axis=1) / varn ** 2
            np.testing.assert_allclose(got[b, :, 0], np.clip(ref, -CLAMP, CLAMP), rtol=0, atol=1e-9)
        clamped.append(np.mean(np.abs(got) == CLAMP))
    assert clamped[0] < 0.5 < clamped[1]


@pytest.mark.parametrize("n_tx,M,varn", [(4, 16, 0.1), (4, 16, 2.0), (8, 4, 0.3), (2, 64, 0.5), (5, 16, 0.2)])
def test_pruned_equals_full_scan_and_modes_agree(S, n_tx, M, varn):
    tb, theta = inputs(S, n_tx, n_tx, M, 9, 2, seed=9 + n_tx)
    a = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M)
    f = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, full_scan=True)
    np.testing.assert_allclose(a, f, rtol=0, atol=1e-12)
    h = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, mode="hard")
    assert np.array_equal(a, h), "soft and hard modes give the same LLRs"


def test_superimposed_offsets_and_shared_phases(S, orc):
    n_tx, n_rx, M, T_d, B = 2, 3, 16, 11, 2
    tb, theta = inputs(S, n_tx, n_rx, M, T_d, B, seed=21)
    cons = orc.qam_constellation(M)
    Xoff = np.zeros((B, T_d, n_tx), np.complex128)
    Xoff[:, :6] = cons[np.random.default_rng(2).integers(0, M, (B, 6, n_tx))]
    for varn in (0.1, 3.0):
        got = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, Xoff=Xoff)
        for b in range(B):
            check_against_oracle(got[b], oracle_llr(orc, tb.Yd[b], tb.PsiD[b], theta[b], M, n_tx, varn, Xoff=Xoff[b]))
    psi = tb.PsiD[0]
    got = gpu_llr(S, tb.Yd, psi, theta, 0.4, n_tx, M, psi_shared=True)
    for b in range(B):
        check_against_oracle(got[b], oracle_llr(orc, tb.Yd[b], psi, theta[b], M, n_tx, 0.4))


def test_mixed_batch_per_trial_varn_and_a_nan_symbol(S, orc):
    n_tx, M, T_d, B = 3, 16, 9, 4
    tb, theta = inputs(S, n_tx, n_tx, M, T_d, B, seed=31)
    varn = np.array([0.1, 2.0, 0.5, 8.0])
    clean = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M)
    for b in range(B):
        check_against_oracle(clean[b], oracle_llr(orc, tb.Yd[b], tb.PsiD[b], theta[b], M, n_tx, varn[b]))
    Yd = tb.Yd.copy()
    Yd[2, 4, 1] = np.nan
    got = gpu_llr(S, Yd, tb.PsiD, theta, varn, n_tx, M)
    assert np.isnan(got[2, 4]).all()
    mask = np.ones(got.shape[:2], bool)
    mask[2, 4] = False
    assert not np.isnan(got[mask]).any()
    assert np.array_equal(got[mask], clean[mask])


def test_chunked_workspace_and_dirty_output_are_bitwise_equal(S):
    import torch

    n_tx, M, T_d, B = 4, 16, 13, 7
    tb, theta = inputs(S, n_tx, n_tx, M, T_d, B, seed=41)
    varn = np.linspace(0.1, 3.0, B)
    one = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M)
    chunked = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, in_flight=3)
    assert np.array_equal(one, chunked)
    dirty = torch.full((B, T_d, n_tx, 4), float("nan"), dtype=torch.float64, device="cuda")
    dirty[::2] = 1e300
    got = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, out=dirty)
    assert np.array_equal(one, got)


def test_hard_bits_follow_kstar_where_it_holds_the_majority(S, orc):
    import torch

    n_tx, n_rx, M, T_d, B, varn = 2, 2, 16, 64, 2, 0.8
    tb, theta = inputs(S, n_tx, n_rx, M, T_d, B, seed=51)
    llr = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M)
    prob = S.Problem(N=tb.PsiD.shape[-1] - 1, n_tx=n_tx, n_rx=n_rx, M=M, T_p=0, T_d=T_d, itera=1, mode="soft")
    ses = S.DeviceSession(prob, B)
    dev = ses.device
    _, _, ks, _ = ses.estep(_t(S, tb.Yd, dev), _t(S, tb.PsiD, dev), _t(S, theta, dev),
                            torch.full((B,), varn, dtype=torch.float64, device=dev))
    ks = ks.cpu().numpy()
    cons = orc.qam_constellation(M)
    table = orc.hypothesis_table(cons, n_tx)
    checked = 0
    for b in range(B):
        d2 = orc.hypothesis_distances(tb.Yd[b], orc.effective_channels(tb.PsiD[b], theta[b], n_tx), table)
        w = np.exp(-(d2 - d2.min(axis=1, keepdims=True)) / varn ** 2)
        post = w[np.arange(T_d), ks[b]] / w.sum(axis=1)
        maj = post > 0.5
        labels = S.qam.bits_of(ks[b], M, n_tx)
        assert np.array_equal((llr[b][maj] < 0), labels[maj].astype(bool))
        checked += maj.sum()
    assert checked > 0


PROFILED = [(4, 16, "k_bit_llr<4, 4>"), (8, 4, "k_bit_llr<8, 2>"), (3, 64, "k_bit_llr<3, 8>"), (1, 4, "k_bit_llr<1, 2>")]

# One bit_llr call per shape under torch.profiler, in a fresh interpreter: a process that already ran other
# profiler sessions and many kernels may deliver no device activity to a later session, which would say nothing
# about the launcher.  The session, its workspace and the inputs are set up, and the kernel launched once, outside
# the trace, so that the trace holds the launches of one call only.
_PROFILE_SCRIPT = r"""
import json, sys
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile
import sbce

out = {}
for n_tx, M in json.loads(sys.argv[1]):
    tb = sbce.signal_model.generate_batch(2, n_tx, n_tx, M, 4, 5, 0.01, 1, seed=61, legacy=False)
    ses = sbce.DeviceSession(sbce.Problem(N=2, n_tx=n_tx, n_rx=n_tx, M=M, T_p=0, T_d=5, itera=1), 1)
    args = [torch.from_numpy(np.ascontiguousarray(a)).to(ses.device) for a in (tb.Yd, tb.PsiD, tb.h, np.full(1, 0.3))]
    llr = ses.bit_llr(*args)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ses.bit_llr(*args, out=llr)
        torch.cuda.synchronize()
    out["%d,%d" % (n_tx, M)] = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
print(json.dumps(out))
"""


@pytest.fixture(scope="module")
def profiled_kernels(S):
    import json
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-c", _PROFILE_SCRIPT, json.dumps([[n, m] for n, m, _ in PROFILED])],
                       cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("n_tx,M,name", PROFILED)
def test_profiler_sees_the_templated_kernel(profiled_kernels, n_tx, M, name):
    """The launcher picks k_bit_llr<n_tx, sqrt M> and no other instantiation."""
    names = profiled_kernels["%d,%d" % (n_tx, M)]
    assert any(re.search(r"(?<![A-Za-z0-9_])" + re.escape(name), n) for n in names), (name, names)
    assert not any("k_bit_llr<" in n and name not in n for n in names), names


def test_accumulate_ber_equals_numpy_count(S):
    import torch

    n_tx, n_rx, M, T_d, B = 3, 3, 16, 21, 5
    prob = S.Problem(N=4, n_tx=n_tx, n_rx=n_rx, M=M, T_p=8, T_d=T_d, itera=2, mode="hard")
    ses = S.DeviceSession(prob, B)
    tb = ses.generate(B, 1.5, seed=7)
    rng = np.random.default_rng(3)
    ks = rng.integers(0, M ** n_tx, (B, T_d)).astype(np.int32)
    acc = torch.zeros(2, dtype=torch.float64, device=ses.device)
    import ctypes as C

    kst = _t(S, ks, ses.device)
    S._lib.check(S._lib.load().sbce_accumulate_ber(C.byref(prob.cfg(B)), kst.data_ptr(), tb["Xd"].data_ptr(), B,
                                                    acc.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    Xd = tb["Xd"].cpu().numpy()
    cons = S.qam.constellation(M)
    idx = np.argmin(np.abs(Xd[..., None] - cons), axis=-1)
    lab = S.qam.bit_labels(M)
    ref = np.count_nonzero(S.qam.bits_of(ks, M, n_tx) != lab[idx])
    assert acc.cpu().numpy().tolist() == [float(ref), float(B * T_d * n_tx * 4)]


def _cfg(S, on_device):
    return S.SweepConfig(N=6, n_tx=2, n_rx=2, M=16, T_p=12, T_d=30, itera=3, monte_iter=6, mode="hard", seed=4,
                         max_batch=4, on_device=on_device, variant="top_tp")


def test_ser_vs_snr_reports_ber_on_the_host_route(S):
    seen = []

    def runner(prob, tb, device):
        res = S.drivers.cuda_runner(prob, tb, device)
        seen.append((tb.idx_d.copy(), np.asarray(res.kstar).copy()))
        return res

    snr = [0.0, 10.0]
    out = S.ser_vs_snr(_cfg(S, False), snr, runner=runner)
    lab = S.qam.bit_labels(16)
    per_point = len(seen) // len(snr)
    for i in range(len(snr)):
        err = tot = 0
        for idx, ks in seen[i * per_point:(i + 1) * per_point]:
            bits = S.qam.bits_of(ks, 16, 2)
            err += np.count_nonzero(bits != lab[idx])
            tot += bits.size
        assert out["ber"][i] == err / tot
    assert out["ber"][0] > 0


def test_ser_vs_snr_reports_ber_on_the_device_route(S):
    import torch

    cfg = _cfg(S, True)
    snr = [0.0, 10.0]
    out = S.ser_vs_snr(cfg, snr)
    lab = S.qam.bit_labels(16)
    cons = S.qam.constellation(16)
    for i, x in enumerate(snr):
        varn = float(S.drivers.snr_to_varn(x))
        prob = S.Problem(N=cfg.N, n_tx=2, n_rx=2, M=16, T_p=cfg.T_p, T_d=cfg.T_d, itera=cfg.itera, mode="hard",
                         psip_shared=True)
        ses = S.DeviceSession(prob, cfg.max_batch)
        err = tot = 0
        for b0 in range(0, cfg.monte_iter, cfg.max_batch):
            nb = min(cfg.max_batch, cfg.monte_iter - b0)
            tb = ses.generate(nb, varn, seed=cfg.seed * 1000003 + i, trial0=b0, pilot_design="top", data_phases="random")
            theta0, _ = ses.ls_start(tb["Yp"], tb["PsiP"], tb["Xp"])
            res = ses.run(tb["Yd"], tb["Yp"], tb["PsiD"], tb["PsiP"], tb["Xp"], tb["varn"], theta0=theta0, h_true=tb["h"])
            torch.cuda.synchronize()
            ks = res.kstar.cpu().numpy()
            idx = np.argmin(np.abs(tb["Xd"].cpu().numpy()[..., None] - cons), axis=-1)
            bits = S.qam.bits_of(ks, 16, 2)
            err += np.count_nonzero(bits != lab[idx])
            tot += bits.size
        assert out["ber"][i] == err / tot
    assert np.isfinite(out["ber"]).all() and np.isfinite(out["ser"]).all()


def test_estimators_bit_llr_equals_the_session(S):
    n_tx, n_rx, M, T_d = 3, 4, 16, 17
    tb, theta = inputs(S, n_tx, n_rx, M, T_d, 1, seed=71)
    Y_d = [tb.Yd[0, t].reshape(-1, 1) for t in range(T_d)]
    PsiTilde_td = tb.PsiD[0].T
    for X_p in (None, [S.qam.constellation(M)[[1, 5, 9]].reshape(-1, 1), S.qam.constellation(M)[[0, 2, 3]].reshape(-1, 1)]):
        got = S.bit_llr(Y_d, PsiTilde_td, theta[0].reshape(-1, 1), M, 0.6, n_tx, X_p=X_p)
        Xoff = None
        if X_p is not None:
            Xoff = np.zeros((1, T_d, n_tx), np.complex128)
            Xoff[0, :2] = np.hstack(X_p).T
        ref = gpu_llr(S, tb.Yd, tb.PsiD, theta, 0.6, n_tx, M, Xoff=Xoff)
        assert got.shape == (T_d, n_tx * 4)
        assert np.array_equal(got, ref[0].reshape(T_d, -1))


def test_bit_llr_rejects_modes_without_a_tree(S):
    for mode in ("pm_beta", "zf", "mmse"):
        prob = S.Problem(N=2, n_tx=2, n_rx=2, M=4, T_p=2, T_d=3, itera=1, mode=mode, partition_r=2)
        ses = S.DeviceSession(prob, 1)
        with pytest.raises(ValueError):
            ses.bit_llr(None, None, None, None)
