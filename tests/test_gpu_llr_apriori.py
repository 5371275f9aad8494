"""Extrinsic bit LLRs with a-priori input (sbce_bit_llr_apriori, k_bit_llr<n_tx, sqrt M, true>) on the GPU,
against the numpy oracle of tests/llr_apriori_oracle.py, against sbce_bit_llr with a zero prior, and against
closed forms."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import llr_apriori_oracle as lao  # noqa: E402
from test_gpu_llr import SHAPES, check_against_oracle, inputs  # noqa: E402

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


def _t(a, dev):
    import torch

    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def session(S, B, n_tx, n_rx, M, T_d, N, mode="soft", full_scan=False, superimposed=False, psi_shared=False,
            in_flight=None):
    prob = S.Problem(N=N, n_tx=n_tx, n_rx=n_rx, M=M, T_p=0, T_d=T_d, itera=1, mode=mode, full_scan=full_scan,
                     superimposed=superimposed, psi_shared=psi_shared)
    return S.DeviceSession(prob, in_flight or B)


def gpu_llr(S, Yd, PsiD, theta, varn, n_tx, M, La=None, mode="soft", full_scan=False, Xoff=None, psi_shared=False,
            in_flight=None, out=None, inplace=False):
    """La None: sbce_bit_llr; else sbce_bit_llr_apriori (inplace: the result overwrites a device copy of La)."""
    import torch

    B, T_d, n_rx = Yd.shape
    ses = session(S, B, n_tx, n_rx, M, T_d, PsiD.shape[-1] - 1, mode, full_scan, Xoff is not None, psi_shared,
                  in_flight)
    dev = ses.device
    vn = np.broadcast_to(np.asarray(varn, np.float64), (B,))
    la = _t(La, dev)
    if inplace:
        out = la
    r = ses.bit_llr(_t(Yd, dev), _t(PsiD, dev), _t(theta, dev), _t(vn, dev), Xp=_t(Xoff, dev), out=out, llr_a=la)
    torch.cuda.synchronize()
    if inplace:
        assert r is la
    return r.cpu().numpy()


def random_prior(shape, seed):
    """Both signs, most inside the clamp, some far beyond it."""
    rng = np.random.default_rng(seed)
    La = 6.0 * rng.standard_normal(shape)
    far = rng.random(shape) < 0.1
    La[far] = np.sign(La[far]) * rng.uniform(33.0, 80.0, far.sum())
    return La


def oracle_ext(orc, Yd, PsiD, theta, M, n_tx, varn, La, Xoff=None):
    """Unclamped oracle values of one trial; the split enumeration for the 2^24-leaf trees."""
    cons = orc.qam_constellation(M)
    f = lao.bit_llr_apriori_split if M ** n_tx > (1 << 20) else lao.bit_llr_apriori
    return f(Yd, PsiD, theta, cons, n_tx, varn, La, Xoff=Xoff, clamp=False)


@pytest.mark.parametrize("n_tx,M", SHAPES)
@pytest.mark.parametrize("regime", ["peaked", "flat"])
def test_every_shape_against_the_oracle(S, orc, n_tx, M, regime):
    big = M ** n_tx > (1 << 16)
    T_d = 3 if big else 7
    B = 1 if big else 2
    tb, theta = inputs(S, n_tx, n_tx, M, T_d, B, seed=100 * n_tx + M)
    varn = 0.1 if regime == "peaked" else {4: 3.0, 16: 6.0, 64: 10.0}[M]
    La = random_prior((B, T_d, n_tx, int(np.log2(M))), seed=7 * n_tx + M)
    got = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La)
    assert got.shape == La.shape
    for b in range(B):
        check_against_oracle(got[b], oracle_ext(orc, tb.Yd[b], tb.PsiD[b], theta[b], M, n_tx, varn, La[b]))


@pytest.mark.parametrize("full_scan", [False, True])
def test_zero_prior_is_bitwise_sbce_bit_llr(S, full_scan):
    for n_tx, M, varn in [(1, 4, 0.7), (2, 64, 0.5), (3, 16, 2.0), (4, 16, 0.3), (5, 16, 0.2), (8, 4, 0.4)]:
        tb, theta = inputs(S, n_tx, n_tx, M, 5, 2, seed=13 + n_tx)
        plain = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, full_scan=full_scan)
        zero = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=np.zeros(plain.shape), full_scan=full_scan)
        assert np.array_equal(plain, zero), (n_tx, M)


@pytest.mark.parametrize("n_rx", [1, 3])
def test_single_stream_qpsk_extrinsic_is_the_channel_llr(S, orc, n_rx):
    """n_tx = 1, QPSK: the I and Q bits separate, so whatever the prior the extrinsic LLRs are the no-prior closed
    form llr_I = -4 Re(h^H y) / varn^2, llr_Q = -4 Im(h^H y) / varn^2 (clamped)."""
    tb, theta = inputs(S, 1, n_rx, 4, 33, 2, seed=5)
    La = random_prior((2, 33, 1, 2), seed=8)
    for varn in (1.3, 0.3):
        got = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, 1, 4, La=La)
        for b in range(2):
            h = orc.effective_channels(tb.PsiD[b], theta[b], 1)[:, :, 0]          # (T_d, n_rx)
            z = np.einsum("tr,tr->t", h.conj(), tb.Yd[b])
            ref = np.stack([-4 * z.real, -4 * z.imag], axis=1) / varn ** 2
            np.testing.assert_allclose(got[b, :, 0], np.clip(ref, -CLAMP, CLAMP), rtol=0, atol=1e-9)


@pytest.mark.parametrize("n_tx", [2, 3, 4])
def test_genie_priors_cancel_the_interference(S, orc, n_tx):
    """QPSK, priors +-32 from the true bits: every bit's extrinsic LLR is the single-stream closed form on
    z_j = y - sum_{s != j} h_s x_s, up to the prior's leakage.  Side v of bit i of stream j is its closed-form part
    (the other streams at their true symbols) times 1 + eps_v, where eps_v is the weight of every other choice of
    the other streams, each damped by e^-32 per bit it gets wrong, relative to that part.  So
    |llr - closed form| <= max_v ln(1 + eps_v), computed here from the exact distances.  varn = 4 keeps the
    likelihood ratios small enough for the leakage to stay below 1e-6."""
    M, n_rx, T_d, B, varn = 4, {2: 3, 3: 4, 4: 6}[n_tx], 16, 2, 4.0
    tb, theta = inputs(S, n_tx, n_rx, M, T_d, B, seed=17 + n_tx)
    cons = orc.qam_constellation(M)
    lab = S.qam.bit_labels(M)
    idx = np.argmin(np.abs(tb.Xd[..., None] - cons), axis=-1)                       # (B, T_d, n_tx)
    La = np.where(lab[idx] == 1, -32.0, 32.0)
    got = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La)
    K = M ** n_tx
    table = orc.hypothesis_table(cons, n_tx)                                          # (K, n_tx)
    bits = S.qam.bits_of(np.arange(K), M, n_tx)                                       # (K, n_tx, 2)
    worst = 0.0
    for b in range(B):
        H = orc.effective_channels(tb.PsiD[b], theta[b], n_tx)                        # (T_d, n_rx, n_tx)
        for t in range(T_d):
            x = cons[idx[b, t]]
            d2 = (np.abs(tb.Yd[b, t][None, :] - table @ H[t].T) ** 2).sum(axis=1)       # (K,)
            for j in range(n_tx):
                others = [s for s in range(n_tx) if s != j]
                zz = H[t][:, j].conj() @ (tb.Yd[b, t] - H[t][:, others] @ x[others])
                ref = np.clip(np.array([-4 * zz.real, -4 * zz.imag]) / varn ** 2, -CLAMP, CLAMP)
                miss = bits != lab[idx[b, t]]                                        # (K, n_tx, 2) against the prior
                wrong = miss[:, others].sum(axis=(1, 2))                              # the other streams' bits
                for i in range(2):
                    # log-weights with the prior of every bit but the one asked for (which cancels in the extrinsic)
                    a = -d2 / varn ** 2 - 32.0 * (wrong + miss[:, j, 1 - i])
                    tol = 0.0
                    for v in (0, 1):
                        side = bits[:, j, i] == v
                        eps = np.exp(np.logaddexp.reduce(a[side & (wrong > 0)]) -
                                     np.logaddexp.reduce(a[side & (wrong == 0)]))
                        tol = max(tol, np.log1p(eps))
                    worst = max(worst, tol)
                    assert abs(got[b, t, j, i] - ref[i]) <= tol + 1e-9, (b, t, j, i, got[b, t, j, i], ref[i], tol)
    assert worst < 1e-6   # the leakage bound is small enough for the comparison to mean something


@pytest.mark.parametrize("n_tx,M,varn", [(4, 16, 0.1), (4, 16, 2.0), (8, 4, 0.3), (2, 64, 0.5), (5, 16, 0.2)])
def test_pruned_equals_full_scan_and_modes_agree(S, n_tx, M, varn):
    tb, theta = inputs(S, n_tx, n_tx, M, 9, 2, seed=9 + n_tx)
    La = random_prior((2, 9, n_tx, int(np.log2(M))), seed=n_tx)
    a = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La)
    f = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La, full_scan=True)
    np.testing.assert_allclose(a, f, rtol=0, atol=1e-12)
    h = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La, mode="hard")
    assert np.array_equal(a, h), "soft and hard modes give the same LLRs"


def test_superimposed_offsets_and_shared_phases(S, orc):
    n_tx, n_rx, M, T_d, B = 2, 3, 16, 11, 2
    tb, theta = inputs(S, n_tx, n_rx, M, T_d, B, seed=21)
    cons = orc.qam_constellation(M)
    Xoff = np.zeros((B, T_d, n_tx), np.complex128)
    Xoff[:, :6] = cons[np.random.default_rng(2).integers(0, M, (B, 6, n_tx))]
    La = random_prior((B, T_d, n_tx, 4), seed=22)
    for varn in (0.1, 3.0):
        got = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La, Xoff=Xoff)
        for b in range(B):
            check_against_oracle(got[b], oracle_ext(orc, tb.Yd[b], tb.PsiD[b], theta[b], M, n_tx, varn, La[b],
                                                    Xoff=Xoff[b]))
    psi = tb.PsiD[0]
    got = gpu_llr(S, tb.Yd, psi, theta, 0.4, n_tx, M, La=La, psi_shared=True)
    for b in range(B):
        check_against_oracle(got[b], oracle_ext(orc, tb.Yd[b], psi, theta[b], M, n_tx, 0.4, La[b]))


def test_mixed_batch_nan_prior_and_infinite_prior(S, orc):
    n_tx, M, T_d, B = 3, 16, 9, 4
    tb, theta = inputs(S, n_tx, n_tx, M, T_d, B, seed=31)
    varn = np.array([0.1, 2.0, 0.5, 8.0])
    La = random_prior((B, T_d, n_tx, 4), seed=32)
    clean = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La)
    for b in range(B):
        check_against_oracle(clean[b], oracle_ext(orc, tb.Yd[b], tb.PsiD[b], theta[b], M, n_tx, varn[b], La[b]))
    bad = La.copy()
    bad[2, 4, 1, 3] = np.nan
    got = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=bad)
    assert np.isnan(got[2, 4]).all()
    mask = np.ones(got.shape[:2], bool)
    mask[2, 4] = False
    assert not np.isnan(got[mask]).any()
    assert np.array_equal(got[mask], clean[mask])
    # an infinite prior reads as +-32
    inf, c32 = La.copy(), La.copy()
    inf[1, 2, 0, 1], c32[1, 2, 0, 1] = -np.inf, -32.0
    inf[3, 5, 2, 0], c32[3, 5, 2, 0] = np.inf, 32.0
    assert np.array_equal(gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=inf),
                          gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=c32))


def test_chunked_workspace_dirty_output_and_in_place_are_bitwise_equal(S):
    import torch

    n_tx, M, T_d, B = 4, 16, 13, 7
    tb, theta = inputs(S, n_tx, n_tx, M, T_d, B, seed=41)
    varn = np.linspace(0.1, 3.0, B)
    La = random_prior((B, T_d, n_tx, 4), seed=42)
    one = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La)
    chunked = gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La, in_flight=3)
    assert np.array_equal(one, chunked)
    dirty = torch.full((B, T_d, n_tx, 4), float("nan"), dtype=torch.float64, device="cuda")
    dirty[::2] = 1e300
    assert np.array_equal(one, gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La, out=dirty))
    assert np.array_equal(one, gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La, inplace=True))
    assert np.array_equal(one, gpu_llr(S, tb.Yd, tb.PsiD, theta, varn, n_tx, M, La=La, inplace=True, in_flight=3))


def test_estimators_bit_llr_with_prior_equals_the_session(S):
    n_tx, n_rx, M, T_d = 3, 4, 16, 17
    tb, theta = inputs(S, n_tx, n_rx, M, T_d, 1, seed=71)
    Y_d = [tb.Yd[0, t].reshape(-1, 1) for t in range(T_d)]
    PsiTilde_td = tb.PsiD[0].T
    La = random_prior((1, T_d, n_tx, 4), seed=72)
    got = S.bit_llr(Y_d, PsiTilde_td, theta[0].reshape(-1, 1), M, 0.6, n_tx, llr_a=La[0].reshape(T_d, -1))
    ref = gpu_llr(S, tb.Yd, tb.PsiD, theta, 0.6, n_tx, M, La=La)
    assert got.shape == (T_d, n_tx * 4)
    assert np.array_equal(got, ref[0].reshape(T_d, -1))
    with pytest.raises(ValueError):
        S.bit_llr(Y_d, PsiTilde_td, theta[0].reshape(-1, 1), M, 0.6, n_tx, llr_a=np.zeros((T_d, 3)))
