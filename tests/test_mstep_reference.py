"""CPU tests of the M-step backward-error reference (tests/mstep_reference.py): the measure accepts a
backward-stable FP64 solve at any conditioning, rejects one that is off by 1e-12 relative, and the
Gaussian-integer builder produces Grams that are exact in FP64 at the conditioning it was asked for."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mstep_reference as mr  # noqa: E402


def hermitian_with_cond(rng, L, kappa):
    Q, _ = np.linalg.qr(rng.standard_normal((L, L)) + 1j * rng.standard_normal((L, L)))
    s = np.geomspace(1.0, 1.0 / kappa, L)
    G = (Q * s) @ Q.conj().T
    return 0.5 * (G + G.conj().T), Q[:, 0]


@pytest.mark.parametrize("L", [16, 64])
@pytest.mark.parametrize("kappa", [1.0, 1e4, 1e8, 1e12])
def test_backward_error_separates_fp64_solve_from_a_1e12_perturbation(L, kappa):
    rng = np.random.default_rng(L + int(np.log10(kappa)))
    G, qmax = hermitian_with_cond(rng, L, kappa)
    B = rng.standard_normal((L, 3)) + 1j * rng.standard_normal((L, 3))
    th = np.linalg.solve(G, B)
    assert mr.backward_error(G, B, th) <= mr.tau(L)
    # 1e-12 relative along the dominant eigenvector: the residual grows by ||G|| 1e-12 ||theta||
    pert = th + 1e-12 * np.linalg.norm(th) * np.outer(qmax, np.ones(3)) / np.sqrt(3)
    assert mr.backward_error(G, B, pert) > mr.tau(L)
    ref = mr.refined_solve(G, B)
    assert mr.backward_error(G, B, ref) < 1e-3 * mr.tau(L)
    assert mr.relerr(th, ref) <= 8 * L * mr.U * max(kappa, np.linalg.cond(G))


@pytest.mark.parametrize("cond", [None, 1e4, 1e8, 1e12])
@pytest.mark.parametrize("shape", [(17, 1, 2, 4, 30), (9, 4, 3, 6, 20), (6, 8, 8, 4, 12)])
def test_integer_inputs_give_an_exact_fp64_gram(shape, cond):
    N1, n_tx, n_rx, T_p, T_d = shape
    inp = mr.integer_inputs(np.random.default_rng(N1 * n_tx), 2, N1, n_tx, n_rx, T_p, T_d, cond=cond)
    for b in range(2):
        args = [inp[k][b] for k in ("PsiP", "Yp", "Xp", "PsiD", "Yd", "m", "R")]
        G64, B64 = mr.system(*args, exact_fp64=True)
        Gld, Bld = mr.system(*args)
        assert np.array_equal(G64, Gld) and np.array_equal(B64, Bld)
        assert np.array_equal(Gld, Gld.conj().T)
        c = inp["cond"][b]
        if cond is None:
            assert c < 1e4
        else:
            assert cond / 10 <= c <= cond * 10, (c, cond)
