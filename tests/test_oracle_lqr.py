"""CPU: solve_DARE()/dlqr() restatement (row f-4) against SciPy's DARE solution, the reference's own text
(oracle/_ref) and its iteration semantics."""
import os

import numpy as np
import pytest
import scipy.linalg as sl

from cpprobotics_b200 import synth
from oracle import oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_text_golden.npz")


@pytest.mark.parametrize("nx,nu", [(4, 1), (5, 2)])
def test_gain_is_close_to_the_exact_dare_solution(nx, nu):
    A, B, Q, R = synth.lqr_inputs(64, nx)
    r = O.dlqr_batched(A, B, Q, R, nx, nu)
    assert r["iters"].min() >= 2 and r["iters"].max() <= 150
    for i in range(0, 64, 5):
        Am = A[:, i].reshape(nx, nx).T.astype(float); Bm = B[:, i].reshape(nu, nx).T.astype(float)
        Xs = sl.solve_discrete_are(Am, Bm, np.eye(nx), np.eye(nu))
        Ks = np.linalg.solve(Bm.T @ Xs @ Bm + np.eye(nu), Bm.T @ Xs @ Am)
        Ko = r["K"][:, i].reshape(nx, nu).T
        # the reference stops when max|dX| < 0.01 (:78,:83): a few 1e-3 from the true fixed point
        assert np.abs(Ko - Ks).max() < 2e-2 * max(1.0, np.abs(Ks).max())


def test_iteration_cap_and_tolerance_semantics():
    A, B, Q, R = synth.lqr_inputs(8, 4)
    r1 = O.dlqr_batched(A, B, Q, R, 4, 1, maxiter=3)
    assert (r1["iters"] == 3).all()
    r0 = O.dlqr_batched(A, B, Q, R, 4, 1, maxiter=0)
    assert (r0["iters"] == 0).all() and np.array_equal(r0["X"], np.repeat(Q[:, None], 8, axis=1))
    tight = O.dlqr_batched(A, B, Q, R, 4, 1, eps=1e-6, maxiter=150)
    loose = O.dlqr_batched(A, B, Q, R, 4, 1)
    assert (tight["iters"] >= loose["iters"]).all()


@pytest.mark.parametrize("nx,nu,lib", [(4, 1, "libref_lqr4.so"), (5, 2, "libref_lqr5.so")])
def test_restatement_is_bitwise_the_reference_text(nx, nu, lib):
    """K and X of the reference's solve_DARE/dlqr (`lib`, the reference source compiled through the shims) on
    200 seeded systems, as stored by tests/golden/make_ref_text_golden.py."""
    G = np.load(GOLDEN)
    A, B, Q, R = (G[f"lqr{nx}_{k}"] for k in "ABQR")
    r = O.dlqr_batched(A, B, Q, R, nx, nu)
    for i in range(200):
        K, X = G[f"lqr{nx}_K"][:, i], G[f"lqr{nx}_X"][:, i]
        assert np.array_equal(K, r["K"][:, i]) and np.array_equal(X, r["X"][:, i])
