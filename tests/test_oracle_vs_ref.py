"""CPU: pins the oracle against the reference's OWN source files, compiled unmodified against header shims
(oracle/shim -> oracle/_ref/libref_*.so; see oracle/shim/README.md for what this does and does not pin).
What those files returned is stored in tests/golden/ref_text_golden.npz (tests/golden/make_ref_text_golden.py
regenerates it where the reference tree is present), so the pin holds in every checkout."""
import os

import numpy as np

import ref_mpc as M
from cpprobotics_b200 import synth
from oracle import oracle as O

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_text_golden.npz"))


def test_ekf_restatement_is_bitwise_the_reference_text():
    n = 3000
    x, P, z, u = synth.ekf_inputs(n, seed=31)
    dt, Q, R = O.ekf_constants()
    lib = O.lib()
    for i in range(n):
        xi, ui = np.ascontiguousarray(x[:, i]), np.ascontiguousarray(u[:, i])
        b = np.zeros(4, np.float32)
        lib.crb_oracle_motion_model(xi, ui, dt, b)
        assert np.array_equal(G["ekf_motion"][:, i], b)
        jb = np.zeros(16, np.float32)
        lib.crb_oracle_jacobF(xi, ui, dt, jb)
        assert np.array_equal(G["ekf_jacobF"][:, i], jb)
        xo, Po = O.ekf_estimation(xi, P[:, i], z[:, i], ui)
        assert np.array_equal(G["ekf_x_out"][:, i], xo) and np.array_equal(G["ekf_P_out"][:, i], Po)


def test_ekf_known_answer_through_the_reference_text():
    x, P = G["ekf_ka_x"], G["ekf_ka_P"]
    np.testing.assert_allclose(x, [0.1, 0.0, 0.010000001, 1.0], atol=1e-8)
    assert abs(P[0] - 0.50495052) < 1e-7 and abs(P[15] - 1.0050495) < 1e-7
    xo, Po = O.ekf_estimation(np.zeros(4, np.float32), np.eye(4, dtype=np.float32).reshape(-1),
                              np.float32([0.1, 0.0]), np.float32([1.0, 0.1]))
    assert np.array_equal(x, xo) and np.array_equal(P, Po)


def test_pf_restatement_is_bitwise_the_reference_text():
    for xv, ref in zip(np.linspace(-0.6, 0.6, 101), G["pf_gauss"]):
        s = float(np.sqrt(np.float32(0.01)))
        assert ref == np.float32(O.gauss_likelihood(xv, s))
    NP = int(G["pf_np"])
    assert NP == 100                                    # src/particle_filter.cpp:21
    px, pw, _ = synth.pf_inputs(NP, seed=9)
    lm = synth.pf_landmarks(4, seed=9)                  # the reference sees <= 4 landmarks (:192-196)
    c = O.pf_constants()
    pxr, pwr, xe, Pe, draws = (G[k] for k in ("pf_px_out", "pf_pw_out", "pf_xEst", "pf_PEst", "pf_draws"))
    lib = O.lib()
    pxo, pwo = np.zeros((NP, 4), np.float32), np.zeros(NP, np.float32)
    for ip in range(NP):
        xx, ww = np.ascontiguousarray(px[:, ip]).copy(), np.array([pw[ip]], np.float32)
        lib.crb_oracle_pf_particle(xx, ww, np.ascontiguousarray(draws[2 * ip:2 * ip + 2]), c["u"], c["rsim_diag"],
                                   np.ascontiguousarray(lm.reshape(-1)), len(lm), float(c["Q"]), c["dt"], c["pi"])
        pxo[ip], pwo[ip] = xx, ww[0]
    assert np.array_equal(pxr, pxo)                     # predict: bit for bit
    s = np.float32(0.0)
    for w in pwo:                                       # pw / pw.sum() with Eigen's float sum (:104)
        s = np.float32(s + w)
    assert np.array_equal(pwr, (pwo / s).astype(np.float32))
    # xEst / PEst (:106-107): the engine accumulates in double (documented), so tolerance here
    pwn, xeo, Peo, _ = O.pf_estimate(np.ascontiguousarray(pxo.T), pwo)
    assert np.abs(xe - xeo).max() < 1e-5 and np.abs(Pe - Peo.T.reshape(-1)).max() < 1e-5


def test_mpc_helpers_are_bitwise_the_reference_text():
    T = int(G["mpc_T"])
    assert T == 6                                       # src/model_predictive_control.cpp:24
    for st, (a, d), r in zip(G["upd_state"], G["upd_ad"], G["upd_out"]):     # update(): :69-81
        assert np.array_equal(r, O.plant_update(st, a, d))
    course = synth.mpc_course()
    cx, cy, cyaw, sp = course
    st, pind = G["crt_state"], G["crt_pind"]
    for i in range(st.shape[1]):
        s = np.ascontiguousarray(st[:, i])
        assert G["crt_nearest"][i] == O.calc_nearest_index(s, cx, cy, int(pind[i]))
        xo, to = O.calc_ref_trajectory(s, cx, cy, cyaw, sp, 1.0, T, int(pind[i]))
        assert G["crt_tind"][i] == to and np.array_equal(G["crt_xref"][i], xo.reshape(-1))


def test_nlp_statement_equals_fg_eval_and_solution_satisfies_it():
    """FG_EVAL::operator() (:199-252) evaluated by the reference's own code: (a) our statement of the cost
    (tests/ref_mpc.nlp_cost) is the same function, (b) the solver's answer is feasible for the reference's
    constraints and its reported cost is the reference's fg[0]."""
    T = 6
    st, xref = G["nlp_state"], G["nlp_xref"]
    r = O.mpc_solve_batched(st, xref, T)
    # the reference evaluated its constraints at this solution when the fixture was made
    np.testing.assert_allclose(r["sol"], G["nlp_sol"], rtol=0, atol=1e-6)
    for i in range(st.shape[1]):
        xr = np.ascontiguousarray(xref[:, i])           # field 4t+k == 4xT column-major
        # (a) random point: cost identity
        v, fg = G["nlp_vars"][i], G["nlp_fg_vars"][i]
        X = v[:4 * T].reshape(4, T); U = v[4 * T:].reshape(2, T - 1)
        p = dict(M.DEFAULTS)
        assert abs(fg[0] - M.nlp_cost(X, U, xr.reshape(T, 4).T.astype(float), p)) <= 1e-9 * abs(fg[0])
        # (b) the oracle's solution
        fg = G["nlp_fg_sol"][i]
        assert abs(fg[0] - r["cost"][i]) <= 2e-5 * max(1.0, fg[0])
        g = fg[1:].reshape(4, T)                        # rows x, y, yaw, v; column 0 = initial state
        assert np.array_equal(g[:, 0].astype(np.float32), st[:, i])
        assert np.abs(g[:, 1:]).max() < 5e-5            # dynamics residuals :242-245 (float32 roll-out)


def test_resampling_restatement_is_bitwise_the_reference_text():
    """resampling() + cumsum() (:111-148) of the reference's own source against oracle.pf_resample in
    reference_mode, on peaked weights (Neff < NP/2 -> resample) and on flat ones (no resample)."""
    for seed, sharp in ((1, True), (2, True), (3, False)):
        px, pw, draws = G[f"rs{seed}_px"], G[f"rs{seed}_pw"], G[f"rs{seed}_draws"]
        pxo, pwo, did_o, neff = O.pf_resample(px, pw, draws, reference_mode=True)
        assert bool(G[f"rs{seed}_did"]) == did_o == sharp
        assert np.array_equal(G[f"rs{seed}_px_out"], pxo) and np.array_equal(G[f"rs{seed}_pw_out"], pwo)
