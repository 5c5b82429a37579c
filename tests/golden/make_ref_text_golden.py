"""Writes tests/golden/ref_text_golden.npz: what the REFERENCE'S OWN SOURCE TEXT (oracle/_ref/libref_*.so, the
unmodified reference sources compiled against the header shims of oracle/shim) returns on the inputs of
tests/test_oracle_vs_ref.py and tests/test_oracle_lqr.py::test_restatement_is_bitwise_the_reference_text.
Those tests compare the oracle with these stored outputs, so they run in any checkout, with or without the
reference tree.  Inputs that come from numpy float arithmetic (normalised weights, reference trajectories,
random points) are stored too, so the comparison does not depend on how the host's numpy rounds.

    make -C oracle ref REF=<reference checkout> && python tests/golden/make_ref_text_golden.py
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from cpprobotics_b200 import synth  # noqa: E402
from oracle import oracle as O  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref")
f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")


def _load(name):
    return C.CDLL(os.path.join(REF, name))


def ekf(out):
    L = _load("libref_ekf.so")
    L.ref_motion_model.argtypes = [f32p, f32p, f32p]
    L.ref_jacobF.argtypes = [f32p, f32p, f32p]
    L.ref_ekf_estimation.argtypes = [f32p] * 6
    n = 3000
    x, P, z, u = synth.ekf_inputs(n, seed=31)
    _, Q, R = O.ekf_constants()
    mm, jf, xo, Po = (np.zeros((k, n), np.float32) for k in (4, 16, 4, 16))
    for i in range(n):
        xi, ui = np.ascontiguousarray(x[:, i]), np.ascontiguousarray(u[:, i])
        a, ja = np.zeros(4, np.float32), np.zeros(16, np.float32)
        L.ref_motion_model(xi, ui, a)
        L.ref_jacobF(xi, ui, ja)
        xr, Pr = xi.copy(), np.ascontiguousarray(P[:, i]).copy()
        L.ref_ekf_estimation(xr, Pr, np.ascontiguousarray(z[:, i]), ui, Q, R)
        mm[:, i], jf[:, i], xo[:, i], Po[:, i] = a, ja, xr, Pr
    out.update(ekf_motion=mm, ekf_jacobF=jf, ekf_x_out=xo, ekf_P_out=Po)
    # known answer: unit covariance, one step from the origin
    xk, Pk = np.zeros(4, np.float32), np.eye(4, dtype=np.float32).reshape(-1).copy()
    L.ref_ekf_estimation(xk, Pk, np.float32([0.1, 0.0]), np.float32([1.0, 0.1]), Q, R)
    out.update(ekf_ka_x=xk, ekf_ka_P=Pk)


def pf(out):
    L = _load("libref_pf.so")
    L.ref_gauss_likelihood.restype = C.c_float
    L.ref_gauss_likelihood.argtypes = [C.c_float, C.c_float]
    L.ref_pf_np.restype = C.c_int
    L.ref_pf_localization.argtypes = [f32p, f32p, f32p, f32p, f32p, C.c_int, f32p, f32p, C.c_float, C.c_uint, f64p]
    L.ref_resampling.restype = C.c_int
    L.ref_resampling.argtypes = [f32p, f32p, C.c_uint, f64p]
    s = float(np.sqrt(np.float32(0.01)))
    out["pf_gauss"] = np.float32([L.ref_gauss_likelihood(xv, s) for xv in np.linspace(-0.6, 0.6, 101)])
    NP = L.ref_pf_np()
    out["pf_np"] = np.int32(NP)
    px, pw, _ = synth.pf_inputs(NP, seed=9)
    lm = synth.pf_landmarks(4, seed=9)
    c = O.pf_constants()
    pxr = np.ascontiguousarray(px.T.reshape(-1)).copy()
    pwr = pw.copy()
    xe, Pe, draws = np.zeros(4, np.float32), np.zeros(16, np.float32), np.zeros(2 * NP)
    L.ref_pf_localization(pxr, pwr, xe, Pe, np.ascontiguousarray(lm.reshape(-1)), len(lm), c["u"], c["rsim_diag"],
                          float(c["Q"]), 4242, draws)
    out.update(pf_px_out=pxr.reshape(NP, 4), pf_pw_out=pwr, pf_xEst=xe, pf_PEst=Pe, pf_draws=draws)
    # resampling: peaked weights (seeds 1, 2: Neff < NP/2) and flat ones (seed 3)
    for seed, sharp in ((1, True), (2, True), (3, False)):
        px, pw, noise = synth.pf_inputs(100, seed=seed)
        lm = synth.pf_landmarks(4, seed=seed)
        if sharp:
            px, pw = O.pf_predict_weight_batched(px, pw, noise, lm)
            pw = (pw / np.float32(pw.sum())).astype(np.float32)
        pxr, pwr, draws = np.ascontiguousarray(px.T.reshape(-1)).copy(), pw.copy(), np.zeros(100)
        did = L.ref_resampling(pxr, pwr, 99 + seed, draws)
        out.update({f"rs{seed}_px": px, f"rs{seed}_pw": pw, f"rs{seed}_draws": draws, f"rs{seed}_did": np.int32(did),
                    f"rs{seed}_px_out": pxr.reshape(100, 4).T.copy(), f"rs{seed}_pw_out": pwr})


def mpc(out):
    L = _load("libref_mpc.so")
    L.ref_mpc_T.restype = C.c_int
    L.ref_update.argtypes = [f32p, C.c_float, C.c_float]
    L.ref_calc_nearest_index.restype = C.c_int
    L.ref_calc_nearest_index.argtypes = [f32p, f32p, f32p, f32p, C.c_int, C.c_int]
    L.ref_calc_ref_trajectory.argtypes = [f32p, f32p, f32p, f32p, f32p, C.c_int, C.c_float, C.POINTER(C.c_int), f32p]
    L.ref_fg_eval.argtypes = [f32p, f64p, f64p]
    T = L.ref_mpc_T()
    out["mpc_T"] = np.int32(T)
    rng = np.random.default_rng(2)
    st_u, ad_u, out_u = [], [], []
    for _ in range(500):
        st = np.float32([rng.uniform(-50, 50), rng.uniform(-50, 50), rng.uniform(-3, 3), rng.uniform(-6, 15.4)])
        a, d = np.float32(rng.uniform(-1.5, 1.5)), np.float32(rng.uniform(-1, 1))
        r = st.copy()
        L.ref_update(r, a, d)
        st_u.append(st); ad_u.append((a, d)); out_u.append(r)
    out.update(upd_state=np.array(st_u), upd_ad=np.array(ad_u, np.float32), upd_out=np.array(out_u))
    cx, cy, cyaw, sp = synth.mpc_course()
    st, pind = synth.mpc_states(400, seed=3, course=(cx, cy, cyaw, sp))
    near, tind, xref = np.zeros(400, np.int32), np.zeros(400, np.int32), np.zeros((400, 4 * T), np.float32)
    for i in range(400):
        s = np.ascontiguousarray(st[:, i])
        near[i] = L.ref_calc_nearest_index(s, cx, cy, cyaw, len(cx), int(pind[i]))
        ti = C.c_int(int(pind[i]))
        L.ref_calc_ref_trajectory(s, cx, cy, cyaw, sp, len(cx), 1.0, C.byref(ti), xref[i])
        tind[i] = ti.value
    out.update(crt_state=st, crt_pind=pind.astype(np.int32), crt_nearest=near, crt_tind=tind, crt_xref=xref)
    # FG_EVAL at random points and at the oracle's solution of 40 problems
    st, pind = synth.mpc_states(40, seed=4, course=(cx, cy, cyaw, sp))
    xref, _ = synth.mpc_xref_numpy(st, pind, T, course=(cx, cy, cyaw, sp))
    r = O.mpc_solve_batched(st, xref, T)
    rng = np.random.default_rng(0)
    v = rng.normal(size=(40, 4 * T + 2 * (T - 1)))
    fg_v, fg_s = np.zeros((40, 1 + 4 * T)), np.zeros((40, 1 + 4 * T))
    for i in range(40):
        xr = np.ascontiguousarray(xref[:, i])
        L.ref_fg_eval(xr, np.ascontiguousarray(v[i]), fg_v[i])
        L.ref_fg_eval(xr, r["sol"][:, i].astype(np.float64), fg_s[i])
    out.update(nlp_state=st, nlp_xref=xref, nlp_vars=v, nlp_fg_vars=fg_v, nlp_sol=r["sol"], nlp_fg_sol=fg_s)


def lqr(out):
    for nx, nu, name in ((4, 1, "libref_lqr4.so"), (5, 2, "libref_lqr5.so")):
        L = _load(name)
        A, B, Q, R = synth.lqr_inputs(200, nx, seed=12)
        K, X = np.zeros((nu * nx, 200), np.float32), np.zeros((nx * nx, 200), np.float32)
        for i in range(200):
            k, xx = np.zeros(nu * nx, np.float32), np.zeros(nx * nx, np.float32)
            a, b = np.ascontiguousarray(A[:, i]), np.ascontiguousarray(B[:, i])
            if nx == 4:
                L.ref_dlqr4.argtypes = [f32p, f32p, f32p, C.c_float, f32p, f32p]
                L.ref_dlqr4(a, b, Q, float(R[0]), k, xx)
            else:
                L.ref_dlqr5.argtypes = [f32p] * 6
                L.ref_dlqr5(a, b, Q, R, k, xx)
            K[:, i], X[:, i] = k, xx
        out.update({f"lqr{nx}_A": A, f"lqr{nx}_B": B, f"lqr{nx}_Q": Q, f"lqr{nx}_R": R, f"lqr{nx}_K": K,
                    f"lqr{nx}_X": X})


def main():
    out = {}
    for part in (ekf, pf, mpc, lqr):
        part(out)
    path = os.path.join(HERE, "ref_text_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, len(out), "arrays,", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
