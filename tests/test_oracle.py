"""CPU: pin the oracle (oracle/oracle.py + oracle/psoap_oracle.c) against the golden vectors produced by the
unmodified reference (tests/golden/make_golden.py)."""
import numpy as np

from conftest import rel_close

N_ORB = {"SB1": 6, "SB2": 7, "ST1": 11, "ST2": 12, "ST3": 13}


def test_fill_bit_exact(golden, oracle):
    g = golden["fills"]
    lw, lwp, amp, l = g["lwl"], g["lwl_predict"], g["amp"], g["l"]
    N, M = lw.shape[1], len(lwp)
    m = np.empty((N, N)); oracle.fill_V11_f(m, lw[0], amp[0], l[0])
    assert np.array_equal(m, g["V11_f"])
    m = np.empty((N, N)); oracle.fill_V11_f_g(m, lw[0], lw[1], amp[0], l[0], amp[1], l[1])
    assert np.array_equal(m, g["V11_f_g"])
    m = np.empty((N, N)); oracle.fill_V11_f_g_h(m, lw[0], lw[1], lw[2], amp[0], l[0], amp[1], l[1], amp[2], l[2])
    assert np.array_equal(m, g["V11_f_g_h"])
    m = np.empty((N, M)); oracle.fill_V12_f(m, lw[0], lwp, amp[0], l[0])
    assert np.array_equal(m, g["V12_f"])
    m = np.empty((33, 33)); oracle.fill_V11_f(m, g["far_lwl"], 0.5, 5.0)
    assert np.array_equal(m, g["far_V11_f"])
    assert (g["far_V11_f"] == 0).any()  # the fixture reaches exp underflow


def test_orbits(golden, oracle):
    g = golden["orbits"]
    dates = g["dates"]
    keys = [k[:-2] for k in g.files if k.endswith("_p")]
    assert len(keys) == 9
    for k in keys:
        model = k.split("_")[0]
        v = oracle.get_velocities(model, g[k + "_p"], dates)
        assert v.shape == g[k + "_v"].shape
        assert np.array_equal(v, g[k + "_v"]), k  # same fsolve, same arithmetic


def test_replicate_wls_and_lnlike(golden, oracle):
    g = golden["lnlike"]
    for k in range(4):
        pre = f"case{k}_"
        model = str(g[pre + "model"])
        p = g[pre + "p"]
        vel = oracle.get_velocities(model, p[:N_ORB[model]], g[pre + "date1D"])
        assert np.array_equal(vel, g[pre + "vel"])
        lwls = oracle.replicate_wls(g[pre + "lwl"], vel, g[pre + "mask"])
        assert np.array_equal(lwls, g[pre + "lwls"])
        # the C replicate with the explicit epoch index
        out = np.empty_like(lwls)
        ep = np.ascontiguousarray(g[pre + "epoch"], dtype=np.int32)
        import ctypes
        oracle.clib().oracle_replicate_wls(oracle._p(out), oracle._p(np.ascontiguousarray(g[pre + "lwl"])),
                                           ep.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), len(ep),
                                           oracle._p(np.ascontiguousarray(vel)), vel.shape[0], vel.shape[1])
        assert np.array_equal(out, lwls)
        N = lwls.shape[1]
        fl, sigma, pg = g[pre + "fl"], g[pre + "sigma"], p[N_ORB[model]:]
        V11 = np.empty((N, N))
        ln = oracle.lnlike[model](V11, *lwls, fl, sigma, *pg)
        assert rel_close(ln, g[pre + "lnlike"], 1e-13)
        ln_c = oracle.lnlike_c(V11, list(lwls), fl, sigma, pg[0::2], pg[1::2])
        assert rel_close(ln_c, g[pre + "lnlike"], 1e-12)
        ln = oracle.lnlike[model](V11, *lwls, fl, sigma, *pg, mu_GP=0.9)
        assert rel_close(ln, g[pre + "lnlike_mu09"], 1e-13)
        assert g[pre + "lnlike_negamp"] == -np.inf and g[pre + "lnlike_nonpd"] == -np.inf
        pn = pg.copy(); pn[0] = -0.1
        assert oracle.lnlike[model](V11, *lwls, fl, sigma, *pn) == -np.inf
        lw2 = lwls.copy(); lw2[:, 1] = lw2[:, 0]
        assert oracle.lnlike[model](V11, *lw2, fl, np.zeros_like(sigma), *pg) == -np.inf
        assert oracle.lnlike_c(V11, list(lw2), fl, np.zeros_like(sigma), pg[0::2], pg[1::2]) == -np.inf
        # farm composition (sample_parallel.Worker.lnprob)
        ch = dict(lwl=g[pre + "lwl"], fl=fl, sigma=sigma, mask=g[pre + "mask"], date1D=g[pre + "date1D"])
        assert rel_close(oracle.chunk_lnprob(model, p, ch), g[pre + "lnlike"], 1e-13)


def test_predict(golden, oracle):
    g = golden["predict"]
    lwls, fl, sigma, lwp, amp, l = g["lwls"], g["fl"], g["sigma"], g["lwl_predict"], g["amp"], g["l"]
    mu, Sig = oracle.predict_f_g(lwls[0], lwls[1], fl, sigma, lwp[0], lwp[1], 0.7, amp[0], l[0], 0.3, amp[1], l[1])
    assert rel_close(mu, g["fg_mu"], 1e-12) and rel_close(Sig, g["fg_Sigma"], 1e-11, 1e-16)
    mu = oracle.predict_f_g(lwls[0], lwls[1], fl, sigma, lwp[0], lwp[1], 0.7, amp[0], l[0], 0.3, amp[1], l[1],
                            get_Sigma=False)
    assert rel_close(mu, g["fg_mu_only"], 1e-12)
    mu, Sig = oracle.predict_f_g_sum(lwls[0], lwls[1], fl, sigma, lwp[0], lwp[1], 1.0, amp[0], l[0], amp[1], l[1])
    assert rel_close(mu, g["fgsum_mu"], 1e-12) and rel_close(Sig, g["fgsum_Sigma"], 1e-11, 1e-16)
    mu, Sig = oracle.predict_f_g_h(lwls[0], lwls[1], lwls[2], fl, sigma, lwp[0], lwp[1], lwp[2], 0.5, 0.3, 0.2,
                                   amp[0], l[0], amp[1], l[1], amp[2], l[2])
    assert rel_close(mu, g["fgh_mu"], 1e-12) and rel_close(Sig, g["fgh_Sigma"], 1e-11, 1e-16)
    mu, Sig = oracle.predict_f_g_h_sum(lwls[0], lwls[1], lwls[2], fl, sigma, lwls[0], lwls[1], lwls[2], 1.0,
                                       amp[0], l[0], amp[1], l[1], amp[2], l[2])
    assert rel_close(mu, g["fghsum_mu"], 1e-12) and rel_close(Sig, g["fghsum_Sigma"], 1e-11, 1e-16)
    assert str(g["predict_f_raises"]) == "NameError"  # reference defect (covariance.py:38), documented


def test_calibration_and_gp_fit(golden, oracle):
    g = golden["calibration"]
    args = (float(g["lwl0"]), float(g["lwl1"]), g["lwl_cal"], g["fl_cal"], g["sigma_cal"], g["lwl_fixed"], g["fl_fixed"],
            g["sigma_fixed"], float(g["amp"]), float(g["l"]))
    for order in (1, 2):
        fl_cor, X = oracle.optimize_calibration_static(*args, order=order, mu_GP=1.0)
        assert rel_close(X, g[f"static_o{order}_X"], 1e-9, 1e-12) and rel_close(fl_cor, g[f"static_o{order}_fl"], 1e-10)
    n_cal, n_fix = len(g["lwl_cal"]), len(g["lwl_fixed"])
    A = np.empty((n_cal, n_cal)); oracle.fill_V11_f(A, g["lwl_cal"], float(g["amp"]), float(g["l"]))
    A[np.diag_indices_from(A)] += g["sigma_cal"] ** 2
    B = np.empty((n_fix, n_fix)); oracle.fill_V11_f(B, g["lwl_fixed"], float(g["amp"]), float(g["l"]))
    B[np.diag_indices_from(B)] += g["sigma_fixed"] ** 2
    C = np.empty((n_cal, n_fix)); oracle.fill_V12_f(C, g["lwl_cal"], g["lwl_fixed"], float(g["amp"]), float(g["l"]))
    fl_cor, X = oracle.optimize_calibration(float(g["lwl0"]), float(g["lwl1"]), g["lwl_cal"], g["fl_cal"],
                                            g["fl_fixed"], A, B, C, order=1, mu_GP=1.0)
    assert rel_close(X, g["general_X"], 1e-9, 1e-12) and rel_close(fl_cor, g["general_fl"], 1e-10)
