"""The oracle (oracle/) against the golden vectors produced by the unmodified reference
(tests/golden/make_golden.py)."""
import numpy as np
import pytest

from oracle import kf as okf, ukf as oukf, resample as ors


def close(a, b, rtol=1e-9, atol=1e-11):
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


# ------------------------------------------------------------------ KF
def test_kf_c1_batch_filter(golden):
    g = golden("kf_c1")
    zs = list(g["zs"])
    out = okf.kf_batch_filter_single(g["x"], g["P"], zs, g["F"], g["Q"], g["H"], g["R"])
    for got, key in zip(out, ["means", "covs", "means_p", "covs_p"]):
        close(got, g[key], rtol=1e-12, atol=1e-13)
    # known answers (SURVEY §8c)
    x, P = okf.kf_predict_single(np.zeros(4), 10 * np.eye(4), g["F"], g["Q"])
    x, P, y, K, S, SI = okf.kf_update_single(x, P, np.array([1., 2.]), g["H"], g["R"])
    close(x, g["one_x"], 1e-13); close(P, g["one_P"], 1e-13)
    close(S, g["one_S"], 1e-13); close(K, g["one_K"], 1e-13)
    assert abs(x[0] - 0.9876558449574127) < 1e-14
    ll = okf.log_likelihood_bank(y[None], S[None])[0]
    assert abs(ll - float(g["one_loglik"])) < 1e-12
    assert abs(ll - (-4.969596859557728)) < 1e-12


@pytest.mark.parametrize("name", ["kf_bank_4_2", "kf_bank_9_3", "kf_bank_1_1", "kf_bank_2_1",
                                  "kf_bank_3_2", "kf_bank_6_3", "kf_bank_5_5"])
def test_kf_bank_vs_reference(golden, name):
    g = golden(name)
    x, P = g["x"], g["P"]
    alpha_sq = float(g["alpha"]) ** 2
    for t in range(g["zs"].shape[0]):
        if "B" in g:
            xp, Pp = okf.kf_predict_bank(x, P, g["F"], g["Q"], alpha_sq, g["B"], g["us"][t])
            o = okf.kf_update_bank(xp, Pp, g["zs"][t], g["H"], g["R"], g["valid"][t])
            o["x_prior"], o["P_prior"] = xp, Pp
        else:
            o = okf.kf_step_bank(x, P, g["zs"][t], g["F"], g["H"], g["Q"], g["R"], alpha_sq, g["valid"][t])
        x, P = o["x"], o["P"]
        v = g["valid"][t]
        close(x, g["ref_x"][t]); close(P, g["ref_P"][t])
        close(o["x_prior"], g["ref_x_prior"][t]); close(o["P_prior"], g["ref_P_prior"][t])
        for k in ["K", "S", "SI"]:
            close(o[k][v], g["ref_" + k][t][v])
        close(o["y"], g["ref_y"][t])
        ll = okf.log_likelihood_bank(o["y"], o["S"])
        close(ll[v], g["ref_loglik"][t][v], rtol=1e-9, atol=1e-9)


def test_kf_c_port_matches(golden):
    import ctypes
    from oracle import cbuild
    lib = cbuild.load()
    for name in ["kf_bank_4_2", "kf_bank_9_3", "kf_bank_3_2"]:
        g = golden(name)
        if "B" in g:
            continue
        x = g["x"].copy(); P = g["P"].copy()
        N, n = x.shape; m = g["H"].shape[-2]
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        for t in range(g["zs"].shape[0]):
            z = np.ascontiguousarray(g["zs"][t]); v = np.ascontiguousarray(g["valid"][t].astype(np.uint8))
            bad = lib.oracle_kf_step_f64(ctypes.c_int64(N), n, m, p(x), p(P),
                                         p(g["F"]), ctypes.c_int64(n * n), p(g["H"]), ctypes.c_int64(m * n),
                                         p(g["Q"]), ctypes.c_int64(n * n), p(g["R"]), ctypes.c_int64(m * m),
                                         p(z), p(v), ctypes.c_double(float(g["alpha"]) ** 2), 1)
            assert bad == 0
            close(x, g["ref_x"][t]); close(P, g["ref_P"][t])


# ------------------------------------------------------------------ UKF
def test_merwe_sigma_points(golden):
    g = golden("ukf_sigma")
    a, b, k = float(g["alpha"]), float(g["beta"]), float(g["kappa"])
    Wm, Wc = oukf.merwe_weights(6, a, b, k)
    close(Wm, g["Wm"], 1e-14); close(Wc, g["Wc"], 1e-14)
    Wm4, Wc4 = oukf.merwe_weights(4, .5, 2, 0)
    close(Wm4, [-3] + [.5] * 8); close(Wc4, [-.25] + [.5] * 8)
    close(oukf.merwe_sigma_points(g["x"], g["P"], a, b, k), g["sigmas"], 1e-13)


@pytest.mark.parametrize("name,fxm,hxm", [("ukf_bank_rae", oukf.FX_CONST_VEL, oukf.HX_RANGE_AZ_EL),
                                         ("ukf_bank_lin", oukf.FX_LINEAR, oukf.HX_LINEAR)])
def test_ukf_bank_vs_reference(golden, name, fxm, hxm):
    g = golden(name)
    x, P = g["x"], g["P"]
    a, b, k, dt = float(g["alpha"]), float(g["beta"]), float(g["kappa"]), float(g["dt"])
    for t in range(g["zs"].shape[0]):
        o = oukf.ukf_step_bank(x, P, g["zs"][t], g["Q"], g["R"], dt, a, b, k, fxm, hxm,
                               F=g["F"], H=g["H"], valid=g["valid"][t])
        x, P = o["x"], o["P"]
        close(x, g["ref_x"][t], rtol=1e-9, atol=1e-9); close(P, g["ref_P"][t], rtol=1e-8, atol=1e-9)
        close(o["x_prior"], g["ref_x_prior"][t]); close(o["P_prior"], g["ref_P_prior"][t], 1e-8, 1e-9)


@pytest.mark.parametrize("name,fxm,hxm", [("ukf_julier_rae", oukf.FX_CONST_VEL, oukf.HX_RANGE_AZ_EL),
                                         ("ukf_julier_lin", oukf.FX_LINEAR, oukf.HX_LINEAR)])
def test_ukf_julier_bank_vs_reference(golden, name, fxm, hxm):
    """JulierSigmaPoints(kappa) (sigma_points.py:211-383) == the Merwe parameterisation alpha=1, beta=0."""
    g = golden(name)
    x, P = g["x"], g["P"]
    k, dt = float(g["kappa"]), float(g["dt"])
    for t in range(g["zs"].shape[0]):
        o = oukf.ukf_step_bank(x, P, g["zs"][t], g["Q"], g["R"], dt, 1.0, 0.0, k, fxm, hxm,
                               F=g["F"], H=g["H"], valid=g["valid"][t])
        x, P = o["x"], o["P"]
        close(x, g["ref_x"][t], rtol=1e-9, atol=1e-9); close(P, g["ref_P"][t], rtol=1e-8, atol=1e-9)
        close(o["x_prior"], g["ref_x_prior"][t]); close(o["P_prior"], g["ref_P_prior"][t], 1e-8, 1e-9)


def test_julier_weights_and_sigma_points(golden):
    from filterpy_b200.kalman import JulierSigmaPoints
    g = golden("julier_sigma")
    for i in range(4):
        k = float(g["kappa%d" % i])
        pts = JulierSigmaPoints(4, k)
        assert pts.num_sigmas() == 9 and (pts.alpha, pts.beta, pts.kappa) == (1.0, 0.0, k)
        close(pts.Wm, g["Wm%d" % i], 1e-15); close(pts.Wc, g["Wc%d" % i], 1e-15)
        Wm, Wc = oukf.merwe_weights(4, 1.0, 0.0, k)
        close(Wm, g["Wm%d" % i], 1e-14); close(Wc, g["Wc%d" % i], 1e-14)
        close(oukf.merwe_sigma_points(g["x"], g["P"], 1.0, 0.0, k), g["sigmas%d" % i], 1e-13)
    with pytest.raises(NotImplementedError):
        JulierSigmaPoints(4, 0., sqrt_method=np.linalg.cholesky)


@pytest.mark.parametrize("name,linear", [("ukf_user_ct_rb", False), ("ukf_user_ct_lin", True)])
def test_ukf_user_models_oracle_vs_reference(golden, name, linear):
    """fx / hx outside the built-in set (coordinated turn with a per-filter rate, offset range / bearing):
    the oracle's single-filter path with the Python callables of workloads.py against the reference."""
    from filterpy_b200.common import workloads as wl
    g = golden(name)
    a, b, k, dt = float(g["alpha"]), float(g["beta"]), float(g["kappa"]), float(g["dt"])
    H, sensor = g["H"], g["sensor"]
    hx = (lambda s: H @ s) if linear else (lambda s: wl.offset_rb_hx(s, sensor[0], sensor[1]))
    for f in range(0, g["x"].shape[0], 5):
        x, P = g["x"][f], g["P"][f]
        om = float(g["omega"][f])
        for t in range(g["zs"].shape[0]):
            x, P, sf = oukf.ukf_predict_single(x, P, g["Q"][f], lambda s, dt: wl.ct_fx(s, dt, om), dt, a, b, k)
            close(x, g["ref_x_prior"][t, f], 1e-9, 1e-9); close(P, g["ref_P_prior"][t, f], 1e-8, 1e-9)
            if g["valid"][t, f]:
                x, P = oukf.ukf_update_single(x, P, sf, g["zs"][t, f], g["R"][f], hx, a, b, k)[:2]
            close(x, g["ref_x"][t, f], 1e-9, 1e-9); close(P, g["ref_P"][t, f], 1e-8, 1e-9)


def test_ukf_single_matches_bank(golden):
    g = golden("ukf_bank_lin")
    a, b, k, dt = float(g["alpha"]), float(g["beta"]), float(g["kappa"]), float(g["dt"])
    F, H = g["F"], g["H"]
    x, P = g["x"][0], g["P"][0]
    for t in range(3):
        x, P, sf = oukf.ukf_predict_single(x, P, g["Q"][0], lambda s, dt: F @ s, dt, a, b, k)
        x, P = oukf.ukf_update_single(x, P, sf, g["zs"][t, 0], g["R"][0], lambda s: H @ s, a, b, k)[:2]
        close(x, g["ref_x"][t, 0], 1e-9, 1e-9); close(P, g["ref_P"][t, 0], 1e-8, 1e-9)


# ------------------------------------------------------------------ resampling
def test_resample_golden(golden):
    g = golden("resample")
    assert list(g["known_sys"]) == [1, 2, 3, 3]
    assert list(ors.systematic_resample_loop([.1, .2, .3, .4], 0.5)) == [1, 2, 3, 3]
    assert list(ors.stratified_resample_loop([.1, .2, .3, .4], np.full(4, .5))) == list(g["known_str"])
    for (i, N, ok, ok_s, seed) in g["meta"]:
        w, u, U = g["w%d" % i], float(g["u%d" % i]), g["U%d" % i]
        for fn in (ors.systematic_resample_loop, ors.systematic_resample_vec, ors.systematic_resample_c):
            if ok:
                got = fn(w, u)
                assert got.dtype == np.int32
                assert np.array_equal(got, g["sys%d" % i]), (fn.__name__, i, N)
            else:
                with pytest.raises(IndexError):
                    fn(w, u)
        for fn in (ors.stratified_resample_loop, ors.stratified_resample_vec, ors.stratified_resample_c):
            if ok_s:
                assert np.array_equal(fn(w, U), g["str%d" % i]), (fn.__name__, i, N)
            else:
                with pytest.raises(IndexError):
                    fn(w, U)


def test_live_reference_resample_and_kf(golden):
    """systematic_resample(w) after np.random.seed(123), and five reference KalmanFilter objects over
    two steps (tests/golden/make_golden.py:gen_spot_checks)."""
    g = golden("spot_checks")
    w, u, ref = g["sys_w"], float(g["sys_u"]), g["sys_idx"]
    assert np.array_equal(ors.systematic_resample_vec(w, u), ref)
    assert np.array_equal(ors.systematic_resample_c(w, u), ref)
    o = None; x, P = g["kf_x"], g["kf_P"]
    for t in range(2):
        o = okf.kf_step_bank(x, P, g["kf_zs"][t], g["kf_F"], g["kf_H"], g["kf_Q"], g["kf_R"]); x, P = o["x"], o["P"]
    for f in range(5):
        close(x[f], g["kf_ref_x"][f], 1e-12); close(P[f], g["kf_ref_P"][f], 1e-12)


# ------------------------------------------------------------------ §8f rows: multinomial resample, RTS smoother
def test_multinomial_oracle_vs_reference_vectors(golden):
    g = golden("resample_multinomial")
    for (i, N, seed) in g["meta"]:
        w, U, ref = g["w%d" % i], g["U%d" % i], g["idx%d" % i]
        assert ref.dtype == np.int64
        assert np.array_equal(ors.multinomial_resample_vec(w, U), ref)
        assert np.array_equal(ors.multinomial_resample_c(w, U), ref)
        if N <= 1000:
            assert np.array_equal(ors.multinomial_resample_loop(w, U), ref)


def test_residual_oracle_vs_reference_vectors(golden):
    """resampling.py:27-76: the restatement (reference-order sums + NumPy's bracket-carrying bisection,
    oracle/resample.py:binsearch_left) reproduces the reference on every golden case; most of these
    cumulative sums are NOT monotone and on at least one the carried bracket decides the answer."""
    g = golden("resample_residual")
    nonmono = dep = 0
    for (i, N, seed, k) in g["meta"]:
        w, U, ref = g["w%d" % i], g["U%d" % i], g["idx%d" % i]
        assert ref.dtype == np.int32 and len(U) == N - k
        with np.errstate(all="ignore"):
            assert np.array_equal(ors.residual_resample_vec(w, U), ref)
            _, k2, c, _ = ors.residual_prepare(w)
        assert k2 == k
        nonmono += bool(np.any(np.diff(c) < 0))
        # NumPy's own searchsorted on the oracle's cumulative sum agrees with the restated bisection
        assert np.array_equal(np.searchsorted(c, U), ref[k:])
        if N <= 4097 and len(U):
            ind = np.array([ors.binsearch_left(c, [u])[0] for u in U])
            dep += not np.array_equal(ind, ref[k:])
    assert nonmono >= 10 and dep >= 1


def test_residual_live_reference(golden):
    """residual_resample(w) after np.random.seed(21) (tests/golden/make_golden.py:gen_spot_checks)."""
    g = golden("spot_checks")
    for N in [3, 50, 3001]:
        w, U, ref = g["res%d_w" % N], g["res%d_U" % N], g["res%d_idx" % N]
        k = int(np.floor(N * w).astype(int).sum())
        assert len(U) == N - k
        assert np.array_equal(ors.residual_resample_vec(w, U), ref)


def test_rts_oracle_vs_reference_vectors(golden):
    g = golden("rts")
    T = g["c1_means"].shape[0]
    out = okf.rts_smoother(g["c1_means"], g["c1_covs"], [g["c1_F"]] * T, [g["c1_Q"]] * T, shift=1)
    for got, key in zip(out, ["c1_x", "c1_P", "c1_K", "c1_Pp"]):
        close(got, g[key], rtol=1e-12, atol=1e-13)
    for form, shift in [("method", 1), ("proc", 0)]:
        out = okf.rts_smoother(g["c1_means"], g["c1_covs"], list(g["tv_Fs"]), list(g["tv_Qs"]), shift=shift)
        for got, key in zip(out, ["x", "P", "K", "Pp"]):
            close(got, g["tv_%s_%s" % (form, key)], rtol=1e-12, atol=1e-13)
    for name in ["b42", "b93"]:
        out = okf.rts_smoother_bank(g[name + "_Xs"], g[name + "_Ps"], g[name + "_F"], g[name + "_Q"])
        for got, key in zip(out, ["x", "P", "K", "Pp"]):
            close(got, g[name + "_" + key], rtol=1e-12, atol=1e-13)


def test_multinomial_and_rts_live_reference(golden):
    """multinomial_resample(w) after np.random.seed(9), and KalmanFilter.rts_smoother on the reference's
    own batch_filter output of a 50-step C1 track (tests/golden/make_golden.py:gen_spot_checks)."""
    g = golden("spot_checks")
    w, U, ref = g["mn_w"], g["mn_U"], g["mn_idx"]
    assert np.array_equal(ors.multinomial_resample_c(w, U), ref)
    out = okf.rts_smoother(g["rts_mu"], g["rts_cov"], [g["rts_F"]] * 50, [g["rts_Q"]] * 50)
    for a, key in zip(out, ["x", "P", "K", "Pp"]):
        close(a, g["rts_" + key], rtol=1e-12, atol=1e-13)


@pytest.mark.parametrize("nm", [2, 3])
def test_imm_and_mmae_oracle_vs_reference_vectors(golden, nm):
    from oracle import imm as oimm
    g = golden("mm")
    zs = g["m%d_zs" % nm]
    T, NT, _ = zs.shape

    def mk(t_):
        return [dict(x=g["m%d_x0" % nm][t_].copy() + j, P=g["m%d_P0" % nm][t_].copy(), F=g["m%d_F" % nm],
                     H=g["m%d_H" % nm], R=g["m%d_R" % nm], Q=g["m%d_Qs" % nm][j]) for j in range(nm)]
    for t_ in range(NT):
        imm = oimm.Imm(mk(t_), g["m%d_mu0" % nm], g["m%d_trans" % nm])
        if t_ == 0:
            close(imm.x, g["imm%d_init_x" % nm]); close(imm.P, g["imm%d_init_P" % nm])
            close(imm.omega, g["imm%d_init_omega" % nm]); close(imm.cbar, g["imm%d_init_cbar" % nm])
        bank = oimm.Mmae(mk(t_), g["m%d_mu0" % nm])
        for k in range(T):
            imm.predict()
            close(imm.x, g["imm%d_xp" % nm][k, t_]); close(imm.P, g["imm%d_Pp" % nm][k, t_])
            imm.update(zs[k, t_])
            close(imm.x, g["imm%d_x" % nm][k, t_]); close(imm.P, g["imm%d_P" % nm][k, t_])
            close(imm.mu, g["imm%d_mu" % nm][k, t_], rtol=1e-8)
            bank.predict(); bank.update(zs[k, t_])
            close(bank.x, g["mmae%d_x" % nm][k, t_]); close(bank.P, g["mmae%d_P" % nm][k, t_])
            close(bank.p, g["mmae%d_p" % nm][k, t_], rtol=1e-8, atol=1e-300)


def test_ukf_rts_oracle_vs_reference_vectors(golden):
    g = golden("ukf_rts")
    al, be, ka = float(g["alpha"]), float(g["beta"]), float(g["kappa"])

    def fx_cv(x, dt):
        o = x.copy()
        o[0::2] = x[0::2] + dt * x[1::2]
        return o
    for name in ("cv", "lin"):
        F = g[name + "_F"]
        fx = fx_cv if name == "cv" else (lambda s, dt: F @ s)
        Xs, Ps = g[name + "_Xs"], g[name + "_Ps"]
        for f in range(Xs.shape[1]):
            x, P, K = oukf.ukf_rts_smoother(Xs[:, f], Ps[:, f], g[name + "_Q"][f], fx, list(g[name + "_dts"]), al, be, ka)
            close(x, g[name + "_x"][:, f], rtol=1e-10, atol=1e-11)
            close(P, g[name + "_P"][:, f], rtol=1e-10, atol=1e-11)
            close(K, g[name + "_K"][:, f], rtol=1e-9, atol=1e-10)
