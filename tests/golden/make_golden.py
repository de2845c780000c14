#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ from the UNMODIFIED reference.

Run with FILTERPY_REFERENCE naming a source checkout of the reference:

    FILTERPY_REFERENCE=<checkout> python tests/golden/make_golden.py

It imports rlabbe/filterpy 1.4.5 (@ 3b51149) from that checkout, feeds it the seeded
synthetic inputs of ``filterpy_b200.common.workloads`` and stores inputs + the reference's
outputs as small ``.npz`` files.  The tests need only the vectors, not the reference:
they compare the oracle (``oracle/``) and the CUDA path against them.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.environ["FILTERPY_REFERENCE"])

from filterpy.kalman import KalmanFilter, UnscentedKalmanFilter, MerweScaledSigmaPoints  # noqa: E402
from filterpy.kalman import predict as kf_predict_proc, update as kf_update_proc          # noqa: E402
from filterpy.monte_carlo import systematic_resample, stratified_resample, multinomial_resample  # noqa: E402
from filterpy.monte_carlo import residual_resample                                                  # noqa: E402
from filterpy.kalman import rts_smoother as rts_proc                                      # noqa: E402
import filterpy                                                                            # noqa: E402

from filterpy_b200.common import workloads as wl                                          # noqa: E402


def save(name, **arrs):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, reference_version=filterpy.__version__, **arrs)
    print("wrote", path, os.path.getsize(path), "bytes")


# ----------------------------------------------------------------------------- KF C1
def gen_kf_c1():
    w = wl.kf_single_cv2d(T=1000, seed=0)
    kf = KalmanFilter(4, 2)
    kf.x = w["x"].copy(); kf.P = w["P"].copy()
    kf.F, kf.H, kf.Q, kf.R = w["F"], w["H"], w["Q"], w["R"]
    means, covs, means_p, covs_p = kf.batch_filter(list(w["zs"]))
    # one-step known answers quoted in SURVEY.md §8c
    k2 = KalmanFilter(4, 2)
    k2.x = np.zeros(4); k2.P = 10 * np.eye(4)
    k2.F, k2.H, k2.Q, k2.R = w["F"], w["H"], w["Q"], w["R"]
    k2.predict(); k2.update(np.array([1., 2.]))
    save("kf_c1", **w, means=means, covs=covs, means_p=means_p, covs_p=covs_p,
         one_x=k2.x, one_P=k2.P, one_S=k2.S, one_K=k2.K,
         one_loglik=k2.log_likelihood, one_maha=float(k2.mahalanobis))


# ----------------------------------------------------------------------------- KF banks
def run_kf_bank(w, steps, alpha=1.0, none_frac=0.0, seed=5, with_control=False):
    N, n = w["x"].shape
    m = w["H"].shape[-2]
    rng = np.random.default_rng(seed)
    valid = rng.random((steps, N)) >= none_frac
    du = 2 if with_control else 0
    B = rng.standard_normal((N, n, du)) if with_control else None
    us = rng.standard_normal((steps, N, du)) if with_control else None
    keys = ["x", "P", "x_prior", "P_prior", "y", "K", "S", "SI", "loglik"]
    out = {k: [] for k in keys}
    filters = []
    for f in range(N):
        kf = KalmanFilter(n, m, dim_u=du)
        kf.x = w["x"][f].copy(); kf.P = w["P"][f].copy()
        kf.F, kf.H, kf.Q, kf.R = w["F"][f], w["H"][f], w["Q"][f], w["R"][f]
        kf.alpha = alpha
        if with_control:
            kf.B = B[f]
        filters.append(kf)
    for t in range(steps):
        rec = {k: [] for k in keys}
        for f, kf in enumerate(filters):
            kf.predict(u=us[t, f] if with_control else None)
            z = w["zs"][t, f] if valid[t, f] else None
            kf.update(z)
            rec["x"].append(kf.x.copy()); rec["P"].append(kf.P.copy())
            rec["x_prior"].append(kf.x_prior.copy()); rec["P_prior"].append(kf.P_prior.copy())
            rec["y"].append(np.asarray(kf.y, float).reshape(m))
            rec["K"].append(kf.K.copy()); rec["S"].append(kf.S.copy()); rec["SI"].append(kf.SI.copy())
            rec["loglik"].append(kf.log_likelihood if z is not None else np.nan)
        for k in keys:
            out[k].append(np.array(rec[k]))
    res = {"ref_" + k: np.array(v) for k, v in out.items()}
    res["valid"] = valid
    res["alpha"] = alpha
    if with_control:
        res["B"] = B; res["us"] = us
    return res


def gen_kf_banks():
    w = wl.kf_bank_cv2d(48, seed=1234, steps=5)
    save("kf_bank_4_2", **w, **run_kf_bank(w, 5, none_frac=0.15))
    w = wl.kf_bank_ca3d(24, seed=4321, steps=3)
    save("kf_bank_9_3", **w, **run_kf_bank(w, 3, alpha=1.02))
    # odd little shapes: random well-conditioned dense models
    rng = np.random.default_rng(99)
    for (n, m) in [(1, 1), (2, 1), (3, 2), (6, 3), (5, 5)]:
        N, steps = 8, 3
        A = rng.standard_normal((N, n, n)) * 0.3
        w = dict(x=rng.standard_normal((N, n)),
                 P=np.einsum("nij,nkj->nik", A, A) + np.eye(n),
                 F=np.eye(n) + 0.1 * rng.standard_normal((N, n, n)),
                 H=rng.standard_normal((N, m, n)),
                 Q=0.01 * np.eye(n) + np.zeros((N, n, n)),
                 R=np.eye(m) * rng.uniform(0.2, 1.0, (N, 1, 1)),
                 zs=rng.standard_normal((steps, N, m)))
        save("kf_bank_%d_%d" % (n, m), **w, **run_kf_bank(w, steps, with_control=(n == 3)))


# ----------------------------------------------------------------------------- UKF
def fx_cv(x, dt):
    o = x.copy()
    o[0::2] = x[0::2] + dt * x[1::2]
    return o


def hx_rae(x):
    px, py, pz = x[0], x[2], x[4]
    return np.array([np.sqrt(px * px + py * py + pz * pz), np.arctan2(py, px),
                     np.arctan2(pz, np.sqrt(px * px + py * py))])


def gen_ukf():
    alpha, beta, kappa = 0.5, 2.0, 0.0
    pts = MerweScaledSigmaPoints(6, alpha, beta, kappa)
    P = np.array([[4, .5, 0, 0, 0, 0], [.5, 2, 0, 0, 0, 0], [0, 0, 3, .2, 0, 0],
                  [0, 0, .2, 1, 0, 0], [0, 0, 0, 0, 5, .1], [0, 0, 0, 0, .1, 1.5]], float)
    x = np.arange(6.0)
    save("ukf_sigma", x=x, P=P, alpha=alpha, beta=beta, kappa=kappa,
         sigmas=pts.sigma_points(x, P), Wm=pts.Wm, Wc=pts.Wc,
         Wm4=MerweScaledSigmaPoints(4, .5, 2, 0).Wm, Wc4=MerweScaledSigmaPoints(4, .5, 2, 0).Wc)
    for name, linear in (("ukf_bank_rae", False), ("ukf_bank_lin", True)):
        N, steps, dt = 16, 5, 0.1
        w = wl.ukf_bank_cv3d(N, seed=2468, steps=steps, dt=dt, linear_hx=linear)
        F, Hlin = w["F"], w["H"]
        fx = (lambda s, dt: F @ s) if linear else fx_cv
        hx = (lambda s: Hlin @ s) if linear else hx_rae
        rng = np.random.default_rng(3)
        valid = rng.random((steps, N)) >= (0.0 if linear else 0.1)
        keys = ["x", "P", "x_prior", "P_prior", "K", "S", "y"]
        out = {k: [] for k in keys}
        ukfs = []
        for f in range(N):
            u = UnscentedKalmanFilter(6, 3, dt, hx, fx, MerweScaledSigmaPoints(6, alpha, beta, kappa))
            u.x = w["x"][f].copy(); u.P = w["P"][f].copy(); u.Q = w["Q"][f]; u.R = w["R"][f]
            ukfs.append(u)
        for t in range(steps):
            rec = {k: [] for k in keys}
            for f, u in enumerate(ukfs):
                u.predict()
                u.update(w["zs"][t, f] if valid[t, f] else None)
                for k in keys:
                    rec[k].append(np.array(getattr(u, k), float).copy())
            for k in keys:
                out[k].append(np.array(rec[k]))
        save(name, **w, valid=valid, dt=dt, alpha=alpha, beta=beta, kappa=kappa,
             **{"ref_" + k: np.array(v) for k, v in out.items()})


def gen_ukf_julier():
    """UKF banks driven by JulierSigmaPoints (sigma_points.py:211-383): kappa > 0 with the range/az/el
    model, kappa < 0 (negative centre weight) with the linear one."""
    from filterpy.kalman import JulierSigmaPoints
    P = np.array([[4, .5, 0, 0], [.5, 2, 0, 0], [0, 0, 3, .2], [0, 0, .2, 1]], float)
    x = np.arange(4.0)
    sig = {}
    for i, k in enumerate([0.0, 1.0, -1.0, 2.5]):
        pts = JulierSigmaPoints(4, k)
        sig.update({"kappa%d" % i: k, "sigmas%d" % i: pts.sigma_points(x, P), "Wm%d" % i: pts.Wm, "Wc%d" % i: pts.Wc})
    save("julier_sigma", x=x, P=P, **sig)
    for name, linear, kappa in (("ukf_julier_rae", False, 1.5), ("ukf_julier_lin", True, -2.0)):
        N, steps, dt = 16, 5, 0.1
        w = wl.ukf_bank_cv3d(N, seed=8642, steps=steps, dt=dt, linear_hx=linear)
        F, Hlin = w["F"], w["H"]
        fx = (lambda s, dt: F @ s) if linear else fx_cv
        hx = (lambda s: Hlin @ s) if linear else hx_rae
        valid = np.random.default_rng(4).random((steps, N)) >= 0.1
        keys = ["x", "P", "x_prior", "P_prior", "K", "S", "y"]
        out = {k: [] for k in keys}
        ukfs = []
        for f in range(N):
            u = UnscentedKalmanFilter(6, 3, dt, hx, fx, JulierSigmaPoints(6, kappa))
            u.x = w["x"][f].copy(); u.P = w["P"][f].copy(); u.Q = w["Q"][f]; u.R = w["R"][f]
            ukfs.append(u)
        for t in range(steps):
            rec = {k: [] for k in keys}
            for f, u in enumerate(ukfs):
                u.predict()
                u.update(w["zs"][t, f] if valid[t, f] else None)
                for k in keys:
                    rec[k].append(np.array(getattr(u, k), float).copy())
            for k in keys:
                out[k].append(np.array(rec[k]))
        save(name, **w, valid=valid, dt=dt, kappa=kappa, **{"ref_" + k: np.array(v) for k, v in out.items()})


def gen_ukf_user():
    """UKF banks with fx / hx OUTSIDE the built-in set: the reference runs the Python callables of
    workloads.py (coordinated turn with a per-filter turn rate passed as fx_args, range / bearing from
    an offset sensor passed as hx_args); the GPU side compiles the CUDA text of the same functions."""
    for name, linear in (("ukf_user_ct_rb", False), ("ukf_user_ct_lin", True)):
        N, steps, dt = 16, 6, 0.5
        w = wl.ukf_bank_ct2d(N, steps=steps, dt=dt, linear_hx=linear)
        Hlin, sensor = w["H"], w["sensor"]
        hx = (lambda s: Hlin @ s) if linear else wl.offset_rb_hx
        valid = np.random.default_rng(5).random((steps, N)) >= 0.1
        keys = ["x", "P", "x_prior", "P_prior", "K", "S", "y"]
        out = {k: [] for k in keys}
        ukfs = []
        for f in range(N):
            u = UnscentedKalmanFilter(4, 2, dt, hx, wl.ct_fx, MerweScaledSigmaPoints(4, 0.5, 2.0, 0.0))
            u.x = w["x"][f].copy(); u.P = w["P"][f].copy(); u.Q = w["Q"][f]; u.R = w["R"][f]
            ukfs.append(u)
        for t in range(steps):
            rec = {k: [] for k in keys}
            for f, u in enumerate(ukfs):
                u.predict(omega=w["omega"][f])
                z = w["zs"][t, f] if valid[t, f] else None
                if linear:
                    u.update(z)
                else:
                    u.update(z, sx=sensor[0], sy=sensor[1])
                for k in keys:
                    rec[k].append(np.array(getattr(u, k), float).copy())
            for k in keys:
                out[k].append(np.array(rec[k]))
        save(name, **w, valid=valid, dt=dt, alpha=0.5, beta=2.0, kappa=0.0,
             **{"ref_" + k: np.array(v) for k, v in out.items()})
    # RTS smoother around the user fx: the reference calls fx(sigma, dt) without keyword arguments there
    # (UKF.py:712), so the turn rate is the callable's default
    N, steps, dt, om = 6, 10, 0.5, 0.07
    w = wl.ukf_bank_ct2d(N, seed=1122, steps=steps, dt=dt, linear_hx=True)
    Hlin = w["H"]
    Xs = np.zeros((steps, N, 4)); Ps = np.zeros((steps, N, 4, 4))
    sm = [np.zeros((steps, N, 4)), np.zeros((steps, N, 4, 4)), np.zeros((steps, N, 4, 4))]
    for f in range(N):
        u = UnscentedKalmanFilter(4, 2, dt, lambda s: Hlin @ s, lambda s, dt, omega=om: wl.ct_fx(s, dt, omega),
                                  MerweScaledSigmaPoints(4, 0.5, 2.0, 0.0))
        u.x = w["x"][f].copy(); u.P = w["P"][f].copy(); u.Q = w["Q"][f]; u.R = w["R"][f]
        mu, cov = u.batch_filter(list(w["zs"][:, f]))
        Xs[:, f] = mu; Ps[:, f] = cov
        for o, v in zip(sm, u.rts_smoother(mu, cov)):
            o[:, f] = v
    save("ukf_user_rts", Xs=Xs, Ps=Ps, x=sm[0], P=sm[1], K=sm[2], Q=w["Q"], H=Hlin, dt=dt, omega=om, alpha=0.5, beta=2.0, kappa=0.0)


# ----------------------------------------------------------------------------- resampling
def gen_resample():
    cases = {}
    meta = []
    i = 0
    for kind in ["heavy", "uniform", "random", "zeros", "degenerate", "dyadic"]:
        for N in [1, 2, 7, 64, 1000, 4097]:
            w = wl.resample_weights(N, kind, seed=97 + N)
            np.random.seed(7 + i)
            st = np.random.get_state()
            try:
                idx = systematic_resample(w)
                ok = 1
            except IndexError:
                idx = np.zeros(0, 'i'); ok = 0
            np.random.set_state(st)
            u = np.random.random()
            np.random.set_state(st)
            try:
                idx_s = stratified_resample(w)
                ok_s = 1
            except IndexError:
                idx_s = np.zeros(0, 'i'); ok_s = 0
            np.random.set_state(st)
            U = np.random.random(N)
            cases["w%d" % i] = w; cases["u%d" % i] = u; cases["U%d" % i] = U
            cases["sys%d" % i] = idx; cases["str%d" % i] = idx_s
            meta.append((i, N, ok, ok_s, 7 + i))
            i += 1
    # the SURVEY known answer: systematic_resample([.1,.2,.3,.4]) with u = 0.5 -> [1,2,3,3]
    import filterpy.monte_carlo.resampling as rs
    old = rs.random
    rs.random = lambda *a: 0.5 if not a else np.full(a[0], 0.5)
    ka = systematic_resample([.1, .2, .3, .4]); ka_s = stratified_resample([.1, .2, .3, .4])
    rs.random = old
    save("resample", meta=np.array(meta), known_sys=ka, known_str=ka_s, **cases)


def gen_multinomial():
    cases = {}
    meta = []
    i = 0
    for kind in ["heavy", "uniform", "zeros", "degenerate", "dyadic"]:
        for N in [1, 2, 7, 1000, 4097]:
            w = wl.resample_weights(N, kind, seed=31 + N)
            np.random.seed(100 + i)
            idx = multinomial_resample(w)
            np.random.seed(100 + i)
            U = np.random.random(N)
            cases["w%d" % i] = w; cases["U%d" % i] = U; cases["idx%d" % i] = idx
            meta.append((i, N, 100 + i))
            i += 1
    save("resample_multinomial", meta=np.array(meta), **cases)


def gen_residual():
    """residual_resample (resampling.py:27-76) on the weight families of the resample goldens: the
    reference's result, the uniforms it drew (random(N - k) after seeding) and k."""
    cases = {}
    meta = []
    i = 0
    for kind in ["heavy", "uniform", "zeros", "degenerate", "dyadic"]:
        for N in [1, 2, 7, 100, 1000, 4097, 20011]:
            w = wl.resample_weights(N, kind, seed=57 + N)
            np.random.seed(300 + i)
            idx = residual_resample(w.copy())
            k = int(np.floor(N * w).astype(int).sum())
            np.random.seed(300 + i)
            U = np.random.random(N - k)
            cases["w%d" % i] = w; cases["U%d" % i] = U; cases["idx%d" % i] = idx
            meta.append((i, N, 300 + i, k))
            i += 1
    save("resample_residual", meta=np.array(meta), **cases)


# ----------------------------------------------------------------------------- RTS smoother
def gen_rts():
    out = {}
    # (1) the C1 single filter: batch_filter then the method (Fs[k+1]) and the procedural form (Fs[k])
    w = wl.kf_single_cv2d(T=200, seed=3)
    kf = KalmanFilter(4, 2)
    kf.x = w["x"].copy(); kf.P = w["P"].copy()
    kf.F, kf.H, kf.Q, kf.R = w["F"], w["H"], w["Q"], w["R"]
    means, covs, _, _ = kf.batch_filter(list(w["zs"]))
    x, P, K, Pp = kf.rts_smoother(means, covs)
    out.update(c1_F=w["F"], c1_Q=w["Q"], c1_means=means, c1_covs=covs, c1_x=x, c1_P=P, c1_K=K, c1_Pp=Pp)
    # per-epoch models: F_k = CV with dt_k, Q_k scaled
    rng = np.random.default_rng(11)
    T = means.shape[0]
    Fs, Qs = [], []
    for k in range(T):
        dt = rng.uniform(0.5, 1.5)
        F = np.eye(4); F[0, 1] = dt; F[2, 3] = dt
        Fs.append(F); Qs.append(w["Q"] * rng.uniform(0.5, 2.0))
    xm, Pm, Km, Ppm = kf.rts_smoother(means, covs, Fs=Fs, Qs=Qs)
    xp, Pq, Kp, Ppp = rts_proc(means, covs, Fs, Qs)
    out.update(tv_Fs=np.array(Fs), tv_Qs=np.array(Qs), tv_method_x=xm, tv_method_P=Pm, tv_method_K=Km, tv_method_Pp=Ppm,
               tv_proc_x=xp, tv_proc_P=Pq, tv_proc_K=Kp, tv_proc_Pp=Ppp)
    # (2) small banks with per-filter models: 4/2, 2/1, 6/3 (generic kernel), column-vector x
    for name, bank in [("b42", wl.kf_bank_cv2d(24, seed=21)), ("b93", wl.kf_bank_ca3d(6, seed=22))]:
        N, n = bank["x"].shape
        T = 30
        m = bank["H"].shape[-2]
        zs = np.random.default_rng(5).normal(size=(T, N, m)) + np.einsum("nij,nj->ni", bank["H"], bank["x"])[None]
        Xs = np.zeros((T, N, n)); Ps = np.zeros((T, N, n, n))
        sm = [np.zeros((T, N, n)), np.zeros((T, N, n, n)), np.zeros((T, N, n, n)), np.zeros((T, N, n, n))]
        for i in range(N):
            f = KalmanFilter(n, m)
            f.x = bank["x"][i].copy(); f.P = bank["P"][i].copy()
            f.F, f.H, f.Q, f.R = bank["F"][i], bank["H"][i], bank["Q"][i], bank["R"][i]
            mu, cov, _, _ = f.batch_filter(list(zs[:, i]))
            Xs[:, i] = mu; Ps[:, i] = cov
            r = f.rts_smoother(mu, cov)
            for o, v in zip(sm, r):
                o[:, i] = v
        out.update({name + "_F": bank["F"], name + "_Q": bank["Q"], name + "_Xs": Xs, name + "_Ps": Ps,
                    name + "_x": sm[0], name + "_P": sm[1], name + "_K": sm[2], name + "_Pp": sm[3]})
    save("rts", **out)


# ----------------------------------------------------------------------------- UKF RTS smoother
def gen_ukf_rts():
    alpha, beta, kappa = 0.5, 2.0, 0.0
    out = {}
    for name, linear in (("cv", False), ("lin", True)):
        N, steps, dt = 6, 12, 0.1
        w = wl.ukf_bank_cv3d(N, seed=1357, steps=steps, dt=dt, linear_hx=True)
        F, Hlin = w["F"], w["H"]
        fx = (lambda s, dt: F @ s) if linear else fx_cv
        hx = lambda s: Hlin @ s                                   # noqa: E731
        dts = list(np.random.default_rng(1).uniform(0.05, 0.15, steps)) if not linear else None
        Xs = np.zeros((steps, N, 6)); Ps = np.zeros((steps, N, 6, 6))
        sm = [np.zeros((steps, N, 6)), np.zeros((steps, N, 6, 6)), np.zeros((steps, N, 6, 6))]
        for f in range(N):
            u = UnscentedKalmanFilter(6, 3, dt, hx, fx, MerweScaledSigmaPoints(6, alpha, beta, kappa))
            u.x = w["x"][f].copy(); u.P = w["P"][f].copy(); u.Q = w["Q"][f]; u.R = w["R"][f]
            mu, cov = u.batch_filter(list(w["zs"][:, f]), dts=dts)
            Xs[:, f] = mu; Ps[:, f] = cov
            r = u.rts_smoother(mu, cov, dts=dts)
            for o, v in zip(sm, r):
                o[:, f] = v
        out.update({name + "_Xs": Xs, name + "_Ps": Ps, name + "_x": sm[0], name + "_P": sm[1], name + "_K": sm[2],
                    name + "_Q": w["Q"], name + "_F": F, name + "_dt": dt,
                    name + "_dts": np.array(dts if dts is not None else [dt] * steps)})
    save("ukf_rts", alpha=alpha, beta=beta, kappa=kappa, **out)


# ----------------------------------------------------------------------------- IMM / MMAE
def mm_models(n_tracks, seed):
    """Two / three CV models (different process noise) per track, dim_x=4, dim_z=2, 1-D x."""
    rng = np.random.default_rng(seed)
    c = wl.kf_single_cv2d(T=1, seed=0)
    x0 = rng.normal(size=(n_tracks, 4)) * 3
    P0 = np.array([np.diag(rng.uniform(1, 5, 4)) for _ in range(n_tracks)])
    qs = [0.05, 1.0, 8.0]
    return dict(F=c["F"], H=c["H"], R=c["R"], Qs=np.array([c["Q"] * q for q in qs]), x0=x0, P0=P0)


def gen_mm():
    from filterpy.kalman import IMMEstimator, MMAEFilterBank
    out = {}
    T, NT = 25, 12
    for nm in (2, 3):
        mdl = mm_models(NT, 40 + nm)
        rng = np.random.default_rng(7 + nm)
        zs = rng.normal(size=(T, NT, 2)) * 2 + np.cumsum(rng.normal(size=(T, NT, 2)), axis=0)
        trans = np.array([[0.9, 0.1], [0.2, 0.8]]) if nm == 2 else np.array([[.9, .05, .05], [.1, .8, .1], [.05, .15, .8]])
        mu0 = np.array([0.6, 0.4]) if nm == 2 else np.array([0.5, 0.3, 0.2])
        rec = {k: np.zeros((T, NT) + shp) for k, shp in [("x", (4,)), ("P", (4, 4)), ("mu", (nm,)), ("xp", (4,)), ("Pp", (4, 4)),
                                                           ("fx", (nm, 4)), ("fP", (nm, 4, 4))]}
        mrec = {k: np.zeros((T, NT) + shp) for k, shp in [("x", (4,)), ("P", (4, 4)), ("p", (nm,))]}
        for t_ in range(NT):
            def mk():
                fs = []
                for j in range(nm):
                    f = KalmanFilter(4, 2)
                    f.x = mdl["x0"][t_].copy() + j; f.P = mdl["P0"][t_].copy()
                    f.F, f.H, f.R, f.Q = mdl["F"], mdl["H"], mdl["R"], mdl["Qs"][j]
                    fs.append(f)
                return fs
            imm = IMMEstimator(mk(), mu0, trans)
            if t_ == 0:
                out["imm%d_init_x" % nm] = imm.x.copy(); out["imm%d_init_P" % nm] = imm.P.copy()
                out["imm%d_init_omega" % nm] = imm.omega.copy(); out["imm%d_init_cbar" % nm] = imm.cbar.copy()
            for k in range(T):
                imm.predict()
                rec["xp"][k, t_] = imm.x; rec["Pp"][k, t_] = imm.P
                imm.update(zs[k, t_])
                rec["x"][k, t_] = imm.x; rec["P"][k, t_] = imm.P; rec["mu"][k, t_] = imm.mu
                for j, f in enumerate(imm.filters):
                    rec["fx"][k, t_, j] = f.x; rec["fP"][k, t_, j] = f.P
            bank = MMAEFilterBank(mk(), list(mu0), dim_x=4)
            for k in range(T):
                bank.predict()
                bank.update(zs[k, t_])
                mrec["x"][k, t_] = bank.x; mrec["P"][k, t_] = bank.P; mrec["p"][k, t_] = bank.p
        out.update({"m%d_zs" % nm: zs, "m%d_trans" % nm: trans, "m%d_mu0" % nm: mu0, "m%d_F" % nm: mdl["F"], "m%d_H" % nm: mdl["H"],
                    "m%d_R" % nm: mdl["R"], "m%d_Qs" % nm: mdl["Qs"][:nm], "m%d_x0" % nm: mdl["x0"], "m%d_P0" % nm: mdl["P0"]})
        out.update({"imm%d_%s" % (nm, k): v for k, v in rec.items()})
        out.update({"mmae%d_%s" % (nm, k): v for k, v in mrec.items()})
    save("mm", **out)


# ----------------------------------------------------------------------------- spot checks
def gen_spot_checks():
    """The reference's public functions called the way a user calls them (seeded global RNG):
    systematic / residual / multinomial resample, a 5-filter KF bank and the RTS smoother of C1."""
    out = {}
    w = wl.resample_weights(20000, "heavy", seed=5)
    np.random.seed(123); st = np.random.get_state()
    out["sys_idx"] = systematic_resample(w)
    np.random.set_state(st)
    out.update(sys_w=w, sys_u=np.random.random())
    b = wl.kf_bank_cv2d(5, seed=11, steps=2)
    xs, Ps = [], []
    for f in range(5):
        kf = KalmanFilter(4, 2); kf.x = b["x"][f].copy(); kf.P = b["P"][f].copy()
        kf.F, kf.H, kf.Q, kf.R = b["F"][f], b["H"][f], b["Q"][f], b["R"][f]
        for t in range(2):
            kf.predict(); kf.update(b["zs"][t, f])
        xs.append(kf.x); Ps.append(kf.P)
    out.update({"kf_" + k: v for k, v in b.items()})
    out.update(kf_ref_x=np.array(xs), kf_ref_P=np.array(Ps))
    rng = np.random.default_rng(5)
    for N in [3, 50, 3001]:
        w = rng.random(N) ** 3
        w /= w.sum()
        np.random.seed(21); idx = residual_resample(w.copy())
        k = int(np.floor(N * w).astype(int).sum())
        np.random.seed(21)
        out.update({"res%d_w" % N: w, "res%d_U" % N: np.random.random(N - k), "res%d_idx" % N: idx})
    rng = np.random.default_rng(0)
    w = rng.random(5000) ** 3
    w /= w.sum()
    np.random.seed(9); idx = multinomial_resample(w)
    np.random.seed(9)
    out.update(mn_w=w, mn_U=np.random.random(len(w)), mn_idx=idx)
    c = wl.kf_single_cv2d(T=50, seed=2)
    kf = KalmanFilter(4, 2)
    kf.x = c["x"].copy(); kf.P = c["P"].copy(); kf.F, kf.H, kf.Q, kf.R = c["F"], c["H"], c["Q"], c["R"]
    mu, cov, _, _ = kf.batch_filter(list(c["zs"]))
    x, P, K, Pp = kf.rts_smoother(mu, cov)
    out.update(rts_F=c["F"], rts_Q=c["Q"], rts_mu=mu, rts_cov=cov, rts_x=x, rts_P=P, rts_K=K, rts_Pp=Pp)
    save("spot_checks", **out)


if __name__ == "__main__":
    if len(sys.argv) > 1:                       # e.g. `make_golden.py gen_ukf_julier`: only the named generators
        for g in sys.argv[1:]:
            globals()[g]()
        sys.exit(0)
    gen_kf_c1()
    gen_kf_banks()
    gen_ukf()
    gen_resample()
    gen_multinomial()
    gen_residual()
    gen_rts()
    gen_ukf_rts()
    gen_mm()
    gen_ukf_julier()
    gen_ukf_user()
    gen_spot_checks()
