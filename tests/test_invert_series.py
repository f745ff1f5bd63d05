"""Joint inversion of time series on the device: gpe_bank_solve_series / gpe_multi_bank_solve_series,
DeviceBank.invert_series / forward_invert_series and MultivariateEmulator.invert_series (DESIGN 4.6g).

``lm_series_ref`` restates the algorithm of include/gpemu.h in numpy with a dense solve of the series' system.  On the CPU
it is checked against a textbook Rauch-Tung-Striebel smoother and an analytic bounded optimum; on the GPU it drives the
library's own cost calls and the device solver must land where it lands."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import scipy.linalg

from tests.conftest import ROOT
from tests.test_invert import CONVERGED, NONFINITE, _bank, _cost, _models, _own_obs, _problem, _prosail, _solve

MAX_ITER, STALLED = 1, 2


def _coupling(T, coupling):
    return np.ones(T - 1) if coupling is None else np.asarray(coupling, dtype=np.float64)


def series_hessian(hess, R, coupling):
    """Dense (T D, T D) Hessian of one series from its diagonal blocks without the coupling (T, D, D)."""
    T, D = hess.shape[:2]
    c = _coupling(T, coupling)
    H = np.zeros((T * D, T * D))
    for t in range(T):
        H[t * D:(t + 1) * D, t * D:(t + 1) * D] = hess[t]
    for t in range(1, T):
        a, b = slice((t - 1) * D, t * D), slice(t * D, (t + 1) * D)
        H[a, a] += c[t - 1] * R
        H[b, b] += c[t - 1] * R
        H[a, b] -= c[t - 1] * R
        H[b, a] -= c[t - 1] * R
    return H


def dense_hessian(blocks, R, coupling):
    """Dense Hessian of one series from the diagonal blocks the solver returns (coupling included)."""
    T = blocks.shape[0]
    c = _coupling(T, coupling)
    own = blocks.copy()
    for t in range(T):
        own[t] -= ((c[t - 1] if t > 0 else 0.0) + (c[t] if t + 1 < T else 0.0)) * R
    return series_hessian(own, R, c)


def lm_series_ref(fgh, x0, R, coupling=None, lower=None, upper=None, prior_mean=None, prior_prec=None, max_iter=50,
                  ftol=1e-10, xtol=1e-10, gtol=0.0, lambda0=1e-3):
    """The algorithm of include/gpemu.h for series.  x0 (S, T, D); fgh(X (n, D), rows) -> f (n,), g (n, D), H (n, D, D)
    of the per-date cost at rows n = s T + t.  Returns x (S, T, D), cost (S), grad (S, T, D), hess (S, T, D, D) diagonal
    blocks with the coupling, cov (S, T, D, D) diagonal blocks of inv(H), status and n_iter (S)."""
    x0 = np.asarray(x0, dtype=np.float64)
    S, T, D = x0.shape
    c = _coupling(T, coupling)
    lo = np.full(D, -np.inf) if lower is None else np.asarray(lower, dtype=np.float64)
    hi = np.full(D, np.inf) if upper is None else np.asarray(upper, dtype=np.float64)
    m = np.zeros((S, T, D)) if prior_mean is None else np.broadcast_to(np.asarray(prior_mean, dtype=np.float64), (S, T, D))

    def evaluate(X, sidx):
        rows = (sidx[:, None] * T + np.arange(T)).ravel()
        f, g, H = (np.array(a, dtype=np.float64) for a in fgh(X.reshape(-1, D), rows))
        f, g, H = f.reshape(len(sidx), T), g.reshape(len(sidx), T, D), H.reshape(len(sidx), T, D, D)
        if prior_prec is not None:
            r = X - m[sidx]
            pr = r @ np.asarray(prior_prec).T
            f = f + 0.5 * np.sum(r * pr, axis=2)
            g = g + pr
            H = H + prior_prec
        fs = f.sum(axis=1)
        for t in range(1, T):
            e = X[:, t] - X[:, t - 1]
            Re = e @ R.T
            fs = fs + 0.5 * c[t - 1] * np.sum(e * Re, axis=1)
            g[:, t] += c[t - 1] * Re
            g[:, t - 1] -= c[t - 1] * Re
        return fs, g, H

    x = np.clip(x0, lo, hi)
    f, g, H = evaluate(x, np.arange(S))
    lam, nu = np.full(S, float(lambda0)), np.full(S, 2.0)
    nev, status = np.zeros(S, dtype=np.int64), np.full(S, -1)
    pred, xt = np.zeros(S), x.copy()
    status[~np.isfinite(f)] = NONFINITE

    def propose(k):
        free = (~(((x[k] <= lo) & (g[k] > 0)) | ((x[k] >= hi) & (g[k] < 0)))).ravel()
        gk = g[k].ravel()
        if np.max(np.abs(gk[free]), initial=0.0) <= gtol:
            return CONVERGED
        Hd = series_hessian(H[k], R, c)
        F = np.flatnonzero(free)
        HF = Hd[np.ix_(F, F)]
        dg = np.abs(np.diag(HF))
        s = np.maximum(dg, 1e-12 * dg.max())
        while True:
            if not lam[k] <= 1e20:
                return STALLED
            try:
                L = np.linalg.cholesky(HF + lam[k] * np.diag(s))
                break
            except np.linalg.LinAlgError:
                lam[k] *= nu[k]
                nu[k] *= 2.0
        step = np.zeros(T * D)
        step[F] = scipy.linalg.cho_solve((L, True), -gk[F])
        t_ = np.clip(x[k] + step.reshape(T, D), lo, hi)
        d = (t_ - x[k]).ravel()
        if np.max(np.abs(d)) <= xtol * (np.max(np.abs(x[k])) + xtol):
            return CONVERGED
        if nev[k] >= max_iter:
            return MAX_ITER
        pred[k] = -(gk @ d + 0.5 * d @ Hd @ d)
        xt[k] = t_
        return -1

    for k in np.flatnonzero(status < 0):
        status[k] = propose(k)
    while np.any(status < 0):
        idx = np.flatnonzero(status < 0)
        ft, gt, Ht = evaluate(xt[idx], idx)
        for j, k in enumerate(idx):
            nev[k] += 1
            with np.errstate(divide="ignore", invalid="ignore"):
                rho = (f[k] - ft[j]) / pred[k]
            if ft[j] < f[k] and rho > 0:
                f_old = f[k]
                x[k], f[k], g[k], H[k] = xt[k], ft[j], gt[j], Ht[j]
                lam[k] *= max(1.0 / 3.0, 1.0 - (2.0 * rho - 1.0) ** 3)
                nu[k] = 2.0
                if abs(f_old - f[k]) <= ftol * abs(f[k]):
                    status[k] = CONVERGED
                    continue
            else:
                lam[k] *= nu[k]
                nu[k] *= 2.0
            status[k] = propose(k)
    hess = H.copy()
    cov = np.full_like(H, np.nan)
    for k in range(S):
        Hd = series_hessian(H[k], R, c)
        for t in range(T):
            hess[k, t] = Hd[t * D:(t + 1) * D, t * D:(t + 1) * D]
        if np.all(np.linalg.eigvalsh(Hd) > 0):
            inv = np.linalg.inv(Hd)
            for t in range(T):
                cov[k, t] = inv[t * D:(t + 1) * D, t * D:(t + 1) * D]
    return {"x": x, "cost": f, "grad": g, "hess": hess, "cov": cov, "status": status, "n_iter": nev}


# ---- CPU: the reference against closed forms -------------------------------------------------------------------------
def _linear_gaussian(A, Wt, y):
    """fgh of cost_n(x) = 1/2 (y_n - A x)^T diag(Wt_n) (y_n - A x), one row of y and Wt per row n."""
    def fgh(X, rows):
        r = X @ A.T - y[rows]
        w = Wt[rows]
        H = np.einsum("ek,ne,el->nkl", A, w, A)
        return 0.5 * np.sum(w * r * r, axis=1), (w * r) @ A, H
    return fgh


def _rts(A, Wt, y, P, m, R, c):
    """Kalman filter + Rauch-Tung-Striebel smoother of one series: x_t = x_t-1 + N(0, inv(c_t R)); observations
    y_t = A x_t + N(0, diag(1 / Wt_t)) and m_t = x_t + N(0, inv(P)); flat prior on x_0."""
    T, D = m.shape
    Hm = np.vstack([A, np.eye(D)])
    mf, Pf, mp, Pp = np.zeros((T, D)), np.zeros((T, D, D)), np.zeros((T, D)), np.zeros((T, D, D))
    for t in range(T):
        Rinv = scipy.linalg.block_diag(np.diag(Wt[t]), P)         # observation precision
        z = np.concatenate([y[t], m[t]])
        if t == 0:
            info = Hm.T @ Rinv @ Hm
            Pf[0] = np.linalg.inv(info)
            mf[0] = Pf[0] @ (Hm.T @ Rinv @ z)
            continue
        mp[t], Pp[t] = mf[t - 1], Pf[t - 1] + np.linalg.inv(c[t - 1] * R)
        # the update in information form: a masked date has a singular observation precision
        Pf[t] = np.linalg.inv(np.linalg.inv(Pp[t]) + Hm.T @ Rinv @ Hm)
        mf[t] = Pf[t] @ (np.linalg.solve(Pp[t], mp[t]) + Hm.T @ Rinv @ z)
    ms, Ps = mf.copy(), Pf.copy()
    for t in range(T - 2, -1, -1):
        G = Pf[t] @ np.linalg.inv(Pp[t + 1])
        ms[t] = mf[t] + G @ (ms[t + 1] - mp[t + 1])
        Ps[t] = Pf[t] + G @ (Ps[t + 1] - Pp[t + 1]) @ G.T
    return ms, Ps


def test_reference_matches_a_rauch_tung_striebel_smoother():
    rs = np.random.RandomState(0)
    S, T, D, E = 3, 9, 3, 4
    A = rs.standard_normal((E, D))
    Q = rs.standard_normal((D, D))
    R = Q @ Q.T + 0.5 * np.eye(D)
    P = np.diag(rs.uniform(0.05, 0.2, D))
    c = rs.uniform(0.2, 3.0, T - 1)                       # irregular dates
    Wt = rs.uniform(0.5, 2.0, (S * T, E))
    Wt[rs.random_sample(S * T) < 0.3] = 0.0               # masked dates
    y = rs.standard_normal((S * T, E))
    m = rs.standard_normal((S, T, D))
    res = lm_series_ref(_linear_gaussian(A, Wt, y), rs.standard_normal((S, T, D)), R, c, prior_mean=m, prior_prec=P,
                        max_iter=100, ftol=0.0, gtol=1e-13)
    assert np.all(res["status"] == CONVERGED)
    for s in range(S):
        ms, Ps = _rts(A, Wt[s * T:(s + 1) * T], y[s * T:(s + 1) * T], P, m[s], R, c)
        assert np.max(np.abs(res["x"][s] - ms)) < 1e-10 * max(1.0, np.abs(ms).max())
        assert np.max(np.abs(res["cov"][s] - Ps)) < 1e-10 * np.abs(Ps).max()


def test_reference_finds_an_analytic_bounded_optimum():
    """Diagonal model, every date observing input 0 beyond the upper bound: input 0 sits on the bound on every date (where
    the smoothness term vanishes), input 1 is the interior solution of its own tridiagonal system."""
    T, D = 7, 2
    rs = np.random.RandomState(1)
    A = np.eye(D)
    w = np.array([1.0, 2.0])
    R = np.diag([3.0, 5.0])
    c = rs.uniform(0.5, 2.0, T - 1)
    y = np.stack([np.full(T, 2.0), rs.uniform(0.2, 0.8, T)], axis=1)
    res = lm_series_ref(_linear_gaussian(A, np.tile(w, (T, 1)), y), np.full((1, T, D), 0.5), R, c, lower=np.zeros(D),
                        upper=np.ones(D), max_iter=100, ftol=0.0, gtol=1e-13)
    assert res["status"][0] == CONVERGED
    assert np.all(res["x"][0, :, 0] == 1.0) and np.all(res["grad"][0, :, 0] < 0)
    H1 = series_hessian(np.full((T, 1, 1), w[1]), R[1:, 1:], c)
    want = np.linalg.solve(H1, w[1] * y[:, 1])
    assert np.max(np.abs(res["x"][0, :, 1] - want)) < 1e-12


def test_header_and_bindings_agree():
    from gp_emulator_b200 import _lib
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "gpemu.h")).read(), flags=re.S)
    lib = _lib.load()
    for name in ("gpe_bank_solve_series", "gpe_multi_bank_solve_series"):
        assert name in _lib.SYMBOLS
        params = re.search(r"\b%s\s*\(([^)]*)\)" % name, text).group(1).split(",")
        assert len(params) == len(getattr(lib, name).argtypes), name
    params = re.search(r"\bgpe_bank_solve_series\s*\(([^)]*)\)", text).group(1)
    names = [p.split()[-1].lstrip("*") for p in params.split(",")]
    assert names[:3] == ["b", "S", "T"] and names[9:11] == ["smooth_prec", "coupling"]


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpemu(lib):
    import gp_emulator_b200 as g
    assert lib.gpe_device_count() > 0, "no GPU visible: the gpu tests must not pass on a fallback"
    return g


def _series(bank, spectra, *a, **k):
    return (bank.forward_invert_series if spectra else bank.invert_series)(*a, **k)


def _spd(rs, D, scale):
    Q = rs.standard_normal((D, D))
    R = Q @ Q.T / D + 0.1 * np.eye(D)
    R = 0.5 * (R + R.T)
    return scale * R


def _trajectory(rs, lo, hi, S, T):
    """Smooth x_true (S, T, D) inside the box: a sine of random phase per input around a random centre."""
    D = len(lo)
    width = hi - lo
    ctr = lo + width * rs.uniform(0.35, 0.65, (S, 1, D))
    ph = rs.uniform(0, 2 * np.pi, (S, 1, D))
    t = np.arange(T)[None, :, None]
    return ctr + 0.2 * width * np.sin(2 * np.pi * t / T + ph)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fwd", "prosail", "band"])
def test_one_date_is_the_point_solver_bit_for_bit(gpemu, kind):
    bank, spectra, lo, hi, rs = _problem(gpemu, kind)
    N, D = 80, len(lo)
    width = hi - lo
    x_true = lo + width * rs.uniform(0.1, 0.9, (N, D))
    obs = _own_obs(bank, spectra, x_true)
    obs = obs * (1.0 + 0.01 * rs.standard_normal(obs.shape))
    w = rs.uniform(0.5, 2.0, obs.shape)
    x0 = np.clip(x_true + 0.05 * width * rs.standard_normal(x_true.shape), lo, hi)
    P = np.diag(1.0 / (0.3 * width) ** 2)
    pm = lo + width * rs.uniform(0.3, 0.7, (N, D))
    kw = dict(lower=lo, upper=hi, prior_mean=pm, prior_precision=P, max_iter=60, want_cov=True)
    ref = _solve(bank, spectra, x0, obs, w, **kw)
    kws = dict(kw, prior_mean=pm[:, None])
    got = _series(bank, spectra, x0[:, None], obs[:, None], w[:, None], smooth_precision=_spd(rs, D, 7.0), **kws)
    for k in ("x", "grad", "hess", "cov"):
        assert np.array_equal(got[k][:, 0], ref[k], equal_nan=True), k
    for k in ("cost", "status", "n_iter"):
        assert np.array_equal(got[k], ref[k], equal_nan=True), k


@pytest.mark.gpu
@pytest.mark.parametrize("D", [3, 12, 20, 32])
def test_one_date_is_the_point_solver_bit_for_bit_at_every_dp(gpemu, D):
    """Band banks whose D selects each compiled instance of the series kernels (DP = 8, 16, 32), with a prior and cov."""
    bank, rs = _bank(gpemu, 16, D)
    N = 120
    x_true = rs.uniform(0.1, 0.9, (N, D))
    obs = _own_obs(bank, False, x_true)
    obs = obs * (1.0 + 0.01 * rs.standard_normal(obs.shape))
    x0 = np.clip(x_true + 0.05 * rs.standard_normal(x_true.shape), 0, 1)
    pm = rs.uniform(0.3, 0.7, (N, D))
    kw = dict(lower=np.zeros(D), upper=np.ones(D), prior_mean=pm, prior_precision=np.eye(D), max_iter=60, want_cov=True)
    ref = bank.invert(x0, obs, **kw)
    got = bank.invert_series(x0[:, None], obs[:, None], smooth_precision=_spd(rs, D, 3.0), **dict(kw, prior_mean=pm[:, None]))
    assert len(np.unique(ref["n_iter"])) > 1
    for k in ("x", "grad", "hess", "cov"):
        assert np.array_equal(got[k][:, 0], ref[k], equal_nan=True), k
    for k in ("cost", "status", "n_iter"):
        assert np.array_equal(got[k], ref[k], equal_nan=True), k


def _masked_problem(gpemu, kind, S, T, rs_seed=3, frac=0.3):
    bank, spectra, lo, hi, rs = _problem(gpemu, kind)
    rs = np.random.RandomState(rs_seed)
    x_true = _trajectory(rs, lo, hi, S, T)
    D = len(lo)
    obs = _own_obs(bank, spectra, x_true.reshape(-1, D))
    obs = obs * (1.0 + 0.01 * rs.standard_normal(obs.shape))
    w = np.tile(rs.uniform(0.5, 2.0, obs.shape[1]), (S * T, 1))
    w[rs.random_sample(S * T) < frac] = 0.0
    K = obs.shape[1]
    return bank, spectra, lo, hi, rs, x_true, obs.reshape(S, T, K), w.reshape(S, T, K)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fwd", "prosail", "band"])
def test_agreement_with_the_reference_driving_the_library_costs(gpemu, kind):
    S, T = 12, 10
    bank, spectra, lo, hi, rs, x_true, obs, w = _masked_problem(gpemu, kind, S, T)
    D, K = len(lo), obs.shape[2]
    width = hi - lo
    x0 = np.clip(x_true + 0.05 * width * rs.standard_normal(x_true.shape), lo, hi)
    R = np.diag(1.0 / (0.1 * width) ** 2)
    c = rs.uniform(0.3, 2.0, T - 1)
    flat_obs, flat_w = obs.reshape(-1, K), w.reshape(-1, K)

    def fgh(X, rows):
        # every evaluation covers all S T rows, as the solver's do (call_N = S T): the same kernel plans
        allx = x0.reshape(-1, D).copy()
        allx[rows] = X
        out = _cost(bank, spectra, allx, flat_obs, flat_w, want_hess=True)
        return out["cost"][rows], out["grad"][rows], out["hess"][rows]

    ref = lm_series_ref(fgh, x0, R, c, lo, hi, max_iter=100)
    got = _series(bank, spectra, x0, obs, w, smooth_precision=R, coupling=c, lower=lo, upper=hi, max_iter=100)
    assert np.array_equal(got["status"], ref["status"])
    ok = ref["status"] == CONVERGED
    assert np.mean(ok) >= 0.5
    assert np.max(np.abs(got["cost"][ok] - ref["cost"][ok]) / np.abs(ref["cost"][ok])) < 1e-8
    dx = got["x"] - ref["x"]
    close = np.max(np.abs(dx) / width, axis=(1, 2)) < 1e-8
    if kind != "prosail":
        assert np.all(close[ok])
    else:
        # the flat-valley clause of test_invert: where the two step arithmetics stop at different points of a weakly
        # determined valley, the quadratic model's cost difference is within 1e-8 of the cost, for a minority of series
        flat = np.array([0.5 * dx[k].ravel() @ dense_hessian(ref["hess"][k], R, c) @ dx[k].ravel()
                         <= 1e-8 * abs(ref["cost"][k]) for k in range(S)])
        assert np.all((close | flat)[ok])
        assert np.sum(~close[ok]) <= S // 4


@pytest.mark.gpu
@pytest.mark.parametrize("spectra", [True, False])
def test_covariance_and_returned_values_have_the_stated_structure(gpemu, spectra):
    bank, rs = _bank(gpemu, 12, 5, W=300 if spectra else 0)
    S, T, D = 20, 8, 5
    x_true = _trajectory(rs, np.zeros(D), np.ones(D), S, T)
    obs = _own_obs(bank, spectra, x_true.reshape(-1, D))
    obs = (obs + 0.01 * rs.standard_normal(obs.shape)).reshape(S, T, -1)
    x0 = np.clip(x_true + 0.1 * rs.standard_normal(x_true.shape), 0, 1)
    R = _spd(rs, D, 20.0)
    c = rs.uniform(0.2, 2.0, T - 1)
    res = _series(bank, spectra, x0, obs, smooth_precision=R, coupling=c, lower=np.zeros(D), upper=np.ones(D),
                  want_cov=True)
    cov = res["cov"]
    assert np.array_equal(cov, cov.transpose(0, 1, 3, 2))
    n_pd = 0
    for s in range(S):
        H = dense_hessian(res["hess"][s], R, c)
        if not np.all(np.linalg.eigvalsh(H) > 0):
            assert np.all(np.isnan(cov[s]))
            continue
        n_pd += 1
        inv = np.linalg.inv(H)
        for t in range(T):
            blk = inv[t * D:(t + 1) * D, t * D:(t + 1) * D]
            assert np.max(np.abs(cov[s, t] - blk)) <= 1e-9 * np.abs(blk).max()
    assert n_pd >= S // 2
    # no prior: grad and hess are the cost call's at the returned x plus the coupling terms
    lib_ = _cost(bank, spectra, res["x"].reshape(-1, D), obs.reshape(S * T, -1), want_hess=True)
    g = lib_["grad"].reshape(S, T, D).copy()
    h = lib_["hess"].reshape(S, T, D, D).copy()
    for t in range(1, T):
        Re = (res["x"][:, t] - res["x"][:, t - 1]) @ R.T
        g[:, t] += c[t - 1] * Re
        g[:, t - 1] -= c[t - 1] * Re
        h[:, t] += c[t - 1] * R
        h[:, t - 1] += c[t - 1] * R
    ulp = 8 * np.finfo(float).eps
    assert np.max(np.abs(res["grad"] - g)) <= ulp * (np.abs(lib_["grad"]).max() + np.abs(g).max())
    assert np.max(np.abs(res["hess"] - h)) <= ulp * np.abs(h).max()
    f = lib_["cost"].reshape(S, T).sum(axis=1)
    for t in range(1, T):
        e = res["x"][:, t] - res["x"][:, t - 1]
        f = f + 0.5 * c[t - 1] * np.einsum("nd,de,ne->n", e, R, e)
    assert np.max(np.abs(res["cost"] - f) / np.abs(f)) < 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("spectra", [True, False])
def test_results_do_not_depend_on_chunking_placement_devices_or_order(lib, gpemu, monkeypatch, spectra):
    import torch
    E, W, D, S, T = 16, 257, 6, 300, 9
    bank, rs = _bank(gpemu, E, D, W=W if spectra else 0)
    x_true = _trajectory(rs, np.zeros(D), np.ones(D), S, T)
    obs = _own_obs(bank, spectra, x_true.reshape(-1, D))
    K = obs.shape[1]
    obs = (obs + 0.01 * rs.standard_normal(obs.shape)).reshape(S, T, K)
    w = np.tile(rs.uniform(0.5, 2.0, K), (S * T, 1))
    w[rs.random_sample(S * T) < 0.3] = 0.0
    w = w.reshape(S, T, K)
    x0 = np.clip(x_true + 0.1 * rs.standard_normal(x_true.shape), 0, 1)
    pm = rs.uniform(0, 1, (S, T, D))
    R, c = _spd(rs, D, 30.0), rs.uniform(0.2, 2.0, T - 1)
    kw = dict(smooth_precision=R, coupling=c, lower=np.zeros(D), upper=np.ones(D), prior_mean=pm,
              prior_precision=0.01 * np.eye(D), want_cov=True)
    keys = ("x", "cost", "grad", "hess", "cov", "status", "n_iter")
    ref = _series(bank, spectra, x0, obs, w, **kw)
    assert len(np.unique(ref["n_iter"])) > 1
    versions = {}
    monkeypatch.setenv("GPE_SLOT_OUT_BYTES", str(8 * T * (3 + 2 * D + 2 * D * D) * 37))     # chunks of about 37 series
    versions["chunks"] = _series(bank, spectra, x0, obs, w, **kw)
    monkeypatch.delenv("GPE_SLOT_OUT_BYTES")
    monkeypatch.setenv("GPE_SOLVE_SUB_POINTS", "23")                                     # solver sub-chunks of 23 series
    versions["sub"] = _series(bank, spectra, x0, obs, w, **kw)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    dev = _series(bank, spectra, t(x0), t(obs), t(w), **{k: (t(v) if isinstance(v, np.ndarray) else v) for k, v in kw.items()})
    versions["device+sub"] = {k: v.cpu().numpy() for k, v in dev.items()}
    monkeypatch.delenv("GPE_SOLVE_SUB_POINTS")
    dev = _series(bank, spectra, t(x0), t(obs), t(w), **{k: (t(v) if isinstance(v, np.ndarray) else v) for k, v in kw.items()})
    versions["device"] = {k: v.cpu().numpy() for k, v in dev.items()}
    inputs, thetas, invQts, invQs, rs2 = _models(E, D, 40, 0)
    B = rs2.standard_normal((E, W)) if spectra else None
    two = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=B, device=[0, 0] if lib.gpe_device_count() == 1 else "all")
    versions["devices"] = _series(two, spectra, x0, obs, w, **kw)
    perm = rs.permutation(S)
    got = _series(bank, spectra, x0[perm], obs[perm], w[perm], **dict(kw, prior_mean=pm[perm]))
    inv = np.argsort(perm)
    versions["permuted"] = {k: got[k][inv] for k in keys}
    for name, v in versions.items():
        for k in keys:
            assert np.array_equal(np.asarray(v[k]), np.asarray(ref[k]), equal_nan=True), (name, k)


@pytest.mark.gpu
def test_gap_filling_beats_per_date_inversion_on_masked_dates(gpemu):
    """Smooth x_true(t), per-row sigma, 40 % of the dates fully masked: every series converges, the truth lies within 6
    posterior sd on every date, and on the masked dates the series RMSE is at most a quarter of per-date invert's (which
    can only return its start there)."""
    bank, rs = _bank(gpemu, 24, 6)
    S, T, D = 64, 46, 6
    lo, hi = np.zeros(D), np.ones(D)
    x_true = _trajectory(rs, lo, hi, S, T)
    mu = _own_obs(bank, False, x_true.reshape(-1, D))
    sigma = 0.01 * np.abs(mu).mean(axis=0) * rs.uniform(0.5, 2.0, mu.shape)
    obs = mu + sigma * rs.standard_normal(mu.shape)
    w = 1.0 / sigma ** 2
    masked = rs.random_sample(S * T) < 0.4
    w[masked] = 0.0
    x0 = np.full((S, T, D), 0.5)
    step = 0.2 * 2 * np.pi / T                 # largest change of x_true between dates
    R = np.eye(D) / step ** 2
    E = mu.shape[1]
    res = bank.invert_series(x0, obs.reshape(S, T, E), w.reshape(S, T, E), smooth_precision=R, lower=lo, upper=hi,
                             max_iter=200, want_cov=True)
    assert np.all(res["status"] == CONVERGED), np.bincount(res["status"])
    sd = np.sqrt(np.einsum("stdd->std", res["cov"]))
    assert np.all(np.abs(res["x"] - x_true) <= 6 * sd)
    point = bank.invert(x0.reshape(-1, D), obs, w, lower=lo, upper=hi, max_iter=200)
    err_series = (res["x"].reshape(-1, D) - x_true.reshape(-1, D))[masked]
    err_point = (point["x"] - x_true.reshape(-1, D))[masked]
    rmse_s, rmse_p = np.sqrt(np.mean(err_series ** 2)), np.sqrt(np.mean(err_point ** 2))
    assert rmse_s <= 0.25 * rmse_p, (rmse_s, rmse_p)


@pytest.mark.gpu
def test_a_non_finite_start_stops_only_its_series(gpemu):
    bank, rs = _bank(gpemu, 12, 5)
    S, T, D = 6, 5, 5
    x_true = _trajectory(rs, np.zeros(D), np.ones(D), S, T)
    obs = _own_obs(bank, False, x_true.reshape(-1, D)).reshape(S, T, -1)
    x0 = x_true.copy()
    x0[2, 3, 1] = np.nan
    res = bank.invert_series(x0, obs, smooth_precision=np.eye(D))
    assert res["status"][2] == NONFINITE and res["n_iter"][2] == 0
    assert np.all(res["status"][np.arange(S) != 2] == CONVERGED)


@pytest.mark.gpu
def test_zero_coupling_leaves_every_date_at_its_own_optimum(gpemu):
    bank, rs = _bank(gpemu, 24, 6)
    S, T, D = 10, 6, 6
    x_true = _trajectory(rs, np.zeros(D), np.ones(D), S, T)
    obs = _own_obs(bank, False, x_true.reshape(-1, D))
    x0 = np.clip(x_true + 0.02 * rs.standard_normal(x_true.shape), 0, 1)
    kw = dict(lower=np.zeros(D), upper=np.ones(D), max_iter=100)
    res = bank.invert_series(x0, obs.reshape(S, T, -1), smooth_precision=_spd(rs, D, 50.0), coupling=np.zeros(T - 1), **kw)
    point = bank.invert(x0.reshape(-1, D), obs, **kw)
    ok = res["status"] == CONVERGED
    assert np.mean(ok) >= 0.8 and np.all(point["status"] == CONVERGED)
    assert np.max(np.abs(res["x"][ok] - point["x"].reshape(S, T, D)[ok])) < 1e-7


def _raw(lib, bank, S, T, x0, obs, obs_ld, R, c, x, cost, info, flags, opts=None, w=None, w_ld=0):
    return lib.gpe_bank_solve_series(bank._h, S, T, x0, obs, obs_ld, w, w_ld, opts, R, c, x, cost, None, None, None, info,
                                     flags, None)


@pytest.mark.gpu
def test_argument_errors(lib, gpemu):
    from gp_emulator_b200 import _lib
    bank, rs = _bank(gpemu, 6, 4)
    S, T, D, E = 3, 4, 4, 6
    H = _lib.HOST_PTRS
    x0, obs = rs.uniform(0, 1, (S * T, D)), rs.standard_normal((S * T, E))
    x, cost, info = np.empty((S * T, D)), np.empty(S), np.empty((S, 2), dtype=np.int32)
    R, c = np.eye(D), np.ones(T - 1)
    a = lambda v: None if v is None else v.ctypes.data

    def call(S=S, T=T, ld=E, R=R, c=c):
        return _raw(lib, bank, S, T, a(x0), a(obs), ld, a(R), a(c), a(x), a(cost), a(info), H)

    assert call() == 0
    assert call(ld=E - 1) != 0 and call(ld=E + 1) != 0
    assert call(R=None) != 0
    Ra = R.copy()
    Ra[0, 1] = 1e-3
    assert call(R=Ra) != 0
    Rn = R.copy()
    Rn[1, 1] = np.nan
    assert call(R=Rn) != 0
    for bad in (-1.0, np.nan, np.inf):
        cb = c.copy()
        cb[1] = bad
        assert call(c=cb) != 0
    assert call(T=0) != 0 and call(S=-1) != 0
    big, rs2 = _bank(gpemu, 2, 33)
    xb = np.zeros((2, 33))
    rc = _raw(lib, big, 1, 2, xb.ctypes.data, np.zeros(2).ctypes.data, 0, np.eye(33).ctypes.data, None, xb.ctypes.data,
              np.empty(1).ctypes.data, np.empty((1, 2), dtype=np.int32).ctypes.data, H)
    assert rc != 0 and "32" in lib.gpe_last_error().decode()


@pytest.mark.gpu
@pytest.mark.parametrize("spectra", [True, False])
def test_red_zones(lib, gpemu, spectra):
    import torch
    from gp_emulator_b200 import _lib
    E, W, D, S, T = 8, 129, 4, 33, 7
    bank, rs = _bank(gpemu, E, D, W=W if spectra else 0)
    K = W if spectra else E
    x_true = _trajectory(rs, np.zeros(D), np.ones(D), S, T)
    obs = _own_obs(bank, spectra, x_true.reshape(-1, D))
    x0 = np.clip(x_true.reshape(-1, D) + 0.05 * rs.standard_normal((S * T, D)), 0, 1)
    R, c = np.eye(D) * 10.0, rs.uniform(0.5, 1.5, T - 1)
    lo, hi = np.zeros(D), np.ones(D)
    opts = _lib.SolveOpts(50, 1e-10, 1e-10, 0.0, 1e-3, lo.ctypes.data, hi.ctypes.data, None, 0, None)
    pad = 64
    sizes = {"x": S * T * D, "cost": S, "grad": S * T * D, "hess": S * T * D * D, "cov": S * T * D * D, "info": S}
    flags = _lib.SOLVE_SPECTRA if spectra else 0
    for device in (False, True):
        bufs = {k: np.full(n + 2 * pad, 7.25) for k, n in sizes.items()}
        if device:
            t = lambda v: torch.from_numpy(np.ascontiguousarray(v)).cuda()
            dbufs = {k: t(v) for k, v in bufs.items()}
            ptr = lambda k: dbufs[k].data_ptr() + 8 * pad
            args = [t(x0), t(obs), t(R), t(c), t(lo), t(hi)]
            dopts = _lib.SolveOpts(50, 1e-10, 1e-10, 0.0, 1e-3, args[4].data_ptr(), args[5].data_ptr(), None, 0, None)
            rc = lib.gpe_bank_solve_series(bank._h, S, T, args[0].data_ptr(), args[1].data_ptr(), K, None, 0, C.byref(dopts),
                                           args[2].data_ptr(), args[3].data_ptr(), ptr("x"), ptr("cost"), ptr("grad"),
                                           ptr("hess"), ptr("cov"), ptr("info"), flags, None)
            torch.cuda.synchronize()
            bufs = {k: v.cpu().numpy() for k, v in dbufs.items()}
        else:
            ptr = lambda k: bufs[k].ctypes.data + 8 * pad
            rc = lib.gpe_bank_solve_series(bank._h, S, T, x0.ctypes.data, obs.ctypes.data, K, None, 0, C.byref(opts),
                                           R.ctypes.data, c.ctypes.data, ptr("x"), ptr("cost"), ptr("grad"), ptr("hess"),
                                           ptr("cov"), ptr("info"), flags | _lib.HOST_PTRS, None)
        assert rc == 0, lib.gpe_last_error()
        for k, v in bufs.items():
            assert np.all(v[:pad] == 7.25) and np.all(v[pad + sizes[k]:] == 7.25), (device, k)
            assert not np.any(v[pad:pad + sizes[k]] == 7.25), (device, k)


@pytest.mark.gpu
def test_multivariate_emulator_invert_series(gpemu):
    mv, g = _prosail(gpemu)
    lo, hi = g["y"].min(axis=0), g["y"].max(axis=0)
    rs = np.random.RandomState(4)
    S, T, D = 4, 6, 10
    x_true = _trajectory(rs, lo, hi, S, T)
    obs = mv.predict(x_true.reshape(-1, D), do_deriv=False).reshape(S, T, -1)
    R = np.diag(1.0 / (0.1 * (hi - lo)) ** 2)
    y0 = np.clip(x_true + 0.02 * (hi - lo) * rs.standard_normal(x_true.shape), lo, hi)
    res = mv.invert_series(obs, y0, smooth=(R, None), bounds=(lo, hi), max_iter=100)
    bank = mv._device_bank()
    ref = bank.forward_invert_series(y0, obs, smooth_precision=R, lower=lo, upper=hi, max_iter=100, want_cov=True)
    for k in ("x", "cost", "cov", "status"):
        assert np.array_equal(res[k], ref[k], equal_nan=True), k
    one = mv.invert_series(obs[1], y0[1], smooth=(R, np.ones(T - 1)), bounds=(lo, hi), max_iter=100)
    assert one["x"].shape == (T, D) and np.array_equal(one["x"], ref["x"][1])
    with pytest.raises(ValueError):
        mv.invert_series(obs, None, smooth=(R, None))
