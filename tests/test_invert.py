"""Inversion on the device: gpe_bank_solve / gpe_multi_bank_solve, DeviceBank.invert / forward_invert and
MultivariateEmulator.invert (bounded Levenberg-Marquardt on the exact cost Hessian, DESIGN 4.6d).

``lm_ref`` restates the algorithm of include/gpemu.h step for step in numpy, with any batch evaluator of f, g, H.  On the
CPU it is checked against analytic optima; on the GPU it drives the library's own cost calls and the device solver must
land where it lands."""
import os
import re

import numpy as np
import pytest
import scipy.linalg

from tests.conftest import ROOT, golden

CONVERGED, MAX_ITER, STALLED, NONFINITE = 0, 1, 2, 3


def lm_ref(fgh, x0, lower=None, upper=None, prior_mean=None, prior_prec=None, max_iter=50, ftol=1e-10, xtol=1e-10,
           gtol=0.0, lambda0=1e-3, indexed=False):
    """The algorithm of include/gpemu.h.  fgh(X (n, D)) -> f (n,), g (n, D), H (n, D, D) without the prior; with
    ``indexed`` fgh(X, idx) is also told which points (rows of x0) it evaluates."""
    x0 = np.asarray(x0, dtype=np.float64)
    N, D = x0.shape
    lo = np.full(D, -np.inf) if lower is None else np.asarray(lower, dtype=np.float64)
    hi = np.full(D, np.inf) if upper is None else np.asarray(upper, dtype=np.float64)
    m = np.zeros((N, D)) if prior_mean is None else np.broadcast_to(np.asarray(prior_mean, dtype=np.float64), (N, D))

    def evaluate(X, idx):
        f, g, H = (np.array(a, dtype=np.float64) for a in (fgh(X, idx) if indexed else fgh(X)))
        if prior_prec is not None:
            r = X - m[idx]
            pr = r @ np.asarray(prior_prec).T
            f = f + 0.5 * np.sum(r * pr, axis=1)
            g = g + pr
            H = H + prior_prec
        return f, g, H

    x = np.clip(x0, lo, hi)
    f, g, H = evaluate(x, np.arange(N))
    lam, nu = np.full(N, float(lambda0)), np.full(N, 2.0)
    nev, status = np.zeros(N, dtype=np.int64), np.full(N, -1)
    pred, xt = np.zeros(N), x.copy()
    status[~np.isfinite(f)] = NONFINITE

    def propose(k):
        free = ~(((x[k] <= lo) & (g[k] > 0)) | ((x[k] >= hi) & (g[k] < 0)))
        if np.max(np.abs(g[k][free]), initial=0.0) <= gtol:
            return CONVERGED
        F = np.flatnonzero(free)
        HF = H[k][np.ix_(F, F)]
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
        step = np.zeros(D)
        step[F] = scipy.linalg.cho_solve((L, True), -g[k][F])
        t = np.clip(x[k] + step, lo, hi)
        d = t - x[k]
        if np.max(np.abs(d)) <= xtol * (np.max(np.abs(x[k])) + xtol):
            return CONVERGED
        if nev[k] >= max_iter:
            return MAX_ITER
        pred[k] = -(g[k] @ d + 0.5 * d @ H[k] @ d)
        xt[k] = t
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
    return {"x": x, "cost": f, "grad": g, "hess": H, "status": status, "n_iter": nev}


def _projected_grad(x, g, lo, hi):
    out = g.copy()
    out[((x <= lo) & (g > 0)) | ((x >= hi) & (g < 0))] = 0.0
    return out


# ---- CPU: the reference on analytic problems ----------------------------------------------------------------------
def _quadratic(A, c):
    def fgh(X):
        r = X - c
        Ar = r @ A.T
        return 0.5 * np.sum(r * Ar, axis=1), Ar, np.broadcast_to(A, (len(X),) + A.shape).copy()
    return fgh


def test_reference_finds_the_minimiser_of_a_quadratic_inside_and_on_the_box():
    rs = np.random.RandomState(0)
    D = 5
    Q = rs.standard_normal((D, D))
    A = Q @ Q.T + 0.5 * np.eye(D)
    c = rs.uniform(-1, 1, (1, D))
    lo, hi = np.full(D, -2.0), np.full(D, 2.0)
    res = lm_ref(_quadratic(A, c), rs.uniform(-2, 2, (8, D)), lo, hi)
    assert np.all(res["status"] == CONVERGED)
    assert np.max(np.abs(res["x"] - c)) < 1e-9
    lo2, hi2 = np.full(D, -0.3), np.full(D, 0.3)               # box cuts the unconstrained minimiser off
    c2 = np.array([[1.0, -1.0, 0.1, 0.5, -0.2]])
    res = lm_ref(_quadratic(A, c2), rs.uniform(-0.3, 0.3, (8, D)), lo2, hi2)
    assert np.all(res["status"] == CONVERGED)
    for k in range(8):
        x, g = res["x"][k], res["grad"][k]
        assert np.all((x >= lo2) & (x <= hi2))
        assert np.max(np.abs(_projected_grad(x, g, lo2, hi2))) < 1e-8
        assert np.all(g[x <= lo2] >= 0) and np.all(g[x >= hi2] <= 0)
        assert np.any(x <= lo2) or np.any(x >= hi2)
    assert np.max(np.abs(res["x"] - res["x"][0])) < 1e-9      # one minimiser for every start


def _rosenbrock(X):
    x1, x2 = X[:, 0], X[:, 1]
    r = np.stack([10 * (x2 - x1 ** 2), 1 - x1], axis=1)
    J = np.zeros((len(X), 2, 2))
    J[:, 0, 0], J[:, 0, 1], J[:, 1, 0] = -20 * x1, 10.0, -1.0
    H = np.einsum("nik,nil->nkl", J, J)
    H[:, 0, 0] += r[:, 0] * -20.0
    return 0.5 * np.sum(r * r, axis=1), np.einsum("nik,ni->nk", J, r), H


def test_reference_solves_a_bounded_rosenbrock_least_squares_problem():
    x0 = np.array([[-1.2, 1.0], [0.0, 0.0], [-1.5, 2.0], [0.4, -0.5]])
    res = lm_ref(_rosenbrock, x0, max_iter=200)
    assert np.all(res["status"] == CONVERGED) and np.max(np.abs(res["x"] - 1.0)) < 1e-8
    lo, hi = np.array([-2.0, -1.0]), np.array([0.5, 2.0])
    res = lm_ref(_rosenbrock, x0, lo, hi, max_iter=200)     # the minimiser is cut off at x1 = 0.5: (0.5, 0.25)
    assert np.all(res["status"] == CONVERGED)
    assert np.max(np.abs(res["x"] - [0.5, 0.25])) < 1e-8
    assert np.all(res["grad"][:, 0] <= 0)


def test_reference_reaches_the_posterior_mode_of_a_linear_gaussian_problem():
    rs = np.random.RandomState(2)
    D, E, N = 4, 6, 5
    A = rs.standard_normal((E, D))
    w = rs.uniform(0.5, 2.0, E)
    y = rs.standard_normal((N, E))
    P = np.diag(rs.uniform(0.5, 3.0, D))
    m = rs.standard_normal((N, D))

    cur = [0]

    def fgh(X):       # one point per call: its own observation row
        r = X @ A.T - y[cur[0]]
        return 0.5 * np.sum(w * r * r, axis=1), (w * r) @ A, np.broadcast_to(A.T @ (w[:, None] * A), (len(X), D, D)).copy()

    # closed form: (A^T W A + P) x = A^T W y + P m
    mode = np.linalg.solve(A.T @ (w[:, None] * A) + P, ((w * y) @ A + m @ P).T).T
    for k in range(N):        # one point per call keeps the observation row aligned with the evaluation
        cur[0] = k
        res = lm_ref(fgh, rs.standard_normal((1, D)), prior_mean=m[k], prior_prec=P)
        assert res["status"][0] == CONVERGED
        assert np.max(np.abs(res["x"][0] - mode[k])) < 1e-9
        assert np.max(np.abs(res["grad"][0])) < 1e-7


def test_solve_constants_mirror_the_header():
    from gp_emulator_b200 import _lib
    text = open(os.path.join(ROOT, "include", "gpemu.h")).read()
    defs = {k: int(v, 0) for k, v in re.findall(r"#define\s+(GPE_[A-Z0-9_]+)\s+(0x[0-9a-fA-F]+|\d+)", text)}
    for cname, pyname in [("GPE_SOLVE_SPECTRA", "SOLVE_SPECTRA"), ("GPE_SOLVE_MAX_D", "SOLVE_MAX_D"),
                          ("GPE_SOLVE_CONVERGED", "SOLVE_CONVERGED"), ("GPE_SOLVE_MAX_ITER", "SOLVE_MAX_ITER"),
                          ("GPE_SOLVE_STALLED", "SOLVE_STALLED"), ("GPE_SOLVE_NONFINITE", "SOLVE_NONFINITE"),
                          ("GPE_SOLVE_DEFAULT_MAX_ITER", "SOLVE_DEFAULT_MAX_ITER")]:
        assert defs[cname] == getattr(_lib, pyname), cname
    assert (CONVERGED, MAX_ITER, STALLED, NONFINITE) == (_lib.SOLVE_CONVERGED, _lib.SOLVE_MAX_ITER, _lib.SOLVE_STALLED,
                                                         _lib.SOLVE_NONFINITE)
    names = [f[0] for f in _lib.SolveOpts._fields_]
    assert names == ["max_iter", "ftol", "xtol", "gtol", "lambda0", "lower", "upper", "prior_mean", "prior_ld", "prior_prec"]


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpemu(lib):
    import gp_emulator_b200 as g
    assert lib.gpe_device_count() > 0, "no GPU visible: the gpu tests must not pass on a fallback"
    return g


def _models(E, D, M, seed):
    rs = np.random.RandomState(seed + 11 * E + 3 * D + M)
    inputs = rs.random_sample((M, D))
    thetas = np.log(rs.uniform(0.5, 3.0, (E, D + 2)))
    invQts = rs.standard_normal((E, M))
    invQs = rs.random_sample((E, M, M))
    return inputs, thetas, invQts, invQs, rs


def _bank(gpemu, E, D, M=40, W=0, seed=0, device=0):
    inputs, thetas, invQts, invQs, rs = _models(E, D, M, seed)
    B = rs.standard_normal((E, W)) if W else None
    return gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=B, device=device), rs


def _prosail(gpemu):
    from tests.test_gpu_parity import _write_prosail_dump
    g = golden("P")
    mv = gpemu.MultivariateEmulator(X=None, y=None, dump=_write_prosail_dump(g))
    return mv, g


def _problem(gpemu, kind):
    """(bank, spectra, lo, hi, rs) of a test problem: the synthetic config-4 bank, the PROSAIL golden model or a band bank."""
    if kind == "fwd":
        bank, rs = _bank(gpemu, 20, 10, W=2101)
        return bank, True, np.zeros(10), np.ones(10), rs
    if kind == "prosail":
        mv, g = _prosail(gpemu)
        return mv._device_bank(), True, g["y"].min(axis=0), g["y"].max(axis=0), np.random.RandomState(5)
    bank, rs = _bank(gpemu, 24, 6)
    return bank, False, np.zeros(6), np.ones(6), rs


def _own_obs(bank, spectra, x):
    if spectra:
        return bank.predict(x, want_var=False, want_deriv=False, want_mu=False, project=True)["fwd"]
    return bank.predict(x, want_var=False, want_deriv=False)["mu"]


def _solve(bank, spectra, *a, **k):
    return (bank.forward_invert if spectra else bank.invert)(*a, **k)


def _cost(bank, spectra, *a, **k):
    return (bank.forward_cost if spectra else bank.cost)(*a, **k)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fwd", "prosail", "band"])
def test_recovery_of_the_inputs_behind_the_library_own_outputs(gpemu, kind):
    bank, spectra, lo, hi, rs = _problem(gpemu, kind)
    N = 200
    width = hi - lo
    x_true = lo + width * rs.uniform(0.2, 0.8, (N, len(lo)))
    x0 = np.clip(x_true + 0.02 * width * rs.standard_normal(x_true.shape), lo, hi)
    obs = _own_obs(bank, spectra, x_true)
    res = _solve(bank, spectra, x0, obs, lower=lo, upper=hi, max_iter=100)
    assert np.all(res["status"] == CONVERGED), np.bincount(res["status"])
    assert np.max(np.abs(res["x"] - x_true) / width) <= 1e-8


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fwd", "prosail", "band"])
def test_agreement_with_the_reference_driving_the_library_costs(gpemu, kind):
    bank, spectra, lo, hi, rs = _problem(gpemu, kind)
    N = 60
    width = hi - lo
    x_true = lo + width * rs.uniform(0.1, 0.9, (N, len(lo)))
    obs = _own_obs(bank, spectra, x_true)
    obs = obs * (1.0 + 0.01 * rs.standard_normal(obs.shape))
    w = rs.uniform(0.5, 2.0, obs.shape[1])
    x0 = np.clip(x_true + 0.05 * width * rs.standard_normal(x_true.shape), lo, hi)

    def fgh(X, idx):
        # every evaluation covers all N rows, as the solver's do (call_N = N): the same kernel plans, so the reference
        # sees bit for bit the solver's values and the comparison isolates the step arithmetic
        rows = x0.copy()
        rows[idx] = X
        out = _cost(bank, spectra, rows, obs, w, want_hess=True)
        return out["cost"][idx], out["grad"][idx], out["hess"][idx]

    ref = lm_ref(fgh, x0, lo, hi, max_iter=100, indexed=True)
    got = _solve(bank, spectra, x0, obs, w, lower=lo, upper=hi, max_iter=100)
    ref_x, ref_c, ref_s = ref["x"], ref["cost"], ref["status"]
    assert np.array_equal(got["status"], ref_s)
    ok = ref_s == CONVERGED
    assert np.max(np.abs(got["cost"][ok] - ref_c[ok]) / np.maximum(np.abs(ref_c[ok]), 1e-300)) < 1e-8
    dx = got["x"] - ref_x
    close = np.max(np.abs(dx) / width, axis=1) < 1e-8
    if kind != "prosail":
        assert np.all(close[ok])                             # x to 1e-8 of the box
    else:
        # The PROSAIL model has weakly determined directions: there the two step arithmetics (warp Cholesky, LAPACK) may
        # stop at different points of a flat valley (up to 1.8e-5 of the box on one input).  Such points must agree as
        # closely as the cost resolves -- the quadratic model's cost difference between the two end points within 1e-8
        # of the cost -- and stay a minority (7 of these 60 points).
        flat = 0.5 * np.einsum("nd,nde,ne->n", dx, ref["hess"], dx) <= 1e-8 * np.abs(ref_c)
        assert np.all((close | flat)[ok])
        assert np.sum(~close[ok]) <= len(close) // 4


@pytest.mark.gpu
def test_cost_is_no_worse_than_scipy_lbfgsb(gpemu):
    from scipy.optimize import minimize
    mv, g = _prosail(gpemu)
    lo, hi = g["y"].min(axis=0), g["y"].max(axis=0)
    rs = np.random.RandomState(9)
    N = 24
    x_true = lo + (hi - lo) * rs.uniform(0.1, 0.9, (N, 10))
    obs = mv.predict(x_true, do_deriv=False) * (1.0 + 0.02 * rs.standard_normal((N, 2101)))
    x0 = lo + (hi - lo) * rs.uniform(0.3, 0.7, (N, 10))
    got = mv.invert(obs, x0, bounds=(lo, hi), max_iter=200)
    for k in range(N):
        sp = minimize(lambda y: mv.cost(y, obs[k]), x0[k], jac=True, method="L-BFGS-B", bounds=list(zip(lo, hi)),
                      options={"maxiter": 2000, "ftol": 1e-15, "gtol": 1e-12})
        if got["status"][k] == CONVERGED:
            assert got["cost"][k] <= sp.fun * (1 + 1e-9) + 1e-300, (k, got["cost"][k], sp.fun)
            pg = _projected_grad(got["x"][k], got["grad"][k], lo, hi)
            assert np.max(np.abs(pg)) <= 1e-6 * max(1.0, np.max(np.abs(got["grad"][k])), abs(got["cost"][k]))
    assert np.mean(got["status"] == CONVERGED) >= 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("spectra", [True, False])
def test_returned_values_are_the_library_values(gpemu, spectra):
    bank, rs = _bank(gpemu, 12, 5, W=300 if spectra else 0)
    N, D = 150, 5
    x_true = rs.uniform(0.2, 0.8, (N, D))
    obs = _own_obs(bank, spectra, x_true)
    obs = obs + 0.01 * rs.standard_normal(obs.shape)
    x0 = np.clip(x_true + 0.1 * rs.standard_normal((N, D)), 0, 1)
    res = _solve(bank, spectra, x0, obs, lower=np.zeros(D), upper=np.ones(D), want_cov=True)
    again = _cost(bank, spectra, res["x"], obs, want_hess=True)
    for k in ("cost", "grad", "hess"):
        assert np.array_equal(res[k], again[k]), k
    cov = res["cov"]
    assert np.array_equal(cov, cov.transpose(0, 2, 1))
    pd = np.all(np.linalg.eigvalsh(res["hess"]) > 0, axis=1)
    assert np.all(np.isnan(cov[~pd]))
    inv = np.linalg.inv(res["hess"][pd])
    assert np.max(np.abs(cov[pd] - inv) / np.abs(inv).max(axis=(1, 2), keepdims=True)) < 1e-10
    # with a prior the outputs differ from the library's by exactly the prior terms
    P = np.diag(rs.uniform(1.0, 5.0, D)) + 0.1
    m = rs.uniform(0, 1, (N, D))
    res = _solve(bank, spectra, x0, obs, lower=np.zeros(D), upper=np.ones(D), prior_mean=m, prior_precision=P)
    lib_ = _cost(bank, spectra, res["x"], obs, want_hess=True)
    r = res["x"] - m
    scale = np.abs(lib_["cost"]) + 0.5 * np.abs(np.einsum("nd,de,ne->n", r, P, r))
    assert np.all(np.abs(res["cost"] - lib_["cost"] - 0.5 * np.einsum("nd,de,ne->n", r, P, r)) <= 1e-14 * scale)
    assert np.max(np.abs(res["grad"] - lib_["grad"] - r @ P.T)) <= 1e-14 * np.abs(res["grad"]).max() + 1e-300
    assert np.max(np.abs(res["hess"] - lib_["hess"] - P)) <= 1e-14 * np.abs(res["hess"]).max()


@pytest.mark.gpu
@pytest.mark.parametrize("spectra", [True, False])
def test_results_do_not_depend_on_placement_chunking_devices_or_order(lib, gpemu, monkeypatch, spectra):
    import torch
    E, W, D, N = 16, 257, 6, 3000
    bank, rs = _bank(gpemu, E, D, W=W if spectra else 0)
    x_true = rs.uniform(0.1, 0.9, (N, D))
    obs = _own_obs(bank, spectra, x_true)
    obs = obs + 0.01 * rs.standard_normal(obs.shape)
    x0 = np.clip(x_true + 0.1 * rs.standard_normal((N, D)), 0, 1)
    w = rs.uniform(0.5, 2.0, obs.shape[1])
    pm = rs.uniform(0, 1, (N, D))
    P = 0.01 * np.eye(D)
    kw = dict(lower=np.zeros(D), upper=np.ones(D), prior_mean=pm, prior_precision=P, want_cov=True)
    keys = ("x", "cost", "grad", "hess", "cov", "status", "n_iter")
    ref = _solve(bank, spectra, x0, obs, w, **kw)
    assert len(np.unique(ref["n_iter"])) > 1             # points leave the active list at different iterations
    versions = {}
    monkeypatch.setenv("GPE_SLOT_OUT_BYTES", str(8 * (3 + 2 * D + 2 * D * D) * 97))     # chunks of 97 points
    versions["chunks"] = _solve(bank, spectra, x0, obs, w, **kw)
    monkeypatch.delenv("GPE_SLOT_OUT_BYTES")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    dev = _solve(bank, spectra, t(x0), t(obs), t(w), lower=t(np.zeros(D)), upper=t(np.ones(D)), prior_mean=t(pm),
                 prior_precision=t(P), want_cov=True)
    versions["device"] = {k: v.cpu().numpy() for k, v in dev.items()}
    inputs, thetas, invQts, invQs, rs2 = _models(E, D, 40, 0)
    B = rs2.standard_normal((E, W)) if spectra else None
    two = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=B, device=[0, 0] if lib.gpe_device_count() == 1 else "all")
    versions["devices"] = _solve(two, spectra, x0, obs, w, **kw)
    perm = rs.permutation(N)
    kwp = dict(kw, prior_mean=pm[perm])
    got = _solve(bank, spectra, x0[perm], obs[perm], w, **kwp)
    inv = np.argsort(perm)
    versions["permuted"] = {k: got[k][inv] for k in keys}
    for name, v in versions.items():
        for k in keys:
            a, b = np.asarray(v[k]), np.asarray(ref[k])
            assert np.array_equal(a, b, equal_nan=True), (name, k)


@pytest.mark.gpu
@pytest.mark.parametrize("spectra", [True, False])
def test_sub_chunks_of_the_solver_scratch_are_invisible(gpemu, monkeypatch, spectra):
    """A call longer than the solver's scratch is solved in sub-chunks (offsets into x0, obs, the prior means and every
    output): forced down to 97 points, host and device pointers give what one sub-chunk gives."""
    import torch
    E, W, D, N = 12, 129, 5, 1000
    bank, rs = _bank(gpemu, E, D, W=W if spectra else 0)
    x_true = rs.uniform(0.1, 0.9, (N, D))
    obs = _own_obs(bank, spectra, x_true)
    obs = obs + 0.01 * rs.standard_normal(obs.shape)
    x0 = np.clip(x_true + 0.1 * rs.standard_normal((N, D)), 0, 1)
    pm = rs.uniform(0, 1, (N, D))
    kw = dict(lower=np.zeros(D), upper=np.ones(D), prior_mean=pm, prior_precision=0.01 * np.eye(D), want_cov=True)
    keys = ("x", "cost", "grad", "hess", "cov", "status", "n_iter")
    ref = _solve(bank, spectra, x0, obs, **kw)
    monkeypatch.setenv("GPE_SOLVE_SUB_POINTS", "97")
    host = _solve(bank, spectra, x0, obs, **kw)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    dev = _solve(bank, spectra, t(x0), t(obs), **{k: (t(v) if isinstance(v, np.ndarray) else v) for k, v in kw.items()})
    dev = {k: v.cpu().numpy() for k, v in dev.items()}
    for name, v in (("host", host), ("device", dev)):
        for k in keys:
            assert np.array_equal(np.asarray(v[k]), np.asarray(ref[k]), equal_nan=True), (name, k)


@pytest.mark.gpu
def test_bounds_statuses_and_one_point_api(gpemu):
    mv, g = _prosail(gpemu)
    bank = mv._device_bank()
    lo, hi = g["y"].min(axis=0), g["y"].max(axis=0)
    rs = np.random.RandomState(3)
    N, D = 40, 10
    x_true = lo + (hi - lo) * rs.uniform(0.2, 0.8, (N, D))
    x_true[:, 2] = hi[2] + 0.3 * (hi[2] - lo[2])               # outside the box on one input
    obs = mv.predict(x_true, do_deriv=False)
    box_lo, box_hi = lo.copy(), hi.copy()
    x0 = lo + (hi - lo) * rs.uniform(0.3, 0.7, (N, D))
    res = mv.invert(obs, x0, bounds=(box_lo, box_hi), max_iter=100)
    assert np.all((res["x"] >= box_lo) & (res["x"] <= box_hi))
    on = res["x"][:, 2] >= box_hi[2]
    assert np.mean(on) > 0.5
    assert np.all(res["grad"][on, 2] <= 0)                     # outward gradient at the active bound
    # NaN observation: nonfinite, returned at x0
    bad = obs[:3].copy()
    bad[1, 17] = np.nan
    r = mv.invert(bad, x0[:3], bounds=(lo, hi))
    assert r["status"][1] == NONFINITE and np.array_equal(r["x"][1], x0[1]) and r["n_iter"][1] == 0
    assert r["status"][0] != NONFINITE
    for it in (0, 1):
        r = bank.forward_invert(x0[:5], obs[:5], lower=lo, upper=hi, max_iter=it)
        assert np.all(r["status"] == MAX_ITER) and np.all(r["n_iter"] == it)
    one = mv.invert(obs[0], x0[0], bounds=(lo, hi))
    assert one["x"].shape == (D,) and isinstance(one["cost"], float) and one["grad"].shape == (D,)
    assert one["hess"].shape == (D, D) and one["cov"].shape == (D, D) and isinstance(one["status"], int)
    many = mv.invert(obs[:4], x0[:4], bounds=(lo, hi))
    assert many["x"].shape == (4, D) and many["cov"].shape == (4, D, D) and many["status"].shape == (4,)
    assert np.array_equal(one["x"], many["x"][0])


@pytest.mark.gpu
@pytest.mark.parametrize("spectra", [True, False])
def test_red_zones(lib, gpemu, spectra):
    """x, hess, cov and info between guard bands, device and host pointers: bands untouched, every element written."""
    import ctypes as C
    import torch
    from gp_emulator_b200 import _lib
    E, W, D, N = 10, 129, 4, 37
    bank, rs = _bank(gpemu, E, D, W=W if spectra else 0)
    x_true = rs.uniform(0.2, 0.8, (N, D))
    obs = _own_obs(bank, spectra, x_true)
    x0 = np.clip(x_true + 0.05 * rs.standard_normal((N, D)), 0, 1)
    ref = _solve(bank, spectra, x0, obs, want_cov=True)
    flags = _lib.SOLVE_SPECTRA if spectra else 0
    gb = 512
    sizes = {"x": N * D, "hess": N * D * D, "cov": N * D * D}
    for host in (False, True):
        opts = _lib.SolveOpts(50, 1e-10, 1e-10, 0.0, 1e-3, None, None, None, 0, None)
        if host:
            bufs = {k: np.full(n + 2 * gb, np.nan) for k, n in sizes.items()}
            info = np.full(2 * N + 2 * gb, -7, dtype=np.int32)
            p = lambda a: a.ctypes.data + a.itemsize * gb
            rc = lib.gpe_bank_solve(bank._h, x0.ctypes.data, N, obs.ctypes.data, obs.shape[1], None, C.byref(opts),
                                    p(bufs["x"]), None, None, p(bufs["hess"]), p(bufs["cov"]), p(info), flags | _lib.HOST_PTRS, None)
        else:
            bufs = {k: torch.full((n + 2 * gb,), float("nan"), dtype=torch.float64, device="cuda") for k, n in sizes.items()}
            info = torch.full((2 * N + 2 * gb,), -7, dtype=torch.int32, device="cuda")
            p = lambda a: a.data_ptr() + a.element_size() * gb
            xd, od = torch.from_numpy(x0).cuda(), torch.from_numpy(obs).cuda()
            rc = lib.gpe_bank_solve(bank._h, xd.data_ptr(), N, od.data_ptr(), obs.shape[1], None, C.byref(opts),
                                    p(bufs["x"]), None, None, p(bufs["hess"]), p(bufs["cov"]), p(info), flags, None)
            bufs = {k: v.cpu().numpy() for k, v in bufs.items()}
            info = info.cpu().numpy()
        assert rc == 0
        for k, n in sizes.items():
            b = bufs[k]
            assert np.all(np.isnan(b[:gb])) and np.all(np.isnan(b[gb + n:])), k
            assert np.array_equal(b[gb:gb + n], ref[k].ravel(), equal_nan=True), k
        assert np.all(info[:gb] == -7) and np.all(info[gb + 2 * N:] == -7)
        assert np.array_equal(info[gb:gb + 2 * N].reshape(N, 2), np.stack([ref["status"], ref["n_iter"]], axis=1))


@pytest.mark.gpu
def test_argument_errors(lib, gpemu):
    import ctypes as C
    from gp_emulator_b200 import _lib
    E, W, D, N = 5, 9, 3, 4
    bank, rs = _bank(gpemu, E, D, W=W)
    nob, _ = _bank(gpemu, E, D)
    x0 = rs.random_sample((N, D)); obs = rs.standard_normal((N, W)); obsE = rs.standard_normal((N, E))
    x = np.empty((N, D)); info = np.empty((N, 2), dtype=np.int32)
    a = lambda v: None if v is None else v.ctypes.data
    H, S = _lib.HOST_PTRS, _lib.SOLVE_SPECTRA

    def call(h=bank._h, n=N, o=obs, ld=W, opts=None, xo=x, inf=info, flags=H | S, x0_=x0):
        return lib.gpe_bank_solve(h, a(x0_), n, a(o), ld, None, C.byref(opts) if opts is not None else None, a(xo), None,
                                  None, None, None, a(inf), flags, None)

    def opts(**k):
        base = dict(max_iter=10, ftol=1e-10, xtol=1e-10, gtol=0.0, lambda0=1e-3, lower=None, upper=None, prior_mean=None,
                    prior_ld=0, prior_prec=None)
        base.update(k)
        return _lib.SolveOpts(**base)
    assert call() == 0
    assert call(h=None) == -1                                         # NULL handle
    assert call(n=-1) == -1
    assert call(xo=None) == -1 and call(inf=None) == -1 and call(x0_=None) == -1 and call(o=None) == -1
    assert call(opts=opts(max_iter=-1)) == -1
    assert call(opts=opts(lambda0=0.0)) == -1 and call(opts=opts(ftol=float("nan"))) == -1
    lo, hi = np.full(D, 0.6), np.full(D, 0.4)
    assert call(opts=opts(lower=a(lo), upper=a(hi))) == -1          # lower > upper
    assert call(opts=opts(lower=a(hi), upper=a(lo))) == 0
    assert call(h=nob._h) == -1                                       # spectra without a basis
    assert call(ld=W + 1) == -1 and call(o=obsE, ld=E, flags=H) == 0 and call(o=obsE, ld=E + 1, flags=H) == -1
    pm = np.zeros((N, D)); P = np.eye(D)
    assert call(opts=opts(prior_mean=a(pm), prior_ld=D)) == -1       # a prior mean without a precision
    assert call(opts=opts(prior_mean=a(pm), prior_ld=D + 1, prior_prec=a(P))) == -1   # host rows must be D apart
    assert call(opts=opts(prior_mean=a(pm), prior_ld=D, prior_prec=a(P))) == 0
    assert call(flags=H | S | 0x4000) == -1                           # unknown flag
    assert lib.gpe_multi_bank_solve(None, a(x0), N, a(obs), W, None, None, a(x), None, None, None, None, a(info), S) == -1
    wide, _ = _bank(gpemu, 3, 33, M=6)                                # D > 32
    xw = rs.random_sample((2, 33)); xwo = np.empty((2, 33)); iw = np.empty((2, 2), dtype=np.int32)
    assert lib.gpe_bank_solve(wide._h, a(xw), 2, a(np.zeros(3)), 0, None, None, a(xwo), None, None, None, None, a(iw), H,
                              None) == -4
    big, _ = _bank(gpemu, 97, 2, M=6, W=8)                            # beyond the forward cost's 96 emulators
    xb = rs.random_sample((2, 2)); xbo = np.empty((2, 2)); ib = np.empty((2, 2), dtype=np.int32)
    assert lib.gpe_bank_solve(big._h, a(xb), 2, a(np.zeros(8)), 0, None, None, a(xbo), None, None, None, None, a(ib), H | S,
                              None) == -4
    with pytest.raises(ValueError):
        bank.forward_invert(x0, obs, lower=np.zeros(D + 1))
    with pytest.raises(gpemu.GpemuError):
        nob.forward_invert(x0, obs)
