"""CPU oracle for the GP prediction hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A numpy/scipy restatement (Python 3) of the reference's prediction arithmetic.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference`` legs may import this
module; nothing under ``gp_emulator_b200/`` does, and the product path raises if its CUDA library is
missing instead of falling back to this file.

Parity pinning: the reference package is Python-2 only (print statements, xrange, tab/space mixing,
``import _gpu_predict`` at module scope), so it cannot be imported as-is.  ``tests/golden/make_golden.py``
loads the reference *source text* from a checkout of it at generation time, applies a purely mechanical
py2->py3 token conversion in memory, executes it, and freezes its outputs into ``tests/golden/*.npz``.
``tests/test_oracle.py`` checks every function below against those frozen reference outputs, so this
oracle is pinned to outputs of the reference itself.

Each function cites the reference file:line it follows (paths relative to the reference checkout).
"""
from __future__ import annotations

import numpy as np
import scipy.spatial.distance as _dist

__all__ = [
    "cross_covariance", "predict", "hessian", "prepare_likelihood", "loglikelihood_and_grad", "predict_longdouble",
    "mv_compress", "mv_predict_point", "mv_predict_batch", "bank_predict", "bank_cost",
    "ref_err", "var_cond_err", "make_S_model", "make_T_model", "make_training_problem",
]


# --------------------------------------------------------------------------------------------------
# single GP
# --------------------------------------------------------------------------------------------------
def cross_covariance(inputs, theta, testing):
    """K* as the reference forms it: (M, N) = b * exp(-0.5 * cdist(sqrt(w) x, sqrt(w) t)^2).

    gp_emulator/GaussianProcess.py:230-234 (same three numpy/scipy calls, same operand order).
    """
    D = inputs.shape[1]
    e = np.exp(theta)
    s = np.sqrt(e[:D])
    a = _dist.cdist(s * inputs, s * testing, "sqeuclidean")
    return e[D] * np.exp(-0.5 * a), e


def _predict_block(inputs, theta, invQ, invQt, testing, do_unc):
    """One un-chunked evaluation; gp_emulator/GaussianProcess.py:228-251."""
    nn, D = testing.shape
    a, e = cross_covariance(inputs, theta, testing)
    mu = np.dot(a.T, invQt)                                   # :237
    var = None
    if do_unc:
        var = e[D] - np.sum(a * np.dot(invQ, a), axis=0)      # :240
    deriv = np.zeros((nn, D))
    for d in range(D):                                        # :244-247
        aa = inputs[:, d].flatten()[None, :] - testing[:, d].flatten()[:, None]
        c = a * aa.T
        deriv[:, d] = e[d] * np.dot(c.T, invQt)
    return mu, var, deriv


def predict(inputs, theta, invQ, invQt, testing, do_unc=True, chunk=50000):
    """``GaussianProcess.cpu_predict`` (gp_emulator/GaussianProcess.py:211-251).

    Returns (mu (N,), var (N,), deriv (N, D)); var is None when ``do_unc`` is False.  The reference
    materialises (M, N) temporaries in one go; test points are independent, so evaluating in chunks
    of ``chunk`` points and concatenating gives the same per-point arithmetic with bounded memory.
    """
    testing = np.ascontiguousarray(testing, dtype=np.float64)
    N, D = testing.shape
    assert D == inputs.shape[1]
    mu = np.empty(N)
    var = np.empty(N) if do_unc else None
    deriv = np.empty((N, D))
    for s in range(0, max(N, 1), chunk):
        blk = testing[s:s + chunk]
        if blk.shape[0] == 0:
            break
        m, v, g = _predict_block(inputs, theta, invQ, invQt, blk, do_unc)
        mu[s:s + chunk] = m
        deriv[s:s + chunk] = g
        if do_unc:
            var[s:s + chunk] = v
    return mu, var, deriv


def hessian(inputs, theta, invQt, testing, chunk=20000):
    """``GaussianProcess.hessian`` (gp_emulator/GaussianProcess.py:345-366): (N, D, D)."""
    testing = np.ascontiguousarray(testing, dtype=np.float64)
    N, D = testing.shape
    hess = np.empty((N, D, D))
    for s in range(0, N, chunk):
        blk = testing[s:s + chunk]
        a, e = cross_covariance(inputs, theta, blk)           # :351-354
        eye_w = np.identity(D) * e[:D]                        # :355
        for d in range(D):                                    # :357-365 (same left-to-right product order)
            for d2 in range(D):
                aa = e[d] * (inputs[:, d].flatten()[None, :] - blk[:, d].flatten()[:, None]) * \
                    e[d2] * (inputs[:, d2].flatten()[None, :] - blk[:, d2].flatten()[:, None]) - eye_w[d, d2]
                cc = a * aa.T
                hess[s:s + chunk, d, d2] = np.dot(cc.T, invQt)
    return hess


def prepare_likelihood(inputs, targets, theta):
    """State consumed by predict: (invQ, invQt).  gp_emulator/GaussianProcess.py:52-72.

    Q = b * exp(-0.5 * sum_d w_d (x_id - x_jd)^2) + exp(theta[D+1]) * I, invQ by explicit inverse.
    """
    n, D = inputs.shape
    e = np.exp(theta)
    Z = np.zeros((n, n))
    for d in range(D):
        col = np.tile(inputs[:, d], (n, 1))
        Z = Z + e[d] * (col - col.T) ** 2
    Z = e[D] * np.exp(-0.5 * Z)
    Q = Z + e[D + 1] * np.eye(n)
    invQ = np.linalg.inv(Q)
    invQt = np.dot(invQ, targets)
    return invQ, invQt


def loglikelihood_and_grad(inputs, targets, theta):
    """The training cost and its gradient at ``theta``: ``(loglik, partial_d (D + 2,))``.

    gp_emulator/GaussianProcess.py:78-95 (loglikelihood = _set_params -> _prepare_likelihood :52-75, then
    0.5 log|Q| + 0.5 t.invQt + 0.5 n log 2 pi) followed by partial_devs (:97-125) at the same theta -- the pair of
    calls scipy's L-BFGS-B makes per evaluation (:171-173).  Same numpy calls, same operand order.
    """
    n, D = inputs.shape
    e = np.exp(theta)
    Z = np.zeros((n, n))
    for d in range(D):                                                  # :61-66
        col = np.tile(inputs[:, d], (n, 1))
        Z = Z + e[d] * (col - col.T) ** 2
    Z = e[D] * np.exp(-0.5 * Z)
    Q = Z + e[D + 1] * np.eye(n)
    invQ = np.linalg.inv(Q)
    invQt = np.dot(invQ, targets)
    logdetQ = 2.0 * np.sum(np.log(np.diag(np.linalg.cholesky(Q))))     # :73-75 (raises LinAlgError if Q is not PD)
    ll = 0.5 * logdetQ + 0.5 * np.dot(targets, invQt) + 0.5 * n * np.log(2.0 * np.pi)   # :90-92
    partial_d = np.zeros(D + 2)
    for d in range(D):                                                  # :108-116
        col = np.tile(inputs[:, d], (n, 1))
        V = ((col - col.T) ** 2).T * Z
        partial_d[d] = np.exp(theta[d]) * (np.dot(invQt, np.dot(V, invQt)) - np.sum(invQ * V)) / 4.0
    partial_d[D] = 0.5 * np.sum(invQ * Z) - 0.5 * np.dot(invQt, np.dot(Z, invQt))        # :117-119
    partial_d[D + 1] = 0.5 * np.trace(invQ) * np.exp(theta[D + 1]) - 0.5 * np.dot(invQt, invQt) * np.exp(theta[D + 1])
    return ll, partial_d


def make_training_problem(M=60, D=4, T=3, B=6, seed=21):
    """Seeded training inputs (M, D), T smooth target vectors (T, M), B thetas drawn as the reference draws its
    L-BFGS-B starts (5 (U - 0.5), gp_emulator/GaussianProcess.py:201) and the target row each theta is paired with."""
    rs = np.random.RandomState(seed)
    inputs = rs.random_sample((M, D))
    k = np.arange(1, T + 1)[:, None]
    targets = np.sin(k * (inputs @ np.linspace(1.0, 2.0, D))[None, :]) + 0.3 * np.cos(3.0 * inputs[:, 0])[None, :] / k
    thetas = 5.0 * (rs.random_sample((B, D + 2)) - 0.5)
    tidx = (np.arange(B) % T).astype(np.int32)
    return inputs, targets, thetas, tidx


def predict_longdouble(inputs, theta, invQ, invQt, testing, do_hess=False):
    """Extended-precision evaluation of the same formulas (x87 80-bit ``np.longdouble``).

    Not a reference function: the arbiter used when two FP64 evaluation orders legitimately differ
    (ill-conditioned variance on trained models, SURVEY.md section 7).  O(N*M*M) in Python-level
    longdouble matmul, keep N small.
    """
    L = np.longdouble
    x = inputs.astype(L)
    t = np.asarray(testing).astype(L)
    e = np.exp(theta.astype(L))
    D = x.shape[1]
    diff = x[None, :, :] - t[:, None, :]                      # (N, M, D)
    r2 = np.sum(e[:D] * diff * diff, axis=2)
    k = e[D] * np.exp(-r2 / 2)                                # (N, M)
    al = invQt.astype(L)
    mu = k @ al
    Sk = k @ invQ.astype(L).T
    var = e[D] - np.sum(k * Sk, axis=1)
    c = k * al
    deriv = e[:D] * np.einsum("nm,nmd->nd", c, diff)
    out = [mu, var, deriv]
    if do_hess:
        wd = e[:D] * diff
        H = np.einsum("nm,nmd,nme->nde", c, wd, wd) - np.einsum("n,de->nde", mu, np.diag(e[:D]))
        out.append(H)
    return tuple(out)


# --------------------------------------------------------------------------------------------------
# multivariate (PCA) emulator and banks
# --------------------------------------------------------------------------------------------------
def mv_compress(X, basis_functions):
    """``MultivariateEmulator.compress`` (gp_emulator/multivariate_gp.py:191-193): (P, N_train)."""
    return X.dot(basis_functions.T).T


def mv_predict_point(models, basis_functions, y, do_deriv=True):
    """``MultivariateEmulator.predict`` for ONE point (gp_emulator/multivariate_gp.py:195-222).

    ``models`` is a list of (inputs, theta, invQ, invQt) per principal component.  Returns
    fwd (W,) and deriv (D, W) exactly as the reference accumulates them (:216, :218).
    """
    y = np.atleast_2d(y)
    W = basis_functions.shape[1]
    fwd = np.zeros(W)
    deriv = np.zeros((y.shape[1], W))
    for i, (inputs, theta, invQ, invQt) in enumerate(models):
        mu, _, grad = predict(inputs, theta, invQ, invQt, y, do_unc=True)
        fwd += mu * basis_functions[i]
        if do_deriv:
            deriv += grad.T @ basis_functions[i][None, :]
    return (fwd, deriv) if do_deriv else fwd


def bank_predict(models, testing, do_hess=False):
    """E independent GPs on shared test inputs (pattern of tests/test_perband_emulator.py:22-37).

    Returns mu (N, E), var (N, E), deriv (N, E, D) [, hess (N, E, D, D)].
    """
    N, D = testing.shape
    E = len(models)
    mu = np.empty((N, E))
    var = np.empty((N, E))
    deriv = np.empty((N, E, D))
    hess = np.empty((N, E, D, D)) if do_hess else None
    for i, (inputs, theta, invQ, invQt) in enumerate(models):
        m, v, g = predict(inputs, theta, invQ, invQt, testing)
        mu[:, i], var[:, i], deriv[:, i, :] = m, v, g
        if do_hess:
            hess[:, i] = hessian(inputs, theta, invQt, testing)
    return (mu, var, deriv, hess) if do_hess else (mu, var, deriv)


def bank_cost(models, testing, obs, weights=None):
    """Least-squares misfit of E per-band GPs against observed bands, and its gradient w.r.t. the inputs, built the way a
    caller of the reference builds it: one ``predict`` per emulator (tests/test_perband_emulator.py:39-47), then
    cost_n = 1/2 sum_e w_e (mu_ne - obs_ne)^2 and grad_nd = sum_e w_e (mu_ne - obs_ne) deriv_ned.  (Not a reference
    function: the checker for ``gpe_bank_cost``, SURVEY.md 8f-3.)"""
    mu, _, deriv = bank_predict(models, testing)
    r = mu - np.asarray(obs)
    w = np.ones(mu.shape[1]) if weights is None else np.asarray(weights)
    return 0.5 * np.sum(w * r * r, axis=1), np.einsum("ne,ned->nd", w * r, deriv)


def mv_predict_batch(models, basis_functions, testing, want_deriv_full=False):
    """Batched semantics for N points (new capability, SURVEY.md section 8a row A5).

    The reference handles one point per call; the batched definition is the row-wise stack of that:
    fwd (N, W) = MU (N, P) @ B, PC-space gradient grad (N, P, D), and optionally the full
    deriv (N, D, W) = einsum('npd,pw->ndw').
    """
    mu, var, grad = bank_predict(models, testing)
    fwd = mu @ basis_functions
    out = [fwd, mu, var, grad]
    if want_deriv_full:
        out.append(np.einsum("npd,pw->ndw", grad, basis_functions))
    return tuple(out)


# --------------------------------------------------------------------------------------------------
# parity metrics (SURVEY.md section 8d) and synthetic model generators
# --------------------------------------------------------------------------------------------------
def ref_err(x, ref):
    """The reference's own metric: max|x - ref| / max|ref| (tests/benchmark.py:51-53)."""
    x = np.asarray(x, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    den = np.max(np.abs(ref)) if ref.size else 1.0
    return float(np.max(np.abs(x - ref)) / den) if ref.size else 0.0


def var_cond_err(var, var_ref, inputs, theta, invQ, testing):
    """Condition-scaled variance error: max_n |dvar_n| / (b + |k_n|^T |invQ| |k_n|)."""
    a, e = cross_covariance(inputs, theta, testing)
    scale = e[inputs.shape[1]] + np.sum(np.abs(a) * (np.abs(invQ) @ np.abs(a)), axis=0)
    return float(np.max(np.abs(np.asarray(var) - np.asarray(var_ref)) / scale))


def make_S_model(M=250, D=10, N=1000, seed=0):
    """Synthetic "S" model exactly as tests/benchmark.py:11-15,28-29 draws it (all U(0,1)), seeded.

    Draw order: inputs, testing, theta, invQ, invQt -- the order benchmark.py consumes the stream.
    Uses the legacy ``RandomState`` so the stream is identical across numpy versions.
    """
    rs = np.random.RandomState(seed)
    inputs = rs.random_sample((M, D))
    testing = rs.random_sample((N, D))
    theta = rs.random_sample(D + 2)
    invQ = rs.random_sample((M, M))
    invQt = rs.random_sample(M)
    return inputs, theta, invQ, invQt, testing


def make_T_model(M=100, D=4, N=200, seed=1, theta=None):
    """A genuinely conditioned model: smooth targets, fixed theta, invQ/invQt via prepare_likelihood."""
    rs = np.random.RandomState(seed)
    inputs = rs.random_sample((M, D))
    testing = rs.random_sample((N, D))
    targets = np.sin(inputs @ np.linspace(1.0, 2.0, D)) + 0.3 * np.cos(3.0 * inputs[:, 0])
    if theta is None:
        theta = np.array([-1.0] * D + [0.0, -8.0])
    invQ, invQt = prepare_likelihood(inputs, targets, theta)
    return inputs, targets, theta, invQ, invQt, testing
