#!/usr/bin/env python
"""End-to-end tour of the drop-in package on one B200 (synthetic "radiative-transfer" model, runs in a few seconds).

    python examples/quickstart.py

1. draw a Latin-hypercube training design (``lhd``), run a toy spectral model on it;
2. build a ``MultivariateEmulator`` (PCA + one GP per component), hyper-parameters fitted with the batched GPU
   training objective (``batched_training=True``; drop the flag for the reference's sequential host fit);
3. predict spectra + Jacobians, one point (the reference's call) and a batch; score 1000 candidates against an observed
   spectrum (``emu.cost``), then invert 1000 noisy spectra at once inside the design's bounds (``emu.invert``: bounded
   Levenberg-Marquardt on the exact Hessian, on the device) and print the retrieved parameters with their Laplace
   posterior standard deviations;
4. per-band ``GaussianProcess`` objects: mean / variance / gradient / Hessian, FP64 and single precision;
5. a per-band bank reduced on the device to a least-squares misfit and its gradient (``DeviceBank.cost``);
6. store and reload an emulator (``EmulatorStorage``).
"""
import os
import sys
import tempfile
import time

import numpy as np
import scipy.stats as ss

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import gp_emulator_b200 as gpe  # noqa: E402


def toy_model(params, wl):
    """(N, 4) parameters -> (N, len(wl)) smooth 'spectra'."""
    a, b, c, d = (params[:, k:k + 1] for k in range(4))
    return a * np.exp(-((wl[None, :] - 0.3 - 0.4 * b) / (0.1 + 0.2 * c)) ** 2) + d * wl[None, :] ** 2 + 0.05 * np.sin(9 * wl)[None, :]


def main():
    np.random.seed(0)
    wl = np.linspace(0.0, 1.0, 400)
    dists = [ss.uniform(0.5, 1.0), ss.uniform(0.0, 1.0), ss.uniform(0.0, 1.0), ss.uniform(0.0, 0.5)]
    y_train = gpe.lhd(dist=dists, size=150)                                   # 1. design
    X_train = toy_model(y_train, wl)

    t0 = time.perf_counter()                                                  # 2. PCA + batched fit
    emu = gpe.MultivariateEmulator(X=X_train, y=y_train, thresh=0.995, n_tries=4, batched_training=True)
    print("fitted %d PCs x 4 starts in %.2f s (%s)" % (emu.n_pcs, time.perf_counter() - t0, emu.training_stats))

    y_test = gpe.lhd(dist=dists, size=1000)                                   # 3. predict
    fwd, jac = emu.predict(y_test[0])
    print("one point: spectrum %s, Jacobian %s" % (fwd.shape, np.shape(jac)))
    fwd_all = emu.predict(y_test, do_deriv=False)
    truth = toy_model(y_test, wl)
    print("batch of %d: rms emulation error %.2e (signal rms %.2f)" % (len(y_test), np.sqrt(np.mean((fwd_all - truth) ** 2)),
                                                                       np.sqrt(np.mean(truth ** 2))))
    noise = np.random.RandomState(1).standard_normal(len(wl))                # 3b. spectrum misfit
    cost, grad = emu.cost(y_test, truth[3] + 0.01 * noise)                   # spectra and Jacobians stay in the kernel
    best = int(np.argmin(cost))
    print("misfit of 1000 candidates against one observed spectrum: best candidate %d (cost %.3f), true one is 3 "
          "(cost %.3f); gradients %s" % (best, cost[best], cost[3], grad.shape))
    sigma = 0.01                                                              # 3c. inversion + Laplace uncertainty
    obs = truth + sigma * np.random.RandomState(2).standard_normal(truth.shape)   # one noisy spectrum per pixel
    lower, upper = np.array([d.ppf(0.0) for d in dists]), np.array([d.ppf(1.0) for d in dists])
    y0 = np.tile(0.5 * (lower + upper), (len(obs), 1))
    t0 = time.perf_counter()                                                  # weights 1 / sigma^2: cost = -log likelihood
    res = emu.invert(obs, y0, weights=np.full(len(wl), 1.0 / sigma ** 2), bounds=(lower, upper))
    sd = np.sqrt(np.diagonal(res["cov"], axis1=1, axis2=2))
    print("inverted %d spectra in %.3f s, status counts %s (converged, max_iter, stalled, nonfinite)" % (
        len(obs), time.perf_counter() - t0, np.bincount(res["status"], minlength=4).tolist()))
    print("pixel 3: retrieved %s +- %s (Laplace sd), truth %s; %.0f%% of all retrieved parameters lie within 3 sd of "
          "the truth" % (np.round(res["x"][3], 4), np.round(sd[3], 4), np.round(y_test[3], 4),
                         100 * np.mean(np.abs(res["x"] - y_test) <= 3 * sd)))

    bands = [40, 120, 200, 280, 360]                                          # 4. per-band GPs
    from gp_emulator_b200.training import fit_bank
    gps, _ = fit_bank(y_train, X_train[:, bands].T, n_tries=10)              # all bands x starts in one batch
    mu, var, grad = gps[0].predict(y_test)
    hess = gps[0].hessian(y_test[:8])
    mu32, var32, _ = gps[0].predict(y_test.astype(np.float32), precision=np.float32)
    print("band %d: |mu - truth| max %.2e, mean predictive sd %.2e, grad %s, hess %s; single-precision path differs by up to %.1e "
          "(a well-fitted GP has large cancelling weights: keep FP64 for conditioned models)" % (
        bands[0], np.max(np.abs(mu - truth[:, bands[0]])), np.sqrt(np.mean(np.maximum(var, 0))), grad.shape, hess.shape,
        np.max(np.abs(mu32 - mu))))

    bank = gpe.DeviceBank(y_train, np.stack([g.theta for g in gps]), np.stack([g.invQt for g in gps]),   # 5. bank misfit
                          np.stack([g.invQ for g in gps]))
    obs = truth[3, bands] + 0.01 * np.random.standard_normal(len(bands))
    out = bank.cost(y_test, obs, weights=np.full(len(bands), 1e4))
    best = int(np.argmin(out["cost"]))
    print("misfit of 1000 candidates against one observation: best candidate %d (cost %.2f), true one is 3 (cost %.2f)" % (
        best, out["cost"][best], out["cost"][3]))

    with tempfile.TemporaryDirectory() as tmp:                                # 6. storage
        store = gpe.EmulatorStorage(os.path.join(tmp, "emulators"))
        store.dump_emulator(emu, ("toy", 400))
        store.dump_emulator(gps[0], ("toy", "band", bands[0]))
        again = store.get_emulator(("toy", 400))
        print("stored keys:", sorted(store.get_keys()), "| reloaded emulator reproduces the spectrum:",
              bool(np.allclose(again.predict(y_test[0], do_deriv=False), fwd)))


if __name__ == "__main__":
    main()
