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
5. a per-band bank reduced on the device to a least-squares misfit and its gradient (``DeviceBank.cost``), then 1000
   band observations inverted at once with each pixel's own sigma and one band masked on a tenth of the pixels
   (per-point weights ``(N, bands)``: ``DeviceBank.invert``);
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
    noise = np.random.RandomState(1).standard_normal(len(wl))                # 3b. look-up-table search
    obs_lut = truth + 0.01 * noise                                            # 1000 observed spectra, one call:
    found = emu.search(obs_lut, candidates=y_test, k=3)                       # the 3 best of 1000 candidates per pixel
    print("look-up table: %d of %d pixels pick their own candidate first; pixel 3: candidates %s, costs %s" % (
        int(np.sum(found["idx"][:, 0] == np.arange(len(obs_lut)))), len(obs_lut), found["idx"][3].tolist(),
        np.round(found["cost"][3], 3).tolist()))
    sigma = 0.01                                                              # 3c. inversion + Laplace uncertainty
    obs = truth + sigma * np.random.RandomState(2).standard_normal(truth.shape)   # one noisy spectrum per pixel
    lower, upper = np.array([d.ppf(0.0) for d in dists]), np.array([d.ppf(1.0) for d in dists])
    w = np.full(len(wl), 1.0 / sigma ** 2)                                    # weights 1 / sigma^2: cost = -log likelihood
    state = np.random.get_state()                                             # (later steps keep their draws)
    np.random.seed(3)
    table = gpe.lhd(dist=dists, size=2000)                                    # starts: the 4 best rows of a seeded table
    np.random.set_state(state)
    t0 = time.perf_counter()
    res = emu.invert(obs, weights=w, bounds=(lower, upper), candidates=table, n_starts=4)
    t_seeded = time.perf_counter() - t0
    t0 = time.perf_counter()
    mid = emu.invert(obs, np.tile(0.5 * (lower + upper), (len(obs), 1)), weights=w, bounds=(lower, upper))
    t_mid = time.perf_counter() - t0
    print("inverted %d spectra from the table in %.3f s (from the box centre: %.3f s); median cost %.1f (box centre: "
          "%.1f); status counts %s (converged, max_iter, stalled, nonfinite)" % (
        len(obs), t_seeded, t_mid, np.median(res["cost"]), np.median(mid["cost"]),
        np.bincount(res["status"], minlength=4).tolist()))
    sd = np.sqrt(np.diagonal(res["cov"], axis1=1, axis2=2))
    print("pixel 3: retrieved %s +- %s (Laplace sd), truth %s; %.0f%% of all retrieved parameters lie within 3 sd of "
          "the truth" % (np.round(res["x"][3], 4), np.round(sd[3], 4), np.round(y_test[3], 4),
                         100 * np.mean(np.abs(res["x"] - y_test) <= 3 * sd)))

    rs = np.random.RandomState(5)                                             # 3d. time series with cloudy dates
    S, T = 200, 46                                                            # 200 pixels x 46 dates a season
    ph = rs.uniform(0, 2 * np.pi, (S, 1, len(dists)))
    y_ts = (lower + upper) / 2 + 0.3 * (upper - lower) * np.sin(2 * np.pi * np.arange(T)[None, :, None] / T + ph)
    obs_ts = toy_model(y_ts.reshape(-1, len(dists)), wl) + sigma * rs.standard_normal((S * T, len(wl)))
    cloudy = rs.random_sample(S * T) < 0.4                                    # 40 % of the dates masked
    w_ts = np.where(cloudy[:, None], 0.0, 1.0 / sigma ** 2) * np.ones(len(wl))
    obs_ts[cloudy] = 0.0                                                      # no data there: any finite value, weight 0
    y0 = table[emu.search(obs_ts, candidates=table, k=1)["idx"][:, 0]]       # starts per date from the table ...
    y0[cloudy] = 0.5 * (lower + upper)                                        # ... and the box centre where it is cloudy
    per_date = emu.invert(obs_ts, y0, weights=w_ts, bounds=(lower, upper), do_cov=False)
    step = 0.3 * (upper - lower) * 2 * np.pi / T                              # largest change of y between dates
    ts = emu.invert_series(obs_ts.reshape(S, T, -1), y0.reshape(S, T, -1), smooth=(np.diag(1.0 / step ** 2), None),
                           weights=w_ts.reshape(S, T, -1), bounds=(lower, upper), do_cov=False)
    err = lambda x: np.abs(x.reshape(-1, len(dists)) - y_ts.reshape(-1, len(dists)))
    rms = lambda e, m: np.sqrt(np.mean(e[m] ** 2))
    print("time series, %d pixels x %d dates, %d %% cloudy: rmse on cloudy dates %.4f per date, %.4f jointly; on clear "
          "dates %.4f per date, %.4f jointly; series status counts %s" % (
        S, T, round(100 * cloudy.mean()), rms(err(per_date["x"]), cloudy), rms(err(ts["x"]), cloudy),
        rms(err(per_date["x"]), ~cloudy), rms(err(ts["x"]), ~cloudy), np.bincount(ts["status"], minlength=4).tolist()))

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
    rs = np.random.RandomState(4)                                             # 5b. per-pixel sigma and masked bands
    sig = 0.005 * rs.uniform(0.5, 3.0, (len(y_test), len(bands)))            # each pixel's own noise level per band
    obs_b = truth[:, bands] + sig * rs.standard_normal(sig.shape)
    wb = 1.0 / sig ** 2                                                       # weights (N, bands): one row per pixel
    masked = rs.random_sample(len(y_test)) < 0.1
    wb[masked, 2] = 0.0                                                       # band 2 unusable there: weight 0
    rb = bank.invert(np.tile(0.5 * (lower + upper), (len(y_test), 1)), obs_b, wb, lower=lower, upper=upper, want_cov=True)
    sdb = np.sqrt(np.diagonal(rb["cov"], axis1=1, axis2=2))
    print("inverted %d band observations with per-pixel sigma, band %d masked on %d of them: status counts %s; median "
          "Laplace sd of parameter 0: %.4f with all bands, %.4f with one masked" % (
        len(y_test), bands[2], int(masked.sum()), np.bincount(rb["status"], minlength=4).tolist(),
        np.nanmedian(sdb[~masked, 0]), np.nanmedian(sdb[masked, 0])))

    with tempfile.TemporaryDirectory() as tmp:                                # 6. storage
        store = gpe.EmulatorStorage(os.path.join(tmp, "emulators"))
        store.dump_emulator(emu, ("toy", 400))
        store.dump_emulator(gps[0], ("toy", "band", bands[0]))
        again = store.get_emulator(("toy", 400))
        print("stored keys:", sorted(store.get_keys()), "| reloaded emulator reproduces the spectrum:",
              bool(np.allclose(again.predict(y_test[0], do_deriv=False), fwd)))


if __name__ == "__main__":
    main()
