"""Joint time-series inversion (gpe_bank_solve_series: DeviceBank.forward_invert_series / invert_series) at config 4
(E = 20 PCs, W = 2101 wavelengths, M = 250, D = 10, spectrum cost) and config 5 (E = 64 bands, M = 250, D = 10, band
cost), T = 73 dates a series, each beside the paths it replaces, in one run.  Synthetic series: a smooth trajectory
x_true(t) in [0, 1]^D (a sine of random phase per input), the bank's own output there plus noise of 1 % of each band's
mean magnitude, weights 1 / sigma^2 per row and 0 on the 30 % of dates that are masked, starts x0 = x_true + 0.1 N(0, 1)
clipped to the box, smoothness precision R = I / (largest change of x_true between dates)^2, coupling all 1.  Wall times around calls that end synchronised (the
solve is synchronous), after a warm-up call at the same size; min / median / max of the timed calls.

  device-resident:  S = 13,699 series (1.0e6 rows), CUDA tensors in and out; beside it per-date invert on the same rows
  host-resident:    S = 1,370 series (1.0e5 rows), numpy in and out; beside it the device-resident time at the same S
  python loop:      the same algorithm (tests/test_invert_series.py lm_series_ref, dense solve per series) around the
                    library's cost + grad + hess calls, evaluations device-resident, on a slice of 20 series
  kernels:          torch.profiler per-kernel times of a device-resident solve of 1.0e5 rows (separate pass): the shares
                    of k_lm_series_step, k_lm_series_output, the cost kernels and the rest

Usage: python tools/invert_series_probe.py [out.json]"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from tools.forward_cost_probe import gpu_info  # noqa: E402
from tools.invert_probe import evals_hist, wall  # noqa: E402

W, M, D, T = 2101, 250, 10, 73
MASKED = 0.3


def repeat(fn, reps):
    import numpy as np
    ts = []
    for _ in range(reps):
        t, r = wall(fn)
        ts.append(t)
    return {"min_s": float(np.min(ts)), "median_s": float(np.median(ts)), "max_s": float(np.max(ts)), "reps": reps}, r


def kernel_shares(fn):
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        wall_s = time.perf_counter() - t0
    total, parts, steps = 0.0, {"k_lm_series_step": 0.0, "k_lm_series_output": 0.0, "cost": 0.0, "other": 0.0}, 0
    for ev in prof.key_averages():
        v = (getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)) / 1e6
        if v <= 0:
            continue
        total += v
        if "k_lm_series_step" in ev.key:
            parts["k_lm_series_step"] += v
            steps += ev.count
        elif "k_lm_series_output" in ev.key:
            parts["k_lm_series_output"] += v
        elif any(k in ev.key for k in ("k_bank", "k_forward_cost", "k_cost_hess", "k_predict", "k_project")):
            parts["cost"] += v
        else:
            parts["other"] += v
    return {"kernel_s": total, "wall_s_profiled": wall_s, "step_launches": steps,
            "kernel_s_by_part": parts, "share_of_kernel_time": {k: v / total for k, v in parts.items()},
            "step_us_per_launch": parts["k_lm_series_step"] / max(steps, 1) * 1e6}


def run_config(name, bank, spectra, line):
    import numpy as np
    import torch
    from tests.test_invert_series import lm_series_ref
    solve_s = bank.forward_invert_series if spectra else bank.invert_series
    solve_p = bank.forward_invert if spectra else bank.invert
    cost = bank.forward_cost if spectra else bank.cost
    step = 0.2 * 2 * np.pi / T
    R = np.eye(D) / step ** 2
    dev = lambda a: torch.as_tensor(a, dtype=torch.float64, device="cuda")
    lo_t, hi_t, R_t = dev(np.zeros(D)), dev(np.ones(D)), dev(R)

    def series(S):
        g = torch.Generator("cuda").manual_seed(S)
        rnd = lambda *s: torch.rand(*s, dtype=torch.float64, device="cuda", generator=g)
        t = torch.arange(T, dtype=torch.float64, device="cuda")[None, :, None]
        xt = (0.35 + 0.3 * rnd(S, 1, D)) + 0.2 * torch.sin(2 * np.pi * t / T + 2 * np.pi * rnd(S, 1, D))
        out = bank.predict(xt.reshape(-1, D), want_var=False, want_deriv=False, project=spectra)
        obs = out["fwd"] if spectra else out["mu"]
        sig = 0.01 * obs.abs().mean(dim=0)                   # noise: 1 % of each band's mean magnitude
        obs = obs + sig * torch.randn(obs.shape, dtype=torch.float64, device="cuda", generator=g)
        K = obs.shape[1]
        w = ((rnd(S * T, 1) >= MASKED).to(torch.float64) / sig ** 2).contiguous()   # 1 / sigma^2, 0 on masked dates
        x0 = (xt + 0.1 * torch.randn(xt.shape, dtype=torch.float64, device="cuda", generator=g)).clamp(0, 1)
        return xt, x0, obs.reshape(S, T, K), w.reshape(S, T, K)

    def rmse(x, xt, w):
        m = (w[..., 0] == 0).reshape(-1).cpu().numpy()
        e = (x.reshape(-1, D) - xt.reshape(-1, D)).cpu().numpy()
        return {"masked": float(np.sqrt(np.mean(e[m] ** 2))), "observed": float(np.sqrt(np.mean(e[~m] ** 2)))}

    S = 13_699
    xt, x0, obs, w = series(S)
    kw = dict(smooth_precision=R_t, lower=lo_t, upper=hi_t)
    solve_s(x0[:10], obs[:10], w[:10], **kw)
    solve_s(x0, obs, w, **kw)                      # warm-up at full size: the solver and cost scratch grow once
    t, r = repeat(lambda: solve_s(x0, obs, w, **kw), 2)
    st = r["status"].cpu().numpy()
    K = obs.shape[2]
    flat = lambda a, k: a.reshape(S * T, k)
    solve_p(flat(x0, D), flat(obs, K), flat(w, K), lower=lo_t, upper=hi_t)
    tp, rp = repeat(lambda: solve_p(flat(x0, D), flat(obs, K), flat(w, K), lower=lo_t, upper=hi_t), 2)
    line(f"{name}_device_1e6", {
        "series": S, "rows": S * T, "series_per_s": S / t["median_s"], "rows_per_s": S * T / t["median_s"], **t,
        "evaluations_after_first": evals_hist(r["n_iter"].cpu().numpy()),
        "status_counts": np.bincount(st, minlength=4).tolist(), "rmse": rmse(r["x"], xt, w),
        "per_date_invert": {"rows_per_s": S * T / tp["median_s"], **tp,
                            "evaluations_after_first": evals_hist(rp["n_iter"].cpu().numpy()),
                            "status_counts": np.bincount(rp["status"].cpu().numpy(), minlength=4).tolist(),
                            "rmse": rmse(rp["x"].reshape(S, T, D), xt, w)}})
    del xt, x0, obs, w, r, rp
    torch.cuda.empty_cache()

    S = 1_370
    xt, x0, obs, w = series(S)
    solve_s(x0, obs, w, **kw)
    t_dev, _ = repeat(lambda: solve_s(x0, obs, w, **kw), 3)
    line(f"{name}_kernels_1e5", kernel_shares(lambda: solve_s(x0, obs, w, **kw)))
    x0h, obsh, wh = x0.cpu().numpy(), obs.cpu().numpy(), w.cpu().numpy()
    kwh = dict(smooth_precision=R, lower=np.zeros(D), upper=np.ones(D))
    solve_s(x0h, obsh, wh, **kwh)
    t_host, r = repeat(lambda: solve_s(x0h, obsh, wh, **kwh), 3)
    line(f"{name}_host_1e5", {"series": S, "rows": S * T, "rows_per_s": S * T / t_host["median_s"], "host": t_host,
                              "device_resident_same_S": t_dev, "evaluations_after_first": evals_hist(r["n_iter"])})

    # the same algorithm as a Python loop around the library's cost + grad + hess (device-resident evaluations)
    n = 20
    x0n = x0h[:n]
    o_dev, w_dev = obs[:n].reshape(n * T, K), w[:n].reshape(n * T, K)

    def fgh(X, rows):
        idx = torch.from_numpy(rows).cuda()
        o = cost(torch.from_numpy(X).cuda(), o_dev[idx], w_dev[idx], want_hess=True)
        return o["cost"].cpu().numpy(), o["grad"].cpu().numpy(), o["hess"].cpu().numpy()
    t, ref = wall(lambda: lm_series_ref(fgh, x0n, R, None, np.zeros(D), np.ones(D)))
    line(f"{name}_python_loop_{n}_series", {"series": n, "rows": n * T, "rows_per_s": n * T / t, "s": t,
                                            "evaluations_after_first": evals_hist(ref["n_iter"])})
    del xt, x0, obs, w
    torch.cuda.empty_cache()


def main():
    import numpy as np
    import gp_emulator_b200 as g
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"config4": {"E": 20, "W": W, "M": M, "D": D, "T": T}, "config5": {"E": 64, "M": M, "D": D, "T": T},
           "masked_dates": MASKED, "gpu": gpu_info()}

    def line(k, v):
        res[k] = v
        print(k, json.dumps(v), flush=True)
        if out_path:                          # written after every result: a partial run keeps what it measured
            with open(out_path, "w") as f:
                json.dump(res, f, indent=1)
    rs = np.random.RandomState(0)
    E = 20
    y = rs.random_sample((M, D))
    hyp = np.vstack([rs.random_sample((D, E)) * 2 - 3, np.ones((1, E)), np.full((1, E), -6.0)])
    wl = np.linspace(0, 1, W)
    B = np.linalg.qr(np.stack([np.cos(np.pi * (k + 1) * wl) for k in range(E)]).T)[0].T
    X = (np.sin(y @ rs.random_sample((D, E))) @ B) + 0.01 * rs.standard_normal((M, W))
    emu = g.MultivariateEmulator(X=X, y=y, hyperparams=hyp, basis_functions=B, n_pcs=E)
    E5 = 64
    inputs = rs.random_sample((M, D))
    thetas = np.vstack([rs.random_sample((D, E5)) * 2 - 3, np.ones((1, E5))]).T
    invQts = rs.standard_normal((E5, M))
    run_config("config5", g.DeviceBank(inputs, thetas, invQts), False, line)
    run_config("config4", emu._device_bank(), True, line)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
