"""Inversion (gpe_bank_solve: DeviceBank.forward_invert / invert, MultivariateEmulator.invert) at config 4 (E = 20 PCs,
W = 2101 wavelengths, M = 250, D = 10, spectrum cost) and config 5 (E = 64 bands, M = 250, D = 10, band cost), each beside
the paths it replaces, in one run.  Synthetic pixels: the bank's own output at random x_true in [0, 1]^D plus noise, one
observation per pixel, starts x0 = x_true + 0.1 N(0, 1) clipped to the box [0, 1]^D.  Wall times around calls that end
synchronised (the solve is synchronous), after a warm-up call of the same kind and size; min / median / max of 3 calls.

  device-resident:  N = 1e6 pixels, CUDA tensors in and out
  host-resident:    N = 1e5 pixels, numpy in and out, pageable and page-locked; beside them the device-resident time at
                    the same N and the inputs' H2D copy alone.  Page-locked minus device-resident is the transfer time the
                    blocking chunk solves leave unoverlapped (pageable adds the staging copies)
  python loop:      the same algorithm (tests/test_invert.py lm_ref) around the library's cost + grad + hess calls,
                    evaluations device-resident (results copied to the host each iteration) and host-resident, N = 1e4
  scipy:            per-pixel scipy.optimize.minimize (L-BFGS-B, bounds) on the library's one-point cost, 200 pixels
  kernels:          torch.profiler per-kernel times of a device-resident solve of 1e5 pixels (separate pass): the share of
                    k_lm_step + compaction + gather, and the idle time per iteration (wall - kernel time, over iterations)
  one point:        MultivariateEmulator.invert against the hand-written 8-step Newton loop it replaced in the quickstart

Usage: python tools/invert_probe.py [out.json]"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from tools.forward_cost_probe import gpu_info  # noqa: E402

W, M, D = 2101, 250, 10


def wall(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def repeat(fn, reps=3):
    """min / median / max seconds of `reps` synchronised calls, and the last call's result."""
    import numpy as np
    ts = []
    for _ in range(reps):
        t, r = wall(fn)
        ts.append(t)
    return {"min_s": float(np.min(ts)), "median_s": float(np.median(ts)), "max_s": float(np.max(ts))}, r


def evals_hist(n_iter):
    import numpy as np
    v = np.asarray(n_iter)
    return {"mean": float(v.mean()), "p50": float(np.percentile(v, 50)), "p90": float(np.percentile(v, 90)),
            "max": int(v.max()), "counts": np.bincount(v).tolist()}


def kernel_share(fn):
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        wall_s = time.perf_counter() - t0
    total = solver = 0.0
    steps = 0
    for ev in prof.key_averages():
        v = (getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)) / 1e6
        if v <= 0:
            continue
        total += v
        if any(k in ev.key for k in ("k_lm_", "DeviceSelect", "DeviceCompact")):
            solver += v
        if "k_lm_step" in ev.key:
            steps += ev.count
    return {"kernel_s": total, "solver_kernels_s": solver, "solver_share": solver / total, "iterations": steps,
            "wall_s_profiled": wall_s, "idle_per_iteration_us": (wall_s - total) / max(steps, 1) * 1e6}


def run_config(name, bank, spectra, rs, res, line):
    import numpy as np
    import torch
    from scipy.optimize import minimize
    from tests.test_invert import lm_ref
    lo, hi = np.zeros(D), np.ones(D)
    solve = bank.forward_invert if spectra else bank.invert
    cost = bank.forward_cost if spectra else bank.cost

    def pixels(n, dev):
        xt = torch.rand(n, D, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(n))
        out = bank.predict(xt, want_var=False, want_deriv=False, project=spectra)
        obs = out["fwd"] if spectra else out["mu"]
        obs = obs * (1 + 0.01 * torch.randn(obs.shape, dtype=torch.float64, device="cuda"))
        x0 = (xt + 0.1 * torch.randn(xt.shape, dtype=torch.float64, device="cuda")).clamp(0, 1)
        return (x0, obs) if dev else (x0.cpu().numpy(), obs.cpu().numpy())

    lo_t, hi_t = torch.zeros(D, dtype=torch.float64, device="cuda"), torch.ones(D, dtype=torch.float64, device="cuda")
    N = 1_000_000
    x0, obs = pixels(N, True)
    solve(x0, obs, lower=lo_t, upper=hi_t)          # warm-up at full size: the solver and cost scratch grow once
    t, r = repeat(lambda: solve(x0, obs, lower=lo_t, upper=hi_t))
    st = r["status"].cpu().numpy()
    line(f"{name}_device_1e6", {"pixels_per_s": N / t["median_s"], **t,
                                "evaluations_after_first": evals_hist(r["n_iter"].cpu().numpy()),
                                "status_counts": np.bincount(st, minlength=4).tolist()})
    del x0, obs, r
    torch.cuda.empty_cache()
    N = 100_000
    x0d, obsd = pixels(N, True)
    solve(x0d, obsd, lower=lo_t, upper=hi_t)
    t_dev, _ = repeat(lambda: solve(x0d, obsd, lower=lo_t, upper=hi_t))
    line(f"{name}_kernels_1e5", kernel_share(lambda: solve(x0d, obsd, lower=lo_t, upper=hi_t)))
    x0, obs = x0d.cpu().numpy(), obsd.cpu().numpy()
    solve(x0, obs, lower=lo, upper=hi)          # warm-up at full size: the pipeline grows its page-locked staging once
    t_host, r = repeat(lambda: solve(x0, obs, lower=lo, upper=hi))
    # page-locked inputs take the direct path (no staging copy): what it adds to the device-resident time is the part of
    # the uploads (and result downloads) that the blocking chunk solves leave unoverlapped
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
    x0p, obsp = pin(x0), pin(obs)
    solve(x0p, obsp, lower=lo, upper=hi)
    t_pin, _ = repeat(lambda: solve(x0p, obsp, lower=lo, upper=hi))
    t_up, _ = repeat(lambda: (obsd.copy_(torch.from_numpy(obsp), non_blocking=True), x0d.copy_(torch.from_numpy(x0p),
                                                                                               non_blocking=True)))
    line(f"{name}_host_1e5", {"pixels_per_s": N / t_host["median_s"], "pageable": t_host, "page_locked": t_pin,
                              "device_resident_same_N": t_dev, "inputs_h2d_alone": t_up,
                              "not_overlapped_page_locked_s": t_pin["median_s"] - t_dev["median_s"],
                              "not_overlapped_pageable_s": t_host["median_s"] - t_dev["median_s"],
                              "evaluations_after_first": evals_hist(r["n_iter"])})
    del x0d, obsd, x0p, obsp
    torch.cuda.empty_cache()

    # the same algorithm as a Python loop around the library's cost + grad + hess
    n = 10_000
    x0, obs = pixels(n, False)
    for dev in (True, False):
        obs_dev = torch.from_numpy(obs).cuda() if dev else None

        def fgh(X, idx):
            if dev:
                o = cost(torch.from_numpy(X).cuda(), obs_dev[torch.from_numpy(idx).cuda()], want_hess=True)
                return o["cost"].cpu().numpy(), o["grad"].cpu().numpy(), o["hess"].cpu().numpy()
            o = cost(X, obs[idx], want_hess=True)
            return o["cost"], o["grad"], o["hess"]
        t, _ = wall(lambda: lm_ref(fgh, x0, lo, hi, indexed=True))
        line(f"{name}_python_loop_{'device' if dev else 'host'}_1e4", {"pixels_per_s": n / t, "s": t})
    # per-pixel scipy
    n = 200
    t0 = time.perf_counter()
    for k in range(n):
        def fg(y, k=k):
            o = cost(y[None], obs[k])
            return o["cost"][0], o["grad"][0]
        minimize(fg, x0[k], jac=True, method="L-BFGS-B", bounds=list(zip(lo, hi)))
    t = time.perf_counter() - t0
    line(f"{name}_scipy_per_pixel_200", {"pixels_per_s": n / t, "s_per_pixel": t / n})


def main():
    import numpy as np
    import torch
    import gp_emulator_b200 as g
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"config4": {"E": 20, "W": W, "M": M, "D": D}, "config5": {"E": 64, "M": M, "D": D}, "gpu": gpu_info()}
    line = lambda k, v: (res.__setitem__(k, v), print(k, json.dumps(v), flush=True))
    rs = np.random.RandomState(0)
    E = 20
    y = rs.random_sample((M, D))
    hyp = np.vstack([rs.random_sample((D, E)) * 2 - 3, np.ones((1, E)), np.full((1, E), -6.0)])
    wl = np.linspace(0, 1, W)
    B = np.linalg.qr(np.stack([np.cos(np.pi * (k + 1) * wl) for k in range(E)]).T)[0].T
    X = (np.sin(y @ rs.random_sample((D, E))) @ B) + 0.01 * rs.standard_normal((M, W))
    emu = g.MultivariateEmulator(X=X, y=y, hyperparams=hyp, basis_functions=B, n_pcs=E)
    run_config("config4", emu._device_bank(), True, rs, res, line)

    # one point: MultivariateEmulator.invert against the quickstart's former Newton loop
    xt = rs.random_sample(D)
    obs = emu.predict(xt, do_deriv=False) * (1 + 0.01 * rs.standard_normal(W))
    y0 = np.clip(xt + 0.1 * rs.standard_normal(D), 0, 1)

    def newton():
        yy, damp = y0.copy(), 0.0
        c, gg, H = emu.cost(yy, obs, do_hess=True)
        for _ in range(8):
            step = np.linalg.solve(H + damp * np.abs(np.diag(H)).max() * np.eye(D), -gg)
            c2, g2, H2 = emu.cost(yy + step, obs, do_hess=True)
            if c2 < c:
                yy, c, gg, H, damp = yy + step, c2, g2, H2, damp / 10
            else:
                damp = max(10 * damp, 1e-3)
        return np.linalg.inv(H)
    inv = lambda: emu.invert(obs, y0, bounds=(np.zeros(D), np.ones(D)))
    for f in (newton, inv):
        f()
    reps = 50
    tn = min(wall(newton)[0] for _ in range(reps))
    ti_, r1 = min((wall(inv) for _ in range(reps)), key=lambda p: p[0])
    line("one_point", {"invert_s": ti_, "newton_loop_8_steps_s": tn, "invert_evaluations_after_first": int(r1["n_iter"])})

    E5 = 64
    inputs = rs.random_sample((M, D))
    thetas = np.vstack([rs.random_sample((D, E5)) * 2 - 3, np.ones((1, E5))]).T
    invQts = rs.standard_normal((E5, M))
    run_config("config5", g.DeviceBank(inputs, thetas, invQts), False, rs, res, line)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
