"""Per-point observation weights (gpe_bank_cost_pw / gpe_bank_solve_pw / gpe_bank_search_pw, DESIGN 4.6f) against the
same calls with one shared weight vector, in one run, at config 4 (E = 20 PCs, W = 2101 wavelengths, M = 250, D = 10,
spectrum cost) and config 5 (E = 64 bands, M = 250, D = 10, band cost).  Synthetic pixels: the bank's own output at random
x_true in [0, 1]^D plus 1 % noise; per-point weights uniform in [0.5, 2] with 10 % zeros.  Wall times around calls that
end synchronised, after a warm-up call of the same kind and size; min / median / max of 3 calls.

  cost:     cost + grad and cost + grad + hess, device-resident N = 1e6 and host-resident N = 1e5 (numpy, page-locked);
            host-resident rates are reported against the PCIe bound: the call's bytes (testing, obs and, per point, the
            weight rows in; cost, grad, hess out) over the H2D rate of a page-locked copy measured in the same run
  curv:     torch.profiler time of the per-point curvature kernel k_forward_cost_curv_pw inside a device-resident
            cost + grad + hess call of 1e5 points (separate pass), beside the call's total kernel time
  solve:    device-resident N = 1e6, host-resident N = 1e5
  search:   a 48-band bank (the largest the per-point band search takes) and the PROSAIL model (12 PCs), K = 1e4
            candidates, k = 8, device-resident N = 1e5

Usage: python tools/point_weights_probe.py [out.json]"""
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
    import numpy as np
    fn()
    ts = [wall(fn)[0] for _ in range(reps)]
    return {"min_s": float(np.min(ts)), "median_s": float(np.median(ts)), "max_s": float(np.max(ts))}


def h2d_rate():
    """GB/s of a 1 GB page-locked host-to-device copy."""
    import torch
    src = torch.empty(1 << 27, dtype=torch.float64).pin_memory()
    dst = torch.empty_like(src, device="cuda")
    t = repeat(lambda: dst.copy_(src, non_blocking=True))
    return src.numel() * 8 / t["median_s"] / 1e9


def kernel_times(fn, names):
    import torch
    from torch.profiler import profile, ProfilerActivity
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    total, part = 0.0, {n: 0.0 for n in names}
    for ev in prof.key_averages():
        v = (getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)) / 1e6
        if v <= 0:
            continue
        total += v
        for n in names:
            if n in ev.key:
                part[n] += v
    return {"kernel_s": total, **{f"{n}_s": v for n, v in part.items()}}


def weights_like(obs, gen):
    import torch
    w = 0.5 + 1.5 * torch.rand(obs.shape, dtype=torch.float64, device=obs.device, generator=gen)
    return w * (torch.rand(obs.shape, dtype=torch.float64, device=obs.device, generator=gen) >= 0.1)


def run_config(name, bank, spectra, line, pcie):
    import numpy as np
    import torch
    K = W if spectra else bank.E
    cost = bank.forward_cost if spectra else bank.cost
    solve = bank.forward_invert if spectra else bank.invert
    gen = torch.Generator("cuda").manual_seed(1)

    def pixels(n):
        xt = torch.rand(n, D, dtype=torch.float64, device="cuda", generator=gen)
        out = bank.predict(xt, want_var=False, want_deriv=False, project=spectra)
        obs = out["fwd"] if spectra else out["mu"]
        obs = obs * (1 + 0.01 * torch.randn(obs.shape, dtype=torch.float64, device="cuda", generator=gen))
        x0 = (xt + 0.1 * torch.randn(xt.shape, dtype=torch.float64, device="cuda", generator=gen)).clamp(0, 1)
        return x0, obs, weights_like(obs, gen)

    lo, hi = torch.zeros(D, dtype=torch.float64, device="cuda"), torch.ones(D, dtype=torch.float64, device="cuda")
    N = 1_000_000
    x0, obs, wN = pixels(N)
    w1 = wN[0].clone()
    for hess in (False, True):
        tag = "cost_grad_hess" if hess else "cost_grad"
        ts = repeat(lambda: cost(x0, obs, w1, want_hess=hess))
        tp = repeat(lambda: cost(x0, obs, wN, want_hess=hess))
        line(f"{name}_{tag}_device_1e6", {"shared": ts, "per_point": tp, "shared_points_per_s": N / ts["median_s"],
                                          "per_point_points_per_s": N / tp["median_s"],
                                          "per_point_over_shared": tp["median_s"] / ts["median_s"]})
    ts = repeat(lambda: solve(x0, obs, w1, lower=lo, upper=hi))
    tp, r = None, None
    tp = repeat(lambda: solve(x0, obs, wN, lower=lo, upper=hi))
    r = solve(x0, obs, wN, lower=lo, upper=hi)
    line(f"{name}_solve_device_1e6", {"shared": ts, "per_point": tp, "per_point_pixels_per_s": N / tp["median_s"],
                                      "per_point_over_shared": tp["median_s"] / ts["median_s"],
                                      "status_counts": np.bincount(r["status"].cpu().numpy(), minlength=4).tolist()})
    del x0, obs, wN, r
    torch.cuda.empty_cache()
    N = 100_000
    x0d, obsd, wNd = pixels(N)
    if spectra:
        line(f"{name}_curv_kernel_1e5", kernel_times(lambda: cost(x0d, obsd, wNd, want_hess=True),
                                                     ["k_forward_cost_curv_pw", "k_forward_cost_pw", "k_cost_hess"]))
    pin = lambda a: a.cpu().pin_memory().numpy()
    x0, obs, wN = pin(x0d), pin(obsd), pin(wNd)
    w1 = np.ascontiguousarray(wN[0])
    for hess in (False, True):
        tag = "cost_grad_hess" if hess else "cost_grad"
        ts = repeat(lambda: cost(x0, obs, w1, want_hess=hess))
        tp = repeat(lambda: cost(x0, obs, wN, want_hess=hess))
        out_b = 8 * (1 + D + (D * D if hess else 0))
        b_shared = 8 * (D + K) + out_b
        b_pp = 8 * (D + 2 * K) + out_b
        line(f"{name}_{tag}_host_1e5", {
            "shared": ts, "per_point": tp, "per_point_points_per_s": N / tp["median_s"],
            "per_point_over_shared": tp["median_s"] / ts["median_s"],
            "bytes_per_point_shared": b_shared, "bytes_per_point_per_point": b_pp, "h2d_gbs": pcie,
            "shared_of_pcie_bound": (b_shared * N / pcie / 1e9) / ts["median_s"],
            "per_point_of_pcie_bound": (b_pp * N / pcie / 1e9) / tp["median_s"]})
    ts = repeat(lambda: solve(x0, obs, w1, lower=np.zeros(D), upper=np.ones(D)))
    tp = repeat(lambda: solve(x0, obs, wN, lower=np.zeros(D), upper=np.ones(D)))
    line(f"{name}_solve_host_1e5", {"shared": ts, "per_point": tp, "per_point_pixels_per_s": N / tp["median_s"],
                                    "per_point_over_shared": tp["median_s"] / ts["median_s"]})
    torch.cuda.empty_cache()


def run_search(name, bank, spectra, lo, hi, line):
    import numpy as np
    import torch
    search = bank.forward_search if spectra else bank.search
    gen = torch.Generator("cuda").manual_seed(2)
    Dd = len(lo)
    lo_t, hi_t = torch.as_tensor(lo, device="cuda"), torch.as_tensor(hi, device="cuda")
    N, K, k = 100_000, 10_000, 8
    cand = lo_t + (hi_t - lo_t) * torch.rand(K, Dd, dtype=torch.float64, device="cuda", generator=gen)
    xt = lo_t + (hi_t - lo_t) * torch.rand(N, Dd, dtype=torch.float64, device="cuda", generator=gen)
    out = bank.predict(xt, want_var=False, want_deriv=False, project=spectra)
    obs = (out["fwd"] if spectra else out["mu"]).contiguous()
    obs = obs * (1 + 0.01 * torch.randn(obs.shape, dtype=torch.float64, device="cuda", generator=gen))
    wN = weights_like(obs, gen)
    w1 = wN[0].clone()
    ts = repeat(lambda: search(cand, obs, w1, k=k))
    tp = repeat(lambda: search(cand, obs, wN, k=k))
    kt = kernel_times(lambda: search(cand, obs, wN, k=k), ["k_search_topk", "k_search_operand_pw", "k_forward_cost"])
    line(f"{name}_search_device_1e5_K1e4_k8", {"shared": ts, "per_point": tp, "per_point_pairs_per_s": N * K / tp["median_s"],
                                               "shared_pairs_per_s": N * K / ts["median_s"],
                                               "per_point_over_shared": tp["median_s"] / ts["median_s"], "kernels": kt})


def main():
    import numpy as np
    import gp_emulator_b200 as g
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"config4": {"E": 20, "W": W, "M": M, "D": D}, "config5": {"E": 64, "M": M, "D": D}, "gpu": gpu_info()}
    line = lambda k, v: (res.__setitem__(k, v), print(k, json.dumps(v), flush=True))
    pcie = h2d_rate()
    line("h2d_page_locked_gbs", pcie)
    rs = np.random.RandomState(0)
    E = 20
    y = rs.random_sample((M, D))
    hyp = np.vstack([rs.random_sample((D, E)) * 2 - 3, np.ones((1, E)), np.full((1, E), -6.0)])
    wl = np.linspace(0, 1, W)
    B = np.linalg.qr(np.stack([np.cos(np.pi * (k + 1) * wl) for k in range(E)]).T)[0].T
    X = (np.sin(y @ rs.random_sample((D, E))) @ B) + 0.01 * rs.standard_normal((M, W))
    emu = g.MultivariateEmulator(X=X, y=y, hyperparams=hyp, basis_functions=B, n_pcs=E)
    run_config("config4", emu._device_bank(), True, line, pcie)
    del emu
    E5 = 64
    inputs = rs.random_sample((M, D))
    thetas = np.vstack([rs.random_sample((D, E5)) * 2 - 3, np.ones((1, E5))]).T
    invQts = rs.standard_normal((E5, M))
    run_config("config5", g.DeviceBank(inputs, thetas, invQts), False, line, pcie)
    E48 = 48
    run_search("bands48", g.DeviceBank(inputs, thetas[:E48], invQts[:E48]), False, np.zeros(D), np.ones(D), line)
    from tests.conftest import golden
    from tests.test_gpu_parity import _write_prosail_dump
    gp = golden("P")
    mv = g.MultivariateEmulator(X=None, y=None, dump=_write_prosail_dump(gp))
    run_search("prosail", mv._device_bank(), True, gp["y"].min(axis=0), gp["y"].max(axis=0), line)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
