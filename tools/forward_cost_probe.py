"""Forward cost (gpe_bank_forward_cost*) at config 4 (E = 20 PCs, W = 2101 wavelengths, M = 250, D = 10) against the
paths it replaces, in one run.  Every timing: warm-up, then CUDA events (device calls) or a host clock around calls that
end synchronised (host calls), repeated until the window is >= 1 s.

  device-resident, N = 1e7:  forward cost + gradient (shared obs), cost only, the bank mean + gradient alone (the bound of
                             the new path), and predict(project=True, project_deriv=True) + a torch reduction, in chunks
  device-resident, per-point obs, N = 2e6 (33.6 GB of spectra): forward cost + gradient
  host-resident:             shared obs and per-point obs (page-locked; against the measured H2D rate of this link),
                             against forward() (fwd + deriv_full to the host) + numpy
  one point:                 MultivariateEmulator.cost against emu.predict(y) + numpy
  kernel:                    k_forward_cost's own time from torch.profiler (separate pass), its share of the live DMMA peak

Usage: python tools/forward_cost_probe.py [out.json]   (the full result is printed as JSON; out.json: also written there)"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

E, W, M, D = 20, 2101, 250, 10


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def timed_device(fn, min_s=1.0):
    """Mean seconds per call of an asynchronous device call, CUDA events, window >= min_s."""
    import torch
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 1
    while True:
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        s = e0.elapsed_time(e1) / 1e3
        if s >= min_s:
            return s / reps
        reps = max(reps * 2, int(reps * min_s / max(s, 1e-6) * 1.1) + 1)


def timed_host(fn, min_s=1.0):
    """Mean seconds per call of a synchronous host call, window >= min_s."""
    fn()
    reps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < min_s:
        fn()
        reps += 1
    return (time.perf_counter() - t0) / reps


def main():
    import numpy as np
    import torch
    import gp_emulator_b200 as g
    from gp_emulator_b200 import _lib
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"config": {"E": E, "W": W, "M": M, "D": D}, "gpu": gpu_info()}
    peaks = _lib.measure_fp64_peaks(0)
    res["fp64_peaks_live"] = peaks
    rs = np.random.RandomState(0)
    y = rs.random_sample((M, D))
    hyp = np.vstack([rs.random_sample((D, E)) * 2 - 3, np.ones((1, E)), np.full((1, E), -6.0)])   # (D + 2, E)
    wl = np.linspace(0, 1, W)
    B = np.linalg.qr(np.stack([np.cos(np.pi * (k + 1) * wl) for k in range(E)]).T)[0].T               # (E, W) orthonormal
    X = (np.sin(y @ rs.random_sample((D, E))) @ B) + 0.01 * rs.standard_normal((M, W))
    emu = g.MultivariateEmulator(X=X, y=y, hyperparams=hyp, basis_functions=B, n_pcs=E)
    bank = emu._device_bank()
    lam = torch.from_numpy(rs.random_sample(W) + 0.5).cuda()
    lam_np = lam.cpu().numpy()
    line = lambda k, v: (res.__setitem__(k, v), print(k, json.dumps(v), flush=True))

    # ---- device-resident -------------------------------------------------------------------------------------------
    N = 10_000_000
    t = torch.rand(N, D, dtype=torch.float64, device="cuda")
    obs1 = torch.from_numpy(emu.predict(np.full(D, 0.5), do_deriv=False)).cuda()
    s = timed_device(lambda: bank.forward_cost(t, obs1, lam))
    line("device_cost_grad_shared_obs", {"N": N, "s": s, "points_per_s": N / s})
    s = timed_device(lambda: bank.forward_cost(t, obs1, lam, want_grad=False))
    line("device_cost_only_shared_obs", {"N": N, "s": s, "points_per_s": N / s})
    s = timed_device(lambda: bank.predict(t, want_var=False, want_deriv=True))
    line("device_bank_mean_grad_alone", {"N": N, "s": s, "points_per_s": N / s})
    s = timed_device(lambda: bank.predict(t, want_var=False, want_deriv=False))
    line("device_bank_mean_alone", {"N": N, "s": s, "points_per_s": N / s})
    CH = 65536                                         # materialise-and-reduce: 11 GB of deriv_full per chunk

    def materialise(tt, obs):
        o = bank.predict(tt, want_var=False, want_deriv=False, project=True, project_deriv=True)
        u = (o["fwd"] - obs) * lam
        cost = 0.5 * (u * (o["fwd"] - obs)).sum(1)
        grad = torch.bmm(o["deriv_full"], u.unsqueeze(2)).squeeze(2)
        return cost, grad
    tc = t[:CH].contiguous()
    s = timed_device(lambda: materialise(tc, obs1))
    line("device_materialise_and_reduce_shared_obs", {"N": CH, "s": s, "points_per_s": CH / s})

    def materialise_cost(tt, obs):
        f = bank.predict(tt, want_var=False, want_deriv=False, project=True)["fwd"] - obs
        return 0.5 * (lam * f * f).sum(1)
    s = timed_device(lambda: materialise_cost(tc, obs1))
    line("device_materialise_and_reduce_cost_only", {"N": CH, "s": s, "points_per_s": CH / s})
    c_new = bank.forward_cost(tc, obs1, lam)
    c_old, g_old = materialise(tc, obs1)
    res["device_agreement_max_rel"] = {
        "cost": float(((c_new["cost"] - c_old).abs().max() / c_old.abs().max()).item()),
        "grad": float(((c_new["grad"] - g_old).abs().max() / g_old.abs().max()).item())}
    del t

    NP = 2_000_000
    tp = torch.rand(NP, D, dtype=torch.float64, device="cuda")
    obsN = obs1.unsqueeze(0) * (1.0 + 0.05 * torch.randn(NP, W, dtype=torch.float64, device="cuda"))
    s = timed_device(lambda: bank.forward_cost(tp, obsN, lam))
    line("device_cost_grad_per_point_obs", {"N": NP, "s": s, "points_per_s": NP / s})
    tpc, opc = tp[:CH].contiguous(), obsN[:CH].contiguous()
    s = timed_device(lambda: materialise(tpc, opc))
    line("device_materialise_and_reduce_per_point_obs", {"N": CH, "s": s, "points_per_s": CH / s})

    # ---- kernel time (profiler pass of its own) ---------------------------------------------------------------------
    from torch.profiler import profile, ProfilerActivity
    tk = tp[:1_000_000].contiguous()
    bank.forward_cost(tk, obs1, lam); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            bank.forward_cost(tk, obs1, lam)
        torch.cuda.synchronize()
    kt = {}
    for ev in prof.key_averages():
        kt[ev.key] = (getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)) / 5 / 1e6
    fc = sum(v for k, v in kt.items() if "k_forward_cost<" in k or "k_forward_costILi" in k)
    useful = 4.0 * E * W * tk.shape[0]                  # fwd tile + s update, 2 E W flop each per point
    executed = 4.0 * 24 * 2176 * tk.shape[0]            # padded to 24 emulators (KS = 6) and Wp = 2176 columns
    line("kernel_k_forward_cost", {"N": tk.shape[0], "s": fc, "points_per_s": tk.shape[0] / fc if fc else None,
                                   "useful_tflops": useful / fc / 1e12 if fc else None,
                                   "executed_dmma_tflops": executed / fc / 1e12 if fc else None,
                                   "share_of_live_dmma_peak": executed / fc / 1e12 / peaks["dmma_tflops"] if fc else None,
                                   "all_kernels_s": {k: v for k, v in kt.items() if v > 0}})
    del tp, obsN, tk
    torch.cuda.empty_cache()

    # ---- host-resident ----------------------------------------------------------------------------------------------
    NH = 2_000_000
    th = rs.random_sample((NH, D))
    o1 = obs1.cpu().numpy()
    s = timed_host(lambda: bank.forward_cost(th, o1, lam_np))
    line("host_cost_grad_shared_obs", {"N": NH, "s": s, "points_per_s": NH / s})
    NHP = 100_000
    thp = torch.from_numpy(th[:NHP]).pin_memory().numpy()
    ohp = torch.empty(NHP, W, dtype=torch.float64).pin_memory().numpy()
    ohp[:] = o1 * (1.0 + 0.05 * rs.standard_normal((NHP, W)))
    s = timed_host(lambda: bank.forward_cost(thp, ohp, lam_np))
    src = torch.empty(1 << 27, dtype=torch.float64).pin_memory()           # 1 GB: this link's H2D rate, same run
    dst = torch.empty_like(src, device="cuda")
    h2d = src.numel() * 8 / timed_device(lambda: dst.copy_(src, non_blocking=True))
    bound = h2d / ((D + W) * 8)
    line("host_cost_grad_per_point_obs", {"N": NHP, "s": s, "points_per_s": NHP / s, "h2d_GBps": h2d / 1e9,
                                          "pcie_bound_points_per_s": bound, "fraction_of_pcie_bound": NHP / s / bound})
    NB = 16384

    def host_materialise(tt, obs):
        f, dfull = bank.forward(tt, want_deriv=True)
        r = f - obs
        u = lam_np * r
        return 0.5 * np.sum(u * r, axis=1), np.einsum("ndw,nw->nd", dfull, u)
    s = timed_host(lambda: host_materialise(th[:NB], o1))
    line("host_materialise_and_reduce_shared_obs", {"N": NB, "s": s, "points_per_s": NB / s})
    s = timed_host(lambda: host_materialise(thp[:NB], ohp[:NB]))
    line("host_materialise_and_reduce_per_point_obs", {"N": NB, "s": s, "points_per_s": NB / s})

    # ---- one point ----------------------------------------------------------------------------------------------------
    y1 = rs.random_sample(D)

    def one_old():
        f, d = emu.predict(y1)
        u = lam_np * (f - o1)
        return 0.5 * np.dot(u, f - o1), d @ u
    s_new = timed_host(lambda: emu.cost(y1, o1, lam_np))
    s_old = timed_host(one_old)
    line("one_point_latency", {"multivariate_cost_us": s_new * 1e6, "predict_plus_numpy_us": s_old * 1e6})
    c1, g1 = emu.cost(y1, o1, lam_np)
    c0, g0 = one_old()
    res["one_point_agreement_rel"] = {"cost": abs(c1 - c0) / abs(c0), "grad": float(np.max(np.abs(g1 - g0)) / np.max(np.abs(g0)))}

    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
