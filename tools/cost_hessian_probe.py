"""Cost Hessian (gpe_bank_forward_cost_ex, gpe_bank_cost_ex) at config 4 (E = 20 PCs, W = 2101 wavelengths, M = 250,
D = 10) and config 5 (E = 64 bands, M = 250, D = 10), each beside the path it replaces, in one run.  Every timing:
warm-up, then CUDA events (device calls) or a host clock around calls that end synchronised (host calls), repeated
until the window is >= 1 s.

  device-resident:  cost + grad + hess, cost + grad alone, the bank's Hessian alone, and the materialise path
                    (predict(want_hess=True[, project_deriv=True]) + a torch reduction, in chunks)
  host-resident:    cost + grad + hess with one shared observation, cost + grad alone, and the materialise path to the
                    host + numpy
  one point:        MultivariateEmulator.cost(do_hess=True) against emu.predict + the PC Hessians + numpy
  kernels:          per-kernel times of one cost + grad + hess call from torch.profiler (separate pass); the Hessian
                    pass's FP64 rate against the live peaks of gpe_measure_fp64_peaks

Usage: python tools/cost_hessian_probe.py [out.json]   (the full result is printed as JSON; out.json: also written there)"""
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from tools.forward_cost_probe import gpu_info, timed_device, timed_host  # noqa: E402

W, M, D = 2101, 250, 10


def kernel_times(fn, reps=3):
    import torch
    from torch.profiler import profile, ProfilerActivity
    fn(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    kt = {}
    for ev in prof.key_averages():
        v = (getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)) / reps / 1e6
        if v > 0:
            kt[ev.key] = v
    return kt


def hessian_pass_share(kt, N, E, peaks):
    """The Hessian pass: every kernel but the mean + gradient pass (k_bank_mean), the forward cost, C and the reducer.
    Counted work per point and emulator: M (D (D + 1) / 2 + D) multiply-adds (the upper triangle of
    sum_j k_j a_j dx_j dx_j^T plus the distances; the kernels form the full D x D, so this is a lower bound)."""
    other = ("k_cost_hess", "k_forward_cost", "k_bank_mean", "k_bank_cost", "Memcpy", "Memset")
    names = [k for k in kt if not any(o in k for o in other)]
    hess_s = sum(kt[k] for k in names)
    if hess_s <= 0:
        return {"hessian_pass_s": None, "kernels": names}
    rate = 2.0 * N * E * M * (D * (D + 1) / 2 + D) / hess_s / 1e12
    return {"hessian_pass_s": hess_s, "kernels": names, "counted_tflops": rate,
            "share_of_live_dfma_peak": rate / peaks["dfma_tflops"], "share_of_live_dmma_peak": rate / peaks["dmma_tflops"]}


def main():
    import numpy as np
    import torch
    import gp_emulator_b200 as g
    from gp_emulator_b200 import _lib
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"config4": {"E": 20, "W": W, "M": M, "D": D}, "config5": {"E": 64, "M": M, "D": D}, "gpu": gpu_info()}
    peaks = _lib.measure_fp64_peaks(0)
    res["fp64_peaks_live"] = peaks
    line = lambda k, v: (res.__setitem__(k, v), print(k, json.dumps(v), flush=True))
    rs = np.random.RandomState(0)

    # ---- config 4: forward cost ---------------------------------------------------------------------------------------
    E = 20
    y = rs.random_sample((M, D))
    hyp = np.vstack([rs.random_sample((D, E)) * 2 - 3, np.ones((1, E)), np.full((1, E), -6.0)])
    wl = np.linspace(0, 1, W)
    B = np.linalg.qr(np.stack([np.cos(np.pi * (k + 1) * wl) for k in range(E)]).T)[0].T
    X = (np.sin(y @ rs.random_sample((D, E))) @ B) + 0.01 * rs.standard_normal((M, W))
    emu = g.MultivariateEmulator(X=X, y=y, hyperparams=hyp, basis_functions=B, n_pcs=E)
    bank = emu._device_bank()
    lam = torch.from_numpy(rs.random_sample(W) + 0.5).cuda()
    lam_np = lam.cpu().numpy()
    Bt = torch.from_numpy(B).cuda()

    N = 1_000_000
    t = torch.rand(N, D, dtype=torch.float64, device="cuda")
    obs1 = torch.from_numpy(emu.predict(np.full(D, 0.5), do_deriv=False)).cuda()
    s = timed_device(lambda: bank.forward_cost(t, obs1, lam, want_hess=True))
    line("c4_device_cost_grad_hess", {"N": N, "s": s, "points_per_s": N / s})
    s = timed_device(lambda: bank.forward_cost(t, obs1, lam))
    line("c4_device_cost_grad", {"N": N, "s": s, "points_per_s": N / s})
    s = timed_device(lambda: bank.predict(t, want_var=False, want_deriv=False, want_hess=True))
    line("c4_device_bank_mean_hess_alone", {"N": N, "s": s, "points_per_s": N / s})
    CH = 16384                                         # 2.75 GB of deriv_full per chunk

    def materialise(tt, obs):
        o = bank.predict(tt, want_var=False, want_deriv=False, want_hess=True, project=True, project_deriv=True)
        r = o["fwd"] - obs
        u = r * lam
        sv = u @ Bt.T                                                        # (n, E)
        J = o["deriv_full"]
        hess = torch.bmm(J * lam, J.transpose(1, 2)) + torch.einsum("nedk,ne->ndk", o["hess"], sv)
        return 0.5 * (u * r).sum(1), torch.bmm(J, u.unsqueeze(2)).squeeze(2), hess
    tc = t[:CH].contiguous()
    s = timed_device(lambda: materialise(tc, obs1))
    line("c4_device_materialise_and_reduce", {"N": CH, "s": s, "points_per_s": CH / s})
    new = bank.forward_cost(tc, obs1, lam, want_hess=True)
    old = materialise(tc, obs1)
    res["c4_device_agreement_max_rel"] = {k: float(((new[k] - o).abs().max() / o.abs().max()).item())
                                         for k, o in zip(("cost", "grad", "hess"), old)}
    kt = kernel_times(lambda: bank.forward_cost(t, obs1, lam, want_hess=True))
    line("c4_kernels", {"N": N, "kernel_s": kt, "hessian_pass": hessian_pass_share(kt, N, E, peaks)})

    NH = 200_000
    th = t[:NH].cpu().numpy()
    o1 = obs1.cpu().numpy()
    s = timed_host(lambda: bank.forward_cost(th, o1, lam_np, want_hess=True))
    line("c4_host_cost_grad_hess_shared_obs", {"N": NH, "s": s, "points_per_s": NH / s})
    s = timed_host(lambda: bank.forward_cost(th, o1, lam_np))
    line("c4_host_cost_grad_shared_obs", {"N": NH, "s": s, "points_per_s": NH / s})
    NB = 4096

    def host_materialise(tt, obs):
        o = bank.predict(tt, want_var=False, want_deriv=False, want_hess=True, project=True, project_deriv=True)
        r = o["fwd"] - obs
        u = lam_np * r
        J = o["deriv_full"]
        hess = np.einsum("ndw,w,nkw->ndk", J, lam_np, J, optimize=True) + np.einsum("nedk,ne->ndk", o["hess"], u @ B.T)
        return 0.5 * np.sum(u * r, axis=1), np.einsum("ndw,nw->nd", J, u), hess
    s = timed_host(lambda: host_materialise(th[:NB], o1))
    line("c4_host_materialise_and_reduce_shared_obs", {"N": NB, "s": s, "points_per_s": NB / s})

    y1 = th[0]

    def one_old():
        f, d = emu.predict(y1)
        hs = bank.predict(y1[None, :], want_var=False, want_deriv=False, want_hess=True)["hess"][0]
        r = f - o1
        u = lam_np * r
        return 0.5 * np.dot(u, r), d @ u, (d * lam_np) @ d.T + np.einsum("edk,e->dk", hs, B @ u)
    s_new = timed_host(lambda: emu.cost(y1, o1, lam_np, do_hess=True))
    s_grad = timed_host(lambda: emu.cost(y1, o1, lam_np))
    s_old = timed_host(one_old)
    line("c4_one_point_latency", {"cost_grad_hess_us": s_new * 1e6, "cost_grad_us": s_grad * 1e6,
                                  "predict_pc_hessians_numpy_us": s_old * 1e6})
    c1, g1, h1 = emu.cost(y1, o1, lam_np, do_hess=True)
    c0, g0, h0 = one_old()
    res["c4_one_point_agreement_rel"] = {"cost": abs(c1 - c0) / abs(c0), "grad": float(np.max(np.abs(g1 - g0)) / np.max(np.abs(g0))),
                                         "hess": float(np.max(np.abs(h1 - h0)) / np.max(np.abs(h0)))}
    del t, tc
    torch.cuda.empty_cache()

    # ---- config 5: band cost ------------------------------------------------------------------------------------------
    E5 = 64
    inputs = rs.random_sample((M, D))
    thetas = np.vstack([rs.random_sample((D, E5)) * 2 - 3, np.ones((1, E5))]).T
    invQts = rs.standard_normal((E5, M))
    bank5 = g.DeviceBank(inputs, thetas, invQts)
    t = torch.rand(N, D, dtype=torch.float64, device="cuda")
    w5 = torch.from_numpy(rs.random_sample(E5) + 0.5).cuda()
    ob5 = bank5.predict(t[:1], want_var=False, want_deriv=False)["mu"][0] * 1.1
    s = timed_device(lambda: bank5.cost(t, ob5, w5, want_hess=True))
    line("c5_device_cost_grad_hess", {"N": N, "s": s, "points_per_s": N / s})
    s = timed_device(lambda: bank5.cost(t, ob5, w5))
    line("c5_device_cost_grad", {"N": N, "s": s, "points_per_s": N / s})
    s = timed_device(lambda: bank5.predict(t, want_var=False, want_deriv=False, want_hess=True))
    line("c5_device_bank_mean_hess_alone", {"N": N, "s": s, "points_per_s": N / s})
    CH5 = 65536

    def materialise5(tt, obs):
        o = bank5.predict(tt, want_var=False, want_deriv=True, want_hess=True)
        r = o["mu"] - obs
        c = w5 * r
        G = o["deriv"]
        hess = torch.einsum("ne,nedk->ndk", c, o["hess"]) + torch.bmm(G.transpose(1, 2) * w5, G)
        return 0.5 * (c * r).sum(1), torch.einsum("ne,ned->nd", c, G), hess
    tc = t[:CH5].contiguous()
    s = timed_device(lambda: materialise5(tc, ob5))
    line("c5_device_materialise_and_reduce", {"N": CH5, "s": s, "points_per_s": CH5 / s})
    new = bank5.cost(tc, ob5, w5, want_hess=True)
    old = materialise5(tc, ob5)
    res["c5_device_agreement_max_rel"] = {k: float(((new[k] - o).abs().max() / o.abs().max()).item())
                                         for k, o in zip(("cost", "grad", "hess"), old)}
    kt = kernel_times(lambda: bank5.cost(t, ob5, w5, want_hess=True))
    line("c5_kernels", {"N": N, "kernel_s": kt, "hessian_pass": hessian_pass_share(kt, N, E5, peaks)})
    th = t[:NH].cpu().numpy()
    o5, w5n = ob5.cpu().numpy(), w5.cpu().numpy()
    s = timed_host(lambda: bank5.cost(th, o5, w5n, want_hess=True))
    line("c5_host_cost_grad_hess_shared_obs", {"N": NH, "s": s, "points_per_s": NH / s})
    s = timed_host(lambda: bank5.cost(th, o5, w5n))
    line("c5_host_cost_grad_shared_obs", {"N": NH, "s": s, "points_per_s": NH / s})

    def host_materialise5(tt, obs):
        o = bank5.predict(tt, want_var=False, want_deriv=True, want_hess=True)
        c = w5n * (o["mu"] - obs)
        G = o["deriv"]
        return np.einsum("ne,nedk->ndk", c, o["hess"]) + np.einsum("e,ned,nek->ndk", w5n, G, G, optimize=True)
    s = timed_host(lambda: host_materialise5(th[:NB], o5))
    line("c5_host_materialise_and_reduce_shared_obs", {"N": NB, "s": s, "points_per_s": NB / s})

    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
