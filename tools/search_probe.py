"""Candidate search (gpe_bank_search: DeviceBank.search / forward_search, invert(candidates=...)) at config 4 (E = 20 PCs,
W = 2101 wavelengths, M = 250, D = 10, spectrum cost) and config 5 (E = 64 bands, band cost), each beside the path it
replaces, in one run.  The GPU name and power limit are read in the same run.

  device-resident:  N = 1e6 pixels, K = 1e4 and 1e5 candidates, k = 1 and 8, CUDA tensors; wall time of the whole call
                    (table, pixel operand, top-k, exact costs of the k winners) and, from a torch.profiler pass, the time of
                    k_search_topk alone.  Pairs/s = N K / time; share of the live DMMA peak at 2 (E + 1) flop per pair.
                    Beside it (a) the torch route a user writes today -- fwd of the candidates, a chunked FP64 matmul over
                    W, torch.topk -- and (b) the same PC-space algorithm unfused in torch (matmul over E, topk), both per
                    pair on a slice of the pixels
  host-resident:    N = 1e5 per-point spectra from numpy (pageable and page-locked) against the PCIe bound (the spectra's
                    bytes over the measured H2D rate)
  one pixel:        search and invert(candidates=...) of one spectrum against a table of K = 1e4
  end to end:       invert from a seeded lhd table (K = 1e4, n_starts 1 and 4) against invert from the box centre, N = 1e4
                    noise-free pixels with x_true over the whole box; config 4 and the PROSAIL golden model; wall time and
                    the fraction of pixels within 1e-6 of the box width of x_true

Usage: python tools/search_probe.py [out.json]"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from tools.forward_cost_probe import gpu_info  # noqa: E402

W, M, D = 2101, 250, 10


def wall(fn, reps=3):
    import torch
    ts, r = [], None
    fn()
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return min(ts), r


def kernel_time(fn, name):
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    tot = {}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
        tot[ev.key] = tot.get(ev.key, 0.0) + us * 1e-6
    return {k: v for k, v in tot.items() if name in k}


def torch_routes(bank, spectra, cand, obs, weights, k, n_slice):
    """(a) materialised fwd + chunked matmul over the observation width + topk, (b) PC-space matmul + topk; seconds per
    pair on the first n_slice pixels."""
    import torch
    Kc = cand.shape[0]
    o = obs[:n_slice]
    w = weights
    out = {}

    def route_a():
        f = bank.predict(cand, want_var=False, want_deriv=False, want_mu=not spectra, project=spectra)
        f = f["fwd"] if spectra else f["mu"]
        half = 0.5 * torch.sum(w * f * f, dim=1)
        best = []
        for c0 in range(0, o.shape[0], 2048):
            sc = half[None, :] - (o[c0:c0 + 2048] * w) @ f.T
            best.append(torch.topk(sc, k, dim=1, largest=False).indices)
        return torch.cat(best)

    def route_b():
        m = bank.predict(cand, want_var=False, want_deriv=False)["mu"]
        if spectra:
            Bm = torch.as_tensor(bank_basis[id(bank)], device=o.device)
            Cm = (Bm * w) @ Bm.T
            a = 0.5 * torch.sum((m @ Cm) * m, dim=1)
            s = -((o * w) @ Bm.T)
        else:
            a = 0.5 * torch.sum(w * m * m, dim=1)
            s = -(o * w)
        best = []
        for c0 in range(0, o.shape[0], 65536):
            sc = a[None, :] + s[c0:c0 + 65536] @ m.T
            best.append(torch.topk(sc, k, dim=1, largest=False).indices)
        return torch.cat(best)

    for name, fn in (("a_materialise_matmul_W_topk", route_a), ("b_pc_space_matmul_topk_unfused", route_b)):
        t, _ = wall(fn, reps=2)
        out[name] = {"pixels": n_slice, "s": t, "pairs_per_s": n_slice * Kc / t}
    return out


bank_basis = {}


def run_config(name, bank, spectra, E, rs, res, line, peak):
    import numpy as np
    import torch
    dev = torch.device("cuda", 0)
    Kw = W if spectra else E
    search = bank.forward_search if spectra else bank.search
    N = 1_000_000
    x_true = torch.as_tensor(rs.random_sample((N, D)), device=dev)
    out = bank.predict(x_true, want_var=False, want_deriv=False, want_mu=True, project=spectra)
    obs = (out["fwd"] if spectra else out["mu"]).contiguous()
    del out
    weights = torch.as_tensor(rs.uniform(0.5, 2.0, Kw), device=dev)
    for K in (10_000, 100_000):
        cand = torch.as_tensor(rs.random_sample((K, D)), device=dev)
        for k in (1, 8):
            t, r = wall(lambda: search(cand, obs, weights, k=k), reps=2)
            kt = kernel_time(lambda: search(cand, obs, weights, k=k), "k_search_topk")
            ktopk = sum(kt.values())
            flop = 2.0 * (E + 1) * N * K
            row = {"N": N, "K": K, "k": k, "call_s": t, "pairs_per_s_call": N * K / t, "k_search_topk_s": ktopk,
                   "pairs_per_s_topk_kernel": N * K / ktopk if ktopk else None,
                   "topk_kernel_dmma_share": flop / ktopk / (peak * 1e12) if ktopk else None,
                   "bound": "FP64 tensor (DMMA) compute: 2 (E + 1) flop per pair; table bytes per CTA are reused by 128 pixels"}
            if k == 8:
                row["torch"] = torch_routes(bank, spectra, cand, obs, weights, k, 10_000 if spectra else 200_000)
            line(f"{name}_device_K{K}_k{k}", row)
        del cand
    # host-resident, N = 1e5 per-point observations
    Nh = 100_000
    cand = rs.random_sample((10_000, D))
    oh = obs[:Nh].cpu().numpy()
    wh = weights.cpu().numpy()
    pinned = torch.empty(oh.shape, dtype=torch.float64).pin_memory()
    pinned.numpy()[:] = oh
    dst = torch.empty(oh.shape, dtype=torch.float64, device=dev)
    th2d, _ = wall(lambda: dst.copy_(pinned, non_blocking=True))
    tp, _ = wall(lambda: search(cand, oh, wh, k=8), reps=2)
    tl, _ = wall(lambda: search(cand, pinned.numpy(), wh, k=8), reps=2)
    td, _ = wall(lambda: search(torch.as_tensor(cand, device=dev), dst, weights, k=8), reps=2)
    line(f"{name}_host_N1e5_K1e4_k8", {"pageable_s": tp, "pinned_s": tl, "device_resident_s": td,
                                       "obs_h2d_alone_s": th2d, "pcie_bound_pixels_per_s": Nh / th2d,
                                       "pinned_pixels_per_s": Nh / tl})
    del obs, x_true
    torch.cuda.empty_cache()


def end_to_end(name, bank, spectra, lo, hi, res, line):
    import numpy as np
    import scipy.stats
    import gp_emulator_b200 as g
    width = hi - lo
    np.random.seed(17)
    table = g.lhd(dist=[scipy.stats.uniform(loc=l, scale=s) for l, s in zip(lo, width)], size=10_000)
    rs = np.random.RandomState(23)
    N = 10_000
    x_true = lo + width * rs.uniform(0, 1, (N, len(lo)))
    f = bank.predict(x_true, want_var=False, want_deriv=False, want_mu=not spectra, project=spectra)
    obs = f["fwd"] if spectra else f["mu"]
    solve = bank.forward_invert if spectra else bank.invert
    row = {"N": N, "K": 10_000}
    runs = {"box_centre": lambda: solve(np.tile(0.5 * (lo + hi), (N, 1)), obs, lower=lo, upper=hi, max_iter=100)}
    for ns in (1, 4):
        runs[f"candidates_n_starts_{ns}"] = lambda ns=ns: solve(None, obs, lower=lo, upper=hi, max_iter=100, candidates=table,
                                                                n_starts=ns)
    for key, fn in runs.items():
        t, r = wall(fn, reps=1)
        err = np.max(np.abs(r["x"] - x_true) / width, axis=1)
        row[key] = {"s": t, "fraction_within_1e-6": float(np.mean(err <= 1e-6)),
                    "fraction_within_1e-8": float(np.mean(err <= 1e-8))}
    line(f"end_to_end_{name}", row)


def main():
    import numpy as np
    import gp_emulator_b200 as g
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"config4": {"E": 20, "W": W, "M": M, "D": D}, "config5": {"E": 64, "M": M, "D": D}, "gpu": gpu_info()}
    line = lambda k, v: (res.__setitem__(k, v), print(k, json.dumps(v), flush=True))
    peaks = g.measure_fp64_peaks(0)
    line("fp64_peaks", peaks)
    rs = np.random.RandomState(0)
    E = 20
    y = rs.random_sample((M, D))
    hyp = np.vstack([rs.random_sample((D, E)) * 2 - 3, np.ones((1, E)), np.full((1, E), -6.0)])
    wl = np.linspace(0, 1, W)
    B = np.linalg.qr(np.stack([np.cos(np.pi * (k + 1) * wl) for k in range(E)]).T)[0].T
    X = (np.sin(y @ rs.random_sample((D, E))) @ B) + 0.01 * rs.standard_normal((M, W))
    emu = g.MultivariateEmulator(X=X, y=y, hyperparams=hyp, basis_functions=B, n_pcs=E)
    bank4 = emu._device_bank()
    bank_basis[id(bank4)] = B
    run_config("config4", bank4, True, E, rs, res, line, peaks["dmma_tflops"])

    # one pixel, K = 1e4
    cand = rs.random_sample((10_000, D))
    obs1 = emu.predict(rs.random_sample(D), do_deriv=False)
    ts, _ = wall(lambda: emu.search(obs1, candidates=cand, k=4), reps=20)
    ti, _ = wall(lambda: emu.invert(obs1, bounds=(np.zeros(D), np.ones(D)), candidates=cand), reps=20)
    tf, _ = wall(lambda: emu.cost(cand[:1], obs1, do_deriv=False), reps=20)
    line("one_pixel_K1e4", {"search_k4_s": ts, "invert_from_candidates_s": ti, "one_point_cost_s": tf})

    end_to_end("config4", bank4, True, np.zeros(D), np.ones(D), res, line)
    from tests.test_gpu_parity import _write_prosail_dump
    from tests.conftest import golden
    gp = golden("P")
    mv = g.MultivariateEmulator(X=None, y=None, dump=_write_prosail_dump(gp))
    end_to_end("prosail", mv._device_bank(), True, gp["y"].min(axis=0), gp["y"].max(axis=0), res, line)

    E5 = 64
    inputs = rs.random_sample((M, D))
    thetas = np.vstack([rs.random_sample((D, E5)) * 2 - 3, np.ones((1, E5))]).T
    invQts = rs.standard_normal((E5, M))
    run_config("config5", g.DeviceBank(inputs, thetas, invQts), False, E5, rs, res, line, peaks["dmma_tflops"])
    if out_path:
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
