#!/usr/bin/env python
"""Headline benchmark: test-point predictions/sec (mean + variance + gradient, M=250, D=10, FP64).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

* workload = BASELINE.json configs[1]: the tests/benchmark.py-style synthetic GaussianProcess
  (M=250, D=10, all-U(0,1) model, seed 0), 1e8 FP64 test points PER GPU generated on the device
  (weak scaling: test points shard trivially, no data-path collective; rank 0 broadcasts the model once).
* a step = one pass of the fused predict kernel over the rank's 1e8 points (one kernel launch);
  `value` = points of all ranks / max-over-ranks device time (CUDA events on the launching stream).
* `e2e` = the same metric through the public drop-in API GaussianProcess.predict() with HOST buffers
  (pinned input, H2D + kernels + D2H inside the timed region) on --e2e-points points per GPU per step.
* `roofline`: the kernel is FP64-arithmetic bound (SURVEY.md section 8d); achieved = N * F(M, D) flop per
  launch / launch duration with F = 2M^2 + M(5D+6) + D + 1 = 139,011; peak = the DMMA (FP64 tensor)
  throughput of THIS GPU measured live by the library's micro-benchmark, because the driver-written
  MEASURED_PEAKS.json holds no FP64 figure.
* `configs`: the other BASELINE.json configurations on the same GPU, outside the headline's timed region -- cfg 1
  (N = 1e5 through the API), cfg 3 (M = 1000, FP64 and TF32), cfg 4 (20 PCs x 2101 wavelengths with back-projection,
  1e7 points in chunks; bound = HBM write), cfg 5 (bank of 64 GPs with gradient and Hessian, 1e7 points in chunks) --
  each with points/s, the kernel, a roofline and parity against the oracle.  `strong_scaling`: configs[1] as written
  (1e8 points in total, N/G per GPU).
* N > 1: `e2e` holds both "torchrun ranks" (every rank streams its own host buffers, max over ranks) and "one
  process" (rank 0 alone calls GaussianProcess(device=[0..N-1]).predict on host buffers: the drop-in call).
* `cpu_baseline` / `--impl reference`: the reference's numpy/scipy cpu_predict (restated in oracle/, the
  reference itself is Python 2 and cannot be imported) on the box's host cores, bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

M, D = 250, 10
F_PER_POINT = 2 * M * M + M * (5 * D + 6) + D + 1          # 139,011 flop (+ M exp), SURVEY.md section 8d
BYTES_PER_POINT = 8 * D + 8 * (2 + D)                      # 176 B
METRIC = "test-point predictions/sec (mean+var+grad, M=250, D=10, FP64)"
DUMP_POINTS = 1 << 19                                      # 12 doubles per point: 48 MiB of --dump-outputs at most


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=float, default=1e8, help="device-resident test points per GPU per step")
    ap.add_argument("--e2e-points", type=float, default=2e7, help="host-resident test points per GPU per step")
    ap.add_argument("--cpu-points", type=float, default=1e5, help="sample size of the CPU baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the cfg 1/3/4/5 block")
    ap.add_argument("--multi-points", type=float, default=1e7, help="host-resident points per GPU of the one-process e2e (N > 1)")
    ap.add_argument("--tripwire", type=int, default=100000, help="prefix and random-subset size of the oracle check")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed (rank 0) as DIR/<name>.npy in float64: "
                         "every point up to %d points, beyond that the same seeded sample of that many points" % DUMP_POINTS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(dirname, outputs, n):
    """Write outputs[name] (first axis = the step's n points) as dirname/<name>.npy, float64, on a fixed sample of rows
    so that two builds given the same arguments can be compared output for output."""
    os.makedirs(dirname, exist_ok=True)
    idx = np.arange(n) if n <= DUMP_POINTS else np.sort(np.random.default_rng(0).choice(n, DUMP_POINTS, replace=False))
    for name, a in outputs.items():
        if a is None:
            continue
        if hasattr(a, "cpu"):   # torch tensor: gather the sample on its device
            import torch
            a = a[torch.from_numpy(idx).to(a.device)].cpu().numpy()
        else:
            a = np.asarray(a)[idx]
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def workload_config(n_points):
    return {"workload": "cfg2 GaussianProcess S-model (tests/benchmark.py recipe, seed 0) M=250 D=10 FP64 "
                        "mu+var+grad, test points per GPU per step below, generated on device",
            "points_per_gpu_per_step": int(n_points),
            "l2": "inputs (%.1f GB per step) larger than L2" % (n_points * D * 8 / 1e9),
            "sharding": "contiguous test-point ranges per rank, model broadcast once, no data-path collective"}


def synthetic_model():
    # the reference benchmark's recipe (tests/benchmark.py:11-15, 28-29): everything U(0, 1), drawn in the order
    # inputs, testing, theta, invQ, invQt; legacy RandomState so the stream is the same on every numpy
    rs = np.random.RandomState(0)
    inputs = rs.random_sample((M, D))
    rs.random_sample((1, D))
    theta = rs.random_sample(D + 2)
    invQ = rs.random_sample((M, M))
    invQt = rs.random_sample(M)
    return {"inputs": inputs, "theta": theta, "invQ": invQ, "invQt": invQt}


# --------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (pynvml)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def _use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core BLAS can take."""
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=os.cpu_count())
        return max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    except Exception:
        return os.cpu_count()


def cpu_baseline(model, npts, repeats=3):
    """Reference cpu_predict semantics (oracle port) on the host cores; best of `repeats`."""
    from oracle import gp_oracle as orc
    threads = _use_all_host_threads()
    testing = np.random.RandomState(1).random_sample((int(npts), D))
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        orc.predict(model["inputs"], model["theta"], model["invQ"], model["invQt"], testing, chunk=100000)
        best = min(best, time.perf_counter() - t0)
    return {"value": npts / best, "unit": "points/s", "cores": int(threads), "kind": "port",
            "sample": "%d points of the same workload (one 1e5-point chunk, as the reference materialises (M,N) "
                      "matrices), best of %d; numpy/scipy cpu_predict restated from GaussianProcess.py:211-251" %
                      (int(npts), repeats)}


def flops_per_point(m, d, hess=False):
    """SURVEY.md section 8d: 2M^2 + M(5D+6) + D + 1 (+ M(D^2+2D) + D with the Hessian); exp evaluations not counted."""
    return 2 * m * m + m * (5 * d + 6) + d + 1 + ((m * (d * d + 2 * d) + d) if hess else 0)


def run_configs(torch, gpe, orc, dev_index, peaks, hbm_gbs, bf16_tflops):
    """BASELINE.json configs 1, 3, 4, 5 on one GPU: throughput, kernel, roofline, parity against the oracle."""
    dev = torch.device("cuda", dev_index)
    P64 = peaks["dmma_tflops"]
    out = {}

    def rate(fn, n_pts, reps=2, warm=1):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return n_pts * reps / (a.elapsed_time(b) * 1e-3)

    def tensor_roofline(pps, flop):
        ach = pps * flop / 1e12
        return {"bound": "tensor", "achieved": ach, "peak": P64, "unit": "TFLOP/s", "frac": ach / P64}

    def errs(got, ref):
        return {k: orc.ref_err(got[k].cpu().numpy() if hasattr(got[k], "cpu") else got[k], v) for k, v in ref.items()}

    # ---- cfg 1: the reference's own CPU-runnable case, N = 1e5, through the drop-in API with plain numpy arrays ------
    M, D, N = 250, 10, 100_000
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=0)
    gp = gpe.GaussianProcess(inputs, [], device=dev_index)
    gp.theta, gp.invQ, gp.invQt = theta, invQ, invQt
    for _ in range(3):
        res = gp.predict(testing)
    t0 = time.perf_counter()
    for _ in range(5):
        res = gp.predict(testing)
    api_pps = 5 * N / (time.perf_counter() - t0)
    t0 = time.perf_counter()
    mu_o, var_o, der_o = orc.predict(inputs, theta, invQ, invQt, testing, chunk=100000)
    cpu_s = time.perf_counter() - t0
    td = torch.from_numpy(testing).to(dev)
    dm = gp._device_model()
    dev_pps = rate(lambda: dm.predict(td), N, reps=20, warm=3)
    out["cfg1"] = {"workload": "GaussianProcess S-model (tests/benchmark.py recipe, seed 0) M=250 D=10, 1e5 test points, FP64 mu+var+grad",
                   "api_numpy_points_per_s": api_pps, "device_resident_points_per_s": dev_pps, "kernel": dm.plan(N),
                   "roofline": tensor_roofline(dev_pps, flops_per_point(M, D)),
                   "oracle_cpu_points_per_s": N / cpu_s,
                   "parity_vs_oracle": errs(dict(zip(("mu", "var", "deriv"), res)), {"mu": mu_o, "var": var_o, "deriv": der_o}),
                   "note": "api = GaussianProcess.predict(numpy in, numpy out): H2D + kernel + D2H + result arrays per call; "
                           "parity over all 1e5 points"}
    del td, gp, dm

    # ---- cfg 3: M = 1000, variance dominated; FP64 and single precision (tcgen05 / TF32) ------------------------------
    M, D, N = 1000, 10, 10_000_000
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, 2000, seed=3)
    m = gpe.DeviceModel(inputs, theta, invQt, invQ, device=dev_index)
    mu_o, var_o, der_o = orc.predict(inputs, theta, invQ, invQt, testing)
    par64 = errs(m.predict(testing), {"mu": mu_o, "var": var_o, "deriv": der_o})
    t = torch.rand(N, D, dtype=torch.float64, device=dev)
    pps64 = rate(lambda: m.predict(t), N, reps=2, warm=1)
    t32 = t.to(torch.float32)
    del t
    o32 = m.predict_f32(testing.astype(np.float32))
    o32x = m.predict_f32(testing.astype(np.float32), fast=False)
    ref32 = dict(zip(("mu", "var", "deriv"), orc.predict(inputs, theta, invQ, invQt, testing.astype(np.float32).astype(np.float64))))
    pps32 = rate(lambda: m.predict_f32(t32), N, reps=3, warm=1)
    pps32x = rate(lambda: m.predict_f32(t32, fast=False), N, reps=2, warm=1)
    tf_peak = bf16_tflops / 2.0 if bf16_tflops else None
    tf_ach = pps32 * 2 * 1024 * 1024 / 1e12
    out["cfg3"] = {"workload": "M=1000 D=10 S-model, 1e7 device-resident test points, mu+var+grad",
                   "fp64": {"points_per_s": pps64, "kernel": m.plan(N), "roofline": tensor_roofline(pps64, flops_per_point(M, D)),
                            "parity_vs_oracle": par64},
                   "tf32": {"points_per_s": pps32, "points_per_s_3xtf32": pps32x,
                            "kernel": "k_predict_tf32_big<DP=12,X3=false> (tcgen05.mma kind::tf32, TMEM accumulators, column passes)",
                            "roofline": {"bound": "tensor", "achieved": tf_ach, "peak": tf_peak, "unit": "TFLOP/s",
                                         "frac": (tf_ach / tf_peak) if tf_peak else None,
                                         "note": "executed TF32 flop (2*Mp^2 per point, Mp=1024) / time; peak = half the measured bf16 "
                                                 "rate of MEASURED_PEAKS.json (no TF32 figure there); the kernel is bound by the FP32 "
                                                 "issue rate of K* generation, not by the tensor pipe (DESIGN 4.3c)"},
                            "error_vs_fp64_oracle": errs(o32, ref32), "error_vs_fp64_oracle_3xtf32": errs(o32x, ref32),
                            "stated_bound": "variance 2^-11 relative to max|var| (one TF32 pass); reference FP32 pass bar 1e-5 "
                                            "(tests/benchmark.py:56) met by mean/gradient, and by the variance with the 3x split at M <= 256"}}
    del t32, m

    # ---- cfg 4: MultivariateEmulator, 20 PCs x 2101 wavelengths, 1e7 test inputs, batched predict + back-projection ----
    M, D, P, W, N, CH = 250, 10, 20, 2101, 10_000_000, 200_000
    rs = np.random.RandomState(4)
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((P, D + 2)); invQts = rs.random_sample((P, M)); invQs = rs.random_sample((P, M, M))
    basis = np.linalg.qr(rs.standard_normal((W, P)))[0].T.copy()
    bank = gpe.DeviceBank(inputs, thetas, invQts, invQs, basis=basis, device=dev_index)
    tt = rs.random_sample((64, D))
    models = [(inputs, thetas[i], invQs[i], invQts[i]) for i in range(P)]
    fwd_o, mu_o, var_o, grad_o, dfull_o = orc.mv_predict_batch(models, basis, tt, want_deriv_full=True)
    got = bank.predict(tt, want_var=True, want_deriv=True, project=True, project_deriv=True)
    par4 = errs(got, {"fwd": fwd_o, "mu": mu_o, "var": var_o, "deriv": grad_o, "deriv_full": dfull_o})
    t = torch.rand(N, D, dtype=torch.float64, device=dev)
    lib = _lib_handle()
    mu_b = torch.empty(CH, P, dtype=torch.float64, device=dev); der_b = torch.empty(CH, P, D, dtype=torch.float64, device=dev)
    fwd_b = torch.empty(CH, W, dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream(dev_index).cuda_stream

    def cfg4_pass(project=True, grad=True):
        for c0 in range(0, N, CH):      # the 168 GB of spectra are produced chunk-wise into one 3.4 GB buffer
            _check(lib.gpe_bank_predict_ex(bank._h, t[c0:c0 + CH].data_ptr(), CH, mu_b.data_ptr(), None,
                                           der_b.data_ptr() if grad else None, None, fwd_b.data_ptr() if project else None, None,
                                           0x01 | (0x04 if grad else 0) | (0x10 if project else 0), st))
    pps4 = rate(cfg4_pass, N, reps=1, warm=1)
    pps4_pc = rate(lambda: cfg4_pass(False), N, reps=1, warm=0)
    pps4_fwd = rate(lambda: cfg4_pass(True, False), N, reps=1, warm=0)   # MultivariateEmulator.predict(do_deriv=False)
    proj_s = 1.0 / pps4 - 1.0 / pps4_pc
    out["cfg4"] = {"workload": "MultivariateEmulator bank P=20 PCs, W=2101 wavelengths, M=250 D=10; 1e7 device-resident test inputs in "
                               "chunks of 2e5: PC means + PC gradients + back-projected spectra fwd (N, 2101)",
                   "points_per_s": pps4, "pc_space_only_points_per_s": pps4_pc,
                   "forward_only_points_per_s": pps4_fwd,
                   "forward_only_note": "PC means (no gradients) + spectra: k_bank_mean<10,10,false>, 23 FP64 instructions per "
                                        "(pair, PC); MultivariateEmulator.predict(do_deriv=False) on a batch",
                   "kernel": "k_bank_mean<10,5,true> (groups of 5 PCs share x_j - t_n; blockIdx.y = group) + k_project_tma<5,1> "
                             "(tensor-map TMA stores)",
                   "roofline": {"bound": "hbm", "achieved": W * 8 / proj_s / 1e9 if proj_s > 0 else None, "peak": hbm_gbs, "unit": "GB/s",
                                "frac": (W * 8 / proj_s / 1e9 / hbm_gbs) if proj_s > 0 else None,
                                "note": "the back-projection kernel alone: algorithmic bytes = 8 W = 16,808 B of spectrum written per "
                                        "point (SURVEY 8d) / its time (step with projection - step without, CUDA events); peak = "
                                        "MEASURED_PEAKS.json hbm_gbs"},
                   "step_roofline": {"bound": "fp64 pipe (instruction issue)", "achieved": pps4_pc * P * M * 36 / 1e12,
                                     "peak": peaks["dfma_tflops"] / 2.0, "unit": "T FP64 instr/s",
                                     "frac": pps4_pc * P * M * 36 / 1e12 / (peaks["dfma_tflops"] / 2.0),
                                     "spectra_GBps_whole_step": pps4 * W * 8 / 1e9,
                                     "note": "the STEP is bound by the P = 20 mean + gradient evaluations, not by the projection "
                                             "(%.0f %% of its time): 36 FP64 instructions per (test, train) pair and PC (2D + 12 + 2D/5: the "
                                             "differences are shared by 5 PCs; 43 in the one-emulator kernel) against the "
                                             "measured DFMA instruction rate" % (100.0 * pps4 / pps4_pc)},
                   "parity_vs_oracle": par4}
    # host-resident: numpy in, PC-space outputs out (1,760 B per point back over PCIe), chunk walk below the C ABI
    Nh = 2_000_000
    h_in = torch.rand(Nh, D, dtype=torch.float64).pin_memory().numpy()
    h_out = {"mu": torch.empty(Nh, P, dtype=torch.float64).pin_memory().numpy(),
             "deriv": torch.empty(Nh, P, D, dtype=torch.float64).pin_memory().numpy()}
    bank.predict(h_in, want_var=False, out=h_out)
    t0 = time.perf_counter()
    bank.predict(h_in, want_var=False, out=h_out)
    out["cfg4"]["host_resident_pc_space_points_per_s"] = Nh / (time.perf_counter() - t0)
    out["cfg4"]["host_resident_note"] = ("pinned numpy in/out through gpe_bank_predict_ex(GPE_HOST_PTRS); %d B per point D2H: the PCIe "
                                         "link (~55 GB/s) allows %.2e points/s" % (8 * P * (1 + D), 55e9 / (8 * P * (1 + D))))
    del t, mu_b, der_b, fwd_b, bank, h_in, h_out

    # ---- cfg 5: per-band bank of 64 GPs sharing test inputs, mean + variance + gradient + Hessian --------------------
    sms = torch.cuda.get_device_properties(dev_index).multi_processor_count
    M, D, E, N, CH = 250, 10, 64, 10_000_000, 64 * sms * 10     # chunks of ten whole waves of 64-point tiles (94,720 points)
    thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)); invQs = rs.random_sample((E, M, M))
    bank = gpe.DeviceBank(inputs, thetas, invQts, invQs, device=dev_index)
    tt = rs.random_sample((40, D))
    models = [(inputs, thetas[i], invQs[i], invQts[i]) for i in range(E)]
    mu_o, var_o, grad_o, hess_o = orc.bank_predict(models, tt, do_hess=True)
    got = bank.predict(tt, want_var=True, want_deriv=True, want_hess=True)
    par5 = errs(got, {"mu": mu_o, "var": var_o, "deriv": grad_o, "hess": hess_o})
    t = torch.rand(N, D, dtype=torch.float64, device=dev)
    ob = {"mu": torch.empty(CH, E, dtype=torch.float64, device=dev), "var": torch.empty(CH, E, dtype=torch.float64, device=dev),
          "deriv": torch.empty(CH, E, D, dtype=torch.float64, device=dev), "hess": torch.empty(CH, E, D, D, dtype=torch.float64, device=dev)}

    def cfg5_pass(n_total):
        for c0 in range(0, n_total, CH):   # 573 GB of outputs in total: produced chunk-wise into one 5.4 GB set of buffers
            n = min(CH, n_total - c0)
            _check(lib.gpe_bank_predict_ex(bank._h, t[c0:c0 + n].data_ptr(), n, ob["mu"].data_ptr(), ob["var"].data_ptr(),
                                           ob["deriv"].data_ptr(), ob["hess"].data_ptr(), None, None, 0x0F, st))
    cfg5_pass(2 * CH)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); cfg5_pass(N); b.record(); torch.cuda.synchronize()
    pps5 = N / (a.elapsed_time(b) * 1e-3)
    out["cfg5"] = {"workload": "bank of 64 S-model GPs sharing 1e7 device-resident test inputs (chunks of 94,720 = ten whole waves of 64-point tiles), M=250 D=10 FP64, "
                               "mu+var+grad+Hessian = 112 doubles per point per emulator",
                   "points_per_s": pps5, "emulator_points_per_s": pps5 * E,
                   "kernel": "64 x k_predict_full<4,8,2,4,10,1,2,true,false,true> (fused Hessian, phase C) per chunk",
                   "roofline": tensor_roofline(pps5 * E, flops_per_point(M, D, hess=True)),
                   "output_GBps": pps5 * E * 112 * 8 / 1e9, "parity_vs_oracle": par5}
    del ob
    # 5b: the same bank consumed on the fly (cost + gradient per point), device- and host-resident
    Nc = 2_000_000
    obs_v = mu_o.mean(axis=0)
    c_o, g_o = orc.bank_cost(models, tt, obs_v)
    oc = bank.cost(tt, obs_v)
    obs_d = torch.from_numpy(obs_v).to(dev)
    pps5b = rate(lambda: bank.cost(t[:Nc], obs_d), Nc, reps=2, warm=1)
    h_in = torch.rand(Nc, D, dtype=torch.float64).pin_memory().numpy()
    bank.cost(h_in, obs_v)
    t0 = time.perf_counter()
    bank.cost(h_in, obs_v)
    out["cfg5"]["on_the_fly_cost"] = {"device_resident_points_per_s": pps5b, "host_resident_points_per_s": Nc / (time.perf_counter() - t0),
                                      "kernel": "k_bank_mean<10,5,true> (groups of 5 emulators on shared differences) + k_bank_cost", "bytes_out_per_point": 8 * (1 + D),
                                      "parity_vs_oracle": {"cost": orc.ref_err(oc["cost"], c_o), "grad": orc.ref_err(oc["grad"], g_o)},
                                      "note": "gpe_bank_cost / gpe_bank_cost_host: least-squares misfit of the 64 means against one observed "
                                              "vector + its gradient, reduced on the device (88 B per point instead of 5.6 KB)"}
    return out


def _lib_handle():
    from gp_emulator_b200 import _lib
    return _lib.load()


def _check(rc):
    from gp_emulator_b200 import _lib
    _lib.check(rc)


def run_reference(args, rank, world):
    if rank != 0:
        return
    model = synthetic_model()
    from oracle import gp_oracle as orc
    npts = int(args.cpu_points)
    threads = _use_all_host_threads()
    testing = np.random.RandomState(1).random_sample((npts, D))
    for _ in range(args.warmup):
        orc.predict(model["inputs"], model["theta"], model["invQ"], model["invQt"], testing[:20000])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = orc.predict(model["inputs"], model["theta"], model["invQ"], model["invQt"], testing, chunk=100000)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("mu", "var", "deriv"), res)), npts)
    value = npts * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.points),
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": int(threads), "kind": "port",
                         "sample": "each step = %d points of the workload on the host CPU (the reference materialises "
                                   "(M,N) matrices, 1e8 points would need 200 GB); numpy/scipy cpu_predict restated "
                                   "in oracle/ (the reference is Python 2 and cannot be imported)" % npts},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch ourselves under torchrun the way the driver does
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29533"),
               os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import gp_emulator_b200 as gpe
    from gp_emulator_b200 import _lib, sharding

    # stdout carries exactly one JSON line: keep NCCL's version banner (NCCL_DEBUG=VERSION prints it there) off it
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    # one process per GPU: keep each rank (and the page-locked buffers it touches first) on its GPU's NUMA node
    numa_cpus = sharding.bind_host_to_gpu(local_rank) if (world > 1 and not os.environ.get("GPE_NO_NUMA_BIND")) else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    model = synthetic_model() if rank == 0 else None
    if world > 1:
        # NCCL initialises lazily and may print (version banner, NCCL_DEBUG output) on fd 1: point fd 1 at stderr
        # until the communicator exists, so that stdout carries exactly one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            host_group = dist.new_group(backend="gloo")   # CPU-side barrier for the phase where rank 0 drives every GPU
            model = sharding.broadcast_model(model, src=0, device=dev)   # the only collective on the path
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    gp = gpe.GaussianProcess(model["inputs"], [], device=local_rank)
    gp.theta, gp.invQ, gp.invQt = model["theta"], model["invQ"], model["invQt"]   # tests/benchmark.py:11-15
    dm = gp._device_model()
    lib = _lib.load()

    N = int(args.points)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    testing = torch.rand(N, D, dtype=torch.float64, device=dev, generator=gen)   # 8 GB >> 126 MB L2
    peaks = gpe.measure_fp64_peaks(local_rank) if rank == 0 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident: `value` and the roofline ------------------------------------------------
    out = None
    for _ in range(args.warmup):
        out = dm.predict(testing)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib.gpe_launch_count()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    evs[0].record()
    for i in range(args.steps):
        out = dm.predict(testing)
        evs[i + 1].record()
    barrier()
    launches = lib.gpe_launch_count() - launches0
    sampler.stop_flag = True
    sampler.join()
    step_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    total_ms = evs[0].elapsed_time(evs[-1])
    if world > 1:
        total_ms = sharding.max_over_ranks(total_ms, device=dev)
    # correctness tripwire inside the bench (SURVEY 8d, cfg 2): a prefix and a random subset of the step's points
    # against the oracle, all three outputs (rank 0)
    trip = None
    if rank == 0:
        nt = min(int(args.tripwire), N)
        idx = torch.cat([torch.arange(nt, device=dev),
                         torch.randint(0, N, (nt,), device=dev, generator=torch.Generator(device=dev).manual_seed(7))])
        trip = {"t": testing[idx].cpu().numpy(), "mu": out["mu"][idx].cpu().numpy(), "var": out["var"][idx].cpu().numpy(),
                "deriv": out["deriv"][idx].cpu().numpy(), "n_prefix": nt, "n_random": nt}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, out, N)
    # ---- configs[1] as written: 1e8 points IN TOTAL, N/G per GPU (strong scaling) ---------------------------------
    strong = None
    Ns = int(round(1e8)) // world
    if Ns <= N:
        ts = testing[:Ns]
        dm.predict(ts)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            dm.predict(ts)
        e1.record()
        barrier()
        s_ms = e0.elapsed_time(e1)
        if world > 1:
            s_ms = sharding.max_over_ranks(s_ms, device=dev)
        strong = {"total_points_per_step": Ns * world, "points_per_gpu_per_step": Ns, "value": Ns * world * args.steps / (s_ms * 1e-3),
                  "unit": "points/s", "ms_per_step": s_ms / args.steps, "scaling": "strong",
                  "note": "BASELINE configs[1] literally: 1e8 test points sharded N/G per GPU, device-resident, max over ranks"}
        del ts
    del out
    torch.cuda.empty_cache()

    # ---- end to end through the public API with host buffers ------------------------------------
    Ne = int(args.e2e_points)
    host_in = torch.rand(Ne, D, dtype=torch.float64).pin_memory().numpy()
    # result buffers are allocated once, page-locked, outside the timed region (a fresh 2 GB pinned allocation
    # costs more than the whole step); every step still moves all inputs H2D and all results D2H
    host_out = {"mu": torch.empty(Ne, dtype=torch.float64).pin_memory().numpy(),
                "var": torch.empty(Ne, dtype=torch.float64).pin_memory().numpy(),
                "deriv": torch.empty(Ne, D, dtype=torch.float64).pin_memory().numpy()}
    for _ in range(max(1, min(args.warmup, 2))):
        gp.predict(host_in, out=host_out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        mu_h, var_h, der_h = gp.predict(host_in, out=host_out)   # H2D + kernels + D2H, returns numpy arrays
        _ = float(mu_h[-1]) + float(der_h[-1, -1])               # the results are on the host
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        e2e_s = sharding.max_over_ranks(e2e_s, device=dev)
    ranks_e2e = Ne * world * args.steps / e2e_s
    # ---- N > 1: the drop-in call itself -- ONE process, ONE GaussianProcess.predict over all N GPUs (gpe_multi_*) ----
    one_proc = None
    if world > 1:
        del host_in, host_out, mu_h, var_h, der_h
        dist.barrier(group=host_group)
        if rank == 0:
            Nm = int(args.multi_points) * world
            gpm = gpe.GaussianProcess(model["inputs"], [], device=list(range(world)))
            gpm.theta, gpm.invQ, gpm.invQt = model["theta"], model["invQ"], model["invQt"]
            m_in = torch.rand(Nm, D, dtype=torch.float64).pin_memory().numpy()
            m_out = {"mu": torch.empty(Nm, dtype=torch.float64).pin_memory().numpy(),
                     "var": torch.empty(Nm, dtype=torch.float64).pin_memory().numpy(),
                     "deriv": torch.empty(Nm, D, dtype=torch.float64).pin_memory().numpy()}
            gpm.predict(m_in, out=m_out)
            l0 = lib.gpe_launch_count()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                mu_m, var_m, der_m = gpm.predict(m_in, out=m_out)
                _ = float(mu_m[-1]) + float(der_m[-1, -1])
            one_s = time.perf_counter() - t0
            # the fan-out must reproduce one GPU bit for bit: check a slice against this rank's single-device model
            chk = dm.predict(torch.from_numpy(m_in[:100000]).to(dev))
            same = all(bool(np.array_equal(chk[k].cpu().numpy(), m_out[k][:100000])) for k in ("mu", "var", "deriv"))
            one_proc = {"value": Nm * args.steps / one_s, "unit": "points/s", "points_per_step": Nm,
                        "h2d_bytes_per_step": Nm * D * 8, "d2h_bytes_per_step": Nm * (2 + D) * 8,
                        "launches": int(lib.gpe_launch_count() - l0), "bit_identical_to_one_gpu": same,
                        "api": "ONE process: GaussianProcess(inputs, targets, device=[0..%d]).predict(pinned numpy in, pinned out) -> "
                               "gpe_multi_predict: one pipeline thread per GPU pulling chunks from a shared cursor" % (world - 1)}
            del m_in, m_out, gpm
        dist.barrier(group=host_group)
    # the same call the way a reference user makes it: plain (pageable) numpy in, fresh numpy arrays out
    pageable_rate = None
    if world == 1:
        Np = min(Ne, 2_000_000)
        plain_in = np.array(host_in[:Np])
        for _ in range(4):   # repeated calls of one size get page-locked result arrays from the 2nd call on (engine._auto_pin);
            mu_p, var_p, der_p = gp.predict(plain_in)   # let torch's pinned cache fill before timing the steady state
        t0 = time.perf_counter()
        for _ in range(3):
            mu_p, var_p, der_p = gp.predict(plain_in)
        pageable_rate = 3 * Np / (time.perf_counter() - t0)
        del plain_in, mu_p, var_p, der_p
        del host_in, host_out

    # ---- opt-in variants of the same workload, reported beside the headline (short, outside every timed region) --
    variants = None
    if rank == 0:
        def _rate(fn, n_pts, reps=3):
            fn(); fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            return n_pts * reps / (a.elapsed_time(b) * 1e-3)
        nv = min(N, 20_000_000)
        tv = testing[:nv]
        sym = gpe.DeviceModel(model["inputs"], model["theta"], model["invQt"], model["invQ"], device=local_rank,
                              symmetric_variance=True)
        t32 = tv.to(torch.float32)
        nh = min(nv, 4_000_000)   # the (N, D, D) Hessian output is 800 B per point
        hout = {"hess": torch.empty(nh, D, D, dtype=torch.float64, device=tv.device)}
        variants = {
            "points": nv,
            "fp64_symmetric_variance_points_per_s": _rate(lambda: sym.predict(tv), nv),
            "fp32_3xtf32_tcgen05_points_per_s": _rate(lambda: dm.predict_f32(t32), nv),
            "fp32_1xtf32_tcgen05_points_per_s": _rate(lambda: dm.predict_f32(t32, fast=True), nv),
            "fp64_mean_gradient_only_points_per_s": _rate(lambda: dm.predict(tv, want_var=False), nv),
            "fp64_with_hessian_points_per_s": _rate(lambda: dm.predict(tv[:nh], want_hess=True, out=hout), nh),
            "note": "same model and test points; symmetric = opt-in upper-triangular fold of invQ (exact identity, "
                    "half the DMMAs); with_hessian = mean + variance + gradient + (N, D, D) Hessian in one fused launch; tf32 = single precision with the variance contraction on tcgen05/TMEM (3x split: var error "
                    "~3e-6, meets the reference FP32 bar 1e-5; 1x: ~6e-5)",
        }
        del sym, t32, tv, hout
        # the caller on the input side of the path (SURVEY 8f-1): cost + gradient of the hyper-parameter fit, one
        # (theta, target) problem per SM, timed through the C ABI with host buffers (wall clock, synchronous call)
        from gp_emulator_b200.training import DeviceTrainer
        rs_t = np.random.RandomState(1)
        nprob = torch.cuda.get_device_properties(local_rank).multi_processor_count
        trainer = DeviceTrainer(model["inputs"], np.sin(model["inputs"].sum(axis=1)), device=local_rank)
        thetas = 5.0 * (rs_t.random_sample((nprob, D + 2)) - 0.5)
        trainer.evaluate(thetas)
        t0 = time.perf_counter()
        for _ in range(5):
            trainer.evaluate(thetas)
        variants["training_objective_evaluations_per_s"] = 5 * nprob / (time.perf_counter() - t0)
        variants["training_note"] = ("loglikelihood + partial_devs (GaussianProcess.py:78-125) for %d thetas per launch, "
                                     "M=%d D=%d: block Gauss-Jordan on DMMA, k_train_eval" % (nprob, M, D))
        trainer.close()
    if rank == 0:
        from oracle import gp_oracle as orc
        _use_all_host_threads()
        mu_o, var_o, der_o = orc.predict(model["inputs"], model["theta"], model["invQ"], model["invQt"], trip["t"], chunk=100000)
        parity = {"mu": orc.ref_err(trip["mu"], mu_o), "var": orc.ref_err(trip["var"], var_o),
                  "deriv": orc.ref_err(trip["deriv"], der_o), "points_checked": int(trip["t"].shape[0]),
                  "what": "%d-point prefix + %d random indices of rank 0's %d points of the last timed step, metric "
                          "max|x - ref| / max|ref| (tests/benchmark.py:51-53), bar 1e-10" % (trip["n_prefix"], trip["n_random"], N)}
        value = N * world * args.steps / (total_ms * 1e-3)
        kern_ms = float(np.mean(step_ms))
        achieved = N * F_PER_POINT / (kern_ms * 1e-3) / 1e12
        peak = peaks["dmma_tflops"]
        # DRAM traffic cannot be observed without a profiler attached: it is IMPORTED from the committed ncu capture of
        # this kernel (profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per point) and scaled to N
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj["dram_bytes_per_point"] * N
                traffic_src = "imported, not measured in this run: %s" % tj.get("source", "profiles/traffic.json")
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(N),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "note": "FP64: achieved = N*139011 flop / mean launch time (CUDA events, one launch per step); "
                                 "peak = DMMA.8x8x4 rate measured live on this GPU (MEASURED_PEAKS.json has no FP64 "
                                 "figure); DFMA peak %.1f, SM %.0f MHz under FP64 load" %
                                 (peaks["dfma_tflops"], peaks["sm_mhz_fp64_load"]),
                         "kernel": dm.plan(N), "kernel_ms": kern_ms,
                         "hbm_GBps": N * BYTES_PER_POINT / (kern_ms * 1e-3) / 1e9},
            "e2e": {"value": ranks_e2e, "unit": "points/s",
                    "h2d_bytes_per_step": Ne * D * 8, "d2h_bytes_per_step": Ne * (2 + D) * 8,
                    "points_per_gpu_per_step": Ne, "mode": "torchrun ranks" if world > 1 else "one process, one GPU",
                    "torchrun_ranks_points_per_s": ranks_e2e, "one_process_all_gpus": one_proc,
                    "pageable_numpy_points_per_s": pageable_rate,   # pageable inputs, fresh result arrays per call (steady state)
                    "host_numa_binding": ("rank pinned to the %d CPUs local to its GPU" % len(numa_cpus)) if numa_cpus else None,
                    "api": "GaussianProcess.predict(numpy pinned in, preallocated pinned out) -> libgpemu two-slot stream pipeline"},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "parity_vs_oracle": parity,
            "variants": variants,
        }
        if one_proc is not None and one_proc["value"] > ranks_e2e:
            # the headline e2e is the call a drop-in user makes: one process, one predict over all N GPUs
            line["e2e"].update({"value": one_proc["value"], "mode": "one process, gpe_multi (GaussianProcess(device=[0..N-1]))",
                                "h2d_bytes_per_step": one_proc["h2d_bytes_per_step"],
                                "d2h_bytes_per_step": one_proc["d2h_bytes_per_step"]})
        line["strong_scaling"] = strong
        if not args.no_cpu_baseline and world == 1:   # reported on rank 0 at N=1 only
            line["cpu_baseline"] = cpu_baseline(model, int(args.cpu_points))
        if not args.no_configs and world == 1:
            del testing
            torch.cuda.empty_cache()
            hbm = bf16 = None
            try:
                mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
                hbm, bf16 = float(mp["hbm_gbs"]), float(mp.get("bf16_tflops_sustained", mp.get("bf16_tflops")))
            except Exception:
                hbm = 6550.0     # the figure B200_PROFILING.md quotes for this pool when the file is absent
            line["configs"] = run_configs(torch, gpe, orc, local_rank, peaks, hbm, bf16)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
