"""Parity of the CUDA path (through the C ABI) with the oracle and the frozen reference outputs.

FP64 tolerance: 1e-10 in the reference's own metric max|x - ref| / max|ref| (tests/benchmark.py:51-53;
north_star asks <= 1e-10 relative), and for the variance of genuinely conditioned models the
condition-scaled metric of SURVEY.md section 8d (|dvar| / (b + |k|^T |invQ| |k|)) <= 1e-10.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import gp_oracle as orc
from tests.conftest import golden

pytestmark = pytest.mark.gpu
TOL = 1e-10


@pytest.fixture(scope="module")
def gpemu(lib):
    import gp_emulator_b200 as g
    assert lib.gpe_device_count() > 0, "no GPU visible: the gpu tests must not pass on a fallback"
    return g


def _check(out, ref_mu, ref_var, ref_deriv, tol=TOL):
    assert orc.ref_err(out["mu"], ref_mu) < tol
    assert orc.ref_err(out["deriv"], ref_deriv) < tol
    if ref_var is not None:
        assert orc.ref_err(out["var"], ref_var) < tol


@pytest.mark.parametrize("tag", ["S250", "S1000", "S37", "S1500"])
def test_golden_S(gpemu, tag):
    g = golden(tag)
    inputs, theta, invQ, invQt, testing = orc.make_S_model(int(g["M"]), int(g["D"]), int(g["N"]), int(g["seed"]))
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    out = m.predict(testing, want_hess="hess" in g)
    _check(out, g["mu"], g["var"], g["deriv"])
    if "hess" in g:
        nh = g["hess"].shape[0]
        assert orc.ref_err(out["hess"][:nh], g["hess"]) < TOL


def test_golden_T_trained_model(gpemu):
    g = golden("T")
    m = gpemu.DeviceModel(g["inputs"], g["theta"], g["invQt"], g["invQ"])
    out = m.predict(g["testing"], want_hess=True)
    assert orc.ref_err(out["mu"], g["mu"]) < TOL
    assert orc.ref_err(out["deriv"], g["deriv"]) < TOL
    assert orc.ref_err(out["hess"], g["hess"]) < TOL
    assert orc.var_cond_err(out["var"], g["var"], g["inputs"], g["theta"], g["invQ"], g["testing"]) < TOL
    # against the extended-precision arbiter: no worse than 2x numpy's own error (SURVEY.md section 8d)
    lmu, lvar, _ = orc.predict_longdouble(g["inputs"], g["theta"], g["invQ"], g["invQt"], g["testing"])
    e_np = np.max(np.abs(g["var"] - lvar))
    e_gpu = np.max(np.abs(out["var"] - lvar))
    assert e_gpu <= 2.0 * e_np + 1e-18


def test_golden_prosail_bank_and_projection(gpemu):
    g = golden("P")
    y, hyp, B, P = g["y"], g["hyperparams"], g["basis_functions"], int(g["n_pcs"])
    invQs = np.stack([orc.prepare_likelihood(y, g["train_data"][i], hyp[:, i])[0] for i in range(P)])
    bank = gpemu.DeviceBank(y, hyp.T, g["invQt"], invQs, basis=B)
    out = bank.predict(g["testing"], want_var=True, want_deriv=True)
    assert orc.ref_err(out["mu"], g["pc_mu"]) < TOL
    assert orc.ref_err(out["deriv"], g["pc_deriv"]) < TOL
    for i in range(P):
        assert orc.var_cond_err(out["var"][:, i], g["pc_var"][:, i], y, hyp[:, i], invQs[i], g["testing"]) < TOL
    outp = bank.predict(g["points"], want_var=False, want_deriv=False, project=True, project_deriv=True)
    assert orc.ref_err(outp["fwd"], g["fwd"]) < TOL
    assert orc.ref_err(outp["deriv_full"][:, :, g["wsub"]], g["deriv_sub"]) < TOL
    gp0 = gpemu.DeviceModel(y, hyp[:, 0], g["invQt"][0])
    assert orc.ref_err(gp0.predict(g["testing"][:8], want_var=False, want_deriv=False, want_hess=True)["hess"],
                       g["hess0"]) < TOL


@pytest.mark.parametrize("M,D,N", [(1, 1, 1), (3, 2, 5), (31, 7, 63), (32, 5, 64), (33, 9, 65), (250, 10, 1000),
                                   (256, 10, 129), (257, 11, 70), (300, 12, 100), (512, 4, 40), (513, 6, 33),
                                   (777, 13, 50), (1000, 10, 130), (1024, 16, 20), (100, 20, 70), (90, 32, 40)])
def test_shapes_against_oracle(gpemu, M, D, N):
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=M + D)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    out = m.predict(testing)
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
    _check(out, mu, var, deriv)
    out2 = m.predict(testing, want_var=False)            # mean-only kernel
    assert orc.ref_err(out2["mu"], mu) < TOL and orc.ref_err(out2["deriv"], deriv) < TOL
    if D <= 16:
        h = m.predict(testing, want_mu=False, want_var=False, want_deriv=False, want_hess=True)["hess"]
        assert orc.ref_err(h, orc.hessian(inputs, theta, invQt, testing)) < TOL


def test_wide_length_scales_and_far_points(gpemu):
    """exp underflow, huge distances and tiny kernels must stay finite and match."""
    rs = np.random.RandomState(5)
    inputs = rs.random_sample((64, 4)) * 10
    theta = np.array([3.0, -4.0, 0.5, 6.0, 1.0, -5.0])
    invQ = rs.standard_normal((64, 64)); invQt = rs.standard_normal(64)
    testing = np.vstack([rs.random_sample((30, 4)) * 10, rs.random_sample((5, 4)) * 1e3, inputs[:5]])
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    out = m.predict(testing)
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
    assert np.all(np.isfinite(out["mu"])) and np.all(np.isfinite(out["var"])) and np.all(np.isfinite(out["deriv"]))
    assert np.max(np.abs(out["mu"] - mu)) <= TOL * max(1.0, np.max(np.abs(mu)))
    assert np.max(np.abs(out["var"] - var)) <= TOL * np.max(np.abs(var))
    assert np.max(np.abs(out["deriv"] - deriv)) <= TOL * max(1.0, np.max(np.abs(deriv)))


def test_empty_and_tiny_inputs(gpemu):
    inputs, theta, invQ, invQt, testing = orc.make_S_model(50, 3, 4, seed=1)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    out = m.predict(np.zeros((0, 3)))
    assert out["mu"].shape == (0,) and out["deriv"].shape == (0, 3)
    out = m.predict(testing[:1])
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing[:1])
    _check(out, mu, var, deriv)
    with pytest.raises(ValueError):
        m.predict(np.zeros((3, 4)))
    m2 = gpemu.DeviceModel(inputs, theta, invQt)  # no invQ uploaded
    with pytest.raises(gpemu.GpemuError):
        m2.predict(testing, want_var=True)


def test_device_pointers_equal_host_streaming_and_shard_invariance(gpemu):
    import torch
    # (60,001 points: every shard below stays on the plan of the whole call -- the 64-point tiles; the plans for a few
    # thousand and for a few hundred points have summation orders of their own and agree with it to rounding only)
    NP = 60_001
    inputs, theta, invQ, invQt, testing = orc.make_S_model(250, 10, NP, seed=8)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    host = m.predict(testing)
    t = torch.from_numpy(testing).cuda()
    dev = m.predict(t)
    torch.cuda.synchronize()
    for k in ("mu", "var", "deriv"):
        assert np.array_equal(dev[k].cpu().numpy(), host[k]), k
    # 1-way result must equal any G-way contiguous split bit for bit (points are independent)
    from gp_emulator_b200.sharding import shard_range
    for world in (2, 3, 8):
        parts = [m.predict(t[slice(*shard_range(NP, r, world))]) for r in range(world)]
        for k in ("mu", "var", "deriv"):
            assert torch.equal(torch.cat([p[k] for p in parts]), dev[k]), (world, k)


def test_pageable_and_pinned_host_paths_multi_chunk(gpemu):
    import torch
    inputs, theta, invQ, invQt, _ = orc.make_S_model(64, 6, 1, seed=3)
    N = (1 << 18) * 2 + 12345       # three pipeline chunks
    testing = np.random.RandomState(0).random_sample((N, 6))
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    a = m.predict(testing)
    tp = torch.from_numpy(testing).pin_memory()
    b = m.predict(tp.numpy())
    for k in ("mu", "var", "deriv"):
        assert np.array_equal(a[k], b[k])
    idx = np.r_[0:50, (1 << 18) - 25:(1 << 18) + 25, N - 50:N]
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing[idx])
    assert orc.ref_err(a["mu"][idx], mu) < TOL and orc.ref_err(a["var"][idx], var) < TOL
    assert orc.ref_err(a["deriv"][idx], deriv) < TOL


def test_bank_host_batches_are_chunked(gpemu, monkeypatch):
    """numpy callers of a bank get their batch walked in chunks BELOW the C ABI (gpe_bank_predict_ex with host pointers:
    H2D / kernels / D2H overlapped, chunk size bounded by the width of the outputs): same values as the device-pointer
    call, every output key, ragged last chunk, pageable and page-locked result arrays."""
    import torch
    rs = np.random.RandomState(12)
    M, D, E, W, N = 60, 4, 5, 300, 1037
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)); invQs = rs.random_sample((E, M, M))
    basis = rs.standard_normal((E, W))
    bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=basis)
    t = rs.random_sample((N, D))
    kw = dict(want_var=True, want_deriv=True, want_hess=True, project=True, project_deriv=True)
    ref = {k: v.cpu().numpy() for k, v in bank.predict(torch.from_numpy(t).cuda(), **kw).items()}
    one = bank.predict(t, **kw)                                            # one chunk
    monkeypatch.setenv("GPE_SLOT_OUT_BYTES", str(8 * 100 * (E * (2 + D + D * D) + W + D * W)))   # 100 points per chunk
    got = bank.predict(t, **kw)                                            # 11 chunks, staged (pageable) path
    pin = bank.predict(torch.from_numpy(t).pin_memory().numpy(), pinned=True, **kw)   # 11 chunks, direct DMA path
    assert set(got) == set(ref) == set(one) == set(pin)
    for k in ref:
        for name, r in (("one", one), ("chunked", got), ("pinned", pin)):
            assert r[k].shape == ref[k].shape and np.array_equal(r[k], ref[k]), (name, k)
    # without the variance the bank's means / gradients come from the shared-difference kernel (predict_bank_mean.cuh):
    # bit-identical between host and device callers of the same request, equal to the variance path to rounding
    ref_nv = {k: v.cpu().numpy() for k, v in bank.predict(torch.from_numpy(t).cuda(), want_var=False, want_deriv=True,
                                                          project=True, project_deriv=True).items()}
    assert orc.ref_err(ref_nv["fwd"], ref["fwd"]) < 1e-13 and orc.ref_err(ref_nv["deriv_full"], ref["deriv_full"]) < 1e-13
    # forward only: the means-only variant of that kernel (larger groups, k * alpha fused into the accumulation)
    ref_f = bank.predict(torch.from_numpy(t).cuda(), want_var=False, want_deriv=False, want_mu=False, project=True)
    fwd = bank.predict(t, want_var=False, want_deriv=False, want_mu=False, project=True)
    assert set(fwd) == {"fwd"} and np.array_equal(fwd["fwd"], ref_f["fwd"].cpu().numpy())  # PC means stay on the device
    assert orc.ref_err(fwd["fwd"], ref_nv["fwd"]) < 1e-13
    f2, d2 = bank.forward(t)
    assert np.array_equal(f2, ref_nv["fwd"]) and np.array_equal(d2, ref_nv["deriv_full"])
    monkeypatch.delenv("GPE_SLOT_OUT_BYTES")
    models = [(inputs, thetas[e], invQs[e], invQts[e]) for e in range(E)]
    mu_o, var_o, grad_o, hess_o = orc.bank_predict(models, t[:200], do_hess=True)
    assert orc.ref_err(got["mu"][:200], mu_o) < TOL and orc.ref_err(got["hess"][:200], hess_o) < TOL


@pytest.mark.parametrize("M,D,E,N", [(60, 4, 5, 1037), (250, 10, 64, 3000), (33, 1, 1, 7), (40, 32, 3, 129)])
def test_bank_cost_reduction_on_the_fly(gpemu, M, D, E, N):
    """gpe_bank_cost: misfit against observations and its gradient, reduced over the emulators on the device, equals
    the E separate predicts + numpy reduction a caller of the reference would write (oracle bank_cost)."""
    import torch
    rs = np.random.RandomState(M + E)
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)); invQs = rs.random_sample((E, M, M))
    bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs)
    t = rs.random_sample((N, D))
    models = [(inputs, thetas[e], invQs[e], invQts[e]) for e in range(E)]
    mu_o = orc.bank_predict(models, t)[0]
    obs1 = mu_o.mean(axis=0) * 1.1                         # one observed vector for every point
    obsN = mu_o * (1.0 + 0.2 * rs.standard_normal(mu_o.shape))
    w = rs.random_sample(E) + 0.5
    for obs, wt in ((obs1, None), (obsN, w), (obs1, w)):
        c_o, g_o = orc.bank_cost(models, t, obs, wt)
        got = bank.cost(t, obs, wt)
        assert got["cost"].shape == (N,) and got["grad"].shape == (N, D)
        assert orc.ref_err(got["cost"], c_o) < TOL and orc.ref_err(got["grad"], g_o) < TOL
    only = bank.cost(t, obs1, want_grad=False)
    assert set(only) == {"cost"} and orc.ref_err(only["cost"], orc.bank_cost(models, t, obs1)[0]) < TOL
    td = torch.from_numpy(t).cuda()
    dev = bank.cost(td, torch.from_numpy(obsN).cuda(), torch.from_numpy(w).cuda())       # device in, device out
    c_o, g_o = orc.bank_cost(models, t, obsN, w)
    assert dev["cost"].is_cuda and orc.ref_err(dev["cost"].cpu().numpy(), c_o) < TOL
    assert orc.ref_err(dev["grad"].cpu().numpy(), g_o) < TOL
    with pytest.raises(ValueError):
        bank.cost(t, np.zeros(E + 1))


def test_device_exp_accuracy(lib, gpemu):
    """The FP64 exp routines behind K* (gpe_math.cuh) against mpmath on [-708, 0]: the table-driven exp_neg_tab of the
    predict kernels <= 1.3 ulp, the polynomial exp_neg <= 1 ulp; exactly 1 at 0, flush to 0 below the normal range."""
    import mpmath as mp
    mp.mp.prec = 120
    rs = np.random.RandomState(3)
    x = np.concatenate([-rs.uniform(0, 708, 30000), -rs.uniform(0, 40, 30000), -10.0 ** rs.uniform(-300, 0, 2000),
                        np.array([0.0, -0.0, -708.0, -707.999, -1e-320, -np.log(2) / 2, -np.log(2) / 128, -745.0, -1e4])])
    ref = [mp.exp(mp.mpf(float(v))) for v in x]
    lib.gpe_debug_exp.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int]
    for which, bound in ((0, 1.3), (1, 1.0)):
        y = np.empty_like(x)
        assert lib.gpe_debug_exp(x.ctypes.data, y.ctypes.data, x.size, which) == 0
        worst = 0.0
        for v, got, r in zip(x, y, ref):
            if v < -708.0:
                assert got == 0.0
                continue
            worst = max(worst, float(abs(mp.mpf(float(got)) - r) / np.spacing(float(r))))
        assert y[np.where(x == 0.0)[0][0]] == 1.0
        assert worst <= bound, (which, worst)


def test_tiny_host_calls_run_on_mapped_buffers(gpemu):
    """Host calls of a few points (the reference's usual call is ONE point) skip the copy engine: the kernels read and
    write the library's page-locked staging buffers directly.  Same numbers as the DMA path that page-locked caller
    arrays take, for every output, at the sizes around the switch (16384 points)."""
    import torch
    inputs, theta, invQ, invQt, testing = orc.make_S_model(120, 6, 16385, seed=31)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    for n in (1, 7, 300, 16384, 16385):
        t = testing[:n]
        got = m.predict(t, want_hess=True, pinned=False)                    # pageable in / out: mapped buffers up to 16384
        tp = torch.from_numpy(t).pin_memory().numpy()
        ref = m.predict(tp, want_hess=True, pinned=True)                    # page-locked in / out: direct DMA
        for k in ("mu", "var", "deriv", "hess"):
            assert np.array_equal(got[k], ref[k]), (n, k)
        mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, t)
        _check(got, mu, var, deriv)
    g32 = m.predict_f32(testing[:3].astype(np.float32))
    assert orc.ref_err(g32["mu"], orc.predict(inputs, theta, invQ, invQt, testing[:3])[0]) < 1e-5


def test_small_batch_plan_threshold(gpemu):
    """Calls of up to 3 * 16 * #SM points run 16-point tiles (lower latency), larger ones 64-point tiles; both sides of
    the switch meet the oracle, and a host call uses one plan for all of its chunks."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    inputs, theta, invQ, invQt, _ = orc.make_S_model(250, 10, 1, seed=17)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    rs = np.random.RandomState(18)
    for N in (48 * sms, 48 * sms + 1):
        testing = rs.random_sample((N, 10))
        out = m.predict(testing)
        idx = np.r_[0:40, N // 2:N // 2 + 40, N - 40:N]
        mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing[idx])
        assert orc.ref_err(out["mu"][idx], mu) < TOL and orc.ref_err(out["var"][idx], var) < TOL
        assert orc.ref_err(out["deriv"][idx], deriv) < TOL
        dev = m.predict(torch.from_numpy(testing).cuda())
        assert np.array_equal(dev["var"].cpu().numpy(), out["var"])


def test_bank_forward_single_call(gpemu):
    """gpe_bank_forward (what MultivariateEmulator.predict runs on for host callers): same values as the two-step
    device path, for one point, a few, and more than one internal chunk; Jacobian optional."""
    rs = np.random.RandomState(13)
    M, D, E, W = 60, 4, 5, 300
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)); invQs = rs.random_sample((E, M, M))
    basis = rs.standard_normal((E, W))
    bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=basis)
    for N in (1, 7, 6001):
        t = rs.random_sample((N, D))
        ref = bank.predict(t, want_var=False, want_deriv=False, project=True, project_deriv=True)
        fwd, dfull = bank.forward(t)
        assert np.array_equal(fwd, ref["fwd"]) and np.array_equal(dfull, ref["deriv_full"]), N
        # forward only: the means-only kernel variant (its own rounding); same request through predict: same bits
        f_only = bank.forward(t, want_deriv=False)
        assert np.array_equal(f_only, bank.predict(t, want_var=False, want_deriv=False, want_mu=False, project=True)["fwd"])
        assert orc.ref_err(f_only, ref["fwd"]) < 1e-13
    models = [(inputs, thetas[i], invQs[i], invQts[i]) for i in range(E)]
    t = rs.random_sample((3, D))
    fwd, dfull = bank.forward(t)
    for k in range(3):
        f_o, d_o = orc.mv_predict_point(models, basis, t[k])
        assert orc.ref_err(fwd[k], f_o) < TOL and orc.ref_err(dfull[k], d_o) < TOL


def test_staged_pipeline_chunk_seams(gpemu):
    """Pageable callers go through the three-slot staged pipeline (copy-in thread / GPU / copy-out thread).  Sizes
    around its chunking decisions must give bit-identical results to the device-resident call, repeatedly (slot
    reuse across calls), for every output combination."""
    import torch
    inputs, theta, invQ, invQt, _ = orc.make_S_model(64, 5, 1, seed=9)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    lib = gpemu._lib.load()
    wave = 64 * torch.cuda.get_device_properties(0).multi_processor_count
    rs = np.random.RandomState(2)
    for N in (1, 3 * wave, 3 * wave + 1, 8 * wave - 1, 8 * wave, 12 * wave + 7, 4 * (1 << 18) + 1, 777_777):
        testing = rs.random_sample((N, 5))
        dev = m.predict(torch.from_numpy(testing).cuda(), want_hess=True)
        torch.cuda.synchronize()
        for rep in range(2):
            host = m.predict(testing, want_hess=True)
            for k in ("mu", "var", "deriv", "hess"):
                assert np.array_equal(host[k], dev[k].cpu().numpy()), (N, rep, k)
        h2 = m.predict(testing, want_mu=False, want_var=True, want_deriv=False)
        assert set(h2) == {"var"} and np.array_equal(h2["var"], dev["var"].cpu().numpy())


def test_staged_pipeline_concurrent_models(gpemu):
    """Two models streaming pageable batches from two Python threads share the copy pool."""
    import threading
    res = {}
    def work(seed):
        inputs, theta, invQ, invQt, _ = orc.make_S_model(80, 4, 1, seed=seed)
        testing = np.random.RandomState(seed).random_sample((400_000, 4))
        m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
        out = m.predict(testing)
        idx = np.r_[0:40, 200_000:200_040, 399_960:400_000]
        mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing[idx])
        res[seed] = max(orc.ref_err(out["mu"][idx], mu), orc.ref_err(out["var"][idx], var), orc.ref_err(out["deriv"][idx], deriv))
    th = [threading.Thread(target=work, args=(s,)) for s in (21, 22, 23)]
    for t in th: t.start()
    for t in th: t.join()
    assert len(res) == 3 and max(res.values()) < TOL, res


def test_mixed_staging_and_auto_pinned_results(gpemu):
    """Inputs and outputs are staged independently: pageable inputs with page-locked results (what repeated calls get
    automatically from the second call of a size on) skip the copy-out; every combination gives the same bits."""
    import torch
    inputs, theta, invQ, invQt, _ = orc.make_S_model(90, 5, 1, seed=41)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    N = 300_017
    testing = np.random.RandomState(42).random_sample((N, 5))
    ref = m.predict(testing, pinned=False)
    assert not torch.from_numpy(ref["deriv"]).is_pinned()
    forced = m.predict(testing, pinned=True)                       # pageable in, page-locked out, several chunks
    assert torch.from_numpy(forced["deriv"]).is_pinned()
    pin_in = torch.from_numpy(testing).pin_memory().numpy()
    mixed = m.predict(pin_in, pinned=False)                        # page-locked in, pageable out
    first = m.predict(testing)                                     # auto: first request of this size -> pageable
    again = m.predict(testing)                                     # second request -> page-locked
    assert torch.from_numpy(again["deriv"]).is_pinned()
    for other in (forced, mixed, first, again):
        for k in ("mu", "var", "deriv"):
            assert np.array_equal(other[k], ref[k]), k
    small = m.predict(testing[:100]); small2 = m.predict(testing[:100])   # below 1 MB: never page-locked
    assert not torch.from_numpy(small2["deriv"]).is_pinned() and np.array_equal(small["mu"], small2["mu"])


def test_one_model_shared_by_threads(gpemu):
    """The numpy reference is re-entrant; here host-pointer calls on one handle are serialised by the library, so
    several Python threads (ctypes releases the GIL) may share one GaussianProcess."""
    import threading
    inputs, theta, invQ, invQt, _ = orc.make_S_model(100, 6, 1, seed=31)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    rs = np.random.RandomState(3)
    batches = [rs.random_sample((n, 6)) for n in (50_000, 120_001, 777, 64_000)]
    want = [m.predict(b) for b in batches]
    got = [None] * len(batches)
    def work(i):
        for _ in range(3):
            got[i] = m.predict(batches[i])
    th = [threading.Thread(target=work, args=(i,)) for i in range(len(batches))]
    for t in th: t.start()
    for t in th: t.join()
    for w, g_ in zip(want, got):
        for k in ("mu", "var", "deriv"):
            assert np.array_equal(w[k], g_[k]), k


def test_preallocated_and_pinned_outputs(gpemu):
    import torch
    inputs, theta, invQ, invQt, testing = orc.make_S_model(120, 7, 70000, seed=6)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    ref = m.predict(testing)
    out = {"mu": torch.empty(70000, dtype=torch.float64).pin_memory().numpy(), "deriv": np.empty((70000, 7))}
    got = m.predict(testing, out=out)
    assert got["mu"] is out["mu"] and got["deriv"] is out["deriv"]
    for k in ("mu", "var", "deriv"):
        assert np.array_equal(got[k], ref[k])
    got = m.predict(testing, pinned=True)
    for k in ("mu", "var", "deriv"):
        assert np.array_equal(got[k], ref[k])
    with pytest.raises(ValueError):
        m.predict(testing, out={"mu": np.empty(5)})
    t = torch.from_numpy(testing).cuda()
    dout = {"var": torch.empty(70000, dtype=torch.float64, device="cuda")}
    got = m.predict(t, out=dout)
    assert got["var"] is dout["var"] and np.array_equal(got["var"].cpu().numpy(), ref["var"])


@pytest.mark.parametrize("M,D,N", [(250, 10, 3000), (256, 10, 129), (64, 4, 500), (37, 3, 1), (100, 7, 257),
                                   (200, 16, 300), (130, 12, 128), (10, 1, 40)])
def test_single_precision_tensor_core_path(gpemu, M, D, N):
    """tcgen05 / TMEM kernels.  Bars: mean and gradient at the reference's own FP32 pass criterion 1e-5
    (tests/benchmark.py:56); variance 1e-5 as well in the default 3xTF32 mode, 5e-4 = 2^-11 (the TF32 input
    rounding; measured ~6e-5 at M = 250) in the single-pass `fast` mode."""
    import torch
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=M + D)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    t32 = testing.astype(np.float32)
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, t32.astype(np.float64))
    o = m.predict_f32(t32)
    assert o["mu"].dtype == np.float32 and o["deriv"].shape == (N, D)
    assert orc.ref_err(o["mu"], mu) < 1e-5 and orc.ref_err(o["deriv"], deriv) < 1e-5
    assert orc.ref_err(o["var"], var) < 1e-5
    of = m.predict_f32(t32, fast=True)
    assert orc.ref_err(of["mu"], mu) < 1e-5 and orc.ref_err(of["deriv"], deriv) < 1e-5
    assert orc.ref_err(of["var"], var) < 5e-4
    o2 = m.predict_f32(t32, want_var=False)
    assert orc.ref_err(o2["mu"], mu) < 1e-5 and orc.ref_err(o2["deriv"], deriv) < 1e-5
    od = m.predict_f32(torch.from_numpy(t32).cuda())
    torch.cuda.synchronize()
    for k in ("mu", "var", "deriv"):
        assert np.array_equal(od[k].cpu().numpy(), o[k])


@pytest.mark.parametrize("M,D,N", [(300, 5, 200), (512, 10, 129), (513, 4, 64), (1000, 10, 300), (1024, 12, 100),
                                   (700, 16, 50)])
def test_single_precision_large_m(gpemu, M, D, N):
    """256 < M <= 1024: column passes over the TMEM columns, K* slabs through a 2-deep A ring, epilogue with K*
    recomputed (predict_tf32_big.cuh).  At M ~ 1000 the FP32 accumulation of 1000-term sums itself costs ~1e-5, so
    the variance bar of the 3xTF32 mode is 3e-5 here (measured 1.1e-5 at M = 1000); fast mode as for small M."""
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=M + D)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    t32 = testing.astype(np.float32)
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, t32.astype(np.float64))
    for fast, bar in ((False, 3e-5), (True, 5e-4)):
        o = m.predict_f32(t32, fast=fast)
        assert orc.ref_err(o["mu"], mu) < 1e-5 and orc.ref_err(o["deriv"], deriv) < 1e-5
        assert orc.ref_err(o["var"], var) < bar, (fast, orc.ref_err(o["var"], var))
    o2 = m.predict_f32(t32, want_var=False)
    assert orc.ref_err(o2["mu"], mu) < 1e-5 and orc.ref_err(o2["deriv"], deriv) < 1e-5


def test_single_precision_limits_and_dropin_routing(gpemu):
    inputs, theta, invQ, invQt, testing = orc.make_S_model(1100, 5, 50, seed=2)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    with pytest.raises(gpemu.GpemuError):
        m.predict_f32(testing.astype(np.float32))          # M > 1024: not served by the tensor-core path
    inputs, theta, invQ, invQt, testing = orc.make_S_model(250, 10, 5000, seed=0)
    gp = gpemu.GaussianProcess(inputs, [])
    gp.theta, gp.invQ, gp.invQt = theta, invQ, invQt
    mu_c, var_c, deriv_c = orc.predict(inputs, theta, invQ, invQt, testing)
    mu, var, deriv = gp.predict(testing, precision=np.float32)    # the reference benchmark's GPU call
    assert mu.dtype == np.float32
    # all three outputs at the reference's FP32 criterion (tests/benchmark.py:56)
    assert orc.ref_err(mu, mu_c) < 1e-5 and orc.ref_err(deriv, deriv_c) < 1e-5 and orc.ref_err(var, var_c) < 1e-5


def test_dropin_class_matches_reference_semantics(gpemu):
    """The reference's benchmark flow (tests/benchmark.py:11-60): overwrite attributes, call predict."""
    inputs, theta, invQ, invQt, testing = orc.make_S_model(250, 10, 2000, seed=0)
    gp = gpemu.GaussianProcess(inputs, [])
    gp.theta, gp.invQ, gp.invQt = theta, invQ, invQt
    mu_c, var_c, deriv_c = orc.predict(inputs, theta, invQ, invQt, testing)
    mu, var, deriv = gp.predict(testing, is_gpu=True, threshold=1e5)
    assert orc.ref_err(mu, mu_c) < TOL and orc.ref_err(var, var_c) < TOL and orc.ref_err(deriv, deriv_c) < TOL
    mu2, deriv2 = gp.predict(testing, do_unc=False)
    assert orc.ref_err(mu2, mu_c) < TOL and orc.ref_err(deriv2, deriv_c) < TOL
    mu3, var3, deriv3 = gp.predict(testing, precision=np.float32)
    assert mu3.dtype == np.float32 and orc.ref_err(mu3, mu_c) < 1e-5  # the reference's own FP32 bar
    assert orc.ref_err(gp.hessian(testing[:100]), orc.hessian(inputs, theta, invQt, testing[:100])) < TOL
    # attributes overwritten in place -> the device copy must follow
    gp.invQt = invQt * 2.0
    mu4 = gp.predict(testing, do_unc=False, do_deriv=False)
    assert orc.ref_err(mu4, 2.0 * mu_c) < TOL
    with pytest.raises(AssertionError):
        gp.predict(np.zeros((3, 9)))


def test_legacy_predict_wrap_entry_point(lib, gpemu):
    inputs, theta, invQ, invQt, testing = orc.make_S_model(250, 10, 1500, seed=4)
    expX = np.exp(theta)
    N = testing.shape[0]
    res = np.zeros(N); err = np.zeros(N); der = np.zeros(N * 10)
    rc = lib.gpe_predict_wrap(expX.ctypes.data, inputs.ravel().ctypes.data, invQt.ctypes.data,
                              np.ascontiguousarray(invQ).ravel().ctypes.data, testing.ravel().ctypes.data,
                              res.ctypes.data, err.ctypes.data, der.ctypes.data, N, 250, 10, 12)
    assert rc == 0, lib.gpe_last_error()
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
    assert orc.ref_err(res, mu) < TOL and orc.ref_err(err, var) < TOL
    assert orc.ref_err(der.reshape(10, N).T, deriv) < TOL   # (D, N) layout, as GaussianProcess.py:321 expects


def test_multivariate_emulator_single_point_and_batch(gpemu):
    g = golden("P")
    mv = gpemu.MultivariateEmulator(X=None, y=None, dump=_write_prosail_dump(g))
    host_models = [(gp.inputs, gp.theta, gp.invQ, gp.invQt) for gp in mv.emulators]
    for k in range(3):
        fwd, d = mv.predict(g["points"][k])
        assert fwd.shape == (2101,) and d.shape == (10, 2101)
        # against the reference's frozen outputs: invQ is re-derived on this host and cond(Q) ~ 3.5e7, so 1e-6 ...
        assert orc.ref_err(fwd, g["fwd"][k]) < 1e-6
        assert orc.ref_err(d[:, g["wsub"]], g["deriv_sub"][k]) < 1e-6
        # ... and against the oracle on the SAME state at the full bar, so that a regression of the device path shows
        f_o, d_o = orc.mv_predict_point(host_models, mv.basis_functions, g["points"][k])
        assert orc.ref_err(fwd, f_o) < TOL and orc.ref_err(d, d_o) < TOL
    fwd_b, d_b = mv.predict(g["points"])
    assert fwd_b.shape == (3, 2101) and d_b.shape == (3, 10, 2101)
    models = [(gp.inputs, gp.theta, gp.invQ, gp.invQt) for gp in mv.emulators]
    ofwd, omu, ovar, ograd = orc.mv_predict_batch(models, mv.basis_functions, g["testing"])
    fwd_t = mv.predict(g["testing"], do_deriv=False)
    assert orc.ref_err(fwd_t, ofwd) < TOL
    pcs = mv.predict_pcs(g["testing"])
    assert orc.ref_err(pcs["mu"], omu) < TOL and orc.ref_err(pcs["deriv"], ograd) < TOL


def _write_prosail_dump(g):
    """Rebuild an npz in the reference's dump format from the fixture (X is not shipped: use B^T-lifted targets)."""
    import os
    import tempfile
    B = g["basis_functions"]
    X = g["train_data"].T @ B        # rank-P stand-in whose compression reproduces train_data (B rows orthonormal)
    f = os.path.join(tempfile.mkdtemp(), "prosail_fixture.npz")
    np.savez_compressed(f, X=X, y=g["y"], hyperparams=g["hyperparams"], thresh=0.99, basis_functions=B,
                        n_pcs=int(g["n_pcs"]))
    return f


def test_full_size_properties_linearity_and_kernel_bound(gpemu):
    """Size-independent properties at bench scale (N = 2e6 device-resident points)."""
    import torch
    inputs, theta, invQ, invQt, _ = orc.make_S_model(250, 10, 1, seed=0)
    N = 2_000_000
    gen = torch.Generator(device="cuda").manual_seed(0)
    t = torch.rand(N, 10, dtype=torch.float64, device="cuda", generator=gen)
    a1 = np.random.RandomState(1).random_sample(250); a2 = np.random.RandomState(2).random_sample(250)
    o1 = gpemu.DeviceModel(inputs, theta, a1, invQ).predict(t)
    o2 = gpemu.DeviceModel(inputs, theta, a2, invQ).predict(t)
    o12 = gpemu.DeviceModel(inputs, theta, a1 + a2, invQ).predict(t)
    # mean and gradient are linear in invQt; the variance does not depend on it
    for k in ("mu", "deriv"):
        err = (o1[k] + o2[k] - o12[k]).abs().max() / o12[k].abs().max()
        assert float(err) < 1e-13, k
    assert torch.equal(o1["var"], o2["var"])
    # scaling invQ by s scales (b - var) by s
    o3 = gpemu.DeviceModel(inputs, theta, a1, 3.0 * invQ).predict(t)
    b = float(np.exp(theta[10]))
    err = ((b - o3["var"]) - 3.0 * (b - o1["var"])).abs().max() / (b - o3["var"]).abs().max()
    assert float(err) < 1e-13
    # spot-check against the oracle on a prefix and a random subset
    idx = np.r_[0:2000, np.random.RandomState(3).randint(0, N, 2000)]
    tt = t[torch.from_numpy(idx).cuda()].cpu().numpy()
    mu, var, deriv = orc.predict(inputs, theta, invQ, a1, tt)
    ii = torch.from_numpy(idx).cuda()
    assert orc.ref_err(o1["mu"][ii].cpu().numpy(), mu) < TOL
    assert orc.ref_err(o1["var"][ii].cpu().numpy(), var) < TOL
    assert orc.ref_err(o1["deriv"][ii].cpu().numpy(), deriv) < TOL


@pytest.mark.parametrize("M,D,N", [(250, 10, 1500), (1000, 10, 100), (300, 6, 200), (37, 3, 70), (200, 8, 130),
                                   (8, 2, 40), (30, 4, 9000), (64, 5, 8000), (100, 10, 7200), (129, 3, 300), (224, 10, 100),
                                   (256, 7, 64), (257, 7, 33), (420, 4, 50), (512, 10, 40), (700, 2, 30), (1024, 6, 20)])
def test_symmetric_variance_option(gpemu, M, D, N):
    """Opt-in k^T T k (upper-triangular fold of invQ): exact identity for ANY invQ, incl. the benchmark's
    non-symmetric random matrix; same 1e-10 bar, mean / gradient bit-identical to the default path.  The shapes cover the
    tile counts of the three configurations (one tile, odd and even numbers of column tiles per warp, Mp = 256 / 512 / 1024
    exactly) and both the 64-point and the small-batch (16-point, run-time tile count) plans."""
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=M)
    m0 = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    m1 = gpemu.DeviceModel(inputs, theta, invQt, invQ, symmetric_variance=True)
    a, b = m0.predict(testing), m1.predict(testing)
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
    assert orc.ref_err(b["var"], var) < TOL
    assert np.array_equal(a["mu"], b["mu"]) and np.array_equal(a["deriv"], b["deriv"])


def test_symmetric_variance_on_trained_model(gpemu):
    g = golden("T")
    m1 = gpemu.DeviceModel(g["inputs"], g["theta"], g["invQt"], g["invQ"], symmetric_variance=True)
    out = m1.predict(g["testing"])
    assert orc.var_cond_err(out["var"], g["var"], g["inputs"], g["theta"], g["invQ"], g["testing"]) < TOL
    _, lvar, _ = orc.predict_longdouble(g["inputs"], g["theta"], g["invQ"], g["invQt"], g["testing"])
    assert np.max(np.abs(out["var"] - lvar)) <= 2.0 * np.max(np.abs(g["var"] - lvar)) + 1e-18


def test_symmetric_variance_auto_mode(gpemu):
    """"auto" folds invQ only when it is symmetric (the inverse of a covariance matrix), never the random invQ of the
    reference benchmark; the drop-in class passes the choice through and both stay inside the parity bars."""
    g = golden("T")
    m = gpemu.DeviceModel(g["inputs"], g["theta"], g["invQt"], g["invQ"], symmetric_variance="auto")
    assert m.symmetric_variance is True
    out = m.predict(g["testing"])
    assert orc.var_cond_err(out["var"], g["var"], g["inputs"], g["theta"], g["invQ"], g["testing"]) < TOL
    inputs, theta, invQ, invQt, testing = orc.make_S_model(100, 5, 300, seed=13)
    ms = gpemu.DeviceModel(inputs, theta, invQt, invQ, symmetric_variance="auto")
    assert ms.symmetric_variance is False
    gp = gpemu.GaussianProcess(g["inputs"], g["targets"], symmetric_variance="auto")
    gp._set_params(g["theta"])
    mu, var, deriv = gp.predict(g["testing"])
    assert gp._dev_model.symmetric_variance is True
    assert orc.ref_err(mu, g["mu"]) < TOL and orc.ref_err(deriv, g["deriv"]) < TOL
    assert orc.var_cond_err(var, g["var"], g["inputs"], g["theta"], gp.invQ, g["testing"]) < TOL
    with pytest.raises(ValueError):
        gpemu.DeviceModel(inputs, theta, invQt, invQ, symmetric_variance="sometimes")


def test_documented_limits_raise_cleanly(gpemu):
    """M > GPE_MAX_TRAIN (variance) is reported as GPE_ERR_UNSUPPORTED, never a wrong answer."""
    rs = np.random.RandomState(1)
    M = 16400
    inputs = rs.random_sample((M, 3)); theta = rs.random_sample(5); invQt = rs.random_sample(M)
    invQ = np.zeros((M, M))          # never read: the limit is checked first
    testing = rs.random_sample((20, 3))
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    with pytest.raises(gpemu.GpemuError, match="M <= 16384"):
        m.predict(testing)
    o = m.predict(testing, want_var=False)               # mean + gradient have no M limit
    mu, _, deriv = orc.predict(inputs, theta, invQ, invQt, testing, do_unc=False)
    assert orc.ref_err(o["mu"], mu) < TOL and orc.ref_err(o["deriv"], deriv) < TOL


@pytest.mark.parametrize("M,D,N", [(1025, 4, 300), (1100, 3, 20), (1500, 10, 2500), (2048, 6, 777), (2500, 10, 100),
                                   (4096, 2, 50), (4500, 3, 40), (6000, 2, 17)])
def test_large_m_variance(gpemu, M, D, N):
    """1024 < M <= GPE_MAX_TRAIN: K* goes through a scratch buffer and the contraction runs in column passes
    (predict_var_large.cuh).  Same formula as GaussianProcess.py:232-247, same tolerance."""
    import torch
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=M % 97)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    out = m.predict(testing, want_hess=(D <= 6))
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
    assert orc.ref_err(out["mu"], mu) < TOL and orc.ref_err(out["var"], var) < TOL
    assert orc.ref_err(out["deriv"], deriv) < TOL
    if D <= 6:
        assert orc.ref_err(out["hess"], orc.hessian(inputs, theta, invQt, testing)) < TOL
    v_only = m.predict(torch.from_numpy(testing).cuda(), want_mu=False, want_deriv=False)["var"]
    assert np.array_equal(v_only.cpu().numpy(), out["var"])


def test_large_m_variance_many_points_and_streams(gpemu):
    """More points than the K* scratch holds (sub-batches) and the host pipeline's three streams sharing it."""
    inputs, theta, invQ, invQt, _ = orc.make_S_model(1300, 5, 1, seed=4)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    N = 60_001
    testing = np.random.RandomState(5).random_sample((N, 5))
    out = m.predict(testing)                                  # pageable: staged pipeline, several chunks
    idx = np.r_[0:30, 9460:9490, 30_000:30_030, N - 30:N]
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing[idx])
    assert orc.ref_err(out["mu"][idx], mu) < TOL and orc.ref_err(out["var"][idx], var) < TOL
    assert orc.ref_err(out["deriv"][idx], deriv) < TOL
    again = m.predict(testing)
    assert np.array_equal(again["var"], out["var"])


@pytest.mark.parametrize("M,D,N", [(50, 13, 70), (120, 16, 33), (300, 20, 40), (64, 32, 65)])
def test_hessian_large_d(gpemu, M, D, N):
    """D > 12 runs the row-block Hessian kernel (k_hessian_rows)."""
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=D)
    theta = theta - 1.5
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    out = m.predict(testing, want_var=False, want_hess=True)
    mu, _, deriv = orc.predict(inputs, theta, invQ, invQt, testing, do_unc=False)
    assert orc.ref_err(out["mu"], mu) < TOL and orc.ref_err(out["deriv"], deriv) < TOL
    assert orc.ref_err(out["hess"], orc.hessian(inputs, theta, invQt, testing)) < TOL


@pytest.mark.parametrize("M,D,N", [(250, 10, 333), (96, 4, 65), (60, 2, 64), (400, 7, 100), (1000, 10, 50), (200, 16, 77),
                                   (180, 12, 130), (57, 10, 40)])
def test_fused_hessian(gpemu, M, D, N):
    """mean + variance + gradient + Hessian in one launch: the Hessian is a second tensor-path contraction against
    the K* tile (predict_full.cuh phase C).  Reference GaussianProcess.py:345-366 for the values."""
    N += 600          # above the few-hundred-point cluster path (predict_tiny.cuh), which pairs with the direct Hessian kernel
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=M + D)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    before = gpemu._lib.load().gpe_launch_count()
    out = m.predict(testing, want_hess=True)
    assert gpemu._lib.load().gpe_launch_count() - before == 1
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
    assert orc.ref_err(out["mu"], mu) < TOL and orc.ref_err(out["var"], var) < TOL
    assert orc.ref_err(out["deriv"], deriv) < TOL
    ho = orc.hessian(inputs, theta, invQt, testing)
    assert orc.ref_err(out["hess"], ho) < TOL
    h = m.predict(testing, want_mu=False, want_var=False, want_deriv=False, want_hess=True)["hess"]
    assert orc.ref_err(h, ho) < TOL


def test_fused_hessian_fallbacks(gpemu):
    """Shapes / data the fused Hessian does not take fall back to the direct kernel (two launches), same values:
    fewer training points than Hessian columns, symmetric-folded variance operand, inputs spanning so many length
    scales that the centred expansion would cancel digits."""
    lib = gpemu._lib.load()
    cases = []
    inputs, theta, invQ, invQt, testing = orc.make_S_model(40, 10, 50, seed=1)          # NC = 56 > M
    cases.append((gpemu.DeviceModel(inputs, theta, invQt, invQ), inputs, theta, invQ, invQt, testing))
    inputs, theta, invQ, invQt, testing = orc.make_S_model(250, 10, 50, seed=2)
    cases.append((gpemu.DeviceModel(inputs, theta, invQt, invQ, symmetric_variance=True), inputs, theta, invQ, invQt, testing))
    inputs, theta, invQ, invQt, testing = orc.make_S_model(250, 10, 50, seed=3)
    theta = theta.copy(); theta[0] += np.log(1.0e6)                                      # 1000x shorter length scale in d = 0
    invQ, invQt = orc.prepare_likelihood(inputs, np.sin(inputs.sum(1)), theta)
    testing = inputs[:50] + 1e-4
    cases.append((gpemu.DeviceModel(inputs, theta, invQt, invQ), inputs, theta, invQ, invQt, testing))
    for m, inputs, theta, invQ, invQt, testing in cases:
        before = lib.gpe_launch_count()
        out = m.predict(testing, want_hess=True)
        assert lib.gpe_launch_count() - before == 2
        mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
        assert orc.ref_err(out["mu"], mu) < TOL and orc.ref_err(out["var"], var) < 1e-9
        assert orc.ref_err(out["hess"], orc.hessian(inputs, theta, invQt, testing)) < TOL


def test_fused_hessian_short_length_scales(gpemu):
    """Training inputs spanning +-30 length scales in every dimension: still inside the fused path's guard
    (max |x'|^2 = 900 <= 2000); the cancellation of the centred expansion must stay far below the bar."""
    lib = gpemu._lib.load()
    rs = np.random.RandomState(11)
    M, D = 250, 6
    inputs = rs.random_sample((M, D))
    theta = np.concatenate([np.full(D, np.log(3600.0)), [0.3, -6.0]])
    invQ, invQt = orc.prepare_likelihood(inputs, np.sin(4 * inputs.sum(1)), theta)
    testing = np.tile(inputs, (3, 1)) + 0.01 * rs.standard_normal((3 * M, D))     # 750 points: the fused plan
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    before = lib.gpe_launch_count()
    out = m.predict(testing, want_hess=True)
    assert lib.gpe_launch_count() - before == 1
    ho = orc.hessian(inputs, theta, invQt, testing)
    assert np.abs(ho).max() > 1.0
    assert orc.ref_err(out["hess"], ho) < TOL


def test_fused_hessian_offset_inputs(gpemu):
    """Inputs far from the origin: the centring of the fused expansion must keep the error at the level of the
    direct formula (which itself is limited by the conditioning of x - t at |x| ~ 1e3)."""
    inputs, theta, _, _, testing = orc.make_S_model(250, 10, 200, seed=5)
    inputs = inputs + 1000.0
    testing = testing + 1000.0
    invQ, invQt = orc.prepare_likelihood(inputs, np.sin(inputs.sum(1)), theta)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    out = m.predict(testing, want_hess=True)
    assert orc.ref_err(out["hess"], orc.hessian(inputs, theta, invQt, testing)) < 1e-10


def test_inplace_edits_are_seen_without_invalidate(gpemu):
    """The reference re-reads inputs / theta / invQ / invQt on every predict (GaussianProcess.py:228-240).  Here the
    device copy is checked bitwise against the arrays (one memcmp) whenever that is cheap next to the call -- always at
    M = 250, and for >= 1000 points at any M -- so an in-place edit of ONE entry gives the new result with no hook."""
    inputs, theta, invQ, invQt, testing = orc.make_S_model(250, 10, 10_000, seed=2)
    gp = gpemu.GaussianProcess(inputs.copy(), [])
    gp.theta, gp.invQ, gp.invQt = theta, invQ.copy(), invQt
    _, v0, _ = gp.predict(testing)
    gp.invQ[101, 7] += 0.5                                # one entry, in place, not on the sampled grid
    _, v1, _ = gp.predict(testing)
    _, var, _ = orc.predict(inputs, theta, gp.invQ, invQt, testing)
    assert orc.ref_err(v1, var) < TOL and not np.array_equal(v0, v1)
    gp.inputs[17, 3] += 0.25                              # the other matrix; a one-point call this time
    m1, v2, d1 = gp.predict(testing[:1])
    mu, var, der = orc.predict(gp.inputs, theta, gp.invQ, invQt, testing[:1])
    assert orc.ref_err(m1, mu) < TOL and orc.ref_err(v2, var) < TOL and orc.ref_err(d1, der) < TOL
    # a large model: tiny calls use the sampled fingerprint (documented), calls of >= 1000 points the full comparison
    inputs, theta, invQ, invQt, testing = orc.make_S_model(600, 4, 1200, seed=3)
    gp = gpemu.GaussianProcess(inputs, [])
    gp.theta, gp.invQ, gp.invQt = theta, invQ.copy(), invQt
    gp.predict(testing[:5])
    gp.invQ[301, 11] -= 0.75
    _, v3, _ = gp.predict(testing)
    assert orc.ref_err(v3, orc.predict(inputs, theta, gp.invQ, invQt, testing)[1]) < TOL
    gp.cache_check = "full"
    gp.invQ[5, 501] += 0.3
    _, v4, _ = gp.predict(testing[:3])
    assert orc.ref_err(v4, orc.predict(inputs, theta, gp.invQ, invQt, testing[:3])[1]) < TOL
    gp.invalidate_device()
    assert gp._dev_model is None


def test_closed_handles_raise(gpemu):
    inputs, theta, invQ, invQt, testing = orc.make_S_model(20, 3, 10, seed=4)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    m.predict(testing)
    m.close()
    with pytest.raises(gpemu.GpemuError):
        m.predict(testing)
    b = gpemu.DeviceBank(inputs, theta[None, :], invQt[None, :], invQ[None, :, :])
    b.close()
    with pytest.raises(gpemu.GpemuError):
        b.predict(testing)


def test_reference_method_aliases(gpemu):
    """cpu_predict / gpu_predict / get_gpu_block exist under the reference's names (GaussianProcess.py:211, 253, 273)."""
    inputs, theta, invQ, invQt, testing = orc.make_S_model(64, 4, 50, seed=2)
    gp = gpemu.GaussianProcess(inputs, [])
    gp.theta, gp.invQ, gp.invQt = theta, invQ, invQt
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
    a = gp.cpu_predict(testing)
    assert len(a) == 3 and orc.ref_err(a[0], mu) < TOL and orc.ref_err(a[1], var) < TOL and orc.ref_err(a[2], deriv) < TOL
    b = gp.cpu_predict(testing, do_unc=False)
    assert len(b) == 2 and orc.ref_err(b[0], mu) < TOL and orc.ref_err(b[1], deriv) < TOL    # (mean-only kernel)
    c = gp.gpu_predict(testing)
    assert all(np.array_equal(x, y) for x, y in zip(a, c))
    s, e = gp.get_gpu_block(10, 4)
    assert list(s) == [0, 4, 7] and list(e) == [4, 7, 10]


def test_one_call_multi_device_fanout(lib, gpemu):
    """gpe_multi_*: with G visible GPUs the batch is split over them; with one GPU the same code path runs two
    copies of the model on device 0 from two host threads.  Bit-identical to the single-device result."""
    inputs, theta, invQ, invQt, testing = orc.make_S_model(250, 10, 100001, seed=12)
    ndev = lib.gpe_device_count()
    devices = list(range(ndev)) if ndev > 1 else [0, 0]
    mm = gpemu.MultiDeviceModel(inputs, theta, invQt, invQ, devices=devices)
    a = mm.predict(testing)
    b = gpemu.DeviceModel(inputs, theta, invQt, invQ).predict(testing)
    for k in ("mu", "var", "deriv"):
        assert np.array_equal(a[k], b[k]), k
    h = mm.predict(testing[:300], want_var=False, want_deriv=False, want_hess=True)["hess"]
    assert orc.ref_err(h, orc.hessian(inputs, theta, invQt, testing[:300])) < TOL
    # a call whose per-device shares fall below the small-batch switch while the call itself does not: the tile plan
    # follows the call, so the fan-out still reproduces the single-device result bit for bit
    single = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    for n in (10_000, 7_104, 300):
        a = mm.predict(testing[:n]); b = single.predict(testing[:n])
        for k in ("mu", "var", "deriv"):
            assert np.array_equal(a[k], b[k]), (n, k)


def test_random_shape_sweep(gpemu):
    """Seeded fuzz over (M, D, N): random shapes, chunked / resident training sets, ragged tiles.  Batches stay small
    (N < 700), so for M <= 256 the calls run the cluster kernel or the 16-point small plan; every compiled instance at
    the batch sizes that select it is covered by tests/test_instance_matrix.py."""
    rs = np.random.RandomState(2026)
    for _ in range(24):
        M = int(rs.choice([rs.randint(1, 64), rs.randint(64, 257), rs.randint(257, 513), rs.randint(513, 1025)]))
        D = int(rs.randint(1, 33))
        N = int(rs.choice([1, rs.randint(2, 200), rs.randint(200, 700)]))
        inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=int(rs.randint(1 << 30)))
        invQ = invQ - 0.5                       # mixed signs: exercises cancellation in the contraction
        theta = theta - 1.0
        m = gpemu.DeviceModel(inputs, theta, invQt, invQ, symmetric_variance=bool(rs.randint(2)))
        out = m.predict(testing)
        mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
        tag = (M, D, N)
        assert orc.ref_err(out["mu"], mu) < TOL, tag
        assert orc.ref_err(out["deriv"], deriv) < TOL, tag
        assert orc.var_cond_err(out["var"], var, inputs, theta, invQ, testing) < TOL, tag
        if D <= 16:
            o32 = m.predict_f32(testing.astype(np.float32), fast=bool(rs.randint(2)))
            assert orc.ref_err(o32["mu"], mu) < 2e-5, tag


def test_single_precision_host_streaming_multi_chunk(gpemu):
    """float32 host arrays go through the same host pipeline as FP64: chunk seams must be invisible."""
    import torch
    inputs, theta, invQ, invQt, _ = orc.make_S_model(96, 5, 1, seed=3)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    N = (1 << 18) + 4321
    t32 = np.random.RandomState(1).random_sample((N, 5)).astype(np.float32)
    a = m.predict_f32(t32)
    b = m.predict_f32(torch.from_numpy(t32).cuda())
    torch.cuda.synchronize()
    for k in ("mu", "var", "deriv"):
        assert np.array_equal(a[k], b[k].cpu().numpy()), k


# ---- round 2: BASELINE configs 4 and 5 under pytest, banks through the host pipeline, one call / all GPUs, guards ----
@pytest.mark.parametrize("M,D,E,N", [(250, 10, 64, 150), (37, 3, 5, 131), (60, 13, 3, 70)])
def test_bank_hessian_against_oracle(gpemu, M, D, E, N):
    """BASELINE config 5: a per-band bank (E GPs, shared inputs and test points) with mean, variance, gradient AND
    Hessian against E separate oracle predict + hessian calls -- the reference pattern of
    tests/test_perband_emulator.py:22-37 + GaussianProcess.hessian (:345-366); point-major strided outputs
    (ld_hess = E*D*D), device and host callers."""
    import torch
    rs = np.random.RandomState(100 + E)
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)); invQs = rs.random_sample((E, M, M))
    bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs)
    t = rs.random_sample((N, D))
    models = [(inputs, thetas[e], invQs[e], invQts[e]) for e in range(E)]
    mu_o, var_o, grad_o, hess_o = orc.bank_predict(models, t, do_hess=True)
    host = bank.predict(t, want_var=True, want_deriv=True, want_hess=True)
    dev = bank.predict(torch.from_numpy(t).cuda(), want_var=True, want_deriv=True, want_hess=True)
    for name, got in (("host", host), ("device", {k: v.cpu().numpy() for k, v in dev.items()})):
        assert got["hess"].shape == (N, E, D, D) and got["deriv"].shape == (N, E, D)
        assert orc.ref_err(got["mu"], mu_o) < TOL, name
        assert orc.ref_err(got["var"], var_o) < TOL, name
        assert orc.ref_err(got["deriv"], grad_o) < TOL, name
        assert orc.ref_err(got["hess"], hess_o) < TOL, name
    # Hessian without the variance (one launch for all emulators, or per-emulator fused launches on big batches)
    h_only = bank.predict(t, want_var=False, want_deriv=False, want_hess=True)
    assert orc.ref_err(h_only["hess"], hess_o) < TOL and orc.ref_err(h_only["mu"], mu_o) < TOL


def test_golden_perband_bank_with_hessian(gpemu):
    """The same pattern against outputs frozen from the reference itself (golden_K: trained per-band GPs)."""
    g = golden("K")
    bank = gpemu.DeviceBank(g["inputs"], g["thetas"], g["invQt"], g["invQ"])
    got = bank.predict(g["testing"], want_var=True, want_deriv=True, want_hess=True)
    assert orc.ref_err(got["mu"], g["mu"]) < TOL and orc.ref_err(got["deriv"], g["deriv"]) < TOL
    assert orc.ref_err(got["hess"], g["hess"]) < TOL
    for e in range(g["thetas"].shape[0]):
        assert orc.var_cond_err(got["var"][:, e], g["var"][:, e], g["inputs"], g["thetas"][e], g["invQ"][e], g["testing"]) < TOL


def test_cfg4_20_components_2101_wavelengths(gpemu):
    """BASELINE config 4: P = 20 PCs, W = 2101 wavelengths, synthetic orthonormal basis; PC-space outputs, spectra and
    full Jacobians against the oracle's batched MultivariateEmulator.predict (multivariate_gp.py:195-222), host and
    device callers."""
    import torch
    M, D, P, W, N = 250, 10, 20, 2101, 96
    rs = np.random.RandomState(4)
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((P, D + 2)); invQts = rs.random_sample((P, M)); invQs = rs.random_sample((P, M, M))
    basis = np.linalg.qr(rs.standard_normal((W, P)))[0].T.copy()
    bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=basis)
    tt = rs.random_sample((N, D))
    models = [(inputs, thetas[i], invQs[i], invQts[i]) for i in range(P)]
    fwd, mu_o, var_o, grad_o, dfull = orc.mv_predict_batch(models, basis, tt, want_deriv_full=True)
    kw = dict(want_var=True, want_deriv=True, project=True, project_deriv=True)
    host = bank.predict(tt, **kw)
    dev = {k: v.cpu().numpy() for k, v in bank.predict(torch.from_numpy(tt).cuda(), **kw).items()}
    for name, got in (("host", host), ("device", dev)):
        assert got["fwd"].shape == (N, W) and got["deriv_full"].shape == (N, D, W)
        for k, ref in (("fwd", fwd), ("mu", mu_o), ("var", var_o), ("deriv", grad_o), ("deriv_full", dfull)):
            assert orc.ref_err(got[k], ref) < TOL, (name, k)
    f2, d2 = bank.forward(tt)           # (no variance: the one-launch bank mean kernel instead of P fused launches)
    assert orc.ref_err(f2, fwd) < TOL and orc.ref_err(d2, dfull) < TOL


def test_golden_cfg4_multivariate_emulator_20pcs(gpemu):
    """The drop-in MultivariateEmulator on a model the REFERENCE built with 20 PCs x 2101 wavelengths (golden_M20):
    single-point predicts as the reference makes them, and the batch call."""
    g = golden("M20")
    B = g["basis_functions"]
    X = g["train_data"].T @ B            # rank-20 stand-in whose compression reproduces train_data
    mv = gpemu.MultivariateEmulator(X=X, y=g["y"], hyperparams=g["hyperparams"], basis_functions=B, n_pcs=20)
    models = [(gp.inputs, gp.theta, gp.invQ, gp.invQt) for gp in mv.emulators]
    for k in range(4):
        fwd, d = mv.predict(g["points"][k])
        assert fwd.shape == (2101,) and d.shape == (10, 2101)
        assert orc.ref_err(fwd, g["fwd"][k]) < 1e-7        # invQ re-derived on this host (cond(Q) ~ 1e6)
        assert orc.ref_err(d[:, g["wsub"]], g["deriv_sub"][k]) < 1e-7
        ofwd, od = orc.mv_predict_point(models, B, g["points"][k])     # same invQ on both sides: the 1e-10 bar
        assert orc.ref_err(fwd, ofwd) < TOL and orc.ref_err(d, od) < TOL
    fb, db = mv.predict(g["points"])
    assert fb.shape == (4, 2101) and db.shape == (4, 10, 2101)
    ofwd, _, _, _, odf = orc.mv_predict_batch(models, B, g["points"], want_deriv_full=True)
    assert orc.ref_err(fb, ofwd) < TOL and orc.ref_err(db, odf) < TOL
    # re-binding one emulator's state re-uploads the bank; in-place edits need invalidate_device()
    mv.emulators[3]._set_params(mv.emulators[3].theta + 0.01)
    models[3] = (mv.emulators[3].inputs, mv.emulators[3].theta, mv.emulators[3].invQ, mv.emulators[3].invQt)
    f2 = mv.predict(g["points"][1], do_deriv=False)
    assert orc.ref_err(f2, orc.mv_predict_point(models, B, g["points"][1])[0]) < TOL and not np.array_equal(f2, fb[1])


@pytest.mark.parametrize("E", [33, 70])
def test_bank_with_more_than_32_emulators_and_a_basis(gpemu, E):
    """The reference has no limit on the number of PCs: banks beyond 32 emulators project in slices of 32 that
    accumulate into the output (ADVICE r01: E > 32 with a basis used to overflow the packed basis image)."""
    import torch
    M, D, W, N = 40, 3, 300, 203
    rs = np.random.RandomState(E)
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)) - 0.5
    basis = rs.standard_normal((E, W))
    bank = gpemu.DeviceBank(inputs, thetas, invQts, None, basis=basis)
    t = rs.random_sample((N, D))
    models = [(inputs, thetas[e], None, invQts[e]) for e in range(E)]
    mu = np.empty((N, E)); grad = np.empty((N, E, D))
    for e in range(E):
        mu[:, e], _, grad[:, e, :] = orc.predict(inputs, thetas[e], None, invQts[e], t, do_unc=False)
    fwd = mu @ basis
    dfull = np.einsum("ned,ew->ndw", grad, basis)
    host = bank.predict(t, want_var=False, want_deriv=True, project=True, project_deriv=True)
    dev = {k: v.cpu().numpy() for k, v in bank.predict(torch.from_numpy(t).cuda(), want_var=False, want_deriv=True,
                                                        project=True, project_deriv=True).items()}
    for name, got in (("host", host), ("device", dev)):
        assert orc.ref_err(got["mu"], mu) < TOL and orc.ref_err(got["deriv"], grad) < TOL, name
        assert orc.ref_err(got["fwd"], fwd) < TOL and orc.ref_err(got["deriv_full"], dfull) < TOL, name


def test_bank_cost_host_streaming_seams(gpemu, monkeypatch):
    """gpe_bank_cost_host: test points and per-point observations stream in, cost + gradient stream out, in chunks."""
    rs = np.random.RandomState(77)
    M, D, E, N = 60, 4, 6, 2500
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)); invQs = rs.random_sample((E, M, M))
    bank = gpemu.DeviceBank(inputs, thetas, invQts)          # (mean + gradient only: the bank needs no invQ)
    t = rs.random_sample((N, D))
    models = [(inputs, thetas[e], invQs[e], invQts[e]) for e in range(E)]
    obsN = rs.random_sample((N, E)); w = rs.random_sample(E) + 0.5
    c_o, g_o = orc.bank_cost(models, t, obsN, w)
    one = bank.cost(t, obsN, w)
    monkeypatch.setenv("GPE_SLOT_OUT_BYTES", str(8 * (1 + D) * 300))     # 300 points per chunk
    many = bank.cost(t, obsN, w)
    shared = bank.cost(t, obsN[0], None)
    monkeypatch.delenv("GPE_SLOT_OUT_BYTES")
    assert orc.ref_err(one["cost"], c_o) < TOL and orc.ref_err(one["grad"], g_o) < TOL
    assert np.array_equal(one["cost"], many["cost"]) and np.array_equal(one["grad"], many["grad"])
    c1, g1 = orc.bank_cost(models, t, obsN[0], None)
    assert orc.ref_err(shared["cost"], c1) < TOL and orc.ref_err(shared["grad"], g1) < TOL


def test_drop_in_classes_spread_one_call_over_all_devices(lib, gpemu):
    """GaussianProcess / MultivariateEmulator / DeviceBank with device="all" (or a list): ONE predict call, every GPU of
    the list -- the reference API has no notion of ranks (GaussianProcess.py:327).  The devices' pipelines pull chunks
    from one cursor; results are bit-identical to one GPU.  With one visible GPU the list [0, 0] runs the same code with
    two resident copies."""
    import torch
    ndev = lib.gpe_device_count()
    devices = "all" if ndev > 1 else [0, 0]
    inputs, theta, invQ, invQt, testing = orc.make_S_model(250, 10, 300_001, seed=12)
    gp1 = gpemu.GaussianProcess(inputs, [], device=0)
    gpn = gpemu.GaussianProcess(inputs, [], device=devices)
    for gp in (gp1, gpn):
        gp.theta, gp.invQ, gp.invQt = theta, invQ, invQt
    a = gp1.predict(testing); b = gpn.predict(testing)
    assert isinstance(gpn._device_model(), gpemu.MultiDeviceModel)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    pin = torch.from_numpy(testing).pin_memory().numpy()
    out = {k: torch.empty(s, dtype=torch.float64).pin_memory().numpy() for k, s in
           (("mu", (300_001,)), ("var", (300_001,)), ("deriv", (300_001, 10)))}
    c = gpn.predict(pin, out=out)                                     # page-locked in and out: direct DMA path
    for x, y in zip(a, c):
        assert np.array_equal(x, y)
    assert np.array_equal(gpn.hessian(testing[:500]), gp1.hessian(testing[:500]))
    mu1 = gpn.predict(testing[:1], do_unc=False, do_deriv=False)
    assert mu1.shape == (1,) and mu1[0] == a[0][0]
    # device-resident data on several devices: one tensor per device
    mm = gpn._device_model()
    parts = [torch.from_numpy(testing[i * 1000:(i + 1) * 1000]).to("cuda:%d" % d) for i, d in enumerate(mm.devices)]
    res = mm.predict(parts)
    for d in set(mm.devices):
        torch.cuda.synchronize(d)
    for i, r in enumerate(res):
        assert np.array_equal(r["var"].cpu().numpy(), gp1.predict(testing[i * 1000:(i + 1) * 1000])[1])
    one = mm.predict(parts[-1])
    assert np.array_equal(one["mu"].cpu().numpy(), res[-1]["mu"].cpu().numpy())
    with pytest.raises(ValueError):
        mm.predict(testing, out={"mu": np.empty(3)})                  # wrong shape is refused, not written past
    with pytest.raises(ValueError):
        mm.predict(testing, out={"mu": np.empty(300_001, dtype=np.float32)})
    # single precision on a multi-device handle is served by one device
    m32 = gpn.predict(testing[:2000], precision=np.float32)
    assert m32[0].dtype == np.float32 and orc.ref_err(m32[0], a[0][:2000]) < 1e-5
    # banks
    rs = np.random.RandomState(5)
    M, D, E, W, N = 60, 4, 5, 300, 40_000
    binp = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)); invQs = rs.random_sample((E, M, M))
    basis = rs.standard_normal((E, W))
    t = rs.random_sample((N, D))
    b1 = gpemu.DeviceBank(binp, thetas, invQts, invQs, basis=basis, device=0)
    bn = gpemu.DeviceBank(binp, thetas, invQts, invQs, basis=basis, device=devices)
    kw = dict(want_var=True, want_deriv=True, want_hess=True, project=True)
    r1 = b1.predict(t, **kw); rn = bn.predict(t, **kw)
    for k in r1:
        assert np.array_equal(r1[k], rn[k]), k
    obs = rs.random_sample((N, E))
    c1 = b1.cost(t, obs); cn = bn.cost(t, obs)
    assert np.array_equal(c1["cost"], cn["cost"]) and np.array_equal(c1["grad"], cn["grad"])
    with pytest.raises(ValueError):
        bn.predict(torch.from_numpy(t).cuda())


def test_large_m_scratch_shared_by_threads_and_streams(gpemu):
    """1024 < M: the per-model K* scratch is handed between streams through an event; wait -> launches -> record is
    one critical section (ADVICE r01: two threads could both pass the wait before either recorded)."""
    import threading
    import torch
    M, D, N = 1100, 4, 6000
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=8)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    ref = orc.predict(inputs, theta, invQ, invQt, testing)
    td = torch.from_numpy(testing).cuda()
    results, errors = {}, []

    def work(i):
        try:
            st = torch.cuda.Stream()
            with torch.cuda.stream(st):
                for _ in range(3):
                    out = m.predict(td)
            st.synchronize()
            results[i] = {k: v.cpu().numpy() for k, v in out.items()}
        except Exception as e:          # pragma: no cover
            errors.append(e)
    threads = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for th in threads: th.start()
    for th in threads: th.join()
    assert not errors
    for i in range(4):
        assert orc.ref_err(results[i]["mu"], ref[0]) < TOL and orc.ref_err(results[i]["var"], ref[1]) < TOL
        assert orc.ref_err(results[i]["deriv"], ref[2]) < TOL


def _guarded(shape, guard=4096):
    """CUDA tensor of `shape` carved out of a buffer with NaN-pattern guard bands on both sides."""
    import torch
    n = int(np.prod(shape)) if len(shape) else 1
    big = torch.full((guard + n + guard,), float("nan"), dtype=torch.float64, device="cuda")
    return big, big[guard:guard + n].view(*shape)


def _guards_intact(big, n, guard=4096):
    import torch
    return bool(torch.isnan(big[:guard]).all()) and bool(torch.isnan(big[guard + n:]).all())


def test_red_zones_around_every_output(gpemu):
    """Stand-in for compute-sanitizer (closed on this pool): every output lives between NaN guard bands; after a sweep
    over all plans (cfg 0/1/2, small-batch plan, symmetric fold, fused / direct Hessian, large M, single precision,
    bank strides, projection slices) the guards must be untouched and every result element written."""
    import torch
    rs = np.random.RandomState(9)
    shapes = [(1, 1, 1), (5, 2, 3), (64, 4, 129), (100, 7, 257), (250, 10, 1000), (250, 10, 7105), (256, 16, 65),
              (300, 6, 200), (512, 10, 97), (700, 12, 50), (1000, 10, 130), (1024, 24, 33), (1100, 3, 500), (96, 32, 70)]
    for (M, D, N) in shapes:
        inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=M + D)
        td = torch.from_numpy(testing).cuda()
        for sym in ((False, True) if M <= 1024 else (False,)):
            m = gpemu.DeviceModel(inputs, theta, invQt, invQ, symmetric_variance=sym)
            for hess in (False, True):
                bufs = {k: _guarded(s) for k, s in (("mu", (N,)), ("var", (N,)), ("deriv", (N, D)), ("hess", (N, D, D)))
                        if hess or k != "hess"}
                for b, v in bufs.values():
                    v.fill_(float("inf"))
                m.predict(td, want_hess=hess, out={k: v for k, (b, v) in bufs.items()})
                torch.cuda.synchronize()
                for k, (b, v) in bufs.items():
                    assert _guards_intact(b, v.numel()), (M, D, N, sym, hess, k)
                    assert bool(torch.isfinite(v).all()), (M, D, N, sym, hess, k)
            m.close()
    # single precision (float32 outputs: guard with a float32 NaN pattern)
    for (M, D, N) in [(250, 10, 300), (100, 3, 129), (600, 10, 200), (1024, 16, 70)]:
        inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=M)
        m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
        lib = gpemu._lib.load()
        t32 = torch.from_numpy(testing.astype(np.float32)).cuda()
        G = 4096
        bufs = {k: torch.full((G + n + G,), float("nan"), dtype=torch.float32, device="cuda")
                for k, n in (("mu", N), ("var", N), ("deriv", N * D))}
        for fast in (0, gpemu._lib.F32_FAST_TF32):
            for b in bufs.values():
                b[G:-G] = float("inf")
            gpemu._lib.check(lib.gpe_predict_f32(m._h, t32.data_ptr(), N, bufs["mu"][G:].data_ptr(), bufs["var"][G:].data_ptr(),
                                                 bufs["deriv"][G:].data_ptr(), 7 | fast,
                                                 torch.cuda.current_stream().cuda_stream))
            torch.cuda.synchronize()
            for k, b in bufs.items():
                assert bool(torch.isnan(b[:G]).all()) and bool(torch.isnan(b[-G:]).all()), (M, D, N, fast, k)
                assert bool(torch.isfinite(b[G:-G]).all()), (M, D, N, fast, k)
        m.close()
    # bank: strided point-major outputs, Hessian, projection (incl. a slice boundary at E = 33 and odd W)
    for (M, D, E, W, N) in [(60, 4, 5, 301, 150), (40, 3, 33, 77, 90), (250, 10, 3, 2101, 70)]:
        inputs = rs.random_sample((M, D))
        thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)); invQs = rs.random_sample((E, M, M))
        basis = rs.standard_normal((E, W))
        bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=basis)
        td = torch.from_numpy(rs.random_sample((N, D))).cuda()
        lib = gpemu._lib.load()
        bufs = {k: _guarded(s) for k, s in (("mu", (N, E)), ("var", (N, E)), ("deriv", (N, E, D)), ("hess", (N, E, D, D)),
                                            ("fwd", (N, W)), ("deriv_full", (N, D, W)))}
        for b, v in bufs.values():
            v.fill_(float("inf"))
        gpemu._lib.check(lib.gpe_bank_predict_ex(bank._h, td.data_ptr(), N, *[bufs[k][1].data_ptr() for k in
                                                 ("mu", "var", "deriv", "hess", "fwd", "deriv_full")], 0x3F,
                                                 torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        for k, (b, v) in bufs.items():
            assert _guards_intact(b, v.numel()), (M, D, E, W, N, k)
            assert bool(torch.isfinite(v).all()), (M, D, E, W, N, k)
        bank.close()


def test_multi_device_nvlink_relay_of_host_traffic(lib, gpemu, monkeypatch):
    """gpe_multi_predict can send a device's host traffic through a partner's PCIe link (host -> partner -> NVLink ->
    device -> NVLink -> partner -> host) when its own link is measured to be much slower; forced here
    (GPE_MULTI_RELAY=force: first half of the device list relays through the second half).  Bit-identical results."""
    import torch
    ndev = lib.gpe_device_count()
    devices = list(range(ndev)) if ndev > 1 else [0, 0]
    inputs, theta, invQ, invQt, _ = orc.make_S_model(250, 10, 1, seed=21)
    N = 700_001
    t = torch.rand(N, 10, dtype=torch.float64, generator=torch.Generator().manual_seed(3)).pin_memory().numpy()
    out = {k: torch.empty(s, dtype=torch.float64).pin_memory().numpy() for k, s in
           (("mu", (N,)), ("var", (N,)), ("deriv", (N, 10)))}
    ref = gpemu.DeviceModel(inputs, theta, invQt, invQ).predict(t)
    monkeypatch.setenv("GPE_MULTI_RELAY", "force")
    mm = gpemu.MultiDeviceModel(inputs, theta, invQt, invQ, devices=devices)
    for _ in range(2):
        for v in out.values():
            v.fill(np.nan)
        got = mm.predict(t, out=out)
        for k in ("mu", "var", "deriv"):
            assert np.array_equal(got[k], ref[k]), k
    mm.close()
    # banks take the same route (test points and per-point observations in, any bank output out)
    rs = np.random.RandomState(6)
    Mb, Db, E, Nb = 60, 4, 5, 300_000
    binp = rs.random_sample((Mb, Db))
    thetas = rs.random_sample((E, Db + 2)); invQts = rs.random_sample((E, Mb)); invQs = rs.random_sample((E, Mb, Mb))
    tb = torch.rand(Nb, Db, dtype=torch.float64, generator=torch.Generator().manual_seed(4)).pin_memory().numpy()
    obs = torch.rand(Nb, E, dtype=torch.float64, generator=torch.Generator().manual_seed(5)).pin_memory().numpy()
    b1 = gpemu.DeviceBank(binp, thetas, invQts, invQs, device=0)
    bn = gpemu.DeviceBank(binp, thetas, invQts, invQs, device=devices)
    r1 = b1.predict(tb, pinned=True); rn = bn.predict(tb, pinned=True)
    for k in r1:
        assert np.array_equal(r1[k], rn[k]), k
    c1 = b1.cost(tb, obs); cn = bn.cost(tb, obs)
    assert np.array_equal(c1["cost"], cn["cost"]) and np.array_equal(c1["grad"], cn["grad"])
    monkeypatch.setenv("GPE_MULTI_RELAY", "off")
    mm = gpemu.MultiDeviceModel(inputs, theta, invQt, invQ, devices=devices)
    got = mm.predict(t, out=out)
    for k in ("mu", "var", "deriv"):
        assert np.array_equal(got[k], ref[k]), k


# ---- banks: mean + gradient on shared input differences (predict_bank_mean.cuh) ----
@pytest.mark.parametrize("M,D,E,N", [
    (250, 10, 20, 1037),   # BASELINE config 4's bank: groups of 5
    (250, 10, 64, 333),    # config 5's bank without the variance: 13 groups, the last one padded
    (37, 3, 7, 131),       # ragged everything, DP = 4
    (60, 5, 3, 1),         # one group of 3, one point, D odd (DP = 6)
    (300, 8, 11, 95),      # two training chunks (M > 256)
    (530, 11, 6, 64),      # three chunks, DP = 12: groups of 3
    (45, 14, 5, 77),       # DP = 16: groups of 3 and 2
    (33, 2, 4, 4097),      # DP = 2, many tiles per CTA
    (20, 20, 4, 50),       # DP = 24: no group kernel, one-emulator path
    (50, 6, 2, 40),        # E < 3: one-emulator path
])
def test_bank_mean_gradient_shared_differences(gpemu, M, D, E, N):
    """Mean and gradient of a bank without the variance (MultivariateEmulator.predict, multivariate_gp.py:195-222; per-band
    banks): E oracle predicts on the same test points against one launch that shares x_j - t_n between the emulators of a
    group.  Host and device callers; mean-only and gradient-only requests."""
    import torch
    rs = np.random.RandomState(7 * M + E)
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.randn(E, M); invQs = rs.random_sample((E, M, M))
    bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs)
    # the group kernel serves calls whose CTAs fill the machine (tiles x groups >= #SMs); smaller calls stay on the
    # one-emulator kernel: the first N points are also run as a call of their own
    n_small = N
    N = N + 32 * torch.cuda.get_device_properties(0).multi_processor_count
    t = rs.random_sample((N, D))
    models = [(inputs, thetas[e], invQs[e], invQts[e]) for e in range(E)]
    mu_o, _, grad_o = orc.bank_predict(models, t)
    host = bank.predict(t, want_var=False, want_deriv=True)
    dev = bank.predict(torch.from_numpy(t).cuda(), want_var=False, want_deriv=True)
    for name, got in (("host", host), ("device", {k: v.cpu().numpy() for k, v in dev.items()})):
        assert got["mu"].shape == (N, E) and got["deriv"].shape == (N, E, D), name
        assert orc.ref_err(got["mu"], mu_o) < TOL, name
        assert orc.ref_err(got["deriv"], grad_o) < TOL, name
        for e in range(E):   # per emulator too: a small-output emulator must not hide behind a large one
            assert orc.ref_err(got["mu"][:, e], mu_o[:, e]) < TOL, (name, e)
            assert orc.ref_err(got["deriv"][:, e], grad_o[:, e]) < TOL, (name, e)
    small = bank.predict(t[:n_small], want_var=False, want_deriv=True)
    assert orc.ref_err(small["mu"], mu_o[:n_small]) < TOL and orc.ref_err(small["deriv"], grad_o[:n_small]) < TOL
    mu_only = bank.predict(t, want_var=False, want_deriv=False)      # means-only variant: larger groups
    assert orc.ref_err(mu_only["mu"], mu_o) < TOL
    for e in range(E):
        assert orc.ref_err(mu_only["mu"][:, e], mu_o[:, e]) < TOL, e
    # the variance path (per-emulator fused launches) agrees with it to rounding
    full = bank.predict(t, want_var=True, want_deriv=True)
    assert orc.ref_err(full["mu"], host["mu"]) < 1e-13 and orc.ref_err(full["deriv"], host["deriv"]) < 1e-13


def test_non_finite_and_far_away_test_points_follow_numpy(gpemu):
    """Edge rows the reference handles by IEEE arithmetic (GaussianProcess.py:228-247): a test point so far away that every
    covariance underflows (mu = 0, var = b, deriv = 0), one with a NaN coordinate (its outputs are NaN, nobody else's) and
    one with an infinite coordinate (exp(-inf) = 0: mu = 0, var = b; the gradient is 0 * inf = NaN in that dimension).
    Same pattern of non-finite values as numpy, same finite values, for the fused, the mean-only and the bank kernels."""
    rs = np.random.RandomState(77)
    M, D, E = 120, 5, 6
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, 70, seed=5)
    testing = testing.copy()
    testing[3] = 1e3                       # exponent ~ -1e6: underflow
    testing[10] = 40.0                     # exponent ~ -2e3: below the normal range
    testing[17, 2] = np.nan
    testing[33, 0] = np.inf
    testing[34, 4] = -np.inf
    testing[50] = 1e200                    # squares overflow to inf

    def same(got, ref, what):
        assert np.array_equal(np.isnan(got), np.isnan(ref)), what
        ok = np.isfinite(ref)
        assert np.array_equal(np.isfinite(got), ok), what
        assert orc.ref_err(got[ok], ref[ok]) < TOL, what

    with np.errstate(all="ignore"):
        mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
    assert mu[3] == 0.0 and mu[50] == 0.0 and np.isnan(mu[17]) and np.isnan(deriv[33, 0]) and mu[33] == 0.0
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    full = m.predict(testing)
    mean_only = m.predict(testing, want_var=False)
    for k, r in (("mu", mu), ("var", var), ("deriv", deriv)):
        same(full[k], r, ("fused", k))
        if k != "var":
            same(mean_only[k], r, ("mean", k))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.randn(E, M)
    bank = gpemu.DeviceBank(inputs, thetas, invQts, None)
    with np.errstate(all="ignore"):
        mu_b, _, grad_b = orc.bank_predict([(inputs, thetas[e], invQ, invQts[e]) for e in range(E)], testing)
    got = bank.predict(testing, want_var=False, want_deriv=True)          # small call: one-emulator kernel
    same(got["mu"], mu_b, "bank mu"); same(got["deriv"], grad_b, "bank deriv")
    big = np.tile(testing, (80, 1))                                        # enough tiles for the group kernels
    got = bank.predict(big, want_var=False, want_deriv=True)
    same(got["mu"], np.tile(mu_b, (80, 1)), "bank mu, groups"); same(got["deriv"], np.tile(grad_b, (80, 1, 1)), "bank deriv, groups")
    same(bank.predict(big, want_var=False, want_deriv=False)["mu"], np.tile(mu_b, (80, 1)), "bank means only, groups")


@pytest.mark.parametrize("M,D,N", [(60, 33, 37), (250, 40, 300), (7, 64, 1), (130, 100, 50), (1100, 36, 20), (40, 256, 33)])
def test_more_than_32_inputs_generic_path(gpemu, M, D, N):
    """D > 32 (the reference loops `for d in range(self.D)`, no limit: GaussianProcess.py:228-247, :345-366): generic
    kernels on the K* scratch + the column-pass variance kernel (predict_generic.cuh).  Mean, variance, gradient and
    Hessian against the oracle, host and device callers, more points than one sub-batch, and through the drop-in class."""
    import torch
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=D)
    theta = theta.copy(); theta[:D] -= np.log(D / 8.0)        # keep sum_d w_d (x - t)^2 in a range where K* is not ~ 0
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
    hess = orc.hessian(inputs, theta, invQt, testing[:8])
    assert np.max(np.abs(mu)) > 1e-3
    host = m.predict(testing, want_hess=True)
    dev = {k: v.cpu().numpy() for k, v in m.predict(torch.from_numpy(testing).cuda(), want_hess=True).items()}
    for name, got in (("host", host), ("device", dev)):
        assert orc.ref_err(got["mu"], mu) < TOL and orc.ref_err(got["var"], var) < TOL, name
        assert orc.ref_err(got["deriv"], deriv) < TOL and orc.ref_err(got["hess"][:8], hess) < TOL, name
    o = m.predict(testing, want_var=False, want_mu=False)
    assert set(o) == {"deriv"} and np.array_equal(o["deriv"], host["deriv"])
    gp = gpemu.GaussianProcess(inputs, np.zeros(M))
    gp.theta, gp.invQ, gp.invQt = theta, invQ, invQt
    r = gp.predict(testing)
    assert orc.ref_err(r[0], mu) < TOL and orc.ref_err(r[1], var) < TOL and orc.ref_err(r[2], deriv) < TOL
    assert orc.ref_err(gp.hessian(testing[:8]), hess) < TOL


def test_more_than_32_inputs_many_points_and_bank(gpemu):
    """Sub-batches of the K* scratch (N > 16 * 4 * #SMs) and a bank of D = 35 emulators (strided point-major outputs)."""
    rs = np.random.RandomState(35)
    M, D, E, N = 90, 35, 3, 12_001
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)) - np.log(D / 8.0); invQts = rs.randn(E, M); invQs = rs.random_sample((E, M, M))
    t = rs.random_sample((N, D))
    bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs)
    got = bank.predict(t, want_var=True, want_deriv=True)
    idx = np.r_[0:40, N - 40:N, rs.randint(0, N, 60)]
    mu_o, var_o, grad_o = orc.bank_predict([(inputs, thetas[e], invQs[e], invQts[e]) for e in range(E)], t[idx])
    assert orc.ref_err(got["mu"][idx], mu_o) < TOL and orc.ref_err(got["var"][idx], var_o) < TOL
    assert orc.ref_err(got["deriv"][idx], grad_o) < TOL
    nv = bank.predict(t[:500], want_var=False, want_deriv=True)
    assert np.array_equal(nv["mu"], got["mu"][:500]) and np.array_equal(nv["deriv"], got["deriv"][:500])


@pytest.mark.parametrize("M,D", [(250, 10), (8, 2), (37, 3), (100, 1), (129, 16), (200, 7), (256, 12), (31, 5)])
def test_handful_of_points_cluster_path(gpemu, M, D):
    """Calls of a few points with variance (what the reference is mostly used for, GaussianProcess.py:327-341) run one
    8-CTA cluster per 16-point tile (predict_tiny.cuh).  Parity at every size around the tile and the switch to the
    16-point plan, host and device callers, strided bank outputs, a symmetric-folded model, outputs requested one by one."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n_max = 16 * (2 * sms // 8)
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, n_max + 40, seed=M + D)
    mu, var, deriv = orc.predict(inputs, theta, invQ, invQt, testing)
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    assert "k_predict_tiny" in m.plan(1) and "k_predict_tiny" in m.plan(n_max) and "k_predict_tiny" not in m.plan(n_max + 1)
    for n in (1, 2, 15, 16, 17, 33, n_max - 1, n_max, n_max + 1):
        o = m.predict(testing[:n])
        assert orc.ref_err(o["mu"], mu[:n]) < TOL and orc.ref_err(o["var"], var[:n]) < TOL, n
        assert orc.ref_err(o["deriv"], deriv[:n]) < TOL, n
    d = m.predict(torch.from_numpy(testing[:19]).cuda(), want_mu=False, want_deriv=False)
    assert set(d) == {"var"} and orc.ref_err(d["var"].cpu().numpy(), var[:19]) < TOL
    ms = gpemu.DeviceModel(inputs, theta, invQt, invQ, symmetric_variance=True)
    assert orc.ref_err(ms.predict(testing[:21])["var"], var[:21]) < TOL
    if M == 250:
        rs = np.random.RandomState(3)
        E = 3
        thetas = rs.random_sample((E, D + 2)); invQts = rs.randn(E, M); invQs = rs.random_sample((E, M, M))
        bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs)
        mu_b, var_b, grad_b = orc.bank_predict([(inputs, thetas[e], invQs[e], invQts[e]) for e in range(E)], testing[:20])
        got = bank.predict(testing[:20], want_var=True, want_deriv=True)
        assert orc.ref_err(got["mu"], mu_b) < TOL and orc.ref_err(got["var"], var_b) < TOL
        assert orc.ref_err(got["deriv"], grad_b) < TOL


def test_concurrent_device_calls_on_shared_handles(gpemu):
    """include/gpemu.h allows device-pointer calls on one handle from several threads, each on its own stream.  The paths
    added in round 2 under that contract: the cluster path (no shared state), the generic D > 32 path (one K* scratch per
    model: mutex + event), and a bank on the shared-difference kernel.  Every thread must get exactly the serial result."""
    import threading
    import torch
    rs = np.random.RandomState(21)
    cases = []
    inputs, theta, invQ, invQt, t = orc.make_S_model(250, 10, 300, seed=3)            # cluster path
    cases.append((gpemu.DeviceModel(inputs, theta, invQt, invQ), t, dict()))
    inputs, theta, invQ, invQt, t = orc.make_S_model(120, 40, 5000, seed=4)           # generic path, several sub-batches
    theta = theta.copy(); theta[:40] -= np.log(5.0)
    cases.append((gpemu.DeviceModel(inputs, theta, invQt, invQ), t, dict()))
    M, D, E = 100, 6, 7                                                                # bank, group kernel (N large enough)
    binp = rs.random_sample((M, D)); thetas = rs.random_sample((E, D + 2)); invQts = rs.randn(E, M)
    cases.append((gpemu.DeviceBank(binp, thetas, invQts), rs.random_sample((6000, D)), dict(want_var=False, want_deriv=True)))
    for handle, t, kw in cases:
        td = torch.from_numpy(np.ascontiguousarray(t)).cuda()
        serial = {k: v.clone() for k, v in handle.predict(td, **kw).items()}
        torch.cuda.synchronize()
        results, errors = [None] * 6, []

        def work(i):
            try:
                s = torch.cuda.Stream()
                with torch.cuda.stream(s):
                    outs = [handle.predict(td, **kw) for _ in range(4)]
                s.synchronize()
                results[i] = outs
            except Exception as e:     # noqa: BLE001 -- reported below
                errors.append(e)

        threads = [threading.Thread(target=work, args=(i,)) for i in range(6)]
        for th in threads: th.start()
        for th in threads: th.join()
        assert not errors, errors
        for outs in results:
            for o in outs:
                for k in serial:
                    assert torch.equal(o[k], serial[k]), (type(handle).__name__, k)
