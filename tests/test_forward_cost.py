"""Forward cost of a bank with a basis (gpe_bank_forward_cost*, DeviceBank.forward_cost, MultivariateEmulator.cost):
the misfit of the back-projected spectra against observed spectra and its input gradient, reduced on the device.

The reference for it is what a user of the reference library writes: materialise fwd (N, W) and deriv_full (N, D, W)
(multivariate_gp.py:216,218, batched) and reduce them in numpy (``mv_cost`` below)."""
import ctypes as C

import numpy as np
import pytest

from oracle import gp_oracle as orc
from tests.conftest import golden

pytestmark = pytest.mark.gpu
TOL = 1e-10


def mv_cost(models, basis, testing, obs, weights=None):
    """cost_n = 1/2 sum_w l_w (fwd_nw - obs_nw)^2, grad_nd = sum_w l_w (fwd_nw - obs_nw) deriv_full_ndw, materialised."""
    fwd, _, _, _, dfull = orc.mv_predict_batch(models, basis, testing, want_deriv_full=True)
    lam = np.ones(basis.shape[1]) if weights is None else np.asarray(weights)
    r = fwd - np.asarray(obs)
    return 0.5 * np.sum(lam * r * r, axis=1), np.einsum("ndw,nw->nd", dfull, lam * r)


@pytest.fixture(scope="module")
def gpemu(lib):
    import gp_emulator_b200 as g
    assert lib.gpe_device_count() > 0, "no GPU visible: the gpu tests must not pass on a fallback"
    return g


def _problem(gpemu, E, W, D, M=40, seed=0, device=0, basis=True):
    rs = np.random.RandomState(seed + 7 * E + W + D)
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)); invQs = rs.random_sample((E, M, M))
    B = rs.standard_normal((E, W)) if basis else None
    bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=B, device=device)
    models = [(inputs, thetas[e], invQs[e], invQts[e]) for e in range(E)]
    return bank, models, B, rs


@pytest.mark.parametrize("E,W,D,N", [(1, 1, 1, 1), (5, 7, 4, 7), (12, 128, 10, 255), (20, 2101, 10, 256),
                                     (32, 129, 16, 3000), (40, 129, 4, 300), (20, 128, 1, 3000), (40, 7, 10, 1)])
def test_oracle_parity(gpemu, E, W, D, N):
    import torch
    bank, models, B, rs = _problem(gpemu, E, W, D)
    t = rs.random_sample((N, D))
    fwd = orc.mv_predict_batch(models, B, t)[0]
    obs1 = fwd.mean(axis=0) * 1.1 + 0.01                                  # one observed spectrum for every point
    obsN = fwd * (1.0 + 0.1 * rs.standard_normal(fwd.shape))
    w = rs.random_sample(W) + 0.5
    wz = w * (rs.random_sample(W) < 0.7)                                 # weights with zeros
    for obs, wt in ((obs1, None), (obsN, w), (obs1, wz), (obsN, None)):
        c_o, g_o = mv_cost(models, B, t, obs, wt)
        got = bank.forward_cost(t, obs, wt)
        assert got["cost"].shape == (N,) and got["grad"].shape == (N, D)
        assert orc.ref_err(got["cost"], c_o) < TOL and orc.ref_err(got["grad"], g_o) < TOL
    only = bank.forward_cost(t, obsN, wz, want_grad=False)
    assert set(only) == {"cost"} and orc.ref_err(only["cost"], mv_cost(models, B, t, obsN, wz)[0]) < TOL
    dev = bank.forward_cost(torch.from_numpy(t).cuda(), torch.from_numpy(obsN).cuda(), torch.from_numpy(w).cuda())
    c_o, g_o = mv_cost(models, B, t, obsN, w)
    assert dev["cost"].is_cuda and orc.ref_err(dev["cost"].cpu().numpy(), c_o) < TOL
    assert orc.ref_err(dev["grad"].cpu().numpy(), g_o) < TOL


def test_device_call_with_padded_observation_rows(lib, gpemu):
    """obs_ld > W through the C ABI (the Python layer always passes contiguous rows)."""
    import torch
    E, W, D, N = 20, 129, 6, 300
    bank, models, B, rs = _problem(gpemu, E, W, D)
    t = rs.random_sample((N, D))
    obs = orc.mv_predict_batch(models, B, t)[0] * (1.0 + 0.1 * rs.standard_normal((N, W)))
    w = rs.random_sample(W)
    ld = W + 5
    big = torch.full((N, ld), float("nan"), dtype=torch.float64, device="cuda")
    big[:, :W] = torch.from_numpy(obs).cuda()
    td, wd = torch.from_numpy(t).cuda(), torch.from_numpy(w).cuda()
    cost = torch.empty(N, dtype=torch.float64, device="cuda"); grad = torch.empty(N, D, dtype=torch.float64, device="cuda")
    assert lib.gpe_bank_forward_cost(bank._h, td.data_ptr(), N, big.data_ptr(), ld, wd.data_ptr(), cost.data_ptr(),
                                     grad.data_ptr(), None) == 0
    torch.cuda.synchronize()
    ref = bank.forward_cost(td, torch.from_numpy(obs).cuda(), wd)
    assert torch.equal(cost, ref["cost"]) and torch.equal(grad, ref["grad"])
    c_o, g_o = mv_cost(models, B, t, obs, w)
    assert orc.ref_err(cost.cpu().numpy(), c_o) < TOL and orc.ref_err(grad.cpu().numpy(), g_o) < TOL


def test_pinned_to_the_reference_outputs(gpemu):
    """PROSAIL emulator: against the reference's own frozen fwd and its Jacobian on the wsub columns, with weights
    nonzero only on wsub."""
    from tests.test_gpu_parity import _write_prosail_dump
    g = golden("P")
    mv = gpemu.MultivariateEmulator(X=None, y=None, dump=_write_prosail_dump(g))
    for i, gp in enumerate(mv.emulators):       # the frozen state the reference's outputs were made with
        gp.invQt = g["invQt"][i]
    rs = np.random.RandomState(5)
    W = g["fwd"].shape[1]
    lam = np.zeros(W)
    lam[g["wsub"]] = rs.random_sample(len(g["wsub"])) + 0.5
    obs = g["fwd"] * (1.0 + 0.05 * rs.standard_normal(g["fwd"].shape))
    r = (g["fwd"] - obs)[:, g["wsub"]] * lam[g["wsub"]]
    c_ref = 0.5 * np.sum(r * (g["fwd"] - obs)[:, g["wsub"]], axis=1)
    g_ref = np.einsum("ndw,nw->nd", g["deriv_sub"], r)
    c, gr = mv.cost(g["points"], obs, lam)
    assert c.shape == (3,) and gr.shape == (3, 10)
    assert orc.ref_err(c, c_ref) < TOL and orc.ref_err(gr, g_ref) < TOL
    for k in range(3):                           # one point: the reference's call shape
        c1, g1 = mv.cost(g["points"][k], obs[k], lam)
        assert isinstance(c1, float) and g1.shape == (10,)
        # (the frozen Jacobian's rounding is relative to its own size, not to a small residual: scale of the batch)
        assert abs(c1 - c_ref[k]) <= TOL * abs(c_ref).max() and np.max(np.abs(g1 - g_ref[k])) <= TOL * abs(g_ref).max()
    c_only = mv.cost(g["points"][0], obs[0], lam, do_deriv=False)
    assert isinstance(c_only, float) and abs(c_only - c_ref[0]) <= TOL * abs(c_ref).max()
    fwd = mv.predict(g["points"][0], do_deriv=False)             # a point scored against its own prediction
    assert mv.cost(g["points"][0], fwd, do_deriv=False) == 0.0


@pytest.mark.parametrize("E", [12, 20, 32, 40])
def test_own_forward_gives_exact_zero(gpemu, E):
    W, D, N = 2101, 10, 300
    bank, models, B, rs = _problem(gpemu, E, W, D)
    t = rs.random_sample((N, D))
    full = bank.predict(t, want_var=False, want_deriv=False, want_mu=False, project=True, project_deriv=True)
    got = bank.forward_cost(t, full["fwd"])
    assert np.all(got["cost"] == 0.0) and np.all(got["grad"] == 0.0)
    fwd = bank.predict(t, want_var=False, want_deriv=False, want_mu=False, project=True)["fwd"]
    assert np.all(bank.forward_cost(t, fwd, want_grad=False)["cost"] == 0.0)


def test_seams_and_placement_are_invisible(lib, gpemu, monkeypatch):
    import torch
    from gp_emulator_b200.engine import _pinned_empty
    E, W, D = 20, 129, 10
    bank, models, B, rs = _problem(gpemu, E, W, D)
    N = 40000
    t = rs.random_sample((N, D))
    obs = rs.standard_normal((N, W))
    w = rs.random_sample(W)
    ref = bank.forward_cost(t, obs, w)                                     # staged, one chunk per pipeline slot plan
    monkeypatch.setenv("GPE_SLOT_OUT_BYTES", str(8 * (D + 1) * 997))       # chunks of 997 points
    seams = bank.forward_cost(t, obs, w)
    monkeypatch.delenv("GPE_SLOT_OUT_BYTES")
    assert np.array_equal(seams["cost"], ref["cost"]) and np.array_equal(seams["grad"], ref["grad"])
    dev = bank.forward_cost(torch.from_numpy(t).cuda(), torch.from_numpy(obs).cuda(), torch.from_numpy(w).cuda())
    assert np.array_equal(dev["cost"].cpu().numpy(), ref["cost"]) and np.array_equal(dev["grad"].cpu().numpy(), ref["grad"])
    two = gpemu.DeviceBank(*_inputs_of(models), basis=B, device=[0, 0] if lib.gpe_device_count() == 1 else "all")
    multi = two.forward_cost(t, obs, w)
    assert np.array_equal(multi["cost"], ref["cost"]) and np.array_equal(multi["grad"], ref["grad"])
    obs1 = obs[0]
    ref1 = bank.forward_cost(t, obs1)
    assert np.array_equal(two.forward_cost(t, obs1)["grad"], ref1["grad"])
    # a tiny call on mapped buffers (pageable inputs) against the same call with page-locked inputs (copied, results
    # staged) and with device pointers.  (Not against rows of the large call: the kernels that form the bank means
    # follow the size of the call.)
    n = 100
    tiny = bank.forward_cost(t[:n], obs[:n], w)
    tp, op = _pinned_empty((n, D)), _pinned_empty((n, W))
    tp[:], op[:] = t[:n], obs[:n]
    staged = bank.forward_cost(tp, op, w)
    dev = bank.forward_cost(torch.from_numpy(t[:n]).cuda(), torch.from_numpy(obs[:n]).cuda(), torch.from_numpy(w).cuda())
    for k in ("cost", "grad"):
        assert np.array_equal(tiny[k], staged[k]) and np.array_equal(tiny[k], dev[k].cpu().numpy())
    assert not np.array_equal(tiny["cost"], np.zeros(n))


def _inputs_of(models):
    inputs = models[0][0]
    return inputs, np.stack([m[1] for m in models]), np.stack([m[3] for m in models]), np.stack([m[2] for m in models])


@pytest.mark.parametrize("E,W,D,N", [(20, 129, 10, 97), (40, 2101, 3, 33), (5, 7, 2, 1)])
def test_red_zones(lib, gpemu, E, W, D, N):
    """Outputs between NaN guard bands, device and host pointers: the bands stay untouched, every element is written."""
    import torch
    bank, models, B, rs = _problem(gpemu, E, W, D)
    t = rs.random_sample((N, D))
    obs = rs.standard_normal((N, W))
    g = 4096
    for host in (False, True):
        mk = (lambda n: np.full(n, np.nan)) if host else (lambda n: torch.full((n,), float("nan"), dtype=torch.float64, device="cuda"))
        cbig, gbig = mk(N + 2 * g), mk(N * D + 2 * g)
        if host:
            p = lambda a: a.ctypes.data + 8 * g
            rc = lib.gpe_bank_forward_cost_host(bank._h, t.ctypes.data, N, obs.ctypes.data, W, None, p(cbig), p(gbig))
        else:
            td, od = torch.from_numpy(t).cuda(), torch.from_numpy(obs).cuda()
            p = lambda a: a.data_ptr() + 8 * g
            rc = lib.gpe_bank_forward_cost(bank._h, td.data_ptr(), N, od.data_ptr(), W, None, p(cbig), p(gbig), None)
            torch.cuda.synchronize()
            cbig, gbig = cbig.cpu().numpy(), gbig.cpu().numpy()
        assert rc == 0
        for big, n in ((cbig, N), (gbig, N * D)):
            assert np.all(np.isnan(big[:g])) and np.all(np.isnan(big[g + n:])) and np.all(np.isfinite(big[g:g + n]))
        c_o, g_o = mv_cost(models, B, t, obs)
        assert orc.ref_err(cbig[g:g + N], c_o) < TOL and orc.ref_err(gbig[g:g + N * D].reshape(N, D), g_o) < TOL


def test_nan_observation_propagates_at_zero_weight(gpemu):
    E, W, D, N = 12, 129, 4, 5
    bank, models, B, rs = _problem(gpemu, E, W, D)
    t = rs.random_sample((N, D))
    obs = rs.standard_normal((N, W))
    obs[2, 17] = np.nan
    w = np.ones(W); w[17] = 0.0
    got = bank.forward_cost(t, obs, w)
    c_o, g_o = mv_cost(models, B, t, obs, w)
    assert np.isnan(c_o[2]) and np.all(np.isnan(g_o[2]))
    assert np.isnan(got["cost"][2]) and np.all(np.isnan(got["grad"][2]))
    keep = [0, 1, 3, 4]
    assert orc.ref_err(got["cost"][keep], c_o[keep]) < TOL and orc.ref_err(got["grad"][keep], g_o[keep]) < TOL


def test_argument_errors(lib, gpemu):
    import torch
    E, W, D, N = 5, 9, 3, 4
    bank, models, B, rs = _problem(gpemu, E, W, D)
    nob, _, _, _ = _problem(gpemu, E, W, D, basis=False)
    t = rs.random_sample((N, D)); obs = rs.standard_normal((N, W)); c = np.empty(N); gr = np.empty((N, D))
    a = lambda x: x.ctypes.data
    host, dev = lib.gpe_bank_forward_cost_host, lib.gpe_bank_forward_cost
    assert host(nob._h, a(t), N, a(obs), W, None, a(c), a(gr)) == -1                 # bank without a basis
    assert host(bank._h, a(t), N, a(obs), W, None, None, None) == -1                 # nothing requested
    assert host(bank._h, a(t), N, None, W, None, a(c), a(gr)) == -1                 # obs NULL, N > 0
    assert host(bank._h, a(t), N, a(obs), W + 1, None, a(c), a(gr)) == -1            # host rows must be contiguous
    assert host(bank._h, a(t), -1, a(obs), W, None, a(c), a(gr)) == -1               # N < 0
    assert host(bank._h, None, 0, None, W, None, a(c), a(gr)) == 0                   # N = 0: nothing to do
    td = torch.from_numpy(t).cuda(); od = torch.from_numpy(obs).cuda()
    cd = torch.empty(N, dtype=torch.float64, device="cuda"); gd = torch.empty(N, D, dtype=torch.float64, device="cuda")
    p = lambda x: x.data_ptr()
    assert dev(nob._h, p(td), N, p(od), W, None, p(cd), p(gd), None) == -1
    assert dev(bank._h, p(td), N, p(od), W, None, None, None, None) == -1
    assert dev(bank._h, p(td), N, None, W, None, p(cd), p(gd), None) == -1
    assert dev(bank._h, p(td), N, p(od), W - 1, None, p(cd), p(gd), None) == -1     # 0 < obs_ld < W
    assert dev(bank._h, p(td), -1, p(od), W, None, p(cd), p(gd), None) == -1
    assert dev(bank._h, p(td), 0, None, W, None, p(cd), p(gd), None) == 0
    assert lib.gpe_multi_bank_forward_cost(None, a(t), N, a(obs), W, None, a(c), a(gr)) == -1
    with pytest.raises(gpemu.GpemuError):
        nob.forward_cost(t, obs)
    with pytest.raises(ValueError):
        bank.forward_cost(t, np.zeros(W + 1))
    with pytest.raises(ValueError):
        bank.forward_cost(t, obs, np.ones(W - 1))
    big, _, _, _ = _problem(gpemu, 97, 8, 2, M=6)                                  # beyond the kernel's shared memory
    with pytest.raises(gpemu.GpemuError):
        big.forward_cost(rs.random_sample((3, 2)), np.zeros(8))
