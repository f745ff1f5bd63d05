"""Input Hessian of the bank costs (gpe_bank_cost_ex, gpe_bank_forward_cost_ex and their host / multi-device variants,
DeviceBank.cost / forward_cost with want_hess, MultivariateEmulator.cost with do_hess), reduced on the device.

The references are what a user of the reference library builds: the per-emulator Hessians of E separate predicts
(``orc.bank_predict(..., do_hess=True)``) and, for the spectra, the materialised Jacobian J (N, D, W) reduced in numpy.
The spectra reference sums over wavelengths and never forms C = basis . diag(l) . basis^T, so the library's C route is
checked independently."""
import numpy as np
import pytest

from oracle import gp_oracle as orc
from tests.conftest import golden

TOL = 1e-10


def bank_cost_hess_ref(models, testing, obs, weights=None):
    """cost, grad, hess of 1/2 sum_e w_e (mu_ne - obs_ne)^2, and the magnitude sum of hess (the same two sums over
    absolute values)."""
    mu, _, G, H = orc.bank_predict(models, testing, do_hess=True)
    w = np.ones(mu.shape[1]) if weights is None else np.asarray(weights)
    r = mu - np.asarray(obs)
    c = w * r
    hess = np.einsum("ne,nedk->ndk", c, H) + np.einsum("e,ned,nek->ndk", w, G, G)
    mag = np.einsum("ne,nedk->ndk", np.abs(c), np.abs(H)) + np.einsum("e,ned,nek->ndk", np.abs(w), np.abs(G), np.abs(G))
    return 0.5 * np.sum(c * r, axis=1), np.einsum("ne,ned->nd", c, G), hess, mag


def mv_cost_hess_ref(models, basis, testing, obs, weights=None):
    """cost, grad, hess of 1/2 sum_w l_w (fwd_nw - obs_nw)^2 with J = d fwd / dx materialised, and the magnitude sum."""
    mu, _, G, H = orc.bank_predict(models, testing, do_hess=True)
    lam = np.ones(basis.shape[1]) if weights is None else np.asarray(weights)
    r = mu @ basis - np.asarray(obs)
    J = np.einsum("ned,ew->ndw", G, basis)
    lr = lam * r
    hess = np.einsum("ndw,w,nkw->ndk", J, lam, J) + np.einsum("nedk,ew,nw->ndk", H, basis, lr)
    mag = np.einsum("ndw,w,nkw->ndk", np.abs(J), np.abs(lam), np.abs(J)) + \
        np.einsum("nedk,ew,nw->ndk", np.abs(H), np.abs(basis), np.abs(lr))
    return 0.5 * np.sum(lr * r, axis=1), np.einsum("ndw,nw->nd", J, lr), hess, mag


def _models(E, D, M, seed):
    rs = np.random.RandomState(seed + 11 * E + 3 * D + M)
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)); invQts = rs.random_sample((E, M)); invQs = rs.random_sample((E, M, M))
    return inputs, thetas, invQts, invQs, rs


def _as_models(inputs, thetas, invQts, invQs):
    return [(inputs, thetas[e], invQs[e], invQts[e]) for e in range(thetas.shape[0])]


def _central_hessian(grad_fn, t, h=1e-5):
    """(N, D, D) central differences of grad_fn (N, D) -> (N, D), one input at a time."""
    N, D = t.shape
    out = np.empty((N, D, D))
    for d in range(D):
        tp, tm = t.copy(), t.copy()
        tp[:, d] += h
        tm[:, d] -= h
        out[:, :, d] = (grad_fn(tp) - grad_fn(tm)) / (2 * h)
    return out


# ---- CPU: the references are the Hessians of the oracle's own costs ------------------------------------------------
@pytest.mark.parametrize("E,D", [(1, 1), (3, 4), (6, 3)])
def test_bank_reference_matches_finite_differences(E, D):
    inputs, thetas, invQts, invQs, rs = _models(E, D, 30, seed=1)
    models = _as_models(inputs, thetas, invQts, invQs)
    t = rs.random_sample((5, D))
    obs = orc.bank_predict(models, t)[0] * 1.2 + 0.1
    w = rs.random_sample(E) + 0.5
    _, _, hess, _ = bank_cost_hess_ref(models, t, obs, w)
    fd = _central_hessian(lambda x: orc.bank_cost(models, x, obs, w)[1], t)
    assert orc.ref_err(hess, fd) < 1e-6


@pytest.mark.parametrize("E,W,D", [(1, 5, 1), (4, 9, 3), (7, 20, 4)])
def test_spectra_reference_matches_finite_differences(E, W, D):
    from tests.test_forward_cost import mv_cost
    inputs, thetas, invQts, invQs, rs = _models(E, D, 30, seed=2)
    models = _as_models(inputs, thetas, invQts, invQs)
    B = rs.standard_normal((E, W))
    t = rs.random_sample((5, D))
    obs = orc.mv_predict_batch(models, B, t)[0] * 1.2 + 0.1
    lam = rs.random_sample(W) + 0.5
    c, g, hess, _ = mv_cost_hess_ref(models, B, t, obs, lam)
    c_o, g_o = mv_cost(models, B, t, obs, lam)
    assert orc.ref_err(c, c_o) < 1e-12 and orc.ref_err(g, g_o) < 1e-12
    fd = _central_hessian(lambda x: mv_cost(models, B, x, obs, lam)[1], t)
    assert orc.ref_err(hess, fd) < 1e-6


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpemu(lib):
    import gp_emulator_b200 as g
    assert lib.gpe_device_count() > 0, "no GPU visible: the gpu tests must not pass on a fallback"
    return g


def _bank(gpemu, E, D, M=40, W=0, seed=0, device=0):
    inputs, thetas, invQts, invQs, rs = _models(E, D, M, seed)
    B = rs.standard_normal((E, W)) if W else None
    bank = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=B, device=device)
    return bank, _as_models(inputs, thetas, invQts, invQs), B, rs


def _err(x, ref):
    """ref_err, with an all-zero reference (a zero weight on a one-emulator bank) matched exactly."""
    return orc.ref_err(x, ref) if np.any(ref != 0) else float(np.max(np.abs(x)))


def _check(got, ref, grad=True):
    """cost, grad against the reference; hess by ref_err and per element against its magnitude sum; exact symmetry."""
    c, g, h, mag = ref
    assert got["hess"].shape == h.shape
    assert np.array_equal(got["hess"], got["hess"].transpose(0, 2, 1))
    assert _err(got["cost"], c) < TOL and (not grad or _err(got["grad"], g) < TOL)
    assert _err(got["hess"], h) < TOL
    assert np.all(np.abs(got["hess"] - h) <= TOL * mag)


# (M, E, D, N): N > 16384 takes the per-emulator fused Hessian; E = 64, D = 24 walks several scratch chunks; D = 40 is
# the generic path
BANK_SHAPES = [(40, 1, 1, 1), (40, 5, 4, 7), (40, 20, 10, 300), (40, 33, 13, 65), (30, 64, 16, 200),
               (30, 64, 24, 2000), (25, 5, 40, 20), (64, 3, 4, 17000)]


@pytest.mark.gpu
@pytest.mark.parametrize("M,E,D,N", BANK_SHAPES)
def test_bank_cost_hessian_parity(gpemu, M, E, D, N):
    bank, models, _, rs = _bank(gpemu, E, D, M)
    t = rs.random_sample((N, D))
    mu = orc.bank_predict(models, t)[0]
    obs1 = mu.mean(axis=0) * 1.1 + 0.01
    obsN = mu * (1.0 + 0.1 * rs.standard_normal(mu.shape))
    w = rs.random_sample(E) + 0.5
    wz = w * (rs.random_sample(E) < 0.7)
    for obs, wt in ((obs1, None), (obsN, w), (obs1, wz)) if N < 10000 else ((obsN, wz),):
        # (the band cost's gradient, one lane of a warp per input in k_bank_cost, has no columns past 32: it is not
        # part of this check for D > 32)
        _check(bank.cost(t, obs, wt, want_hess=True), bank_cost_hess_ref(models, t, obs, wt), grad=D <= 32)


# (E, W, D, N); E = 96 is the forward cost's largest bank
FWD_SHAPES = [(1, 7, 1, 1), (5, 7, 4, 7), (20, 2101, 10, 100), (33, 129, 13, 65), (20, 129, 16, 300),
              (96, 300, 4, 40), (5, 64, 40, 10), (3, 7, 4, 17000)]


@pytest.mark.gpu
@pytest.mark.parametrize("E,W,D,N", FWD_SHAPES)
def test_forward_cost_hessian_parity(gpemu, E, W, D, N):
    bank, models, B, rs = _bank(gpemu, E, D, M=64 if N > 10000 else 30, W=W)
    t = rs.random_sample((N, D))
    fwd = orc.mv_predict_batch(models, B, t)[0]
    obs1 = fwd.mean(axis=0) * 1.1 + 0.01
    obsN = fwd * (1.0 + 0.1 * rs.standard_normal(fwd.shape))
    w = rs.random_sample(W) + 0.5
    wz = w * (rs.random_sample(W) < 0.7)
    for obs, wt in ((obs1, None), (obsN, w), (obs1, wz)) if N < 10000 else ((obsN, wz),):
        _check(bank.forward_cost(t, obs, wt, want_hess=True), mv_cost_hess_ref(models, B, t, obs, wt))


@pytest.mark.gpu
def test_bank_cost_hessian_pinned_to_reference_outputs(gpemu):
    """golden_K: mu, deriv and hess frozen from the reference itself."""
    g = golden("K")
    bank = gpemu.DeviceBank(g["inputs"], g["thetas"], g["invQt"], g["invQ"])
    rs = np.random.RandomState(3)
    E = g["mu"].shape[1]
    obs = g["mu"] * (1.0 + 0.2 * rs.standard_normal(g["mu"].shape))
    w = rs.random_sample(E) + 0.5
    c = w * (g["mu"] - obs)
    ref = np.einsum("ne,nedk->ndk", c, g["hess"]) + np.einsum("e,ned,nek->ndk", w, g["deriv"], g["deriv"])
    got = bank.cost(g["testing"], obs, w, want_hess=True)
    assert orc.ref_err(got["hess"], ref) < TOL
    assert np.array_equal(got["hess"], got["hess"].transpose(0, 2, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("E,D", [(5, 4), (20, 10), (64, 13)])
def test_bank_own_prediction_gives_the_gauss_newton_term(gpemu, E, D):
    bank, models, _, rs = _bank(gpemu, E, D)
    N = 200
    t = rs.random_sample((N, D))
    w = rs.random_sample(E) + 0.5
    own = bank.predict(t, want_var=False, want_deriv=True)
    got = bank.cost(t, own["mu"], w, want_hess=True)
    assert np.all(got["cost"] == 0.0) and np.all(got["grad"] == 0.0)
    gn = np.einsum("e,ned,nek->ndk", w, own["deriv"], own["deriv"])
    assert orc.ref_err(got["hess"], gn) < 1e-12
    ev = np.linalg.eigvalsh(got["hess"])
    assert np.all(ev >= -1e-12 * np.abs(ev).max(axis=1, keepdims=True))


@pytest.mark.gpu
@pytest.mark.parametrize("E,W,D", [(5, 129, 4), (20, 2101, 10), (40, 300, 6)])
def test_forward_own_prediction_gives_the_gauss_newton_term(gpemu, E, W, D):
    bank, models, B, rs = _bank(gpemu, E, D, W=W)
    N = 100
    t = rs.random_sample((N, D))
    lam = rs.random_sample(W) + 0.5
    own = bank.predict(t, want_var=False, want_deriv=False, want_mu=False, project=True, project_deriv=True)
    got = bank.forward_cost(t, own["fwd"], lam, want_hess=True)
    assert np.all(got["cost"] == 0.0) and np.all(got["grad"] == 0.0)
    J = own["deriv_full"]
    gn = np.einsum("ndw,w,nkw->ndk", J, lam, J)
    assert orc.ref_err(got["hess"], gn) < 1e-12
    ev = np.linalg.eigvalsh(got["hess"])
    assert np.all(ev >= -1e-12 * np.abs(ev).max(axis=1, keepdims=True))


def _device_ex(lib, bank, kind, t, obs, w, ld):
    """The device entry point with observation rows ld >= K wide (padded with NaN past K)."""
    import torch
    N, D = t.shape
    K = obs.shape[1]
    big = torch.full((N, ld), float("nan"), dtype=torch.float64, device="cuda")
    big[:, :K] = torch.from_numpy(obs).cuda()
    td, wd = torch.from_numpy(t).cuda(), torch.from_numpy(w).cuda()
    out = {"cost": torch.empty(N, dtype=torch.float64, device="cuda"),
           "grad": torch.empty(N, D, dtype=torch.float64, device="cuda"),
           "hess": torch.empty(N, D, D, dtype=torch.float64, device="cuda")}
    fn = lib.gpe_bank_cost_ex if kind == "bank" else lib.gpe_bank_forward_cost_ex
    assert fn(bank._h, td.data_ptr(), N, big.data_ptr(), ld, wd.data_ptr(), out["cost"].data_ptr(),
              out["grad"].data_ptr(), out["hess"].data_ptr(), None) == 0
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("kind,E,W,D,N", [("bank", 64, 0, 24, 2000), ("bank", 20, 0, 10, 30000),
                                          ("fwd", 20, 129, 10, 3000), ("fwd", 40, 2101, 6, 300)])
def test_placement_chunking_and_devices_are_invisible(lib, gpemu, monkeypatch, kind, E, W, D, N):
    import torch
    bank, models, B, rs = _bank(gpemu, E, D, M=30, W=W)
    K = E if kind == "bank" else W
    call = (lambda b, *a, **k: b.cost(*a, **k)) if kind == "bank" else (lambda b, *a, **k: b.forward_cost(*a, **k))
    t = rs.random_sample((N, D))
    obs = rs.standard_normal((N, K))
    w = rs.random_sample(K)
    ref = call(bank, t, obs, w, want_hess=True)
    plain = call(bank, t, obs, w)
    assert np.array_equal(plain["cost"], ref["cost"]) and np.array_equal(plain["grad"], ref["grad"])
    versions = []
    monkeypatch.setenv("GPE_SLOT_OUT_BYTES", str(8 * (1 + D + D * D) * 997))       # chunks of 997 points
    versions.append(call(bank, t, obs, w, want_hess=True))
    monkeypatch.delenv("GPE_SLOT_OUT_BYTES")
    dev = call(bank, torch.from_numpy(t).cuda(), torch.from_numpy(obs).cuda(), torch.from_numpy(w).cuda(), want_hess=True)
    versions.append({k: v.cpu().numpy() for k, v in dev.items()})
    versions.append(_device_ex(lib, bank, kind, t, obs, w, K + 5))
    inputs, thetas, invQts, invQs, _ = _models(E, D, 30, 0)
    two = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=B, device=[0, 0] if lib.gpe_device_count() == 1 else "all")
    versions.append(call(two, t, obs, w, want_hess=True))
    for v in versions:
        for k in ("cost", "grad", "hess"):
            assert np.array_equal(v[k], ref[k]), k
    only = call(bank, t, obs, w, want_grad=False, want_hess=True)          # no gradient requested
    assert set(only) == {"cost", "hess"} and np.array_equal(only["cost"], call(bank, t, obs, w, want_grad=False)["cost"])
    assert orc.ref_err(only["hess"], ref["hess"]) < 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bank", "fwd"])
def test_hessian_matches_finite_differences_of_the_library_gradient(gpemu, kind):
    E, W, D, N = 8, 129, 5, 20
    bank, models, B, rs = _bank(gpemu, E, D, W=W if kind == "fwd" else 0)
    t = rs.random_sample((N, D))
    K = E if kind == "bank" else W
    obs = rs.standard_normal(K)
    w = rs.random_sample(K) + 0.5
    call = bank.cost if kind == "bank" else bank.forward_cost
    hess = call(t, obs, w, want_hess=True)["hess"]
    fd = _central_hessian(lambda x: call(x, obs, w)["grad"], t)
    assert orc.ref_err(hess, fd) < 1e-6


@pytest.mark.gpu
def test_one_point_calls(gpemu):
    from tests.test_gpu_parity import _write_prosail_dump
    g = golden("P")
    mv = gpemu.MultivariateEmulator(X=None, y=None, dump=_write_prosail_dump(g))
    rs = np.random.RandomState(7)
    pts = g["points"]
    D = pts.shape[1]
    obs = mv.predict(pts[0], do_deriv=False) * 1.05
    lam = rs.random_sample(obs.shape[0]) + 0.5
    c, gr, h = mv.cost(pts, obs, lam, do_hess=True)
    assert c.shape == (len(pts),) and gr.shape == (len(pts), D) and h.shape == (len(pts), D, D)
    for k in range(len(pts)):
        c1, g1, h1 = mv.cost(pts[k], obs, lam, do_hess=True)
        assert isinstance(c1, float) and g1.shape == (D,) and h1.shape == (D, D)
        assert np.array_equal(h1, h1.T)
        assert abs(c1 - c[k]) <= TOL * abs(c).max() and np.max(np.abs(g1 - gr[k])) <= TOL * np.abs(gr).max()
        assert np.max(np.abs(h1 - h[k])) <= TOL * np.abs(h).max()
        c2, h2 = mv.cost(pts[k], obs, lam, do_deriv=False, do_hess=True)
        # (without the gradient the PC means come from the mean-only kernel: equal to the last bits)
        assert abs(c2 - c1) <= TOL * abs(c).max() and np.max(np.abs(h2 - h1)) <= TOL * np.abs(h).max()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,E,W,D,N", [("bank", 20, 0, 10, 97), ("bank", 64, 0, 24, 900), ("fwd", 40, 2101, 3, 33),
                                          ("fwd", 5, 7, 2, 1)])
def test_red_zones(lib, gpemu, kind, E, W, D, N):
    """hess between NaN guard bands, device and host pointers: the bands stay untouched, every element is written."""
    import torch
    bank, models, B, rs = _bank(gpemu, E, D, M=30, W=W)
    K = E if kind == "bank" else W
    t = rs.random_sample((N, D))
    obs = rs.standard_normal((N, K))
    ref = bank_cost_hess_ref(models, t, obs) if kind == "bank" else mv_cost_hess_ref(models, B, t, obs)
    g, n = 4096, N * D * D
    for host in (False, True):
        if host:
            hbig = np.full(n + 2 * g, np.nan)
            fn = lib.gpe_bank_cost_host_ex if kind == "bank" else lib.gpe_bank_forward_cost_host_ex
            assert fn(bank._h, t.ctypes.data, N, obs.ctypes.data, K, None, None, None, hbig.ctypes.data + 8 * g) == 0
        else:
            hd = torch.full((n + 2 * g,), float("nan"), dtype=torch.float64, device="cuda")
            td, od = torch.from_numpy(t).cuda(), torch.from_numpy(obs).cuda()
            fn = lib.gpe_bank_cost_ex if kind == "bank" else lib.gpe_bank_forward_cost_ex
            assert fn(bank._h, td.data_ptr(), N, od.data_ptr(), K, None, None, None, hd.data_ptr() + 8 * g, None) == 0
            torch.cuda.synchronize()
            hbig = hd.cpu().numpy()
        assert np.all(np.isnan(hbig[:g])) and np.all(np.isnan(hbig[g + n:])) and np.all(np.isfinite(hbig[g:g + n]))
        assert orc.ref_err(hbig[g:g + n].reshape(N, D, D), ref[2]) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bank", "fwd"])
def test_nan_observation_propagates_at_zero_weight(gpemu, kind):
    E, W, D, N = 12, 129, 4, 5
    bank, models, B, rs = _bank(gpemu, E, D, W=W if kind == "fwd" else 0)
    K = E if kind == "bank" else W
    t = rs.random_sample((N, D))
    obs = rs.standard_normal((N, K))
    obs[2, 7] = np.nan
    w = np.ones(K); w[7] = 0.0
    if kind == "bank":
        got, ref = bank.cost(t, obs, w, want_hess=True), bank_cost_hess_ref(models, t, obs, w)
    else:
        got, ref = bank.forward_cost(t, obs, w, want_hess=True), mv_cost_hess_ref(models, B, t, obs, w)
    assert np.all(np.isnan(ref[2][2])) and np.all(np.isnan(got["hess"][2]))
    keep = [0, 1, 3, 4]
    assert orc.ref_err(got["hess"][keep], ref[2][keep]) < TOL


@pytest.mark.gpu
def test_argument_errors(lib, gpemu):
    import torch
    E, W, D, N = 5, 9, 3, 4
    bank, models, B, rs = _bank(gpemu, E, D, W=W)
    nob, _, _, _ = _bank(gpemu, E, D)
    t = rs.random_sample((N, D)); obs = rs.standard_normal((N, W)); h = np.empty((N, D, D))
    a = lambda x: x.ctypes.data
    assert lib.gpe_bank_cost_host_ex(bank._h, a(t), N, a(obs), E, None, None, None, None) == -1        # nothing requested
    assert lib.gpe_bank_forward_cost_host_ex(bank._h, a(t), N, a(obs), W, None, None, None, None) == -1
    assert lib.gpe_bank_forward_cost_host_ex(nob._h, a(t), N, a(obs), W, None, None, None, a(h)) == -1   # no basis
    td, od = torch.from_numpy(t).cuda(), torch.from_numpy(obs).cuda()
    hd = torch.empty(N, D, D, dtype=torch.float64, device="cuda")
    assert lib.gpe_bank_cost_ex(bank._h, td.data_ptr(), N, od.data_ptr(), W, None, None, None, None, None) == -1
    assert lib.gpe_bank_forward_cost_ex(nob._h, td.data_ptr(), N, od.data_ptr(), W, None, None, None, hd.data_ptr(),
                                        None) == -1
    assert lib.gpe_multi_bank_cost_ex(None, a(t), N, a(obs), E, None, None, None, a(h)) == -1           # NULL handle
    assert lib.gpe_multi_bank_forward_cost_ex(None, a(t), N, a(obs), W, None, None, None, a(h)) == -1
    with pytest.raises(gpemu.GpemuError):
        nob.forward_cost(t, obs, want_hess=True)
    big, _, _, _ = _bank(gpemu, 97, 2, M=6, W=8)                                    # beyond the forward cost's limit
    with pytest.raises(gpemu.GpemuError):
        big.forward_cost(rs.random_sample((3, 2)), np.zeros(8), want_hess=True)
