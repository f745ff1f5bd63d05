"""Per-point observation weights (DESIGN 4.6f): gpe_bank_cost_pw, gpe_bank_solve_pw, gpe_bank_search_pw and their
multi-device counterparts, DeviceBank.cost / forward_cost / search / forward_search / invert / forward_invert and the
MultivariateEmulator calls with (N, K) weights.

The references restate the formulas with w_e -> w_ne and l_w -> l_nw in numpy; on the CPU they are checked against
central differences, and the expanded search forms against a per-wavelength brute force.  On the GPU the library is
checked for the equivalence contract (rows all equal to w give the shared-w call bit for bit), against the references, for
exact masking by zero weights, for invariance, and for recovery of the inputs behind per-pixel noisy observations."""
import ctypes as C
import re

import numpy as np
import pytest

from oracle import gp_oracle as orc
from tests.conftest import ROOT
from tests.test_cost_hessian import TOL, _as_models, _central_hessian, _err
from tests.test_cost_hessian import _bank as _ref_bank
from tests.test_cost_hessian import _models as _ref_models
from tests.test_invert import CONVERGED, _bank, _own_obs, _problem, _prosail, _solve, lm_ref
from tests.test_search import U, brute_costs, check_against_brute

NEW = ("gpe_bank_cost_pw", "gpe_bank_solve_pw", "gpe_bank_search_pw", "gpe_multi_bank_cost_pw", "gpe_multi_bank_solve_pw",
       "gpe_multi_bank_search_pw")


def band_pw_ref(models, t, obs, w):
    """cost, grad, hess of 1/2 sum_e w_ne (mu_ne - obs_ne)^2 and the magnitude sum of hess."""
    mu, _, G, H = orc.bank_predict(models, t, do_hess=True)
    r = mu - obs
    c = w * r
    hess = np.einsum("ne,nedk->ndk", c, H) + np.einsum("ne,ned,nek->ndk", w, G, G)
    mag = np.einsum("ne,nedk->ndk", np.abs(c), np.abs(H)) + np.einsum("ne,ned,nek->ndk", np.abs(w), np.abs(G), np.abs(G))
    return 0.5 * np.sum(c * r, axis=1), np.einsum("ne,ned->nd", c, G), hess, mag


def fwd_pw_ref(models, B, t, obs, lam):
    """cost, grad, hess of 1/2 sum_w l_nw (fwd_nw - obs_nw)^2 with the Jacobian materialised, and the magnitude sum."""
    mu, _, G, H = orc.bank_predict(models, t, do_hess=True)
    r = mu @ B - obs
    J = np.einsum("ned,ew->ndw", G, B)
    lr = lam * r
    hess = np.einsum("ndw,nw,nkw->ndk", J, lam, J) + np.einsum("nedk,ew,nw->ndk", H, B, lr)
    mag = np.einsum("ndw,nw,nkw->ndk", np.abs(J), np.abs(lam), np.abs(J)) + \
        np.einsum("nedk,ew,nw->ndk", np.abs(H), np.abs(B), np.abs(lr))
    return 0.5 * np.sum(lr * r, axis=1), np.einsum("ndw,nw->nd", J, lr), hess, mag


def search_forms(m, obs, w, basis=None):
    """The expanded per-point-weight forms of include/gpemu.h: table rows (K, Ew), pixel operands (N, Ew), the constant
    c_n, and the score's rounding bound (N, K)."""
    if basis is None:
        tbl = np.concatenate([0.5 * (m * m), m], axis=1)
        op = np.concatenate([w, -(w * obs)], axis=1)
    else:
        E = m.shape[1]
        iu = np.triu_indices(E)
        Cn = np.einsum("ew,nw,fw->nef", basis, w, basis)
        Cn[:, np.arange(E), np.arange(E)] *= 0.5
        s = -((w * obs) @ basis.T)
        tbl = np.concatenate([m[:, iu[0]] * m[:, iu[1]], m], axis=1)
        op = np.concatenate([Cn[:, iu[0], iu[1]], s], axis=1)
    c = 0.5 * np.sum(w * obs * obs, axis=1)
    bound = op.shape[1] * U * (np.abs(op) @ np.abs(tbl).T)
    return tbl, op, c, bound


def _masked(rs, w, frac=0.1):
    return w * (rs.random_sample(w.shape) >= frac)


# ---- CPU -----------------------------------------------------------------------------------------------------------
def test_header_and_bindings_agree(lib):
    from gp_emulator_b200 import _lib
    hdr = open(f"{ROOT}/include/gpemu.h").read()
    for name in NEW:
        m = re.search(r"int\s+%s\s*\(([^;]*)\)\s*;" % name, hdr)
        assert m, name
        args = [a.strip() for a in m.group(1).split(",")]
        assert len(args) == len(getattr(lib, name).argtypes), name
        assert any(a.endswith("weights_ld") and a.startswith("int64_t") for a in args), name
        assert name in _lib.SYMBOLS
    for key, val in (("GPE_SEARCH_PW_MAX_E_BANDS", _lib.SEARCH_PW_MAX_E_BANDS),
                     ("GPE_SEARCH_PW_MAX_E_SPECTRA", _lib.SEARCH_PW_MAX_E_SPECTRA)):
        assert int(re.search(r"#define %s (\d+)" % key, hdr).group(1)) == val
    # the widths the existing k_search_topk instances reach (96 columns) are what the limits come from
    assert 2 * _lib.SEARCH_PW_MAX_E_BANDS <= 96 < 2 * (_lib.SEARCH_PW_MAX_E_BANDS + 1)
    e = _lib.SEARCH_PW_MAX_E_SPECTRA
    assert e * (e + 1) // 2 + e <= 96 < (e + 1) * (e + 2) // 2 + e + 1


@pytest.mark.parametrize("E,D", [(1, 1), (4, 3), (7, 2)])
def test_band_reference_matches_finite_differences(E, D):
    inputs, thetas, invQts, invQs, rs = _ref_models(E, D, 30, seed=3)
    models = _as_models(inputs, thetas, invQts, invQs)
    t = rs.random_sample((5, D))
    obs = orc.bank_predict(models, t)[0] * 1.2 + 0.1
    w = _masked(rs, rs.random_sample((5, E)) + 0.5, 0.3)
    c, g, h, _ = band_pw_ref(models, t, obs, w)
    cost = lambda x: band_pw_ref(models, x, obs, w)[0]
    fd_g = np.stack([(cost(t + 1e-6 * np.eye(D)[d]) - cost(t - 1e-6 * np.eye(D)[d])) / 2e-6 for d in range(D)], axis=1)
    assert orc.ref_err(g, fd_g) < 1e-6
    assert orc.ref_err(h, _central_hessian(lambda x: band_pw_ref(models, x, obs, w)[1], t)) < 1e-6
    # rows all equal to w: the shared-weight reference of the Hessian tests
    from tests.test_cost_hessian import bank_cost_hess_ref
    ws = np.tile(w[0], (5, 1))
    for a, b in zip(band_pw_ref(models, t, obs, ws)[:3], bank_cost_hess_ref(models, t, obs, w[0])[:3]):
        assert orc.ref_err(a, b) < 1e-13


@pytest.mark.parametrize("E,W,D", [(1, 5, 1), (4, 9, 3), (6, 20, 2)])
def test_spectra_reference_matches_finite_differences(E, W, D):
    inputs, thetas, invQts, invQs, rs = _ref_models(E, D, 30, seed=4)
    models = _as_models(inputs, thetas, invQts, invQs)
    B = rs.standard_normal((E, W))
    t = rs.random_sample((5, D))
    obs = orc.mv_predict_batch(models, B, t)[0] * 1.2 + 0.1
    lam = _masked(rs, rs.random_sample((5, W)) + 0.5, 0.3)
    c, g, h, _ = fwd_pw_ref(models, B, t, obs, lam)
    cost = lambda x: fwd_pw_ref(models, B, x, obs, lam)[0]
    fd_g = np.stack([(cost(t + 1e-6 * np.eye(D)[d]) - cost(t - 1e-6 * np.eye(D)[d])) / 2e-6 for d in range(D)], axis=1)
    assert orc.ref_err(g, fd_g) < 1e-6
    assert orc.ref_err(h, _central_hessian(lambda x: fwd_pw_ref(models, B, x, obs, lam)[1], t)) < 1e-6
    # the C_n route of the library: hess = sum_e s_ne H_ne + G^T C_n G
    mu, _, G, H = orc.bank_predict(models, t, do_hess=True)
    s = (lam * (mu @ B - obs)) @ B.T
    Cn = np.einsum("ew,nw,fw->nef", B, lam, B)
    h2 = np.einsum("ne,nedk->ndk", s, H) + np.einsum("ned,nef,nfk->ndk", G, Cn, G)
    assert orc.ref_err(h2, h) < 1e-12


@pytest.mark.parametrize("spectra", [False, True])
def test_expanded_search_scores_agree_with_a_per_wavelength_brute_force(spectra):
    rs = np.random.RandomState(7)
    E, W, K, N = (5, 33, 300, 20) if spectra else (9, 9, 300, 20)
    m = rs.standard_normal((K, E))
    B = rs.standard_normal((E, W)) if spectra else None
    fwd = m if B is None else m @ B
    obs = fwd[rs.randint(0, K, N)] + 0.3 * rs.standard_normal((N, W))
    w = _masked(rs, rs.uniform(0.5, 2.0, (N, W)))
    tbl, op, c, bound = search_forms(m, obs, w, B)
    assert tbl.shape[1] == (E * (E + 1) // 2 + E if spectra else 2 * E)
    score = op @ tbl.T
    brute = np.stack([brute_costs(m, obs[n:n + 1], w[n], B)[0] for n in range(N)])
    assert np.all(np.abs(score + c[:, None] - brute) <= bound + 4 * U * np.abs(brute))
    # the ranking the library's forms give is the brute force's up to the rounding bound
    k = 5
    sel = np.argsort(score, axis=1, kind="stable")[:, :k]
    idx = np.stack([sel[n][np.lexsort((sel[n], brute[n, sel[n]]))] for n in range(N)])
    check_against_brute(idx, np.take_along_axis(brute, idx, axis=1), brute, bound)


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpemu(lib):
    import gp_emulator_b200 as g
    assert lib.gpe_device_count() > 0, "no GPU visible: the gpu tests must not pass on a fallback"
    return g


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(d):
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in d.items()}


def _same(a, b, keys, what=""):
    for k in keys:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k]), equal_nan=True), (what, k)


def _cost(bank, spectra, *a, **k):
    return (bank.forward_cost if spectra else bank.cost)(*a, **k)


def _search(bank, spectra, *a, **k):
    return (bank.forward_search if spectra else bank.search)(*a, **k)


def _two_devices(lib, gpemu, kind):
    """The problem's bank on two devices (the same device twice on a one-GPU machine)."""
    devs = [0, 0] if lib.gpe_device_count() == 1 else "all"
    if kind == "prosail":
        from tests.test_gpu_parity import _write_prosail_dump
        from tests.conftest import golden
        mv = gpemu.MultivariateEmulator(X=None, y=None, dump=_write_prosail_dump(golden("P")), device=devs)
        return mv._device_bank()
    from tests.test_invert import _models
    E, D, W = (20, 10, 2101) if kind == "fwd" else (24, 6, 0)
    inputs, thetas, invQts, invQs, rs = _models(E, D, 40, 0)
    B = rs.standard_normal((E, W)) if W else None
    return gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=B, device=devs)


def _data(bank, spectra, lo, hi, rs, N, noise=0.01):
    width = hi - lo
    x_true = lo + width * rs.uniform(0.1, 0.9, (N, len(lo)))
    obs = _own_obs(bank, spectra, x_true)
    obs = obs * (1.0 + noise * rs.standard_normal(obs.shape))
    x0 = np.clip(x_true + 0.05 * width * rs.standard_normal(x_true.shape), lo, hi)
    return x_true, obs, x0


SOLVE_KEYS = ("x", "cost", "grad", "hess", "cov", "status", "n_iter")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "fwd", "prosail"])
def test_rows_equal_to_the_shared_weights_reproduce_the_shared_call(lib, gpemu, kind):
    bank, spectra, lo, hi, rs = _problem(gpemu, kind)
    N = 300
    x_true, obs, x0 = _data(bank, spectra, lo, hi, rs, N)
    w = rs.uniform(0.5, 2.0, obs.shape[1])
    wN = np.tile(w, (N, 1))
    keys = ("cost", "grad", "hess")
    ref = _cost(bank, spectra, x0, obs, w, want_hess=True)
    _same(_cost(bank, spectra, x0, obs, wN, want_hess=True), ref, keys, "host")
    _same(_np(_cost(bank, spectra, _t(x0), _t(obs), _t(wN), want_hess=True)), ref, keys, "device")
    _same(_cost(_two_devices(lib, gpemu, kind), spectra, x0, obs, wN, want_hess=True), ref, keys, "devices")
    ref1 = _cost(bank, spectra, x0, obs[0], w, want_hess=True)                 # one shared observation
    _same(_cost(bank, spectra, x0, obs[0], wN, want_hess=True), ref1, keys, "shared obs")
    kw = dict(lower=lo, upper=hi, want_cov=True, max_iter=100)
    sref = _solve(bank, spectra, x0, obs, w, **kw)
    _same(_solve(bank, spectra, x0, obs, wN, **kw), sref, SOLVE_KEYS, "solve host")
    dev = _solve(bank, spectra, _t(x0), _t(obs), _t(wN), lower=_t(lo), upper=_t(hi), want_cov=True, max_iter=100)
    _same(_np(dev), sref, SOLVE_KEYS, "solve device")
    if not spectra or bank.E <= 12:
        K = 500
        cand = lo + (hi - lo) * rs.uniform(0, 1, (K, len(lo)))
        f = _search(bank, spectra, cand, obs, w, k=4)
        g = _search(bank, spectra, cand, obs, wN, k=4)
        # the two forms rank by different expanded sums: the exact costs of the chosen candidates agree bit for bit
        # wherever the same candidates are chosen
        same = np.all(f["idx"] == g["idx"], axis=1)
        assert np.mean(same) > 0.9
        assert np.array_equal(f["cost"][same], g["cost"][same])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "fwd"])
def test_per_point_costs_match_the_numpy_reference(gpemu, kind):
    spectra = kind == "fwd"
    E, D, W, N = (20, 10, 2101, 100) if spectra else (24, 6, 0, 300)
    bank, models, B, rs = _ref_bank(gpemu, E, D, 30, W=W)
    t = rs.random_sample((N, D))
    ref_out = orc.mv_predict_batch(models, B, t)[0] if spectra else orc.bank_predict(models, t)[0]
    obs = ref_out * (1.0 + 0.1 * rs.standard_normal(ref_out.shape))
    w = _masked(rs, rs.uniform(0.5, 2.0, obs.shape))
    got = _cost(bank, spectra, t, obs, w, want_hess=True)
    ref = fwd_pw_ref(models, B, t, obs, w) if spectra else band_pw_ref(models, t, obs, w)
    c, g, h, mag = ref
    assert np.array_equal(got["hess"], got["hess"].transpose(0, 2, 1))
    assert _err(got["cost"], c) < TOL and _err(got["grad"], g) < TOL and _err(got["hess"], h) < TOL
    assert np.all(np.abs(got["hess"] - h) <= TOL * mag)
    got_d = _np(_cost(bank, spectra, _t(t), _t(obs), _t(w), want_hess=True))
    _same(got_d, got, ("cost", "grad", "hess"), "device")


@pytest.mark.gpu
def test_per_point_prosail_costs_match_one_shared_call_per_point(gpemu):
    mv, g = _prosail(gpemu)
    bank = mv._device_bank()
    rs = np.random.RandomState(2)
    lo, hi = g["y"].min(axis=0), g["y"].max(axis=0)
    N = 12
    _, obs, x0 = _data(bank, True, lo, hi, rs, N, noise=0.05)
    w = _masked(rs, rs.uniform(0.5, 2.0, obs.shape))
    got = mv.cost(x0, obs, w, do_hess=True)
    for n in range(N):
        c, gr, h = mv.cost(x0[n], obs[n], w[n], do_hess=True)
        assert abs(got[0][n] - c) <= TOL * abs(c)
        assert orc.ref_err(got[1][n], gr) < TOL and orc.ref_err(got[2][n], h) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "fwd", "prosail"])
def test_masked_observations_do_not_reach_any_output(gpemu, kind):
    bank, spectra, lo, hi, rs = _problem(gpemu, kind)
    N = 200
    _, obs, x0 = _data(bank, spectra, lo, hi, rs, N)
    w = _masked(rs, rs.uniform(0.5, 2.0, obs.shape))
    assert np.any(w == 0)
    other = np.where(w == 0, obs + 1e3 * rs.standard_normal(obs.shape), obs)
    keys = ("cost", "grad", "hess")
    _same(_cost(bank, spectra, x0, other, w, want_hess=True), _cost(bank, spectra, x0, obs, w, want_hess=True), keys)
    kw = dict(lower=lo, upper=hi, want_cov=True)
    _same(_solve(bank, spectra, x0, other, w, **kw), _solve(bank, spectra, x0, obs, w, **kw), SOLVE_KEYS, "solve")
    if not spectra or bank.E <= 12:
        cand = lo + (hi - lo) * rs.uniform(0, 1, (400, len(lo)))
        _same(_search(bank, spectra, cand, other, w, k=5), _search(bank, spectra, cand, obs, w, k=5), ("idx", "cost"))


@pytest.mark.gpu
@pytest.mark.parametrize("spectra", [True, False])
def test_results_do_not_depend_on_chunking_placement_devices_or_order(lib, gpemu, monkeypatch, spectra):
    E, W, D, N = 12, 257, 6, 3000
    bank, rs = _bank(gpemu, E, D, W=W if spectra else 0)
    x_true = rs.uniform(0.1, 0.9, (N, D))
    obs = _own_obs(bank, spectra, x_true)
    obs = obs + 0.01 * rs.standard_normal(obs.shape)
    x0 = np.clip(x_true + 0.1 * rs.standard_normal((N, D)), 0, 1)
    w = _masked(rs, rs.uniform(0.5, 2.0, obs.shape))
    kw = dict(lower=np.zeros(D), upper=np.ones(D), want_cov=True)
    cand = rs.uniform(0, 1, (700, D))
    ref = {"cost": _cost(bank, spectra, x0, obs, w, want_hess=True), "solve": _solve(bank, spectra, x0, obs, w, **kw),
           "search": _search(bank, spectra, cand, obs, w, k=5)}
    assert len(np.unique(ref["solve"]["n_iter"])) > 1
    keys = {"cost": ("cost", "grad", "hess"), "solve": SOLVE_KEYS, "search": ("idx", "cost")}

    def run(b, x, o, ww, c=cand):
        return {"cost": _cost(b, spectra, x, o, ww, want_hess=True), "solve": _solve(b, spectra, x, o, ww, **kw),
                "search": _search(b, spectra, c, o, ww, k=5)}
    versions = {}
    monkeypatch.setenv("GPE_SLOT_OUT_BYTES", str(8 * (3 + 2 * D + 2 * D * D) * 97))     # streamed chunks of 97 points
    versions["chunks"] = run(bank, x0, obs, w)
    monkeypatch.delenv("GPE_SLOT_OUT_BYTES")
    monkeypatch.setenv("GPE_SOLVE_SUB_POINTS", "97")                                   # solver sub-chunks
    versions["sub"] = {"solve": _solve(bank, spectra, x0, obs, w, **kw)}
    monkeypatch.delenv("GPE_SOLVE_SUB_POINTS")
    dev = run(bank, _t(x0), _t(obs), _t(w), _t(cand))
    versions["device"] = {k: _np(v) for k, v in dev.items()}
    from tests.test_invert import _models
    inputs, thetas, invQts, invQs, rs2 = _models(E, D, 40, 0)
    B = rs2.standard_normal((E, W)) if spectra else None
    two = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=B, device=[0, 0] if lib.gpe_device_count() == 1 else "all")
    versions["devices"] = run(two, x0, obs, w)
    perm = rs.permutation(N)
    got = run(bank, x0[perm], obs[perm], w[perm])
    inv = np.argsort(perm)
    versions["permuted"] = {k: {kk: vv[inv] for kk, vv in v.items()} for k, v in got.items()}
    for name, v in versions.items():
        for call, out in v.items():
            _same(out, ref[call], keys[call], (name, call))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "fwd", "prosail"])
def test_per_pixel_sigma_with_masked_bands_recovers_the_inputs(gpemu, kind):
    """Pixels from the model's own output plus noise at per-pixel sigma, with some bands masked: the solve lands within a
    few of its own Laplace standard deviations of x_true, and those follow each pixel's sigma."""
    bank, spectra, lo, hi, rs = _problem(gpemu, kind)
    N = 200
    width = hi - lo
    x_true = lo + width * rs.uniform(0.2, 0.8, (N, len(lo)))
    clean = _own_obs(bank, spectra, x_true)
    sigma = np.abs(clean).mean() * 1e-4 * rs.uniform(0.5, 5.0, (N, 1)) * rs.uniform(0.5, 1.5, clean.shape)
    w = 1.0 / sigma ** 2
    mask = rs.random_sample(clean.shape) < 0.1
    w[mask] = 0.0
    obs = clean + sigma * rs.standard_normal(clean.shape)
    obs[mask] = 1e6                                  # masked entries: any finite value
    x0 = np.clip(x_true + 0.02 * width * rs.standard_normal(x_true.shape), lo, hi)
    res = _solve(bank, spectra, x0, obs, w, lower=lo, upper=hi, max_iter=100, want_cov=True)
    assert np.all(res["status"] == CONVERGED), np.bincount(res["status"])
    sd = np.sqrt(np.einsum("ndd->nd", res["cov"]))
    assert np.all(np.isfinite(sd))
    assert np.all(np.abs(res["x"] - x_true) <= 6 * sd), np.max(np.abs(res["x"] - x_true) / sd)
    # the standard deviations scale with each pixel's own sigma
    assert np.corrcoef(np.log(sd[:, 0]), np.log(sigma.mean(axis=1)))[0, 1] > 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fwd", "prosail", "band"])
def test_agreement_with_the_reference_driving_the_per_point_costs(gpemu, kind):
    bank, spectra, lo, hi, rs = _problem(gpemu, kind)
    N = 60
    width = hi - lo
    _, obs, x0 = _data(bank, spectra, lo, hi, rs, N)
    w = _masked(rs, rs.uniform(0.5, 2.0, obs.shape))

    def fgh(X, idx):
        rows = x0.copy()
        rows[idx] = X
        out = _cost(bank, spectra, rows, obs, w, want_hess=True)
        return out["cost"][idx], out["grad"][idx], out["hess"][idx]

    ref = lm_ref(fgh, x0, lo, hi, max_iter=100, indexed=True)
    got = _solve(bank, spectra, x0, obs, w, lower=lo, upper=hi, max_iter=100)
    ref_x, ref_c, ref_s = ref["x"], ref["cost"], ref["status"]
    assert np.array_equal(got["status"], ref_s)
    ok = ref_s == CONVERGED
    assert np.max(np.abs(got["cost"][ok] - ref_c[ok]) / np.maximum(np.abs(ref_c[ok]), 1e-300)) < 1e-8
    dx = got["x"] - ref_x
    close = np.max(np.abs(dx) / width, axis=1) < 1e-8
    if kind != "prosail":
        assert np.all(close[ok])
    else:   # flat valleys of the PROSAIL model: as test_invert.test_agreement_with_the_reference_driving_the_library_costs
        flat = 0.5 * np.einsum("nd,nde,ne->n", dx, ref["hess"], dx) <= 1e-8 * np.abs(ref_c)
        assert np.all((close | flat)[ok])
        assert np.sum(~close[ok]) <= len(close) // 4


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "prosail"])
@pytest.mark.parametrize("k", [1, 5, 16])
def test_search_matches_an_exact_brute_force(gpemu, kind, k):
    bank, spectra, lo, hi, rs = _problem(gpemu, kind)
    N, K = 150, 2000
    cand = lo + (hi - lo) * rs.uniform(0, 1, (K, len(lo)))
    _, obs, _ = _data(bank, spectra, lo, hi, rs, N, noise=0.02)
    w = _masked(rs, rs.uniform(0.5, 2.0, obs.shape))
    got = _search(bank, spectra, cand, obs, w, k=k)
    # brute force: the library's cost of every candidate against every row, with that row's weights
    brute = np.stack([_cost(bank, spectra, cand, obs[n], w[n], want_grad=False)["cost"] for n in range(N)])
    c_n = 0.5 * np.sum(w * obs * obs, axis=1)
    check_against_brute(got["idx"], got["cost"], brute, 1e-10 * (np.abs(brute) + c_n[:, None]))
    assert np.all(got["idx"] >= 0)
    # the returned costs are bit for bit those of the per-point cost call
    for j in range(k):
        c = _cost(bank, spectra, cand[got["idx"][:, j]], obs, w, want_grad=False)["cost"]
        assert np.array_equal(c, got["cost"][:, j])


@pytest.mark.gpu
def test_searches_beyond_the_operand_width_are_unsupported(lib, gpemu, monkeypatch):
    from gp_emulator_b200 import _lib
    big, rs = _bank(gpemu, 49, 3)
    N, K, E = 4, 10, 49
    obs, w = rs.standard_normal((N, E)), rs.uniform(0.5, 2, (N, E))
    cand = rs.uniform(0, 1, (K, 3))
    idx, cost = np.empty((N, 2), dtype=np.int64), np.empty((N, 2))
    a = lambda v: v.ctypes.data
    rc = lib.gpe_bank_search_pw(big._h, a(cand), K, a(obs), N, E, a(w), E, 2, a(idx), a(cost), _lib.HOST_PTRS, None)
    assert rc == -4 and b"48" in lib.gpe_last_error()
    assert big.search(cand, obs, w[0], k=2)["idx"].shape == (N, 2)          # shared weights: served
    ok48, _ = _bank(gpemu, 48, 3)
    assert ok48.search(cand, obs[:, :48], w[:, :48], k=2)["idx"].shape == (N, 2)
    fwd, spectra, lo, hi, rs = _problem(gpemu, "fwd")
    obsW = _own_obs(fwd, True, rs.uniform(0, 1, (N, 10)))
    with pytest.raises(gpemu.GpemuError, match="12"):
        fwd.forward_search(rs.uniform(0, 1, (K, 10)), obsW, np.ones_like(obsW), k=2)
    mv, g = _prosail(gpemu)
    y = g["y"][:3]
    spec = mv.predict(y, do_deriv=False)
    wN = np.ones_like(spec)
    assert mv.invert(spec, weights=wN, bounds=(g["y"].min(axis=0), g["y"].max(axis=0)))["x"].shape == y.shape
    monkeypatch.setattr(mv, "n_pcs", 13)             # the check reads the emulator's PC count before any upload
    with pytest.raises(ValueError, match="12.*y0"):
        mv.invert(spec, weights=wN)


@pytest.mark.gpu
def test_argument_errors(lib, gpemu):
    from gp_emulator_b200 import _lib
    E, W, D, N = 5, 9, 3, 4
    bank, rs = _bank(gpemu, E, D, W=W)
    x = rs.random_sample((N, D))
    obs, w = rs.standard_normal((N, W)), rs.uniform(0.5, 2, (N, W))
    obsE, wE = rs.standard_normal((N, E)), rs.uniform(0.5, 2, (N, E))
    cost = np.empty(N)
    a = lambda v: None if v is None else v.ctypes.data
    H, S = _lib.HOST_PTRS, _lib.SOLVE_SPECTRA

    def cost_call(o=obs, wt=w, ld=W, flags=H | S):
        return lib.gpe_bank_cost_pw(bank._h, a(x), N, a(o), o.shape[1], a(wt), ld, a(cost), None, None, flags, None)
    assert cost_call() == 0 and cost_call(o=obsE, wt=wE, ld=E, flags=H) == 0 and cost_call(ld=0) == 0
    assert cost_call(ld=W + 1) == -1 and cost_call(ld=W - 1) == -1 and cost_call(o=obsE, wt=wE, ld=E + 1, flags=H) == -1
    assert cost_call(wt=None, ld=W) == -1 and cost_call(ld=-1) == -1
    assert cost_call(flags=H | S | 0x4000) == -1
    assert lib.gpe_multi_bank_cost_pw(None, a(x), N, a(obs), W, a(w), W, a(cost), None, None, S) == -1
    xo, info = np.empty((N, D)), np.empty((N, 2), dtype=np.int32)
    solve = lambda ld, flags=H | S: lib.gpe_bank_solve_pw(bank._h, a(x), N, a(obs), W, a(w), ld, None, a(xo), None, None,
                                                          None, None, a(info), flags, None)
    assert solve(W) == 0 and solve(W + 1) == -1 and solve(W - 1) == -1 and solve(W, H | S | 0x4000) == -1
    idx = np.empty((N, 2), dtype=np.int64)
    cand = rs.random_sample((7, D))
    srch = lambda ld, o=obsE, wt=wE, flags=H: lib.gpe_bank_search_pw(bank._h, a(cand), 7, a(o), N, o.shape[1], a(wt), ld, 2,
                                                                      a(idx), None, flags, None)
    assert srch(E) == 0 and srch(E + 1) == -1 and srch(E - 1) == -1 and srch(E, flags=H | 0x4000) == -1
    # device pointers: rows may be further apart than K, but not closer
    import torch
    xd, od = _t(x), _t(np.concatenate([obsE, np.zeros((N, 3))], axis=1))
    wd = _t(np.concatenate([wE, np.zeros((N, 3))], axis=1))
    cd = torch.empty(N, dtype=torch.float64, device="cuda")
    dcall = lambda ld: lib.gpe_bank_cost_pw(bank._h, xd.data_ptr(), N, od.data_ptr(), E + 3, wd.data_ptr(), ld, cd.data_ptr(),
                                            None, None, 0, None)
    assert dcall(E + 3) == 0 and dcall(E - 1) == -1
    torch.cuda.synchronize()
    ref = bank.cost(x, obsE, wE, want_grad=False)["cost"]
    assert np.array_equal(cd.cpu().numpy(), ref)
    with pytest.raises(ValueError):
        bank.cost(x, obsE, wE[:, :-1])
    with pytest.raises(ValueError):
        bank.invert(x, obsE, wE[:-1])


@pytest.mark.gpu
@pytest.mark.parametrize("spectra", [True, False])
def test_red_zones(lib, gpemu, spectra):
    """cost, grad, hess of the cost call, x / hess / cov / info of the solve and idx / cost of the search between guard
    bands, device and host pointers: bands untouched, every element written."""
    import torch
    from gp_emulator_b200 import _lib
    E, W, D, N = 10, 129, 4, 37
    bank, rs = _bank(gpemu, E, D, W=W if spectra else 0)
    x_true = rs.uniform(0.2, 0.8, (N, D))
    obs = _own_obs(bank, spectra, x_true) * (1 + 0.01 * rs.standard_normal((N, W if spectra else E)))
    Kw = obs.shape[1]
    w = _masked(rs, rs.uniform(0.5, 2.0, obs.shape))
    x0 = np.clip(x_true + 0.05 * rs.standard_normal((N, D)), 0, 1)
    cand = rs.uniform(0, 1, (50, D))
    cref = _cost(bank, spectra, x0, obs, w, want_hess=True)
    sref = _solve(bank, spectra, x0, obs, w, want_cov=True)
    flags = _lib.SOLVE_SPECTRA if spectra else 0
    gb, k = 512, 3
    for host in (False, True):
        if host:
            mk = lambda n, dt=np.float64, fill=np.nan: np.full(n + 2 * gb, fill, dtype=dt)
            p = lambda b: b.ctypes.data + b.itemsize * gb
            arg = lambda v: np.ascontiguousarray(v).ctypes.data
            keep = []
            fl, st = flags | _lib.HOST_PTRS, None
            back = lambda b: b
        else:
            mk = lambda n, dt=np.float64, fill=np.nan: torch.full((n + 2 * gb,), fill, device="cuda",
                                                                 dtype=torch.int32 if dt == np.int32 else
                                                                 torch.int64 if dt == np.int64 else torch.float64)
            p = lambda b: b.data_ptr() + b.element_size() * gb
            keep = [_t(x0), _t(obs), _t(w), _t(cand)]
            arg = {id(v): t for v, t in zip((x0, obs, w, cand), keep)}
            arg = (lambda d: (lambda v: d[id(v)].data_ptr()))(arg)
            fl, st = flags, None
            back = lambda b: b.cpu().numpy()
        bufs = {"cost": mk(N), "grad": mk(N * D), "hess": mk(N * D * D)}
        rc = lib.gpe_bank_cost_pw(bank._h, arg(x0), N, arg(obs), Kw, arg(w), Kw, p(bufs["cost"]), p(bufs["grad"]),
                                  p(bufs["hess"]), fl, st)
        assert rc == 0
        sb = {"x": mk(N * D), "hess": mk(N * D * D), "cov": mk(N * D * D)}
        info = mk(2 * N, np.int32, -7)
        opts = _lib.SolveOpts(50, 1e-10, 1e-10, 0.0, 1e-3, None, None, None, 0, None)
        rc = lib.gpe_bank_solve_pw(bank._h, arg(x0), N, arg(obs), Kw, arg(w), Kw, C.byref(opts), p(sb["x"]), None, None,
                                   p(sb["hess"]), p(sb["cov"]), p(info), fl, st)
        assert rc == 0
        rb = {"idx": mk(N * k, np.int64, -7), "cost": mk(N * k)}
        rc = lib.gpe_bank_search_pw(bank._h, arg(cand), 50, arg(obs), N, Kw, arg(w), Kw, k, p(rb["idx"]), p(rb["cost"]), fl, st)
        assert rc == 0
        if not host:
            torch.cuda.synchronize()
        for bset, ref, names in ((bufs, cref, ("cost", "grad", "hess")), (sb, sref, ("x", "hess", "cov"))):
            for name in names:
                b, n = back(bset[name]), np.asarray(ref[name]).size
                assert np.all(np.isnan(b[:gb])) and np.all(np.isnan(b[gb + n:])), name
                assert np.array_equal(b[gb:gb + n], np.asarray(ref[name]).ravel(), equal_nan=True), name
        inf = back(info)
        assert np.all(inf[:gb] == -7) and np.all(inf[gb + 2 * N:] == -7)
        assert np.array_equal(inf[gb:gb + 2 * N].reshape(N, 2), np.stack([sref["status"], sref["n_iter"]], axis=1))
        ref = _search(bank, spectra, cand, obs, w, k=k)
        ri, rcst = back(rb["idx"]), back(rb["cost"])
        assert np.all(ri[:gb] == -7) and np.all(ri[gb + N * k:] == -7)
        assert np.all(np.isnan(rcst[:gb])) and np.all(np.isnan(rcst[gb + N * k:]))
        assert np.array_equal(ri[gb:gb + N * k], ref["idx"].ravel())
        assert np.array_equal(rcst[gb:gb + N * k], ref["cost"].ravel(), equal_nan=True)
