"""Candidate search on the device: gpe_bank_search / gpe_multi_bank_search, DeviceBank.search / forward_search,
MultivariateEmulator.search and the candidate-started invert (DESIGN 4.6e).

``search_ref`` restates the selection rule of include/gpemu.h in numpy: rank by the expanded form a_k + s_n . m_k under the
(score, index) order, NaN scores never selected, -1 / NaN for missing slots, then sort by (exact cost, index).  On the CPU
it is checked against a per-wavelength brute force; on the GPU the library is checked against the library's own costs of
every candidate."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from tests.conftest import ROOT
from tests.test_invert import CONVERGED, NONFINITE, _models, _own_obs, _problem, _prosail

U = 2.0 ** -53


def search_ref(m, obs, k, weights=None, basis=None):
    """Top-k of every row of obs (N, K_obs) against the candidate means m (K, E): band cost without basis, spectrum cost
    (m . basis against obs) with it.  Returns idx (N, k) in (exact cost, index) order, cost (N, k), the scores (N, K)
    and their rounding bound (N, K)."""
    m = np.asarray(m, dtype=np.float64)
    K, E = m.shape
    w = np.ones(obs.shape[1]) if weights is None else np.asarray(weights, dtype=np.float64)
    if basis is None:
        with np.errstate(over="ignore"):
            a = 0.5 * np.sum(w * m * m, axis=1)
        s = -(w * obs)
        fwd = m
    else:
        Cm = (basis * w) @ basis.T
        a = 0.5 * np.einsum("ke,ef,kf->k", m, Cm, m)
        s = -((w * obs) @ basis.T)
        fwd = m @ basis
    with np.errstate(invalid="ignore", over="ignore"):
        score = a[None, :] + s @ m.T
        bound = E * U * (np.abs(a)[None, :] + np.abs(s) @ np.abs(m).T)
    N = obs.shape[0]
    idx = np.full((N, k), -1, dtype=np.int64)
    cost = np.full((N, k), np.nan)
    for n in range(N):
        ok = np.flatnonzero(~np.isnan(score[n]))
        order = ok[np.lexsort((ok, score[n, ok]))][:k]
        with np.errstate(invalid="ignore", over="ignore"):
            c = 0.5 * np.sum(w * (fwd[order] - obs[n]) ** 2, axis=1)
        srt = np.lexsort((order, np.where(np.isnan(c), np.inf, c), np.isnan(c)))
        idx[n, :len(order)] = order[srt]
        cost[n, :len(order)] = c[srt]
    return idx, cost, score, bound


def brute_costs(m, obs, weights=None, basis=None):
    """Per-wavelength costs of every (row, candidate) pair, (N, K)."""
    w = np.ones(obs.shape[1]) if weights is None else weights
    fwd = m if basis is None else m @ basis
    return 0.5 * np.sum(w * (fwd[None, :, :] - obs[:, None, :]) ** 2, axis=2)


def check_against_brute(idx, cost, brute, slack):
    """idx (N, k) is the top k of brute (N, K) up to near-ties within slack (N, K); rows sorted by (cost, index)."""
    N, k = idx.shape
    for n in range(N):
        sel = idx[n][idx[n] >= 0]
        finite = np.flatnonzero(~np.isnan(brute[n]))
        assert len(sel) == min(k, len(finite)), n
        if len(sel) == 0:
            continue
        assert len(set(sel.tolist())) == len(sel)
        kth = np.max(brute[n, sel])
        others = np.setdiff1d(finite, sel)
        # no unselected candidate is better than a selected one by more than the rounding slack of both
        if len(others):
            worst = sel[np.argmax(brute[n, sel])]
            assert np.all(brute[n, others] >= kth - slack[n, others] - slack[n, worst]), n
        c = cost[n, :len(sel)]
        assert np.all((c[:-1] < c[1:]) | ((c[:-1] == c[1:]) & (sel[:-1] < sel[1:]))), n


# ---- CPU -----------------------------------------------------------------------------------------------------------
def test_search_constants_and_argtypes_mirror_the_header(lib):
    from gp_emulator_b200 import _lib
    text = open(os.path.join(ROOT, "include", "gpemu.h")).read()
    defs = {k: int(v, 0) for k, v in re.findall(r"#define\s+(GPE_[A-Z0-9_]+)\s+(0x[0-9a-fA-F]+|\d+)", text)}
    assert defs["GPE_SEARCH_MAX_K"] == _lib.SEARCH_MAX_K == 16
    ctype = {"gpe_bank*": C.c_void_p, "gpe_multi*": C.c_void_p, "const double*": C.c_void_p, "double*": C.c_void_p,
             "int64_t*": C.c_void_p, "int64_t": C.c_int64, "int": C.c_int, "unsigned": C.c_uint, "void*": C.c_void_p}
    for name in ("gpe_bank_search", "gpe_multi_bank_search"):
        proto = re.search(r"int\s+%s\(([^)]*)\);" % name, text).group(1)
        params = [re.sub(r"\s+\w+$", "", p.strip()).replace(" *", "*") for p in proto.split(",")]
        assert [ctype[p] for p in params] == list(getattr(lib, name).argtypes), name
        assert getattr(lib, name).restype is C.c_int
        assert name in _lib.SYMBOLS


@pytest.mark.parametrize("spectra", [False, True])
def test_reference_agrees_with_a_per_wavelength_brute_force(spectra):
    rs = np.random.RandomState(3 + spectra)
    for trial in range(6):
        E, K, N, W = rs.randint(1, 9), rs.randint(1, 60), rs.randint(1, 12), rs.randint(1, 30)
        k = rs.randint(1, min(K, 16) + 1)
        m = rs.standard_normal((K, E))
        basis = rs.standard_normal((E, W)) if spectra else None
        obs = rs.standard_normal((N, W if spectra else E))
        w = rs.uniform(0.5, 2.0, obs.shape[1]) if trial % 2 else None
        m[rs.randint(K)] = np.nan                                   # a NaN candidate is never chosen
        obs[rs.randint(N)] = np.nan                                 # a NaN observation gets nothing
        idx, cost, _, bound = search_ref(m, obs, k, w, basis)
        brute = brute_costs(m, obs, w, basis)
        for n in range(N):
            if np.isnan(obs[n]).any():
                assert np.all(idx[n] == -1) and np.all(np.isnan(cost[n]))
        check_against_brute(idx, cost, brute, 4 * bound + 1e-12 * np.abs(brute))
        ok = idx >= 0
        assert np.allclose(cost[ok], np.take_along_axis(brute, np.maximum(idx, 0), 1)[ok], rtol=1e-12, atol=1e-12)


def test_reference_breaks_ties_by_index_and_keeps_infinite_scores():
    m = np.array([[1.0], [1.0], [0.0], [2.0]])
    idx, cost, _, _ = search_ref(m, np.array([[1.0]]), 3)
    assert idx.tolist() == [[0, 1, 2]] and cost.tolist() == [[0.0, 0.0, 0.5]]
    big = np.array([[1e300], [np.nan]])
    idx, cost, _, _ = search_ref(big, np.array([[-1e300]]), 2)
    assert idx.tolist() == [[0, -1]] and np.isinf(cost[0, 0]) and np.isnan(cost[0, 1])


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpemu(lib):
    import gp_emulator_b200 as g
    assert lib.gpe_device_count() > 0, "no GPU visible: the gpu tests must not pass on a fallback"
    return g


_PROBLEMS = {}


def _cached(gpemu, kind):
    if kind not in _PROBLEMS:
        _PROBLEMS[kind] = _problem(gpemu, kind)
    return _PROBLEMS[kind]


def _search(bank, spectra, *a, **kw):
    return (bank.forward_search if spectra else bank.search)(*a, **kw)


def _cost(bank, spectra, x, obs, w):
    return (bank.forward_cost if spectra else bank.cost)(x, obs, w, want_grad=False)["cost"]


def _host_search(lib, bank, spectra, cand, obs, N, obs_ld, w, k):
    """C-level host call (obs_ld = 0 with N > 1 has no Python spelling)."""
    from gp_emulator_b200 import _lib
    idx, cost = np.empty((N, k), dtype=np.int64), np.empty((N, k))
    flags = _lib.HOST_PTRS | (_lib.SOLVE_SPECTRA if spectra else 0)
    rc = lib.gpe_bank_search(bank._h, cand.ctypes.data, len(cand), obs.ctypes.data, N, obs_ld,
                             None if w is None else w.ctypes.data, k, idx.ctypes.data, cost.ctypes.data, flags, None)
    assert rc == 0, lib.gpe_last_error()
    return idx, cost


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "fwd", "prosail"])
@pytest.mark.parametrize("K", [100, 300])
@pytest.mark.parametrize("k", [1, 5, 16])
def test_against_an_exact_brute_force(lib, gpemu, kind, K, k):
    bank, spectra, lo, hi, rs = _cached(gpemu, kind)
    rs = np.random.RandomState(K + k)
    N = 23
    cand = lo + (hi - lo) * rs.uniform(0, 1, (K, len(lo)))
    x_true = lo + (hi - lo) * rs.uniform(0, 1, (N, len(lo)))
    obs_all = _own_obs(bank, spectra, x_true)
    obs_all = obs_all * (1.0 + 0.01 * rs.standard_normal(obs_all.shape))
    for shared in (False, True):
        for weighted in (False, True):
            w = rs.uniform(0.5, 2.0, obs_all.shape[1]) if weighted else None
            obs = np.ascontiguousarray(obs_all[0]) if shared else obs_all
            if shared:
                idx, cost = _host_search(lib, bank, spectra, cand, obs, N, 0, w, k)
                rows = np.broadcast_to(obs, obs_all.shape)
            else:
                got = _search(bank, spectra, cand, obs, w, k=k)
                idx, cost = got["idx"], got["cost"]
                rows = obs
            # brute force: the library's cost of every candidate against every row
            brute = np.stack([_cost(bank, spectra, cand, np.ascontiguousarray(rows[n]), w) for n in range(N)])
            ww = np.ones(rows.shape[1]) if w is None else w
            c_n = 0.5 * np.sum(ww * rows * rows, axis=1)
            slack = 1e-10 * (np.abs(brute) + c_n[:, None])
            check_against_brute(idx, cost, brute, slack)
            # every cost is, bit for bit, the cost call of those candidates on the same N points
            for j in range(k):
                assert np.all(idx[:, j] >= 0)
                assert np.array_equal(cost[:, j], _cost(bank, spectra, cand[idx[:, j]], obs, w))


def _setup(gpemu, kind, K=300, N=97, seed=0):
    bank, spectra, lo, hi, _ = _cached(gpemu, kind)
    rs = np.random.RandomState(seed)
    cand = lo + (hi - lo) * rs.uniform(0, 1, (K, len(lo)))
    x_true = lo + (hi - lo) * rs.uniform(0, 1, (N, len(lo)))
    obs = _own_obs(bank, spectra, x_true) * (1.0 + 0.01 * rs.standard_normal((N, 1)))
    w = rs.uniform(0.5, 2.0, obs.shape[1])
    return bank, spectra, lo, hi, cand, obs, w


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "fwd"])
def test_results_do_not_depend_on_placement_chunking_devices_order_or_split(lib, gpemu, monkeypatch, kind):
    import torch
    bank, spectra, lo, hi, cand, obs, w = _setup(gpemu, kind)
    k = 6
    ref = _search(bank, spectra, cand, obs, w, k=k)
    dev = _search(bank, spectra, torch.as_tensor(cand, device="cuda"), torch.as_tensor(obs, device="cuda"), w, k=k)
    torch.cuda.synchronize()
    for key in ("idx", "cost"):
        assert np.array_equal(dev[key].cpu().numpy(), ref[key])
    monkeypatch.setenv("GPE_SLOT_OUT_BYTES", str(2 * k * 8 * 13))   # chunks of 13 pixels
    seam = _search(bank, spectra, cand, obs, w, k=k)
    monkeypatch.delenv("GPE_SLOT_OUT_BYTES")
    for key in ("idx", "cost"):
        assert np.array_equal(seam[key], ref[key])
    E, D, W = (20, 10, 2101) if spectra else (24, 6, 0)
    inputs, thetas, invQts, invQs, brs = _models(E, D, 40, 0)          # the bank of tests.test_invert._bank
    basis = brs.standard_normal((E, W)) if W else None
    for devices in ([0, 0], "all"):
        multi = gpemu.DeviceBank(inputs, thetas, invQts, invQs, basis=basis, device=devices)
        got = _search(multi, spectra, cand, obs, w, k=k)
        multi.close()
        for key in ("idx", "cost"):
            assert np.array_equal(got[key], ref[key]), devices
    rs = np.random.RandomState(1)
    pn = rs.permutation(len(obs))
    got = _search(bank, spectra, cand, obs[pn], w, k=k)
    for key in ("idx", "cost"):
        assert np.array_equal(got[key], ref[key][pn])
    pc = rs.permutation(len(cand))
    got = _search(bank, spectra, cand[pc], obs, w, k=k)
    assert np.array_equal(pc[got["idx"]], ref["idx"])
    assert np.array_equal(got["cost"], ref["cost"])
    for n in (0, 50, 96):                                  # one pixel: the candidate groups spread over CTAs
        one = _search(bank, spectra, cand, obs[n], w, k=k)
        assert np.array_equal(one["idx"][0], ref["idx"][n])
        assert np.allclose(one["cost"][0], ref["cost"][n], rtol=1e-13, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "fwd"])
def test_nan_rows_nan_candidates_and_k_equal_to_K(gpemu, kind):
    bank, spectra, lo, hi, cand, obs, w = _setup(gpemu, kind, K=16, N=9)
    obs = obs.copy()
    obs[4] = np.nan
    cand = cand.copy()
    cand[7] = np.nan
    got = _search(bank, spectra, cand, obs, w, k=16)                   # k = K
    for n in range(9):
        if n == 4:                                                     # a NaN observation: nothing is selectable
            assert np.all(got["idx"][n] == -1) and np.all(np.isnan(got["cost"][n]))
            continue
        assert sorted(got["idx"][n][:15].tolist()) == [i for i in range(16) if i != 7]   # the NaN candidate never
        assert got["idx"][n][15] == -1 and np.isnan(got["cost"][n][15])


@pytest.mark.gpu
def test_argument_errors(lib, gpemu):
    from gp_emulator_b200 import _lib
    bank, spectra, lo, hi, cand, obs, w = _setup(gpemu, "band", K=20, N=4)
    idx, cost = np.empty((4, 16), dtype=np.int64), np.empty((4, 16))
    H = _lib.HOST_PTRS

    def call(b=bank._h, K=20, k=2, flags=H, obs_ld=24, i=idx.ctypes.data, c=cost.ctypes.data, N=4):
        return lib.gpe_bank_search(b, cand.ctypes.data, K, obs.ctypes.data, N, obs_ld, None, k, i, c, flags, None)

    assert call() == 0
    for bad in (dict(k=0), dict(k=17), dict(k=21), dict(K=0, k=1), dict(flags=H | _lib.SOLVE_SPECTRA), dict(obs_ld=7),
                dict(i=None, c=None), dict(flags=H | 0x4000), dict(N=-1), dict(b=None)):
        assert call(**bad) == -1, bad
    assert call(N=0) == 0
    rs = np.random.RandomState(0)
    E = 97
    big = gpemu.DeviceBank(rs.random_sample((10, 2)), np.zeros((E, 4)), rs.standard_normal((E, 10)))
    o = np.zeros((1, E))
    rc = lib.gpe_bank_search(big._h, cand[:, :2].copy().ctypes.data, 20, o.ctypes.data, 1, E, None, 1, idx.ctypes.data,
                             cost.ctypes.data, H, None)
    assert rc == -4
    big.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "fwd"])
def test_red_zones(lib, gpemu, kind):
    import torch
    from gp_emulator_b200 import _lib
    bank, spectra, lo, hi, cand, obs, w = _setup(gpemu, kind, K=150, N=33)
    k, pad = 5, 64
    flags = _lib.SOLVE_SPECTRA if spectra else 0
    ref = _search(bank, spectra, cand, obs, w, k=k)
    # host
    zi = np.full(33 * k + 2 * pad, -7, dtype=np.int64)
    zc = np.full(33 * k + 2 * pad, 12345.5)
    rc = lib.gpe_bank_search(bank._h, cand.ctypes.data, 150, obs.ctypes.data, 33, obs.shape[1], w.ctypes.data, k,
                             zi[pad:].ctypes.data, zc[pad:].ctypes.data, flags | _lib.HOST_PTRS, None)
    assert rc == 0
    assert np.all(zi[:pad] == -7) and np.all(zi[-pad:] == -7) and np.all(zc[:pad] == 12345.5) and np.all(zc[-pad:] == 12345.5)
    assert np.array_equal(zi[pad:-pad].reshape(33, k), ref["idx"]) and np.array_equal(zc[pad:-pad].reshape(33, k), ref["cost"])
    # device
    di = torch.full((33 * k + 2 * pad,), -7, dtype=torch.int64, device="cuda")
    dc = torch.full((33 * k + 2 * pad,), 12345.5, dtype=torch.float64, device="cuda")
    tc, to, tw = (torch.as_tensor(a, device="cuda") for a in (cand, obs, w))
    rc = lib.gpe_bank_search(bank._h, tc.data_ptr(), 150, to.data_ptr(), 33, obs.shape[1], tw.data_ptr(), k,
                             di[pad:].data_ptr(), dc[pad:].data_ptr(), flags, None)
    assert rc == 0
    torch.cuda.synchronize()
    zi, zc = di.cpu().numpy(), dc.cpu().numpy()
    assert np.all(zi[:pad] == -7) and np.all(zi[-pad:] == -7) and np.all(zc[:pad] == 12345.5) and np.all(zc[-pad:] == 12345.5)
    assert np.array_equal(zi[pad:-pad].reshape(33, k), ref["idx"]) and np.array_equal(zc[pad:-pad].reshape(33, k), ref["cost"])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "fwd"])
def test_invert_from_candidates(gpemu, kind):
    bank, spectra, lo, hi, cand, obs, w = _setup(gpemu, kind, K=300, N=40)
    solve = bank.forward_invert if spectra else bank.invert
    found = _search(bank, spectra, cand, obs, w, k=3)
    one = solve(None, obs, w, lower=lo, upper=hi, candidates=cand)
    ref = solve(cand[found["idx"][:, 0]], obs, w, lower=lo, upper=hi)
    for key in ref:
        assert np.array_equal(one[key], ref[key]), key
    assert np.array_equal(one["candidate"], found["idx"][:, 0])
    three = solve(None, obs, w, lower=lo, upper=hi, candidates=cand, n_starts=3)
    runs = [solve(cand[found["idx"][:, j]], obs, w, lower=lo, upper=hi) for j in range(3)]
    costs = np.stack([r["cost"] for r in runs], axis=1)
    best = np.argmin(np.where(np.isnan(costs), np.inf, costs), axis=1)   # first minimum: ties to the better-ranked start
    for key in ref:
        want = np.stack([runs[b][key][n] for n, b in enumerate(best)])
        assert np.array_equal(three[key], want), key
    assert np.array_equal(three["candidate"], found["idx"][np.arange(40), best])


@pytest.mark.gpu
def test_point_without_a_candidate_comes_back_nonfinite(gpemu):
    bank, spectra, lo, hi, cand, obs, w = _setup(gpemu, "band", K=50, N=5)
    obs = obs.copy()
    obs[2] = np.nan
    res = bank.invert(None, obs, w, lower=lo, upper=hi, candidates=cand, n_starts=2)
    assert res["status"][2] == NONFINITE and res["n_iter"][2] == 0 and np.all(np.isnan(res["x"][2]))
    assert res["candidate"][2] == -1
    assert np.all(res["status"][[0, 1, 3, 4]] == CONVERGED)


@pytest.mark.gpu
def test_multivariate_emulator_search_and_invert_use_the_training_design(gpemu):
    mv, g = _prosail(gpemu)
    lo, hi = g["y"].min(axis=0), g["y"].max(axis=0)
    rs = np.random.RandomState(2)
    x_true = lo + (hi - lo) * rs.uniform(0.1, 0.9, (3, 10))
    obs = mv.predict(x_true, do_deriv=False)
    s1 = mv.search(obs[0], k=4)
    assert s1["idx"].shape == (4,) and s1["cost"].shape == (4,)
    s_all = mv._device_bank().forward_search(np.atleast_2d(mv.y_train), obs[:1], k=4)
    assert np.array_equal(s1["idx"], s_all["idx"][0]) and np.array_equal(s1["cost"], s_all["cost"][0])
    r1 = mv.invert(obs[0], bounds=(lo, hi))
    r2 = mv.invert(obs[0], bounds=(lo, hi), candidates=mv.y_train)
    assert isinstance(r1["cost"], float) and isinstance(r1["candidate"], int)
    for key in r1:
        assert np.array_equal(np.asarray(r1[key]), np.asarray(r2[key])), key
    rn = mv.invert(obs, bounds=(lo, hi), n_starts=2)
    assert rn["x"].shape == (3, 10) and rn["candidate"].shape == (3,)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "fwd"])
def test_starts_from_a_latin_hypercube_table_reach_x_true_anywhere_in_the_box(gpemu, kind):
    """Noise-free observations of x_true drawn over the whole box; starts from a seeded lhd table of K = 4096 rows, the
    4 best of each pixel."""
    import scipy.stats
    bank, spectra, lo, hi, _ = _cached(gpemu, kind)
    width = hi - lo
    np.random.seed(17)
    table = gpemu.lhd(dist=[scipy.stats.uniform(loc=l, scale=s) for l, s in zip(lo, width)], size=4096)
    rs = np.random.RandomState(23)
    N = 100
    x_true = lo + width * rs.uniform(0, 1, (N, len(lo)))
    obs = _own_obs(bank, spectra, x_true)
    solve = bank.forward_invert if spectra else bank.invert
    res = solve(None, obs, lower=lo, upper=hi, max_iter=100, candidates=table, n_starts=4)
    assert np.max(np.abs(res["x"] - x_true) / width) <= 1e-8
