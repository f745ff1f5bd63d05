"""Every compiled FP64 predict instance against the oracle, at the batch sizes that select it.

The FP64 predict path is a table of template instances: ``predict_full_inst.cu`` is compiled once per padded input width
(``DPS`` in the Makefile) and instantiates ``k_predict_full`` for every row of ``kShape``; the host picks one per call from
(M, D, N) in ``plan_full`` / ``plan_call``.  Most oracle comparisons elsewhere run small batches, which land on the cluster
kernel or the 16-point small plan.  This file:

1. derives the list of fused instances from the build (CPU) and generates one sweep case per (DP, cfg, nt_act), plus a
   small-plan case per even cfg 0 nt_act; a test asserts the sweep covers every instance but the ``UNREACHABLE`` ones;
2. runs each case with N chosen so that every CTA loops over >= 3 tiles and the last tile is ragged, checks that the plan
   names the expected instance, and compares mu / var / deriv (and the fused Hessian for DP <= 16) with the oracle per
   point, on host arrays, an aligned device tensor (TMA prefetch) and a misaligned device view (in-line loads);
3. covers the other per-DP kernels: mean-only and Hessian-only calls of a model without invQ, the large-M variance path
   and the shared-difference bank kernels for every (DP, G, grad) that is compiled.

Errors are per point, scaled by the point's own magnitude sum, so that a wrong tile of small values cannot hide behind a
large one elsewhere.  Failure messages name the instance, DP, M, D and N.
"""
import os
import re

import numpy as np
import pytest

from oracle import gp_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-10

# ------------------------------------------------------------------------------------------------------------------
# 1. the instance matrix, derived from the build
# ------------------------------------------------------------------------------------------------------------------


def _read(*parts):
    with open(os.path.join(ROOT, *parts)) as f:
        return f.read()


def build_dps():
    """``DPS`` of the Makefile: the padded input widths predict_full_inst.cu is compiled for."""
    m = re.search(r"^DPS\s*:=\s*(.+)$", _read("Makefile"), re.M)
    return [int(x) for x in m.group(1).split()]


def build_shapes():
    """``kShape`` rows of predict_full_inst.cu: {cfg: (MT, WR, WC, MINB, KB, nt_lo, nt_max)}."""
    src = _read("gp_emulator_b200", "csrc", "predict_full_inst.cu")
    body = re.search(r"kShape\[\d+\]\s*=\s*\{(.*?)\n\};", src, re.S).group(1)
    rows = re.findall(r"\{\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*\}", body)
    return {cfg: tuple(int(v) for v in row) for cfg, row in enumerate(rows)}


def build_launches():
    """``launch_cfg<CFG, NT, EXACT>`` instantiations of launch_full: [(cfg, NT, exact)]."""
    src = _read("gp_emulator_b200", "csrc", "predict_full_inst.cu")
    body = re.search(r"static cudaError_t launch_full\(.*?\n\}", src, re.S).group(0)
    return [(int(c), int(n), e == "true") for c, n, e in re.findall(r"launch_cfg<(\d+),\s*(\d+),\s*(true|false)>", body)]


def full_name(dp, cfg, nt, fullnt, sym):
    """Instance name in the format of predict_full_inst.cu::full_name (what gpe_model_plan reports)."""
    mt, wr, wc, minb, kb, _, _ = build_shapes()[cfg]
    b = lambda x: "true" if x else "false"
    return "k_predict_full<%d,%d,%d,%d,%d,%d,%d,%s,%s,false>" % (mt, nt, wr, wc, dp, minb, kb, b(fullnt), b(sym))


def expected_instances():
    """Every non-Hessian k_predict_full instance the build compiles: launch_cfg<CFG, NT, EXACT> instantiates the
    predicate-free (FULLNT) kernel, and with EXACT = false also the column-predicated one, each plain and folded."""
    names = set()
    for dp in build_dps():
        for cfg, nt, exact in build_launches():
            for sym in (False, True):
                names.add(full_name(dp, cfg, nt, True, sym))
                if not exact:
                    names.add(full_name(dp, cfg, nt, False, sym))
    return names


def _unreachable():
    out = {}
    for dp in build_dps():
        for sym in (False, True):
            # cfg 1 runs for 256 < m32 and m64 <= 512, so nt_act = m64 / 64 is 5..8, and 5, 6, 7 and 8 all have their own
            # FULLNT instance: launch_cfg<1, 8, false> is only ever called with nt_act = 8, never with predicates.
            out[full_name(dp, 1, 8, False, sym)] = "cfg 1: nt_act is always 5..8"
        if dp >= 24:
            for sym in (False, True):
                # nt_act = 16 needs 960 < M <= 1024, so Mp = 1024.  The fixed carve-up, 192 + 256 + 16 (Mp + 4) 8
                # + 2 * 16 (D + 1) 8 + 4 * 16 (D + 1) 8 + 8 * 16 * 8 rounded to 128, is 152,320 B at D = 24 and
                # 158,464 B at D = 32, which leaves 78,080 / 71,936 B of the 230,400.  The smallest chunked plan needs
                # two 32 KB ring stages (Mp * 32) and 64 training rows of (x_pitch + 1) 8 = 216 / 280 B: 79,360 / 83,456 B.
                # plan_full is invalid for M = 961..1024 and the large-M path takes the call
                # (k_predict_mean2<DP,true> + k_var_large, checked in test_large_m_path).
                out[full_name(dp, 2, 16, True, sym)] = "DP >= 24: the cfg 2 nt_act = 16 plan exceeds shared memory"
    return out


UNREACHABLE = _unreachable()

# The sweep: which (cfg, nt_act) plan_full picks for M (mirrors gpemu.cu::plan_full).  Extending kShape or DPS means
# extending these tables, or test_sweep_covers_every_compiled_instance fails.
SWEEP_DPS = (2, 4, 6, 8, 10, 12, 16, 24, 32)
SWEEP_CFGS = {   # cfg: (TN, column-tile width of M, nt_act range)
    0: (64, 32, range(1, 9)),
    1: (32, 64, range(5, 9)),
    2: (16, 64, range(9, 17)),
}
SMALL_TN = 16


# --- a port of plan_full's shared-memory arithmetic, to pick M where the plan depends on more than the tile width ------
_SMEM_CAP = 232448 - 2048


def _x_pitch(dp):
    return dp if (dp // 2) & 1 else dp + 2


def _up(x, a):
    return (x + a - 1) // a * a


def plan_full(M, D, DP, small_Mp=0):
    """gpemu.cu::plan_full: None where the fused plan is invalid, else the fields the sweep uses."""
    m32, m64 = _up(M, 32), _up(M, 64)
    if small_Mp:
        cfg, TN, WC, GH, Mp = 2, 16, 8, 4, small_Mp
    elif m32 <= 256:
        cfg, TN, WC, GH, Mp = 0, 64, 4, 1, m32
    elif m64 <= 512:
        cfg, TN, WC, GH, Mp = 1, 32, 8, 2, m64
    elif m64 <= 1024:
        cfg, TN, WC, GH, Mp = 2, 16, 8, 4, m64
    else:
        return None
    nt = Mp // (32 if cfg == 0 and not small_Mp else 64)
    kblk = (M + 3) // 4
    stage = (2 if cfg == 0 else 1) * Mp * 32
    off = 192 + 256 + TN * (Mp + 4) * 8 + 2 * _up(TN * (D + 1) * 8, 16)
    off += _up(GH * TN * (D + 1) * 8, 16) if GH > 1 else 0
    off += WC * TN * 8
    nc = kbh = 0
    if DP <= 16:
        off += _up(TN * D * 8, 16)
        nc = (DP * (DP + 1) // 2 + 7) // 8 * 8
        kbh = stage // (nc * 32)
    fixed = _up(off, 128)
    m4, row = _up(M, 4), (_x_pitch(DP) + 1) * 8
    avail = _SMEM_CAP - fixed
    if avail >= m4 * row + 3 * stage:
        jc, nchunks = m4, 1
    else:
        if avail < 2 * stage + 64 * row:
            return None
        jc = min((avail - 2 * stage) // row // 4 * 4, 256, m4)
        nchunks = (M + jc - 1) // jc
    nstage = min(8, (avail - jc * row) // stage)
    if nstage < 2 or fixed + nstage * stage + jc * row > _SMEM_CAP:
        return None
    return dict(cfg=cfg, TN=TN, Mp=Mp, nt=nt, kblk=kblk, JC=jc, nchunks=nchunks, NC=nc, kbh=kbh)


def small_plan(M, D, DP):
    """The 16-point plan gpe_model_create_ex builds beside a cfg 0 plan, or None."""
    f = plan_full(M, D, DP)
    if f is None or f["cfg"] != 0 or f["Mp"] % 64:
        return None
    fs = plan_full(M, D, DP, f["Mp"])
    ok = fs is not None and (fs["JC"], fs["nchunks"], fs["kblk"]) == (f["JC"], f["nchunks"], f["kblk"])
    return fs if ok else None


def _m_choices(width, nt):
    """An exact multiple of the column-tile width, and a ragged M in the same nt_act: M % 4 != 0, not a multiple of 32,
    so the last k-block and the padded columns are partial."""
    return width * nt, width * (nt - 1) + 5


def sweep_cases():
    """One case per (DP, cfg, nt_act) and one small-plan case per even cfg 0 nt_act: dicts with dp, cfg, nt, M, D,
    small (16-point plan) and the instance name the default (sym False) model must report."""
    cases = []
    for dp in SWEEP_DPS:
        i = 0
        for cfg, (_, width, nts) in SWEEP_CFGS.items():
            for nt in nts:
                D = 1 if dp == 2 else (dp if i % 2 == 0 else dp - 1)
                exact, ragged = _m_choices(width, nt)
                for M in ((exact, ragged) if i % 2 == 0 else (ragged, exact)):
                    f = plan_full(M, D, dp)
                    if f is not None and (f["cfg"], f["nt"]) == (cfg, nt):
                        cases.append(dict(dp=dp, cfg=cfg, nt=nt, M=M, D=D, small=False))
                        break
                i += 1
        for nt in range(2, 9, 2):
            D = 1 if dp == 2 else (dp if i % 2 == 0 else dp - 1)
            exact, ragged = _m_choices(32, nt)
            for M in ((exact, ragged) if i % 2 == 0 else (ragged, exact)):
                if small_plan(M, D, dp) is not None:
                    cases.append(dict(dp=dp, cfg=0, nt=nt, M=M, D=D, small=True))
                    break
            i += 1
    for c in cases:
        c["names"] = {sym: (full_name(c["dp"], 2, 16, False, sym) if c["small"] else full_name(c["dp"], c["cfg"], c["nt"], True, sym))
                      for sym in (False, True)}
        c["id"] = "dp%d-%s-nt%d-M%d-D%d" % (c["dp"], "small" if c["small"] else "cfg%d" % c["cfg"], c["nt"], c["M"], c["D"])
    return cases


CASES = sweep_cases()


def test_build_tables_parse():
    """The parsers find what the build compiles: every kShape row's nt_act range has a launch, every DP is in DPS."""
    shapes, launches = build_shapes(), build_launches()
    assert len(shapes) >= 3 and build_dps()
    for cfg, (_, _, _, _, _, lo, hi) in shapes.items():
        assert {n for c, n, _ in launches if c == cfg} >= set(range(lo, hi + 1)), cfg


def test_sweep_covers_every_compiled_instance():
    """Every k_predict_full instance the build compiles is named by a sweep case, except the UNREACHABLE ones; a DP
    added to DPS or a shape added to kShape without extending the sweep fails here."""
    expected = expected_instances()
    assert set(UNREACHABLE) <= expected
    covered = {n for c in CASES for n in c["names"].values()}
    assert covered <= expected
    missing = expected - set(UNREACHABLE) - covered
    assert not missing, "instances without a sweep case: %s" % sorted(missing)
    assert set(SWEEP_DPS) == set(build_dps())
    assert set(SWEEP_CFGS) == set(build_shapes())
    # both training-set layouts (resident, chunked) of each cfg are reached
    for cfg in SWEEP_CFGS:
        layouts = {plan_full(c["M"], c["D"], c["dp"])["nchunks"] > 1 for c in CASES if c["cfg"] == cfg and not c["small"]}
        assert layouts == {False, True}, cfg
    # and the port agrees with the shapes the unreachable entries rest on
    for dp in (24, 32):
        assert all(plan_full(M, D, dp) is None for M in range(961, 1025) for D in (dp - 1, dp))


# ------------------------------------------------------------------------------------------------------------------
# helpers for the GPU tests
# ------------------------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def gpemu(lib):
    import gp_emulator_b200 as g
    assert lib.gpe_device_count() > 0, "no GPU visible: the gpu tests must not pass on a fallback"
    return g


@pytest.fixture(scope="module")
def sms(gpemu):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _model_data(M, D, N, seed):
    """The S model with mixed signs (invQ - 0.5, invQt - 0.5, theta - 1)."""
    inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed=seed)
    return inputs, theta - 1.0, invQ - 0.5, invQt - 0.5, testing


def _plant(testing, inputs, rows, rs):
    """Test rows equal to training rows (x - t exactly 0) and rows so far away that every k underflows to 0."""
    for i, n in enumerate(rows):
        if i % 2 == 0:
            testing[n] = inputs[rs.randint(inputs.shape[0])]
        else:
            testing[n] = 1.0e3 * (1 + (i % 3))


def _tile_rows(tiles, TN, N):
    return np.unique(np.concatenate([np.arange(t * TN, min((t + 1) * TN, N)) for t in tiles]))


def _scaled(diff, scale):
    """|diff| / scale per entry; where the scale is 0 (every k underflowed) the result must be exact."""
    diff = np.abs(diff)
    with np.errstate(divide="ignore", invalid="ignore"):
        e = np.where(scale > 0, diff / np.where(scale > 0, scale, 1.0), np.where(diff == 0, 0.0, np.inf))
    return e


def _mean_scales(inputs, theta, invQt, t):
    """Per-point magnitude sums: sum_j |k_nj invQt_j| for mu, w_d sum_j |k_nj (x_jd - t_nd) invQt_j| for deriv."""
    a, e = orc.cross_covariance(inputs, theta, t)            # (M, N)
    ka = np.abs(a) * np.abs(invQt)[:, None]
    D = inputs.shape[1]
    ds = np.empty((t.shape[0], D))
    buf = np.empty_like(ka)
    for d in range(D):
        np.subtract(inputs[:, d][:, None], t[:, d][None, :], out=buf)
        np.abs(buf, out=buf)
        buf *= ka
        ds[:, d] = e[d] * buf.sum(0)
    return ka.sum(0), ds


def _var_err(var, var_ref, inputs, theta, invQ, t):
    """orc.var_cond_err per point: |dvar_n| / (b + |k_n|^T |invQ| |k_n|)."""
    a, e = orc.cross_covariance(inputs, theta, t)
    scale = e[inputs.shape[1]] + np.sum(np.abs(a) * (np.abs(invQ) @ np.abs(a)), axis=0)
    return np.abs(np.asarray(var) - var_ref) / scale


def _check_var(tag, var, var_ref, var_scale_fn):
    e, at = _worst(var_scale_fn(var, var_ref))
    assert e < TOL, "%s: var error %.3g (condition-scaled) at row %s" % (tag, e, at)
    return e


def _hess_scale(inputs, theta, invQt, t):
    """sum_j |k_nj invQt_j| (|w_d (x_jd - t_nd)| |w_e (x_je - t_ne)| + delta_de w_d): the Hessian's magnitude sum."""
    a, e = orc.cross_covariance(inputs, theta, t)
    D = inputs.shape[1]
    ka = (np.abs(a) * np.abs(invQt)[:, None]).T               # (N, M)
    out = np.empty((t.shape[0], D, D))
    for s in range(0, t.shape[0], 256):
        wd = np.abs(e[:D] * (inputs[None, :, :] - t[s:s + 256, None, :]))      # (n, M, D)
        out[s:s + 256] = np.matmul((wd * ka[s:s + 256, :, None]).transpose(0, 2, 1), wd)
        out[s:s + 256] += ka[s:s + 256].sum(1)[:, None, None] * np.diag(e[:D])[None]
    return out


def _worst(err):
    i = int(np.argmax(err))
    return float(err.flat[i]), np.unravel_index(i, err.shape)


def _check_mean(tag, got, mu, deriv, mu_s, der_s, tol=TOL, rows=None):
    rows = slice(None) if rows is None else rows
    e_mu, at_mu = _worst(_scaled(got["mu"][rows] - mu, mu_s))
    assert e_mu < tol, "%s: mu error %.3g at row %s" % (tag, e_mu, at_mu)
    e_d, at_d = _worst(_scaled(got["deriv"][rows] - deriv, der_s))
    assert e_d < tol, "%s: deriv error %.3g at (row, d) %s" % (tag, e_d, at_d)
    return max(e_mu, e_d)


def _check_hess(tag, hess, ref, scale, tol=TOL):
    e, at = _worst(_scaled(hess - ref, scale))
    assert e < tol, "%s: Hessian error %.3g at (row, d, e) %s" % (tag, e, at)
    return e


def _sample_rows(N, TN, grid, n_seeded, seed):
    """Rows for the oracle checks that cost O(D^2) per point: the first and last tiles, the tiles on either side of each
    gridDim boundary, and n_seeded seeded rows."""
    ntiles = (N + TN - 1) // TN
    tiles = {0, ntiles - 1}
    for b in range(grid, ntiles, grid):
        tiles |= {b - 1, b}
    rows = _tile_rows(sorted(tiles), TN, N)
    rs = np.random.RandomState(seed)
    return np.unique(np.concatenate([rows, rs.randint(0, N, n_seeded)]))


def _device_views(testing):
    """An aligned CUDA tensor (16-byte start: the TMA prefetch path) and a view 8 bytes off a 16-byte boundary (every
    tile takes the in-line load path): one row in for odd D, a one-element offset into a flat buffer for even D."""
    import torch
    N, D = testing.shape
    aligned = torch.from_numpy(testing).cuda()
    assert aligned.data_ptr() % 16 == 0
    if D % 2:
        big = torch.empty((N + 1, D), dtype=torch.float64, device="cuda")
        big[1:] = aligned
        mis = big[1:]
    else:
        flat = torch.empty(N * D + 1, dtype=torch.float64, device="cuda")
        flat[1:] = aligned.reshape(-1)
        mis = flat[1:].view(N, D)
    assert mis.data_ptr() % 16 == 8 and mis.is_contiguous()
    return aligned, mis


def _device_call(m, t, **kw):
    """One call on device data, and the number of kernel launches it made (a host call makes one per streamed chunk)."""
    from gp_emulator_b200 import _lib
    lib = _lib.load()
    before = lib.gpe_launch_count()
    out = {k: v.cpu().numpy() for k, v in m.predict(t, **kw).items()}
    return out, lib.gpe_launch_count() - before


def _three_calls(tag, m, testing, dev, mis, launches=None, **kw):
    """Host arrays, aligned and misaligned device data: bit-identical results; `launches`: what the aligned device call
    must launch."""
    host = m.predict(testing, **kw)
    a, n = _device_call(m, dev, **kw)
    if launches is not None:
        assert n == launches, "%s: %d kernel launches, expected %d" % (tag, n, launches)
    b = {k: v.cpu().numpy() for k, v in m.predict(mis, **kw).items()}
    for k in host:
        assert np.array_equal(host[k], a[k], equal_nan=True), "%s: %s differs between host and aligned device data" % (tag, k)
        assert np.array_equal(host[k], b[k], equal_nan=True), "%s: %s differs between host and misaligned device data" % (tag, k)
    return host


_WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    """Prints the largest per-point scaled error seen in each family when the module ends (visible with -s)."""
    yield
    for k in sorted(_WORST):
        print("\ninstance matrix: largest per-point scaled error, %-10s %.3g" % (k, _WORST[k]), end="")


def _note(family, err):
    _WORST[family] = max(_WORST.get(family, 0.0), err)


def _plan_head(plan):
    return plan.split(" (")[0]


# ------------------------------------------------------------------------------------------------------------------
# 2. fused instances against the oracle
# ------------------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_plan_names_every_reachable_instance(gpemu, sms):
    """m.plan(N) of every sweep case names its expected instance, and across the sweep the reported names are exactly
    the compiled instances minus UNREACHABLE.  The fused line also reports the training-set layout, and each cfg is
    reached both resident (nchunks = 1) and chunked."""
    reported, layouts = set(), set()
    for c in CASES:
        M, D = c["M"], c["D"]
        N = _n_case(c, sms)
        inputs = np.random.RandomState(M + D).random_sample((M, D))
        theta, invQ, invQt = np.zeros(D + 2), np.eye(M), np.ones(M)
        for sym in (False, True):
            m = gpemu.DeviceModel(inputs, theta, invQt, invQ, symmetric_variance=sym)
            plan = m.plan(N)
            assert _plan_head(plan) == c["names"][sym], (c["id"], N, sym, plan)
            f = plan_full(M, D, c["dp"], 64 * c["nt"] // 2 if c["small"] else 0)
            assert "JC=%d, nchunks=%d)" % (f["JC"], f["nchunks"]) in plan, (c["id"], plan)
            reported.add(c["names"][sym])
            if not c["small"]:
                layouts.add((c["cfg"], f["nchunks"] > 1))
            m.close()
    assert reported == expected_instances() - set(UNREACHABLE), sorted(reported ^ (expected_instances() - set(UNREACHABLE)))
    assert layouts == {(cfg, ch) for cfg in SWEEP_CFGS for ch in (False, True)}


def _n_case(c, sms):
    """Every CTA runs >= 3 tiles and the last tile is ragged; the small plan stays just under its 3 * 16 * #SM bound."""
    if c["small"]:
        return 3 * 16 * sms - 5
    TN = SWEEP_CFGS[c["cfg"]][0]
    return 3 * sms * TN + TN // 2 + 1


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c["id"] for c in CASES])
def test_fused_instance_against_oracle(gpemu, sms, case):
    """Default and symmetric-folded model, three calls each (host, aligned device, misaligned device), per-point errors
    against the oracle; for DP <= 16 the fused Hessian against the oracle on a row sample."""
    dp, M, D = case["dp"], case["M"], case["D"]
    N = _n_case(case, sms)
    TN = SMALL_TN if case["small"] else SWEEP_CFGS[case["cfg"]][0]
    ntiles = (N + TN - 1) // TN
    grid = min(ntiles, sms)
    tag = "%s (DP %d, M %d, D %d, N %d)" % (case["names"][False], dp, M, D, N)
    inputs, theta, invQ, invQt, testing = _model_data(M, D, N, seed=1000 * dp + M + D)
    rs = np.random.RandomState(M * D + 1)
    planted = np.concatenate([np.arange(3) * 7 + 1,                           # first tile
                              (grid + 1) * TN + np.arange(3) * 5,             # a second-round tile
                              N - 1 - np.arange(3) * 3])                      # the ragged last tile
    _plant(testing, inputs, planted, rs)

    mu_o, var_o, der_o = orc.predict(inputs, theta, invQ, invQt, testing)
    mu_s, der_s = _mean_scales(inputs, theta, invQt, testing)
    a, ex = orc.cross_covariance(inputs, theta, testing)
    v_scale = ex[D] + np.sum(np.abs(a) * (np.abs(invQ) @ np.abs(a)), axis=0)
    del a
    var_err = lambda v, ref: np.abs(v - ref) / v_scale
    dev, mis = _device_views(testing)

    outs = {}
    for sym in (False, True):
        m = gpemu.DeviceModel(inputs, theta, invQt, invQ, symmetric_variance=sym)
        name = case["names"][sym]
        assert _plan_head(m.plan(N)) == name, (tag, m.plan(N))
        stag = "%s (DP %d, M %d, D %d, N %d)" % (name, dp, M, D, N)
        out = _three_calls(stag, m, testing, dev, mis)
        err = _check_mean(stag, out, mu_o, der_o, mu_s, der_s)
        ev = _check_var(stag, out["var"], var_o, var_err)
        _note("small plan" if case["small"] else "fused", max(err, ev))
        outs[sym] = (m, out)
    # phase A (mean and gradient) is the same code in both forms
    for k in ("mu", "deriv"):
        assert np.array_equal(outs[False][1][k], outs[True][1][k]), "%s: %s differs between plain and folded model" % (tag, k)

    if dp > 16 or case["small"]:
        return
    # fused Hessian: one launch when build_hessian_operand takes the model (NC <= M, kbh >= 1; the centred-radius guard
    # holds for inputs in [0, 1) at these length scales), two otherwise
    plan = outs[False][0].plan(N)
    Mp = int(re.search(r"Mp=(\d+)", plan).group(1))
    kbps = 2 if case["cfg"] == 0 else 1
    nc = (dp * (dp + 1) // 2 + 7) // 8 * 8
    fused = nc <= M and nc <= Mp and kbps * Mp // nc >= 1
    rows = _sample_rows(N, TN, grid, 1000, seed=dp + M)
    h_ref = orc.hessian(inputs, theta, invQt, testing[rows])
    h_scale = _hess_scale(inputs, theta, invQt, testing[rows])
    m = outs[False][0]
    htag = tag + (" + fused Hessian" if fused else " + direct Hessian")
    out, n = _device_call(m, dev, want_hess=True)
    assert n == (1 if fused else 2), "%s: %d kernel launches" % (htag, n)
    _check_mean(htag, out, mu_o, der_o, mu_s, der_s)
    _check_var(htag, out["var"], var_o, var_err)
    _note("Hessian", _check_hess(htag, out["hess"][rows], h_ref, h_scale))
    if case["cfg"] == 0 and fused:
        # Hessian only, symmetric-folded model: phase B is skipped, so the Hessian still rides on the fused kernel
        ms = outs[True][0]
        h, n = _device_call(ms, dev, want_mu=False, want_var=False, want_deriv=False, want_hess=True)
        h = h["hess"]
        assert n == 1, "%s (Hessian only, folded model): %d kernel launches" % (htag, n)
        _note("Hessian", _check_hess(htag + " (Hessian only, folded model)", h[rows], h_ref, h_scale))
    for m, _ in outs.values():
        m.close()


# ------------------------------------------------------------------------------------------------------------------
# 3. the other per-DP kernels
# ------------------------------------------------------------------------------------------------------------------
_MEAN_TN = 32           # predict_mean.cuh::kMeanTN
_MEAN_CTAS = (12, 8)    # CTAs per SM of the mean + gradient and of the Hessian launches (gpemu.cu::predict_device)


def _dp_d(dp, i):
    return 1 if dp == 2 else (dp if i % 2 == 0 else dp - 1)


MEAN_CASES = [(dp, _dp_d(dp, i), M) for i, dp in enumerate(SWEEP_DPS) for M in (203, 300)]   # resident; 256 + 44


@pytest.mark.gpu
@pytest.mark.parametrize("dp,D,M", MEAN_CASES, ids=["dp%d-D%d-M%d" % c for c in MEAN_CASES])
def test_mean_and_hessian_kernels(gpemu, sms, dp, D, M):
    """A model without invQ (no fused plan): mean + gradient from k_predict_mean / k_predict_mean2 as the DP selects,
    the Hessian from k_predict_mean<DP,true> (DP <= 12) or k_hessian_rows.  M = 203 keeps the training set resident,
    M = 300 takes two chunks with a ragged last one; N makes both grids loop."""
    N = _MEAN_CTAS[0] * sms * _MEAN_TN + 17
    inputs, theta, _, invQt, testing = _model_data(M, D, N, seed=7 * dp + M)
    rs = np.random.RandomState(dp + M)
    _plant(testing, inputs, [1, 5, N - 1, N - 4, _MEAN_CTAS[1] * sms * _MEAN_TN + 3], rs)
    m = gpemu.DeviceModel(inputs, theta, invQt)
    plan = m.plan(N)
    kern = "k_predict_mean" if dp == 12 or dp >= 24 else "k_predict_mean2"
    assert _plan_head(plan) == "%s<%d,false>" % (kern, dp), plan
    tag = "%s<%d,false> (DP %d, M %d, D %d, N %d)" % (kern, dp, dp, M, D, N)
    rows = np.unique(np.concatenate([_sample_rows(N, _MEAN_TN, _MEAN_CTAS[0] * sms, 1000, seed=dp),
                                     _sample_rows(N, _MEAN_TN, _MEAN_CTAS[1] * sms, 0, seed=dp)]))
    t = testing[rows]
    mu_o, _, der_o = orc.predict(inputs, theta, None, invQt, t, do_unc=False)
    mu_s, der_s = _mean_scales(inputs, theta, invQt, t)
    dev, mis = _device_views(testing)
    out = _three_calls(tag, m, testing, dev, mis, want_var=False)
    _note("mean", _check_mean(tag, out, mu_o, der_o, mu_s, der_s, rows=rows))
    hk = "k_predict_mean<%d,true>" % dp if dp <= 12 else "k_hessian_rows<%d,%d>" % (dp, 4 if dp <= 16 else 2)
    htag = "%s (DP %d, M %d, D %d, N %d)" % (hk, dp, M, D, N)
    h = _three_calls(htag, m, testing, dev, mis, launches=1, want_mu=False, want_var=False, want_deriv=False, want_hess=True)["hess"]
    _note("Hessian", _check_hess(htag, h[rows], orc.hessian(inputs, theta, invQt, t), _hess_scale(inputs, theta, invQt, t)))


LARGE_CASES = [(dp, _dp_d(dp, i), 1100) for i, dp in enumerate((8, 12, 16, 24, 32))] + [(24, 24, 1000), (32, 31, 961), (32, 32, 1024)]


@pytest.mark.gpu
@pytest.mark.parametrize("dp,D,M", LARGE_CASES, ids=["dp%d-D%d-M%d" % c for c in LARGE_CASES])
def test_large_m_path(gpemu, sms, dp, D, M):
    """k_predict_mean2<DP,true> + k_var_large: M = 1100 at the DPs without a test elsewhere, and M = 961..1024 at DP 24 / 32,
    where the cfg 2 nt_act = 16 plan does not fit (UNREACHABLE).  N spans several K*-scratch sub-batches."""
    N = 16 * sms * 4 + 37
    inputs, theta, invQ, invQt, testing = _model_data(M, D, N, seed=11 * dp + M)
    _plant(testing, inputs, [0, 3, 16 * sms * 4 + 1, N - 1, N - 2], np.random.RandomState(dp))
    m = gpemu.DeviceModel(inputs, theta, invQt, invQ)
    plan = m.plan(N)
    assert plan.startswith("k_predict_mean2<%d,true> + k_var_large" % dp), plan
    tag = "k_predict_mean2<%d,true> + k_var_large (DP %d, M %d, D %d, N %d)" % (dp, dp, M, D, N)
    mu_o, var_o, der_o = orc.predict(inputs, theta, invQ, invQt, testing)
    mu_s, der_s = _mean_scales(inputs, theta, invQt, testing)
    dev, mis = _device_views(testing)
    out = _three_calls(tag, m, testing, dev, mis)
    err = _check_mean(tag, out, mu_o, der_o, mu_s, der_s)
    ev = _check_var(tag, out["var"], var_o, lambda v, ref: _var_err(v, ref, inputs, theta, invQ, testing))
    _note("large-M", max(err, ev))


def bank_group_ok(dp, G, grad):
    """launch.h::bank_group_ok: the group sizes the shared-difference bank kernel is compiled for."""
    if not grad:
        return dp <= 16 and G in (4, 5, 8, 10)
    if dp <= 10:
        return 3 <= G <= 5
    return (dp == 12 and G in (3, 4)) or (dp == 16 and G in (2, 3))


def test_bank_group_table_matches_the_launcher():
    """The (DP, G, grad) list above is what predict_full_inst.cu::launch_bank_mean dispatches."""
    src = _read("gp_emulator_b200", "csrc", "launch.h")
    body = re.search(r"inline bool bank_group_ok\(.*?\n\}", src, re.S).group(0)
    assert "G == 4 || G == 5 || G == 8 || G == 10" in body and "G >= 3 && G <= 5" in body
    assert "DP == 12) return G == 3 || G == 4" in body and "DP == 16) return G == 2 || G == 3" in body


BANK_CASES = [(dp, G, grad) for dp in SWEEP_DPS for grad in (True, False) for G in range(2, 11) if bank_group_ok(dp, G, grad)]


@pytest.mark.gpu
@pytest.mark.parametrize("dp,G,grad", BANK_CASES, ids=["dp%d-G%d-%s" % (d, g, "grad" if r else "mean") for d, g, r in BANK_CASES])
def test_bank_group_kernel(gpemu, sms, monkeypatch, dp, G, grad):
    """k_bank_mean<DP,G,GRAD> for every compiled (DP, G, grad): G forced at bank creation, E = 2G + 1 so the last group
    is ragged, N large enough that the group kernel is chosen and its grid loops.  Each emulator is checked per point."""
    import torch
    i = BANK_CASES.index((dp, G, grad))
    D, M = _dp_d(dp, i), (45 if i % 2 == 0 else 300)
    E = 2 * G + 1
    N = 32 * sms + 17
    assert (N + 31) // 32 * ((E + G - 1) // G) >= sms
    rs = np.random.RandomState(100 * dp + 10 * G + grad)
    inputs = rs.random_sample((M, D))
    thetas = rs.random_sample((E, D + 2)) - 1.0
    invQts = rs.random_sample((E, M)) - 0.5
    t = rs.random_sample((N, D))
    _plant(t, inputs, [2, 9, 32 * sms + 1, N - 1], rs)
    monkeypatch.setenv("GPE_BANK_G" if grad else "GPE_BANK_G_MEAN", str(G))
    bank = gpemu.DeviceBank(inputs, thetas, invQts)
    monkeypatch.delenv("GPE_BANK_G" if grad else "GPE_BANK_G_MEAN")
    tag = "k_bank_mean<%d,%d,%s> (DP %d, M %d, D %d, E %d, N %d)" % (dp, G, "true" if grad else "false", dp, M, D, E, N)
    host = bank.predict(t, want_var=False, want_deriv=grad)
    dev, n = _device_call(bank, torch.from_numpy(t).cuda(), want_var=False, want_deriv=grad)
    assert n == 1, "%s: %d kernel launches" % (tag, n)
    for k in host:
        assert np.array_equal(host[k], dev[k]), "%s: %s differs between host and device data" % (tag, k)
    worst = 0.0
    for e in range(E):
        mu_o, _, der_o = orc.predict(inputs, thetas[e], None, invQts[e], t, do_unc=False)
        mu_s, der_s = _mean_scales(inputs, thetas[e], invQts[e], t)
        etag = "%s emulator %d" % (tag, e)
        em, at = _worst(_scaled(host["mu"][:, e] - mu_o, mu_s))
        assert em < TOL, "%s: mu error %.3g at row %s" % (etag, em, at)
        worst = max(worst, em)
        if grad:
            ed, at = _worst(_scaled(host["deriv"][:, e] - der_o, der_s))
            assert ed < TOL, "%s: deriv error %.3g at (row, d) %s" % (etag, ed, at)
            worst = max(worst, ed)
    _note("bank group", worst)
