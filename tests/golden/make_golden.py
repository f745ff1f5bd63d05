#!/usr/bin/env python
"""Freeze outputs of the REFERENCE implementation into tests/golden/*.npz.

Needs a checkout of the reference project; the fixtures it writes are committed, so the tests need neither the
reference nor this script.

The reference package is Python 2 (print statements, xrange, tab/space mixing) and imports its compiled
``_gpu_predict`` at module scope, so it cannot be imported.  This script reads the reference *source text*,
applies a purely mechanical token-level py2->py3 conversion IN MEMORY (nothing is written to disk, no
reference source enters this repository) and executes the result.  All arithmetic that produces the
goldens is therefore the reference's own numpy/scipy code:

  GaussianProcess.predict / cpu_predict   gp_emulator/GaussianProcess.py:211-251, 327-341
  GaussianProcess.hessian                 gp_emulator/GaussianProcess.py:345-366
  GaussianProcess._set_params             gp_emulator/GaussianProcess.py:52-75, 127-139
  MultivariateEmulator (dump=...) .predict gp_emulator/multivariate_gp.py:40-121, 195-222
  GaussianProcess.loglikelihood / partial_devs  gp_emulator/GaussianProcess.py:78-125
  lhd                                     gp_emulator/lhd.py:11-269
  GaussianProcess.get_gpu_block           gp_emulator/GaussianProcess.py:253-270
  per-band bank pattern (E x predict + hessian on shared inputs)   tests/test_perband_emulator.py:22-47
  MultivariateEmulator(X=, y=, hyperparams=) with 20 PCs x 2101 wavelengths (BASELINE config 4)

    python tests/golden/make_golden.py REFERENCE_DIR [--only S1500]
"""
import hashlib
import os
import re
import sys
import types

import numpy as np

if len(sys.argv) < 2 or sys.argv[1].startswith("-"):
    sys.exit(__doc__)
REF = sys.argv[1]
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import gp_oracle as orc  # noqa: E402  (input generators only; outputs come from the reference)


def py2to3(src):
    src = src.expandtabs(8)
    src = re.sub(r"^(\s*)import _gpu_predict\s*$", r"\1pass", src, flags=re.M)
    src = src.replace("xrange", "range").replace("np.int(", "int(")
    src = re.sub(r"^(\s*)print (.*?),?\s*$", r"\1print(\2)", src, flags=re.M)
    src = re.sub(r"raise ValueError, (\".*?\")", r"raise ValueError(\1)", src)
    src = src.replace("from GaussianProcess import GaussianProcess", "")
    # py2 `range` is a list the reference assigns into (get_gpu_block, GaussianProcess.py:259,266)
    src = re.sub(r"^(\s*\w+ = )range\((.*)\)\s*$", r"\1list(range(\2))", src, flags=re.M)
    # numpy of the reference's era let a boolean mask be shorter than the axis it indexes (multivariate_gp.py:159:
    # 250 singular values against the 2101 rows of the full V); current numpy raises, so make the truncation explicit
    src = src.replace("V [ pcnt_var_explained <= thresh ]", "V [ :s.size ][ pcnt_var_explained <= thresh ]")
    return src


def load_reference():
    gp_mod = types.ModuleType("ref_GaussianProcess")
    with open(os.path.join(REF, "gp_emulator", "GaussianProcess.py")) as f:
        exec(compile(py2to3(f.read()), "ref:GaussianProcess.py", "exec"), gp_mod.__dict__)
    mv_mod = types.ModuleType("ref_multivariate_gp")
    mv_mod.GaussianProcess = gp_mod.GaussianProcess
    with open(os.path.join(REF, "gp_emulator", "multivariate_gp.py")) as f:
        exec(compile(py2to3(f.read()), "ref:multivariate_gp.py", "exec"), mv_mod.__dict__)
    return gp_mod.GaussianProcess, mv_mod.MultivariateEmulator


def sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a, dtype=np.float64).tobytes())
    return h.hexdigest()


def ref_gp(RefGP, inputs, theta, invQ, invQt):
    gp = RefGP(inputs, [])
    gp.theta, gp.invQ, gp.invQt = theta, invQ, invQt      # exactly how tests/benchmark.py:11-15 sets them
    return gp


def main():
    RefGP, RefMV = load_reference()

    # ---- S: tests/benchmark.py-style all-U(0,1) model (config 1 and config 3 shapes) ---------------
    only = sys.argv[sys.argv.index("--only") + 1] if "--only" in sys.argv else None   # regenerate one fixture
    for tag, (M, D, N, seed, nh) in {"S250": (250, 10, 300, 0, 40), "S1000": (1000, 10, 64, 3, 0),
                                     "S37": (37, 3, 130, 5, 130), "S1500": (1500, 6, 48, 7, 8)}.items():
        if only and tag != only:
            continue
        inputs, theta, invQ, invQt, testing = orc.make_S_model(M, D, N, seed)
        gp = ref_gp(RefGP, inputs, theta, invQ, invQt)
        mu, var, deriv = gp.predict(testing)
        mu2, deriv2 = gp.predict(testing, do_unc=False)
        assert np.array_equal(mu, mu2) and np.array_equal(deriv, deriv2)
        out = dict(M=M, D=D, N=N, seed=seed, input_sha=sha(inputs, theta, invQ, invQt, testing), mu=mu, var=var,
                   deriv=deriv)
        if nh:
            out["hess"] = gp.hessian(testing[:nh])
        np.savez_compressed(os.path.join(HERE, "golden_%s.npz" % tag), **out)
        print(tag, "mu[:2]", mu[:2], "var[:2]", var[:2])

    # ---- L: training objective and gradient (loglikelihood + partial_devs) at the reference's start distribution ----
    if not only or only == "L":
        out = {}
        for tag, (M, D, T, B, seed) in {"a": (60, 4, 3, 6, 21), "b": (250, 10, 2, 4, 22), "c": (33, 2, 1, 5, 23)}.items():
            inputs, targets, thetas, tidx = orc.make_training_problem(M, D, T, B, seed)
            ll = np.empty(B); grad = np.empty((B, D + 2))
            for n in range(B):
                gp = RefGP(inputs, targets[tidx[n]])
                ll[n] = gp.loglikelihood(thetas[n])
                grad[n] = gp.partial_devs(thetas[n])
            out.update({"shape_" + tag: np.array([M, D, T, B, seed]), "ll_" + tag: ll, "grad_" + tag: grad,
                        "sha_" + tag: sha(inputs, targets, thetas)})
            print("L%s  ll[:2]" % tag, ll[:2])
        np.savez_compressed(os.path.join(HERE, "golden_L.npz"), **out)
    # ---- U: lhd designs under a seeded legacy numpy RNG (gp_emulator/lhd.py:11-269) ---------------------------------
    if not only or only == "U":
        import scipy.stats as ss
        lhd_mod = types.ModuleType("ref_lhd")
        with open(os.path.join(REF, "gp_emulator", "lhd.py")) as f:
            exec(compile(py2to3(f.read()), "ref:lhd.py", "exec"), lhd_mod.__dict__)
        d0, d1, d2, d3 = ss.uniform(loc=-1, scale=2), ss.norm(loc=0, scale=1), ss.beta(2, 5), ss.expon(scale=1 / 1.5)
        out = {}
        np.random.seed(5); out["single"] = lhd_mod.lhd(dist=d0, size=5)
        np.random.seed(6); out["dims"] = lhd_mod.lhd(dist=d1, size=7, dims=5)
        np.random.seed(7); out["multi"] = lhd_mod.lhd(dist=(d1, d2, d3), size=6)
        np.random.seed(8); out["big"] = lhd_mod.lhd(dist=(d0, d1, d2, d3), size=100)
        np.random.seed(9); out["space"] = lhd_mod.lhd(dist=(d0, d1, d2, d3), size=12, form="spacefilling", iterations=7)
        np.savez_compressed(os.path.join(HERE, "golden_U.npz"), **out)
        print("U   single", out["single"].ravel())
    # ---- B: block boundaries of the reference's host chunker (GaussianProcess.get_gpu_block, :253-270) --------------
    if not only or only == "B":
        gp = RefGP(np.zeros((3, 2)), [])
        cases = [(10, 4), (12345, 1000), (100000, 200000), (900000, 100000), (200001, 200000), (7, 7), (8, 7), (1, 5)]
        out = {"cases": np.array(cases)}
        for i, (size, block) in enumerate(cases):
            a, b = gp.get_gpu_block(size, block)
            out["start_%d" % i] = np.asarray(a, dtype=np.int64); out["end_%d" % i] = np.asarray(b, dtype=np.int64)
        np.savez_compressed(os.path.join(HERE, "golden_B.npz"), **out)
        print("B   ", [(out["start_0"].tolist(), out["end_0"].tolist())])
    # ---- K: per-band bank -- E GaussianProcess objects on the same inputs, own theta / targets, each predicted and
    # differentiated twice separately (the loop of tests/test_perband_emulator.py:22-47) -------------------------------
    if not only or only == "K":
        rs = np.random.RandomState(31)
        M, D, E, N = 60, 4, 5, 40
        inputs = rs.random_sample((M, D)); testing = rs.random_sample((N, D))
        thetas = rs.random_sample((E, D + 2)) - 0.5
        targets = np.sin(inputs.sum(axis=1))[None, :] * (1.0 + rs.random_sample((E, 1))) + 0.1 * rs.standard_normal((E, M))
        mu = np.empty((N, E)); var = np.empty((N, E)); deriv = np.empty((N, E, D)); hess = np.empty((N, E, D, D))
        invQ = np.empty((E, M, M)); invQt = np.empty((E, M))
        for e in range(E):
            gp = RefGP(inputs, targets[e])
            gp._set_params(np.r_[thetas[e, :D + 1], -4.0])
            invQ[e], invQt[e] = gp.invQ, gp.invQt
            mu[:, e], var[:, e], deriv[:, e, :] = gp.predict(testing)
            hess[:, e] = gp.hessian(testing)
        thetas[:, D + 1] = -4.0
        np.savez_compressed(os.path.join(HERE, "golden_K.npz"), inputs=inputs, testing=testing, thetas=thetas, invQ=invQ,
                            invQt=invQt, mu=mu, var=var, deriv=deriv, hess=hess)
        print("K    mu[0]", mu[0])
    # ---- M20: BASELINE config 4 -- MultivariateEmulator with 2101 wavelengths compressed to 20 PCs, built by the
    # reference's own constructor (SVD + per-PC _set_params), single-point predicts (all the reference supports) ------
    if not only or only == "M20":
        rs = np.random.RandomState(41)
        M, D, W = 250, 10, 2101
        y = rs.random_sample((M, D))
        lam = np.linspace(0.0, 1.0, W)
        # smooth synthetic spectra: a few dozen parameter-dependent bumps, so the singular values decay slowly enough
        X = np.zeros((M, W))
        for k in range(40):
            a = rs.standard_normal(D)
            X += np.cos(y @ a + k)[:, None] * np.exp(-0.5 * ((lam - rs.random_sample()) / (0.02 + 0.1 * rs.random_sample())) ** 2)[None, :]
        s = np.linalg.svd(X, compute_uv=False)
        frac = s.cumsum() / s.sum()
        thresh = 0.5 * (frac[19] + frac[20])                      # exactly 20 components pass `<= thresh`
        hyper = np.tile(np.r_[[-0.5] * D, 0.0, -6.0][:, None], (1, 20)) + 0.3 * rs.standard_normal((D + 2, 20))
        hyper[D + 1] = -6.0
        mv = RefMV(X=X, y=y, hyperparams=hyper, thresh=thresh)
        assert mv.n_pcs == 20, mv.n_pcs
        pts = np.vstack([y[3], rs.random_sample((3, D))])
        wsub = np.arange(0, W, 5)
        fwd = np.empty((4, W)); dsub = np.empty((4, D, wsub.size))
        for k in range(4):
            f, d = mv.predict(pts[k])
            fwd[k] = f; dsub[k] = np.asarray(d)[:, wsub]
        np.savez_compressed(os.path.join(HERE, "golden_M20.npz"), y=y, hyperparams=hyper, thresh=thresh,
                            basis_functions=mv.basis_functions, n_pcs=20, train_data=mv.compress(X),
                            invQt=np.stack([g.invQt for g in mv.emulators]), points=pts, fwd=fwd, wsub=wsub, deriv_sub=dsub)
        print("M20  n_pcs", mv.n_pcs, "fwd[0,:3]", fwd[0, :3])
    if only and only not in ("T", "P"):
        return
    # ---- T: genuinely conditioned model through the reference's own _set_params ---------------------
    inputs, targets, theta, _, _, testing = orc.make_T_model(M=100, D=4, N=200, seed=1)
    gp = RefGP(inputs, targets)
    gp._set_params(theta)
    mu, var, deriv = gp.predict(testing)
    hess = gp.hessian(testing)
    np.savez_compressed(os.path.join(HERE, "golden_T.npz"), inputs=inputs, targets=targets, theta=theta,
                        invQ=gp.invQ, invQt=gp.invQt, testing=testing, mu=mu, var=var, deriv=deriv, hess=hess)
    print("T   mu[:2]", mu[:2], "var[:2]", var[:2])

    # ---- P: the reference's trained PROSAIL MultivariateEmulator (data/prosail_30_0_30_0.npz) -------
    mv = RefMV(dump=os.path.join(REF, "data", "prosail_30_0_30_0.npz"))
    y = mv.y_train
    lo, hi = y.min(axis=0), y.max(axis=0)
    rs = np.random.RandomState(11)
    testing = lo + (hi - lo) * rs.random_sample((48, y.shape[1]))
    P = mv.n_pcs
    pc_mu = np.empty((48, P)); pc_var = np.empty((48, P)); pc_deriv = np.empty((48, P, y.shape[1]))
    for i, g in enumerate(mv.emulators):
        pc_mu[:, i], pc_var[:, i], pc_deriv[:, i, :] = g.predict(testing)
    hess0 = mv.emulators[0].hessian(testing[:8])
    pts = np.vstack([y[0], testing[0], testing[1]])
    wsub = np.arange(0, mv.basis_functions.shape[1], 7)
    fwd = np.empty((3, mv.basis_functions.shape[1])); dsub = np.empty((3, y.shape[1], wsub.size))
    for k in range(3):
        f, d = mv.predict(pts[k])
        fwd[k] = f
        dsub[k] = np.asarray(d)[:, wsub]
    np.savez_compressed(
        os.path.join(HERE, "golden_P.npz"), y=y, hyperparams=mv.hyperparams, basis_functions=mv.basis_functions,
        n_pcs=P, train_data=mv.compress(mv.X_train), invQt=np.stack([g.invQt for g in mv.emulators]),
        testing=testing, pc_mu=pc_mu, pc_var=pc_var, pc_deriv=pc_deriv, hess0=hess0, points=pts, fwd=fwd,
        wsub=wsub, deriv_sub=dsub)
    print("P   n_pcs", P, "fwd[0,:3]", fwd[0, :3])
    for fn in sorted(os.listdir(HERE)):
        if fn.endswith(".npz"):
            print("%-18s %8d bytes" % (fn, os.path.getsize(os.path.join(HERE, fn))))


if __name__ == "__main__":
    main()
