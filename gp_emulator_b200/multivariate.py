"""Drop-in ``MultivariateEmulator`` (reference gp_emulator/multivariate_gp.py:38-222): PCA-compressed
multivariate output, one GP per principal component, prediction on the B200 engine.

Construction (SVD, npz load/save, per-PC training) is host-side numpy, same npz wire format as the
reference (``X, y, hyperparams, thresh, basis_functions, n_pcs``).  ``predict`` keeps the reference's
single-point call and return shapes, and additionally accepts N > 1 points (the reference cannot:
multivariate_gp.py:216 fails to broadcast), evaluated as one bank launch plus one back-projection.
"""
from __future__ import annotations

import os
import shutil

import numpy as np

from .engine import DeviceBank, resolve_devices
from .gaussian_process import GaussianProcess


class MultivariateEmulator(object):
    def __init__(self, dump=None, X=None, y=None, hyperparams=None, thresh=0.98, n_tries=5, device=0,
                 batched_training=False, basis_functions=None, n_pcs=None):
        """See reference multivariate_gp.py:40-121.  ``X`` (N_train, N_full) model outputs, ``y``
        (N_train, N_params) the parameters that produced them, ``hyperparams`` (N_params + 2, n_pcs).
        ``device``: GPU index, list of indices or ``"all"`` (host batches are then spread over all of them per call)."""
        if basis_functions is not None and n_pcs is None:      # (EmulatorStorage hands a stored basis back in)
            n_pcs = basis_functions.shape[0]
        if dump is not None:
            if X is not None or y is not None:
                raise ValueError("You specified both a dump file and X and y")
            with np.load(dump) as f:
                X = f["X"]
                y = f["y"]
                hyperparams = f["hyperparams"]
                if "thresh" in f:
                    thresh = float(f["thresh"])
                if "basis_functions" in f:
                    basis_functions = f["basis_functions"]
                    n_pcs = int(f["n_pcs"])
            if basis_functions is None:
                # older dumps carry no basis: decompose once and rewrite the file (reference :79-90)
                self.calculate_decomposition(X, thresh)
                basis_functions, n_pcs = self.basis_functions, self.n_pcs
                tmp = os.path.join("/tmp", os.path.basename(dump))
                np.savez_compressed(tmp, X=X, y=y, hyperparams=hyperparams, thresh=thresh,
                                    basis_functions=basis_functions, n_pcs=n_pcs)
                shutil.move(tmp if tmp.endswith(".npz") else tmp + ".npz", dump)
        else:
            if X is None or y is None:
                raise ValueError("Need to specify both X and y")
            assert X.shape[0] == y.shape[0]
            assert X.ndim == 2
            assert y.ndim == 2

        self.X_train = X
        self.y_train = y
        self.thresh = thresh
        self.device = device
        if basis_functions is None:
            self.calculate_decomposition(X, thresh)
            basis_functions, n_pcs = self.basis_functions, self.n_pcs
        self.n_pcs = int(n_pcs)
        self.basis_functions = basis_functions
        if hyperparams is not None:
            assert (y.shape[1] + 2 == hyperparams.shape[0]) and (self.n_pcs == hyperparams.shape[1])
        self._bank, self._bank_key = None, None
        self.train_emulators(X, y, hyperparams=hyperparams, n_tries=n_tries, batched=batched_training)

    def dump_emulator(self, fname):
        """Save for reuse, reference npz format (multivariate_gp.py:124-137)."""
        np.savez_compressed(fname, X=self.X_train, y=self.y_train, hyperparams=self.hyperparams,
                            thresh=self.thresh, basis_functions=self.basis_functions, n_pcs=self.n_pcs)

    def calculate_decomposition(self, X, thresh):
        """PCA by SVD; keep the components whose cumulative singular-value share is <= thresh
        (reference multivariate_gp.py:140-160)."""
        # (the reference asks LAPACK for the full (N_full, N_full) right factor and uses its first min(N_train, N_full)
        # rows; the economy factorisation returns just those rows -- same singular values, vectors equal to the last
        # bit or two -- and is 14x cheaper at 250 x 2101)
        _, s, V = np.linalg.svd(X, full_matrices=False)
        keep = (s.cumsum() / s.sum()) <= thresh
        self.basis_functions = V[: keep.size][keep]
        self.n_pcs = int(np.sum(keep))

    def train_emulators(self, X, y, hyperparams, n_tries=2, batched=False):
        """One GP per PC on the compressed outputs (reference multivariate_gp.py:162-188).

        ``batched=True`` (only meaningful when ``hyperparams`` is None): all ``n_pcs * n_tries`` L-BFGS-B descents run
        in lockstep, their cost + gradient evaluations served by one GPU launch per round (``training.py``) -- the PCs
        share the training inputs ``y``, so they are one batch of (theta, target vector) problems.
        """
        self.emulators = []
        train_data = self.compress(X)
        self.hyperparams = np.zeros((2 + y.shape[1], self.n_pcs))
        gps = [GaussianProcess(np.atleast_2d(y), train_data[i], device=self.device) for i in range(self.n_pcs)]
        if hyperparams is None and batched:
            from .training import DeviceTrainer, minimise_batched
            D = y.shape[1]
            # the same random draws, in the same order, as n_pcs sequential learn_hyperparameters calls
            starts = [(i, th) for i in range(self.n_pcs) for th in 5.0 * (np.random.rand(n_tries, D + 2) - 0.5)]
            trainer = DeviceTrainer(np.atleast_2d(y), train_data, device=resolve_devices(self.device)[0])
            try:
                fits, self.training_stats = minimise_batched(trainer.evaluate, starts)
            finally:
                trainer.close()
            for i, gp in enumerate(gps):
                mine = fits[i * n_tries:(i + 1) * n_tries]
                best = int(np.argsort(np.array([f[1] for f in mine]))[0])
                print("After %d, the minimum cost was %e" % (n_tries, mine[best][1]))
                self.hyperparams[:, i] = mine[best][0]
                gp._set_params(self.hyperparams[:, i])
        else:
            for i, gp in enumerate(gps):
                if hyperparams is None:
                    self.hyperparams[:, i] = gp.learn_hyperparameters(n_tries=n_tries)[1]
                else:
                    self.hyperparams[:, i] = hyperparams[:, i]
                    gp._set_params(hyperparams[:, i])
        self.emulators = gps
        self.invalidate_device()

    def compress(self, X):
        """Project full-rank vectors onto the PC basis (reference multivariate_gp.py:191-193)."""
        return X.dot(self.basis_functions.T).T

    def _device_bank(self):
        """Device copy of the per-PC GPs and the basis, rebuilt when any emulator's state is rebound (each
        ``GaussianProcess`` counts assignments to inputs / theta / invQ / invQt, so ``emulators[i]._set_params(...)``
        is seen) or the basis is replaced.  In-place edits of an emulator's arrays need ``invalidate_device()``."""
        key = (tuple((id(g), g._version) for g in self.emulators), id(self.basis_functions), self.n_pcs, str(self.device))
        if self._bank is None or key != self._bank_key:
            if self._bank is not None:
                self._bank.close()
            gps = self.emulators
            self._bank = DeviceBank(np.atleast_2d(self.y_train), np.stack([g.theta for g in gps]),
                                    np.stack([g.invQt for g in gps]), np.stack([g.invQ for g in gps]),
                                    basis=self.basis_functions[: self.n_pcs], device=self.device)
            self._bank_key = key
        return self._bank

    def invalidate_device(self):
        """Drop the device copy of the emulator bank (the next predict re-uploads it)."""
        if self._bank is not None:
            self._bank.close()
        self._bank, self._bank_key = None, None

    def predict(self, y, do_deriv=True, is_gpu=True):
        """Reconstruct the full output (and its Jacobian) at parameter vector(s) ``y``.

        One point, as in the reference (multivariate_gp.py:195-222): returns ``fwd (N_full,)`` and
        ``deriv (N_params, N_full)``.  N > 1 points (new): ``fwd (N, N_full)``, ``deriv (N, N_params, N_full)``.
        """
        bank = self._device_bank()
        if isinstance(y, np.ndarray) or not hasattr(y, "is_cuda"):
            # host caller: one library call (latency matters: the reference is used one point per call)
            y2 = np.atleast_2d(y)
            res = bank.forward(y2, want_deriv=do_deriv)
            fwd, dfull = res if do_deriv else (res, None)
        else:                                # torch CUDA tensor: everything stays on the device
            y2 = y if y.dim() == 2 else y.reshape(1, -1)
            out = bank.predict(y2, want_var=False, want_deriv=False, project=True, project_deriv=do_deriv)
            fwd, dfull = out["fwd"], out.get("deriv_full")
        if y2.shape[0] == 1:
            return (fwd[0], dfull[0]) if do_deriv else fwd[0]
        return (fwd, dfull) if do_deriv else fwd

    def cost(self, y, obs, weights=None, do_deriv=True, do_hess=False):
        """Misfit of the reconstructed output at parameter vector(s) ``y`` against observed output(s) ``obs`` and its
        gradient in ``y``: ``cost = 1/2 sum_w weights_w (fwd_w - obs_w)^2``, ``grad_d = sum_w weights_w (fwd_w - obs_w)
        deriv_dw`` with fwd / deriv those of ``predict``, reduced on the device without forming them.  ``do_hess``: also
        the exact Hessian in ``y`` (for Newton steps; with weights 1 / sigma^2, ``inv(hess)`` at the optimum is the
        Laplace approximation of the posterior covariance).

        ``obs`` (N_full,) is shared by every point, (N, N_full) is one per point; ``weights`` (N_full,) or None (all 1).
        Returns the requested items in the order cost, grad, hess -- one point: ``float``, ``(N_params,)``,
        ``(N_params, N_params)``; N points: ``(N,)``, ``(N, N_params)``, ``(N, N_params, N_params)`` -- and the cost
        alone, not in a tuple, when it is the only one.  Host arrays or CUDA tensors, as ``predict``.
        """
        bank = self._device_bank()
        if isinstance(y, np.ndarray) or not hasattr(y, "is_cuda"):
            y2 = np.atleast_2d(y)
        else:
            y2 = y if y.dim() == 2 else y.reshape(1, -1)
        out = bank.forward_cost(y2, obs, weights, want_grad=do_deriv, want_hess=do_hess)
        res = [out["cost"]] + ([out["grad"]] if do_deriv else []) + ([out["hess"]] if do_hess else [])
        if y2.shape[0] == 1:
            c = res[0]
            res = [float(c[0]) if isinstance(c, np.ndarray) else c[0]] + [a[0] for a in res[1:]]
        return tuple(res) if len(res) > 1 else res[0]

    def invert(self, obs, y0, weights=None, bounds=None, prior=None, max_iter=50, ftol=1e-10, xtol=1e-10, gtol=0.0,
               do_cov=True):
        """Retrieve the parameters whose reconstructed output best fits ``obs``: per point, the minimiser of ``cost``
        (plus ``1/2 (y - m)^T P (y - m)`` with ``prior = (m, P)``) inside ``bounds = (lower, upper)``, by bounded
        Levenberg-Marquardt on the exact Hessian with every iteration on the device (``DeviceBank.forward_invert``).
        With weights 1 / sigma^2 the cost is a negative log-likelihood and ``cov = inv(hess)`` at the optimum is the
        Laplace approximation of the posterior covariance.

        ``y0`` (N_params,) or (N, N_params) starting points; ``obs`` (N_full,) shared or (N, N_full) one per point;
        ``lower`` / ``upper`` (N_params,) or None; ``m`` (N_params,) or (N, N_params), ``P`` (N_params, N_params).
        Returns a dict ``x``, ``cost``, ``grad``, ``hess``, ``cov`` (with ``do_cov``), ``status``, ``n_iter`` -- one point:
        ``(N_params,)``, ``float``, ``(N_params,)``, ``(N_params, N_params)``, ..., ``int``, ``int``; N points: the same with
        a leading N.  Host arrays or CUDA tensors, as ``predict``."""
        bank = self._device_bank()
        if isinstance(y0, np.ndarray) or not hasattr(y0, "is_cuda"):
            y2 = np.atleast_2d(y0)
        else:
            y2 = y0 if y0.dim() == 2 else y0.reshape(1, -1)
        lower, upper = bounds if bounds is not None else (None, None)
        m, P = prior if prior is not None else (None, None)
        out = bank.forward_invert(y2, obs, weights, lower=lower, upper=upper, prior_mean=m, prior_precision=P,
                                  max_iter=max_iter, ftol=ftol, xtol=xtol, gtol=gtol, want_cov=do_cov)
        if y2.shape[0] == 1:
            one = {k: v[0] for k, v in out.items()}
            for k in ("cost", "status", "n_iter"):
                one[k] = (float if k == "cost" else int)(one[k]) if isinstance(one[k], np.generic) else one[k]
            return one
        return out

    def predict_pcs(self, y, do_unc=True, do_deriv=True):
        """PC-space outputs for N points: dict with mu (N, P), var (N, P), deriv (N, P, D)."""
        return self._device_bank().predict(np.atleast_2d(y), want_var=do_unc, want_deriv=do_deriv)
