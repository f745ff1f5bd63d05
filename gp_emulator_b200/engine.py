"""Handles on device-resident models: thin, typed wrappers over the libgpemu C ABI.

``DeviceModel`` is one trained GP on one GPU, ``DeviceBank`` is E GPs that share training inputs and test
points (the per-PC emulators of a MultivariateEmulator, or a per-band bank).  Test points may be

* numpy arrays (host): the library streams them through its chunked host pipeline and the results
  come back as numpy arrays; or
* torch CUDA tensors (device): the call is asynchronous on torch's current stream and the results are
  torch CUDA tensors -- PyTorch is used only to own the device buffers.
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from . import _lib
from ._lib import (WANT_DERIV, WANT_DERIV_FULL, WANT_FWD, WANT_HESS, WANT_MU, WANT_VAR, HOST_PTRS, GpemuError, addr, check,
                   f64c)


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _pinned_empty(shape):
    """numpy array backed by torch's caching pinned-host allocator (the view keeps the block alive)."""
    import torch
    return torch.empty(shape, dtype=torch.float64, pin_memory=True).numpy()


def resolve_devices(device):
    """``device`` argument of the drop-in classes -> list of device indices: an int, a list of ints, or "all"."""
    if isinstance(device, str):
        if device != "all":
            raise ValueError('device must be an index, a list of indices or "all"')
        n = _lib.load().gpe_device_count()
        if n < 1:
            raise GpemuError("no CUDA device available; gp_emulator_b200 has no CPU fallback")
        return list(range(n))
    if isinstance(device, (list, tuple)):
        if not device:
            raise ValueError("empty device list")
        return [int(d) for d in device]
    return [int(device)]


# Result arrays of host calls.  A fresh pageable numpy array costs page faults + a CPU copy out of the staging buffer
# every call (the kernel zero-fills its pages: ~26 GB/s on the GPU box against 52 GB/s for warm pages); a page-locked
# one costs ~0.7 s/GB to create but is then recycled by torch's caching host allocator and lets the D2H copy land in
# it directly.  ``pinned=None`` (the default) therefore switches to page-locked results from the second request of
# the same total size on, for sizes where it pays and stays bounded.
# Auto-pinned result arrays that callers still hold count against ``AUTO_PIN_BUDGET`` bytes (page-locked memory is
# not swappable: a caller that keeps every result must not be able to lock down the host); beyond it fresh results are
# pageable again.
_AUTO_PIN_MIN, _AUTO_PIN_MAX = 1 << 20, 1 << 30
AUTO_PIN_BUDGET = 4 << 30
_pin_requests = {}
_pin_outstanding = [0]


def _auto_pin(nbytes):
    if not (_AUTO_PIN_MIN <= nbytes <= _AUTO_PIN_MAX):
        return False
    if len(_pin_requests) > 512:
        _pin_requests.clear()
    seen = _pin_requests.get(nbytes, 0)
    _pin_requests[nbytes] = seen + 1
    return seen >= 1 and _pin_outstanding[0] + nbytes <= AUTO_PIN_BUDGET


def _auto_pinned_empty(shape):
    """Page-locked result array charged to the auto-pin budget until the caller drops it."""
    a = _pinned_empty(shape)
    n = a.nbytes
    _pin_outstanding[0] += n

    def _release(n=n):
        _pin_outstanding[0] -= n
    weakref.finalize(a, _release)
    return a


def _weights_ld(shape, K, N):
    """Row pitch of the weights of a call with observations K wide: 0 for one (K,) vector shared by every point (or
    None), K for one row per point (N, K)."""
    if shape is None or tuple(shape) == (K,):
        return 0
    if tuple(shape) == (N, K):
        return K
    raise ValueError(f"weights must be ({K},) or ({N}, {K})")


def _check_out(out, k, shape):
    a = out[k]
    if not isinstance(a, np.ndarray) or a.shape != shape or a.dtype != np.float64 or not a.flags.c_contiguous:
        raise ValueError(f"out[{k!r}] must be a C-contiguous float64 numpy array of shape {shape}")


class _Handle:
    """Owner of one libgpemu handle: ``close()`` destroys it and later use raises instead of reaching freed memory."""

    def _own(self, h, destroy):
        self._hh = h
        self._fin = weakref.finalize(self, destroy, h)

    @property
    def _h(self):
        if self._hh is None:
            raise GpemuError("this device handle has been closed")
        return self._hh

    def close(self):
        self._fin()
        self._hh = None


def _current_stream_ptr(device_index):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device_index).cuda_stream)


def _host_result_factory(pinned, N, D, missing):
    """Allocator for the result arrays a host call has to create (see ``DeviceModel.predict`` for ``pinned``)."""
    if pinned is None:
        per_point = {"mu": 1, "var": 1, "deriv": D, "hess": D * D}
        if bool(missing) and _auto_pin(8 * N * sum(per_point[k] for k in missing)):
            return _auto_pinned_empty
        return np.empty
    return _pinned_empty if pinned else np.empty


class DeviceModel(_Handle):
    """One GP resident on one device.  Mirrors the state ``GaussianProcess.predict`` reads
    (reference gp_emulator/GaussianProcess.py:228-249): inputs (M, D), theta (D+2), invQ (M, M), invQt (M)."""

    def __init__(self, inputs, theta, invQt, invQ=None, device=0, symmetric_variance=False):
        """``symmetric_variance=True`` opts into evaluating k^T invQ k through the upper-triangular fold of invQ
        (exact identity for any invQ, half the tensor-core work, rounding differs at the 1e-16 level);
        ``"auto"`` folds only when ``invQ`` is symmetric to 1e-6 of its largest entry -- what the inverse of a
        covariance matrix is (``_prepare_likelihood``: ~3e-10), unlike the random ``invQ`` of the reference benchmark."""
        inputs = f64c(inputs)
        if inputs.ndim != 2:
            raise ValueError("inputs must be (M, D)")
        self.M, self.D = inputs.shape
        theta = f64c(theta).ravel()
        if theta.size < self.D + 1:
            raise ValueError(f"theta must hold at least D+1 = {self.D + 1} entries, got {theta.size}")
        expx = np.exp(theta[: self.D + 1])
        invQt = f64c(invQt).ravel()
        if invQt.size != self.M:
            raise ValueError("invQt must have M entries")
        if invQ is not None:
            invQ = f64c(invQ)
            if invQ.shape != (self.M, self.M):
                raise ValueError("invQ must be (M, M)")
        self.device = int(device)
        self.has_var = invQ is not None
        h = C.c_void_p()
        self.symmetric_variance = _symmetric_choice(symmetric_variance, invQ, self.M)
        check(_lib.load().gpe_model_create_ex(self.device, self.M, self.D, addr(inputs), addr(expx), addr(invQt),
                                              addr(invQ), _lib.OPT_SYMMETRIC_VARIANCE if self.symmetric_variance else 0,
                                              C.byref(h)))
        self._own(h, _lib.load().gpe_model_destroy)

    def predict(self, testing, want_var=True, want_deriv=True, want_hess=False, want_mu=True, out=None,
                pinned=None):
        """Returns a dict with the requested arrays among mu (N,), var (N,), deriv (N, D), hess (N, D, D).

        ``out`` may hold preallocated result arrays under the same keys (float64, C-contiguous, right shape;
        numpy for host calls, CUDA tensors for device calls): they are filled in place and returned.  Fresh host
        results are ordinary numpy arrays; ``pinned`` chooses their memory: False pageable (staged through the
        library's page-locked buffers), True page-locked (the D2H copy lands in them directly; ~0.7 s per GB the
        first time a size is seen, then recycled by torch's caching allocator), None (default) page-locked from the
        second request of the same size on -- repeated calls, as in an optimisation loop, then run at the pinned rate.
        """
        lib = _lib.load()
        D = self.D
        if want_var and not self.has_var:
            raise GpemuError("variance requested but the model was uploaded without invQ")
        flags = (WANT_MU if want_mu else 0) | (WANT_VAR if want_var else 0) | (WANT_DERIV if want_deriv else 0) | (
            WANT_HESS if want_hess else 0)
        wanted = [k for k, w in (("mu", want_mu), ("var", want_var), ("deriv", want_deriv), ("hess", want_hess)) if w]
        out = dict(out) if out else {}
        if _is_torch(testing):
            import torch
            t = testing
            if not t.is_cuda or t.device.index != self.device:
                raise ValueError(f"torch test points must live on cuda:{self.device}")
            if t.dtype != torch.float64 or t.dim() != 2 or t.shape[1] != D:
                raise ValueError(f"testing must be float64 (N, {D})")
            t = t.contiguous()
            N = t.shape[0]
            shapes = {"mu": (N,), "var": (N,), "deriv": (N, D), "hess": (N, D, D)}
            for k in wanted:
                if k not in out:
                    out[k] = torch.empty(shapes[k], dtype=torch.float64, device=t.device)
                elif (tuple(out[k].shape) != shapes[k] or out[k].dtype != torch.float64 or not out[k].is_cuda
                      or not out[k].is_contiguous()):
                    raise ValueError(f"out[{k!r}] must be a contiguous float64 CUDA tensor of shape {shapes[k]}")
            check(lib.gpe_predict(self._h, addr(t), N, addr(out.get("mu")), addr(out.get("var")),
                                  addr(out.get("deriv")), addr(out.get("hess")), flags,
                                  _current_stream_ptr(self.device)))
            return {k: out[k] for k in wanted}
        t = f64c(testing)
        if t.ndim != 2 or t.shape[1] != D:
            raise ValueError(f"testing must be (N, {D})")
        N = t.shape[0]
        shapes = {"mu": (N,), "var": (N,), "deriv": (N, D), "hess": (N, D, D)}
        missing = [k for k in wanted if k not in out]
        mk = _host_result_factory(pinned, N, D, missing)
        for k in wanted:
            if k not in out:
                out[k] = mk(shapes[k])
            else:
                _check_out(out, k, shapes[k])
        check(lib.gpe_predict(self._h, addr(t), N, addr(out.get("mu")), addr(out.get("var")),
                              addr(out.get("deriv")), addr(out.get("hess")), flags | HOST_PTRS, None))
        return {k: out[k] for k in wanted}


    def plan(self, n_points):
        """Name and tile plan of the kernel a mean + variance + gradient call of ``n_points`` runs (diagnostic)."""
        buf = C.create_string_buffer(512)
        _lib.load().gpe_model_plan(self._h, int(n_points), buf, 512)
        return buf.value.decode()

    def predict_f32(self, testing, want_var=True, want_deriv=True, fast=None):
        """Single-precision prediction on the tcgen05 / TMEM path (M <= 256): float32 in, float32 out.

        numpy float32 (N, D) -> numpy results; torch float32 CUDA tensor -> torch results (asynchronous).
        The variance contraction runs on the tensor cores: 3xTF32 split by default (FP32-grade, meets the
        reference's 1e-5 FP32 criterion); ``fast=True`` uses a single TF32 pass (error ~1e-4, ~1.7x faster).
        ``fast=None`` (default) = split for M <= 256, single pass above (where FP32 accumulation dominates the
        error anyway); ``fast=False`` forces the split for any M.
        """
        lib = _lib.load()
        D = self.D
        if want_var and not self.has_var:
            raise GpemuError("variance requested but the model was uploaded without invQ")
        flags = WANT_MU | (WANT_VAR if want_var else 0) | (WANT_DERIV if want_deriv else 0) | (
            _lib.F32_FAST_TF32 if fast else (_lib.F32_FORCE_3X if fast is False else 0))
        if _is_torch(testing):
            import torch
            t = testing
            if not t.is_cuda or t.device.index != self.device or t.dtype != torch.float32 or t.dim() != 2 \
                    or t.shape[1] != D:
                raise ValueError(f"testing must be a float32 (N, {D}) tensor on cuda:{self.device}")
            t = t.contiguous()
            N = t.shape[0]
            mk = lambda *s: torch.empty(*s, dtype=torch.float32, device=t.device)
            out = {"mu": mk(N)}
            if want_var: out["var"] = mk(N)
            if want_deriv: out["deriv"] = mk(N, D)
            check(lib.gpe_predict_f32(self._h, addr(t), N, addr(out["mu"]), addr(out.get("var")),
                                      addr(out.get("deriv")), flags, _current_stream_ptr(self.device)))
            return out
        t = np.ascontiguousarray(testing, dtype=np.float32)
        if t.ndim != 2 or t.shape[1] != D:
            raise ValueError(f"testing must be (N, {D})")
        N = t.shape[0]
        out = {"mu": np.empty(N, dtype=np.float32)}
        if want_var: out["var"] = np.empty(N, dtype=np.float32)
        if want_deriv: out["deriv"] = np.empty((N, D), dtype=np.float32)
        check(lib.gpe_predict_f32(self._h, addr(t), N, addr(out["mu"]), addr(out.get("var")),
                                  addr(out.get("deriv")), flags | HOST_PTRS, None))
        return out


def _symmetric_choice(symmetric_variance, invQ, M):
    if isinstance(symmetric_variance, str):
        if symmetric_variance != "auto":
            raise ValueError('symmetric_variance must be True, False or "auto"')
        return bool(invQ is not None and M > 1
                    and float(np.max(np.abs(invQ - invQ.T))) <= 1e-6 * float(np.max(np.abs(invQ))))
    return bool(symmetric_variance)


class MultiDeviceModel(_Handle):
    """One GP resident on several GPUs of the box, one call (``gpe_multi_*``).

    Host arrays: the batch is cut into chunks that the devices' pipelines (one host thread each inside the library, no
    Python threads, no collective) pull from a shared cursor, so GPUs behind slower PCIe paths take fewer chunks.
    Device data: a CUDA tensor that lives on one of the handle's devices is predicted there; a list with one tensor per
    device (``None`` for devices without work) is predicted on all of them asynchronously.  Results are bit-identical
    to ``DeviceModel`` on one GPU.
    """

    def __init__(self, inputs, theta, invQt, invQ=None, devices=None, symmetric_variance=False):
        inputs = f64c(inputs)
        if inputs.ndim != 2:
            raise ValueError("inputs must be (M, D)")
        self.M, self.D = inputs.shape
        theta = f64c(theta).ravel()
        if theta.size < self.D + 1:
            raise ValueError(f"theta must hold at least D+1 = {self.D + 1} entries, got {theta.size}")
        expx = np.exp(theta[: self.D + 1])
        invQt = f64c(invQt).ravel()
        if invQt.size != self.M:
            raise ValueError("invQt must have M entries")
        invQ = None if invQ is None else f64c(invQ)
        if invQ is not None and invQ.shape != (self.M, self.M):
            raise ValueError("invQ must be (M, M)")
        lib = _lib.load()
        self.devices = resolve_devices("all" if devices is None else devices)
        self.device = self.devices[0]
        self.has_var = invQ is not None
        self.symmetric_variance = _symmetric_choice(symmetric_variance, invQ, self.M)
        self._state = (inputs, theta, invQt, invQ)      # for the lazily built single-precision model
        self._f32_model = None
        arr = (C.c_int * len(self.devices))(*self.devices)
        h = C.c_void_p()
        check(lib.gpe_multi_create(len(self.devices), arr, self.M, self.D, addr(inputs), addr(expx), addr(invQt),
                                   addr(invQ), _lib.OPT_SYMMETRIC_VARIANCE if self.symmetric_variance else 0,
                                   C.byref(h)))
        self._own(h, lib.gpe_multi_destroy)

    def close(self):
        if self._f32_model is not None:
            self._f32_model.close()
            self._f32_model = None
        super().close()

    def predict(self, testing, want_var=True, want_deriv=True, want_hess=False, want_mu=True, out=None, pinned=None):
        """Same contract as ``DeviceModel.predict``; ``testing`` may also be a list of per-device CUDA tensors, in
        which case a list of result dicts (``None`` where there was no work) is returned."""
        D = self.D
        if want_var and not self.has_var:
            raise GpemuError("variance requested but the model was uploaded without invQ")
        flags = (WANT_MU if want_mu else 0) | (WANT_VAR if want_var else 0) | (WANT_DERIV if want_deriv else 0) | (
            WANT_HESS if want_hess else 0)
        wanted = [k for k, w in (("mu", want_mu), ("var", want_var), ("deriv", want_deriv), ("hess", want_hess)) if w]
        if isinstance(testing, (list, tuple)) or _is_torch(testing):
            return self._predict_tensors(testing, flags, wanted, out)
        t = f64c(testing)
        if t.ndim != 2 or t.shape[1] != D:
            raise ValueError(f"testing must be (N, {D})")
        N = t.shape[0]
        shapes = {"mu": (N,), "var": (N,), "deriv": (N, D), "hess": (N, D, D)}
        out = dict(out) if out else {}
        mk = _host_result_factory(pinned, N, D, [k for k in wanted if k not in out])
        for k in wanted:
            if k not in out:
                out[k] = mk(shapes[k])
            else:
                _check_out(out, k, shapes[k])
        check(_lib.load().gpe_multi_predict(self._h, addr(t), N, addr(out.get("mu")), addr(out.get("var")),
                                            addr(out.get("deriv")), addr(out.get("hess")), flags))
        return {k: out[k] for k in wanted}

    def _predict_tensors(self, testing, flags, wanted, out):
        import torch
        single = _is_torch(testing)
        G, D = len(self.devices), self.D
        per_dev = [None] * G
        if single:
            if not testing.is_cuda or testing.device.index not in self.devices:
                raise ValueError(f"torch test points must live on one of the devices {self.devices}")
            per_dev[self.devices.index(testing.device.index)] = testing
            outs = [dict(out) if (out and per_dev[g] is not None) else {} for g in range(G)]
        else:
            if len(testing) != G:
                raise ValueError(f"need one tensor (or None) per device: {G} entries")
            per_dev = list(testing)
            outs = [dict(o) if o else {} for o in (out if out else [None] * G)]
        ptrs = {k: (C.c_void_p * G)() for k in ("t", "mu", "var", "deriv", "hess", "st")}
        Ns = (C.c_int64 * G)()
        keep = []
        for g, t in enumerate(per_dev):
            if t is None or t.shape[0] == 0:
                continue
            if not t.is_cuda or t.device.index != self.devices[g] or t.dtype != torch.float64 or t.dim() != 2 \
                    or t.shape[1] != D:
                raise ValueError(f"entry {g} must be a float64 (N, {D}) tensor on cuda:{self.devices[g]}")
            t = t.contiguous()
            keep.append(t)
            n = t.shape[0]
            shapes = {"mu": (n,), "var": (n,), "deriv": (n, D), "hess": (n, D, D)}
            for k in wanted:
                if k not in outs[g]:
                    outs[g][k] = torch.empty(shapes[k], dtype=torch.float64, device=t.device)
                elif (tuple(outs[g][k].shape) != shapes[k] or outs[g][k].dtype != torch.float64
                      or outs[g][k].device != t.device or not outs[g][k].is_contiguous()):
                    raise ValueError(f"out[{k!r}] must be a contiguous float64 tensor of shape {shapes[k]} on {t.device}")
                ptrs[k][g] = outs[g][k].data_ptr()
            ptrs["t"][g] = t.data_ptr()
            Ns[g] = n
            ptrs["st"][g] = torch.cuda.current_stream(self.devices[g]).cuda_stream
        check(_lib.load().gpe_multi_predict_device(self._h, ptrs["t"], Ns, ptrs["mu"], ptrs["var"], ptrs["deriv"],
                                                   ptrs["hess"], flags, ptrs["st"]))
        res = [({k: outs[g][k] for k in wanted} if Ns[g] > 0 else None) for g in range(G)]
        if single:
            return next(r for r in res if r is not None) if any(r is not None for r in res) else \
                {k: torch.empty((0,) + ((D,) if k == "deriv" else (D, D) if k == "hess" else ()), dtype=torch.float64,
                                device=testing.device) for k in wanted}
        return res

    def predict_f32(self, testing, want_var=True, want_deriv=True, fast=None):
        """Single precision (tcgen05 path): served by one device (the first of the handle, or the tensor's own)."""
        dev = testing.device.index if _is_torch(testing) else self.devices[0]
        if self._f32_model is None or self._f32_model.device != dev:
            if self._f32_model is not None:
                self._f32_model.close()
            inputs, theta, invQt, invQ = self._state
            self._f32_model = DeviceModel(inputs, theta, invQt, invQ, device=dev)
        return self._f32_model.predict_f32(testing, want_var=want_var, want_deriv=want_deriv, fast=fast)


class DeviceBank(_Handle):
    """E GPs sharing training inputs and test points; optional PCA basis (E, W) for back-projection.

    ``device`` is one index, a list of indices or ``"all"``.  On several devices (``gpe_multi_bank_*``) host arrays are
    streamed through every GPU of the list in one call; CUDA tensors are only accepted by single-device banks."""

    def __init__(self, inputs, thetas, invQts, invQs=None, basis=None, device=0):
        inputs = f64c(inputs)
        if inputs.ndim != 2:
            raise ValueError("inputs must be (M, D)")
        self.M, self.D = inputs.shape
        thetas = f64c(thetas)
        if thetas.ndim != 2 or thetas.shape[1] < self.D + 1:
            raise ValueError("thetas must be (E, >= D+1)")
        self.E = thetas.shape[0]
        expx = f64c(np.exp(thetas[:, : self.D + 1]))
        invQts = f64c(invQts)
        if invQts.shape != (self.E, self.M):
            raise ValueError("invQts must be (E, M)")
        if invQs is not None:
            invQs = f64c(invQs)
            if invQs.shape != (self.E, self.M, self.M):
                raise ValueError("invQs must be (E, M, M)")
        self.W = 0
        if basis is not None:
            basis = f64c(basis)
            if basis.ndim != 2 or basis.shape[0] != self.E:
                raise ValueError("basis must be (E, W)")
            self.W = basis.shape[1]
        self.devices = resolve_devices(device)
        self.device = self.devices[0]
        self.multi = len(self.devices) > 1
        self.has_var = invQs is not None
        lib = _lib.load()
        h = C.c_void_p()
        if self.multi:
            arr = (C.c_int * len(self.devices))(*self.devices)
            check(lib.gpe_multi_bank_create(len(self.devices), arr, self.E, self.M, self.D, addr(inputs), addr(expx),
                                            addr(invQts), addr(invQs), addr(basis), self.W, C.byref(h)))
            self._own(h, lib.gpe_multi_destroy)
        else:
            check(lib.gpe_bank_create(self.device, self.E, self.M, self.D, addr(inputs), addr(expx),
                                      addr(invQts), addr(invQs), addr(basis), self.W, C.byref(h)))
            self._own(h, lib.gpe_bank_destroy)

    def _host_call(self, t, N, out, flags):
        lib = _lib.load()
        args = [addr(out.get(k)) for k in ("mu", "var", "deriv", "hess", "fwd", "deriv_full")]
        if self.multi:
            check(lib.gpe_multi_bank_predict(self._h, addr(t), N, *args, flags))
        else:
            check(lib.gpe_bank_predict_ex(self._h, addr(t), N, *args, flags | HOST_PTRS, None))

    def predict(self, testing, want_var=True, want_deriv=True, want_hess=False, project=False,
                project_deriv=False, want_mu=True, out=None, pinned=False):
        """Point-major outputs: mu (N, E), var (N, E), deriv (N, E, D), hess (N, E, D, D);
        with ``project``: fwd (N, W) = mu @ basis; with ``project_deriv``: deriv_full (N, D, W).

        numpy in -> numpy out: ONE library call, the chunk walk (H2D, kernels, D2H overlapped; chunks bounded by the
        width of the outputs) happens below the C ABI (``gpe_bank_predict_ex`` with host pointers), on every device of
        the bank.  ``out`` may hold preallocated (ideally page-locked) result arrays, ``pinned=True`` makes fresh ones
        page-locked.  torch CUDA in -> torch CUDA out, asynchronous on the current stream (single-device banks).
        With ``project_deriv`` the PC gradients ``deriv`` are returned too (device callers: they are its operand)."""
        D, E, W = self.D, self.E, self.W
        if want_var and not self.has_var:
            raise GpemuError("variance requested but the bank was uploaded without invQ")
        if (project or project_deriv) and W == 0:
            raise GpemuError("bank has no basis functions to project onto")
        if _is_torch(testing):
            if self.multi:
                raise ValueError("a multi-device bank takes host arrays; use one DeviceBank per device for CUDA tensors")
            import torch
            t = testing.contiguous()
            if t.dim() != 2 or t.shape[1] != D or t.dtype != torch.float64 or not t.is_cuda \
                    or t.device.index != self.device:
                raise ValueError(f"testing must be float64 (N, {D}) on cuda:{self.device}")
            return self._predict_device(t, want_var, want_deriv, want_hess, project, project_deriv)
        th = f64c(testing)
        if th.ndim != 2 or th.shape[1] != D:
            raise ValueError(f"testing must be float64 (N, {D})")
        N = th.shape[0]
        want = (("mu", want_mu, (N, E), WANT_MU), ("var", want_var, (N, E), WANT_VAR),
                ("deriv", want_deriv, (N, E, D), WANT_DERIV), ("hess", want_hess, (N, E, D, D), WANT_HESS),
                ("fwd", project, (N, W), WANT_FWD), ("deriv_full", project_deriv, (N, D, W), WANT_DERIV_FULL))
        out = dict(out) if out else {}
        res, flags = {}, 0
        mk = _pinned_empty if pinned else np.empty
        for k, w, shape, bit in want:
            if not w:
                continue
            if k in out:
                _check_out(out, k, shape)
                res[k] = out[k]
            else:
                res[k] = mk(shape)
            flags |= bit
        if not res:
            raise ValueError("no output requested")
        if N > 0:
            self._host_call(th, N, res, flags)
        return res

    def cost(self, testing, obs, weights=None, want_grad=True, want_hess=False):
        """Least-squares misfit of the bank's means against observations, reduced over the emulators on the device:
        ``cost (N,) = 1/2 sum_e w_e (mu_ne - obs_ne)^2`` and ``grad (N, D) = sum_e w_e (mu_ne - obs_ne) deriv_ned``
        (``gpe_bank_cost``).  ``obs`` is (E,) -- one observation for every point -- or (N, E); ``weights`` (E,) or None.
        ``want_hess``: also ``hess (N, D, D)``, the exact input Hessian of the cost (``gpe_bank_cost_ex``).
        numpy in -> numpy out (streamed below the C ABI, all devices of the bank); torch CUDA in -> torch CUDA out
        (asynchronous on the current stream, single-device banks).

        Per-point weights: ``weights`` may also be (N, K) -- one row per point, e.g. 1 / sigma^2 of the point's own
        uncertainties -- through the ``_pw`` entry points (include/gpemu.h, DESIGN 4.6f); rows all equal to a vector w give
        the (K,) call's results bit for bit.  A weight of 0 with a finite observation masks that entry exactly (the result
        does not depend on the observation's value); a NaN observation still gives NaN.  Data that marks gaps with NaN:
        ``weights = np.where(np.isnan(obs), 0.0, weights); obs = np.where(np.isnan(obs), 0.0, obs)``."""
        lib = _lib.load()
        return self._reduce(testing, obs, weights, want_grad, want_hess, self.E,
                            lib.gpe_multi_bank_cost_ex if self.multi else lib.gpe_bank_cost_host_ex, lib.gpe_bank_cost_ex)

    def forward_cost(self, testing, obs, weights=None, want_grad=True, want_hess=False):
        """Least-squares misfit of the back-projected spectra against observed spectra, per point:
        ``cost (N,) = 1/2 sum_w w_w (fwd_nw - obs_nw)^2`` and ``grad (N, D) = sum_w w_w (fwd_nw - obs_nw) deriv_full_ndw``
        (``gpe_bank_forward_cost``), with fwd / deriv_full those of ``predict(project=True, project_deriv=True)``.  The
        spectra never leave the kernel.  ``obs`` is (W,) -- one observed spectrum for every point -- or (N, W);
        ``weights`` (W,) or None.  ``want_hess``: also ``hess (N, D, D)``, the exact input Hessian of the cost
        (``gpe_bank_forward_cost_ex``).  numpy in -> numpy out (streamed below the C ABI, all devices of the bank); torch
        CUDA in -> torch CUDA out (asynchronous on the current stream, single-device banks).  Per-point weights (N, W)
        as in ``cost``."""
        if self.W == 0:
            raise GpemuError("bank has no basis functions to project onto")
        lib = _lib.load()
        return self._reduce(testing, obs, weights, want_grad, want_hess, self.W,
                            lib.gpe_multi_bank_forward_cost_ex if self.multi else lib.gpe_bank_forward_cost_host_ex,
                            lib.gpe_bank_forward_cost_ex)

    def _reduce(self, testing, obs, weights, want_grad, want_hess, K, host_fn, device_fn):
        """Shape checks and routing of the cost calls (observations K wide): host arrays to host_fn, CUDA tensors to
        device_fn on the current stream; per-point (N, K) weights to the ``_pw`` entry points."""
        D = self.D
        lib = _lib.load()
        flags = _lib.SOLVE_SPECTRA if device_fn is lib.gpe_bank_forward_cost_ex else 0
        if not _is_torch(testing):
            th = f64c(testing)
            if th.ndim != 2 or th.shape[1] != D:
                raise ValueError(f"testing must be float64 (N, {D})")
            N = th.shape[0]
            o = f64c(obs.cpu().numpy() if _is_torch(obs) else obs)
            if o.shape == (K,):
                obs_ld = 0
            elif o.shape == (N, K):
                obs_ld = K
            else:
                raise ValueError(f"obs must be ({K},) or ({N}, {K})")
            wt = None
            if weights is not None:
                wt = f64c(weights.cpu().numpy() if _is_torch(weights) else weights)
            w_ld = _weights_ld(None if wt is None else wt.shape, K, N)
            out = {"cost": np.empty(N)}
            if want_grad:
                out["grad"] = np.empty((N, D))
            if want_hess:
                out["hess"] = np.empty((N, D, D))
            outs = (addr(out["cost"]), addr(out.get("grad")), addr(out.get("hess")))
            if N > 0 and w_ld:
                if self.multi:
                    check(lib.gpe_multi_bank_cost_pw(self._h, addr(th), N, addr(o), obs_ld, addr(wt), w_ld, *outs, flags))
                else:
                    check(lib.gpe_bank_cost_pw(self._h, addr(th), N, addr(o), obs_ld, addr(wt), w_ld, *outs, flags | HOST_PTRS,
                                               None))
            elif N > 0:
                check(host_fn(self._h, addr(th), N, addr(o), obs_ld, addr(wt), *outs))
            return out
        if self.multi:
            raise ValueError("a multi-device bank takes host arrays; use one DeviceBank per device for CUDA tensors")
        import torch
        dev = torch.device("cuda", self.device)
        t = testing.contiguous()
        if t.dim() != 2 or t.shape[1] != D or t.dtype != torch.float64:
            raise ValueError(f"testing must be float64 (N, {D})")
        N = t.shape[0]
        o = torch.as_tensor(np.asarray(obs, dtype=np.float64) if not _is_torch(obs) else obs, dtype=torch.float64,
                            device=dev).contiguous()
        if tuple(o.shape) == (K,):
            obs_ld = 0
        elif tuple(o.shape) == (N, K):
            obs_ld = K
        else:
            raise ValueError(f"obs must be ({K},) or ({N}, {K})")
        wt = None
        if weights is not None:
            wt = torch.as_tensor(np.asarray(weights, dtype=np.float64) if not _is_torch(weights) else weights,
                                 dtype=torch.float64, device=dev).contiguous()
        w_ld = _weights_ld(None if wt is None else tuple(wt.shape), K, N)
        out = {"cost": torch.empty(N, dtype=torch.float64, device=dev)}
        if want_grad:
            out["grad"] = torch.empty(N, D, dtype=torch.float64, device=dev)
        if want_hess:
            out["hess"] = torch.empty(N, D, D, dtype=torch.float64, device=dev)
        outs = (addr(out["cost"]), addr(out.get("grad")), addr(out.get("hess")))
        if w_ld:
            check(lib.gpe_bank_cost_pw(self._h, addr(t), N, addr(o), obs_ld, addr(wt), w_ld, *outs, flags,
                                       _current_stream_ptr(self.device)))
        else:
            check(device_fn(self._h, addr(t), N, addr(o), obs_ld, addr(wt), *outs, _current_stream_ptr(self.device)))
        return out

    def search(self, candidates, obs, weights=None, k=1):
        """Per point, the ``k`` rows of the candidate table ``candidates`` (K, D) whose band cost (``cost``) against the
        point's observation is smallest: a look-up-table retrieval, or the starting points of ``invert``
        (``gpe_bank_search``).  ``obs`` is (E,) -- one point -- or (N, E); ``weights`` (E,) or None; 1 <= k <=
        min(K, ``SEARCH_MAX_K``).  Returns ``{"idx": (N, k) int64, "cost": (N, k)}``: row n lists the chosen candidates in
        ascending order of (cost, index), and ``cost`` is bit for bit the ``cost`` of those candidates against row n in a
        call of the same N points.  Candidates are ranked by the expanded form ``a_k + s_n . m_k`` of the cost, whose
        rounding may swap candidates whose costs differ by about ``E u (|a_k| + sum_e |s_ne m_ke|)`` (include/gpemu.h).
        A point with fewer than k candidates of non-NaN score gets ``idx = -1`` and ``cost = NaN`` in its last slots.
        ``weights`` may be (N, E), one row per point (``gpe_bank_search_pw``; banks of up to ``SEARCH_PW_MAX_E_BANDS`` (48)
        emulators), with the masking rules of ``cost``.
        numpy in -> numpy out (all devices of the bank); a torch CUDA tensor among ``candidates`` / ``obs`` -> torch CUDA
        out (asynchronous on the current stream, single-device banks)."""
        return self._search(False, candidates, obs, weights, k)

    def forward_search(self, candidates, obs, weights=None, k=1):
        """``search`` with the spectrum cost of ``forward_cost``: ``obs`` (W,) or (N, W), ``weights`` (W,), (N, W) or None.
        With per-point weights the search takes banks of up to ``SEARCH_PW_MAX_E_SPECTRA`` (12) emulators."""
        if self.W == 0:
            raise GpemuError("bank has no basis functions to project onto")
        return self._search(True, candidates, obs, weights, k)

    def _search(self, spectra, candidates, obs, weights, k):
        D, K_obs = self.D, (self.W if spectra else self.E)
        lib = _lib.load()
        k = int(k)
        flags = _lib.SOLVE_SPECTRA if spectra else 0
        if _is_torch(candidates) or _is_torch(obs):
            if self.multi:
                raise ValueError("a multi-device bank takes host arrays; use one DeviceBank per device for CUDA tensors")
            import torch
            tdev = torch.device("cuda", self.device)
            arr = lambda a: None if a is None else torch.as_tensor(
                a if _is_torch(a) else np.asarray(a, dtype=np.float64), dtype=torch.float64, device=tdev).contiguous()
            c, o, wt = arr(candidates), arr(obs), arr(weights)
            shape = lambda a: tuple(a.shape)
            empty = lambda s, dt: torch.empty(s, dtype=torch.int64 if dt is np.int64 else torch.float64, device=tdev)
        else:
            arr = lambda a: None if a is None else f64c(a.cpu().numpy() if _is_torch(a) else a)
            c, o, wt = arr(candidates), arr(obs), arr(weights)
            shape = lambda a: a.shape
            empty = lambda s, dt: np.empty(s, dtype=dt)
        if len(shape(c)) != 2 or shape(c)[1] != D:
            raise ValueError(f"candidates must be (K, {D})")
        if shape(o) == (K_obs,):
            N, obs_ld = 1, 0
        elif len(shape(o)) == 2 and shape(o)[1] == K_obs:
            N, obs_ld = shape(o)[0], K_obs
        else:
            raise ValueError(f"obs must be ({K_obs},) or (N, {K_obs})")
        w_ld = _weights_ld(None if wt is None else shape(wt), K_obs, N)
        out = {"idx": empty((N, k), np.int64), "cost": empty((N, k), np.float64)}
        if w_ld:
            args = (addr(c), shape(c)[0], addr(o), N, obs_ld, addr(wt), w_ld, k, addr(out["idx"]), addr(out["cost"]))
            if _is_torch(c):
                check(lib.gpe_bank_search_pw(self._h, *args, flags, _current_stream_ptr(self.device)))
            elif self.multi:
                check(lib.gpe_multi_bank_search_pw(self._h, *args, flags))
            else:
                check(lib.gpe_bank_search_pw(self._h, *args, flags | HOST_PTRS, None))
            return out
        args = (addr(c), shape(c)[0], addr(o), N, obs_ld, addr(wt), k, addr(out["idx"]), addr(out["cost"]))
        if _is_torch(c):
            check(lib.gpe_bank_search(self._h, *args, flags, _current_stream_ptr(self.device)))
        elif self.multi:
            check(lib.gpe_multi_bank_search(self._h, *args, flags))
        else:
            check(lib.gpe_bank_search(self._h, *args, flags | HOST_PTRS, None))
        return out

    def invert(self, x0, obs, weights=None, lower=None, upper=None, prior_mean=None, prior_precision=None,
               max_iter=_lib.SOLVE_DEFAULT_MAX_ITER, ftol=1e-10, xtol=1e-10, gtol=0.0, lambda0=1e-3, want_cov=False,
               candidates=None, n_starts=1):
        """Per point, the inputs that minimise the band cost of ``cost`` plus an optional Gaussian prior,
        ``f(x) = cost(x) + 1/2 (x - prior_mean)^T prior_precision (x - prior_mean)``, inside the box ``lower <= x <= upper``:
        bounded Levenberg-Marquardt on the exact Hessian, every iteration on the device (``gpe_bank_solve``; the
        algorithm and the stopping tests are stated in include/gpemu.h).

        ``x0`` (N, D) starting points; ``obs`` (E,) or (N, E); ``weights`` (E,), (N, E) or None (per-point rows as in
        ``cost``: ``gpe_bank_solve_pw``, and with 1 / sigma^2 of each point ``cov`` is its Laplace posterior); ``lower`` / ``upper`` (D,) or
        None (entries may be infinite); ``prior_mean`` (D,) or (N, D), ``prior_precision`` (D, D).  Returns a dict:
        ``x`` (N, D), ``cost`` (N,), ``grad`` (N, D) and ``hess`` (N, D, D) at x (prior included), ``cov`` (N, D, D) =
        inv(hess) with ``want_cov`` (NaN where hess is not positive definite), ``status`` (N,) int32 (``SOLVE_*`` of
        ``_lib``) and ``n_iter`` (N,) int32, the evaluations after the first.  numpy in -> numpy out (all devices of the
        bank); torch CUDA in -> torch CUDA out (single-device banks; the call returns when the results are written).

        Starting points from a candidate table: with ``x0=None`` and ``candidates`` (K, D), the ``n_starts`` best
        candidates of each point (``search``) are each solved from, and each point keeps the result of the lowest returned
        cost (prior included; ties go to the better-ranked start, NaN loses).  ``candidate`` (N,) int64 is then added: the
        index of the winning start in ``candidates``.  A point without a candidate of non-NaN score comes back with status
        ``SOLVE_NONFINITE``, NaN x and ``n_iter`` 0.  With ``n_starts=1`` the result is that of
        ``invert(candidates[idx[:, 0]], ...)``, bit for bit."""
        return self._solve(False, x0, obs, weights, lower, upper, prior_mean, prior_precision, max_iter, ftol, xtol, gtol,
                           lambda0, want_cov, candidates, n_starts)

    def forward_invert(self, x0, obs, weights=None, lower=None, upper=None, prior_mean=None, prior_precision=None,
                       max_iter=_lib.SOLVE_DEFAULT_MAX_ITER, ftol=1e-10, xtol=1e-10, gtol=0.0, lambda0=1e-3,
                       want_cov=False, candidates=None, n_starts=1):
        """``invert`` with the spectrum cost of ``forward_cost``: ``obs`` (W,) or (N, W), ``weights`` (W,) or None; the
        starts from ``candidates`` are chosen by ``forward_search``."""
        if self.W == 0:
            raise GpemuError("bank has no basis functions to project onto")
        return self._solve(True, x0, obs, weights, lower, upper, prior_mean, prior_precision, max_iter, ftol, xtol, gtol,
                           lambda0, want_cov, candidates, n_starts)

    def invert_series(self, x0, obs, weights=None, smooth_precision=None, coupling=None, lower=None, upper=None,
                      prior_mean=None, prior_precision=None, max_iter=_lib.SOLVE_DEFAULT_MAX_ITER, ftol=1e-10, xtol=1e-10,
                      gtol=0.0, lambda0=1e-3, want_cov=False):
        """Per series of T dates, the inputs that minimise the summed band cost of ``cost`` plus the optional Gaussian
        prior of ``invert`` on every date plus a temporal smoothness prior,
        ``1/2 sum_t coupling[t-1] (x_t - x_t-1)^T smooth_precision (x_t - x_t-1)``, inside the box: the Levenberg-Marquardt
        of ``invert`` on the block-tridiagonal Hessian of the whole series, every iteration on the device
        (``gpe_bank_solve_series``; the objective and the algorithm are stated in include/gpemu.h).

        ``x0`` (S, T, D) or (T, D) for one series; ``obs`` (E,) or (S, T, E); ``weights`` (E,), (S, T, E) or None -- a date
        whose weights are all 0 is masked and filled in by the smoothness prior; ``smooth_precision`` (D, D) symmetric PSD,
        required; ``coupling`` (T - 1,) >= 0 or None (all 1): with 1 / (days between dates) the prior is a random walk over
        irregular dates, a 0 cuts the chain; ``prior_mean`` (D,) or (S, T, D); the other arguments as ``invert``.  Returns
        ``x`` and ``grad`` (S, T, D), ``hess`` (S, T, D, D) the diagonal blocks of the Hessian (the off-diagonal ones are
        ``-coupling[t-1] smooth_precision``), ``cov`` (S, T, D, D) the diagonal blocks of its inverse with ``want_cov``,
        ``cost``, ``status`` and ``n_iter`` (S,) -- without the leading S (scalars for the last three) for one series.
        numpy in -> numpy out (all devices of the bank); torch CUDA in -> torch CUDA out (single-device banks)."""
        if smooth_precision is None:
            raise ValueError("smooth_precision (D, D) is required")
        return self._solve(False, x0, obs, weights, lower, upper, prior_mean, prior_precision, max_iter, ftol, xtol, gtol,
                           lambda0, want_cov, series=(smooth_precision, coupling))

    def forward_invert_series(self, x0, obs, weights=None, smooth_precision=None, coupling=None, lower=None, upper=None,
                              prior_mean=None, prior_precision=None, max_iter=_lib.SOLVE_DEFAULT_MAX_ITER, ftol=1e-10,
                              xtol=1e-10, gtol=0.0, lambda0=1e-3, want_cov=False):
        """``invert_series`` with the spectrum cost of ``forward_cost``: ``obs`` (W,) or (S, T, W), ``weights`` (W,),
        (S, T, W) or None."""
        if self.W == 0:
            raise GpemuError("bank has no basis functions to project onto")
        if smooth_precision is None:
            raise ValueError("smooth_precision (D, D) is required")
        return self._solve(True, x0, obs, weights, lower, upper, prior_mean, prior_precision, max_iter, ftol, xtol, gtol,
                           lambda0, want_cov, series=(smooth_precision, coupling))

    def _solve_from_candidates(self, spectra, candidates, n_starts, obs, weights, solve):
        """Multi-start solve: ``solve(x0)`` from each of the ``n_starts`` best candidates, the best result per point."""
        found = self._search(spectra, candidates, obs, weights, n_starts)
        idx = found["idx"]
        if _is_torch(idx):
            import torch
            cand = torch.as_tensor(candidates if _is_torch(candidates) else np.asarray(candidates, dtype=np.float64),
                                   dtype=torch.float64, device=idx.device)
            where = lambda m, a, b: torch.where(m.reshape(m.shape + (1,) * (a.dim() - 1)), a, b)
            isnan = torch.isnan
        else:
            cand = f64c(candidates.cpu().numpy() if _is_torch(candidates) else candidates)
            where = lambda m, a, b: np.where(m.reshape(m.shape + (1,) * (a.ndim - 1)), a, b)
            isnan = np.isnan
        best, win = None, None
        for j in range(int(n_starts)):
            ij = idx[:, j]
            res = solve(cand[ij.clip(min=0) if _is_torch(ij) else np.clip(ij, 0, None)])
            if best is None:
                best, win = res, ij
                continue
            c, bc = res["cost"], best["cost"]
            take = (ij >= 0) & ((c < bc) | (isnan(bc) & ~isnan(c)))
            best = {key: where(take, res[key], best[key]) for key in best}
            win = where(take, ij, win)
        none = idx[:, 0] < 0
        if bool(none.any()):
            for key, v in best.items():
                if key == "status":
                    best[key] = where(none, v * 0 + _lib.SOLVE_NONFINITE, v)
                elif key == "n_iter":
                    best[key] = where(none, v * 0, v)
                else:
                    best[key] = where(none, v * float("nan"), v)
        best["candidate"] = win
        return best

    def _solve(self, spectra, x0, obs, weights, lower, upper, prior_mean, prior_precision, max_iter, ftol, xtol, gtol,
               lambda0, want_cov, candidates=None, n_starts=1, series=None):
        if x0 is None:
            if candidates is None:
                raise ValueError("give the starting points x0 or a candidate table")
            return self._solve_from_candidates(
                spectra, candidates, n_starts, obs, weights,
                lambda s: self._solve(spectra, s, obs, weights, lower, upper, prior_mean, prior_precision, max_iter, ftol,
                                      xtol, gtol, lambda0, want_cov))
        if candidates is not None:
            raise ValueError("give x0 or candidates, not both")
        D, K = self.D, (self.W if spectra else self.E)
        lib = _lib.load()
        dev = _is_torch(x0)
        if dev:
            if self.multi:
                raise ValueError("a multi-device bank takes host arrays; use one DeviceBank per device for CUDA tensors")
            import torch
            tdev = torch.device("cuda", self.device)
            arr = lambda a: None if a is None else torch.as_tensor(
                a if _is_torch(a) else np.asarray(a, dtype=np.float64), dtype=torch.float64, device=tdev).contiguous()
            shape = lambda a: tuple(a.shape)
            empty = lambda *s: torch.empty(*s, dtype=torch.float64, device=tdev)
            info_empty = lambda n: torch.empty(n, 2, dtype=torch.int32, device=tdev)
        else:
            arr = lambda a: None if a is None else f64c(a.cpu().numpy() if _is_torch(a) else a)
            shape = lambda a: a.shape
            empty = np.empty
            info_empty = lambda n: np.empty((n, 2), dtype=np.int32)
        x0 = arr(x0)
        if series is not None:
            # series: the (S, T, ...) arrays become rows n = s T + t of the point solver's arguments
            if len(shape(x0)) == 3 and shape(x0)[2] == D:
                lead = tuple(shape(x0)[:2])
            elif len(shape(x0)) == 2 and shape(x0)[1] == D:
                lead = (shape(x0)[0],)
            else:
                raise ValueError(f"x0 must be (S, T, {D}) or (T, {D})")
            S, T = (lead[0], lead[1]) if len(lead) == 2 else (1, lead[0])
            rows = lambda a, w: a.reshape(S * T, w) if a is not None and tuple(shape(a)) == lead + (w,) else a
            x0, obs, weights, prior_mean = rows(x0, D), rows(arr(obs), K), rows(arr(weights), K), rows(arr(prior_mean), D)
            smooth, cpl = arr(series[0]), arr(series[1])
            if shape(smooth) != (D, D):
                raise ValueError(f"smooth_precision must be ({D}, {D})")
            if cpl is not None and shape(cpl) != (T - 1,):
                raise ValueError(f"coupling must be ({T - 1},)")
        if len(shape(x0)) != 2 or shape(x0)[1] != D:
            raise ValueError(f"x0 must be (N, {D})")
        N = shape(x0)[0]
        o = arr(obs)
        if shape(o) == (K,):
            obs_ld = 0
        elif shape(o) == (N, K):
            obs_ld = K
        else:
            raise ValueError(f"obs must be ({K},) or ({N}, {K})")
        wt, lo, hi, pm, pp = (arr(a) for a in (weights, lower, upper, prior_mean, prior_precision))
        w_ld = _weights_ld(None if wt is None else shape(wt), K, N)
        for name, a, want in (("lower", lo, (D,)), ("upper", hi, (D,)), ("prior_precision", pp, (D, D))):
            if a is not None and shape(a) != want:
                raise ValueError(f"{name} must be {want}")
        prior_ld = 0
        if pm is not None:
            if shape(pm) == (N, D):
                prior_ld = D
            elif shape(pm) != (D,):
                raise ValueError(f"prior_mean must be ({D},) or ({N}, {D})")
        opts = _lib.SolveOpts(int(max_iter), float(ftol), float(xtol), float(gtol), float(lambda0), addr(lo), addr(hi),
                              addr(pm), prior_ld, addr(pp))
        n_out = N if series is None else S
        out = {"x": empty((N, D)), "cost": empty(n_out), "grad": empty((N, D)), "hess": empty((N, D, D))}
        if want_cov:
            out["cov"] = empty((N, D, D))
        info = info_empty(n_out)
        flags = _lib.SOLVE_SPECTRA if spectra else 0
        args = (addr(x0), N, addr(o), obs_ld, addr(wt), C.byref(opts), addr(out["x"]), addr(out["cost"]),
                addr(out["grad"]), addr(out["hess"]), addr(out.get("cov")), addr(info))
        if series is not None:
            args = (S, T, addr(x0), addr(o), obs_ld, addr(wt), w_ld, C.byref(opts), addr(smooth), addr(cpl)) + args[6:]
            if dev:
                check(lib.gpe_bank_solve_series(self._h, *args, flags, _current_stream_ptr(self.device)))
            elif self.multi:
                check(lib.gpe_multi_bank_solve_series(self._h, *args, flags))
            else:
                check(lib.gpe_bank_solve_series(self._h, *args, flags | HOST_PTRS, None))
            out["status"], out["n_iter"] = info[:, 0], info[:, 1]
            one = len(lead) == 1
            for key in ("x", "grad", "hess", "cov"):
                if key in out:
                    out[key] = out[key].reshape(lead + tuple(shape(out[key])[1:]))
            if one:
                for key in ("cost", "status", "n_iter"):
                    out[key] = out[key][0]
            return out
        if w_ld:
            args = args[:5] + (w_ld,) + args[5:]
            if dev:
                check(lib.gpe_bank_solve_pw(self._h, *args, flags, _current_stream_ptr(self.device)))
            elif self.multi:
                check(lib.gpe_multi_bank_solve_pw(self._h, *args, flags))
            else:
                check(lib.gpe_bank_solve_pw(self._h, *args, flags | HOST_PTRS, None))
        elif dev:
            check(lib.gpe_bank_solve(self._h, *args, flags, _current_stream_ptr(self.device)))
        elif self.multi:
            check(lib.gpe_multi_bank_solve(self._h, *args, flags))
        else:
            check(lib.gpe_bank_solve(self._h, *args, flags | HOST_PTRS, None))
        out["status"], out["n_iter"] = info[:, 0], info[:, 1]
        return out

    def forward(self, testing, want_deriv=True):
        """numpy (N, D) -> fwd (N, W) [, deriv_full (N, D, W)]: one call, nothing but the spectra (and Jacobians)
        crosses PCIe.  This is what ``MultivariateEmulator.predict`` (reference multivariate_gp.py:195-222) runs on."""
        res = self.predict(testing, want_var=False, want_deriv=False, want_mu=False, project=True,
                           project_deriv=want_deriv)
        return (res["fwd"], res["deriv_full"]) if want_deriv else res["fwd"]

    def _predict_device(self, t, want_var, want_deriv, want_hess, project, project_deriv):
        import torch
        lib = _lib.load()
        D, E = self.D, self.E
        dev = t.device
        N = t.shape[0]
        mk = lambda *s: torch.empty(*s, dtype=torch.float64, device=dev)
        out = {"mu": mk(N, E)}
        flags = WANT_MU
        if want_var: out["var"] = mk(N, E); flags |= WANT_VAR
        if want_deriv or project_deriv: out["deriv"] = mk(N, E, D); flags |= WANT_DERIV
        if want_hess: out["hess"] = mk(N, E, D, D); flags |= WANT_HESS
        if project: out["fwd"] = mk(N, self.W); flags |= WANT_FWD
        if project_deriv: out["deriv_full"] = mk(N, D, self.W); flags |= WANT_DERIV_FULL
        check(lib.gpe_bank_predict_ex(self._h, addr(t), N, addr(out["mu"]), addr(out.get("var")),
                                      addr(out.get("deriv")), addr(out.get("hess")), addr(out.get("fwd")),
                                      addr(out.get("deriv_full")), flags, _current_stream_ptr(self.device)))
        return out
