"""
Device-resident RV model: the B200 replacement for ``evidence.rvmodel`` on the likelihood hot
path.  Same constructor, attributes and scalar protocol as the reference classes
(evidence/rvmodel/__init__.py:10-80 ``BaseModel``, :84-219 ``RVModel``), plus the batched entry
points the vectorised samplers call:

    model = RVModel(fixedpardict, datadict, parnames)        # same arguments as the reference
    model.log_likelihood(x)              -> float            # scalar protocol (batch of 1)
    model.log_likelihood_batch(X[B,ndim]) -> ndarray[B]      # one launch for the whole batch
    model.set_priors(priordict); model.prior_transform_batch(U); model.transform_loglike_batch(U)
    model.log_likelihood_device(theta_cuda_tensor) -> cuda tensor   # no host round trip

All arithmetic runs in hand-written sm_100a CUDA behind the C-ABI of include/rvlnl.h
(evidence_b200/csrc/rvlnl.cu).  There is no CPU fallback.
"""
import ctypes
from ctypes import POINTER, byref, c_double, c_int32, c_uint64, c_void_p

import numpy as np

from . import _abi
from .layout import compile_model

_dp = POINTER(c_double)


class DeviceError(RuntimeError):
    pass


def _ptr(a):
    return a.ctypes.data_as(_dp)


class BaseModel(object):
    """
    Mirrors evidence/rvmodel/__init__.py:10-57: keeps ``fixedpardict``, the SORTED ``parnames``
    (:43), the instrument list (:46) and the concatenated data with an ``inst_id`` column
    (:50-55).  ``datadict[inst]['data']`` may be a pandas DataFrame (what ``config.read_data``
    produces, evidence/config.py:102-114) or any mapping of column name -> array.
    """

    def __init__(self, fixedpardict, datadict, parnames):
        self.fixedpardict = fixedpardict
        self.parnames = sorted(parnames)
        self.insts = list(datadict.keys())
        self.datadict = datadict
        cols = {}
        ids = []
        for i, instrument in enumerate(self.insts):
            tab = datadict[instrument]["data"]
            n = len(tab[_first_key(tab)])
            try:  # the reference adds the id column to the caller's frame too (:52)
                tab["inst_id"] = np.zeros(n, dtype=int) + i
            except Exception:
                pass
            for key in _keys(tab):
                if key == "inst_id":
                    continue
                cols.setdefault(key, []).append(np.asarray(tab[key]))
            ids.append(np.zeros(n, dtype=np.int32) + i)
        self._columns = {k: np.concatenate(v) for k, v in cols.items()
                         if len(v) == len(self.insts)}
        self._inst_id = np.concatenate(ids) if ids else np.zeros(0, dtype=np.int32)
        try:
            import pandas as pd
            frame = dict(self._columns)
            frame["inst_id"] = self._inst_id
            self.data = pd.DataFrame(frame)
        except ImportError:  # pandas is only needed for the reference-compatible .data view
            self.data = dict(self._columns, inst_id=self._inst_id)

    def logL(self, residuals, var):
        """Host helper kept for custom post-processing (evidence/rvmodel/__init__.py:59-80)."""
        n = len(residuals)
        cte = -0.5 * n * np.log(2 * np.pi)
        return cte - np.sum(np.log(np.sqrt(var))) - np.sum(residuals ** 2 / (2 * var))


def _keys(tab):
    return list(tab.columns) if hasattr(tab, "columns") else list(tab.keys())


# ---------------------------------------------------------------------- model curves: host logic
# Output of one rvl_kepler_rv call is capped: larger requests are cut into row chunks.
CURVE_CHUNK_BYTES = 256 << 20


def planet_mask(nplanets, planets=None, exclude=None):
    """Bit mask (bit p = planet p + 1) of the planets to sum: ``planets`` (a planet number 1..K or
    an iterable of them; None = all) minus ``exclude`` (the same forms)."""
    def numbers(sel, what):
        if sel is None:
            return []
        sel = [sel] if np.ndim(sel) == 0 else list(sel)
        out = []
        for k in sel:
            if int(k) != k or not 1 <= int(k) <= nplanets:
                raise ValueError(f"{what}: {k!r} is not a planet number in 1..{nplanets}")
            out.append(int(k))
        return out
    chosen = range(1, nplanets + 1) if planets is None else numbers(planets, "planets")
    mask = 0
    for k in chosen:
        mask |= 1 << (k - 1)
    for k in numbers(exclude, "exclude_planet"):
        mask &= ~(1 << (k - 1))
    return mask


def curve_chunks(B, T, max_bytes=CURVE_CHUNK_BYTES):
    """Row ranges [lo, hi) that cut a [B, T] float64 output into pieces of at most ``max_bytes``
    (at least one row each)."""
    rows = max(1, max_bytes // (8 * T)) if T > 0 else max(1, B)
    return [(lo, min(B, lo + rows)) for lo in range(0, B, rows)]


def planet_param_names(desc, k):
    """(name, rvl_param) of every quantity that planet ``k`` (1-based) of a compiled
    ``rvl_model_desc`` reads, in modelk's parametrisation (evidence/rvmodel/__init__.py:411-456)."""
    pl = desc.planet[k - 1]
    pre = f"planet{k}_"
    e_names = {_abi.RVL_ECC_SECOS_SESIN: ("secos", "sesin"), _abi.RVL_ECC_ECOS_ESIN: ("ecos", "esin"),
               _abi.RVL_ECC_DIRECT: ("ecc", "omega")}[pl.ecc_mode]
    return [(pre + ("logk1" if pl.amp_is_log else "k1"), pl.amp),
            (pre + ("logperiod" if pl.period_is_log else "period"), pl.period),
            (pre + e_names[0], pl.e1), (pre + e_names[1], pl.e2),
            (pre + ("ml0" if pl.phase_mode == _abi.RVL_PHASE_ML0 else "ma0"), pl.phase),
            (pre + "epoch", pl.epoch)]


def pardict_row(pardict, parnames, desc, mask):
    """
    theta row (sorted ``parnames`` order) for a reference-style ``pardict``, for the planets in
    ``mask``.  Free names come from ``pardict``; a free name that none of those planets reads may be
    missing and is filled with 0 (it cannot reach their velocities).  A missing free name that they
    read raises KeyError, as the reference's lookup would.  The device model was compiled with the
    fixed values, so a fixed name they read whose ``pardict`` value differs raises ValueError.
    """
    row = np.zeros(len(parnames), dtype=np.float64)
    used = set()
    for k in range(1, desc.n_planets + 1):
        if not (mask >> (k - 1)) & 1:
            continue
        for name, par in planet_param_names(desc, k):
            if par.slot >= 0:
                used.add(par.slot)
            elif name in pardict and float(pardict[name]) != par.value:
                raise ValueError(f"{name} = {pardict[name]!r} differs from the model's fixed value "
                                 f"{par.value!r}")
    for i, name in enumerate(parnames):
        if name in pardict:
            row[i] = float(pardict[name])
        elif i in used:
            raise KeyError(name)
    return row


def host_drift(pardict, time):
    """RVModel.drift (evidence/rvmodel/__init__.py:222-273) on the host, the reference's own
    elementwise numpy arithmetic: lin*tt + quad*tt**2 + cub*tt**3 + quar*tt**4 with
    tt = (time - tref)/365.25, tref = pardict['drift_tref'] if present, else time[0] of ``time``."""
    time = np.asarray(time, dtype=np.float64)
    lin = pardict.get("drift_lin", 0.0)
    quad = pardict.get("drift_quad", 0.0)
    cub = pardict.get("drift_cub", 0.0)
    quar = pardict.get("drift_quar", 0.0)
    tref = pardict["drift_tref"] if "drift_tref" in pardict else time[0]
    tt = (time - tref) / 365.25
    return lin * tt + quad * tt ** 2 + cub * tt ** 3 + quar * tt ** 4


def _first_key(tab):
    return _keys(tab)[0]


class RVModel(BaseModel):
    """
    Drop-in for evidence.rvmodel.RVModel whose likelihood runs on a B200.

    Extra keyword arguments (all optional): ``device`` (CUDA device index, default: current),
    ``devices`` (a list of device indices, or ``"all"``: ONE model over several GPUs of the box --
    ``rvl_create_multi``; every host-buffer batch call then splits its rows over them),
    ``linpar_dict`` (name -> per-epoch array, the reference's ``self.linpar_dict``,
    evidence/rvmodel/__init__.py:131-136, 210-212), ``tol`` / ``itmax`` (Newton tolerance and
    cap; the reference hard-codes 1e-4 and 10000, :466, :491).
    """

    def __init__(self, fixedpardict, datadict, parnames, device=None, linpar_dict=None,
                 tol=1.0e-4, itmax=10000, devices=None):
        super().__init__(fixedpardict, datadict, parnames)
        # structure from the free names only (:118-139)
        self.nplanets = sum("k1" in p for p in self.parnames)
        self.drift_in_model = any("drift" in p for p in self.parnames)
        self.linpar_in_model = any("linpar" in p for p in self.parnames)
        self.jitter_in_model = any("jitter" in p for p in self.parnames)
        self.linpar_dict = dict(linpar_dict or {}) if self.linpar_in_model else {}

        tkey = "rjd" if "rjd" in self._columns else "jdb"  # :141-144
        self.time = np.ascontiguousarray(self._columns[tkey], dtype=np.float64).copy()
        self.vrad = np.ascontiguousarray(self._columns["vrad"], dtype=np.float64).copy()
        self.svrad = np.ascontiguousarray(self._columns["svrad"], dtype=np.float64).copy()
        self.ndim = len(self.parnames)

        self._desc, _ = compile_model(self.parnames, self.fixedpardict, self.insts,
                                      self.time[0] if len(self.time) else 0.0,
                                      linpar_names=list(self.linpar_dict.keys()),
                                      tol=tol, itmax=itmax)
        self._lib = _abi.load()
        self._h = c_void_p()
        self.device_index = None if device is None else int(device)  # None: the current device
        if devices is not None:
            if device is not None:
                raise ValueError("give either device or devices")
            devs = [] if devices == "all" else [int(d) for d in devices]
            arr = (c_int32 * max(1, len(devs)))(*devs)
            rc = self._lib.rvl_create_multi(byref(self._h), arr if devs else None, len(devs))
        else:
            rc = self._lib.rvl_create(byref(self._h), -1 if device is None else int(device))
        if rc != 0:
            msg = self._lib.rvl_last_error(None).decode()
            raise DeviceError(f"rvl_create failed ({_abi.RVL_ERRORS.get(rc, rc)}): {msg}")
        ids = np.ascontiguousarray(self._inst_id, dtype=np.int32)
        self._check(self._lib.rvl_set_data(self._h, _ptr(self.time), _ptr(self.vrad),
                                           _ptr(self.svrad),
                                           ids.ctypes.data_as(POINTER(c_int32)),
                                           len(self.time), len(self.insts)))
        for j, name in enumerate(self.linpar_dict):
            col = np.ascontiguousarray(self.linpar_dict[name], dtype=np.float64)
            self._check(self._lib.rvl_set_linpar(self._h, j, _ptr(col), len(col)))
        self._check(self._lib.rvl_set_model(self._h, byref(self._desc)))
        self._priors_set = False
        self._one_in = np.empty((1, max(1, self.ndim)), dtype=np.float64)
        self._one_out = np.empty(1, dtype=np.float64)

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc):
        if rc != 0:
            msg = self._lib.rvl_last_error(self._h).decode()
            raise DeviceError(f"librvlnl: {_abi.RVL_ERRORS.get(rc, rc)}: {msg}")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.rvl_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name, value):
        self._check(self._lib.rvl_set_option(self._h, name.encode(), int(value)))

    def desc_bytes(self):
        """Raw bytes of the compiled ``rvl_model_desc`` (tests feed them to the C checker)."""
        return bytes(self._desc)

    def _as_batch(self, X, what):
        X = np.ascontiguousarray(X, dtype=np.float64)
        if X.ndim == 1:
            X = X.reshape(1, -1)
        if X.ndim != 2 or X.shape[1] != self.ndim:
            raise ValueError(f"{what} must have shape (B, {self.ndim}), got {X.shape}")
        return X

    # ------------------------------------------------------------------ likelihood
    def log_likelihood(self, x):
        """Scalar protocol of the reference (evidence/rvmodel/__init__.py:157-219): batch of 1."""
        self._one_in[0, :self.ndim] = x
        self._check(self._lib.rvl_loglike(self._h, _ptr(self._one_in), 1, _ptr(self._one_out)))
        return float(self._one_out[0])

    def log_likelihood_batch(self, X, out=None):
        """lnL for every row of ``X`` (theta in sorted-parnames order); one kernel launch."""
        if not (type(X) is np.ndarray and X.dtype == np.float64 and X.ndim == 2
                and X.shape[1] == self.ndim and X.flags.c_contiguous):
            X = self._as_batch(X, "X")  # (the usual case above skips the conversions)
        B = X.shape[0]
        if out is None:
            out = np.empty(B, dtype=np.float64)
        elif not (out.dtype == np.float64 and out.flags.c_contiguous and out.size >= B):
            raise ValueError("out must be a C-contiguous float64 array with at least B elements")
        rc = self._lib.rvl_loglike(self._h, X.ctypes.data, B, out.ctypes.data)
        if rc != 0:
            self._check(rc)
        return out

    def log_likelihood_device(self, theta, out=None):
        """
        lnL for a CUDA float64 tensor ``theta[B, ndim]`` without leaving the device; enqueued on
        torch's current stream.
        """
        import torch
        if not (theta.is_cuda and theta.dtype == torch.float64 and theta.is_contiguous()):
            raise ValueError("theta must be a contiguous CUDA float64 tensor")
        if theta.dim() != 2 or theta.shape[1] != self.ndim:
            raise ValueError(f"theta must have shape (B, {self.ndim})")
        B = theta.shape[0]
        if out is None:
            out = torch.empty(B, dtype=torch.float64, device=theta.device)
        stream = torch.cuda.current_stream(theta.device).cuda_stream
        self._check(self._lib.rvl_loglike_dev(self._h, c_void_p(theta.data_ptr()), B,
                                              c_void_p(out.data_ptr()), c_void_p(stream)))
        return out

    def log_likelihood_device_scatter(self, theta, out, peer_ptrs, offset):
        """
        ``log_likelihood_device`` whose producing kernel also stores lnL into the peer-mapped
        buffers ``peer_ptrs`` (device addresses, e.g. torch symmetric memory ``buffer_ptrs``) at
        element ``offset``: the all-gather of the multi-GPU path without a separate collective.
        """
        import torch
        if not (theta.is_cuda and theta.dtype == torch.float64 and theta.is_contiguous()):
            raise ValueError("theta must be a contiguous CUDA float64 tensor")
        B = theta.shape[0]
        arr = (c_uint64 * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
        stream = torch.cuda.current_stream(theta.device).cuda_stream
        self._check(self._lib.rvl_loglike_dev_scatter(
            self._h, c_void_p(theta.data_ptr()), B, c_void_p(out.data_ptr()), arr, len(peer_ptrs),
            int(offset), c_void_p(stream)))
        return out

    def log_likelihood_device_gather(self, theta, out, peer_ptrs, rank, offset, flag_offset, seq):
        """
        The all-gather inside the likelihood launch (``rvl_loglike_dev_gather``): lnL goes into every
        peer buffer at element ``offset``, the finished launch stores ``seq`` into completion slot
        ``flag_offset + rank`` of every peer buffer, and a one-warp kernel behind it waits for all
        ranks' slots of this rank's own buffer.  Stream-ordered; no barrier, no collective.
        """
        import torch
        if not (theta.is_cuda and theta.dtype == torch.float64 and theta.is_contiguous()):
            raise ValueError("theta must be a contiguous CUDA float64 tensor")
        B = theta.shape[0]
        arr = (c_uint64 * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
        stream = torch.cuda.current_stream(theta.device).cuda_stream
        self._check(self._lib.rvl_loglike_dev_gather(
            self._h, c_void_p(theta.data_ptr()), B, c_void_p(out.data_ptr()), arr, len(peer_ptrs),
            int(rank), int(offset), int(flag_offset), int(seq), c_void_p(stream)))
        return out

    def log_likelihood_gather_host(self, X, out_all, peer_ptrs, rank, flag_offset, seq):
        """
        Per-rank host-buffer form of the fused all-gather (``rvl_loglike_gather``): this rank's rows
        ``X[B, ndim]`` (host, ideally page-locked) in, ``out_all[world * B]`` (host) = lnL of all
        ranks out.  One synchronous call per step.
        """
        B = X.shape[0]
        arr = (c_uint64 * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
        rc = self._lib.rvl_loglike_gather(self._h, X.ctypes.data, B, out_all.ctypes.data, arr,
                                          len(peer_ptrs), int(rank), int(flag_offset), int(seq))
        if rc != 0:
            self._check(rc)
        return out_all

    def device_count(self):
        n = c_int32()
        self._check(self._lib.rvl_device_count(self._h, byref(n)))
        return n.value

    def reset(self):
        """Re-arm the handle after a faulted launch (``rvl_reset``)."""
        self._check(self._lib.rvl_reset(self._h))

    # ------------------------------------------------------------------ priors
    def set_priors(self, priordict):
        """
        Stage the unit-cube transform of ``priordict`` (name -> prior, as built by
        ``evidence_b200.priors.prior_constructor``) in sorted-parnames order
        (evidence/ultranest/__init__.py:132-135).
        """
        from .priors import device_descriptors
        descs, tables = device_descriptors([priordict[p] for p in self.parnames])
        arr = (_abi.rvl_prior_desc * len(descs))(*descs)
        tptr = _ptr(tables) if tables.size else None
        self._check(self._lib.rvl_set_priors(self._h, arr, len(descs), tptr, tables.size))
        self._priors_set = True

    def prior_transform_batch(self, U):
        U = self._as_batch(U, "U")
        theta = np.empty_like(U)
        self._check(self._lib.rvl_transform(self._h, _ptr(U), U.shape[0], _ptr(theta)))
        return theta

    def transform_loglike_batch(self, U, return_theta=True):
        """Fused u -> theta -> lnL for a batch of unit-cube points."""
        U = self._as_batch(U, "U")
        B = U.shape[0]
        lnl = np.empty(B, dtype=np.float64)
        theta = np.empty_like(U) if return_theta else None
        self._check(self._lib.rvl_transform_loglike(
            self._h, _ptr(U), B, _ptr(theta) if return_theta else None, _ptr(lnl)))
        return (theta, lnl) if return_theta else lnl

    def transform_loglike_device(self, U, theta=None, lnl=None):
        import torch
        if not (U.is_cuda and U.dtype == torch.float64 and U.is_contiguous()):
            raise ValueError("U must be a contiguous CUDA float64 tensor")
        B = U.shape[0]
        if theta is None:
            theta = torch.empty_like(U)
        if lnl is None:
            lnl = torch.empty(B, dtype=torch.float64, device=U.device)
        stream = torch.cuda.current_stream(U.device).cuda_stream
        self._check(self._lib.rvl_transform_loglike_dev(
            self._h, c_void_p(U.data_ptr()), B, c_void_p(theta.data_ptr()),
            c_void_p(lnl.data_ptr()), c_void_p(stream)))
        return theta, lnl

    # ------------------------------------------------------------------ model curves
    def kepler_rv_batch(self, X, time, planets=None):
        """
        Keplerian velocity of every row of ``X`` (theta, sorted-parnames order) at ``time``: the sum
        over ``planets`` (planet numbers 1..K; None = all) of modelk, in planet order
        (evidence/rvmodel/__init__.py:343-463).  Returns ``(rv[B, T], ok[B])``; a row with an
        invalid Keplerian among the summed planets is NaN with ``ok`` False.  Solves that stopped
        at the Newton cap (which the reference drops silently) raise a RuntimeWarning.
        """
        X = self._as_batch(X, "X")
        time = np.ascontiguousarray(time, dtype=np.float64).reshape(-1)
        mask = planet_mask(self.nplanets, planets)
        B, T = X.shape[0], time.shape[0]
        rv = np.empty((B, T), dtype=np.float64)
        inv = np.zeros(B, dtype=np.uint32)
        caps = c_uint64(0)
        for lo, hi in curve_chunks(B, T):
            self._check(self._lib.rvl_kepler_rv(
                self._h, X[lo:].ctypes.data, hi - lo, time.ctypes.data, T, mask,
                rv[lo:].ctypes.data, inv[lo:].ctypes.data, byref(caps)))
        if caps.value:
            import warnings
            warnings.warn(f"{caps.value} Kepler solves stopped at the Newton cap "
                          f"(itmax = {self._desc.itmax}); their last iterate was used",
                          RuntimeWarning, stacklevel=2)
        return rv, (inv & np.uint32(mask)) == 0

    def kepler_rv_device(self, theta, times, planets=None, out=None):
        """
        ``kepler_rv_batch`` for CUDA float64 tensors ``theta[B, ndim]`` and ``times[T]``, enqueued
        on torch's current stream.  Returns ``(rv[B, T], ok[B])`` as CUDA tensors (no cap report).
        """
        import torch
        for name, v in (("theta", theta), ("times", times)):
            if not (v.is_cuda and v.dtype == torch.float64 and v.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous CUDA float64 tensor")
        if theta.dim() != 2 or theta.shape[1] != self.ndim or times.dim() != 1:
            raise ValueError(f"need theta of shape (B, {self.ndim}) and 1-D times")
        mask = planet_mask(self.nplanets, planets)
        B, T = theta.shape[0], times.shape[0]
        if out is None:
            out = torch.empty((B, T), dtype=torch.float64, device=theta.device)
        elif not (out.is_cuda and out.dtype == torch.float64 and out.is_contiguous()
                  and tuple(out.shape) == (B, T)):
            raise ValueError(f"out must be a contiguous CUDA float64 tensor of shape ({B}, {T})")
        inv = torch.zeros(B, dtype=torch.int32, device=theta.device)
        stream = torch.cuda.current_stream(theta.device).cuda_stream
        self._check(self._lib.rvl_kepler_rv_dev(
            self._h, c_void_p(theta.data_ptr()), B, c_void_p(times.data_ptr()), T, mask,
            c_void_p(out.data_ptr()), c_void_p(inv.data_ptr()), None, c_void_p(stream)))
        return out, (inv & mask) == 0

    def _curve(self, pardict, time, mask):
        row = pardict_row(pardict, self.parnames, self._desc, mask)
        time = np.asarray(time, dtype=np.float64).reshape(-1)
        ks = [k for k in range(1, self.nplanets + 1) if (mask >> (k - 1)) & 1]
        rv, ok = self.kepler_rv_batch(row[None], time, ks if ks else [])
        return rv[0] if ok[0] else None

    def modelk(self, pardict, time, planet):
        """Velocity of planet ``planet`` (1..K) at ``time`` (evidence/rvmodel/__init__.py:388-463);
        None for an invalid Keplerian (e > 1)."""
        return self._curve(pardict, time, planet_mask(self.nplanets, planet))

    def kep_rv(self, pardict, time, exclude_planet=None):
        """Sum of the planets' velocities at ``time`` (evidence/rvmodel/__init__.py:343-385); None
        if a summed planet is invalid.  ``exclude_planet``: a planet number, or an iterable of
        them, left out of the sum (what a phase fold of one planet subtracts)."""
        return self._curve(pardict, time, planet_mask(self.nplanets, exclude=exclude_planet))

    def drift(self, pardict, time):
        """evidence/rvmodel/__init__.py:222-273, on the host (see ``host_drift``)."""
        return host_drift(pardict, time)

    def residuals_batch(self, X):
        """
        Residuals and variances at the data epochs for every row of ``X``, composed in the
        reference's order (evidence/rvmodel/__init__.py:183-215): rvm = offset[inst] + kep_rv
        (device) + drift + sum of linear-parameter terms; res = vrad - rvm, var = svrad**2
        (+ jitter**2).  Returns ``(res[B, N], var[B, N])``; rows with an invalid Keplerian are NaN.
        """
        X = self._as_batch(X, "X")
        B = X.shape[0]
        d = self._desc

        def column(par):  # a model quantity for every row: a theta column or the fixed value
            return X[:, par.slot] if par.slot >= 0 else np.full(B, par.value)
        ids = self._inst_id
        rvm = np.zeros((B, len(self.time)))
        rvm += np.stack([column(d.offset[i]) for i in range(len(self.insts))], 1)[:, ids]
        ok = np.ones(B, dtype=bool)
        if self.nplanets > 0:
            kep, ok = self.kepler_rv_batch(X, self.time)
            rvm += kep
        if self.drift_in_model:
            coef = {nm: column(d.drift[j])[:, None]
                    for j, nm in enumerate(("lin", "quad", "cub", "quar"))}
            tt = (self.time - d.tref) / 365.25
            rvm += (coef["lin"] * tt + coef["quad"] * tt ** 2 + coef["cub"] * tt ** 3
                    + coef["quar"] * tt ** 4)
        for j, name in enumerate(self.linpar_dict):
            rvm += column(d.linpar[j])[:, None] * np.asarray(self.linpar_dict[name], dtype=np.float64)
        res = self.vrad - rvm
        var = np.broadcast_to(self.svrad ** 2, res.shape).copy()
        if self.jitter_in_model:
            var += np.stack([column(d.jitter[i]) for i in range(len(self.insts))], 1)[:, ids] ** 2
        res[~ok] = np.nan
        var[~ok] = np.nan
        return res, var

    # ------------------------------------------------------------------ host helpers
    def linear_parameter(self, time, indicator, kernel=None, timescale=0.5, filter_type="lp"):
        """
        Smoothed, [-1, 1]-normalised activity-indicator series for a ``linpar`` term: same
        signature and result as evidence/rvmodel/__init__.py:276-340 (kernels 'gaussian', 'box',
        'epanechnikov'; low-/high-pass).  Host side, runs once per model (the O(N^2) loop of the
        reference is a single broadcast here); feed the result to ``linpar_dict``.
        """
        time = np.asarray(time, dtype=np.float64)
        indicator = np.asarray(indicator, dtype=np.float64)
        assert len(time) == len(indicator), "time and indicator have to have the same length."
        if kernel is None:
            smoothed = indicator
        else:
            rt = time / (365.25 * timescale)
            delta = rt[None, :] - rt[:, None]  # row k: renorm_time - renorm_time[k]
            if kernel == "gaussian":
                w = np.exp(-0.5 * delta ** 2)
            elif kernel == "box":
                w = (np.abs(delta) <= 1.0).astype(np.float64)
            elif kernel == "epanechnikov":
                w = (np.abs(delta) <= 1.0) * (1.0 - delta ** 2)
            else:
                raise ValueError(f"Chosen kernel ('{kernel}') is not a valid option.")
            w = w / np.sum(w, axis=1, keepdims=True)
            low = np.sum(w * indicator[None, :], axis=1)
            if filter_type == "lp":
                smoothed = low
            elif filter_type == "hp":
                smoothed = indicator - low
            else:
                raise ValueError("filter_type has to be 'lp' or 'hp'")
        lo, hi = np.min(smoothed), np.max(smoothed)
        return 2.0 * (smoothed - lo) / (hi - lo) - 1.0

    # ------------------------------------------------------------------ reference FFI / stats
    def true_anomaly(self, ma, ecc, tol=1.0e-4):
        """Device version of evidence/rvmodel/__init__.py:466-494 (same signature)."""
        ma = np.ascontiguousarray(ma, dtype=np.float64)
        nu = np.zeros_like(ma)
        rc = self._lib.rvl_trueanomaly(self._h, _ptr(ma), len(ma), float(ecc), _ptr(nu),
                                       int(1.0e4), float(tol))
        if rc not in (0, -1):  # -1 = iteration cap, ignored like the reference (:490)
            self._check(rc)
        return nu

    def counters(self):
        c = _abi.rvl_counters_t()
        self._check(self._lib.rvl_counters(self._h, byref(c)))
        return {"n_points": c.n_points, "n_solves": c.n_solves,
                "n_newton_iters": c.n_newton_iters, "n_cap_hits": c.n_cap_hits,
                "n_invalid": c.n_invalid}

    def reset_counters(self):
        self._check(self._lib.rvl_reset_counters(self._h))

    def last_kernel_ms(self):
        ms = c_double()
        self._check(self._lib.rvl_last_kernel_ms(self._h, byref(ms)))
        return ms.value

    def last_gather_wait_ms(self):
        ms = c_double()
        self._check(self._lib.rvl_last_gather_wait_ms(self._h, byref(ms)))
        return ms.value

    def launch_count(self):
        n = c_uint64()
        self._check(self._lib.rvl_launch_count(self._h, byref(n)))
        return n.value

    def fp64_peak_tflops(self):
        v = c_double()
        self._check(self._lib.rvl_fp64_peak(self._h, byref(v)))
        return v.value

    def device_info(self):
        a, b, c = c_int32(), c_int32(), c_int32()
        self._check(self._lib.rvl_device_info(self._h, byref(a), byref(b), byref(c)))
        return {"sm_count": a.value, "smem_optin": b.value, "clock_khz": c.value}
