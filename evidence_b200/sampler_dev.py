"""
The slice-sampling nested sampler of ``evidence_b200.sampler`` with its bookkeeping on the device.

``sampler.nested_sample`` keeps the live points, brackets and masks in numpy and crosses the
host/device boundary for every likelihood batch; a run is then bound by that bookkeeping
(0.3 - 1.4 M lnL/s against 30 M lnL/s of the kernel, DESIGN.md section 9).  Here every array of
the run -- live points, walkers, brackets, candidates, evidence terms -- is a torch tensor on the
likelihood's device and the likelihood is called through the device entry point
(``RVModel.transform_loglike_device``: u -> theta -> lnL without leaving the GPU).  The host only
sequences the launches and reads back two scalars per round (loop exits).

``nested_sample_ensemble`` runs R independent runs of one model in lockstep: the walkers of all
runs share every bookkeeping and likelihood launch (``rvl_slice_phase_runs``), each run with its
own random streams.

Same algorithm (SURVEY.md 8f row 1; the scheme of PolyChord / UltraNest's step samplers that the
reference configures at evidence/ultranest/__init__.py:175): per round the k worst live points are
retired with the shrinkage 1/n for n = nlive, nlive-1, ..; k walkers started from surviving live
points take ``nsteps`` slice moves along whitened random directions under L > L*_k, with the next
m stepping-out positions and shrinkage candidates of every walker evaluated speculatively in one
launch (see ``sampler._slice_moves``).  Differences from the numpy sampler: the random numbers come
from torch's generator (so the two are statistically, not bit-wise, equivalent), and candidates
outside the unit cube are clamped before they are evaluated and rejected afterwards (no compaction
of the batch, hence no synchronisation to learn its size).  Circular coordinates (``wrapped``) follow
the rule of ``sampler``: taken modulo 1 in every candidate (``rvl_slice_phase_wrapped`` in the
kernels), whitened about their circular mean.

There is no CPU fallback in the product: ``fused`` must be a device callable.  (The function itself
is device-agnostic torch code, which is how the CPU tests drive it with an analytic likelihood.)
"""
import math

import numpy as np

from .sampler import NestedResult, lineage_bootstrap, retire_groups, wrap_mask


def _wrap_unit(torch, p):
    """p modulo 1 with 1 -> 0 (``sampler.wrap_unit``)."""
    q = p - torch.floor(p)
    return torch.where(q >= 1.0, torch.zeros_like(q), q)


def _whitening(torch, u, wrapped=None):
    """Lower Cholesky factor of the covariance of u[n, d]; ``wrapped`` (bool tensor [d] with at least
    one True, or None): those coordinates about their circular mean (``sampler.recentre``)."""
    if wrapped is not None:
        ang = 2.0 * math.pi * u
        mu = torch.atan2(torch.sin(ang).mean(0), torch.cos(ang).mean(0)) / (2.0 * math.pi)
        u = torch.where(wrapped, _wrap_unit(torch, u - mu + 0.5), u)
    d = u.shape[1]
    cov = torch.cov(u.T).reshape(d, d) + torch.eye(d, dtype=u.dtype, device=u.device) * 1e-18
    L, info = torch.linalg.cholesky_ex(cov)
    diag = torch.diag(torch.sqrt(torch.clamp(torch.diagonal(cov), min=1e-30)))
    return torch.where(info.reshape(1, 1) == 0, L, diag)


def _slice_moves(torch, gen, fused, u, theta, lmin, chol, nsteps, m, max_expand, max_shrink,
                 m_out=None, wrapped=None):
    """k walkers, nsteps slice moves each, everything on u.device.  Returns (u, theta, lnL, ncall);
    lnL is NaN for a walker that never moved.  ``wrapped`` (bool tensor [d] or None): those
    coordinates of every candidate are taken modulo 1 before the cube test and kept so."""
    k, d = u.shape
    dev, f64 = u.device, u.dtype
    lcur = torch.full((k,), float("nan"), dtype=f64, device=dev)
    rows = torch.arange(k, device=dev)
    # stepping out has no sequential dependence at all (the positions are lo - j, hi + j): with
    # room in the launch every one of the max_expand positions of both sides is evaluated at once
    # and the phase needs ONE launch and no read-back
    mo = m if m_out is None else max(1, min(int(m_out), max_expand))
    steps = torch.arange(mo, device=dev, dtype=f64)
    isteps = torch.arange(mo, device=dev)
    hi_clamp = 1.0 - 2.0 ** -53
    ncall = 0

    def fold(points):
        return points if wrapped is None else torch.where(wrapped, _wrap_unit(torch, points), points)

    def evaluate(points):
        """lnL (and theta) of points[k, n, d]; -inf outside the unit cube."""
        nonlocal ncall
        n = points.shape[1]
        inside = ((points >= 0.0) & (points < 1.0)).all(dim=-1)
        th, ll = fused(points.clamp(0.0, hi_clamp).reshape(k * n, d).contiguous())
        ncall += k * n
        ll = torch.where(inside, ll.reshape(k, n), torch.full_like(inside, -math.inf, dtype=f64))
        return ll, th.reshape(k, n, d)

    for _ in range(nsteps):
        z = torch.randn((k, d), generator=gen, dtype=f64, device=dev)
        z = z / torch.linalg.norm(z, dim=1, keepdim=True)
        dirn = z @ chol.T
        r = torch.rand((k,), generator=gen, dtype=f64, device=dev)
        lo, hi = -r, 1.0 - r
        # ---- stepping out: the next m unit steps of both sides in one launch
        grow_lo = torch.ones(k, dtype=torch.bool, device=dev)
        grow_hi = torch.ones(k, dtype=torch.bool, device=dev)
        done_lo = torch.zeros(k, dtype=torch.long, device=dev)
        done_hi = torch.zeros(k, dtype=torch.long, device=dev)
        n_out = (max_expand + mo - 1) // mo
        for _e in range(n_out):
            edges = torch.cat([lo[:, None] - steps[None, :], hi[:, None] + steps[None, :]], dim=1)
            mask = torch.cat([grow_lo[:, None] & (done_lo[:, None] + isteps[None, :] < max_expand),
                              grow_hi[:, None] & (done_hi[:, None] + isteps[None, :] < max_expand)], dim=1)
            ll, _ = evaluate(fold(u[:, None, :] + edges[:, :, None] * dirn[:, None, :]))
            above = (ll > lmin) & mask
            run_lo = torch.cumprod(above[:, :mo].to(torch.long), dim=1).sum(dim=1)
            run_hi = torch.cumprod(above[:, mo:].to(torch.long), dim=1).sum(dim=1)
            lo = lo - run_lo.to(f64)
            hi = hi + run_hi.to(f64)
            done_lo = done_lo + run_lo
            done_hi = done_hi + run_hi
            if n_out == 1:
                break
            grow_lo = grow_lo & (run_lo == mo) & (done_lo < max_expand)
            grow_hi = grow_hi & (run_hi == mo) & (done_hi < max_expand)
            if not bool((grow_lo | grow_hi).any()):  # one scalar back per launch
                break
        # ---- shrinkage: the next m candidates, each drawn as if the ones before it were rejected
        pending = torch.ones(k, dtype=torch.bool, device=dev)
        draws = torch.rand((max_shrink, k), generator=gen, dtype=f64, device=dev)
        it = 0
        while it < max_shrink:
            mm = min(m, max_shrink - it)
            lo_s, hi_s = lo, hi
            ts = []
            for j in range(mm):
                t = lo_s + (hi_s - lo_s) * draws[it + j]
                ts.append(t)
                lo_s = torch.where(t < 0, t, lo_s)
                hi_s = torch.where(t >= 0, t, hi_s)
            T = torch.stack(ts, dim=1)
            cand = fold(u[:, None, :] + T[:, :, None] * dirn[:, None, :])
            ll, th = evaluate(cand)
            acc = (ll > lmin) & pending[:, None]
            hit = acc.any(dim=1)
            first = acc.to(torch.int8).argmax(dim=1)
            u = torch.where(hit[:, None], cand[rows, first], u)
            theta = torch.where(hit[:, None], th[rows, first], theta)
            lcur = torch.where(hit, ll[rows, first], lcur)
            pending = pending & ~hit
            lo = torch.where(pending, lo_s, lo)
            hi = torch.where(pending, hi_s, hi)
            it += mm
            if not bool(pending.any()):
                break
    return u, theta, lcur, ncall


def _wrap_bits(wrap):
    """The mask of rvl_slice_phase_wrapped (uint32[4]) for a bool per dimension; None without a True."""
    import ctypes
    if wrap is None or not np.any(wrap):
        return None
    bits = (ctypes.c_uint32 * 4)()
    for j in np.flatnonzero(np.asarray(wrap, dtype=bool)):
        bits[j >> 5] |= 1 << (int(j) & 31)
    return bits


class _NativeSlice:
    """
    The slice moves of a round through the hand-written kernels of csrc/rvslice.cu
    (``rvl_slice_phase``): per move 3-4 bookkeeping launches around 2-3 likelihood launches, nothing
    read back.  Stepping out evaluates all ``n_out`` positions of both sides at once; shrinkage runs
    ``rounds`` launches of ``m`` speculated candidates per walker (a walker whose bracket is not
    resolved after rounds * m candidates keeps its position -- counted in ``unresolved``; with the
    defaults, 24 candidates, that is a few 1e-3 of the moves on the RV posteriors).  ``wrap`` (bool
    per dimension, or None): circular coordinates, through ``rvl_slice_phase_wrapped``.
    """

    def __init__(self, torch, k, d, dev, seed, n_out=8, m=8, rounds=3, wrap=None):
        import ctypes
        from . import _abi
        self.torch, self.k, self.d, self.n_out, self.m, self.rounds = torch, k, d, n_out, m, rounds
        self.lib = _abi.load()
        f64 = torch.float64
        z = lambda *shape, dt=f64: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
        self.dirn, self.lo, self.hi, self.lo2, self.hi2 = z(k, d), z(k), z(k), z(k), z(k)
        self.tval, self.pending = z(k, m), z(k, dt=torch.int32)
        self.cand_o, self.inside_o = z(k * 2 * n_out, d), z(k * 2 * n_out, dt=torch.uint8)
        self.th_o, self.ll_o = z(k * 2 * n_out, d), z(k * 2 * n_out)
        self.cand, self.inside = z(k * m, d), z(k * m, dt=torch.uint8)
        self.th, self.ll = z(k * m, d), z(k * m)
        self.stats = z(2, dt=torch.int64)
        self.args = _abi.rvl_slice_args()
        self.args.k, self.args.d, self.args.n_out, self.args.m = k, d, n_out, m
        self.args.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        for name, t in (("dirn", self.dirn), ("lo", self.lo), ("hi", self.hi), ("lo2", self.lo2),
                        ("hi2", self.hi2), ("tval", self.tval), ("pending", self.pending),
                        ("cand_out", self.cand_o), ("inside_out", self.inside_o), ("ll_out", self.ll_o),
                        ("cand", self.cand), ("inside", self.inside), ("cand_ll", self.ll),
                        ("cand_th", self.th), ("stats", self.stats)):
            setattr(self.args, name, t.data_ptr())
        self._byref = ctypes.byref(self.args)
        self.wrap_bits = _wrap_bits(wrap)
        self.move = 0

    def _phase(self, ph):
        stream = self.torch.cuda.current_stream().cuda_stream
        if self.wrap_bits is None:
            rc = self.lib.rvl_slice_phase(ph, self._byref, stream)
        else:
            rc = self.lib.rvl_slice_phase_wrapped(ph, self._byref, self.wrap_bits, stream)
        if rc != 0:
            raise RuntimeError("rvl_slice_phase: " + self.lib.rvl_slice_last_error().decode())

    @staticmethod
    def _writes_in_place(fused):
        """Does ``fused`` take ``theta=`` / ``lnl=`` output tensors (RVModel.transform_loglike_device)?"""
        import inspect
        try:
            params = inspect.signature(fused).parameters
        except (TypeError, ValueError):
            return False
        return "theta" in params and "lnl" in params

    def _eval(self, fused, pts, th_out, ll_out):
        if self._inplace:
            fused(pts, theta=th_out, lnl=ll_out)
        else:
            th, ll = fused(pts)
            th_out.copy_(th)
            ll_out.copy_(ll)

    def moves(self, fused, u, theta, lcur, lmin, chol, nsteps):
        """nsteps slice moves of the k walkers u (updated in place with theta and lcur)."""
        a = self.args
        self._inplace = self._writes_in_place(fused)
        chol = chol.contiguous()
        a.lmin, a.chol = lmin.data_ptr(), chol.data_ptr()
        a.u, a.theta, a.lcur = u.data_ptr(), theta.data_ptr(), lcur.data_ptr()
        ncall = 0
        for _ in range(nsteps):
            a.move, a.shrink_round = self.move & 0xFFFFFFFF, 0
            self.move += 1
            self._phase(0)
            self._eval(fused, self.cand_o, self.th_o, self.ll_o)
            self._phase(1)
            for r in range(self.rounds):
                self._eval(fused, self.cand, self.th, self.ll)
                a.shrink_round = r + 1
                self._phase(2 if r + 1 < self.rounds else 3)
            ncall += self.k * (2 * self.n_out + self.rounds * self.m)
        return ncall


def nested_sample_device(fused, ndim, nlive=400, dlogz=0.5, frac_remain=0.01, seed=0, nsteps=None,
                         batch_fraction=0.2, speculate=None, device="cuda", max_expand=16,
                         max_shrink=64, max_calls=2_000_000_000, verbose=False, num_bootstraps=30,
                         native=None, native_m=8, native_rounds=3, native_out=8, wrapped=None):
    """
    Nested sampling with every array on ``device``.  ``fused(U[n, ndim]) -> (theta[n, ndim],
    lnL[n])`` maps unit-cube points to parameters and log-likelihoods on that device
    (``RVModel.transform_loglike_device``).  Returns the same ``NestedResult`` as
    ``sampler.nested_sample`` (arrays as numpy).

    ``native`` (default: on a CUDA device): the slice moves run through the hand-written bookkeeping
    kernels of csrc/rvslice.cu (``_NativeSlice``) instead of ~150 small torch launches per move;
    ``native_out`` stepping-out positions per side, ``native_rounds`` x ``native_m`` shrinkage
    candidates per walker and move, all speculated.  The torch formulation below it is the same
    sampler for CPU tensors (tests) and the statistical cross-check of the kernels.

    ``wrapped`` (bool per dimension, UltraNest's ``wrapped_params``): circular coordinates, as in
    ``sampler.nested_sample``; None or no True leaves the run exactly as without it.
    """
    import torch
    dev = torch.device(device)
    f64 = torch.float64
    gen = torch.Generator(device=dev).manual_seed(int(seed))
    if native is None:
        native = dev.type == "cuda"
    nsteps = nsteps or max(4, 3 * ndim)  # the reference's default (evidence/ultranest/__init__.py:335)
    wmask = wrap_mask(wrapped, ndim)
    wrap = torch.as_tensor(wmask, device=dev) if wmask.any() else None
    k = max(1, min(int(batch_fraction * nlive), nlive - 2))
    m = max(1, min(6, 512 // k)) if speculate is None else max(1, int(speculate))
    m_out = max(m, min(max_expand, 4096 // (2 * k)))  # a likelihood launch costs the same up to ~4096 points
    u_live = torch.rand((nlive, ndim), generator=gen, dtype=f64, device=dev)
    th_live, l_live = fused(u_live)
    th_live, l_live = th_live.clone(), l_live.clone()
    ncall = nlive
    # the shrinkage of one round is the same every round: n = nlive, nlive-1, .., nlive-k+1
    shrink = 1.0 / (nlive - torch.arange(k, dtype=f64, device=dev))
    before = -(torch.cumsum(shrink, 0) - shrink)          # ln X offset before each retirement
    logw_rel = before + torch.log1p(-torch.exp(-shrink))   # ln w_j - ln X(start of the round)
    round_shrink = float(shrink.sum())
    logx = 0.0
    logz = torch.tensor(-math.inf, dtype=f64, device=dev)
    dead_theta, dead_logl, dead_logw = [], [], []
    # threads (see sampler.lineage_bootstrap): slot and birth constraint of every point
    root_live = torch.arange(nlive, device=dev)
    birth_live = torch.full((nlive,), -math.inf, dtype=f64, device=dev)
    dead_root, dead_birth = [], []
    niter = 0
    natives, move_no = {}, 0
    l_sorted, order = torch.sort(l_live, stable=True)
    # points tied with the k-th worst are retired with it (a plateau goes as a whole: retire_groups);
    # the count rides on the one read-back per round
    kk = int((l_sorted <= l_sorted[k - 1]).sum())
    while True:
        kk = min(kk, nlive - 2)
        worst, keep = order[:kk], order[kk:]
        if kk == k:
            logw, dx = logx + logw_rel, round_shrink
        else:  # a plateau round (rare: invalid-Keplerian sentinels at the start of a run)
            dlx, lw = retire_groups(l_sorted[:kk].cpu().numpy(), nlive)
            logw, dx = logx + torch.from_numpy(lw).to(dev), -float(dlx.sum())
        logz = torch.logaddexp(logz, torch.logsumexp(l_sorted[:kk] + logw, 0))
        dead_theta.append(th_live[worst])
        dead_logl.append(l_sorted[:kk])
        dead_logw.append(logw)
        dead_root.append(root_live[worst])
        dead_birth.append(birth_live[worst])
        logx -= dx
        niter += kk
        lmin = l_sorted[kk - 1]
        chol = _whitening(torch, u_live[keep], wrap)
        starts = keep[torch.randint(0, len(keep), (kk,), generator=gen, device=dev)]
        if native:
            if kk not in natives:
                natives[kk] = _NativeSlice(torch, kk, ndim, dev, seed, n_out=native_out, m=native_m,
                                           rounds=native_rounds, wrap=wmask)
            natives[kk].move = move_no
            u_new, th_new = u_live[starts].clone(), th_live[starts].clone()
            l_new = torch.full((kk,), float("nan"), dtype=f64, device=dev)
            nc = natives[kk].moves(fused, u_new, th_new, l_new, lmin.reshape(1).clone(), chol, nsteps)
            move_no += nsteps
        else:
            u_new, th_new, l_new, nc = _slice_moves(torch, gen, fused, u_live[starts].clone(),
                                                    th_live[starts].clone(), lmin, chol, nsteps, m,
                                                    max_expand, max_shrink, m_out=m_out, wrapped=wrap)
        ncall += nc
        stuck = ~torch.isfinite(l_new)  # a walker that never moved is a copy of its start point
        l_new = torch.where(stuck, l_live[starts], l_new)
        u_live[worst], th_live[worst], l_live[worst] = u_new, th_new, l_new
        birth_live[worst] = lmin  # (root = slot: the thread continues with the point written into it)
        if ncall > max_calls:
            raise RuntimeError("nested_sample_device: max_calls exceeded")
        # UltraNest's two criteria (evidence/ultranest/__init__.py:181-185); one read-back per round
        l_sorted, order = torch.sort(l_live, stable=True)
        log_remain = l_sorted[-1] + logx
        total = torch.logaddexp(logz, log_remain)
        tied = (l_sorted <= l_sorted[k - 1]).sum().to(f64)
        lr, tt, lz, kk = (float(x) for x in torch.stack([log_remain, total, logz, tied]).cpu())
        kk = int(kk)
        if verbose and (niter // k) % 20 == 0:
            print(f"it={niter} lnZ={lz:.3f} ln(remain/Z)={lr - lz:.2f} ncall={ncall}")
        if lr - tt < math.log(frac_remain) and tt - lz < dlogz:
            break
    logw_live = torch.full((nlive,), logx - math.log(nlive), dtype=f64, device=dev)
    logz = torch.logaddexp(logz, torch.logsumexp(l_sorted + logw_live, 0))
    dead_theta.append(th_live[order])
    dead_logl.append(l_sorted)
    dead_logw.append(logw_live)
    dead_root.append(root_live[order])
    dead_birth.append(birth_live[order])
    theta = torch.cat(dead_theta)
    logl = torch.cat(dead_logl)
    logwt = logl + torch.cat(dead_logw) - logz
    p = torch.exp(logwt)
    h_info = float((p * logl).sum() - logz)                 # H = sum p_i ln L_i - ln Z
    weights = torch.exp(logwt - logwt.max())
    weights = weights / weights.sum()
    nsamp = max(1, int(1.0 / float((weights ** 2).sum())))
    pos = (float(torch.rand((), generator=gen, dtype=f64, device=dev)) +
           torch.arange(nsamp, dtype=f64, device=dev)) / nsamp
    idx = torch.clamp(torch.searchsorted(torch.cumsum(weights, 0), pos), max=len(weights) - 1)
    skilling = math.sqrt(max(h_info, 0.0) / nlive)
    bs_std, _ = lineage_bootstrap(torch.cat(dead_birth).cpu().numpy(), logl.cpu().numpy(),
                                  torch.cat(dead_root).cpu().numpy(), nlive,
                                  np.random.default_rng([int(seed), 0xB007]), num_bootstraps)
    return NestedResult(logz=float(logz), logzerr=float(max(skilling, bs_std)),
                        logzerr_skilling=skilling, logzerr_bootstrap=bs_std,
                        ncall=int(ncall), niter=int(niter), information=h_info,
                        samples=theta[idx].cpu().numpy(), weighted_samples=theta.cpu().numpy(),
                        weights=weights.cpu().numpy(), logl=logl.cpu().numpy(), nlive=nlive,
                        seed=seed, method="slice-device" + ("-native" if native else ""),
                        unresolved_moves=int(sum(int(n.stats[0]) for n in natives.values())),
                        accepted_moves=int(sum(int(n.stats[1]) for n in natives.values())),
                        wrapped=wmask)


# ------------------------------------------------------------------------------------------------
# ensembles: R independent runs of one model, advanced in lockstep through shared launches
# ------------------------------------------------------------------------------------------------
def _ensemble_seeds(seeds):
    """The seeds of an ensemble as uint64 values; an empty list or a repeated seed is an error (two
    identical runs would be counted as two independent ones)."""
    vals = [int(s) & 0xFFFFFFFFFFFFFFFF for s in np.atleast_1d(np.asarray(seeds, dtype=object))]
    if not vals:
        raise ValueError("seeds: an ensemble needs at least one seed")
    if len(set(vals)) != len(vals):
        dup = sorted({v for v in vals if vals.count(v) > 1})
        raise ValueError(f"seeds: {dup} given more than once; identical runs are not independent")
    return vals


def _walker_layout(counts):
    """(run_of, walker_of), int32 [sum(counts)]: the walkers of run r are walkers 0 .. counts[r] - 1
    of that run, runs in order; a run with count 0 (finished) has none."""
    counts = np.asarray(counts, dtype=np.int64)
    run_of = np.repeat(np.arange(len(counts), dtype=np.int32), counts)
    first = np.concatenate([[0], np.cumsum(counts)[:-1]])
    walker_of = (np.arange(len(run_of)) - np.repeat(first, counts)).astype(np.int32)
    return run_of, walker_of


class _NativeSliceRuns(_NativeSlice):
    """
    The kernels of an ensemble: ``rvl_slice_runs_init`` / ``_whiten`` / ``_starts`` and the slice
    moves of ``_NativeSlice.moves`` through ``rvl_slice_phase_runs``.  One set of walker and
    candidate buffers for all runs, grown by ``reserve`` when a round needs more walkers (a plateau
    round) and otherwise reused; the first k rows of each are the walkers of the round.
    """

    # buffer -> (rows per walker, trailing shape: "d" or "m", dtype name)
    _BUFFERS = {"u": (1, "d", "float64"), "theta": (1, "d", "float64"), "lcur": (1, None, "float64"),
                "dirn": (1, "d", "float64"), "lo": (1, None, "float64"), "hi": (1, None, "float64"),
                "lo2": (1, None, "float64"), "hi2": (1, None, "float64"), "tval": (1, "m", "float64"),
                "pending": (1, None, "int32"), "cand_o": ("2n", "d", "float64"),
                "inside_o": ("2n", None, "uint8"), "th_o": ("2n", "d", "float64"),
                "ll_o": ("2n", None, "float64"), "cand": ("m", "d", "float64"),
                "inside": ("m", None, "uint8"), "th": ("m", "d", "float64"), "ll": ("m", None, "float64"),
                "start": (1, None, "int64"), "lstart": (1, None, "float64")}
    _ARGS = {"u": "u", "theta": "theta", "lcur": "lcur", "dirn": "dirn", "lo": "lo", "hi": "hi",
             "lo2": "lo2", "hi2": "hi2", "tval": "tval", "pending": "pending", "cand_o": "cand_out",
             "inside_o": "inside_out", "ll_o": "ll_out", "cand": "cand", "inside": "inside",
             "ll": "cand_ll", "th": "cand_th"}

    def __init__(self, torch, d, dev, seeds, nlive, n_out=8, m=8, rounds=3, wrap=None):
        import ctypes
        from . import _abi
        self.torch, self.d, self.dev, self.n_out, self.m, self.rounds = torch, d, dev, n_out, m, rounds
        self.lib = _abi.load()
        R = self.n_runs = len(seeds)
        self.wrap_bits = _wrap_bits(wrap)
        f64 = torch.float64
        self.seeds = torch.from_numpy(np.array(seeds, dtype=np.uint64).view(np.int64)).to(dev)
        self.chol = torch.zeros((R, d, d), dtype=f64, device=dev)
        self.stats = torch.zeros((R, 2), dtype=torch.int64, device=dev)
        self.u_live = torch.zeros((R, nlive, d), dtype=f64, device=dev)
        self.runs = _abi.rvl_slice_runs(n_runs=R, seeds=self.seeds.data_ptr(), chol=self.chol.data_ptr(),
                                        stats=self.stats.data_ptr())
        self.live = _abi.rvl_slice_live(nlive=nlive, d=d, u_live=self.u_live.data_ptr())
        self.args = _abi.rvl_slice_args(d=d, n_out=n_out, m=m)
        self._byref, self._runs, self._live = (ctypes.byref(self.args), ctypes.byref(self.runs),
                                               ctypes.byref(self.live))
        self.cap, self.k, self.move, self._full = 0, 0, 0, {}

    def reserve(self, k):
        """Make the buffers hold k walkers (reallocated only when k exceeds the capacity)."""
        torch = self.torch
        if k > self.cap:
            rows = {1: 1, "2n": 2 * self.n_out, "m": self.m}
            tail = {None: (), "d": (self.d,), "m": (self.m,)}
            self._full = {name: torch.zeros((k * rows[r],) + tail[t], dtype=getattr(torch, dt), device=self.dev)
                          for name, (r, t, dt) in self._BUFFERS.items()}
            self.cap = k
        for name, (r, _, _) in self._BUFFERS.items():
            setattr(self, name, self._full[name][:k * {1: 1, "2n": 2 * self.n_out, "m": self.m}[r]])
        for name, field in self._ARGS.items():
            setattr(self.args, field, getattr(self, name).data_ptr())
        self.live.start, self.live.lstart = self.start.data_ptr(), self.lstart.data_ptr()
        self.k = self.args.k = k

    def _stream(self):
        return self.torch.cuda.current_stream().cuda_stream

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what}: " + self.lib.rvl_slice_last_error().decode())

    def _phase(self, ph):
        self._check(self.lib.rvl_slice_phase_runs(ph, self._byref, self._runs, self.wrap_bits, self._stream()),
                    "rvl_slice_phase_runs")

    def init(self):
        """u_live[r] = the initial live points of run r, from its seed."""
        self._check(self.lib.rvl_slice_runs_init(self._runs, self._live, self._stream()), "rvl_slice_runs_init")
        return self.u_live

    def setup_round(self, th_live, l_live, order, kk, lmin, run_of, walker_of, round_no):
        """Whitening of every run and the starts of the round's walkers (the layout run_of /
        walker_of, int32 device tensors of the reserved length)."""
        lv, rn = self.live, self.runs
        lv.th_live, lv.l_live, lv.order, lv.kk = (th_live.data_ptr(), l_live.data_ptr(), order.data_ptr(),
                                                  kk.data_ptr())
        lv.round = round_no & 0xFFFFFFFF
        rn.lmin, rn.run_of, rn.walker_of = lmin.data_ptr(), run_of.data_ptr(), walker_of.data_ptr()
        self._check(self.lib.rvl_slice_runs_whiten(self._runs, self._live, self.wrap_bits, self._stream()),
                    "rvl_slice_runs_whiten")
        self._check(self.lib.rvl_slice_runs_starts(self._byref, self._runs, self._live, self._stream()),
                    "rvl_slice_runs_starts")


def nested_sample_ensemble(fused, ndim, seeds, nlive=400, dlogz=0.5, frac_remain=0.01, nsteps=None,
                           wrapped=None, device="cuda", native_m=8, native_rounds=3, native_out=8,
                           num_bootstraps=30, max_calls=2_000_000_000):
    """
    R = len(seeds) independent runs of ``nested_sample_device`` (native kernels, batch_fraction 0.2)
    on one likelihood, advanced in lockstep: every bookkeeping launch and every likelihood launch
    carries the walkers of all runs still active.  Returns one ``NestedResult`` per seed, in the
    order of ``seeds`` -- e.g. for the median ln Z per model of the reference's model selection
    (evidence/fip_criterion.py:245-266) or the run-to-run scatter of ln Z.

    Each run has the retirement, plateau, stuck-walker and termination rules, slice moves and
    lineage bootstrap of ``nested_sample_device``, but its own random streams, keyed by its seed:
    initial points, starts and moves from the kernels' Philox generator (``rvl_slice_runs_*``,
    ``rvl_slice_phase_runs``), the whitening from its own points in a fixed order.  A run's chain
    is therefore the same whatever other runs share the ensemble -- exactly so when the row values
    of ``fused`` do not depend on the rest of the batch (its ln Z then to the last bits of a batched
    sum).  The RV kernel's rows can change in the last bits with their position in the batch
    (DESIGN.md section 4): with the RV model runs are independent statistically, not bit for bit.
    The streams differ from those of ``nested_sample_device`` with the same seed.

    The host reads back one [R, 4] tensor per round (loop exits and tie counts), plus the retired
    values of a run in a plateau round (``retire_groups``), as the single-run sampler does.
    """
    import torch
    seeds = _ensemble_seeds(seeds)
    wmask = wrap_mask(wrapped, ndim)
    dev = torch.device(device)
    if dev.type != "cuda":
        raise ValueError("nested_sample_ensemble runs the kernels of csrc/rvslice.cu: device must be CUDA")
    R, f64 = len(seeds), torch.float64
    nsteps = nsteps or max(4, 3 * ndim)
    k = max(1, min(int(0.2 * nlive), nlive - 2))
    per_walker = nsteps * (2 * native_out + native_rounds * native_m)  # lnL calls per walker and round
    ns = _NativeSliceRuns(torch, ndim, dev, seeds, nlive, n_out=native_out, m=native_m,
                          rounds=native_rounds, wrap=wmask)
    u_live = ns.init()
    th, ll = fused(u_live.reshape(R * nlive, ndim))
    th_live, l_live = th.reshape(R, nlive, ndim).clone(), ll.reshape(R, nlive).clone()
    ncall = np.full(R, nlive, dtype=np.int64)
    shrink = 1.0 / (nlive - torch.arange(k, dtype=f64, device=dev))
    before = -(torch.cumsum(shrink, 0) - shrink)
    logw_rel = before + torch.log1p(-torch.exp(-shrink))
    round_shrink = float(shrink.sum())
    logx = np.zeros(R)
    logz = torch.full((R,), -math.inf, dtype=f64, device=dev)
    root_live = torch.arange(nlive, device=dev).repeat(R, 1)
    birth_live = torch.full((R, nlive), -math.inf, dtype=f64, device=dev)
    records = []  # (runs, theta [n, kk, d], logl, logw, root, birth [n, kk]) per retirement group
    niter = np.zeros(R, dtype=np.int64)
    active = np.ones(R, dtype=bool)
    move_no = round_no = 0
    l_sorted, order = torch.sort(l_live, dim=1, stable=True)
    kk = (l_sorted <= l_sorted[:, k - 1:k]).sum(1).cpu().numpy()
    # what the host decides for a round goes to the device in two copies from page-locked buffers,
    # queued before the round's launches: [kk (0 = finished) | run_of | walker_of | regular runs] and
    # [ln X before | ln X after the round's retirement]
    up_i = torch.empty(R + 2 * R * nlive + R, dtype=torch.int32).pin_memory()
    up_f = torch.empty(2 * R, dtype=f64).pin_memory()
    dev_i = torch.empty(up_i.shape, dtype=torch.int32, device=dev)
    dev_f = torch.empty(up_f.shape, dtype=f64, device=dev)
    while active.any():
        act = np.flatnonzero(active)
        kk = np.minimum(kk, nlive - 2)
        regular, plateau = act[kk[act] == k], act[kk[act] != k]
        logx_before = logx.copy()
        logx[regular] -= round_shrink
        lws = {}
        for r in plateau:  # rare: invalid-Keplerian sentinels at the start of a run
            dlx, lws[r] = retire_groups(l_sorted[r, :int(kk[r])].cpu().numpy(), nlive)
            logx[r] -= -float(dlx.sum())
        niter[act] += kk[act]
        # the round's walkers: kk[r] for every active run, walker j of run r replaces order[r][j]
        counts = np.where(active, kk, 0)
        run_of, walker_of = _walker_layout(counts)
        K, G = len(run_of), len(regular)
        n_up = R + 2 * K + G
        up_i[:n_up] = torch.from_numpy(np.concatenate([counts.astype(np.int32), run_of, walker_of,
                                                       regular.astype(np.int32)]))
        up_f[:R], up_f[R:] = torch.from_numpy(logx_before), torch.from_numpy(logx)
        dev_i[:n_up].copy_(up_i[:n_up], non_blocking=True)
        dev_f.copy_(up_f, non_blocking=True)
        kk_dev, run_t, walker_t = dev_i[:R].long(), dev_i[R:R + K], dev_i[R + K:R + 2 * K]
        if G:
            idx = dev_i[R + 2 * K:n_up].long()
            ls = l_sorted[idx, :k]
            logw = dev_f[idx][:, None] + logw_rel
            logz[idx] = torch.logaddexp(logz[idx], torch.logsumexp(ls + logw, 1))
            worst = order[idx, :k]
            rows = idx[:, None]
            records.append((regular, th_live[rows, worst], ls, logw, root_live[rows, worst],
                            birth_live[rows, worst]))
        for r in plateau:
            n = int(kk[r])
            logw = logx_before[r] + torch.from_numpy(lws[r]).to(dev)
            ls = l_sorted[r, :n]
            logz[r] = torch.logaddexp(logz[r], torch.logsumexp(ls + logw, 0))
            worst = order[r, :n]
            records.append((np.array([r]), th_live[r, worst][None], ls[None], logw[None],
                            root_live[r, worst][None], birth_live[r, worst][None]))
        ns.reserve(K)
        lmin = l_sorted.gather(1, (kk_dev - 1).clamp(min=0)[:, None]).reshape(R)
        ns.setup_round(th_live, l_live, order, kk_dev, lmin, run_t, walker_t, round_no)
        ns.move = move_no
        ns.moves(fused, ns.u, ns.theta, ns.lcur, lmin, ns.chol, nsteps)
        move_no += nsteps
        round_no += 1
        ncall += counts * per_walker
        stuck = ~torch.isfinite(ns.lcur)  # a walker that never moved is a copy of its start point
        l_new = torch.where(stuck, ns.lstart, ns.lcur)
        run_l = run_t.long()
        dst = run_l * nlive + order[run_l, walker_t.long()]
        u_live.view(-1, ndim)[dst] = ns.u
        th_live.view(-1, ndim)[dst] = ns.theta
        l_live.view(-1)[dst] = l_new
        birth_live.view(-1)[dst] = lmin[run_l]
        if (ncall > max_calls).any():
            raise RuntimeError("nested_sample_ensemble: max_calls exceeded")
        l_sorted, order = torch.sort(l_live, dim=1, stable=True)
        log_remain = l_sorted[:, -1] + dev_f[R:]
        total = torch.logaddexp(logz, log_remain)
        tied = (l_sorted <= l_sorted[:, k - 1:k]).sum(1).to(f64)
        back = torch.stack([log_remain, total, logz, tied], 1).cpu().numpy()  # one read-back per round
        kk = back[:, 3].astype(np.int64)
        for r in act:
            lr, tt, lz = back[r, :3]
            if lr - tt < math.log(frac_remain) and tt - lz < dlogz:
                # UltraNest's two criteria met: the final live points join the dead ones
                logw_live = torch.full((nlive,), logx[r] - math.log(nlive), dtype=f64, device=dev)
                logz[r] = torch.logaddexp(logz[r], torch.logsumexp(l_sorted[r] + logw_live, 0))
                o = order[r]
                records.append((np.array([r]), th_live[r, o][None], l_sorted[r][None], logw_live[None],
                                root_live[r, o][None], birth_live[r, o][None]))
                active[r] = False
    return _ensemble_results(records, logz.cpu().numpy(), ns.stats.cpu().numpy(), seeds, ncall, niter,
                             nlive, ndim, wmask, num_bootstraps)


def _ensemble_results(records, logz, stats, seeds, ncall, niter, nlive, ndim, wmask, num_bootstraps):
    """One NestedResult per run from the retirement records of an ensemble (host numpy; each run's
    arrays in the order its points died, as nested_sample_device keeps them)."""
    import torch
    host = [torch.cat([rec[1 + j].reshape((-1, ndim) if j == 0 else (-1,)) for rec in records]).cpu().numpy()
            for j in range(5)]
    pieces = [[] for _ in seeds]
    off = 0
    for rec in records:
        n_kk = rec[2].shape[1]
        for p, r in enumerate(rec[0]):
            pieces[r].append(slice(off + p * n_kk, off + (p + 1) * n_kk))
        off += len(rec[0]) * n_kk
    out = []
    for r, seed in enumerate(seeds):
        theta, logl, logw, root, birth = (np.concatenate([a[s] for s in pieces[r]]) for a in host)
        lz = float(logz[r])
        logwt = logl + logw - lz
        h_info = float((np.exp(logwt) * logl).sum() - lz)
        weights = np.exp(logwt - logwt.max())
        weights = weights / weights.sum()
        nsamp = max(1, int(1.0 / float((weights ** 2).sum())))
        pos = (np.random.default_rng([seed, 0x5A3D]).random() + np.arange(nsamp)) / nsamp
        idx = np.minimum(np.searchsorted(np.cumsum(weights), pos), len(weights) - 1)
        skilling = math.sqrt(max(h_info, 0.0) / nlive)
        bs_std, _ = lineage_bootstrap(birth, logl, root, nlive, np.random.default_rng([seed, 0xB007]),
                                      num_bootstraps)
        out.append(NestedResult(logz=lz, logzerr=float(max(skilling, bs_std)), logzerr_skilling=skilling,
                                logzerr_bootstrap=bs_std, ncall=int(ncall[r]), niter=int(niter[r]),
                                information=h_info, samples=theta[idx], weighted_samples=theta,
                                weights=weights, logl=logl, nlive=nlive, seed=seed,
                                method="slice-device-native-ensemble",
                                unresolved_moves=int(stats[r, 0]), accepted_moves=int(stats[r, 1]),
                                wrapped=wmask))
    return out
