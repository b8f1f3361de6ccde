"""
Small, seeded, fully vectorised nested samplers.

The reference delegates sampling to third-party packages (UltraNest, PolyChord) that are not part
of its repository and are absent from this image (SURVEY.md 8c).  The runner in
``evidence_b200.ultranest`` uses UltraNest when it is importable; this module is the stand-in
that makes end-to-end ln Z runs possible without it, and -- because it is deterministic for a
given seed -- lets the SAME sampler code be driven by the device likelihood and by the CPU oracle
to check that the two agree on ln Z (BASELINE.json north_star).

Two replacement schemes for classic nested sampling (Skilling 2006):

``nested_sample`` (default, method='slice'): the k worst live points are retired per round
(prior volume shrinks by 1/n for n = nlive, nlive-1, ..., the dynamic-live-point bookkeeping) and
k walkers started from surviving live points take ``nsteps`` slice-sampling moves along random
directions whitened by the live-point covariance, under the hard constraint L > L*_k -- the
scheme of PolyChord and of UltraNest's step samplers (the reference configures UltraNest with a
RegionSliceSampler, evidence/ultranest/__init__.py:175).  All k walkers are advanced in lock-step,
so every likelihood call is one batch of up to k points.  Robust for the multimodal period
posteriors of RV models.

``nested_sample_ellipsoid``: rejection sampling from a single bounding ellipsoid of the live
points (MultiNest with one ellipsoid / nestle's 'single' bound); candidates are drawn in batches
of ``ndraw`` -- the large batches the device path is built for -- and consumed in order.  Efficient
for unimodal problems only.

Circular coordinates (``wrapped``, UltraNest's ``wrapped_params``; opt-in): the slice samplers take
a wrapped coordinate of every candidate modulo 1 instead of rejecting it outside [0, 1), so the
walkers move on the torus (``wrap_unit``), and whiten with the covariance of the live points
re-centred on their circular mean in those coordinates (``recentre``).  Nested sampling needs
points uniform in the cube under L > L*; the torus has the same uniform measure, so this is valid
for any coordinate and helps where lnL is periodic (an argument of periastron whose posterior
straddles 0 = 2 pi is then one mode, not two on opposite faces of the cube).

ln Z uncertainty: the larger of Skilling's estimate sqrt(H / nlive) and a bootstrap over the run's
threads (``lineage_bootstrap``, the estimate UltraNest's ``num_bootstraps`` makes); likelihood
plateaus (tied values, e.g. the model's -1e30) are retired as a whole (``retire_groups``).
"""
import numpy as np


class NestedResult(dict):
    __getattr__ = dict.get


def _logaddexp(a, b):
    return np.logaddexp(a, b)


def _bounding_ellipsoid(u, enlarge, wrapped=None):
    """Centre, Cholesky factor of the enlarged bounding ellipsoid of points u[n, d]."""
    n, d = u.shape
    ctr = u.mean(axis=0)
    delta = u - ctr
    cov = delta.T @ delta / max(1, n - 1)
    cov += np.eye(d) * 1e-14 * max(1e-300, np.trace(cov) / d)
    try:
        L = np.linalg.cholesky(cov)
    except np.linalg.LinAlgError:
        L = np.diag(np.sqrt(np.maximum(np.diag(cov), 1e-30)))
    y = np.linalg.solve(L, delta.T)
    rmax = np.sqrt(np.max(np.sum(y * y, axis=0)))
    return ctr, L * (rmax * enlarge)


def _draw_in_ellipsoid(rng, ctr, L, n):
    d = len(ctr)
    z = rng.standard_normal((n, d))
    z /= np.linalg.norm(z, axis=1, keepdims=True)
    r = rng.random(n) ** (1.0 / d)
    return ctr + (z * r[:, None]) @ L.T


def nested_sample_ellipsoid(loglike, transform, ndim, nlive=400, ndraw=4096, dlogz=0.5,
                            frac_remain=0.01, enlarge=1.15, seed=0, max_calls=50_000_000,
                            update_interval=None, verbose=False):
    """
    loglike(theta[n, ndim]) -> lnL[n] and transform(u[n, ndim]) -> theta[n, ndim] are the
    vectorised callbacks (UltraNest's ``vectorized=True`` convention).

    Stops when the live points' remaining evidence falls below ``frac_remain`` of the total, or
    their ln Z contribution below ``dlogz`` -- the two UltraNest criteria the reference sets
    (evidence/ultranest/__init__.py:181-185).
    """
    rng = np.random.default_rng(seed)
    u_live = rng.random((nlive, ndim))
    th_live = transform(u_live)
    l_live = np.asarray(loglike(th_live), dtype=np.float64)
    ncall = nlive
    update_interval = update_interval or max(1, nlive // 2)

    logz = -np.inf
    h_info = 0.0
    logx = 0.0  # ln prior volume
    dead_theta, dead_logl, dead_logw = [], [], []
    pool_u = np.zeros((0, ndim))
    pool_th = np.zeros((0, ndim))
    pool_l = np.zeros(0)
    pool_pos = 0
    since_update = update_interval  # force a bound on first use
    ctr = L = None
    it = 0
    log_shrink = np.log1p(-1.0 / (nlive + 1.0))  # E[ln t] per iteration ~ -1/nlive
    while True:
        worst = int(np.argmin(l_live))
        lstar = l_live[worst]
        logx_new = logx - 1.0 / nlive
        logw = np.log(np.exp(logx) - np.exp(logx_new)) if logx > -700 else logx + np.log1p(-np.exp(-1.0 / nlive))
        contrib = lstar + logw
        logz_new = _logaddexp(logz, contrib)
        if np.isfinite(logz_new):
            h_info = (np.exp(contrib - logz_new) * lstar
                      + (np.exp(logz - logz_new) * (h_info + logz) if np.isfinite(logz) else 0.0)
                      - logz_new)
        logz = logz_new
        dead_theta.append(th_live[worst].copy())
        dead_logl.append(lstar)
        dead_logw.append(logw)
        logx = logx_new
        it += 1

        # replacement: next pooled candidate above the new threshold
        found = False
        while not found:
            while pool_pos < len(pool_l):
                k = pool_pos
                pool_pos += 1
                if pool_l[k] > lstar:
                    u_live[worst], th_live[worst], l_live[worst] = pool_u[k], pool_th[k], pool_l[k]
                    found = True
                    break
            if found:
                break
            if since_update >= update_interval or ctr is None:
                ctr, L = _bounding_ellipsoid(u_live, enlarge)
                since_update = 0
            cand = _draw_in_ellipsoid(rng, ctr, L, ndraw)
            inside = np.all((cand >= 0.0) & (cand < 1.0), axis=1)
            cand = cand[inside]
            if len(cand) == 0:
                continue
            pool_u = cand
            pool_th = transform(cand)
            pool_l = np.asarray(loglike(pool_th), dtype=np.float64)
            pool_pos = 0
            ncall += len(cand)
            if ncall > max_calls:
                raise RuntimeError("nested_sample: max_calls exceeded")
        since_update += 1

        # termination on the live points' remaining evidence
        lmax = np.max(l_live)
        log_remain = lmax + logx
        if it % 50 == 0 or True:
            if log_remain - _logaddexp(logz, log_remain) < np.log(frac_remain) or \
                    _logaddexp(logz, log_remain) - logz < dlogz * 1e-3:
                break
        if verbose and it % 500 == 0:
            print(f"it={it} lnZ={logz:.3f} remain={log_remain - logz:.2f} ncall={ncall}")

    # final live-point contribution
    logw_live = logx - np.log(nlive)
    for k in np.argsort(l_live):
        contrib = l_live[k] + logw_live
        logz_new = _logaddexp(logz, contrib)
        h_info = (np.exp(contrib - logz_new) * l_live[k]
                  + np.exp(logz - logz_new) * (h_info + logz) - logz_new)
        logz = logz_new
        dead_theta.append(th_live[k].copy())
        dead_logl.append(l_live[k])
        dead_logw.append(logw_live)
    dead_logl = np.array(dead_logl)
    dead_logw = np.array(dead_logw)
    logwt = dead_logl + dead_logw - logz
    weights = np.exp(logwt - np.max(logwt))
    weights /= weights.sum()
    theta = np.array(dead_theta)
    # equally weighted posterior samples (systematic resampling, seeded)
    nsamp = max(1, int(1.0 / np.sum(weights ** 2)))
    pos = (rng.random() + np.arange(nsamp)) / nsamp
    idx = np.minimum(np.searchsorted(np.cumsum(weights), pos), len(weights) - 1)
    return NestedResult(logz=float(logz), logzerr=float(np.sqrt(max(h_info, 0.0) / nlive)),
                        ncall=int(ncall), niter=int(it), information=float(h_info),
                        samples=theta[idx], weighted_samples=theta, weights=weights,
                        logl=dead_logl, nlive=nlive, seed=seed)



# ------------------------------------------------------------------------------------------
# evidence bookkeeping shared by the samplers: tie-aware retirement and the lineage bootstrap
# ------------------------------------------------------------------------------------------
def retire_groups(l_sorted, n_live):
    """
    Shrinkage bookkeeping for retiring the points with (ascending) log-likelihoods ``l_sorted`` from
    a set of ``n_live`` live points, one after the other.  Returns (dlogx[len], logw_rel[len]): the
    change of ln X caused by each point and its ln weight relative to ln X at the start.

    Distinct values: the classic E[ln t] = -1/n with n = n_live, n_live - 1, ...  A group of g points
    with the SAME value (a likelihood plateau -- e.g. the -1e30 the model returns for an invalid
    Keplerian, evidence/rvmodel/__init__.py:198-203) is retired as a whole: X shrinks by
    (n - g) / n and every member gets 1/g of that shell (Fowlie, Handley & Su 2020; UltraNest does
    the same).  Charging each tied point its own 1/n instead over-estimates X whenever the
    replacements are drawn from L > L_plateau, and with it ln Z (+0.17 for a 70 % plateau).
    """
    l_sorted = np.asarray(l_sorted, dtype=np.float64)
    m = len(l_sorted)
    dlogx, logw_rel = np.empty(m), np.empty(m)
    n_cur, logx, i = int(n_live), 0.0, 0
    while i < m:
        j = i
        while j + 1 < m and l_sorted[j + 1] == l_sorted[i]:
            j += 1
        g = j - i + 1
        if g >= n_cur:
            raise ValueError("every live point has the same log-likelihood: nothing to integrate")
        step = -1.0 / n_cur if g == 1 else np.log((n_cur - g) / n_cur)
        shell = logx + np.log1p(-np.exp(step))  # ln (X_before - X_after)
        logw_rel[i:j + 1] = shell - np.log(g)
        dlogx[i:j + 1] = step / g
        logx += step
        n_cur -= g
        i = j + 1
    return dlogx, logw_rel


def lineage_bootstrap(birth, death, root, n_roots, rng, num=30):
    """
    Scatter of ln Z under resampling of the run's THREADS (what UltraNest's ``num_bootstraps``
    estimates, evidence/ultranest/__init__.py:172, and nestcheck's bootstrap, Higson et al. 2018): a
    run with n live points is n single-live-point runs merged -- the thread of a slot is the sequence
    of points that occupied it, each born under the constraint at which its predecessor was replaced
    (``root`` = slot).  A bootstrap draws n_roots threads with replacement, keeps their points (with
    multiplicity) and integrates the evidence again with the number of live points THOSE threads had
    at each death.  It contains the shrinkage noise that Skilling's sqrt(H/n) estimates and adds the
    variance of how the posterior mass is spread over the threads; like every within-run estimate it
    cannot see a mode that no live point ever found.
    Returns (std of ln Z over the bootstraps, the ln Z values).
    """
    birth, death = np.asarray(birth, dtype=np.float64), np.asarray(death, dtype=np.float64)
    root = np.asarray(root)
    order = np.argsort(death, kind="stable")
    birth, death, root = birth[order], death[order], root[order]
    birth_sorted_idx = np.argsort(birth, kind="stable")
    out = []
    for _ in range(int(num)):
        mult = np.bincount(rng.integers(0, n_roots, n_roots), minlength=n_roots)[root].astype(np.float64)
        # live count just before death i: points born below L_i minus points that died below L_i
        born = np.concatenate([[0.0], np.cumsum(mult[birth_sorted_idx])])
        n_born = born[np.searchsorted(birth[birth_sorted_idx], death, side="left")]
        dead_before = np.concatenate([[0.0], np.cumsum(mult)])[:-1]
        n_alive = n_born - dead_before
        use = (mult > 0) & (n_alive > 0)
        if use.sum() < 2:
            continue
        # each kept point (multiplicity c) compresses ln X by c / n_alive
        dl = np.where(use, mult / np.maximum(n_alive, 1e-300), 0.0)
        logx_after = -np.cumsum(dl)
        logx_before = logx_after + dl
        with np.errstate(divide="ignore"):
            logw = np.where(use, logx_before + np.log1p(-np.exp(-np.maximum(dl, 1e-300))), -np.inf)
        terms = death + logw
        mx = np.max(terms[np.isfinite(terms)])
        out.append(mx + np.log(np.sum(np.exp(terms[np.isfinite(terms)] - mx))))
    out = np.array(out)
    return (float(np.std(out)) if len(out) > 1 else 0.0), out

# ------------------------------------------------------------------------------------------
# slice-sampling replacement (default)
# ------------------------------------------------------------------------------------------
def wrap_mask(wrapped, ndim):
    """The circular coordinates as a bool array [ndim] (all False for None)."""
    if wrapped is None:
        return np.zeros(ndim, dtype=bool)
    w = np.asarray(wrapped, dtype=bool).reshape(-1)
    if w.shape != (ndim,):
        raise ValueError(f"wrapped: {len(w)} entries for {ndim} dimensions")
    return w


def wrap_unit(p):
    """p modulo 1: p - floor(p) (exact), and 0 where that rounds to 1.0 -- only for p in
    (-2^-54, 0), where 1 is the same point as 0.  The rule of rvl_slice_phase_wrapped."""
    q = p - np.floor(p)
    return np.where(q >= 1.0, 0.0, q)


def recentre(u, wrapped):
    """u[n, d] with every circular coordinate j moved to frac(u_j - mu_j + 1/2), mu_j the circular
    mean atan2(mean sin 2 pi u_j, mean cos 2 pi u_j) / 2 pi: a mode that straddles the seam then
    lies in the middle of [0, 1), and its covariance does not depend on where it sits."""
    ang = 2.0 * np.pi * u[:, wrapped]
    mu = np.arctan2(np.sin(ang).mean(axis=0), np.cos(ang).mean(axis=0)) / (2.0 * np.pi)
    v = u.copy()
    v[:, wrapped] = wrap_unit(u[:, wrapped] - mu + 0.5)
    return v


def _whitening(u, wrapped=None):
    """Lower Cholesky factor of the covariance of the live points u[n, d]; circular coordinates
    (``wrapped``, a bool mask with at least one True) about their circular mean."""
    if wrapped is not None:
        u = recentre(u, wrapped)
    d = u.shape[1]
    cov = np.cov(u.T).reshape(d, d) + np.eye(d) * 1e-18
    try:
        return np.linalg.cholesky(cov)
    except np.linalg.LinAlgError:
        return np.diag(np.sqrt(np.maximum(np.diag(cov), 1e-30)))


def _slice_moves(rng, loglike, transform, u, lmin, chol, nsteps, max_expand=16, max_shrink=64,
                 fused=None, speculate=None, wrapped=None):
    """Advance k walkers u[k, d] by nsteps slice moves under L > lmin; all evaluations batched.
    ``fused(u) -> (theta, lnL)``, when given, replaces the transform + loglike pair of every
    evaluation by one call (one device round trip instead of two).  ``speculate`` = m: every call
    evaluates the next m stepping-out positions of both sides, and then the next m shrinkage
    candidates, of every walker at once.  The chain is EXACTLY the sequential one (m = 1) -- the
    extra evaluations are discarded -- but it needs ~3x fewer, larger device calls, which is
    what a latency-bound accelerator wants.  None: chosen from the number of walkers.  ``wrapped``
    (bool mask with at least one True, or None): those coordinates of every candidate are taken
    modulo 1 before the cube test, and an accepted candidate keeps the wrapped value."""
    k, d = u.shape
    theta = transform(u)
    lcur = np.full(k, np.nan)
    ncall = 0

    def evaluate(points, mask):
        """lnL of points[mask] (inside the cube only); -inf elsewhere."""
        nonlocal ncall
        out = np.full(len(points), -np.inf)
        th = np.zeros_like(points)
        idx = np.where(mask & np.all((points >= 0.0) & (points < 1.0), axis=1))[0]
        if len(idx):
            if fused is not None:
                th[idx], out[idx] = fused(points[idx])
            else:
                th[idx] = transform(points[idx])
                out[idx] = loglike(th[idx])
            ncall += len(idx)
        return out, th

    # look-ahead depth: enough to fill a device call (a call costs the same up to ~1e3 points),
    # none when the walkers alone already do (the host bookkeeping then dominates)
    m = max(1, min(6, 512 // max(1, k))) if speculate is None else max(1, int(speculate))
    for _ in range(nsteps):
        z = rng.standard_normal((k, d))
        z /= np.linalg.norm(z, axis=1, keepdims=True)
        dirn = z @ chol.T
        r = rng.random(k)
        lo, hi = -r, 1.0 - r
        # ---- stepping out: both sides and the next m unit steps of each in ONE call.  The edge
        # positions lo, lo-1, ... do not depend on earlier results, so evaluating m of them ahead
        # and keeping the run of successes is the sequential rule evaluated speculatively.
        grow_lo, grow_hi = np.ones(k, dtype=bool), np.ones(k, dtype=bool)
        done_lo, done_hi = np.zeros(k, dtype=int), np.zeros(k, dtype=int)
        steps = np.arange(m)
        while grow_lo.any() or grow_hi.any():
            e_lo, e_hi = np.empty((k, m)), np.empty((k, m))
            a_lo, a_hi = lo, hi
            for j in range(m):  # unit steps applied one by one: the roundings of the sequential rule
                e_lo[:, j], e_hi[:, j] = a_lo, a_hi
                a_lo, a_hi = a_lo - 1.0, a_hi + 1.0
            edges = np.concatenate([e_lo, e_hi], axis=1)                      # [k, 2m]
            mask = np.concatenate([grow_lo[:, None] & (done_lo[:, None] + steps[None, :] < max_expand),
                                   grow_hi[:, None] & (done_hi[:, None] + steps[None, :] < max_expand)],
                                  axis=1)
            pts = u[:, None, :] + edges[:, :, None] * dirn[:, None, :]
            if wrapped is not None:
                pts[..., wrapped] = wrap_unit(pts[..., wrapped])
            l_e, _ = evaluate(pts.reshape(-1, d), mask.reshape(-1))
            above = (l_e.reshape(k, 2 * m) > lmin) & mask
            run_lo = np.cumprod(above[:, :m], axis=1).sum(axis=1)              # leading successes
            run_hi = np.cumprod(above[:, m:], axis=1).sum(axis=1)
            for j in range(m):
                lo = np.where(run_lo > j, lo - 1.0, lo)
                hi = np.where(run_hi > j, hi + 1.0, hi)
            done_lo += run_lo
            done_hi += run_hi
            grow_lo &= (run_lo == m) & (done_lo < max_expand)
            grow_hi &= (run_hi == m) & (done_hi < max_expand)
        # ---- shrinkage: the next m candidates of a walker, generated as if each one before it were
        # rejected (which is the only case in which the sequential rule would draw it), in ONE call;
        # the first accepted one is taken.  Same chain as one candidate per call.
        pending = np.ones(k, dtype=bool)
        draws = rng.random((max_shrink, k))
        it = 0
        while it < max_shrink and pending.any():
            mm = min(m, max_shrink - it)
            lo_s, hi_s = lo.copy(), hi.copy()
            T = np.empty((k, mm))
            for j in range(mm):
                t = lo_s + (hi_s - lo_s) * draws[it + j]
                T[:, j] = t
                lo_s = np.where(t < 0, t, lo_s)
                hi_s = np.where(t >= 0, t, hi_s)
            cand = u[:, None, :] + T[:, :, None] * dirn[:, None, :]            # [k, mm, d]
            if wrapped is not None:
                cand[..., wrapped] = wrap_unit(cand[..., wrapped])
            l_c, th_c = evaluate(cand.reshape(-1, d), np.repeat(pending, mm))
            l_c = l_c.reshape(k, mm)
            acc = l_c > lmin
            hit = pending & acc.any(axis=1)
            first = np.argmax(acc, axis=1)
            rows = np.where(hit)[0]
            if len(rows):
                sel = first[rows]
                u[rows] = cand[rows, sel]
                theta[rows] = th_c.reshape(k, mm, d)[rows, sel]
                lcur[rows] = l_c[rows, sel]
            pending &= ~hit
            lo = np.where(pending, lo_s, lo)
            hi = np.where(pending, hi_s, hi)
            it += mm
        # walkers that never found a point keep their position (the bracket collapsed)
    return u, theta, lcur, ncall


def nested_sample(loglike, transform, ndim, nlive=400, ndraw=4096, dlogz=0.5, frac_remain=0.01,
                  seed=0, nsteps=None, batch_fraction=0.2, method="slice", max_calls=500_000_000,
                  verbose=False, fused=None, speculate=None, num_bootstraps=30, wrapped=None, **kw):
    """
    Seeded vectorised nested sampling; see the module docstring.  ``loglike(theta[n, ndim])`` and
    ``transform(u[n, ndim])`` follow UltraNest's ``vectorized=True`` convention.  Returns a
    ``NestedResult`` (logz, logzerr, ncall, niter, samples, ...).  ``fused(u[n, ndim]) ->
    (theta[n, ndim], lnL[n])`` (method='slice'): the device's fused u -> theta -> lnL call; it must
    return what ``transform`` followed by ``loglike`` returns, and then the run is identical.
    ``wrapped`` (bool per dimension, UltraNest's ``wrapped_params``): circular coordinates of the
    slice method (module docstring); None or no True leaves the run exactly as without it.  The
    result's ``wrapped`` holds the mask.
    """
    wmask = wrap_mask(wrapped, ndim)
    if method == "ellipsoid":
        if wmask.any():
            # an ellipsoid longer than 1 along a circular axis covers some points twice: its
            # proposal would not be uniform on the torus
            raise ValueError("method='ellipsoid' does not support wrapped (circular) coordinates")
        res = nested_sample_ellipsoid(loglike, transform, ndim, nlive=nlive, ndraw=ndraw,
                                      dlogz=dlogz, frac_remain=frac_remain, seed=seed,
                                      max_calls=max_calls, verbose=verbose, **kw)
        res["wrapped"] = wmask
        return res
    wrap = wmask if wmask.any() else None
    rng = np.random.default_rng(seed)
    nsteps = nsteps or max(4, 3 * ndim)  # the reference's default (evidence/ultranest/__init__.py:335)
    k = max(1, min(int(batch_fraction * nlive), nlive - 2, ndraw))
    u_live = rng.random((nlive, ndim))
    th_live = transform(u_live)
    l_live = np.asarray(loglike(th_live), dtype=np.float64).copy()
    ncall = nlive
    logz, h_info, logx = -np.inf, 0.0, 0.0
    dead_theta, dead_logl, dead_logw = [], [], []
    # threads: the slot a point occupies, and the constraint it was born under (lineage_bootstrap)
    root_live, birth_live = np.arange(nlive), np.full(nlive, -np.inf)
    dead_root, dead_birth = [], []
    niter = 0

    def absorb(lval, logw):
        nonlocal logz, h_info
        contrib = lval + logw
        new = np.logaddexp(logz, contrib)
        if np.isfinite(new):
            h_info = (np.exp(contrib - new) * lval
                      + (np.exp(logz - new) * (h_info + logz) if np.isfinite(logz) else 0.0) - new)
        logz = new

    while True:
        order = np.argsort(l_live, kind="stable")
        # the k worst -- and everything tied with the k-th: a plateau is retired as a whole, before
        # any replacement is drawn from above it (retire_groups)
        kk = k
        while kk < nlive - 2 and l_live[order[kk]] == l_live[order[k - 1]]:
            kk += 1
        worst = order[:kk]
        dlogx, logw_rel = retire_groups(l_live[worst], nlive)
        for i, j in enumerate(worst):
            absorb(l_live[j], logx + logw_rel[i])
            dead_theta.append(th_live[j].copy())
            dead_logl.append(l_live[j])
            dead_logw.append(logx + logw_rel[i])
            dead_root.append(root_live[j])
            dead_birth.append(birth_live[j])
            niter += 1
        logx += float(np.sum(dlogx))
        lmin = l_live[worst[-1]]
        keep = order[kk:]
        chol = _whitening(u_live[keep], wrap)
        starts = keep[rng.integers(0, len(keep), kk)]
        u_new, th_new, l_new, nc = _slice_moves(rng, loglike, transform, u_live[starts].copy(),
                                                lmin, chol, nsteps, fused=fused,
                                                speculate=speculate, wrapped=wrap)
        ncall += nc
        stuck = ~np.isfinite(l_new)  # a walker that never moved is a copy of its start point
        l_new = np.where(stuck, l_live[starts], l_new)
        th_new[stuck] = th_live[starts][stuck]
        u_live[worst], th_live[worst], l_live[worst] = u_new, th_new, l_new
        birth_live[worst] = lmin  # (the thread of a slot continues with the point written into it)
        if ncall > max_calls:
            raise RuntimeError("nested_sample: max_calls exceeded")
        log_remain = np.max(l_live) + logx
        total = np.logaddexp(logz, log_remain)
        if verbose and (niter // k) % 20 == 0:
            print(f"it={niter} lnZ={logz:.3f} ln(remain/Z)={log_remain - logz:.2f} ncall={ncall}")
        # UltraNest's two criteria (evidence/ultranest/__init__.py:181-185): remaining fraction
        # of the evidence in the live points, and their possible ln Z contribution
        if log_remain - total < np.log(frac_remain) and total - logz < dlogz:
            break

    logw_live = logx - np.log(nlive)
    for j in np.argsort(l_live, kind="stable"):
        absorb(l_live[j], logw_live)
        dead_theta.append(th_live[j].copy())
        dead_logl.append(l_live[j])
        dead_logw.append(logw_live)
        dead_root.append(root_live[j])
        dead_birth.append(birth_live[j])
    dead_logl, dead_logw = np.array(dead_logl), np.array(dead_logw)
    logwt = dead_logl + dead_logw - logz
    weights = np.exp(logwt - np.max(logwt))
    weights /= weights.sum()
    theta = np.array(dead_theta)
    nsamp = max(1, int(1.0 / np.sum(weights ** 2)))
    pos = (rng.random() + np.arange(nsamp)) / nsamp
    idx = np.minimum(np.searchsorted(np.cumsum(weights), pos), len(weights) - 1)
    skilling = float(np.sqrt(max(h_info, 0.0) / nlive))
    bs_std, bs = lineage_bootstrap(dead_birth, dead_logl, dead_root, nlive,
                                   np.random.default_rng([int(seed), 0xB007]), num_bootstraps)
    # reported uncertainty: the thread bootstrap (which contains the shrinkage noise) where it is
    # larger than Skilling's estimate
    return NestedResult(logz=float(logz), logzerr=float(max(skilling, bs_std)),
                        logzerr_skilling=skilling, logzerr_bootstrap=bs_std,
                        ncall=int(ncall), niter=int(niter), information=float(h_info),
                        samples=theta[idx], weighted_samples=theta, weights=weights,
                        logl=dead_logl, nlive=nlive, seed=seed, method="slice", wrapped=wmask)
