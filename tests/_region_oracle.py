"""
Host restatement of the MLFriends region kernels of evidence_b200/csrc/rvslice.cu
(`rvl_region_runs_radius`, `rvl_region_runs_draw`, `rvl_region_runs_pick`).

TEST INFRASTRUCTURE ONLY.  The random words come from the generator of `oracle.slice_oracle`
(Philox4x32-10, the seed as key, `u01`) with the kernels' counters; distances are `dist2` of
tests/_slice_travel_oracle.py, in the kernels' operation order.  The radius and the pick are
therefore reproduced bit for bit.  A candidate of the draw kernel goes through log, sin, cos and pow,
which are not correctly rounded on the device: its coordinates agree to about 1e-15, and its accept
flag can differ only where a test sits within that of a ball surface or a cube face (``near``).

``nearest_image=False`` / ``first_ball=False`` drop rule 4 / rule 7 of the draw (for the tests that
show each rule is needed for a uniform density); the kernels always apply both.
"""
import numpy as np

import _slice_travel_oracle as to
from oracle import slice_oracle as so

TAG_BOOT, TAG_REGION = 0x42540000, 0x52000000
TWO_PI = 6.283185307179586
NEAR = 1e-12


def _wrap_unit(p):
    q = p - np.floor(p)
    return np.where(q >= 1.0, 0.0, q)


def boot_chosen(seed, round_no, b, n):
    """The survivors drawn by bootstrap b (bool [n]): index 4q + t is floor(word_t n / 2^32) of the
    words (x, y, z, w) of counter (round, TAG_BOOT + b, q, 0)."""
    q = np.arange((n + 3) // 4, dtype=np.uint64)
    x, y, z, w = so.draw(seed, round_no, TAG_BOOT + b, q)
    words = np.stack([x, y, z, w], 1).reshape(-1)[:n]
    chosen = np.zeros(n, dtype=bool)
    chosen[((words * np.uint64(n)) >> np.uint64(32)).astype(np.int64)] = True
    return chosen


def radius(seeds, u_live, order, kk, chol, nboot, round_no, wrap=None, rad2=None):
    """rad2[R]: for each run with kk[r] > 0, the max over bootstraps b < nboot of rho2_b = max over the
    survivors not drawn of min over the drawn ones of D (0 when none is left out); runs with kk[r] = 0
    keep rad2[r] (default 0)."""
    R = u_live.shape[0]
    out = np.zeros(R) if rad2 is None else np.array(rad2, dtype=np.float64)
    for r in range(R):
        k = int(kk[r])
        if k <= 0:
            continue
        pts = u_live[r][np.asarray(order[r][k:])]
        n = len(pts)
        X = to.linv(chol[r])
        best = 0.0
        for b in range(nboot):
            chosen = boot_chosen(seeds[r], round_no, b, n)
            left, sel = pts[~chosen], pts[chosen]
            if len(left) == 0:
                continue
            a = np.repeat(left, len(sel), 0)
            c = np.tile(sel, (len(left), 1))
            D = to.dist2(a, c, X, wrap).reshape(len(left), len(sel))
            best = max(best, float(np.fmin.reduce(D, axis=1).max()))
        out[r] = best
    return out


def draw(seeds, u_live, order, kk, chol, rad2, slot_base, batch, round_no, wrap=None, nearest_image=True,
         first_ball=True):
    """The draw kernel for every slot: (x [S, d], flag [S] bool, near [S] bool, count [R], offs [R + 1],
    cand [offs[R], d]).  x is every slot's candidate (also where rejected); near marks the slots whose
    flag rests on a comparison within NEAR (relative) of its bound."""
    R, nlive, d = u_live.shape
    slot_base = np.asarray(slot_base, dtype=np.int64)
    S = int(slot_base[-1])
    x_all, flag, near = np.full((S, d), np.nan), np.zeros(S, bool), np.zeros(S, bool)
    circ = np.zeros(d, bool) if wrap is None else np.asarray(wrap, bool)
    tag = TAG_REGION + (int(batch) << 8)
    for r in range(R):
        k, s0, ns = int(kk[r]), int(slot_base[r]), int(slot_base[r + 1] - slot_base[r])
        if k <= 0 or ns <= 0:
            continue
        pts = u_live[r][np.asarray(order[r][k:])]
        n = len(pts)
        s = np.arange(ns, dtype=np.uint64)
        x0, _, z0, w0 = so.draw(seeds[r], round_no, tag, s)
        i = ((x0 * np.uint64(n)) >> np.uint64(32)).astype(np.int64)
        v = so.u01(z0, w0)
        Z = np.empty((ns, d))
        for c in range(d):
            x, y, z, w = so.draw(seeds[r], round_no, tag + 1 + (c >> 1), s)
            rad = np.sqrt(-2.0 * np.log(so.u01(x, y)))
            ang = TWO_PI * so.u01(z, w)
            Z[:, c] = rad * np.sin(ang) if c & 1 else rad * np.cos(ang)
        n2 = np.zeros(ns)
        for c in range(d):
            n2 = n2 + Z[:, c] * Z[:, c]
        scale = np.sqrt(rad2[r]) * (v ** (1.0 / d) / np.sqrt(n2))
        L = chol[r]
        ok, nr = np.ones(ns, bool), np.zeros(ns, bool)
        x = np.empty((ns, d))
        for c in range(d):
            acc = np.zeros(ns)
            for l in range(c + 1):
                acc = acc + L[c, l] * Z[:, l]
            dc = scale * acc
            p = pts[i, c] + dc
            if circ[c]:
                if nearest_image:
                    ok &= np.abs(dc) <= 0.5
                    nr |= np.abs(np.abs(dc) - 0.5) <= NEAR
                x[:, c] = _wrap_unit(p)
            else:
                ok &= (p >= 0.0) & (p < 1.0)
                nr |= (np.abs(p) <= NEAR) | (np.abs(p - 1.0) <= NEAR)
                x[:, c] = p
        if first_ball:
            X = to.linv(L)
            for j in range(n - 1):
                before = j < i
                if not before.any():
                    continue
                D = to.dist2(x, np.repeat(pts[j:j + 1], ns, 0), X, wrap)
                ok &= ~(before & (D <= rad2[r]))
                nr |= before & (np.abs(D - rad2[r]) <= NEAR * rad2[r])
        x_all[s0:s0 + ns], flag[s0:s0 + ns], near[s0:s0 + ns] = x, ok, nr
    count = np.array([int(flag[slot_base[r]:slot_base[r + 1]].sum()) for r in range(R)], np.int64)
    offs = np.concatenate([[0], np.cumsum(count)])
    return x_all, flag, near, count, offs, x_all[flag]


def pick(kk, lmin, offs, cand, cand_th, cand_ll, run_of, walker_of, u, theta, lcur, filled):
    """The pick kernel on copies of the walker buffers: (u, theta, lcur, filled, above)."""
    u, theta, lcur = u.copy(), theta.copy(), lcur.copy()
    R = len(kk)
    filled, above = np.array(filled, dtype=np.int64), np.zeros(R, np.int64)
    for r in range(R):
        need = int(kk[r])
        if need <= 0:
            continue
        rows = np.arange(offs[r], offs[r + 1])
        rows = rows[cand_ll[rows] > lmin[r]]
        f0 = int(filled[r])
        for w in np.flatnonzero(np.asarray(run_of) == r):
            t = int(walker_of[w]) - f0
            if 0 <= t < len(rows) and int(walker_of[w]) < need:
                u[w], theta[w], lcur[w] = cand[rows[t]], cand_th[rows[t]], cand_ll[rows[t]]
        filled[r] = min(need, f0 + len(rows))
        above[r] = len(rows)
    return u, theta, lcur, filled, above
