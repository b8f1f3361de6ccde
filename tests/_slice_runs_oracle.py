"""
Host restatement of the ensemble set-up kernels of evidence_b200/csrc/rvslice.cu
(`rvl_slice_runs_init`, `rvl_slice_runs_whiten`, `rvl_slice_runs_starts`).

TEST INFRASTRUCTURE ONLY.  The random draws reuse the generator of `oracle.slice_oracle` (Philox4x32-10,
the seed as key, `u01`), so the initial points and starts are reproduced bit for bit.  The whitening
is restated in the kernel's operation order (sums over the survivors in order, one rounding per
operation: the library is built with -fmad=false and IEEE division and square root), so without
circular coordinates it is reproduced bit for bit too; with them it depends on the device's sin, cos
and atan2, which are not correctly rounded.
"""
import numpy as np

from oracle import slice_oracle as so

TAG_INIT, TAG_START = 0x494E0000, 0x53540000
TWO_PI = 6.283185307179586


def init_points(seeds, nlive, d):
    """u_live[R][nlive][d]: coordinate c of point p of run r is the u01 of counter
    (0, TAG_INIT + c // 2, p, 0) under seeds[r], words (x, y) for even c and (z, w) for odd c."""
    out = np.empty((len(seeds), nlive, d))
    p = np.arange(nlive, dtype=np.uint64)[:, None]
    c = np.arange(d, dtype=np.uint64)[None, :]
    for r, seed in enumerate(seeds):
        x, y, z, w = so.draw(seed, 0, np.uint64(TAG_INIT) + (c >> np.uint64(1)), p)
        out[r] = np.where((c & np.uint64(1)) == 1, so.u01(z, w), so.u01(x, y))
    return out


def start_slots(seeds, nlive, order, kk, run_of, walker_of, round_no):
    """The start slot of every walker: survivor floor(x n / 2^32) of its run, x the first word of
    counter (round, TAG_START, j, 0) under the run's seed, n = nlive - kk[r]."""
    slots = np.empty(len(run_of), dtype=np.int64)
    for w, (r, j) in enumerate(zip(run_of, walker_of)):
        x, _, _, _ = so.draw(seeds[r], round_no, TAG_START, np.uint64(j))
        n = nlive - int(kk[r])
        slots[w] = order[r][int(kk[r]) + ((int(x) * n) >> 32)]
    return slots


def _wrap_unit(p):
    q = p - np.floor(p)
    return np.where(q >= 1.0, 0.0, q)


def whiten(u_live, order, kk, wrap=None):
    """(chol [R][d][d], failed [R]) in the kernel's order: circular means, means, covariance
    (sum over the survivors in order, / (n - 1), + 1e-18 on the diagonal), then Cholesky column by
    column (pivot: cov_jj - L_j0^2 - L_j1^2 - .., sequentially; below it: (cov_ij - sum_l L_il L_jl)
    / pivot); diag(sqrt(max(cov_jj, 1e-30))) where a pivot is not > 0.  A run with kk = 0 is
    skipped (its factor stays 0 here)."""
    R, nlive, d = u_live.shape
    wrap = np.zeros(d, bool) if wrap is None else np.asarray(wrap, bool)
    out, failed = np.zeros((R, d, d)), np.zeros(R, bool)
    for r in range(R):
        if int(kk[r]) == 0:
            continue
        rows = np.asarray(order[r][int(kk[r]):])
        n = len(rows)
        x = u_live[r][rows]  # [n, d]
        v = x.copy()
        for c in np.flatnonzero(wrap):
            ss = cs = 0.0
            for i in range(n):
                ang = TWO_PI * x[i, c]
                ss += np.sin(ang)
                cs += np.cos(ang)
            mu = np.arctan2(ss / n, cs / n) / TWO_PI
            v[:, c] = _wrap_unit(x[:, c] - mu + 0.5)
        mean = np.zeros(d)
        for i in range(n):
            mean = mean + v[i]
        mean = mean / n
        dev = v - mean
        acc = np.zeros((d, d))
        for i in range(n):
            acc = acc + dev[i][:, None] * dev[i][None, :]
        cov = np.tril(acc / (n - 1))
        cov[np.diag_indices(d)] += 1e-18
        L = cov.copy()
        ok = True
        for j in range(d):
            s = L[j, j]
            for l in range(j):
                s = s - L[j, l] * L[j, l]
            if not s > 0.0:
                ok = False
                break
            L[j, j] = np.sqrt(s)
            for i in range(j + 1, d):
                t = L[i, j]
                for l in range(j):
                    t = t - L[i, l] * L[j, l]
                L[i, j] = t / L[j, j]
        if not ok:
            L = np.diag(np.sqrt(np.fmax(np.diag(cov), 1e-30)))
        out[r], failed[r] = L, not ok
    return out, failed
