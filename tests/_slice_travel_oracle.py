"""
Host restatement of the adaptive-moves kernels of evidence_b200/csrc/rvslice.cu
(`rvl_slice_runs_radius`, `rvl_slice_runs_travel`).

TEST INFRASTRUCTURE ONLY.  Every value is formed in the kernels' operation order, one IEEE rounding
per operation (the library is built with -fmad=false and IEEE division), so the results are
reproduced bit for bit:
  Linv = L^-1 column by column: Linv_cc = 1 / L_cc, Linv_ic = -(s / L_ii) with
         s = 0, s = s + L_il Linv_lc for l = c .. i - 1
  y_i  = 0, y_i = y_i + Linv_il delta_l for l = 0 .. i
  D    = 0, D = D + y_i y_i for i = 0 .. d - 1
with delta = a - b and delta_c - rint(delta_c) (half to even) in a circular coordinate.

The loops below run over all indices at once and add the terms of the zero triangle too: a term
0 * x is a signed zero, and adding it changes neither a nonzero sum nor the +0 a sum starts from
(x + (-0) = x, +0 + (-0) = +0), so the sums are the kernels' sums.
"""
import numpy as np


def linv(L):
    """L^-1 of a lower factor L [d][d], in the kernel's order (the upper triangle is +0)."""
    d = L.shape[0]
    X = np.zeros((d, d))
    for i in range(d):
        s = np.zeros(d)
        for l in range(i):
            s = s + L[i, l] * X[l, :]  # column c takes the terms l >= c; X[l, c] = +0 for c > l
        X[i, :i] = -(s[:i] / L[i, i])
        X[i, i] = 1.0 / L[i, i]
    return X


def delta(a, b, wrap=None):
    """a - b [..., d]; a circular coordinate minus its nearest integer (half to even)."""
    x = a - b
    if wrap is not None and np.any(wrap):
        w = np.asarray(wrap, bool)
        x = np.where(w, x - np.rint(x), x)
    return x


def dist2(a, b, X, wrap=None):
    """D(a, b) = |X delta|^2 for points a, b [P, d] (X = linv(L)), in the kernel's order."""
    dl = delta(a, b, wrap)
    d = X.shape[0]
    y = np.zeros(dl.shape)
    for l in range(d):
        y = y + dl[:, l:l + 1] * X[:, l][None, :]  # y_i takes the terms l <= i; X[i, l] = +0 for l > i
    D = np.zeros(dl.shape[0])
    for i in range(d):
        D = D + y[:, i] * y[:, i]
    return D


def radius(u_live, order, kk, chol, wrap=None, rad2=None):
    """rad2[R]: for each run with kk[r] > 0, the max over its survivors u_live[r][order[r][kk[r]:]] of
    the min over the other survivors of D; 0 with fewer than two; runs with kk[r] = 0 keep rad2[r]
    (default 0)."""
    R = u_live.shape[0]
    out = np.zeros(R) if rad2 is None else np.array(rad2, dtype=np.float64)
    for r in range(R):
        if int(kk[r]) <= 0:
            continue
        pts = u_live[r][np.asarray(order[r][int(kk[r]):])]
        n = len(pts)
        if n < 2:
            out[r] = 0.0
            continue
        X = linv(chol[r])
        best = 0.0
        for i in range(n):
            D = dist2(np.repeat(pts[i:i + 1], n, 0), pts, X, wrap)
            D[i] = np.inf
            best = max(best, float(np.fmin.reduce(D)))
        out[r] = best
    return out


def travel(u_end, run_of, start, u_live, kk, chol, rad2, wrap=None, far=None):
    """far[R]: for each run with kk[r] > 0, the number of walkers w with run_of[w] = r and
    D(u_end[w], u_live[r][start[w]]) > rad2[r]; runs with kk[r] = 0 keep far[r] (default 0)."""
    R = u_live.shape[0]
    out = np.zeros(R, np.int32) if far is None else np.array(far, dtype=np.int32)
    run_of, start = np.asarray(run_of), np.asarray(start)
    for r in range(R):
        if int(kk[r]) <= 0:
            continue
        w = np.flatnonzero(run_of == r)
        if len(w) == 0:
            out[r] = 0
            continue
        D = dist2(u_end[w], u_live[r][start[w]], linv(chol[r]), wrap)
        out[r] = int(np.count_nonzero(D > rad2[r]))
    return out
