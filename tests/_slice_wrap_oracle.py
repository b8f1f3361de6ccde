"""
Host restatement of `rvl_slice_phase_wrapped` (evidence_b200/csrc/rvslice.cu, the kWrap = true
kernels): the phases of oracle/slice_oracle.py with circular coordinates.

TEST INFRASTRUCTURE ONLY.  It reuses the generator, the direction and the bookkeeping of
`oracle.slice_oracle` and restates the three places where a candidate is written: a coordinate of
the mask `wrap` ([d] bool) is stored as `wrap_unit(p)` instead of the clamped p, and it never
makes the candidate outside the cube.  floor and the subtraction are exact, so the device matches
this bit for bit from its direction onward, as it matches the unwrapped oracle.  The mask is an
argument, not part of the `SliceState`, which stays that of the unwrapped oracle.
"""
import numpy as np

from oracle import slice_oracle as so


def wrap_unit(p):
    """A circular coordinate taken modulo 1: q = p - floor(p) (exact), and q = 0 where that rounds
    to 1.0 -- only for p in (-2^-54, 0), where 1 is the same point as 0.  Result in [0, 1)."""
    p = np.asarray(p, dtype=np.float64)
    q = p - np.floor(p)
    return np.where(q >= 1.0, 0.0, q)


def candidates(u, dirn, t, wrap):
    """write_candidate<kWrap> for every walker: p = u + t d (t [k] or [k, n]); returns (stored
    points, inside flags).  Coordinates of the mask are stored as wrap_unit(p) and do not take part
    in the inside test; the others are clamped and tested as in so._candidates."""
    t = np.asarray(t, dtype=np.float64)
    if t.ndim == 1:
        p = u + t[:, None] * dirn
    else:
        p = u[:, None, :] + t[:, :, None] * dirn[:, None, :]
    wrap = np.asarray(wrap, dtype=bool)
    inside = ((p >= 0.0) & (p < 1.0)) | wrap
    out = np.where(wrap, wrap_unit(p), np.fmin(np.fmax(p, 0.0), so.HI_CLAMP))
    return out, inside.all(axis=-1).astype(np.uint8)


def slice_begin(st, wrap, dirn=None):
    """Phase 0 (so.slice_begin with wrapped stepping-out candidates).  Returns (z, the oracle's own
    direction)."""
    z = so.normals(st)
    own = so.direction(st, z)
    st.dirn = own.copy() if dirn is None else np.array(dirn, dtype=np.float64).reshape(st.k, st.d)
    x, y, _, _ = so.draw(st.seed, st.move, so.TAG_BRACKET, np.arange(st.k, dtype=np.uint64))
    r0 = so.u01(x, y)
    lo, hi = -r0, 1.0 - r0
    st.lo, st.hi = lo, hi
    st.pending = np.ones(st.k, dtype=np.int32)
    steps = np.arange(st.n_out, dtype=np.float64)
    t = np.concatenate([lo[:, None] - steps[None, :], hi[:, None] + steps[None, :]], axis=1)
    st.cand_out, st.inside_out = candidates(st.u, st.dirn, t, wrap)
    return z, own


def _propose_shrink(st, wrap, rows, lo, hi):
    """so._propose_shrink with wrapped shrinkage candidates."""
    lo, hi = lo.copy(), hi.copy()
    walkers = rows.astype(np.uint64)
    u, dirn = st.u[rows], st.dirn[rows]
    for j in range(st.m):
        tag = (so.TAG_SHRINK + st.shrink_round * 64 + j) & 0xFFFFFFFF
        x, y, _, _ = so.draw(st.seed, st.move, tag, walkers)
        t = lo + (hi - lo) * so.u01(x, y)
        st.tval[rows, j] = t
        st.cand[rows, j], st.inside[rows, j] = candidates(u, dirn, t, wrap)
        neg = t < 0.0
        lo = np.where(neg, t, lo)
        hi = np.where(neg, hi, t)
    st.lo2[rows], st.hi2[rows] = lo, hi


def slice_mid(st, wrap):
    """Phase 1 (so.slice_mid)."""
    n = st.n_out
    ok = (st.inside_out != 0) & (st.ll_out > st.lmin)
    st.lo = st.lo - so._run(ok[:, :n]).astype(np.float64)
    st.hi = st.hi + so._run(ok[:, n:]).astype(np.float64)
    _propose_shrink(st, wrap, np.arange(st.k), st.lo, st.hi)


def slice_end(st, wrap, propose_more):
    """Phase 2 (propose_more) or 3 (so.slice_end); an accepted point is the stored candidate, so its
    circular coordinates are already in [0, 1)."""
    pend = st.pending != 0
    ok = (st.inside != 0) & (st.cand_ll > st.lmin)
    hit = pend & ok.any(axis=1)
    first = np.argmax(ok, axis=1)
    acc = np.nonzero(hit)[0]
    st.u[acc] = st.cand[acc, first[acc]]
    st.theta[acc] = st.cand_th[acc, first[acc]]
    st.lcur[acc] = st.cand_ll[acc, first[acc]]
    st.pending[acc] = 0
    st.stats[1] += np.uint64(len(acc))
    rej = pend & ~hit
    st.lo[rej], st.hi[rej] = st.lo2[rej], st.hi2[rej]
    if not propose_more:
        st.stats[0] += np.uint64(int(rej.sum()))
        return
    still = np.nonzero(rej)[0]
    if len(still):
        _propose_shrink(st, wrap, still, st.lo2[still], st.hi2[still])
    done = np.nonzero(~rej)[0]
    st.cand[done], _ = candidates(st.u[done], st.dirn[done], np.zeros((len(done), st.m)), wrap)
    st.inside[done] = 0


def phase(ph, st, wrap, dirn=None):
    """rvl_slice_phase_wrapped(ph) with the mask `wrap` on the state; phase 0 returns (z, the
    oracle's own direction)."""
    if ph == 0:
        return slice_begin(st, wrap, dirn)
    if ph == 1:
        return slice_mid(st, wrap)
    if ph in (2, 3):
        return slice_end(st, wrap, ph == 2)
    raise ValueError("phase must be 0, 1, 2 or 3")
