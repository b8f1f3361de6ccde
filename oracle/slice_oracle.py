"""
Host restatement of the slice-sampler bookkeeping kernels (evidence_b200/csrc/rvslice.cu).

TEST INFRASTRUCTURE ONLY (checker of `rvl_slice_phase`).

Each kernel is restated statement by statement, vectorised over the walkers in numpy, with the same
float64 operations in the same order (the library is built with -fmad=false and IEEE div/sqrt: one
rounding per operation).  The only thing that cannot be reproduced bit for bit is the direction:
the device's log/sin/cos are not correctly rounded (1-2 ulp), so `slice_begin` takes the device's
`dirn` when it is given and continues from it; everything downstream of the direction -- brackets,
shrinkage offsets, candidates, inside flags, acceptance, copies, counts -- is then bit-identical.

The state is a `SliceState` whose arrays mirror the buffers of `rvl_slice_args`, shaped per walker:
cand_out [k][2 n_out][d], inside_out / ll_out [k][2 n_out], cand / cand_th [k][m][d],
inside / cand_ll / tval [k][m].
"""
from dataclasses import dataclass

import numpy as np

M32 = np.uint64(0xFFFFFFFF)
HI_CLAMP = 1.0 - 2.0 ** -53
TAG_DIR, TAG_BRACKET, TAG_SHRINK = 0x44495200, 0x42524B00, 0x53480000
KEY_HI_CONST = 0x51CE
TWO_PI = 6.283185307179586


def philox4x32(ctr, k0, k1):
    """Philox4x32-10: counter words (x, y, z, w) and key (k0, k1), each a uint32 value or array
    (broadcast); returns the four output words as uint64 arrays holding uint32 values."""
    x, y, z, w = (np.asarray(c, dtype=np.uint64) & M32 for c in ctr)
    k0 = np.asarray(k0, dtype=np.uint64) & M32
    k1 = np.asarray(k1, dtype=np.uint64) & M32
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * x  # < 2^64: the full 32 x 32 product
        p1 = np.uint64(0xCD9E8D57) * z
        x, y, z, w = (p1 >> np.uint64(32)) ^ y ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ w ^ k1, p0 & M32
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return x, y, z, w


def u01(a, b):
    """The kernel's uniform from two words: 52 random bits, ((v >> 1) + 0.5) 2^-52, in
    [2^-53, 1 - 2^-53] -- strictly inside (0, 1), every operation exact."""
    a = np.asarray(a, dtype=np.uint64)
    b = np.asarray(b, dtype=np.uint64)
    v = (a << np.uint64(21)) ^ (b >> np.uint64(11))  # 53 bits
    return ((v >> np.uint64(1)).astype(np.float64) + 0.5) * 2.0 ** -52


def key(seed):
    """The generator's key: the seed alone (the walker is a counter word)."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return seed & 0xFFFFFFFF, ((seed >> 32) + KEY_HI_CONST) & 0xFFFFFFFF


def draw(seed, move, tag, walkers):
    """The four words of counter (move, tag, walker, 0) for every walker."""
    k0, k1 = key(seed)
    return philox4x32((move & 0xFFFFFFFF, tag & 0xFFFFFFFF, walkers, 0), k0, k1)


@dataclass
class SliceState:
    k: int
    d: int
    n_out: int
    m: int
    seed: int
    move: int
    shrink_round: int
    lmin: float
    chol: np.ndarray        # [d][d]
    u: np.ndarray           # [k][d]
    theta: np.ndarray       # [k][d]
    lcur: np.ndarray        # [k]
    dirn: np.ndarray        # [k][d]
    lo: np.ndarray          # [k]
    hi: np.ndarray
    lo2: np.ndarray
    hi2: np.ndarray
    tval: np.ndarray        # [k][m]
    pending: np.ndarray     # [k] int32
    cand_out: np.ndarray    # [k][2 n_out][d]
    inside_out: np.ndarray  # [k][2 n_out] uint8
    ll_out: np.ndarray      # [k][2 n_out]
    cand: np.ndarray        # [k][m][d]
    inside: np.ndarray      # [k][m] uint8
    cand_ll: np.ndarray     # [k][m]
    cand_th: np.ndarray     # [k][m][d]
    stats: np.ndarray       # [2] uint64: unresolved walkers, accepted moves

    def copy(self):
        return SliceState(**{f: (v.copy() if isinstance(v, np.ndarray) else v)
                             for f, v in self.__dict__.items()})


def _candidates(u, dirn, t):
    """write_candidate for every walker: p = u + t d (t [k] or [k, n]); returns (clamped points,
    inside flags) with inside = 0 <= p < 1 in every coordinate (False for NaN)."""
    t = np.asarray(t, dtype=np.float64)
    if t.ndim == 1:
        p = u + t[:, None] * dirn
        inside = ((p >= 0.0) & (p < 1.0)).all(axis=-1)
    else:
        p = u[:, None, :] + t[:, :, None] * dirn[:, None, :]
        inside = ((p >= 0.0) & (p < 1.0)).all(axis=-1)
    return np.fmin(np.fmax(p, 0.0), HI_CLAMP), inside.astype(np.uint8)


def normals(st):
    """z ~ N(0, I) of slice_begin: Box-Muller, coordinates 2i and 2i+1 share counter word i
    (cos for even j, sin for odd j).  numpy's log/sin/cos: within an ulp or two of the device."""
    walkers = np.arange(st.k, dtype=np.uint64)[:, None]
    j = np.arange(st.d, dtype=np.uint64)[None, :]
    x, y, z, w = draw(st.seed, st.move, np.uint64(TAG_DIR) + (j >> np.uint64(1)), walkers)
    rad = np.sqrt(-2.0 * np.log(u01(x, y)))
    ang = TWO_PI * u01(z, w)
    return np.where((j & np.uint64(1)) == 1, rad * np.sin(ang), rad * np.cos(ang))


def norm2(z):
    """Squared norm in the kernel's order: per-lane sums over j = lane, lane + 32, .. from 0.0, then
    the xor butterfly 16, 8, 4, 2, 1."""
    k, d = z.shape
    part = np.zeros((k, 32))
    for j in range(d):
        part[:, j % 32] = part[:, j % 32] + z[:, j] * z[:, j]
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        part = part + part[:, lanes ^ o]
    return part[:, 0]


def direction(st, z):
    """dirn = chol z * (1 / sqrt(|z|^2)); acc += chol[j][l] z[l] for l = 0..j, one rounding each."""
    inv = 1.0 / np.sqrt(norm2(z))
    acc = np.zeros((st.k, st.d))
    for l in range(st.d):
        acc[:, l:] = acc[:, l:] + st.chol[l:, l][None, :] * z[:, l:l + 1]
    return acc * inv[:, None]


def slice_begin(st, dirn=None):
    """Phase 0.  Returns (z, the oracle's own direction); st.dirn is `dirn` when given, else that
    direction."""
    z = normals(st)
    own = direction(st, z)
    st.dirn = own.copy() if dirn is None else np.array(dirn, dtype=np.float64).reshape(st.k, st.d)
    x, y, _, _ = draw(st.seed, st.move, TAG_BRACKET, np.arange(st.k, dtype=np.uint64))
    r0 = u01(x, y)
    lo, hi = -r0, 1.0 - r0
    st.lo, st.hi = lo, hi
    st.pending = np.ones(st.k, dtype=np.int32)
    steps = np.arange(st.n_out, dtype=np.float64)
    t = np.concatenate([lo[:, None] - steps[None, :], hi[:, None] + steps[None, :]], axis=1)
    st.cand_out, st.inside_out = _candidates(st.u, st.dirn, t)
    return z, own


def _propose_shrink(st, rows, lo, hi):
    """m shrinkage candidates of the walkers `rows` from their brackets (lo, hi), each drawn as if
    the ones before it had been rejected; writes tval, cand, inside, lo2, hi2 of those rows."""
    lo, hi = lo.copy(), hi.copy()
    walkers = rows.astype(np.uint64)
    u, dirn = st.u[rows], st.dirn[rows]
    for j in range(st.m):
        tag = (TAG_SHRINK + st.shrink_round * 64 + j) & 0xFFFFFFFF
        x, y, _, _ = draw(st.seed, st.move, tag, walkers)
        t = lo + (hi - lo) * u01(x, y)
        st.tval[rows, j] = t
        st.cand[rows, j], st.inside[rows, j] = _candidates(u, dirn, t)
        neg = t < 0.0
        lo = np.where(neg, t, lo)
        hi = np.where(neg, hi, t)
    st.lo2[rows], st.hi2[rows] = lo, hi


def _run(success):
    """Length of the run of successes from the first slot."""
    return np.cumprod(success, axis=1).sum(axis=1)


def slice_mid(st):
    """Phase 1: final bracket from the runs of successes (inside and lnL > lmin, strictly) on both
    sides, then the first m shrinkage candidates."""
    n = st.n_out
    ok = (st.inside_out != 0) & (st.ll_out > st.lmin)
    run_lo, run_hi = _run(ok[:, :n]), _run(ok[:, n:])
    st.lo = st.lo - run_lo.astype(np.float64)
    st.hi = st.hi + run_hi.astype(np.float64)
    _propose_shrink(st, np.arange(st.k), st.lo, st.hi)


def slice_end(st, propose_more):
    """Phase 2 (propose_more) or 3: accept the first candidate that is inside and above lmin; a
    pending walker without one takes the bracket (lo2, hi2).  Phase 2 then proposes m more
    candidates for the walkers still pending and writes t = 0 candidates with inside = 0 for the
    others; phase 3 counts the walkers left pending."""
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
        _propose_shrink(st, still, st.lo2[still], st.hi2[still])
    done = np.nonzero(~rej)[0]
    st.cand[done], _ = _candidates(st.u[done], st.dirn[done], np.zeros((len(done), st.m)))
    st.inside[done] = 0


def phase(ph, st, dirn=None):
    """rvl_slice_phase(ph) on the state; phase 0 returns (z, the oracle's own direction)."""
    if ph == 0:
        return slice_begin(st, dirn)
    if ph == 1:
        return slice_mid(st)
    if ph in (2, 3):
        return slice_end(st, ph == 2)
    raise ValueError("phase must be 0, 1, 2 or 3")
