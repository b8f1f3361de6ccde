"""CPU tests of oracle/slice_oracle.py, the host restatement of the slice-sampler kernels: its
Philox4x32-10 against Random123's known answers, its uniform at the extreme words, the unit-cube
test of its candidates, and the bookkeeping of one whole move on a hand-checked case."""
import numpy as np

from oracle import slice_oracle as so

FF = 0xFFFFFFFF


def _hex(words):
    return tuple("%08x" % int(w) for w in words)


def test_philox_known_answers():
    # Random123's kat_vectors for philox4x32_10: counter (x, y, z, w), key (k0, k1)
    assert _hex(so.philox4x32((0, 0, 0, 0), 0, 0)) == ("6627e8d5", "e169c58d", "bc57ac4c", "9b00dbd8")
    assert _hex(so.philox4x32((FF, FF, FF, FF), FF, FF)) == (
        "408f276d", "41c83b0e", "a20bc7c6", "6d5451fd")
    assert _hex(so.philox4x32((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344),
                              0xa4093822, 0x299f31d0)) == ("d16cfe09", "94fdcceb", "5001e420", "24126ea1")


def test_philox_is_vectorised_elementwise():
    ctr = np.arange(5, dtype=np.uint64)
    got = np.stack(so.philox4x32((7, ctr, 3, 0), 11, 13))
    for i in range(5):
        assert np.array_equal(got[:, i], np.stack(so.philox4x32((7, i, 3, 0), 11, 13)))


def test_u01_is_strictly_inside_the_unit_interval_at_the_extreme_words():
    lo, hi = so.u01(0, 0), so.u01(FF, FF)
    assert lo == 2.0 ** -53 and 0.0 < lo
    assert hi == 1.0 - 2.0 ** -53 and hi < 1.0
    # (2^53 - 1) + 0.5 rounds to 2^53 in float64: the 53-bit form would return exactly 1.0 here
    assert (float(2 ** 53 - 1) + 0.5) * 2.0 ** -53 == 1.0
    # the low 11 bits of b are not used
    assert so.u01(FF, 0xFFFFF800) == hi and so.u01(0, 0x7FF) == lo
    v = so.u01(np.arange(1000, dtype=np.uint64) * 0x9E3779B9 & FF, np.arange(1000, dtype=np.uint64))
    assert np.all((v > 0.0) & (v < 1.0))


def test_key_is_the_seed_alone():
    assert so.key(0) == (0, 0x51CE)
    assert so.key(2 ** 32 + 7) == (7, 1 + 0x51CE)
    assert so.key(2 ** 64 - 1) == (FF, (FF + 0x51CE) & FF)


def test_candidate_inside_semantics_at_the_cube_faces():
    u = np.array([[0.0, 0.5], [1.0, 0.5], [0.5, 0.5], [0.25, 0.5]])
    dirn = np.array([[0.0, 0.1], [0.0, 0.1], [0.6, 0.0], [-0.5, 0.0]])
    pts, inside = so._candidates(u, dirn, np.array([1.0, 1.0, 1.0, 1.0]))
    # p = 0 is inside; p = 1 is outside and clamped to the largest double below 1; p < 0 clamps to 0
    assert inside.tolist() == [1, 0, 0, 0]
    assert pts[0].tolist() == [0.0, 0.6]
    assert pts[1, 0] == 1.0 - 2.0 ** -53 and pts[2, 0] == 1.0 - 2.0 ** -53 and pts[3, 0] == 0.0
    _, inside = so._candidates(np.array([[0.5, np.nan]]), np.zeros((1, 2)), np.zeros(1))
    assert inside.tolist() == [0]


def test_norm_order_is_the_warp_butterfly():
    z = np.random.default_rng(3).standard_normal((4, 77))
    n2 = so.norm2(z)
    assert np.allclose(n2, (z * z).sum(1), rtol=1e-14, atol=0)
    part = np.zeros((4, 32))
    for j in range(77):
        part[:, j % 32] += z[:, j] ** 2
    for o in (16, 8, 4, 2, 1):
        part = part + part[:, np.arange(32) ^ o]
    assert np.array_equal(part[:, 0], n2) and np.all(part == part[:, :1])


def _state(k=3, d=2, n_out=2, m=2, lmin=0.0):
    z = lambda *s, dt=np.float64: np.zeros(s, dtype=dt)  # noqa: E731
    return so.SliceState(k=k, d=d, n_out=n_out, m=m, seed=5, move=2, shrink_round=0, lmin=lmin,
                         chol=np.eye(d) * 0.1, u=np.full((k, d), 0.5), theta=z(k, d),
                         lcur=np.full(k, np.nan), dirn=z(k, d), lo=z(k), hi=z(k), lo2=z(k), hi2=z(k),
                         tval=z(k, m), pending=z(k, dt=np.int32), cand_out=z(k, 2 * n_out, d),
                         inside_out=z(k, 2 * n_out, dt=np.uint8), ll_out=z(k, 2 * n_out),
                         cand=z(k, m, d), inside=z(k, m, dt=np.uint8), cand_ll=z(k, m),
                         cand_th=z(k, m, d), stats=z(2, dt=np.uint64))


def test_one_move_by_hand():
    st = _state()
    dirn = np.array([[0.1, 0.0], [0.0, -0.1], [0.05, 0.05]])
    so.phase(0, st, dirn=dirn)
    assert np.array_equal(st.dirn, dirn) and st.pending.tolist() == [1, 1, 1]
    assert np.all((st.lo < 0) & (st.hi > 0)) and np.array_equal(st.hi - st.lo, np.ones(3))
    assert np.array_equal(st.cand_out[:, 1], st.u + (st.lo - 1.0)[:, None] * dirn)
    lo0, hi0 = st.lo.copy(), st.hi.copy()
    # runs: walker 0 lo T F -> 1, hi F T -> 0; walker 1 ll == lmin and NaN -> 0, 0; walker 2 all T
    st.ll_out[:] = [[1.0, -1.0, -1.0, 1.0], [0.0, 1.0, np.nan, 1.0], [1.0, 1.0, 1.0, 1.0]]
    so.phase(1, st)
    assert np.array_equal(st.lo, lo0 - [1.0, 0.0, 2.0]) and np.array_equal(st.hi, hi0 + [0.0, 0.0, 2.0])
    t0 = st.tval[:, 0]
    assert np.all((t0 > st.lo) & (t0 < st.hi))
    lo1 = np.where(t0 < 0, t0, st.lo)
    hi1 = np.where(t0 < 0, st.hi, t0)
    assert np.all((st.tval[:, 1] > lo1) & (st.tval[:, 1] < hi1))
    assert np.array_equal(st.cand[:, 1], st.u + st.tval[:, 1:2] * dirn)
    # walker 0 accepts its second candidate, walker 1 none (-inf, == lmin), walker 2 its first
    st.cand_ll[:] = [[np.nan, 2.0], [-np.inf, 0.0], [3.0, 4.0]]
    st.cand_th[:] = np.arange(12, dtype=np.float64).reshape(3, 2, 2)
    cand = st.cand.copy()
    so.phase(3, st)  # a move of one shrinkage round
    assert st.pending.tolist() == [0, 1, 0] and st.stats.tolist() == [1, 2]
    assert np.array_equal(st.u[0], cand[0, 1]) and np.array_equal(st.u[2], cand[2, 0])
    assert np.array_equal(st.u[1], [0.5, 0.5]) and np.isnan(st.lcur[1])
    assert st.theta.tolist() == [[2.0, 3.0], [0.0, 0.0], [8.0, 9.0]]
    assert st.lcur[0] == 2.0 and st.lcur[2] == 3.0
    assert st.lo[1] == st.lo2[1] and st.hi[1] == st.hi2[1]


def test_phase_2_proposes_for_pending_walkers_only():
    st = _state()
    so.phase(0, st, dirn=np.array([[0.1, 0.0], [0.0, -0.1], [0.05, 0.05]]))
    st.ll_out[:] = -1.0
    so.phase(1, st)
    st.cand_ll[:] = [[1.0, 1.0], [-1.0, -1.0], [-1.0, -1.0]]
    tval, lo2 = st.tval.copy(), st.lo2.copy()
    st.shrink_round = 1
    so.phase(2, st)
    assert st.pending.tolist() == [0, 1, 1] and st.stats.tolist() == [0, 1]
    assert st.inside[0].tolist() == [0, 0] and np.array_equal(st.cand[0], np.repeat(st.u[:1], 2, 0))
    assert np.array_equal(st.tval[0], tval[0]) and st.lo2[0] == lo2[0]
    # the pending walkers drew new offsets inside their shrunken brackets
    assert np.all((st.tval[1:, 0] > st.lo[1:]) & (st.tval[1:, 0] < st.hi[1:]))
    assert not np.any(st.tval[1:] == tval[1:])
