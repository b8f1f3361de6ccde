"""
CPU tests of MLFriends region sampling (sampler_dev.nested_sample_ensemble(method='mlfriends')):
the host restatement of its kernels (tests/_region_oracle.py) -- hand-worked radii, uniform draws on
a union of balls in the plane and on a torus, the pick order -- the batch-size rule, the C-ABI struct
and the argument checks.  The device side is tests/test_gpu_region.py.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy import stats

import _region_oracle as ro
from evidence_b200 import _abi
from evidence_b200.sampler_dev import _region_batch, nested_sample_ensemble
from oracle import slice_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- radius -------------------------------------------------------------------------------------
def test_bootstrap_indices_are_philox_words():
    """Index 4q + t of bootstrap b: floor(word_t n / 2^32), words of counter (round, TAG_BOOT + b, q, 0)."""
    n, seed = 7, 99
    chosen = ro.boot_chosen(seed, 3, 5, n)
    want = np.zeros(n, bool)
    for t in range(n):
        words = so.draw(seed, 3, ro.TAG_BOOT + 5, np.uint64(t // 4))
        want[(int(words[t % 4]) * n) >> 32] = True
    assert np.array_equal(chosen, want)


def test_radius_by_hand():
    """d = 1, L = 2 (D = ((a - b) / 2)^2): survivors 0.1, 0.2, 0.5, 0.9 after one retired point; each
    bootstrap's value worked out from its drawn set by hand; a run of two survivors whose bootstrap
    drew both has radius 0; a run with kk = 0 keeps its value."""
    pos = np.array([0.7, 0.1, 0.2, 0.5, 0.9])          # slot 0 is retired (order puts it first)
    u = np.stack([pos[:, None], pos[:, None]])
    order = np.array([[0, 1, 2, 3, 4]] * 2)
    chol = np.full((2, 1, 1), 2.0)
    seed, nboot = 5, 6
    want = 0.0
    surv = pos[1:]
    for b in range(nboot):
        ch = ro.boot_chosen(seed, 0, b, 4)
        for i in np.flatnonzero(~ch):
            want = max(want, min(((surv[i] - surv[j]) / 2.0) ** 2 for j in np.flatnonzero(ch)))
    got = ro.radius([seed, seed], u, order, np.array([1, 0]), chol, nboot, 0, rad2=[0.0, -3.0])
    assert got[0] == want and got[1] == -3.0
    assert want > 0
    # two survivors, one bootstrap: find a seed whose draw takes both, and one whose draw does not
    two = np.array([[[0.1], [0.3], [0.6]]])
    both = next(s for s in range(100) if ro.boot_chosen(s, 0, 0, 2).all())
    one = next(s for s in range(100) if not ro.boot_chosen(s, 0, 0, 2).all())
    assert ro.radius([both], two, np.array([[0, 1, 2]]), np.array([1]), np.ones((1, 1, 1)), 1, 0)[0] == 0.0
    assert ro.radius([one], two, np.array([[0, 1, 2]]), np.array([1]), np.ones((1, 1, 1)), 1, 0)[0] == \
        (0.6 - 0.3) ** 2


# ---- uniform draws on a union of balls ------------------------------------------------------------
def _cells_inside(member, ncell, sub=5):
    """The cells of an ncell x ncell grid of the unit square entirely inside the region (sub x sub
    points of every cell tested)."""
    g = (np.arange(sub) + 0.5) / sub
    inside = np.zeros((ncell, ncell), bool)
    for a in range(ncell):
        for b in range(ncell):
            p = np.stack(np.meshgrid((a + g) / ncell, (b + g) / ncell, indexing="ij"), -1).reshape(-1, 2)
            inside[a, b] = member(p).all()
    return inside


def _uniform_p(x, inside, ncell):
    """Chi-square p-value of equal counts over the cells inside; x [N, 2]."""
    cell = np.minimum((x * ncell).astype(int), ncell - 1)
    counts = np.zeros((ncell, ncell))
    np.add.at(counts, (cell[:, 0], cell[:, 1]), 1)
    obs = counts[inside]
    return stats.chisquare(obs).pvalue, obs


def _draw_many(seeds, u, order, kk, chol, rad2, n_slots, wrap=None, **kw):
    out = []
    for b in range(n_slots // 20000):
        x, flag, *_ = ro.draw(seeds, u, order, kk, chol, rad2, [0, 20000], b, 0, wrap, **kw)
        out.append(x[flag])
    return np.concatenate(out)


def test_draws_uniform_on_overlapping_discs():
    """Three overlapping discs of radius 0.18 (whitening 2 I, rho2 = 0.0081) in the unit square: the
    accepted points lie in the union and are uniform over the cells inside it; without rule 7 (each
    point through its first ball) the overlaps are over-filled and the same test fails."""
    centres = np.array([[0.9, 0.9], [0.3, 0.4], [0.45, 0.5], [0.35, 0.6]])   # slot 0 retired
    u, order, kk = centres[None], np.array([[0, 1, 2, 3]]), np.array([1])
    chol, rad2 = np.array([2.0 * np.eye(2)]), np.array([(0.18 / 2.0) ** 2])

    def member(p):
        return (((p[:, None, :] - centres[None, 1:, :]) ** 2).sum(-1) <= 0.18 ** 2).any(1)
    x = _draw_many([17], u, order, kk, chol, rad2, 200000)
    assert member(x).all() and len(x) > 100000
    inside = _cells_inside(member, 24)
    p, obs = _uniform_p(x, inside, 24)
    assert inside.sum() > 60 and p > 1e-3, (p, obs.min(), obs.max())
    y = _draw_many([17], u, order, kk, chol, rad2, 200000, first_ball=False)
    assert _uniform_p(y, inside, 24)[0] < 1e-6


def test_draws_uniform_on_a_torus():
    """Coordinate 0 circular, whitening diag(1, 0.2), rho = 0.7: each ball is wider than half the
    circle.  The accepted points are uniform over the cells inside the union of the nearest-image
    balls; without rule 4 (|delta_c| <= 1/2) the part of a ball beyond half the circle lands a second
    time on the other side and the same test fails."""
    centres = np.array([[0.0, 0.0], [0.5, 0.45], [0.1, 0.55]])
    u, order, kk = centres[None], np.array([[0, 1, 2]]), np.array([1])
    chol, rad2 = np.array([np.diag([1.0, 0.2])]), np.array([0.49])
    wrap = np.array([True, False])

    def member(p):
        dl = p[:, None, :] - centres[None, 1:, :]
        dl[..., 0] -= np.rint(dl[..., 0])
        return ((dl[..., 0] ** 2 + (dl[..., 1] / 0.2) ** 2) <= 0.49).any(1)
    x = _draw_many([23], u, order, kk, chol, rad2, 200000, wrap)
    assert member(x).all() and (x[:, 0] >= 0).all() and (x[:, 0] < 1).all()
    inside = _cells_inside(member, 20)
    p, obs = _uniform_p(x, inside, 20)
    assert inside.sum() > 60 and p > 1e-3, (p, obs.min(), obs.max())
    y = _draw_many([23], u, order, kk, chol, rad2, 200000, wrap, nearest_image=False)
    assert _uniform_p(y, inside, 20)[0] < 1e-6


# ---- pick ---------------------------------------------------------------------------------------
def test_pick_fills_walkers_in_row_order():
    """Walker j of run r takes the (j - filled[r])-th row of run r above lmin[r], in row order; rows
    beyond the walkers are counted in `above` but not taken; a run with kk = 0 is left alone."""
    d = 2
    kk = np.array([3, 0, 2])
    lmin = np.array([0.0, 0.0, 5.0])
    offs = np.array([0, 5, 5, 9])
    cand_ll = np.array([-1.0, 2.0, 3.0, -4.0, 7.0, 6.0, 4.0, 9.0, 8.0])
    cand = np.arange(9 * d, dtype=float).reshape(9, d)
    cand_th = -cand
    run_of = np.array([2, 0, 0, 2, 0], np.int32)
    walker_of = np.array([0, 0, 1, 1, 2], np.int32)
    z = np.zeros((5, d))
    u, th, lc, filled, above = ro.pick(kk, lmin, offs, cand, cand_th, cand_ll, run_of, walker_of, z, z,
                                       np.full(5, np.nan), [1, 0, 0])
    # run 0 had walker 0 filled: rows above 0 are 1, 2, 4 -> its walkers 1, 2 (w = 2, 4) take rows 1, 2
    assert np.isnan(lc[1]) and np.array_equal(u[1], z[1])
    assert lc[2] == 2.0 and np.array_equal(u[2], cand[1]) and np.array_equal(th[2], -cand[1])
    assert lc[4] == 3.0 and np.array_equal(u[4], cand[2]) and np.array_equal(th[4], -cand[2])
    # run 2: rows above 5 are 5, 7, 8 -> its walkers 0, 1 (w = 0, 3) take rows 5, 7
    assert lc[0] == 6.0 and lc[3] == 9.0 and np.array_equal(u[3], cand[7])
    assert list(filled) == [3, 0, 2] and list(above) == [3, 0, 3]


# ---- batch sizes --------------------------------------------------------------------------------
def test_batch_size_rule():
    """c = clamp(ceil(1.5 need / eff), need, ndraw_max); 0 for a run that needs nothing."""
    need = np.array([10, 10, 10, 0, 3, 40])
    eff = np.array([1.0, 0.1, 1e-6, 0.5, 2.0, 0.3])
    assert list(_region_batch(need, eff, 65536)) == [15, 150, 65536, 0, 3, 200]
    assert list(_region_batch([100], [1.0], 120)) == [120]
    assert list(_region_batch([100], [1.0], 50)) == [50]  # ndraw_max wins over need


def test_method_argument_checks():
    f = lambda u: (u, -(u ** 2).sum(1))  # noqa: E731
    with pytest.raises(ValueError, match="'slice' or 'mlfriends'"):
        nested_sample_ensemble(f, 2, [1], method="ellipsoid")
    with pytest.raises(ValueError, match="adaptive_nsteps"):
        nested_sample_ensemble(f, 2, [1], method="mlfriends", adaptive_nsteps="move-distance")


# ---- ABI ----------------------------------------------------------------------------------------
def test_struct_size_matches_the_header(built_lib):
    src = '#include <stdio.h>\n#include "rvlnl.h"\nint main(){printf("%zu\\n",sizeof(rvl_region_args));return 0;}'
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        got = int(subprocess.check_output([exe]))
    assert got == ctypes.sizeof(_abi.rvl_region_args) == 112


def test_abi_argument_checks(built_lib):
    """NULL pointers, B < 1, d above RVL_MAX_DIM and a mask bit at or above d: RVL_EINVAL and a message,
    before anything reaches the device."""
    lib = _abi.load()
    g = _abi.rvl_region_args(num_bootstraps=4)
    runs = _abi.rvl_slice_runs(n_runs=2)
    live = _abi.rvl_slice_live(nlive=10, d=3)
    args = _abi.rvl_slice_args(k=4, d=3)
    G, RN, LV, A = (ctypes.byref(x) for x in (g, runs, live, args))
    rad = lambda *a, bits=None: lib.rvl_region_runs_radius(*a, bits, None)  # noqa: E731
    drw = lambda *a, bits=None: lib.rvl_region_runs_draw(*a, bits, None)  # noqa: E731
    pck = lambda *a: lib.rvl_region_runs_pick(*a, None)  # noqa: E731

    def err():
        return lib.rvl_slice_last_error().decode()
    for fn in (rad, drw):
        assert fn(None, RN, LV) == -1 and "region is NULL" in err()
        assert fn(G, None, LV) == -1 and "runs is NULL" in err()
        assert fn(G, RN, None) == -1 and "live is NULL" in err()
        assert fn(G, RN, LV) == -1 and "must be set" in err()
    runs.seeds, runs.chol, live.u_live, live.order, live.kk = 8, 8, 8, 8, 8
    assert rad(G, RN, LV) == -1 and "rad2 must be set" in err()
    assert drw(G, RN, LV) == -1 and "draw:" in err()
    g.rad2 = 8
    for field, value in (("d", 0), ("d", 129), ("nlive", 2)):
        old = getattr(live, field)
        setattr(live, field, value)
        assert rad(G, RN, LV) == -1 and "bad sizes" in err()
        assert drw(G, RN, LV) == -1 and "bad sizes" in err()
        setattr(live, field, old)
    for b in (0, -1):
        g.num_bootstraps = b
        assert rad(G, RN, LV) == -1 and "num_bootstraps" in err()
    g.num_bootstraps = 4
    bits = (ctypes.c_uint32 * 4)(0b1000, 0, 0, 0)
    assert rad(G, RN, LV, bits=bits) == -1 and "bit 3 set, but d = 3" in err()
    assert drw(G, RN, LV, bits=bits) == -1 and "bit 3 set, but d = 3" in err()
    live.nlive = 300000
    assert rad(G, RN, LV) == -1 and "nlive too large" in err()
    live.nlive = 10
    g.batch = 65536
    assert drw(G, RN, LV) == -1 and "batch" in err()
    g.batch = 0
    assert pck(None, A, RN, LV) == -1 and "region is NULL" in err()
    assert pck(G, None, RN, LV) == -1 and "args is NULL" in err()
    assert pck(G, A, None, LV) == -1 and "runs is NULL" in err()
    assert pck(G, A, RN, None) == -1 and "live is NULL" in err()
    args.d = 4
    assert pck(G, A, RN, LV) == -1 and "bad sizes" in err()
    args.d = 3
    assert pck(G, A, RN, LV) == -1 and "pick: a device address is missing" in err()
