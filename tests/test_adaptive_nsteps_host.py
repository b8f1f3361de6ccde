"""
CPU tests of the adaptive number of moves (adaptive_nsteps='move-distance' of the device samplers):
the host restatement of the spacing and travel kernels (tests/_slice_travel_oracle.py) on hand-worked
points, the adaptation rule, the walker layout of an adaptive round, the move numbers, the settings
that reject it, and the argument checks of the C-ABI.  The device side is
tests/test_gpu_adaptive_nsteps.py.
"""
import ctypes

import numpy as np
import pytest

import _slice_travel_oracle as to
from evidence_b200 import _abi
from evidence_b200 import priors
from evidence_b200 import sampler as hs
from evidence_b200 import ultranest as runner
from evidence_b200.sampler_dev import (_adapt_nsteps, _adaptive_layout, _adaptive_settings, _move_base,
                                       _walker_layout, nested_sample_device)

DIAG = np.diag([0.5, 0.25])  # L^-1 = diag(2, 4): D = 4 dx^2 + 16 dy^2, exact in binary


def test_linv_and_distance_by_hand():
    """L = [[1, 0], [1/2, 1/2]]: L^-1 = [[1, 0], [-1, 2]], D = dx^2 + (2 dy - dx)^2; and against a
    solve on random factors (to rounding)."""
    X = to.linv(np.array([[1.0, 0.0], [0.5, 0.5]]))
    assert X.tolist() == [[1.0, 0.0], [-1.0, 2.0]]
    a, b = np.array([[0.75, 0.5]]), np.array([[0.25, 0.25]])
    assert to.dist2(a, b, X).tolist() == [0.25 + 0.0]  # dx = 1/2, 2 dy - dx = 0
    rng = np.random.default_rng(1)
    for d in (2, 7, 26):
        A = rng.normal(size=(d, d))
        L = np.linalg.cholesky(A @ A.T + d * np.eye(d))
        X = to.linv(L)
        assert np.allclose(X @ L, np.eye(d), atol=1e-12)
        p, q = rng.uniform(size=(5, d)), rng.uniform(size=(5, d))
        want = (np.linalg.solve(L, (p - q).T) ** 2).sum(0)
        assert np.allclose(to.dist2(p, q, X), want, rtol=1e-12)


def test_radius_by_hand():
    """Three points (1/8, 1/4), (3/8, 1/4), (1/8, 3/4) under L = diag(1/2, 1/4): pair distances 1/4, 4
    and 17/4, nearest neighbours 1/4, 1/4, 4: rho^2 = 4.  The circular dy = -1/2 stays -1/2 (rint
    rounds half to even), so wrapping coordinate 1 changes nothing here; (1/8, 1/8) - (1/8, 7/8) is
    dy = -3/4, D = 9, and 1/4 wrapped, D = 1."""
    u = np.array([[[0.125, 0.25], [0.375, 0.25], [0.125, 0.75]]])
    assert to.radius(u, np.array([[0, 1, 2]]), [0], DIAG[None], rad2=[7.0]).tolist() == [7.0]  # kk = 0: kept
    u4 = np.concatenate([np.array([[[0.5, 0.5]]]), u], axis=1)  # point 0 retired (kk = 1)
    order4 = np.array([[0, 1, 2, 3]])
    for wrap in (None, [False, True]):
        assert to.radius(u4, order4, [1], DIAG[None], wrap).tolist() == [4.0]
    assert to.delta(np.array([0.25]), np.array([0.75]), [True]).tolist() == [-0.5]
    assert to.delta(np.array([0.75]), np.array([0.25]), [True]).tolist() == [0.5]
    a, b = np.array([[0.125, 0.125]]), np.array([[0.125, 0.875]])
    assert to.dist2(a, b, to.linv(DIAG)).tolist() == [9.0]
    assert to.dist2(a, b, to.linv(DIAG), [False, True]).tolist() == [1.0]


def test_duplicate_points_have_no_spacing():
    """Survivors in identical pairs: every nearest neighbour is at 0, rho^2 = 0; then a walker that
    did not move is not far (0 > 0 is false) and one that moved is."""
    p = np.array([[0.25, 0.5], [0.25, 0.5], [0.75, 0.125], [0.75, 0.125]])
    u = np.concatenate([np.array([[0.5, 0.5]]), p])[None]
    order, kk = np.array([[0, 1, 2, 3, 4]]), np.array([1])
    rad2 = to.radius(u, order, kk, DIAG[None])
    assert rad2.tolist() == [0.0]
    u_end = np.array([[0.25, 0.5], [0.75, 0.25]])  # walker 0 stuck on survivor 1, walker 1 moved
    far = to.travel(u_end, [0, 0], [1, 3], u, kk, DIAG[None], rad2)
    assert far.tolist() == [1]


def test_travel_by_hand():
    """Two runs, rho^2 = 4 and 1/4: a walker is far only when D > rho^2 strictly; a run with kk = 0
    keeps its count."""
    u = np.array([[[0.5, 0.5], [0.125, 0.25], [0.375, 0.25]],
                  [[0.5, 0.5], [0.125, 0.25], [0.375, 0.25]],
                  [[0.5, 0.5], [0.5, 0.5], [0.5, 0.5]]])
    chol = np.stack([DIAG, DIAG, DIAG])
    rad2 = np.array([4.0, 0.25, 1.0])
    # D from (1/8, 1/4): to (1/8, 3/4) 4 (not > 4), to (5/8, 1/4) 1, to (3/8, 1/4) 1/4 (not > 1/4)
    u_end = np.array([[0.125, 0.75], [0.625, 0.25], [0.375, 0.25], [0.625, 0.25]])
    run_of, start = [0, 1, 1, 0], [1, 1, 1, 1]
    far = to.travel(u_end, run_of, start, u, [1, 1, 0], chol, rad2, far=[9, 9, 9])
    assert far.tolist() == [0, 1, 9]
    rad2[0] = 3.75
    assert to.travel(u_end, run_of, start, u, [1, 1, 0], chol, rad2).tolist() == [1, 1, 0]


@pytest.mark.parametrize("n, far, kk, floor, want", [
    (10, 19, 40, 1, 15),   # 2 far < kk: n + n // 2
    (10, 20, 40, 1, 10),   # 2 far == kk: unchanged
    (10, 30, 40, 1, 10),   # 4 far == 3 kk: unchanged
    (10, 31, 40, 1, 7),    # 4 far > 3 kk: n - n // 3
    (21, 40, 40, 21, 21),  # the floor
    (22, 40, 40, 21, 21),  # 22 - 7 = 15: the floor
    (80, 0, 40, 21, 84),   # the cap
    (84, 0, 40, 21, 84),
    (1, 0, 40, 1, 2),      # at least one more
])
def test_adaptation_rule(n, far, kk, floor, want):
    assert _adapt_nsteps([n], [far], [kk], floor, 84).tolist() == [want]


def test_adaptation_is_per_run_and_integer():
    n = np.array([21, 21, 40, 84, 30])
    far = np.array([0, 40, 39, 0, 30])
    kk = np.array([40, 40, 40, 40, 40])
    got = _adapt_nsteps(n, far, kk, 21, 84)
    assert got.tolist() == [31, 21, 27, 84, 30] and got.dtype == np.int64


def test_adaptive_layout_orders_runs_and_keeps_a_prefix():
    run_of, walker_of, ks = _adaptive_layout([3, 0, 2, 1], [5, 9, 5, 7])
    assert run_of.tolist() == [3, 0, 0, 0, 2, 2] and walker_of.tolist() == [0, 0, 1, 2, 0, 1]
    assert run_of.dtype == walker_of.dtype == np.int32
    assert ks == [6, 6, 6, 6, 6, 1, 1]  # run 1 has no walkers: its 9 moves launch nothing
    rng = np.random.default_rng(2)
    for _ in range(50):
        counts = rng.integers(0, 6, size=8)
        n_r = rng.integers(3, 12, size=8)
        run_of, walker_of, ks = _adaptive_layout(counts, n_r)
        assert sorted(zip(run_of.tolist(), walker_of.tolist())) == sorted(zip(*_walker_layout(counts)))
        for j, kj in enumerate(ks):
            moving = n_r[run_of] > j
            assert moving[:kj].all() and not moving[kj:].any()
        assert len(ks) == (n_r[counts > 0].max() if counts.any() else 0)
    # equal counts: the layout of _walker_layout, every move over all walkers
    run_of, walker_of, ks = _adaptive_layout([3, 1, 2], [21, 21, 21])
    assert [run_of.tolist(), walker_of.tolist()] == [a.tolist() for a in _walker_layout([3, 1, 2])]
    assert ks == [6] * 21


def test_move_numbers():
    assert _move_base(0, 84) == 0 and _move_base(3, 84) == 252
    assert [_move_base(i, 21) for i in range(4)] == [0, 21, 42, 63]  # max_nsteps == nsteps: the fixed run's
    last_ok = 2 ** 32 // 16 - 1  # its last move, last_ok * 16 + 15, is 2^32 - 1
    assert _move_base(last_ok, 16) + 15 == 2 ** 32 - 1
    with pytest.raises(OverflowError, match="32 bits"):
        _move_base(last_ok + 1, 16)


def test_settings():
    assert _adaptive_settings(None, None, 21) == (False, 21)
    assert _adaptive_settings("move-distance", None, 21) == (True, 84)
    assert _adaptive_settings("move-distance", 21, 21) == (True, 21)
    with pytest.raises(ValueError, match="below nsteps"):
        _adaptive_settings("move-distance", 20, 21)
    with pytest.raises(ValueError, match="move-distance"):
        _adaptive_settings("volume", None, 21)
    with pytest.raises(ValueError, match="max_nsteps applies"):
        _adaptive_settings(None, 40, 21)


def test_torch_formulation_and_host_sampler_reject_it():
    import torch

    def fused(U):
        return U, -0.5 * ((U - 0.5) ** 2).sum(1) / 0.01
    for kw in (dict(device="cpu"), dict(device="cpu", native=False)):
        with pytest.raises(ValueError, match="native kernels"):
            nested_sample_device(fused, 2, nlive=20, adaptive_nsteps="move-distance", **kw)
    f = lambda th: -0.5 * np.sum(th ** 2, axis=1)  # noqa: E731
    for method in ("slice", "ellipsoid"):
        with pytest.raises(ValueError, match="device samplers"):
            hs.nested_sample(f, lambda u: u, 2, nlive=50, method=method, adaptive_nsteps="move-distance")
    with pytest.raises(ValueError, match="device samplers"):
        hs.nested_sample(f, lambda u: u, 2, nlive=50, max_nsteps=10)
    del torch


class Toy:
    """The reference's scalar model protocol."""

    def __init__(self):
        self.parnames = ["a", "b"]
        self.datadict, self.fixedpardict = {}, {}

    def log_likelihood(self, x):
        return -0.5 * np.sum(((np.asarray(x) - 3.0) / 0.5) ** 2)


@pytest.mark.parametrize("method", ["slice", "ellipsoid"])
def test_runner_rejects_it_without_the_device_sampler(tmp_path, method):
    model = Toy()
    priordict = {p: priors.Uniform(0.0, 6.0) for p in model.parnames}
    rundict = {"target": "toy", "runid": "a", "save_dir": str(tmp_path)}
    settings = {"nlive": 40, "sampler": "builtin", "seed": 1, "builtin_method": method,
                "builtin_adaptive_nsteps": "move-distance"}
    with pytest.raises(ValueError, match="slice-device"):
        runner.run(model, rundict, priordict, settings)
    settings["builtin_adaptive_nsteps"] = "sometimes"
    with pytest.raises(ValueError, match="False or 'move-distance'"):
        runner.run(model, rundict, priordict, settings)
    settings["builtin_adaptive_nsteps"] = False  # the default: the run as before
    out = runner.run(model, rundict, priordict, settings)
    assert np.isfinite(out.logZ) and "adaptive" not in out.sampler_impl


def test_runner_note_and_default():
    s = runner.set_ultrasettings({"target": "t", "runid": "r"}, None, 3, 0, "now", ["a", "b", "c"])
    assert s["builtin_adaptive_nsteps"] is False
    note = runner._nsteps_note("move-distance", [21, 31, 46, 46, 30])
    assert note == "; adaptive nsteps (move-distance): moves per round min 21, median 31, max 46 over 5 rounds"


def test_abi_argument_checks(built_lib):
    """Bad sizes, missing addresses and mask bits at or above d: RVL_EINVAL and a message."""
    lib = _abi.load()
    runs = _abi.rvl_slice_runs(n_runs=2)
    live = _abi.rvl_slice_live(nlive=10, d=3)
    a = _abi.rvl_slice_args(k=4, d=3, n_out=2, m=2)
    rad = lambda rn, lv, bits=None, r2=8: lib.rvl_slice_runs_radius(rn, lv, bits, r2, None)  # noqa: E731
    trav = lambda args, bits=None, far=8: lib.rvl_slice_runs_travel(  # noqa: E731
        args, ctypes.byref(runs), ctypes.byref(live), bits, 8, far, None)

    def err():
        return lib.rvl_slice_last_error().decode()
    assert rad(None, ctypes.byref(live)) == -1 and "runs is NULL" in err()
    assert rad(ctypes.byref(runs), None) == -1 and "live is NULL" in err()
    assert rad(ctypes.byref(runs), ctypes.byref(live)) == -1 and "must be set" in err()
    live.u_live, live.kk, runs.chol = 8, 8, 8
    assert rad(ctypes.byref(runs), ctypes.byref(live), r2=None) == -1 and "rad2 must be set" in err()
    assert rad(ctypes.byref(runs), ctypes.byref(live)) == -1 and "live->order" in err()
    for field, value in (("nlive", 2), ("d", 0), ("d", 129)):
        old = getattr(live, field)
        setattr(live, field, value)
        assert rad(ctypes.byref(runs), ctypes.byref(live)) == -1 and "bad sizes" in err()
        assert trav(ctypes.byref(a)) == -1 and "bad sizes" in err()
        setattr(live, field, old)
    runs.n_runs = 0
    assert rad(ctypes.byref(runs), ctypes.byref(live)) == -1 and "bad sizes" in err()
    runs.n_runs = 2
    bits = (ctypes.c_uint32 * 4)(0b1000, 0, 0, 0)
    live.order = 8
    assert rad(ctypes.byref(runs), ctypes.byref(live), bits) == -1 and "bit 3 set, but d = 3" in err()
    assert trav(ctypes.byref(a), bits) == -1 and "bit 3 set, but d = 3" in err()
    assert trav(None) == -1 and "args is NULL" in err()
    a.d = 4
    assert trav(ctypes.byref(a)) == -1 and "args->d == live->d" in err()
    a.d, a.k = 3, 0
    assert trav(ctypes.byref(a)) == -1 and "args->k > 0" in err()
    a.k = 4
    assert trav(ctypes.byref(a)) == -1 and "must be set" in err()  # args->u, run_of, start missing
    a.u, runs.run_of, live.start = 8, 8, 8
    assert trav(ctypes.byref(a), far=None) == -1 and "far must be set" in err()
