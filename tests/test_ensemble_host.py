"""
CPU tests of the ensemble sampler (evidence_b200.sampler_dev.nested_sample_ensemble): the C-ABI
structs, the host restatement of the set-up kernels (tests/_slice_runs_oracle.py), the walker layout
and the buffers, and argument validation.  The device side is tests/test_gpu_ensemble.py.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest

import _slice_runs_oracle as ro
from evidence_b200 import _abi
from evidence_b200.sampler_dev import _NativeSliceRuns, _ensemble_seeds, _walker_layout, nested_sample_ensemble
from oracle import slice_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_struct_sizes_match_the_header(built_lib):
    src = ('#include <stdio.h>\n#include "rvlnl.h"\nint main(){printf("%zu %zu\\n",'
           'sizeof(rvl_slice_runs),sizeof(rvl_slice_live));return 0;}')
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    assert got == [ctypes.sizeof(_abi.rvl_slice_runs), ctypes.sizeof(_abi.rvl_slice_live)] == [56, 72]


def test_initial_points_are_philox_uniforms():
    """Coordinate c of point p of run r: u01 of counter (0, TAG_INIT + c // 2, p, 0) under seeds[r];
    each run's points depend on its seed alone."""
    u = ro.init_points([7, 2 ** 64 - 1], 5, 3)
    for r, seed in enumerate([7, 2 ** 64 - 1]):
        for p in range(5):
            for c in range(3):
                x, y, z, w = so.philox4x32((0, ro.TAG_INIT + c // 2, p, 0), *so.key(seed))
                want = so.u01(z, w) if c & 1 else so.u01(x, y)
                assert u[r, p, c] == want
    assert np.array_equal(ro.init_points([2 ** 64 - 1], 5, 3)[0], u[1])
    assert np.all((u > 0) & (u < 1))


def test_start_draws():
    """A walker's start: survivor floor(x n / 2^32) of its run, x the first word of counter
    (round, TAG_START, j, 0); the same walker of the same run draws the same start whatever the
    layout, and the draws cover the survivors uniformly."""
    nlive, kk = 50, np.array([10, 3])
    order = np.stack([np.random.default_rng(r).permutation(nlive) for r in range(2)])
    run_of, walker_of = _walker_layout([10, 3])
    slots = ro.start_slots([11, 12], nlive, order, kk, run_of, walker_of, 4)
    x = so.philox4x32((4, ro.TAG_START, 2, 0), *so.key(12))[0]
    assert slots[10 + 2] == order[1][3 + (int(x) * (nlive - 3) >> 32)]
    alone = ro.start_slots([99, 12], nlive, order, kk, np.zeros(3, np.int32) + 1, np.arange(3), 4)
    assert np.array_equal(alone, slots[10:])
    assert set(slots[:10]) <= set(order[0][10:])
    many = ro.start_slots([5], nlive, order[:1], [10], np.zeros(20000, np.int32), np.arange(20000), 0)
    counts = np.bincount(many, minlength=nlive)[order[0][10:]]
    assert counts.min() > 0.8 * 20000 / 40 and counts.max() < 1.2 * 20000 / 40


def degenerate_points(nlive, d):
    """Points whose coordinate 1 repeats coordinate 0 exactly: the pivot of coordinate 1 is 1e-18
    plus rounding, and for these points (the survivors order[kk = 8:] = 8 .. nlive - 1) it rounds
    to <= 0."""
    u = np.random.default_rng(7).uniform(0.3, 0.7, (nlive, d))
    u[:, 1] = u[:, 0]
    return u


def test_whitening_restatement():
    """Without circular coordinates: the covariance of the survivors (numpy's, to rounding) and its
    Cholesky factor; a run whose survivors repeat one coordinate exactly falls back to the diagonal;
    with circular coordinates the factor does not depend on where on the circle the mode sits."""
    rng = np.random.default_rng(3)
    R, nlive, d = 3, 40, 4
    u = rng.uniform(0.3, 0.7, (R, nlive, d))
    order = np.argsort(rng.uniform(size=(R, nlive)), axis=1, kind="stable")
    kk = np.array([8, 1, 8])
    u[2] = degenerate_points(nlive, d)
    order[2] = np.arange(nlive)
    L, failed = ro.whiten(u, order, kk)
    assert failed.tolist() == [False, False, True]
    for r in range(2):
        cov = np.cov(u[r][order[r][kk[r]:]].T) + 1e-18 * np.eye(d)
        assert np.allclose(L[r] @ L[r].T, cov, rtol=1e-12, atol=1e-16)
        assert np.allclose(L[r], np.linalg.cholesky(cov), rtol=1e-12, atol=1e-16)
    cov2 = np.cov(u[2][order[2][8:]].T) + 1e-18 * np.eye(d)
    assert np.allclose(L[2], np.diag(np.sqrt(np.diag(cov2))), rtol=1e-13)
    wrap = np.array([True, False, False, True])
    a = rng.uniform(-0.05, 0.05, (1, nlive, d)) + 0.5
    b = a.copy()
    b[..., wrap] = ro._wrap_unit(b[..., wrap] + 0.5)  # the mode moved onto the seam
    La, _ = ro.whiten(a, order[:1], kk[:1], wrap)
    Lb, _ = ro.whiten(b, order[:1], kk[:1], wrap)
    assert np.allclose(La, Lb, rtol=1e-9, atol=1e-15)


def test_walker_layout():
    run_of, walker_of = _walker_layout([3, 0, 2, 1])
    assert run_of.tolist() == [0, 0, 0, 2, 2, 3] and walker_of.tolist() == [0, 1, 2, 0, 1, 0]
    assert run_of.dtype == walker_of.dtype == np.int32
    run_of, walker_of = _walker_layout([0, 0])  # every run finished
    assert len(run_of) == len(walker_of) == 0


def test_buffers_grow_for_a_plateau_round(built_lib):
    """Rounds of 2 x 8 walkers, then a plateau round with 8 + 30: the buffers grow once and are
    reused (views of the first k rows) when the round shrinks again."""
    import torch
    ns = _NativeSliceRuns(torch, 3, torch.device("cpu"), [1, 2], 50, n_out=2, m=3, rounds=2)
    ns.reserve(16)
    base = ns._full["cand"].data_ptr()
    assert ns.cand_o.shape == (16 * 4, 3) and ns.cand.shape == (16 * 3, 3) and ns.args.k == 16
    ns.reserve(38)
    assert ns.cap == 38 and ns.cand.shape == (38 * 3, 3) and ns.args.k == 38
    grown = ns._full["cand"].data_ptr()
    ns.reserve(8)
    assert ns.cap == 38 and ns._full["cand"].data_ptr() == grown != base
    assert ns.u.shape == (8, 3) and ns.args.k == 8 and ns.args.cand == grown
    assert ns.args.u == ns.u.data_ptr() and ns.live.start == ns.start.data_ptr()


def test_argument_validation():
    """Duplicate seeds (also after reduction to 64 bits), no seeds, and a wrap mask of the wrong
    length are rejected before anything reaches a device."""
    fused = None
    with pytest.raises(ValueError, match="more than once"):
        nested_sample_ensemble(fused, 3, [1, 2, 1])
    with pytest.raises(ValueError, match="more than once"):
        _ensemble_seeds([5, 5 + 2 ** 64])
    with pytest.raises(ValueError, match="at least one seed"):
        nested_sample_ensemble(fused, 3, [])
    with pytest.raises(ValueError, match="entries for 3 dimensions"):
        nested_sample_ensemble(fused, 3, [1, 2], wrapped=[True, False])
    with pytest.raises(ValueError, match="CUDA"):
        nested_sample_ensemble(fused, 3, [1, 2], device="cpu")


def test_abi_argument_checks(built_lib):
    """The new entry points check their arguments on the host: RVL_EINVAL and a message."""
    lib = _abi.load()
    a = _abi.rvl_slice_args(k=4, d=3, n_out=2, m=2)
    runs = _abi.rvl_slice_runs(n_runs=2)
    assert lib.rvl_slice_phase_runs(0, ctypes.byref(a), None, None, None) == -1
    assert "runs is NULL" in lib.rvl_slice_last_error().decode()
    assert lib.rvl_slice_phase_runs(0, ctypes.byref(a), ctypes.byref(runs), None, None) == -1
    assert "must all be set" in lib.rvl_slice_last_error().decode()
    runs.n_runs = 0
    assert lib.rvl_slice_phase_runs(0, ctypes.byref(a), ctypes.byref(runs), None, None) == -1
    assert "n_runs" in lib.rvl_slice_last_error().decode()
    bits = (ctypes.c_uint32 * 4)(0b1000, 0, 0, 0)
    assert lib.rvl_slice_phase_runs(0, ctypes.byref(a), ctypes.byref(runs), bits, None) == -1
    assert "bit 3 set, but d = 3" in lib.rvl_slice_last_error().decode()
    live = _abi.rvl_slice_live(nlive=2, d=3)
    runs.n_runs = 1
    for fn in (lambda: lib.rvl_slice_runs_init(ctypes.byref(runs), ctypes.byref(live), None),
               lambda: lib.rvl_slice_runs_whiten(ctypes.byref(runs), ctypes.byref(live), None, None),
               lambda: lib.rvl_slice_runs_starts(ctypes.byref(a), ctypes.byref(runs), ctypes.byref(live), None)):
        assert fn() == -1
        assert "bad sizes" in lib.rvl_slice_last_error().decode()
    live.nlive, runs.seeds, live.u_live = 10, 8, 8
    assert lib.rvl_slice_runs_whiten(ctypes.byref(runs), ctypes.byref(live), None, None) == -1
    assert "must be set" in lib.rvl_slice_last_error().decode()
    a.d = 4
    assert lib.rvl_slice_runs_starts(ctypes.byref(a), ctypes.byref(runs), ctypes.byref(live), None) == -1
    assert "args->d == live->d" in lib.rvl_slice_last_error().decode()
