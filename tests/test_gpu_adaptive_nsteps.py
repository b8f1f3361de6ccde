"""
The adaptive number of moves on the GPU: `rvl_slice_runs_radius` / `_travel` against their host
restatement (tests/_slice_travel_oracle.py), bit for bit; the samplers with adaptive_nsteps =
'move-distance' and max_nsteps = nsteps against the fixed ones; the independence of the runs of an
ensemble with adaptive moves; the evidence of a Gaussian started from too few moves; the runner.
"""
import ctypes
import math

import numpy as np
import pytest

import _slice_travel_oracle as to
from test_gpu_ensemble import gauss_columns
from test_gpu_slice_kernels import same_bits

pytestmark = pytest.mark.gpu

SENT_RAD, SENT_FAR = -7.25e300, -5


def _factor(rng, d):
    """A lower factor with positive diagonal and NaN above it (never read)."""
    L = np.tril(rng.normal(0.0, 0.05 / np.sqrt(d), (d, d)), -1) + np.diag(rng.uniform(0.05, 0.2, d))
    L[np.triu_indices(d, 1)] = np.nan
    return L


def _case(d, nlive, R, wrapped, seed):
    """Live points, orders and kk of R runs (run 1: kk = 0; run 2: two survivors; the survivors of run 0
    include a duplicate pair and a pair exactly 1/2 apart in coordinate 0), factors, a wrap mask with
    points on both sides of the seam, and walkers: some stuck on their start, some moved a little,
    some far, a few of the kk = 0 run (ignored)."""
    rng = np.random.default_rng([d, nlive, R, wrapped, seed])
    u = rng.uniform(size=(R, nlive, d))
    wrap = None
    if wrapped:
        wrap = rng.uniform(size=d) < 0.5
        wrap[0] = True
        seam = np.where(rng.uniform(size=(R, nlive)) < 0.5, rng.uniform(0.97, 1.0, (R, nlive)),
                        rng.uniform(0.0, 0.03, (R, nlive)))
        u[:, :, 0] = seam
    order = np.stack([rng.permutation(nlive) for _ in range(R)])
    kk = rng.integers(1, max(2, nlive // 4), size=R)
    kk[1 % R] = 0 if R > 1 else kk[0]
    if R > 2:
        kk[2] = nlive - 2
    s0 = order[0][kk[0]:]
    u[0, s0[1]] = u[0, s0[0]]                       # a duplicate pair
    u[0, s0[2], 0], u[0, s0[3], 0] = 0.25, 0.75      # delta_0 = -1/2 exactly
    chol = np.stack([_factor(rng, d) for _ in range(R)])
    runs = [r for r in range(R) if kk[r] > 0]
    K = 6 * R
    run_of = rng.choice(runs, size=K).astype(np.int32)
    if R > 1:
        run_of[:2] = 1  # walkers of a run with kk = 0: ignored
    start = np.array([order[r][kk[r] + rng.integers(0, max(1, nlive - kk[r]))] for r in run_of], np.int64)
    u_start = u[run_of, start]
    step = rng.normal(size=(K, d)) * 0.002
    u_end = np.clip(u_start + step, 0.0, 1.0 - 2.0 ** -53)
    if wrap is not None:
        q = u_start + step
        u_end[:, wrap] = (q - np.floor(q))[:, wrap]
    kind = rng.uniform(size=K)
    u_end[kind < 0.3] = u_start[kind < 0.3]                 # stuck
    u_end[kind > 0.65] = 1.0 - u_start[kind > 0.65]         # the mirrored point: far in any d
    return u, order, kk, chol, wrap, run_of, start, u_end


def _bits(wrap):
    from evidence_b200.sampler_dev import _wrap_bits
    return _wrap_bits(wrap)


def _run_kernels(u, order, kk, chol, wrap, run_of, start, u_end):
    import torch
    from evidence_b200 import _abi
    lib = _abi.load()
    R, nlive, d = u.shape
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    t = dict(u=cuda(u), order=cuda(order.astype(np.int64)), kk=cuda(kk.astype(np.int64)), chol=cuda(chol),
             run_of=cuda(run_of), start=cuda(start), u_end=cuda(u_end),
             rad2=cuda(np.full(R, SENT_RAD)), far=cuda(np.full(R, SENT_FAR, np.int32)))
    runs = _abi.rvl_slice_runs(n_runs=R, run_of=t["run_of"].data_ptr(), chol=t["chol"].data_ptr())
    live = _abi.rvl_slice_live(nlive=nlive, d=d, u_live=t["u"].data_ptr(), order=t["order"].data_ptr(),
                               kk=t["kk"].data_ptr(), start=t["start"].data_ptr())
    args = _abi.rvl_slice_args(k=len(run_of), d=d, u=t["u_end"].data_ptr())
    bits = _bits(wrap)
    stream = torch.cuda.current_stream().cuda_stream
    assert lib.rvl_slice_runs_radius(ctypes.byref(runs), ctypes.byref(live), bits, t["rad2"].data_ptr(),
                                     stream) == 0, lib.rvl_slice_last_error().decode()
    assert lib.rvl_slice_runs_travel(ctypes.byref(args), ctypes.byref(runs), ctypes.byref(live), bits,
                                     t["rad2"].data_ptr(), t["far"].data_ptr(), stream) == 0, \
        lib.rvl_slice_last_error().decode()
    torch.cuda.synchronize()
    return t["rad2"].cpu().numpy(), t["far"].cpu().numpy()


@pytest.mark.parametrize("wrapped", [False, True])
@pytest.mark.parametrize("d, nlive, R", [(2, 650, 5), (7, 200, 64), (26, 650, 3), (128, 80, 3)])
def test_kernels_match_the_restatement(d, nlive, R, wrapped):
    u, order, kk, chol, wrap, run_of, start, u_end = _case(d, nlive, R, wrapped, 0)
    rad2, far = _run_kernels(u, order, kk, chol, wrap, run_of, start, u_end)
    want_rad2 = to.radius(u, order, kk, chol, wrap, rad2=np.full(R, SENT_RAD))
    assert same_bits(rad2, want_rad2)
    want_far = to.travel(u_end, run_of, start, u, kk, chol, want_rad2, wrap, far=np.full(R, SENT_FAR))
    assert np.array_equal(far, want_far)
    skipped = kk == 0
    assert np.all(rad2[skipped] == SENT_RAD) and np.all(far[skipped] == SENT_FAR)
    assert np.all(rad2[~skipped] >= 0) and np.all(far[~skipped] >= 0)
    assert 0 < far[~skipped].sum() < np.isin(run_of, np.flatnonzero(~skipped)).sum()  # both kinds occur
    # a run's values do not depend on the others: run 0 alone
    u0, o0, k0, c0 = u[:1], order[:1], kk[:1], chol[:1]
    sel = run_of == 0
    r1, f1 = _run_kernels(u0, o0, k0, c0, wrap, run_of[sel], start[sel], u_end[sel])
    assert same_bits(r1, rad2[:1]) and f1[0] == far[0]


def _gauss_kw():
    return dict(nlive=100, nsteps=8, device="cuda")


def _same_run(x, y, exact_logz):
    for f in ("samples", "weighted_samples", "logl"):
        assert same_bits(x[f], y[f]), f
    assert (x.ncall, x.niter, x.accepted_moves, x.unresolved_moves) == (
        y.ncall, y.niter, y.accepted_moves, y.unresolved_moves)
    if exact_logz:
        assert x.logz == y.logz and x.logzerr == y.logzerr
    else:
        assert abs(x.logz - y.logz) <= 1e-12 and abs(x.logzerr - y.logzerr) <= 1e-9


def test_cap_at_nsteps_is_the_fixed_sampler():
    """adaptive_nsteps='move-distance' with max_nsteps = nsteps: the runs of adaptive_nsteps=None, bit
    for bit, for the ensemble and for the single-run sampler (wrapped too); every round at nsteps."""
    from evidence_b200.sampler_dev import nested_sample_device, nested_sample_ensemble
    kw = _gauss_kw()
    a = nested_sample_ensemble(gauss_columns, 4, [3, 4, 5], **kw)
    b = nested_sample_ensemble(gauss_columns, 4, [3, 4, 5], adaptive_nsteps="move-distance", max_nsteps=8, **kw)
    for x, y in zip(a, b):
        _same_run(x, y, True)
        assert x.nsteps_history is None and set(y.nsteps_history) == {8}
        assert len(y.nsteps_history) == (y.ncall - 100) // (20 * 8 * 40)
    for wrapped in (None, [True, False, False, True]):
        x = nested_sample_device(gauss_columns, 4, seed=7, wrapped=wrapped, **kw)
        y = nested_sample_device(gauss_columns, 4, seed=7, wrapped=wrapped, adaptive_nsteps="move-distance",
                                 max_nsteps=8, **kw)
        _same_run(x, y, True)
        assert set(y.nsteps_history) == {8} and len(y.nsteps_history) == x.niter // 20


def test_runs_do_not_interact_with_adaptive_moves():
    """R = 6 runs with adaptive moves (nsteps 2, cap 8) on a likelihood whose rows do not depend on the
    batch: each run equals the same seed run alone -- chain, nsteps_history, ncall, ln Z to 1e-12 --
    and the runs' histories differ (so moves launched prefixes of the walkers)."""
    from evidence_b200.sampler_dev import nested_sample_ensemble
    kw = dict(nlive=100, nsteps=2, device="cuda", adaptive_nsteps="move-distance")
    seeds = [11, 12, 13, 14, 15, 16]
    ens = nested_sample_ensemble(gauss_columns, 4, seeds, **kw)
    for s, x in zip(seeds, ens):
        y = nested_sample_ensemble(gauss_columns, 4, [s], **kw)[0]
        _same_run(x, y, False)
        assert x.nsteps_history == y.nsteps_history
        per_move = 2 * 8 + 3 * 8
        assert x.ncall == 100 + sum(20 * n * per_move for n in x.nsteps_history)
    hist = [tuple(r.nsteps_history) for r in ens]
    assert len(set(hist)) >= 2, hist
    assert all(2 <= n <= 8 for h in hist for n in h)


ND10, SIG10 = 10, 0.6
LNZ10 = ND10 * math.log(math.sqrt(2 * math.pi) * SIG10 / 20)


def gauss10(U):
    """A d = 10 Gaussian of width 0.6 in a box of 20 (ln Z = LNZ10); rows independent of the batch."""
    th = -10 + 20 * U
    return th, -0.5 * ((th / SIG10) ** 2).sum(1)


def _lnz_stats(res):
    z = np.array([r.logz for r in res])
    return z.mean(), z.std(ddof=1) / math.sqrt(len(z))


def test_adaptive_moves_engage_from_too_few():
    """The d = 10 Gaussian started at nsteps = 2 (cap 40), R = 16: every run's count rises above 2, and
    the mean ln Z lies closer to the analytic value than that of the same runs at a fixed 2 moves; the
    single-run sampler adapts too.  The rule does not promise an unbiased ln Z from such a start: it
    settles where about half the walkers leave the largest nearest-neighbour gap of the survivors,
    9 - 13 moves here, which leaves ln Z about 0.5 high (DESIGN.md section 9.1)."""
    from evidence_b200.sampler_dev import nested_sample_device, nested_sample_ensemble
    seeds = list(range(200, 216))
    ada = nested_sample_ensemble(gauss10, ND10, seeds, nlive=200, nsteps=2, max_nsteps=40,
                                 adaptive_nsteps="move-distance", device="cuda")
    fix = nested_sample_ensemble(gauss10, ND10, seeds, nlive=200, nsteps=2, device="cuda")
    (ma, sa), (mf, sf) = _lnz_stats(ada), _lnz_stats(fix)
    top = [max(r.nsteps_history) for r in ada]
    print(f"adaptive 2..40: mean {ma:.3f} (se {sa:.3f}), fixed 2: mean {mf:.3f} (se {sf:.3f}), analytic "
          f"{LNZ10:.3f}; max n per run {top}, median {[int(np.median(r.nsteps_history)) for r in ada]}")
    assert all(t > 2 for t in top), top
    assert abs(ma - LNZ10) < abs(mf - LNZ10), (ma, mf, LNZ10)
    one = nested_sample_device(gauss10, ND10, nlive=200, nsteps=2, seed=3, adaptive_nsteps="move-distance",
                               device="cuda")
    assert max(one.nsteps_history) > 2 and np.isfinite(one.logz)


def test_adaptive_moves_keep_the_evidence():
    """The d = 10 Gaussian started at the reference's 3 ndim = 30 moves (default cap 120), R = 16: no
    round goes below 30, and the mean ln Z lies within 3 standard errors of the analytic value."""
    from evidence_b200.sampler_dev import nested_sample_ensemble
    res = nested_sample_ensemble(gauss10, ND10, list(range(200, 216)), nlive=200, nsteps=30,
                                 adaptive_nsteps="move-distance", device="cuda")
    m, se = _lnz_stats(res)
    print(f"adaptive 30..120: mean {m:.3f} (se {se:.3f}), analytic {LNZ10:.3f}; "
          f"max n per run {[max(r.nsteps_history) for r in res]}")
    assert all(min(r.nsteps_history) >= 30 and max(r.nsteps_history) <= 120 for r in res)
    assert abs(m - LNZ10) < 3 * se, (m, LNZ10, se)


def test_runner(tmp_path):
    """run() with 'slice-device' and run_ensemble with 'builtin_adaptive_nsteps': 'move-distance':
    the outputs carry the history and the implementation string names it."""
    from evidence_b200 import synth
    from evidence_b200 import ultranest as runner
    from evidence_b200.rvmodel import RVModel
    case = synth.make_case(1, seed=4, n_epochs=96)
    model = RVModel(case.fixedpardict, case.datadict(pandas=True), case.parnames)
    settings = {"nlive": 100, "nsteps": 4, "seed": 40, "sampler": "builtin", "builtin_method": "slice-device",
                "builtin_adaptive_nsteps": "move-distance"}
    rundict = {"target": "synth", "runid": "ad", "save_dir": str(tmp_path), "nplanets": 1}
    out = runner.run(model, dict(rundict), case.priordict, settings)
    assert "adaptive nsteps (move-distance)" in out.sampler_impl and np.isfinite(out.logZ)
    assert len(out.nsteps_history) > 0 and min(out.nsteps_history) >= 4 and max(out.nsteps_history) <= 16
    outs = runner.run_ensemble(model, dict(rundict, runid="ade"), case.priordict, settings, nruns=2)
    for o in outs:
        assert "adaptive nsteps (move-distance)" in o.sampler_impl and np.isfinite(o.logZ)
        assert len(o.nsteps_history) > 0 and min(o.nsteps_history) >= 4
    plain = runner.run(model, dict(rundict, runid="plain"), case.priordict,
                       dict(settings, builtin_adaptive_nsteps=False))
    assert "adaptive" not in plain.sampler_impl and not hasattr(plain, "nsteps_history")
    model.close()
