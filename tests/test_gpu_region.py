"""
MLFriends region sampling on the GPU: `rvl_region_runs_radius` / `_draw` / `_pick` against their host
restatement (tests/_region_oracle.py); uniform device draws on a union of discs and on a torus; the
independence of the runs of an ensemble; ln Z of analytic problems at R = 32; the runner.
"""
import ctypes
import math

import numpy as np
import pytest
from scipy import integrate, special

import _region_oracle as ro
from test_gpu_adaptive_nsteps import _case
from test_gpu_ensemble import gauss_columns
from test_gpu_slice_kernels import same_bits
from test_region_host import _cells_inside, _uniform_p

pytestmark = pytest.mark.gpu

SENT_RAD = -7.25e300


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


class _Dev:
    """Device copies of a case and the structs of the region entry points."""

    def __init__(self, seeds, u, order, kk, chol, round_no):
        import torch
        from evidence_b200 import _abi
        self.lib = _abi.load()
        R, nlive, d = u.shape
        self.t = dict(seeds=_cuda(np.array(seeds, np.uint64).view(np.int64)), u=_cuda(u),
                      order=_cuda(np.asarray(order, np.int64)), kk=_cuda(np.asarray(kk, np.int64)), chol=_cuda(chol),
                      rad2=_cuda(np.full(R, SENT_RAD)), count=torch.zeros(R, dtype=torch.int32, device="cuda"),
                      offs=torch.zeros(R + 1, dtype=torch.int32, device="cuda"))
        t = self.t
        self.runs = _abi.rvl_slice_runs(n_runs=R, seeds=t["seeds"].data_ptr(), chol=t["chol"].data_ptr())
        self.live = _abi.rvl_slice_live(nlive=nlive, d=d, round=round_no, u_live=t["u"].data_ptr(),
                                        order=t["order"].data_ptr(), kk=t["kk"].data_ptr())
        self.g = _abi.rvl_region_args(rad2=t["rad2"].data_ptr(), count=t["count"].data_ptr(),
                                      offs=t["offs"].data_ptr())
        self.d, self.R = d, R

    def _err(self, rc):
        assert rc == 0, self.lib.rvl_slice_last_error().decode()

    def radius(self, nboot, bits):
        import torch
        self.g.num_bootstraps = nboot
        self._err(self.lib.rvl_region_runs_radius(ctypes.byref(self.g), ctypes.byref(self.runs),
                                                  ctypes.byref(self.live), bits, torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        return self.t["rad2"].cpu().numpy()

    def draw(self, rad2, slot_base, batch, bits):
        """(stage, flag, count, offs, cand) after one draw."""
        import torch
        S, d = int(slot_base[-1]), self.d
        t = self.t
        t["rad2"].copy_(torch.from_numpy(np.asarray(rad2, np.float64)))
        t.update(base=_cuda(np.asarray(slot_base, np.int32)), stage=torch.full((max(S, 1), d), np.nan,
                 dtype=torch.float64, device="cuda"), flag=torch.full((max(S, 1),), 7, dtype=torch.uint8, device="cuda"),
                 cand=torch.full((max(S, 1), d), np.nan, dtype=torch.float64, device="cuda"))
        g = self.g
        g.batch, g.max_slots = batch, int(np.diff(slot_base).max())
        g.slot_base, g.stage, g.flag, g.cand = (t[n].data_ptr() for n in ("base", "stage", "flag", "cand"))
        self._err(self.lib.rvl_region_runs_draw(ctypes.byref(g), ctypes.byref(self.runs), ctypes.byref(self.live),
                                                bits, torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        return (t["stage"].cpu().numpy()[:S], t["flag"].cpu().numpy()[:S], t["count"].cpu().numpy(),
                t["offs"].cpu().numpy(), t["cand"].cpu().numpy())


def _bits(wrap):
    from evidence_b200.sampler_dev import _wrap_bits
    return _wrap_bits(wrap)


@pytest.mark.parametrize("wrapped", [False, True])
@pytest.mark.parametrize("d, nlive, R, nboot", [(2, 650, 5, 4), (7, 200, 64, 3), (15, 375, 4, 5), (40, 120, 3, 3)])
def test_radius_matches_the_restatement(d, nlive, R, nboot, wrapped):
    """Bit for bit, d = 2..40, n up to 650, R up to 64; a run with kk = 0 keeps its value; a run's
    radius does not depend on the other runs."""
    u, order, kk, chol, wrap, *_ = _case(d, nlive, R, wrapped, 1)
    seeds = [1000 + 7 * r for r in range(R)]
    got = _Dev(seeds, u, order, kk, chol, 9).radius(nboot, _bits(wrap))
    want = ro.radius(seeds, u, order, kk, chol, nboot, 9, wrap, rad2=np.full(R, SENT_RAD))
    assert same_bits(got, want)
    assert np.all(got[kk == 0] == SENT_RAD) and np.all(got[kk > 0] > 0)
    alone = _Dev(seeds[:1], u[:1], order[:1], kk[:1], chol[:1], 9).radius(nboot, _bits(wrap))
    assert same_bits(alone, got[:1])


@pytest.mark.parametrize("wrapped", [False, True])
@pytest.mark.parametrize("d, nlive, R", [(2, 300, 4), (7, 200, 8), (15, 375, 3)])
def test_draw_matches_the_restatement(d, nlive, R, wrapped):
    """Every accepted candidate within 1e-12 of the restatement's (device log, sin, cos, pow against
    numpy's); accept flags identical except where a test sits within 1e-12 of a ball surface or cube
    face (their number is printed); the compacted rows are the accepted slots, run by run in slot
    order, with counts and offsets to match; a run with kk = 0 draws nothing."""
    u, order, kk, chol, wrap, *_ = _case(d, nlive, R, wrapped, 2)
    # survivors in the middle of the cube (the circular coordinate keeps its points on the seam) and
    # balls of a few tenths of the cube: all three rules reject some candidates
    rng = np.random.default_rng([d, R])
    if wrap is None:
        u = 0.5 + (u - 0.5) * 0.6
    else:
        u = np.where(wrap, u, 0.5 + (u - 0.5) * 0.6)
    rad2 = rng.uniform(0.3, 3.0, R)
    slots = rng.integers(50, 3000, R)
    slots[kk == 0] = 40          # slots of a finished run: nothing drawn
    base = np.concatenate([[0], np.cumsum(slots)])
    seeds = [2 ** 64 - 1 - r for r in range(R)]
    dev = _Dev(seeds, u, order, kk, chol, 4)
    stage, flag, count, offs, cand = dev.draw(rad2, base, 3, _bits(wrap))
    x, want, near, wcount, woffs, _ = ro.draw(seeds, u, order, kk, chol, rad2, base, 3, 4, wrap)
    live = np.repeat(kk > 0, slots)
    assert np.all(flag[~live] == 7)                      # a run with kk = 0 is skipped: flags untouched
    flag = flag.astype(bool) & live
    differ = flag != want
    print(f"d {d} R {R} wrapped {wrapped}: {len(flag)} slots, {flag.sum()} accepted, {near.sum()} near a "
          f"surface or face, {differ.sum()} flags differ")
    assert not np.any(differ & ~near)
    both = flag & want
    assert np.all(np.abs(stage[both] - x[both]) <= 1e-12)
    assert 0 < flag.sum() < len(flag)
    for r in range(R):
        sl = slice(base[r], base[r + 1])
        assert count[r] == flag[sl].sum()
        assert same_bits(cand[offs[r]:offs[r + 1]], stage[sl][flag[sl]])
        if kk[r] == 0:
            assert count[r] == 0
    assert offs[0] == 0 and np.array_equal(np.diff(offs), count)
    if not differ.any():
        assert np.array_equal(count, wcount) and np.array_equal(offs, woffs)


def test_pick_matches_the_restatement():
    """Bit for bit: R = 5 runs (one with kk = 0, one filled before the batch), walkers interleaved at
    random, rows above and below each run's constraint."""
    import torch
    from evidence_b200 import _abi
    lib = _abi.load()
    rng = np.random.default_rng(5)
    R, d, nlive = 5, 6, 60
    kk = np.array([12, 0, 5, 30, 7])
    filled0 = np.array([3, 0, 5, 0, 6])
    rows = np.array([40, 0, 10, 25, 3])
    offs = np.concatenate([[0], np.cumsum(rows)])
    N = int(offs[-1])
    cand, cand_th, cand_ll = rng.uniform(size=(N, d)), rng.normal(size=(N, d)), rng.normal(size=N)
    lmin = rng.normal(size=R) * 0.5
    run_of = np.repeat(np.arange(R, dtype=np.int32), kk)
    walker_of = np.concatenate([np.arange(k) for k in kk]).astype(np.int32)
    perm = rng.permutation(len(run_of))
    run_of, walker_of = run_of[perm], walker_of[perm]
    K = len(run_of)
    u0, th0, lc0 = rng.uniform(size=(K, d)), rng.uniform(size=(K, d)), np.full(K, np.nan)
    t = dict(kk=_cuda(kk.astype(np.int64)), lmin=_cuda(lmin), offs=_cuda(offs.astype(np.int32)), cand=_cuda(cand),
             th=_cuda(cand_th), ll=_cuda(cand_ll), sel=torch.zeros(N, dtype=torch.int32, device="cuda"),
             run_of=_cuda(run_of), walker_of=_cuda(walker_of), u=_cuda(u0), theta=_cuda(th0), lcur=_cuda(lc0),
             fa=_cuda(np.stack([filled0, np.full(R, -9)]).astype(np.int32)))
    g = _abi.rvl_region_args(offs=t["offs"].data_ptr(), cand=t["cand"].data_ptr(), cand_th=t["th"].data_ptr(),
                             cand_ll=t["ll"].data_ptr(), sel=t["sel"].data_ptr(), filled=t["fa"][0].data_ptr(),
                             above=t["fa"][1].data_ptr())
    runs = _abi.rvl_slice_runs(n_runs=R, run_of=t["run_of"].data_ptr(), walker_of=t["walker_of"].data_ptr(),
                               lmin=t["lmin"].data_ptr())
    live = _abi.rvl_slice_live(nlive=nlive, d=d, kk=t["kk"].data_ptr())
    args = _abi.rvl_slice_args(k=K, d=d, u=t["u"].data_ptr(), theta=t["theta"].data_ptr(), lcur=t["lcur"].data_ptr())
    assert lib.rvl_region_runs_pick(ctypes.byref(g), ctypes.byref(args), ctypes.byref(runs), ctypes.byref(live),
                                    None) == 0, lib.rvl_slice_last_error().decode()
    torch.cuda.synchronize()
    wu, wth, wlc, wf, wa = ro.pick(kk, lmin, offs, cand, cand_th, cand_ll, run_of, walker_of, u0, th0, lc0, filled0)
    assert same_bits(t["u"].cpu().numpy(), wu) and same_bits(t["theta"].cpu().numpy(), wth)
    assert same_bits(t["lcur"].cpu().numpy(), wlc)
    fa = t["fa"].cpu().numpy()
    assert np.array_equal(fa[0], wf)
    assert np.array_equal(fa[1][kk > 0], wa[kk > 0]) and fa[1][1] == -9   # kk = 0: untouched
    assert 0 < np.isfinite(wlc).sum() < K


def _device_draws(seeds, u, order, kk, chol, rad2, wrap, batches=10, slots=20000):
    dev = _Dev(seeds, u, order, kk, chol, 0)
    out = []
    for b in range(batches):
        stage, flag, *_ = dev.draw(rad2, [0, slots], b, _bits(wrap))
        out.append(stage[flag.astype(bool)])
    return np.concatenate(out)


def test_device_draws_uniform_on_overlapping_discs():
    """The discs of test_region_host.test_draws_uniform_on_overlapping_discs, 200000 device slots."""
    centres = np.array([[0.9, 0.9], [0.3, 0.4], [0.45, 0.5], [0.35, 0.6]])
    x = _device_draws([17], centres[None], np.array([[0, 1, 2, 3]]), np.array([1]), np.array([2.0 * np.eye(2)]),
                      np.array([0.0081]), None)

    def member(p):
        return (((p[:, None, :] - centres[None, 1:, :]) ** 2).sum(-1) <= 0.18 ** 2 * (1 + 1e-12)).any(1)
    assert member(x).all() and len(x) > 100000
    p, obs = _uniform_p(x, _cells_inside(member, 24), 24)
    assert p > 1e-3, (p, obs.min(), obs.max())


def test_device_draws_uniform_on_a_torus():
    """The torus of test_region_host.test_draws_uniform_on_a_torus (balls wider than half the circle)."""
    centres = np.array([[0.0, 0.0], [0.5, 0.45], [0.1, 0.55]])
    wrap = np.array([True, False])
    x = _device_draws([23], centres[None], np.array([[0, 1, 2]]), np.array([1]), np.array([np.diag([1.0, 0.2])]),
                      np.array([0.49]), wrap)

    def member(p):
        dl = p[:, None, :] - centres[None, 1:, :]
        dl[..., 0] -= np.rint(dl[..., 0])
        return ((dl[..., 0] ** 2 + (dl[..., 1] / 0.2) ** 2) <= 0.49 * (1 + 1e-12)).any(1)
    assert member(x).all() and (x[:, 0] >= 0).all() and (x[:, 0] < 1).all()
    p, obs = _uniform_p(x, _cells_inside(member, 20), 20)
    assert p > 1e-3, (p, obs.min(), obs.max())


def _same_run(x, y):
    for f in ("samples", "weighted_samples", "logl"):
        assert same_bits(x[f], y[f]), f
    assert (x.ncall, x.niter, x.region_draws) == (y.ncall, y.niter, y.region_draws)
    assert abs(x.logz - y.logz) <= 1e-12 and abs(x.logzerr - y.logzerr) <= 1e-9


def test_runs_do_not_interact():
    """With a likelihood whose rows do not depend on the batch, the run of seed 5 is the same in the
    ensembles [3, 4, 5, 6], [5] and [6, 5, 3] (chain, ncall, region draws, ln Z to 1e-12); the runs
    differ from each other and report the method."""
    from evidence_b200.sampler_dev import nested_sample_ensemble
    kw = dict(nlive=100, device="cuda", method="mlfriends")
    a = nested_sample_ensemble(gauss_columns, 4, [3, 4, 5, 6], **kw)
    b = nested_sample_ensemble(gauss_columns, 4, [5], **kw)
    c = nested_sample_ensemble(gauss_columns, 4, [6, 5, 3], **kw)
    _same_run(a[2], b[0])
    _same_run(a[2], c[1])
    _same_run(a[0], c[2])
    assert len({r.ncall for r in a}) > 1
    for r in a:
        assert r.method == "mlfriends-device-ensemble" and r.region_draws >= r.ncall - 100 > 0
        assert r.accepted_moves == 0 and r.nsteps_history is None


# ---- analytic evidence, R = 32 -------------------------------------------------------------------
def _check_lnz(res, want, tag):
    z = np.array([r.logz for r in res])
    err = np.median([r.logzerr for r in res])
    se = z.std(ddof=1) / math.sqrt(len(z))
    print(f"{tag}: mean {z.mean():.4f} (analytic {want:.4f}, se {se:.4f}), std {z.std(ddof=1):.4f}, "
          f"median logzerr {err:.4f}, calls/run {np.mean([r.ncall for r in res]):.0f}, "
          f"region draws/run {np.mean([r.region_draws for r in res]):.0f}")
    assert abs(z.mean() - want) < 3 * se, (z.mean(), want, se)
    assert z.std(ddof=1) < 1.5 * err, (z.std(ddof=1), err)


def _ensemble(fused, ndim, nlive, **kw):
    from evidence_b200.sampler_dev import nested_sample_ensemble
    return nested_sample_ensemble(fused, ndim, list(range(300, 332)), nlive=nlive, device="cuda",
                                  method="mlfriends", **kw)


def test_gaussian():
    """The d = 4 Gaussian of test_gpu_ensemble.test_analytic_evidence."""
    ndim, sig = 4, 0.6

    def fused(U):
        th = -10 + 20 * U
        return th, -0.5 * ((th / sig) ** 2).sum(1)
    _check_lnz(_ensemble(fused, ndim, 250), ndim * math.log(math.sqrt(2 * math.pi) * sig / 20), "gaussian d 4")


MIX_D, MIX_W = 6, (0.75, 0.25)
MIX_S = (0.04, 0.04 * (MIX_W[1] / MIX_W[0]) ** (1 / MIX_D))


def mixture(U):
    """Two normalised Gaussians at u = 0.3 and 0.7 (every coordinate), weights 3/4 and 1/4, widths 0.04
    and 0.04 (1/3)^(1/6), so that both peaks have the same lnL: ln Z = ln(sum of the weights times
    their mass in the cube) = 0 to 1e-30."""
    import torch
    out = []
    for w, s, c in zip(MIX_W, MIX_S, (0.3, 0.7)):
        out.append(math.log(w) - MIX_D * math.log(s * math.sqrt(2 * math.pi)) - 0.5 * (((U - c) / s) ** 2).sum(1))
    return U.clone(), torch.logaddexp(out[0], out[1])


def test_gaussian_mixture():
    """Two separated modes of unequal weight and equal peak height, d = 6: both kept to the end (the
    mean is right and the scatter follows the reported error).  A mode whose peak lies below the
    other's dies out before the end, and its last survivors then stretch the bootstrapped radius
    across both modes; without clustering the efficiency collapses there (DESIGN.md section 9.1)."""
    _check_lnz(_ensemble(mixture, MIX_D, 300), 0.0, "mixture d 6")


SHELL_R, SHELL_W, SHELL_C, SHELL_BOX = 2.0, 0.1, 3.5, 6.0


def shells(d):
    def fused(U):
        import torch
        th = SHELL_BOX * (2 * U - 1)
        out = []
        for sgn in (-1.0, 1.0):
            x = th.clone()
            x[:, 0] = x[:, 0] - sgn * SHELL_C
            rho = torch.sqrt((x ** 2).sum(1))
            out.append(-0.5 * ((rho - SHELL_R) / SHELL_W) ** 2 - math.log(SHELL_W * math.sqrt(2 * math.pi)))
        return th, torch.logaddexp(out[0], out[1])
    return fused


def shells_lnz(d):
    """Two disjoint shells inside the box: ln Z = ln(2 S_(d-1) int rho^(d-1) g(rho) drho / (2 box)^d), g the
    normalised radial Gaussian, S_(d-1) = 2 pi^(d/2) / Gamma(d/2) -- a 1-D quadrature."""
    g = lambda r: r ** (d - 1) * math.exp(-0.5 * ((r - SHELL_R) / SHELL_W) ** 2) / (SHELL_W * math.sqrt(2 * math.pi))  # noqa: E731
    radial, _ = integrate.quad(g, 0.0, SHELL_R + 20 * SHELL_W, points=[SHELL_R], epsabs=0, epsrel=1e-12)
    area = 2 * math.pi ** (d / 2) / special.gamma(d / 2)
    return math.log(2 * area * radial) - d * math.log(2 * SHELL_BOX)


@pytest.mark.parametrize("d", [2, 5])
def test_gaussian_shells(d):
    _check_lnz(_ensemble(shells(d), d, 300), shells_lnz(d), f"shells d {d}")


def test_wrapped_von_mises():
    """The periodic problem of test_slice_wrap (two von Mises coordinates with the mode on the seam,
    three narrow Gaussians) with its mask."""
    from test_slice_wrap import KAPPA, PERIODIC_LNZ, PERIODIC_WRAP, S

    def fused(U):
        import torch
        ll = (KAPPA * (torch.cos(2 * math.pi * U[:, :2]) - 1.0)).sum(1) - (((U[:, 2:] - 0.5) ** 2) / (2 * S * S)).sum(1)
        return U.clone(), ll
    _check_lnz(_ensemble(fused, 5, 200, wrapped=PERIODIC_WRAP), float(PERIODIC_LNZ), "von Mises d 5, wrapped")


def test_runner(tmp_path):
    """run() and run_ensemble with 'builtin_method': 'mlfriends-device' (the wrap mask applied);
    'builtin_adaptive_nsteps' is rejected with it."""
    from evidence_b200 import synth
    from evidence_b200 import ultranest as runner
    from evidence_b200.rvmodel import RVModel
    case = synth.make_case(1, seed=4, n_epochs=96)
    model = RVModel(case.fixedpardict, case.datadict(pandas=True), case.parnames)
    settings = {"nlive": 100, "seed": 40, "sampler": "builtin", "builtin_method": "mlfriends-device",
                "builtin_wrap": True}
    rundict = {"target": "synth", "runid": "ml", "save_dir": str(tmp_path), "nplanets": 1}
    out = runner.run(model, dict(rundict), case.priordict, settings)
    assert "mlfriends-device" in out.sampler_impl and out.sampler_impl.endswith("wrapped: planet1_omega")
    assert np.isfinite(out.logZ) and out.nlike > 100
    outs = runner.run_ensemble(model, dict(rundict, runid="mle"), case.priordict, settings, nruns=2)
    assert len(outs) == 2 and len({o.logZ for o in outs}) == 2
    for o in outs:
        assert "MLFriends" in o.sampler_impl and np.isfinite(o.logZ)
    for fn in (runner.run, runner.run_ensemble):
        with pytest.raises(ValueError, match="adaptive_nsteps"):
            fn(model, dict(rundict, runid="bad"), case.priordict, dict(settings, builtin_adaptive_nsteps="move-distance"))
    model.close()
