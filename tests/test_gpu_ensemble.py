"""
The ensemble sampler on the GPU: `rvl_slice_phase_runs` against per-run `rvl_slice_phase` launches,
the set-up kernels against their host restatement (tests/_slice_runs_oracle.py), independence of the
runs, the evidence of a Gaussian, agreement with the single-run sampler on an RV case, and the runner.
"""
import ctypes
import math

import numpy as np
import pytest

import _slice_runs_oracle as ro
from test_gpu_slice_kernels import (DTYPE, PAD, PER_WALKER, SENTINEL, Device, _dims, fabricated,
                                    random_state, same_bits)
from test_gpu_slice_wrap import WrappedDevice

pytestmark = pytest.mark.gpu


class RunsDevice:
    """The walkers of several SliceStates in one launch, walker j of run r at row pos[r][j], phases
    through rvl_slice_phase_runs; PAD sentinel rows after the k walkers."""

    def __init__(self, sts, pos, wrap):
        import torch
        from evidence_b200 import _abi
        self.torch, self.lib, self.sts, self.pos = torch, _abi.load(), sts, pos
        st0 = sts[0]
        self.k = K = sum(s.k for s in sts)
        run_of, walker_of = np.empty(K, np.int32), np.empty(K, np.int32)
        for r, p in enumerate(pos):
            run_of[p], walker_of[p] = r, np.arange(len(p))
        self.buf = {}
        for name, shape in PER_WALKER.items():
            dt = DTYPE.get(name, np.float64)
            host = np.full((K + PAD,) + _dims(st0, shape), SENTINEL[dt], dt)
            for st, p in zip(sts, pos):
                host[p] = getattr(st, name)
            self.buf[name] = torch.from_numpy(host).cuda()
        cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
        self.run_of, self.walker_of = cuda(run_of), cuda(walker_of)
        self.seeds = cuda(np.array([s.seed for s in sts], np.uint64).view(np.int64))
        self.lmin = cuda(np.array([s.lmin for s in sts]))
        self.chol = cuda(np.stack([s.chol for s in sts]))
        self.stats = cuda(np.stack([s.stats for s in sts]).view(np.int64))
        a = self.args = _abi.rvl_slice_args()
        a.k, a.d, a.n_out, a.m = K, st0.d, st0.n_out, st0.m
        a.seed, a.lmin, a.chol, a.stats = 12345, 0, 0, 0  # ignored: the runs' own are used
        for name, t in self.buf.items():
            setattr(a, name, t.data_ptr())
        self.runs = _abi.rvl_slice_runs(n_runs=len(sts), run_of=self.run_of.data_ptr(),
                                        walker_of=self.walker_of.data_ptr(), seeds=self.seeds.data_ptr(),
                                        lmin=self.lmin.data_ptr(), chol=self.chol.data_ptr(),
                                        stats=self.stats.data_ptr())
        self.bits = None
        if wrap is not None:
            self.bits = (ctypes.c_uint32 * 4)()
            for j in np.flatnonzero(wrap):
                self.bits[j >> 5] |= 1 << (int(j) & 31)

    def set(self, r, name, values):
        self.buf[name][self.torch.from_numpy(self.pos[r]).cuda()] = self.torch.from_numpy(
            np.ascontiguousarray(values)).cuda()

    def phase(self, ph, move, shrink_round):
        self.args.move, self.args.shrink_round = move, shrink_round
        rc = self.lib.rvl_slice_phase_runs(ph, ctypes.byref(self.args), ctypes.byref(self.runs), self.bits,
                                           self.torch.cuda.current_stream().cuda_stream)
        assert rc == 0, self.lib.rvl_slice_last_error().decode()
        self.torch.cuda.synchronize()


@pytest.mark.parametrize("wrapped", [False, True])
@pytest.mark.parametrize("d", [15, 40])
def test_runs_kernels_match_per_run_launches(d, wrapped):
    """R = 5 runs (k_r = 1, 3, 7, 40, 13; seeds that differ in their low bits), walkers interleaved
    at random: every buffer after every phase 0, 1, 2, 2, 3 equals that of the same run launched alone
    through rvl_slice_phase (_wrapped), bit for bit, and so do the per-run counters."""
    ks = [1, 3, 7, 40, 13]
    seeds = [2 ** 40 + 2, 2 ** 40 + 3, 4, 5, 2 ** 64 - 1]
    n_out, m, move = 4, 6, 9
    rng = np.random.default_rng([d, wrapped])
    wrap = (rng.uniform(size=d) < 0.4) if wrapped else None
    if wrapped:
        wrap[0] = True
    sts, lls = [], []
    for r, (k, seed) in enumerate(zip(ks, seeds)):
        st = random_state(k, d, n_out, m, seed, move, rng)
        st.stats = np.array([r, 10 * r], np.uint64)
        made = fabricated(st, rng)
        # each run its own constraint: lmin and the made-up lnL values moved by 2 r
        st.lmin += 2.0 * r
        lls.append(lambda i, made=made, off=2.0 * r: {n: v if n == "cand_th" else v + off
                                                      for n, v in made(i).items()})
        sts.append(st)
    perm = rng.permutation(sum(ks))
    pos = np.split(perm, np.cumsum(ks)[:-1])
    alone = [WrappedDevice(st, wrap) if wrapped else Device(st) for st in sts]
    ens = RunsDevice(sts, pos, wrap)
    steps = [(0, 0), (1, 0), (2, 1), (2, 2), (3, 3)]
    for i, (ph, sr) in enumerate(steps):
        if i > 0:
            for r in range(len(sts)):
                for name, v in lls[r](i - 1).items():
                    alone[r].set(name, v)
                    ens.set(r, name, v)
        for dev in alone:
            dev.phase(ph, move, sr)
        ens.phase(ph, move, sr)
        got = {n: t.cpu().numpy() for n, t in ens.buf.items()}
        for r, dev in enumerate(alone):
            want = dev.read()
            for name in PER_WALKER:
                assert same_bits(got[name][pos[r]], want[name][:ks[r]]), (ph, sr, r, name)
            assert same_bits(ens.stats.cpu().numpy().view(np.uint64)[r], want["stats"][:2]), (ph, r)
        for name in PER_WALKER:
            assert np.all(got[name][ens.k:] == SENTINEL[got[name].dtype.type]), (ph, name, "past row k")


def _ensemble_buffers(seeds, nlive, d):
    import torch
    from evidence_b200.sampler_dev import _NativeSliceRuns
    return _NativeSliceRuns(torch, d, torch.device("cuda"), seeds, nlive, n_out=2, m=3, rounds=2)


def test_initial_points_and_starts_match_the_restatement():
    import torch
    from evidence_b200.sampler_dev import _walker_layout
    seeds, nlive, d = [0, 1, 2 ** 64 - 1, 77], 60, 7
    ns = _ensemble_buffers(seeds, nlive, d)
    u = ns.init().cpu().numpy()
    assert same_bits(u, ro.init_points(seeds, nlive, d))
    rng = np.random.default_rng(4)
    ns.u_live.copy_(torch.from_numpy(rng.uniform(size=(4, nlive, d))))
    th = torch.from_numpy(rng.normal(size=(4, nlive, d))).cuda()
    ll = torch.from_numpy(rng.normal(size=(4, nlive))).cuda()
    _, order = torch.sort(ll, dim=1, stable=True)
    kk = np.array([12, 1, 58, 30])
    run_of, walker_of = _walker_layout(kk)
    perm = rng.permutation(len(run_of))
    run_of, walker_of = run_of[perm], walker_of[perm]
    ns.reserve(len(run_of))
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    lmin = torch.zeros(4, dtype=torch.float64, device="cuda")
    ns.setup_round(th, ll, order, cuda(kk.astype(np.int64)), lmin, cuda(run_of), cuda(walker_of), 6)
    torch.cuda.synchronize()
    slots = ro.start_slots(seeds, nlive, order.cpu().numpy(), kk, run_of, walker_of, 6)
    assert np.array_equal(ns.start.cpu().numpy(), slots)
    u_host, th_host, l_host = ns.u_live.cpu().numpy(), th.cpu().numpy(), ll.cpu().numpy()
    assert same_bits(ns.u.cpu().numpy(), u_host[run_of, slots])
    assert same_bits(ns.theta.cpu().numpy(), th_host[run_of, slots])
    assert same_bits(ns.lstart.cpu().numpy(), l_host[run_of, slots])
    assert np.all(np.isnan(ns.lcur.cpu().numpy()))


@pytest.mark.parametrize("wrapped", [False, True])
def test_whitening_matches_the_restatement(wrapped):
    """Bit for bit without circular coordinates, within 1e-12 with them; the run whose survivors
    repeat a coordinate gets the diagonal; a run with kk = 0 (finished) keeps its factor."""
    import torch
    from evidence_b200.sampler_dev import _wrap_bits
    from test_ensemble_host import degenerate_points
    seeds, nlive, d = [3, 4, 5, 6], 40, 4
    ns = _ensemble_buffers(seeds, nlive, d)
    rng = np.random.default_rng(9)
    u = rng.uniform(0.3, 0.7, (4, nlive, d))
    u[0, :, 3] = ro._wrap_unit(u[0, :, 3] + 0.5)  # a mode across the seam in coordinate 3
    u[2] = degenerate_points(nlive, d)
    order = np.argsort(rng.uniform(size=(4, nlive)), axis=1, kind="stable")
    order[2] = np.arange(nlive)
    kk = np.array([8, 1, 8, 0])
    wrap = np.array([False, False, True, True]) if wrapped else None
    ns.wrap_bits = _wrap_bits(wrap)
    ns.u_live.copy_(torch.from_numpy(u))
    ns.chol[3] = 7.0
    run_of, walker_of = np.zeros(1, np.int32), np.zeros(1, np.int32)
    ns.reserve(1)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    th = torch.zeros((4, nlive, d), dtype=torch.float64, device="cuda")
    ns.setup_round(th, th[:, :, 0].contiguous(), cuda(order), cuda(kk), th[:, 0, 0].contiguous(),
                   cuda(run_of), cuda(walker_of), 0)
    got = ns.chol.cpu().numpy()
    assert np.all(got[3] == 7.0)
    want, failed = ro.whiten(u[:3], order[:3], kk[:3], wrap)
    assert failed.tolist() == [False, False, True]
    if wrapped:
        assert np.abs(got[:3] - want).max() <= 1e-12
    else:
        assert same_bits(got[:3], want)
    assert np.count_nonzero(got[2] - np.diag(np.diag(got[2]))) == 0


S_IND = 0.1


def gauss_columns(U):
    """lnL of a Gaussian (width 0.1 about 1/2, d = 4) written column by column: a row's value does
    not depend on the rest of the batch."""
    import torch
    ll = torch.zeros(U.shape[0], dtype=U.dtype, device=U.device)
    for c in range(U.shape[1]):
        ll = ll + (-0.5) * ((U[:, c] - 0.5) / S_IND) ** 2
    return U.clone(), ll


def gauss_plateau(U):
    """gauss_columns with lnL = -1e30 where u_0 < 0.3: a plateau that the first rounds retire."""
    import torch
    th, ll = gauss_columns(U)
    return th, torch.where(U[:, 0] < 0.3, torch.full_like(ll, -1e30), ll)


@pytest.mark.parametrize("fused", [gauss_columns, gauss_plateau])
def test_runs_do_not_interact(fused):
    """The run of seed 5 is the same in the ensembles [3, 4, 5, 6], [5] and [6, 5, 3]; the runs of
    an ensemble do not all end in the same round (so runs drop out while others go on)."""
    from evidence_b200.sampler_dev import nested_sample_ensemble
    kw = dict(nlive=100, nsteps=8, device="cuda")
    a = nested_sample_ensemble(fused, 4, [3, 4, 5, 6], **kw)
    b = nested_sample_ensemble(fused, 4, [5], **kw)
    c = nested_sample_ensemble(fused, 4, [6, 5, 3], **kw)
    for x in (b[0], c[1]):
        y = a[2]
        assert x.seed == y.seed == 5
        for f in ("samples", "weighted_samples", "logl"):
            assert same_bits(x[f], y[f]), f
        assert np.allclose(x.weights, y.weights, rtol=1e-11, atol=0)  # through ln Z: a batched sum
        assert (x.ncall, x.niter, x.accepted_moves, x.unresolved_moves) == (
            y.ncall, y.niter, y.accepted_moves, y.unresolved_moves)
        assert abs(x.logz - y.logz) <= 1e-12 and abs(x.logzerr - y.logzerr) <= 1e-9
    for r3, r6 in ((a[0], c[2]), (a[3], c[0])):
        assert same_bits(r3.weighted_samples, r6.weighted_samples) and r3.ncall == r6.ncall
    if fused is gauss_columns:  # every round retires k = 20 points: ncall = nlive + rounds 20 x 320
        rounds = [(r.ncall - 100) / (20 * 8 * (2 * 8 + 3 * 8)) for r in a]
        assert all(x == int(x) for x in rounds) and len(set(rounds)) > 1, rounds
    else:
        assert all(r.logl.min() == -1e30 for r in a)
        assert len({r.niter for r in a}) > 1 and len({r.ncall for r in a}) > 1


def test_analytic_evidence():
    """The Gaussian of test_native_slice_kernels_on_an_analytic_gaussian, R = 32: the mean ln Z within
    3 standard errors of the analytic value, the run-to-run scatter below 3 x the median reported
    uncertainty."""
    from evidence_b200.sampler_dev import nested_sample_ensemble
    ndim, sig = 4, 0.6

    def fused(U):
        th = -10 + 20 * U
        return th, -0.5 * ((th / sig) ** 2).sum(1)
    want = ndim * math.log(math.sqrt(2 * math.pi) * sig / 20)
    res = nested_sample_ensemble(fused, ndim, list(range(100, 132)), nlive=250, nsteps=10, device="cuda")
    z = np.array([r.logz for r in res])
    err = np.median([r.logzerr for r in res])
    assert abs(z.mean() - want) < 3 * z.std(ddof=1) / math.sqrt(len(z)), (z.mean(), want, z.std(ddof=1))
    assert z.std(ddof=1) < 3 * err, (z.std(ddof=1), err)
    assert all(r.unresolved_moves < 0.01 * r.accepted_moves for r in res)
    print(f"R = 32: mean {z.mean():.4f} (analytic {want:.4f}), std {z.std(ddof=1):.4f}, median logzerr {err:.4f}")


def test_same_sampler_as_the_single_run_one_on_the_rv_model():
    """Seeds 0-15 as an ensemble and as 16 nested_sample_device runs (different streams): the means of
    ln Z agree within 3 combined standard errors, every run finds the period within 2 %, and the
    model counted exactly the evaluations the ensemble reports.  16 runs a side, not 8: the run-to-run
    scatter of ln Z on this posterior is 1-2 and heavy-tailed, and with 8 the standard error itself is
    too uncertain for a 3-sigma bound (profiles/r6_ensemble.txt, section 2)."""
    from evidence_b200 import synth
    from evidence_b200.rvmodel import RVModel
    from evidence_b200.sampler_dev import nested_sample_device, nested_sample_ensemble
    case = synth.make_case(1, seed=4, n_epochs=96)
    model = RVModel(case.fixedpardict, case.datadict(), case.parnames)
    model.set_priors(case.priordict)
    fused = model.transform_loglike_device
    model.reset_counters()
    n = 16
    ens = nested_sample_ensemble(fused, case.ndim, list(range(n)), nlive=200, device="cuda")
    assert model.counters()["n_points"] == sum(r.ncall for r in ens)
    one = [nested_sample_device(fused, case.ndim, nlive=200, seed=s, device="cuda") for s in range(n)]
    za, zb = np.array([r.logz for r in ens]), np.array([r.logz for r in one])
    se = math.sqrt(za.var(ddof=1) / n + zb.var(ddof=1) / n)
    assert abs(za.mean() - zb.mean()) < 3 * se, (za.mean(), zb.mean(), se)
    col = case.parnames.index("planet1_period")
    for r in ens:
        per = np.median(r.samples[:, col])
        assert abs(per - case.truth["planet1_period"]) / case.truth["planet1_period"] < 0.02, (r.seed, per)
    print(f"ensemble {za.mean():.3f} +- {za.std(ddof=1):.3f}, single {zb.mean():.3f} +- {zb.std(ddof=1):.3f}")
    model.close()


def test_runner(tmp_path):
    """run_ensemble with R = 3 writes three pickles (runids {runid}_0..2) with the attributes run()
    sets and three weighted_post.txt files."""
    import os
    import pickle
    from evidence_b200 import synth
    from evidence_b200 import ultranest as runner
    from evidence_b200.rvmodel import RVModel
    case = synth.make_case(1, seed=4, n_epochs=96)
    model = RVModel(case.fixedpardict, case.datadict(pandas=True), case.parnames)
    outs = runner.run_ensemble(model, {"target": "synth", "runid": "ens", "save_dir": str(tmp_path), "nplanets": 1},
                               case.priordict, {"nlive": 100, "nsteps": 8, "seed": 40}, nruns=3)
    assert len(outs) == 3 and len({o.file_root for o in outs}) == 3
    attrs = {"runtime", "walltime", "rundict", "datadict", "fixedpardict", "model_name", "nlive", "nrepeats",
             "isodate", "ncores", "parnames", "ndim", "sampler", "sampler_impl", "base_dir", "file_root",
             "logZ", "logZerr", "nlike", "samples", "device_counters", "evals_per_second"}
    for i, o in enumerate(outs):
        assert o.file_root.startswith(f"synth_ens_{i}_k1_")
        assert o.rundict["runid"] == f"ens_{i}" and f"run {i} of 3, seed {40 + i}" in o.sampler_impl
        assert attrs <= set(vars(o)), attrs - set(vars(o))
        with open(os.path.join(os.path.dirname(o.base_dir), o.file_root + ".pkl"), "rb") as f:
            p = pickle.load(f)
        assert p.logZ == o.logZ and p.file_root == o.file_root
        post = np.loadtxt(os.path.join(o.base_dir, "run1", "chains", "weighted_post.txt"), skiprows=1)
        assert post.shape[1] == 2 + case.ndim and abs(post[:, 0].sum() - 1.0) < 1e-9
        assert np.isfinite(o.logZ) and o.nlike > 0
    assert len({o.logZ for o in outs}) == 3
    total = sum(o.nlike for o in outs)  # the rate is the ensemble's: all runs' evaluations, one wall time
    assert all(abs(o.evals_per_second * o.walltime - total) <= 1e-6 * total for o in outs)
    model.close()
