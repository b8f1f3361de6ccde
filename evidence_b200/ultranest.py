"""
Vectorised UltraNest runner on the device likelihood.

Same entry point as the reference runner -- ``run(model, rundict, priordict, ultrasettings)``
(evidence/ultranest/__init__.py:32-259) -- with the same defaults (:333-338), file-root naming
(:347-375), wrapped-parameter rule (:159-162) and ``Output`` attribute set (:200-229), so
post-processing and pickles stay compatible.  What changes is the hot loop: the ``prior`` and
``loglike`` callbacks are the BATCHED device transform / likelihood
(``vectorized=True``, which the reference has commented out at :171), fed with ``ndraw_min`` ..
``ndraw_max`` points per call.

Extra ``ultrasettings`` keys (the "config switch"):
    'vectorized' (True), 'ndraw_min' (4096), 'ndraw_max' (65536), 'seed' (None),
    'stepsampler' ('region-slice' like the reference | 'population-slice' | 'none'),
    'sampler' ('auto' | 'ultranest' | 'builtin'),
    'builtin_method' ('slice' | 'slice-device' | 'ellipsoid' | 'mlfriends-device': MLFriends region
    sampling on the device, ``sampler_dev.nested_sample_ensemble(method='mlfriends')``, run as an
    ensemble of one seed, at most 'ndraw_max' candidates per batch),
    'builtin_wrap' (False: the built-in slice samplers and 'mlfriends-device' take the wrapped
    parameters -- the ones UltraNest gets as ``wrapped_params`` -- as circular coordinates; 'ellipsoid'
    rejects it),
    'builtin_adaptive_nsteps' (False | 'move-distance': the device sampler adapts each run's number of
    moves per round, ``sampler_dev.nested_sample_device(adaptive_nsteps=...)``; 'slice-device' and
    ``run_ensemble`` only, 'slice' and 'ellipsoid' reject it),
    'postprocess' (False), 'plot' (False)

``run_ensemble`` runs several seeded runs of the built-in device sampler ('mlfriends-device' or, for
any other 'builtin_method', the slice sampler) through shared launches and writes each as ``run()``
would (one run directory, pickle and ``weighted_post.txt`` per run).

UltraNest is a third-party package that is not part of the reference repository (SURVEY.md 8c).
When it is importable it is used; otherwise -- or with ``'sampler': 'builtin'`` -- the seeded
vectorised nested sampler of ``evidence_b200.sampler`` produces ln Z from the same callbacks.
"""
import datetime
import os
import pickle
import time
from pathlib import Path

import numpy as np

try:  # MPI is optional, as in the reference (:21-29)
    from mpi4py import MPI
    comm = MPI.COMM_WORLD
    rank, size = comm.Get_rank(), comm.Get_size()
except ImportError:
    comm, rank, size = None, 0, 1


class Output:
    """Attribute bag of a run, pickled as such (evidence/ultranest/__init__.py:200-229, 262-297):
    the reference's post-processing un-pickles it and reads attributes (``output.file_root``,
    ``output.rundict``, ``output.datadict``, ... -- evidence/post_processing.py:34-89)."""


def _torch_device(model):
    import torch
    idx = getattr(model, "device_index", None)
    return torch.device("cuda", torch.cuda.current_device() if idx is None else idx)


def make_callbacks(model, priordict):
    """(prior, loglike) in UltraNest's vectorised convention, both one device launch per call."""
    if hasattr(model, "set_priors"):
        model.set_priors(priordict)

        def prior(cube):
            return model.prior_transform_batch(np.atleast_2d(cube))

        def loglike(theta):
            return model.log_likelihood_batch(np.atleast_2d(theta))
    else:  # any object with the reference's scalar protocol (:125-146)
        parnames = model.parnames

        def prior(cube):
            cube = np.atleast_2d(cube)
            out = np.empty_like(cube)
            for i, p in enumerate(parnames):
                out[:, i] = priordict[p].ppf(cube[:, i])
            return out

        def loglike(theta):
            return np.array([model.log_likelihood(row) for row in np.atleast_2d(theta)])
    return prior, loglike


def run(model, rundict, priordict, ultrasettings=None):
    """
    Run nested sampling on ``model`` (an ``evidence_b200.rvmodel.RVModel`` or any object with the
    reference's model protocol) and return the ``Output`` object (the reference returns None and
    only pickles it; the pickle is written here too).
    """
    parnames = model.parnames
    ndim = len(parnames)
    nderived = 0
    isodate = datetime.datetime.today().isoformat()
    if size > 1:
        isodate = comm.bcast(isodate, root=0)
    settings = set_ultrasettings(rundict, ultrasettings, ndim, nderived, isodate, parnames)

    # circular parameters, evidence/ultranest/__init__.py:159-162
    wrapped = np.array([("omega" in p) or ("ml0" in p) for p in parnames], dtype=bool)
    prior, loglike = make_callbacks(model, priordict)

    which = settings["sampler"]
    if which == "auto":
        try:
            import ultranest  # noqa: F401
            which = "ultranest"
        except ImportError:
            which = "builtin"

    ti = time.process_time()
    t_wall = time.perf_counter()
    if which == "ultranest":
        import ultranest
        import ultranest.stepsampler
        sampler = ultranest.ReactiveNestedSampler(
            parnames, loglike, prior, log_dir=settings["log_dir"], num_test_samples=100,
            wrapped_params=wrapped, num_bootstraps=settings["num_bootstraps"],
            vectorized=settings["vectorized"], ndraw_min=settings["ndraw_min"],
            ndraw_max=settings["ndraw_max"])
        if settings["stepsampler"] == "region-slice":  # the reference's choice (:175)
            sampler.stepsampler = ultranest.stepsampler.RegionSliceSampler(
                nsteps=settings["nsteps"], adaptive_nsteps="move-distance")
        elif settings["stepsampler"] == "population-slice":
            import ultranest.popstepsampler as pop
            sampler.stepsampler = pop.PopulationSliceSampler(
                popsize=settings["ndraw_min"], nsteps=settings["nsteps"],
                generate_direction=pop.generate_region_oriented_direction)
        sampler.run(min_num_live_points=settings["nlive"],
                    cluster_num_live_points=int(0.1 * settings["nlive"]),
                    dlogz=settings["dlogz"], frac_remain=settings["frac_remain"])
        sampler.print_results()
        res = sampler.results
        logz, logzerr, ncall, samples = res["logz"], res["logzerr"], res["ncall"], res["samples"]
        name = "UltraNest"
        impl = f"ultranest {getattr(ultranest, '__version__', '?')}, vectorized={settings['vectorized']}, " \
               f"stepsampler={settings['stepsampler']}"
        if settings["plot"]:
            sampler.plot()
    else:
        from .sampler import nested_sample
        os.makedirs(settings["log_dir"], exist_ok=True)
        # the device model evaluates u -> theta -> lnL in one call (rvl_transform_loglike)
        fused = getattr(model, "transform_loglike_batch", None) if hasattr(model, "set_priors") else None
        # the circular parameters UltraNest gets, only when asked for
        builtin_wrapped = wrapped if settings["builtin_wrap"] else None
        adaptive = _adaptive_setting(settings)
        if adaptive is not None and settings["builtin_method"] != "slice-device":
            raise ValueError(f"'builtin_adaptive_nsteps': {adaptive!r} needs 'builtin_method': 'slice-device', "
                             f"not {settings['builtin_method']!r}")
        if settings["builtin_method"] == "mlfriends-device":
            # MLFriends region sampling on the likelihood's device: an ensemble of one seed
            from .sampler_dev import nested_sample_ensemble
            if not hasattr(model, "transform_loglike_device"):
                raise ValueError("'builtin_method': 'mlfriends-device' needs the device model")
            res = nested_sample_ensemble(model.transform_loglike_device, ndim,
                                         [0 if settings["seed"] is None else settings["seed"]],
                                         nlive=settings["nlive"], dlogz=settings["dlogz"],
                                         frac_remain=settings["frac_remain"], wrapped=builtin_wrapped,
                                         device=_torch_device(model), num_bootstraps=settings["num_bootstraps"],
                                         method="mlfriends", ndraw_max=settings["ndraw_max"])[0]
        elif settings["builtin_method"] == "slice-device":
            # the whole run on the likelihood's device (evidence_b200.sampler_dev)
            from .sampler_dev import nested_sample_device
            if not hasattr(model, "transform_loglike_device"):
                raise ValueError("'builtin_method': 'slice-device' needs the device model")
            res = nested_sample_device(model.transform_loglike_device, ndim,
                                       nlive=settings["nlive"], dlogz=settings["dlogz"],
                                       frac_remain=settings["frac_remain"], nsteps=settings["nsteps"],
                                       seed=0 if settings["seed"] is None else settings["seed"],
                                       device=_torch_device(model), wrapped=builtin_wrapped,
                                       adaptive_nsteps=adaptive)
        else:
            res = nested_sample(loglike, prior, ndim, nlive=settings["nlive"], fused=fused,
                                ndraw=settings["ndraw_min"], dlogz=settings["dlogz"],
                                frac_remain=settings["frac_remain"], nsteps=settings["nsteps"],
                                method=settings["builtin_method"], wrapped=builtin_wrapped,
                                seed=0 if settings["seed"] is None else settings["seed"])
        logz, logzerr, ncall, samples = res.logz, res.logzerr, res.ncall, res.samples
        # the reference's post-processing knows 'PolyChord' and 'UltraNest' only and, for the latter,
        # reads run1/chains/weighted_post.txt (evidence/post_processing.py:66-88): same label, same
        # file, and the implementation named beside it
        name = "UltraNest"
        impl = f"evidence_b200.sampler ({settings['builtin_method']}); ultranest not used"
        if settings["builtin_method"] == "mlfriends-device":
            impl = (f"evidence_b200.sampler_dev (mlfriends-device: MLFriends region sampling, "
                    f"{settings['num_bootstraps']} bootstraps); ultranest not used")
        if builtin_wrapped is not None:
            impl += "; wrapped: " + (", ".join(p for p, w in zip(parnames, wrapped) if w) or "none")
        if adaptive is not None:
            impl += _nsteps_note(adaptive, res.nsteps_history)
        write_weighted_post(settings["log_dir"], parnames, res)
    tf = time.process_time()
    t_wall = time.perf_counter() - t_wall
    if size > 1:
        ti = comm.reduce(ti, op=MPI.MIN, root=0)
        tf = comm.reduce(tf, op=MPI.MAX, root=0)

    history = res.nsteps_history if which != "ultranest" else None
    return _output(model, rundict, settings, isodate, parnames, name, impl, logz, logzerr, ncall, samples,
                   ti, tf, t_wall, nsteps_history=history)


def _output(model, rundict, settings, isodate, parnames, name, impl, logz, logzerr, ncall, samples,
            ti, tf, t_wall, evals=None, nsteps_history=None):
    """The ``Output`` of a run (rank 0; None elsewhere), pickled as ``<file_root>.pkl``: process time
    tf - ti, wall time t_wall; ``evals``: the lnL evaluations those times cover (default: ncall);
    ``nsteps_history``: the moves per round of an adaptive run (set as an attribute when given)."""
    ndim = len(parnames)
    output = None
    if rank == 0:
        import pandas as pd
        output = Output()
        output.runtime = datetime.timedelta(seconds=tf - ti)
        output.walltime = t_wall
        output.rundict = rundict.copy()
        output.datadict = dict(getattr(model, "datadict", {}))  # host tables (frames / arrays) only
        output.fixedpardict = dict(getattr(model, "fixedpardict", {}))
        model_path = getattr(model, "model_path", None)
        output.model_name = str(Path(model_path).stem) if model_path else type(model).__name__
        output.nlive = settings["nlive"]
        output.nrepeats = settings["nsteps"]
        output.isodate = isodate
        output.ncores = size
        output.parnames = parnames
        output.ndim = ndim
        output.sampler = name
        output.sampler_impl = impl
        output.base_dir = settings["log_dir"]
        output.file_root = settings["file_root"]
        output.logZ = float(logz)
        output.logZerr = float(logzerr)
        output.nlike = int(ncall)
        output.samples = pd.DataFrame(np.asarray(samples), columns=parnames)
        if nsteps_history is not None:
            output.nsteps_history = list(nsteps_history)
        if hasattr(model, "counters"):  # observability added by the device path
            output.device_counters = model.counters()
            output.evals_per_second = (output.nlike if evals is None else evals) / max(t_wall, 1e-9)
        if "prior_names" in rundict:
            output.priors = rundict["prior_names"]
        if "star_params" in rundict:
            output.starparams = rundict["star_params"]
        print(f"\nTotal run time was: {output.runtime}")
        dump2pickle(output, output.file_root + ".pkl")
        if settings["postprocess"]:
            from evidence.post_processing import postprocess  # the reference's own (unchanged)
            postprocess(str(Path(output.base_dir).parent.absolute()))
    return output


def run_ensemble(model, rundict, priordict, ultrasettings=None, nruns=4, seeds=None):
    """
    ``nruns`` independent runs of the built-in device sampler on ``model`` (the device model, as for
    ``'builtin_method': 'slice-device'``), advanced together through shared launches
    (``sampler_dev.nested_sample_ensemble``).  Returns a list of ``Output``: output i is what ``run()``
    writes for ``rundict['runid'] = f"{runid}_{i}"`` and seed ``seeds[i]`` -- its own pickle, file
    root and ``run1/chains/weighted_post.txt`` -- so that the reference's post-processing and
    ``fip_criterion`` (median ln Z over run directories, evidence/fip_criterion.py:245-266) scan
    them as separately launched runs.  ``seeds`` (default: seed, seed + 1, .. from the settings'
    'seed', 0 when None) sets nruns.  Every output's runtime, walltime, ``device_counters`` and
    ``evals_per_second`` (all runs' evaluations over the wall time) are those of the whole ensemble,
    which is what the GPU did; ``nlike`` is the run's own count.  Settings as for ``run()``;
    'builtin_method': 'mlfriends-device' runs MLFriends region sampling
    (``nested_sample_ensemble(method='mlfriends')``), any other value the slice sampler;
    'builtin_wrap' and 'builtin_adaptive_nsteps' are honoured, and 'postprocess' runs the reference's
    post-processing on each run's own directory (``<save_dir>/<file_root>``), as ``run()`` does.
    """
    from .sampler_dev import nested_sample_ensemble
    if not hasattr(model, "transform_loglike_device"):
        raise ValueError("run_ensemble needs the device model (transform_loglike_device)")
    parnames = model.parnames
    ndim = len(parnames)
    isodate = datetime.datetime.today().isoformat()
    if size > 1:
        isodate = comm.bcast(isodate, root=0)
    base = set_ultrasettings(dict(rundict), ultrasettings, ndim, 0, isodate, parnames)
    if seeds is None:
        seed0 = 0 if base["seed"] is None else int(base["seed"])
        seeds = [seed0 + i for i in range(int(nruns))]
    seeds = [int(s) for s in seeds]
    wrapped = np.array([("omega" in p) or ("ml0" in p) for p in parnames], dtype=bool)
    builtin_wrapped = wrapped if base["builtin_wrap"] else None
    adaptive = _adaptive_setting(base)
    mlfriends = base["builtin_method"] == "mlfriends-device"
    if adaptive is not None and mlfriends:
        raise ValueError(f"'builtin_adaptive_nsteps': {adaptive!r} needs the slice sampler, not "
                         "'builtin_method': 'mlfriends-device'")
    region = dict(method="mlfriends", ndraw_max=base["ndraw_max"]) if mlfriends else {}
    model.set_priors(priordict)
    ti = time.process_time()
    t_wall = time.perf_counter()
    results = nested_sample_ensemble(model.transform_loglike_device, ndim, seeds, nlive=base["nlive"],
                                     dlogz=base["dlogz"], frac_remain=base["frac_remain"],
                                     nsteps=base["nsteps"], wrapped=builtin_wrapped,
                                     device=_torch_device(model), num_bootstraps=base["num_bootstraps"],
                                     adaptive_nsteps=adaptive, **region)
    tf = time.process_time()
    t_wall = time.perf_counter() - t_wall
    if size > 1:
        ti = comm.reduce(ti, op=MPI.MIN, root=0)
        tf = comm.reduce(tf, op=MPI.MAX, root=0)
    runid = rundict["runid"].replace(" ", "")
    outputs = []
    for i, (seed, res) in enumerate(zip(seeds, results)):
        rd = dict(rundict, runid=f"{runid}_{i}")
        settings = set_ultrasettings(rd, ultrasettings, ndim, 0, isodate, parnames)
        os.makedirs(settings["log_dir"], exist_ok=True)
        write_weighted_post(settings["log_dir"], parnames, res)
        kind = "mlfriends-device: MLFriends region sampling" if mlfriends else "slice-device"
        impl = (f"evidence_b200.sampler_dev ensemble ({kind}): run {i} of {len(seeds)}, seed {seed}; "
                "ultranest not used")
        if builtin_wrapped is not None:
            impl += "; wrapped: " + (", ".join(p for p, w in zip(parnames, wrapped) if w) or "none")
        if adaptive is not None:
            impl += _nsteps_note(adaptive, res.nsteps_history)
        outputs.append(_output(model, rd, settings, isodate, parnames, "UltraNest", impl, res.logz,
                               res.logzerr, res.ncall, res.samples, ti, tf, t_wall,
                               evals=sum(r.ncall for r in results), nsteps_history=res.nsteps_history))
    return outputs


def _adaptive_setting(settings):
    """The samplers' ``adaptive_nsteps`` for the setting 'builtin_adaptive_nsteps': None when it is
    False or None, 'move-distance' as is; anything else is a ValueError."""
    value = settings["builtin_adaptive_nsteps"]
    if value is False or value is None:
        return None
    if value != "move-distance":
        raise ValueError(f"'builtin_adaptive_nsteps': {value!r}; False or 'move-distance'")
    return value


def _nsteps_note(adaptive, history):
    """The implementation string's note on the adapted number of moves per round."""
    h = np.asarray(history)
    return (f"; adaptive nsteps ({adaptive}): moves per round min {h.min()}, median {np.median(h):g}, "
            f"max {h.max()} over {len(h)} rounds")


def write_weighted_post(log_dir, parnames, res):
    """``<log_dir>/run1/chains/weighted_post.txt`` in UltraNest's layout (``weight logl <params>``,
    space separated), which the reference's post-processing reads for the log-likelihoods and
    weights of the posterior (evidence/post_processing.py:85-88)."""
    pts, w, logl = res.get("weighted_samples"), res.get("weights"), res.get("logl")
    if pts is None or w is None or logl is None:
        return None
    chains = os.path.join(log_dir, "run1", "chains")
    os.makedirs(chains, exist_ok=True)
    path = os.path.join(chains, "weighted_post.txt")
    np.savetxt(path, np.column_stack([np.asarray(w), np.asarray(logl), np.asarray(pts)]),
               header=" ".join(["weight", "logl"] + list(parnames)), comments="")
    return path


def dump2pickle(output, filename, savedir=None):
    """Pickle the ``Output`` OBJECT next to the run directory, like
    evidence/ultranest/__init__.py:262-297 (``datadict`` included: post-processing reads it)."""
    pickledir = Path(output.base_dir).parent if savedir is None else savedir
    os.makedirs(pickledir, exist_ok=True)
    with open(os.path.join(pickledir, filename), "wb") as f:
        pickle.dump(output, f)


def set_ultrasettings(rundict, ultrasettings, ndim, nderived, isodate, parnames):
    """Defaults + user settings + file-root naming, evidence/ultranest/__init__.py:300-388."""
    settings = {"nlive": 25 * ndim, "nsteps": 3 * ndim, "dlogz": 0.5, "frac_remain": 0.01,
                "num_bootstraps": 30,
                # the device-path switch
                "vectorized": True, "ndraw_min": 4096, "ndraw_max": 65536, "seed": None,
                "stepsampler": "region-slice", "sampler": "auto", "builtin_method": "slice",
                "builtin_wrap": False, "builtin_adaptive_nsteps": False,
                "postprocess": False, "plot": False}
    if ultrasettings is not None:
        if type(ultrasettings) is not dict:
            raise TypeError("ultrasettings has to be a dictionary")
        settings.update(ultrasettings)

    rundict["target"] = rundict["target"].replace(" ", "")
    rundict["runid"] = rundict["runid"].replace(" ", "")
    file_root = rundict["target"] + "_" + rundict["runid"]
    if rundict.get("comment", "") != "":
        file_root += "-" + rundict["comment"]
    if rundict.get("nplanets") is not None:
        file_root += f'_k{rundict["nplanets"]}'
    drift_order = sum(1 for p in parnames
                      if "drift" in p and p[6:] in ("lin", "quad", "cub", "quar"))
    if drift_order > 0:
        file_root += f"_d{drift_order}"
    file_root += f'_nlive{settings["nlive"]}_ncores{size}_ultranest_{isodate}'
    base_dir = os.path.join(rundict.get("save_dir", ""), file_root, "ultraresults")
    settings.update({"log_dir": base_dir, "file_root": file_root})
    return settings
