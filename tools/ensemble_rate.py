"""Ensembles of nested-sampling runs (sampler_dev.nested_sample_ensemble) against the same runs one
after another (nested_sample_device), measured:
  1. wall time of R = 1, 4, 16, 64 runs (seeds 0 .. R-1) as one ensemble and as R sequential runs,
     the two alternated, twice (the 64 sequential runs once), on two workloads: the RV case of profiles/r2_lnz_scatter.txt
     (make_case(1, seed=4, n_epochs=96), nlive = 200, nsteps = 21) and the config-2 model of
     profiles/r2_sampler_rate.txt (make_case(2, seed=11, n_epochs=300), nlive = 200, nsteps = 12);
  2. on the RV case at R = 32, without and with the reference's wrap mask (omega, ml0): mean and
     standard deviation of ln Z across runs next to the median reported logzerr; and seeds 0-15 as
     an ensemble against 16 single runs (the comparison of tests/test_gpu_ensemble.py);
  3. the same for the d = 4 Gaussian of tests/test_gpu_ensemble.py::test_analytic_evidence.
usage: python tools/ensemble_rate.py [output file]"""
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from evidence_b200 import synth  # noqa: E402
from evidence_b200.rvmodel import RVModel  # noqa: E402
from evidence_b200.sampler_dev import nested_sample_device, nested_sample_ensemble  # noqa: E402

OUT = open(sys.argv[1], "w") if len(sys.argv) > 1 else None  # written line by line


def out(s=""):
    print(s, flush=True)
    if OUT:
        OUT.write(s + "\n")
        OUT.flush()


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return f"{name}, power limit / max SM clock: {q.stdout.strip()}"
    except (OSError, subprocess.SubprocessError):
        return f"{name}, power limit not readable"


def model_of(n_planets, seed, n_epochs):
    case = synth.make_case(n_planets, seed=seed, n_epochs=n_epochs)
    model = RVModel(case.fixedpardict, case.datadict(), case.parnames)
    model.set_priors(case.priordict)
    return case, model


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, res


out(f"# {card()}")
out(f"# torch {torch.__version__}, {time.strftime('%Y-%m-%d %H:%M:%S')}")
out("# command: python tools/ensemble_rate.py profiles/r6_ensemble.txt")
workloads = {"rv (1 planet, 96 epochs, nsteps 21)": (model_of(1, 4, 96), 21),
             "config 2 (2 planets, 300 epochs, nsteps 12)": (model_of(2, 11, 300), 12)}
out("\n## 1. wall time: ensemble vs sequential runs, nlive = 200, seeds 0 .. R-1")
out(f"{'workload':44s} {'R':>3s} {'mode':10s} {'rep':>3s} {'wall s':>8s} {'s/run':>7s} {'ncall':>11s} {'M lnL/s':>8s}")
for wname, ((case, model), nsteps) in workloads.items():
    fused = model.transform_loglike_device
    nested_sample_ensemble(fused, case.ndim, [0, 1], nlive=200, nsteps=nsteps)  # warm-up (modules, allocator)
    nested_sample_device(fused, case.ndim, nlive=200, seed=0, nsteps=nsteps)
    for R in (1, 4, 16, 64):
        best = {}
        for rep in range(2):
            for mode in ("ensemble", "sequential"):
                if mode == "sequential" and R == 64 and rep == 1:
                    continue  # 64 runs one after another take minutes: timed once
                if mode == "ensemble":
                    dt, res = timed(lambda: nested_sample_ensemble(fused, case.ndim, list(range(R)), nlive=200,
                                                                   nsteps=nsteps))
                else:
                    dt, res = timed(lambda: [nested_sample_device(fused, case.ndim, nlive=200, seed=s, nsteps=nsteps)
                                             for s in range(R)])
                nc = sum(r.ncall for r in res)
                best[mode] = min(best.get(mode, math.inf), dt)
                out(f"{wname:44s} {R:3d} {mode:10s} {rep:3d} {dt:8.2f} {dt / R:7.3f} {nc:11d} {nc / dt / 1e6:8.2f}")
        out(f"{wname:44s} {R:3d} speed-up of the ensemble (best of 2 each): {best['sequential'] / best['ensemble']:.2f}x")
    model.close()

out("\n## 2. run-to-run scatter of ln Z, RV case, R = 32 (seeds 0-31), nlive = 200, nsteps = 21")
case, model = model_of(1, 4, 96)
wrap = np.array([("omega" in p) or ("ml0" in p) for p in case.parnames])
for tag, w in (("no mask", None), ("omega/ml0 wrapped", wrap)):
    dt, res = timed(lambda: nested_sample_ensemble(model.transform_loglike_device, case.ndim, list(range(32)),
                                                   nlive=200, nsteps=21, wrapped=w))
    z = np.array([r.logz for r in res])
    e = np.median([r.logzerr for r in res])
    out(f"{tag:20s} mean lnZ {z.mean():9.3f}  std {z.std(ddof=1):6.3f}  median logzerr {e:6.3f}  "
        f"std / logzerr {z.std(ddof=1) / e:5.2f}  median {np.median(z):9.3f}  ({dt:.1f} s)")
out("\nensemble against single runs (nested_sample_device, other random streams), the same seeds:")
ens = nested_sample_ensemble(model.transform_loglike_device, case.ndim, list(range(16)), nlive=200, nsteps=21)
one = [nested_sample_device(model.transform_loglike_device, case.ndim, nlive=200, seed=s, nsteps=21)
       for s in range(16)]
for n in (8, 16):
    za, zb = np.array([r.logz for r in ens[:n]]), np.array([r.logz for r in one[:n]])
    se = math.sqrt(za.var(ddof=1) / n + zb.var(ddof=1) / n)
    out(f"seeds 0-{n - 1:<2d} ensemble mean {za.mean():9.3f} (std {za.std(ddof=1):5.3f})  single mean "
        f"{zb.mean():9.3f} (std {zb.std(ddof=1):5.3f})  difference / combined standard error "
        f"{(za.mean() - zb.mean()) / se:5.2f}")
out("single runs, seeds 0-15: " + " ".join(f"{r.logz:.2f}" for r in one))
out("ensemble,    seeds 0-15: " + " ".join(f"{r.logz:.2f}" for r in ens))
model.close()

out("\n## 3. the d = 4 Gaussian of test_analytic_evidence (nlive = 250, nsteps = 10), R = 32 (seeds 100-131)")


def gauss(U):
    th = -10 + 20 * U
    return th, -0.5 * ((th / 0.6) ** 2).sum(1)


want = 4 * math.log(math.sqrt(2 * math.pi) * 0.6 / 20)
res = nested_sample_ensemble(gauss, 4, list(range(100, 132)), nlive=250, nsteps=10)
z = np.array([r.logz for r in res])
e = np.median([r.logzerr for r in res])
out(f"analytic {want:.4f}  mean {z.mean():.4f}  (mean - analytic) / standard error "
    f"{(z.mean() - want) / (z.std(ddof=1) / math.sqrt(32)):.2f}  std {z.std(ddof=1):.4f}  median logzerr {e:.4f}  "
    f"std / logzerr {z.std(ddof=1) / e:.2f}")
