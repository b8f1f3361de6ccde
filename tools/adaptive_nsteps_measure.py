"""The adaptive number of moves (adaptive_nsteps='move-distance') of the device samplers, measured:
  1. the RV case of profiles/r2_lnz_scatter.txt (make_case(1, seed=4, n_epochs=96), nlive = 200), R = 32
     (seeds 0-31), one ensemble each: fixed nsteps 21, 42, 84; adaptive from 21 with cap 84; the same
     with the reference's wrap mask (omega, ml0).  Mean, std and median of ln Z, mean and median
     reported logzerr, std / median logzerr, lnL calls per run, wall time, median and maximum moves
     per round, unresolved moves;
  2. the same rows for the config-2 model of profiles/r6_ensemble.txt (make_case(2, seed=11,
     n_epochs=300), nlive = 200), fixed 3 ndim against adaptive from 3 ndim, and for the d = 4 Gaussian
     of tests/test_gpu_ensemble.py::test_analytic_evidence (nlive 250, nsteps 10), with its analytic ln Z;
  3. kernel time of rvl_slice_runs_radius + _travel per round (CUDA events over 50 rounds after 5
     warm-up rounds, random points) at nlive 200, d 7, R 1/32/64 and nlive 650, d 26, R 1/16, kk = 0.2
     nlive per run, next to the measured time per round of section 1 where a workload has that shape.
usage: python tools/adaptive_nsteps_measure.py [output file]"""
import ctypes
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from evidence_b200 import _abi, synth  # noqa: E402
from evidence_b200.rvmodel import RVModel  # noqa: E402
from evidence_b200.sampler_dev import nested_sample_ensemble  # noqa: E402

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


HEAD = (f"{'configuration':34s} {'mean lnZ':>9s} {'std':>6s} {'median':>9s} {'err mean':>8s} {'err med':>7s} "
        f"{'std/err':>7s} {'calls/run':>10s} {'wall s':>7s} {'n med':>5s} {'n max':>5s} {'unres/acc':>9s}")


def row(tag, dt, res, want=None):
    z = np.array([r.logz for r in res])
    e = np.array([r.logzerr for r in res])
    hist = np.concatenate([r.nsteps_history for r in res]) if res[0].nsteps_history is not None else None
    nmed = f"{np.median(hist):5.0f}" if hist is not None else f"{'-':>5s}"
    nmax = f"{hist.max():5d}" if hist is not None else f"{'-':>5s}"
    unres = sum(r.unresolved_moves for r in res) / max(1, sum(r.accepted_moves for r in res))
    out(f"{tag:34s} {z.mean():9.3f} {z.std(ddof=1):6.3f} {np.median(z):9.3f} {e.mean():8.3f} {np.median(e):7.3f} "
        f"{z.std(ddof=1) / np.median(e):7.2f} {np.mean([r.ncall for r in res]):10.0f} {dt:7.1f} {nmed} {nmax} "
        f"{unres:9.2e}")
    if want is not None:
        out(f"{'':34s} analytic {want:.4f}: (mean - analytic) / standard error "
            f"{(z.mean() - want) / (z.std(ddof=1) / math.sqrt(len(z))):.2f}")
    rounds = max(len(r.nsteps_history) for r in res) if hist is not None else None
    return dt / rounds if rounds else None


out(f"# {card()}")
out(f"# torch {torch.__version__}, {time.strftime('%Y-%m-%d %H:%M:%S')}")
out("# command: python tools/adaptive_nsteps_measure.py profiles/r7_adaptive_nsteps.txt")
out("# n med / n max: median and maximum over all runs and rounds of the moves per walker (adaptive rows);")
out("# unres/acc: unresolved over accepted moves, all runs; wall s: the whole ensemble")

out("\n## 1. RV case, R = 32 (seeds 0-31), nlive = 200, d = 7")
out(HEAD)
case, model = model_of(1, 4, 96)
fused = model.transform_loglike_device
wrap = np.array([("omega" in p) or ("ml0" in p) for p in case.parnames])
seeds = list(range(32))
nested_sample_ensemble(fused, case.ndim, [0, 1], nlive=200, nsteps=21)  # warm-up (modules, allocator)
nested_sample_ensemble(fused, case.ndim, [0, 1], nlive=200, nsteps=21, adaptive_nsteps="move-distance")
per_round = {}
for tag, kw in (("fixed 21", dict(nsteps=21)), ("fixed 42", dict(nsteps=42)), ("fixed 84", dict(nsteps=84)),
                ("adaptive 21..84", dict(nsteps=21, adaptive_nsteps="move-distance")),
                ("adaptive 21..84, omega wrapped", dict(nsteps=21, adaptive_nsteps="move-distance", wrapped=wrap))):
    dt, res = timed(lambda: nested_sample_ensemble(fused, case.ndim, seeds, nlive=200, **kw))
    per_round[tag] = row(tag, dt, res)
model.close()

out("\n## 2. config-2 model, R = 32 (seeds 0-31), nlive = 200; d = 4 Gaussian, R = 32 (seeds 100-131), nlive = 250")
out(HEAD)
case, model = model_of(2, 11, 300)
fused = model.transform_loglike_device
n3 = 3 * case.ndim
nested_sample_ensemble(fused, case.ndim, [0, 1], nlive=200, nsteps=n3)
for tag, kw in ((f"config 2 (d {case.ndim}): fixed {n3}", dict(nsteps=n3)),
                (f"config 2 (d {case.ndim}): adaptive {n3}..{4 * n3}", dict(nsteps=n3, adaptive_nsteps="move-distance"))):
    dt, res = timed(lambda: nested_sample_ensemble(fused, case.ndim, seeds, nlive=200, **kw))
    row(tag, dt, res)
model.close()


def gauss(U):
    th = -10 + 20 * U
    return th, -0.5 * ((th / 0.6) ** 2).sum(1)


want = 4 * math.log(math.sqrt(2 * math.pi) * 0.6 / 20)
for tag, kw in (("gaussian d 4: fixed 10", dict(nsteps=10)),
                ("gaussian d 4: adaptive 10..40", dict(nsteps=10, adaptive_nsteps="move-distance"))):
    dt, res = timed(lambda: nested_sample_ensemble(gauss, 4, list(range(100, 132)), nlive=250, **kw))
    row(tag, dt, res, want)

out("\n## 3. rvl_slice_runs_radius + rvl_slice_runs_travel per round, CUDA events, random points, kk = 0.2 nlive")
lib = _abi.load()


def kernel_ms(nlive, d, R, rounds=50, warm=5):
    rng = np.random.default_rng([nlive, d, R])
    kk = int(0.2 * nlive)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    L = np.stack([np.tril(rng.normal(0, 0.01, (d, d)), -1) + np.diag(rng.uniform(0.05, 0.2, d)) for _ in range(R)])
    order = np.stack([rng.permutation(nlive) for _ in range(R)]).astype(np.int64)
    run_of = np.repeat(np.arange(R, dtype=np.int32), kk)
    start = np.concatenate([order[r][kk + rng.integers(0, nlive - kk, kk)] for r in range(R)]).astype(np.int64)
    t = dict(u=cuda(rng.uniform(size=(R, nlive, d))), order=cuda(order), kk=cuda(np.full(R, kk, np.int64)),
             chol=cuda(L), run_of=cuda(run_of), start=cuda(start), u_end=cuda(rng.uniform(size=(R * kk, d))),
             rad2=torch.zeros(R, dtype=torch.float64, device="cuda"),
             far=torch.zeros(R, dtype=torch.int32, device="cuda"))
    runs = _abi.rvl_slice_runs(n_runs=R, run_of=t["run_of"].data_ptr(), chol=t["chol"].data_ptr())
    live = _abi.rvl_slice_live(nlive=nlive, d=d, u_live=t["u"].data_ptr(), order=t["order"].data_ptr(),
                               kk=t["kk"].data_ptr(), start=t["start"].data_ptr())
    args = _abi.rvl_slice_args(k=R * kk, d=d, u=t["u_end"].data_ptr())
    stream = torch.cuda.current_stream().cuda_stream

    def one():
        assert lib.rvl_slice_runs_radius(ctypes.byref(runs), ctypes.byref(live), None, t["rad2"].data_ptr(),
                                         stream) == 0
        assert lib.rvl_slice_runs_travel(ctypes.byref(args), ctypes.byref(runs), ctypes.byref(live), None,
                                         t["rad2"].data_ptr(), t["far"].data_ptr(), stream) == 0
    for _ in range(warm):
        one()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(rounds):
        one()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / rounds


out(f"{'nlive':>5s} {'d':>3s} {'R':>3s} {'radius+travel ms':>16s}  round total")
for nlive, d, R in ((200, 7, 1), (200, 7, 32), (200, 7, 64), (650, 26, 1), (650, 26, 16)):
    ms = kernel_ms(nlive, d, R)
    if (nlive, d, R) == (200, 7, 32) and per_round.get("adaptive 21..84"):
        total = (f"{1e3 * per_round['adaptive 21..84']:.1f} ms (section 1, adaptive 21..84: ensemble wall time "
                 "over its rounds)")
    else:
        total = "not measured (no workload of this shape above)"
    out(f"{nlive:5d} {d:3d} {R:3d} {ms:16.4f}  {total}")
