"""MLFriends region sampling (nested_sample_ensemble(method='mlfriends')) measured against the slice ensemble:
  1. the RV case of profiles/r7_adaptive_nsteps.txt (make_case(1, seed=4, n_epochs=96), nlive = 200), R = 32
     (seeds 0-31): MLFriends without and with omega wrapped; the slice sampler at fixed 21 and 84 moves
     (the rows of r7, measured again here); one run of the UltraNest test double (region sampling);
  2. the config-2 model of r6 / r7 (make_case(2, seed=11, n_epochs=300), nlive = 200), R = 32: MLFriends
     against the slice sampler at 3 ndim moves;
  3. the mixture (d = 6) and Gaussian-shell (d = 2, 5) problems of tests/test_gpu_region.py, R = 32:
     MLFriends against the slice sampler at 3 ndim moves, with their analytic ln Z;
  4. kernel time (CUDA events, 50 rounds after 5 warm-up rounds, random points) of rvl_region_runs_radius
     (30 bootstraps), one _draw of 1.5 kk / 0.25 slots per run and one _pick, at nlive 200 / d 7 / R 32 and
     nlive 375 / d 15 / R 32, kk = 0.2 nlive, beside the measured time per round of section 1 or 2.
Columns: mean, std and median ln Z, median reported logzerr, std / median logzerr, lnL calls per run,
wall time of the ensemble, region efficiency (replacements per geometric draw) and geometric draws per run.
usage: python tools/region_measure.py [output file]"""
import ctypes
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from evidence_b200 import _abi, synth  # noqa: E402
from evidence_b200 import ultranest as runner  # noqa: E402
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


def model_of(n_planets, seed, n_epochs, pandas=False):
    case = synth.make_case(n_planets, seed=seed, n_epochs=n_epochs)
    model = RVModel(case.fixedpardict, case.datadict(pandas=pandas), case.parnames)
    model.set_priors(case.priordict)
    return case, model


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, res


HEAD = (f"{'configuration':36s} {'mean lnZ':>9s} {'std':>7s} {'median':>9s} {'err med':>7s} {'std/err':>7s} "
        f"{'calls/run':>10s} {'wall s':>7s} {'eff':>7s} {'draws/run':>10s}")
SEEDS = list(range(32))


def row(tag, dt, res, want=None):
    z = np.array([r.logz for r in res])
    e = np.median([r.logzerr for r in res])
    region = res[0].get("region_draws") is not None
    eff = f"{np.sum([r.niter for r in res]) / np.sum([r.region_draws for r in res]):7.4f}" if region else f"{'-':>7s}"
    draws = f"{np.mean([r.region_draws for r in res]):10.0f}" if region else f"{'-':>10s}"
    out(f"{tag:36s} {z.mean():9.3f} {z.std(ddof=1):7.3f} {np.median(z):9.3f} {e:7.3f} {z.std(ddof=1) / e:7.2f} "
        f"{np.mean([r.ncall for r in res]):10.0f} {dt:7.1f} {eff} {draws}")
    if want is not None:
        out(f"{'':36s} analytic {want:.4f}: (mean - analytic) / standard error "
            f"{(z.mean() - want) / (z.std(ddof=1) / math.sqrt(len(z))):.2f}")
    rounds = max(r.niter for r in res) / (0.2 * res[0].nlive)
    return dt / rounds


def ensemble(tag, fused, ndim, nlive, want=None, **kw):
    t0 = time.perf_counter()
    try:
        dt, res = timed(lambda: nested_sample_ensemble(fused, ndim, SEEDS, nlive=nlive, **kw))
    except RuntimeError as e:  # max_calls: a run whose efficiency collapsed
        out(f"{tag:36s} stopped after {time.perf_counter() - t0:.1f} s: {e}")
        return None
    return row(tag, dt, res, want)


out(f"# {card()}")
out(f"# torch {torch.__version__}, {time.strftime('%Y-%m-%d %H:%M:%S')}")
out("# command: python tools/region_measure.py profiles/r8_mlfriends.txt")
out("# eff: replacements (niter) over geometric draws, all runs; wall s: the whole ensemble")

out("\n## 1. RV case, R = 32 (seeds 0-31), nlive = 200, d = 7")
out(HEAD)
case, model = model_of(1, 4, 96)
fused = model.transform_loglike_device
wrap = np.array([("omega" in p) or ("ml0" in p) for p in case.parnames])
nested_sample_ensemble(fused, case.ndim, [0, 1], nlive=200, nsteps=21)  # warm-up (modules, allocator)
per_round = {}
cap = dict(method="mlfriends", max_calls=500_000_000)  # bounds a run whose region efficiency collapses
for tag, kw in (("mlfriends", cap), ("mlfriends, omega wrapped", dict(cap, wrapped=wrap)),
                ("slice, fixed 21", dict(nsteps=21)), ("slice, fixed 84", dict(nsteps=84))):
    per_round[tag] = ensemble(tag, fused, case.ndim, 200, **kw)
model.close()
sys.path.insert(0, os.path.join(ROOT, "tests", "doubles"))
with tempfile.TemporaryDirectory() as tmp:
    case, m2 = model_of(1, 4, 96, pandas=True)
    t0 = time.perf_counter()
    un = runner.run(m2, {"target": "synth", "runid": "un", "save_dir": tmp, "nplanets": 1}, case.priordict,
                    {"nlive": 200, "sampler": "ultranest", "stepsampler": "none", "ndraw_min": 256, "ndraw_max": 4096})
    out(f"{'UltraNest test double (region), 1 run':36s} {un.logZ:9.3f} {'-':>7s} {'-':>9s} {un.logZerr:7.3f} {'-':>7s} "
        f"{un.nlike:10d} {time.perf_counter() - t0:7.1f}")
    m2.close()

out("\n## 2. config-2 model, R = 32 (seeds 0-31), nlive = 200")
out(HEAD)
case, model = model_of(2, 11, 300)
fused = model.transform_loglike_device
n3 = 3 * case.ndim
per_round["config 2"] = ensemble(f"config 2 (d {case.ndim}): mlfriends", fused, case.ndim, 200, **cap)
ensemble(f"config 2 (d {case.ndim}): slice, fixed {n3}", fused, case.ndim, 200, nsteps=n3)
model.close()

out("\n## 3. mixture and Gaussian shells of tests/test_gpu_region.py, R = 32 (seeds 0-31)")
out(HEAD)
import test_gpu_region as tg  # noqa: E402

for tag, fn, d, nlive, want in (("mixture d 6", tg.mixture, 6, 300, 0.0),
                                ("shells d 2", tg.shells(2), 2, 300, tg.shells_lnz(2)),
                                ("shells d 5", tg.shells(5), 5, 300, tg.shells_lnz(5))):
    ensemble(f"{tag}: mlfriends", fn, d, nlive, want, method="mlfriends")
    ensemble(f"{tag}: slice, fixed {3 * d}", fn, d, nlive, want, nsteps=3 * d)

out("\n## 4. region kernels per round, CUDA events, random points, kk = 0.2 nlive, 30 bootstraps")
lib = _abi.load()


def kernel_ms(nlive, d, R, rounds=50, warm=5):
    rng = np.random.default_rng([nlive, d, R])
    kk = int(0.2 * nlive)
    slots = int(1.5 * kk / 0.25)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    L = np.stack([np.tril(rng.normal(0, 0.01, (d, d)), -1) + np.diag(rng.uniform(0.05, 0.2, d)) for _ in range(R)])
    order = np.stack([rng.permutation(nlive) for _ in range(R)]).astype(np.int64)
    S = R * slots
    i32, f64 = torch.int32, torch.float64
    t = dict(seeds=cuda(np.arange(R, dtype=np.int64)), u=cuda(0.5 + 0.3 * (rng.uniform(size=(R, nlive, d)) - 0.5)),
             order=cuda(order), kk=cuda(np.full(R, kk, np.int64)), chol=cuda(L), lmin=cuda(np.zeros(R)),
             run_of=cuda(np.repeat(np.arange(R, dtype=np.int32), kk)),
             walker_of=cuda(np.tile(np.arange(kk, dtype=np.int32), R)),
             base=cuda(np.arange(R + 1, dtype=np.int32) * slots), rad2=torch.zeros(R, dtype=f64, device="cuda"),
             stage=torch.zeros((S, d), dtype=f64, device="cuda"), flag=torch.zeros(S, dtype=torch.uint8, device="cuda"),
             count=torch.zeros(R, dtype=i32, device="cuda"), offs=torch.zeros(R + 1, dtype=i32, device="cuda"),
             cand=torch.zeros((S, d), dtype=f64, device="cuda"), th=torch.zeros((S, d), dtype=f64, device="cuda"),
             ll=cuda(rng.normal(size=S)), sel=torch.zeros(S, dtype=i32, device="cuda"),
             fa=torch.zeros((2, R), dtype=i32, device="cuda"), wu=torch.zeros((R * kk, d), dtype=f64, device="cuda"),
             wth=torch.zeros((R * kk, d), dtype=f64, device="cuda"), wl=torch.zeros(R * kk, dtype=f64, device="cuda"))
    runs = _abi.rvl_slice_runs(n_runs=R, seeds=t["seeds"].data_ptr(), chol=t["chol"].data_ptr(),
                               run_of=t["run_of"].data_ptr(), walker_of=t["walker_of"].data_ptr(),
                               lmin=t["lmin"].data_ptr())
    live = _abi.rvl_slice_live(nlive=nlive, d=d, u_live=t["u"].data_ptr(), order=t["order"].data_ptr(),
                               kk=t["kk"].data_ptr())
    g = _abi.rvl_region_args(num_bootstraps=30, max_slots=slots, rad2=t["rad2"].data_ptr(),
                             slot_base=t["base"].data_ptr(), stage=t["stage"].data_ptr(), flag=t["flag"].data_ptr(),
                             count=t["count"].data_ptr(), offs=t["offs"].data_ptr(), cand=t["cand"].data_ptr(),
                             cand_th=t["th"].data_ptr(), cand_ll=t["ll"].data_ptr(), sel=t["sel"].data_ptr(),
                             filled=t["fa"][0].data_ptr(), above=t["fa"][1].data_ptr())
    args = _abi.rvl_slice_args(k=R * kk, d=d, u=t["wu"].data_ptr(), theta=t["wth"].data_ptr(), lcur=t["wl"].data_ptr())
    stream = torch.cuda.current_stream().cuda_stream
    G, RN, LV = ctypes.byref(g), ctypes.byref(runs), ctypes.byref(live)
    calls = {"radius": lambda: lib.rvl_region_runs_radius(G, RN, LV, None, stream),
             "draw": lambda: lib.rvl_region_runs_draw(G, RN, LV, None, stream),
             "pick": lambda: lib.rvl_region_runs_pick(G, ctypes.byref(args), RN, LV, stream)}
    ms = {}
    for name, fn in calls.items():
        for _ in range(warm):
            assert fn() == 0, lib.rvl_slice_last_error().decode()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(rounds):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms[name] = e0.elapsed_time(e1) / rounds
    acc = int(t["offs"][-1])
    return ms, slots, acc


out(f"{'nlive':>5s} {'d':>3s} {'R':>3s} {'slots/run':>9s} {'accepted':>8s} {'radius ms':>9s} {'draw ms':>8s} "
    f"{'pick ms':>8s}  round (measured above)")
for nlive, d, R, key in ((200, 7, 32, "mlfriends"), (375, 15, 32, None)):
    ms, slots, acc = kernel_ms(nlive, d, R)
    pr = per_round.get(key) if key else None
    total = sum(ms.values())
    share = (f"{1e3 * pr:.1f} ms per round (section 1, {key}); the three kernels {100 * total / (1e3 * pr):.1f} %"
             if pr else "not measured (no workload of this shape above)")
    out(f"{nlive:5d} {d:3d} {R:3d} {slots:9d} {acc:8d} {ms['radius']:9.4f} {ms['draw']:8.4f} {ms['pick']:8.4f}  {share}")
