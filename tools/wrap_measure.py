"""Circular coordinates in the built-in slice samplers (rvl_slice_phase_wrapped), measured:
  1. time per move of the three bookkeeping kernels at k = 2048, d = 15, without and with a mask,
     alternated in one process (CUDA events; likelihood launches excluded);
  2. ln Z of the periodic problem of tests/test_gpu_slice_wrap.py, seeds 0-3, without and with
     wrapping, next to the analytic value;
  3. ln Z of make_case(1, seed=4, n_epochs=96) (nlive = 200, nsteps = 3 ndim) from the device
     sampler without a mask, with omega / ml0 wrapped (the reference's rule) and with omega + ma0
     wrapped, next to the UltraNest test double;
  4. the same on two cases with the true omega near 0 = 2 pi, at e = 0.12 and e = 0.02.
usage: python tools/wrap_measure.py [output file]"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from scipy.special import i0e  # noqa: E402

from evidence_b200 import synth  # noqa: E402
from evidence_b200 import ultranest as runner  # noqa: E402
from evidence_b200.rvmodel import RVModel  # noqa: E402
from evidence_b200.sampler_dev import _NativeSlice, nested_sample_device  # noqa: E402

lines = []


def out(s=""):
    print(s, flush=True)
    lines.append(s)


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return f"{name}, power limit / max SM clock: {q.stdout.strip()}"
    except (OSError, subprocess.SubprocessError):
        return f"{name}, power limit not readable"


out(f"# {card()}")
out(f"# torch {torch.__version__}, {time.strftime('%Y-%m-%d %H:%M:%S')}")

# ---- 1. kernels alone, per move (phases 0, 1, 2, 2, 3)
k, d = 2048, 15
dev = torch.device("cuda")
rng = np.random.default_rng(0)
mask = np.zeros(d, bool)
mask[[3, 9]] = True  # two circular coordinates, like omega and ml0 of a 2-planet model
kern = {}
for tag, w in (("no mask", None), ("mask", mask)):
    ns = _NativeSlice(torch, k, d, dev, 5, n_out=8, m=8, rounds=3, wrap=w)
    u = torch.from_numpy(rng.uniform(0.2, 0.8, (k, d))).cuda()
    th, lc = u.clone(), torch.full((k,), np.nan, dtype=torch.float64, device=dev)
    lmin = torch.tensor([-1.0], dtype=torch.float64, device=dev)
    chol = torch.eye(d, dtype=torch.float64, device=dev) * 0.05
    a = ns.args
    a.lmin, a.chol, a.u, a.theta, a.lcur = lmin.data_ptr(), chol.data_ptr(), u.data_ptr(), th.data_ptr(), lc.data_ptr()
    ns.ll_o.fill_(0.0)  # every stepping-out candidate succeeds ...
    ns.ll.fill_(-2.0)   # ... every shrinkage candidate fails: the longest move
    kern[tag] = (ns, (u, th, lc, lmin, chol))


def move(ns, nmoves):
    for i in range(nmoves):
        ns.args.move, ns.args.shrink_round = i, 0
        ns._phase(0)
        ns._phase(1)
        for r in range(ns.rounds):
            ns.args.shrink_round = r + 1
            ns._phase(2 if r + 1 < ns.rounds else 3)


NMOVES, REPS = 50, 7
times = {t: [] for t in kern}
for tag in kern:
    move(kern[tag][0], 5)  # warm-up
for rep in range(REPS):
    for tag in (list(kern) if rep % 2 == 0 else list(kern)[::-1]):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        move(kern[tag][0], NMOVES)
        e1.record()
        e1.synchronize()
        times[tag].append(e0.elapsed_time(e1) * 1e3 / NMOVES)
out()
out(f"## 1. bookkeeping kernels per move (5 launches), k = {k}, d = {d}, n_out = 8, m = 8, 3 rounds;")
out(f"##    {REPS} x {NMOVES} moves, alternated; us per move: median [min, max]")
for tag, v in times.items():
    out(f"{tag:8s} {np.median(v):8.2f} [{min(v):.2f}, {max(v):.2f}]")
out(f"ratio mask / no mask (medians): {np.median(times['mask']) / np.median(times['no mask']):.4f}")

# ---- 2. periodic problem
KAPPA, S = 50.0, 0.03
want = 2 * np.log(i0e(KAPPA)) + 3 * np.log(S * np.sqrt(2 * np.pi))


def periodic(U):
    ll = (KAPPA * (torch.cos(2 * np.pi * U[:, :2]) - 1.0)).sum(1) - ((U[:, 2:] - 0.5) ** 2).sum(1) / (2 * S * S)
    return U.clone(), ll


out()
out(f"## 2. periodic problem, d = 5 (von Mises kappa = 50 in u0, u1, mode on the seam; Gaussians s = 0.03),")
out(f"##    identity transform, nlive = 200, nsteps = 15, native kernels; analytic ln Z = {want:.4f}")
out("wrap   seed     lnZ     err   (lnZ-want)/err   ncall")
for w in (None, [True, True, False, False, False]):
    for seed in range(4):
        r = nested_sample_device(periodic, 5, nlive=200, seed=seed, device="cuda", wrapped=w)
        out(f"{'yes' if w else 'no ':5s} {seed:4d} {r.logz:9.4f} {r.logzerr:6.3f} {(r.logz - want) / r.logzerr:12.2f}"
            f" {r.ncall:10d}")

# ---- 3. the RV case of ADVICE
case = synth.make_case(1, seed=4, n_epochs=96)
model = RVModel(case.fixedpardict, case.datadict(), case.parnames)
model.set_priors(case.priordict)
wrapped = np.array([("omega" in p) or ("ml0" in p) for p in case.parnames])
out()
out(f"## 3. make_case(1, seed=4, n_epochs=96), ndim = {case.ndim}, nlive = 200, nsteps = {3 * case.ndim};"
    f" true omega = {case.truth['planet1_omega']:.3f} rad")
out(f"##    wrapped by the reference's rule: {[p for p, w in zip(case.parnames, wrapped) if w]}")
sys.path.insert(0, os.path.join(ROOT, "tests", "doubles"))
import tempfile  # noqa: E402


def rv_case(case, model):
    """Device sampler, seeds 0-3: no mask, the reference's rule (omega, ml0), and omega + ma0; then
    the UltraNest test double (region sampling, which wraps by the reference's rule)."""
    rule = np.array([("omega" in p) or ("ml0" in p) for p in case.parnames])
    both = np.array([("omega" in p) or ("ma0" in p) or ("ml0" in p) for p in case.parnames])
    out("sampler                      seed      lnZ     err      ncall    s")
    for tag, w in (("slice-device", None), ("slice-device, omega", rule), ("slice-device, omega + ma0", both)):
        vals = []
        for seed in range(4):
            t0 = time.perf_counter()
            r = nested_sample_device(model.transform_loglike_device, case.ndim, nlive=200, nsteps=3 * case.ndim,
                                     seed=seed, device="cuda", wrapped=w)
            vals.append(r.logz)
            out(f"{tag:28s} {seed:4d} {r.logz:9.3f} {r.logzerr:6.3f} {r.ncall:10d} {time.perf_counter() - t0:5.2f}")
        out(f"{tag:28s} mean {np.mean(vals):9.3f}, scatter {np.std(vals, ddof=1):.3f}")
    with tempfile.TemporaryDirectory() as tmp:
        m2 = RVModel(case.fixedpardict, case.datadict(pandas=True), case.parnames)
        t0 = time.perf_counter()
        un = runner.run(m2, {"target": "synth", "runid": "un", "save_dir": tmp, "nplanets": 1}, case.priordict,
                        {"nlive": 200, "sampler": "ultranest", "stepsampler": "none", "ndraw_min": 256,
                         "ndraw_max": 4096})
        out(f"{'UltraNest test double (region)':28s} {'-':>4s} {un.logZ:9.3f} {un.logZerr:6.3f} {un.nlike:10d}"
            f" {time.perf_counter() - t0:5.2f}")
        m2.close()


rv_case(case, model)
model.close()
out("(the double on the CPU oracle, profiles/r2_lnz_scatter.txt: -203.08 +- 0.46 region sampling,"
    " -202.82 +- 0.44 population slice)")

# ---- 4. omega near 0 = 2 pi: measured (e = 0.12) and not (e = 0.02)
for seed in (112, 101):
    case = synth.make_case(1, seed=seed, n_epochs=96)
    t = case.truth
    out()
    out(f"## 4. make_case(1, seed={seed}, n_epochs=96), nlive = 200, nsteps = {3 * case.ndim}; true omega ="
        f" {t['planet1_omega']:.3f} rad, e = {t['planet1_ecc']:.3f}, K = {t['planet1_k1']:.2f} m/s,"
        f" ma0 = {t['planet1_ma0']:.3f} rad")
    model = RVModel(case.fixedpardict, case.datadict(), case.parnames)
    model.set_priors(case.priordict)
    rv_case(case, model)
    model.close()

if len(sys.argv) > 1:
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], "w") as f:
        f.write("\n".join(lines) + "\n")
