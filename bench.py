#!/usr/bin/env python
"""
bench.py — headline benchmark of the B200-native RV log-likelihood path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): RV lnL evals/sec (K-planet, batched) at 1/2/4/8 B200, plus the fraction of
the FP64 roofline.  Workload at every N: BASELINE.json configs[2], the configuration the metric
is quoted on -- 4-planet model, 3 instruments, 5000 epochs, a batched lnL sweep; one step = one
batch of theta per GPU (rows sharded over the ranks, weak scaling; per-rank lnL vectors gathered
inside the step by the fused all-gather over NVLink).  The batch is a function of --steps only
(`batch_for`): large enough that K steps are >= 2 s of device work.

One JSON line on stdout (rank 0).  `value` = device-timed throughput with theta resident in HBM;
`e2e` = the same metric through the public host-buffer call (page-locked host theta -> kernel ->
gathered lnL in host memory: rvl_loglike at N = 1, rvl_loglike_gather per rank at N > 1);
`roofline` = algorithmic FP64 flops of the likelihood kernel / its CUDA-event time / the FP64
peak measured in the same run by a register-resident DFMA loop (MEASURED_PEAKS.json has no FP64
row); `parity` = max |lnL - reference| over >= 1e4 theta of the bench model evaluated BEFORE the
timed region (the run exits non-zero when it fails); `gather_check` (N > 1) = the fused
all-gather's vector against NCCL's; `cpu_baseline` = the reference implementation itself
(oracle/_ref, staged by oracle/Makefile) on the box's host cores.

`--impl reference` times that CPU implementation alone, on the same config/metric.

`--dump-outputs DIR` writes the lnL vector of the last timed step (what the caller of the step
receives: at N > 1 the gathered vector of all ranks) to DIR/lnl.npy in float64, so that two builds
run with the same arguments, and therefore the same seeded theta, can be compared row for row.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "RV lnL evals/sec (K-planet, batched)"
UNIT = "lnL/s"
CONFIG_ID = 3          # BASELINE.json configs[2]: N = 5000 epochs, K = 4 planets, 3 instruments
LATENCY_CONFIG = 2     # configs[1]: the UltraNest ndraw = 4096 call, reported as a latency line
LATENCY_BATCH = 4096
STRESS_TOTAL = 10_000_000  # configs[4]: 1e7 theta x 1e4 epochs x 3 planets over all ranks
NOMINAL_RATE = 4.5e6   # lnL/s/GPU on config 3: only used to size the batch deterministically
DUMP_BYTES = 64_000_000  # --dump-outputs: at most this much in all


def batch_for(steps):
    """theta rows per GPU and step: a power-of-two multiple of 131072 inside configs[2]'s 1e4-1e6
    range such that `steps` steps are >= 2 s of device work.  A function of --steps only, so that
    both arms (and every N) state the same config."""
    b = 131072
    while steps * b < 2.0 * NOMINAL_RATE and b < 1048576:
        b *= 2
    return b


def algorithmic_flops(n_epochs, n_planets, drift_order, mean_iters):
    """SURVEY.md 8(d): F = N [K (51 + 46 I) + 48 + 2 d] FP64 flops per lnL."""
    return n_epochs * (n_planets * (51.0 + 46.0 * mean_iters) + 48.0 + 2.0 * drift_order)


def dump_outputs(dirpath, lnl):
    """Write the last timed step's lnL vector as DIR/lnl.npy (float64).  A vector larger than half
    of DUMP_BYTES (N = 8 at the largest batch) is replaced by a fixed seeded sample of a quarter of
    that size, with the rows' positions in DIR/lnl_rows.npy (float64, exact)."""
    lnl = np.ascontiguousarray(lnl, dtype=np.float64)
    os.makedirs(dirpath, exist_ok=True)
    out = {"lnl": lnl}
    if lnl.nbytes > DUMP_BYTES // 2:
        rows = np.sort(np.random.default_rng(0).choice(lnl.size, DUMP_BYTES // 32, replace=False))
        out = {"lnl": lnl[rows], "lnl_rows": rows.astype(np.float64)}
    for name, arr in out.items():
        np.save(os.path.join(dirpath, name + ".npy"), arr)
    return sorted(out)


def workload_config(case, batch, world):
    return {"workload": f"config{CONFIG_ID} (BASELINE.json configs[2]): {case.n_planets}-planet Keplerian, "
                        f"{case.n_inst} instruments, {case.n_epochs} epochs, batched lnL sweep, "
                        f"{batch} theta per step per GPU",
            "n_epochs": case.n_epochs, "n_planets": case.n_planets, "n_inst": case.n_inst,
            "ndim": case.ndim, "batch_per_gpu": batch, "global_batch": batch * world,
            "parallelism": f"rows sharded x{world}, lnL all-gather",
            "l2": "flushed (256 MiB write) between timed steps"}


# ------------------------------------------------------------------------------------------
# CPU side: the reference implementation (oracle/_ref: the reference's own RVModel + C solver,
# staged by oracle/Makefile) or, where that is absent, the restatement (oracle/rv_oracle.py).
# Test infrastructure: used here as the checker (parity) and as the timed CPU baseline only.
# ------------------------------------------------------------------------------------------
_W = {}


def _cpu_model(key):
    """Per worker process: one CPU model per (config, variant) key, built on first use."""
    if key not in _W:
        from evidence_b200 import synth
        from oracle import ref_runner, rv_oracle
        config, variant = key
        case = synth.make_case(config)
        parnames, fixed = variant_names(case, variant)
        if ref_runner.available():
            _W[key] = ("reference", ref_runner.make_model(fixed, case.datadict(), parnames))
        else:
            _W[key] = ("port", rv_oracle.OracleRVModel(fixed, case.datadict(), parnames))
    return _W[key]


def _cpu_eval(task):
    key, block = task
    kind, model = _cpu_model(key)
    if kind == "reference":
        from oracle import ref_runner
        return ref_runner.loglike_rows(model, block)
    return model.log_likelihood_batch(block)


def cpu_kind():
    from oracle import ref_runner, rv_oracle
    rv_oracle.build()
    return "reference" if ref_runner.available() else "port"


def kind_text(kind):
    return ("the unmodified reference RVModel.log_likelihood (evidence/rvmodel, staged in oracle/_ref) "
            "looped over rows, its own trueanomaly.c" if kind == "reference" else
            "numpy restatement of RVModel.log_likelihood (oracle/rv_oracle.py)")


def make_pool(cores):
    import multiprocessing as mp
    return mp.get_context("fork").Pool(cores)


def pool_rate(pool, cores, key, theta, seconds):
    """lnL/s of the CPU arm over a bounded sample of `theta` (rows repeated to fill ~`seconds`)."""
    probe = theta[: max(cores * 2, 32)]
    t0 = time.perf_counter()  # first touch builds the models in the workers
    pool.map(_cpu_eval, [(key, b) for b in np.array_split(probe, cores)])
    t0 = time.perf_counter()
    pool.map(_cpu_eval, [(key, b) for b in np.array_split(probe, cores)])
    rate0 = len(probe) / (time.perf_counter() - t0)
    n = int(max(len(probe), rate0 * seconds))
    sample = np.tile(theta, (-(-n // len(theta)), 1))[:n]
    t0 = time.perf_counter()
    pool.map(_cpu_eval, [(key, b) for b in np.array_split(sample, cores * 4)])
    dt = time.perf_counter() - t0
    return n / dt, n, dt


def run_reference(args, rank, world, emit):
    """The CPU arm: the reference on all host cores; every step is a bounded sample of the
    workload, sized so that warmup + steps together take about two minutes."""
    if rank != 0:
        return
    from evidence_b200 import synth
    kind = cpu_kind()
    case = synth.make_case(CONFIG_ID)
    B = batch_for(args.steps)
    cores = os.cpu_count() or 1
    theta = case.draw_theta(8192, seed=1000)  # rows of the step's batch (same seed as rank 0's)
    n_steps = args.warmup + args.steps
    per_step_s = min(12.0, max(0.5, 110.0 / max(1, n_steps)))
    key = (CONFIG_ID, "bench")
    rates = []
    with make_pool(cores) as pool:
        rate0, _, _ = pool_rate(pool, cores, key, theta, 2.0)
        n = int(max(cores * 2, rate0 * per_step_s))
        sample = np.tile(theta, (-(-n // len(theta)), 1))[:n]
        tasks = [(key, b) for b in np.array_split(sample, cores * 4)]
        for k in range(n_steps):
            t0 = time.perf_counter()
            pool.map(_cpu_eval, tasks)
            dt = time.perf_counter() - t0
            if k >= args.warmup:
                rates.append(n / dt)
    value = float(np.mean(rates)) if rates else 0.0
    sample_txt = (f"{n} lnL evaluations per step (rows of the {B}-theta batch) on {cores} processes; "
                  + kind_text(kind))
    emit({"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
          "steps": args.steps, "warmup": args.warmup,
          "ms_per_step": 1e3 * n / value if value else None, "higher_is_better": True,
          "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
          "config": workload_config(case, B, world),
          "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                           "sample": sample_txt},
          "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


# ------------------------------------------------------------------------------------------
# parity sets: theta of the bench model, evaluated on the device before the timed region and on
# the CPU by the reference (SURVEY.md 8(d) "parity check in the same run")
# ------------------------------------------------------------------------------------------
def variant_names(case, variant):
    """(parnames, fixedpardict) of the bench model ("bench") or of the same model with every planet
    re-parametrised as secos / sesin / ml0 ("secos": the parametrisation whose e > 1 is the
    reference's -1e30 sentinel, evidence/rvmodel/__init__.py:425-431, 198-203)."""
    if variant == "bench":
        return list(case.parnames), dict(case.fixedpardict)
    names = []
    for p in case.parnames:
        p = p.replace("_ecc", "_secos").replace("_omega", "_sesin").replace("_ma0", "_ml0")
        names.append(p)
    return sorted(names), dict(case.fixedpardict)


def parity_sets(case):
    """[(name, variant, theta, abs_bar)]; bar None = reported only."""
    rng = np.random.default_rng(20260)
    names = case.parnames
    K = case.n_planets
    ecc_cols = [names.index(f"planet{k}_ecc") for k in range(1, K + 1)]
    sets = []
    sets.append(("prior_draws", "bench", case.draw_theta(8192, seed=4242), 1e-9))
    th = case.draw_theta(1024, seed=4243)  # one planet per row just above the prior's e < 0.95
    for i in range(len(th)):
        th[i, ecc_cols[i % K]] = rng.uniform(0.95, 0.97)
    sets.append(("ecc_0.95_0.97", "bench", th, 1e-9))
    th = case.draw_theta(512, seed=4244)
    for j, p in enumerate(names):
        if p.endswith("_jitter"):
            th[:, j] = 0.0
    sets.append(("jitter_zero", "bench", th, 1e-9))
    th = case.draw_theta(512, seed=4245)  # chaotic-Newton regime: bounded by the solver tolerance
    for i in range(len(th)):
        th[i, ecc_cols[i % K]] = rng.uniform(0.97, 1.0)
    sets.append(("ecc_0.97_1.00", "bench", th, 1e-5))
    # secos / sesin parametrisation: ~30 % of the rows have one planet with e > 1 -> -1e30
    vnames, _ = variant_names(case, "secos")
    base = case.draw_theta(512, seed=4246)
    th = np.empty((512, len(vnames)))
    for j, p in enumerate(vnames):
        src = p.replace("_secos", "_ecc").replace("_sesin", "_omega").replace("_ml0", "_ma0")
        th[:, j] = base[:, names.index(src)]
    for k in range(1, K + 1):
        e = rng.uniform(0.0, 0.9, 512)
        bad = rng.random(512) < 0.3 / K
        e[bad] = rng.uniform(1.0001, 1.5, bad.sum())
        w = rng.uniform(0.0, 2 * np.pi, 512)
        th[:, vnames.index(f"planet{k}_secos")] = np.sqrt(e) * np.cos(w)
        th[:, vnames.index(f"planet{k}_sesin")] = np.sqrt(e) * np.sin(w)
    sets.append(("secos_sesin_invalid", "secos", th, 1e-9))
    return sets


def parity_verdict(sets, got, want, kind, classify=None):
    """Compare device and CPU values set by set; returns (report, ok).

    The e > 0.97 set: Newton from E = M has attracting cycles for e in (0.98, 0.99] -- about 1.5e-7 of
    such solves never converge IN THE REFERENCE'S OWN ARITHMETIC (profiles/r2_newton_cap.txt); the
    reference then aborts the whole trueanomaly() call at 10000 iterations, ignores the return code
    (evidence/rvmodel/__init__.py:490) and uses a partly zero-filled nu, while the device keeps the
    last iterate and counts the event.  Which (theta, epoch) ends in a cycle follows the last bit of
    sin/cos, so either side may hit it alone.  Rows over the bar are therefore re-examined one by one
    (`classify`: device cap counter, and the C port's cap counter for the reference's arithmetic) and
    reported as `cap_rows` instead of failing the run."""
    out = {"n": 0, "max_abs": 0.0, "sentinels_equal": True, "n_sentinels": 0, "checker": kind,
           "bar": "abs <= max(1e-9, 1e-13 |lnL|) (SURVEY.md 8d); -1e30 sentinels identical", "sets": {}}
    ok = True
    for (name, _, theta, bar), g, w in zip(sets, got, want):
        sent = w == -1e30
        sent_ok = bool(np.array_equal(g == -1e30, sent))
        err = np.where(sent, 0.0, np.abs(g - w))
        bound = np.maximum(bar, 1e-13 * np.abs(w))
        cap_rows = []
        if bar > 1e-9 and classify is not None:
            over = np.nonzero(err > bound)[0]
            for i in over[:16]:
                dev_caps, ref_caps = classify(theta[i])
                if dev_caps or ref_caps:
                    cap_rows.append({"row": int(i), "abs_err": float(err[i]), "device_cap_hits": int(dev_caps),
                                     "reference_cap_hits": int(ref_caps)})
                    err[i] = 0.0
        passed = bool(sent_ok and np.all(err <= bound))
        rep = {"n": int(len(w)), "max_abs": float(err.max()), "bar_abs": bar,
               "max_abs_lnl": float(np.abs(np.where(sent, 0.0, w)).max()),
               "bit_identical": int(np.sum((g == w) & ~sent)), "sentinels": int(sent.sum()),
               "pass": passed}
        if cap_rows:
            rep["cap_rows"] = cap_rows
        out["sets"][name] = rep
        out["n_sentinels"] += int(sent.sum())
        out["sentinels_equal"] = out["sentinels_equal"] and sent_ok
        if bar <= 1e-9:  # the north-star bar; the e > 0.97 set is reported beside it
            out["n"] += int(len(w))
            out["max_abs"] = max(out["max_abs"], float(err.max()))
        else:
            out["max_abs_high_ecc"] = float(err.max())
        ok = ok and passed
    out["pass"] = ok
    return out, ok


# ------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "50", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); smax.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(np.max(smax)) if smax else None,
                "power_w_max": float(np.max(power)) if power else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# extras (every N): configs[2]'s sweep sizes, the configs[1] latency line, the configs[4] stress
# ------------------------------------------------------------------------------------------
class Ranks:
    """max-over-ranks reduction of device times (every multi-GPU number is the slowest rank's)."""

    def __init__(self, torch, dist, world):
        self.torch, self.dist, self.world = torch, dist, world

    def max(self, *vals):
        if self.world == 1:
            return [float(v) for v in vals]
        t = self.torch.tensor(vals, dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def sum(self, *vals):
        if self.world == 1:
            return [float(v) for v in vals]
        t = self.torch.tensor(vals, dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in t]

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()


def timed_ms(torch, fn, reps):
    """Mean device time of fn() over `reps` calls (CUDA events on the launching stream)."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.mean([a.elapsed_time(b) for a, b in ev]))


def sweep_sizes(model, case, rank, world, ranks, torch, peak):
    """BASELINE.json configs[2]: the batched lnL sweep at 1e4, 1e5 and 1e6 points in total, rows
    sharded over the ranks (strong scaling of a fixed total)."""
    from evidence_b200.multigpu import shard_bounds
    out = []
    for total in (10_000, 100_000, 1_000_000):
        lo, hi, _ = shard_bounds(total, world, rank)
        theta = torch.from_numpy(case.draw_theta(hi - lo, seed=300 + rank)).cuda()
        lnl = torch.empty(hi - lo, dtype=torch.float64, device="cuda")
        model.log_likelihood_device(theta, out=lnl)
        ranks.barrier()
        model.reset_counters()
        ms = timed_ms(torch, lambda: model.log_likelihood_device(theta, out=lnl), 3)
        c = model.counters()
        mean_it = c["n_newton_iters"] / max(1, c["n_solves"])
        (ms,) = ranks.max(ms)
        F = algorithmic_flops(case.n_epochs, case.n_planets, case.drift, mean_it)
        rate = total / (ms * 1e-3)
        out.append({"total_points": total, "lnl_per_s": rate, "ms": ms,
                    "frac_of_fp64_peak": rate * F / 1e12 / (peak * world) if peak else None})
    return out


def latency_line(make_model, rank, world, ranks, torch, peak, gather_mode):
    """BASELINE.json configs[1]: one UltraNest-sized call, ndraw = 4096 theta per GPU (2 planets +
    linear drift, 1000 epochs).  A latency measurement: the kernel is one launch of ~0.13 ms."""
    from evidence_b200 import synth
    case = synth.make_case(LATENCY_CONFIG)
    model = make_model(case)
    B = LATENCY_BATCH
    theta_host = case.draw_theta(B, seed=1000 + rank)
    theta = torch.from_numpy(theta_host).cuda()
    lnl = torch.empty(B, dtype=torch.float64, device="cuda")
    fused = None
    if world > 1 and gather_mode != "nccl":
        from evidence_b200.multigpu import FusedGatherLikelihood
        fused = FusedGatherLikelihood(model, B)
        step = lambda: fused.evaluate_local(theta)
    elif world > 1:
        from evidence_b200.multigpu import ShardedLikelihood
        sh = ShardedLikelihood(lambda blk: model.log_likelihood_device(blk, out=lnl), case.ndim)
        step = lambda: sh.evaluate_local(theta)
    else:
        step = lambda: model.log_likelihood_device(theta, out=lnl)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    model.set_option("timing", 1)
    for _ in range(10):
        step()
    ranks.barrier()
    model.reset_counters()
    steps, tot, kms = 200, 0.0, []
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        flush.zero_()
        a.record()
        step()
        b.record()
        kms.append(model.last_kernel_ms())
    ranks.barrier()
    tot = float(sum(a.elapsed_time(b) for a, b in ev))
    c = model.counters()
    model.set_option("timing", 0)
    # end to end, host buffers, one library call per step
    th_pin = torch.from_numpy(theta_host).pin_memory()
    out_pin = torch.empty(B * world, dtype=torch.float64).pin_memory()
    th_np, out_np = th_pin.numpy(), out_pin.numpy()
    shared = None
    if fused is not None:
        try:  # host consumers: the gather through a host segment shared by the ranks
            from evidence_b200.multigpu import SharedHostGather
            shared = SharedHostGather(model, B)
            call = lambda: shared.evaluate_local_host(th_np)
        except Exception as exc:  # noqa: BLE001
            print(f"shared-host gather unavailable ({exc!r}); using rvl_loglike_gather", file=sys.stderr)
            call = lambda: fused.evaluate_local_host(th_np, out_np)
    else:
        call = lambda: model.log_likelihood_batch(th_np, out=out_np[:B])
    for _ in range(10):
        call()
    ranks.barrier()
    gc.collect(); gc.disable()
    marks = [time.perf_counter()]
    for _ in range(steps):
        call()
        marks.append(time.perf_counter())
    gc.enable()
    us = np.diff(np.array(marks)) * 1e6
    e2e_s = marks[-1] - marks[0]
    tot, e2e_s = ranks.max(tot, e2e_s)
    mean_it = c["n_newton_iters"] / max(1, c["n_solves"])
    F = algorithmic_flops(case.n_epochs, case.n_planets, case.drift, mean_it)
    k_ms = float(np.mean(kms))
    res = {"workload": f"config{LATENCY_CONFIG} (configs[1]): 2 planets + linear drift, 2 instruments, "
                       f"1000 epochs, UltraNest vectorized ndraw = {B} theta per GPU and call",
           "lnl_per_s": world * B * steps / (tot * 1e-3), "us_per_step": 1e3 * tot / steps,
           "kernel_us": 1e3 * k_ms, "frac_of_fp64_peak": B * F / (k_ms * 1e-3) / 1e12 / peak if peak else None,
           "e2e_lnl_per_s": world * B * steps / e2e_s,
           "e2e_api": ("rvl_loglike" if world == 1 else
                       "rvl_loglike_scatter_host + rvl_wait_host_flags" if shared is not None else "rvl_loglike_gather"),
           "e2e_us_per_call_percentiles_1_50_99": [float(x) for x in np.percentile(us, [1, 50, 99])]}
    if shared is not None:
        shared.close()
    model.close()
    return res


def stress(make_model, rank, world, ranks, torch, peak):
    """BASELINE.json configs[4]: raw kernel stress, 1e7 parameter vectors x 1e4 epochs x 3 planets
    (rows sharded over the ranks), Kepler solves/s against the FP64 peak.  Everything stays on the
    device: U ~ torch.rand, the prior transform fused in front of the likelihood."""
    from evidence_b200 import synth
    from evidence_b200.multigpu import shard_bounds
    case = synth.make_case(5)
    model = make_model(case)
    model.set_priors(case.priordict)
    model.set_option("timing", 1)
    lo, hi, _ = shard_bounds(STRESS_TOTAL, world, rank)
    rows = hi - lo
    gen = torch.Generator(device="cuda").manual_seed(5 + rank)
    U = torch.rand((100_000, case.ndim), dtype=torch.float64, device="cuda", generator=gen)
    model.transform_loglike_device(U)  # warm launch
    U = torch.rand((rows, case.ndim), dtype=torch.float64, device="cuda", generator=gen)
    theta = torch.empty_like(U)
    lnl = torch.empty(rows, dtype=torch.float64, device="cuda")
    ranks.barrier()
    model.reset_counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    model.transform_loglike_device(U, theta=theta, lnl=lnl)
    e1.record()
    torch.cuda.synchronize()
    total_ms, k_ms = e0.elapsed_time(e1), model.last_kernel_ms()
    c = model.counters()
    finite = bool(torch.isfinite(lnl).all().item())
    total_ms, k_ms = ranks.max(total_ms, k_ms)
    solves, iters, caps = ranks.sum(c["n_solves"], c["n_newton_iters"], c["n_cap_hits"])
    mean_it = iters / max(1.0, solves)
    F = algorithmic_flops(case.n_epochs, case.n_planets, case.drift, mean_it)
    ach = STRESS_TOTAL * F / (k_ms * 1e-3) / 1e12
    res = {"workload": f"configs[4] stress: N={case.n_epochs} K={case.n_planets}, {STRESS_TOTAL} theta in total "
                       f"({rows} per GPU), u -> theta -> lnL on the device",
           "kepler_solves": int(solves), "kernel_ms": k_ms, "total_ms_with_prior_transform": total_ms,
           "kepler_solves_per_s": solves / (k_ms * 1e-3), "lnl_per_s": STRESS_TOTAL / (k_ms * 1e-3),
           "mean_newton_iters": mean_it, "achieved_tflops": ach,
           "frac_of_fp64_peak": ach / (peak * world) if peak else None,
           "newton_cap_hits": int(caps), "all_finite": finite}
    model.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="theta per GPU and step (default: batch_for(steps))")
    ap.add_argument("--no-extras", action="store_true", help="skip cpu baseline, sweeps, latency line, stress")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run parity check (profiling runs)")
    ap.add_argument("--e2e-gather", default="shared-host", choices=["shared-host", "device"],
                    help="multi-GPU end-to-end call: lnL stored by the kernels straight into a host segment "
                         "shared by the ranks (rvl_loglike_scatter_host; default), or gathered on the devices "
                         "and copied back (rvl_loglike_gather)")
    ap.add_argument("--gather", default="fused", choices=["fused", "fused-barrier", "nccl"],
                    help="multi-GPU: the all-gather fused into the likelihood launch over NVLink "
                         "symmetric memory (peer stores + completion flags; default), the same with "
                         "a symmetric-memory barrier, or NCCL all_gather")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the lnL vector of the last timed step to DIR/lnl.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    # stdout carries exactly ONE JSON line: libraries that print to fd 1 (NCCL's version banner,
    # torchrun notices) are sent to stderr for the duration of the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    if args.impl == "reference":
        run_reference(args, rank, world, emit)
        return

    from evidence_b200 import synth
    case = synth.make_case(CONFIG_ID)
    B, K, W = (args.batch or batch_for(args.steps)), args.steps, args.warmup

    # ---- the CPU checker starts first (rank 0): worker processes are forked BEFORE CUDA / NCCL
    # exist in this process, and evaluate the parity sets while the device warms up
    pool, psets, want_async, kind = None, None, None, None
    cores = os.cpu_count() or 1
    if not args.no_parity:
        psets = parity_sets(case)
        if rank == 0:
            kind = cpu_kind()
            pool = make_pool(cores)
            tasks, owner = [], []
            for si, (_, variant, th, _) in enumerate(psets):
                for blk in np.array_split(th, max(1, len(th) // 32)):
                    tasks.append(((CONFIG_ID, variant), blk))
                    owner.append(si)
            want_async = pool.map_async(_cpu_eval, tasks, chunksize=1)
    elif rank == 0 and world == 1 and not args.no_extras:
        kind = cpu_kind()
        pool = make_pool(cores)

    import torch
    import torch.distributed as dist
    from evidence_b200 import build
    from evidence_b200.multigpu import ShardedLikelihood
    from evidence_b200.rvmodel import RVModel

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); "
                         "use --impl reference for the CPU arm")
    build.build()
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ranks = Ranks(torch, dist, world)

    def make_model(c, names=None, fixed=None):
        return RVModel(dict(fixed if fixed is not None else c.fixedpardict), c.datadict(),
                       list(names if names is not None else c.parnames), device=local_rank)

    model = make_model(case)
    theta_host = case.draw_theta(B, seed=1000 + rank)
    theta = torch.from_numpy(theta_host).cuda()
    lnl = torch.empty(B, dtype=torch.float64, device="cuda")
    sharded = ShardedLikelihood(lambda blk: model.log_likelihood_device(blk, out=lnl), case.ndim)
    fused, shared = None, None
    gather = "none" if world == 1 else "nccl all_gather"
    if world > 1 and args.gather != "nccl":
        try:  # all-gather fused into the producing kernel over NVLink symmetric memory
            from evidence_b200.multigpu import FusedGatherLikelihood
            sig = "flags" if args.gather == "fused" else "barrier"
            fused = FusedGatherLikelihood(model, B, signal=sig)
            gather = ("fused into the likelihood launch (peer stores over NVLink symmetric memory + "
                      + ("completion flags)" if sig == "flags" else "symmetric-memory barrier)"))
        except Exception as exc:  # symmetric memory unavailable: NCCL all-gather
            print(f"fused gather unavailable ({exc!r}); using NCCL all_gather", file=sys.stderr)
            fused = None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def step():
        return fused.evaluate_local(theta) if fused is not None else sharded.evaluate_local(theta)

    # ---- parity, device side: every rank evaluates the sets on its own GPU (through the C-ABI host
    # call), rank 0 compares with the CPU reference; the ranks must agree bit for bit
    parity, parity_ok, got = None, True, None
    if psets is not None:
        got = []
        vmodels = {"bench": model}
        for name, variant, th, _ in psets:
            if variant not in vmodels:
                vn, vf = variant_names(case, variant)
                vmodels[variant] = make_model(case, vn, vf)
            got.append(vmodels[variant].log_likelihood_batch(np.ascontiguousarray(th)))
        for v, m in vmodels.items():
            if v != "bench":
                m.close()
        if world > 1:
            mine = torch.from_numpy(np.concatenate(got)).cuda()
            allv = torch.empty(world * mine.numel(), dtype=torch.float64, device="cuda")
            dist.all_gather_into_tensor(allv, mine)
            ranks_agree = bool((allv.view(world, -1) == mine.unsqueeze(0)).all().item())
        else:
            ranks_agree = True

    # ---- gather check (N > 1): the fused all-gather's vector against NCCL's, same launch inputs
    gather_check = None
    if world > 1:
        local = model.log_likelihood_device(theta, out=lnl).clone()
        ref_all = torch.empty(world * B, dtype=torch.float64, device="cuda")
        dist.all_gather_into_tensor(ref_all, local)
        gather_check = {"n": world * B, "against": "torch.distributed.all_gather_into_tensor (NCCL) of "
                                                   "rvl_loglike_dev on the same theta"}
        if fused is not None:
            g1 = fused.evaluate_local(theta).clone()
            gather_check["device_call_equal"] = bool(torch.equal(g1, ref_all))
            if fused.signal == "flags":
                th_pin0 = torch.from_numpy(theta_host).pin_memory()
                out0 = torch.empty(world * B, dtype=torch.float64).pin_memory()
                fused.evaluate_local_host(th_pin0.numpy(), out0.numpy())
                gather_check["host_call_equal"] = bool(torch.equal(out0, ref_all.cpu()))
                if args.e2e_gather == "shared-host":
                    try:
                        from evidence_b200.multigpu import SharedHostGather
                        shared = SharedHostGather(model, B)
                        got_sh = shared.evaluate_local_host(th_pin0.numpy())
                        gather_check["shared_host_call_equal"] = bool(np.array_equal(got_sh, ref_all.cpu().numpy()))
                    except Exception as exc:  # shared memory / registration unavailable: device gather
                        print(f"shared-host gather unavailable ({exc!r}); using rvl_loglike_gather", file=sys.stderr)
                        shared = None
                del th_pin0, out0
        else:
            g1 = sharded.evaluate_local(theta)
            gather_check["device_call_equal"] = bool(torch.equal(g1, ref_all))
        flags = [float(all(v for k, v in gather_check.items() if k.endswith("_equal")))]
        t = torch.tensor(flags, dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        gather_check["pass"] = bool(t.item() == 1.0)
        del ref_all, g1, local

    # At N = 1 a step IS one launch of the likelihood kernel (the work list, the per-point
    # constants and the slice sums all live inside it), so the step's CUDA events time the kernel;
    # with an all-gather in the step the library records its own events around the kernel.
    inner_events = world > 1
    model.set_option("timing", 1 if inner_events else 0)
    for _ in range(W):
        step()
    ranks.barrier()
    peak = max(model.fp64_peak_tflops(), model.fp64_peak_tflops())  # after warm-up: clocks are up
    model.reset_counters()
    launches0 = model.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(K)]
    kms, wms = [], []
    clocks = ClockSampler(local_rank)
    ranks.barrier()
    t_wall = time.perf_counter()
    for k in range(K):
        flush.zero_()  # L2 flush, outside the per-step events
        ev[k][0].record()
        last = step()
        ev[k][1].record()
        if inner_events:
            kms.append(model.last_kernel_ms())
            if fused is not None and fused.signal == "flags":
                wms.append(model.last_gather_wait_ms())
    ranks.barrier()
    t_wall = time.perf_counter() - t_wall
    if args.dump_outputs and rank == 0:  # before the end-to-end calls re-use the buffers
        dump_outputs(args.dump_outputs, last.cpu().numpy())
    dev_ms = float(sum(a.elapsed_time(b) for a, b in ev))
    launches = model.launch_count() - launches0
    if not inner_events:
        if launches != K:
            raise SystemExit(f"expected one launch per step, counted {launches} in {K} steps")
        kms = [a.elapsed_time(b) for a, b in ev]
    cnt = model.counters()

    model.set_option("timing", 0)
    # ---- end to end: ONE public host-buffer call per step -- page-locked host theta read in place
    # by the kernel over PCIe, lnL (N > 1: the gathered vector of all ranks) back in host memory
    th_pin = torch.from_numpy(theta_host).pin_memory()
    out_all_pin = torch.empty(B * world, dtype=torch.float64).pin_memory()
    th_np, out_np = th_pin.numpy(), out_all_pin.numpy()
    host_gather = fused is not None and fused.signal == "flags"
    shared_out = [None]

    def e2e_step():
        if world == 1:
            model.log_likelihood_batch(th_np, out=out_np)  # rvl_loglike
        elif shared is not None:
            shared_out[0] = shared.evaluate_local_host(th_np)  # rvl_loglike_scatter_host + host flags
        elif host_gather:
            fused.evaluate_local_host(th_np, out_np)       # rvl_loglike_gather
        else:  # NCCL fallback: H2D, kernel, all-gather, D2H of the gathered vector
            theta.copy_(th_pin, non_blocking=True)
            gathered = sharded.evaluate_local(theta)
            out_all_pin.copy_(gathered, non_blocking=True)
            torch.cuda.synchronize()

    for _ in range(W):
        e2e_step()
    ranks.barrier()
    # a full collection of the interpreter's heap (torch, numpy, ... imported) takes ~45 ms and
    # would land inside this wall-clock region: collect now, keep the collector off while timing
    gc.collect()
    gc.disable()
    t0 = time.perf_counter()
    marks = [t0]
    for k in range(K):
        e2e_step()
        marks.append(time.perf_counter())
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    gc.enable()
    e2e_ms = np.diff(np.array(marks)) * 1e3  # per call (every call ends with a stream sync)
    clk = clocks.stop()  # the sampler covers both timed regions
    res_np = shared_out[0] if shared_out[0] is not None else out_np
    e2e_equal = (bool(np.array_equal(res_np[rank * B:(rank + 1) * B], lnl.cpu().numpy()))
                 if world == 1 or host_gather or shared is not None else None)

    dev_ms, e2e_s = ranks.max(dev_ms, e2e_s)

    mean_it = cnt["n_newton_iters"] / max(1, cnt["n_solves"])
    F = algorithmic_flops(case.n_epochs, case.n_planets, case.drift, mean_it)
    k_ms = float(np.mean(kms))
    traffic = None  # DRAM bytes per launch from the committed `ncu --set full` capture (profiles/)
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = f"config{CONFIG_ID}_B{B}"
        if key in prof:
            traffic = prof[key]["dram_bytes_per_launch"]
    except (OSError, ValueError, KeyError):
        pass
    achieved = B * F / (k_ms * 1e-3) / 1e12
    value = world * B * K / (dev_ms * 1e-3)
    h2d = int(B * case.ndim * 8)
    d2h = int(B * 8) if shared is not None else int(B * world * 8)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(case, B, world),
        "gather": gather,
        "clocks": clk,
        "e2e": {"value": world * B * K / e2e_s, "unit": UNIT,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": ("rvl_loglike (page-locked theta read in place, lnL written in place)" if world == 1 else
                        "rvl_loglike_scatter_host + rvl_wait_host_flags, per rank and step (page-locked theta read in "
                        "place; every rank's kernel stores its lnL block into a host segment shared by the ranks)"
                        if shared is not None else
                        "rvl_loglike_gather, one call per rank and step (page-locked theta read in place; gathered "
                        "lnL of all ranks copied to host memory)" if host_gather else
                        "torch copies around rvl_loglike_dev + NCCL all_gather"),
                "ms_per_call_percentiles_1_50_99": [float(x) for x in np.percentile(e2e_ms, [1, 50, 99])],
                "result_equals_device_path": e2e_equal},
        "gpu_launches": int(launches),
        "roofline": {"bound": "fp64", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                     "frac": achieved / peak if peak else None, "traffic": traffic,
                     "kernel": "rv_lnl_kernel", "kernel_ms": k_ms,
                     "kernel_ms_source": ("library CUDA events around the kernel" if inner_events else
                                          "the step's CUDA events (one launch per step)"),
                     "flops_per_lnl": F, "mean_newton_iters": mean_it,
                     "peak_source": "DFMA loop measured in this run (rvl_fp64_peak); "
                                    "MEASURED_PEAKS.json has no FP64 row",
                     "peak_nominal": 148 * 64 * 2 * 1.965e9 / 1e12,
                     "hbm_bytes_per_lnl": 8 * (case.ndim + 1)},
        "wall_s_timed_region": t_wall,
        "kepler_solves_per_s": value * case.n_epochs * case.n_planets,
        "newton_cap_hits": cnt["n_cap_hits"],
    }
    if gather_check is not None:
        line["gather_check"] = gather_check
    if wms:  # what the exchange costs beyond the rank's own kernel (CUDA events around the wait)
        (wmax,) = ranks.max(float(np.mean(wms)))
        line["gather_cost"] = {"wait_after_kernel_ms_mean_rank0": float(np.mean(wms)),
                               "wait_after_kernel_ms_mean_max_over_ranks": wmax,
                               "nvlink_bytes_per_step_per_rank": int(8 * B * (world - 1)),
                               "note": "time between the end of this rank's likelihood kernel and the arrival of "
                                       "the last peer's completion flag: rank skew + NVLink latency"}

    # ---- parity verdict (the CPU side has been running since the start)
    if psets is not None:
        if rank == 0:
            res = want_async.get()
            want = [np.concatenate([r for r, o in zip(res, owner) if o == si]) for si in range(len(psets))]
            def classify(row):
                """Newton-cap events of one theta row: (device counter, C-port counter)."""
                from evidence_b200.layout import compile_model
                from oracle import rv_oracle
                model.reset_counters()
                model.log_likelihood(row)
                dev = model.counters()["n_cap_hits"]
                t_, v_, s_, ids_ = case.arrays()
                desc, _ = compile_model(case.parnames, case.fixedpardict, case.insts, t_[0])
                _, _, ref = rv_oracle.c_loglike_batch(bytes(desc), t_, v_, s_, ids_, case.n_inst, row[None, :])
                return dev, ref

            parity, parity_ok = parity_verdict(psets, got, want, kind, classify)
            parity["ranks_bit_identical"] = ranks_agree
            parity["checker_text"] = kind_text(kind)
            parity_ok = parity_ok and ranks_agree
            line["parity"] = parity

    if not args.no_extras:
        try:
            line["sweep_total_points"] = sweep_sizes(model, case, rank, world, ranks, torch, peak)
            line["latency_ndraw4096"] = latency_line(make_model, rank, world, ranks, torch, peak, args.gather)
            line["stress"] = stress(make_model, rank, world, ranks, torch, peak)
        except Exception as exc:  # extras must never cost the headline line
            line["extras_error"] = repr(exc)
            if world > 1:
                raise
    if rank == 0 and world == 1 and not args.no_extras and pool is not None:
        try:
            key = (CONFIG_ID, "bench")
            rate, n, dt = pool_rate(pool, cores, key, theta_host[:8192], 12.0)
            line["cpu_baseline"] = {
                "value": rate, "unit": UNIT, "cores": cores, "kind": kind,
                "sample": f"{n} lnL evaluations (rows of the step's {B}-theta batch), {dt:.1f} s on {cores} processes; "
                          + kind_text(kind)}
        except Exception as exc:
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": kind,
                                    "sample": "failed: " + repr(exc)}
    if pool is not None:
        pool.terminate()
    if shared is not None:
        shared.close()
    if rank == 0:
        emit(line)
    model.close()
    failed = (not parity_ok) or (gather_check is not None and not gather_check.get("pass", True))
    if world > 1:
        t = torch.tensor([1.0 if failed else 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        failed = bool(t.item() > 0)
        dist.destroy_process_group()
    if failed:
        print("bench.py: parity / gather check FAILED (see the JSON line)", file=sys.stderr)
        sys.exit(3)


if __name__ == "__main__":
    main()
