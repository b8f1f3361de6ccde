"""
Rate of the model velocity curves (rvl_kepler_rv_dev) against the likelihood kernel on the same theta.

Config 3 (N = 5000 epochs, K = 4 planets), B = 16 384 prior draws: curves at the 5000 data times and
on a 4096-point grid, device form, CUDA events around >= 1 s of back-to-back calls after warm-up.
Reports Kepler solves/s, the share of the in-run FP64 peak (rvl_fp64_peak) with the per-solve flop
count K (51 + 46 I) of DESIGN.md section 5 (I = mean Newton iterations, from the likelihood's counter
on the same theta), the likelihood kernel's solves/s at the data times, the prepare pass alone (a
call with T = 0), and the oracle's kep_rv on one host core for scale.  The card's name and power
limit are read in the same run.

    python tests/diag/kepler_rv_bench.py [--B 16384] [--seconds 1.0]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def timed(fn, seconds):
    """ms per call of fn (enqueue on the current stream), CUDA events, >= `seconds` of calls."""
    import torch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    reps = max(5, int(np.ceil(seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3))))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=16384)
    ap.add_argument("--grid", type=int, default=4096)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--cpu-rows", type=int, default=4)
    args = ap.parse_args()
    import torch
    from evidence_b200 import _abi, synth
    from evidence_b200.rvmodel import RVModel
    from oracle.rv_oracle import OracleRVModel

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(f"card: {smi.splitlines()[0] if smi else 'unknown'}")
    print(f"library: {_abi.LIB_PATH}")
    case = synth.make_case(3)
    m = RVModel(case.fixedpardict, case.datadict(), case.parnames, device=0)
    B, K = args.B, m.nplanets
    theta_h = case.draw_theta(B, seed=77)
    theta = torch.from_numpy(theta_h).cuda()
    t_data = torch.from_numpy(m.time).cuda()
    t_grid = torch.linspace(float(m.time.min()) - 200.0, float(m.time.max()) + 200.0, args.grid,
                            dtype=torch.float64, device="cuda")
    peak = m.fp64_peak_tflops()
    print(f"rvl_fp64_peak: {peak:.2f} TFLOP/s (in-run)")

    # the likelihood on the same theta: its Newton iteration count and its rate
    m.reset_counters()
    m.log_likelihood_batch(theta_h)
    c = m.counters()
    I = c["n_newton_iters"] / c["n_solves"]
    lnl_out = torch.empty(B, dtype=torch.float64, device="cuda")
    ms_l, reps = timed(lambda: m.log_likelihood_device(theta, out=lnl_out), args.seconds)
    sol_l = B * len(m.time) * K / (ms_l * 1e-3)
    flop = 51 + 46 * I
    print(f"config 3, B = {B}, K = {K}, N = {len(m.time)}; mean Newton iterations I = {I:.3f}, "
          f"{flop:.1f} flop per solve")
    print(f"rv_lnl_kernel (data times)   : {ms_l:8.3f} ms/call ({reps} calls)  "
          f"{sol_l:.3e} solves/s  {sol_l * flop / (peak * 1e12):.3f} of the FP64 peak")

    results = {}
    for label, tt in (("data times", t_data), ("grid", t_grid)):
        T = tt.shape[0]
        out = torch.empty((B, T), dtype=torch.float64, device="cuda")
        ms, reps = timed(lambda: m.kepler_rv_device(theta, tt, out=out), args.seconds)
        sol = B * T * K / (ms * 1e-3)
        results[label] = sol
        print(f"kepler_rv {label:<11} T={T:5d}: {ms:8.3f} ms/call ({reps} calls)  {sol:.3e} solves/s  "
              f"{sol * flop / (peak * 1e12):.3f} of the FP64 peak  {sol / sol_l:.3f} x the likelihood")
    # the prepare pass alone: a call with no times derives the constants and writes the invalid bits
    empty = torch.zeros(0, dtype=torch.float64, device="cuda")
    ms_p, reps = timed(lambda: m.kepler_rv_device(theta, empty), min(args.seconds, 0.3))
    print(f"prepare pass (T = 0 call)    : {ms_p * 1e3:8.1f} us/call ({reps} calls)")
    # the same rows' curves agree at the data times with the likelihood-path residuals
    rv_dev, ok = m.kepler_rv_device(theta[:64], t_data)
    rv_host, ok_h = m.kepler_rv_batch(theta_h[:64], m.time)
    assert np.array_equal(rv_dev.cpu().numpy(), rv_host) and bool(ok.all())

    om = OracleRVModel(case.fixedpardict, case.datadict(), case.parnames)
    rows = theta_h[:args.cpu_rows]
    t0 = time.perf_counter()
    want = [om.kep_rv(dict(dict(zip(m.parnames, r)), **case.fixedpardict), om.time) for r in rows]
    dt = time.perf_counter() - t0
    sol_c = len(rows) * len(om.time) * K / dt
    err = max(float(np.max(np.abs(rv_host[i] - w))) for i, w in enumerate(want))
    print(f"oracle kep_rv, one host core : {dt / len(rows) * 1e3:8.1f} ms/row ({len(rows)} rows)  "
          f"{sol_c:.3e} solves/s ({1e9 / sol_c:.0f} ns/solve); device / host = {results['data times'] / sol_c:.0f}x; "
          f"max |dv| on those rows {err:.2e}")
    m.close()


if __name__ == "__main__":
    main()
