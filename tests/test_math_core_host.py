"""
CPU tests of the likelihood kernel's FP64 core (evidence_b200/csrc/rvl_math.h) one operation at a
time, through the host build of the device probe (tests/device_probe/ops.h), against mpmath:
  * the five step series advance_{final,tiny,small,mid,medium} over the whole range of steps each is
    used for, and chains of up to 12 steps as a Newton solve takes them;
  * newton_step, kepler_rv2 and log_mantissa (through rvl::rcp);
  * split_pos / split_raw against np.frexp and on every value the log-determinant must flag;
  * mean_anomaly bit for bit against numpy (an FMA-formed M breaks parity with the reference).
Also: the probe cross-compiles for sm_100a with the library's flags, and the sin/cos path
thresholds of the lean loop are defined once (evidence_b200/csrc/rvl_lean.h).
tests/test_gpu_math_core.py runs the same operations on the device.
"""
import glob
import os
import re
import subprocess

import numpy as np
import pytest

from _mp import sincos_dd, sincos_err
from _probe import (ADVANCE_RANGE, angles, build_device_probe, chain_args, chain_total, check_kepler_rv2,
                    check_log_mantissa, check_newton_step, host_probe, log_mantissa_args,
                    mean_anomaly_args, split_args, steps)
from _util import ROOT

assert host_probe  # a fixture

SINCOS_BAR = 2.3e-16  # about one ulp of 1, as for sincos_fast (test_host_emul.py)
HALF_ULP_1 = 2.0**-53


def _start(rng, n):
    """E and its correctly rounded (sin E, cos E)."""
    E = angles(rng, n)
    ref = sincos_dd(E)
    return E, ref[:, 0].copy(), ref[:, 1].copy()


@pytest.mark.parametrize("op", list(ADVANCE_RANGE))
def test_advance_series_vs_mpmath(host_probe, op):
    rng = np.random.default_rng(list(ADVANCE_RANGE).index(op) + 11)
    n = 20000
    E, s, c = _start(rng, n)
    d = steps(rng, n, ADVANCE_RANGE[op])
    out = host_probe(op, s, c, d)
    err = sincos_err(out[:, 0], out[:, 1], sincos_dd(E, d))
    big = np.abs(d) >= ADVANCE_RANGE[op] / 2
    print(f"{op}: |d| < {ADVANCE_RANGE[op]:.4g}: max error {err.max():.3g} "
          f"(upper half of the range {err[big].max():.3g})")
    assert err.max() <= SINCOS_BAR, (op, float(err.max()), float(d[np.argmax(err)]))


def test_chains_of_steps_vs_mpmath(host_probe):
    """k = 1..12 steps with the series the loop picks for each: the error grows by at most half an
    ulp per step beyond the first."""
    rng = np.random.default_rng(23)
    n = 12000
    E, s, c = _start(rng, n)
    d0, q, k = chain_args(rng, n)
    out = host_probe("chain", s, c, d0, q, k)
    from mpmath.libmp import from_float, mpf_add, mpf_cos_sin, mpf_sub, round_nearest, to_float
    err = np.empty(n)
    for i, tot in enumerate(chain_total(d0, q, k)):
        cc, ss = mpf_cos_sin(mpf_add(from_float(float(E[i])), tot, 2200, round_nearest), 120, round_nearest)
        err[i] = max(abs(to_float(mpf_sub(from_float(float(out[i, 0])), ss, 120))),
                     abs(to_float(mpf_sub(from_float(float(out[i, 1])), cc, 120))))
    bar = SINCOS_BAR + (k - 1) * HALF_ULP_1
    worst = {int(j): float(err[k == j].max()) for j in range(1, 13)}
    print("max error after k steps:", {j: f"{v:.3g}" for j, v in worst.items()})
    assert np.all(err <= bar), [(j, v) for j, v in worst.items() if v > SINCOS_BAR + (j - 1) * HALF_ULP_1]


def test_newton_step(host_probe):
    worst = check_newton_step(host_probe, np.random.default_rng(31), 20000)
    print(f"newton_step: max error / bar {worst:.3f}")


def test_kepler_rv2(host_probe):
    worst = check_kepler_rv2(host_probe, np.random.default_rng(37), 20000)
    print(f"kepler_rv2: max error {worst:.3f} ulp of the result scale")


def test_log_mantissa(host_probe):
    worst = check_log_mantissa(host_probe, log_mantissa_args(np.random.default_rng(41), 50000))
    print(f"log_mantissa: max error {worst:.3f} ulp")


def test_split_pos_and_split_raw(host_probe):
    good, bad = split_args(np.random.default_rng(43))
    fm, fe = np.frexp(good)
    p = host_probe("split_pos", good)
    r = host_probe("split_raw", good)
    assert np.array_equal(p[:, 0], 2 * fm) and np.array_equal(p[:, 1], fe - 1) and np.all(p[:, 2] == 1.0)
    assert np.array_equal(r[:, 0], 2 * fm) and np.array_equal(r[:, 1], fe - 1 + 1023)
    assert np.all((r[:, 1].astype(np.int64) - 1) % 2**32 < 0x7FE)
    p = host_probe("split_pos", bad)
    r = host_probe("split_raw", bad)
    assert np.all(p[:, 2] == 0.0)
    # item_epochs keeps the unsigned maximum of be - 1: at least 0x7fe exactly when a term is bad
    assert np.all((r[:, 1].astype(np.int64) - 1) % 2**32 >= 0x7FE)


def test_mean_anomaly_is_numpys(host_probe):
    nmot, t, epoch, m0 = mean_anomaly_args(np.random.default_rng(47), 200000)
    got = host_probe("mean_anomaly", nmot, t, epoch, m0)[:, 0]
    assert np.array_equal(got, nmot * (t - epoch) + m0)


def test_probe_cross_compiles(tmp_path):
    so = build_device_probe(tmp_path)
    res = subprocess.run([os.path.join(os.path.dirname(_nvcc()), "cuobjdump"), "--list-elf", so],
                         capture_output=True, text=True, check=True)
    assert "sm_100a" in res.stdout, res.stdout


def _nvcc():
    from evidence_b200 import build
    return build.nvcc_path()


def test_path_thresholds_have_one_home():
    """The thresholds that pick the sin/cos path of a pass are defined in rvl_lean.h alone: no source
    of the library or of its host replays and probe keeps a copy of their values."""
    values = re.compile(r"0x(40F86A00|3F500000|3FA00000|3FC00000|3FE80000)\b", re.I)
    names = re.compile(r"\bkHi(TrigMax|Tiny|Small|Mid|Medium)\s*=")
    home = os.path.join(ROOT, "evidence_b200", "csrc", "rvl_lean.h")
    files = [f for pat in ("evidence_b200/csrc/*", "tests/host_emul/*.cpp", "tests/device_probe/*", "tools/*.cu")
             for f in glob.glob(os.path.join(ROOT, pat))]
    assert home in files
    found = []
    for f in files:
        with open(f) as fh:
            text = fh.read()
        if values.search(text) or names.search(text):
            found.append(os.path.relpath(f, ROOT))
    assert found == ["evidence_b200/csrc/rvl_lean.h"], found
