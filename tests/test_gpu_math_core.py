"""
GPU tests of the likelihood kernel's FP64 core (evidence_b200/csrc/rvl_math.h) one operation at a
time: the device probe (tests/device_probe/probe.cu, built with the library's nvcc flags) runs each
operation as the kernel calls it -- coefficients through rvl::load_ktab() and through
rvl::load_ktab_pinned(), which must agree bit for bit, and table rows read from shared memory
through rvl::SmemSinTab.
  * Every operation that does not go through the reciprocal seed gives the same bits as the host
    build of the same source, which tests/test_math_core_host.py, test_sintab.py and
    test_host_emul.py check against mpmath: sincos_tab and sincos_fast on 1.1e6 arguments, the five
    step series, chains of steps, exp_cr, split_pos / split_raw and mean_anomaly.
  * The arithmetic that only the device has -- the MUFU.RCP64H seed (rcp.approx.ftz.f64) and what
    is built on it: rcp, newton_step, kepler_rv2, log_mantissa -- against mpmath, and exp_cr
    against the nearest double.
Run with -s to see the measured errors.
"""
import numpy as np
import pytest

from _mp import sincos_args
from _probe import (ADVANCE_RANGE, DeviceProbe, angles, build_device_probe, chain_args,
                    check_kepler_rv2, check_log_mantissa, check_newton_step, check_rcp, exp_args,
                    exp_nearest, first_diffs, host_probe, log_mantissa_args, mean_anomaly_args,
                    rcp_args, split_args, steps)

pytestmark = pytest.mark.gpu
assert host_probe  # a fixture

N = 200000


@pytest.fixture(scope="module")
def dev(tmp_path_factory):
    return DeviceProbe(build_device_probe(tmp_path_factory.mktemp("probe_dev")))


def _bit_sets():
    """(op, argument columns) of every operation whose device and host builds must agree bit for bit."""
    rng = np.random.default_rng(101)
    x = sincos_args()
    yield "sincos_tab", (x,)
    yield "sincos_fast", (x,)
    for op, bound in ADVANCE_RANGE.items():
        E = angles(rng, N)
        yield op, (np.sin(E), np.cos(E), steps(rng, N, bound))
    E = angles(rng, N)
    yield "chain", (np.sin(E), np.cos(E)) + chain_args(rng, N)
    yield "exp_cr", (np.concatenate([exp_args(), rng.uniform(-700.0, 700.0, N)]),)
    good, bad = split_args(rng)
    yield "split_pos", (np.concatenate([good, bad]),)
    yield "split_raw", (np.concatenate([good, bad]),)
    yield "mean_anomaly", mean_anomaly_args(rng, N)


def test_bit_identical_to_host_build(dev, host_probe):
    report = {}
    for op, args in _bit_sets():
        got, want = dev(op, *args), host_probe(op, *args)
        nbad, first = first_diffs(got, want, args)
        report[op] = len(args[0])
        assert nbad == 0, (op, f"{nbad} of {len(args[0])} differ from the host build", first)
    print("bit-identical to the host build, with both coefficient loaders (arguments):", report)


def test_reciprocal_seed_and_refinement(dev):
    from mpmath import libmp as lm
    x1, x2 = rcp_args(np.random.default_rng(103), N)
    x = np.concatenate([x1, x2])
    y0 = dev("rcp_seed", x)[:, 0]
    rel = np.array([abs(lm.to_float(lm.mpf_sub(lm.mpf_mul(lm.from_float(a), lm.from_float(b)), lm.fone, 400)))
                    for a, b in zip(x.tolist(), y0.tolist())])
    print(f"rcp_seed: max |1 - x y0| = {rel.max():.3g} = 2^{np.log2(rel.max()):.2f}")
    assert rel.max() <= 2.0**-19
    for name, xs in (("[0.01, 2]", x1), ("[1e-30, 1e30]", x2)):
        worst, off = check_rcp(dev, xs)
        print(f"rcp over {name}: max error {worst:.3f} ulp, {100 * off:.2f} % not correctly rounded")
        assert worst <= 1.0, (name, worst)


def test_newton_step(dev):
    worst = check_newton_step(dev, np.random.default_rng(107), N)
    print(f"newton_step: max error / bar {worst:.3f}")


def test_kepler_rv2(dev):
    worst = check_kepler_rv2(dev, np.random.default_rng(109), N)
    print(f"kepler_rv2: max error {worst:.3f} ulp of the result scale")


def test_log_mantissa(dev):
    worst = check_log_mantissa(dev, log_mantissa_args(np.random.default_rng(113), N))
    print(f"log_mantissa: max error {worst:.3f} ulp")


def test_exp_cr_is_correctly_rounded(dev):
    x = exp_args()
    y = dev("exp_cr", x)[:, 0]
    want = exp_nearest(x)
    bad = np.nonzero(y != want)[0]
    print(f"exp_cr: {len(bad)} of {len(x)} not the nearest double (|x| up to {np.abs(x).max()!r})")
    assert len(bad) == 0, [(float(x[i]), float(y[i]), float(want[i])) for i in bad[:5]]
