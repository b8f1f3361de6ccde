"""The FP64 core of the likelihood kernel one operation at a time (tests/device_probe): builds of the
probe for the device and the host, argument sets, and the checks against mpmath that both
tests/test_math_core_host.py and tests/test_gpu_math_core.py apply."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from _util import ROOT

PROBE_DIR = os.path.join(ROOT, "tests", "device_probe")
K_IN, K_OUT = 8, 4
# the Op enum of ops.h, in order
OPS = ["sincos_tab", "sincos_fast", "advance_final", "advance_tiny", "advance_small", "advance_mid",
       "advance_medium", "chain", "rcp_seed", "rcp", "newton_step", "kepler_rv2", "log_mantissa",
       "exp_cr", "split_pos", "split_raw", "mean_anomaly"]
OP = {name: i for i, name in enumerate(OPS)}

# each advance series and the sizes of step it is used for (|d| < bound; the final series is the one
# of the reference tolerance: valid below 2e-4)
ADVANCE_RANGE = {"advance_final": 2e-4, "advance_tiny": 2.0**-10, "advance_small": 2.0**-5,
                 "advance_mid": 2.0**-3, "advance_medium": 0.75}

dp = ctypes.POINTER(ctypes.c_double)


def build_device_probe(outdir):
    """nvcc with the library's own flags (sm_100a, -fmad=false): the probe compiles as the kernel does."""
    from evidence_b200 import build
    so = os.path.join(str(outdir), "libprobe_dev.so")
    cmd = [build.nvcc_path()] + build.NVCC_FLAGS + ["-o", so, os.path.join(PROBE_DIR, "probe.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, " ".join(cmd) + "\n" + res.stdout + res.stderr
    return so


def build_host_probe(outdir):
    """g++ with contraction off, as tests/host_emul is built."""
    so = os.path.join(str(outdir), "libprobe_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so,
                    os.path.join(PROBE_DIR, "host.cpp"), "-lm"], check=True)
    return so


def _pack(args):
    a = np.zeros((len(args[0]), K_IN))
    for k, col in enumerate(args):
        a[:, k] = col
    return np.ascontiguousarray(a)


class HostProbe:
    def __init__(self, so):
        self.lib = ctypes.CDLL(so)

    def __call__(self, op, *args):
        a = _pack(args)
        out = np.empty((len(a), K_OUT))
        rc = self.lib.host_run(OP[op], a.ctypes.data_as(dp), out.ctypes.data_as(dp), ctypes.c_longlong(len(a)))
        assert rc == 0, op
        return out


class DeviceProbe:
    """Runs an operation with both coefficient loaders (rvl::load_ktab, rvl::load_ktab_pinned),
    checks that they give the same bits and returns the result."""

    def __init__(self, so):
        self.lib = ctypes.CDLL(so)

    def run(self, op, pinned, *args):
        a = _pack(args)
        out = np.empty((len(a), K_OUT))
        rc = self.lib.probe_run(OP[op], int(pinned), a.ctypes.data_as(dp), out.ctypes.data_as(dp),
                                ctypes.c_longlong(len(a)))
        assert rc == 0, f"probe_run({op}): CUDA error {rc}"
        return out

    def __call__(self, op, *args):
        plain, pinned = self.run(op, 0, *args), self.run(op, 1, *args)
        assert bits_equal(plain, pinned), (op, "load_ktab and load_ktab_pinned differ")
        return plain


@pytest.fixture(scope="module")
def host_probe(tmp_path_factory):
    return HostProbe(build_host_probe(tmp_path_factory.mktemp("probe_host")))


def bits_equal(a, b):
    return np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))


def first_diffs(a, b, args, n=5):
    bad = np.nonzero((np.asarray(a).view(np.uint64) != np.asarray(b).view(np.uint64)).any(axis=1))[0]
    return len(bad), [(tuple(float(v[i]) for v in args), a[i].tolist(), b[i].tolist()) for i in bad[:n]]


# ---- argument sets ------------------------------------------------------------------------------

def angles(rng, n):
    """E for the advance tests: half over the loop's whole range, half in [-7, 7]."""
    return np.concatenate([rng.uniform(-1e5, 1e5, n - n // 2), rng.uniform(-7.0, 7.0, n // 2)])


def steps(rng, n, bound):
    """d over (-bound, bound): uniform, log-uniform in size down to 1e-3 of the bound, and the
    edges: one ulp below the bound (the largest step the series is used for), 0, +-tiny."""
    edge = np.nextafter(bound, 0.0)
    special = np.array([edge, -edge, np.nextafter(edge, 0.0), -np.nextafter(edge, 0.0), 0.0, -0.0,
                        1e-300, -1e-300, bound / 2, -bound / 2])
    m = n - len(special)
    sign = np.where(rng.random(m - m // 2) < 0.5, -1.0, 1.0)
    logu = sign * bound * 10.0 ** rng.uniform(-3.0, 0.0, m - m // 2)
    d = np.concatenate([rng.uniform(-bound, bound, m // 2), logu, special])
    return np.clip(d, -edge, edge)


def chain_args(rng, n):
    """Geometrically shrinking steps, as a Newton solve takes them: d0 = first step, q = ratio of
    successive steps, k = 1..12 steps (the reference stops at a step <= 1e-4)."""
    d0 = np.where(rng.random(n) < 0.5, -1.0, 1.0) * 10.0 ** rng.uniform(-4.0, np.log10(0.7), n)
    q = 10.0 ** rng.uniform(-3.0, np.log10(0.6), n) * np.where(rng.random(n) < 0.2, -1.0, 1.0)
    k = rng.integers(1, 13, n).astype(np.float64)
    return d0, q, k


def chain_total(d0, q, k):
    """The steps of the chain op, d_(i+1) = d_i q rounded as the op rounds them, and their sum taken
    exactly (as a list of mpmath values)."""
    from mpmath.libmp import fzero, from_float, mpf_add, round_nearest
    total = []
    for a, b, m in zip(d0.tolist(), q.tolist(), k.astype(int).tolist()):
        t, d = fzero, a
        for _ in range(m):
            t = mpf_add(t, from_float(d), 2200, round_nearest)
            d = float(np.float64(d) * np.float64(b))
        total.append(t)
    return total


def rcp_args(rng, n):
    """The two uses of rvl::rcp: Newton denominators 1 - e cos E in [0.01, 2] and variances."""
    x1 = np.concatenate([rng.uniform(0.01, 2.0, n // 2 - 6), [0.01, 2.0, 1.0, np.nextafter(1.0, 0), 0.5, 1.5]])
    x2 = 10.0 ** rng.uniform(-30.0, 30.0, n - n // 2)
    return x1, x2


def split_args(rng):
    """(positive normal values, values the split must flag)."""
    tiny_n = np.finfo(np.float64).tiny
    good = np.concatenate([
        rng.uniform(1.0, 2.0, 20000) * np.ldexp(1.0, rng.integers(-1022, 1024, 20000)),
        rng.uniform(1e-6, 1e6, 20000),
        [tiny_n, np.nextafter(tiny_n, 1.0), np.finfo(np.float64).max, 1.0, np.nextafter(1.0, 2.0),
         np.nextafter(2.0, 1.0), 2.0, 0.5],
    ])
    sub = rng.uniform(0.0, 1.0, 2000) * tiny_n
    bad = np.concatenate([
        sub[sub > 0], -sub[sub > 0], [5e-324, np.nextafter(tiny_n, 0.0), -5e-324],
        [0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan, -tiny_n, -1.0, -np.finfo(np.float64).max],
        -good[:5000],
        np.array([0x7FF0000000000001, 0x7FF8000000000000, 0xFFF8000000000001], dtype=np.uint64).view(np.float64),
    ])
    return np.ascontiguousarray(good), np.ascontiguousarray(bad)


def mean_anomaly_args(rng, n):
    """nmot = 2 pi / P, epoch times, epochs of the elements, M0 as the models meet them."""
    nmot = 2 * np.pi / (10.0 ** rng.uniform(-0.5, 4.5, n))
    t = rng.uniform(-2e4, 2e4, n)
    epoch = np.where(rng.random(n) < 0.5, 0.0, rng.uniform(-1e4, 1e4, n))
    m0 = rng.uniform(-np.pi, 2 * np.pi, n)
    return nmot, t, epoch, m0


def exp_args():
    """test_host_emul.py::test_exp_cr_is_correctly_rounded's arguments and the ends of the range
    exp_cr computes itself (|x| < 700; beyond that it calls the library)."""
    rng = np.random.default_rng(1)
    x = np.concatenate([rng.uniform(-10, 10, 12000), rng.uniform(-690, 690, 4000),
                        rng.uniform(-1e-3, 1e-3, 1000), [0.0, 1.0, -1.0, 0.5 * np.log(2), 699.9, -699.9]])
    edge = [700.0]
    for _ in range(64):
        edge.append(np.nextafter(edge[-1], 0.0))
    edge = np.array(edge[1:])
    return np.ascontiguousarray(np.concatenate([x, edge, -edge, rng.uniform(699.0, 700.0, 500) * np.array([1, -1] * 250)]))


# ---- checks against mpmath ----------------------------------------------------------------------

def _exact():
    from mpmath import libmp
    return libmp


def check_rcp(run, x):
    """rvl::rcp within one ulp of 1/x; returns (max error in ulp, share not correctly rounded)."""
    lm = _exact()
    y = run("rcp", x)[:, 0]
    # x y - 1 exactly (the product of two doubles has 106 bits)
    res = np.array([lm.to_float(lm.mpf_sub(lm.mpf_mul(lm.from_float(a), lm.from_float(b)), lm.fone, 400))
                    for a, b in zip(x.tolist(), y.tolist())])
    err_ulp = np.abs(res) * y / np.spacing(y)  # |y - 1/x| = |x y - 1| / x, 1/x = y (1 + 2^-52)
    off = float(np.mean(y != 1.0 / x))  # numpy's division is correctly rounded
    return float(err_ulp.max()), off


def check_newton_step(run, rng, n):
    """rvl::newton_step: d = E_new - E exactly, and E_new within half an ulp of E plus the reference's
    update E - f/f' (f formed as the kernel forms it) by no more than 2 ulp of f/f'; returns the
    largest error over its bar."""
    lm = _exact()
    rn = lm.round_nearest
    ec = np.concatenate([rng.uniform(0.0, 0.99, n // 2), 0.99 - rng.uniform(0, 1e-3, n - n // 2)])
    M = np.concatenate([rng.uniform(-1e4, 1e4, n // 2), rng.uniform(-7.0, 7.0, n - n // 2)])
    E = M + rng.uniform(-1.0, 1.0, n) * 10.0 ** rng.uniform(-12, 0, n)
    s, c = np.sin(E), np.cos(E)
    out = run("newton_step", E, s, c, M, ec)
    En, d = out[:, 0], out[:, 1]
    assert np.array_equal(d, En - E), "d is not E_new - E"
    # f = RN(RN(E - ec s) - M) (E - ec s with one rounding: RVL_FMA_F), f' = 1 - ec c exactly
    f = np.array([lm.to_float(lm.mpf_sub(lm.from_float(e), lm.mpf_mul(lm.from_float(a), lm.from_float(b)), 53, rn))
                  for e, a, b in zip(E.tolist(), ec.tolist(), s.tolist())]) - M
    ref, q = [], []
    for e, fv, a, b in zip(E.tolist(), f.tolist(), ec.tolist(), c.tolist()):
        fp = lm.mpf_sub(lm.fone, lm.mpf_mul(lm.from_float(a), lm.from_float(b)), 400)
        qq = lm.mpf_div(lm.from_float(fv), fp, 400)
        q.append(abs(lm.to_float(qq)))
        ref.append(lm.mpf_sub(lm.from_float(e), qq, 400))
    err = np.array([abs(lm.to_float(lm.mpf_sub(lm.from_float(g), r, 400))) for g, r in zip(En.tolist(), ref)])
    bar = 0.5 * np.spacing(np.abs(En)) + 4.5e-16 * np.array(q)
    worst = float(np.max(err / bar))
    assert worst <= 1.0, worst
    return worst


def check_kepler_rv2(run, rng, n):
    """rvl::kepler_rv2 against (A c - A ec + Bs s) / (1 - ec c) + Ce from the same doubles, e up to
    0.99 and c near 1 (the denominator near 0.01); returns the max error in ulp of the result scale."""
    lm = _exact()
    e = np.concatenate([rng.uniform(0.0, 0.99, n // 2), 0.99 - rng.uniform(0, 1e-3, n - n // 2)])
    E = np.concatenate([rng.uniform(-7.0, 7.0, n // 2), rng.uniform(-0.05, 0.05, n - n // 2)])
    s, c = np.sin(E), np.cos(E)
    K = 10.0 ** rng.uniform(-1.0, 3.0, n)
    w = rng.uniform(0.0, 2 * np.pi, n)
    A = K * np.cos(w)
    Bs = -K * np.sin(w) * np.sqrt(1 - e * e)
    Ce = K * (e * np.cos(w))
    mAec = -(A * e)
    rv = run("kepler_rv2", s, c, e, A, Bs, Ce, mAec)[:, 0]
    F = lm.from_float
    err = np.empty(n)
    for i in range(n):
        num = lm.mpf_add(lm.mpf_add(lm.mpf_mul(F(A[i]), F(c[i])), F(mAec[i]), 400),
                         lm.mpf_mul(F(Bs[i]), F(s[i])), 400)
        den = lm.mpf_sub(lm.fone, lm.mpf_mul(F(e[i]), F(c[i])), 400)
        want = lm.mpf_add(lm.mpf_div(num, den, 400), F(Ce[i]), 400)
        err[i] = abs(lm.to_float(lm.mpf_sub(F(rv[i]), want, 400)))
    scale = (np.abs(A * c) + np.abs(mAec) + np.abs(Bs * s)) / (1 - e * c) + np.abs(Ce)
    worst = float(np.max(err / np.spacing(scale)))
    assert worst <= 4.0, worst
    return worst


SQRT2 = float.fromhex("0x1.6a09e667f3bcdp+0")  # log_mantissa halves m above this


def log_mantissa_args(rng, n):
    r2 = SQRT2
    near = [r2]
    for _ in range(8):
        near = [np.nextafter(near[0], 0.0)] + near + [np.nextafter(near[-1], 2.0)]
    special = [1.0, 1.0 + 2.0**-52, 1.0 + 2.0**-51, 2.0 - 2.0**-52, 2.0 - 2.0**-51, 1.5, 2.0**0.5]
    return np.concatenate([rng.uniform(1.0, 2.0, n - len(near) - len(special)), near, special])


def check_log_mantissa(run, m):
    """ln(m) (ln(m / 2), half = 1, above sqrt 2) within one ulp of the correctly rounded value;
    returns the max error in ulp."""
    lm = _exact()
    out = run("log_mantissa", m)
    got, half = out[:, 0], out[:, 1]
    assert np.array_equal(half, (m > SQRT2).astype(np.float64))
    want = np.array([lm.to_float(lm.mpf_log(lm.mpf_shift(lm.from_float(v), -int(h)), 160), rnd=lm.round_nearest)
                     for v, h in zip(m.tolist(), half.tolist())])
    err = np.abs(got - want)
    ulp = np.where(want == 0.0, 5e-324, np.spacing(np.abs(want)))
    worst = float(np.max(err / ulp))
    assert worst <= 1.0, worst
    return worst


def exp_nearest(x):
    import mpmath
    with mpmath.workprec(200):
        return np.array([float(mpmath.exp(mpmath.mpf(float(v)))) for v in x])
