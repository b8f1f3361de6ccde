"""mpmath references for the tests of the kernel's FP64 core (evidence_b200/csrc/rvl_math.h)."""
import numpy as np


def sincos_args():
    """1.1e6 arguments over the lean loop's sin/cos range |x| < 1e5, with its edges: multiples of
    the table step 2 pi / 1024 and their neighbours, halfway points, tiny values, the ends."""
    rng = np.random.default_rng(7)
    h = 2 * np.pi / 1024
    k = rng.integers(-16000, 16000, 60000).astype(np.float64)
    tiny = np.ldexp(1.0, -np.arange(1, 1075, 7))  # down to the smallest denormal
    edge = 1e5 - np.ldexp(1.0, -np.arange(0, 37, 2))
    return np.ascontiguousarray(np.concatenate([
        rng.uniform(-1e5, 1e5, 700000),
        rng.uniform(-1e4, 1e4, 100000),
        rng.uniform(-7.0, 7.0, 100000),
        k * h,                                            # multiples of 2 pi / 1024 (= pi / 512)
        k * h * (1 + rng.uniform(-4e-16, 4e-16, len(k))),  # ... and their neighbours
        k * h + h / 2,                                    # halfway between two rows
        rng.uniform(-1e-3, 1e-3, 20000),
        tiny, -tiny, [0.0, -0.0, 5e-324, -5e-324],
        edge, -edge,
    ]))


def sincos_dd(x, d=None):
    """(sin, cos) of x (of x + d, the sum taken exactly, when d is given) as double-doubles from
    120-bit mpmath: columns sin hi, cos hi, sin lo, cos lo; the hi parts are correctly rounded."""
    from mpmath.libmp import from_float, mpf_add, mpf_cos_sin, mpf_sub, round_nearest, to_float
    rn = round_nearest
    out = np.empty((len(x), 4))
    dl = [None] * len(x) if d is None else np.asarray(d, dtype=np.float64).tolist()
    for i, (v, w) in enumerate(zip(np.asarray(x, dtype=np.float64).tolist(), dl)):
        a = from_float(v) if w is None else mpf_add(from_float(v), from_float(w), 2200, rn)
        c, s = mpf_cos_sin(a, 120, rn)
        sh, ch = to_float(s, rnd=rn), to_float(c, rnd=rn)
        out[i] = (sh, ch, to_float(mpf_sub(s, from_float(sh), 120, rn), rnd=rn),
                  to_float(mpf_sub(c, from_float(ch), 120, rn), rnd=rn))
    return out


def sincos_err(s, c, ref):
    """max(|s - sin|, |c - cos|) per argument against sincos_dd's double-doubles: s - hi is exact
    (the two are a few ulp apart), so the error is known to ~1e-32."""
    return np.maximum(np.abs((s - ref[:, 0]) - ref[:, 2]), np.abs((c - ref[:, 1]) - ref[:, 3]))
