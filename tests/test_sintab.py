"""
CPU tests of the table sin/cos of the lean Newton loop (rvl::sincos_tab in
evidence_b200/csrc/rvl_math.h, table evidence_b200/csrc/rvl_sintab.h):
  * the committed table is exactly what oracle/make_sintab.py generates;
  * sincos_tab against mpmath on 10^6 arguments over the loop's range |x| < 1e5;
  * a host lock-step replay of the lean loop (tests/host_emul/emul_tab.cpp) against the
    reference's golden lnL and the C oracle's Newton iteration totals.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from _mp import sincos_args, sincos_dd, sincos_err
from _util import ROOT, lnl_close, load_golden, oracle_model

from evidence_b200.layout import compile_model
from oracle import rv_oracle

HERE = os.path.dirname(os.path.abspath(__file__))
dp = ctypes.POINTER(ctypes.c_double)


@pytest.fixture(scope="module")
def lib():
    so = os.path.join(HERE, "host_emul", "libemul_tab.so")
    src = os.path.join(HERE, "host_emul", "emul_tab.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                    "-o", so, src, "-lm"], check=True)
    return ctypes.CDLL(so)


def test_committed_table_is_the_generators_output():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import make_sintab
    finally:
        sys.path.pop(0)
    with open(make_sintab.OUT) as f:
        assert f.read() == make_sintab.render()


def _eval(fn, x):
    s = np.empty_like(x)
    c = np.empty_like(x)
    fn(x.ctypes.data_as(dp), ctypes.c_int(len(x)), s.ctypes.data_as(dp), c.ctypes.data_as(dp))
    return s, c


def test_sincos_tab_accuracy(lib):
    x = sincos_args()
    assert len(x) >= 10**6 and np.abs(x).max() < 1e5
    ref = sincos_dd(x)
    report = {}
    for name, fn in (("sincos_tab", lib.emul_sincos_tab), ("sincos_fast", lib.emul_sincos_fast)):
        s, c = _eval(fn, x)
        err = sincos_err(s, c, ref)
        off = np.mean(np.concatenate([s != ref[:, 0], c != ref[:, 1]]))  # share of the 2n values
        report[name] = (float(err.max()), float(off))
    print("max abs error, share of values not correctly rounded:", report)
    err, off = report["sincos_tab"]
    assert err <= 1.2e-16, report
    assert off <= 0.01, report
    assert report["sincos_tab"][1] < report["sincos_fast"][1], report
    # tiny arguments: sin x = x and cos x = 1 exactly, like the correctly rounded values
    t = np.ascontiguousarray(np.concatenate([np.ldexp(1.0, -np.arange(30, 1075, 7)), [5e-324]]))
    s, c = _eval(lib.emul_sincos_tab, t)
    assert np.array_equal(s, t) and np.all(c == 1.0)


def _replay(lib, desc, om, theta, U):
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    out = np.empty(len(theta))
    st = (ctypes.c_longlong * 11)()
    ids = np.ascontiguousarray(om.inst_id, dtype=np.int32)
    lib.emul_tab_loglike(ctypes.byref(desc), om.time.ctypes.data_as(dp), om.vrad.ctypes.data_as(dp),
                         om.svrad.ctypes.data_as(dp), ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                         ctypes.c_int(len(om.time)), theta.ctypes.data_as(dp),
                         ctypes.c_longlong(len(theta)), ctypes.c_int(U), out.ctypes.data_as(dp), st)
    return out, list(st)


def _cases():
    for name in ("cfg1", "cfg2", "cfg3", "cfg5", "edge_mixed"):
        meta, z = load_golden(name)
        n = min(len(z["theta"]), 64)
        yield name, meta, z, meta["parnames"], meta["fixed"], z["theta"][:n], z["lnl"][:n]
    meta, z = load_golden("kat_51peg")
    for case, want in zip(meta["cases"], z["lnl"]):
        yield ("kat_51peg/" + case["name"], meta, z, case["parnames"], case["fixed"],
               np.array(case["theta"], dtype=np.float64)[None], np.array([want]))


@pytest.mark.parametrize("U", [2, 4])
def test_lean_loop_replay_vs_reference(lib, U):
    paths = np.zeros(11, dtype=np.int64)
    for name, meta, z, parnames, fixed, theta, want in _cases():
        om = oracle_model(meta, z, parnames, fixed)
        desc, _ = compile_model(parnames, fixed, meta["insts"], om.time[0])
        got, st = _replay(lib, desc, om, theta, U)
        paths += np.array(st)
        if name == "edge_mixed":
            # rows with e > 0.97 follow chaotic Newton trajectories (see DESIGN.md): bounded by
            # the reference's own solver tolerance, as in test_host_emul.py
            e1 = theta[:, parnames.index("planet1_secos")] ** 2 + theta[:, parnames.index("planet1_sesin")] ** 2
            e2 = np.hypot(theta[:, parnames.index("planet2_ecos")], theta[:, parnames.index("planet2_esin")])
            calm = (e1 <= 0.97) & (e2 <= 0.97)
            ok, worst = lnl_close(got[calm], want[calm])
            assert ok, (name, worst)
            ok, worst = lnl_close(got, want, abs_tol=1e-5)
            assert ok, (name, worst)
            theta = theta[calm]  # (their Newton step counts are chaotic too)
            _, st = _replay(lib, desc, om, theta, U)
        elif "clamp" in name:  # the 51 Peg case at the clamp e = 0.99: the same chaotic regime
            ok, worst = lnl_close(got, want, abs_tol=1e-5)
            assert ok, (name, worst)
            continue
        else:
            ok, worst = lnl_close(got, want)
        assert ok, (name, worst)
        _, iters, caps = rv_oracle.c_loglike_batch(bytes(desc), om.time, om.vrad, om.svrad, om.inst_id,
                                                   len(meta["insts"]), theta)
        assert abs(st[9] - iters) <= 1e-6 * iters + 5, (name, st[9], iters)
        assert st[10] == caps == 0, name
    solves = paths[7] * 32 * U
    # every solve started in the lean loop; a few chaotic e > 0.97 ones restarted in the general loop
    assert paths[0] == paths[7] and paths[8] <= 1e-3 * paths[7], paths
    print("warp passes per warp-solve (pass 1, table >= 0.75, medium, mid, small, tiny, "
          "final):", np.round(paths[:7] / paths[7], 3), f"{paths[9] / solves:.3f} steps per solve")
