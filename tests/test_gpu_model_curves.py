"""
GPU tests of the model velocity curves (rvl_kepler_rv / RVModel.kepler_rv_batch, modelk, kep_rv,
residuals_batch) against the oracle's restatement of the reference's modelk / kep_rv.

Bar: |dv| <= 1e-10 sum|K_p| + 1e-12 on rows whose eccentricities are all below 0.97 -- the true-anomaly
bar of the solver test carried through K (cos(nu + omega) + e cos omega).  Above 0.97 Newton from E = M
is chaotic (DESIGN.md section 3): 1e-5 sum|K_p|, with rows that hit the iteration cap reported.  Rows
with a logperiod on which numpy's exp is not the nearest double carry the reference's own last bit of
P: 1e-8 sum|K_p| (the rule of test_random_model_structures_vs_numpy_oracle).
"""
import warnings

import numpy as np
import pytest

from _util import device_model, lnl_close, load_golden, oracle_model, tables_of

pytestmark = pytest.mark.gpu

CFGS = ["cfg1", "cfg2", "cfg3", "cfg5", "edge_mixed"]


def _exp_nearest(v):
    import mpmath
    with mpmath.workprec(200):
        return float(mpmath.exp(mpmath.mpf(float(v))))


def _pardicts(names, fixed, theta):
    out = []
    for row in np.atleast_2d(theta):
        pd = {n: float(v) for n, v in zip(names, row)}
        pd.update(fixed)  # fixed wins (:178)
        out.append(pd)
    return out


def _planet(pd, k):
    """(|K|, P, e, numpy's exp of logperiod is the nearest double) of planet k, the oracle's way."""
    pre = f"planet{k}_"
    amp = pd[pre + "k1"] if pre + "k1" in pd else np.exp(pd[pre + "logk1"])
    exact = True
    if pre + "period" in pd:
        per = pd[pre + "period"]
    else:
        per = np.exp(pd[pre + "logperiod"])
        exact = per == _exp_nearest(pd[pre + "logperiod"])
    if pre + "secos" in pd:
        e = pd[pre + "secos"] ** 2 + pd[pre + "sesin"] ** 2
    elif pre + "ecos" in pd:
        e = np.sqrt(pd[pre + "ecos"] ** 2 + pd[pre + "esin"] ** 2)
    else:
        e = pd[pre + "ecc"]
    return abs(amp), per, e, exact


def _bars(pds, planets):
    """Per-row bar and whether the row is in the chaotic high-e regime."""
    bars, hot = [], []
    for pd in pds:
        info = [_planet(pd, k) for k in planets]
        ksum = sum(i[0] for i in info)
        high = any(i[2] >= 0.97 for i in info)
        exact = all(i[3] for i in info)
        rel = 1e-5 if high else (1e-10 if exact else 1e-8)
        bars.append(rel * ksum + 1e-12)
        hot.append(high)
    return np.array(bars), np.array(hot, dtype=bool)


def _device_curves(m, theta, time, planets):
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        rv, ok = m.kepler_rv_batch(theta, time, planets)
    return rv, ok, sum("Newton cap" in str(x.message) for x in w)


def _check(m, om, names, fixed, theta, time, planets, label):
    """Device curves of ``planets`` for every row against the oracle; returns rows that capped."""
    pds = _pardicts(names, fixed, theta)
    rv, ok, capped = _device_curves(m, theta, time, planets)
    bars, hot = _bars(pds, planets)
    reported = []
    for b, pd in enumerate(pds):
        if list(planets) == list(range(1, om.nplanets + 1)):
            want = om.kep_rv(pd, time)  # the reference's own sum
        else:  # a subset: the planets' modelk added in planet order, like kep_rv does
            parts = [om.modelk(pd, time, k) for k in planets]
            want = None if any(p is None for p in parts) else np.sum(parts, axis=0)
        if want is None:
            assert not ok[b] and np.all(np.isnan(rv[b])), (label, b)
            continue
        assert ok[b] and np.all(np.isfinite(rv[b])), (label, b)
        err = float(np.max(np.abs(rv[b] - want))) if len(time) else 0.0
        if err > bars[b]:
            # only a row in the chaotic regime whose solves hit the cap may miss the bar: report it
            _, _, c = _device_curves(m, theta[b:b + 1], time, planets)
            assert hot[b] and c > 0, (label, b, err, bars[b])
            reported.append((label, b, err))
    assert capped == 0 or any(hot), label
    return reported


def _grid(om, pds):
    pmax = max(_planet(pd, k)[1] for pd in pds for k in range(1, om.nplanets + 1))
    return np.linspace(om.time.min() - pmax, om.time.max() + pmax, 3001)


@pytest.mark.parametrize("name", CFGS)
def test_golden_rows_every_planet_and_the_sum(name):
    meta, z = load_golden(name)
    m, om = device_model(meta, z), oracle_model(meta, z)
    names, fixed, theta = meta["parnames"], meta["fixed"], z["theta"]
    pds = _pardicts(m.parnames, fixed, theta)
    reported = []
    for time in (om.time, _grid(om, pds)):
        for k in range(1, m.nplanets + 1):
            reported += _check(m, om, m.parnames, fixed, theta, time, [k], (name, k))
        reported += _check(m, om, m.parnames, fixed, theta, time, list(range(1, m.nplanets + 1)),
                           (name, "sum"))
    print("cap rows:", reported)
    m.close()


def test_golden_kat_51peg_every_case():
    meta, z = load_golden("kat_51peg")
    for case in meta["cases"]:
        m = device_model(meta, z, case["parnames"], case["fixed"])
        om = oracle_model(meta, z, case["parnames"], case["fixed"])
        theta = np.array([case["theta"]])
        pds = _pardicts(m.parnames, case["fixed"], theta)
        times = [om.time] + ([_grid(om, pds)] if m.nplanets else [])
        for time in times:
            for k in range(1, m.nplanets + 1):
                _check(m, om, m.parnames, case["fixed"], theta, time, [k], (case["name"], k))
            rv, ok, _ = _device_curves(m, theta, time, None)
            want = om.kep_rv(pds[0], time) if m.nplanets else np.zeros(len(time))
            if want is None:
                assert not ok[0] and np.all(np.isnan(rv[0])) and m.kep_rv(pds[0], time) is None
            else:
                bars, _ = _bars(pds, range(1, m.nplanets + 1))
                assert np.max(np.abs(rv[0] - want)) <= bars[0], case["name"]
                assert np.array_equal(m.kep_rv(pds[0], time), rv[0])
        m.close()


@pytest.fixture(scope="module")
def cfg2():
    meta, z = load_golden("cfg2")
    m, om = device_model(meta, z), oracle_model(meta, z)
    yield meta, z, m, om
    m.close()


def test_edge_shapes(cfg2):
    meta, z, m, om = cfg2
    theta = z["theta"][:40]
    rng = np.random.default_rng(3)
    both = [1, 2]
    _check(m, om, m.parnames, meta["fixed"], theta[:1], om.time, both, "B=1")
    for T in (1, 31, 33):
        _check(m, om, m.parnames, meta["fixed"], theta, rng.uniform(50000, 56000, T), both, ("T", T))
    _check(m, om, m.parnames, meta["fixed"], theta, rng.permutation(om.time), both, "unsorted")
    # |M| >= 1e5 everywhere: the general Newton loop with libdevice sin/cos (the oracle: glibc)
    far = 52500.0 + np.linspace(2.0e7, 2.1e7, 257)
    pds = _pardicts(m.parnames, meta["fixed"], theta)
    assert min(2 * np.pi / _planet(pd, k)[1] * 2e7 for pd in pds for k in both) >= 1e5
    rv, ok, _ = _device_curves(m, theta, far, both)
    for b, pd in enumerate(pds):
        bar = 1e-9 * sum(_planet(pd, k)[0] for k in both)
        assert ok[b] and np.max(np.abs(rv[b] - om.kep_rv(pd, far))) <= bar, b
    # empty batches and an empty time axis
    rv, ok = m.kepler_rv_batch(theta[:0], om.time)
    assert rv.shape == (0, len(om.time)) and ok.shape == (0,)
    rv, ok = m.kepler_rv_batch(theta, np.zeros(0))
    assert rv.shape == (len(theta), 0) and ok.all()
    with pytest.raises(ValueError):
        m.kepler_rv_batch(theta, om.time, planets=[3])


def test_model_without_planets():
    meta, z = load_golden("cfg1")
    names = [p for p in meta["parnames"] if "planet" not in p]
    m = device_model(meta, z, names, {})
    X = np.random.default_rng(0).uniform(0, 3, (17, len(names)))
    rv, ok = m.kepler_rv_batch(X, m.time)
    assert np.array_equal(rv, np.zeros_like(rv)) and ok.all()
    pd = dict(zip(m.parnames, X[0]))
    assert np.array_equal(m.kep_rv(pd, m.time), np.zeros(len(m.time)))
    m.close()


def test_excluding_the_invalid_planet():
    """edge_mixed: rows whose planet 1 (secos/sesin) is invalid still have valid curves without it."""
    meta, z = load_golden("edge_mixed")
    m, om = device_model(meta, z), oracle_model(meta, z)
    pds = _pardicts(m.parnames, meta["fixed"], z["theta"])
    bad1 = np.array([om.modelk(pd, om.time, 1) is None for pd in pds])
    valid23 = np.array([om.modelk(pd, om.time, 2) is not None and om.modelk(pd, om.time, 3) is not None
                        for pd in pds])
    rows = np.flatnonzero(bad1 & valid23)
    assert len(rows) >= 1
    theta = z["theta"][rows]
    _check(m, om, m.parnames, meta["fixed"], theta, om.time, [2, 3], "without planet 1")
    rv, ok = m.kepler_rv_batch(theta, om.time)
    assert not ok.any() and np.all(np.isnan(rv))
    for b in rows:
        assert m.kep_rv(pds[b], om.time) is None and m.modelk(pds[b], om.time, 1) is None
        got = m.kep_rv(pds[b], om.time, exclude_planet=1)
        want = om.modelk(pds[b], om.time, 2) + om.modelk(pds[b], om.time, 3)
        bars, _ = _bars([pds[b]], [2, 3])
        assert got is not None and np.max(np.abs(got - want)) <= bars[0]
    m.close()


def test_determinism_and_form_independence(cfg2):
    import torch
    meta, z, m, om = cfg2
    theta = z["theta"]
    time = np.linspace(om.time.min() - 100, om.time.max() + 100, 1001)
    rv, ok = m.kepler_rv_batch(theta, time)
    for _ in range(3):
        again, ok2 = m.kepler_rv_batch(theta, time)
        assert np.array_equal(again, rv) and np.array_equal(ok2, ok)
    for b in (0, 17, len(theta) - 1):  # a row alone, and inside other batches
        assert np.array_equal(m.kepler_rv_batch(theta[b:b + 1], time)[0][0], rv[b])
        assert np.array_equal(m.kepler_rv_batch(theta[b:b + 5], time)[0][0], rv[b])
    perm = np.random.default_rng(1).permutation(len(theta))
    assert np.array_equal(m.kepler_rv_batch(theta[perm], time)[0], rv[perm])
    # the host form and the device form
    dev, dok = m.kepler_rv_device(torch.from_numpy(theta).cuda(), torch.from_numpy(time).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(dev.cpu().numpy(), rv) and np.array_equal(dok.cpu().numpy(), ok)
    # a likelihood call in between leaves the curves alone (shared per-point scratch)
    m.log_likelihood_batch(theta)
    assert np.array_equal(m.kepler_rv_batch(theta, time)[0], rv)
    # a multi-device handle runs the call on its first device
    mm = device_model(meta, z, devices="all")
    assert np.array_equal(mm.kepler_rv_batch(theta, time)[0], rv)
    mm.close()


@pytest.mark.parametrize("name", CFGS)
def test_residuals_reproduce_the_likelihood(name):
    """logL(residuals_batch) equals the likelihood kernel's lnL on the golden rows."""
    meta, z = load_golden(name)
    m = device_model(meta, z)
    theta = z["theta"]
    res, var = m.residuals_batch(theta)
    lnl = m.log_likelihood_batch(theta)
    valid = lnl != -1e30
    assert np.all(np.isnan(res[~valid])) and np.all(np.isfinite(res[valid]))
    got = np.array([m.logL(res[b], var[b]) for b in np.flatnonzero(valid)])
    ok, worst = lnl_close(got, lnl[valid])
    assert ok, (name, worst)
    # and the golden values of the reference itself, to the suite's bar where e < 0.97
    ok, worst = lnl_close(got, z["lnl"][valid], abs_tol=1e-5)
    assert ok, (name, worst)
    m.close()
