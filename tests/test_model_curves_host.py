"""CPU tests of the host logic behind RVModel.modelk / kep_rv / drift / kepler_rv_batch: pardict ->
theta row, planet selection -> mask, output chunking, and the host drift against the oracle."""
import numpy as np
import pytest

from _util import load_golden
from evidence_b200.layout import compile_model
from evidence_b200.rvmodel import (curve_chunks, host_drift, pardict_row, planet_mask,
                                   planet_param_names)
from oracle.rv_oracle import OracleRVModel

# two planets: planet 1 fully free (k1, period, secos/sesin, ma0), planet 2 with a fixed logperiod
# and ecc/omega, ml0; fixed epochs; one instrument with a free offset and a free linear drift
FREE = ["planet1_k1", "planet1_period", "planet1_secos", "planet1_sesin", "planet1_ma0",
        "planet2_logk1", "planet2_ecc", "planet2_omega", "planet2_ml0", "harps_offset", "drift_lin"]
FIXED = {"planet1_epoch": 55000.0, "planet2_epoch": 55010.0, "planet2_logperiod": 3.5}


def _model():
    desc, names = compile_model(FREE, FIXED, ["harps"], 54000.0)
    return desc, names


def _pardict(names):
    return dict({n: 0.1 * (i + 1) for i, n in enumerate(names)}, **FIXED)


def test_planet_param_names_follow_the_parametrisation():
    desc, names = _model()
    assert [n for n, _ in planet_param_names(desc, 1)] == [
        "planet1_k1", "planet1_period", "planet1_secos", "planet1_sesin", "planet1_ma0", "planet1_epoch"]
    p2 = dict(planet_param_names(desc, 2))
    assert list(p2) == ["planet2_logk1", "planet2_logperiod", "planet2_ecc", "planet2_omega",
                        "planet2_ml0", "planet2_epoch"]
    assert p2["planet2_logperiod"].slot == -1 and p2["planet2_logperiod"].value == 3.5
    assert p2["planet2_ecc"].slot == names.index("planet2_ecc")


def test_pardict_row_free_and_fixed_names():
    desc, names = _model()
    pd = _pardict(names)
    row = pardict_row(pd, names, desc, planet_mask(2))
    assert row.tolist() == [pd[n] for n in names]
    # fixed values equal to the model's are accepted, whatever their type
    pd2 = dict(pd, planet2_logperiod=np.float64(3.5))
    assert np.array_equal(pardict_row(pd2, names, desc, planet_mask(2)), row)


def test_pardict_row_missing_names():
    desc, names = _model()
    pd = _pardict(names)
    # names no summed planet reads may be missing: filled with 0
    for gone in ("harps_offset", "drift_lin", "planet2_ecc"):
        del pd[gone]
    row = pardict_row(pd, names, desc, planet_mask(2, [1]))
    for gone in ("harps_offset", "drift_lin", "planet2_ecc"):
        assert row[names.index(gone)] == 0.0
    assert row[names.index("planet1_k1")] == pd["planet1_k1"]
    # ... but a name a summed planet reads raises KeyError naming it
    with pytest.raises(KeyError, match="planet2_ecc"):
        pardict_row(pd, names, desc, planet_mask(2))
    # the fixed names may be missing altogether: the model was compiled with them
    pd3 = {n: v for n, v in _pardict(names).items() if n not in FIXED}
    assert pardict_row(pd3, names, desc, planet_mask(2)).shape == (len(names),)


def test_pardict_row_changed_fixed_value():
    desc, names = _model()
    pd = dict(_pardict(names), planet2_logperiod=3.6)
    with pytest.raises(ValueError, match="planet2_logperiod"):
        pardict_row(pd, names, desc, planet_mask(2))
    with pytest.raises(ValueError, match="planet1_epoch"):
        pardict_row(dict(_pardict(names), planet1_epoch=1.0), names, desc, planet_mask(2, 1))
    # a planet that is not summed does not read it
    assert pardict_row(pd, names, desc, planet_mask(2, 1)).shape == (len(names),)


def test_planet_mask():
    assert planet_mask(3) == 0b111
    assert planet_mask(0) == 0
    assert planet_mask(3, 2) == 0b010
    assert planet_mask(3, [1, 3]) == 0b101
    assert planet_mask(3, np.array([3])) == 0b100
    assert planet_mask(3, []) == 0
    assert planet_mask(3, exclude=2) == 0b101
    assert planet_mask(3, exclude=(1, 2)) == 0b100
    assert planet_mask(3, [1, 2], exclude=[2]) == 0b001
    assert planet_mask(8) == 0xFF
    for bad in (0, 4, 1.5, [1, 5]):
        with pytest.raises(ValueError):
            planet_mask(3, bad)
    with pytest.raises(ValueError):
        planet_mask(3, exclude=4)


def test_curve_chunks():
    mib = 1 << 20
    assert curve_chunks(10, 100) == [(0, 10)]
    # 256 MiB of float64 at T = 4096 is 8192 rows
    assert curve_chunks(20000, 4096) == [(0, 8192), (8192, 16384), (16384, 20000)]
    assert curve_chunks(5, 10, max_bytes=80) == [(0, 1), (1, 2), (2, 3), (3, 4), (4, 5)]
    # a single row larger than the cap still goes in one piece
    assert curve_chunks(3, 64 * mib) == [(0, 1), (1, 2), (2, 3)]
    assert curve_chunks(0, 100) == []
    assert curve_chunks(7, 0) == [(0, 7)]
    for B, T in ((1, 1), (12345, 3001), (100000, 5000)):
        ch = curve_chunks(B, T)
        assert ch[0][0] == 0 and ch[-1][1] == B
        assert all(a[1] == b[0] for a, b in zip(ch, ch[1:]))
        assert all(8 * (hi - lo) * T <= 256 * mib or hi - lo == 1 for lo, hi in ch)


@pytest.mark.parametrize("name", ["cfg2", "kat_51peg"])
def test_host_drift_matches_the_oracle_bit_for_bit(name):
    meta, z = load_golden(name)
    from _util import tables_of
    om = OracleRVModel({}, tables_of(meta, z), ["x_offset"])
    rng = np.random.default_rng(7)
    grid = np.linspace(om.time.min() - 300.0, om.time.max() + 300.0, 3001)
    for time in (om.time, grid, rng.permutation(om.time)):
        for pd in ({"drift_lin": 0.37},
                   {"drift_lin": -1.25, "drift_quad": 0.031, "drift_cub": -2e-3, "drift_quar": 1e-4},
                   {"drift_quad": 0.5, "drift_tref": 55123.5},
                   {"drift_lin": 0.2, "drift_quar": -3e-5, "drift_tref": float(time[-1])}):
            want = OracleRVModel.drift(pd, time)
            got = host_drift(pd, time)
            assert got.dtype == np.float64 and np.array_equal(got, want), pd
