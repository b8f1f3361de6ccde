"""CPU tests of bench.py's host logic: batch sizing, parity sets, the parity verdict (incl. the
Newton-cap classification of the high-eccentricity set) -- no device involved."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from evidence_b200 import synth  # noqa: E402


def test_batch_is_a_function_of_steps_only():
    assert bench.batch_for(20) == 524288 and bench.batch_for(100) == 131072 and bench.batch_for(1) == 1048576
    for k in (1, 5, 20, 50, 1000):
        b = bench.batch_for(k)
        assert 131072 <= b <= 1048576 and (k * b >= 2.0 * bench.NOMINAL_RATE or b == 1048576)
    case = synth.make_case(bench.CONFIG_ID)
    a = bench.workload_config(case, bench.batch_for(20), 8)
    assert a["global_batch"] == 8 * 524288 and "gather" not in a and a["n_epochs"] == 5000 and a["n_planets"] == 4


def test_parity_sets_cover_what_survey_8d_asks():
    case = synth.make_case(bench.CONFIG_ID)
    sets = {name: (variant, th, bar) for name, variant, th, bar in bench.parity_sets(case)}
    assert sum(len(v[1]) for v in sets.values() if v[2] <= 1e-9) >= 10_000
    ecc = [case.parnames.index(f"planet{k}_ecc") for k in range(1, 5)]
    hi = sets["ecc_0.95_0.97"][1][:, ecc].max(axis=1)
    assert np.all((hi >= 0.95) & (hi <= 0.97))
    jit = [i for i, p in enumerate(case.parnames) if p.endswith("_jitter")]
    assert np.all(sets["jitter_zero"][1][:, jit] == 0.0)
    vh = sets["ecc_0.97_1.00"][1][:, ecc].max(axis=1)
    assert np.all(vh >= 0.97) and sets["ecc_0.97_1.00"][2] == 1e-5
    # the secos / sesin variant: same data, re-parametrised; ~30 % of the rows hold an e > 1 planet
    names, fixed = bench.variant_names(case, "secos")
    assert names == sorted(names) and "planet1_secos" in names and "planet1_ml0" in names
    th = sets["secos_sesin_invalid"][1]
    e = np.stack([th[:, names.index(f"planet{k}_secos")] ** 2 + th[:, names.index(f"planet{k}_sesin")] ** 2
                  for k in range(1, 5)], axis=1)
    frac = np.mean(e.max(axis=1) > 1.0)
    assert 0.15 < frac < 0.45 and not np.any((e > 0.9001) & (e < 1.0))


def test_parity_verdict_passes_fails_and_classifies_cap_rows():
    case = synth.make_case(bench.CONFIG_ID)
    sets = bench.parity_sets(case)
    rng = np.random.default_rng(0)
    want = [rng.uniform(-1e6, -1e4, len(th)) for _, _, th, _ in sets]
    want[4][:50] = -1e30
    got = [w.copy() for w in want]
    got[0][3] += 5e-10            # inside the absolute bar
    got[3][7] += 2e-6             # inside the high-e bar
    rep, ok = bench.parity_verdict(sets, got, want, "reference")
    assert ok and rep["n"] >= 10_000 and rep["sentinels_equal"] and rep["n_sentinels"] == 50
    assert rep["max_abs"] >= 4e-10 and rep["max_abs_high_ecc"] >= 1e-6
    bad = [g.copy() for g in got]
    bad[1][0] += 1e-6             # over the bar max(1e-9, 1e-13 |lnL|) <= 1e-7 here
    assert not bench.parity_verdict(sets, bad, want, "reference")[1]
    bad = [g.copy() for g in got]
    bad[4][0] = -5.0              # a sentinel that is not one on the device
    rep, ok = bench.parity_verdict(sets, bad, want, "reference")
    assert not ok and not rep["sentinels_equal"]
    # a high-e row far off: fails unless one side reports a Newton-cap event for it
    bad = [g.copy() for g in got]
    bad[3][11] += 14.0
    assert not bench.parity_verdict(sets, bad, want, "reference", classify=lambda row: (0, 0))[1]
    rep, ok = bench.parity_verdict(sets, bad, want, "reference", classify=lambda row: (1, 0))
    assert ok and rep["sets"]["ecc_0.97_1.00"]["cap_rows"][0]["row"] == 11


def test_dump_outputs_writes_float64_within_the_size_cap(tmp_path, monkeypatch):
    lnl = np.random.default_rng(1).uniform(-1e5, -1e4, 4096)
    assert bench.dump_outputs(str(tmp_path / "a"), lnl) == ["lnl"]
    back = np.load(tmp_path / "a" / "lnl.npy")
    assert back.dtype == np.float64 and np.array_equal(back, lnl)
    # a vector over the cap: the same seeded sample of rows every time, with the rows' positions
    monkeypatch.setattr(bench, "DUMP_BYTES", 64_000)
    big = np.arange(bench.DUMP_BYTES // 8 + 10, dtype=np.float64)
    for d in ("b", "c"):
        assert bench.dump_outputs(str(tmp_path / d), big) == ["lnl", "lnl_rows"]
    files = [tmp_path / d / f"{n}.npy" for d in ("b", "c") for n in ("lnl", "lnl_rows")]
    assert sum(f.stat().st_size for f in files[:2]) <= bench.DUMP_BYTES
    got, rows = np.load(files[0]), np.load(files[1])
    assert got.dtype == rows.dtype == np.float64 and np.array_equal(got, big[rows.astype(np.int64)])
    assert np.array_equal(np.load(files[2]), got) and np.all(np.diff(rows) > 0)
