"""
Circular (wrapped) coordinates of the built-in slice samplers, on the CPU: the rule of
`rvl_slice_phase_wrapped` in the oracle, the circular whitening of both samplers, the host sampler
on a periodic problem with known evidence, the runner's `builtin_wrap` setting, and the argument
checks of the new entry point (library only, no GPU).
"""
import ctypes

import numpy as np
import pytest
from scipy.special import i0e

from evidence_b200 import priors
from evidence_b200 import sampler as hs
from evidence_b200 import ultranest as runner
from oracle import slice_oracle as so

import _slice_wrap_oracle as wo

KAPPA, S = 50.0, 0.03


def periodic_lnl(u):
    """Two circular dimensions with their mode on the seam (von Mises in 2 pi u), three Gaussian."""
    return ((KAPPA * (np.cos(2 * np.pi * u[:, :2]) - 1.0)).sum(1)
            - (((u[:, 2:] - 0.5) ** 2) / (2 * S * S)).sum(1))


PERIODIC_LNZ = 2 * np.log(i0e(KAPPA)) + 3 * np.log(S * np.sqrt(2 * np.pi))
PERIODIC_WRAP = np.array([True, True, False, False, False])


@pytest.mark.parametrize("p,want", [(-2.0 ** -60, 0.0), (1.0, 0.0), (3.25, 0.25), (-0.75, 0.25),
                                    (1.0 - 2.0 ** -53, 1.0 - 2.0 ** -53), (0.0, 0.0),
                                    (-2.0 ** -53, 1.0 - 2.0 ** -53)])
def test_wrap_rule_edge_values(p, want):
    for f in (wo.wrap_unit, hs.wrap_unit):
        got = float(f(np.array([p]))[0])
        assert got == want and (got != 0.0 or np.signbit(got) == np.signbit(want)), (f, p, got)


def _state(k, d, n_out, m, seed, rng, scale=0.4):
    chol = np.tril(rng.normal(0.0, 0.1 * scale, (d, d)), -1) + np.diag(rng.uniform(0.5, 1.0, d) * scale)
    junk = lambda *s: rng.normal(0.0, 3.0, s)  # noqa: E731
    u = rng.uniform(0.0, 1.0, (k, d))
    u[0], u[1] = 0.0, 1.0 - 2.0 ** -53
    return so.SliceState(
        k=k, d=d, n_out=n_out, m=m, seed=seed, move=3, shrink_round=0, lmin=0.25, chol=chol,
        u=u, theta=junk(k, d), lcur=junk(k), dirn=junk(k, d), lo=junk(k), hi=junk(k), lo2=junk(k),
        hi2=junk(k), tval=junk(k, m), pending=np.full(k, 7, np.int32),
        cand_out=junk(k, 2 * n_out, d), inside_out=np.full((k, 2 * n_out), 0x77, np.uint8),
        ll_out=junk(k, 2 * n_out), cand=junk(k, m, d), inside=np.full((k, m), 0x77, np.uint8),
        cand_ll=junk(k, m), cand_th=junk(k, m, d), stats=np.array([5, 9], np.uint64))


def _move(st, rng, phase):
    """Phases 0, 1, 2, 3 of an oracle (phase(ph, st)) with made-up likelihoods; the state after
    each."""
    out = [phase(0, st) and st.copy()]
    st.ll_out = np.where(rng.uniform(size=st.ll_out.shape) < 0.6, 1.0, 0.0)
    for ph, sr in ((1, 0), (2, 1), (3, 2)):
        st.shrink_round = sr
        phase(ph, st)
        out.append(st.copy())
        st.cand_ll = np.where(rng.uniform(size=st.cand_ll.shape) < 0.3, 1.0, 0.0)
        st.cand_th = rng.normal(size=st.cand_th.shape)
    return out


def test_oracle_without_a_wrapped_coordinate_is_the_unwrapped_oracle():
    """The wrapped restatement with an all-false mask gives every buffer of oracle/slice_oracle.py."""
    k, d, n_out, m = 9, 37, 3, 4
    a = _state(k, d, n_out, m, 17, np.random.default_rng(0))
    b = a.copy()
    none = np.zeros(d, dtype=bool)
    for sa, sb in zip(_move(a, np.random.default_rng(1), so.phase),
                      _move(b, np.random.default_rng(1), lambda ph, st: wo.phase(ph, st, none))):
        for name, v in sa.__dict__.items():
            if isinstance(v, np.ndarray):
                assert np.array_equal(v, getattr(sb, name), equal_nan=True), name


def test_oracle_wraps_the_masked_coordinates_only():
    """Wrapped coordinates of every candidate lie in [0, 1) and equal wrap_unit(u + t dirn); the
    inside flag is the cube test of the other coordinates; accepted points stay in [0, 1)."""
    k, d, n_out, m = 16, 6, 4, 5
    rng = np.random.default_rng(2)
    st = _state(k, d, n_out, m, 5, rng, scale=0.8)
    wrap = np.array([True, False, True, False, False, True])
    wo.phase(0, st, wrap)
    t = np.concatenate([st.lo[:, None] - np.arange(n_out), st.hi[:, None] + np.arange(n_out)], axis=1)
    p = st.u[:, None, :] + t[:, :, None] * st.dirn[:, None, :]
    assert np.array_equal(st.cand_out[..., wrap], wo.wrap_unit(p[..., wrap]))
    assert np.array_equal(st.cand_out[..., ~wrap], np.clip(p[..., ~wrap], 0.0, so.HI_CLAMP))
    want_in = ((p[..., ~wrap] >= 0) & (p[..., ~wrap] < 1)).all(-1)
    assert np.array_equal(st.inside_out.astype(bool), want_in)
    assert (~((p[..., wrap] >= 0) & (p[..., wrap] < 1))).any()  # the seam was crossed
    states = _move(st, rng, lambda ph, s: wo.phase(ph, s, wrap))
    assert np.all((states[0].cand_out[..., wrap] >= 0.0) & (states[0].cand_out[..., wrap] < 1.0))
    for s in states[1:]:
        assert np.all((s.cand[..., wrap] >= 0.0) & (s.cand[..., wrap] < 1.0))
        assert np.all((s.u >= 0.0) & (s.u < 1.0))
    assert states[-1].stats[1] > 9  # some walkers moved


def _seam_set(rng, n=400, d=4):
    """Points of a correlated cluster centred at u0 = 0.97 (across the seam) in dimension 0."""
    cov = np.array([[1.0, 0.6, 0.0, 0.2], [0.6, 1.0, 0.1, 0.0], [0.0, 0.1, 1.0, 0.0],
                    [0.2, 0.0, 0.0, 1.0]]) * 0.03 ** 2
    x = rng.multivariate_normal([0.97, 0.5, 0.4, 0.6], cov[:d, :d], n)
    x[:, 0] = hs.wrap_unit(x[:, 0])
    return x


def test_circular_whitening_does_not_depend_on_where_the_mode_sits():
    import torch
    from evidence_b200 import sampler_dev
    u = _seam_set(np.random.default_rng(3))
    assert (u[:, 0] < 0.1).any() and (u[:, 0] > 0.9).any()
    middle = u.copy()
    middle[:, 0] = hs.wrap_unit(u[:, 0] - 0.47)  # the same set with its mode at 0.5
    wrap = np.array([True, False, False, False])
    want = hs._whitening(middle)
    assert np.abs(hs._whitening(u, wrap) - want).max() < 1e-12
    assert np.abs(hs._whitening(u) - want).max() > 0.1  # the plain covariance spans the cube
    tw = torch.as_tensor(wrap)
    got = sampler_dev._whitening(torch, torch.from_numpy(u), tw).numpy()
    assert np.abs(got - sampler_dev._whitening(torch, torch.from_numpy(middle)).numpy()).max() < 1e-12
    # with no mask: bitwise the factor of the plain covariance
    assert np.array_equal(hs._whitening(u, None), np.linalg.cholesky(np.cov(u.T) + np.eye(4) * 1e-18))


def test_host_sampler_without_a_mask_is_unchanged():
    f = lambda th: -0.5 * np.sum(th ** 2, axis=1)  # noqa: E731
    g = lambda u: -10 + 20 * u  # noqa: E731
    a = hs.nested_sample(f, g, 3, nlive=80, seed=4)
    for w in (None, [False] * 3, np.zeros(3, bool)):
        b = hs.nested_sample(f, g, 3, nlive=80, seed=4, wrapped=w)
        assert b.logz == a.logz and b.ncall == a.ncall and np.array_equal(b.samples, a.samples)
        assert b.wrapped.tolist() == [False] * 3


@pytest.mark.parametrize("seed", [0, 1])
def test_host_sampler_on_a_periodic_problem(seed):
    """Identity prior transform, d = 5: von Mises (kappa = 50) in two circular dimensions with the
    mode on the seam, narrow Gaussians in three: ln Z = 2 ln i0e(kappa) + 3 ln(s sqrt(2 pi))."""
    r = hs.nested_sample(periodic_lnl, lambda u: u, 5, nlive=100, seed=seed, wrapped=PERIODIC_WRAP)
    assert abs(r.logz - PERIODIC_LNZ) < 3 * r.logzerr, (r.logz, r.logzerr, PERIODIC_LNZ)
    assert r.wrapped.tolist() == PERIODIC_WRAP.tolist()
    # the posterior of a circular coordinate straddles the seam
    x = r.samples[:, 0]
    assert np.mean(x < 0.1) > 0.3 and np.mean(x > 0.9) > 0.3 and np.all((x >= 0) & (x < 1))


def test_device_sampler_torch_formulation_on_a_periodic_problem():
    """The torch formulation of sampler_dev (CPU tensors) with the same mask and problem."""
    import torch
    from evidence_b200.sampler_dev import nested_sample_device

    def fused(U):
        return U, torch.from_numpy(periodic_lnl(U.numpy()))
    r = nested_sample_device(fused, 5, nlive=100, seed=1, device="cpu", wrapped=PERIODIC_WRAP)
    assert abs(r.logz - PERIODIC_LNZ) < 3 * r.logzerr, (r.logz, r.logzerr, PERIODIC_LNZ)
    assert r.wrapped.tolist() == PERIODIC_WRAP.tolist()
    assert np.all((r.samples[:, :2] >= 0) & (r.samples[:, :2] < 1))


def test_ellipsoid_rejects_a_mask():
    f = lambda th: -0.5 * np.sum(th ** 2, axis=1)  # noqa: E731
    with pytest.raises(ValueError, match="wrapped"):
        hs.nested_sample(f, lambda u: u, 2, nlive=50, method="ellipsoid", wrapped=[True, False])
    r = hs.nested_sample(f, lambda u: u, 2, nlive=50, method="ellipsoid", wrapped=[False, False])
    assert np.isfinite(r.logz)
    with pytest.raises(ValueError, match="dimensions"):
        hs.nested_sample(f, lambda u: u, 2, nlive=50, wrapped=[True])


class PlanetToy:
    """The reference's scalar model protocol with one circular-by-name parameter."""

    def __init__(self):
        self.parnames = sorted(["planet1_omega", "planet1_k1", "planet1_ml0"])
        self.datadict, self.fixedpardict = {}, {}

    def log_likelihood(self, x):
        return -0.5 * np.sum(((np.asarray(x) - 3.0) / 0.5) ** 2)


@pytest.mark.parametrize("method", ["slice", "ellipsoid"])
@pytest.mark.parametrize("wrap", [None, False, True])
def test_runner_passes_the_mask_only_when_asked(tmp_path, monkeypatch, wrap, method):
    seen = {}
    real = hs.nested_sample

    def spy(*a, **kw):
        seen["wrapped"] = kw.get("wrapped")
        return real(*a, **kw)
    monkeypatch.setattr(hs, "nested_sample", spy)
    model = PlanetToy()
    priordict = {p: priors.Uniform(0.0, 6.0) for p in model.parnames}
    settings = {"nlive": 60, "sampler": "builtin", "seed": 1, "ndraw_min": 256, "builtin_method": method}
    if wrap is not None:
        settings["builtin_wrap"] = wrap
    rundict = {"target": "toy", "runid": "w", "save_dir": str(tmp_path), "nplanets": 1}
    if wrap and method == "ellipsoid":
        with pytest.raises(ValueError, match="wrapped"):
            runner.run(model, rundict, priordict, settings)
        assert seen["wrapped"].tolist() == [False, True, True]
        return
    out = runner.run(model, rundict, priordict, settings)
    if wrap:
        # the mask UltraNest would get: names containing omega or ml0 (sorted: k1, ml0, omega)
        assert seen["wrapped"].tolist() == [False, True, True]
        assert out.sampler_impl.endswith("wrapped: planet1_ml0, planet1_omega")
    else:
        assert seen["wrapped"] is None and "wrapped" not in out.sampler_impl
    assert np.isfinite(out.logZ)


def test_wrapped_entry_point_rejects_bits_at_or_above_d(built_lib):
    """Mask bits at or above d: RVL_EINVAL and a message, before anything reaches the device; the
    size and phase checks of rvl_slice_phase hold for the new entry point too."""
    from evidence_b200 import _abi
    lib = _abi.load()
    for d, word, bit in ((3, 0, 3), (3, 0, 31), (32, 1, 0), (33, 1, 1), (100, 3, 4), (127, 3, 31),
                         (1, 2, 7)):
        a = _abi.rvl_slice_args()
        a.k, a.d, a.n_out, a.m = 4, d, 2, 2
        bits = (ctypes.c_uint32 * 4)()
        bits[0] = 1  # a valid bit beside the bad one
        bits[word] |= 1 << bit
        assert lib.rvl_slice_phase_wrapped(0, ctypes.byref(a), bits, None) == -1  # RVL_EINVAL
        msg = lib.rvl_slice_last_error().decode()
        assert f"bit {32 * word + bit} set, but d = {d}" in msg, msg
    a = _abi.rvl_slice_args()
    a.k, a.d, a.n_out, a.m = 4, 3, 2, 65
    assert lib.rvl_slice_phase_wrapped(1, ctypes.byref(a), None, None) == -1
    assert "bad sizes" in lib.rvl_slice_last_error().decode()
    a.m = 2
    bits = (ctypes.c_uint32 * 4)(0b101, 0, 0, 0)
    assert lib.rvl_slice_phase_wrapped(4, ctypes.byref(a), bits, None) == -1
    assert "phase must be" in lib.rvl_slice_last_error().decode()
    assert lib.rvl_slice_phase_wrapped(0, None, bits, None) == -1
