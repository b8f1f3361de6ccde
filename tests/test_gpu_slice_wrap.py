"""
Circular (wrapped) coordinates on the GPU: `rvl_slice_phase_wrapped` against the oracle buffer by
buffer, walkers crossing the seam, the device sampler on a periodic problem with known evidence, and
an RV fit through the runner whose argument of periastron sits at 0 = 2 pi.
"""
import ctypes

import numpy as np
import pytest
from scipy import stats
from scipy.special import i0e

import _slice_wrap_oracle as wo
from test_gpu_slice_kernels import (SEEDS, SHAPES, Device, check, dirn_tolerance, fabricated,
                                    random_state, run_move)

pytestmark = pytest.mark.gpu


class WrappedDevice(Device):
    """Device buffers of a SliceState with a wrap mask, phases through rvl_slice_phase_wrapped."""

    def __init__(self, st, wrap):
        super().__init__(st)
        self.bits = (ctypes.c_uint32 * 4)()
        for j in np.flatnonzero(wrap):
            self.bits[j >> 5] |= 1 << (int(j) & 31)

    def phase(self, ph, move, shrink_round):
        self.args.move, self.args.shrink_round = move, shrink_round
        rc = self.lib.rvl_slice_phase_wrapped(ph, ctypes.byref(self.args), self.bits,
                                              self.torch.cuda.current_stream().cuda_stream)
        assert rc == 0, self.lib.rvl_slice_last_error().decode()
        self.torch.cuda.synchronize()


def wrapped_state(k, d, n_out, m, seed, move, rng):
    """random_state and a mask (first and last coordinate always circular), with walkers 0 and 1
    on the seam: u = 0 and u = 1 - 2^-53 in every circular coordinate."""
    st = random_state(k, d, n_out, m, seed, move, rng)
    wrap = rng.uniform(size=d) < 0.5
    wrap[0] = wrap[d - 1] = True
    st.u[0, wrap] = 0.0
    if k > 1:
        st.u[1, wrap] = 1.0 - 2.0 ** -53
    return st, wrap


def run_wrapped_move(st, wrap, dev, lls):
    """test_gpu_slice_kernels.run_move against the wrapped restatement: phases 0 -> 1 -> 2 -> 2 -> 3
    on the device and on the host, every buffer checked after each.  Returns the device buffers."""
    seen = []
    dev.phase(0, st.move, 0)
    d_dirn = dev.read()["dirn"][:st.k]
    z, own = wo.phase(0, st, wrap, dirn=d_dirn)
    assert np.all(np.abs(d_dirn - own) <= dirn_tolerance(st, z)), "direction off by more than 32 ulp"
    seen.append(check(dev, st, "phase 0"))
    for i, (ph, sr) in enumerate([(1, 0), (2, 1), (2, 2), (3, 3)]):
        for name, v in lls(i).items():
            dev.set(name, v)
            setattr(st, name, v.copy())
        st.shrink_round = sr
        dev.phase(ph, st.move, sr)
        wo.phase(ph, st, wrap)
        seen.append(check(dev, st, f"phase {ph}, round {sr}"))
    return seen


@pytest.mark.parametrize("move", [0, 0xFFFFFFFF])
@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("k,d,n_out,m", SHAPES)
def test_wrapped_phases_match_the_oracle(k, d, n_out, m, seed, move):
    """Every buffer bit for bit after phases 0, 1, 2, 2, 3 (direction: within 32 ulp), sentinel rows
    untouched; the walkers on the seam cross it."""
    rng = np.random.default_rng([k, d, n_out, m, seed % 1000, move & 1, 0xA7])
    st, w = wrapped_state(k, d, n_out, m, seed, move, rng)
    u0 = st.u.copy()
    seen = run_wrapped_move(st, w, WrappedDevice(st, w), fabricated(st, rng))
    b0 = seen[0]
    t = np.concatenate([b0["lo"][:k, None] - np.arange(n_out), b0["hi"][:k, None] + np.arange(n_out)], axis=1)
    p = u0[:, None, :] + t[:, :, None] * b0["dirn"][:k, None, :]
    crossed = ((p[..., w] < 0.0) | (p[..., w] >= 1.0)).any(axis=(1, 2))
    assert crossed[:min(k, 2)].all()
    c = b0["cand_out"][:k][..., w]
    assert np.all((c >= 0.0) & (c < 1.0))
    assert np.all((seen[-1]["u"][:k][:, w] >= 0.0) & (seen[-1]["u"][:k][:, w] < 1.0))


def test_all_zero_bits_are_the_unwrapped_kernels():
    """A mask without a bit (NULL or zeros) gives the same bits as rvl_slice_phase."""
    rng = np.random.default_rng(11)
    st = random_state(37, 33, 3, 6, 9, 4, rng)
    lls = fabricated(st, rng)
    plain = run_move(st.copy(), Device(st), lls, check_each=False)

    class Zero(WrappedDevice):
        def __init__(self, s, null):
            Device.__init__(self, s)
            self.bits = None if null else (ctypes.c_uint32 * 4)()
    for null in (True, False):
        got = run_move(st.copy(), Zero(st, null), lls, check_each=False)
        for a, b in zip(plain, got):
            for name in a:
                assert np.array_equal(a[name].view(np.uint8), b[name].view(np.uint8)), (null, name)


def _band_ball(d, R=0.3):
    """lnL = 0 on {u0 in [0.9, 1) or [0, 0.1)} x {|u_1.. - 0.5| < R}, -1 elsewhere."""
    def fused(U):
        import torch
        band = (U[:, 0] >= 0.9) | (U[:, 0] < 0.1)
        ball = ((U[:, 1:] - 0.5) ** 2).sum(1) < R * R
        return U.clone(), torch.where(band & ball, 0.0, -1.0).to(U.dtype)
    return fused


@pytest.mark.parametrize("wrap", [True, False])
def test_walkers_cross_the_seam(wrap):
    """All walkers start in [0.9, 1) of a band that wraps around to [0, 0.1): after 10 chained
    moves half of them are in [0, 0.1) and the band is filled uniformly.  Without the mask the
    walkers cannot reach the other half through the cube."""
    import torch
    from evidence_b200.sampler_dev import _NativeSlice
    k, d, R, nsteps = 4096, 3, 0.3, 10
    rng = np.random.default_rng(21)
    g = rng.standard_normal((k, d - 1))
    u0 = np.empty((k, d))
    u0[:, 0] = 0.9 + 0.1 * rng.uniform(size=k)
    u0[:, 1:] = 0.5 + R * rng.uniform(size=(k, 1)) ** (1.0 / (d - 1)) * g / np.linalg.norm(g, axis=1, keepdims=True)
    mask = np.array([True] + [False] * (d - 1)) if wrap else None
    ns = _NativeSlice(torch, k, d, torch.device("cuda"), 77, n_out=8, m=8, rounds=3, wrap=mask)
    u = torch.from_numpy(u0).cuda()
    theta, lcur = u.clone(), torch.full((k,), np.nan, dtype=torch.float64, device="cuda")
    ns.moves(_band_ball(d, R), u, theta, lcur, torch.tensor([-0.5], dtype=torch.float64, device="cuda"),
             torch.eye(d, dtype=torch.float64, device="cuda") * 0.1, nsteps)
    x = u.cpu().numpy()
    assert np.all((x[:, 0] >= 0.9) | (x[:, 0] < 0.1)) and np.all(((x[:, 1:] - 0.5) ** 2).sum(1) < R * R)
    unresolved, accepted = ns.stats.cpu().numpy().tolist()
    assert unresolved < 1e-3 * k * nsteps and unresolved + accepted == k * nsteps
    lower = int((x[:, 0] < 0.1).sum())
    if wrap:
        p_share = stats.binomtest(lower, k, 0.5).pvalue
        p_band = stats.kstest(wo.wrap_unit(x[:, 0] + 0.1) / 0.2, "uniform").pvalue
        assert p_share > 1e-3 and p_band > 1e-3, (lower / k, p_share, p_band)
    else:
        assert lower < 0.01 * k, lower / k


KAPPA, S = 50.0, 0.03
PERIODIC_LNZ = 2 * np.log(i0e(KAPPA)) + 3 * np.log(S * np.sqrt(2 * np.pi))


def periodic_fused(U):
    """Identity prior transform, d = 5: von Mises (kappa = 50) in 2 pi u_0, 2 pi u_1 with the mode on
    the seam, Gaussians of width 0.03 about 1/2 in u_2 .. u_4."""
    import torch
    ll = (KAPPA * (torch.cos(2 * np.pi * U[:, :2]) - 1.0)).sum(1) - ((U[:, 2:] - 0.5) ** 2).sum(1) / (2 * S * S)
    return U.clone(), ll


def test_device_sampler_on_a_periodic_problem():
    """ln Z = 2 ln i0e(kappa) + 3 ln(s sqrt(2 pi)) within 3 reported sigma for seeds 0-3, with the
    two von Mises coordinates wrapped; the posterior is one mode across the seam."""
    from evidence_b200.sampler_dev import nested_sample_device
    wrap = [True, True, False, False, False]
    for seed in range(4):
        r = nested_sample_device(periodic_fused, 5, nlive=200, seed=seed, device="cuda", wrapped=wrap)
        assert r.method.endswith("native") and r.wrapped.tolist() == wrap
        assert abs(r.logz - PERIODIC_LNZ) < 3 * r.logzerr, (seed, r.logz, r.logzerr, PERIODIC_LNZ)
        x = r.samples[:, 0]
        assert np.all((x >= 0) & (x < 1)) and np.mean(x < 0.1) > 0.3 and np.mean(x > 0.9) > 0.3
        assert r.unresolved_moves < 0.01 * r.accepted_moves


def omega_near_zero_case():
    """The first 1-planet synthetic case (config 1, 96 epochs, seeds from 100) whose true omega is
    within 0.3 rad of 0 = 2 pi and is measured: e >= 0.1 and K >= 10 m/s (seed 112: e = 0.12,
    omega = -0.23).  At smaller e only omega + M0 is constrained; that ridge wraps around in ma0
    too, which the reference's rule leaves unwrapped (profiles/r5_wrapped_sampler.txt, section 4)."""
    from evidence_b200 import synth
    for seed in range(100, 400):
        case = synth.make_case(1, seed=seed, n_epochs=96)
        t = case.truth
        w = t["planet1_omega"]
        if min(w, 2 * np.pi - w) < 0.3 and t["planet1_ecc"] >= 0.1 and t["planet1_k1"] >= 10.0:
            return case
    raise AssertionError("no case with omega near 0")


def test_rv_fit_with_omega_on_the_seam(tmp_path):
    """run() with builtin_method='slice-device' and builtin_wrap=True on an RV case whose omega
    posterior straddles 0 = 2 pi: the mask the runner derives reaches the kernels, the posterior of
    omega is one mode across the seam with every sample in [0, 2 pi), and the planet is found."""
    from evidence_b200 import ultranest as runner
    from evidence_b200.rvmodel import RVModel
    case = omega_near_zero_case()
    model = RVModel(case.fixedpardict, case.datadict(pandas=True), case.parnames)
    out = runner.run(model, {"target": "synth", "runid": "wrap", "save_dir": str(tmp_path), "nplanets": 1},
                     case.priordict, {"nlive": 200, "sampler": "builtin", "builtin_method": "slice-device",
                                      "builtin_wrap": True, "seed": 1})
    assert out.sampler_impl.endswith("wrapped: planet1_omega")
    assert np.isfinite(out.logZ) and 0 < out.logZerr < 2.0
    assert out.device_counters["n_points"] == out.nlike
    w = out.samples["planet1_omega"].to_numpy()
    assert np.all((w >= 0.0) & (w < 2 * np.pi))
    # both sides of the seam (the posterior is about -0.2 +- 0.2 rad: most of it below 2 pi)
    assert np.mean(w < 1.0) > 0.02 and np.mean(w > 2 * np.pi - 1.0) > 0.5
    mean = np.arctan2(np.sin(w).mean(), np.cos(w).mean())
    truth = case.truth["planet1_omega"]
    assert abs(np.angle(np.exp(1j * (mean - truth)))) < 0.5, (mean, truth)
    per = np.median(out.samples["planet1_period"])
    assert abs(per - case.truth["planet1_period"]) / case.truth["planet1_period"] < 0.02
    model.close()
