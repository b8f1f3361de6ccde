"""
The slice-sampler kernels of evidence_b200/csrc/rvslice.cu (`rvl_slice_phase`) against their host
restatement, oracle/slice_oracle.py, buffer by buffer after every phase.

The likelihood values the kernels read (`ll_out`, `cand_ll`, `cand_th`) are made up by the tests, so
no likelihood code is involved.  The direction is compared within a few ulp (the device's log, sin
and cos are not correctly rounded); the oracle then continues from the device's direction and every
other buffer must be bit-identical.  Every per-walker buffer has PAD extra rows of a sentinel that
must survive every phase.
"""
import ctypes

import numpy as np
import pytest

from oracle import slice_oracle as so

PAD = 4
SENTINEL = {np.float64: -7.25e300, np.uint8: 0xA5, np.int32: 0x5A5A5A5A, np.uint64: 0xDEADBEEF}
LMIN = 0.25

# buffer -> (shape of one walker's rows, dtype); stats ([2]) is padded the same way
PER_WALKER = {
    "u": ("d",), "theta": ("d",), "lcur": (), "dirn": ("d",), "lo": (), "hi": (), "lo2": (),
    "hi2": (), "tval": ("m",), "pending": (), "cand_out": ("2n", "d"), "inside_out": ("2n",),
    "ll_out": ("2n",), "cand": ("m", "d"), "inside": ("m",), "cand_ll": ("m",),
    "cand_th": ("m", "d"),
}
DTYPE = {"pending": np.int32, "inside_out": np.uint8, "inside": np.uint8}


def _dims(st, shape):
    return tuple({"d": st.d, "m": st.m, "2n": 2 * st.n_out}[s] for s in shape)


def random_state(k, d, n_out, m, seed, move, rng, chol_scale=0.15):
    """Inputs and scratch of k walkers; scratch holds junk that the kernels must overwrite or keep."""
    chol = np.tril(rng.normal(0.0, 0.3 * chol_scale / np.sqrt(d), (d, d)), -1)
    chol += np.diag(rng.uniform(0.5, 1.0, d) * chol_scale)
    chol[np.triu_indices(d, 1)] = np.nan  # the kernel reads only l <= j
    junk = lambda *s: rng.normal(0.0, 3.0, s)  # noqa: E731
    return so.SliceState(
        k=k, d=d, n_out=n_out, m=m, seed=seed, move=move, shrink_round=0, lmin=LMIN, chol=chol,
        u=rng.uniform(0.02, 0.98, (k, d)), theta=junk(k, d), lcur=junk(k), dirn=junk(k, d),
        lo=junk(k), hi=junk(k), lo2=junk(k), hi2=junk(k), tval=junk(k, m),
        pending=np.full(k, 7, np.int32), cand_out=junk(k, 2 * n_out, d),
        inside_out=np.full((k, 2 * n_out), 0x77, np.uint8), ll_out=junk(k, 2 * n_out),
        cand=junk(k, m, d), inside=np.full((k, m), 0x77, np.uint8), cand_ll=junk(k, m),
        cand_th=junk(k, m, d), stats=np.array([5, 9], np.uint64))


def fake_ll(rng, shape, p_success):
    """lnL values around LMIN: above it with probability p_success (including +inf), else below it,
    exactly equal, NaN or -inf."""
    above = rng.choice([LMIN + 1.0, np.nextafter(LMIN, 1.0), np.inf], shape, p=[0.8, 0.1, 0.1])
    below = rng.choice([LMIN - 1.0, LMIN, np.nextafter(LMIN, 0.0), np.nan, -np.inf], shape)
    return np.where(rng.uniform(size=shape) < p_success, above, below)


class Device:
    """Device buffers of one SliceState, with PAD sentinel rows, and rvl_slice_phase on them."""

    def __init__(self, st):
        import torch
        from evidence_b200 import _abi
        self.torch, self.lib, self.st0 = torch, _abi.load(), st
        self.buf = {}
        for name, shape in PER_WALKER.items():
            dt = DTYPE.get(name, np.float64)
            host = np.full((st.k + PAD,) + _dims(st, shape), SENTINEL[dt], dt)
            host[:st.k] = getattr(st, name)
            self.buf[name] = torch.from_numpy(host).cuda()
        stats = np.full(2 + PAD, SENTINEL[np.uint64], np.uint64)
        stats[:2] = st.stats
        self.buf["stats"] = torch.from_numpy(stats.view(np.int64)).cuda()
        self.chol = torch.from_numpy(np.ascontiguousarray(st.chol)).cuda()
        self.lmin = torch.tensor([st.lmin], dtype=torch.float64, device="cuda")
        a = self.args = _abi.rvl_slice_args()
        a.k, a.d, a.n_out, a.m, a.seed = st.k, st.d, st.n_out, st.m, st.seed
        a.lmin, a.chol = self.lmin.data_ptr(), self.chol.data_ptr()
        for name, t in self.buf.items():
            setattr(a, name, t.data_ptr())

    def set(self, name, values):
        self.buf[name][:self.st0.k] = self.torch.from_numpy(np.ascontiguousarray(values)).cuda()

    def phase(self, ph, move, shrink_round):
        self.args.move, self.args.shrink_round = move, shrink_round
        rc = self.lib.rvl_slice_phase(ph, ctypes.byref(self.args),
                                      self.torch.cuda.current_stream().cuda_stream)
        assert rc == 0, self.lib.rvl_slice_last_error().decode()
        self.torch.cuda.synchronize()

    def read(self):
        out = {n: t.cpu().numpy() for n, t in self.buf.items()}
        out["stats"] = out["stats"].view(np.uint64)
        return out


def same_bits(a, b):
    """Bit-identical, except that any NaN equals any NaN."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    if a.dtype != np.float64:
        return np.array_equal(a, b)
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.int64),
                                                               b[~nan].view(np.int64))


def dirn_tolerance(st, z):
    """32 2^-53 sum_l |chol_jl z_l| / |z| per element (z: the oracle's normals)."""
    terms = np.abs(np.nan_to_num(np.tril(st.chol))[None, :, :] * z[:, None, :]).sum(-1)
    return 32 * 2.0 ** -53 * terms / np.sqrt((z * z).sum(1))[:, None]


def check(dev, st, where):
    """Every buffer of the device equals the oracle's; the sentinel rows are untouched."""
    got = dev.read()
    for name, g in got.items():
        if name == "stats":
            assert same_bits(g[:2], st.stats), (where, name, g[:2], st.stats)
            assert np.all(g[2:] == SENTINEL[np.uint64]), (where, name)
            continue
        want = getattr(st, name)
        rows = g[:st.k].reshape(want.shape)
        if name != "dirn":
            bad = ~np.array([same_bits(r, w) for r, w in zip(rows, want)])
            assert not bad.any(), (where, name, np.nonzero(bad)[0][:8], rows[bad][:2], want[bad][:2])
        assert np.all(g[st.k:] == SENTINEL[g.dtype.type]), (where, name, "write past row k")
    return got


def run_move(st, dev, lls, check_each=True):
    """Phases 0 -> 1 -> 2 -> 2 -> 3 on the device and on the oracle, the made-up likelihoods of each
    phase from lls(phase_no) -> {buffer: values}.  Returns the device buffers after each phase."""
    seen = []
    dev.phase(0, st.move, 0)
    d_dirn = dev.read()["dirn"][:st.k]
    z, own = so.phase(0, st, dirn=d_dirn)
    assert np.all(np.abs(d_dirn - own) <= dirn_tolerance(st, z)), "direction off by more than 32 ulp"
    seen.append(check(dev, st, "phase 0") if check_each else dev.read())
    for i, (ph, sr) in enumerate([(1, 0), (2, 1), (2, 2), (3, 3)]):
        for name, v in lls(i).items():
            dev.set(name, v)
            setattr(st, name, v.copy())
        st.shrink_round = sr
        dev.phase(ph, st.move, sr)
        so.phase(ph, st)
        seen.append(check(dev, st, f"phase {ph}, round {sr}") if check_each else dev.read())
    return seen


def fabricated(st, rng, p_out=0.6, p_cand=0.2):
    draws = [{"ll_out": fake_ll(rng, (st.k, 2 * st.n_out), p_out)}]
    for _ in range(3):
        draws.append({"cand_ll": fake_ll(rng, (st.k, st.m), p_cand),
                      "cand_th": rng.normal(size=(st.k, st.m, st.d))})
    return lambda i: draws[i]


SHAPES = [(1, 1, 1, 1), (5, 7, 8, 8), (64, 32, 4, 6), (37, 33, 3, 64), (9, 128, 2, 5), (130, 3, 16, 1)]
SEEDS = [0, 1, 2 ** 32 + 7, 2 ** 64 - 1]


@pytest.mark.gpu
@pytest.mark.parametrize("move", [0, 0xFFFFFFFF])
@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("k,d,n_out,m", SHAPES)
def test_phases_match_the_oracle(k, d, n_out, m, seed, move):
    rng = np.random.default_rng([k, d, n_out, m, seed % 1000, move & 1])
    st = random_state(k, d, n_out, m, seed, move, rng)
    run_move(st, Device(st), fabricated(st, rng))


T = LMIN + 1.0
UP, DOWN = np.nextafter(LMIN, 1.0), np.nextafter(LMIN, 0.0)
NAN, NINF, PINF = np.nan, -np.inf, np.inf


@pytest.mark.gpu
def test_likelihood_patterns():
    """Runs of successes end at the first failure; lnL == lmin, NaN and -inf fail; the first
    candidate above lmin is accepted, whatever follows it."""
    k, d, n_out, m = 5, 3, 4, 4
    st = random_state(k, d, n_out, m, 99, 3, np.random.default_rng(1), chol_scale=0.01)
    st.u[:] = 0.5  # every candidate inside the cube
    ll_out = np.array([
        [T, 0.0, T, T, T, T, T, T],            # lo: 1, hi: 4
        [0.0, T, T, T, T, T, 0.0, T],          # 0, 2
        [LMIN, T, T, T, T, NAN, T, T],         # 0, 1
        [T, T, NINF, T, PINF, PINF, PINF, 0.0],  # 2, 3
        [UP, 0.0, T, T, DOWN, T, T, T],        # 1, 0
    ])
    runs_lo, runs_hi = np.array([1, 0, 0, 2, 1]), np.array([4, 2, 1, 3, 0])
    cand_ll = [
        np.array([[LMIN, NAN, NINF, 1.3], [0.0] * 4, [2.0, 2.1, 2.2, 2.3], [0.0, LMIN, UP, 3.3],
                  [NAN] * 4]),
        np.array([[9.0] * 4, [0.0, 1.1, 1.2, 1.3], [9.0] * 4, [9.0] * 4, [NINF, LMIN, DOWN, NAN]]),
    ]
    th = [np.random.default_rng(i).normal(size=(k, m, d)) for i in range(2)]
    rounds = [{"ll_out": ll_out}, {"cand_ll": cand_ll[0], "cand_th": th[0]},
              {"cand_ll": cand_ll[1], "cand_th": th[1]}]
    dev = Device(st)
    dev.phase(0, st.move, 0)
    b0 = dev.read()
    so.phase(0, st, dirn=b0["dirn"][:k])
    check(dev, st, "phase 0")
    assert np.all(b0["inside_out"][:k] == 1)
    for i, (ph, sr) in enumerate([(1, 0), (2, 1), (3, 2)]):
        for name, v in rounds[i].items():
            dev.set(name, v)
            setattr(st, name, v.copy())
        before = dev.read()
        st.shrink_round = sr
        dev.phase(ph, st.move, sr)
        so.phase(ph, st)
        after = check(dev, st, f"phase {ph}")
        if ph == 1:
            assert np.array_equal(after["lo"][:k], b0["lo"][:k] - runs_lo)
            assert np.array_equal(after["hi"][:k], b0["hi"][:k] + runs_hi)
        elif ph == 2:  # walker 0 takes candidate 3, 2 candidate 0, 3 candidate 2; 1 and 4 go on
            assert after["pending"][:k].tolist() == [0, 1, 0, 0, 1]
            for w, j in ((0, 3), (2, 0), (3, 2)):
                assert same_bits(after["u"][w], before["cand"][w, j])
                assert same_bits(after["theta"][w], th[0][w, j])
                assert after["lcur"][w] == cand_ll[0][w, j]
            for w in (1, 4):
                assert after["lo"][w] == before["lo2"][w] and after["hi"][w] == before["hi2"][w]
        else:  # walker 1 takes candidate 1; walker 4 is left unresolved and keeps its position
            assert after["pending"][:k].tolist() == [0, 0, 0, 0, 1]
            assert same_bits(after["u"][1], before["cand"][1, 1]) and after["lcur"][1] == 1.1
            assert same_bits(after["u"][4], b0["u"][4]) and same_bits(after["theta"][4], b0["theta"][4])
            assert same_bits(after["lcur"][4], b0["lcur"][4])
            assert after["stats"][:2].tolist() == [5 + 1, 9 + 4]


@pytest.mark.gpu
def test_cube_boundary_is_exact():
    """A zero row of chol makes dirn[j] = 0, so p_j = u_j for every candidate: u_j = 1.0 is outside
    (and never accepted, although lnL > lmin), u_j = 0.0 inside.  j = d - 1 >= 32, so only the
    warp-wide vote sees it."""
    k, d, n_out, m = 8, 40, 3, 4
    st = random_state(k, d, n_out, m, 7, 11, np.random.default_rng(2), chol_scale=0.01)
    st.chol[d - 1, :d] = 0.0
    st.u[:, :] = 0.5
    st.u[0::2, d - 1] = 1.0
    st.u[1::2, d - 1] = 0.0
    out = k // 2
    seen = run_move(st, Device(st), lambda i: ({"ll_out": np.full((k, 2 * n_out), T)} if i == 0 else
                                               {"cand_ll": np.full((k, m), T),
                                                "cand_th": np.full((k, m, d), float(i))}))
    b0, b1, _, _, b3 = seen
    assert np.all(b0["dirn"][:k, d - 1] == 0.0)
    ins = b0["inside_out"][:k]
    assert np.all(ins[0::2] == 0) and np.all(ins[1::2] == 1)
    c = b0["cand_out"][:k, :, d - 1]
    assert np.all(c[0::2] == 1.0 - 2.0 ** -53) and np.all(c[1::2] == 0.0)
    # the walkers inside step out the whole n_out on both sides; the others not at all
    assert np.array_equal((b0["lo"] - b1["lo"])[:k], np.tile([0.0, n_out], out))
    assert np.all(b1["inside"][:k][0::2] == 0)
    # the inside walkers accept their first candidate, with u[d-1] still exactly 0
    assert b3["pending"][:k].tolist() == [1, 0] * out
    assert np.all(b3["u"][1:k:2, d - 1] == 0.0) and np.all(b3["theta"][1:k:2] == 1.0)
    assert same_bits(b3["u"][0:k:2], st.u[0::2]) and np.all(b3["u"][0:k:2, d - 1] == 1.0)
    assert b3["stats"][:2].tolist() == [5 + out, 9 + out]


@pytest.mark.gpu
def test_launch_shape_independence_and_repeatability():
    """The first 5 walkers give the same bits at k = 5 and k = 64, and a rerun the same bits."""
    rng = np.random.default_rng(5)
    big = random_state(64, 9, 4, 6, 2 ** 40 + 3, 12, rng)
    lls = fabricated(big, rng)
    small = big.copy()
    small.k = 5
    for name in PER_WALKER:
        setattr(small, name, getattr(big, name)[:5].copy())
    runs = [run_move(s.copy(), Device(s), f, check_each=False)
            for s, f in ((big, lls), (big, lls),
                         (small, lambda i: {n: v[:5] for n, v in lls(i).items()}))]
    for a, b, c in zip(*runs):
        for name in PER_WALKER:
            assert same_bits(a[name], b[name]), name
            assert same_bits(a[name][:5], c[name][:5]), name


@pytest.mark.gpu
def test_seeds_draw_independent_streams():
    """No bracket draw of one seed reappears under another seed (k = 64, phase 0): seeds 1..4,
    s and s ^ 1, s and s + 2^32."""
    k = 64

    def draws(seed):
        st = random_state(k, 3, 1, 1, seed, 0, np.random.default_rng(0))
        dev = Device(st)
        dev.phase(0, 0, 0)
        return dev.read()["hi"][:k]
    s = 0x0123456789ABCDEF
    for group in ([1, 2, 3, 4], [s, s ^ 1], [s, s + 2 ** 32]):
        hs = {seed: draws(seed) for seed in group}
        for a in group:
            for b in group:
                if a < b:
                    shared = np.intersect1d(hs[a], hs[b])
                    assert len(shared) == 0, (f"seeds {a} and {b} share {len(shared)} of their {k} "
                                              "bracket draws")


def _host_gauss(pts):
    ll = -0.5 * (((pts - 0.5) / 0.15) ** 2).sum(1)
    return 3.0 * pts - 1.0, ll


@pytest.mark.gpu
def test_whole_move_through_the_driver():
    """_NativeSlice.moves (nsteps = 1, 3 shrinkage rounds) with a host likelihood equals the oracle
    rerun from the kernel's direction: u, theta, lcur and stats bit for bit."""
    import torch
    from evidence_b200.sampler_dev import _NativeSlice
    k, d, n_out, m, seed = 50, 6, 4, 5, 2024
    rng = np.random.default_rng(8)
    u0 = 0.5 + rng.uniform(-0.1, 0.1, (k, d))
    th0, l0 = _host_gauss(u0)
    lmin = float(np.quantile(l0, 0.3))

    def fused(U):
        th, ll = _host_gauss(U.cpu().numpy())
        return torch.from_numpy(th).cuda(), torch.from_numpy(ll).cuda()
    chol = np.linalg.cholesky(np.diag(np.full(d, 0.02)) + 0.005)
    ns = _NativeSlice(torch, k, d, torch.device("cuda"), seed, n_out=n_out, m=m, rounds=3)
    ns.move = 17
    u, theta = torch.from_numpy(u0.copy()).cuda(), torch.from_numpy(th0.copy()).cuda()
    lcur = torch.full((k,), np.nan, dtype=torch.float64, device="cuda")
    ns.moves(fused, u, theta, lcur, torch.tensor([lmin], dtype=torch.float64, device="cuda"),
             torch.from_numpy(chol).cuda(), 1)
    torch.cuda.synchronize()

    st = random_state(k, d, n_out, m, seed, 17, rng)
    st.lmin, st.chol, st.u, st.theta = lmin, chol, u0.copy(), th0.copy()
    st.lcur, st.stats = np.full(k, np.nan), np.zeros(2, np.uint64)
    so.phase(0, st, dirn=ns.dirn.cpu().numpy())
    _, st.ll_out = _host_gauss(st.cand_out.reshape(-1, d))
    st.ll_out = st.ll_out.reshape(k, 2 * n_out)
    so.phase(1, st)
    for r in range(3):
        th, ll = _host_gauss(st.cand.reshape(-1, d))
        st.cand_th, st.cand_ll = th.reshape(k, m, d), ll.reshape(k, m)
        st.shrink_round = r + 1
        so.phase(2 if r < 2 else 3, st)
    assert same_bits(u.cpu().numpy(), st.u) and same_bits(theta.cpu().numpy(), st.theta)
    assert same_bits(lcur.cpu().numpy(), st.lcur)
    assert ns.stats.cpu().numpy().view(np.uint64).tolist() == st.stats.tolist()
    moved = np.isfinite(st.lcur)
    assert moved.sum() > k // 2 and np.all(st.lcur[moved] > lmin)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [2, 5])
def test_moves_keep_the_uniform_distribution_on_a_ball(d):
    """Walkers uniform in a ball of radius 0.3 at the centre of the cube (the region lnL > lmin) stay
    uniform over 10 chained moves: (r / R)^d and the angle in the (x0, x1) plane stay uniform.  The
    stepping-out cap (8 unit steps of length 0.15 per side) never binds."""
    import torch
    from scipy import stats
    from evidence_b200.sampler_dev import _NativeSlice
    k, R, nsteps = 4096, 0.3, 10
    rng = np.random.default_rng(d)
    g = rng.standard_normal((k, d))
    u0 = 0.5 + R * rng.uniform(size=(k, 1)) ** (1.0 / d) * g / np.linalg.norm(g, axis=1, keepdims=True)

    def fused(U):
        return U, -((U - 0.5) ** 2).sum(1)
    ns = _NativeSlice(torch, k, d, torch.device("cuda"), 123, n_out=8, m=8, rounds=3)
    u = torch.from_numpy(u0).cuda()
    theta, lcur = u.clone(), torch.full((k,), np.nan, dtype=torch.float64, device="cuda")
    ns.moves(fused, u, theta, lcur, torch.tensor([-R * R], dtype=torch.float64, device="cuda"),
             torch.eye(d, dtype=torch.float64, device="cuda") * 0.15, nsteps)
    x = u.cpu().numpy() - 0.5
    r = np.linalg.norm(x, axis=1)
    unresolved, accepted = ns.stats.cpu().numpy().tolist()
    assert np.all(r < R * (1 + 1e-12))
    assert unresolved < 1e-3 * k * nsteps and unresolved + accepted == k * nsteps
    assert np.mean(np.abs(x - (u0 - 0.5)).max(1) > 0) > 0.999  # (almost) every walker moved
    p_r = stats.kstest((r / R) ** d, "uniform").pvalue
    p_a = stats.kstest(np.mod(np.arctan2(x[:, 1], x[:, 0]), 2 * np.pi) / (2 * np.pi), "uniform").pvalue
    assert p_r > 1e-3 and p_a > 1e-3, (p_r, p_a)


@pytest.mark.parametrize("field,value,phase", [("k", 0, 0), ("d", 129, 0), ("n_out", 0, 1),
                                               ("m", 65, 2), (None, None, 4)])
def test_argument_validation(built_lib, field, value, phase):
    """Bad sizes or phase: RVL_EINVAL and a message, before anything reaches the device."""
    from evidence_b200 import _abi
    lib = _abi.load()
    a = _abi.rvl_slice_args()
    a.k, a.d, a.n_out, a.m = 4, 3, 2, 2
    if field:
        setattr(a, field, value)
    assert lib.rvl_slice_phase(phase, ctypes.byref(a), None) == -1  # RVL_EINVAL
    msg = lib.rvl_slice_last_error().decode()
    assert ("phase must be" if field is None else "bad sizes") in msg
