"""GPU (-m gpu): recorder traces of a whole population in one call (sgmm_rollout_trace_population, csrc/sgmm_trace_pop.cu).

Row i of every column must be bit-identical to sgmm_rollout_trace of individual i alone (the reference this file compares
against), whose columns in turn equal the C oracle's; fitness / trades equal the exact population rollout and the oracle.
Covered: H = 32 and 256, with and without the adversary, fee and phi settings, population sizes beyond the SM count, ragged
and chunk-crossing lengths, forced batching, seeded children and adversaries, the rounding-edge episodes of
tests/test_gpu_rounding_edges.py and tests/test_gpu_exact256.py, column subsets, output canaries, the device analytics of
backtest_population (the shipped ARL agent included) and the refusals.  The CPU tests (no marker) check the fixtures.
"""
import ctypes as C

import numpy as np
import pytest

F32 = np.float32
TICK = 0.001
PHI = 1e-4
FLIP = 0x8000000000000000
BATCH_ENV = "SGMM_EXACT256_BATCH_BYTES"
ADV_THR = F32(0.54930615)                         # largest fp32 y with round(tanh(y)) == 0 (tests/golden/tanh_threshold.npz)
ADV_ULP = np.nextafter(ADV_THR, F32(np.inf)) - ADV_THR
LARGE_K = [(1 << 22) - 1, 1 << 22, (1 << 22) + 5, 1 << 23, (1 << 24) + 3, (1 << 30) - 3]
DYADIC_LARGE_SCALE = F32(1 << 14)
ORACLE_COLS = ("off_a", "off_b", "adv_a", "adv_b", "fill_buy", "fill_sell", "inventory", "cash", "reward", "pnl_reward",
               "inventory_reward", "fee_paid", "raw_a", "raw_b")
ANALYTICS_COLS = ("wealth", "inventory", "fill_buy", "fill_sell")


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


def bits32(a):
    return np.asarray(a, np.float32).view(np.uint32)


def bits(a):
    a = np.asarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else (a.view(np.uint32) if a.dtype == np.float32 else a)


# ----------------------------------------------------------------------------------------------
# fixtures copied from tests/test_gpu_rounding_edges.py and tests/test_gpu_exact256.py: transparent policies (raw = scale *
# (z1, z2) exactly, for every inventory), boundary adversaries on the tanh threshold, scripted episodes
# ----------------------------------------------------------------------------------------------
def transparent_genome(hidden=32, scale=1.0, swap=False):
    H = hidden
    W1, b1 = np.zeros((H, 3), F32), np.zeros(H, F32)
    W2, b2 = np.zeros((H, H), F32), np.zeros(H, F32)
    W3, b3 = np.zeros((2, H), F32), np.zeros(2, F32)
    W1[0, 0], W1[1, 0], W1[2, 1], W1[3, 1] = 1, -1, 1, -1           # relu(z1), relu(-z1), relu(z2), relu(-z2)
    for j in range(4):
        W2[j, j] = 1
    a, b = (1, 0) if swap else (0, 1)
    W3[a, 0], W3[a, 1], W3[b, 2], W3[b, 3] = scale, -scale, scale, -scale
    return np.concatenate([W1.ravel(), b1, W2.ravel(), b2, W3.ravel(), b3]).astype(F32)


def boundary_adversary(sign_a, sign_b):
    g = np.zeros(1250, F32)
    g[1] = 1.0                              # h0 = relu(fill_sell_prev)
    g[5] = 1.0                              # h1 = relu(fill_buy_prev)
    g[48] = sign_a * ADV_ULP                # V2[0, 0]
    g[61] = sign_b * ADV_ULP                # V2[1, 1]
    g[72], g[73] = sign_a * ADV_THR, sign_b * ADV_THR
    return g


def genomes_of(hidden=32, scale=1.0):
    g0, g1 = transparent_genome(hidden, scale), transparent_genome(hidden, scale, swap=True)
    return np.stack([g0, g1, g0, g1])


def adversaries():
    return np.stack([boundary_adversary(1, -1), boundary_adversary(-1, 1), boundary_adversary(-1, 1), boundary_adversary(1, -1)])


def z_for(q):
    """An fp32 z with fl(z * 5) == q, or None."""
    q = F32(q)
    z = F32(q / F32(5))
    for d in range(-8, 9):
        c = z
        for _ in range(abs(d)):
            c = np.nextafter(c, F32(np.inf) if d > 0 else F32(-np.inf), dtype=F32)
        if F32(c * F32(5)) == q:
            return c
    return None


def quote_targets(K):
    out = []
    for c in (K + 0.5, K - 0.5):
        t = F32(c)
        out += [t, np.nextafter(t, F32(np.inf), dtype=F32), np.nextafter(t, F32(-np.inf), dtype=F32)]
    out.append(F32(K))
    return out


def _prices(rng, T, start_ticks=3500, step=0.001, decimals=3):
    bid_t = start_ticks + np.cumsum(rng.choice([-1, 0, 1], size=T))
    bid = np.round(bid_t * step, decimals)
    ask = np.round((bid_t + rng.choice([1, 2], size=T, p=[0.9, 0.1])) * step, decimals)
    mid = np.round((bid_t + rng.choice([-1, 0, 1, 2], size=T)) * step, decimals) + step / 2
    return mid, ask, bid


def touch_bounds(ask, bid, ka, kb, tick):
    return ask + ka.astype(np.float64) * tick, bid - kb.astype(np.float64) * tick


def _episode_ties(rng):
    T = 320
    mid, ask, bid = _prices(rng, T)
    ka, kb = rng.integers(-6, 7, size=T), rng.integers(-6, 7, size=T)
    z = np.zeros((2, T), F32)
    for t in range(T):
        for s, K in ((0, ka[t]), (1, kb[t])):
            while True:
                c = int(rng.integers(0, 7))
                zz = z_for(quote_targets(int(K))[c])
                if zz is not None:
                    break
                K = rng.integers(-6, 7)
                (ka if s == 0 else kb)[t] = K
            z[s, t] = zz
    for lo, side in ((40, 0), (90, 1), (200, 0), (260, 1)):        # inventory held at +-2
        for t in range(lo, lo + 12):
            (kb if side == 0 else ka)[t] = 6
            z[1 - side, t] = z_for(F32(-5.5 if t % 2 else -5.0))
    bmax, smin = touch_bounds(ask, bid, ka, kb, TICK)
    for lo, side in ((40, 0), (90, 1), (200, 0), (260, 1)):
        (bmax if side == 0 else smin)[lo:lo + 12] = np.nan
    special = rng.choice(np.arange(T), size=40, replace=False)
    kinds = [("a", np.nan), ("b", np.nan), ("a", np.inf), ("a", -np.inf), ("b", -np.inf), ("b", np.inf)]
    for i, t in enumerate(special):
        side, v = kinds[i % len(kinds)]
        (bmax if side == "a" else smin)[t] = v
    return dict(z1=z[0], z2=z[1], mid=mid, ask=ask, bid=bid, bmax=bmax, smin=smin, scale=F32(1))


def _episode_large(rng):
    T = 260
    mid, ask, bid = _prices(rng, T)
    ka, kb = rng.integers(-6, 7, size=T), rng.integers(-6, 7, size=T)
    z = np.zeros((2, T), F32)
    for t in range(T):
        z[0, t] = z_for(F32(rng.integers(-6, 7)))
        z[1, t] = z_for(F32(rng.integers(-6, 7)))
    cases = [(sgn * K0, c) for K0 in LARGE_K for sgn in (1, -1)
             for c in quote_targets(sgn * K0) + [F32(sgn * K0 + 1), F32(sgn * K0 - 1)]]
    cases = [(K, c, z_for(c)) for K, c in cases if abs(float(c)) <= (1 << 30)]
    for t, (K, c, zz) in enumerate([x for x in cases if x[2] is not None]):
        s = t % 2
        (ka if s == 0 else kb)[t] = K
        z[s, t] = zz
    bmax, smin = touch_bounds(ask, bid, ka, kb, TICK)
    return dict(z1=z[0], z2=z[1], mid=mid, ask=ask, bid=bid, bmax=bmax, smin=smin, scale=F32(1))


def _episode_dyadic(rng):
    T = 300
    mid, ask, bid = _prices(rng, T)
    z = (rng.integers(-32, 33, size=(2, T)) / 8.0).astype(F32)
    tie = rng.random((2, T)) < 0.5
    z[tie] = (rng.choice([-7, -5, -3, -1, 1, 3, 5, 7], size=int(tie.sum())) / 2.0).astype(F32)
    q = z * F32(5)
    k = np.rint(q).astype(np.int64) + rng.choice([-1, 0, 0, 1], size=(2, T))
    bmax, smin = touch_bounds(ask, bid, k[0], k[1], TICK)
    special = rng.choice(np.arange(T), size=30, replace=False)
    for i, t in enumerate(special):
        (bmax if i % 2 == 0 else smin)[t] = [np.nan, np.inf, -np.inf][i % 3]
    return dict(z1=z[0], z2=z[1], mid=mid, ask=ask, bid=bid, bmax=bmax, smin=smin, scale=F32(1))


def _episode_dyadic_large(rng):
    """|q| from 40 960 ticks to ~2^30 and (scale 2^14 * 13056 * 5) beyond K_CLAMP."""
    T = 240
    mid, ask, bid = _prices(rng, T)
    mags = [0.5, 51.0, 51.25, 102.5, 205.0, 3328.0, 13056.0]
    z = (rng.choice(mags, size=(2, T)) * rng.choice([-1, 1], size=(2, T))).astype(F32)
    q = (z * DYADIC_LARGE_SCALE) * F32(5)
    k = q.astype(np.int64) + rng.choice([-1, 0, 1], size=(2, T))
    lim = rng.random((2, T)) < 0.2
    k[lim] = rng.choice([K * s for K in LARGE_K for s in (1, -1)], size=int(lim.sum()))
    bmax, smin = touch_bounds(ask, bid, k[0], k[1], TICK)
    return dict(z1=z[0], z2=z[1], mid=mid, ask=ask, bid=bid, bmax=bmax, smin=smin, scale=DYADIC_LARGE_SCALE)


def make_episode(name):
    """dyadic_huge: the dyadic_large episode under policies of twice its scale, |q| up to 2.14e9 ticks (exactly), beyond
    K_CLAMP = 2^30 but inside int32 (the offsets' type)."""
    if name == "dyadic_huge":
        return dict(make_episode("dyadic_large"), scale=F32(2) * DYADIC_LARGE_SCALE)
    rng = np.random.default_rng({"ties": 11, "large": 12, "dyadic": 13, "dyadic_large": 14}[name])
    return {"ties": _episode_ties, "large": _episode_large, "dyadic": _episode_dyadic,
            "dyadic_large": _episode_dyadic_large}[name](rng)


def edge_episode_h256(seed=7):
    """tests/test_gpu_exact256.py: q on K +- 0.5 ties, thresholds up to near K_CLAMP with q on and around them, NaN / inf bounds."""
    rng = np.random.default_rng(seed)
    cases = [(K, c) for K in range(-6, 7) for c in quote_targets(K)]
    cases += [(s * K0, c) for K0 in LARGE_K for s in (1, -1) for c in quote_targets(s * K0) + [F32(s * K0 + 1), F32(s * K0 - 1)]]
    cases = [(K, z_for(c)) for K, c in cases if abs(float(c)) <= (1 << 30)]
    cases = [(K, z) for K, z in cases if z is not None]
    T = 2 * len(cases) + 40
    bid_t = 3500 + np.cumsum(rng.choice([-1, 0, 1], size=T))
    bid = np.round(bid_t * TICK, 3)
    ask = np.round((bid_t + rng.choice([1, 2], size=T, p=[0.9, 0.1])) * TICK, 3)
    mid = np.round((bid_t + rng.choice([-1, 0, 1, 2], size=T)) * TICK, 3) + TICK / 2
    ka, kb = rng.integers(-6, 7, size=T), rng.integers(-6, 7, size=T)
    z = np.array([[z_for(F32(k)) for k in rng.integers(-6, 7, size=T)] for _ in range(2)], F32)
    for i, (K, zz) in enumerate(cases):
        t, s = 2 * i + (i % 2), i % 2
        (ka if s == 0 else kb)[t] = K
        z[s, t] = zz
    bmax, smin = ask + ka.astype(np.float64) * TICK, bid - kb.astype(np.float64) * TICK
    for i, t in enumerate(rng.choice(np.arange(T), size=24, replace=False)):
        (bmax if i % 2 == 0 else smin)[t] = [np.nan, np.inf, -np.inf][i % 3]
    return (z[0], z[1], mid, ask, bid, bmax, smin)


def bz_of(ep):
    return (ep["z1"], ep["z2"], ep["mid"], ep["ask"], ep["bid"], ep["bmax"], ep["smin"])


# ----------------------------------------------------------------------------------------------
# CPU: the fixtures are what they claim
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hidden", [32, 256])
def test_transparent_policy_outputs_its_inputs(hidden):
    from oracle import oracle as orc
    ep = make_episode("ties")
    g0, g1 = transparent_genome(hidden), transparent_genome(hidden, swap=True)
    for t in range(0, ep["z1"].size, 7):
        for iv in range(5):
            x = [ep["z1"][t], ep["z2"][t], (iv - 2) / 2.0]
            want = np.array([ep["z1"][t], ep["z2"][t]], F32)
            assert np.array_equal(bits32(orc.mlp_forward(g0, x, hidden=hidden)), bits32(want))
            assert np.array_equal(bits32(orc.mlp_forward(g1, x, hidden=hidden)), bits32(want[::-1]))


def test_episodes_reach_ties_and_beyond_k_clamp():
    q = np.concatenate([make_episode("ties")["z1"], make_episode("ties")["z2"]]) * F32(5)
    for K in (-5, -4, 4, 5):
        assert (q == F32(K + 0.5)).any() and (q == F32(K - 0.5)).any()
    ep = make_episode("dyadic_huge")
    z = np.concatenate([ep["z1"], ep["z2"]])
    ql = np.abs((z * ep["scale"]) * F32(5))
    assert (ql > (1 << 30)).any() and (ql < (1 << 31)).all()
    assert np.array_equal(ql.astype(np.float64), np.abs(z.astype(np.float64) * float(ep["scale"]) * 5))    # exact
    bz = edge_episode_h256()
    assert np.isnan(bz[5]).any() and np.isinf(bz[6]).any()


# ----------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sg():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import sgmm_b200
    return sgmm_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


_BUNDLES = {}


def synthetic(sg, orc, T):
    """A synthetic bundle of exactly T bars (cached per module)."""
    if T not in _BUNDLES:
        from sgmm_b200 import synthetic as syn
        days = max(1, -(-T // syn.BARS_PER_DAY))
        bundle = syn.synthetic_bundle(days, first_day=80)
        stats = syn.train_stats_of(bundle)
        bundle = tuple(a[:T] for a in bundle)
        z1, z2 = orc.normalise(bundle, stats)
        _BUNDLES[T] = (sg.Bundle.from_arrays(bundle, stats, TICK), (z1, z2) + tuple(bundle[2:]), bundle)
    return _BUNDLES[T]


def genomes(P, seed, hidden=32, out_scale=4.0):
    from sgmm_b200 import synthetic as syn
    return syn.policy_like_genomes(P, hidden=hidden, seed=seed, out_scale=out_scale, out_bias=(0.1, 0.1))[1]


def adv_genomes(P, seed):
    return (np.random.default_rng(seed).standard_normal((P, 1250)) * 0.6).astype(F32)


def check_rows(sg, bun, G, A, fit, trd, cols, *, phi, fee, hidden=32, rows=None):
    """Row i of every returned column, fitness[i] and trades[i] equal rollout_trace of individual i alone, bit for bit."""
    fit, trd = fit.cpu().numpy(), trd.cpu().numpy()
    host = {k: v.cpu().numpy() for k, v in cols.items()}
    for i in (range(len(G)) if rows is None else rows):
        f1, t1, tr1 = sg.rollout_trace(bun, G[i], None if A is None else A[i], phi=phi, fee_rate=fee, hidden=hidden)
        assert (bits64(fit[i]), trd[i]) == (bits64(f1), t1), i
        for k, v in host.items():
            assert np.array_equal(bits(v[i]), bits(tr1[k])), (i, k)


def check_oracle(orc, bz, G, A, fit, trd, cols, *, phi, fee, hidden=32, rows=None):
    """The oracle's columns, the derived columns computed from them, fitness / trades of its population rollout."""
    fo, to = orc.rollout_population(bz, phi, TICK, fee, genomes=G, adv_genomes=A, use_adv=A is not None, hidden=hidden, nthreads=8)
    assert np.array_equal(bits64(fit.cpu().numpy()), bits64(fo)) and np.array_equal(trd.cpu().numpy(), to)
    mid, ask, bid = (np.asarray(bz[k], np.float64) for k in (2, 3, 4))
    host = {k: v.cpu().numpy() for k, v in cols.items()}
    for i in (range(len(G)) if rows is None else rows):
        f1, t1, tro = orc.rollout(G[i], None if A is None else A[i], bz, phi, TICK, fee, hidden=hidden, trace=True)
        for k in ORACLE_COLS:
            assert np.array_equal(bits(host[k][i]), bits(tro[k])), (i, k)
        inv = tro["inventory"].astype(np.float64)
        assert np.array_equal(bits64(host["spread"][i]), bits64(ask - bid))
        assert np.array_equal(bits64(host["unrealized_pnl"][i]), bits64(inv * mid))
        assert np.array_equal(bits64(host["wealth"][i]), bits64(tro["cash"] + inv * mid))
        assert np.array_equal(bits64(host["cum_reward"][i]), bits64(np.cumsum(tro["reward"])))
        assert np.array_equal(bits64(host["cum_fees"][i]), bits64(np.cumsum(tro["fee_paid"])))
        assert np.array_equal(host["skew"][i], tro["off_b"] - tro["off_a"])


def cuda(x):
    import torch
    return None if x is None else torch.from_numpy(np.ascontiguousarray(x)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("use_adv", [False, True])
@pytest.mark.parametrize("fee", [0.0, 3e-4, -1e-4])
@pytest.mark.parametrize("phi", [0.0, 1e-4, 0.01])
def test_h32_rows_fee_phi(sg, orc, use_adv, fee, phi):
    bun, bz, _ = synthetic(sg, orc, 300)
    G = genomes(3, seed=1)
    A = adv_genomes(3, seed=1) if use_adv else None
    fit, trd, cols = sg.rollout_trace_population(bun, cuda(G), cuda(A), phi=phi, fee_rate=fee)
    assert sorted(cols) == sorted(n for n, _ in sg._lib.Trace._fields_)
    check_rows(sg, bun, G, A, fit, trd, cols, phi=phi, fee=fee)
    check_oracle(orc, bz, G, A, fit, trd, cols, phi=phi, fee=fee)
    fe, te = sg.rollout_population(bun, cuda(G), cuda(A), phi=phi, fee_rate=fee, precision="exact")
    assert fe.equal(fit) and te.equal(trd)
    assert trd.cpu().numpy().min() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("T", [0, 1, 2, 127, 1000, 2049])
@pytest.mark.parametrize("P", [1, 3, 33, 149])
def test_h32_sizes_and_lengths(sg, orc, P, T):
    bun, bz, _ = synthetic(sg, orc, T)
    assert bun.T == T
    G = genomes(P, seed=P + T)
    A = adv_genomes(P, seed=P + T)
    for adv in (None, A):
        fit, trd, cols = sg.rollout_trace_population(bun, cuda(G), cuda(adv), phi=PHI, fee_rate=3e-4)
        assert all(v.shape == (P, T) for v in cols.values())
        check_rows(sg, bun, G, adv, fit, trd, cols, phi=PHI, fee=3e-4)
        fe, te = sg.rollout_population(bun, cuda(G), cuda(adv), phi=PHI, fee_rate=3e-4)
        assert fe.equal(fit) and te.equal(trd)
        if T > 0:
            check_oracle(orc, bz, G, adv, fit, trd, cols, phi=PHI, fee=3e-4, rows=[0, P - 1])


@pytest.mark.gpu
@pytest.mark.parametrize("P", [3, 149])
def test_h32_full_length_episode(sg, orc, P):
    bun, bz, _ = synthetic(sg, orc, 14400)
    G = genomes(P, seed=P, out_scale=3.0)
    A = adv_genomes(P, seed=P)
    for adv in (None, A):
        fit, trd, cols = sg.rollout_trace_population(bun, cuda(G), cuda(adv), phi=PHI, fee_rate=3e-4)
        rows = range(P) if P <= 3 else [0, 1, 47, 100, P - 1]
        check_rows(sg, bun, G, adv, fit, trd, cols, phi=PHI, fee=3e-4, rows=rows)
        check_oracle(orc, bz, G, adv, fit, trd, cols, phi=PHI, fee=3e-4, rows=[0, P - 1])
        assert trd.cpu().numpy().min() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("use_adv", [False, True])
def test_h256_rows(sg, orc, use_adv):
    bun, bz, _ = synthetic(sg, orc, 300)
    G = genomes(5, seed=4, hidden=256)
    A = adv_genomes(5, seed=4) if use_adv else None
    fit, trd, cols = sg.rollout_trace_population(bun, cuda(G), cuda(A), phi=PHI, fee_rate=3e-4, hidden=256)
    check_rows(sg, bun, G, A, fit, trd, cols, phi=PHI, fee=3e-4, hidden=256)
    check_oracle(orc, bz, G, A, fit, trd, cols, phi=PHI, fee=3e-4, hidden=256)
    fe, te = sg.rollout_population(bun, cuda(G), cuda(A), phi=PHI, fee_rate=3e-4, hidden=256, precision="exact")
    assert fe.equal(fit) and te.equal(trd)


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [32, 256])
@pytest.mark.parametrize("use_adv", [False, True])
def test_several_batches_equal_one(sg, orc, hidden, use_adv, monkeypatch):
    bun, bz, _ = synthetic(sg, orc, 200)
    P = 7
    G = genomes(P, seed=5, hidden=hidden)
    A = adv_genomes(P, seed=5) if use_adv else None
    kw = dict(phi=PHI, fee_rate=3e-4, hidden=hidden)
    seeded = dict(master=cuda(G[0]), count=P, sigma=0.05, seed=3, generation=1, first_index=2,
                  adv_master=None if A is None else cuda(A[0]), adv_sigma=0.1)
    whole = sg.rollout_trace_population(bun, cuda(G), cuda(A), **kw)
    whole_s = sg.rollout_trace_population(bun, **seeded, **kw)
    monkeypatch.setenv(BATCH_ENV, str(200 * 40 * 2 + 1))            # two individuals' tables per batch: 4 batches
    parts = sg.rollout_trace_population(bun, cuda(G), cuda(A), **kw)
    monkeypatch.setenv(BATCH_ENV, "1")                              # one individual per batch (H = 256 seeded: + staged genome)
    parts_s = sg.rollout_trace_population(bun, **seeded, **kw)
    for x, y in ((whole, parts), (whole_s, parts_s)):
        assert x[0].equal(y[0]) and x[1].equal(y[1])
        assert all(x[2][k].equal(y[2][k]) for k in x[2])
    check_oracle(orc, bz, G, A, *parts, phi=PHI, fee=3e-4, hidden=hidden, rows=[0, P - 1])


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [32, 256])
def test_seeded_children_equal_explicit(sg, orc, hidden):
    bun, bz, _ = synthetic(sg, orc, 300)
    master = genomes(1, seed=8, hidden=hidden)[0]
    am = adv_genomes(1, seed=8)[0]
    P, seed, gen, first = 6, 77, 4, 10
    kids = np.stack([orc.mutate(master, 0.05, seed, gen, first + i) for i in range(P)])
    akids = np.stack([orc.mutate(am, 0.1, seed ^ FLIP, gen, first + i) for i in range(P)])
    for adv in (False, True):
        fs, ts, cs = sg.rollout_trace_population(bun, master=cuda(master), count=P, sigma=0.05, seed=seed, generation=gen,
                                                 first_index=first, adv_master=cuda(am) if adv else None, adv_sigma=0.1,
                                                 phi=PHI, fee_rate=3e-4, hidden=hidden)
        A = akids if adv else None
        fe, te, ce = sg.rollout_trace_population(bun, cuda(kids), cuda(A), phi=PHI, fee_rate=3e-4, hidden=hidden)
        assert fs.equal(fe) and ts.equal(te) and all(cs[k].equal(ce[k]) for k in cs)
        fo, to = orc.rollout_population(bz, PHI, TICK, 3e-4, master=master, sigma=0.05, seed=seed, generation=gen,
                                        first_index=first, count=P, adv_master=am if adv else None, adv_sigma=0.1,
                                        use_adv=adv, hidden=hidden)
        assert np.array_equal(bits64(fs.cpu().numpy()), bits64(fo)) and np.array_equal(ts.cpu().numpy(), to)
        check_rows(sg, bun, kids, A, fs, ts, cs, phi=PHI, fee=3e-4, hidden=hidden, rows=[0, 3])


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "fee", "adv"])
@pytest.mark.parametrize("name", ["ties", "large", "dyadic", "dyadic_large", "dyadic_huge"])
def test_rounding_edges_h32(sg, orc, name, variant):
    ep = make_episode(name)
    fee = 3e-4 if variant == "fee" else 0.0
    G = genomes_of(32, ep["scale"])
    A = adversaries() if variant == "adv" else None
    bun = sg.Bundle(*bz_of(ep), TICK)
    fit, trd, cols = sg.rollout_trace_population(bun, cuda(G), cuda(A), phi=PHI, fee_rate=fee)
    check_rows(sg, bun, G, A, fit, trd, cols, phi=PHI, fee=fee)
    check_oracle(orc, bz_of(ep), G, A, fit, trd, cols, phi=PHI, fee=fee)
    if A is not None:
        assert (cols["adv_a"].cpu().numpy() != 0).any() and (cols["adv_b"].cpu().numpy() != 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "fee", "adv"])
def test_rounding_edges_h256(sg, orc, variant):
    bz = edge_episode_h256()
    fee = 3e-4 if variant == "fee" else 0.0
    G = genomes_of(256)
    A = adversaries() if variant == "adv" else None
    bun = sg.Bundle(*bz, TICK)
    fit, trd, cols = sg.rollout_trace_population(bun, cuda(G), cuda(A), phi=PHI, fee_rate=fee, hidden=256)
    check_rows(sg, bun, G, A, fit, trd, cols, phi=PHI, fee=fee, hidden=256)
    check_oracle(orc, bz, G, A, fit, trd, cols, phi=PHI, fee=fee, hidden=256)


SUBSETS = [(), ("wealth",), ("cash",), ("cum_fees",), ("cum_reward", "skew"), ANALYTICS_COLS, ("raw_a", "adv_b", "fee_paid"),
           ("cash", "wealth", "cum_fees", "unrealized_pnl")]


@pytest.mark.gpu
@pytest.mark.parametrize("use_adv", [False, True])
def test_column_subsets_and_canaries(sg, orc, use_adv):
    import torch
    L = sg._lib
    bun, bz, _ = synthetic(sg, orc, 2100)
    T, P, pad = bun.T, 5, 64
    G = genomes(P, seed=2)
    A = adv_genomes(P, seed=2) if use_adv else None
    fit0, trd0, full = sg.rollout_trace_population(bun, cuda(G), cuda(A), phi=PHI, fee_rate=3e-4)
    names = [n for n, _ in L.Trace._fields_]
    g, a = cuda(G), cuda(A)
    canary = {torch.int32: -3, torch.float32: -3.5, torch.float64: 12345.5}
    for subset in SUBSETS + [(n,) for n in names]:
        bufs = {}
        for n in names:                                             # every column between canaries; only the subset is passed
            buf = torch.full((P * T + 2 * pad,), canary[full[n].dtype], dtype=full[n].dtype, device="cuda")
            bufs[n] = buf
        tr = L.Trace(*[bufs[n][pad:].data_ptr() if n in subset else None for n in names])
        fit = torch.full((P + 2 * pad,), 12345.5, dtype=torch.float64, device="cuda")
        trd = torch.full((P + 2 * pad,), -777, dtype=torch.int32, device="cuda")
        mm = L.Population(32, 0, P, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
        ap = None if a is None else C.byref(L.Population(32, 0, P, a.data_ptr(), None, 0.0, 0.0, 0, 0, 0))
        L.check(L.lib().sgmm_rollout_trace_population(bun.handle, C.byref(mm), ap, C.byref(L.RolloutParams(PHI, 3e-4, 0, 0, 0, 0)),
                                                      C.byref(tr), fit[pad:].data_ptr(), trd[pad:].data_ptr(), None))
        torch.cuda.synchronize()
        for n, buf in bufs.items():
            c = canary[buf.dtype]
            if n in subset:
                assert (buf[:pad] == c).all() and (buf[pad + P * T:] == c).all(), (subset, n)
                assert torch.equal(buf[pad:pad + P * T].view(P, T), full[n]), (subset, n)
            else:
                assert (buf == c).all(), (subset, n)                 # not passed: untouched
        assert (fit[:pad] == 12345.5).all() and (fit[pad + P:] == 12345.5).all() and torch.equal(fit[pad:pad + P], fit0)
        assert (trd[:pad] == -777).all() and (trd[pad + P:] == -777).all() and torch.equal(trd[pad:pad + P], trd0)
    # trace == NULL: fitness and trades only
    fit = torch.empty(P, dtype=torch.float64, device="cuda")
    trd = torch.empty(P, dtype=torch.int32, device="cuda")
    mm = L.Population(32, 0, P, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    ap = None if a is None else C.byref(L.Population(32, 0, P, a.data_ptr(), None, 0.0, 0.0, 0, 0, 0))
    L.check(L.lib().sgmm_rollout_trace_population(bun.handle, C.byref(mm), ap, C.byref(L.RolloutParams(PHI, 3e-4, 4, 0, 0, 0)),
                                                  None, fit.data_ptr(), trd.data_ptr(), None))
    assert torch.equal(fit, fit0) and torch.equal(trd, trd0)
    f2, t2, c2 = sg.rollout_trace_population(bun, g, a, phi=PHI, fee_rate=3e-4, columns=("wealth", "raw_b"))
    assert sorted(c2) == ["raw_b", "wealth"] and c2["wealth"].equal(full["wealth"]) and c2["raw_b"].equal(full["raw_b"])


def _summary_of_row(sg, bun, bundle, g, a, phi, fee, hidden=32):
    from sgmm_b200 import StrategyRecorder
    _, _, tr = sg.rollout_trace(bun, g, a, phi=phi, fee_rate=fee, hidden=hidden)
    df = StrategyRecorder.from_trace(tr, bundle).to_dataframe()
    df["is_trade"] = (df["fill_buy"] != 0) | (df["fill_sell"] != 0)
    return df


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [32, 256])
def test_backtest_population_summary(sg, orc, hidden):
    from sgmm_b200.analytics import KEYS
    bun, bz, bundle = synthetic(sg, orc, 1500)
    P = 4
    G = genomes(P, seed=6, hidden=hidden)
    A = adv_genomes(P, seed=6)
    for adv in (None, A):
        fit, trd, summ = sg.backtest_population(bun, cuda(G), cuda(adv), phi=PHI, fee_rate=3e-4, hidden=hidden)
        fe, te, _ = sg.rollout_trace_population(bun, cuda(G), cuda(adv), phi=PHI, fee_rate=3e-4, hidden=hidden, columns=())
        assert fit.equal(fe) and trd.equal(te)
        s = summ.cpu().numpy()
        for i in range(P):
            df = _summary_of_row(sg, bun, bundle, G[i], None if adv is None else adv[i], PHI, 3e-4, hidden)
            want = sg.StrategyAnalytics(df).summary_dict
            assert np.array_equal(bits64(s[i]), bits64([want[k] for k in KEYS])), i
            o = orc.analytics(df["wealth"].to_numpy(), df["inventory"].to_numpy(), df["is_trade"].to_numpy())
            assert np.array_equal(bits64(s[i]), bits64(o)), i
    # the row of a population trace, moved to numpy, is a valid StrategyRecorder.from_trace argument
    _, _, cols = sg.rollout_trace_population(bun, cuda(G), phi=PHI, fee_rate=3e-4, hidden=hidden)
    from sgmm_b200 import StrategyRecorder
    df = StrategyRecorder.from_trace({k: v[1].cpu().numpy() for k, v in cols.items()}, bundle).to_dataframe()
    ref = _summary_of_row(sg, bun, bundle, G[1], None, PHI, 3e-4, hidden)
    for k in ("off_a", "inventory", "cash", "wealth", "cum_reward", "cum_fees", "realized_pnl", "unrealized_pnl"):
        assert np.array_equal(bits(df[k].to_numpy()), bits(ref[k].to_numpy())), k


@pytest.mark.gpu
def test_backtest_population_with_shipped_arl_agent(sg, orc, golden):
    """The shipped ARL agent on its golden backtest bundle (tests/test_gpu_parity.py), in a population with DRL-like agents."""
    b, c = golden.backtest, golden.ckpt
    s1, s2 = b["arl.s1_pred"], b["arl.s2_pred"]
    z1 = ((s1 - c["train_stats_s1_m"][()]) / c["train_stats_s1_s"][()]).astype(np.float32)
    z2 = ((s2 - c["train_stats_s2_m"][()]) / c["train_stats_s2_s"][()]).astype(np.float32)
    fb, fs = b["arl.fill_buy"], b["arl.fill_sell"]
    my_ask = b["arl.ask"] + b["arl.off_a"] * 0.001
    my_bid = b["arl.bid"] - b["arl.off_b"] * 0.001
    arrays = (z1, z2, b["arl.mid"], b["arl.ask"], b["arl.bid"],
              np.where(fs == 1, my_ask, my_ask - 0.0005), np.where(fb == 1, my_bid, my_bid + 0.0005))
    bun = sg.Bundle(*arrays, 0.001)
    G = np.concatenate([c["510300_with_adv"].reshape(1, -1).astype(F32), genomes(3, seed=9)])
    fit, trd, summ = sg.backtest_population(bun, cuda(G), phi=1e-4)
    _, _, cols = sg.rollout_trace_population(bun, cuda(G), phi=1e-4)
    assert np.array_equal(cols["off_a"][0].cpu().numpy(), b["arl.off_a"])
    assert np.array_equal(cols["inventory"][0].cpu().numpy(), b["arl.inventory"])
    assert np.array_equal(bits64(cols["cash"][0].cpu().numpy()), bits64(b["arl.cash"]))
    host = (s1, s2) + arrays[2:]
    s = summ.cpu().numpy()
    for i in range(len(G)):
        df = _summary_of_row(sg, bun, host, G[i], None, 1e-4, 0.0)
        want = sg.StrategyAnalytics(df).summary_dict
        assert np.array_equal(bits64(s[i]), bits64([want[k] for k in sg.analytics.KEYS])), i
        o = orc.analytics(df["wealth"].to_numpy(), df["inventory"].to_numpy(), df["is_trade"].to_numpy())
        assert np.array_equal(bits64(s[i]), bits64(o)), i
    f1, t1, _ = sg.rollout_trace(bun, G[0], phi=1e-4)
    assert (bits64(fit[0].item()), trd[0].item()) == (bits64(f1), t1)


@pytest.mark.gpu
def test_refusals(sg, orc):
    import torch
    L = sg._lib
    bun, _, _ = synthetic(sg, orc, 40)
    G = genomes(2, seed=1)
    g = cuda(G)
    a = cuda(adv_genomes(3, seed=1))
    f = torch.empty(3, dtype=torch.float64, device="cuda")
    t = torch.empty(3, dtype=torch.int32, device="cuda")
    run = L.lib().sgmm_rollout_trace_population
    mm = L.Population(32, 0, 2, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    for prec in (1, 2, 3):                                          # BF16, TF32, F16
        rc = run(bun.handle, C.byref(mm), None, C.byref(L.RolloutParams(PHI, 0.0, prec, 0, 0, 0)), None, f.data_ptr(), t.data_ptr(), None)
        assert rc == L.ERR_UNSUPPORTED and b"SGMM_PRECISION_EXACT" in L.lib().sgmm_last_error(), prec
    f32, exact = L.RolloutParams(PHI, 0.0, 0, 0, 0, 0), L.RolloutParams(PHI, 0.0, 4, 0, 0, 0)
    for hidden in (64, 128):
        gh = torch.zeros(2, hidden * hidden + 7 * hidden + 2, dtype=torch.float32, device="cuda")
        mh = L.Population(hidden, 0, 2, gh.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
        for prm in (f32, exact):
            assert run(bun.handle, C.byref(mh), None, C.byref(prm), None, f.data_ptr(), t.data_ptr(), None) == L.ERR_UNSUPPORTED
    ap = L.Population(32, 0, 3, a.data_ptr(), None, 0.0, 0.0, 0, 0, 0)           # adv.count != mm.count
    assert run(bun.handle, C.byref(mm), C.byref(ap), C.byref(f32), None, f.data_ptr(), t.data_ptr(), None) == L.ERR_INVALID
    assert run(None, C.byref(mm), None, C.byref(f32), None, f.data_ptr(), t.data_ptr(), None) == L.ERR_INVALID
    assert run(bun.handle, C.byref(mm), None, None, None, f.data_ptr(), t.data_ptr(), None) == L.ERR_INVALID
    assert run(bun.handle, C.byref(mm), None, C.byref(f32), None, None, t.data_ptr(), None) == L.ERR_INVALID
    assert run(bun.handle, C.byref(mm), None, C.byref(f32), None, f.data_ptr(), None, None) == L.ERR_INVALID
    m0 = L.Population(32, 0, 0, None, None, 0.0, 0.0, 0, 0, 0)                    # count == 0: nothing to do
    assert run(bun.handle, C.byref(m0), None, C.byref(f32), None, None, None, None) == L.OK
    fit, trd, cols = sg.rollout_trace_population(bun, torch.zeros(0, 1250, device="cuda"), phi=PHI)
    assert fit.numel() == 0 and all(v.shape == (0, 40) for v in cols.values())
    with pytest.raises(ValueError):
        sg.rollout_trace_population(bun, g, phi=PHI, columns=("wealth", "nope"))
    with pytest.raises(ValueError):
        sg.rollout_trace_population(bun, g, master=g[0], phi=PHI)
    # F32 and EXACT give the same trace at H = 32 and at H = 256
    g256 = cuda(genomes(2, seed=3, hidden=256))
    for gg, hidden in ((g, 32), (g256, 256)):
        outs = []
        for prec in (0, 4):
            mh = L.Population(hidden, 0, 2, gg.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
            w = torch.empty(2, 40, dtype=torch.float64, device="cuda")
            tr = L.Trace(*[w.data_ptr() if n == "wealth" else None for n, _ in L.Trace._fields_])
            L.check(run(bun.handle, C.byref(mh), None, C.byref(L.RolloutParams(PHI, 0.0, prec, 0, 0, 0)), C.byref(tr),
                        f.data_ptr(), t.data_ptr(), None))
            outs.append((w.clone(), f[:2].clone()))
        assert outs[0][0].equal(outs[1][0]) and outs[0][1].equal(outs[1][1])
