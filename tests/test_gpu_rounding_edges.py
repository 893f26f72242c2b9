"""Every rollout route at the inputs where rounding code goes wrong: quotes exactly on a rounding tie, one ulp either
side of it, adversary outputs exactly on and just beyond the tanh rounding boundary, NaN / infinite bounds, fill
thresholds of millions of ticks up to K_CLAMP, and operating points other than tick 0.001 / phi 1e-4.

The policies are TRANSPARENT: W1 copies +z1, -z1, +z2, -z2 into hidden units 0-3, W2 is the identity on them and W3 takes
the differences, so in SGMM-F32 order raw = s * (z1, z2) exactly for every inventory.  The bundle's signals then choose
q = raw*5 bar by bar, and its bounds choose the integer fill thresholds (Ka, Kb) bar by bar.

Episodes:
  ties          |K| <= 6, q on K +- 0.5 (even and odd K, both signs), one ulp either side, exactly K; NaN and +-inf bounds;
                inventory driven to +-2.  Exact routes bitwise; tensor-core routes: outputs within TAU and, given the
                offsets they took, the env bit for bit.
  large         thresholds +-(2^22 - 1), +-2^22, +-(2^22 + 5), +-2^23, +-(2^24 + 3) and near K_CLAMP, q on and around
                them.  Exact routes bitwise (z needs the full fp32 mantissa here: out of the tensor-core routes' range).
  dyadic        z in 1/8 Z (q in 0.625 Z: ties at +-2.5, +-7.5, ...).  Every product and sum on the bf16 / f16 / tf32
                paths is exact, so EVERY route equals the oracle bit for bit in closed loop.
  dyadic_large  8-bit z times W3 = 2^14: q of millions of ticks up to 2^30, thresholds one tick either side.  Every
                route equals the oracle bit for bit in closed loop.

The CPU tests (no marker) check on the oracle that each fixture is what it claims to be.
"""
import numpy as np
import pytest

ADV_THR = np.float32(0.54930615)                  # largest fp32 y with round(tanh(y)) == 0 (tests/golden/tanh_threshold.npz)
ADV_ULP = np.nextafter(ADV_THR, np.float32(np.inf)) - ADV_THR
TAU = {"bf16": 0.12, "tf32": 0.03, "f16": 0.03}   # tests/test_gpu_tc32.py
TAU_256 = 0.05                                    # tests/test_gpu_spec256.py
TICK = 0.001
PHI = 1e-4
LARGE_K = [(1 << 22) - 1, 1 << 22, (1 << 22) + 5, 1 << 23, (1 << 24) + 3, (1 << 30) - 3]
DYADIC_LARGE_SCALE = np.float32(1 << 14)
EPISODES = ("ties", "large", "dyadic", "dyadic_large")
TENSOR_EPISODES = ("ties", "dyadic", "dyadic_large")
VARIANTS = {"plain": (0.0, False), "fee": (3e-4, False), "adv": (0.0, True)}
F32 = np.float32


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


def bits32(a):
    return np.asarray(a, np.float32).view(np.uint32)


# ----------------------------------------------------------------------------------------------
# fixtures: transparent policies, boundary adversaries, scripted episodes
# ----------------------------------------------------------------------------------------------
def transparent_genome(hidden=32, scale=1.0, swap=False):
    """raw = scale * (z1, z2) (or (z2, z1) with ``swap``) for every inventory, exactly (models/model.py:31-36 layout)."""
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
    """AdversaryPolicy (models/model.py:40-50) whose output y_a is ADV_THR after a bar without a sell fill and the next float
    beyond it after one (sign_a = +1: displacement 0 / +1; -1: the mirror, 0 / -1); y_b likewise driven by fill_buy_prev."""
    g = np.zeros(1250, F32)
    g[3 * 0 + 1] = 1.0                      # h0 = relu(fill_sell_prev)
    g[3 * 1 + 2] = 1.0                      # h1 = relu(fill_buy_prev)
    g[48 + 0] = sign_a * ADV_ULP            # V2[0, 0]
    g[48 + 12 + 1] = sign_b * ADV_ULP       # V2[1, 1]
    g[72], g[73] = sign_a * ADV_THR, sign_b * ADV_THR
    return g


def genomes_of(hidden=32, scale=1.0):
    g0, g1 = transparent_genome(hidden, scale), transparent_genome(hidden, scale, swap=True)
    return np.stack([g0, g1, g0, g1])


def adversaries():
    return np.stack([boundary_adversary(1, -1), boundary_adversary(-1, 1), boundary_adversary(-1, 1), boundary_adversary(1, -1)])


def z_for(q):
    """An fp32 z with fl(z * 5) == q, or None (not every fp32 q is a product of 5)."""
    q = F32(q)
    z = F32(q / F32(5))
    for d in range(-8, 9):
        c = z
        for _ in range(abs(d)):
            c = np.nextafter(c, F32(np.inf) if d > 0 else F32(-np.inf), dtype=F32)
        if F32(c * F32(5)) == q:
            return c
    return None


def rint_even(q):
    return int(np.rint(np.float64(q)))


def quote_targets(K):
    """q on and around K's rounding boundaries: K + 0.5, K - 0.5, one ulp either side of each, and K itself
    (fp32-rounded where the value is not representable)."""
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
    """Bounds whose integer thresholds are ka / kb: the quote at the threshold itself (fl(best +- fl(k*tick)),
    market_env.py:30-31)."""
    return ask + ka.astype(np.float64) * tick, bid - kb.astype(np.float64) * tick


def _episode_ties(rng):
    """~300 bars, |K| <= 6, every quote category, NaN / inf bounds, inventory gates."""
    T = 320
    mid, ask, bid = _prices(rng, T)
    ka, kb = rng.integers(-6, 7, size=T), rng.integers(-6, 7, size=T)
    z = np.zeros((2, T), F32)
    cat = np.zeros((2, T), np.int32)
    for t in range(T):
        for s, K in ((0, ka[t]), (1, kb[t])):
            while True:
                c = int(rng.integers(0, 7))
                zz = z_for(quote_targets(int(K))[c])
                if zz is not None:
                    break
                K = rng.integers(-6, 7)
                (ka if s == 0 else kb)[t] = K
            z[s, t], cat[s, t] = zz, c
    # runs that push the inventory to +-2 and hold it there: one side never fills (NaN bound), the other always could
    for lo, side in ((40, 0), (90, 1), (200, 0), (260, 1)):
        for t in range(lo, lo + 12):
            (kb if side == 0 else ka)[t] = 6
            z[1 - side, t] = z_for(F32(-5.5 if t % 2 else -5.0))
            cat[1 - side, t] = -1
    bmax, smin = touch_bounds(ask, bid, ka, kb, TICK)
    for lo, side in ((40, 0), (90, 1), (200, 0), (260, 1)):
        (bmax if side == 0 else smin)[lo:lo + 12] = np.nan
    special = rng.choice(np.arange(T), size=40, replace=False)
    kinds = [("a", np.nan), ("b", np.nan), ("a", np.inf), ("a", -np.inf), ("b", -np.inf), ("b", np.inf)]
    for i, t in enumerate(special):
        side, v = kinds[i % len(kinds)]
        (bmax if side == "a" else smin)[t] = v
    return dict(z1=z[0], z2=z[1], mid=mid, ask=ask, bid=bid, bmax=bmax, smin=smin, scale=F32(1), cat=cat)


def _episode_large(rng):
    """Thresholds of millions of ticks, q on and around them (|q| <= 2^30), both signs; small bars in between."""
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
        s = t % 2                                                   # alternate sides: ask on even bars, bid on odd ones
        (ka if s == 0 else kb)[t] = K
        z[s, t] = zz
    assert len(cases) < T
    bmax, smin = touch_bounds(ask, bid, ka, kb, TICK)
    return dict(z1=z[0], z2=z[1], mid=mid, ask=ask, bid=bid, bmax=bmax, smin=smin, scale=F32(1))


def _episode_dyadic(rng):
    """z in 1/8 Z within [-4, 4]: q in 0.625 Z with ties at +-2.5, +-7.5, +-12.5, +-17.5; thresholds on both sides
    of the rounded value so that the rounding decides the fill."""
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
    """8-bit z times W3 = 2^14: |q| from 40 960 ticks to ~2^30; thresholds at q - 1, q, q + 1 and at the listed limits."""
    T = 240
    mid, ask, bid = _prices(rng, T)
    mags = [0.5, 51.0, 51.25, 102.5, 205.0, 3328.0, 13056.0]       # at most 8 significant bits, < 2^15 (f16 range)
    z = (rng.choice(mags, size=(2, T)) * rng.choice([-1, 1], size=(2, T))).astype(F32)
    q = (z * DYADIC_LARGE_SCALE) * F32(5)
    k = q.astype(np.int64) + rng.choice([-1, 0, 1], size=(2, T))
    lim = rng.random((2, T)) < 0.2
    k[lim] = rng.choice([K * s for K in LARGE_K for s in (1, -1)], size=int(lim.sum()))
    bmax, smin = touch_bounds(ask, bid, k[0], k[1], TICK)
    return dict(z1=z[0], z2=z[1], mid=mid, ask=ask, bid=bid, bmax=bmax, smin=smin, scale=DYADIC_LARGE_SCALE)


def make_episode(name):
    rng = np.random.default_rng({"ties": 11, "large": 12, "dyadic": 13, "dyadic_large": 14}[name])
    return {"ties": _episode_ties, "large": _episode_large, "dyadic": _episode_dyadic,
            "dyadic_large": _episode_dyadic_large}[name](rng)


def bz_of(ep):
    return (ep["z1"], ep["z2"], ep["mid"], ep["ask"], ep["bid"], ep["bmax"], ep["smin"])


def brute_thresholds(ep, tick=TICK):
    """(Ka, Kb) from the reference's fp64 quotes (market_env.py:30-31,37-38) by brute force around the real-arithmetic
    solution: INT32_MIN never, INT32_MAX always (the prologue's K_CLAMP = 2^30 search range)."""
    imin, imax, clamp = np.iinfo(np.int32).min, np.iinfo(np.int32).max, 1 << 30

    def one(best, bound, ask):
        quote = (lambda k: best + np.float64(k) * tick) if ask else (lambda k: best - np.float64(k) * tick)
        touch = (lambda k: quote(k) <= bound) if ask else (lambda k: quote(k) >= bound)
        if not touch(-clamp):
            return imin
        if touch(clamp):
            return imax
        e = int(np.floor((bound - best) / tick if ask else (best - bound) / tick))
        ks = [k for k in range(e - 8, e + 9) if touch(k)]
        assert ks and not touch(max(ks) + 1) and max(ks) < e + 8
        return max(ks)

    ka = np.array([one(a, b, True) for a, b in zip(ep["ask"], ep["bmax"])], np.int64)
    kb = np.array([one(b, s, False) for b, s in zip(ep["bid"], ep["smin"])], np.int64)
    return ka, kb


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


@pytest.fixture(scope="module")
def episodes():
    return {n: make_episode(n) for n in EPISODES}


# ----------------------------------------------------------------------------------------------
# CPU: each fixture is what it claims to be (checked on the oracle)
# ----------------------------------------------------------------------------------------------
def test_tie_quotes_exist_for_small_thresholds(orc):
    for K in range(-6, 7):
        z = z_for(K + 0.5)
        assert z is not None and F32(z * F32(5)) == F32(K + 0.5), K
        assert orc.quantise([z, z])[0] == (K if K % 2 == 0 else K + 1)          # half to even
    assert F32(F32(0.1) * F32(5)) == 0.5 and z_for(0.5) == F32(0.1)
    assert F32(F32(-0.90000004) * F32(5)) == -4.5 and z_for(-4.5) == F32(-0.90000004)
    for z, k in ((2.5, 12), (-2.5, -12), (1.5, 8), (-1.5, -8), (0.5, 2), (-0.5, -2)):  # dyadic ties
        assert F32(z) * F32(5) == F32(z * 5) and orc.quantise([z / 1.0, 0.0])[0] == k


@pytest.mark.parametrize("hidden", [32, 256])
def test_transparent_policy_outputs_its_inputs(orc, episodes, hidden):
    for name, ep in episodes.items():
        g0, g1 = transparent_genome(hidden, ep["scale"]), transparent_genome(hidden, ep["scale"], swap=True)
        for t in range(0, ep["z1"].size, 7 if hidden == 256 else 1):
            for iv in range(5):
                x = [ep["z1"][t], ep["z2"][t], (iv - 2) / 2.0]
                want = np.array([ep["z1"][t], ep["z2"][t]], F32) * ep["scale"]
                assert np.array_equal(bits32(orc.mlp_forward(g0, x, hidden=hidden)), bits32(want)), (name, t, iv)
                assert np.array_equal(bits32(orc.mlp_forward(g1, x, hidden=hidden)), bits32(want[::-1])), (name, t, iv)


def test_boundary_adversary_sits_on_the_tanh_threshold(orc):
    T_BITS, BEYOND = 0x3F0C9F54, 0x3F0C9F55
    assert bits32(ADV_THR) == T_BITS
    for sa, sb in ((1, -1), (-1, 1)):
        g = boundary_adversary(sa, sb)
        for inv in range(-2, 3):
            for fs in (0, 1):
                for fb in (0, 1):
                    pre, d = orc.adv_forward(g, [inv / 2.0, float(fs), float(fb)])
                    assert bits32(abs(pre[0])) == (BEYOND if fs else T_BITS) and np.sign(pre[0]) == sa
                    assert bits32(abs(pre[1])) == (BEYOND if fb else T_BITS) and np.sign(pre[1]) == sb
                    assert d.tolist() == [sa * fs, sb * fb]


@pytest.mark.parametrize("name", EPISODES)
def test_scripted_episode_covers_its_cases(orc, episodes, name):
    ep = episodes[name]
    ka, kb = brute_thresholds(ep)
    imin, imax = np.iinfo(np.int32).min, np.iinfo(np.int32).max
    qa, qb = ep["z1"] * ep["scale"] * F32(5), ep["z2"] * ep["scale"] * F32(5)
    assert np.abs(qa).max() <= (1 << 30) and np.abs(qb).max() <= (1 << 30)
    fo, to, tr = orc.rollout(transparent_genome(32, ep["scale"]), None, bz_of(ep), PHI, TICK, 0.0, trace=True)
    assert np.array_equal(tr["off_a"], [rint_even(q) for q in qa]) and np.array_equal(tr["off_b"], [rint_even(q) for q in qb])
    fs, fb = tr["fill_sell"] == 1, tr["fill_buy"] == 1
    if name in ("ties", "dyadic"):
        assert ((ka == imin).sum() > 0) and ((ka == imax).sum() > 0) and ((kb == imin).sum() > 0) and ((kb == imax).sum() > 0)
        assert np.isnan(ep["bmax"]).any() and np.isnan(ep["smin"]).any()
        assert tr["inventory"].max() == 2 and tr["inventory"].min() == -2 and (fs & fb).any()
        inv_prev = np.concatenate([[0], tr["inventory"][:-1]])
        assert ((inv_prev == 2) & (tr["off_b"] <= kb)).any() and ((inv_prev == -2) & (tr["off_a"] <= ka)).any()  # gated
        # the tie rule decides fills: rounding half away from zero would fill differently on some bars
        away = lambda q: (np.sign(q) * np.floor(np.abs(q).astype(np.float64) + 0.5)).astype(np.int64)
        ties_a = (qa - np.floor(qa) == 0.5)
        assert ((away(qa) <= ka) != (tr["off_a"] <= ka))[ties_a].any()
        assert ((away(qb) <= kb) != (tr["off_b"] <= kb))[qb - np.floor(qb) == 0.5].any()
    if name == "ties":
        for s, (q, K) in enumerate(((qa, ka), (qb, kb))):
            fin = np.abs(K) <= 6
            for K0 in (-5, -4, 4, 5):                                     # even and odd, both signs, every category
                for c in range(7):
                    sel = fin & (K == K0) & (ep["cat"][s] == c)
                    if sel.any():
                        assert np.all(q[sel] == quote_targets(K0)[c])
            cats = set(ep["cat"][s][fin & (np.abs(K) >= 1)].tolist())
            assert cats >= set(range(7)), (s, cats)
            for parity in (0, 1):
                for sgn in (1, -1):
                    sel = fin & (K % 2 == parity) & (np.sign(K) == sgn) & (q == K + F32(0.5))
                    assert sel.any(), (s, parity, sgn)
    if name == "large":
        for K0 in LARGE_K:
            for K in (K0, -K0):
                sel = np.concatenate([ka == K, kb == K])
                q = np.concatenate([qa, qb])[sel].astype(np.float64)
                assert sel.sum() >= 3 and (q >= K).any() and (q < K).any(), K
        # the |K| >= 2^22 cases where filling is decided by one half tick
        for K, q in (((1 << 22) + 5, (1 << 22) + 5.5), (-(1 << 23), -(1 << 23) + 0.5)):   # q on the tie beyond the threshold
            assert (((qa == F32(q)) & (ka == K)) | ((qb == F32(q)) & (kb == K))).any()
        assert fs.any() and fb.any() and (~fs).any() and (~fb).any()
    if name == "dyadic":
        for q in (2.5, 7.5, 12.5, 17.5):
            assert (qa == q).any() and (qa == -q).any() and (qb == q).any() and (qb == -q).any()
    if name == "dyadic_large":
        for K0 in LARGE_K:
            assert (np.abs(ka) == K0).any() or (np.abs(kb) == K0).any()
        assert np.abs(qa).max() > (1 << 29) and (np.abs(ka - qa.astype(np.int64)) <= 1).sum() > 100
        assert fs.any() and fb.any() and (~fs).any() and (~fb).any()


# ----------------------------------------------------------------------------------------------
# GPU: the routes
# ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sg():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import sgmm_b200
    return sgmm_b200


def _bundle(sg, ep, tick=TICK):
    return sg.Bundle(ep["z1"], ep["z2"], ep["mid"], ep["ask"], ep["bid"], ep["bmax"], ep["smin"], tick)


@pytest.mark.gpu
@pytest.mark.parametrize("name", EPISODES)
def test_prologue_thresholds_are_the_chosen_ones(sg, episodes, name):
    ep = episodes[name]
    ka, kb = _bundle(sg, ep).thresholds()
    wa, wb = brute_thresholds(ep)
    assert np.array_equal(ka, wa) and np.array_equal(kb, wb)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("name", EPISODES)
def test_exact_routes_equal_the_oracle(sg, orc, episodes, name, variant):
    """rollout_kernel_h32 (U = 1, 2, 4), the small-population path (5- and 20-state) and the trace kernel, bit for bit."""
    import torch
    ep = episodes[name]
    fee, use_adv = VARIANTS[variant]
    G = genomes_of(32, ep["scale"])
    A = adversaries() if use_adv else None
    bz, bun = bz_of(ep), _bundle(sg, ep)
    fo, to = orc.rollout_population(bz, PHI, TICK, fee, genomes=G, adv_genomes=A, use_adv=use_adv, nthreads=4)
    g = torch.from_numpy(G).cuda()
    a = None if A is None else torch.from_numpy(A).cuda()
    for units in (0, 1, 2, 4):                       # 0: the small-population path (P <= 148)
        f, t = sg.rollout_population(bun, g, a, phi=PHI, fee_rate=fee, units_per_lane=units)
        assert np.array_equal(bits64(f.cpu().numpy()), bits64(fo)), (units, f.cpu().numpy(), fo)
        assert np.array_equal(t.cpu().numpy(), to), units
    for i in range(2):
        adv = None if A is None else A[i]
        fo1, to1, tro = orc.rollout(G[i], adv, bz, PHI, TICK, fee, trace=True)
        fg, tg, trg = sg.rollout_trace(bun, G[i], adv, phi=PHI, fee_rate=fee)
        for k in ("off_a", "off_b", "adv_a", "adv_b", "fill_buy", "fill_sell", "inventory"):
            assert np.array_equal(trg[k], tro[k]), (i, k)
        for k in ("raw_a", "raw_b"):
            assert np.array_equal(bits32(trg[k]), bits32(tro[k])), (i, k)
        for k in ("cash", "reward", "pnl_reward", "inventory_reward", "fee_paid"):
            assert np.array_equal(bits64(trg[k]), bits64(tro[k])), (i, k)
        assert (bits64(fg), tg) == (bits64(fo1), to1) == (bits64(fo[i]), to[i])
        if use_adv:
            assert (tro["adv_a"] != 0).any() and (tro["adv_b"] != 0).any()


def _tensor_checks(orc, ep, name, G, A, fee, fit, trd, raw, act, hidden, tau):
    """Given the kernel's offsets the env is the oracle's bit for bit; on dyadic episodes the whole closed loop is."""
    bz, T = bz_of(ep), ep["z1"].size
    small = (np.abs(ep["z1"] * ep["scale"] * 5) <= 16) & (np.abs(ep["z2"] * ep["scale"] * 5) <= 16)
    for i in range(G.shape[0]):
        adv = None if A is None else A[i]
        fo, to, tro = orc.rollout(None, adv, bz, PHI, TICK, fee, forced_actions=act[i], trace=True)
        assert fo == fit[i] and to == trd[i], (i, fo, fit[i], to, trd[i])
        inv_before = np.concatenate([[0], tro["inventory"][:-1]])
        taken = np.rint(raw[i, np.arange(T), inv_before + 2] * F32(5)).astype(np.int32)
        assert np.array_equal(taken, act[i]), i
        want = np.stack([ep["z1"], ep["z2"]], 1) * ep["scale"]
        want = want[:, ::-1] if i % 2 else want
        if name.startswith("dyadic"):
            fc, tc, trc = orc.rollout(G[i], adv, bz, PHI, TICK, fee, hidden=hidden, trace=True)
            for iv in range(5):
                assert np.array_equal(bits32(raw[i, :, iv]), bits32(want)), (i, iv)
            assert np.array_equal(act[i, :, 0], trc["off_a"]) and np.array_equal(act[i, :, 1], trc["off_b"]), i
            assert bits64(fit[i]) == bits64(fc) and trd[i] == tc, i
        else:
            d = np.abs(raw[i][small] * F32(5) - want[small][:, None, :] * F32(5))
            assert d.max() <= tau, (i, d.max())


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "tf32", "f16"])
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("name", TENSOR_EPISODES)
def test_tc32_routes(sg, orc, episodes, name, variant, precision):
    import torch
    ep = episodes[name]
    fee, use_adv = VARIANTS[variant]
    G = genomes_of(32, ep["scale"])
    A = adversaries() if use_adv else None
    bun = _bundle(sg, ep)
    fit, trd, raw, act = sg.rollout_tc_audit(bun, G, A, phi=PHI, fee_rate=fee, hidden=32, precision=precision)
    f2, t2 = sg.rollout_population(bun, torch.from_numpy(G).cuda(), None if A is None else torch.from_numpy(A).cuda(),
                                   phi=PHI, fee_rate=fee, precision=precision)
    assert torch.equal(f2, fit) and torch.equal(t2, trd)
    _tensor_checks(orc, ep, name, G, A, fee, fit.cpu().numpy(), trd.cpu().numpy(), raw.cpu().numpy(), act.cpu().numpy(),
                   32, TAU[precision])


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "fee"])
@pytest.mark.parametrize("name", TENSOR_EPISODES)
def test_spec256_route(sg, orc, episodes, name, variant):
    import torch
    ep = episodes[name]
    fee, _ = VARIANTS[variant]
    G = genomes_of(256, ep["scale"])
    bun = _bundle(sg, ep)
    fit, trd, raw, act = sg.rollout_spec256_audit(bun, G, phi=PHI, fee_rate=fee)
    f2, t2 = sg.rollout_population(bun, torch.from_numpy(G).cuda(), phi=PHI, fee_rate=fee, hidden=256)
    assert torch.equal(f2, fit) and torch.equal(t2, trd)
    _tensor_checks(orc, ep, name, G, None, fee, fit.cpu().numpy(), trd.cpu().numpy(), raw.cpu().numpy(), act.cpu().numpy(),
                   256, TAU_256)


# ----------------------------------------------------------------------------------------------
# other operating points: price grids and ticks, phi, fees (a negative fee is a maker rebate)
# ----------------------------------------------------------------------------------------------
GRIDS = {                       # start bid, price step, decimals, tick
    "3dp_tick0.01": (3.480, 0.001, 3, 0.01),          # the reference's default tick on the 3-decimal data
    "2dp_35": (35.00, 0.01, 2, 0.01),
    "4dp_0.9": (0.9000, 0.0001, 4, 0.0001),
    "1dp_3800_tick0.2": (3800.0, 0.2, 1, 0.2),
}


def grid_bundle(name, T=240, seed=0):
    """Bars on another price grid: bid random walk, spread 1-2 steps, next-bar extremes -1..3 steps beyond the touch,
    ~2 % NaN bounds, AR(1) / iid signals as in synthetic.py."""
    start, step, dec, _ = GRIDS[name]
    rng = np.random.default_rng(1000 + seed)
    n = T + 1
    bt = int(round(start / step)) + np.cumsum(rng.choice([-2, -1, 0, 1, 2], size=n, p=[.1, .22, .36, .22, .1]))
    at = bt + rng.choice([1, 2], size=n, p=[.9, .1])
    bid, ask = np.round(bt * step, dec), np.round(at * step, dec)
    mid = (ask + bid) / 2.0
    bmax = np.round((at + rng.choice([-1, 0, 1, 2, 3], size=n, p=[.04, .51, .3, .11, .04])) * step, dec)
    smin = np.round((bt - rng.choice([-1, 0, 1, 2, 3], size=n, p=[.04, .51, .3, .11, .04])) * step, dec)
    bmax[rng.random(n) < 0.02] = np.nan
    smin[rng.random(n) < 0.02] = np.nan
    s1 = (2.24 + 0.37 * rng.standard_normal(n)).astype(F32)
    s2 = (0.04 + 0.55 * rng.standard_normal(n)).astype(F32)
    return (s1[:-1], s2[:-1], mid[1:].copy(), ask[:-1].copy(), bid[:-1].copy(), bmax[:-1].copy(), smin[:-1].copy())


@pytest.mark.gpu
@pytest.mark.parametrize("fee", [0.0, 3e-4, -1e-4])
@pytest.mark.parametrize("grid", list(GRIDS))
def test_operating_points_sweep(sg, orc, grid, fee):
    """policy_like_genomes on other price grids and ticks, phi in {0, 1e-4, 0.01}: the exact routes bitwise, the
    tensor-core routes bit for bit given the offsets they took."""
    import torch
    from sgmm_b200 import synthetic
    tick = GRIDS[grid][3]
    bundle = grid_bundle(grid)
    stats = synthetic.train_stats_of(bundle)
    bz = orc.normalise(bundle, stats) + bundle[2:]
    bun = sg.Bundle.from_arrays(bundle, stats, tick)
    _, G = synthetic.policy_like_genomes(6, seed=7, out_scale=6.0, out_bias=(0.1, 0.1))
    _, G256 = synthetic.policy_like_genomes(4, hidden=256, seed=8, out_scale=4.0, out_bias=(0.1, 0.1))
    g = torch.from_numpy(G).cuda()
    for phi in (0.0, 1e-4, 0.01):
        fo, to = orc.rollout_population(bz, phi, tick, fee, genomes=G, nthreads=4)
        assert to.max() > 0
        for units in (0, 4):
            f, t = sg.rollout_population(bun, g, phi=phi, fee_rate=fee, units_per_lane=units)
            assert np.array_equal(bits64(f.cpu().numpy()), bits64(fo)) and np.array_equal(t.cpu().numpy(), to), (phi, units)
        fo1, to1, tro = orc.rollout(G[0], None, bz, phi, tick, fee, trace=True)
        fg, tg, trg = sg.rollout_trace(bun, G[0], phi=phi, fee_rate=fee)
        for k in ("off_a", "off_b", "fill_buy", "fill_sell", "inventory"):
            assert np.array_equal(trg[k], tro[k]), (phi, k)
        for k in ("cash", "reward", "fee_paid"):
            assert np.array_equal(bits64(trg[k]), bits64(tro[k])), (phi, k)
        for precision in ("bf16", "tf32", "f16"):
            fit, trd, _, act = sg.rollout_tc_audit(bun, G, phi=phi, fee_rate=fee, hidden=32, precision=precision)
            fit, trd, act = fit.cpu().numpy(), trd.cpu().numpy(), act.cpu().numpy()
            for i in range(G.shape[0]):
                assert orc.rollout(None, None, bz, phi, tick, fee, forced_actions=act[i]) == (fit[i], trd[i]), (phi, precision, i)
        fit, trd, _, act = sg.rollout_spec256_audit(bun, G256, phi=phi, fee_rate=fee)
        fit, trd, act = fit.cpu().numpy(), trd.cpu().numpy(), act.cpu().numpy()
        for i in range(G256.shape[0]):
            assert orc.rollout(None, None, bz, phi, tick, fee, forced_actions=act[i]) == (fit[i], trd[i]), (phi, i)
