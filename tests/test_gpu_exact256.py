"""GPU (-m gpu): bit-exact episodes at hidden width 256 (SGMM_PRECISION_EXACT, csrc/sgmm_exact256.cu).

The exact H = 256 path is a CUDA-core policy table of every (bar, inventory) pair in SGMM-F32 order plus the walk kernels
of the small-population path.  Everything here is compared with the C oracle at hidden=256 BIT FOR BIT: population
fitness and trades (explicit genomes, seeded children, host and pipelined entries, several batches), the adversary,
quotes on rounding ties, every trace column, the device GA against a GA composed from oracle rollouts, and DRLEngine.
The CPU tests (no marker) check on the oracle that the transparent fixtures are what they claim.
"""
import ctypes as C
import os

import numpy as np
import pytest

H = 256
G256 = H * H + 7 * H + 2
F32 = np.float32
ADV_THR = F32(0.54930615)                         # largest fp32 y with round(tanh(y)) == 0 (tests/golden/tanh_threshold.npz)
ADV_ULP = np.nextafter(ADV_THR, F32(np.inf)) - ADV_THR
TICK = 0.001
BATCH_ENV = "SGMM_EXACT256_BATCH_BYTES"


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


def bits32(a):
    return np.asarray(a, np.float32).view(np.uint32)


# ----------------------------------------------------------------------------------------------
# transparent policies (as in tests/test_gpu_rounding_edges.py): raw = scale * (z1, z2) exactly, for every inventory
# ----------------------------------------------------------------------------------------------
def transparent_genome(hidden=H, scale=1.0, swap=False):
    W1, b1 = np.zeros((hidden, 3), F32), np.zeros(hidden, F32)
    W2, b2 = np.zeros((hidden, hidden), F32), np.zeros(hidden, F32)
    W3, b3 = np.zeros((2, hidden), F32), np.zeros(2, F32)
    W1[0, 0], W1[1, 0], W1[2, 1], W1[3, 1] = 1, -1, 1, -1           # relu(z1), relu(-z1), relu(z2), relu(-z2)
    for j in range(4):
        W2[j, j] = 1
    a, b = (1, 0) if swap else (0, 1)
    W3[a, 0], W3[a, 1], W3[b, 2], W3[b, 3] = scale, -scale, scale, -scale
    return np.concatenate([W1.ravel(), b1, W2.ravel(), b2, W3.ravel(), b3]).astype(F32)


def genomes_of(hidden=H, scale=1.0):
    g0, g1 = transparent_genome(hidden, scale), transparent_genome(hidden, scale, swap=True)
    return np.stack([g0, g1, g0, g1])


def boundary_adversary(sign_a, sign_b):
    """y_a is ADV_THR after a bar without a sell fill and the next float beyond it after one; y_b likewise (fill_buy)."""
    g = np.zeros(1250, F32)
    g[1] = 1.0                              # h0 = relu(fill_sell_prev)
    g[5] = 1.0                              # h1 = relu(fill_buy_prev)
    g[48] = sign_a * ADV_ULP                # V2[0, 0]
    g[61] = sign_b * ADV_ULP                # V2[1, 1]
    g[72], g[73] = sign_a * ADV_THR, sign_b * ADV_THR
    return g


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


LARGE_K = [(1 << 22) - 1, 1 << 22, (1 << 22) + 5, 1 << 23, (1 << 24) + 3, (1 << 30) - 3]


def edge_episode(seed=7):
    """q on K +- 0.5 for even and odd K of both signs, one ulp either side and exactly K (|K| <= 6), then thresholds of
    +-2^22 ... near K_CLAMP with q on and around them; NaN / inf bounds."""
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
        t, s = 2 * i + (i % 2), i % 2                       # ask on even cases, bid on odd ones
        (ka if s == 0 else kb)[t] = K
        z[s, t] = zz
    bmax, smin = ask + ka.astype(np.float64) * TICK, bid - kb.astype(np.float64) * TICK
    for i, t in enumerate(rng.choice(np.arange(T), size=24, replace=False)):
        (bmax if i % 2 == 0 else smin)[t] = [np.nan, np.inf, -np.inf][i % 3]
    return (z[0], z[1], mid, ask, bid, bmax, smin)


def test_transparent_h256_policy_outputs_its_inputs():
    from oracle import oracle as orc
    bz = edge_episode()
    g0, g1 = transparent_genome(), transparent_genome(swap=True)
    for t in range(0, bz[0].size, 5):
        for iv in range(5):
            x = [bz[0][t], bz[1][t], (iv - 2) / 2.0]
            want = np.array([bz[0][t], bz[1][t]], F32)
            assert np.array_equal(bits32(orc.mlp_forward(g0, x, hidden=H)), bits32(want))
            assert np.array_equal(bits32(orc.mlp_forward(g1, x, hidden=H)), bits32(want[::-1]))


def test_edge_episode_has_ties_of_both_parities():
    z1, z2 = edge_episode()[:2]
    q = np.concatenate([z1, z2]) * F32(5)
    for K in (-5, -4, 4, 5):
        assert (q == F32(K + 0.5)).any() and (q == F32(K - 0.5)).any() and (q == F32(K)).any()
    assert (np.abs(q) > (1 << 29)).any() and (np.abs(q) == (1 << 22) + 5.5).any()


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


def _synthetic(sg, orc, days, first_day, T=None, tick=TICK):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(days, first_day=first_day)
    if T is not None:
        bundle = tuple(a[:T] for a in bundle)
    stats = synthetic.train_stats_of(synthetic.synthetic_bundle(days, first_day=first_day))
    z1, z2 = orc.normalise(bundle, stats)
    return sg.Bundle.from_arrays(bundle, stats, tick), (z1, z2) + tuple(bundle[2:]), bundle, stats


def _genomes(P, seed, out_scale=4.0):
    from sgmm_b200 import synthetic
    _, g = synthetic.policy_like_genomes(P, hidden=H, seed=seed, out_scale=out_scale, out_bias=(0.1, 0.1))
    return g


def _adv(P, seed):
    return (np.random.default_rng(seed).standard_normal((P, 1250)) * 0.6).astype(F32)


def _same(f, t, fo, to):
    f = f.cpu().numpy() if hasattr(f, "cpu") else np.asarray(f)
    t = t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t)
    assert np.array_equal(bits64(f), bits64(fo)), (f, fo)
    assert np.array_equal(t, to), (t, to)


@pytest.mark.gpu
@pytest.mark.parametrize("fee", [0.0, 3e-4, -1e-4])
@pytest.mark.parametrize("phi", [0.0, 1e-4, 0.01])
def test_population_bitwise_fee_phi(sg, orc, fee, phi):
    import torch
    bun, bz, _, _ = _synthetic(sg, orc, 1, 90, T=160)
    G = _genomes(5, seed=3)
    fo, to = orc.rollout_population(bz, phi, TICK, fee, genomes=G, hidden=H)
    f, t = sg.rollout_population(bun, torch.from_numpy(G).cuda(), phi=phi, fee_rate=fee, hidden=H, precision="exact")
    _same(f, t, fo, to)
    assert to.max() > 0
    f, t = sg.rollout_population(bun, G, phi=phi, fee_rate=fee, hidden=H, precision="exact")     # host entry
    _same(f, t, fo, to)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [0, 1, 2, 127, 128, 129, 1000])
@pytest.mark.parametrize("P", [1, 3, 33])
def test_ragged_lengths_and_population_sizes(sg, orc, T, P):
    import torch
    bun, bz, _, _ = _synthetic(sg, orc, 5, 91, T=T)
    assert bun.T == T
    G = _genomes(P, seed=T + P)
    fo, to = orc.rollout_population(bz, 1e-4, TICK, 3e-4, genomes=G, hidden=H)
    f, t = sg.rollout_population(bun, torch.from_numpy(G).cuda(), phi=1e-4, fee_rate=3e-4, hidden=H, precision="exact")
    _same(f, t, fo, to)


@pytest.mark.gpu
def test_seeded_children_equal_explicit_through_every_entry(sg, orc):
    import torch
    bun, bz, _, _ = _synthetic(sg, orc, 1, 93, T=300)
    master = _genomes(1, seed=8)[0]
    kids = np.stack([orc.mutate(master, 0.05, 77, 4, 10 + i) for i in range(6)])
    fo, to = orc.rollout_population(bz, 1e-4, TICK, 0.0, master=master, sigma=0.05, seed=77, generation=4, first_index=10,
                                    count=6, hidden=H)
    fs, ts = sg.rollout_seeded(bun, torch.from_numpy(master).cuda(), count=6, sigma=0.05, seed=77, generation=4,
                               first_index=10, phi=1e-4, hidden=H, precision="exact")
    _same(fs, ts, fo, to)
    fe, te = sg.rollout_population(bun, torch.from_numpy(kids).cuda(), phi=1e-4, hidden=H, precision="exact")
    _same(fe, te, fo, to)
    fh, th = sg.rollout_population(bun, kids, phi=1e-4, hidden=H, precision="exact")
    _same(fh, th, fo, to)
    pend = [sg.rollout_population_async(bun, torch.from_numpy(kids[i:i + 3]).pin_memory(), phi=1e-4, hidden=H,
                                        precision="exact") for i in (0, 3)]
    fa, ta = zip(*[p.result() for p in pend])
    _same(np.concatenate(fa), np.concatenate(ta), fo, to)
    # an explicit genome row that is only 4-byte aligned is staged, not misread
    flat = torch.zeros(G256 * 2 + 1, dtype=torch.float32, device="cuda")
    flat[1:1 + G256] = torch.from_numpy(kids[2]).cuda()
    mm = sg._lib.Population(H, 0, 1, flat.data_ptr() + 4, None, 0.0, 0.0, 0, 0, 0)
    prm = sg._lib.RolloutParams(1e-4, 0.0, 4, 0, 0, 0)
    of = torch.empty(1, dtype=torch.float64, device="cuda")
    ot = torch.empty(1, dtype=torch.int32, device="cuda")
    sg._lib.check(sg._lib.lib().sgmm_rollout_population(bun.handle, C.byref(mm), None, C.byref(prm), of.data_ptr(),
                                                        ot.data_ptr(), None))
    _same(of, ot, fo[2:3], to[2:3])


@pytest.mark.gpu
def test_multi_day_episode(sg, orc):
    import torch
    bun, bz, _, _ = _synthetic(sg, orc, 12, 100)
    assert bun.T >= 2880
    G = _genomes(2, seed=12, out_scale=3.0)
    A = _adv(2, seed=12)
    for adv in (None, A):
        fo, to = orc.rollout_population(bz, 1e-4, TICK, 3e-4, genomes=G, adv_genomes=adv, use_adv=adv is not None, hidden=H)
        f, t = sg.rollout_population(bun, torch.from_numpy(G).cuda(), None if adv is None else torch.from_numpy(adv).cuda(),
                                     phi=1e-4, fee_rate=3e-4, hidden=H, precision="exact")
        _same(f, t, fo, to)
        assert to.min() > 100


@pytest.mark.gpu
@pytest.mark.parametrize("use_adv", [False, True])
def test_several_batches_equal_one(sg, orc, use_adv, monkeypatch):
    import torch
    bun, bz, _, _ = _synthetic(sg, orc, 1, 94, T=200)
    P = 7
    G = _genomes(P, seed=5)
    A = _adv(P, seed=5) if use_adv else None
    g = torch.from_numpy(G).cuda()
    a = None if A is None else torch.from_numpy(A).cuda()
    master = torch.from_numpy(G[0]).cuda()
    whole = sg.rollout_population(bun, g, a, phi=1e-4, hidden=H, precision="exact")
    whole_s = sg.rollout_seeded(bun, master, count=P, sigma=0.05, seed=3, generation=1, phi=1e-4, hidden=H, precision="exact",
                                adv_master=None if a is None else a[0], adv_sigma=0.1)
    monkeypatch.setenv(BATCH_ENV, str(200 * 48 * 2 + 1))            # two individuals' tables per batch: 4 batches
    parts = sg.rollout_population(bun, g, a, phi=1e-4, hidden=H, precision="exact")
    monkeypatch.setenv(BATCH_ENV, "1")                              # one individual per batch (seeded: + staged genome)
    parts_s = sg.rollout_seeded(bun, master, count=P, sigma=0.05, seed=3, generation=1, phi=1e-4, hidden=H, precision="exact",
                                adv_master=None if a is None else a[0], adv_sigma=0.1)
    for x, y in ((whole, parts), (whole_s, parts_s)):
        assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])
    fo, to = orc.rollout_population(bz, 1e-4, TICK, 0.0, genomes=G, adv_genomes=A, use_adv=use_adv, hidden=H)
    _same(parts[0], parts[1], fo, to)
    fo, to = orc.rollout_population(bz, 1e-4, TICK, 0.0, master=G[0], sigma=0.05, seed=3, generation=1, count=P,
                                    adv_master=None if A is None else A[0], adv_sigma=0.1, use_adv=use_adv, hidden=H)
    _same(parts_s[0], parts_s[1], fo, to)


@pytest.mark.gpu
@pytest.mark.parametrize("fee", [0.0, 3e-4])
def test_adversary_bitwise(sg, orc, fee):
    import torch
    bun, bz, _, _ = _synthetic(sg, orc, 1, 95, T=400)
    P = 9
    G = _genomes(P, seed=6)
    A = _adv(P, seed=6)
    fo, to = orc.rollout_population(bz, 1e-4, TICK, fee, genomes=G, adv_genomes=A, use_adv=True, hidden=H)
    f, t = sg.rollout_population(bun, torch.from_numpy(G).cuda(), torch.from_numpy(A).cuda(), phi=1e-4, fee_rate=fee,
                                 hidden=H, precision="exact")
    _same(f, t, fo, to)
    f, t = sg.rollout_population(bun, G, A, phi=1e-4, fee_rate=fee, hidden=H, precision="exact")
    _same(f, t, fo, to)
    fo2, _ = orc.rollout_population(bz, 1e-4, TICK, fee, genomes=G, hidden=H)
    assert not np.array_equal(fo, fo2)                                # the adversary changes the episodes


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "fee", "adv"])
def test_rounding_edges_bitwise(sg, orc, variant):
    """Transparent H = 256 policies put q = raw*5 on K +- 0.5 ties, one ulp either side and exactly on K, and on thresholds
    of millions of ticks; boundary adversaries sit exactly on and one float beyond the tanh rounding threshold."""
    import torch
    bz = edge_episode()
    bun = sg.Bundle(*bz, TICK)
    fee = 3e-4 if variant == "fee" else 0.0
    G = genomes_of()
    A = adversaries() if variant == "adv" else None
    fo, to = orc.rollout_population(bz, 1e-4, TICK, fee, genomes=G, adv_genomes=A, use_adv=A is not None, hidden=H)
    f, t = sg.rollout_population(bun, torch.from_numpy(G).cuda(), None if A is None else torch.from_numpy(A).cuda(),
                                 phi=1e-4, fee_rate=fee, hidden=H, precision="exact")
    _same(f, t, fo, to)
    for i in range(2):
        adv = None if A is None else A[i]
        fo1, to1, tro = orc.rollout(G[i], adv, bz, 1e-4, TICK, fee, hidden=H, trace=True)
        fg, tg, trg = sg.rollout_trace(bun, G[i], adv, phi=1e-4, fee_rate=fee, hidden=H)
        for k in ("off_a", "off_b", "adv_a", "adv_b", "fill_buy", "fill_sell", "inventory"):
            assert np.array_equal(trg[k], tro[k]), (i, k)
        assert (bits64(fg), tg) == (bits64(fo1), to1) == (bits64(fo[i]), to[i])
        if A is not None:
            assert (tro["adv_a"] != 0).any() and (tro["adv_b"] != 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("use_adv", [False, True])
def test_trace_every_column_and_recorder(sg, orc, use_adv):
    bun, bz, bundle, _ = _synthetic(sg, orc, 1, 96, T=500)
    g = _genomes(1, seed=9)[0]
    a = _adv(1, seed=9)[0] if use_adv else None
    fo, to, tro = orc.rollout(g, a, bz, 1e-4, TICK, 3e-4, hidden=H, trace=True)
    fg, tg, trg = sg.rollout_trace(bun, g, a, phi=1e-4, fee_rate=3e-4, hidden=H)
    for k in ("off_a", "off_b", "adv_a", "adv_b", "fill_buy", "fill_sell", "inventory"):
        assert np.array_equal(trg[k], tro[k]), k
    for k in ("raw_a", "raw_b"):
        assert np.array_equal(bits32(trg[k]), bits32(tro[k])), k
    for k in ("cash", "reward", "pnl_reward", "inventory_reward", "fee_paid"):
        assert np.array_equal(bits64(trg[k]), bits64(tro[k])), k
    assert (bits64(fg), tg) == (bits64(fo), to)
    # derived columns (Env/recorder.py:45-51) from the oracle's own columns
    mid = np.asarray(bundle[2], np.float64)
    inv = tro["inventory"].astype(np.float64)
    assert np.array_equal(bits64(trg["spread"]), bits64(np.asarray(bundle[3]) - np.asarray(bundle[4])))
    assert np.array_equal(bits64(trg["unrealized_pnl"]), bits64(inv * mid))
    assert np.array_equal(bits64(trg["wealth"]), bits64(tro["cash"] + inv * mid))
    assert np.array_equal(bits64(trg["cum_reward"]), bits64(np.cumsum(tro["reward"])))
    assert np.array_equal(bits64(trg["cum_fees"]), bits64(np.cumsum(tro["fee_paid"])))
    assert np.array_equal(trg["skew"], tro["off_b"] - tro["off_a"])
    if use_adv:
        assert (tro["adv_a"] != 0).any()
    from sgmm_b200 import StrategyRecorder
    df = StrategyRecorder.from_trace(trg, bundle).to_dataframe()
    assert len(df) == bun.T and np.array_equal(df["off_a"].to_numpy(), tro["off_a"])
    assert np.array_equal(bits64(df["wealth"].to_numpy()), bits64(trg["wealth"]))


def _oracle_ga(orc, train_bz, val_bz, master, adv_master, *, pop, sigma, phi, tick, fee, use_arl, seed, gens, patience):
    FLIP = 0x8000000000000000
    master = master.copy()
    adv_master = None if adv_master is None else adv_master.copy()
    s_mm = s_adv = F32(sigma)
    best_val, stale = -np.inf, 0
    best_master = master.copy()
    hist = {k: [] for k in ("train_f", "val_f", "train_trades", "val_trades", "sigma")}
    for gen in range(gens):
        fit, trd = orc.rollout_population(train_bz, phi, tick, fee, master=master, sigma=float(s_mm),
                                          adv_master=adv_master, adv_sigma=float(s_adv), use_adv=use_arl,
                                          seed=seed, generation=gen, count=pop, hidden=H)
        best = int(np.argmax(fit))                                        # model.py:74
        master = orc.mutate(master, float(s_mm), seed, gen, best)
        if use_arl:
            adv_master = orc.mutate(adv_master, float(s_adv), seed ^ FLIP, gen, int(np.argmax(-fit)))
        vf, vt = orc.rollout(master, None, val_bz, phi, tick, fee, hidden=H)   # drl_engine.py:129-140
        hist["train_f"].append(fit[best]); hist["train_trades"].append(trd[best])
        hist["val_f"].append(vf); hist["val_trades"].append(vt); hist["sigma"].append(s_mm)
        if vf > best_val:
            best_val, stale, best_master = vf, 0, master.copy()
        else:
            stale += 1
        if stale >= patience:
            s_mm = F32(s_mm * F32(0.5))
            if use_arl:
                s_adv = F32(s_adv * F32(0.5))
            stale = 0
    return hist, master, adv_master, best_master, best_val, float(s_mm)


@pytest.mark.gpu
@pytest.mark.parametrize("use_arl", [False, True])
def test_device_ga_matches_oracle_ga(sg, orc, use_arl):
    from sgmm_b200.engine import DeviceGA
    train, tz, _, stats = _synthetic(sg, orc, 1, 50, T=180)
    from sgmm_b200 import synthetic
    vb = tuple(a[:150] for a in synthetic.synthetic_bundle(1, first_day=52))
    val = sg.Bundle.from_arrays(vb, stats, TICK)
    vz = orc.normalise(vb, stats) + tuple(vb[2:])
    master = _genomes(1, seed=21, out_scale=1.0)[0]
    adv_master = (np.random.default_rng(4).standard_normal(1250) * 0.5).astype(F32) if use_arl else None
    gens, pop, patience = 6, 10, 2
    ga = DeviceGA(master, adv_master, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=use_arl, seed=77,
                  max_generations=gens, patience=patience, hidden=H, precision="exact")
    for _ in range(gens):
        ga.generation(train, val)
    h = ga.history(gens)
    st = ga.status()
    mm, adv, best = ga.masters()
    ga.close()
    ho, m_o, a_o, b_o, bv_o, s_o = _oracle_ga(orc, tz, vz, master, adv_master, pop=pop, sigma=0.05, phi=1e-4, tick=TICK,
                                               fee=0.0, use_arl=use_arl, seed=77, gens=gens, patience=patience)
    assert np.array_equal(bits64(h["train_f"]), bits64(ho["train_f"]))
    assert np.array_equal(bits64(h["val_f"]), bits64(ho["val_f"]))
    assert h["train_trades"].tolist() == ho["train_trades"] and h["val_trades"].tolist() == ho["val_trades"]
    assert np.array_equal(h["sigma"], np.array(ho["sigma"], F32))
    assert np.array_equal(bits32(mm), bits32(m_o)) and np.array_equal(bits32(best), bits32(b_o))
    if use_arl:
        assert np.array_equal(bits32(adv), bits32(a_o))
    assert st["generation"] == gens and st["best_val"] == bv_o and st["sigma"] == s_o


@pytest.mark.gpu
def test_drl_engine_exact_h256_with_arl(sg, orc, tmp_path):
    import torch
    from sgmm_b200 import synthetic
    tb = tuple(a[:200] for a in synthetic.synthetic_bundle(1, first_day=60))
    vb = tuple(a[:160] for a in synthetic.synthetic_bundle(1, first_day=61))
    stats = synthetic.train_stats_of(tb)
    eng = sg.DRLEngine(pop_size=8, phi=1e-4, tick_size=TICK, use_arl=True, save_dir=str(tmp_path), seed=5,
                       hidden_dim=H, precision="exact")
    policy, hist = eng.train(tb, vb, stats, generations=4, output_prefix="x256", verbose=False)
    w = policy.get_weights().detach().cpu().numpy()
    assert w.size == G256
    vz = orc.normalise(vb, stats) + tuple(vb[2:])
    fo, to = orc.rollout(w, None, vz, 1e-4, TICK, 0.0, hidden=H)
    assert fo == max(hist["val_f"])
    fe, te = sg.evaluate_individual(w, None, vb, 1e-4, TICK, 0.0, stats)
    assert (bits64(fe), te) == (bits64(fo), to)
    snap = sg.TradingPolicy(hidden_dim=H)
    snap.load_state_dict(torch.load(os.path.join(str(tmp_path), "x256_best_val_0.0001.pth")))
    assert np.array_equal(bits32(snap.get_weights().detach().cpu().numpy()), bits32(w))
    fa, ta = sg.evaluate_individual(w, _adv(1, 3)[0], vb, 1e-4, TICK, 3e-4, stats, use_arl=True)
    fo, to = orc.rollout(w, _adv(1, 3)[0], vz, 1e-4, TICK, 3e-4, hidden=H)
    assert (bits64(fa), ta) == (bits64(fo), to)
    with pytest.raises(ValueError):
        sg.evaluate_individual(w[:-1], None, vb, 1e-4, TICK, 0.0, stats)


@pytest.mark.gpu
def test_output_canaries_untouched(sg, orc):
    import torch
    bun, bz, _, _ = _synthetic(sg, orc, 1, 97, T=130)
    P, pad = 5, 64
    G = _genomes(P, seed=2)
    A = _adv(P, seed=2)
    L = sg._lib
    g = torch.from_numpy(G).cuda()
    a = torch.from_numpy(A).cuda()
    for adv in (None, a):
        fit = torch.full((P + 2 * pad,), 12345.5, dtype=torch.float64, device="cuda")
        trd = torch.full((P + 2 * pad,), -777, dtype=torch.int32, device="cuda")
        mm = L.Population(H, 0, P, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
        ap = None if adv is None else C.byref(L.Population(32, 0, P, adv.data_ptr(), None, 0.0, 0.0, 0, 0, 0))
        prm = L.RolloutParams(1e-4, 0.0, 4, 0, 0, 0)
        L.check(L.lib().sgmm_rollout_population(bun.handle, C.byref(mm), ap, C.byref(prm), fit[pad:].data_ptr(),
                                                trd[pad:].data_ptr(), None))
        torch.cuda.synchronize()
        f, t = fit.cpu().numpy(), trd.cpu().numpy()
        assert (f[:pad] == 12345.5).all() and (f[pad + P:] == 12345.5).all()
        assert (t[:pad] == -777).all() and (t[pad + P:] == -777).all()
        fo, to = orc.rollout_population(bz, 1e-4, TICK, 0.0, genomes=G, adv_genomes=None if adv is None else A,
                                        use_adv=adv is not None, hidden=H)
        _same(f[pad:pad + P], t[pad:pad + P], fo, to)
    # trace columns: every column of T values between canaries
    T = bun.T
    cols, keep = {}, []
    for name, _ in L.Trace._fields_:
        dt = torch.int32 if name in ("off_a", "off_b", "adv_a", "adv_b", "fill_buy", "fill_sell", "inventory", "skew") else (
            torch.float32 if name in ("raw_a", "raw_b") else torch.float64)
        buf = torch.full((T + 2 * pad,), -3, dtype=dt, device="cuda")
        keep.append(buf)
        cols[name] = buf
    tr = L.Trace(*[cols[n][pad:].data_ptr() for n, _ in L.Trace._fields_])
    fit = torch.full((1 + 2 * pad,), 12345.5, dtype=torch.float64, device="cuda")
    trd = torch.full((1 + 2 * pad,), -777, dtype=torch.int32, device="cuda")
    gg = g[0].contiguous()
    L.check(L.lib().sgmm_rollout_trace(bun.handle, gg.data_ptr(), H, a[0].data_ptr(), None, C.byref(L.RolloutParams(1e-4, 0.0, 0, 0, 0, 0)),
                                       C.byref(tr), fit[pad:].data_ptr(), trd[pad:].data_ptr(), None))
    torch.cuda.synchronize()
    for n, buf in cols.items():
        b = buf.cpu().numpy()
        assert (b[:pad] == -3).all() and (b[pad + T:] == -3).all(), n
    f, t = fit.cpu().numpy(), trd.cpu().numpy()
    assert (f[:pad] == 12345.5).all() and (f[pad + 1:] == 12345.5).all() and (t[pad + 1:] == -777).all()
    fo, to = orc.rollout(G[0], A[0], bz, 1e-4, TICK, 0.0, hidden=H)
    assert (bits64(f[pad]), t[pad]) == (bits64(fo), to)


@pytest.mark.gpu
def test_guards(sg, orc):
    import torch
    from sgmm_b200.engine import DeviceGA
    bun, bz, _, _ = _synthetic(sg, orc, 1, 98, T=40)
    L = sg._lib
    G = _genomes(2, seed=1)
    g = torch.from_numpy(G).cuda()
    out_f = torch.empty(2, dtype=torch.float64, device="cuda")
    out_t = torch.empty(2, dtype=torch.int32, device="cuda")
    raw = torch.zeros(2 * bun.T * 10, dtype=torch.float32, device="cuda")
    act = torch.zeros(2 * bun.T * 2, dtype=torch.int32, device="cuda")
    exact = L.RolloutParams(1e-4, 0.0, 4, 0, 0, 0)
    for hidden in (32, 256):
        gh = torch.zeros(2, hidden * hidden + 7 * hidden + 2, dtype=torch.float32, device="cuda")
        mm = L.Population(hidden, 0, 2, gh.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
        rc = L.lib().sgmm_rollout_tc_audit(bun.handle, C.byref(mm), None, C.byref(exact), out_f.data_ptr(), out_t.data_ptr(),
                                           raw.data_ptr(), act.data_ptr(), None)
        assert rc == L.ERR_INVALID, hidden
    for hidden in (64, 128):
        gh = torch.zeros(2, hidden * hidden + 7 * hidden + 2, dtype=torch.float32, device="cuda")
        mm = L.Population(hidden, 0, 2, gh.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
        rc = L.lib().sgmm_rollout_population(bun.handle, C.byref(mm), None, C.byref(exact), out_f.data_ptr(),
                                             out_t.data_ptr(), None)
        assert rc in (L.ERR_UNSUPPORTED, L.ERR_INVALID), hidden
    with pytest.raises(L.SgmmError):
        DeviceGA(np.zeros(64 * 64 + 7 * 64 + 2, F32), None, pop_size=4, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=False,
                 seed=1, max_generations=2, hidden=64, precision="exact")
    # F32 (0) at H = 256 stays refused; BF16 with the adversary stays refused; EXACT at H = 32 is the F32 route
    mm = L.Population(H, 0, 2, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    rc = L.lib().sgmm_rollout_population(bun.handle, C.byref(mm), None, C.byref(L.RolloutParams(1e-4, 0.0, 0, 0, 0, 0)),
                                         out_f.data_ptr(), out_t.data_ptr(), None)
    assert rc == L.ERR_UNSUPPORTED and b"EXACT" in L.lib().sgmm_last_error()
    from sgmm_b200 import synthetic
    _, g32 = synthetic.policy_like_genomes(3, seed=4)
    f0, t0 = sg.rollout_population(bun, torch.from_numpy(g32).cuda(), phi=1e-4)
    f4, t4 = sg.rollout_population(bun, torch.from_numpy(g32).cuda(), phi=1e-4, precision="exact")
    prm = L.RolloutParams(1e-4, 0.0, 4, 0, 0, 0)
    assert torch.equal(f0, f4) and torch.equal(t0, t4)
    g32d = torch.from_numpy(g32).cuda()
    mm32 = L.Population(32, 0, 3, g32d.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    of = torch.empty(3, dtype=torch.float64, device="cuda")
    ot = torch.empty(3, dtype=torch.int32, device="cuda")
    L.check(L.lib().sgmm_rollout_population(bun.handle, C.byref(mm32), None, C.byref(prm), of.data_ptr(), ot.data_ptr(), None))
    torch.cuda.synchronize()
    assert torch.equal(of, f0) and torch.equal(ot, t0)
