"""Risk-adjusted training objectives (sgmm_rollout_objective, sgmm_ga_set_objective, ``objective=`` in Python).

The contract (include/sgmm.h, SGMM_OBJECTIVE_*), restated:
  REWARD   0  the reference's total reward, -50 without trades (the default)
  PNL      1  StrategyAnalytics "Total PnL"     (analytics.KEYS[0])
  PNL_MAP  2  StrategyAnalytics "PnLMAP (Eff)"  (analytics.KEYS[2])
  SHARPE   3  StrategyAnalytics "Sharpe", the trade Sharpe (analytics.KEYS[4])
For an episode with trace columns wealth = cash + inventory * mid_next (cash: buy leg, then sell leg) and
is_trade = fill_buy | fill_sell, v is that StrategyAnalytics column and
    fitness = trades == 0 ? v - 50 : (v is NaN ? -50 : v),   trades unchanged.

``stream_objective`` restates the streaming evaluation of the device walk (chunks of bars, a cash chain in bar order,
first / last wealth, sum |inventory|, the wealth differences of consecutive trade rows, numpy pairwise sums) in Python
floats; the CPU tests hold it to ``oracle.analytics`` on crafted and oracle traces.  The GPU tests hold the device to
``backtest_population`` (trace + device analytics) and to the oracle composition (trace -> wealth -> oracle.analytics),
and whole GAs to the GA composed from oracle traces with the (1,lambda), truncation-selection and ES updates of
tests/test_gpu_ga_parents.py and tests/test_gpu_ga_es.py.
"""
import ctypes as C

import numpy as np
import pytest

FLIP = 0x8000000000000000
TICK = 0.001
OBJECTIVES = ("reward", "pnl", "pnl_map", "sharpe")
KEY = {"pnl": 0, "pnl_map": 2, "sharpe": 4}
CHUNK = 1024                                      # bars per chunk of the device walk (any value gives the same bits)


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


def bits32(a):
    return np.asarray(a, np.float32).view(np.uint32)


# ------------------------------------------------------------------------------------------------ the definition
def fitness_of(v, trades):
    """The contract's post-processing of a StrategyAnalytics value."""
    v = float(v)
    if trades == 0:
        return v - 50.0
    return -50.0 if v != v else v


def post(summary, trades, objective):
    """fitness of backtest_population's / oracle.analytics' summary rows."""
    s = np.atleast_2d(np.asarray(summary, np.float64))
    return np.array([fitness_of(row[KEY[objective]], int(t)) for row, t in zip(s, np.atleast_1d(trades))], np.float64)


def stream_objective(fill_buy, fill_sell, inventory, my_bid, my_ask, mid, fee, objective, chunk=CHUNK):
    """The device walk's evaluation: returns (fitness, trades)."""
    T = len(mid)
    cash, w0, wl, prev, seen, diffs, abs_sum, trades = 0.0, 0.0, 0.0, 0.0, False, [], 0, 0
    for c0 in range(0, T, chunk):
        for t in range(c0, min(T, c0 + chunk)):
            fb, fs = bool(fill_buy[t]), bool(fill_sell[t])
            if fb:
                cash = cash - (float(my_bid[t]) + float(my_bid[t]) * fee)
            if fs:
                cash = cash + (float(my_ask[t]) - float(my_ask[t]) * fee)
            w = cash + float(inventory[t]) * float(mid[t])
            if t == 0:
                w0 = w
            if t == T - 1:
                wl = w
            abs_sum += abs(int(inventory[t]))
            if fb or fs:
                trades += 1
                if seen:
                    diffs.append(w - prev)
                prev, seen = w, True
    total = wl - w0
    if objective == "pnl":
        v = total
    elif objective == "pnl_map":
        mp = abs_sum / T if T > 0 else 0.0
        v = 0.0 if mp == 0.0 else total / mp
    else:
        v = 0.0
        if trades >= 2:
            d = np.array(diffs, np.float64)
            m = d.size
            mean = np.sum(d) / m                                  # numpy's pairwise sum, the device's np_pairwise_sum
            var = np.sum((mean - d) * (mean - d)) / (m - 1) if m > 1 else np.nan
            sd = np.sqrt(var)
            v = np.nan if sd != sd else (0.0 if sd == 0.0 else mean / sd)
    return fitness_of(v, trades), trades


def oracle_objective(orc, tr, mid, objective):
    """The oracle composition: trace -> wealth -> oracle.analytics -> the contract's post-processing."""
    inv = tr["inventory"].astype(np.float64)
    wealth = tr["cash"] + inv * np.asarray(mid, np.float64)
    is_trade = (tr["fill_buy"] | tr["fill_sell"]).astype(bool)
    s = orc.analytics(wealth, tr["inventory"], is_trade)
    return post(s, int(is_trade.sum()), objective)[0], int(is_trade.sum())


def quotes_of(tr, bz, tick):
    ask, bid = np.asarray(bz[3], np.float64), np.asarray(bz[4], np.float64)
    oa = (tr["off_a"] + tr["adv_a"]).astype(np.float64)
    ob = (tr["off_b"] + tr["adv_b"]).astype(np.float64)
    return bid - ob * tick, ask + oa * tick


def crafted_trace(kind, T=40, seed=0):
    """Trace columns with a chosen trade pattern; wealth follows the env's cash rule."""
    rng = np.random.default_rng(seed)
    mid = np.round(3.5 + np.cumsum(rng.choice([-1, 0, 1], size=T)) * TICK, 3) + TICK / 2
    my_bid, my_ask = mid - TICK * rng.integers(0, 3, size=T), mid + TICK * rng.integers(0, 3, size=T)
    fb, fs = np.zeros(T, np.int32), np.zeros(T, np.int32)
    if kind == "one":
        fb[T // 2] = 1
    elif kind == "two":
        fb[3], fs[T - 5] = 1, 1
    elif kind == "zero_std":                         # the same wealth step between every two trade rows
        mid[:] = 4.0
        my_bid[:], my_ask[:] = 3.75, 4.25
        fb[::4], fs[2::4] = 1, 1
    elif kind == "map0":                             # buy and sell in the same bars: inventory stays 0
        fb[::3], fs[::3] = 1, 1
    elif kind == "many":
        fb, fs = (rng.random(T) < 0.3).astype(np.int32), (rng.random(T) < 0.3).astype(np.int32)
    inv = np.zeros(T, np.int32)
    cur = 0
    for t in range(T):
        if cur >= 2:
            fb[t] = 0
        if cur <= -2:
            fs[t] = 0
        cur += int(fb[t]) - int(fs[t])
        inv[t] = cur
    return fb, fs, inv, my_bid, my_ask, mid


def env_wealth(fb, fs, my_bid, my_ask, inv, mid, fee):
    cash, out = 0.0, np.zeros(len(mid))
    for t in range(len(mid)):
        if fb[t]:
            cash -= my_bid[t] + my_bid[t] * fee
        if fs[t]:
            cash += my_ask[t] - my_ask[t] * fee
        out[t] = cash + float(inv[t]) * float(mid[t])
    return out


# ------------------------------------------------------------------------------------------------ CPU
@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


@pytest.mark.parametrize("kind,T", [("none", 40), ("one", 40), ("two", 40), ("zero_std", 40), ("map0", 40), ("many", 40),
                                    ("none", 0), ("one", 1), ("many", 2047), ("many", 2048), ("many", 2049)])
@pytest.mark.parametrize("fee", [0.0, 3e-4, -1e-4])
def test_stream_restatement_equals_oracle_analytics_on_crafted_traces(orc, kind, T, fee):
    fb, fs, inv, my_bid, my_ask, mid = crafted_trace(kind, T, seed=T)
    wealth = env_wealth(fb, fs, my_bid, my_ask, inv, mid, fee)
    is_trade = (fb | fs).astype(bool)
    s = orc.analytics(wealth, inv, is_trade)
    for obj in KEY:
        f, trades = stream_objective(fb, fs, inv, my_bid, my_ask, mid, fee, obj)
        assert trades == int(is_trade.sum())
        assert bits64(f) == bits64(post(s, trades, obj)[0]), (kind, T, obj)
    if kind == "two":
        assert np.isnan(s[4]) and stream_objective(fb, fs, inv, my_bid, my_ask, mid, fee, "sharpe")[0] == -50.0
    if kind == "zero_std" and fee == 0.0:
        assert s[4] == 0.0 and s[5] > 2
    if kind == "map0":
        assert s[1] == 0.0 and s[2] == 0.0 and is_trade.any()
    if kind == "none" or T == 0:
        assert all(stream_objective(fb, fs, inv, my_bid, my_ask, mid, fee, o)[0] == -50.0 for o in KEY)


@pytest.mark.parametrize("T", [1, 2047, 2048, 2049])
@pytest.mark.parametrize("use_adv", [False, True])
def test_stream_restatement_equals_oracle_analytics_on_oracle_traces(orc, T, use_adv):
    from sgmm_b200 import synthetic as syn
    bundle = syn.synthetic_bundle(-(-T // syn.BARS_PER_DAY), first_day=81)
    stats = syn.train_stats_of(bundle)
    bundle = tuple(a[:T] for a in bundle)
    bz = orc.normalise(bundle, stats) + tuple(bundle[2:])
    G = syn.policy_like_genomes(3, seed=T, out_scale=4.0, out_bias=(0.1, 0.1))[1]
    A = (np.random.default_rng(T).standard_normal((3, 1250)) * 0.6).astype(np.float32)
    for i in range(3):
        for fee in (0.0, 3e-4):
            _, _, tr = orc.rollout(G[i], A[i] if use_adv else None, bz, 1e-4, TICK, fee, trace=True)
            my_bid, my_ask = quotes_of(tr, bz, TICK)
            for obj in KEY:
                f, trades = stream_objective(tr["fill_buy"], tr["fill_sell"], tr["inventory"], my_bid, my_ask, bz[2], fee, obj)
                fo, to = oracle_objective(orc, tr, bz[2], obj)
                assert trades == to and bits64(f) == bits64(fo), (i, fee, obj)


def test_python_argument_errors_before_any_device_call(tmp_path):
    import sgmm_b200
    m = np.zeros(1250, np.float32)
    kw = dict(pop_size=8, sigma=0.05, phi=0.0, fee_rate=0.0, use_arl=False, seed=1, max_generations=2)
    for bad in ("Sharpe", "max_dd", "", None, 3, ["pnl"]):
        with pytest.raises(ValueError):
            sgmm_b200.DeviceGA(m, objective=bad, **kw)
        with pytest.raises(ValueError):
            sgmm_b200.DeviceGASweep(m, runs=[dict(seed=1, phi=0.0)], pop_size=8, use_arl=False, max_generations=2,
                                    objective=bad)
        with pytest.raises(ValueError):
            sgmm_b200.DRLEngine(save_dir=str(tmp_path / "never"), objective=bad)
        with pytest.raises(ValueError):
            sgmm_b200.rollout_population(None, m[None], phi=0.0, objective=bad)
        with pytest.raises(ValueError):
            sgmm_b200.rollout_seeded(None, m, count=1, sigma=0.05, seed=1, generation=0, phi=0.0, objective=bad)
    for obj in ("pnl", "pnl_map", "sharpe"):
        for prec in ("bf16", "tf32", "f16"):
            with pytest.raises(ValueError):
                sgmm_b200.DeviceGA(m, objective=obj, precision=prec, **kw)
            with pytest.raises(ValueError):
                sgmm_b200.rollout_population(None, m[None], phi=0.0, precision=prec, objective=obj)
        with pytest.raises(ValueError, match="precision='exact'"):
            sgmm_b200.DRLEngine(save_dir=str(tmp_path / "never"), hidden_dim=256, objective=obj)
        with pytest.raises(ValueError):
            sgmm_b200.DRLEngine(save_dir=str(tmp_path / "never"), precision="bf16", objective=obj)
    assert not (tmp_path / "never").exists()


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def sg():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import sgmm_b200
    return sgmm_b200


_BUNDLES = {}


def synthetic(sg, orc, T):
    if T not in _BUNDLES:
        from sgmm_b200 import synthetic as syn
        days = max(1, -(-T // syn.BARS_PER_DAY))
        bundle = syn.synthetic_bundle(days, first_day=80)
        stats = syn.train_stats_of(bundle)
        bundle = tuple(a[:T] for a in bundle)
        _BUNDLES[T] = (sg.Bundle.from_arrays(bundle, stats, TICK), orc.normalise(bundle, stats) + tuple(bundle[2:]))
    return _BUNDLES[T]


def genomes(P, seed, hidden=32):
    from sgmm_b200 import synthetic as syn
    return syn.policy_like_genomes(P, hidden=hidden, seed=seed, out_scale=4.0, out_bias=(0.1, 0.1))[1]


def adv_genomes(P, seed):
    return (np.random.default_rng(seed).standard_normal((P, 1250)) * 0.6).astype(np.float32)


def cuda(x):
    import torch
    return None if x is None else torch.from_numpy(np.ascontiguousarray(x)).cuda()


def check_population(sg, orc, bun, bz, G, A, *, phi, fee, hidden=32, rows=(), seeded=None):
    """Every objective of the population equals backtest_population's column post-processed, bit for bit, and the oracle
    composition on `rows`; the reward through the objective entry equals rollout_population."""
    import torch
    from sgmm_b200.analytics import backtest_population
    kw = dict(phi=phi, fee_rate=fee, hidden=hidden)
    if seeded is None:
        fr, tr = sg.rollout_population(bun, cuda(G), cuda(A), precision="exact", **kw)
        bf, bt, summ = backtest_population(bun, cuda(G), cuda(A), **kw)
    else:
        fr, tr = sg.rollout_seeded(bun, precision="exact", **seeded, **kw)
        sk = dict(seeded)
        sk["master"] = sk["master"].reshape(-1)
        bf, bt, summ = backtest_population(bun, **sk, **kw)
    assert fr.equal(bf) and tr.equal(bt)
    summ, bt = summ.cpu().numpy(), bt.cpu().numpy()
    for obj in OBJECTIVES:
        if seeded is None:
            f, t = sg.rollout_population(bun, cuda(G), cuda(A), precision="exact", objective=obj, **kw)
        else:
            f, t = sg.rollout_seeded(bun, precision="exact", objective=obj, **seeded, **kw)
        torch.cuda.synchronize()
        assert t.equal(tr), obj
        if obj == "reward":
            assert f.equal(fr)
            continue
        got = f.cpu().numpy()
        assert np.array_equal(bits64(got), bits64(post(summ, bt, obj))), obj
        for i in rows:
            _, _, tro = orc.rollout(G[i], None if A is None else A[i], bz, phi, TICK, fee, hidden=hidden, trace=True)
            fo, to = oracle_objective(orc, tro, bz[2], obj)
            assert bt[i] == to and bits64(got[i]) == bits64(fo), (obj, i)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 50, 401, 1000])
def test_h32_population_sizes(sg, orc, P):
    bun, bz = synthetic(sg, orc, 2049)
    G = genomes(P, seed=P)
    check_population(sg, orc, bun, bz, G, None, phi=1e-4, fee=3e-4, rows=[0, P - 1])
    master = G[0]
    kids = np.stack([orc.mutate(master, 0.05, 7, 3, 5 + i) for i in range(P)])
    seeded = dict(master=cuda(master), count=P, sigma=0.05, seed=7, generation=3, first_index=5)
    check_population(sg, orc, bun, bz, kids, None, phi=1e-4, fee=3e-4, rows=[0, P - 1], seeded=seeded)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [50, 401])
def test_h32_adversary(sg, orc, P):
    bun, bz = synthetic(sg, orc, 2049)
    check_population(sg, orc, bun, bz, genomes(P, seed=P + 1), adv_genomes(P, seed=P), phi=1e-4, fee=3e-4, rows=[0, P - 1])


@pytest.mark.gpu
@pytest.mark.parametrize("fee", [3e-4, -1e-4])
@pytest.mark.parametrize("phi", [0.0, 0.01])
def test_h32_fee_phi(sg, orc, fee, phi):
    bun, bz = synthetic(sg, orc, 2049)
    G, A = genomes(50, seed=3), adv_genomes(50, seed=3)
    for adv in (None, A):
        check_population(sg, orc, bun, bz, G, adv, phi=phi, fee=fee, rows=[0, 49])


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 14400])
def test_h32_lengths(sg, orc, T):
    bun, bz = synthetic(sg, orc, T)
    G, A = genomes(50, seed=T), adv_genomes(50, seed=T)
    for adv in (None, A):
        check_population(sg, orc, bun, bz, G, adv, phi=1e-4, fee=3e-4, rows=[0, 49])


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [32, 256])
def test_several_batches_equal_one(sg, orc, hidden, monkeypatch):
    bun, bz = synthetic(sg, orc, 200)
    P = 7
    G, A = genomes(P, seed=5, hidden=hidden), adv_genomes(P, seed=5)
    for adv in (None, A):
        whole = {o: sg.rollout_population(bun, cuda(G), cuda(adv), phi=1e-4, fee_rate=3e-4, hidden=hidden, precision="exact",
                                          objective=o) for o in OBJECTIVES}
        monkeypatch.setenv("SGMM_EXACT256_BATCH_BYTES", "1")          # one individual per batch
        for o in OBJECTIVES:
            f, t = sg.rollout_population(bun, cuda(G), cuda(adv), phi=1e-4, fee_rate=3e-4, hidden=hidden, precision="exact",
                                         objective=o)
            assert f.equal(whole[o][0]) and t.equal(whole[o][1]), o
        monkeypatch.delenv("SGMM_EXACT256_BATCH_BYTES")
    check_population(sg, orc, bun, bz, G, A, phi=1e-4, fee=3e-4, hidden=hidden, rows=[0, P - 1])


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "fee", "adv"])
def test_rounding_edge_episode(sg, orc, variant):
    import test_gpu_trace_population as tp                 # the rounding-edge fixtures of tests/test_gpu_rounding_edges.py
    ep = tp.make_episode("ties")
    fee = 3e-4 if variant == "fee" else 0.0
    G = tp.genomes_of(32, ep["scale"])
    A = tp.adversaries() if variant == "adv" else None
    bun = sg.Bundle(*tp.bz_of(ep), TICK)
    check_population(sg, orc, bun, tp.bz_of(ep), G, A, phi=1e-4, fee=fee, rows=range(len(G)))


@pytest.mark.gpu
@pytest.mark.parametrize("use_adv", [False, True])
def test_h256_exact(sg, orc, use_adv):
    bun, bz = synthetic(sg, orc, 300)
    G = genomes(5, seed=4, hidden=256)
    check_population(sg, orc, bun, bz, G, adv_genomes(5, seed=4) if use_adv else None, phi=1e-4, fee=3e-4, hidden=256,
                     rows=[0, 4])


@pytest.mark.gpu
def test_c_entry_reward_and_refusals(sg, orc):
    import torch
    from sgmm_b200 import _lib
    L = _lib.lib()
    bun, _ = synthetic(sg, orc, 300)
    G = cuda(genomes(20, seed=9))
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    mm = _lib.Population(32, 0, 20, G.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    f0, t0 = sg.rollout_population(bun, G, phi=1e-4, fee_rate=3e-4)
    f, t = torch.empty_like(f0), torch.empty_like(t0)
    for prec in (0, 4):
        prm = _lib.RolloutParams(1e-4, 3e-4, prec, 0, 0, 0)
        assert L.sgmm_rollout_objective(bun.handle, C.byref(mm), None, C.byref(prm), 0, f.data_ptr(), t.data_ptr(), stream) == 0
        torch.cuda.synchronize()
        assert f.equal(f0) and t.equal(t0)
    prm = _lib.RolloutParams(1e-4, 3e-4, 0, 0, 0, 0)
    for bad in (-1, 4, 1 << 20):
        assert L.sgmm_rollout_objective(bun.handle, C.byref(mm), None, C.byref(prm), bad, f.data_ptr(), t.data_ptr(), stream) == _lib.ERR_INVALID
    for prec in (1, 2, 3):
        prm = _lib.RolloutParams(1e-4, 3e-4, prec, 0, 0, 0)
        for obj in (1, 2, 3):
            assert L.sgmm_rollout_objective(bun.handle, C.byref(mm), None, C.byref(prm), obj, f.data_ptr(), t.data_ptr(),
                                            stream) == _lib.ERR_UNSUPPORTED


# ---- whole GAs
@pytest.fixture(scope="module")
def data(sg):
    from sgmm_b200 import synthetic as syn
    tb = syn.synthetic_bundle(2, first_day=70)
    vb = syn.synthetic_bundle(1, first_day=72)
    stats = syn.train_stats_of(tb)
    return tb, vb, stats, sg.Bundle.from_arrays(tb, stats, TICK), sg.Bundle.from_arrays(vb, stats, TICK)


def masters(seed, use_arl=True, hidden=32):
    from sgmm_b200 import synthetic as syn
    from sgmm_b200.policy import genome_len
    if hidden == 32:
        mm = syn.policy_like_genomes(1, seed=seed, out_scale=1.0)[0]
    else:
        mm = (np.random.default_rng(seed).standard_normal(genome_len(hidden)) * 0.05).astype(np.float32)
    adv = (np.random.default_rng(seed + 4).standard_normal(1250) * 0.5).astype(np.float32) if use_arl else None
    return mm, adv


def run_ga(sg, train, val, m, a, gens, **kw):
    ga = sg.DeviceGA(m, a, max_generations=gens, **kw)
    for _ in range(gens):
        ga.generation(train, val)
    out = ga.history(gens), ga.status(), ga.masters()
    ga.close()
    return out


def assert_same(x, y, what=""):
    (hx, sx, mx), (hy, sy, my) = x[:3], y[:3]
    for k in hx:
        assert np.array_equal(hx[k].view(np.uint8), hy[k].view(np.uint8)), (what, k)
    assert sx == sy, (what, sx, sy)
    for p, q, name in zip(mx, my, ("mm", "adv", "best")):
        assert np.array_equal(bits32(p), bits32(q)), (what, name)


def oracle_fitness(orc, z, genomes_, advs, objective, *, phi, fee, hidden):
    out = [oracle_objective(orc, orc.rollout(g, a, z, phi, TICK, fee, hidden=hidden, trace=True)[2], z[2], objective)
           for g, a in zip(genomes_, advs)]
    return np.array([o[0] for o in out], np.float64), np.array([o[1] for o in out], np.int32)


def oracle_ga(orc, tz, vz, master, adv_master, objective, *, pop, sigma, phi, fee, use_arl, seed, gens, patience,
              hidden=32, update="best", mu=1, lr=None):
    """The reference's generation loop (drl_engine.py) with fitness = the objective of oracle traces; update "best" is
    the (1,lambda) rule, "parents" truncation selection with equal weights, "es" the evolution strategy."""
    import test_gpu_ga_es as es_ref
    import test_gpu_ga_parents as par_ref
    master = master.copy()
    adv_master = None if adv_master is None else adv_master.copy()
    es = es_ref.ESRef(lr, master.size, use_arl) if update == "es" else None
    s_mm = s_adv = np.float32(sigma)
    best_val, stale, best_master = -np.inf, 0, master.copy()
    hist = {k: [] for k in ("train_f", "val_f", "train_trades", "val_trades", "sigma")}
    for gen in range(gens):
        kids = [orc.mutate(master, float(s_mm), seed, gen, i) for i in range(pop)]
        akids = [orc.mutate(adv_master, float(s_adv), seed ^ FLIP, gen, i) if use_arl else None for i in range(pop)]
        fit, trd = oracle_fitness(orc, tz, kids, akids, objective, phi=phi, fee=fee, hidden=hidden)
        best = es_ref.rank_order(fit, 1)[0]
        if update == "best":
            master = kids[best]
            if use_arl:
                adv_master = akids[es_ref.rank_order(fit, -1)[0]]
        elif update == "parents":
            w = np.full(mu, np.float32(1.0) / np.float32(mu), np.float32)
            master = par_ref.recombine(master, s_mm, seed, gen, par_ref.select_parents(fit, mu, 1), w)
            if use_arl:
                adv_master = par_ref.recombine(adv_master, s_adv, seed ^ FLIP, gen, par_ref.select_parents(fit, mu, -1), w)
        else:
            master, new_adv, _ = es.step(fit, master, adv_master, s_mm, s_adv, seed, gen)
            if use_arl:
                adv_master = new_adv
        vf, vt = oracle_fitness(orc, vz, [master], [None], objective, phi=phi, fee=fee, hidden=hidden)
        hist["train_f"].append(fit[best]); hist["train_trades"].append(trd[best])
        hist["val_f"].append(vf[0]); hist["val_trades"].append(vt[0]); hist["sigma"].append(s_mm)
        if vf[0] > best_val:
            best_val, stale, best_master = vf[0], 0, master.copy()
        else:
            stale += 1
        if stale >= patience:
            s_mm = np.float32(s_mm * np.float32(0.5))
            if use_arl:
                s_adv = np.float32(s_adv * np.float32(0.5))
            stale = 0
    return hist, master, adv_master, best_master, best_val, s_mm


def check_against_oracle(got, ref, use_arl):
    h, st, (m, a, b) = got
    ho, m_o, a_o, b_o, bv_o, s_o = ref
    assert np.array_equal(bits64(h["train_f"]), bits64(ho["train_f"]))
    assert np.array_equal(bits64(h["val_f"]), bits64(ho["val_f"]))
    assert h["train_trades"].tolist() == ho["train_trades"] and h["val_trades"].tolist() == ho["val_trades"]
    assert np.array_equal(h["sigma"], np.array(ho["sigma"], np.float32))
    assert np.array_equal(bits32(m), bits32(m_o)) and np.array_equal(bits32(b), bits32(b_o))
    assert st["best_val"] == bv_o and st["sigma"] == s_o
    if use_arl:
        assert np.array_equal(bits32(a), bits32(a_o))


def zs(orc, data):
    tb, vb, stats, _, _ = data
    return orc.normalise(tb, stats) + tb[2:], orc.normalise(vb, stats) + vb[2:]


@pytest.mark.gpu
@pytest.mark.parametrize("objective", ["pnl", "pnl_map", "sharpe"])
@pytest.mark.parametrize("use_arl", [False, True])
def test_ga_matches_oracle_composed_ga(sg, orc, data, objective, use_arl):
    tz, vz = zs(orc, data)
    _, _, _, train, val = data
    pop, gens, seed = 16, 5, 31 + int(use_arl)
    m0, a0 = masters(13, use_arl)
    got = run_ga(sg, train, val, m0, a0, gens, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=use_arl,
                 seed=seed, patience=1, objective=objective)
    ref = oracle_ga(orc, tz, vz, m0, a0, objective, pop=pop, sigma=0.05, phi=1e-4, fee=3e-4, use_arl=use_arl, seed=seed,
                    gens=gens, patience=1)
    check_against_oracle(got, ref, use_arl)
    assert got[1]["sigma"] < np.float32(0.05)                      # sigma decayed at least once


@pytest.mark.gpu
@pytest.mark.parametrize("objective", ["pnl_map", "sharpe"])
@pytest.mark.parametrize("update", ["parents", "es"])
def test_ga_composes_with_parents_and_es(sg, orc, data, objective, update):
    tz, vz = zs(orc, data)
    _, _, _, train, val = data
    pop, gens, seed = 16, 4, 41
    m0, a0 = masters(17, True)
    kw = dict(parents=5) if update == "parents" else dict(es_lr=0.02)
    got = run_ga(sg, train, val, m0, a0, gens, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=True, seed=seed,
                 patience=1, objective=objective, **kw)
    ref = oracle_ga(orc, tz, vz, m0, a0, objective, pop=pop, sigma=0.05, phi=1e-4, fee=0.0, use_arl=True, seed=seed,
                    gens=gens, patience=1, update=update, mu=5, lr=0.02)
    check_against_oracle(got, ref, True)


@pytest.mark.gpu
def test_h256_exact_ga_matches_oracle_composed_ga(sg, orc):
    from sgmm_b200 import synthetic as syn
    full = syn.synthetic_bundle(1, first_day=60)
    tb = tuple(np.ascontiguousarray(x[:240]) for x in full)
    vb = tuple(np.ascontiguousarray(x[240:400]) for x in full)
    stats = syn.train_stats_of(full)
    train, val = sg.Bundle.from_arrays(tb, stats, TICK), sg.Bundle.from_arrays(vb, stats, TICK)
    tz, vz = orc.normalise(tb, stats) + tb[2:], orc.normalise(vb, stats) + vb[2:]
    m0, a0 = masters(5, True, hidden=256)
    got = run_ga(sg, train, val, m0, a0, 3, pop_size=6, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=True, seed=9, patience=1,
                 hidden=256, precision="exact", objective="sharpe")
    ref = oracle_ga(orc, tz, vz, m0, a0, "sharpe", pop=6, sigma=0.05, phi=1e-4, fee=0.0, use_arl=True, seed=9, gens=3,
                    patience=1, hidden=256)
    check_against_oracle(got, ref, True)


@pytest.mark.gpu
def test_sweep_shards_graph_and_reward_call(sg, data):
    import torch
    from sgmm_b200.dist import device_tensor
    _, _, _, train, val = data
    runs = [dict(seed=11, phi=0.0, fee_rate=0.0, sigma=0.05, patience=1),
            dict(seed=12, phi=1e-4, fee_rate=3e-4, sigma=0.02, patience=2),
            dict(seed=2 ** 63 + 5, phi=0.01, fee_rate=-1e-4, sigma=0.08, patience=3)]
    K, pop, gens = len(runs), 24, 5
    mm = np.stack([masters(3 + r)[0] for r in range(K)])
    adv = np.stack([masters(3 + r)[1] for r in range(K)])
    for obj in ("pnl", "sharpe"):                                   # sweep runs equal their solo GAs
        ga = sg.DeviceGASweep(mm, adv, runs=runs, pop_size=pop, use_arl=True, max_generations=gens, objective=obj)
        for _ in range(gens):
            ga.generation(train, val)
        for r in range(K):
            solo = run_ga(sg, train, val, mm[r], adv[r], gens, pop_size=pop, use_arl=True, precision="exact", objective=obj,
                          **runs[r])
            assert_same((ga.history(r, gens), ga.status(r), ga.masters(r)), solo, f"{obj} run {r}")
        ga.close()
    m0, a0 = masters(23)
    kw = dict(pop_size=50, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=True, seed=77, patience=2, objective="pnl_map")
    shards = [sg.DeviceGA(m0, a0, shard=(0, 25, 25), max_generations=gens, **kw),
              sg.DeviceGA(m0, a0, shard=(25, 25, 25), max_generations=gens, **kw)]
    views = []
    for ga in shards:
        _, _, base, bb, nb, my = ga.buffers()
        views.append((device_tensor(base, nb * bb, torch.uint8, ga.device), bb, my))
    for _ in range(gens):
        for ga in shards:
            ga.evaluate(train)
        for (dst, bb, _), (src, _, my) in ((views[0], views[1]), (views[1], views[0])):
            dst[my * bb:(my + 1) * bb].copy_(src[my * bb:(my + 1) * bb])
        for ga in shards:
            ga.select(val)
    whole = run_ga(sg, train, val, m0, a0, gens, **kw)
    for i, ga in enumerate(shards):
        assert_same((ga.history(gens), ga.status(), ga.masters()), whole, f"shard {i}")
        ga.close()
    kw = dict(pop_size=300, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=True, seed=3, patience=2, max_generations=8,
              objective="sharpe")                                  # a captured generation's replay equals eager ones
    eager = sg.DeviceGA(m0, a0, **kw)
    for _ in range(7):
        eager.generation(train, val)
    graphed = sg.DeviceGA(m0, a0, **kw)
    graphed.generation(train, val)
    torch.cuda.synchronize()
    g = graphed.capture(train, val)
    for _ in range(6):
        g.replay()
    torch.cuda.synchronize()
    assert_same((eager.history(7), eager.status(), eager.masters()), (graphed.history(7), graphed.status(), graphed.masters()))
    eager.close()
    graphed.close()
    from sgmm_b200 import _lib                                      # set_objective(REWARD) gives the bits of no call
    kw = dict(pop_size=24, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=True, seed=5, patience=1)
    plain = run_ga(sg, train, val, m0, a0, 3, **kw)
    ga = sg.DeviceGA(m0, a0, max_generations=3, **kw)
    assert _lib.lib().sgmm_ga_set_objective(ga._h, 0, C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
    for _ in range(3):
        ga.generation(train, val)
    assert_same((ga.history(3), ga.status(), ga.masters()), plain, "reward")
    ga.close()


@pytest.mark.gpu
def test_set_objective_refusals(sg, data):
    import torch
    from sgmm_b200 import _lib
    L = _lib.lib()
    _, _, _, train, val = data
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    m0, a0 = masters(1)
    kw = dict(sigma=0.05, phi=0.0, fee_rate=0.0, use_arl=True, seed=1, max_generations=3, pop_size=8)
    ga = sg.DeviceGA(m0, a0, **kw)
    for bad in (-1, 4, 99):
        assert L.sgmm_ga_set_objective(ga._h, bad, stream) == _lib.ERR_INVALID
    assert L.sgmm_ga_set_objective(None, 1, stream) == _lib.ERR_INVALID
    assert L.sgmm_ga_set_objective(ga._h, 3, stream) == 0 and L.sgmm_ga_set_objective(ga._h, 1, stream) == 0
    ga.generation(train, val)
    assert L.sgmm_ga_set_objective(ga._h, 2, stream) == _lib.ERR_INVALID
    assert "already" in L.sgmm_last_error().decode()
    with pytest.raises(_lib.SgmmError):
        ga.set_objective("pnl")
    ga.close()
    ga = sg.DeviceGA(m0, a0, **kw)                                  # evaluate alone closes the window too
    ga.evaluate(train)
    assert L.sgmm_ga_set_objective(ga._h, 1, stream) == _lib.ERR_INVALID
    ga.close()
    for prec in ("bf16", "f16", "tf32"):
        ga = sg.DeviceGA(m0, a0, precision=prec, **kw)
        for obj in (1, 2, 3):
            assert L.sgmm_ga_set_objective(ga._h, obj, stream) == _lib.ERR_UNSUPPORTED
        assert L.sgmm_ga_set_objective(ga._h, 0, stream) == 0
        ga.close()


@pytest.mark.gpu
def test_drl_engine_objective_equals_its_device_compositions(sg, data, tmp_path):
    import torch
    tb, vb, stats, train, val = data
    gens, pop = 6, 20
    torch.manual_seed(5)
    eng = sg.DRLEngine(pop_size=pop, phi=1e-4, tick_size=TICK, use_arl=True, patience=2, seed=99, objective="sharpe",
                       save_dir=str(tmp_path / "e"))
    m0 = eng.mm_evolver.master_policy.get_weights().clone()
    a0 = eng.adv_evolver.master_policy.get_weights().clone()
    policy, hist = eng.train(tb, vb, stats, generations=gens, log_every=3, verbose=False)
    h, st, (mm, adv, best) = run_ga(sg, train, val, m0, a0, gens, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=0.0,
                                    use_arl=True, seed=99, patience=2, objective="sharpe")
    assert np.array_equal(bits64(hist["val_f"]), bits64(h["val_f"]))
    assert np.array_equal(bits64(hist["train_f"]), bits64(h["train_f"]))
    assert hist["train_trades"] == h["train_trades"].tolist()
    want = best if st["best_val"] > -np.inf else mm
    assert np.array_equal(bits32(policy.get_weights().numpy()), bits32(want))
    assert np.array_equal(bits32(eng.adv_evolver.master_policy.get_weights().numpy()), bits32(adv))
    if st["best_val"] > -np.inf:
        snap = sg.TradingPolicy(hidden_dim=32)
        snap.load_state_dict(torch.load(str(tmp_path / "e" / "agent_best_val_0.0001.pth")))
        assert np.array_equal(bits32(snap.get_weights().numpy()), bits32(best))       # the checkpoint
    eng2 = sg.DRLEngine(pop_size=pop, phi=1e-4, tick_size=TICK, use_arl=True, patience=2, objective="pnl_map",
                        save_dir=str(tmp_path / "s"))
    eng2.mm_evolver.master_policy.set_weights(m0)
    eng2.adv_evolver.master_policy.set_weights(a0)
    out = eng2.train_sweep(tb, vb, stats, gens, phis=[1e-4, 0.01], seeds=[5, 6], log_every=3, verbose=False)
    sw = sg.DeviceGASweep(m0, a0, runs=[dict(seed=5, phi=1e-4, patience=2), dict(seed=6, phi=0.01, patience=2)],
                          pop_size=pop, use_arl=True, max_generations=gens, objective="pnl_map")
    for _ in range(gens):
        sw.generation(train, val)
    for r in range(2):
        p, hh = out[r]
        hs, ss = sw.history(r, gens), sw.status(r)
        assert np.array_equal(bits64(hh["val_f"]), bits64(hs["val_f"]))
        assert np.array_equal(bits64(hh["train_f"]), bits64(hs["train_f"]))
        mm_r, _, b = sw.masters(r)
        assert np.array_equal(bits32(p.get_weights().numpy()), bits32(b if ss["best_val"] > -np.inf else mm_r))
    sw.close()
