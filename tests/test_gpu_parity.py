"""GPU (-m gpu): the CUDA path, called through the C ABI, against the oracle and the golden
fixtures.  Integer work (offsets, fills, inventory, trades) and -- because the kernels implement
the oracle's SGMM-F32 order exactly -- every fp32/fp64 quantity are compared BIT-EXACTLY.  The only
tolerance in this file is the reference-facing one: fitness within 1e-5 relative of the imported
reference's own output (tests/golden/ref_rollouts.npz), as BASELINE.json's north_star states.
"""
import numpy as np
import pytest
import torch

from conftest import REF_CASES, ref_case

pytestmark = pytest.mark.gpu

REL_TOL_VS_REFERENCE = 1e-5


@pytest.fixture(scope="module")
def sg():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import sgmm_b200
    return sgmm_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


def bits32(a):
    return np.asarray(a, np.float32).view(np.uint32)


# ----------------------------------------------------------------------------------------------
# bundle prologue: integer fill thresholds
# ----------------------------------------------------------------------------------------------
def test_fill_thresholds_match_exact_fp64_quotes(sg):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(3, first_day=20)
    stats = synthetic.train_stats_of(bundle)
    b = sg.Bundle.from_arrays(bundle, stats, 0.001)
    ka, kb = b.thresholds()
    _, _, mid, ask, bid, bmax, smin = bundle
    tick = 0.001
    ks = np.arange(-40, 41)
    for t in range(len(mid)):
        qa = ask[t] + ks * tick          # numpy: int*float -> f64 product, then f64 add (two roundings)
        qb = bid[t] - ks * tick
        ta = ks[qa <= bmax[t]]
        tb = ks[qb >= smin[t]]
        want_a = ta.max() if ta.size else np.iinfo(np.int32).min
        want_b = tb.max() if tb.size else np.iinfo(np.int32).min
        assert ka[t] == want_a, (t, ka[t], want_a)
        assert kb[t] == want_b, (t, kb[t], want_b)
    assert (ka == np.iinfo(np.int32).min).sum() == np.isnan(bmax).sum()


# exact-touch grids: (first price, step, decimals, tick) -- the 3.400-3.599 grid of SURVEY 7.4-2, the reference's default tick
# 0.01 on the same 3-decimal prices, 2-decimal prices near 35, 4-decimal prices near 0.9 and 1-decimal prices near 3800
EXACT_TOUCH_GRIDS = [(3.400, 0.001, 3, 0.001), (3.400, 0.001, 3, 0.01), (34.00, 0.01, 2, 0.01), (0.8800, 0.0001, 4, 0.0001),
                     (3800.0, 0.2, 1, 0.2)]


def test_fill_thresholds_adversarial_grid(sg):
    """SURVEY 7.4-2: on a 3.400-3.599 grid ~10 % of exact-touch cases differ between
    fl(p +- fl(k*tick)) and the fused/real-arithmetic value; the thresholds must follow the former.
    The same holds on every price grid and tick in EXACT_TOUCH_GRIDS."""
    for first, step, dec, tick in EXACT_TOUCH_GRIDS:
        p = np.round(first + np.arange(200) * step, dec)
        ks = np.arange(-12, 13)
        ask = np.repeat(p, ks.size)
        k = np.tile(ks, p.size)
        bound_a = np.round(ask + k * tick, dec)            # "exact touch" bounds on the price grid
        bound_b = np.round(ask - k * tick, dec)
        z = np.zeros(ask.size, np.float32)
        b = sg.Bundle(z, z, ask, ask, ask, bound_a, bound_b, tick)
        ka, kb = b.thresholds()
        kk = np.arange(-40, 41)
        for i in range(ask.size):
            assert ka[i] == kk[(ask[i] + kk * tick) <= bound_a[i]].max(), (tick, i)
            assert kb[i] == kk[(ask[i] - kk * tick) >= bound_b[i]].max(), (tick, i)
        naive = np.round((bound_a - ask) / tick).astype(int)
        assert (naive != ka).sum() > 0, "grid should contain cases where the naive integer engine is wrong"
    # infinities
    z1 = np.zeros(4, np.float32)
    b2 = sg.Bundle(z1, z1, np.ones(4), np.ones(4), np.ones(4), np.array([np.inf, -np.inf, np.nan, 1.0]),
                   np.array([-np.inf, np.inf, np.nan, 1.0]), 0.001)
    ka2, kb2 = b2.thresholds()
    imin, imax = np.iinfo(np.int32).min, np.iinfo(np.int32).max
    assert ka2.tolist() == [imax, imin, imin, 0] and kb2.tolist() == [imax, imin, imin, 0]


# ----------------------------------------------------------------------------------------------
# trace kernel: teacher-forced replay of the reference's golden backtests (env arithmetic)
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["drl", "arl", "glft", "foic"])
def test_device_replay_of_golden_backtests_bit_exact(sg, golden, name):
    b = golden.backtest
    T = 960
    off = np.stack([b[f"{name}.off_a"], b[f"{name}.off_b"]], 1).astype(np.int32)
    fb, fs = b[f"{name}.fill_buy"], b[f"{name}.fill_sell"]
    z = np.zeros(T, np.float32)
    bun = sg.Bundle(z, z, b[f"{name}.mid"], b[f"{name}.ask"], b[f"{name}.bid"],
                    np.where(fs == 1, np.inf, -np.inf), np.where(fb == 1, -np.inf, np.inf), 0.001)
    fit, trades, tr = sg.rollout_trace(bun, None, None, off, phi=1e-4, fee_rate=0.0)
    assert np.array_equal(tr["fill_buy"], fb) and np.array_equal(tr["fill_sell"], fs)
    assert np.array_equal(tr["inventory"], b[f"{name}.inventory"])
    for col in ("cash", "reward", "pnl_reward", "inventory_reward", "fee_paid"):
        assert np.array_equal(bits64(tr[col]), bits64(b[f"{name}.{col}"])), col
    assert trades == int(((fb == 1) | (fs == 1)).sum())
    assert fit == np.cumsum(b[f"{name}.reward"])[-1]
    df = sg.StrategyRecorder.from_trace(tr, (b[f"{name}.s1_pred"], b[f"{name}.s2_pred"], b[f"{name}.mid"],
                                             b[f"{name}.ask"], b[f"{name}.bid"], None, None)).to_dataframe()
    # the derived columns come from the kernel (running fp64 sums in bar order) and equal the reference's pandas columns bit for bit
    for c in ("wealth", "cum_reward", "spread", "skew", "cum_fees", "realized_pnl", "unrealized_pnl"):
        assert np.array_equal(df[c].to_numpy(), b[f"{name}.{c}"]), c
        if c in tr:
            assert np.array_equal(np.asarray(tr[c], df[c].to_numpy().dtype), b[f"{name}.{c}"]), c
    assert all(k in tr for k in ("spread", "wealth", "cum_reward", "skew", "cum_fees", "unrealized_pnl"))


def test_device_policy_reproduces_arl_checkpoint_actions(sg, golden):
    """960/960 recorded actions of the shipped ARL agent, closed loop on the device."""
    b, c = golden.backtest, golden.ckpt
    s1, s2 = b["arl.s1_pred"], b["arl.s2_pred"]
    z1 = ((s1 - c["train_stats_s1_m"][()]) / c["train_stats_s1_s"][()]).astype(np.float32)
    z2 = ((s2 - c["train_stats_s2_m"][()]) / c["train_stats_s2_s"][()]).astype(np.float32)
    fb, fs = b["arl.fill_buy"], b["arl.fill_sell"]
    my_ask = b["arl.ask"] + b["arl.off_a"] * 0.001
    my_bid = b["arl.bid"] - b["arl.off_b"] * 0.001
    bun = sg.Bundle(z1, z2, b["arl.mid"], b["arl.ask"], b["arl.bid"],
                    np.where(fs == 1, my_ask, my_ask - 0.0005), np.where(fb == 1, my_bid, my_bid + 0.0005), 0.001)
    fit, trades, tr = sg.rollout_trace(bun, c["510300_with_adv"], phi=1e-4)
    assert np.array_equal(tr["off_a"], b["arl.off_a"]) and np.array_equal(tr["off_b"], b["arl.off_b"])
    assert np.array_equal(tr["inventory"], b["arl.inventory"])
    assert np.array_equal(bits64(tr["reward"]), bits64(b["arl.reward"]))
    assert np.array_equal(bits64(tr["cash"]), bits64(b["arl.cash"]))
    # the population kernel on the same episode
    g = torch.from_numpy(c["510300_with_adv"].copy()).reshape(1, -1).cuda()
    f2, t2 = sg.rollout_population(bun, g, phi=1e-4)
    assert f2.item() == fit and t2.item() == trades
    assert abs(fit - b["arl.cum_reward"][-1]) <= 1e-12


# ----------------------------------------------------------------------------------------------
# closed loop vs the oracle (bit-exact) and vs the imported reference (1e-5 relative)
# ----------------------------------------------------------------------------------------------
def _case_bundle(sg, orc, cs):
    z1, z2 = orc.normalise(cs["bundle"], cs["stats"])
    bz = (z1, z2) + cs["bundle"][2:]
    bun = sg.Bundle.from_arrays(cs["bundle"], cs["stats"], cs["tick"])
    return bz, bun


@pytest.mark.parametrize("name", REF_CASES)
def test_trace_kernel_vs_oracle_bitwise(sg, orc, golden, name):
    cs = ref_case(golden.ref, name)
    bz, bun = _case_bundle(sg, orc, cs)
    for i in range(min(4, cs["genomes"].shape[0])):
        adv = cs["adv"][i] if cs["use_arl"] else None
        fo, to, tro = orc.rollout(cs["genomes"][i], adv, bz, cs["phi"], cs["tick"], cs["fee"], trace=True)
        fg, tg, trg = sg.rollout_trace(bun, cs["genomes"][i], adv, phi=cs["phi"], fee_rate=cs["fee"])
        for k in ("off_a", "off_b", "adv_a", "adv_b", "fill_buy", "fill_sell", "inventory"):
            assert np.array_equal(trg[k], tro[k]), (name, i, k)
        for k in ("raw_a", "raw_b"):
            assert np.array_equal(bits32(trg[k]), bits32(tro[k])), (name, i, k)
        for k in ("cash", "reward", "pnl_reward", "inventory_reward", "fee_paid"):
            assert np.array_equal(bits64(trg[k]), bits64(tro[k])), (name, i, k)
        assert (bits64(fg), tg) == (bits64(fo), to)


@pytest.mark.parametrize("units", [1, 2, 4])
@pytest.mark.parametrize("name", REF_CASES)
def test_population_kernel_vs_oracle_and_reference(sg, orc, golden, name, units):
    cs = ref_case(golden.ref, name)
    bz, bun = _case_bundle(sg, orc, cs)
    P = cs["genomes"].shape[0]
    g = torch.from_numpy(cs["genomes"]).cuda()
    a = torch.from_numpy(cs["adv"]).cuda() if cs["use_arl"] else None
    fit, trd = sg.rollout_population(bun, g, a, phi=cs["phi"], fee_rate=cs["fee"], units_per_lane=units)
    fit, trd = fit.cpu().numpy(), trd.cpu().numpy()
    fo, to = orc.rollout_population(bz, cs["phi"], cs["tick"], cs["fee"], genomes=cs["genomes"],
                                    adv_genomes=cs["adv"], use_adv=cs["use_arl"], nthreads=4)
    assert np.array_equal(bits64(fit), bits64(fo)), (fit, fo)          # bit-exact vs the oracle
    assert np.array_equal(trd, to)
    # vs the imported reference: trades identical, fitness within 1e-5 relative -- except for a
    # trajectory the oracle itself flags as having hit a near-tie of the reference's rounding
    n_ok = 0
    for i in range(P):
        if trd[i] == cs["trades"][i] and abs(fit[i] - cs["fitness"][i]) <= REL_TOL_VS_REFERENCE * abs(cs["fitness"][i]):
            n_ok += 1
        else:
            assert cs["margin"][i] < 1e-4, (name, i, fit[i], cs["fitness"][i])
    assert n_ok >= P - 1


def test_host_entry_matches_device_entry(sg, orc, golden):
    cs = ref_case(golden.ref, "arl_fee")
    bz, bun = _case_bundle(sg, orc, cs)
    f_dev, t_dev = sg.rollout_population(bun, torch.from_numpy(cs["genomes"]).cuda(), torch.from_numpy(cs["adv"]).cuda(),
                                         phi=cs["phi"], fee_rate=cs["fee"])
    f_host, t_host = sg.rollout_population(bun, cs["genomes"], cs["adv"], phi=cs["phi"], fee_rate=cs["fee"])
    assert isinstance(f_host, np.ndarray)
    assert np.array_equal(bits64(f_host), bits64(f_dev.cpu().numpy())) and np.array_equal(t_host, t_dev.cpu().numpy())
    # list-of-tensors form (what NeuroEvolution.ask returns)
    f_list, _ = sg.rollout_population(bun, [torch.from_numpy(x.copy()) for x in cs["genomes"]],
                                      [torch.from_numpy(x.copy()) for x in cs["adv"]], phi=cs["phi"], fee_rate=cs["fee"])
    assert np.array_equal(bits64(f_list), bits64(f_host))


def test_evaluate_individual_drop_in(sg, golden):
    cs = ref_case(golden.ref, "fresh")
    for i in range(3):
        f, n = sg.evaluate_individual(torch.from_numpy(cs["genomes"][i].copy()), None, cs["bundle"], cs["phi"],
                                      cs["tick"], cs["fee"], cs["stats"], use_arl=False)
        assert isinstance(f, np.float64) and isinstance(n, int)
        assert n == cs["trades"][i] and abs(f - cs["fitness"][i]) <= REL_TOL_VS_REFERENCE * abs(cs["fitness"][i])
    cs = ref_case(golden.ref, "arl")
    f, n = sg.evaluate_individual(torch.from_numpy(cs["genomes"][2].copy()), torch.from_numpy(cs["adv"][2].copy()),
                                  cs["bundle"], cs["phi"], cs["tick"], cs["fee"], cs["stats"], use_arl=True)
    assert n == cs["trades"][2] and abs(f - cs["fitness"][2]) <= REL_TOL_VS_REFERENCE * abs(cs["fitness"][2])
    # use_arl=False ignores the adversary weights (drl_engine.py:17-21)
    f2, _ = sg.evaluate_individual(torch.from_numpy(cs["genomes"][2].copy()), torch.from_numpy(cs["adv"][2].copy()),
                                   cs["bundle"], cs["phi"], cs["tick"], cs["fee"], cs["stats"], use_arl=False)
    f3, _ = sg.evaluate_individual(torch.from_numpy(cs["genomes"][2].copy()), None,
                                   cs["bundle"], cs["phi"], cs["tick"], cs["fee"], cs["stats"], use_arl=False)
    assert f2 == f3


# ----------------------------------------------------------------------------------------------
# edge cases: empty / ragged sizes
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [0, 1, 2, 127, 128, 129, 511, 513, 1000])
@pytest.mark.parametrize("P", [1, 3, 33])
def test_ragged_sizes(sg, orc, T, P):
    from sgmm_b200 import synthetic
    full = synthetic.synthetic_bundle(5, first_day=30)
    bundle = tuple(a[:T] for a in full)
    stats = synthetic.train_stats_of(full)
    _, genomes = synthetic.policy_like_genomes(P, seed=T + P, out_scale=6.0, out_bias=(0.1, 0.1))
    z1, z2 = orc.normalise(bundle, stats)
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    fo, to = orc.rollout_population((z1, z2) + bundle[2:], 1e-4, 0.001, 0.0, genomes=genomes, nthreads=4)
    for units in (1, 2, 4):
        for warps in (0, 1, 3):
            f, t = sg.rollout_population(bun, torch.from_numpy(genomes).cuda(), phi=1e-4, units_per_lane=units,
                                         warps_per_cta=warps)
            assert np.array_equal(bits64(f.cpu().numpy()), bits64(fo)), (T, P, units, warps)
            assert np.array_equal(t.cpu().numpy(), to)
    if T == 0:
        assert np.all(fo == -50.0) and np.all(to == 0)


def test_empty_population(sg):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(1)
    bun = sg.Bundle.from_arrays(bundle, synthetic.train_stats_of(bundle), 0.001)
    f, t = sg.rollout_population(bun, torch.zeros(0, 1250, device="cuda"), phi=1e-4)
    assert f.numel() == 0 and t.numel() == 0


# ----------------------------------------------------------------------------------------------
# device-resident ask: counter-based children, bit-identical to the oracle's
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_adv", [False, True])
def test_seeded_children_match_oracle(sg, orc, use_adv):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(2, first_day=40)
    stats = synthetic.train_stats_of(bundle)
    z1, z2 = orc.normalise(bundle, stats)
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    master, _ = synthetic.policy_like_genomes(1, seed=3, out_scale=6.0, out_bias=(0.1, 0.1))
    adv_master = np.random.default_rng(9).standard_normal(1250).astype(np.float32) if use_adv else None
    kw = dict(count=45, sigma=0.05, seed=0x1234_5678_9ABC_DEF0, generation=7, first_index=1000)
    fo, to = orc.rollout_population((z1, z2) + bundle[2:], 1e-4, 0.001, 0.0, master=master, adv_master=adv_master,
                                    adv_sigma=0.3, use_adv=use_adv, nthreads=4, **kw)
    f, t = sg.rollout_seeded(bun, torch.from_numpy(master).cuda(),
                             adv_master=None if adv_master is None else torch.from_numpy(adv_master).cuda(),
                             adv_sigma=0.3, phi=1e-4, **kw)
    assert np.array_equal(bits64(f.cpu().numpy()), bits64(fo)) and np.array_equal(t.cpu().numpy(), to)
    # explicit genomes built by the oracle's mutate give the same answer: ask is layout-independent
    kids = np.stack([orc.mutate(master, 0.05, kw["seed"], 7, 1000 + i) for i in range(45)])
    if not use_adv:
        f2, _ = sg.rollout_population(bun, torch.from_numpy(kids).cuda(), phi=1e-4)
        assert np.array_equal(bits64(f2.cpu().numpy()), bits64(fo))
    # sharding invariance: two shards == one population
    fa, _ = sg.rollout_seeded(bun, torch.from_numpy(master).cuda(), count=20, sigma=0.05, seed=kw["seed"], generation=7,
                              first_index=1000, adv_master=None if adv_master is None else torch.from_numpy(adv_master).cuda(),
                              adv_sigma=0.3, phi=1e-4)
    fb, _ = sg.rollout_seeded(bun, torch.from_numpy(master).cuda(), count=25, sigma=0.05, seed=kw["seed"], generation=7,
                              first_index=1020, adv_master=None if adv_master is None else torch.from_numpy(adv_master).cuda(),
                              adv_sigma=0.3, phi=1e-4)
    assert np.array_equal(torch.cat([fa, fb]).cpu().numpy(), f.cpu().numpy())


# ----------------------------------------------------------------------------------------------
# GA on the device vs the same GA composed from oracle pieces
# ----------------------------------------------------------------------------------------------
def _oracle_ga(orc, train_bz, val_bz, master, adv_master, *, pop, sigma, phi, tick, fee, use_arl, seed, gens, patience):
    FLIP = 0x8000000000000000
    master = master.copy()
    adv_master = None if adv_master is None else adv_master.copy()
    s_mm = s_adv = np.float32(sigma)
    best_val, stale = -np.inf, 0
    best_master = master.copy()
    hist = {k: [] for k in ("train_f", "val_f", "train_trades", "val_trades", "sigma")}
    for gen in range(gens):
        fit, trd = orc.rollout_population(train_bz, phi, tick, fee, master=master, sigma=float(s_mm),
                                          adv_master=adv_master, adv_sigma=float(s_adv), use_adv=use_arl,
                                          seed=seed, generation=gen, count=pop, nthreads=4)
        best = int(np.argmax(fit))                                        # model.py:74
        master = orc.mutate(master, float(s_mm), seed, gen, best)         # master <- best child
        if use_arl:
            abest = int(np.argmax(-fit))                                  # drl_engine.py:124-125
            adv_master = orc.mutate(adv_master, float(s_adv), seed ^ FLIP, gen, abest)
        vf, vt = orc.rollout(master, None, val_bz, phi, tick, fee)      # drl_engine.py:129-140
        hist["train_f"].append(fit[best]); hist["train_trades"].append(trd[best])
        hist["val_f"].append(vf); hist["val_trades"].append(vt); hist["sigma"].append(s_mm)
        if vf > best_val:
            best_val, stale, best_master = vf, 0, master.copy()
        else:
            stale += 1
        if stale >= patience:
            s_mm = np.float32(s_mm * np.float32(0.5))
            if use_arl:
                s_adv = np.float32(s_adv * np.float32(0.5))
            stale = 0
    return hist, master, adv_master, best_master, best_val, float(s_mm)


@pytest.mark.parametrize("use_arl,phi,tick", [pytest.param(False, 1e-4, 0.001, id="False"), pytest.param(True, 1e-4, 0.001, id="True"),
                                              pytest.param(False, 0.01, 0.01, id="False-reference_defaults"),
                                              pytest.param(True, 0.01, 0.01, id="True-reference_defaults")])
def test_device_ga_matches_oracle_ga(sg, orc, use_arl, phi, tick):
    """phi = 0.01, tick 0.01: DRLEngine's and FTPEnv's own defaults (Env/drl_engine.py, Env/market_env.py)."""
    from sgmm_b200 import synthetic
    from sgmm_b200.engine import DeviceGA
    tb = synthetic.synthetic_bundle(2, first_day=50)
    vb = synthetic.synthetic_bundle(1, first_day=52)
    stats = synthetic.train_stats_of(tb)
    train = sg.Bundle.from_arrays(tb, stats, tick)
    val = sg.Bundle.from_arrays(vb, stats, tick)
    tz = orc.normalise(tb, stats) + tb[2:]
    vz = orc.normalise(vb, stats) + vb[2:]
    master, _ = synthetic.policy_like_genomes(1, seed=21, out_scale=1.0)
    adv_master = (np.random.default_rng(4).standard_normal(1250) * 0.5).astype(np.float32) if use_arl else None
    gens, pop, patience = 9, 24, 3
    ga = DeviceGA(master, adv_master, pop_size=pop, sigma=0.05, phi=phi, fee_rate=0.0, use_arl=use_arl, seed=77,
                  max_generations=gens, patience=patience)
    for _ in range(gens):
        ga.generation(train, val)
    h = ga.history(gens)
    st = ga.status()
    mm, adv, best = ga.masters()
    ho, m_o, a_o, b_o, bv_o, s_o = _oracle_ga(orc, tz, vz, master, adv_master, pop=pop, sigma=0.05, phi=phi, tick=tick, fee=0.0,
                                               use_arl=use_arl, seed=77, gens=gens, patience=patience)
    assert np.array_equal(bits64(h["train_f"]), bits64(ho["train_f"]))
    assert np.array_equal(bits64(h["val_f"]), bits64(ho["val_f"]))
    assert h["train_trades"].tolist() == ho["train_trades"] and h["val_trades"].tolist() == ho["val_trades"]
    assert np.array_equal(h["sigma"], np.array(ho["sigma"], np.float32))
    assert np.array_equal(bits32(mm), bits32(m_o)) and np.array_equal(bits32(best), bits32(b_o))
    if use_arl:
        assert np.array_equal(bits32(adv), bits32(a_o))
    assert st["generation"] == gens and st["best_val"] == bv_o and st["sigma"] == s_o


def test_drl_engine_train_drop_in(sg, tmp_path, capsys):
    from sgmm_b200 import synthetic
    tb = synthetic.synthetic_bundle(2, first_day=60)
    vb = synthetic.synthetic_bundle(1, first_day=62)
    stats = synthetic.train_stats_of(tb)
    torch.manual_seed(0)
    eng = sg.DRLEngine(pop_size=50, sigma=0.05, phi=1e-4, tick_size=0.001, save_dir=str(tmp_path / "ck"), use_arl=True)
    assert hasattr(eng, "mm_evolver") and hasattr(eng, "adv_evolver")
    policy, hist = eng.train(tb, vb, stats, generations=6)
    assert sorted(hist) == ['gen', 'train_f', 'train_trades', 'val_f', 'val_trades']
    assert hist['gen'] == list(range(6)) and all(len(hist[k]) == 6 for k in hist)
    assert isinstance(policy, sg.TradingPolicy)
    out = capsys.readouterr().out
    assert "Gen 000 | ARL:ON | Best Train:" in out and "Gen 005" in out
    ck = tmp_path / "ck" / "agent_best_val_0.0001.pth"
    assert ck.exists()
    sd = torch.load(ck, weights_only=True)
    assert list(sd.keys()) == [f"net.{i}.{p}" for i in (0, 2, 4) for p in ("weight", "bias")]
    # the returned policy is the best-on-validation master and reproduces its validation fitness
    f, n = sg.evaluate_individual(policy.get_weights(), None, vb, 1e-4, 0.001, 0.0, stats)
    assert f == max(hist['val_f'])
    # best train fitness of a generation is the max over that generation's children: monotone link
    assert all(np.isfinite(hist['train_f']))


# ----------------------------------------------------------------------------------------------
# full-size properties (BASELINE config 2: P=4096, T=14400)
# ----------------------------------------------------------------------------------------------
def test_full_size_properties(sg, orc):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(60)
    stats = synthetic.train_stats_of(bundle)
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    assert bun.T == 14400
    P = 4096
    _, genomes = synthetic.policy_like_genomes(P, seed=0, out_scale=1.0)
    g = torch.from_numpy(genomes).cuda()
    f4, t4 = sg.rollout_population(bun, g, phi=1e-4)
    f1, t1 = sg.rollout_population(bun, g, phi=1e-4, units_per_lane=1)
    f2, t2 = sg.rollout_population(bun, g, phi=1e-4, units_per_lane=2, warps_per_cta=5)
    assert torch.equal(f4, f1) and torch.equal(f4, f2) and torch.equal(t4, t1) and torch.equal(t4, t2)
    # permutation equivariance: individuals do not interact
    perm = torch.randperm(P, generator=torch.Generator().manual_seed(1)).cuda()
    fp, tp = sg.rollout_population(bun, g[perm].contiguous(), phi=1e-4)
    assert torch.equal(fp, f4[perm]) and torch.equal(tp, t4[perm])
    assert int(t4.max()) <= bun.T and int(t4.min()) >= 0
    assert torch.isfinite(f4).all()
    # a seeded sample against the oracle, full length
    idx = [0, 1, 777, 2048, 4095]
    z1, z2 = orc.normalise(bundle, stats)
    fo, to = orc.rollout_population((z1, z2) + bundle[2:], 1e-4, 0.001, 0.0, genomes=genomes[idx], nthreads=5)
    assert np.array_equal(bits64(f4.cpu().numpy()[idx]), bits64(fo)) and np.array_equal(t4.cpu().numpy()[idx], to)
    # checksum of checksums is launch-geometry independent
    assert f4.sum().item() == f1.sum().item()


# ----------------------------------------------------------------------------------------------
# benchmark rules (FOIC / GLFT) through the device step core vs the imported reference
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["glft", "glft_wide", "foic", "foic_1_2"])
@pytest.mark.parametrize("fee", [0.0, 0.0003])
def test_benchmark_policies_closed_loop_vs_reference(sg, name, fee):
    import os
    from conftest import GOLDEN
    from sgmm_b200.benchmarks import FOICPolicy, GLFTPolicy
    ref = np.load(os.path.join(GOLDEN, "ref_benchmarks.npz"))
    bundle = tuple(ref[f"bundle.{k}"] for k in ("s1", "s2", "mid_next", "best_ask", "best_bid", "buy_max", "sell_min"))
    pol = {"glft": GLFTPolicy(gamma=0.0001, kappa=3000, A=0.1, sigma=0.0005),
           "glft_wide": GLFTPolicy(gamma=0.01, kappa=1500, A=0.1, sigma=0.02),
           "foic": FOICPolicy(0, 0), "foic_1_2": FOICPolicy(1, 2)}[name]
    z = np.zeros(len(bundle[0]), np.float32)
    bun = sg.Bundle(z, z, *bundle[2:], 0.001)
    fit, trades, tr = sg.rollout_table(bun, pol.table(bundle, 0.001), phi=1e-4, fee_rate=fee)
    key = f"{name}.fee{fee}"
    for k in ("off_a", "off_b", "fill_buy", "fill_sell", "inventory"):
        assert np.array_equal(tr[k], ref[f"{key}.{k}"]), k
    for k in ("cash", "reward", "pnl_reward", "fee_paid"):
        assert np.array_equal(bits64(tr[k]), bits64(ref[f"{key}.{k}"])), k
    assert trades == int(((ref[f"{key}.fill_buy"] == 1) | (ref[f"{key}.fill_sell"] == 1)).sum())


def test_ga_generation_cuda_graph_replay_matches_eager(sg):
    from sgmm_b200 import synthetic
    from sgmm_b200.engine import DeviceGA
    tb = synthetic.synthetic_bundle(1, first_day=110)
    vb = synthetic.synthetic_bundle(1, first_day=111)
    stats = synthetic.train_stats_of(tb)
    train = sg.Bundle.from_arrays(tb, stats, 0.001)
    val = sg.Bundle.from_arrays(vb, stats, 0.001)
    master, _ = synthetic.policy_like_genomes(1, seed=41)
    kw = dict(pop_size=37, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=False, seed=5, max_generations=8, patience=2)
    eager = DeviceGA(master, None, **kw)
    for _ in range(6):
        eager.generation(train, val)
    graphed = DeviceGA(master, None, **kw)
    graphed.generation(train, val)                     # generation 0 eagerly (configures the kernels)
    torch.cuda.synchronize()
    g = graphed.capture(train, val)                    # capture advances nothing (capture does not execute)
    for _ in range(5):
        g.replay()
    torch.cuda.synchronize()
    he, hg = eager.history(6), graphed.history(6)
    for k in he:
        assert np.array_equal(he[k].view(np.uint8), hg[k].view(np.uint8)), k
    assert np.array_equal(eager.masters()[0], graphed.masters()[0])
