"""CPU: the C-ABI library loads and exports every declared symbol; the reference-named host
surface (FTPEnv, policies, NeuroEvolution, StrategyRecorder, sharding helpers) behaves like the
reference.  No compute entry point that needs a GPU is called here."""
import os
import re
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, REF_CASES, ref_case

import sgmm_b200
from sgmm_b200 import _lib
from sgmm_b200.dist import shard_bounds


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "sgmm.h")).read()
    declared = set(re.findall(r"\b(sgmm_[a-z0-9_]+)\s*\(", header))
    declared -= {"sgmm_bundle", "sgmm_ga"}
    assert declared, "no declarations parsed"
    L = _lib.lib()
    for name in sorted(declared):
        assert hasattr(L, name), f"libsgmm_b200.so does not export {name}"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert L.sgmm_version() == 101


def test_struct_layouts_match_header():
    import ctypes as C
    assert C.sizeof(_lib.Population) == 64
    assert C.sizeof(_lib.RolloutParams) == 32
    assert C.sizeof(_lib.Trace) == 20 * 8
    assert C.sizeof(_lib.EnvState) == 56 and C.sizeof(_lib.StepInfo) == 40
    assert C.sizeof(_lib.GaConfig) == 80 and C.sizeof(_lib.GaStatus) == 32
    L = _lib.lib()
    for which, struct in enumerate((_lib.Population, _lib.RolloutParams, _lib.Trace, _lib.EnvState, _lib.StepInfo,
                                    _lib.GaConfig, _lib.GaStatus)):
        assert L.sgmm_abi_sizeof(which) == C.sizeof(struct), struct.__name__
    assert L.sgmm_abi_sizeof(99) < 0


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libsgmm_b200.so")
    with pytest.raises(_lib.SgmmLibraryError):
        _lib.lib()


def test_error_reporting_invalid_arguments():
    import ctypes as C
    L = _lib.lib()
    h = C.c_void_p()
    rc = L.sgmm_bundle_create(C.byref(h), -1, None, None, None, None, None, None, None, 0.001, 0, None)
    assert rc == _lib.ERR_INVALID and b"T < 0" in L.sgmm_last_error()
    rc = L.sgmm_bundle_create(C.byref(h), 0, None, None, None, None, None, None, None, 0.0, 0, None)
    assert rc == _lib.ERR_INVALID and b"tick_size" in L.sgmm_last_error()
    with pytest.raises(_lib.SgmmError):
        _lib.check(L.sgmm_env_init(None, 0.0, 0.0, 0.0))


@pytest.mark.parametrize("name", ["drl", "arl", "glft", "foic"])
def test_ftpenv_shim_replays_golden_backtests_bit_exact(golden, name):
    """Same replay as the oracle's, through the product's FTPEnv (host build of the step core)."""
    b = golden.backtest
    env = sgmm_b200.FTPEnv(phi=1e-4, tick_size=0.001, fee_rate=0.0)
    assert env.reset() == (0, 0.0)
    for t in range(960):
        fb, fs = b[f"{name}.fill_buy"][t], b[f"{name}.fill_sell"][t]
        reward, info = env.step(np.array([b[f"{name}.off_a"][t], b[f"{name}.off_b"][t]]),
                                b[f"{name}.mid"][t], b[f"{name}.ask"][t], b[f"{name}.bid"][t],
                                np.inf if fs else -np.inf, -np.inf if fb else np.inf)
        assert (info['fill_buy'], info['fill_sell']) == (fb, fs)
        assert env.inventory == b[f"{name}.inventory"][t]
        assert env.cash == b[f"{name}.cash"][t] and reward == b[f"{name}.reward"][t]
        assert info['pnl_reward'] == b[f"{name}.pnl_reward"][t]
        assert isinstance(reward, np.float64)
        assert np.signbit(info['inventory_reward']) == np.signbit(b[f"{name}.inventory_reward"][t])


@pytest.mark.parametrize("name", ["fee", "arl_fee"])
def test_ftpenv_shim_vs_imported_reference_trace(golden, name):
    """Fill decisions against real bounds, fees and adversary displacement (unpinned by the
    parquets) against the imported reference's per-step trace."""
    cs = ref_case(golden.ref, name)
    _, _, mid, ask, bid, bmax, smin = cs["bundle"]
    for i in range(2):
        tr = {k: v[i] for k, v in cs["trace"].items()}
        env = sgmm_b200.FTPEnv(phi=cs["phi"], tick_size=cs["tick"], fee_rate=cs["fee"])
        for t in range(len(mid)):
            adv = np.array([tr["adv_a"][t], tr["adv_b"][t]], np.float32) if cs["use_arl"] else None
            r, info = env.step(np.array([tr["off_a"][t], tr["off_b"][t]]), mid[t], ask[t], bid[t], bmax[t], smin[t],
                               adv_action=adv)
            assert (info['fill_buy'], info['fill_sell']) == (tr["fill_buy"][t], tr["fill_sell"][t])
            assert env.inventory == tr["inventory"][t] and env.cash == tr["cash"][t]
            assert r == tr["reward"][t] and info['fee_paid'] == tr["fee_paid"][t]


def test_ftpenv_attributes_are_writable():
    env = sgmm_b200.FTPEnv()
    assert (env.phi, env.tick_size, env.fee_rate, env.i_max, env.i_min) == (0.01, 0.01, 0.0, 2, -2)
    env.inventory = 2
    r, info = env.step([0, 0], 1.0, 1.01, 0.99, 2.0, 0.0)      # capped long: cannot buy, sells
    assert info['fill_buy'] == 0 and info['fill_sell'] == 1 and env.inventory == 1
    env.i_max = 1
    r, info = env.step([0, 0], 1.0, 1.01, 0.99, -1.0, 0.0)
    assert info['fill_buy'] == 0
    r, info = env.step([0, 0], 1.0, 1.01, 0.99, np.nan, np.nan)
    assert info['fill_buy'] == 0 and info['fill_sell'] == 0


def test_policy_checkpoint_contract(golden, tmp_path):
    pol = sgmm_b200.TradingPolicy()
    assert list(pol.state_dict().keys()) == [f"net.{i}.{p}" for i in (0, 2, 4) for p in ("weight", "bias")]
    assert [tuple(v.shape) for v in pol.state_dict().values()] == [(32, 3), (32,), (32, 32), (32,), (2, 32), (2,)]
    g = torch.from_numpy(golden.ckpt["510300_with_adv"].copy())
    pol.set_weights(g)
    assert torch.equal(pol.get_weights(), g)
    assert torch.equal(pol.state_dict()["net.2.weight"].reshape(-1), g[128:1152])
    p = tmp_path / "a.pth"
    torch.save(pol.state_dict(), p)
    pol2 = sgmm_b200.TradingPolicy()
    pol2.load_state_dict(torch.load(p, weights_only=True))
    assert torch.equal(pol2.get_weights(), g)
    # fresh policies: orthogonal gain 0.9, bias 0.05 (models/model.py:18-21)
    fresh = sgmm_b200.TradingPolicy()
    w = fresh.net[2].weight
    assert torch.allclose(w @ w.T, 0.81 * torch.eye(32), atol=1e-5)
    assert torch.all(fresh.net[0].bias == 0.05)
    adv = sgmm_b200.AdversaryPolicy()
    assert list(adv.state_dict().keys()) == ["fc.0.weight", "fc.0.bias", "fc.2.weight", "fc.2.bias"]
    adv.set_weights(g)                                         # consumes the first 74 floats (model.py:52-57)
    assert torch.equal(adv.fc[0].weight.reshape(-1), g[:36]) and torch.equal(adv.fc[2].bias, g[72:74])
    assert sgmm_b200.genome_len(32) == 1250 and sgmm_b200.genome_len(256) == 67330


def test_policy_forward_matches_oracle_order_within_fp32_noise(golden):
    from oracle import oracle
    g = golden.ckpt["510300_with_adv"]
    pol = sgmm_b200.TradingPolicy()
    pol.set_weights(torch.from_numpy(g.copy()))
    rng = np.random.default_rng(0)
    for _ in range(50):
        x = np.array([rng.normal(), rng.normal(), rng.integers(-2, 3) / 2.0], np.float32)
        want = pol.forward(torch.from_numpy(x).reshape(1, 3)).numpy().ravel()
        got = oracle.mlp_forward(g, x)
        assert np.max(np.abs(want - got)) < 5e-6


def test_neuroevolution_ask_tell_semantics():
    ne = sgmm_b200.NeuroEvolution(population_size=7, sigma=0.05)
    assert ne.pop_size == 7 and ne.sigma == 0.05
    base = ne.master_policy.get_weights()
    pop = ne.ask()
    assert len(pop) == 7 and all(p.shape == (1250,) and p.dtype == torch.float32 for p in pop)
    d = torch.stack(pop) - base
    assert 0.04 < d.std().item() < 0.06
    best = ne.tell(pop, [0.0, 2.0, 2.0, -1.0, 1.0, 0.5, 0.1])       # first maximum, no elitism
    assert best == 2.0 and torch.equal(ne.master_policy.get_weights(), pop[1])


def test_recorder_rows_and_derived_columns(golden):
    b = golden.backtest
    rec = sgmm_b200.StrategyRecorder()
    for t in range(5):
        info = {'pnl_reward': b["drl.pnl_reward"][t], 'inventory_reward': b["drl.inventory_reward"][t],
                'fee_paid': 0.0, 'fill_buy': b["drl.fill_buy"][t], 'fill_sell': b["drl.fill_sell"][t]}
        rec.record(t, b["drl.mid"][t], b["drl.ask"][t], b["drl.bid"][t], (b["drl.off_a"][t], b["drl.off_b"][t]),
                   b["drl.reward"][t], b["drl.inventory"][t], b["drl.cash"][t], info)
    df = rec.to_dataframe()
    assert list(df.columns[:13]) == ['step', 'mid', 'ask', 'bid', 'off_a', 'off_b', 'reward', 'inventory', 'cash',
                                     'pnl_reward', 'inventory_reward', 'fee_paid', 'is_trade']
    for c in ("spread", "wealth", "cum_reward", "skew", "cum_fees", "realized_pnl", "unrealized_pnl"):
        assert np.array_equal(df[c].to_numpy(), b[f"drl.{c}"][:5]), c
    # trace-fed recorder reproduces the whole golden frame
    trace = {k: b[f"arl.{k}"] for k in ("off_a", "off_b", "reward", "inventory", "cash", "fee_paid", "pnl_reward",
                                         "inventory_reward", "fill_buy", "fill_sell")}
    bundle = (b["arl.s1_pred"], b["arl.s2_pred"], b["arl.mid"], b["arl.ask"], b["arl.bid"], None, None)
    df2 = sgmm_b200.StrategyRecorder.from_trace(trace, bundle).to_dataframe()
    for c in ("spread", "wealth", "cum_reward", "skew", "cum_fees", "realized_pnl", "unrealized_pnl"):
        assert np.array_equal(df2[c].to_numpy(), b[f"arl.{c}"]), c
    rec3 = sgmm_b200.StrategyRecorder()
    rec3.record_detailed(0, 1.0, 1.01, 0.99, (1, 2), 0.5, 0, 0.0,
                         {'pnl_reward': 0.5, 'inventory_reward': -0.0, 'fill_buy': 1, 'fill_sell': 0}, 2.0, 0.1)
    assert rec3.to_dataframe()['spread'][0] == pytest.approx(0.02)


def test_normalise_matches_reference_dtypes(golden):
    for name in REF_CASES:
        cs = ref_case(golden.ref, name)
        z1, z2 = sgmm_b200.normalise(cs["bundle"], cs["stats"])
        assert z1.dtype == np.float32
        assert np.array_equal(z1, cs["trace"]["z1"][0]) and np.array_equal(z2, cs["trace"]["z2"][0])


def test_shard_bounds_partition():
    for P in (1, 7, 50, 4096, 65536, 65537):
        for R in (1, 2, 3, 4, 8):
            seen = []
            for r in range(R):
                first, count, stride = shard_bounds(P, R, r)
                assert stride == -(-P // R) and 0 <= count <= stride
                seen += list(range(first, first + count))
            assert seen == list(range(P))
            assert R * stride <= P + 64


def test_synthetic_bundle_shape_and_determinism():
    from sgmm_b200 import synthetic
    a = synthetic.synthetic_bundle(2)
    b = synthetic.synthetic_bundle(2)
    assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(a, b))
    assert [len(x) for x in a] == [480] * 7
    assert a[0].dtype == np.float32 and a[2].dtype == np.float64
    s1, s2, mid, ask, bid, bmax, smin = a
    spread = np.round((ask - bid) / 0.001).astype(int)
    assert set(np.unique(spread)) <= {1, 2}
    assert 0.002 < np.isnan(bmax).mean() < 0.03
    touch0 = np.nanmean(bmax >= ask)
    assert 0.9 < touch0 <= 1.0


def test_benchmark_policy_tables_match_reference_actions():
    """FOIC / GLFT offset tables (host closed form) against the imported reference's benchmark run
    (tests/golden/ref_benchmarks.npz: Env/benchmarks.py driven by the loop of main.py:99-132)."""
    from conftest import GOLDEN
    from sgmm_b200.benchmarks import FOICPolicy, GLFTPolicy
    ref = np.load(os.path.join(GOLDEN, "ref_benchmarks.npz"))
    bundle = tuple(ref[f"bundle.{k}"] for k in ("s1", "s2", "mid_next", "best_ask", "best_bid", "buy_max", "sell_min"))
    pols = {"glft": GLFTPolicy(gamma=0.0001, kappa=3000, A=0.1, sigma=0.0005),
            "glft_wide": GLFTPolicy(gamma=0.01, kappa=1500, A=0.1, sigma=0.02),
            "foic": FOICPolicy(0, 0), "foic_1_2": FOICPolicy(1, 2)}
    for name, pol in pols.items():
        tab = pol.table(bundle, 0.001)
        assert tab.shape == (480, 5, 2) and tab.dtype == np.int32
        inv_prev = np.concatenate([[0], ref[f"{name}.fee0.0.inventory"][:-1]])
        t = np.arange(480)
        assert np.array_equal(tab[t, inv_prev + 2, 0], ref[f"{name}.fee0.0.off_a"])
        assert np.array_equal(tab[t, inv_prev + 2, 1], ref[f"{name}.fee0.0.off_b"])
    assert np.array_equal(FOICPolicy(1, 2).get_action(-1), [1, 2])
    a = GLFTPolicy(gamma=0.0001, kappa=3000, A=0.1, sigma=0.0005).get_action(1)
    assert a[0] > a[1] and a.dtype == np.float64            # long inventory skews the quotes down


def test_ftpenv_fractional_offsets_quote_as_given():
    """Env/market_env.py:23,30-31 uses the offsets as given, floats included: 1.7 quotes at 1.7 ticks, not at 1."""
    import sgmm_b200
    env = sgmm_b200.FTPEnv(phi=1e-4, tick_size=0.001, fee_rate=3e-4)
    ask, bid, mid = 3.481, 3.480, 3.4815
    # ask quote = 3.481 + 1.7 * 0.001 = 3.4827: fills against buy_max 3.4828, would NOT fill at int(1.7) -> 3.482 ... both fill;
    # use a bound between the two quotes to tell them apart
    my_ask = ask + 1.7 * 0.001
    r, info = env.step([1.7, 5.0], mid, ask, bid, buy_max=3.4825, sell_min=float("nan"))
    assert info["fill_sell"] == 0 and my_ask > 3.4825                # truncation to 1 tick (3.482) would have filled
    r, info = env.step([1.7, 5.0], mid, ask, bid, buy_max=3.4828, sell_min=float("nan"))
    assert info["fill_sell"] == 1
    fee = my_ask * 3e-4
    want_pnl = 0.0 + ((my_ask - mid) - fee)
    assert info["pnl_reward"] == want_pnl and env.cash == 0.0 + (my_ask - fee) and env.inventory == -1
    assert r == want_pnl - 1e-4 * 1
    # integral floats and numpy integers take the integer entry and agree with the real-valued one
    e1, e2 = sgmm_b200.FTPEnv(1e-4, 0.001, 0.0), sgmm_b200.FTPEnv(1e-4, 0.001, 0.0)
    r1, i1 = e1.step(np.array([2, -1]), mid, ask, bid, 3.49, 3.47, adv_action=np.array([0.6, -0.4]))
    r2, i2 = e2.step([2.0, -1.0], mid, ask, bid, 3.49, 3.47, adv_action=np.array([0.6, -0.4]))
    assert r1 == r2 and i1 == i2 and e1.cash == e2.cash


def test_adversary_genome_lengths_accepted():
    from sgmm_b200.engine import _as_adv_matrix
    import torch
    a74 = torch.arange(74, dtype=torch.float32)
    m = _as_adv_matrix(a74)
    assert m.shape == (1, 1250) and torch.equal(m[0, :74], a74) and float(m[0, 74:].abs().sum()) == 0.0
    assert _as_adv_matrix(torch.zeros(3, 1250)).shape == (3, 1250)
    assert _as_adv_matrix([torch.zeros(2000), torch.ones(2000)]).shape == (2, 1250)
    with pytest.raises(ValueError):
        _as_adv_matrix(torch.zeros(73))


def test_reference_staging_recipe(tmp_path):
    """stage() copies the reference's hot-path files byte for byte and the manifest detects any edit; where oracle/_ref is
    staged, it holds byte-identical copies of the reference's files."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import stage_ref
    finally:
        sys.path.pop(0)
    src, dst = tmp_path / "reference", tmp_path / "staged"
    for k, rel in enumerate(stage_ref.FILES):
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_bytes(f"# stand-in {k}\n".encode() + bytes(range(256)))
    manifest = stage_ref.stage(ref=str(src), dst=str(dst))
    assert set(manifest["files"]) == set(stage_ref.FILES) and stage_ref.staged(str(dst))
    for rel in stage_ref.FILES:
        assert (dst / rel).read_bytes() == (src / rel).read_bytes()
    (dst / stage_ref.FILES[0]).write_bytes(b"edited\n")
    assert not stage_ref.staged(str(dst))
    (dst / stage_ref.FILES[-1]).unlink()
    assert not stage_ref.staged(str(dst))
    if os.path.exists(os.path.join(stage_ref.DST, "MANIFEST.json")):
        assert stage_ref.staged()
    if os.path.isdir(stage_ref.REF) and os.path.isdir(stage_ref.DST):
        for rel in stage_ref.FILES:
            assert open(os.path.join(stage_ref.REF, rel), "rb").read() == open(os.path.join(stage_ref.DST, rel), "rb").read()
    tracked = __import__("subprocess").run(["git", "ls-files", "oracle/_ref"], cwd=ROOT, capture_output=True, text=True).stdout
    assert tracked.strip() == "", "reference sources must never be committed"
