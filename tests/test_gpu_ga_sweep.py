"""A sweep of K independent GA runs in the same launches (sgmm_ga_create_sweep, DeviceGASweep, DRLEngine.train_sweep).

Every run of a sweep must be bit-identical to the solo DeviceGA of its seed, phi, fee, sigma and patience, whatever its
position in the sweep, the number of runs, the batching of the policy table and the bundle lengths."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sg():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import sgmm_b200
    return sgmm_b200


@pytest.fixture(scope="module")
def data(sg):
    from sgmm_b200 import synthetic
    tb = synthetic.synthetic_bundle(2, first_day=70)
    vb = synthetic.synthetic_bundle(1, first_day=72)
    stats = synthetic.train_stats_of(tb)
    return tb, vb, stats, sg.Bundle.from_arrays(tb, stats, 0.001), sg.Bundle.from_arrays(vb, stats, 0.001)


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


def bits32(a):
    return np.asarray(a, np.float32).view(np.uint32)


# five runs: distinct seeds, phi in {0, 1e-4, 0.01}, fee in {0, 3e-4, -1e-4}, different sigmas, patience in {1, 2, 3}
RUNS5 = [dict(seed=11, phi=0.0, fee_rate=0.0, sigma=0.05, patience=1),
         dict(seed=12, phi=1e-4, fee_rate=3e-4, sigma=0.02, patience=2),
         dict(seed=13, phi=0.01, fee_rate=-1e-4, sigma=0.08, patience=3),
         dict(seed=2 ** 63 + 5, phi=1e-4, fee_rate=0.0, sigma=0.05, patience=2),
         dict(seed=15, phi=0.01, fee_rate=3e-4, sigma=0.03, patience=1)]


def masters_of(K, seed=0, use_arl=False):
    from sgmm_b200 import synthetic
    mm = np.stack([synthetic.policy_like_genomes(1, seed=seed + 31 * r, out_scale=1.0)[0] for r in range(K)])
    adv = None
    if use_arl:
        adv = (np.random.default_rng(seed + 4).standard_normal((K, 1250)) * 0.5).astype(np.float32)
    return mm, adv


def read_run(ga, run, gens, solo=False):
    if solo:
        return ga.history(gens), ga.status(), ga.masters()
    return ga.history(run, gens), ga.status(run), ga.masters(run)


def assert_same(a, b, what=""):
    ha, sa, ma = a
    hb, sb, mb = b
    for k in ha:
        assert np.array_equal(ha[k].view(np.uint8), hb[k].view(np.uint8)), (what, k)
    assert sa == sb, (what, sa, sb)
    for x, y, name in zip(ma, mb, ("mm", "adv", "best")):
        assert np.array_equal(bits32(x), bits32(y)), (what, name)


def run_sweep(sg, train, val, runs, mm, adv, *, pop, use_arl, gens):
    ga = sg.DeviceGASweep(mm, adv, runs=runs, pop_size=pop, use_arl=use_arl, max_generations=gens)
    for _ in range(gens):
        ga.generation(train, val)
    out = [read_run(ga, r, gens) for r in range(len(runs))]
    ga.close()
    return out


def run_solo(sg, train, val, run, mm, adv, *, pop, use_arl, gens):
    ga = sg.DeviceGA(mm, adv, pop_size=pop, use_arl=use_arl, max_generations=gens, precision="exact", **run)
    for _ in range(gens):
        ga.generation(train, val)
    out = read_run(ga, 0, gens, solo=True)
    ga.close()
    return out


@pytest.mark.parametrize("use_arl", [False, True])
@pytest.mark.parametrize("pop", [1, 24, 50])
def test_every_run_equals_its_solo_ga(sg, data, pop, use_arl):
    _, _, _, train, val = data
    gens = 10
    mm, adv = masters_of(len(RUNS5), seed=pop, use_arl=use_arl)
    sweep = run_sweep(sg, train, val, RUNS5, mm, adv, pop=pop, use_arl=use_arl, gens=gens)
    decayed = 0
    for r, run in enumerate(RUNS5):
        solo = run_solo(sg, train, val, run, mm[r], None if adv is None else adv[r], pop=pop, use_arl=use_arl, gens=gens)
        assert_same(sweep[r], solo, f"run {r}")
        decayed += int(sweep[r][1]["sigma"] != np.float32(run["sigma"]))
    assert decayed >= 1                                   # some runs' sigmas decayed
    assert sweep[0][0]["sigma"][0] == np.float32(RUNS5[0]["sigma"])


def test_sweep_run_matches_oracle_ga(sg, data):
    from oracle import oracle as orc
    from test_gpu_parity import _oracle_ga
    tb, vb, stats, train, val = data
    tz = orc.normalise(tb, stats) + tb[2:]
    vz = orc.normalise(vb, stats) + vb[2:]
    runs = [RUNS5[0], dict(seed=77, phi=1e-4, fee_rate=3e-4, sigma=0.05, patience=3)]
    mm, adv = masters_of(2, seed=5, use_arl=True)
    gens, pop = 9, 24
    (h, st, (m, a, b)) = run_sweep(sg, train, val, runs, mm, adv, pop=pop, use_arl=True, gens=gens)[1]
    ho, m_o, a_o, b_o, bv_o, s_o = _oracle_ga(orc, tz, vz, mm[1], adv[1], pop=pop, sigma=0.05, phi=1e-4, tick=0.001,
                                               fee=3e-4, use_arl=True, seed=77, gens=gens, patience=3)
    assert np.array_equal(bits64(h["train_f"]), bits64(ho["train_f"]))
    assert np.array_equal(bits64(h["val_f"]), bits64(ho["val_f"]))
    assert h["train_trades"].tolist() == ho["train_trades"] and h["val_trades"].tolist() == ho["val_trades"]
    assert np.array_equal(h["sigma"], np.array(ho["sigma"], np.float32))
    assert np.array_equal(bits32(m), bits32(m_o)) and np.array_equal(bits32(b), bits32(b_o))
    assert np.array_equal(bits32(a), bits32(a_o))
    assert st["best_val"] == bv_o and st["sigma"] == s_o


@pytest.mark.parametrize("use_arl", [False, True])
def test_position_independence(sg, data, use_arl):
    _, _, _, train, val = data
    gens, pop = 8, 24
    runs = [dict(seed=100 + r, phi=(1e-4, 0.01, 0.0)[r % 3], fee_rate=(0.0, 3e-4, -1e-4)[r % 3], sigma=0.05, patience=2)
            for r in range(9)]
    mm, adv = masters_of(9, seed=3, use_arl=use_arl)
    nine = run_sweep(sg, train, val, runs, mm, adv, pop=pop, use_arl=use_arl, gens=gens)
    alone = run_sweep(sg, train, val, runs[8:], mm[8:], None if adv is None else adv[8:], pop=pop, use_arl=use_arl, gens=gens)
    assert_same(nine[8], alone[0], "last of 9 vs alone")
    twins = run_sweep(sg, train, val, [runs[4], runs[4]], np.stack([mm[4], mm[4]]),
                      None if adv is None else np.stack([adv[4], adv[4]]), pop=pop, use_arl=use_arl, gens=gens)
    assert_same(twins[0], twins[1], "twins")
    assert_same(twins[0], nine[4], "twin vs run 4 of 9")


@pytest.mark.parametrize("use_arl,K,pop", [(False, 9, 50), (True, 4, 50)])
def test_large_sweeps_and_batches_inside_runs(sg, data, monkeypatch, use_arl, K, pop):
    """K*lambda above SMALL_POP_MAX (400) without the adversary and above 148 with it; then a batch budget that cuts
    the table every 7 individuals, so that batch boundaries fall inside runs."""
    _, _, _, train, val = data
    gens = 6
    runs = [dict(seed=200 + r, phi=(1e-4, 0.01)[r % 2], fee_rate=(0.0, 3e-4, -1e-4)[r % 3], sigma=0.04, patience=2)
            for r in range(K)]
    mm, adv = masters_of(K, seed=9, use_arl=use_arl)
    assert K * pop > (400 if not use_arl else 148)
    whole = run_sweep(sg, train, val, runs, mm, adv, pop=pop, use_arl=use_arl, gens=gens)
    monkeypatch.setenv("SGMM_EXACT256_BATCH_BYTES", str(7 * train.T * 48))
    batched = run_sweep(sg, train, val, runs, mm, adv, pop=pop, use_arl=use_arl, gens=gens)
    monkeypatch.delenv("SGMM_EXACT256_BATCH_BYTES")
    for r in range(K):
        assert_same(whole[r], batched[r], f"batched run {r}")
    for r in (0, K - 1):                                  # and equal to the solo GAs
        solo = run_solo(sg, train, val, runs[r], mm[r], None if adv is None else adv[r], pop=pop, use_arl=use_arl, gens=gens)
        assert_same(whole[r], solo, f"solo run {r}")


@pytest.mark.parametrize("T", [1, 2641])
def test_bundle_shapes(sg, T):
    from sgmm_b200 import synthetic
    full = synthetic.synthetic_bundle(12, first_day=80)
    tb = tuple(np.ascontiguousarray(x[:T]) for x in full)
    vb = synthetic.synthetic_bundle(2, first_day=95)
    vb = tuple(np.ascontiguousarray(x[:333]) for x in vb)
    stats = synthetic.train_stats_of(full)
    train, val = sg.Bundle.from_arrays(tb, stats, 0.001), sg.Bundle.from_arrays(vb, stats, 0.001)
    assert train.T == T and val.T == 333
    runs = RUNS5[:3]
    for use_arl in (False, True):
        mm, adv = masters_of(3, seed=T, use_arl=use_arl)
        sweep = run_sweep(sg, train, val, runs, mm, adv, pop=24, use_arl=use_arl, gens=5)
        for r in range(3):
            solo = run_solo(sg, train, val, runs[r], mm[r], None if adv is None else adv[r], pop=24, use_arl=use_arl, gens=5)
            assert_same(sweep[r], solo, f"T={T} arl={use_arl} run {r}")


def test_graph_replay_and_phases(sg, data):
    _, _, _, train, val = data
    mm, adv = masters_of(4, seed=17, use_arl=True)
    runs = RUNS5[:4]
    kw = dict(runs=runs, pop_size=30, use_arl=True, max_generations=8)
    eager = sg.DeviceGASweep(mm, adv, **kw)
    for _ in range(7):
        eager.generation(train, val)
    graphed = sg.DeviceGASweep(mm, adv, **kw)
    graphed.generation(train, val)                        # one eager generation allocates the table buffer
    torch.cuda.synchronize()
    g = graphed.capture(train, val)
    for _ in range(6):
        g.replay()
    torch.cuda.synchronize()
    phased = sg.DeviceGASweep(mm, adv, **kw)
    for _ in range(7):
        phased.evaluate(train)
        phased.select(val)
    for r in range(4):
        e = read_run(eager, r, 7)
        assert_same(e, read_run(graphed, r, 7), f"graph run {r}")
        assert_same(e, read_run(phased, r, 7), f"phases run {r}")
    for x in (eager, graphed, phased):
        x.close()


def test_refusals(sg, data, tmp_path):
    from sgmm_b200 import _lib
    L = _lib.lib()
    _, _, _, train, val = data
    dev = torch.cuda.current_device()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    mm, adv = masters_of(2, seed=1, use_arl=True)
    runs = (_lib.GaRun * 2)(_lib.GaRun(1, 0.0, 0.0, 0.05, 2), _lib.GaRun(2, 1e-4, 0.0, 0.05, 2))

    def create(cfg, K=2, run=runs, m=mm, a=adv):
        h = C.c_void_p()
        rc = L.sgmm_ga_create_sweep(C.byref(h), C.byref(cfg), K, run, None if m is None else m.ctypes.data,
                                    None if a is None else a.ctypes.data, dev, stream)
        if rc == 0:
            L.sgmm_ga_destroy(h)
        return rc, L.sgmm_last_error().decode()

    def cfg(hidden=32, use_arl=1, pop=8, first=0, count=8, stride=0, precision=0):
        return _lib.GaConfig(hidden, use_arl, pop, first, count, stride, 0.0, 0, 0.0, 0.0, 0, 4, precision)
    assert create(cfg())[0] == 0
    assert create(cfg(precision=4))[0] == 0                                   # EXACT
    for prec in (1, 2, 3):                                                    # BF16, TF32, F16
        rc, msg = create(cfg(precision=prec))
        assert rc == _lib.ERR_UNSUPPORTED and "exact" in msg
    rc, msg = create(cfg(hidden=256))
    assert rc == _lib.ERR_UNSUPPORTED and "hidden" in msg
    for K in (0, -1):
        rc, msg = create(cfg(), K=K)
        assert rc == _lib.ERR_INVALID and "run" in msg
    assert create(cfg(), run=None)[0] == _lib.ERR_INVALID
    assert create(cfg(), m=None)[0] == _lib.ERR_INVALID
    rc, msg = create(cfg(), a=None)
    assert rc == _lib.ERR_INVALID and "use_arl" in msg
    assert create(cfg(use_arl=0), a=None)[0] == 0
    for sharded in (cfg(count=4, stride=4), cfg(first=4, count=4, stride=4), cfg(count=4)):
        rc, msg = create(sharded)
        assert rc == _lib.ERR_INVALID and "rank" in msg
    assert L.sgmm_abi_sizeof(7) == C.sizeof(_lib.GaRun) == 32
    # run-less read-backs and the shard buffers refuse a multi-run handle; run indices are checked
    ga = sg.DeviceGASweep(mm, adv, runs=[dict(seed=1, phi=0.0), dict(seed=2, phi=0.0)], pop_size=8, use_arl=True,
                          max_generations=3)
    ga.generation(train, val)
    s = _lib.GaStatus()
    buf = np.empty(1250, np.float32)
    h64 = np.empty(3, np.float64)
    checks = [L.sgmm_ga_status_host(ga._h, C.byref(s), stream),
              L.sgmm_ga_master_host(ga._h, buf.ctypes.data, None, None, stream),
              L.sgmm_ga_history_host(ga._h, 3, h64.ctypes.data, None, None, None, None, stream),
              L.sgmm_ga_buffers(ga._h, None, None, None, None, None, None)]
    for rc in checks:
        assert rc == _lib.ERR_INVALID
    assert L.sgmm_ga_status_host(ga._h, C.byref(s), stream) == _lib.ERR_INVALID
    assert "sgmm_ga_run_status_host" in L.sgmm_last_error().decode()
    for bad in (-1, 2):
        assert L.sgmm_ga_run_status_host(ga._h, bad, C.byref(s), stream) == _lib.ERR_INVALID
        assert "out of range" in L.sgmm_last_error().decode()
        assert L.sgmm_ga_run_master_host(ga._h, bad, buf.ctypes.data, None, None, stream) == _lib.ERR_INVALID
        assert L.sgmm_ga_run_history_host(ga._h, bad, 3, h64.ctypes.data, None, None, None, None, stream) == _lib.ERR_INVALID
    assert ga.status(1)["generation"] == 1
    ga.close()
    # the run_* entries accept run 0 of a one-run GA
    solo = sg.DeviceGA(mm[0], adv[0], pop_size=8, sigma=0.05, phi=0.0, fee_rate=0.0, use_arl=True, seed=1, max_generations=3)
    solo.generation(train, val)
    assert L.sgmm_ga_run_status_host(solo._h, 0, C.byref(s), stream) == 0 and s.generation == 1
    assert L.sgmm_ga_status_host(solo._h, C.byref(s), stream) == 0
    assert L.sgmm_ga_run_status_host(solo._h, 1, C.byref(s), stream) == _lib.ERR_INVALID
    solo.close()
    # DRLEngine.train_sweep refusals
    tb, vb, stats, _, _ = data
    with pytest.raises(ValueError, match="different lengths"):
        sg.DRLEngine(pop_size=8, save_dir=str(tmp_path)).train_sweep(tb, vb, stats, 1, phis=[0.0, 1e-4], seeds=[1, 2, 3])
    with pytest.raises(ValueError, match="hidden_dim"):
        sg.DRLEngine(pop_size=8, hidden_dim=256, save_dir=str(tmp_path)).train_sweep(tb, vb, stats, 1)
    with pytest.raises(ValueError, match="exact"):
        sg.DRLEngine(pop_size=8, precision="bf16", save_dir=str(tmp_path)).train_sweep(tb, vb, stats, 1)


def test_drl_engine_train_sweep_equals_train(sg, data, tmp_path):
    tb, vb, stats, _, _ = data
    phis, fees, seeds = [1e-4, 0.01, 0.0], [0.0, 3e-4, -1e-4], [7, 8, 2 ** 62 + 9]
    gens = 8
    torch.manual_seed(3)
    eng = sg.DRLEngine(pop_size=20, phi=0.01, tick_size=0.001, use_arl=True, patience=2, save_dir=str(tmp_path / "sweep"))
    mm0 = eng.mm_evolver.master_policy.get_weights().clone()
    adv0 = eng.adv_evolver.master_policy.get_weights().clone()
    out = eng.train_sweep(tb, vb, stats, gens, phis=phis, fee_rates=fees, seeds=seeds, log_every=3, verbose=False)
    assert len(out) == 3
    assert torch.equal(eng.mm_evolver.master_policy.get_weights(), mm0)             # the engine's evolvers are untouched
    assert torch.equal(eng.adv_evolver.master_policy.get_weights(), adv0) and eng.mm_evolver.sigma == 0.05
    for r in range(3):
        solo = sg.DRLEngine(pop_size=20, phi=phis[r], fee_rate=fees[r], tick_size=0.001, use_arl=True, patience=2,
                            seed=seeds[r], save_dir=str(tmp_path / f"solo{r}"))
        solo.mm_evolver.master_policy.set_weights(mm0)
        solo.adv_evolver.master_policy.set_weights(adv0)
        policy, hist = solo.train(tb, vb, stats, generations=gens, log_every=3, verbose=False)
        sp, sh = out[r]
        assert sorted(sh) == sorted(hist) and sh["gen"] == hist["gen"]
        for k in ("train_f", "val_f"):
            assert np.array_equal(bits64(sh[k]), bits64(hist[k])), (r, k)
        assert sh["train_trades"] == hist["train_trades"] and sh["val_trades"] == hist["val_trades"]
        sa, sb = sp.state_dict(), policy.state_dict()
        assert list(sa) == list(sb)
        for k in sa:
            assert np.array_equal(bits32(sa[k].numpy()), bits32(sb[k].numpy())), (r, k)
        ck = tmp_path / "sweep" / f"agent_run{r}_best_val_{phis[r]}.pth"
        assert ck.exists()
        snap = sg.TradingPolicy(hidden_dim=32)
        snap.load_state_dict(torch.load(ck, weights_only=True))
        assert torch.equal(snap.get_weights(), sp.get_weights())                        # the best-on-validation master
        assert os.path.exists(tmp_path / f"solo{r}" / f"agent_best_val_{phis[r]}.pth")


def test_handles_collected_during_a_capture(sg, data):
    """A bundle and a sweep that only a reference cycle keeps alive, collected by the garbage collector in the middle of a
    graph capture, leave the capture valid; they are destroyed at the next release outside it."""
    import gc
    from sgmm_b200 import _lib
    _, vb, stats, train, val = data
    mm, _ = masters_of(2, seed=8)
    ga = sg.DeviceGASweep(mm, None, runs=RUNS5[:2], pop_size=8, use_arl=False, max_generations=4)
    ga.generation(train, val)
    doomed_bundle = sg.Bundle.from_arrays(vb, stats, 0.001)
    doomed_ga = sg.DeviceGASweep(mm, None, runs=RUNS5[:2], pop_size=8, use_arl=False, max_generations=4)
    doomed_bundle.cycle, doomed_ga.cycle = doomed_bundle, doomed_ga
    del doomed_bundle, doomed_ga
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        gc.collect()                                      # finalises both inside the capture
        ga.generation(train, val)
    assert len(_lib._DEFERRED) >= 2
    g.replay()
    torch.cuda.synchronize()
    _lib.release("sgmm_bundle_destroy", 0)                # no handle: only drains
    assert _lib._DEFERRED == []
    solo = sg.DeviceGASweep(mm, None, runs=RUNS5[:2], pop_size=8, use_arl=False, max_generations=4)
    for _ in range(2):
        solo.generation(train, val)
    for r in range(2):
        assert_same(read_run(ga, r, 2), read_run(solo, r, 2), f"run {r}")
    ga.close()
    solo.close()
