"""GPU (-m gpu): the adversary on the H = 256 tensor-core path (SGMM_PRECISION_BF16, csrc/sgmm_spec256.cu).

With an adversary, spec256_kernel writes q = raw*5 of every (bar, inventory) and walk_account_kernel<Walk20> (the 20-state
walk of the exact paths) runs the episode over that table.  Parity is stated as for the plain H = 256 path
(tests/test_gpu_spec256.py): policy outputs within TAU ticks of the fp32 oracle, and GIVEN the market maker's offsets the
kernel took, the adversary's displacements, fills, rewards and fitness are the oracle's bit for bit.
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_rounding_edges import TENSOR_EPISODES, _bundle, _tensor_checks, adversaries, genomes_of, make_episode

pytestmark = pytest.mark.gpu

H = 256
F32 = np.float32
TAU = 0.05                     # ticks on raw*5 (tests/test_gpu_spec256.py)
TICK = 0.001
PHI = 1e-4
ADV_SEED_FLIP = 0x8000000000000000
BATCH_ENV = "SGMM_EXACT256_BATCH_BYTES"


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


def bits32(a):
    return np.asarray(a, np.float32).view(np.uint32)


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


def _synthetic(sg, orc, days, first_day, T=None):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(days, first_day=first_day)
    if T is not None:
        bundle = tuple(a[:T] for a in bundle)
    stats = synthetic.train_stats_of(synthetic.synthetic_bundle(days, first_day=first_day))
    z1, z2 = orc.normalise(bundle, stats)
    return sg.Bundle.from_arrays(bundle, stats, TICK), (z1, z2) + tuple(bundle[2:]), stats


def _genomes(P, seed, out_scale=4.0):
    from sgmm_b200 import synthetic
    _, g = synthetic.policy_like_genomes(P, hidden=H, seed=seed, out_scale=out_scale, out_bias=(0.1, 0.1))
    return g


def _adv(P, seed):
    return (np.random.default_rng(seed).standard_normal((P, 1250)) * 0.6).astype(F32)


def _np(*xs):
    return [x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x) for x in xs]


def _replay(orc, bz, fee, A, fit, trd, act, raw=None):
    """Teacher-forced: the oracle's env with the adversary, on the market maker's offsets the kernel took, gives the
    kernel's fitness and trades bit for bit; the offsets are the policy's at the oracle's pre-step inventory."""
    displaced = 0
    for i in range(fit.shape[0]):
        fo, to, tro = orc.rollout(None, A[i], bz, PHI, TICK, fee, forced_actions=act[i], trace=True)
        assert bits64(fo) == bits64(fit[i]) and to == trd[i], (i, fo, fit[i], to, trd[i])
        displaced += int((tro["adv_a"] != 0).sum() + (tro["adv_b"] != 0).sum())
        if raw is not None:
            T = act.shape[1]
            inv_before = np.concatenate([[0], tro["inventory"][:-1]])
            taken = np.rint(raw[i, np.arange(T), inv_before + 2] * F32(5)).astype(np.int32)
            assert np.array_equal(taken, act[i]), i
    return displaced


def test_policy_outputs_are_the_plain_kernels_and_within_tolerance(sg, orc):
    bun, bz, _ = _synthetic(sg, orc, 1, 90)
    G, A = _genomes(4, seed=11), _adv(4, seed=11)
    _, _, raw, _ = _np(*sg.rollout_tc_audit(bun, G, A, phi=PHI, hidden=H))
    _, _, raw0, _ = _np(*sg.rollout_spec256_audit(bun, G, phi=PHI))
    assert np.array_equal(bits32(raw), bits32(raw0))
    worst, flips = 0.0, 0
    for i in range(G.shape[0]):
        for t in range(bun.T):
            for iv in range(5):
                q_o = orc.mlp_forward(G[i], [bz[0][t], bz[1][t], (iv - 2) / 2.0], hidden=H) * F32(5)
                q_k = raw[i, t, iv] * F32(5)
                worst = max(worst, float(np.max(np.abs(q_o - q_k))))
                margin = np.abs(np.abs(q_o - np.floor(q_o)) - 0.5)
                flips += int(np.sum((np.rint(q_o) != np.rint(q_k)) & (margin > TAU)))
    print(f"max |d(raw*5)| = {worst:.4g} ticks (tolerance {TAU})")
    assert worst <= TAU and flips == 0


@pytest.mark.parametrize("fee", [0.0, 3e-4, -1e-4])
def test_teacher_forced_env_bit_exact(sg, orc, fee):
    bun, bz, _ = _synthetic(sg, orc, 2, 91)
    G, A = _genomes(6, seed=12), _adv(6, seed=12)
    fit, trd, raw, act = _np(*sg.rollout_tc_audit(bun, G, A, phi=PHI, fee_rate=fee, hidden=H))
    assert _replay(orc, bz, fee, A, fit, trd, act, raw) > 0               # some quotes were displaced
    f0, _, _, _ = _np(*sg.rollout_spec256_audit(bun, G, phi=PHI, fee_rate=fee))
    assert not np.array_equal(bits64(fit), bits64(f0))                     # the adversary changes the episodes
    assert trd.max() > 0


def test_every_entry_agrees(sg, orc):
    import torch
    bun, bz, _ = _synthetic(sg, orc, 1, 92)
    G, A = _genomes(6, seed=13), _adv(6, seed=13)
    fa, ta, _, _ = _np(*sg.rollout_tc_audit(bun, G, A, phi=PHI, fee_rate=3e-4, hidden=H))
    fd, td = _np(*sg.rollout_population(bun, torch.from_numpy(G).cuda(), torch.from_numpy(A).cuda(), phi=PHI, fee_rate=3e-4,
                                        hidden=H))
    fh, th = sg.rollout_population(bun, G, A, phi=PHI, fee_rate=3e-4, hidden=H)
    pend = [sg.rollout_population_async(bun, torch.from_numpy(G[i:i + 3]).pin_memory(), torch.from_numpy(A[i:i + 3]).pin_memory(),
                                        phi=PHI, fee_rate=3e-4, hidden=H) for i in (0, 3)]
    fy, ty = (np.concatenate(x) for x in zip(*[p.result() for p in pend]))
    f74, t74 = _np(*sg.rollout_population(bun, torch.from_numpy(G).cuda(), torch.from_numpy(A[:, :74].copy()).cuda(),
                                          phi=PHI, fee_rate=3e-4, hidden=H))    # native 74-float AdversaryPolicy genomes
    for f, t in ((fd, td), (fh, th), (fy, ty), (f74, t74)):
        assert np.array_equal(bits64(f), bits64(fa)) and np.array_equal(t, ta)


def test_seeded_children_and_adversaries_equal_explicit(sg, orc):
    import torch
    bun, bz, _ = _synthetic(sg, orc, 1, 93)
    master, adv_master = _genomes(1, seed=14)[0], _adv(1, seed=14)[0]
    seed, gen, first, n = 77, 4, 10, 6
    kids = np.stack([orc.mutate(master, 0.05, seed, gen, first + i) for i in range(n)])
    akids = np.stack([orc.mutate(adv_master, 0.1, seed ^ ADV_SEED_FLIP, gen, first + i) for i in range(n)])
    fs, ts = _np(*sg.rollout_seeded(bun, torch.from_numpy(master).cuda(), count=n, sigma=0.05, seed=seed, generation=gen,
                                    first_index=first, adv_master=torch.from_numpy(adv_master).cuda(), adv_sigma=0.1, phi=PHI,
                                    hidden=H))
    fe, te, _, act = _np(*sg.rollout_tc_audit(bun, kids, akids, phi=PHI, hidden=H))
    assert np.array_equal(bits64(fs), bits64(fe)) and np.array_equal(ts, te)
    _replay(orc, bz, 0.0, akids, fe, te, act)


@pytest.mark.parametrize("T", [0, 1, 24, 25, 26, 51, 130])
def test_ragged_lengths_and_many_individuals(sg, orc, T):
    import torch
    P = 150 if T <= 26 else 5                   # more individuals than SMs: the persistent loop of spec256_kernel
    bun, bz, _ = _synthetic(sg, orc, 1, 94, T=T)
    assert bun.T == T
    G, A = _genomes(P, seed=T), _adv(P, seed=T)
    fit, trd, raw, act = sg.rollout_tc_audit(bun, G, A, phi=PHI, fee_rate=3e-4, hidden=H)
    f2, t2 = sg.rollout_population(bun, torch.from_numpy(G).cuda(), torch.from_numpy(A).cuda(), phi=PHI, fee_rate=3e-4,
                                   hidden=H)
    assert torch.equal(f2, fit) and torch.equal(t2, trd)
    fit, trd, raw, act = _np(fit, trd, raw, act)
    if T == 0:
        assert (fit == -50.0).all() and (trd == 0).all()
        return
    sel = np.arange(0, P, max(1, P // 7))
    _replay(orc, bz, 3e-4, A[sel], fit[sel], trd[sel], act[sel], raw[sel])


def test_empty_population(sg, orc):
    import torch
    bun, _, _ = _synthetic(sg, orc, 1, 95, T=40)
    f, t = sg.rollout_population(bun, torch.zeros(0, 67330, device="cuda"), torch.zeros(0, 1250, device="cuda"), phi=PHI,
                                 hidden=H)
    assert f.numel() == 0 and t.numel() == 0
    f, t, raw, act = sg.rollout_tc_audit(bun, np.zeros((0, 67330), F32), np.zeros((0, 1250), F32), phi=PHI, hidden=H)
    assert f.numel() == 0 and raw.numel() == 0 and act.numel() == 0


def test_forced_batches_equal_one(sg, orc, monkeypatch):
    import torch
    bun, bz, _ = _synthetic(sg, orc, 1, 96, T=200)
    P = 7
    G, A = _genomes(P, seed=15), _adv(P, seed=15)
    g, a = torch.from_numpy(G).cuda(), torch.from_numpy(A).cuda()
    master = torch.from_numpy(G[0]).cuda()

    def run():
        return (sg.rollout_population(bun, g, a, phi=PHI, hidden=H),
                sg.rollout_seeded(bun, master, count=P, sigma=0.05, seed=3, generation=1, phi=PHI, hidden=H, adv_master=a[0],
                                  adv_sigma=0.1),
                sg.rollout_tc_audit(bun, G, A, phi=PHI, hidden=H))

    whole = run()
    for budget in (200 * 40 * 3 + 1, 1):        # three individuals per batch (3 + 3 + 1), then one
        monkeypatch.setenv(BATCH_ENV, str(budget))
        parts = run()
        for x, y in zip(whole, parts):
            for u, v in zip(x, y):
                assert torch.equal(u, v), budget
    fit, trd, _, act = _np(*whole[2])
    _replay(orc, bz, 0.0, A, fit, trd, act)


@pytest.mark.parametrize("name", TENSOR_EPISODES)
def test_rounding_edges_with_boundary_adversaries(sg, orc, name):
    """Transparent policies on rounding ties and dyadic values, boundary adversaries exactly on and one float beyond the tanh
    threshold: teacher-forced bit-exact everywhere, and on the dyadic episodes the whole closed loop equals the oracle."""
    import torch
    ep = make_episode(name)
    G, A = genomes_of(H, ep["scale"]), adversaries()
    bun = _bundle(sg, ep)
    fit, trd, raw, act = sg.rollout_tc_audit(bun, G, A, phi=PHI, hidden=H)
    f2, t2 = sg.rollout_population(bun, torch.from_numpy(G).cuda(), torch.from_numpy(A).cuda(), phi=PHI, hidden=H)
    assert torch.equal(f2, fit) and torch.equal(t2, trd)
    _tensor_checks(orc, ep, name, G, A, 0.0, *_np(fit, trd, raw, act), hidden=H, tau=TAU)


@pytest.mark.parametrize("out_scale,fee", [(300.0, 0.0), (4e4, 3e-4)])
def test_large_offsets(sg, orc, out_scale, fee):
    bun, bz, _ = _synthetic(sg, orc, 1, 97, T=240)
    G, A = _genomes(9, seed=3, out_scale=out_scale), _adv(9, seed=3)
    fit, trd, raw, act = _np(*sg.rollout_tc_audit(bun, G, A, phi=PHI, fee_rate=fee, hidden=H))
    assert np.abs(act).max() > 50 * out_scale / 300.0
    assert _replay(orc, bz, fee, A, fit, trd, act, raw) > 0


@pytest.mark.parametrize("fee", [0.0, 3e-4])
def test_offsets_beyond_k_clamp(sg, orc, fee):
    """Policy outputs of up to 3.2e9 ticks: the offsets are clamped to +-2^30 before the displacement.  (Policy-like genomes
    cannot get there on this path: output weights beyond the f16 range make the outputs NaN, which is out of contract.)
    Transparent policies on the dyadic_large episode with z x 3 (every value still exact in f16) reach them exactly."""
    from test_gpu_rounding_edges import DYADIC_LARGE_SCALE, bz_of
    ep = make_episode("dyadic_large")
    ep["z1"], ep["z2"] = ep["z1"] * F32(3), ep["z2"] * F32(3)
    bz, bun = bz_of(ep), _bundle(sg, ep)
    G, A = genomes_of(H, DYADIC_LARGE_SCALE), _adv(4, seed=6)
    fit, trd, raw, act = _np(*sg.rollout_tc_audit(bun, G, A, phi=PHI, fee_rate=fee, hidden=H))
    q = np.abs(raw * F32(5))
    assert (q > (1 << 30)).any() and (q < (1 << 30)).any()
    assert np.abs(act).max() == 1 << 30
    assert _replay(orc, bz, fee, A, fit, trd, act) > 0


def _composed_ga(sg, orc, train, val, master, adv_master, *, pop, sigma, seed, gens, patience):
    """The GA of Env/drl_engine.py:92-171 from rollout_seeded calls on the same routes: train argmax -> market maker,
    argmin -> adversary (orc.mutate), validation of the new master through the plain H = 256 rollout."""
    import torch
    s_mm = s_adv = F32(sigma)
    best_val, stale, best_master = -np.inf, 0, master.copy()
    hist = {k: [] for k in ("train_f", "val_f", "train_trades", "val_trades", "sigma")}
    for gen in range(gens):
        fit, trd = _np(*sg.rollout_seeded(train, torch.from_numpy(master).cuda(), count=pop, sigma=float(s_mm), seed=seed,
                                          generation=gen, adv_master=torch.from_numpy(adv_master).cuda(),
                                          adv_sigma=float(s_adv), phi=PHI, hidden=H))
        best = int(np.argmax(fit))
        master = orc.mutate(master, float(s_mm), seed, gen, best)
        adv_master = orc.mutate(adv_master, float(s_adv), seed ^ ADV_SEED_FLIP, gen, int(np.argmax(-fit)))
        vf, vt = _np(*sg.rollout_population(val, torch.from_numpy(master[None]).cuda(), phi=PHI, hidden=H))
        hist["train_f"].append(fit[best]); hist["train_trades"].append(trd[best])
        hist["val_f"].append(vf[0]); hist["val_trades"].append(vt[0]); hist["sigma"].append(s_mm)
        if vf[0] > best_val:
            best_val, stale, best_master = vf[0], 0, master.copy()
        else:
            stale += 1
        if stale >= patience:
            s_mm, s_adv, stale = F32(s_mm * F32(0.5)), F32(s_adv * F32(0.5)), 0
    return hist, master, adv_master, best_master, best_val


def _ga_bundles(sg, orc):
    from sgmm_b200 import synthetic
    train, _, stats = _synthetic(sg, orc, 1, 50, T=180)
    vb = tuple(a[:150] for a in synthetic.synthetic_bundle(1, first_day=52))
    return train, sg.Bundle.from_arrays(vb, stats, TICK)


def test_device_ga_equals_composed_ga(sg, orc):
    from sgmm_b200.engine import DeviceGA
    train, val = _ga_bundles(sg, orc)
    master, adv_master = _genomes(1, seed=21, out_scale=1.0)[0], (np.random.default_rng(4).standard_normal(1250) * 0.5).astype(F32)
    gens, pop, patience = 6, 10, 2
    ga = DeviceGA(master, adv_master, pop_size=pop, sigma=0.05, phi=PHI, fee_rate=0.0, use_arl=True, seed=77,
                  max_generations=gens, patience=patience, hidden=H, precision="bf16")
    for _ in range(gens):
        ga.generation(train, val)
    h, st, (mm, adv, best) = ga.history(gens), ga.status(), ga.masters()
    ga.close()
    ho, m_o, a_o, b_o, bv_o = _composed_ga(sg, orc, train, val, master, adv_master, pop=pop, sigma=0.05, seed=77, gens=gens,
                                           patience=patience)
    assert np.array_equal(bits64(h["train_f"]), bits64(ho["train_f"]))
    assert np.array_equal(bits64(h["val_f"]), bits64(ho["val_f"]))
    assert h["train_trades"].tolist() == ho["train_trades"] and h["val_trades"].tolist() == ho["val_trades"]
    assert np.array_equal(h["sigma"], np.array(ho["sigma"], F32))
    assert np.array_equal(bits32(mm), bits32(m_o)) and np.array_equal(bits32(best), bits32(b_o))
    assert np.array_equal(bits32(adv), bits32(a_o))
    assert st["generation"] == gens and st["best_val"] == bv_o


def test_device_ga_graph_replay_equals_eager(sg, orc):
    import torch
    from sgmm_b200.engine import DeviceGA
    train, val = _ga_bundles(sg, orc)
    master, adv_master = _genomes(1, seed=22, out_scale=1.0)[0], _adv(1, seed=22)[0]
    kw = dict(pop_size=12, sigma=0.05, phi=PHI, fee_rate=3e-4, use_arl=True, seed=5, max_generations=8, patience=2, hidden=H)
    eager = DeviceGA(master, adv_master, **kw)
    for _ in range(5):
        eager.generation(train, val)
    graphed = DeviceGA(master, adv_master, **kw)
    graphed.generation(train, val)                  # generation 0 eagerly: configures the kernels, sizes the code buffers
    torch.cuda.synchronize()
    g = graphed.capture(train, val)
    for _ in range(4):
        g.replay()
    torch.cuda.synchronize()
    he, hg = eager.history(5), graphed.history(5)
    for k in he:
        assert np.array_equal(he[k].view(np.uint8), hg[k].view(np.uint8)), k
    for x, y in zip(eager.masters(), graphed.masters()):
        assert np.array_equal(bits32(x), bits32(y))
    eager.close(); graphed.close()


def test_drl_engine_h256_with_arl(sg, orc, tmp_path):
    import os
    import torch
    from sgmm_b200 import synthetic
    tb = tuple(a[:200] for a in synthetic.synthetic_bundle(1, first_day=60))
    vb = tuple(a[:160] for a in synthetic.synthetic_bundle(1, first_day=61))
    stats = synthetic.train_stats_of(tb)
    eng = sg.DRLEngine(pop_size=8, phi=PHI, tick_size=TICK, use_arl=True, save_dir=str(tmp_path), seed=5, hidden_dim=H)
    policy, hist = eng.train(tb, vb, stats, generations=4, output_prefix="s256", verbose=False)
    assert set(hist) == {"gen", "train_f", "val_f", "train_trades", "val_trades"}       # Env/drl_engine.py:86-89
    assert len(hist["val_f"]) == 4
    w = policy.get_weights().detach().cpu().numpy()
    assert w.size == H * H + 7 * H + 2
    fv, _ = _np(*sg.rollout_population(sg.Bundle.from_arrays(vb, stats, TICK), torch.from_numpy(w[None]).cuda(), phi=PHI,
                                       hidden=H))
    assert fv[0] == max(hist["val_f"])
    snap = sg.TradingPolicy(hidden_dim=H)
    snap.load_state_dict(torch.load(os.path.join(str(tmp_path), "s256_best_val_0.0001.pth")))
    assert np.array_equal(bits32(snap.get_weights().detach().cpu().numpy()), bits32(w))


def test_output_canaries_untouched(sg, orc):
    import torch
    bun, bz, _ = _synthetic(sg, orc, 1, 98, T=130)
    P, pad, T = 5, 64, 130
    G, A = _genomes(P, seed=2), _adv(P, seed=2)
    L = sg._lib
    g, a = torch.from_numpy(G).cuda(), torch.from_numpy(A).cuda()
    fit = torch.full((P + 2 * pad,), 12345.5, dtype=torch.float64, device="cuda")
    trd = torch.full((P + 2 * pad,), -777, dtype=torch.int32, device="cuda")
    raw = torch.full((P * T * 10 + 2 * pad,), -3.0, dtype=torch.float32, device="cuda")
    act = torch.full((P * T * 2 + 2 * pad,), -3, dtype=torch.int32, device="cuda")
    mm = L.Population(H, 0, P, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    ap = L.Population(32, 0, P, a.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    prm = L.RolloutParams(PHI, 0.0, 1, 0, 0, 0)
    L.check(L.lib().sgmm_rollout_tc_audit(bun.handle, C.byref(mm), C.byref(ap), C.byref(prm), fit[pad:].data_ptr(),
                                          trd[pad:].data_ptr(), raw[pad:].data_ptr(), act[pad:].data_ptr(), None))
    torch.cuda.synchronize()
    for buf, n, fill in ((fit, P, 12345.5), (trd, P, -777), (raw, P * T * 10, -3.0), (act, P * T * 2, -3)):
        b = buf.cpu().numpy()
        assert (b[:pad] == fill).all() and (b[pad + n:] == fill).all()
    f, t, ac = _np(fit[pad:pad + P], trd[pad:pad + P], act[pad:pad + P * T * 2].reshape(P, T, 2))
    _replay(orc, bz, 0.0, A, f, t, ac)
    fit.fill_(12345.5)
    L.check(L.lib().sgmm_rollout_population(bun.handle, C.byref(mm), C.byref(ap), C.byref(prm), fit[pad:].data_ptr(),
                                            trd[pad:].data_ptr(), None))
    torch.cuda.synchronize()
    fb = fit.cpu().numpy()
    assert (fb[:pad] == 12345.5).all() and (fb[pad + P:] == 12345.5).all()
    assert np.array_equal(bits64(fb[pad:pad + P]), bits64(f))


def test_refusals(sg, orc):
    import torch
    from sgmm_b200.engine import DeviceGA
    bun, _, _ = _synthetic(sg, orc, 1, 99, T=40)
    L = sg._lib
    g = torch.from_numpy(_genomes(2, seed=1)).cuda()
    a = torch.from_numpy(_adv(3, seed=1)).cuda()
    out_f = torch.empty(3, dtype=torch.float64, device="cuda")
    out_t = torch.empty(3, dtype=torch.int32, device="cuda")
    mm = L.Population(H, 0, 2, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    ap = L.Population(32, 0, 2, a.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    for precision in (0, 2, 3):                       # F32, TF32, F16 at H = 256 with an adversary
        prm = L.RolloutParams(PHI, 0.0, precision, 0, 0, 0)
        rc = L.lib().sgmm_rollout_population(bun.handle, C.byref(mm), C.byref(ap), C.byref(prm), out_f.data_ptr(),
                                             out_t.data_ptr(), None)
        assert rc == L.ERR_UNSUPPORTED, precision
    a3 = L.Population(32, 0, 3, a.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    rc = L.lib().sgmm_rollout_population(bun.handle, C.byref(mm), C.byref(a3), C.byref(L.RolloutParams(PHI, 0.0, 1, 0, 0, 0)),
                                         out_f.data_ptr(), out_t.data_ptr(), None)
    assert rc == L.ERR_INVALID
    for precision in ("tf32", "f16"):
        with pytest.raises(L.SgmmError):
            DeviceGA(_genomes(1, seed=1)[0], _adv(1, seed=1)[0], pop_size=4, sigma=0.05, phi=PHI, fee_rate=0.0, use_arl=True,
                     seed=1, max_generations=2, hidden=H, precision=precision)
