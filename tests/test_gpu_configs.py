"""GPU (-m gpu): BASELINE.json configs[2..4] at their full sizes, the unmodified reference's outputs, and the round-2
entry points (H = 256 GA, pipelined host entry, sharding through DRLEngine's building blocks).

Everything goes through the C ABI.  Integer work and every fp32 / fp64 quantity of the exact path are compared BIT-EXACTLY
with the oracle; against the reference's own Python (its outputs recorded in tests/golden/ref_long.npz) the tolerance is the one
BASELINE.json states: trades identical, fitness within 1e-5 relative, and a differing trajectory is excused only when the
oracle's own raw*5 comes within NEAR_TIE_TICKS of a rounding boundary somewhere along it (MKL's fp32 summation order is
not the SGMM-F32 order; the difference is ~1e-7 relative and flips a rounding only at such near-ties).
"""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

REL_TOL_VS_REFERENCE = 1e-5
NEAR_TIE_TICKS = 1e-4


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


# ----------------------------------------------------------------------------------------------
# config 5 length: T = 60 000 bars = 469 chunks of the 4-stage bar ring and the 2-stage record buffers
# ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bundle250(sg, orc):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(250, first_day=500)
    stats = synthetic.train_stats_of(bundle)
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    assert bun.T == 60000
    z1, z2 = orc.normalise(bundle, stats)
    return bundle, stats, bun, (z1, z2) + bundle[2:]


@pytest.mark.parametrize("P", [3, 33, 700])
def test_t60000_exact_path_bitwise(sg, orc, bundle250, P):
    from sgmm_b200 import synthetic
    bundle, stats, bun, bz = bundle250
    _, genomes = synthetic.policy_like_genomes(P, seed=60 + P, out_scale=3.0, out_bias=(0.1, 0.1))
    fit, trd = sg.rollout_population(bun, torch.from_numpy(genomes).cuda(), phi=1e-4)
    fit, trd = fit.cpu().numpy(), trd.cpu().numpy()
    # the oracle runs ~0.7 M env-steps/s on 8 threads: all of the small populations, a spread sample of the large one
    idx = np.arange(P) if P <= 40 else np.unique(np.concatenate([np.arange(0, P, 23), [P - 1, P - 2, 27, 28, 29]]))
    fo, to = orc.rollout_population(bz, 1e-4, 0.001, 0.0, genomes=genomes[idx])
    assert np.array_equal(bits64(fit[idx]), bits64(fo)), "fitness differs from the oracle at T = 60000"
    assert np.array_equal(trd[idx], to)
    assert trd.max() > 1000                      # the policies trade through the whole episode


def test_t60000_seeded_children_bitwise(sg, orc, bundle250):
    from sgmm_b200 import synthetic
    bundle, stats, bun, bz = bundle250
    master, _ = synthetic.policy_like_genomes(1, seed=5, out_scale=3.0, out_bias=(0.1, 0.1))
    fs, ts = sg.rollout_seeded(bun, torch.from_numpy(master).cuda(), count=40, sigma=0.05, seed=9, generation=3,
                               first_index=65000, phi=1e-4)
    fo, to = orc.rollout_population(bz, 1e-4, 0.001, 0.0, master=master, sigma=0.05, seed=9, generation=3,
                                    first_index=65000, count=40)
    assert np.array_equal(bits64(fs.cpu().numpy()), bits64(fo)) and np.array_equal(ts.cpu().numpy(), to)


# ----------------------------------------------------------------------------------------------
# config 3: 2048 market makers + 2048 adversaries x 14 400 bars
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fee", [0.0, 3e-5])
def test_config3_full_size_adversary_sampled_pairs_bitwise(sg, orc, fee):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(60)
    stats = synthetic.train_stats_of(bundle)
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    P = 2048
    _, genomes = synthetic.policy_like_genomes(P, seed=2, out_scale=4.0, out_bias=(0.1, 0.1))
    adv = (np.random.default_rng(3).standard_normal((P, 1250)) * 0.5).astype(np.float32)
    fit, trd = sg.rollout_population(bun, torch.from_numpy(genomes).cuda(), torch.from_numpy(adv).cuda(), phi=1e-4, fee_rate=fee)
    fit, trd = fit.cpu().numpy(), trd.cpu().numpy()
    idx = np.array([0, 1, 27, 28, 511, 1024, 2046, 2047])
    z1, z2 = orc.normalise(bundle, stats)
    fo, to = orc.rollout_population((z1, z2) + bundle[2:], 1e-4, 0.001, fee, genomes=genomes[idx], adv_genomes=adv[idx], use_adv=True)
    assert np.array_equal(bits64(fit[idx]), bits64(fo)) and np.array_equal(trd[idx], to)
    # the adversary matters: without it the same market makers earn something else
    f0, _ = sg.rollout_population(bun, torch.from_numpy(genomes[idx]).cuda(), phi=1e-4, fee_rate=fee)
    assert not np.array_equal(f0.cpu().numpy(), fit[idx])


# ----------------------------------------------------------------------------------------------
# config 4: H = 256, T = 28 800, with fee -- policy outputs within tolerance, env bit-exact given the offsets
# ----------------------------------------------------------------------------------------------
def test_config4_h256_t28800_fee_teacher_forced(sg, orc):
    from sgmm_b200 import synthetic
    TAU = 0.05
    bundle = synthetic.synthetic_bundle(120, first_day=300)
    stats = synthetic.train_stats_of(bundle)
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    assert bun.T == 28800
    z1, z2 = orc.normalise(bundle, stats)
    bz = (z1, z2) + bundle[2:]
    _, genomes = synthetic.policy_like_genomes(3, hidden=256, seed=44, out_scale=4.0, out_bias=(0.1, 0.1))
    fit, trd, raw, act = sg.rollout_spec256_audit(bun, genomes, phi=1e-4, fee_rate=3e-4)
    f2, t2 = sg.rollout_population(bun, torch.from_numpy(genomes).cuda(), phi=1e-4, fee_rate=3e-4, hidden=256)
    assert torch.equal(f2, fit) and torch.equal(t2, trd)
    fit, trd, raw, act = fit.cpu().numpy(), trd.cpu().numpy(), raw.cpu().numpy(), act.cpu().numpy()
    worst = 0.0
    for i in range(3):
        fo, to, tro = orc.rollout(None, None, bz, 1e-4, 0.001, 3e-4, forced_actions=act[i], trace=True)
        assert fo == fit[i] and to == trd[i], (i, fo, fit[i], to, trd[i])
        inv_before = np.concatenate([[0], tro["inventory"][:-1]])
        taken = np.rint(raw[i, np.arange(bun.T), inv_before + 2] * np.float32(5.0)).astype(np.int32)
        assert np.array_equal(taken, act[i])
        for t in range(i, bun.T, 997):               # sampled bars, every inventory, incl. the last tiles
            for iv in range(5):
                want = orc.mlp_forward(genomes[i], [z1[t], z2[t], (iv - 2) / 2.0], hidden=256)
                worst = max(worst, float(np.max(np.abs((want - raw[i, t, iv]) * np.float32(5.0)))))
    assert worst <= TAU, worst
    assert trd.min() > 100


def test_h256_f16_accumulator_envelope(sg, orc):
    """The hidden layer accumulates in f16 (TMEM); state the envelope: with the hidden weights scaled x8 (activations
    ~8x the orthogonal-init scale) the outputs stay within a RELATIVE tolerance of the fp32 oracle and nothing
    overflows; the tolerance in ticks grows with the activation scale, as f16's 11-bit significand dictates."""
    from sgmm_b200 import synthetic
    bundle = tuple(a[:200] for a in synthetic.synthetic_bundle(1, first_day=95))
    stats = synthetic.train_stats_of(synthetic.synthetic_bundle(1, first_day=95))
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    z1, z2 = orc.normalise(bundle, stats)
    H = 256
    _, genomes = synthetic.policy_like_genomes(2, hidden=H, seed=8, out_scale=1.0)
    g = genomes.copy()
    w2 = slice(4 * H, 4 * H + H * H)
    g[:, w2] *= np.float32(8.0)
    fit, trd, raw, act = sg.rollout_spec256_audit(bun, g, phi=1e-4)
    raw = raw.cpu().numpy()
    assert np.isfinite(raw).all() and np.isfinite(fit.cpu().numpy()).all()
    worst_rel = 0.0
    for i in range(2):
        for t in range(0, 200, 7):
            for iv in range(5):
                want = orc.mlp_forward(g[i], [z1[t], z2[t], (iv - 2) / 2.0], hidden=H)
                scale = max(1.0, float(np.max(np.abs(want))))
                worst_rel = max(worst_rel, float(np.max(np.abs(want - raw[i, t, iv]))) / scale)
    print("x8 hidden weights: max relative output error", worst_rel)
    assert worst_rel <= 4e-3          # ~8 f16 ulps (2^-11 each) of accumulated rounding


# ----------------------------------------------------------------------------------------------
# the unmodified reference at config-2 length
# ----------------------------------------------------------------------------------------------
def _reference_outputs(bundle, genomes, adv, fee, use_arl):
    """The reference's own fitness and trades on these episodes, as oracle/make_golden_long.py recorded them (its
    evaluate_individual in a Pool, run by oracle/run_ref.py) into tests/golden/ref_long.npz."""
    from sgmm_b200 import synthetic
    g = np.load(os.path.join(GOLDEN, "ref_long.npz"))
    P = genomes.shape[0]
    _, want = synthetic.policy_like_genomes(int(g["P"]), seed=int(g["genome_seed"]), out_scale=float(g["out_scale"]),
                                            out_bias=tuple(g["out_bias"]))
    assert np.array_equal(want, genomes) and len(bundle[0]) == 240 * int(g["days"]), "not the recorded episodes"
    if use_arl:
        assert np.array_equal(adv, (np.random.default_rng(int(g["adv_seed"])).standard_normal((P, 1250))
                                    * float(g["adv_scale"])).astype(np.float32)), "not the recorded adversaries"
    name = {(False, 0.0): "plain", (True, 0.0): "arl", (False, 3e-4): "fee", (True, 3e-4): "arl_fee"}[(use_arl, fee)]
    assert bool(g[f"{name}.use_arl"]) == use_arl and float(g[f"{name}.fee"]) == fee
    return g[f"{name}.fitness"].copy(), g[f"{name}.trades"].copy()


@pytest.mark.parametrize("use_arl,fee", [(False, 0.0), (True, 0.0), (False, 3e-4), (True, 3e-4)])
def test_cuda_vs_live_reference_8_individuals_14400_bars(sg, orc, use_arl, fee):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(60)
    stats = synthetic.train_stats_of(bundle)
    P = 8
    _, genomes = synthetic.policy_like_genomes(P, seed=12, out_scale=5.0, out_bias=(0.1, 0.1))
    adv = (np.random.default_rng(13).standard_normal((P, 1250)) * 0.5).astype(np.float32) if use_arl else None
    f_ref, t_ref = _reference_outputs(bundle, genomes, adv, fee, use_arl)
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    fit, trd = sg.rollout_population(bun, genomes, adv, phi=1e-4, fee_rate=fee)            # host entry (numpy in / out)
    z1, z2 = orc.normalise(bundle, stats)
    bz = (z1, z2) + bundle[2:]
    excused = 0
    for i in range(P):
        same = (trd[i] == t_ref[i]) and abs(fit[i] - f_ref[i]) <= REL_TOL_VS_REFERENCE * max(1.0, abs(f_ref[i]))
        if same:
            continue
        # a differing trajectory is acceptable only if the fp32 result itself sits on a rounding boundary somewhere
        _, _, tr = orc.rollout(genomes[i], adv[i] if use_arl else None, bz, 1e-4, 0.001, fee, trace=True)
        q = np.stack([tr["raw_a"], tr["raw_b"]], 1).astype(np.float32) * np.float32(5.0)
        margin = float(np.min(np.abs(np.abs(q - np.floor(q)) - 0.5)))
        assert margin <= NEAR_TIE_TICKS, (i, trd[i], t_ref[i], fit[i], f_ref[i], margin)
        excused += 1
    print(f"use_arl={use_arl} fee={fee}: {P - excused}/{P} trajectories identical to the reference "
          f"(trades equal, fitness within {REL_TOL_VS_REFERENCE} relative); {excused} excused at a logged near-tie")
    assert excused <= 2
    assert t_ref.min() > 100


# ----------------------------------------------------------------------------------------------
# H = 256 as a trainable config: device GA with spec256 for population and validation
# ----------------------------------------------------------------------------------------------
def test_h256_device_ga_matches_composed_rollouts(sg, orc):
    from sgmm_b200 import synthetic
    from sgmm_b200.engine import DeviceGA
    tb = tuple(a[:300] for a in synthetic.synthetic_bundle(2, first_day=120))
    vb = tuple(a[:200] for a in synthetic.synthetic_bundle(1, first_day=122))
    stats = synthetic.train_stats_of(tb)
    train = sg.Bundle.from_arrays(tb, stats, 0.001)
    val = sg.Bundle.from_arrays(vb, stats, 0.001)
    H, pop, gens = 256, 20, 4
    master, _ = synthetic.policy_like_genomes(1, hidden=H, seed=9, out_scale=4.0, out_bias=(0.1, 0.1))
    ga = DeviceGA(master, None, pop_size=pop, sigma=0.02, phi=1e-4, fee_rate=3e-4, use_arl=False, seed=123,
                  max_generations=gens, patience=2, hidden=H)
    for _ in range(gens):
        ga.generation(train, val)
    h = ga.history()
    assert len(h["val_f"]) == gens
    # compose the same GA from the public rollouts: children from the oracle's counter-based mutate, evaluated by the
    # same tensor-core kernel as explicit genomes (bit-identical to the seeded path), numpy argmax, validation rollout
    m = master.copy()
    sigma = np.float32(0.02)
    best_val, stale = -np.inf, 0
    for g in range(gens):
        kids = np.stack([orc.mutate(m, float(sigma), 123, g, i) for i in range(pop)])
        f, t = sg.rollout_population(train, torch.from_numpy(kids).cuda(), phi=1e-4, fee_rate=3e-4, hidden=H)
        f, t = f.cpu().numpy(), t.cpu().numpy()
        b = int(np.argmax(f))
        m = kids[b]
        fv, tv = sg.rollout_population(val, torch.from_numpy(m[None]).cuda(), phi=1e-4, fee_rate=3e-4, hidden=H)
        assert h["train_f"][g] == f[b] and h["train_trades"][g] == t[b], g
        assert h["val_f"][g] == fv.item() and h["val_trades"][g] == tv.item(), g
        assert h["sigma"][g] == sigma
        if fv.item() > best_val:
            best_val, stale = fv.item(), 0
        else:
            stale += 1
        if stale >= 2:
            sigma, stale = np.float32(sigma * np.float32(0.5)), 0
    mm, _, best = ga.masters()
    assert np.array_equal(mm, m)
    assert ga.status()["best_val"] == best_val


def test_drl_engine_hidden_dim_256(sg, tmp_path):
    from sgmm_b200 import synthetic
    tb = tuple(a[:240] for a in synthetic.synthetic_bundle(1, first_day=130))
    vb = tuple(a[:120] for a in synthetic.synthetic_bundle(1, first_day=131))
    stats = synthetic.train_stats_of(tb)
    torch.manual_seed(3)
    eng = sg.DRLEngine(pop_size=12, phi=1e-4, tick_size=0.001, fee_rate=3e-4, save_dir=str(tmp_path), seed=4, hidden_dim=256)
    assert eng.mm_evolver.master_policy.net[0].out_features == 256
    policy, hist = eng.train(tb, vb, stats, generations=3, verbose=False)
    assert len(hist["val_f"]) == 3 and policy.net[2].weight.shape == (256, 256)
    sd = torch.load(tmp_path / "agent_best_val_0.0001.pth", weights_only=True)
    assert sd["net.2.weight"].shape == (256, 256)
    # the returned policy reproduces its validation fitness through the same path
    val = sg.Bundle.from_arrays(vb, stats, 0.001)
    f, _ = sg.rollout_population(val, policy.get_weights().reshape(1, -1).cuda(), phi=1e-4, fee_rate=3e-4, hidden=256)
    assert f.item() == max(hist["val_f"])


# ----------------------------------------------------------------------------------------------
# pipelined host entry; repeated train() calls; in-process second device
# ----------------------------------------------------------------------------------------------
def test_pipelined_host_entry_matches_synchronous(sg):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(2, first_day=140)
    stats = synthetic.train_stats_of(bundle)
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    batches = [synthetic.policy_like_genomes(n, seed=70 + k, out_scale=4.0)[1] for k, n in enumerate((50, 0, 333, 7, 120))]
    want = [sg.rollout_population(bun, g, phi=1e-4, fee_rate=3e-5) if len(g) else (np.empty(0), np.empty(0, np.int32)) for g in batches]
    pend = [sg.rollout_population_async(bun, torch.from_numpy(g).pin_memory() if len(g) else torch.empty(0, 1250), phi=1e-4, fee_rate=3e-5)
            for g in batches]                       # five submissions, two in flight at a time
    for (f, t), p in zip(want, pend):
        fa, ta = p.result()
        assert np.array_equal(bits64(fa), bits64(f)) and np.array_equal(ta, t)
    # tensor-core precision through the same entry
    f16, t16 = sg.rollout_population(bun, batches[0], phi=1e-4, precision="f16")
    fa, ta = sg.rollout_population_async(bun, torch.from_numpy(batches[0]).pin_memory(), phi=1e-4, precision="f16").result()
    assert np.array_equal(bits64(fa), bits64(f16)) and np.array_equal(ta, t16)


def test_repeated_train_calls_draw_fresh_noise(sg, tmp_path):
    from sgmm_b200 import synthetic
    tb = synthetic.synthetic_bundle(1, first_day=150)
    vb = synthetic.synthetic_bundle(1, first_day=151)
    stats = synthetic.train_stats_of(tb)

    def run(seed, calls=1):
        torch.manual_seed(0)
        eng = sg.DRLEngine(pop_size=16, phi=1e-4, tick_size=0.001, save_dir=str(tmp_path), seed=seed)
        return [eng.train(tb, vb, stats, generations=2, verbose=False)[1]["train_f"] for _ in range(calls)]
    a, b = run(5, 2)
    assert a != b                                    # the second train() call does not replay the first one's noise
    assert run(5)[0] == a                            # an explicit seed is reproducible
    torch.manual_seed(0)
    e1 = sg.DRLEngine(pop_size=16, phi=1e-4, tick_size=0.001, save_dir=str(tmp_path))      # seed=None: torch's generator
    e2 = sg.DRLEngine(pop_size=16, phi=1e-4, tick_size=0.001, save_dir=str(tmp_path))
    e2.mm_evolver.master_policy.set_weights(e1.mm_evolver.master_policy.get_weights())
    h1 = e1.train(tb, vb, stats, generations=2, verbose=False)[1]["train_f"]
    h2 = e2.train(tb, vb, stats, generations=2, verbose=False)[1]["train_f"]
    assert h1 != h2                                  # two engines of a sweep are independent, like the reference's randn


def test_sigma_argument_is_not_forwarded_like_the_reference(sg, tmp_path):
    eng = sg.DRLEngine(pop_size=5, sigma=0.9, save_dir=str(tmp_path))
    assert eng.mm_evolver.sigma == 0.05              # Env/drl_engine.py:77 builds NeuroEvolution(population_size=pop_size)


def test_second_device_in_process_if_present(sg):
    """cudaFuncAttributeMaxDynamicSharedMemorySize is per device: a second device in the same process must work."""
    if torch.cuda.device_count() < 2:
        pytest.skip("one visible device")
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(1, first_day=160)
    stats = synthetic.train_stats_of(bundle)
    _, genomes = synthetic.policy_like_genomes(40, seed=1, out_scale=4.0)
    res = []
    for d in (0, 1):
        bun = sg.Bundle.from_arrays(bundle, stats, 0.001, device=d)
        with torch.cuda.device(d):
            f, t = sg.rollout_population(bun, torch.from_numpy(genomes).to(f"cuda:{d}"), phi=1e-4)
            f16, _ = sg.rollout_population(bun, torch.from_numpy(genomes).to(f"cuda:{d}"), phi=1e-4, precision="f16")
        res.append((f.cpu(), t.cpu(), f16.cpu()))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1]) and torch.equal(res[0][2], res[1][2])


# ----------------------------------------------------------------------------------------------
# memory safety without compute-sanitizer (closed on this pool): canaries around every output buffer
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hidden,precision,use_adv,P,T", [(32, "f32", True, 29, 131), (32, "f32", False, 3, 1), (32, "f16", False, 17, 51),
                                                           (32, "tf32", True, 9, 26), (32, "bf16", True, 150, 25), (256, "bf16", False, 5, 27)])
def test_kernels_write_nothing_outside_their_output_buffers(sg, hidden, precision, use_adv, P, T):
    import ctypes as C
    from sgmm_b200 import _lib, synthetic
    from sgmm_b200.engine import _params
    bundle = tuple(a[:T] for a in synthetic.synthetic_bundle(1, first_day=180))
    stats = synthetic.train_stats_of(synthetic.synthetic_bundle(1, first_day=180))
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    _, genomes = synthetic.policy_like_genomes(P, hidden=hidden, seed=P, out_scale=4.0)
    g = torch.from_numpy(genomes).cuda()
    adv = torch.from_numpy((np.random.default_rng(1).standard_normal((P, 1250)) * 0.5).astype(np.float32)).cuda() if use_adv else None
    PAD = 64
    CAN_F, CAN_I = -1.2345e300, -77777777
    fit = torch.full((P + 2 * PAD,), CAN_F, dtype=torch.float64, device="cuda")
    trd = torch.full((P + 2 * PAD,), CAN_I, dtype=torch.int32, device="cuda")
    audit = precision != "f32"
    raw = torch.full((P * T * 10 + 2 * PAD,), 7.25, dtype=torch.float32, device="cuda") if audit else None
    act = torch.full((P * T * 2 + 2 * PAD,), CAN_I, dtype=torch.int32, device="cuda") if audit else None
    mm = _lib.Population(hidden, 0, P, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    ad = _lib.Population(32, 0, P, adv.data_ptr(), None, 0.0, 0.0, 0, 0, 0) if use_adv else None
    prm = _params(1e-4, 3e-5, hidden=hidden, precision=precision)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    L = _lib.lib()
    if audit:
        _lib.check(L.sgmm_rollout_tc_audit(bun.handle, C.byref(mm), None if ad is None else C.byref(ad), C.byref(prm),
                                           fit.data_ptr() + PAD * 8, trd.data_ptr() + PAD * 4, raw.data_ptr() + PAD * 4,
                                           act.data_ptr() + PAD * 4, st))
    else:
        _lib.check(L.sgmm_rollout_population(bun.handle, C.byref(mm), None if ad is None else C.byref(ad), C.byref(prm),
                                             fit.data_ptr() + PAD * 8, trd.data_ptr() + PAD * 4, st))
    torch.cuda.synchronize()
    for buf, can, n in ((fit, CAN_F, P), (trd, CAN_I, P)) + (((raw, 7.25, P * T * 10), (act, CAN_I, P * T * 2)) if audit else ()):
        assert bool((buf[:PAD] == can).all()) and bool((buf[PAD + n:] == can).all()), "a kernel wrote outside its output buffer"
    assert bool((fit[PAD:PAD + P] != CAN_F).all()) and bool((trd[PAD:PAD + P] != CAN_I).all())
    if audit:
        assert bool((act[PAD:PAD + P * T * 2] != CAN_I).all())


# ----------------------------------------------------------------------------------------------
# the GA's validation rollout: policy table for every (bar, inventory) + automaton scan + reference-order sum
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("days,T", [(1, 0), (1, 1), (1, 7), (1, 240), (9, 2049), (12, 2880), (250, 60000)])
@pytest.mark.parametrize("fee", [0.0, 3e-4])
def test_validation_fast_path_is_bit_identical_to_the_sequential_kernel_and_the_oracle(sg, orc, days, T, fee):
    """sgmm_one.cu (one individual's episode as 5T parallel policy evaluations + a prefix scan over the 5-state automaton)
    against rollout_kernel_h32 and the oracle: empty, single-bar, ragged, chunk-boundary (2048 + 1) and 60 000-bar episodes."""
    from sgmm_b200 import synthetic
    from sgmm_b200.engine import DeviceGA
    vb = tuple(a[:T] for a in synthetic.synthetic_bundle(days, first_day=400))
    tb = synthetic.synthetic_bundle(1, first_day=399)
    stats = synthetic.train_stats_of(tb)
    train, val = sg.Bundle.from_arrays(tb, stats, 0.001), sg.Bundle.from_arrays(vb, stats, 0.001)
    master, _ = synthetic.policy_like_genomes(1, seed=T + 1, out_scale=4.0, out_bias=(0.1, 0.1))
    ga = DeviceGA(master, None, pop_size=6, sigma=0.05, phi=1e-4, fee_rate=fee, use_arl=False, seed=3, max_generations=3)
    ga.generation(train, val)
    ga.generation(train, val)
    h = ga.history(2)
    mm, _, _ = ga.masters()
    ga.close()
    f, t = sg.rollout_population(val, torch.from_numpy(mm[None]).cuda(), phi=1e-4, fee_rate=fee)        # the sequential kernel
    z1, z2 = orc.normalise(vb, stats)
    fo, to = orc.rollout(mm, None, (z1, z2) + vb[2:], 1e-4, 0.001, fee)
    assert h["val_f"][1] == f.item() == fo, (h["val_f"][1], f.item(), fo)
    assert h["val_trades"][1] == t.item() == to
    if T >= 240:
        assert to > 0


@pytest.mark.parametrize("name", ["plain", "arl", "fee", "arl_fee"])
def test_cuda_matches_the_committed_long_reference_vectors(sg, orc, name):
    """tests/golden/ref_long.npz: the unmodified reference on 8 individuals x 14 400 bars (oracle/make_golden_long.py) --
    the config-2 length pinned by committed vectors, with every trajectory's minimum rounding margin logged."""
    from test_oracle_golden import _long_case, check_against_long_reference
    bundle, stats, genomes, adv, fee, f_ref, t_ref = _long_case(name)
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    fit, trd = sg.rollout_population(bun, torch.from_numpy(genomes).cuda(), None if adv is None else torch.from_numpy(adv).cuda(),
                                     phi=1e-4, fee_rate=fee, units_per_lane=4)                       # the population kernel
    check_against_long_reference(name, fit.cpu().numpy(), trd.cpu().numpy(), orc)
    if adv is None:                                                                                  # and the small-population path
        f2, t2 = sg.rollout_population(bun, torch.from_numpy(genomes).cuda(), phi=1e-4, fee_rate=fee)
        assert torch.equal(f2, fit) and torch.equal(t2, trd)


@pytest.mark.parametrize("days,T", [(1, 0), (1, 1), (1, 7), (9, 2049), (60, 14400)])
@pytest.mark.parametrize("use_adv,fee", [(False, 0.0), (True, 0.0), (True, 3e-4)])
def test_small_population_path_equals_sequential_kernel_and_oracle(sg, orc, days, T, use_adv, fee):
    """The launcher's two routes for a small population -- policy table + automaton scan (sgmm_one.cu: 5 states, 20 with the
    adversary) and the sequential kernel (pinned by units_per_lane) -- against each other and the oracle, explicit and seeded."""
    from sgmm_b200 import synthetic
    bundle = tuple(a[:T] for a in synthetic.synthetic_bundle(days, first_day=420))
    stats = synthetic.train_stats_of(synthetic.synthetic_bundle(1, first_day=419))
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    P = 7
    master, genomes = synthetic.policy_like_genomes(P, seed=T + 3, out_scale=4.0, out_bias=(0.1, 0.1))
    adv = (np.random.default_rng(T + 4).standard_normal((P, 1250)) * 0.6).astype(np.float32) if use_adv else None
    g = torch.from_numpy(genomes).cuda()
    a = None if adv is None else torch.from_numpy(adv).cuda()
    f_small, t_small = sg.rollout_population(bun, g, a, phi=1e-4, fee_rate=fee)
    f_seq, t_seq = sg.rollout_population(bun, g, a, phi=1e-4, fee_rate=fee, units_per_lane=1)
    assert torch.equal(f_small, f_seq) and torch.equal(t_small, t_seq)
    z1, z2 = orc.normalise(bundle, stats)
    bz = (z1, z2) + bundle[2:]
    fo, to = orc.rollout_population(bz, 1e-4, 0.001, fee, genomes=genomes, adv_genomes=adv, use_adv=use_adv)
    assert np.array_equal(bits64(f_small.cpu().numpy()), bits64(fo)) and np.array_equal(t_small.cpu().numpy(), to)
    # seeded children (and seeded adversaries): both routes regenerate the same genomes
    am = None if adv is None else torch.from_numpy(adv[0]).cuda()
    kw = dict(count=9, sigma=0.05, seed=21, generation=2, first_index=5, adv_master=am, phi=1e-4, fee_rate=fee)
    fs1, ts1 = sg.rollout_seeded(bun, torch.from_numpy(master).cuda(), **kw)
    fs2, ts2 = sg.rollout_seeded(bun, torch.from_numpy(master).cuda(), units_per_lane=4, **kw)
    assert torch.equal(fs1, fs2) and torch.equal(ts1, ts2)
