"""Truncation selection with weighted recombination (sgmm_ga_set_parents, DeviceGA / DeviceGASweep / DRLEngine ``parents``).

The rank order (NaN first, then descending fitness -- the adversary's ascending --, ties to the lower index, -0.0 == +0.0)
and the recombined master ``m + sigma * sum_k w_k eps_k`` must match the references below bit for bit; ``w = [1, 0, ...]``
must be the (1,lambda) GA at any mu, on every population route.  The references: ``select_parents`` is a numpy ``lexsort``
restatement of the order; ``recombine`` draws every parent's noise from the CPU oracle (``oracle.mutate`` of a zero master
with sigma 1 is the noise itself) and chains an exact binary32 fused multiply-add, checked against libm's ``fmaf``."""
import ctypes as C
import ctypes.util
import functools

import numpy as np
import pytest

FLIP = 0x8000000000000000


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


def bits32(a):
    return np.asarray(a, np.float32).view(np.uint32)


def lexsort_order(f, sign=1):
    """numpy restatement of the rank order: NaN first, then descending sign*f, then ascending index."""
    f = np.asarray(f, np.float64)
    v = sign * f
    nan = np.isnan(v)
    key = np.where(nan, 0.0, -v) + 0.0                            # + 0.0: -0.0 -> +0.0
    return np.lexsort((np.arange(f.size), key, ~nan))


def select_parents(f, mu, sign=1):
    """The first ``mu`` children of the rank order as int64[mu]; ``sign=-1`` is the adversary's order."""
    f = np.asarray(f, np.float64)
    if not 1 <= mu <= f.size:
        raise ValueError(f"mu={mu} outside 1..{f.size}")
    return lexsort_order(f, sign)[:mu].astype(np.int64)


def fmaf(a, b, c):
    """binary32 fused multiply-add, element-wise and exact (libm's fmaf).  a*b is exact in binary64 (24 + 24 bits); the
    binary64 sum s = a*b + c and its exact error e (TwoSum) give the true value s + e.  Rounding s to binary32 rounds
    s + e the same way unless s lies exactly halfway between two binary32 values and e != 0: then e decides."""
    a, b, c = (np.asarray(x, np.float32) for x in (a, b, c))
    p = a.astype(np.float64) * b.astype(np.float64)
    c64 = c.astype(np.float64)
    s = p + c64
    bv = s - p
    e = (p - (s - bv)) + (c64 - bv)
    r = s.astype(np.float32)
    d = s - r.astype(np.float64)
    nb = np.nextafter(r, np.where(d > 0, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32))
    half = (d != 0) & (d == nb.astype(np.float64) - s) & (e != 0)
    return np.where(half & (np.sign(e) == np.sign(d)), nb, r).astype(np.float32)


def noise(G, seed, generation, individual):
    """eps of one child: the oracle's child of a zero master with sigma 1 (0 + n*1 == n)."""
    from oracle import oracle as orc
    return orc.mutate(np.zeros(G, np.float32), 1.0, seed, generation, int(individual))


def recombine(master, sigma, seed, generation, idx, w):
    """m + (w0*eps_0 -> fmaf(w_k, eps_k, acc) in rank order) * sigma, every operation one binary32 rounding."""
    m = np.asarray(master, np.float32)
    w = np.asarray(w, np.float32)
    if len(idx) == 0 or w.size != len(idx):
        raise ValueError("one weight per parent, at least one parent")
    acc = w[0] * noise(m.size, seed, generation, idx[0])
    for k in range(1, len(idx)):
        acc = fmaf(w[k], noise(m.size, seed, generation, idx[k]), acc)
    return (m + acc * np.float32(sigma)).astype(np.float32)


PALETTE = np.array([-50.0, -50.0, -50.0, 0.0, -0.0, np.inf, -np.inf, np.nan, 1.5, 1.5, 2.0, -3.0, 1e-300, -1e-300])


def crafted(n, kind, seed=0):
    rng = np.random.default_rng(seed + n)
    if kind == "palette":                                         # ties everywhere, NaN, +-inf, +-0.0
        return PALETTE[rng.integers(0, PALETTE.size, n)]
    if kind == "plateau":                                         # every child at the no-trade penalty
        return np.full(n, -50.0)
    if kind == "cut":                                             # a tie of 7 values spanning every small cut
        f = rng.standard_normal(n) - 100.0
        f[rng.permutation(n)[:min(n, 7)]] = -100.0 + 0.25
        f[rng.permutation(n)[:min(n, 3)]] = 5.0
        return f
    return rng.standard_normal(n)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("n", [1, 2, 50, 4097])
@pytest.mark.parametrize("kind", ["palette", "plateau", "cut", "normal"])
def test_select_parents_is_the_rank_order(n, kind):
    """the lexsort restatement against a literal comparator sort, and mu = 1 against the oracle's numpy argmax"""
    from oracle import oracle as orc
    f = crafted(n, kind)
    for sign in (1, -1):
        def before(i, j):
            a, b = sign * f[i], sign * f[j]
            if np.isnan(a) != np.isnan(b):
                return -1 if np.isnan(a) else 1
            if not np.isnan(a) and a != b:
                return -1 if a > b else 1
            return -1 if i < j else (1 if i > j else 0)
        literal = sorted(range(n), key=functools.cmp_to_key(before))
        for mu in sorted({1, 2, 7, 50, 1024, n}):
            if mu <= n:
                assert select_parents(f, mu, sign).tolist() == literal[:mu], (kind, n, sign, mu)
        assert select_parents(f, 1, sign)[0] == orc.argmax(sign * f)      # mu = 1 is the (1,lambda) argmax


def test_select_parents_details():
    f = np.array([1.0, np.nan, 2.0, np.nan, -0.0, 0.0, 2.0])
    assert select_parents(f, 7).tolist() == [1, 3, 2, 6, 0, 4, 5]
    assert select_parents(f, 7, -1).tolist() == [1, 3, 4, 5, 0, 2, 6]
    with pytest.raises(ValueError):
        select_parents(f, 8)
    with pytest.raises(ValueError):
        select_parents(f, 0)


def test_fmaf_is_libm_fmaf():
    libm = C.CDLL(ctypes.util.find_library("m"))
    libm.fmaf.restype = C.c_float
    libm.fmaf.argtypes = [C.c_float, C.c_float, C.c_float]
    rng = np.random.default_rng(11)
    n = 20000
    a = (rng.standard_normal(n) * 2.0 ** rng.integers(-30, 30, n)).astype(np.float32)
    b = rng.standard_normal(n).astype(np.float32)
    c = (rng.standard_normal(n) * 2.0 ** rng.integers(-40, 20, n)).astype(np.float32)
    # products with a 2^-24 tail land exactly halfway between binary32 values; a tiny c then decides the rounding
    k = rng.integers(1, 2 ** 11, n)
    j = rng.integers(1, 2 ** 11, n)
    a2 = (1.0 + k * 2.0 ** -12).astype(np.float32)
    b2 = (1.0 + j * 2.0 ** -12).astype(np.float32)
    c2 = (rng.choice([-1.0, 0.0, 1.0], n) * 2.0 ** -60).astype(np.float32)
    for x, y, z in ((a, b, c), (a2, b2, c2), (a, b, -(a * b))):
        got = fmaf(x, y, z)
        ref = np.array([libm.fmaf(float(p), float(q), float(r)) for p, q, r in zip(x, y, z)], np.float32)
        assert np.array_equal(bits32(got), bits32(ref))


def test_recombine_with_one_weight_is_mutate():
    from oracle import oracle as orc
    rng = np.random.default_rng(3)
    for G in (1250, 67330, 5):
        m = rng.standard_normal(G).astype(np.float32)
        for idx in (0, 17, 2 ** 33 + 1):
            a = recombine(m, 0.05, 7, 3, [idx], [1.0])
            assert np.array_equal(bits32(a), bits32(orc.mutate(m, 0.05, 7, 3, idx)))
            z = recombine(m, 0.05, 7, 3, [idx, 4, 9], [1.0, 0.0, 0.0])
            assert np.array_equal(bits32(z), bits32(a))


def test_python_argument_errors_before_any_device_call(tmp_path):
    import sgmm_b200
    kw = dict(pop_size=8, sigma=0.05, phi=0.0, fee_rate=0.0, use_arl=False, seed=1, max_generations=2)
    m = np.zeros(1250, np.float32)
    bad = [dict(parents=0), dict(parents=9), dict(parents=1025), dict(parents=2.5), dict(parents=True),
           dict(parents=2, weights=[1.0]), dict(parents=2, weights=[1.0, -1.0]), dict(parents=2, weights=[0.0, 0.0]),
           dict(parents=2, weights=[1.0, np.inf]), dict(parents=2, weights=[np.nan, 1.0]), dict(weights=[1.0, 1.0])]
    for b in bad:
        with pytest.raises(ValueError):
            sgmm_b200.DeviceGA(m, **kw, **b)
        with pytest.raises(ValueError):
            sgmm_b200.DeviceGASweep(m, runs=[dict(seed=1, phi=0.0)], pop_size=8, use_arl=False, max_generations=2, **b)
    with pytest.raises(ValueError):
        sgmm_b200.DRLEngine(pop_size=8, parents=9, save_dir=str(tmp_path))
    with pytest.raises(ValueError):
        sgmm_b200.DRLEngine(pop_size=8, parents=2, parent_weights=[1.0, -0.5], save_dir=str(tmp_path))


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def sg():
    import torch
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


def masters(seed, use_arl=True, hidden=32):
    from sgmm_b200 import synthetic
    from sgmm_b200.policy import genome_len
    if hidden == 32:
        mm = synthetic.policy_like_genomes(1, seed=seed, out_scale=1.0)[0]
    else:
        mm = (np.random.default_rng(seed).standard_normal(genome_len(hidden)) * 0.05).astype(np.float32)
    adv = (np.random.default_rng(seed + 4).standard_normal(1250) * 0.5).astype(np.float32) if use_arl else None
    return mm, adv


def weights_of(kind, mu):
    if kind == "equal":
        return None
    if kind == "logrank":
        w = np.log(mu + 0.5) - np.log(np.arange(1, mu + 1))
        return (w / w.sum()).astype(np.float32)
    if kind == "onehot":
        return np.eye(1, mu, dtype=np.float32)[0]
    raise ValueError(kind)


def full_w(w, mu):
    return np.full(mu, np.float32(1.0) / np.float32(mu), np.float32) if w is None else np.asarray(w, np.float32)


def write_fitness(sg, ga, f):
    import torch
    from sgmm_b200.dist import device_tensor
    fp, tp, *_ = ga.buffers()
    device_tensor(fp, f.size, torch.float64, ga.device).copy_(torch.from_numpy(np.ascontiguousarray(f, np.float64)))
    device_tensor(tp, f.size, torch.int32, ga.device).copy_(torch.arange(f.size, dtype=torch.int32))


CRAFTED = [(lam, mu) for lam in (1, 50, 4097, 65536) for mu in sorted({1, 2, 50, 1024, lam}) if mu <= min(lam, 1024)]


@pytest.mark.gpu
@pytest.mark.parametrize("lam,mu", CRAFTED)
def test_crafted_fitness_select_and_recombine(sg, data, lam, mu):
    _, _, _, _, val = data
    sigma, seed = 0.05, 1234
    m0, a0 = masters(lam + mu)
    for kind in ("palette", "plateau", "cut", "normal"):
        f = crafted(lam, kind, seed=mu)
        w = np.ones(1, np.float32) if mu == 1 else weights_of("logrank" if kind == "cut" else "equal", mu)
        ga = sg.DeviceGA(m0, a0, pop_size=lam, sigma=sigma, phi=1e-4, fee_rate=0.0, use_arl=True, seed=seed,
                         max_generations=1, parents=mu, weights=w)
        write_fitness(sg, ga, f)
        ga.select(val)
        pm, pa = ga.parents()
        om, oa = select_parents(f, mu, 1), select_parents(f, mu, -1)
        assert np.array_equal(pm, om), (kind, "mm")
        assert np.array_equal(pa, oa), (kind, "adv")
        mm, adv, _ = ga.masters()
        assert np.array_equal(bits32(mm), bits32(recombine(m0, sigma, seed, 0, om, full_w(w, mu)))), kind
        assert np.array_equal(bits32(adv), bits32(recombine(a0, sigma, seed ^ FLIP, 0, oa, full_w(w, mu)))), kind
        st, h = ga.status(), ga.history()
        assert st["last_best_index"] == om[0]
        assert bits64(h["train_f"][0]) == bits64(f[om[0]]) and h["train_trades"][0] == om[0]
        ga.close()


def run_ga(sg, train, val, m, a, gens, **kw):
    ga = sg.DeviceGA(m, a, max_generations=gens, **kw)
    for _ in range(gens):
        ga.generation(train, val)
    out = ga.history(gens), ga.status(), ga.masters(), ga.parents()
    ga.close()
    return out


def assert_same(x, y, what=""):
    (hx, sx, mx, _), (hy, sy, my, _) = x, y
    for k in hx:
        assert np.array_equal(hx[k].view(np.uint8), hy[k].view(np.uint8)), (what, k)
    assert sx == sy, (what, sx, sy)
    for p, q, name in zip(mx, my, ("mm", "adv", "best")):
        assert np.array_equal(bits32(p), bits32(q)), (what, name)


def oracle_ga(orc, tz, vz, master, adv_master, *, pop, mu, w, sigma, phi, tick, fee, use_arl, seed, gens, patience,
              hidden=32):
    """The GA composed from oracle rollouts + the select_parents / recombine references (drl_engine.py's loop with truncation selection)."""
    master = master.copy()
    adv_master = None if adv_master is None else adv_master.copy()
    s_mm = s_adv = np.float32(sigma)
    best_val, stale, best_master = -np.inf, 0, master.copy()
    hist = {k: [] for k in ("train_f", "val_f", "train_trades", "val_trades", "sigma")}
    last = None
    for gen in range(gens):
        fit, trd = orc.rollout_population(tz, phi, tick, fee, master=master, sigma=float(s_mm), adv_master=adv_master,
                                          adv_sigma=float(s_adv), use_adv=use_arl, seed=seed, generation=gen, count=pop,
                                          hidden=hidden, nthreads=4)
        pm = select_parents(fit, mu, 1)
        master = recombine(master, float(s_mm), seed, gen, pm, w)
        pa = np.zeros(mu, np.int64)
        if use_arl:
            pa = select_parents(fit, mu, -1)
            adv_master = recombine(adv_master, float(s_adv), seed ^ FLIP, gen, pa, w)
        last = (pm, pa)
        vf, vt = orc.rollout(master, None, vz, phi, tick, fee, hidden=hidden)
        hist["train_f"].append(fit[pm[0]]); hist["train_trades"].append(trd[pm[0]])
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
    return hist, master, adv_master, best_master, best_val, s_mm, last


def check_against_oracle(got, ref, use_arl):
    (h, st, (m, a, b), (pm, pa)) = got
    ho, m_o, a_o, b_o, bv_o, s_o, (pm_o, pa_o) = ref
    assert np.array_equal(bits64(h["train_f"]), bits64(ho["train_f"]))
    assert np.array_equal(bits64(h["val_f"]), bits64(ho["val_f"]))
    assert h["train_trades"].tolist() == ho["train_trades"] and h["val_trades"].tolist() == ho["val_trades"]
    assert np.array_equal(h["sigma"], np.array(ho["sigma"], np.float32))
    assert np.array_equal(bits32(m), bits32(m_o)) and np.array_equal(bits32(b), bits32(b_o))
    assert st["best_val"] == bv_o and st["sigma"] == s_o and st["last_best_index"] == pm_o[0]
    assert np.array_equal(pm, pm_o)
    if use_arl:
        assert np.array_equal(bits32(a), bits32(a_o)) and np.array_equal(pa, pa_o)


@pytest.mark.gpu
@pytest.mark.parametrize("mu,wkind,use_arl", [(2, "equal", False), (7, "logrank", True), (24, "equal", True),
                                              (7, "onehot", False), (2, "logrank", True)])
def test_ga_matches_oracle_composed_ga(sg, data, mu, wkind, use_arl):
    from oracle import oracle as orc
    tb, vb, stats, train, val = data
    tz = orc.normalise(tb, stats) + tb[2:]
    vz = orc.normalise(vb, stats) + vb[2:]
    pop, gens, seed = 24, 10, 41 + mu
    m0, a0 = masters(mu, use_arl)
    w = weights_of(wkind, mu)
    got = run_ga(sg, train, val, m0, a0, gens, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=use_arl, seed=seed,
                 patience=1, parents=mu, weights=w)
    ref = oracle_ga(orc, tz, vz, m0, a0, pop=pop, mu=mu, w=full_w(w, mu), sigma=0.05, phi=1e-4, tick=0.001, fee=3e-4,
                    use_arl=use_arl, seed=seed, gens=gens, patience=1)
    check_against_oracle(got, ref, use_arl)
    assert got[1]["sigma"] < np.float32(0.05)                      # sigma decayed at least once


@pytest.mark.gpu
def test_h256_exact_matches_oracle_composed_ga(sg):
    from oracle import oracle as orc
    from sgmm_b200 import synthetic
    full = synthetic.synthetic_bundle(1, first_day=60)
    tb = tuple(np.ascontiguousarray(x[:240]) for x in full)
    vb = tuple(np.ascontiguousarray(x[240:400]) for x in full)
    stats = synthetic.train_stats_of(full)
    train, val = sg.Bundle.from_arrays(tb, stats, 0.001), sg.Bundle.from_arrays(vb, stats, 0.001)
    tz = orc.normalise(tb, stats) + tb[2:]
    vz = orc.normalise(vb, stats) + vb[2:]
    m0, a0 = masters(5, True, hidden=256)
    mu, pop, gens = 3, 6, 4
    w = weights_of("logrank", mu)
    got = run_ga(sg, train, val, m0, a0, gens, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=True, seed=9,
                 patience=1, parents=mu, weights=w, hidden=256, precision="exact")
    ref = oracle_ga(orc, tz, vz, m0, a0, pop=pop, mu=mu, w=w, sigma=0.05, phi=1e-4, tick=0.001, fee=0.0, use_arl=True,
                    seed=9, gens=gens, patience=1, hidden=256)
    check_against_oracle(got, ref, True)


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,precision", [(32, "f32"), (32, "f16"), (256, "bf16")])
def test_onehot_weights_equal_the_default_ga(sg, data, hidden, precision):
    _, _, _, train, val = data
    m0, a0 = masters(17, True, hidden=hidden)
    kw = dict(pop_size=40, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=True, seed=5, patience=2, hidden=hidden,
              precision=precision)
    gens = 6
    base = run_ga(sg, train, val, m0, a0, gens, **kw)
    five = run_ga(sg, train, val, m0, a0, gens, parents=5, weights=[1, 0, 0, 0, 0], **kw)
    one = run_ga(sg, train, val, m0, a0, gens, weights=[1.0], **kw)     # mu = 1 through the selection kernels
    assert_same(base, five, "w=[1,0,0,0,0]")
    assert_same(base, one, "w=[1]")
    assert five[3][0][0] == base[3][0][0] == base[1]["last_best_index"]
    assert five[3][1][0] == base[3][1][0]


@pytest.mark.gpu
def test_sweep_runs_equal_their_solo_gas(sg, data):
    from sgmm_b200 import synthetic
    _, _, _, train, val = data
    # a three-bar bundle: most children sit on the -50 no-trade plateau, at different levels per run
    full = synthetic.synthetic_bundle(2, first_day=80)
    stats = synthetic.train_stats_of(full)
    short = sg.Bundle.from_arrays(tuple(np.ascontiguousarray(x[:3]) for x in full), stats, 0.001)
    runs = [dict(seed=11, phi=0.0, fee_rate=0.0, sigma=0.05, patience=1),
            dict(seed=12, phi=1e-4, fee_rate=3e-4, sigma=0.02, patience=2),
            dict(seed=2 ** 63 + 5, phi=0.01, fee_rate=-1e-4, sigma=0.08, patience=3)]
    K, pop, gens, mu = len(runs), 24, 6, 5
    mm = np.stack([masters(3 + r)[0] for r in range(K)])
    adv = np.stack([masters(3 + r)[1] for r in range(K)])
    w = weights_of("logrank", mu)
    for tr in (train, short):
        ga = sg.DeviceGASweep(mm, adv, runs=runs, pop_size=pop, use_arl=True, max_generations=gens, parents=mu, weights=w)
        for _ in range(gens):
            ga.generation(tr, val)
        for r in range(K):
            sweep = ga.history(r, gens), ga.status(r), ga.masters(r), ga.parents(r)
            solo = run_ga(sg, tr, val, mm[r], adv[r], gens, pop_size=pop, use_arl=True, precision="exact", parents=mu,
                          weights=w, **runs[r])
            assert_same(sweep, solo, f"run {r}")
            assert np.array_equal(sweep[3][0], solo[3][0]) and np.array_equal(sweep[3][1], solo[3][1])
        ga.close()


@pytest.mark.gpu
def test_two_shards_on_one_device_equal_the_unsharded_ga(sg, data):
    import torch
    from sgmm_b200.dist import device_tensor
    _, _, _, train, val = data
    m0, a0 = masters(23)
    pop, mu, gens = 50, 7, 5
    kw = dict(pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=True, seed=77, patience=2, max_generations=gens,
              parents=mu, weights=weights_of("logrank", mu))
    stride = 25
    shards = [sg.DeviceGA(m0, a0, shard=(0, 25, stride), **kw), sg.DeviceGA(m0, a0, shard=(25, 25, stride), **kw)]
    views = []
    for ga in shards:
        _, _, base, bb, nb, my = ga.buffers()
        assert nb == 2
        views.append((device_tensor(base, nb * bb, torch.uint8, ga.device), bb, my))
    for _ in range(gens):
        for ga in shards:
            ga.evaluate(train)
        for (dst, bb, _), (src, _, my) in ((views[0], views[1]), (views[1], views[0])):
            dst[my * bb:(my + 1) * bb].copy_(src[my * bb:(my + 1) * bb])
        for ga in shards:
            ga.select(val)
    whole = run_ga(sg, train, val, m0, a0, gens, **{k: v for k, v in kw.items() if k != "max_generations"})
    for i, ga in enumerate(shards):
        got = ga.history(gens), ga.status(), ga.masters(), ga.parents()
        assert_same(got, whole, f"shard {i}")
        assert np.array_equal(got[3][0], whole[3][0])
        ga.close()


@pytest.mark.gpu
def test_captured_generation_equals_eager(sg, data):
    import torch
    _, _, _, train, val = data
    m0, a0 = masters(29)
    kw = dict(pop_size=40, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=True, seed=3, patience=2, max_generations=8,
              parents=6)
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
    a = eager.history(7), eager.status(), eager.masters(), eager.parents()
    b = graphed.history(7), graphed.status(), graphed.masters(), graphed.parents()
    assert_same(a, b, "graph")
    assert np.array_equal(a[3][0], b[3][0]) and np.array_equal(a[3][1], b[3][1])
    eager.close()
    graphed.close()


@pytest.mark.gpu
def test_set_parents_refusals(sg, data):
    import torch
    from sgmm_b200 import _lib
    L = _lib.lib()
    _, _, _, train, val = data
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    m0, a0 = masters(1)
    ga = sg.DeviceGA(m0, a0, pop_size=8, sigma=0.05, phi=0.0, fee_rate=0.0, use_arl=True, seed=1, max_generations=3)

    def setp(mu, w=None):
        arr = None if w is None else np.ascontiguousarray(w, np.float32)
        return L.sgmm_ga_set_parents(ga._h, mu, None if arr is None else arr.ctypes.data, stream)
    for mu, w in ((0, None), (-1, None), (9, None), (1025, None), (2, [1.0, -1.0]), (2, [0.0, 0.0]), (2, [np.nan, 1.0]),
                  (2, [np.inf, 1.0]), (1, [-0.5])):
        assert setp(mu, w) == _lib.ERR_INVALID, (mu, w)
    assert L.sgmm_ga_set_parents(None, 2, None, stream) == _lib.ERR_INVALID
    assert setp(3) == 0 and setp(2, [1.0, 0.0]) == 0                # a second call before the first generation is fine
    ga.n_parents = 2
    ga.generation(train, val)
    assert setp(2) == _lib.ERR_INVALID
    assert "already" in L.sgmm_last_error().decode()
    pm, pa = ga.parents()
    assert pm[0] == ga.status()["last_best_index"]
    one = np.zeros(1, np.int64)
    assert L.sgmm_ga_parents_host(ga._h, 1, one.ctypes.data, None, stream) == 0 and one[0] == pm[0]
    assert L.sgmm_ga_run_parents_host(ga._h, 1, 1, one.ctypes.data, None, stream) == _lib.ERR_INVALID
    assert L.sgmm_ga_run_parents_host(ga._h, 0, -1, one.ctypes.data, None, stream) == _lib.ERR_INVALID
    ga.close()
    # evaluate alone also closes the window; a sweep takes one setting for all runs and refuses the run-less read-back
    ga = sg.DeviceGA(m0, a0, pop_size=8, sigma=0.05, phi=0.0, fee_rate=0.0, use_arl=True, seed=1, max_generations=3)
    ga.evaluate(train)
    assert setp(2) == _lib.ERR_INVALID
    ga.close()
    sw = sg.DeviceGASweep(np.stack([m0, m0]), np.stack([a0, a0]), runs=[dict(seed=1, phi=0.0), dict(seed=2, phi=0.0)],
                          pop_size=8, use_arl=True, max_generations=2, parents=3)
    sw.generation(train, val)
    assert L.sgmm_ga_parents_host(sw._h, 1, one.ctypes.data, None, stream) == _lib.ERR_INVALID
    assert sw.parents(1)[0].shape == (3,)
    sw.close()


@pytest.mark.gpu
def test_drl_engine_parents_equal_their_device_compositions(sg, data, tmp_path):
    import torch
    tb, vb, stats, train, val = data
    gens, mu, pop = 7, 4, 20
    w = weights_of("logrank", mu)
    torch.manual_seed(5)
    eng = sg.DRLEngine(pop_size=pop, phi=1e-4, tick_size=0.001, use_arl=True, patience=2, seed=99, parents=mu,
                       parent_weights=w, save_dir=str(tmp_path / "e"))
    m0 = eng.mm_evolver.master_policy.get_weights().clone()
    a0 = eng.adv_evolver.master_policy.get_weights().clone()
    policy, hist = eng.train(tb, vb, stats, generations=gens, log_every=3, verbose=False)
    ref = run_ga(sg, train, val, m0, a0, gens, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=True, seed=99,
                 patience=2, parents=mu, weights=w)
    h, st, (mm, adv, best), _ = ref
    assert np.array_equal(bits64(hist["val_f"]), bits64(h["val_f"]))
    assert np.array_equal(bits64(hist["train_f"]), bits64(h["train_f"]))
    assert np.array_equal(bits32(policy.get_weights().numpy()), bits32(best))          # the recombined best-on-validation
    assert np.array_equal(bits32(eng.adv_evolver.master_policy.get_weights().numpy()), bits32(adv))
    eng2 = sg.DRLEngine(pop_size=pop, phi=1e-4, tick_size=0.001, use_arl=True, patience=2, parents=mu, parent_weights=w,
                        save_dir=str(tmp_path / "s"))
    eng2.mm_evolver.master_policy.set_weights(m0)
    eng2.adv_evolver.master_policy.set_weights(a0)
    out = eng2.train_sweep(tb, vb, stats, gens, phis=[1e-4, 0.01], seeds=[5, 6], log_every=3, verbose=False)
    sw = sg.DeviceGASweep(m0, a0, runs=[dict(seed=5, phi=1e-4, patience=2), dict(seed=6, phi=0.01, patience=2)],
                          pop_size=pop, use_arl=True, max_generations=gens, parents=mu, weights=w)
    for _ in range(gens):
        sw.generation(train, val)
    for r in range(2):
        p, hh = out[r]
        hs, ss = sw.history(r, gens), sw.status(r)
        assert np.array_equal(bits64(hh["val_f"]), bits64(hs["val_f"]))
        _, _, b = sw.masters(r)
        assert np.array_equal(bits32(p.get_weights().numpy()), bits32(b if ss["best_val"] > -np.inf else sw.masters(r)[0]))
    sw.close()
