"""Natural-gradient evolution strategy (sgmm_ga_set_es, DeviceGA / DeviceGASweep / DRLEngine ``es_lr``).

The definition (include/sgmm.h) is restated below in numpy binary32, one rounding per operation:
``utilities`` -- centered ranks of the truncation-selection order (NaN first, then descending fitness, the adversary's
ascending, ties to the lower index, -0.0 == +0.0) --, ``es_sum`` -- index order in segments of 256 children, an exact
binary32 fma chain inside a segment, a pairwise tree over the segments --, ``es_grad`` and ``adam``.  Every child's noise
comes from the CPU oracle (``oracle.mutate`` of a zero master with sigma 1 is the noise itself).  The CPU tests check
this restatement against a literal comparator sort, a float64 sum and a scalar restatement of Adam on Python floats;
the GPU tests hold the device to it bit for bit."""
import ctypes as C
import ctypes.util
import functools
import math
import os
import struct
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

FLIP = 0x8000000000000000
SEGMENT = 256
B1, B2, EPS = np.float32(0.9), np.float32(0.999), np.float32(1e-8)
ONE = np.float32(1.0)


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


def bits32(a):
    return np.asarray(a, np.float32).view(np.uint32)


# ------------------------------------------------------------------------------------------------ the definition
def rank_order(f, sign=1):
    """Children in rank order: NaN first, then descending sign*f, then ascending index."""
    f = np.asarray(f, np.float64)
    v = sign * f
    nan = np.isnan(v)
    key = np.where(nan, 0.0, -v) + 0.0                            # + 0.0: -0.0 -> +0.0
    return np.lexsort((np.arange(f.size), key, ~nan))


def ranks(f, sign=1):
    order = rank_order(f, sign)
    r = np.empty(order.size, np.int64)
    r[order] = np.arange(order.size)
    return r


def utilities(f, sign=1):
    """u_i = fl(fl((float)(lambda-1-r_i) / (float)(lambda-1)) - 0.5f), float32[lambda] in index order."""
    lam = np.asarray(f).size
    if lam < 2:
        raise ValueError("centered ranks need lambda >= 2")
    r = ranks(f, sign)
    return ((lam - 1 - r).astype(np.float32) / np.float32(lam - 1) - np.float32(0.5)).astype(np.float32)


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


def noise_rows(G, seed, generation, n, start=0):
    """eps of children start .. n-1 as float32[n - start, G]: the oracle's child of a zero master with sigma 1
    (0 + eps*1 == eps).  The oracle releases the GIL inside its C call, so the rows are drawn on a thread pool."""
    from oracle import oracle as orc
    z = np.zeros(G, np.float32)
    with ThreadPoolExecutor(max_workers=max(1, min(16, os.cpu_count() or 1))) as ex:
        return np.stack(list(ex.map(lambda i: orc.mutate(z, 1.0, seed, generation, i), range(start, n))))


def es_sum(u, eps):
    """sum_i u_i eps_i: segments of 256 children in index order (u*eps, then fmaf(u, eps, acc)), then a pairwise tree."""
    u = np.asarray(u, np.float32)
    segs = []
    for s0 in range(0, u.size, SEGMENT):
        acc = (u[s0] * eps[s0]).astype(np.float32)
        for i in range(s0 + 1, min(u.size, s0 + SEGMENT)):
            acc = fmaf(u[i], eps[i], acc)
        segs.append(acc)
    while len(segs) > 1:
        nxt = [(segs[k] + segs[k + 1]).astype(np.float32) for k in range(0, len(segs) - 1, 2)]
        if len(segs) % 2:
            nxt.append(segs[-1])
        segs = nxt
    return segs[0]


def es_grad(S, lam, sigma):
    """g = fl(S * fl(1 / fl((float)lambda * sigma)))"""
    return (S * (ONE / (np.float32(lam) * np.float32(sigma)))).astype(np.float32)


def adam(theta, m, v, p1, p2, g, lr):
    """One Adam ascent step; p1, p2 are this step's powers (already multiplied by b1, b2).  Returns (theta, m, v)."""
    m = (B1 * m + (ONE - B1) * g).astype(np.float32)
    v = (B2 * v + (ONE - B2) * (g * g)).astype(np.float32)
    mh = m / (ONE - p1)
    vh = v / (ONE - p2)
    theta = (theta + np.float32(lr) * (mh / (np.sqrt(vh) + EPS))).astype(np.float32)
    return theta, m, v


class ESRef:
    """The evolution strategy's state of one run (both masters' moments and the shared powers) and its update."""

    def __init__(self, lr, G, use_arl):
        self.lr, self.use_arl = np.float32(lr), use_arl
        self.m, self.v = np.zeros(G, np.float32), np.zeros(G, np.float32)
        self.am, self.av = np.zeros(1250, np.float32), np.zeros(1250, np.float32)
        self.p1, self.p2 = ONE, ONE

    def step(self, fit, master, adv_master, sigma, adv_sigma, seed, generation):
        """New (master, adv_master) and the step's {utilities, grad, adv_utilities, adv_grad} from the run's fitness."""
        lam = np.asarray(fit).size
        self.p1, self.p2 = np.float32(self.p1 * B1), np.float32(self.p2 * B2)
        u = utilities(fit, 1)
        g = es_grad(es_sum(u, noise_rows(master.size, seed, generation, lam)), lam, sigma)
        master, self.m, self.v = adam(master, self.m, self.v, self.p1, self.p2, g, self.lr)
        out = {"utilities": u, "grad": g, "adv_utilities": np.zeros(lam, np.float32), "adv_grad": np.zeros(1250, np.float32)}
        if self.use_arl:
            au = utilities(fit, -1)
            ag = es_grad(es_sum(au, noise_rows(1250, seed ^ FLIP, generation, lam)), lam, adv_sigma)
            adv_master, self.am, self.av = adam(adv_master, self.am, self.av, self.p1, self.p2, ag, self.lr)
            out.update(adv_utilities=au, adv_grad=ag)
        return master, adv_master, out


PALETTE = np.array([-50.0, -50.0, -50.0, 0.0, -0.0, np.inf, -np.inf, np.nan, 1.5, 1.5, 2.0, -3.0, 1e-300, -1e-300])


def crafted(n, kind, seed=0):
    rng = np.random.default_rng(seed + n)
    if kind == "palette":                                         # ties everywhere, NaN, +-inf, +-0.0
        return PALETTE[rng.integers(0, PALETTE.size, n)]
    if kind == "plateau":                                         # every child at the no-trade penalty
        return np.full(n, -50.0)
    if kind == "borders":                                         # ties that straddle every segment border
        f = rng.standard_normal(n)
        for b in range(SEGMENT, n + SEGMENT, SEGMENT):
            f[max(0, b - 3):min(n, b + 3)] = [np.nan, -0.0, 0.0, 0.0, 7.0, np.nan][:min(n, b + 3) - max(0, b - 3)]
        return f
    return rng.standard_normal(n)


KINDS = ("palette", "plateau", "borders", "normal")


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("n", [2, 3, 255, 256, 257, 4097])
@pytest.mark.parametrize("kind", KINDS)
def test_ranks_are_a_literal_comparator_sort(n, kind):
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
        r = ranks(f, sign)
        assert [int(x) for x in np.argsort(r)] == literal, (kind, n, sign)
        u = utilities(f, sign)
        for i in (literal[0], literal[-1], literal[n // 2]):   # u = fl(fl((n-1-r)/(n-1)) - 0.5) on Python floats
            ref = fl(fl(float(n - 1 - r[i]) / float(n - 1)) - 0.5)
            assert bits32(u[i]) == bits32(ref)
        assert u[literal[0]] == 0.5 and u[literal[-1]] == -0.5


def test_utility_details():
    f = np.array([1.0, np.nan, 2.0, np.nan, -0.0, 0.0, 2.0])
    assert ranks(f).tolist() == [4, 0, 2, 1, 5, 6, 3]
    assert ranks(f, -1).tolist() == [4, 0, 5, 1, 2, 3, 6]
    assert utilities([3.0, 3.0]).tolist() == [0.5, -0.5]
    with pytest.raises(ValueError):
        utilities([1.0])


def fl(x):
    """round a Python float (binary64) to binary32"""
    return struct.unpack("f", struct.pack("f", x))[0]


@pytest.mark.parametrize("lam", [2, 257, 4097])
def test_es_sum_is_within_its_rounding_bound_of_a_float64_sum(lam):
    rng = np.random.default_rng(lam)
    G = 333
    eps = rng.standard_normal((lam, G)).astype(np.float32)
    u = utilities(rng.standard_normal(lam))
    S = es_sum(u, eps)
    exact = (u.astype(np.float64)[:, None] * eps.astype(np.float64)).sum(0)
    mag = np.abs(u.astype(np.float64)[:, None] * eps.astype(np.float64)).sum(0)
    depth = math.ceil(math.log2(max(1, -(-lam // SEGMENT))))
    n = min(lam, SEGMENT) + depth                                  # roundings on any product's path to the sum
    assert np.all(np.abs(S.astype(np.float64) - exact) <= n * 2.0 ** -24 / (1 - n * 2.0 ** -24) * mag)
    # the fma chain keeps every product exact: a segment of one child is that child's product, rounded once
    assert np.array_equal(bits32(es_sum(u[:1], eps[:1])), bits32(u[0] * eps[0]))


def test_es_sum_tree_order():
    """the tree's order: segments s0..s4 combine as ((s0+s1)+(s2+s3))+s4, an odd last segment moving up unchanged"""
    lam = 4 * SEGMENT + 1
    eps = np.zeros((lam, 1), np.float32)
    u = np.zeros(lam, np.float32)
    vals = np.float32([1.0, 2.0 ** -24, 2.0 ** -24, 2.0 ** -24, 2.0 ** -22])   # one child per segment carries a value
    for s, x in enumerate(vals):
        u[s * SEGMENT], eps[s * SEGMENT, 0] = 1.0, x
    got = es_sum(u, eps)[0]
    assert got == np.float32(1.0 + 3 * 2.0 ** -23)                 # ((1 + 2^-24) + (2^-24 + 2^-24)) + 2^-22
    seq = vals[0]
    for x in vals[1:]:
        seq = np.float32(seq + x)
    assert seq == np.float32(1.0 + 2.0 ** -22)                     # left to right the three 2^-24 vanish


def test_adam_is_a_scalar_binary32_restatement():
    rng = np.random.default_rng(2)
    n = 3000
    theta = rng.standard_normal(n).astype(np.float32)
    m = (rng.standard_normal(n) * 1e-2).astype(np.float32)
    v = np.abs(rng.standard_normal(n) * 1e-4).astype(np.float32)
    g = (rng.standard_normal(n) * 10.0 ** rng.integers(-6, 3, n)).astype(np.float32)
    g[:5] = [0.0, -0.0, 1e-30, -1e-38, 3e4]
    p1, p2 = ONE, ONE
    for step in range(3):
        p1, p2 = np.float32(p1 * B1), np.float32(p2 * B2)
        lr = 0.01
        nt, nm, nv = adam(theta, m, v, p1, p2, g, lr)
        for i in range(n):                                         # Python floats, fl() after every operation
            b1, b2, e = float(B1), float(B2), float(EPS)
            mi = fl(fl(b1 * float(m[i])) + fl(fl(1.0 - b1) * float(g[i])))
            vi = fl(fl(b2 * float(v[i])) + fl(fl(1.0 - b2) * fl(float(g[i]) * float(g[i]))))
            mh = fl(mi / fl(1.0 - float(p1)))
            vh = fl(vi / fl(1.0 - float(p2)))
            ti = fl(float(theta[i]) + fl(fl(lr) * fl(mh / fl(fl(math.sqrt(vh)) + e))))
            assert (bits32(nm[i]), bits32(nv[i]), bits32(nt[i])) == (bits32(mi), bits32(vi), bits32(ti)), (step, i)
        theta, m, v = nt, nm, nv
    assert float(p1) == fl(fl(fl(0.9) * fl(0.9)) * fl(0.9))


def test_fmaf_is_libm_fmaf():
    libm = C.CDLL(ctypes.util.find_library("m"))
    libm.fmaf.restype = C.c_float
    libm.fmaf.argtypes = [C.c_float, C.c_float, C.c_float]
    rng = np.random.default_rng(12)
    n = 20000
    a = (rng.standard_normal(n) * 2.0 ** rng.integers(-30, 30, n)).astype(np.float32)
    b = rng.standard_normal(n).astype(np.float32)
    c = (rng.standard_normal(n) * 2.0 ** rng.integers(-40, 20, n)).astype(np.float32)
    k, j = rng.integers(1, 2 ** 11, n), rng.integers(1, 2 ** 11, n)
    a2, b2 = (1.0 + k * 2.0 ** -12).astype(np.float32), (1.0 + j * 2.0 ** -12).astype(np.float32)
    c2 = (rng.choice([-1.0, 0.0, 1.0], n) * 2.0 ** -60).astype(np.float32)
    for x, y, z in ((a, b, c), (a2, b2, c2), (a, b, -(a * b))):
        ref = np.array([libm.fmaf(float(p), float(q), float(r)) for p, q, r in zip(x, y, z)], np.float32)
        assert np.array_equal(bits32(fmaf(x, y, z)), bits32(ref))


def test_python_argument_errors_before_any_device_call(tmp_path):
    import sgmm_b200
    kw = dict(sigma=0.05, phi=0.0, fee_rate=0.0, use_arl=False, seed=1, max_generations=2)
    m = np.zeros(1250, np.float32)
    bad = [dict(pop_size=8, es_lr=0.0), dict(pop_size=8, es_lr=-1e-3), dict(pop_size=8, es_lr=float("nan")),
           dict(pop_size=8, es_lr=float("inf")), dict(pop_size=8, es_lr=1e-50), dict(pop_size=8, es_lr=True),
           dict(pop_size=8, es_lr="0.01"), dict(pop_size=1, es_lr=0.01), dict(pop_size=8, es_lr=0.01, parents=2),
           dict(pop_size=8, es_lr=0.01, weights=[1.0]), dict(pop_size=8, es_lr=0.01, parents=2, weights=[1.0, 0.0])]
    for b in bad:
        with pytest.raises(ValueError):
            sgmm_b200.DeviceGA(m, **kw, **b)
        with pytest.raises(ValueError):
            sgmm_b200.DeviceGASweep(m, runs=[dict(seed=1, phi=0.0)], use_arl=False, max_generations=2, **b)
    for b in (dict(pop_size=8, es_lr=0.0), dict(pop_size=1, es_lr=0.01), dict(pop_size=8, es_lr=0.01, parents=2),
              dict(pop_size=8, es_lr=0.01, parent_weights=[1.0])):
        with pytest.raises(ValueError):
            sgmm_b200.DRLEngine(save_dir=str(tmp_path / "never"), **b)
    assert not (tmp_path / "never").exists()


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


def write_fitness(ga, f):
    import torch
    from sgmm_b200.dist import device_tensor
    fp, tp, *_ = ga.buffers()
    device_tensor(fp, f.size, torch.float64, ga.device).copy_(torch.from_numpy(np.ascontiguousarray(f, np.float64)))
    device_tensor(tp, f.size, torch.int32, ga.device).copy_(torch.arange(f.size, dtype=torch.int32))


def read_fitness(ga, n):
    import torch
    from sgmm_b200.dist import device_tensor
    fp, *_ = ga.buffers()
    torch.cuda.synchronize()
    return device_tensor(fp, n, torch.float64, ga.device).cpu().numpy().copy()


LR = 0.02


@pytest.mark.gpu
@pytest.mark.parametrize("lam", [2, 50, 257, 4097, 65536])
def test_crafted_fitness_one_generation(sg, data, lam):
    _, _, _, _, val = data
    sigma, seed = 0.05, 4321
    m0, a0 = masters(lam)
    exact = lam <= 4097
    if exact:
        eps, aeps = noise_rows(m0.size, seed, 0, lam), noise_rows(1250, seed ^ FLIP, 0, lam)
    grads = []
    for kind in KINDS:
        f = crafted(lam, kind, seed=7)
        ga = sg.DeviceGA(m0, a0, pop_size=lam, sigma=sigma, phi=1e-4, fee_rate=0.0, use_arl=True, seed=seed,
                         max_generations=1, es_lr=LR)
        write_fitness(ga, f)
        ga.select(val)
        es = ga.es_state()
        u, au = utilities(f, 1), utilities(f, -1)
        assert np.array_equal(bits32(es["utilities"]), bits32(u)), kind
        assert np.array_equal(bits32(es["adv_utilities"]), bits32(au)), kind
        st, h = ga.status(), ga.history()
        best = rank_order(f, 1)[0]
        assert st["last_best_index"] == best and h["train_trades"][0] == best
        assert bits64(h["train_f"][0]) == bits64(f[best])
        mm, adv, _ = ga.masters()
        if exact:
            g, ag = es_grad(es_sum(u, eps), lam, sigma), es_grad(es_sum(au, aeps), lam, sigma)
            assert np.array_equal(bits32(es["grad"]), bits32(g)), kind
            assert np.array_equal(bits32(es["adv_grad"]), bits32(ag)), kind
            z = np.zeros_like
            assert np.array_equal(bits32(mm), bits32(adam(m0, z(m0), z(m0), B1, B2, g, LR)[0])), kind
            assert np.array_equal(bits32(adv), bits32(adam(a0, z(a0), z(a0), B1, B2, ag, LR)[0])), kind
        elif kind == "normal":
            grads.append((es["grad"], es["adv_grad"]))
            again = sg.DeviceGA(m0, a0, pop_size=lam, sigma=sigma, phi=1e-4, fee_rate=0.0, use_arl=True, seed=seed,
                                max_generations=1, es_lr=LR)
            write_fitness(again, f)
            again.select(val)
            e2 = again.es_state()
            assert np.array_equal(bits32(e2["grad"]), bits32(es["grad"]))
            assert np.array_equal(bits32(e2["adv_grad"]), bits32(es["adv_grad"]))
            assert np.array_equal(bits32(again.masters()[0]), bits32(mm))
            again.close()
            # against a float64 sum: every product is exact in binary64, at most 256 chained + 8 tree roundings
            S64 = np.zeros(m0.size)
            A64 = np.zeros(m0.size)
            for c0 in range(0, lam, 4096):
                e = noise_rows(m0.size, seed, 0, min(lam, c0 + 4096), start=c0)
                p = u[c0:c0 + e.shape[0]].astype(np.float64)[:, None] * e.astype(np.float64)
                S64 += p.sum(0)
                A64 += np.abs(p).sum(0)
            scale = 1.0 / (np.float64(np.float32(lam) * np.float32(sigma)))
            n = SEGMENT + 8 + 3
            bound = n * 2.0 ** -24 / (1 - n * 2.0 ** -24) * A64 * scale + np.spacing(np.abs(es["grad"])).astype(np.float64)
            assert np.all(np.abs(es["grad"].astype(np.float64) - S64 * scale) <= bound)
        ga.close()


def run_ga(sg, train, val, m, a, gens, **kw):
    ga = sg.DeviceGA(m, a, max_generations=gens, **kw)
    for _ in range(gens):
        ga.generation(train, val)
    out = ga.history(gens), ga.status(), ga.masters(), ga.es_state()
    ga.close()
    return out


def assert_same(x, y, what=""):
    (hx, sx, mx, ex), (hy, sy, my, ey) = x, y
    for k in hx:
        assert np.array_equal(hx[k].view(np.uint8), hy[k].view(np.uint8)), (what, k)
    assert sx == sy, (what, sx, sy)
    for p, q, name in zip(mx, my, ("mm", "adv", "best")):
        assert np.array_equal(bits32(p), bits32(q)), (what, name)
    for k in ex:
        assert np.array_equal(bits32(ex[k]), bits32(ey[k])), (what, k)


def oracle_ga(orc, tz, vz, master, adv_master, *, pop, lr, sigma, phi, tick, fee, use_arl, seed, gens, patience,
              hidden=32):
    """The GA composed from oracle rollouts and the ES reference (drl_engine.py's loop with the ES update)."""
    master = master.copy()
    adv_master = None if adv_master is None else adv_master.copy()
    ref = ESRef(lr, master.size, use_arl)
    s_mm = s_adv = np.float32(sigma)
    best_val, stale, best_master = -np.inf, 0, master.copy()
    hist = {k: [] for k in ("train_f", "val_f", "train_trades", "val_trades", "sigma")}
    last, best = None, None
    for gen in range(gens):
        fit, trd = orc.rollout_population(tz, phi, tick, fee, master=master, sigma=float(s_mm), adv_master=adv_master,
                                          adv_sigma=float(s_adv), use_adv=use_arl, seed=seed, generation=gen, count=pop,
                                          hidden=hidden, nthreads=4)
        best = rank_order(fit, 1)[0]
        master, new_adv, last = ref.step(fit, master, adv_master, s_mm, s_adv, seed, gen)
        if use_arl:
            adv_master = new_adv
        vf, vt = orc.rollout(master, None, vz, phi, tick, fee, hidden=hidden)
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
    return hist, master, adv_master, best_master, best_val, s_mm, last, best


def check_against_oracle(got, ref, use_arl):
    h, st, (m, a, b), es = got
    ho, m_o, a_o, b_o, bv_o, s_o, es_o, best_o = ref
    assert np.array_equal(bits64(h["train_f"]), bits64(ho["train_f"]))
    assert np.array_equal(bits64(h["val_f"]), bits64(ho["val_f"]))
    assert h["train_trades"].tolist() == ho["train_trades"] and h["val_trades"].tolist() == ho["val_trades"]
    assert np.array_equal(h["sigma"], np.array(ho["sigma"], np.float32))
    assert np.array_equal(bits32(m), bits32(m_o)) and np.array_equal(bits32(b), bits32(b_o))
    assert st["best_val"] == bv_o and st["sigma"] == s_o and st["last_best_index"] == best_o
    for k in ("utilities", "grad") + (("adv_utilities", "adv_grad") if use_arl else ()):
        assert np.array_equal(bits32(es[k]), bits32(es_o[k])), k
    if use_arl:
        assert np.array_equal(bits32(a), bits32(a_o))


@pytest.mark.gpu
@pytest.mark.parametrize("use_arl", [False, True])
def test_ga_matches_oracle_composed_ga(sg, data, use_arl):
    from oracle import oracle as orc
    tb, vb, stats, train, val = data
    tz = orc.normalise(tb, stats) + tb[2:]
    vz = orc.normalise(vb, stats) + vb[2:]
    pop, gens, seed = 24, 8, 61 + int(use_arl)
    m0, a0 = masters(13, use_arl)
    got = run_ga(sg, train, val, m0, a0, gens, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=use_arl,
                 seed=seed, patience=1, es_lr=LR)
    ref = oracle_ga(orc, tz, vz, m0, a0, pop=pop, lr=LR, sigma=0.05, phi=1e-4, tick=0.001, fee=3e-4, use_arl=use_arl,
                    seed=seed, gens=gens, patience=1)
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
    pop, gens = 6, 3
    got = run_ga(sg, train, val, m0, a0, gens, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=True, seed=9,
                 patience=1, es_lr=LR, hidden=256, precision="exact")
    ref = oracle_ga(orc, tz, vz, m0, a0, pop=pop, lr=LR, sigma=0.05, phi=1e-4, tick=0.001, fee=0.0, use_arl=True,
                    seed=9, gens=gens, patience=1, hidden=256)
    check_against_oracle(got, ref, True)


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,precision", [(32, "f16"), (32, "bf16"), (256, "bf16")])
def test_tensor_core_ga_takes_the_reference_update_of_its_own_fitness(sg, data, hidden, precision):
    _, _, _, train, val = data
    m0, a0 = masters(19, True, hidden=hidden)
    pop, gens, seed = 40, 4, 8
    ga = sg.DeviceGA(m0, a0, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=True, seed=seed, patience=1,
                     hidden=hidden, precision=precision, max_generations=gens, es_lr=LR)
    ref = ESRef(LR, m0.size, True)
    m, a = m0.copy(), a0.copy()
    for gen in range(gens):
        ga.evaluate(train)
        f = read_fitness(ga, pop)
        st = ga.status()
        m, a, out = ref.step(f, m, a, np.float32(st["sigma"]), np.float32(st["adv_sigma"]), seed, gen)
        ga.select(val)
        gm, ga_, _ = ga.masters()
        assert np.array_equal(bits32(gm), bits32(m)), gen
        assert np.array_equal(bits32(ga_), bits32(a)), gen
        es = ga.es_state()
        for k in out:
            assert np.array_equal(bits32(es[k]), bits32(out[k])), (gen, k)
    ga.close()


@pytest.mark.gpu
def test_sweep_runs_equal_their_solo_gas(sg, data):
    _, _, _, train, val = data
    runs = [dict(seed=11, phi=0.0, fee_rate=0.0, sigma=0.05, patience=1),
            dict(seed=12, phi=1e-4, fee_rate=3e-4, sigma=0.02, patience=2),
            dict(seed=2 ** 63 + 5, phi=0.01, fee_rate=-1e-4, sigma=0.08, patience=3)]
    K, pop, gens = len(runs), 24, 6
    mm = np.stack([masters(3 + r)[0] for r in range(K)])
    adv = np.stack([masters(3 + r)[1] for r in range(K)])
    ga = sg.DeviceGASweep(mm, adv, runs=runs, pop_size=pop, use_arl=True, max_generations=gens, es_lr=LR)
    for _ in range(gens):
        ga.generation(train, val)
    for r in range(K):
        sweep = ga.history(r, gens), ga.status(r), ga.masters(r), ga.es_state(r)
        solo = run_ga(sg, train, val, mm[r], adv[r], gens, pop_size=pop, use_arl=True, precision="exact", es_lr=LR,
                      **runs[r])
        assert_same(sweep, solo, f"run {r}")
    ga.close()


@pytest.mark.gpu
def test_two_shards_on_one_device_equal_the_unsharded_ga(sg, data):
    import torch
    from sgmm_b200.dist import device_tensor
    _, _, _, train, val = data
    m0, a0 = masters(23)
    pop, gens, stride = 50, 5, 25
    kw = dict(pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=True, seed=77, patience=2, max_generations=gens,
              es_lr=LR)
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
        got = ga.history(gens), ga.status(), ga.masters(), ga.es_state()
        assert_same(got, whole, f"shard {i}")
        ga.close()


@pytest.mark.gpu
def test_captured_generation_equals_eager(sg, data):
    import torch
    _, _, _, train, val = data
    m0, a0 = masters(29)
    kw = dict(pop_size=300, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=True, seed=3, patience=2, max_generations=8,
              es_lr=LR)
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
    a = eager.history(7), eager.status(), eager.masters(), eager.es_state()
    b = graphed.history(7), graphed.status(), graphed.masters(), graphed.es_state()
    assert_same(a, b, "graph")
    eager.close()
    graphed.close()


@pytest.mark.gpu
def test_set_es_refusals(sg, data):
    import torch
    from sgmm_b200 import _lib
    L = _lib.lib()
    _, _, _, train, val = data
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    m0, a0 = masters(1)
    kw = dict(sigma=0.05, phi=0.0, fee_rate=0.0, use_arl=True, seed=1, max_generations=3)
    ga = sg.DeviceGA(m0, a0, pop_size=8, **kw)
    u = np.zeros(8, np.float32)
    assert L.sgmm_ga_run_es_host(ga._h, 0, u.ctypes.data, None, None, None, stream) == _lib.ERR_INVALID   # no ES set
    for lr in (0.0, -0.01, float("nan"), float("inf"), float("-inf")):
        assert L.sgmm_ga_set_es(ga._h, lr, stream) == _lib.ERR_INVALID, lr
    assert L.sgmm_ga_set_es(None, 0.01, stream) == _lib.ERR_INVALID
    assert L.sgmm_ga_set_es(ga._h, 0.5, stream) == 0 and L.sgmm_ga_set_es(ga._h, LR, stream) == 0   # again before a generation
    assert L.sgmm_ga_set_parents(ga._h, 2, None, stream) == _lib.ERR_INVALID                 # ES first, then parents
    assert "exclude" in L.sgmm_last_error().decode()
    assert L.sgmm_ga_run_es_host(ga._h, 0, u.ctypes.data, None, None, None, stream) == 0 and not u.any()
    ga.generation(train, val)
    assert L.sgmm_ga_set_es(ga._h, LR, stream) == _lib.ERR_INVALID
    assert "already" in L.sgmm_last_error().decode()
    es = ga.es_state()
    assert L.sgmm_ga_es_host(ga._h, u.ctypes.data, None, None, None, stream) == 0
    assert np.array_equal(u, es["utilities"]) and sorted(u.tolist()) == sorted(utilities(np.arange(8.0)).tolist())
    assert L.sgmm_ga_run_es_host(ga._h, 1, u.ctypes.data, None, None, None, stream) == _lib.ERR_INVALID
    assert L.sgmm_ga_run_es_host(ga._h, -1, u.ctypes.data, None, None, None, stream) == _lib.ERR_INVALID
    assert L.sgmm_ga_run_es_host(ga._h, 0, None, None, None, None, stream) == 0
    ga.close()
    ga = sg.DeviceGA(m0, a0, pop_size=8, parents=2, **kw)                 # parents first, then the ES
    assert L.sgmm_ga_set_es(ga._h, LR, stream) == _lib.ERR_INVALID
    ga.close()
    ga = sg.DeviceGA(m0, a0, pop_size=8, **kw)                            # evaluate alone closes the window too
    ga.evaluate(train)
    assert L.sgmm_ga_set_es(ga._h, LR, stream) == _lib.ERR_INVALID
    ga.close()
    one = sg.DeviceGA(m0, a0, pop_size=1, **kw)                           # lambda < 2
    assert L.sgmm_ga_set_es(one._h, LR, stream) == _lib.ERR_INVALID
    one.close()
    sw = sg.DeviceGASweep(np.stack([m0, m0]), np.stack([a0, a0]), runs=[dict(seed=1, phi=0.0), dict(seed=2, phi=0.0)],
                          pop_size=8, use_arl=True, max_generations=2, es_lr=LR)
    sw.generation(train, val)
    assert L.sgmm_ga_es_host(sw._h, u.ctypes.data, None, None, None, stream) == _lib.ERR_INVALID
    assert sw.es_state(1)["utilities"].shape == (8,) and sw.es_state(1)["adv_grad"].any()
    sw.close()
    sw = sg.DeviceGASweep(m0, None, runs=[dict(seed=1, phi=0.0)], pop_size=1, use_arl=False, max_generations=2)
    assert L.sgmm_ga_set_es(sw._h, LR, stream) == _lib.ERR_INVALID
    sw.close()


@pytest.mark.gpu
def test_drl_engine_es_equals_its_device_compositions(sg, data, tmp_path):
    import torch
    tb, vb, stats, train, val = data
    gens, pop = 7, 20
    torch.manual_seed(5)
    eng = sg.DRLEngine(pop_size=pop, phi=1e-4, tick_size=0.001, use_arl=True, patience=2, seed=99, es_lr=LR,
                       save_dir=str(tmp_path / "e"))
    m0 = eng.mm_evolver.master_policy.get_weights().clone()
    a0 = eng.adv_evolver.master_policy.get_weights().clone()
    policy, hist = eng.train(tb, vb, stats, generations=gens, log_every=3, verbose=False)
    h, st, (mm, adv, best), _ = run_ga(sg, train, val, m0, a0, gens, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=0.0,
                                       use_arl=True, seed=99, patience=2, es_lr=LR)
    assert np.array_equal(bits64(hist["val_f"]), bits64(h["val_f"]))
    assert np.array_equal(bits64(hist["train_f"]), bits64(h["train_f"]))
    assert hist["train_trades"] == h["train_trades"].tolist()
    assert st["best_val"] > -np.inf
    assert np.array_equal(bits32(policy.get_weights().numpy()), bits32(best))          # the best-on-validation master
    assert np.array_equal(bits32(eng.adv_evolver.master_policy.get_weights().numpy()), bits32(adv))
    ck = torch.load(str(tmp_path / "e" / "agent_best_val_0.0001.pth"))
    snap = sg.TradingPolicy(hidden_dim=32)
    snap.load_state_dict(ck)
    assert np.array_equal(bits32(snap.get_weights().numpy()), bits32(best))           # the checkpoint
    eng2 = sg.DRLEngine(pop_size=pop, phi=1e-4, tick_size=0.001, use_arl=True, patience=2, es_lr=LR,
                        save_dir=str(tmp_path / "s"))
    eng2.mm_evolver.master_policy.set_weights(m0)
    eng2.adv_evolver.master_policy.set_weights(a0)
    out = eng2.train_sweep(tb, vb, stats, gens, phis=[1e-4, 0.01], seeds=[5, 6], log_every=3, verbose=False)
    sw = sg.DeviceGASweep(m0, a0, runs=[dict(seed=5, phi=1e-4, patience=2), dict(seed=6, phi=0.01, patience=2)],
                          pop_size=pop, use_arl=True, max_generations=gens, es_lr=LR)
    for _ in range(gens):
        sw.generation(train, val)
    for r, phi in enumerate((1e-4, 0.01)):
        p, hh = out[r]
        hs, ss = sw.history(r, gens), sw.status(r)
        assert np.array_equal(bits64(hh["val_f"]), bits64(hs["val_f"]))
        mm_r, _, b = sw.masters(r)
        want = b if ss["best_val"] > -np.inf else mm_r
        assert np.array_equal(bits32(p.get_weights().numpy()), bits32(want))
        if ss["best_val"] > -np.inf:
            snap.load_state_dict(torch.load(str(tmp_path / "s" / f"agent_run{r}_best_val_{phi}.pth")))
            assert np.array_equal(bits32(snap.get_weights().numpy()), bits32(b))
    sw.close()
