"""The tensor-core routes at the shapes the benchmark and the GA run: policy outputs against a float64 reference for EVERY
individual, bar and inventory.

tc32_kernel walks groups of individuals in a persistent loop (sgmm_tc32.cu): a CTA's second and later groups restage
B1 / B2 / B3 and the adversary table and carry the pipeline phases (gt, gc) over from the group before.  spec256_kernel
walks individuals the same way (sgmm_spec256.cu: gt, W2 restaged per individual).  Teacher-forced replay cannot see a
wrong policy there: a group that ran on stale weights, or a late chunk that read the wrong A1 tile, takes wrong offsets
and the env still replays them bit for bit.  So every case here compares the audit table with the reference row by row,
at P = 4096 x T = 14 400 (the tensor_core_h32 workload: a second group on every CTA), at group 2 with an odd length
(3-4 groups per CTA, a partial last group, chunk counts that are no multiple of the A1 ring or of the TMEM buffers),
and at H = 256 with 4-5 individuals per CTA and T = 28 800 (config 4).  Checks of each case:

  outputs      |raw*5 - ref*5| <= TAU for every (individual, bar, inventory, side), all finite, and the rounded offset
               equals the reference's wherever the reference is more than TAU + 1e-3 tick from a rounding boundary;
  production   rollout_population returns the audit's fitness and trades bit for bit;
  offsets      every offset the kernel took is one of the five rounded outputs of its bar, for every individual;
  boundaries   for individuals at group and grid boundaries (and a spread): teacher-forced replay of the oracle's env bit
               for bit, the offsets along the replayed inventory path are the rounded outputs of those rows, and the
               closed loop equals the fp32 oracle's up to its first near-tie.

The CPU tests (no marker) pin the reference to the oracle and show that every case can see the mix-ups it targets:
the individuals a scheduling bug would confuse, and the bars a stale chunk would supply, differ by more than 2 TAU on
almost every row, so such a mix-up shows as an error above TAU.
"""
import functools
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

# stated tolerances on raw*5 (ticks), as in tests/test_gpu_tc32.py and tests/test_gpu_spec256.py, except BF16 at H = 32:
# over 5.9e8 outputs per population the bf16 rounding of W2, A2 and A3 alone reaches 0.19 tick (a bf16-operand emulation
# of the same layers gives the kernel's worst outputs to 5e-5 tick), above the 0.12 that holds on the small audit shapes;
# DESIGN.md section 3 states 0.25 at population scale
TAU = {"bf16": 0.25, "tf32": 0.03, "f16": 0.03, "spec256": 0.05}
PHI = 1e-4
TICK = 0.001
F32 = np.float32
SPREAD = 16                   # individuals spread over the population, checked next to the boundary ones
SEP_FRACTION = 0.95           # share of rows on which two confusable individuals (or bars) must differ by > 2 TAU

# name -> hidden, precision, fee, adversary, (days, first_day, T), population a*SMs + b, explicit group (0: the library's)
CASES = {
    "tc32-bf16":          (32, "bf16", 0.0, False, (60, 200, None), (0, 4096), 0),
    "tc32-tf32":          (32, "tf32", 0.0, False, (60, 200, None), (0, 4096), 0),
    "tc32-f16":           (32, "f16", 0.0, False, (60, 200, None), (0, 4096), 0),
    "tc32-f16-fee":       (32, "f16", 3e-4, False, (60, 260, None), (0, 4096), 0),
    "tc32-f16-adv-fee":   (32, "f16", 3e-4, True, (60, 260, None), (0, 4096), 0),
    "tc32-bf16-adv-fee":  (32, "bf16", 3e-4, True, (60, 320, None), (0, 4096), 0),
    "tc32-g2-tf32":       (32, "tf32", 0.0, False, (11, 380, 2413), (6, 1), 2),
    "tc32-g2-f16-adv":    (32, "f16", 0.0, True, (11, 400, 2413), (6, 1), 2),
    "spec256":            (256, "bf16", 0.0, False, (120, 420, None), (4, 3), 0),
    "spec256-fee":        (256, "bf16", 3e-4, False, (120, 420, None), (4, 3), 0),
    "spec256-qtab-fee":   (256, "bf16", 3e-4, True, (60, 560, None), (4, 3), 0),
}


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


@pytest.fixture(scope="module")
def sg():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import sgmm_b200
    return sgmm_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


# ----------------------------------------------------------------------------------------------
# the float64 reference and the inputs of the cases
# ----------------------------------------------------------------------------------------------
def policy_ref(genomes, z1, z2, hidden):
    """TradingPolicy (3 -> H -> H -> 2, relu, genome W1[H,3] | b1 | W2[H,H] | b2 | W3[2,H] | b3) in float64 for every bar
    of (z1, z2) and every inventory -2..2 (input inv/2): raw outputs [p, T, 5, 2] on the genomes' device."""
    H = hidden
    g = torch.as_tensor(genomes).to(torch.float64)
    dev, p = g.device, g.shape[0]
    W1, b1 = g[:, :3 * H].reshape(p, H, 3), g[:, 3 * H:4 * H]
    W2, b2 = g[:, 4 * H:4 * H + H * H].reshape(p, H, H), g[:, 4 * H + H * H:5 * H + H * H]
    W3, b3 = g[:, 5 * H + H * H:7 * H + H * H].reshape(p, 2, H), g[:, 7 * H + H * H:]
    z1 = torch.as_tensor(z1).to(dev, torch.float64)
    z2 = torch.as_tensor(z2).to(dev, torch.float64)
    T = z1.shape[0]
    inv2 = (torch.arange(5, dtype=torch.float64, device=dev) - 2) / 2
    x = torch.stack([z1.repeat_interleave(5), z2.repeat_interleave(5), inv2.repeat(T),
                     torch.ones(5 * T, dtype=torch.float64, device=dev)], 1)              # row t*5 + inv+2
    h = torch.matmul(x, torch.cat([W1, b1[:, :, None]], 2).transpose(1, 2)).relu_()       # [p, 5T, H]
    h = torch.baddbmm(b2[:, None, :], h, W2.transpose(1, 2)).relu_()
    return torch.baddbmm(b3[:, None, :], h, W3.transpose(1, 2)).view(p, T, 5, 2)


@functools.lru_cache(maxsize=4)
def _genomes(P, hidden, seed):
    from sgmm_b200 import synthetic
    return synthetic.policy_like_genomes(P, hidden=hidden, seed=seed, out_scale=6.0 if hidden == 32 else 4.0,
                                         out_bias=(0.1, 0.1))


def _adv(P, seed):
    return (np.random.default_rng(seed).standard_normal((P, 1250)) * 0.7).astype(F32)


@functools.lru_cache(maxsize=2)
def _episode(days, first_day, T):
    """(bundle 7-tuple, normalised bundle for the oracle, train stats) of ``days`` synthetic days, cut to ``T`` bars."""
    from oracle import oracle
    from sgmm_b200 import synthetic
    full = synthetic.synthetic_bundle(days, first_day=first_day)
    bundle = full if T is None else tuple(a[:T] for a in full)
    stats = synthetic.train_stats_of(full)
    z1, z2 = oracle.normalise(bundle, stats)
    return bundle, (z1, z2) + tuple(bundle[2:]), stats


def _seed(name):
    return 1000 + list(CASES).index(name)


def _tc32_group(count, sms):
    """tc32_group_size (sgmm_tc32.cu): the even group of at most 16 that minimises waves x group, the larger on a tie."""
    best, best_cost = 2, None
    for g in range(2, 17, 2):
        groups = -(-count // g)
        cost = -(-groups // sms) * g
        if best_cost is None or cost <= best_cost:
            best, best_cost = g, cost
    return best


def _layout(name, sms):
    """Population, group, grid and the individuals a scheduling bug would confuse with their neighbours at ``sms`` SMs:
    (P, G, C, per_cta, boundary individuals, confusable distances)."""
    hidden, _, _, _, _, (a, b), group = CASES[name]
    P = a * sms + b
    if hidden == 32:
        G = group or _tc32_group(P, sms)
        groups = -(-P // G)
        C = min(groups, sms)
        per_cta = -(-groups // C)
        edge = [0, 1, G - 1, G, C * G - 1, C * G, C * G + 1, P - 2, P - 1]
        dists = (1, G, C * G)
    else:
        G, C = 1, min(P, sms)
        per_cta = -(-P // C)
        edge = [0, sms - 1, sms, sms + 1, 2 * sms, P - 1]
        dists = (1, sms)
    spread = np.linspace(0, P - 1, SPREAD + 2).astype(int)[1:-1].tolist()
    return P, G, C, per_cta, sorted(set(edge + spread)), dists


def _separation(genomes, z1, z2, hidden, pairs, lags=()):
    """max |d(ref*5)| over the two outputs of a row (bar, inventory), on a sample of bars: between individuals i and j of
    each of ``pairs``, and between bar t and bar t - lag of each individual i of ``pairs``."""
    bars = np.arange(max(lags, default=0), len(z1), 193)
    out = []
    for i, j in pairs:
        q = policy_ref(genomes[[i, j]], z1[bars], z2[bars], hidden) * 5
        out.append((q[0] - q[1]).abs().amax(-1).flatten())
    for lag in lags:
        for i in {i for i, _ in pairs}:
            q0 = policy_ref(genomes[[i]], z1[bars], z2[bars], hidden) * 5
            q1 = policy_ref(genomes[[i]], z1[bars - lag], z2[bars - lag], hidden) * 5
            out.append((q0 - q1).abs().amax(-1).flatten())
    return torch.cat(out)


def _confusable_pairs(P, edge, dists):
    return [(i, i + s * d) for i in edge for d in dists for s in (-1, 1) if 0 <= i + s * d < P]


# ----------------------------------------------------------------------------------------------
# CPU: the reference is the oracle's policy, and every case can see the mix-ups it targets
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hidden", [32, 256])
def test_reference_agrees_with_the_oracle(hidden):
    from oracle import oracle
    _, bz, _ = _episode(60, 200, None)
    master, kids = _genomes(9, hidden, 7)
    G = np.concatenate([master[None], kids])
    bars = np.concatenate([np.arange(0, 14400, 331), [14399]])
    ref = policy_ref(G, bz[0][bars], bz[1][bars], hidden).numpy()
    worst = 0.0
    for i in range(G.shape[0]):
        for k, t in enumerate(bars):
            for iv in range(5):
                want = oracle.mlp_forward(G[i], [bz[0][t], bz[1][t], (iv - 2) / 2.0], hidden=hidden)
                worst = max(worst, float(np.max(np.abs(want.astype(np.float64) - ref[i, k, iv]))) * 5)
    print(f"H = {hidden}: max |d(raw*5)| between the fp32 oracle and the float64 reference = {worst:.3g} ticks")
    assert worst <= 1e-4
    assert np.abs(ref).max() * 5 > 5                                      # the sample spans several ticks


@pytest.mark.parametrize("sms", [148, 160])
@pytest.mark.parametrize("name", list(CASES))
def test_each_case_separates_what_it_could_confuse(name, sms):
    """At ``sms`` SMs: neighbours at distance 1, group and grid x group (tc32) or SM count (spec256) of every boundary
    individual, and bars t - 25 (the chunk before) and t - 100 (one trip round the A1 ring), differ by more than 2 TAU."""
    hidden, precision, _, _, ep, _, _ = CASES[name]
    tau = TAU["spec256" if hidden == 256 else precision]
    P, _, _, _, edge, dists = _layout(name, sms)
    _, bz, _ = _episode(*ep)
    G = _genomes(P, hidden, _seed(name))[1]
    d = _separation(G, bz[0], bz[1], hidden, _confusable_pairs(P, edge, dists), lags=(25, 100))
    frac = float((d > 2 * tau).double().mean())
    print(f"{name} at {sms} SMs: {frac:.4f} of {d.numel()} rows differ by > 2 TAU")
    assert frac >= SEP_FRACTION


# ----------------------------------------------------------------------------------------------
# GPU: the cases
# ----------------------------------------------------------------------------------------------
def _audit_outputs(g, z1, z2, raw, act, hidden, tau, budget=4 << 30):
    """Every row of ``raw`` [P, T, 5, 2] against the reference, on the device, in chunks of individuals.  Returns the worst
    error with where it is, error counts, the rounding flips (all, and those outside the near-tie margin), the number of
    non-finite outputs and of taken offsets that are none of their bar's five rounded outputs."""
    P, T = raw.shape[:2]
    chunk = max(1, budget // (T * 5 * hidden * 8 * 2))
    st = dict(worst=-1.0, at=None, over_half=0, flips=0, outside=0, nonfinite=0, off_row=0)
    for i0 in range(0, P, chunk):
        i1 = min(P, i0 + chunk)
        q_r = policy_ref(g[i0:i1], z1, z2, hidden) * 5.0
        q_k = raw[i0:i1] * 5.0                      # fp32: the product the kernel rounds (drl_engine.py:39)
        st["nonfinite"] += int((~torch.isfinite(q_k)).sum())
        err = (q_k.double() - q_r).abs()
        m, k = torch.max(err.view(-1), 0)
        if float(m) > st["worst"]:
            i, t, iv, o = (int(x) for x in np.unravel_index(int(k), err.shape))
            st["worst"], st["at"] = float(m), (i0 + i, t, iv - 2, "ab"[o], float(q_k[i, t, iv, o]), float(q_r[i, t, iv, o]))
        st["over_half"] += int((err > tau / 2).sum())
        r_k, r_r = torch.round(q_k).double(), torch.round(q_r)
        flip = r_k != r_r
        margin = (q_r - q_r.floor() - 0.5).abs()
        st["flips"] += int(flip.sum())
        st["outside"] += int((flip & (margin > tau + 1e-3)).sum())
        st["off_row"] += int((~(act[i0:i1, :, None, :].double() == r_k).all(-1).any(-1)).sum())
        del q_r, q_k, err, r_k, r_r, flip, margin
    return st


def _check_individual(orc, bz, fee, hidden, tau, G, A, fit, trd, raw, act, i, closed_loop):
    """Teacher-forced replay and the offsets along its path; with ``closed_loop`` the fp32 oracle's own episode up to
    its first near-tie.  Returns (problems, identical closed loop or None)."""
    a = None if A is None else A[i]
    problems = []
    fo, to, tro = orc.rollout(None, a, bz, PHI, TICK, fee, forced_actions=act, trace=True)
    if bits64(fo) != bits64(fit) or to != trd:
        problems.append(f"individual {i}: teacher-forced ({fo}, {to}) != kernel ({fit}, {trd})")
    T = act.shape[0]
    inv_before = np.concatenate([[0], tro["inventory"][:-1]])
    taken = np.rint(raw[np.arange(T), inv_before + 2] * F32(5)).astype(np.int32)
    if not np.array_equal(taken, act):
        problems.append(f"individual {i}: offsets differ from rint(raw*5) on the path from bar {int(np.argmax((taken != act).any(1)))}")
    if not closed_loop:
        return problems, None
    fo, to, tro = orc.rollout(G[i], a, bz, PHI, TICK, fee, hidden=hidden, trace=True)
    diff = (tro["off_a"] != act[:, 0]) | (tro["off_b"] != act[:, 1])
    if not diff.any():
        if bits64(fo) != bits64(fit) or to != trd:
            problems.append(f"individual {i}: same offsets as the oracle, ({fo}, {to}) != ({fit}, {trd})")
        return problems, True
    t = int(np.argmax(diff))
    q = np.array([tro["raw_a"][t], tro["raw_b"][t]], F32) * F32(5)
    margin = float(np.min(np.abs(np.abs(q - np.floor(q)) - 0.5)))
    if margin > tau:
        problems.append(f"individual {i}: closed loop leaves the oracle at bar {t}, {margin:.4f} tick from a rounding boundary")
    return problems, False


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_outputs_within_tolerance_at_scale(sg, orc, name):
    hidden, precision, fee, use_adv, ep, _, group = CASES[name]
    tau = TAU["spec256" if hidden == 256 else precision]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    P, G_, C, per_cta, edge, dists = _layout(name, sms)
    if hidden == 32 and not group:
        assert P > 16 * sms                 # some CTA runs two groups whatever group size the library picks
    assert per_cta >= 2
    t0 = time.time()
    bundle, bz, stats = _episode(*ep)
    bun = sg.Bundle.from_arrays(bundle, stats, TICK)
    T = bun.T
    G = _genomes(P, hidden, _seed(name))[1]
    A = _adv(P, _seed(name)) if use_adv else None
    g = torch.from_numpy(G).cuda()
    a = None if A is None else torch.from_numpy(A).cuda()
    z1, z2 = (torch.from_numpy(z).cuda() for z in bz[:2])
    sep = _separation(g, z1, z2, hidden, _confusable_pairs(P, edge, dists), lags=(25, 100))
    assert float((sep > 2 * tau).double().mean()) >= SEP_FRACTION      # a mix-up of this shape shows as an error > TAU

    fit, trd, raw, act = sg.rollout_tc_audit(bun, g, a, phi=PHI, fee_rate=fee, hidden=hidden, group=group, precision=precision)
    f2, t2 = sg.rollout_population(bun, g, a, phi=PHI, fee_rate=fee, hidden=hidden, precision=precision, units_per_lane=group)
    assert torch.equal(f2.view(torch.int64), fit.view(torch.int64)) and torch.equal(t2, trd), "production != audit"
    st = _audit_outputs(g, z1, z2, raw, act, hidden, tau)
    fit, trd = fit.cpu().numpy(), trd.cpu().numpy()
    loop = edge if hidden == 32 else [sms, sms + 1, 2 * sms, P - 1]
    rows = {i: (raw[i].cpu().numpy(), act[i].cpu().numpy()) for i in edge}
    del raw, act
    torch.cuda.empty_cache()
    orc.lib()                                       # loaded once before the oracle runs on several threads
    with ThreadPoolExecutor(8) as ex:
        res = list(ex.map(lambda i: _check_individual(orc, bz, fee, hidden, tau, G, A, fit[i], trd[i], *rows[i], i, i in loop), edge))
    problems = [p for r, _ in res for p in r]
    same = sum(1 for _, s in res if s)
    shape = f"{per_cta} groups of {G_} per CTA on {C} CTAs" if hidden == 32 else f"{per_cta} individuals per CTA on {C} CTAs"
    print(f"\n{name}: P = {P}, T = {T} ({shape}); max |d(raw*5)| = {st['worst']:.4g} ticks (TAU {tau}) at (i, t, inv, side, "
          f"kernel, ref) = {st['at']}; {st['over_half']} outputs over TAU/2; {st['flips']} of {P * T * 10} rounded outputs "
          f"flip, {st['outside']} outside the near-tie margin; closed loop identical to the oracle for {same} of {len(loop)}; "
          f"{time.time() - t0:.1f} s")
    assert st["nonfinite"] == 0, st
    assert st["worst"] <= tau, st
    assert st["outside"] == 0, st
    assert st["off_row"] == 0, f"{st['off_row']} taken offsets are none of their bar's rounded outputs"
    assert not problems, problems[:5]


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,use_adv", [(32, False), (256, False), (256, True)])
def test_seeded_children_at_scale(sg, orc, hidden, use_adv):
    """The GA's evaluation path: children generated inside the kernel (make_source in every group / individual) equal
    the children materialised with oracle.mutate, bit for bit, for the whole population."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    P = 4096 if hidden == 32 else 4 * sms + 3
    precision = "bf16"
    bundle, bz, stats = _episode(60, 620, None)
    bun = sg.Bundle.from_arrays(bundle, stats, TICK)
    master = _genomes(1, hidden, 31)[0]
    seed, gen, first = 91, 5, 17
    kids = torch.from_numpy(np.stack([orc.mutate(master, 0.05, seed, gen, first + i) for i in range(P)])).cuda()
    adv_master = akids = None
    if use_adv:
        adv_master = _adv(1, 32)[0]
        akids = torch.from_numpy(np.stack([orc.mutate(adv_master, 0.1, seed ^ 0x8000000000000000, gen, first + i)
                                           for i in range(P)])).cuda()
        adv_master = torch.from_numpy(adv_master).cuda()
    fs, ts = sg.rollout_seeded(bun, torch.from_numpy(master).cuda(), count=P, sigma=0.05, seed=seed, generation=gen,
                               first_index=first, adv_master=adv_master, adv_sigma=0.1, phi=PHI, fee_rate=3e-4,
                               hidden=hidden, precision=precision)
    fe, te = sg.rollout_population(bun, kids, akids, phi=PHI, fee_rate=3e-4, hidden=hidden, precision=precision)
    assert torch.equal(fs.view(torch.int64), fe.view(torch.int64)) and torch.equal(ts, te)
    assert int((te > 0).sum()) > P // 2 and fe.unique().numel() > P // 2          # the episodes are not all alike
