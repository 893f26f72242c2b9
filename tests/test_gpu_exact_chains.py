"""GPU (-m gpu): the two-chain exact H = 32 rollout (rollout2_kernel_h32) bit for bit against the single-chain kernel
(SGMM_ROLLOUT_CHAINS=1) and the oracle, on fitness and trades.

The launcher reads SGMM_ROLLOUT_CHAINS and SGMM_ROLLOUT_BURN_IN once per process, so every setting runs in a child
process that writes its results to an .npz (this file is also that child's script).  Episode lengths straddle the
kernel's round of 256 bars and its default burn-in of 4; burn-in 0 makes the stitch repair almost every round, and a
crafted policy whose cold starts never join the true trajectory drives the repair across whole blocks.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
ROUND, BURN = 256, 4
TS = [1, 2, BURN - 1, BURN + 1, ROUND - 1, ROUND, ROUND + 1, 2 * ROUND - 1, 2 * ROUND + 1, 2049, 14400, 60000]
# (P, fee, seeded, units_per_lane): 401 takes U = 1, 6*148*4 + 3 two waves, 8192 + 5 a ragged last CTA
POPS = [(401, 0.0, False, 0), (4096, 3e-4, True, 0), (6 * 148 * 4 + 3, 0.0, True, 0), (8192 + 5, 3e-4, False, 0),
        (1000, 3e-4, False, 2)]
CASES = [(T,) + p for T in TS for p in POPS] + [(T, 600, 0.0, False, 4) for T in (ROUND + 1, 14400)]
PHI, TICK = 1e-4, 0.001


def bundle_of(T):
    from sgmm_b200 import synthetic
    days = max(1, -(-T // 240))
    bundle = tuple(a[:T] for a in synthetic.synthetic_bundle(days, first_day=300))
    stats = synthetic.train_stats_of(synthetic.synthetic_bundle(1, first_day=299))
    return bundle, stats


def case_population(T, P, seeded):
    from sgmm_b200 import synthetic
    master, genomes = synthetic.policy_like_genomes(1 if seeded else P, seed=T + P, out_scale=2.0, out_bias=(0.1, 0.1))
    return master, genomes


def crafted_genome():
    """Inventory +1 and -1 absorb: there both sides fill every bar (q ~ -2.5e8 at +1, ~ -5e8 at -1, so the records
    differ); at 0 the policy buys when z1 > 0.1 and sells when z1 < -0.1.  A cold start joins the true trajectory only
    when it lands on the same side."""
    H = 32
    g = np.zeros(H * H + 7 * H + 2, np.float32)
    g[3 * 0 + 0], g[3 * 1 + 0] = 1e3, -1e3                    # h1_0 = relu(1e3 z1), h1_1 = relu(-1e3 z1)
    g[3 * 2 + 2], g[3 * 3 + 2] = 1e8, -1e8                    # h1_2 = relu(1e8 inv/2), h1_3 = relu(-1e8 inv/2)
    w2 = 4 * H
    for j in range(4):
        g[w2 + j * H + j] = 1.0                               # h2_j = h1_j
    w3a, w3b = 5 * H + H * H, 6 * H + H * H
    g[w3a + 1], g[w3b + 0] = -1e3, -1e3                        # sell on z1 < 0, buy on z1 > 0
    for w3 in (w3a, w3b):
        g[w3 + 2], g[w3 + 3] = -1.0, -2.0
    g[7 * H + H * H:] = 1e5
    return g


def run_child(out):
    """Child process: every case under this process's SGMM_ROLLOUT_* settings."""
    import torch
    import sgmm_b200
    res = {}
    for T in sorted({c[0] for c in CASES}):
        bundle, stats = bundle_of(T)
        bun = sgmm_b200.Bundle.from_arrays(bundle, stats, TICK)
        for (t, P, fee, seeded, U) in CASES:
            if t != T:
                continue
            master, genomes = case_population(T, P, seeded)
            if seeded:
                f, tr = sgmm_b200.rollout_seeded(bun, torch.from_numpy(master).cuda(), count=P, sigma=0.05, seed=T + 7,
                                                 generation=2, phi=PHI, fee_rate=fee, units_per_lane=U)
            else:
                f, tr = sgmm_b200.rollout_population(bun, torch.from_numpy(genomes).cuda(), phi=PHI, fee_rate=fee,
                                                     units_per_lane=U)
            res[f"f_{T}_{P}_{fee}_{seeded}_{U}"] = f.cpu().numpy()
            res[f"t_{T}_{P}_{fee}_{seeded}_{U}"] = tr.cpu().numpy()
        if T == 14400:
            g = np.repeat(crafted_genome()[None], 1200, 0)
            for U in (0, 1):
                f, tr = sgmm_b200.rollout_population(bun, torch.from_numpy(g).cuda(), phi=PHI, units_per_lane=U)
                res[f"crafted_f_{U}"], res[f"crafted_t_{U}"] = f.cpu().numpy(), tr.cpu().numpy()
        bun.close()
    np.savez(out, **res)


SETTINGS = {"one": {"SGMM_ROLLOUT_CHAINS": "1"}, "two": {"SGMM_ROLLOUT_CHAINS": "2"},
            "burn0": {"SGMM_ROLLOUT_CHAINS": "2", "SGMM_ROLLOUT_BURN_IN": "0"},
            "burn8": {"SGMM_ROLLOUT_CHAINS": "2", "SGMM_ROLLOUT_BURN_IN": "8"},
            "burn32": {"SGMM_ROLLOUT_CHAINS": "2", "SGMM_ROLLOUT_BURN_IN": "32"}}


@pytest.fixture(scope="module")
def results(tmp_path_factory):
    d = tmp_path_factory.mktemp("chains")
    out = {}
    for name, env in SETTINGS.items():
        e = {k: v for k, v in os.environ.items() if not k.startswith("SGMM_ROLLOUT_")}
        e.update(env)
        p = str(d / f"{name}.npz")
        r = subprocess.run([sys.executable, os.path.abspath(__file__), p], env=e, cwd=ROOT, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        out[name] = dict(np.load(p))
    return out


def bits64(a):
    return np.asarray(a, np.float64).view(np.uint64)


@pytest.mark.gpu
@pytest.mark.parametrize("setting", ["two", "burn0", "burn8", "burn32"])
def test_two_chains_equal_one_chain_bitwise(results, setting):
    ref, got = results["one"], results[setting]
    assert sorted(ref) == sorted(got)
    for k in ref:
        a, b = ref[k], got[k]
        assert a.shape == b.shape, k
        if k.startswith("f_") or k.startswith("crafted_f"):
            bad = np.flatnonzero(bits64(a) != bits64(b))
        else:
            bad = np.flatnonzero(a != b)
        assert bad.size == 0, (k, bad[:10], a[bad[:3]], b[bad[:3]])


@pytest.mark.gpu
@pytest.mark.parametrize("T", TS)
def test_two_chains_match_the_oracle(results, T):
    """A sample of every case's individuals (first, last, and spread between) against the C oracle."""
    from oracle import oracle as orc
    bundle, stats = bundle_of(T)
    z1, z2 = orc.normalise(bundle, stats)
    bz = (z1, z2) + bundle[2:]
    for (t, P, fee, seeded, U) in CASES:
        if t != T:
            continue
        idx = np.unique(np.r_[0, 1, P - 2, P - 1, np.linspace(0, P - 1, 12).astype(int)])
        master, genomes = case_population(T, P, seeded)
        key = f"{T}_{P}_{fee}_{seeded}_{U}"
        for name in ("two", "burn0"):
            f, tr = results[name]["f_" + key], results[name]["t_" + key]
            for i in idx:
                if seeded:
                    fo, to = orc.rollout_population(bz, PHI, TICK, fee, master=master, sigma=0.05, seed=T + 7,
                                                    generation=2, first_index=int(i), count=1)
                else:
                    fo, to = orc.rollout_population(bz, PHI, TICK, fee, genomes=genomes[i:i + 1])
                assert bits64(f[i]) == bits64(fo[0]) and tr[i] == to[0], (name, key, i, f[i], fo[0], tr[i], to[0])


@pytest.mark.gpu
def test_never_joining_policy_is_repaired(results):
    """The crafted policy on 14 400 bars: the CPU oracle shows that many rounds' cold starts never join the true
    trajectory inside their block; the device still gives the oracle's bits with every burn-in."""
    from oracle import oracle as orc
    bundle, stats = bundle_of(14400)
    z1, z2 = orc.normalise(bundle, stats)
    bz = (z1, z2) + bundle[2:]
    g = crafted_genome()
    fo, to, tr = orc.rollout(g, None, bz, PHI, TICK, 0.0, trace=True)
    inv = tr["inventory"]                                      # after each bar
    never = 0
    N = (ROUND + BURN) // 2
    for r in range(14400 // ROUND):
        cs = r * ROUND + N - BURN                              # the cold start's first bar
        _, _, trc = orc.rollout(g, None, tuple(a[cs:(r + 1) * ROUND] for a in bz), PHI, TICK, 0.0, trace=True)
        cold = trc["inventory"][BURN:]                         # after bars N .. ROUND - 1 of the round
        never += bool((cold != inv[r * ROUND + N:(r + 1) * ROUND]).all())
    assert never >= 5, never
    for name in SETTINGS:
        for U in (0, 1):
            f, t = results[name][f"crafted_f_{U}"], results[name][f"crafted_t_{U}"]
            assert (bits64(f) == bits64(fo)).all() and (t == to).all(), (name, U, f[:2], fo, t[:2], to)


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    run_child(sys.argv[1])
