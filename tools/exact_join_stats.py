"""How soon does a rollout started cold (inventory 0) at bar s join the true trajectory?  Bench inputs (configs[1])."""
import sys, numpy as np
import os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sgmm_b200 import synthetic
from oracle import oracle

PHI, TICK, FEE = 1e-4, 0.001, 0.0
bundle = synthetic.synthetic_bundle(60)
stats = synthetic.train_stats_of(bundle)
z1, z2 = oracle.normalise(bundle, stats)
bz = (z1, z2) + tuple(np.asarray(a) for a in bundle[2:])
T = len(z1)
_, genomes = synthetic.policy_like_genomes(4096, 32, seed=0, sigma=0.05, out_scale=1.0)
adv = np.zeros(1250, np.float32)
rng = np.random.default_rng(1)
idx = rng.choice(4096, int(sys.argv[1]) if len(sys.argv) > 1 else 48, replace=False)
W = 4096
delays, trades, zero_at = [], [], []
for i in idx:
    f, tr, tt = oracle.rollout(genomes[i], adv, bz, PHI, TICK, FEE, trace=True)
    trades.append(tr)
    post = tt["inventory"]
    enter = np.concatenate([[0], post[:-1]])          # inventory entering bar t
    for s in range(512, T - W, 1024):
        sl = tuple(a[s:s + W] for a in bz)
        _, _, ts = oracle.rollout(genomes[i], adv, sl, PHI, TICK, FEE, trace=True)
        e2 = np.concatenate([[0], ts["inventory"][:-1]])
        eq = np.nonzero(e2 == enter[s:s + W])[0]
        d = int(eq[0]) if eq.size else W
        if eq.size:   # once joined the two must agree for ever after (state = inventory)
            assert np.array_equal(e2[eq[0]:], enter[s + eq[0]:s + W])
        delays.append(d)
        zero_at.append(enter[s] == 0)
delays = np.array(delays)
print("individuals", len(idx), "starts", delays.size, "trades/episode median", int(np.median(trades)),
      "min", int(np.min(trades)), "max", int(np.max(trades)))
print("true inventory at a start = 0 (guess right at once):", float(np.mean(zero_at)))
for q in (0.5, 0.9, 0.99, 0.999, 1.0):
    print(f"delay quantile {q}: {np.quantile(delays, q):.0f} bars")
for B in (0, 8, 16, 24, 32, 48, 64, 128, 256, 512, 1024):
    print(f"P(not joined after {B} bars) = {np.mean(delays > B):.4f}")
print("never joined within", W, ":", int(np.sum(delays >= W)))
