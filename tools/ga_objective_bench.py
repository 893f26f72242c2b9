"""Cost of the training objectives (sgmm_rollout_objective, DeviceGA ``objective``) against the reward, in one process.

    python tools/ga_objective_bench.py [--out FILE] [--reps N]

Workload (synthetic bundles, phi = 1e-4, fee 0):
  - 4 096 explicit H = 32 genomes x 60 days (14 400 bars): sgmm_rollout_population (the reward, the headline kernel),
    sgmm_rollout_objective for PNL, PNL_MAP and SHARPE (the policy-table route), and backtest_population (population
    trace + device analytics: the composition an objective replaces).  CUDA events over `reps` calls, arms alternated
    over three rounds, median reported;
  - a captured GA generation (H = 32 exact, no adversary, one-day validation), reward against each objective, at
    lambda = 50 x one day (240 bars) and lambda = 4 096 x 60 days;
  - PNL_MAP against the reward at H = 256 EXACT, 592 explicit genomes x 60 days (both on the policy-table route).
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import sgmm_b200  # noqa: E402
from exact256_bench import card  # noqa: E402
from ga_sweep_bench import graph_time  # noqa: E402
from sgmm_b200 import synthetic  # noqa: E402
from sgmm_b200.analytics import backtest_population  # noqa: E402
from sgmm_b200.policy import genome_len  # noqa: E402

OBJECTIVES = ("reward", "pnl", "pnl_map", "sharpe")


def bundles(days):
    tb = synthetic.synthetic_bundle(days, first_day=10)
    vb = synthetic.synthetic_bundle(1, first_day=100)
    stats = synthetic.train_stats_of(tb)
    return sgmm_b200.Bundle.from_arrays(tb, stats, 0.001), sgmm_b200.Bundle.from_arrays(vb, stats, 0.001)


def call_time(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def alternate(arms, reps):
    t = {k: [] for k in arms}
    for _ in range(3):
        for k, fn in arms.items():
            t[k].append(call_time(fn, reps))
    return {k: round(statistics.median(v), 4) for k, v in t.items()}, {k: [round(x, 4) for x in v] for k, v in t.items()}


def rollouts(train, P, reps):
    g = torch.from_numpy(synthetic.policy_like_genomes(P, seed=5, out_scale=4.0, out_bias=(0.1, 0.1))[1]).cuda()
    kw = dict(phi=1e-4, fee_rate=0.0)
    arms = {o: (lambda o=o: sgmm_b200.rollout_population(train, g, objective=o, **kw)) for o in OBJECTIVES}
    arms["backtest_population"] = lambda: backtest_population(train, g, **kw)
    ref = {o: sgmm_b200.rollout_population(train, g, objective=o, **kw) for o in OBJECTIVES}
    _, trd, summ = backtest_population(train, g, **kw)
    same_trades = all(ref[o][1].equal(trd) for o in OBJECTIVES)
    med, rounds = alternate(arms, reps)
    return {"hidden": 32, "P": P, "T": train.T, "reps": reps, "ms": med, "ms_rounds": rounds,
            "vs_reward": {k: round(v / med["reward"], 3) for k, v in med.items()}, "trades_equal_backtest": same_trades}


def generations(train, val, pop, reps):
    mm = synthetic.policy_like_genomes(1, seed=3, out_scale=1.0)[0]
    gas = {o: sgmm_b200.DeviceGA(mm, None, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=0.0, use_arl=False, seed=7,
                                 max_generations=4, precision="exact", objective=o) for o in OBJECTIVES}
    for ga in gas.values():
        ga.generation(train, val)
    torch.cuda.synchronize()
    graphs = {o: ga.capture(train, val) for o, ga in gas.items()}
    t = {o: [] for o in OBJECTIVES}
    for _ in range(3):
        for o in OBJECTIVES:
            t[o].append(graph_time(graphs[o].replay, reps))
    med = {o: round(statistics.median(v), 4) for o, v in t.items()}
    del graphs
    for ga in gas.values():
        ga.close()
    return {"hidden": 32, "lambda": pop, "T": train.T, "T_val": val.T, "reps": reps, "ms_per_generation": med,
            "vs_reward": {k: round(v / med["reward"], 3) for k, v in med.items()},
            "ms_rounds": {o: [round(x, 4) for x in v] for o, v in t.items()}}


def h256(train, P, reps):
    g = torch.from_numpy((np.random.default_rng(1).standard_normal((P, genome_len(256))) * 0.05).astype(np.float32)).cuda()
    arms = {o: (lambda o=o: sgmm_b200.rollout_population(train, g, phi=1e-4, hidden=256, precision="exact", objective=o))
            for o in ("reward", "pnl_map")}
    med, rounds = alternate(arms, reps)
    return {"hidden": 256, "precision": "exact", "P": P, "T": train.T, "reps": reps, "ms": med, "ms_rounds": rounds,
            "pnl_map_vs_reward": round(med["pnl_map"] / med["reward"], 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ga_objective_bench needs a CUDA device")
    res = {"card": card()}
    print(json.dumps(res["card"]), flush=True)
    one = bundles(1)
    big = bundles(60)
    res["rollouts"] = rollouts(big[0], 4096, args.reps)
    print(json.dumps(res["rollouts"]), flush=True)
    res["generations"] = [generations(*one, 50, 10 * args.reps), generations(*big, 4096, args.reps)]
    for p in res["generations"]:
        print(json.dumps(p), flush=True)
    res["h256_exact"] = h256(big[0], 592, max(2, args.reps // 10))
    print(json.dumps(res["h256_exact"]), flush=True)
    s = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
