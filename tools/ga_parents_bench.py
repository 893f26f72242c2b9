"""Cost of truncation selection (DeviceGA / DeviceGASweep ``parents``): captured generations with mu = 1 against mu > 1.

    python tools/ga_parents_bench.py [--out FILE] [--reps N]

Workload (synthetic bundles, a one-day validation bundle, phi = 1e-4):
  - lambda = 50 x one day (240 bars), the reference's scale: mu in {1, 5, 25}, with and without the adversary;
  - lambda = 4 096 x 60 days (14 400 bars), hidden 32 exact: mu in {1, 64, 512};
  - hidden 256 (config 4's genome, G = 67 330) with fee 3e-4, mu in {1, 1024}: BF16 at lambda = 16 384 x one day, EXACT at
    lambda = 2 048 x one day (the population and the days are cut from config 4's 16 384 x 120 days to keep the run short).
mu = 1 is the default GA (ga_tell_kernel); mu > 1 runs ga_select_kernel + ga_recombine_kernel with equal weights.  Both are
CUDA graphs captured after one eager generation and timed with CUDA events over `reps` replays, the two alternated over
three rounds (median reported).  A torch.profiler pass in a separate run splits one eager generation of each mu > 1 point
into kernels, plus lambda = 65 536 x one day with mu = 1024 (config 5's population on one device).  For information only:
the final best validation fitness of 8 seeds x 100 generations at lambda = 50 x one day, mu = 1 against mu = 10 (equal
weights), run as two 8-run sweeps.  The card's name and power limit are read in the same run.
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
from spec256_adv_bench import kernel_times  # noqa: E402
from sgmm_b200 import synthetic  # noqa: E402
from sgmm_b200.policy import genome_len  # noqa: E402


def bundles(days):
    tb = synthetic.synthetic_bundle(days, first_day=10)
    vb = synthetic.synthetic_bundle(1, first_day=100)
    stats = synthetic.train_stats_of(tb)
    return sgmm_b200.Bundle.from_arrays(tb, stats, 0.001), sgmm_b200.Bundle.from_arrays(vb, stats, 0.001)


def make(pop, mu, use_arl, hidden, precision, fee):
    mm = (synthetic.policy_like_genomes(1, seed=3, out_scale=1.0)[0] if hidden == 32 else
          (np.random.default_rng(3).standard_normal(genome_len(hidden)) * 0.05).astype(np.float32))
    adv = (np.random.default_rng(4).standard_normal(1250) * 0.5).astype(np.float32) if use_arl else None
    return sgmm_b200.DeviceGA(mm, adv, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=fee, use_arl=use_arl, seed=7,
                              max_generations=4, patience=15, hidden=hidden, precision=precision, parents=mu)


def point(train, val, pop, mu, use_arl, reps, hidden=32, precision="exact", fee=0.0):
    gas = [make(pop, 1, use_arl, hidden, precision, fee), make(pop, mu, use_arl, hidden, precision, fee)]
    for ga in gas:
        ga.generation(train, val)                             # eager generation: allocates, configures the kernels
    torch.cuda.synchronize()
    graphs = [ga.capture(train, val) for ga in gas]
    t = [[], []]
    for _ in range(3):
        for i in (0, 1):
            t[i].append(graph_time(graphs[i].replay, reps))
    t1, tm = statistics.median(t[0]), statistics.median(t[1])
    out = {"hidden": hidden, "precision": precision, "lambda": pop, "T": train.T, "T_val": val.T, "use_arl": use_arl,
           "mu": mu, "reps": reps, "mu1_ms_per_generation": round(t1, 4), "mu_ms_per_generation": round(tm, 4),
           "extra_ms": round(tm - t1, 4), "mu1_ms_rounds": [round(x, 4) for x in t[0]],
           "mu_ms_rounds": [round(x, 4) for x in t[1]]}
    del graphs
    for ga in gas:
        ga.close()
    return out


def split(train, val, pop, mu, use_arl, hidden=32, precision="exact", fee=0.0):
    ga = make(pop, mu, use_arl, hidden, precision, fee)
    ga.generation(train, val)
    torch.cuda.synchronize()
    kt = kernel_times(lambda: ga.generation(train, val))
    ga.close()
    return {"hidden": hidden, "precision": precision, "lambda": pop, "T": train.T, "use_arl": use_arl, "mu": mu,
            "select_ms": kt.get("sgmm::ga_select_kernel"), "recombine_ms": kt.get("sgmm::ga_recombine_kernel"),
            "kernels_ms": kt}


def quality(train, val, mu, seeds=8, gens=100):
    mm = np.stack([synthetic.policy_like_genomes(1, seed=50 + r, out_scale=1.0)[0] for r in range(seeds)])
    runs = [dict(seed=9000 + r, phi=1e-4) for r in range(seeds)]
    sw = sgmm_b200.DeviceGASweep(mm, None, runs=runs, pop_size=50, use_arl=False, max_generations=gens, parents=mu)
    for _ in range(gens):
        sw.generation(train, val)
    best = [float(sw.status(r)["best_val"]) for r in range(seeds)]
    sw.close()
    return {"mu": mu, "lambda": 50, "T": train.T, "generations": gens, "best_val_f": [round(b, 4) for b in best],
            "mean": round(float(np.mean(best)), 4), "median": round(float(np.median(best)), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--profile", action="store_true", help="the torch.profiler kernel split (run it separately)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ga_parents_bench needs a CUDA device")
    res = {"card": card()}
    print(json.dumps(res["card"]), flush=True)
    one = bundles(1)
    big = bundles(60)
    if args.profile:
        res["kernel_split"] = []
        for args_ in ((one, 50, 5, False), (one, 50, 25, True), (big, 4096, 64, False), (big, 4096, 512, False),
                      (one, 65536, 1024, False)):
            s = split(*args_[0], *args_[1:])
            print(json.dumps(s), flush=True)
            res["kernel_split"].append(s)
        for prec, pop in (("bf16", 16384), ("exact", 2048)):
            s = split(*one, pop, 1024, False, hidden=256, precision=prec, fee=3e-4)
            print(json.dumps(s), flush=True)
            res["kernel_split"].append(s)
    else:
        res["points"] = []
        cases = [(one, 50, mu, arl, args.reps) for arl in (False, True) for mu in (5, 25)]
        cases += [(big, 4096, mu, False, max(10, args.reps // 10)) for mu in (64, 512)]
        for c in cases:
            p = point(*c[0], *c[1:])
            print(json.dumps(p), flush=True)
            res["points"].append(p)
        for prec, pop in (("bf16", 16384), ("exact", 2048)):
            p = point(*one, pop, 1024, False, max(10, args.reps // 10), hidden=256, precision=prec, fee=3e-4)
            print(json.dumps(p), flush=True)
            res["points"].append(p)
        res["quality_info_only"] = [quality(*one, mu) for mu in (1, 10)]
        print(json.dumps(res["quality_info_only"]), flush=True)
    s = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
