"""Cost of the natural-gradient evolution strategy (DeviceGA ``es_lr``): captured generations with the (1,lambda) rule,
truncation selection and the ES, in the same process.

    python tools/ga_es_bench.py [--out FILE] [--reps N] [--profile]

Workload (synthetic bundles, a one-day validation bundle, phi = 1e-4, Adam step 0.01):
  - lambda = 50 x one day (240 bars), the reference's scale, with and without the adversary: (1,lambda), mu = 25, ES;
  - lambda = 4 096 x 60 days (14 400 bars), hidden 32 exact: (1,lambda), mu = 512, ES;
  - lambda = 65 536 x one day, hidden 32 exact, one GPU: (1,lambda), ES;
  - hidden 256 (G = 67 330) BF16 with fee 3e-4 at lambda = 16 384 x one day: (1,lambda), ES.
Every arm is a CUDA graph captured after one eager generation and timed with CUDA events over `reps` replays; the arms
are alternated over three rounds (median reported).  ``--profile`` (run it separately) splits one eager ES generation of
each point into kernels with torch.profiler.  For information only: the best validation fitness of 8 seeds x 100
generations at lambda = 50 x one day for (1,lambda), mu = 12 (lambda/4) and the ES, run as 8-run sweeps.  The card's name
and power limit are read in the same run.
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

LR = 0.01


def bundles(days):
    tb = synthetic.synthetic_bundle(days, first_day=10)
    vb = synthetic.synthetic_bundle(1, first_day=100)
    stats = synthetic.train_stats_of(tb)
    return sgmm_b200.Bundle.from_arrays(tb, stats, 0.001), sgmm_b200.Bundle.from_arrays(vb, stats, 0.001)


def make(pop, use_arl, hidden, precision, fee, **update):
    mm = (synthetic.policy_like_genomes(1, seed=3, out_scale=1.0)[0] if hidden == 32 else
          (np.random.default_rng(3).standard_normal(genome_len(hidden)) * 0.05).astype(np.float32))
    adv = (np.random.default_rng(4).standard_normal(1250) * 0.5).astype(np.float32) if use_arl else None
    return sgmm_b200.DeviceGA(mm, adv, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=fee, use_arl=use_arl, seed=7,
                              max_generations=4, patience=15, hidden=hidden, precision=precision, **update)


def point(train, val, pop, use_arl, reps, mu=None, hidden=32, precision="exact", fee=0.0):
    arms = {"one_lambda": {}, "es": {"es_lr": LR}}
    if mu:
        arms[f"mu{mu}"] = {"parents": mu}
    gas = {k: make(pop, use_arl, hidden, precision, fee, **kw) for k, kw in arms.items()}
    for ga in gas.values():
        ga.generation(train, val)                             # eager generation: configures the kernels
    torch.cuda.synchronize()
    graphs = {k: ga.capture(train, val) for k, ga in gas.items()}
    t = {k: [] for k in arms}
    for _ in range(3):
        for k in arms:
            t[k].append(graph_time(graphs[k].replay, reps))
    med = {k: statistics.median(v) for k, v in t.items()}
    out = {"hidden": hidden, "precision": precision, "lambda": pop, "T": train.T, "T_val": val.T, "use_arl": use_arl,
           "reps": reps, "ms_per_generation": {k: round(v, 4) for k, v in med.items()},
           "es_extra_ms": round(med["es"] - med["one_lambda"], 4),
           "es_extra_pct": round(100.0 * (med["es"] / med["one_lambda"] - 1.0), 2),
           "ms_rounds": {k: [round(x, 4) for x in v] for k, v in t.items()}}
    if mu:
        out[f"mu{mu}_extra_pct"] = round(100.0 * (med[f"mu{mu}"] / med["one_lambda"] - 1.0), 2)
    del graphs
    for ga in gas.values():
        ga.close()
    return out


def split(train, val, pop, use_arl, hidden=32, precision="exact", fee=0.0):
    ga = make(pop, use_arl, hidden, precision, fee, es_lr=LR)
    ga.generation(train, val)
    torch.cuda.synchronize()
    kt = kernel_times(lambda: ga.generation(train, val))
    ga.close()
    return {"hidden": hidden, "precision": precision, "lambda": pop, "T": train.T, "use_arl": use_arl,
            "rank_ms": kt.get("sgmm::es_rank_kernel"), "grad_ms": kt.get("sgmm::es_grad_kernel"),
            "adam_ms": kt.get("sgmm::es_adam_kernel"), "kernels_ms": kt}


def quality(train, val, seeds=8, gens=100, **update):
    mm = np.stack([synthetic.policy_like_genomes(1, seed=50 + r, out_scale=1.0)[0] for r in range(seeds)])
    runs = [dict(seed=9000 + r, phi=1e-4) for r in range(seeds)]
    sw = sgmm_b200.DeviceGASweep(mm, None, runs=runs, pop_size=50, use_arl=False, max_generations=gens, **update)
    for _ in range(gens):
        sw.generation(train, val)
    best = [float(sw.status(r)["best_val"]) for r in range(seeds)]
    sw.close()
    return {"update": update or "one_lambda", "lambda": 50, "T": train.T, "generations": gens,
            "best_val_f": [round(b, 4) for b in best], "mean": round(float(np.mean(best)), 4),
            "median": round(float(np.median(best)), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--profile", action="store_true", help="the torch.profiler kernel split (run it separately)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ga_es_bench needs a CUDA device")
    res = {"card": card(), "es_lr": LR}
    print(json.dumps(res["card"]), flush=True)
    one = bundles(1)
    big = bundles(60)
    if args.profile:
        res["kernel_split"] = []
        for a in ((one, 50, False), (one, 50, True), (big, 4096, False), (one, 65536, False), (one, 65536, True)):
            s = split(*a[0], *a[1:])
            print(json.dumps(s), flush=True)
            res["kernel_split"].append(s)
        s = split(*one, 16384, False, hidden=256, precision="bf16", fee=3e-4)
        print(json.dumps(s), flush=True)
        res["kernel_split"].append(s)
    else:
        res["points"] = []
        cases = [(one, 50, arl, args.reps, 25) for arl in (False, True)]
        cases += [(big, 4096, False, max(10, args.reps // 10), 512), (one, 65536, False, max(10, args.reps // 10), None)]
        for c in cases:
            p = point(*c[0], *c[1:])
            print(json.dumps(p), flush=True)
            res["points"].append(p)
        p = point(*one, 16384, False, max(10, args.reps // 10), hidden=256, precision="bf16", fee=3e-4)
        print(json.dumps(p), flush=True)
        res["points"].append(p)
        res["quality_info_only"] = [quality(*one), quality(*one, parents=12), quality(*one, es_lr=LR)]
        print(json.dumps(res["quality_info_only"]), flush=True)
    s = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
