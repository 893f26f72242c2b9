"""Time a GA sweep (DeviceGASweep: K runs in the same launches) against K solo DeviceGA runs replayed back to back.

    python tools/ga_sweep_bench.py [--out FILE] [--reps N]

Workload: synthetic bundles, lambda = 50 per run, a training bundle of one day (240 bars) and of 15 days (3 600 bars), a
one-day validation bundle, with and without the adversary, K in {1, 2, 4, 8, 16, 32}; plus one point past the
small-population break-even, K = 4 x lambda = 4 096 x one day, where every solo GA runs rollout_kernel_h32 and the sweep
still takes the policy-table path.  Runs differ in seed, phi (0, 1e-4, 0.01) and fee (0, 3e-4).
Both sides are CUDA graphs captured after one eager generation: the sweep's one graph per generation, and the K solo
graphs replayed one after the other.  Each side is warmed up, then timed with CUDA events over `reps` (>= 200) replays.
Reported: ms per generation of the sweep and of the K solo GAs, run-generations per second of both, and the ratio.  After
timing, the masters and status of every run are compared with its solo GA (both advanced the same generations).  A
torch.profiler pass splits one eager generation of the K = 8, one-day, no-adversary sweep and of its solo GAs into kernels.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import sgmm_b200  # noqa: E402
from exact256_bench import card  # noqa: E402
from spec256_adv_bench import kernel_times  # noqa: E402
from sgmm_b200 import synthetic  # noqa: E402


def bundles(days):
    tb = synthetic.synthetic_bundle(days, first_day=10)
    vb = synthetic.synthetic_bundle(1, first_day=40)
    stats = synthetic.train_stats_of(tb)
    return sgmm_b200.Bundle.from_arrays(tb, stats, 0.001), sgmm_b200.Bundle.from_arrays(vb, stats, 0.001)


def runs_of(K):
    return [dict(seed=1000 + r, phi=(0.0, 1e-4, 0.01)[r % 3], fee_rate=(0.0, 3e-4)[r % 2], sigma=0.05, patience=3)
            for r in range(K)]


def graph_time(replay, reps):
    for _ in range(10):
        replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def point(K, pop, days, use_arl, reps):
    train, val = bundles(days)
    runs = runs_of(K)
    mm = np.stack([synthetic.policy_like_genomes(1, seed=r, out_scale=1.0)[0] for r in range(K)])
    adv = (np.random.default_rng(K).standard_normal((K, 1250)) * 0.5).astype(np.float32) if use_arl else None
    gens = 1 + 2 * (10 + reps)
    sweep = sgmm_b200.DeviceGASweep(mm, adv, runs=runs, pop_size=pop, use_arl=use_arl, max_generations=gens)
    solos = [sgmm_b200.DeviceGA(mm[r], None if adv is None else adv[r], pop_size=pop, use_arl=use_arl, max_generations=gens,
                                precision="exact", **runs[r]) for r in range(K)]
    sweep.generation(train, val)                             # eager generation 0: allocates the table buffers
    for s in solos:
        s.generation(train, val)
    torch.cuda.synchronize()
    gs = sweep.capture(train, val)
    gsolo = [s.capture(train, val) for s in solos]
    t_sweep = graph_time(gs.replay, reps)
    t_solo = graph_time(lambda: [g.replay() for g in gsolo], reps)
    same = True
    for r in range(K):
        a, b = sweep.masters(r), solos[r].masters()
        same &= all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(a, b))
        same &= sweep.status(r) == solos[r].status()
    out = {"K": K, "lambda": pop, "T": train.T, "T_val": val.T, "use_arl": use_arl, "reps": reps,
           "sweep_ms_per_generation": round(t_sweep, 4), "solo_ms_per_K_generations": round(t_solo, 4),
           "sweep_run_generations_per_s": round(K * 1e3 / t_sweep, 1),
           "solo_run_generations_per_s": round(K * 1e3 / t_solo, 1),
           "speedup": round(t_solo / t_sweep, 3), "runs_bit_identical_to_solo": bool(same)}
    del gs, gsolo
    sweep.close()
    for s in solos:
        s.close()
    return out


def profile_split(K, pop, days):
    train, val = bundles(days)
    runs = runs_of(K)
    mm = np.stack([synthetic.policy_like_genomes(1, seed=r, out_scale=1.0)[0] for r in range(K)])
    sweep = sgmm_b200.DeviceGASweep(mm, None, runs=runs, pop_size=pop, use_arl=False, max_generations=8)
    solos = [sgmm_b200.DeviceGA(mm[r], None, pop_size=pop, use_arl=False, max_generations=8, precision="exact", **runs[r])
             for r in range(K)]
    sweep.generation(train, val)
    for s in solos:
        s.generation(train, val)
    torch.cuda.synchronize()
    out = {"K": K, "lambda": pop, "T": train.T, "sweep_one_generation_ms": kernel_times(lambda: sweep.generation(train, val)),
           "solo_K_generations_ms": kernel_times(lambda: [s.generation(train, val) for s in solos])}
    sweep.close()
    for s in solos:
        s.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ga_sweep_bench needs a CUDA device")
    res = {"card": card(), "points": []}
    for days in (1, 15):
        for use_arl in (False, True):
            for K in (1, 2, 4, 8, 16, 32):
                p = point(K, 50, days, use_arl, args.reps)
                print(json.dumps(p), flush=True)
                res["points"].append(p)
    for use_arl in (False, True):                           # past the small-population break-even of a solo GA
        p = point(4, 4096, 1, use_arl, args.reps)
        print(json.dumps(p), flush=True)
        res["points"].append(p)
    res["kernel_split"] = profile_split(8, 50, 1)
    print(json.dumps(res["kernel_split"]), flush=True)
    s = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
