"""Time the adversary on the H = 256 tensor-core path (spec256 q tables + walk_account_kernel<Walk20>) with CUDA events.

    python tools/spec256_adv_bench.py [--out FILE] [--skip-ga]

Shapes: 592 x 14 400 bars, fee 3e-4: BF16 without the adversary, BF16 with it (the q-table route), EXACT with it; then a
torch.profiler pass of the BF16 adversary route in the same run splits its time into spec256_kernel and
walk_account_kernel<Walk20>.  One config-4 GA generation (16 384 seeded children x 28 800 bars, fee 3e-4, then the
validation rollout): use_arl in BF16 next to use_arl=False BF16 and use_arl EXACT.  Every timed call is preceded by a
warm-up call of the same shape and by a 512 MB write that evicts the 126 MB L2.  The card's name and power limit are read
in the same run.
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
from exact256_bench import bun_of, card, flush_l2, timed  # noqa: E402
from sgmm_b200 import synthetic  # noqa: E402
from sgmm_b200.engine import DeviceGA  # noqa: E402


def kernel_times(fn):
    """Device time per kernel name (ms) of one call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kt = {}
    for ev in prof.key_averages():
        if ev.device_type is not None and "kernel" in ev.key:
            k = ev.key.split("(")[0]
            kt[k] = kt.get(k, 0.0) + ev.device_time_total / 1e3
    return {k: round(v, 3) for k, v in kt.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-ga", action="store_true")
    args = ap.parse_args()
    res = {"card": card(), "rows": []}
    print(res["card"], flush=True)

    def row(name, P, T, ms, extra=None):
        r = {"case": name, "P": P, "T": T, "ms_median": round(ms[0], 3), "ms_min": round(ms[1], 3), "ms_max": round(ms[2], 3),
             "G_env_steps_per_s": round(P * T / ms[0] / 1e6, 4)}
        if extra:
            r.update(extra)
        res["rows"].append(r)
        print(r, flush=True)

    P = 592
    bun = bun_of(60)
    _, g = synthetic.policy_like_genomes(P, hidden=256, seed=P)
    g = torch.from_numpy(g).cuda()
    a = torch.from_numpy((np.random.default_rng(P).standard_normal((P, 1250)) * 0.6).astype(np.float32)).cuda()
    cases = (("bf16, no adversary", None, "bf16"), ("bf16 + adversary (q table + Walk20 walk)", a, "bf16"),
             ("exact + adversary", a, "exact"))
    for name, adv, prec in cases:
        ms = timed(lambda: sgmm_b200.rollout_population(bun, g, adv, phi=1e-4, fee_rate=3e-4, hidden=256, precision=prec), 5)
        row(name, P, bun.T, ms)
    kt = kernel_times(lambda: sgmm_b200.rollout_population(bun, g, a, phi=1e-4, fee_rate=3e-4, hidden=256))
    spec = sum(v for k, v in kt.items() if "spec256_kernel" in k)
    walk = sum(v for k, v in kt.items() if "walk_account_kernel" in k)
    res["kernels_bf16_adv_592x14400_ms"] = kt
    res["walk_share_bf16_adv_592x14400"] = round(walk / (spec + walk), 3) if spec + walk > 0 else None
    print("kernels:", kt, "walk share:", res["walk_share_bf16_adv_592x14400"], flush=True)

    if not args.skip_ga:
        bun4, val = bun_of(120), bun_of(120)
        m, _ = synthetic.policy_like_genomes(1, hidden=256, seed=0)
        am = (np.random.default_rng(1).standard_normal(1250) * 0.5).astype(np.float32)
        for arl, prec in ((False, "bf16"), (True, "bf16"), (True, "exact")):
            def make():
                return DeviceGA(m, am if arl else None, pop_size=16384, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=arl,
                                seed=1, max_generations=4, hidden=256, precision=prec)
            warm = make()
            warm.generation(bun4, val)                               # warm-up: modules, code buffers of both bundles
            torch.cuda.synchronize()
            ga = make()
            flush_l2()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ga.generation(bun4, val)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            row(f"config-4 GA generation (use_arl={arl}, {prec})", 16384, bun4.T, (ms, ms, ms),
                {"note": "population + validation rollout"})
            warm.close(); ga.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
