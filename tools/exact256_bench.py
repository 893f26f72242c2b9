"""Time the bit-exact H = 256 path (SGMM_PRECISION_EXACT, csrc/sgmm_exact256.cu) with CUDA events.

    python tools/exact256_bench.py [--out FILE] [--skip-ga]

Shapes: 1 x 28 800 bars (BASELINE config 4's validation rollout), 50 x 240 (the reference's population of 50 over one
day), 592 x 14 400, and one config-4 GA generation (16 384 seeded children x 28 800 bars, fee 3e-4, then the validation
rollout) with EXACT next to BF16.  Every timed call is preceded by a warm-up call of the same shape and by a 512 MB write
that evicts the 126 MB L2.  Reports ms, env-steps/s, and the executed FLOP/s (5 x 133 632 FLOP per env-step: the
policy of all five inventories of every bar) over the measured FP32 FFMA peak; the table kernel's own time at 592 x 14 400
comes from torch.profiler in the same run.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import sgmm_b200  # noqa: E402
from sgmm_b200 import synthetic  # noqa: E402
from sgmm_b200.engine import DeviceGA  # noqa: E402

FLOP_PER_ENV_STEP = 5 * 2 * (3 * 256 + 256 * 256 + 2 * 256)       # 5 x 133 632 executed per bar
_flush = None


def flush_l2():
    global _flush
    if _flush is None:
        _flush = torch.empty(128 << 20, dtype=torch.float32, device="cuda")
    _flush.fill_(1.0)


def timed(fn, reps):
    fn()                                                            # warm-up of this shape
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush_l2()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(min(ts)), float(max(ts))


def bun_of(days, T=None):
    b = synthetic.synthetic_bundle(days)
    if T is not None:
        b = tuple(a[:T] for a in b)
    return sgmm_b200.Bundle.from_arrays(b, synthetic.train_stats_of(b), 0.001)


def card():
    """The card's name, and its power limit and maximum SM clock where nvidia-smi (a read-only query) is available."""
    out = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60)
        out["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.stdout.strip() else ""
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-ga", action="store_true")
    args = ap.parse_args()
    peak = sgmm_b200.measure_fp32_peak(0)
    res = {"card": card(), "fp32_peak_tflops": round(peak, 2), "rows": []}
    print(res["card"], "FP32 FFMA peak", round(peak, 2), "TFLOP/s", flush=True)

    def row(name, P, T, ms, extra=None):
        r = {"case": name, "P": P, "T": T, "ms_median": round(ms[0], 4), "ms_min": round(ms[1], 4), "ms_max": round(ms[2], 4),
             "G_env_steps_per_s": round(P * T / ms[0] / 1e6, 4),
             "executed_tflops": round(P * T * FLOP_PER_ENV_STEP / ms[0] / 1e9, 2)}
        r["share_of_fp32_peak"] = round(r["executed_tflops"] / peak, 3)
        if extra:
            r.update(extra)
        res["rows"].append(r)
        print(r, flush=True)

    for (P, days, T, reps) in ((1, 120, None, 20), (50, 1, None, 20), (592, 60, None, 3)):
        bun = bun_of(days, T)
        _, g = synthetic.policy_like_genomes(P, hidden=256, seed=P)
        g = torch.from_numpy(g).cuda()
        ms = timed(lambda: sgmm_b200.rollout_population(bun, g, phi=1e-4, fee_rate=3e-4, hidden=256, precision="exact"), reps)
        row("exact rollout (table + walk)", P, bun.T, ms)
        if P == 592:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                sgmm_b200.rollout_population(bun, g, phi=1e-4, fee_rate=3e-4, hidden=256, precision="exact")
                torch.cuda.synchronize()
            kt = {}
            for ev in prof.key_averages():
                if ev.device_type is not None and "kernel" in ev.key:
                    kt[ev.key.split("(")[0]] = kt.get(ev.key.split("(")[0], 0.0) + ev.device_time_total / 1e3
            tab = [v for k, v in kt.items() if "exact256_table" in k]
            res["kernels_592x14400_ms"] = {k: round(v, 3) for k, v in kt.items()}
            if tab:
                row("exact256_table_kernel alone", P, bun.T, (tab[0], tab[0], tab[0]))
            print("kernels:", res["kernels_592x14400_ms"], flush=True)
            ms = timed(lambda: sgmm_b200.rollout_population(bun, g, phi=1e-4, fee_rate=3e-4, hidden=256), reps)
            row("bf16 spec256 rollout (same shape, for scale)", P, bun.T, ms)

    if not args.skip_ga:
        bun4 = bun_of(120)
        val = bun_of(120)
        m, _ = synthetic.policy_like_genomes(1, hidden=256, seed=0)
        for prec in ("bf16", "exact"):
            def make(pop):
                return DeviceGA(m, None, pop_size=pop, sigma=0.05, phi=1e-4, fee_rate=3e-4, use_arl=False, seed=1,
                                max_generations=4, hidden=256, precision=prec)
            warm = make(16384)
            warm.generation(bun4, val)                               # warm-up: modules, code buffers of both bundles
            torch.cuda.synchronize()
            ga = make(16384)
            flush_l2()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ga.generation(bun4, val)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            row(f"config-4 GA generation ({prec})", 16384, bun4.T, (ms, ms, ms),
                {"note": "population + validation rollout; FLOP columns count 5 policy evaluations per env-step"})
            warm.close(); ga.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
