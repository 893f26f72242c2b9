"""A/B of the exact H = 32 rollout: one chain per warp (SGMM_ROLLOUT_CHAINS=1, rollout_kernel_h32) against two time blocks per
warp (=2, rollout2_kernel_h32), alternating child processes (the launcher reads the knobs once per process).

Workload: bench.py's headline (synthetic_bundle(60) = 14 400 bars, policy_like_genomes(4096, seed=0, sigma=0.05), phi 1e-4,
no fee), CUDA events around each rollout with a 256 MiB L2 flush between steps.  Also times U = 1 (P = 592) and U = 2 (P =
4096 pinned) and U = 1 at P = 4096.  Reports the card's name and power limit, each arm's spread over processes and whether its outputs equal the
single-chain arm's.
args: [pairs] [out.json]; extra settings through EXTRA="BURN_IN=32;BURN_IN=8" (each a two-chain arm with that burn-in)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r"""
import sys, json, numpy as np, torch
sys.path.insert(0, ROOT)
import sgmm_b200
from sgmm_b200 import synthetic
bundle = synthetic.synthetic_bundle(60)
bun = sgmm_b200.Bundle.from_arrays(bundle, synthetic.train_stats_of(bundle), 0.001)
out = {}
for name, P, U in (("p4096", 4096, 0), ("p592_u1", 592, 0), ("p4096_u2", 4096, 2), ("p4096_u1", 4096, 1)):
    _, genomes = synthetic.policy_like_genomes(P, 32, seed=0, sigma=0.05, out_scale=1.0)
    g = torch.from_numpy(genomes).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        f, t = sgmm_b200.rollout_population(bun, g, phi=1e-4, units_per_lane=U)
    torch.cuda.synchronize()
    ms = []
    for _ in range(STEPS):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); f, t = sgmm_b200.rollout_population(bun, g, phi=1e-4, units_per_lane=U); e1.record()
        torch.cuda.synchronize(); ms.append(e0.elapsed_time(e1))
    out[name] = {"ms_median": float(np.median(ms)), "ms_min": float(min(ms)), "ms_max": float(max(ms)),
                 "checksum_fitness": float(np.asarray(f.cpu().numpy(), np.float64).view(np.uint64).sum() % (1 << 61)),
                 "trades_sum": int(t.sum().item())}
print("RESULT " + json.dumps(out))
"""


def run(env_extra, steps):
    env = {k: v for k, v in os.environ.items() if not k.startswith("SGMM_ROLLOUT_")}
    env.update(env_extra)
    code = CHILD.replace("ROOT", repr(ROOT)).replace("STEPS", str(steps))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    if r.returncode != 0 or not line:
        raise SystemExit(f"child failed ({env_extra}):\n{r.stdout[-2000:]}\n{r.stderr[-2000:]}")
    return json.loads(line[0][7:])


def main():
    pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    out_path = sys.argv[2] if len(sys.argv) > 2 else None
    arms = {"chains1": {"SGMM_ROLLOUT_CHAINS": "1"}, "chains2": {"SGMM_ROLLOUT_CHAINS": "2"}}
    for s in filter(None, os.environ.get("EXTRA", "").split(";")):
        k, v = s.split("=")
        arms[f"chains2_{k.lower()}{v}"] = {"SGMM_ROLLOUT_CHAINS": "2", "SGMM_ROLLOUT_" + k: v}
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    runs = {a: [] for a in arms}
    for i in range(pairs):
        for a, env in arms.items():
            runs[a].append(run(env, 20))
            print(a, i, json.dumps(runs[a][-1]), flush=True)
    summary = {"device": smi, "pairs": pairs, "steps_per_process": 20, "arms": {}}
    for a in arms:
        summary["arms"][a] = {}
        for case in runs[a][0]:
            med = [r[case]["ms_median"] for r in runs[a]]
            summary["arms"][a][case] = {"ms_median_per_process": med, "ms_median": sorted(med)[len(med) // 2],
                                        "spread_ms": [min(med), max(med)],
                                        "same_outputs_every_process": len({(r[case]["checksum_fitness"], r[case]["trades_sum"])
                                                                           for r in runs[a]}) == 1,
                                        "checksum": [runs[a][0][case]["checksum_fitness"], runs[a][0][case]["trades_sum"]]}
    b = summary["arms"]["chains1"]
    for a in arms:
        for case in b:
            summary["arms"][a][case]["speedup_vs_chains1"] = b[case]["ms_median"] / summary["arms"][a][case]["ms_median"]
            summary["arms"][a][case]["same_outputs_as_chains1"] = summary["arms"][a][case]["checksum"] == b[case]["checksum"]
    print(json.dumps(summary, indent=1))
    if out_path:
        with open(out_path, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
