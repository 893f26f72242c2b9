"""A/B of two builds of libsgmm_b200.so on the exact H = 32 rollout: the same shapes timed in alternating child processes,
one library per process (the launcher reads its environment knobs once per process).

Workload: bench.py's inputs (synthetic_bundle(60) = 14 400 bars, policy_like_genomes(P, seed=0, sigma=0.05), phi 1e-4,
no fee), CUDA events around each rollout with a 256 MiB L2 flush between steps, 20 steps per process.  Shapes:
  p4096       the bench shape (auto geometry: two chains per warp, U = 4)
  p592_u1     P = 592 (auto: U = 1, two chains)
  p4096_u2    P = 4096 pinned to U = 2 (one chain)
  p4096_1ch   P = 4096 with SGMM_ROLLOUT_CHAINS=1 (one chain, U = 4)
  adv2048     2048 market makers with their own adversaries (bench.py config 3's shape, one chain, U = 4)
Reports the card's name and power limit, each shape's median and spread over processes for each library, whether the new
library's median lies within the old one's spread, and whether every process of both libraries returned the same fitness
and trade bits.
usage: lib_ab_bench.py OLD.so NEW.so [pairs] [out.json]"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r"""
import hashlib, json, sys
import numpy as np, torch
sys.path.insert(0, ROOT)
import sgmm_b200
from sgmm_b200 import _lib, synthetic
_lib.LIB_PATH = __LIB__
bundle = synthetic.synthetic_bundle(60)
bun = sgmm_b200.Bundle.from_arrays(bundle, synthetic.train_stats_of(bundle), 0.001)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
_, g4096 = synthetic.policy_like_genomes(4096, 32, seed=0, sigma=0.05, out_scale=1.0)
adv = torch.from_numpy((np.random.default_rng(3).standard_normal((2048, 1250)) * 0.5).astype(np.float32)).cuda()
SHAPES = {"p4096": (4096, 0, False), "p592_u1": (592, 0, False), "p4096_u2": (4096, 2, False),
          "p4096_1ch": (4096, 0, False), "adv2048": (2048, 0, True)}
out = {}
for name in CASES:
    P, U, with_adv = SHAPES[name]
    g = torch.from_numpy(g4096[:P].copy()).cuda()
    run = lambda: sgmm_b200.rollout_population(bun, g, adv if with_adv else None, phi=1e-4, units_per_lane=U)
    for _ in range(3):
        f, t = run()
    torch.cuda.synchronize()
    ms = []
    for _ in range(STEPS):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); f, t = run(); e1.record()
        torch.cuda.synchronize(); ms.append(e0.elapsed_time(e1))
    digest = hashlib.sha256(f.cpu().numpy().astype(np.float64).tobytes() + t.cpu().numpy().astype(np.int32).tobytes())
    out[name] = {"ms_median": float(np.median(ms)), "ms_min": float(min(ms)), "ms_max": float(max(ms)),
                 "outputs_sha256": digest.hexdigest()}
print("RESULT " + json.dumps(out))
"""


def run(lib, cases, env_extra, steps):
    env = {k: v for k, v in os.environ.items() if not k.startswith("SGMM_ROLLOUT_")}
    env.update(env_extra)
    code = CHILD.replace("ROOT", repr(ROOT)).replace("__LIB__", repr(os.path.abspath(lib)))
    code = code.replace("CASES", repr(cases)).replace("STEPS", str(steps))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    if r.returncode != 0 or not line:
        raise SystemExit(f"child failed ({lib}, {cases}):\n{r.stdout[-2000:]}\n{r.stderr[-2000:]}")
    return json.loads(line[0][7:])


def main():
    if len(sys.argv) < 3:
        raise SystemExit(__doc__)
    libs = {"old": sys.argv[1], "new": sys.argv[2]}
    pairs = int(sys.argv[3]) if len(sys.argv) > 3 else 5
    out_path = sys.argv[4] if len(sys.argv) > 4 else None
    # (cases, environment) per process; SGMM_ROLLOUT_CHAINS is read once per process, so its shape runs alone
    groups = [(["p4096", "p592_u1", "p4096_u2", "adv2048"], {}), (["p4096_1ch"], {"SGMM_ROLLOUT_CHAINS": "1"})]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    runs = {k: [] for k in libs}
    for i in range(pairs):
        for k, lib in libs.items():
            res = {}
            for cases, env in groups:
                res.update(run(lib, cases, env, 20))
            runs[k].append(res)
            print(k, i, json.dumps(res), flush=True)
    summary = {"device": smi, "pairs": pairs, "steps_per_process": 20, "libraries": libs, "shapes": {}}
    for case in runs["old"][0]:
        row = {}
        for k in libs:
            med = [r[case]["ms_median"] for r in runs[k]]
            row[k] = {"ms_median_per_process": med, "ms_median": sorted(med)[len(med) // 2], "spread_ms": [min(med), max(med)]}
        row["combined_spread_ms"] = [min(row[k]["spread_ms"][0] for k in libs), max(row[k]["spread_ms"][1] for k in libs)]
        row["new_minus_old_ms"] = row["new"]["ms_median"] - row["old"]["ms_median"]
        row["new_median_within_old_spread"] = row["old"]["spread_ms"][0] <= row["new"]["ms_median"] <= row["old"]["spread_ms"][1]
        row["same_outputs_every_process"] = len({r[case]["outputs_sha256"] for k in libs for r in runs[k]}) == 1
        summary["shapes"][case] = row
    print(json.dumps(summary, indent=1))
    if out_path:
        with open(out_path, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
