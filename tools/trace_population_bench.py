"""Time the population trace (sgmm_rollout_trace_population) with CUDA events.

    python tools/trace_population_bench.py [--out FILE] [--loop-reps N]

Shapes at T = 14 400 bars (60 synthetic days), phi 1e-4, fee 3e-4: P in {1, 50, 592, 4096} at H = 32 without and with the
adversary, P in {50, 592} at H = 256 (exact).  Each shape is timed with every column, with the four columns of
backtest_population (wealth, inventory, fill_buy, fill_sell) and with none (fitness and trades only), and set against
  - the exact population rollout of the same shape (sgmm_rollout_population; no outputs: the floor), and
  - P back-to-back sgmm_rollout_trace calls writing into rows of the same device columns (the loop this call replaces);
    timed at P <= 592, extrapolated linearly from the P = 592 loop above that and labelled so.
Output bytes per second count the columns written (120 B per individual and bar with every column, 20 B with the analytics
subset) against the 7.7 TB/s HBM3e figure of the data sheet.  A torch.profiler pass of the largest shapes splits the call
into its kernels.  Every timed call is preceded by a warm-up call of the same shape and by a 512 MB write that evicts the
126 MB L2.  The card's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import sgmm_b200  # noqa: E402
from exact256_bench import bun_of, card, flush_l2, timed  # noqa: E402
from spec256_adv_bench import kernel_times  # noqa: E402
from sgmm_b200 import _lib, synthetic  # noqa: E402
from sgmm_b200.engine import _TRACE_F32, _TRACE_I32, _stream  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
ANALYTICS = ("wealth", "inventory", "fill_buy", "fill_sell")
NAMES = [n for n, _ in _lib.Trace._fields_]


def col_bytes(names):
    return sum(4 if n in _TRACE_I32 or n in _TRACE_F32 else 8 for n in names)


def trace_loop(bun, g, a, cols, fit, trd, hidden, n):
    """n back-to-back sgmm_rollout_trace calls, individual i into row i of the columns."""
    L = _lib.lib()
    prm = _lib.RolloutParams(1e-4, 3e-4, 0, 0, 0, 0)
    st = _stream(bun.device)
    T = bun.T
    for i in range(n):
        tr = _lib.Trace(*[cols[k].data_ptr() + i * T * cols[k].element_size() if k in cols else None for k in NAMES])
        _lib.check(L.sgmm_rollout_trace(bun.handle, g[i].data_ptr(), hidden, None if a is None else a[i].data_ptr(), None,
                                        C.byref(prm), C.byref(tr), fit[i:].data_ptr(), trd[i:].data_ptr(), st))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--loop-reps", type=int, default=1)
    args = ap.parse_args()
    res = {"card": card(), "T": None, "rows": [], "kernels_ms": {}}
    print(res["card"], flush=True)
    bun = bun_of(60)
    T = bun.T
    res["T"] = T
    loop_592 = {}

    def row(r):
        res["rows"].append(r)
        print(r, flush=True)

    for hidden, use_adv, sizes in ((32, False, (1, 50, 592, 4096)), (32, True, (1, 50, 592, 4096)), (256, False, (50, 592)),
                                   (256, True, (50, 592))):
        for P in sizes:
            _, g = synthetic.policy_like_genomes(P, hidden=hidden, seed=P)
            g = torch.from_numpy(g).cuda()
            a = torch.from_numpy((np.random.default_rng(P).standard_normal((P, 1250)) * 0.6).astype(np.float32)).cuda() if use_adv else None
            kw = dict(phi=1e-4, fee_rate=3e-4, hidden=hidden)
            base = {"hidden": hidden, "adversary": use_adv, "P": P, "T": T}
            floor = timed(lambda: sgmm_b200.rollout_population(bun, g, a, precision="exact", **kw), 3)
            row(dict(base, case="exact rollout_population (floor, no outputs)", ms_median=round(floor[0], 3),
                     ms_min=round(floor[1], 3), ms_max=round(floor[2], 3)))
            for label, columns in (("all columns", None), ("analytics subset", ANALYTICS), ("no columns", ())):
                names = NAMES if columns is None else list(columns)
                ms = timed(lambda: sgmm_b200.rollout_trace_population(bun, g, a, columns=columns, **kw), 3)
                nbytes = P * T * col_bytes(names)
                row(dict(base, case=f"population trace, {label}", ms_median=round(ms[0], 3), ms_min=round(ms[1], 3),
                         ms_max=round(ms[2], 3), output_bytes=nbytes, output_TB_per_s=round(nbytes / ms[0] / 1e9, 3),
                         share_of_hbm=round(nbytes / ms[0] / 1e9 / (HBM_BYTES_PER_S / 1e12), 4),
                         over_floor=round(ms[0] / floor[0], 2)))
                if label == "all columns":
                    t_all = ms[0]
            if P > 1 and P <= 592:
                cols = {k: torch.empty(P, T, dtype=torch.int32 if k in _TRACE_I32 else (torch.float32 if k in _TRACE_F32 else
                                                                                        torch.float64), device="cuda")
                        for k in NAMES}
                fit = torch.empty(P, dtype=torch.float64, device="cuda")
                trd = torch.empty(P, dtype=torch.int32, device="cuda")
                ms = timed(lambda: trace_loop(bun, g, a, cols, fit, trd, hidden, P), args.loop_reps)
                f2, t2, c2 = sgmm_b200.rollout_trace_population(bun, g, a, **kw)
                same = bool(f2.equal(fit) and t2.equal(trd) and all(c2[k].equal(cols[k]) for k in NAMES))
                del cols, c2
                if P == 592:
                    loop_592[(hidden, use_adv)] = ms[0]
                row(dict(base, case="sequential rollout_trace loop, all columns", ms_median=round(ms[0], 3), ms_min=round(ms[1], 3),
                         ms_max=round(ms[2], 3), measured=True, population_speedup=round(ms[0] / t_all, 2),
                         identical_outputs=same))
            elif P > 592 and (hidden, use_adv) in loop_592:
                ms = loop_592[(hidden, use_adv)] * P / 592
                row(dict(base, case="sequential rollout_trace loop, all columns", ms_median=round(ms, 3), measured=False,
                         note="extrapolated linearly from the measured P = 592 loop", population_speedup=round(ms / t_all, 2)))
            if P == max(sizes):
                for label, columns in (("all columns", None), ("analytics subset", ANALYTICS), ("no columns", ())):
                    flush_l2()
                    kt = kernel_times(lambda: sgmm_b200.rollout_trace_population(bun, g, a, columns=columns, **kw))
                    res["kernels_ms"][f"H={hidden} adv={use_adv} P={P} {label}"] = kt
                    print(label, kt, flush=True)
            del g, a
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:                              # one row per line
            f.write('{"card": %s, "T": %d,\n "rows": [\n  ' % (json.dumps(res["card"]), res["T"]))
            f.write(",\n  ".join(json.dumps(r) for r in res["rows"]))
            f.write('],\n "kernels_ms": {\n  ')
            f.write(",\n  ".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in res["kernels_ms"].items()))
            f.write("}}\n")


if __name__ == "__main__":
    main()
