#!/usr/bin/env python
"""bench.py -- population env-steps/s of the signal-gated market-making rollout on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one full population rollout (BASELINE.json configs[1]: P = 4096 individuals per GPU x
T = 14 400 bars = 60 synthetic 510300-shaped days, H = 32, no fee, phi = 1e-4): every individual's
policy MLP + quantisation + FPT env step for every bar, fitness and trade count out.  At N > 1 the
population is sharded by contiguous global index (weak scaling: 4096 individuals per GPU) and each
step ends with the ONE all-gather of the packed fitness / trade block that a sharded GA generation performs.

--dump-outputs DIR writes, after the timed steps, what the last timed step returned -- fitness and trade count of the
whole population, for the exact rollout and for each tensor-core precision -- as DIR/<name>.npy in float64.  The inputs
are seeded, so two builds of the project can be compared array for array.

  value   whole-job env-steps/s, genomes and bars resident in HBM, CUDA-event timed per step
  e2e     the same through the host-buffer C-ABI entries: pinned host genomes H2D + kernel + fitness/trades D2H
          inside the timed region, every step.  value = the pipelined entry (sgmm_rollout_population_host_async:
          batch k+1 uploads under batch k's kernel); sync_value = one synchronous call per step
  roofline  FP32 CUDA-core roofline (SURVEY.md 8d: compute-bound; 2368 algorithmic FLOP / env-step)
            against the FFMA peak measured live on this device; hbm sub-object for the bar/genome stream
  tensor_core_h32   the same workload through the tensor-core rollout (sgmm_tc32.cu)
  configs   BASELINE.json configs[2..4]: adversarial co-training (2048 + 2048), H = 256 with fee at 16 384 x 28 800,
            and 65 536 x 60 000 strong-scaled over the ranks through ShardedGA (GA generations/s, bit-identity flag)
  cpu_baseline / --impl reference   the UNMODIFIED reference (oracle/_ref, staged from /root/reference by build())
            running its own Pool.starmap(evaluate_individual) on the box's host cores; the C oracle port as a
            second figure
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

P_PER_GPU = 4096
N_DAYS = 60
HIDDEN = 32
PHI, TICK, FEE = 1e-4, 0.001, 0.0
FLOP_PER_STEP = 2368.0               # SURVEY.md 8d: 2*(3H + H^2 + 2H) at H = 32
FLOP_PER_STEP_ADV = 2488.0           # + the adversary's (36 + 24) MACs
FLOP_PER_STEP_H256 = 133632.0
METRIC = "population_env_steps_per_sec"
UNIT = "env-steps/s"
REF_SAMPLE_BARS = 2400               # 10 days: the reference arm's bounded sample of the 60-day bundle


def workload_config(n_gpus):
    return {"workload": "configs[1]: DRL agent, population 4096 per GPU, 60 synthetic 510300-shaped days "
                        "(T=14400 bars), H=32 MLP 3-32-32-2, no fee, phi=1e-4, tick=0.001",
            "population_per_gpu": P_PER_GPU, "population_total": P_PER_GPU * n_gpus, "bars": N_DAYS * 240,
            "hidden": HIDDEN, "fee_rate": FEE, "phi": PHI, "sharding": f"population x{n_gpus} (weak)",
            "l2": "256 MiB device memset between timed steps (flushes the 126 MB L2); per-step CUDA events "
                  "exclude the flush"}


def make_inputs(p_total):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(N_DAYS)
    stats = synthetic.train_stats_of(bundle)
    master, genomes = synthetic.policy_like_genomes(p_total, HIDDEN, seed=0, sigma=0.05, out_scale=1.0)
    return bundle, stats, master, genomes


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows[-3:]]
        sm, smax, reasons = [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU arms: the unmodified reference (oracle/_ref) and the C oracle port
# ------------------------------------------------------------------------------------------------
def cpu_port_rate(bundle, stats, genomes, target_seconds, threads=0):
    """env-steps/s of the CPU oracle port on a bounded sample (all host threads)."""
    from oracle import oracle
    z1, z2 = oracle.normalise(bundle, stats)
    bz = (z1, z2) + tuple(bundle[2:])
    cores = threads or oracle.max_threads()
    T = len(z1)
    probe_n = max(cores, 8)
    t0 = time.perf_counter()
    oracle.rollout_population(bz, PHI, TICK, FEE, genomes=genomes[:probe_n], nthreads=cores)
    probe = time.perf_counter() - t0
    n = int(max(probe_n, min(genomes.shape[0], probe_n * target_seconds / max(probe, 1e-3))))
    n = max(cores, (n // cores) * cores)
    n = min(n, genomes.shape[0])
    t0 = time.perf_counter()
    fit, trd = oracle.rollout_population(bz, PHI, TICK, FEE, genomes=genomes[:n], nthreads=cores)
    dt = time.perf_counter() - t0
    return n * T / dt, cores, n, T, dt, fit


def ref_staged():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import stage_ref
        return stage_ref.staged()
    finally:
        sys.path.pop(0)


def run_ref_subprocess(bundle, stats, genomes, *, bars, mode, procs, torch_threads, steps, warmup, timeout=900):
    """Run oracle/run_ref.py (the unmodified reference from oracle/_ref) on `genomes` x the first `bars` bars.
    Returns (seconds per timed step, fitness, trades)."""
    with tempfile.TemporaryDirectory() as d:
        keys = ("s1", "s2", "mid_next", "best_ask", "best_bid", "buy_max", "sell_min")
        np.savez(os.path.join(d, "in.npz"), **{k: np.asarray(a)[:bars] for k, a in zip(keys, bundle)},
                 s1_m=stats["s1_m"], s1_s=stats["s1_s"], s2_m=stats["s2_m"], s2_s=stats["s2_s"],
                 genomes=genomes, phi=PHI, tick=TICK, fee=FEE, use_arl=False)
        cmd = [sys.executable, os.path.join(ROOT, "oracle", "run_ref.py"), "--in", os.path.join(d, "in.npz"),
               "--out", os.path.join(d, "out.npz"), "--mode", mode, "--procs", str(procs),
               "--torch-threads", str(torch_threads), "--steps", str(steps), "--warmup", str(warmup)]
        env = dict(os.environ, CUDA_VISIBLE_DEVICES="")          # the reference is a CPU program
        subprocess.run(cmd, check=True, timeout=timeout, env=env, stdout=subprocess.DEVNULL)
        o = np.load(os.path.join(d, "out.npz"))
        return o["seconds"].copy(), o["fitness"].copy(), o["trades"].copy()


def reference_rates(bundle, stats, genomes, steps, warmup, per_step_individuals_per_core=16):
    """The reference's own population evaluation (Env/drl_engine.py:91,104-115) on the box's host cores.
    Headline = Pool over ALL host cores with one torch thread per worker (the strongest configuration of the unmodified
    code); also the as-shipped Pool(8) with torch's default threads and a single process with one thread."""
    cores = os.cpu_count() or 8
    n = min(genomes.shape[0], per_step_individuals_per_core * cores)
    secs, fit, trd = run_ref_subprocess(bundle, stats, genomes[:n], bars=REF_SAMPLE_BARS, mode="pool", procs=cores,
                                        torch_threads=1, steps=steps, warmup=warmup)
    out = {"value": n * REF_SAMPLE_BARS * len(secs) / float(secs.sum()), "cores": cores, "individuals": n,
           "bars": REF_SAMPLE_BARS, "seconds": [float(x) for x in secs]}
    try:        # as shipped: Pool(processes=8), torch default intra-op threads in every worker
        n8 = min(genomes.shape[0], 32)
        s8, _, _ = run_ref_subprocess(bundle, stats, genomes[:n8], bars=REF_SAMPLE_BARS, mode="pool", procs=8,
                                      torch_threads=0, steps=1, warmup=0)
        out["as_shipped_pool8"] = {"value": n8 * REF_SAMPLE_BARS / float(s8[0]), "individuals": n8, "bars": REF_SAMPLE_BARS,
                                   "note": "Pool(processes=8), torch default threads per worker (Env/drl_engine.py:91 verbatim)"}
        n1 = 4
        s1, _, _ = run_ref_subprocess(bundle, stats, genomes[:n1], bars=REF_SAMPLE_BARS, mode="single", procs=1,
                                      torch_threads=1, steps=1, warmup=0)
        out["single_process_1thread"] = {"value": n1 * REF_SAMPLE_BARS / float(s1[0]), "individuals": n1, "bars": REF_SAMPLE_BARS}
    except Exception as e:          # secondary figures only
        out["secondary_error"] = str(e)
    return out, fit, trd


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    bundle, stats, master, genomes = make_inputs(P_PER_GPU)
    port_rate, port_cores, pn, pT, pdt, _ = cpu_port_rate(bundle, stats, genomes, target_seconds=4.0)
    port = {"value": port_rate, "unit": UNIT, "cores": port_cores, "kind": "port",
            "sample": f"{pn} individuals x {pT} bars in {pdt:.1f} s (C oracle port, pthreads)"}
    if ref_staged():
        r, _, _ = reference_rates(bundle, stats, genomes, steps=args.steps, warmup=args.warmup)
        value, kind, cores = r["value"], "reference", r["cores"]
        total = sum(r["seconds"])
        sample = (f"{r['individuals']} individuals x {r['bars']} bars per step: the unmodified reference (oracle/_ref) running "
                  f"Pool({cores}).starmap(evaluate_individual) with one torch thread per worker")
        extra = {k: r[k] for k in ("as_shipped_pool8", "single_process_1thread", "secondary_error") if k in r}
        nsteps = len(r["seconds"])
    else:       # oracle/_ref did not travel (never the case after build() where /root/reference exists): the C port
        rates = []
        for i in range(args.warmup + args.steps):
            rate, cores, n, T, dt, _ = cpu_port_rate(bundle, stats, genomes, target_seconds=max(2.0, 20.0 / max(1, args.steps)))
            if i >= args.warmup:
                rates.append((n * T, dt))
        total = sum(r[1] for r in rates)
        value, kind, nsteps = sum(r[0] for r in rates) / total, "port", len(rates)
        sample = f"{n} individuals x {T} bars per step (C oracle port, pthreads over {cores} host threads; oracle/_ref not staged)"
        extra = {}
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * total / max(1, nsteps), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32 policy / f64 env", "data": "synthetic",
           "config": workload_config(args.gpus),
           "cpu_baseline": dict({"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                                 "c_port": port}, **extra),
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


def traffic_for(kernel, P, T):
    """dram bytes of one launch of `kernel` at (P, T) from the committed ncu capture summary, else None."""
    try:
        rows = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        for r in rows:
            if r.get("kernel") == kernel and r.get("P") == P and r.get("T") == T:
                return r.get("dram_bytes"), r.get("source")
    except Exception:
        pass
    return None, None


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import sgmm_b200
    from sgmm_b200 import _lib, synthetic
    from sgmm_b200.engine import DeviceGA
    from sgmm_b200.dist import ShardedGA

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    p_total = P_PER_GPU * n_gpus
    bundle, stats, master, genomes_all = make_inputs(p_total)
    first = rank * P_PER_GPU
    genomes = genomes_all[first:first + P_PER_GPU]
    T = len(bundle[0])
    G = HIDDEN * HIDDEN + 7 * HIDDEN + 2
    bun = sgmm_b200.Bundle.from_arrays(bundle, stats, TICK, device=local)
    g_dev = torch.from_numpy(genomes).to(dev)
    g_pin = torch.from_numpy(genomes).pin_memory()
    outs_pin = [(torch.empty(P_PER_GPU, dtype=torch.float64).pin_memory(), torch.empty(P_PER_GPU, dtype=torch.int32).pin_memory())
                for _ in range(2)]
    fit_pin, trd_pin = outs_pin[0]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # the sharded step's exchange: ONE all-gather of the packed (fitness f64 | trades i32) block per rank
    blk = P_PER_GPU * 12
    gather = torch.empty(world * blk, dtype=torch.uint8, device=dev)
    mine = gather[rank * blk:(rank + 1) * blk]
    fit_view = mine[:P_PER_GPU * 8].view(torch.float64)
    trd_view = mine[P_PER_GPU * 8:].view(torch.int32)

    import ctypes as C
    L = _lib.lib()
    mm_dev = _lib.Population(HIDDEN, 0, P_PER_GPU, g_dev.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    mm_pin = _lib.Population(HIDDEN, 0, P_PER_GPU, g_pin.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    TC_MODES = (("tf32", 2), ("f16", 3), ("bf16", 1))
    prm = {"f32": _lib.RolloutParams(PHI, FEE, 0, 0, 0, 0)}
    prm.update({name: _lib.RolloutParams(PHI, FEE, code, 0, 0, 0) for name, code in TC_MODES})

    def step_device(mode="f32"):
        st = C.c_void_p(torch.cuda.current_stream(local).cuda_stream)
        _lib.check(L.sgmm_rollout_population(bun.handle, C.byref(mm_dev), None, C.byref(prm[mode]), fit_view.data_ptr(),
                                             trd_view.data_ptr(), st))
        if world > 1:
            dist.all_gather_into_tensor(gather, mine)

    def step_e2e_sync(mode="f32"):
        st = C.c_void_p(torch.cuda.current_stream(local).cuda_stream)
        _lib.check(L.sgmm_rollout_population_host(bun.handle, C.byref(mm_pin), None, C.byref(prm[mode]), fit_pin.data_ptr(),
                                                  trd_pin.data_ptr(), st))
        return float(fit_pin[0])

    def run_e2e_pipelined(mode, steps):
        """K batches through sgmm_rollout_population_host_async, two in flight; every batch has its own H2D of the
        genomes and D2H of fitness / trades.  Returns wall seconds (first submit .. last result read)."""
        tickets = []
        acc = 0.0
        t0 = time.perf_counter()
        for k in range(steps):
            f, t = outs_pin[k % 2]
            if len(tickets) == 2:
                tk, fo = tickets.pop(0)
                _lib.check(L.sgmm_rollout_wait(bun.handle, tk))
                acc += float(fo[0])                                  # the host reads the step's result
            tk = C.c_int32(-1)
            _lib.check(L.sgmm_rollout_population_host_async(bun.handle, C.byref(mm_pin), None, C.byref(prm[mode]),
                                                            f.data_ptr(), t.data_ptr(), C.byref(tk)))
            tickets.append((tk.value, f))
        for tk, fo in tickets:
            _lib.check(L.sgmm_rollout_wait(bun.handle, tk))
            acc += float(fo[0])
        return time.perf_counter() - t0, acc

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def last_outputs(prefix=""):
        """Fitness and trades of the whole population as the last device step left them in the gathered block."""
        rows = gather.view(world, blk)
        return {prefix + "fitness": rows[:, :P_PER_GPU * 8].contiguous().view(torch.float64).flatten().cpu().numpy(),
                prefix + "trades": rows[:, P_PER_GPU * 8:].contiguous().view(torch.int32).flatten().cpu().numpy().astype(np.float64)}

    def time_device(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for (e0, e1) in evs:
            flush.fill_(1)                                  # L2 flush, outside the step's event pair
            e0.record()
            fn()
            e1.record()
        barrier()
        return [e0.elapsed_time(e1) for (e0, e1) in evs]

    # ---- warm-up -------------------------------------------------------------------------------
    W = max(3, args.warmup)
    for _ in range(W):
        for mode in prm:
            step_device(mode)
            step_e2e_sync(mode)
    for mode in prm:
        run_e2e_pipelined(mode, 3)
    barrier()
    fp32_peak = sgmm_b200.measure_fp32_peak(local)

    # ---- device-timed steps (the contract's timed region) ---------------------------------------
    K = args.steps
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.25)
    t_wall0 = time.perf_counter()
    step_ms = time_device(step_device, K)
    t_wall1 = time.perf_counter()
    checksum = float(fit_view.sum().item())
    outputs = last_outputs()
    # ---- end-to-end steps (host buffers, copies inside the timed region) ----------------------
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        step_e2e_sync()
    barrier()
    e2e_sync_s = time.perf_counter() - t0
    barrier()
    e2e_pipe_s, _ = run_e2e_pipelined("f32", K)
    barrier()
    # ---- the same measurements for the tensor-core rollout, per precision ---------------------------
    tc_raw = {}
    for mode, _ in TC_MODES:
        ms = time_device(lambda m=mode: step_device(m), K)
        csum = float(fit_view.sum().item())
        outputs.update(last_outputs(f"tensor_core_{mode}_"))
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            step_e2e_sync(mode)
        barrier()
        es = time.perf_counter() - t0
        ep, _ = run_e2e_pipelined(mode, K)
        barrier()
        tc_raw[mode] = {"ms": ms, "e2e_sync_s": es, "e2e_pipe_s": ep, "checksum": csum}
    clocks = sampler.stop(t_wall0, time.perf_counter())

    vals = [sum(step_ms), e2e_sync_s, e2e_pipe_s]
    for mode, _ in TC_MODES:
        vals += [sum(tc_raw[mode]["ms"]), tc_raw[mode]["e2e_sync_s"], tc_raw[mode]["e2e_pipe_s"]]
    tt = torch.tensor(vals, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_ms, e2e_sync_s, e2e_pipe_s = tt[0].item(), tt[1].item(), tt[2].item()
    for k, (mode, _) in enumerate(TC_MODES):
        tc_raw[mode]["dev_ms"], tc_raw[mode]["e2e_sync_s"], tc_raw[mode]["e2e_pipe_s"] = (tt[3 + 3 * k].item(), tt[4 + 3 * k].item(),
                                                                                        tt[5 + 3 * k].item())

    # ---- GA generations/s at every N (ask + rollout + all-gather + tell + validation rollout + select) ----
    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def ga_rate_of(train_b, val_b, pop, ngen, master_np, precision=None, hidden=32, fee=FEE, use_graph=None):
        """Generations/s: single rank = CUDA-graph replay of the whole generation; sharded = eager (evaluate, ONE NCCL
        all-gather, select).  Wall time between device synchronisations, max over ranks."""
        def make(shard=None):
            return DeviceGA(master_np, None, pop_size=pop, sigma=0.05, phi=PHI, fee_rate=fee, use_arl=False, seed=0,
                            max_generations=2 * ngen + 6, device=local, precision=precision, hidden=hidden, shard=shard)
        if world > 1:
            runner = ShardedGA(make, pop)
            ga, run = runner.ga, (lambda: runner.generation(train_b, val_b))
        else:
            ga = make()
            run = lambda: ga.generation(train_b, val_b)       # noqa: E731
        run(); run()
        barrier()
        if world == 1 and (use_graph if use_graph is not None else True):
            graph = ga.capture(train_b, val_b)
            run = graph.replay
            run()
        barrier()
        t0 = time.perf_counter()
        for _ in range(ngen):
            run()
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        colls = getattr(runner, "collectives", 0) if world > 1 else 0
        h = ga.history()
        ga.close()
        return ngen / dt, (colls / (ngen + 2) if world > 1 else 0), float(h["val_f"][-1])

    val = sgmm_b200.Bundle.from_arrays(synthetic.synthetic_bundle(12, first_day=N_DAYS), stats, TICK, device=local)
    ga_rate, ga_colls, _ = ga_rate_of(bun, val, p_total, 5, master)
    ga_rate_tc = {mode: ga_rate_of(bun, val, p_total, 5, master, precision=mode)[0] for mode, _ in TC_MODES}
    ga_small = ga_small_arl = None
    if world == 1:
        # the reference's own scale (BASELINE configs[0]): population 50, one training day, one validation day
        d1 = synthetic.synthetic_bundle(1, first_day=200)
        st1 = synthetic.train_stats_of(d1)
        t1 = sgmm_b200.Bundle.from_arrays(d1, st1, TICK, device=local)
        v1 = sgmm_b200.Bundle.from_arrays(synthetic.synthetic_bundle(1, first_day=201), st1, TICK, device=local)
        ga_small = ga_rate_of(t1, v1, 50, 200, master)[0]
        # the reference's default pipeline co-trains the adversary (pipeline/agent_trainer.py:79: USE_ARL=True)
        adv0 = (np.random.default_rng(4).standard_normal(1250) * 0.5).astype(np.float32)
        ga0 = DeviceGA(master, adv0, pop_size=50, sigma=0.05, phi=PHI, fee_rate=FEE, use_arl=True, seed=0, max_generations=420, device=local)
        ga0.generation(t1, v1); ga0.generation(t1, v1); torch.cuda.synchronize()
        gr0 = ga0.capture(t1, v1); gr0.replay(); torch.cuda.synchronize()
        t0_ = time.perf_counter()
        for _ in range(200):
            gr0.replay()
        torch.cuda.synchronize()
        ga_small_arl = 200 / (time.perf_counter() - t0_)
        ga0.close()

    # ---- BASELINE.json configs[2..4] -------------------------------------------------------------
    configs = {}
    sms = torch.cuda.get_device_properties(local).multi_processor_count
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    tensor_peak = peaks.get("bf16_tflops_sustained", 1400.0)

    def guarded(name, fn):
        try:
            configs[name] = fn()
        except Exception as e:          # a secondary section must never take the headline down
            configs[name] = {"error": f"{type(e).__name__}: {e}"}

    def config3():
        """Adversarial co-training: 2048 market makers each meeting its own adversary (2048 adversary genomes), the
        displacement fused into the step; per GPU, weak-scaled like the headline."""
        P3 = 2048
        adv = (np.random.default_rng(3).standard_normal((P3, 1250)) * 0.5).astype(np.float32)
        a_dev = torch.from_numpy(adv).to(dev)
        g3 = g_dev[:P3].contiguous()
        out = {}
        for mode in ("f32",) + tuple(m for m, _ in TC_MODES if getattr(sgmm_b200.engine, "TC_ADVERSARY", False)):
            def run(m=mode):
                sgmm_b200.rollout_population(bun, g3, a_dev, phi=PHI, fee_rate=FEE, precision=m)
            run(); run()
            ms = time_device(run, min(K, 5))
            per = max_over_ranks(sum(ms)) / len(ms)
            v = P3 * T * n_gpus / (per * 1e-3)
            tf = FLOP_PER_STEP_ADV * P3 * T / (per * 1e-3) / 1e12
            out[mode] = {"value": v, "unit": UNIT, "ms_per_step": per,
                         "roofline": ({"bound": "fp32", "achieved": tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": tf / fp32_peak}
                                      if mode == "f32" else
                                      {"bound": "tensor", "achieved": tf, "peak": tensor_peak, "unit": "TFLOP/s", "frac": tf / tensor_peak})}
        return dict(out, workload=f"configs[2]: {P3} market makers + {P3} adversaries per GPU x {T} bars, H=32, adversary "
                                  "displacement fused in the step", algorithmic_flop_per_env_step=FLOP_PER_STEP_ADV)

    def config4():
        """With-fee variant, 256x256 hidden layers on tcgen05, population 16384, 120 days -- full size, rank 0's GPU only."""
        P4, D4, fee4 = 16384, 120, 3e-4
        b4 = synthetic.synthetic_bundle(D4, first_day=300)
        s4 = synthetic.train_stats_of(b4)
        bun4 = sgmm_b200.Bundle.from_arrays(b4, s4, TICK, device=local)
        val4 = sgmm_b200.Bundle.from_arrays(synthetic.synthetic_bundle(24, first_day=300 + D4), s4, TICK, device=local)
        m256, _ = synthetic.policy_like_genomes(1, hidden=256, seed=0)
        md = torch.from_numpy(m256).to(dev)
        T4 = bun4.T

        def run():
            return sgmm_b200.rollout_seeded(bun4, md, count=P4, sigma=0.05, seed=1, generation=0, phi=PHI, fee_rate=fee4, hidden=256)
        run(); torch.cuda.synchronize()
        ms = time_device(run, 5)
        per = sum(ms) / len(ms)
        st4 = P4 * T4
        alg = st4 * FLOP_PER_STEP_H256 / per / 1e9
        rate, _, vf = ga_rate_of(bun4, val4, P4, 3, m256, precision="bf16", hidden=256, fee=fee4, use_graph=False) if world == 1 else (None, 0, None)
        bun4.close(); val4.close()
        return {"workload": f"configs[3]: population {P4} x {T4} bars ({D4} days), H=256 MLP 3-256-256-2, fee_rate {fee4}, seeded children",
                "kernel": "spec256_kernel (tcgen05 kind::f16: f16 operands, f16 layer-2 accumulator in TMEM, fp32 output layer; "
                          "5-inventory speculation) + account_kernel (fp64 env arithmetic)",
                "value": st4 / per * 1e3, "unit": UNIT, "ms_per_step": per, "per_step_ms": ms, "launches_timed": len(ms),
                "roofline": {"bound": "tensor", "achieved": alg, "peak": tensor_peak, "unit": "TFLOP/s", "frac": alg / tensor_peak,
                             "executed_hidden_tflops": st4 * (128 / 25) * 131072 / per / 1e9,
                             "algorithmic_flop_per_env_step": FLOP_PER_STEP_H256},
                "ga_generations_per_sec": rate, "ga_last_val_f": vf}

    def config5():
        """Population scaling sweep: 65536 individuals x 250 days, STRONG-scaled over the ranks through
        ShardedGA.generation (evaluate shard + ONE NCCL all-gather + identical select on every rank)."""
        P5, D5 = 65536, 250
        b5 = synthetic.synthetic_bundle(D5, first_day=500)
        s5 = synthetic.train_stats_of(b5)
        bun5 = sgmm_b200.Bundle.from_arrays(b5, s5, TICK, device=local)
        val5 = sgmm_b200.Bundle.from_arrays(synthetic.synthetic_bundle(25, first_day=500 + D5), s5, TICK, device=local)
        rate, colls, vf = ga_rate_of(bun5, val5, P5, 3, master, use_graph=False)
        out = {"workload": f"configs[4]: population {P5} x {bun5.T} bars ({D5} days), H=32, no fee, seeded children; population "
                           f"sharded over {world} rank(s), strong scaling",
               "scaling": "strong", "ga_generations_per_sec": rate, "ms_per_generation": 1e3 / rate,
               "value": P5 * bun5.T * rate, "unit": UNIT, "collectives_per_generation": colls, "ga_last_val_f": vf}
        bun5.close(); val5.close()
        return out

    def sharded_identity():
        """The sharded GA must reproduce the single-rank GA bit for bit (children come from the counter-based stream):
        every rank runs both on a small problem and compares history and masters."""
        tb = synthetic.synthetic_bundle(3, first_day=80)
        vb = synthetic.synthetic_bundle(1, first_day=83)
        s = synthetic.train_stats_of(tb)
        tr = sgmm_b200.Bundle.from_arrays(tb, s, TICK, device=local)
        va = sgmm_b200.Bundle.from_arrays(vb, s, TICK, device=local)
        m0, _ = synthetic.policy_like_genomes(1, seed=31)
        a0 = (np.random.default_rng(6).standard_normal(1250) * 0.5).astype(np.float32)
        pop, gens = 1001, 6          # not divisible by the world size on purpose
        kw = dict(pop_size=pop, sigma=0.05, phi=PHI, fee_rate=0.0, use_arl=True, seed=99, max_generations=gens, patience=2, device=local)
        sh = ShardedGA(lambda shard: DeviceGA(m0, a0, shard=shard, **kw), pop)
        ref = DeviceGA(m0, a0, **kw)
        for _ in range(gens):
            sh.generation(tr, va)
            ref.generation(tr, va)
        h, hr = sh.ga.history(gens), ref.history(gens)
        ok = all(np.array_equal(h[k].view(np.uint8), hr[k].view(np.uint8)) for k in h)
        ok = ok and all(np.array_equal(x, y) for x, y in zip(sh.ga.masters(), ref.masters()))
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        sh.ga.close(); ref.close()
        return bool(flag.item())

    def config0():
        """The reference's own scale (configs[0]): population 50 (Env/drl_engine.py:70), no fee, phi 1e-4 -- one day and the
        15-day training set of the replication report; seeded children, CUDA-graph replay (device time, rank 0's GPU)."""
        out = {"workload": "configs[0]: population 50, H=32, no fee, phi=1e-4; one synthetic day (240 bars) and 15 days (3600 bars)"}
        md = torch.from_numpy(master).to(dev)
        for days in (1, 15):
            b0 = synthetic.synthetic_bundle(days, first_day=200)
            bun0 = sgmm_b200.Bundle.from_arrays(b0, synthetic.train_stats_of(b0), TICK, device=local)
            run = lambda: sgmm_b200.rollout_seeded(bun0, md, count=50, sigma=0.05, seed=1, generation=0, phi=PHI)      # noqa: E731
            run(); run(); torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                for _ in range(10):
                    run()
            gr.replay(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); gr.replay(); e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 10
            out[f"{days}_day"] = {"bars": bun0.T, "ms_per_rollout": ms, "value": 50 * bun0.T / ms * 1e3, "unit": UNIT}
            bun0.close()
        return out

    if world == 1:
        guarded("config0_reference_scale", config0)
    guarded("config3_adversarial", config3)
    if world == 1:
        guarded("config4_h256_fee", config4)
    guarded("config5_population_sweep", config5)
    if world > 1:
        guarded("sharded_ga_bit_identical", sharded_identity)

    if rank == 0:
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        steps_per_step = p_total * T
        value = steps_per_step * K / (dev_ms * 1e-3)
        kernel_s = (dev_ms / K) * 1e-3                       # the rollout kernel is the whole device step
        achieved_tflops = FLOP_PER_STEP * P_PER_GPU * T / kernel_s / 1e12
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        hbm_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        alg_bytes = P_PER_GPU * G * 4 + T * 48 + P_PER_GPU * 12       # genomes once + bars once + outputs
        traffic, traffic_src = traffic_for("rollout_kernel_h32", P_PER_GPU, T)
        # ---- cpu_baseline: the unmodified reference on this box's host cores (N = 1 only), the C port beside it
        cpu = None
        if world == 1:
            port_rate, port_cores, pn, pT, pdt, _ = cpu_port_rate(bundle, stats, genomes, target_seconds=6.0)
            port = {"value": port_rate, "unit": UNIT, "cores": port_cores, "kind": "port",
                    "sample": f"{pn} individuals x {pT} bars in {pdt:.1f} s (C oracle port, pthreads)"}
            cpu = port
            if ref_staged():
                try:
                    r, _, _ = reference_rates(bundle, stats, genomes, steps=1, warmup=0, per_step_individuals_per_core=32)
                    cpu = dict({"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "reference",
                                "sample": f"{r['individuals']} individuals x {r['bars']} bars in {r['seconds'][0]:.1f} s: the unmodified "
                                          f"reference (oracle/_ref) running Pool({r['cores']}).starmap(evaluate_individual), one torch "
                                          "thread per worker", "c_port": port},
                               **{k: r[k] for k in ("as_shipped_pool8", "single_process_1thread", "secondary_error") if k in r})
                except Exception as e:
                    cpu = dict(port, reference_error=str(e))
        # tensor-core rollout: algorithmic FLOPs as above; EXECUTED tensor FLOPs per unit of two 128-row tiles
        # (= 50 env-steps): L1 128x64x16, L2 2 x 128x32x48, L3 2 x 128x16x48, x2 FLOP per MAC
        tc_exec_flop_per_step = {"bf16": 2.0 * (128 * 64 * 16 + 2 * 128 * 32 * 48 + 2 * 128 * 16 * 48) / 50.0,
                                 "tf32": 2.0 * (128 * 64 * 16 + 2 * 128 * 32 * 40 + 2 * 128 * 16 * 40) / 50.0}
        tc_exec_flop_per_step["f16"] = tc_exec_flop_per_step["bf16"]
        tol = {"bf16": "policy outputs within 0.12 tick of the fp32 oracle; 3 of 1920 offsets of the golden ARL audit set flip, all at "
                       "near-ties of the fp32 result",
               "f16": "f16 operands, f16 accumulators for layers 1-2 (fp32 for the output layer): policy outputs within 0.03 tick of "
                      "the fp32 oracle (measured 0.0105); 0 of 1920 offsets of the golden ARL audit set flip",
               "tf32": "policy outputs within 0.03 tick of the fp32 oracle (measured 0.011); 0 of 1920 offsets of the golden ARL "
                       "audit set flip: the reference's shipped backtest is reproduced exactly (actions, trades, fitness)"}
        tc = {"kernel": "tc32_kernel (sgmm_tc32.cu): all three policy layers on tcgen05 (accumulators in TMEM, A operands chained "
                        "through tensor memory), 5-inventory speculation, grouped GEMM over 14 individuals per CTA; "
                        "tests/test_gpu_tc32.py states the tolerances; the env step given the offsets is bit-exact"}
        h2d, d2h = P_PER_GPU * G * 4 * n_gpus, P_PER_GPU * 12 * n_gpus
        for mode, _ in TC_MODES:
            r = tc_raw[mode]
            tc_value = steps_per_step * K / (r["dev_ms"] * 1e-3)
            tc_kernel_s = (r["dev_ms"] / K) * 1e-3
            tc_alg_tflops = FLOP_PER_STEP * P_PER_GPU * T / tc_kernel_s / 1e12
            tc[mode] = {"value": tc_value, "unit": UNIT, "ms_per_step": r["dev_ms"] / K, "per_step_ms": r["ms"],
                        "speedup_vs_exact_kernel": tc_value / value, "tolerance": tol[mode],
                        "e2e": {"value": steps_per_step * K / r["e2e_pipe_s"], "unit": UNIT, "ms_per_step": 1e3 * r["e2e_pipe_s"] / K,
                                "sync_value": steps_per_step * K / r["e2e_sync_s"], "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                        "roofline": {"bound": "tensor", "achieved": tc_alg_tflops, "peak": tensor_peak, "unit": "TFLOP/s",
                                     "frac": tc_alg_tflops / tensor_peak, "traffic": None,
                                     "executed_tflops": tc_exec_flop_per_step[mode] * P_PER_GPU * T / tc_kernel_s / 1e12,
                                     "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (tf32 nominal peak is half)"
                                                     if "bf16_tflops_sustained" in peaks else "fallback 1400"),
                                     "note": "algorithmic = 2368 FLOP/env-step; executed counts the 5-inventory speculation and the "
                                             "K / N padding"},
                        "ga_generations_per_sec": ga_rate_tc.get(mode), "checksum": r["checksum"]}
        launches = K * (1 + len(TC_MODES))
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": W,
            "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 policy (SGMM-F32 order, FFMA2) / int32 fills / f64 env", "data": "synthetic",
            "config": workload_config(n_gpus),
            "e2e": {"value": steps_per_step * K / e2e_pipe_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_pipe_s / K,
                    "entry": "sgmm_rollout_population_host_async + sgmm_rollout_wait (pinned host genomes in, fitness/trades out, every "
                             "step; two batches in flight so the H2D of step k+1 overlaps the kernel of step k; bundle resident)",
                    "sync_value": steps_per_step * K / e2e_sync_s, "sync_ms_per_step": 1e3 * e2e_sync_s / K,
                    "sync_entry": "sgmm_rollout_population_host (one synchronous call per step)"},
            "gpu_launches": launches,          # K exact-kernel + K tensor-core rollouts per mode in the device-timed regions
            "clocks": clocks,
            "roofline": {"bound": "fp32", "achieved": achieved_tflops, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": achieved_tflops / fp32_peak if fp32_peak else None,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "rollout_kernel_h32 (exact SGMM-F32 order)",
                         "algorithmic_flop_per_env_step": FLOP_PER_STEP,
                         "peak_source": "FFMA/FFMA2 peak measured live on this device by sgmm_measure_fp32_peak "
                                        "(MEASURED_PEAKS.json has no fp32 figure; theoretical 74.4 TFLOP/s at 1965 MHz)",
                         "note": "compute-bound on the FP32 CUDA-core pipe (SURVEY.md 8d); bound is neither hbm nor tensor. "
                                 "traffic = dram__bytes_read+write of one launch from the committed ncu capture of this (P, T) "
                                 "(profiles/traffic.json), null when no capture of this shape is committed",
                         "hbm": {"achieved": alg_bytes / kernel_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": alg_bytes / kernel_s / 1e9 / hbm_peak, "algorithmic_bytes_per_launch": alg_bytes,
                                 "peak_source": hbm_src}},
            "roofline_hbm": {"bound": "hbm", "achieved": alg_bytes / kernel_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": alg_bytes / kernel_s / 1e9 / hbm_peak, "traffic": traffic,
                             "note": "reported for completeness: the bar/genome stream is <0.1% of HBM peak by construction"},
            "cpu_baseline": cpu,
            "per_step_ms": step_ms,
            "ga_generations_per_sec": ga_rate,
            "ga_collectives_per_generation": ga_colls,
            "ga_workload": f"population {p_total} x {T} bars train + 2880 bars validation"
                           + (" (CUDA-graph replay)" if world == 1 else f" sharded over {world} ranks (eager: evaluate, one NCCL all-gather, select)"),
            "ga_generations_per_sec_config0_pop50_1day": ga_small,
            "ga_generations_per_sec_config0_pop50_1day_arl": ga_small_arl,
            "tensor_core_h32": tc,
            "configs": configs,
            "checksum": checksum,
        }
        emit(out)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(obj):
    """The ONE JSON line of the contract goes to the real stdout; everything libraries print while the
    benchmark runs (NCCL's version banner, for instance) was redirected to stderr."""
    line = json.dumps(obj) + "\n"
    if _REAL_STDOUT is None:
        sys.stdout.write(line); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line.encode())


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                      # fd 1 -> stderr for the duration of the run
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the CUDA path's outputs (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
