"""Population rollout, per-individual evaluation and the GA engine on the B200.

Reference surface kept verbatim (Env/drl_engine.py):
  ``evaluate_individual(mm_weights, adv_weights, bundle, phi, tick_size, fee_rate, train_stats,
  use_arl=False) -> (total_reward, trades)``                                           (:9-67)
  ``DRLEngine(pop_size, sigma, phi, tick_size, fee_rate, use_arl, save_dir)``, ``.mm_evolver``,
  ``.adv_evolver``, ``.train(train_bundle, val_bundle, train_stats, generations, output_prefix)
  -> (master_policy, history)``                                                        (:69-178)
plus the population-level calls the reference spells ``Pool.starmap`` (:104-115).
Everything computes through the C ABI of libsgmm_b200.so; nothing here touches ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import OrderedDict

import numpy as np
import torch

from . import _lib
from .bundle import Bundle
from .policy import NeuroEvolution, TradingPolicy, genome_len

ADV_SEED_FLIP = 0x8000000000000000       # adversary noise stream = seed with the top bit flipped


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


PRECISION_F32, PRECISION_BF16, PRECISION_TF32, PRECISION_F16, PRECISION_EXACT = 0, 1, 2, 3, 4


def _precision(precision, hidden):
    """None -> the default of the width: hidden=32 bit-exact SGMM-F32 path, hidden=256 tcgen05 path.
    "bf16" with hidden=32 selects the tensor-core rollout of sgmm_tc32.cu (all three layers on tcgen05).
    "exact" is SGMM-F32 order at any width the library builds: the F32 path at hidden=32, the CUDA-core policy-table
    path of sgmm_exact256.cu at hidden=256."""
    if precision is None:
        return PRECISION_BF16 if hidden == 256 else PRECISION_F32
    if precision in ("exact", PRECISION_EXACT):
        return PRECISION_F32 if hidden == 32 else PRECISION_EXACT
    if precision in ("f32", "fp32", PRECISION_F32):
        return PRECISION_F32
    if precision in ("bf16", "tensor", PRECISION_BF16):
        return PRECISION_BF16
    if precision in ("tf32", PRECISION_TF32):
        return PRECISION_TF32
    if precision in ("f16", "fp16", PRECISION_F16):
        return PRECISION_F16
    raise ValueError(f"unknown precision {precision!r}")


def _params(phi, fee_rate, units_per_lane=0, warps_per_cta=0, hidden=32, precision=None):
    prec = _precision(precision, hidden)
    return _lib.RolloutParams(float(phi), float(fee_rate), prec, 0, int(units_per_lane), int(warps_per_cta))


def _as_f32_matrix(x, width):
    """Accept a list of 1-D tensors (NeuroEvolution.ask), a 2-D tensor or ndarray."""
    if isinstance(x, (list, tuple)):
        x = torch.stack([torch.as_tensor(w, dtype=torch.float32).reshape(-1) for w in x])
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x, np.float32))
    x = x.to(torch.float32)
    if x.dim() == 1:
        x = x.reshape(1, -1)
    if x.shape[1] != width:
        raise ValueError(f"genome length {x.shape[1]} != {width}")
    return x.contiguous()


def _as_adv_matrix(x):
    """Adversary genomes: the reference's AdversaryPolicy.set_weights consumes the first 74 floats of whatever vector it
    is handed (models/model.py:52-57) -- a 1250-float TradingPolicy-sized child of the adversary evolver (:63) or a native
    74-float AdversaryPolicy.get_weights().  Anything of at least 74 floats is accepted; the kernels read [P, 1250] rows,
    so shorter rows are zero padded and longer ones cut."""
    if isinstance(x, (list, tuple)):
        x = torch.stack([torch.as_tensor(w, dtype=torch.float32).reshape(-1) for w in x])
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x, np.float32))
    x = x.to(torch.float32)
    if x.dim() == 1:
        x = x.reshape(1, -1)
    n = x.shape[1]
    if n < 74:
        raise ValueError(f"adversary genome has {n} floats; AdversaryPolicy needs 74 (models/model.py:40-57)")
    if n == 1250:
        return x.contiguous()
    out = torch.zeros(x.shape[0], 1250, dtype=torch.float32, device=x.device)
    out[:, :min(n, 1250)] = x[:, :1250]
    return out


def rollout_population(bundle: Bundle, genomes, adv_genomes=None, *, phi, fee_rate=0.0, hidden=32,
                       units_per_lane=0, warps_per_cta=0, precision=None):
    """One episode per individual (the reference's ``pool.starmap(evaluate_individual, ...)``).

    ``genomes``: [P, G] float32 -- CUDA tensor (device path, returns CUDA tensors, no sync) or
    CPU tensor / ndarray / list of tensors (end-to-end path through ``sgmm_rollout_population_host``:
    H2D, kernel, D2H, returns numpy arrays).  ``adv_genomes``: optional [P, 1250] (use_arl).
    Returns ``(fitness float64[P], trades int32[P])``.
    """
    G = genome_len(hidden)
    g = _as_f32_matrix(genomes, G)
    P = g.shape[0]
    a = None if adv_genomes is None else _as_adv_matrix(adv_genomes)
    if a is not None and a.shape[0] != P:
        raise ValueError("adversary population size differs from the market-maker population")
    L = _lib.lib()
    mm = _lib.Population(hidden, 0, P, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    adv = None if a is None else _lib.Population(32, 0, P, a.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    prm = _params(phi, fee_rate, units_per_lane, warps_per_cta, hidden, precision)
    advp = None if adv is None else C.byref(adv)
    if g.is_cuda:
        if g.device.index != bundle.device or (a is not None and a.device != g.device):
            raise ValueError("genomes must live on the bundle's device")
        fit = torch.empty(P, dtype=torch.float64, device=g.device)
        trd = torch.empty(P, dtype=torch.int32, device=g.device)
        _lib.check(L.sgmm_rollout_population(bundle.handle, C.byref(mm), advp, C.byref(prm),
                                             fit.data_ptr(), trd.data_ptr(), _stream(bundle.device)))
        return fit, trd
    if a is not None and a.is_cuda:
        raise ValueError("mixing CPU market-maker genomes with CUDA adversary genomes")
    fit = np.empty(P, np.float64)
    trd = np.empty(P, np.int32)
    _lib.check(L.sgmm_rollout_population_host(bundle.handle, C.byref(mm), advp, C.byref(prm),
                                              fit.ctypes.data, trd.ctypes.data, _stream(bundle.device)))
    return fit, trd


class PendingRollout:
    """A batch in flight on one of the bundle's two pipelined streams (``sgmm_rollout_population_host_async``).
    Keeps the pinned host buffers alive; ``result()`` waits and returns ``(fitness, trades)`` as numpy arrays."""

    def __init__(self, bundle, ticket, keep, fit, trd):
        self._bundle, self._ticket, self._keep, self._fit, self._trd = bundle, ticket, keep, fit, trd

    def result(self):
        if self._ticket is not None:
            _lib.check(_lib.lib().sgmm_rollout_wait(self._bundle.handle, self._ticket))
            self._ticket = None
        return self._fit.numpy(), self._trd.numpy()


def rollout_population_async(bundle: Bundle, genomes, adv_genomes=None, *, phi, fee_rate=0.0, hidden=32,
                             precision=None, out=None) -> PendingRollout:
    """Pipelined end-to-end evaluation of one batch of HOST genomes: H2D + kernel + D2H are enqueued on one of two
    internal streams and the call returns at once, so the upload of the next batch overlaps this batch's kernel
    (at most two batches in flight).  ``genomes`` should be a pinned CPU tensor (a pageable one is staged by the
    driver and does not overlap).  ``out = (fitness f64[P], trades i32[P])`` pinned CPU tensors may be passed to be
    reused across batches."""
    g = _as_f32_matrix(genomes, genome_len(hidden))
    if g.is_cuda:
        raise ValueError("rollout_population_async takes host genomes; device genomes need no pipelining")
    P = g.shape[0]
    a = None if adv_genomes is None else _as_adv_matrix(adv_genomes)
    if a is not None and (a.is_cuda or a.shape[0] != P):
        raise ValueError("adversary genomes must be host tensors of the same population size")
    if out is None:
        fit = torch.empty(P, dtype=torch.float64).pin_memory()
        trd = torch.empty(P, dtype=torch.int32).pin_memory()
    else:
        fit, trd = out
        if fit.numel() != P or trd.numel() != P or fit.dtype != torch.float64 or trd.dtype != torch.int32:
            raise ValueError("out must be (float64[P], int32[P])")
    mm = _lib.Population(hidden, 0, P, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    adv = None if a is None else _lib.Population(32, 0, P, a.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    prm = _params(phi, fee_rate, 0, 0, hidden, precision)
    ticket = C.c_int32(-1)
    _lib.check(_lib.lib().sgmm_rollout_population_host_async(bundle.handle, C.byref(mm), None if adv is None else C.byref(adv),
                                                            C.byref(prm), fit.data_ptr(), trd.data_ptr(), C.byref(ticket)))
    return PendingRollout(bundle, ticket.value, (g, a), fit, trd)


def rollout_seeded(bundle: Bundle, master, *, count, sigma, seed, generation, first_index=0,
                   adv_master=None, adv_sigma=None, phi, fee_rate=0.0, hidden=32,
                   units_per_lane=0, warps_per_cta=0, precision=None):
    """Evaluate children ``first_index .. first_index+count-1`` of ``master`` without ever storing
    them: child i = master + sigma*N(0,1)[Philox(seed, generation, i)] is generated inside the
    kernel (device-resident ``ask``, models/model.py:65-71).  ``master`` (and ``adv_master``) are
    CUDA float32 tensors; returns CUDA tensors."""
    G = genome_len(hidden)
    m = torch.as_tensor(master, dtype=torch.float32, device=f"cuda:{bundle.device}").contiguous()
    if m.numel() != G:
        raise ValueError(f"master length {m.numel()} != {G}")
    fit = torch.empty(count, dtype=torch.float64, device=m.device)
    trd = torch.empty(count, dtype=torch.int32, device=m.device)
    mm = _lib.Population(hidden, 0, count, None, m.data_ptr(), float(sigma), 0.0, int(seed), int(generation),
                         int(first_index))
    advp = None
    if adv_master is not None:
        am = _as_adv_matrix(torch.as_tensor(adv_master, dtype=torch.float32, device=m.device)).reshape(-1)
        adv = _lib.Population(32, 0, count, None, am.data_ptr(), float(sigma if adv_sigma is None else adv_sigma),
                              0.0, int(seed) ^ ADV_SEED_FLIP, int(generation), int(first_index))
        advp = C.byref(adv)
    prm = _params(phi, fee_rate, units_per_lane, warps_per_cta, hidden, precision)
    _lib.check(_lib.lib().sgmm_rollout_population(bundle.handle, C.byref(mm), advp, C.byref(prm),
                                                  fit.data_ptr(), trd.data_ptr(), _stream(bundle.device)))
    return fit, trd


TC_ADVERSARY = True          # the tensor-core rollouts carry the adversary (20-state automaton; H=256: q tables + walk)


def rollout_tc_audit(bundle: Bundle, genomes, adv_genomes=None, *, phi, fee_rate=0.0, hidden=32, group=0, precision="bf16"):
    """Tensor-core rollout (hidden=32: sgmm_tc32.cu, hidden=256: sgmm_spec256.cu) with its audit
    outputs: returns ``(fitness, trades, raw_table float32[P,T,5,2], act_trace int32[P,T,2])`` as
    CUDA tensors -- the policy outputs for every (bar, inventory) and the offsets actually taken (the market maker's,
    before the adversary's displacement when ``adv_genomes`` is given, at hidden 32 and 256)."""
    g = _as_f32_matrix(genomes, genome_len(hidden)).to(f"cuda:{bundle.device}")
    P, T = g.shape[0], bundle.T
    fit = torch.empty(P, dtype=torch.float64, device=g.device)
    trd = torch.empty(P, dtype=torch.int32, device=g.device)
    raw = torch.zeros(P, T, 5, 2, dtype=torch.float32, device=g.device)
    act = torch.zeros(P, T, 2, dtype=torch.int32, device=g.device)
    mm = _lib.Population(hidden, 0, P, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    advp = None
    if adv_genomes is not None:
        a = _as_adv_matrix(adv_genomes).to(g.device)
        if a.shape[0] != P:
            raise ValueError("adversary population size differs from the market-maker population")
        adv = _lib.Population(32, 0, P, a.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
        advp = C.byref(adv)
    prm = _params(phi, fee_rate, units_per_lane=group, hidden=hidden, precision=precision)
    _lib.check(_lib.lib().sgmm_rollout_tc_audit(bundle.handle, C.byref(mm), advp, C.byref(prm), fit.data_ptr(),
                                                trd.data_ptr(), raw.data_ptr(), act.data_ptr(), _stream(bundle.device)))
    return fit, trd, raw, act


def rollout_spec256_audit(bundle: Bundle, genomes, *, phi, fee_rate=0.0):
    return rollout_tc_audit(bundle, genomes, phi=phi, fee_rate=fee_rate, hidden=256)


_TRACE_I32 = ("off_a", "off_b", "adv_a", "adv_b", "fill_buy", "fill_sell", "inventory", "skew")
_TRACE_F64 = ("cash", "reward", "pnl_reward", "inventory_reward", "fee_paid",
              "spread", "wealth", "cum_reward", "cum_fees", "unrealized_pnl")      # the last five: Env/recorder.py:45-51, on the device
_TRACE_F32 = ("raw_a", "raw_b")


def rollout_trace(bundle: Bundle, genome=None, adv_genome=None, forced_actions=None, *, phi,
                  fee_rate=0.0, hidden=32):
    """Per-step trace of one individual: the recorder row contract (Env/recorder.py:8-36,
    main.py:74-90) at hidden 32 or 256, policy in SGMM-F32 order.  ``forced_actions`` int32[T,2] replaces the policy
    (teacher-forced replay).
    Returns ``(fitness, trades, dict of numpy arrays of length T)``."""
    dev = torch.device(f"cuda:{bundle.device}")
    T = bundle.T
    cols = {k: torch.zeros(T, dtype=torch.int32, device=dev) for k in _TRACE_I32}
    cols.update({k: torch.zeros(T, dtype=torch.float64, device=dev) for k in _TRACE_F64})
    cols.update({k: torch.zeros(T, dtype=torch.float32, device=dev) for k in _TRACE_F32})
    tr = _lib.Trace(*[cols[n].data_ptr() for n, _ in _lib.Trace._fields_])
    g = None if genome is None else torch.as_tensor(genome, dtype=torch.float32).reshape(-1).to(dev).contiguous()
    a = None if adv_genome is None else torch.as_tensor(adv_genome, dtype=torch.float32).reshape(-1).to(dev).contiguous()
    f = None
    if forced_actions is not None:
        f = torch.as_tensor(np.ascontiguousarray(forced_actions, np.int32)).reshape(-1).to(dev).contiguous()
        if f.numel() != 2 * T:
            raise ValueError("forced_actions must be [T, 2]")
    if g is not None and g.numel() != genome_len(hidden):
        raise ValueError("bad genome length")
    fit = torch.zeros(1, dtype=torch.float64, device=dev)
    trd = torch.zeros(1, dtype=torch.int32, device=dev)
    prm = _params(phi, fee_rate)
    _lib.check(_lib.lib().sgmm_rollout_trace(
        bundle.handle, None if g is None else g.data_ptr(), hidden, None if a is None else a.data_ptr(),
        None if f is None else f.data_ptr(), C.byref(prm), C.byref(tr), fit.data_ptr(), trd.data_ptr(),
        _stream(bundle.device)))
    out = {k: v.cpu().numpy() for k, v in cols.items()}
    return float(fit.item()), int(trd.item()), out


def _population(bundle, genomes, adv_genomes, master, count, sigma, seed, generation, first_index, adv_master, adv_sigma, hidden):
    """The (mm, adv) Population structs of explicit CUDA genomes or seeded children, and the tensors they point into."""
    dev = torch.device(f"cuda:{bundle.device}")
    G = genome_len(hidden)
    if (genomes is None) == (master is None):
        raise ValueError("pass either genomes or master (seeded children)")
    if genomes is not None:
        g = _as_f32_matrix(genomes, G).to(dev)
        P = g.shape[0]
        mm = _lib.Population(hidden, 0, P, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    else:
        if count is None or sigma is None or seed is None:
            raise ValueError("seeded children need count, sigma and seed")
        g = torch.as_tensor(master, dtype=torch.float32).reshape(-1).to(dev).contiguous()
        if g.numel() != G:
            raise ValueError(f"master length {g.numel()} != {G}")
        P = int(count)
        mm = _lib.Population(hidden, 0, P, None, g.data_ptr(), float(sigma), 0.0, int(seed), int(generation), int(first_index))
    a, adv = None, None
    if adv_genomes is not None:
        a = _as_adv_matrix(adv_genomes).to(dev)
        if a.shape[0] != P:
            raise ValueError("adversary population size differs from the market-maker population")
        adv = _lib.Population(32, 0, P, a.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    elif adv_master is not None:
        if master is None:
            raise ValueError("a seeded adversary (adv_master) goes with seeded market makers (master)")
        a = _as_adv_matrix(torch.as_tensor(adv_master, dtype=torch.float32).to(dev)).reshape(-1)
        adv = _lib.Population(32, 0, P, None, a.data_ptr(), float(sigma if adv_sigma is None else adv_sigma), 0.0,
                              int(seed) ^ ADV_SEED_FLIP, int(generation), int(first_index))
    return mm, adv, (g, a)


def rollout_trace_population(bundle: Bundle, genomes=None, adv_genomes=None, *, master=None, count=None, sigma=None, seed=None,
                             generation=0, first_index=0, adv_master=None, adv_sigma=None, phi, fee_rate=0.0, hidden=32,
                             columns=None):
    """Backtest a whole population in one call: the per-step recorder trace of every individual (``sgmm_rollout_trace_population``).

    The population is ``genomes`` [P, G] (explicit; any tensor or array, moved to the bundle's device) or the seeded children
    ``first_index .. first_index+count-1`` of ``master`` (child i = master + sigma*N(0,1)[Philox(seed, generation, i)], as
    :func:`rollout_seeded`); the adversary is ``adv_genomes`` [P, >=74] or seeded from ``adv_master`` (noise stream
    ``seed ^ ADV_SEED_FLIP``, sigma ``adv_sigma``).  hidden 32 or 256, policy in SGMM-F32 order.
    ``columns``: names out of the trace columns (default: all); the others are neither written nor computed.
    Returns ``(fitness float64[P], trades int32[P], {column: [P, T] CUDA tensor})`` with no host copy: row i of every column
    and fitness[i] / trades[i] are bit-identical to :func:`rollout_trace` of individual i alone, and fitness / trades to the
    exact :func:`rollout_population`.  (All columns take 120 B per individual and bar: 7.1 GB at 4096 x 14 400.)"""
    mm, adv, keep = _population(bundle, genomes, adv_genomes, master, count, sigma, seed, generation, first_index, adv_master,
                                adv_sigma, hidden)
    dev = torch.device(f"cuda:{bundle.device}")
    P, T = mm.count, bundle.T
    names = [n for n, _ in _lib.Trace._fields_]
    wanted = names if columns is None else list(columns)
    unknown = [c for c in wanted if c not in names]
    if unknown:
        raise ValueError(f"unknown trace columns {unknown}")
    cols = {}
    for k in wanted:
        dt = torch.int32 if k in _TRACE_I32 else (torch.float32 if k in _TRACE_F32 else torch.float64)
        cols[k] = torch.empty(P, T, dtype=dt, device=dev)
    tr = _lib.Trace(*[cols[n].data_ptr() if n in cols and cols[n].numel() else None for n in names])
    fit = torch.empty(P, dtype=torch.float64, device=dev)
    trd = torch.empty(P, dtype=torch.int32, device=dev)
    prm = _params(phi, fee_rate, hidden=hidden, precision="exact")
    _lib.check(_lib.lib().sgmm_rollout_trace_population(bundle.handle, C.byref(mm), None if adv is None else C.byref(adv),
                                                        C.byref(prm), C.byref(tr), fit.data_ptr(), trd.data_ptr(),
                                                        _stream(bundle.device)))
    return fit, trd, cols


def rollout_table(bundle: Bundle, table, *, phi, fee_rate=0.0):
    """Walk an inventory-indexed offset table int32[T,5,2] (FOIC / GLFT benchmarks, see
    :mod:`benchmarks`) through the device step core.  Returns ``(fitness, trades, trace dict)``."""
    dev = torch.device(f"cuda:{bundle.device}")
    T = bundle.T
    tab = torch.as_tensor(np.ascontiguousarray(table, np.int32)).reshape(-1).to(dev).contiguous()
    if tab.numel() != T * 10:
        raise ValueError("table must be [T, 5, 2]")
    cols = {k: torch.zeros(T, dtype=torch.int32, device=dev) for k in _TRACE_I32}
    cols.update({k: torch.zeros(T, dtype=torch.float64, device=dev) for k in _TRACE_F64})
    cols.update({k: torch.zeros(T, dtype=torch.float32, device=dev) for k in _TRACE_F32})
    tr = _lib.Trace(*[cols[n].data_ptr() for n, _ in _lib.Trace._fields_])
    fit = torch.zeros(1, dtype=torch.float64, device=dev)
    trd = torch.zeros(1, dtype=torch.int32, device=dev)
    prm = _params(phi, fee_rate)
    _lib.check(_lib.lib().sgmm_rollout_table(bundle.handle, tab.data_ptr(), C.byref(prm), C.byref(tr),
                                             fit.data_ptr(), trd.data_ptr(), _stream(bundle.device)))
    return float(fit.item()), int(trd.item()), {k: v.cpu().numpy() for k, v in cols.items()}


def measure_fp32_peak(device=0) -> float:
    """Sustained FP32 FMA TFLOP/s of the device (roofline denominator for H=32)."""
    v = C.c_double()
    _lib.check(_lib.lib().sgmm_measure_fp32_peak(int(device), C.byref(v), _stream(device)))
    return v.value


# ------------------------------------------------------------------------------------------------
# evaluate_individual: reference signature, one individual per call
# ------------------------------------------------------------------------------------------------
_BUNDLE_CACHE: "OrderedDict[tuple, Bundle]" = OrderedDict()
_BUNDLE_CACHE_MAX = 8


def _content_key(arrays):
    """Cheap content fingerprint of a host bundle: lengths, dtypes and a CRC of every array's bytes (14 400 bars x 7
    arrays = 0.7 MB: ~0.2 ms, negligible next to the upload it saves).  Keyed on content, not on ``id()``: an in-place
    edit of a cached bundle's arrays must not silently evaluate stale device data."""
    import zlib
    key = []
    for a in arrays:
        a = np.ascontiguousarray(a)
        key.append((a.shape, a.dtype.str, zlib.crc32(a.view(np.uint8).reshape(-1)) if a.size else 0))
    return tuple(key)


def _cached_bundle(bundle, train_stats, tick_size, device=None) -> Bundle:
    """Upload a host 7-tuple once; later calls with the same CONTENT reuse the device copy (the
    reference re-pickles the bundle to its workers every generation, drl_engine.py:104-115)."""
    if isinstance(bundle, Bundle):
        return bundle
    dev = torch.cuda.current_device() if device is None else int(device)
    key = (_content_key(bundle), float(tick_size), dev,
           tuple((k, float(train_stats[k]), np.asarray(train_stats[k]).dtype.str)
                 for k in ("s1_m", "s1_s", "s2_m", "s2_s")))
    b = _BUNDLE_CACHE.get(key)
    if b is None:
        b = Bundle.from_arrays(bundle, train_stats, tick_size, dev)
        _BUNDLE_CACHE[key] = b
        while len(_BUNDLE_CACHE) > _BUNDLE_CACHE_MAX:
            _BUNDLE_CACHE.popitem(last=False)[1].close()
    else:
        _BUNDLE_CACHE.move_to_end(key)
    return b


_HIDDEN_OF_LEN = {genome_len(32): 32, genome_len(256): 256}


def evaluate_individual(mm_weights, adv_weights, bundle, phi, tick_size, fee_rate, train_stats,
                        use_arl=False):
    """Drop-in for Env/drl_engine.py:9-67 -> ``(np.float64 total_reward, int trades)``.  The policy width follows from
    the genome length, as the reference's ``TradingPolicy.set_weights`` of the matching width does (1250 floats: H=32,
    67 330: H=256); both are evaluated in SGMM-F32 order, bit-identical to the reference's fp32 arithmetic."""
    dev_bundle = _cached_bundle(bundle, train_stats, tick_size)
    adv = adv_weights if (use_arl and adv_weights is not None) else None      # :17-21
    mm = torch.as_tensor(mm_weights, dtype=torch.float32).reshape(1, -1).cpu()
    hidden = _HIDDEN_OF_LEN.get(mm.shape[1])
    if hidden is None:
        raise ValueError(f"genome length {mm.shape[1]} is neither {genome_len(32)} (hidden 32) nor {genome_len(256)} (hidden 256)")
    if adv is not None:
        adv = torch.as_tensor(adv, dtype=torch.float32).reshape(1, -1).cpu()
    fit, trd = rollout_population(dev_bundle, mm, adv, phi=phi, fee_rate=fee_rate, hidden=hidden, precision="exact")
    return np.float64(fit[0]), int(trd[0])


# ------------------------------------------------------------------------------------------------
# DRLEngine
# ------------------------------------------------------------------------------------------------
class DeviceGA:
    """Thin owner of a ``sgmm_ga`` handle (include/sgmm.h): ask/evaluate/tell/validate/select on
    the device, one call per generation, no host round trip."""

    def __init__(self, mm_master, adv_master=None, *, pop_size, sigma, phi, fee_rate, use_arl, seed,
                 max_generations, patience=15, hidden=32, device=None, shard=None, precision=None):
        self.device = torch.cuda.current_device() if device is None else int(device)
        first, count, stride = (0, pop_size, 0) if shard is None else shard
        cfg = _lib.GaConfig(hidden, int(bool(use_arl)), pop_size, first, count, stride, float(sigma), patience,
                            float(phi), float(fee_rate), int(seed) & 0xFFFFFFFFFFFFFFFF, int(max_generations),
                            _precision(precision, hidden))
        m = np.ascontiguousarray(torch.as_tensor(mm_master).detach().cpu().numpy(), np.float32)
        a = None
        if use_arl:
            a = np.ascontiguousarray(_as_adv_matrix(torch.as_tensor(adv_master).detach().cpu()).reshape(-1).numpy(), np.float32)
        self.G = genome_len(hidden)
        self.pop_size, self.shard, self.max_generations = pop_size, (first, count), max_generations
        self._h = C.c_void_p()
        _lib.check(_lib.lib().sgmm_ga_create(C.byref(self._h), C.byref(cfg), m.ctypes.data,
                                             None if a is None else a.ctypes.data, self.device,
                                             _stream(self.device)))

    def buffers(self):
        """``(fitness_slice, trades_slice, gather_base, block_bytes, n_blocks, my_block)``: raw device addresses of
        this rank's result slices and of the rank-blocked gather buffer (include/sgmm.h, sgmm_ga_buffers)."""
        p = [C.c_void_p() for _ in range(3)]
        bb, nb, mb = C.c_int64(), C.c_int32(), C.c_int32()
        _lib.check(_lib.lib().sgmm_ga_buffers(self._h, *[C.byref(x) for x in p], C.byref(bb), C.byref(nb), C.byref(mb)))
        return p[0].value, p[1].value, p[2].value, bb.value, nb.value, mb.value

    def evaluate(self, train: Bundle):
        _lib.check(_lib.lib().sgmm_ga_evaluate(self._h, train.handle, _stream(self.device)))

    def select(self, val: Bundle):
        _lib.check(_lib.lib().sgmm_ga_select(self._h, val.handle, _stream(self.device)))

    def generation(self, train: Bundle, val: Bundle):
        _lib.check(_lib.lib().sgmm_ga_generation(self._h, train.handle, val.handle, _stream(self.device)))

    def capture(self, train: Bundle, val: Bundle):
        """Capture one generation (ask + rollout + tell + validation rollout + select: 4 kernels, no
        host round trip) into a CUDA graph; ``graph.replay()`` then advances the GA by one generation.
        Call :meth:`generation` once before capturing (first launches configure the kernels)."""
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.generation(train, val)
        return g

    def status(self):
        s = _lib.GaStatus()
        _lib.check(_lib.lib().sgmm_ga_status_host(self._h, C.byref(s), _stream(self.device)))
        return {"generation": s.generation, "stale": s.stale, "sigma": s.sigma, "adv_sigma": s.adv_sigma,
                "best_val": s.best_val, "last_best_index": s.last_best_index}

    def masters(self):
        mm = np.empty(self.G, np.float32)
        adv = np.empty(1250, np.float32)
        best = np.empty(self.G, np.float32)
        _lib.check(_lib.lib().sgmm_ga_master_host(self._h, mm.ctypes.data, adv.ctypes.data, best.ctypes.data,
                                                  _stream(self.device)))
        return mm, adv, best

    def history(self, n=None):
        """History columns of the first ``n`` generations (default: the generations completed so far)."""
        n = self.status()["generation"] if n is None else int(n)
        n = max(0, min(n, self.max_generations))
        tf, vf = np.empty(n, np.float64), np.empty(n, np.float64)
        tt, vt = np.empty(n, np.int32), np.empty(n, np.int32)
        sg = np.empty(n, np.float32)
        _lib.check(_lib.lib().sgmm_ga_history_host(self._h, n, tf.ctypes.data, vf.ctypes.data, tt.ctypes.data,
                                                   vt.ctypes.data, sg.ctypes.data, _stream(self.device)))
        return {"train_f": tf, "val_f": vf, "train_trades": tt, "val_trades": vt, "sigma": sg}

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().sgmm_ga_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DRLEngine:
    """Drop-in for Env/drl_engine.py:69-178.  Same constructor, attributes and return values; the generation loop
    runs on the device (:class:`DeviceGA`).

    * ``sigma`` is accepted and -- exactly like the reference (drl_engine.py:77,81 build ``NeuroEvolution(population_size=
      pop_size)`` without it) -- NOT forwarded: the evolvers start at 0.05; set ``engine.mm_evolver.sigma`` to change it.
    * Extra keyword arguments expose what the reference hard-codes or leaves to the global RNG: ``seed`` (``None`` = drawn
      from torch's global generator at every ``train`` call, so repeated runs and phi sweeps are independent like the
      reference's unseeded ``torch.randn``, models/model.py:69; an integer = reproducible, with the ``train`` call count
      folded in), ``device``, ``patience`` (15, :155), ``hidden_dim`` (32 or 256, models/model.py:7), ``precision``
      (``None`` / "f32": bit-exact population evaluation at hidden 32; "tf32" / "f16" / "bf16": tensor-core rollout;
      ``None`` at hidden 256 runs the tensor-core path, with ``use_arl`` too; "exact" runs population, validation and
      adversary bit-exact at hidden 32 and 256).
    * When ``torch.distributed`` is initialised with more than one rank, ``train`` shards the population over the ranks
      (:class:`dist.ShardedGA`: one NCCL all-gather of fitness + trades per generation) -- the multi-GPU replacement of
      the ``Pool(8).starmap`` of drl_engine.py:91,115.  Every rank returns the identical policy and history; rank 0
      writes the checkpoint.
    """

    def __init__(self, pop_size=50, sigma=0.05, phi=0.01, tick_size=0.01, fee_rate=0.0, use_arl=False,
                 save_dir="checkpoints/drl", seed=None, device=None, patience=15, precision=None, hidden_dim=32,
                 group=None):
        self.precision = precision
        self.phi = phi
        self.tick_size = tick_size
        self.fee_rate = fee_rate
        self.save_dir = save_dir
        os.makedirs(self.save_dir, exist_ok=True)
        self.use_arl = use_arl
        self.seed = seed
        self.device = device
        self.patience = patience
        self.hidden_dim = hidden_dim
        self.group = group
        self._train_calls = 0
        self.mm_evolver = NeuroEvolution(population_size=pop_size, hidden_dim=hidden_dim)      # drl_engine.py:77
        if self.use_arl:
            self.adv_evolver = NeuroEvolution(population_size=pop_size)                        # :81

    def _run_seed(self):
        """Philox key of this ``train`` call."""
        call = self._train_calls
        self._train_calls += 1
        if self.seed is None:
            return int(torch.randint(0, 2 ** 62, (), dtype=torch.int64).item())
        # splitmix-style fold of the call counter: call 0 keeps the caller's seed verbatim
        return (int(self.seed) + call * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF

    def train(self, train_bundle, val_bundle, train_stats, generations=100, output_prefix="agent",
              log_every=5, verbose=True):
        import torch.distributed as tdist
        dev = torch.cuda.current_device() if self.device is None else int(self.device)
        train = _cached_bundle(train_bundle, train_stats, self.tick_size, dev)
        val = _cached_bundle(val_bundle, train_stats, self.tick_size, dev)
        history = {'gen': [], 'train_f': [], 'val_f': [], 'train_trades': [], 'val_trades': []}
        save_path = os.path.join(self.save_dir, f"{output_prefix}_best_val_{self.phi}.pth")
        sharded = tdist.is_available() and tdist.is_initialized() and tdist.get_world_size(self.group) > 1
        rank = tdist.get_rank(self.group) if sharded else 0
        seed = self._run_seed()
        if sharded:                                  # every rank must use rank 0's key (seed=None draws per process)
            t = torch.tensor([seed & 0x7FFFFFFFFFFFFFFF], dtype=torch.int64, device=f"cuda:{dev}")
            tdist.broadcast(t, src=tdist.get_global_rank(self.group, 0) if self.group is not None else 0, group=self.group)
            seed = int(t.item())
        pop = self.mm_evolver.pop_size

        def make(shard=None):
            return DeviceGA(self.mm_evolver.master_policy.get_weights(),
                            self.adv_evolver.master_policy.get_weights() if self.use_arl else None,
                            pop_size=pop, sigma=self.mm_evolver.sigma, phi=self.phi,
                            fee_rate=self.fee_rate, use_arl=self.use_arl, seed=seed,
                            max_generations=max(1, generations), patience=self.patience, device=dev,
                            precision=self.precision, hidden=self.hidden_dim, shard=shard)
        if sharded:
            from .dist import ShardedGA
            runner = ShardedGA(make, pop, group=self.group)
            ga = runner.ga
        else:
            runner = ga = make()
        saved_val = -np.inf

        def checkpoint(best_val):
            """drl_engine.py:144-150 saves on every improvement; here at every poll that saw one, so that an
            interrupted run keeps the best-on-validation master found so far."""
            nonlocal saved_val
            if best_val > saved_val:
                saved_val = best_val
                if rank == 0:
                    _, _, best = ga.masters()
                    snap = TradingPolicy(hidden_dim=self.hidden_dim)
                    snap.set_weights(torch.from_numpy(best))
                    torch.save(snap.state_dict(), save_path)

        try:
            logged = 0
            for gen in range(generations):
                runner.generation(train, val)                   # ask + evaluate (+ all-gather) + tell + validate + select
                if gen % log_every == 0:                        # drl_engine.py:169-171
                    h = ga.history(gen + 1)
                    best_so_far = np.maximum.accumulate(h["val_f"])
                    checkpoint(float(best_so_far[gen]))
                    if verbose and rank == 0:
                        for g in range(logged, gen + 1):
                            if g > 0 and h["sigma"][g] != h["sigma"][g - 1]:
                                print(f">>> Sigma decayed to {h['sigma'][g]:.4f} due to no improvement")
                        tag = "*" if (gen == 0 or h["val_f"][gen] > best_so_far[gen - 1]) else ""
                        arl = "ARL:ON" if self.use_arl else "ARL:OFF"
                        print(f"Gen {gen:03d} | {arl} | Best Train: {h['train_f'][gen]:.2f} | Val: {h['val_f'][gen]:.2f}{tag}")
                    logged = gen + 1
            h = ga.history(generations)
            st = ga.status()
            mm, adv, best = ga.masters()
            improved = generations > 0 and st["best_val"] > -np.inf
            if improved:
                checkpoint(float(st["best_val"]))
        finally:
            ga.close()
        history['gen'] = list(range(generations))
        history['train_f'] = [np.float64(x) for x in h["train_f"]]
        history['val_f'] = [np.float64(x) for x in h["val_f"]]
        history['train_trades'] = [int(x) for x in h["train_trades"]]
        history['val_trades'] = [int(x) for x in h["val_trades"]]
        self.mm_evolver.sigma = float(st["sigma"])
        if self.use_arl:
            self.adv_evolver.sigma = float(st["adv_sigma"])
            self.adv_evolver.master_policy.set_weights(torch.from_numpy(adv))
        # drl_engine.py:144-150,174-176: the checkpoint holds the master of the best validation
        # generation and is loaded back into the returned policy
        self.mm_evolver.master_policy.set_weights(torch.from_numpy(best if improved else mm))
        return self.mm_evolver.master_policy, history
