"""A bundle carries state from call to call; no result may depend on it.

State of a bundle (include/sgmm.h): the grow-only code buffer, scratch of about ten kernels in five layouts (step codes of
spec256, 48 B policy tables of the small-population path and of the exact H = 256 path with staged seeded children, 40 B q
tables of spec256 with the adversary, raw tables of the population trace, the table of the single H = 256 trace); the event
that orders its users across streams; the buffers a capture has used (retired, not freed, when outgrown); one leg table per
fee rate of the tensor-core adversary path; the host workspaces of the synchronous and the pipelined host entries.

Every result here is compared with a reference that has no history: the exact routes with the C oracle bit for bit (through
a reference run on a fresh bundle, itself checked against the oracle), the tensor-core routes with the same call on a
freshly created bundle bit for bit (those kernels are deterministic).

  A  history: every ordered pair (X, Y) of the routes below on one bundle -- Y in X's leftovers (X's footprint covers
     Y's), Y growing the buffer, Y shrinking after its own growth -- at T = 300 and a few pairs at T = 2049 (across the
     2048-bar chunk of the walk and the trace); batch loops forced by SGMM_EXACT256_BATCH_BYTES (batch k runs in batch
     k-1's leftovers)
  B  streams: one sequence of calls over three side streams and the legacy default stream with no host synchronisation,
     the buffer growing in the middle; two pipelined host batches in flight, the second growing the buffer
  C  graph capture: captured GA generations replayed before and after a call that outgrows (so retires) the captured
     buffers; refusals under capture (buffer too small, no leg table for the fee) leave the bundle and later captures working
  D  leg tables: fee rates alternating over two streams, -0.0 as a key of its own (sign of zero kept bit for bit), the
     64-table limit
"""
import numpy as np
import pytest
import torch

from test_gpu_rounding_edges import bits32, bits64, boundary_adversary, transparent_genome

F32 = np.float32
T0 = 300                       # the shape of the pair matrix
T_RAGGED = 2049
TICK, PHI, FEE = 0.001, 1e-4, 3e-4
BATCH_ENV = "SGMM_EXACT256_BATCH_BYTES"
G256 = 256 * 256 + 7 * 256 + 2
K_CLAMP_SCALE = F32(1.15e8)    # transparent output layer: |q| = 5 * 1.15e8 * |z| beyond K_CLAMP = 2^30 for |z| > 1.87, and
                               # inside int32 (the offsets' type, include/sgmm.h) for |z| < 3.73 (checked on the episodes)
ADV_SCALE = F32(5.5e7)         # with the adversary offsets are clamped to +-K_CLAMP (include/sgmm.h): |q| up to ~2^30 only
TC_SCALE = F32(1 << 14)        # the same within the f16 range of the tensor-core operands
SEED, GEN, FIRST, SIGMA, ADV_SIGMA = 31, 3, 5, 0.05, 0.1

# name: (hidden, adversary, seeded, tensor-core precision or None, sizes tiny / normal / big, scratch layout)
#   scratch layouts (words of 8 B the call reserves in the code buffer, default batch budget):
#     "table"  (6P + 1) T                         small-population path (sgmm_one.cu)
#     "codes"  P T                                spec256 step codes (sgmm_spec256.cu)
#     "batch"  (floor((P w + T - 1) / T) + 1) T   batches of w words per individual (exact256, spec256 + adversary,
#                                                 population trace)
#     "trace"  ceil((5 T + G/2) / T) T            single H = 256 trace (sgmm_rollout.cu)
ROUTES = {
    "small32":             (32, False, False, None, (1, 8, 50), "table"),
    "small32_adv":         (32, True, False, None, (1, 8, 50), "table"),
    "seq32":               (32, False, False, None, (401, 401, 401), None),     # rollout_kernel_h32: no scratch
    "tc32":                (32, False, False, "bf16", (8, 8, 8), None),        # no scratch
    "tc32_adv":            (32, True, False, "f16", (8, 8, 8), None),          # leg table only
    "spec256":             (256, False, False, "bf16", (1, 8, 300), "codes"),
    "spec256_adv":         (256, True, False, "bf16", (1, 8, 60), "batch"),
    "exact256":            (256, False, False, None, (1, 8, 50), "batch"),
    "exact256_seeded_adv": (256, True, True, None, (1, 2, 3), "batch"),
    "tracepop32_adv":      (32, True, False, None, (1, 8, 60), "batch"),
    "tracepop256_seeded":  (256, False, True, None, (1, 2, 3), "batch"),
    "trace256":            (256, True, False, None, (1, 1, 1), "trace"),
}
NAMES = list(ROUTES)
SIZES = ("tiny", "normal", "big")
TENSOR = {n for n, r in ROUTES.items() if r[3] is not None}


def count_of(name, size):
    return ROUTES[name][4][SIZES.index(size)]


def batch_words(name, T):
    """Words per individual of a batched route (ScratchLease::reserve_in_batches' per_ind)."""
    return {"spec256_adv": 5 * T, "exact256": 6 * T, "exact256_seeded_adv": 6 * T + G256 // 2, "tracepop32_adv": 5 * T,
            "tracepop256_seeded": 5 * T + G256 // 2}[name]


def footprint(name, size, T, batch_bytes=2 << 30):
    """8-byte words of the bundle's code buffer a call reserves (sgmm_account.cu ScratchLease)."""
    P, kind = count_of(name, size), ROUTES[name][5]
    if kind is None:
        return 0
    if kind == "table":
        return (6 * P + 1) * T
    if kind == "codes":
        return P * T
    if kind == "trace":
        return -(-(5 * T + G256 // 2) // T) * T
    w = batch_words(name, T)
    nb = min(max(batch_bytes // (w * 8), 1), P)
    return ((nb * w + T - 1) // T + 1) * T


def capacity(words):
    return words + words // 4          # the lease allocates 1.25x what it was asked for


def pair_kind(x, y, case, T):
    """Whether the pair (x, y) exercises `case` at T: "covers" = x's footprint holds y's (y reads x's leftovers), "grows" =
    y outgrows the buffer x left."""
    if case == "covers":
        fx = footprint(x, "big", T)
        return fx > 0 and footprint(y, "normal", T) > 0 and fx >= footprint(y, "normal", T)
    fy = footprint(y, "big", T)
    return fy > capacity(footprint(x, "tiny", T))


# ----------------------------------------------------------------------------------------------
# populations and episodes
# ----------------------------------------------------------------------------------------------
def mm_genomes(P, hidden, seed, scale):
    """Policy-like genomes; rows 0 and 1 transparent (raw = scale * (z1, z2), and swapped)."""
    from sgmm_b200 import synthetic as syn
    G = syn.policy_like_genomes(P, hidden=hidden, seed=seed, out_scale=4.0, out_bias=(0.1, 0.1))[1]
    G[0] = transparent_genome(hidden, scale)
    if P > 1:
        G[1] = transparent_genome(hidden, scale, swap=True)
    return G


def adv_genomes(P, seed):
    """Random adversaries; rows 0 and 1 on the tanh rounding threshold (tests/test_gpu_rounding_edges.py)."""
    A = (np.random.default_rng(seed).standard_normal((P, 1250)) * 0.6).astype(F32)
    A[0] = boundary_adversary(1, -1)
    if P > 1:
        A[1] = boundary_adversary(-1, 1)
    return A


_POPS = {}


def population(name, size):
    """Host and device arrays of one (route, size): explicit G / A, or the seeded master (and adversary master)."""
    key = (name, size)
    if key not in _POPS:
        hidden, adv, seeded, tensor, _, _ = ROUTES[name]
        P = count_of(name, size)
        seed = 1000 + 10 * NAMES.index(name) + SIZES.index(size)
        if seeded:
            from sgmm_b200 import synthetic as syn
            G = syn.policy_like_genomes(1, hidden=hidden, seed=seed, out_scale=4.0, out_bias=(0.1, 0.1))[0][None, :]
            A = (np.random.default_rng(seed).standard_normal((1, 1250)) * 0.6).astype(F32) if adv else None
        else:
            G = mm_genomes(P, hidden, seed, TC_SCALE if tensor else (ADV_SCALE if adv else K_CLAMP_SCALE))
            A = adv_genomes(P, seed) if adv else None
        cuda = lambda x: None if x is None else torch.from_numpy(np.ascontiguousarray(x)).cuda()
        _POPS[key] = dict(P=P, G=G, A=A, g=cuda(G), a=cuda(A))
        torch.cuda.synchronize()
    return _POPS[key]


def children(orc, master, P):
    return np.stack([orc.mutate(master, SIGMA, SEED, GEN, FIRST + i) for i in range(P)])


def adv_children(orc, adv_master, P):
    return np.stack([orc.mutate(adv_master, ADV_SIGMA, SEED ^ 0x8000000000000000, GEN, FIRST + i) for i in range(P)])


_DATA = {}


def episode(orc, T):
    """(host 7-tuple, train stats, normalised 7-tuple of the oracle) of a synthetic episode of exactly T bars."""
    if T not in _DATA:
        from sgmm_b200 import synthetic as syn
        bundle = tuple(a[:T] for a in syn.synthetic_bundle(-(-T // syn.BARS_PER_DAY), first_day=130))
        stats = syn.train_stats_of(bundle)
        _DATA[T] = (bundle, stats, tuple(orc.normalise(bundle, stats)) + tuple(bundle[2:]))
    return _DATA[T]


def fresh(sg, orc, T):
    bundle, stats, _ = episode(orc, T)
    return sg.Bundle.from_arrays(bundle, stats, TICK)


# ----------------------------------------------------------------------------------------------
# the routes
# ----------------------------------------------------------------------------------------------
def run(sg, bun, name, size, fee=FEE):
    """One call of route `name` at `size` on `bun` (current stream); every output it has, as tensors or arrays."""
    hidden, adv, seeded, tensor, _, _ = ROUTES[name]
    p = population(name, size)
    P, g, a = p["P"], p["g"], p["a"]
    if name in ("small32", "small32_adv", "seq32", "exact256"):
        f, t = sg.rollout_population(bun, g, a, phi=PHI, fee_rate=fee, hidden=hidden, precision="exact")
        return dict(fitness=f, trades=t)
    if tensor is not None:
        f, t, raw, act = sg.rollout_tc_audit(bun, g, a, phi=PHI, fee_rate=fee, hidden=hidden, precision=tensor)
        return dict(fitness=f, trades=t, raw_table=raw, act_trace=act)
    if name == "exact256_seeded_adv":
        f, t = sg.rollout_seeded(bun, g[0], count=P, sigma=SIGMA, seed=SEED, generation=GEN, first_index=FIRST, adv_master=a[0],
                                 adv_sigma=ADV_SIGMA, phi=PHI, fee_rate=fee, hidden=hidden, precision="exact")
        return dict(fitness=f, trades=t)
    if name == "tracepop32_adv":
        f, t, cols = sg.rollout_trace_population(bun, g, a, phi=PHI, fee_rate=fee, hidden=hidden)
        return dict(fitness=f, trades=t, **cols)
    if name == "tracepop256_seeded":
        f, t, cols = sg.rollout_trace_population(bun, master=g[0], count=P, sigma=SIGMA, seed=SEED, generation=GEN,
                                                 first_index=FIRST, phi=PHI, fee_rate=fee, hidden=hidden)
        return dict(fitness=f, trades=t, **cols)
    if name == "trace256":
        f, t, cols = sg.rollout_trace(bun, p["G"][0], p["A"][0], phi=PHI, fee_rate=fee, hidden=hidden)
        return dict(fitness=np.array([f]), trades=np.array([t], np.int32), **{k: v[None] for k, v in cols.items()})
    raise KeyError(name)


def host(out):
    return {k: (v.cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in out.items()}


def assert_same(out, ref, what):
    """Every output bit for bit (float bits, so -0.0 != 0.0 and NaN == NaN of the same payload)."""
    out, ref = host(out), host(ref)
    assert sorted(out) == sorted(ref), what
    for k in ref:
        assert out[k].shape == ref[k].shape and out[k].dtype == ref[k].dtype, (what, k)
        assert np.array_equal(np.ascontiguousarray(out[k]).view(np.uint8), np.ascontiguousarray(ref[k]).view(np.uint8)), (what, k)


ORACLE_COLS = ("off_a", "off_b", "adv_a", "adv_b", "fill_buy", "fill_sell", "inventory", "cash", "reward", "pnl_reward",
               "inventory_reward", "fee_paid", "raw_a", "raw_b")


def check_oracle(orc, name, size, out, T, fee=FEE):
    """An exact route's outputs equal the oracle bit for bit: fitness / trades of every individual, and every trace column
    (the recorder's derived ones computed from the oracle's) of a sample of rows."""
    hidden, adv, seeded, tensor, _, _ = ROUTES[name]
    assert tensor is None
    _, _, bz = episode(orc, T)
    p, out = population(name, size), host(out)
    P = p["P"]
    if seeded:
        G = children(orc, p["G"][0], P)
        A = adv_children(orc, p["A"][0], P) if adv else None
        fo, to = orc.rollout_population(bz, PHI, TICK, fee, master=p["G"][0], sigma=SIGMA, adv_master=None if A is None else p["A"][0],
                                        adv_sigma=ADV_SIGMA, use_adv=adv, seed=SEED, generation=GEN, first_index=FIRST, count=P,
                                        hidden=hidden, nthreads=8)
    else:
        G, A = p["G"], p["A"]
        fo, to = orc.rollout_population(bz, PHI, TICK, fee, genomes=G, adv_genomes=A, use_adv=adv, hidden=hidden, nthreads=8)
    assert np.array_equal(bits64(out["fitness"]), bits64(fo)), (name, size)
    assert np.array_equal(out["trades"], to), (name, size)
    if "cash" not in out:
        return
    mid, ask, bid = (np.asarray(bz[k], np.float64) for k in (2, 3, 4))
    for i in sorted({0, 1, P - 1} & set(range(P))):
        f1, t1, tro = orc.rollout(G[i], None if A is None else A[i], bz, PHI, TICK, fee, hidden=hidden, trace=True)
        assert (bits64(f1), t1) == (bits64(fo[i]), to[i])
        for k in ORACLE_COLS:
            assert np.array_equal(np.asarray(out[k][i]).view(np.uint8), tro[k].view(np.uint8)), (name, size, i, k)
        inv = tro["inventory"].astype(np.float64)
        assert np.array_equal(bits64(out["spread"][i]), bits64(ask - bid))
        assert np.array_equal(bits64(out["unrealized_pnl"][i]), bits64(inv * mid))
        assert np.array_equal(bits64(out["wealth"][i]), bits64(tro["cash"] + inv * mid))
        assert np.array_equal(bits64(out["cum_reward"][i]), bits64(np.cumsum(tro["reward"])))
        assert np.array_equal(bits64(out["cum_fees"][i]), bits64(np.cumsum(tro["fee_paid"])))
        assert np.array_equal(out["skew"][i], tro["off_b"] - tro["off_a"])


def check_replay(orc, name, size, out, T, fee):
    """A tensor-core route's fitness / trades equal the oracle's env driven by the offsets it took (teacher-forced)."""
    hidden, adv, _, tensor, _, _ = ROUTES[name]
    _, _, bz = episode(orc, T)
    p, out = population(name, size), host(out)
    for i in range(p["P"]):
        fo, to = orc.rollout(None, None if p["A"] is None else p["A"][i], bz, PHI, TICK, fee, forced_actions=out["act_trace"][i])
        assert (bits64(fo), to) == (bits64(out["fitness"][i]), out["trades"][i]), (name, i)


_REFS = {}


def reference(sg, orc, name, size, T=T0):
    """The outputs of (route, size) on a fresh bundle; exact routes checked against the oracle once."""
    key = (name, size, T)
    if key not in _REFS:
        out = host(run(sg, fresh(sg, orc, T), name, size))
        if name not in TENSOR:
            check_oracle(orc, name, size, out, T)
        _REFS[key] = out
    return _REFS[key]


@pytest.fixture(scope="module")
def sg():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import sgmm_b200
    return sgmm_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


# ----------------------------------------------------------------------------------------------
# CPU: the sizes do what the pair cases claim
# ----------------------------------------------------------------------------------------------
def test_route_sizes_cover_the_pair_cases():
    """"covers": X at its big size reserves at least what Y reads at its normal size, for every pair of scratch users but
    the single H = 256 trace (fixed at one genome) before the two seeded H = 256 routes (one staged 269 KB genome more).
    "grows": Y at its big size outgrows the buffer of every X at its tiny size, except where Y is that trace.  Forced
    batches: the exact H = 256, spec256-with-adversary and population-trace routes run several batches."""
    scratch = [n for n in NAMES if ROUTES[n][5] is not None]
    misses = {(x, y) for x in scratch for y in scratch if not pair_kind(x, y, "covers", T0)}
    assert misses == {("trace256", "exact256_seeded_adv"), ("trace256", "tracepop256_seeded")}
    misses = {(x, y) for x in NAMES for y in scratch if not pair_kind(x, y, "grows", T0)}
    assert misses == {(x, "trace256") for x in ("trace256", "exact256_seeded_adv", "tracepop256_seeded")}
    for n in scratch:
        if n != "trace256":
            assert footprint(n, "big", T0) > capacity(footprint(n, "normal", T0)), n          # the shrink case shrinks
    for n in ("spec256_adv", "exact256", "exact256_seeded_adv", "tracepop32_adv", "tracepop256_seeded"):
        P, w = count_of(n, "normal"), batch_words(n, T0)
        assert max(FORCED_BATCH_BYTES // (8 * w), 1) < P, n
    for x, y in RAGGED_PAIRS:
        assert pair_kind(x, y, "covers", T_RAGGED), (x, y)


def test_transparent_outputs_reach_beyond_k_clamp_inside_int32(orc):
    """The exact routes' transparent rows quote beyond K_CLAMP on some bars of both episodes and stay inside int32; with
    the adversary (whose displaced offsets are clamped to +-K_CLAMP) they reach 2^29 and stay within K_CLAMP."""
    for T in (T0, T_RAGGED):
        _, _, bz = episode(orc, T)
        z = np.abs(np.concatenate([bz[0], bz[1]]))
        q = (z * K_CLAMP_SCALE * F32(5)).astype(np.float64)
        assert q.max() < 2.0 ** 31 and (q > 2.0 ** 30).sum() >= 10, (T, q.max(), (q > 2.0 ** 30).sum())
        q = (z * ADV_SCALE * F32(5)).astype(np.float64)
        assert q.max() < 2.0 ** 30 - 2 and (q > 2.0 ** 29).sum() >= 10, (T, q.max(), (q > 2.0 ** 29).sum())


# ----------------------------------------------------------------------------------------------
# A. history independence
# ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["covers", "grows"])
@pytest.mark.parametrize("x", NAMES)
def test_every_route_after_x(sg, orc, x, case):
    """Y after X on one bundle equals Y's reference for every Y: "covers" runs X at its big size and Y at its normal size
    (Y in X's leftovers), "grows" X at its tiny size and Y at its big size (Y outgrows X's buffer)."""
    sx, sy = ("big", "normal") if case == "covers" else ("tiny", "big")
    for y in NAMES:
        ref = reference(sg, orc, y, sy)
        bun = fresh(sg, orc, T0)
        run(sg, bun, x, sx)
        assert_same(run(sg, bun, y, sy), ref, (x, y, case))
        bun.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n in NAMES if ROUTES[n][5] not in (None, "trace")])
def test_route_after_its_own_growth(sg, orc, name):
    """The same route at a smaller population on the buffer it grew: tables of another stride under it."""
    bun = fresh(sg, orc, T0)
    assert_same(run(sg, bun, name, "big"), reference(sg, orc, name, "big"), (name, "big"))
    assert_same(run(sg, bun, name, "normal"), reference(sg, orc, name, "normal"), (name, "normal"))
    assert_same(run(sg, bun, name, "tiny"), reference(sg, orc, name, "tiny"), (name, "tiny"))


RAGGED_PAIRS = [("spec256_adv", "small32"), ("exact256", "tracepop32_adv"), ("tracepop32_adv", "small32_adv"),
                ("small32_adv", "exact256"), ("spec256", "tracepop256_seeded"), ("tracepop256_seeded", "spec256_adv")]


@pytest.mark.gpu
def test_ragged_length_pairs(sg, orc):
    """A few pairs at T = 2049, and one route shrinking after its own growth there."""
    for x, y in RAGGED_PAIRS:
        ref = reference(sg, orc, y, "normal", T_RAGGED)
        bun = fresh(sg, orc, T_RAGGED)
        run(sg, bun, x, "big")
        assert_same(run(sg, bun, y, "normal"), ref, (x, y))
    bun = fresh(sg, orc, T_RAGGED)
    run(sg, bun, "tracepop32_adv", "big")
    assert_same(run(sg, bun, "tracepop32_adv", "normal"), reference(sg, orc, "tracepop32_adv", "normal", T_RAGGED), "shrink")


FORCED_BATCH_BYTES = 3 * 48 * T0       # three 48 B tables of T0 bars: 2-3 individuals per batch, seeded H = 256 one


@pytest.mark.gpu
@pytest.mark.parametrize("T", [T0, T_RAGGED])
def test_forced_batches_run_in_the_previous_batch_leftovers(sg, orc, T, monkeypatch):
    """Several batches per call: batch k in batch k-1's leftovers, the results those of one batch."""
    names = ("spec256_adv", "exact256", "exact256_seeded_adv", "tracepop32_adv", "tracepop256_seeded")
    refs = {(n, s): reference(sg, orc, n, s, T) for n in names for s in ("normal", "big")}
    monkeypatch.setenv(BATCH_ENV, str(FORCED_BATCH_BYTES))
    bun = fresh(sg, orc, T)
    for n in names:
        for s in ("big", "normal"):
            assert_same(run(sg, bun, n, s), refs[(n, s)], (n, s, T))


# ----------------------------------------------------------------------------------------------
# B. streams
# ----------------------------------------------------------------------------------------------
STREAM_SEQUENCE = [("small32", "normal"), ("spec256", "normal"), ("tracepop32_adv", "normal"), ("tc32_adv", "normal"),
                   ("exact256", "big"),                                    # grows the buffer
                   ("small32_adv", "normal"), ("spec256_adv", "normal"), ("tracepop256_seeded", "normal"),
                   ("seq32", "normal"), ("exact256_seeded_adv", "normal"), ("spec256", "big"), ("tc32", "normal"),
                   ("small32", "big"), ("exact256", "normal")]


@pytest.mark.gpu
def test_calls_on_different_streams_are_ordered(sg, orc):
    """The sequence once on the default stream, once with call i on stream i % 4 (three side streams and the legacy
    default stream) and no host synchronisation in between: the same bits, equal to the references."""
    refs = [reference(sg, orc, n, s) for n, s in STREAM_SEQUENCE]
    assert footprint("exact256", "big", T0) > capacity(max(footprint(n, s, T0) for n, s in STREAM_SEQUENCE[:4]))
    bun = fresh(sg, orc, T0)
    single = [host(run(sg, bun, n, s)) for n, s in STREAM_SEQUENCE]
    streams = [torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.default_stream()]
    assert streams[3].cuda_stream == 0
    bun = fresh(sg, orc, T0)
    torch.cuda.synchronize()
    outs = []
    for i, (n, s) in enumerate(STREAM_SEQUENCE):
        with torch.cuda.stream(streams[i % 4]):
            outs.append(run(sg, bun, n, s))
    torch.cuda.synchronize()
    for (n, s), out, one, ref in zip(STREAM_SEQUENCE, outs, single, refs):
        assert_same(out, one, (n, s, "streams"))
        assert_same(one, ref, (n, s, "single stream"))


ASYNC_ROUTES = [("small32", None), ("small32_adv", None), ("spec256", None), ("spec256_adv", None), ("exact256", "exact")]


@pytest.mark.gpu
def test_pipelined_batches_in_flight(sg, orc):
    """Two batches in flight on the bundle's two pipelined streams, the second (another route, big) growing the code
    buffer while the first runs: both equal the synchronous host entry, and the references."""
    for i, (n1, p1) in enumerate(ASYNC_ROUTES):
        n2, p2 = ASYNC_ROUTES[(i + 1) % len(ASYNC_ROUTES)]
        bun = fresh(sg, orc, T0)
        assert footprint(n2, "big", T0) > capacity(footprint(n1, "normal", T0))
        pend = []
        for n, s, prec in ((n1, "normal", p1), (n2, "big", p2)):
            pop = population(n, s)
            g = torch.from_numpy(pop["G"]).pin_memory()
            a = None if pop["A"] is None else torch.from_numpy(pop["A"]).pin_memory()
            pend.append((n, s, prec, pop, sg.rollout_population_async(bun, g, a, phi=PHI, fee_rate=FEE, hidden=ROUTES[n][0],
                                                                       precision=prec)))
        for n, s, prec, pop, pr in pend:
            f, t = (x.copy() for x in pr.result())
            fs, ts = sg.rollout_population(bun, pop["G"], pop["A"], phi=PHI, fee_rate=FEE, hidden=ROUTES[n][0], precision=prec)
            assert np.array_equal(bits64(f), bits64(fs)) and np.array_equal(t, ts), (n1, n, s)
            ref = reference(sg, orc, n, s)
            assert np.array_equal(bits64(f), bits64(ref["fitness"])) and np.array_equal(t, ref["trades"]), (n1, n, s)


# ----------------------------------------------------------------------------------------------
# C. graph capture
# ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [32, 256])
def test_captured_generation_replays_across_a_retired_buffer(sg, orc, hidden):
    """A captured GA generation (H = 32 small population; EXACT at H = 256) replayed, then a larger population trace on
    the same train and val bundles (both outgrow the captured buffers, which must be retired, not freed), then replayed
    again: history and masters equal an eager GA bit for bit, the trace equals the oracle."""
    from sgmm_b200 import synthetic as syn
    from sgmm_b200.engine import DeviceGA
    tb, stats, tz = episode(orc, T0)
    vb = tuple(a[:240] for a in syn.synthetic_bundle(1, first_day=140))
    master = syn.policy_like_genomes(1, hidden=hidden, seed=17, out_scale=2.0, out_bias=(0.1, 0.1))[0]
    pop = 24 if hidden == 32 else 4
    kw = dict(pop_size=pop, sigma=0.05, phi=PHI, fee_rate=FEE, use_arl=False, seed=9, max_generations=6, patience=2, hidden=hidden,
              precision=None if hidden == 32 else "exact")
    bundles = lambda: (sg.Bundle.from_arrays(tb, stats, TICK), sg.Bundle.from_arrays(vb, stats, TICK))
    train_e, val_e = bundles()
    eager = DeviceGA(master, None, **kw)
    for _ in range(5):
        eager.generation(train_e, val_e)
    train, val = bundles()
    graphed = DeviceGA(master, None, **kw)
    graphed.generation(train, val)
    torch.cuda.synchronize()
    g = graphed.capture(train, val)
    g.replay()
    g.replay()
    P = 130                                         # 651 T words: beyond 1.25x what either generation reserved
    G, A = mm_genomes(P, 32, 77, ADV_SCALE), adv_genomes(P, 77)
    f, t, cols = sg.rollout_trace_population(train, torch.from_numpy(G).cuda(), torch.from_numpy(A).cuda(), phi=PHI, fee_rate=FEE)
    fv, tv, _ = sg.rollout_trace_population(val, torch.from_numpy(G).cuda(), torch.from_numpy(A).cuda(), phi=PHI, fee_rate=FEE,
                                            columns=("wealth",))
    g.replay()
    g.replay()
    torch.cuda.synchronize()
    fo, to = orc.rollout_population(tz, PHI, TICK, FEE, genomes=G, adv_genomes=A, use_adv=True, nthreads=8)
    assert np.array_equal(bits64(f.cpu().numpy()), bits64(fo)) and np.array_equal(t.cpu().numpy(), to)
    vz = tuple(orc.normalise(vb, stats)) + tuple(vb[2:])
    fvo, tvo = orc.rollout_population(vz, PHI, TICK, FEE, genomes=G, adv_genomes=A, use_adv=True, nthreads=8)
    assert np.array_equal(bits64(fv.cpu().numpy()), bits64(fvo)) and np.array_equal(tv.cpu().numpy(), tvo)
    for i in (0, 1, P - 1):
        _, _, tro = orc.rollout(G[i], A[i], tz, PHI, TICK, FEE, trace=True)
        for k in ORACLE_COLS:
            assert np.array_equal(cols[k][i].cpu().numpy().view(np.uint8), tro[k].view(np.uint8)), (i, k)
    he, hg = eager.history(5), graphed.history(5)
    for k in he:
        assert np.array_equal(he[k].view(np.uint8), hg[k].view(np.uint8)), k
    for x, y in zip(eager.masters(), graphed.masters()):
        assert np.array_equal(bits32(x), bits32(y))
    assert graphed.status()["generation"] == 5
    eager.close()
    graphed.close()


def _capture(fn):
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    return graph, out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["small32", "spec256", "spec256_adv", "exact256", "tracepop32_adv"])
def test_capture_refuses_a_buffer_it_would_have_to_grow(sg, orc, name):
    """Under a capture the buffer cannot grow: the call is refused with its message, the capture ends cleanly, eager calls
    stay correct, and a capture made after one eager call of that size replays correctly."""
    ref_big = reference(sg, orc, name, "big")         # (populations uploaded before any capture)
    bun = fresh(sg, orc, T0)
    assert_same(run(sg, bun, name, "normal"), reference(sg, orc, name, "normal"), "eager")
    torch.cuda.synchronize()
    with pytest.raises(sg.SgmmError) as err:
        _capture(lambda: run(sg, bun, name, "big"))
    assert err.value.code == -1 and "run one rollout of this size outside the stream capture first" in str(err.value)
    assert not torch.cuda.is_current_stream_capturing()
    assert_same(run(sg, bun, name, "big"), ref_big, "eager after the refusal")
    torch.cuda.synchronize()
    graph, out = _capture(lambda: run(sg, bun, name, "big"))
    graph.replay()
    torch.cuda.synchronize()
    assert_same(out, ref_big, "replay")
    assert_same(run(sg, bun, name, "normal"), reference(sg, orc, name, "normal"), "eager after the replay")


@pytest.mark.gpu
def test_capture_refuses_a_fee_rate_without_leg_table(sg, orc):
    """A tensor-core adversary rollout at a new fee rate under capture is refused; afterwards the eager call and a capture
    of it equal a fresh bundle."""
    bun = fresh(sg, orc, T0)
    run(sg, bun, "tc32_adv", "normal")
    torch.cuda.synchronize()
    with pytest.raises(sg.SgmmError) as err:
        _capture(lambda: run(sg, bun, "tc32_adv", "normal", fee=2e-4))
    assert err.value.code == -1 and "no leg table for fee_rate" in str(err.value)
    assert not torch.cuda.is_current_stream_capturing()
    ref = host(run(sg, fresh(sg, orc, T0), "tc32_adv", "normal", fee=2e-4))
    assert_same(run(sg, bun, "tc32_adv", "normal", fee=2e-4), ref, "eager after the refusal")
    torch.cuda.synchronize()
    graph, out = _capture(lambda: run(sg, bun, "tc32_adv", "normal", fee=2e-4))
    graph.replay()
    torch.cuda.synchronize()
    assert_same(out, ref, "replay")


# ----------------------------------------------------------------------------------------------
# D. leg tables and fee keys
# ----------------------------------------------------------------------------------------------
FEES_D = (3e-4, 0.0, -1e-4, 3e-4, -0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "tf32", "f16"])
def test_leg_tables_over_two_streams(sg, orc, precision):
    """One bundle, fee rates 3e-4, 0, -1e-4, 3e-4, -0.0 alternating over two side streams: each equals a fresh bundle."""
    pop = population("tc32_adv", "normal")
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    bun = fresh(sg, orc, T0)
    torch.cuda.synchronize()
    outs = []
    for i, fee in enumerate(FEES_D):
        with torch.cuda.stream(streams[i % 2]):
            outs.append(sg.rollout_tc_audit(bun, pop["g"], pop["a"], phi=PHI, fee_rate=fee, hidden=32, precision=precision))
    torch.cuda.synchronize()
    for fee, out in zip(FEES_D, outs):
        ref = sg.rollout_tc_audit(fresh(sg, orc, T0), pop["g"], pop["a"], phi=PHI, fee_rate=fee, hidden=32, precision=precision)
        assert_same(dict(enumerate(out)), dict(enumerate(ref)), (precision, fee))


@pytest.mark.gpu
def test_negative_zero_fee_rate_equals_the_oracle(sg, orc):
    """fee_rate = -0.0 on a bundle that has already run every route at fee 0.0: the exact routes equal the oracle run with
    -0.0 bit for bit (the sign of zero of fee_paid / cum_fees of both traces included), the tensor-core routes the oracle's
    env driven by their offsets."""
    bun = fresh(sg, orc, T0)
    for name in NAMES:
        run(sg, bun, name, "normal", fee=0.0)
    _, _, bz = episode(orc, T0)
    for name in NAMES:
        out = run(sg, bun, name, "normal", fee=-0.0)
        if name in TENSOR:
            check_replay(orc, name, "normal", out, T0, -0.0)
            assert_same(out, run(sg, fresh(sg, orc, T0), name, "normal", fee=-0.0), (name, "fresh"))
        else:
            check_oracle(orc, name, "normal", out, T0, fee=-0.0)
    g, a = population("small32_adv", "normal")["G"][2], population("small32_adv", "normal")["A"][2]
    f, t, tr = sg.rollout_trace(bun, g, a, phi=PHI, fee_rate=-0.0)
    fo, to, tro = orc.rollout(g, a, bz, PHI, TICK, -0.0, trace=True)
    assert (bits64(f), t) == (bits64(fo), to) and tro["fill_buy"].any()
    for k in ORACLE_COLS:
        assert np.array_equal(tr[k].view(np.uint8), tro[k].view(np.uint8)), k
    assert np.array_equal(bits64(tr["cum_fees"]), bits64(np.cumsum(tro["fee_paid"])))


@pytest.mark.gpu
def test_sixty_four_leg_tables_then_refusal(sg, orc):
    """64 distinct fee rates build 64 leg tables; the 65th is refused with SGMM_ERR_NOMEM and its message; the first 64
    still give what a fresh bundle gives."""
    pop = population("tc32_adv", "normal")
    fees = [k * 1e-5 for k in range(64)]
    call = lambda b, fee: sg.rollout_tc_audit(b, pop["g"], pop["a"], phi=PHI, fee_rate=fee, hidden=32, precision="bf16")
    bun = fresh(sg, orc, T0)
    first = [host(dict(enumerate(call(bun, fee)))) for fee in fees]
    with pytest.raises(sg.SgmmError) as err:
        call(bun, 7.77e-4)
    assert err.value.code == -3 and "more than 64 distinct fee rates on one bundle" in str(err.value)
    for fee, one in zip(fees, first):
        assert_same(dict(enumerate(call(bun, fee))), one, (fee, "again"))
        assert_same(dict(enumerate(call(fresh(sg, orc, T0), fee))), one, (fee, "fresh"))
