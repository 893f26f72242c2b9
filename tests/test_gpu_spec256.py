"""GPU (-m gpu): the H=256 tensor-core path (tcgen05; f16 operands, f16 layer-2 accumulator in TMEM, fp32 output layer;
BASELINE.json config 4).  The rollout kernel does the integer half of the env step and records 64-bit step codes; the
fp64 accounting is a second kernel (sgmm_account.cu).  Parity is stated in two halves:

  (1) POLICY OUTPUTS vs the fp32 oracle (SGMM-F32 order, oracle/sgmm_oracle.c) for EVERY (bar,
      inventory) pair: |d(raw*5)| <= TAU_TICKS, and the rounded offsets are identical wherever the
      oracle's own distance to a rounding boundary exceeds TAU_TICKS (no tick flips outside the
      stated tolerance);
  (2) GIVEN the offsets the kernel took, fills, inventory, trade count, rewards and fitness are
      BIT-IDENTICAL to the oracle's env (teacher-forced replay of the kernel's action trace).
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TAU_TICKS = 0.05          # stated tolerance on raw*5 (ticks); measured max is 0.008 (f16), 0.025 with bf16 operands


@pytest.fixture(scope="module")
def sg():
    assert torch.cuda.is_available()
    import sgmm_b200
    return sgmm_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


def _setup(sg, orc, days, first_day, P, seed, T=None, out_scale=4.0):
    from sgmm_b200 import synthetic
    bundle = synthetic.synthetic_bundle(days, first_day=first_day)
    if T is not None:
        bundle = tuple(a[:T] for a in bundle)
    stats = synthetic.train_stats_of(synthetic.synthetic_bundle(days, first_day=first_day))
    z1, z2 = orc.normalise(bundle, stats)
    bun = sg.Bundle.from_arrays(bundle, stats, 0.001)
    _, genomes = synthetic.policy_like_genomes(P, hidden=256, seed=seed, out_scale=out_scale, out_bias=(0.1, 0.1))
    return bundle, (z1, z2) + bundle[2:], bun, genomes


@pytest.mark.parametrize("fee", [0.0, 3e-4])
def test_policy_outputs_within_tolerance_and_env_bit_exact(sg, orc, fee):
    bundle, bz, bun, genomes = _setup(sg, orc, 1, 90, 4, seed=11)
    T = bun.T
    fit, trd, raw, act = sg.rollout_spec256_audit(bun, genomes, phi=1e-4, fee_rate=fee)
    fit, trd, raw, act = fit.cpu().numpy(), trd.cpu().numpy(), raw.cpu().numpy(), act.cpu().numpy()
    worst = 0.0
    flips_outside = 0
    for i in range(genomes.shape[0]):
        for t in range(T):
            for iv in range(5):
                want = orc.mlp_forward(genomes[i], [bz[0][t], bz[1][t], (iv - 2) / 2.0], hidden=256)
                q_o = want * np.float32(5.0)
                q_k = raw[i, t, iv] * np.float32(5.0)
                worst = max(worst, float(np.max(np.abs(q_o - q_k))))
                margin = np.abs(np.abs(q_o - np.floor(q_o)) - 0.5)
                k_o, k_k = np.rint(q_o), np.rint(q_k)
                flips_outside += int(np.sum((k_o != k_k) & (margin > TAU_TICKS)))
        # (2) teacher-forced: the oracle's env on the kernel's own action trace
        fo, to, tro = orc.rollout(None, None, bz, 1e-4, 0.001, fee, forced_actions=act[i], trace=True)
        assert fo == fit[i] and to == trd[i], (i, fo, fit[i], to, trd[i])
        # the trace is the policy's choice at the walked inventory
        inv_before = np.concatenate([[0], tro["inventory"][:-1]])
        taken = np.rint(raw[i, np.arange(T), inv_before + 2] * np.float32(5.0)).astype(np.int32)
        assert np.array_equal(taken, act[i])
    print(f"max |d(raw*5)| = {worst:.4g} ticks (tolerance {TAU_TICKS})")
    assert worst <= TAU_TICKS
    assert flips_outside == 0


@pytest.mark.parametrize("T", [1, 24, 25, 26, 51, 130])
def test_ragged_lengths_and_many_individuals(sg, orc, T):
    P = 150 if T <= 26 else 5            # more individuals than SMs exercises the persistent loop
    bundle, bz, bun, genomes = _setup(sg, orc, 1, 91, P, seed=T, T=T)
    fit, trd, raw, act = sg.rollout_spec256_audit(bun, genomes, phi=1e-4)
    f2, t2 = sg.rollout_population(bun, torch.from_numpy(genomes).cuda(), phi=1e-4, hidden=256)
    assert torch.equal(f2, fit) and torch.equal(t2, trd)
    fit, trd, act = fit.cpu().numpy(), trd.cpu().numpy(), act.cpu().numpy()
    for i in range(0, P, max(1, P // 7)):
        fo, to = orc.rollout(None, None, bz, 1e-4, 0.001, 0.0, forced_actions=act[i])
        assert fo == fit[i] and to == trd[i]


@pytest.mark.parametrize("out_scale,fee", [(300.0, 0.0), (40000.0, 3e-4)])
def test_large_offsets_through_the_step_codes(sg, orc, out_scale, fee):
    """Offsets of hundreds to tens of thousands of ticks (both signs, both sides filling in one bar): the two int32 offset
    fields of the step code and the accounting kernel reproduce the oracle's env bit for bit on the kernel's actions."""
    bundle, bz, bun, genomes = _setup(sg, orc, 1, 93, 9, seed=3, T=333, out_scale=out_scale)
    fit, trd, raw, act = sg.rollout_spec256_audit(bun, genomes, phi=1e-4, fee_rate=fee)
    fit, trd, act = fit.cpu().numpy(), trd.cpu().numpy(), act.cpu().numpy()
    assert np.abs(act).max() > 50 * out_scale / 300.0          # the case is what it claims to be
    both = 0
    for i in range(genomes.shape[0]):
        fo, to, tro = orc.rollout(None, None, bz, 1e-4, 0.001, fee, forced_actions=act[i], trace=True)
        assert fo == fit[i] and to == trd[i], (i, fo, fit[i], to, trd[i])
        both += int(np.sum(tro["fill_buy"] & tro["fill_sell"])) if "fill_buy" in tro else 0
    print("bars with both sides filled:", both)


def test_closed_loop_diverges_from_fp32_oracle_only_at_near_ties(sg, orc):
    """Closed loop against the fp32 oracle: the walked trajectory is identical to the oracle's up to
    the first bar where the oracle's own raw*5 is within TAU_TICKS of a rounding boundary (bf16 may
    round the other way there; the MDP is chaotic afterwards, SURVEY.md 7.4-1)."""
    bundle, bz, bun, genomes = _setup(sg, orc, 2, 92, 6, seed=5)
    fit, trd, raw, act = sg.rollout_spec256_audit(bun, genomes, phi=1e-4)
    fit, trd, act = fit.cpu().numpy(), trd.cpu().numpy(), act.cpu().numpy()
    identical = 0
    for i in range(genomes.shape[0]):
        fo, to, tro = orc.rollout(genomes[i], None, bz, 1e-4, 0.001, 0.0, hidden=256, trace=True)
        diff = (tro["off_a"] != act[i, :, 0]) | (tro["off_b"] != act[i, :, 1])
        if not diff.any():
            identical += 1
            assert fo == fit[i] and to == trd[i]
            continue
        t = int(np.argmax(diff))
        q = np.array([tro["raw_a"][t], tro["raw_b"][t]], np.float32) * np.float32(5.0)
        margin = np.min(np.abs(np.abs(q - np.floor(q)) - 0.5))
        assert margin <= TAU_TICKS, (i, t, q)
    print("closed-loop trajectories identical to the fp32 oracle:", identical, "of", genomes.shape[0])


def test_seeded_children_and_argument_checks(sg, orc):
    from sgmm_b200 import _lib
    bundle, bz, bun, genomes = _setup(sg, orc, 1, 93, 1, seed=3, T=60)
    master = genomes[0]
    kids = np.stack([orc.mutate(master, 0.05, 77, 4, 10 + i) for i in range(5)])
    f_exp, t_exp = sg.rollout_population(bun, torch.from_numpy(kids).cuda(), phi=1e-4, hidden=256)
    f_seed, t_seed = sg.rollout_seeded(bun, torch.from_numpy(master).cuda(), count=5, sigma=0.05, seed=77,
                                       generation=4, first_index=10, phi=1e-4, hidden=256)
    assert torch.equal(f_exp, f_seed) and torch.equal(t_exp, t_seed)
    import ctypes as C
    g = torch.from_numpy(genomes).cuda()
    mm = _lib.Population(256, 0, 1, g.data_ptr(), None, 0.0, 0.0, 0, 0, 0)
    prm = _lib.RolloutParams(1e-4, 0.0, 0, 0, 0, 0)              # precision F32 with H=256: refused loudly
    out_f = torch.empty(1, dtype=torch.float64, device="cuda")
    out_t = torch.empty(1, dtype=torch.int32, device="cuda")
    rc = _lib.lib().sgmm_rollout_population(bun.handle, C.byref(mm), None, C.byref(prm), out_f.data_ptr(),
                                            out_t.data_ptr(), None)
    assert rc == _lib.ERR_UNSUPPORTED
