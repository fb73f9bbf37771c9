"""Per-joint feedback policies on the CUDA library (the policy images: episode_kernel_policy, episode_kernel_policy_r128 and
step_kernel_policy) against the oracle with the policy (tests/oracle_policy), bit for bit in fitness, ticks, statistics and counters,
under every execution strategy: bulk and warp mode, forced group widths, parking with tails, the overflow wave, the 128-register
image, regrouping of draining warps, re-runs after a capacity overflow and the 33-44-body class, over three encodings; policy
stepping tick by tick; zero weights against open loop on CUDA; a 65536-creature evaluation; the fast library runs the policy path;
the call contract is the oracle's. Needs a GPU; tests/test_policy.py checks the oracle and the device code on the CPU."""
import os
import random
import sys

import numpy as np
import pytest

from gym_rem2d_b200 import Individual, constants as K, policy, terrain
from gym_rem2d_b200.capi import Engine
from gym_rem2d_b200.flatten import flatten_population
from gym_rem2d_b200.population import random_population

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "oracle_policy"))
from oracle_policy import OraclePolicyEngine  # noqa: E402
from tests.test_policy import assert_state_equal, assert_stats_equal, check_contract, n_joints, same  # noqa: E402

pytestmark = pytest.mark.gpu

BULK, WARP = "0", "1000000"
THREADS = max(8, os.cpu_count() or 8)


def weights(pop, H=8, scale=0.05, seed=0):
    """Small feedback (many creatures still live long enough to be parked), or large with scale ~1."""
    return policy.random_weights(n_joints(pop), H, scale, rng=seed)


def oracle_eval(pop, ys, W, max_ticks=K.EVALUATION_STEPS, step=K.TERRAIN_STEP):
    o = OraclePolicyEngine(threads=THREADS)
    o.set_terrain(ys, step)
    o.set_stats(True)
    if W is not None:
        o.set_policy(W)
    f, t = o.evaluate(pop, max_ticks)
    return f, t, o.counters(), o.read_stats()


def gpu_eval(pop, ys, W, max_ticks=K.EVALUATION_STEPS, step=K.TERRAIN_STEP, stats=True, precision="exact", **options):
    g = Engine(device=0, precision=precision)
    g.set_terrain(ys, step)
    for k, v in options.items():
        g.set_option(k, v)
    g.set_stats(stats)
    if W is not None:
        g.set_policy(W)
    f, t = g.evaluate(pop, max_ticks)
    out = f, t, g.counters(), (g.read_stats() if stats else None)
    g.close()
    return out


def assert_run_equal(a, b, what):
    (fa, ta, ca, sa), (fb, tb, cb, sb) = a, b
    assert same(ta, tb) and same(fa, fb), what
    assert ca == cb, what
    assert_stats_equal(sa, sb, what)


@pytest.mark.parametrize("mode", [BULK, WARP])
@pytest.mark.parametrize("enc,n,seed,H,scale", [("direct", 512, 11, 1, 0.05), ("lsystem", 512, 12, 8, 0.1), ("ce", 256, 13, 16, 1.0)])
def test_full_episodes_match_the_oracle(enc, n, seed, H, scale, mode, monkeypatch):
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", mode)
    random.seed(seed)
    pop = flatten_population([Individual.random(encoding=enc) for _ in range(n)])
    xs, ys = terrain.generate_terrain()
    W = weights(pop, H, scale, seed)
    ref = oracle_eval(pop, ys, W)
    assert_run_equal(gpu_eval(pop, ys, W), ref, "%s mode %s" % (enc, mode))
    # without statistics the policy images accumulate into scratch: same results
    f0, t0, c0, _ = gpu_eval(pop, ys, W, stats=False)
    assert same(f0, ref[0]) and same(t0, ref[1]) and c0 == ref[2]


def test_forced_group_widths_parking_and_tails():
    pop = random_population(1024, ("lsystem",), seed=81, workers=4)
    xs, ys = terrain.generate_terrain()
    W = weights(pop, 8, 0.05, 81)
    ref = oracle_eval(pop, ys, W)
    assert (ref[1] > 140).sum() > 20                       # long-lived creatures: parked and finished by tail launches
    for gs in range(6):
        assert_run_equal(gpu_eval(pop, ys, W, warp_mode_max=0, group_shift=gs, tail_group_shift=max(gs, 1), smem_budget_kb=16,
                                  park_ticks=130), ref, "group_shift %d" % gs)
    for park in (8, 64, 0):
        assert_run_equal(gpu_eval(pop, ys, W, warp_mode_max=0, park_ticks=park), ref, "park_ticks %d" % park)


def test_ea_configured_population_overflow_wave_image_and_largest_class():
    """A population as run_deap configures it, tiled: the overflow wave runs, and the 33-44-body class is filled."""
    from gym_rem2d_b200 import ea
    from gym_rem2d_b200.modules import get_module_list
    random.seed(21); np.random.seed(21)
    cfg = ea.default_config(enc="lsystem")
    base = flatten_population([Individual.random(get_module_list(), cfg) for _ in range(2048)], 7)
    assert (np.diff(base.body_off) > 32).sum() > 40
    xs, ys = terrain.generate_terrain()
    Wb = weights(base, 8, 0.05, 21)
    fo, to, co, so = oracle_eval(base, ys, Wb)
    tiles = 24
    idx = np.tile(np.arange(2048), tiles)
    pop = base.select(idx)
    nbs = np.diff(base.body_off)
    j0 = np.asarray(base.body_off[:-1], np.int64) - np.arange(2048)
    W = Wb[np.concatenate([np.arange(j0[c], j0[c] + nbs[c] - 1) for c in idx])]
    bodies = np.concatenate([np.arange(base.body_off[c], base.body_off[c + 1]) for c in idx])
    want = {k: (v[bodies] if k == "ground_ticks" else v[idx]) for k, v in so.items()}
    for options in (dict(), dict(overflow_wave=0), dict(image=1)):
        f, t, c, s = gpu_eval(pop, ys, W, **options)
        assert same(t, np.tile(to, tiles)) and same(f, np.tile(fo, tiles)), options
        assert_stats_equal(s, want, str(options))


@pytest.mark.parametrize("mode", [BULK, WARP])
def test_capacity_overflow_reruns(mode, monkeypatch):
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", mode)
    random.seed(41)
    pop = flatten_population([Individual.random(encoding="direct") for _ in range(96)])
    ys = np.full(200, 5.0)
    W = weights(pop, 4, 0.1, 41)
    ref = oracle_eval(pop, ys, W, 150, step=0.15)
    assert_run_equal(gpu_eval(pop, ys, W, 150, step=0.15), ref, "overflow %s" % mode)


@pytest.mark.parametrize("options", [
    dict(warp_mode_max=0, park_ticks=0, smem_budget_kb=24),
    dict(warp_mode_max=0, park_ticks=0, smem_budget_kb=40, group_shift=0),
    dict(warp_mode_max=0, park_ticks=140, park_cap=0.0625, tail_group_shift=1, smem_budget_kb=24),
])
def test_draining_warps(options):
    pop = random_population(3072, ("lsystem",), seed=71, workers=4)
    xs, ys = terrain.generate_terrain()
    W = weights(pop, 8, 0.05, 71)
    assert_run_equal(gpu_eval(pop, ys, W, **options), oracle_eval(pop, ys, W), str(options))


@pytest.mark.parametrize("gs", [None, 0, 1, 2, 3, 4, 5])
@pytest.mark.parametrize("enc,seed", [("direct", 31), ("lsystem", 32), ("ce", 33)])
def test_policy_stepping_matches_the_oracle(enc, seed, gs):
    random.seed(seed)
    pop = flatten_population([Individual.random(encoding=enc) for _ in range(96)])
    xs, ys = terrain.generate_terrain()
    W = weights(pop, 8, 1.0, seed)
    g, o = Engine(device=0), OraclePolicyEngine(threads=THREADS)
    if gs is not None:
        g.set_option("group_shift", gs)
    for e in (g, o):
        e.set_terrain(ys, K.TERRAIN_STEP)
        e.set_policy(W)
        e.upload(pop)
    for t in range(60):
        for e in (g, o):
            e.step(1 + t % 3)
        if t % 6 == 5:
            assert_state_equal(g.read_state(max_pairs=16), o.read_state(max_pairs=16), "%s gs %s call %d" % (enc, gs, t))
    assert same(g.fitness(), o.fitness()) and same(g.ticks(), o.ticks()) and g.counters() == o.counters()
    g.close()


def test_zero_weights_equal_open_loop_on_cuda():
    pop = random_population(4096, ("lsystem", "ce"), seed=91, workers=8)
    xs, ys = terrain.generate_terrain()
    zero = np.zeros((n_joints(pop), policy.n_params(8)))
    assert_run_equal(gpu_eval(pop, ys, zero), gpu_eval(pop, ys, None), "zero weights")


def test_bench_sized_population_matches_the_oracle_on_a_subset():
    """65536 creatures with a policy on the GPU; creatures are independent, so 4096 of them alone on the oracle."""
    pop = random_population(65536, ("lsystem",), seed=2024, workers=8)
    xs, ys = terrain.generate_terrain()
    W = weights(pop, 8, 0.05, 2024)
    f, t, c, s = gpu_eval(pop, ys, W)
    sub = np.random.default_rng(5).choice(65536, 4096, replace=False)
    nbs = np.diff(pop.body_off)
    j0 = np.asarray(pop.body_off[:-1], np.int64) - np.arange(pop.n_creatures)
    Ws = W[np.concatenate([np.arange(j0[c], j0[c] + nbs[c] - 1) for c in sub])]
    fo, to, co, so = oracle_eval(pop.select(sub), ys, Ws)
    assert same(f[sub], fo) and same(t[sub], to)
    bodies = np.concatenate([np.arange(pop.body_off[c], pop.body_off[c + 1]) for c in sub])
    assert_stats_equal({k: (v[bodies] if k == "ground_ticks" else v[sub]) for k, v in s.items()}, so, "subset")


def test_fast_build_runs_the_policy():
    pop = random_population(2048, ("lsystem",), seed=92, workers=4)
    xs, ys = terrain.generate_terrain()
    W = weights(pop, 8, 1.0, 92)
    f0, t0, _, _ = gpu_eval(pop, ys, None, precision="fast", stats=False)
    f1, t1, _, s1 = gpu_eval(pop, ys, W, precision="fast")
    assert not same(f0, f1) and s1["ground_ticks"].shape == (pop.n_bodies,) and (s1["end_reason"] > 0).all()
    g = Engine(device=0, precision="fast")
    g.set_terrain(ys, K.TERRAIN_STEP)
    g.set_policy(W)
    g.upload(pop)
    g.step(20)
    assert g.ticks().max() == 20
    g.close()


def test_contract_equals_the_oracle():
    xs, ys = terrain.generate_terrain()

    def make():
        g = Engine(device=0)
        g.set_terrain(ys, K.TERRAIN_STEP)
        return g
    random.seed(3)
    check_contract(make, ys, flatten_population([Individual.random(encoding="direct") for _ in range(16)]))
