"""Closed-loop control on the CUDA library (step_kernel_targets and observations_kernel) against the oracle with joint targets
(tests/oracle_ext), bit for bit: state, observations, fitness, ticks and counters, over three encodings, every forced group
shift, mixed plain and target calls, held targets, the 33-44-body class, sine outputs fed back as targets, and a 300-tick
feedback loop over 4096 creatures. The fast library exports the functions and runs them. Needs a GPU; tests/test_closed_loop.py
checks the oracle and the device code on the CPU."""
import os
import random
import sys

import numpy as np
import pytest

from gym_rem2d_b200 import Individual, constants as K, terrain
from gym_rem2d_b200.capi import Engine
from gym_rem2d_b200.env import BatchedModular2D
from gym_rem2d_b200.flatten import flatten_population
from gym_rem2d_b200.population import random_population

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "oracle_ext"))
from oracle_ext import OracleExtEngine  # noqa: E402

pytestmark = pytest.mark.gpu

STATE = ("pose", "vel", "joint_impulse", "limit_state", "motor_speed", "alive", "ticks", "awake", "wod", "n_contacts",
         "n_touching", "touching_pairs", "touching_impulse")
OBS = ("joint_angle", "joint_speed", "root", "ground")
THREADS = max(8, os.cpu_count() or 8)


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def pair(pop, ys, precision="exact", **options):
    g = Engine(device=0, precision=precision)
    o = OracleExtEngine(threads=THREADS)
    for e in (g, o):
        e.set_terrain(ys, K.TERRAIN_STEP)
    for k, v in options.items():
        g.set_option(k, v)
    for e in (g, o):
        e.upload(pop)
    return g, o


def assert_same_run(g, o, what, max_pairs=16):
    sg, so = g.read_state(max_pairs=max_pairs), o.read_state(max_pairs=max_pairs)
    for k in STATE:
        assert same(sg[k], so[k]), "%s: %s differs in %d values" % (what, k, (sg[k] != so[k]).sum())
    og, oo = g.read_observations(), o.read_observations()
    for k in OBS:
        assert same(og[k], oo[k]), "%s: observation %s differs in %d values" % (what, k, (og[k] != oo[k]).sum())
    assert same(g.fitness(), o.fitness()) and same(g.ticks(), o.ticks()), what
    assert g.counters() == o.counters(), what


def drive(engines, pop, n_calls, n_ticks, seed, plain_every=0):
    """Mixed calls on every engine: random targets in [-pi/2, pi/2] held for n_ticks, a plain call every plain_every-th."""
    rng = np.random.default_rng(seed)
    nj = pop.n_bodies - pop.n_creatures
    for i in range(n_calls):
        t = rng.uniform(-np.pi / 2, np.pi / 2, nj)
        for e in engines:
            if plain_every and i % plain_every == plain_every - 1:
                e.step(n_ticks)
            else:
                e.step_targets(t, n_ticks)


@pytest.mark.parametrize("gs", range(6))
@pytest.mark.parametrize("enc,seed", [("direct", 31), ("lsystem", 32), ("ce", 33)])
def test_targets_match_the_oracle(enc, seed, gs):
    random.seed(seed)
    pop = flatten_population([Individual.random(encoding=enc) for _ in range(96)])
    xs, ys = terrain.generate_terrain()
    g, o = pair(pop, ys, group_shift=gs)
    for n_ticks, plain_every in ((1, 4), (7, 3)):
        drive((g, o), pop, 12, n_ticks, seed * 10 + gs + n_ticks, plain_every)
        assert_same_run(g, o, "%s gs %d n_ticks %d" % (enc, gs, n_ticks))
    g.close()


def test_targets_match_the_oracle_in_the_largest_class():
    """A population as run_deap configures it (max_size 40): the 33-44-body class is filled."""
    from gym_rem2d_b200 import ea
    from gym_rem2d_b200.modules import get_module_list
    random.seed(21); np.random.seed(21)
    cfg = ea.default_config(enc="lsystem")
    base = flatten_population([Individual.random(get_module_list(), cfg) for _ in range(640)], 7)
    nb = np.diff(base.body_off)
    pop = base.select(np.nonzero(nb > 16)[0])
    assert (np.diff(pop.body_off) > 32).sum() > 40
    xs, ys = terrain.generate_terrain()
    g, o = pair(pop, ys)
    drive((g, o), pop, 20, 1, 5, plain_every=5)
    assert_same_run(g, o, "33-44 class, 1 tick", max_pairs=32)
    drive((g, o), pop, 6, 7, 6, plain_every=3)
    assert_same_run(g, o, "33-44 class, 7 ticks", max_pairs=32)
    g.close()


@pytest.mark.parametrize("enc", ["direct", "lsystem", "ce"])
def test_sine_outputs_as_targets_reproduce_plain_stepping_on_cuda(enc):
    random.seed(50 + len(enc))
    pop = flatten_population([Individual.random(encoding=enc) for _ in range(256)])
    xs, ys = terrain.generate_terrain()
    plain, ctl = Engine(device=0), Engine(device=0)
    o = OracleExtEngine()
    for e in (plain, ctl, o):
        e.set_terrain(ys, K.TERRAIN_STEP)
        e.upload(pop)
    T = 150
    sine = o.sine_outputs(T)
    for t in range(T):
        plain.step(1)
        ctl.step_targets(sine[t], 1)
        if t % 15 == 14:
            a, b = plain.read_state(max_pairs=16), ctl.read_state(max_pairs=16)
            for k in STATE:
                assert same(a[k], b[k]), "%s tick %d: %s" % (enc, t, k)
    assert same(plain.fitness(), ctl.fitness()) and same(plain.ticks(), ctl.ticks())
    assert plain.counters() == ctl.counters()
    plain.close(); ctl.close()


def test_closed_loop_feedback_run_matches_the_oracle():
    """4096 creatures, 300 ticks, each engine driven by a feedback policy of its own observations."""
    pop = random_population(4096, ("lsystem",), seed=61, workers=8)
    xs, ys = terrain.generate_terrain()
    g, o = pair(pop, ys)
    creature = np.repeat(np.arange(pop.n_creatures), np.diff(pop.body_off) - 1)
    phase = np.arange(pop.n_bodies - pop.n_creatures) * 0.7

    def policy(ob, t):
        grounded = ob["ground"][np.asarray(pop.body_off[:-1])][creature]
        return (-0.8 * ob["joint_angle"].astype(np.float64) - 0.05 * ob["joint_speed"] + 0.6 * np.sin(0.2 * t + phase)
                + 0.3 * grounded)

    for t in range(300):
        for e in (g, o):
            e.step_targets(policy(e.read_observations(), t), 1)
    assert_same_run(g, o, "closed loop")
    assert (g.ticks() == 300).any() and (g.ticks() < 300).any()
    g.close()


def test_batched_env_on_cuda():
    random.seed(71)
    individuals = [Individual.random(encoding="lsystem") for _ in range(64)]
    env = BatchedModular2D(device=0)
    env.reset(individuals)
    o = OracleExtEngine()
    o.set_terrain(env.terrain_y, K.TERRAIN_STEP)
    o.upload(env.table)
    for t in range(40):
        target = -0.5 * env.observe()["joint_angle"].astype(np.float64)
        env.step(1, targets=target)
        o.step_targets(-0.5 * o.read_observations()["joint_angle"].astype(np.float64), 1)
    for k in OBS:
        assert same(env.observe()[k], o.read_observations()[k]), k
    env.close()


def test_fast_library_exports_and_runs_targets():
    """The fused-multiply-add build takes targets and observes; its results are not bit-compared (contraction changes the
    controller line), only checked for sanity."""
    random.seed(81)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(128)])
    xs, ys = terrain.generate_terrain()
    g = Engine(device=0, precision="fast")
    assert hasattr(g.lib, "rem2d_step_targets") and hasattr(g.lib, "rem2d_read_observations")
    g.set_terrain(ys, K.TERRAIN_STEP)
    g.upload(pop)
    for t in range(50):
        ob = g.read_observations()
        g.step_targets(-0.5 * ob["joint_angle"].astype(np.float64), 1)
    ob = g.read_observations()
    assert all(np.isfinite(ob[k]).all() for k in ("joint_angle", "joint_speed", "root"))
    assert (g.ticks() > 0).all() and set(np.unique(ob["ground"])) <= {0, 1}
    g.close()
