"""Closed-loop control of stepping runs (rem2d_step_targets / rem2d_read_observations, include/rem2d_control.h) on the CPU: the
oracle with the extension headers (tests/oracle_ext) against plain oracle stepping and against the stated control rule, the
frozen sine controllers, the observations against read_state, the call contract, the Python layer, and the device code of
step_kernel_targets and of the observation gather (-DREM2D_TARGETS, the targets build of the emulation in tests/emu) against the
oracle, bit for bit."""
import ctypes as C
import os
import random
import sys

import numpy as np
import pytest

from gym_rem2d_b200 import Individual, constants as K, terrain
from gym_rem2d_b200.capi import Observation, Rem2dError
from gym_rem2d_b200.env import BatchedModular2D
from gym_rem2d_b200.flatten import flatten_population
from oracle.oracle import OracleEngine

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))
sys.path.insert(0, os.path.join(HERE, "oracle_ext"))
import emu  # noqa: E402
import oracle_ext  # noqa: E402
from oracle_ext import OracleExtEngine  # noqa: E402

STATE = ("pose", "vel", "joint_impulse", "limit_state", "motor_speed", "alive", "ticks", "awake", "wod", "n_contacts",
         "n_touching", "touching_pairs", "touching_impulse")
OBS = ("joint_angle", "joint_speed", "root", "ground")


def population(enc, n, seed):
    random.seed(seed)
    return flatten_population([Individual.random(encoding=enc) for _ in range(n)])


def engine(cls, ys, pop=None, **cfg):
    e = cls(threads=8, **cfg)
    e.set_terrain(ys, K.TERRAIN_STEP)
    if pop is not None:
        e.upload(pop)
    return e


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def assert_state_equal(a, b, what=""):
    for k in STATE:
        assert same(a[k], b[k]), "%s: %s differs in %d values" % (what, k, (a[k] != b[k]).sum())


def joints(pop):
    """(A, B) global body indices of every joint in table order."""
    body_off = np.asarray(pop.body_off, np.int64)
    nbs = np.diff(body_off)
    c = np.repeat(np.arange(pop.n_creatures), nbs - 1)
    k = np.arange(pop.n_bodies - pop.n_creatures) - (body_off[:-1] - np.arange(pop.n_creatures))[c]
    return body_off[c] + np.asarray(pop.joint_parent, np.int64), body_off[c] + k + 1


def observations_from_state(pop, st):
    """The observations recomputed from read_state: pose, vel and touching_pairs (max_pairs large enough)."""
    A, B = joints(pop)
    ang = st["pose"][:, 2]
    w = st["vel"][:, 2]
    body_off = np.asarray(pop.body_off, np.int64)
    ground = np.zeros(pop.n_bodies, np.int32)
    pairs = st["touching_pairs"][:, :, 0]
    for c in range(pop.n_creatures):
        ground[body_off[c] + np.unique(pairs[c][pairs[c] >= 0])] = 1
    return dict(joint_angle=(ang[B] - ang[A]) - np.float32(0.0), joint_speed=w[B] - w[A],
                root=np.concatenate([st["pose"][body_off[:-1]], st["vel"][body_off[:-1]]], axis=1), ground=ground)


@pytest.mark.parametrize("enc", ["direct", "lsystem", "ce"])
def test_sine_outputs_as_targets_reproduce_plain_stepping(enc):
    pop = population(enc, 64, 40 + len(enc))
    xs, ys = terrain.generate_terrain()
    plain, ctl = engine(OracleEngine, ys, pop), engine(OracleExtEngine, ys, pop)
    T = 150
    sine = ctl.sine_outputs(T)
    for t in range(T):
        plain.step(1)
        ctl.step_targets(sine[t], 1)
        a, b = plain.read_state(max_pairs=16), ctl.read_state(max_pairs=16)
        assert_state_equal(a, b, "%s tick %d" % (enc, t))
        assert same(plain.fitness(), ctl.fitness()) and same(plain.ticks(), ctl.ticks())
    assert (b["ticks"] == T).any() and (b["ticks"] < T).any()          # some lived to the end, some died on the way
    assert plain.counters() == ctl.counters()


def test_the_control_rule():
    pop = population("lsystem", 64, 3)
    xs, ys = terrain.generate_terrain()
    ctl = engine(OracleExtEngine, ys, pop)
    A, B = joints(pop)
    creature = np.repeat(np.arange(pop.n_creatures), np.diff(pop.body_off) - 1)
    rng = np.random.default_rng(0)
    p_gain = ctl.cfg.p_gain
    checked = 0
    for t in range(40):
        before = ctl.read_state()
        target = rng.uniform(-np.pi / 2, np.pi / 2, pop.n_bodies - pop.n_creatures)
        ctl.step_targets(target, 1)
        after = ctl.read_state()
        ang = before["pose"][:, 2]
        angle_before = (ang[B] - ang[A]) - np.float32(0.0)
        want = ((target - angle_before.astype(np.float64)) * p_gain).astype(np.float32)
        live = before["alive"][creature] == 1
        assert same(after["motor_speed"][live], want[live]), "tick %d" % t
        assert same(after["motor_speed"][~live], before["motor_speed"][~live])        # dead creatures are not stepped
        checked += live.sum()
    assert checked > 1000


def test_sine_controllers_are_frozen_during_target_ticks():
    """A plain tick after k target ticks uses the sine output indexed by plain ticks only."""
    pop = population("ce", 48, 5)
    xs, ys = terrain.generate_terrain()
    ctl = engine(OracleExtEngine, ys, pop)
    sine = ctl.sine_outputs(4)
    A, B = joints(pop)
    creature = np.repeat(np.arange(pop.n_creatures), np.diff(pop.body_off) - 1)
    rng = np.random.default_rng(1)
    ctl.step(2)                                          # plain ticks 0 and 1
    for plain_tick, k in ((2, 3), (3, 5)):
        for _ in range(k):
            ctl.step_targets(rng.uniform(-1, 1, pop.n_bodies - pop.n_creatures), 1)
        before = ctl.read_state()
        ctl.step(1)
        after = ctl.read_state()
        ang = before["pose"][:, 2]
        angle_before = (ang[B] - ang[A]) - np.float32(0.0)
        live = before["alive"][creature] == 1
        want = ((sine[plain_tick] - angle_before.astype(np.float64)) * ctl.cfg.p_gain).astype(np.float32)
        assert live.sum() > 100 and same(after["motor_speed"][live], want[live]), "plain tick %d after %d target ticks" % (plain_tick, k)


def test_sine_outputs_follow_plain_ticks_only():
    pop = population("direct", 32, 6)
    xs, ys = terrain.generate_terrain()
    ctl = engine(OracleExtEngine, ys, pop)
    sine = ctl.sine_outputs(6)
    ctl.step(2)
    assert same(ctl.sine_outputs(4), sine[2:6])
    ctl.step_targets(np.zeros(pop.n_bodies - pop.n_creatures), 7)
    assert same(ctl.sine_outputs(4), sine[2:6])
    ctl.step(1)
    assert same(ctl.sine_outputs(3), sine[3:6])


@pytest.mark.parametrize("flat", [True, False])
def test_observations_equal_read_state(flat):
    pop = population("lsystem", 96, 8 + flat)
    xs, ys = terrain.flat_terrain() if flat else terrain.generate_terrain()
    ctl = engine(OracleExtEngine, ys, pop)
    rng = np.random.default_rng(2)
    for t in range(60):
        if t % 3:
            ctl.step_targets(rng.uniform(-np.pi / 2, np.pi / 2, pop.n_bodies - pop.n_creatures), 1 + t % 2)
        else:
            ctl.step(1)
        st = ctl.read_state(max_pairs=64)
        assert (st["n_touching"] <= 64).all()
        ob, ref = ctl.read_observations(), observations_from_state(pop, st)
        for k in OBS:
            assert same(ob[k], ref[k]), "tick %d: %s" % (t, k)
    assert ob["ground"].any() and not ob["ground"].all()


def test_contract():
    pop = population("direct", 16, 3)
    xs, ys = terrain.generate_terrain()
    nj = pop.n_bodies - pop.n_creatures
    ctl = engine(OracleExtEngine, ys)
    lib = ctl.lib
    zeros = np.zeros(nj)
    assert lib.rem2d_step_targets(ctl.h, zeros.ctypes.data, 1) != 0          # no population uploaded
    assert lib.rem2d_read_observations(ctl.h, C.byref(Observation())) != 0
    ctl.upload(pop)
    ctl.step(3)
    ref = ctl.read_state(max_pairs=8)

    def unchanged():
        assert_state_equal(ctl.read_state(max_pairs=8), ref, "after a failed call")

    for bad in (np.nan, np.inf, -np.inf):
        t = np.zeros(nj)
        t[nj // 2] = bad
        with pytest.raises(Rem2dError):
            ctl.step_targets(t, 1)
        unchanged()
    assert lib.rem2d_step_targets(ctl.h, None, 1) != 0                      # NULL targets
    assert lib.rem2d_step_targets(ctl.h, zeros.ctypes.data, -1) != 0        # negative tick count
    unchanged()
    with pytest.raises(ValueError):
        ctl.step_targets(np.zeros(nj + 1), 1)
    ctl.step_targets(zeros, 0)                                              # zero ticks: nothing changes
    unchanged()
    assert lib.rem2d_read_observations(ctl.h, None) != 0
    # NULL members are skipped
    full = ctl.read_observations()
    v = Observation()
    ground = np.full(pop.n_bodies, -7, np.int32)
    v.ground = ground.ctypes.data
    assert lib.rem2d_read_observations(ctl.h, C.byref(v)) == 0
    assert same(ground, full["ground"])
    # consumed by a whole-episode run until the next reset / upload
    for consume in (lambda: ctl.run_episodes(50), lambda: ctl.evaluate(pop, 50)):
        consume()
        with pytest.raises(Rem2dError):
            ctl.step_targets(zeros, 1)
        with pytest.raises(Rem2dError):
            ctl.read_observations()
        ctl.reset()
        ctl.step_targets(zeros, 1)
        ctl.read_observations()
    # the plain oracle does not have the extension
    plain = engine(OracleEngine, ys, pop)
    assert not hasattr(plain.lib, "rem2d_step_targets")
    with pytest.raises(Rem2dError):
        plain.step_targets(zeros, 1)
    with pytest.raises(Rem2dError):
        plain.read_observations()


def test_batched_env_takes_targets_and_observes():
    """BatchedModular2D.step(targets=...) and observe() (here on the oracle with joint targets): numpy and CPU torch inputs,
    an unchanged return value."""
    import torch
    random.seed(11)
    individuals = [Individual.random(encoding="lsystem") for _ in range(12)]
    env = BatchedModular2D(lib_path=oracle_ext.build())
    env.reset(individuals)
    ref = OracleExtEngine()
    ref.set_terrain(env.terrain_y, K.TERRAIN_STEP)
    ref.upload(env.table)
    nj = env.table.n_bodies - env.table.n_creatures
    for t in range(6):
        ob = env.observe()
        target = -0.5 * ob["joint_angle"].astype(np.float64)
        reward, done = env.step(1, targets=torch.from_numpy(target) if t % 2 else target)
        ref.step_targets(target, 1)
        x, wod, alive = ref.read_roots()
        x = x.astype(np.float64)
        assert same(reward, np.where((x < 0) | (wod > x), -100.0, x)) and done.dtype == bool and done.shape == (env.table.n_creatures,)
    for k in OBS:
        assert same(env.observe()[k], ref.read_observations()[k])
    with pytest.raises(ValueError):
        env.step(1, targets=np.zeros(nj - 1))
    env.step(2)                                           # plain ticks still work
    env.close()


# ------------------------------------------------------------------ device code of step_kernel_targets on the CPU

@pytest.fixture(scope="module")
def lsystem_world():
    random.seed(5)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(300)])
    xs, ys = terrain.generate_terrain()
    return pop, ys


@pytest.mark.parametrize("ticks_per_call", [1, 3])
@pytest.mark.parametrize("gs", range(6))
def test_emulated_targets_kernel_equals_the_oracle(lsystem_world, gs, ticks_per_call):
    pop, ys = lsystem_world
    klass = emu.class_of(22)
    nbs = np.diff(pop.body_off)
    creatures = np.nonzero((nbs >= 3) & (nbs <= 22))[0][5 * gs:5 * gs + (32 >> gs)]
    n_calls = 60 // ticks_per_call
    rng = np.random.default_rng(gs * 10 + ticks_per_call)
    nj = pop.n_bodies - pop.n_creatures
    targets = rng.uniform(-np.pi / 2, np.pi / 2, (n_calls, nj))
    r = emu.step(pop, ys, creatures, gs, ticks_per_call, variant="targets", targets=targets, klass=klass)
    sub = pop.select(creatures)
    j0 = np.asarray(pop.body_off[:-1], np.int64) - np.arange(pop.n_creatures)
    jsel = np.concatenate([np.arange(j0[c], j0[c] + nbs[c] - 1) for c in creatures])
    bsel = np.concatenate([np.arange(pop.body_off[c], pop.body_off[c + 1]) for c in creatures])
    o = engine(OracleExtEngine, ys, sub)
    for i in range(n_calls):
        o.step_targets(targets[i, jsel], ticks_per_call)
    st, ob = o.read_state(), o.read_observations()
    what = "G = %d, %d ticks per call" % (1 << gs, ticks_per_call)
    assert same(r["ticks"][creatures], st["ticks"]) and same(r["alive"][creatures], st["alive"]), what
    assert same(r["fitness"][creatures], o.fitness()), what
    for k in ("pose", "vel"):
        assert same(r[k][bsel], st[k]), (what, k)
    for k in ("joint_impulse", "motor_speed"):
        assert same(r[k][jsel], st[k]), (what, k)
    assert same(r["joint_angle"][jsel], ob["joint_angle"]) and same(r["joint_speed"][jsel], ob["joint_speed"]), what
    assert same(r["root"][creatures], ob["root"]) and same(r["ground"][bsel], ob["ground"]), what
    assert r["counters"] == o.counters(), what
