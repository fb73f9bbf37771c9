"""Per-joint feedback policies (rem2d_set_policy, include/rem2d_policy.h) on the CPU: the oracle with the extension headers and
the policy (tests/oracle_policy) against a host loop built from independent pieces (read_observations, the sine outputs, the numpy network of
gym_rem2d_b200.policy and rem2d_step_targets), zero weights against open loop, the call contract, the Python layer, and the
device code of the policy images (-DREM2D_POLICY, the emulation in tests/emu_policy) against the oracle, bit for bit."""
import os
import random
import sys

import numpy as np
import pytest

from gym_rem2d_b200 import Individual, constants as K, policy, terrain
from gym_rem2d_b200.capi import Rem2dError
from gym_rem2d_b200.env import BatchedModular2D, evaluate_population
from gym_rem2d_b200.flatten import flatten_population
from oracle.oracle import OracleEngine

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu_policy"))
sys.path.insert(0, os.path.join(HERE, "oracle_policy"))
import emu_policy  # noqa: E402
import oracle_policy  # noqa: E402
from oracle_policy import OraclePolicyEngine  # noqa: E402

STATE = ("pose", "vel", "joint_impulse", "limit_state", "motor_speed", "alive", "ticks", "awake", "wod", "n_contacts",
         "n_touching", "touching_pairs", "touching_impulse")
NAMES = ("end_reason", "max_x", "joint_work", "airborne_ticks", "ground_ticks")
END_RUNNING, END_ORIGIN, END_WALL, END_GOAL, END_STEPS = 0, 1, 2, 3, 4


def population(enc, n, seed):
    random.seed(seed)
    return flatten_population([Individual.random(encoding=enc) for _ in range(n)])


def n_joints(pop):
    return pop.n_bodies - pop.n_creatures


def engine(ys, pop=None, weights=None, stats=False, cls=OraclePolicyEngine, **cfg):
    e = cls(threads=8, **cfg)
    e.set_terrain(ys, K.TERRAIN_STEP)
    if stats:
        e.set_stats(True)
    if weights is not None:
        e.set_policy(weights)
    if pop is not None:
        e.upload(pop)
    return e


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def assert_state_equal(a, b, what=""):
    for k in STATE:
        assert same(a[k], b[k]), "%s: %s differs in %d values" % (what, k, (a[k] != b[k]).sum())


def assert_stats_equal(a, b, what=""):
    for k in NAMES:
        assert same(a[k], b[k]), "%s: %s differs in %d values" % (what, k, (a[k] != b[k]).sum())


def host_loop(pop, ys, weights, n_ticks, on_tick=None):
    """The policy by hand, on the oracle with joint targets and no policy: every tick reads the observations, takes the sine
    outputs of rem2d_control_sine_outputs (target ticks do not advance the oscillators, so tick t uses output t), evaluates
    gym_rem2d_b200.policy.forward in numpy and steps one tick with rem2d_step_targets(s + u). The episode statistics are
    recomputed from their definitions (include/rem2d_stats.h) from the state after every tick. Returns the engine and the
    statistics."""
    o = engine(ys, pop)
    sine = o.sine_outputs(n_ticks)
    n, body_off = pop.n_creatures, np.asarray(pop.body_off, np.int64)
    nbs, j0, parent = np.diff(body_off), body_off[:-1] - np.arange(n), np.asarray(pop.joint_parent, np.int64)
    st = dict(end_reason=np.zeros(n, np.int32), max_x=np.full(n, -np.inf, np.float32), joint_work=np.zeros(n, np.float64),
              airborne_ticks=np.zeros(n, np.int32), ground_ticks=np.zeros(pop.n_bodies, np.int32))
    ticks = np.zeros(n, np.int32)
    for t in range(n_ticks):
        u = policy.forward(weights, policy.features(o.read_observations(), sine[t], pop))
        o.step_targets(sine[t] + u, 1)
        s = o.read_state(max_pairs=64)
        if on_tick:
            on_tick(t, s)
        x, wod, alive = o.read_roots()
        adv = s["ticks"] > ticks
        if not adv.any():
            break
        ticks = s["ticks"].copy()
        assert (s["n_touching"] <= 64).all()
        xd, died = x.astype(np.float64), adv & (alive == 0)
        why = np.where(x < np.float32(0), END_ORIGIN, np.where(wod > xd, END_WALL, np.where(xd > o.cfg.env_length, END_GOAL,
                       np.where(ticks >= o.cfg.evaluation_steps, END_STEPS, END_RUNNING))))
        st["end_reason"][died] = why[died]
        take = adv & (x > st["max_x"])
        st["max_x"][take] = x[take]
        w, mimp = s["vel"][:, 2].astype(np.float64), s["joint_impulse"][:, 3].astype(np.float64)
        for k in range(int(nbs.max()) - 1):
            cs = np.nonzero(adv & (nbs - 1 > k))[0]
            j = j0[cs] + k
            st["joint_work"][cs] = st["joint_work"][cs] + np.abs(mimp[j] * (w[body_off[cs] + k + 1] - w[body_off[cs] + parent[j]]))
        pairs = s["touching_pairs"][:, :, 0]
        for c in np.nonzero(adv)[0]:
            bodies = np.unique(pairs[c][pairs[c] >= 0])
            st["ground_ticks"][body_off[c] + bodies] += 1
            st["airborne_ticks"][c] += len(bodies) == 0
    return o, st


# (encoding, hidden units, weight scale): every encoding, every H of {1, 8, 16} and every scale of {0.1, 1, 10} (10 saturates)
CASES = [("direct", 1, 0.1), ("lsystem", 8, 1.0), ("ce", 16, 10.0), ("direct", 16, 1.0), ("lsystem", 1, 10.0), ("ce", 8, 0.1)]


@pytest.mark.parametrize("enc,H,scale", CASES)
def test_host_loop_reproduces_policy_stepping_and_episodes(enc, H, scale):
    pop = population(enc, 40, 200 + H)
    xs, ys = terrain.generate_terrain()
    W = policy.random_weights(n_joints(pop), H, scale, rng=H)
    T = 300
    # stepping: rem2d_step of a population uploaded with the policy, tick by tick
    stepped = engine(ys, pop, W)

    def compare(t, s):
        stepped.step(1)
        assert_state_equal(stepped.read_state(max_pairs=64), s, "%s H %d scale %g tick %d" % (enc, H, scale, t))

    ref, st = host_loop(pop, ys, W, T, compare)
    assert stepped.counters() == ref.counters()
    # whole episodes of T ticks, with statistics
    o = engine(ys, weights=W, stats=True)
    f, t = o.evaluate(pop, T)
    assert same(f, ref.fitness()) and same(t, ref.ticks())
    assert (t < T).any() and t.max() > 100
    assert_stats_equal(o.read_stats(), st, "%s H %d scale %g" % (enc, H, scale))
    # the policy changes the motion
    f0, t0 = engine(ys).evaluate(pop, T)
    assert not same(f, f0)


def no_negative_zero_sine(o, pop, T):
    """The sine outputs of the first T ticks: s + (+0.0) would turn an output of exactly -0.0 into +0.0."""
    s = o.sine_outputs(T)
    return not (np.signbit(s) & (s == 0.0)).any()


@pytest.mark.parametrize("enc", ["direct", "lsystem", "ce"])
def test_zero_feedback_reproduces_open_loop(enc):
    pop = population(enc, 64, 300 + len(enc))
    xs, ys = terrain.generate_terrain()
    plain = engine(ys, stats=True)
    fp, tp = plain.evaluate(pop, K.EVALUATION_STEPS)
    sp, cp = plain.read_stats(), plain.counters()
    plain.reset()
    assert no_negative_zero_sine(plain, pop, int(tp.max()))
    nj = n_joints(pop)
    zero = np.zeros((nj, policy.n_params(8)))
    input_only = policy.random_weights(nj, 8, 1.0, rng=4)
    input_only[:, 9 * 8:] = 0.0                                   # w2 = b2 = 0: the hidden layer is computed and ignored
    for W in (zero, input_only):
        o = engine(ys, weights=W, stats=True)
        f, t = o.evaluate(pop, K.EVALUATION_STEPS)
        assert same(f, fp) and same(t, tp) and o.counters() == cp
        assert_stats_equal(o.read_stats(), sp, enc)


def check_contract(make, ys, pop):
    """The call contract of include/rem2d_policy.h on the engine that make() creates (with the terrain set)."""
    nj = n_joints(pop)
    A = policy.random_weights(nj, 4, 1.0, rng=1)
    B = policy.random_weights(nj, 2, 1.0, rng=2)

    def run(e, n=40):
        e.upload(pop)
        e.step(n)
        return e.read_state(max_pairs=16)

    ref_a, ref_b, ref_plain = run(make_with(make, A)), run(make_with(make, B)), run(make())
    assert not same(ref_a["pose"], ref_plain["pose"]) and not same(ref_a["pose"], ref_b["pose"])
    # rejected calls keep the previous policy
    e = make_with(make, A)
    lib = e.lib
    for bad in (0, 17, -1):
        assert lib.rem2d_set_policy(e.h, B.ctypes.data, nj, bad) != 0
    assert lib.rem2d_set_policy(e.h, B.ctypes.data, -1, 2) != 0
    for v in (np.nan, np.inf, -np.inf):
        bad = B.copy()
        bad[nj // 2, 3] = v
        with pytest.raises(Rem2dError):
            e.set_policy(bad)
    assert_state_equal(run(e), ref_a, "after rejected set_policy calls")
    # the upload takes a snapshot: a later set_policy changes nothing of the current population, not even after a reset
    e.upload(pop)
    e.set_policy(B)
    e.step(40)
    assert_state_equal(e.read_state(max_pairs=16), ref_a, "set_policy after the upload")
    e.reset()                                                   # the reset keeps the uploaded policy
    e.step(40)
    assert_state_equal(e.read_state(max_pairs=16), ref_a, "after a reset")
    assert_state_equal(run(e), ref_b, "the next upload takes the new policy")
    # a joint-count mismatch at upload changes nothing
    e.reset()
    e.step(10)
    before = e.read_state(max_pairs=16)
    other = population("direct", 5, 9)
    assert n_joints(other) != nj
    with pytest.raises(Rem2dError):
        e.upload(other)
    assert_state_equal(e.read_state(max_pairs=16), before, "after a refused upload")
    e.step(30)
    assert_state_equal(e.read_state(max_pairs=16), ref_b, "stepping on after a refused upload")
    # clearing: open loop again
    e.set_policy(None)
    assert_state_equal(run(e), ref_plain, "after clearing the policy")
    # step_targets overrides the policy: the policy is not evaluated
    targets = np.random.default_rng(3).uniform(-1, 1, nj)
    runs = []
    for w in (A, None):
        t = make_with(make, w)
        t.upload(pop)
        t.step_targets(targets, 9)
        runs.append(t.read_state(max_pairs=16))
    assert_state_equal(runs[0], runs[1], "step_targets with a policy")
    # statistics compose with the policy; without statistics read_stats is refused after a policy run
    s = make_with(make, A)
    s.set_stats(True)
    s.evaluate(pop, 200)
    assert s.read_stats()["ground_ticks"].shape == (pop.n_bodies,)
    s.set_stats(False)
    s.evaluate(pop, 200)
    with pytest.raises(Rem2dError):
        s.read_stats()
    for bad_shape in (np.zeros((nj, 12)), np.zeros(nj * 11), np.zeros((nj, 171))):
        with pytest.raises(ValueError):
            s.set_policy(bad_shape)


def make_with(make, weights):
    e = make()
    if weights is not None:
        e.set_policy(weights)
    return e


def test_contract():
    xs, ys = terrain.generate_terrain()
    check_contract(lambda: engine(ys), ys, population("direct", 16, 3))
    # the plain oracle does not have the extension
    plain = engine(ys, cls=OracleEngine)
    assert not hasattr(plain.lib, "rem2d_set_policy")
    with pytest.raises(Rem2dError):
        plain.set_policy(None)


def test_step_targets_ignore_the_policy():
    """rem2d_step_targets on a population uploaded with a policy is rem2d_step_targets without one; the oscillators are frozen,
    so the plain ticks around it are policy ticks on the same sine outputs."""
    pop = population("lsystem", 24, 12)
    xs, ys = terrain.generate_terrain()
    nj = n_joints(pop)
    W = policy.random_weights(nj, 3, 1.0, rng=6)
    targets = np.random.default_rng(7).uniform(-1, 1, nj)
    a, b = engine(ys, pop, W), engine(ys, pop)
    a.step_targets(targets, 9)
    b.step_targets(targets, 9)
    assert_state_equal(a.read_state(max_pairs=16), b.read_state(max_pairs=16), "step_targets")
    # then a policy tick uses sine output 0 (no plain tick has run)
    sine = a.sine_outputs(1)[0]
    u = policy.forward(W, policy.features(a.read_observations(), sine, pop))
    a.step(1)
    b.step_targets(sine + u, 1)
    assert_state_equal(a.read_state(max_pairs=16), b.read_state(max_pairs=16), "policy tick after step_targets")


def test_policy_module():
    assert policy.n_params(1) == 11 and policy.n_params(16) == 161
    assert [policy.hidden_size(10 * h + 1) for h in (1, 8, 16)] == [1, 8, 16]
    for P in (0, 10, 12, 171, 1):
        with pytest.raises(ValueError):
            policy.hidden_size(P)
    with pytest.raises(ValueError):
        policy.n_params(17)
    W = policy.random_weights(5, 3, 2.0, rng=0)
    assert W.shape == (5, 31) and W.dtype == np.float64
    x = np.random.default_rng(1).normal(size=(5, 8))
    # the definition, one joint at a time in plain Python floats
    for j in range(5):
        u = W[j, 30]
        for k in range(3):
            acc = W[j, 24 + k]
            for i in range(8):
                acc = acc + W[j, 8 * k + i] * x[j, i]
            u = u + W[j, 27 + k] * (acc / (1.0 + abs(acc)))
        assert policy.forward(W, x)[j] == u
    # features: the columns of the observations
    pop = population("lsystem", 6, 2)
    xs, ys = terrain.generate_terrain()
    o = engine(ys, pop)
    o.step(30)
    ob = o.read_observations()
    s = o.sine_outputs(1)[0]
    f = policy.features(ob, s, pop)
    assert f.shape == (n_joints(pop), 8) and f.dtype == np.float64
    assert same(f[:, 0].copy(), s) and same(f[:, 1].copy(), ob["joint_angle"].astype(np.float64))


def test_python_layer():
    """Engine.set_policy (numpy and CPU tensors, H inferred), BatchedModular2D.reset / evaluate (policy per call, none = open
    loop) and evaluate_population(policy=...), here on the oracle with the extension headers."""
    import torch
    random.seed(21)
    inds = [Individual.random(encoding="lsystem") for _ in range(12)]
    env = BatchedModular2D(lib_path=oracle_policy.build())
    open_loop = env.evaluate(inds, steps=300)
    nj = env.table.n_bodies - env.table.n_creatures
    W = policy.random_weights(nj, 5, 1.0, rng=8)
    ref = engine(env.terrain_y, weights=W)
    f_ref, _ = ref.evaluate(env.table, 300)
    assert same(env.evaluate(inds, steps=300, policy=W), f_ref)
    assert same(env.evaluate(inds, steps=300, policy=torch.from_numpy(W)), f_ref)
    assert same(env.evaluate(inds, steps=300), open_loop)                 # left out: open loop again
    fit = evaluate_population(inds, EVALUATION_STEPS=300, env=env, as_torch=False, policy=W)
    assert same(fit, f_ref)
    env.reset(inds, policy=W)
    env.step(20)
    ref.upload(env.table)
    ref.step(20)
    assert_state_equal(env.engine.read_state(max_pairs=16), ref.read_state(max_pairs=16), "BatchedModular2D.reset(policy=...)")
    env.reset(inds)
    env.step(20)
    plain = engine(env.terrain_y, env.table)
    plain.step(20)
    assert_state_equal(env.engine.read_state(max_pairs=16), plain.read_state(max_pairs=16), "BatchedModular2D.reset() after a policy")
    with pytest.raises(ValueError):
        env.evaluate(inds, steps=10, policy=np.zeros((nj, 20)))
    with pytest.raises(Rem2dError):
        env.evaluate(inds, steps=10, policy=np.zeros((nj + 1, 11)))
    env.close()


# ------------------------------------------------------------------ device code of the policy images on the CPU

@pytest.fixture(scope="module")
def world():
    random.seed(5)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(400)])
    xs, ys = terrain.generate_terrain()
    W = policy.random_weights(n_joints(pop), 6, 1.0, rng=11)
    o = engine(ys, weights=W, stats=True)
    fo, to = o.evaluate(pop, K.EVALUATION_STEPS)
    return pop, ys, W, fo, to, o.read_stats()


def subset(stats, pop, creatures):
    bodies = np.concatenate([np.arange(pop.body_off[c], pop.body_off[c + 1]) for c in creatures])
    return {k: (v[bodies] if k == "ground_ticks" else v[creatures]) for k, v in stats.items() if k in NAMES}


def sub_weights(W, pop, creatures):
    j0 = np.asarray(pop.body_off[:-1], np.int64) - np.arange(pop.n_creatures)
    nbs = np.diff(pop.body_off)
    return W[np.concatenate([np.arange(j0[c], j0[c] + nbs[c] - 1) for c in creatures])]


@pytest.mark.parametrize("gs", range(6))
def test_emulated_policy_stepping_equals_the_oracle(world, gs):
    pop, ys, W, fo, to, so = world
    klass = emu_policy.class_of(22)
    nbs = np.diff(pop.body_off)
    creatures = np.nonzero((nbs >= 3) & (nbs <= 22))[0][7 * gs:7 * gs + (32 >> gs)]
    n_ticks = 300
    r = emu_policy.step(pop, ys, creatures, gs, n_ticks, W, klass=klass)
    sub = pop.select(creatures)
    o = engine(ys, sub, sub_weights(W, pop, creatures))
    o.step(n_ticks)
    st = o.read_state()
    bsel = np.concatenate([np.arange(pop.body_off[c], pop.body_off[c + 1]) for c in creatures])
    what = "G = %d" % (1 << gs)
    assert same(r["ticks"][creatures], st["ticks"]) and same(r["fitness"][creatures], o.fitness()), what
    assert same(r["pose"][bsel], st["pose"]) and same(r["vel"][bsel], st["vel"]), what
    assert r["counters"] == o.counters(), what


@pytest.mark.parametrize("nb", [8, 12, 22, 44])
def test_emulated_policy_queue_with_regrouping_equals_the_oracle(world, nb):
    pop, ys, W, fo, to, so = world
    klass = emu_policy.class_of(nb)
    nbs = np.diff(pop.body_off)
    fit = np.nonzero((nbs >= 3) & (nbs <= nb))[0]
    order = fit[np.argsort(-nbs[fit], kind="stable")][:40]
    r = emu_policy.queue(pop, ys, order, 0, klass[3], K.EVALUATION_STEPS, klass, W)
    assert len(r["gs_seq"]) > 1                                    # the warp regrouped
    assert same(r["ticks"][order], to[order]) and same(r["fitness"][order], fo[order])
    assert_stats_equal(subset(r, pop, order), subset(so, pop, order), "NB %d" % nb)


def test_emulation_refuses_bad_hidden_sizes(world):
    pop, ys, W, fo, to, so = world
    klass = emu_policy.class_of(22)
    for bad in (np.zeros((n_joints(pop), 1)), np.zeros((n_joints(pop), 171))):    # H = 0 and H = 17
        with pytest.raises(RuntimeError):
            emu_policy.step(pop, ys, [0], 0, 1, bad, klass=klass)
