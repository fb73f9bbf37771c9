"""Episode statistics of whole-episode runs (rem2d_set_stats / rem2d_read_stats, include/rem2d_stats.h) on the CPU: the oracle
with the extension headers (tests/oracle_ext) against the definitions recomputed from a stepping run of the plain oracle, every
end reason, the call contract, and the device code of the statistics images (-DREM2D_STATS, the statistics build of the
emulation in tests/emu) against the oracle, bit for bit."""
import ctypes as C
import os
import random
import sys

import numpy as np
import pytest

from gym_rem2d_b200 import Individual, constants as K, terrain
from gym_rem2d_b200.capi import Rem2dError, END_RUNNING, END_ORIGIN, END_WALL, END_GOAL, END_STEPS
from gym_rem2d_b200.flatten import flatten_population
from oracle.oracle import OracleEngine

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))
sys.path.insert(0, os.path.join(HERE, "oracle_ext"))
import emu  # noqa: E402
from oracle_ext import OracleExtEngine  # noqa: E402

NAMES = ("end_reason", "max_x", "joint_work", "airborne_ticks", "ground_ticks")
ENCODINGS = ("direct", "lsystem", "ce", "cppn")


def population(enc, n, seed):
    random.seed(seed)
    return flatten_population([Individual.random(encoding=enc) for _ in range(n)])


def oracle(ys, stats=True, **cfg):
    o = OracleExtEngine(threads=8, **cfg)
    o.set_terrain(ys, K.TERRAIN_STEP)
    o.set_stats(stats)
    return o


def stats_by_stepping(pop, ys, n_ticks, **cfg):
    """The five statistics from their definitions, recomputed from the state an oracle stepping run reports after every tick."""
    o = OracleEngine(threads=8, **cfg)          # the plain oracle: only what rem2d.h reports
    o.set_terrain(ys, K.TERRAIN_STEP)
    o.upload(pop)
    n, nbod = pop.n_creatures, pop.n_bodies
    body_off = np.asarray(pop.body_off, np.int64)
    nbs = np.diff(body_off)
    j0 = body_off[:-1] - np.arange(n)
    parent = np.asarray(pop.joint_parent, np.int64)
    env_length, steps, terminate = o.cfg.env_length, o.cfg.evaluation_steps, o.cfg.terminate
    end = np.zeros(n, np.int32)
    max_x = np.full(n, -np.inf, np.float32)
    work = np.zeros(n, np.float64)
    airborne = np.zeros(n, np.int32)
    ground = np.zeros(nbod, np.int32)
    ticks = np.zeros(n, np.int32)
    for _ in range(n_ticks):
        o.step(1)
        st = o.read_state(max_pairs=64)
        x, wod, alive = o.read_roots()
        adv = st["ticks"] > ticks
        if not adv.any():
            break
        ticks = st["ticks"].copy()
        assert (st["n_touching"] <= 64).all()
        # end reason: the comparisons of the termination rule, in its precedence, at the tick the creature died
        died = adv & (alive == 0)
        if terminate:
            xd = x.astype(np.float64)
            why = np.where(x < np.float32(0), END_ORIGIN, np.where(wod > xd, END_WALL, np.where(xd > env_length, END_GOAL,
                           np.where(ticks >= steps, END_STEPS, END_RUNNING))))
            end[died] = why[died]
        take = adv & (x > max_x)
        max_x[take] = x[take]
        # joint work: one running double per creature, joints in order (vectorised over creatures, sequential over joints)
        w = st["vel"][:, 2].astype(np.float64)
        mimp = st["joint_impulse"][:, 3].astype(np.float64)
        for k in range(int(nbs.max()) - 1):
            cs = np.nonzero(adv & (nbs - 1 > k))[0]
            j = j0[cs] + k
            term = np.abs(mimp[j] * (w[body_off[cs] + k + 1] - w[body_off[cs] + parent[j]]))
            work[cs] = work[cs] + term
        # ground contact per body, once per tick; airborne: no body touches
        pairs = st["touching_pairs"][:, :, 0]
        for c in np.nonzero(adv)[0]:
            bodies = np.unique(pairs[c][pairs[c] >= 0])
            ground[body_off[c] + bodies] += 1
            if len(bodies) == 0:
                airborne[c] += 1
    return dict(end_reason=end, max_x=max_x, joint_work=work, airborne_ticks=airborne, ground_ticks=ground), ticks


def assert_stats_equal(a, b, what=""):
    for k in NAMES:
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, (what, k)
        assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), "%s: %s differs in %d values" % (
            what, k, (a[k] != b[k]).sum())


@pytest.mark.parametrize("flat", [True, False])
@pytest.mark.parametrize("enc", ENCODINGS)
def test_oracle_equals_the_definitions(enc, flat):
    pop = population(enc, 48, 100 + ENCODINGS.index(enc) * 2 + flat)
    xs, ys = terrain.flat_terrain() if flat else terrain.generate_terrain()
    n_ticks = 400
    ref, ticks = stats_by_stepping(pop, ys, n_ticks)
    o = oracle(ys)
    fo, to = o.evaluate(pop, n_ticks)
    assert np.array_equal(to, ticks)
    assert_stats_equal(o.read_stats(), ref, "%s flat=%s" % (enc, flat))
    assert (ref["joint_work"] > 0).any() and (ref["ground_ticks"] > 0).any()


def _reasons(ys, max_ticks, **cfg):
    pop = population("lsystem", 96, 7)
    o = oracle(ys, **cfg)
    f, t = o.evaluate(pop, max_ticks)
    return pop, o, f, t, o.read_stats()


def test_every_end_reason_occurs_and_agrees_with_fitness_and_ticks():
    xs, ys = terrain.generate_terrain()
    # default rule: random creatures are caught by the wall of death
    pop, o, f, t, s = _reasons(ys, K.EVALUATION_STEPS)
    r = s["end_reason"]
    assert (r == END_WALL).any(), np.bincount(r)
    assert not (r == END_RUNNING).any()
    assert (t[r != END_STEPS] < K.EVALUATION_STEPS).all()
    # a slope down to the left and no wall: they slide back past the origin (root x < 0, which the wall rule would catch too)
    xs = np.arange(200) * K.TERRAIN_STEP
    slope = K.TERRAIN_HEIGHT + 0.6 * (xs - K.TERRAIN_STEP * K.TERRAIN_STARTPAD / 2)
    pop, o, f, t, s = _reasons(slope, K.EVALUATION_STEPS, wod_speed=0.0, evaluation_steps=600)
    r = s["end_reason"]
    assert (r == END_ORIGIN).any(), np.bincount(r)
    assert (s["max_x"][r == END_ORIGIN] > 0).all() and (t[r == END_ORIGIN] < 600).all()
    # a short course: some reach the goal, with the bonus in their fitness
    pop, o, f, t, s = _reasons(ys, K.EVALUATION_STEPS, env_length=3.0)
    r = s["end_reason"]
    assert (r == END_GOAL).any(), np.bincount(r)
    assert (f[r == END_GOAL] > 3.0).all() and (f[r != END_GOAL] <= 3.0).all()
    assert (s["max_x"][r == END_GOAL] > 3.0).all()
    # a short episode: the step limit ends it
    pop, o, f, t, s = _reasons(ys, K.EVALUATION_STEPS, evaluation_steps=40)
    r = s["end_reason"]
    assert (r == END_STEPS).any(), np.bincount(r)
    assert (t[r == END_STEPS] == 40).all() and (t[r != END_STEPS] < 40).all()
    # the run stops before the episodes end
    pop, o, f, t, s = _reasons(ys, 60)
    r = s["end_reason"]
    assert (r == END_RUNNING).any(), np.bincount(r)
    assert (t[r == END_RUNNING] == 60).all() and (t[r != END_RUNNING] < 60).all()
    # no termination rule: everything is still running at the horizon
    pop, o, f, t, s = _reasons(ys, 120, terminate=0)
    assert (s["end_reason"] == END_RUNNING).all() and (t == 120).all()
    # the ticks a creature ran are split into airborne ticks and ticks with a body on the ground
    nbs = np.diff(pop.body_off)
    per_creature = np.add.reduceat(s["ground_ticks"], pop.body_off[:-1])
    assert (s["airborne_ticks"] <= t).all() and (per_creature <= t * nbs).all()


def test_statistics_never_change_results():
    """The oracle with statistics, recording or not, computes what the plain oracle computes."""
    pop = population("ce", 64, 9)
    xs, ys = terrain.generate_terrain()
    plain = OracleEngine(threads=8)
    plain.set_terrain(ys, K.TERRAIN_STEP)
    f, t = plain.evaluate(pop, K.EVALUATION_STEPS)
    out = [(f, t, plain.counters())]
    for on in (False, True, False):
        o = oracle(ys, stats=on)
        f, t = o.evaluate(pop, K.EVALUATION_STEPS)
        out.append((f, t, o.counters()))
    for f, t, c in out[1:]:
        assert np.array_equal(f, out[0][0]) and np.array_equal(t, out[0][1]) and c == out[0][2]


def test_plain_oracle_has_no_statistics():
    o = OracleEngine()
    assert not hasattr(o.lib, "rem2d_read_stats")
    with pytest.raises(Rem2dError):
        o.set_stats(True)


def check_contract(o, pop):
    """The call contract of the statistics on engine `o`, terrain set, statistics off and nothing uploaded: the oracle's here,
    the CUDA library's in tests/test_episode_stats_gpu.py."""
    with pytest.raises(Rem2dError):
        o.read_stats()                          # no population
    o.upload(pop)
    with pytest.raises(Rem2dError):
        o.read_stats()                          # no run since the upload
    o.evaluate(pop, 200)
    with pytest.raises(Rem2dError):
        o.read_stats()                          # uploaded with statistics off
    o.set_stats(True)
    o.run_episodes(200)
    with pytest.raises(Rem2dError):
        o.read_stats()                          # the flag applies from the next upload on
    o.evaluate(pop, 200)
    full = o.read_stats()
    # NULL pointers are skipped
    from gym_rem2d_b200.capi import EpisodeStats
    jw = np.full(pop.n_creatures, -1.0)
    v = EpisodeStats()
    v.joint_work = jw.ctypes.data
    assert o.lib.rem2d_read_stats(o.h, C.byref(v)) == 0
    assert np.array_equal(jw, full["joint_work"])
    o.run_episodes(200)
    assert_stats_equal(o.read_stats(), full, "re-run")
    # the run consumed the per-creature state: stepping is refused and leaves the statistics readable
    with pytest.raises(Rem2dError):
        o.step(1)
    with pytest.raises(Rem2dError):
        o.step_targets(np.zeros(pop.n_bodies - pop.n_creatures), 1)
    assert_stats_equal(o.read_stats(), full, "after a refused step")
    o.reset()
    o.step(1)
    with pytest.raises(Rem2dError):
        o.read_stats()                          # the stepping path records none
    o.run_episodes(200)
    o.read_stats()
    o.reset()
    with pytest.raises(Rem2dError):
        o.read_stats()
    o.upload(pop)
    with pytest.raises(Rem2dError):
        o.read_stats()


def test_contract():
    xs, ys = terrain.generate_terrain()
    check_contract(oracle(ys, stats=False), population("direct", 16, 3))


# ------------------------------------------------------------------ device code of the statistics images on the CPU

def subset(stats, pop, creatures):
    """The statistics of `creatures` only (ground_ticks of their bodies)."""
    bodies = np.concatenate([np.arange(pop.body_off[c], pop.body_off[c + 1]) for c in creatures])
    return {k: (v[bodies] if k == "ground_ticks" else v[creatures]) for k, v in stats.items() if k in NAMES}


@pytest.fixture(scope="module")
def world():
    random.seed(5)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(400)])
    xs, ys = terrain.generate_terrain()
    o = oracle(ys)
    fo, to = o.evaluate(pop, K.EVALUATION_STEPS)
    return pop, ys, fo, to, o.read_stats()


@pytest.mark.parametrize("gs", range(6))
def test_emulated_stepping_entry_equals_the_oracle(world, gs):
    pop, ys, fo, to, so = world
    klass = emu.class_of(22)
    nbs = np.diff(pop.body_off)
    creatures = np.nonzero((nbs >= 3) & (nbs <= 22))[0][7 * gs:7 * gs + (32 >> gs)]
    n_ticks = 300
    r = emu.step(pop, ys, creatures, gs, n_ticks, variant="stats", klass=klass)
    o = oracle(ys)
    fc, tc = o.evaluate(pop.select(creatures), n_ticks)
    assert np.array_equal(r["ticks"][creatures], tc) and np.array_equal(r["fitness"][creatures], fc)
    assert_stats_equal(subset(r, pop, creatures), o.read_stats(), "G = %d" % (1 << gs))


@pytest.mark.parametrize("nb", [8, 12, 22, 44])
def test_emulated_queue_with_regrouping_equals_the_oracle(world, nb):
    pop, ys, fo, to, so = world
    klass = emu.class_of(nb)
    nbs = np.diff(pop.body_off)
    fit = np.nonzero((nbs >= 3) & (nbs <= nb))[0]
    order = fit[np.argsort(-nbs[fit], kind="stable")][:40]          # the largest creatures of the class first, as the host queues
    r = emu.queue(pop, ys, order, 0, klass[3], K.EVALUATION_STEPS, klass, variant="stats")
    assert np.array_equal(r["ticks"][order], to[order]) and np.array_equal(r["fitness"][order], fo[order])
    assert_stats_equal(subset(r, pop, order), subset(so, pop, order), "NB %d" % nb)
