"""Regrouping of a draining episode warp, on the CPU emulation of the device code (tests/emu, its queue entry): once the class
queue is empty, Sim::episodes (rem2d_device.cuh, the loop of the episode kernel) packs the surviving creatures of the warp into
wider lane groups, up to the class's widest group shift. Results must equal the oracle bit for bit, and the work counters must
be those of the creatures' whole episodes, also when a creature overflows its class after a regroup."""
import os
import random
import sys

import numpy as np
import pytest

from gym_rem2d_b200 import Individual, constants as K, terrain
from gym_rem2d_b200.flatten import flatten_population
from oracle.oracle import OracleEngine

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu  # noqa: E402


@pytest.fixture(scope="module")
def world():
    random.seed(5)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(400)])
    xs, ys = terrain.generate_terrain()
    o = OracleEngine(threads=8)
    o.set_terrain(ys, K.TERRAIN_STEP)
    fo, to = o.evaluate(pop, K.EVALUATION_STEPS)
    return pop, ys, fo, to


def oracle_counters(pop, ys, creatures):
    o = OracleEngine(threads=8)
    o.set_terrain(ys, K.TERRAIN_STEP)
    o.evaluate(pop.select(np.sort(creatures)), K.EVALUATION_STEPS)
    return o.counters()


def queue(world, order, gs, klass, max_gs=None):
    pop, ys, _, _ = world
    return emu.queue(pop, ys, order, gs, klass[3] if max_gs is None else max_gs, K.EVALUATION_STEPS, klass[:3])


@pytest.mark.parametrize("gs", [0, 2])
@pytest.mark.parametrize("nb", [8, 12, 22, 44])
def test_draining_warp_widens_to_the_class_cap_and_matches_the_oracle(world, nb, gs):
    pop, ys, fo, to = world
    klass = emu.class_of(nb)
    nbs = np.diff(pop.body_off)
    fit = np.nonzero((nbs >= 3) & (nbs <= nb))[0]
    order = fit[np.argsort(-nbs[fit], kind="stable")][:40]          # the largest creatures of the class first, as the host queues
    r = queue(world, order, gs, klass)
    seq = r["gs_seq"]
    assert seq[0] == gs and seq == sorted(set(seq)), seq
    assert seq[-1] == klass[3], "the last creature runs at the class's widest group shift: %s" % seq
    assert len(seq) >= min(3, klass[3] - gs + 1), "the warp widened fewer times than it could: %s" % seq
    assert (r["finish_gs"][order] > gs).any()
    assert np.array_equal(r["ticks"][order], to[order])
    assert np.array_equal(r["fitness"][order], fo[order])
    assert (r["alive"][order] == 0).all() and (r["status"][order] == 0).all()
    assert r["counters"] == oracle_counters(pop, ys, order)


def test_counters_equal_the_stepping_entry(world):
    """The queue's counters are the sum of what the stepping entry counts for each creature's whole episode."""
    pop, ys, _, to = world
    klass = emu.class_of(22)
    nbs = np.diff(pop.body_off)
    order = np.nonzero((nbs >= 17) & (nbs <= 22))[0][:40]
    r = queue(world, order, 0, klass)
    total = {}
    for first in range(0, len(order), 32):
        se = emu.step(pop, ys, order[first:first + 32], 0, K.EVALUATION_STEPS, klass=klass[:3])
        for k, v in se["counters"].items():
            total[k] = total.get(k, 0) + v
    assert r["counters"] == total


def test_overflow_in_a_widened_group_removes_all_its_work(world):
    """A creature that overflows its contact pool after its warp widened (status != 0: the host re-runs it in the next
    class up) must leave no work in the counters, including the ticks it ran in its narrower group before the regroup."""
    pop, ys, fo, to = world
    nbs = np.diff(pop.body_off)
    order = np.nonzero((nbs >= 17) & (nbs <= 22))[0][:12]     # 12 creatures, 32 lanes: the queue is empty from the start
    klass = (22, 50, 6, 5)                                     # a contact pool small enough to overflow late
    r = queue(world, order, 0, klass)
    over = order[r["status"][order] != 0]
    assert len(over) >= 1
    assert (r["finish_gs"][over] > 0).all(), "the overflow must happen in a widened group"
    assert r["gs_seq"][:2] == [0, 1]
    rest = order[r["status"][order] == 0]
    r2 = queue(world, rest, 0, klass)
    assert r["counters"] == r2["counters"]
    assert r["counters"] == oracle_counters(pop, ys, rest)
    assert np.array_equal(r["ticks"][rest], to[rest]) and np.array_equal(r["fitness"][rest], fo[rest])


def test_one_and_two_body_classes_never_widen(world):
    pop, ys, fo, to = world
    nbs = np.diff(pop.body_off)
    for nb in (1, 2):
        klass = emu.class_of(nb)
        assert klass[3] == 0
        order = np.nonzero(nbs == nb)[0][:40]
        r = queue(world, order, 0, klass)
        assert r["gs_seq"] == [0]
        assert np.array_equal(r["ticks"][order], to[order]) and np.array_equal(r["fitness"][order], fo[order])


def test_a_wider_group_never_needs_more_hot_rows():
    """A warp launched with groups of 2^gs lanes has make_hot_layout(L, gs).rows rows of shared memory; its widened groups
    must fit in them."""
    L = emu.lib()
    for nb, nc, nt, cap in emu.classes():
        rows = [L.rem2d_emu_hot_rows(nb, nc, nt, gs) for gs in range(6)]
        for gs in range(6):
            for wide in range(gs, 6):
                assert rows[wide] <= rows[gs], (nb, gs, wide, rows)
