"""The device code of the CUDA kernels, executed on the CPU (tests/emu: one host thread per lane, barriers for
__syncwarp/__shfl_sync), against the oracle — bit for bit, for every group size the kernels are launched with.

This is how the lane-group logic of gym_rem2d_b200/csrc/rem2d_device.cuh (static modulo schedule of the velocity
sweeps, strided per-body/joint/contact loops, leader sections, group barriers) is checked in a container without a
GPU; the `-m gpu` tests then check the same code as compiled by nvcc, plus the queue / park / tail logic of the kernels.
"""
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

INT_KEYS = ("alive", "ticks", "limit_state", "n_contacts", "n_touching", "touching_pairs")
FLT_KEYS = ("pose", "vel", "joint_impulse", "motor_speed", "touching_impulse", "wod")


def oracle_state(sub, ys, step, n_ticks, **cfg):
    o = OracleEngine(threads=4, **cfg)
    o.set_terrain(ys, step)
    o.upload(sub)
    o.step(n_ticks)
    return o.read_state(max_pairs=24), o.counters(), o.fitness()


def check(sub, ys, gs, n_ticks, step=K.TERRAIN_STEP, **cfg):
    so, co, fo = oracle_state(sub, ys, step, n_ticks, **cfg)
    per = 32 >> gs
    out, total = [], dict.fromkeys(co, 0)
    for first in range(0, sub.n_creatures, per):          # one emulated warp per `per` creatures
        idx = np.arange(first, min(first + per, sub.n_creatures))
        se = emu.step(sub, ys, idx, gs, n_ticks, terrain_step=step, **cfg)
        b0, b1 = sub.body_off[idx[0]], sub.body_off[idx[-1] + 1]
        j0, j1 = b0 - idx[0], b1 - idx[-1] - 1
        sl = {"pose": slice(b0, b1), "vel": slice(b0, b1), "joint_impulse": slice(j0, j1), "limit_state": slice(j0, j1),
              "motor_speed": slice(j0, j1)}
        for k in INT_KEYS + FLT_KEYS:
            s = sl.get(k, slice(idx[0], idx[-1] + 1))
            assert np.array_equal(se[k][s], so[k][s]), "gs=%d creatures %s: %s differs" % (gs, idx, k)
        assert np.array_equal(se["fitness"][idx], fo[idx])
        out.append(se["sched_P"][idx])
        total = {k: v + se["counters"][k] for k, v in total.items()}
    assert total == co
    return out


@pytest.fixture(scope="module")
def lsystem_pop():
    random.seed(12)
    return flatten_population([Individual.random(encoding="lsystem") for _ in range(64)])


@pytest.mark.parametrize("gs", [0, 1, 2, 3, 4, 5])
def test_every_group_size_matches_the_oracle_on_large_creatures(lsystem_pop, gs):
    nbs = np.diff(lsystem_pop.body_off)
    big = np.sort(np.argsort(-nbs, kind="stable")[:max(2, 32 >> gs)])
    sub = lsystem_pop.select(big)
    xs, ys = terrain.generate_terrain()
    out = check(sub, ys, gs, 45)
    if gs >= 2:
        # the schedule really pipelines: period well below the number of constraints of a 17-21 body creature
        assert max(int(p.max()) for p in out) <= 8
        assert min(int(p.min()) for p in out) >= 3


@pytest.mark.parametrize("gs", [1, 2, 3])
def test_mixed_sizes_in_one_warp_full_episode_lengths(lsystem_pop, gs):
    """Groups of one warp hold creatures of different sizes (different periods, skews and lifetimes: groups finish their
    sweeps at different passes and die at different ticks)."""
    idx = np.arange(0, 32 >> gs) * 2 + 5
    sub = lsystem_pop.select(idx)
    xs, ys = terrain.generate_terrain()
    check(sub, ys, gs, 140)


@pytest.mark.parametrize("enc,gs", [("direct", 2), ("ce", 1), ("cppn", 2)])
def test_other_encodings_flat_and_rough(enc, gs):
    random.seed(3)
    pop = flatten_population([Individual.random(encoding=enc) for _ in range(24)])
    xs, ys = terrain.flat_terrain() if enc == "direct" else terrain.generate_terrain()
    check(pop.select(np.arange(16)), ys, gs, 70)


@pytest.mark.parametrize("gs", [2, 5])
def test_inclined_terrain_no_sleep_fixed_horizon(lsystem_pop, gs):
    nbs = np.diff(lsystem_pop.body_off)
    sub = lsystem_pop.select(np.sort(np.argsort(-nbs, kind="stable")[:8 if gs == 2 else 2]))
    xs = np.arange(200) * K.TERRAIN_STEP
    ys = K.TERRAIN_HEIGHT - 0.6 * (xs - K.TERRAIN_STEP * K.TERRAIN_STARTPAD / 2)
    check(sub, ys, gs, 60, terminate=0, allow_sleep=0)


def test_spilled_hot_contacts_fall_back_to_the_sequential_sweep():
    """More touching contacts than the class stages in shared memory (forced here with a class that stages ONE): the extra
    ones spill to the cold block, the tick's sweeps are not scheduled and the group leader runs them sequentially."""
    random.seed(41)
    pop = flatten_population([Individual.random(encoding="direct") for _ in range(16)])
    ys = np.full(200, 5.0)
    nbs = np.diff(pop.body_off)
    ok = np.nonzero(nbs >= 3)[0][:4]
    so, _, _ = oracle_state(pop.select(ok), ys, 0.15, 50)
    se = emu.step(pop.select(ok), ys, np.arange(len(ok)), 2, 50, klass=(12, 64, 1), terrain_step=0.15)
    for k in INT_KEYS + FLT_KEYS:
        assert np.array_equal(se[k], so[k]), k
    assert so["n_touching"].max() > 1
