"""Regrouping of draining episode warps on the GPU: once its class queue is empty, a queue-mode warp packs its surviving
creatures into wider lane groups (Sim::episodes, rem2d_device.cuh), and so does a tail launch narrower than a warp per
creature. Results must stay bit-identical to the oracle, and the work counters must not depend on how the warps were
laid out. Needs a GPU; tests/test_regroup.py checks the same code on the CPU emulation."""
import numpy as np
import pytest

from gym_rem2d_b200 import constants as K, terrain
from gym_rem2d_b200.capi import Engine
from gym_rem2d_b200.population import random_population
from oracle.oracle import OracleEngine

pytestmark = pytest.mark.gpu


def _oracle_eval(pop, ys):
    o = OracleEngine(threads=max(8, (__import__("os").cpu_count() or 8)))
    o.set_terrain(ys, K.TERRAIN_STEP)
    fo, to = o.evaluate(pop, K.EVALUATION_STEPS)
    return fo, to, o.counters()


def _gpu_eval(pop, ys, **options):
    g = Engine(device=0)
    g.set_terrain(ys, K.TERRAIN_STEP)
    for k, v in options.items():
        g.set_option(k, v)
    fg, tg = g.evaluate(pop, K.EVALUATION_STEPS)
    out = fg, tg, g.counters()
    g.close()
    return out


@pytest.mark.parametrize("options", [
    dict(warp_mode_max=0, park_ticks=0, smem_budget_kb=24),                                    # several rounds, no parking
    dict(warp_mode_max=0, park_ticks=0, smem_budget_kb=40, group_shift=0),                     # every class starts at G = 1
    dict(warp_mode_max=0, park_ticks=140, park_cap=0.0625, tail_group_shift=1, smem_budget_kb=24),   # narrow tail launches
])
def test_draining_warps_match_the_oracle(options):
    pop = random_population(3072, ("lsystem",), seed=71, workers=4)
    xs, ys = terrain.generate_terrain()
    fo, to, co = _oracle_eval(pop, ys)
    fg, tg, cg = _gpu_eval(pop, ys, **options)
    assert np.array_equal(tg, to), "ticks differ for %d creatures" % (tg != to).sum()
    assert np.array_equal(fg, fo)
    assert cg == co


def test_config3_counters_do_not_depend_on_the_grid():
    """Config 3's 16384 creatures with the default grids and with the grids of a quarter of the shared memory: identical
    results and work counters."""
    pop = random_population(16384, ("lsystem",), seed=2, workers=8)
    xs, ys = terrain.generate_terrain()
    f1, t1, c1 = _gpu_eval(pop, ys)
    f2, t2, c2 = _gpu_eval(pop, ys, smem_budget_kb=56)
    assert np.array_equal(t1, t2) and np.array_equal(f1, f2)
    assert c1 == c2
