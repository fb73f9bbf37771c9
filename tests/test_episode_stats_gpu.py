"""Episode statistics of the CUDA library (the statistics images of the episode kernel) against the oracle, bit for bit, under
every execution strategy: bulk and warp mode, parking and tail launches, forced group widths, refill rounds, the overflow wave,
the 128-register image, re-runs after a capacity overflow and regrouping of draining warps (reference: the oracle with
statistics, tests/oracle_ext). Statistics never change results, in the exact and in the fast build, and the call contract is the
oracle's. Needs a GPU; tests/test_episode_stats.py checks the oracle and the device code on the CPU."""
import os
import random
import sys

import numpy as np
import pytest

from gym_rem2d_b200 import Individual, constants as K, terrain
from gym_rem2d_b200.capi import Engine
from gym_rem2d_b200.flatten import flatten_population
from gym_rem2d_b200.population import random_population

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "oracle_ext"))
from oracle_ext import OracleExtEngine  # noqa: E402
from tests.test_episode_stats import check_contract, population  # noqa: E402

pytestmark = pytest.mark.gpu

NAMES = ("end_reason", "max_x", "joint_work", "airborne_ticks", "ground_ticks")
BULK, WARP = "0", "1000000"


def assert_stats_equal(a, b, what=""):
    for k in NAMES:
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, (what, k)
        assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), "%s: %s differs in %d values" % (
            what, k, (a[k] != b[k]).sum())


def oracle_eval(pop, ys, max_ticks=K.EVALUATION_STEPS, step=K.TERRAIN_STEP):
    o = OracleExtEngine(threads=max(8, os.cpu_count() or 8))
    o.set_terrain(ys, step)
    o.set_stats(True)
    f, t = o.evaluate(pop, max_ticks)
    return f, t, o.read_stats()


def gpu_eval(pop, ys, max_ticks=K.EVALUATION_STEPS, step=K.TERRAIN_STEP, stats=True, precision="exact", **options):
    g = Engine(device=0, precision=precision)
    g.set_terrain(ys, step)
    for k, v in options.items():
        g.set_option(k, v)
    g.set_stats(stats)
    f, t = g.evaluate(pop, max_ticks)
    out = f, t, g.counters(), (g.read_stats() if stats else None)
    g.close()
    return out


@pytest.mark.parametrize("mode", [BULK, WARP])
@pytest.mark.parametrize("enc,n,seed", [("direct", 512, 11), ("lsystem", 512, 12), ("ce", 256, 13)])
def test_full_episodes_match_the_oracle(enc, n, seed, mode, monkeypatch):
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", mode)
    random.seed(seed)
    pop = flatten_population([Individual.random(encoding=enc) for _ in range(n)])
    xs, ys = terrain.generate_terrain()
    fo, to, so = oracle_eval(pop, ys)
    fg, tg, cg, sg = gpu_eval(pop, ys)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo)
    assert_stats_equal(sg, so, "%s mode %s" % (enc, mode))
    f0, t0, c0, _ = gpu_eval(pop, ys, stats=False)
    assert np.array_equal(f0, fg) and np.array_equal(t0, tg) and c0 == cg


def test_park_thresholds(monkeypatch):
    random.seed(51)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(300)])
    xs, ys = terrain.generate_terrain()
    fo, to, so = oracle_eval(pop, ys, 400)
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", BULK)
    for park in (8, 64, 0):
        fg, tg, cg, sg = gpu_eval(pop, ys, 400, park_ticks=park)
        assert np.array_equal(tg, to) and np.array_equal(fg, fo), park
        assert_stats_equal(sg, so, "park %d" % park)


def test_forced_group_widths_refill_rounds_and_tails():
    pop = random_population(1024, ("lsystem",), seed=81, workers=4)
    xs, ys = terrain.generate_terrain()
    fo, to, so = oracle_eval(pop, ys)
    for gs in range(6):
        fg, tg, cg, sg = gpu_eval(pop, ys, warp_mode_max=0, group_shift=gs, tail_group_shift=max(gs, 1), smem_budget_kb=16,
                                  park_ticks=130)
        assert np.array_equal(tg, to) and np.array_equal(fg, fo), gs
        assert_stats_equal(sg, so, "group_shift %d" % gs)


def test_ea_configured_population_overflow_wave_and_image():
    from gym_rem2d_b200 import ea
    from gym_rem2d_b200.modules import get_module_list
    random.seed(21); np.random.seed(21)
    cfg = ea.default_config(enc="lsystem")
    base = flatten_population([Individual.random(get_module_list(), cfg) for _ in range(2048)], 7)
    xs, ys = terrain.generate_terrain()
    fo, to, so = oracle_eval(base, ys)
    tiles = 24
    idx = np.tile(np.arange(2048), tiles)
    pop = base.select(idx)
    bodies = np.concatenate([np.arange(base.body_off[c], base.body_off[c + 1]) for c in idx])
    want = {k: (v[bodies] if k == "ground_ticks" else v[idx]) for k, v in so.items()}
    for options in (dict(), dict(overflow_wave=0), dict(image=1)):
        g = Engine(device=0)
        g.set_terrain(ys, K.TERRAIN_STEP)
        for k, v in options.items():
            g.set_option(k, v)
        g.set_stats(True)
        fg, tg = g.evaluate(pop, K.EVALUATION_STEPS)
        assert np.array_equal(tg, np.tile(to, tiles)) and np.array_equal(fg, np.tile(fo, tiles)), options
        assert_stats_equal(g.read_stats(), want, str(options))
        if not options:
            assert g.launch_count() > 2 * 9
        g.close()


@pytest.mark.parametrize("mode", [BULK, WARP])
def test_capacity_overflow_reruns(mode, monkeypatch):
    """Short terrain edges overflow the contact pools: creatures are re-run from tick 0 in a larger class, and their statistics
    must be those of the re-run alone."""
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", mode)
    random.seed(41)
    pop = flatten_population([Individual.random(encoding="direct") for _ in range(96)])
    ys = np.full(200, 5.0)
    fo, to, so = oracle_eval(pop, ys, 150, step=0.15)
    fg, tg, cg, sg = gpu_eval(pop, ys, 150, step=0.15)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo)
    assert_stats_equal(sg, so, "overflow %s" % mode)


@pytest.mark.parametrize("options", [
    dict(warp_mode_max=0, park_ticks=0, smem_budget_kb=24),
    dict(warp_mode_max=0, park_ticks=0, smem_budget_kb=40, group_shift=0),
    dict(warp_mode_max=0, park_ticks=140, park_cap=0.0625, tail_group_shift=1, smem_budget_kb=24),
])
def test_draining_warps(options):
    pop = random_population(3072, ("lsystem",), seed=71, workers=4)
    xs, ys = terrain.generate_terrain()
    fo, to, so = oracle_eval(pop, ys)
    fg, tg, cg, sg = gpu_eval(pop, ys, **options)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo)
    assert_stats_equal(sg, so, str(options))


def test_fast_build_results_do_not_change():
    pop = random_population(2048, ("lsystem", "ce"), seed=91, workers=4)
    xs, ys = terrain.generate_terrain()
    f0, t0, c0, _ = gpu_eval(pop, ys, precision="fast", stats=False)
    f1, t1, c1, s1 = gpu_eval(pop, ys, precision="fast")
    assert np.array_equal(f0, f1) and np.array_equal(t0, t1) and c0 == c1
    assert s1["ground_ticks"].shape == (pop.n_bodies,) and (s1["end_reason"] > 0).all()


def test_python_interfaces():
    from gym_rem2d_b200.env import BatchedModular2D, evaluate_population
    random.seed(3)
    inds = [Individual.random(encoding="lsystem") for _ in range(64)]
    env = BatchedModular2D()
    fit_plain = env.evaluate(inds)
    assert env.last_stats is None
    fit, stats = evaluate_population(inds, env=env, as_torch=False, return_stats=True)
    assert np.array_equal(fit, fit_plain)
    table = env.table
    n, nb = table.n_creatures, table.n_bodies
    assert stats["end_reason"].shape == (n,) and stats["max_x"].dtype == np.float32 and stats["joint_work"].dtype == np.float64
    assert stats["airborne_ticks"].shape == (n,) and stats["ground_ticks"].shape == (nb,)
    fo, to, so = oracle_eval(table, env.terrain_y)
    assert_stats_equal(stats, so, "evaluate_population")
    assert evaluate_population(inds, env=env, as_torch=False).shape == (n,)
    env2 = BatchedModular2D(stats=True)
    env2.evaluate(table=table)
    assert_stats_equal(env2.last_stats, so, "BatchedModular2D(stats=True)")
    env.close(); env2.close()


def test_contract_equals_the_oracle():
    """The statistics' call contract that tests/test_episode_stats.py checks on the oracle, on the CUDA library."""
    xs, ys = terrain.generate_terrain()
    g = Engine(device=0)
    g.set_terrain(ys, K.TERRAIN_STEP)
    check_contract(g, population("direct", 16, 3))
    g.close()
