"""Parity of the CUDA path against the CPU oracle, through the C-ABI (pin P4). Needs a GPU.

Integer / index results (contact pairs, limit states, tick counts) must be identical; float32 state is
compared for exact equality as well: both sides perform the same IEEE operations in the same order
(no FMA contraction, shared portable sin/cos), which is far stricter than the 1e-4 relative bound the
north star asks for over the first 100 ticks.
"""
import random

import numpy as np
import pytest

from gym_rem2d_b200 import Individual, constants as K, terrain
from gym_rem2d_b200.capi import Engine
from gym_rem2d_b200.flatten import flatten_population
from oracle.oracle import OracleEngine

pytestmark = pytest.mark.gpu


def engines(ys, **cfg):
    g, o = Engine(device=0, **cfg), OracleEngine(threads=8, **cfg)
    for e in (g, o):
        e.set_terrain(ys, K.TERRAIN_STEP)
    return g, o


def assert_same_state(sg, so, what):
    for k in ("alive", "ticks", "limit_state", "n_contacts", "n_touching", "touching_pairs", "awake"):
        assert np.array_equal(sg[k], so[k]), "%s: %s differs" % (what, k)
    for k in ("pose", "vel", "joint_impulse", "motor_speed", "touching_impulse", "wod"):
        same = sg[k] == so[k]
        assert same.all(), "%s: %s differs in %d of %d values, max abs err %g" % (
            what, k, (~same).sum(), same.size, np.abs(sg[k].astype(np.float64) - so[k]).max())


@pytest.mark.parametrize("enc,flat,n,seed", [("direct", True, 256, 1), ("lsystem", False, 192, 2), ("ce", False, 128, 3),
                                             ("cppn", False, 96, 4)])
def test_first_100_ticks_bit_exact(enc, flat, n, seed):
    random.seed(seed)
    pop = flatten_population([Individual.random(encoding=enc) for _ in range(n)])
    xs, ys = terrain.flat_terrain() if flat else terrain.generate_terrain()
    g, o = engines(ys)
    g.upload(pop); o.upload(pop)
    assert_same_state(g.read_state(max_pairs=24), o.read_state(max_pairs=24), "tick 0")
    for t in (1, 1, 1, 7, 10, 30, 50):
        g.step(t); o.step(t)
        assert_same_state(g.read_state(max_pairs=24), o.read_state(max_pairs=24), "%s after +%d" % (enc, t))


# rem2d_run_episodes picks its execution mode by population size: one warp per creature (REM2D_WARP_MODE_MAX, default
# 24 per SM) for small populations, lane-per-creature bulk warps + tail warps otherwise. Both must equal the oracle.
BULK, WARP = "0", "1000000"


@pytest.mark.parametrize("mode", [BULK, WARP])
@pytest.mark.parametrize("enc,n,seed", [("direct", 512, 11), ("lsystem", 512, 12), ("ce", 256, 13)])
def test_full_episode_fitness_identical(enc, n, seed, mode, monkeypatch):
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", mode)
    random.seed(seed)
    pop = flatten_population([Individual.random(encoding=enc) for _ in range(n)])
    xs, ys = terrain.generate_terrain()
    g, o = engines(ys)
    fg, tg = g.evaluate(pop, K.EVALUATION_STEPS)
    fo, to = o.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg, to)
    assert np.array_equal(fg, fo)
    assert g.counters() == o.counters()
    assert tg.min() >= 20 and fg.max() > 5.0


def test_fixed_horizon_and_reset_reproducible():
    random.seed(21)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(96)])
    xs, ys = terrain.generate_terrain()
    g, o = engines(ys, terminate=0)
    g.upload(pop); o.upload(pop)
    g.step(300); o.step(300)
    s1 = g.read_state(max_pairs=24)
    assert_same_state(s1, o.read_state(max_pairs=24), "fixed horizon 300")
    assert (s1["ticks"] == 300).all()
    g.reset(); g.step(300)
    assert_same_state(g.read_state(max_pairs=24), s1, "after reset")


def test_single_body_creatures_sleep_and_die_like_the_oracle():
    random.seed(5)
    inds = [Individual.random(encoding="ce") for _ in range(200)]
    pop = flatten_population(inds)
    keep = np.nonzero(np.diff(pop.body_off) == 1)[0][:64]
    assert len(keep) >= 16
    sub = pop.select(keep)
    xs, ys = terrain.generate_terrain()
    g, o = engines(ys)
    g.upload(sub); o.upload(sub)
    for _ in range(5):
        g.step(30); o.step(30)
        assert_same_state(g.read_state(max_pairs=8), o.read_state(max_pairs=8), "single-body")


@pytest.mark.parametrize("mode", [BULK, WARP])
def test_episode_kernel_matches_stepping_kernel(mode, monkeypatch):
    """rem2d_run_episodes (persistent kernel, lanes refilled from a queue / a warp per creature) vs reset + step."""
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", mode)
    random.seed(31)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(700)])
    xs, ys = terrain.generate_terrain()
    g = Engine(device=0)
    g.set_terrain(ys, K.TERRAIN_STEP)
    g.upload(pop)
    g.step(K.EVALUATION_STEPS)
    f1, t1, c1 = g.fitness(), g.ticks(), g.counters()
    g.run_episodes(K.EVALUATION_STEPS)
    f2, t2, c2 = g.fitness(), g.ticks(), g.counters()
    assert np.array_equal(f1, f2) and np.array_equal(t1, t2) and c1 == c2
    with pytest.raises(Exception):
        g.step(1)                      # stepping state was consumed by the episode kernel
    g.reset(); g.step(3)
    assert (g.read_state()["ticks"] == 3).all()


@pytest.mark.parametrize("mode", [BULK, WARP])
def test_capacity_overflow_is_promoted_to_a_larger_class(mode, monkeypatch):
    """A terrain with very short edges makes every body overlap dozens of edge proxies: the contact pool of the
    creature's own class overflows and the library must transparently re-run it in a larger class."""
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", mode)
    random.seed(41)
    pop = flatten_population([Individual.random(encoding="direct") for _ in range(96)])
    ys = np.full(200, 5.0)
    step = 0.15                       # 199 edges cover x in [0, 29.9]; a 1 m wide box overlaps ~12 edge proxies
    g, o = Engine(device=0), OracleEngine(threads=8)
    for e in (g, o):
        e.set_terrain(ys, step)
    fg, tg = g.evaluate(pop, 150)
    fo, to = o.evaluate(pop, 150)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo)
    # (work counters are not compared here: aborted attempts in too-small classes are counted as work)
    assert g.counters()["ticks"] >= o.counters()["ticks"]


def test_park_cap_and_thresholds_do_not_change_results(monkeypatch):
    """The tail mode (warp-per-creature wavefront) is an execution strategy: whatever the park threshold, results
    must be identical to the oracle. A threshold of 8 ticks with 300 creatures exceeds the park cap of small classes,
    so both the parked and the not-parked continuation are exercised."""
    random.seed(51)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(300)])
    xs, ys = terrain.generate_terrain()
    o = OracleEngine(threads=8)
    o.set_terrain(ys, K.TERRAIN_STEP)
    fo, to = o.evaluate(pop, 400)
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", BULK)
    for park in ("8", "64", "0"):
        monkeypatch.setenv("REM2D_PARK_TICKS", park)
        g = Engine(device=0)
        g.set_terrain(ys, K.TERRAIN_STEP)
        fg, tg = g.evaluate(pop, 400)
        assert np.array_equal(tg, to) and np.array_equal(fg, fo), park
        assert g.counters() == o.counters(), park


def test_config2_direct_flat_1024_and_config4_mixed_cppn_ce(monkeypatch):
    """BASELINE.json configs 2 and 4 at test size: 1024 direct-encoding creatures on flat terrain (default mode for this
    size: a warp per creature), and a mixed CPPN / CE population on rough terrain (forced to the bulk mode) —
    per-creature fitness and lifetime identical to the oracle."""
    from gym_rem2d_b200.population import random_population
    pop2 = random_population(1024, ("direct",), seed=1, workers=4)
    xs, ys = terrain.flat_terrain()
    g, o = engines(ys)
    fg, tg = g.evaluate(pop2, K.EVALUATION_STEPS)
    fo, to = o.evaluate(pop2, K.EVALUATION_STEPS)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo)
    pop4 = random_population(768, ("cppn", "ce"), seed=3, workers=4)
    xs, ys = terrain.generate_terrain()
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", BULK)
    g, o = engines(ys)
    fg, tg = g.evaluate(pop4, K.EVALUATION_STEPS)
    fo, to = o.evaluate(pop4, K.EVALUATION_STEPS)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo)
    assert g.counters() == o.counters()


@pytest.mark.parametrize("tan_slope", [0.6, -0.35])
def test_inclined_terrain_and_no_sleep_bit_exact(tan_slope):
    """Edge chains that are not axis-aligned (sliding and tumbling creatures, manifolds across collinear edges, bodies that
    start inside the slope) with sleeping disabled and a fixed horizon: state after every block of ticks identical to the
    oracle."""
    random.seed(61)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(160)])
    xs = np.arange(200) * K.TERRAIN_STEP
    x_start = K.TERRAIN_STEP * K.TERRAIN_STARTPAD / 2          # creatures are built around (x_start, TERRAIN_HEIGHT + 2)
    ys = K.TERRAIN_HEIGHT - tan_slope * (xs - x_start)
    g, o = Engine(device=0, terminate=0, allow_sleep=0), OracleEngine(threads=8, terminate=0, allow_sleep=0)
    for e in (g, o):
        e.set_terrain(ys, K.TERRAIN_STEP)
    g.upload(pop); o.upload(pop)
    for t in (20, 40, 60, 80):
        g.step(t); o.step(t)
        assert_same_state(g.read_state(max_pairs=16), o.read_state(max_pairs=16), "incline %.2f after +%d" % (tan_slope, t))


# ---------------------------------------------------------------------------------------------------------------------
# The PRODUCTION execution path at test size (VERDICT r1, item 1): persistent bulk warps whose lanes are REFILLED from the
# class queue (first-wave grid < n_batches), parking at 256 ticks with a 1/16 cap and on-demand tail launches that see
# late-parked creatures. A small shared-memory budget forces several refill rounds with a few thousand creatures.
def _oracle_eval(pop, ys, steps=K.EVALUATION_STEPS, **cfg):
    o = OracleEngine(threads=max(8, (__import__("os").cpu_count() or 8)), **cfg)
    o.set_terrain(ys, K.TERRAIN_STEP)
    fo, to = o.evaluate(pop, steps)
    return fo, to, o.counters()


@pytest.mark.parametrize("budget_kb,park", [("24", None), ("40", "140"), ("16", "256")])
def test_lane_refill_rounds_and_late_parking_match_the_oracle(budget_kb, park, monkeypatch):
    from gym_rem2d_b200.population import random_population
    pop = random_population(3072, ("lsystem",), seed=71, workers=4)
    xs, ys = terrain.generate_terrain()
    fo, to, co = _oracle_eval(pop, ys)
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", "0")
    monkeypatch.setenv("REM2D_SMEM_BUDGET_KB", budget_kb)      # per-SM budget: every class gets fewer warps than batches
    if park is not None:
        monkeypatch.setenv("REM2D_PARK_TICKS", park)
        monkeypatch.setenv("REM2D_PARK_CAP", "0.0625")
    g = Engine(device=0)
    g.set_terrain(ys, K.TERRAIN_STEP)
    fg, tg = g.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg, to), "ticks differ for %d creatures" % (tg != to).sum()
    assert np.array_equal(fg, fo)
    assert g.counters() == co
    assert (to > 256).sum() >= 3, "the population must contain creatures that outlive the park threshold"
    # same handle, second evaluation (buffers and queues are reused)
    fg2, tg2 = g.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg2, to) and np.array_equal(fg2, fo)


@pytest.mark.parametrize("terminate", [1, 0])
def test_config1_single_creature_1000_ticks(terminate):
    """BASELINE config 1: ONE direct-encoding creature (seed 0), flat terrain, 1000 ticks with the termination rule on and
    off — state after every 100 ticks and the episode result identical to the oracle."""
    random.seed(0)
    np.random.seed(0)
    pop = flatten_population([Individual.random(encoding="direct")])
    xs, ys = terrain.flat_terrain()
    g, o = engines(ys, terminate=terminate)
    g.upload(pop); o.upload(pop)
    for _ in range(10):
        g.step(100); o.step(100)
        assert_same_state(g.read_state(max_pairs=24), o.read_state(max_pairs=24), "config 1, terminate=%d" % terminate)
    if not terminate:
        assert (g.read_state()["ticks"] == 1000).all()
    fg, tg = g.evaluate(pop, 1000)
    fo, to = o.evaluate(pop, 1000)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo)


def test_config3_16384_lsystem_rough_full_size():
    """BASELINE config 3 at its stated size: 16384 L-system creatures (seed 2), rough terrain, whole episodes in the default
    execution mode for this size (bulk warps, under-filled GPU -> park at 160 ticks)."""
    from gym_rem2d_b200.population import random_population
    pop = random_population(16384, ("lsystem",), seed=2, workers=8)
    xs, ys = terrain.generate_terrain()
    fo, to, co = _oracle_eval(pop, ys)
    g = Engine(device=0)
    g.set_terrain(ys, K.TERRAIN_STEP)
    fg, tg = g.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo)
    assert g.counters() == co


def test_config4_4096_cppn_ce_rough():
    from gym_rem2d_b200.population import random_population
    pop = random_population(4096, ("cppn", "ce"), seed=3, workers=8)
    xs, ys = terrain.generate_terrain()
    fo, to, co = _oracle_eval(pop, ys)
    g = Engine(device=0)
    g.set_terrain(ys, K.TERRAIN_STEP)
    fg, tg = g.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo)
    assert g.counters() == co


def test_full_size_population_is_order_independent():
    """BASELINE's full size (65536 L-system creatures, the bench population) through a size-independent property: a creature's
    fitness and lifetime do not depend on its position in the population - a permuted population lands on other lanes, other
    rounds of the class queues and other tail launches, and must give the permuted results; 4096 of them are also checked
    against the oracle."""
    from gym_rem2d_b200.population import random_population
    pop = random_population(65536, ("lsystem",), seed=2, workers=8)
    xs, ys = terrain.generate_terrain()
    g = Engine(device=0)
    g.set_terrain(ys, K.TERRAIN_STEP)
    f, t = g.evaluate(pop, K.EVALUATION_STEPS)
    perm = np.random.RandomState(5).permutation(65536)
    f2, t2 = g.evaluate(pop.select(perm), K.EVALUATION_STEPS)
    assert np.array_equal(t2, t[perm]) and np.array_equal(f2, f[perm])
    sample = np.sort(perm[:4096])
    fo, to, _ = _oracle_eval(pop.select(sample), ys)
    assert np.array_equal(t[sample], to) and np.array_equal(f[sample], fo)
    g.close()


def test_ea_configured_population_mixed_widths_and_overflow_wave():
    """A population as run_deap configures it (max_size 40: creatures of up to 41 bodies) that does not fit on the GPU at once:
    the 33-44 body class runs 8 lanes per creature next to one-lane classes, the first wave is sized to 75 % of the shared
    memory, every class queues an overflow wave behind the first launches, and the lifetime hint reorders the class queues.
    2048 distinct creatures (checked against the oracle), tiled 24 times."""
    from gym_rem2d_b200 import ea
    from gym_rem2d_b200.modules import get_module_list
    random.seed(21); np.random.seed(21)
    cfg = ea.default_config(enc="lsystem")
    base = flatten_population([Individual.random(get_module_list(), cfg) for _ in range(2048)], 7)
    nb = np.diff(base.body_off)
    assert (nb > 32).sum() > 100 and nb.max() <= 44
    xs, ys = terrain.generate_terrain()
    fo, to, co = _oracle_eval(base, ys)
    pop = base.select(np.tile(np.arange(2048), 24))
    g = Engine(device=0)
    g.set_terrain(ys, K.TERRAIN_STEP)
    fg, tg = g.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg, np.tile(to, 24)) and np.array_equal(fg, np.tile(fo, 24))
    assert g.launch_count() > 2 * 9                         # first launches + overflow waves (+ tails)
    g.set_priority(np.tile(to, 24).astype(np.float32))      # longest-lived first: another order, the same results
    fg2, tg2 = g.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg2, tg) and np.array_equal(fg2, fg)
    g.set_option("overflow_wave", 0)
    fg3, tg3 = g.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg3, tg) and np.array_equal(fg3, fg)
    g.close()


# ---------------------------------------------------------------------------------------------------------------------
# Lanes per creature (group shift): the same kernels with G = 1, 2, 4, 8, 32 lanes per creature must all equal the oracle.
@pytest.mark.parametrize("gs", ["0", "1", "2", "3", "5"])
def test_every_group_size_stepping_kernel_bit_exact(gs, monkeypatch):
    monkeypatch.setenv("REM2D_GROUP_SHIFT", gs)
    random.seed(81)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(160)])
    xs, ys = terrain.generate_terrain()
    g, o = engines(ys)
    g.upload(pop); o.upload(pop)
    for t in (1, 9, 40, 60):
        g.step(t); o.step(t)
        assert_same_state(g.read_state(max_pairs=24), o.read_state(max_pairs=24), "gs=%s after +%d" % (gs, t))
    assert g.counters() == o.counters()


@pytest.mark.parametrize("gs,tail_gs", [("0", "5"), ("1", "3"), ("2", "5"), ("3", "4"), ("4", "2")])
def test_every_group_size_queue_and_tail_modes_full_episodes(gs, tail_gs, monkeypatch):
    from gym_rem2d_b200.population import random_population
    pop = random_population(1536, ("lsystem",), seed=83, workers=4)
    xs, ys = terrain.generate_terrain()
    fo, to, co = _oracle_eval(pop, ys)
    monkeypatch.setenv("REM2D_GROUP_SHIFT", gs)
    monkeypatch.setenv("REM2D_TAIL_GROUP_SHIFT", tail_gs)
    monkeypatch.setenv("REM2D_WARP_MODE_MAX", "0")
    monkeypatch.setenv("REM2D_SMEM_BUDGET_KB", "30")
    monkeypatch.setenv("REM2D_PARK_TICKS", "130")
    monkeypatch.setenv("REM2D_PARK_CAP", "0.1")
    g = Engine(device=0)
    g.set_terrain(ys, K.TERRAIN_STEP)
    fg, tg = g.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg, to), "ticks differ for %d creatures" % (tg != to).sum()
    assert np.array_equal(fg, fo)
    assert g.counters() == co


def test_set_option_and_read_roots():
    random.seed(91)
    pop = flatten_population([Individual.random(encoding="direct") for _ in range(40)])
    xs, ys = terrain.generate_terrain()
    g, o = engines(ys)
    g.set_option("group_shift", 2)
    with pytest.raises(Exception):
        g.set_option("no_such_option", 1)
    g.upload(pop); o.upload(pop)
    g.step(50); o.step(50)
    xg, wg, ag = g.read_roots()
    xo, wo, ao = o.read_roots()
    assert np.array_equal(xg, xo) and np.array_equal(wg, wo) and np.array_equal(ag, ao)
    root = pop.body_off[:-1]
    assert np.array_equal(xg, g.read_state()["pose"][root, 0])


def test_priority_hint_changes_the_schedule_not_the_results():
    from gym_rem2d_b200.population import random_population
    pop = random_population(2048, ("lsystem",), seed=97, workers=4)
    xs, ys = terrain.generate_terrain()
    fo, to, co = _oracle_eval(pop, ys)
    g = Engine(device=0)
    g.set_option("warp_mode_max", 0); g.set_option("group_shift", 0); g.set_option("smem_budget_kb", 20)
    g.set_terrain(ys, K.TERRAIN_STEP)
    g.set_priority(to.astype(np.float32))            # a perfect hint: the real lifetimes
    fg, tg = g.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo) and g.counters() == co
    g.set_priority(np.random.RandomState(0).uniform(0, 400, pop.n_creatures))      # a useless one
    fg, tg = g.evaluate(pop, K.EVALUATION_STEPS)
    assert np.array_equal(tg, to) and np.array_equal(fg, fo)


def test_fast_precision_build_keeps_the_fitness_distribution():
    """Engine(precision="fast") = the same kernels compiled with fused multiply-adds: not bit-identical any more (individual
    trajectories diverge chaotically after contact events), judged on the fitness distribution of whole episodes."""
    from gym_rem2d_b200.population import random_population
    from tests.test_fitness_distribution import ks_statistic
    pop = random_population(4096, ("lsystem",), seed=2, workers=4)
    xs, ys = terrain.generate_terrain()
    res = {}
    for precision in ("exact", "fast"):
        g = Engine(device=0, precision=precision)
        g.set_terrain(ys, K.TERRAIN_STEP)
        res[precision] = g.evaluate(pop, K.EVALUATION_STEPS)
    (fe, te), (ff, tf) = res["exact"], res["fast"]
    assert not np.array_equal(fe, ff)                       # it really is a different arithmetic
    assert ks_statistic(fe, ff) <= 0.02 and abs(fe.mean() - ff.mean()) <= 0.01
    assert np.mean(te == tf) >= 0.9
