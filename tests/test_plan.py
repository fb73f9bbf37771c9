"""The episode planner of the CUDA library (rem2d_host_util.h: plan_upload, plan_launch, step_group_shift), run on the CPU
through the emulation build: the plans of the populations the benchmark and the GPU tests run, and properties every plan has.
The planner is plain arithmetic on the class sizes, the SM count, the resident warps per SM and the options, so none of
this needs a GPU."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu  # noqa: E402

# B200: 148 SMs; 9 and 16 resident warps per SM for the 202- and 126-register episode kernel images (occupancy API).
N_SMS, MAX_WARPS = 148, (9, 16)

# Per capacity class: the number of creatures and the sum of their cost estimates (1 for a lone body, 3.5 + bodies
# otherwise), as rem2d_upload computes them for the named population.
LOADS = {
    # bench.py's population: random_population(65536, ("lsystem",), seed=2)
    "bench": ([16438, 9818, 11984, 4914, 3807, 1500, 17075, 0, 0],
             [16438.0, 53999.0, 83203.0, 46681.0, 49531.5, 27039.0, 396092.5, 0.0, 0.0]),
    # BASELINE config 3: random_population(16384, ("lsystem",), seed=2)
    "config3": ([4158, 2445, 3022, 1217, 927, 350, 4265, 0, 0],
               [4158.0, 13447.5, 20991.0, 11523.5, 12067.5, 6272.0, 98828.5, 0.0, 0.0]),
    # test_ea_configured_population_mixed_widths_and_overflow_wave: 2048 creatures of ea.default_config(enc="lsystem")
    # (seed 21), tiled 24 times
    "ea_configured": ([12456, 6984, 8400, 5496, 1608, 3648, 3096, 2088, 5376],
                     [12456.0, 38412.0, 58104.0, 55332.0, 22524.0, 67104.0, 75108.0, 65292.0, 225648.0]),
    # BASELINE config 2 at its size: random_population(1024, ("direct",), seed=1)
    "config2": ([16, 99, 587, 319, 3, 0, 0, 0, 0],
               [16.0, 544.5, 4113.5, 2916.5, 40.5, 0.0, 0.0, 0.0, 0.0]),
    # random_population(768, ("cppn", "ce"), seed=3) (test_config2_direct_flat_1024_and_config4_mixed_cppn_ce)
    "config4_768": ([380, 56, 205, 21, 9, 9, 88, 0, 0],
                   [380.0, 308.0, 1499.5, 199.5, 121.5, 162.5, 2110.0, 0.0, 0.0]),
    # random_population(3072, ("lsystem",), seed=71) (test_lane_refill_rounds_and_late_parking_match_the_oracle)
    "refill_3072": ([785, 451, 565, 210, 184, 67, 810, 0, 0],
                   [785.0, 2480.5, 3911.5, 1973.0, 2398.0, 1222.5, 18797.0, 0.0, 0.0]),
    # random_population(1536, ("lsystem",), seed=83) (test_every_group_size_queue_and_tail_modes_full_episodes)
    "group_shift_1536": ([371, 225, 273, 100, 105, 42, 420, 0, 0],
                        [371.0, 1237.5, 1889.5, 962.0, 1362.5, 750.0, 9705.0, 0.0, 0.0]),
    # random_population(2048, ("lsystem",), seed=97) (test_priority_hint_changes_the_schedule_not_the_results)
    "priority_2048": ([470, 323, 372, 177, 105, 43, 558, 0, 0],
                     [470.0, 1776.5, 2574.0, 1664.5, 1375.5, 773.5, 12924.0, 0.0, 0.0]),
}

# name: (population, options, max_ticks). The options are the ones the GPU tests and tools force.
GS_OPTIONS = {"warp_mode_max": 0, "smem_budget_kb": 30, "park_ticks": 130, "park_cap": 0.1}
CASES = {
    "bench": ("bench", {}, 10000),
    "bench_class_gs": ("bench", {"class_gs_6": 1, "class_gs_8": 5}, 10000),
    "bench_image_1": ("bench", {"image": 1}, 10000),
    "config3": ("config3", {}, 10000),
    "ea_configured": ("ea_configured", {}, 10000),
    "ea_configured_no_overflow_wave": ("ea_configured", {"overflow_wave": 0}, 10000),
    "config2_warp_mode": ("config2", {}, 10000),
    "config2_bulk": ("config2", {"warp_mode_max": 0}, 10000),
    "config4_bulk": ("config4_768", {"warp_mode_max": 0}, 10000),
    "config4_bulk_150_ticks": ("config4_768", {"warp_mode_max": 0}, 150),
    "refill_24": ("refill_3072", {"warp_mode_max": 0, "smem_budget_kb": 24}, 10000),
    "refill_40_park_140": ("refill_3072", {"warp_mode_max": 0, "smem_budget_kb": 40, "park_ticks": 140, "park_cap": 0.0625}, 10000),
    "refill_16_park_256": ("refill_3072", {"warp_mode_max": 0, "smem_budget_kb": 16, "park_ticks": 256, "park_cap": 0.0625}, 10000),
    **{"group_shift_%d" % g: ("group_shift_1536", dict(group_shift=g, **GS_OPTIONS), 10000) for g in range(5)},
    "priority": ("priority_2048", {"warp_mode_max": 0, "group_shift": 0, "smem_budget_kb": 20}, 10000),
}

# The plans, as the scheduler computed them before it was turned into pure functions.
PLANS = {
    "bench": dict(image=0, all_fit=False, warp_mode=False, park_ticks=200,
                  gs=[0, 0, 0, 0, 0, 0, 0, 0, 3], grid=[14, 46, 71, 40, 42, 23, 342, 0, 0],
                  grid2=[500, 261, 304, 114, 77, 24, 192, 0, 0], park_cap=[2368, 2368, 2368, 1228, 951, 375, 2368, 0, 0],
                  order=[7, 6, 5, 4, 3, 8, 2, 1, 0], step_gs=[0, 0, 0, 0, 0, 0, 0, 0, 0]),
    "bench_class_gs": dict(image=0, all_fit=False, warp_mode=False, park_ticks=200,
                           gs=[0, 0, 0, 0, 0, 0, 1, 0, 5], grid=[10, 35, 54, 30, 32, 17, 448, 0, 0],
                           grid2=[504, 272, 321, 124, 87, 30, 620, 0, 0], park_cap=[2368, 2368, 2368, 1228, 951, 375, 2368, 0, 0],
                           order=[7, 5, 4, 6, 3, 2, 1, 8, 0], step_gs=[0, 0, 0, 0, 0, 0, 1, 0, 5]),
    "bench_image_1": dict(image=1, all_fit=False, warp_mode=False, park_ticks=200,
                          gs=[0, 0, 0, 0, 0, 0, 0, 0, 3], grid=[14, 46, 71, 40, 42, 23, 342, 0, 0],
                          grid2=[500, 261, 304, 114, 77, 24, 192, 0, 0], park_cap=[2368, 2368, 2368, 1228, 951, 375, 2368, 0, 0],
                          order=[7, 6, 5, 4, 3, 8, 2, 1, 0], step_gs=[0, 0, 0, 0, 0, 0, 0, 0, 0]),
    "config3": dict(image=1, all_fit=True, warp_mode=False, park_ticks=160,
                    gs=[0, 0, 1, 2, 2, 2, 2, 2, 2], grid=[130, 77, 189, 153, 116, 44, 534, 0, 0],
                    grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[1039, 611, 755, 304, 231, 87, 1066, 0, 0],
                    order=[8, 7, 6, 5, 4, 1, 3, 2, 0], step_gs=[0, 0, 1, 1, 1, 1, 1, 1, 1]),
    "ea_configured": dict(image=0, all_fit=False, warp_mode=False, park_ticks=200,
                          gs=[0, 0, 0, 0, 0, 0, 0, 0, 3], grid=[6, 20, 30, 29, 12, 35, 40, 34, 506],
                          grid2=[384, 199, 233, 143, 39, 79, 57, 32, 838], park_cap=[2368, 1746, 2100, 1374, 402, 912, 774, 522, 1344],
                          order=[7, 6, 5, 4, 3, 8, 2, 1, 0], step_gs=[0, 0, 0, 0, 0, 0, 0, 0, 0]),
    "ea_configured_no_overflow_wave": dict(image=0, all_fit=False, warp_mode=False, park_ticks=200,
                                           gs=[0, 0, 0, 0, 0, 0, 0, 0, 3], grid=[8, 27, 41, 39, 16, 47, 53, 46, 675],
                                           grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[2368, 1746, 2100, 1374, 402, 912, 774, 522, 1344],
                                           order=[7, 6, 5, 4, 3, 8, 2, 1, 0], step_gs=[0, 0, 0, 0, 0, 0, 0, 0, 0]),
    "config2_warp_mode": dict(image=1, all_fit=True, warp_mode=True, park_ticks=0,
                              gs=[0, 0, 1, 3, 5, 5, 5, 5, 5], grid=[1, 4, 37, 80, 3, 0, 0, 0, 0],
                              grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[16, 32, 146, 79, 3, 0, 0, 0, 0],
                              order=[8, 7, 6, 5, 4, 3, 2, 1, 0], step_gs=[0, 0, 5, 5, 5, 5, 5, 5, 5]),
    "config2_bulk": dict(image=1, all_fit=True, warp_mode=False, park_ticks=160,
                         gs=[0, 0, 1, 3, 5, 5, 5, 5, 5], grid=[1, 4, 37, 80, 3, 0, 0, 0, 0],
                         grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[16, 32, 146, 79, 3, 0, 0, 0, 0],
                         order=[1, 2, 8, 0, 7, 6, 5, 4, 3], step_gs=[0, 0, 5, 5, 5, 5, 5, 5, 5]),
    "config4_bulk": dict(image=1, all_fit=True, warp_mode=False, park_ticks=160,
                         gs=[0, 0, 1, 3, 5, 5, 5, 5, 5], grid=[12, 2, 13, 6, 9, 9, 88, 0, 0],
                         grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[95, 32, 51, 21, 9, 9, 32, 0, 0],
                         order=[1, 2, 8, 0, 7, 6, 5, 4, 3], step_gs=[0, 0, 5, 5, 5, 5, 5, 5, 5]),
    "config4_bulk_150_ticks": dict(image=1, all_fit=True, warp_mode=False, park_ticks=0,
                                   gs=[0, 0, 1, 3, 5, 5, 5, 5, 5], grid=[12, 2, 13, 6, 9, 9, 88, 0, 0],
                                   grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[95, 32, 51, 21, 9, 9, 32, 0, 0],
                                   order=[1, 2, 8, 0, 7, 6, 5, 4, 3], step_gs=[0, 0, 5, 5, 5, 5, 5, 5, 5]),
    "refill_24": dict(image=0, all_fit=False, warp_mode=False, park_ticks=200,
                      gs=[0, 0, 0, 0, 0, 0, 0, 0, 3], grid=[18, 15, 18, 7, 6, 3, 26, 0, 0],
                      grid2=[7, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[196, 112, 141, 52, 46, 32, 202, 0, 0],
                      order=[7, 6, 5, 4, 3, 8, 2, 1, 0], step_gs=[0, 0, 3, 3, 3, 3, 3, 3, 3]),
    "refill_40_park_140": dict(image=1, all_fit=True, warp_mode=False, park_ticks=140,
                               gs=[0, 0, 1, 3, 3, 3, 3, 3, 3], grid=[25, 15, 36, 53, 46, 17, 203, 0, 0],
                               grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[49, 32, 35, 32, 32, 32, 50, 0, 0],
                               order=[8, 7, 1, 6, 2, 5, 4, 0, 3], step_gs=[0, 0, 3, 3, 3, 3, 3, 3, 3]),
    "refill_16_park_256": dict(image=0, all_fit=False, warp_mode=False, park_ticks=256,
                               gs=[0, 0, 0, 0, 0, 0, 0, 0, 3], grid=[1, 3, 5, 2, 3, 1, 24, 0, 0],
                               grid2=[24, 12, 13, 5, 3, 2, 2, 0, 0], park_cap=[49, 32, 35, 32, 32, 32, 50, 0, 0],
                               order=[7, 6, 5, 4, 3, 8, 2, 1, 0], step_gs=[0, 0, 3, 3, 3, 3, 3, 3, 3]),
    "group_shift_0": dict(image=1, all_fit=True, warp_mode=False, park_ticks=130,
                          gs=[0, 0, 0, 0, 0, 0, 0, 0, 0], grid=[12, 8, 9, 4, 4, 2, 14, 0, 0],
                          grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[37, 32, 32, 32, 32, 32, 42, 0, 0],
                          order=[8, 7, 6, 5, 4, 3, 2, 1, 0], step_gs=[0, 0, 0, 0, 0, 0, 0, 0, 0]),
    "group_shift_1": dict(image=1, all_fit=True, warp_mode=False, park_ticks=130,
                          gs=[1, 1, 1, 1, 1, 1, 1, 1, 1], grid=[24, 15, 18, 7, 7, 3, 27, 0, 0],
                          grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[37, 32, 32, 32, 32, 32, 42, 0, 0],
                          order=[8, 7, 6, 5, 4, 3, 2, 1, 0], step_gs=[1, 1, 1, 1, 1, 1, 1, 1, 1]),
    "group_shift_2": dict(image=1, all_fit=True, warp_mode=False, park_ticks=130,
                          gs=[2, 2, 2, 2, 2, 2, 2, 2, 2], grid=[47, 29, 35, 13, 14, 6, 53, 0, 0],
                          grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[37, 32, 32, 32, 32, 32, 42, 0, 0],
                          order=[8, 7, 6, 5, 4, 3, 2, 1, 0], step_gs=[2, 2, 2, 2, 2, 2, 2, 2, 2]),
    "group_shift_3": dict(image=1, all_fit=True, warp_mode=False, park_ticks=130,
                          gs=[3, 3, 3, 3, 3, 3, 3, 3, 3], grid=[93, 57, 69, 25, 27, 11, 105, 0, 0],
                          grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[37, 32, 32, 32, 32, 32, 42, 0, 0],
                          order=[8, 7, 6, 5, 4, 3, 2, 1, 0], step_gs=[3, 3, 3, 3, 3, 3, 3, 3, 3]),
    "group_shift_4": dict(image=0, all_fit=False, warp_mode=False, park_ticks=130,
                          gs=[4, 4, 4, 4, 4, 4, 4, 4, 4], grid=[11, 39, 60, 30, 43, 21, 210, 0, 0],
                          grid2=[175, 74, 77, 20, 10, 0, 0, 0, 0], park_cap=[37, 32, 32, 32, 32, 32, 42, 0, 0],
                          order=[8, 7, 6, 5, 4, 3, 2, 1, 0], step_gs=[4, 4, 4, 4, 4, 4, 4, 4, 4]),
    "priority": dict(image=1, all_fit=True, warp_mode=False, park_ticks=160,
                     gs=[0, 0, 0, 0, 0, 0, 0, 0, 0], grid=[15, 11, 12, 6, 4, 2, 18, 0, 0],
                     grid2=[0, 0, 0, 0, 0, 0, 0, 0, 0], park_cap=[117, 80, 93, 44, 32, 32, 139, 0, 0],
                     order=[8, 7, 6, 5, 4, 3, 2, 1, 0], step_gs=[0, 0, 0, 0, 0, 0, 0, 0, 0]),
}


def plan(load, options, max_ticks):
    return emu.plan(*load, options=options, max_ticks=max_ticks, n_sms=N_SMS, max_warps_per_sm=MAX_WARPS)


@pytest.mark.parametrize("name", sorted(CASES))
def test_pinned_plans(name):
    population, options, max_ticks = CASES[name]
    assert plan(LOADS[population], options, max_ticks) == PLANS[name]


def test_class_table():
    assert emu.classes() == [(1, 10, 3, 0), (2, 16, 4, 0), (4, 28, 4, 1), (8, 48, 6, 3), (12, 64, 6, 5), (16, 80, 6, 5),
                             (22, 104, 6, 5), (32, 144, 8, 5), (44, 192, 10, 5)]


def random_cases(n, seed):
    """Random class histograms (empty classes, a handful of creatures, up to 300000) with random option sets."""
    rng = np.random.RandomState(seed)
    lo = [1, 2, 3, 5, 9, 13, 17, 23, 33]
    hi = [nb for nb, _, _, _ in emu.classes()]
    for _ in range(n):
        scale = np.exp(rng.uniform(0, np.log(3e5)))
        members = np.where(rng.rand(9) < rng.uniform(0.2, 1.0), (scale * rng.rand(9)).astype(np.int64), 0)
        bodies = rng.uniform(lo, hi)
        work = members * np.where(bodies < 1.5, 1.0, 3.5 + bodies)
        options = {}
        if rng.rand() < 0.15:
            options["group_shift"] = int(rng.randint(-1, 8))
        for k in range(9):
            if rng.rand() < 0.05:
                options["class_gs_%d" % k] = int(rng.randint(-1, 7))
        if rng.rand() < 0.3:
            options["smem_budget_kb"] = float(rng.choice([10, 24, 40, 100, 226, 226.5, 227, rng.uniform(5, 240)]))
        if rng.rand() < 0.3:
            options["overflow_wave"] = int(rng.randint(0, 2))
        if rng.rand() < 0.2:
            options["image"] = int(rng.randint(-1, 2))
        if rng.rand() < 0.2:
            options["park_ticks"] = int(rng.choice([-1, 0, 130, 160, 256, 20000]))
        if rng.rand() < 0.2:
            options["park_cap"] = float(rng.choice([-1, 0, 0.0625, 0.25, 1.0]))
        if rng.rand() < 0.3:
            options["warp_mode_max"] = int(rng.choice([-1, 0, 10 ** 6, rng.randint(0, 20000)]))
        max_ticks = int(rng.choice([0, 150, 200, 1000, 10000]))
        yield (members.tolist(), work.tolist()), options, max_ticks


def hot_bytes(k, gs):
    nb, nc, nt, _ = emu.classes()[k]
    return emu.lib().rem2d_emu_hot_rows(nb, nc, nt, gs) * 128


def all_cases():
    yield from (((LOADS[p], o, t), name) for name, (p, o, t) in sorted(CASES.items()))
    yield from ((c, "random %d" % i) for i, c in enumerate(random_cases(2000, seed=1)))


def test_plan_properties():
    table = emu.classes()
    for (load, options, max_ticks), name in all_cases():
        members = load[0]
        p = plan(load, options, max_ticks)
        for k, (nb, _, _, table_gs) in enumerate(table):
            gs = p["gs"][k]
            forced = options.get("group_shift", -1)
            forced = forced if forced >= 0 else options.get("class_gs_%d" % k, -1)
            assert 0 <= gs <= 5, name
            assert gs == min(5, forced) if forced >= 0 else gs <= table_gs, name
            if members[k]:
                assert p["grid"][k] >= 1, name
            else:
                assert p["grid"][k] == 0 and p["grid2"][k] == 0, name
            if options.get("overflow_wave", 1) or p["all_fit"]:
                assert (p["grid"][k] + p["grid2"][k]) * (32 >> gs) >= members[k], name
        assert sorted(p["order"]) == list(range(len(table))), name
        smem = [hot_bytes(k, 5 if p["warp_mode"] else p["gs"][k]) for k in p["order"]]
        assert smem == sorted(smem, reverse=True), name
