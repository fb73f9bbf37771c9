#!/usr/bin/env python
"""Per-tick cost of closed-loop control (include/rem2d_control.h) against plain stepping, on L-system populations. Plain mode
is step(1) + read_roots per tick; target mode is step_targets(1) + read_observations + read_roots with a trivial numpy policy
(target = -0.5 * joint angle). The two modes run on two engines with the same population, alternating in blocks of 20 one-tick
calls, 200 calls per mode and population; both engines are reset after 100 calls so that most creatures stay ahead of the wall
of death. Reports the device ms per tick (rem2d_last_step_ms: the kernels, plus the copy of the targets in target mode) and
the wall ms per tick of the whole call sequence, with the card name and power limit read in the same run, as JSON (also
written to --out).

  python tools/closed_loop_cost.py [--pops 4096,65536] [--calls 200] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gym_rem2d_b200 import constants as K, terrain  # noqa: E402
from gym_rem2d_b200.capi import Engine  # noqa: E402
from gym_rem2d_b200.population import random_population  # noqa: E402

BLOCK = 20


def card():
    return subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()


def plain_tick(e):
    e.step(1)
    e.read_roots()


def target_tick(e):
    ob = e.read_observations()
    e.step_targets(-0.5 * ob["joint_angle"].astype(np.float64), 1)
    e.read_roots()


def measure(n, calls):
    pop = random_population(n, ("lsystem",), seed=2, workers=min(32, os.cpu_count() or 1))
    xs, ys = terrain.generate_terrain()
    modes = {"plain": plain_tick, "targets": target_tick}
    engines = {}
    for m, fn in modes.items():
        e = Engine(device=0)
        e.set_terrain(ys, K.TERRAIN_STEP)
        e.upload(pop)
        for _ in range(BLOCK):                     # warm-up: module load, buffers
            fn(e)
        e.reset()
        engines[m] = e
    dev = {m: [] for m in modes}
    wall = {m: [] for m in modes}
    for b in range(calls // BLOCK):
        if b * BLOCK == calls // 2:
            for e in engines.values():
                e.reset()
        for m in (("plain", "targets") if b % 2 == 0 else ("targets", "plain")):
            e, fn = engines[m], modes[m]
            t0 = time.perf_counter()
            for _ in range(BLOCK):
                fn(e)
                dev[m].append(e.last_step_ms())
            wall[m].append((time.perf_counter() - t0) * 1e3 / BLOCK)       # every call ends in a device synchronise
    res = {"population": "random_population(%d, ('lsystem',), seed=2), generate_terrain()" % n, "n_creatures": n,
           "n_joints": int(pop.n_bodies - pop.n_creatures), "calls_per_mode": calls}
    for m in modes:
        res[m] = {"device_ms_per_tick_median": float(np.median(dev[m])), "device_ms_per_tick_mean": float(np.mean(dev[m])),
                  "wall_ms_per_tick_median": float(np.median(wall[m])), "wall_ms_per_tick_mean": float(np.mean(wall[m])),
                  "wall_ms_per_tick_blocks": wall[m]}
    res["wall_ratio_targets_over_plain"] = res["targets"]["wall_ms_per_tick_median"] / res["plain"]["wall_ms_per_tick_median"]
    res["device_ratio_targets_over_plain"] = res["targets"]["device_ms_per_tick_median"] / res["plain"]["device_ms_per_tick_median"]
    for e in engines.values():
        e.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pops", default="4096,65536")
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"card": card(), "policy": "target = -0.5 * joint_angle (numpy, float64)",
           "results": [measure(int(n), a.calls) for n in a.pops.split(",")]}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
