#!/usr/bin/env python
"""Cost of recording episode statistics (rem2d_set_stats): whole evaluations of the bench population with statistics off and
on, alternating, in one process. Prints creature-steps/s per evaluation, the medians and the relative cost, with the card
name and power limit read in the same run, as JSON (also written to --out). Fitness and lifetimes of the two must be identical.

  python tools/stats_cost.py [--pop 65536] [--rounds 5] [--out FILE]
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


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pop", type=int, default=65536)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    pop = random_population(a.pop, ("lsystem",), seed=2, workers=min(32, os.cpu_count() or 1))
    xs, ys = terrain.generate_terrain()
    engines = {}
    for on in (False, True):
        e = Engine(device=0)
        e.set_terrain(ys, K.TERRAIN_STEP)
        e.set_stats(on)
        e.evaluate(pop, K.EVALUATION_STEPS)          # warm-up: module load, buffers
        engines[on] = e
    rates = {False: [], True: []}
    ref = None
    for r in range(a.rounds):
        for on in ((False, True) if r % 2 == 0 else (True, False)):
            e = engines[on]
            t0 = time.perf_counter()
            f, t = e.evaluate(pop, K.EVALUATION_STEPS)     # returns after the device finished (results copied to the host)
            dt = time.perf_counter() - t0
            if on:
                e.read_stats()
            rates[on].append(float(t.sum()) / dt)
            if ref is None:
                ref = (f, t)
            assert np.array_equal(f, ref[0]) and np.array_equal(t, ref[1]), "statistics changed the results"
    off, on = float(np.median(rates[False])), float(np.median(rates[True]))
    res = {"card": card(), "population": "random_population(%d, ('lsystem',), seed=2), generate_terrain()" % a.pop,
           "rounds": a.rounds, "creature_steps_per_s_off": rates[False], "creature_steps_per_s_on": rates[True],
           "median_off": off, "median_on": on, "cost_percent": 100.0 * (off - on) / off,
           "creature_steps": int(ref[1].sum())}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
