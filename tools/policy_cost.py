#!/usr/bin/env python
"""Cost of the per-joint feedback policy (rem2d_set_policy, include/rem2d_policy.h): whole evaluations of the bench population
in three modes, in alternating blocks in one process: open loop, a zero-weight policy with H = 8 (the same motion as open
loop, so the difference is the policy's overhead alone) and random weights with H = 8. Prints creature-steps/s per evaluation,
the medians and spreads, and the upload time with and without weights, with the card name and power limit read in the same
run, as JSON (also written to --out). The zero-weight policy must reproduce the open-loop fitness and lifetimes.

  python tools/policy_cost.py [--pop 65536] [--rounds 5] [--hidden 8] [--scale 0.1] [--out FILE]
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

from gym_rem2d_b200 import constants as K, policy, terrain  # noqa: E402
from gym_rem2d_b200.capi import Engine  # noqa: E402
from gym_rem2d_b200.population import random_population  # noqa: E402

MODES = ("open_loop", "zero_policy", "random_policy")


def card():
    return subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()


def spread(v):
    return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pop", type=int, default=65536)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--hidden", type=int, default=8)
    ap.add_argument("--scale", type=float, default=0.1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    pop = random_population(a.pop, ("lsystem",), seed=2, workers=min(32, os.cpu_count() or 1))   # the bench population
    xs, ys = terrain.generate_terrain()
    nj = pop.n_bodies - pop.n_creatures
    weights = {"open_loop": None, "zero_policy": np.zeros((nj, policy.n_params(a.hidden))),
               "random_policy": policy.random_weights(nj, a.hidden, a.scale, rng=0)}
    engines, set_ms = {}, {}
    for m in MODES:
        e = Engine(device=0)
        e.set_terrain(ys, K.TERRAIN_STEP)
        if weights[m] is not None:
            t0 = time.perf_counter()
            e.set_policy(weights[m])
            set_ms[m] = 1e3 * (time.perf_counter() - t0)
        e.evaluate(pop, K.EVALUATION_STEPS)          # warm-up: module load, buffers
        engines[m] = e
    rates = {m: [] for m in MODES}
    upload_ms = {"open_loop": [], "zero_policy": []}
    results = {}
    for r in range(a.rounds):
        for m in (MODES if r % 2 == 0 else MODES[::-1]):
            e = engines[m]
            t0 = time.perf_counter()
            f, t = e.evaluate(pop, K.EVALUATION_STEPS)     # returns after the device finished (results copied to the host)
            dt = time.perf_counter() - t0
            rates[m].append(float(t.sum()) / dt)
            results.setdefault(m, (f, t))
            assert np.array_equal(f, results[m][0]) and np.array_equal(t, results[m][1]), "%s is not deterministic" % m
            if m in upload_ms:                              # upload (table + weights snapshot) and world build, synchronised
                t0 = time.perf_counter()
                e.upload(pop)
                e.counters()
                upload_ms[m].append(1e3 * (time.perf_counter() - t0))
    (f0, t0), (fz, tz) = results["open_loop"], results["zero_policy"]
    assert np.array_equal(f0, fz) and np.array_equal(t0, tz), "the zero-weight policy changed the results"
    med = {m: float(np.median(rates[m])) for m in MODES}
    res = {"card": card(), "population": "random_population(%d, ('lsystem',), seed=2), generate_terrain()" % a.pop,
           "n_joints": nj, "hidden": a.hidden, "weights_bytes": int(weights["zero_policy"].nbytes),
           "random_scale": a.scale, "rounds": a.rounds,
           "creature_steps_per_s": {m: rates[m] for m in MODES},
           "creature_steps_per_s_spread": {m: spread(rates[m]) for m in MODES},
           "overhead_percent_zero_policy": 100.0 * (med["open_loop"] - med["zero_policy"]) / med["open_loop"],
           "creature_steps": {m: int(results[m][1].sum()) for m in MODES},
           "upload_ms": {m: spread(v) for m, v in upload_ms.items()}, "set_policy_ms": set_ms}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
