"""ctypes handle on the CPU emulation of the device code of the policy images (tests/emu_policy/librem2d_emu_policy.so: the
harness of tests/emu with -DREM2D_POLICY -DREM2D_STATS). TEST INFRASTRUCTURE ONLY. Outputs are those of tests/emu/emu.py, the
episode statistics included."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

from gym_rem2d_b200 import constants as K
from gym_rem2d_b200.capi import Config, Engine, Population, load_library, N_COUNTERS, COUNTER_NAMES

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "emu"))
from emu import EmuOut, class_of  # noqa: E402,F401

_lib = None


def lib():
    global _lib
    if _lib is None:
        subprocess.check_call(["make", "-s", "-C", HERE])
        L = C.CDLL(os.path.join(HERE, "librem2d_emu_policy.so"))
        common = [C.POINTER(Population), C.c_void_p, C.c_int, C.c_double, C.POINTER(Config), C.c_int, C.c_int, C.c_int, C.c_int]
        policy = [C.c_void_p, C.c_int, C.POINTER(EmuOut)]          # weights, hidden units, outputs
        L.rem2d_emu_policy_step.argtypes = common + [C.c_void_p, C.c_int, C.c_int, C.c_int] + policy
        L.rem2d_emu_policy_queue.argtypes = common + [C.c_int, C.c_void_p, C.c_int, C.c_int] + policy
        _lib = L
    return _lib


def _run(entry, pop, ys, weights, terrain_step, klass, gs, cfg_over, max_pairs, args):
    """Calls `entry` on one warp with the policy `weights` [n_joints of the table, 10 * H + 1]. Every output is indexed like the
    table of `pop`; the entries of creatures the warp did not run keep -1 (NaN for floats)."""
    binder = Engine.__new__(Engine)                      # only for _pop_struct (no native handle)
    s, keep = Engine._pop_struct(binder, pop)
    cfg = Config()
    load_library().rem2d_default_config(C.byref(cfg))
    for k, v in cfg_over.items():
        setattr(cfg, k, v)
    w = np.ascontiguousarray(weights, np.float64)
    n, nb, nj = pop.n_creatures, pop.n_bodies, pop.n_bodies - pop.n_creatures
    shapes = dict(pose=((nb, 3), np.float32), vel=((nb, 3), np.float32), joint_impulse=((nj, 4), np.float32),
                  limit_state=(nj, np.int32), motor_speed=(nj, np.float32), alive=(n, np.int32), ticks=(n, np.int32),
                  fitness=(n, np.float64), wod=(n, np.float64), n_contacts=(n, np.int32), n_touching=(n, np.int32),
                  touching_pairs=((n, max_pairs, 2), np.int32), touching_impulse=((n, max_pairs, 4), np.float32),
                  sched_P=(n, np.int32), sched_smax=(n, np.int32), status=(n, np.int32), finish_gs=(n, np.int32),
                  joint_angle=(nj, np.float32), joint_speed=(nj, np.float32), root=((n, 6), np.float32), ground=(nb, np.int32),
                  end_reason=(n, np.int32), max_x=(n, np.float32), joint_work=(n, np.float64), airborne_ticks=(n, np.int32),
                  ground_ticks=(nb, np.int32))
    st = {k: np.full(shape, np.nan if np.dtype(dt).kind == "f" else -1, dt) for k, (shape, dt) in shapes.items()}
    st.update(counters=np.zeros(N_COUNTERS, np.uint64), n_syncs=np.zeros(1, np.int64), gs_seq=np.zeros(64, np.int32),
              n_seq=np.zeros(1, np.int32))
    o = EmuOut(max_pairs=max_pairs, max_seq=len(st["gs_seq"]))
    for k, a in st.items():
        setattr(o, k, a.ctypes.data)
    ys = np.ascontiguousarray(ys, np.float64)
    rc = getattr(lib(), entry)(C.byref(s), ys.ctypes.data, len(ys), float(terrain_step), C.byref(cfg), klass[0], klass[1], klass[2],
                               gs, *args, w.ctypes.data, (w.shape[1] - 1) // 10, C.byref(o))
    if rc != 0:
        raise RuntimeError("%s failed: %d" % (entry, rc))
    st["counters"] = dict(zip(COUNTER_NAMES, (int(v) for v in st["counters"])))
    st["gs_seq"] = st.pop("gs_seq")[:int(st.pop("n_seq")[0])].tolist()
    return st


def step(pop, ys, creatures, gs, n_ticks, weights, klass=None, n_calls=1, terrain_step=K.TERRAIN_STEP, max_pairs=24, **cfg_over):
    """One emulated warp of step_kernel_policy: `creatures` (<= 32 >> gs) of `pop`, a group of 1 << gs lanes each, reset and
    then n_calls launches of n_ticks ticks. `klass` = (bodies, pool slots, staged contacts); the class of the largest creature
    by default."""
    creatures = np.ascontiguousarray(creatures, np.int32)
    klass = klass or class_of(int(np.diff(pop.body_off)[creatures].max()))
    return _run("rem2d_emu_policy_step", pop, ys, weights, terrain_step, klass, gs, cfg_over, max_pairs,
                (creatures.ctypes.data, len(creatures), int(n_calls), int(n_ticks)))


def queue(pop, ys, order, gs, max_gs, max_ticks, klass, weights, terrain_step=K.TERRAIN_STEP, max_pairs=24, **cfg_over):
    """One emulated warp of the queue-mode policy episode kernel, parking off: the creatures `order` of `pop` are pulled in that
    order by groups of 1 << gs lanes, which widen up to max_gs as the warp drains; gs_seq lists the group shifts it ran at."""
    order = np.ascontiguousarray(order, np.int32)
    return _run("rem2d_emu_policy_queue", pop, ys, weights, terrain_step, klass, gs, cfg_over, max_pairs,
                (int(max_gs), order.ctypes.data, len(order), int(max_ticks)))
