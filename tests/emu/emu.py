"""ctypes handle on the CPU emulation of the CUDA device code (tests/emu: librem2d_emu.so, and librem2d_emu_stats.so /
librem2d_emu_targets.so for the statistics and joint-target variants). TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os
import subprocess

import numpy as np

from gym_rem2d_b200 import constants as K
from gym_rem2d_b200.capi import Config, Engine, Population, load_library, N_COUNTERS, COUNTER_NAMES

HERE = os.path.dirname(os.path.abspath(__file__))
VARIANTS = {"plain": "librem2d_emu.so", "stats": "librem2d_emu_stats.so", "targets": "librem2d_emu_targets.so"}
STATS = ("end_reason", "max_x", "joint_work", "airborne_ticks", "ground_ticks")
OBS = ("joint_angle", "joint_speed", "root", "ground")


class EmuOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("pose", "vel", "joint_impulse", "limit_state", "motor_speed", "alive", "ticks", "fitness",
                                          "wod", "n_contacts", "n_touching", "touching_pairs", "touching_impulse", "sched_P",
                                          "sched_smax", "counters", "n_syncs", "status", "finish_gs", "gs_seq", "n_seq") + OBS + STATS] + \
               [("max_pairs", C.c_int32), ("max_seq", C.c_int32)]


_libs = {}


def lib(variant="plain"):
    if variant not in _libs:
        subprocess.check_call(["make", "-s", "-C", HERE, VARIANTS[variant]])
        L = C.CDLL(os.path.join(HERE, VARIANTS[variant]))
        common = [C.POINTER(Population), C.c_void_p, C.c_int, C.c_double, C.POINTER(Config), C.c_int, C.c_int, C.c_int, C.c_int]
        L.rem2d_emu_step.argtypes = common + [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(EmuOut)]
        L.rem2d_emu_queue.argtypes = common + [C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(EmuOut)]
        L.rem2d_emu_classes.argtypes = [C.c_void_p]
        L.rem2d_emu_plan.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        _libs[variant] = L
    return _libs[variant]


_classes = None


def classes():
    """The capacity classes of the CUDA library: (bodies, contact-pool slots, staged touching contacts, widest group shift)."""
    global _classes
    if _classes is None:
        out = np.zeros((64, 4), np.int32)
        n = lib().rem2d_emu_classes(out.ctypes.data)
        _classes = [tuple(int(v) for v in row) for row in out[:n]]
    return _classes


def class_of(nb):
    for cl in classes():
        if nb <= cl[0]:
            return cl
    raise ValueError(nb)


# the Options fields the planner reads, in the order rem2d_emu_plan takes them (rem2d_set_option names)
PLAN_OPTIONS = ("warp_mode_max", "park_ticks", "park_cap", "overflow_wave", "image", "smem_budget_kb", "group_shift")


def plan(members, work, options=None, max_ticks=10000, n_sms=148, max_warps_per_sm=(9, 16)):
    """The CUDA library's episode plan for a population with `members` creatures and a cost estimate of `work` per capacity
    class, on `n_sms` SMs with `max_warps_per_sm` resident warps per SM for the two kernel images, with the planner options
    `options` (a dict: PLAN_OPTIONS and "class_gs_<k>"; the library's defaults for the rest)."""
    L, n = lib(), len(classes())
    members, work = np.ascontiguousarray(members, np.int32), np.ascontiguousarray(work, np.float64)
    assert members.shape == (n,) and work.shape == (n,)
    warps = np.ascontiguousarray(max_warps_per_sm, np.int32)
    names = PLAN_OPTIONS + tuple("class_gs_%d" % k for k in range(n))
    unknown = set(options or {}) - set(names)
    if unknown:
        raise ValueError("not a planner option: %s" % sorted(unknown))
    opt = np.array([(options or {}).get(k, np.nan) for k in names], np.float64)
    out = np.zeros(4 + 6 * n, np.int32)
    L.rem2d_emu_plan(n_sms, warps.ctypes.data, members.ctypes.data, work.ctypes.data, opt.ctypes.data, int(max_ticks),
                     out.ctypes.data)
    cols = out[4:].reshape(6, n)
    return dict(image=int(out[0]), all_fit=bool(out[1]), warp_mode=bool(out[2]), park_ticks=int(out[3]),
                **{k: cols[i].tolist() for i, k in enumerate(("gs", "grid", "grid2", "park_cap", "order", "step_gs"))})


def _run(entry, variant, pop, ys, terrain_step, klass, gs, cfg_over, max_pairs, args):
    """Calls `entry` of the `variant` library on one warp. Every output is indexed like the table of `pop` (creature, body,
    joint); the entries of creatures the warp did not run keep -1 (NaN for floats)."""
    binder = Engine.__new__(Engine)                      # only for _pop_struct (no native handle)
    s, keep = Engine._pop_struct(binder, pop)
    cfg = Config()
    load_library().rem2d_default_config(C.byref(cfg))
    for k, v in cfg_over.items():
        setattr(cfg, k, v)
    n, nb, nj = pop.n_creatures, pop.n_bodies, pop.n_bodies - pop.n_creatures
    shapes = dict(pose=((nb, 3), np.float32), vel=((nb, 3), np.float32), joint_impulse=((nj, 4), np.float32),
                  limit_state=(nj, np.int32), motor_speed=(nj, np.float32), alive=(n, np.int32), ticks=(n, np.int32),
                  fitness=(n, np.float64), wod=(n, np.float64), n_contacts=(n, np.int32), n_touching=(n, np.int32),
                  touching_pairs=((n, max_pairs, 2), np.int32), touching_impulse=((n, max_pairs, 4), np.float32),
                  sched_P=(n, np.int32), sched_smax=(n, np.int32), status=(n, np.int32), finish_gs=(n, np.int32),
                  joint_angle=(nj, np.float32), joint_speed=(nj, np.float32), root=((n, 6), np.float32), ground=(nb, np.int32))
    if variant == "stats":
        shapes.update(end_reason=(n, np.int32), max_x=(n, np.float32), joint_work=(n, np.float64), airborne_ticks=(n, np.int32),
                      ground_ticks=(nb, np.int32))
    st = {k: np.full(shape, np.nan if np.dtype(dt).kind == "f" else -1, dt) for k, (shape, dt) in shapes.items()}
    st.update(counters=np.zeros(N_COUNTERS, np.uint64), n_syncs=np.zeros(1, np.int64), gs_seq=np.zeros(64, np.int32),
              n_seq=np.zeros(1, np.int32))
    o = EmuOut(max_pairs=max_pairs, max_seq=len(st["gs_seq"]))
    for k, a in st.items():
        setattr(o, k, a.ctypes.data)
    ys = np.ascontiguousarray(ys, np.float64)
    rc = getattr(lib(variant), entry)(C.byref(s), ys.ctypes.data, len(ys), float(terrain_step), C.byref(cfg), klass[0], klass[1],
                                      klass[2], gs, *args, C.byref(o))
    if rc != 0:
        raise RuntimeError("%s (%s) failed: %d" % (entry, variant, rc))
    st["counters"] = dict(zip(COUNTER_NAMES, (int(v) for v in st["counters"])))
    st["gs_seq"] = st.pop("gs_seq")[:int(st.pop("n_seq")[0])].tolist()
    return st


def step(pop, ys, creatures, gs, n_ticks, variant="plain", targets=None, klass=None, terrain_step=K.TERRAIN_STEP, max_pairs=24,
         **cfg_over):
    """One emulated warp of the stepping kernel: `creatures` (<= 32 >> gs) of `pop`, a group of 1 << gs lanes each, reset and
    then n_ticks ticks. variant "targets" takes targets[n_calls, n_joints of the table]: call i holds targets[i] for n_ticks
    ticks, as rem2d_step_targets does. `klass` = (bodies, pool slots, staged contacts); the class of the largest creature by
    default."""
    creatures = np.ascontiguousarray(creatures, np.int32)
    klass = klass or class_of(int(np.diff(pop.body_off)[creatures].max()))
    n_calls, t = 1, None
    if targets is not None:
        t = np.ascontiguousarray(targets, np.float64)
        n_calls = len(t)
    return _run("rem2d_emu_step", variant, pop, ys, terrain_step, klass, gs, cfg_over, max_pairs,
                (creatures.ctypes.data, len(creatures), None if t is None else t.ctypes.data, n_calls, int(n_ticks)))


def queue(pop, ys, order, gs, max_gs, max_ticks, klass, variant="plain", terrain_step=K.TERRAIN_STEP, max_pairs=24, **cfg_over):
    """One emulated warp of the queue-mode episode kernel, parking off: the creatures `order` of `pop` are pulled in that order
    by groups of 1 << gs lanes, which widen up to max_gs as the warp drains. Each creature's outputs are its state at the end of
    its episode; gs_seq lists the group shifts the warp ran at."""
    order = np.ascontiguousarray(order, np.int32)
    return _run("rem2d_emu_queue", variant, pop, ys, terrain_step, klass, gs, cfg_over, max_pairs,
                (int(max_gs), order.ctypes.data, len(order), int(max_ticks)))
