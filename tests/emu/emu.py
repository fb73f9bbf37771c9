"""ctypes handle on the CPU emulation of the CUDA device code (tests/emu/librem2d_emu.so). TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os
import subprocess

import numpy as np

from gym_rem2d_b200.capi import Config, Engine, Population, load_library, N_COUNTERS, COUNTER_NAMES

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "librem2d_emu.so")


class EmuOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("pose", "vel", "joint_impulse", "limit_state", "motor_speed", "alive", "ticks", "fitness",
                                          "wod", "n_contacts", "n_touching", "touching_pairs", "touching_impulse")] + \
               [("max_pairs", C.c_int32), ("sched_P", C.c_void_p), ("sched_smax", C.c_void_p), ("counters", C.c_void_p),
                ("n_syncs", C.c_void_p)]


def build():
    subprocess.check_call(["make", "-s", "-C", HERE])
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.rem2d_emu_run.argtypes = [C.POINTER(Population), C.c_void_p, C.c_int, C.c_double, C.POINTER(Config), C.c_int, C.c_int,
                                       C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(EmuOut)]
        _lib.rem2d_emu_classes.argtypes = [C.c_void_p]
        _lib.rem2d_emu_plan.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    return _lib


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


def run(pop, ys, step, creatures, gs, n_ticks, max_pairs=24, klass=None, **cfg_over):
    """One emulated warp: `creatures` (<= 32 >> gs) of `pop`, reset + n_ticks ticks with groups of 1 << gs lanes."""
    L = lib()
    binder = Engine.__new__(Engine)                      # only for _pop_struct (no native handle)
    s, keep = Engine._pop_struct(binder, pop)
    cfg = Config()
    load_library().rem2d_default_config(C.byref(cfg))
    for k, v in cfg_over.items():
        setattr(cfg, k, v)
    creatures = np.ascontiguousarray(creatures, np.int32)
    nbs = np.diff(pop.body_off)[creatures]
    klass = klass or class_of(int(nbs.max()))
    n, nb, nj = len(creatures), int(nbs.sum()), int(nbs.sum()) - len(creatures)
    ys = np.ascontiguousarray(ys, np.float64)
    st = dict(pose=np.zeros((nb, 3), np.float32), vel=np.zeros((nb, 3), np.float32), joint_impulse=np.zeros((nj, 4), np.float32),
              limit_state=np.zeros(nj, np.int32), motor_speed=np.zeros(nj, np.float32), alive=np.zeros(n, np.int32),
              ticks=np.zeros(n, np.int32), fitness=np.zeros(n, np.float64), wod=np.zeros(n, np.float64),
              n_contacts=np.zeros(n, np.int32), n_touching=np.zeros(n, np.int32),
              touching_pairs=np.full((n, max_pairs, 2), -1, np.int32), touching_impulse=np.zeros((n, max_pairs, 4), np.float32),
              sched_P=np.zeros(n, np.int32), sched_smax=np.zeros(n, np.int32), counters=np.zeros(N_COUNTERS, np.uint64),
              n_syncs=np.zeros(1, np.int64))
    o = EmuOut()
    for k, a in st.items():
        setattr(o, k, a.ctypes.data)
    o.max_pairs = max_pairs
    rc = L.rem2d_emu_run(C.byref(s), ys.ctypes.data, len(ys), float(step), C.byref(cfg), klass[0], klass[1], klass[2], gs,
                         creatures.ctypes.data, n, int(n_ticks), C.byref(o))
    if rc != 0:
        raise RuntimeError("rem2d_emu_run failed: %d" % rc)
    st["counters"] = dict(zip(COUNTER_NAMES, (int(v) for v in st["counters"])))
    return st
