"""ctypes binding of the C-ABI declared in include/rem2d.h.

The product library is ``csrc/librem2d_cuda.so`` (hand-written CUDA for sm_100a). There is NO CPU
fallback: if the library is missing, or no CUDA device is usable, loading/creating raises.
The binding class itself is library-agnostic because the CPU oracle exports the same ABI; only the
tests point it at the oracle's shared object (see oracle/oracle.py) — nothing in this package does.
"""
import ctypes as C
import os

import numpy as np

# The library runs one stream per capacity class (+ one per tail-mode launch); with the default 8 hardware queues, streams
# alias and stream-waits block unrelated launches. Must be set before the CUDA context exists.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

HERE = os.path.dirname(os.path.abspath(__file__))
CUDA_LIB = os.environ.get("REM2D_CUDA_LIB") or os.path.join(HERE, "csrc", "librem2d_cuda.so")   # env override: A/B builds
# optional build with fused multiply-adds (`make -C gym_rem2d_b200/csrc fast`): NOT bit-identical to the oracle, fitness distribution
# unchanged (KS 0.002), 1.06x on the bench population (profiles/r2_fma.txt). Engine(precision="fast") selects it; default = exact.
CUDA_LIB_FAST = os.path.join(HERE, "csrc", "librem2d_cuda_fma.so")

N_COUNTERS = 12
COUNTER_NAMES = ["ticks", "body_ticks", "joint_vsolves", "p1_vsolves", "m2_vsolves", "joint_psolves",
                 "point_psolves", "narrow", "toi_calls", "toi_events", "gjk_iters", "toi_root_iters"]


class Config(C.Structure):
    _fields_ = [("dt", C.c_float), ("velocity_iterations", C.c_int32), ("position_iterations", C.c_int32),
                ("gravity_y", C.c_float), ("module_friction", C.c_float), ("terrain_friction", C.c_float),
                ("p_gain", C.c_double), ("wod_speed", C.c_double), ("env_length", C.c_double),
                ("evaluation_steps", C.c_int32), ("continuous", C.c_int32), ("allow_sleep", C.c_int32),
                ("terminate", C.c_int32), ("device", C.c_int32), ("stream", C.c_void_p),
                ("sincos_mode", C.c_int32), ("reserved", C.c_int32)]


class Population(C.Structure):
    _fields_ = [("n_creatures", C.c_int32), ("n_bodies", C.c_int32), ("n_joints", C.c_int32),
                ("body_off", C.c_void_p), ("shape", C.c_void_p), ("hx", C.c_void_p), ("hy", C.c_void_p),
                ("x0", C.c_void_p), ("y0", C.c_void_p), ("a0", C.c_void_p), ("joint_parent", C.c_void_p),
                ("anchor_a", C.c_void_p), ("anchor_b", C.c_void_p), ("lower", C.c_void_p), ("upper", C.c_void_p),
                ("max_torque", C.c_void_p), ("ctrl", C.c_void_p)]


class StateView(C.Structure):
    _fields_ = [("pose", C.c_void_p), ("vel", C.c_void_p), ("joint_impulse", C.c_void_p),
                ("limit_state", C.c_void_p), ("motor_speed", C.c_void_p), ("alive", C.c_void_p), ("ticks", C.c_void_p), ("awake", C.c_void_p),
                ("wod", C.c_void_p), ("n_contacts", C.c_void_p), ("n_touching", C.c_void_p),
                ("touching_pairs", C.c_void_p), ("touching_impulse", C.c_void_p), ("max_pairs", C.c_int32),
                ("reserved", C.c_int32)]


class EpisodeStats(C.Structure):
    _fields_ = [("end_reason", C.c_void_p), ("max_x", C.c_void_p), ("joint_work", C.c_void_p),
                ("airborne_ticks", C.c_void_p), ("ground_ticks", C.c_void_p)]


# rem2d_episode_stats.end_reason values (include/rem2d_stats.h)
END_RUNNING, END_ORIGIN, END_WALL, END_GOAL, END_STEPS = 0, 1, 2, 3, 4
END_REASONS = {END_RUNNING: "running", END_ORIGIN: "origin", END_WALL: "wall", END_GOAL: "goal", END_STEPS: "steps"}


class Observation(C.Structure):
    _fields_ = [("joint_angle", C.c_void_p), ("joint_speed", C.c_void_p), ("root", C.c_void_p), ("ground", C.c_void_p)]


class Rem2dError(RuntimeError):
    pass


_LIBS = {}


def load_library(path=None):
    path = path or CUDA_LIB
    if path in _LIBS:
        return _LIBS[path]
    if not os.path.exists(path):
        raise Rem2dError(
            "rem2d: native library %s is missing — build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)" % path)
    lib = C.CDLL(path)
    H = C.c_void_p
    lib.rem2d_default_config.argtypes = [C.POINTER(Config)]
    lib.rem2d_default_config.restype = None
    lib.rem2d_abi_version.restype = C.c_int
    lib.rem2d_backend.restype = C.c_char_p
    lib.rem2d_create.argtypes = [C.POINTER(Config), C.POINTER(H)]
    lib.rem2d_destroy.argtypes = [H]
    lib.rem2d_last_error.argtypes = [H]
    lib.rem2d_last_error.restype = C.c_char_p
    lib.rem2d_set_terrain.argtypes = [H, C.c_void_p, C.c_int32, C.c_double]
    lib.rem2d_upload.argtypes = [H, C.POINTER(Population)]
    lib.rem2d_reset.argtypes = [H]
    lib.rem2d_step.argtypes = [H, C.c_int32]
    lib.rem2d_read_state.argtypes = [H, C.POINTER(StateView)]
    lib.rem2d_fitness.argtypes = [H, C.c_void_p]
    lib.rem2d_get_counters.argtypes = [H, C.c_void_p]
    lib.rem2d_evaluate.argtypes = [H, C.POINTER(Population), C.c_int32, C.c_void_p, C.c_void_p]
    lib.rem2d_run_episodes.argtypes = [H, C.c_int32]
    lib.rem2d_ticks.argtypes = [H, C.c_void_p]
    lib.rem2d_last_step_ms.argtypes = [H]
    lib.rem2d_last_step_ms.restype = C.c_float
    lib.rem2d_measure_fp32_peak.argtypes = [H, C.POINTER(C.c_double)]
    lib.rem2d_launch_count.argtypes = [H]
    lib.rem2d_launch_count.restype = C.c_int64
    lib.rem2d_set_option.argtypes = [H, C.c_char_p, C.c_double]
    lib.rem2d_read_roots.argtypes = [H, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rem2d_set_priority.argtypes = [H, C.c_void_p, C.c_int32]
    if hasattr(lib, "rem2d_read_stats"):          # the episode statistics extension (include/rem2d_stats.h)
        lib.rem2d_set_stats.argtypes = [H, C.c_int32]
        lib.rem2d_read_stats.argtypes = [H, C.POINTER(EpisodeStats)]
    if hasattr(lib, "rem2d_step_targets"):        # the closed-loop control extension (include/rem2d_control.h)
        lib.rem2d_step_targets.argtypes = [H, C.c_void_p, C.c_int32]
        lib.rem2d_read_observations.argtypes = [H, C.POINTER(Observation)]
    if hasattr(lib, "rem2d_set_policy"):          # the feedback policy extension (include/rem2d_policy.h)
        lib.rem2d_set_policy.argtypes = [H, C.c_void_p, C.c_int32, C.c_int32]
    _LIBS[path] = lib
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Engine:
    """One handle (= one device). Thin, explicit wrapper: every method is one C-ABI call."""

    def __init__(self, lib_path=None, device=0, stream=None, precision="exact", **overrides):
        if precision not in ("exact", "fast"):
            raise ValueError("precision must be 'exact' (bit-identical to the oracle) or 'fast' (fused multiply-adds)")
        if lib_path is None and precision == "fast":
            lib_path = CUDA_LIB_FAST
        self.precision = precision
        self.lib = load_library(lib_path)
        self.cfg = Config()
        self.lib.rem2d_default_config(C.byref(self.cfg))
        self.cfg.device = device
        self.cfg.stream = stream
        for k, v in overrides.items():
            if not hasattr(self.cfg, k):
                raise TypeError("unknown config field %r" % k)
            setattr(self.cfg, k, v)
        self.h = C.c_void_p()
        rc = self.lib.rem2d_create(C.byref(self.cfg), C.byref(self.h))
        if rc != 0:
            msg = self.lib.rem2d_last_error(None)
            raise Rem2dError("rem2d_create failed (%d): %s" % (rc, msg.decode() if msg else "?"))
        self.pop = None
        self._keep = None

    @property
    def backend(self):
        return self.lib.rem2d_backend().decode()

    def _check(self, rc, what):
        if rc != 0:
            msg = self.lib.rem2d_last_error(self.h)
            raise Rem2dError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.rem2d_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_terrain(self, ys, step):
        ys = np.ascontiguousarray(ys, dtype=np.float64)
        self._check(self.lib.rem2d_set_terrain(self.h, _ptr(ys), len(ys), float(step)), "rem2d_set_terrain")

    def _pop_struct(self, pop):
        arrs = dict(
            body_off=np.ascontiguousarray(pop.body_off, np.int32), shape=np.ascontiguousarray(pop.shape, np.uint8),
            hx=np.ascontiguousarray(pop.hx, np.float32), hy=np.ascontiguousarray(pop.hy, np.float32),
            x0=np.ascontiguousarray(pop.x0, np.float32), y0=np.ascontiguousarray(pop.y0, np.float32),
            a0=np.ascontiguousarray(pop.a0, np.float32), joint_parent=np.ascontiguousarray(pop.joint_parent, np.int16),
            anchor_a=np.ascontiguousarray(pop.anchor_a, np.float32), anchor_b=np.ascontiguousarray(pop.anchor_b, np.float32),
            lower=np.ascontiguousarray(pop.lower, np.float32), upper=np.ascontiguousarray(pop.upper, np.float32),
            max_torque=np.ascontiguousarray(pop.max_torque, np.float32), ctrl=np.ascontiguousarray(pop.ctrl, np.float64))
        s = Population()
        s.n_creatures = pop.n_creatures
        s.n_bodies = pop.n_bodies
        s.n_joints = pop.n_bodies - pop.n_creatures
        for k, a in arrs.items():
            setattr(s, k, a.ctypes.data)
        return s, arrs

    def upload(self, pop):
        s, keep = self._pop_struct(pop)
        self._check(self.lib.rem2d_upload(self.h, C.byref(s)), "rem2d_upload")
        self.pop = pop

    def reset(self):
        self._check(self.lib.rem2d_reset(self.h), "rem2d_reset")

    def step(self, n_ticks=1):
        self._check(self.lib.rem2d_step(self.h, int(n_ticks)), "rem2d_step")

    def run_episodes(self, max_ticks):
        """Whole episodes of the uploaded population from tick 0 (persistent episode kernel on the GPU)."""
        self._check(self.lib.rem2d_run_episodes(self.h, int(max_ticks)), "rem2d_run_episodes")

    def ticks(self):
        out = np.zeros(self.pop.n_creatures, np.int32)
        self._check(self.lib.rem2d_ticks(self.h, _ptr(out)), "rem2d_ticks")
        return out

    def fitness(self):
        out = np.zeros(self.pop.n_creatures, np.float64)
        self._check(self.lib.rem2d_fitness(self.h, _ptr(out)), "rem2d_fitness")
        return out

    def counters(self):
        out = np.zeros(N_COUNTERS, np.uint64)
        self._check(self.lib.rem2d_get_counters(self.h, _ptr(out)), "rem2d_get_counters")
        return dict(zip(COUNTER_NAMES, (int(v) for v in out)))

    def evaluate(self, pop, max_ticks):
        """Batched evaluate(): host table in, (fitness float64[n], ticks int32[n]) out."""
        s, keep = self._pop_struct(pop)
        fit = np.zeros(pop.n_creatures, np.float64)
        ticks = np.zeros(pop.n_creatures, np.int32)
        self._check(self.lib.rem2d_evaluate(self.h, C.byref(s), int(max_ticks), _ptr(fit), _ptr(ticks)), "rem2d_evaluate")
        self.pop = pop
        return fit, ticks

    def last_step_ms(self):
        return float(self.lib.rem2d_last_step_ms(self.h))

    def measure_fp32_peak(self):
        """GFLOP/s of non-fused FP32 multiply/add issue on this device (CUDA build only)."""
        v = C.c_double(0.0)
        self._check(self.lib.rem2d_measure_fp32_peak(self.h, C.byref(v)), "rem2d_measure_fp32_peak")
        return v.value

    def launch_count(self):
        return int(self.lib.rem2d_launch_count(self.h))

    def set_option(self, name, value):
        """Execution-strategy option (never changes results): see include/rem2d.h, rem2d_set_option."""
        self._check(self.lib.rem2d_set_option(self.h, name.encode(), float(value)), "rem2d_set_option(%s)" % name)

    def set_priority(self, expected_ticks):
        """Scheduling hint for the next upload / evaluate: expected lifetime per creature (None clears). Never changes results."""
        if expected_ticks is None:
            self._check(self.lib.rem2d_set_priority(self.h, None, 0), "rem2d_set_priority")
            return
        a = np.ascontiguousarray(expected_ticks, np.float32)
        self._check(self.lib.rem2d_set_priority(self.h, _ptr(a), len(a)), "rem2d_set_priority")

    def read_roots(self):
        """(root x float32[n], wall-of-death position float64[n], alive int32[n]) — what a step-wise driver needs per tick."""
        n = self.pop.n_creatures
        x, wod, alive = np.zeros(n, np.float32), np.zeros(n, np.float64), np.zeros(n, np.int32)
        self._check(self.lib.rem2d_read_roots(self.h, _ptr(x), _ptr(wod), _ptr(alive)), "rem2d_read_roots")
        return x, wod, alive

    def read_state(self, max_pairs=0):
        pop = self.pop
        nb, nj, nc = pop.n_bodies, pop.n_bodies - pop.n_creatures, pop.n_creatures
        st = dict(pose=np.zeros((nb, 3), np.float32), vel=np.zeros((nb, 3), np.float32),
                  joint_impulse=np.zeros((nj, 4), np.float32), limit_state=np.zeros(nj, np.int32),
                  motor_speed=np.zeros(nj, np.float32),
                  alive=np.zeros(nc, np.int32), ticks=np.zeros(nc, np.int32), awake=np.zeros(nc, np.int32),
                  wod=np.zeros(nc, np.float64), n_contacts=np.zeros(nc, np.int32), n_touching=np.zeros(nc, np.int32))
        if max_pairs > 0:
            st["touching_pairs"] = np.full((nc, max_pairs, 2), -1, np.int32)
            st["touching_impulse"] = np.zeros((nc, max_pairs, 4), np.float32)
        v = StateView()
        for k, a in st.items():
            setattr(v, k, a.ctypes.data)
        v.max_pairs = max_pairs
        self._check(self.lib.rem2d_read_state(self.h, C.byref(v)), "rem2d_read_state")
        return st

    def _require_stats(self):
        if not hasattr(self.lib, "rem2d_read_stats"):
            raise Rem2dError("%s does not record episode statistics (include/rem2d_stats.h)" % self.backend)

    def set_stats(self, on=True):
        """Record episode statistics in the whole-episode runs of every later upload / evaluate (never changes results)."""
        self._require_stats()
        self._check(self.lib.rem2d_set_stats(self.h, 1 if on else 0), "rem2d_set_stats")

    def read_stats(self):
        """Episode statistics of the last run_episodes / evaluate of a population uploaded with set_stats(True): a dict of
        end_reason int32[n] (END_*), max_x float32[n], joint_work float64[n], airborne_ticks int32[n] and ground_ticks
        int32[n_bodies] (aligned with the table's bodies). Definitions: include/rem2d_stats.h."""
        self._require_stats()
        pop = self.pop
        if pop is None:
            raise Rem2dError("rem2d_read_stats: no population uploaded")
        nc, nb = pop.n_creatures, pop.n_bodies
        st = dict(end_reason=np.zeros(nc, np.int32), max_x=np.zeros(nc, np.float32), joint_work=np.zeros(nc, np.float64),
                  airborne_ticks=np.zeros(nc, np.int32), ground_ticks=np.zeros(nb, np.int32))
        v = EpisodeStats()
        for k, a in st.items():
            setattr(v, k, a.ctypes.data)
        self._check(self.lib.rem2d_read_stats(self.h, C.byref(v)), "rem2d_read_stats")
        return st

    def _require_control(self):
        if not hasattr(self.lib, "rem2d_step_targets"):
            raise Rem2dError("%s does not take joint targets (include/rem2d_control.h)" % self.backend)

    def step_targets(self, targets, n_ticks=1):
        """Advances every living creature by up to ``n_ticks`` ticks with the P-controller driven to ``targets`` (float64
        [n_joints], target angles in radians in table order, held for all ticks) instead of the sine controllers, which are
        not advanced. Semantics: include/rem2d_control.h."""
        self._require_control()
        if self.pop is None:
            raise Rem2dError("rem2d_step_targets: no population uploaded")
        nj = self.pop.n_bodies - self.pop.n_creatures
        t = np.ascontiguousarray(targets, np.float64)
        if t.shape != (nj,):
            raise ValueError("targets must have shape (%d,) (one per joint), got %s" % (nj, t.shape))
        self._check(self.lib.rem2d_step_targets(self.h, _ptr(t), int(n_ticks)), "rem2d_step_targets")

    def read_observations(self):
        """End-of-tick observations of the uploaded population: a dict of joint_angle float32[n_joints] (the angle the next
        tick's P-controller uses), joint_speed float32[n_joints], root float32[n, 6] (x, y, angle, vx, vy, omega of body 0)
        and ground int32[n_bodies] (1: touching terrain). Definitions: include/rem2d_control.h."""
        self._require_control()
        pop = self.pop
        if pop is None:
            raise Rem2dError("rem2d_read_observations: no population uploaded")
        nc, nb = pop.n_creatures, pop.n_bodies
        ob = dict(joint_angle=np.zeros(nb - nc, np.float32), joint_speed=np.zeros(nb - nc, np.float32),
                  root=np.zeros((nc, 6), np.float32), ground=np.zeros(nb, np.int32))
        v = Observation()
        for k, a in ob.items():
            setattr(v, k, a.ctypes.data)
        self._check(self.lib.rem2d_read_observations(self.h, C.byref(v)), "rem2d_read_observations")
        return ob

    def set_policy(self, weights):
        """Per-joint feedback policy for every later upload / evaluate (include/rem2d_policy.h): float64 weights of shape
        (n_joints, 10 * H + 1), a numpy array or a CPU tensor, one row per joint in table order (gym_rem2d_b200.policy); None
        clears it. The upload takes a snapshot; an upload with another joint count is refused while a policy is set."""
        if not hasattr(self.lib, "rem2d_set_policy"):
            raise Rem2dError("%s does not run feedback policies (include/rem2d_policy.h)" % self.backend)
        if weights is None:
            self._check(self.lib.rem2d_set_policy(self.h, None, 0, 0), "rem2d_set_policy")
            return
        from .policy import hidden_size
        if hasattr(weights, "detach"):                # torch tensor: host memory only
            if weights.device.type != "cpu":
                raise ValueError("policy weights must be on the host (a numpy array or a CPU tensor)")
            weights = weights.detach().numpy()
        w = np.ascontiguousarray(weights, np.float64)
        if w.ndim != 2:
            raise ValueError("policy weights must have shape (n_joints, 10 * H + 1), got %s" % (w.shape,))
        H = hidden_size(w.shape[1])
        self._check(self.lib.rem2d_set_policy(self.h, _ptr(w), w.shape[0], H), "rem2d_set_policy")
