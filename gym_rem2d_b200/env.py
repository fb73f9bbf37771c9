"""Host-side mirror of the reference's evaluation interface, backed by the CUDA library.

Reference interface kept (paths under /root/reference/ModularER_2D):
  * ``Modular2D`` env: ``seed / reset(tree=, module_list=) / step(action) -> (0, reward, done, 0) /
    render / close`` (gym_rem2D/envs/Modular2DEnv.py:127-773, registered as Modular2DLocomotion-v0 in
    gym_rem2D/__init__.py:5-7). ``ModularEnv`` is an alias (BASELINE north_star naming).
  * ``evaluate(individual, EVALUATION_STEPS=10000, HEADLESS=True, INTERVAL=100, ENV_LENGTH=100,
    TREE_DEPTH=None, CONTROLLER=None) -> float``  (REM2D_main.py:350-378).
New, batched entry points: ``BatchedModular2D`` and ``evaluate_population`` — what
``toolbox.map(toolbox.evaluate, population)`` (REM2D_main.py:267,291) becomes.
All physics runs in csrc/librem2d_cuda.so; there is no CPU path here.
"""
import numpy as np

from . import constants as K
from . import terrain as _terrain
from .capi import Engine
from .flatten import flatten_population, flatten_tree, pack


class _Box:
    """Minimal stand-in for gym.spaces.Box (gym is not a dependency)."""

    def __init__(self, low, high, dtype=np.float32):
        self.low = np.asarray(low, dtype=dtype)
        self.high = np.asarray(high, dtype=dtype)
        self.shape = self.low.shape
        self.dtype = dtype

    def sample(self):
        return np.random.uniform(np.maximum(self.low, -1e6), np.minimum(self.high, 1e6)).astype(self.dtype)


class BatchedModular2D:
    """A whole population of creatures, each in its own world, stepped together on one GPU. With ``stats=True`` every
    ``evaluate`` also leaves the episode statistics of the population in ``last_stats`` (``Engine.read_stats``)."""

    def __init__(self, device=0, stream=None, max_perturbance=K.MAX_PERTURBANCE_TERRAIN, lib_path=None, precision="exact", stats=False,
                 **config):
        self.engine = Engine(lib_path=lib_path, device=device, stream=stream, precision=precision, **config)
        self.max_perturbance = max_perturbance
        self.table = None
        self.stats = bool(stats)
        self._engine_stats = False
        self._engine_policy = False
        self.last_stats = None
        self.seed(K.TERRAIN_SEED)

    def seed(self, seed=None):
        """Regenerates the terrain like ``Modular2D.seed`` + ``_generate_terrain`` (Modular2DEnv.py:171,188)."""
        self._seed = K.TERRAIN_SEED if seed is None else seed
        self.terrain_x, self.terrain_y = _terrain.generate_terrain(self._seed, self.max_perturbance)
        self.engine.set_terrain(self.terrain_y, K.TERRAIN_STEP)
        return [self._seed]

    def _set_policy(self, policy):
        """The policy of the next upload: the given weights, or none (open loop), clearing one set by an earlier call."""
        if policy is not None or self._engine_policy:
            self.engine.set_policy(policy)
            self._engine_policy = policy is not None

    def reset(self, individuals=None, table=None, tree_depth=None, policy=None):
        """Builds one world per individual (genome.create -> flatten -> upload). ``policy``: float64 weights of a per-joint
        feedback policy, shape (n_joints, 10 * H + 1) (``Engine.set_policy``; gym_rem2d_b200.policy); later ``step`` calls
        without targets run it. None: the genome's open-loop sine controllers."""
        if table is None:
            table = flatten_population(individuals, tree_depth)
        self.table = table
        self._set_policy(policy)
        self.engine.upload(table)

    def step(self, n_ticks=1, targets=None):
        """Advances every living creature by ``n_ticks`` ticks. Returns (reward, done) arrays formed like ``Modular2D.step``
        (Modular2DEnv.py:642-649): reward = root x, or -100 with done = True when the root is left of the origin or behind the
        wall of death. A creature whose episode ended with success (x > ENV_LENGTH) or at the step limit keeps reporting its
        x — only the two death rules give -100, as in the reference.

        ``targets`` (numpy array or CPU torch tensor of shape (n_joints,), radians, table joint order) drives every joint's
        P-controller to its target for these ticks instead of the genome's sine oscillators, which pause
        (``Engine.step_targets``; include/rem2d_control.h). ``observe()`` gives the feedback for the next call."""
        if targets is None:
            self.engine.step(n_ticks)
        else:
            if hasattr(targets, "detach"):            # torch tensor: host memory only
                if targets.device.type != "cpu":
                    raise ValueError("targets must be on the host (a numpy array or a CPU tensor)")
                targets = targets.detach().numpy()
            self.engine.step_targets(targets, n_ticks)
        x, wod, _alive = self.engine.read_roots()          # 16 bytes per creature, not the whole state block
        x = x.astype(np.float64)
        dead = (x < 0.0) | (wod > x)
        return np.where(dead, -100.0, x), dead

    def observe(self):
        """End-of-tick observations for closed-loop control: a dict of joint_angle float32[n_joints], joint_speed
        float32[n_joints], root float32[n, 6] (x, y, angle, vx, vy, omega) and ground int32[n_bodies]
        (``Engine.read_observations``)."""
        return self.engine.read_observations()

    def fitness(self):
        return self.engine.fitness()

    def evaluate(self, individuals=None, table=None, steps=K.EVALUATION_STEPS, tree_depth=None, stats=None, policy=None):
        """Whole episodes for the whole population: float64 fitness per individual, as ``evaluate`` returns. ``stats``
        (default: the constructor's) also records the episode statistics, left in ``last_stats``; they never change results.
        ``policy``: per-joint feedback policy weights for this population, shape (n_joints, 10 * H + 1) (``reset``); None:
        open loop."""
        if table is None:
            table = flatten_population(individuals, tree_depth)
        self.table = table
        stats = self.stats if stats is None else bool(stats)
        if stats != self._engine_stats:
            self.engine.set_stats(stats)
            self._engine_stats = stats
        self._set_policy(policy)
        fit, ticks = self.engine.evaluate(table, steps)
        self.last_ticks = ticks
        self.last_stats = self.engine.read_stats() if stats else None
        return fit

    def close(self):
        self.engine.close()


class Modular2D:
    """Single-creature facade with the reference env's method signatures (one world on the GPU)."""
    metadata = {'render.modes': ['human', 'rgb_array'], 'video.frames_per_second': K.FPS}
    hardcore = False

    def __init__(self, random_seed=None, device=0):
        self._batched = BatchedModular2D(device=device)
        high = np.array([np.inf] * 24)
        self.action_space = _Box(np.array([-1, -1, -1, -1]), np.array([1, 1, 1, 1]))
        self.observation_space = _Box(-high, high)
        self.tree_morphology = None
        self.seed(random_seed)

    def seed(self, seed=None):
        return self._batched.seed(seed)

    def reset(self, tree=None, module_list=None):
        self.tree_morphology = tree
        if tree is not None:
            self._batched.reset(table=pack([flatten_tree(tree, module_list)]))
        return

    def step(self, action):
        """Like the reference, ignores ``action``: the genome's controllers drive the joints (closed-loop control:
        ``BatchedModular2D.step(targets=...)``)."""
        if self.tree_morphology is None:
            raise Exception("no tree_morphology")
        reward, done = self._batched.step(1)
        return 0, float(reward[0]), bool(done[0]), 0

    def render(self, mode='human', path=None):
        """Headless replacement of the pyglet viewer (Modular2DEnv.py:655-738): rasterises the current state of the creature.
        ``rgb_array`` returns the image; ``human`` writes it as a PNG (``path`` or ./rem2d_frame_<tick>.png) and returns
        the file name - there is no window on a GPU box."""
        from . import render as _render
        if self.tree_morphology is None:
            raise Exception("no tree_morphology")
        b = self._batched
        st = b.engine.read_state()
        img = _render.render_creature(b.table, 0, st["pose"], b.terrain_y, wod=float(st["wod"][0]))
        if mode == 'rgb_array':
            return img
        path = path or "rem2d_frame_%05d.png" % int(st["ticks"][0])
        _render.write_png(path, img)
        return path

    def close(self):
        self._batched.close()


ModularEnv = Modular2D

_env = None


def getEnv():
    """Process-wide env singleton (REM2D_main.py:57-67)."""
    global _env
    if _env is None:
        _env = BatchedModular2D()
    return _env


def evaluate(individual, EVALUATION_STEPS=10000, HEADLESS=True, INTERVAL=100, ENV_LENGTH=100, TREE_DEPTH=None,
             CONTROLLER=None):
    """Drop-in for REM2D_main.evaluate: one individual, whole episode, Python float fitness."""
    if TREE_DEPTH is None:
        try:
            TREE_DEPTH = individual.tree_depth
        except AttributeError:
            raise Exception("Tree depth not defined in evaluation")
    if not HEADLESS:
        raise NotImplementedError("HEADLESS=False needs the pyglet viewer, which is out of scope of this path")
    env = getEnv()
    cfg = env.engine.cfg
    if cfg.evaluation_steps != EVALUATION_STEPS or cfg.env_length != ENV_LENGTH:
        env.close()
        globals()["_env"] = env = BatchedModular2D(evaluation_steps=EVALUATION_STEPS, env_length=float(ENV_LENGTH))
    env.seed(K.TERRAIN_SEED)
    return float(env.evaluate([individual], steps=EVALUATION_STEPS, tree_depth=TREE_DEPTH)[0])


def evaluate_population(individuals, EVALUATION_STEPS=10000, TREE_DEPTH=None, env=None, as_torch=True, return_stats=False,
                        policy=None):
    """Batched evaluate: fitness of every individual (torch.float32 tensor on the host by default). With ``return_stats``,
    ``(fitness, stats)``: the episode statistics of ``Engine.read_stats`` (numpy arrays; ground_ticks per body of the
    flattened table). ``policy``: per-joint feedback policy weights for the flattened population (``BatchedModular2D.reset``)."""
    env = env or getEnv()
    env.seed(K.TERRAIN_SEED)
    fit = env.evaluate(individuals, steps=EVALUATION_STEPS, tree_depth=TREE_DEPTH, stats=True if return_stats else None,
                       policy=policy)
    if as_torch:
        import torch
        fit = torch.from_numpy(fit.astype(np.float32))
    return (fit, env.last_stats) if return_stats else fit
