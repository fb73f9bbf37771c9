"""Pins for the CPU oracle (oracle/rem2d_oracle.c).

* control_pin: controller + P-control + wall of death against the reference's own step() run on a
  frozen fake Box2D world (tests/golden/control_pin.json)                               (a9, a10, a12)
* analytic known answers for the Box2D-2.3 restatement (SURVEY.md 8c, pin P3): free fall, resting
  contact depth and manifold, interior-vertex circle contacts, motor torque saturation, limit snap,
  sleeping, wall-of-death lifetime, momentum conservation, Coulomb friction and rolling on inclines,
  time of impact.
The oracle is parity-UNPINNED against real pybox2d (not installable); these tests pin what can be.
"""
import json
import math
import os
import random
import sys

import numpy as np
import pytest

from gym_rem2d_b200 import Individual, constants as K, terrain
from gym_rem2d_b200.encodings.direct import DirectEncoding
from gym_rem2d_b200.flatten import CreatureTable, flatten_tree, pack, flatten_population
from gym_rem2d_b200.modules import get_module_list
from oracle.oracle import OracleEngine

F32 = np.float32


def flat_engine(**kw):
    e = OracleEngine(**kw)
    xs, ys = terrain.flat_terrain()
    e.set_terrain(ys, K.TERRAIN_STEP)
    return e


def single(shape, hx, hy, x=5.0, y=7.0, a=0.0):
    c = CreatureTable()
    c.shape, c.hx, c.hy, c.x0, c.y0, c.a0 = [shape], [hx], [hy], [x], [y], [a]
    c.node_index, c.type_ref, c.ctrl = [0], [0], [(0.0, 0.0, 0.0, 0.0, 0.0)]
    return c


def add_child(c, parent, shape, hx, hy, x, y, a, anchor_a, anchor_b, ctrl=(0.0, 0.0, 0.0, 0.0, 0.0)):
    c.shape.append(shape); c.hx.append(hx); c.hy.append(hy); c.x0.append(x); c.y0.append(y); c.a0.append(a)
    c.node_index.append(len(c.shape) - 1); c.type_ref.append(0); c.ctrl.append(ctrl)
    c.joint_parent.append(parent); c.anchor_a.append(anchor_a); c.anchor_b.append(anchor_b)
    c.lower.append(float(F32(-math.pi / 2))); c.upper.append(float(F32(math.pi / 2))); c.max_torque.append(50.0)
    return c


def test_control_pin_matches_reference_step(golden_dir):
    pin = json.load(open(os.path.join(golden_dir, "control_pin.json")))
    random.seed(pin["seed"])
    g = DirectEncoding(get_module_list())
    pop = pack([flatten_tree(g.create(8), g.moduleList)])
    e = flat_engine(dt=0.0)          # dt = 0: Box2D skips Solve/SolveTOI, bodies stay frozen like the fake world
    e.upload(pop)
    assert pin["step_args"][1:] == [180, 60] and F32(pin["step_args"][0]) == F32(0.02)
    for t, ref in enumerate(pin["ticks"]):
        e.step(1)
        st = e.read_state()
        assert np.array_equal(st["motor_speed"], np.array(ref["motor_speed"], F32)), t
        assert st["wod"][0] == ref["wod"]
        assert bool(st["alive"][0]) == (not ref["done"])
    # frozen at x = 5 -> reward 5 -> fitness 5 while alive
    assert e.fitness()[0] == 5.0


def test_free_fall_closed_form():
    e = flat_engine(terminate=0)
    e.upload(pack([single(0, 0.25, 0.25, y=9.0)]))
    y = F32(9.0); v = F32(0.0); dt = F32(0.02)
    for k in range(20):
        e.step(1)
        v = F32(v + F32(dt * F32(-10.0)))       # symplectic Euler in float32, Box2D operation order
        y = F32(y + F32(dt * v))
        st = e.read_state()
        assert st["pose"][0, 1] == y and st["vel"][0, 1] == v and st["pose"][0, 0] == 5.0
    # closed form y_k = y0 - g dt^2 k(k+1)/2 within float32 accumulation error
    assert abs(float(y) - (9.0 - 10 * 0.02 ** 2 * 20 * 21 / 2)) < 1e-5


def test_box_rests_at_linear_slop_with_two_point_manifold():
    e = flat_engine(terminate=0)
    e.upload(pack([single(0, 0.5, 0.25, y=5.5)]))
    e.step(150)
    st = e.read_state(max_pairs=8)
    # polygon skin 0.01 + edge skin 0.01; the position solver only pushes while separation < -linearSlop,
    # so the box comes to rest with a separation in [-linearSlop, 0]
    sep = st["pose"][0, 1] - (5.0 + 0.25 + 0.02)
    assert -0.005 - 1e-4 <= sep <= 1e-4
    # the box spans three terrain edges; sequential impulses leave a tilt well inside the slop band
    assert abs(st["pose"][0, 2]) < 0.01 and np.all(np.abs(st["vel"][0]) < 1e-3)
    assert st["n_touching"][0] >= 1
    # weight is carried by the normal impulses: sum = m g dt = (4 * .5 * .25) * 10 * 0.02
    imp = st["touching_impulse"][0][: st["n_touching"][0]]
    assert abs(imp[:, :2].sum() - 0.5 * 10 * 0.02) < 1e-3
    e.step(100)
    assert e.read_state()["awake"][0] == 0          # a lone body at rest goes to sleep after 0.5 s


def test_circle_on_interior_vertex_touches_two_edges():
    e = flat_engine(terminate=0)
    x_vertex = 10 * K.TERRAIN_STEP
    e.upload(pack([single(1, 0.3, 0.0, x=x_vertex, y=5.4)]))
    e.step(120)
    st = e.read_state(max_pairs=8)
    pairs = st["touching_pairs"][0][: st["n_touching"][0]]
    sep = st["pose"][0, 1] - (5.0 + 0.3 + 0.01)
    assert -0.005 - 1e-4 <= sep <= 1e-4
    assert st["n_touching"][0] in (1, 2) and set(pairs[:, 1]) <= {9, 10}


def _pendulum(ctrl, angle=0.0):
    # root box far above ground (no contacts in the horizon), child bar hanging from its centre
    c = single(0, 0.5, 0.5, y=40.0)
    add_child(c, 0, 0, 0.1, 0.4, 5.0, 40.0 - 0.4, angle, (0.0, 0.0), (0.0, 0.4), ctrl)
    return c


def test_motor_impulse_saturates_at_dt_times_max_torque():
    e = flat_engine(terminate=0)
    # huge offset error -> P-controller asks for a speed the 50 N m motor cannot reach in one tick
    c = _pendulum((0.0, 0.0, 0.0, 1.5, 0.0))
    c.max_torque[0] = 2.0             # the stock 50 N m never saturates on modules this light
    e.upload(pack([c]))
    e.step(1)
    st = e.read_state()
    assert st["motor_speed"][0] == F32(1.9 * 1.5)
    assert st["joint_impulse"][0, 3] == F32(0.02) * F32(2.0)         # clamp at dt * maxMotorTorque


def test_limit_snap_from_outside_range():
    e = flat_engine(terminate=0)
    e.upload(pack([_pendulum((0.0, 0.0, 0.0, 0.0, 0.0), angle=2.0)]))
    st0 = e.read_state()
    e.step(1)
    st = e.read_state()
    rel = st["pose"][1, 2] - st["pose"][0, 2]
    assert st["limit_state"][0] == 2                                  # at upper limit
    # position solver pulls the angle back by up to 8 degrees per iteration, 60 iterations
    assert rel <= math.pi / 2 + 2.5 / 180 * math.pi


def test_wall_of_death_lifetime_and_fitness_latch():
    e = flat_engine()
    e.upload(pack([single(0, 0.25, 0.25)]))
    e.step(10000)
    st = e.read_state()
    # wod = 0.04 k passes x = 5 shortly after tick 125 (double accumulation of 0.04)
    assert 125 <= st["ticks"][0] <= 127 and st["alive"][0] == 0
    assert abs(e.fitness()[0] - 5.0) < 1e-3


def test_sincos_modes_agree_over_100_ticks():
    """portable sin/cos (mode 0 float = what the CUDA build uses, mode 2 double) vs libm sinf/cosf (mode 1) as
    upstream Box2D uses: both portable kernels must track the libm build equally well."""
    random.seed(11)
    pop = flatten_population([Individual.random(encoding="direct") for _ in range(16)])
    xs, ys = terrain.generate_terrain()
    out = []
    for mode in (0, 1, 2):
        e = OracleEngine(sincos_mode=mode)
        e.set_terrain(ys, K.TERRAIN_STEP)
        e.upload(pop)
        e.step(100)
        out.append(e.read_state()["pose"])
    for k in (0, 2):
        err = np.abs(out[k] - out[1]) / np.maximum(1.0, np.abs(out[1]))
        # chaotic divergence after contact events is expected for a few creatures; the bulk must agree tightly
        assert np.median(err) < 1e-5
        assert np.mean(err.max(axis=1) < 1e-4) > 0.7


def test_portable_float_sincos_is_accurate():
    """rot_set mode 0 (the float kernel, used for |a| < 65536) restated in numpy float32 with the same operation order, against
    float64 math over the whole range it serves. The restatement equals the device function bit for bit (the CPU build of
    tests/probe). Its error grows with the quadrant count: 7.7e-8 below 8192, up to 9.6e-7 between 8192 and 65536
    (measured on 4e6 random angles per band; tests/test_device_geometry.py states the same bounds for the device function)."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "probe"))
    import probe
    rng = np.random.default_rng(0)
    small = np.concatenate([np.linspace(-40, 40, 200001), np.linspace(-8191.99, 8191.99, 100001), rng.uniform(-8192, 8192, 200000)])
    large = rng.uniform(8192, 65535.99, 400000) * rng.choice([-1.0, 1.0], 400000)
    a = np.concatenate([small, large]).astype(F32)
    kf = np.floor(a * F32(0.636619747) + F32(0.5)).astype(F32)
    r = ((a - kf * F32(1.5703125)) - kf * F32(4.837512969970703125e-4)) - kf * F32(7.54978995489188216e-8)
    z = r * r
    sr = ((F32(-1.9515295891e-4) * z + F32(8.3321608736e-3)) * z - F32(1.6666654611e-1)) * z * r + r
    cr = ((F32(2.443315711809948e-5) * z - F32(1.388731625493765e-3)) * z + F32(4.166664568298827e-2)) * z * z - F32(0.5) * z + F32(1.0)
    n = kf.astype(np.int64) & 3
    s = np.where(n == 0, sr, np.where(n == 1, cr, np.where(n == 2, -sr, -cr)))
    c = np.where(n == 0, cr, np.where(n == 1, -sr, np.where(n == 2, -cr, sr)))
    ds, dc = probe.rot_set(a)
    assert np.array_equal(s.view(np.uint32), ds.view(np.uint32)) and np.array_equal(c.view(np.uint32), dc.view(np.uint32))
    err = np.maximum(np.abs(s - np.sin(a.astype(np.float64))), np.abs(c - np.cos(a.astype(np.float64))))
    band = np.abs(a) < 8192
    assert err[band].max() < 1.0e-7
    assert err[~band].max() < 1.2e-6


def test_counters_and_threads_are_consistent():
    random.seed(5)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(24)])
    xs, ys = terrain.generate_terrain()
    res = []
    for th in (1, 3):
        e = OracleEngine(threads=th)
        e.set_terrain(ys, K.TERRAIN_STEP)
        fit, ticks = e.evaluate(pop, 10000)
        res.append((fit, ticks, e.counters()))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])
    assert res[0][2] == res[1][2]
    assert res[0][2]["ticks"] == int(res[0][1].sum())
    assert np.all(res[0][1] >= 40)     # the wall of death reaches x = 5 at tick 125; creatures pushed backwards die earlier


def test_jointed_free_fall_conserves_linear_and_angular_momentum():
    """Internal constraint impulses (point-to-point, motor, limit) are equal and opposite: while a driven 3-body chain is in
    free fall, its centre of mass follows the closed-form trajectory of a single body, its horizontal momentum stays zero
    and its angular momentum about the centre of mass stays at its initial value (zero) — independent of what the
    controllers do. Checks the sign conventions and lever arms of the restated revolute solver (velocity AND position
    phase: the position solver moves bodies without touching velocities, so the centre of mass must not move either)."""
    e = flat_engine(terminate=0)

    def place(parent_pose, anchor_a, angle, anchor_b):       # child centre such that the two anchors coincide
        px, py, pa = parent_pose
        ax = px + math.cos(pa) * anchor_a[0] - math.sin(pa) * anchor_a[1]
        ay = py + math.sin(pa) * anchor_a[0] + math.cos(pa) * anchor_a[1]
        return (ax - (math.cos(angle) * anchor_b[0] - math.sin(angle) * anchor_b[1]),
                ay - (math.sin(angle) * anchor_b[0] + math.cos(angle) * anchor_b[1]), angle)

    c = single(0, 0.5, 0.5, y=60.0)
    p1 = place((5.0, 60.0, 0.0), (0.0, 0.0), 0.3, (0.0, 0.4))
    add_child(c, 0, 0, 0.1, 0.4, p1[0], p1[1], 0.3, (0.0, 0.0), (0.0, 0.4), (1.2, 0.5, 0.35, 0.2, 0.0))
    p2 = place(p1, (0.0, -0.4), -0.2, (0.3, 0.0))
    add_child(c, 1, 0, 0.3, 0.15, p2[0], p2[1], -0.2, (0.0, -0.4), (0.3, 0.0), (0.9, 1.5, 0.5, -0.3, 0.0))
    e.upload(pack([c]))
    hx, hy = np.array(c.hx), np.array(c.hy)
    m = K.MODULE_DENSITY * 4.0 * hx * hy                                  # b2PolygonShape::ComputeMass of a box
    inertia = m * ((2 * hx) ** 2 + (2 * hy) ** 2) / 12.0
    st = e.read_state()
    com0 = (m[:, None] * st["pose"][:, :2].astype(np.float64)).sum(0) / m.sum()
    moved = False
    for k in range(1, 41):
        e.step(1)
        st = e.read_state()
        p, v = st["pose"].astype(np.float64), st["vel"].astype(np.float64)
        assert st["n_contacts"][0] == 0
        com = (m[:, None] * p[:, :2]).sum(0) / m.sum()
        vcom = (m[:, None] * v[:, :2]).sum(0) / m.sum()
        assert abs(com[0] - com0[0]) < 2e-5 and abs(vcom[0]) < 2e-5
        assert abs(com[1] - (com0[1] - 10.0 * 0.02 ** 2 * k * (k + 1) / 2)) < 2e-4
        assert abs(vcom[1] + 10.0 * 0.02 * k) < 2e-5
        r = p[:, :2] - com
        u = v[:, :2] - vcom
        L = (inertia * v[:, 2]).sum() + (m * (r[:, 0] * u[:, 1] - r[:, 1] * u[:, 0])).sum()
        assert abs(L) < 5e-4, (k, L)
        moved |= abs(st["pose"][1, 2] - st["pose"][0, 2] - 0.3) > 0.05
    assert moved                                                           # the motors did drive the joints


def test_motor_cannot_push_a_joint_through_its_limit():
    """A controller offset of 2.5 rad asks for an angle beyond the +pi/2 joint limit: the P-controlled motor drives the joint
    into the limit, where the 3x3 (point + limit) solve and the position solver hold it within the angular slop."""
    e = flat_engine(terminate=0)
    c = _pendulum((0.0, 0.0, 0.0, 2.5, 0.0))
    e.upload(pack([c]))
    seen_limit = False
    for k in range(60):
        e.step(1)
        st = e.read_state()
        rel = float(st["pose"][1, 2]) - float(st["pose"][0, 2])
        assert rel <= math.pi / 2 + 2.0 * (2.0 / 180.0 * math.pi) + 1e-6, (k, rel)
        seen_limit |= st["limit_state"][0] == 2
    assert seen_limit and rel > math.pi / 2 - 0.1                     # it got there and stays there
    # Box2D's convention: the impulse of an active UPPER limit is <= 0. In the steady state it balances the saturated motor
    # (+dt * maxMotorTorque = 0.02 * 50) exactly, because nothing else exerts a torque about the joint in free fall.
    assert st["joint_impulse"][0, 3] == F32(0.02) * F32(50.0)
    assert st["joint_impulse"][0, 2] <= 0.0 and abs(float(st["joint_impulse"][0, 2]) + 1.0) < 1e-3


@pytest.mark.parametrize("tan_slope", [0.3, 0.45, 0.6, 1.0])
def test_coulomb_friction_on_an_incline(tan_slope):
    """A box on an inclined edge chain: b2MixFriction gives mu = sqrt(2.5 * 0.1) = 0.5, so the box sticks while
    tan(theta) < 0.5 and otherwise slides with a = g (sin(theta) - mu cos(theta)) — friction clamp against the accumulated
    normal impulse, manifold ids across collinear edges and warm starting all have to be right for this to come out."""
    th = math.atan(tan_slope)
    xs = np.arange(200) * K.TERRAIN_STEP
    e = OracleEngine(terminate=0, allow_sleep=0)
    e.set_terrain(60.0 - tan_slope * xs, K.TERRAIN_STEP)
    x0, hx, hy = 10.0, 0.5, 0.25
    d = hy + 0.02                                                      # just above the surface, aligned with it
    cx, cy = x0 + math.sin(th) * d, 60.0 - tan_slope * x0 + math.cos(th) * d
    e.upload(pack([single(0, hx, hy, x=cx, y=cy, a=-th)]))
    v_along = []
    for k in range(101):
        e.step(1)
        st = e.read_state()
        v_along.append(float(st["vel"][0, 0]) * math.cos(th) - float(st["vel"][0, 1]) * math.sin(th))
    accel = (v_along[100] - v_along[40]) / (60 * 0.02)
    expected = max(0.0, 10.0 * (math.sin(th) - 0.5 * math.cos(th)))
    if expected == 0.0:
        assert abs(v_along[100]) < 1e-4 and abs(float(st["pose"][0, 0]) - cx) < 2e-3
    else:
        assert abs(accel - expected) < 0.01 * expected + 1e-3, (accel, expected)
    assert abs(float(st["pose"][0, 2]) + th) < 0.01                    # it slides, it does not tumble


def test_time_of_impact_stops_a_fast_small_body_at_the_edge_chain():
    """Continuous collision: a circle of radius 0.1 dropped from 55 m above the (zero-thickness) edge chain moves 0.66 m per
    tick when it arrives; the discrete step alone would put it below the terrain. SolveTOI must stop it at the surface."""
    e = flat_engine(terminate=0)
    e.upload(pack([single(1, 0.1, 0.1, x=5.1, y=60.0)]))
    lowest, events = 1e9, 0
    for k in range(260):
        e.step(1)
        st = e.read_state()
        lowest = min(lowest, float(st["pose"][0, 1]))
    events = e.counters()["toi_events"]
    assert events >= 1
    assert lowest > K.TERRAIN_HEIGHT + 0.1 - 3 * 0.005 - 1e-4          # never deeper than the TOI target separation
    assert abs(float(st["pose"][0, 1]) - (K.TERRAIN_HEIGHT + 0.1)) < 0.011 and abs(float(st["vel"][0, 1])) < 1e-3   # at rest on it


@pytest.mark.parametrize("tan_slope", [0.3, 1.0, 2.0])
def test_disc_rolls_without_slipping_until_the_slope_exceeds_three_mu(tan_slope):
    """A disc (I = m r^2 / 2) on an incline rolls with a = 2/3 g sin(theta) and v = omega r as long as tan(theta) < 3 mu = 1.5;
    on a steeper slope the contact slips and the centre accelerates like a sliding body. Pins the circle mass data, the
    edge-circle manifold, and the friction impulse acting at the contact point (torque as well as force)."""
    th = math.atan(tan_slope)
    xs = np.arange(200) * K.TERRAIN_STEP
    e = OracleEngine(terminate=0, allow_sleep=0)
    e.set_terrain(80.0 - tan_slope * xs, K.TERRAIN_STEP)
    r, x0 = 0.25, 6.0
    cx, cy = x0 + math.sin(th) * (r + 0.005), 80.0 - tan_slope * x0 + math.cos(th) * (r + 0.005)
    e.upload(pack([single(1, r, r, x=cx, y=cy)]))
    v = []
    for k in range(101):
        e.step(1)
        st = e.read_state()
        v.append((float(st["vel"][0, 0]) * math.cos(th) - float(st["vel"][0, 1]) * math.sin(th), float(st["vel"][0, 2])))
    accel = (v[100][0] - v[40][0]) / (60 * 0.02)
    slip_ratio = v[100][0] / (-v[100][1] * r)
    if tan_slope < 1.5:
        assert abs(accel - 10.0 * math.sin(th) * 2.0 / 3.0) < 0.01 * accel and abs(slip_ratio - 1.0) < 0.01
    else:
        assert abs(accel - 10.0 * (math.sin(th) - 0.5 * math.cos(th))) < 0.02 * accel and slip_ratio > 1.2


def test_results_do_not_depend_on_population_order_or_company():
    """Size-independent property of the path: every creature is its own world, so its fitness and lifetime depend neither on
    its position in the population nor on which other creatures are evaluated with it (what makes sharding by individual
    and the tiled populations of the GPU tests legitimate)."""
    random.seed(17)
    pop = flatten_population([Individual.random(encoding="lsystem") for _ in range(48)])
    xs, ys = terrain.generate_terrain()
    e = OracleEngine(threads=4)
    e.set_terrain(ys, K.TERRAIN_STEP)
    f, t = e.evaluate(pop, 400)
    perm = np.random.RandomState(3).permutation(48)
    f2, t2 = e.evaluate(pop.select(perm), 400)
    assert np.array_equal(f2, f[perm]) and np.array_equal(t2, t[perm])
    sub = np.array([5, 5, 40, 0, 17])
    f3, t3 = e.evaluate(pop.select(sub), 400)
    assert np.array_equal(f3, f[sub]) and np.array_equal(t3, t[sub])
    f4, t4 = e.evaluate(pop, 400)                     # and an evaluation leaves nothing behind in the engine
    assert np.array_equal(f4, f) and np.array_equal(t4, t)
