"""The geometry kernels of the device code (gym_rem2d_b200/csrc/rem2d_device.cuh) against plain float64 references.

The oracle and the device code are two restatements of Box2D 2.3 by the same hands and are tested against each other bit
for bit; a mistake they share would pass those tests. Here the narrow phase (Sim::contact_update: edge vs circle, edge vs
box), the GJK distance (Sim::gjk), the time of impact (Sim::time_of_impact) and the float sin/cos (rot_set) are run on
batches of poses through tests/probe (the device code's own functions, built with g++ on the CPU and with nvcc for the
GPU) and compared with references written from the definitions of the operations, in float64, without the oracle.

Tolerances are a small multiple of 2^-23 (|coordinate| + 1) (plus the stated rot_set error times the body's extent where
the body is rotated). Near a decision boundary (within the tolerance of a threshold) the reference accepts either branch,
but the output must then be what the reference computes for the branch taken; such cases are counted and must be rare in
the random batches. The CPU tests check the g++ build; the gpu tests check that the nvcc -fmad=false build equals it bit for
bit (so the CPU tests check what the B200 runs) and that the fused-multiply-add build stays within the same tolerances.
"""
import math
import os
import sys

import numpy as np
import pytest

from gym_rem2d_b200 import constants as K, terrain

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "probe"))
import probe  # noqa: E402

F32 = np.float32
ULP = 2.0 ** -23
SLOP = 0.005                      # b2_linearSlop
POLY_R = 2.0 * SLOP               # b2_polygonRadius: skin of boxes and terrain edges
EP_RADIUS = 2.0 * POLY_R          # b2EPCollider: total radius of edge + box
MAX_ROT = 0.5 * math.pi           # b2_maxRotation per step
TOL_K = 16                        # tolerance = TOL_K * 2^-23 * (|coordinate| + 1) + rotation term
# rot_set: largest |error| against float64 sin/cos per band of |angle| (stated bounds; see test_rot_set_*)
ROT_BANDS = ((0.0, 8192.0, 1.0e-7), (8192.0, 65536.0, 1.2e-6), (65536.0, 2.0 ** 24, 4.0e-8))
MT_CIRCLES, MT_FACE_A, MT_FACE_B = 0, 1, 2
LV = np.array([(-1.0, -1.0), (1.0, -1.0), (1.0, 1.0), (-1.0, 1.0)])          # box vertices / (hx, hy)
LN = np.array([(0.0, -1.0), (1.0, 0.0), (0.0, 1.0), (-1.0, 0.0)])            # box face normals
BOX_SIZES = (0.1, 0.25, 0.4, 0.5)          # half extents modules.py produces (default 0.2 x 0.8, and 0.5 ... 1.0)
RADII = (0.25, 0.375, 0.5)                 # circle radii modules.py produces


def mkid(ia, ib, ta, tb):
    return ia | (ib << 8) | (ta << 16) | (tb << 24)


def rot_bound(a):
    a = np.abs(np.asarray(a, np.float64))
    return np.select([a < lo_hi[1] for lo_hi in ROT_BANDS], [b[2] for b in ROT_BANDS], ROT_BANDS[-1][2])


def tolerance(coord, angle=0.0, extent=0.0):
    return TOL_K * ULP * (np.abs(coord) + 1.0) + 4.0 * rot_bound(angle) * extent


# ------------------------------------------------------------------ cases
def f32(v):
    return np.asarray(v, F32).astype(np.float64)


def seed4_edges():
    """The 199 edges of the seed-4 terrain, as the library stores them (float32 vertices at i * TERRAIN_STEP)."""
    xs, ys = terrain.generate_terrain()
    i = np.arange(len(ys) - 1)
    return np.stack([f32(i * K.TERRAIN_STEP), f32(ys[:-1]), f32((i + 1) * K.TERRAIN_STEP), f32(ys[1:])], 1)


def synthetic_edges(rng):
    """200 terrain-like edges (left to right, one TERRAIN_STEP wide) far from the origin, where float32 ulps are largest:
    flat, shallow, steep and negative slopes, and the steepest edge of the seed-4 terrain."""
    t4 = seed4_edges()
    steep = t4[np.argmax(np.abs(t4[:, 3] - t4[:, 1]))]
    i = rng.integers(150, 199, 200)
    i[:20] = 198                                                # the last edge: x ~ 199 * TERRAIN_STEP
    dy = np.concatenate([np.zeros(30), rng.uniform(-0.2, 0.2, 70), rng.uniform(-3.0, 3.0, 60), rng.choice([-1, 1], 40) * 5.0])
    y1 = rng.uniform(3.0, 8.0, 200)
    e = np.stack([f32(i * K.TERRAIN_STEP), f32(y1), f32((i + 1) * K.TERRAIN_STEP), f32(y1 + dy)], 1)
    e[0] = steep
    return e


def edge_frame(e):
    v1, v2 = e[..., 0:2], e[..., 2:4]
    d = v2 - v1
    L = np.hypot(d[..., 0], d[..., 1])
    t = d / L[..., None]
    n1 = np.stack([t[..., 1], -t[..., 0]], -1)                # b2EPCollider's normal1 (right of v1 -> v2)
    return v1, v2, t, n1, L


def box_extent_along(hx, hy, ang, n):
    c, s = np.cos(ang), np.sin(ang)
    return hx * np.abs(c * n[..., 0] + s * n[..., 1]) + hy * np.abs(-s * n[..., 0] + c * n[..., 1])


def contact_cases(edges, rng, n_box, n_circle):
    """Random bodies around the edges of a table: touching, near, far, in front of and behind the edge, near endpoints."""
    ne = len(edges)
    out = []
    for circle, n in ((0, n_box), (1, n_circle)):
        e = rng.integers(0, ne, n)
        v1, v2, t, n1, L = edge_frame(edges[e])
        u = rng.uniform(-0.3, 1.3, n)
        near_end = rng.random(n) < 0.25
        u[near_end] = rng.choice([0.0, 1.0], near_end.sum()) + rng.normal(0, 0.05, near_end.sum()) / L[near_end]
        if circle:
            hx = rng.choice(RADII, n); hy = np.zeros(n)
            ang = rng.uniform(-4 * math.pi, 4 * math.pi, n)
            ext = hx + POLY_R
        else:
            hx = rng.choice(BOX_SIZES, n); hy = rng.choice(BOX_SIZES, n)
            ang = rng.uniform(-math.pi, math.pi, n)
            big = rng.random(n) < 0.1
            ang[big] = rng.uniform(-40.0, 40.0, big.sum())
            ext = box_extent_along(hx, hy, ang, n1) + EP_RADIUS
        side = np.where(rng.random(n) < 0.6, -1.0, 1.0)           # -1: above a terrain edge (front == false)
        off = side * (ext + rng.uniform(-0.08, 0.04, n))
        wide = rng.random(n) < 0.2
        off[wide] = rng.uniform(-1.2, 1.2, wide.sum())
        c = v1 + u[:, None] * (v2 - v1) + off[:, None] * n1
        out.append(dict(edge=e, circle=np.full(n, circle), hx=f32(hx), hy=f32(hy), x=f32(c[:, 0]), y=f32(c[:, 1]), angle=f32(ang)))
    return {k: np.concatenate([o[k] for o in out]) for k in out[0]}


def structured_box_cases(edges, e_idx, rng):
    """Boxes at the places where the edge-box narrow phase goes wrong: faces parallel to the edge (exactly, +-1 ulp,
    +-1e-4 rad) at separations 0.02 +- a few ulps and in contact, corners at and within 1e-6 of an endpoint's x, boxes
    behind and straddling the edge line, angles beyond +-2 pi and near +-65536."""
    cs = []

    def add(e, hx, hy, x, y, a):
        cs.append((e, 0, hx, hy, x, y, a))

    for e in e_idx:
        v1, v2, t, n1, L = edge_frame(edges[e])
        base = math.atan2(t[1], t[0])
        for hx, hy in ((0.1, 0.4), (0.25, 0.25), (0.5, 0.5)):
            for k in range(4):
                a0 = F32(base + k * math.pi / 2)
                for a in (a0, np.nextafter(a0, F32(10)), np.nextafter(a0, F32(-10)), F32(a0 + 1e-4), F32(a0 - 1e-4),
                          F32(a0 + 2 * math.pi * 3), F32(a0 - 2 * math.pi * 5)):
                    h = box_extent_along(hx, hy, float(a), n1)
                    for side in (-1.0, 1.0):
                        for sep in (0.02, 0.02 + 4e-6, 0.02 - 4e-6, 0.019, 0.0, -0.01, -0.2):
                            for u in (0.5, 0.02):
                                c = v1 + u * (v2 - v1) + side * (h + sep) * n1
                                add(e, hx, hy, c[0], c[1], a)
            # corners at (and within 1e-6 of) an endpoint's x, tilted boxes touching the edge line
            for a in (0.3, -0.7, 1.1, F32(65535.5), F32(-65536.0)):
                a = float(F32(a))
                ca, sa = math.cos(a), math.sin(a)
                corners = np.array([(ca * x - sa * y, sa * x + ca * y) for x, y in LV * (hx, hy)])
                for vend in (v1, v2):
                    for j in range(4):
                        for dx in (0.0, 1e-6, -1e-6):
                            for dy in (0.0, 0.005, -0.01):
                                cx = vend[0] + dx - corners[j, 0]
                                # the corner on (or just off) the edge line at that x, body above or below it
                                ly = v1[1] + (vend[0] + dx - v1[0]) * t[1] / t[0]
                                for sgn in (1.0, -1.0):
                                    cy = ly + sgn * dy - corners[j, 1]
                                    add(e, hx, hy, cx, cy, a)
            # straddling: centroid on (and just off) the edge line
            for a in rng.uniform(-math.pi, math.pi, 6):
                for d in (0.0, 1e-7, -1e-7, 0.1, -0.1):
                    c = v1 + 0.5 * (v2 - v1) + d * n1
                    add(e, hx, hy, c[0], c[1], a)
    a = np.array(cs, np.float64)
    return dict(edge=a[:, 0].astype(np.int64), circle=a[:, 1].astype(np.int64), hx=f32(a[:, 2]), hy=f32(a[:, 3]),
                x=f32(a[:, 4]), y=f32(a[:, 5]), angle=f32(a[:, 6]))


def structured_circle_cases(edges, e_idx):
    """Circles with centres on the perpendicular through an endpoint (u == 0, v == 0) and on the edge line, at the contact
    distance +- a few ulps."""
    cs = []
    for e in e_idx:
        v1, v2, t, n1, L = edge_frame(edges[e])
        for r in RADII:
            for end, tdir in ((v1, -1.0), (v2, 1.0)):
                for s in (-1.0, 1.0):
                    for d in (r + POLY_R, r + POLY_R + 4e-6, r + POLY_R - 4e-6, 0.5 * r, 0.0):
                        c = end + s * d * n1
                        cs.append((e, 1, r, 0.0, c[0], c[1], 0.3))
                        c = end + tdir * d * t                       # on the edge line beyond the endpoint
                        cs.append((e, 1, r, 0.0, c[0], c[1], -2.0))
            for u in (0.25, 0.5, 0.75):
                c = v1 + u * (v2 - v1)
                cs.append((e, 1, r, 0.0, c[0], c[1], 7.0))           # centre on the edge line
    a = np.array(cs, np.float64)
    return dict(edge=a[:, 0].astype(np.int64), circle=a[:, 1].astype(np.int64), hx=f32(a[:, 2]), hy=f32(a[:, 3]),
                x=f32(a[:, 4]), y=f32(a[:, 5]), angle=f32(a[:, 6]))


def cat(*ds):
    return {k: np.concatenate([d[k] for d in ds]) for k in ds[0]}


def flat_edges(edges):
    """The flat edges of a table (the start pad of the seed-4 terrain): endpoint perpendiculars are exact in float32."""
    return np.nonzero(edges[:, 1] == edges[:, 3])[0]


# ------------------------------------------------------------------ float64 references
class Decider:
    """Records the branches of one evaluation of a reference. A comparison within `tol` of its threshold (or an arg-min/max
    with several candidates within `tol`) is ambiguous: every alternative is explored by `outcomes`."""

    def __init__(self, forced, tol):
        self.forced, self.tol, self.taken, self.nopt = forced, tol, [], []

    def _pick(self, options):
        k = len(self.taken)
        j = self.forced[k] if k < len(self.forced) else 0
        self.taken.append(j)
        self.nopt.append(len(options))
        return options[j]

    def le(self, a, b):                       # a <= b
        d = a - b
        return self._pick([d <= 0, not d <= 0] if abs(d) <= self.tol else [d <= 0])

    def ge(self, a, b):                       # a >= b
        return self.le(b, a)

    def sign(self, d):                        # -1, 0, +1 for the clip distances (0: kept, no crossing point)
        default = -1 if d < 0 else (0 if d == 0 else 1)
        return self._pick([default] + [s for s in (-1, 0, 1) if s != default] if abs(d) <= self.tol else [default])

    def argbest(self, vals, largest):         # first index of the max (min): strict improvement, as the kernels scan
        best = 0
        for i in range(1, len(vals)):
            if (vals[i] > vals[best]) if largest else (vals[i] < vals[best]):
                best = i
        alt = [i for i in range(len(vals)) if i != best and abs(vals[i] - vals[best]) <= self.tol]
        return self._pick([best] + alt)


def outcomes(fn, tol, cap=256):
    """Every result of reference `fn(decider)` over the ambiguous branches; the first one takes the default branches."""
    res, stack = [], [[]]
    while stack and len(res) < cap:
        forced = stack.pop()
        d = Decider(forced, tol)
        res.append(fn(d))
        for k in range(len(forced), len(d.taken)):
            for alt in range(1, d.nopt[k]):
                stack.append(d.taken[:k] + [alt])
    return res


def ref_edge_box(v1, v2, p, ang, hx, hy, D):
    """b2CollideEdgeAndPolygon (b2EPCollider) without ghost vertices, in float64: edge (v1, v2) in the world frame, box of half
    extents (hx, hy) at (p, ang). Returns (count, type, normal, local point, points, ids); normal and local point in the frame
    of the reference face (world for face A, box for face B), points in the box frame (face A) or the world (face B)."""
    none = (0, None, None, None, [], [])
    c, s = math.cos(ang), math.sin(ang)
    R = lambda v: np.array([c * v[0] - s * v[1], s * v[0] + c * v[1]])
    lv = LV * (hx, hy)
    pv = [p + R(v) for v in lv]
    pn = [R(n) for n in LN]
    d = v2 - v1
    edge1 = d / math.hypot(d[0], d[1])
    normal1 = np.array([edge1[1], -edge1[0]])
    front = D.ge(float(normal1 @ (p - v1)), 0.0)
    normal = normal1 if front else -normal1
    edge_sep = min(float(normal @ (v - v1)) for v in pv)                 # edge axis: the separation of the box from the edge
    if not D.le(edge_sep, EP_RADIUS):
        return none
    seps = []
    for i in range(4):                                                   # polygon axes: each box face against the segment
        n = -pn[i]
        seps.append(min(float(n @ (pv[i] - v1)), float(n @ (pv[i] - v2))))
        if not D.le(seps[i], EP_RADIUS):
            return none                                                  # a separating box face
    poly = D.argbest(seps, True)
    primary_poly = not D.le(seps[poly], 0.98 * edge_sep + 0.001)        # hysteresis of b2EPCollider
    if not primary_poly:
        typ = MT_FACE_A
        best = D.argbest([float(normal @ n) for n in pn], False)         # incident face: most anti-parallel to the normal
        i1, i2 = best, (best + 1) % 4
        ie = [(pv[i1], mkid(0, i1, 1, 0)), (pv[i2], mkid(0, i2, 1, 0))]
        rf = (0, 1, v1, v2, normal1) if front else (1, 0, v2, v1, -normal1)
    else:
        typ = MT_FACE_B
        ie = [(v1, mkid(0, poly, 0, 1)), (v2, mkid(0, poly, 0, 1))]
        j = (poly + 1) % 4
        rf = (poly, j, pv[poly], pv[j], pn[poly])
    ri1, ri2, rv1, rv2, rn = rf
    side1 = np.array([rn[1], -rn[0]])

    def clip(vin, n, off, ia):
        d0, d1 = float(n @ vin[0][0]) - off, float(n @ vin[1][0]) - off
        s0, s1 = D.sign(d0), D.sign(d1)
        out = [v for v, sg in zip(vin, (s0, s1)) if sg <= 0]
        if s0 * s1 < 0:
            w = d0 / (d0 - d1)
            out.append((vin[0][0] + w * (vin[1][0] - vin[0][0]), mkid(ia, (vin[0][1] >> 8) & 0xff, 0, 1)))
        return out

    cp = clip(ie, side1, float(side1 @ rv1), ri1)
    if len(cp) < 2:
        return none
    cp = clip(cp, -side1, float(-side1 @ rv2), ri2)
    if len(cp) < 2:
        return none
    pts, ids = [], []
    for v, id_ in cp[:2]:
        if D.le(float(rn @ (v - rv1)), EP_RADIUS):
            if not primary_poly:
                w = v - p
                pts.append(np.array([c * w[0] + s * w[1], -s * w[0] + c * w[1]]))
                ids.append(id_)
            else:
                pts.append(v)
                ids.append(mkid((id_ >> 8) & 0xff, id_ & 0xff, (id_ >> 24) & 0xff, (id_ >> 16) & 0xff))
    if not primary_poly:
        ln, lp = rn, rv1
    else:
        ln, lp = LN[ri1], lv[ri1]
    return (len(pts), typ, ln, lp, pts, ids)


def manifold_matches(dev, i, ref, tol):
    count, typ, ln, lp, pts, ids = ref
    if int(dev["count"][i]) != count:
        return False
    if count == 0:
        return True
    if int(dev["type"][i]) != typ or [int(x) for x in dev["ids"][i, :count]] != ids:
        return False
    close = lambda a, b: np.abs(np.asarray(a, np.float64) - b).max() <= tol
    return close(dev["normal"][i], ln) and close(dev["local_point"][i], lp) and all(close(dev["points"][i, k], pts[k]) for k in range(count))


def ref_edge_circle(v1, v2, q, rad):
    """b2CollideEdgeAndCircle in float64 (vectorised): closest point of the segment to the centre, by Voronoi region of the
    segment (0: vertex v1, 1: vertex v2, 2: interior). Returns per region: distance, margin of the region test, normal."""
    e = v2 - v1
    ee = np.einsum("ij,ij->i", e, e)
    L = np.sqrt(ee)
    u = np.einsum("ij,ij->i", e, v2 - q) / L          # distance of the centre's projection before v2
    v = np.einsum("ij,ij->i", e, q - v1) / L          # ... after v1
    proj = v1 + (v / L)[:, None] * e
    n = np.stack([-e[:, 1], e[:, 0]], 1) / L[:, None]
    side = np.einsum("ij,ij->i", n, q - v1)
    n = np.where((side < 0)[:, None], -n, n)
    dist = [np.hypot(*(q - v1).T), np.hypot(*(q - v2).T), np.abs(side)]
    region = np.where(v <= 0, 0, np.where(u <= 0, 1, 2))
    return dict(dist=dist, region=region, u=u, v=v, normal=n, side=side, rad=rad + POLY_R)


# ---- distances between the edge and a body's core (GJK / TOI references)
def _dot(a, b):
    return a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]


def _cross(a, b):
    return a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]


def seg_point_dist(a, b, p):
    ab = b - a
    t = np.clip(_dot(p - a, ab) / np.maximum(_dot(ab, ab), 1e-300), 0.0, 1.0)
    d = p - (a + t[..., None] * ab)
    return np.sqrt(_dot(d, d))


def core_vertices(circle, hx, hy, cx, cy, ang):
    """World vertices of the core shape (box: its 4 corners; circle: its centre, repeated) in float64; shapes broadcast."""
    c, s = np.cos(ang), np.sin(ang)
    lx, ly = LV[:, 0] * hx[..., None], LV[:, 1] * hy[..., None]
    lx = np.where(circle[..., None] != 0, 0.0, lx)
    ly = np.where(circle[..., None] != 0, 0.0, ly)
    return np.stack([cx[..., None] + c[..., None] * lx - s[..., None] * ly, cy[..., None] + s[..., None] * lx + c[..., None] * ly], -1)


def edge_core_distance(v1, v2, pv):
    """Exact distance between the segment (v1, v2) and the convex hull of pv (4 corners in counter-clockwise order, or a
    point repeated): the minimum of the vertex-segment distances both ways, 0 where they intersect."""
    v1, v2 = v1[..., None, :], v2[..., None, :]
    q1 = np.roll(pv, -1, axis=-2)
    d = np.minimum(seg_point_dist(v1, v2, pv).min(-1),
                   np.minimum(seg_point_dist(pv, q1, v1).min(-1), seg_point_dist(pv, q1, v2).min(-1)))
    e = q1 - pv
    inside = (_cross(e, v1 - pv) >= 0).all(-1) & (np.abs(e).sum(-1) > 0).all(-1)
    o1, o2 = _cross(e, v1 - pv), _cross(e, v2 - pv)
    o3, o4 = _cross(v2 - v1, pv - v1), _cross(v2 - v1, q1 - v1)
    crossing = ((o1 * o2 < 0) & (o3 * o4 < 0)).any(-1)
    return np.where(inside | crossing, 0.0, d)


# ------------------------------------------------------------------ checks
def check_rot_set(a, s, c):
    a64 = np.asarray(a, np.float64)
    err = np.maximum(np.abs(s - np.sin(a64)), np.abs(c - np.cos(a64)))
    bound = rot_bound(a64)
    bad = np.nonzero(err > bound)[0]
    assert len(bad) == 0, "rot_set(%r): error %.3g > %.3g" % (float(a[bad[0]]), err[bad[0]], bound[bad[0]])
    return err


def rot_set_angles(rng):
    """Per band: seeded random angles of both signs, and the structured ones (+-0, multiples of pi/2 and their float
    neighbours, the switch to the double kernel at 65536)."""
    bands = []
    for lo, hi, _ in ROT_BANDS:
        a = F32(rng.uniform(lo, hi, 400000) * rng.choice([-1.0, 1.0], 400000))
        bands.append(a[(np.abs(a) >= lo) & (np.abs(a) < hi)])
    k = np.concatenate([np.arange(-64, 65), np.array([1000, 5215, 41721, 41722, 10 ** 5, 10 ** 6]) * rng.choice([-1, 1], 6)])
    m = F32(k * (math.pi / 2))
    special = np.concatenate([np.array([0.0, -0.0, 65535.99, 65536.0, -65536.0, -65535.99, 8192.0, -8192.0], F32),
                              np.nextafter(np.array([65536.0, -65536.0], F32), F32(0)),
                              m, np.nextafter(m, F32(np.inf)), np.nextafter(m, F32(-np.inf))]).astype(F32)
    return bands, special


def check_contacts(cases, edges, dev, where):
    """Every contact_update result against the float64 references and the reference-free geometric checks. Returns
    (number of boundary cases, largest deviation from the default-branch reference in units of the tolerance)."""
    n = len(cases["edge"])
    e = edges[cases["edge"]]
    v1, v2 = e[:, 0:2], e[:, 2:4]
    p = np.stack([cases["x"], cases["y"]], 1)
    ang, hx, hy = cases["angle"], cases["hx"], cases["hy"]
    coord = np.maximum(np.abs(p).max(1), np.abs(e).max(1))
    tol = tolerance(coord, ang, hx + hy)
    circ = cases["circle"] != 0
    boundary, worst = 0, 0.0
    # ---- circles
    ci = np.nonzero(circ)[0]
    if len(ci):
        r = ref_edge_circle(v1[ci], v2[ci], p[ci], hx[ci])
        for k, i in enumerate(ci):
            t = tol[i]
            regions = [r["region"][k]] + [g for g, m in ((0, abs(r["v"][k])), (1, abs(r["u"][k]))) if m <= t and g != r["region"][k]]
            if r["region"][k] != 2 and min(abs(r["u"][k]), abs(r["v"][k])) <= t:
                regions.append(2)
            ok_any, ok_default = False, False
            for j, g in enumerate(regions):
                dist = r["dist"][g][k]
                touch, near = dist <= r["rad"][k], abs(dist - r["rad"][k]) <= t
                cnt = int(dev["count"][i])
                if cnt == 0:
                    ok = (not touch) or near
                else:
                    ok = (touch or near) and cnt == 1 and np.all(dev["points"][i, 0] == 0)
                    if g == 2:
                        nrm = r["normal"][k]
                        flip = abs(r["side"][k]) <= t
                        ok = ok and dev["type"][i] == MT_FACE_A and dev["ids"][i, 0] == mkid(0, 0, 1, 0) and \
                            np.array_equal(dev["local_point"][i], F32(v1[i])) and \
                            (np.abs(dev["normal"][i] - nrm).max() <= t or (flip and np.abs(dev["normal"][i] + nrm).max() <= t))
                        if ok and not flip:
                            worst = max(worst, np.abs(dev["normal"][i] - nrm).max() / t)
                    else:
                        ok = ok and dev["type"][i] == MT_CIRCLES and dev["ids"][i, 0] == mkid(g, 0, 0, 0) and \
                            np.array_equal(dev["local_point"][i], F32((v1, v2)[g][i]))
                    ok = ok and (dev["touching"][i] == 1)
                ok_any |= ok
                ok_default |= ok and j == 0 and not (abs(r["dist"][g][k] - r["rad"][k]) <= t)
            assert ok_any, "%s edge-circle case %d: %r vs region %d dist %.9g rad %.9g" % (
                where, i, {kk: dev[kk][i] for kk in dev}, r["region"][k], r["dist"][r["region"][k]][k], r["rad"][k])
            boundary += not ok_default
    # ---- boxes
    for i in np.nonzero(~circ)[0]:
        t = tol[i]
        fn = lambda D, i=i: ref_edge_box(v1[i], v2[i], p[i], float(ang[i]), float(hx[i]), float(hy[i]), D)
        res = outcomes(fn, t)
        matched = [manifold_matches(dev, i, ref, t) for ref in res]
        assert any(matched), "%s edge-box case %d (edge %s, pose %r, hx %r hy %r): device %r, reference %r" % (
            where, i, e[i], (p[i], ang[i]), hx[i], hy[i], {kk: dev[kk][i] for kk in dev}, res[0])
        if not matched[0] or len(res) > 1:
            boundary += 1
        elif res[0][0]:
            count, typ, ln, lp, pts, ids = res[0]
            worst = max(worst, max(np.abs(dev["points"][i, k] - pts[k]).max() for k in range(count)) / t,
                        np.abs(dev["normal"][i] - ln).max() / t)
        check_box_geometry(dev, i, v1[i], v2[i], p[i], float(ang[i]), float(hx[i]), float(hy[i]), t, where)
    return boundary, worst


def check_box_geometry(dev, i, v1, v2, p, ang, hx, hy, t, where):
    """Checks that do not depend on Box2D's algorithm: a unit normal on the centroid's side of the edge, points on the incident
    face, separations that are the float64 signed distances to the reference face and at most the total radius, and no
    contact at all where the separating-axis separation exceeds the total radius."""
    c, s = math.cos(ang), math.sin(ang)
    R = lambda v: np.array([c * v[0] - s * v[1], s * v[0] + c * v[1]])
    pv = [p + R(v) for v in LV * (hx, hy)]
    pn = [R(n) for n in LN]
    d = v2 - v1
    n1 = np.array([d[1], -d[0]]) / math.hypot(d[0], d[1])
    sat = max(max(min(float(n1 @ (v - v1)) for v in pv), min(float(-n1 @ (v - v1)) for v in pv)),
              max(min(float(pn[j] @ (v1 - pv[j])), float(pn[j] @ (v2 - pv[j]))) for j in range(4)))
    count = int(dev["count"][i])
    msg = "%s edge-box case %d" % (where, i)
    if sat > EP_RADIUS + t:
        assert count == 0, msg + ": separating-axis separation %.9g but %d points" % (sat, count)
    if count == 0:
        return
    ln, lp = dev["normal"][i].astype(np.float64), dev["local_point"][i].astype(np.float64)
    assert abs(math.hypot(*ln) - 1.0) <= t, msg + ": normal not unit"
    typ = int(dev["type"][i])
    for k in range(count):
        pt = dev["points"][i, k].astype(np.float64)
        idk = int(dev["ids"][i, k])
        if typ == MT_FACE_A:
            assert float(ln @ (p - v1)) >= -t, msg + ": normal points away from the centroid"
            P = p + R(pt)                                                 # the point lies on a face of the box
            assert min(abs(hx - abs(pt[0])), abs(hy - abs(pt[1]))) <= t and abs(pt[0]) <= hx + t and abs(pt[1]) <= hy + t, \
                msg + ": point %d not on a box face" % k
            off = float(n1 @ (p - v1))                                    # (a centroid on the edge line: either side)
            nref = (n1 if off >= 0 else -n1) if abs(off) > t else (n1 if float(ln @ n1) >= 0 else -n1)
            sd = float(nref @ (P - v1))                                   # signed distance to the edge (reference face)
            sep = float(ln @ (P - lp))
        else:
            P = pt                                                        # the point lies on the edge
            assert seg_point_dist(v1, v2, P) <= t, msg + ": point %d not on the edge" % k
            face = idk & 0xff
            sd = float(pn[face] @ (P - pv[face]))                         # signed distance to the box face named by the id
            sep = float(R(ln) @ (P - (p + R(lp))))
        assert abs(sep - sd) <= t, msg + ": point %d separation %.9g, float64 distance to the reference face %.9g" % (k, sep, sd)
        assert sd <= EP_RADIUS + t, msg + ": point %d kept at separation %.9g" % (k, sd)


def distance_cases(rng, edges, n):
    e = edges[rng.integers(0, len(edges), n)]
    v1, v2, t, n1, L = edge_frame(e)
    circle = (rng.random(n) < 0.3).astype(np.int64)
    hx = np.where(circle, rng.choice(RADII, n), rng.choice(BOX_SIZES, n))
    hy = np.where(circle, 0.0, rng.choice(BOX_SIZES, n))
    u = rng.uniform(-0.5, 1.5, n)
    off = rng.choice([-1.0, 1.0], n) * rng.uniform(0.0, 1.5, n)
    c = v1 + u[:, None] * (v2 - v1) + off[:, None] * n1
    ang = rng.uniform(-8.0, 8.0, n)
    return e, dict(circle=circle, hx=f32(hx), hy=f32(hy), x=f32(c[:, 0]), y=f32(c[:, 1]), angle=f32(ang))


def check_distance(e, b, d):
    pv = core_vertices(b["circle"], b["hx"], b["hy"], b["x"], b["y"], b["angle"])
    ref = edge_core_distance(e[:, 0:2], e[:, 2:4], pv)
    coord = np.maximum(np.abs(np.stack([b["x"], b["y"]], 1)).max(1), np.abs(e).max(1))
    tol = tolerance(coord, b["angle"], b["hx"] + b["hy"])
    err = np.abs(d - ref)
    bad = np.nonzero(err > tol)[0]
    assert len(bad) == 0, "gjk case %d: %.9g, float64 distance %.9g" % (bad[0], d[bad[0]], ref[bad[0]])
    return (err / tol).max()


def toi_cases(rng, edges, n):
    """Sweeps of one step toward and along the edges: pure translations (half of them) and rotations by up to
    b2_maxRotation, hitting the interior or an endpoint corner, grazing, starting within the target, angles beyond 2 pi."""
    e = edges[rng.integers(0, len(edges), n)]
    v1, v2, t, n1, L = edge_frame(e)
    circle = (rng.random(n) < 0.3).astype(np.int64)
    hx = np.where(circle, rng.choice(RADII, n), rng.choice(BOX_SIZES, n))
    hy = np.where(circle, 0.0, rng.choice(BOX_SIZES, n))
    a0 = rng.uniform(-math.pi, math.pi, n)
    far = rng.random(n) < 0.15
    a0[far] = rng.uniform(-30.0, 30.0, far.sum())
    rotating = rng.random(n) < 0.5
    da = np.where(rotating, rng.uniform(-MAX_ROT, MAX_ROT, n), 0.0)
    ext = np.where(circle, hx, np.hypot(hx, hy)) + 0.02
    side = np.where(rng.random(n) < 0.8, -1.0, 1.0)
    u0 = rng.uniform(-0.4, 1.4, n)
    start = side * (ext + rng.uniform(-0.05, 1.0, n))
    c0 = v1 + u0[:, None] * (v2 - v1) + start[:, None] * n1
    mv = rng.uniform(0.0, 2.0, n)                                     # up to b2_maxTranslation
    dirn = -side[:, None] * n1 + rng.normal(0, 0.6, (n, 2))
    graze = rng.random(n) < 0.15                                      # along the edge at about the target distance
    dirn[graze] = t[graze] * rng.choice([-1.0, 1.0], graze.sum())[:, None]
    corner = rng.random(n) < 0.15                                     # toward an endpoint
    endp = np.where(rng.random(n)[:, None] < 0.5, v1, v2)
    dirn[corner] = endp[corner] - c0[corner]
    dirn /= np.hypot(dirn[:, 0], dirn[:, 1])[:, None]
    c1 = c0 + mv[:, None] * dirn
    sweep = np.stack([c0[:, 0], c0[:, 1], a0, c1[:, 0], c1[:, 1], a0 + da, np.zeros(n)], 1)
    sweep = f32(sweep)
    sweep[~rotating, 5] = sweep[~rotating, 2]
    return e, dict(circle=circle, hx=f32(hx), hy=f32(hy)), sweep, ~rotating


def sweep_distance(e, b, sweep, t):
    """float64 distance between the edge and the core along the linear sweep, at times t [n, m]."""
    c0, a0, c1, a1 = sweep[:, None, 0:2], sweep[:, None, 2], sweep[:, None, 3:5], sweep[:, None, 5]
    c = (1 - t)[..., None] * c0 + t[..., None] * c1
    a = (1 - t) * a0 + t * a1
    bc = lambda k: np.broadcast_to(b[k][:, None], t.shape)
    pv = core_vertices(bc("circle"), bc("hx"), bc("hy"), c[..., 0], c[..., 1], a)
    return edge_core_distance(np.broadcast_to(e[:, None, 0:2], c.shape), np.broadcast_to(e[:, None, 2:4], c.shape), pv)


def min_distance(e, b, sweep, lo, hi, iters=40):
    """Minimum of the distance over [lo, hi] of a pure translation (convex in t): dense samples plus ternary refinement."""
    ts = lo[:, None] + (hi - lo)[:, None] * np.linspace(0.0, 1.0, 65)[None, :]
    d = sweep_distance(e, b, sweep, ts)
    k = d.argmin(1)
    step = (hi - lo) / 64
    a, z = np.maximum(lo, ts[np.arange(len(k)), k] - step), np.minimum(hi, ts[np.arange(len(k)), k] + step)
    for _ in range(iters):
        m1, m2 = a + (z - a) / 3, z - (z - a) / 3
        d1 = sweep_distance(e, b, sweep, m1[:, None])[:, 0]
        d2 = sweep_distance(e, b, sweep, m2[:, None])[:, 0]
        z = np.where(d1 < d2, m2, z)
        a = np.where(d1 < d2, a, m1)
    return np.minimum(d.min(1), sweep_distance(e, b, sweep, (0.5 * (a + z))[:, None])[:, 0])


def check_toi(e, b, sweep, translation, touching, t):
    """Results of time_of_impact against the float64 distance along the sweep. Returns (largest deviation of a touching
    result from the target in units of its tolerance, number of failed results)."""
    n = len(t)
    total = np.where(b["circle"] != 0, b["hx"], POLY_R) + POLY_R
    target = np.maximum(SLOP, total - 3 * SLOP)
    tol = 0.25 * SLOP
    coord = np.maximum(np.abs(sweep[:, [0, 1, 3, 4]]).max(1), np.abs(e).max(1))
    m = tolerance(coord, np.abs(sweep[:, [2, 5]]).max(1), b["hx"] + b["hy"])
    t64 = t.astype(np.float64)
    d_t = sweep_distance(e, b, sweep, t64[:, None])[:, 0]
    d_1 = sweep_distance(e, b, sweep, np.ones((n, 1)))[:, 0]
    overlapped = ~touching & (t == 0)
    separated = ~touching & (t == 1)
    failed = ~touching & (t > 0) & (t < 1)
    i = np.nonzero(touching & (d_t > target + tol + m))[0]
    assert len(i) == 0, "toi case %d: touching at t=%.9g where the distance is %.9g > target %.9g" % (i[0], t[i[0]], d_t[i[0]], target[i[0]])
    i = np.nonzero(touching & (t > 0) & (d_t < target - tol - m))[0]
    assert len(i) == 0, "toi case %d: touching at t=%.9g where the distance is %.9g < target %.9g" % (i[0], t[i[0]], d_t[i[0]], target[i[0]])
    i = np.nonzero(overlapped & (d_t > m))[0]
    assert len(i) == 0, "toi case %d: overlapped at t = 0 but the distance is %.9g" % (i[0], d_t[i[0]])
    i = np.nonzero(separated & (d_1 < target + tol - m))[0]
    assert len(i) == 0, "toi case %d: separated, but the distance at t = 1 is %.9g" % (i[0], d_1[i[0]])
    # Pure translation: conservative advancement is exact, nothing before t may come closer than the target. For rotating
    # sweeps Box2D itself can step over a contact between the samples it looks at, so only t and t = 1 are checked there.
    # (A sweep that starts within the target reports touching at t = 0.)
    tr = np.nonzero(translation & ((touching & (t > 0)) | separated))[0]
    dmin = min_distance(e[tr], {k: v[tr] for k, v in b.items()}, sweep[tr], np.zeros(len(tr)), t64[tr])
    bad = np.nonzero(dmin < target[tr] - tol - m[tr])[0]
    assert len(bad) == 0, "toi case %d (translation): distance %.9g before t=%.9g" % (tr[bad[0]], dmin[bad[0]], t[tr[bad[0]]])
    dev = np.abs(d_t - target)[touching & (t > 0)] / (tol + m[touching & (t > 0)])
    return (dev.max() if len(dev) else 0.0), int(failed.sum()), int((failed & translation).sum())


# ------------------------------------------------------------------ fixtures
def make_tables():
    rng = np.random.default_rng(2024)
    t4, syn = seed4_edges(), synthetic_edges(rng)
    steep = int(np.argmax(np.abs(t4[:, 3] - t4[:, 1])))
    batches = []
    for name, edges, n in (("seed-4 terrain", t4, 9000), ("synthetic edges", syn, 5000)):
        rnd = contact_cases(edges, rng, int(n * 0.7), n - int(n * 0.7))
        pick = np.unique(np.concatenate([[0, 20, 100, 198 if len(edges) > 199 else steep, steep], rng.integers(0, len(edges), 3)]))
        pick = pick[pick < len(edges)]
        flat = flat_edges(edges)[:2]
        st = cat(structured_box_cases(edges, pick[:3], rng), structured_circle_cases(edges, np.concatenate([pick, flat])))
        batches.append((name, edges, rnd, st))
    return batches


@pytest.fixture(scope="module")
def tables():
    return make_tables()


@pytest.fixture(scope="module")
def distance_batch():
    rng = np.random.default_rng(77)
    edges = np.concatenate([seed4_edges(), synthetic_edges(rng)])
    e, b = distance_cases(rng, edges, 12000)
    return e, b


@pytest.fixture(scope="module")
def toi_batch():
    rng = np.random.default_rng(31)
    edges = np.concatenate([seed4_edges(), synthetic_edges(rng)])
    return toi_cases(rng, edges, 12000)


def run_contacts(kind, edges, cases):
    return probe.contact_update(edges, cases["edge"], cases["circle"], cases["hx"], cases["hy"], cases["x"], cases["y"],
                                cases["angle"], kind=kind)


# ------------------------------------------------------------------ CPU tests (g++ build of the device code)
def test_rot_set_matches_float64_per_band():
    """rot_set (the device's b2Rot::Set) against float64 sin/cos. Stated bounds per band of |angle|: < 8192: 1.0e-7;
    8192 - 65536: 1.2e-6 (the float kernel's reduction loses bits as the quadrant count grows); >= 65536, the double kernel:
    4e-8 (the float rounding of the result)."""
    bands, special = rot_set_angles(np.random.default_rng(5))
    for (lo, hi, bound), a in zip(ROT_BANDS, bands):
        s, c = probe.rot_set(a)
        err = check_rot_set(a, s, c)
        assert err.max() > 0.25 * bound, "band [%g, %g): bound %.3g is not tight (max error %.3g)" % (lo, hi, bound, err.max())
    s, c = probe.rot_set(special)
    check_rot_set(special, s, c)
    assert s[0] == 0 and s[1] == 0 and c[0] == 1 and c[1] == 1


def test_rot_set_switches_to_the_double_kernel_at_65536():
    a = np.array([65536.0, -65536.0, 1e5, -3e6], F32)
    s, c = probe.rot_set(a)
    for x, si, co in zip(a, s, c):
        # the double kernel rounds the float64 result to float: equal to float(sin), float(cos) except at a rounding tie
        assert abs(float(si) - math.sin(float(x))) <= 0.5 * np.spacing(F32(abs(math.sin(float(x))))) + 1e-15
        assert abs(float(co) - math.cos(float(x))) <= 0.5 * np.spacing(F32(abs(math.cos(float(x))))) + 1e-15


def test_contact_update_matches_float64_references(tables):
    """Sim::contact_update (edge vs circle, edge vs box) on the random and the structured cases of both edge tables."""
    for name, edges, rnd, st in tables:
        dev = run_contacts("emu", edges, rnd)
        boundary, worst = check_contacts(rnd, edges, dev, name + " random")
        n = len(rnd["edge"])
        assert boundary <= 0.005 * n, "%s: %d of %d random cases at a decision boundary" % (name, boundary, n)
        assert (dev["count"] > 0).mean() > 0.3 and (dev["count"] == 2).sum() > 0.05 * n       # the batch does reach contacts
        assert ((dev["type"] == MT_FACE_B) & (dev["count"] > 0)).sum() > 0.01 * n
        dev = run_contacts("emu", edges, st)
        check_contacts(st, edges, dev, name + " structured")


def test_contact_update_carries_impulses_by_feature_id(tables):
    """Warm starting: impulses follow the feature ids of the new manifold (in either slot of the old one), others start at 0."""
    name, edges, rnd, st = tables[0]
    dev = run_contacts("emu", edges, rnd)
    n = len(rnd["edge"])
    rng = np.random.default_rng(9)
    old_count = np.where(dev["count"] > 0, rng.integers(1, 3, n), rng.integers(0, 3, n))
    swap = rng.random(n) < 0.5
    ids = np.where(swap[:, None], dev["ids"][:, ::-1], dev["ids"])
    stale = rng.random(n) < 0.2
    ids[stale, 0] ^= 0x100
    old_imp = rng.uniform(0.1, 1.0, (n, 4)).astype(F32)
    out = probe.contact_update(edges, rnd["edge"], rnd["circle"], rnd["hx"], rnd["hy"], rnd["x"], rnd["y"], rnd["angle"],
                               old_i=np.concatenate([old_count[:, None], ids], 1), old_imp=old_imp)
    for i in range(n):
        for k in range(int(out["count"][i])):
            want = (0.0, 0.0)
            for j in range(int(old_count[i])):
                if ids[i, j] == out["ids"][i, k]:
                    want = tuple(old_imp[i, 2 * j:2 * j + 2])
                    break
            assert tuple(out["impulses"][i, 2 * k:2 * k + 2]) == want, i


def test_gjk_distance_matches_float64(distance_batch):
    e, b = distance_batch
    d, cache, metric = probe.distance(e, **b)
    check_distance(e, b, d)
    assert (d == 0).mean() > 0.02 and (d > 0.5).mean() > 0.1
    # warm start: the cache of a nearby pose gives the distance of the cold call at the new pose
    rng = np.random.default_rng(3)
    n = len(d)
    b2 = dict(b, x=f32(b["x"] + rng.normal(0, 2e-3, n)), y=f32(b["y"] + rng.normal(0, 2e-3, n)),
              angle=f32(b["angle"] + rng.normal(0, 2e-3, n)))
    cold, _, _ = probe.distance(e, **b2)
    warm, _, _ = probe.distance(e, cache=cache, metric=metric, **b2)
    check_distance(e, b2, warm)
    coord = np.maximum(np.abs(np.stack([b2["x"], b2["y"]], 1)).max(1), np.abs(e).max(1))
    assert np.all(np.abs(warm - cold) <= tolerance(coord, b2["angle"], b2["hx"] + b2["hy"]))


def test_time_of_impact_matches_float64_distance_along_the_sweep(toi_batch):
    e, b, sweep, translation = toi_batch
    touching, t = probe.toi(e, b["circle"], b["hx"], b["hy"], sweep)
    worst, failed, failed_translation = check_toi(e, b, sweep, translation, touching, t)
    n = len(t)
    assert touching.mean() > 0.2 and (~touching & (t == 1)).mean() > 0.2      # both outcomes well represented
    assert failed_translation == 0 and failed <= 0.002 * n


# ------------------------------------------------------------------ GPU tests (nvcc builds of the device code)
def _all_probes(kind, tables, distance_batch, toi_batch):
    out = {}
    bands, special = rot_set_angles(np.random.default_rng(5))
    a = np.concatenate(bands + [special])
    out["rot_set"] = probe.rot_set(a, kind=kind) + (a,)
    for name, edges, rnd, st in tables:
        out[name] = (run_contacts(kind, edges, rnd), run_contacts(kind, edges, st))
    e, b = distance_batch
    out["gjk"] = probe.distance(e, kind=kind, **b)
    e, b, sweep, tr = toi_batch
    out["toi"] = probe.toi(e, b["circle"], b["hx"], b["hy"], sweep, kind=kind)
    return out


def _bits(x):
    x = np.ascontiguousarray(x)
    return x.view(np.uint32) if x.dtype == F32 else x


@pytest.mark.gpu
def test_cuda_probe_equals_cpu_probe_bit_for_bit(tables, distance_batch, toi_batch):
    assert probe.lib("cuda").probe_fmad() == 0
    cpu = _all_probes("emu", tables, distance_batch, toi_batch)
    gpu = _all_probes("cuda", tables, distance_batch, toi_batch)
    for key in cpu:
        c, g = cpu[key], gpu[key]
        for x, y in zip(c, g):
            if isinstance(x, dict):
                for k in x:
                    assert np.array_equal(_bits(x[k]), _bits(y[k])), "%s: %s differs" % (key, k)
            else:
                assert np.array_equal(_bits(x), _bits(y)), "%s differs" % key


@pytest.mark.gpu
def test_fma_probe_is_within_the_float64_tolerances(tables, distance_batch, toi_batch):
    """The fused-multiply-add build (Engine(precision="fast")) is not bit-identical, but must meet the same references."""
    assert probe.lib("fma").probe_fmad() == 1
    bands, special = rot_set_angles(np.random.default_rng(5))
    for a in bands + [special]:
        s, c = probe.rot_set(a, kind="fma")
        check_rot_set(a, s, c)
    for name, edges, rnd, st in tables:
        for cases, what in ((rnd, "random"), (st, "structured")):
            boundary, worst = check_contacts(cases, edges, run_contacts("fma", edges, cases), name + " " + what + " (fma)")
            if what == "random":
                assert boundary <= 0.005 * len(cases["edge"])
    e, b = distance_batch
    check_distance(e, b, probe.distance(e, kind="fma", **b)[0])
    e, b, sweep, tr = toi_batch
    touching, t = probe.toi(e, b["circle"], b["hx"], b["hy"], sweep, kind="fma")
    worst, failed, failed_translation = check_toi(e, b, sweep, tr, touching, t)
    assert failed_translation == 0 and failed <= 0.002 * len(t)
