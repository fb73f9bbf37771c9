/* rem2d_oracle.c — CPU ORACLE for the REM2D evaluation path.  TEST INFRASTRUCTURE, NOT THE PRODUCT.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load
 * the library built from this file. The product path is gym_rem2d_b200/csrc (CUDA) and must never
 * route through here.
 *
 * PARITY UNPINNED against real pybox2d: the arithmetic of the reference's hot path lives in the
 * third-party wheel Box2D==2.3.10 (/root/reference/requirements.txt:1; bundles Box2D C++ 2.3.x), which
 * is neither vendored in /root/reference nor installable here (no wheel, no swig, no network), and the
 * reference has no tests or golden vectors for this path. This file therefore RESTATES the published
 * Box2D 2.3 algorithm for exactly the scene the reference builds (SURVEY.md Appendix A/E):
 *   dynamic bodies with one box or one circle fixture, 199 static ghost-less edge bodies, revolute
 *   joints with motor + limit, default world flags (sleeping, warm starting, continuous physics).
 * What *is* pinned: the episode semantics around Step (controllers, P-control, wall of death, fitness
 * latch) against the reference's own Python run on a frozen fake world (tests/golden/control_pin.json),
 * and analytic known answers (tests/test_oracle.py).
 *
 * Reference call sites restated (paths under /root/reference/ModularER_2D):
 *   REM2D_main.py:350-378            evaluate(): episode loop, termination, fitness          -> tick()
 *   gym_rem2D/envs/Modular2DEnv.py:565-598  reset(): new b2World, terrain edges, robot       -> world_build()
 *   gym_rem2D/envs/Modular2DEnv.py:600-653  PID + step(): wod, controllers, motor speeds,
 *                                           world.Step(1/50, 180, 60), reward/done            -> tick()
 *   Controller/m_controller.py:17-21        Controller.update                                 -> tick()
 *   gym_rem2D/morph/simple_module.py:286-298, circular_module.py:191-202  fixtures/bodies     -> world_build()
 *   gym_rem2D/morph/module_utility.py:19-32 revolute joint definition                         -> world_build()
 * Box2D 2.3 pieces restated (upstream file names for orientation): b2World::Step/Solve/SolveTOI,
 * b2ContactManager::Collide/FindNewContacts/AddPair, b2BroadPhase/b2DynamicTree::MoveProxy (fat AABB
 * rule only; the tree itself is replaced by the terrain's x-grid), b2CollideEdgeAndPolygon,
 * b2CollideEdgeAndCircle, b2Contact::Update, b2Island::Solve/SolveTOI, b2ContactSolver,
 * b2RevoluteJoint, b2TimeOfImpact, b2Distance (GJK), b2Sweep.
 *
 * All arithmetic is IEEE float32 in upstream's operation order; build with -ffp-contract=off.
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <float.h>
#include <pthread.h>

#include "../include/rem2d.h"

/* ---------------------------------------------------------------- Box2D settings (A.1) */
#define B2_PI 3.14159265359f
#define B2_EPSILON FLT_EPSILON
#define B2_MAX_FLOAT FLT_MAX
#define B2_LINEAR_SLOP 0.005f
#define B2_ANGULAR_SLOP (2.0f / 180.0f * B2_PI)
#define B2_POLYGON_RADIUS (2.0f * B2_LINEAR_SLOP)
#define B2_AABB_EXTENSION 0.1f
#define B2_AABB_MULTIPLIER 2.0f
#define B2_VELOCITY_THRESHOLD 1.0f
#define B2_MAX_LINEAR_CORRECTION 0.2f
#define B2_MAX_ANGULAR_CORRECTION (8.0f / 180.0f * B2_PI)
#define B2_MAX_TRANSLATION 2.0f
#define B2_MAX_TRANSLATION_SQ (B2_MAX_TRANSLATION * B2_MAX_TRANSLATION)
#define B2_MAX_ROTATION (0.5f * B2_PI)
#define B2_MAX_ROTATION_SQ (B2_MAX_ROTATION * B2_MAX_ROTATION)
#define B2_BAUMGARTE 0.2f
#define B2_TOI_BAUMGARTE 0.75f
#define B2_MAX_SUB_STEPS 8
#define B2_MAX_TOI_CONTACTS 32
#define B2_TIME_TO_SLEEP 0.5f
#define B2_LINEAR_SLEEP_TOL 0.01f
#define B2_ANGULAR_SLEEP_TOL (2.0f / 180.0f * B2_PI)
/* upstream Box2D: 8; the pybox2d build raises it to 16. Only bounds the TOI push-back loop. */
#define B2_MAX_POLYGON_VERTICES 16

#define MAX_EDGES 256

typedef struct { float x, y; } V2;
typedef struct { float x, y, z; } V3;
typedef struct { float s, c; } Rot;
typedef struct { V2 p; Rot q; } Xf;
typedef struct { V2 lo, hi; } AABB;
typedef struct { V2 localCenter, c0, c; float a0, a, alpha0; } Sweep;

/* contact feature id: 4 bytes compared as one key */
typedef struct { uint8_t indexA, indexB, typeA, typeB; } Feature;
#define F_VERTEX 0
#define F_FACE 1
typedef struct { V2 v; Feature id; } ClipVertex;

#define M_CIRCLES 0
#define M_FACE_A 1
#define M_FACE_B 2
typedef struct { V2 localPoint; float normalImpulse, tangentImpulse; Feature id; } ManifoldPoint;
typedef struct { ManifoldPoint points[2]; V2 localNormal, localPoint; int type, pointCount; } Manifold;

#define CF_ENABLED 1u
#define CF_TOUCHING 2u
#define CF_ISLAND 4u
#define CF_TOI 8u

typedef struct {
    int body, edge;       /* fixture B = module body, fixture A = terrain edge (always) */
    unsigned flags;
    int toiCount;
    float toi;
    float friction, restitution;
    Manifold m;
} Contact;

typedef struct {
    int shape;            /* REM2D_SHAPE_* */
    int count;            /* polygon vertex count (4) */
    V2 verts[4], normals[4];
    float radius;         /* shape radius: polygonRadius for boxes, r for circles */
    Xf xf;
    Sweep sweep;
    V2 v;
    float w;
    float mass, invMass, I, invI;
    float sleepTime;
    int awake;
    int islandFlag, islandIndex;
    AABB fat;             /* broad-phase proxy AABB */
    int moved;            /* proxy is in the broad-phase move buffer */
} Body;

#define LIMIT_INACTIVE 0
#define LIMIT_LOWER 1
#define LIMIT_UPPER 2
#define LIMIT_EQUAL 3

typedef struct {
    int bodyA, bodyB;
    V2 localAnchorA, localAnchorB;
    float lower, upper, maxMotorTorque, motorSpeed, referenceAngle;
    V3 impulse;
    float motorImpulse;
    int limitState;
    int islandFlag;
    /* solver temp */
    int indexA, indexB;
    V2 rA, rB, localCenterA, localCenterB;
    float invMassA, invMassB, invIA, invIB;
    V3 mex, mey, mez;     /* m_mass columns */
    float motorMass;
} Joint;

typedef struct { double amplitude, phase, frequency, offset, i_state, output; } Ctrl;

typedef struct {
    int nb, nj;
    Body* bodies;
    Joint* joints;
    Ctrl* ctrl;
    Contact* contacts;    /* creation order: [0] oldest ... [nc-1] newest */
    int nc, cap;
    float edge_alpha0[MAX_EDGES]; /* sweep.alpha0 of the static edge bodies */
    float inv_dt0;
    int newFixture;
    int overflow;         /* island scratch capacity exceeded (never seen; reported by rem2d_step) */
    /* episode */
    int alive, ticks;
    double wod, fitness;
} World;

struct rem2d_handle {
    rem2d_config cfg;
    int n_edges;
    V2 ev1[MAX_EDGES], ev2[MAX_EDGES];
    AABB efat[MAX_EDGES];
    float terrain_step;
    int have_terrain;
    /* copy of the uploaded table */
    rem2d_population pop;
    void* pop_mem[16];
    int have_pop;
    World* worlds;
    int n_worlds;
    uint64_t counters[REM2D_N_COUNTERS];
    char err[256];
    int threads;
};

static __thread char g_create_err[256];

/* per-thread counters, merged after a step */
typedef struct { uint64_t c[REM2D_N_COUNTERS]; } Counters;

/* ---------------------------------------------------------------- math helpers (b2Math.h) */
static inline V2 v2(float x, float y) { V2 r = {x, y}; return r; }
static inline V2 vadd(V2 a, V2 b) { return v2(a.x + b.x, a.y + b.y); }
static inline V2 vsub(V2 a, V2 b) { return v2(a.x - b.x, a.y - b.y); }
static inline V2 vneg(V2 a) { return v2(-a.x, -a.y); }
static inline V2 vscale(float s, V2 a) { return v2(s * a.x, s * a.y); }
static inline float vdot(V2 a, V2 b) { return a.x * b.x + a.y * b.y; }
static inline float vcross(V2 a, V2 b) { return a.x * b.y - a.y * b.x; }
static inline V2 vcross_vs(V2 a, float s) { return v2(s * a.y, -s * a.x); }
static inline V2 vcross_sv(float s, V2 a) { return v2(-s * a.y, s * a.x); }
static inline float vlen(V2 a) { return sqrtf(a.x * a.x + a.y * a.y); }
static inline float vlen2(V2 a) { return a.x * a.x + a.y * a.y; }
static inline float fmin2(float a, float b) { return a < b ? a : b; }
static inline float fmax2(float a, float b) { return a > b ? a : b; }
static inline float fclamp(float a, float lo, float hi) { return fmax2(lo, fmin2(a, hi)); }
static inline float fabs2(float a) { return a > 0.0f ? a : -a; }
static inline float vnormalize(V2* a) {
    float len = vlen(*a);
    if (len < B2_EPSILON) return 0.0f;
    float inv = 1.0f / len;
    a->x *= inv; a->y *= inv;
    return len;
}
static inline V2 rmul(Rot q, V2 v) { return v2(q.c * v.x - q.s * v.y, q.s * v.x + q.c * v.y); }
static inline V2 rmulT(Rot q, V2 v) { return v2(q.c * v.x + q.s * v.y, -q.s * v.x + q.c * v.y); }
static inline V2 xmul(Xf T, V2 v) {
    return v2((T.q.c * v.x - T.q.s * v.y) + T.p.x, (T.q.s * v.x + T.q.c * v.y) + T.p.y);
}
static inline V2 xmulT(Xf T, V2 v) {
    float px = v.x - T.p.x, py = v.y - T.p.y;
    return v2(T.q.c * px + T.q.s * py, -T.q.s * px + T.q.c * py);
}
/* b2MulT(A, B) for transforms */
static inline Xf xfmulT(Xf A, Xf B) {
    Xf C;
    C.q.s = A.q.c * B.q.s - A.q.s * B.q.c;
    C.q.c = A.q.c * B.q.c + A.q.s * B.q.s;
    C.p = rmulT(A.q, vsub(B.p, A.p));
    return C;
}

/* ---------------------------------------------------------------- sin / cos
 * b2Rot::Set uses libm sinf/cosf (mode 1). Mode 0 ("portable", default) is a float kernel with a fixed
 * operation order that the CUDA build reproduces bit for bit; mode 2 is the same idea in double precision
 * (3-term Cody-Waite by pi/2 + degree-13/14 minimax; also used for the controllers' double-precision sin). */
static const double PIO2_1 = 1.57079632673412561417e+00;  /* first 33 bits of pi/2 */
static const double PIO2_2 = 6.07710050630396597660e-11;  /* next 33 bits */
static const double PIO2_2T = 2.02226624879595063154e-21; /* tail */
static const double TWO_OVER_PI = 6.36619772367581382433e-01;

static inline void sincos_kernel(double x, double* s, double* c) {
    double kd = floor(x * TWO_OVER_PI + 0.5);
    double r = ((x - kd * PIO2_1) - kd * PIO2_2) - kd * PIO2_2T;
    double z = r * r;
    double ps = -1.66666666666666324348e-01 + z * (8.33333333332248946124e-03 + z * (-1.98412698298579493134e-04 +
                z * (2.75573137070700676789e-06 + z * (-2.50507602534068634195e-08 + z * 1.58969099521155010221e-10))));
    double pc = 4.16666666666666019037e-02 + z * (-1.38888888888741095749e-03 + z * (2.48015872894767294178e-05 +
                z * (-2.75573143513906633035e-07 + z * (2.08757232129817482790e-09 + z * -1.13596475577881948265e-11))));
    double sr = r + (r * z) * ps;
    double cr = (1.0 - 0.5 * z) + (z * z) * pc;
    long long n = (long long)kd & 3LL;
    switch (n) {
    case 0: *s = sr; *c = cr; break;
    case 1: *s = cr; *c = -sr; break;
    case 2: *s = -sr; *c = -cr; break;
    default: *s = -cr; *c = sr; break;
    }
}
/* Float variant used for body rotations (mode 0): Cody-Waite by pi/2 with short constants + Cephes-style minimax
 * kernels, plain float mul/add in a fixed order. Over 100 ticks it tracks the libm build as closely as the double
 * kernel does (tests/test_oracle.py); huge angles fall back to the double kernel. */
static inline void sincos_kernel_f32(float a, float* s, float* c) {
    if (!(fabs2(a) < 65536.0f)) {
        double ds, dc;
        sincos_kernel((double)a, &ds, &dc);
        *s = (float)ds; *c = (float)dc;
        return;
    }
    float kf = floorf(a * 0.636619747f + 0.5f);
    float r = ((a - kf * 1.5703125f) - kf * 4.837512969970703125e-4f) - kf * 7.54978995489188216e-8f;
    float z = r * r;
    float sr = ((-1.9515295891e-4f * z + 8.3321608736e-3f) * z - 1.6666654611e-1f) * z * r + r;
    float cr = ((2.443315711809948e-5f * z - 1.388731625493765e-3f) * z + 4.166664568298827e-2f) * z * z - 0.5f * z + 1.0f;
    int n = (int)kf & 3;
    switch (n) {
    case 0: *s = sr; *c = cr; break;
    case 1: *s = cr; *c = -sr; break;
    case 2: *s = -sr; *c = -cr; break;
    default: *s = -cr; *c = sr; break;
    }
}
static int g_sincos_mode = 0; /* set per step call from cfg (all handles of a process share it) */
static inline Rot rot_set(float a) {
    Rot q;
    if (g_sincos_mode == 1) { q.s = sinf(a); q.c = cosf(a); return q; }
    if (g_sincos_mode == 0) { sincos_kernel_f32(a, &q.s, &q.c); return q; }
    double s, c;                 /* mode 2: double-precision portable kernel */
    sincos_kernel((double)a, &s, &c);
    q.s = (float)s; q.c = (float)c;
    return q;
}
static inline double sin_f64(double x) {
    double s, c;
    sincos_kernel(x, &s, &c);
    return s;
}

/* ---------------------------------------------------------------- sweeps (b2Sweep) */
static inline Xf sweep_xf(const Sweep* s, float beta) {
    Xf xf;
    xf.p = vadd(vscale(1.0f - beta, s->c0), vscale(beta, s->c));
    float angle = (1.0f - beta) * s->a0 + beta * s->a;
    xf.q = rot_set(angle);
    xf.p = vsub(xf.p, rmul(xf.q, s->localCenter));
    return xf;
}
static inline void sweep_advance(Sweep* s, float alpha) {
    float beta = (alpha - s->alpha0) / (1.0f - s->alpha0);
    s->c0 = vadd(s->c0, vscale(beta, vsub(s->c, s->c0)));
    s->a0 += beta * (s->a - s->a0);
    s->alpha0 = alpha;
}
static inline void sweep_normalize(Sweep* s) {
    float twoPi = 2.0f * B2_PI;
    float d = twoPi * floorf(s->a0 / twoPi);
    s->a0 -= d;
    s->a -= d;
}
static inline void body_sync_transform(Body* b) {
    b->xf.q = rot_set(b->sweep.a);
    b->xf.p = vsub(b->sweep.c, rmul(b->xf.q, b->sweep.localCenter));
}
static inline void body_advance(Body* b, float alpha) {
    sweep_advance(&b->sweep, alpha);
    b->sweep.c = b->sweep.c0;
    b->sweep.a = b->sweep.a0;
    body_sync_transform(b);
}
static inline void body_set_awake(Body* b, int flag) {
    if (flag) {
        if (!b->awake) { b->awake = 1; b->sleepTime = 0.0f; }
    } else {
        b->awake = 0; b->sleepTime = 0.0f;
        b->v = v2(0.0f, 0.0f); b->w = 0.0f;
    }
}

/* ---------------------------------------------------------------- shapes, AABBs, broad phase (A.2, A.3) */
static AABB shape_aabb(const Body* b, Xf xf) {
    AABB r;
    if (b->shape == REM2D_SHAPE_CIRCLE) {
        V2 p = vadd(xf.p, rmul(xf.q, v2(0.0f, 0.0f)));
        r.lo = v2(p.x - b->radius, p.y - b->radius);
        r.hi = v2(p.x + b->radius, p.y + b->radius);
        return r;
    }
    V2 lo = xmul(xf, b->verts[0]), hi = lo;
    for (int i = 1; i < b->count; ++i) {
        V2 v = xmul(xf, b->verts[i]);
        lo = v2(fmin2(lo.x, v.x), fmin2(lo.y, v.y));
        hi = v2(fmax2(hi.x, v.x), fmax2(hi.y, v.y));
    }
    r.lo = v2(lo.x - b->radius, lo.y - b->radius);
    r.hi = v2(hi.x + b->radius, hi.y + b->radius);
    return r;
}
static inline AABB aabb_fatten(AABB a) {
    AABB r;
    r.lo = v2(a.lo.x - B2_AABB_EXTENSION, a.lo.y - B2_AABB_EXTENSION);
    r.hi = v2(a.hi.x + B2_AABB_EXTENSION, a.hi.y + B2_AABB_EXTENSION);
    return r;
}
static inline int aabb_overlap(AABB a, AABB b) {
    V2 d1 = vsub(b.lo, a.hi), d2 = vsub(a.lo, b.hi);
    if (d1.x > 0.0f || d1.y > 0.0f) return 0;
    if (d2.x > 0.0f || d2.y > 0.0f) return 0;
    return 1;
}
static inline int aabb_contains(AABB a, AABB b) {
    return a.lo.x <= b.lo.x && a.lo.y <= b.lo.y && b.hi.x <= a.hi.x && b.hi.y <= a.hi.y;
}
/* b2Body::SynchronizeFixtures -> b2Fixture::Synchronize -> b2BroadPhase::MoveProxy */
static void body_synchronize_fixtures(Body* b) {
    Xf xf1;
    xf1.q = rot_set(b->sweep.a0);
    xf1.p = vsub(b->sweep.c0, rmul(xf1.q, b->sweep.localCenter));
    AABB a1 = shape_aabb(b, xf1), a2 = shape_aabb(b, b->xf), u;
    u.lo = v2(fmin2(a1.lo.x, a2.lo.x), fmin2(a1.lo.y, a2.lo.y));
    u.hi = v2(fmax2(a1.hi.x, a2.hi.x), fmax2(a1.hi.y, a2.hi.y));
    V2 disp = vsub(b->xf.p, xf1.p);
    if (aabb_contains(b->fat, u)) return;
    AABB f = aabb_fatten(u);
    V2 d = vscale(B2_AABB_MULTIPLIER, disp);
    if (d.x < 0.0f) f.lo.x += d.x; else f.hi.x += d.x;
    if (d.y < 0.0f) f.lo.y += d.y; else f.hi.y += d.y;
    b->fat = f;
    b->moved = 1;
}

static int world_find_contact(const World* w, int body, int edge) {
    for (int i = 0; i < w->nc; ++i)
        if (w->contacts[i].body == body && w->contacts[i].edge == edge) return i;
    return -1;
}

/* b2ContactManager::FindNewContacts -> b2BroadPhase::UpdatePairs -> AddPair.
 * Pairs are sorted by (proxyIdA, proxyIdB): terrain proxies were created first in edge order, module
 * proxies afterwards in body order, so the order is ascending (edge, body). Each new contact is
 * prepended to the world list / body lists, i.e. becomes the newest. */
static void world_find_new_contacts(rem2d_handle* h, World* w) {
    int any = 0, elo = h->n_edges, ehi = -1;
    int blo[64], bhi[64];
    for (int b = 0; b < w->nb; ++b) {
        Body* B = &w->bodies[b];
        if (!B->moved) continue;
        any = 1;
        /* conservative candidate range on the terrain's uniform x grid (stands in for the dynamic tree
         * query; the exact fat-AABB test below decides) */
        double l = floor(((double)B->fat.lo.x - 0.25) / (double)h->terrain_step) - 1.0;
        double u = ceil(((double)B->fat.hi.x + 0.25) / (double)h->terrain_step) + 1.0;
        blo[b] = l < 0.0 ? 0 : (l > (double)(h->n_edges - 1) ? h->n_edges : (int)l);
        bhi[b] = u < 0.0 ? -1 : (u > (double)(h->n_edges - 1) ? h->n_edges - 1 : (int)u);
        if (blo[b] < elo) elo = blo[b];
        if (bhi[b] > ehi) ehi = bhi[b];
    }
    if (!any) return;
    for (int e = elo; e <= ehi; ++e) {
        for (int b = 0; b < w->nb; ++b) {
            Body* B = &w->bodies[b];
            if (!B->moved) continue;
            if (e < blo[b] || e > bhi[b]) continue;
            if (!aabb_overlap(h->efat[e], B->fat)) continue;
            if (world_find_contact(w, b, e) >= 0) continue;
            /* ShouldCollide: one body dynamic, no joint between them, (0xFFFF & 0x20) && (0x1 & 0x1) */
            if (w->nc == w->cap) {
                w->cap = w->cap ? 2 * w->cap : 32;
                w->contacts = (Contact*)realloc(w->contacts, sizeof(Contact) * (size_t)w->cap);
            }
            Contact* c = &w->contacts[w->nc++];
            memset(c, 0, sizeof(*c));
            c->body = b; c->edge = e;
            c->flags = CF_ENABLED;
            c->toiCount = 0;
            c->toi = 1.0f;
            c->friction = sqrtf(h->cfg.terrain_friction * h->cfg.module_friction);  /* b2MixFriction */
            c->restitution = 0.0f;                                                   /* b2MixRestitution: max(0,0) */
            c->m.pointCount = 0;
            body_set_awake(B, 1);
        }
    }
    for (int b = 0; b < w->nb; ++b) w->bodies[b].moved = 0;
}

static void world_destroy_contact(World* w, int i) {
    Contact* c = &w->contacts[i];
    if (c->m.pointCount > 0) body_set_awake(&w->bodies[c->body], 1);
    memmove(&w->contacts[i], &w->contacts[i + 1], sizeof(Contact) * (size_t)(w->nc - i - 1));
    w->nc--;
}

/* ---------------------------------------------------------------- narrow phase (A.4) */
static int clip_segment_to_line(ClipVertex out[2], const ClipVertex in[2], V2 normal, float offset, int vertexIndexA) {
    int n = 0;
    float d0 = vdot(normal, in[0].v) - offset;
    float d1 = vdot(normal, in[1].v) - offset;
    if (d0 <= 0.0f) out[n++] = in[0];
    if (d1 <= 0.0f) out[n++] = in[1];
    if (d0 * d1 < 0.0f) {
        float interp = d0 / (d0 - d1);
        out[n].v = vadd(in[0].v, vscale(interp, vsub(in[1].v, in[0].v)));
        out[n].id.indexA = (uint8_t)vertexIndexA;
        out[n].id.indexB = in[0].id.indexB;
        out[n].id.typeA = F_VERTEX;
        out[n].id.typeB = F_FACE;
        ++n;
    }
    return n;
}

/* b2CollideEdgeAndPolygon / b2EPCollider::Collide for an edge without ghost vertices */
static void collide_edge_polygon(Manifold* m, V2 v1, V2 v2_, Xf xfA, const Body* B, Xf xfB) {
    Xf xf = xfmulT(xfA, xfB);
    V2 centroidB = xmul(xf, v2(0.0f, 0.0f));
    V2 edge1 = vsub(v2_, v1);
    vnormalize(&edge1);
    V2 normal1 = v2(edge1.y, -edge1.x);
    float offset1 = vdot(normal1, vsub(centroidB, v1));
    int front = offset1 >= 0.0f;
    V2 normal, lowerLimit, upperLimit;
    if (front) { normal = normal1; lowerLimit = vneg(normal1); upperLimit = vneg(normal1); }
    else { normal = vneg(normal1); lowerLimit = normal1; upperLimit = normal1; }
    V2 pv[4], pn[4];
    int count = B->count;
    for (int i = 0; i < count; ++i) { pv[i] = xmul(xf, B->verts[i]); pn[i] = rmul(xf.q, B->normals[i]); }
    float radius = 2.0f * B2_POLYGON_RADIUS;
    m->pointCount = 0;
    /* ComputeEdgeSeparation */
    float edgeSep = B2_MAX_FLOAT;
    for (int i = 0; i < count; ++i) {
        float s = vdot(normal, vsub(pv[i], v1));
        if (s < edgeSep) edgeSep = s;
    }
    if (edgeSep > radius) return;
    /* ComputePolygonSeparation */
    int polyType = 0 /* unknown */, polyIndex = -1;
    float polySep = -B2_MAX_FLOAT;
    V2 perp = v2(-normal.y, normal.x);
    for (int i = 0; i < count; ++i) {
        V2 n = vneg(pn[i]);
        float s1 = vdot(n, vsub(pv[i], v1));
        float s2 = vdot(n, vsub(pv[i], v2_));
        float s = fmin2(s1, s2);
        if (s > radius) { polyType = 1; polyIndex = i; polySep = s; break; }
        if (vdot(n, perp) >= 0.0f) {
            if (vdot(vsub(n, upperLimit), normal) < -B2_ANGULAR_SLOP) continue;
        } else {
            if (vdot(vsub(n, lowerLimit), normal) < -B2_ANGULAR_SLOP) continue;
        }
        if (s > polySep) { polyType = 1; polyIndex = i; polySep = s; }
    }
    if (polyType != 0 && polySep > radius) return;
    const float k_relativeTol = 0.98f, k_absoluteTol = 0.001f;
    int primaryIsPoly;
    if (polyType == 0) primaryIsPoly = 0;
    else if (polySep > k_relativeTol * edgeSep + k_absoluteTol) primaryIsPoly = 1;
    else primaryIsPoly = 0;

    ClipVertex ie[2];
    int rf_i1, rf_i2;
    V2 rf_v1, rf_v2, rf_normal;
    if (!primaryIsPoly) {
        m->type = M_FACE_A;
        int best = 0;
        float bestValue = vdot(normal, pn[0]);
        for (int i = 1; i < count; ++i) {
            float value = vdot(normal, pn[i]);
            if (value < bestValue) { bestValue = value; best = i; }
        }
        int i1 = best, i2 = i1 + 1 < count ? i1 + 1 : 0;
        ie[0].v = pv[i1]; ie[0].id.indexA = 0; ie[0].id.indexB = (uint8_t)i1; ie[0].id.typeA = F_FACE; ie[0].id.typeB = F_VERTEX;
        ie[1].v = pv[i2]; ie[1].id.indexA = 0; ie[1].id.indexB = (uint8_t)i2; ie[1].id.typeA = F_FACE; ie[1].id.typeB = F_VERTEX;
        if (front) { rf_i1 = 0; rf_i2 = 1; rf_v1 = v1; rf_v2 = v2_; rf_normal = normal1; }
        else { rf_i1 = 1; rf_i2 = 0; rf_v1 = v2_; rf_v2 = v1; rf_normal = vneg(normal1); }
    } else {
        m->type = M_FACE_B;
        ie[0].v = v1; ie[0].id.indexA = 0; ie[0].id.indexB = (uint8_t)polyIndex; ie[0].id.typeA = F_VERTEX; ie[0].id.typeB = F_FACE;
        ie[1].v = v2_; ie[1].id.indexA = 0; ie[1].id.indexB = (uint8_t)polyIndex; ie[1].id.typeA = F_VERTEX; ie[1].id.typeB = F_FACE;
        rf_i1 = polyIndex; rf_i2 = rf_i1 + 1 < count ? rf_i1 + 1 : 0;
        rf_v1 = pv[rf_i1]; rf_v2 = pv[rf_i2]; rf_normal = pn[rf_i1];
    }
    V2 side1 = v2(rf_normal.y, -rf_normal.x), side2 = vneg(side1);
    float sideOffset1 = vdot(side1, rf_v1), sideOffset2 = vdot(side2, rf_v2);
    ClipVertex cp1[2], cp2[2];
    int np = clip_segment_to_line(cp1, ie, side1, sideOffset1, rf_i1);
    if (np < 2) return;
    np = clip_segment_to_line(cp2, cp1, side2, sideOffset2, rf_i2);
    if (np < 2) return;
    if (!primaryIsPoly) { m->localNormal = rf_normal; m->localPoint = rf_v1; }
    else { m->localNormal = B->normals[rf_i1]; m->localPoint = B->verts[rf_i1]; }
    int pointCount = 0;
    for (int i = 0; i < 2; ++i) {
        float separation = vdot(rf_normal, vsub(cp2[i].v, rf_v1));
        if (separation <= radius) {
            ManifoldPoint* cp = &m->points[pointCount];
            if (!primaryIsPoly) {
                cp->localPoint = xmulT(xf, cp2[i].v);
                cp->id = cp2[i].id;
            } else {
                cp->localPoint = cp2[i].v;
                cp->id.typeA = cp2[i].id.typeB; cp->id.typeB = cp2[i].id.typeA;
                cp->id.indexA = cp2[i].id.indexB; cp->id.indexB = cp2[i].id.indexA;
            }
            ++pointCount;
        }
    }
    m->pointCount = pointCount;
}

/* b2CollideEdgeAndCircle for an edge without ghost vertices (circle centre m_p = 0) */
static void collide_edge_circle(Manifold* m, V2 A, V2 Bv, float edgeRadius, Xf xfA, const Body* body, Xf xfB) {
    m->pointCount = 0;
    V2 mp = v2(0.0f, 0.0f);
    V2 Q = xmulT(xfA, xmul(xfB, mp));
    V2 e = vsub(Bv, A);
    float u = vdot(e, vsub(Bv, Q));
    float v = vdot(e, vsub(Q, A));
    float radius = edgeRadius + body->radius;
    Feature cf; cf.indexB = 0; cf.typeB = F_VERTEX;
    if (v <= 0.0f) {
        V2 P = A, d = vsub(Q, P);
        float dd = vdot(d, d);
        if (dd > radius * radius) return;
        cf.indexA = 0; cf.typeA = F_VERTEX;
        m->pointCount = 1; m->type = M_CIRCLES; m->localNormal = v2(0.0f, 0.0f); m->localPoint = P;
        m->points[0].id = cf; m->points[0].localPoint = mp;
        return;
    }
    if (u <= 0.0f) {
        V2 P = Bv, d = vsub(Q, P);
        float dd = vdot(d, d);
        if (dd > radius * radius) return;
        cf.indexA = 1; cf.typeA = F_VERTEX;
        m->pointCount = 1; m->type = M_CIRCLES; m->localNormal = v2(0.0f, 0.0f); m->localPoint = P;
        m->points[0].id = cf; m->points[0].localPoint = mp;
        return;
    }
    float den = vdot(e, e);
    V2 P = vscale(1.0f / den, vadd(vscale(u, A), vscale(v, Bv)));
    V2 d = vsub(Q, P);
    float dd = vdot(d, d);
    if (dd > radius * radius) return;
    V2 n = v2(-e.y, e.x);
    if (vdot(n, vsub(Q, A)) < 0.0f) n = v2(-n.x, -n.y);
    vnormalize(&n);
    cf.indexA = 0; cf.typeA = F_FACE;
    m->pointCount = 1; m->type = M_FACE_A; m->localNormal = n; m->localPoint = A;
    m->points[0].id = cf; m->points[0].localPoint = mp;
}

static inline int feature_eq(Feature a, Feature b) {
    return a.indexA == b.indexA && a.indexB == b.indexB && a.typeA == b.typeA && a.typeB == b.typeB;
}
static const Xf XF_IDENTITY = {{0.0f, 0.0f}, {0.0f, 1.0f}};

/* b2Contact::Update (no listener, no sensors) */
static void contact_update(rem2d_handle* h, World* w, Contact* c, Counters* cnt) {
    Manifold old = c->m;
    c->flags |= CF_ENABLED;
    int wasTouching = (c->flags & CF_TOUCHING) != 0;
    Body* B = &w->bodies[c->body];
    cnt->c[REM2D_CNT_NARROW]++;
    if (B->shape == REM2D_SHAPE_CIRCLE)
        collide_edge_circle(&c->m, h->ev1[c->edge], h->ev2[c->edge], B2_POLYGON_RADIUS, XF_IDENTITY, B, B->xf);
    else
        collide_edge_polygon(&c->m, h->ev1[c->edge], h->ev2[c->edge], XF_IDENTITY, B, B->xf);
    int touching = c->m.pointCount > 0;
    for (int i = 0; i < c->m.pointCount; ++i) {
        ManifoldPoint* mp2 = &c->m.points[i];
        mp2->normalImpulse = 0.0f; mp2->tangentImpulse = 0.0f;
        for (int j = 0; j < old.pointCount; ++j) {
            if (feature_eq(old.points[j].id, mp2->id)) {
                mp2->normalImpulse = old.points[j].normalImpulse;
                mp2->tangentImpulse = old.points[j].tangentImpulse;
                break;
            }
        }
    }
    if (touching != wasTouching) body_set_awake(B, 1);
    if (touching) c->flags |= CF_TOUCHING; else c->flags &= ~CF_TOUCHING;
}

/* b2ContactManager::Collide — newest contact first */
static void world_collide(rem2d_handle* h, World* w, Counters* cnt) {
    for (int i = w->nc - 1; i >= 0; --i) {
        Contact* c = &w->contacts[i];
        Body* B = &w->bodies[c->body];
        if (!B->awake) continue;                     /* static side is never "active" */
        if (!aabb_overlap(h->efat[c->edge], B->fat)) { world_destroy_contact(w, i); continue; }
        contact_update(h, w, c, cnt);
    }
}

/* ---------------------------------------------------------------- contact solver (A.5, A.6, E.4, E.5) */
typedef struct { V2 rA, rB; float normalImpulse, tangentImpulse, normalMass, tangentMass, velocityBias; } VCPoint;
typedef struct {
    VCPoint points[2];
    V2 normal;
    float nm_exx, nm_exy, nm_eyx, nm_eyy;   /* normalMass (2x2) */
    float k_exx, k_exy, k_eyx, k_eyy;       /* K */
    int indexA, indexB;
    float invMassA, invMassB, invIA, invIB, friction, restitution, tangentSpeed;
    int pointCount, contactIndex;
} VelCon;
typedef struct {
    V2 localPoints[2], localNormal, localPoint;
    int indexA, indexB;
    float invMassA, invMassB;
    V2 localCenterA, localCenterB;
    float invIA, invIB;
    int type;
    float radiusA, radiusB;
    int pointCount;
} PosCon;
typedef struct { V2 c; float a; } Position;
typedef struct { V2 v; float w; } Velocity;

/* Island body table: index < nb -> dynamic module body; index >= nb -> static terrain body (all zero) */
#define ISL_MAX_BODIES 384      /* <= 64 modules + the static edge bodies they touch */
#define ISL_MAX_CONTACTS 320
typedef struct {
    int count;
    int bodyIdx[ISL_MAX_BODIES]; /* >= 0: module body index, < 0: static edge -(e+1) */
    Position pos[ISL_MAX_BODIES];
    Velocity vel[ISL_MAX_BODIES];
    int ncontacts;
    int contactIdx[ISL_MAX_CONTACTS];
    VelCon vc[ISL_MAX_CONTACTS];
    PosCon pc[ISL_MAX_CONTACTS];
    int njoints;
    int jointIdx[64];
} Island;

static void world_manifold(const Manifold* m, Xf xfA, float radiusA, Xf xfB, float radiusB, V2* normalOut, V2 points[2]) {
    if (m->pointCount == 0) return;
    if (m->type == M_CIRCLES) {
        V2 normal = v2(1.0f, 0.0f);
        V2 pointA = xmul(xfA, m->localPoint), pointB = xmul(xfB, m->points[0].localPoint);
        V2 d = vsub(pointA, pointB);
        if (vdot(d, d) > B2_EPSILON * B2_EPSILON) { normal = vsub(pointB, pointA); vnormalize(&normal); }
        V2 cA = vadd(pointA, vscale(radiusA, normal)), cB = vsub(pointB, vscale(radiusB, normal));
        points[0] = vscale(0.5f, vadd(cA, cB));
        *normalOut = normal;
    } else if (m->type == M_FACE_A) {
        V2 normal = rmul(xfA.q, m->localNormal);
        V2 planePoint = xmul(xfA, m->localPoint);
        for (int i = 0; i < m->pointCount; ++i) {
            V2 clipPoint = xmul(xfB, m->points[i].localPoint);
            V2 cA = vadd(clipPoint, vscale(radiusA - vdot(vsub(clipPoint, planePoint), normal), normal));
            V2 cB = vsub(clipPoint, vscale(radiusB, normal));
            points[i] = vscale(0.5f, vadd(cA, cB));
        }
        *normalOut = normal;
    } else {
        V2 normal = rmul(xfB.q, m->localNormal);
        V2 planePoint = xmul(xfB, m->localPoint);
        for (int i = 0; i < m->pointCount; ++i) {
            V2 clipPoint = xmul(xfA, m->points[i].localPoint);
            V2 cB = vadd(clipPoint, vscale(radiusB - vdot(vsub(clipPoint, planePoint), normal), normal));
            V2 cA = vsub(clipPoint, vscale(radiusA, normal));
            points[i] = vscale(0.5f, vadd(cA, cB));
        }
        *normalOut = vneg(normal);
    }
}

/* b2ContactSolver constructor */
static void csolver_setup(World* w, Island* is, float dtRatio, int warmStarting, const int* islandIndexOfBody,
                          const int* islandIndexOfContactEdge) {
    for (int i = 0; i < is->ncontacts; ++i) {
        Contact* c = &w->contacts[is->contactIdx[i]];
        Body* B = &w->bodies[c->body];
        VelCon* vc = &is->vc[i];
        PosCon* pc = &is->pc[i];
        vc->friction = c->friction; vc->restitution = c->restitution; vc->tangentSpeed = 0.0f;
        vc->indexA = islandIndexOfContactEdge[i]; vc->indexB = islandIndexOfBody[c->body];
        vc->invMassA = 0.0f; vc->invMassB = B->invMass; vc->invIA = 0.0f; vc->invIB = B->invI;
        vc->contactIndex = i; vc->pointCount = c->m.pointCount;
        vc->k_exx = vc->k_exy = vc->k_eyx = vc->k_eyy = 0.0f;
        vc->nm_exx = vc->nm_exy = vc->nm_eyx = vc->nm_eyy = 0.0f;
        pc->indexA = vc->indexA; pc->indexB = vc->indexB;
        pc->invMassA = 0.0f; pc->invMassB = B->invMass;
        pc->localCenterA = v2(0.0f, 0.0f); pc->localCenterB = B->sweep.localCenter;
        pc->invIA = 0.0f; pc->invIB = B->invI;
        pc->localNormal = c->m.localNormal; pc->localPoint = c->m.localPoint;
        pc->pointCount = c->m.pointCount;
        pc->radiusA = B2_POLYGON_RADIUS; pc->radiusB = B->radius;
        pc->type = c->m.type;
        for (int j = 0; j < c->m.pointCount; ++j) {
            ManifoldPoint* cp = &c->m.points[j];
            VCPoint* vcp = &vc->points[j];
            if (warmStarting) {
                vcp->normalImpulse = dtRatio * cp->normalImpulse;
                vcp->tangentImpulse = dtRatio * cp->tangentImpulse;
            } else { vcp->normalImpulse = 0.0f; vcp->tangentImpulse = 0.0f; }
            vcp->rA = v2(0.0f, 0.0f); vcp->rB = v2(0.0f, 0.0f);
            vcp->normalMass = 0.0f; vcp->tangentMass = 0.0f; vcp->velocityBias = 0.0f;
            pc->localPoints[j] = cp->localPoint;
        }
    }
}

static void csolver_init_velocity(World* w, Island* is) {
    for (int i = 0; i < is->ncontacts; ++i) {
        VelCon* vc = &is->vc[i];
        PosCon* pc = &is->pc[i];
        const Manifold* m = &w->contacts[is->contactIdx[vc->contactIndex]].m;
        float radiusA = pc->radiusA, radiusB = pc->radiusB;
        int indexA = vc->indexA, indexB = vc->indexB;
        float mA = vc->invMassA, mB = vc->invMassB, iA = vc->invIA, iB = vc->invIB;
        V2 localCenterA = pc->localCenterA, localCenterB = pc->localCenterB;
        V2 cA = is->pos[indexA].c; float aA = is->pos[indexA].a;
        V2 vA = is->vel[indexA].v; float wA = is->vel[indexA].w;
        V2 cB = is->pos[indexB].c; float aB = is->pos[indexB].a;
        V2 vB = is->vel[indexB].v; float wB = is->vel[indexB].w;
        Xf xfA, xfB;
        xfA.q = rot_set(aA); xfB.q = rot_set(aB);
        xfA.p = vsub(cA, rmul(xfA.q, localCenterA));
        xfB.p = vsub(cB, rmul(xfB.q, localCenterB));
        V2 wpoints[2];
        world_manifold(m, xfA, radiusA, xfB, radiusB, &vc->normal, wpoints);
        int pointCount = vc->pointCount;
        for (int j = 0; j < pointCount; ++j) {
            VCPoint* vcp = &vc->points[j];
            vcp->rA = vsub(wpoints[j], cA);
            vcp->rB = vsub(wpoints[j], cB);
            float rnA = vcross(vcp->rA, vc->normal), rnB = vcross(vcp->rB, vc->normal);
            float kNormal = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
            vcp->normalMass = kNormal > 0.0f ? 1.0f / kNormal : 0.0f;
            V2 tangent = vcross_vs(vc->normal, 1.0f);
            float rtA = vcross(vcp->rA, tangent), rtB = vcross(vcp->rB, tangent);
            float kTangent = mA + mB + iA * rtA * rtA + iB * rtB * rtB;
            vcp->tangentMass = kTangent > 0.0f ? 1.0f / kTangent : 0.0f;
            vcp->velocityBias = 0.0f;
            float vRel = vdot(vc->normal, vsub(vsub(vadd(vB, vcross_sv(wB, vcp->rB)), vA), vcross_sv(wA, vcp->rA)));
            if (vRel < -B2_VELOCITY_THRESHOLD) vcp->velocityBias = -vc->restitution * vRel;
        }
        if (vc->pointCount == 2) {
            VCPoint* vcp1 = &vc->points[0];
            VCPoint* vcp2 = &vc->points[1];
            float rn1A = vcross(vcp1->rA, vc->normal), rn1B = vcross(vcp1->rB, vc->normal);
            float rn2A = vcross(vcp2->rA, vc->normal), rn2B = vcross(vcp2->rB, vc->normal);
            float k11 = mA + mB + iA * rn1A * rn1A + iB * rn1B * rn1B;
            float k22 = mA + mB + iA * rn2A * rn2A + iB * rn2B * rn2B;
            float k12 = mA + mB + iA * rn1A * rn2A + iB * rn1B * rn2B;
            const float k_maxConditionNumber = 1000.0f;
            if (k11 * k11 < k_maxConditionNumber * (k11 * k22 - k12 * k12)) {
                vc->k_exx = k11; vc->k_exy = k12; vc->k_eyx = k12; vc->k_eyy = k22;
                /* b2Mat22::GetInverse */
                float a = k11, b = k12, cc = k12, d = k22;
                float det = a * d - b * cc;
                if (det != 0.0f) det = 1.0f / det;
                vc->nm_exx = det * d; vc->nm_eyx = -det * b;
                vc->nm_exy = -det * cc; vc->nm_eyy = det * a;
            } else {
                vc->pointCount = 1;
            }
        }
    }
}

static void csolver_warm_start(Island* is) {
    for (int i = 0; i < is->ncontacts; ++i) {
        VelCon* vc = &is->vc[i];
        int indexA = vc->indexA, indexB = vc->indexB;
        float mA = vc->invMassA, iA = vc->invIA, mB = vc->invMassB, iB = vc->invIB;
        V2 vA = is->vel[indexA].v; float wA = is->vel[indexA].w;
        V2 vB = is->vel[indexB].v; float wB = is->vel[indexB].w;
        V2 normal = vc->normal, tangent = vcross_vs(normal, 1.0f);
        for (int j = 0; j < vc->pointCount; ++j) {
            VCPoint* vcp = &vc->points[j];
            V2 P = vadd(vscale(vcp->normalImpulse, normal), vscale(vcp->tangentImpulse, tangent));
            wA -= iA * vcross(vcp->rA, P);
            vA = vsub(vA, vscale(mA, P));
            wB += iB * vcross(vcp->rB, P);
            vB = vadd(vB, vscale(mB, P));
        }
        is->vel[indexA].v = vA; is->vel[indexA].w = wA;
        is->vel[indexB].v = vB; is->vel[indexB].w = wB;
    }
}

static void csolver_solve_velocity(Island* is, Counters* cnt) {
    for (int i = 0; i < is->ncontacts; ++i) {
        VelCon* vc = &is->vc[i];
        int indexA = vc->indexA, indexB = vc->indexB;
        float mA = vc->invMassA, iA = vc->invIA, mB = vc->invMassB, iB = vc->invIB;
        int pointCount = vc->pointCount;
        V2 vA = is->vel[indexA].v; float wA = is->vel[indexA].w;
        V2 vB = is->vel[indexB].v; float wB = is->vel[indexB].w;
        V2 normal = vc->normal, tangent = vcross_vs(normal, 1.0f);
        float friction = vc->friction;
        for (int j = 0; j < pointCount; ++j) {
            VCPoint* vcp = &vc->points[j];
            V2 dv = vsub(vsub(vadd(vB, vcross_sv(wB, vcp->rB)), vA), vcross_sv(wA, vcp->rA));
            float vt = vdot(dv, tangent) - vc->tangentSpeed;
            float lambda = vcp->tangentMass * (-vt);
            float maxFriction = friction * vcp->normalImpulse;
            float newImpulse = fclamp(vcp->tangentImpulse + lambda, -maxFriction, maxFriction);
            lambda = newImpulse - vcp->tangentImpulse;
            vcp->tangentImpulse = newImpulse;
            V2 P = vscale(lambda, tangent);
            vA = vsub(vA, vscale(mA, P)); wA -= iA * vcross(vcp->rA, P);
            vB = vadd(vB, vscale(mB, P)); wB += iB * vcross(vcp->rB, P);
        }
        if (vc->pointCount == 1) {
            cnt->c[REM2D_CNT_P1_VSOLVES]++;
            VCPoint* vcp = &vc->points[0];
            V2 dv = vsub(vsub(vadd(vB, vcross_sv(wB, vcp->rB)), vA), vcross_sv(wA, vcp->rA));
            float vn = vdot(dv, normal);
            float lambda = -vcp->normalMass * (vn - vcp->velocityBias);
            float newImpulse = fmax2(vcp->normalImpulse + lambda, 0.0f);
            lambda = newImpulse - vcp->normalImpulse;
            vcp->normalImpulse = newImpulse;
            V2 P = vscale(lambda, normal);
            vA = vsub(vA, vscale(mA, P)); wA -= iA * vcross(vcp->rA, P);
            vB = vadd(vB, vscale(mB, P)); wB += iB * vcross(vcp->rB, P);
        } else {
            cnt->c[REM2D_CNT_M2_VSOLVES]++;
            VCPoint* cp1 = &vc->points[0];
            VCPoint* cp2 = &vc->points[1];
            V2 a = v2(cp1->normalImpulse, cp2->normalImpulse);
            V2 dv1 = vsub(vsub(vadd(vB, vcross_sv(wB, cp1->rB)), vA), vcross_sv(wA, cp1->rA));
            V2 dv2 = vsub(vsub(vadd(vB, vcross_sv(wB, cp2->rB)), vA), vcross_sv(wA, cp2->rA));
            float vn1 = vdot(dv1, normal), vn2 = vdot(dv2, normal);
            V2 b = v2(vn1 - cp1->velocityBias, vn2 - cp2->velocityBias);
            /* b -= K a */
            b = vsub(b, v2(vc->k_exx * a.x + vc->k_eyx * a.y, vc->k_exy * a.x + vc->k_eyy * a.y));
            V2 x;
            int solved = 0;
            /* case 1 */
            x = vneg(v2(vc->nm_exx * b.x + vc->nm_eyx * b.y, vc->nm_exy * b.x + vc->nm_eyy * b.y));
            if (x.x >= 0.0f && x.y >= 0.0f) solved = 1;
            if (!solved) { /* case 2 */
                x.x = -cp1->normalMass * b.x; x.y = 0.0f;
                vn1 = 0.0f; vn2 = vc->k_exy * x.x + b.y;
                if (x.x >= 0.0f && vn2 >= 0.0f) solved = 1;
            }
            if (!solved) { /* case 3 */
                x.x = 0.0f; x.y = -cp2->normalMass * b.y;
                vn1 = vc->k_eyx * x.y + b.x; vn2 = 0.0f;
                if (x.y >= 0.0f && vn1 >= 0.0f) solved = 1;
            }
            if (!solved) { /* case 4 */
                x.x = 0.0f; x.y = 0.0f;
                vn1 = b.x; vn2 = b.y;
                if (vn1 >= 0.0f && vn2 >= 0.0f) solved = 1;
            }
            if (solved) {
                V2 d = vsub(x, a);
                V2 P1 = vscale(d.x, normal), P2 = vscale(d.y, normal);
                vA = vsub(vA, vscale(mA, vadd(P1, P2)));
                wA -= iA * (vcross(cp1->rA, P1) + vcross(cp2->rA, P2));
                vB = vadd(vB, vscale(mB, vadd(P1, P2)));
                wB += iB * (vcross(cp1->rB, P1) + vcross(cp2->rB, P2));
                cp1->normalImpulse = x.x; cp2->normalImpulse = x.y;
            }
        }
        is->vel[indexA].v = vA; is->vel[indexA].w = wA;
        is->vel[indexB].v = vB; is->vel[indexB].w = wB;
    }
}

static void csolver_store_impulses(World* w, Island* is) {
    for (int i = 0; i < is->ncontacts; ++i) {
        VelCon* vc = &is->vc[i];
        Manifold* m = &w->contacts[is->contactIdx[vc->contactIndex]].m;
        for (int j = 0; j < vc->pointCount; ++j) {
            m->points[j].normalImpulse = vc->points[j].normalImpulse;
            m->points[j].tangentImpulse = vc->points[j].tangentImpulse;
        }
    }
}

static void psm_init(const PosCon* pc, Xf xfA, Xf xfB, int index, V2* normal, V2* point, float* separation) {
    if (pc->type == M_CIRCLES) {
        V2 pointA = xmul(xfA, pc->localPoint), pointB = xmul(xfB, pc->localPoints[0]);
        *normal = vsub(pointB, pointA);
        vnormalize(normal);
        *point = vscale(0.5f, vadd(pointA, pointB));
        *separation = vdot(vsub(pointB, pointA), *normal) - pc->radiusA - pc->radiusB;
    } else if (pc->type == M_FACE_A) {
        *normal = rmul(xfA.q, pc->localNormal);
        V2 planePoint = xmul(xfA, pc->localPoint);
        V2 clipPoint = xmul(xfB, pc->localPoints[index]);
        *separation = vdot(vsub(clipPoint, planePoint), *normal) - pc->radiusA - pc->radiusB;
        *point = clipPoint;
    } else {
        *normal = rmul(xfB.q, pc->localNormal);
        V2 planePoint = xmul(xfB, pc->localPoint);
        V2 clipPoint = xmul(xfA, pc->localPoints[index]);
        *separation = vdot(vsub(clipPoint, planePoint), *normal) - pc->radiusA - pc->radiusB;
        *point = clipPoint;
        *normal = vneg(*normal);
    }
}

/* SolvePositionConstraints (toi = 0) / SolveTOIPositionConstraints (toi = 1) */
static int csolver_solve_position(Island* is, int toi, int toiIndexA, int toiIndexB, Counters* cnt) {
    float minSeparation = 0.0f;
    for (int i = 0; i < is->ncontacts; ++i) {
        PosCon* pc = &is->pc[i];
        int indexA = pc->indexA, indexB = pc->indexB;
        V2 localCenterA = pc->localCenterA, localCenterB = pc->localCenterB;
        float mA, iA, mB, iB;
        if (!toi) { mA = pc->invMassA; iA = pc->invIA; mB = pc->invMassB; iB = pc->invIB; }
        else {
            mA = 0.0f; iA = 0.0f;
            if (indexA == toiIndexA || indexA == toiIndexB) { mA = pc->invMassA; iA = pc->invIA; }
            mB = 0.0f; iB = 0.0f;
            if (indexB == toiIndexA || indexB == toiIndexB) { mB = pc->invMassB; iB = pc->invIB; }
        }
        V2 cA = is->pos[indexA].c; float aA = is->pos[indexA].a;
        V2 cB = is->pos[indexB].c; float aB = is->pos[indexB].a;
        for (int j = 0; j < pc->pointCount; ++j) {
            cnt->c[REM2D_CNT_POINT_PSOLVES]++;
            Xf xfA, xfB;
            xfA.q = rot_set(aA); xfB.q = rot_set(aB);
            xfA.p = vsub(cA, rmul(xfA.q, localCenterA));
            xfB.p = vsub(cB, rmul(xfB.q, localCenterB));
            V2 normal, point; float separation;
            psm_init(pc, xfA, xfB, j, &normal, &point, &separation);
            V2 rA = vsub(point, cA), rB = vsub(point, cB);
            minSeparation = fmin2(minSeparation, separation);
            float C = fclamp((toi ? B2_TOI_BAUMGARTE : B2_BAUMGARTE) * (separation + B2_LINEAR_SLOP), -B2_MAX_LINEAR_CORRECTION, 0.0f);
            float rnA = vcross(rA, normal), rnB = vcross(rB, normal);
            float K = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
            float impulse = K > 0.0f ? -C / K : 0.0f;
            V2 P = vscale(impulse, normal);
            cA = vsub(cA, vscale(mA, P)); aA -= iA * vcross(rA, P);
            cB = vadd(cB, vscale(mB, P)); aB += iB * vcross(rB, P);
        }
        is->pos[indexA].c = cA; is->pos[indexA].a = aA;
        is->pos[indexB].c = cB; is->pos[indexB].a = aB;
    }
    return minSeparation >= (toi ? -1.5f * B2_LINEAR_SLOP : -3.0f * B2_LINEAR_SLOP);
}

/* ---------------------------------------------------------------- revolute joint (A.7, E.6) */
static inline V3 v3cross(V3 a, V3 b) { V3 r = {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; return r; }
static inline float v3dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline V3 mat33_solve33(const Joint* j, V3 b) {
    float det = v3dot(j->mex, v3cross(j->mey, j->mez));
    if (det != 0.0f) det = 1.0f / det;
    V3 x;
    x.x = det * v3dot(b, v3cross(j->mey, j->mez));
    x.y = det * v3dot(j->mex, v3cross(b, j->mez));
    x.z = det * v3dot(j->mex, v3cross(j->mey, b));
    return x;
}
static inline V2 mat33_solve22(const Joint* j, V2 b) {
    float a11 = j->mex.x, a12 = j->mey.x, a21 = j->mex.y, a22 = j->mey.y;
    float det = a11 * a22 - a12 * a21;
    if (det != 0.0f) det = 1.0f / det;
    return v2(det * (a22 * b.x - a12 * b.y), det * (a11 * b.y - a21 * b.x));
}

static void joint_init_velocity(World* w, Island* is, Joint* j, float dtRatio) {
    Body* bA = &w->bodies[j->bodyA];
    Body* bB = &w->bodies[j->bodyB];
    j->indexA = bA->islandIndex; j->indexB = bB->islandIndex;
    j->localCenterA = bA->sweep.localCenter; j->localCenterB = bB->sweep.localCenter;
    j->invMassA = bA->invMass; j->invMassB = bB->invMass;
    j->invIA = bA->invI; j->invIB = bB->invI;
    float aA = is->pos[j->indexA].a; V2 vA = is->vel[j->indexA].v; float wA = is->vel[j->indexA].w;
    float aB = is->pos[j->indexB].a; V2 vB = is->vel[j->indexB].v; float wB = is->vel[j->indexB].w;
    Rot qA = rot_set(aA), qB = rot_set(aB);
    j->rA = rmul(qA, vsub(j->localAnchorA, j->localCenterA));
    j->rB = rmul(qB, vsub(j->localAnchorB, j->localCenterB));
    float mA = j->invMassA, mB = j->invMassB, iA = j->invIA, iB = j->invIB;
    int fixedRotation = (iA + iB == 0.0f);
    j->mex.x = mA + mB + j->rA.y * j->rA.y * iA + j->rB.y * j->rB.y * iB;
    j->mey.x = -j->rA.y * j->rA.x * iA - j->rB.y * j->rB.x * iB;
    j->mez.x = -j->rA.y * iA - j->rB.y * iB;
    j->mex.y = j->mey.x;
    j->mey.y = mA + mB + j->rA.x * j->rA.x * iA + j->rB.x * j->rB.x * iB;
    j->mez.y = j->rA.x * iA + j->rB.x * iB;
    j->mex.z = j->mez.x;
    j->mey.z = j->mez.y;
    j->mez.z = iA + iB;
    j->motorMass = iA + iB;
    if (j->motorMass > 0.0f) j->motorMass = 1.0f / j->motorMass;
    if (fixedRotation) j->motorImpulse = 0.0f;
    if (!fixedRotation) {
        float jointAngle = aB - aA - j->referenceAngle;
        if (fabs2(j->upper - j->lower) < 2.0f * B2_ANGULAR_SLOP) j->limitState = LIMIT_EQUAL;
        else if (jointAngle <= j->lower) {
            if (j->limitState != LIMIT_LOWER) j->impulse.z = 0.0f;
            j->limitState = LIMIT_LOWER;
        } else if (jointAngle >= j->upper) {
            if (j->limitState != LIMIT_UPPER) j->impulse.z = 0.0f;
            j->limitState = LIMIT_UPPER;
        } else { j->limitState = LIMIT_INACTIVE; j->impulse.z = 0.0f; }
    } else j->limitState = LIMIT_INACTIVE;
    /* warm starting is always on for the discrete solver */
    j->impulse.x *= dtRatio; j->impulse.y *= dtRatio; j->impulse.z *= dtRatio;
    j->motorImpulse *= dtRatio;
    V2 P = v2(j->impulse.x, j->impulse.y);
    vA = vsub(vA, vscale(mA, P));
    wA -= iA * (vcross(j->rA, P) + j->motorImpulse + j->impulse.z);
    vB = vadd(vB, vscale(mB, P));
    wB += iB * (vcross(j->rB, P) + j->motorImpulse + j->impulse.z);
    is->vel[j->indexA].v = vA; is->vel[j->indexA].w = wA;
    is->vel[j->indexB].v = vB; is->vel[j->indexB].w = wB;
}

static void joint_solve_velocity(Island* is, Joint* j, float dt) {
    V2 vA = is->vel[j->indexA].v; float wA = is->vel[j->indexA].w;
    V2 vB = is->vel[j->indexB].v; float wB = is->vel[j->indexB].w;
    float mA = j->invMassA, mB = j->invMassB, iA = j->invIA, iB = j->invIB;
    int fixedRotation = (iA + iB == 0.0f);
    if (j->limitState != LIMIT_EQUAL && !fixedRotation) {
        float Cdot = wB - wA - j->motorSpeed;
        float impulse = -j->motorMass * Cdot;
        float oldImpulse = j->motorImpulse;
        float maxImpulse = dt * j->maxMotorTorque;
        j->motorImpulse = fclamp(oldImpulse + impulse, -maxImpulse, maxImpulse);
        impulse = j->motorImpulse - oldImpulse;
        wA -= iA * impulse;
        wB += iB * impulse;
    }
    if (j->limitState != LIMIT_INACTIVE && !fixedRotation) {
        V2 Cdot1 = vsub(vsub(vadd(vB, vcross_sv(wB, j->rB)), vA), vcross_sv(wA, j->rA));
        float Cdot2 = wB - wA;
        V3 Cdot = {Cdot1.x, Cdot1.y, Cdot2};
        V3 impulse = mat33_solve33(j, Cdot);
        impulse.x = -impulse.x; impulse.y = -impulse.y; impulse.z = -impulse.z;
        if (j->limitState == LIMIT_EQUAL) {
            j->impulse.x += impulse.x; j->impulse.y += impulse.y; j->impulse.z += impulse.z;
        } else if (j->limitState == LIMIT_LOWER) {
            float newImpulse = j->impulse.z + impulse.z;
            if (newImpulse < 0.0f) {
                V2 rhs = vadd(vneg(Cdot1), vscale(j->impulse.z, v2(j->mez.x, j->mez.y)));
                V2 reduced = mat33_solve22(j, rhs);
                impulse.x = reduced.x; impulse.y = reduced.y; impulse.z = -j->impulse.z;
                j->impulse.x += reduced.x; j->impulse.y += reduced.y; j->impulse.z = 0.0f;
            } else {
                j->impulse.x += impulse.x; j->impulse.y += impulse.y; j->impulse.z += impulse.z;
            }
        } else if (j->limitState == LIMIT_UPPER) {
            float newImpulse = j->impulse.z + impulse.z;
            if (newImpulse > 0.0f) {
                V2 rhs = vadd(vneg(Cdot1), vscale(j->impulse.z, v2(j->mez.x, j->mez.y)));
                V2 reduced = mat33_solve22(j, rhs);
                impulse.x = reduced.x; impulse.y = reduced.y; impulse.z = -j->impulse.z;
                j->impulse.x += reduced.x; j->impulse.y += reduced.y; j->impulse.z = 0.0f;
            } else {
                j->impulse.x += impulse.x; j->impulse.y += impulse.y; j->impulse.z += impulse.z;
            }
        }
        V2 P = v2(impulse.x, impulse.y);
        vA = vsub(vA, vscale(mA, P));
        wA -= iA * (vcross(j->rA, P) + impulse.z);
        vB = vadd(vB, vscale(mB, P));
        wB += iB * (vcross(j->rB, P) + impulse.z);
    } else {
        V2 Cdot = vsub(vsub(vadd(vB, vcross_sv(wB, j->rB)), vA), vcross_sv(wA, j->rA));
        V2 impulse = mat33_solve22(j, vneg(Cdot));
        j->impulse.x += impulse.x; j->impulse.y += impulse.y;
        vA = vsub(vA, vscale(mA, impulse));
        wA -= iA * vcross(j->rA, impulse);
        vB = vadd(vB, vscale(mB, impulse));
        wB += iB * vcross(j->rB, impulse);
    }
    is->vel[j->indexA].v = vA; is->vel[j->indexA].w = wA;
    is->vel[j->indexB].v = vB; is->vel[j->indexB].w = wB;
}

static int joint_solve_position(Island* is, Joint* j) {
    V2 cA = is->pos[j->indexA].c; float aA = is->pos[j->indexA].a;
    V2 cB = is->pos[j->indexB].c; float aB = is->pos[j->indexB].a;
    float angularError = 0.0f, positionError = 0.0f;
    int fixedRotation = (j->invIA + j->invIB == 0.0f);
    if (j->limitState != LIMIT_INACTIVE && !fixedRotation) {
        float angle = aB - aA - j->referenceAngle;
        float limitImpulse = 0.0f;
        if (j->limitState == LIMIT_EQUAL) {
            float C = fclamp(angle - j->lower, -B2_MAX_ANGULAR_CORRECTION, B2_MAX_ANGULAR_CORRECTION);
            limitImpulse = -j->motorMass * C;
            angularError = fabs2(C);
        } else if (j->limitState == LIMIT_LOWER) {
            float C = angle - j->lower;
            angularError = -C;
            C = fclamp(C + B2_ANGULAR_SLOP, -B2_MAX_ANGULAR_CORRECTION, 0.0f);
            limitImpulse = -j->motorMass * C;
        } else if (j->limitState == LIMIT_UPPER) {
            float C = angle - j->upper;
            angularError = C;
            C = fclamp(C - B2_ANGULAR_SLOP, 0.0f, B2_MAX_ANGULAR_CORRECTION);
            limitImpulse = -j->motorMass * C;
        }
        aA -= j->invIA * limitImpulse;
        aB += j->invIB * limitImpulse;
    }
    {
        Rot qA = rot_set(aA), qB = rot_set(aB);
        V2 rA = rmul(qA, vsub(j->localAnchorA, j->localCenterA));
        V2 rB = rmul(qB, vsub(j->localAnchorB, j->localCenterB));
        V2 C = vsub(vsub(vadd(cB, rB), cA), rA);
        positionError = vlen(C);
        float mA = j->invMassA, mB = j->invMassB, iA = j->invIA, iB = j->invIB;
        float kexx = mA + mB + iA * rA.y * rA.y + iB * rB.y * rB.y;
        float kexy = -iA * rA.x * rA.y - iB * rB.x * rB.y;
        float keyx = kexy;
        float keyy = mA + mB + iA * rA.x * rA.x + iB * rB.x * rB.x;
        /* impulse = -K.Solve(C) */
        float a11 = kexx, a12 = keyx, a21 = kexy, a22 = keyy;
        float det = a11 * a22 - a12 * a21;
        if (det != 0.0f) det = 1.0f / det;
        V2 impulse = vneg(v2(det * (a22 * C.x - a12 * C.y), det * (a11 * C.y - a21 * C.x)));
        cA = vsub(cA, vscale(mA, impulse));
        aA -= iA * vcross(rA, impulse);
        cB = vadd(cB, vscale(mB, impulse));
        aB += iB * vcross(rB, impulse);
    }
    is->pos[j->indexA].c = cA; is->pos[j->indexA].a = aA;
    is->pos[j->indexB].c = cB; is->pos[j->indexB].a = aB;
    return positionError <= B2_LINEAR_SLOP && angularError <= B2_ANGULAR_SLOP;
}

/* ---------------------------------------------------------------- b2World::Solve + b2Island::Solve (A.5, A.9, E.3) */
static void island_solve(rem2d_handle* h, World* w, Island* is, float dt, float dtRatio, Counters* cnt,
                         const int* islandIndexOfBody, const int* islandIndexOfContactEdge) {
    float hdt = dt;
    V2 gravity = v2(0.0f, h->cfg.gravity_y);
    for (int i = 0; i < is->count; ++i) {
        if (is->bodyIdx[i] < 0) {          /* static terrain body */
            is->pos[i].c = v2(0.0f, 0.0f); is->pos[i].a = 0.0f;
            is->vel[i].v = v2(0.0f, 0.0f); is->vel[i].w = 0.0f;
            continue;
        }
        Body* b = &w->bodies[is->bodyIdx[i]];
        V2 c = b->sweep.c; float a = b->sweep.a;
        V2 v = b->v; float ww = b->w;
        b->sweep.c0 = b->sweep.c; b->sweep.a0 = b->sweep.a;
        /* v += h * (gravityScale * gravity + invMass * force); w += h * invI * torque */
        V2 force = v2(0.0f, 0.0f);
        v = vadd(v, vscale(hdt, vadd(vscale(1.0f, gravity), vscale(b->invMass, force))));
        ww += hdt * b->invI * 0.0f;
        v = vscale(1.0f / (1.0f + hdt * 0.0f), v);
        ww *= 1.0f / (1.0f + hdt * 0.0f);
        is->pos[i].c = c; is->pos[i].a = a;
        is->vel[i].v = v; is->vel[i].w = ww;
        cnt->c[REM2D_CNT_BODY_TICKS]++;
    }
    csolver_setup(w, is, dtRatio, 1, islandIndexOfBody, islandIndexOfContactEdge);
    csolver_init_velocity(w, is);
    csolver_warm_start(is);
    for (int i = 0; i < is->njoints; ++i) joint_init_velocity(w, is, &w->joints[is->jointIdx[i]], dtRatio);
    for (int it = 0; it < h->cfg.velocity_iterations; ++it) {
        for (int j = 0; j < is->njoints; ++j) joint_solve_velocity(is, &w->joints[is->jointIdx[j]], dt);
        cnt->c[REM2D_CNT_JOINT_VSOLVES] += (uint64_t)is->njoints;
        csolver_solve_velocity(is, cnt);
    }
    csolver_store_impulses(w, is);
    for (int i = 0; i < is->count; ++i) {
        V2 c = is->pos[i].c; float a = is->pos[i].a;
        V2 v = is->vel[i].v; float ww = is->vel[i].w;
        V2 translation = vscale(hdt, v);
        if (vdot(translation, translation) > B2_MAX_TRANSLATION_SQ) {
            float ratio = B2_MAX_TRANSLATION / vlen(translation);
            v = vscale(ratio, v);
        }
        float rotation = hdt * ww;
        if (rotation * rotation > B2_MAX_ROTATION_SQ) {
            float ratio = B2_MAX_ROTATION / fabs2(rotation);
            ww *= ratio;
        }
        c = vadd(c, vscale(hdt, v));
        a += hdt * ww;
        is->pos[i].c = c; is->pos[i].a = a;
        is->vel[i].v = v; is->vel[i].w = ww;
    }
    int positionSolved = 0;
    for (int it = 0; it < h->cfg.position_iterations; ++it) {
        int contactsOkay = csolver_solve_position(is, 0, 0, 0, cnt);
        int jointsOkay = 1;
        for (int j = 0; j < is->njoints; ++j) {
            int ok = joint_solve_position(is, &w->joints[is->jointIdx[j]]);
            jointsOkay = jointsOkay && ok;
        }
        cnt->c[REM2D_CNT_JOINT_PSOLVES] += (uint64_t)is->njoints;
        if (contactsOkay && jointsOkay) { positionSolved = 1; break; }
    }
    for (int i = 0; i < is->count; ++i) {
        if (is->bodyIdx[i] < 0) continue;
        Body* b = &w->bodies[is->bodyIdx[i]];
        b->sweep.c = is->pos[i].c; b->sweep.a = is->pos[i].a;
        b->v = is->vel[i].v; b->w = is->vel[i].w;
        body_sync_transform(b);
    }
    if (h->cfg.allow_sleep) {
        float minSleepTime = B2_MAX_FLOAT;
        const float linTolSqr = B2_LINEAR_SLEEP_TOL * B2_LINEAR_SLEEP_TOL;
        const float angTolSqr = B2_ANGULAR_SLEEP_TOL * B2_ANGULAR_SLEEP_TOL;
        for (int i = 0; i < is->count; ++i) {
            if (is->bodyIdx[i] < 0) continue;
            Body* b = &w->bodies[is->bodyIdx[i]];
            if (b->w * b->w > angTolSqr || vdot(b->v, b->v) > linTolSqr) { b->sleepTime = 0.0f; minSleepTime = 0.0f; }
            else { b->sleepTime += hdt; minSleepTime = fmin2(minSleepTime, b->sleepTime); }
        }
        if (minSleepTime >= B2_TIME_TO_SLEEP && positionSolved) {
            for (int i = 0; i < is->count; ++i)
                if (is->bodyIdx[i] >= 0) body_set_awake(&w->bodies[is->bodyIdx[i]], 0);
        }
    }
}

static void world_solve(rem2d_handle* h, World* w, float dt, float dtRatio, Counters* cnt) {
    for (int b = 0; b < w->nb; ++b) w->bodies[b].islandFlag = 0;
    for (int i = 0; i < w->nc; ++i) w->contacts[i].flags &= ~CF_ISLAND;
    for (int j = 0; j < w->nj; ++j) w->joints[j].islandFlag = 0;
    static __thread Island is_storage;
    Island* is = &is_storage;
    int islandIndexOfBody[64];
    int islandIndexOfContactEdge[ISL_MAX_CONTACTS];
    int stack[ISL_MAX_BODIES];
    /* seeds: world body list, newest first; terrain bodies (older) are static and never seeds */
    for (int seed = w->nb - 1; seed >= 0; --seed) {
        Body* S = &w->bodies[seed];
        if (S->islandFlag) continue;
        if (!S->awake) continue;
        is->count = 0; is->ncontacts = 0; is->njoints = 0;
        int sp = 0;
        stack[sp++] = seed;
        S->islandFlag = 1;
        while (sp > 0) {
            int bi = stack[--sp];
            if (bi < 0) {      /* static terrain body: joins the island, propagates nothing */
                is->bodyIdx[is->count++] = bi;
                continue;
            }
            Body* b = &w->bodies[bi];
            b->islandIndex = is->count;
            islandIndexOfBody[bi] = is->count;
            is->bodyIdx[is->count++] = bi;
            body_set_awake(b, 1);
            /* contact list of the body, newest first */
            for (int ci = w->nc - 1; ci >= 0; --ci) {
                Contact* c = &w->contacts[ci];
                if (c->body != bi) continue;
                if (c->flags & CF_ISLAND) continue;
                if (!(c->flags & CF_ENABLED) || !(c->flags & CF_TOUCHING)) continue;
                if (is->ncontacts == ISL_MAX_CONTACTS || is->count + sp >= ISL_MAX_BODIES - 1) { w->overflow = 1; continue; }
                c->flags |= CF_ISLAND;
                /* the other body is this edge's static body. Each edge is its own b2Body; its island flag
                 * is cleared after every island, and within an island it is added once. */
                int already = -1;
                for (int k = 0; k < is->ncontacts; ++k)
                    if (w->contacts[is->contactIdx[k]].edge == c->edge) { already = k; break; }
                is->contactIdx[is->ncontacts] = ci;
                if (already >= 0) islandIndexOfContactEdge[is->ncontacts] = -1000 - already; /* resolved below */
                else { islandIndexOfContactEdge[is->ncontacts] = -1; stack[sp++] = -(c->edge + 1); }
                is->ncontacts++;
            }
            /* joint list of the body, newest first: joints to children (descending), then to the parent */
            for (int ji = w->nj - 1; ji >= 0; --ji) {
                Joint* j = &w->joints[ji];
                if (j->bodyA != bi && j->bodyB != bi) continue;
                if (j->islandFlag) continue;
                int other = j->bodyA == bi ? j->bodyB : j->bodyA;
                is->jointIdx[is->njoints++] = ji;
                j->islandFlag = 1;
                if (w->bodies[other].islandFlag) continue;
                stack[sp++] = other;
                w->bodies[other].islandFlag = 1;
            }
        }
        /* resolve island indices of the static edge bodies (they were appended when popped) */
        for (int k = 0; k < is->ncontacts; ++k) {
            int e = w->contacts[is->contactIdx[k]].edge;
            for (int i = 0; i < is->count; ++i)
                if (is->bodyIdx[i] == -(e + 1)) { islandIndexOfContactEdge[k] = i; break; }
        }
        island_solve(h, w, is, dt, dtRatio, cnt, islandIndexOfBody, islandIndexOfContactEdge);
    }
    /* synchronize fixtures of island bodies (body list order, newest first), then look for new contacts */
    for (int b = w->nb - 1; b >= 0; --b) {
        if (!w->bodies[b].islandFlag) continue;
        body_synchronize_fixtures(&w->bodies[b]);
    }
    world_find_new_contacts(h, w);
}

/* ---------------------------------------------------------------- GJK distance + time of impact (A.8, E.9) */
typedef struct { const V2* verts; int count; float radius; } Proxy;
typedef struct { float metric; int count; int indexA[3], indexB[3]; } SimplexCache;
typedef struct { V2 wA, wB, w; float a; int indexA, indexB; } SimplexVertex;
typedef struct { SimplexVertex v[3]; int count; } Simplex;

static inline int proxy_support(const Proxy* p, V2 d) {
    int best = 0;
    float bestValue = vdot(p->verts[0], d);
    for (int i = 1; i < p->count; ++i) {
        float value = vdot(p->verts[i], d);
        if (value > bestValue) { best = i; bestValue = value; }
    }
    return best;
}
static float simplex_metric(const Simplex* s) {
    if (s->count == 2) return vlen(vsub(s->v[0].w, s->v[1].w));
    if (s->count == 3) return vcross(vsub(s->v[1].w, s->v[0].w), vsub(s->v[2].w, s->v[0].w));
    return 0.0f;
}
static void simplex_solve2(Simplex* s) {
    V2 w1 = s->v[0].w, w2 = s->v[1].w, e12 = vsub(w2, w1);
    float d12_2 = -vdot(w1, e12);
    if (d12_2 <= 0.0f) { s->v[0].a = 1.0f; s->count = 1; return; }
    float d12_1 = vdot(w2, e12);
    if (d12_1 <= 0.0f) { s->v[1].a = 1.0f; s->count = 1; s->v[0] = s->v[1]; return; }
    float inv_d12 = 1.0f / (d12_1 + d12_2);
    s->v[0].a = d12_1 * inv_d12; s->v[1].a = d12_2 * inv_d12; s->count = 2;
}
static void simplex_solve3(Simplex* s) {
    V2 w1 = s->v[0].w, w2 = s->v[1].w, w3 = s->v[2].w;
    V2 e12 = vsub(w2, w1);
    float w1e12 = vdot(w1, e12), w2e12 = vdot(w2, e12);
    float d12_1 = w2e12, d12_2 = -w1e12;
    V2 e13 = vsub(w3, w1);
    float w1e13 = vdot(w1, e13), w3e13 = vdot(w3, e13);
    float d13_1 = w3e13, d13_2 = -w1e13;
    V2 e23 = vsub(w3, w2);
    float w2e23 = vdot(w2, e23), w3e23 = vdot(w3, e23);
    float d23_1 = w3e23, d23_2 = -w2e23;
    float n123 = vcross(e12, e13);
    float d123_1 = n123 * vcross(w2, w3), d123_2 = n123 * vcross(w3, w1), d123_3 = n123 * vcross(w1, w2);
    if (d12_2 <= 0.0f && d13_2 <= 0.0f) { s->v[0].a = 1.0f; s->count = 1; return; }
    if (d12_1 > 0.0f && d12_2 > 0.0f && d123_3 <= 0.0f) {
        float inv = 1.0f / (d12_1 + d12_2);
        s->v[0].a = d12_1 * inv; s->v[1].a = d12_2 * inv; s->count = 2; return;
    }
    if (d13_1 > 0.0f && d13_2 > 0.0f && d123_2 <= 0.0f) {
        float inv = 1.0f / (d13_1 + d13_2);
        s->v[0].a = d13_1 * inv; s->v[2].a = d13_2 * inv; s->count = 2; s->v[1] = s->v[2]; return;
    }
    if (d12_1 <= 0.0f && d23_2 <= 0.0f) { s->v[1].a = 1.0f; s->count = 1; s->v[0] = s->v[1]; return; }
    if (d13_1 <= 0.0f && d23_1 <= 0.0f) { s->v[2].a = 1.0f; s->count = 1; s->v[0] = s->v[2]; return; }
    if (d23_1 > 0.0f && d23_2 > 0.0f && d123_1 <= 0.0f) {
        float inv = 1.0f / (d23_1 + d23_2);
        s->v[1].a = d23_1 * inv; s->v[2].a = d23_2 * inv; s->count = 2; s->v[0] = s->v[2]; return;
    }
    float inv = 1.0f / (d123_1 + d123_2 + d123_3);
    s->v[0].a = d123_1 * inv; s->v[1].a = d123_2 * inv; s->v[2].a = d123_3 * inv; s->count = 3;
}

/* b2Distance with useRadii = false; returns the distance, updates the cache */
static float gjk_distance(SimplexCache* cache, const Proxy* pA, Xf xfA, const Proxy* pB, Xf xfB, Counters* cnt) {
    Simplex s;
    /* ReadCache */
    s.count = cache->count;
    for (int i = 0; i < s.count; ++i) {
        SimplexVertex* v = &s.v[i];
        v->indexA = cache->indexA[i]; v->indexB = cache->indexB[i];
        v->wA = xmul(xfA, pA->verts[v->indexA]);
        v->wB = xmul(xfB, pB->verts[v->indexB]);
        v->w = vsub(v->wB, v->wA);
        v->a = 0.0f;
    }
    if (s.count > 1) {
        float metric1 = cache->metric, metric2 = simplex_metric(&s);
        if (metric2 < 0.5f * metric1 || 2.0f * metric1 < metric2 || metric2 < B2_EPSILON) s.count = 0;
    }
    if (s.count == 0) {
        SimplexVertex* v = &s.v[0];
        v->indexA = 0; v->indexB = 0;
        v->wA = xmul(xfA, pA->verts[0]); v->wB = xmul(xfB, pB->verts[0]);
        v->w = vsub(v->wB, v->wA);
        v->a = 1.0f;
        s.count = 1;
    }
    const int k_maxIters = 20;
    int saveA[3], saveB[3], saveCount = 0;
    int iter = 0;
    while (iter < k_maxIters) {
        saveCount = s.count;
        for (int i = 0; i < saveCount; ++i) { saveA[i] = s.v[i].indexA; saveB[i] = s.v[i].indexB; }
        if (s.count == 2) simplex_solve2(&s);
        else if (s.count == 3) simplex_solve3(&s);
        if (s.count == 3) break;
        /* search direction */
        V2 d;
        if (s.count == 1) d = vneg(s.v[0].w);
        else {
            V2 e12 = vsub(s.v[1].w, s.v[0].w);
            float sgn = vcross(e12, vneg(s.v[0].w));
            d = sgn > 0.0f ? vcross_sv(1.0f, e12) : vcross_vs(e12, 1.0f);
        }
        if (vlen2(d) < B2_EPSILON * B2_EPSILON) break;
        SimplexVertex* vertex = &s.v[s.count];
        vertex->indexA = proxy_support(pA, rmulT(xfA.q, vneg(d)));
        vertex->wA = xmul(xfA, pA->verts[vertex->indexA]);
        vertex->indexB = proxy_support(pB, rmulT(xfB.q, d));
        vertex->wB = xmul(xfB, pB->verts[vertex->indexB]);
        vertex->w = vsub(vertex->wB, vertex->wA);
        ++iter;
        cnt->c[REM2D_CNT_GJK_ITERS]++;
        int duplicate = 0;
        for (int i = 0; i < saveCount; ++i)
            if (vertex->indexA == saveA[i] && vertex->indexB == saveB[i]) { duplicate = 1; break; }
        if (duplicate) break;
        ++s.count;
    }
    /* witness points */
    V2 a, b;
    if (s.count == 1) { a = s.v[0].wA; b = s.v[0].wB; }
    else if (s.count == 2) {
        a = vadd(vscale(s.v[0].a, s.v[0].wA), vscale(s.v[1].a, s.v[1].wA));
        b = vadd(vscale(s.v[0].a, s.v[0].wB), vscale(s.v[1].a, s.v[1].wB));
    } else {
        a = vadd(vadd(vscale(s.v[0].a, s.v[0].wA), vscale(s.v[1].a, s.v[1].wA)), vscale(s.v[2].a, s.v[2].wA));
        b = a;
    }
    float distance = vlen(vsub(a, b));
    /* WriteCache */
    cache->metric = simplex_metric(&s);
    cache->count = s.count;
    for (int i = 0; i < s.count; ++i) { cache->indexA[i] = s.v[i].indexA; cache->indexB[i] = s.v[i].indexB; }
    return distance;
}

#define SEP_POINTS 0
#define SEP_FACE_A 1
#define SEP_FACE_B 2
typedef struct { const Proxy* pA; const Proxy* pB; Sweep sA, sB; int type; V2 localPoint, axis; } SepFn;

static void sep_init(SepFn* f, const SimplexCache* cache, const Proxy* pA, const Sweep* sA, const Proxy* pB, const Sweep* sB, float t1) {
    f->pA = pA; f->pB = pB; f->sA = *sA; f->sB = *sB;
    Xf xfA = sweep_xf(&f->sA, t1), xfB = sweep_xf(&f->sB, t1);
    if (cache->count == 1) {
        f->type = SEP_POINTS;
        V2 pointA = xmul(xfA, pA->verts[cache->indexA[0]]), pointB = xmul(xfB, pB->verts[cache->indexB[0]]);
        f->axis = vsub(pointB, pointA);
        vnormalize(&f->axis);
        f->localPoint = v2(0.0f, 0.0f);
    } else if (cache->indexA[0] == cache->indexA[1]) {
        f->type = SEP_FACE_B;
        V2 b1 = pB->verts[cache->indexB[0]], b2 = pB->verts[cache->indexB[1]];
        f->axis = vcross_vs(vsub(b2, b1), 1.0f);
        vnormalize(&f->axis);
        V2 normal = rmul(xfB.q, f->axis);
        f->localPoint = vscale(0.5f, vadd(b1, b2));
        V2 pointB = xmul(xfB, f->localPoint);
        V2 pointA = xmul(xfA, pA->verts[cache->indexA[0]]);
        float s = vdot(vsub(pointA, pointB), normal);
        if (s < 0.0f) f->axis = vneg(f->axis);
    } else {
        f->type = SEP_FACE_A;
        V2 a1 = pA->verts[cache->indexA[0]], a2 = pA->verts[cache->indexA[1]];
        f->axis = vcross_vs(vsub(a2, a1), 1.0f);
        vnormalize(&f->axis);
        V2 normal = rmul(xfA.q, f->axis);
        f->localPoint = vscale(0.5f, vadd(a1, a2));
        V2 pointA = xmul(xfA, f->localPoint);
        V2 pointB = xmul(xfB, pB->verts[cache->indexB[0]]);
        float s = vdot(vsub(pointB, pointA), normal);
        if (s < 0.0f) f->axis = vneg(f->axis);
    }
}
static float sep_find_min(const SepFn* f, int* indexA, int* indexB, float t) {
    Xf xfA = sweep_xf(&f->sA, t), xfB = sweep_xf(&f->sB, t);
    if (f->type == SEP_POINTS) {
        V2 axisA = rmulT(xfA.q, f->axis), axisB = rmulT(xfB.q, vneg(f->axis));
        *indexA = proxy_support(f->pA, axisA);
        *indexB = proxy_support(f->pB, axisB);
        V2 pointA = xmul(xfA, f->pA->verts[*indexA]), pointB = xmul(xfB, f->pB->verts[*indexB]);
        return vdot(vsub(pointB, pointA), f->axis);
    } else if (f->type == SEP_FACE_A) {
        V2 normal = rmul(xfA.q, f->axis);
        V2 pointA = xmul(xfA, f->localPoint);
        V2 axisB = rmulT(xfB.q, vneg(normal));
        *indexA = -1;
        *indexB = proxy_support(f->pB, axisB);
        V2 pointB = xmul(xfB, f->pB->verts[*indexB]);
        return vdot(vsub(pointB, pointA), normal);
    } else {
        V2 normal = rmul(xfB.q, f->axis);
        V2 pointB = xmul(xfB, f->localPoint);
        V2 axisA = rmulT(xfA.q, vneg(normal));
        *indexB = -1;
        *indexA = proxy_support(f->pA, axisA);
        V2 pointA = xmul(xfA, f->pA->verts[*indexA]);
        return vdot(vsub(pointA, pointB), normal);
    }
}
static float sep_evaluate(const SepFn* f, int indexA, int indexB, float t) {
    Xf xfA = sweep_xf(&f->sA, t), xfB = sweep_xf(&f->sB, t);
    if (f->type == SEP_POINTS) {
        V2 pointA = xmul(xfA, f->pA->verts[indexA]), pointB = xmul(xfB, f->pB->verts[indexB]);
        return vdot(vsub(pointB, pointA), f->axis);
    } else if (f->type == SEP_FACE_A) {
        V2 normal = rmul(xfA.q, f->axis);
        V2 pointA = xmul(xfA, f->localPoint);
        V2 pointB = xmul(xfB, f->pB->verts[indexB]);
        return vdot(vsub(pointB, pointA), normal);
    } else {
        V2 normal = rmul(xfB.q, f->axis);
        V2 pointB = xmul(xfB, f->localPoint);
        V2 pointA = xmul(xfA, f->pA->verts[indexA]);
        return vdot(vsub(pointA, pointB), normal);
    }
}

#define TOI_UNKNOWN 0
#define TOI_FAILED 1
#define TOI_OVERLAPPED 2
#define TOI_TOUCHING 3
#define TOI_SEPARATED 4

static int time_of_impact(float* tOut, const Proxy* pA, Sweep sweepA, const Proxy* pB, Sweep sweepB, float tMax, Counters* cnt) {
    cnt->c[REM2D_CNT_TOI_CALLS]++;
    int state = TOI_UNKNOWN;
    *tOut = tMax;
    sweep_normalize(&sweepA);
    sweep_normalize(&sweepB);
    float totalRadius = pA->radius + pB->radius;
    float target = fmax2(B2_LINEAR_SLOP, totalRadius - 3.0f * B2_LINEAR_SLOP);
    float tolerance = 0.25f * B2_LINEAR_SLOP;
    float t1 = 0.0f;
    const int k_maxIterations = 20;
    int iter = 0;
    SimplexCache cache;
    cache.count = 0; cache.metric = 0.0f;
    for (;;) {
        Xf xfA = sweep_xf(&sweepA, t1), xfB = sweep_xf(&sweepB, t1);
        float distance = gjk_distance(&cache, pA, xfA, pB, xfB, cnt);
        if (distance <= 0.0f) { state = TOI_OVERLAPPED; *tOut = 0.0f; break; }
        if (distance < target + tolerance) { state = TOI_TOUCHING; *tOut = t1; break; }
        SepFn fcn;
        sep_init(&fcn, &cache, pA, &sweepA, pB, &sweepB, t1);
        int done = 0;
        float t2 = tMax;
        int pushBackIter = 0;
        for (;;) {
            int indexA, indexB;
            float s2 = sep_find_min(&fcn, &indexA, &indexB, t2);
            if (s2 > target + tolerance) { state = TOI_SEPARATED; *tOut = tMax; done = 1; break; }
            if (s2 > target - tolerance) { t1 = t2; break; }
            float s1 = sep_evaluate(&fcn, indexA, indexB, t1);
            if (s1 < target - tolerance) { state = TOI_FAILED; *tOut = t1; done = 1; break; }
            if (s1 <= target + tolerance) { state = TOI_TOUCHING; *tOut = t1; done = 1; break; }
            int rootIterCount = 0;
            float a1 = t1, a2 = t2;
            for (;;) {
                float t;
                if (rootIterCount & 1) t = a1 + (target - s1) * (a2 - a1) / (s2 - s1);
                else t = 0.5f * (a1 + a2);
                ++rootIterCount;
                cnt->c[REM2D_CNT_TOI_ROOT_ITERS]++;
                float s = sep_evaluate(&fcn, indexA, indexB, t);
                if (fabs2(s - target) < tolerance) { t2 = t; break; }
                if (s > target) { a1 = t; s1 = s; } else { a2 = t; s2 = s; }
                if (rootIterCount == 50) break;
            }
            ++pushBackIter;
            if (pushBackIter == B2_MAX_POLYGON_VERTICES) break;
        }
        ++iter;
        if (done) break;
        if (iter == k_maxIterations) { state = TOI_FAILED; *tOut = t1; break; }
    }
    return state;
}

/* b2Island::SolveTOI for {edge (static, index 0), module (index 1), further static edges} */
static void island_solve_toi(rem2d_handle* h, World* w, Island* is, float subDt, Counters* cnt,
                             const int* islandIndexOfBody, const int* islandIndexOfContactEdge) {
    for (int i = 0; i < is->count; ++i) {
        if (is->bodyIdx[i] < 0) {
            is->pos[i].c = v2(0.0f, 0.0f); is->pos[i].a = 0.0f;
            is->vel[i].v = v2(0.0f, 0.0f); is->vel[i].w = 0.0f;
        } else {
            Body* b = &w->bodies[is->bodyIdx[i]];
            is->pos[i].c = b->sweep.c; is->pos[i].a = b->sweep.a;
            is->vel[i].v = b->v; is->vel[i].w = b->w;
        }
    }
    csolver_setup(w, is, 1.0f, 0, islandIndexOfBody, islandIndexOfContactEdge);
    for (int i = 0; i < 20; ++i) {
        int contactsOkay = csolver_solve_position(is, 1, 0, 1, cnt);
        if (contactsOkay) break;
    }
    /* leap of faith to the new safe state (toiIndexA = 0 is the static edge: unchanged) */
    {
        Body* b = &w->bodies[is->bodyIdx[1]];
        b->sweep.c0 = is->pos[1].c;
        b->sweep.a0 = is->pos[1].a;
    }
    csolver_init_velocity(w, is);
    for (int it = 0; it < h->cfg.velocity_iterations; ++it) csolver_solve_velocity(is, cnt);
    float hdt = subDt;
    for (int i = 0; i < is->count; ++i) {
        V2 c = is->pos[i].c; float a = is->pos[i].a;
        V2 v = is->vel[i].v; float ww = is->vel[i].w;
        V2 translation = vscale(hdt, v);
        if (vdot(translation, translation) > B2_MAX_TRANSLATION_SQ) {
            float ratio = B2_MAX_TRANSLATION / vlen(translation);
            v = vscale(ratio, v);
        }
        float rotation = hdt * ww;
        if (rotation * rotation > B2_MAX_ROTATION_SQ) {
            float ratio = B2_MAX_ROTATION / fabs2(rotation);
            ww *= ratio;
        }
        c = vadd(c, vscale(hdt, v));
        a += hdt * ww;
        is->pos[i].c = c; is->pos[i].a = a;
        is->vel[i].v = v; is->vel[i].w = ww;
        if (is->bodyIdx[i] >= 0) {
            Body* b = &w->bodies[is->bodyIdx[i]];
            b->sweep.c = c; b->sweep.a = a;
            b->v = v; b->w = ww;
            body_sync_transform(b);
        }
    }
}

/* b2World::SolveTOI (m_stepComplete is always true here: no sub-stepping) */
static void world_solve_toi(rem2d_handle* h, World* w, float dt, Counters* cnt) {
    static __thread Island is_storage;
    Island* is = &is_storage;
    for (int b = 0; b < w->nb; ++b) { w->bodies[b].islandFlag = 0; w->bodies[b].sweep.alpha0 = 0.0f; }
    for (int e = 0; e < h->n_edges; ++e) w->edge_alpha0[e] = 0.0f;
    for (int i = 0; i < w->nc; ++i) {
        w->contacts[i].flags &= ~(CF_TOI | CF_ISLAND);
        w->contacts[i].toiCount = 0;
        w->contacts[i].toi = 1.0f;
    }
    for (;;) {
        int minContact = -1;
        float minAlpha = 1.0f;
        for (int ci = w->nc - 1; ci >= 0; --ci) {      /* world contact list: newest first */
            Contact* c = &w->contacts[ci];
            if (!(c->flags & CF_ENABLED)) continue;
            if (c->toiCount > B2_MAX_SUB_STEPS) continue;
            float alpha = 1.0f;
            if (c->flags & CF_TOI) alpha = c->toi;
            else {
                Body* bB = &w->bodies[c->body];
                int activeB = bB->awake;          /* A is static: never active, always "collides" */
                if (!activeB) continue;
                float aA0 = w->edge_alpha0[c->edge];
                float alpha0 = aA0;
                if (aA0 < bB->sweep.alpha0) { alpha0 = bB->sweep.alpha0; w->edge_alpha0[c->edge] = alpha0; }
                else if (bB->sweep.alpha0 < aA0) { alpha0 = aA0; sweep_advance(&bB->sweep, alpha0); }
                V2 everts[2] = { h->ev1[c->edge], h->ev2[c->edge] };
                V2 cverts[1] = { {0.0f, 0.0f} };
                Proxy pA = { everts, 2, B2_POLYGON_RADIUS };
                Proxy pB;
                if (bB->shape == REM2D_SHAPE_CIRCLE) { pB.verts = cverts; pB.count = 1; pB.radius = bB->radius; }
                else { pB.verts = bB->verts; pB.count = bB->count; pB.radius = bB->radius; }
                Sweep sA;
                memset(&sA, 0, sizeof(sA));
                sA.alpha0 = w->edge_alpha0[c->edge];
                float t;
                int state = time_of_impact(&t, &pA, sA, &pB, bB->sweep, 1.0f, cnt);
                float beta = t;
                if (state == TOI_TOUCHING) alpha = fmin2(alpha0 + (1.0f - alpha0) * beta, 1.0f);
                else alpha = 1.0f;
                c->toi = alpha;
                c->flags |= CF_TOI;
            }
            if (alpha < minAlpha) { minContact = ci; minAlpha = alpha; }
        }
        if (minContact < 0 || 1.0f - 10.0f * B2_EPSILON < minAlpha) break;
        cnt->c[REM2D_CNT_TOI_EVENTS]++;
        Contact* mc = &w->contacts[minContact];
        Body* bB = &w->bodies[mc->body];
        int eA = mc->edge;
        Sweep backupB = bB->sweep;
        float backupA = w->edge_alpha0[eA];
        w->edge_alpha0[eA] = minAlpha;           /* bA->Advance(minAlpha) on a static body */
        body_advance(bB, minAlpha);
        contact_update(h, w, mc, cnt);
        mc->flags &= ~CF_TOI;
        ++mc->toiCount;
        if (!(mc->flags & CF_ENABLED) || !(mc->flags & CF_TOUCHING)) {
            mc->flags &= ~CF_ENABLED;
            w->edge_alpha0[eA] = backupA;
            bB->sweep = backupB;
            body_sync_transform(bB);
            continue;
        }
        body_set_awake(bB, 1);
        /* build the TOI island: [edge eA, module, other static edges touched by the module] */
        int islandIndexOfBody[64];
        int islandIndexOfContactEdge[ISL_MAX_CONTACTS];
        unsigned char edgeFlag[MAX_EDGES];
        memset(edgeFlag, 0, sizeof(edgeFlag));
        is->count = 0; is->ncontacts = 0; is->njoints = 0;
        is->bodyIdx[is->count++] = -(eA + 1);
        islandIndexOfBody[mc->body] = is->count;
        bB->islandIndex = is->count;
        is->bodyIdx[is->count++] = mc->body;
        is->contactIdx[is->ncontacts] = minContact;
        islandIndexOfContactEdge[is->ncontacts] = 0;
        is->ncontacts++;
        edgeFlag[eA] = 1;
        bB->islandFlag = 1;
        mc->flags |= CF_ISLAND;
        for (int ci = w->nc - 1; ci >= 0; --ci) {   /* the module's contact list, newest first */
            Contact* c = &w->contacts[ci];
            if (c->body != mc->body) continue;
            if (is->count == 2 * B2_MAX_TOI_CONTACTS) break;
            if (is->ncontacts == B2_MAX_TOI_CONTACTS) break;
            if (c->flags & CF_ISLAND) continue;
            int e = c->edge;
            float backup = w->edge_alpha0[e];
            if (!edgeFlag[e]) w->edge_alpha0[e] = minAlpha;     /* other->Advance(minAlpha) */
            contact_update(h, w, c, cnt);
            if (!(c->flags & CF_ENABLED) || !(c->flags & CF_TOUCHING)) { w->edge_alpha0[e] = backup; continue; }
            c->flags |= CF_ISLAND;
            is->contactIdx[is->ncontacts] = ci;
            if (edgeFlag[e]) {
                for (int i = 0; i < is->count; ++i)
                    if (is->bodyIdx[i] == -(e + 1)) { islandIndexOfContactEdge[is->ncontacts] = i; break; }
                is->ncontacts++;
                continue;
            }
            edgeFlag[e] = 1;
            islandIndexOfContactEdge[is->ncontacts] = is->count;
            is->ncontacts++;
            is->bodyIdx[is->count++] = -(e + 1);
        }
        float subDt = (1.0f - minAlpha) * dt;
        island_solve_toi(h, w, is, subDt, cnt, islandIndexOfBody, islandIndexOfContactEdge);
        /* reset island flags and synchronize broad-phase proxies */
        bB->islandFlag = 0;
        body_synchronize_fixtures(bB);
        for (int ci = 0; ci < w->nc; ++ci)
            if (w->contacts[ci].body == mc->body) w->contacts[ci].flags &= ~(CF_TOI | CF_ISLAND);
        world_find_new_contacts(h, w);
    }
}

/* b2World::Step */
static void world_step(rem2d_handle* h, World* w, Counters* cnt) {
    float dt = h->cfg.dt;
    if (w->newFixture) { world_find_new_contacts(h, w); w->newFixture = 0; }
    float inv_dt = dt > 0.0f ? 1.0f / dt : 0.0f;
    float dtRatio = w->inv_dt0 * dt;
    world_collide(h, w, cnt);
    if (dt > 0.0f) world_solve(h, w, dt, dtRatio, cnt);
    if (h->cfg.continuous && dt > 0.0f) world_solve_toi(h, w, dt, cnt);
    if (dt > 0.0f) w->inv_dt0 = inv_dt;
}

/* ---------------------------------------------------------------- episode: Modular2D.step + evaluate() */
static void tick(rem2d_handle* h, World* w, Counters* cnt) {
    if (!w->alive) return;
    /* Modular2DEnv.py:613-614 */
    w->wod += h->cfg.wod_speed;
    /* Modular2DEnv.py:620-623: controller.update(0) for every expressed node, root included */
    for (int b = 0; b < w->nb; ++b) {
        Ctrl* c = &w->ctrl[b];
        c->phase += 0.0;
        c->i_state += c->frequency;
        c->output = c->amplitude * sin_f64(c->i_state + c->phase) + c->offset;
    }
    /* Modular2DEnv.py:631-632 + PID (:600-605); the setter wakes both bodies (b2RevoluteJoint::SetMotorSpeed) */
    for (int k = 0; k < w->nj; ++k) {
        Joint* j = &w->joints[k];
        float currentAngle = w->bodies[j->bodyB].sweep.a - w->bodies[j->bodyA].sweep.a - j->referenceAngle;
        double angleDifference = w->ctrl[k + 1].output - (double)currentAngle;
        double speed = angleDifference * h->cfg.p_gain;
        body_set_awake(&w->bodies[j->bodyA], 1);
        body_set_awake(&w->bodies[j->bodyB], 1);
        j->motorSpeed = (float)speed;
    }
    world_step(h, w, cnt);
    cnt->c[REM2D_CNT_TICKS]++;
    int i = w->ticks;           /* loop index of evaluate() */
    w->ticks++;
    if (h->cfg.terminate) {
        /* Modular2DEnv.py:642-649 */
        double reward = (double)w->bodies[0].xf.p.x;
        if (w->bodies[0].xf.p.x < 0.0f) reward = -100.0;
        if (w->wod > (double)w->bodies[0].xf.p.x) reward = -100.0;
        /* REM2D_main.py:370-377 */
        if (reward < -10.0) { w->alive = 0; }
        else if (reward > h->cfg.env_length) {
            reward += (double)(h->cfg.evaluation_steps - i) / (double)h->cfg.evaluation_steps;
            w->fitness = reward;
            w->alive = 0;
        } else if (reward > 0.0) w->fitness = reward;
        if (w->ticks >= h->cfg.evaluation_steps) w->alive = 0;
    } else {
        double reward = (double)w->bodies[0].xf.p.x;
        if (reward > 0.0) w->fitness = reward;
    }
}

/* ---------------------------------------------------------------- world construction */
static void body_init(Body* b, int shape, float hx, float hy, float x, float y, float a) {
    memset(b, 0, sizeof(*b));
    b->shape = shape;
    float density = 1.0f;
    float mass, I;
    V2 center;
    if (shape == REM2D_SHAPE_CIRCLE) {
        b->count = 0;
        b->radius = hx;
        /* b2CircleShape::ComputeMass, m_p = 0 */
        mass = density * B2_PI * b->radius * b->radius;
        center = v2(0.0f, 0.0f);
        I = mass * (0.5f * b->radius * b->radius + vdot(center, center));
    } else {
        /* b2PolygonShape::SetAsBox + ComputeMass */
        b->count = 4;
        b->radius = B2_POLYGON_RADIUS;
        b->verts[0] = v2(-hx, -hy); b->verts[1] = v2(hx, -hy); b->verts[2] = v2(hx, hy); b->verts[3] = v2(-hx, hy);
        b->normals[0] = v2(0.0f, -1.0f); b->normals[1] = v2(1.0f, 0.0f); b->normals[2] = v2(0.0f, 1.0f); b->normals[3] = v2(-1.0f, 0.0f);
        V2 cen = v2(0.0f, 0.0f);
        float area = 0.0f, II = 0.0f;
        V2 s = v2(0.0f, 0.0f);
        for (int i = 0; i < 4; ++i) s = vadd(s, b->verts[i]);
        s = vscale(1.0f / 4.0f, s);
        const float k_inv3 = 1.0f / 3.0f;
        for (int i = 0; i < 4; ++i) {
            V2 e1 = vsub(b->verts[i], s);
            V2 e2 = i + 1 < 4 ? vsub(b->verts[i + 1], s) : vsub(b->verts[0], s);
            float D = vcross(e1, e2);
            float triangleArea = 0.5f * D;
            area += triangleArea;
            cen = vadd(cen, vscale(triangleArea * k_inv3, vadd(e1, e2)));
            float ex1 = e1.x, ey1 = e1.y, ex2 = e2.x, ey2 = e2.y;
            float intx2 = ex1 * ex1 + ex2 * ex1 + ex2 * ex2;
            float inty2 = ey1 * ey1 + ey2 * ey1 + ey2 * ey2;
            II += (0.25f * k_inv3 * D) * (intx2 + inty2);
        }
        mass = density * area;
        cen = vscale(1.0f / area, cen);
        center = vadd(cen, s);
        I = density * II;
        I += mass * (vdot(center, center) - vdot(cen, cen));
    }
    /* b2Body::ResetMassData */
    b->mass = mass;
    V2 localCenter = vscale(mass, center);
    b->I = I;
    if (b->mass > 0.0f) { b->invMass = 1.0f / b->mass; localCenter = vscale(b->invMass, localCenter); }
    else { b->mass = 1.0f; b->invMass = 1.0f; }
    if (b->I > 0.0f) { b->I -= b->mass * vdot(localCenter, localCenter); b->invI = 1.0f / b->I; }
    else { b->I = 0.0f; b->invI = 0.0f; }
    b->xf.p = v2(x, y);
    b->xf.q = rot_set(a);
    b->sweep.localCenter = localCenter;
    b->sweep.c0 = b->sweep.c = xmul(b->xf, localCenter);
    b->sweep.a0 = b->sweep.a = a;
    b->sweep.alpha0 = 0.0f;
    b->v = v2(0.0f, 0.0f); b->w = 0.0f;
    b->awake = 1; b->sleepTime = 0.0f;
    /* b2Fixture::CreateProxies: fat AABB of the initial pose, proxy goes into the move buffer */
    b->fat = aabb_fatten(shape_aabb(b, b->xf));
    b->moved = 1;
}

static void world_free(World* w) {
    free(w->bodies); free(w->joints); free(w->ctrl); free(w->contacts);
    memset(w, 0, sizeof(*w));
}

static int world_build(rem2d_handle* h, World* w, int c) {
    const rem2d_population* p = &h->pop;
    int b0 = p->body_off[c], b1 = p->body_off[c + 1];
    int nb = b1 - b0, nj = nb - 1, j0 = b0 - c;
    if (nb < 1 || nb > 64) return REM2D_E_CAPACITY;
    world_free(w);
    w->nb = nb; w->nj = nj;
    w->bodies = (Body*)calloc((size_t)nb, sizeof(Body));
    w->joints = (Joint*)calloc((size_t)(nj > 0 ? nj : 1), sizeof(Joint));
    w->ctrl = (Ctrl*)calloc((size_t)nb, sizeof(Ctrl));
    for (int i = 0; i < nb; ++i) {
        body_init(&w->bodies[i], p->shape[b0 + i], p->hx[b0 + i], p->hy[b0 + i], p->x0[b0 + i], p->y0[b0 + i], p->a0[b0 + i]);
        const double* cc = &p->ctrl[(size_t)(b0 + i) * 5];
        w->ctrl[i].amplitude = cc[0]; w->ctrl[i].phase = cc[1]; w->ctrl[i].frequency = cc[2];
        w->ctrl[i].offset = cc[3]; w->ctrl[i].i_state = cc[4]; w->ctrl[i].output = 0.0;
    }
    for (int k = 0; k < nj; ++k) {
        Joint* j = &w->joints[k];
        j->bodyA = p->joint_parent[j0 + k];
        j->bodyB = k + 1;
        if (j->bodyA < 0 || j->bodyA > k) return REM2D_E_INVALID;
        j->localAnchorA = v2(p->anchor_a[2 * (j0 + k)], p->anchor_a[2 * (j0 + k) + 1]);
        j->localAnchorB = v2(p->anchor_b[2 * (j0 + k)], p->anchor_b[2 * (j0 + k) + 1]);
        j->lower = p->lower[j0 + k]; j->upper = p->upper[j0 + k];
        j->maxMotorTorque = p->max_torque[j0 + k];
        j->referenceAngle = 0.0f;
        j->motorSpeed = 0.0f;
        j->limitState = LIMIT_INACTIVE;
    }
    w->nc = 0;
    w->inv_dt0 = 0.0f;
    w->newFixture = 1;
    w->alive = 1; w->ticks = 0; w->wod = 0.0; w->fitness = 0.0;
    memset(w->edge_alpha0, 0, sizeof(w->edge_alpha0));
    return REM2D_OK;
}

/* ---------------------------------------------------------------- C-ABI */
void rem2d_default_config(rem2d_config* cfg) {
    memset(cfg, 0, sizeof(*cfg));
    cfg->dt = (float)(1.0 / 50);
    cfg->velocity_iterations = 180;
    cfg->position_iterations = 60;
    cfg->gravity_y = -10.0f;
    cfg->module_friction = (float)0.1;
    cfg->terrain_friction = 2.5f;
    cfg->p_gain = 1.9;
    cfg->wod_speed = 0.04;
    cfg->env_length = 100.0;
    cfg->evaluation_steps = 10000;
    cfg->continuous = 1;
    cfg->allow_sleep = 1;
    cfg->terminate = 1;
    cfg->device = 0;
    cfg->stream = NULL;
    cfg->sincos_mode = 0;
}
int rem2d_abi_version(void) { return REM2D_ABI_VERSION; }
const char* rem2d_backend(void) { return "oracle-c"; }

int rem2d_create(const rem2d_config* cfg, rem2d_handle** out) {
    if (!cfg || !out) { snprintf(g_create_err, sizeof(g_create_err), "rem2d_create: NULL argument"); return REM2D_E_INVALID; }
    rem2d_handle* h = (rem2d_handle*)calloc(1, sizeof(rem2d_handle));
    if (!h) return REM2D_E_NOMEM;
    h->cfg = *cfg;
    h->threads = 0;
    *out = h;
    return REM2D_OK;
}
static void free_pop(rem2d_handle* h) {
    for (int i = 0; i < 16; ++i) { free(h->pop_mem[i]); h->pop_mem[i] = NULL; }
    h->have_pop = 0;
}
int rem2d_destroy(rem2d_handle* h) {
    if (!h) return REM2D_E_INVALID;
    for (int i = 0; i < h->n_worlds; ++i) world_free(&h->worlds[i]);
    free(h->worlds);
    free_pop(h);
    free(h);
    return REM2D_OK;
}
const char* rem2d_last_error(rem2d_handle* h) { return h ? h->err : g_create_err; }

int rem2d_set_terrain(rem2d_handle* h, const double* y, int32_t n, double step) {
    if (!h || !y || n < 2 || n > MAX_EDGES) { if (h) snprintf(h->err, sizeof(h->err), "set_terrain: bad arguments"); return REM2D_E_INVALID; }
    h->n_edges = n - 1;
    h->terrain_step = (float)step;
    for (int i = 0; i < n - 1; ++i) {
        /* edgeShape.vertices = [(x_i, y_i), (x_{i+1}, y_{i+1})] (Modular2DEnv.py:294-302): doubles -> float32 */
        h->ev1[i] = v2((float)((double)i * step), (float)y[i]);
        h->ev2[i] = v2((float)((double)(i + 1) * step), (float)y[i + 1]);
        /* b2EdgeShape::ComputeAABB with identity transform, then the proxy's fat AABB */
        V2 lo = v2(fmin2(h->ev1[i].x, h->ev2[i].x), fmin2(h->ev1[i].y, h->ev2[i].y));
        V2 hi = v2(fmax2(h->ev1[i].x, h->ev2[i].x), fmax2(h->ev1[i].y, h->ev2[i].y));
        AABB a;
        a.lo = v2(lo.x - B2_POLYGON_RADIUS, lo.y - B2_POLYGON_RADIUS);
        a.hi = v2(hi.x + B2_POLYGON_RADIUS, hi.y + B2_POLYGON_RADIUS);
        h->efat[i] = aabb_fatten(a);
    }
    h->have_terrain = 1;
    return REM2D_OK;
}

static void* dup_mem(const void* src, size_t bytes) {
    void* p = malloc(bytes ? bytes : 1);
    if (p && bytes) memcpy(p, src, bytes);
    return p;
}
int rem2d_upload(rem2d_handle* h, const rem2d_population* pop) {
    if (!h || !pop || pop->n_creatures < 0) return REM2D_E_INVALID;
    if (pop->n_joints != pop->n_bodies - pop->n_creatures) { snprintf(h->err, sizeof(h->err), "upload: n_joints != n_bodies - n_creatures"); return REM2D_E_INVALID; }
    free_pop(h);
    size_t nb = (size_t)pop->n_bodies, nj = (size_t)pop->n_joints, nc = (size_t)pop->n_creatures;
    h->pop = *pop;
    int k = 0;
    h->pop.body_off = (const int32_t*)(h->pop_mem[k++] = dup_mem(pop->body_off, (nc + 1) * 4));
    h->pop.shape = (const uint8_t*)(h->pop_mem[k++] = dup_mem(pop->shape, nb));
    h->pop.hx = (const float*)(h->pop_mem[k++] = dup_mem(pop->hx, nb * 4));
    h->pop.hy = (const float*)(h->pop_mem[k++] = dup_mem(pop->hy, nb * 4));
    h->pop.x0 = (const float*)(h->pop_mem[k++] = dup_mem(pop->x0, nb * 4));
    h->pop.y0 = (const float*)(h->pop_mem[k++] = dup_mem(pop->y0, nb * 4));
    h->pop.a0 = (const float*)(h->pop_mem[k++] = dup_mem(pop->a0, nb * 4));
    h->pop.joint_parent = (const int16_t*)(h->pop_mem[k++] = dup_mem(pop->joint_parent, nj * 2));
    h->pop.anchor_a = (const float*)(h->pop_mem[k++] = dup_mem(pop->anchor_a, nj * 8));
    h->pop.anchor_b = (const float*)(h->pop_mem[k++] = dup_mem(pop->anchor_b, nj * 8));
    h->pop.lower = (const float*)(h->pop_mem[k++] = dup_mem(pop->lower, nj * 4));
    h->pop.upper = (const float*)(h->pop_mem[k++] = dup_mem(pop->upper, nj * 4));
    h->pop.max_torque = (const float*)(h->pop_mem[k++] = dup_mem(pop->max_torque, nj * 4));
    h->pop.ctrl = (const double*)(h->pop_mem[k++] = dup_mem(pop->ctrl, nb * 5 * 8));
    h->have_pop = 1;
    return rem2d_reset(h);
}

int rem2d_reset(rem2d_handle* h) {
    if (!h || !h->have_pop) { if (h) snprintf(h->err, sizeof(h->err), "reset: no population uploaded"); return REM2D_E_INVALID; }
    if (!h->have_terrain) { snprintf(h->err, sizeof(h->err), "reset: no terrain set"); return REM2D_E_INVALID; }
    g_sincos_mode = h->cfg.sincos_mode;
    int n = h->pop.n_creatures;
    if (h->n_worlds != n) {
        for (int i = 0; i < h->n_worlds; ++i) world_free(&h->worlds[i]);
        free(h->worlds);
        h->worlds = (World*)calloc((size_t)(n > 0 ? n : 1), sizeof(World));
        h->n_worlds = n;
    }
    for (int c = 0; c < n; ++c) {
        int rc = world_build(h, &h->worlds[c], c);
        if (rc != REM2D_OK) { snprintf(h->err, sizeof(h->err), "reset: creature %d cannot be built (%d)", c, rc); return rc; }
    }
    memset(h->counters, 0, sizeof(h->counters));
    return REM2D_OK;
}

/* TEST-ONLY entry point of the oracle-backed Box2D shim (tests/golden/oracle_box2d.py): what the reference's Modular2D.step
 * does to the world between its own Python statements - `joint.motorSpeed = v` for every joint (b2RevoluteJoint::SetMotorSpeed
 * wakes both bodies, Modular2DEnv.py:631-632) followed by ONE world.Step (Modular2DEnv.py:634). No controllers, no wall of
 * death, no episode bookkeeping: the reference's unmodified Python does those around this call. */
int rem2d_oracle_world_step(rem2d_handle* h, int creature, const float* motor_speed, int n_joints) {
    if (!h || !h->have_pop || creature < 0 || creature >= h->n_worlds) return REM2D_E_INVALID;
    World* w = &h->worlds[creature];
    if (n_joints != w->nj) return REM2D_E_INVALID;
    g_sincos_mode = h->cfg.sincos_mode;
    Counters cnt;
    memset(&cnt, 0, sizeof(cnt));
    for (int k = 0; k < w->nj; ++k) {
        Joint* j = &w->joints[k];
        body_set_awake(&w->bodies[j->bodyA], 1);
        body_set_awake(&w->bodies[j->bodyB], 1);
        j->motorSpeed = motor_speed[k];
    }
    world_step(h, w, &cnt);
    for (int i = 0; i < REM2D_N_COUNTERS; ++i) h->counters[i] += cnt.c[i];
    return REM2D_OK;
}

int rem2d_oracle_set_threads(rem2d_handle* h, int n) { if (!h) return REM2D_E_INVALID; h->threads = n; return REM2D_OK; }

typedef struct { rem2d_handle* h; int n_ticks; int* next; Counters cnt; } StepJob;
static void* step_worker(void* arg) {
    StepJob* job = (StepJob*)arg;
    rem2d_handle* h = job->h;
    const int chunk = 8;
    for (;;) {
        int c0 = __atomic_fetch_add(job->next, chunk, __ATOMIC_RELAXED);   /* dynamic schedule over creatures */
        if (c0 >= h->n_worlds) break;
        int c1 = c0 + chunk < h->n_worlds ? c0 + chunk : h->n_worlds;
        for (int c = c0; c < c1; ++c) {
            World* w = &h->worlds[c];
            for (int t = 0; t < job->n_ticks && w->alive; ++t) tick(h, w, &job->cnt);
        }
    }
    return NULL;
}

int rem2d_step(rem2d_handle* h, int32_t n_ticks) {
    if (!h || !h->have_pop || n_ticks < 0) return REM2D_E_INVALID;
    g_sincos_mode = h->cfg.sincos_mode;
    int nt = h->threads > 0 ? h->threads : 1;
    if (nt > 256) nt = 256;
    int next = 0;
    StepJob* jobs = (StepJob*)calloc((size_t)nt, sizeof(StepJob));
    pthread_t* tids = (pthread_t*)calloc((size_t)nt, sizeof(pthread_t));
    for (int i = 0; i < nt; ++i) { jobs[i].h = h; jobs[i].n_ticks = n_ticks; jobs[i].next = &next; }
    for (int i = 1; i < nt; ++i) pthread_create(&tids[i], NULL, step_worker, &jobs[i]);
    step_worker(&jobs[0]);
    for (int i = 1; i < nt; ++i) pthread_join(tids[i], NULL);
    for (int i = 0; i < nt; ++i)
        for (int k = 0; k < REM2D_N_COUNTERS; ++k) h->counters[k] += jobs[i].cnt.c[k];
    free(jobs); free(tids);
    for (int c = 0; c < h->n_worlds; ++c)
        if (h->worlds[c].overflow) { snprintf(h->err, sizeof(h->err), "step: island scratch overflow in creature %d", c); return REM2D_E_CAPACITY; }
    return REM2D_OK;
}

int rem2d_read_state(rem2d_handle* h, rem2d_state_view* out) {
    if (!h || !out || !h->have_pop) return REM2D_E_INVALID;
    const rem2d_population* p = &h->pop;
    for (int c = 0; c < h->n_worlds; ++c) {
        World* w = &h->worlds[c];
        int b0 = p->body_off[c], j0 = b0 - c;
        for (int i = 0; i < w->nb; ++i) {
            Body* b = &w->bodies[i];
            if (out->pose) { out->pose[3 * (b0 + i)] = b->xf.p.x; out->pose[3 * (b0 + i) + 1] = b->xf.p.y; out->pose[3 * (b0 + i) + 2] = b->sweep.a; }
            if (out->vel) { out->vel[3 * (b0 + i)] = b->v.x; out->vel[3 * (b0 + i) + 1] = b->v.y; out->vel[3 * (b0 + i) + 2] = b->w; }
        }
        for (int k = 0; k < w->nj; ++k) {
            Joint* j = &w->joints[k];
            if (out->joint_impulse) {
                float* o = &out->joint_impulse[4 * (j0 + k)];
                o[0] = j->impulse.x; o[1] = j->impulse.y; o[2] = j->impulse.z; o[3] = j->motorImpulse;
            }
            if (out->limit_state) out->limit_state[j0 + k] = j->limitState;
            if (out->motor_speed) out->motor_speed[j0 + k] = j->motorSpeed;
        }
        if (out->alive) out->alive[c] = w->alive;
        if (out->ticks) out->ticks[c] = w->ticks;
        if (out->awake) { int a = 0; for (int i = 0; i < w->nb; ++i) a |= w->bodies[i].awake; out->awake[c] = a; }
        if (out->wod) out->wod[c] = w->wod;
        if (out->n_contacts) out->n_contacts[c] = w->nc;
        int nt = 0;
        for (int i = 0; i < w->nc; ++i) nt += (w->contacts[i].flags & CF_TOUCHING) ? 1 : 0;
        if (out->n_touching) out->n_touching[c] = nt;
        if (out->touching_pairs && out->max_pairs > 0) {
            int32_t* tp = &out->touching_pairs[(size_t)c * out->max_pairs * 2];
            float* ti = out->touching_impulse ? &out->touching_impulse[(size_t)c * out->max_pairs * 4] : NULL;
            for (int k = 0; k < out->max_pairs * 2; ++k) tp[k] = -1;
            if (ti) for (int k = 0; k < out->max_pairs * 4; ++k) ti[k] = 0.0f;
            int k = 0;
            for (int b = 0; b < w->nb && k < out->max_pairs; ++b)
                for (int e = 0; e < h->n_edges && k < out->max_pairs; ++e) {
                    int ci = world_find_contact(w, b, e);
                    if (ci < 0 || !(w->contacts[ci].flags & CF_TOUCHING)) continue;
                    tp[2 * k] = b; tp[2 * k + 1] = e;
                    if (ti) {
                        const Manifold* m = &w->contacts[ci].m;
                        ti[4 * k] = m->points[0].normalImpulse;
                        ti[4 * k + 1] = m->pointCount > 1 ? m->points[1].normalImpulse : 0.0f;
                        ti[4 * k + 2] = m->points[0].tangentImpulse;
                        ti[4 * k + 3] = m->pointCount > 1 ? m->points[1].tangentImpulse : 0.0f;
                    }
                    ++k;
                }
        }
    }
    return REM2D_OK;
}

int rem2d_fitness(rem2d_handle* h, double* out) {
    if (!h || !out || !h->have_pop) return REM2D_E_INVALID;
    for (int c = 0; c < h->n_worlds; ++c) out[c] = h->worlds[c].fitness;
    return REM2D_OK;
}
int rem2d_get_counters(rem2d_handle* h, uint64_t* out) {
    if (!h || !out) return REM2D_E_INVALID;
    memcpy(out, h->counters, sizeof(h->counters));
    return REM2D_OK;
}
int rem2d_run_episodes(rem2d_handle* h, int32_t max_ticks) {
    int rc = rem2d_reset(h);
    if (rc) return rc;
    return rem2d_step(h, max_ticks);
}
int rem2d_ticks(rem2d_handle* h, int32_t* out) {
    if (!h || !out || !h->have_pop) return REM2D_E_INVALID;
    for (int c = 0; c < h->n_worlds; ++c) out[c] = h->worlds[c].ticks;
    return REM2D_OK;
}
int rem2d_evaluate(rem2d_handle* h, const rem2d_population* pop, int32_t max_ticks, double* fitness_out, int32_t* ticks_out) {
    int rc = rem2d_upload(h, pop);
    if (rc) return rc;
    rc = rem2d_step(h, max_ticks);
    if (rc) return rc;
    if (fitness_out) { rc = rem2d_fitness(h, fitness_out); if (rc) return rc; }
    if (ticks_out) for (int c = 0; c < h->n_worlds; ++c) ticks_out[c] = h->worlds[c].ticks;
    return REM2D_OK;
}
int rem2d_measure_fp32_peak(rem2d_handle* h, double* gflops) { (void)h; if (gflops) *gflops = 0.0; return REM2D_E_INVALID; }
float rem2d_last_step_ms(rem2d_handle* h) { (void)h; return 0.0f; }
int64_t rem2d_launch_count(rem2d_handle* h) { (void)h; return 0; }
/* execution-strategy options of the CUDA build: accepted and ignored (they never change results) */
int rem2d_set_option(rem2d_handle* h, const char* name, double value) {
    static const char* known[] = {"warp_mode_max", "park_ticks", "park_cap", "smem_budget_kb",
                                  "group_shift", "tail_group_shift", "trace", "image", "overflow_wave"};
    (void)value;
    if (!h || !name) return REM2D_E_INVALID;
    for (size_t i = 0; i < sizeof(known) / sizeof(known[0]); ++i) if (!strcmp(known[i], name)) return REM2D_OK;
    if (!strncmp(name, "class_gs_", 9) && strlen(name) == 10) return REM2D_OK;
    snprintf(h->err, sizeof(h->err), "set_option: unknown option %s", name);
    return REM2D_E_INVALID;
}
int rem2d_set_priority(rem2d_handle* h, const float* expected_ticks, int32_t n) { (void)expected_ticks; (void)n; return h ? REM2D_OK : REM2D_E_INVALID; }
int rem2d_read_roots(rem2d_handle* h, float* root_x, double* wod, int32_t* alive) {
    if (!h || !h->have_pop) return REM2D_E_INVALID;
    for (int c = 0; c < h->n_worlds; ++c) {
        World* w = &h->worlds[c];
        if (root_x) root_x[c] = w->bodies[0].xf.p.x;
        if (wod) wod[c] = w->wod;
        if (alive) alive[c] = w->alive;
    }
    return REM2D_OK;
}
