// rem2d_device.cuh — device code of the batched REM2D step for sm_100a.
//
// Mapping: a GROUP of G = 2^gs LANES = ONE CREATURE (one Box2D world of the reference), 32/G creatures per warp, one warp
// per CTA; G is a run-time value per launch (1 for the small capacity classes, 2-8 for the large ones, 32 for the
// latency-oriented warp-per-creature launches). Nothing on this path is a dense contraction, so there are no tensor-core
// instructions; the per-tick work is a long chain of dependent fp32 operations on ~1-3 KB of state per creature. The lanes of
// a group share that chain: the 180 velocity iterations run as a STATIC MODULO SCHEDULE of Box2D's sequential-impulse order
// (see Sim::build_schedule), the per-body / per-joint / per-contact loops of the other phases are strided over the group.
//
//  * cold state (poses, sweeps, fat AABBs, contact pool + manifolds, joint definitions, controller state)
//    lives in HBM in a lane-interleaved block per batch of 32 creatures: word w of lane l is at
//    block[w*32 + l], so every access with a warp-uniform word index is one coalesced 128-byte line;
//  * hot state of the two iteration loops (180 velocity iterations, <= 60 position iterations) is staged
//    in shared memory in the same [word][lane] layout: bank == lane, so the per-lane *divergent* body /
//    joint / contact indices of different creatures are bank-conflict free by construction.
//
// Arithmetic restates Box2D 2.3 (b2World::Step and below) for the reference's scene — see
// oracle/rem2d_oracle.c for the plain-C restatement this is tested against bit for bit. The terrain
// side of every contact is a static body with identity transform, which removes all "A" terms
// (invMassA = invIA = 0, vA = wA = 0, xfA = I) exactly, up to the sign of zeros.
// Compile with -fmad=false: upstream Box2D builds do not contract multiply-adds.
//
// Reference call sites (under /root/reference/ModularER_2D): Modular2DEnv.py:607-653 (step),
// :600-605 (PID), Controller/m_controller.py:17-21, REM2D_main.py:362-377 (episode loop).
#pragma once
#ifdef REM2D_EMU
#include "rem2d_emu_shim.h"      // tests/emu: lanes are host threads (test infrastructure, never a product path)
// the two atomics of the park hand-over in Sim::episodes, which the emulation (parking off) compiles but never executes
inline int atomicCAS(int* p, int cmp, int v) { __atomic_compare_exchange_n(p, &cmp, v, false, __ATOMIC_ACQ_REL, __ATOMIC_ACQUIRE); return cmp; }
inline int atomicExch(int* p, int v) { return __atomic_exchange_n(p, v, __ATOMIC_ACQ_REL); }
#else
#include <cuda_runtime.h>
#endif
#include <stdint.h>
#include <float.h>

#include "../../include/rem2d.h"
#include "../../include/rem2d_stats.h"
#include "../../include/rem2d_policy.h"

namespace rem2d {

// ------------------------------------------------------------------ Box2D settings (SURVEY.md A.1)
#define RB_PI 3.14159265359f
#define RB_EPS FLT_EPSILON
#define RB_MAXF FLT_MAX
#define RB_LINEAR_SLOP 0.005f
#define RB_ANGULAR_SLOP (2.0f / 180.0f * RB_PI)
#define RB_POLY_RADIUS (2.0f * RB_LINEAR_SLOP)
#define RB_AABB_EXT 0.1f
#define RB_AABB_MULT 2.0f
#define RB_MAX_LIN_CORR 0.2f
#define RB_MAX_ANG_CORR (8.0f / 180.0f * RB_PI)
#define RB_MAX_TRANS 2.0f
#define RB_MAX_ROT (0.5f * RB_PI)
#define RB_BAUMGARTE 0.2f
#define RB_TOI_BAUMGARTE 0.75f
#define RB_MAX_SUBSTEPS 8
#define RB_TIME_TO_SLEEP 0.5f
#define RB_LIN_SLEEP_TOL 0.01f
#define RB_ANG_SLEEP_TOL (2.0f / 180.0f * RB_PI)
#define RB_MAX_POLY_VERTS 16   // pybox2d build value; bounds the TOI push-back loop only

#define RB_MAX_EDGES 200       // terrain edges (199 used)
#define RB_TOI_ISLAND_CAP 32   // b2_maxTOIContacts: Box2D stops adding contacts to a TOI mini-island at 32

struct V2 { float x, y; };
struct Rot { float s, c; };

__device__ __forceinline__ V2 mk(float x, float y) { V2 r; r.x = x; r.y = y; return r; }
__device__ __forceinline__ V2 operator+(V2 a, V2 b) { return mk(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ V2 operator-(V2 a, V2 b) { return mk(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ V2 operator-(V2 a) { return mk(-a.x, -a.y); }
__device__ __forceinline__ V2 operator*(float s, V2 a) { return mk(s * a.x, s * a.y); }
__device__ __forceinline__ float dot(V2 a, V2 b) { return a.x * b.x + a.y * b.y; }
__device__ __forceinline__ float cross(V2 a, V2 b) { return a.x * b.y - a.y * b.x; }
__device__ __forceinline__ V2 cross_vs(V2 a, float s) { return mk(s * a.y, -s * a.x); }
__device__ __forceinline__ V2 cross_sv(float s, V2 a) { return mk(-s * a.y, s * a.x); }
__device__ __forceinline__ float len(V2 a) { return sqrtf(a.x * a.x + a.y * a.y); }
__device__ __forceinline__ float min2(float a, float b) { return a < b ? a : b; }
__device__ __forceinline__ float max2(float a, float b) { return a > b ? a : b; }
__device__ __forceinline__ float clampf(float a, float lo, float hi) { return max2(lo, min2(a, hi)); }
__device__ __forceinline__ float abs2(float a) { return a > 0.0f ? a : -a; }
__device__ __forceinline__ float normalize(V2& a) {
    float l = len(a);
    if (l < RB_EPS) return 0.0f;
    float inv = 1.0f / l;
    a.x *= inv; a.y *= inv;
    return l;
}
__device__ __forceinline__ V2 rmul(Rot q, V2 v) { return mk(q.c * v.x - q.s * v.y, q.s * v.x + q.c * v.y); }
__device__ __forceinline__ V2 rmulT(Rot q, V2 v) { return mk(q.c * v.x + q.s * v.y, -q.s * v.x + q.c * v.y); }
// b2Mul(xf, v) with xf = (p, q)
__device__ __forceinline__ V2 xmul(V2 p, Rot q, V2 v) {
    return mk((q.c * v.x - q.s * v.y) + p.x, (q.s * v.x + q.c * v.y) + p.y);
}
__device__ __forceinline__ V2 xmulT(V2 p, Rot q, V2 v) {
    float px = v.x - p.x, py = v.y - p.y;
    return mk(q.c * px + q.s * py, -q.s * px + q.c * py);
}

// ------------------------------------------------------------------ portable sin/cos
// Same operation sequence as oracle/rem2d_oracle.c:sincos_kernel (double precision, no contraction):
// 3-term Cody-Waite reduction by pi/2 + degree-13/14 minimax kernels, result rounded to float.
__device__ __forceinline__ void sincos_kernel(double x, double& s, double& c) {
    const double PIO2_1 = 1.57079632673412561417e+00, PIO2_2 = 6.07710050630396597660e-11,
                 PIO2_2T = 2.02226624879595063154e-21, TWO_OVER_PI = 6.36619772367581382433e-01;
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
    if (n == 0) { s = sr; c = cr; }
    else if (n == 1) { s = cr; c = -sr; }
    else if (n == 2) { s = -sr; c = -cr; }
    else { s = -cr; c = sr; }
}
// b2Rot::Set: float kernel, same operation sequence as oracle sincos_kernel_f32 (Cody-Waite by pi/2 with short
// constants + Cephes-style minimax polynomials); huge angles use the double kernel.
// (the huge-angle path is a real call: rot_set is inlined at ~20 sites and the double kernel would be 10 % of the code)
static __device__ __noinline__ Rot rot_set_huge(float a) {
    Rot q;
    double s, c;
    sincos_kernel((double)a, s, c);
    q.s = (float)s; q.c = (float)c;
    return q;
}
__device__ __forceinline__ Rot rot_set(float a) {
    Rot q;
    if (!(abs2(a) < 65536.0f)) return rot_set_huge(a);
    float kf = floorf(a * 0.636619747f + 0.5f);
    float r = ((a - kf * 1.5703125f) - kf * 4.837512969970703125e-4f) - kf * 7.54978995489188216e-8f;
    float z = r * r;
    float sr = ((-1.9515295891e-4f * z + 8.3321608736e-3f) * z - 1.6666654611e-1f) * z * r + r;
    float cr = ((2.443315711809948e-5f * z - 1.388731625493765e-3f) * z + 4.166664568298827e-2f) * z * z - 0.5f * z + 1.0f;
    int n = (int)kf & 3;
    if (n == 0) { q.s = sr; q.c = cr; }
    else if (n == 1) { q.s = cr; q.c = -sr; }
    else if (n == 2) { q.s = -sr; q.c = -cr; }
    else { q.s = -cr; q.c = sr; }
    return q;
}

// ------------------------------------------------------------------ cold state layout (words per lane)
enum { S_NB, S_NC, S_ALIVE, S_TICKS, S_WOD_LO, S_WOD_HI, S_FIT_LO, S_FIT_HI, S_INVDT0, S_NEWFIX, S_STATUS,
       S_NADV, S_ADV0, S_COUNT = S_ADV0 + 8 };
enum { BF_CX, BF_CY, BF_A, BF_VX, BF_VY, BF_W, BF_C0X, BF_C0Y, BF_A0, BF_ALPHA0, BF_QS, BF_QC,
       BF_FLX, BF_FLY, BF_FHX, BF_FHY, BF_SLEEP, BF_INVM, BF_INVI, BF_HX, BF_HY, BF_FLAGS, BF_COUNT };
enum { JF_META, JF_LAAX, JF_LAAY, JF_LABX, JF_LABY, JF_IMPX, JF_IMPY, JF_IMPZ, JF_MIMP, JF_MSPEED, JF_LIMIT,
       JF_LOWER, JF_UPPER, JF_MAXT, JF_AMP, JF_PHASE = JF_AMP + 2, JF_FREQ = JF_PHASE + 2, JF_OFFS = JF_FREQ + 2,
       JF_ISTATE = JF_OFFS + 2, JF_COUNT = JF_ISTATE + 2 };
enum { CF_KEY, CF_TOI, CF_LNX, CF_LNY, CF_LPX, CF_LPY, CF_P0X, CF_P0Y, CF_P0N, CF_P0T, CF_P0ID,
       CF_P1X, CF_P1Y, CF_P1N, CF_P1T, CF_P1ID, CF_COUNT };

// body flags
#define BFL_AWAKE 1
#define BFL_MOVED 2
#define BFL_ISLAND 4
#define BFL_CIRCLE 8
// contact key: body | edge << 8 | flags << 16 | toiCount << 24
#define CK_ENABLED 0x01
#define CK_TOUCHING 0x02
#define CK_ISLAND 0x04
#define CK_TOIFLAG 0x08
#define CK_TYPE_SHIFT 4      // 2 bits: manifold type
#define CK_COUNT_SHIFT 6     // 2 bits: manifold pointCount
#define CK_DESTROY_MARK 0x80000000      // top bit of the toiCount byte (toiCount <= 9): contact is to be destroyed (Sim::collide)
#define MT_CIRCLES 0
#define MT_FACE_A 1
#define MT_FACE_B 2
// HJ_META / PJ_META: a | b << 8 | limit << 16 | flags | j << 24; flags: this joint is the last one of its body A (B) in island order
#define HJM_LAST_A (1 << 18)
#define HJM_LAST_B (1 << 19)
// status bits
#define ST_POOL_OVERFLOW 1     // contact pool (NC) exhausted

// hot (shared memory) layout, words per lane: 5*NB + 17*NJ + 21*NT
enum { HB_VX, HB_VY, HB_W, HB_INVM, HB_INVI, HB_COUNT };                 // position phase: CX, CY, A reuse 0..2
enum { HJ_META, HJ_RAX, HJ_RAY, HJ_RBX, HJ_RBY, HJ_EXX, HJ_EYX, HJ_EYY, HJ_INV2, HJ_INV3, HJ_MMASS,
       HJ_IMPX, HJ_IMPY, HJ_IMPZ, HJ_MIMP, HJ_MSPEED, HJ_MAXIMP, HJ_COUNT };   // INV2/INV3: 1/det of the 2x2 / 3x3 blocks
// position-phase overlay of a joint slot
enum { PJ_META = HJ_META, PJ_LAAX, PJ_LAAY, PJ_LABX, PJ_LABY, PJ_LOWER, PJ_UPPER };
enum { HC_META, HC_NX, HC_NY, HC_R0X, HC_R0Y, HC_NM0, HC_TM0, HC_NI0, HC_TI0, HC_R1X, HC_R1Y, HC_NM1, HC_TM1,
       HC_NI1, HC_TI1, HC_K11, HC_K12, HC_K22, HC_IXX, HC_IXY, HC_IYY, HC_COUNT };
// position-phase overlay of a contact slot
enum { PC_META = HC_META, PC_LNX, PC_LNY, PC_LPX, PC_LPY, PC_P0X, PC_P0Y, PC_P1X, PC_P1Y, PC_RADB };

struct Terrain {           // read-only, shared by every creature (Modular2DEnv.py:294-306)
    float v1x[RB_MAX_EDGES], v1y[RB_MAX_EDGES], v2x[RB_MAX_EDGES], v2y[RB_MAX_EDGES];
    float flx[RB_MAX_EDGES], fly[RB_MAX_EDGES], fhx[RB_MAX_EDGES], fhy[RB_MAX_EDGES];   // fat AABBs of the edge proxies
    int n_edges;
    float step;
};

struct Consts {
    float dt, gravity_y, friction;   // friction = sqrtf(module * terrain)
    int vel_iters, pos_iters, continuous, allow_sleep, terminate, evaluation_steps;
    double p_gain, wod_speed, env_length;
};

// device copy of the flattened population table (+ island joint order)
struct DevPop {
    const int32_t* body_off; const uint8_t* shape; const float *hx, *hy, *x0, *y0, *a0;
    const int16_t* joint_parent; const float *anchor_a, *anchor_b, *lower, *upper, *max_torque;
    const double* ctrl; const uint8_t* joint_order;
};
// work counters kept in registers and flushed once per launch
struct Cnt { unsigned int c[REM2D_N_COUNTERS]; };   // per lane per launch; summed into 64-bit totals

// When the queue-mode episode kernel hands a creature over to the tail mode (launches of the same kernel).
struct ParkPolicy {
    int ticks;        // park a creature that is still alive after this many ticks (0: never park)
    int cap;          // at most this many creatures of the class are parked
    // Always off (lead_x = 0, late_from = class size): the rejected lead and late-start park tests of the episode kernel.
    // Deleting them takes episode_kernel from 202 to 200 registers; at 200, 10 instead of 9 warps fit per SM, so the
    // occupancy-based grid sizing (size_grids, rem2d_host_util.h) hands out other first-wave grids.
    float lead_x;     // > 0: park a creature whose root has reached x >= lead_x after lead_from ticks
    int lead_from;
    int late_from;    // creatures pulled from this position of the class queue on park after late_ticks ticks
    int late_ticks;
    // diagnostics (trace option): every 4th tick lane 0 of each warp records {globaltimer us, live creatures | tick << 8 |
    // smid << 24}; REM2D_TRACE_SAMPLES entries per warp. Null in production.
    unsigned int* trace;
    unsigned int* tail_trace;   // per park slot: {us parked, us tail warp started, us finished, ticks run by the tail warp}
    int wide_gs;      // a creature whose group already has this many lanes (log2) is not parked: the tail launch is no wider
};
#define REM2D_TRACE_SAMPLES 1024

// The class queue of an episode launch and where finished creatures are written (indexed by creature).
struct EpisodeQueue {
    const int* __restrict__ order; int n_order; int* queue;      // creatures in pull order; pull counter
    DevPop p; int max_ticks;
    double* fitness; int* ticks; int* alive; int* status;
};

// Episode statistics (include/rem2d_stats.h, rem2d_episode_stats), accumulated by the statistics images of the episode kernel only
// (-DREM2D_STATS): indexed by creature, ground_ticks by global body index body_off[c] + b. Zeroed when a creature is pulled.
struct EpisodeStats {
    int32_t* end_reason; float* max_x; double* joint_work; int32_t* airborne_ticks; int32_t* ground_ticks;
    const int32_t* body_off;
};

// Per-joint feedback policy (include/rem2d_policy.h), evaluated by the policy images only (-DREM2D_POLICY): the weights of global
// joint j start at w + j * (10 * n_hidden + 1); body_off locates a creature's first joint (body_off[c] - c).
struct PolicyWeights {
    const double* w; const int32_t* body_off; int n_hidden;
};

// Capacities and section offsets of one capacity class. The layout is a RUN-TIME value (kernel parameter, i.e. constant
// bank): all classes execute the SAME code image. With one template instantiation per class, warps of 7 different
// 365 KB kernels shared each SM's instruction cache and every class ran 1.4-5x slower than alone (measured, DESIGN.md).
// Within a section the words are element-major (element * FIELD_COUNT + field), so that field offsets are immediates.
struct Layout {
    int nb, nj, nc, nt;                        // bodies, joints, contact-pool slots, hot (shared memory) touching contacts
    int off_joint, off_cont, off_edge, off_spill, off_ring, words;      // cold block, words per lane (bodies start at S_COUNT)
    int hot_words;                                            // hot block with one lane per creature, words per lane
};
#define RB_RING 8             // end-of-iteration body poses kept by the pipelined position sweeps (iterations in flight)
#define RB_SCHED_ROWS 20      // slots per period of the static schedule (shared-memory rows per warp); longer periods fall back
#define RB_MAX_SKEW 24        // iteration skew bound of a schedule (ring depth of the position-phase end-of-iteration states)
__host__ __device__ inline Layout make_layout(int NB, int NC, int NT) {
    Layout L;
    L.nb = NB; L.nj = NB - 1 > 0 ? NB - 1 : 1; L.nc = NC; L.nt = NT;
    L.off_joint = S_COUNT + BF_COUNT * NB;
    L.off_cont = L.off_joint + JF_COUNT * L.nj;
    L.off_edge = L.off_cont + CF_COUNT * NC;                  // alpha0 of the static edge bodies
    L.off_spill = L.off_edge + RB_MAX_EDGES;                  // touching contacts beyond NT spill to HBM
    L.off_ring = L.off_spill + HC_COUNT * (NC - NT);          // RB_RING x NB x (cx, cy, a)
    L.words = L.off_ring + RB_RING * 3 * NB;
    L.hot_words = HB_COUNT * NB + HJ_COUNT * L.nj + HC_COUNT * NT;
    return L;
}
// Hot block of one warp for groups of G = 2^gs lanes per creature: rows of 32 words. Element e of a creature lives in row
// (section + (e >> gs) * FIELD_COUNT + field), column (group * G + (e & (G-1))). Sections: bodies, joints, hot contacts, then
// (G > 1 only) one scratch word per body for the scheduler and RB_SCHED_ROWS rows of schedule entries (column = lane).
struct HotLayout { int hj_off, hc_off, aux_off, sch_off, rows; };
__host__ __device__ inline HotLayout make_hot_layout(const Layout& L, int gs) {
    const int G = 1 << gs;
    const int rb = (L.nb + G - 1) >> gs, rj = (L.nj + G - 1) >> gs, rt = (L.nt + G - 1) >> gs;
    HotLayout H;
    H.hj_off = HB_COUNT * rb;
    H.hc_off = H.hj_off + HJ_COUNT * rj;
    H.aux_off = H.hc_off + HC_COUNT * rt;
    H.sch_off = H.aux_off + (gs ? rb : 0);
    H.rows = H.sch_off + (gs ? RB_SCHED_ROWS : 0);
    return H;
}

// Observation of one creature at the end of a tick (include/rem2d_control.h, rem2d_read_observations) from its cold column g,
// nb bodies: the outputs are already offset to the creature's first joint (joint_angle, joint_speed), its root row (root[6])
// and its first body (ground). The values are those rem2d_read_state decodes from the same column.
__device__ __forceinline__ void observe_column(const float* g, const Layout& L, int nb, float* joint_angle, float* joint_speed,
                                               float* root, int32_t* ground) {
    auto B = [&](int f, int i) { return g[(S_COUNT + i * BF_COUNT + f) * 32]; };
    for (int j = 0; j < nb - 1; ++j) {
        const int a = __float_as_int(g[(L.off_joint + j * JF_COUNT + JF_META) * 32]) & 0xff, b = j + 1;
        joint_angle[j] = B(BF_A, b) - B(BF_A, a) - 0.0f;          // the currentAngle of Sim::tick_pre
        joint_speed[j] = B(BF_W, b) - B(BF_W, a);
    }
    root[0] = B(BF_CX, 0); root[1] = B(BF_CY, 0); root[2] = B(BF_A, 0);
    root[3] = B(BF_VX, 0); root[4] = B(BF_VY, 0); root[5] = B(BF_W, 0);
    unsigned long long m = 0ull;                                   // bodies with a touching terrain contact
    const int n_pool = __float_as_int(g[S_NC * 32]);
    for (int q = 0; q < n_pool; ++q) {
        const int key = __float_as_int(g[(L.off_cont + q * CF_COUNT + CF_KEY) * 32]);
        if (((key >> 16) & 0xff) & CK_TOUCHING) m |= 1ull << (key & 0xff);
    }
    for (int b = 0; b < nb; ++b) ground[b] = (int32_t)((m >> b) & 1ull);
}

// One creature. All G lanes of the creature's group hold the same Sim (same cold column `g`, same hot column base `h`) and call
// every member function TOGETHER; functions marked "leader" are executed by sub == 0 only and everything the other lanes need
// afterwards is broadcast or read after a group barrier. With G == 1 the code degenerates to the sequential per-lane form.
// Group barriers use the group's own lane mask, so groups of a warp never wait for each other inside a phase.
// Phase timing (diagnostic builds only, -DREM2D_PHASE_TIMING: tools/phase_breakdown.py): clock64 deltas per tick phase
#ifdef REM2D_PHASE_TIMING
#define REM2D_N_PHASES 16
#define PHASE(i) do { long long t_ = clock64(); ph[phase_cur] += t_ - phase_t0; phase_t0 = t_; phase_cur = (i); } while (0)
#else
#define PHASE(i) do { } while (0)
#endif
enum { PH_LOOP, PH_CONTROL, PH_COLLIDE, PH_STAGE, PH_SCHEDULE, PH_VELOCITY, PH_STORE, PH_POSITION, PH_FINALIZE, PH_FINDNEW, PH_TOI_SCAN,
       PH_TOI_EVENTS, PH_BUILD, PH_PARK };

struct Sim {
    Layout L;
#ifdef REM2D_PHASE_TIMING
public:
    long long ph[REM2D_N_PHASES]; long long phase_t0; int phase_cur;
#endif
    int gs, G, sub, lead;     // lanes per creature = 1 << gs; my index in the group; absolute lane of the group leader
    unsigned gmask;           // lanes of my group
    int hj_off, hc_off, aux_off, sch_off;   // section rows of the hot block for this gs
    int e_shift, e_mask;      // element -> (row, column): (e >> gs, e & (G-1))
    float* g;                 // cold block of this batch, already offset by the creature's column
    float* h;                 // hot block of this warp in shared memory, already offset by the group's first column
    const Terrain* __restrict__ ter;
    const Consts* __restrict__ k;
    Cnt cnt;
    int nb, nj;
    // schedule of the current tick (group-uniform): period (slots), largest iteration skew; sched_P == 0: sequential fallback
    int sched_P, sched_smax;
#ifdef REM2D_STATS
    EpisodeStats st;          // where the statistics go, and the creature this group is ticking (set before every tick)
    int st_c;
#endif
#ifdef REM2D_TARGETS
    const double* tgt;        // caller-supplied target angles of this creature's joints (step_kernel_targets, include/rem2d_control.h)
#endif
#ifdef REM2D_POLICY
    PolicyWeights pol;        // the population's policy, and the weights of this creature's first joint (set before every tick)
    const double* __restrict__ pw;
    __device__ __forceinline__ void set_policy_creature(int c) { pw = pol.w + (size_t)(pol.body_off[c] - c) * (10 * pol.n_hidden + 1); }
#endif

    // ---- accessors
    __device__ __forceinline__ float& S(int f) { return g[f * 32]; }
    __device__ __forceinline__ int Si(int f) { return __float_as_int(g[f * 32]); }
    __device__ __forceinline__ void setSi(int f, int v) { g[f * 32] = __int_as_float(v); }
    __device__ __forceinline__ double Sd(int f) { return __hiloint2double(Si(f + 1), Si(f)); }
    __device__ __forceinline__ void setSd(int f, double v) { setSi(f, __double2loint(v)); setSi(f + 1, __double2hiint(v)); }
    __device__ __forceinline__ float& B(int f, int i) { return g[(S_COUNT + i * BF_COUNT + f) * 32]; }
    __device__ __forceinline__ int Bi(int f, int i) { return __float_as_int(B(f, i)); }
    __device__ __forceinline__ void setBi(int f, int i, int v) { B(f, i) = __int_as_float(v); }
    __device__ __forceinline__ float& J(int f, int j) { return g[(L.off_joint + j * JF_COUNT + f) * 32]; }
    __device__ __forceinline__ int Ji(int f, int j) { return __float_as_int(J(f, j)); }
    __device__ __forceinline__ void setJi(int f, int j, int v) { J(f, j) = __int_as_float(v); }
    __device__ __forceinline__ double Jd(int f, int j) { return __hiloint2double(Ji(f + 1, j), Ji(f, j)); }
    __device__ __forceinline__ void setJd(int f, int j, double v) { setJi(f, j, __double2loint(v)); setJi(f + 1, j, __double2hiint(v)); }
    __device__ __forceinline__ float& C(int f, int c) { return g[(L.off_cont + c * CF_COUNT + f) * 32]; }
    __device__ __forceinline__ int Ci(int f, int c) { return __float_as_int(C(f, c)); }
    __device__ __forceinline__ void setCi(int f, int c, int v) { C(f, c) = __int_as_float(v); }
    __device__ __forceinline__ float& EA(int e) { return g[(L.off_edge + e) * 32]; }
    __device__ __forceinline__ float& RING(int r, int b, int f) { return g[(L.off_ring + (r * L.nb + b) * 3 + f) * 32]; }
    // lane = lane index in the warp; hot = the warp's hot block
    __device__ __forceinline__ void set_group(int gshift, int lane, float* hot) {
        gs = gshift; G = 1 << gs; sub = lane & (G - 1); lead = lane & ~(G - 1);
        gmask = gs == 5 ? 0xffffffffu : (((1u << G) - 1u) << lead);
        const HotLayout H = make_hot_layout(L, gs);
        hj_off = H.hj_off; hc_off = H.hc_off; aux_off = H.aux_off; sch_off = H.sch_off;
        e_shift = gs; e_mask = G - 1;
        h = hot + lead;
        sched_P = 0; sched_smax = 0;
    }
    // ---- group primitives
    __device__ __forceinline__ void gsync() { __syncwarp(gmask); }
    __device__ __forceinline__ int bcast(int v) { return gs ? __shfl_sync(gmask, v, lead) : v; }
    __device__ __forceinline__ bool leader() const { return sub == 0; }
    __device__ __forceinline__ float group_min(float v) {
        for (int o = G >> 1; o > 0; o >>= 1) v = min2(v, __shfl_xor_sync(gmask, v, o));
        return v;
    }
    __device__ __forceinline__ bool group_any(bool v) { return gs ? (__ballot_sync(gmask, v) != 0u) : v; }
    // "does any lane that is executing this instruction together with me ..." - a scheduling hint only (results never depend on it)
    __device__ __forceinline__ bool warp_any_converged(bool v) {
#ifdef REM2D_EMU
        return group_any(v);
#else
        return __any_sync(__activemask(), v) != 0;
#endif
    }
    __device__ __forceinline__ bool group_all(bool v) { return gs ? (__ballot_sync(gmask, v) == gmask) : v; }
    __device__ __forceinline__ float* hot_elem(int section, int count, int e) {     // field 0 of element e
        return h + ((section + (e >> e_shift) * count) << 5) + (e & e_mask);
    }
    __device__ __forceinline__ float& HB(int f, int i) { return hot_elem(0, HB_COUNT, i)[f * 32]; }
    __device__ __forceinline__ float& HJ(int f, int j) { return hot_elem(hj_off, HJ_COUNT, j)[f * 32]; }
    __device__ __forceinline__ int HJi(int f, int j) { return __float_as_int(HJ(f, j)); }
    __device__ __forceinline__ int& AUX(int b) { return *(int*)hot_elem(aux_off, 1, b); }           // scheduler scratch, one word per body
    __device__ __forceinline__ int& SCH(int p, int lane_in_group) { return *(int*)(h + ((sch_off + p) << 5) + lane_in_group); }
    // Hot contact slot t: shared memory for t < NT, a spill region of the cold block otherwise. The callee gets the
    // address of field 0 and the stride between fields; the two call sites are specialised by the compiler
    // (LDS/STS vs LDG/STG).
    template <class F>
    __device__ __forceinline__ void for_contacts(int nt, F f) {
        const int n1 = nt < L.nt ? nt : L.nt;
        for (int t = 0; t < n1; ++t) f(hot_elem(hc_off, HC_COUNT, t), 32, t);
        for (int t = L.nt; t < nt; ++t) f(g + (L.off_spill + (t - L.nt) * HC_COUNT) * 32, 32, t);
    }
    template <class F>
    __device__ __forceinline__ void with_contact(int t, F f) {
        if (t < L.nt) f(hot_elem(hc_off, HC_COUNT, t), 32);
        else f(g + (L.off_spill + (t - L.nt) * HC_COUNT) * 32, 32);
    }

    __device__ __forceinline__ int key_body(int key) { return key & 0xff; }
    __device__ __forceinline__ int key_edge(int key) { return (key >> 8) & 0xff; }
    __device__ __forceinline__ int key_flags(int key) { return (key >> 16) & 0xff; }
    __device__ __forceinline__ int key_toicount(int key) { return (key >> 24) & 0xff; }

    // ---- bodies
    __device__ __forceinline__ void set_awake(int b, bool flag) {
        int fl = Bi(BF_FLAGS, b);
        if (flag) {
            if (!(fl & BFL_AWAKE)) { setBi(BF_FLAGS, b, fl | BFL_AWAKE); B(BF_SLEEP, b) = 0.0f; }
        } else {
            setBi(BF_FLAGS, b, fl & ~BFL_AWAKE);
            B(BF_SLEEP, b) = 0.0f;
            B(BF_VX, b) = 0.0f; B(BF_VY, b) = 0.0f; B(BF_W, b) = 0.0f;
        }
    }
    __device__ __forceinline__ void sync_transform(int b) {     // localCenter == 0: xf.p == sweep.c
        Rot q = rot_set(B(BF_A, b));
        B(BF_QS, b) = q.s; B(BF_QC, b) = q.c;
    }
    // tight AABB of the shape at pose (p, q)   (b2PolygonShape/b2CircleShape::ComputeAABB)
    __device__ __forceinline__ void shape_aabb(int b, V2 p, Rot q, V2& lo, V2& hi) {
        float hx = B(BF_HX, b), hy = B(BF_HY, b);
        if (Bi(BF_FLAGS, b) & BFL_CIRCLE) {
            V2 z = mk(0.0f, 0.0f);
            V2 c = p + rmul(q, z);
            lo = mk(c.x - hx, c.y - hx); hi = mk(c.x + hx, c.y + hx);
            return;
        }
        V2 v0 = xmul(p, q, mk(-hx, -hy));
        lo = v0; hi = v0;
        V2 v;
        v = xmul(p, q, mk(hx, -hy)); lo = mk(min2(lo.x, v.x), min2(lo.y, v.y)); hi = mk(max2(hi.x, v.x), max2(hi.y, v.y));
        v = xmul(p, q, mk(hx, hy));  lo = mk(min2(lo.x, v.x), min2(lo.y, v.y)); hi = mk(max2(hi.x, v.x), max2(hi.y, v.y));
        v = xmul(p, q, mk(-hx, hy)); lo = mk(min2(lo.x, v.x), min2(lo.y, v.y)); hi = mk(max2(hi.x, v.x), max2(hi.y, v.y));
        lo = mk(lo.x - RB_POLY_RADIUS, lo.y - RB_POLY_RADIUS);
        hi = mk(hi.x + RB_POLY_RADIUS, hi.y + RB_POLY_RADIUS);
    }
    // b2Body::SynchronizeFixtures -> b2DynamicTree::MoveProxy (fat AABB rule)
    __device__ void synchronize_fixtures(int b) {
        Rot q1 = rot_set(B(BF_A0, b));
        V2 p1 = mk(B(BF_C0X, b), B(BF_C0Y, b));
        V2 p2 = mk(B(BF_CX, b), B(BF_CY, b));
        Rot q2; q2.s = B(BF_QS, b); q2.c = B(BF_QC, b);
        V2 lo1, hi1, lo2, hi2;
        shape_aabb(b, p1, q1, lo1, hi1);
        shape_aabb(b, p2, q2, lo2, hi2);
        V2 lo = mk(min2(lo1.x, lo2.x), min2(lo1.y, lo2.y)), hi = mk(max2(hi1.x, hi2.x), max2(hi1.y, hi2.y));
        V2 disp = p2 - p1;
        float flx = B(BF_FLX, b), fly = B(BF_FLY, b), fhx = B(BF_FHX, b), fhy = B(BF_FHY, b);
        if (flx <= lo.x && fly <= lo.y && hi.x <= fhx && hi.y <= fhy) return;
        lo = mk(lo.x - RB_AABB_EXT, lo.y - RB_AABB_EXT);
        hi = mk(hi.x + RB_AABB_EXT, hi.y + RB_AABB_EXT);
        V2 d = RB_AABB_MULT * disp;
        if (d.x < 0.0f) lo.x += d.x; else hi.x += d.x;
        if (d.y < 0.0f) lo.y += d.y; else hi.y += d.y;
        B(BF_FLX, b) = lo.x; B(BF_FLY, b) = lo.y; B(BF_FHX, b) = hi.x; B(BF_FHY, b) = hi.y;
        setBi(BF_FLAGS, b, Bi(BF_FLAGS, b) | BFL_MOVED);
    }
    __device__ __forceinline__ bool overlap_edge(int e, int b) {
        return overlap_edge_box(e, B(BF_FLX, b), B(BF_FLY, b), B(BF_FHX, b), B(BF_FHY, b));
    }
    __device__ __forceinline__ bool overlap_edge_box(int e, float blx, float bly, float bhx, float bhy) {
        float alx = __ldg(&ter->flx[e]), aly = __ldg(&ter->fly[e]), ahx = __ldg(&ter->fhx[e]), ahy = __ldg(&ter->fhy[e]);
        float d1x = blx - ahx, d1y = bly - ahy, d2x = alx - bhx, d2y = aly - bhy;
        if (d1x > 0.0f || d1y > 0.0f) return false;
        if (d2x > 0.0f || d2y > 0.0f) return false;
        return true;
    }


    // ---- world construction: b2Body/b2Fixture creation (mass data, sweep, proxy fat AABB), joints, controllers and
    // episode scalars of creature c (c < 0: empty column). Mirrors oracle world_build()/body_init(). Group-cooperative: bodies,
    // joints and the edge table are strided over the lanes of the group; ends with a group barrier.
    __device__ void build_world(const DevPop& p, int c) {
        PHASE(PH_BUILD);
        if (c < 0) {
            if (leader()) { for (int w = 0; w < S_COUNT; ++w) g[w * 32] = 0.0f; setSi(S_NB, 0); setSi(S_ALIVE, 0); }
            nb = 0; nj = 0;
            gsync();
            return;
        }
        const int b0 = p.body_off[c], j0 = b0 - c;
        nb = p.body_off[c + 1] - b0; nj = nb - 1;
        if (leader()) {
            for (int w = 0; w < S_COUNT; ++w) g[w * 32] = 0.0f;
            setSi(S_NB, nb); setSi(S_NC, 0); setSi(S_ALIVE, 1); setSi(S_TICKS, 0);
            setSd(S_WOD_LO, 0.0); setSd(S_FIT_LO, 0.0);
            S(S_INVDT0) = 0.0f; setSi(S_NEWFIX, 1); setSi(S_STATUS, 0); setSi(S_NADV, 0);
        }
        for (int e = sub; e < RB_MAX_EDGES; e += G) EA(e) = 0.0f;
        for (int i = sub; i < nb; i += G) {
            const int shape = p.shape[b0 + i];
            const float hx = p.hx[b0 + i], hy = p.hy[b0 + i];
            const float density = 1.0f;
            float mass, I;
            V2 center;
            if (shape == REM2D_SHAPE_CIRCLE) {
                mass = density * RB_PI * hx * hx;
                center = mk(0.0f, 0.0f);
                I = mass * (0.5f * hx * hx + dot(center, center));
            } else {
                V2 v[4] = { mk(-hx, -hy), mk(hx, -hy), mk(hx, hy), mk(-hx, hy) };
                V2 cen = mk(0.0f, 0.0f), s = mk(0.0f, 0.0f);
                float area = 0.0f, II = 0.0f;
                for (int q = 0; q < 4; ++q) s = s + v[q];
                s = (1.0f / 4.0f) * s;
                const float k_inv3 = 1.0f / 3.0f;
                for (int q = 0; q < 4; ++q) {
                    V2 e1 = v[q] - s, e2 = q + 1 < 4 ? v[q + 1] - s : v[0] - s;
                    float D = cross(e1, e2);
                    float triangleArea = 0.5f * D;
                    area += triangleArea;
                    cen = cen + (triangleArea * k_inv3) * (e1 + e2);
                    float intx2 = e1.x * e1.x + e2.x * e1.x + e2.x * e2.x;
                    float inty2 = e1.y * e1.y + e2.y * e1.y + e2.y * e2.y;
                    II += (0.25f * k_inv3 * D) * (intx2 + inty2);
                }
                mass = density * area;
                cen = (1.0f / area) * cen;
                center = cen + s;
                I = density * II;
                I += mass * (dot(center, center) - dot(cen, cen));
            }
            float invMass, invI;
            V2 localCenter = mass * center;
            if (mass > 0.0f) { invMass = 1.0f / mass; localCenter = invMass * localCenter; }
            else { mass = 1.0f; invMass = 1.0f; }
            if (I > 0.0f) { I -= mass * dot(localCenter, localCenter); invI = 1.0f / I; }
            else { invI = 0.0f; }
            const float x = p.x0[b0 + i], y = p.y0[b0 + i], a = p.a0[b0 + i];
            Rot q = rot_set(a);
            V2 cpos = xmul(mk(x, y), q, localCenter);          // localCenter == 0 for boxes and circles
            B(BF_CX, i) = cpos.x; B(BF_CY, i) = cpos.y; B(BF_A, i) = a;
            B(BF_C0X, i) = cpos.x; B(BF_C0Y, i) = cpos.y; B(BF_A0, i) = a; B(BF_ALPHA0, i) = 0.0f;
            B(BF_VX, i) = 0.0f; B(BF_VY, i) = 0.0f; B(BF_W, i) = 0.0f;
            B(BF_QS, i) = q.s; B(BF_QC, i) = q.c;
            B(BF_SLEEP, i) = 0.0f; B(BF_INVM, i) = invMass; B(BF_INVI, i) = invI;
            B(BF_HX, i) = hx; B(BF_HY, i) = hy;
            setBi(BF_FLAGS, i, BFL_AWAKE | BFL_MOVED | (shape == REM2D_SHAPE_CIRCLE ? BFL_CIRCLE : 0));
            V2 lo, hi;
            shape_aabb(i, mk(x, y), q, lo, hi);
            B(BF_FLX, i) = lo.x - RB_AABB_EXT; B(BF_FLY, i) = lo.y - RB_AABB_EXT;
            B(BF_FHX, i) = hi.x + RB_AABB_EXT; B(BF_FHY, i) = hi.y + RB_AABB_EXT;
        }
        for (int j = sub; j < nj; j += G) {
            setJi(JF_META, j, (int)p.joint_parent[j0 + j] | ((int)p.joint_order[j0 + j] << 8));
            J(JF_LAAX, j) = p.anchor_a[2 * (j0 + j)]; J(JF_LAAY, j) = p.anchor_a[2 * (j0 + j) + 1];
            J(JF_LABX, j) = p.anchor_b[2 * (j0 + j)]; J(JF_LABY, j) = p.anchor_b[2 * (j0 + j) + 1];
            J(JF_IMPX, j) = 0.0f; J(JF_IMPY, j) = 0.0f; J(JF_IMPZ, j) = 0.0f; J(JF_MIMP, j) = 0.0f;
            J(JF_MSPEED, j) = 0.0f; setJi(JF_LIMIT, j, 0);
            J(JF_LOWER, j) = p.lower[j0 + j]; J(JF_UPPER, j) = p.upper[j0 + j]; J(JF_MAXT, j) = p.max_torque[j0 + j];
            const double* cc = &p.ctrl[(size_t)(b0 + j + 1) * 5];     // controller of body j+1 drives joint j
            setJd(JF_AMP, j, cc[0]); setJd(JF_PHASE, j, cc[1]); setJd(JF_FREQ, j, cc[2]);
            setJd(JF_OFFS, j, cc[3]); setJd(JF_ISTATE, j, cc[4]);
        }
        gsync();
    }

    // ---- contact pool (creation order; index nc-1 is the newest == head of Box2D's lists)
    __device__ int find_contact(int nc, int b, int e) {
        int want = b | (e << 8);
        for (int i = 0; i < nc; ++i)
            if ((Ci(CF_KEY, i) & 0xffff) == want) return i;
        return -1;
    }
    // b2ContactManager::FindNewContacts: new pairs in ascending (edge, body) order, each becomes the newest
    // The first pass asks, body by body over the body's own edge range, whether ANY new pair exists (almost never: a handful
    // per episode); only then the pairs are enumerated in Box2D's order over the union of the ranges.
    __device__ void find_new_contacts() {
        int elo = ter->n_edges, ehi = -1;
        bool any = false, has = false;
        int nc = Si(S_NC);
        for (int b = 0; b < nb; ++b) {
            if (!(Bi(BF_FLAGS, b) & BFL_MOVED)) continue;
            any = true;
            const float blx = B(BF_FLX, b), bly = B(BF_FLY, b), bhx = B(BF_FHX, b), bhy = B(BF_FHY, b);
            double l = floor(((double)blx - 0.25) / (double)ter->step) - 1.0;
            double u = ceil(((double)bhx + 0.25) / (double)ter->step) + 1.0;
            int il = l < 0.0 ? 0 : (l > (double)(ter->n_edges - 1) ? ter->n_edges : (int)l);
            int iu = u < 0.0 ? -1 : (u > (double)(ter->n_edges - 1) ? ter->n_edges - 1 : (int)u);
            if (il < elo) elo = il;
            if (iu > ehi) ehi = iu;
            if (!has)
                for (int e = il; e <= iu; ++e)
                    if (overlap_edge_box(e, blx, bly, bhx, bhy) && find_contact(nc, b, e) < 0) { has = true; break; }
        }
        if (!any) return;
        if (!has) { elo = 0; ehi = -1; }
        for (int e = elo; e <= ehi; ++e) {
            for (int b = 0; b < nb; ++b) {
                if (!(Bi(BF_FLAGS, b) & BFL_MOVED)) continue;
                if (!overlap_edge(e, b)) continue;
                if (find_contact(nc, b, e) >= 0) continue;
                if (nc == L.nc) { setSi(S_STATUS, Si(S_STATUS) | ST_POOL_OVERFLOW); continue; }
                setCi(CF_KEY, nc, b | (e << 8) | (CK_ENABLED << 16));
                C(CF_TOI, nc) = 1.0f;
                C(CF_P0N, nc) = 0.0f; C(CF_P0T, nc) = 0.0f; C(CF_P1N, nc) = 0.0f; C(CF_P1T, nc) = 0.0f;
                ++nc;
                set_awake(b, true);
            }
        }
        setSi(S_NC, nc);
        for (int b = 0; b < nb; ++b) setBi(BF_FLAGS, b, Bi(BF_FLAGS, b) & ~BFL_MOVED);
    }
    // Group-cooperative FindNewContacts (G > 1): the broad-phase queries of the moved proxies - edge range of the fat AABB,
    // overlap tests against the edge proxies, "is this pair already a contact" scans of the pool, all of them chains of cold
    // loads - are strided over the lanes, one body per lane at a time; each body leaves a bit mask of its NEW pairs in its
    // scratch word, and the leader turns the masks into contacts in Box2D's pair order (ascending edge, then body). New pairs
    // are rare (a handful per episode), so the leader's part is usually empty. Ends with a group barrier.
    __device__ void find_new_contacts_group() {
        if (gs == 0) { find_new_contacts(); return; }
        const int nc0 = bcast(Si(S_NC));
        bool has = false, special = false;
        for (int b = sub; b < nb; b += G) {
            int w = 0;
            if (Bi(BF_FLAGS, b) & BFL_MOVED) {
                double l = floor(((double)B(BF_FLX, b) - 0.25) / (double)ter->step) - 1.0;
                double u = ceil(((double)B(BF_FHX, b) + 0.25) / (double)ter->step) + 1.0;
                int il = l < 0.0 ? 0 : (l > (double)(ter->n_edges - 1) ? ter->n_edges : (int)l);
                int iu = u < 0.0 ? -1 : (u > (double)(ter->n_edges - 1) ? ter->n_edges - 1 : (int)u);
                if (iu - il >= 24) special = true;            // (a proxy spanning > 24 edges: the leader scans it the slow way)
                else {
                    int mask = 0;
                    const float blx = B(BF_FLX, b), bly = B(BF_FLY, b), bhx = B(BF_FHX, b), bhy = B(BF_FHY, b);
                    for (int e = il; e <= iu; ++e)
                        if (overlap_edge_box(e, blx, bly, bhx, bhy) && find_contact(nc0, b, e) < 0) mask |= 1 << (e - il);
                    if (mask) { w = il | (mask << 8); has = true; }
                }
            }
            AUX(b) = w;
        }
        special = group_any(special);
        has = group_any(has);
        gsync();                              // publishes the scratch words
        if (leader()) {
            if (special) find_new_contacts();
            else if (has) {
                int nc = nc0;
                int elo = ter->n_edges, ehi = -1;
                for (int b = 0; b < nb; ++b) {
                    const int w = AUX(b);
                    if (!w) continue;
                    const int il = w & 0xff, m = (int)((unsigned)w >> 8);
                    if (il < elo) elo = il;
                    const int top = il + 31 - __clz(m);
                    if (top > ehi) ehi = top;
                }
                for (int e = elo; e <= ehi; ++e)
                    for (int b = 0; b < nb; ++b) {
                        const int w = AUX(b);
                        const int k = e - (w & 0xff);
                        if (!w || k < 0 || k >= 24 || !(((unsigned)w >> (8 + k)) & 1u)) continue;
                        if (nc == L.nc) { setSi(S_STATUS, Si(S_STATUS) | ST_POOL_OVERFLOW); continue; }
                        setCi(CF_KEY, nc, b | (e << 8) | (CK_ENABLED << 16));
                        C(CF_TOI, nc) = 1.0f;
                        C(CF_P0N, nc) = 0.0f; C(CF_P0T, nc) = 0.0f; C(CF_P1N, nc) = 0.0f; C(CF_P1T, nc) = 0.0f;
                        ++nc;
                        set_awake(b, true);
                    }
                setSi(S_NC, nc);
            }
        }
        gsync();
        if (!special)
            for (int b = sub; b < nb; b += G) setBi(BF_FLAGS, b, Bi(BF_FLAGS, b) & ~BFL_MOVED);
        gsync();
    }
    __device__ void destroy_contact(int i) {
        int nc = Si(S_NC);
        int key = Ci(CF_KEY, i);
        if ((key_flags(key) >> CK_COUNT_SHIFT) & 3) set_awake(key_body(key), true);
        for (int k = i; k < nc - 1; ++k) {
            float tmp[CF_COUNT];                      // all loads first: 16 independent global loads in flight
#pragma unroll
            for (int f = 0; f < CF_COUNT; ++f) tmp[f] = C(f, k + 1);
#pragma unroll
            for (int f = 0; f < CF_COUNT; ++f) C(f, k) = tmp[f];
        }
        setSi(S_NC, nc - 1);
    }

    // ---- narrow phase. Edge frame == world frame (static body at the origin).
    struct Clip { V2 v; int id; };   // id = indexA | indexB<<8 | typeA<<16 | typeB<<24  (vertex 0, face 1)
    __device__ __forceinline__ int mkid(int ia, int ib, int ta, int tb) { return ia | (ib << 8) | (ta << 16) | (tb << 24); }
    __device__ __forceinline__ int clip_segment(Clip out[2], const Clip in[2], V2 normal, float offset, int vertexIndexA) {
        int n = 0;
        float d0 = dot(normal, in[0].v) - offset;
        float d1 = dot(normal, in[1].v) - offset;
        if (d0 <= 0.0f) out[n++] = in[0];
        if (d1 <= 0.0f) out[n++] = in[1];
        if (d0 * d1 < 0.0f) {
            float interp = d0 / (d0 - d1);
            out[n].v = in[0].v + interp * (in[1].v - in[0].v);
            out[n].id = mkid(vertexIndexA, (in[0].id >> 8) & 0xff, 0, 1);
            ++n;
        }
        return n;
    }

    // Evaluate the manifold of contact c at the body's current transform and write it to the pool
    // (b2Contact::Update incl. warm-start impulse matching by feature id).
    __device__ void contact_update(int c) {
        cnt.c[REM2D_CNT_NARROW]++;
        int key = Ci(CF_KEY, c);
        int b = key_body(key), e = key_edge(key);
        int flags = key_flags(key);
        int oldCount = (flags >> CK_COUNT_SHIFT) & 3;
        int oldId0 = Ci(CF_P0ID, c), oldId1 = Ci(CF_P1ID, c);
        float oldN0 = C(CF_P0N, c), oldT0 = C(CF_P0T, c), oldN1 = C(CF_P1N, c), oldT1 = C(CF_P1T, c);
        bool wasTouching = (flags & CK_TOUCHING) != 0;
        flags |= CK_ENABLED;
        V2 v1 = mk(__ldg(&ter->v1x[e]), __ldg(&ter->v1y[e])), v2 = mk(__ldg(&ter->v2x[e]), __ldg(&ter->v2y[e]));
        V2 p = mk(B(BF_CX, b), B(BF_CY, b));
        Rot q; q.s = B(BF_QS, b); q.c = B(BF_QC, b);
        int type = 0, count = 0;
        V2 ln = mk(0.0f, 0.0f), lp = mk(0.0f, 0.0f), pt[2];
        int pid[2];
        pt[0] = pt[1] = mk(0.0f, 0.0f); pid[0] = pid[1] = 0;
        if (Bi(BF_FLAGS, b) & BFL_CIRCLE) {
            // b2CollideEdgeAndCircle, circle centre m_p = 0 -> Q = xfB.p
            float rad = RB_POLY_RADIUS + B(BF_HX, b);
            V2 Q = p, A = v1, Bv = v2, ee = Bv - A;
            float u = dot(ee, Bv - Q), v = dot(ee, Q - A);
            if (v <= 0.0f) {
                V2 d = Q - A; float dd = dot(d, d);
                if (!(dd > rad * rad)) { count = 1; type = MT_CIRCLES; lp = A; pid[0] = mkid(0, 0, 0, 0); }
            } else if (u <= 0.0f) {
                V2 d = Q - Bv; float dd = dot(d, d);
                if (!(dd > rad * rad)) { count = 1; type = MT_CIRCLES; lp = Bv; pid[0] = mkid(1, 0, 0, 0); }
            } else {
                float den = dot(ee, ee);
                V2 P = (1.0f / den) * (u * A + v * Bv);
                V2 d = Q - P; float dd = dot(d, d);
                if (!(dd > rad * rad)) {
                    V2 n = mk(-ee.y, ee.x);
                    if (dot(n, Q - A) < 0.0f) n = mk(-n.x, -n.y);
                    normalize(n);
                    count = 1; type = MT_FACE_A; ln = n; lp = A; pid[0] = mkid(0, 0, 1, 0);
                }
            }
        } else {
            // b2CollideEdgeAndPolygon (b2EPCollider) without ghost vertices; xf = xfB
            float hx = B(BF_HX, b), hy = B(BF_HY, b);
            V2 lv[4] = { mk(-hx, -hy), mk(hx, -hy), mk(hx, hy), mk(-hx, hy) };
            V2 lnrm[4] = { mk(0.0f, -1.0f), mk(1.0f, 0.0f), mk(0.0f, 1.0f), mk(-1.0f, 0.0f) };
            V2 centroidB = xmul(p, q, mk(0.0f, 0.0f));
            V2 edge1 = v2 - v1;
            normalize(edge1);
            V2 normal1 = mk(edge1.y, -edge1.x);
            float offset1 = dot(normal1, centroidB - v1);
            bool front = offset1 >= 0.0f;
            V2 normal = front ? normal1 : -normal1;
            V2 pv[4], pn[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { pv[i] = xmul(p, q, lv[i]); pn[i] = rmul(q, lnrm[i]); }
            const float radius = 2.0f * RB_POLY_RADIUS;
            float edgeSep = RB_MAXF;
#pragma unroll
            for (int i = 0; i < 4; ++i) { float s = dot(normal, pv[i] - v1); if (s < edgeSep) edgeSep = s; }
            bool hit = !(edgeSep > radius);
            int polyIndex = -1; float polySep = -RB_MAXF; bool polyKnown = false;
            if (hit) {
                for (int i = 0; i < 4; ++i) {
                    V2 n = -pn[i];
                    float s1 = dot(n, pv[i] - v1), s2 = dot(n, pv[i] - v2);
                    float s = min2(s1, s2);
                    if (s > radius) { polyKnown = true; polyIndex = i; polySep = s; break; }
                    // the adjacency test of b2EPCollider can never reject without ghost vertices:
                    // dot(n - (-normal), normal) = dot(n, normal) + 1 >= 0 > -angularSlop
                    if (s > polySep) { polyKnown = true; polyIndex = i; polySep = s; }
                }
                if (polyKnown && polySep > radius) hit = false;
            }
            if (hit) {
                bool primaryPoly = polyKnown && (polySep > 0.98f * edgeSep + 0.001f);
                Clip ie[2];
                int rf_i1, rf_i2; V2 rf_v1, rf_v2, rf_n;
                if (!primaryPoly) {
                    type = MT_FACE_A;
                    int best = 0; float bestValue = dot(normal, pn[0]);
                    for (int i = 1; i < 4; ++i) { float value = dot(normal, pn[i]); if (value < bestValue) { bestValue = value; best = i; } }
                    int i1 = best, i2 = i1 + 1 < 4 ? i1 + 1 : 0;
                    ie[0].v = pv[i1]; ie[0].id = mkid(0, i1, 1, 0);
                    ie[1].v = pv[i2]; ie[1].id = mkid(0, i2, 1, 0);
                    if (front) { rf_i1 = 0; rf_i2 = 1; rf_v1 = v1; rf_v2 = v2; rf_n = normal1; }
                    else { rf_i1 = 1; rf_i2 = 0; rf_v1 = v2; rf_v2 = v1; rf_n = -normal1; }
                } else {
                    type = MT_FACE_B;
                    ie[0].v = v1; ie[0].id = mkid(0, polyIndex, 0, 1);
                    ie[1].v = v2; ie[1].id = mkid(0, polyIndex, 0, 1);
                    rf_i1 = polyIndex; rf_i2 = rf_i1 + 1 < 4 ? rf_i1 + 1 : 0;
                    rf_v1 = pv[rf_i1]; rf_v2 = pv[rf_i2]; rf_n = pn[rf_i1];
                }
                V2 side1 = mk(rf_n.y, -rf_n.x), side2 = -side1;
                float so1 = dot(side1, rf_v1), so2 = dot(side2, rf_v2);
                Clip cp1[2], cp2[2];
                int np = clip_segment(cp1, ie, side1, so1, rf_i1);
                if (np >= 2) np = clip_segment(cp2, cp1, side2, so2, rf_i2);
                if (np >= 2) {
                    if (!primaryPoly) { ln = rf_n; lp = rf_v1; }
                    else { ln = lnrm[rf_i1]; lp = lv[rf_i1]; }
                    for (int i = 0; i < 2; ++i) {
                        float separation = dot(rf_n, cp2[i].v - rf_v1);
                        if (separation <= radius) {
                            if (!primaryPoly) { pt[count] = xmulT(p, q, cp2[i].v); pid[count] = cp2[i].id; }
                            else {
                                pt[count] = cp2[i].v;
                                int id = cp2[i].id;
                                pid[count] = mkid((id >> 8) & 0xff, id & 0xff, (id >> 24) & 0xff, (id >> 16) & 0xff);
                            }
                            ++count;
                        }
                    }
                }
            }
        }
        // impulse matching by feature id
        float n0 = 0.0f, t0 = 0.0f, n1 = 0.0f, t1 = 0.0f;
        if (count > 0) {
            if (oldCount > 0 && oldId0 == pid[0]) { n0 = oldN0; t0 = oldT0; }
            else if (oldCount > 1 && oldId1 == pid[0]) { n0 = oldN1; t0 = oldT1; }
        }
        if (count > 1) {
            if (oldCount > 0 && oldId0 == pid[1]) { n1 = oldN0; t1 = oldT0; }
            else if (oldCount > 1 && oldId1 == pid[1]) { n1 = oldN1; t1 = oldT1; }
        }
        bool touching = count > 0;
        if (touching != wasTouching) set_awake(b, true);
        flags &= ~(CK_TOUCHING | (3 << CK_TYPE_SHIFT) | (3 << CK_COUNT_SHIFT));
        if (touching) flags |= CK_TOUCHING;
        flags |= (type << CK_TYPE_SHIFT) | (count << CK_COUNT_SHIFT);
        setCi(CF_KEY, c, (key & 0xff00ffff) | (flags << 16));
        if (count > 0) {
            C(CF_LNX, c) = ln.x; C(CF_LNY, c) = ln.y; C(CF_LPX, c) = lp.x; C(CF_LPY, c) = lp.y;
            C(CF_P0X, c) = pt[0].x; C(CF_P0Y, c) = pt[0].y; C(CF_P0N, c) = n0; C(CF_P0T, c) = t0; setCi(CF_P0ID, c, pid[0]);
        }
        if (count > 1) {
            C(CF_P1X, c) = pt[1].x; C(CF_P1Y, c) = pt[1].y; C(CF_P1N, c) = n1; C(CF_P1T, c) = t1; setCi(CF_P1ID, c, pid[1]);
        }
    }

    // b2ContactManager::Collide, newest contact first. Group-cooperative: the narrow phase of the pool contacts is strided over
    // the lanes (descending, so that G == 1 keeps Box2D's order exactly); contacts whose fat AABBs stopped overlapping are only
    // MARKED and then removed by the leader, newest first. This is the sequential result: a contact is looked at only if its
    // body is awake, and neither b2Contact::Update nor the destruction can change the awake flag of an awake body, so no
    // contact's treatment depends on what happened to another contact of the same pass.
    __device__ void collide() {
        const int nc = bcast(Si(S_NC));
        bool marked = false;
        for (int i = nc - 1 - sub; i >= 0; i -= G) {
            int key = Ci(CF_KEY, i);
            int b = key_body(key);
            if (!(Bi(BF_FLAGS, b) & BFL_AWAKE)) continue;
            if (!overlap_edge(key_edge(key), b)) { setCi(CF_KEY, i, key | CK_DESTROY_MARK); marked = true; continue; }
            contact_update(i);
        }
        if (group_any(marked)) {
            gsync();                      // (a vote synchronises the lanes but is not a memory barrier)
            if (leader())
                for (int i = nc - 1; i >= 0; --i)
                    if (Ci(CF_KEY, i) & CK_DESTROY_MARK) destroy_contact(i);
        }
        gsync();
    }

    // ---- contact constraints in shared memory
    // Build the velocity constraint of pool contact c in hot slot t from the CURRENT solver pose of its body
    // (b2ContactSolver ctor + InitializeVelocityConstraints). cB/aB are passed in.
    __device__ __forceinline__ void contact_init_velocity(float* hc, const int st, int c, V2 cB, float aB, float mB, float iB, float dtRatio, bool warm) {
        int key = Ci(CF_KEY, c);
        int b = key_body(key);
        int flags = key_flags(key);
        int type = (flags >> CK_TYPE_SHIFT) & 3, count = (flags >> CK_COUNT_SHIFT) & 3;
        float radiusB = (Bi(BF_FLAGS, b) & BFL_CIRCLE) ? B(BF_HX, b) : RB_POLY_RADIUS;
        const float radiusA = RB_POLY_RADIUS;
        Rot qB = rot_set(aB);
        V2 pB = cB;                                  // xfB.p = cB - R(aB) * 0
        V2 ln = mk(C(CF_LNX, c), C(CF_LNY, c)), lp = mk(C(CF_LPX, c), C(CF_LPY, c));
        V2 l0 = mk(C(CF_P0X, c), C(CF_P0Y, c)), l1 = mk(C(CF_P1X, c), C(CF_P1Y, c));
        V2 normal, wp0, wp1 = mk(0.0f, 0.0f);
        if (type == MT_CIRCLES) {
            normal = mk(1.0f, 0.0f);
            V2 pointA = lp, pointB = xmul(pB, qB, l0);
            V2 d = pointA - pointB;
            if (dot(d, d) > RB_EPS * RB_EPS) { normal = pointB - pointA; normalize(normal); }
            V2 cA = pointA + radiusA * normal, cBp = pointB - radiusB * normal;
            wp0 = 0.5f * (cA + cBp);
        } else if (type == MT_FACE_A) {
            normal = ln;
            V2 planePoint = lp;
            V2 clip = xmul(pB, qB, l0);
            V2 cA = clip + (radiusA - dot(clip - planePoint, normal)) * normal, cBp = clip - radiusB * normal;
            wp0 = 0.5f * (cA + cBp);
            if (count > 1) {
                clip = xmul(pB, qB, l1);
                cA = clip + (radiusA - dot(clip - planePoint, normal)) * normal; cBp = clip - radiusB * normal;
                wp1 = 0.5f * (cA + cBp);
            }
        } else {
            V2 nrm = rmul(qB, ln);
            V2 planePoint = xmul(pB, qB, lp);
            V2 clip = l0;
            V2 cBp = clip + (radiusB - dot(clip - planePoint, nrm)) * nrm, cA = clip - radiusA * nrm;
            wp0 = 0.5f * (cA + cBp);
            if (count > 1) {
                clip = l1;
                cBp = clip + (radiusB - dot(clip - planePoint, nrm)) * nrm; cA = clip - radiusA * nrm;
                wp1 = 0.5f * (cA + cBp);
            }
            normal = -nrm;
        }
        V2 tangent = cross_vs(normal, 1.0f);
        V2 r0 = wp0 - cB, r1 = wp1 - cB;
        float rn0 = cross(r0, normal), rt0 = cross(r0, tangent);
        float kN0 = mB + iB * rn0 * rn0, kT0 = mB + iB * rt0 * rt0;
        hc[HC_NX * st] = normal.x; hc[HC_NY * st] = normal.y;
        hc[HC_R0X * st] = r0.x; hc[HC_R0Y * st] = r0.y;
        hc[HC_NM0 * st] = kN0 > 0.0f ? 1.0f / kN0 : 0.0f;
        hc[HC_TM0 * st] = kT0 > 0.0f ? 1.0f / kT0 : 0.0f;
        hc[HC_NI0 * st] = warm ? dtRatio * C(CF_P0N, c) : 0.0f;
        hc[HC_TI0 * st] = warm ? dtRatio * C(CF_P0T, c) : 0.0f;
        int vcount = count;
        if (count > 1) {
            float rn1 = cross(r1, normal), rt1 = cross(r1, tangent);
            float kN1 = mB + iB * rn1 * rn1, kT1 = mB + iB * rt1 * rt1;
            hc[HC_R1X * st] = r1.x; hc[HC_R1Y * st] = r1.y;
            hc[HC_NM1 * st] = kN1 > 0.0f ? 1.0f / kN1 : 0.0f;
            hc[HC_TM1 * st] = kT1 > 0.0f ? 1.0f / kT1 : 0.0f;
            hc[HC_NI1 * st] = warm ? dtRatio * C(CF_P1N, c) : 0.0f;
            hc[HC_TI1 * st] = warm ? dtRatio * C(CF_P1T, c) : 0.0f;
            float k11 = mB + iB * rn0 * rn0, k22 = mB + iB * rn1 * rn1, k12 = mB + iB * rn0 * rn1;
            if (k11 * k11 < 1000.0f * (k11 * k22 - k12 * k12)) {
                hc[HC_K11 * st] = k11; hc[HC_K12 * st] = k12; hc[HC_K22 * st] = k22;
                float det = k11 * k22 - k12 * k12;
                if (det != 0.0f) det = 1.0f / det;
                hc[HC_IXX * st] = det * k22; hc[HC_IXY * st] = -det * k12; hc[HC_IYY * st] = det * k11;
            } else vcount = 1;
        }
        hc[HC_META * st] = __int_as_float(b | (vcount << 8) | (c << 16));
    }

    // one sequential-impulse pass over hot contact slot t (b2ContactSolver::SolveVelocityConstraints)
    __device__ __forceinline__ void contact_solve_velocity(float* hc, const int st) {
        int meta = __float_as_int(hc[HC_META * st]);
        int b = meta & 0xff, count = (meta >> 8) & 3;
        float mB = HB(HB_INVM, b), iB = HB(HB_INVI, b);
        V2 vB = mk(HB(HB_VX, b), HB(HB_VY, b)); float wB = HB(HB_W, b);
        V2 normal = mk(hc[HC_NX * st], hc[HC_NY * st]), tangent = cross_vs(normal, 1.0f);
        const float friction = k->friction;
        V2 r0 = mk(hc[HC_R0X * st], hc[HC_R0Y * st]);
        {   // friction, point 0
            V2 dv = vB + cross_sv(wB, r0);
            float vt = dot(dv, tangent);
            float lambda = hc[HC_TM0 * st] * (-vt);
            float ti = hc[HC_TI0 * st];
            float maxF = friction * hc[HC_NI0 * st];
            float ni = clampf(ti + lambda, -maxF, maxF);
            lambda = ni - ti; hc[HC_TI0 * st] = ni;
            V2 P = lambda * tangent;
            vB = vB + mB * P; wB += iB * cross(r0, P);
        }
        if (count == 1) {
            V2 dv = vB + cross_sv(wB, r0);
            float vn = dot(dv, normal);
            float lambda = -hc[HC_NM0 * st] * vn;
            float ni0 = hc[HC_NI0 * st];
            float ni = max2(ni0 + lambda, 0.0f);
            lambda = ni - ni0; hc[HC_NI0 * st] = ni;
            V2 P = lambda * normal;
            vB = vB + mB * P; wB += iB * cross(r0, P);
        } else {
            V2 r1 = mk(hc[HC_R1X * st], hc[HC_R1Y * st]);
            {   // friction, point 1
                V2 dv = vB + cross_sv(wB, r1);
                float vt = dot(dv, tangent);
                float lambda = hc[HC_TM1 * st] * (-vt);
                float ti = hc[HC_TI1 * st];
                float maxF = friction * hc[HC_NI1 * st];
                float ni = clampf(ti + lambda, -maxF, maxF);
                lambda = ni - ti; hc[HC_TI1 * st] = ni;
                V2 P = lambda * tangent;
                vB = vB + mB * P; wB += iB * cross(r1, P);
            }
            float a1 = hc[HC_NI0 * st], a2 = hc[HC_NI1 * st];
            V2 dv1 = vB + cross_sv(wB, r0), dv2 = vB + cross_sv(wB, r1);
            float vn1 = dot(dv1, normal), vn2 = dot(dv2, normal);
            float k11 = hc[HC_K11 * st], k12 = hc[HC_K12 * st], k22 = hc[HC_K22 * st];
            float bx = vn1 - (k11 * a1 + k12 * a2), by = vn2 - (k12 * a1 + k22 * a2);
            float x1, x2; bool solved = false;
            x1 = -(hc[HC_IXX * st] * bx + hc[HC_IXY * st] * by); x2 = -(hc[HC_IXY * st] * bx + hc[HC_IYY * st] * by);
            if (x1 >= 0.0f && x2 >= 0.0f) solved = true;
            if (!solved) { x1 = -hc[HC_NM0 * st] * bx; x2 = 0.0f; vn2 = k12 * x1 + by; if (x1 >= 0.0f && vn2 >= 0.0f) solved = true; }
            if (!solved) { x1 = 0.0f; x2 = -hc[HC_NM1 * st] * by; vn1 = k12 * x2 + bx; if (x2 >= 0.0f && vn1 >= 0.0f) solved = true; }
            if (!solved) { x1 = 0.0f; x2 = 0.0f; if (bx >= 0.0f && by >= 0.0f) solved = true; }
            if (solved) {
                float d1 = x1 - a1, d2 = x2 - a2;
                V2 P1 = d1 * normal, P2 = d2 * normal;
                vB = vB + mB * (P1 + P2);
                wB += iB * (cross(r0, P1) + cross(r1, P2));
                hc[HC_NI0 * st] = x1; hc[HC_NI1 * st] = x2;
            }
        }
        HB(HB_VX, b) = vB.x; HB(HB_VY, b) = vB.y; HB(HB_W, b) = wB;
    }

    // The same solve in three pieces - loads, arithmetic, stores - for the FUSED slots of the scheduled sweeps (solve_velocity):
    // a slot in which lanes of the warp hold a revolute joint and other lanes a contact runs both kinds as ONE straight-line
    // sequence (all loads, both computations, then the stores), so the two dependency chains overlap instead of being
    // serialised by a divergent branch. Friction of point 0 and the normal solve of a one-point manifold are straight-line;
    // a two-point manifold continues from the post-friction velocity in contact_v_two. Every path performs exactly the
    // operations of contact_solve_velocity.
    struct CV { int b, count; float mB, iB, wB, tm0, ti0, ni0, nm0, o_ti0, o_ni0, wF, w1; V2 vB, normal, tangent, r0, vF, v1; };
    // (`on` = false: an idle lane of a fused slot - it computes on zeros and neither loads nor stores)
    #define LDP(x) (on ? (x) : 0.0f)
    __device__ __forceinline__ void contact_v_load(const float* hc, const int st, const int meta, CV& c, const bool on = true) {
        c.b = meta & 0xff; c.count = (meta >> 8) & 3;
        c.mB = LDP(HB(HB_INVM, c.b)); c.iB = LDP(HB(HB_INVI, c.b));
        c.vB = mk(LDP(HB(HB_VX, c.b)), LDP(HB(HB_VY, c.b))); c.wB = LDP(HB(HB_W, c.b));
        c.normal = mk(LDP(hc[HC_NX * st]), LDP(hc[HC_NY * st])); c.tangent = cross_vs(c.normal, 1.0f);
        c.r0 = mk(LDP(hc[HC_R0X * st]), LDP(hc[HC_R0Y * st]));
        c.tm0 = LDP(hc[HC_TM0 * st]); c.ti0 = LDP(hc[HC_TI0 * st]); c.ni0 = LDP(hc[HC_NI0 * st]); c.nm0 = LDP(hc[HC_NM0 * st]);
    }
    __device__ __forceinline__ void contact_v_compute(CV& c) {
        const float friction = k->friction;
        V2 vB = c.vB; float wB = c.wB;
        {   // friction, point 0
            V2 dv = vB + cross_sv(wB, c.r0);
            float vt = dot(dv, c.tangent);
            float lambda = c.tm0 * (-vt);
            float maxF = friction * c.ni0;
            float ni = clampf(c.ti0 + lambda, -maxF, maxF);
            lambda = ni - c.ti0; c.o_ti0 = ni;
            V2 P = lambda * c.tangent;
            vB = vB + c.mB * P; wB += c.iB * cross(c.r0, P);
        }
        c.vF = vB; c.wF = wB;
        {   // one-point manifold: normal constraint
            V2 dv = vB + cross_sv(wB, c.r0);
            float vn = dot(dv, c.normal);
            float lambda = -c.nm0 * vn;
            float ni = max2(c.ni0 + lambda, 0.0f);
            lambda = ni - c.ni0; c.o_ni0 = ni;
            V2 P = lambda * c.normal;
            c.v1 = vB + c.mB * P; c.w1 = wB + c.iB * cross(c.r0, P);
        }
    }
    __device__ __forceinline__ void contact_v_store1(float* hc, const int st, const CV& c) {
        hc[HC_TI0 * st] = c.o_ti0;
        if (c.count == 1) {
            hc[HC_NI0 * st] = c.o_ni0;
            HB(HB_VX, c.b) = c.v1.x; HB(HB_VY, c.b) = c.v1.y; HB(HB_W, c.b) = c.w1;
        }
    }
    __device__ __forceinline__ void contact_v_two(float* hc, const int st, const CV& c) {
        V2 vB = c.vF; float wB = c.wF;
        const V2 normal = c.normal, tangent = c.tangent, r0 = c.r0;
        const float mB = c.mB, iB = c.iB, friction = k->friction;
        V2 r1 = mk(hc[HC_R1X * st], hc[HC_R1Y * st]);
        {   // friction, point 1
            V2 dv = vB + cross_sv(wB, r1);
            float vt = dot(dv, tangent);
            float lambda = hc[HC_TM1 * st] * (-vt);
            float ti = hc[HC_TI1 * st];
            float maxF = friction * hc[HC_NI1 * st];
            float ni = clampf(ti + lambda, -maxF, maxF);
            lambda = ni - ti; hc[HC_TI1 * st] = ni;
            V2 P = lambda * tangent;
            vB = vB + mB * P; wB += iB * cross(r1, P);
        }
        float a1 = c.ni0, a2 = hc[HC_NI1 * st];
        V2 dv1 = vB + cross_sv(wB, r0), dv2 = vB + cross_sv(wB, r1);
        float vn1 = dot(dv1, normal), vn2 = dot(dv2, normal);
        float k11 = hc[HC_K11 * st], k12 = hc[HC_K12 * st], k22 = hc[HC_K22 * st];
        float bx = vn1 - (k11 * a1 + k12 * a2), by = vn2 - (k12 * a1 + k22 * a2);
        float x1, x2; bool solved = false;
        x1 = -(hc[HC_IXX * st] * bx + hc[HC_IXY * st] * by); x2 = -(hc[HC_IXY * st] * bx + hc[HC_IYY * st] * by);
        if (x1 >= 0.0f && x2 >= 0.0f) solved = true;
        if (!solved) { x1 = -c.nm0 * bx; x2 = 0.0f; vn2 = k12 * x1 + by; if (x1 >= 0.0f && vn2 >= 0.0f) solved = true; }
        if (!solved) { x1 = 0.0f; x2 = -hc[HC_NM1 * st] * by; vn1 = k12 * x2 + bx; if (x2 >= 0.0f && vn1 >= 0.0f) solved = true; }
        if (!solved) { x1 = 0.0f; x2 = 0.0f; if (bx >= 0.0f && by >= 0.0f) solved = true; }
        if (solved) {
            float d1 = x1 - a1, d2 = x2 - a2;
            V2 P1 = d1 * normal, P2 = d2 * normal;
            vB = vB + mB * (P1 + P2);
            wB += iB * (cross(r0, P1) + cross(r1, P2));
            hc[HC_NI0 * st] = x1; hc[HC_NI1 * st] = x2;
        }
        HB(HB_VX, c.b) = vB.x; HB(HB_VY, c.b) = vB.y; HB(HB_W, c.b) = wB;
    }

    __device__ __forceinline__ void count_contact_solves(int nt, int vit) {
        int n1 = 0, n2 = 0;
        for_contacts(nt, [&](float* hc, const int st, int) { if (((__float_as_int(hc[HC_META * st]) >> 8) & 3) == 1) ++n1; else ++n2; });
        cnt.c[REM2D_CNT_P1_VSOLVES] += (unsigned)(n1 * vit);
        cnt.c[REM2D_CNT_M2_VSOLVES] += (unsigned)(n2 * vit);
    }
    // position manifold of point j of hot (position overlay) slot t; returns separation
    __device__ __forceinline__ float psm(const float* hc, const int st, int type, int j, V2 cB, float aB, V2& normal, V2& point) {
        Rot qB = rot_set(aB);
        V2 lp = mk(hc[PC_LPX * st], hc[PC_LPY * st]);
        V2 lpt = j == 0 ? mk(hc[PC_P0X * st], hc[PC_P0Y * st]) : mk(hc[PC_P1X * st], hc[PC_P1Y * st]);
        const float radiusA = RB_POLY_RADIUS;
        float radiusB = hc[PC_RADB * st];
        if (type == MT_CIRCLES) {
            V2 pointA = lp, pointB = xmul(cB, qB, mk(hc[PC_P0X * st], hc[PC_P0Y * st]));
            normal = pointB - pointA;
            normalize(normal);
            point = 0.5f * (pointA + pointB);
            return dot(pointB - pointA, normal) - radiusA - radiusB;
        } else if (type == MT_FACE_A) {
            normal = mk(hc[PC_LNX * st], hc[PC_LNY * st]);
            V2 clip = xmul(cB, qB, lpt);
            point = clip;
            return dot(clip - lp, normal) - radiusA - radiusB;
        } else {
            V2 nrm = rmul(qB, mk(hc[PC_LNX * st], hc[PC_LNY * st]));
            V2 planePoint = xmul(cB, qB, lp);
            V2 clip = lpt;
            float sep = dot(clip - planePoint, nrm) - radiusA - radiusB;
            point = clip;
            normal = -nrm;
            return sep;
        }
    }
    // one pass of Solve(TOI)PositionConstraints over hot slot t; returns the min separation seen
    template <bool COUNT = true>
    __device__ __forceinline__ float contact_solve_position(float* hc, const int st, float baumgarte, float minSeparation) {
        int meta = __float_as_int(hc[PC_META * st]);
        int b = meta & 0xff, count = (meta >> 8) & 3, type = (meta >> 10) & 3;
        float mB = HB(HB_INVM, b), iB = HB(HB_INVI, b);
        V2 cB = mk(HB(HB_VX, b), HB(HB_VY, b)); float aB = HB(HB_W, b);     // position overlay: c, a
        for (int j = 0; j < count; ++j) {
            if (COUNT) cnt.c[REM2D_CNT_POINT_PSOLVES]++;
            V2 normal, point;
            float separation = psm(hc, st, type, j, cB, aB, normal, point);
            V2 rB = point - cB;
            minSeparation = min2(minSeparation, separation);
            float Cc = clampf(baumgarte * (separation + RB_LINEAR_SLOP), -RB_MAX_LIN_CORR, 0.0f);
            float rnB = cross(rB, normal);
            float K = mB + iB * rnB * rnB;
            float impulse = K > 0.0f ? -Cc / K : 0.0f;
            V2 P = impulse * normal;
            cB = cB + mB * P; aB += iB * cross(rB, P);
        }
        HB(HB_VX, b) = cB.x; HB(HB_VY, b) = cB.y; HB(HB_W, b) = aB;
        return minSeparation;
    }
    // copy the position-constraint data of pool contact c into hot slot t
    __device__ __forceinline__ void contact_init_position(float* hc, const int st, int c) {
        int key = Ci(CF_KEY, c);
        int b = key_body(key), flags = key_flags(key);
        int type = (flags >> CK_TYPE_SHIFT) & 3, count = (flags >> CK_COUNT_SHIFT) & 3;
        hc[PC_META * st] = __int_as_float(b | (count << 8) | (type << 10));
        hc[PC_LNX * st] = C(CF_LNX, c); hc[PC_LNY * st] = C(CF_LNY, c);
        hc[PC_LPX * st] = C(CF_LPX, c); hc[PC_LPY * st] = C(CF_LPY, c);
        hc[PC_P0X * st] = C(CF_P0X, c); hc[PC_P0Y * st] = C(CF_P0Y, c);
        hc[PC_P1X * st] = C(CF_P1X, c); hc[PC_P1Y * st] = C(CF_P1Y, c);
        hc[PC_RADB * st] = (Bi(BF_FLAGS, b) & BFL_CIRCLE) ? B(BF_HX, b) : RB_POLY_RADIUS;
    }

    // ---- revolute joints in shared memory (b2RevoluteJoint)
    // One b2RevoluteJoint::SolveVelocityConstraints. Lanes of a warp disagree on the limit state of their s-th joint,
    // so a branchy version executes the 2x2 (limit inactive) and the 3x3 (at a limit) paths one after the other.
    // Here both candidates are computed unconditionally from the same inputs and the results are selected: the two
    // dependency chains overlap, there is no reconvergence overhead, and every value is bit-identical to the branchy
    // evaluation (each candidate uses exactly the operations of its Box2D path).
    // Loads / arithmetic / stores of the solve as separate pieces (see CV above for why).
    struct JV { int a, b, limit; bool act; float mA, iA, mB, iB, wA, wB, exx, eyx, eyy, d2, det, jx, jy, jz, mspeed, mmass, mimp, maximp;
                float o_mimp, o_jx, o_jy, o_jz, o_wA, o_wB; V2 vA, vB, rA, rB, o_vA, o_vB; };
    __device__ __forceinline__ void joint_v_load(int s, const int meta, JV& r, const bool on = true) {
        r.a = meta & 0xff; r.b = (meta >> 8) & 0xff; r.limit = (meta >> 16) & 3;
        r.mA = LDP(HB(HB_INVM, r.a)); r.iA = LDP(HB(HB_INVI, r.a)); r.mB = LDP(HB(HB_INVM, r.b)); r.iB = LDP(HB(HB_INVI, r.b));
        r.vA = mk(LDP(HB(HB_VX, r.a)), LDP(HB(HB_VY, r.a))); r.wA = LDP(HB(HB_W, r.a));
        r.vB = mk(LDP(HB(HB_VX, r.b)), LDP(HB(HB_VY, r.b))); r.wB = LDP(HB(HB_W, r.b));
        r.rA = mk(LDP(HJ(HJ_RAX, s)), LDP(HJ(HJ_RAY, s))); r.rB = mk(LDP(HJ(HJ_RBX, s)), LDP(HJ(HJ_RBY, s)));
        r.exx = LDP(HJ(HJ_EXX, s)); r.eyx = LDP(HJ(HJ_EYX, s)); r.eyy = LDP(HJ(HJ_EYY, s));
        r.d2 = LDP(HJ(HJ_INV2, s)); r.det = LDP(HJ(HJ_INV3, s));
        r.jx = LDP(HJ(HJ_IMPX, s)); r.jy = LDP(HJ(HJ_IMPY, s)); r.jz = LDP(HJ(HJ_IMPZ, s));
        r.mspeed = LDP(HJ(HJ_MSPEED, s)); r.mmass = LDP(HJ(HJ_MMASS, s)); r.mimp = LDP(HJ(HJ_MIMP, s)); r.maximp = LDP(HJ(HJ_MAXIMP, s));
    }
    __device__ __forceinline__ void joint_v_compute(JV& r) {
        const float mA = r.mA, iA = r.iA, mB = r.mB, iB = r.iB, exx = r.exx, eyx = r.eyx, eyy = r.eyy, d2 = r.d2, det = r.det;
        const float jx = r.jx, jy = r.jy, jz = r.jz;
        const V2 vA = r.vA, vB = r.vB, rA = r.rA, rB = r.rB;
        float wA = r.wA, wB = r.wB;
        const int limit = r.limit;
        {   // motor
            float Cdot = wB - wA - r.mspeed;
            float impulse = -r.mmass * Cdot;
            float oldImpulse = r.mimp;
            float maxImpulse = r.maximp;
            float ni = clampf(oldImpulse + impulse, -maxImpulse, maxImpulse);
            r.o_mimp = ni;
            impulse = ni - oldImpulse;
            wA -= iA * impulse; wB += iB * impulse;
        }
        // relative velocity of the anchor points: the same expression in both Box2D paths
        const V2 Cdot1 = vB + cross_sv(wB, rB) - vA - cross_sv(wA, rA);
        // ---- candidate 1: point-to-point constraint only (limit inactive), Solve22(-Cdot)
        const V2 nb_ = -Cdot1;
        const V2 imp2 = mk(d2 * (eyy * nb_.x - eyx * nb_.y), d2 * (exx * nb_.y - eyx * nb_.x));
        const V2 vA2 = vA - mA * imp2; const float wA2 = wA - iA * cross(rA, imp2);
        const V2 vB2 = vB + mB * imp2; const float wB2 = wB + iB * cross(rB, imp2);
        // ---- candidate 2: point + angular limit, Solve33 and, if the limit impulse changes sign, the reduced Solve22
        const float ezx = -rA.y * iA - rB.y * iB, ezy = rA.x * iA + rB.x * iB, ezz = iA + iB;
        const float Cdot2 = wB - wA;
        const float cx = eyy * ezz - ezy * ezy, cy = ezy * ezx - eyx * ezz, cz = eyx * ezy - eyy * ezx;   // ey x ez
        float ix = det * (Cdot1.x * cx + Cdot1.y * cy + Cdot2 * cz);
        const float bx = Cdot1.y * ezz - Cdot2 * ezy, by = Cdot2 * ezx - Cdot1.x * ezz, bz = Cdot1.x * ezy - Cdot1.y * ezx;   // b x ez
        float iy = det * (exx * bx + eyx * by + ezx * bz);
        const float ex2 = eyy * Cdot2 - ezy * Cdot1.y, ey2 = ezy * Cdot1.x - eyx * Cdot2, ez2 = eyx * Cdot1.y - eyy * Cdot1.x;   // ey x b
        float iz = det * (exx * ex2 + eyx * ey2 + ezx * ez2);
        ix = -ix; iy = -iy; iz = -iz;
        const float newImpulse = jz + iz;
        const bool reduce = (limit == 1) ? (newImpulse < 0.0f) : (newImpulse > 0.0f);
        const V2 rhs = -Cdot1 + jz * mk(ezx, ezy);
        const float rx = d2 * (eyy * rhs.x - eyx * rhs.y), ry = d2 * (exx * rhs.y - eyx * rhs.x);
        const float px = reduce ? rx : ix, py = reduce ? ry : iy, pz = reduce ? -jz : iz;
        const V2 P = mk(px, py);
        const V2 vA3 = vA - mA * P; const float wA3 = wA - iA * (cross(rA, P) + pz);
        const V2 vB3 = vB + mB * P; const float wB3 = wB + iB * (cross(rB, P) + pz);
        const float jz3 = reduce ? 0.0f : jz + iz;
        // ---- select
        const bool act = limit != 0;
        r.act = act;
        r.o_jx = jx + (act ? px : imp2.x);
        r.o_jy = jy + (act ? py : imp2.y);
        r.o_jz = jz3;
        r.o_vA = mk(act ? vA3.x : vA2.x, act ? vA3.y : vA2.y); r.o_wA = act ? wA3 : wA2;
        r.o_vB = mk(act ? vB3.x : vB2.x, act ? vB3.y : vB2.y); r.o_wB = act ? wB3 : wB2;
    }
    __device__ __forceinline__ void joint_v_store(int s, const JV& r) {
        HJ(HJ_MIMP, s) = r.o_mimp;
        HJ(HJ_IMPX, s) = r.o_jx;
        HJ(HJ_IMPY, s) = r.o_jy;
        if (r.act) HJ(HJ_IMPZ, s) = r.o_jz;
        HB(HB_VX, r.a) = r.o_vA.x; HB(HB_VY, r.a) = r.o_vA.y; HB(HB_W, r.a) = r.o_wA;
        HB(HB_VX, r.b) = r.o_vB.x; HB(HB_VY, r.b) = r.o_vB.y; HB(HB_W, r.b) = r.o_wB;
    }
    __device__ __forceinline__ void joint_solve_velocity(int s) { joint_solve_velocity(s, HJi(HJ_META, s)); }
    __device__ __forceinline__ void joint_solve_velocity(int s, const int meta) {
        JV r;
        joint_v_load(s, meta, r);
        joint_v_compute(r);
        joint_v_store(s, r);
    }
    __device__ __forceinline__ bool joint_solve_position(int s) {
        int meta = HJi(PJ_META, s);
        int a = meta & 0xff, b = (meta >> 8) & 0xff, limit = (meta >> 16) & 3;
        float mA = HB(HB_INVM, a), iA = HB(HB_INVI, a), mB = HB(HB_INVM, b), iB = HB(HB_INVI, b);
        V2 cA = mk(HB(HB_VX, a), HB(HB_VY, a)); float aA = HB(HB_W, a);
        V2 cB = mk(HB(HB_VX, b), HB(HB_VY, b)); float aB = HB(HB_W, b);
        float angularError = 0.0f, positionError = 0.0f;
        {   // angular limit, evaluated for every lane and selected (lanes disagree on the limit state)
            const float motorMass = HJ(HJ_MMASS, s);      // 1 / (iA + iB): this slot survives the position overlay
            const float angle = aB - aA - 0.0f;
            const float Cl = angle - HJ(PJ_LOWER, s), Cu = angle - HJ(PJ_UPPER, s);
            const float Ccl = clampf(Cl + RB_ANGULAR_SLOP, -RB_MAX_ANG_CORR, 0.0f);
            const float Ccu = clampf(Cu - RB_ANGULAR_SLOP, 0.0f, RB_MAX_ANG_CORR);
            const float limitImpulse = -motorMass * (limit == 1 ? Ccl : Ccu);
            const float aA1 = aA - iA * limitImpulse, aB1 = aB + iB * limitImpulse;
            const bool act = limit != 0;
            angularError = act ? (limit == 1 ? -Cl : Cu) : 0.0f;
            aA = act ? aA1 : aA; aB = act ? aB1 : aB;
        }
        Rot qA = rot_set(aA), qB = rot_set(aB);
        V2 rA = rmul(qA, mk(HJ(PJ_LAAX, s), HJ(PJ_LAAY, s)) - mk(0.0f, 0.0f));
        V2 rB = rmul(qB, mk(HJ(PJ_LABX, s), HJ(PJ_LABY, s)) - mk(0.0f, 0.0f));
        V2 Cv = cB + rB - cA - rA;
        positionError = len(Cv);
        float kexx = mA + mB + iA * rA.y * rA.y + iB * rB.y * rB.y;
        float kexy = -iA * rA.x * rA.y - iB * rB.x * rB.y;
        float keyy = mA + mB + iA * rA.x * rA.x + iB * rB.x * rB.x;
        float det = kexx * keyy - kexy * kexy;
        if (det != 0.0f) det = 1.0f / det;
        V2 imp = -mk(det * (keyy * Cv.x - kexy * Cv.y), det * (kexx * Cv.y - kexy * Cv.x));
        cA = cA - mA * imp; aA -= iA * cross(rA, imp);
        cB = cB + mB * imp; aB += iB * cross(rB, imp);
        HB(HB_VX, a) = cA.x; HB(HB_VY, a) = cA.y; HB(HB_W, a) = aA;
        HB(HB_VX, b) = cB.x; HB(HB_VY, b) = cB.y; HB(HB_W, b) = aB;
        return positionError <= RB_LINEAR_SLOP && angularError <= RB_ANGULAR_SLOP;
    }

    // ---- b2World::Solve for the creature's single island (+ SynchronizeFixtures + FindNewContacts)
    // solve_pre: integrate velocities, stage + warm start the constraints, build the schedule; returns false if the island
    // sleeps. solve_velocity: the 180 sequential-impulse iterations. solve_post: store impulses, integrate positions, position
    // iterations, sleeping, SynchronizeFixtures + FindNewContacts. All group-cooperative (every lane of the group calls them).
    __device__ bool solve_pre(float dtRatio, int& nt_out) {
        const float hdt = k->dt;
        nt_out = 0;
        // a creature is one island (tree of joints); it is solved iff its seed body is awake. Jointed
        // creatures are always awake here (the motor-speed setter woke them); a lone body may sleep.
        bool anyAwake = false;
        for (int b = sub; b < nb; b += G) anyAwake |= (Bi(BF_FLAGS, b) & BFL_AWAKE) != 0;
        if (!group_any(anyAwake)) return false;
        for (int b = sub; b < nb; b += G) {
            set_awake(b, true);
            float cx = B(BF_CX, b), cy = B(BF_CY, b), a = B(BF_A, b);
            B(BF_C0X, b) = cx; B(BF_C0Y, b) = cy; B(BF_A0, b) = a;
            V2 v = mk(B(BF_VX, b), B(BF_VY, b)); float w = B(BF_W, b);
            float invM = B(BF_INVM, b), invI = B(BF_INVI, b);
            V2 gravity = mk(0.0f, k->gravity_y), force = mk(0.0f, 0.0f);
            v = v + hdt * (1.0f * gravity + invM * force);
            w += hdt * invI * 0.0f;
            v = (1.0f / (1.0f + hdt * 0.0f)) * v;
            w *= 1.0f / (1.0f + hdt * 0.0f);
            HB(HB_VX, b) = v.x; HB(HB_VY, b) = v.y; HB(HB_W, b) = w;
            HB(HB_INVM, b) = invM; HB(HB_INVI, b) = invI;
            cnt.c[REM2D_CNT_BODY_TICKS]++;
        }
        // contact constraints: touching contacts, newest first (per-body list order is what matters:
        // contacts of different bodies only share the static terrain and commute exactly). The leader lists them (slot t
        // remembers its pool index), the group builds the constraints.
        int nt = 0;
        if (leader()) {
            const int nc = Si(S_NC);
            for (int c = nc - 1; c >= 0; --c) {
                int fl = key_flags(Ci(CF_KEY, c));
                if (!(fl & CK_ENABLED) || !(fl & CK_TOUCHING)) continue;
                with_contact(nt, [&](float* hc, const int st) { hc[HC_META * st] = __int_as_float(c); });
                ++nt;
            }
        }
        nt = bcast(nt);
        gsync();
        for (int t = sub; t < nt; t += G)
            with_contact(t, [&](float* hc, const int st) {
                const int c = __float_as_int(hc[HC_META * st]);
                const int b = key_body(Ci(CF_KEY, c));
                contact_init_velocity(hc, st, c, mk(B(BF_CX, b), B(BF_CY, b)), B(BF_A, b), B(BF_INVM, b), B(BF_INVI, b), dtRatio, true);
            });
        // joints: InitVelocityConstraints in island order (slot s = s-th joint of the island); the warm-start impulses are
        // scaled and stored here and APPLIED below in Box2D's order
        for (int s = sub; s < nj; s += G) {
            int jm = Ji(JF_META, s);
            int j = (jm >> 8) & 0xff;                  // joint index solved s-th
            int a = Ji(JF_META, j) & 0xff, b = j + 1;
            float aA = B(BF_A, a), aB = B(BF_A, b);
            float mA = B(BF_INVM, a), iA = B(BF_INVI, a), mB = B(BF_INVM, b), iB = B(BF_INVI, b);
            Rot qA = rot_set(aA), qB = rot_set(aB);
            V2 rA = rmul(qA, mk(J(JF_LAAX, j), J(JF_LAAY, j)) - mk(0.0f, 0.0f));
            V2 rB = rmul(qB, mk(J(JF_LABX, j), J(JF_LABY, j)) - mk(0.0f, 0.0f));
            float exx = mA + mB + rA.y * rA.y * iA + rB.y * rB.y * iB;
            float eyx = -rA.y * rA.x * iA - rB.y * rB.x * iB;
            float ezx = -rA.y * iA - rB.y * iB;
            float eyy = mA + mB + rA.x * rA.x * iA + rB.x * rB.x * iB;
            float ezy = rA.x * iA + rB.x * iB;
            float ezz = iA + iB;
            float motorMass = iA + iB;
            if (motorMass > 0.0f) motorMass = 1.0f / motorMass;
            float impx = J(JF_IMPX, j), impy = J(JF_IMPY, j), impz = J(JF_IMPZ, j), mimp = J(JF_MIMP, j);
            int limit = Ji(JF_LIMIT, j);
            float jointAngle = aB - aA - 0.0f;
            float lower = J(JF_LOWER, j), upper = J(JF_UPPER, j);
            if (jointAngle <= lower) { if (limit != 1) impz = 0.0f; limit = 1; }
            else if (jointAngle >= upper) { if (limit != 2) impz = 0.0f; limit = 2; }
            else { limit = 0; impz = 0.0f; }
            setJi(JF_LIMIT, j, limit);
            impx *= dtRatio; impy *= dtRatio; impz *= dtRatio; mimp *= dtRatio;
            HJ(HJ_META, s) = __int_as_float(a | (b << 8) | (limit << 16) | (j << 24));
            HJ(HJ_RAX, s) = rA.x; HJ(HJ_RAY, s) = rA.y; HJ(HJ_RBX, s) = rB.x; HJ(HJ_RBY, s) = rB.y;
            HJ(HJ_EXX, s) = exx; HJ(HJ_EYX, s) = eyx; HJ(HJ_EYY, s) = eyy;
            {
                float inv2 = exx * eyy - eyx * eyx;
                if (inv2 != 0.0f) inv2 = 1.0f / inv2;
                float cx = eyy * ezz - ezy * ezy, cy = ezy * ezx - eyx * ezz, cz = eyx * ezy - eyy * ezx;
                float inv3 = exx * cx + eyx * cy + ezx * cz;
                if (inv3 != 0.0f) inv3 = 1.0f / inv3;
                HJ(HJ_INV2, s) = inv2; HJ(HJ_INV3, s) = inv3;
            }
            HJ(HJ_MMASS, s) = motorMass;
            HJ(HJ_IMPX, s) = impx; HJ(HJ_IMPY, s) = impy; HJ(HJ_IMPZ, s) = impz; HJ(HJ_MIMP, s) = mimp;
            HJ(HJ_MSPEED, s) = J(JF_MSPEED, j);
            HJ(HJ_MAXIMP, s) = hdt * J(JF_MAXT, j);
        }
        gsync();
        // warm start in Box2D's order: all contacts (b2ContactSolver::WarmStart), then the joints in island order. The
        // additions to a body's velocity do not commute in float arithmetic, so the leader applies them one after the other.
        if (leader()) {
            for_contacts(nt, [&](float* hc, const int st, int) {
                int meta = __float_as_int(hc[HC_META * st]);
                int b = meta & 0xff, count = (meta >> 8) & 3;
                float mB = HB(HB_INVM, b), iB = HB(HB_INVI, b);
                V2 vB = mk(HB(HB_VX, b), HB(HB_VY, b)); float wB = HB(HB_W, b);
                V2 normal = mk(hc[HC_NX * st], hc[HC_NY * st]), tangent = cross_vs(normal, 1.0f);
                {
                    V2 r = mk(hc[HC_R0X * st], hc[HC_R0Y * st]);
                    V2 P = hc[HC_NI0 * st] * normal + hc[HC_TI0 * st] * tangent;
                    wB += iB * cross(r, P); vB = vB + mB * P;
                }
                if (count > 1) {
                    V2 r = mk(hc[HC_R1X * st], hc[HC_R1Y * st]);
                    V2 P = hc[HC_NI1 * st] * normal + hc[HC_TI1 * st] * tangent;
                    wB += iB * cross(r, P); vB = vB + mB * P;
                }
                HB(HB_VX, b) = vB.x; HB(HB_VY, b) = vB.y; HB(HB_W, b) = wB;
            });
            for (int s = 0; s < nj; ++s) {
                const int meta = HJi(HJ_META, s);
                const int a = meta & 0xff, b = (meta >> 8) & 0xff;
                const float mA = HB(HB_INVM, a), iA = HB(HB_INVI, a), mB = HB(HB_INVM, b), iB = HB(HB_INVI, b);
                const V2 rA = mk(HJ(HJ_RAX, s), HJ(HJ_RAY, s)), rB = mk(HJ(HJ_RBX, s), HJ(HJ_RBY, s));
                const float impz = HJ(HJ_IMPZ, s), mimp = HJ(HJ_MIMP, s);
                V2 vA = mk(HB(HB_VX, a), HB(HB_VY, a)); float wA = HB(HB_W, a);
                V2 vB = mk(HB(HB_VX, b), HB(HB_VY, b)); float wB = HB(HB_W, b);
                V2 P = mk(HJ(HJ_IMPX, s), HJ(HJ_IMPY, s));
                vA = vA - mA * P; wA -= iA * (cross(rA, P) + mimp + impz);
                vB = vB + mB * P; wB += iB * (cross(rB, P) + mimp + impz);
                HB(HB_VX, a) = vA.x; HB(HB_VY, a) = vA.y; HB(HB_W, a) = wA;
                HB(HB_VX, b) = vB.x; HB(HB_VY, b) = vB.y; HB(HB_W, b) = wB;
            }
            if (gs) {      // the last joint of every body in island order (it closes the body's position iteration, see solve_post)
                unsigned long long seen = 0ull;
                for (int s = nj - 1; s >= 0; --s) {
                    int meta = HJi(HJ_META, s);
                    const int a = meta & 0xff, b = (meta >> 8) & 0xff;
                    if (!((seen >> a) & 1ull)) { meta |= HJM_LAST_A; seen |= 1ull << a; }
                    if (!((seen >> b) & 1ull)) { meta |= HJM_LAST_B; seen |= 1ull << b; }
                    HJ(HJ_META, s) = __int_as_float(meta);
                }
            }
        }
        nt_out = nt;
        PHASE(PH_SCHEDULE);
        build_schedule(nt, false);
        return true;
    }
    // ---------------- static modulo schedule of one sequential-impulse sweep
    // Box2D solves the constraints of an island one after the other, every iteration in the same order (velocity: joints in
    // island order, then contacts; position: contacts, then joints). Two constraints commute EXACTLY iff they share no body,
    // so the order only matters per body: each body sees its incident constraints in sequence order, iteration after
    // iteration. The schedule gives constraint c a time tau_c = skew_c * P + slot_c such that, for every body, the times of its
    // incident constraints increase in sequence order and span less than one period P: iteration `it` of c then runs at time
    // (it + skew_c) * P + slot_c, every body still sees exactly Box2D's order (bit-identical results), at most G constraints
    // share a slot (one per lane), and in steady state every lane solves one constraint per slot - consecutive iterations
    // are software-pipelined across the creature's joint tree. Built greedily in sequence order (each constraint at the
    // earliest slot after its bodies' previous constraints that has a free lane), the period is tried upwards from the lower
    // bound max(ceil(n/G), max body degree); measured on L-system creatures: the achieved period IS that bound for 97 % of
    // them (tests/emu + tools/sched_sim.py). The run is then fully static: at slot p of super-step T lane l executes entry
    // SCH(p, l) for iteration T - skew - no readiness checks, one group barrier per slot.
    // Entry: bit 31 valid | bit 30 contact | skew << 8 | index (joint slot s or hot contact slot t).
    // Times are packed as (skew << 5 | slot); AUX(b) = deg | rem << 6 | first << 12 | last << 22 (10-bit times, 0x3ff = none).
    #define SCH_VALID 0x80000000
    #define SCH_CONTACT 0x40000000
    __device__ __forceinline__ int sched_body_b(bool contact, int idx) {
        if (contact) return __float_as_int(hot_elem(hc_off, HC_COUNT, idx)[HC_META * 32]) & 0xff;
        return (HJi(HJ_META, idx) >> 8) & 0xff;
    }
    __device__ bool try_schedule(int n, int nt, bool position_order, int P, int& smax_out) {      // leader
        int smax = 0;
        for (int q = 0; q < n; ++q) {
            // q-th constraint of the sweep
            bool contact; int idx;
            if (position_order) { contact = q < nt; idx = contact ? q : q - nt; }
            else { contact = q >= nj; idx = contact ? q - nj : q; }
            const int ub = sched_body_b(contact, idx);
            const int ua = contact ? -1 : (HJi(HJ_META, idx) & 0xff);
            int lo = 0, hi = 0x7fffffff;
            const int wb = AUX(ub);
            const int wa = ua >= 0 ? AUX(ua) : 0;
            {
                const int first = (wb >> 12) & 0x3ff, last = (wb >> 22) & 0x3ff, rem = (wb >> 6) & 0x3f;
                if (first != 0x3ff) {
                    int t = last + 1; if ((t & 31) == P) t = (t & ~31) + 32;
                    lo = t;
                    int pp = (first & 31) + (P - rem), ss = first >> 5;
                    if (pp >= P) { pp -= P; ++ss; }
                    hi = (ss << 5) | pp;
                }
            }
            if (ua >= 0) {
                const int first = (wa >> 12) & 0x3ff, last = (wa >> 22) & 0x3ff, rem = (wa >> 6) & 0x3f;
                if (first != 0x3ff) {
                    int t = last + 1; if ((t & 31) == P) t = (t & ~31) + 32;
                    if (t > lo) lo = t;
                    int pp = (first & 31) + (P - rem), ss = first >> 5;
                    if (pp >= P) { pp -= P; ++ss; }
                    const int h2 = (ss << 5) | pp;
                    if (h2 < hi) hi = h2;
                }
            }
            // lane: constraint idx lives in hot column (idx & (G-1)), so the lane with that index reads and writes its fields
            // without shared-memory bank conflicts; it is preferred when it is free in the earliest possible slot or the next
            // one, otherwise any free lane of the earliest slot with one takes the constraint
            int t = lo, lane_k = -1;
            {
                const int pref = idx & (G - 1);
                int t2 = lo;
                for (int tries = 0; tries < 2 && t2 <= hi; ++tries) {
                    if (SCH(t2 & 31, pref) == 0) { t = t2; lane_k = pref; break; }
                    ++t2; if ((t2 & 31) == P) t2 = (t2 & ~31) + 32;
                }
            }
            while (lane_k < 0 && t <= hi) {
                const int pslot = t & 31;
                for (int kk = 0; kk < G; ++kk)
                    if (SCH(pslot, kk) == 0) { lane_k = kk; break; }
                if (lane_k >= 0) break;
                ++t; if ((t & 31) == P) t = (t & ~31) + 32;
            }
            if (lane_k < 0) return false;
            const int skew = t >> 5;
            if (skew > RB_MAX_SKEW) return false;
            if (skew > smax) smax = skew;
            SCH(t & 31, lane_k) = (int)(SCH_VALID | (contact ? SCH_CONTACT : 0u) | (unsigned)(skew << 8) | (unsigned)idx);
            {
                int w = AUX(ub);
                if (((w >> 12) & 0x3ff) == 0x3ff) w = (w & ~(0x3ff << 12)) | (t << 12);
                w = (w & ~(0x3ff << 22)) | (t << 22);
                w -= 1 << 6;
                AUX(ub) = w;
            }
            if (ua >= 0) {
                int w = AUX(ua);
                if (((w >> 12) & 0x3ff) == 0x3ff) w = (w & ~(0x3ff << 12)) | (t << 12);
                w = (w & ~(0x3ff << 22)) | (t << 22);
                w -= 1 << 6;
                AUX(ua) = w;
            }
        }
        smax_out = smax;
        return true;
    }
    // Builds the schedule of this tick's velocity sweep (position_order = false; needs the staged HJ_META / HC_META) or
    // position sweep (true; needs the overlaid PJ_META / PC_META, same low bits). Sets sched_P (0: no schedule, the leader
    // runs the sweep sequentially) and sched_smax. Group-cooperative; ends with a group barrier.
    __device__ void build_schedule(int nt, bool position_order) {
        sched_P = 0; sched_smax = 0;
        if (gs == 0) return;
        const int n = nj + nt;
        if (nt > L.nt || n == 0) { gsync(); return; }      // spilled contacts (rare): sequential sweep
        // degrees
        for (int b = sub; b < nb; b += G) AUX(b) = 0;
        gsync();
        int P = 0;
        if (leader()) {
            for (int s = 0; s < nj; ++s) { const int m = HJi(HJ_META, s); AUX(m & 0xff) += 1; AUX((m >> 8) & 0xff) += 1; }
            for (int t = 0; t < nt; ++t) AUX(sched_body_b(true, t)) += 1;
            int maxdeg = 1;
            for (int b = 0; b < nb; ++b) { const int d = AUX(b); if (d > maxdeg) maxdeg = d; }
            P = (n + G - 1) >> gs;
            if (maxdeg > P) P = maxdeg;
        }
        P = bcast(P);
        gsync();
        for (;;) {
            if (P > RB_SCHED_ROWS) { P = 0; break; }
            for (int q = 0; q < P; ++q) SCH(q, sub) = 0;
            for (int b = sub; b < nb; b += G) { const int d = AUX(b) & 0x3f; AUX(b) = d | (d << 6) | (0x3ff << 12) | (0x3ff << 22); }
            gsync();
            int ok = 0, smax = 0;
            if (leader()) ok = try_schedule(n, nt, position_order, P, smax) ? 1 : 0;
            ok = bcast(ok);
            if (ok) { sched_smax = bcast(smax); break; }
            ++P;
            gsync();
        }
        sched_P = P;
        gsync();
    }

    // ---------------- velocity iterations: the hot loop (everything in shared memory)
    // NB: equal limits (|upper-lower| < 2*angularSlop) do not occur: limits are -+pi/2 (module_utility.py:28-29)
    __device__ void solve_velocity(int nt) {
        PHASE(PH_VELOCITY);
        const int vit = k->vel_iters;
        if (sched_P) {
            const int P = sched_P, total = (vit + sched_smax) * P;
            int pslot = 0, T = 0;
            // the schedule and the constraints' index words are constant during the sweeps: the next slot's entry and index
            // word are fetched while the current slot computes (they head the slot's chain of dependent shared-memory loads)
            int e = SCH(0, sub);
            int meta = __float_as_int(hot_elem((e & SCH_CONTACT) ? hc_off : hj_off, (e & SCH_CONTACT) ? HC_COUNT : HJ_COUNT, e < 0 ? (e & 0xff) : 0)[0]);
            for (int q = 0; q < total; ++q) {
                int pnext = pslot + 1, Tnext = T;
                if (pnext == P) { pnext = 0; ++Tnext; }
                const int e_next = SCH(pnext, sub);
                const int meta_next = __float_as_int(hot_elem((e_next & SCH_CONTACT) ? hc_off : hj_off, (e_next & SCH_CONTACT) ? HC_COUNT : HJ_COUNT,
                                                              e_next < 0 ? (e_next & 0xff) : 0)[0]);
                const int it = T - ((e >> 8) & 0xff);
                const bool act = e < 0 && it >= 0 && it < vit;
                const bool isj = act && !(e & SCH_CONTACT), isc = act && (e & SCH_CONTACT);
                // Wide groups (latency-bound launches: tails, small populations): a slot in which some lane of the warp has a
                // contact runs the revolute solve AND the contact solve in every lane as one straight-line sequence - loads,
                // both computations, stores (idle lanes compute on zeros: their loads and stores are predicated off) - so that the two
                // dependency chains overlap instead of being serialised by a divergent branch: the slot then takes about
                // max(joint, contact) instead of their sum. Narrow groups are throughput-bound and keep the divergent form.
                if (gs >= 3 && warp_any_converged(isc)) {
                    // (index word 0 for the idle lanes: bodies 0 / 0, always valid addresses)
                    JV jr; CV cr;
                    float* hc = hot_elem(hc_off, HC_COUNT, isc ? (e & 0xff) : 0);
                    joint_v_load(isj ? (e & 0xff) : 0, isj ? meta : 0, jr, isj);
                    contact_v_load(hc, 32, isc ? meta : 0, cr, isc);
                    joint_v_compute(jr);
                    contact_v_compute(cr);
                    if (isj) joint_v_store(e & 0xff, jr);
                    if (isc) { contact_v_store1(hc, 32, cr); if (cr.count != 1) contact_v_two(hc, 32, cr); }
                } else {
                    if (isj) joint_solve_velocity(e & 0xff, meta);
                    if (isc) contact_solve_velocity(hot_elem(hc_off, HC_COUNT, e & 0xff), 32);
                }
                gsync();
                pslot = pnext; T = Tnext; e = e_next; meta = meta_next;
            }
            return;
        }
        if (leader())
            for (int it = 0; it < vit; ++it) {
                for (int s = 0; s < nj; ++s) joint_solve_velocity(s);
                for_contacts(nt, [&](float* hc, const int st, int) { contact_solve_velocity(hc, st); });
            }
        gsync();
    }
    __device__ void solve_post(int nt) {
        PHASE(PH_STORE);
        const float hdt = k->dt;
        const int vit = k->vel_iters;
        if (leader()) cnt.c[REM2D_CNT_JOINT_VSOLVES] += (unsigned)(vit * nj);
        // store impulses
        for (int t = sub; t < nt; t += G)
            with_contact(t, [&](float* hc, const int st) {
                int meta = __float_as_int(hc[HC_META * st]);
                int c = (meta >> 16) & 0xffff, count = (meta >> 8) & 3;
                cnt.c[count == 1 ? REM2D_CNT_P1_VSOLVES : REM2D_CNT_M2_VSOLVES] += (unsigned)vit;
                C(CF_P0N, c) = hc[HC_NI0 * st]; C(CF_P0T, c) = hc[HC_TI0 * st];
                if (count > 1) { C(CF_P1N, c) = hc[HC_NI1 * st]; C(CF_P1T, c) = hc[HC_TI1 * st]; }
                contact_init_position(hc, st, c);          // position constraints overlay the hot contact slot
            });
        for (int s = sub; s < nj; s += G) {
            int j = (HJi(HJ_META, s) >> 24) & 0xff;
            J(JF_IMPX, j) = HJ(HJ_IMPX, s); J(JF_IMPY, j) = HJ(HJ_IMPY, s); J(JF_IMPZ, j) = HJ(HJ_IMPZ, s);
            J(JF_MIMP, j) = HJ(HJ_MIMP, s);
            HJ(PJ_LAAX, s) = J(JF_LAAX, j); HJ(PJ_LAAY, s) = J(JF_LAAY, j);      // position overlay of the hot joint slot
            HJ(PJ_LABX, s) = J(JF_LABX, j); HJ(PJ_LABY, s) = J(JF_LABY, j);
            HJ(PJ_LOWER, s) = J(JF_LOWER, j); HJ(PJ_UPPER, s) = J(JF_UPPER, j);
        }
        // integrate positions; velocities go back to the cold block, the hot body slots become (c, a)
        for (int b = sub; b < nb; b += G) {
            V2 c = mk(B(BF_CX, b), B(BF_CY, b)); float a = B(BF_A, b);
            V2 v = mk(HB(HB_VX, b), HB(HB_VY, b)); float w = HB(HB_W, b);
            V2 translation = hdt * v;
            if (dot(translation, translation) > RB_MAX_TRANS * RB_MAX_TRANS) {
                float ratio = RB_MAX_TRANS / len(translation);
                v = ratio * v;
            }
            float rotation = hdt * w;
            if (rotation * rotation > RB_MAX_ROT * RB_MAX_ROT) {
                float ratio = RB_MAX_ROT / abs2(rotation);
                w *= ratio;
            }
            c = c + hdt * v; a += hdt * w;
            B(BF_VX, b) = v.x; B(BF_VY, b) = v.y; B(BF_W, b) = w;
            HB(HB_VX, b) = c.x; HB(HB_VY, b) = c.y; HB(HB_W, b) = a;
        }
        gsync();
        PHASE(PH_POSITION);
        int positionSolved = 0;
        const int pit = k->pos_iters;
        const int psmax = sched_smax + (nt > 0 ? 1 : 0);
        if (sched_P && nj > 0 && psmax < RB_RING && pit <= 64) {      // (nj > 0: every body has a joint that files its pose)
            // Pipelined position iterations on the velocity schedule. A position sweep solves the contacts first and the joints
            // after them, i.e. every body sees the SAME cyclic order of its constraints as in a velocity sweep, only the
            // iteration starts at its contacts: the schedule is reused with the joints one period later than the contacts
            // (skew + 1). Box2D stops after the first iteration in which every constraint was within tolerance, which is only
            // known when the slowest-skewed constraint has finished that iteration - lanes have then run ahead by up to
            // psmax iterations. Every body therefore files its pose at the end of each iteration (after its last joint) in a
            // ring of RB_RING entries, and on convergence at iteration K the poses of iteration K are restored: exactly the
            // state of the sequential loop at its break.
            const int P = sched_P;
            unsigned long long bad = 0ull;        // bit it: one of MY constraints was out of tolerance in iteration it
            int stopK = -1;
            for (int T = 0; T < pit + psmax && stopK < 0; ++T) {
                for (int pslot = 0; pslot < P; ++pslot) {
                    const int e = SCH(pslot, sub);
                    const bool isc = (e & SCH_CONTACT) != 0;
                    const int it = T - ((e >> 8) & 0xff) - (isc || nt == 0 ? 0 : 1);
                    const bool act = e < 0 && it >= 0 && it < pit;
                    if (act && isc) {
                        const float ms = contact_solve_position<false>(hot_elem(hc_off, HC_COUNT, e & 0xff), 32, RB_BAUMGARTE, 0.0f);
                        if (!(ms >= -3.0f * RB_LINEAR_SLOP)) bad |= 1ull << it;
                    }
                    if (act && !isc) {
                        const int sj = e & 0xff;
                        if (!joint_solve_position(sj)) bad |= 1ull << it;
                        const int meta = HJi(PJ_META, sj);
                        if (meta & HJM_LAST_A) { const int a = meta & 0xff; RING(it & (RB_RING - 1), a, 0) = HB(HB_VX, a); RING(it & (RB_RING - 1), a, 1) = HB(HB_VY, a); RING(it & (RB_RING - 1), a, 2) = HB(HB_W, a); }
                        if (meta & HJM_LAST_B) { const int b = (meta >> 8) & 0xff; RING(it & (RB_RING - 1), b, 0) = HB(HB_VX, b); RING(it & (RB_RING - 1), b, 1) = HB(HB_VY, b); RING(it & (RB_RING - 1), b, 2) = HB(HB_W, b); }
                    }
                    gsync();
                }
                const int d = T - psmax;          // every constraint has finished iteration d
                if (d >= 0 && !group_any(((bad >> d) & 1ull) != 0ull)) stopK = d;
            }
            const int iters = stopK >= 0 ? stopK + 1 : pit;
            positionSolved = stopK >= 0 ? 1 : 0;
            if (stopK >= 0 && psmax > 0)
                for (int b = sub; b < nb; b += G) {
                    HB(HB_VX, b) = RING(stopK & (RB_RING - 1), b, 0); HB(HB_VY, b) = RING(stopK & (RB_RING - 1), b, 1);
                    HB(HB_W, b) = RING(stopK & (RB_RING - 1), b, 2);
                }
            if (leader()) {
                cnt.c[REM2D_CNT_JOINT_PSOLVES] += (unsigned)(iters * nj);
                int points = 0;
                for (int t = 0; t < nt; ++t) points += (__float_as_int(hot_elem(hc_off, HC_COUNT, t)[PC_META * 32]) >> 8) & 3;
                cnt.c[REM2D_CNT_POINT_PSOLVES] += (unsigned)(iters * points);
            }
        } else {
            if (leader()) {
                for (int it = 0; it < pit; ++it) {
                    float minSep = 0.0f;
                    for_contacts(nt, [&](float* hc, const int st, int) { minSep = contact_solve_position(hc, st, RB_BAUMGARTE, minSep); });
                    bool contactsOkay = minSep >= -3.0f * RB_LINEAR_SLOP;
                    bool jointsOkay = true;
                    for (int s = 0; s < nj; ++s) { bool ok = joint_solve_position(s); jointsOkay = jointsOkay && ok; }
                    cnt.c[REM2D_CNT_JOINT_PSOLVES] += (unsigned)nj;
                    if (contactsOkay && jointsOkay) { positionSolved = 1; break; }
                }
            }
            positionSolved = bcast(positionSolved);
        }
        gsync();
        // copy back, synchronize transforms, sleep management
        PHASE(PH_FINALIZE);
        float minSleepTime = RB_MAXF;
        for (int b = sub; b < nb; b += G) {
            B(BF_CX, b) = HB(HB_VX, b); B(BF_CY, b) = HB(HB_VY, b); B(BF_A, b) = HB(HB_W, b);
            sync_transform(b);
            if (k->allow_sleep) {
                float w = B(BF_W, b); V2 v = mk(B(BF_VX, b), B(BF_VY, b));
                if (w * w > RB_ANG_SLEEP_TOL * RB_ANG_SLEEP_TOL || dot(v, v) > RB_LIN_SLEEP_TOL * RB_LIN_SLEEP_TOL) {
                    B(BF_SLEEP, b) = 0.0f; minSleepTime = 0.0f;
                } else {
                    float st = B(BF_SLEEP, b) + hdt;
                    B(BF_SLEEP, b) = st; minSleepTime = min2(minSleepTime, st);
                }
            }
        }
        if (gs) minSleepTime = group_min(minSleepTime);
        if (k->allow_sleep && minSleepTime >= RB_TIME_TO_SLEEP && positionSolved)
            for (int b = sub; b < nb; b += G) set_awake(b, false);
        for (int b = sub; b < nb; b += G) synchronize_fixtures(b);      // (independent per body: any order)
        gsync();
        PHASE(PH_FINDNEW);
        find_new_contacts_group();
    }

    // ---- continuous collision: b2TimeOfImpact / b2Distance with proxy A = terrain edge (identity frame)
    struct Sweep { V2 c0, c; float a0, a, alpha0; };
    struct Prox { V2 v[4]; int count; float radius; };
    struct SimplexCache { float metric; int count; int ia[3], ib[3]; };
    struct SV { V2 wA, wB, w; float a; int ia, ib; };

    __device__ __forceinline__ void sweep_xf(const Sweep& s, float beta, V2& p, Rot& q) {
        p = (1.0f - beta) * s.c0 + beta * s.c;
        float angle = (1.0f - beta) * s.a0 + beta * s.a;
        q = rot_set(angle);
        p = p - rmul(q, mk(0.0f, 0.0f));
    }
    __device__ __forceinline__ int support(const V2* v, int count, V2 d) {
        int best = 0; float bestValue = dot(v[0], d);
        for (int i = 1; i < count; ++i) { float value = dot(v[i], d); if (value > bestValue) { best = i; bestValue = value; } }
        return best;
    }
    __device__ __forceinline__ float metric(const SV* s, int count) {
        if (count == 2) return len(s[0].w - s[1].w);
        if (count == 3) return cross(s[1].w - s[0].w, s[2].w - s[0].w);
        return 0.0f;
    }
    __device__ float gjk(SimplexCache& cache, const V2* ev, const Prox& pb, V2 pB, Rot qB) {
        SV s[3]; int count = cache.count;
        for (int i = 0; i < count; ++i) {
            s[i].ia = cache.ia[i]; s[i].ib = cache.ib[i];
            s[i].wA = ev[s[i].ia];
            s[i].wB = xmul(pB, qB, pb.v[s[i].ib]);
            s[i].w = s[i].wB - s[i].wA; s[i].a = 0.0f;
        }
        if (count > 1) {
            float m1 = cache.metric, m2 = metric(s, count);
            if (m2 < 0.5f * m1 || 2.0f * m1 < m2 || m2 < RB_EPS) count = 0;
        }
        if (count == 0) {
            s[0].ia = 0; s[0].ib = 0; s[0].wA = ev[0]; s[0].wB = xmul(pB, qB, pb.v[0]);
            s[0].w = s[0].wB - s[0].wA; s[0].a = 1.0f; count = 1;
        }
        int saveA[3], saveB[3], saveCount = 0, iter = 0;
        while (iter < 20) {
            saveCount = count;
            for (int i = 0; i < saveCount; ++i) { saveA[i] = s[i].ia; saveB[i] = s[i].ib; }
            if (count == 2) {
                V2 w1 = s[0].w, w2 = s[1].w, e12 = w2 - w1;
                float d12_2 = -dot(w1, e12);
                if (d12_2 <= 0.0f) { s[0].a = 1.0f; count = 1; }
                else {
                    float d12_1 = dot(w2, e12);
                    if (d12_1 <= 0.0f) { s[1].a = 1.0f; count = 1; s[0] = s[1]; }
                    else { float inv = 1.0f / (d12_1 + d12_2); s[0].a = d12_1 * inv; s[1].a = d12_2 * inv; count = 2; }
                }
            } else if (count == 3) {
                V2 w1 = s[0].w, w2 = s[1].w, w3 = s[2].w;
                V2 e12 = w2 - w1; float w1e12 = dot(w1, e12), w2e12 = dot(w2, e12); float d12_1 = w2e12, d12_2 = -w1e12;
                V2 e13 = w3 - w1; float w1e13 = dot(w1, e13), w3e13 = dot(w3, e13); float d13_1 = w3e13, d13_2 = -w1e13;
                V2 e23 = w3 - w2; float w2e23 = dot(w2, e23), w3e23 = dot(w3, e23); float d23_1 = w3e23, d23_2 = -w2e23;
                float n123 = cross(e12, e13);
                float d123_1 = n123 * cross(w2, w3), d123_2 = n123 * cross(w3, w1), d123_3 = n123 * cross(w1, w2);
                if (d12_2 <= 0.0f && d13_2 <= 0.0f) { s[0].a = 1.0f; count = 1; }
                else if (d12_1 > 0.0f && d12_2 > 0.0f && d123_3 <= 0.0f) { float inv = 1.0f / (d12_1 + d12_2); s[0].a = d12_1 * inv; s[1].a = d12_2 * inv; count = 2; }
                else if (d13_1 > 0.0f && d13_2 > 0.0f && d123_2 <= 0.0f) { float inv = 1.0f / (d13_1 + d13_2); s[0].a = d13_1 * inv; s[2].a = d13_2 * inv; count = 2; s[1] = s[2]; }
                else if (d12_1 <= 0.0f && d23_2 <= 0.0f) { s[1].a = 1.0f; count = 1; s[0] = s[1]; }
                else if (d13_1 <= 0.0f && d23_1 <= 0.0f) { s[2].a = 1.0f; count = 1; s[0] = s[2]; }
                else if (d23_1 > 0.0f && d23_2 > 0.0f && d123_1 <= 0.0f) { float inv = 1.0f / (d23_1 + d23_2); s[1].a = d23_1 * inv; s[2].a = d23_2 * inv; count = 2; s[0] = s[2]; }
                else { float inv = 1.0f / (d123_1 + d123_2 + d123_3); s[0].a = d123_1 * inv; s[1].a = d123_2 * inv; s[2].a = d123_3 * inv; count = 3; }
            }
            if (count == 3) break;
            V2 d;
            if (count == 1) d = -s[0].w;
            else {
                V2 e12 = s[1].w - s[0].w;
                float sgn = cross(e12, -s[0].w);
                d = sgn > 0.0f ? cross_sv(1.0f, e12) : cross_vs(e12, 1.0f);
            }
            if (dot(d, d) < RB_EPS * RB_EPS) break;
            SV& vtx = s[count];
            vtx.ia = support(ev, 2, -d);
            vtx.wA = ev[vtx.ia];
            vtx.ib = support(pb.v, pb.count, rmulT(qB, d));
            vtx.wB = xmul(pB, qB, pb.v[vtx.ib]);
            vtx.w = vtx.wB - vtx.wA;
            ++iter;
            cnt.c[REM2D_CNT_GJK_ITERS]++;
            bool dup = false;
            for (int i = 0; i < saveCount; ++i) if (vtx.ia == saveA[i] && vtx.ib == saveB[i]) { dup = true; break; }
            if (dup) break;
            ++count;
        }
        V2 a, b;
        if (count == 1) { a = s[0].wA; b = s[0].wB; }
        else if (count == 2) { a = s[0].a * s[0].wA + s[1].a * s[1].wA; b = s[0].a * s[0].wB + s[1].a * s[1].wB; }
        else { a = s[0].a * s[0].wA + s[1].a * s[1].wA + s[2].a * s[2].wA; b = a; }
        float distance = len(a - b);
        cache.metric = metric(s, count);
        cache.count = count;
        for (int i = 0; i < count; ++i) { cache.ia[i] = s[i].ia; cache.ib[i] = s[i].ib; }
        return distance;
    }

    struct SepFn { int type; V2 localPoint, axis; };
    __device__ __forceinline__ float sep_find_min(const SepFn& f, const V2* ev, const Prox& pb, const Sweep& sw, int& ia, int& ib, float t) {
        V2 pB; Rot qB; sweep_xf(sw, t, pB, qB);
        if (f.type == 0) {
            ia = support(ev, 2, f.axis);
            ib = support(pb.v, pb.count, rmulT(qB, -f.axis));
            V2 pointA = ev[ia], pointB = xmul(pB, qB, pb.v[ib]);
            return dot(pointB - pointA, f.axis);
        } else if (f.type == 1) {
            V2 normal = f.axis, pointA = f.localPoint;
            ia = -1;
            ib = support(pb.v, pb.count, rmulT(qB, -normal));
            V2 pointB = xmul(pB, qB, pb.v[ib]);
            return dot(pointB - pointA, normal);
        } else {
            V2 normal = rmul(qB, f.axis), pointB = xmul(pB, qB, f.localPoint);
            ib = -1;
            ia = support(ev, 2, -normal);
            V2 pointA = ev[ia];
            return dot(pointA - pointB, normal);
        }
    }
    __device__ __forceinline__ float sep_eval(const SepFn& f, const V2* ev, const Prox& pb, const Sweep& sw, int ia, int ib, float t) {
        V2 pB; Rot qB; sweep_xf(sw, t, pB, qB);
        if (f.type == 0) { V2 pointA = ev[ia], pointB = xmul(pB, qB, pb.v[ib]); return dot(pointB - pointA, f.axis); }
        else if (f.type == 1) { V2 pointB = xmul(pB, qB, pb.v[ib]); return dot(pointB - f.localPoint, f.axis); }
        else { V2 normal = rmul(qB, f.axis), pointB = xmul(pB, qB, f.localPoint); V2 pointA = ev[ia]; return dot(pointA - pointB, normal); }
    }
    // returns true iff the TOI state is "touching"; t receives output.t
    __device__ bool time_of_impact(const V2* ev, const Prox& pb, Sweep sw, float& tOut) {
        cnt.c[REM2D_CNT_TOI_CALLS]++;
        const float tMax = 1.0f;
        tOut = tMax;
        {   // b2Sweep::Normalize
            float twoPi = 2.0f * RB_PI;
            float d = twoPi * floorf(sw.a0 / twoPi);
            sw.a0 -= d; sw.a -= d;
        }
        float totalRadius = RB_POLY_RADIUS + pb.radius;
        float target = max2(RB_LINEAR_SLOP, totalRadius - 3.0f * RB_LINEAR_SLOP);
        float tolerance = 0.25f * RB_LINEAR_SLOP;
        float t1 = 0.0f;
        int iter = 0;
        SimplexCache cache; cache.count = 0; cache.metric = 0.0f;
        bool touching = false;
        for (;;) {
            V2 pB; Rot qB; sweep_xf(sw, t1, pB, qB);
            float distance = gjk(cache, ev, pb, pB, qB);
            if (distance <= 0.0f) { tOut = 0.0f; break; }                         // overlapped
            if (distance < target + tolerance) { touching = true; tOut = t1; break; }
            SepFn f;
            if (cache.count == 1) {
                f.type = 0;
                V2 pointA = ev[cache.ia[0]], pointB = xmul(pB, qB, pb.v[cache.ib[0]]);
                f.axis = pointB - pointA; normalize(f.axis); f.localPoint = mk(0.0f, 0.0f);
            } else if (cache.ia[0] == cache.ia[1]) {
                f.type = 2;
                V2 b1 = pb.v[cache.ib[0]], b2 = pb.v[cache.ib[1]];
                f.axis = cross_vs(b2 - b1, 1.0f); normalize(f.axis);
                V2 normal = rmul(qB, f.axis);
                f.localPoint = 0.5f * (b1 + b2);
                V2 pointB = xmul(pB, qB, f.localPoint), pointA = ev[cache.ia[0]];
                float s = dot(pointA - pointB, normal);
                if (s < 0.0f) f.axis = -f.axis;
            } else {
                f.type = 1;
                V2 a1 = ev[cache.ia[0]], a2 = ev[cache.ia[1]];
                f.axis = cross_vs(a2 - a1, 1.0f); normalize(f.axis);
                V2 normal = f.axis;
                f.localPoint = 0.5f * (a1 + a2);
                V2 pointA = f.localPoint, pointB = xmul(pB, qB, pb.v[cache.ib[0]]);
                float s = dot(pointB - pointA, normal);
                if (s < 0.0f) f.axis = -f.axis;
            }
            bool done = false;
            float t2 = tMax;
            int pushBackIter = 0;
            for (;;) {
                int ia, ib;
                float s2 = sep_find_min(f, ev, pb, sw, ia, ib, t2);
                if (s2 > target + tolerance) { tOut = tMax; done = true; break; }                 // separated
                if (s2 > target - tolerance) { t1 = t2; break; }
                float s1 = sep_eval(f, ev, pb, sw, ia, ib, t1);
                if (s1 < target - tolerance) { tOut = t1; done = true; break; }                   // failed
                if (s1 <= target + tolerance) { touching = true; tOut = t1; done = true; break; }
                int rootIter = 0;
                float a1 = t1, a2 = t2;
                for (;;) {
                    float t;
                    if (rootIter & 1) t = a1 + (target - s1) * (a2 - a1) / (s2 - s1);
                    else t = 0.5f * (a1 + a2);
                    ++rootIter;
                    cnt.c[REM2D_CNT_TOI_ROOT_ITERS]++;
                    float s = sep_eval(f, ev, pb, sw, ia, ib, t);
                    if (abs2(s - target) < tolerance) { t2 = t; break; }
                    if (s > target) { a1 = t; s1 = s; } else { a2 = t; s2 = s; }
                    if (rootIter == 50) break;
                }
                ++pushBackIter;
                if (pushBackIter == RB_MAX_POLY_VERTS) break;
            }
            ++iter;
            if (done) break;
            if (iter == 20) { tOut = t1; break; }                                                  // failed
        }
        return touching;
    }

    // b2DistanceProxy::Set of body b's shape (circle: its centre and radius; box: its 4 vertices and the polygon skin)
    __device__ __forceinline__ Prox body_proxy(int b) {
        Prox pb;
        float hx = B(BF_HX, b), hy = B(BF_HY, b);
        if (Bi(BF_FLAGS, b) & BFL_CIRCLE) { pb.count = 1; pb.radius = hx; pb.v[0] = mk(0.0f, 0.0f); pb.v[1] = pb.v[2] = pb.v[3] = pb.v[0]; }
        else { pb.count = 4; pb.radius = RB_POLY_RADIUS; pb.v[0] = mk(-hx, -hy); pb.v[1] = mk(hx, -hy); pb.v[2] = mk(hx, hy); pb.v[3] = mk(-hx, hy); }
        return pb;
    }

    __device__ __forceinline__ void body_advance(int b, float alpha) {
        float alpha0 = B(BF_ALPHA0, b);
        float beta = (alpha - alpha0) / (1.0f - alpha0);
        V2 c0 = mk(B(BF_C0X, b), B(BF_C0Y, b)), c = mk(B(BF_CX, b), B(BF_CY, b));
        float a0 = B(BF_A0, b), a = B(BF_A, b);
        c0 = c0 + beta * (c - c0);
        a0 += beta * (a - a0);
        B(BF_C0X, b) = c0.x; B(BF_C0Y, b) = c0.y; B(BF_A0, b) = a0; B(BF_ALPHA0, b) = alpha;
        B(BF_CX, b) = c0.x; B(BF_CY, b) = c0.y; B(BF_A, b) = a0;
        sync_transform(b);
    }
    __device__ __forceinline__ void set_edge_alpha(int e, float alpha) {
        EA(e) = alpha;
        int n = Si(S_NADV);
        if (n < 8) setSi(S_ADV0 + n, e);
        setSi(S_NADV, n + 1);
    }

    // time of impact of pool contact c against its body's sweep (the body of b2World::SolveTOI's inner loop); leaves the
    // sweeps untouched when both alpha0 are equal (always the case in the first scan of a step)
    __device__ float contact_toi(int c, int key) {
        int b = key_body(key), e = key_edge(key);
        float aA0 = EA(e), aB0 = B(BF_ALPHA0, b);
        float alpha0 = aA0;
        Sweep sw;
        sw.c0 = mk(B(BF_C0X, b), B(BF_C0Y, b)); sw.c = mk(B(BF_CX, b), B(BF_CY, b));
        sw.a0 = B(BF_A0, b); sw.a = B(BF_A, b); sw.alpha0 = aB0;
        if (aA0 < aB0) { alpha0 = aB0; set_edge_alpha(e, alpha0); }
        else if (aB0 < aA0) {
            alpha0 = aA0;
            float beta = (alpha0 - sw.alpha0) / (1.0f - sw.alpha0);
            sw.c0 = sw.c0 + beta * (sw.c - sw.c0);
            sw.a0 += beta * (sw.a - sw.a0);
            sw.alpha0 = alpha0;
            B(BF_C0X, b) = sw.c0.x; B(BF_C0Y, b) = sw.c0.y; B(BF_A0, b) = sw.a0; B(BF_ALPHA0, b) = alpha0;
        }
        V2 ev[2] = { mk(__ldg(&ter->v1x[e]), __ldg(&ter->v1y[e])), mk(__ldg(&ter->v2x[e]), __ldg(&ter->v2y[e])) };
        Prox pb = body_proxy(b);
        float t;
        bool touching = time_of_impact(ev, pb, sw, t);
        float alpha = 1.0f;
        if (touching) alpha = min2(alpha0 + (1.0f - alpha0) * t, 1.0f);
        return alpha;
    }

    // b2World::SolveTOI. Group-cooperative: the first scan over the contacts - one time-of-impact query per contact of an awake
    // body, every sweep still at alpha0 = 0, so the queries are independent - is strided over the lanes and leaves its results
    // in the pool (toi + toiFlag) exactly as Box2D caches them; the leader then runs Box2D's loop, which finds the cached
    // values, and handles TOI events (rare: 2 % of the ticks) sequentially.
    __device__ void solve_toi() {
        PHASE(PH_TOI_SCAN);
        const float dt = k->dt;
        for (int b = sub; b < nb; b += G) { setBi(BF_FLAGS, b, Bi(BF_FLAGS, b) & ~BFL_ISLAND); B(BF_ALPHA0, b) = 0.0f; }
        if (leader()) {   // alpha0 of the static edge bodies: clear what the previous step dirtied
            int n = Si(S_NADV);
            if (n > 8) { for (int e = 0; e < RB_MAX_EDGES; ++e) EA(e) = 0.0f; }
            else for (int i = 0; i < n; ++i) EA(Si(S_ADV0 + i)) = 0.0f;
            setSi(S_NADV, 0);
        }
        int nc = bcast(Si(S_NC));
        gsync();
        for (int c = nc - 1 - sub; c >= 0; c -= G) {
            int key = Ci(CF_KEY, c);
            key &= ~((CK_TOIFLAG | CK_ISLAND) << 16);
            key &= 0x00ffffff;                                    // toiCount = 0
            float alpha = 1.0f;
            if ((key_flags(key) & CK_ENABLED) && (Bi(BF_FLAGS, key_body(key)) & BFL_AWAKE)) {
                alpha = contact_toi(c, key);
                key |= CK_TOIFLAG << 16;
            }
            setCi(CF_KEY, c, key);
            C(CF_TOI, c) = alpha;
        }
        gsync();
        PHASE(PH_TOI_EVENTS);
        if (leader()) solve_toi_events(dt);
        gsync();
    }
    __device__ void solve_toi_events(const float dt) {       // leader
        int nc;
        for (;;) {
            nc = Si(S_NC);
            int minContact = -1; float minAlpha = 1.0f;
            for (int c = nc - 1; c >= 0; --c) {
                int key = Ci(CF_KEY, c);
                int fl = key_flags(key);
                if (!(fl & CK_ENABLED)) continue;
                if (key_toicount(key) > RB_MAX_SUBSTEPS) continue;
                float alpha = 1.0f;
                if (fl & CK_TOIFLAG) alpha = C(CF_TOI, c);
                else {
                    if (!(Bi(BF_FLAGS, key_body(key)) & BFL_AWAKE)) continue;
                    alpha = contact_toi(c, key);
                    C(CF_TOI, c) = alpha;
                    setCi(CF_KEY, c, key | (CK_TOIFLAG << 16));
                }
                if (alpha < minAlpha) { minContact = c; minAlpha = alpha; }
            }
            if (minContact < 0 || 1.0f - 10.0f * RB_EPS < minAlpha) break;
            cnt.c[REM2D_CNT_TOI_EVENTS]++;
            int mkey = Ci(CF_KEY, minContact);
            int mb = key_body(mkey), eA = key_edge(mkey);
            // backups
            float bk_c0x = B(BF_C0X, mb), bk_c0y = B(BF_C0Y, mb), bk_a0 = B(BF_A0, mb), bk_al = B(BF_ALPHA0, mb);
            float bk_cx = B(BF_CX, mb), bk_cy = B(BF_CY, mb), bk_a = B(BF_A, mb);
            float bk_ea = EA(eA);
            set_edge_alpha(eA, minAlpha);
            body_advance(mb, minAlpha);
            contact_update(minContact);
            mkey = Ci(CF_KEY, minContact);
            mkey &= ~(CK_TOIFLAG << 16);
            mkey += 1 << 24;                                       // ++toiCount
            setCi(CF_KEY, minContact, mkey);
            if (!(key_flags(mkey) & CK_ENABLED) || !(key_flags(mkey) & CK_TOUCHING)) {
                setCi(CF_KEY, minContact, mkey & ~(CK_ENABLED << 16));
                EA(eA) = bk_ea;
                B(BF_C0X, mb) = bk_c0x; B(BF_C0Y, mb) = bk_c0y; B(BF_A0, mb) = bk_a0; B(BF_ALPHA0, mb) = bk_al;
                B(BF_CX, mb) = bk_cx; B(BF_CY, mb) = bk_cy; B(BF_A, mb) = bk_a;
                sync_transform(mb);
                continue;
            }
            set_awake(mb, true);
            // TOI mini-island: this module + its touching contacts (joints are NOT part of it)
            int isl[RB_TOI_ISLAND_CAP]; int ni = 0;
            isl[ni++] = minContact;
            setCi(CF_KEY, minContact, mkey | (CK_ISLAND << 16));
            for (int c = nc - 1; c >= 0; --c) {
                int key = Ci(CF_KEY, c);
                if (key_body(key) != mb) continue;
                if (key_flags(key) & CK_ISLAND) continue;
                if (ni == RB_TOI_ISLAND_CAP) break;
                int e = key_edge(key);
                bool inIsland = false;
                for (int i = 0; i < ni; ++i) inIsland |= (key_edge(Ci(CF_KEY, isl[i])) == e);
                float backup = EA(e);
                if (!inIsland) set_edge_alpha(e, minAlpha);
                contact_update(c);
                key = Ci(CF_KEY, c);
                if (!(key_flags(key) & CK_ENABLED) || !(key_flags(key) & CK_TOUCHING)) { EA(e) = backup; continue; }
                setCi(CF_KEY, c, key | (CK_ISLAND << 16));
                isl[ni++] = c;
            }
            float subDt = (1.0f - minAlpha) * dt;
            // b2Island::SolveTOI: only the module moves
            float mB = B(BF_INVM, mb), iB = B(BF_INVI, mb);
            HB(HB_INVM, mb) = mB; HB(HB_INVI, mb) = iB;
            HB(HB_VX, mb) = B(BF_CX, mb); HB(HB_VY, mb) = B(BF_CY, mb); HB(HB_W, mb) = B(BF_A, mb);   // position overlay
            const int nt = ni;
            for_contacts(nt, [&](float* hc, const int st, int t) { contact_init_position(hc, st, isl[t]); });
            for (int it = 0; it < 20; ++it) {
                float minSep = 0.0f;
                for_contacts(nt, [&](float* hc, const int st, int) { minSep = contact_solve_position(hc, st, RB_TOI_BAUMGARTE, minSep); });
                if (minSep >= -1.5f * RB_LINEAR_SLOP) break;
            }
            V2 cB = mk(HB(HB_VX, mb), HB(HB_VY, mb)); float aB = HB(HB_W, mb);
            B(BF_C0X, mb) = cB.x; B(BF_C0Y, mb) = cB.y; B(BF_A0, mb) = aB;      // leap of faith
            for_contacts(nt, [&](float* hc, const int st, int t) { contact_init_velocity(hc, st, isl[t], cB, aB, mB, iB, 1.0f, false); });
            HB(HB_VX, mb) = B(BF_VX, mb); HB(HB_VY, mb) = B(BF_VY, mb); HB(HB_W, mb) = B(BF_W, mb);
            const int vit = k->vel_iters;
            for (int it = 0; it < vit; ++it)
                for_contacts(nt, [&](float* hc, const int st, int) { contact_solve_velocity(hc, st); });
            count_contact_solves(nt, vit);
            {
                V2 v = mk(HB(HB_VX, mb), HB(HB_VY, mb)); float w = HB(HB_W, mb);
                V2 translation = subDt * v;
                if (dot(translation, translation) > RB_MAX_TRANS * RB_MAX_TRANS) { float ratio = RB_MAX_TRANS / len(translation); v = ratio * v; }
                float rotation = subDt * w;
                if (rotation * rotation > RB_MAX_ROT * RB_MAX_ROT) { float ratio = RB_MAX_ROT / abs2(rotation); w *= ratio; }
                cB = cB + subDt * v; aB += subDt * w;
                B(BF_CX, mb) = cB.x; B(BF_CY, mb) = cB.y; B(BF_A, mb) = aB;
                B(BF_VX, mb) = v.x; B(BF_VY, mb) = v.y; B(BF_W, mb) = w;
                sync_transform(mb);
            }
            synchronize_fixtures(mb);
            for (int c = 0; c < nc; ++c) {
                int key = Ci(CF_KEY, c);
                if (key_body(key) == mb) setCi(CF_KEY, c, key & ~((CK_TOIFLAG | CK_ISLAND) << 16));
            }
            find_new_contacts();
        }
    }

    // ---- Modular2D.step + the body of evaluate()'s loop: tick_pre -> solve_velocity -> tick_post, all group-cooperative.
    // b2World::Step = FindNewContacts (first step) -> Collide -> Solve -> SolveTOI.
    __device__ bool tick_pre(int& nt) {
        PHASE(PH_CONTROL);
        if (leader()) {
            double wod = Sd(S_WOD_LO) + k->wod_speed;
            setSd(S_WOD_LO, wod);
        }
#ifdef REM2D_POLICY
        // the policy's inputs are the state at the start of the tick (rem2d_read_observations): first the bodies with a
        // touching terrain contact, a mask over the pool (order-free, strided over the group)
        unsigned long long ground = 0ull;
        const int n_pool = Si(S_NC);
        for (int q = sub; q < n_pool; q += G) {
            const int key = Ci(CF_KEY, q);
            if (key_flags(key) & CK_TOUCHING) ground |= 1ull << key_body(key);
        }
        for (int o = G >> 1; o > 0; o >>= 1) ground |= __shfl_xor_sync(gmask, ground, o);
        const int H = pol.n_hidden, P = 10 * H + 1;
        const double root_a = (double)B(BF_A, 0), root_vx = (double)B(BF_VX, 0), root_vy = (double)B(BF_VY, 0);
#endif
        for (int j = sub; j < nj; j += G) {
#ifdef REM2D_TARGETS
            // the controller output is the caller's target; the sine controller is not advanced (i_state unchanged)
            const double out = tgt[j];
#else
            double ist = Jd(JF_ISTATE, j) + Jd(JF_FREQ, j);
            setJd(JF_ISTATE, j, ist);
            double s, c;
            sincos_kernel(ist + (Jd(JF_PHASE, j) + 0.0), s, c);
            double out = Jd(JF_AMP, j) * s + Jd(JF_OFFS, j);
#endif
            int a = Ji(JF_META, j) & 0xff, b = j + 1;
            float currentAngle = B(BF_A, b) - B(BF_A, a) - 0.0f;
#ifdef REM2D_POLICY
            {   // the joint's network (include/rem2d_policy.h): target = sine output + u, in this order of operations
                const double* __restrict__ w = pw + (size_t)j * P;
                const double x[REM2D_POLICY_FEATURES] = {out, (double)currentAngle, (double)(B(BF_W, b) - B(BF_W, a)),
                                                         (double)((ground >> b) & 1ull), (double)((ground >> a) & 1ull),
                                                         root_a, root_vx, root_vy};
                double u = __ldg(w + 10 * H);
                for (int k = 0; k < H; ++k) {
                    double acc = __ldg(w + 8 * H + k);
#pragma unroll
                    for (int i = 0; i < REM2D_POLICY_FEATURES; ++i) acc = acc + __ldg(w + 8 * k + i) * x[i];
                    u = u + __ldg(w + 9 * H + k) * (acc / (1.0 + fabs(acc)));
                }
                out = out + u;
            }
#endif
            double speed = (out - (double)currentAngle) * k->p_gain;
            set_awake(a, true); set_awake(b, true);       // (lanes may wake the same body: identical idempotent writes)
            J(JF_MSPEED, j) = (float)speed;
        }
        const float dt = k->dt;
        const int newfix = bcast(Si(S_NEWFIX));
        gsync();
        if (newfix) {
            PHASE(PH_FINDNEW);
            find_new_contacts_group();
            if (leader()) setSi(S_NEWFIX, 0);
            gsync();
        }
        float dtRatio = S(S_INVDT0) * dt;
        PHASE(PH_COLLIDE);
        collide();
        nt = 0;
        PHASE(PH_STAGE);
        return dt > 0.0f ? solve_pre(dtRatio, nt) : false;
    }
    __device__ void tick_post(bool solved, int nt) {
        const float dt = k->dt;
        if (solved) solve_post(nt);
        if (k->continuous && dt > 0.0f) solve_toi();
        PHASE(PH_LOOP);
        if (leader()) {
            if (dt > 0.0f) S(S_INVDT0) = 1.0f / dt;
            cnt.c[REM2D_CNT_TICKS]++;
            int i = Si(S_TICKS);
            setSi(S_TICKS, i + 1);
            float x = B(BF_CX, 0);
            double wod = Sd(S_WOD_LO);
            double reward = (double)x;
            if (k->terminate) {
                if (x < 0.0f) reward = -100.0;
                if (wod > (double)x) reward = -100.0;
                if (reward < -10.0) setSi(S_ALIVE, 0);
                else if (reward > k->env_length) {
                    reward += (double)(k->evaluation_steps - i) / (double)k->evaluation_steps;
                    setSd(S_FIT_LO, reward);
                    setSi(S_ALIVE, 0);
                } else if (reward > 0.0) setSd(S_FIT_LO, reward);
                if (i + 1 >= k->evaluation_steps) setSi(S_ALIVE, 0);
            } else if (reward > 0.0) setSd(S_FIT_LO, reward);
        }
#ifdef REM2D_STATS
        stats_tick();
#endif
        gsync();
    }
#ifdef REM2D_STATS
    // ---- episode statistics (statistics images only). Each is defined by the state at the end of the tick, as
    // rem2d_read_state / rem2d_read_roots report it, and accumulated in the order of oracle/rem2d_oracle.c:tick().
    // Zero the statistics of creature c, pulled into this group (after build_world: nb is set).
    __device__ void stats_begin(int c) {
        const int b0 = st.body_off[c];
        for (int b = sub; b < nb; b += G) st.ground_ticks[b0 + b] = 0;
        if (leader()) {
            st.end_reason[c] = REM2D_END_RUNNING;
            st.max_x[c] = __int_as_float((int)0xff800000);       // -inf
            st.joint_work[c] = 0.0;
            st.airborne_ticks[c] = 0;
        }
    }
    __device__ void stats_tick() {
        gsync();                                         // the tick's writes to bodies, joints and contacts are done
        const int c = st_c, b0 = st.body_off[c];
        // bodies with a touching terrain contact: a mask over the pool (order-free, strided over the group)
        unsigned long long m = 0ull;
        const int n_pool = Si(S_NC);
        for (int q = sub; q < n_pool; q += G) {
            const int key = Ci(CF_KEY, q);
            if (key_flags(key) & CK_TOUCHING) m |= 1ull << key_body(key);
        }
        for (int o = G >> 1; o > 0; o >>= 1) m |= __shfl_xor_sync(gmask, m, o);
        for (int b = sub; b < nb; b += G)
            if ((m >> b) & 1ull) st.ground_ticks[b0 + b] += 1;
        // joint work: the group computes the terms, the leader adds them to the running sum in joint order
        double work = 0.0;
        if (leader()) work = st.joint_work[c];
        for (int base = 0; base < nj; base += G) {
            const int j = base + sub;
            double t = 0.0;
            if (j < nj) {
                const int a = Ji(JF_META, j) & 0xff;
                t = fabs((double)J(JF_MIMP, j) * ((double)B(BF_W, j + 1) - (double)B(BF_W, a)));
            }
            const int n = nj - base < G ? nj - base : G;
            for (int i = 0; i < n; ++i) {
                const double v = gs ? __shfl_sync(gmask, t, lead + i) : t;
                if (leader()) work += v;
            }
        }
        if (leader()) {
            st.joint_work[c] = work;
            if (m == 0ull) st.airborne_ticks[c] += 1;
            const float x = B(BF_CX, 0);
            if (x > st.max_x[c]) st.max_x[c] = x;
            // the comparisons of the termination rule above, in its precedence
            const double wod = Sd(S_WOD_LO);
            int why = REM2D_END_RUNNING;
            if (k->terminate) {
                if (x < 0.0f) why = REM2D_END_ORIGIN;
                else if (wod > (double)x) why = REM2D_END_WALL;
                else if ((double)x > k->env_length) why = REM2D_END_GOAL;
                else if (Si(S_TICKS) >= k->evaluation_steps) why = REM2D_END_STEPS;
            }
            if (why != REM2D_END_RUNNING) st.end_reason[c] = why;
        }
    }
#endif
    __device__ void tick() {
        int nt;
        bool solved = tick_pre(nt);
        if (solved) solve_velocity(nt);
        tick_post(solved, nt);
    }

    // ---- whole episodes: the loop of the episode kernel (rem2d_kernels.cu) in both modes, WARP-cooperative.
    // Queue mode: every group without a creature pulls the next one of the class queue, builds its world in the group's column
    // and ticks it until its episode ends; long-lived creatures are parked for the tail mode. Tail mode (tail = true): the groups
    // start with their parked creatures (my, column g) and nothing to pull. `tslot` is the park slot of a tail creature (-1:
    // none). Hooks: sample(sim, iteration, live lanes) before every iteration, regrouped(sim, old gs) after a regroup,
    // finished(sim, creature, tslot, iterations) on the leader of a group whose creature ended, now_us() for the park trace.
    //
    // Regrouping: once the queue is empty (some group of the warp failed a pull; pulls are monotone, so every later pull fails
    // too), the warp's dead groups would idle until the last live creature ends. Instead the warp packs its n live creatures onto
    // groups 0..n-1, in order, with the largest width 2^gs' <= 32 / n (at most max_gs), and repeats that as more creatures end.
    // Exact: every width runs the same code on the creature's own cold column, the hot block is staged from it at every tick
    // (solve_pre) and written back (solve_post), and make_hot_layout(L, gs').rows never exceeds the rows at a narrower gs, so
    // the widened groups fit in the shared memory the warp was launched with (tests/test_regroup.py).
    template <class Hooks>
    __device__ __forceinline__ void episodes(const int lane, const bool tail, const int max_gs, float* hot, const EpisodeQueue& Q,
                                             const ParkPolicy& park, float* park_state, int* park_creature, int* park_count,
                                             int my, int tslot, Hooks& hooks) {
        int loop_iter = 0, park_at = park.ticks;
        bool exhausted = tail, drained = tail;
        Cnt snapshot = cnt;
        for (;;) {
            if (my < 0 && !exhausted) {
                int idx = 0;
                if (leader()) idx = atomicAdd(Q.queue, 1);
                idx = bcast(idx);
                if (idx < Q.n_order) {
                    my = Q.order[idx]; build_world(Q.p, my); snapshot = cnt;
#ifdef REM2D_STATS
                    stats_begin(my);
#endif
                    park_at = idx >= park.late_from ? park.late_ticks : park.ticks;
                }
                else exhausted = true;
            }
            const unsigned live = __ballot_sync(0xffffffffu, my >= 0);
            hooks.sample(*this, loop_iter, live);
            ++loop_iter;
            if (!live) break;
            if (!drained) drained = __any_sync(0xffffffffu, exhausted);
            if (drained && gs < max_gs && (__popc(live) >> gs) << (gs + 1) <= 32) {
                const int old = gs;
                regroup(lane, live, max_gs, hot, my, park_at, tslot, snapshot);
                exhausted = true;
                hooks.regrouped(*this, old);
            }
            if (my >= 0) {                                            // group-uniform
#ifdef REM2D_STATS
                st_c = my;
#endif
#ifdef REM2D_POLICY
                set_policy_creature(my);
#endif
                tick();
                PHASE(PH_PARK);
                const int t = Si(S_TICKS), st = Si(S_STATUS), al = Si(S_ALIVE);    // (written before tick()'s last group barrier)
                if (!al || t >= Q.max_ticks || st) {
                    if (leader()) {
                        Q.fitness[my] = Sd(S_FIT_LO); Q.ticks[my] = t; Q.alive[my] = al; Q.status[my] = st;
                        hooks.finished(*this, my, tslot, loop_iter);
                    }
                    // a creature that outgrew a capacity of this class is re-run by the host in the next class up:
                    // its partial work must not be counted
                    if (st) cnt = snapshot;
                    my = -1;
                } else if (!tail && park.ticks > 0 && gs < park.wide_gs &&
                           (t >= park_at || (park.lead_x > 0.0f && t >= park.lead_from && B(BF_CX, 0) >= park.lead_x))) {
                    // long-lived creature: park its state; the latency-oriented tail mode (one warp per creature) finishes it.
                    // (the counter never exceeds the cap: the host hands every counted slot to a tail launch)
                    int slot = -1;
                    if (leader()) {
                        int seen = *(volatile int*)park_count;
                        while (seen < park.cap) {
                            const int prev = atomicCAS(park_count, seen, seen + 1);
                            if (prev == seen) { slot = seen; break; }
                            seen = prev;
                        }
                    }
                    slot = bcast(slot);
                    if (slot >= 0) {
                        float* dst = park_state + (size_t)(slot >> 5) * L.words * 32 + (slot & 31);
                        for (int w = sub; w < L.words; w += G) dst[w * 32] = g[w * 32];
                        __threadfence();                                 // the column is visible before the slot is published
                        gsync();
                        if (leader()) {
                            if (park.tail_trace) park.tail_trace[slot * 4] = hooks.now_us();
                            __threadfence();
                            atomicExch(&park_creature[slot], my + 1);    // 0 = allocated but not yet published
                        }
                        my = -1;
                    }
                }
                gsync();          // the leader's reads of this creature's scalars are done before the column is rebuilt
                PHASE(PH_LOOP);
            }
        }
    }
    // Packs the live creatures of the warp onto the first groups, widened to the largest gs' <= max_gs with n_live << gs' <= 32
    // (see episodes). Each creature takes its id, cold column, park threshold and park slot along. Its work so far, summed over
    // the lanes of its old group, moves to the counters of its new leader lane, so that `cnt = snapshot` after an overflow still
    // removes all of it.
    __device__ __forceinline__ void regroup(const int lane, const unsigned live, const int max_gs, float* hot, int& my, int& park_at,
                                            int& tslot, Cnt& snapshot) {
        const int n = __popc(live) >> gs;
        int ngs = gs + 1;
        while (ngs < max_gs && n << (ngs + 1) <= 32) ++ngs;
        __syncwarp();                      // hot columns and cold columns change owners: earlier accesses are done
        const unsigned leads = __ballot_sync(0xffffffffu, my >= 0 && leader());
        unsigned m = leads;
        for (int i = lane >> ngs; i > 0 && m; --i) m &= m - 1;       // the (lane >> ngs)-th live creature, in lane order
        const bool has = m != 0u;
        const int src = has ? __ffs((int)m) - 1 : lane;
        const bool new_leader = has && (lane & ((1 << ngs) - 1)) == 0;
#pragma unroll
        for (int i = 0; i < REM2D_N_COUNTERS; ++i) {
            unsigned w = my >= 0 ? cnt.c[i] - snapshot.c[i] : 0u;
            for (int o = G >> 1; o > 0; o >>= 1) w += __shfl_xor_sync(gmask, w, o);
            if (my >= 0) cnt.c[i] = snapshot.c[i];
            w = __shfl_sync(0xffffffffu, w, src);
            snapshot.c[i] = cnt.c[i];
            if (new_leader) cnt.c[i] += w;
        }
        my = __shfl_sync(0xffffffffu, my, src);
        park_at = __shfl_sync(0xffffffffu, park_at, src);
        tslot = __shfl_sync(0xffffffffu, tslot, src);
        const unsigned long long col = __shfl_sync(0xffffffffu, (unsigned long long)g, src);
        set_group(ngs, lane, hot);
        if (has) { g = (float*)col; nb = Si(S_NB); nj = nb - 1; }
        else { my = -1; tslot = -1; nb = nj = 0; }
    }
};

}  // namespace rem2d
