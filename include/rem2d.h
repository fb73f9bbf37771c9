/* rem2d.h — C-ABI of the batched REM2D evaluation library.
 *
 * Two shared libraries export exactly these symbols:
 *   gym_rem2d_b200/csrc/librem2d_cuda.so   the product: hand-written CUDA for sm_100a
 *   oracle/librem2d_oracle.so              the CPU oracle (test infrastructure only)
 *
 * What it replaces in the reference (paths under /root/reference/ModularER_2D):
 *   the per-individual pybox2d loop  REM2D_main.py:350-378 (evaluate)  ->  Modular2DEnv.py:565-653
 *   (reset/step)  ->  Box2D b2World::Step(1/50, 180, 60)  (Modular2DEnv.py:634), i.e. the SWIG
 *   surface b2World(), CreateStaticBody, CreateDynamicBody, CreateJoint, Step, body.position/.angle,
 *   joint.angle, joint.motorSpeed (call sites Modular2DEnv.py:144,226,301,572,634;
 *   simple_module.py:286-298; circular_module.py:191-202; module_utility.py:19-32).
 * The boundary sits one level above that surface: a flattened population table in, fitness/state out.
 *
 * Conventions: return 0 = OK, negative = error (see REM2D_E_*); no exceptions cross the ABI; the
 * caller owns every buffer it passes (inputs are copied during the call, outputs are written into
 * caller memory); all pointers are HOST pointers; a handle is bound to one device and is not
 * thread-safe, different handles are independent.
 */
#ifndef REM2D_H
#define REM2D_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define REM2D_ABI_VERSION 1

#define REM2D_OK 0
#define REM2D_E_INVALID (-1)   /* bad argument / call order */
#define REM2D_E_CUDA (-2)      /* CUDA runtime error (text in rem2d_last_error) */
#define REM2D_E_CAPACITY (-3)  /* creature larger than the largest compiled capacity class */
#define REM2D_E_NOMEM (-4)

#define REM2D_SHAPE_BOX 0
#define REM2D_SHAPE_CIRCLE 1

typedef struct rem2d_handle rem2d_handle;

/* Constants of the path. rem2d_default_config() fills the reference's values (file:line cited there). */
typedef struct rem2d_config {
    float dt;                  /* 1/FPS = 1/50                      Modular2DEnv.py:26,634 */
    int32_t velocity_iterations; /* 180                             Modular2DEnv.py:634 */
    int32_t position_iterations; /* 60                              Modular2DEnv.py:634 */
    float gravity_y;           /* -10, pybox2d b2World() default */
    float module_friction;     /* 0.1                               simple_module.py:289 */
    float terrain_friction;    /* 2.5                               Modular2DEnv.py:62,162 */
    double p_gain;             /* 1.9                               Modular2DEnv.py:601 */
    double wod_speed;          /* 0.04 per tick                     Modular2DEnv.py:52,107-108 */
    double env_length;         /* 100                               REM2D_main.py:350,372 */
    int32_t evaluation_steps;  /* 10000 (bonus term denominator)    REM2D_main.py:350,373 */
    int32_t continuous;        /* 1: TOI / continuous collision on (b2World default) */
    int32_t allow_sleep;       /* 1 (b2World default) */
    int32_t terminate;         /* 1: wall-of-death / x<0 termination and fitness latch per tick
                                  (Modular2DEnv.py:642-649, REM2D_main.py:370-377); 0: fixed horizon */
    int32_t device;            /* CUDA device ordinal (ignored by the oracle) */
    void* stream;              /* cudaStream_t to order work on; NULL = default stream */
    int32_t sincos_mode;       /* oracle only: 0 = portable float sin/cos (bit-identical to the CUDA build),
                                  1 = libm sinf/cosf as upstream Box2D's b2Rot::Set, 2 = portable double kernel */
    int32_t reserved;
} rem2d_config;

/* Flattened population (SoA, CSR by creature). Emitted by gym_rem2d_b200/flatten.py, which restates
 * Modular2D.create_robot (Modular2DEnv.py:517-563) and the module create()/create_joint geometry.
 * Creature c owns bodies body_off[c] .. body_off[c+1]-1 (creation order, root first) and one joint
 * per non-root body: global joint index = global body index - (c+1); joint k of a creature connects
 * local body joint_parent[k] (A) to local body k+1 (B). */
typedef struct rem2d_population {
    int32_t n_creatures;
    int32_t n_bodies;
    int32_t n_joints;                /* = n_bodies - n_creatures */
    const int32_t* body_off;         /* [n_creatures+1] */
    const uint8_t* shape;            /* [n_bodies] REM2D_SHAPE_* */
    const float* hx;                 /* [n_bodies] half width, or radius for circles */
    const float* hy;                 /* [n_bodies] half height (0 for circles) */
    const float* x0;                 /* [n_bodies] initial pose, already float32 as Box2D stores it */
    const float* y0;
    const float* a0;
    const int16_t* joint_parent;     /* [n_joints] local index of body A */
    const float* anchor_a;           /* [n_joints*2] localAnchorA */
    const float* anchor_b;           /* [n_joints*2] localAnchorB */
    const float* lower;              /* [n_joints] lowerAngle  (-pi/2) */
    const float* upper;              /* [n_joints] upperAngle  (+pi/2) */
    const float* max_torque;         /* [n_joints] maxMotorTorque (50) */
    const double* ctrl;              /* [n_bodies*5] amplitude, phase, frequency, offset, i_state
                                        (Controller/m_controller.py:5-21; the root's is never used) */
} rem2d_population;

/* Snapshot of the simulation state for parity tests. Every pointer may be NULL (skipped). */
typedef struct rem2d_state_view {
    float* pose;            /* [n_bodies*3] x, y, angle   (body.position / body.angle) */
    float* vel;             /* [n_bodies*3] vx, vy, omega */
    float* joint_impulse;   /* [n_joints*4] accumulated impulse x, y, z(limit), motor */
    int32_t* limit_state;   /* [n_joints]   0 inactive, 1 at lower, 2 at upper */
    float* motor_speed;     /* [n_joints]   last joint.motorSpeed written by the P-controller */
    int32_t* alive;         /* [n_creatures] 1 while the episode runs */
    int32_t* ticks;         /* [n_creatures] ticks simulated so far */
    int32_t* awake;         /* [n_creatures] Box2D island awake flag */
    double* wod;            /* [n_creatures] wall-of-death position */
    int32_t* n_contacts;    /* [n_creatures] number of contact objects (fat-AABB overlaps) */
    int32_t* n_touching;    /* [n_creatures] of which touching (manifold pointCount > 0) */
    int32_t* touching_pairs;/* [n_creatures*max_pairs*2] (local body, edge) of touching contacts,
                               ascending (body, edge); unused slots = -1 */
    float* touching_impulse;/* [n_creatures*max_pairs*4] normalImpulse p0,p1, tangentImpulse p0,p1 */
    int32_t max_pairs;
    int32_t reserved;
} rem2d_state_view;

/* Work counters (sums over all creatures since rem2d_reset), used for the roofline's algorithmic FLOPs. */
#define REM2D_N_COUNTERS 12
#define REM2D_CNT_TICKS 0          /* creature-ticks simulated */
#define REM2D_CNT_BODY_TICKS 1     /* sum of awake bodies over ticks */
#define REM2D_CNT_JOINT_VSOLVES 2  /* revolute velocity solves */
#define REM2D_CNT_P1_VSOLVES 3     /* 1-point manifold velocity solves */
#define REM2D_CNT_M2_VSOLVES 4     /* 2-point (block) manifold velocity solves */
#define REM2D_CNT_JOINT_PSOLVES 5  /* revolute position solves */
#define REM2D_CNT_POINT_PSOLVES 6  /* contact point position solves */
#define REM2D_CNT_NARROW 7         /* narrow-phase evaluations (body x edge) */
#define REM2D_CNT_TOI_CALLS 8      /* time-of-impact queries */
#define REM2D_CNT_TOI_EVENTS 9     /* TOI sub-steps taken */
#define REM2D_CNT_GJK_ITERS 10     /* GJK support iterations */
#define REM2D_CNT_TOI_ROOT_ITERS 11/* TOI root finder evaluations */

void rem2d_default_config(rem2d_config* cfg);
int rem2d_abi_version(void);
/* "cuda-sm_100a" or "oracle-c" */
const char* rem2d_backend(void);

int rem2d_create(const rem2d_config* cfg, rem2d_handle** out);
int rem2d_destroy(rem2d_handle* h);
/* NULL handle: error of the last failed rem2d_create on this thread */
const char* rem2d_last_error(rem2d_handle* h);

/* 200-vertex height field, x_i = i*step (Modular2DEnv.py:188-310; same for every creature because
 * evaluate() reseeds with 4 before each reset, REM2D_main.py:358). y is float64 as the reference
 * computes it; the library rounds to float32 where Box2D would. */
int rem2d_set_terrain(rem2d_handle* h, const double* y, int32_t n_vertices, double step);

/* Copy the population in and build the worlds (replaces Modular2D.reset's world construction). */
int rem2d_upload(rem2d_handle* h, const rem2d_population* pop);
/* Back to tick 0 of the uploaded population (new b2World, wod = 0, fitness = 0). */
int rem2d_reset(rem2d_handle* h);
/* Advance every alive creature by up to n_ticks ticks of Modular2D.step (controllers, P-control,
 * world.Step, reward/WOD/termination, fitness latch). */
int rem2d_step(rem2d_handle* h, int32_t n_ticks);
int rem2d_read_state(rem2d_handle* h, rem2d_state_view* out);
/* fitness as evaluate() would return it so far (REM2D_main.py:361-378) */
int rem2d_fitness(rem2d_handle* h, double* out_n_creatures);
int rem2d_get_counters(rem2d_handle* h, uint64_t* out_REM2D_N_COUNTERS);
/* Whole episodes for the uploaded population, from tick 0 to termination (or max_ticks), on the persistent
 * episode kernel; results via rem2d_fitness / rem2d_ticks. Per-creature stepping state is not kept: call
 * rem2d_reset before using rem2d_step / rem2d_read_state again. */
int rem2d_run_episodes(rem2d_handle* h, int32_t max_ticks);
int rem2d_ticks(rem2d_handle* h, int32_t* out_n_creatures);
/* Batched evaluate(): upload + run_episodes(max_ticks) + fitness; ticks_out may be NULL. This is the
 * call toolbox.map(toolbox.evaluate, population) (REM2D_main.py:267,291) turns into. */
int rem2d_evaluate(rem2d_handle* h, const rem2d_population* pop, int32_t max_ticks,
                   double* fitness_out, int32_t* ticks_out);
/* Device time of the kernels launched by the last rem2d_step / rem2d_evaluate, in milliseconds,
 * measured with CUDA events on cfg.stream (0 for the oracle: use wall clock). */
float rem2d_last_step_ms(rem2d_handle* h);
/* CUDA build only: measured non-fused FP32 (FMUL/FADD) issue peak of the device in GFLOP/s — the roofline
 * denominator of the step kernel, which is built without FMA contraction for bit parity with Box2D. */
int rem2d_measure_fp32_peak(rem2d_handle* h, double* gflops);
/* Number of kernels this library launched since rem2d_create. */
int64_t rem2d_launch_count(rem2d_handle* h);
/* Tuning / diagnostic option by name (execution strategy only, never results): "warp_mode_max", "park_ticks", "park_cap",
 * "smem_budget_kb", "group_shift", "class_gs_<k>", "tail_group_shift", "overflow_wave", "image", "trace" (DESIGN.md section 4).
 * Unknown names return REM2D_E_INVALID. The oracle accepts the same names and ignores them. */
int rem2d_set_option(rem2d_handle* h, const char* name, double value);
/* Optional scheduling hint for the NEXT rem2d_upload / rem2d_evaluate: expected lifetime of every creature in ticks (an EA passes
 * the lifetime of the parent). Creatures expected to outlive the wall of death's arrival at the start pad (>= 130 ticks) are
 * started first, so that the sequential ticks of the long-lived creatures - which bound the run time of a generation - overlap
 * the bulk instead of following it (the multiprocessing.Pool of REM2D_main.py:256-262 has the same problem with its static chunks).
 * Never changes results. n must equal the population size of the next upload, otherwise the hint is dropped; NULL clears it. */
int rem2d_set_priority(rem2d_handle* h, const float* expected_ticks, int32_t n);
/* Cheap per-creature read-out for step-wise drivers (what Modular2D.step needs to form its reward, Modular2DEnv.py:642-649):
 * root x (= robot.components[0].position[0]), wall-of-death position, alive flag. Any pointer may be NULL. Valid after
 * rem2d_upload / rem2d_reset / rem2d_step. */
int rem2d_read_roots(rem2d_handle* h, float* root_x, double* wod, int32_t* alive);

#ifdef __cplusplus
}
#endif
#endif /* REM2D_H */
