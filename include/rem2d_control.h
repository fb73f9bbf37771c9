/* rem2d_control.h — closed-loop control of stepping runs: an extension of the C-ABI in rem2d.h.
 *
 * Exported by gym_rem2d_b200/csrc/librem2d_cuda.so (both precisions) and by the test oracle with the extension headers
 * (tests/oracle_ext/librem2d_oracle_ext.so: the CPU oracle, unchanged, plus the two functions below).
 * The plain oracle (oracle/librem2d_oracle.so) exports rem2d.h only.
 *
 * rem2d_step_targets(h, targets, n_ticks):
 *   targets is a host array of n_joints float64, one per joint in table order (global joint index = global body index - (c+1),
 *   as in rem2d.h). Each value is a target angle in radians: the same quantity as the controller output the sine controllers
 *   compute (Modular2DEnv.py:631-632).
 *   Every alive creature advances up to n_ticks ticks exactly as rem2d_step advances it, with one difference in the controller
 *   stage: the target of joint j is targets[j], held for all n_ticks. Everything else is unchanged:
 *     speed = (target - (double)currentAngle) * p_gain, written as float32 to the joint's motor speed;
 *     both bodies of the joint are woken;
 *     the wall of death, Collide / Solve / SolveTOI, reward and termination, the fitness latch and the work counters.
 *   The sine controllers are not advanced: i_state is unchanged, so a later rem2d_step continues every oscillator from where its
 *   last plain tick left it.
 *   A non-finite target, a NULL pointer, n_ticks < 0, no uploaded population, or per-creature state consumed by
 *   rem2d_run_episodes / rem2d_evaluate returns REM2D_E_INVALID; in every such case nothing is stepped. Dead creatures are not
 *   stepped and their targets are ignored. rem2d_last_step_ms reports the device time of the call, the copy of the targets
 *   included.
 *
 * rem2d_read_observations(h, out) writes the end-of-tick state. Any pointer of out may be NULL (skipped). Valid wherever
 * rem2d_read_roots is valid. Every value equals what rem2d_read_state reports for the same state:
 *   joint_angle  the currentAngle the next tick's P-controller uses: pose_a[B] - pose_a[A] - 0.0f (float32), where A is
 *                joint_parent[k] and B is k+1, both local to the creature;
 *   joint_speed  omega_B - omega_A (float32);
 *   root         x, y, angle, vx, vy, omega of body 0;
 *   ground       1 if the body has a touching terrain contact, else 0 (the definition behind ground_ticks in rem2d_stats.h).
 * Bit-identical between the CUDA library (exact precision) and the oracle.
 */
#ifndef REM2D_CONTROL_H
#define REM2D_CONTROL_H

#include "rem2d.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rem2d_observation {   /* any pointer may be NULL (skipped) */
    float* joint_angle;    /* [n_joints]       */
    float* joint_speed;    /* [n_joints]       */
    float* root;           /* [n_creatures*6]  */
    int32_t* ground;       /* [n_bodies]       */
} rem2d_observation;

int rem2d_step_targets(rem2d_handle* h, const double* targets, int32_t n_ticks);
int rem2d_read_observations(rem2d_handle* h, rem2d_observation* out);

#ifdef __cplusplus
}
#endif
#endif /* REM2D_CONTROL_H */
