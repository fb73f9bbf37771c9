/* rem2d_policy.h — per-joint neural feedback controllers: an extension of the C-ABI in rem2d.h.
 *
 * Exported by gym_rem2d_b200/csrc/librem2d_cuda.so (both precisions) and by the test oracle with the policy
 * (tests/oracle_policy/librem2d_oracle_policy.so: the CPU oracle with the other extension headers, unchanged, plus the policy
 * tick below).
 * The plain oracle (oracle/librem2d_oracle.so) exports rem2d.h only.
 *
 * A population uploaded with a policy has one small network per joint; the weights differ per joint and come from the caller.
 * Every tick, for every joint j of a live creature:
 *  1. Oscillator. The sine controller advances exactly as in a plain tick: i_state += frequency, then
 *     s = amplitude * sin(i_state + phase) + offset (float64, the portable sin).
 *  2. Features, eight float64 values read from the state at the start of the tick, i.e. the end-of-tick state that
 *     rem2d_read_observations reports (identical values):
 *       x0 = s
 *       x1 = (double)joint_angle[j]      the currentAngle the P-controller uses
 *       x2 = (double)joint_speed[j]      omega_B - omega_A, float32
 *       x3 = ground[B], x4 = ground[A]   0.0 or 1.0; A is joint_parent[j], B is j+1 (local to the creature)
 *       x5 = (double)root angle, x6 = (double)root vx, x7 = (double)root vy
 *  3. Network, H hidden units (1 <= H <= REM2D_POLICY_MAX_HIDDEN). For each hidden unit k:
 *       acc = b1[k]; acc = acc + W1[k][i] * x_i for i = 0..7, in that order; h_k = acc / (1.0 + fabs(acc))   (softsign)
 *     then u = b2; u = u + w2[k] * h_k for k = 0..H-1. Separate multiplies and adds (no fused multiply-add in the exact build).
 *  4. Target: target = s + u. From here the tick is exactly rem2d_step_targets' tick: speed = (target - (double)currentAngle)
 *     * p_gain written as float32, both bodies woken; Collide, Solve, SolveTOI, the termination rule, the fitness latch and the
 *     work counters are unchanged.
 * Softsign rather than tanh: it is exact IEEE float64 arithmetic everywhere, with no transcendental function to match.
 * target = s + u: with all weights zero the policy is the open-loop controller (u = +0.0), so an evolutionary search can start
 * from existing genomes and evolve the feedback; a caller who wants a purely reactive controller zeroes amplitude and offset.
 *
 * Weight layout: P = 10 * H + 1 float64 per joint: W1 (H x 8, row-major), b1 (H), w2 (H), b2. Joints in table order (global
 * joint index = global body index - (c+1), as in rem2d.h): joint j's block starts at weights[j * P].
 *
 * rem2d_set_policy(h, weights, n_joints, n_hidden):
 *   The policy applies to every later upload (rem2d_upload, rem2d_evaluate) until it is changed; the upload takes a snapshot,
 *   so a later rem2d_set_policy never changes a population that is already uploaded. The weights are copied during the call.
 *   weights == NULL clears the policy. n_hidden outside 1..REM2D_POLICY_MAX_HIDDEN, n_joints < 0 or a non-finite weight
 *   return REM2D_E_INVALID and keep the previous policy. While a policy is set, an upload whose population has another
 *   n_joints returns REM2D_E_INVALID before anything changes.
 *   For a population uploaded with a policy, rem2d_run_episodes, rem2d_evaluate and rem2d_step run policy ticks and
 *   rem2d_reset keeps the policy; rem2d_step_targets still overrides the controller as rem2d_control.h states (the policy is
 *   not evaluated and the oscillators are frozen). Episode statistics (rem2d_stats.h) compose with the policy, with
 *   unchanged definitions.
 * Bit-identical between the CUDA library (exact precision) and the oracle.
 */
#ifndef REM2D_POLICY_H
#define REM2D_POLICY_H

#include "rem2d.h"

#ifdef __cplusplus
extern "C" {
#endif

#define REM2D_POLICY_FEATURES 8
#define REM2D_POLICY_MAX_HIDDEN 16

int rem2d_set_policy(rem2d_handle* h, const double* weights, int32_t n_joints, int32_t n_hidden);

#ifdef __cplusplus
}
#endif
#endif /* REM2D_POLICY_H */
