/* rem2d_stats.h — episode statistics of whole-episode runs: an extension of the C-ABI in rem2d.h.
 *
 * Exported by gym_rem2d_b200/csrc/librem2d_cuda.so (both precisions) and by the test oracle with the extension headers
 * (tests/oracle_ext/librem2d_oracle_ext.so: the CPU oracle, unchanged, plus the accumulation below after every tick).
 * The plain oracle (oracle/librem2d_oracle.so) exports rem2d.h only.
 *
 * Every value is defined by the state at the end of a tick (after Collide, Solve, SolveTOI and the termination rule) as
 * rem2d_read_state / rem2d_read_roots report it, over the ticks the creature ran, so a stepping run can recompute it:
 *   end_reason      how the episode ended (the comparisons of the termination rule, in this precedence): REM2D_END_ORIGIN
 *                   root x < 0, REM2D_END_WALL wall of death > root x, REM2D_END_GOAL reward > env_length, REM2D_END_STEPS
 *                   evaluation_steps reached; REM2D_END_RUNNING alive when the run stopped (always with terminate = 0);
 *   max_x           largest root x (-inf if no tick ran; NaN is never taken);
 *   joint_work      running float64 sum, every tick, joints in order: |motor impulse * (omega_B - omega_A)|;
 *   airborne_ticks  ticks at whose end no body of the creature has a touching terrain contact;
 *   ground_ticks    per body (body order of the uploaded table): ticks at whose end the body has a touching terrain contact.
 * Bit-identical between the CUDA library and the oracle, whatever the execution strategy.
 */
#ifndef REM2D_STATS_H
#define REM2D_STATS_H

#include "rem2d.h"

#ifdef __cplusplus
extern "C" {
#endif

#define REM2D_END_RUNNING 0
#define REM2D_END_ORIGIN 1
#define REM2D_END_WALL 2
#define REM2D_END_GOAL 3
#define REM2D_END_STEPS 4
typedef struct rem2d_episode_stats {   /* any pointer may be NULL (skipped) */
    int32_t* end_reason;     /* [n_creatures] */
    float* max_x;            /* [n_creatures] */
    double* joint_work;      /* [n_creatures] */
    int32_t* airborne_ticks; /* [n_creatures] */
    int32_t* ground_ticks;   /* [n_bodies]    */
} rem2d_episode_stats;
/* Record episode statistics in whole-episode runs of every later upload (rem2d_upload / rem2d_evaluate) until changed.
 * Never changes results. */
int rem2d_set_stats(rem2d_handle* h, int32_t on);
/* Statistics of the last rem2d_run_episodes / rem2d_evaluate. REM2D_E_INVALID if that run's upload was made with statistics
 * off, if no such run happened since the upload, or after rem2d_reset / rem2d_step (the stepping path does not record them). */
int rem2d_read_stats(rem2d_handle* h, rem2d_episode_stats* out);

#ifdef __cplusplus
}
#endif
#endif /* REM2D_STATS_H */
