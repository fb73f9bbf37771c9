/* rem2d_oracle_policy.c — TEST INFRASTRUCTURE: the CPU oracle with the extension headers (tests/oracle_ext, compiled here
 * unchanged) and the per-joint feedback policy of include/rem2d_policy.h.
 *
 * tests/oracle_ext/rem2d_oracle_ext.c is included as it is. The five entries whose behaviour the policy changes (rem2d_upload,
 * rem2d_step, rem2d_run_episodes, rem2d_evaluate, rem2d_destroy) are first declared with assembler names ext_*, so the
 * included definitions are emitted under those (hidden) names and stay callable from here as rem2d_upload etc.; this unit exports its
 * own versions under the public names (policy_* in C, rem2d_* in the library). Everything else, the statistics, joint targets,
 * observations and test-only sine outputs included, is the oracle extension's.
 *
 * A population uploaded with a policy runs tick_policy: the features of every joint from the state at the start of the tick,
 * the sine controllers advanced as tick() does, the network, and then tick_target's body with target = s + u. The stepping
 * path and the whole-episode loop (recording the statistics when they are on) run it through the extension's run_worlds; the
 * call contract is the CUDA library's. Build: make -C tests/oracle_policy. Used by tests/oracle_policy/oracle_policy.py. */
#include <stdint.h>
struct rem2d_handle;
struct rem2d_population;
int rem2d_upload(struct rem2d_handle* h, const struct rem2d_population* pop) __asm__("ext_upload") __attribute__((visibility("hidden")));
int rem2d_step(struct rem2d_handle* h, int32_t n_ticks) __asm__("ext_step") __attribute__((visibility("hidden")));
int rem2d_run_episodes(struct rem2d_handle* h, int32_t max_ticks) __asm__("ext_run_episodes") __attribute__((visibility("hidden")));
int rem2d_evaluate(struct rem2d_handle* h, const struct rem2d_population* pop, int32_t max_ticks, double* fitness_out,
                   int32_t* ticks_out) __asm__("ext_evaluate") __attribute__((visibility("hidden")));
int rem2d_destroy(struct rem2d_handle* h) __asm__("ext_destroy") __attribute__((visibility("hidden")));

#include "../oracle_ext/rem2d_oracle_ext.c"
#include "../../include/rem2d_policy.h"

/* rem2d_set_policy per handle, and the snapshot of the current upload: {H, weights...} (H first, so that the snapshot alone
 * is what the ticks need: it travels as the Job's targets pointer) */
typedef struct PolEntry {
    rem2d_handle* h;
    double* w; int on, nj, hidden;
    double* up;                        /* NULL: the current upload has no policy */
    struct PolEntry* next;
} PolEntry;
static PolEntry* g_pol = NULL;

static PolEntry* pol_of(rem2d_handle* h) {
    if (!h) return NULL;
    pthread_mutex_lock(&g_entries_lock);
    PolEntry* e = g_pol;
    while (e && e->h != h) e = e->next;
    if (!e && (e = (PolEntry*)calloc(1, sizeof(PolEntry)))) { e->h = h; e->next = g_pol; g_pol = e; }
    pthread_mutex_unlock(&g_entries_lock);
    return e;
}

/* tick() with the controller output of joint k computed by its network (include/rem2d_policy.h) from the state at the start of
 * the tick; `wt` holds the weights of the creature's first joint, H the hidden units. The sine controllers advance as in tick(). */
static void tick_policy(rem2d_handle* h, World* w, const double* wt, int H, Counters* cnt) {
    if (!w->alive) return;
    uint64_t ground = 0;
    for (int i = 0; i < w->nc; ++i)
        if (w->contacts[i].flags & CF_TOUCHING) ground |= 1ull << w->contacts[i].body;
    const Body* r = &w->bodies[0];
    const double root_a = (double)r->sweep.a, root_vx = (double)r->v.x, root_vy = (double)r->v.y;
    for (int b = 0; b < w->nb; ++b) {
        Ctrl* c = &w->ctrl[b];
        c->phase += 0.0;
        c->i_state += c->frequency;
        c->output = c->amplitude * sin_f64(c->i_state + c->phase) + c->offset;
    }
    const int P = 10 * H + 1;
    double target[64];
    for (int k = 0; k < w->nj; ++k) {
        const Joint* j = &w->joints[k];
        const Body *A = &w->bodies[j->bodyA], *B = &w->bodies[j->bodyB];
        const double s = w->ctrl[k + 1].output;
        const float angle = B->sweep.a - A->sweep.a - j->referenceAngle, speed = B->w - A->w;
        const double x[REM2D_POLICY_FEATURES] = {s, (double)angle, (double)speed, (double)((ground >> j->bodyB) & 1ull),
                                                 (double)((ground >> j->bodyA) & 1ull), root_a, root_vx, root_vy};
        const double* W = wt + (size_t)k * P;
        double u = W[10 * H];
        for (int q = 0; q < H; ++q) {
            double acc = W[8 * H + q];
            for (int i = 0; i < REM2D_POLICY_FEATURES; ++i) acc = acc + W[8 * q + i] * x[i];
            u = u + W[9 * H + q] * (acc / (1.0 + fabs(acc)));
        }
        target[k] = s + u;
    }
    tick_target(h, w, target, cnt);
}
/* creature-ticks of run_worlds; job->targets is the upload's snapshot {H, weights...} */
static void tick_policied(Job* job, World* w, int c) {
    const int H = (int)job->targets[0];
    tick_policy(job->h, w, job->targets + 1 + (size_t)(job->h->pop.body_off[c] - c) * (10 * H + 1), H, &job->cnt);
}
static void tick_policied_recorded(Job* job, World* w, int c) { tick_policied(job, w, c); accumulate(job->h, job->e, w, c); }

/* run_whole of the extension with policy ticks */
static int run_whole_policy(rem2d_handle* h, Entry* s, const double* up, int32_t n_ticks) {
    s->consumed = 1;
    if (n_ticks < 0) return REM2D_E_INVALID;
    if (!s->upload_on) return run_worlds(h, s, up, tick_policied, n_ticks);
    const int n = h->pop.n_creatures, nb = h->pop.n_bodies;
    free_arrays(s);
    s->n = n; s->nb = nb;
    s->end_reason = (int32_t*)calloc((size_t)(n > 0 ? n : 1), sizeof(int32_t));
    s->airborne_ticks = (int32_t*)calloc((size_t)(n > 0 ? n : 1), sizeof(int32_t));
    s->ground_ticks = (int32_t*)calloc((size_t)(nb > 0 ? nb : 1), sizeof(int32_t));
    s->max_x = (float*)malloc(sizeof(float) * (size_t)(n > 0 ? n : 1));
    s->joint_work = (double*)calloc((size_t)(n > 0 ? n : 1), sizeof(double));
    if (!s->end_reason || !s->airborne_ticks || !s->ground_ticks || !s->max_x || !s->joint_work) { free_arrays(s); return REM2D_E_NOMEM; }
    for (int c = 0; c < n; ++c) s->max_x[c] = -INFINITY;
    int rc = run_worlds(h, s, up, tick_policied_recorded, n_ticks);
    s->valid = rc == REM2D_OK;
    return rc;
}

int rem2d_set_policy(rem2d_handle* h, const double* weights, int32_t n_joints, int32_t n_hidden) {
    PolEntry* e = pol_of(h);
    if (!e) return REM2D_E_INVALID;
    if (!weights) { free(e->w); e->w = NULL; e->on = 0; e->nj = e->hidden = 0; return REM2D_OK; }
    if (n_hidden < 1 || n_hidden > REM2D_POLICY_MAX_HIDDEN || n_joints < 0) {
        snprintf(h->err, sizeof(h->err), "set_policy: need 1 <= n_hidden <= 16 and n_joints >= 0");
        return REM2D_E_INVALID;
    }
    const size_t n = (size_t)n_joints * (10 * n_hidden + 1);
    for (size_t i = 0; i < n; ++i)
        if (!isfinite(weights[i])) { snprintf(h->err, sizeof(h->err), "set_policy: weight %zu is not finite", i); return REM2D_E_INVALID; }
    double* w = (double*)malloc(sizeof(double) * (n ? n : 1));
    if (!w) return REM2D_E_NOMEM;
    memcpy(w, weights, sizeof(double) * n);
    free(e->w);
    e->w = w; e->on = 1; e->nj = n_joints; e->hidden = n_hidden;
    return REM2D_OK;
}

int policy_upload(rem2d_handle* h, const rem2d_population* pop) __asm__("rem2d_upload");
int policy_upload(rem2d_handle* h, const rem2d_population* pop) {
    PolEntry* e = pol_of(h);
    if (e && pop && e->on && pop->n_joints != e->nj) {
        snprintf(h->err, sizeof(h->err), "upload: the policy set with rem2d_set_policy has %d joints, the population %d", e->nj, pop->n_joints);
        return REM2D_E_INVALID;
    }
    if (e) {
        free(e->up);
        e->up = NULL;
        if (e->on) {
            const size_t n = (size_t)e->nj * (10 * e->hidden + 1);
            if (!(e->up = (double*)malloc(sizeof(double) * (n + 1)))) return REM2D_E_NOMEM;
            e->up[0] = (double)e->hidden;
            memcpy(e->up + 1, e->w, sizeof(double) * n);
        }
    }
    return rem2d_upload(h, pop);                     /* the extension's */
}
int policy_step(rem2d_handle* h, int32_t n_ticks) __asm__("rem2d_step");
int policy_step(rem2d_handle* h, int32_t n_ticks) {
    PolEntry* p = pol_of(h);
    if (!p || !p->up) return rem2d_step(h, n_ticks);
    Entry* e = entry_of(h);
    if (refuse_step(h, e, n_ticks, "step")) return REM2D_E_INVALID;
    e->valid = 0;                        /* the stepping path records no statistics */
    return run_worlds(h, e, p->up, tick_policied, n_ticks);
}
int policy_run_episodes(rem2d_handle* h, int32_t max_ticks) __asm__("rem2d_run_episodes");
int policy_run_episodes(rem2d_handle* h, int32_t max_ticks) {
    PolEntry* p = pol_of(h);
    if (!p || !p->up) return rem2d_run_episodes(h, max_ticks);
    int rc = rem2d_reset(h);
    return rc ? rc : run_whole_policy(h, entry_of(h), p->up, max_ticks);
}
int policy_evaluate(rem2d_handle* h, const rem2d_population* pop, int32_t max_ticks, double* fitness_out, int32_t* ticks_out)
    __asm__("rem2d_evaluate");
int policy_evaluate(rem2d_handle* h, const rem2d_population* pop, int32_t max_ticks, double* fitness_out, int32_t* ticks_out) {
    int rc = policy_upload(h, pop);
    if (rc) return rc;
    PolEntry* p = pol_of(h);
    rc = p && p->up ? run_whole_policy(h, entry_of(h), p->up, max_ticks) : run_whole(h, entry_of(h), max_ticks);
    if (!rc && fitness_out) rc = rem2d_fitness(h, fitness_out);
    if (!rc && ticks_out) rc = rem2d_ticks(h, ticks_out);
    return rc;
}
int policy_destroy(rem2d_handle* h) __asm__("rem2d_destroy");
int policy_destroy(rem2d_handle* h) {
    if (!h) return REM2D_E_INVALID;
    pthread_mutex_lock(&g_entries_lock);
    for (PolEntry** p = &g_pol; *p; p = &(*p)->next)
        if ((*p)->h == h) { PolEntry* e = *p; *p = e->next; free(e->w); free(e->up); free(e); break; }
    pthread_mutex_unlock(&g_entries_lock);
    return rem2d_destroy(h);                         /* the extension's */
}
