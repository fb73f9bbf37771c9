/* rem2d_oracle_control.c — TEST INFRASTRUCTURE: the CPU oracle with the joint-target stepping and the observations of
 * include/rem2d_control.h.
 *
 * The oracle (oracle/rem2d_oracle.c) is compiled here unchanged; this unit adds rem2d_step_targets, which runs the oracle's
 * world_step with tick()'s P-control and episode bookkeeping but takes the controller output from the targets (the sine
 * controllers are not advanced), and rem2d_read_observations. Everything else is the oracle's code path. Like the CUDA library,
 * it refuses to step or observe after rem2d_run_episodes / rem2d_evaluate until rem2d_upload / rem2d_reset: that flag lives in a
 * side table, because the oracle's handle is its own. Also exports rem2d_control_sine_outputs (test only). Build:
 * make -C tests/control_oracle. Used by the closed-loop tests. */
#define rem2d_destroy oracle_destroy
#define rem2d_upload oracle_upload
#define rem2d_reset oracle_reset
#define rem2d_step oracle_step
#define rem2d_run_episodes oracle_run_episodes
#define rem2d_evaluate oracle_evaluate
#include "../../oracle/rem2d_oracle.c"
#undef rem2d_destroy
#undef rem2d_upload
#undef rem2d_reset
#undef rem2d_step
#undef rem2d_run_episodes
#undef rem2d_evaluate
#include "../../include/rem2d_control.h"

typedef struct ControlEntry {
    rem2d_handle* h;
    int consumed;             /* state consumed by a whole-episode run (the CUDA library's rule) */
    struct ControlEntry* next;
} ControlEntry;
static ControlEntry* g_entries = NULL;
static pthread_mutex_t g_entries_lock = PTHREAD_MUTEX_INITIALIZER;

static ControlEntry* entry_of(rem2d_handle* h) {
    pthread_mutex_lock(&g_entries_lock);
    ControlEntry* e = g_entries;
    while (e && e->h != h) e = e->next;
    if (!e && (e = (ControlEntry*)calloc(1, sizeof(ControlEntry)))) { e->h = h; e->next = g_entries; g_entries = e; }
    pthread_mutex_unlock(&g_entries_lock);
    return e;
}
static void set_consumed(rem2d_handle* h, int v) {
    ControlEntry* e = h ? entry_of(h) : NULL;
    if (e) e->consumed = v;
}

/* tick() with the controller output of joint k taken from t[k]: no controller update, the rest as tick() does it */
static void tick_target(rem2d_handle* h, World* w, const double* t, Counters* cnt) {
    if (!w->alive) return;
    w->wod += h->cfg.wod_speed;
    for (int k = 0; k < w->nj; ++k) {
        Joint* j = &w->joints[k];
        float currentAngle = w->bodies[j->bodyB].sweep.a - w->bodies[j->bodyA].sweep.a - j->referenceAngle;
        double angleDifference = t[k] - (double)currentAngle;
        double speed = angleDifference * h->cfg.p_gain;
        body_set_awake(&w->bodies[j->bodyA], 1);
        body_set_awake(&w->bodies[j->bodyB], 1);
        j->motorSpeed = (float)speed;
    }
    world_step(h, w, cnt);
    cnt->c[REM2D_CNT_TICKS]++;
    int i = w->ticks;
    w->ticks++;
    if (h->cfg.terminate) {
        double reward = (double)w->bodies[0].xf.p.x;
        if (w->bodies[0].xf.p.x < 0.0f) reward = -100.0;
        if (w->wod > (double)w->bodies[0].xf.p.x) reward = -100.0;
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

/* rem2d_step of the oracle (same dynamic schedule over creatures, same counters) with tick_target */
typedef struct { rem2d_handle* h; const double* targets; int n_ticks; int* next; Counters cnt; } TargetJob;
static void* target_worker(void* arg) {
    TargetJob* job = (TargetJob*)arg;
    rem2d_handle* h = job->h;
    const int chunk = 8;
    for (;;) {
        int c0 = __atomic_fetch_add(job->next, chunk, __ATOMIC_RELAXED);
        if (c0 >= h->n_worlds) break;
        int c1 = c0 + chunk < h->n_worlds ? c0 + chunk : h->n_worlds;
        for (int c = c0; c < c1; ++c) {
            World* w = &h->worlds[c];
            const double* t = job->targets + (h->pop.body_off[c] - c);
            for (int k = 0; k < job->n_ticks && w->alive; ++k) tick_target(h, w, t, &job->cnt);
        }
    }
    return NULL;
}

int rem2d_step_targets(rem2d_handle* h, const double* targets, int32_t n_ticks) {
    if (!h) return REM2D_E_INVALID;
    ControlEntry* e = entry_of(h);
    if (!targets || n_ticks < 0 || !h->have_pop || !e || e->consumed) {
        snprintf(h->err, sizeof(h->err), "step_targets: NULL targets / negative tick count / no population / state consumed by rem2d_run_episodes");
        return REM2D_E_INVALID;
    }
    for (int j = 0; j < h->pop.n_joints; ++j)
        if (!isfinite(targets[j])) { snprintf(h->err, sizeof(h->err), "step_targets: target %d is not finite", j); return REM2D_E_INVALID; }
    g_sincos_mode = h->cfg.sincos_mode;
    int nt = h->threads > 0 ? h->threads : 1;
    if (nt > 256) nt = 256;
    int next = 0;
    TargetJob* jobs = (TargetJob*)calloc((size_t)nt, sizeof(TargetJob));
    pthread_t* tids = (pthread_t*)calloc((size_t)nt, sizeof(pthread_t));
    for (int i = 0; i < nt; ++i) { jobs[i].h = h; jobs[i].targets = targets; jobs[i].n_ticks = n_ticks; jobs[i].next = &next; }
    for (int i = 1; i < nt; ++i) pthread_create(&tids[i], NULL, target_worker, &jobs[i]);
    target_worker(&jobs[0]);
    for (int i = 1; i < nt; ++i) pthread_join(tids[i], NULL);
    for (int i = 0; i < nt; ++i)
        for (int k = 0; k < REM2D_N_COUNTERS; ++k) h->counters[k] += jobs[i].cnt.c[k];
    free(jobs); free(tids);
    for (int c = 0; c < h->n_worlds; ++c)
        if (h->worlds[c].overflow) { snprintf(h->err, sizeof(h->err), "step: island scratch overflow in creature %d", c); return REM2D_E_CAPACITY; }
    return REM2D_OK;
}

int rem2d_read_observations(rem2d_handle* h, rem2d_observation* out) {
    if (!h || !out) return REM2D_E_INVALID;
    ControlEntry* e = entry_of(h);
    if (!h->have_pop || !e || e->consumed) {
        snprintf(h->err, sizeof(h->err), "read_observations: no population / state consumed by rem2d_run_episodes");
        return REM2D_E_INVALID;
    }
    const rem2d_population* p = &h->pop;
    for (int c = 0; c < h->n_worlds; ++c) {
        const World* w = &h->worlds[c];
        const int b0 = p->body_off[c], j0 = b0 - c;
        for (int k = 0; k < w->nj; ++k) {
            const Joint* j = &w->joints[k];
            const Body *A = &w->bodies[j->bodyA], *B = &w->bodies[j->bodyB];
            if (out->joint_angle) out->joint_angle[j0 + k] = B->sweep.a - A->sweep.a - j->referenceAngle;
            if (out->joint_speed) out->joint_speed[j0 + k] = B->w - A->w;
        }
        if (out->root) {
            const Body* r = &w->bodies[0];
            float* o = &out->root[(size_t)c * 6];
            o[0] = r->xf.p.x; o[1] = r->xf.p.y; o[2] = r->sweep.a; o[3] = r->v.x; o[4] = r->v.y; o[5] = r->w;
        }
        if (out->ground) {
            uint64_t m = 0;
            for (int i = 0; i < w->nc; ++i)
                if (w->contacts[i].flags & CF_TOUCHING) m |= 1ull << w->contacts[i].body;
            for (int b = 0; b < w->nb; ++b) out->ground[b0 + b] = (int32_t)((m >> b) & 1ull);
        }
    }
    return REM2D_OK;
}

/* TEST ONLY: the next T outputs of every joint's sine controller from the current state of the worlds, out[t * n_joints + j],
 * computed as tick() computes them (phase += 0.0, i_state += frequency, amplitude * sin_f64(i_state + phase) + offset) on a copy:
 * the worlds are not changed. Feeding out[t] to the t-th one-tick rem2d_step_targets reproduces T plain ticks. */
int rem2d_control_sine_outputs(rem2d_handle* h, int32_t T, double* out) {
    if (!h || !out || T < 0 || !h->have_pop) return REM2D_E_INVALID;
    g_sincos_mode = h->cfg.sincos_mode;
    const int nj = h->pop.n_joints;
    for (int c = 0; c < h->n_worlds; ++c) {
        const World* w = &h->worlds[c];
        const int j0 = h->pop.body_off[c] - c;
        for (int k = 0; k < w->nj; ++k) {
            Ctrl cc = w->ctrl[k + 1];
            for (int t = 0; t < T; ++t) {
                cc.phase += 0.0;
                cc.i_state += cc.frequency;
                out[(size_t)t * nj + j0 + k] = cc.amplitude * sin_f64(cc.i_state + cc.phase) + cc.offset;
            }
        }
    }
    return REM2D_OK;
}

int rem2d_destroy(rem2d_handle* h) {
    if (!h) return REM2D_E_INVALID;
    pthread_mutex_lock(&g_entries_lock);
    for (ControlEntry** p = &g_entries; *p; p = &(*p)->next)
        if ((*p)->h == h) { ControlEntry* e = *p; *p = e->next; free(e); break; }
    pthread_mutex_unlock(&g_entries_lock);
    return oracle_destroy(h);
}
int rem2d_upload(rem2d_handle* h, const rem2d_population* pop) {
    set_consumed(h, 0);
    return oracle_upload(h, pop);
}
int rem2d_reset(rem2d_handle* h) {
    set_consumed(h, 0);
    return oracle_reset(h);
}
int rem2d_step(rem2d_handle* h, int32_t n_ticks) {
    ControlEntry* e = h ? entry_of(h) : NULL;
    if (e && e->consumed) { snprintf(h->err, sizeof(h->err), "step: per-creature state was consumed by rem2d_run_episodes; call rem2d_reset first"); return REM2D_E_INVALID; }
    return oracle_step(h, n_ticks);
}
int rem2d_run_episodes(rem2d_handle* h, int32_t max_ticks) {
    int rc = oracle_run_episodes(h, max_ticks);
    set_consumed(h, 1);
    return rc;
}
int rem2d_evaluate(rem2d_handle* h, const rem2d_population* pop, int32_t max_ticks, double* fitness_out, int32_t* ticks_out) {
    int rc = oracle_evaluate(h, pop, max_ticks, fitness_out, ticks_out);
    set_consumed(h, 1);
    return rc;
}
