/* rem2d_oracle_ext.c — TEST INFRASTRUCTURE: the CPU oracle with the extension headers include/rem2d_stats.h (episode
 * statistics) and include/rem2d_control.h (joint-target stepping and observations).
 *
 * The oracle (oracle/rem2d_oracle.c) is compiled here unchanged; this unit adds
 *  - rem2d_set_stats / rem2d_read_stats: the whole-episode runs of a population uploaded with statistics on run the oracle's
 *    own tick() creature by creature and accumulate the statistics from the World after every tick, i.e. after the
 *    termination rule;
 *  - rem2d_step_targets, which runs the oracle's world_step with tick()'s P-control and episode bookkeeping but takes the
 *    controller output from the targets (the sine controllers are not advanced), and rem2d_read_observations;
 *  - rem2d_control_sine_outputs (test only).
 * Everything else is the oracle's code path: results, counters and the stepping entry are those of oracle/librem2d_oracle.so.
 * The call contract is the CUDA library's: a whole-episode run consumes the per-creature state, and until the next
 * rem2d_upload / rem2d_reset the stepping calls and rem2d_read_observations are refused, before they change anything (the
 * statistics of the run stay readable). The per-handle flags and statistics live in a side table, because the oracle's handle
 * is its own. Build: make -C tests/oracle_ext. Used by tests/oracle_ext/oracle_ext.py. */
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
#include "../../include/rem2d_stats.h"
#include "../../include/rem2d_control.h"

typedef struct Entry {
    rem2d_handle* h;
    int on, upload_on, valid;          /* rem2d_set_stats flag, its value at the upload, "the arrays hold the last run's" */
    int consumed;                      /* state consumed by a whole-episode run */
    int n, nb;
    int32_t *end_reason, *airborne_ticks, *ground_ticks;
    float* max_x;
    double* joint_work;
    struct Entry* next;
} Entry;
static Entry* g_entries = NULL;
static pthread_mutex_t g_entries_lock = PTHREAD_MUTEX_INITIALIZER;

static Entry* entry_of(rem2d_handle* h) {
    if (!h) return NULL;
    pthread_mutex_lock(&g_entries_lock);
    Entry* e = g_entries;
    while (e && e->h != h) e = e->next;
    if (!e && (e = (Entry*)calloc(1, sizeof(Entry)))) { e->h = h; e->next = g_entries; g_entries = e; }
    pthread_mutex_unlock(&g_entries_lock);
    return e;
}
static void free_arrays(Entry* e) {
    free(e->end_reason); free(e->airborne_ticks); free(e->ground_ticks); free(e->max_x); free(e->joint_work);
    e->end_reason = e->airborne_ticks = e->ground_ticks = NULL; e->max_x = NULL; e->joint_work = NULL;
}

/* the statistics of creature c after one tick of its world (definitions: include/rem2d_stats.h) */
static void accumulate(const rem2d_handle* h, Entry* s, const World* w, int c) {
    const float x = w->bodies[0].xf.p.x;
    if (h->cfg.terminate) {       /* the comparisons of the termination rule in tick(), in its precedence */
        int why = REM2D_END_RUNNING;
        if (x < 0.0f) why = REM2D_END_ORIGIN;
        else if (w->wod > (double)x) why = REM2D_END_WALL;
        else if ((double)x > h->cfg.env_length) why = REM2D_END_GOAL;
        else if (w->ticks >= h->cfg.evaluation_steps) why = REM2D_END_STEPS;
        if (why != REM2D_END_RUNNING) s->end_reason[c] = why;
    }
    if (x > s->max_x[c]) s->max_x[c] = x;
    double work = s->joint_work[c];
    for (int k = 0; k < w->nj; ++k) {
        const Joint* j = &w->joints[k];
        work += fabs((double)j->motorImpulse * ((double)w->bodies[j->bodyB].w - (double)w->bodies[j->bodyA].w));
    }
    s->joint_work[c] = work;
    uint64_t ground = 0;
    for (int i = 0; i < w->nc; ++i)
        if (w->contacts[i].flags & CF_TOUCHING) ground |= 1ull << w->contacts[i].body;
    if (!ground) s->airborne_ticks[c]++;
    int32_t* g = &s->ground_ticks[h->pop.body_off[c]];
    for (int b = 0; b < w->nb; ++b)
        if ((ground >> b) & 1ull) g[b]++;
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

/* The stepping loop of the oracle's rem2d_step (dynamic schedule over the worlds in chunks of 8, per-thread counters summed at
 * the end, the island-overflow check) with the creature-tick `fn`: tick + accumulate or tick_target. */
typedef struct Job { rem2d_handle* h; Entry* e; const double* targets; void (*fn)(struct Job*, World*, int); int n_ticks; int* next; Counters cnt; } Job;
static void tick_recorded(Job* job, World* w, int c) { tick(job->h, w, &job->cnt); accumulate(job->h, job->e, w, c); }
static void tick_targeted(Job* job, World* w, int c) { tick_target(job->h, w, job->targets + (job->h->pop.body_off[c] - c), &job->cnt); }
static void* worker(void* arg) {
    Job* job = (Job*)arg;
    rem2d_handle* h = job->h;
    const int chunk = 8;
    for (;;) {
        int c0 = __atomic_fetch_add(job->next, chunk, __ATOMIC_RELAXED);
        if (c0 >= h->n_worlds) break;
        int c1 = c0 + chunk < h->n_worlds ? c0 + chunk : h->n_worlds;
        for (int c = c0; c < c1; ++c) {
            World* w = &h->worlds[c];
            for (int t = 0; t < job->n_ticks && w->alive; ++t) job->fn(job, w, c);
        }
    }
    return NULL;
}
static int run_worlds(rem2d_handle* h, Entry* e, const double* targets, void (*fn)(Job*, World*, int), int n_ticks) {
    g_sincos_mode = h->cfg.sincos_mode;
    int nt = h->threads > 0 ? h->threads : 1;
    if (nt > 256) nt = 256;
    int next = 0;
    Job* jobs = (Job*)calloc((size_t)nt, sizeof(Job));
    pthread_t* tids = (pthread_t*)calloc((size_t)nt, sizeof(pthread_t));
    for (int i = 0; i < nt; ++i) { jobs[i].h = h; jobs[i].e = e; jobs[i].targets = targets; jobs[i].fn = fn; jobs[i].n_ticks = n_ticks; jobs[i].next = &next; }
    for (int i = 1; i < nt; ++i) pthread_create(&tids[i], NULL, worker, &jobs[i]);
    worker(&jobs[0]);
    for (int i = 1; i < nt; ++i) pthread_join(tids[i], NULL);
    for (int i = 0; i < nt; ++i)
        for (int k = 0; k < REM2D_N_COUNTERS; ++k) h->counters[k] += jobs[i].cnt.c[k];
    free(jobs); free(tids);
    for (int c = 0; c < h->n_worlds; ++c)
        if (h->worlds[c].overflow) { snprintf(h->err, sizeof(h->err), "step: island scratch overflow in creature %d", c); return REM2D_E_CAPACITY; }
    return REM2D_OK;
}

/* Whole episodes from the state oracle_upload / oracle_reset just built: the recorded loop if the population was uploaded with
 * statistics on, the oracle's own stepping loop otherwise (what oracle_run_episodes / oracle_evaluate run after their reset,
 * never the refusing rem2d_step below). Either way the state is consumed afterwards, as in the CUDA library. */
static int run_whole(rem2d_handle* h, Entry* s, int32_t n_ticks) {
    s->consumed = 1;
    if (!s->upload_on) return oracle_step(h, n_ticks);
    if (n_ticks < 0) return REM2D_E_INVALID;
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
    int rc = run_worlds(h, s, NULL, tick_recorded, n_ticks);
    s->valid = rc == REM2D_OK;
    return rc;
}

/* The CUDA library's rule for the stepping calls: no population, a negative tick count or state consumed by a whole-episode
 * run are refused before anything changes, the statistics' valid flag included. */
static int refuse_step(rem2d_handle* h, Entry* e, int32_t n_ticks, const char* what) {
    if (!h) return 1;
    if (!e || !h->have_pop || n_ticks < 0 || e->consumed) {
        snprintf(h->err, sizeof(h->err), "%s: no population / negative tick count / state consumed by rem2d_run_episodes; call rem2d_reset first", what);
        return 1;
    }
    return 0;
}

int rem2d_destroy(rem2d_handle* h) {
    if (!h) return REM2D_E_INVALID;
    pthread_mutex_lock(&g_entries_lock);
    for (Entry** p = &g_entries; *p; p = &(*p)->next)
        if ((*p)->h == h) { Entry* e = *p; *p = e->next; free_arrays(e); free(e); break; }
    pthread_mutex_unlock(&g_entries_lock);
    return oracle_destroy(h);
}
int rem2d_upload(rem2d_handle* h, const rem2d_population* pop) {
    Entry* e = entry_of(h);
    if (e) { e->valid = 0; e->consumed = 0; e->upload_on = e->on; }
    return oracle_upload(h, pop);
}
int rem2d_reset(rem2d_handle* h) {
    Entry* e = entry_of(h);
    if (e) { e->valid = 0; e->consumed = 0; }
    return oracle_reset(h);
}
int rem2d_step(rem2d_handle* h, int32_t n_ticks) {
    Entry* e = entry_of(h);
    if (refuse_step(h, e, n_ticks, "step")) return REM2D_E_INVALID;
    e->valid = 0;                        /* the stepping path records no statistics */
    return oracle_step(h, n_ticks);
}
int rem2d_run_episodes(rem2d_handle* h, int32_t max_ticks) {
    int rc = rem2d_reset(h);
    return rc ? rc : run_whole(h, entry_of(h), max_ticks);
}
int rem2d_evaluate(rem2d_handle* h, const rem2d_population* pop, int32_t max_ticks, double* fitness_out, int32_t* ticks_out) {
    int rc = rem2d_upload(h, pop);
    if (!rc) rc = run_whole(h, entry_of(h), max_ticks);
    if (!rc && fitness_out) rc = rem2d_fitness(h, fitness_out);
    if (!rc && ticks_out) rc = rem2d_ticks(h, ticks_out);
    return rc;
}

int rem2d_set_stats(rem2d_handle* h, int32_t on) {
    Entry* s = entry_of(h);
    if (!s) return REM2D_E_INVALID;
    s->on = on != 0;
    return REM2D_OK;
}
int rem2d_read_stats(rem2d_handle* h, rem2d_episode_stats* out) {
    Entry* s = entry_of(h);
    if (!s || !out) return REM2D_E_INVALID;
    if (!h->have_pop || !s->valid) {
        snprintf(h->err, sizeof(h->err), "read_stats: no statistics: run rem2d_run_episodes / rem2d_evaluate on a population uploaded with rem2d_set_stats(1)");
        return REM2D_E_INVALID;
    }
    if (out->end_reason) memcpy(out->end_reason, s->end_reason, sizeof(int32_t) * (size_t)s->n);
    if (out->max_x) memcpy(out->max_x, s->max_x, sizeof(float) * (size_t)s->n);
    if (out->joint_work) memcpy(out->joint_work, s->joint_work, sizeof(double) * (size_t)s->n);
    if (out->airborne_ticks) memcpy(out->airborne_ticks, s->airborne_ticks, sizeof(int32_t) * (size_t)s->n);
    if (out->ground_ticks) memcpy(out->ground_ticks, s->ground_ticks, sizeof(int32_t) * (size_t)s->nb);
    return REM2D_OK;
}

int rem2d_step_targets(rem2d_handle* h, const double* targets, int32_t n_ticks) {
    Entry* e = entry_of(h);
    if (refuse_step(h, e, n_ticks, "step_targets")) return REM2D_E_INVALID;
    if (!targets) { snprintf(h->err, sizeof(h->err), "step_targets: NULL targets"); return REM2D_E_INVALID; }
    for (int j = 0; j < h->pop.n_joints; ++j)
        if (!isfinite(targets[j])) { snprintf(h->err, sizeof(h->err), "step_targets: target %d is not finite", j); return REM2D_E_INVALID; }
    e->valid = 0;
    return run_worlds(h, e, targets, tick_targeted, n_ticks);
}

int rem2d_read_observations(rem2d_handle* h, rem2d_observation* out) {
    if (!h || !out) return REM2D_E_INVALID;
    Entry* e = entry_of(h);
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
