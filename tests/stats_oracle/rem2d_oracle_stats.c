/* rem2d_oracle_stats.c — TEST INFRASTRUCTURE: the CPU oracle with the episode statistics of include/rem2d_stats.h.
 *
 * The oracle (oracle/rem2d_oracle.c) is compiled here unchanged; this unit adds rem2d_set_stats / rem2d_read_stats and, in the
 * whole-episode runs of a population uploaded with statistics on, runs the oracle's own tick() creature by creature and
 * accumulates the statistics from the World after every tick, i.e. after the termination rule. Everything else is the oracle's
 * code path: results, counters and the stepping entry are the same as oracle/librem2d_oracle.so's. Per-handle statistics live
 * in a side table, because the oracle's handle is its own. Build: make -C tests/stats_oracle. Used by the statistics tests. */
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

typedef struct StatsEntry {
    rem2d_handle* h;
    int on, upload_on, valid;          /* rem2d_set_stats flag, its value at the upload, "the arrays hold the last run's" */
    int n, nb;
    int32_t *end_reason, *airborne_ticks, *ground_ticks;
    float* max_x;
    double* joint_work;
    struct StatsEntry* next;
} StatsEntry;
static StatsEntry* g_entries = NULL;
static pthread_mutex_t g_entries_lock = PTHREAD_MUTEX_INITIALIZER;

static StatsEntry* entry_of(rem2d_handle* h) {
    pthread_mutex_lock(&g_entries_lock);
    StatsEntry* e = g_entries;
    while (e && e->h != h) e = e->next;
    if (!e && (e = (StatsEntry*)calloc(1, sizeof(StatsEntry)))) { e->h = h; e->next = g_entries; g_entries = e; }
    pthread_mutex_unlock(&g_entries_lock);
    return e;
}
static void free_arrays(StatsEntry* e) {
    free(e->end_reason); free(e->airborne_ticks); free(e->ground_ticks); free(e->max_x); free(e->joint_work);
    e->end_reason = e->airborne_ticks = e->ground_ticks = NULL; e->max_x = NULL; e->joint_work = NULL;
}

/* the statistics of creature c after one tick of its world (definitions: include/rem2d_stats.h) */
static void accumulate(const rem2d_handle* h, StatsEntry* s, const World* w, int c) {
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

/* rem2d_step of the oracle (same dynamic schedule over creatures, same counters) with the accumulation after every tick */
typedef struct { rem2d_handle* h; StatsEntry* s; int n_ticks; int* next; Counters cnt; } RecordJob;
static void* record_worker(void* arg) {
    RecordJob* job = (RecordJob*)arg;
    rem2d_handle* h = job->h;
    const int chunk = 8;
    for (;;) {
        int c0 = __atomic_fetch_add(job->next, chunk, __ATOMIC_RELAXED);
        if (c0 >= h->n_worlds) break;
        int c1 = c0 + chunk < h->n_worlds ? c0 + chunk : h->n_worlds;
        for (int c = c0; c < c1; ++c) {
            World* w = &h->worlds[c];
            for (int t = 0; t < job->n_ticks && w->alive; ++t) {
                tick(h, w, &job->cnt);
                accumulate(h, job->s, w, c);
            }
        }
    }
    return NULL;
}
static int run_recorded(rem2d_handle* h, StatsEntry* s, int32_t n_ticks) {
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
    g_sincos_mode = h->cfg.sincos_mode;
    int nt = h->threads > 0 ? h->threads : 1;
    if (nt > 256) nt = 256;
    int next = 0;
    RecordJob* jobs = (RecordJob*)calloc((size_t)nt, sizeof(RecordJob));
    pthread_t* tids = (pthread_t*)calloc((size_t)nt, sizeof(pthread_t));
    for (int i = 0; i < nt; ++i) { jobs[i].h = h; jobs[i].s = s; jobs[i].n_ticks = n_ticks; jobs[i].next = &next; }
    for (int i = 1; i < nt; ++i) pthread_create(&tids[i], NULL, record_worker, &jobs[i]);
    record_worker(&jobs[0]);
    for (int i = 1; i < nt; ++i) pthread_join(tids[i], NULL);
    for (int i = 0; i < nt; ++i)
        for (int k = 0; k < REM2D_N_COUNTERS; ++k) h->counters[k] += jobs[i].cnt.c[k];
    free(jobs); free(tids);
    for (int c = 0; c < h->n_worlds; ++c)
        if (h->worlds[c].overflow) { snprintf(h->err, sizeof(h->err), "step: island scratch overflow in creature %d", c); return REM2D_E_CAPACITY; }
    s->valid = 1;
    return REM2D_OK;
}

int rem2d_destroy(rem2d_handle* h) {
    if (!h) return REM2D_E_INVALID;
    pthread_mutex_lock(&g_entries_lock);
    for (StatsEntry** p = &g_entries; *p; p = &(*p)->next)
        if ((*p)->h == h) { StatsEntry* e = *p; *p = e->next; free_arrays(e); free(e); break; }
    pthread_mutex_unlock(&g_entries_lock);
    return oracle_destroy(h);
}
int rem2d_upload(rem2d_handle* h, const rem2d_population* pop) {
    StatsEntry* s = h ? entry_of(h) : NULL;
    if (s) { s->valid = 0; s->upload_on = s->on; }
    return oracle_upload(h, pop);
}
int rem2d_reset(rem2d_handle* h) {
    StatsEntry* s = h ? entry_of(h) : NULL;
    if (s) s->valid = 0;
    return oracle_reset(h);
}
int rem2d_step(rem2d_handle* h, int32_t n_ticks) {
    StatsEntry* s = h ? entry_of(h) : NULL;
    if (s) s->valid = 0;                 /* the stepping path records no statistics */
    return oracle_step(h, n_ticks);
}
int rem2d_run_episodes(rem2d_handle* h, int32_t max_ticks) {
    int rc = rem2d_reset(h);
    if (rc) return rc;
    return run_recorded(h, entry_of(h), max_ticks);
}
int rem2d_evaluate(rem2d_handle* h, const rem2d_population* pop, int32_t max_ticks, double* fitness_out, int32_t* ticks_out) {
    int rc = rem2d_upload(h, pop);
    if (rc) return rc;
    rc = run_recorded(h, entry_of(h), max_ticks);
    if (rc) return rc;
    if (fitness_out) { rc = rem2d_fitness(h, fitness_out); if (rc) return rc; }
    if (ticks_out) for (int c = 0; c < h->n_worlds; ++c) ticks_out[c] = h->worlds[c].ticks;
    return REM2D_OK;
}
int rem2d_set_stats(rem2d_handle* h, int32_t on) {
    StatsEntry* s = h ? entry_of(h) : NULL;
    if (!s) return REM2D_E_INVALID;
    s->on = on != 0;
    return REM2D_OK;
}
int rem2d_read_stats(rem2d_handle* h, rem2d_episode_stats* out) {
    StatsEntry* s = h ? entry_of(h) : NULL;
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
