// rem2d_host_util.h — host-side helpers shared by the CUDA library (rem2d_cuda.cu) and the CPU emulation harness of the device
// code (tests/emu, test infrastructure): the capacity classes, the options and the episode planner (pure functions: no CUDA
// calls, no handle state), the joint order and the terrain / constant tables.
#pragma once
#include <stdint.h>
#include <math.h>
#include <algorithm>

// Capacity classes: NB bodies, NC contact-pool slots (fat-AABB overlaps), NT touching contacts staged in shared memory (further
// touching contacts, up to NC, spill to the cold block: correct but slower), GS = largest log2(lanes per creature) the automatic
// choice may give the class (plan_upload; 1-2 body creatures have nothing to share). Hot words per creature = 5*NB + 17*(NB-1)
// + 21*NT (+ schedule rows per warp when lanes are shared); shared memory, not registers, bounds the resident creatures per SM,
// so lanes are the free resource: a group of 2^gs lanes shares one creature's solver sweeps (static modulo schedule,
// rem2d_device.cuh) and its per-body / per-joint / per-contact loops.
#define N_CLASSES 9
struct ClassDims { int nb, nc, nt, gs; };
static const ClassDims class_dims[N_CLASSES] = {
    {1, 10, 3, 0}, {2, 16, 4, 0}, {4, 28, 4, 1}, {8, 48, 6, 3}, {12, 64, 6, 5}, {16, 80, 6, 5}, {22, 104, 6, 5}, {32, 144, 8, 5},
    {44, 192, 10, 5},
};
// Widest group shift a draining episode warp of class k launched at group shift gs regroups its survivors to (Sim::episodes):
// the class's automatic cap, or the launch's own width if that was forced wider.
static inline int widest_group_shift(int k, int gs) { return std::max(gs, class_dims[k].gs); }
static inline int class_hot_bytes(int k, int gs) {      // shared memory of a warp (CTA) of class k, groups of 2^gs lanes
    return rem2d::make_hot_layout(rem2d::make_layout(class_dims[k].nb, class_dims[k].nc, class_dims[k].nt), gs).rows * 128;
}

// Tuning / diagnostic options (rem2d_set_option; the REM2D_* environment variables of the same names are read ONCE, at
// rem2d_create, as initial values - tools/sweep_groups.py, tools/ea_pop_sweep.py and the tests use them). Defaults are the measured optimum.
struct Options {
    int warp_mode_max = -1;      // largest population that runs one warp per creature from tick 0 (-1: 48 per SM)
    int park_ticks = -1;         // park threshold of the queue mode (-1: automatic, 0: never park)
    double park_cap = -1.0;      // fraction of a class that may be parked (-1: automatic)
    int overflow_wave = 1;       // queue the CTAs a class could not seat in its first wave behind the first launches (see plan_upload)
    int image = -1;              // kernel image of the episode launches (-1: automatic, 0: ~200 registers, 1: 128 registers)
    double smem_budget_kb = 227.0;
    int group_shift = -1;        // log2 lanes per creature in the queue / step kernels (-1: per class default)
    int class_gs[N_CLASSES] = {-1, -1, -1, -1, -1, -1, -1, -1, -1};   // per capacity class ("class_gs_<k>", -1: default)
    int tail_group_shift = 5;    // log2 lanes per creature of the tail launches (few creatures are parked by default: a warp each)
    int trace = 0;
};

// ------------------------------------------------------------------ episode planner
// The device and the uploaded population as the planner sees them.
struct PlanInput {
    int n_sms = 0;
    int max_warps_per_sm[2] = {8, 16};  // resident warps of the two episode kernel images per SM by registers (occupancy API)
    int members[N_CLASSES] = {};        // creatures per capacity class
    double work[N_CLASSES] = {};        // sum of the per-creature cost estimates of the class
};

// Decided at upload: lanes per creature, grids and kernel image of the queue-mode episode launches.
struct UploadPlan {
    int image;                  // kernel image of the population (0: 200 registers, 1: 128 registers)
    bool all_fit;               // every creature has a group from the start with one lane each (forced widths kept)
    int gs[N_CLASSES];          // log2 lanes per creature of the queue mode
    int grid[N_CLASSES];        // resident warps of the first wave
    int grid2[N_CLASSES];       // overflow wave (same group width) for the creatures that do not fit in the first round
};

// Decided at the start of each rem2d_run_episodes.
struct LaunchPlan {
    bool warp_mode;             // one warp per creature from tick 0, no parking
    int park_ticks;             // park threshold of the queue launches (0: no parking, no tail launches)
    int park_cap[N_CLASSES];    // most creatures of the class that may be parked
    int order[N_CLASSES];       // launch order of the classes
};

// Resident warps of the persistent episode kernels (grid[]) for the group shifts gs[]. All classes run concurrently, so the
// shared memory of the SMs (227 KB each, first_wave_frac of it) and the resident-warp limit set by the register file are divided
// among them in proportion to their work; a class never gets more warps than it has creatures, and what it cannot use is
// handed to the others. Without this the largest class would occupy every SM until its last creature dies and the remaining
// classes would run after it. Returns true iff EVERY creature of every class has a group from the start (one round,
// under-filled GPU).
static bool size_grids(const PlanInput& in, const Options& o, const int gs[N_CLASSES], int image, double first_wave_frac,
                       double warp_frac, int grid[N_CLASSES]) {
    double budget = (double)in.n_sms * o.smem_budget_kb * 1024.0 * 0.98 * first_wave_frac;
    double work[N_CLASSES], smem[N_CLASSES];
    bool fixed[N_CLASSES];
    for (int k = 0; k < N_CLASSES; ++k) {
        work[k] = in.work[k]; fixed[k] = in.members[k] == 0; smem[k] = class_hot_bytes(k, gs[k]) + 1024.0;
        // a group of G lanes is one resident creature: G times the warps for the same residency, and the creature ticks
        // p(G) times faster (measured tick latencies, profiles/r2_timeline_*.txt)
        static const double speedup[6] = {1.0, 1.15, 1.5, 1.9, 2.2, 2.5};
        work[k] *= (double)(1 << gs[k]) / speedup[gs[k]];
        grid[k] = 0;
    }
    // warps_k = W * work_k with W such that sum_k warps_k * smem_k = budget: every class then needs about the same
    // number of sequential creature-lifetimes per group times its own tick latency, i.e. the classes finish together.
    // The register file bounds the resident warps as well (max_warps_per_sm, from the occupancy API): a launch whose
    // CTAs do not fit waits for the CTAs of the classes launched before it to EXIT, which serialises the classes
    // (measured: the small classes started 400 ms late when 9 warps per SM fit and the grids asked for 9.7).
    double warp_budget = (double)in.n_sms * in.max_warps_per_sm[image] * warp_frac;
    bool all_fit = true;
    for (int round = 0; round <= N_CLASSES; ++round) {
        double denom = 0.0, wsum = 0.0;
        for (int k = 0; k < N_CLASSES; ++k) if (!fixed[k]) { denom += work[k] * smem[k]; wsum += work[k]; }
        if (denom <= 0.0) break;
        const double W = std::max(0.0, std::min(budget / denom, warp_budget / wsum));
        bool changed = false;
        for (int k = 0; k < N_CLASSES; ++k) {
            if (fixed[k]) continue;
            const int per = 32 >> gs[k], need = (in.members[k] + per - 1) / per;    // one group per creature
            if ((int)(W * work[k]) >= need) {        // the class fits entirely: fix it and give the rest back
                grid[k] = need;
                budget -= need * smem[k];
                warp_budget -= need;
                fixed[k] = true; changed = true;
            }
        }
        if (!changed) {
            for (int k = 0; k < N_CLASSES; ++k)
                if (!fixed[k]) { grid[k] = std::max(1, (int)(W * work[k])); all_fit = false; }
            break;
        }
    }
    for (int k = 0; k < N_CLASSES; ++k)
        if (in.members[k] && grid[k] < 1) grid[k] = 1;
    return all_fit;
}

// Lanes per creature of every class for the uploaded population, then the grids. Throughput and latency pull in opposite
// directions: one lane per creature issues the fewest instructions per creature-tick, a group of G lanes ticks a creature
// up to ~2x faster but spends more issue slots on it (idle lanes in the sweeps, leader sections). Measured on B200
// (tools/sweep_groups.py): with 65536 creatures the GPU is throughput-bound and G = 1 everywhere is fastest; when the
// population leaves the GPU under-filled (every creature resident from the start) the run time is one creature lifetime
// times the tick latency, and wider groups win. So: start from G = 1 and widen the groups of the large classes (up to the
// class table's value) as long as every creature of every class still has a group from the start. Explicit options
// ("group_shift", "class_gs_<k>") override the choice.
static UploadPlan plan_upload(const PlanInput& in, const Options& o) {
    UploadPlan p{};
    bool forced[N_CLASSES];
    for (int k = 0; k < N_CLASSES; ++k) {
        const int f = o.group_shift >= 0 ? o.group_shift : o.class_gs[k];
        forced[k] = f >= 0;
        p.gs[k] = forced[k] ? std::min(5, f) : 0;
    }
    // under-filled GPU <=> everything fits with one lane per creature in the 128-register image: then widen (below)
    p.image = 1;
    p.all_fit = size_grids(in, o, p.gs, p.image, 1.0, 0.97, p.grid);
    if (!p.all_fit) {
        // Throughput-bound: one lane per creature - except the largest class (33-44 bodies): its 4.6 KB of solver state per
        // creature make a 32-creature CTA 148 KB of shared memory, ONE resident warp per SM at a 5 ms tick. 8 lanes per creature
        // (4 creatures, 19 KB per CTA) pack the same residency into warps that tick twice as fast and fit beside the other
        // classes' CTAs. Measured on EA-configured populations (max_size 40; tools/ea_pop_sweep.py, profiles/r2_ea_pop_sweep.txt):
        // 1.5-1.6x on the whole evaluation (1946 -> 1271 ms, 3311 -> 2112, 5925 -> 3676); widening the 23-32 body class as well
        // gains nothing, the smaller classes lose (the bench population, <= 21 bodies, is unaffected).
        for (int k = 0; k < N_CLASSES; ++k)
            if (!forced[k]) p.gs[k] = class_dims[k].nb > 32 ? 3 : 0;
        p.image = o.image >= 0 ? o.image : 0;
        // Mixed widths: the cost model's tick latencies are those of one-lane warps on moderately loaded SMs; next to
        // hundreds of 8-lane warps the one-lane classes tick 2x slower than modelled (4.8 ms against 1.55 ms for the wide
        // class) and a first wave that asks for all of the shared memory does not even fit (736 of 822 CTAs resident,
        // the launches behind them held back). With an overflow wave it is better to seat 75 % statically and let the
        // queued CTAs take the rest as it frees up: 3560 -> 2610 ms, 1930 -> 1600, 1155 -> 1130 ms on the three
        // EA-configured populations; all-one-lane populations (the bench) lose 4 % with it and keep the full first wave.
        bool mixed = false;
        for (int k = 0; k < N_CLASSES; ++k) mixed |= in.members[k] > 0 && p.gs[k] > 0;
        const double first_wave_frac = mixed && o.overflow_wave && o.smem_budget_kb > 226.0 ? 0.75 : 1.0;
        size_grids(in, o, p.gs, p.image, first_wave_frac, 0.97, p.grid);
        // Throughput-bound population: one lane per creature, lanes refilled from the class queue.
        // OVERFLOW WAVE (default): the first-wave grids above come from a static cost model; when it is off for a population -
        // measured on an EA-configured one: the 33-44 body class done after 1.9 s, the others at 3.1-3.6 s, with the freed 18 MB
        // of shared memory idle in between (profiles/r2_timeline_ea_gen2_before.txt) - nothing could use the resources of a
        // class that has finished. So every class also queues, BEHIND all first launches, the CTAs it could not seat: the
        // work distributor places them as earlier CTAs exit, they pull from the same class queue, and a CTA that finds its
        // queue empty exits at once. The hardware does the balancing.
        for (int k = 0; k < N_CLASSES && o.overflow_wave; ++k) {
            const int per = 32 >> p.gs[k], left = in.members[k] - p.grid[k] * per;
            if (left > 0) p.grid2[k] = (left + per - 1) / per;
        }
        return p;
    }
    // widest uniform group width (capped per class) with which every creature has a group from the start AND the warps fill
    // at most 60 % of the resident-warp limit: wide groups are issue-bound before the SMs are full. Measured optimum
    // (tools/small_pop.py): 16384 creatures -> 4 lanes, 8192 -> 8, 4096 -> 8-16, <= 1024 -> 32; one lane always fits (all_fit)
    for (int gs = 5;; --gs) {
        for (int k = 0; k < N_CLASSES; ++k)
            if (!forced[k]) p.gs[k] = std::min(gs, class_dims[k].gs);
        if (gs == 0 || size_grids(in, o, p.gs, p.image, 1.0, 0.6, p.grid)) { size_grids(in, o, p.gs, p.image, 1.0, 0.97, p.grid); return p; }
    }
}

static LaunchPlan plan_launch(const PlanInput& in, const UploadPlan& up, int max_ticks, const Options& o) {
    LaunchPlan p{};
    // creatures still alive after park_ticks are finished by tail-mode launches (REM2D_PARK_TICKS=0 disables parking)
    // Measured on B200 (tools/sweep_groups.py, 65536 L-system creatures): parking at 200-256 ticks (~0.5-1.4 % of the creatures)
    // is the best trade: a tail warp finishes a creature 3-4x sooner than its bulk lane would, but it occupies a whole warp, so
    // earlier thresholds (thousands of parked creatures) slow the bulk down more than they shorten the critical path; later
    // ones leave the longest-lived creatures on the slow path. Drain / late-start parking never paid off. The number of
    // parked creatures per class is bounded (a quarter of the class, at most 16 per SM): in an evolved population where most creatures live
    // long, the rest simply stay on their lanes.
    int park_ticks = 200;            // measured (tools/sweep_groups.py, 65536 creatures): 256 -> 820 ms, 200 -> 790 ms, 160 -> 930 ms
    double cap_frac = 0.25;
    // Under-filled GPU (every creature of every class has a group from the start, e.g. 16384 creatures): tail warps find
    // free SM resources, so parking earlier pays (16384 creatures: 450 -> 413 ms with 160 ticks and a quarter of a class).
    bool single_round = true;
    for (int k = 0; k < N_CLASSES; ++k)
        if (in.members[k] && up.grid[k] * (32 >> up.gs[k]) < in.members[k]) single_round = false;
    if (single_round) park_ticks = 160;
    if (o.park_ticks >= 0) park_ticks = o.park_ticks;
    if (o.park_cap >= 0.0) cap_frac = o.park_cap;
    // Small populations: one warp per creature from tick 0 (mode 2). All creatures then advance at the low tail-mode tick
    // latency and the run takes about one creature lifetime. Measured (tools/small_pop.py, L-system creatures): 2.4x faster
    // than the bulk mode at 128 creatures, 1.9x at 1024, 1.2x at 6144, break-even near 10^4, 0.6x at 16384 (the bulk mode has
    // 32x the lane efficiency).
    int n_creatures = 0;
    for (int k = 0; k < N_CLASSES; ++k) n_creatures += in.members[k];
    p.warp_mode = n_creatures <= (o.warp_mode_max >= 0 ? o.warp_mode_max : in.n_sms * 48);
    p.park_ticks = !p.warp_mode && park_ticks < max_ticks ? park_ticks : 0;
    for (int k = 0; k < N_CLASSES; ++k)
        p.park_cap[k] = std::min(in.members[k], std::max(32, std::min((int)(in.n_sms * 64 * cap_frac), (int)(in.members[k] * cap_frac))));
    // Launch order = decreasing shared memory per CTA (first-fit decreasing): the work distributor places the CTAs of the
    // launches in order, and a CTA that finds no SM with enough free shared memory holds back every launch behind it.
    // Measured (profiles/r2_timeline_ea_gen2_before.txt): with the 33-44 body class at 8 lanes per creature (22 KB per CTA)
    // launched first, its 822 CTAs left < 109 KB free on every SM, the 23-32 body class (109 KB per CTA) could not start, and
    // all seven smaller classes waited behind it until the first launch had finished (1.3 s of a 3.8 s evaluation).
    for (int k = 0; k < N_CLASSES; ++k) p.order[k] = k;
    std::stable_sort(p.order, p.order + N_CLASSES, [&](int a, int b) {
        const int sa = class_hot_bytes(a, p.warp_mode ? 5 : up.gs[a]), sb = class_hot_bytes(b, p.warp_mode ? 5 : up.gs[b]);
        return sa != sb ? sa > sb : a > b;
    });
    return p;
}

// Group shift of the stepping kernels (rem2d_reset / rem2d_step: static creature -> column mapping, no residency limit): the
// option if given, else as wide as keeps all warps of the population resident at once (a single creature gets a whole warp).
static int step_group_shift(const PlanInput& in, int k, const Options& o) {
    const int f = o.group_shift >= 0 ? o.group_shift : o.class_gs[k];
    if (f >= 0) return std::min(5, f);
    int total = 0;
    for (int q = 0; q < N_CLASSES; ++q) total += (in.members[q] + 31) / 32;
    int gs = 0;
    while (gs < 5 && (total << (gs + 1)) <= in.n_sms * 8) ++gs;
    return class_dims[k].nb <= 2 ? 0 : gs;
}

// joint order inside the creature's island: DFS of b2World::Solve from the newest body, each body's joint
// list newest first (SURVEY.md A.9). Pure topology, so it is computed once on the host.
static inline void island_joint_order(int nb, const int16_t* parent, uint8_t* order) {
    const int nj = nb - 1;
    if (nj <= 0) return;
    char bodyFlag[64] = {0}, jointFlag[64] = {0};      // nb <= 44 (largest capacity class)
    int stack[64], sp = 0, n = 0;
    stack[sp++] = nb - 1;
    bodyFlag[nb - 1] = 1;
    while (sp > 0) {
        const int b = stack[--sp];
        for (int j = nj - 1; j >= 0; --j) {
            if (parent[j] != b && j + 1 != b) continue;
            if (jointFlag[j]) continue;
            const int other = parent[j] == b ? j + 1 : parent[j];
            order[n++] = (uint8_t)j;
            jointFlag[j] = 1;
            if (bodyFlag[other]) continue;
            stack[sp++] = other;
            bodyFlag[other] = 1;
        }
    }
}


// Terrain table from the reference's 200-vertex height field (Modular2DEnv.py:294-306): edgeShape vertices are Python doubles
// rounded to float32; fat AABB = b2EdgeShape::ComputeAABB (radius = polygonRadius) + aabbExtension, single float ops.
static inline void fill_terrain(rem2d::Terrain* t, const double* y, int n, double step) {
    memset(t, 0, sizeof(rem2d::Terrain));
    t->n_edges = n - 1;
    t->step = (float)step;
    for (int i = 0; i < n - 1; ++i) {
        float x1 = (float)((double)i * step), y1 = (float)y[i], x2 = (float)((double)(i + 1) * step), y2 = (float)y[i + 1];
        t->v1x[i] = x1; t->v1y[i] = y1; t->v2x[i] = x2; t->v2y[i] = y2;
        volatile float lox = (x1 < x2 ? x1 : x2), loy = (y1 < y2 ? y1 : y2), hix = (x1 > x2 ? x1 : x2), hiy = (y1 > y2 ? y1 : y2);
        volatile float a;
        a = lox - RB_POLY_RADIUS; t->flx[i] = a - RB_AABB_EXT;
        a = loy - RB_POLY_RADIUS; t->fly[i] = a - RB_AABB_EXT;
        a = hix + RB_POLY_RADIUS; t->fhx[i] = a + RB_AABB_EXT;
        a = hiy + RB_POLY_RADIUS; t->fhy[i] = a + RB_AABB_EXT;
    }
}
static inline rem2d::Consts make_consts(const rem2d_config* cfg) {
    rem2d::Consts k;
    k.dt = cfg->dt; k.gravity_y = cfg->gravity_y;
    k.friction = sqrtf(cfg->terrain_friction * cfg->module_friction);       // b2MixFriction
    k.vel_iters = cfg->velocity_iterations; k.pos_iters = cfg->position_iterations;
    k.continuous = cfg->continuous; k.allow_sleep = cfg->allow_sleep; k.terminate = cfg->terminate;
    k.evaluation_steps = cfg->evaluation_steps;
    k.p_gain = cfg->p_gain; k.wod_speed = cfg->wod_speed; k.env_length = cfg->env_length;
    return k;
}
