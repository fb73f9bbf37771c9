// rem2d_emu.cpp — TEST INFRASTRUCTURE: runs gym_rem2d_b200/csrc/rem2d_device.cuh (the device code of the CUDA kernels) on
// the CPU, one host thread per lane of a warp (see rem2d_emu_shim.h), so that the lane-group logic can be compared with the
// oracle without a GPU. The Makefile builds this one source once per variant of the device code: librem2d_emu.so (plain),
// librem2d_emu_stats.so (-DREM2D_STATS, the statistics images of the episode kernel) and librem2d_emu_targets.so
// (-DREM2D_TARGETS, step_kernel_targets). The variants change the layout of rem2d::Sim, so each is a library of its own, built
// with hidden visibility: only the extern "C" entries are exported and no library binds another's inline functions. Entries:
//  - rem2d_emu_step: one warp of the stepping kernel, up to 32 >> gs creatures with a group of 1 << gs lanes each, reset and
//    then n_calls launches of ticks_per_call ticks; with targets, call i holds targets[i] like rem2d_step_targets;
//  - rem2d_emu_queue: one warp of the queue-mode episode kernel (Sim::episodes, parking off, regrouping of a draining warp);
//  - the capacity classes and the episode planner of rem2d_host_util.h.
// Build: make -C tests/emu. Used by tests/emu/emu.py only.
#include <cstring>
#include <functional>
#include <thread>
#include <vector>
#include <algorithm>

#define REM2D_EMU 1
#include "../../gym_rem2d_b200/csrc/rem2d_device.cuh"
#include "../../gym_rem2d_b200/csrc/rem2d_host_util.h"

#define EMU_API extern "C" __attribute__((visibility("default")))

thread_local emu::Ctx* emu::ctx = nullptr;
using namespace rem2d;

struct EmuOut {       // caller-allocated; every pointer is optional (NULL: skipped). Indexed like the table: by creature, body
                      // and joint of pop. A creature's entries are written when its run ends.
    float* pose; float* vel; float* joint_impulse; int32_t* limit_state; float* motor_speed;        // like rem2d_state_view
    int32_t* alive; int32_t* ticks; double* fitness; double* wod; int32_t* n_contacts; int32_t* n_touching;
    int32_t* touching_pairs; float* touching_impulse;
    int32_t* sched_P; int32_t* sched_smax;       // schedule of the creature's last tick (diagnostics)
    uint64_t* counters;                           // [REM2D_N_COUNTERS], summed over the warp
    int64_t* n_syncs;                             // barriers executed by the warp
    int32_t* status; int32_t* finish_gs;          // status; group shift of the creature's group when its run ended
    int32_t* gs_seq; int32_t* n_seq;              // queue: the group shifts the warp ran at, in order (the first is gs)
    float* joint_angle; float* joint_speed; float* root; int32_t* ground;                  // like rem2d_observation
    int32_t* end_reason; float* max_x; double* joint_work; int32_t* airborne_ticks; int32_t* ground_ticks;   // REM2D_STATS
    int32_t max_pairs, max_seq;
};

template <class T> static void put(T* dst, size_t i, T v) { if (dst) dst[i] = v; }

// What every run shares: the terrain, the constants, the island joint order and the device view of the population, and (with
// REM2D_STATS) the statistics of every creature of the table.
struct World {
    const rem2d_population* pop; Terrain ter; Consts k; std::vector<uint8_t> jorder; DevPop dp; Layout L;
    std::vector<float> cold, hot;
#ifdef REM2D_STATS
    std::vector<int32_t> end_reason, airborne_ticks, ground_ticks; std::vector<float> max_x; std::vector<double> joint_work;
#endif
    World(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg, int NB, int NC,
          int NT, int gs) : pop(pop), L(make_layout(NB, NC, NT)) {
        fill_terrain(&ter, terrain_y, n_vertices, step);
        k = make_consts(cfg);
        jorder.assign((size_t)std::max(pop->n_joints, 1), 0);
        for (int c = 0; c < pop->n_creatures; ++c) {
            int nb = pop->body_off[c + 1] - pop->body_off[c], j0 = pop->body_off[c] - c;
            island_joint_order(nb, pop->joint_parent + j0, jorder.data() + j0);
        }
        dp.body_off = pop->body_off; dp.shape = pop->shape; dp.hx = pop->hx; dp.hy = pop->hy; dp.x0 = pop->x0; dp.y0 = pop->y0; dp.a0 = pop->a0;
        dp.joint_parent = pop->joint_parent; dp.anchor_a = pop->anchor_a; dp.anchor_b = pop->anchor_b; dp.lower = pop->lower;
        dp.upper = pop->upper; dp.max_torque = pop->max_torque; dp.ctrl = pop->ctrl; dp.joint_order = jorder.data();
        cold.assign((size_t)L.words * 32, 0.0f);
        hot.assign((size_t)make_hot_layout(L, gs).rows * 32, 0.0f);
#ifdef REM2D_STATS
        const size_t n = std::max(pop->n_creatures, 1);
        end_reason.assign(n, 0); airborne_ticks.assign(n, 0); max_x.assign(n, 0.0f); joint_work.assign(n, 0.0);
        ground_ticks.assign((size_t)std::max(pop->n_bodies, 1), 0);
#endif
    }
    // the Sim of `lane`, with groups of 1 << gs lanes, on column lane >> gs of the warp's block as in the kernels
    void init(Sim& sim, int gs, int lane) {
        sim.L = L; sim.set_group(gs, lane, hot.data());
        sim.g = cold.data() + (lane >> gs);
        sim.ter = &ter; sim.k = &k;
        for (int i = 0; i < REM2D_N_COUNTERS; ++i) sim.cnt.c[i] = 0u;
#ifdef REM2D_STATS
        sim.st = EpisodeStats{end_reason.data(), max_x.data(), joint_work.data(), airborne_ticks.data(), ground_ticks.data(), pop->body_off};
        sim.st_c = -1;
#endif
    }
    // -1: a creature index out of range, -3: a creature larger than the class
    int check(const int32_t* creatures, int n) const {
        for (int i = 0; i < n; ++i) {
            const int c = creatures[i];
            if (c < 0 || c >= pop->n_creatures) return -1;
            if (pop->body_off[c + 1] - pop->body_off[c] > L.nb) return -3;
        }
        return 0;
    }
    // The leader of the group that ran creature c writes its outputs from the group's cold column after the creature's last tick.
    void decode(Sim& sim, int c, EmuOut* out) {
        const float* g = sim.g;
        auto S = [&](int f) { return __float_as_int(g[f * 32]); };
        auto B = [&](int f, int b) { return g[(S_COUNT + b * BF_COUNT + f) * 32]; };
        auto J = [&](int f, int j) { return g[(L.off_joint + j * JF_COUNT + f) * 32]; };
        auto C = [&](int f, int q) { return g[(L.off_cont + q * CF_COUNT + f) * 32]; };
        const int b0 = pop->body_off[c], nb = pop->body_off[c + 1] - b0, j0 = b0 - c;
        for (int b = 0; b < nb; ++b)
            for (int f = 0; f < 3; ++f) { put(out->pose, 3 * (b0 + b) + f, B(BF_CX + f, b)); put(out->vel, 3 * (b0 + b) + f, B(BF_VX + f, b)); }
        for (int j = 0; j < nb - 1; ++j) {
            const int fields[4] = {JF_IMPX, JF_IMPY, JF_IMPZ, JF_MIMP};
            for (int f = 0; f < 4; ++f) put(out->joint_impulse, 4 * (j0 + j) + f, J(fields[f], j));
            put(out->limit_state, j0 + j, __float_as_int(J(JF_LIMIT, j)));
            put(out->motor_speed, j0 + j, J(JF_MSPEED, j));
        }
        put(out->alive, c, S(S_ALIVE)); put(out->ticks, c, S(S_TICKS)); put(out->status, c, S(S_STATUS));
        put(out->fitness, c, __hiloint2double(S(S_FIT_HI), S(S_FIT_LO)));
        put(out->wod, c, __hiloint2double(S(S_WOD_HI), S(S_WOD_LO)));
        put(out->sched_P, c, sim.sched_P); put(out->sched_smax, c, sim.sched_smax); put(out->finish_gs, c, sim.gs);
        // touching contacts in the order of rem2d_read_state: by (body, edge)
        const int nc = S(S_NC);
        std::vector<std::pair<int, int>> pairs;
        for (int q = 0; q < nc; ++q) {
            const int key = __float_as_int(C(CF_KEY, q));
            if ((key >> 16) & CK_TOUCHING) pairs.push_back({((key & 0xff) << 8) | ((key >> 8) & 0xff), q});
        }
        std::sort(pairs.begin(), pairs.end());
        put(out->n_contacts, c, nc); put(out->n_touching, c, (int32_t)pairs.size());
        for (int q = 0; q < out->max_pairs; ++q) {
            int32_t tp[2] = {-1, -1}; float ti[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            if (q < (int)pairs.size()) {
                const int pq = pairs[q].second, key = __float_as_int(C(CF_KEY, pq)), count = (key >> (16 + CK_COUNT_SHIFT)) & 3;
                tp[0] = key & 0xff; tp[1] = (key >> 8) & 0xff;
                ti[0] = C(CF_P0N, pq); ti[1] = count > 1 ? C(CF_P1N, pq) : 0.0f; ti[2] = C(CF_P0T, pq); ti[3] = count > 1 ? C(CF_P1T, pq) : 0.0f;
            }
            const size_t at = (size_t)c * out->max_pairs + q;
            for (int i = 0; i < 2; ++i) put(out->touching_pairs, 2 * at + i, tp[i]);
            for (int i = 0; i < 4; ++i) put(out->touching_impulse, 4 * at + i, ti[i]);
        }
        std::vector<float> angle(nb), speed(nb), root(6); std::vector<int32_t> ground(nb);
        observe_column(g, L, nb, angle.data(), speed.data(), root.data(), ground.data());
        for (int j = 0; j < nb - 1; ++j) { put(out->joint_angle, j0 + j, angle[j]); put(out->joint_speed, j0 + j, speed[j]); }
        for (int i = 0; i < 6; ++i) put(out->root, 6 * (size_t)c + i, root[i]);
        for (int b = 0; b < nb; ++b) put(out->ground, b0 + b, ground[b]);
#ifdef REM2D_STATS
        put(out->end_reason, c, end_reason[c]); put(out->max_x, c, max_x[c]); put(out->joint_work, c, joint_work[c]);
        put(out->airborne_ticks, c, airborne_ticks[c]);
        for (int b = 0; b < nb; ++b) put(out->ground_ticks, b0 + b, ground_ticks[b0 + b]);
#endif
    }
};

// Runs body(lane) on n_lanes host threads, the lanes of one warp; returns the sum of the lanes' work counters.
static void run_lanes(int n_lanes, EmuOut* out, const std::function<void(Sim&, int)>& body) {
    emu::Warp warp;
    std::vector<Cnt> cnts(n_lanes);
    std::vector<std::thread> th;
    for (int l = 0; l < n_lanes; ++l)
        th.emplace_back([&, l]() {
            emu::Ctx ctx; ctx.warp = &warp; ctx.lane = l; memset(ctx.local_sense, 0, sizeof(ctx.local_sense));
            emu::ctx = &ctx;
            Sim sim;
            body(sim, l);
            cnts[l] = sim.cnt;
        });
    for (auto& t : th) t.join();
    for (int i = 0; i < REM2D_N_COUNTERS && out->counters; ++i) { uint64_t v = 0; for (auto& c : cnts) v += c.c[i]; out->counters[i] = v; }
    if (out->n_syncs) *out->n_syncs = warp.n_syncs.load();
}

// Stepping: `creatures` (at most 32 >> gs), built at tick 0 and then driven by n_calls launches of ticks_per_call ticks, like
// rem2d_reset + n_calls x rem2d_step (rem2d_step_targets in the targets build: call i holds targets[i], [n_calls][n_joints of
// the table]). The targets build requires targets, the others reject them.
EMU_API int rem2d_emu_step(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg,
                           int NB, int NC, int NT, int gs, const int32_t* creatures, int n, const double* targets, int n_calls,
                           int ticks_per_call, EmuOut* out) {
#ifdef REM2D_TARGETS
    if (!targets) return -1;
#else
    if (targets) return -1;
#endif
    if (gs < 0 || gs > 5 || n < 1 || n > (32 >> gs) || n_calls < 0 || ticks_per_call < 0) return -1;
    World w(pop, terrain_y, n_vertices, step, cfg, NB, NC, NT, gs);
    if (int rc = w.check(creatures, n)) return rc;
    run_lanes(n << gs, out, [&](Sim& sim, int lane) {
        w.init(sim, gs, lane);
        const int c = creatures[lane >> gs];
        sim.build_world(w.dp, c);
#ifdef REM2D_STATS
        sim.stats_begin(c);
        sim.st_c = c;
#endif
        for (int call = 0; call < n_calls; ++call) {
#ifdef REM2D_TARGETS
            // as step_kernel_targets: one launch per call, the creature's joint targets located through body_off
            sim.nb = sim.Si(S_NB); sim.nj = sim.nb - 1;
            sim.tgt = targets + (size_t)call * pop->n_joints + (pop->body_off[c] - c);
#endif
            for (int t = 0; t < ticks_per_call; ++t) {
                if (!sim.bcast(sim.Si(S_ALIVE))) break;
                sim.tick();
            }
#ifdef REM2D_TARGETS
            sim.gsync();
#endif
        }
        if (sim.leader()) w.decode(sim, c, out);
    });
    return 0;
}

// One warp of the queue-mode episode kernel (Sim::episodes, parking off): the creatures `order` are pulled in that order by
// groups of 1 << gs lanes, which widen up to max_gs as the warp drains, and run until their episode ends or max_ticks.
EMU_API int rem2d_emu_queue(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg,
                            int NB, int NC, int NT, int gs, int max_gs, const int32_t* order, int n_order, int max_ticks, EmuOut* out) {
    if (gs < 0 || gs > 5 || max_gs < gs || max_gs > 5 || n_order < 0) return -1;
    World w(pop, terrain_y, n_vertices, step, cfg, NB, NC, NT, gs);
    if (int rc = w.check(order, n_order)) return rc;
    const size_t n = std::max(pop->n_creatures, 1);
    std::vector<double> fitness(n); std::vector<int32_t> ticks(n), alive(n), status(n);      // what Q writes; decode reports it
    int queue = 0;
    const EpisodeQueue Q{order, n_order, &queue, w.dp, max_ticks, fitness.data(), ticks.data(), alive.data(), status.data()};
    const ParkPolicy off = {0, 0, 0.0f, 0, n_order, 0, nullptr, nullptr, 0};
    int32_t n_seq = 0;
    if (out->max_seq > 0) put(out->gs_seq, n_seq++, gs);
    struct Hooks {
        World& w; EmuOut* out; int32_t& n_seq;
        void sample(Sim&, int, unsigned) {}
        void regrouped(Sim& sim, int) { if (emu::ctx->lane == 0 && n_seq < out->max_seq) put(out->gs_seq, n_seq++, sim.gs); }
        void finished(Sim& sim, int my, int, int) { w.decode(sim, my, out); }
        unsigned now_us() { return 0u; }
    };
    run_lanes(32, out, [&](Sim& sim, int lane) {
        w.init(sim, gs, lane);
        Hooks hooks{w, out, n_seq};
        sim.episodes(lane, false, max_gs, w.hot.data(), Q, off, nullptr, nullptr, nullptr, -1, -1, hooks);
    });
    put(out->n_seq, 0, n_seq);
    return 0;
}

EMU_API int rem2d_emu_hot_rows(int NB, int NC, int NT, int gs) { return make_hot_layout(make_layout(NB, NC, NT), gs).rows; }

// The capacity classes of the CUDA library: out[4 * k ..] = {nb, nc, nt, gs} of class k. Returns the number of classes.
EMU_API int rem2d_emu_classes(int32_t* out) {
    for (int k = 0; k < N_CLASSES; ++k) {
        out[4 * k] = class_dims[k].nb; out[4 * k + 1] = class_dims[k].nc; out[4 * k + 2] = class_dims[k].nt; out[4 * k + 3] = class_dims[k].gs;
    }
    return N_CLASSES;
}

// The episode planner of the CUDA library (plan_upload, plan_launch, step_group_shift) for the given device and class sizes.
// opt[] holds the Options fields the planner reads, in the order warp_mode_max, park_ticks, park_cap, overflow_wave, image,
// smem_budget_kb, group_shift, class_gs[0..N_CLASSES); NaN keeps the default. out = {image, all_fit, warp_mode, park_ticks}
// followed by N_CLASSES values each of gs, grid, grid2, park_cap, order and the stepping kernels' group shift.
EMU_API int rem2d_emu_plan(int n_sms, const int32_t* max_warps_per_sm, const int32_t* members, const double* work,
                           const double* opt, int max_ticks, int32_t* out) {
    PlanInput in;
    in.n_sms = n_sms;
    for (int i = 0; i < 2; ++i) in.max_warps_per_sm[i] = max_warps_per_sm[i];
    for (int k = 0; k < N_CLASSES; ++k) { in.members[k] = members[k]; in.work[k] = work[k]; }
    Options o;
    auto set = [&](int i, auto& field) { if (!std::isnan(opt[i])) field = opt[i]; };
    set(0, o.warp_mode_max); set(1, o.park_ticks); set(2, o.park_cap); set(3, o.overflow_wave); set(4, o.image);
    set(5, o.smem_budget_kb); set(6, o.group_shift);
    for (int k = 0; k < N_CLASSES; ++k) set(7 + k, o.class_gs[k]);
    const UploadPlan up = plan_upload(in, o);
    const LaunchPlan lp = plan_launch(in, up, max_ticks, o);
    out[0] = up.image; out[1] = up.all_fit; out[2] = lp.warp_mode; out[3] = lp.park_ticks;
    for (int k = 0; k < N_CLASSES; ++k) {
        int32_t* col = out + 4 + k;
        col[0] = up.gs[k]; col[N_CLASSES] = up.grid[k]; col[2 * N_CLASSES] = up.grid2[k]; col[3 * N_CLASSES] = lp.park_cap[k];
        col[4 * N_CLASSES] = lp.order[k]; col[5 * N_CLASSES] = step_group_shift(in, k, o);
    }
    return 0;
}
