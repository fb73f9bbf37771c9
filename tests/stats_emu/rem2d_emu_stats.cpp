// rem2d_emu_stats.cpp — TEST INFRASTRUCTURE: the device code of the statistics images of the episode kernel (-DREM2D_STATS) on
// the CPU, through the emulation shim of tests/emu (one host thread per lane). Two entries: a warp stepping its creatures from
// tick 0 like the stepping entry of tests/emu, and one warp of the queue-mode episode kernel (Sim::episodes, with regrouping) like
// tests/regroup_emu. Build: make -C tests/stats_emu. Used by tests/test_episode_stats.py only.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>
#include <algorithm>
#include <functional>

#define REM2D_EMU 1
#define REM2D_STATS 1
#include "../../gym_rem2d_b200/csrc/rem2d_device.cuh"
#include "../../gym_rem2d_b200/csrc/rem2d_host_util.h"

thread_local emu::Ctx* emu::ctx = nullptr;
using namespace rem2d;

struct EmuStatsOut {             // caller-allocated, indexed by creature (ground_ticks by body of the table)
    double* fitness; int32_t* ticks; int32_t* status;
    int32_t* end_reason; float* max_x; double* joint_work; int32_t* airborne_ticks; int32_t* ground_ticks;
};
struct World {
    Terrain ter; Consts k; std::vector<uint8_t> jorder; DevPop dp; EpisodeStats st;
    World(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg, EmuStatsOut* out) {
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
        st = EpisodeStats{out->end_reason, out->max_x, out->joint_work, out->airborne_ticks, out->ground_ticks, pop->body_off};
    }
};
static int check(const rem2d_population* pop, const int32_t* creatures, int n, int NB) {
    for (int i = 0; i < n; ++i) {
        const int c = creatures[i];
        if (c < 0 || c >= pop->n_creatures) return -1;
        if (pop->body_off[c + 1] - pop->body_off[c] > NB) return -3;
    }
    return 0;
}
static void run_lanes(int n_lanes, emu::Warp& warp, const std::function<void(int)>& body) {
    std::vector<std::thread> th;
    for (int l = 0; l < n_lanes; ++l)
        th.emplace_back([&, l]() {
            emu::Ctx ctx; ctx.warp = &warp; ctx.lane = l; memset(ctx.local_sense, 0, sizeof(ctx.local_sense));
            emu::ctx = &ctx;
            body(l);
        });
    for (auto& t : th) t.join();
}

// Stepping: up to 32 >> gs creatures, a group of 1 << gs lanes each, ticked from tick 0 until their episode ends or n_ticks.
extern "C" int rem2d_emu_stats_step(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg,
                                    int NB, int NC, int NT, int gs, const int32_t* creatures, int n, int n_ticks, EmuStatsOut* out) {
    if (gs < 0 || gs > 5 || n < 1 || n > (32 >> gs)) return -1;
    if (int rc = check(pop, creatures, n, NB)) return rc;
    const Layout L = make_layout(NB, NC, NT);
    std::vector<float> cold((size_t)L.words * 32, 0.0f), hot((size_t)make_hot_layout(L, gs).rows * 32, 0.0f);
    World w(pop, terrain_y, n_vertices, step, cfg, out);
    emu::Warp warp;
    run_lanes(n << gs, warp, [&](int lane) {
        Sim sim;
        sim.L = L; sim.set_group(gs, lane, hot.data());
        sim.g = cold.data() + (lane >> gs);
        sim.ter = &w.ter; sim.k = &w.k; sim.st = w.st;
        for (int i = 0; i < REM2D_N_COUNTERS; ++i) sim.cnt.c[i] = 0u;
        const int c = creatures[lane >> gs];
        sim.build_world(w.dp, c);
        sim.stats_begin(c);
        sim.st_c = c;
        for (int t = 0; t < n_ticks; ++t) {
            if (!sim.bcast(sim.Si(S_ALIVE))) break;
            sim.tick();
        }
        if (sim.leader()) {
            out->fitness[c] = sim.Sd(S_FIT_LO); out->ticks[c] = sim.Si(S_TICKS); out->status[c] = sim.Si(S_STATUS);
        }
    });
    return 0;
}

struct NoHooks {
    void sample(Sim&, int, unsigned) {}
    void regrouped(Sim&, int) {}
    void finished(Sim&, int, int, int) {}
    unsigned now_us() { return 0u; }
};

// One warp of the queue-mode episode kernel (parking off): the creatures `order` are pulled in that order by groups of 1 << gs
// lanes, which widen up to max_gs as the warp drains.
extern "C" int rem2d_emu_stats_queue(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg,
                                     int NB, int NC, int NT, int gs, int max_gs, const int32_t* order, int n_order, int max_ticks,
                                     EmuStatsOut* out) {
    if (gs < 0 || gs > 5 || max_gs < gs || max_gs > 5 || n_order < 0) return -1;
    if (int rc = check(pop, order, n_order, NB)) return rc;
    const Layout L = make_layout(NB, NC, NT);
    std::vector<float> cold((size_t)L.words * 32, 0.0f), hot((size_t)make_hot_layout(L, gs).rows * 32, 0.0f);
    World w(pop, terrain_y, n_vertices, step, cfg, out);
    std::vector<int32_t> alive((size_t)std::max(pop->n_creatures, 1), 0);
    int queue = 0;
    const EpisodeQueue Q{order, n_order, &queue, w.dp, max_ticks, out->fitness, out->ticks, alive.data(), out->status};
    const ParkPolicy off = {0, 0, 0.0f, 0, n_order, 0, nullptr, nullptr, 0};
    emu::Warp warp;
    run_lanes(32, warp, [&](int lane) {
        Sim sim;
        sim.L = L; sim.set_group(gs, lane, hot.data());
        sim.g = cold.data() + (lane >> gs);
        sim.ter = &w.ter; sim.k = &w.k; sim.st = w.st; sim.st_c = -1;
        for (int i = 0; i < REM2D_N_COUNTERS; ++i) sim.cnt.c[i] = 0u;
        NoHooks hooks;
        sim.episodes(lane, false, max_gs, hot.data(), Q, off, nullptr, nullptr, nullptr, -1, -1, hooks);
    });
    return 0;
}
