// rem2d_emu_queue.cpp — TEST INFRASTRUCTURE: one warp of the queue-mode episode kernel on the CPU. Runs Sim::episodes of
// gym_rem2d_b200/csrc/rem2d_device.cuh (the loop of episode_kernel, with its regrouping of draining warps) through the emulation
// shim of tests/emu, one host thread per lane. Build: make -C tests/regroup_emu. Used by tests/test_regroup.py only.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>
#include <algorithm>

#define REM2D_EMU 1
#include "../../gym_rem2d_b200/csrc/rem2d_device.cuh"
#include "../../gym_rem2d_b200/csrc/rem2d_host_util.h"

thread_local emu::Ctx* emu::ctx = nullptr;
using namespace rem2d;

static std::vector<uint8_t> joint_orders(const rem2d_population* pop) {
    std::vector<uint8_t> order((size_t)std::max(pop->n_joints, 1), 0);
    for (int c = 0; c < pop->n_creatures; ++c) {
        int nb = pop->body_off[c + 1] - pop->body_off[c], j0 = pop->body_off[c] - c;
        island_joint_order(nb, pop->joint_parent + j0, order.data() + j0);
    }
    return order;
}
static DevPop dev_pop(const rem2d_population* pop, const uint8_t* joint_order) {
    DevPop dp;
    dp.body_off = pop->body_off; dp.shape = pop->shape; dp.hx = pop->hx; dp.hy = pop->hy; dp.x0 = pop->x0; dp.y0 = pop->y0; dp.a0 = pop->a0;
    dp.joint_parent = pop->joint_parent; dp.anchor_a = pop->anchor_a; dp.anchor_b = pop->anchor_b; dp.lower = pop->lower; dp.upper = pop->upper;
    dp.max_torque = pop->max_torque; dp.ctrl = pop->ctrl; dp.joint_order = joint_order;
    return dp;
}

struct EmuQueueOut {             // caller-allocated; per-creature arrays are indexed by creature and written for the queued ones
    double* fitness; int32_t* ticks; int32_t* alive; int32_t* status;
    int32_t* finish_gs;                                          // group shift of the creature's group when its episode ended
    uint64_t* counters;                                          // [REM2D_N_COUNTERS]
    int32_t* gs_seq; int32_t max_seq; int32_t* n_seq;            // group shifts the warp ran at, in order (the first is gs)
};
struct EmuHooks {
    EmuQueueOut* out;
    void sample(Sim&, int, unsigned) {}
    void regrouped(Sim& sim, int) {
        if (emu::ctx->lane == 0 && *out->n_seq < out->max_seq) out->gs_seq[(*out->n_seq)++] = sim.gs;
    }
    void finished(Sim& sim, int my, int, int) { out->finish_gs[my] = sim.gs; }
    unsigned now_us() { return 0u; }
};

// One warp of the queue-mode episode kernel (Sim::episodes, parking off): the creatures `order` are pulled in that order by groups
// of 1 << gs lanes, which widen up to max_gs as the warp drains, and run until their episode ends or max_ticks.
extern "C" int rem2d_emu_queue(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg,
                               int NB, int NC, int NT, int gs, int max_gs, const int32_t* order, int n_order, int max_ticks,
                               EmuQueueOut* out) {
    if (gs < 0 || gs > 5 || max_gs < gs || max_gs > 5 || n_order < 0) return -1;
    for (int i = 0; i < n_order; ++i) {
        const int c = order[i];
        if (c < 0 || c >= pop->n_creatures) return -1;
        if (pop->body_off[c + 1] - pop->body_off[c] > NB) return -3;
    }
    const Layout L = make_layout(NB, NC, NT);
    std::vector<float> cold((size_t)L.words * 32, 0.0f), hot((size_t)make_hot_layout(L, gs).rows * 32, 0.0f);
    Terrain ter; fill_terrain(&ter, terrain_y, n_vertices, step);
    Consts k = make_consts(cfg);
    const std::vector<uint8_t> jorder = joint_orders(pop);
    const DevPop dp = dev_pop(pop, jorder.data());
    int queue = 0;
    const EpisodeQueue Q{order, n_order, &queue, dp, max_ticks, out->fitness, out->ticks, out->alive, out->status};
    const ParkPolicy off = {0, 0, 0.0f, 0, n_order, 0, nullptr, nullptr, 0};
    *out->n_seq = 0;
    if (out->max_seq > 0) { out->gs_seq[0] = gs; *out->n_seq = 1; }

    emu::Warp warp;
    std::vector<Cnt> cnts(32);
    auto lane_main = [&](int lane) {
        emu::Ctx ctx; ctx.warp = &warp; ctx.lane = lane; memset(ctx.local_sense, 0, sizeof(ctx.local_sense));
        emu::ctx = &ctx;
        Sim sim;
        sim.L = L; sim.set_group(gs, lane, hot.data());
        sim.g = cold.data() + (lane >> gs);               // column q = lane >> gs of the warp's block, as in the kernel
        sim.ter = &ter; sim.k = &k;
        for (int i = 0; i < REM2D_N_COUNTERS; ++i) sim.cnt.c[i] = 0u;
        EmuHooks hooks{out};
        sim.episodes(lane, false, max_gs, hot.data(), Q, off, nullptr, nullptr, nullptr, -1, -1, hooks);
        cnts[lane] = sim.cnt;
    };
    std::vector<std::thread> th;
    for (int l = 0; l < 32; ++l) th.emplace_back(lane_main, l);
    for (auto& t : th) t.join();
    for (int i = 0; i < REM2D_N_COUNTERS; ++i) { uint64_t v = 0; for (auto& c : cnts) v += c.c[i]; out->counters[i] = v; }
    return 0;
}
