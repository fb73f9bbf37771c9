// rem2d_emu_control.cpp — TEST INFRASTRUCTURE: the device code of step_kernel_targets (-DREM2D_TARGETS) and the observation
// gather of observations_kernel (rem2d::observe_column) on the CPU, through the emulation shim of tests/emu (one host thread per
// lane). One call = one warp: up to 32 >> gs creatures, a group of 1 << gs lanes each, built at tick 0 and then driven by
// n_calls target calls of ticks_per_call ticks each, like rem2d_reset + n_calls x rem2d_step_targets. Build:
// make -C tests/control_emu. Used by tests/test_closed_loop.py only.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>
#include <algorithm>

#define REM2D_EMU 1
#define REM2D_TARGETS 1
#include "../../gym_rem2d_b200/csrc/rem2d_device.cuh"
#include "../../gym_rem2d_b200/csrc/rem2d_host_util.h"

thread_local emu::Ctx* emu::ctx = nullptr;
using namespace rem2d;

struct EmuControlOut {           // caller-allocated, indexed like the table (creature, body, joint)
    double* fitness; int32_t* ticks; int32_t* alive;
    float* pose; float* vel; float* joint_impulse; float* motor_speed;
    float* joint_angle; float* joint_speed; float* root; int32_t* ground;
    uint64_t* counters;                                                      // [REM2D_N_COUNTERS]
};

// targets: [n_calls][n_joints of the table]; call i holds targets[i] for ticks_per_call ticks
extern "C" int rem2d_emu_control_step(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg,
                                      int NB, int NC, int NT, int gs, const int32_t* creatures, int n, const double* targets, int n_calls,
                                      int ticks_per_call, EmuControlOut* out) {
    const int G = 1 << gs;
    if (gs < 0 || gs > 5 || n < 1 || n > (32 >> gs) || n_calls < 0 || ticks_per_call < 0) return -1;
    for (int i = 0; i < n; ++i) {
        const int c = creatures[i];
        if (c < 0 || c >= pop->n_creatures) return -1;
        if (pop->body_off[c + 1] - pop->body_off[c] > NB) return -3;
    }
    const Layout L = make_layout(NB, NC, NT);
    std::vector<float> cold((size_t)L.words * 32, 0.0f), hot((size_t)make_hot_layout(L, gs).rows * 32, 0.0f);
    Terrain ter; fill_terrain(&ter, terrain_y, n_vertices, step);
    Consts k = make_consts(cfg);
    std::vector<uint8_t> order((size_t)std::max(pop->n_joints, 1), 0);
    for (int c = 0; c < pop->n_creatures; ++c) {
        int nb = pop->body_off[c + 1] - pop->body_off[c], j0 = pop->body_off[c] - c;
        island_joint_order(nb, pop->joint_parent + j0, order.data() + j0);
    }
    DevPop dp;
    dp.body_off = pop->body_off; dp.shape = pop->shape; dp.hx = pop->hx; dp.hy = pop->hy; dp.x0 = pop->x0; dp.y0 = pop->y0; dp.a0 = pop->a0;
    dp.joint_parent = pop->joint_parent; dp.anchor_a = pop->anchor_a; dp.anchor_b = pop->anchor_b; dp.lower = pop->lower; dp.upper = pop->upper;
    dp.max_torque = pop->max_torque; dp.ctrl = pop->ctrl; dp.joint_order = order.data();

    emu::Warp warp;
    const int n_lanes = n * G;
    std::vector<Cnt> cnts(n_lanes);
    auto lane_main = [&](int lane) {
        emu::Ctx ctx; ctx.warp = &warp; ctx.lane = lane; memset(ctx.local_sense, 0, sizeof(ctx.local_sense));
        emu::ctx = &ctx;
        Sim sim;
        sim.L = L; sim.set_group(gs, lane, hot.data());
        sim.g = cold.data() + (lane >> gs);
        sim.ter = &ter; sim.k = &k;
        for (int i = 0; i < REM2D_N_COUNTERS; ++i) sim.cnt.c[i] = 0u;
        const int c = creatures[lane >> gs];
        sim.build_world(dp, c);
        // as step_kernel_targets: one launch per call, the creature's joint targets located through body_off
        for (int call = 0; call < n_calls; ++call) {
            sim.nb = sim.Si(S_NB); sim.nj = sim.nb - 1;
            sim.tgt = targets + (size_t)call * pop->n_joints + (pop->body_off[c] - c);
            for (int t = 0; t < ticks_per_call; ++t) {
                if (!sim.bcast(sim.Si(S_ALIVE))) break;
                sim.tick();
            }
            sim.gsync();
        }
        cnts[lane] = sim.cnt;
    };
    std::vector<std::thread> th;
    for (int l = 0; l < n_lanes; ++l) th.emplace_back(lane_main, l);
    for (auto& t : th) t.join();

    for (int i = 0; i < REM2D_N_COUNTERS; ++i) { uint64_t v = 0; for (auto& c : cnts) v += c.c[i]; out->counters[i] = v; }
    for (int i = 0; i < n; ++i) {
        const float* g = cold.data() + i;
        auto B = [&](int f, int b) { return g[(S_COUNT + b * BF_COUNT + f) * 32]; };
        auto J = [&](int f, int j) { return g[(L.off_joint + j * JF_COUNT + f) * 32]; };
        const int c = creatures[i], b0 = pop->body_off[c], nb = pop->body_off[c + 1] - b0, j0 = b0 - c;
        for (int b = 0; b < nb; ++b) {
            float* p = &out->pose[3 * (b0 + b)]; float* v = &out->vel[3 * (b0 + b)];
            p[0] = B(BF_CX, b); p[1] = B(BF_CY, b); p[2] = B(BF_A, b);
            v[0] = B(BF_VX, b); v[1] = B(BF_VY, b); v[2] = B(BF_W, b);
        }
        for (int j = 0; j < nb - 1; ++j) {
            float* o = &out->joint_impulse[4 * (j0 + j)];
            o[0] = J(JF_IMPX, j); o[1] = J(JF_IMPY, j); o[2] = J(JF_IMPZ, j); o[3] = J(JF_MIMP, j);
            out->motor_speed[j0 + j] = J(JF_MSPEED, j);
        }
        out->alive[c] = __float_as_int(g[S_ALIVE * 32]); out->ticks[c] = __float_as_int(g[S_TICKS * 32]);
        out->fitness[c] = __hiloint2double(__float_as_int(g[S_FIT_HI * 32]), __float_as_int(g[S_FIT_LO * 32]));
        observe_column(g, L, nb, out->joint_angle + j0, out->joint_speed + j0, out->root + (size_t)c * 6, out->ground + b0);
    }
    return 0;
}
