// rem2d_emu.cpp — TEST INFRASTRUCTURE: runs gym_rem2d_b200/csrc/rem2d_device.cuh (the device code of the CUDA kernels) on
// the CPU, one host thread per lane of a warp (see rem2d_emu_shim.h), so that the lane-group logic can be compared with the
// oracle without a GPU. One call = one warp: up to 32 >> gs creatures, each owned by a group of 1 << gs lanes, stepped like
// rem2d_step (reset + n ticks). Also exports the capacity classes and the episode planner of rem2d_host_util.h. Build:
// make -C tests/emu. Used by tests/emu/emu.py only.
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

struct EmuOut {                  // caller-allocated, concatenated over the creatures of the call in call order
    float* pose; float* vel; float* joint_impulse; int32_t* limit_state; float* motor_speed;
    int32_t* alive; int32_t* ticks; double* fitness; double* wod; int32_t* n_contacts; int32_t* n_touching;
    int32_t* touching_pairs; float* touching_impulse; int32_t max_pairs;     // like rem2d_state_view
    int32_t* sched_P; int32_t* sched_smax;                                   // [n] schedule of the last tick (diagnostics)
    uint64_t* counters;                                                      // [REM2D_N_COUNTERS]
    int64_t* n_syncs;                                                        // barriers executed by the warp
};

extern "C" int rem2d_emu_hot_rows(int NB, int NC, int NT, int gs) { return make_hot_layout(make_layout(NB, NC, NT), gs).rows; }

// The capacity classes of the CUDA library: out[4 * k ..] = {nb, nc, nt, gs} of class k. Returns the number of classes.
extern "C" int rem2d_emu_classes(int32_t* out) {
    for (int k = 0; k < N_CLASSES; ++k) {
        out[4 * k] = class_dims[k].nb; out[4 * k + 1] = class_dims[k].nc; out[4 * k + 2] = class_dims[k].nt; out[4 * k + 3] = class_dims[k].gs;
    }
    return N_CLASSES;
}

// The episode planner of the CUDA library (plan_upload, plan_launch, step_group_shift) for the given device and class sizes.
// opt[] holds the Options fields the planner reads, in the order warp_mode_max, park_ticks, park_cap, overflow_wave, image,
// smem_budget_kb, group_shift, class_gs[0..N_CLASSES); NaN keeps the default. out = {image, all_fit, warp_mode, park_ticks}
// followed by N_CLASSES values each of gs, grid, grid2, park_cap, order and the stepping kernels' group shift.
extern "C" int rem2d_emu_plan(int n_sms, const int32_t* max_warps_per_sm, const int32_t* members, const double* work,
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

extern "C" int rem2d_emu_run(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg,
                             int NB, int NC, int NT, int gs, const int32_t* creatures, int n, int n_ticks, EmuOut* out) {
    const int G = 1 << gs;
    if (n < 1 || n > (32 >> gs)) return -1;
    const Layout L = make_layout(NB, NC, NT);
    const HotLayout H = make_hot_layout(L, gs);
    for (int i = 0; i < n; ++i) {
        int c = creatures[i];
        if (c < 0 || c >= pop->n_creatures) return -1;
        if (pop->body_off[c + 1] - pop->body_off[c] > NB) return -3;
    }
    std::vector<float> cold((size_t)L.words * 32, 0.0f), hot((size_t)H.rows * 32, 0.0f);
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
    std::vector<int> sP(n_lanes, 0), sS(n_lanes, 0);
    auto lane_main = [&](int lane) {
        emu::Ctx ctx; ctx.warp = &warp; ctx.lane = lane; memset(ctx.local_sense, 0, sizeof(ctx.local_sense));
        emu::ctx = &ctx;
        Sim sim;
        sim.L = L; sim.set_group(gs, lane, hot.data());
        sim.g = cold.data() + (lane >> gs);
        sim.ter = &ter; sim.k = &k;
        for (int i = 0; i < REM2D_N_COUNTERS; ++i) sim.cnt.c[i] = 0u;
        sim.build_world(dp, creatures[lane >> gs]);
        for (int t = 0; t < n_ticks; ++t) {
            if (!sim.bcast(sim.Si(S_ALIVE))) break;
            sim.tick();
        }
        cnts[lane] = sim.cnt; sP[lane] = sim.sched_P; sS[lane] = sim.sched_smax;
    };
    std::vector<std::thread> th;
    for (int l = 0; l < n_lanes; ++l) th.emplace_back(lane_main, l);
    for (auto& t : th) t.join();

    for (int i = 0; i < REM2D_N_COUNTERS; ++i) { uint64_t v = 0; for (auto& c : cnts) v += c.c[i]; out->counters[i] = v; }
    if (out->n_syncs) *out->n_syncs = warp.n_syncs.load();
    auto asint = [](float f) { int i; memcpy(&i, &f, 4); return i; };
    int bo = 0, jo = 0;
    for (int i = 0; i < n; ++i) {
        const float* g = cold.data() + i;
        auto S = [&](int f) { return g[f * 32]; };
        auto B = [&](int f, int b) { return g[(S_COUNT + b * BF_COUNT + f) * 32]; };
        auto J = [&](int f, int j) { return g[(L.off_joint + j * JF_COUNT + f) * 32]; };
        auto C = [&](int f, int q) { return g[(L.off_cont + q * CF_COUNT + f) * 32]; };
        const int c = creatures[i], nb = pop->body_off[c + 1] - pop->body_off[c];
        for (int b = 0; b < nb; ++b) {
            out->pose[3 * (bo + b)] = B(BF_CX, b); out->pose[3 * (bo + b) + 1] = B(BF_CY, b); out->pose[3 * (bo + b) + 2] = B(BF_A, b);
            out->vel[3 * (bo + b)] = B(BF_VX, b); out->vel[3 * (bo + b) + 1] = B(BF_VY, b); out->vel[3 * (bo + b) + 2] = B(BF_W, b);
        }
        for (int j = 0; j < nb - 1; ++j) {
            float* o = &out->joint_impulse[4 * (jo + j)];
            o[0] = J(JF_IMPX, j); o[1] = J(JF_IMPY, j); o[2] = J(JF_IMPZ, j); o[3] = J(JF_MIMP, j);
            out->limit_state[jo + j] = asint(J(JF_LIMIT, j));
            out->motor_speed[jo + j] = J(JF_MSPEED, j);
        }
        out->alive[i] = asint(S(S_ALIVE)); out->ticks[i] = asint(S(S_TICKS));
        { int lo = asint(S(S_FIT_LO)), hi = asint(S(S_FIT_HI)); uint64_t u = ((uint64_t)(uint32_t)hi << 32) | (uint32_t)lo; memcpy(&out->fitness[i], &u, 8); }
        { int lo = asint(S(S_WOD_LO)), hi = asint(S(S_WOD_HI)); uint64_t u = ((uint64_t)(uint32_t)hi << 32) | (uint32_t)lo; memcpy(&out->wod[i], &u, 8); }
        int nc = asint(S(S_NC)), ntouch = 0;
        std::vector<std::pair<int, int>> pairs;
        for (int q = 0; q < nc; ++q) {
            int key = asint(C(CF_KEY, q));
            if (!((key >> 16) & CK_TOUCHING)) continue;
            ++ntouch;
            pairs.push_back({((key & 0xff) << 8) | ((key >> 8) & 0xff), q});
        }
        out->n_contacts[i] = nc; out->n_touching[i] = ntouch;
        std::sort(pairs.begin(), pairs.end());
        for (int q = 0; q < out->max_pairs; ++q) {
            int32_t* tp = &out->touching_pairs[((size_t)i * out->max_pairs + q) * 2];
            float* ti = &out->touching_impulse[((size_t)i * out->max_pairs + q) * 4];
            tp[0] = tp[1] = -1; ti[0] = ti[1] = ti[2] = ti[3] = 0.0f;
            if (q < (int)pairs.size()) {
                int pq = pairs[q].second, key = asint(C(CF_KEY, pq));
                int count = (key >> (16 + CK_COUNT_SHIFT)) & 3;
                tp[0] = key & 0xff; tp[1] = (key >> 8) & 0xff;
                ti[0] = C(CF_P0N, pq); ti[1] = count > 1 ? C(CF_P1N, pq) : 0.0f; ti[2] = C(CF_P0T, pq); ti[3] = count > 1 ? C(CF_P1T, pq) : 0.0f;
            }
        }
        out->sched_P[i] = sP[i * G]; out->sched_smax[i] = sS[i * G];
        bo += nb; jo += nb - 1;
    }
    return 0;
}
