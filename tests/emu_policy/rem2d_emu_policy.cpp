// rem2d_emu_policy.cpp — TEST INFRASTRUCTURE: the device code of the policy images (-DREM2D_POLICY -DREM2D_STATS: the episode
// kernel's episode_kernel_policy*, and step_kernel_policy's tick with the statistics compiled in) on the CPU, through the
// harness of tests/emu/rem2d_emu.cpp, which is included as it is (World, run_lanes, EmuOut, decode, the planner entries).
// Its two run entries are renamed on inclusion and not used: in this build every Sim needs the policy, which they do not set.
// This unit's entries set it as the kernels do:
//  - rem2d_emu_policy_step: one warp of the stepping kernel, up to 32 >> gs creatures with a group of 1 << gs lanes each,
//    reset and then n_calls launches of ticks_per_call ticks; the weights of a creature are located through body_off at every
//    launch, as step_kernel_policy does from lane_creature;
//  - rem2d_emu_policy_queue: one warp of the queue-mode episode kernel (Sim::episodes sets the weights before every tick,
//    parking off, regrouping of a draining warp).
// weights: [n_joints of the table][10 * n_hidden + 1] (include/rem2d_policy.h). Build: make -C tests/emu_policy. Used by
// tests/emu_policy/emu_policy.py only.
#define rem2d_emu_step rem2d_emu_step_without_policy
#define rem2d_emu_queue rem2d_emu_queue_without_policy
#include "../emu/rem2d_emu.cpp"
#undef rem2d_emu_step
#undef rem2d_emu_queue

static bool policy_ok(const double* weights, int n_hidden) {
    return weights && n_hidden >= 1 && n_hidden <= REM2D_POLICY_MAX_HIDDEN;
}

EMU_API int rem2d_emu_policy_step(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg,
                                  int NB, int NC, int NT, int gs, const int32_t* creatures, int n, int n_calls, int ticks_per_call,
                                  const double* weights, int n_hidden, EmuOut* out) {
    if (gs < 0 || gs > 5 || n < 1 || n > (32 >> gs) || n_calls < 0 || ticks_per_call < 0 || !policy_ok(weights, n_hidden)) return -1;
    World w(pop, terrain_y, n_vertices, step, cfg, NB, NC, NT, gs);
    if (int rc = w.check(creatures, n)) return rc;
    run_lanes(n << gs, out, [&](Sim& sim, int lane) {
        w.init(sim, gs, lane);
        sim.pol = PolicyWeights{weights, pop->body_off, n_hidden};
        const int c = creatures[lane >> gs];
        sim.build_world(w.dp, c);
        sim.stats_begin(c);
        sim.st_c = c;
        for (int call = 0; call < n_calls; ++call) {
            sim.nb = sim.Si(S_NB); sim.nj = sim.nb - 1;
            sim.set_policy_creature(c);
            for (int t = 0; t < ticks_per_call; ++t) {
                if (!sim.bcast(sim.Si(S_ALIVE))) break;
                sim.tick();
            }
            sim.gsync();
        }
        if (sim.leader()) w.decode(sim, c, out);
    });
    return 0;
}

EMU_API int rem2d_emu_policy_queue(const rem2d_population* pop, const double* terrain_y, int n_vertices, double step, const rem2d_config* cfg,
                                   int NB, int NC, int NT, int gs, int max_gs, const int32_t* order, int n_order, int max_ticks,
                                   const double* weights, int n_hidden, EmuOut* out) {
    if (gs < 0 || gs > 5 || max_gs < gs || max_gs > 5 || n_order < 0 || !policy_ok(weights, n_hidden)) return -1;
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
        sim.pol = PolicyWeights{weights, pop->body_off, n_hidden};
        Hooks hooks{w, out, n_seq};
        sim.episodes(lane, false, max_gs, w.hot.data(), Q, off, nullptr, nullptr, nullptr, -1, -1, hooks);
    });
    put(out->n_seq, 0, n_seq);
    return 0;
}
