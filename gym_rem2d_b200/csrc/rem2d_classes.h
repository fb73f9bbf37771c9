// rem2d_classes.h — the launch interface of the three kernels (rem2d_kernels.cu; one translation unit per kernel so that
// they compile in parallel) and the host's per-class view of it. All classes run the SAME code: the class only selects a
// Layout (the capacity classes themselves are in rem2d_host_util.h).
#pragma once
#include <cuda_runtime.h>
#include "rem2d_device.cuh"

// When the queue-mode episode kernel hands a creature over to the tail mode (launches of the same kernel).
struct ParkPolicy {
    int ticks;        // park a creature that is still alive after this many ticks (0: never park)
    int cap;          // at most this many creatures of the class are parked
    // Always off (lead_x = 0, late_from = class size): the rejected lead and late-start park tests of the episode kernel.
    // Deleting them takes episode_kernel from 202 to 200 registers; at 200, 10 instead of 9 warps fit per SM, so the
    // occupancy-based grid sizing (size_grids, rem2d_host_util.h) hands out other first-wave grids.
    float lead_x;     // > 0: park a creature whose root has reached x >= lead_x after lead_from ticks
    int lead_from;
    int late_from;    // creatures pulled from this position of the class queue on park after late_ticks ticks
    int late_ticks;
    // diagnostics (trace option): every 4th tick lane 0 of each warp records {globaltimer us, live creatures | tick << 8 |
    // smid << 24}; REM2D_TRACE_SAMPLES entries per warp. Null in production.
    unsigned int* trace;
    unsigned int* tail_trace;   // per park slot: {us parked, us tail warp started, us finished, ticks run by the tail warp}
};
#define REM2D_TRACE_SAMPLES 1024

// Launchers (rem2d_kernels.cu).
cudaError_t rem2d_set_kernel_attributes(int max_hot_bytes);
int rem2d_episode_blocks_per_sm(int image, int dyn_smem_bytes);
void rem2d_launch_reset(const rem2d::Layout& L, int gs, int n_batches, cudaStream_t st, float* state, const int* lane_creature, rem2d::DevPop p);
void rem2d_launch_step(const rem2d::Layout& L, int gs, int n_batches, cudaStream_t st, float* state, int n_ticks, const rem2d::Terrain* ter,
                       const rem2d::Consts* k, unsigned long long* counters);
void rem2d_launch_episode(const rem2d::Layout& L, int image, int gs, int grid, cudaStream_t st, float* slots, const int* order, int n_order, int* queue,
                          rem2d::DevPop p, const rem2d::Terrain* ter, const rem2d::Consts* k, int max_ticks, double* fitness,
                          int* ticks, int* alive, int* status, unsigned long long* counters, ParkPolicy park, float* park_state,
                          int* park_creature, int* park_count);
void rem2d_launch_tail(const rem2d::Layout& L, int image, int gs, cudaStream_t st, float* park_state, int* park_creature, int first_slot,
                       int n_parked, const rem2d::Terrain* ter, const rem2d::Consts* k, int max_ticks, double* fitness, int* ticks,
                       int* alive, int* status, unsigned long long* counters, unsigned int* tail_trace);

// Per-class view used by the host code.
struct ClassOps {
    rem2d::Layout L;
    int nb, nc, nt, nj, off_body, off_joint, off_cont, off_edge, words, hot_words;
    explicit ClassOps(int NB, int NC, int NT) : L(rem2d::make_layout(NB, NC, NT)) {
        nb = L.nb; nc = L.nc; nt = L.nt; nj = L.nj; off_body = rem2d::S_COUNT; off_joint = L.off_joint; off_cont = L.off_cont;
        off_edge = L.off_edge; words = L.words; hot_words = L.hot_words;
    }
    template <class... A> void reset(A... a) const { rem2d_launch_reset(L, a...); }
    template <class... A> void step(A... a) const { rem2d_launch_step(L, a...); }
    template <class... A> void episode(A... a) const { rem2d_launch_episode(L, a...); }
    template <class... A> void tail(A... a) const { rem2d_launch_tail(L, a...); }
};
