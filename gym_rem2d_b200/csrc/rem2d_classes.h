// rem2d_classes.h — the launch interface of the three kernels (rem2d_kernels.cu; one translation unit per kernel so that
// they compile in parallel, one more for the episode kernel with statistics, one for the step kernel with joint targets and one
// each for the episode and step kernels with a feedback policy) and the host's per-class view of it. All classes run the SAME code: the class only selects a
// Layout (the capacity classes themselves are in rem2d_host_util.h).
#pragma once
#include <cuda_runtime.h>
#include "rem2d_device.cuh"

using rem2d::ParkPolicy;
using rem2d::PolicyWeights;

// Launchers (rem2d_kernels.cu). The episode and tail launchers take the statistics' destinations and the policy: a policy
// launches the policy images (rem2d_launch_*_policy, which need stats != nullptr), otherwise stats == nullptr launches the images
// without statistics and anything else the statistics images (rem2d_launch_*_stats), all called through them.
cudaError_t rem2d_set_kernel_attributes(int max_hot_bytes);
// image 0 / 1: the episode kernel images without statistics, 2 / 3: the statistics images, 4 / 5: the policy images, with the
// same register caps
int rem2d_episode_blocks_per_sm(int image, int dyn_smem_bytes);
int rem2d_episode_blocks_per_sm_stats(int image, int dyn_smem_bytes);
int rem2d_episode_blocks_per_sm_policy(int image, int dyn_smem_bytes);
void rem2d_launch_reset(const rem2d::Layout& L, int gs, int n_batches, cudaStream_t st, float* state, const int* lane_creature, rem2d::DevPop p);
void rem2d_launch_step(const rem2d::Layout& L, int gs, int n_batches, cudaStream_t st, float* state, int n_ticks, const rem2d::Terrain* ter,
                       const rem2d::Consts* k, unsigned long long* counters);
// the step kernel with caller-supplied joint targets (include/rem2d_control.h): targets[j] for global joint j, held for n_ticks
void rem2d_launch_step_targets(const rem2d::Layout& L, int gs, int n_batches, cudaStream_t st, float* state, int n_ticks,
                               const rem2d::Terrain* ter, const rem2d::Consts* k, unsigned long long* counters, const int* lane_creature,
                               const int32_t* body_off, const double* targets);
// the step kernel with the feedback policy (include/rem2d_policy.h)
void rem2d_launch_step_policy(const rem2d::Layout& L, int gs, int n_batches, cudaStream_t st, float* state, int n_ticks,
                              const rem2d::Terrain* ter, const rem2d::Consts* k, unsigned long long* counters, const int* lane_creature,
                              const PolicyWeights& pol);
void rem2d_launch_episode(const rem2d::Layout& L, int image, int gs, int max_gs, int grid, cudaStream_t st, float* slots, const int* order, int n_order, int* queue,
                          rem2d::DevPop p, const rem2d::Terrain* ter, const rem2d::Consts* k, int max_ticks, double* fitness,
                          int* ticks, int* alive, int* status, unsigned long long* counters, ParkPolicy park, float* park_state,
                          int* park_creature, int* park_count, const rem2d::EpisodeStats* stats, const PolicyWeights* policy);
void rem2d_launch_episode_stats(const rem2d::Layout& L, int image, int gs, int max_gs, int grid, cudaStream_t st, float* slots, const int* order,
                                int n_order, int* queue, rem2d::DevPop p, const rem2d::Terrain* ter, const rem2d::Consts* k, int max_ticks,
                                double* fitness, int* ticks, int* alive, int* status, unsigned long long* counters, ParkPolicy park,
                                float* park_state, int* park_creature, int* park_count, const rem2d::EpisodeStats* stats, const PolicyWeights* policy);
void rem2d_launch_tail(const rem2d::Layout& L, int image, int gs, int max_gs, cudaStream_t st, float* park_state, int* park_creature, int first_slot,
                       int n_parked, const rem2d::Terrain* ter, const rem2d::Consts* k, int max_ticks, double* fitness, int* ticks,
                       int* alive, int* status, unsigned long long* counters, unsigned int* tail_trace, const rem2d::EpisodeStats* stats,
                       const PolicyWeights* policy);
void rem2d_launch_tail_stats(const rem2d::Layout& L, int image, int gs, int max_gs, cudaStream_t st, float* park_state, int* park_creature,
                             int first_slot, int n_parked, const rem2d::Terrain* ter, const rem2d::Consts* k, int max_ticks, double* fitness,
                             int* ticks, int* alive, int* status, unsigned long long* counters, unsigned int* tail_trace,
                             const rem2d::EpisodeStats* stats, const PolicyWeights* policy);
void rem2d_launch_episode_policy(const rem2d::Layout& L, int image, int gs, int max_gs, int grid, cudaStream_t st, float* slots, const int* order,
                                 int n_order, int* queue, rem2d::DevPop p, const rem2d::Terrain* ter, const rem2d::Consts* k, int max_ticks,
                                 double* fitness, int* ticks, int* alive, int* status, unsigned long long* counters, ParkPolicy park,
                                 float* park_state, int* park_creature, int* park_count, const rem2d::EpisodeStats* stats,
                                 const PolicyWeights* policy);
void rem2d_launch_tail_policy(const rem2d::Layout& L, int image, int gs, int max_gs, cudaStream_t st, float* park_state, int* park_creature,
                              int first_slot, int n_parked, const rem2d::Terrain* ter, const rem2d::Consts* k, int max_ticks, double* fitness,
                              int* ticks, int* alive, int* status, unsigned long long* counters, unsigned int* tail_trace,
                              const rem2d::EpisodeStats* stats, const PolicyWeights* policy);

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
    template <class... A> void step_targets(A... a) const { rem2d_launch_step_targets(L, a...); }
    template <class... A> void step_policy(A... a) const { rem2d_launch_step_policy(L, a...); }
    template <class... A> void episode(A... a) const { rem2d_launch_episode(L, a...); }
    template <class... A> void tail(A... a) const { rem2d_launch_tail(L, a...); }
};
