// rem2d_kernels.cu — the three kernels of the hot path (reset, step, episode with its queue and tail modes). Compiled once per
// kernel (-DREM2D_KERNEL_ID=0..2) so the translation units build in parallel; every capacity class and every group size runs the
// same code with its own Layout and group shift (kernel parameters). REM2D_KERNEL_ID=3 compiles the episode kernel once more
// with the episode statistics (REM2D_STATS): two more images, launched only by evaluations that record statistics, so that
// the images of every other evaluation stay exactly what they are without them. REM2D_KERNEL_ID=4 compiles the step kernel once
// more with caller-supplied joint targets (REM2D_TARGETS, include/rem2d_control.h): step_kernel_targets, launched only by
// rem2d_step_targets, so that step_kernel stays exactly what it is. REM2D_KERNEL_ID=5 compiles the episode kernel with the
// per-joint feedback policy and the statistics (REM2D_POLICY, include/rem2d_policy.h): episode_kernel_policy and its
// 128-register twin, launched only by evaluations of a population uploaded with a policy (with statistics off, the host points
// the statistics at scratch); REM2D_KERNEL_ID=6 compiles the step kernel with the policy: step_kernel_policy.
//
// Lane mapping (all kernels): a warp holds 32 >> gs creatures, each owned by a group of G = 1 << gs lanes (rem2d_device.cuh).
// Cold state: blocks of 32 creature columns; creature column q lives in block q >> 5, column q & 31.
#include <cstdlib>
#if REM2D_KERNEL_ID == 3
#define REM2D_STATS 1
#endif
#if REM2D_KERNEL_ID == 4
#define REM2D_TARGETS 1
#endif
#if REM2D_KERNEL_ID == 5
#define REM2D_STATS 1
#define REM2D_POLICY 1
#endif
#if REM2D_KERNEL_ID == 6
#define REM2D_POLICY 1
#endif
#include "rem2d_classes.h"

using namespace rem2d;

#ifdef REM2D_PHASE_TIMING      // the kernels time their own loop phases through the Sim's accumulators
#undef PHASE
#define PHASE(i) do { long long t_ = clock64(); sim.ph[sim.phase_cur] += t_ - sim.phase_t0; sim.phase_t0 = t_; sim.phase_cur = (i); } while (0)
#endif

#if REM2D_KERNEL_ID == 0
// Build the world of every creature of a class (static creature -> column mapping, used by rem2d_step).
__global__ void __launch_bounds__(32) reset_kernel(const __grid_constant__ Layout L, int gs, float* state, const int* __restrict__ lane_creature,
                                                   int n_columns, DevPop p) {
    const int lane = threadIdx.x;
    const int q = blockIdx.x * (32 >> gs) + (lane >> gs);
    if (q >= n_columns) return;                                  // (whole groups: n_columns is a multiple of 32)
    Sim sim;
    sim.L = L; sim.set_group(gs, lane, nullptr);
    sim.g = state + (size_t)(q >> 5) * L.words * 32 + (q & 31);
#ifdef REM2D_PHASE_TIMING
    for (int i = 0; i < REM2D_N_PHASES; ++i) sim.ph[i] = 0;
    sim.phase_t0 = clock64(); sim.phase_cur = PH_LOOP;
#endif
    sim.build_world(p, lane_creature[q]);
}
void rem2d_launch_reset(const Layout& L, int gs, int n_batches, cudaStream_t st, float* state, const int* lane_creature, DevPop p) {
    reset_kernel<<<n_batches << gs, 32, 0, st>>>(L, gs, state, lane_creature, n_batches * 32, p);
}
#endif

#if REM2D_KERNEL_ID == 1 || REM2D_KERNEL_ID == 4 || REM2D_KERNEL_ID == 6
#if defined(REM2D_TARGETS)
#define STEP_KERNEL step_kernel_targets
#elif defined(REM2D_POLICY)
#define STEP_KERNEL step_kernel_policy
#else
#define STEP_KERNEL step_kernel
#endif
// Each group advances its creature by up to n_ticks ticks. The targets image takes the controller output of global joint j from
// targets[j]; lane_creature and body_off locate the creature's first joint. The policy image locates the weights of the
// creature's joints through lane_creature and the policy's body_off.
__global__ void __launch_bounds__(32, 1) STEP_KERNEL(const __grid_constant__ Layout L, int gs, float* state, int n_ticks,
                                                     const Terrain* __restrict__ ter, const Consts* __restrict__ k,
                                                     unsigned long long* counters
#ifdef REM2D_TARGETS
                                                     , const int* __restrict__ lane_creature, const int32_t* __restrict__ body_off,
                                                     const double* __restrict__ targets
#endif
#ifdef REM2D_POLICY
                                                     , const int* __restrict__ lane_creature, const __grid_constant__ PolicyWeights pol
#endif
                                                     ) {
    extern __shared__ float hot[];
    const int lane = threadIdx.x;
    const int q = blockIdx.x * (32 >> gs) + (lane >> gs);
    Sim sim;
    sim.L = L; sim.set_group(gs, lane, hot);
    sim.g = state + (size_t)(q >> 5) * L.words * 32 + (q & 31);
    sim.ter = ter; sim.k = k;
#pragma unroll
    for (int i = 0; i < REM2D_N_COUNTERS; ++i) sim.cnt.c[i] = 0u;
    sim.nb = sim.Si(S_NB); sim.nj = sim.nb - 1;
#ifdef REM2D_TARGETS
    if (sim.nb > 0) { const int c = lane_creature[q]; sim.tgt = targets + (body_off[c] - c); }   // (padding columns: nb = 0)
#endif
#ifdef REM2D_POLICY
    sim.pol = pol;
    if (sim.nb > 0) sim.set_policy_creature(lane_creature[q]);                                  // (padding columns: nb = 0)
#endif
#ifdef REM2D_PHASE_TIMING
    for (int i = 0; i < REM2D_N_PHASES; ++i) sim.ph[i] = 0;
    sim.phase_t0 = clock64(); sim.phase_cur = PH_LOOP;
#endif
    if (sim.nb > 0) {
        for (int t = 0; t < n_ticks; ++t) {
            if (!sim.bcast(sim.Si(S_ALIVE))) break;
            sim.tick();
        }
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < REM2D_N_COUNTERS; ++i) {
        unsigned long long v = sim.cnt.c[i];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0 && v) atomicAdd(&counters[i], v);
    }
}
#if REM2D_KERNEL_ID == 1
void rem2d_launch_step(const Layout& L, int gs, int n_batches, cudaStream_t st, float* state, int n_ticks, const Terrain* ter, const Consts* k,
                       unsigned long long* counters) {
    step_kernel<<<n_batches << gs, 32, make_hot_layout(L, gs).rows * 128, st>>>(L, gs, state, n_ticks, ter, k, counters);
}
#elif REM2D_KERNEL_ID == 4
void rem2d_launch_step_targets(const Layout& L, int gs, int n_batches, cudaStream_t st, float* state, int n_ticks, const Terrain* ter,
                               const Consts* k, unsigned long long* counters, const int* lane_creature, const int32_t* body_off,
                               const double* targets) {
    step_kernel_targets<<<n_batches << gs, 32, make_hot_layout(L, gs).rows * 128, st>>>(L, gs, state, n_ticks, ter, k, counters, lane_creature,
                                                                                        body_off, targets);
}
#else
void rem2d_launch_step_policy(const Layout& L, int gs, int n_batches, cudaStream_t st, float* state, int n_ticks, const Terrain* ter,
                              const Consts* k, unsigned long long* counters, const int* lane_creature, const PolicyWeights& pol) {
    step_kernel_policy<<<n_batches << gs, 32, make_hot_layout(L, gs).rows * 128, st>>>(L, gs, state, n_ticks, ter, k, counters, lane_creature,
                                                                                       pol);
}
#endif
#endif

#if REM2D_KERNEL_ID == 2 || REM2D_KERNEL_ID == 3 || REM2D_KERNEL_ID == 5
// Whole episodes, two modes of ONE kernel (one code image: co-resident warps of both modes share the instruction cache).
//
// mode 0, queue: every group pulls the next creature of its class from a queue (big creatures first), builds its world in
// the group's column of the warp's state block, ticks it until the episode ends, writes fitness / ticks and pulls the next
// one. Groups of a warp are therefore always busy until the queue drains, instead of idling until the longest-lived
// creature of a fixed batch dies; and the cold state of the resident warps stays L2-resident. Creatures that live longer
// than the park threshold are parked for mode 1. With gs = 5 and one warp per creature this is the latency-oriented
// execution of SMALL populations (every creature has its own warp from tick 0).
//
// mode 1, tail: takes over parked creatures (one per group, normally gs = 5: a whole warp per creature) and finishes them:
// the long-lived creatures bound the makespan, and a 32-lane schedule ticks a large creature several times faster than
// the throughput-oriented groups of the queue mode.
// The loop of both modes is Sim::episodes (rem2d_device.cuh, shared with the CPU emulation); once its class queue is empty, a
// warp regroups its surviving creatures into wider groups, up to the class's widest group shift (max_gs).

// Hooks of Sim::episodes: the trace samples, the phase-timing flush on a regroup and the tail traces.
struct KernelHooks {
    const ParkPolicy& park;
    unsigned long long* counters;
    int lane, mode;
    __device__ __forceinline__ unsigned now_us() {
        unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        return (unsigned)(t / 1000ull);
    }
    __device__ __forceinline__ void sample(Sim& sim, int loop_iter, unsigned live) {
        if (park.trace && lane == 0 && (loop_iter & 3) == 0 && (loop_iter >> 2) < REM2D_TRACE_SAMPLES) {
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            unsigned int* tr = park.trace + ((size_t)blockIdx.x * REM2D_TRACE_SAMPLES + (loop_iter >> 2)) * 2;
            tr[0] = now_us();
            tr[1] = (unsigned)(__popc(live) >> sim.gs) | ((unsigned)(loop_iter & 0xffff) << 8) | (smid << 24);
        }
    }
    // warp-cycles per phase as seen by lane 0, per (mode, group shift): counters[REM2D_N_COUNTERS + ((mode * 6 + gs) * 16 + phase)]
    __device__ __forceinline__ void flush_phases(Sim& sim, int gs) {
#ifdef REM2D_PHASE_TIMING
        if (lane == 0) {
            PHASE(PH_LOOP);
            for (int i = 0; i < REM2D_N_PHASES; ++i) {
                if (sim.ph[i] > 0) atomicAdd(&counters[REM2D_N_COUNTERS + (mode * 6 + gs) * REM2D_N_PHASES + i], (unsigned long long)sim.ph[i]);
                sim.ph[i] = 0;
            }
        }
#endif
    }
    __device__ __forceinline__ void regrouped(Sim& sim, int old_gs) { flush_phases(sim, old_gs); }
    __device__ __forceinline__ void finished(Sim&, int, int tslot, int loop_iter) {
        if (tslot >= 0 && park.tail_trace) {
            park.tail_trace[tslot * 4 + 2] = now_us();
            park.tail_trace[tslot * 4 + 3] = (unsigned)loop_iter;
        }
    }
};

// Dynamic shared memory: make_hot_layout(L, gs).rows * 128 B (gs = the launch's group shift; regrouping only widens, and
// never needs more rows).
// Two images of the same code that differ only in their register cap (__launch_bounds__): IMAGE 0, 200 registers (<= 9 warps per
// SM), for throughput-bound populations - every class runs one lane per creature, shared memory allows 3-12 warps per SM anyway
// and the uncapped code is ~3 % faster; IMAGE 1, 128 registers (16 warps per SM, no spills), for under-filled GPUs - the creatures
// are spread over wide lane groups and the resident-warp limit is what bounds how wide. All launches of one evaluation (queue
// and tail) use the same image, so co-resident warps still share one code image in the instruction cache.
static __device__ __forceinline__ void episode_body(const Layout& L, int gs, int max_gs, int mode, float* slots,
                                                        const int* __restrict__ order, int n_order, int* queue, DevPop p,
                                                        const Terrain* __restrict__ ter, const Consts* __restrict__ k, int max_ticks,
                                                        double* fitness, int* ticks, int* alive, int* status,
                                                        unsigned long long* counters, ParkPolicy park, float* park_state,
                                                        int* park_creature, int* park_count, int first_slot, int n_slots
#ifdef REM2D_STATS
                                                        , const EpisodeStats& stats
#endif
#ifdef REM2D_POLICY
                                                        , const PolicyWeights& pol
#endif
                                                        ) {
    extern __shared__ float hot[];
    const int lane = threadIdx.x;
    const bool tail = mode != 0;
    Sim sim;
    sim.L = L; sim.set_group(gs, lane, hot);
    sim.ter = ter; sim.k = k;
#ifdef REM2D_STATS
    sim.st = stats; sim.st_c = -1;
#endif
#ifdef REM2D_POLICY
    sim.pol = pol;
#endif
#pragma unroll
    for (int i = 0; i < REM2D_N_COUNTERS; ++i) sim.cnt.c[i] = 0u;
    int my = -1, tslot = -1;
#ifdef REM2D_PHASE_TIMING
    for (int i = 0; i < REM2D_N_PHASES; ++i) sim.ph[i] = 0;
    sim.phase_t0 = clock64(); sim.phase_cur = PH_LOOP;
#endif
    KernelHooks hooks{park, counters, lane, tail ? 1 : 0};
    const int q = blockIdx.x * (32 >> gs) + (lane >> gs);           // my group's column / park slot index
    if (tail) {
        // the slot was allocated by a queue-mode warp that may still be running: wait until its column has been published
        const int slot = first_slot + q;
        if (q < n_slots) {
            if (sim.leader()) {
                int v;
                while ((v = atomicAdd(&park_creature[slot], 0)) == 0) __nanosleep(500);
                my = v - 1;
                __threadfence();
            }
            my = sim.bcast(my);
            tslot = slot;
            if (park.tail_trace && sim.leader()) park.tail_trace[slot * 4 + 1] = hooks.now_us();
            sim.g = park_state + (size_t)(slot >> 5) * L.words * 32 + (slot & 31);
            sim.nb = sim.Si(S_NB); sim.nj = sim.nb - 1;
        } else { sim.g = nullptr; sim.nb = sim.nj = 0; }
    } else {
        sim.g = slots + (size_t)(q >> 5) * L.words * 32 + (q & 31);
    }
    const EpisodeQueue Q{order, n_order, queue, p, max_ticks, fitness, ticks, alive, status};
    sim.episodes(lane, tail, max_gs, hot, Q, park, park_state, park_creature, park_count, my, tslot, hooks);
    __syncwarp();
    hooks.flush_phases(sim, sim.gs);
#pragma unroll
    for (int i = 0; i < REM2D_N_COUNTERS; ++i) {
        unsigned long long v = sim.cnt.c[i];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0 && v) atomicAdd(&counters[i], v);
    }
}
#define EPISODE_PARAMS const __grid_constant__ Layout L, int gs, int max_gs, int mode, float* slots, const int* __restrict__ order, int n_order, int* queue, \
                       DevPop p, const Terrain* __restrict__ ter, const Consts* __restrict__ k, int max_ticks, double* fitness, int* ticks, \
                       int* alive, int* status, unsigned long long* counters, ParkPolicy park, float* park_state, int* park_creature,      \
                       int* park_count, int first_slot, int n_slots
#define EPISODE_ARGS L, gs, max_gs, mode, slots, order, n_order, queue, p, ter, k, max_ticks, fitness, ticks, alive, status, counters, park, park_state, \
                     park_creature, park_count, first_slot, n_slots
#if REM2D_KERNEL_ID == 2
__global__ void __launch_bounds__(32, 1) episode_kernel(EPISODE_PARAMS) { episode_body(EPISODE_ARGS); }
__global__ void __launch_bounds__(32, 16) episode_kernel_r128(EPISODE_PARAMS) { episode_body(EPISODE_ARGS); }
#define EPISODE_IMAGE0 episode_kernel
#define EPISODE_IMAGE1 episode_kernel_r128
#define EPISODE_FN(name) name
#define STATS_ARG
#elif REM2D_KERNEL_ID == 3
// the statistics images: the same code and register caps, the statistics' destinations as a trailing parameter
__global__ void __launch_bounds__(32, 1) episode_kernel_stats(EPISODE_PARAMS, const __grid_constant__ EpisodeStats stats) {
    episode_body(EPISODE_ARGS, stats);
}
__global__ void __launch_bounds__(32, 16) episode_kernel_stats_r128(EPISODE_PARAMS, const __grid_constant__ EpisodeStats stats) {
    episode_body(EPISODE_ARGS, stats);
}
#define EPISODE_IMAGE0 episode_kernel_stats
#define EPISODE_IMAGE1 episode_kernel_stats_r128
#define EPISODE_FN(name) name##_stats
#define STATS_ARG , *stats
#else
// the policy images: the same code and register caps, the statistics' destinations and the policy as trailing parameters
__global__ void __launch_bounds__(32, 1) episode_kernel_policy(EPISODE_PARAMS, const __grid_constant__ EpisodeStats stats,
                                                               const __grid_constant__ PolicyWeights pol) {
    episode_body(EPISODE_ARGS, stats, pol);
}
__global__ void __launch_bounds__(32, 16) episode_kernel_policy_r128(EPISODE_PARAMS, const __grid_constant__ EpisodeStats stats,
                                                                     const __grid_constant__ PolicyWeights pol) {
    episode_body(EPISODE_ARGS, stats, pol);
}
#define EPISODE_IMAGE0 episode_kernel_policy
#define EPISODE_IMAGE1 episode_kernel_policy_r128
#define EPISODE_FN(name) name##_policy
#define STATS_ARG , *stats, *policy
#endif

// Launchers: policy != nullptr launches the policy images (kernel 5's unit; stats must then point somewhere), otherwise stats ==
// nullptr launches the images without statistics (kernel 2's unit) and anything else the statistics images (kernel 3's unit), so
// that every launch of one evaluation uses the same image.
void EPISODE_FN(rem2d_launch_episode)(const Layout& L, int image, int gs, int max_gs, int grid, cudaStream_t st, float* slots, const int* order,
                                      int n_order, int* queue, DevPop p, const Terrain* ter, const Consts* k, int max_ticks, double* fitness,
                                      int* ticks, int* alive, int* status, unsigned long long* counters, ParkPolicy park, float* park_state,
                                      int* park_creature, int* park_count, const EpisodeStats* stats, const PolicyWeights* policy) {
#if REM2D_KERNEL_ID == 2
    if (policy) {
        rem2d_launch_episode_policy(L, image, gs, max_gs, grid, st, slots, order, n_order, queue, p, ter, k, max_ticks, fitness, ticks, alive,
                                    status, counters, park, park_state, park_creature, park_count, stats, policy);
        return;
    }
    if (stats) {
        rem2d_launch_episode_stats(L, image, gs, max_gs, grid, st, slots, order, n_order, queue, p, ter, k, max_ticks, fitness, ticks, alive,
                                   status, counters, park, park_state, park_creature, park_count, stats, nullptr);
        return;
    }
#endif
    const int smem = make_hot_layout(L, gs).rows * 128;
    if (image) EPISODE_IMAGE1<<<grid, 32, smem, st>>>(L, gs, max_gs, 0, slots, order, n_order, queue, p, ter, k, max_ticks, fitness, ticks, alive,
                                                      status, counters, park, park_state, park_creature, park_count, 0, 0 STATS_ARG);
    else EPISODE_IMAGE0<<<grid, 32, smem, st>>>(L, gs, max_gs, 0, slots, order, n_order, queue, p, ter, k, max_ticks, fitness, ticks, alive, status,
                                                counters, park, park_state, park_creature, park_count, 0, 0 STATS_ARG);
}
// resident CTAs (= warps) of the episode kernel per SM for a given dynamic shared-memory size: registers AND shared memory.
// image 0 / 1: the images without statistics, 2 / 3: the statistics images, 4 / 5: the policy images of the same register caps.
int EPISODE_FN(rem2d_episode_blocks_per_sm)(int image, int dyn_smem_bytes) {
#if REM2D_KERNEL_ID == 2
    if (image >= 4) return rem2d_episode_blocks_per_sm_policy(image - 4, dyn_smem_bytes);
    if (image >= 2) return rem2d_episode_blocks_per_sm_stats(image - 2, dyn_smem_bytes);
#endif
    int n = 0;
    cudaError_t e = image ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, EPISODE_IMAGE1, 32, (size_t)dyn_smem_bytes)
                          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, EPISODE_IMAGE0, 32, (size_t)dyn_smem_bytes);
    if (e != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
void EPISODE_FN(rem2d_launch_tail)(const Layout& L, int image, int gs, int max_gs, cudaStream_t st, float* park_state, int* park_creature,
                                   int first_slot, int n_parked, const Terrain* ter, const Consts* k, int max_ticks, double* fitness, int* ticks,
                                   int* alive, int* status, unsigned long long* counters, unsigned int* tail_trace, const EpisodeStats* stats,
                                   const PolicyWeights* policy) {
#if REM2D_KERNEL_ID == 2
    if (policy) {
        rem2d_launch_tail_policy(L, image, gs, max_gs, st, park_state, park_creature, first_slot, n_parked, ter, k, max_ticks, fitness, ticks,
                                 alive, status, counters, tail_trace, stats, policy);
        return;
    }
    if (stats) {
        rem2d_launch_tail_stats(L, image, gs, max_gs, st, park_state, park_creature, first_slot, n_parked, ter, k, max_ticks, fitness, ticks,
                                alive, status, counters, tail_trace, stats, nullptr);
        return;
    }
#endif
    ParkPolicy none = {0, 0, 0.0f, 0, 0, 0, nullptr, tail_trace, 0};
    const int per = 32 >> gs, grid = (n_parked + per - 1) / per, smem = make_hot_layout(L, gs).rows * 128;
    if (image) EPISODE_IMAGE1<<<grid, 32, smem, st>>>(L, gs, max_gs, 1, nullptr, nullptr, 0, nullptr, DevPop(), ter, k, max_ticks, fitness, ticks,
                                                      alive, status, counters, none, park_state, park_creature, nullptr, first_slot,
                                                      n_parked STATS_ARG);
    else EPISODE_IMAGE0<<<grid, 32, smem, st>>>(L, gs, max_gs, 1, nullptr, nullptr, 0, nullptr, DevPop(), ter, k, max_ticks, fitness, ticks, alive,
                                                status, counters, none, park_state, park_creature, nullptr, first_slot, n_parked STATS_ARG);
}
#endif

// Attributes: every translation unit sets those of its own kernel; rem2d_set_kernel_attributes (kernel 0's unit) calls all.
// All kernels that can be resident together should agree on the shared-memory carve-out of the SM: a small-smem kernel
// (tail) would otherwise pin its SMs in a large-L1 configuration and lock the big episode CTAs of other classes out
// (measured: 1.4x slower whole run when a tail kernel was resident next to the episode kernels).
cudaError_t rem2d_attr_step(int max_hot_bytes);
cudaError_t rem2d_attr_episode(int max_hot_bytes);
cudaError_t rem2d_attr_episode_stats(int max_hot_bytes);
cudaError_t rem2d_attr_step_targets(int max_hot_bytes);
cudaError_t rem2d_attr_episode_policy(int max_hot_bytes);
cudaError_t rem2d_attr_step_policy(int max_hot_bytes);
#if REM2D_KERNEL_ID == 0
cudaError_t rem2d_set_kernel_attributes(int max_hot_bytes) {
    cudaError_t e = rem2d_attr_step(max_hot_bytes);
    if (e != cudaSuccess) return e;
    if ((e = rem2d_attr_step_targets(max_hot_bytes)) != cudaSuccess) return e;
    if ((e = rem2d_attr_step_policy(max_hot_bytes)) != cudaSuccess) return e;
    if ((e = rem2d_attr_episode(max_hot_bytes)) != cudaSuccess) return e;
    if ((e = rem2d_attr_episode_stats(max_hot_bytes)) != cudaSuccess) return e;
    return rem2d_attr_episode_policy(max_hot_bytes);
}
#elif REM2D_KERNEL_ID == 1 || REM2D_KERNEL_ID == 4 || REM2D_KERNEL_ID == 6
#if REM2D_KERNEL_ID == 1
cudaError_t rem2d_attr_step(int max_hot_bytes) {
#elif REM2D_KERNEL_ID == 4
cudaError_t rem2d_attr_step_targets(int max_hot_bytes) {
#else
cudaError_t rem2d_attr_step_policy(int max_hot_bytes) {
#endif
    cudaError_t e = cudaFuncSetAttribute(STEP_KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, max_hot_bytes);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(STEP_KERNEL, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}
#elif REM2D_KERNEL_ID == 2 || REM2D_KERNEL_ID == 3 || REM2D_KERNEL_ID == 5
cudaError_t EPISODE_FN(rem2d_attr_episode)(int max_hot_bytes) {
    cudaError_t e = cudaFuncSetAttribute(EPISODE_IMAGE0, cudaFuncAttributeMaxDynamicSharedMemorySize, max_hot_bytes);
    if (e != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(EPISODE_IMAGE0, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(EPISODE_IMAGE1, cudaFuncAttributeMaxDynamicSharedMemorySize, max_hot_bytes)) != cudaSuccess) return e;
    return cudaFuncSetAttribute(EPISODE_IMAGE1, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}
#endif
