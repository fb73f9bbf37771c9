// rem2d_kernels.cu — the three kernels of the hot path (reset, step, episode with its queue and tail modes). Compiled once per
// kernel (-DREM2D_KERNEL_ID=0..2) so the translation units build in parallel; every capacity class and every group size runs the
// same code with its own Layout and group shift (kernel parameters).
//
// Lane mapping (all kernels): a warp holds 32 >> gs creatures, each owned by a group of G = 1 << gs lanes (rem2d_device.cuh).
// Cold state: blocks of 32 creature columns; creature column q lives in block q >> 5, column q & 31.
#include <cstdlib>
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

#if REM2D_KERNEL_ID == 1
// Each group advances its creature by up to n_ticks ticks.
__global__ void __launch_bounds__(32, 1) step_kernel(const __grid_constant__ Layout L, int gs, float* state, int n_ticks,
                                                     const Terrain* __restrict__ ter, const Consts* __restrict__ k,
                                                     unsigned long long* counters) {
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
void rem2d_launch_step(const Layout& L, int gs, int n_batches, cudaStream_t st, float* state, int n_ticks, const Terrain* ter, const Consts* k,
                       unsigned long long* counters) {
    step_kernel<<<n_batches << gs, 32, make_hot_layout(L, gs).rows * 128, st>>>(L, gs, state, n_ticks, ter, k, counters);
}
#endif

#if REM2D_KERNEL_ID == 2
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
// Dynamic shared memory: make_hot_layout(L, gs).rows * 128 B.
// Two images of the same code that differ only in their register cap (__launch_bounds__): IMAGE 0, 200 registers (<= 9 warps per
// SM), for throughput-bound populations - every class runs one lane per creature, shared memory allows 3-12 warps per SM anyway
// and the uncapped code is ~3 % faster; IMAGE 1, 128 registers (16 warps per SM, no spills), for under-filled GPUs - the creatures
// are spread over wide lane groups and the resident-warp limit is what bounds how wide. All launches of one evaluation (queue
// and tail) use the same image, so co-resident warps still share one code image in the instruction cache.
static __device__ __forceinline__ void episode_body(const Layout& L, int gs, int mode, float* slots,
                                                        const int* __restrict__ order, int n_order, int* queue, DevPop p,
                                                        const Terrain* __restrict__ ter, const Consts* __restrict__ k, int max_ticks,
                                                        double* fitness, int* ticks, int* alive, int* status,
                                                        unsigned long long* counters, ParkPolicy park, float* park_state,
                                                        int* park_creature, int* park_count, int first_slot, int n_slots) {
    extern __shared__ float hot[];
    const int lane = threadIdx.x;
    const bool tail = mode != 0;
    Sim sim;
    sim.L = L; sim.set_group(gs, lane, hot);
    sim.ter = ter; sim.k = k;
#pragma unroll
    for (int i = 0; i < REM2D_N_COUNTERS; ++i) sim.cnt.c[i] = 0u;
    int my = -1, loop_iter = 0, park_at = park.ticks;
    bool exhausted = false;
#ifdef REM2D_PHASE_TIMING
    for (int i = 0; i < REM2D_N_PHASES; ++i) sim.ph[i] = 0;
    sim.phase_t0 = clock64(); sim.phase_cur = PH_LOOP;
#endif
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
            if (park.tail_trace && sim.leader()) {
                unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
                park.tail_trace[slot * 4 + 1] = (unsigned)(t / 1000ull);
            }
            sim.g = park_state + (size_t)(slot >> 5) * L.words * 32 + (slot & 31);
            sim.nb = sim.Si(S_NB); sim.nj = sim.nb - 1;
        } else { sim.g = nullptr; sim.nb = sim.nj = 0; }
        exhausted = true;
    } else {
        sim.g = slots + (size_t)(q >> 5) * L.words * 32 + (q & 31);
    }
    Cnt snapshot = sim.cnt;
    for (;;) {
        if (my < 0 && !exhausted) {
            int idx = 0;
            if (sim.leader()) idx = atomicAdd(queue, 1);
            idx = sim.bcast(idx);
            if (idx < n_order) {
                my = order[idx]; sim.build_world(p, my); snapshot = sim.cnt;
                park_at = idx >= park.late_from ? park.late_ticks : park.ticks;
            }
            else exhausted = true;
        }
        const unsigned live = __ballot_sync(0xffffffffu, my >= 0);
        if (park.trace && lane == 0 && (loop_iter & 3) == 0 && (loop_iter >> 2) < REM2D_TRACE_SAMPLES) {
            unsigned long long t; unsigned smid;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            unsigned int* tr = park.trace + ((size_t)blockIdx.x * REM2D_TRACE_SAMPLES + (loop_iter >> 2)) * 2;
            tr[0] = (unsigned)(t / 1000ull);
            tr[1] = (unsigned)(__popc(live) >> gs) | ((unsigned)(loop_iter & 0xffff) << 8) | (smid << 24);
        }
        ++loop_iter;
        if (!live) break;
        if (my >= 0) {                                            // group-uniform
            sim.tick();
            PHASE(PH_PARK);
            const int t = sim.Si(S_TICKS), st = sim.Si(S_STATUS), al = sim.Si(S_ALIVE);    // (written before tick()'s last group barrier)
            if (!al || t >= max_ticks || st) {
                if (sim.leader()) { fitness[my] = sim.Sd(S_FIT_LO); ticks[my] = t; alive[my] = al; status[my] = st; }
                // a creature that outgrew a capacity of this class is re-run by the host in the next class up:
                // its partial work must not be counted
                if (st) sim.cnt = snapshot;
                my = -1;
            } else if (!tail && park.ticks > 0 &&
                       (t >= park_at || (park.lead_x > 0.0f && t >= park.lead_from && sim.B(BF_CX, 0) >= park.lead_x))) {
                // long-lived creature: park its state; the latency-oriented tail mode (one warp per creature) finishes it.
                // (the counter never exceeds the cap: the host hands every counted slot to a tail launch)
                int slot = -1;
                if (sim.leader()) {
                    int seen = *(volatile int*)park_count;
                    while (seen < park.cap) {
                        const int prev = atomicCAS(park_count, seen, seen + 1);
                        if (prev == seen) { slot = seen; break; }
                        seen = prev;
                    }
                }
                slot = sim.bcast(slot);
                if (slot >= 0) {
                    float* dst = park_state + (size_t)(slot >> 5) * L.words * 32 + (slot & 31);
                    for (int w = sim.sub; w < L.words; w += sim.G) dst[w * 32] = sim.g[w * 32];
                    __threadfence();                                 // the column is visible before the slot is published
                    sim.gsync();
                    if (sim.leader()) {
                        if (park.tail_trace) {
                            unsigned long long tt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tt));
                            park.tail_trace[slot * 4] = (unsigned)(tt / 1000ull);
                        }
                        __threadfence();
                        atomicExch(&park_creature[slot], my + 1);    // 0 = allocated but not yet published
                    }
                    my = -1;
                }
            }
            sim.gsync();          // the leader's reads of this creature's scalars are done before the column is rebuilt
            PHASE(PH_LOOP);
        }
    }
    if (tail && park.tail_trace && sim.leader() && q < n_slots) {
        unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        park.tail_trace[(first_slot + q) * 4 + 2] = (unsigned)(t / 1000ull);
        park.tail_trace[(first_slot + q) * 4 + 3] = (unsigned)loop_iter - 1u;
    }
    __syncwarp();
#ifdef REM2D_PHASE_TIMING
    // warp-cycles per phase as seen by lane 0, per (mode, group shift): counters[REM2D_N_COUNTERS + ((mode * 6 + gs) * 16 + phase)]
    if (lane == 0) {
        PHASE(PH_LOOP);
        for (int i = 0; i < REM2D_N_PHASES; ++i)
            if (sim.ph[i] > 0) atomicAdd(&counters[REM2D_N_COUNTERS + ((tail ? 6 : 0) + gs) * REM2D_N_PHASES + i], (unsigned long long)sim.ph[i]);
    }
#endif
#pragma unroll
    for (int i = 0; i < REM2D_N_COUNTERS; ++i) {
        unsigned long long v = sim.cnt.c[i];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0 && v) atomicAdd(&counters[i], v);
    }
}
#define EPISODE_PARAMS const __grid_constant__ Layout L, int gs, int mode, float* slots, const int* __restrict__ order, int n_order, int* queue, \
                       DevPop p, const Terrain* __restrict__ ter, const Consts* __restrict__ k, int max_ticks, double* fitness, int* ticks, \
                       int* alive, int* status, unsigned long long* counters, ParkPolicy park, float* park_state, int* park_creature,      \
                       int* park_count, int first_slot, int n_slots
#define EPISODE_ARGS L, gs, mode, slots, order, n_order, queue, p, ter, k, max_ticks, fitness, ticks, alive, status, counters, park, park_state, \
                     park_creature, park_count, first_slot, n_slots
__global__ void __launch_bounds__(32, 1) episode_kernel(EPISODE_PARAMS) { episode_body(EPISODE_ARGS); }
__global__ void __launch_bounds__(32, 16) episode_kernel_r128(EPISODE_PARAMS) { episode_body(EPISODE_ARGS); }

void rem2d_launch_episode(const Layout& L, int image, int gs, int grid, cudaStream_t st, float* slots, const int* order, int n_order, int* queue,
                          DevPop p, const Terrain* ter, const Consts* k, int max_ticks, double* fitness, int* ticks, int* alive, int* status,
                          unsigned long long* counters, ParkPolicy park, float* park_state, int* park_creature, int* park_count) {
    const int smem = make_hot_layout(L, gs).rows * 128;
    if (image) episode_kernel_r128<<<grid, 32, smem, st>>>(L, gs, 0, slots, order, n_order, queue, p, ter, k, max_ticks, fitness, ticks, alive,
                                                            status, counters, park, park_state, park_creature, park_count, 0, 0);
    else episode_kernel<<<grid, 32, smem, st>>>(L, gs, 0, slots, order, n_order, queue, p, ter, k, max_ticks, fitness, ticks, alive, status,
                                                counters, park, park_state, park_creature, park_count, 0, 0);
}
// resident CTAs (= warps) of the episode kernel per SM for a given dynamic shared-memory size: registers AND shared memory
int rem2d_episode_blocks_per_sm(int image, int dyn_smem_bytes) {
    int n = 0;
    cudaError_t e = image ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, episode_kernel_r128, 32, (size_t)dyn_smem_bytes)
                          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, episode_kernel, 32, (size_t)dyn_smem_bytes);
    if (e != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
void rem2d_launch_tail(const Layout& L, int image, int gs, cudaStream_t st, float* park_state, int* park_creature, int first_slot, int n_parked,
                       const Terrain* ter, const Consts* k, int max_ticks, double* fitness, int* ticks, int* alive, int* status,
                       unsigned long long* counters, unsigned int* tail_trace) {
    ParkPolicy none = {0, 0, 0.0f, 0, 0, 0, nullptr, tail_trace};
    const int per = 32 >> gs, grid = (n_parked + per - 1) / per, smem = make_hot_layout(L, gs).rows * 128;
    if (image) episode_kernel_r128<<<grid, 32, smem, st>>>(L, gs, 1, nullptr, nullptr, 0, nullptr, DevPop(), ter, k, max_ticks, fitness, ticks,
                                                            alive, status, counters, none, park_state, park_creature, nullptr, first_slot,
                                                            n_parked);
    else episode_kernel<<<grid, 32, smem, st>>>(L, gs, 1, nullptr, nullptr, 0, nullptr, DevPop(), ter, k, max_ticks, fitness, ticks, alive, status,
                                                counters, none, park_state, park_creature, nullptr, first_slot, n_parked);
}
#endif

// Attributes: every translation unit sets those of its own kernel; rem2d_set_kernel_attributes (kernel 0's unit) calls all.
// All kernels that can be resident together should agree on the shared-memory carve-out of the SM: a small-smem kernel
// (tail) would otherwise pin its SMs in a large-L1 configuration and lock the big episode CTAs of other classes out
// (measured: 1.4x slower whole run when a tail kernel was resident next to the episode kernels).
cudaError_t rem2d_attr_step(int max_hot_bytes);
cudaError_t rem2d_attr_episode(int max_hot_bytes);
#if REM2D_KERNEL_ID == 0
cudaError_t rem2d_set_kernel_attributes(int max_hot_bytes) {
    cudaError_t e = rem2d_attr_step(max_hot_bytes);
    if (e != cudaSuccess) return e;
    return rem2d_attr_episode(max_hot_bytes);
}
#elif REM2D_KERNEL_ID == 1
cudaError_t rem2d_attr_step(int max_hot_bytes) {
    cudaError_t e = cudaFuncSetAttribute(step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_hot_bytes);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(step_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}
#elif REM2D_KERNEL_ID == 2
cudaError_t rem2d_attr_episode(int max_hot_bytes) {
    cudaError_t e = cudaFuncSetAttribute(episode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_hot_bytes);
    if (e != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(episode_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(episode_kernel_r128, cudaFuncAttributeMaxDynamicSharedMemorySize, max_hot_bytes)) != cudaSuccess) return e;
    return cudaFuncSetAttribute(episode_kernel_r128, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}
#endif
